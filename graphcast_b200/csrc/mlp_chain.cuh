// Fused layer CHAINS on tcgen05 tensor cores (sm_100a): up to GCB_MAX_CHAIN fused layers
// (see mlp_tc.cuh for one layer) over the same rows in ONE persistent kernel.
//
//   layer l:  y_l[r] = residual_l[r] + LN|swish( concat_s A_{l,s}(r) @ W_l + b_l + gathered addends )
//   where a segment A_{l,s} is an external operand image, an external fp32 table (gathered /
//   fan-in summed by the producer warps), or the RESULT OF AN EARLIER LAYER of the chain.
//
// A cluster pair owns a 128-row tile (N-split: CTA r computes output columns [256r, 256r+256)
// of every layer, the A block of each K-step is fetched once and multicast to both CTAs, as in
// mlp_tc.cuh) and takes it through the layers.  A layer whose result later layers consume
// ("keep") writes it, as an operand image, into a per-cluster SCRATCH ring in global memory:
// (lag * max_distance + 1) slots of 264 KB per kept layer and cluster, 40 MB for a whole
// two-layer MLP launch.  The ring is rewritten in place tile after tile by the same cluster and
// read back within microseconds, so it lives in the 126 MB L2 and never has to be written to
// HBM; the consumer streams it with the same TMA bulk copies as any other operand image.  This
// keeps the [rows, 512] hidden activation of every MLP (84 GB of HBM traffic per 0.25 degree
// step when the two linears were separate launches) on chip.
//
// Schedule.  Work is a sequence of UNITS (tile, layer); per cluster, step s runs the units
// (tile_{s - l*lag}, layer l) for l = 0..L-1 (or L-1..0: gcb_chain_desc.order), i.e. a tile advances one layer per `lag` steps, so
// that between a layer's MMAs and the dependent layer's MMAs the tensor pipe has `lag` other
// units to execute while the epilogue converts the accumulator and hands it over.  TMEM holds
// two 128x256 fp32 accumulators (unit u uses buffer u & 1).
//
// Hand-over protocol of a kept layer's scratch slot (both CTAs write half of the columns and
// both read all of them):
//   h_full[q][slot]  count 8: the 4 epilogue warps of BOTH CTAs arrive (release.cluster) after
//                    their st.global + fence.proxy.async; the TMA warp of each CTA waits
//                    (acquire.cluster) before the first bulk copy out of the slot.
//   h_free[q][slot]  count 2 x consumers: every consuming unit's MMA warp commits
//                    (tcgen05.commit, multicast to both CTAs) after its last MMA, i.e. when all
//                    bulk copies out of the slot have landed and been consumed in that CTA; the
//                    epilogue warps wait for it before overwriting the slot.
#pragma once
#include <type_traits>

#include "mlp_tc.cuh"

namespace gcb {

constexpr int kChainSlotsMax = 5;
constexpr int kScratchTileBytes = (kMaxN / kKStep) * GCB_A_IMAGE_BLOCK;   // 32 x 8448 = 270336
constexpr int kChainTailBytes = 3072;
// Epilogue warpgroups.  The epilogue is the critical path of every unit and is bound by
// instruction latency (one warp per scheduler: ncu source view, profiles/r02_ncu_full_chain_*): two
// warpgroups (warps 4-7 and 8-11) take alternate 32-column chunks of the unit's accumulator, warp w
// and w + 4 sharing a TMEM lane quarter.  Warps 12-15 gather the pre-activation addends (chunk c ->
// staging buffer c & 1 -> epilogue group c & 1); fp32-table segments are produced by the otherwise
// idle warps 2-3 of the issue warpgroup.
#ifndef GCB_EPI_GROUPS
#define GCB_EPI_GROUPS 2
#endif
constexpr int kEpiGroups = GCB_EPI_GROUPS;
constexpr int kGatherGroups = 3 - kEpiGroups;                  // producer warpgroups left: 1 or 2
constexpr int kATableWarps = 2;                                // warps 2 and 3
static_assert(kEpiGroups == 1 || kEpiGroups == 2, "one or two epilogue warpgroups");

// kBig: room for 8 instead of 4 [512]-float parameter vectors (biases, LayerNorm scale / offset):
// chains of two MLPs; costs 8 KB of shared memory (one operand stage in some variants).
template <bool kSplit, bool kPre, bool kBig>
struct ChainConfig {
  static constexpr int kParamVecs = kBig ? 8 : 4;
  static constexpr int kAStageBytes = kSplit ? 2 * kAPartBytes : kAPartBytes;
  static constexpr int kBStageBytes = kSplit ? 2 * kBPartBytes : kBPartBytes;
  static constexpr int kStageBytes = kAStageBytes + kBStageBytes;
  static constexpr int kParamBytes = kParamVecs * kMaxN * 4;
  static constexpr int kGRegionBytes = kPre ? kGBytes : 0;
  static constexpr int kFixedBytes =
      kParamBytes + kEpiGroups * kEpiStageBytes + kGRegionBytes + kEpiGroups * kLnxBytes + kChainTailBytes;
  static constexpr int kFit = (kSmemLimit - kFixedBytes) / kStageBytes;
#ifdef GCB_FORCE_STAGES          // experiment: sensitivity of a launch to the ring depth
  static constexpr int kStages = GCB_FORCE_STAGES < kFit ? GCB_FORCE_STAGES : kFit;
#else
  static constexpr int kStages = kFit < 12 ? kFit : 12;
#endif
  static constexpr int kSmemBytes = kStages * kStageBytes + kFixedBytes;
  static_assert(kStages >= 4, "operand ring too shallow");
};

struct ChainSeg {
  const float* table;
  const int32_t* idx;
  const uint8_t* img;
  int ld, k_valid, fan, ksteps;
  int src_q;          // >= 0: scratch ring q (result of an earlier layer); else external
  int pad_;
};

// kKindLN*: LayerNorm without residual / with an fp32 residual / with an operand-image residual
enum { kKindPlain = 0, kKindSwish = 1, kKindLN = 2, kKindLNRes = 3, kKindLNImg = 4 };

struct ChainLayer {
  const uint8_t* w;
  const float* residual;
  float* out;
  float* out_y;
  uint8_t* out_img;
  const uint8_t* res_img;
  int ld_res, ld_out, ld_outy;
  int nseg, ksteps, n_pre, kind;
  int bias_off, scale_off, offset_off;   // float offsets into the parameter area, -1 = none
  int keep_q;                            // scratch ring this layer writes, -1 = none
  int has_table;                         // some segment is an fp32 table (producer warps)
  int res_q;                             // residual = the kept result in scratch ring res_q, -1 = none
};

template <bool kSplit, bool kPre, bool kBig>
__global__ void __launch_bounds__(kThreads, 1)
mlp_chain_tc_kernel(const __grid_constant__ gcb_chain_desc d, const int nq, const int nslots) {
  using Cfg = ChainConfig<kSplit, kPre, kBig>;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* stage_base = smem;
  float* s_param = reinterpret_cast<float*>(smem + Cfg::kStages * Cfg::kStageBytes);
  float* s_epi = s_param + Cfg::kParamBytes / 4;                    // [kEpiGroups][4][32][36]
  float* s_g = s_epi + kEpiGroups * 4 * 32 * kEpiRowFloats;         // [2][128][36] (kPre only)
  float2* s_lnx = reinterpret_cast<float2*>(reinterpret_cast<uint8_t*>(s_g) + Cfg::kGRegionBytes);  // [kEpiGroups][2][128]
  uint8_t* tail = reinterpret_cast<uint8_t*>(s_lnx) + kEpiGroups * kLnxBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);          // [12]
  uint64_t* empty_bar = full_bar + 12;                             // [12]
  uint64_t* tmem_full_bar = empty_bar + 12;                        // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;                    // [2]
  uint64_t* g_full_bar = tmem_empty_bar + 2;                       // [2]
  uint64_t* g_empty_bar = g_full_bar + 2;                          // [2]
  uint64_t* lnx_bar = g_empty_bar + 2;                             // [kEpiGroups][2]
  uint64_t* h_full_bar = lnx_bar + 4;                              // [GCB_MAX_CHAIN][kChainSlotsMax]
  uint64_t* h_free_bar = h_full_bar + GCB_MAX_CHAIN * kChainSlotsMax;
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(h_free_bar + GCB_MAX_CHAIN * kChainSlotsMax);
  ChainLayer* s_layer = reinterpret_cast<ChainLayer*>(tmem_base_slot + 2);           // [4]
  ChainSeg* s_seg = reinterpret_cast<ChainSeg*>(s_layer + GCB_MAX_CHAIN);            // [4][3]
  PreAddInfo* s_pre = reinterpret_cast<PreAddInfo*>(s_seg + GCB_MAX_CHAIN * 3);      // [4][2]
  static_assert((2 * 12 + 12 + 2 * GCB_MAX_CHAIN * kChainSlotsMax) * 8 + 8 +
                    GCB_MAX_CHAIN * (sizeof(ChainLayer) + 3 * sizeof(ChainSeg) + 2 * sizeof(PreAddInfo))
                    <= kChainTailBytes, "tail region too small");

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int L = d.nlayers;
  const int lag = d.lag > 0 ? d.lag : 1;
  // Unit order inside a step: ascending (layer 0 first) or descending.  Descending, a kept
  // result is consumed (by the next layer, one step later) BEFORE the producing layer's next
  // unit writes again, so lag*distance slots per scratch ring suffice instead of lag*distance+1
  // - what keeps the rings of a 4-layer chain inside the L2.  It shortens the distance between
  // dependent units from L+1 to L-1 units, so it is used for chains of 3 and more layers.
  const bool desc = d.order != 0;
  const long long rows_total = d.rows;
  const int num_tiles = (d.rows + kTileM - 1) / kTileM;
  const uint32_t crank = ptx::cluster_ctarank();
  const uint32_t cid = ptx::cluster_id_x();
  const uint32_t ncl = ptx::num_clusters_x();
  const uint32_t peer = crank ^ 1u;
  constexpr uint16_t cmask = 3;
  // Tiles of this cluster: cid, cid + ncl, ...
  const int T = (num_tiles > static_cast<int>(cid))
                    ? (num_tiles - static_cast<int>(cid) + static_cast<int>(ncl) - 1) / static_cast<int>(ncl)
                    : 0;
  const int nsteps = T > 0 ? T + (L - 1) * lag : 0;
  uint8_t* const scratch = static_cast<uint8_t*>(d.scratch) +
                           static_cast<size_t>(cid) * nq * nslots * kScratchTileBytes;
  auto scratch_slot = [&](int q, int ti) -> uint8_t* {
    return scratch + (static_cast<size_t>(q) * nslots + (ti % nslots)) * kScratchTileBytes;
  };
  bool any_table = false;
  for (int l = 0; l < L; ++l)
    for (int s = 0; s < d.layer[l].nseg; ++s)
      any_table = any_table || (d.layer[l].seg_from[s] < 0 && d.layer[l].seg[s].img == nullptr);

  // ---- one-time setup ---------------------------------------------------------
  {
    // Parameter vectors in layer order: [bias] [ln scale, ln offset] per layer (every thread
    // derives the same offsets, so no synchronisation is needed before the copy).
    int off = 0;
    for (int l = 0; l < L; ++l) {
      const gcb_chain_layer& gl = d.layer[l];
      if (gl.bias != nullptr) {
        for (int i = threadIdx.x; i < kMaxN; i += kThreads) s_param[off + i] = gl.bias[i];
        off += kMaxN;
      }
      if (gl.ln_scale != nullptr) {
        for (int i = threadIdx.x; i < kMaxN; i += kThreads) {
          s_param[off + i] = gl.ln_scale[i];
          s_param[off + kMaxN + i] = gl.ln_offset[i];
        }
        off += 2 * kMaxN;
      }
    }
  }
  if (threadIdx.x == 0) {
    int off = 0, q = 0;
    int q_of_layer[GCB_MAX_CHAIN];
    int consumers[GCB_MAX_CHAIN];
    for (int l = 0; l < L; ++l) { q_of_layer[l] = -1; consumers[l] = 0; }
    for (int l = 0; l < L; ++l) {
      const gcb_chain_layer& gl = d.layer[l];
      ChainLayer& cl = s_layer[l];
      cl.w = static_cast<const uint8_t*>(gl.w_packed);
      cl.residual = gl.residual; cl.out = gl.out; cl.out_y = gl.out_y;
      cl.out_img = static_cast<uint8_t*>(gl.out_img);
      cl.res_img = static_cast<const uint8_t*>(gl.residual_img);
      cl.ld_res = gl.ld_res; cl.ld_out = gl.ld_out; cl.ld_outy = gl.ld_out_y;
      cl.nseg = gl.nseg; cl.n_pre = gl.n_pre_add;
      cl.res_q = gl.residual_keep > 0 ? q_of_layer[gl.residual_keep - 1] : -1;
      cl.kind = gl.ln_scale != nullptr
                    ? (gl.residual != nullptr
                           ? kKindLNRes
                           : ((gl.residual_img != nullptr || gl.residual_keep > 0) ? kKindLNImg : kKindLN))
                    : (gl.act == GCB_ACT_SWISH ? kKindSwish : kKindPlain);
      cl.bias_off = -1; cl.scale_off = -1; cl.offset_off = -1;
      if (gl.bias != nullptr) { cl.bias_off = off; off += kMaxN; }
      if (gl.ln_scale != nullptr) { cl.scale_off = off; cl.offset_off = off + kMaxN; off += 2 * kMaxN; }
      cl.keep_q = -1;
      if (gl.keep) { cl.keep_q = q; q_of_layer[l] = q; ++q; }
      int ks = 0, has_table = 0;
      for (int s = 0; s < gl.nseg; ++s) {
        ChainSeg& cs = s_seg[l * 3 + s];
        const int from = gl.seg_from[s];
        cs.table = gl.seg[s].table; cs.idx = gl.seg[s].idx;
        cs.img = static_cast<const uint8_t*>(gl.seg[s].img);
        cs.ld = gl.seg[s].ld; cs.k_valid = gl.seg[s].k_valid; cs.fan = gl.seg[s].fan;
        cs.ksteps = (from >= 0 ? kMaxN : gl.seg[s].k) / kKStep;
        cs.src_q = from >= 0 ? q_of_layer[from] : -1;
        if (from >= 0) { cs.img = nullptr; ++consumers[from]; }
        else if (cs.img == nullptr) has_table = 1;
        ks += cs.ksteps;
      }
      cl.ksteps = ks; cl.has_table = has_table;
      for (int s = 0; s < gl.n_pre_add; ++s) {
        s_pre[l * 2 + s].table = gl.pre_add[s].table;
        s_pre[l * 2 + s].idx = gl.pre_add[s].idx;
        s_pre[l * 2 + s].ld = gl.pre_add[s].ld;
      }
    }
    for (int s = 0; s < Cfg::kStages; ++s) {
      ptx::mbar_init(&full_bar[s], any_table ? 1 + kATableWarps : 1);   // TMA lane (+ the A-table warps)
      ptx::mbar_init(&empty_bar[s], 2);                   // tcgen05.commit of both CTAs
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(&tmem_full_bar[b], 1);
      ptx::mbar_init(&tmem_empty_bar[b], 4 * kEpiGroups);   // every epilogue warp
      ptx::mbar_init(&g_full_bar[b], 4);        // the 4 warps of the gather group that filled it
      ptx::mbar_init(&g_empty_bar[b], 4);       // the 4 warps of the epilogue group that read it
      for (int eg = 0; eg < kEpiGroups; ++eg) ptx::mbar_init(&lnx_bar[eg * 2 + b], 1);
    }
    for (int l = 0; l < L; ++l) {
      if (q_of_layer[l] < 0) continue;
      for (int sl = 0; sl < nslots; ++sl) {
        ptx::mbar_init(&h_full_bar[q_of_layer[l] * kChainSlotsMax + sl], 8 * kEpiGroups);
        ptx::mbar_init(&h_free_bar[q_of_layer[l] * kChainSlotsMax + sl],
                       2 * (consumers[l] > 0 ? consumers[l] : 1));
      }
    }
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_base_slot, kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::cluster_sync_all();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_base_slot;

  // ---- roles ------------------------------------------------------------------
  // Register re-allocation per warpgroup (setmaxnreg): the epilogue is the critical path of
  // every unit and, at the 128 registers a 512-thread CTA starts with, it spills its residual /
  // staging values to local memory inside the chunk loops; the issue warps need a fraction of
  // that.  One epilogue group: 56 x 4 + 216 x 4 + 112 x 8 warps = 1984; two: 72 x 4 + 176 x 8 +
  // 88 x 4 = 2048 of the 2048 register slices of the SM.
  constexpr int kRegsCtl = kEpiGroups == 2 ? 72 : 56;
  constexpr int kRegsEpi = kEpiGroups == 2 ? 176 : 216;
  constexpr int kRegsProd = kEpiGroups == 2 ? 88 : 112;
  if (warp < 4) {
    ptx::setmaxnreg_dec<kRegsCtl>();
  if (warp == 0) {
    // ===== TMA warp (converged; every lane polls, one elected lane issues) =====
    const uint32_t b_bytes = Cfg::kBStageBytes;
    const size_t b_block = 2 * kBPartBytes;
    const size_t b_stride = 2 * b_block;                          // n = 512: two blocks per K-step
    const uint32_t a_bytes = Cfg::kAStageBytes;
    const uint32_t a_half = a_bytes / 2;
    uint32_t stage = 0, phase = 0, tu = 0;
    const uint64_t keep_policy = ptx::l2_policy_evict_last();
    for (int st = 0; st < nsteps; ++st) {
      for (int li = 0; li < L; ++li) {
        const int l = desc ? L - 1 - li : li;
        const int ti = st - l * lag;
        if (ti < 0 || ti >= T) continue;
        const uint32_t tile = cid + static_cast<uint32_t>(ti) * ncl;
        const int nseg = s_layer[l].nseg;
        const uint8_t* b_ptr = s_layer[l].w + static_cast<size_t>(crank) * b_block;
        const bool tr = tracing(tu);
        long long blocked = 0, hwait = 0;
        for (int s = 0; s < nseg; ++s) {
          const ChainSeg sg = s_seg[l * 3 + s];
          const uint8_t* a_ptr = nullptr;
          bool a_copy = false;
          const bool a_scratch = sg.src_q >= 0;
          if (sg.src_q >= 0) {
            const long long w0 = tr ? clock64() : 0;
            // Poll at CTA scope (a cluster-scope acquire per retry is far more expensive), then
            // take the cluster-scope acquire once on the completed phase.
            ptx::mbar_wait(&h_full_bar[sg.src_q * kChainSlotsMax + (ti % nslots)],
                           static_cast<uint32_t>(ti / nslots) & 1u);
            ptx::mbar_wait_cluster(&h_full_bar[sg.src_q * kChainSlotsMax + (ti % nslots)],
                                   static_cast<uint32_t>(ti / nslots) & 1u);
            if (tr) hwait += clock64() - w0;
            a_ptr = scratch_slot(sg.src_q, ti) + crank * a_half;
            a_copy = true;
          } else if (sg.img != nullptr) {
            a_ptr = sg.img + static_cast<size_t>(tile) * sg.ksteps * GCB_A_IMAGE_BLOCK + crank * a_half;
            a_copy = true;
          }
          const uint32_t tx = b_bytes + (a_copy ? a_bytes : 0u);
          for (int k = 0; k < sg.ksteps; ++k) {
            const long long w0 = tr ? clock64() : 0;
            ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
            if (tr) blocked += clock64() - w0;
            uint8_t* a_dst = stage_base + stage * Cfg::kStageBytes;
            if (ptx::elect_one()) {
              ptx::mbar_arrive_expect_tx(&full_bar[stage], tx);
              if (a_scratch)
                ptx::bulk_g2s_multicast_hint(a_dst + crank * a_half, a_ptr, a_half, &full_bar[stage], cmask, keep_policy);
              else if (a_copy)
                ptx::bulk_g2s_multicast(a_dst + crank * a_half, a_ptr, a_half, &full_bar[stage], cmask);
              ptx::bulk_g2s(a_dst + Cfg::kAStageBytes, b_ptr, b_bytes, &full_bar[stage]);
            }
            __syncwarp();
            a_ptr += GCB_A_IMAGE_BLOCK;
            b_ptr += b_stride;
            if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
          }
        }
        if (lane == 0) { trace_val(tu, 7, blocked); trace_val(tu, 8, hwait); trace_val(tu, 11, l); }
        ++tu;
      }
    }
  } else if (warp == 1) {
    // ===== MMA warp =====
    const uint32_t idesc = ptx::make_idesc_bf16(kTileM, kUnitN);
    uint32_t stage = 0, phase = 0, u = 0;
    for (int st = 0; st < nsteps; ++st) {
      for (int li = 0; li < L; ++li) {
        const int l = desc ? L - 1 - li : li;
        const int ti = st - l * lag;
        if (ti < 0 || ti >= T) continue;
        const uint32_t buf = u & 1;
        ptx::mbar_wait(&tmem_empty_bar[buf], ((u >> 1) & 1) ^ 1);
        ptx::tc_fence_after_sync();
        if (lane == 0) trace(u, 0);
        const uint32_t dcol = tmem_base + buf * kUnitN;
        const int ksteps = s_layer[l].ksteps;
        const bool tr = tracing(u);
        long long starved = 0;
        for (int ks = 0; ks < ksteps; ++ks) {
          const long long w0 = tr ? clock64() : 0;
          ptx::mbar_wait(&full_bar[stage], phase);
          if (tr) starved += clock64() - w0;
          ptx::tc_fence_after_sync();
          if (ks == 0 && lane == 0) trace(u, 1);
          const uint32_t sa = ptx::smem_addr(stage_base + stage * Cfg::kStageBytes);
          const uint32_t sb = sa + Cfg::kAStageBytes;
          const uint64_t a_hi = ptx::make_smem_desc(sa, kALbo, 128);
          const uint64_t b_hi = ptx::make_smem_desc(sb, kBLbo, 128);
          if (ptx::elect_one()) {
            ptx::mma_bf16_ss(dcol, a_hi, b_hi, idesc, ks > 0 ? 1u : 0u);
            if (kSplit) {
              const uint64_t a_lo = a_hi + (kAPartBytes >> 4);
              const uint64_t b_lo = b_hi + (kBPartBytes >> 4);
              ptx::mma_bf16_ss(dcol, a_hi, b_lo, idesc, 1u);
              ptx::mma_bf16_ss(dcol, a_lo, b_hi, idesc, 1u);
            }
            ptx::mma_commit_multicast(&empty_bar[stage], cmask);
          }
          __syncwarp();
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
        if (ptx::elect_one()) {
          ptx::mma_commit(&tmem_full_bar[buf]);
          // Every scratch slot this unit read is reusable (in both CTAs) once these MMAs retire.
          const int nseg = s_layer[l].nseg;
          for (int s = 0; s < nseg; ++s) {
            const int q = s_seg[l * 3 + s].src_q;
            if (q >= 0) ptx::mma_commit_multicast(&h_free_bar[q * kChainSlotsMax + (ti % nslots)], cmask);
          }
        }
        __syncwarp();
        if (lane == 0) { trace(u, 2); trace_val(u, 6, starved); }
        ++u;
      }
    }
  } else if (any_table) {
    // ===== A-table warps (2 and 3): segments given as fp32 tables =====
    // Gather through the segment's index, optional fan-in sum, split to bf16 hi / lo, store in
    // the UMMA K-major core-matrix layout.  They arrive on EVERY K-step's full barrier (for image
    // / scratch K-steps without writing anything), so the barrier count is uniform.
    const int t64 = threadIdx.x - 64;
    const int sub = t64 & 3;                        // which float4 of the 16-wide K-step
    const int rg = t64 >> 2;                        // 0..15; rows rg + 16*i
    const uint32_t sts_off = (sub >> 1) * kALbo + (sub & 1) * 8;
    uint32_t stage = 0, phase = 0;
    for (int st = 0; st < nsteps; ++st) {
      for (int li = 0; li < L; ++li) {
        const int l = desc ? L - 1 - li : li;
        const int ti = st - l * lag;
        if (ti < 0 || ti >= T) continue;
        const uint32_t tile = cid + static_cast<uint32_t>(ti) * ncl;
        const int nseg = s_layer[l].nseg;
        for (int s = 0; s < nseg; ++s) {
          const ChainSeg sg = s_seg[l * 3 + s];
          const bool is_tab = sg.src_q < 0 && sg.img == nullptr;
          int src[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            src[i] = -1;
            if (is_tab) {
              const long long grow = static_cast<long long>(tile) * kTileM + rg + 16 * i;
              if (grow < rows_total) src[i] = sg.idx ? __ldg(sg.idx + grow) : static_cast<int>(grow);
            }
          }
          for (int k = 0; k < sg.ksteps; ++k) {
            float4 cur[8];
            if (is_tab) {
              const int koff = k * kKStep + sub * 4;
              const bool kvalid = koff < sg.k_valid;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                if (kvalid && src[i] >= 0) {
                  const float* p = sg.table + static_cast<long long>(src[i]) * sg.fan * sg.ld + koff;
                  acc = __ldg(reinterpret_cast<const float4*>(p));
                  for (int j = 1; j < sg.fan; ++j) {
                    const float4 t = __ldg(reinterpret_cast<const float4*>(p + static_cast<long long>(j) * sg.ld));
                    acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
                  }
                }
                cur[i] = acc;
              }
            }
            ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
            if (is_tab) {
              uint8_t* a_hi = stage_base + stage * Cfg::kStageBytes;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                uint2 hi, lo;
                ptx::split_bf16x4(cur[i], hi, lo);
                const uint32_t off = sts_off + (rg + 16 * i) * 16;
                *reinterpret_cast<uint2*>(a_hi + off) = hi;
                if (kSplit) *reinterpret_cast<uint2*>(a_hi + kAPartBytes + off) = lo;
              }
              ptx::fence_proxy_async_smem();
            }
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&full_bar[stage]);
            if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  }
  } else if (warp < 4 + 4 * kEpiGroups) {
    // ===== epilogue =====
    ptx::setmaxnreg_inc<kRegsEpi>();
    const int eg = (warp - 4) >> 2;               // epilogue group: chunks with (chunk & 1) == eg
    const int ew = warp & 3;                      // TMEM lane quarter
    const uint32_t lane_base = static_cast<uint32_t>(ew * 32) << 16;
    float* my_epi = s_epi + (eg * 4 + ew) * 32 * kEpiRowFloats;
    float2* my_lnx = s_lnx + eg * 2 * kTileM;     // [2][128] of this group
    uint64_t* my_lnx_bar = lnx_bar + eg * 2;
    const int cg = lane & 7;
    const int rsub = lane >> 3;
    const int col_base = static_cast<int>(crank) * kUnitN;   // my 256 columns of every layer
    uint32_t g_count = 0, ln_count = 0, u = 0;
    const uint64_t keep_policy = ptx::l2_policy_evict_last();

    // Per-unit context, passed BY VALUE: as mutable locals captured by reference these lived in
    // local memory and every use in the chunk loops was an LDL on the critical path.
    struct EpiCtx {
      float* out_ptr; float* outy_ptr; const float* res_ptr;
      long long ld_out, ld_outy, ld_res;
      uint8_t* img0;                  // external operand image of this TILE (block base), or null
      uint8_t* img1;                  // scratch slot of this tile, or null
      const uint8_t* res_img;         // residual as an operand image: block base of this TILE, or null
      const float* s_bias; const float* s_scale; const float* s_offset;
      int n_pre;
      int trace_u;                    // unit index when this unit is traced, else -1
    };

    auto finish_unit = [&](auto kind_tag, const EpiCtx cx, uint32_t g_count_in, uint32_t taddr,
                           long long row0, float mean, float rstd) -> uint32_t {
      constexpr int kind = decltype(kind_tag)::value;
      uint32_t g_count = g_count_in;
      // Compile-time leanness: a swish layer only feeds later layers (operand image / scratch, no
      // fp32 output, no residual) and a plain layer has no residual (validate_chain enforces both),
      // so those paths - and the registers they keep alive - exist in the LayerNorm variant only.
      constexpr bool is_ln = kind >= kKindLN;
      float* const out_ptr = kind == kKindSwish ? nullptr : cx.out_ptr;
      float* const outy_ptr = kind == kKindSwish ? nullptr : cx.outy_ptr;
      const float* const res_ptr = kind == kKindLNRes ? cx.res_ptr : nullptr;
      const uint8_t* const res_img = kind == kKindLNImg ? cx.res_img : nullptr;
      const long long ld_out = cx.ld_out, ld_outy = cx.ld_outy, ld_res = cx.ld_res;
      uint8_t* const img0 = cx.img0; uint8_t* const img1 = cx.img1;
      const float* const s_bias = cx.s_bias; const float* const s_scale = cx.s_scale;
      const float* const s_offset = cx.s_offset;
      const int n_pre = cx.n_pre;
      const bool rows_full = row0 + 32 <= rows_total;
      const bool want_img = (img0 != nullptr) || (img1 != nullptr);
      // Residual of the CURRENT chunk, requested at the end of the previous one.
      //   rr     fp32 master, coalesced layout: rows rsub + 4i, 16 bytes at column cg*4
      //   rh/rl  operand image (hi | lo bf16), thread = row layout: the four 16-byte pieces
      //          (K-step ks2, chunk c) of this thread's row
      float4 rr[8];
      uint4 rh[4], rl[4];
      const size_t row_off = static_cast<size_t>(ew * 32 + lane) * 16;
      auto load_res = [&](int c0) {
        if (kind == kKindLNRes && rows_full) {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            rr[i] = *reinterpret_cast<const float4*>(res_ptr + (row0 + rsub + 4 * i) * ld_res + col_base + c0 + cg * 4);
        }
        if (kind == kKindLNImg) {
          const uint8_t* b = res_img + static_cast<size_t>((col_base + c0) >> 4) * GCB_A_IMAGE_BLOCK + row_off;
#pragma unroll
          for (int ks2 = 0; ks2 < 2; ++ks2) {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              rh[ks2 * 2 + c] = *reinterpret_cast<const uint4*>(b + ks2 * GCB_A_IMAGE_BLOCK + c * kALbo);
              rl[ks2 * 2 + c] = *reinterpret_cast<const uint4*>(b + ks2 * GCB_A_IMAGE_BLOCK + c * kALbo + kAPartBytes);
            }
          }
        }
      };
      constexpr int kChunkStep = 32 * kEpiGroups;          // my chunks: eg, eg + kEpiGroups, ...
      load_res(32 * eg);
      const bool trp = cx.trace_u >= 0 && ew == 0 && lane == 0 && eg == 0;
      long long t_ld = 0, t_math = 0, t_f32 = 0, t_img = 0;
      for (int c0 = 32 * eg; c0 < kUnitN; c0 += kChunkStep) {
        const int gc0 = col_base + c0;
        const int col = gc0 + cg * 4;
        float v[32];
        long long tp = trp ? clock64() : 0;
        ptx::tmem_ld32(taddr + c0, v);
        if (trp) { const long long t = clock64(); t_ld += t - tp; tp = t; }
        if (s_bias != nullptr) {
          float b[32];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(&b[4 * q]) = *reinterpret_cast<const float4*>(s_bias + gc0 + 4 * q);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] += b[j];
        }
        if (kPre && !is_ln && n_pre > 0) {
          // staging buffer = chunk parity; with two epilogue groups that is my group index and
          // every fill of that buffer is mine
          const uint32_t gb = kEpiGroups == 2 ? static_cast<uint32_t>(eg) : (g_count & 1);
          ptx::mbar_wait(&g_full_bar[gb], (kEpiGroups == 2 ? g_count : (g_count >> 1)) & 1);
          const float* gp = s_g + gb * kGBufFloats + (ew * 32 + lane) * kEpiRowFloats;
          float g[32];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(&g[4 * q]) = *reinterpret_cast<const float4*>(gp + 4 * q);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] += g[j];
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&g_empty_bar[gb]);
          ++g_count;
        }
        if (kind == kKindSwish) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = swish_f(v[j]);
        }
        if (is_ln) {
          float g[32];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(&g[4 * q]) = *reinterpret_cast<const float4*>(s_scale + gc0 + 4 * q);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = (v[j] - mean) * rstd * g[j];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(&g[4 * q]) = *reinterpret_cast<const float4*>(s_offset + gc0 + 4 * q);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] += g[j];
        }
        if (trp) { const long long t = clock64(); t_math += t - tp; tp = t; }
        if (out_ptr != nullptr || outy_ptr != nullptr) {
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(my_epi + lane * kEpiRowFloats + q * 4) =
                make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          __syncwarp();
          if (rows_full) {
            float4 y[8];
#pragma unroll
            for (int i = 0; i < 8; ++i)
              y[i] = *reinterpret_cast<const float4*>(my_epi + (rsub + 4 * i) * kEpiRowFloats + cg * 4);
            if (outy_ptr != nullptr) {
#pragma unroll
              for (int i = 0; i < 8; ++i)
                *reinterpret_cast<float4*>(outy_ptr + (row0 + rsub + 4 * i) * ld_outy + col) = y[i];
            }
            if (res_ptr != nullptr) {
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                y[i].x += rr[i].x; y[i].y += rr[i].y; y[i].z += rr[i].z; y[i].w += rr[i].w;
              }
            }
            if (out_ptr != nullptr) {
#pragma unroll
              for (int i = 0; i < 8; ++i)
                *reinterpret_cast<float4*>(out_ptr + (row0 + rsub + 4 * i) * ld_out + col) = y[i];
            }
            if (want_img && res_ptr != nullptr) {
#pragma unroll
              for (int i = 0; i < 8; ++i)
                *reinterpret_cast<float4*>(my_epi + (rsub + 4 * i) * kEpiRowFloats + cg * 4) = y[i];
            }
          } else {
            for (int i = 0; i < 8; ++i) {
              const int r = rsub + 4 * i;
              const long long grow = row0 + r;
              if (grow < rows_total) {
                for (int e = 0; e < 4; ++e) {
                  const float yv = my_epi[r * kEpiRowFloats + cg * 4 + e];
                  const float ov = yv + (res_ptr ? res_ptr[grow * ld_res + col + e] : 0.f);
                  if (outy_ptr != nullptr) outy_ptr[grow * ld_outy + col + e] = yv;
                  if (out_ptr != nullptr) out_ptr[grow * ld_out + col + e] = ov;
                  if (want_img) my_epi[r * kEpiRowFloats + cg * 4 + e] = ov;
                }
              }
            }
          }
          __syncwarp();
          if (want_img && res_ptr != nullptr) {
#pragma unroll
            for (int q = 0; q < 8; ++q)
              *reinterpret_cast<float4*>(&v[4 * q]) =
                  *reinterpret_cast<const float4*>(my_epi + lane * kEpiRowFloats + q * 4);
            __syncwarp();
          }
        } else if (want_img && res_ptr != nullptr) {
          // Image-only result with an fp32 residual: transpose the coalesced residual rows to the
          // thread = row layout through the tile.
          if (rows_full) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              *reinterpret_cast<float4*>(my_epi + (rsub + 4 * i) * kEpiRowFloats + cg * 4) = rr[i];
            __syncwarp();
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 t = *reinterpret_cast<const float4*>(my_epi + lane * kEpiRowFloats + q * 4);
              v[4 * q] += t.x; v[4 * q + 1] += t.y; v[4 * q + 2] += t.z; v[4 * q + 3] += t.w;
            }
            __syncwarp();
          } else {
            const long long grow = row0 + lane;
            if (grow < rows_total) {
              const float* rp = res_ptr + grow * ld_res + gc0;
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float4 t = *reinterpret_cast<const float4*>(rp + 4 * q);
                v[4 * q] += t.x; v[4 * q + 1] += t.y; v[4 * q + 2] += t.z; v[4 * q + 3] += t.w;
              }
            }
          }
        }
        if (trp) { const long long t = clock64(); t_f32 += t - tp; tp = t; }
        if (kind == kKindLNImg) {
          // Residual held as an operand image (x = hi + lo, two bf16): already in this thread's
          // row layout.  A packed word holds element 2k in its low and 2k+1 in its high half.
#pragma unroll
          for (int pc = 0; pc < 4; ++pc) {
            const uint32_t hw[4] = {rh[pc].x, rh[pc].y, rh[pc].z, rh[pc].w};
            const uint32_t lw[4] = {rl[pc].x, rl[pc].y, rl[pc].z, rl[pc].w};
#pragma unroll
            for (int k2 = 0; k2 < 4; ++k2) {
              v[pc * 8 + 2 * k2] += __uint_as_float(hw[k2] << 16) + __uint_as_float(lw[k2] << 16);
              v[pc * 8 + 2 * k2 + 1] += __uint_as_float(hw[k2] & 0xffff0000u) + __uint_as_float(lw[k2] & 0xffff0000u);
            }
          }
        }
        if (want_img) {
          // thread = row: the 16-byte pieces of 32 consecutive rows are contiguous -> 512-byte
          // coalesced warp stores, to the external image and / or the scratch slot.
          const size_t boff = static_cast<size_t>(gc0 >> 4) * GCB_A_IMAGE_BLOCK + row_off;
#pragma unroll
          for (int ks2 = 0; ks2 < 2; ++ks2) {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              const float* x = &v[ks2 * 16 + c * 8];
              uint2 h0, l0, h1, l1;
              ptx::split_bf16x4(make_float4(x[0], x[1], x[2], x[3]), h0, l0);
              ptx::split_bf16x4(make_float4(x[4], x[5], x[6], x[7]), h1, l1);
              const size_t o = boff + ks2 * GCB_A_IMAGE_BLOCK + c * kALbo;
              if (img0 != nullptr) {
                *reinterpret_cast<uint4*>(img0 + o) = make_uint4(h0.x, h0.y, h1.x, h1.y);
                *reinterpret_cast<uint4*>(img0 + o + kAPartBytes) = make_uint4(l0.x, l0.y, l1.x, l1.y);
              }
              if (img1 != nullptr) {       // scratch slot: keep these lines in the L2
                ptx::st_global_v4_hint(img1 + o, make_uint4(h0.x, h0.y, h1.x, h1.y), keep_policy);
                ptx::st_global_v4_hint(img1 + o + kAPartBytes, make_uint4(l0.x, l0.y, l1.x, l1.y), keep_policy);
              }
            }
          }
        }
        // Next chunk's residual: requested once this chunk's values are dead (no extra registers);
        // the line is already in L2 (prefetched a step ahead), so the TMEM load and LayerNorm
        // math of the next chunk cover its latency.
        if (c0 + kChunkStep < kUnitN) load_res(c0 + kChunkStep);
        if (trp) { const long long t = clock64(); t_img += t - tp; tp = t; }
      }
      if (trp) {
        trace_val(cx.trace_u, 12, t_ld); trace_val(cx.trace_u, 13, t_math);
        trace_val(cx.trace_u, 14, t_f32); trace_val(cx.trace_u, 15, t_img);
      }
      return g_count;
    };

    auto unit_stats = [&](const float* s_bias, uint32_t taddr, LnStats& st) {
      for (int c0 = 0; c0 < kUnitN; c0 += 32) {
        float v[32];
        ptx::tmem_ld32(taddr + c0, v);
        if (s_bias != nullptr) {
          float b[32];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(&b[4 * q]) = *reinterpret_cast<const float4*>(s_bias + col_base + c0 + 4 * q);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] += b[j];
        }
        st.add_block(v, 32);
      }
    };

    for (int st = 0; st < nsteps; ++st) {
      for (int li = 0; li < L; ++li) {
        const int l = desc ? L - 1 - li : li;
        const int ti = st - l * lag;
        if (ti < 0 || ti >= T) continue;
        const uint32_t tile = cid + static_cast<uint32_t>(ti) * ncl;
        const long long row0 = static_cast<long long>(tile) * kTileM + ew * 32;
        const ChainLayer& cl = s_layer[l];
        EpiCtx cx;
        cx.out_ptr = cl.out; cx.outy_ptr = cl.out_y; cx.res_ptr = cl.residual;
        cx.ld_out = cl.ld_out; cx.ld_outy = cl.ld_outy; cx.ld_res = cl.ld_res;
        cx.s_bias = cl.bias_off >= 0 ? s_param + cl.bias_off : nullptr;
        cx.s_scale = cl.scale_off >= 0 ? s_param + cl.scale_off : nullptr;
        cx.s_offset = cl.offset_off >= 0 ? s_param + cl.offset_off : nullptr;
        cx.n_pre = cl.n_pre;
        cx.trace_u = tracing(u) ? static_cast<int>(u) : -1;
        cx.img0 = cl.out_img != nullptr
                      ? cl.out_img + static_cast<size_t>(tile) * (kMaxN / kKStep) * GCB_A_IMAGE_BLOCK
                      : nullptr;
        cx.img1 = nullptr;
        cx.res_img = cl.res_img != nullptr
                         ? cl.res_img + static_cast<size_t>(tile) * (kMaxN / kKStep) * GCB_A_IMAGE_BLOCK
                         : nullptr;
        // Residual = the kept result of an earlier layer: the slot this CTA's epilogue wrote for
        // this tile (same threads, same rows and columns: program order makes it visible, and the
        // slot cannot be rewritten before these warps reach tile ti + nslots themselves).
        if (cl.res_q >= 0) cx.res_img = scratch_slot(cl.res_q, ti);
        if (eg == 0 && ti + 1 < T && (cl.residual != nullptr || cl.res_img != nullptr)) {
          // Pull the residual of this layer's NEXT tile into L2 now (a whole step ahead).
          const uint32_t ntile = tile + ncl;
          if (cl.residual != nullptr) {
            const long long nrow = static_cast<long long>(ntile) * kTileM + ew * 32 + lane;
            if (nrow < rows_total) ptx::bulk_prefetch_l2(cl.residual + nrow * cl.ld_res + col_base, kUnitN * 4);
          } else if (ew == 0 && lane < kUnitN / kKStep) {
            ptx::bulk_prefetch_l2(cl.res_img + (static_cast<size_t>(ntile) * (kMaxN / kKStep) +
                                                (col_base >> 4) + lane) * GCB_A_IMAGE_BLOCK,
                                  GCB_A_IMAGE_BLOCK);
          }
        }
        const int keep_q = cl.keep_q;
        const int kind = cl.kind;
        if (keep_q >= 0) {
          // previous readers of this slot (tile ti - nslots) are done in both CTAs
          const long long w0 = tracing(u) ? clock64() : 0;
          ptx::mbar_wait(&h_free_bar[keep_q * kChainSlotsMax + (ti % nslots)],
                         (static_cast<uint32_t>(ti / nslots) & 1u) ^ 1u);
          if (ew == 0 && lane == 0 && eg == 0) trace_val(u, 9, clock64() - w0);
          cx.img1 = scratch_slot(keep_q, ti);
        }
        const uint32_t buf = u & 1;
        ptx::mbar_wait(&tmem_full_bar[buf], (u >> 1) & 1);
        ptx::tc_fence_after_sync();
        if (ew == 0 && lane == 0 && eg == 0) trace(u, 3);
        const uint32_t taddr = tmem_base + lane_base + buf * kUnitN;
        if (kind >= kKindLN) {
          const uint32_t lb = ln_count & 1, par = (ln_count >> 1) & 1;
          LnStats st;
          unit_stats(cx.s_bias, taddr, st);
          const float mean_h = st.shift + st.mean;
          const float m2_h = st.m2;
          const int myrow = ew * 32 + lane;
          // (with two epilogue groups both compute the statistics of all 256 columns and run
          // their own exchange with the same group of the partner CTA: no coupling between groups)
          ptx::st_async_f32x2(ptx::mapa(ptx::smem_addr(&my_lnx[lb * kTileM + myrow]), peer), mean_h, m2_h,
                              ptx::mapa(ptx::smem_addr(&my_lnx_bar[lb]), peer));
          if (ew == 0 && lane == 0) ptx::mbar_arrive_expect_tx(&my_lnx_bar[lb], kTileM * 8);
          ptx::mbar_wait(&my_lnx_bar[lb], par);
          const float2 other = my_lnx[lb * kTileM + myrow];
          const float delta = other.x - mean_h;
          const float mean = 0.5f * (mean_h + other.x);
          const float var = (m2_h + other.y + delta * delta * (0.5f * kUnitN)) * (1.0f / (2 * kUnitN));
          const float rstd = rsqrtf(var + 1e-5f);
          if (ew == 0 && lane == 0 && eg == 0) trace(u, 4);
          if (kind == kKindLNRes)
            g_count = finish_unit(std::integral_constant<int, kKindLNRes>{}, cx, g_count, taddr, row0, mean, rstd);
          else if (kind == kKindLNImg)
            g_count = finish_unit(std::integral_constant<int, kKindLNImg>{}, cx, g_count, taddr, row0, mean, rstd);
          else
            g_count = finish_unit(std::integral_constant<int, kKindLN>{}, cx, g_count, taddr, row0, mean, rstd);
          ++ln_count;
        } else if (kind == kKindSwish) {
          g_count = finish_unit(std::integral_constant<int, kKindSwish>{}, cx, g_count, taddr, row0, 0.f, 1.f);
        } else {
          g_count = finish_unit(std::integral_constant<int, kKindPlain>{}, cx, g_count, taddr, row0, 0.f, 1.f);
        }
        if (ew == 0 && lane == 0 && eg == 0) trace(u, 5);
        // accumulator free for the MMA warp
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar[buf]);
        if (keep_q >= 0) {
          // Hand the slot to the TMA warps of both CTAs: my generic-proxy global stores must be
          // visible to their async-proxy bulk copies.
          ptx::fence_proxy_async_global();
          __syncwarp();
          if (lane == 0) {
            uint64_t* hb = &h_full_bar[keep_q * kChainSlotsMax + (ti % nslots)];
            ptx::mbar_arrive_release_cluster(hb);
            ptx::mbar_arrive_remote(ptx::mapa(ptx::smem_addr(hb), peer));
          }
        }
        if (ew == 0 && lane == 0 && eg == 0) trace(u, 10);
        ++u;
      }
    }
  } else {
    // ===== gather warps: pre-activation addends of the split edge MLP =====
    ptx::setmaxnreg_dec<kRegsProd>();
    const int first_warp = 4 + 4 * kEpiGroups;
    const int group = (warp - first_warp) >> 2;        // 0 (.. 1 with a single epilogue group)
    const int tid_g = threadIdx.x - 32 * first_warp - group * 128;
    if (kPre) {
      // Thread (rp, cgp): rows rp + 16*p (p < 8), 16-byte column group cgp of each 32-column
      // chunk: 8 lanes read one 128-byte line segment of a gathered row.  Chunk c goes to staging
      // buffer c & 1; with two gather groups group g fills the chunks of its parity.
      const int cgp = tid_g & 7, rp = tid_g >> 3;
      uint32_t gc = 0;
      const int gcol_lo = static_cast<int>(crank) * kUnitN, gcol_hi = gcol_lo + kUnitN;
      for (int st = 0; st < nsteps; ++st) {
        for (int li = 0; li < L; ++li) {
          const int l = desc ? L - 1 - li : li;
          const int ti = st - l * lag;
          if (ti < 0 || ti >= T) continue;
          const int n_pre = s_layer[l].n_pre;
          if (n_pre == 0 || s_layer[l].kind >= kKindLN) continue;
          const uint32_t tile = cid + static_cast<uint32_t>(ti) * ncl;
          const long long trow0 = static_cast<long long>(tile) * kTileM;
          const float* p0[8];
          const float* p1[8];
#pragma unroll
          for (int p = 0; p < 8; ++p) {
            const long long grow = trow0 + rp + 16 * p;
            p0[p] = nullptr; p1[p] = nullptr;
            if (grow < rows_total) {
              const PreAddInfo a = s_pre[l * 2];
              p0[p] = a.table + (a.idx ? static_cast<long long>(__ldg(a.idx + grow)) : grow) * a.ld + cgp * 4;
              if (n_pre > 1) {
                const PreAddInfo b = s_pre[l * 2 + 1];
                p1[p] = b.table + (b.idx ? static_cast<long long>(__ldg(b.idx + grow)) : grow) * b.ld + cgp * 4;
              }
            }
          }
          for (int c0 = gcol_lo; c0 < gcol_hi; c0 += 32, ++gc) {
            const uint32_t gb = gc & 1;
            if (kGatherGroups == 2 && gb != static_cast<uint32_t>(group)) continue;
            float4 acc[8];
#pragma unroll
            for (int p = 0; p < 8; ++p)
              acc[p] = p0[p] ? __ldg(reinterpret_cast<const float4*>(p0[p] + c0)) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (n_pre > 1) {
#pragma unroll
              for (int p = 0; p < 8; ++p) {
                if (p1[p]) {
                  const float4 t = __ldg(reinterpret_cast<const float4*>(p1[p] + c0));
                  acc[p].x += t.x; acc[p].y += t.y; acc[p].z += t.z; acc[p].w += t.w;
                }
              }
            }
            ptx::mbar_wait(&g_empty_bar[gb], ((gc >> 1) & 1) ^ 1);
            float* gdst = s_g + gb * kGBufFloats + rp * kEpiRowFloats + cgp * 4;
#pragma unroll
            for (int p = 0; p < 8; ++p)
              *reinterpret_cast<float4*>(gdst + 16 * p * kEpiRowFloats) = acc[p];
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&g_full_bar[gb]);
          }
        }
      }
    }
  }

  // ---- teardown ---------------------------------------------------------------
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::cluster_sync_all();
  if (warp == 2) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace gcb
