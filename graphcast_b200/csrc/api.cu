// C ABI of graphcast_b200 (see include/graphcast_b200.h): argument checking,
// kernel launches and the orchestration of one GraphCast step.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/graphcast_b200.h"
#include "aux_kernels.cuh"
#include "mlp_simt.cuh"
#include "mlp_tc.cuh"
#include "mlp_chain.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define GCB_CHECK_ARG(cond, msg) \
  do {                           \
    if (!(cond)) return fail(GCB_ERR_INVALID, std::string("invalid argument: ") + (msg)); \
  } while (0)

#define GCB_CUDA(expr)                                                              \
  do {                                                                              \
    cudaError_t e_ = (expr);                                                        \
    if (e_ != cudaSuccess)                                                          \
      return fail(GCB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_)); \
  } while (0)

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

uint16_t f32_to_bf16_rne(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<uint16_t>((u >> 16) | 0x40);  // NaN
  const uint32_t lsb = (u >> 16) & 1u;
  u += 0x7fffu + lsb;
  return static_cast<uint16_t>(u >> 16);
}
float bf16_to_f32(uint16_t h) {
  uint32_t u = static_cast<uint32_t>(h) << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

int sm_count_cached() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// ---- optional per-launch profiling (CUDA events on the launching stream) ----------
struct ProfRec {
  cudaEvent_t beg, end;
  int kind;
  double flops, bytes;
};
bool g_prof_on = false;
std::vector<ProfRec> g_prof;
std::vector<cudaEvent_t> g_event_pool;

cudaEvent_t pool_event() {
  if (!g_event_pool.empty()) {
    cudaEvent_t e = g_event_pool.back();
    g_event_pool.pop_back();
    return e;
  }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}

struct ProfScope {
  bool on;
  cudaStream_t st;
  ProfRec rec;
  ProfScope(cudaStream_t s, int kind, double flops, double bytes) : on(g_prof_on), st(s) {
    if (!on) return;
    rec.kind = kind; rec.flops = flops; rec.bytes = bytes;
    rec.beg = pool_event(); rec.end = pool_event();
    cudaEventRecord(rec.beg, st);
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(rec.end, st);
    g_prof.push_back(rec);
  }
};

int validate_layer(const gcb_layer_desc* d) {
  GCB_CHECK_ARG(d != nullptr, "null descriptor");
  GCB_CHECK_ARG(d->rows >= 0, "rows < 0");
  GCB_CHECK_ARG(d->n == 256 || d->n == 512, "n must be 256 or 512");
  GCB_CHECK_ARG(d->n_valid > 0 && d->n_valid <= d->n, "n_valid out of range");
  GCB_CHECK_ARG(d->nseg >= 1 && d->nseg <= 3, "nseg must be 1..3");
  if (d->out_img != nullptr)
    GCB_CHECK_ARG(aligned16(d->out_img) && d->n == 512 && d->n_valid == 512,
                  "out_img requires n = n_valid = 512");
  int ksteps = 0;
  for (int s = 0; s < d->nseg; ++s) {
    const gcb_segment& g = d->seg[s];
    GCB_CHECK_ARG(g.k > 0 && g.k % 16 == 0, "segment k must be a positive multiple of 16");
    ksteps += g.k / 16;
    if (g.img != nullptr) {
      GCB_CHECK_ARG(aligned16(g.img), "segment image unaligned");
      continue;
    }
    GCB_CHECK_ARG(g.table != nullptr && aligned16(g.table), "segment table null/unaligned");
    GCB_CHECK_ARG(g.k_valid > 0 && g.k_valid <= g.k && g.k_valid % 4 == 0,
                  "segment k_valid must be a multiple of 4 and <= k");
    GCB_CHECK_ARG(g.ld % 4 == 0 && g.ld >= g.k_valid, "segment ld must be a multiple of 4 and >= k_valid");
    GCB_CHECK_ARG(g.fan >= 1, "segment fan must be >= 1");
  }
  GCB_CHECK_ARG(ksteps <= gcb::kMaxKSteps, "K too large");
  GCB_CHECK_ARG(d->bias != nullptr, "bias is null");
  GCB_CHECK_ARG((d->ln_scale == nullptr) == (d->ln_offset == nullptr), "ln_scale/ln_offset mismatch");
  GCB_CHECK_ARG(d->out != nullptr || d->out_y != nullptr || d->out_img != nullptr, "no output");
  if (d->out) GCB_CHECK_ARG(aligned16(d->out) && d->ld_out % 4 == 0 && d->ld_out >= d->n_valid, "out unaligned");
  if (d->out_y) GCB_CHECK_ARG(aligned16(d->out_y) && d->ld_out_y % 4 == 0 && d->ld_out_y >= d->n_valid, "out_y unaligned");
  if (d->residual) GCB_CHECK_ARG(aligned16(d->residual) && d->ld_res % 4 == 0, "residual unaligned");
  GCB_CHECK_ARG(d->act == GCB_ACT_NONE || d->act == GCB_ACT_SWISH, "unknown activation");
  GCB_CHECK_ARG(!(d->act == GCB_ACT_SWISH && d->ln_scale != nullptr),
                "a layer is swish OR LayerNorm, not both");
  GCB_CHECK_ARG(d->n_pre_add >= 0 && d->n_pre_add <= 2, "n_pre_add must be 0..2");
  if (d->n_pre_add > 0) {
    GCB_CHECK_ARG(d->ln_scale == nullptr, "pre_add cannot be combined with LayerNorm");
    GCB_CHECK_ARG(d->n_valid == d->n, "pre_add requires n_valid == n");
    for (int i = 0; i < d->n_pre_add; ++i)
      GCB_CHECK_ARG(d->pre_add[i].table != nullptr && aligned16(d->pre_add[i].table) &&
                        d->pre_add[i].ld % 4 == 0 && d->pre_add[i].ld >= d->n,
                    "pre_add table null/unaligned");
  }
  if (d->precision == GCB_PREC_FP32_SIMT) {
    GCB_CHECK_ARG(d->w_f32 != nullptr, "w_f32 is null (FP32_SIMT)");
  } else {
    GCB_CHECK_ARG(d->precision == GCB_PREC_BF16X3 || d->precision == GCB_PREC_BF16, "unknown precision");
    GCB_CHECK_ARG(d->w_packed != nullptr && aligned16(d->w_packed), "w_packed null/unaligned");
  }
  return GCB_OK;
}

int g_cluster_size = 2;   // CTAs per cluster sharing the weight stream (1, 2 or 4)

template <bool kSplit, bool kSwish, bool kLN>
int launch_tc_variant(const gcb_layer_desc& d, cudaStream_t stream) {
  using Cfg = gcb::TcConfig<kSplit, kLN>;
  auto kernel = gcb::mlp_layer_tc_kernel<kSplit, kSwish, kLN>;
  static bool attr_set[64] = {false};
  static int max_clusters[64][5] = {{0}};
  int dev = 0;
  GCB_CUDA(cudaGetDevice(&dev));
  GCB_CHECK_ARG(dev >= 0 && dev < 64, "device index out of range");
  if (!attr_set[dev]) {
    GCB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  Cfg::kSmemBytes));
    attr_set[dev] = true;
  }
  const int csize = g_cluster_size;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.blockDim = dim3(gcb::kThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = csize;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (max_clusters[dev][csize] == 0) {
    cfg.gridDim = dim3(sm_count_cached() / csize * csize);
    int nc = 0;
    GCB_CUDA(cudaOccupancyMaxActiveClusters(&nc, kernel, &cfg));
    if (nc <= 0) return fail(GCB_ERR_CUDA, "no resident cluster fits on this device");
    max_clusters[dev][csize] = nc;
  }
  const int tiles = (d.rows + gcb::kTileM - 1) / gcb::kTileM;
  // N-split schedule (n = n_valid = 512, cluster of 2): one tile per cluster at a time;
  // otherwise every CTA of the cluster has its own tile.  Same rule as in the kernel.
  const bool nsplit = (csize == 2 && d.n == 512 && d.n_valid == 512);
  int clusters = nsplit ? tiles : (tiles + csize - 1) / csize;
  if (clusters > max_clusters[dev][csize]) clusters = max_clusters[dev][csize];
  cfg.gridDim = dim3(clusters * csize);
  GCB_CUDA(cudaLaunchKernelEx(&cfg, kernel, d));
  return GCB_OK;
}

template <bool kSplit>
int launch_tc(const gcb_layer_desc& d, cudaStream_t stream) {
  const bool swish = d.act == GCB_ACT_SWISH, ln = d.ln_scale != nullptr;
  if (swish) return launch_tc_variant<kSplit, true, false>(d, stream);
  if (ln) return launch_tc_variant<kSplit, false, true>(d, stream);
  return launch_tc_variant<kSplit, false, false>(d, stream);
}

int launch_simt(const gcb_layer_desc& d, cudaStream_t stream) {
  const size_t smem = (static_cast<size_t>(gcb::kSimtRows) * d.n + gcb::kSimtRows * 17 +
                       static_cast<size_t>(gcb::kSimtK) * d.n) * sizeof(float);
  static bool attr_set[64] = {false};
  int dev = 0;
  GCB_CUDA(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && !attr_set[dev]) {
    GCB_CUDA(cudaFuncSetAttribute(gcb::mlp_layer_simt_kernel,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
    attr_set[dev] = true;
  }
  const int grid = (d.rows + gcb::kSimtRows - 1) / gcb::kSimtRows;
  gcb::mlp_layer_simt_kernel<<<grid, gcb::kSimtThreads, smem, stream>>>(d);
  GCB_CUDA(cudaGetLastError());
  return GCB_OK;
}

// ---- fused layer chains (mlp_chain.cuh) -----------------------------------------------
struct ChainShape {
  int nq = 0;          // kept layers (scratch rings)
  int maxdist = 1;     // largest (consumer layer - producer layer)
  int nslots = 2;
  bool pre = false;
  bool big = false;    // more than 4 parameter vectors
};

int validate_chain(const gcb_chain_desc* d, ChainShape* shape) {
  GCB_CHECK_ARG(d != nullptr, "null descriptor");
  GCB_CHECK_ARG(d->rows >= 0, "rows < 0");
  GCB_CHECK_ARG(d->nlayers >= 1 && d->nlayers <= GCB_MAX_CHAIN, "nlayers must be 1..GCB_MAX_CHAIN");
  GCB_CHECK_ARG(d->precision == GCB_PREC_BF16X3 || d->precision == GCB_PREC_BF16,
                "chains run on the tensor-core path only (BF16X3 / BF16)");
  GCB_CHECK_ARG(d->lag >= 0 && d->lag <= 2, "lag must be 0 (default), 1 or 2");
  ChainShape sh;
  int vecs = 0;
  for (int l = 0; l < d->nlayers; ++l) {
    const gcb_chain_layer& g = d->layer[l];
    GCB_CHECK_ARG(g.nseg >= 1 && g.nseg <= 3, "nseg must be 1..3");
    for (int s = 0; s < g.nseg; ++s) {
      const int from = g.seg_from[s];
      if (from >= 0) {
        GCB_CHECK_ARG(from < l && d->layer[from].keep, "seg_from must name an earlier layer with keep = 1");
        if (l - from > sh.maxdist) sh.maxdist = l - from;
        continue;
      }
      const gcb_segment& sg = g.seg[s];
      GCB_CHECK_ARG(sg.k > 0 && sg.k % 16 == 0, "segment k must be a positive multiple of 16");
      if (sg.img != nullptr) {
        GCB_CHECK_ARG(aligned16(sg.img), "segment image unaligned");
        continue;
      }
      GCB_CHECK_ARG(sg.table != nullptr && aligned16(sg.table), "segment table null/unaligned");
      GCB_CHECK_ARG(sg.k_valid > 0 && sg.k_valid <= sg.k && sg.k_valid % 4 == 0,
                    "segment k_valid must be a multiple of 4 and <= k");
      GCB_CHECK_ARG(sg.ld % 4 == 0 && sg.ld >= sg.k_valid, "segment ld must be a multiple of 4 and >= k_valid");
      GCB_CHECK_ARG(sg.fan >= 1, "segment fan must be >= 1");
    }
    GCB_CHECK_ARG(g.w_packed != nullptr && aligned16(g.w_packed), "w_packed null/unaligned");
    GCB_CHECK_ARG((g.ln_scale == nullptr) == (g.ln_offset == nullptr), "ln_scale/ln_offset mismatch");
    GCB_CHECK_ARG(g.act == GCB_ACT_NONE || g.act == GCB_ACT_SWISH, "unknown activation");
    GCB_CHECK_ARG(!(g.act == GCB_ACT_SWISH && g.ln_scale != nullptr),
                  "a chain layer is swish OR LayerNorm, not both");
    GCB_CHECK_ARG(g.out || g.out_y || g.out_img || g.keep, "layer has no output");
    if (g.act == GCB_ACT_SWISH)
      GCB_CHECK_ARG(!g.out && !g.out_y && !g.residual,
                    "a swish chain layer delivers operand images only (out_img / keep)");
    if (g.ln_scale == nullptr)
      GCB_CHECK_ARG(!g.residual && !g.residual_img, "residual needs a LayerNorm layer in a chain");
    if (g.residual_img)
      GCB_CHECK_ARG(aligned16(g.residual_img) && !g.residual && !g.out,
                    "residual_img excludes residual and out");
    if (g.residual_keep != 0) {
      const int from = g.residual_keep - 1;
      GCB_CHECK_ARG(from >= 0 && from < l && d->layer[from].keep && g.ln_scale != nullptr &&
                        !g.residual && !g.residual_img && !g.out,
                    "residual_keep must name an earlier kept layer (LayerNorm layers; excludes residual*/out)");
      if (l - from > sh.maxdist) sh.maxdist = l - from;
    }
    if (g.out) GCB_CHECK_ARG(aligned16(g.out) && g.ld_out % 4 == 0 && g.ld_out >= 512, "out unaligned");
    if (g.out_y) GCB_CHECK_ARG(aligned16(g.out_y) && g.ld_out_y % 4 == 0 && g.ld_out_y >= 512, "out_y unaligned");
    if (g.out_img) GCB_CHECK_ARG(aligned16(g.out_img), "out_img unaligned");
    if (g.residual) GCB_CHECK_ARG(aligned16(g.residual) && g.ld_res % 4 == 0 && g.ld_res >= 512, "residual unaligned");
    GCB_CHECK_ARG(g.n_pre_add >= 0 && g.n_pre_add <= 2, "n_pre_add must be 0..2");
    if (g.n_pre_add > 0) {
      GCB_CHECK_ARG(g.ln_scale == nullptr, "pre_add cannot be combined with LayerNorm");
      for (int i = 0; i < g.n_pre_add; ++i)
        GCB_CHECK_ARG(g.pre_add[i].table != nullptr && aligned16(g.pre_add[i].table) &&
                          g.pre_add[i].ld % 4 == 0 && g.pre_add[i].ld >= 512,
                      "pre_add table null/unaligned");
      sh.pre = true;
    }
    vecs += (g.bias ? 1 : 0) + (g.ln_scale ? 2 : 0);
    if (g.keep) ++sh.nq;
  }
  GCB_CHECK_ARG(vecs <= 8, "too many bias / LayerNorm vectors for one chain (at most 8)");
  sh.big = vecs > 4;
  const int lag = d->lag > 0 ? d->lag : 1;
  GCB_CHECK_ARG(d->order == 0 || (d->order == 1 && d->nlayers >= 3),
                "order must be 0, or 1 for chains of at least 3 layers");
  sh.nslots = lag * sh.maxdist + (d->order == 0 ? 1 : 0);
  GCB_CHECK_ARG(sh.nslots <= gcb::kChainSlotsMax, "lag x distance too large");
  if (sh.nq > 0) {
    GCB_CHECK_ARG(d->scratch != nullptr && aligned16(d->scratch), "scratch null/unaligned");
    const long long need = static_cast<long long>(sm_count_cached() / 2) * sh.nq * sh.nslots *
                           gcb::kScratchTileBytes;
    GCB_CHECK_ARG(d->scratch_bytes >= need, "scratch too small for this chain (kept layers x slots)");
  }
  *shape = sh;
  return GCB_OK;
}

template <bool kSplit, bool kPre, bool kBig>
int launch_chain_variant(const gcb_chain_desc& d, const ChainShape& sh, cudaStream_t stream) {
  using Cfg = gcb::ChainConfig<kSplit, kPre, kBig>;
  auto kernel = gcb::mlp_chain_tc_kernel<kSplit, kPre, kBig>;
  static bool attr_set[64] = {false};
  static int max_clusters[64] = {0};
  int dev = 0;
  GCB_CUDA(cudaGetDevice(&dev));
  GCB_CHECK_ARG(dev >= 0 && dev < 64, "device index out of range");
  if (!attr_set[dev]) {
    GCB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_set[dev] = true;
    // The scratch ring is accessed with the L2 evict_last policy.  Experiment switch: with
    // GCB_L2_PERSIST_MB > 0 those lines also get a persisting set-aside of that size (at most 79 MB
    // on B200).  Measured at 0.25 degree: DRAM traffic per step 183 -> 147 GB with the full
    // set-aside, but the step gets SLOWER (75.3 -> 80.2 ms; the gathers lose the L2 they lived in),
    // so the default is no set-aside (profiles/r02_l2_persist_experiment.log).
    static bool l2_set[64] = {false};
    if (!l2_set[dev]) {
      l2_set[dev] = true;
      int max_persist = 0;
      cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev);
      long long want = 0;
      if (const char* e = getenv("GCB_L2_PERSIST_MB")) want = atoll(e) * (1ll << 20);
      if (want > max_persist) want = max_persist;
      if (want > 0 && cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, static_cast<size_t>(want)) != cudaSuccess)
        cudaGetLastError();
    }
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.blockDim = dim3(gcb::kThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (max_clusters[dev] == 0) {
    cfg.gridDim = dim3(sm_count_cached() / 2 * 2);
    int nc = 0;
    GCB_CUDA(cudaOccupancyMaxActiveClusters(&nc, kernel, &cfg));
    if (nc <= 0) return fail(GCB_ERR_CUDA, "no resident cluster fits on this device");
    if (nc > sm_count_cached() / 2) nc = sm_count_cached() / 2;   // the scratch is sized for SMs / 2
    max_clusters[dev] = nc;
  }
  const int tiles = (d.rows + gcb::kTileM - 1) / gcb::kTileM;
  int clusters = tiles < max_clusters[dev] ? tiles : max_clusters[dev];
  cfg.gridDim = dim3(clusters * 2);
  GCB_CUDA(cudaLaunchKernelEx(&cfg, kernel, d, sh.nq, sh.nslots));
  return GCB_OK;
}

struct StepCtx {
  const gcb_model* m;
  cudaStream_t stream;
  int launches;
};

gcb_segment seg(const float* table, const int32_t* idx, int ld, int k, int k_valid, int fan = 1) {
  gcb_segment s;
  memset(&s, 0, sizeof(s));
  s.table = table; s.idx = idx; s.ld = ld; s.k = k; s.k_valid = k_valid; s.fan = fan;
  return s;
}

gcb_segment seg_img(const void* img, int k) {
  gcb_segment s;
  memset(&s, 0, sizeof(s));
  s.img = img; s.k = k; s.k_valid = k; s.fan = 1;
  return s;
}

struct MlpOut {
  const void* residual_img = nullptr;   // residual as an operand image (fused path only)
  const float* residual = nullptr;   // fp32 [rows,512], added to the result
  float* out = nullptr;              // residual + y (fp32)
  int ld_out = 512;
  float* out_y = nullptr;            // y alone (fp32)
  void* out_img = nullptr;           // residual + y as an operand image
};

// Two-layer MLP: hidden = swish(concat(segs) @ W0 + b0 [+ gathered addends]);
// y = [LN](hidden @ W1 + b1), delivered as MlpOut says.  Fused (gcb_model.fuse, tensor-core
// precisions, n1 = 512): ONE chain launch, the hidden activation stays in the L2-resident
// scratch.  Otherwise two launches with the hidden activation as an operand image in HBM.
int run_mlp(StepCtx& c, const gcb_mlp& w, int rows, int nseg, const gcb_segment* segs,
            const MlpOut& o, const void* w0_packed_override = nullptr,
            const float* w0_f32_override = nullptr, int n_pre = 0, const gcb_pre_add* pre = nullptr) {
  if (rows == 0) return GCB_OK;
  int k0 = 0;
  for (int s = 0; s < nseg; ++s) k0 += segs[s].k;
  if (w0_packed_override == nullptr && k0 != w.k0)
    return fail(GCB_ERR_INVALID, "run_mlp: segment widths do not match the weight");
  if (c.m->fuse && c.m->precision != GCB_PREC_FP32_SIMT && w.n1 == 512 && w.n1_valid == 512 &&
      o.ld_out == 512) {
    gcb_chain_desc ch;
    memset(&ch, 0, sizeof(ch));
    ch.rows = rows; ch.nlayers = 2; ch.precision = c.m->precision; ch.lag = c.m->chain_lag;
    ch.scratch = c.m->chain_scratch; ch.scratch_bytes = c.m->chain_scratch_bytes;
    gcb_chain_layer& a = ch.layer[0];
    a.nseg = nseg;
    for (int s = 0; s < nseg; ++s) { a.seg[s] = segs[s]; a.seg_from[s] = -1; }
    a.w_packed = w0_packed_override ? w0_packed_override : w.w0_packed;
    a.bias = w.b0; a.act = GCB_ACT_SWISH; a.keep = 1;
    a.n_pre_add = n_pre;
    for (int i = 0; i < n_pre; ++i) a.pre_add[i] = pre[i];
    gcb_chain_layer& b = ch.layer[1];
    b.nseg = 1; b.seg_from[0] = 0; b.seg[0].k = 512; b.seg_from[1] = b.seg_from[2] = -1;
    b.w_packed = w.w1_packed; b.bias = w.b1; b.ln_scale = w.ln_scale; b.ln_offset = w.ln_offset;
    b.act = GCB_ACT_NONE;
    b.residual = o.residual; b.ld_res = 512; b.residual_img = o.residual_img;
    b.out = o.out; b.ld_out = 512; b.out_y = o.out_y; b.ld_out_y = 512; b.out_img = o.out_img;
    int rc = gcb_chain_forward(&ch, c.stream);
    if (rc) return rc;
    c.launches += 1;
    return GCB_OK;
  }
  if (o.residual_img != nullptr)
    return fail(GCB_ERR_INVALID, "run_mlp: an image residual needs the fused path");
  gcb_layer_desc l0;
  memset(&l0, 0, sizeof(l0));
  l0.rows = rows; l0.n = 512; l0.n_valid = 512; l0.nseg = nseg;
  for (int s = 0; s < nseg; ++s) l0.seg[s] = segs[s];
  l0.w_packed = w0_packed_override ? w0_packed_override : w.w0_packed;
  l0.w_f32 = w0_packed_override ? w0_f32_override : w.w0_f32;
  l0.bias = w.b0;
  l0.n_pre_add = n_pre;
  for (int i = 0; i < n_pre; ++i) l0.pre_add[i] = pre[i];
  l0.act = GCB_ACT_SWISH;
  l0.out_img = c.m->hidden;          // hidden activations go straight to operand-image form
  l0.precision = c.m->precision;
  int rc = gcb_layer_forward(&l0, c.stream);
  if (rc) return rc;
  gcb_layer_desc l1;
  memset(&l1, 0, sizeof(l1));
  l1.rows = rows; l1.n = w.n1; l1.n_valid = w.n1_valid; l1.nseg = 1;
  l1.seg[0] = seg_img(c.m->hidden, 512);
  l1.w_packed = w.w1_packed; l1.w_f32 = w.w1_f32; l1.bias = w.b1;
  l1.ln_scale = w.ln_scale; l1.ln_offset = w.ln_offset;
  l1.act = GCB_ACT_NONE;
  l1.residual = o.residual; l1.ld_res = 512;
  l1.out = o.out; l1.ld_out = o.ld_out;
  l1.out_y = o.out_y; l1.ld_out_y = 512;
  l1.out_img = o.out_img;
  l1.precision = c.m->precision;
  rc = gcb_layer_forward(&l1, c.stream);
  if (rc) return rc;
  c.launches += 2;
  return GCB_OK;
}

// Node-level projection P = v @ W (no bias, no activation), v given as an operand image.
int run_projection(StepCtx& c, const void* w_packed, const float* w_f32, const void* v_img,
                   int rows, float* out) {
  if (rows == 0) return GCB_OK;
  gcb_layer_desc l;
  memset(&l, 0, sizeof(l));
  l.rows = rows; l.n = 512; l.n_valid = 512; l.nseg = 1;
  l.seg[0] = seg_img(v_img, 512);
  l.w_packed = w_packed; l.w_f32 = w_f32; l.bias = c.m->zero_bias;
  l.act = GCB_ACT_NONE;
  l.out = out; l.ld_out = 512;
  l.precision = c.m->precision;
  int rc = gcb_layer_forward(&l, c.stream);
  if (rc) return rc;
  c.launches += 1;
  return GCB_OK;
}

// Edge MLP  LN.MLP([e | vs[snd] | vr[rcv]]).  With pregather the first layer is evaluated as
// e @ W_e + (vs @ W_s)[snd] + (vr @ W_r)[rcv]: two node-level projections, then an edge layer
// with K = 512 whose epilogue adds the gathered projections before the activation.
int run_edge_mlp(StepCtx& c, const gcb_mlp& w, const gcb_mlp_split* split, int rows,
                 const void* e_img,
                 const float* vs, const void* vs_img, int n_s, const int32_t* snd, float* proj_s,
                 const float* vr, const void* vr_img, int n_r, const int32_t* rcv, float* proj_r,
                 const MlpOut& o) {
  const int D = 512;
  gcb_segment s[3];
  s[0] = seg_img(e_img, D);
  if (!c.m->pregather) {
    s[1] = seg(vs, snd, D, D, D);
    s[2] = seg(vr, rcv, D, D, D);
    return run_mlp(c, w, rows, 3, s, o);
  }
  int rc;
  if ((rc = run_projection(c, split->ws_packed, split->ws_f32, vs_img, n_s, proj_s))) return rc;
  if ((rc = run_projection(c, split->wr_packed, split->wr_f32, vr_img, n_r, proj_r))) return rc;
  gcb_pre_add pre[2];
  pre[0].table = proj_s; pre[0].idx = snd; pre[0].ld = D; pre[0].pad_ = 0;
  pre[1].table = proj_r; pre[1].idx = rcv; pre[1].ld = D; pre[1].pad_ = 0;
  return run_mlp(c, w, rows, 1, s, o, split->we_packed, split->we_f32, 2, pre);
}

int to_image(StepCtx& c, const float* src, int ld, int fan, long long rows, int k, void* img) {
  int rc = gcb_rows_to_image(src, ld, fan, rows, k, img, c.stream);
  if (rc) return rc;
  c.launches += 1;
  return GCB_OK;
}

}  // namespace

extern "C" {

int gcb_abi_version(void) { return GCB_ABI_VERSION; }

const char* gcb_last_error(void) { return g_err.c_str(); }

int gcb_sm_count(int device) {
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return -1;
  return n;
}

int64_t gcb_a_image_bytes(int64_t rows, int32_t k) {
  if (rows < 0 || k <= 0 || k % 16 != 0) return -1;
  const int64_t tiles = (rows + gcb::kTileM - 1) / gcb::kTileM;
  return tiles * (k / 16) * GCB_A_IMAGE_BLOCK;
}

int64_t gcb_packed_weight_bytes(int32_t k, int32_t n) {
  if (k <= 0 || n <= 0 || k % 16 != 0) return -1;
  return static_cast<int64_t>(k) * n * 4;   // bf16 hi + bf16 lo per element
}

int gcb_pack_weight_host(const float* w, int32_t k_rows, int32_t n_cols, int32_t k, int32_t n,
                         void* dst) {
  GCB_CHECK_ARG(w != nullptr && dst != nullptr, "null pointer");
  GCB_CHECK_ARG(k > 0 && k % 16 == 0 && n > 0 && n % 256 == 0, "k must be a multiple of 16, n of 256");
  GCB_CHECK_ARG(k_rows <= k && n_cols <= n && k_rows >= 0 && n_cols >= 0, "real shape exceeds padded shape");
  // Image order: [K-step][256-column block h][hi | lo][K chunk c][256 rows][8 elements]:
  // one contiguous 16 KB block per (K-step, h) = the B tile of one unit's K-step.
  GCB_CHECK_ARG(n % 256 == 0, "n must be a multiple of 256");
  uint16_t* img = static_cast<uint16_t*>(dst);
  const int ksteps = k / 16, halves = n / 256;
  for (int ks = 0; ks < ksteps; ++ks)
    for (int h = 0; h < halves; ++h) {
      uint16_t* hi = img + (static_cast<size_t>(ks) * halves + h) * 8192;   // 16 KB per block
      uint16_t* lo = hi + 4096;
      for (int c = 0; c < 2; ++c)
        for (int r = 0; r < 256; ++r)
          for (int j = 0; j < 8; ++j) {
            const int kk = ks * 16 + c * 8 + j, nn = h * 256 + r;
            const float v = (kk < k_rows && nn < n_cols) ? w[static_cast<size_t>(kk) * n_cols + nn] : 0.f;
            const uint16_t hv = f32_to_bf16_rne(v);
            const uint16_t lv = f32_to_bf16_rne(v - bf16_to_f32(hv));
            const size_t off = (static_cast<size_t>(c) * 256 + r) * 8 + j;
            hi[off] = hv;
            lo[off] = lv;
          }
    }
  return GCB_OK;
}

int gcb_layer_forward(const gcb_layer_desc* d, void* stream) {
  int rc = validate_layer(d);
  if (rc) return rc;
  if (d->rows == 0) return GCB_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  double kv = 0, a_elems = 0;
  for (int i = 0; i < d->nseg; ++i) {
    const double w = d->seg[i].img ? d->seg[i].k : d->seg[i].k_valid;
    kv += w;
    a_elems += w * (d->seg[i].img ? 1 : d->seg[i].fan);
  }
  const double rows = d->rows;
  a_elems += static_cast<double>(d->n_pre_add) * d->n_valid;
  const double flops = 2.0 * rows * kv * d->n_valid;
  const double bytes = 4.0 * (rows * a_elems + kv * d->n_valid +
                              rows * d->n_valid * ((d->out ? 1 : 0) + (d->out_y ? 1 : 0) +
                                                   (d->residual ? 1 : 0) + (d->out_img ? 1 : 0)));
  ProfScope prof(st, d->precision == GCB_PREC_FP32_SIMT ? GCB_KIND_LAYER_SIMT : GCB_KIND_LAYER_TC,
                 flops, bytes);
  switch (d->precision) {
    case GCB_PREC_BF16X3: return launch_tc<true>(*d, st);
    case GCB_PREC_BF16: return launch_tc<false>(*d, st);
    default: return launch_simt(*d, st);
  }
}

int64_t gcb_chain_scratch_bytes(int32_t device, int32_t n_keep_layers, int32_t lag,
                                int32_t max_distance) {
  if (n_keep_layers < 0 || n_keep_layers > GCB_MAX_CHAIN || lag < 0 || lag > 2 || max_distance < 1)
    return -1;
  int sms = 0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0)
    return -1;
  const int nslots = (lag > 0 ? lag : 1) * max_distance + 1;
  if (nslots > gcb::kChainSlotsMax) return -1;
  return static_cast<int64_t>(sms / 2) * n_keep_layers * nslots * gcb::kScratchTileBytes;
}

int gcb_chain_forward(const gcb_chain_desc* d, void* stream) {
  ChainShape sh;
  int rc = validate_chain(d, &sh);
  if (rc) return rc;
  if (d->rows == 0) return GCB_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // Algorithmic work of the launch: 2*rows*K*n flops per layer; bytes = external A operands
  // (incl. gathers) + gathered addends + weights + residual + outputs; results handed over
  // inside the chain are not HBM traffic.
  double flops = 0, bytes = 0;
  const double rows = d->rows;
  for (int l = 0; l < d->nlayers; ++l) {
    const gcb_chain_layer& g = d->layer[l];
    double kv = 0, a_elems = 0;
    for (int s = 0; s < g.nseg; ++s) {
      if (g.seg_from[s] >= 0) { kv += 512; continue; }
      const double w = g.seg[s].img ? g.seg[s].k : g.seg[s].k_valid;
      kv += w;
      a_elems += w * (g.seg[s].img ? 1 : g.seg[s].fan);
    }
    a_elems += 512.0 * g.n_pre_add;
    flops += 2.0 * rows * kv * 512;
    bytes += 4.0 * (rows * a_elems + kv * 512 +
                    rows * 512 * ((g.out ? 1 : 0) + (g.out_y ? 1 : 0) + (g.residual ? 1 : 0) +
                                  (g.out_img ? 1 : 0)));
    // (a residual_img that is also a segment of the chain is read from HBM once: not counted again)
  }
  ProfScope prof(st, GCB_KIND_CHAIN_TC, flops, bytes);
  const int variant = (d->precision == GCB_PREC_BF16X3 ? 4 : 0) | (sh.pre ? 2 : 0) | (sh.big ? 1 : 0);
  switch (variant) {
    case 7: return launch_chain_variant<true, true, true>(*d, sh, st);
    case 6: return launch_chain_variant<true, true, false>(*d, sh, st);
    case 5: return launch_chain_variant<true, false, true>(*d, sh, st);
    case 4: return launch_chain_variant<true, false, false>(*d, sh, st);
    case 3: return launch_chain_variant<false, true, true>(*d, sh, st);
    case 2: return launch_chain_variant<false, true, false>(*d, sh, st);
    case 1: return launch_chain_variant<false, false, true>(*d, sh, st);
    default: return launch_chain_variant<false, false, false>(*d, sh, st);
  }
}

int gcb_segment_sum(const float* msg, int32_t ld_msg, const int32_t* row_ptr, int32_t num_nodes,
                    float* out, int32_t ld_out, int32_t width, void* stream) {
  return gcb_segment_sum_heavy(msg, ld_msg, row_ptr, num_nodes, nullptr, 0, out, ld_out, width, stream);
}

namespace {
int segment_sum_launch(const float* msg, int32_t ld_msg, const int32_t* row_ptr, int32_t num_nodes,
                       const int32_t* heavy, int32_t num_heavy, float* out, int32_t ld_out,
                       int32_t width, void* img, long long num_edges, void* stream);
}

int gcb_segment_sum_heavy(const float* msg, int32_t ld_msg, const int32_t* row_ptr,
                          int32_t num_nodes, const int32_t* heavy, int32_t num_heavy, float* out,
                          int32_t ld_out, int32_t width, void* stream) {
  return segment_sum_launch(msg, ld_msg, row_ptr, num_nodes, heavy, num_heavy, out, ld_out, width,
                            nullptr, 0, stream);
}

namespace {
// img (optional): operand image of the [num_nodes, 512] result, written by the same kernel.
int segment_sum_launch(const float* msg, int32_t ld_msg, const int32_t* row_ptr, int32_t num_nodes,
                       const int32_t* heavy, int32_t num_heavy, float* out, int32_t ld_out,
                       int32_t width, void* img, long long num_edges, void* stream) {
  GCB_CHECK_ARG(msg && row_ptr && out, "null pointer");
  GCB_CHECK_ARG(num_heavy >= 0 && (num_heavy == 0 || heavy != nullptr), "heavy list is null");
  GCB_CHECK_ARG(width == 512, "segment_sum supports width 512");
  GCB_CHECK_ARG(ld_msg % 4 == 0 && ld_out % 4 == 0 && aligned16(msg) && aligned16(out), "unaligned");
  if (num_nodes == 0) return GCB_OK;
  const int warps_per_block = 8;
  long long blocks = (static_cast<long long>(num_nodes) + warps_per_block - 1) / warps_per_block;
  const long long cap = static_cast<long long>(sm_count_cached()) * 16;
  if (blocks > cap) blocks = cap;
  // algorithmic bytes: every message row read once, every node row written once (+ its image)
  ProfScope prof(static_cast<cudaStream_t>(stream), GCB_KIND_SEGMENT_SUM, 0.0,
                 4.0 * width * (static_cast<double>(num_edges) + num_nodes * (img ? 2.0 : 1.0)));
  gcb::segment_sum_kernel<4><<<static_cast<int>(blocks) + num_heavy, 256, 0,
                              static_cast<cudaStream_t>(stream)>>>(
      msg, ld_msg, row_ptr, num_nodes, out, ld_out, heavy, num_heavy,
      static_cast<unsigned char*>(img));
  GCB_CUDA(cudaGetLastError());
  return GCB_OK;
}
}  // namespace

int gcb_pack_grid_features(const float* planes, int32_t n_ch, int64_t n_nodes, const float* mean,
                           const float* scale, const float* node_static, int32_t n_static,
                           float* feats, int32_t ld, void* stream) {
  GCB_CHECK_ARG(planes && feats, "null pointer");
  GCB_CHECK_ARG(n_ch > 0 && n_static >= 0 && ld >= n_ch + n_static, "ld too small");
  GCB_CHECK_ARG(n_static == 0 || node_static != nullptr, "node_static is null");
  if (n_nodes == 0) return GCB_OK;
  dim3 grid(static_cast<unsigned>((n_nodes + 31) / 32), static_cast<unsigned>((ld + 31) / 32));
  ProfScope prof(static_cast<cudaStream_t>(stream), GCB_KIND_PACK, 0.0,
                 4.0 * n_nodes * (static_cast<double>(n_ch) + n_static + ld));
  gcb::pack_grid_features_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      planes, n_ch, n_nodes, mean, scale, node_static, n_static, feats, ld);
  GCB_CUDA(cudaGetLastError());
  return GCB_OK;
}

int gcb_pack_grid_image(const float* planes, int32_t n_ch, int64_t n_nodes, const float* mean,
                        const float* scale, const float* node_static, int32_t n_static,
                        int32_t k, void* img, void* stream) {
  GCB_CHECK_ARG(planes && img && aligned16(img), "null/unaligned pointer");
  GCB_CHECK_ARG(n_ch > 0 && n_static >= 0 && k % 16 == 0 && k >= n_ch + n_static, "k too small");
  GCB_CHECK_ARG(n_static == 0 || node_static != nullptr, "node_static is null");
  if (n_nodes == 0) return GCB_OK;
  const size_t smem = 32 * static_cast<size_t>(k + 4) * sizeof(float);
  GCB_CHECK_ARG(smem <= 96 * 1024, "k too large");
  static bool attr_set[64] = {false};     // per device: the opt-in is a per-context attribute
  int dev = 0;
  GCB_CUDA(cudaGetDevice(&dev));
  GCB_CHECK_ARG(dev >= 0 && dev < 64, "device index out of range");
  if (!attr_set[dev]) {
    GCB_CUDA(cudaFuncSetAttribute(gcb::pack_grid_image_kernel,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    attr_set[dev] = true;
  }
  const long long padded = (n_nodes + 127) / 128 * 128;
  ProfScope prof(static_cast<cudaStream_t>(stream), GCB_KIND_PACK, 0.0,
                 4.0 * n_nodes * (static_cast<double>(n_ch) + n_static + k));
  gcb::pack_grid_image_kernel<<<static_cast<unsigned>(padded / 32), 256, smem,
                                static_cast<cudaStream_t>(stream)>>>(
      planes, n_ch, n_nodes, mean, scale, node_static, n_static, k, static_cast<unsigned char*>(img));
  GCB_CUDA(cudaGetLastError());
  return GCB_OK;
}

int gcb_unpack_grid_outputs(const float* y, int32_t ld_y, int32_t n_out, int64_t n_nodes,
                            const float* scale, const float* offset, const float* add_planes,
                            const int32_t* add_plane_index, float* planes_out, void* stream) {
  GCB_CHECK_ARG(y && planes_out, "null pointer");
  GCB_CHECK_ARG(n_out > 0 && ld_y >= n_out, "ld_y too small");
  GCB_CHECK_ARG((add_planes == nullptr) == (add_plane_index == nullptr), "add_planes/index mismatch");
  if (n_nodes == 0) return GCB_OK;
  dim3 grid(static_cast<unsigned>((n_nodes + 31) / 32), static_cast<unsigned>((n_out + 31) / 32));
  ProfScope prof(static_cast<cudaStream_t>(stream), GCB_KIND_UNPACK, 0.0,
                 4.0 * n_nodes * n_out * (add_planes ? 3.0 : 2.0));
  gcb::unpack_grid_outputs_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      y, ld_y, n_out, n_nodes, scale, offset, add_planes, add_plane_index, planes_out);
  GCB_CUDA(cudaGetLastError());
  return GCB_OK;
}

int gcb_toa_incident_solar_radiation(const float* table, int32_t n_times, int32_t bins,
                                     const float* sin_lat, const float* cos_lat,
                                     const float* cos_lon, const float* sin_lon, int32_t n_lat,
                                     int32_t n_lon, float* out, void* stream) {
  GCB_CHECK_ARG(table && sin_lat && cos_lat && cos_lon && sin_lon && out, "null pointer");
  GCB_CHECK_ARG(bins >= 1 && bins <= 2048, "bins must be in [1, 2048]");
  GCB_CHECK_ARG(n_times >= 0 && n_times <= 65535 && n_lat >= 0 && n_lat <= 65535 && n_lon >= 0,
                "grid too large");
  if (n_times == 0 || n_lat == 0 || n_lon == 0) return GCB_OK;
  dim3 grid(static_cast<unsigned>((n_lon + 255) / 256), static_cast<unsigned>(n_lat),
            static_cast<unsigned>(n_times));
  ProfScope prof(static_cast<cudaStream_t>(stream), GCB_KIND_PACK, 0.0,
                 4.0 * n_times * static_cast<double>(n_lat) * n_lon);
  gcb::tisr_kernel<<<grid, 256, static_cast<size_t>(bins) * 5 * sizeof(float),
                     static_cast<cudaStream_t>(stream)>>>(
      table, bins, sin_lat, cos_lat, cos_lon, sin_lon, n_lat, n_lon, out);
  GCB_CUDA(cudaGetLastError());
  return GCB_OK;
}

int gcb_gather_rows(const float* src, int32_t ld_src, const int32_t* idx, int64_t n, float* dst,
                    int32_t ld_dst, int32_t width, void* stream) {
  GCB_CHECK_ARG(n >= 0 && width > 0 && width % 4 == 0 && ld_src % 4 == 0 && ld_dst % 4 == 0 &&
                    ld_src >= width && ld_dst >= width, "bad width / ld");
  if (n == 0) return GCB_OK;
  GCB_CHECK_ARG(src && idx && dst && aligned16(src) && aligned16(dst), "null/unaligned pointer");
  long long blocks = (n + 7) / 8;
  const long long cap = static_cast<long long>(sm_count_cached()) * 8;
  if (blocks > cap) blocks = cap;
  ProfScope prof(static_cast<cudaStream_t>(stream), GCB_KIND_GATHER, 0.0, 8.0 * n * width);
  gcb::gather_rows_kernel<<<static_cast<int>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      src, ld_src, idx, n, dst, ld_dst, width);
  GCB_CUDA(cudaGetLastError());
  return GCB_OK;
}

static int image_rows(bool to_image, void* img, const int32_t* idx, int64_t first_row, int64_t n,
                      void* buf, void* stream) {
  GCB_CHECK_ARG(n >= 0 && first_row >= 0, "bad row range");
  if (n == 0) return GCB_OK;
  GCB_CHECK_ARG(img && buf && (to_image || idx) && aligned16(img) && aligned16(buf),
                "null/unaligned pointer");
  long long blocks = (n + 7) / 8;
  const long long cap = static_cast<long long>(sm_count_cached()) * 8;
  if (blocks > cap) blocks = cap;
  ProfScope prof(static_cast<cudaStream_t>(stream), GCB_KIND_GATHER, 0.0, 4096.0 * n);
  if (to_image)
    gcb::image_rows_kernel<true><<<static_cast<int>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<unsigned char*>(img), idx, first_row, n, static_cast<unsigned char*>(buf));
  else
    gcb::image_rows_kernel<false><<<static_cast<int>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<unsigned char*>(img), idx, first_row, n, static_cast<unsigned char*>(buf));
  GCB_CUDA(cudaGetLastError());
  return GCB_OK;
}

int gcb_image_rows_pack(const void* img, const int32_t* idx, int64_t n, void* buf, void* stream) {
  return image_rows(false, const_cast<void*>(img), idx, 0, n, buf, stream);
}

int gcb_image_rows_unpack(const void* buf, int64_t n, void* img, int64_t first_row, void* stream) {
  return image_rows(true, img, nullptr, first_row, n, const_cast<void*>(buf), stream);
}

int gcb_rows_to_image(const float* src, int32_t ld, int32_t fan, int64_t rows, int32_t k,
                      void* img, void* stream) {
  GCB_CHECK_ARG(src && img && aligned16(src) && aligned16(img), "null/unaligned pointer");
  GCB_CHECK_ARG(k > 0 && k % 16 == 0 && ld % 4 == 0 && ld >= k && fan >= 1, "bad k / ld / fan");
  if (rows == 0) return GCB_OK;
  const size_t smem = 32 * static_cast<size_t>(k + 4) * sizeof(float);
  static bool attr_set[64] = {false};     // per device: the opt-in is a per-context attribute
  int dev = 0;
  GCB_CUDA(cudaGetDevice(&dev));
  GCB_CHECK_ARG(dev >= 0 && dev < 64, "device index out of range");
  if (!attr_set[dev]) {
    GCB_CUDA(cudaFuncSetAttribute(gcb::rows_to_image_kernel,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    attr_set[dev] = true;
  }
  GCB_CHECK_ARG(smem <= 96 * 1024, "k too large");
  const long long padded = (rows + 127) / 128 * 128;      // zero-fill the tail of the last tile
  const unsigned grid = static_cast<unsigned>((padded + 31) / 32);
  ProfScope prof(static_cast<cudaStream_t>(stream), GCB_KIND_ROWS_TO_IMAGE, 0.0,
                 4.0 * rows * k * (fan + 1.0));
  gcb::rows_to_image_kernel<<<grid, 256, smem, static_cast<cudaStream_t>(stream)>>>(
      src, ld, fan, rows, k, static_cast<unsigned char*>(img));
  GCB_CUDA(cudaGetLastError());
  return GCB_OK;
}

namespace {

// One recorded step per (model, buffers, stream): gcb_forward runs eagerly the first time it
// sees a key (attribute / occupancy queries happen there), captures the same launch sequence
// into a CUDA graph the second time, and replays it afterwards.
struct StepGraph {
  std::vector<unsigned char> key;
  cudaGraphExec_t exec = nullptr;
  int launches = 0;
};
std::vector<StepGraph> g_step_graphs;
bool g_graph_replay = true;

void drop_step_graphs() {
  for (auto& g : g_step_graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  g_step_graphs.clear();
}

int forward_eager(const gcb_model* m, const void* grid_in_img, float* grid_out, void* stream,
                  int32_t* launches);

}  // namespace

int gcb_set_graph_replay(int32_t enabled) {
  g_graph_replay = enabled != 0;
  if (!g_graph_replay) drop_step_graphs();
  return GCB_OK;
}

int gcb_forward(const gcb_model* m, const void* grid_in_img, float* grid_out, void* stream,
                int32_t* launches) {
  GCB_CHECK_ARG(m && grid_in_img && grid_out, "null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  bool replay = g_graph_replay && !g_prof_on && st != nullptr && st != cudaStreamLegacy &&
                st != cudaStreamPerThread;
  if (replay) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
      cudaGetLastError();
      replay = false;               // the caller is capturing: just contribute the launches
    }
  }
  if (!replay) return forward_eager(m, grid_in_img, grid_out, stream, launches);

  std::vector<unsigned char> key(sizeof(gcb_model) + 4 * sizeof(void*));
  memcpy(key.data(), m, sizeof(gcb_model));
  const void* extra[4] = {grid_in_img, grid_out, stream,
                          reinterpret_cast<const void*>(static_cast<intptr_t>(g_cluster_size))};
  memcpy(key.data() + sizeof(gcb_model), extra, sizeof(extra));
  StepGraph* g = nullptr;
  for (auto& e : g_step_graphs)
    if (e.key == key) { g = &e; break; }
  int32_t n = 0;
  if (g == nullptr) {
    const int rc = forward_eager(m, grid_in_img, grid_out, stream, &n);
    if (rc != GCB_OK) return rc;
    if (g_step_graphs.size() >= 8) {
      if (g_step_graphs.front().exec) cudaGraphExecDestroy(g_step_graphs.front().exec);
      g_step_graphs.erase(g_step_graphs.begin());
    }
    StepGraph e;
    e.key = std::move(key);
    e.launches = n;
    g_step_graphs.push_back(std::move(e));
    if (launches) *launches = n;
    return GCB_OK;
  }
  if (g->exec == nullptr) {
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
      cudaGetLastError();
      g_graph_replay = false;
      return forward_eager(m, grid_in_img, grid_out, stream, launches);
    }
    const int rc = forward_eager(m, grid_in_img, grid_out, stream, &n);
    cudaGraph_t graph = nullptr;
    cudaError_t e = cudaStreamEndCapture(st, &graph);
    if (rc == GCB_OK && e == cudaSuccess) e = cudaGraphInstantiate(&g->exec, graph, 0);
    if (graph) cudaGraphDestroy(graph);
    if (rc != GCB_OK || e != cudaSuccess) {
      cudaGetLastError();
      g->exec = nullptr;
      g_graph_replay = false;       // never retry; fall back to plain launches
      if (rc != GCB_OK) return rc;
      return forward_eager(m, grid_in_img, grid_out, stream, launches);
    }
  }
  GCB_CUDA(cudaGraphLaunch(g->exec, st));
  if (launches) *launches = g->launches;
  return GCB_OK;
}

namespace {

int check_model(const gcb_model* m) {
  GCB_CHECK_ARG(m->msg_steps >= 1 && m->msg_steps <= GCB_MAX_MSG_STEPS, "msg_steps out of range");
  GCB_CHECK_ARG(m->hidden && m->edge_a_img && m->edge_b && m->mesh_in_img &&
                    m->grid_lat && m->grid_lat_img && m->mesh_lat && m->mesh_lat_img &&
                    m->mesh_agg && m->mesh_agg_img && m->mesh_edge && m->mesh_edge_img &&
                    m->mesh_msg && m->grid_agg_img,
                "workspace pointer is null");
  if (m->pregather)
    GCB_CHECK_ARG(m->zero_bias && m->proj_grid && m->proj_mesh_a && m->proj_mesh_b,
                  "pregather needs zero_bias and the proj_* buffers");
  if (m->fuse) GCB_CHECK_ARG(m->chain_scratch != nullptr, "fuse needs chain_scratch");
  GCB_CHECK_ARG(m->num_grid_owned >= 0 && m->num_grid_owned <= m->num_grid &&
                    m->num_mesh_owned >= 0 && m->num_mesh_owned <= m->num_mesh,
                "owned row counts out of range");
  return GCB_OK;
}

// Latent streams as images only (gcb_model.image_residual)?
bool img_only(const gcb_model* m) {
  return m->image_residual && m->fuse && m->pregather && m->precision != GCB_PREC_FP32_SIMT;
}
// Output of an MLP that CREATES a latent stream (master + image, or image only).
MlpOut latent_new(const gcb_model* m, float* master, void* img) {
  MlpOut o;
  o.out_img = img;
  if (!img_only(m)) o.out = master;
  return o;
}
// Output of an MLP that UPDATES a latent stream in place: x += y.
MlpOut latent_update(const gcb_model* m, float* master, void* img) {
  MlpOut o;
  o.out_img = img;
  if (img_only(m)) { o.residual_img = img; }
  else { o.residual = master; o.out = master; }
  return o;
}

// Rows that node updates cover: all of them, or the owned prefix of a partition's local table.
int grid_rows(const gcb_model* m) { return m->num_grid_owned > 0 ? m->num_grid_owned : m->num_grid; }
int mesh_rows(const gcb_model* m) { return m->num_mesh_owned > 0 ? m->num_mesh_owned : m->num_mesh; }

// ---- deep chains ("mega" mode) -----------------------------------------------------------
// With image-only latents on one GPU the step is composed of chains of up to four layers, so
// that whole blocks of the message-passing step are one launch and their intermediates stay
// in the L2-resident scratch: [edge embedder MLP -> edge MLP] of the two bipartite graphs (the
// embedded edge latents never exist in HBM), [node MLP -> sender / receiver projections of the
// NEXT edge MLP], and the first processor step's [edge embedder -> edge MLP].
bool mega(const gcb_model* m) {
  return img_only(m) && m->deep_chains && m->num_grid_owned == 0 && m->num_mesh_owned == 0 &&
         m->proj_grid_b != nullptr;
}

struct Chain {
  gcb_chain_desc d;
  Chain(const gcb_model* m, int rows, int order) {
    memset(&d, 0, sizeof(d));
    d.rows = rows; d.precision = m->precision; d.lag = m->chain_lag; d.order = order;
    d.scratch = m->chain_scratch; d.scratch_bytes = m->chain_scratch_bytes;
  }
  gcb_chain_layer& add() {
    gcb_chain_layer& l = d.layer[d.nlayers++];
    l.seg_from[0] = l.seg_from[1] = l.seg_from[2] = -1;
    return l;
  }
  int last() const { return d.nlayers - 1; }
  // first linear of an MLP over external segments (swish, kept for the second linear)
  gcb_chain_layer& mlp0(const gcb_mlp& w, int nseg, const gcb_segment* segs, const void* w0 = nullptr) {
    gcb_chain_layer& l = add();
    l.nseg = nseg;
    for (int s = 0; s < nseg; ++s) l.seg[s] = segs[s];
    l.w_packed = w0 ? w0 : w.w0_packed; l.bias = w.b0; l.act = GCB_ACT_SWISH; l.keep = 1;
    return l;
  }
  // first linear of an MLP whose single input is the kept result of layer `from`
  gcb_chain_layer& mlp0_from(const gcb_mlp& w, int from, const void* w0 = nullptr) {
    gcb_chain_layer& l = add();
    l.nseg = 1; l.seg_from[0] = from; l.seg[0].k = 512;
    l.w_packed = w0 ? w0 : w.w0_packed; l.bias = w.b0; l.act = GCB_ACT_SWISH; l.keep = 1;
    return l;
  }
  // second linear + LayerNorm of the MLP whose first linear is the previous layer
  gcb_chain_layer& mlp1(const gcb_mlp& w) {
    const int from = last();
    gcb_chain_layer& l = add();
    l.nseg = 1; l.seg_from[0] = from; l.seg[0].k = 512;
    l.w_packed = w.w1_packed; l.bias = w.b1; l.ln_scale = w.ln_scale; l.ln_offset = w.ln_offset;
    l.ld_res = l.ld_out = l.ld_out_y = 512;
    return l;
  }
  // node-level projection of the kept result of layer `from` (no bias, no activation)
  gcb_chain_layer& proj(int from, const void* w_packed, float* out) {
    gcb_chain_layer& l = add();
    l.nseg = 1; l.seg_from[0] = from; l.seg[0].k = 512;
    l.w_packed = w_packed; l.out = out; l.ld_out = 512;
    return l;
  }
  int run(StepCtx& c) {
    const int rc = gcb_chain_forward(&d, c.stream);
    if (rc == GCB_OK) c.launches += 1;
    return rc;
  }
};

void set_pre(gcb_chain_layer& l, const float* ps, const int32_t* snd, const float* pr, const int32_t* rcv) {
  l.n_pre_add = 2;
  l.pre_add[0].table = ps; l.pre_add[0].idx = snd; l.pre_add[0].ld = 512;
  l.pre_add[1].table = pr; l.pre_add[1].idx = rcv; l.pre_add[1].ld = 512;
}

int mega_encode(StepCtx& c, const void* grid_in_img) {
  const gcb_model* m = c.m;
  int rc;
  gcb_segment s[3];
  const int D = 512;
  {  // vg0 = LN.MLP(grid_in) -> grid_lat_img;  proj_grid = vg0 @ W_s(grid2mesh)
    Chain ch(m, m->num_grid, 1);
    s[0] = seg_img(grid_in_img, m->c_in_pad);
    ch.mlp0(m->enc_grid, 1, s);
    gcb_chain_layer& l1 = ch.mlp1(m->enc_grid);
    l1.out_img = m->grid_lat_img; l1.keep = 1;
    ch.proj(ch.last(), m->proc_e_g2m_split.ws_packed, m->proj_grid);
    if ((rc = ch.run(c))) return rc;
  }
  {  // vm0 = LN.MLP(mesh_in) -> mesh_lat_img;  proj_mesh_a = vm0 @ W_r(grid2mesh)
    Chain ch(m, m->num_mesh, 1);
    s[0] = seg_img(m->mesh_in_img, m->c_in_pad);
    ch.mlp0(m->enc_mesh, 1, s);
    gcb_chain_layer& l1 = ch.mlp1(m->enc_mesh);
    l1.out_img = m->mesh_lat_img; l1.keep = 1;
    ch.proj(ch.last(), m->proc_e_g2m_split.wr_packed, m->proj_mesh_a);
    if ((rc = ch.run(c))) return rc;
  }
  {  // e1 = LN.MLP(edge feats);  m1 = LN.MLP([e1 | vg0[snd] | vm0[rcv]]) -> edge_b
    Chain ch(m, m->e_g2m, 1);
    s[0] = seg(m->g2m_feat, nullptr, 4, 16, 4);
    ch.mlp0(m->enc_e_g2m, 1, s);
    ch.mlp1(m->enc_e_g2m).keep = 1;
    set_pre(ch.mlp0_from(m->proc_e_g2m, ch.last(), m->proc_e_g2m_split.we_packed),
            m->proj_grid, m->g2m_snd, m->proj_mesh_a, m->g2m_rcv);
    ch.mlp1(m->proc_e_g2m).out = m->edge_b;
    if ((rc = ch.run(c))) return rc;
  }
  if ((rc = segment_sum_launch(m->edge_b, D, m->g2m_row_ptr, m->num_mesh, m->g2m_heavy,
                               m->n_g2m_heavy, m->mesh_agg, D, D, m->mesh_agg_img, m->e_g2m,
                               c.stream))) return rc;
  c.launches += 1;
  {  // vm1 = vm0 + LN.MLP([vm0 | agg1]);  projections of the first processor step
    Chain ch(m, m->num_mesh, 1);
    s[0] = seg_img(m->mesh_lat_img, D);
    s[1] = seg_img(m->mesh_agg_img, D);
    ch.mlp0(m->proc_n_mesh_g2m, 2, s);
    gcb_chain_layer& l1 = ch.mlp1(m->proc_n_mesh_g2m);
    l1.residual_img = m->mesh_lat_img; l1.out_img = m->mesh_lat_img; l1.keep = 1;
    const int v = ch.last();
    ch.proj(v, m->proc_e_mesh_split[0].ws_packed, m->proj_mesh_a);
    ch.proj(v, m->proc_e_mesh_split[0].wr_packed, m->proj_mesh_b);
    if ((rc = ch.run(c))) return rc;
  }
  {  // vg1 = vg0 + LN.MLP([vg0]);  proj_grid_b = vg1 @ W_r(mesh2grid)
    Chain ch(m, m->num_grid, 1);
    s[0] = seg_img(m->grid_lat_img, D);
    ch.mlp0(m->proc_n_grid_g2m, 1, s);
    gcb_chain_layer& l1 = ch.mlp1(m->proc_n_grid_g2m);
    l1.residual_img = m->grid_lat_img; l1.out_img = m->grid_lat_img; l1.keep = 1;
    ch.proj(ch.last(), m->proc_e_m2g_split.wr_packed, m->proj_grid_b);
    if ((rc = ch.run(c))) return rc;
  }
  return GCB_OK;
}

int mega_process_step(StepCtx& c, int k) {
  const gcb_model* m = c.m;
  GCB_CHECK_ARG(k >= 0 && k < m->msg_steps, "message-passing step out of range");
  int rc;
  gcb_segment s[3];
  const int D = 512;
  const bool last = (k == m->msg_steps - 1);
  if (k == 0) {
    // e0 = LN.MLP(edge feats);  m = LN.MLP([e0 | v[snd] | v[rcv]]);  e1 = e0 + m  (e0 stays on chip)
    Chain ch(m, m->e_mesh, 1);
    s[0] = seg(m->mesh_feat, nullptr, 4, 16, 4);
    ch.mlp0(m->enc_e_mesh, 1, s);
    ch.mlp1(m->enc_e_mesh).keep = 1;
    const int e0 = ch.last();
    set_pre(ch.mlp0_from(m->proc_e_mesh[0], e0, m->proc_e_mesh_split[0].we_packed),
            m->proj_mesh_a, m->mesh_snd, m->proj_mesh_b, m->mesh_rcv);
    gcb_chain_layer& l3 = ch.mlp1(m->proc_e_mesh[0]);
    l3.out_y = m->mesh_msg;
    if (!last) { l3.residual_keep = e0 + 1; l3.out_img = m->mesh_edge_img; }
    if ((rc = ch.run(c))) return rc;
  } else {
    Chain ch(m, m->e_mesh, 0);
    s[0] = seg_img(m->mesh_edge_img, D);
    set_pre(ch.mlp0(m->proc_e_mesh[k], 1, s, m->proc_e_mesh_split[k].we_packed),
            m->proj_mesh_a, m->mesh_snd, m->proj_mesh_b, m->mesh_rcv);
    gcb_chain_layer& l1 = ch.mlp1(m->proc_e_mesh[k]);
    l1.out_y = m->mesh_msg;
    if (!last) { l1.residual_img = m->mesh_edge_img; l1.out_img = m->mesh_edge_img; }
    if ((rc = ch.run(c))) return rc;
  }
  if ((rc = segment_sum_launch(m->mesh_msg, D, m->mesh_row_ptr, m->num_mesh, nullptr, 0, m->mesh_agg,
                               D, D, m->mesh_agg_img, m->e_mesh, c.stream))) return rc;
  c.launches += 1;
  {  // v += LN.MLP([v | agg]);  projections of the next edge MLP (next step, or mesh2grid senders)
    Chain ch(m, m->num_mesh, 1);
    s[0] = seg_img(m->mesh_lat_img, D);
    s[1] = seg_img(m->mesh_agg_img, D);
    ch.mlp0(m->proc_n_mesh[k], 2, s);
    gcb_chain_layer& l1 = ch.mlp1(m->proc_n_mesh[k]);
    l1.residual_img = m->mesh_lat_img; l1.out_img = m->mesh_lat_img; l1.keep = 1;
    const int v = ch.last();
    if (!last) {
      ch.proj(v, m->proc_e_mesh_split[k + 1].ws_packed, m->proj_mesh_a);
      ch.proj(v, m->proc_e_mesh_split[k + 1].wr_packed, m->proj_mesh_b);
    } else {
      ch.proj(v, m->proc_e_m2g_split.ws_packed, m->proj_mesh_a);
    }
    if ((rc = ch.run(c))) return rc;
  }
  return GCB_OK;
}

int mega_decode(StepCtx& c, float* grid_out) {
  const gcb_model* m = c.m;
  int rc;
  gcb_segment s[3];
  const int D = 512;
  GCB_CHECK_ARG(m->e_m2g == 3 * m->num_grid, "mesh2grid must have fan-in 3");
  {  // e3 = LN.MLP(edge feats);  m3 = LN.MLP([e3 | v[snd] | vg1[rcv]]) -> edge_b
    Chain ch(m, m->e_m2g, 1);
    s[0] = seg(m->m2g_feat, nullptr, 4, 16, 4);
    ch.mlp0(m->enc_e_m2g, 1, s);
    ch.mlp1(m->enc_e_m2g).keep = 1;
    set_pre(ch.mlp0_from(m->proc_e_m2g, ch.last(), m->proc_e_m2g_split.we_packed),
            m->proj_mesh_a, m->m2g_snd, m->proj_grid_b, m->m2g_rcv);
    ch.mlp1(m->proc_e_m2g).out = m->edge_b;
    if ((rc = ch.run(c))) return rc;
  }
  if ((rc = to_image(c, m->edge_b, D, 3, m->num_grid, D, m->grid_agg_img))) return rc;
  {  // vg2 = vg1 + LN.MLP([vg1 | agg3])
    Chain ch(m, m->num_grid, 0);
    s[0] = seg_img(m->grid_lat_img, D);
    s[1] = seg_img(m->grid_agg_img, D);
    ch.mlp0(m->proc_n_grid_m2g, 2, s);
    gcb_chain_layer& l1 = ch.mlp1(m->proc_n_grid_m2g);
    l1.residual_img = m->grid_lat_img; l1.out_img = m->grid_lat_img;
    if ((rc = ch.run(c))) return rc;
  }
  // out = MLP(vg2), no LayerNorm (deep_typed_graph_net.py:314-322)
  s[0] = seg_img(m->grid_lat_img, D);
  MlpOut o; o.out = grid_out; o.ld_out = 256;
  return run_mlp(c, m->dec_grid, m->num_grid, 1, s, o);
}

// ---------------- encoder: grid2mesh_gnn (graphcast.py:550-604) ----------------
int stage_encode(StepCtx& c, const void* grid_in_img) {
  if (mega(c.m)) return mega_encode(c, grid_in_img);
  const gcb_model* m = c.m;
  int rc;
  gcb_segment s[3];
  const int D = 512;
  MlpOut o;
  // vg0 = LN.MLP(grid_in)  -> grid_lat (+ image)
  s[0] = seg_img(grid_in_img, m->c_in_pad);
  o = latent_new(m, m->grid_lat, m->grid_lat_img);
  if ((rc = run_mlp(c, m->enc_grid, m->num_grid, 1, s, o))) return rc;
  // vm0 = LN.MLP(mesh_in)  -> mesh_lat (+ image)
  s[0] = seg_img(m->mesh_in_img, m->c_in_pad);
  o = latent_new(m, m->mesh_lat, m->mesh_lat_img);
  if ((rc = run_mlp(c, m->enc_mesh, m->num_mesh, 1, s, o))) return rc;
  // e1 = LN.MLP(g2m edge feats)  -> image only (its fp32 form is never needed)
  s[0] = seg(m->g2m_feat, nullptr, 4, 16, 4);
  o = MlpOut(); o.out_img = m->edge_a_img;
  if ((rc = run_mlp(c, m->enc_e_g2m, m->e_g2m, 1, s, o))) return rc;
  // m1 = LN.MLP([e1 | vg0[snd] | vm0[rcv]])  -> edge_b   (edge residual e1+m1 is dead)
  o = MlpOut(); o.out = m->edge_b;
  if ((rc = run_edge_mlp(c, m->proc_e_g2m, &m->proc_e_g2m_split, m->e_g2m, m->edge_a_img,
                         m->grid_lat, m->grid_lat_img, m->num_grid, m->g2m_snd, m->proj_grid,
                         m->mesh_lat, m->mesh_lat_img, mesh_rows(m), m->g2m_rcv, m->proj_mesh_a, o)))
    return rc;
  // agg1 = segment_sum(m1)
  if ((rc = segment_sum_launch(m->edge_b, D, m->g2m_row_ptr, mesh_rows(m), m->g2m_heavy,
                               m->n_g2m_heavy, m->mesh_agg, D, D, m->mesh_agg_img, m->e_g2m,
                               c.stream))) return rc;
  c.launches += 1;
  // vm1 = vm0 + LN.MLP([vm0 | agg1])  (in place)
  s[0] = seg_img(m->mesh_lat_img, D);
  s[1] = seg_img(m->mesh_agg_img, D);
  o = latent_update(m, m->mesh_lat, m->mesh_lat_img);
  if ((rc = run_mlp(c, m->proc_n_mesh_g2m, mesh_rows(m), 2, s, o))) return rc;
  // vg1 = vg0 + LN.MLP([vg0])  (in place; grid nodes receive nothing in grid2mesh)
  s[0] = seg_img(m->grid_lat_img, D);
  o = latent_update(m, m->grid_lat, m->grid_lat_img);
  return run_mlp(c, m->proc_n_grid_g2m, grid_rows(m), 1, s, o);
}

// ---------------- processor: mesh_gnn (graphcast.py:606-639) --------------------
int stage_process_embed(StepCtx& c) {
  const gcb_model* m = c.m;
  if (mega(m)) return GCB_OK;      // folded into the first step's edge chain
  gcb_segment s[3];
  s[0] = seg(m->mesh_feat, nullptr, 4, 16, 4);
  MlpOut o = latent_new(m, m->mesh_edge, m->mesh_edge_img);
  return run_mlp(c, m->enc_e_mesh, m->e_mesh, 1, s, o);
}

int stage_process_step(StepCtx& c, int k) {
  const gcb_model* m = c.m;
  if (mega(m)) return mega_process_step(c, k);
  GCB_CHECK_ARG(k >= 0 && k < m->msg_steps, "message-passing step out of range");
  int rc;
  gcb_segment s[3];
  const int D = 512;
  const bool last = (k == m->msg_steps - 1);
  // m = LN.MLP([e | v[snd] | v[rcv]]) -> mesh_msg;  e += m (skipped on the last step: the
  // updated edge latents are never read again).
  MlpOut o;
  if (!last) o = latent_update(m, m->mesh_edge, m->mesh_edge_img);
  o.out_y = m->mesh_msg;
  if ((rc = run_edge_mlp(c, m->proc_e_mesh[k], &m->proc_e_mesh_split[k], m->e_mesh, m->mesh_edge_img,
                         m->mesh_lat, m->mesh_lat_img, m->num_mesh, m->mesh_snd, m->proj_mesh_a,
                         m->mesh_lat, m->mesh_lat_img, mesh_rows(m), m->mesh_rcv, m->proj_mesh_b, o)))
    return rc;
  if ((rc = segment_sum_launch(m->mesh_msg, D, m->mesh_row_ptr, mesh_rows(m), nullptr, 0, m->mesh_agg,
                               D, D, m->mesh_agg_img, m->e_mesh, c.stream))) return rc;
  c.launches += 1;
  // v += LN.MLP([v | agg])
  s[0] = seg_img(m->mesh_lat_img, D);
  s[1] = seg_img(m->mesh_agg_img, D);
  o = latent_update(m, m->mesh_lat, m->mesh_lat_img);
  return run_mlp(c, m->proc_n_mesh[k], mesh_rows(m), 2, s, o);
}

// ---------------- decoder: mesh2grid_gnn (graphcast.py:641-678) ------------------
int stage_decode(StepCtx& c, float* grid_out) {
  const gcb_model* m = c.m;
  if (mega(m)) return mega_decode(c, grid_out);
  int rc;
  gcb_segment s[3];
  const int D = 512;
  const int ng = grid_rows(m);
  GCB_CHECK_ARG(m->e_m2g == 3 * ng, "mesh2grid must have fan-in 3 over the (owned) grid rows");
  s[0] = seg(m->m2g_feat, nullptr, 4, 16, 4);
  MlpOut o; o.out_img = m->edge_a_img;
  if ((rc = run_mlp(c, m->enc_e_m2g, m->e_m2g, 1, s, o))) return rc;
  // m3 = LN.MLP([e3 | v[snd] | vg1[rcv]]) -> edge_b
  o = MlpOut(); o.out = m->edge_b;
  if ((rc = run_edge_mlp(c, m->proc_e_m2g, &m->proc_e_m2g_split, m->e_m2g, m->edge_a_img,
                         m->mesh_lat, m->mesh_lat_img, m->num_mesh, m->m2g_snd, m->proj_mesh_a,
                         m->grid_lat, m->grid_lat_img, ng, m->m2g_rcv, m->proj_grid, o)))
    return rc;
  // sum of the 3 incoming messages of every grid node, as an operand image
  if ((rc = to_image(c, m->edge_b, D, 3, ng, D, m->grid_agg_img))) return rc;
  // vg2 = vg1 + LN.MLP([vg1 | agg3])  (in place)
  s[0] = seg_img(m->grid_lat_img, D);
  s[1] = seg_img(m->grid_agg_img, D);
  o = latent_update(m, m->grid_lat, m->grid_lat_img);
  if ((rc = run_mlp(c, m->proc_n_grid_m2g, ng, 2, s, o))) return rc;
  // out = MLP(vg2), no LayerNorm (deep_typed_graph_net.py:314-322)
  s[0] = seg_img(m->grid_lat_img, D);
  o = MlpOut(); o.out = grid_out; o.ld_out = 256;
  return run_mlp(c, m->dec_grid, ng, 1, s, o);
}

int forward_eager(const gcb_model* m, const void* grid_in_img, float* grid_out, void* stream,
                  int32_t* launches) {
  int rc = check_model(m);
  if (rc) return rc;
  StepCtx c{m, static_cast<cudaStream_t>(stream), 0};
  if ((rc = stage_encode(c, grid_in_img))) return rc;
  if ((rc = stage_process_embed(c))) return rc;
  for (int k = 0; k < m->msg_steps; ++k)
    if ((rc = stage_process_step(c, k))) return rc;
  if ((rc = stage_decode(c, grid_out))) return rc;
  if (launches) *launches = c.launches;
  return GCB_OK;
}

}  // namespace

int gcb_forward_stage(const gcb_model* m, int32_t stage, int32_t step, const void* grid_in_img,
                      float* grid_out, void* stream, int32_t* launches) {
  GCB_CHECK_ARG(m != nullptr, "null model");
  int rc = check_model(m);
  if (rc) return rc;
  StepCtx c{m, static_cast<cudaStream_t>(stream), 0};
  switch (stage) {
    case GCB_STAGE_ENCODE:
      GCB_CHECK_ARG(grid_in_img != nullptr, "ENCODE needs grid_in_img");
      rc = stage_encode(c, grid_in_img);
      break;
    case GCB_STAGE_PROCESS_EMBED: rc = stage_process_embed(c); break;
    case GCB_STAGE_PROCESS_STEP: rc = stage_process_step(c, step); break;
    case GCB_STAGE_DECODE:
      GCB_CHECK_ARG(grid_out != nullptr, "DECODE needs grid_out");
      rc = stage_decode(c, grid_out);
      break;
    default: return fail(GCB_ERR_INVALID, "invalid argument: unknown stage");
  }
  if (launches) *launches = c.launches;
  return rc;
}

int gcb_set_cluster_size(int32_t ctas) {
  GCB_CHECK_ARG(ctas == 1 || ctas == 2 || ctas == 4, "cluster size must be 1, 2 or 4");
  g_cluster_size = ctas;
  return GCB_OK;
}

int gcb_debug_trace(long long* device_buffer) {
  // device_buffer: [kTraceTiles * kTraceEvents] int64 on the device, or NULL to disable.
  GCB_CUDA(cudaMemcpyToSymbol(gcb::g_trace, &device_buffer, sizeof(device_buffer)));
  return GCB_OK;
}

int gcb_debug_flags(int flags) {
  GCB_CUDA(cudaMemcpyToSymbol(gcb::g_dbg_flags, &flags, sizeof(flags)));
  return GCB_OK;
}

int gcb_profile_begin(void) {
  for (auto& r : g_prof) { g_event_pool.push_back(r.beg); g_event_pool.push_back(r.end); }
  g_prof.clear();
  g_prof_on = true;
  return GCB_OK;
}

int gcb_profile_end(int32_t capacity, int32_t* kinds, float* ms, double* flops, double* bytes,
                    int32_t* count) {
  g_prof_on = false;
  GCB_CHECK_ARG(count != nullptr, "count is null");
  const int n = static_cast<int>(g_prof.size());
  *count = n;
  for (int i = 0; i < n && i < capacity; ++i) {
    GCB_CUDA(cudaEventSynchronize(g_prof[i].end));
    float t = 0.f;
    GCB_CUDA(cudaEventElapsedTime(&t, g_prof[i].beg, g_prof[i].end));
    if (kinds) kinds[i] = g_prof[i].kind;
    if (ms) ms[i] = t;
    if (flops) flops[i] = g_prof[i].flops;
    if (bytes) bytes[i] = g_prof[i].bytes;
  }
  for (auto& r : g_prof) { g_event_pool.push_back(r.beg); g_event_pool.push_back(r.end); }
  g_prof.clear();
  return GCB_OK;
}

int gcb_selftest_layer(int32_t rows, int32_t k, int32_t n, int32_t precision, float* rel_err) {
  GCB_CHECK_ARG(rows > 0 && k > 0 && k % 16 == 0 && (n == 256 || n == 512) && rel_err, "bad shape");
  std::vector<float> ha(static_cast<size_t>(rows) * k), hw(static_cast<size_t>(k) * n), hb(n), hs(n), ho(n);
  uint32_t st = 12345u;
  auto rnd = [&]() { st = st * 1664525u + 1013904223u; return (static_cast<float>(st >> 8) / 8388608.0f) - 1.0f; };
  for (auto& v : ha) v = rnd();
  const float wscale = 1.0f / sqrtf(static_cast<float>(k));
  for (auto& v : hw) v = rnd() * wscale;
  for (int i = 0; i < n; ++i) { hb[i] = 0.1f * rnd(); hs[i] = 1.0f + 0.1f * rnd(); ho[i] = 0.1f * rnd(); }
  std::vector<uint8_t> himg(static_cast<size_t>(gcb_packed_weight_bytes(k, n)));
  int rc = gcb_pack_weight_host(hw.data(), k, n, k, n, himg.data());
  if (rc) return rc;
  float *da = nullptr, *dw = nullptr, *db = nullptr, *ds = nullptr, *dof = nullptr, *o1 = nullptr, *o2 = nullptr;
  void* dimg = nullptr;
  GCB_CUDA(cudaMalloc(&da, ha.size() * 4));
  GCB_CUDA(cudaMalloc(&dw, hw.size() * 4));
  GCB_CUDA(cudaMalloc(&db, n * 4));
  GCB_CUDA(cudaMalloc(&ds, n * 4));
  GCB_CUDA(cudaMalloc(&dof, n * 4));
  GCB_CUDA(cudaMalloc(&o1, static_cast<size_t>(rows) * n * 4));
  GCB_CUDA(cudaMalloc(&o2, static_cast<size_t>(rows) * n * 4));
  GCB_CUDA(cudaMalloc(&dimg, himg.size()));
  GCB_CUDA(cudaMemcpy(da, ha.data(), ha.size() * 4, cudaMemcpyHostToDevice));
  GCB_CUDA(cudaMemcpy(dw, hw.data(), hw.size() * 4, cudaMemcpyHostToDevice));
  GCB_CUDA(cudaMemcpy(db, hb.data(), n * 4, cudaMemcpyHostToDevice));
  GCB_CUDA(cudaMemcpy(ds, hs.data(), n * 4, cudaMemcpyHostToDevice));
  GCB_CUDA(cudaMemcpy(dof, ho.data(), n * 4, cudaMemcpyHostToDevice));
  GCB_CUDA(cudaMemcpy(dimg, himg.data(), himg.size(), cudaMemcpyHostToDevice));
  gcb_layer_desc d;
  memset(&d, 0, sizeof(d));
  d.rows = rows; d.n = n; d.n_valid = n; d.nseg = 1;
  d.seg[0].table = da; d.seg[0].ld = k; d.seg[0].k = k; d.seg[0].k_valid = k; d.seg[0].fan = 1;
  d.w_packed = dimg; d.w_f32 = dw; d.bias = db; d.ln_scale = ds; d.ln_offset = dof;
  d.act = GCB_ACT_NONE;
  d.out = o1; d.ld_out = n;
  d.precision = precision;
  rc = gcb_layer_forward(&d, nullptr);
  if (rc) return rc;
  d.out = o2; d.precision = GCB_PREC_FP32_SIMT;
  rc = gcb_layer_forward(&d, nullptr);
  if (rc) return rc;
  GCB_CUDA(cudaDeviceSynchronize());
  std::vector<float> r1(static_cast<size_t>(rows) * n), r2(r1.size());
  GCB_CUDA(cudaMemcpy(r1.data(), o1, r1.size() * 4, cudaMemcpyDeviceToHost));
  GCB_CUDA(cudaMemcpy(r2.data(), o2, r2.size() * 4, cudaMemcpyDeviceToHost));
  double maxd = 0, maxr = 0;
  for (size_t i = 0; i < r1.size(); ++i) {
    const double dd = fabs(static_cast<double>(r1[i]) - r2[i]);
    if (!(dd <= maxd)) maxd = dd;   // propagates NaN
    if (fabs(r2[i]) > maxr) maxr = fabs(r2[i]);
  }
  *rel_err = static_cast<float>(maxd / (maxr > 0 ? maxr : 1.0));
  cudaFree(da); cudaFree(dw); cudaFree(db); cudaFree(ds); cudaFree(dof); cudaFree(o1); cudaFree(o2); cudaFree(dimg);
  return GCB_OK;
}

}  // extern "C"
