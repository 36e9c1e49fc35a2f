/* graphcast_b200 -- C ABI of the B200-native GraphCast hot path.
 *
 * This is the drop-in boundary: a plain C interface (pointers and sizes, no
 * torch / C++ types) over hand-written sm_100a CUDA kernels.  The reference is
 * pure Python/JAX and has no FFI of its own; each entry point below names the
 * reference function (file:line under /root/reference) whose work it replaces.
 * The Python mirror (graphcast_b200/graphcast.py, rollout.py) binds these with
 * ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every pointer inside gcb_* structs is a DEVICE pointer unless stated;
 *     buffers are owned by the caller (PyTorch allocations in the Python host);
 *   - all functions take a CUDA stream (cudaStream_t passed as void*) and are
 *     asynchronous with respect to the host; nothing here allocates or syncs;
 *   - return value 0 = success; otherwise a negative gcb_status and
 *     gcb_last_error() describes the failure (thread-local string);
 *   - float tensors are fp32 row-major; node/edge feature tables are
 *     [rows, ld] with ld a multiple of 4 (16-byte rows).
 */
#ifndef GRAPHCAST_B200_H_
#define GRAPHCAST_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GCB_ABI_VERSION 2

typedef enum {
  GCB_OK = 0,
  GCB_ERR_INVALID = -1,  /* bad argument (shape, alignment, null pointer) */
  GCB_ERR_CUDA = -2,     /* a CUDA runtime call / launch failed */
  GCB_ERR_UNSUPPORTED = -3
} gcb_status;

/* Arithmetic of the dense MLP contractions.
 *   BF16X3    : every fp32 operand is split x = hi + lo (two bf16), the product is
 *               formed as hi*hi + hi*lo + lo*hi on tcgen05 tensor cores with fp32
 *               accumulation in TMEM.  ~2^-17 relative operand error: this is the
 *               parity mode (<= 1e-4 vs the fp32 oracle over a full step).
 *   BF16      : single bf16 product (the numerics of the reference's
 *               casting.Bfloat16Cast demo stack, utils/casting.py:31-65); fast,
 *               does NOT meet the 1e-4 gate.
 *   FP32_SIMT : fp32 FFMA on CUDA cores; slow validation arm for the tensor path. */
typedef enum { GCB_PREC_BF16X3 = 0, GCB_PREC_BF16 = 1, GCB_PREC_FP32_SIMT = 2 } gcb_precision;

typedef enum { GCB_ACT_NONE = 0, GCB_ACT_SWISH = 1 } gcb_activation;

/* One K-segment of a layer input.  The logical input row r of the layer is the
 * concatenation over segments of
 *     sum_{j < fan} table[(idx ? idx[r] : r) * fan + j, 0:k_valid]   (zero padded to k)
 * i.e. a gathered node/edge row (jax_gather, utils/typed_graph_net.py:124-125,
 * 431-445) or, with fan > 1, a fixed fan-in segment sum of consecutive rows
 * (jraph.segment_sum for the mesh2grid graph, typed_graph_net.py:535-537). */
typedef struct {
  const float* table;   /* [*, ld] fp32 */
  const int32_t* idx;   /* [rows] gather index or NULL (identity) */
  int32_t ld;           /* row stride in floats, multiple of 4 */
  int32_t k;            /* padded width, multiple of 16 */
  int32_t k_valid;      /* real width (<= k, multiple of 4) */
  int32_t fan;          /* >= 1 */
  /* Alternative source: an operand image (see below) of a [rows, k] matrix, identity
   * rows.  When non-NULL, table/idx/ld/k_valid/fan are ignored and the K-steps of this
   * segment are streamed by TMA bulk copies instead of the gather warps. */
  const void* img;
} gcb_segment;

/* A gathered pre-activation addend:  y_pre[r, :] += table[(idx ? idx[r] : r), 0:n].
 * Used for the algebraically split first edge-MLP layer
 *     [e | v_s | v_r] @ W  =  e @ W_e + (v @ W_s)[senders] + (v @ W_r)[receivers]
 * where the node-level projections are computed once per node instead of per edge
 * (the reference's newer DeepGNN does the same, utils/deep_gnn.py:106-108,245-260). */
typedef struct {
  const float* table;   /* [*, ld] fp32 */
  const int32_t* idx;   /* [rows] gather index or NULL */
  int32_t ld;
  int32_t pad_;
} gcb_pre_add;

/* One fused linear layer over `rows` rows:
 *     z   = concat(segments)                         [rows, K],  K = sum k
 *     y   = act(z @ W + bias + sum_p pre_add_p)      [rows, n]
 *     y   = LayerNorm(y) * ln_scale + ln_offset      (if ln_scale != NULL; eps 1e-5)
 * A layer has either the swish activation or LayerNorm, not both (GCB_ERR_INVALID);
 * LayerNorm statistics are over the n_valid columns.
 *     out_y[r] = y[r]                                (if out_y  != NULL)
 *     out[r]   = (residual ? residual[r] : 0) + y[r] (if out    != NULL)
 * Replaces one hk.Linear (+ jax.nn.swish | + hk.LayerNorm + residual add) of
 * build_mlp_with_maybe_layer_norm (utils/legacy/deep_typed_graph_net.py:205-247),
 * the concat of jraph.concatenated_args, and the residuals of _process_step
 * (deep_typed_graph_net.py:380-389). */
typedef struct {
  int32_t rows;
  int32_t n;            /* padded output width: 256 or 512 */
  int32_t n_valid;      /* real output width (<= n); columns beyond are not stored */
  int32_t nseg;         /* 1..3 */
  gcb_segment seg[3];
  const void* w_packed; /* bf16 hi/lo tile image made by gcb_pack_weight_* */
  const float* w_f32;   /* [K, n] fp32 row-major (FP32_SIMT arm only) */
  const float* bias;    /* [n] */
  const float* ln_scale;  /* [n] or NULL */
  const float* ln_offset; /* [n] or NULL (required iff ln_scale) */
  int32_t act;          /* gcb_activation */
  const float* residual; int32_t ld_res;
  float* out;   int32_t ld_out;
  float* out_y; int32_t ld_out_y;
  int32_t precision;    /* gcb_precision */
  int32_t n_pre_add;    /* 0..2; requires ln_scale == NULL and n_valid % 32 == 0 */
  gcb_pre_add pre_add[2];
  /* Operand images.  The "A image" of a [rows, k] fp32 matrix is its bf16 hi/lo split
   * stored tile by tile in the exact shared-memory layout of the tensor-core A operand:
   * for row tile t (128 rows) and K-step s (16 columns) one block of GCB_A_IMAGE_BLOCK
   * bytes = [hi: 2 chunks x (128 rows x 16 B), 64 B skew | lo: same], blocks ordered
   * [t][s].  gcb_a_image_bytes(rows, k) gives the buffer size.
   *   out_img != NULL : the layer result (out semantics: residual + y; n = n_valid = 512)
   *                     is ALSO written as an image, ready to be a segment.img later. */
  void* out_img;
} gcb_layer_desc;

#define GCB_A_IMAGE_BLOCK 8448
int64_t gcb_a_image_bytes(int64_t rows, int32_t k);

/* img[r, 0:k] = sum_{j < fan} src[(r*fan + j), 0:k]  as an operand image (k multiple of
 * 16, k <= ld).  fan = 1 converts an fp32 matrix; fan = 3 is the mesh2grid aggregation
 * (jraph.segment_sum over the 3 incoming edges of a grid node, typed_graph_net.py:535-537). */
int gcb_rows_to_image(const float* src, int32_t ld, int32_t fan, int64_t rows, int32_t k,
                      void* img, void* stream);

/* dst[i, 0:width] = src[idx[i], 0:width] for i < n (fp32, width a multiple of 4).  Packs the
 * boundary rows of a latent table into the contiguous send buffer of the per-step halo exchange
 * of the node-partitioned processor (the reference's analogue: the all_gather in front of every
 * sharded gather, utils/gather_scatter_ops.py:423). */
int gcb_gather_rows(const float* src, int32_t ld_src, const int32_t* idx, int64_t n, float* dst,
                    int32_t ld_dst, int32_t width, void* stream);

/* Same (reference analogue: utils/gather_scatter_ops.py:423 all_gather before a sharded gather, and
 * its shard-local fast path :102-144) for a latent stream that exists only as an operand image of a
 * [*, 512] matrix.  A packed row is
 * 2048 bytes (per 8-column piece the image's 16 bytes of bf16 hi, then its 16 bytes of lo):
 *   pack:   buf[i] = image row idx[i]                 (send side)
 *   unpack: image row first_row + i = buf[i]          (receive side; bit-identical to the owner's) */
int gcb_image_rows_pack(const void* img, const int32_t* idx, int64_t n, void* buf, void* stream);
int gcb_image_rows_unpack(const void* buf, int64_t n, void* img, int64_t first_row, void* stream);

int gcb_abi_version(void);
const char* gcb_last_error(void);

/* Number of resident SMs used for persistent grids on `device` (query helper). */
int gcb_sm_count(int device);

/* Bytes of the packed bf16 weight image for a [k, n] layer (k multiple of 16). */
int64_t gcb_packed_weight_bytes(int32_t k, int32_t n);

/* Host-side packing (pure CPU, no CUDA): fp32 W[k_rows, n_cols] (row-major, ld =
 * n_cols) -> image for a layer of padded shape [k, n]; rows/cols beyond the real
 * ones are zero.  `dst` has gcb_packed_weight_bytes(k, n) bytes. */
int gcb_pack_weight_host(const float* w, int32_t k_rows, int32_t n_cols, int32_t k, int32_t n,
                         void* dst);

/* CTAs per thread-block cluster of the tensor-core layer kernel (1, 2 or 4; default
 * 2).  The CTAs of a cluster process consecutive row tiles in lockstep and receive
 * each weight tile once from L2 through TMA multicast.  Process-wide tuning knob. */
int gcb_set_cluster_size(int32_t ctas);

/* Launch one fused layer. */
int gcb_layer_forward(const gcb_layer_desc* d, void* stream);

/* out[i, :] = sum_{e in [row_ptr[i], row_ptr[i+1])} msg[e, :]   (width 512).
 * Deterministic receiver-sorted segmented sum; replaces jraph.segment_sum as
 * called from _node_update (utils/typed_graph_net.py:532-538). */
int gcb_segment_sum(const float* msg, int32_t ld_msg, const int32_t* row_ptr, int32_t num_nodes,
                    float* out, int32_t ld_out, int32_t width, void* stream);

/* Same, with the receivers of more than 256 in-edges listed in `heavy` (node ids, host-computed
 * from row_ptr): those are summed by one thread block each instead of one warp (the mesh
 * nodes next to the poles receive thousands of grid points).  Deterministic. */
int gcb_segment_sum_heavy(const float* msg, int32_t ld_msg, const int32_t* row_ptr,
                          int32_t num_nodes, const int32_t* heavy, int32_t num_heavy, float* out,
                          int32_t ld_out, int32_t width, void* stream);

/* Channel packing, device side.  planes: [n_ch, n_nodes] (channel-major, i.e. the
 * (batch-sliced) variables stacked in dataset_to_stacked order);  feats:
 * [n_nodes, ld] with columns [0,n_ch) = (planes - mean) / scale (mean/scale per
 * channel, NULL = identity), columns [n_ch, n_ch+n_static) = node_static, and
 * zero padding up to ld.  Replaces _inputs_to_grid_node_features
 * (weathernext1_graph/graphcast.py:680-699), the structural-feature concat of
 * _run_grid2mesh_gnn (:561-568) and normalization.normalize
 * (utils/normalization.py:29-48). */
int gcb_pack_grid_features(const float* planes, int32_t n_ch, int64_t n_nodes,
                           const float* mean, const float* scale,
                           const float* node_static, int32_t n_static,
                           float* feats, int32_t ld, void* stream);

/* Same packing, delivered directly as the operand image of the [n_nodes, k] feature matrix
 * (k = padded channel count, multiple of 16, >= n_ch + n_static): what gcb_forward consumes. */
int gcb_pack_grid_image(const float* planes, int32_t n_ch, int64_t n_nodes, const float* mean,
                        const float* scale, const float* node_static, int32_t n_static,
                        int32_t k, void* img, void* stream);

/* Inverse for the outputs: y [n_nodes, ld_y] -> planes_out [n_out, n_nodes] with
 *   planes_out[c] = y[:, c] * scale[c] + offset[c] + (add_plane_index[c] >= 0 ?
 *                   add_planes[add_plane_index[c]] : 0).
 * Replaces _grid_node_outputs_to_prediction (graphcast.py:701-723) and
 * InputsAndResiduals._unnormalize_prediction_and_add_input
 * (utils/normalization.py:113-132).  scale/offset/add_* may be NULL. */
int gcb_unpack_grid_outputs(const float* y, int32_t ld_y, int32_t n_out, int64_t n_nodes,
                            const float* scale, const float* offset,
                            const float* add_planes, const int32_t* add_plane_index,
                            float* planes_out, void* stream);

/* ---- fused layer chains ---------------------------------------------------------------
 * A CHAIN runs up to GCB_MAX_CHAIN fused layers over the same `rows` rows in ONE kernel: a
 * cluster pair owns a 128-row tile and takes it through layer 0, 1, ... while the intermediate
 * results stay on chip -- each layer that later layers consume writes its result (as an
 * operand image) into a small per-cluster SCRATCH ring that lives in the 126 MB L2 and is
 * streamed back by TMA as the A operand of the consumer; it is overwritten in place tile after
 * tile, so it never has to reach HBM.  This is how the two linears of every MLP of
 * build_mlp_with_maybe_layer_norm (utils/legacy/deep_typed_graph_net.py:205-247) execute as one
 * launch with the [rows, 512] hidden activation never written to HBM.
 * All layers of a chain have n = n_valid = 512.  Layer results are bit-identical to running the
 * same layers one by one through gcb_layer_forward. */
#define GCB_MAX_CHAIN 6

typedef struct {
  int32_t nseg;             /* 1..3 */
  gcb_segment seg[3];       /* as in gcb_layer_desc; ignored when seg_from[s] >= 0 (set k only) */
  int32_t seg_from[3];      /* -1: external segment (table / img);  j >= 0: the result of layer j
                             * (j < this layer, which must have keep = 1), k = 512 */
  const void* w_packed; const float* bias;      /* bias may be NULL (= 0) */
  const float* ln_scale; const float* ln_offset;
  int32_t act;              /* gcb_activation; SWISH and LayerNorm are mutually exclusive here */
  int32_t keep;             /* 1: later layers of the chain consume this layer's result */
  const float* residual; int32_t ld_res;
  /* Alternative: the residual given as an operand image (x = hi + lo, two bf16: 2^-17 relative)
   * of the [rows, 512] stream -- typically the SAME buffer as out_img (updated in place) and as a
   * segment of an earlier layer, so that a latent has ONE representation in HBM instead of an
   * fp32 master plus an image.  Excludes `residual` and `out`; LayerNorm layers only. */
  const void* residual_img;
  /* Or the kept result of an earlier layer of this chain: 0 = none, j + 1 = layer j (keep = 1).
   * Excludes residual / residual_img / out.  (vg1 = vg0 + MLP(vg0) with vg0 never leaving the chip.) */
  int32_t residual_keep;
  float* out;   int32_t ld_out;      /* residual + y, fp32 (optional) */
  float* out_y; int32_t ld_out_y;    /* y alone, fp32 (optional) */
  void* out_img;                     /* residual + y as an operand image (optional) */
  int32_t n_pre_add; gcb_pre_add pre_add[2];
} gcb_chain_layer;

typedef struct {
  int32_t rows;
  int32_t nlayers;          /* 1..GCB_MAX_CHAIN */
  int32_t precision;        /* GCB_PREC_BF16X3 or GCB_PREC_BF16 */
  int32_t lag;              /* tiles a layer runs ahead of the next one (1 or 2; 0 = default 1) */
  int32_t order;            /* unit order inside a pipeline step: 0 = layer 0 first; 1 = last layer
                             * first (one scratch slot less per ring; for chains of >= 3 layers) */
  int32_t pad_;
  void* scratch;            /* gcb_chain_scratch_bytes() bytes, 16-byte aligned */
  int64_t scratch_bytes;    /* size of `scratch` (checked against what this chain needs) */
  gcb_chain_layer layer[GCB_MAX_CHAIN];
} gcb_chain_desc;

/* Scratch bytes a chain launch needs on `device` (depends on the resident cluster count). */
int64_t gcb_chain_scratch_bytes(int32_t device, int32_t n_keep_layers, int32_t lag,
                                int32_t max_distance);
int gcb_chain_forward(const gcb_chain_desc* d, void* stream);

/* Top-of-atmosphere incident solar radiation on a lat / lon grid, integrated over a period ending
 * at each timestamp (replaces solar_radiation.get_toa_incident_solar_radiation,
 * weathernext/utils/solar_radiation.py:443-521; the forcing GraphCast needs at every target time).
 *   table   [n_times, bins, 5] (device): per integration bin cos / sin of the solar declination,
 *           cos / sin of the hour angle at longitude 0, and weight * TSI / d_au^2 * dx - host-side
 *           scalars, see graphcast_b200/forcings.py
 *   sin_lat, cos_lat [n_lat]; cos_lon, sin_lon [n_lon] (device)
 *   out     [n_times, n_lat, n_lon] float32, J/m^2. */
int gcb_toa_incident_solar_radiation(const float* table, int32_t n_times, int32_t bins,
                                     const float* sin_lat, const float* cos_lat,
                                     const float* cos_lon, const float* sin_lon, int32_t n_lat,
                                     int32_t n_lon, float* out, void* stream);

/* ---- whole-step orchestration -------------------------------------------------- */

/* One two-layer MLP (+ optional LayerNorm) of the model. */
typedef struct {
  const void* w0_packed; const float* w0_f32; const float* b0;   /* [k0, 512] */
  const void* w1_packed; const float* w1_f32; const float* b1;   /* [512, n1] */
  const float* ln_scale; const float* ln_offset;                 /* [n1] or NULL */
  int32_t k0;            /* padded K of layer 0 (sum of its segments) */
  int32_t n1;            /* padded output width (256 or 512) */
  int32_t n1_valid;
} gcb_mlp;

/* Row blocks of a [1536,512] first edge-MLP layer, each packed as its own [512,512] layer. */
typedef struct {
  const void* we_packed; const float* we_f32;
  const void* ws_packed; const float* ws_f32;
  const void* wr_packed; const float* wr_f32;
} gcb_mlp_split;

#define GCB_MAX_MSG_STEPS 64

/* Everything one forward step needs.  Edge arrays are in EXECUTION order
 * (receiver-sorted for grid2mesh and mesh; the reference's own order for
 * mesh2grid, which is receiver-sorted with fan-in 3). */
typedef struct {
  int32_t num_grid, num_mesh;
  int32_t e_g2m, e_mesh, e_m2g;
  int32_t c_in_pad;       /* padded width of the packed input features (mult. of 16) */
  int32_t c_in_valid;     /* real width incl. the 3 structural features (mult. of 4 pad ok) */
  int32_t msg_steps;
  int32_t precision;
  int32_t pregather;      /* 1: split first edge-MLP layers (needs the *_split weights + proj_*) */

  /* static graph */
  const int32_t* g2m_snd; const int32_t* g2m_rcv; const int32_t* g2m_row_ptr;
  const float*   g2m_feat;   /* [e_g2m, 4] */
  const int32_t* g2m_heavy; int32_t n_g2m_heavy;   /* receivers with > 256 in-edges */
  const int32_t* mesh_snd; const int32_t* mesh_rcv; const int32_t* mesh_row_ptr;
  const float*   mesh_feat;  /* [e_mesh, 4] */
  const int32_t* m2g_snd; const int32_t* m2g_rcv;
  const float*   m2g_feat;   /* [e_m2g, 4] */
  const float*   mesh_in;    /* [num_mesh, c_in_pad]: zeros + structural (graphcast.py:573-583) */

  /* weights */
  gcb_mlp enc_grid, enc_mesh, enc_e_g2m, proc_e_g2m, proc_n_mesh_g2m, proc_n_grid_g2m;
  gcb_mlp enc_e_mesh;
  gcb_mlp proc_e_mesh[GCB_MAX_MSG_STEPS];
  gcb_mlp proc_n_mesh[GCB_MAX_MSG_STEPS];
  gcb_mlp enc_e_m2g, proc_e_m2g, proc_n_grid_m2g, dec_grid;

  /* pregather only: first-layer weights of the four edge-MLP families split by rows
   * into edge / sender / receiver blocks ([512,512] each; b0 stays in the MLP). */
  gcb_mlp_split proc_e_g2m_split, proc_e_m2g_split;
  gcb_mlp_split proc_e_mesh_split[GCB_MAX_MSG_STEPS];
  const float* zero_bias;   /* [512] zeros */
  float* proj_grid;         /* [num_grid, 512] */
  float* proj_mesh_a;       /* [num_mesh, 512] */
  float* proj_mesh_b;       /* [num_mesh, 512] */

  /* workspace: fp32 masters (residual streams, gather tables, messages) and operand
   * images (gcb_a_image_bytes) of everything that is consumed as an identity-row A
   * operand -- those are streamed by TMA. */
  void* hidden;         /* image [max_rows, 512]: hidden activations of the current MLP */
  void* edge_a_img;     /* image [max(e_g2m,e_m2g), 512]: embedded bipartite edge latents */
  float* edge_b;        /* [max(e_g2m,e_m2g), 512] bipartite messages */
  const void* mesh_in_img;  /* image [num_mesh, c_in_pad] of mesh_in (static) */
  float* grid_lat;  void* grid_lat_img;    /* [num_grid, 512] latent grid nodes */
  float* mesh_lat;  void* mesh_lat_img;    /* [num_mesh, 512] latent mesh nodes */
  float* mesh_agg;  void* mesh_agg_img;    /* [num_mesh, 512] segment sums */
  float* mesh_edge; void* mesh_edge_img;   /* [e_mesh, 512] latent mesh edges */
  float* mesh_msg;      /* [e_mesh, 512] */
  void* grid_agg_img;   /* image [num_grid, 512]: summed mesh2grid messages */

  /* Fused execution: 1 = every MLP (both linears, activation, LayerNorm, residual) is ONE
   * gcb_chain_forward launch and its hidden activation never reaches HBM (needs chain_scratch;
   * tensor-core precisions only -- the FP32_SIMT validation arm always runs layer by layer).
   * 0 = one launch per linear through `hidden` (the round-1 path, kept as the reference the
   * fused path must reproduce bit for bit). */
  int32_t fuse;
  int32_t chain_lag;        /* gcb_chain_desc.lag for those launches (0 = default) */
  /* Node-partitioned execution (one rank of BASELINE config 4): the local node tables hold
   * [owned rows | halo rows]; node updates, aggregation and the decoder cover the owned rows
   * only, gathers and sender projections all local rows.  0 = every row is owned. */
  int32_t num_grid_owned;
  int32_t num_mesh_owned;
  void* chain_scratch;      /* chain_scratch_bytes >= gcb_chain_scratch_bytes(device, 3, lag, 2) */
  /* 1 (needs fuse, pregather and a tensor-core precision): the latent streams grid_lat, mesh_lat
   * and mesh_edge live in HBM ONLY as operand images; the residual of every update is read back
   * from the image (x = hi + lo, two bf16: 2^-17 relative per update, cf. the 2^-17 operand split
   * of the BF16X3 products) and the fp32 masters are neither written nor read.  Halves the HBM
   * bytes of every residual update.  0 = fp32 masters next to the images (round-1 layout). */
  int32_t image_residual;
  /* 1 (with image_residual, one GPU): compose the step from chains of up to four layers --
   * [edge embedder MLP -> edge MLP], [node MLP -> projections of the next edge MLP] -- so that the
   * embedded edge latents and the inputs of the projections never reach HBM (needs proj_grid_b). */
  int32_t deep_chains;
  float* proj_grid_b;       /* [num_grid, 512]: receiver projection of the mesh2grid edge MLP */
  int64_t chain_scratch_bytes;
} gcb_model;

/* Stage-wise execution of the same step: gcb_forward == ENCODE, PROCESS_EMBED, PROCESS_STEP for
 * step = 0..msg_steps-1, DECODE, in this order on one stream.  Used by the stage-wise parity
 * tests and by the node-partitioned processor, which exchanges halo rows of mesh_lat between
 * PROCESS_STEP calls (reference analogue: the all_gather / psum_scatter pair around every
 * sharded gather / segment sum, utils/gather_scatter_ops.py:278,423).
 *   ENCODE         grid2mesh GNN (graphcast.py:550-604): reads grid_in_img; leaves grid_lat = vg1,
 *                  mesh_lat = vm1 (fp32 + images)
 *   PROCESS_EMBED  mesh edge embedding (deep_typed_graph_net.py:250-271 for the mesh GNN)
 *   PROCESS_STEP   one InteractionNetwork step + residuals (deep_typed_graph_net.py:372-393)
 *   DECODE         mesh2grid GNN + output MLP (graphcast.py:641-678): writes grid_out */
typedef enum {
  GCB_STAGE_ENCODE = 0, GCB_STAGE_PROCESS_EMBED = 1, GCB_STAGE_PROCESS_STEP = 2, GCB_STAGE_DECODE = 3
} gcb_stage;
int gcb_forward_stage(const gcb_model* m, int32_t stage, int32_t step, const void* grid_in_img,
                      float* grid_out, void* stream, int32_t* launches);

/* One 6 h step for one batch element:
 *   grid_in_img  operand image of [num_grid, c_in_pad]  (from gcb_pack_grid_image)
 *   grid_out [num_grid, 256]       (columns [0, n_out) valid)
 * Replaces GraphCast.__call__'s _run_grid2mesh_gnn / _run_mesh_gnn /
 * _run_mesh2grid_gnn (weathernext1_graph/graphcast.py:309-323, 550-678) and the
 * DeepTypedGraphNet / InteractionNetwork machinery under them
 * (utils/legacy/deep_typed_graph_net.py:180-401, utils/typed_graph_net.py:272-546).
 * `launches` (host pointer, may be NULL) receives the number of kernels launched. */
int gcb_forward(const gcb_model* m, const void* grid_in_img, float* grid_out, void* stream,
                int32_t* launches);

/* gcb_forward replays a CUDA graph of its launch sequence from the third call with the same
 * (model contents, buffers, stream) on: the first call runs the launches directly, the second
 * captures them.  Needs a non-legacy stream (a NULL / legacy / per-thread default stream, an
 * active gcb_profile_begin, or a caller that is itself capturing all fall back to direct
 * launches).  Not thread-safe.  enabled = 0 disables replay and drops the recorded graphs. */
int gcb_set_graph_replay(int32_t enabled);

/* Per-launch profiling.  Between gcb_profile_begin() and gcb_profile_end() every
 * kernel launched through this ABI is bracketed by CUDA events on its stream.
 * gcb_profile_end synchronises them and returns, per launch (in launch order,
 * at most `capacity` entries; *count = total launches): its kind, duration in ms,
 * and its ALGORITHMIC flops / HBM bytes (layer / chain: 2*rows*K*n flops per layer; inputs
 * incl. gathers + weights + outputs bytes, results handed over inside a chain excluded.
 * segment sum inside gcb_forward: message rows read + node rows written; through the public
 * gcb_segment_sum* entry points only the output bytes -- the caller adds edges*width*4).
 * Not thread safe. */
typedef enum {
  GCB_KIND_LAYER_TC = 0, GCB_KIND_SEGMENT_SUM = 1, GCB_KIND_PACK = 2, GCB_KIND_UNPACK = 3,
  GCB_KIND_LAYER_SIMT = 4, GCB_KIND_ROWS_TO_IMAGE = 5, GCB_KIND_CHAIN_TC = 6, GCB_KIND_GATHER = 7
} gcb_kernel_kind;
int gcb_profile_begin(void);
int gcb_profile_end(int32_t capacity, int32_t* kinds, float* ms, double* flops, double* bytes,
                    int32_t* count);

/* Debug: timeline trace of CTA 0 of the tensor-core layer kernel.  `device_buffer`
 * (64 tiles x 8 events of int64 clock64 values; NULL disables) receives, per tile:
 * [0] MMA: accumulator free  [1] MMA: first operands landed  [2] MMA: last commit issued
 * [3] epilogue: accumulator ready  [4] epilogue: LayerNorm statistics done
 * [5] epilogue: tile stored. */
int gcb_debug_trace(long long* device_buffer);

/* Debug only: experiment switches of the tensor-core kernel for performance attribution
 * (0 = production behaviour).  2: skip all global stores of the epilogue (results are NOT
 * produced); 4: N-split pairs stream the whole A block per CTA instead of multicasting halves
 * (same results); 16: L2-prefetch the A blocks of the next tile (same results). */
int gcb_debug_flags(int flags);

/* Device self-test of the tensor-core layer against the FP32_SIMT arm on random
 * data (used by tests and __graft_entry__.smoke); returns max |diff| / max |ref|
 * through *rel_err.  Allocates its own scratch. */
int gcb_selftest_layer(int32_t rows, int32_t k, int32_t n, int32_t precision, float* rel_err);

#ifdef __cplusplus
}
#endif
#endif /* GRAPHCAST_B200_H_ */
