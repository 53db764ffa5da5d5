/*
 * hbr.h -- C ABI of libhbr_b200.so: the B200 (sm_100a) implementation of the NeRF hot path of
 * RishabhSri14/Human-Body-Reconstruction.
 *
 * The reference is pure Python; the binding a maintainer adds on the reference side is a ctypes
 * stub (see INTEGRATION.md).  Every entry point replaces one reference interface, cited as
 * file:line into the reference tree.  Conventions:
 *   - plain C: raw pointers + sizes, no torch / C++ types in any signature;
 *   - pointers are DEVICE pointers unless the parameter name ends in _host; the library never
 *     allocates, frees or synchronises: callers own every buffer (PyTorch caching allocator) and
 *     pass the stream (cudaStream_t as void*) the work is enqueued on;
 *   - return 0 on success, a negative hbr_status otherwise; hbr_last_error() gives the message
 *     (thread local).  Nothing throws, nothing exits.  There is no CPU fallback: calling without a
 *     CUDA device returns HBR_ERR_CUDA;
 *   - entry points are re-entrant and stateless (safe on different devices/streams concurrently).
 */
#ifndef HBR_B200_H_
#define HBR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HBR_ABI_VERSION 2
#define HBR_MAX_LEVELS 32

typedef enum {
  HBR_OK = 0,
  HBR_ERR_ARG = -1,       /* bad argument (shape, alignment, unsupported configuration) */
  HBR_ERR_CUDA = -2,      /* CUDA runtime error (message holds cudaGetErrorString) */
  HBR_ERR_UNSUPPORTED = -3
} hbr_status;

typedef enum { HBR_F32 = 0, HBR_F16 = 1, HBR_U8 = 2, HBR_BF16 = 3 } hbr_dtype;

/* Geometry of a HashEncoder instance: hash_encoding.py:6-39.
 * scale[l] = N_min * b**l is computed by the HOST with the reference's torch expression
 * (hash_encoding.py:13,153) and handed over; the kernels never recompute it (SURVEY Q1/Q2). */
typedef struct {
  float mu[3];                    /* bbox minimum, hash_encoding.py:21 / train_hash2.py:117 */
  float sigma;                    /* bbox diagonal (scalar), hash_encoding.py:20 / train_hash2.py:119 */
  int32_t L;                      /* levels */
  int32_t F;                      /* features per entry: 1, 2 or 4 */
  int32_t E;                      /* extra zero columns appended to the output, hash_encoding.py:148 */
  uint32_t T;                     /* entries per level (any T; power-of-two takes the uint32 fast path) */
  float scale[HBR_MAX_LEVELS];
} hbr_hash_geom;

/* Shape of MLP_3D(num_sig=2, num_col=2, h_size=64): test_hash.py:21-51.
 * Parameters live in ONE flat fp32 buffer in state_dict order:
 *   sig_model.0.{weight(64,in0),bias(64)} sig_model.2.{(64,64),(64)} sig_model.4.{(16,64),(16)}
 *   col_model.0.{(64,15+d_view),(64)}     col_model.2.{(64,64),(64)} col_model.4.{(3,64),(3)}      */
typedef struct {
  int32_t in0;                    /* L*F+E, <= 64 */
  int32_t d_view;                 /* direction-encoding width, 15+d_view <= 64 */
} hbr_mlp_dims;

int hbr_abi_version(void);
const char* hbr_last_error(void);
/* number of floats in the flat MLP parameter buffer for these dims */
int64_t hbr_mlp_param_count(const hbr_mlp_dims* dims);
/* floats per point of the activation / pre-activation-gradient scratch used by the fp32 MLP */
int64_t hbr_mlp_act_floats(void);

/* ---- a2/a3/a4: HashEncoder.forward, hash_encoding.py:146-170 ------------------------------------
 * x: (n,3) row-major, fp32 or fp16 (nerf2mesh.py:40 feeds fp16).  table: (L,T,F) fp32.
 * y: n rows of L*F+E floats, row pitch y_stride floats. */
int hbr_hash_encode_fwd(const void* x, int x_dtype, int64_t n, const float* table,
                        const hbr_hash_geom* geom_host, float* y, int64_t y_stride, void* stream);

/* a5: autograd of the above (16 x embedding_dense_backward): dtable[l,h,:] += w * dy[:, lF:(l+1)F].
 * dtable (L,T,F) fp32 is ACCUMULATED into (caller zeroes it).  Only levels [level_begin, level_end) are processed,
 * so a caller can split the pass into level chunks and overlap the all-reduce of a finished chunk (multi-GPU). */
int hbr_hash_encode_bwd(const void* x, int x_dtype, int64_t n, const float* dy, int64_t dy_stride,
                        const hbr_hash_geom* geom_host, float* dtable, int level_begin, int level_end, void* stream);

/* Gradient with respect to the POSITIONS (the reference detaches the interpolation weights and has none):
 * dx (n,3) fp32 is OVERWRITTEN with dL/dx = sum_l (s_l/sigma) dL/du_l, the trilinear weights differentiated at the cells
 * and fracs of the forward (truncation toward zero: d frac / du = 1).  dy: rows of dy_stride floats, the first L*F
 * columns used (the E aux columns are ignored).  x fp32 or fp16.  Deterministic: no atomics. */
int hbr_hash_encode_dx(const void* x, int x_dtype, int64_t n, const float* table, const hbr_hash_geom* geom_host,
                       const float* dy, int64_t dy_stride, float* dx, void* stream);

/* a2/a5/a9 for the training step: the same two kernels with the sample positions formed inside from the rays --
 * point (r, s) = rays_o[r] + rays_d[r] * t[r * t_ray_stride + s], multiply and add rounded separately exactly like
 * hbr_ray_points (vol_renderer.py:165, helper.py:48) -- so the (R*S,3) position tensor is never written or read.
 * t is (S) shared (t_ray_stride = 0) or (R,S) per ray (t_ray_stride >= S).  The forward writes y (R*S, y_stride) as
 * y_dtype = HBR_F32 or, for the autocast path (train_hash2.py:218), already rounded to the MLP's 16-bit operand
 * format (HBR_F16 | HBR_BF16: y_stride even, y 4-byte aligned) -- the rounding the MLP's first Linear applies to its
 * input under autocast -- which halves the feature traffic and lets hbr_mlp_*_tc skip its conversion pass. */
int hbr_hash_encode_fwd_rays(const float* rays_o, const float* rays_d, const float* t, int64_t t_ray_stride, int64_t R,
                             int64_t S, const float* table, const hbr_hash_geom* geom_host, void* y, int64_t y_stride,
                             int y_dtype, void* stream);
int hbr_hash_encode_bwd_rays(const float* rays_o, const float* rays_d, const float* t, int64_t t_ray_stride, int64_t R,
                             int64_t S, const float* dy, int64_t dy_stride, const hbr_hash_geom* geom_host, float* dtable,
                             int level_begin, int level_end, void* stream);

/* a5 for the multi-GPU training step (SURVEY 8e): the whole scatter-add in ONE launch that walks `nchunks` level chunks
 * [level_bounds[c], level_bounds[c+1]) (level_bounds[0] = 0, level_bounds[nchunks] = L) in chunk-major CTA order and
 * counts every finished CTA into done[c] (nchunks device words the caller zeroes beforehand; chunk c of dtable is
 * complete when done[c] == ceil(n / 128), the value hbr_hash_bwd_stream_tiles returns).  hbr_allreduce_peer_stream,
 * running beside it on another stream, exchanges chunk c over NVLink while the later chunks are still accumulated. */
int64_t hbr_hash_bwd_stream_tiles(int64_t n);
int hbr_hash_encode_bwd_stream(const void* x, int x_dtype, int64_t n, const float* dy, int64_t dy_stride,
                               const hbr_hash_geom* geom_host, float* dtable, const int* level_bounds, int nchunks,
                               unsigned int* done, void* stream);
int hbr_hash_encode_bwd_rays_stream(const float* rays_o, const float* rays_d, const float* t, int64_t t_ray_stride, int64_t R,
                                    int64_t S, const float* dy, int64_t dy_stride, const hbr_hash_geom* geom_host,
                                    float* dtable, const int* level_bounds, int nchunks, unsigned int* done, void* stream);

/* a5, level-major traversal: dy_lm is (L, n, F) -- hbr_mlp_bwd_tc writes d(features) so with dfeat_stride =
 * HBR_DFEAT_LEVEL_MAJOR -- and a co-resident grid (hbr_hash_bwd_lm_ctas(n) CTAs, 1024 points each, positions kept in
 * registers) walks the levels in order, all CTAs roughly in lockstep, so the table gradient is finished level by level.
 * level_bounds / nchunks / done as for hbr_hash_encode_bwd_stream (chunk c complete when done[c] == hbr_hash_bwd_lm_ctas(n));
 * all three NULL / 0: no counters.  Same arithmetic, run merging and pairing as hbr_hash_encode_bwd; E must be 0. */
int64_t hbr_hash_bwd_lm_ctas(int64_t n);
int hbr_hash_encode_bwd_lm(const void* x, int x_dtype, int64_t n, const float* dy_lm, const hbr_hash_geom* geom_host,
                           float* dtable, const int* level_bounds, int nchunks, unsigned int* done, void* stream);
int hbr_hash_encode_bwd_rays_lm(const float* rays_o, const float* rays_d, const float* t, int64_t t_ray_stride, int64_t R,
                                int64_t S, const float* dy_lm, const hbr_hash_geom* geom_host, float* dtable,
                                const int* level_bounds, int nchunks, unsigned int* done, void* stream);

/* Parity probe: the hash indices hash_encoding.py:161-162 computes (hash_func, :41-55), and the
 * n-linear weights of :142-143.  idx: (L,n,8) int32, w: (L,n,8) fp32 (either may be NULL). */
int hbr_hash_indices(const void* x, int x_dtype, int64_t n, const hbr_hash_geom* geom_host,
                     int32_t* idx, float* w, void* stream);

/* ---- a6: PositionalEncoder.forward, encoder.py:25-32 ---------------------------------------------
 * d: (n,dim) -> out (n, dim*2*num_freq) fp32: per component sin(2 d k), k<num_freq, then cos.
 * With x_dtype = HBR_F16 the intermediate products and the result are rounded to fp16 like the
 * reference's fp16 tensor ops (nerf2mesh.py:69-81), then widened. */
int hbr_dir_encode(const void* d, int d_dtype, int64_t n, int dim, int num_freq, float* out, void* stream);

/* ---- a7: MLP_3D.forward / backward in fp32 (CUDA cores), test_hash.py:52-77 ----------------------
 * feat (n,in0) pitch feat_stride; dirs (n_dirs_rows, d_view): row index = point / dir_group, so one
 * row per ray serves its S samples (vol_renderer.py:177-183 repeats it; dir_group = S) -- pass
 * dir_group = 1 for a per-point tensor.  dirs == NULL gives the density-only branch (test_hash.py:77).
 * out (n,4) = [rgb, density]  (or (n,1) density when dirs == NULL).
 * act: optional (hbr_mlp_act_floats(), n) scratch that keeps the activations for the backward pass. */
int hbr_mlp_fwd_f32(const float* feat, int64_t feat_stride, const float* dirs, int64_t dir_group, int64_t n,
                    const float* params, const hbr_mlp_dims* dims, float* out, float* act, void* stream);

/* dout (n,4).  dparams (flat, same layout as params) is ACCUMULATED into.  dfeat (n,in0) and
 * ddirs (n/dir_group, d_view; accumulated with atomics, caller zeroes; may be NULL) are written.
 * act is the buffer hbr_mlp_fwd_f32 filled; dz is scratch of the same size.
 * dirs == NULL: the backward of the density-only forward -- dout is (n), the gradient of the density; only the three layers
 * of the density head are walked and only their parameter gradients accumulated (ddirs must be NULL).  This is the sigma-net
 * pass of SDF mode's eikonal stencil (test_hash.py:78-105: six density-only evaluations per sample). */
int hbr_mlp_bwd_f32(const float* feat, int64_t feat_stride, const float* dirs, int64_t dir_group, int64_t n,
                    const float* params, const hbr_mlp_dims* dims, const float* dout, const float* act,
                    float* dz, float* dfeat, int64_t dfeat_stride, float* ddirs, float* dparams, void* stream);

/* ---- a7 on the tensor cores: 16-bit operands, fp32 accumulation in TMEM (tcgen05) ------------------------
 * Same contract as the fp32 pair; this is what runs under autocast (train_hash2.py:218).  `operand` is the tensor-core
 * operand format: HBR_F16 under torch.autocast(float16) -- the reference trainer's precision -- or HBR_BF16 under
 * torch.autocast(bfloat16).  No activation is kept between the passes: the backward kernel recomputes them in shared
 * memory from feat, takes ELU' / LeakyReLU' from `out` (the (n,4) result of the forward call), and keeps the
 * weight-gradient accumulators in TMEM across all tiles of a persistent CTA.  dfeat / ddirs may be NULL; dparams (flat
 * fp32) and ddirs are ACCUMULATED into.  grad_scale (> 0, a power of two; 1 = off) multiplies dout before it is rounded
 * to the operand format and is divided out of every result: fp16's 5 exponent bits underflow on the gradients of a
 * mean-reduced loss unless the caller scales (the reference's GradScaler, train_hash2.py:156,226) or passes it here. */
/* scratch: optional device buffer of hbr_mlp_tc_scratch_bytes(dims) bytes, 256-byte aligned (NULL = none).  With it a
 * small prep kernel builds the 16-bit operand image once per call and the backward sums per-CTA gradient rows with a
 * reduce kernel; without it every CTA converts the parameters itself and flushes its gradients with atomics. */
int64_t hbr_mlp_tc_scratch_bytes(const hbr_mlp_dims* dims);
/* Builds the operand image of `params` in `scratch` (what hbr_mlp_fwd_tc / _bwd_tc do themselves unless image_ready): lets a
 * caller run it on another stream, beside the hash-grid kernel of the step. */
int hbr_mlp_tc_prepare(const float* params, const hbr_mlp_dims* dims, int operand, void* scratch, void* stream);
/* Sums the per-CTA gradient rows a hbr_mlp_bwd_tc call with defer_reduce != 0 left in `scratch` into dparams (accumulating):
 * the second half of that call, for callers that want it on another stream beside the hash-grid backward. */
int hbr_mlp_tc_reduce_grads(const hbr_mlp_dims* dims, int64_t n, void* scratch, float* dparams, void* stream);
/* image_ready != 0: the operand image in `scratch` was built by an earlier call for these very parameters and operand
 * format (the forward call of the same step): skip the prep kernel.
 * n_dev / dir_rows (both may be NULL): compacted sample lists (hbr_compact_samples): at most n points, the live count is
 * read from *n_dev on the device; point p uses direction row dir_rows[p] instead of p / dir_group. */
/* feat_dtype: HBR_F32 (n, feat_stride) fp32 features, or the operand format itself -- features already rounded to it by
 * hbr_hash_encode_fwd_rays (contiguous rows of in0 16-bit values; in0 must be 32, or 64 for the wide shape): the kernels
 * then copy the rows straight into their operand tile. */
int hbr_mlp_fwd_tc(const void* feat, int feat_dtype, int64_t feat_stride, const float* dirs, int64_t dir_group, int64_t n,
                   const float* params, const hbr_mlp_dims* dims, int operand, float* out, void* scratch, int image_ready,
                   const unsigned long long* n_dev, const int32_t* dir_rows, void* stream);
/* dfeat_stride == HBR_DFEAT_LEVEL_MAJOR: dfeat is written as (in0/2 levels, n, 2) instead of (n, in0) -- the layout
 * hbr_hash_encode_bwd*_lm reads level by level with coalesced loads (in0 = 32, even n, 16-byte aligned, n_dev NULL). */
#define HBR_DFEAT_LEVEL_MAJOR (-1)
int hbr_mlp_bwd_tc(const void* feat, int feat_dtype, int64_t feat_stride, const float* dirs, int64_t dir_group, int64_t n,
                   const float* params, const hbr_mlp_dims* dims, int operand, const float* out, const float* dout,
                   float* dfeat, int64_t dfeat_stride, float* ddirs, float* dparams, float grad_scale, void* scratch,
                   int image_ready, int defer_reduce, const unsigned long long* n_dev, const int32_t* dir_rows, void* stream);
/* ---- a2 + a7 fused (the training step's field evaluation under autocast): hash-grid encoder + MLP_3D in ONE kernel per
 * direction -- HashEncoder.forward (hash_encoding.py:146-170) feeding MLP_3D.forward (test_hash.py:52-72) as
 * vol_renderer.py:179,211 chains them.  Covers the reference's configuration family F = 2, L = 16, E = 0, power-of-two T,
 * d_view <= 25; anything else uses the separate entry points.  x (n,3) fp32 sample positions.  The forward writes the
 * 16-bit features (operand format) it fed to the tensor cores to feat16 (n,32) for the backward recompute; the backward scatter-adds
 * d(features) into dtable (L,T,2) straight from the accumulator.  dparams / dtable / ddirs are ACCUMULATED into. */
int hbr_field_fwd_tc(const float* x, int64_t n, const float* table, const hbr_hash_geom* geom_host, const float* dirs,
                     int64_t dir_group, const float* params, const hbr_mlp_dims* dims, int operand, float* out,
                     void* feat16, void* scratch, void* stream);
int hbr_field_bwd_tc(const float* x, int64_t n, const hbr_hash_geom* geom_host, const float* dirs, int64_t dir_group,
                     const float* params, const hbr_mlp_dims* dims, int operand, const void* feat16, const float* out,
                     const float* dout, float* dtable, float* ddirs, float* dparams, float grad_scale, void* scratch,
                     void* stream);
/* a2 + a7 + a9 for the training step's forward in ONE kernel: what hbr_hash_encode_fwd_rays followed by hbr_mlp_fwd_tc
 * computes (same arithmetic), with the gather on dedicated warps of the tensor-core kernel feeding its tile groups through
 * shared memory -- no fp32 features, the layer chain hidden behind the gather.  Same configuration family as
 * hbr_field_fwd_tc.  out (R*S,4) = [rgb, sigma]; feat16 (R*S,32) 16-bit features (operand format) for the backward. */
int hbr_field_fwd_rays_tc(const float* rays_o, const float* rays_d, const float* t, int64_t t_ray_stride, int64_t R, int64_t S,
                          const float* table, const hbr_hash_geom* geom_host, const float* dirs, const float* params,
                          const hbr_mlp_dims* dims, int operand, float* out, void* feat16, void* scratch, int image_ready,
                          void* stream);
/* ---- a7 backward + a5 in one kernel (the training step's backward under autocast): what hbr_mlp_bwd_tc followed by
 * hbr_hash_encode_bwd_rays computes -- the autograd of MLP_3D.forward (test_hash.py:52-72) chained into the autograd of
 * HashEncoder.forward (hash_encoding.py:146-170; 16 x embedding_dense_backward) for the sample positions o + d t of
 * vol_renderer.py:165 -- with the scatter-add running on dedicated warps of the MLP kernel, tile by tile, beside the layer
 * chains of the following tiles: no fp32 d(feature) tensor, and the two phases overlap on every SM.  Same configuration
 * family as hbr_field_*_tc.  feat16 (R*S,32): the 16-bit features hbr_hash_encode_fwd_rays wrote (operand format).
 * t: (S) shared (t_ray_stride = 0) or (R,S).  dirs (R,d_view).  dtable (L,T,2) / dparams / ddirs are ACCUMULATED into.
 * scratch / image_ready / defer_reduce as in hbr_mlp_bwd_tc. */
int hbr_field_bwd_rays_tc(const void* feat16, const float* rays_o, const float* rays_d, const float* t, int64_t t_ray_stride,
                          int64_t R, int64_t S, const hbr_hash_geom* geom_host, const float* dirs, const float* params,
                          const hbr_mlp_dims* dims, int operand, const float* out, const float* dout, float* dtable,
                          float* ddirs, float* dparams, float grad_scale, void* scratch, int image_ready, int defer_reduce,
                          void* stream);
/* ---- a8: strat_sampler, helper.py:231-232: t[s] = lin[s] + (u[s] * span) / count with span = tf - tn, count = num_samples,
 * each operation rounded on its own (bit-identical to the reference's three elementwise ops).  lin = torch.linspace(tn, tf, S)
 * and u = torch.rand_like(lin) are produced by the caller (same RNG stream, Q9). */
int hbr_strat_depths(const float* lin, const float* u, float span, float count, int64_t S, float* t, void* stream);

/* The loss of train_hash2.py:177,221 -- scale * (nn.MSELoss (mean) of a against gt, plus that of b when b != NULL) -- as one
 * kernel per direction (scale = 2 with b == NULL serves the non-hierarchical step, where the trainer adds the same MSE
 * twice).  loss (1 float) must be zero on entry and is accumulated into; gout is the scalar upstream gradient on the
 * device; da / db receive gout * scale * 2 (x - gt) / n.  n = number of elements of each tensor. */
int hbr_mse_pair_fwd(const float* a, const float* b, const float* gt, int64_t n, float scale, float* loss, void* stream);
int hbr_mse_pair_bwd(const float* a, const float* b, const float* gt, int64_t n, float scale, const float* gout, float* da,
                     float* db, void* stream);

/* ---- a9: sample positions, vol_renderer.py:165 / helper.py:48 -------------------------------------
 * pts[r,s,:] = o[r,:] + d[r,:]*t  (separate multiply and add).  t is (S) shared (t_ray_stride = 0)
 * or (R,S) per ray (t_ray_stride = S). */
int hbr_ray_points(const float* rays_o, const float* rays_d, const float* t, int64_t t_ray_stride,
                   int64_t R, int64_t S, float* pts, void* stream);

/* a9: Volume_Renderer.get_mask, vol_renderer.py:133-140: mask[p] = grid[((p-mu)/sigma*G).long()],
 * negative cells wrap (Python indexing).  grid: G^3 bytes (torch.bool). */
int hbr_occupancy_mask(const float* pts, int64_t n, const uint8_t* grid, int G, const float* mu3_host,
                       float sigma, uint8_t* mask, void* stream);

/* ---- 8f row 3: the occupancy grid of vol_renderer.py:106-140 as a live empty-space skipper ---------------------------
 * hbr_occupancy_update = Volume_Renderer.update_grid (vol_renderer.py:116-131): cells of grid (G^3 bytes) hit by a point
 * with alpha > 0 are set; if no point hit anything the whole grid is set (the reference's fallback).  flags2: two zeroed
 * 32-bit words of device scratch (left zeroed).
 * hbr_compact_samples: sample positions from the rays (as hbr_ray_points), looked up in the grid (as hbr_occupancy_mask);
 * only the live ones are written: pts_c (<= R*S, 3), ray_c (their ray), rowmap (R*S): sample -> compacted row or -1;
 * *count (zero on entry) receives the number of live samples and is what the consumers read as n_dev.  Each ray's live
 * samples are contiguous and in order; rays appear in arbitrary order. */
int hbr_occupancy_update(const float* pts, int64_t n, const float* alpha, int64_t alpha_stride, uint8_t* grid, int G,
                         const float* mu3_host, float sigma, unsigned int* flags2, void* stream);
int hbr_compact_samples(const float* rays_o, const float* rays_d, const float* t, int64_t t_ray_stride, int64_t R, int64_t S,
                        const uint8_t* grid, int G, const float* mu3_host, float sigma, float* pts_c, int32_t* ray_c,
                        int32_t* rowmap, unsigned long long* count, void* stream);
/* The encoder on a compacted list: x (<= n_max, 3) fp32, live count *n_dev (NULL = n_max); y as hbr_hash_encode_fwd_rays. */
int hbr_hash_encode_fwd_pts(const float* x, int64_t n_max, const unsigned long long* n_dev, const float* table,
                            const hbr_hash_geom* geom_host, void* y, int64_t y_stride, int y_dtype, void* stream);
int hbr_hash_encode_bwd_pts(const float* x, int64_t n_max, const unsigned long long* n_dev, const float* dy, int64_t dy_stride,
                            const hbr_hash_geom* geom_host, float* dtable, int level_begin, int level_end, void* stream);

/* ---- a10: calc_color (NeRF mode), helper.py:53-107, and its backward (SURVEY A.3) ------------------
 * One warp per ray.  rgb/sigma are addressed as rgb[(r*S+s)*rgb_stride + c], sigma[(r*S+s)*sigma_stride]
 * so both the reference's separate (R,S,3)/(R,S) tensors (strides 3,1) and the MLP's packed (R*S,4)
 * output (rgb = out, sigma = out+3, strides 4,4) are accepted.  dir_norm: (R) or NULL (=> scalar).
 * mask: optional (R*S) bytes; masked-out samples contribute sigma = rgb = 0 (vol_renderer.py:213-216).
 * rowmap: optional (R*S) int32 from hbr_compact_samples: sample i reads rgb / sigma (and its gradients are written) at
 * row rowmap[i] of the compacted tensors; rowmap[i] < 0 = skipped sample (as masked out).
 * C (R,3), w (R,S).
 * ert_tau: early ray termination, opt-in (<= 0 = off, the reference's behaviour): once the optical depth accumulated over
 * whole 32-sample chunks exceeds ert_tau, the rest of the ray is skipped (weight 0, gradient 0).  At ert_tau = 104 the
 * skipped transmittances exp(-depth) are exactly 0 in fp32, so results are bit-identical whenever the depth stays above
 * the threshold afterwards (always for sigma >= 0).  Pass the same value to the backward. */
int hbr_composite_fwd(const float* t, int64_t t_ray_stride, const float* rgb, int64_t rgb_stride,
                      const float* sigma, int64_t sigma_stride, const float* dir_norm, float dir_norm_scalar,
                      const uint8_t* mask, const int32_t* rowmap, int64_t R, int64_t S, float* C, float* w, float ert_tau,
                      void* stream);
int hbr_composite_bwd(const float* t, int64_t t_ray_stride, const float* rgb, int64_t rgb_stride,
                      const float* sigma, int64_t sigma_stride, const float* dir_norm, float dir_norm_scalar,
                      const uint8_t* mask, const int32_t* rowmap, int64_t R, int64_t S, const float* gC,
                      float* drgb, int64_t drgb_stride, float* dsigma, int64_t dsigma_stride, float ert_tau,
                      void* stream);
/* The same compositor with per-ray depth and opacity maps, formed in the same pass from the same weights:
 *   depth (R) = sum_s w_s t_s   -- distance along the unit ray direction, in the units of t (p = o + d t with |d| = 1);
 *                                 z-depth is depth / dir_norm.  Not normalised by the opacity, not clamped.
 *   opacity (R) = sum_s w_s     -- w may be negative (LeakyReLU density), so opacity can leave [0, 1] like the weights.
 * Either map may be NULL (not written).  Every input form of hbr_composite_fwd is accepted (shared / per-ray t, dir_norm
 * tensor or scalar, mask, rowmap, ert_tau: skipped chunks contribute 0); C and w are bit-identical to hbr_composite_fwd's.
 * bwd: gD, gA (R) are the gradients of depth and opacity (NULL = 0; gC may be NULL too); the per-sample term of the
 * closed-form backward becomes c_s = gC.rgb_s + gD t_s + gA, d(rgb) = w gC is unchanged.  With gD = gA = 0 the gradients
 * equal hbr_composite_bwd's.  One kernel per call, the colour-only kernels with the map code compiled in. */
int hbr_composite_maps_fwd(const float* t, int64_t t_ray_stride, const float* rgb, int64_t rgb_stride,
                           const float* sigma, int64_t sigma_stride, const float* dir_norm, float dir_norm_scalar,
                           const uint8_t* mask, const int32_t* rowmap, int64_t R, int64_t S, float* C, float* w,
                           float* depth, float* opacity, float ert_tau, void* stream);
int hbr_composite_maps_bwd(const float* t, int64_t t_ray_stride, const float* rgb, int64_t rgb_stride,
                           const float* sigma, int64_t sigma_stride, const float* dir_norm, float dir_norm_scalar,
                           const uint8_t* mask, const int32_t* rowmap, int64_t R, int64_t S, const float* gC,
                           const float* gD, const float* gA, float* drgb, int64_t drgb_stride, float* dsigma,
                           int64_t dsigma_stride, float ert_tau, void* stream);

/* ---- a11: hierarchical_sampling, helper.py:23-51 --------------------------------------------------
 * w (R,S) coarse weights (negatives treated as 0; written back clamped when clamp_in_place != 0,
 * helper.py:36), t (S) coarse depths, u (R,S) uniforms (draw #2), cand (S) candidate depths
 * rand(S)*(tf-tn)+tn (draw #3, helper.py:43).  t_fine (R,2S): sorted merge of t and cand[inds]. */
int hbr_hier_sample(float* w, const float* t, const float* u, const float* cand, int64_t R, int64_t S,
                    int clamp_in_place, float* t_fine, void* stream);

/* ---- 8f row 4: SDF mode (--use_sdf) -----------------------------------------------------------------
 * hbr_composite_sdf_fwd/bwd = the SDF branch of calc_color (helper.py:76-86,102-105): phi = VarModel (helper.py:18-21,
 * b = its sharpness parameter, ONE float on the device), alpha_i = relu(1 - phi(s_{i+1}) / phi(s_i)) (last sample 0),
 * T = exclusive cumprod(1 - alpha), C = sum T alpha rgb.  One warp per ray; rgb / sdf addressed like hbr_composite_fwd
 * ((r*S+s)*stride).  from_density != 0: the sdf column holds the density head's LeakyReLU output d and the SDF value
 * 2*sigmoid(d > 0 ? d : 100 d) - 1 (test_hash.py:59-60 on the recovered pre-activation) is formed in the kernel, the
 * gradient handed back is then with respect to d.  The -10 clamp of helper.py:76 is applied in the kernel (gradient 0).
 * bwd: gw (R,S) optional gradient of the weights; db_ray (R): per-ray partial sums of dL/db (the caller adds them up). */
int hbr_composite_sdf_fwd(const float* rgb, int64_t rgb_stride, const float* sdf, int64_t sdf_stride, int from_density,
                          const float* b, int64_t R, int64_t S, float* C, float* w, void* stream);
int hbr_composite_sdf_bwd(const float* rgb, int64_t rgb_stride, const float* sdf, int64_t sdf_stride, int from_density,
                          const float* b, int64_t R, int64_t S, const float* gC, const float* gw, float* drgb,
                          int64_t drgb_stride, float* dsdf, int64_t dsdf_stride, float* db_ray, void* stream);
/* The eikonal term, MLP_3D.finite_difference_normals_approximator + eikonal_value (test_hash.py:86-105, helper.py:293-297),
 * as a 6-point stencil around ONE encoder + density-head pass instead of six:
 * hbr_sdf_stencil_points: x (n,3) -> pts (6,n,3), slab 2*axis = clamp(x + eps e_axis, lo, hi), slab 2*axis+1 = clamp(x - eps
 * e_axis, lo, hi) (lo / hi = MLP_3D.min_bound / max_bound, host floats);
 * hbr_sdf_eikonal_fwd: dens6 (6,n) = LeakyReLU density-head output at those points -> norm (n) = |0.5 (s+ - s-) / eps| with
 * s = 2 sigmoid(pre-activation) - 1; grads (n,3) optional (the central differences themselves);
 * hbr_sdf_eikonal_bwd: gnorm (n) -> ddens6 (6,n). */
int hbr_sdf_stencil_points(const float* x, int64_t n, float eps, const float* lo3_host, const float* hi3_host, float* pts,
                           void* stream);
int hbr_sdf_eikonal_fwd(const float* dens6, int64_t n, float eps, float* norm, float* grads, void* stream);
int hbr_sdf_eikonal_bwd(const float* dens6, int64_t n, float eps, const float* gnorm, float* ddens6, void* stream);

/* ---- a13: nerf2mesh.py:27-40,69-86 density grid -----------------------------------------------------
 * Grid point p = (i*res + j)*res + k  <->  (x[j], y[i], z[k]) with x,y,z = np.linspace(min,max,res)
 * evaluated in float64 (numpy 1.23 semantics, Nerf.yml:119) and rounded to fp16 (nerf2mesh.py:31-40).
 * hbr_grid_points writes the fp16 positions of flat range [p0, p0+count) as (count,3) halfs. */
int hbr_grid_points(const double* min3_host, const double* max3_host, int res, int64_t p0, int64_t count,
                    void* pts_f16, void* stream);
/* Evaluates the field on [p0, p0+count) in chunks: fp16 positions -> fp32 encoder -> fp32 MLP with the
 * single encoded view direction dir_enc (1, d_view) = PositionalEncoder((0,0,1) fp16) (nerf2mesh.py:69-70,81).
 * out: count rows of 4 floats [rgb, density]; with dir_enc == NULL, count floats (density only).
 * pts_scratch: (chunk,3) halfs, feat_scratch: (chunk, L*F+E) floats.  z-slab / multi-GPU sharding = one
 * [p0, p0+count) range per rank. */
/* field_mode: 0 = automatic -- the density-only query of the reference's shape (dir_enc == NULL, in0 == 32) runs its MLP on
 * the tensor cores at fp32-level accuracy (hbr_mlp_density_tf32x3), everything else on the fp32 CUDA-core kernel;
 * 1 = fp32 CUDA-core kernel always. */
int hbr_grid_density(const double* min3_host, const double* max3_host, int res, int64_t p0, int64_t count,
                     const float* table, const hbr_hash_geom* geom_host, const float* params,
                     const hbr_mlp_dims* dims, const float* dir_enc, float* out, void* pts_scratch,
                     float* feat_scratch, int64_t chunk, int field_mode, void* stream);
/* Density head of MLP_3D (test_hash.py:52-62: sig_model on the (n,32) fp32 features, output 0, LeakyReLU) for n points,
 * as nerf2mesh.py:80-82 evaluates it (no autocast: fp32), on the tensor cores: every fp32 operand split into two TF32
 * parts, three tcgen05.mma.kind::tf32 terms per product, fp32 accumulation -- within 1e-5 of the fp32 CUDA-core kernel.
 * feat: contiguous rows of 32 floats, 16-byte aligned.  out: n floats. */
int hbr_mlp_density_tf32x3(const float* feat, int64_t n, const float* params, const hbr_mlp_dims* dims, float* out,
                           void* stream);

/* ---- a14: marching cubes at iso over density (n0,n1,n2) fp32, inside test d < iso -------------------
 * Cells i in [i_begin, i_end) along axis 0 (slab ownership for multi-GPU).  counts[0] = vertices
 * (grid edges owned by the slab whose end points straddle iso), counts[1] = triangles.  counts is a
 * 2 x uint64 device buffer the caller zeroes. */
int hbr_mc_count(const float* density, int n0, int n1, int n2, float iso, int i_begin, int i_end,
                 unsigned long long* counts, void* stream);
/* Emits welded vertices (grid-index coordinates, axis order 0,1,2) and triangles.  edge_id is a
 * (3, n0, n1, n2) int32 scratch.  cursors: 2 x uint64 device counters the caller zeroes. verts has
 * room for max_verts x 3 floats, faces for max_faces x 3 int32. */
int hbr_mc_emit(const float* density, int n0, int n1, int n2, float iso, int i_begin, int i_end,
                int32_t* edge_id, float* verts, int64_t max_verts, int32_t* faces, int64_t max_faces,
                unsigned long long* cursors, void* stream);

/* ---- sparse marching cubes: the res^3 grid above, meshed brick by brick ---------------------------------------------
 * A brick is HBR_MC_BRICK^3 cells; nb = ceil((res-1)/8) bricks per axis, brick b = (bi*nb + bj)*nb + bk holds the cells
 * [8B, min(8B+8, res-1)) per axis and is evaluated on its 9^3 points, indices past res-1 clamped to res-1.  Brick
 * densities are brick-major (n, 9, 9, 9) fp32.  The coarse lattice is the (nb+1)^3 grid points min(8c, res-1), flat index
 * (ci*(nb+1) + cj)*(nb+1) + ck.  Positions are hbr_grid_points' fp16 values and the field is hbr_grid_density's (same
 * field_mode, dir_enc = NULL), so every value equals the dense grid's at the same index.
 * The brick map (nb^3 int32) holds HBR_BRICK_INACTIVE, HBR_BRICK_PENDING (to be evaluated) or the brick's slot >= 0: its
 * row in the caller's brick-density and scratch arrays.  Scans run in tiles of HBR_SCAN_TILE entries; `block_sums` is
 * ceil(n / HBR_SCAN_TILE) + 1 int64. */
#define HBR_MC_BRICK 8
#define HBR_BRICK_INACTIVE (-1)
#define HBR_BRICK_PENDING (-2)
#define HBR_SCAN_TILE 4096
/* pts_scratch: (chunk,3) halfs, feat_scratch: (chunk, L*F+E) floats.  out: (nb+1)^3 floats. */
int hbr_coarse_density(const double* min3_host, const double* max3_host, int res, const float* table,
                       const hbr_hash_geom* geom_host, const float* params, const hbr_mlp_dims* dims, float* out,
                       void* pts_scratch, float* feat_scratch, int64_t chunk, int field_mode, void* stream);
/* out: (n, 9, 9, 9) floats for the bricks listed in bricks (n int32 brick indices). */
int hbr_brick_density(const double* min3_host, const double* max3_host, int res, const int32_t* bricks, int64_t n,
                      const float* table, const hbr_hash_geom* geom_host, const float* params, const hbr_mlp_dims* dims,
                      float* out, void* pts_scratch, float* feat_scratch, int64_t chunk, int field_mode, void* stream);
/* Seed: map[b] = PENDING where the 8 coarse values at brick b's corners are not all on one side of iso, else INACTIVE. */
int hbr_brick_seed(const float* coarse, int nb, float iso, int32_t* map, void* stream);
/* Compaction of the PENDING bricks in brick-index order, by a scan (no atomics).  hbr_brick_pending_count writes the
 * per-tile counts, exclusively scanned, to block_sums and the total to block_sums[ceil(nb^3 / HBR_SCAN_TILE)];
 * hbr_brick_compact then writes list[m] = the m-th pending brick and sets its map entry to the slot base + m. */
int hbr_brick_pending_count(const int32_t* map, int nb, int64_t* block_sums, void* stream);
int hbr_brick_compact(int32_t* map, int nb, const int64_t* block_sums, int32_t base, int32_t* list, void* stream);
/* Closure step over the n bricks just evaluated (list, their densities dens (n,9,9,9)): each of a brick's 6 boundary
 * planes of 9x9 points that is not on the outer grid boundary and holds points on both sides of iso makes the neighbour
 * across it PENDING if it was INACTIVE. */
int hbr_brick_closure(const float* dens, const int32_t* list, int64_t n, int nb, float iso, int32_t* map, void* stream);
/* Marching cubes over the cells of the n bricks in slot order (list[s] = the brick in slot s, dens (n,9,9,9)); every map
 * entry is INACTIVE or a slot.  A crossing grid edge gets one vertex, emitted by the first active brick among those
 * containing it, in the order o, o-e_u, o-e_v, o-e_u-e_v (o = min(p/8, nb-1) of its lower end point p; u < v the other
 * axes, a step back only where p lies on an interior brick plane).
 * hbr_brick_mc_count writes the local vertex id of every (point, axis) of each brick to eid (n, 3, 9, 9, 9) uint16
 * (0xffff: no vertex of this brick) and offsets (n+1, 2) int64: the exclusive scans of the per-brick vertex and triangle
 * counts, totals in row n.  hbr_brick_mc_emit writes vertices (grid-index coordinates along axes 0,1,2, the dense
 * route's arithmetic) and triangles (the dense route's tables and winding): brick s's go to the rows from offsets[s]. */
int hbr_brick_mc_count(const float* dens, const int32_t* list, int64_t n, const int32_t* map, int nb, int res, float iso,
                       uint16_t* eid, int64_t* offsets, int64_t* block_sums, void* stream);
int hbr_brick_mc_emit(const float* dens, const int32_t* list, int64_t n, const int32_t* map, int nb, int res, float iso,
                      const uint16_t* eid, const int64_t* offsets, float* verts, int32_t* faces, void* stream);

/* ---- connected components of a triangle mesh (floater removal after marching cubes) -------------------------------
 * faces (nf, 3) int32 index nv vertices (0 <= nv <= INT32_MAX; indices are NOT range-checked here).  Two vertices are
 * connected when a chain of faces joins them through shared vertices; a vertex no face uses is its own component.
 * label[v] = the smallest vertex index of v's component; face_count[r] / vertex_count[r] = the component's faces (a face
 * belongs to the component of its first vertex) and vertices at its root r (label[r] == r), 0 at every other index.  All
 * three nv-int32 outputs are written in full; the result does not depend on thread order. */
int hbr_mesh_components(const int32_t* faces, int64_t nf, int64_t nv, int32_t* label, int32_t* face_count,
                        int32_t* vertex_count, void* stream);

/* a14: torchmcubes.grid_interp (nerf2mesh.py:99): trilinear samples of vol (C, n0, n1, n2) fp32 at pts (n,3) given as
 * (x, y, z) = (index along axis 2, axis 1, axis 0) in grid-index units (the order torchmcubes returns vertices in),
 * clamped to the volume; out (n, C). */
int hbr_grid_interp(const float* vol, int C, int n0, int n1, int n2, const float* pts, int64_t n, float* out, void* stream);

/* ---- 8f row 1: the optimiser step of train_hash2.py:141-142,227-228 (torch.optim.Adam / AdamW) as ONE pass --------
 * param / grad / exp_avg / exp_avg_sq: n fp32 each (the flat table or MLP buffer).  step >= 1 is the 1-based step count.
 * grad is multiplied by inv_scale (GradScaler unscale, 1.0 without AMP); with found_inf != NULL and *found_inf != 0 the
 * step is skipped (GradScaler's inf check).  decoupled_weight_decay != 0 = AdamW. */
int hbr_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, double lr, double beta1,
                  double beta2, double eps, double weight_decay, int decoupled_weight_decay, int64_t step,
                  double inv_scale, const float* found_inf, void* stream);
/* The same step with every per-step scalar on the device (torch's "capturable" contract), so that the optimiser can be
 * captured in the CUDA graph of the training step and a step GradScaler skips does not advance the bias correction:
 * hbr_adam_tick: *step_dev += 1 unless *found_inf != 0 (once per optimiser step, before the updates);
 * hbr_adam_step_dev: reads the step count and the learning rate from the device; grad is multiplied by
 * inv_scale / *grad_scale_dev (grad_scale_dev may be NULL). */
int hbr_adam_tick(long long* step_dev, const float* found_inf, void* stream);
int hbr_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const float* lr_dev,
                      double beta1, double beta2, double eps, double weight_decay, int decoupled_weight_decay,
                      const long long* step_dev, double inv_scale, const float* grad_scale_dev, const float* found_inf,
                      void* stream);

/* ---- 8f row 2: on-device ray generation, replacing the CPU TensorDataset + DataLoader of train_hash2.py:74-96,211-215 ----
 * get_od (helper.py:176-208) evaluated per requested ray: ray id = view * H*W + row * W + col (the order of the
 * reference's flattened (rays_o, rays_d, dir_norm, gt) dataset); ids from ray_ids (n_rays int64 on the device) or, with
 * ray_ids == NULL, the consecutive range [first, first + n_rays).  c2w: (n_views,4,4) fp32 row-major on the device;
 * fx, fy, cx, cy = K[0,0], K[1,1], K[0,2], K[1,2] converted to float (the reference's K is int64, train_hash2.py:67-72).
 * images (optional, with gt): (n_views,H,W,3) fp32 in [0,1] or uint8 (then gt = u8 / 255 as torchvision's ToTensor).
 * Outputs: rays_o (n,3), unit rays_d (n,3), dir_norm (n,1), gt (n,3).  bad_id (optional device int): set to 1 when an id
 * falls outside [0, n_views*H*W) (that ray is written as zeros). */
int hbr_ray_gen(const float* c2w, int64_t n_views, int H, int W, float fx, float fy, float cx, float cy,
                const int64_t* ray_ids, int64_t first, int64_t n_rays, const void* images, int image_dtype, float* rays_o,
                float* rays_d, float* dir_norm, float* gt, int* bad_id, void* stream);
/* find_bounding_box (helper.py:109-141): bounds[0..2] = min, bounds[3..5] = max over every pixel of every view of
 * o + d*t0 and o + d*t1 (t0 = near, t1 = far + 1.5 in the reference).  The caller initialises bounds to (+1e7 x3, -1e7 x3)
 * like helper.py:121-122. */
int hbr_ray_bbox(const float* c2w, int64_t n_views, int H, int W, float fx, float fy, float cx, float cy, float t0, float t1,
                 float* bounds, void* stream);

/* ---- 8e: the data-parallel step's gradient exchange over NVLink peer memory (csrc/comm.cu) -------------------------
 * The reference has no multi-process path (train_hash2.py:134 wraps only the MLP in nn.DataParallel); this replaces the
 * NCCL all-reduce dist.GradAllReduce would issue on the flat gradient buffer.
 * hbr_peer_alloc: a zero-filled device allocation that other processes of this node can map (plain cudaMalloc, so a
 * CUDA IPC handle addresses it exactly); hbr_peer_export / hbr_peer_import turn it into / open a 64-byte handle that the
 * host side passes between ranks (e.g. torch.distributed.all_gather_object); hbr_peer_release unmaps an imported
 * pointer, hbr_peer_free frees an owned one. */
#define HBR_MAX_PEERS 8
#define HBR_PEER_MAX_CTAS 128
#define HBR_PEER_HANDLE_BYTES 64
#define HBR_PEER_FLAG_BYTES (HBR_PEER_MAX_CTAS * HBR_MAX_PEERS * 4)
int hbr_peer_alloc(void** ptr, int64_t bytes);
int hbr_peer_free(void* ptr);
int hbr_peer_export(void* ptr, unsigned char handle[HBR_PEER_HANDLE_BYTES]);
int hbr_peer_import(const unsigned char handle[HBR_PEER_HANDLE_BYTES], void** ptr);
int hbr_peer_release(void* ptr);
/* In-place all-reduce of n fp32 (n % 4 == 0) over `world` ranks: every rank calls it with bufs[q] / flags[q] = ITS
 * mapping of rank q's buffer and of rank q's HBR_PEER_FLAG_BYTES zero-initialised flag words (bufs[rank] is its own), on
 * the stream that produced its buffer; result = scale * sum over ranks, bit-identical on every rank.  multicast: an NVLS
 * multicast mapping of the same buffers (switch-side reduction) or NULL (plain peer loads/stores).  ctas <= 0 picks the
 * default; the grid never exceeds the SM count (the flag barriers need co-resident CTAs) and must be the same on every
 * rank.  status: optional device word set to 1 if a barrier timed out (10 s) -- the buffer is then undefined. */
int hbr_allreduce_peer(void* const* bufs, void* const* flags, void* multicast, int rank, int world, int64_t n, float scale,
                       int ctas, unsigned int* status, void* stream);

/* The same exchange as ONE launch over a list of pieces [piece_off[i], piece_off[i] + piece_n[i]) of the region (floats,
 * multiples of 4; at most HBR_MAX_LEVELS + 2 pieces), meant to run on a side stream BESIDE the kernel that produces them:
 * piece i is exchanged as soon as the local counter done[piece_done_idx[i]] has reached piece_need[i] (0 = complete when
 * the kernel starts) and the other ranks report the same.  Enqueue it AFTER the producer (hbr_hash_encode_bwd*_stream) so
 * that a device that serialises the two launches still terminates.  Same result, status and grid rules as above. */
int hbr_allreduce_peer_stream(void* const* bufs, void* const* flags, void* multicast, int rank, int world, int npieces,
                              const int64_t* piece_off, const int64_t* piece_n, const unsigned int* piece_need,
                              const int* piece_done_idx, const unsigned int* done, float scale, int ctas,
                              unsigned int* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HBR_B200_H_ */
