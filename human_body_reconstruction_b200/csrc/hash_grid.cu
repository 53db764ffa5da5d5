// Multiresolution hash-grid encoder: forward gather, backward warp-aggregated scatter-add, index probe.
// Replaces HashEncoder.forward (hash_encoding.py:146-170) and its autograd (16 x embedding_dense_backward).
//
// Mapping (both directions): CTA = 128 consecutive points x all levels, 256 threads; thread (p, g) owns
// point p and the levels l = g, g+2, ...  A warp is 32 CONSECUTIVE points -- when the caller is the
// volume renderer these are consecutive samples of one ray, which share cells on the coarse levels
// (SURVEY appendix C): the forward gathers coalesce into few L1 lines and the backward merges runs of
// equal cells with shuffles before issuing one red.global.add.v2.f32 per distinct entry.
// Rows of y / dy cross shared memory so global traffic is full 128-byte lines.
#include "common.cuh"

namespace hbr {

#ifndef HBR_HASH_TILE
#define HBR_HASH_TILE 128
#endif
constexpr int kTilePts = HBR_HASH_TILE;          // points per CTA
constexpr int kHashThreads = 2 * kTilePts;       // two threads per point (alternating levels)

template <int F> struct FeatVec;
template <> struct FeatVec<1> { using type = float; };
template <> struct FeatVec<2> { using type = float2; };
template <> struct FeatVec<4> { using type = float4; };

template <int F>
__device__ __forceinline__ void load_feat(const float* __restrict__ base, uint32_t idx, float v[F]) {
  if (F == 1) {
    v[0] = __ldg(base + idx);
  } else if (F == 2) {
    const float2 t = __ldg(reinterpret_cast<const float2*>(base) + idx);
    v[0] = t.x; v[1] = t.y;
  } else {
    const float4 t = __ldg(reinterpret_cast<const float4*>(base) + idx);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
}

// Explicit red.global (no return value).  atomicAdd() with an unused result is lowered to RED as well -- unless the kernel
// contains a memory fence: the streamed variants below (a gpu-scope fence before the completion count) then got ATOMG for
// every gradient update, whose returned values the LSU has to track: measured 257 us against 183 us for the same reductions.
__device__ __forceinline__ void red_add_f32(float* p, float a) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(a) : "memory");
}
__device__ __forceinline__ void red_add_v2(float* p, float a, float b) {
  asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

template <int F>
__device__ __forceinline__ void red_feat(float* base, uint32_t idx, const float v[F]) {
  if (F == 1) {
    red_add_f32(base + idx, v[0]);
  } else if (F == 2) {
    red_add_v2(base + 2 * (size_t)idx, v[0], v[1]);
  } else {
    red_add_v4(base + 4 * (size_t)idx, v[0], v[1], v[2], v[3]);
  }
}

template <typename XT>
__device__ __forceinline__ void load_point(const XT* __restrict__ x, long long gp, long long n, float p[3]) {
  if (gp < n) {
    p[0] = load_coord(x + gp * 3 + 0);
    p[1] = load_coord(x + gp * 3 + 1);
    p[2] = load_coord(x + gp * 3 + 2);
  } else {
    p[0] = p[1] = p[2] = 0.f;
  }
}

// Sample positions formed in the kernel from the rays: point gp = (ray gp / S, sample gp % S), p = o + d * t with the
// multiply and the add rounded separately -- bit-identical to hbr_ray_points (vol_renderer.py:165, helper.py:48) -- so
// the (R*S,3) position tensor of the training step never exists.  t is (S) shared (t_stride = 0) or (R,S) per ray.
struct RaySrc {
  const float* o;
  const float* d;
  const float* t;
  long long S, t_stride;
};
struct RayPts {};                                  // tag: positions come from a RaySrc
__device__ __forceinline__ void load_point(const RaySrc& rs, long long gp, long long n, float p[3]) {
  if (gp < n) {
    long long ray, smp;
    if (n <= 0xffffffffLL) {                      // 32-bit division (the 64-bit one is a ~100-instruction subroutine)
      const unsigned q = (unsigned)gp / (unsigned)rs.S;
      ray = q;
      smp = (long long)((unsigned)gp - q * (unsigned)rs.S);
    } else {
      ray = gp / rs.S;
      smp = gp - ray * rs.S;
    }
    const float tt = __ldg(rs.t + ray * rs.t_stride + smp);
#pragma unroll
    for (int a = 0; a < 3; ++a) p[a] = __fadd_rn(__ldg(rs.o + ray * 3 + a), __fmul_rn(__ldg(rs.d + ray * 3 + a), tt));
  } else {
    p[0] = p[1] = p[2] = 0.f;
  }
}
template <typename XT> struct PointSrc { using type = const XT*; };
template <> struct PointSrc<RayPts> { using type = RaySrc; };

// ---- forward ------------------------------------------------------------------------------------------
// PAIR: 0 = eight 8-byte gathers per level (default); 1 = (x, x+1) corner pairs of an even x share one aligned 16-byte
// slot: one LDG.128 per pair, the odd-x second load predicated.  Measured at 524 288 points, T = 2^19, cold L2: PAIR 0
// with 4 levels unrolled (32 gathers in flight per thread) 104 us, 2 levels 109 us, 8 levels 107 us; PAIR 1 124 us
// (the 16-byte loads double the L1 traffic of the odd-x half); a mixed variant (one 16-byte gather for lanes with an even
// x, two 8-byte gathers for the others, i.e. 25 % fewer L1 wavefronts on the hashed levels) 112 us against 107 us in the
// same step -- pairing only pays in the backward, where it halves the number of reductions.  ncu: the kernel runs at
// 83 % of the L1TEX wavefront peak (l1tex__data_pipe_lsu_wavefronts), 49 % of L2 throughput, 9 % of HBM.
// YT: float (the module's output, hash_encoding.py:165) or a 16-bit operand format (uint16_t bits of bf16 / fp16, selected by
// y_fmt): the rounding the MLP applies to its input under autocast, done here so the training step neither writes nor
// re-reads fp32 features (64 B/point instead of 128, and the MLP kernels copy the rows straight into their operand tile).
template <int F, bool POW2, typename XT, int PAIR = 0, int UNR = 4, typename YT = float>
__global__ void __launch_bounds__(kHashThreads)
hash_fwd_kernel(const typename PointSrc<XT>::type x, long long n, const float* __restrict__ table, YT* __restrict__ y,
                long long y_stride, const __grid_constant__ HashGeom g, int y_fmt, const unsigned long long* __restrict__ n_dev) {
  extern __shared__ float tile[];                    // [kTilePts][pitch]
  if (n_dev != nullptr) {                            // compacted sample lists: the live count lives on the device
    n = min(n, (long long)__ldg(n_dev));
    if ((long long)blockIdx.x * kTilePts >= n) return;
  }
  const int C = g.L * F;
  const int pitch = C | 1;                           // odd pitch: conflict-free column writes
  const int p = threadIdx.x & (kTilePts - 1);
  const int grp = threadIdx.x / kTilePts;
  const long long base = (long long)blockIdx.x * kTilePts;
  float pt[3];
  load_point(x, base + p, n, pt);

#pragma unroll UNR
  for (int l = grp; l < g.L; l += 2) {
    const float s = g.scale[l];
    long long ix, iy, iz;
    float fx, fy, fz;
    cell_of(pt[0], g.mu[0], g.sigma, s, ix, fx);
    cell_of(pt[1], g.mu[1], g.sigma, s, iy, fy);
    cell_of(pt[2], g.mu[2], g.sigma, s, iz, fz);
    uint32_t idx[8];
    corner_indices<POW2>(ix, iy, iz, g.T, idx);
    const float* lvl = table + (size_t)l * g.T * F;
    float v[8][F];
    if (F == 2 && POW2 && PAIR == 1) {
      const bool even = !(ix & 1);
#pragma unroll
      for (int c = 0; c < 8; c += 2) {
        const float4 q0 = __ldg(reinterpret_cast<const float4*>(lvl) + (idx[c] >> 1));
        float4 q1 = q0;
        if (!even) q1 = __ldg(reinterpret_cast<const float4*>(lvl) + (idx[c + 1] >> 1));
        const bool o0 = idx[c] & 1, o1 = idx[c + 1] & 1;
        v[c][0] = o0 ? q0.z : q0.x;     v[c][F - 1] = o0 ? q0.w : q0.y;
        v[c + 1][0] = o1 ? q1.z : q1.x; v[c + 1][F - 1] = o1 ? q1.w : q1.y;
      }
    } else {
#pragma unroll
      for (int c = 0; c < 8; ++c) load_feat<F>(lvl, idx[c], v[c]);        // 8 independent gathers in flight
    }
    float w[8];
    corner_weights(fx, fy, fz, w);
    // sum over corners in index order, multiply and add rounded separately (hash_encoding.py:144)
#pragma unroll
    for (int f = 0; f < F; ++f) {
      float acc = __fmul_rn(v[0][f], w[0]);
#pragma unroll
      for (int c = 1; c < 8; ++c) acc = __fadd_rn(acc, __fmul_rn(v[c][f], w[c]));
      tile[p * pitch + l * F + f] = acc;
    }
  }
  __syncthreads();
  const int cols = C + g.E;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (sizeof(YT) == 2) {
    // 16-bit rows: pairs of columns packed into one 32-bit store (cols is even for the 16-bit path: checked by the caller)
    uint32_t* y32 = reinterpret_cast<uint32_t*>(y);
    const int half = cols >> 1;
    for (int e = threadIdx.x; e < kTilePts * half; e += kHashThreads) {
      const int r = e / half, c = (e - r * half) * 2;
      const long long gp = base + r;
      if (gp >= n) break;
      const float a = c < C ? tile[r * pitch + c] : 0.f, b = c + 1 < C ? tile[r * pitch + c + 1] : 0.f;
      uint32_t v;
      if (y_fmt == HBR_F16) {
        const __half2 hh = __floats2half2_rn(a, b);
        v = *reinterpret_cast<const uint32_t*>(&hh);
      } else {
        const __nv_bfloat162 hh = __floats2bfloat162_rn(a, b);
        v = *reinterpret_cast<const uint32_t*>(&hh);
      }
      y32[(gp * y_stride + c) >> 1] = v;
    }
  } else {
    for (int r = warp; r < kTilePts; r += kHashThreads / 32) {
      const long long gp = base + r;
      if (gp >= n) break;
      for (int c = lane; c < cols; c += 32) y[gp * y_stride + c] = (YT)(c < C ? tile[r * pitch + c] : 0.f);
    }
  }
}

// ---- backward -----------------------------------------------------------------------------------------
// STREAM (multi-GPU gradient exchange, comm.cu: allreduce_stream_kernel): ONE launch walks the level chunks
// [bounds[c], bounds[c+1]) in chunk-major CTA order -- CTA b serves chunk b / tiles, tile b % tiles, and CTAs are
// dispatched in index order, so chunk c of the table gradient is complete long before the launch ends -- and every CTA
// counts itself into done[c] (all its reductions ordered before the count by a gpu-scope fence).  The all-reduce kernel
// running beside this one on another stream watches the counters and puts chunk c on the wire while the later chunks
// are still being accumulated.  Against one launch per chunk there are no launch gaps or per-chunk tails.
struct ChunkPlan {
  int nchunks;
  int bounds[HBR_MAX_LEVELS + 1];
  unsigned* done;                                  // [nchunks] counters, zeroed by the caller before the launch
  unsigned tiles;
  int order[HBR_MAX_LEVELS];                       // level-major kernel: the levels in visiting order (bounds index this list)
};

template <int F, bool POW2, typename XT, bool STREAM = false>
__global__ void __launch_bounds__(kHashThreads)
hash_bwd_kernel(const typename PointSrc<XT>::type x, long long n, const float* __restrict__ dy, long long dy_stride,
                float* __restrict__ dtable, const __grid_constant__ HashGeom g, int l_begin, int l_end,
                const unsigned long long* __restrict__ n_dev, const __grid_constant__ ChunkPlan plan) {
  extern __shared__ float tile[];
  if (n_dev != nullptr) {
    n = min(n, (long long)__ldg(n_dev));
    if ((long long)blockIdx.x * kTilePts >= n) return;
  }
  unsigned bidx = blockIdx.x, chunk = 0;
  if (STREAM) {
    chunk = blockIdx.x / plan.tiles;
    bidx = blockIdx.x - chunk * plan.tiles;
    l_begin = plan.bounds[chunk];
    l_end = plan.bounds[chunk + 1];
  }
  const int C = g.L * F;
  const int pitch = C | 1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long base = (long long)bidx * kTilePts;
  const int c0 = l_begin * F, c1 = l_end * F;
  if (C == 32 && dy_stride == 32 && ((uintptr_t)dy & 15) == 0) {
    // the tile is one contiguous 16 KB block of dy: four independent float4 loads per thread, all in flight before the
    // first shared-memory store (a one-load-at-a-time loop here cost a quarter of the kernel in long-scoreboard stalls)
    const float4* src = reinterpret_cast<const float4*>(dy + base * 32);
    float4 q[kTilePts * 8 / kHashThreads];
#pragma unroll
    for (int it = 0; it < kTilePts * 8 / kHashThreads; ++it) {
      const int idx = it * kHashThreads + threadIdx.x;          // float4 index in the tile: row = idx / 8
      const int c = (idx & 7) * 4;                              // a level chunk reads only its own columns of dy
      q[it] = (base + idx / 8 < n && c + 4 > c0 && c < c1) ? __ldg(src + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int it = 0; it < kTilePts * 8 / kHashThreads; ++it) {
      const int idx = it * kHashThreads + threadIdx.x, r = idx >> 3, c = (idx & 7) * 4;
      float* t = tile + r * pitch + c;                          // odd pitch: scalar stores, conflict-free
      t[0] = q[it].x; t[1] = q[it].y; t[2] = q[it].z; t[3] = q[it].w;
    }
  } else {
    for (int r = warp; r < kTilePts; r += kHashThreads / 32) {
      const long long gp = base + r;
      for (int c = c0 + lane; c < c1; c += 32) tile[r * pitch + c] = gp < n ? __ldg(dy + gp * dy_stride + c) : 0.f;
    }
  }
  const int p = threadIdx.x & (kTilePts - 1);
  const int grp = threadIdx.x / kTilePts;
  const bool valid = base + p < n;
  float pt[3];
  load_point(x, base + p, n, pt);
  __syncthreads();

  for (int l = l_begin + grp; l < l_end; l += 2) {
    const float s = g.scale[l];
    long long ix, iy, iz;
    float fx, fy, fz;
    cell_of(pt[0], g.mu[0], g.sigma, s, ix, fx);
    cell_of(pt[1], g.mu[1], g.sigma, s, iy, fy);
    cell_of(pt[2], g.mu[2], g.sigma, s, iz, fz);
    float w[8];
    corner_weights(fx, fy, fz, w);
    float gy[F];
#pragma unroll
    for (int f = 0; f < F; ++f) gy[f] = tile[p * pitch + l * F + f];
    float val[8][F];
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
      for (int f = 0; f < F; ++f) val[c][f] = w[c] * gy[f];

    // Runs of consecutive lanes in the same cell (a ray crosses a cell in one contiguous stretch).
    const long long pix = __shfl_up_sync(kFull, ix, 1);
    const long long piy = __shfl_up_sync(kFull, iy, 1);
    const long long piz = __shfl_up_sync(kFull, iz, 1);
    const int pvalid = __shfl_up_sync(kFull, (int)valid, 1);
    const bool head = lane == 0 || !valid || !pvalid || pix != ix || piy != iy || piz != iz;
    const unsigned heads = __ballot_sync(kFull, head);
    if (heads != kFull) {
      const unsigned above = lane == 31 ? 0u : (heads & (0xfffffffeu << lane));
      const int end = above ? (__ffs(above) - 1) : 32;                    // first lane of the next run
      const int maxrun = __reduce_max_sync(kFull, head ? end - lane : 0);
      for (int d = 1; d < maxrun; d <<= 1) {
#pragma unroll
        for (int c = 0; c < 8; ++c)
#pragma unroll
          for (int f = 0; f < F; ++f) {
            const float t = __shfl_down_sync(kFull, val[c][f], d);
            if (lane + d < end) val[c][f] += t;
          }
      }
    }
    if (head && valid) {
      uint32_t idx[8];
      corner_indices<POW2>(ix, iy, iz, g.T, idx);
      float* lvl = dtable + (size_t)l * g.T * F;
      if (F == 2 && POW2 && g.T >= 2 && !(ix & 1)) {       // T = 1 has no (e, e^1) slot pair
        // even x: corners (x, x+1) hash to entries e and e^1 -- one aligned 16-byte slot, one red.global.add.v4.f32
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
          const bool odd = idx[c] & 1;
          const float4 q = odd ? make_float4(val[c + 1][0], val[c + 1][F - 1], val[c][0], val[c][F - 1])
                               : make_float4(val[c][0], val[c][F - 1], val[c + 1][0], val[c + 1][F - 1]);
          red_add_v4(lvl + 4 * (size_t)(idx[c] >> 1), q.x, q.y, q.z, q.w);
        }
      } else {
#pragma unroll
        for (int c = 0; c < 8; ++c) red_feat<F>(lvl, idx[c], val[c]);
      }
    }
  }
  if (STREAM) {
    __syncthreads();                                // every thread's reductions have been issued ...
    if (threadIdx.x == 0) {
      __threadfence();                              // ... and are ordered (gpu scope) before the count
      atomicAdd(plan.done + chunk, 1u);
    }
  }
}

// ---- backward, level-major traversal (the multi-GPU training step, SURVEY 8e) --------------------------------------------
// dy arrives level-major, (L, n, F) -- hbr_mlp_bwd_tc writes it so on request -- and the grid is small enough to be
// co-resident: CTA b owns kLmPts consecutive points (thread t: points b*kLmPts + j*256 + t, j < kLmPer; their normalised
// positions stay in registers) and walks the LEVELS in order, all CTAs roughly in lockstep.  So the table gradient is
// finished level by level: after the last level of chunk c every CTA counts itself into done[c] (its reductions ordered
// before the count by a gpu-scope fence taken by one thread, while the other warps go on with the next chunk), and the
// all-reduce kernel beside it (comm.cu: allreduce_stream_kernel) puts chunk c on the wire while the finer levels -- where
// most of the reductions are -- are still being accumulated.  Same arithmetic, run merging and (x, x+1) pairing as
// hash_bwd_kernel; no shared memory (the per-level dy reads are coalesced 8-byte loads), positions formed once.
#ifndef HBR_LM_PER
#define HBR_LM_PER 4
#endif
#ifndef HBR_LM_MINB
#define HBR_LM_MINB 4
#endif
constexpr int kLmThreads = 256;
constexpr int kLmPer = HBR_LM_PER;                  // points per thread
constexpr int kLmPts = kLmThreads * kLmPer;         // points per CTA

template <int F, bool POW2, typename XT>
__global__ void __launch_bounds__(kLmThreads, HBR_LM_MINB)
hash_bwd_lm_kernel(const typename PointSrc<XT>::type x, long long n, const float* __restrict__ dy, float* __restrict__ dtable,
                   const __grid_constant__ HashGeom g, const __grid_constant__ ChunkPlan plan) {
  using FV = typename FeatVec<F>::type;
  const int lane = threadIdx.x & 31;
  const long long base = (long long)blockIdx.x * kLmPts + threadIdx.x;
  float un[kLmPer][3];
  bool valid[kLmPer];
#pragma unroll
  for (int j = 0; j < kLmPer; ++j) {
    const long long gp = base + j * kLmThreads;
    valid[j] = gp < n;
    float pt[3];
    load_point(x, gp, n, pt);
#pragma unroll
    for (int a = 0; a < 3; ++a) un[j][a] = __fdiv_rn(__fsub_rn(pt[a], g.mu[a]), g.sigma);   // level-independent part of cell_of
  }
  for (int c = 0; c < plan.nchunks; ++c) {
    const int b0 = plan.bounds[c], b1 = plan.bounds[c + 1];
#pragma unroll 1
    for (int i = b0; i < b1; ++i) {
      // odd warps walk the chunk's levels backwards, so that cheap (coarse: shuffle merges) and expensive (fine: one
      // reduction per corner) levels are in flight together; chunks pairing level c with L-1-c were measured too: no gain
      const int l = plan.order[((threadIdx.x >> 5) & 1) ? b1 - 1 - (i - b0) : i];
      const float s = g.scale[l];
      const FV* dyl = reinterpret_cast<const FV*>(dy) + (size_t)l * n;
      float* lvl = dtable + (size_t)l * g.T * F;
      FV gyv[kLmPer];
#pragma unroll
      for (int j = 0; j < kLmPer; ++j) {            // all loads of the level in flight before the first use
        const long long gp = base + j * kLmThreads;
        gyv[j] = valid[j] ? __ldg(dyl + gp) : FV{};
      }
#pragma unroll
      for (int j = 0; j < kLmPer; ++j) {
        const float* gy = reinterpret_cast<const float*>(&gyv[j]);
        const bool vj = valid[j];
        long long ix, iy, iz;
        float fx, fy, fz;
        {
          const float ux = __fmul_rn(un[j][0], s), uy = __fmul_rn(un[j][1], s), uz = __fmul_rn(un[j][2], s);
          ix = __float2ll_rz(ux); fx = __fsub_rn(ux, __ll2float_rn(ix));
          iy = __float2ll_rz(uy); fy = __fsub_rn(uy, __ll2float_rn(iy));
          iz = __float2ll_rz(uz); fz = __fsub_rn(uz, __ll2float_rn(iz));
        }
        float w[8];
        corner_weights(fx, fy, fz, w);
        float val[8][F];
#pragma unroll
        for (int q = 0; q < 8; ++q)
#pragma unroll
          for (int f = 0; f < F; ++f) val[q][f] = w[q] * gy[f];
        // runs of consecutive lanes in the same cell (a ray crosses a cell in one contiguous stretch)
        const long long pix = __shfl_up_sync(kFull, ix, 1);
        const long long piy = __shfl_up_sync(kFull, iy, 1);
        const long long piz = __shfl_up_sync(kFull, iz, 1);
        const int pvalid = __shfl_up_sync(kFull, (int)vj, 1);
        const bool head = lane == 0 || !vj || !pvalid || pix != ix || piy != iy || piz != iz;
        const unsigned heads = __ballot_sync(kFull, head);
        if (heads != kFull) {
          const unsigned above = lane == 31 ? 0u : (heads & (0xfffffffeu << lane));
          const int end = above ? (__ffs(above) - 1) : 32;
          const int maxrun = __reduce_max_sync(kFull, head ? end - lane : 0);
          for (int d = 1; d < maxrun; d <<= 1) {
#pragma unroll
            for (int q = 0; q < 8; ++q)
#pragma unroll
              for (int f = 0; f < F; ++f) {
                const float tt = __shfl_down_sync(kFull, val[q][f], d);
                if (lane + d < end) val[q][f] += tt;
              }
          }
        }
        if (head && vj) {
          uint32_t idx[8];
          corner_indices<POW2>(ix, iy, iz, g.T, idx);
          if (F == 2 && POW2 && g.T >= 2 && !(ix & 1)) {
#pragma unroll
            for (int q = 0; q < 8; q += 2) {
              const bool odd = idx[q] & 1;
              const float4 v4 = odd ? make_float4(val[q + 1][0], val[q + 1][F - 1], val[q][0], val[q][F - 1])
                                    : make_float4(val[q][0], val[q][F - 1], val[q + 1][0], val[q + 1][F - 1]);
              red_add_v4(lvl + 4 * (size_t)(idx[q] >> 1), v4.x, v4.y, v4.z, v4.w);
            }
          } else {
#pragma unroll
            for (int q = 0; q < 8; ++q) red_feat<F>(lvl, idx[q], val[q]);
          }
        }
      }
    }
    if (plan.done != nullptr) {
      __syncthreads();                              // every thread's reductions of this chunk have been issued ...
      if (threadIdx.x == 0) {
        __threadfence();                            // ... and are ordered (gpu scope) before the count
        atomicAdd(plan.done + c, 1u);
      }
    }
  }
}

// ---- parity probe: indices and weights ------------------------------------------------------------------
template <bool POW2, typename XT>
__global__ void hash_idx_kernel(const XT* __restrict__ x, long long n, int32_t* __restrict__ idx_out,
                                float* __restrict__ w_out, const __grid_constant__ HashGeom g) {
  const long long gp = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int l = blockIdx.y;
  if (gp >= n) return;
  float pt[3];
  load_point(x, gp, n, pt);
  long long ix, iy, iz;
  float fx, fy, fz;
  const float s = g.scale[l];
  cell_of(pt[0], g.mu[0], g.sigma, s, ix, fx);
  cell_of(pt[1], g.mu[1], g.sigma, s, iy, fy);
  cell_of(pt[2], g.mu[2], g.sigma, s, iz, fz);
  uint32_t idx[8];
  corner_indices<POW2>(ix, iy, iz, g.T, idx);
  float w[8];
  corner_weights(fx, fy, fz, w);
  const size_t o = ((size_t)l * n + gp) * 8;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    if (idx_out) idx_out[o + c] = (int32_t)idx[c];
    if (w_out) w_out[o + c] = w[c];
  }
}

// ---- input gradient: dL/dx ---------------------------------------------------------------------------------
// The forward's mapping and gathers, with the feature gradient dy in place of the output: per level the 8 corner rows are
// contracted with dy (g_c = sum_f dy[lF+f] v_c[f]) and differentiated through the trilinear weights.  The cells and fracs
// come from the same cell_of pipeline; the truncation toward zero has slope 1 on both sides of 0, so d(frac)/du = 1 and
//   dL/du_x = sum_c g_c (bit_x(c) ? +1 : -1) wy wz   (y, z alike),   dx_a = sum_l (s_l / sigma) dL/du_a.
// Each of the two threads of a point sums its own levels in order; the odd-level thread leaves its partial sum in shared
// memory and the even-level thread adds it: a fixed order, no atomics, bitwise reproducible.  dx is overwritten.
template <int F, bool POW2, typename XT, int UNR = 4>
__global__ void __launch_bounds__(kHashThreads)
hash_dx_kernel(const XT* __restrict__ x, long long n, const float* __restrict__ table, const float* __restrict__ dy,
               long long dy_stride, float* __restrict__ dx, const __grid_constant__ HashGeom g) {
  extern __shared__ float tile[];                    // [kTilePts][pitch] rows of dy, then [kTilePts][3] odd-level partials
  const int C = g.L * F;
  const int pitch = C | 1;
  float* part = tile + kTilePts * pitch;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long base = (long long)blockIdx.x * kTilePts;
  for (int r = warp; r < kTilePts; r += kHashThreads / 32) {
    const long long gp = base + r;
    for (int c = lane; c < C; c += 32) tile[r * pitch + c] = gp < n ? __ldg(dy + gp * dy_stride + c) : 0.f;
  }
  const int p = threadIdx.x & (kTilePts - 1);
  const int grp = threadIdx.x / kTilePts;
  float pt[3];
  load_point(x, base + p, n, pt);
  __syncthreads();

  float acc[3] = {0.f, 0.f, 0.f};
#pragma unroll UNR
  for (int l = grp; l < g.L; l += 2) {
    const float s = g.scale[l];
    long long ix, iy, iz;
    float fx, fy, fz;
    cell_of(pt[0], g.mu[0], g.sigma, s, ix, fx);
    cell_of(pt[1], g.mu[1], g.sigma, s, iy, fy);
    cell_of(pt[2], g.mu[2], g.sigma, s, iz, fz);
    uint32_t idx[8];
    corner_indices<POW2>(ix, iy, iz, g.T, idx);
    const float* lvl = table + (size_t)l * g.T * F;
    float v[8][F];
#pragma unroll
    for (int c = 0; c < 8; ++c) load_feat<F>(lvl, idx[c], v[c]);          // 8 independent gathers in flight
    float gc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      gc[c] = 0.f;
#pragma unroll
      for (int f = 0; f < F; ++f) gc[c] = fmaf(tile[p * pitch + l * F + f], v[c][f], gc[c]);
    }
    const float wx[2] = {1.f - fx, fx}, wy[2] = {1.f - fy, fy}, wz[2] = {1.f - fz, fz};
    float du[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const int bx = c & 1, by = (c >> 1) & 1, bz = (c >> 2) & 1;
      const float sg = bx ? gc[c] : -gc[c], sy = by ? gc[c] : -gc[c], sz = bz ? gc[c] : -gc[c];
      du[0] = fmaf(sg, wy[by] * wz[bz], du[0]);
      du[1] = fmaf(sy, wx[bx] * wz[bz], du[1]);
      du[2] = fmaf(sz, wx[bx] * wy[by], du[2]);
    }
    const float k = s / g.sigma;
#pragma unroll
    for (int a = 0; a < 3; ++a) acc[a] = fmaf(k, du[a], acc[a]);
  }
  if (grp == 1) {
#pragma unroll
    for (int a = 0; a < 3; ++a) part[p * 3 + a] = acc[a];
  }
  __syncthreads();
  const long long gp = base + p;
  if (grp == 0 && gp < n) {
#pragma unroll
    for (int a = 0; a < 3; ++a) dx[gp * 3 + a] = acc[a] + part[p * 3 + a];
  }
}

static int check_geom(const hbr_hash_geom* g) {
  HBR_REQUIRE(g != nullptr, "geom is NULL");
  HBR_REQUIRE(g->L >= 1 && g->L <= HBR_MAX_LEVELS, "L=%d out of range [1,%d]", g->L, HBR_MAX_LEVELS);
  HBR_REQUIRE(g->F == 1 || g->F == 2 || g->F == 4, "F=%d unsupported (1, 2 or 4)", g->F);
  HBR_REQUIRE(g->T >= 1 && g->T <= (1u << 30), "T=%u out of range", g->T);
  HBR_REQUIRE(g->E >= 0, "E=%d negative", g->E);
  return HBR_OK;
}

template <int F, bool POW2, typename XT>
static int launch_fwd(const void* x, int64_t n, const float* table, const HashGeom& g, float* y, int64_t ys, cudaStream_t st) {
  const size_t smem = (size_t)kTilePts * ((g.L * F) | 1) * sizeof(float);
  const unsigned grid = (unsigned)ceil_div(n, kTilePts);
  auto k = hash_fwd_kernel<F, POW2, XT>;
  HBR_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<grid, kHashThreads, smem, st>>>(static_cast<const XT*>(x), n, table, y, ys, g, HBR_F32, nullptr);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}
template <int F, bool POW2, typename XT>
static int launch_bwd(const void* x, int64_t n, const float* dy, int64_t ds, const HashGeom& g, float* dt, int l0, int l1,
                      cudaStream_t st) {
  const size_t smem = (size_t)kTilePts * ((g.L * F) | 1) * sizeof(float);
  HBR_CUDA(cudaFuncSetAttribute(hash_bwd_kernel<F, POW2, XT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  hash_bwd_kernel<F, POW2, XT><<<(unsigned)ceil_div(n, kTilePts), kHashThreads, smem, st>>>(
      static_cast<const XT*>(x), n, dy, ds, dt, g, l0, l1, nullptr, ChunkPlan{});
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}
template <int F, bool POW2, typename XT>
static int launch_dx(const void* x, int64_t n, const float* table, const float* dy, int64_t ds, const HashGeom& g, float* dx,
                     cudaStream_t st) {
  const size_t smem = (size_t)kTilePts * (((g.L * F) | 1) + 3) * sizeof(float);
  auto k = hash_dx_kernel<F, POW2, XT>;
  HBR_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<(unsigned)ceil_div(n, kTilePts), kHashThreads, smem, st>>>(static_cast<const XT*>(x), n, table, dy, ds, dx, g);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}
// the training step's variants: positions from the rays, features in fp32 or in the MLP's 16-bit operand format
template <int F, bool POW2, typename YT>
static int launch_fwd_rays(const RaySrc& rs, int64_t n, const float* table, const HashGeom& g, void* y, int64_t ys, int y_fmt,
                           cudaStream_t st) {
  const size_t smem = (size_t)kTilePts * ((g.L * F) | 1) * sizeof(float);
  auto k = hash_fwd_kernel<F, POW2, RayPts, 0, 4, YT>;
  HBR_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<(unsigned)ceil_div(n, kTilePts), kHashThreads, smem, st>>>(rs, n, table, static_cast<YT*>(y), ys, g, y_fmt, nullptr);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}
template <int F, bool POW2>
static int launch_bwd_rays(const RaySrc& rs, int64_t n, const float* dy, int64_t ds, const HashGeom& g, float* dt, int l0,
                           int l1, cudaStream_t st) {
  const size_t smem = (size_t)kTilePts * ((g.L * F) | 1) * sizeof(float);
  auto k = hash_bwd_kernel<F, POW2, RayPts>;
  HBR_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<(unsigned)ceil_div(n, kTilePts), kHashThreads, smem, st>>>(rs, n, dy, ds, dt, g, l0, l1, nullptr, ChunkPlan{});

  HBR_LAUNCH_CHECK();
  return HBR_OK;
}
// compacted sample lists (SURVEY 8f row 3): explicit fp32 positions, at most n of them, the live count on the device
template <int F, bool POW2, typename YT>
static int launch_fwd_pts(const float* x, int64_t n, const unsigned long long* n_dev, const float* table, const HashGeom& g,
                          void* y, int64_t ys, int y_fmt, cudaStream_t st) {
  const size_t smem = (size_t)kTilePts * ((g.L * F) | 1) * sizeof(float);
  auto k = hash_fwd_kernel<F, POW2, float, 0, 4, YT>;
  HBR_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<(unsigned)ceil_div(n, kTilePts), kHashThreads, smem, st>>>(x, n, table, static_cast<YT*>(y), ys, g, y_fmt, n_dev);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}
template <int F, bool POW2>
static int launch_bwd_pts(const float* x, int64_t n, const unsigned long long* n_dev, const float* dy, int64_t ds,
                          const HashGeom& g, float* dt, int l0, int l1, cudaStream_t st) {
  const size_t smem = (size_t)kTilePts * ((g.L * F) | 1) * sizeof(float);
  auto k = hash_bwd_kernel<F, POW2, float>;
  HBR_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<(unsigned)ceil_div(n, kTilePts), kHashThreads, smem, st>>>(x, n, dy, ds, dt, g, l0, l1, n_dev, ChunkPlan{});
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

// one launch over all level chunks in chunk-major CTA order, counting finished CTAs per chunk (ChunkPlan above)
template <int F, bool POW2, typename XT>
static int launch_bwd_stream(const typename PointSrc<XT>::type src, int64_t n, const float* dy, int64_t ds, const HashGeom& g,
                             float* dt, ChunkPlan plan, cudaStream_t st) {
  const size_t smem = (size_t)kTilePts * ((g.L * F) | 1) * sizeof(float);
  auto k = hash_bwd_kernel<F, POW2, XT, true>;
  HBR_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t tiles = ceil_div(n, kTilePts);
  HBR_REQUIRE(tiles * plan.nchunks < (1LL << 31), "too many CTAs: %lld tiles x %d chunks", (long long)tiles, plan.nchunks);
  plan.tiles = (unsigned)tiles;
  k<<<(unsigned)(tiles * plan.nchunks), kHashThreads, smem, st>>>(src, n, dy, ds, dt, g, 0, 0, nullptr, plan);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}
static int make_plan(const hbr_hash_geom* geom, const int* bounds, int nchunks, unsigned* done, ChunkPlan& plan) {
  HBR_REQUIRE(bounds != nullptr && done != nullptr, "NULL level_bounds / done");
  HBR_REQUIRE(nchunks >= 1 && nchunks <= geom->L, "nchunks=%d out of range [1,%d]", nchunks, geom->L);
  HBR_REQUIRE(bounds[0] == 0 && bounds[nchunks] == geom->L, "level_bounds must run from 0 to L");
  for (int c = 0; c < nchunks; ++c) HBR_REQUIRE(bounds[c] < bounds[c + 1], "level_bounds must increase");
  plan = ChunkPlan{};
  plan.nchunks = nchunks;
  for (int c = 0; c <= nchunks; ++c) plan.bounds[c] = bounds[c];
  for (int l = 0; l < geom->L; ++l) plan.order[l] = l;
  plan.done = done;
  return HBR_OK;
}

template <int F, bool POW2, typename XT>
static int launch_bwd_lm(const typename PointSrc<XT>::type src, int64_t n, const float* dy, const HashGeom& g, float* dt,
                         const ChunkPlan& plan, cudaStream_t st) {
  const int64_t ctas = ceil_div(n, kLmPts);
  HBR_REQUIRE(ctas < (1LL << 31), "too many points: %lld", (long long)n);
  hash_bwd_lm_kernel<F, POW2, XT><<<(unsigned)ctas, kLmThreads, 0, st>>>(src, n, dy, dt, g, plan);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

#define HBR_DISPATCH_HASH(FN, ...)                                                             \
  do {                                                                                         \
    const bool p2 = is_pow2(g.T);                                                              \
    const bool h = x_dtype == HBR_F16;                                                         \
    switch (g.F) {                                                                             \
      case 1:                                                                                  \
        return p2 ? (h ? FN<1, true, __half>(__VA_ARGS__) : FN<1, true, float>(__VA_ARGS__))   \
                  : (h ? FN<1, false, __half>(__VA_ARGS__) : FN<1, false, float>(__VA_ARGS__)); \
      case 2:                                                                                  \
        return p2 ? (h ? FN<2, true, __half>(__VA_ARGS__) : FN<2, true, float>(__VA_ARGS__))   \
                  : (h ? FN<2, false, __half>(__VA_ARGS__) : FN<2, false, float>(__VA_ARGS__)); \
      default:                                                                                 \
        return p2 ? (h ? FN<4, true, __half>(__VA_ARGS__) : FN<4, true, float>(__VA_ARGS__))   \
                  : (h ? FN<4, false, __half>(__VA_ARGS__) : FN<4, false, float>(__VA_ARGS__)); \
    }                                                                                          \
  } while (0)

}  // namespace hbr

using namespace hbr;

extern "C" int hbr_hash_encode_fwd(const void* x, int x_dtype, int64_t n, const float* table,
                                   const hbr_hash_geom* geom, float* y, int64_t y_stride, void* stream) {
  if (int rc = check_geom(geom)) return rc;
  HBR_REQUIRE(x_dtype == HBR_F32 || x_dtype == HBR_F16, "x_dtype %d", x_dtype);
  HBR_REQUIRE(n >= 0 && n < (1LL << 40), "n=%lld", (long long)n);
  if (n == 0) return HBR_OK;
  HBR_REQUIRE(x && table && y, "NULL pointer");
  HBR_REQUIRE(y_stride >= geom->L * geom->F + geom->E, "y_stride %lld too small", (long long)y_stride);
  HBR_REQUIRE((uintptr_t)table % 16 == 0, "table must be 16-byte aligned");
  const HashGeom g = to_device_geom(*geom);
  HBR_DISPATCH_HASH(launch_fwd, x, n, table, g, y, y_stride, as_stream(stream));
}

extern "C" int hbr_hash_encode_bwd(const void* x, int x_dtype, int64_t n, const float* dy, int64_t dy_stride,
                                   const hbr_hash_geom* geom, float* dtable, int level_begin, int level_end,
                                   void* stream) {
  if (int rc = check_geom(geom)) return rc;
  HBR_REQUIRE(x_dtype == HBR_F32 || x_dtype == HBR_F16, "x_dtype %d", x_dtype);
  HBR_REQUIRE(n >= 0 && n < (1LL << 40), "n=%lld", (long long)n);
  if (n == 0) return HBR_OK;
  HBR_REQUIRE(x && dy && dtable, "NULL pointer");
  HBR_REQUIRE(dy_stride >= geom->L * geom->F, "dy_stride %lld too small", (long long)dy_stride);
  HBR_REQUIRE((uintptr_t)dtable % 16 == 0, "dtable must be 16-byte aligned");
  HBR_REQUIRE(level_begin >= 0 && level_begin <= level_end && level_end <= geom->L, "level range [%d,%d)", level_begin,
              level_end);
  if (level_begin == level_end) return HBR_OK;
  const HashGeom g = to_device_geom(*geom);
  HBR_DISPATCH_HASH(launch_bwd, x, n, dy, dy_stride, g, dtable, level_begin, level_end, as_stream(stream));
}

extern "C" int hbr_hash_encode_dx(const void* x, int x_dtype, int64_t n, const float* table, const hbr_hash_geom* geom,
                                  const float* dy, int64_t dy_stride, float* dx, void* stream) {
  if (int rc = check_geom(geom)) return rc;
  HBR_REQUIRE(x_dtype == HBR_F32 || x_dtype == HBR_F16, "x_dtype %d", x_dtype);
  HBR_REQUIRE(n >= 0 && n < (1LL << 40), "n=%lld", (long long)n);
  if (n == 0) return HBR_OK;
  HBR_REQUIRE(x && table && dy && dx, "NULL pointer");
  HBR_REQUIRE(dy_stride >= geom->L * geom->F, "dy_stride %lld too small", (long long)dy_stride);
  HBR_REQUIRE((uintptr_t)table % 16 == 0, "table must be 16-byte aligned");
  const HashGeom g = to_device_geom(*geom);
  HBR_DISPATCH_HASH(launch_dx, x, n, table, dy, dy_stride, g, dx, as_stream(stream));
}

extern "C" int hbr_hash_indices(const void* x, int x_dtype, int64_t n, const hbr_hash_geom* geom,
                                int32_t* idx, float* w, void* stream) {
  if (int rc = check_geom(geom)) return rc;
  HBR_REQUIRE(x_dtype == HBR_F32 || x_dtype == HBR_F16, "x_dtype %d", x_dtype);
  if (n == 0) return HBR_OK;
  HBR_REQUIRE(x && (idx || w), "NULL pointer");
  const HashGeom g = to_device_geom(*geom);
  const dim3 grid((unsigned)ceil_div(n, 256), g.L);
  cudaStream_t st = as_stream(stream);
  const bool p2 = is_pow2(g.T);
  if (x_dtype == HBR_F16) {
    if (p2) hash_idx_kernel<true, __half><<<grid, 256, 0, st>>>((const __half*)x, n, idx, w, g);
    else hash_idx_kernel<false, __half><<<grid, 256, 0, st>>>((const __half*)x, n, idx, w, g);
  } else {
    if (p2) hash_idx_kernel<true, float><<<grid, 256, 0, st>>>((const float*)x, n, idx, w, g);
    else hash_idx_kernel<false, float><<<grid, 256, 0, st>>>((const float*)x, n, idx, w, g);
  }
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

static int check_rays(const float* o, const float* d, const float* t, int64_t t_rs, int64_t R, int64_t S) {
  HBR_REQUIRE(R >= 0 && S >= 1 && R < (1LL << 40) / S, "R=%lld S=%lld", (long long)R, (long long)S);
  HBR_REQUIRE(t_rs == 0 || t_rs >= S, "t_ray_stride %lld", (long long)t_rs);
  HBR_REQUIRE(R == 0 || (o && d && t), "NULL ray pointer");
  return HBR_OK;
}

extern "C" int hbr_hash_encode_fwd_rays(const float* rays_o, const float* rays_d, const float* t, int64_t t_ray_stride, int64_t R,
                                        int64_t S, const float* table, const hbr_hash_geom* geom, void* y, int64_t y_stride,
                                        int y_dtype, void* stream) {
  if (int rc = check_geom(geom)) return rc;
  if (int rc = check_rays(rays_o, rays_d, t, t_ray_stride, R, S)) return rc;
  HBR_REQUIRE(y_dtype == HBR_F32 || y_dtype == HBR_F16 || y_dtype == HBR_BF16, "y_dtype %d", y_dtype);
  const int64_t n = R * S;
  if (n == 0) return HBR_OK;
  HBR_REQUIRE(table && y, "NULL pointer");
  const int cols = geom->L * geom->F + geom->E;
  HBR_REQUIRE(y_stride >= cols, "y_stride %lld too small", (long long)y_stride);
  HBR_REQUIRE((uintptr_t)table % 16 == 0, "table must be 16-byte aligned");
  HBR_REQUIRE(y_dtype == HBR_F32 || (cols % 2 == 0 && y_stride % 2 == 0 && (uintptr_t)y % 4 == 0),
              "16-bit features need an even column count / stride and a 4-byte aligned buffer");
  const HashGeom g = to_device_geom(*geom);
  const RaySrc rs{rays_o, rays_d, t, S, t_ray_stride};
  cudaStream_t st = as_stream(stream);
  const bool p2 = is_pow2(g.T);
#define HBR_FWD_RAYS(F_)                                                                                              \
  (y_dtype == HBR_F32 ? (p2 ? launch_fwd_rays<F_, true, float>(rs, n, table, g, y, y_stride, y_dtype, st)              \
                            : launch_fwd_rays<F_, false, float>(rs, n, table, g, y, y_stride, y_dtype, st))            \
                      : (p2 ? launch_fwd_rays<F_, true, uint16_t>(rs, n, table, g, y, y_stride, y_dtype, st)           \
                            : launch_fwd_rays<F_, false, uint16_t>(rs, n, table, g, y, y_stride, y_dtype, st)))
  switch (g.F) {
    case 1: return HBR_FWD_RAYS(1);
    case 2: return HBR_FWD_RAYS(2);
    default: return HBR_FWD_RAYS(4);
  }
#undef HBR_FWD_RAYS
}

extern "C" int hbr_hash_encode_bwd_rays(const float* rays_o, const float* rays_d, const float* t, int64_t t_ray_stride, int64_t R,
                                        int64_t S, const float* dy, int64_t dy_stride, const hbr_hash_geom* geom, float* dtable,
                                        int level_begin, int level_end, void* stream) {
  if (int rc = check_geom(geom)) return rc;
  if (int rc = check_rays(rays_o, rays_d, t, t_ray_stride, R, S)) return rc;
  const int64_t n = R * S;
  if (n == 0) return HBR_OK;
  HBR_REQUIRE(dy && dtable, "NULL pointer");
  HBR_REQUIRE(dy_stride >= geom->L * geom->F, "dy_stride %lld too small", (long long)dy_stride);
  HBR_REQUIRE((uintptr_t)dtable % 16 == 0, "dtable must be 16-byte aligned");
  HBR_REQUIRE(level_begin >= 0 && level_begin <= level_end && level_end <= geom->L, "level range [%d,%d)", level_begin,
              level_end);
  if (level_begin == level_end) return HBR_OK;
  const HashGeom g = to_device_geom(*geom);
  const RaySrc rs{rays_o, rays_d, t, S, t_ray_stride};
  cudaStream_t st = as_stream(stream);
  const bool p2 = is_pow2(g.T);
  switch (g.F) {
    case 1: return p2 ? launch_bwd_rays<1, true>(rs, n, dy, dy_stride, g, dtable, level_begin, level_end, st)
                      : launch_bwd_rays<1, false>(rs, n, dy, dy_stride, g, dtable, level_begin, level_end, st);
    case 2: return p2 ? launch_bwd_rays<2, true>(rs, n, dy, dy_stride, g, dtable, level_begin, level_end, st)
                      : launch_bwd_rays<2, false>(rs, n, dy, dy_stride, g, dtable, level_begin, level_end, st);
    default: return p2 ? launch_bwd_rays<4, true>(rs, n, dy, dy_stride, g, dtable, level_begin, level_end, st)
                       : launch_bwd_rays<4, false>(rs, n, dy, dy_stride, g, dtable, level_begin, level_end, st);
  }
}

extern "C" int hbr_hash_encode_fwd_pts(const float* x, int64_t n_max, const unsigned long long* n_dev, const float* table,
                                       const hbr_hash_geom* geom, void* y, int64_t y_stride, int y_dtype, void* stream) {
  if (int rc = check_geom(geom)) return rc;
  HBR_REQUIRE(y_dtype == HBR_F32 || y_dtype == HBR_F16 || y_dtype == HBR_BF16, "y_dtype %d", y_dtype);
  HBR_REQUIRE(n_max >= 0 && n_max < (1LL << 40), "n_max=%lld", (long long)n_max);
  if (n_max == 0) return HBR_OK;
  HBR_REQUIRE(x && table && y, "NULL pointer");
  const int cols = geom->L * geom->F + geom->E;
  HBR_REQUIRE(y_stride >= cols && (uintptr_t)table % 16 == 0, "y_stride / table alignment");
  HBR_REQUIRE(y_dtype == HBR_F32 || (cols % 2 == 0 && y_stride % 2 == 0 && (uintptr_t)y % 4 == 0),
              "16-bit features need an even column count / stride and a 4-byte aligned buffer");
  const HashGeom g = to_device_geom(*geom);
  cudaStream_t st = as_stream(stream);
  const bool p2 = is_pow2(g.T);
#define HBR_FWD_PTS(F_)                                                                                               \
  (y_dtype == HBR_F32 ? (p2 ? launch_fwd_pts<F_, true, float>(x, n_max, n_dev, table, g, y, y_stride, y_dtype, st)     \
                            : launch_fwd_pts<F_, false, float>(x, n_max, n_dev, table, g, y, y_stride, y_dtype, st))   \
                      : (p2 ? launch_fwd_pts<F_, true, uint16_t>(x, n_max, n_dev, table, g, y, y_stride, y_dtype, st)  \
                            : launch_fwd_pts<F_, false, uint16_t>(x, n_max, n_dev, table, g, y, y_stride, y_dtype, st)))
  switch (g.F) {
    case 1: return HBR_FWD_PTS(1);
    case 2: return HBR_FWD_PTS(2);
    default: return HBR_FWD_PTS(4);
  }
#undef HBR_FWD_PTS
}

extern "C" int hbr_hash_encode_bwd_pts(const float* x, int64_t n_max, const unsigned long long* n_dev, const float* dy,
                                       int64_t dy_stride, const hbr_hash_geom* geom, float* dtable, int level_begin,
                                       int level_end, void* stream) {
  if (int rc = check_geom(geom)) return rc;
  HBR_REQUIRE(n_max >= 0 && n_max < (1LL << 40), "n_max=%lld", (long long)n_max);
  if (n_max == 0) return HBR_OK;
  HBR_REQUIRE(x && dy && dtable, "NULL pointer");
  HBR_REQUIRE(dy_stride >= geom->L * geom->F && (uintptr_t)dtable % 16 == 0, "dy_stride / dtable alignment");
  HBR_REQUIRE(level_begin >= 0 && level_begin <= level_end && level_end <= geom->L, "level range [%d,%d)", level_begin,
              level_end);
  if (level_begin == level_end) return HBR_OK;
  const HashGeom g = to_device_geom(*geom);
  cudaStream_t st = as_stream(stream);
  const bool p2 = is_pow2(g.T);
  switch (g.F) {
    case 1: return p2 ? launch_bwd_pts<1, true>(x, n_max, n_dev, dy, dy_stride, g, dtable, level_begin, level_end, st)
                      : launch_bwd_pts<1, false>(x, n_max, n_dev, dy, dy_stride, g, dtable, level_begin, level_end, st);
    case 2: return p2 ? launch_bwd_pts<2, true>(x, n_max, n_dev, dy, dy_stride, g, dtable, level_begin, level_end, st)
                      : launch_bwd_pts<2, false>(x, n_max, n_dev, dy, dy_stride, g, dtable, level_begin, level_end, st);
    default: return p2 ? launch_bwd_pts<4, true>(x, n_max, n_dev, dy, dy_stride, g, dtable, level_begin, level_end, st)
                       : launch_bwd_pts<4, false>(x, n_max, n_dev, dy, dy_stride, g, dtable, level_begin, level_end, st);
  }
}

extern "C" int64_t hbr_hash_bwd_stream_tiles(int64_t n) { return ceil_div(n, kTilePts); }
extern "C" int64_t hbr_hash_bwd_lm_ctas(int64_t n) { return ceil_div(n, kLmPts); }

static int make_lm_plan(const hbr_hash_geom* geom, const int* bounds, int nchunks, unsigned* done, ChunkPlan& plan) {
  if (bounds == nullptr) {                          // one chunk over all levels, no counters
    HBR_REQUIRE(done == nullptr, "done without level_bounds");
    plan = ChunkPlan{};
    plan.nchunks = 1;
    plan.bounds[0] = 0;
    plan.bounds[1] = geom->L;
    for (int l = 0; l < geom->L; ++l) plan.order[l] = l;
    return HBR_OK;
  }
  return make_plan(geom, bounds, nchunks, done, plan);
}

extern "C" int hbr_hash_encode_bwd_lm(const void* x, int x_dtype, int64_t n, const float* dy_lm, const hbr_hash_geom* geom,
                                      float* dtable, const int* level_bounds, int nchunks, unsigned int* done, void* stream) {
  if (int rc = check_geom(geom)) return rc;
  HBR_REQUIRE(x_dtype == HBR_F32 || x_dtype == HBR_F16, "x_dtype %d", x_dtype);
  HBR_REQUIRE(n > 0 && n < (1LL << 38), "n=%lld", (long long)n);
  HBR_REQUIRE(x && dy_lm && dtable, "NULL pointer");
  HBR_REQUIRE((uintptr_t)dtable % 16 == 0 && (uintptr_t)dy_lm % (4 * geom->F) == 0 && geom->E == 0, "alignment / E != 0");
  ChunkPlan plan;
  if (int rc = make_lm_plan(geom, level_bounds, nchunks, done, plan)) return rc;
  const HashGeom g = to_device_geom(*geom);
  cudaStream_t st = as_stream(stream);
  const bool p2 = is_pow2(g.T), h = x_dtype == HBR_F16;
#define HBR_BWD_LM(F_)                                                                                            \
  (p2 ? (h ? launch_bwd_lm<F_, true, __half>((const __half*)x, n, dy_lm, g, dtable, plan, st)                      \
           : launch_bwd_lm<F_, true, float>((const float*)x, n, dy_lm, g, dtable, plan, st))                       \
      : (h ? launch_bwd_lm<F_, false, __half>((const __half*)x, n, dy_lm, g, dtable, plan, st)                     \
           : launch_bwd_lm<F_, false, float>((const float*)x, n, dy_lm, g, dtable, plan, st)))
  switch (g.F) {
    case 1: return HBR_BWD_LM(1);
    case 2: return HBR_BWD_LM(2);
    default: return HBR_BWD_LM(4);
  }
#undef HBR_BWD_LM
}

extern "C" int hbr_hash_encode_bwd_rays_lm(const float* rays_o, const float* rays_d, const float* t, int64_t t_ray_stride,
                                           int64_t R, int64_t S, const float* dy_lm, const hbr_hash_geom* geom, float* dtable,
                                           const int* level_bounds, int nchunks, unsigned int* done, void* stream) {
  if (int rc = check_geom(geom)) return rc;
  if (int rc = check_rays(rays_o, rays_d, t, t_ray_stride, R, S)) return rc;
  const int64_t n = R * S;
  HBR_REQUIRE(n > 0 && n < (1LL << 38), "n=%lld", (long long)n);
  HBR_REQUIRE(dy_lm && dtable, "NULL pointer");
  HBR_REQUIRE((uintptr_t)dtable % 16 == 0 && (uintptr_t)dy_lm % (4 * geom->F) == 0 && geom->E == 0, "alignment / E != 0");
  ChunkPlan plan;
  if (int rc = make_lm_plan(geom, level_bounds, nchunks, done, plan)) return rc;
  const HashGeom g = to_device_geom(*geom);
  const RaySrc rs{rays_o, rays_d, t, S, t_ray_stride};
  cudaStream_t st = as_stream(stream);
  const bool p2 = is_pow2(g.T);
  switch (g.F) {
    case 1: return p2 ? launch_bwd_lm<1, true, RayPts>(rs, n, dy_lm, g, dtable, plan, st)
                      : launch_bwd_lm<1, false, RayPts>(rs, n, dy_lm, g, dtable, plan, st);
    case 2: return p2 ? launch_bwd_lm<2, true, RayPts>(rs, n, dy_lm, g, dtable, plan, st)
                      : launch_bwd_lm<2, false, RayPts>(rs, n, dy_lm, g, dtable, plan, st);
    default: return p2 ? launch_bwd_lm<4, true, RayPts>(rs, n, dy_lm, g, dtable, plan, st)
                       : launch_bwd_lm<4, false, RayPts>(rs, n, dy_lm, g, dtable, plan, st);
  }
}


extern "C" int hbr_hash_encode_bwd_stream(const void* x, int x_dtype, int64_t n, const float* dy, int64_t dy_stride,
                                          const hbr_hash_geom* geom, float* dtable, const int* level_bounds, int nchunks,
                                          unsigned int* done, void* stream) {
  if (int rc = check_geom(geom)) return rc;
  HBR_REQUIRE(x_dtype == HBR_F32 || x_dtype == HBR_F16, "x_dtype %d", x_dtype);
  HBR_REQUIRE(n > 0 && n < (1LL << 38), "n=%lld", (long long)n);     // n = 0 would leave the counters at zero: not allowed
  HBR_REQUIRE(x && dy && dtable, "NULL pointer");
  HBR_REQUIRE(dy_stride >= geom->L * geom->F && (uintptr_t)dtable % 16 == 0, "dy_stride / dtable alignment");
  ChunkPlan plan;
  if (int rc = make_plan(geom, level_bounds, nchunks, done, plan)) return rc;
  const HashGeom g = to_device_geom(*geom);
  cudaStream_t st = as_stream(stream);
  const bool p2 = is_pow2(g.T), h = x_dtype == HBR_F16;
#define HBR_BWD_STREAM(F_)                                                                                                       \
  (p2 ? (h ? launch_bwd_stream<F_, true, __half>((const __half*)x, n, dy, dy_stride, g, dtable, plan, st)                         \
           : launch_bwd_stream<F_, true, float>((const float*)x, n, dy, dy_stride, g, dtable, plan, st))                          \
      : (h ? launch_bwd_stream<F_, false, __half>((const __half*)x, n, dy, dy_stride, g, dtable, plan, st)                        \
           : launch_bwd_stream<F_, false, float>((const float*)x, n, dy, dy_stride, g, dtable, plan, st)))
  switch (g.F) {
    case 1: return HBR_BWD_STREAM(1);
    case 2: return HBR_BWD_STREAM(2);
    default: return HBR_BWD_STREAM(4);
  }
#undef HBR_BWD_STREAM
}

extern "C" int hbr_hash_encode_bwd_rays_stream(const float* rays_o, const float* rays_d, const float* t, int64_t t_ray_stride,
                                               int64_t R, int64_t S, const float* dy, int64_t dy_stride,
                                               const hbr_hash_geom* geom, float* dtable, const int* level_bounds, int nchunks,
                                               unsigned int* done, void* stream) {
  if (int rc = check_geom(geom)) return rc;
  if (int rc = check_rays(rays_o, rays_d, t, t_ray_stride, R, S)) return rc;
  const int64_t n = R * S;
  HBR_REQUIRE(n > 0 && n < (1LL << 38), "n=%lld", (long long)n);
  HBR_REQUIRE(dy && dtable, "NULL pointer");
  HBR_REQUIRE(dy_stride >= geom->L * geom->F && (uintptr_t)dtable % 16 == 0, "dy_stride / dtable alignment");
  ChunkPlan plan;
  if (int rc = make_plan(geom, level_bounds, nchunks, done, plan)) return rc;
  const HashGeom g = to_device_geom(*geom);
  const RaySrc rs{rays_o, rays_d, t, S, t_ray_stride};
  cudaStream_t st = as_stream(stream);
  const bool p2 = is_pow2(g.T);
  switch (g.F) {
    case 1: return p2 ? launch_bwd_stream<1, true, RayPts>(rs, n, dy, dy_stride, g, dtable, plan, st)
                      : launch_bwd_stream<1, false, RayPts>(rs, n, dy, dy_stride, g, dtable, plan, st);
    case 2: return p2 ? launch_bwd_stream<2, true, RayPts>(rs, n, dy, dy_stride, g, dtable, plan, st)
                      : launch_bwd_stream<2, false, RayPts>(rs, n, dy, dy_stride, g, dtable, plan, st);
    default: return p2 ? launch_bwd_stream<4, true, RayPts>(rs, n, dy, dy_stride, g, dtable, plan, st)
                       : launch_bwd_stream<4, false, RayPts>(rs, n, dy, dy_stride, g, dtable, plan, st);
  }
}
