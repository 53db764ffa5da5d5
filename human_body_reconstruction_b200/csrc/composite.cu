// Ray sampling, direction encoding, alpha compositing (forward/backward) and hierarchical resampling.
// Replaces helper.py:53-107 (calc_color), :23-51 (hierarchical_sampling), vol_renderer.py:165,133-140,
// encoder.py:25-32.  One warp per ray: lanes take samples s = 32*i + lane so that the (R,S,*) tensors
// are read as contiguous 128..512-byte runs; prefix/suffix sums are warp shuffles with a carry between
// the 32-sample chunks.
#include "common.cuh"
#include <math_constants.h>

namespace hbr {

constexpr int kRaysPerCta = 8;

// ---- vol_renderer.py:165: o + d*t -----------------------------------------------------------------------
__global__ void ray_points_kernel(const float* __restrict__ o, const float* __restrict__ d, const float* __restrict__ t,
                                  long long t_rs, long long R, long long S, float* __restrict__ pts) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R * S) return;
  const long long r = i / S, s = i - r * S;
  const float tt = __ldg(t + r * t_rs + s);
#pragma unroll
  for (int k = 0; k < 3; ++k) pts[i * 3 + k] = __fadd_rn(__ldg(o + r * 3 + k), __fmul_rn(__ldg(d + r * 3 + k), tt));
}

// ---- vol_renderer.py:133-140 ------------------------------------------------------------------------------
struct Mu3 { float v[3]; };
__global__ void occupancy_kernel(const float* __restrict__ pts, long long n, const uint8_t* __restrict__ grid, int G,
                                 Mu3 mu, float sigma, uint8_t* __restrict__ mask) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  long long q[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float u = __fmul_rn(__fdiv_rn(__fsub_rn(__ldg(pts + i * 3 + k), mu.v[k]), sigma), (float)G);
    long long c = __float2ll_rz(u);
    if (c < 0) c += G;                       // Python-style negative index
    c = c < 0 ? 0 : (c >= G ? G - 1 : c);    // the reference would raise here; clamp instead of faulting
    q[k] = c;
  }
  mask[i] = grid[(q[0] * G + q[1]) * G + q[2]] ? 1 : 0;
}

// ---- encoder.py:25-32 ----------------------------------------------------------------------------------
template <typename XT>
__global__ void dir_encode_kernel(const XT* __restrict__ d, long long n, int dim, int nf, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // over n*dim*nf
  const long long total = n * dim * nf;
  if (i >= total) return;
  const int k = (int)(i % nf);
  const long long rc = i / nf;                 // row*dim + comp
  float s, c;
  if (sizeof(XT) == 2) {
    // fp16 tensor ops: every intermediate is rounded to fp16 (2*x, *k, sin/cos)
    const float x = __half2float(reinterpret_cast<const __half*>(d)[rc]);
    const float two_x = __half2float(__float2half_rn(2.f * x));
    const float a = __half2float(__float2half_rn(two_x * (float)k));
    s = __half2float(__float2half_rn(sinf(a)));
    c = __half2float(__float2half_rn(cosf(a)));
  } else {
    const float x = reinterpret_cast<const float*>(d)[rc];
    const float a = __fmul_rn(__fmul_rn(2.f, x), (float)k);
    s = sinf(a);
    c = cosf(a);
  }
  float* o = out + rc * (2 * nf);
  o[k] = s;
  o[nf + k] = c;
}

// ---- calc_color forward ------------------------------------------------------------------------------------
struct SampleIn {
  float delta, sig, p;       // p = clamp(sigma)*delta
  bool keep;                 // sigma >= -10 (gradient passes)
};

// row: where sample gs lives in the rgb / sigma tensors (gs itself, or its compacted row; < 0 = skipped sample)
__device__ __forceinline__ long long sample_row(const int32_t* __restrict__ rowmap, long long gs, int s, int S) {
  return rowmap == nullptr ? gs : (s < S ? (long long)__ldg(rowmap + gs) : -1);
}

__device__ __forceinline__ SampleIn load_sample(const float* __restrict__ tr, const float* __restrict__ sigma,
                                                long long sig_st, const uint8_t* __restrict__ mask, long long gs,
                                                int s, int S, float dnr, bool& live, long long row) {
  SampleIn q;
  live = s < S && row >= 0 && (mask == nullptr || mask[gs]);
  float delta = 0.f;
  if (s + 1 < S) delta = __fsub_rn(__ldg(tr + s + 1), __ldg(tr + s));   // helper.py:67, last delta stays 0
  q.delta = __fmul_rn(delta, dnr);                                       // :71
  const float raw = live ? __ldg(sigma + row * sig_st) : 0.f;
  q.keep = !(raw < -10.f);
  q.sig = q.keep ? raw : -10.f;                                          // :76
  q.p = s < S ? __fmul_rn(q.sig, q.delta) : 0.f;                         // :77
  return q;
}

// MAPS: also depth = sum_s w_s t_s and opacity = sum_s w_s per ray (either pointer may be NULL); without it the kernel is
// exactly the colour-only compositor (hbr_composite_fwd), the maps code is compiled out.
template <bool MAPS>
__global__ void __launch_bounds__(kRaysPerCta * 32)
composite_fwd_kernel(const float* __restrict__ t, long long t_rs, const float* __restrict__ rgb, long long rgb_st,
                     const float* __restrict__ sigma, long long sig_st, const float* __restrict__ dn, float dn_scalar,
                     const uint8_t* __restrict__ mask, const int32_t* __restrict__ rowmap, long long R, int S,
                     float* __restrict__ C, float* __restrict__ w_out, float ert_tau, float* __restrict__ depth,
                     float* __restrict__ opac) {
  // ert_tau: early ray termination (opt-in; +inf = off, the reference's behaviour).  Once the optical depth accumulated
  // over whole 32-sample chunks exceeds ert_tau the remaining chunks are skipped and get weight 0.  With the default
  // threshold 104 the transmittance exp(-depth) of every skipped sample is EXACTLY 0 in fp32 (exp(-104) underflows), so
  // the result is bit-identical as long as the depth does not fall back below the threshold -- always when sigma >= 0;
  // MLP_3D's LeakyReLU density can be slightly negative, which is why this is not on by default (SURVEY H8).
  const int lane = threadIdx.x & 31;
  const long long ray = (long long)blockIdx.x * kRaysPerCta + (threadIdx.x >> 5);
  if (ray >= R) return;
  const float* tr = t + ray * t_rs;
  const float dnr = dn ? __ldg(dn + ray) : dn_scalar;
  float carry = 0.f, c0 = 0.f, c1 = 0.f, c2 = 0.f, dsum = 0.f, asum = 0.f;
  for (int s0 = 0; s0 < S; s0 += 32) {
    const int s = s0 + lane;
    const long long gs = ray * S + s;
    bool live;
    const long long row = sample_row(rowmap, gs, s, S);
    const SampleIn q = load_sample(tr, sigma, sig_st, mask, gs, s, S, dnr, live, row);
    const float incl = carry + warp_incl_scan(q.p, lane);               // cumsum(prod), helper.py:93
    float prev = __shfl_up_sync(kFull, incl, 1);
    if (lane == 0) prev = carry;
    const float T = s == 0 ? 1.f : expf(-prev);                          // roll by one, T[0]=1 (:94-95)
    const float alpha = 1.f - expf(-q.p);                                // :91
    const float w = s < S ? __fmul_rn(T, alpha) : 0.f;                   // :102
    if (s < S) {
      if (w_out) w_out[gs] = w;
      if (MAPS) {
        dsum += w * __ldg(tr + s);
        asum += w;
      }
      if (live) {
        const float* c = rgb + row * rgb_st;
        c0 += w * __ldg(c + 0);
        c1 += w * __ldg(c + 1);
        c2 += w * __ldg(c + 2);
      }
    }
    carry = __shfl_sync(kFull, incl, 31);
    if (carry > ert_tau) {                                               // warp-uniform
      if (w_out)
        for (int s2 = s0 + 32 + lane; s2 < S; s2 += 32) w_out[ray * S + s2] = 0.f;
      break;
    }
  }
  c0 = warp_sum(c0); c1 = warp_sum(c1); c2 = warp_sum(c2);
  if (lane == 0) { C[ray * 3 + 0] = c0; C[ray * 3 + 1] = c1; C[ray * 3 + 2] = c2; }
  if (MAPS) {
    dsum = warp_sum(dsum); asum = warp_sum(asum);
    if (lane == 0) {
      if (depth) depth[ray] = dsum;
      if (opac) opac[ray] = asum;
    }
  }
}

// ---- calc_color backward (SURVEY A.3) -------------------------------------------------------------------
// MAPS: per-ray gradients gD of depth = sum w t and gA of opacity = sum w enter the per-sample term as
// c_s = g.rgb_s + gD t_s + gA (NULL = 0; gC may be NULL too); d(rgb) = w g is unchanged.  Without MAPS the code is compiled
// out and the kernel is exactly hbr_composite_bwd's.
template <int NCH, bool MAPS>
__global__ void __launch_bounds__(kRaysPerCta * 32)
composite_bwd_kernel(const float* __restrict__ t, long long t_rs, const float* __restrict__ rgb, long long rgb_st,
                     const float* __restrict__ sigma, long long sig_st, const float* __restrict__ dn, float dn_scalar,
                     const uint8_t* __restrict__ mask, const int32_t* __restrict__ rowmap, long long R, int S,
                     const float* __restrict__ gC, float* __restrict__ drgb, long long drgb_st, float* __restrict__ dsig,
                     long long dsig_st, float ert_tau, const float* __restrict__ gD, const float* __restrict__ gA) {
  const int lane = threadIdx.x & 31;
  const long long ray = (long long)blockIdx.x * kRaysPerCta + (threadIdx.x >> 5);
  if (ray >= R) return;
  const float* tr = t + ray * t_rs;
  const float dnr = dn ? __ldg(dn + ray) : dn_scalar;
  float g0 = 0.f, g1 = 0.f, g2 = 0.f, gd = 0.f, ga = 0.f;
  if (!MAPS || gC) { g0 = __ldg(gC + ray * 3 + 0); g1 = __ldg(gC + ray * 3 + 1); g2 = __ldg(gC + ray * 3 + 2); }
  if (MAPS) {
    if (gD) gd = __ldg(gD + ray);
    if (gA) ga = __ldg(gA + ray);
  }
  const bool packed = drgb_st == 4 && dsig_st == 4 && dsig == drgb + 3;

  float Tk[NCH], ek[NCH], ck[NCH], dk[NCH];     // transmittance, exp(-p), g.rgb, delta*[keep]
  float carry = 0.f;
  bool done = false;                             // early ray termination: the forward skipped the chunks from here on
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    const int s = i * 32 + lane;
    Tk[i] = 0.f; ek[i] = 1.f; ck[i] = 0.f; dk[i] = 0.f;
    if (i * 32 < S && !done) {
      const long long gs = ray * S + s;
      bool live;
      const long long row = sample_row(rowmap, gs, s, S);
      const SampleIn q = load_sample(tr, sigma, sig_st, mask, gs, s, S, dnr, live, row);
      const float incl = carry + warp_incl_scan(q.p, lane);
      float prev = __shfl_up_sync(kFull, incl, 1);
      if (lane == 0) prev = carry;
      carry = __shfl_sync(kFull, incl, 31);
      if (s < S) {
        Tk[i] = s == 0 ? 1.f : expf(-prev);
        ek[i] = expf(-q.p);
        if (live) {
          const float* c = rgb + row * rgb_st;
          ck[i] = g0 * __ldg(c + 0) + g1 * __ldg(c + 1) + g2 * __ldg(c + 2);
          dk[i] = q.keep ? q.delta : 0.f;
        }
        if (MAPS) ck[i] = __fadd_rn(__fmaf_rn(gd, __ldg(tr + s), ck[i]), ga);   // gD = gA = 0: ck unchanged
      }
      done = carry > ert_tau;                    // warp-uniform; skipped chunks keep T = 0: zero weights, zero gradients
    }
  }
  float rcarry = 0.f;                            // sum of w*c over all later chunks
#pragma unroll
  for (int i = NCH - 1; i >= 0; --i) {
    if (i * 32 < S) {
      const int s = i * 32 + lane;
      const long long gs = ray * S + s;
      const float w = Tk[i] * (1.f - ek[i]);
      const float wc = w * ck[i];
      const float rin = warp_rincl_scan(wc, lane);
      float after = __shfl_down_sync(kFull, rin, 1);
      if (lane == 31) after = 0.f;
      const float suffix = rcarry + after;       // sum_{j>k} w_j c_j
      rcarry += __shfl_sync(kFull, rin, 0);
      if (s < S) {
        const long long row = sample_row(rowmap, gs, s, S);
        const bool live = row >= 0 && (mask == nullptr || mask[gs]);
        const float dp = Tk[i] * ek[i] * ck[i] - suffix;
        const float ds = live ? dk[i] * dp : 0.f;
        const float r0 = live ? w * g0 : 0.f, r1 = live ? w * g1 : 0.f, r2 = live ? w * g2 : 0.f;
        if (row >= 0) {                          // skipped samples of a compacted list have no gradient row
          if (packed) {
            *reinterpret_cast<float4*>(drgb + row * 4) = make_float4(r0, r1, r2, ds);
          } else {
            float* o = drgb + row * drgb_st;
            o[0] = r0; o[1] = r1; o[2] = r2;
            dsig[row * dsig_st] = ds;
          }
        }
      }
    }
  }
}

// ---- hierarchical_sampling (helper.py:36-47) --------------------------------------------------------------
constexpr int kHierWarps = 4;

__global__ void __launch_bounds__(kHierWarps * 32)
hier_sample_kernel(float* __restrict__ w, const float* __restrict__ t, const float* __restrict__ u,
                   const float* __restrict__ cand, long long R, int S, int P2, int clamp_in_place,
                   float* __restrict__ t_fine) {
  extern __shared__ float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* cdf = sm + (size_t)warp * (S + P2);
  float* arr = cdf + S;
  const long long ray = (long long)blockIdx.x * kHierWarps + warp;
  if (ray >= R) return;
  float* wr = w + ray * S;
  float part = 0.f;
  for (int s = lane; s < S; s += 32) {
    float v = wr[s];
    if (v < 0.f) { v = 0.f; if (clamp_in_place) wr[s] = 0.f; }           // :36
    v = __fadd_rn(v, 1e-5f);                                              // :38
    cdf[s] = v;
    part += v;
  }
  const float total = warp_sum(part);
  __syncwarp();
  for (int s = lane; s < S; s += 32) cdf[s] = __fdiv_rn(cdf[s], total);  // pdf
  __syncwarp();
  if (lane == 0) {                                                        // sequential cumsum == torch CPU order (:39)
    float acc = 0.f;
    for (int s = 0; s < S; ++s) { acc = __fadd_rn(acc, cdf[s]); cdf[s] = acc; }
  }
  __syncwarp();
  for (int s = lane; s < P2; s += 32) {
    float v = CUDART_INF_F;
    if (s < S) {
      v = __ldg(t + s);
    } else if (s < 2 * S) {
      const float uu = __ldg(u + ray * S + (s - S));
      int lo = 0, hi = S;                                                 // searchsorted(right=True) (:41)
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cdf[mid] <= uu) lo = mid + 1; else hi = mid;
      }
      v = __ldg(cand + min(lo, S - 1));                                   // clamp + gather (:44-45)
    }
    arr[s] = v;
  }
  __syncwarp();
  for (int k = 2; k <= P2; k <<= 1) {                                     // bitonic sort (:47)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = lane; i < P2; i += 32) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const float a = arr[i], b = arr[ixj];
          const bool asc = (i & k) == 0;
          if ((a > b) == asc) { arr[i] = b; arr[ixj] = a; }
        }
      }
      __syncwarp();
    }
  }
  for (int s = lane; s < 2 * S; s += 32) t_fine[ray * 2 * S + s] = arr[s];
}

}  // namespace hbr

using namespace hbr;

extern "C" int hbr_ray_points(const float* o, const float* d, const float* t, int64_t t_rs, int64_t R, int64_t S,
                              float* pts, void* stream) {
  HBR_REQUIRE(R >= 0 && S >= 0, "negative size");
  if (R * S == 0) return HBR_OK;
  HBR_REQUIRE(o && d && t && pts, "NULL pointer");
  HBR_REQUIRE(t_rs == 0 || t_rs >= S, "t_ray_stride %lld", (long long)t_rs);
  ray_points_kernel<<<(unsigned)ceil_div(R * S, 256), 256, 0, as_stream(stream)>>>(o, d, t, t_rs, R, S, pts);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

extern "C" int hbr_occupancy_mask(const float* pts, int64_t n, const uint8_t* grid, int G, const float* mu3,
                                  float sigma, uint8_t* mask, void* stream) {
  if (n == 0) return HBR_OK;
  HBR_REQUIRE(pts && grid && mu3 && mask && G > 0, "bad argument");
  Mu3 mu{{mu3[0], mu3[1], mu3[2]}};
  occupancy_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, as_stream(stream)>>>(pts, n, grid, G, mu, sigma, mask);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

extern "C" int hbr_dir_encode(const void* d, int d_dtype, int64_t n, int dim, int num_freq, float* out, void* stream) {
  HBR_REQUIRE(d_dtype == HBR_F32 || d_dtype == HBR_F16, "d_dtype %d", d_dtype);
  HBR_REQUIRE(dim >= 1 && num_freq >= 1 && num_freq <= 127, "dim=%d num_freq=%d", dim, num_freq);
  if (n == 0) return HBR_OK;
  HBR_REQUIRE(d && out, "NULL pointer");
  const long long total = (long long)n * dim * num_freq;
  const unsigned grid = (unsigned)ceil_div(total, 256);
  if (d_dtype == HBR_F16) dir_encode_kernel<__half><<<grid, 256, 0, as_stream(stream)>>>((const __half*)d, n, dim, num_freq, out);
  else dir_encode_kernel<float><<<grid, 256, 0, as_stream(stream)>>>((const float*)d, n, dim, num_freq, out);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

static int check_composite(const float* t, int64_t t_rs, const float* rgb, const float* sigma, int64_t R, int64_t S) {
  HBR_REQUIRE(R >= 0 && S >= 1 && S <= 1024, "R=%lld S=%lld (S must be 1..1024)", (long long)R, (long long)S);
  HBR_REQUIRE(t && rgb && sigma, "NULL pointer");
  HBR_REQUIRE(t_rs == 0 || t_rs >= S, "t_ray_stride %lld", (long long)t_rs);
  return HBR_OK;
}

extern "C" int hbr_composite_fwd(const float* t, int64_t t_rs, const float* rgb, int64_t rgb_st, const float* sigma,
                                 int64_t sig_st, const float* dn, float dn_scalar, const uint8_t* mask, const int32_t* rowmap,
                                 int64_t R, int64_t S, float* C, float* w, float ert_tau, void* stream) {
  if (R == 0) return HBR_OK;
  if (int rc = check_composite(t, t_rs, rgb, sigma, R, S)) return rc;
  HBR_REQUIRE(C != nullptr, "C is NULL");
  if (!(ert_tau > 0.f)) ert_tau = 3.0e38f;                           // <= 0 / NaN: off (no fp32 optical depth exceeds it)
  composite_fwd_kernel<false><<<(unsigned)ceil_div(R, kRaysPerCta), kRaysPerCta * 32, 0, as_stream(stream)>>>(
      t, t_rs, rgb, rgb_st, sigma, sig_st, dn, dn_scalar, mask, rowmap, R, (int)S, C, w, ert_tau, nullptr, nullptr);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

extern "C" int hbr_composite_maps_fwd(const float* t, int64_t t_rs, const float* rgb, int64_t rgb_st, const float* sigma,
                                      int64_t sig_st, const float* dn, float dn_scalar, const uint8_t* mask,
                                      const int32_t* rowmap, int64_t R, int64_t S, float* C, float* w, float* depth,
                                      float* opacity, float ert_tau, void* stream) {
  if (R == 0) return HBR_OK;
  if (int rc = check_composite(t, t_rs, rgb, sigma, R, S)) return rc;
  HBR_REQUIRE(C != nullptr, "C is NULL");
  if (!(ert_tau > 0.f)) ert_tau = 3.0e38f;
  composite_fwd_kernel<true><<<(unsigned)ceil_div(R, kRaysPerCta), kRaysPerCta * 32, 0, as_stream(stream)>>>(
      t, t_rs, rgb, rgb_st, sigma, sig_st, dn, dn_scalar, mask, rowmap, R, (int)S, C, w, ert_tau, depth, opacity);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

template <bool MAPS>
static int composite_bwd_launch(const float* t, int64_t t_rs, const float* rgb, int64_t rgb_st, const float* sigma,
                                int64_t sig_st, const float* dn, float dn_scalar, const uint8_t* mask, const int32_t* rowmap,
                                int64_t R, int64_t S, const float* gC, const float* gD, const float* gA, float* drgb,
                                int64_t drgb_st, float* dsig, int64_t dsig_st, float ert_tau, void* stream) {
  if (!(ert_tau > 0.f)) ert_tau = 3.0e38f;
  if (drgb_st == 4 && dsig_st == 4 && dsig == drgb + 3)
    HBR_REQUIRE((uintptr_t)drgb % 16 == 0, "packed gradient buffer must be 16-byte aligned");
  const unsigned grid = (unsigned)ceil_div(R, kRaysPerCta);
  cudaStream_t st = as_stream(stream);
#define HBR_CB(N)                                                                                                      \
  composite_bwd_kernel<N, MAPS><<<grid, kRaysPerCta * 32, 0, st>>>(t, t_rs, rgb, rgb_st, sigma, sig_st, dn, dn_scalar, \
                                                                   mask, rowmap, R, (int)S, gC, drgb, drgb_st, dsig,   \
                                                                   dsig_st, ert_tau, gD, gA)
  if (S <= 128) HBR_CB(4);
  else if (S <= 256) HBR_CB(8);
  else if (S <= 512) HBR_CB(16);
  else HBR_CB(32);
#undef HBR_CB
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

extern "C" int hbr_composite_bwd(const float* t, int64_t t_rs, const float* rgb, int64_t rgb_st, const float* sigma,
                                 int64_t sig_st, const float* dn, float dn_scalar, const uint8_t* mask, const int32_t* rowmap,
                                 int64_t R, int64_t S, const float* gC, float* drgb, int64_t drgb_st, float* dsig,
                                 int64_t dsig_st, float ert_tau, void* stream) {
  if (R == 0) return HBR_OK;
  if (int rc = check_composite(t, t_rs, rgb, sigma, R, S)) return rc;
  HBR_REQUIRE(gC && drgb && dsig, "NULL pointer");
  return composite_bwd_launch<false>(t, t_rs, rgb, rgb_st, sigma, sig_st, dn, dn_scalar, mask, rowmap, R, S, gC, nullptr,
                                     nullptr, drgb, drgb_st, dsig, dsig_st, ert_tau, stream);
}

extern "C" int hbr_composite_maps_bwd(const float* t, int64_t t_rs, const float* rgb, int64_t rgb_st, const float* sigma,
                                      int64_t sig_st, const float* dn, float dn_scalar, const uint8_t* mask,
                                      const int32_t* rowmap, int64_t R, int64_t S, const float* gC, const float* gD,
                                      const float* gA, float* drgb, int64_t drgb_st, float* dsig, int64_t dsig_st,
                                      float ert_tau, void* stream) {
  if (R == 0) return HBR_OK;
  if (int rc = check_composite(t, t_rs, rgb, sigma, R, S)) return rc;
  HBR_REQUIRE(drgb && dsig, "NULL pointer");
  return composite_bwd_launch<true>(t, t_rs, rgb, rgb_st, sigma, sig_st, dn, dn_scalar, mask, rowmap, R, S, gC, gD, gA,
                                    drgb, drgb_st, dsig, dsig_st, ert_tau, stream);
}

extern "C" int hbr_hier_sample(float* w, const float* t, const float* u, const float* cand, int64_t R, int64_t S,
                               int clamp_in_place, float* t_fine, void* stream) {
  if (R == 0) return HBR_OK;
  HBR_REQUIRE(S >= 1 && S <= 2048, "S=%lld (1..2048)", (long long)S);
  HBR_REQUIRE(w && t && u && cand && t_fine, "NULL pointer");
  int P2 = 2;
  while (P2 < 2 * S) P2 <<= 1;
  const size_t smem = (size_t)kHierWarps * (S + P2) * sizeof(float);
  HBR_CUDA(cudaFuncSetAttribute(hier_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  hier_sample_kernel<<<(unsigned)ceil_div(R, kHierWarps), kHierWarps * 32, smem, as_stream(stream)>>>(
      w, t, u, cand, R, (int)S, P2, clamp_in_place, t_fine);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}
