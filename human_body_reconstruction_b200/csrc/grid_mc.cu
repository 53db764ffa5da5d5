// nerf2mesh.py hot loop: density grid evaluation (nerf2mesh.py:27-40,69-86) and marching cubes (:98).
#include "common.cuh"
#include "mlp_layout.cuh"
#include "mc_tables.h"

namespace hbr {

// ---- grid positions: np.linspace in float64, meshgrid 'xy', cast to fp16 (nerf2mesh.py:31-40) -------------
struct GridAxes {
  double start[3], stop[3], step[3];
  int res;
};

__device__ __forceinline__ double linspace_at(double start, double stop, double step, int i, int res) {
  if (res > 1 && i == res - 1) return stop;                 // numpy pins the end point
  return __dadd_rn(__dmul_rn((double)i, step), start);      // arange(num)*step + start, no FMA
}

// grid point (i, j, k)  <->  (x[j], y[i], z[k])   (meshgrid default 'xy' indexing)
__device__ __forceinline__ void grid_point(const GridAxes& ax, int i, int j, int k, __half* __restrict__ dst) {
  dst[0] = __double2half(linspace_at(ax.start[0], ax.stop[0], ax.step[0], j, ax.res));
  dst[1] = __double2half(linspace_at(ax.start[1], ax.stop[1], ax.step[1], i, ax.res));
  dst[2] = __double2half(linspace_at(ax.start[2], ax.stop[2], ax.step[2], k, ax.res));
}

__global__ void grid_points_kernel(GridAxes ax, long long p0, long long count, __half* __restrict__ pts) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= count) return;
  const long long p = p0 + q;
  const int res = ax.res;
  // flat index p = (i*res + j)*res + k
  grid_point(ax, (int)(p / ((long long)res * res)), (int)((p / res) % res), (int)(p % res), pts + q * 3);
}

// ---- the brick lattice of the sparse route (HBR_MC_BRICK^3 cells per brick, hbr.h) --------------------------------
// coarse lattice point c = (ci*(nb+1) + cj)*(nb+1) + ck is grid point min(8c, res-1) per axis; points [q0, q0+count)
__global__ void coarse_points_kernel(GridAxes ax, int nb, long long q0, long long count, __half* __restrict__ pts) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= count) return;
  const long long c = q0 + q;
  const int m = nb + 1, last = ax.res - 1;
  const int ci = (int)(c / ((long long)m * m)), cj = (int)((c / m) % m), ck = (int)(c % m);
  grid_point(ax, min(ci * HBR_MC_BRICK, last), min(cj * HBR_MC_BRICK, last), min(ck * HBR_MC_BRICK, last), pts + q * 3);
}

// brick-major points: point q = s*729 + (li*9 + lj)*9 + lk is grid point min(8*B + l, res-1) per axis of brick B = bricks[s]
__global__ void brick_points_kernel(GridAxes ax, int nb, const int32_t* __restrict__ bricks, long long q0, long long count,
                                    __half* __restrict__ pts) {
  constexpr int P = HBR_MC_BRICK + 1;
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= count) return;
  const long long g = q0 + q;
  const int b = __ldg(bricks + g / (P * P * P)), l = (int)(g % (P * P * P));
  const int bi = b / (nb * nb), bj = (b / nb) % nb, bk = b % nb, last = ax.res - 1;
  grid_point(ax, min(bi * HBR_MC_BRICK + l / (P * P), last), min(bj * HBR_MC_BRICK + (l / P) % P, last),
             min(bk * HBR_MC_BRICK + l % P, last), pts + q * 3);
}

// ---- marching cubes ----------------------------------------------------------------------------------------
__device__ __forceinline__ bool inside(float d, float iso) { return d < iso; }

// counts[0] += crossing edges owned by grid points with i in [i_begin,i_end); counts[1] += triangles of the
// cells with i in [i_begin, min(i_end, n0-1)).
__global__ void __launch_bounds__(256)
mc_count_kernel(const float* __restrict__ d, int n0, int n1, int n2, float iso, int i_begin, int i_end,
                unsigned long long* __restrict__ counts) {
  const long long plane = (long long)n1 * n2;
  const long long total = (long long)(i_end - i_begin) * plane;
  unsigned nv = 0, nt = 0;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(q % n2);
    const int j = (int)((q / n2) % n1);
    const int i = i_begin + (int)(q / plane);
    const long long o = (long long)i * plane + (long long)j * n2 + k;
    const bool in0 = inside(__ldg(d + o), iso);
    const bool hi = i + 1 < n0, hj = j + 1 < n1, hk = k + 1 < n2;
    bool c[8];
    c[0] = in0;
    c[1] = hi ? inside(__ldg(d + o + plane), iso) : in0;
    c[2] = hj ? inside(__ldg(d + o + n2), iso) : in0;
    c[4] = hk ? inside(__ldg(d + o + 1), iso) : in0;
    nv += (hi && c[1] != in0) + (hj && c[2] != in0) + (hk && c[4] != in0);
    if (hi && hj && hk) {
      c[3] = inside(__ldg(d + o + plane + n2), iso);
      c[5] = inside(__ldg(d + o + plane + 1), iso);
      c[6] = inside(__ldg(d + o + n2 + 1), iso);
      c[7] = inside(__ldg(d + o + plane + n2 + 1), iso);
      unsigned cs = 0;
#pragma unroll
      for (int v = 0; v < 8; ++v) cs |= (unsigned)c[v] << v;
      nt += kMcNumTris[cs];
    }
  }
  nv = __reduce_add_sync(kFull, nv);
  nt = __reduce_add_sync(kFull, nt);
  if ((threadIdx.x & 31) == 0) {
    if (nv) atomicAdd(counts + 0, (unsigned long long)nv);
    if (nt) atomicAdd(counts + 1, (unsigned long long)nt);
  }
}

// pass 1: one welded vertex per owned crossing edge; edge_id[a][i][j][k] = vertex index or -1
__global__ void __launch_bounds__(256)
mc_vertices_kernel(const float* __restrict__ d, int n0, int n1, int n2, float iso, int i_begin, int i_end,
                   int32_t* __restrict__ edge_id, float* __restrict__ verts, long long max_verts,
                   unsigned long long* __restrict__ cursors) {
  const long long plane = (long long)n1 * n2, vol = (long long)n0 * plane;
  const long long total = (long long)(i_end - i_begin) * plane;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(q % n2);
    const int j = (int)((q / n2) % n1);
    const int i = i_begin + (int)(q / plane);
    const long long o = (long long)i * plane + (long long)j * n2 + k;
    const float d0 = __ldg(d + o);
    const bool in0 = inside(d0, iso);
    const long long step[3] = {plane, (long long)n2, 1};
    const bool has[3] = {i + 1 < n0, j + 1 < n1, k + 1 < n2};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      int32_t id = -1;
      if (has[a]) {
        const float d1 = __ldg(d + o + step[a]);
        if (inside(d1, iso) != in0) {
          const unsigned long long slot = atomicAdd(cursors + 0, 1ULL);
          if ((long long)slot < max_verts) {
            const float tt = (iso - d0) / (d1 - d0);
            float p[3] = {(float)i, (float)j, (float)k};
            p[a] += tt;
            verts[slot * 3 + 0] = p[0]; verts[slot * 3 + 1] = p[1]; verts[slot * 3 + 2] = p[2];
            id = (int32_t)slot;
          }
        }
      }
      edge_id[(size_t)a * vol + o] = id;
    }
  }
}

// pass 2: triangles of every cell from the case table, referencing the welded vertices
__global__ void __launch_bounds__(256)
mc_faces_kernel(const float* __restrict__ d, int n0, int n1, int n2, float iso, int i_begin, int i_end,
                const int32_t* __restrict__ edge_id, int32_t* __restrict__ faces, long long max_faces,
                unsigned long long* __restrict__ cursors) {
  const long long plane = (long long)n1 * n2, vol = (long long)n0 * plane;
  const int ie = min(i_end, n0 - 1);
  const long long total = (long long)max(ie - i_begin, 0) * (n1 - 1) * (n2 - 1);
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(q % (n2 - 1));
    const int j = (int)((q / (n2 - 1)) % (n1 - 1));
    const int i = i_begin + (int)(q / ((long long)(n1 - 1) * (n2 - 1)));
    const long long o = (long long)i * plane + (long long)j * n2 + k;
    unsigned cs = 0;
#pragma unroll
    for (int v = 0; v < 8; ++v) {
      const long long ov = o + (v & 1) * plane + ((v >> 1) & 1) * n2 + ((v >> 2) & 1);
      cs |= (unsigned)inside(__ldg(d + ov), iso) << v;
    }
    const int nt = kMcNumTris[cs];
    if (nt == 0) continue;
    const unsigned long long slot = atomicAdd(cursors + 1, (unsigned long long)nt);
    for (int t = 0; t < nt; ++t) {
      if ((long long)(slot + t) >= max_faces) break;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int e = kMcTris[cs][t * 3 + c];
        const int a = e >> 2, lo = e & 1, hi = (e >> 1) & 1;
        // edge e runs along axis a from the cell corner whose other coordinates (increasing axis order) are (lo,hi)
        int off[3];
        off[a] = 0;
        off[a == 0 ? 1 : 0] = lo;
        off[a == 2 ? 1 : 2] = hi;
        const long long oe = o + off[0] * plane + off[1] * n2 + off[2];
        faces[(slot + t) * 3 + c] = edge_id[(size_t)a * vol + oe];
      }
    }
  }
}

// torchmcubes.grid_interp (nerf2mesh.py:99): trilinear sample of vol (C, n0, n1, n2) at points given as (x, y, z) =
// (index along axis 2, axis 1, axis 0) in grid-index units, clamped to the volume.  out (n, C).
__global__ void __launch_bounds__(256)
grid_interp_kernel(const float* __restrict__ vol, int C, int n0, int n1, int n2, const float* __restrict__ pts,
                   long long n, float* __restrict__ out) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n) return;
  const float x = fminf(fmaxf(__ldg(pts + q * 3 + 0), 0.f), (float)(n2 - 1));
  const float y = fminf(fmaxf(__ldg(pts + q * 3 + 1), 0.f), (float)(n1 - 1));
  const float z = fminf(fmaxf(__ldg(pts + q * 3 + 2), 0.f), (float)(n0 - 1));
  const int k0 = min((int)x, max(n2 - 2, 0)), j0 = min((int)y, max(n1 - 2, 0)), i0 = min((int)z, max(n0 - 2, 0));
  const int k1 = min(k0 + 1, n2 - 1), j1 = min(j0 + 1, n1 - 1), i1 = min(i0 + 1, n0 - 1);
  const float fx = x - (float)k0, fy = y - (float)j0, fz = z - (float)i0;
  const long long plane = (long long)n1 * n2, volsz = (long long)n0 * plane;
  for (int c = 0; c < C; ++c) {
    const float* v = vol + (long long)c * volsz;
    auto at = [&](int i, int j, int k) { return __ldg(v + (long long)i * plane + (long long)j * n2 + k); };
    const float c00 = at(i0, j0, k0) * (1.f - fx) + at(i0, j0, k1) * fx;
    const float c01 = at(i0, j1, k0) * (1.f - fx) + at(i0, j1, k1) * fx;
    const float c10 = at(i1, j0, k0) * (1.f - fx) + at(i1, j0, k1) * fx;
    const float c11 = at(i1, j1, k0) * (1.f - fx) + at(i1, j1, k1) * fx;
    const float c0 = c00 * (1.f - fy) + c01 * fy, c1 = c10 * (1.f - fy) + c11 * fy;
    out[q * C + c] = c0 * (1.f - fz) + c1 * fz;
  }
}

}  // namespace hbr

using namespace hbr;

extern "C" int hbr_grid_interp(const float* vol, int C, int n0, int n1, int n2, const float* pts, int64_t n, float* out,
                               void* stream) {
  HBR_REQUIRE(C >= 1 && n0 >= 1 && n1 >= 1 && n2 >= 1 && n >= 0, "bad shape");
  if (n == 0) return HBR_OK;
  HBR_REQUIRE(vol && pts && out, "NULL pointer");
  grid_interp_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, as_stream(stream)>>>(vol, C, n0, n1, n2, pts, n, out);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

static GridAxes make_axes(const double* min3, const double* max3, int res) {
  GridAxes ax;
  ax.res = res;
  for (int a = 0; a < 3; ++a) {
    ax.start[a] = min3[a];
    ax.stop[a] = max3[a];
    ax.step[a] = res > 1 ? (max3[a] - min3[a]) / (double)(res - 1) : 0.0;     // numpy: delta / div
  }
  return ax;
}

extern "C" int hbr_grid_points(const double* min3, const double* max3, int res, int64_t p0, int64_t count,
                               void* pts_f16, void* stream) {
  HBR_REQUIRE(min3 && max3 && res >= 1, "bad argument");
  const int64_t total = (int64_t)res * res * res;
  HBR_REQUIRE(p0 >= 0 && count >= 0 && p0 + count <= total, "range [%lld,+%lld) outside the %d^3 grid",
              (long long)p0, (long long)count, res);
  if (count == 0) return HBR_OK;
  HBR_REQUIRE(pts_f16 != nullptr, "NULL pointer");
  grid_points_kernel<<<(unsigned)ceil_div(count, 256), 256, 0, as_stream(stream)>>>(make_axes(min3, max3, res), p0, count,
                                                                                   (__half*)pts_f16);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

// The field at `count` points whose fp16 positions points(s, c) writes to pts_scratch for points [s, s+c), chunk by chunk:
// encoder -> density head (or the full MLP with dir_enc).  Every dense and sparse density query runs through here.
template <class Points>
static int field_at_points(Points&& points, int64_t count, const float* table, const hbr_hash_geom* geom,
                           const float* params, const hbr_mlp_dims* dims, const float* dir_enc, float* out,
                           void* pts_scratch, float* feat_scratch, int64_t chunk, int field_mode, void* stream) {
  HBR_REQUIRE(geom && dims && chunk >= 1, "bad argument");
  HBR_REQUIRE(field_mode == 0 || field_mode == 1, "field_mode %d", field_mode);
  HBR_REQUIRE(dims->in0 == geom->L * geom->F + geom->E, "MLP input width %d != encoder width %d", dims->in0,
              geom->L * geom->F + geom->E);
  const int ow = dir_enc ? 4 : 1;
  for (int64_t s = 0; s < count; s += chunk) {
    const int64_t c = count - s < chunk ? count - s : chunk;
    if (int rc = points(s, c)) return rc;
    if (int rc = hbr_hash_encode_fwd(pts_scratch, HBR_F16, c, table, geom, feat_scratch, dims->in0, stream)) return rc;
    if (!dir_enc && field_mode == 0 && dims->in0 == 32) {
      if (int rc = hbr_mlp_density_tf32x3(feat_scratch, c, params, dims, out + s, stream)) return rc;
      continue;
    }
    // one direction row for all points: dir_group >= c maps every point to row 0 (nerf2mesh.py:69-70)
    if (int rc = hbr_mlp_fwd_f32(feat_scratch, dims->in0, dir_enc, c, c, params, dims, out + s * ow, nullptr, stream))
      return rc;
  }
  return HBR_OK;
}

extern "C" int hbr_grid_density(const double* min3, const double* max3, int res, int64_t p0, int64_t count,
                                const float* table, const hbr_hash_geom* geom, const float* params,
                                const hbr_mlp_dims* dims, const float* dir_enc, float* out, void* pts_scratch,
                                float* feat_scratch, int64_t chunk, int field_mode, void* stream) {
  return field_at_points([&](int64_t s, int64_t c) { return hbr_grid_points(min3, max3, res, p0 + s, c, pts_scratch, stream); },
                         count, table, geom, params, dims, dir_enc, out, pts_scratch, feat_scratch, chunk, field_mode, stream);
}

static int brick_count(int res) { return res >= 2 ? (int)ceil_div(res - 1, HBR_MC_BRICK) : 0; }

extern "C" int hbr_coarse_density(const double* min3, const double* max3, int res, const float* table,
                                  const hbr_hash_geom* geom, const float* params, const hbr_mlp_dims* dims, float* out,
                                  void* pts_scratch, float* feat_scratch, int64_t chunk, int field_mode, void* stream) {
  HBR_REQUIRE(min3 && max3 && res >= 2, "bad argument (res %d < 2)", res);
  HBR_REQUIRE(out && pts_scratch && feat_scratch, "NULL pointer");
  const int nb = brick_count(res);
  const int64_t count = (int64_t)(nb + 1) * (nb + 1) * (nb + 1);
  const GridAxes ax = make_axes(min3, max3, res);
  auto points = [&](int64_t s, int64_t c) {
    coarse_points_kernel<<<(unsigned)ceil_div(c, 256), 256, 0, as_stream(stream)>>>(ax, nb, s, c, (__half*)pts_scratch);
    HBR_LAUNCH_CHECK();
    return (int)HBR_OK;
  };
  return field_at_points(points, count, table, geom, params, dims, nullptr, out, pts_scratch, feat_scratch, chunk, field_mode,
                         stream);
}

extern "C" int hbr_brick_density(const double* min3, const double* max3, int res, const int32_t* bricks, int64_t n,
                                 const float* table, const hbr_hash_geom* geom, const float* params,
                                 const hbr_mlp_dims* dims, float* out, void* pts_scratch, float* feat_scratch, int64_t chunk,
                                 int field_mode, void* stream) {
  HBR_REQUIRE(min3 && max3 && res >= 2 && n >= 0, "bad argument");
  if (n == 0) return HBR_OK;
  HBR_REQUIRE(bricks && out && pts_scratch && feat_scratch, "NULL pointer");
  const int nb = brick_count(res);
  constexpr int P = HBR_MC_BRICK + 1;
  const GridAxes ax = make_axes(min3, max3, res);
  auto points = [&](int64_t s, int64_t c) {
    brick_points_kernel<<<(unsigned)ceil_div(c, 256), 256, 0, as_stream(stream)>>>(ax, nb, bricks, s, c, (__half*)pts_scratch);
    HBR_LAUNCH_CHECK();
    return (int)HBR_OK;
  };
  return field_at_points(points, n * P * P * P, table, geom, params, dims, nullptr, out, pts_scratch, feat_scratch, chunk,
                         field_mode, stream);
}

static int check_mc(const float* d, int n0, int n1, int n2, int i_begin, int i_end) {
  HBR_REQUIRE(d != nullptr, "density is NULL");
  HBR_REQUIRE(n0 >= 1 && n1 >= 1 && n2 >= 1, "bad grid shape (%d,%d,%d)", n0, n1, n2);
  HBR_REQUIRE(0 <= i_begin && i_begin <= i_end && i_end <= n0, "slab [%d,%d) outside [0,%d)", i_begin, i_end, n0);
  return HBR_OK;
}

extern "C" int hbr_mc_count(const float* d, int n0, int n1, int n2, float iso, int i_begin, int i_end,
                            unsigned long long* counts, void* stream) {
  if (int rc = check_mc(d, n0, n1, n2, i_begin, i_end)) return rc;
  HBR_REQUIRE(counts != nullptr, "counts is NULL");
  const long long total = (long long)(i_end - i_begin) * n1 * n2;
  if (total == 0) return HBR_OK;
  const int grid = (int)min64(ceil_div(total, 256), (long long)sm_count() * 16);
  mc_count_kernel<<<grid, 256, 0, as_stream(stream)>>>(d, n0, n1, n2, iso, i_begin, i_end, counts);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

extern "C" int hbr_mc_emit(const float* d, int n0, int n1, int n2, float iso, int i_begin, int i_end,
                           int32_t* edge_id, float* verts, int64_t max_verts, int32_t* faces, int64_t max_faces,
                           unsigned long long* cursors, void* stream) {
  if (int rc = check_mc(d, n0, n1, n2, i_begin, i_end)) return rc;
  HBR_REQUIRE(edge_id && verts && faces && cursors, "NULL pointer");
  // faces of the last cell layer of the slab reference vertices on plane i_end, owned by the next slab:
  // single-device callers pass the whole grid; slab callers emit vertices for [i_begin, min(i_end+1,n0)).
  const int v_end = i_end < n0 ? i_end + 1 : n0;
  const long long totv = (long long)(v_end - i_begin) * n1 * n2;
  if (totv == 0) return HBR_OK;
  cudaStream_t st = as_stream(stream);
  const int gridv = (int)min64(ceil_div(totv, 256), (long long)sm_count() * 16);
  mc_vertices_kernel<<<gridv, 256, 0, st>>>(d, n0, n1, n2, iso, i_begin, v_end, edge_id, verts, max_verts, cursors);
  HBR_LAUNCH_CHECK();
  if (n1 > 1 && n2 > 1 && n0 > 1) {
    const long long totc = (long long)max(min(i_end, n0 - 1) - i_begin, 0) * (n1 - 1) * (n2 - 1);
    if (totc > 0) {
      const int gridc = (int)min64(ceil_div(totc, 256), (long long)sm_count() * 16);
      mc_faces_kernel<<<gridc, 256, 0, st>>>(d, n0, n1, n2, iso, i_begin, i_end, edge_id, faces, max_faces, cursors);
      HBR_LAUNCH_CHECK();
    }
  }
  return HBR_OK;
}
