// Sparse marching cubes (hbr.h, "sparse marching cubes"): seed bricks from the coarse lattice, close the active set over
// brick faces, compact it by a scan, and mesh the active bricks' cells with one welded vertex per crossing grid edge.
// Memory is the nb^3 brick map plus per-active-brick arrays; nothing here is sized by res^3.
#include "common.cuh"
#include "mc_tables.h"

namespace hbr {

constexpr int kB = HBR_MC_BRICK;             // cells per brick and axis
constexpr int kP = kB + 1;                   // points per brick and axis
constexpr int kPts = kP * kP * kP;           // 729
constexpr int kEdges = 3 * kPts;             // (axis, point) slots per brick
constexpr uint16_t kNoVertex = 0xffff;
static_assert(kEdges < kNoVertex, "local edge ids must fit 16 bits");

__device__ __forceinline__ bool inside(float d, float iso) { return d < iso; }

__device__ __forceinline__ void brick_coords(int b, int nb, int B[3]) {
  B[0] = b / (nb * nb);
  B[1] = (b / nb) % nb;
  B[2] = b % nb;
}

// ---- block-wide exclusive scan (blockDim.x a multiple of 32, <= 1024); sh: 32 entries ----------------------------
__device__ long long block_excl_scan(long long v, long long* sh, long long& total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  long long x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long y = __shfl_up_sync(kFull, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) sh[w] = x;
  __syncthreads();
  if (w == 0) {
    long long s = lane < nw ? sh[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long y = __shfl_up_sync(kFull, s, o);
      if (lane >= o) s += y;
    }
    if (lane < nw) sh[lane] = s;
  }
  __syncthreads();
  total = sh[nw - 1];
  const long long excl = x - v + (w > 0 ? sh[w - 1] : 0);
  __syncthreads();
  return excl;
}

// ---- device-wide exclusive scan in tiles of HBR_SCAN_TILE: tile sums, one CTA scans them, then each tile emits --------
constexpr int kScanThreads = 512;
constexpr int kScanItems = HBR_SCAN_TILE / kScanThreads;

template <class Op>
__global__ void __launch_bounds__(kScanThreads) scan_tiles_kernel(Op op, long long n, long long* __restrict__ block_sums) {
  __shared__ long long sh[32];
  const long long i0 = (long long)blockIdx.x * HBR_SCAN_TILE + (long long)threadIdx.x * kScanItems;
  long long v = 0;
#pragma unroll
  for (int r = 0; r < kScanItems; ++r)
    if (i0 + r < n) v += op.get(i0 + r);
  long long total;
  block_excl_scan(v, sh, total);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// in place: block_sums[0..tiles) -> exclusive prefix, *total_out = the sum
__global__ void __launch_bounds__(kScanThreads) scan_sums_kernel(long long* __restrict__ block_sums, long long tiles,
                                                                  long long* __restrict__ total_out) {
  __shared__ long long sh[32];
  long long carry = 0;
  for (long long base = 0; base < tiles; base += kScanThreads) {
    const long long i = base + threadIdx.x;
    const long long v = i < tiles ? block_sums[i] : 0;
    long long total;
    const long long e = block_excl_scan(v, sh, total);
    if (i < tiles) block_sums[i] = carry + e;
    carry += total;
  }
  if (threadIdx.x == 0) *total_out = carry;
}

template <class Op>
__global__ void __launch_bounds__(kScanThreads) scan_emit_kernel(Op op, long long n, const long long* __restrict__ block_sums) {
  __shared__ long long sh[32];
  const long long i0 = (long long)blockIdx.x * HBR_SCAN_TILE + (long long)threadIdx.x * kScanItems;
  long long v[kScanItems], s = 0;
#pragma unroll
  for (int r = 0; r < kScanItems; ++r) {
    v[r] = i0 + r < n ? op.get(i0 + r) : 0;
    s += v[r];
  }
  long long total;
  long long run = block_sums[blockIdx.x] + block_excl_scan(s, sh, total);
#pragma unroll
  for (int r = 0; r < kScanItems; ++r) {
    if (i0 + r < n) op.put(i0 + r, run, v[r]);
    run += v[r];
  }
}

template <class Op>
static int scan_sums(Op op, long long n, long long* block_sums, long long* total_out, cudaStream_t st) {
  const long long tiles = ceil_div(n, HBR_SCAN_TILE);
  scan_tiles_kernel<<<(unsigned)tiles, kScanThreads, 0, st>>>(op, n, block_sums);
  HBR_LAUNCH_CHECK();
  scan_sums_kernel<<<1, kScanThreads, 0, st>>>(block_sums, tiles, total_out);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

struct PendingOp {                            // select PENDING map entries; put: list them and give them slots
  int32_t* map;
  int32_t* list;
  int32_t base;
  __device__ long long get(long long i) const { return map[i] == HBR_BRICK_PENDING; }
  __device__ void put(long long i, long long excl, long long v) const {
    if (v) {
      list[excl] = (int32_t)i;
      map[i] = base + (int32_t)excl;
    }
  }
};

struct ColumnOp {                             // column c of an (n+1, 2) int64 array of counts -> exclusive prefix, in place
  long long* a;
  int c;
  __device__ long long get(long long i) const { return a[2 * i + c]; }
  __device__ void put(long long i, long long excl, long long) const { a[2 * i + c] = excl; }
};

// ---- selection ----------------------------------------------------------------------------------------------------
__global__ void brick_seed_kernel(const float* __restrict__ coarse, int nb, float iso, int32_t* __restrict__ map) {
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= (long long)nb * nb * nb) return;
  int B[3];
  brick_coords((int)b, nb, B);
  const int m = nb + 1;
  int nin = 0;
#pragma unroll
  for (int v = 0; v < 8; ++v)
    nin += inside(__ldg(coarse + ((long long)(B[0] + (v & 1)) * m + B[1] + ((v >> 1) & 1)) * m + B[2] + (v >> 2)), iso);
  map[b] = (nin != 0 && nin != 8) ? HBR_BRICK_PENDING : HBR_BRICK_INACTIVE;
}

// one warp per (brick, face): face f = 2*axis + side, the 9x9 points at local index 0 (side 0) or 8 (side 1) along axis
__global__ void __launch_bounds__(256)
brick_closure_kernel(const float* __restrict__ dens, const int32_t* __restrict__ list, long long n, int nb, float iso,
                     int32_t* __restrict__ map) {
  const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gw >= n * 6) return;
  const long long s = gw / 6;
  const int f = (int)(gw % 6), a = f >> 1, side = f & 1;
  int B[3];
  brick_coords(__ldg(list + s), nb, B);
  if (side == 0 ? B[a] == 0 : B[a] == nb - 1) return;          // the outer grid boundary: no neighbour
  const int step[3] = {kP * kP, kP, 1};
  const int u = a == 0 ? 1 : 0, v = a == 2 ? 1 : 2;
  const float* d = dens + s * kPts + side * kB * step[a];
  bool in = false, out = false;
  for (int r = lane; r < kP * kP; r += 32) {
    const bool x = inside(__ldg(d + (r / kP) * step[u] + (r % kP) * step[v]), iso);
    in |= x;
    out |= !x;
  }
  if (__any_sync(kFull, in) && __any_sync(kFull, out) && lane == 0) {
    B[a] += side ? 1 : -1;
    const long long nbr = ((long long)B[0] * nb + B[1]) * nb + B[2];
    if (map[nbr] == HBR_BRICK_INACTIVE) map[nbr] = HBR_BRICK_PENDING;      // racing writers store the same value
  }
}

// ---- brick marching cubes -----------------------------------------------------------------------------------------
// The brick that emits the vertex of the edge from grid point p along axis a: the first active brick containing the edge
// among o, o-e_u, o-e_v, o-e_u-e_v (o = min(p/8, nb-1); a step back along u only where p_u is an interior brick plane).
// The calling brick contains the edge, so one of them is active.
__device__ __forceinline__ int edge_owner(const int p[3], int a, int nb, const int32_t* __restrict__ map) {
  const int u = a == 0 ? 1 : 0, v = a == 2 ? 1 : 2;
  int o[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) o[k] = min(p[k] / kB, nb - 1);
  const bool su = p[u] % kB == 0 && p[u] > 0 && p[u] / kB < nb;
  const bool sv = p[v] % kB == 0 && p[v] > 0 && p[v] / kB < nb;
  const int b0 = (o[0] * nb + o[1]) * nb + o[2];
  if (!su && !sv) return b0;
  const int du = su ? (u == 0 ? nb * nb : nb) : 0;              // u < v, so u is axis 0 or 1
  const int dv = sv ? (v == 1 ? nb : 1) : 0;                    // v is axis 1 or 2
  if (__ldg(map + b0) >= 0) return b0;
  if (su && __ldg(map + b0 - du) >= 0) return b0 - du;
  if (sv && __ldg(map + b0 - dv) >= 0) return b0 - dv;
  return b0 - du - dv;
}

__device__ __forceinline__ int local_index(int li, int lj, int lk) { return (li * kP + lj) * kP + lk; }

struct BrickCtx {
  int b, B[3], ncell[3];
};

__device__ __forceinline__ BrickCtx brick_ctx(int b, int nb, int res) {
  BrickCtx c;
  c.b = b;
  brick_coords(b, nb, c.B);
#pragma unroll
  for (int k = 0; k < 3; ++k) c.ncell[k] = min(kB, res - 1 - kB * c.B[k]);
  return c;
}

// edge slot q = a*729 + local point: a crossing edge of this brick's cells?  (l: its local lower end point)
__device__ __forceinline__ bool crossing_edge(const float* d, const BrickCtx& c, int q, float iso, int& a, int l[3]) {
  a = q / kPts;
  const int r = q % kPts;
  l[0] = r / (kP * kP);
  l[1] = (r / kP) % kP;
  l[2] = r % kP;
  const int u = a == 0 ? 1 : 0, v = a == 2 ? 1 : 2;
  if (l[a] >= c.ncell[a] || l[u] > c.ncell[u] || l[v] > c.ncell[v]) return false;
  const int step = a == 0 ? kP * kP : (a == 1 ? kP : 1);
  return inside(d[r], iso) != inside(d[r + step], iso);
}

__device__ __forceinline__ unsigned cell_case(const float* d, int ci, int cj, int ck, float iso) {
  unsigned cs = 0;
#pragma unroll
  for (int v = 0; v < 8; ++v)
    cs |= (unsigned)inside(d[local_index(ci + (v & 1), cj + ((v >> 1) & 1), ck + (v >> 2))], iso) << v;
  return cs;
}

constexpr int kMcThreads = 256;

// one CTA per brick: local vertex ids of the brick's owned crossing edges in slot order, vertex and triangle counts
__global__ void __launch_bounds__(kMcThreads)
brick_mc_count_kernel(const float* __restrict__ dens, const int32_t* __restrict__ list, int nb, int res, float iso,
                      const int32_t* __restrict__ map, uint16_t* __restrict__ eid, long long* __restrict__ counts) {
  __shared__ float d[kPts];
  __shared__ long long sh[32];
  const long long s = blockIdx.x;
  for (int r = threadIdx.x; r < kPts; r += kMcThreads) d[r] = __ldg(dens + s * kPts + r);
  const BrickCtx c = brick_ctx(__ldg(list + s), nb, res);
  __syncthreads();
  long long nv = 0;
  for (int q0 = 0; q0 < kEdges; q0 += kMcThreads) {
    const int q = q0 + threadIdx.x;
    bool own = false;
    if (q < kEdges) {
      int a, l[3];
      if (crossing_edge(d, c, q, iso, a, l)) {
        const int p[3] = {kB * c.B[0] + l[0], kB * c.B[1] + l[1], kB * c.B[2] + l[2]};
        own = edge_owner(p, a, nb, map) == c.b;
      }
    }
    long long total;
    const long long e = block_excl_scan(own, sh, total);
    if (q < kEdges) eid[s * kEdges + q] = own ? (uint16_t)(nv + e) : kNoVertex;
    nv += total;
  }
  long long nt = 0;
  for (int cell = threadIdx.x; cell < kB * kB * kB; cell += kMcThreads) {
    const int ci = cell / (kB * kB), cj = (cell / kB) % kB, ck = cell % kB;
    if (ci < c.ncell[0] && cj < c.ncell[1] && ck < c.ncell[2]) nt += kMcNumTris[cell_case(d, ci, cj, ck, iso)];
  }
  long long total;
  block_excl_scan(nt, sh, total);
  if (threadIdx.x == 0) {
    counts[2 * s + 0] = nv;
    counts[2 * s + 1] = total;
  }
}

__global__ void __launch_bounds__(kMcThreads)
brick_mc_emit_kernel(const float* __restrict__ dens, const int32_t* __restrict__ list, int nb, int res, float iso,
                     const int32_t* __restrict__ map, const uint16_t* __restrict__ eid, const long long* __restrict__ offsets,
                     float* __restrict__ verts, int32_t* __restrict__ faces) {
  __shared__ float d[kPts];
  __shared__ long long sh[32];
  const long long s = blockIdx.x;
  for (int r = threadIdx.x; r < kPts; r += kMcThreads) d[r] = __ldg(dens + s * kPts + r);
  const BrickCtx c = brick_ctx(__ldg(list + s), nb, res);
  const long long vbase = __ldg(offsets + 2 * s), fbase = __ldg(offsets + 2 * s + 1);
  __syncthreads();
  for (int q = threadIdx.x; q < kEdges; q += kMcThreads) {
    const uint16_t id = __ldg(eid + s * kEdges + q);
    if (id == kNoVertex) continue;
    const int a = q / kPts, r = q % kPts;
    const int step = a == 0 ? kP * kP : (a == 1 ? kP : 1);
    const float d0 = d[r], d1 = d[r + step];
    const float tt = (iso - d0) / (d1 - d0);                  // hbr_mc_emit's arithmetic
    float p[3] = {(float)(kB * c.B[0] + r / (kP * kP)), (float)(kB * c.B[1] + (r / kP) % kP), (float)(kB * c.B[2] + r % kP)};
    p[a] += tt;
    float* o = verts + (vbase + id) * 3;
    o[0] = p[0]; o[1] = p[1]; o[2] = p[2];
  }
  long long fdone = 0;
  for (int c0 = 0; c0 < kB * kB * kB; c0 += kMcThreads) {
    const int cell = c0 + threadIdx.x;
    const int ci = cell / (kB * kB), cj = (cell / kB) % kB, ck = cell % kB;
    unsigned cs = 0;
    int nt = 0;
    if (ci < c.ncell[0] && cj < c.ncell[1] && ck < c.ncell[2]) {
      cs = cell_case(d, ci, cj, ck, iso);
      nt = kMcNumTris[cs];
    }
    long long total;
    const long long slot = fbase + fdone + block_excl_scan(nt, sh, total);
    fdone += total;
    for (int t = 0; t < nt; ++t) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const int e = kMcTris[cs][t * 3 + k];
        const int a = e >> 2, lo = e & 1, hi = (e >> 1) & 1;
        int p[3] = {kB * c.B[0] + ci, kB * c.B[1] + cj, kB * c.B[2] + ck};
        p[a == 0 ? 1 : 0] += lo;
        p[a == 2 ? 1 : 2] += hi;
        const int ob = edge_owner(p, a, nb, map);
        const long long os = __ldg(map + ob);
        int O[3];
        brick_coords(ob, nb, O);
        const int q = a * kPts + local_index(p[0] - kB * O[0], p[1] - kB * O[1], p[2] - kB * O[2]);
        faces[(slot + t) * 3 + k] = (int32_t)(__ldg(offsets + 2 * os) + __ldg(eid + os * kEdges + q));
      }
    }
  }
}

}  // namespace hbr

using namespace hbr;

static long long brick_total(int nb) { return (long long)nb * nb * nb; }

extern "C" int hbr_brick_seed(const float* coarse, int nb, float iso, int32_t* map, void* stream) {
  HBR_REQUIRE(nb >= 1 && nb <= 1290, "nb %d outside [1, 1290]", nb);            // nb^3 brick indices fit int32
  HBR_REQUIRE(coarse && map, "NULL pointer");
  brick_seed_kernel<<<(unsigned)ceil_div(brick_total(nb), 256), 256, 0, as_stream(stream)>>>(coarse, nb, iso, map);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

extern "C" int hbr_brick_pending_count(const int32_t* map, int nb, int64_t* block_sums, void* stream) {
  HBR_REQUIRE(nb >= 1 && nb <= 1290, "nb %d outside [1, 1290]", nb);
  HBR_REQUIRE(map && block_sums, "NULL pointer");
  const long long n = brick_total(nb);
  long long* bs = (long long*)block_sums;
  return scan_sums(PendingOp{const_cast<int32_t*>(map), nullptr, 0}, n, bs, bs + ceil_div(n, HBR_SCAN_TILE),
                   as_stream(stream));
}

extern "C" int hbr_brick_compact(int32_t* map, int nb, const int64_t* block_sums, int32_t base, int32_t* list, void* stream) {
  HBR_REQUIRE(nb >= 1 && nb <= 1290 && base >= 0, "bad argument");
  HBR_REQUIRE(map && block_sums && list, "NULL pointer");
  const long long n = brick_total(nb);
  scan_emit_kernel<<<(unsigned)ceil_div(n, HBR_SCAN_TILE), kScanThreads, 0, as_stream(stream)>>>(
      PendingOp{map, list, base}, n, (const long long*)block_sums);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

extern "C" int hbr_brick_closure(const float* dens, const int32_t* list, int64_t n, int nb, float iso, int32_t* map,
                                 void* stream) {
  HBR_REQUIRE(nb >= 1 && nb <= 1290 && n >= 0, "bad argument");
  if (n == 0) return HBR_OK;
  HBR_REQUIRE(dens && list && map, "NULL pointer");
  brick_closure_kernel<<<(unsigned)ceil_div(n * 6 * 32, 256), 256, 0, as_stream(stream)>>>(dens, list, n, nb, iso, map);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}

static int check_brick_mc(const float* dens, const int32_t* list, int64_t n, const int32_t* map, int nb, int res) {
  HBR_REQUIRE(res >= 2 && nb == (int)ceil_div(res - 1, HBR_MC_BRICK), "nb %d does not match res %d", nb, res);
  HBR_REQUIRE(nb <= 1290 && n >= 0 && n <= brick_total(nb) && n <= 0x7fffffff, "bad brick count %lld", (long long)n);
  HBR_REQUIRE(n == 0 || (dens && list && map), "NULL pointer");
  return HBR_OK;
}

extern "C" int hbr_brick_mc_count(const float* dens, const int32_t* list, int64_t n, const int32_t* map, int nb, int res,
                                  float iso, uint16_t* eid, int64_t* offsets, int64_t* block_sums, void* stream) {
  if (int rc = check_brick_mc(dens, list, n, map, nb, res)) return rc;
  HBR_REQUIRE(offsets && block_sums && (n == 0 || eid), "NULL pointer");
  cudaStream_t st = as_stream(stream);
  long long* off = (long long*)offsets;
  if (n == 0) {
    HBR_CUDA(cudaMemsetAsync(off, 0, 2 * sizeof(long long), st));
    return HBR_OK;
  }
  brick_mc_count_kernel<<<(unsigned)n, kMcThreads, 0, st>>>(dens, list, nb, res, iso, map, eid, off);
  HBR_LAUNCH_CHECK();
  long long* bs = (long long*)block_sums;
  for (int col = 0; col < 2; ++col) {
    if (int rc = scan_sums(ColumnOp{off, col}, n, bs, off + 2 * n + col, st)) return rc;
    scan_emit_kernel<<<(unsigned)ceil_div(n, HBR_SCAN_TILE), kScanThreads, 0, st>>>(ColumnOp{off, col}, n, bs);
    HBR_LAUNCH_CHECK();
  }
  return HBR_OK;
}

extern "C" int hbr_brick_mc_emit(const float* dens, const int32_t* list, int64_t n, const int32_t* map, int nb, int res,
                                 float iso, const uint16_t* eid, const int64_t* offsets, float* verts, int32_t* faces,
                                 void* stream) {
  if (int rc = check_brick_mc(dens, list, n, map, nb, res)) return rc;
  if (n == 0) return HBR_OK;
  HBR_REQUIRE(eid && offsets && verts && faces, "NULL pointer");
  brick_mc_emit_kernel<<<(unsigned)n, kMcThreads, 0, as_stream(stream)>>>(dens, list, nb, res, iso, map, eid,
                                                                         (const long long*)offsets, verts, faces);
  HBR_LAUNCH_CHECK();
  return HBR_OK;
}
