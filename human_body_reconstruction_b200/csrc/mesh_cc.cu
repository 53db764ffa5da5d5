// Connected components of a triangle mesh (hbr.h, "connected components"): union-find over the label array, which is the
// parent array.  Four launches: init (label[v] = v, counts 0), hook (one thread per face: unite(a,b), unite(a,c)),
// flatten (one thread per vertex: label[v] = root, vertex count), face count (one thread per face).
//
// Linking.  unite() finds both roots with path halving and links the larger root under the smaller one with
// atomicCAS(&label[hi], hi, lo).  A parent is always smaller than its child, so there are no cycles and each component's
// final root is its minimum vertex index: the labels do not depend on the order the threads run in, and the integer counts
// are exact.  Path halving lowers a non-root entry to its grandparent with atomicMin; a non-root never becomes a root
// again, so this never races with a successful CAS, and any ancestor is a valid parent.  Every write to label is a min
// (the CAS included: hi -> lo < hi), so an entry only ever decreases along its chain of ancestors; the flatten pass can
// therefore halve paths while other threads store final roots, and its last atomicMin(&label[v], root) leaves the root
// there whatever order the stores land in (the root is the smallest ancestor).
//
// Counting.  Most faces of a marching-cubes mesh belong to one giant component, so the counts are added per warp: lanes
// holding the same root (__match_any_sync) add once, which keeps same-address atomics on the giant root 32x fewer.
//
// Termination.  find() walks strictly decreasing indices, so it ends.  A CAS fails only when label[hi] is no longer hi,
// i.e. another thread linked hi: every failed CAS is paid for by a link, and there are at most nv - 1 links in total.  This
// needs find() to see those links: label is read with ld.relaxed.gpu (L2, coherent with other SMs' atomics).  A read from
// L1 could keep returning a stale label[hi] == hi, and the retry would spin on it forever.
#include "common.cuh"

namespace hbr {

constexpr int kCcThreads = 256;

__device__ __forceinline__ int32_t ld_label(const int32_t* p) {
  int32_t v;
  asm volatile("ld.relaxed.gpu.global.b32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// root of x, halving the path on the way (label[x] <- label[label[x]])
__device__ __forceinline__ int32_t find_root(int32_t* label, int32_t x) {
  int32_t p = ld_label(label + x);
  while (p != x) {
    const int32_t g = ld_label(label + p);
    if (g != p) atomicMin(label + x, g);
    x = g;
    p = ld_label(label + x);
  }
  return x;
}

__device__ __forceinline__ void unite(int32_t* label, int32_t a, int32_t b) {
  while (true) {
    a = find_root(label, a);
    b = find_root(label, b);
    if (a == b) return;
    const int32_t lo = min(a, b), hi = max(a, b);
    if (atomicCAS(label + hi, hi, lo) == hi) return;
    a = lo;                                     // hi was linked meanwhile: look again from both sides
    b = hi;
  }
}

__global__ void __launch_bounds__(kCcThreads)
cc_init_kernel(long long nv, int32_t* __restrict__ label, int32_t* __restrict__ face_count, int32_t* __restrict__ vertex_count) {
  const long long v = (long long)blockIdx.x * kCcThreads + threadIdx.x;
  if (v >= nv) return;
  label[v] = (int32_t)v;
  face_count[v] = 0;
  vertex_count[v] = 0;
}

__global__ void __launch_bounds__(kCcThreads)
cc_hook_kernel(const int32_t* __restrict__ faces, long long nf, int32_t* label) {
  const long long f = (long long)blockIdx.x * kCcThreads + threadIdx.x;
  if (f >= nf) return;
  const int32_t a = __ldg(faces + 3 * f), b = __ldg(faces + 3 * f + 1), c = __ldg(faces + 3 * f + 2);
  unite(label, a, b);
  unite(label, a, c);
}

// count[r] += the lanes of this warp holding r (every lane of the warp must call it; ok = false lanes add nothing)
__device__ __forceinline__ void add_per_warp(int32_t* count, int32_t r, bool ok) {
  const unsigned same = __match_any_sync(kFull, ok ? r : -1);
  if (ok && (threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(count + r, __popc(same));
}

__global__ void __launch_bounds__(kCcThreads)
cc_flatten_kernel(long long nv, int32_t* label, int32_t* __restrict__ vertex_count) {
  const long long v = (long long)blockIdx.x * kCcThreads + threadIdx.x;
  const bool ok = v < nv;
  int32_t r = 0;
  if (ok) {
    r = find_root(label, (int32_t)v);
    atomicMin(label + v, r);
  }
  add_per_warp(vertex_count, r, ok);
}

__global__ void __launch_bounds__(kCcThreads)
cc_face_count_kernel(const int32_t* __restrict__ faces, long long nf, const int32_t* __restrict__ label,
                     int32_t* __restrict__ face_count) {
  const long long f = (long long)blockIdx.x * kCcThreads + threadIdx.x;
  const bool ok = f < nf;
  add_per_warp(face_count, ok ? __ldg(label + __ldg(faces + 3 * f)) : 0, ok);
}

}  // namespace hbr

using namespace hbr;

extern "C" int hbr_mesh_components(const int32_t* faces, int64_t nf, int64_t nv, int32_t* label, int32_t* face_count,
                                   int32_t* vertex_count, void* stream) {
  HBR_REQUIRE(nf >= 0 && nv >= 0 && nv <= 0x7fffffff, "bad size: nf %lld, nv %lld", (long long)nf, (long long)nv);
  HBR_REQUIRE(nf == 0 || nv > 0, "%lld faces but no vertices", (long long)nf);
  HBR_REQUIRE(nf == 0 || faces, "NULL pointer");
  HBR_REQUIRE(nv == 0 || (label && face_count && vertex_count), "NULL pointer");
  if (nv == 0) return HBR_OK;
  cudaStream_t st = as_stream(stream);
  const unsigned vblocks = (unsigned)ceil_div(nv, kCcThreads), fblocks = (unsigned)ceil_div(nf, kCcThreads);
  cc_init_kernel<<<vblocks, kCcThreads, 0, st>>>(nv, label, face_count, vertex_count);
  HBR_LAUNCH_CHECK();
  if (nf > 0) {
    cc_hook_kernel<<<fblocks, kCcThreads, 0, st>>>(faces, nf, label);
    HBR_LAUNCH_CHECK();
  }
  cc_flatten_kernel<<<vblocks, kCcThreads, 0, st>>>(nv, label, vertex_count);
  HBR_LAUNCH_CHECK();
  if (nf > 0) {
    cc_face_count_kernel<<<fblocks, kCcThreads, 0, st>>>(faces, nf, label, face_count);
    HBR_LAUNCH_CHECK();
  }
  return HBR_OK;
}
