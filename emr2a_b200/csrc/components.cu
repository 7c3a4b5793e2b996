// Connected components of an edge list on the GPU: a lock-free union-find over a caller-owned int64 parent[n]
// (emr2a_components_union / emr2a_components_finish).  It turns the pairs of the near-duplicate self-join into groups
// (Engine.duplicate_groups): the pairs of a band are folded into the forest and dropped, so no pair list has to be
// kept.  The scheme is that of ECL-CC (Jaiganesh & Burtscher, HPDC 2018): path halving on every find, roots hooked
// with one compare-and-swap, plain (volatile) loads, no locks.
//
// Correctness:
//  * Invariant: parent[v] <= v for every v, at every moment.  The start state is any forest that satisfies it
//    (arange(n), or the output of an earlier finish).  A halving store writes parent[v] = parent[parent[v]], an
//    ancestor of v, so it keeps the invariant; a racing halving store can only write an ancestor that is not the
//    newest one, which loses a shortcut, never a link.  Halving stores go to non-roots and hooks to roots (the CAS
//    expects parent[hi] == hi), and a non-root never becomes a root again, so a store never undoes a hook.
//  * A root hi is hooked only under a root lo < hi of the other endpoint's tree (atomicCAS(&parent[hi], hi, lo)).  A
//    failed CAS means hi was hooked meanwhile: both roots are found again from what the CAS returned, and the loop
//    ends when they are equal.  The roots of an edge only decrease, so it ends.
//  * With parent[v] <= v the root of a tree is its smallest vertex, and a hook keeps the smaller of two roots, so the
//    smallest vertex of a component is never hooked.  After every edge has been processed both ends of each edge
//    share a root, so each component is one tree, rooted at its smallest vertex.
//  * After the finish parent[v] = root(v) = the smallest vertex of v's component.  That label does not depend on the
//    edge order, the thread schedule, how the edges were split over calls, or how many GPUs produced them.
//
// The finish is pointer jumping in rounds, one launch per round: every v sets parent[v] = parent[parent[v]].  Only
// v's own thread writes parent[v] in a round, so a final root is never overwritten, and a read of a slot another
// thread updates in the same round returns an ancestor either way.  A round at least halves every vertex's distance
// to its root, and a tree of n vertices is less than n deep, so ceil(log2 n) rounds always suffice: the time is
// bounded whatever shape the union left.  (A single pass in which every thread walks to its root with path halving
// is as fast on shallow trees but, on a chain the union built from a path given in descending order, its run time
// depended on the thread schedule and reached seconds.)
//
// Both kernels read parent[] at random: they are bound by the latency of random global accesses, not by bandwidth.
#include "common.cuh"

namespace emr2a {

__device__ __forceinline__ int64_t parent_load(const int64_t* p, int64_t v) {
  return *reinterpret_cast<const volatile int64_t*>(p + v);
}

// Root of v with path halving: every visited vertex is pointed at its grandparent on the way up.
__device__ __forceinline__ int64_t find_root(int64_t* parent, int64_t v) {
  int64_t p = parent_load(parent, v);
  while (p != v) {
    const int64_t gp = parent_load(parent, p);
    if (gp == p) return p;
    *reinterpret_cast<volatile int64_t*>(parent + v) = gp;
    v = gp;
    p = parent_load(parent, v);
  }
  return v;
}

__global__ void __launch_bounds__(256) components_union_kernel(int64_t* parent, int64_t n,
                                                               const int64_t* __restrict__ edges, int64_t m,
                                                               unsigned long long* __restrict__ bad_edges) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < m; e += stride) {
    const int64_t a = edges[2 * e], b = edges[2 * e + 1];
    if (a < 0 || a >= n || b < 0 || b >= n) {          // checked before parent[] is touched
      atomicAdd(bad_edges, 1ull);
      continue;
    }
    int64_t ra = find_root(parent, a), rb = find_root(parent, b);
    while (ra != rb) {
      const int64_t lo = ra < rb ? ra : rb, hi = ra < rb ? rb : ra;
      const int64_t old = static_cast<int64_t>(atomicCAS(reinterpret_cast<unsigned long long*>(parent + hi),
                                                         static_cast<unsigned long long>(hi),
                                                         static_cast<unsigned long long>(lo)));
      if (old == hi) break;
      ra = find_root(parent, old);                      // hi was hooked meanwhile: climb from where it went
      rb = find_root(parent, lo);
    }
  }
}

// One round of pointer jumping: parent[v] = parent[parent[v]].
__global__ void __launch_bounds__(256) components_jump_kernel(int64_t* parent, int64_t n) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t v = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; v < n; v += stride) {
    const int64_t p = parent_load(parent, v);
    const int64_t gp = parent_load(parent, p);
    if (gp != p) *reinterpret_cast<volatile int64_t*>(parent + v) = gp;
  }
}

static unsigned grid_for(int64_t items) {
  const int64_t want = (items + 255) / 256, cap = static_cast<int64_t>(sm_count()) * 16;
  return static_cast<unsigned>(want < cap ? want : cap);
}

// Row numbers travel in the low 32 bits of the packed keys as 0xFFFFFFFF - row, so a row set has fewer than that
// many rows.
static const int64_t kMaxVertices = 0xFFFFFFFFLL;

}  // namespace emr2a

using namespace emr2a;

extern "C" int emr2a_components_union(int64_t* parent, int64_t n, const int64_t* edges, int64_t m,
                                      uint64_t* bad_edges_out, void* stream) {
  if (n < 0 || m < 0 || (n > 0 && !parent) || (m > 0 && (!edges || !bad_edges_out)))
    return fail(EMR2A_ERR_INVALID, "components_union: bad arguments (n=%lld m=%lld)", (long long)n, (long long)m);
  if (n >= kMaxVertices)
    return fail(EMR2A_ERR_INVALID, "components_union: n=%lld must be below 2^32 - 1", (long long)n);
  if (m == 0) return EMR2A_OK;
  components_union_kernel<<<grid_for(m), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      parent, n, edges, m, reinterpret_cast<unsigned long long*>(bad_edges_out));
  EMR2A_LAUNCH_CHECK("components_union_kernel");
  return EMR2A_OK;
}

extern "C" int emr2a_components_finish(int64_t* parent, int64_t n, void* stream) {
  if (n < 0 || (n > 0 && !parent))
    return fail(EMR2A_ERR_INVALID, "components_finish: bad arguments (n=%lld)", (long long)n);
  if (n >= kMaxVertices)
    return fail(EMR2A_ERR_INVALID, "components_finish: n=%lld must be below 2^32 - 1", (long long)n);
  if (n == 0) return EMR2A_OK;
  int rounds = 1;                                       // 2^rounds >= n > the depth of any tree
  while ((int64_t(1) << rounds) < n) ++rounds;
  for (int r = 0; r < rounds; ++r) {
    components_jump_kernel<<<grid_for(n), 256, 0, static_cast<cudaStream_t>(stream)>>>(parent, n);
    EMR2A_LAUNCH_CHECK("components_jump_kernel");
  }
  return EMR2A_OK;
}
