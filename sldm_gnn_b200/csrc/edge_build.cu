// edge_build.cu -- proximity edges between vehicle trajectories (SURVEY 8f rank 4).
//
// Reference: the O(V^2 T) Python double loop of src/gbuilder.py:88-112 (offline packs) and :244-268
// (GraphOnlineCreator, the per-window cost of rcv.py:77).  For every ORDERED pair (i, j), i != j:
//   dists = || x[i,:,0:2] - x[j,:,0:2] ||_2 over the frames where both presence flags x[.,:,4] exceed 0.5
//   edge (i, j) exists iff dists is non-empty and min(dists) <= m_radius
//   edge_attr = [min, max, mean, mean of squares] of dists (float32, numpy's pairwise summation)
// Edges come out in (i, j) lexicographic order.  Here: one CTA per source vehicle i; pass 1 counts the edges of every
// row, a single-CTA scan turns the counts into offsets, pass 2 recomputes the pair statistics and writes each row's edges
// in ascending j (block-wide exclusive scan of the flags per chunk of 256 targets): deterministic, no atomics.
// Any number of frames: both trajectories are read through L1 (the source's loads are warp-uniform broadcasts), min / max
// are taken over squared distances (sqrt_rn is monotone, so sqrt(min s) == min sqrt(s) bit for bit), and the sums are
// streamed through numpy's pairwise-summation tree, so no per-thread or shared storage grows with T.
// Bound: FP32 issue and L1/L2 traffic, linear in the V^2 T pair-frames (DESIGN.md §5, "Proximity edges").
#include "common.cuh"
#include <math.h>

namespace sldm {

// numpy's float32 pairwise_sum (numpy/_core/src/umath/loops_utils.h.src), which np.add.reduce and ndarray.mean use:
//   n < 8:        sequential from 0
//   8 <= n <= 128: eight running sums over whole blocks of 8, combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)),
//                  then the remainder sequentially
//   n > 128:      pw(a, n2) + pw(a + n2, n - n2) with n2 = n/2 rounded down to a multiple of 8
constexpr int kEbLeaf = 128;
__host__ __device__ constexpr int np_pw_split(int n) { return n / 2 - (n / 2) % 8; }
// depth of the recursion for n elements; the right half is never the smaller one, so it sets the depth
constexpr int np_pw_depth(int n) { return n <= kEbLeaf ? 0 : 1 + np_pw_depth(n - np_pw_split(n)); }
constexpr int kEbStack = np_pw_depth(INT32_MAX);   // 25 levels cover every n an int32 frame count allows
static_assert(kEbStack <= 32, "path bits of the summation tree must fit in a uint32_t");

// squared distance of frame (a, b), rounded like np.linalg.norm(axis=1) before its sqrt: unfused dx*dx + dy*dy
__device__ __forceinline__ float sq_dist(const float* a, const float* b) {
  const float dx = __fsub_rn(__ldg(a), __ldg(b)), dy = __fsub_rn(__ldg(a + 1), __ldg(b + 1));
  return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
}
__device__ __forceinline__ bool co_present(const float* a, const float* b) { return __ldg(a + 4) > 0.5f && __ldg(b + 4) > 0.5f; }

// the next co-present distance at or after frame cursors (a, b), which then move past it; one must exist
__device__ __forceinline__ float next_dist(const float*& a, const float*& b, int64_t F) {
  for (;;) {
    const bool on = co_present(a, b);
    const float s = on ? sq_dist(a, b) : 0.f;
    a += F; b += F;
    if (on) return __fsqrt_rn(s);
  }
}

__device__ __forceinline__ float tree8(const float (&r)[8]) {
  return __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])), __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
}

// numpy's pairwise sums of the n co-present distances d of trajectories a, b (frame stride F) and of d*d, in one walk.
// The leaves of the recursion (<= 128 elements) are summed as their elements arrive; a finished leaf is added to the
// left halves waiting on the stack in the tree's post-order, so every addition is numpy's, in numpy's order.
// Running sums start at 0: 0 + a == a for the non-negative d and d*d, so a leaf needs no special first block.
__device__ __forceinline__ float2 pair_sums(const float* a, const float* b, int64_t F, int n) {
  float stk_s[kEbStack], stk_q[kEbStack];   // sum of the finished left half at each level of the current path
  uint32_t right = 0;                       // bit l: the node at depth l+1 of the path is its parent's right half
  int depth = 0, m = n;                     // m: size of the node being descended into
  float s, q;
  for (;;) {
    while (m > kEbLeaf) { m = np_pw_split(m); ++depth; }
    float r[8], rq[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { r[k] = 0.f; rq[k] = 0.f; }
    for (int g = m >> 3; g > 0; --g) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float d = next_dist(a, b, F);
        r[k] = __fadd_rn(r[k], d); rq[k] = __fadd_rn(rq[k], __fmul_rn(d, d));
      }
    }
    s = tree8(r); q = tree8(rq);               // 0 when m < 8: numpy's sequential sum from 0
    for (int k = m & 7; k > 0; --k) {
      const float d = next_dist(a, b, F);
      s = __fadd_rn(s, d); q = __fadd_rn(q, __fmul_rn(d, d));
    }
    while (depth > 0 && ((right >> (depth - 1)) & 1u)) {   // right half done: pw(left) + pw(right), up the tree
      --depth;
      right &= ~(1u << depth);
      s = __fadd_rn(stk_s[depth], s); q = __fadd_rn(stk_q[depth], q);
    }
    if (depth == 0) break;
    stk_s[depth - 1] = s; stk_q[depth - 1] = q;            // left half done: park it, descend into the right half
    right |= 1u << (depth - 1);
    int p = n;                                              // size of the parent, from the root along the path
    for (int l = 0; l < depth - 1; ++l) { const int h = np_pw_split(p); p = ((right >> l) & 1u) ? p - h : h; }
    m = p - np_pw_split(p);
  }
  return make_float2(s, q);
}

// T <= 128: whatever n is, numpy sums the window's distances as one leaf, so a single walk gives n, the squared min /
// max and both sums.  Elements are taken eight at a time; the first incomplete block is numpy's sequential tail.
struct LeafStats { int n; float s_mn, s_mx; float2 sums; };
__device__ __forceinline__ LeafStats pair_stats_one_leaf(const float* a, const float* b, int64_t F, int T) {
  LeafStats st; st.n = 0; st.s_mn = INFINITY; st.s_mx = 0.f;
  float r[8], rq[8], v[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { r[k] = 0.f; rq[k] = 0.f; }
  int t = 0, got;
  for (;;) {
    got = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      v[k] = 0.f;
      if (got == k) {
        while (t < T && !co_present(a, b)) { a += F; b += F; ++t; }
        if (t < T) {
          const float s = sq_dist(a, b);
          st.s_mn = fminf(st.s_mn, s); st.s_mx = fmaxf(st.s_mx, s);
          v[k] = __fsqrt_rn(s); ++got;
          a += F; b += F; ++t;
        }
      }
    }
    if (got < 8) break;
#pragma unroll
    for (int k = 0; k < 8; ++k) { r[k] = __fadd_rn(r[k], v[k]); rq[k] = __fadd_rn(rq[k], __fmul_rn(v[k], v[k])); }
    st.n += 8;
  }
  float s = tree8(r), q = tree8(rq);
#pragma unroll
  for (int k = 0; k < 7; ++k)
    if (k < got) { s = __fadd_rn(s, v[k]); q = __fadd_rn(q, __fmul_rn(v[k], v[k])); }
  st.n += got;
  st.sums = make_float2(s, q);
  return st;
}

template <bool FILL>
__global__ void __launch_bounds__(256)
k_edge_rows(const float* __restrict__ x, int V, int T, int F, float radius, int32_t* __restrict__ rowcnt,
            const int32_t* __restrict__ rowoff, int64_t* __restrict__ edge_index, int64_t E_cap,
            float* __restrict__ edge_attr) {
  __shared__ int s_scan[256 / 32 + 1];
  const int i = blockIdx.x;
  const int64_t row = (int64_t)T * F;
  const float* xi = x + (int64_t)i * row;
  int run = FILL ? rowoff[i] : 0;                 // edges of this row written so far (uniform across the CTA)
  for (int j0 = 0; j0 < V; j0 += 256) {
    const int j = j0 + threadIdx.x;
    const float* xj = x + (int64_t)min(j, V - 1) * row;
    int n = 0;
    float s_mn = INFINITY, s_mx = 0.f;            // over squared distances
    float2 sums = make_float2(0.f, 0.f);
    if (FILL && T <= kEbLeaf) {
      if (j < V && j != i) {
        const LeafStats st = pair_stats_one_leaf(xi, xj, F, T);
        n = st.n; s_mn = st.s_mn; s_mx = st.s_mx; sums = st.sums;
      }
    } else if (j < V && j != i) {
      const float* a = xi; const float* b = xj;
      for (int t = 0; t < T; ++t, a += F, b += F) {
        if (co_present(a, b)) {
          const float s = sq_dist(a, b);
          s_mn = fminf(s_mn, s);
          if (FILL) s_mx = fmaxf(s_mx, s);
          ++n;
        }
      }
    }
    const float mn = __fsqrt_rn(s_mn);
    const int flag = (n > 0 && mn <= radius) ? 1 : 0;
    int total;
    const int pre = block_exclusive_scan_256(flag, total, s_scan);
    if (FILL && flag) {
      if (T > kEbLeaf) sums = pair_sums(xi, xj, F, n);   // n is known now: stream the frames through numpy's tree
      const int64_t e = run + pre;
      edge_index[e] = i;
      edge_index[E_cap + e] = j;
      *reinterpret_cast<float4*>(edge_attr + 4 * e) =
          make_float4(mn, __fsqrt_rn(s_mx), __fdiv_rn(sums.x, (float)n), __fdiv_rn(sums.y, (float)n));
    }
    run += total;
  }
  if (!FILL && threadIdx.x == 0) rowcnt[i] = run;
}

// offsets[i] = exclusive prefix of counts; offsets[V] = total; single CTA (V is a few hundred .. a few thousand)
__global__ void __launch_bounds__(256)
k_edge_offsets(const int32_t* __restrict__ cnt, int V, int32_t* __restrict__ off) {
  __shared__ int s_scan[256 / 32 + 1];
  int carry = 0;
  for (int c = 0; c < V; c += 256) {
    const int i = c + threadIdx.x;
    const int v = i < V ? cnt[i] : 0;
    int total;
    const int p = block_exclusive_scan_256(v, total, s_scan);
    if (i < V) off[i] = carry + p;
    carry += total;
  }
  if (threadIdx.x == 0) off[V] = carry;
}

}  // namespace sldm

using namespace sldm;

// Pass 1: counts[V] and offsets[V+1] (offsets[V] = number of edges E; the host reads it to size the outputs).
extern "C" int sldm_edge_build_count(const float* x, int64_t V, int32_t T, int32_t F, float m_radius,
                                     int32_t* counts, int32_t* offsets, sldm_stream_t stream) {
  SLDM_REQUIRE(V >= 0 && T >= 0, SLDM_EINVAL, "sldm_edge_build_count: negative size");
  SLDM_REQUIRE(F >= 5, SLDM_ESHAPE, "sldm_edge_build_count: need >= 5 temporal features (X, Y, ., ., presence), got %d", F);
  SLDM_REQUIRE(V < ((int64_t)1 << 24), SLDM_EUNSUPPORTED, "sldm_edge_build_count: too many vehicles");
  SLDM_REQUIRE(offsets != nullptr && (V == 0 || (x != nullptr && counts != nullptr)), SLDM_EINVAL, "sldm_edge_build_count: NULL pointer");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (V > 0) {
    k_edge_rows<false><<<(unsigned)V, 256, 0, s>>>(x, (int)V, T, F, m_radius, counts, nullptr, nullptr, 0, nullptr);
    SLDM_LAUNCH_CHECK("k_edge_rows<count>");
  }
  k_edge_offsets<<<1, 256, 0, s>>>(counts, (int)V, offsets);
  SLDM_LAUNCH_CHECK("k_edge_offsets");
  return SLDM_OK;
}

// Pass 2: edge_index int64 [2, E] and edge_attr fp32 [E, 4] (16-byte aligned), E = offsets[V] as read by the host.
extern "C" int sldm_edge_build_fill(const float* x, int64_t V, int32_t T, int32_t F, float m_radius,
                                    const int32_t* offsets, int64_t E, int64_t* edge_index, float* edge_attr,
                                    sldm_stream_t stream) {
  SLDM_REQUIRE(V >= 0 && T >= 0 && E >= 0, SLDM_EINVAL, "sldm_edge_build_fill: negative size");
  SLDM_REQUIRE(F >= 5, SLDM_ESHAPE, "sldm_edge_build_fill: need >= 5 temporal features, got %d", F);
  if (V == 0 || E == 0) return SLDM_OK;
  SLDM_REQUIRE(x && offsets && edge_index && edge_attr, SLDM_EINVAL, "sldm_edge_build_fill: NULL pointer");
  SLDM_REQUIRE((reinterpret_cast<uintptr_t>(edge_attr) & 15u) == 0, SLDM_EINVAL, "sldm_edge_build_fill: edge_attr must be 16-byte aligned");
  k_edge_rows<true><<<(unsigned)V, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, (int)V, T, F, m_radius, nullptr, offsets, edge_index, E, edge_attr);
  SLDM_LAUNCH_CHECK("k_edge_rows<fill>");
  return SLDM_OK;
}
