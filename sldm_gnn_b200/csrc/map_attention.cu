// map_attention.cu -- MapSpatialAttention (src/models/map/mapattention.py:21-56), the step between the map-graph
// SageBlock and the vehicle-graph SageBlock (src/models/grusage.py:171-179).  SURVEY 8f rank 3.
//
// Reference (plain torch, 7 launches, materialises [B,S,2] and [B,S]):
//   diff = pos[:,None,:] - centroids[None,:,:] ; dists = norm(diff, dim=2)            # [B,S]
//   neg, idx = topk(-dists, k) ; kd = -neg                                            # K nearest segments
//   score = attn_mlp(kd[...,None]) = W2 . relu(W1*kd + b1) + b2                       # Linear(1,H) -> ReLU -> Linear(H,1)
//   w = softmax(score, dim=1) ; ctx = sum_k w_k * emb[idx_k]                          # [B,D]
// Here: one warp per vehicle scans the centroids (staged in shared memory, coalesced), keeps a per-lane sorted list
// of the K nearest, the warp merges the 32 lists with K rounds of a 64-bit (distance, index) min-reduction, then the
// MLP, softmax and the weighted sum of K embedding rows run in registers.  Nothing of size B*S ever touches memory.
// Ties in distance are broken towards the LOWER segment index (torch.topk leaves that unspecified).
// Backward: per-vehicle kernel for the softmax / MLP chain (parameter gradients as per-CTA partials, reduced in fixed
// order), and a deterministic gather for d_emb over a membership CSR keyed by the selected segment (no atomics).
// Bound: the scan is FP32-issue bound (B*S distance evaluations), everything else HBM: B*(8 + K*D*4 + D*4) bytes.
#include "common.cuh"
#include <algorithm>
#include <math.h>

namespace sldm {

constexpr int kMaK = 8;          // K <= 8
constexpr int kMaH = 64;         // hidden width of the score MLP <= 64 (reference: 16)
constexpr int kMaTile = 4096;    // centroids per shared-memory tile (32 KB); a map that fits is loaded once per CTA

__device__ __forceinline__ unsigned long long pack_key(float d, int idx) {
  // d >= 0: its bit pattern orders like the value; NaN sorts last
  return ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)idx;
}

template <int K>
__global__ void __launch_bounds__(256)
k_map_attention_fwd(const float* __restrict__ pos, int64_t B, const float2* __restrict__ cent, int S,
                    const float* __restrict__ emb, int D, const float* __restrict__ W1, const float* __restrict__ b1,
                    const float* __restrict__ W2, const float* __restrict__ b2, int H,
                    float* __restrict__ ctx, int64_t* __restrict__ idx_out, float* __restrict__ dist_out,
                    float* __restrict__ w_out) {
  __shared__ float2 s_c[kMaTile];
  __shared__ float s_w1[kMaH], s_b1[kMaH], s_w2[kMaH];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int h = threadIdx.x; h < H; h += 256) { s_w1[h] = W1[h]; s_b1[h] = b1[h]; s_w2[h] = W2[h]; }
  // persistent over groups of 8 vehicles (one per warp).  A map of at most kMaTile segments is staged ONCE per CTA -- with
  // one group per CTA the kernel spent its time filling shared memory (16 KB per 8 vehicles) rather than scanning.
  const bool single = S <= kMaTile;
  if (single) {
    for (int i = threadIdx.x; i < S; i += 256) s_c[i] = __ldg(cent + i);
  }
  __syncthreads();
  for (int64_t vb = blockIdx.x; vb * 8 < B; vb += gridDim.x) {
  const int64_t b = vb * 8 + warp;
  const bool live = b < B;
  const float px = live ? __ldg(pos + 2 * b) : 0.f, py = live ? __ldg(pos + 2 * b + 1) : 0.f;
  // The K best (distance, index) keys of the WARP live in lanes 0..K-1 (ascending).  A round looks at 32 segments, one
  // per lane; a ballot on the squared distance against the warp's current K-th best finds the few that can enter, and each
  // of those is inserted with a warp-uniform shift (no per-lane lists, no divergence: per-lane sorted lists cost 5.4k warp
  // instructions per vehicle at 15/32 active lanes -- ncu, profiles/r01j).
  unsigned long long L = ~0ull;
  float thr2 = INFINITY;                           // squared distance a candidate must not exceed
  for (int t0 = 0; t0 < S; t0 += kMaTile) {
    const int tn = min(kMaTile, S - t0);
    if (!single) {
      __syncthreads();
      for (int i = threadIdx.x; i < tn; i += 256) s_c[i] = __ldg(cent + t0 + i);
      __syncthreads();
    }
    if (live) {
      int i0 = 0;
      if (t0 == 0) {
        // bootstrap: the first 32 segments are sorted with a warp bitonic network (15 compare-exchange steps) instead of
        // 32 serial insertions; lanes 0..K-1 then hold the K best so far
        unsigned long long key = ~0ull;
        if (lane < tn) {
          const float dx = __fsub_rn(px, s_c[lane].x), dy = __fsub_rn(py, s_c[lane].y);
          key = pack_key(__fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy))), lane);
        }
#pragma unroll
        for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
          for (int j = k >> 1; j > 0; j >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, j);
            const bool take_min = ((lane & k) == 0) == ((lane & j) == 0);
            key = (take_min == (other < key)) ? other : key;
          }
        }
        L = lane < K ? key : ~0ull;
        const unsigned long long worst = __shfl_sync(0xffffffffu, L, K - 1);
        if (worst != ~0ull) {
          const float wd = __uint_as_float((unsigned)(worst >> 32));
          thr2 = __fmul_rn(__fmul_rn(wd, wd), 1.000001f);
        }
        i0 = 32;
      }
      // afterwards: 64 segments per round (two per lane): one ballot per 32, the filter rarely fires
      for (; i0 < tn; i0 += 64) {
        float d2[2];
        unsigned pass[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int i = i0 + 32 * h + lane;
          d2[h] = INFINITY;
          if (i < tn) {
            const float dx = __fsub_rn(px, s_c[i].x), dy = __fsub_rn(py, s_c[i].y);
            // dx*dx + dy*dy without FMA contraction: the same operations torch.norm performs
            d2[h] = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
          }
          pass[h] = __ballot_sync(0xffffffffu, i < tn && d2[h] <= thr2);
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          unsigned m = pass[h];
          while (m) {
            const int srcl = __ffs(m) - 1;
            m &= m - 1;
            const float c2 = __shfl_sync(0xffffffffu, d2[h], srcl);
            if (c2 <= thr2) {                      // the threshold may have tightened inside this round (uniform)
              const unsigned long long key = pack_key(__fsqrt_rn(c2), t0 + i0 + 32 * h + srcl);
              const bool lt = L < key;
              const unsigned long long prev = __shfl_up_sync(0xffffffffu, L, 1);
              const int prevlt = __shfl_up_sync(0xffffffffu, (int)lt, 1);
              if (lane < K) L = lt ? L : ((lane == 0 || prevlt) ? key : prev);
              const unsigned long long worst = __shfl_sync(0xffffffffu, L, K - 1);
              if (worst != ~0ull) {                // list full: tighten the filter (inflated by a few ulp so that a
                const float wd = __uint_as_float((unsigned)(worst >> 32));        // candidate that would TIE after the
                thr2 = __fmul_rn(__fmul_rn(wd, wd), 1.000001f);                    // rounding of sqrt still gets in)
              }
            }
          }
        }
      }
    }
  }
  if (live) {
  const float kd = __uint_as_float((unsigned)(L >> 32));          // lane k (< K): the k-th nearest
  const int kidx = (int)(unsigned)(L & 0xffffffffu);
  // score MLP + softmax on lanes 0..K-1
  float score = -INFINITY;
  if (lane < K) {
    float acc = 0.f;
    for (int h = 0; h < H; ++h) {
      const float pre = fmaf(s_w1[h], kd, s_b1[h]);
      acc = fmaf(s_w2[h], pre > 0.f ? pre : 0.f, acc);
    }
    score = acc + __ldg(b2);
  }
  float mx = score;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  const float ex = lane < K ? expf(score - mx) : 0.f;
  float den = ex;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) den += __shfl_xor_sync(0xffffffffu, den, o);
  const float w = __fdiv_rn(ex, den);
  if (lane < K) {
    idx_out[b * K + lane] = kidx;
    dist_out[b * K + lane] = kd;
    w_out[b * K + lane] = w;
  }
  // ctx = sum_k w_k emb[idx_k]   (k ascending); the broadcasts happen before the column loop (not every lane enters it)
  float wk[K]; int ik[K];
#pragma unroll
  for (int k = 0; k < K; ++k) { wk[k] = __shfl_sync(0xffffffffu, w, k); ik[k] = __shfl_sync(0xffffffffu, kidx, k); }
  for (int c = lane; c < D; c += 32) {
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) acc = fmaf(wk[k], __ldg(emb + (int64_t)ik[k] * D + c), acc);
    ctx[b * D + c] = acc;
  }
  }   // live
  }   // vehicle groups
}

// ---------------------------------------------------------------------------------------------------------------
// Grid path.  The map is fixed for the life of the module (a registered buffer of the reference class), the positions
// change every call: the centroids are binned ONCE into a uniform G x G grid over their bounding box (about four per
// cell), and a query walks square rings of cells around its own cell until the K-th best distance is provably smaller
// than the distance to anything not yet visited.  ~40 candidates per vehicle instead of S, the same (distance, index)
// keys as the exhaustive scan above, hence bit-identical idx / dist / w / ctx (tests/test_map_attention.py).
//   grid buffer: [MapGridHeader 64 B][cell_start int32 G*G+1][cursor int32 G*G][entries float4 S = {x, y, index, -}]
// Cell of a point: clamp(floor((v - min) / w), 0, G-1) per axis; cell ids are row-major, so a run of cells of one grid
// row is one contiguous run of entries.  `slack` (4e-6 x the largest coordinate magnitude, ~30x the rounding error of
// the cell arithmetic) is taken off every geometric bound: a larger slack only costs an extra ring, never an answer.
struct MapGridHeader { float minx, miny, wx, wy, inv_wx, inv_wy, slack; int32_t G; int32_t pad[8]; };
static_assert(sizeof(MapGridHeader) == 64, "grid header layout");
constexpr int kMaGridMax = 512;
// centroids per cell on average: with 4 the K = 5 nearest are almost always inside the 3 x 3 block around the own cell, so
// the lanes of a warp stop together (with 2, ~20% of the lanes needed a second ring and the other lanes idled through it)
constexpr double kMaCellLoad = 4.0;

struct MapGridLayout { int G; int64_t off_start, off_cursor, off_entries, total; };
static MapGridLayout map_grid_layout(int64_t S) {
  MapGridLayout L;
  int64_t g = (int64_t)ceil(sqrt((double)std::max<int64_t>(S, 1) / kMaCellLoad));
  L.G = (int)std::max<int64_t>(1, std::min<int64_t>(g, kMaGridMax));
  const int64_t cells = (int64_t)L.G * L.G;
  L.off_start = 64;
  L.off_cursor = L.off_start + align_bytes((cells + 1) * 4);
  L.off_entries = L.off_cursor + align_bytes(cells * 4);
  L.total = L.off_entries + align_bytes(std::max<int64_t>(S, 1) * 16);
  return L;
}

__device__ __forceinline__ int grid_coord(float v, float mn, float inv_w, int G) {
  const float f = floorf((v - mn) * inv_w);
  return (int)fminf(fmaxf(f, 0.f), (float)(G - 1));      // NaN -> 0
}

// one CTA: bounding box, counts, exclusive scan, fill.  Runs once per map.
__global__ void __launch_bounds__(1024)
k_map_grid_build(const float2* __restrict__ cent, int S, int G, MapGridHeader* __restrict__ hdr,
                 int* __restrict__ cell_start, int* __restrict__ cursor, float4* __restrict__ entries) {
  __shared__ float s_red[4][32];
  __shared__ int s_warp[33];
  __shared__ MapGridHeader s_h;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cells = G * G;
  float mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
  for (int i = tid; i < S; i += 1024) {
    const float2 c = cent[i];
    if (isfinite(c.x) && isfinite(c.y)) {
      mnx = fminf(mnx, c.x); mxx = fmaxf(mxx, c.x);
      mny = fminf(mny, c.y); mxy = fmaxf(mxy, c.y);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o)); mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
    mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o)); mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
  }
  if (lane == 0) { s_red[0][warp] = mnx; s_red[1][warp] = mxx; s_red[2][warp] = mny; s_red[3][warp] = mxy; }
  for (int i = tid; i < cells; i += 1024) cursor[i] = 0;
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < 32; ++w) {
      mnx = fminf(mnx, s_red[0][w]); mxx = fmaxf(mxx, s_red[1][w]);
      mny = fminf(mny, s_red[2][w]); mxy = fmaxf(mxy, s_red[3][w]);
    }
    if (!(mnx <= mxx)) { mnx = mxx = 0.f; mny = mxy = 0.f; }       // no finite centroid at all
    float wx = (mxx - mnx) / (float)G, wy = (mxy - mny) / (float)G;
    if (!(wx > 0.f) || !isfinite(wx)) wx = 1.f;                    // degenerate extent: everything in column 0
    if (!(wy > 0.f) || !isfinite(wy)) wy = 1.f;
    MapGridHeader h;
    h.minx = mnx; h.miny = mny; h.wx = wx; h.wy = wy; h.inv_wx = 1.f / wx; h.inv_wy = 1.f / wy;
    h.slack = 4e-6f * fmaxf(fmaxf(fabsf(mnx), fabsf(mxx)), fmaxf(fabsf(mny), fabsf(mxy)));
    h.G = G;
    for (int i = 0; i < 8; ++i) h.pad[i] = 0;
    s_h = h;
    *hdr = h;
  }
  __syncthreads();
  const MapGridHeader h = s_h;
  auto cell_of = [&](const float2 c) {
    if (!(isfinite(c.x) && isfinite(c.y))) return 0;
    return grid_coord(c.y, h.miny, h.inv_wy, G) * G + grid_coord(c.x, h.minx, h.inv_wx, G);
  };
  for (int i = tid; i < S; i += 1024) atomicAdd(&cursor[cell_of(cent[i])], 1);
  __syncthreads();
  // exclusive scan of the cell counts: a contiguous slice per thread, the 1024 slice totals scanned by warps
  const int per = (cells + 1023) / 1024;
  const int lo = min(tid * per, cells), hi = min(lo + per, cells);
  int sum = 0;
  for (int i = lo; i < hi; ++i) sum += cursor[i];
  int inc = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const int w = s_warp[lane];
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    s_warp[lane] = winc - w;
  }
  __syncthreads();
  int run = s_warp[warp] + inc - sum;
  for (int i = lo; i < hi; ++i) {
    const int c = cursor[i];
    cell_start[i] = run;
    cursor[i] = run;
    run += c;
  }
  if (tid == 0) cell_start[cells] = S;
  __syncthreads();
  // fill.  The order inside a cell is whatever the atomics give: the search keys are (distance, index), a total order,
  // so the selected set does not depend on the order of the visits.
  for (int i = tid; i < S; i += 1024) {
    const float2 c = cent[i];
    const int at = atomicAdd(&cursor[cell_of(c)], 1);
    entries[at] = make_float4(c.x, c.y, __int_as_float(i), 0.f);
  }
}

// thread = vehicle for the search and the score MLP; the context rows are then written warp-cooperatively (lane = column)
template <int K>
__global__ void __launch_bounds__(256, 5)
k_map_attention_grid_fwd(const float* __restrict__ pos, int64_t B, const MapGridHeader* __restrict__ hdr,
                         const int* __restrict__ cell_start, const float4* __restrict__ entries,
                         const float* __restrict__ emb, int D, const float* __restrict__ W1, const float* __restrict__ b1,
                         const float* __restrict__ W2, const float* __restrict__ b2, int H,
                         float* __restrict__ ctx, int64_t* __restrict__ idx_out, float* __restrict__ dist_out,
                         float* __restrict__ w_out) {
  __shared__ float s_w1[kMaH], s_b1[kMaH], s_w2[kMaH];
  __shared__ float2 s_sel[8][K][32];               // (softmax weight, element offset of the embedding row) per warp / k / vehicle
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int h = threadIdx.x; h < H; h += 256) { s_w1[h] = W1[h]; s_b1[h] = b1[h]; s_w2[h] = W2[h]; }
  __syncthreads();
  const int64_t b = (int64_t)blockIdx.x * 256 + threadIdx.x;
  const bool live = b < B;
  unsigned long long L[K];                         // the K best (distance, index) keys so far, ascending
#pragma unroll
  for (int k = 0; k < K; ++k) L[k] = ~0ull;
  if (live) {
    const float px = __ldg(pos + 2 * b), py = __ldg(pos + 2 * b + 1);
    const float minx = __ldg(&hdr->minx), miny = __ldg(&hdr->miny), wx = __ldg(&hdr->wx), wy = __ldg(&hdr->wy);
    const float slack = __ldg(&hdr->slack);
    const int G = __ldg(&hdr->G);
    const int cx = grid_coord(px, minx, __ldg(&hdr->inv_wx), G), cy = grid_coord(py, miny, __ldg(&hdr->inv_wy), G);
    float thr2 = INFINITY;                         // squared distance a candidate must not exceed
    auto scan = [&](int beg, int end) {
      for (int e = beg; e < end; ++e) {
        const float4 c = __ldg(entries + e);
        const float dx = __fsub_rn(px, c.x), dy = __fsub_rn(py, c.y);
        // dx*dx + dy*dy without FMA contraction: the same operations torch.norm performs
        const float d2 = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
        if (!(d2 > thr2)) {                        // (NaN passes: the exact key comparison below decides)
          const unsigned long long key = pack_key(__fsqrt_rn(d2), __float_as_int(c.z));
          if (key < L[K - 1]) {
            L[K - 1] = key;
#pragma unroll
            for (int k = K - 1; k > 0; --k) {
              const unsigned long long a = L[k - 1], bk = L[k];
              const bool sw = bk < a;
              L[k - 1] = sw ? bk : a;
              L[k] = sw ? a : bk;
            }
            if (L[K - 1] != ~0ull) {               // list full: tighten the filter (inflated by a few ulp so that a
              const float wd = __uint_as_float((unsigned)(L[K - 1] >> 32));   // candidate that would TIE after the
              thr2 = __fmul_rn(__fmul_rn(wd, wd), 1.000001f);                  // rounding of sqrt still gets in)
            }
          }
        }
      }
    };
    // the 3 x 3 block around the own cell first (three runs of entries, one per grid row), then ring by ring
    {
      const int xa = max(cx - 1, 0), xb = min(cx + 1, G - 1);
      for (int y = max(cy - 1, 0); y <= min(cy + 1, G - 1); ++y)
        scan(__ldg(cell_start + y * G + xa), __ldg(cell_start + y * G + xb + 1));
    }
    for (int r = 1;; ++r) {
      const int x0 = cx - r, x1 = cx + r, y0 = cy - r, y1 = cy + r;
      if (r > 1) {
        const int xa = max(x0, 0), xb = min(x1, G - 1);
        if (y0 >= 0) scan(__ldg(cell_start + y0 * G + xa), __ldg(cell_start + y0 * G + xb + 1));
        if (y1 <= G - 1) scan(__ldg(cell_start + y1 * G + xa), __ldg(cell_start + y1 * G + xb + 1));
        for (int y = max(y0 + 1, 0); y <= min(y1 - 1, G - 1); ++y) {
          if (x0 >= 0) scan(__ldg(cell_start + y * G + x0), __ldg(cell_start + y * G + x0 + 1));
          if (x1 <= G - 1) scan(__ldg(cell_start + y * G + x1), __ldg(cell_start + y * G + x1 + 1));
        }
      }
      // everything within Chebyshev ring r (clipped to the grid) has been seen.  A centroid not seen yet lies beyond one
      // of the block's four edges that are still inside the grid; its distance is at least the distance to that edge.
      float bound = INFINITY;
      bool more = false;
      if (x0 > 0) { more = true; bound = fminf(bound, px - (minx + (float)x0 * wx)); }
      if (x1 < G - 1) { more = true; bound = fminf(bound, (minx + (float)(x1 + 1) * wx) - px); }
      if (y0 > 0) { more = true; bound = fminf(bound, py - (miny + (float)y0 * wy)); }
      if (y1 < G - 1) { more = true; bound = fminf(bound, (miny + (float)(y1 + 1) * wy) - py); }
      if (!more) break;                            // the whole grid has been visited
      if (L[K - 1] != ~0ull && __uint_as_float((unsigned)(L[K - 1] >> 32)) < bound - slack) break;
    }
  }
  // score MLP + softmax per thread (same operation order as the exhaustive kernel: its warp butterfly adds pairs 4, 2, 1 apart)
  float w[K];
  int ki[K];
  {
    float kd[K], sc[K], ex8[8];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      kd[k] = __uint_as_float((unsigned)(L[k] >> 32));
      ki[k] = (int)(unsigned)(L[k] & 0xffffffffu);
      sc[k] = 0.f;
    }
    for (int h = 0; h < H; ++h) {
      const float w1 = s_w1[h], bb = s_b1[h], w2 = s_w2[h];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const float pre = fmaf(w1, kd[k], bb);
        sc[k] = fmaf(w2, pre > 0.f ? pre : 0.f, sc[k]);
      }
    }
    const float bias2 = __ldg(b2);
    float mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < K; ++k) { sc[k] += bias2; mx = fmaxf(mx, sc[k]); }
#pragma unroll
    for (int k = 0; k < 8; ++k) ex8[k] = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) ex8[k] = expf(sc[k] - mx);
    const float den = ((ex8[0] + ex8[4]) + (ex8[2] + ex8[6])) + ((ex8[1] + ex8[5]) + (ex8[3] + ex8[7]));
#pragma unroll
    for (int k = 0; k < K; ++k) w[k] = __fdiv_rn(ex8[k], den);
    if (live) {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        idx_out[b * K + k] = ki[k];
        dist_out[b * K + k] = kd[k];
        w_out[b * K + k] = w[k];
      }
    }
  }
  // ctx = sum_k w_k emb[idx_k]   (k ascending): the warp walks its 32 vehicles, lane = column.  (weight, row offset) pairs
  // go through shared memory: one broadcast 8-byte read per neighbour instead of two shuffles and 64-bit index arithmetic.
#pragma unroll
  for (int k = 0; k < K; ++k)
    s_sel[warp][k][lane] = make_float2(w[k], __uint_as_float(live ? (unsigned)ki[k] * (unsigned)D : 0u));
  __syncwarp();
  const int64_t b0 = (int64_t)blockIdx.x * 256 + warp * 32;
  const int nv = (int)min((int64_t)32, B - b0);
  if (D == 32) {
    const float* const e0 = emb + lane;
    float* const c0 = ctx + b0 * 32 + lane;
#pragma unroll 4
    for (int v = 0; v < nv; ++v) {
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const float2 t = s_sel[warp][k][v];
        acc = fmaf(t.x, __ldg(e0 + __float_as_uint(t.y)), acc);
      }
      c0[v * 32] = acc;
    }
  } else {
    for (int v = 0; v < nv; ++v) {
      for (int c = lane; c < D; c += 32) {
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const float2 t = s_sel[warp][k][v];
          acc = fmaf(t.x, __ldg(emb + __float_as_uint(t.y) + c), acc);
        }
        ctx[(b0 + v) * D + c] = acc;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------- backward --
// Three streaming kernels (all reductions in a fixed order, no atomics):
//   k_map_attention_bwd_ds   per vehicle: gw_k = <emb[idx_k], dctx_b>, ds_k = w_k (gw_k - sum_j w_j gw_j) = dL/dscore_k
//   k_map_attention_bwd_mlp  per vehicle: the score MLP's parameter gradients from (dist, ds), per-CTA partials
//                            part[cta][0:H] = dW1, [H:2H] = db1, [2H:3H] = dW2, [3H] = db2, summed by k_map_attention_reduce
//   k_map_attention_demb     d_emb[s,:] = sum over the (vehicle, k) pairs that selected segment s of w * dctx[vehicle,:]

// LPV lanes share a vehicle (LPV = 8: four vehicles per warp, float4 columns; LPV = 32: scalar columns, any D / alignment).
// The loop is latency bound (index -> embedding row -> dot product), so the indices, weights and the first dctx columns of
// the NEXT vehicle are fetched while the current one is reduced.
template <int K, int LPV>
__global__ void __launch_bounds__(256)
k_map_attention_bwd_ds(const float* __restrict__ dctx, int64_t B, const float* __restrict__ emb, int D,
                       const int64_t* __restrict__ idx, const float* __restrict__ wgt, float* __restrict__ ds_out) {
  constexpr int VPW = 32 / LPV;                    // vehicles per warp
  constexpr int CW = LPV == 8 ? 4 : 1;             // columns per lane and step
  const int lane = threadIdx.x & 31, sub = lane % LPV;
  const int c0 = CW * sub;
  const int64_t wglobal = ((int64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
  const int64_t stride = (((int64_t)gridDim.x * 256) >> 5) * VPW;
  const int64_t Bp = round_up<int64_t>(B, VPW);    // padded to whole warps so that the shuffles stay convergent
  unsigned off_n[K];
  float w_n[K];
  float4 g_n;
  auto fetch = [&](int64_t bb) {
    const bool live = bb < B;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      off_n[k] = live ? (unsigned)__ldg(idx + bb * K + k) * (unsigned)D : 0u;
      w_n[k] = live ? __ldg(wgt + bb * K + k) : 0.f;
    }
    g_n = make_float4(0.f, 0.f, 0.f, 0.f);
    if (live && c0 < D) {
      if constexpr (LPV == 8) g_n = __ldg(reinterpret_cast<const float4*>(dctx + bb * D + c0));
      else g_n.x = __ldg(dctx + bb * D + c0);
    }
  };
  int64_t b = wglobal * VPW + lane / LPV;
  if (b < Bp) fetch(b);
  for (; b < Bp; b += stride) {
    const bool live = b < B;
    unsigned off[K];
    float gw[K], wk[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { off[k] = off_n[k]; wk[k] = w_n[k]; gw[k] = 0.f; }
    float4 g = g_n;
    if (live) {
      for (int c = c0; c < D; c += 32) {
        if (c != c0) {
          if constexpr (LPV == 8) g = __ldg(reinterpret_cast<const float4*>(dctx + b * D + c));
          else g.x = __ldg(dctx + b * D + c);
        }
        if constexpr (LPV == 8) {
          float4 e[K];
#pragma unroll
          for (int k = 0; k < K; ++k) e[k] = __ldg(reinterpret_cast<const float4*>(emb + off[k] + c));
          if (c == c0 && b + stride < Bp) fetch(b + stride);
#pragma unroll
          for (int k = 0; k < K; ++k) gw[k] = fmaf(e[k].w, g.w, fmaf(e[k].z, g.z, fmaf(e[k].y, g.y, fmaf(e[k].x, g.x, gw[k]))));
        } else {
          float e[K];
#pragma unroll
          for (int k = 0; k < K; ++k) e[k] = __ldg(emb + off[k] + c);
          if (c == c0 && b + stride < Bp) fetch(b + stride);
#pragma unroll
          for (int k = 0; k < K; ++k) gw[k] = fmaf(e[k], g.x, gw[k]);
        }
      }
      if (c0 >= D && b + stride < Bp) fetch(b + stride);       // lanes beyond the columns of a narrow D
    } else if (b + stride < Bp) {
      fetch(b + stride);
    }
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int o = LPV / 2; o > 0; o >>= 1) gw[k] += __shfl_xor_sync(0xffffffffu, gw[k], o);
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) dot = fmaf(wk[k], gw[k], dot);
    float mine = 0.f;                              // lane `sub` (< K) of the group stores ds_sub
#pragma unroll
    for (int k = 0; k < K; ++k) mine = (sub == k) ? wk[k] * (gw[k] - dot) : mine;
    if (live && sub < K) ds_out[b * K + sub] = mine;
  }
}

// lane = (hidden unit, vehicle slot): HL lanes cover the hidden units (two per lane when H > 32), 32 / HL vehicles are in
// flight per warp.  The K terms of a vehicle cancel (sum_k ds_k = 0), so they are summed locally first and only the
// residual enters the running sums; every lane takes its vehicles in index order; CTAs own contiguous vehicle ranges.
__global__ void __launch_bounds__(256)
k_map_attention_bwd_mlp(const float* __restrict__ dist, const float* __restrict__ ds, int64_t B, int K, int64_t per_cta,
                        const float* __restrict__ W1, const float* __restrict__ b1, const float* __restrict__ W2,
                        int H, int HL, float* __restrict__ part) {
  __shared__ float s_p[8][3 * kMaH + 1];
  __shared__ float s_g[8][32][7];                  // per lane: a1[2], a2[2], a3[2], a4
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int EG = 32 / HL, hl = lane % HL, eg = lane / HL;
  float w1[2], bb[2], w2[2];
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int h = hl + 32 * q;
    const bool on = h < H && (q == 0 || HL == 32);
    w1[q] = on ? __ldg(W1 + h) : 0.f; bb[q] = on ? __ldg(b1 + h) : 0.f; w2[q] = on ? __ldg(W2 + h) : 0.f;
  }
  float a1[2] = {0.f, 0.f}, a2[2] = {0.f, 0.f}, a3[2] = {0.f, 0.f}, a4 = 0.f;
  const int64_t beg = (int64_t)blockIdx.x * per_cta, end = min(B, beg + per_cta);
  for (int64_t v0 = beg + warp * 32; v0 < end; v0 += 256) {
    const int64_t v = v0 + lane;
    float d_l[kMaK], s_l[kMaK];
#pragma unroll
    for (int k = 0; k < kMaK; ++k) {
      const bool on = v < end && k < K;
      d_l[k] = on ? __ldg(dist + v * K + k) : 0.f;
      s_l[k] = on ? __ldg(ds + v * K + k) : 0.f;              // ds = 0: a padded slot contributes nothing
    }
    for (int j = 0; j < HL; ++j) {                            // HL = 32 / EG rounds, EG vehicles per round
      const int src = j * EG + eg;
      float l1[2] = {0.f, 0.f}, l2[2] = {0.f, 0.f}, l3[2] = {0.f, 0.f}, l4 = 0.f;
#pragma unroll
      for (int k = 0; k < kMaK; ++k) {
        if (k < K) {
          const float d = __shfl_sync(0xffffffffu, d_l[k], src);
          const float g = __shfl_sync(0xffffffffu, s_l[k], src);
          l4 += g;
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            if (q == 1 && HL < 32) break;                      // H <= 32: one hidden unit per lane
            const float pre = fmaf(w1[q], d, bb[q]);
            const bool pos = pre > 0.f;
            l3[q] = fmaf(g, pos ? pre : 0.f, l3[q]);
            const float da = pos ? g * w2[q] : 0.f;
            l1[q] = fmaf(da, d, l1[q]);
            l2[q] += da;
          }
        }
      }
      a4 += l4;
#pragma unroll
      for (int q = 0; q < 2; ++q) { a1[q] += l1[q]; a2[q] += l2[q]; a3[q] += l3[q]; }
    }
  }
  // combine the element slots of a warp in slot order, then the warps in warp order
  s_g[warp][lane][0] = a1[0]; s_g[warp][lane][1] = a1[1]; s_g[warp][lane][2] = a2[0]; s_g[warp][lane][3] = a2[1];
  s_g[warp][lane][4] = a3[0]; s_g[warp][lane][5] = a3[1]; s_g[warp][lane][6] = a4;
  __syncwarp();
  if (lane < HL) {
    float t[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int e = 0; e < EG; ++e)
#pragma unroll
      for (int v = 0; v < 7; ++v) t[v] += s_g[warp][e * HL + lane][v];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int h = lane + 32 * q;
      if (h < H && (q == 0 || HL == 32)) { s_p[warp][h] = t[q]; s_p[warp][H + h] = t[2 + q]; s_p[warp][2 * H + h] = t[4 + q]; }
    }
    if (lane == 0) s_p[warp][3 * H] = t[6];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * H + 1; i += 256) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += s_p[w][i];
    part[(int64_t)blockIdx.x * (3 * H + 1) + i] = s;
  }
}

// one CTA per segment; members from the membership CSR in ascending position order.  A warp takes 32 members at a time
// (ids and weights loaded coalesced, broadcast by shuffle) so that the dctx row loads of a block are independent; the
// warps are combined in warp order (deterministic).
constexpr int kDembWarps = 4;   // 128-thread CTAs: 16 per SM, so a 2048-segment map is ONE wave and all segments walk the
                                // vehicles in step -- the K segments that share a dctx row find it in L2
template <int K>
__global__ void __launch_bounds__(32 * kDembWarps)
k_map_attention_demb(const float* __restrict__ dctx, int D, const float* __restrict__ wgt,
                     const int32_t* __restrict__ ptr, const int32_t* __restrict__ members, float* __restrict__ demb) {
  extern __shared__ float sm[];                    // [kDembWarps][D]
  const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int beg = __ldg(ptr + s), end = __ldg(ptr + s + 1);
  for (int c0 = 0; c0 < D; c0 += 32) {
    const int c = c0 + lane;
    const bool on = c < D;
    float acc = 0.f;
    // member ids and weights of the NEXT block are fetched while the 32 row loads of the current one are in flight
    int i0 = beg + warp * 32;
    int p_n = 0;
    float w_n = 0.f;
    if (i0 + lane < end) { p_n = __ldg(members + i0 + lane); w_n = __ldg(wgt + p_n); }
    for (; i0 < end; i0 += 32 * kDembWarps) {
      const float wp = w_n;
      const unsigned rowoff = (unsigned)(p_n / K) * (unsigned)D;       // B * D < 2^32 (checked on the host)
      const int cnt = min(32, end - i0);
      const int inext = i0 + 32 * kDembWarps + lane;
      p_n = 0; w_n = 0.f;
      if (inext < end) p_n = __ldg(members + inext);
      if (cnt == 32) {
        float r[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          // the shuffle is executed by ALL lanes, also those beyond column D (it sat inside the `on ?` branch once:
          // with D < 32 and a segment of >= 32 members the source lanes 16.. were not in the shuffle -> wild offsets)
          const unsigned ro = __shfl_sync(0xffffffffu, rowoff, j);
          r[j] = on ? __ldg(dctx + ro + c) : 0.f;
        }
        if (inext < end) w_n = __ldg(wgt + p_n);
#pragma unroll
        for (int j = 0; j < 32; ++j) acc = fmaf(__shfl_sync(0xffffffffu, wp, j), r[j], acc);
      } else {
        if (inext < end) w_n = __ldg(wgt + p_n);
        for (int j = 0; j < cnt; ++j) {
          const unsigned ro = __shfl_sync(0xffffffffu, rowoff, j);
          const float wj = __shfl_sync(0xffffffffu, wp, j);
          if (on) acc = fmaf(wj, __ldg(dctx + ro + c), acc);
        }
      }
    }
    if (on) sm[warp * D + c] = acc;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < D; c += 32 * kDembWarps) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kDembWarps; ++w) t += sm[w * D + c];
    demb[(int64_t)s * D + c] = t;
  }
}

// one warp per output: lanes stride over the partials (index order), then a fixed butterfly
__global__ void __launch_bounds__(256)
k_map_attention_reduce(const float* __restrict__ part, int nparts, int H, float* __restrict__ dW1,
                       float* __restrict__ db1, float* __restrict__ dW2, float* __restrict__ db2) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= 3 * H + 1) return;
  float s = 0.f;
  for (int k = lane; k < nparts; k += 32) s += part[(int64_t)k * (3 * H + 1) + i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) {
    if (i < H) dW1[i] = s; else if (i < 2 * H) db1[i - H] = s; else if (i < 3 * H) dW2[i - 2 * H] = s; else db2[0] = s;
  }
}

// ------------------------------------------------------------------------------------------------------ K > 8 --
// The kernels above keep K-long arrays per thread: the grid search a sorted list of K 64-bit keys (48 registers at K = 8,
// the cap of its __launch_bounds__(256, 5)), k_map_attention_bwd_ds K embedding rows in flight (116 registers at K = 8).
// A 32-key list alone would take 64 registers.  For 8 < K <= 32 every kernel below works with one WARP per vehicle and
// the warp's K best (distance, index) keys in lanes 0..K-1, the structure of k_map_attention_fwd.  Same keys, same
// distance arithmetic, same tie rule: the selected set is exactly the K nearest, whatever the visit order.
constexpr int kMaKWide = 32;
constexpr int64_t kMaCsrMax = ((int64_t)1 << 31) - ((int64_t)1 << 20);   // pairs of the int32 membership CSR

// Offers one candidate (squared distance c2, segment ci; both warp-uniform) to the warp's ascending list L (lanes
// 0..K-1) with a warp-uniform shift: a lane keeps its key if it is smaller, else takes the candidate (lane 0, or the left
// neighbour's key is smaller) or the left neighbour's key.  Then the filter is tightened to the new K-th best, inflated
// by a few ulp so that a candidate that would TIE after the rounding of sqrt still gets in.  NaN passes the filter: the
// exact key comparison decides, and a vehicle whose distances are all NaN still fills its list with valid indices.
__device__ __forceinline__ void ma_offer(unsigned long long& L, float& thr2, float c2, int ci, int lane, int K) {
  if (c2 > thr2) return;                           // the threshold may have tightened inside this round (uniform)
  const unsigned long long key = pack_key(__fsqrt_rn(c2), ci);
  const bool lt = L < key;
  const unsigned long long prev = __shfl_up_sync(0xffffffffu, L, 1);
  const int prevlt = __shfl_up_sync(0xffffffffu, (int)lt, 1);
  if (lane < K) L = lt ? L : ((lane == 0 || prevlt) ? key : prev);
  const unsigned long long worst = __shfl_sync(0xffffffffu, L, K - 1);
  if (worst != ~0ull) {
    const float wd = __uint_as_float((unsigned)(worst >> 32));
    thr2 = __fmul_rn(__fmul_rn(wd, wd), 1.000001f);
  }
}

// One round of up to 32 candidates, lane i holding (d2, ci) when `has`: a ballot against the threshold picks the few
// that can enter, and they are offered in lane order.
__device__ __forceinline__ void ma_round(unsigned long long& L, float& thr2, bool has, float d2, int ci, int lane, int K) {
  unsigned m = __ballot_sync(0xffffffffu, has && !(d2 > thr2));
  while (m) {
    const int src = __ffs(m) - 1;
    m &= m - 1;
    ma_offer(L, thr2, __shfl_sync(0xffffffffu, d2, src), __shfl_sync(0xffffffffu, ci, src), lane, K);
  }
}

// dx*dx + dy*dy without FMA contraction: the same operations torch.norm performs
__device__ __forceinline__ float ma_d2(float px, float py, float cx, float cy) {
  const float dx = __fsub_rn(px, cx), dy = __fsub_rn(py, cy);
  return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
}

// The epilogue of both K > 8 forward kernels, so that they return the same bits: the score MLP on lanes 0..K-1, the
// softmax max and denominator by the 32-lane butterfly, w = ex / den (IEEE), the saved tensors, then
// ctx = sum_k w_k emb[idx_k] as one FMA chain in ascending k, lane = column.  The (weight, row) pairs are broadcast through
// the warp's 32 slots of shared memory.  Called by the whole warp.
__device__ __forceinline__ void ma_wide_epilogue(unsigned long long L, int lane, int K, int64_t b,
                                                 const float* s_w1, const float* s_b1, const float* s_w2, int H,
                                                 const float* __restrict__ b2, const float* __restrict__ emb, int D,
                                                 float* s_wt, int* s_ix, float* __restrict__ ctx, int64_t* __restrict__ idx_out,
                                                 float* __restrict__ dist_out, float* __restrict__ w_out) {
  const float kd = __uint_as_float((unsigned)(L >> 32));          // lane k (< K): the k-th nearest
  const int kidx = (int)(unsigned)(L & 0xffffffffu);
  float score = -INFINITY;
  if (lane < K) {
    float acc = 0.f;
    for (int h = 0; h < H; ++h) {
      const float pre = fmaf(s_w1[h], kd, s_b1[h]);
      acc = fmaf(s_w2[h], pre > 0.f ? pre : 0.f, acc);
    }
    score = acc + __ldg(b2);
  }
  float mx = score;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  const float ex = lane < K ? expf(score - mx) : 0.f;
  float den = ex;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) den += __shfl_xor_sync(0xffffffffu, den, o);
  const float w = __fdiv_rn(ex, den);
  if (lane < K) {
    idx_out[b * K + lane] = kidx;
    dist_out[b * K + lane] = kd;
    w_out[b * K + lane] = w;
    s_wt[lane] = w;
    s_ix[lane] = kidx;
  }
  __syncwarp();
  if (D == 32) {
    float acc = 0.f;
#pragma unroll 8
    for (int k = 0; k < K; ++k) acc = fmaf(s_wt[k], __ldg(emb + (int64_t)s_ix[k] * 32 + lane), acc);
    ctx[b * 32 + lane] = acc;
  } else {
    for (int c = lane; c < D; c += 32) {
      float acc = 0.f;
#pragma unroll 8
      for (int k = 0; k < K; ++k) acc = fmaf(s_wt[k], __ldg(emb + (int64_t)s_ix[k] * D + c), acc);
      ctx[b * D + c] = acc;
    }
  }
  __syncwarp();                                    // the slots are rewritten by the warp's next vehicle
}

// Exhaustive scan for K > 8: k_map_attention_fwd with a runtime K and the shared insertion and epilogue.
__global__ void __launch_bounds__(256)
k_map_attention_fwd_wide(const float* __restrict__ pos, int64_t B, const float2* __restrict__ cent, int S,
                         const float* __restrict__ emb, int D, const float* __restrict__ W1, const float* __restrict__ b1,
                         const float* __restrict__ W2, const float* __restrict__ b2, int H, int K,
                         float* __restrict__ ctx, int64_t* __restrict__ idx_out, float* __restrict__ dist_out,
                         float* __restrict__ w_out) {
  __shared__ float2 s_c[kMaTile];
  __shared__ float s_w1[kMaH], s_b1[kMaH], s_w2[kMaH];
  __shared__ float s_wt[8][32];
  __shared__ int s_ix[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int h = threadIdx.x; h < H; h += 256) { s_w1[h] = W1[h]; s_b1[h] = b1[h]; s_w2[h] = W2[h]; }
  const bool single = S <= kMaTile;
  if (single) {
    for (int i = threadIdx.x; i < S; i += 256) s_c[i] = __ldg(cent + i);
  }
  __syncthreads();
  for (int64_t vb = blockIdx.x; vb * 8 < B; vb += gridDim.x) {
    const int64_t b = vb * 8 + warp;
    const bool live = b < B;                       // warp-uniform
    const float px = live ? __ldg(pos + 2 * b) : 0.f, py = live ? __ldg(pos + 2 * b + 1) : 0.f;
    unsigned long long L = ~0ull;
    float thr2 = INFINITY;
    for (int t0 = 0; t0 < S; t0 += kMaTile) {
      const int tn = min(kMaTile, S - t0);
      if (!single) {
        __syncthreads();
        for (int i = threadIdx.x; i < tn; i += 256) s_c[i] = __ldg(cent + t0 + i);
        __syncthreads();
      }
      if (live) {
        int i0 = 0;
        if (t0 == 0) {
          // bootstrap: the first 32 segments sorted by a warp bitonic network; S >= K, so lanes 0..K-1 get real keys
          unsigned long long key = ~0ull;
          if (lane < tn) key = pack_key(__fsqrt_rn(ma_d2(px, py, s_c[lane].x, s_c[lane].y)), lane);
#pragma unroll
          for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
            for (int j = k >> 1; j > 0; j >>= 1) {
              const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, j);
              const bool take_min = ((lane & k) == 0) == ((lane & j) == 0);
              key = (take_min == (other < key)) ? other : key;
            }
          }
          L = lane < K ? key : ~0ull;
          const float wd = __uint_as_float((unsigned)(__shfl_sync(0xffffffffu, L, K - 1) >> 32));
          thr2 = __fmul_rn(__fmul_rn(wd, wd), 1.000001f);
          i0 = 32;
        }
        for (; i0 < tn; i0 += 32) {
          const int i = i0 + lane;
          const bool has = i < tn;
          ma_round(L, thr2, has, has ? ma_d2(px, py, s_c[i].x, s_c[i].y) : INFINITY, t0 + i, lane, K);
        }
      }
    }
    if (live) ma_wide_epilogue(L, lane, K, b, s_w1, s_b1, s_w2, H, b2, emb, D, s_wt[warp], s_ix[warp], ctx, idx_out, dist_out, w_out);
  }
}

// Grid search for K > 8, one warp per vehicle: the cells of k_map_attention_grid_fwd in the same order (the 3 x 3 block
// around the own cell, then square rings) and the same stopping rule; a run of entries is taken 32 at a time, one per lane.
__global__ void __launch_bounds__(256)
k_map_attention_grid_fwd_wide(const float* __restrict__ pos, int64_t B, const MapGridHeader* __restrict__ hdr,
                              const int* __restrict__ cell_start, const float4* __restrict__ entries,
                              const float* __restrict__ emb, int D, const float* __restrict__ W1, const float* __restrict__ b1,
                              const float* __restrict__ W2, const float* __restrict__ b2, int H, int K,
                              float* __restrict__ ctx, int64_t* __restrict__ idx_out, float* __restrict__ dist_out,
                              float* __restrict__ w_out) {
  __shared__ float s_w1[kMaH], s_b1[kMaH], s_w2[kMaH];
  __shared__ float s_wt[8][32];
  __shared__ int s_ix[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int h = threadIdx.x; h < H; h += 256) { s_w1[h] = W1[h]; s_b1[h] = b1[h]; s_w2[h] = W2[h]; }
  __syncthreads();
  const int64_t b = (int64_t)blockIdx.x * 8 + warp;
  if (b >= B) return;                              // warp-uniform; no block barrier follows
  const float px = __ldg(pos + 2 * b), py = __ldg(pos + 2 * b + 1);
  const float minx = __ldg(&hdr->minx), miny = __ldg(&hdr->miny), wx = __ldg(&hdr->wx), wy = __ldg(&hdr->wy);
  const float slack = __ldg(&hdr->slack);
  const int G = __ldg(&hdr->G);
  const int cx = grid_coord(px, minx, __ldg(&hdr->inv_wx), G), cy = grid_coord(py, miny, __ldg(&hdr->inv_wy), G);
  unsigned long long L = ~0ull;
  float thr2 = INFINITY;
  auto scan = [&](int beg, int end) {
    for (int e0 = beg; e0 < end; e0 += 32) {
      const int e = e0 + lane;
      const bool has = e < end;
      float d2 = INFINITY;
      int ci = 0;
      if (has) {
        const float4 c = __ldg(entries + e);
        d2 = ma_d2(px, py, c.x, c.y);
        ci = __float_as_int(c.z);
      }
      ma_round(L, thr2, has, d2, ci, lane, K);
    }
  };
  {
    const int xa = max(cx - 1, 0), xb = min(cx + 1, G - 1);
    for (int y = max(cy - 1, 0); y <= min(cy + 1, G - 1); ++y)
      scan(__ldg(cell_start + y * G + xa), __ldg(cell_start + y * G + xb + 1));
  }
  for (int r = 1;; ++r) {
    const int x0 = cx - r, x1 = cx + r, y0 = cy - r, y1 = cy + r;
    if (r > 1) {
      const int xa = max(x0, 0), xb = min(x1, G - 1);
      if (y0 >= 0) scan(__ldg(cell_start + y0 * G + xa), __ldg(cell_start + y0 * G + xb + 1));
      if (y1 <= G - 1) scan(__ldg(cell_start + y1 * G + xa), __ldg(cell_start + y1 * G + xb + 1));
      for (int y = max(y0 + 1, 0); y <= min(y1 - 1, G - 1); ++y) {
        if (x0 >= 0) scan(__ldg(cell_start + y * G + x0), __ldg(cell_start + y * G + x0 + 1));
        if (x1 <= G - 1) scan(__ldg(cell_start + y * G + x1), __ldg(cell_start + y * G + x1 + 1));
      }
    }
    float bound = INFINITY;
    bool more = false;
    if (x0 > 0) { more = true; bound = fminf(bound, px - (minx + (float)x0 * wx)); }
    if (x1 < G - 1) { more = true; bound = fminf(bound, (minx + (float)(x1 + 1) * wx) - px); }
    if (y0 > 0) { more = true; bound = fminf(bound, py - (miny + (float)y0 * wy)); }
    if (y1 < G - 1) { more = true; bound = fminf(bound, (miny + (float)(y1 + 1) * wy) - py); }
    if (!more) break;                              // the whole grid has been visited
    const unsigned long long worst = __shfl_sync(0xffffffffu, L, K - 1);
    if (worst != ~0ull && __uint_as_float((unsigned)(worst >> 32)) < bound - slack) break;
  }
  ma_wide_epilogue(L, lane, K, b, s_w1, s_b1, s_w2, H, b2, emb, D, s_wt[warp], s_ix[warp], ctx, idx_out, dist_out, w_out);
}

// ds for K > 8, one warp per vehicle, lane = neighbour k: gw_k = <emb[idx_k], dctx_b> streams the lane's own embedding
// row (16-byte loads when VEC), sum_j w_j gw_j by the 32-lane butterfly (fixed order), ds_k = w_k (gw_k - sum_j w_j gw_j).
template <bool VEC>
__global__ void __launch_bounds__(256)
k_map_attention_bwd_ds_wide(const float* __restrict__ dctx, int64_t B, const float* __restrict__ emb, int D, int K,
                            const int64_t* __restrict__ idx, const float* __restrict__ wgt, float* __restrict__ ds_out) {
  const int lane = threadIdx.x & 31;
  const int64_t b = ((int64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
  if (b >= B) return;                              // warp-uniform
  const bool on = lane < K;
  const float wk = on ? __ldg(wgt + b * K + lane) : 0.f;
  float gw = 0.f;
  if (on) {
    const float* row = emb + __ldg(idx + b * K + lane) * (int64_t)D;
    const float* g = dctx + b * D;
    if constexpr (VEC) {
#pragma unroll 4
      for (int c = 0; c < D; c += 4) {
        const float4 e = __ldg(reinterpret_cast<const float4*>(row + c));
        const float4 x = __ldg(reinterpret_cast<const float4*>(g + c));
        gw = fmaf(e.w, x.w, fmaf(e.z, x.z, fmaf(e.y, x.y, fmaf(e.x, x.x, gw))));
      }
    } else {
#pragma unroll 4
      for (int c = 0; c < D; ++c) gw = fmaf(__ldg(row + c), __ldg(g + c), gw);
    }
  }
  float dot = wk * gw;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
  if (on) ds_out[b * K + lane] = wk * (gw - dot);
}

// The MLP gradients for K > 8: lanes and partials as in k_map_attention_bwd_mlp, but every lane reads its vehicle's K
// (dist, ds) pairs itself (the HL lanes of a vehicle slot read the same words).  The K terms of a vehicle are still summed
// locally before they enter the running sums (they cancel: sum_k ds_k = 0).
__global__ void __launch_bounds__(256)
k_map_attention_bwd_mlp_wide(const float* __restrict__ dist, const float* __restrict__ ds, int64_t B, int K, int64_t per_cta,
                             const float* __restrict__ W1, const float* __restrict__ b1, const float* __restrict__ W2,
                             int H, int HL, float* __restrict__ part) {
  __shared__ float s_p[8][3 * kMaH + 1];
  __shared__ float s_g[8][32][7];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int EG = 32 / HL, hl = lane % HL, eg = lane / HL;
  float w1[2], bb[2], w2[2];
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int h = hl + 32 * q;
    const bool on = h < H && (q == 0 || HL == 32);
    w1[q] = on ? __ldg(W1 + h) : 0.f; bb[q] = on ? __ldg(b1 + h) : 0.f; w2[q] = on ? __ldg(W2 + h) : 0.f;
  }
  float a1[2] = {0.f, 0.f}, a2[2] = {0.f, 0.f}, a3[2] = {0.f, 0.f}, a4 = 0.f;
  const int64_t beg = (int64_t)blockIdx.x * per_cta, end = min(B, beg + per_cta);
  for (int64_t v = beg + warp * EG + eg; v < end; v += 8 * EG) {
    float l1[2] = {0.f, 0.f}, l2[2] = {0.f, 0.f}, l3[2] = {0.f, 0.f}, l4 = 0.f;
    for (int k = 0; k < K; ++k) {
      const float d = __ldg(dist + v * K + k), g = __ldg(ds + v * K + k);
      l4 += g;
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        if (q == 1 && HL < 32) break;
        const float pre = fmaf(w1[q], d, bb[q]);
        const bool pos = pre > 0.f;
        l3[q] = fmaf(g, pos ? pre : 0.f, l3[q]);
        const float da = pos ? g * w2[q] : 0.f;
        l1[q] = fmaf(da, d, l1[q]);
        l2[q] += da;
      }
    }
    a4 += l4;
#pragma unroll
    for (int q = 0; q < 2; ++q) { a1[q] += l1[q]; a2[q] += l2[q]; a3[q] += l3[q]; }
  }
  // combine the vehicle slots of a warp in slot order, then the warps in warp order
  s_g[warp][lane][0] = a1[0]; s_g[warp][lane][1] = a1[1]; s_g[warp][lane][2] = a2[0]; s_g[warp][lane][3] = a2[1];
  s_g[warp][lane][4] = a3[0]; s_g[warp][lane][5] = a3[1]; s_g[warp][lane][6] = a4;
  __syncwarp();
  if (lane < HL) {
    float t[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int e = 0; e < EG; ++e)
#pragma unroll
      for (int v = 0; v < 7; ++v) t[v] += s_g[warp][e * HL + lane][v];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int h = lane + 32 * q;
      if (h < H && (q == 0 || HL == 32)) { s_p[warp][h] = t[q]; s_p[warp][H + h] = t[2 + q]; s_p[warp][2 * H + h] = t[4 + q]; }
    }
    if (lane == 0) s_p[warp][3 * H] = t[6];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * H + 1; i += 256) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += s_p[w][i];
    part[(int64_t)blockIdx.x * (3 * H + 1) + i] = s;
  }
}

// k_map_attention_demb for K = 9..32: one instance per K (K only divides the member position)
template <int KK>
static void launch_demb_wide(int K, unsigned S, size_t smb, cudaStream_t s, const float* dctx, int D, const float* w,
                             const int32_t* rp, const int32_t* mem, float* demb) {
  if (K == KK) k_map_attention_demb<KK><<<S, 32 * kDembWarps, smb, s>>>(dctx, D, w, rp, mem, demb);
  else if constexpr (KK < kMaKWide) launch_demb_wide<KK + 1>(K, S, smb, s, dctx, D, w, rp, mem, demb);
}

// kernel for the MLP gradients: the partial count is fixed by B alone (workspace sizing)
static int mlp_grid(int64_t B) { return (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div<int64_t>(B, 256), (int64_t)num_sms() * 4)); }

}  // namespace sldm

using namespace sldm;

// workspace: [ds: B * 8 floats][partials: mlp_grid(B) x (3H + 1) floats]
extern "C" int64_t sldm_map_attention_workspace_bytes(int64_t B, int32_t H) {
  if (B < 0 || H < 0) return -1;
  return align_bytes(B * kMaK * 4) + align_bytes((int64_t)mlp_grid(B) * (3 * H + 1) * 4);
}

// the same layout with B * max(K, 8) floats for ds: equal to the query above for K <= 8
extern "C" int64_t sldm_map_attention_workspace_bytes_k(int64_t B, int32_t H, int32_t K) {
  if (B < 0 || H < 0 || K < 1 || K > kMaKWide) return -1;
  return align_bytes(B * std::max<int64_t>(K, kMaK) * 4) + align_bytes((int64_t)mlp_grid(B) * (3 * H + 1) * 4);
}

extern "C" int sldm_map_attention_max_k(void) { return kMaKWide; }

extern "C" int sldm_map_attention_forward(const float* pos, int64_t B, const float* centroids, int64_t S,
                                          const float* emb, int32_t D, int32_t K,
                                          const float* W1, const float* b1, const float* W2, const float* b2, int32_t H,
                                          float* ctx, int64_t* idx_out, float* dist_out, float* w_out,
                                          sldm_stream_t stream) {
  SLDM_REQUIRE(B >= 0 && S >= 0 && D >= 1, SLDM_EINVAL, "sldm_map_attention_forward: bad sizes");
  SLDM_REQUIRE(K >= 1 && K <= kMaKWide, SLDM_EUNSUPPORTED, "sldm_map_attention_forward: k_neighbors=%d outside 1..%d", K, kMaKWide);
  SLDM_REQUIRE(H >= 1 && H <= kMaH, SLDM_EUNSUPPORTED, "sldm_map_attention_forward: MLP width %d outside 1..%d", H, kMaH);
  SLDM_REQUIRE(S >= K, SLDM_ESHAPE, "selected index k out of range");   // torch.topk's message
  SLDM_REQUIRE(S < ((int64_t)1 << 31), SLDM_EUNSUPPORTED, "sldm_map_attention_forward: S too large");
  if (B == 0) return SLDM_OK;
  SLDM_REQUIRE(pos && centroids && emb && W1 && b1 && W2 && b2 && ctx && idx_out && dist_out && w_out, SLDM_EINVAL,
               "sldm_map_attention_forward: NULL pointer");
  SLDM_REQUIRE((reinterpret_cast<uintptr_t>(centroids) & 7u) == 0, SLDM_EINVAL, "sldm_map_attention_forward: centroids must be 8-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div<int64_t>(B, 8), (int64_t)num_sms() * 8);
  const float2* c2 = reinterpret_cast<const float2*>(centroids);
  if (K > kMaK) {
    k_map_attention_fwd_wide<<<grid, 256, 0, s>>>(pos, B, c2, (int)S, emb, D, W1, b1, W2, b2, H, K, ctx, idx_out, dist_out, w_out);
    SLDM_LAUNCH_CHECK("k_map_attention_fwd_wide");
    return SLDM_OK;
  }
#define SLDM_MA(KK) k_map_attention_fwd<KK><<<grid, 256, 0, s>>>(pos, B, c2, (int)S, emb, D, W1, b1, W2, b2, H, ctx, idx_out, dist_out, w_out)
  switch (K) {
    case 1: SLDM_MA(1); break; case 2: SLDM_MA(2); break; case 3: SLDM_MA(3); break; case 4: SLDM_MA(4); break;
    case 5: SLDM_MA(5); break; case 6: SLDM_MA(6); break; case 7: SLDM_MA(7); break; default: SLDM_MA(8); break;
  }
#undef SLDM_MA
  SLDM_LAUNCH_CHECK("k_map_attention_fwd");
  return SLDM_OK;
}

extern "C" int64_t sldm_map_grid_bytes(int64_t S) {
  if (S < 0 || S >= ((int64_t)1 << 31)) return -1;
  return map_grid_layout(S).total;
}

extern "C" int sldm_map_grid_build(const float* centroids, int64_t S, void* grid, int64_t grid_bytes, sldm_stream_t stream) {
  SLDM_REQUIRE(S >= 0 && S < ((int64_t)1 << 31), SLDM_EINVAL, "sldm_map_grid_build: bad S");
  const MapGridLayout L = map_grid_layout(S);
  SLDM_REQUIRE(grid != nullptr && grid_bytes >= L.total, SLDM_EWORKSPACE, "sldm_map_grid_build: grid buffer too small");
  SLDM_REQUIRE(S == 0 || centroids != nullptr, SLDM_EINVAL, "sldm_map_grid_build: NULL centroids");
  SLDM_REQUIRE((reinterpret_cast<uintptr_t>(centroids) & 7u) == 0 && (reinterpret_cast<uintptr_t>(grid) & 15u) == 0, SLDM_EINVAL,
               "sldm_map_grid_build: centroids must be 8-byte, the grid buffer 16-byte aligned");
  uint8_t* g = static_cast<uint8_t*>(grid);
  k_map_grid_build<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float2*>(centroids), (int)S, L.G, reinterpret_cast<MapGridHeader*>(g),
      reinterpret_cast<int*>(g + L.off_start), reinterpret_cast<int*>(g + L.off_cursor), reinterpret_cast<float4*>(g + L.off_entries));
  SLDM_LAUNCH_CHECK("k_map_grid_build");
  return SLDM_OK;
}

extern "C" int sldm_map_attention_forward_grid(const float* pos, int64_t B, const void* grid, int64_t grid_bytes, int64_t S,
                                               const float* emb, int32_t D, int32_t K,
                                               const float* W1, const float* b1, const float* W2, const float* b2, int32_t H,
                                               float* ctx, int64_t* idx_out, float* dist_out, float* w_out,
                                               sldm_stream_t stream) {
  SLDM_REQUIRE(B >= 0 && S >= 0 && D >= 1, SLDM_EINVAL, "sldm_map_attention_forward_grid: bad sizes");
  SLDM_REQUIRE(K >= 1 && K <= kMaKWide, SLDM_EUNSUPPORTED, "sldm_map_attention_forward_grid: k_neighbors=%d outside 1..%d", K, kMaKWide);
  SLDM_REQUIRE(H >= 1 && H <= kMaH, SLDM_EUNSUPPORTED, "sldm_map_attention_forward_grid: MLP width %d outside 1..%d", H, kMaH);
  SLDM_REQUIRE(S >= K, SLDM_ESHAPE, "selected index k out of range");   // torch.topk's message
  SLDM_REQUIRE(S * (int64_t)D < ((int64_t)1 << 32), SLDM_EUNSUPPORTED, "sldm_map_attention_forward_grid: S * D must stay below 2^32");
  if (B == 0) return SLDM_OK;
  const MapGridLayout L = map_grid_layout(S);
  SLDM_REQUIRE(grid != nullptr && grid_bytes >= L.total, SLDM_EWORKSPACE, "sldm_map_attention_forward_grid: grid buffer too small");
  SLDM_REQUIRE(pos && emb && W1 && b1 && W2 && b2 && ctx && idx_out && dist_out && w_out, SLDM_EINVAL,
               "sldm_map_attention_forward_grid: NULL pointer");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const uint8_t* g = static_cast<const uint8_t*>(grid);
  if (K > kMaK) {
    k_map_attention_grid_fwd_wide<<<(unsigned)ceil_div<int64_t>(B, 8), 256, 0, s>>>(
        pos, B, reinterpret_cast<const MapGridHeader*>(g), reinterpret_cast<const int*>(g + L.off_start),
        reinterpret_cast<const float4*>(g + L.off_entries), emb, D, W1, b1, W2, b2, H, K, ctx, idx_out, dist_out, w_out);
    SLDM_LAUNCH_CHECK("k_map_attention_grid_fwd_wide");
    return SLDM_OK;
  }
  const unsigned nblk = (unsigned)ceil_div<int64_t>(B, 256);
#define SLDM_MG(KK) k_map_attention_grid_fwd<KK><<<nblk, 256, 0, s>>>(pos, B, reinterpret_cast<const MapGridHeader*>(g), \
      reinterpret_cast<const int*>(g + L.off_start), reinterpret_cast<const float4*>(g + L.off_entries), emb, D, W1, b1, W2, b2, H, \
      ctx, idx_out, dist_out, w_out)
  switch (K) {
    case 1: SLDM_MG(1); break; case 2: SLDM_MG(2); break; case 3: SLDM_MG(3); break; case 4: SLDM_MG(4); break;
    case 5: SLDM_MG(5); break; case 6: SLDM_MG(6); break; case 7: SLDM_MG(7); break; default: SLDM_MG(8); break;
  }
#undef SLDM_MG
  SLDM_LAUNCH_CHECK("k_map_attention_grid_fwd");
  return SLDM_OK;
}

// csr: membership CSR of the selected segments: sldm_csr_build_pairs(NULL, idx (as [B*K] int64), B*K, csr_nodes >= S, ...)
extern "C" int sldm_map_attention_backward(const float* dctx, int64_t B, const float* emb, int64_t S, int32_t D, int32_t K,
                                           const int64_t* idx, const float* dist, const float* w,
                                           const float* W1, const float* b1, const float* W2, int32_t H,
                                           const int32_t* csr, int64_t csr_nodes,
                                           float* demb, float* dW1, float* db1, float* dW2, float* db2,
                                           void* workspace, int64_t workspace_bytes, sldm_stream_t stream) {
  SLDM_REQUIRE(B >= 0 && S >= 0 && D >= 1 && D <= 1024, SLDM_EINVAL, "sldm_map_attention_backward: bad sizes");
  SLDM_REQUIRE(S * (int64_t)D < ((int64_t)1 << 32) && B * (int64_t)D < ((int64_t)1 << 32), SLDM_EUNSUPPORTED,
               "sldm_map_attention_backward: S * D and B * D must stay below 2^32");
  SLDM_REQUIRE(K >= 1 && K <= kMaKWide && H >= 1 && H <= kMaH, SLDM_EUNSUPPORTED, "sldm_map_attention_backward: K / H out of range");
  SLDM_REQUIRE(K <= kMaK || B * K < kMaCsrMax, SLDM_EUNSUPPORTED,
               "sldm_map_attention_backward: B * K = %lld exceeds the int32 membership CSR", (long long)(B * K));
  SLDM_REQUIRE(dW1 && db1 && dW2 && db2, SLDM_EINVAL, "sldm_map_attention_backward: NULL gradient output");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (B == 0) {
    SLDM_CUDA(cudaMemsetAsync(dW1, 0, H * 4, s)); SLDM_CUDA(cudaMemsetAsync(db1, 0, H * 4, s));
    SLDM_CUDA(cudaMemsetAsync(dW2, 0, H * 4, s)); SLDM_CUDA(cudaMemsetAsync(db2, 0, 4, s));
    if (demb && S > 0) SLDM_CUDA(cudaMemsetAsync(demb, 0, (size_t)S * D * 4, s));
    return SLDM_OK;
  }
  SLDM_REQUIRE(dctx && emb && idx && dist && w && W1 && b1 && W2, SLDM_EINVAL, "sldm_map_attention_backward: NULL pointer");
  SLDM_REQUIRE(workspace != nullptr && workspace_bytes >= sldm_map_attention_workspace_bytes_k(B, H, K), SLDM_EWORKSPACE,
               "sldm_map_attention_backward: workspace too small");
  float* const ds = static_cast<float*>(workspace);
  float* const part = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + align_bytes(B * std::max(K, kMaK) * 4));
  const bool vec = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(dctx) | reinterpret_cast<uintptr_t>(emb)) & 15u) == 0;
  // persistent grid: exactly the CTAs that are resident at once (the loop prefetches across iterations)
  auto ds_grid = [&](auto kernel, int vpw) {
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0);
    return (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div<int64_t>(B, 8 * vpw), (int64_t)num_sms() * std::max(per_sm, 1)));
  };
  const int mgrid = mlp_grid(B);
  const int64_t per_cta = round_up<int64_t>(ceil_div<int64_t>(B, mgrid), 256);   // vehicles per CTA
  int HL = 1;
  while (HL < H && HL < 32) HL <<= 1;              // lanes across the hidden units
  if (K > kMaK) {
    const unsigned nblk = (unsigned)ceil_div<int64_t>(B, 8);
    if (vec) k_map_attention_bwd_ds_wide<true><<<nblk, 256, 0, s>>>(dctx, B, emb, D, K, idx, w, ds);
    else k_map_attention_bwd_ds_wide<false><<<nblk, 256, 0, s>>>(dctx, B, emb, D, K, idx, w, ds);
    SLDM_LAUNCH_CHECK("k_map_attention_bwd_ds_wide");
    k_map_attention_bwd_mlp_wide<<<mgrid, 256, 0, s>>>(dist, ds, B, K, per_cta, W1, b1, W2, H, HL, part);
    SLDM_LAUNCH_CHECK("k_map_attention_bwd_mlp_wide");
  } else {
#define SLDM_MB(KK) do { if (vec) k_map_attention_bwd_ds<KK, 8><<<ds_grid(k_map_attention_bwd_ds<KK, 8>, 4), 256, 0, s>>>(dctx, B, emb, D, idx, w, ds); \
                         else k_map_attention_bwd_ds<KK, 32><<<ds_grid(k_map_attention_bwd_ds<KK, 32>, 1), 256, 0, s>>>(dctx, B, emb, D, idx, w, ds); } while (0)
    switch (K) {
      case 1: SLDM_MB(1); break; case 2: SLDM_MB(2); break; case 3: SLDM_MB(3); break; case 4: SLDM_MB(4); break;
      case 5: SLDM_MB(5); break; case 6: SLDM_MB(6); break; case 7: SLDM_MB(7); break; default: SLDM_MB(8); break;
    }
#undef SLDM_MB
    SLDM_LAUNCH_CHECK("k_map_attention_bwd_ds");
    k_map_attention_bwd_mlp<<<mgrid, 256, 0, s>>>(dist, ds, B, K, per_cta, W1, b1, W2, H, HL, part);
    SLDM_LAUNCH_CHECK("k_map_attention_bwd_mlp");
  }
  k_map_attention_reduce<<<ceil_div(3 * H + 1, 8), 256, 0, s>>>(part, mgrid, H, dW1, db1, dW2, db2);
  SLDM_LAUNCH_CHECK("k_map_attention_reduce");
  if (demb != nullptr && S > 0) {
    SLDM_REQUIRE(csr != nullptr && csr_nodes >= S, SLDM_EINVAL, "sldm_map_attention_backward: membership CSR missing / too small");
    CsrLayout L = csr_layout(csr_nodes, B * K);
    const int32_t* rp = csr + L.off[SLDM_CSR_ROWPTR_DST];
    const int32_t* mem = csr + L.off[SLDM_CSR_COL_SRC];
    const size_t smb = (size_t)kDembWarps * D * sizeof(float);
#define SLDM_ME(KK) k_map_attention_demb<KK><<<(unsigned)S, 32 * kDembWarps, smb, s>>>(dctx, D, w, rp, mem, demb)
    if (K > kMaK) launch_demb_wide<kMaK + 1>(K, (unsigned)S, smb, s, dctx, D, w, rp, mem, demb);
    else switch (K) {
      case 1: SLDM_ME(1); break; case 2: SLDM_ME(2); break; case 3: SLDM_ME(3); break; case 4: SLDM_ME(4); break;
      case 5: SLDM_ME(5); break; case 6: SLDM_ME(6); break; case 7: SLDM_ME(7); break; default: SLDM_ME(8); break;
    }
#undef SLDM_ME
    SLDM_LAUNCH_CHECK("k_map_attention_demb");
  }
  return SLDM_OK;
}
