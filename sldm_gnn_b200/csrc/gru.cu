// gru.cu -- fused GRU layers over short sequences (the sequence head in front of the vehicle-graph SageBlock).
//
// Replaces `gru_out, hlast = self.gru(x); x = hlast[-1]` (src/models/grusage.py:160-161; nn.GRU(input 6, hidden 96,
// one layer, batch_first) built at grusage.py:55-60) and its autograd backward.  torch runs that as 16 x (2 GEMMs +
// a cell kernel) forward and as many again backward, with every gate tensor making a round trip through HBM; here the
// whole recurrence of a tile of 64 sequences stays on one SM:
//
//   forward  (k_gru_fwd):  W_hh [3H,H] lives in shared memory (row stride H+4 floats: conflict-free 128-bit loads with
//            lane = hidden unit), a warp owns 8 sequences for all T steps (its h rows are read as shared-memory
//            broadcasts), a lane owns H/32 hidden units x 3 gates x 8 rows = 72 fp32 accumulators at H = 96; the gate
//            math of a (row, unit) is local to its thread, so the time loop needs no block-level barrier at all.
//            When training it writes h_{t-1}, r, z, n and (W_hn h + b_hn) per step -- what torch's fused cell saves --
//            as one [T, N, 5, H] buffer: a warp's output of a step is 8 x 5H contiguous floats (with five [N, T, H]
//            arrays the 128-byte pieces were 6 KB apart and the stores cost 3.6 ms on top of 5.7 ms of arithmetic).
//   backward (k_gru_bwd):  the same tiling walks t = T-1 .. 0 with W_hh transposed in shared memory
//            (dh_{t-1} = dh_t z + [dr dz dn r] W_hh); it emits the hidden-gate gradients dgh [T,N,3H] and accumulates
//            dW_ih, db_ih, db_hh per CTA in registers (fixed order; the per-CTA partials are summed by the caller).
//   wgrad    (k_gru_wgrad): dW_hh = dgh^T h_prev over the T*N rows, one persistent CTA per SM (below).
//
// Stacked layers (nn.GRU(num_layers = L)) run layer by layer on the same kernels: a layer above the first reads the
// output sequence h_seq [T,N,H] of the layer below through k_gru_proj (gi = h_seq W_ih^T + b_ih, [T,N,3H]) and
// k_gru_fwd's gi mode; backward, k_gru_bwd's deep mode takes the per-step upstream gradient dh_seq and writes
// dgi [T,N,3H], from which k_gru_wgrad gives dW_ih (against h_seq) and k_gru_proj the layer below's dh_seq.
//
// Arithmetic: FP32 FMA in sequential k order, expf / tanhf / IEEE division like ATen's gru_cell_forward, i.e. the
// reference's own formulas (aten/src/ATen/native/cuda/RNN.cu); bound by the FP32 pipe (2*3H*H flops per sequence and
// step each way), not by HBM.  Limits: H in {32, 64, 96}, layer 0's input width <= 8 and its x tile must fit shared
// memory; the layers above have no limit on T.
#include "common.cuh"
#include <algorithm>

namespace sldm {
namespace {

constexpr int kGruRows = 64;      // sequences per CTA
constexpr int kGruRpw = 8;        // sequences per warp
constexpr int kGruThreads = 256;
constexpr int kGruMaxI = 8;
constexpr int kGruLdi = 9;        // W_ih row stride in shared memory (odd: conflict-free scalar loads)
constexpr int64_t kGruSmemMax = 227 * 1024;

__device__ __forceinline__ float gru_sigmoid(float v) { return 1.0f / (1.0f + expf(-v)); }

__device__ __forceinline__ void fma4(float& acc, const float4& a, const float4& b) {
  acc = fmaf(a.x, b.x, acc);
  acc = fmaf(a.y, b.y, acc);
  acc = fmaf(a.z, b.z, acc);
  acc = fmaf(a.w, b.w, acc);
}

// Packed FP32 FMA of sm_100 (fma.rn.f32x2 -> FFMA2): two FMAs per issue slot at the same pipe rate (tools/ffma2_probe.cu:
// a register-tiled 8 x 9 outer product reaches 56 TFLOP/s with FFMA and 65 with FFMA2 on B200).  Used by k_gru_wgrad
// (4.03 -> 3.75 ms).  In the recurrence kernels a k-paired FFMA2 main loop (even k in the low half of an accumulator pair,
// odd k in the high half) measured slower than scalar FFMA (forward 5.70 vs 5.34 ms: 144 accumulator registers and ~80
// pair-shuffling MOVs per 288 FFMA2), so they keep the scalar loop.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 ffma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 f32x2_dup(float v) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %1};" : "=l"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ void load_x_tile(float* xs, const float* __restrict__ x, int64_t row0, int nrows, int TI) {
  const float* xg = x + row0 * TI;
  for (int i = threadIdx.x; i < kGruRows * TI; i += kGruThreads) xs[i] = i < nrows * TI ? __ldg(xg + i) : 0.f;
}

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// GI = false: layer 0, the input product x W_ih^T (I <= 8) is computed here from a shared-memory tile of x.
// GI = true : a layer of a stack, fed the precomputed input pre-activations gi [T,N,3H] (b_ih included, k_gru_proj);
//             a warp prefetches step t+1's [8][3H] slice with cp.async while step t's W_hh product runs.  Nothing in
//             shared memory depends on T, so this mode has no sequence-length limit.
// h_seq [T,N,H] (NULL unless a layer above reads it) receives h_t of every step; h_last may be NULL.
template <int H, bool SAVE, bool GI>
__global__ void __launch_bounds__(kGruThreads, 1)
k_gru_fwd(const float* __restrict__ x, const float* __restrict__ gi, int64_t N, int T, int I,
          const float* __restrict__ W_ih, const float* __restrict__ W_hh,
          const float* __restrict__ b_ih, const float* __restrict__ b_hh,
          float* __restrict__ h_last, float* __restrict__ saved, float* __restrict__ h_seq) {
  constexpr int U = H / 32, LDW = H + 4, G3 = 3 * H;
  extern __shared__ __align__(16) float sm[];
  float* Ws = sm;                        // [3H][LDW]
  float* hs = Ws + 3 * H * LDW;          // [64][H]   current hidden state of the tile
  float* bs = hs + kGruRows * H;         // b_ir+b_hr | b_iz+b_hz | b_in | b_hn   (GI: b_hr | b_hz | 0 | b_hn)
  float* Wi = bs + 4 * H;                // [3H][9]                               (GI: absent)
  float* xs = Wi + 3 * H * kGruLdi;      // [64][T*I]                             (GI: absent)
  float* gs = Wi;                        // GI: [64][3H] gi of the current step
  const int tid = threadIdx.x, w = tid >> 5, l = tid & 31;
  const int64_t row0 = (int64_t)blockIdx.x * kGruRows;
  const int nrows = (int)min((int64_t)kGruRows, N - row0);
  const int TI = T * I;

  for (int i = tid; i < 3 * H * (H / 4); i += kGruThreads) {
    const int r = i / (H / 4), c = i % (H / 4);
    *reinterpret_cast<float4*>(Ws + r * LDW + 4 * c) = __ldg(reinterpret_cast<const float4*>(W_hh) + i);
  }
  if (GI) {
    for (int i = tid; i < H; i += kGruThreads) {
      bs[i] = __ldg(b_hh + i);
      bs[H + i] = __ldg(b_hh + H + i);
      bs[2 * H + i] = 0.f;
      bs[3 * H + i] = __ldg(b_hh + 2 * H + i);
    }
  } else {
    for (int i = tid; i < 3 * H * I; i += kGruThreads) Wi[(i / I) * kGruLdi + (i % I)] = __ldg(W_ih + i);
    for (int i = tid; i < H; i += kGruThreads) {
      bs[i] = __ldg(b_ih + i) + __ldg(b_hh + i);
      bs[H + i] = __ldg(b_ih + H + i) + __ldg(b_hh + H + i);
      bs[2 * H + i] = __ldg(b_ih + 2 * H + i);
      bs[3 * H + i] = __ldg(b_hh + 2 * H + i);
    }
  }
  for (int i = tid; i < kGruRows * H; i += kGruThreads) hs[i] = 0.f;
  if (!GI) load_x_tile(xs, x, row0, nrows, TI);
  __syncthreads();

  const int r0 = w * kGruRpw;
  const float* hrow = hs + r0 * H;
  const float* wrow = Ws + l * LDW;
  float* gw = gs + r0 * G3;                                   // GI: the warp's [8][3H] slice
  const int nv = max(0, min(kGruRpw, nrows - r0));           // valid rows of the warp
  auto prefetch_gi = [&](int t) {                             // rows of one step are contiguous in gi
    const float* src = gi + ((int64_t)t * N + row0 + r0) * G3;
    for (int i = l; i < nv * G3 / 4; i += 32) cp_async16(gw + 4 * i, src + 4 * i);
    cp_async_commit();
  };
  if (GI) prefetch_gi(0);
  float hreg[kGruRpw][U];
#pragma unroll
  for (int i = 0; i < kGruRpw; ++i)
#pragma unroll
    for (int u = 0; u < U; ++u) hreg[i][u] = 0.f;

  for (int t = 0; t < T; ++t) {
    float ar[kGruRpw][U], az[kGruRpw][U], an[kGruRpw][U], ai[kGruRpw][U];
    if (GI) {
      cp_async_wait<0>();
      __syncwarp();
#pragma unroll
      for (int i = 0; i < kGruRpw; ++i)
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const float* g = gw + i * G3 + l + 32 * u;
          ar[i][u] = g[0]; az[i][u] = g[H]; ai[i][u] = g[2 * H]; an[i][u] = 0.f;
        }
      __syncwarp();   // the slice is in registers: step t+1's copy may overwrite it
      if (t + 1 < T) prefetch_gi(t + 1);
    } else {
#pragma unroll
      for (int i = 0; i < kGruRpw; ++i)
#pragma unroll
        for (int u = 0; u < U; ++u) ar[i][u] = az[i][u] = an[i][u] = ai[i][u] = 0.f;
    }

    // hidden part: [8 rows] x [3 gates x U units] over k, h rows as broadcasts, weights one row per lane
#pragma unroll 2
    for (int k = 0; k < H; k += 4) {
      float4 hv[kGruRpw];
#pragma unroll
      for (int i = 0; i < kGruRpw; ++i) hv[i] = *reinterpret_cast<const float4*>(hrow + i * H + k);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float4 w0 = *reinterpret_cast<const float4*>(wrow + (u * 32) * LDW + k);
        const float4 w1 = *reinterpret_cast<const float4*>(wrow + (H + u * 32) * LDW + k);
        const float4 w2 = *reinterpret_cast<const float4*>(wrow + (2 * H + u * 32) * LDW + k);
#pragma unroll
        for (int i = 0; i < kGruRpw; ++i) {
          fma4(ar[i][u], hv[i], w0);
          fma4(az[i][u], hv[i], w1);
          fma4(an[i][u], hv[i], w2);
        }
      }
    }
    if (SAVE) {
#pragma unroll
      for (int i = 0; i < kGruRpw; ++i)
        if (r0 + i < nrows) {
          float* o = saved + (((int64_t)t * N + row0 + r0 + i) * 5) * H + l;
#pragma unroll
          for (int u = 0; u < U; ++u) o[32 * u] = hreg[i][u];
        }
    }
    // input part (I <= 8): r and z continue their accumulators, the n gate keeps its input half apart
    for (int i2 = 0; i2 < (GI ? 0 : I); ++i2) {
      float xv[kGruRpw];
#pragma unroll
      for (int i = 0; i < kGruRpw; ++i) xv[i] = xs[(r0 + i) * TI + t * I + i2];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float wr = Wi[(l + 32 * u) * kGruLdi + i2];
        const float wz = Wi[(H + l + 32 * u) * kGruLdi + i2];
        const float wn = Wi[(2 * H + l + 32 * u) * kGruLdi + i2];
#pragma unroll
        for (int i = 0; i < kGruRpw; ++i) {
          ar[i][u] = fmaf(xv[i], wr, ar[i][u]);
          az[i][u] = fmaf(xv[i], wz, az[i][u]);
          ai[i][u] = fmaf(xv[i], wn, ai[i][u]);
        }
      }
    }
    // gates (ATen gru_cell_forward): r, z = sigmoid, n = tanh(i_n + b_in + r (h_n + b_hn)), h' = n + z (h - n)
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int j = l + 32 * u;
      const float br = bs[j], bz = bs[H + j], bin = bs[2 * H + j], bhn = bs[3 * H + j];
#pragma unroll
      for (int i = 0; i < kGruRpw; ++i) {
        const float rg = gru_sigmoid(ar[i][u] + br);
        const float zg = gru_sigmoid(az[i][u] + bz);
        const float hn = an[i][u] + bhn;
        const float ng = tanhf(ai[i][u] + bin + rg * hn);
        if (SAVE && r0 + i < nrows) {
          float* o = saved + (((int64_t)t * N + row0 + r0 + i) * 5) * H + j;
          o[H] = rg; o[2 * H] = zg; o[3 * H] = ng; o[4 * H] = hn;
        }
        hreg[i][u] = ng + zg * (hreg[i][u] - ng);
      }
    }
    __syncwarp();   // every lane has finished reading the warp's h rows
#pragma unroll
    for (int i = 0; i < kGruRpw; ++i)
#pragma unroll
      for (int u = 0; u < U; ++u) hs[(r0 + i) * H + l + 32 * u] = hreg[i][u];
    if (h_seq != nullptr) {
#pragma unroll
      for (int i = 0; i < kGruRpw; ++i)
        if (r0 + i < nrows) {
#pragma unroll
          for (int u = 0; u < U; ++u) h_seq[((int64_t)t * N + row0 + r0 + i) * H + l + 32 * u] = hreg[i][u];
        }
    }
    __syncwarp();
  }
  if (h_last == nullptr) return;
#pragma unroll
  for (int i = 0; i < kGruRpw; ++i)
    if (r0 + i < nrows) {
#pragma unroll
      for (int u = 0; u < U; ++u) h_last[(row0 + r0 + i) * H + l + 32 * u] = hreg[i][u];
    }
}

// per-CTA partial layout (floats): [28*U][32 lanes]: v = (u*3+g)*8 + i2 -> dW_ih[g*H + 32u + lane][i2];
// v = 24U + u*3 + g -> db_ih[g*H + 32u + lane]; v = 27U + u -> db_hh[2H + 32u + lane] (its r and z thirds equal db_ih's)
// DEEP = false: layer 0, dW_ih accumulated here against the x tile.  DEEP = true: a layer of a stack (its input is the
// layer below's h_seq, dW_ih comes from k_gru_wgrad over dgi); no x tile, so no sequence-length limit, and the dW_ih
// slots of the partials are written as zeros.  dh_last may be NULL (zeros: the hlast of a lower layer is unused);
// dh_seq [T,N,H] (may be NULL) is the upstream gradient of h_t, added to dh at the top of step t; dgi [T,N,3H] (may be
// NULL) receives [dr~ dz~ dn~], the input-side pre-activation gradients.
template <int H, bool DEEP>
__global__ void __launch_bounds__(kGruThreads, 1)
k_gru_bwd(const float* __restrict__ x, int64_t N, int T, int I, const float* __restrict__ W_hh,
          const float* __restrict__ dh_last, const float* __restrict__ dh_seq, const float* __restrict__ saved,
          float* __restrict__ dgh, float* __restrict__ gin_out, float* __restrict__ dgi, float* __restrict__ parts) {
  constexpr int U = H / 32, G3 = 3 * H, LDT = 3 * H + 4, V = 28 * U;
  extern __shared__ __align__(16) float sm[];
  float* Wt = sm;                       // [H][LDT]: Wt[j][k] = W_hh[k][j]
  float* gs = Wt + H * LDT;             // [64][3H]  hidden-gate gradients of the current step
  float* xs = gs + kGruRows * G3;       // [64][T*I]  (DEEP: absent)
  const int tid = threadIdx.x, w = tid >> 5, l = tid & 31;
  const int64_t row0 = (int64_t)blockIdx.x * kGruRows;
  const int nrows = (int)min((int64_t)kGruRows, N - row0);
  const int TI = T * I;

  for (int i = tid; i < G3 * H; i += kGruThreads) Wt[(i % H) * LDT + (i / H)] = __ldg(W_hh + i);
  if (!DEEP) load_x_tile(xs, x, row0, nrows, TI);
  __syncthreads();

  const int r0 = w * kGruRpw;
  float dh[kGruRpw][U];
#pragma unroll
  for (int i = 0; i < kGruRpw; ++i)
#pragma unroll
    for (int u = 0; u < U; ++u)
      dh[i][u] = dh_last != nullptr && r0 + i < nrows ? __ldg(dh_last + (row0 + r0 + i) * H + l + 32 * u) : 0.f;
  float dWi[U][3][kGruMaxI], dbi[U][3], dbn[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    dbn[u] = 0.f;
#pragma unroll
    for (int g = 0; g < 3; ++g) {
      dbi[u][g] = 0.f;
#pragma unroll
      for (int i2 = 0; i2 < kGruMaxI; ++i2) dWi[u][g][i2] = 0.f;
    }
  }
  const float* grow = gs + r0 * G3;
  const float* wrow = Wt + l * LDT;

  for (int t = T - 1; t >= 0; --t) {
    if (dh_seq != nullptr) {
#pragma unroll
      for (int i = 0; i < kGruRpw; ++i)
        if (r0 + i < nrows) {
#pragma unroll
          for (int u = 0; u < U; ++u) dh[i][u] += __ldg(dh_seq + ((int64_t)t * N + row0 + r0 + i) * H + l + 32 * u);
        }
    }
    // cell backward (ATen gru_cell_backward) for the thread's (row, unit) pairs
#pragma unroll
    for (int i = 0; i < kGruRpw; ++i) {
      const bool valid = r0 + i < nrows;
      float xv[kGruMaxI];
#pragma unroll
      for (int i2 = 0; i2 < kGruMaxI; ++i2) xv[i2] = !DEEP && i2 < I ? xs[(r0 + i) * TI + t * I + i2] : 0.f;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int j = l + 32 * u;
        const int64_t tr = (int64_t)t * N + row0 + r0 + i;     // row of the [T, N, ...] buffers
        float rg = 0.f, zg = 0.f, ng = 0.f, hn = 0.f, hpv = 0.f;
        if (valid) {
          const float* o = saved + tr * 5 * H + j;
          hpv = __ldg(o); rg = __ldg(o + H); zg = __ldg(o + 2 * H); ng = __ldg(o + 3 * H); hn = __ldg(o + 4 * H);
        }
        const float g = dh[i][u];
        const float gig = g * (hpv - ng) * (1.f - zg) * zg;
        const float ghx = g * zg;
        const float gin = g * (1.f - zg) * (1.f - ng * ng);
        const float ghn = gin * rg;
        const float grg = gin * hn * (1.f - rg) * rg;
        if (valid) {
          float* og = dgh + tr * G3 + j;
          og[0] = grg; og[H] = gig; og[2 * H] = ghn;
          if (gin_out != nullptr) gin_out[tr * H + j] = gin;
          if (dgi != nullptr) {
            float* oi = dgi + tr * G3 + j;
            oi[0] = grg; oi[H] = gig; oi[2 * H] = gin;
          }
        }
        float* gr = gs + (r0 + i) * G3 + j;
        gr[0] = grg; gr[H] = gig; gr[2 * H] = ghn;
        dh[i][u] = ghx;
        dbi[u][0] += grg; dbi[u][1] += gig; dbi[u][2] += gin; dbn[u] += ghn;
        if (!DEEP) {
#pragma unroll
          for (int i2 = 0; i2 < kGruMaxI; ++i2) {
            dWi[u][0][i2] = fmaf(grg, xv[i2], dWi[u][0][i2]);
            dWi[u][1][i2] = fmaf(gig, xv[i2], dWi[u][1][i2]);
            dWi[u][2][i2] = fmaf(gin, xv[i2], dWi[u][2][i2]);
          }
        }
      }
    }
    __syncwarp();
    // dh_{t-1} = dh_t z + dgh W_hh : [8 rows] x [U units] over k = 0..3H
#pragma unroll 2
    for (int k = 0; k < G3; k += 4) {
      float4 gv[kGruRpw];
#pragma unroll
      for (int i = 0; i < kGruRpw; ++i) gv[i] = *reinterpret_cast<const float4*>(grow + i * G3 + k);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float4 wv = *reinterpret_cast<const float4*>(wrow + (32 * u) * LDT + k);
#pragma unroll
        for (int i = 0; i < kGruRpw; ++i) fma4(dh[i][u], gv[i], wv);
      }
    }
    __syncwarp();
  }

  // parameter-gradient partials: warps combined in index order
  __syncthreads();
  float* red = sm;   // [8 warps][V][32]  (fits in Wt + gs for every supported H)
  {
    float* mine = red + (w * V) * 32 + l;
#pragma unroll
    for (int u = 0; u < U; ++u) {
#pragma unroll
      for (int g = 0; g < 3; ++g) {
#pragma unroll
        for (int i2 = 0; i2 < kGruMaxI; ++i2) mine[((u * 3 + g) * 8 + i2) * 32] = dWi[u][g][i2];
        mine[(24 * U + u * 3 + g) * 32] = dbi[u][g];
      }
      mine[(27 * U + u) * 32] = dbn[u];
    }
  }
  __syncthreads();
  for (int o = tid; o < V * 32; o += kGruThreads) {
    float s = 0.f;
#pragma unroll
    for (int ww = 0; ww < kGruThreads / 32; ++ww) s += red[ww * V * 32 + o];
    parts[(int64_t)blockIdx.x * (V * 32) + o] = s;
  }
}

// dW_hh = dgh^T . h_prev over the T*N rows: [3H, H] accumulated in registers by a persistent CTA per SM (thread = 6 gate
// rows x H/8 hidden columns), 32-row chunks of both operands double-buffered in shared memory with cp.async; h_prev is
// read in place from the saved buffer (row stride ps = 5H).  cuBLAS takes 6.1 ms for this 288 x 96 x 3.3 M product at the
// C2 shape (30 TFLOP/s); rows are summed in index order per CTA, the per-CTA tiles by the caller.  The same kernel gives
// dW_ih of a stacked layer as dgi^T . h_seq of the layer below (ps = H).
constexpr int kGruWgChunk = 32;

template <int H>
__global__ void __launch_bounds__(4 * H, 1)
k_gru_wgrad(const float* __restrict__ dgh, const float* __restrict__ saved, int64_t ps, int64_t rows,
            float* __restrict__ parts) {
  constexpr int G3 = 3 * H, CW = H / 8, CH = kGruWgChunk, NT = 4 * H;
  extern __shared__ __align__(16) float sm[];
  float* Gs = sm;                  // [2][CH][3H]
  float* Ps = sm + 2 * CH * G3;    // [2][CH][H]
  const int tid = threadIdx.x, b = tid & 7, a = tid >> 3;
  f32x2 acc[6][CW / 2];          // pairs of adjacent hidden columns (FFMA2: the gate value is duplicated, h_prev pairs are natural)
#pragma unroll
  for (int m = 0; m < 6; ++m)
#pragma unroll
    for (int n = 0; n < CW / 2; ++n) acc[m][n] = 0ull;
  const int64_t nchunks = ceil_div<int64_t>(rows, CH);

  auto load = [&](int stage, int64_t c) {
    const int64_t r0 = c * CH;
    const int nr = (int)min((int64_t)CH, rows - r0);
    float* gd = Gs + stage * CH * G3;
    const float* gsrc = dgh + r0 * G3;
    for (int i = tid; i < CH * G3 / 4; i += NT) {
      if (i / (G3 / 4) < nr) cp_async16(gd + 4 * i, gsrc + 4 * i);
      else *reinterpret_cast<float4*>(gd + 4 * i) = f4zero();
    }
    float* pd = Ps + stage * CH * H;
    for (int i = tid; i < CH * H / 4; i += NT) {
      const int r = i / (H / 4), c4 = i % (H / 4);
      if (r < nr) cp_async16(pd + 4 * i, saved + (r0 + r) * ps + 4 * c4);
      else *reinterpret_cast<float4*>(pd + 4 * i) = f4zero();
    }
    cp_async_commit();
  };

  int stage = 0;
  if ((int64_t)blockIdx.x < nchunks) load(0, blockIdx.x);
  for (int64_t c = blockIdx.x; c < nchunks; c += gridDim.x) {
    const int64_t nxt = c + gridDim.x;
    if (nxt < nchunks) { load(stage ^ 1, nxt); cp_async_wait<1>(); }
    else cp_async_wait<0>();
    __syncthreads();
    const float* g = Gs + stage * CH * G3 + 6 * a;
    const float* p = Ps + stage * CH * H + CW * b;
#pragma unroll 4
    for (int r = 0; r < CH; ++r) {
      const float2 g0 = *reinterpret_cast<const float2*>(g + r * G3);
      const float2 g1 = *reinterpret_cast<const float2*>(g + r * G3 + 2);
      const float2 g2 = *reinterpret_cast<const float2*>(g + r * G3 + 4);
      const f32x2 gv[6] = {f32x2_dup(g0.x), f32x2_dup(g0.y), f32x2_dup(g1.x), f32x2_dup(g1.y), f32x2_dup(g2.x), f32x2_dup(g2.y)};
#pragma unroll
      for (int q = 0; q < CW / 4; ++q) {
        const ulonglong2 pv = *reinterpret_cast<const ulonglong2*>(p + r * H + 4 * q);
#pragma unroll
        for (int m = 0; m < 6; ++m) {
          acc[m][2 * q + 0] = ffma2(gv[m], pv.x, acc[m][2 * q + 0]);
          acc[m][2 * q + 1] = ffma2(gv[m], pv.y, acc[m][2 * q + 1]);
        }
      }
    }
    __syncthreads();
    stage ^= 1;
  }
  float* out = parts + (int64_t)blockIdx.x * G3 * H;
#pragma unroll
  for (int m = 0; m < 6; ++m)
#pragma unroll
    for (int q = 0; q < CW / 4; ++q) {
      ulonglong2 v;
      v.x = acc[m][2 * q]; v.y = acc[m][2 * q + 1];
      *reinterpret_cast<ulonglong2*>(out + (6 * a + m) * H + CW * b + 4 * q) = v;
    }
}


// Input projection of a stacked layer and its data gradient: row GEMMs over the T*N rows against W_ih [3H,H],
//   FWD: gi[r] = b_ih + h_seq[r] . W_ih^T   ([H] -> [3H]);      BWD: dY[r] = dgi[r] . W_ih   ([3H] -> [H]).
// W_ih sits in shared memory as Ws[n][k] (row stride K+4: conflict-free 128-bit loads with lane = output column, as in
// the recurrences); a persistent CTA per SM streams chunks of 8*RM input rows, one H-wide k panel at a time,
// double-buffered with cp.async.  A warp owns RM rows (read as broadcasts), a lane NO/32 output columns; each output is
// one FP32 FMA chain in sequential k order (FWD starts from the bias).
template <int H, bool FWD>
__global__ void __launch_bounds__(kGruThreads, 1)
k_gru_proj(const float* __restrict__ in, int64_t rows, const float* __restrict__ W_ih, const float* __restrict__ b_ih,
           float* __restrict__ out) {
  constexpr int K = FWD ? H : 3 * H, NO = FWD ? 3 * H : H, LDW = K + 4, CN = NO / 32, RM = FWD ? 8 : 16;
  constexpr int P = K / H, CH = (kGruThreads / 32) * RM;
  extern __shared__ __align__(16) float sm[];
  float* Ws = sm;                 // [NO][LDW]
  float* Xs = Ws + NO * LDW;      // [2][CH][H]
  const int tid = threadIdx.x, w = tid >> 5, l = tid & 31;
  for (int i = tid; i < 3 * H * H; i += kGruThreads) {
    if (FWD) Ws[(i / H) * LDW + i % H] = __ldg(W_ih + i);        // W_ih[n][k]
    else Ws[(i % H) * LDW + i / H] = __ldg(W_ih + i);            // W_ih[k][n]
  }
  float bias[CN];
#pragma unroll
  for (int c = 0; c < CN; ++c) bias[c] = FWD ? __ldg(b_ih + l + 32 * c) : 0.f;
  const int64_t nchunks = ceil_div<int64_t>(rows, CH);

  auto load = [&](int stage, int64_t c, int p) {
    const int64_t r0 = c * CH;
    const int nr = (int)min((int64_t)CH, rows - r0);
    float* d = Xs + stage * CH * H;
    const float* src = in + r0 * K + p * H;
    for (int i = tid; i < CH * H / 4; i += kGruThreads) {
      const int r = i / (H / 4), c4 = i % (H / 4);
      if (r < nr) cp_async16(d + 4 * i, src + (int64_t)r * K + 4 * c4);
      else *reinterpret_cast<float4*>(d + 4 * i) = f4zero();
    }
    cp_async_commit();
  };

  float acc[RM][CN];
  int stage = 0, p = 0;
  int64_t c = blockIdx.x;
  if (c < nchunks) load(0, c, 0);
  __syncthreads();   // the weights are in shared memory
  while (c < nchunks) {
    int64_t c2 = c;
    int p2 = p + 1;
    if (p2 == P) { p2 = 0; c2 += gridDim.x; }
    if (c2 < nchunks) { load(stage ^ 1, c2, p2); cp_async_wait<1>(); }
    else cp_async_wait<0>();
    __syncthreads();
    if (p == 0) {
#pragma unroll
      for (int i = 0; i < RM; ++i)
#pragma unroll
        for (int cc = 0; cc < CN; ++cc) acc[i][cc] = bias[cc];
    }
    const float* xr = Xs + stage * CH * H + w * RM * H;
    const float* wr = Ws + l * LDW + p * H;
#pragma unroll 2
    for (int k = 0; k < H; k += 4) {
      float4 xv[RM];
#pragma unroll
      for (int i = 0; i < RM; ++i) xv[i] = *reinterpret_cast<const float4*>(xr + i * H + k);
#pragma unroll
      for (int cc = 0; cc < CN; ++cc) {
        const float4 wv = *reinterpret_cast<const float4*>(wr + 32 * cc * LDW + k);
#pragma unroll
        for (int i = 0; i < RM; ++i) fma4(acc[i][cc], xv[i], wv);
      }
    }
    if (p == P - 1) {
      const int64_t rb = c * CH + w * RM;
#pragma unroll
      for (int i = 0; i < RM; ++i)
        if (rb + i < rows) {
#pragma unroll
          for (int cc = 0; cc < CN; ++cc) out[(rb + i) * NO + l + 32 * cc] = acc[i][cc];
        }
    }
    __syncthreads();
    stage ^= 1; c = c2; p = p2;
  }
}

int64_t gru_wgrad_tiles(int64_t rows) {
  return std::min<int64_t>(num_sms(), ceil_div<int64_t>(rows, kGruWgChunk));
}

template <int H>
int gru_wgrad_launch(const float* dgh, const float* a, int64_t ps, int64_t rows, float* parts, cudaStream_t s) {
  const int64_t smem = 2ll * kGruWgChunk * 4 * H * 4;
  SLDM_OPT_IN_SMEM((k_gru_wgrad<H>), smem);
  k_gru_wgrad<H><<<(unsigned)gru_wgrad_tiles(rows), 4 * H, (size_t)smem, s>>>(dgh, a, ps, rows, parts);
  SLDM_LAUNCH_CHECK("k_gru_wgrad");
  return SLDM_OK;
}

int64_t gru_fwd_smem(int H, int T, int I) {
  return 4ll * (3ll * H * (H + 4) + (int64_t)kGruRows * H + 3ll * H * kGruLdi + 4ll * H + (int64_t)kGruRows * T * I);
}
int64_t gru_fwd_gi_smem(int H) {
  return 4ll * (3ll * H * (H + 4) + (int64_t)kGruRows * H + 4ll * H + (int64_t)kGruRows * 3 * H);
}
int64_t gru_bwd_smem(int H, int T, int I) {   // I = 0: the deep mode (no x tile)
  const int64_t main_part = (int64_t)H * (3 * H + 4) + (int64_t)kGruRows * 3 * H;
  const int64_t red = 8ll * 28 * (H / 32) * 32;
  return 4ll * (std::max(main_part, red) + (int64_t)kGruRows * T * I);
}
constexpr int gru_proj_rows(bool fwd) { return (kGruThreads / 32) * (fwd ? 8 : 16); }
int64_t gru_proj_smem(int H, bool fwd) {
  return 4ll * (fwd ? 3ll * H * (H + 4) : (int64_t)H * (3 * H + 4)) + 4ll * 2 * gru_proj_rows(fwd) * H;
}
bool gru_hidden_ok(int32_t H) { return H == 32 || H == 64 || H == 96; }

int gru_check(const char* who, int64_t N, int32_t T, int32_t I, int32_t H) {
  SLDM_REQUIRE(N >= 0 && T >= 1 && I >= 1, SLDM_EINVAL, "%s: bad sizes N=%lld T=%d I=%d", who, (long long)N, T, I);
  SLDM_REQUIRE(gru_hidden_ok(H), SLDM_EUNSUPPORTED, "%s: hidden size %d (fused path: 32, 64, 96)", who, H);
  SLDM_REQUIRE(I <= kGruMaxI, SLDM_EUNSUPPORTED, "%s: input width %d > %d", who, I, kGruMaxI);
  SLDM_REQUIRE(std::max(gru_fwd_smem(H, T, I), gru_bwd_smem(H, T, I)) <= kGruSmemMax, SLDM_EUNSUPPORTED,
               "%s: %d steps x %d inputs do not fit the shared-memory tile", who, T, I);
  SLDM_REQUIRE(ceil_div<int64_t>(N, kGruRows) < (1ll << 31), SLDM_EUNSUPPORTED, "%s: N too large", who);
  return SLDM_OK;
}
// a layer fed by the layer below (gi / dh_seq): no input width, no shared-memory limit on T
int gru_check_deep(const char* who, int64_t N, int32_t T, int32_t H) {
  SLDM_REQUIRE(N >= 0 && T >= 1, SLDM_EINVAL, "%s: bad sizes N=%lld T=%d", who, (long long)N, T);
  SLDM_REQUIRE(gru_hidden_ok(H), SLDM_EUNSUPPORTED, "%s: hidden size %d (fused path: 32, 64, 96)", who, H);
  SLDM_REQUIRE(ceil_div<int64_t>(N, kGruRows) < (1ll << 31), SLDM_EUNSUPPORTED, "%s: N too large", who);
  return SLDM_OK;
}

template <int H, bool SAVE, bool GI>
int gru_fwd_go(const float* x, const float* gi, int64_t N, int T, int I, const float* W_ih, const float* W_hh,
               const float* b_ih, const float* b_hh, float* h_last, float* saved, float* h_seq, cudaStream_t s) {
  const int64_t smem = GI ? gru_fwd_gi_smem(H) : gru_fwd_smem(H, T, I);
  const unsigned grid = (unsigned)ceil_div<int64_t>(N, kGruRows);
  SLDM_OPT_IN_SMEM((k_gru_fwd<H, SAVE, GI>), kGruSmemMax);
  k_gru_fwd<H, SAVE, GI><<<grid, kGruThreads, (size_t)smem, s>>>(x, gi, N, T, I, W_ih, W_hh, b_ih, b_hh, h_last,
                                                                  saved, h_seq);
  SLDM_LAUNCH_CHECK("k_gru_fwd");
  return SLDM_OK;
}

template <int H>
int gru_fwd_launch(const float* x, const float* gi, int64_t N, int T, int I, const float* W_ih, const float* W_hh,
                   const float* b_ih, const float* b_hh, float* h_last, float* saved, float* h_seq, cudaStream_t s) {
  if (gi != nullptr)
    return saved != nullptr ? gru_fwd_go<H, true, true>(x, gi, N, T, I, W_ih, W_hh, b_ih, b_hh, h_last, saved, h_seq, s)
                            : gru_fwd_go<H, false, true>(x, gi, N, T, I, W_ih, W_hh, b_ih, b_hh, h_last, saved, h_seq, s);
  return saved != nullptr ? gru_fwd_go<H, true, false>(x, gi, N, T, I, W_ih, W_hh, b_ih, b_hh, h_last, saved, h_seq, s)
                          : gru_fwd_go<H, false, false>(x, gi, N, T, I, W_ih, W_hh, b_ih, b_hh, h_last, saved, h_seq, s);
}

template <int H, bool DEEP>
int gru_bwd_go(const float* x, int64_t N, int T, int I, const float* W_hh, const float* dh_last, const float* dh_seq,
               const float* saved, float* dgh, float* gin, float* dgi, float* parts, cudaStream_t s) {
  const int64_t smem = gru_bwd_smem(H, T, DEEP ? 0 : I);
  const unsigned grid = (unsigned)ceil_div<int64_t>(N, kGruRows);
  SLDM_OPT_IN_SMEM((k_gru_bwd<H, DEEP>), kGruSmemMax);
  k_gru_bwd<H, DEEP><<<grid, kGruThreads, (size_t)smem, s>>>(x, N, T, I, W_hh, dh_last, dh_seq, saved, dgh, gin, dgi,
                                                             parts);
  SLDM_LAUNCH_CHECK("k_gru_bwd");
  return SLDM_OK;
}

template <int H>
int gru_bwd_launch(const float* x, int64_t N, int T, int I, const float* W_hh, const float* dh_last, const float* dh_seq,
                   const float* saved, float* dgh, float* gin, float* dgi, float* parts, cudaStream_t s) {
  return x == nullptr ? gru_bwd_go<H, true>(x, N, T, I, W_hh, dh_last, dh_seq, saved, dgh, gin, dgi, parts, s)
                      : gru_bwd_go<H, false>(x, N, T, I, W_hh, dh_last, dh_seq, saved, dgh, gin, dgi, parts, s);
}

template <int H, bool FWD>
int gru_proj_launch(const float* in, int64_t rows, const float* W_ih, const float* b_ih, float* out, cudaStream_t s) {
  const int64_t smem = gru_proj_smem(H, FWD);
  const unsigned grid = (unsigned)std::min<int64_t>(num_sms(), ceil_div<int64_t>(rows, gru_proj_rows(FWD)));
  SLDM_OPT_IN_SMEM((k_gru_proj<H, FWD>), smem);
  k_gru_proj<H, FWD><<<grid, kGruThreads, (size_t)smem, s>>>(in, rows, W_ih, b_ih, out);
  SLDM_LAUNCH_CHECK("k_gru_proj");
  return SLDM_OK;
}

int gru_forward_impl(const char* who, const float* x, const float* gi, int64_t N, int32_t T, int32_t I, int32_t H,
                     const float* W_ih, const float* W_hh, const float* b_ih, const float* b_hh, float* h_last,
                     float* saved, float* h_seq, sldm_stream_t stream) {
  int rc = gi != nullptr ? gru_check_deep(who, N, T, H) : gru_check(who, N, T, I, H);
  if (rc) return rc;
  if (N == 0) return SLDM_OK;
  SLDM_REQUIRE(W_hh && b_hh && (gi ? x == nullptr : x && W_ih && b_ih), SLDM_EINVAL, "%s: NULL pointer", who);
  SLDM_REQUIRE((reinterpret_cast<uintptr_t>(W_hh) & 15u) == 0, SLDM_EINVAL, "%s: W_hh must be 16-byte aligned", who);
  SLDM_REQUIRE((reinterpret_cast<uintptr_t>(gi) & 15u) == 0, SLDM_EINVAL, "%s: gi must be 16-byte aligned", who);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (H) {
    case 32: return gru_fwd_launch<32>(x, gi, N, T, I, W_ih, W_hh, b_ih, b_hh, h_last, saved, h_seq, s);
    case 64: return gru_fwd_launch<64>(x, gi, N, T, I, W_ih, W_hh, b_ih, b_hh, h_last, saved, h_seq, s);
    default: return gru_fwd_launch<96>(x, gi, N, T, I, W_ih, W_hh, b_ih, b_hh, h_last, saved, h_seq, s);
  }
}

int gru_backward_impl(const char* who, const float* x, int64_t N, int32_t T, int32_t I, int32_t H, const float* W_hh,
                      const float* dh_last, const float* dh_seq, const float* saved, float* dgh, float* dgi_n,
                      float* dgi, float* partials, int64_t partial_rows, sldm_stream_t stream) {
  int rc = x == nullptr ? gru_check_deep(who, N, T, H) : gru_check(who, N, T, I, H);
  if (rc) return rc;
  if (N == 0) return SLDM_OK;
  SLDM_REQUIRE(W_hh && saved && dgh && partials, SLDM_EINVAL, "%s: NULL pointer", who);
  SLDM_REQUIRE(partial_rows >= ceil_div<int64_t>(N, kGruRows), SLDM_EWORKSPACE,
               "%s: %lld partial rows < %lld", who, (long long)partial_rows, (long long)ceil_div<int64_t>(N, kGruRows));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (H) {
    case 32: return gru_bwd_launch<32>(x, N, T, I, W_hh, dh_last, dh_seq, saved, dgh, dgi_n, dgi, partials, s);
    case 64: return gru_bwd_launch<64>(x, N, T, I, W_hh, dh_last, dh_seq, saved, dgh, dgi_n, dgi, partials, s);
    default: return gru_bwd_launch<96>(x, N, T, I, W_hh, dh_last, dh_seq, saved, dgh, dgi_n, dgi, partials, s);
  }
}

int gru_wgrad_impl(const char* who, const float* dgh, const float* a, int64_t a_stride, int64_t N, int32_t T, int32_t H,
                   float* partials, int64_t partial_tiles, sldm_stream_t stream) {
  SLDM_REQUIRE(N >= 0 && T >= 1, SLDM_EINVAL, "%s: bad sizes N=%lld T=%d", who, (long long)N, T);
  SLDM_REQUIRE(gru_hidden_ok(H), SLDM_EUNSUPPORTED, "%s: hidden size %d (fused path: 32, 64, 96)", who, H);
  SLDM_REQUIRE(a_stride >= H && a_stride % 4 == 0, SLDM_EINVAL, "%s: row stride %lld (>= H, a multiple of 4)", who,
               (long long)a_stride);
  const int64_t rows = N * (int64_t)T;
  if (rows == 0) return SLDM_OK;
  SLDM_REQUIRE(dgh && a && partials, SLDM_EINVAL, "%s: NULL pointer", who);
  SLDM_REQUIRE(partial_tiles >= gru_wgrad_tiles(rows), SLDM_EWORKSPACE, "%s: %lld partial tiles < %lld", who,
               (long long)partial_tiles, (long long)gru_wgrad_tiles(rows));
  SLDM_REQUIRE(((reinterpret_cast<uintptr_t>(dgh) | reinterpret_cast<uintptr_t>(a) |
                 reinterpret_cast<uintptr_t>(partials)) & 15u) == 0, SLDM_EINVAL, "%s: buffers must be 16-byte aligned", who);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (H) {
    case 32: return gru_wgrad_launch<32>(dgh, a, a_stride, rows, partials, s);
    case 64: return gru_wgrad_launch<64>(dgh, a, a_stride, rows, partials, s);
    default: return gru_wgrad_launch<96>(dgh, a, a_stride, rows, partials, s);
  }
}

template <bool FWD>
int gru_project_impl(const char* who, const float* in, int64_t rows, int32_t H, const float* W_ih, const float* b_ih,
                     float* out, sldm_stream_t stream) {
  SLDM_REQUIRE(rows >= 0, SLDM_EINVAL, "%s: bad row count %lld", who, (long long)rows);
  SLDM_REQUIRE(gru_hidden_ok(H), SLDM_EUNSUPPORTED, "%s: hidden size %d (fused path: 32, 64, 96)", who, H);
  if (rows == 0) return SLDM_OK;
  SLDM_REQUIRE(in && W_ih && out && (!FWD || b_ih), SLDM_EINVAL, "%s: NULL pointer", who);
  SLDM_REQUIRE((reinterpret_cast<uintptr_t>(in) & 15u) == 0, SLDM_EINVAL, "%s: input must be 16-byte aligned", who);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (H) {
    case 32: return gru_proj_launch<32, FWD>(in, rows, W_ih, b_ih, out, s);
    case 64: return gru_proj_launch<64, FWD>(in, rows, W_ih, b_ih, out, s);
    default: return gru_proj_launch<96, FWD>(in, rows, W_ih, b_ih, out, s);
  }
}

}  // namespace
}  // namespace sldm

using namespace sldm;

extern "C" int sldm_gru_supported(int32_t T, int32_t I, int32_t H) {
  return gru_hidden_ok(H) && T >= 1 && I >= 1 && I <= kGruMaxI &&
         std::max(gru_fwd_smem(H, T, I), gru_bwd_smem(H, T, I)) <= kGruSmemMax;
}

extern "C" int sldm_gru_stack_supported(int32_t T, int32_t I, int32_t H) {
  return sldm_gru_supported(T, I, H) && std::max(gru_fwd_gi_smem(H), gru_bwd_smem(H, T, 0)) <= kGruSmemMax &&
         std::max(gru_proj_smem(H, true), gru_proj_smem(H, false)) <= kGruSmemMax;
}

extern "C" int64_t sldm_gru_partial_rows(int64_t N) { return N < 0 ? -1 : ceil_div<int64_t>(N, kGruRows); }
extern "C" int64_t sldm_gru_partial_width(int32_t H) { return H > 0 && H % 32 == 0 ? 28ll * H : -1; }

extern "C" int sldm_gru_forward(const float* x, int64_t N, int32_t T, int32_t I, int32_t H,
                                const float* W_ih, const float* W_hh, const float* b_ih, const float* b_hh,
                                float* h_last, float* saved, sldm_stream_t stream) {
  int rc = gru_check("sldm_gru_forward", N, T, I, H);
  if (rc) return rc;
  if (N == 0) return SLDM_OK;
  SLDM_REQUIRE(x && h_last, SLDM_EINVAL, "sldm_gru_forward: NULL pointer");
  return gru_forward_impl("sldm_gru_forward", x, nullptr, N, T, I, H, W_ih, W_hh, b_ih, b_hh, h_last, saved, nullptr,
                          stream);
}

extern "C" int sldm_gru_layer_forward(const float* x, const float* gi, int64_t N, int32_t T, int32_t I, int32_t H,
                                      const float* W_ih, const float* W_hh, const float* b_ih, const float* b_hh,
                                      float* h_last, float* saved, float* h_seq, sldm_stream_t stream) {
  return gru_forward_impl("sldm_gru_layer_forward", x, gi, N, T, I, H, W_ih, W_hh, b_ih, b_hh, h_last, saved, h_seq,
                          stream);
}

extern "C" int sldm_gru_backward(const float* x, int64_t N, int32_t T, int32_t I, int32_t H, const float* W_hh,
                                 const float* dh_last, const float* saved, float* dgh, float* dgi_n, float* partials,
                                 int64_t partial_rows, sldm_stream_t stream) {
  int rc = gru_check("sldm_gru_backward", N, T, I, H);
  if (rc) return rc;
  if (N == 0) return SLDM_OK;
  SLDM_REQUIRE(x && dh_last, SLDM_EINVAL, "sldm_gru_backward: NULL pointer");
  return gru_backward_impl("sldm_gru_backward", x, N, T, I, H, W_hh, dh_last, nullptr, saved, dgh, dgi_n, nullptr,
                           partials, partial_rows, stream);
}

extern "C" int sldm_gru_layer_backward(const float* x, int64_t N, int32_t T, int32_t I, int32_t H, const float* W_hh,
                                       const float* dh_last, const float* dh_seq, const float* saved, float* dgh,
                                       float* dgi_n, float* dgi, float* partials, int64_t partial_rows,
                                       sldm_stream_t stream) {
  return gru_backward_impl("sldm_gru_layer_backward", x, N, T, I, H, W_hh, dh_last, dh_seq, saved, dgh, dgi_n, dgi,
                           partials, partial_rows, stream);
}

extern "C" int sldm_gru_project_forward(const float* h_seq, int64_t rows, int32_t H, const float* W_ih,
                                        const float* b_ih, float* gi, sldm_stream_t stream) {
  return gru_project_impl<true>("sldm_gru_project_forward", h_seq, rows, H, W_ih, b_ih, gi, stream);
}

extern "C" int sldm_gru_project_backward(const float* dgi, int64_t rows, int32_t H, const float* W_ih, float* dy,
                                         sldm_stream_t stream) {
  return gru_project_impl<false>("sldm_gru_project_backward", dgi, rows, H, W_ih, nullptr, dy, stream);
}

extern "C" int64_t sldm_gru_wgrad_tiles(int64_t N, int32_t T) {
  if (N < 0 || T < 1) return -1;
  return gru_wgrad_tiles(N * (int64_t)T);
}

extern "C" int sldm_gru_wgrad(const float* dgh, const float* saved, int64_t N, int32_t T, int32_t H,
                              float* partials, int64_t partial_tiles, sldm_stream_t stream) {
  return gru_wgrad_impl("sldm_gru_wgrad", dgh, saved, 5ll * H, N, T, H, partials, partial_tiles, stream);
}

extern "C" int sldm_gru_wgrad_strided(const float* dg, const float* a, int64_t a_stride, int64_t N, int32_t T,
                                      int32_t H, float* partials, int64_t partial_tiles, sldm_stream_t stream) {
  return gru_wgrad_impl("sldm_gru_wgrad_strided", dg, a, a_stride, N, T, H, partials, partial_tiles, stream);
}
