// Radial-MLP hidden layer (K = 8) on CUDA cores, sm_100a.
//
// Reference op (paths under /root/reference):
//   edge_weight = ScalarMLPFunction(edge_embedding)            nequip/nn/mlp.py:80-195, 262-268
//   built with depth 1 by InteractionBlock                     nequip/nn/interaction_block.py:119-127, 196
//     h   = silu(emb @ (W1 * a1))          [E, NB] x [NB, H]   (NB = 8 Bessel functions, H = 128)   <- here
//     w   =      h   @ (W2 * a2)           [E, H ] x [H, W]    nqb_gemm.cu (unfused) / the fused TP kernels
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/nqb.h"
#include "nqb_tc.cuh"

namespace {

constexpr int H = 128;       // hidden width == K of the second-layer GEMM
constexpr int NB = 8;        // Bessel functions

// ---------------------------------------------------------------------------------------------
// first radial layer on CUDA cores (K = 8): h = silu(emb @ W1s)  and its backward
//   gemb[e, k] = sum_m gh[e, m] * silu'(pre[e, m]) * W1s[k, m],  pre recomputed from emb
// (feeds / follows the grouped tensor-core GEMM of the second layer, nqb_gemm.cu)
// ---------------------------------------------------------------------------------------------
// Persistent warps: lane = 4 hidden units whose 8 x 4 first-layer weights live in registers for the whole
// kernel; a warp walks over edges (grid-stride), reads the 8 basis values of the edge (one broadcast
// 32-byte load) and writes the edge's 128 activations as one 512-byte row.  (The first version re-staged
// the 4 KB weight matrix per 8 edges -- as many bytes as it wrote.)
__device__ __forceinline__ float sigmoid_fast(float p) { return __fdividef(1.0f, 1.0f + expf(-p)); }

__global__ void __launch_bounds__(256) k_hidden_fwd(const float* __restrict__ emb, const float* __restrict__ W1s,
                                                    int64_t E, float* __restrict__ h, float* __restrict__ h_lo) {
  const int lane = threadIdx.x & 31, m0 = lane * 4;
  float w[NB][4];
#pragma unroll
  for (int k = 0; k < NB; ++k) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(W1s + k * H + m0));
    w[k][0] = t.x; w[k][1] = t.y; w[k][2] = t.z; w[k][3] = t.w;
  }
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t e = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); e < E; e += nwarps) {
    const float4 x0 = __ldg(reinterpret_cast<const float4*>(emb + e * NB));
    const float4 x1 = __ldg(reinterpret_cast<const float4*>(emb + e * NB + 4));
    const float x[NB] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
    float o[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float p = 0.f;
#pragma unroll
      for (int k = 0; k < NB; ++k) p = fmaf(x[k], w[k][q], p);
      o[q] = p * sigmoid_fast(p);
    }
    __stcs(reinterpret_cast<float4*>(h + e * H + m0), make_float4(o[0], o[1], o[2], o[3]));
    if (h_lo) __stcs(reinterpret_cast<float4*>(h_lo + e * H + m0), make_float4(tf32_lo(o[0]), tf32_lo(o[1]), tf32_lo(o[2]), tf32_lo(o[3])));
  }
}

__global__ void __launch_bounds__(256) k_hidden_bwd(const float* __restrict__ emb, const float* __restrict__ W1s,
                                                    const float* __restrict__ gh, int64_t E, float* __restrict__ gemb) {
  const int lane = threadIdx.x & 31, m0 = lane * 4;
  float w[NB][4];
#pragma unroll
  for (int k = 0; k < NB; ++k) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(W1s + k * H + m0));
    w[k][0] = t.x; w[k][1] = t.y; w[k][2] = t.z; w[k][3] = t.w;
  }
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t e = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); e < E; e += nwarps) {  // warp = edge
  const float4 x0 = __ldg(reinterpret_cast<const float4*>(emb + e * NB));
  const float4 x1 = __ldg(reinterpret_cast<const float4*>(emb + e * NB + 4));
  const float x[NB] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
  const float4 g4 = __ldcs(reinterpret_cast<const float4*>(gh + e * H + m0));
  const float g[4] = {g4.x, g4.y, g4.z, g4.w};
  float acc[NB];
#pragma unroll
  for (int k = 0; k < NB; ++k) acc[k] = 0.f;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float p = 0.f;
#pragma unroll
    for (int k = 0; k < NB; ++k) p = fmaf(x[k], w[k][q], p);
    const float sg = sigmoid_fast(p);
    const float gp = g[q] * (sg * (1.0f + p * (1.0f - sg)));
#pragma unroll
    for (int k = 0; k < NB; ++k) acc[k] = fmaf(gp, w[k][q], acc[k]);
  }
  // reduce the 8 partial sums over the 32 lanes (halving butterfly: 4 + 2 + 1 + 2 shuffles)
#pragma unroll
  for (int o = 16, c = NB; o >= 1; o >>= 1) {
    if (c > 1) {
      c >>= 1;
      const bool up = (lane & o) != 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (j < c) {
          const float mine = up ? acc[j + c] : acc[j];
          const float theirs = up ? acc[j] : acc[j + c];
          acc[j] = mine + __shfl_xor_sync(0xffffffffu, theirs, o);
        }
      }
    } else {
      acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], o);
    }
  }
  // after the three halving steps lane bits (16, 8, 4) select the component: k = 4*b16 + 2*b8 + b4
  if ((lane & 3) == 0) {
    const int k = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
    gemb[e * NB + k] = acc[0];
  }
  }  // edge loop
}


// ---------------------------------------------------------------------------------------------
// v2 of the two kernels (round 2).  The ncu launch list of one step (profiles/r02_launches_li3po4_step.csv)
// has k_hidden_fwd at 109 us and k_hidden_bwd at 183 us per layer -- 2.4x / 3.5x their HBM floors
// (0.32 GB each way).  v1 runs 4 CTAs per SM (55-63 registers) with ONE edge per warp iteration and the
// edge's basis values fetched by a dependent broadcast load at the top of every iteration: 32 edges in
// flight per SM, each paying a full DRAM latency before its arithmetic starts.  v2:
//   * a warp owns a BATCH of 32 consecutive edges; lane j fetches edge j's 8 basis values with two
//     coalesced 16-byte loads (1 KB per warp) and the batch after that is already in flight while the
//     current one is computed; inside the batch the values of edge j are broadcast with warp shuffles,
//     so no load sits on the critical path of an edge;
//   * packed FFMA2 arithmetic (two hidden units per instruction), sigmoid from ex2.approx / rcp.approx
//     (5 instructions; <= 2 ulp each, the result agrees with v1 to ~1e-7 relative);
//   * backward: four edges per inner iteration -- their four grad_h rows are loaded up front and the
//     4 x 8 partial sums are reduced with one 32-value halving butterfly (31 shuffles instead of
//     4 x 9) that leaves element `lane` in lane `lane`: grad_emb is written as one 128-byte row.
// Selected by hidden_variant() below (NQB_HIDDEN_VARIANT / nqb_mlp_hidden_set_variant).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// 1 / (1 + exp(-p));  p -> -inf gives rcp(inf) = 0, p -> +inf gives rcp(1) = 1
__device__ __forceinline__ float sigmoid_v2(float p) { return rcp_approx(1.0f + ex2_approx(p * -1.4426950408889634f)); }

struct Basis8 { float4 a, b; };
__device__ __forceinline__ Basis8 load_basis(const float* __restrict__ emb, int64_t e, int64_t E) {
  Basis8 r;
  if (e < E) {
    r.a = __ldg(reinterpret_cast<const float4*>(emb + e * NB));
    r.b = __ldg(reinterpret_cast<const float4*>(emb + e * NB + 4));
  } else {
    r.a = make_float4(0.f, 0.f, 0.f, 0.f);
    r.b = r.a;
  }
  return r;
}
// the 8 basis values of the batch's edge j (held by lane j), broadcast to every lane
__device__ __forceinline__ void bcast_basis(const Basis8& mine, int j, float (&x)[NB]) {
  x[0] = __shfl_sync(0xffffffffu, mine.a.x, j); x[1] = __shfl_sync(0xffffffffu, mine.a.y, j);
  x[2] = __shfl_sync(0xffffffffu, mine.a.z, j); x[3] = __shfl_sync(0xffffffffu, mine.a.w, j);
  x[4] = __shfl_sync(0xffffffffu, mine.b.x, j); x[5] = __shfl_sync(0xffffffffu, mine.b.y, j);
  x[6] = __shfl_sync(0xffffffffu, mine.b.z, j); x[7] = __shfl_sync(0xffffffffu, mine.b.w, j);
}
// pre-activations of this lane's 4 hidden units: p[q] = sum_k x[k] * W1s[k, m0 + q]  (k ascending, as v1)
__device__ __forceinline__ void preact4(const float (&x)[NB], const float2 (&w01)[NB], const float2 (&w23)[NB],
                                        float2& p01, float2& p23) {
  p01 = make_float2(0.f, 0.f);
  p23 = p01;
#pragma unroll
  for (int k = 0; k < NB; ++k) {
    const float2 xx = make_float2(x[k], x[k]);
    p01 = __ffma2_rn(xx, w01[k], p01);
    p23 = __ffma2_rn(xx, w23[k], p23);
  }
}

// kLo: also write the tf32 low parts of h to h_lo (as k_hidden_fwd does); h itself is the same either way
template <bool kLo>
__global__ void __launch_bounds__(256) k_hidden_fwd2(const float* __restrict__ emb, const float* __restrict__ W1s,
                                                     int64_t E, float* __restrict__ h, float* __restrict__ h_lo) {
  const int lane = threadIdx.x & 31, m0 = lane * 4;
  float2 w01[NB], w23[NB];
#pragma unroll
  for (int k = 0; k < NB; ++k) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(W1s + k * H + m0));
    w01[k] = make_float2(t.x, t.y);
    w23[k] = make_float2(t.z, t.w);
  }
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t nbatch = (E + 31) >> 5;
  int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  Basis8 cur = load_basis(emb, b * 32 + lane, b < nbatch ? E : 0);
  for (; b < nbatch; b += nwarps) {
    const int64_t bn = b + nwarps;
    const Basis8 nxt = load_basis(emb, bn * 32 + lane, bn < nbatch ? E : 0);  // in flight during this batch
    const int64_t e0 = b * 32;
    const int cnt = (int)((E - e0) < 32 ? (E - e0) : 32);  // warp-uniform
    float* hrow = h + e0 * H + m0;
#pragma unroll 2
    for (int j = 0; j < cnt; ++j) {
      float x[NB];
      bcast_basis(cur, j, x);
      float2 p01, p23;
      preact4(x, w01, w23, p01, p23);
      float4 o;  // __fmul_rn: no FMA contraction into tf32_lo's subtraction, h_lo is the low part of the stored h
      o.x = __fmul_rn(p01.x, sigmoid_v2(p01.x));
      o.y = __fmul_rn(p01.y, sigmoid_v2(p01.y));
      o.z = __fmul_rn(p23.x, sigmoid_v2(p23.x));
      o.w = __fmul_rn(p23.y, sigmoid_v2(p23.y));
      __stcs(reinterpret_cast<float4*>(hrow + (int64_t)j * H), o);
      if (kLo)
        __stcs(reinterpret_cast<float4*>(h_lo + e0 * H + m0 + (int64_t)j * H),
               make_float4(tf32_lo(o.x), tf32_lo(o.y), tf32_lo(o.z), tf32_lo(o.w)));
    }
    cur = nxt;
  }
}

__global__ void __launch_bounds__(256) k_hidden_bwd2(const float* __restrict__ emb, const float* __restrict__ W1s,
                                                     const float* __restrict__ gh, int64_t E, float* __restrict__ gemb) {
  const int lane = threadIdx.x & 31, m0 = lane * 4;
  float2 w01[NB], w23[NB];
#pragma unroll
  for (int k = 0; k < NB; ++k) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(W1s + k * H + m0));
    w01[k] = make_float2(t.x, t.y);
    w23[k] = make_float2(t.z, t.w);
  }
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t nbatch = (E + 31) >> 5;
  int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  Basis8 cur = load_basis(emb, b * 32 + lane, b < nbatch ? E : 0);
  for (; b < nbatch; b += nwarps) {
    const int64_t bn = b + nwarps;
    const Basis8 nxt = load_basis(emb, bn * 32 + lane, bn < nbatch ? E : 0);
    const int64_t e0 = b * 32;
    const int cnt = (int)((E - e0) < 32 ? (E - e0) : 32);  // warp-uniform
    const float* grow = gh + e0 * H + m0;
#pragma unroll 1
    for (int j0 = 0; j0 < cnt; j0 += 4) {  // four edges per iteration
      float4 g[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        g[u] = (j0 + u < cnt) ? __ldcs(reinterpret_cast<const float4*>(grow + (int64_t)(j0 + u) * H))
                              : make_float4(0.f, 0.f, 0.f, 0.f);
      float v[32];  // v[u * 8 + k]: this lane's share of grad_emb[e0 + j0 + u, k]
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float x[NB];
        bcast_basis(cur, (j0 + u) & 31, x);
        float2 p01, p23;
        preact4(x, w01, w23, p01, p23);
        // gp[q] = grad_h[q] * silu'(p[q]),  silu'(p) = s (1 + p (1 - s))
        const float s0 = sigmoid_v2(p01.x), s1 = sigmoid_v2(p01.y), s2 = sigmoid_v2(p23.x), s3 = sigmoid_v2(p23.y);
        const float2 gp01 = make_float2(g[u].x * (s0 * fmaf(p01.x, 1.0f - s0, 1.0f)), g[u].y * (s1 * fmaf(p01.y, 1.0f - s1, 1.0f)));
        const float2 gp23 = make_float2(g[u].z * (s2 * fmaf(p23.x, 1.0f - s2, 1.0f)), g[u].w * (s3 * fmaf(p23.y, 1.0f - s3, 1.0f)));
#pragma unroll
        for (int k = 0; k < NB; ++k) {
          const float2 t = __ffma2_rn(gp23, w23[k], __fmul2_rn(gp01, w01[k]));
          v[u * 8 + k] = t.x + t.y;
        }
      }
      // halving butterfly over the 32 lanes: after the step with offset o a lane keeps the half of its values
      // whose element index has bit o equal to its own lane bit o; after five steps lane l holds element l
#define NQB_HALVE(O, C)                                                        \
  {                                                                            \
    const bool up = (lane & (O)) != 0;                                         \
    _Pragma("unroll") for (int j = 0; j < (C); ++j) {                          \
      const float mine = up ? v[j + (C)] : v[j];                               \
      const float theirs = up ? v[j] : v[j + (C)];                             \
      v[j] = mine + __shfl_xor_sync(0xffffffffu, theirs, (O));                 \
    }                                                                          \
  }
      NQB_HALVE(16, 16)
      NQB_HALVE(8, 8)
      NQB_HALVE(4, 4)
      NQB_HALVE(2, 2)
      NQB_HALVE(1, 1)
#undef NQB_HALVE
      // element `lane` = (edge j0 + lane / 8, component lane % 8): 128 contiguous bytes per warp
      if (j0 + (lane >> 3) < cnt) gemb[(e0 + j0) * NB + lane] = v[0];
    }
    cur = nxt;
  }
}

}  // namespace

extern "C" int nqb_set_error(const char* msg);  // defined in nqb_runtime.cu
extern "C" void nqb_count_launch(void);

// persistent grid: 8 CTAs of 256 threads per SM (or fewer when there is less work)
static unsigned hidden_grid(int64_t threads) {
  static int sms_dev[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  dev &= 63;
  if (sms_dev[dev] == 0) {
    cudaDeviceGetAttribute(&sms_dev[dev], cudaDevAttrMultiProcessorCount, dev);
    if (sms_dev[dev] <= 0) sms_dev[dev] = 148;
  }
  const int sms = sms_dev[dev];
  const int64_t need = (threads + 255) / 256, cap = (int64_t)sms * 8;
  return (unsigned)(need < cap ? need : cap);
}

// Kernel generation: 2 = the batched kernels above, 1 = the round-1 kernels (kept for A/B timing and as the
// reference of the v2 parity test).  Default NQB_HIDDEN_VARIANT_DEFAULT, overridden by the environment variable
// NQB_HIDDEN_VARIANT or at run time by nqb_mlp_hidden_set_variant().
#ifndef NQB_HIDDEN_VARIANT_DEFAULT
#define NQB_HIDDEN_VARIANT_DEFAULT 2
#endif
static int g_hidden_variant = 0;  // 0 = not initialised
static int hidden_variant() {
  if (g_hidden_variant == 0) {
    const char* e = getenv("NQB_HIDDEN_VARIANT");
    g_hidden_variant = (e != nullptr && (e[0] == '1' || e[0] == '2')) ? (e[0] - '0') : NQB_HIDDEN_VARIANT_DEFAULT;
  }
  return g_hidden_variant;
}
extern "C" int nqb_mlp_hidden_set_variant(int variant) {  // returns the previous one; 0 = query only
  const int prev = hidden_variant();
  if (variant == 1 || variant == 2) g_hidden_variant = variant;
  return prev;
}

// v2: persistent grid of exactly the resident CTAs (occupancy x SMs), so that a warp sees several batches and
// its next batch is always prefetched; fewer CTAs when there are fewer batches than warps
template <typename K>
static unsigned hidden_grid2(K kernel, int which, int64_t E) {
  static int ctas_dev[3][64] = {{0}, {0}, {0}};
  int dev = 0;
  cudaGetDevice(&dev);
  dev &= 63;
  if (ctas_dev[which][dev] == 0) {
    int sms = 0, occ = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, 256, 0) != cudaSuccess || occ <= 0) occ = 2;
    ctas_dev[which][dev] = (sms > 0 ? sms : 148) * occ;
  }
  const int64_t need = (((E + 31) >> 5) + 7) / 8;  // 8 warps per CTA, one batch of 32 edges per warp
  return (unsigned)(need < ctas_dev[which][dev] ? need : ctas_dev[which][dev]);
}

extern "C" int nqb_mlp_hidden_fwd(const float* emb, const float* W1s, int64_t E, int num_bessel, int hidden, float* h,
                                  float* h_lo, nqb_stream_t st) {
  if (num_bessel != NB || hidden != H) return nqb_set_error("nqb_mlp_hidden_fwd: only num_bessel=8, hidden=128 is built");
  if (E < 0) return nqb_set_error("nqb_mlp_hidden_fwd: negative size");
  if (E == 0) return 0;
  if (!emb || !W1s || !h) return nqb_set_error("nqb_mlp_hidden_fwd: null pointer");
  const int64_t threads = E * 32;
  // the variant alone picks the kernel: asking for h_lo must not change h
  if (hidden_variant() == 2 && h_lo == nullptr)
    k_hidden_fwd2<false><<<hidden_grid2(k_hidden_fwd2<false>, 0, E), 256, 0, (cudaStream_t)st>>>(emb, W1s, E, h, nullptr);
  else if (hidden_variant() == 2)
    k_hidden_fwd2<true><<<hidden_grid2(k_hidden_fwd2<true>, 2, E), 256, 0, (cudaStream_t)st>>>(emb, W1s, E, h, h_lo);
  else
    k_hidden_fwd<<<hidden_grid(threads), 256, 0, (cudaStream_t)st>>>(emb, W1s, E, h, h_lo);
  nqb_count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return nqb_set_error(cudaGetErrorString(e));
  return 0;
}

extern "C" int nqb_mlp_hidden_bwd(const float* emb, const float* W1s, const float* grad_h, int64_t E, int num_bessel,
                                  int hidden, float* grad_emb, nqb_stream_t st) {
  if (num_bessel != NB || hidden != H) return nqb_set_error("nqb_mlp_hidden_bwd: only num_bessel=8, hidden=128 is built");
  if (E < 0) return nqb_set_error("nqb_mlp_hidden_bwd: negative size");
  if (E == 0) return 0;
  if (!emb || !W1s || !grad_h || !grad_emb) return nqb_set_error("nqb_mlp_hidden_bwd: null pointer");
  const int64_t threads = E * 32;
  if (hidden_variant() == 2)
    k_hidden_bwd2<<<hidden_grid2(k_hidden_bwd2, 1, E), 256, 0, (cudaStream_t)st>>>(emb, W1s, grad_h, E, grad_emb);
  else
    k_hidden_bwd<<<hidden_grid(threads), 256, 0, (cudaStream_t)st>>>(emb, W1s, grad_h, E, grad_emb);
  nqb_count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return nqb_set_error(cudaGetErrorString(e));
  return 0;
}
