// common.cuh -- shared device code of libmappo_b200 (sm_100a).
//
// Data layout inside a CTA: every activation tile is kept TRANSPOSED in shared memory,
// tile[feature][row] with leading dimension LD = TR + 4 floats.  With that layout
//   * a thread's 4 consecutive rows are one aligned float4 (LDS.128),
//   * the three GEMM shapes of an MLP layer (forward  Y = X W^T, input grad dX = dY W, weight grad
//     dW = dY^T X) all read both operands with unit or odd stride, i.e. bank-conflict free,
//   * LayerNorm statistics are a walk down a column with consecutive rows in consecutive banks.
// Weights live in shared memory in the PyTorch [out][in] layout with an ODD leading dimension.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "../../include/mappo_b200.h"

namespace mappo {

constexpr int kMaxHeads = MAPPO_MAX_HEADS;
constexpr int kMaxLayers = MAPPO_MAX_LAYERS;
constexpr float kLnEps = 1e-5f;          // nn.LayerNorm default eps (mlp.py:19,47; rnn.py:22)

// Host/device description of one net: the C-ABI desc + layout, flattened for pass-by-value.
struct NetDev {
  int in_dim, hid, layer_n, use_fn, use_relu, recurrent, n_heads, is_critic;
  int head_dim[kMaxHeads];
  int head_total;
  mappo_net_layout_t g;      // offsets in the flat global parameter / gradient vector
};

// Offsets of the shared-memory weight image (odd leading dimensions).
struct SmemW {
  int fn_w, fn_b, fc1_w, ld1, fc1_b, ln1_w, ln1_b;
  int fc2_w[kMaxLayers], fc2_b[kMaxLayers], ln2_w[kMaxLayers], ln2_b[kMaxLayers];
  int ldh;                   // leading dimension of every [*, H] matrix (H | 1)
  int wih, whh, bih, bhh, rln_w, rln_b;
  int head_w, head_b;
  int total;                 // floats, rounded up to a multiple of 4
};

__host__ __device__ inline SmemW make_smem_w(const NetDev& n, bool with_gru) {
  SmemW s;
  int o = 0;
  const int H = n.hid;
  s.ld1 = n.in_dim | 1;
  s.ldh = H | 1;
  s.fn_w = o; o += n.use_fn ? n.in_dim : 0;
  s.fn_b = o; o += n.use_fn ? n.in_dim : 0;
  s.fc1_w = o; o += H * s.ld1;
  s.fc1_b = o; o += H;
  s.ln1_w = o; o += H;
  s.ln1_b = o; o += H;
  for (int l = 0; l < kMaxLayers; ++l) {
    const bool on = l < n.layer_n;
    s.fc2_w[l] = o; o += on ? H * s.ldh : 0;
    s.fc2_b[l] = o; o += on ? H : 0;
    s.ln2_w[l] = o; o += on ? H : 0;
    s.ln2_b[l] = o; o += on ? H : 0;
  }
  const bool gru = with_gru && n.recurrent;
  s.wih = o; o += gru ? 3 * H * s.ldh : 0;
  s.whh = o; o += gru ? 3 * H * s.ldh : 0;
  s.bih = o; o += gru ? 3 * H : 0;
  s.bhh = o; o += gru ? 3 * H : 0;
  s.rln_w = o; o += (with_gru && n.recurrent) ? H : 0;
  s.rln_b = o; o += (with_gru && n.recurrent) ? H : 0;
  s.head_w = o; o += n.head_total * s.ldh;
  s.head_b = o; o += n.head_total;
  s.total = (o + 3) & ~3;
  return s;
}

// ---------------------------------------------------------------------------------------------
// weight image: global flat params -> shared memory
// ---------------------------------------------------------------------------------------------
// Weights go global -> shared with cp.async (LDGSTS): no register staging, every copy of a thread in flight at
// once, so the whole image costs one L2/HBM latency instead of one per element.  Call cp_async_wait_all() (done at
// the end of load_weights / load_gru_w) and then a block barrier before the first use.
__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

__device__ __forceinline__ void copy_vec(float* dst, const float* __restrict__ src, int n, int tid, int nt) {
  for (int i = tid; i < n; i += nt) cp_async4(dst + i, src + i);
}
__device__ __forceinline__ void copy_mat(float* dst, int ldd, const float* __restrict__ src, int rows, int cols,
                                         int tid, int nt) {
  const int n = rows * cols;
  for (int i = tid; i < n; i += nt) {
    const int r = i / cols, c = i - r * cols;
    cp_async4(dst + r * ldd + c, src + i);
  }
}

__device__ inline void load_weights(float* sW, const SmemW& s, const NetDev& n, const float* __restrict__ p,
                                    bool with_gru, int tid, int nt) {
  const int H = n.hid;
  if (n.use_fn) {
    copy_vec(sW + s.fn_w, p + n.g.fn_w, n.in_dim, tid, nt);
    copy_vec(sW + s.fn_b, p + n.g.fn_b, n.in_dim, tid, nt);
  }
  copy_mat(sW + s.fc1_w, s.ld1, p + n.g.fc1_w, H, n.in_dim, tid, nt);
  copy_vec(sW + s.fc1_b, p + n.g.fc1_b, H, tid, nt);
  copy_vec(sW + s.ln1_w, p + n.g.ln1_w, H, tid, nt);
  copy_vec(sW + s.ln1_b, p + n.g.ln1_b, H, tid, nt);
  for (int l = 0; l < n.layer_n; ++l) {
    copy_mat(sW + s.fc2_w[l], s.ldh, p + n.g.fc2_w[l], H, H, tid, nt);
    copy_vec(sW + s.fc2_b[l], p + n.g.fc2_b[l], H, tid, nt);
    copy_vec(sW + s.ln2_w[l], p + n.g.ln2_w[l], H, tid, nt);
    copy_vec(sW + s.ln2_b[l], p + n.g.ln2_b[l], H, tid, nt);
  }
  if (with_gru && n.recurrent) {
    copy_mat(sW + s.wih, s.ldh, p + n.g.gru_wih, 3 * H, H, tid, nt);
    copy_mat(sW + s.whh, s.ldh, p + n.g.gru_whh, 3 * H, H, tid, nt);
    copy_vec(sW + s.bih, p + n.g.gru_bih, 3 * H, tid, nt);
    copy_vec(sW + s.bhh, p + n.g.gru_bhh, 3 * H, tid, nt);
    copy_vec(sW + s.rln_w, p + n.g.rnn_ln_w, H, tid, nt);
    copy_vec(sW + s.rln_b, p + n.g.rnn_ln_b, H, tid, nt);
  }
  copy_mat(sW + s.head_w, s.ldh, p + n.g.head_w, n.head_total, H, tid, nt);
  copy_vec(sW + s.head_b, p + n.g.head_b, n.head_total, tid, nt);
  cp_async_wait_all();
}

// ---------------------------------------------------------------------------------------------
// tile primitives.  TR rows per tile, NT = 4*TR threads, thread (tx = tid&15, ty = tid>>4) owns rows
// 4*ty..4*ty+3 and output columns tx + 16*j.
// ---------------------------------------------------------------------------------------------
template <int TR> struct Tile {
  static constexpr int LD = TR + 4;
  static constexpr int NT = 4 * TR;
  static constexpr int NTY = TR / 4;
};

enum Act { ACT_NONE = 0, ACT_TANH = 1, ACT_RELU = 2 };

__device__ __forceinline__ float act_fwd(float z, int act) {
  return act == ACT_RELU ? fmaxf(z, 0.f) : (act == ACT_TANH ? tanhf(z) : z);
}
// derivative from the activation OUTPUT a
__device__ __forceinline__ float act_bwd(float a, int act) {
  return act == ACT_RELU ? (a > 0.f ? 1.f : 0.f) : (act == ACT_TANH ? 1.f - a * a : 1.f);
}

// outT[n][r] = act( bias[n] + sum_{k<K} inT[k][r] * W[n*sn + k*sk] ),  n < N  (N <= 16*NJ)
// forward  : W = weight [N][K] (ld odd): sn = ld, sk = 1
// input grad: W = weight [K][N]         : sn = 1,  sk = ld   (contraction over the weight's rows)
template <int TR, int NJ>
__device__ __forceinline__ void tile_mm(const float* __restrict__ inT, int K, const float* __restrict__ W, int sn,
                                        int sk, int N, const float* __restrict__ bias, int act,
                                        float* __restrict__ outT, int tid, bool accumulate = false) {
  constexpr int LD = Tile<TR>::LD;
  const int tx = tid & 15, r0 = (tid >> 4) * 4;
  float acc[4][NJ];
  int wof[NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const int n = min(tx + 16 * j, N - 1);
    wof[j] = n * sn;
    acc[0][j] = acc[1][j] = acc[2][j] = acc[3][j] = 0.f;
  }
  const float* ap = inT + r0;
#pragma unroll 4
  for (int k = 0; k < K; ++k) {
    const float4 a = *reinterpret_cast<const float4*>(ap + k * LD);
    const float* wk = W + k * sk;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const float w = wk[wof[j]];
      acc[0][j] = fmaf(a.x, w, acc[0][j]);
      acc[1][j] = fmaf(a.y, w, acc[1][j]);
      acc[2][j] = fmaf(a.z, w, acc[2][j]);
      acc[3][j] = fmaf(a.w, w, acc[3][j]);
    }
  }
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const int n = tx + 16 * j;
    if (n < N) {
      const float b = bias ? bias[n] : 0.f;
      if (accumulate) {
        const float4 e = *reinterpret_cast<const float4*>(outT + n * LD + r0);
        acc[0][j] += e.x; acc[1][j] += e.y; acc[2][j] += e.z; acc[3][j] += e.w;
      }
      float4 o;
      o.x = act_fwd(acc[0][j] + b, act);
      o.y = act_fwd(acc[1][j] + b, act);
      o.z = act_fwd(acc[2][j] + b, act);
      o.w = act_fwd(acc[3][j] + b, act);
      *reinterpret_cast<float4*>(outT + n * LD + r0) = o;
    }
  }
}

// Two independent products of the same shape in ONE k loop (twice the independent FMA chains per thread: the rollout CTAs run one
// warp per scheduler, so instruction-level parallelism is the only latency hiding there):
//   sum == true :  out1T[n][r] = ((sum_k in2T[k][r] W2[n][k]) + ((sum_k in1T[k][r] W1[n][k]) + b1[n])) + b2[n]
//                  -- bit-identical to tile_mm(in1, W1, b1 -> out1) followed by tile_mm(in2, W2, b2 -> out1, accumulate = true)
//   sum == false:  out1T = in1 W1^T + b1,  out2T = in2 W2^T + b2
// Forward orientation only (W row-major [N][K] with leading dimension ld), N == 16 * NJ.
template <int TR, int NJ>
__device__ __forceinline__ void tile_mm2(const float* __restrict__ in1T, const float* __restrict__ W1, const float* __restrict__ b1,
                                         const float* __restrict__ in2T, const float* __restrict__ W2, const float* __restrict__ b2,
                                         int K, int ld, float* __restrict__ out1T, float* __restrict__ out2T, bool sum, int tid) {
  constexpr int LD = Tile<TR>::LD;
  const int tx = tid & 15, r0 = (tid >> 4) * 4;
  float acc1[4][NJ], acc2[4][NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    acc1[0][j] = acc1[1][j] = acc1[2][j] = acc1[3][j] = 0.f;
    acc2[0][j] = acc2[1][j] = acc2[2][j] = acc2[3][j] = 0.f;
  }
  const float* ap1 = in1T + r0;
  const float* ap2 = in2T + r0;
  const float* w1 = W1 + tx * ld;
  const float* w2 = W2 + tx * ld;
#pragma unroll 4
  for (int k = 0; k < K; ++k) {
    const float4 a1 = *reinterpret_cast<const float4*>(ap1 + k * LD);
    const float4 a2 = *reinterpret_cast<const float4*>(ap2 + k * LD);
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const float u = w1[16 * j * ld + k], v = w2[16 * j * ld + k];
      acc1[0][j] = fmaf(a1.x, u, acc1[0][j]);
      acc1[1][j] = fmaf(a1.y, u, acc1[1][j]);
      acc1[2][j] = fmaf(a1.z, u, acc1[2][j]);
      acc1[3][j] = fmaf(a1.w, u, acc1[3][j]);
      acc2[0][j] = fmaf(a2.x, v, acc2[0][j]);
      acc2[1][j] = fmaf(a2.y, v, acc2[1][j]);
      acc2[2][j] = fmaf(a2.z, v, acc2[2][j]);
      acc2[3][j] = fmaf(a2.w, v, acc2[3][j]);
    }
  }
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const int n = tx + 16 * j;
    const float c1 = b1[n], c2 = b2[n];
    float4 o1, o2;
    o1.x = acc1[0][j] + c1; o1.y = acc1[1][j] + c1; o1.z = acc1[2][j] + c1; o1.w = acc1[3][j] + c1;
    if (sum) {
      o1.x = (acc2[0][j] + o1.x) + c2; o1.y = (acc2[1][j] + o1.y) + c2; o1.z = (acc2[2][j] + o1.z) + c2; o1.w = (acc2[3][j] + o1.w) + c2;
      *reinterpret_cast<float4*>(out1T + n * LD + r0) = o1;
    } else {
      o2.x = acc2[0][j] + c2; o2.y = acc2[1][j] + c2; o2.z = acc2[2][j] + c2; o2.w = acc2[3][j] + c2;
      *reinterpret_cast<float4*>(out1T + n * LD + r0) = o1;
      *reinterpret_cast<float4*>(out2T + n * LD + r0) = o2;
    }
  }
}

// Fused layer: Y = LayerNorm(act(X W^T + b)) * gamma + beta for N == 16*NJ output features, the LayerNorm statistics
// taken with warp shuffles across the 16 threads that share a row (no shared-memory pass, no extra barriers).
// Optionally also leaves act(.) in AT and (mean, rstd) per row for a later backward pass.
template <int TR, int NJ>
__device__ __forceinline__ void tile_mm_ln(const float* __restrict__ inT, int K, const float* __restrict__ W, int ldw,
                                           const float* __restrict__ bias, int act, const float* __restrict__ gamma,
                                           const float* __restrict__ beta, float* __restrict__ AT,
                                           float* __restrict__ YT, float* __restrict__ mean, float* __restrict__ rstd,
                                           int tid) {
  constexpr int LD = Tile<TR>::LD;
  constexpr float invN = 1.0f / (16.f * NJ);
  const int tx = tid & 15, r0 = (tid >> 4) * 4;
  float acc[4][NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) acc[0][j] = acc[1][j] = acc[2][j] = acc[3][j] = 0.f;
  const float* ap = inT + r0;
  const float* wp = W + tx * ldw;
#pragma unroll 4
  for (int k = 0; k < K; ++k) {
    const float4 a = *reinterpret_cast<const float4*>(ap + k * LD);
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const float w = wp[16 * j * ldw + k];
      acc[0][j] = fmaf(a.x, w, acc[0][j]);
      acc[1][j] = fmaf(a.y, w, acc[1][j]);
      acc[2][j] = fmaf(a.z, w, acc[2][j]);
      acc[3][j] = fmaf(a.w, w, acc[3][j]);
    }
  }
  float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const float b = bias[tx + 16 * j];
#pragma unroll
    for (int i = 0; i < 4; ++i) { acc[i][j] = act_fwd(acc[i][j] + b, act); s[i] += acc[i][j]; }
  }
#pragma unroll
  for (int o = 8; o > 0; o >>= 1)
#pragma unroll
    for (int i = 0; i < 4; ++i) s[i] += __shfl_xor_sync(0xffffffffu, s[i], o);
  float m[4], v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 4; ++i) m[i] = s[i] * invN;
#pragma unroll
  for (int j = 0; j < NJ; ++j)
#pragma unroll
    for (int i = 0; i < 4; ++i) { const float d = acc[i][j] - m[i]; v[i] = fmaf(d, d, v[i]); }
#pragma unroll
  for (int o = 8; o > 0; o >>= 1)
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], o);
  float rs[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) rs[i] = 1.0f / sqrtf(v[i] * invN + kLnEps);
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const int n = tx + 16 * j;
    const float g = gamma[n], be = beta[n];
    if (AT) *reinterpret_cast<float4*>(AT + n * LD + r0) = make_float4(acc[0][j], acc[1][j], acc[2][j], acc[3][j]);
    float4 y;
    y.x = fmaf((acc[0][j] - m[0]) * rs[0], g, be);
    y.y = fmaf((acc[1][j] - m[1]) * rs[1], g, be);
    y.z = fmaf((acc[2][j] - m[2]) * rs[2], g, be);
    y.w = fmaf((acc[3][j] - m[3]) * rs[3], g, be);
    *reinterpret_cast<float4*>(YT + n * LD + r0) = y;
  }
  if (tx == 0 && mean) {
#pragma unroll
    for (int i = 0; i < 4; ++i) { mean[r0 + i] = m[i]; rstd[r0 + i] = rs[i]; }
  }
}

// Weight gradient: g[o*ldg + k] += sum_r dYT[o][r] * XT[k][r],  o < No (No <= NTY*NI), k < Nk (Nk <= 16*NJ).
// g is the CTA-private slot in global memory (plain read-modify-write, same thread every tile).
template <int TR, int NI, int NJ>
__device__ __forceinline__ void tile_dw(const float* __restrict__ dYT, int No, const float* __restrict__ XT, int Nk,
                                        float* __restrict__ g, int ldg, int tid) {
  constexpr int LD = Tile<TR>::LD;
  constexpr int NTY = Tile<TR>::NTY;
  const int tx = tid & 15, ty = tid >> 4;
  float acc[NI][NJ];
  int ao[NI], bo[NJ];
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    ao[i] = min(ty + NTY * i, No - 1) * LD;
#pragma unroll
    for (int j = 0; j < NJ; ++j) acc[i][j] = 0.f;
  }
#pragma unroll
  for (int j = 0; j < NJ; ++j) bo[j] = min(tx + 16 * j, Nk - 1) * LD;
#pragma unroll 2
  for (int r = 0; r < TR; r += 4) {
    float4 a[NI], b[NJ];
#pragma unroll
    for (int i = 0; i < NI; ++i) a[i] = *reinterpret_cast<const float4*>(dYT + ao[i] + r);
#pragma unroll
    for (int j = 0; j < NJ; ++j) b[j] = *reinterpret_cast<const float4*>(XT + bo[j] + r);
#pragma unroll
    for (int i = 0; i < NI; ++i)
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        acc[i][j] = fmaf(a[i].x, b[j].x, acc[i][j]);
        acc[i][j] = fmaf(a[i].y, b[j].y, acc[i][j]);
        acc[i][j] = fmaf(a[i].z, b[j].z, acc[i][j]);
        acc[i][j] = fmaf(a[i].w, b[j].w, acc[i][j]);
      }
  }
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const int o = ty + NTY * i;
    if (o < No) {
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        const int k = tx + 16 * j;
        if (k < Nk) g[o * ldg + k] += acc[i][j];
      }
    }
  }
}

// g1[n] += sum_r AT[n][r]              (bias / LN-beta gradients), n < N, one thread per n (strided)
template <int TR>
__device__ __forceinline__ void tile_colsum(const float* __restrict__ AT, int N, float* __restrict__ g1, int tid) {
  constexpr int LD = Tile<TR>::LD;
  for (int n = tid; n < N; n += Tile<TR>::NT) {
    float s = 0.f;
#pragma unroll 4
    for (int r = 0; r < TR; r += 4) {
      const float4 a = *reinterpret_cast<const float4*>(AT + n * LD + r);
      s += (a.x + a.y) + (a.z + a.w);
    }
    g1[n] += s;
  }
}

// LayerNorm parameter gradients: gw[n] += sum_r dYT[n][r] * xhat[n][r], gb[n] += sum_r dYT[n][r]
// with xhat = (AT - mean[r]) * rstd[r].
template <int TR>
__device__ __forceinline__ void tile_ln_param_grads(const float* __restrict__ dYT, const float* __restrict__ AT,
                                                    const float* __restrict__ mean, const float* __restrict__ rstd,
                                                    int N, float* __restrict__ gw, float* __restrict__ gb, int tid) {
  constexpr int LD = Tile<TR>::LD;
  for (int n = tid; n < N; n += Tile<TR>::NT) {
    float sw = 0.f, sb = 0.f;
#pragma unroll 4
    for (int r = 0; r < TR; ++r) {
      const float d = dYT[n * LD + r];
      sw = fmaf(d, (AT[n * LD + r] - mean[r]) * rstd[r], sw);
      sb += d;
    }
    gw[n] += sw;
    gb[n] += sb;
  }
}

// Row-wise LayerNorm over N features of AT -> YT (may alias AT is NOT allowed), statistics kept.
// red: scratch of 4*TR floats.  Ends with a __syncthreads().
template <int TR>
__device__ __forceinline__ void tile_layernorm(const float* __restrict__ AT, int N, const float* __restrict__ gamma,
                                               const float* __restrict__ beta, float* __restrict__ YT,
                                               float* __restrict__ mean, float* __restrict__ rstd,
                                               float* __restrict__ red, int tid) {
  constexpr int LD = Tile<TR>::LD;
  const int r = tid % TR, q = tid / TR;
  float s = 0.f;
  for (int n = q; n < N; n += 4) s += AT[n * LD + r];
  red[q * TR + r] = s;
  __syncthreads();
  const float m = ((red[r] + red[TR + r]) + (red[2 * TR + r] + red[3 * TR + r])) / (float)N;
  __syncthreads();
  float v = 0.f;
  for (int n = q; n < N; n += 4) {
    const float d = AT[n * LD + r] - m;
    v = fmaf(d, d, v);
  }
  red[q * TR + r] = v;
  __syncthreads();
  const float var = ((red[r] + red[TR + r]) + (red[2 * TR + r] + red[3 * TR + r])) / (float)N;
  const float rs = 1.0f / sqrtf(var + kLnEps);
  for (int n = q; n < N; n += 4) {
    const float xh = (AT[n * LD + r] - m) * rs;
    YT[n * LD + r] = gamma ? fmaf(xh, gamma[n], beta[n]) : xh;
  }
  if (q == 0) {
    mean[r] = m;
    rstd[r] = rs;
  }
  __syncthreads();
}

// Backward of  Y = LN(A) * gamma + beta  followed by the activation that produced A (A = act(Z)):
// dT holds dL/dY on entry and dL/dZ on exit (in place).  act == ACT_NONE stops at dL/dA.
// Ends with a __syncthreads().
template <int TR>
__device__ __forceinline__ void tile_layernorm_bwd(float* __restrict__ dT, const float* __restrict__ AT,
                                                   const float* __restrict__ mean, const float* __restrict__ rstd,
                                                   const float* __restrict__ gamma, int N, int act,
                                                   float* __restrict__ red, int tid) {
  constexpr int LD = Tile<TR>::LD;
  const int r = tid % TR, q = tid / TR;
  const float m = mean[r], rs = rstd[r];
  float s1 = 0.f, s2 = 0.f;
  for (int n = q; n < N; n += 4) {
    const float dx = dT[n * LD + r] * gamma[n];
    s1 += dx;
    s2 = fmaf(dx, (AT[n * LD + r] - m) * rs, s2);
  }
  __syncthreads();                       // red may still be in use by a previous reader
  red[q * TR + r] = s1;
  red[4 * TR + q * TR + r] = s2;
  __syncthreads();
  const float invN = 1.0f / (float)N;
  const float a1 = ((red[r] + red[TR + r]) + (red[2 * TR + r] + red[3 * TR + r])) * invN;
  const float a2 = ((red[4 * TR + r] + red[5 * TR + r]) + (red[6 * TR + r] + red[7 * TR + r])) * invN;
  for (int n = q; n < N; n += 4) {
    const float a = AT[n * LD + r];
    const float xh = (a - m) * rs;
    const float dx = dT[n * LD + r] * gamma[n];
    const float dA = rs * (dx - a1 - xh * a2);
    dT[n * LD + r] = dA * act_bwd(a, act);
  }
  __syncthreads();
}

// block reduction of NV doubles per thread into out[] with one atomicAdd per value per CTA
template <int NV>
__device__ __forceinline__ void block_accumulate(double (&v)[NV], double* __restrict__ out, double* sred /*[NV*32]*/,
                                                 int tid, int nt) {
  const int lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    double x = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) sred[i * 32 + warp] = x;
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      double x = lane < nw ? sred[i * 32 + lane] : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
      if (lane == 0) atomicAdd(out + i, x);
    }
  }
  __syncthreads();
}

// ValueNorm.running_mean_var (utils/valuenorm.py:32-36)
__device__ __forceinline__ void vn_mean_var(const float* __restrict__ vn, float& mean, float& var) {
  const float d = fmaxf(vn[2], 1e-5f);
  mean = vn[0] / d;
  const float msq = vn[1] / d;
  var = fmaxf(msq - mean * mean, 1e-2f);
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-(function, DEVICE) setting: remember what was configured per device
// ordinal, so that a process driving several GPUs configures each of them (one static instance per call site)
struct SmemConfig {
  size_t bytes[64];
  size_t& slot() {
    int d = 0;
    cudaGetDevice(&d);
    return bytes[d & 63];
  }
};

// ---- thread-block clusters: barrier and distributed shared memory (DSMEM) -----------------------------------------------------
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_cta_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// store into the shared memory of CTA `rank` of this cluster, at the address `local` has in this CTA's own window
__device__ __forceinline__ void st_cluster_f32(const float* local, uint32_t rank, float v) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"((uint32_t)__cvta_generic_to_shared(local)), "r"(rank));
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(remote), "f"(v) : "memory");
}
// the two halves of a cluster barrier, for threads that have work to do between signalling and waiting (not .aligned: callable
// where a warp may have diverged); arrive releases and wait acquires this thread's shared / DSMEM writes at cluster scope
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait;" ::: "memory"); }

// ---- programmatic dependent launch (PDL) for the chains of small dependent kernels of an optimiser step -------------------------
// A kernel launched with launch_pdl() may be SCHEDULED while its stream predecessor still runs: its CTAs take their SMs and park in
// pdl_prologue() (griddepcontrol.wait) until the predecessor grid has completed and flushed, so the ~2 us of launch / scheduling
// latency between two dependent kernels of a CUDA graph disappears.  Every kernel of such a chain calls pdl_prologue() first (it
// also lets ITS successor start scheduling: griddepcontrol.launch_dependents); without the launch attribute both are no-ops.
bool pdl_enabled();     // api.cu: env MAPPO_B200_PDL
__device__ __forceinline__ void pdl_prologue() {
  asm volatile("griddepcontrol.launch_dependents;");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg;
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = &attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// error plumbing (api.cu)
void set_error(const char* fmt, ...);
int check_launch(const char* what);

NetDev make_net_dev(const mappo_net_desc_t* d);

}  // namespace mappo
