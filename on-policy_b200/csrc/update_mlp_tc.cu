// update_mlp_tc.cu -- the fused MLP training step on Blackwell tensor cores (tcgen05.mma kind::tf32, fp32
// accumulators in TMEM, weights delivered by one TMA bulk copy).  Same contract as update_mlp_kernel (update_mlp.cu):
// index-driven gather -> forward -> losses -> backward -> per-CTA gradient slot, one launch per net per step.
//
// Tile = 128 rows = UMMA M = the 128 TMEM lanes, TWO threads per row: warps w and w + 4 address the same 32 TMEM lanes,
// warpgroup g owns hidden columns [32 g, 32 g + 32).  After each MMA a thread pulls ITS half row of the accumulator out
// of TMEM (tcgen05.ld 32x32b) and does activation / LayerNorm in registers; the two halves of a row meet on a 64-thread
// named barrier and swap their partial sums through shared memory (PairXch).  One thread per row was a 16 K-instruction
// dependent chain on one warp per scheduler; two halve it.
//
// Operand layout: every operand is K-major, no swizzle ("interleaved" canonical layout): an R x K operand is stored
// as [K/4][R(+pad)][4] floats, i.e. the 16-byte unit of 4 consecutive K-elements of row r sits at
// ((k/4)*S + r)*16 with S >= R; descriptor SBO = 128 B (next 8 rows), LBO = S*16 B (next 4 K-elements).
// (MN-major tf32 operands in this layout produce no output on sm_100a -- tests/cuda/tc_probe.cu -- so the
// weight-gradient GEMMs dW = dY^T X, whose contraction runs over the ROWS, read explicitly transposed tiles:
// thread r scatters its row as column r of a [rows/4][features + 1][4] tile; the odd feature stride S = F + 1
// makes those 4-byte stores bank-conflict free.)  The dX GEMMs read a transposed weight image built once per step.
//
// LayerNorm affine parameters and biases are folded into the GEMMs: the tiles hold xhat (pre-affine) plus a
// constant-1 feature, the weight image holds W' = W diag(gamma) and b' = b + W beta in the column of the 1-feature.
// dW' accumulates in TMEM across the tiles of a CTA; at the end dW = dW' diag(gamma) + db' beta^T, db = dW'[:, one],
// dgamma = colsum(dW' .* W), dbeta = W^T db'  (chain rule of the folding), written to the CTA's gradient slot.
#include "tc64.cuh"
#include "p2p.cuh"

namespace mappo {




// dW = dW' diag(gamma_in) + db' beta_in^T, db = dW'[:, one], dgamma_in = colsum(dW' .* W), dbeta_in = W^T db'   (chain rule of the
// folding) from the slot-summed raw accumulators.  Grid: blockIdx.y = layer (0 fc2, 1 fc1, 2 heads), blockIdx.x = block
// of 16 input features; 256 threads = 16 features x 16 groups of 4 output rows.  Every CTA also emits its sum(g^2).
// The body works on one (bx, by) unit with 256 threads `tid`; part_g / part_b / sred are that unit's shared scratch.  `active`
// == false: the unit only takes part in the barriers (tc_tail_kernel runs four units per CTA, not all of them populated).
struct UnfoldScratch { float part_g[16][17], part_b[16][17], sred[8]; };
__device__ __forceinline__ void tc_unfold_unit(const NetDev& n, const float* p, const float* raw, float* g, float* sumsq_part,
                                               int bx, int by, int grid_x, int tid, bool active, UnfoldScratch& S,
                                               float* g_mirror = nullptr) {
  const TcImage m = make_tc_image(n);
  const TcRaw R = make_tc_raw(m);
  const int kx = tid & 15, og = tid >> 4;
  const int sec = by, k = bx * 16 + kx;                 // for the heads (sec == 2) k < 64 always (grid_x == 4)
  const int in = n.in_dim, Atot = n.head_total;
  float sq = 0.f;
  auto put = [&](int off, float v) { g[off] = v; if (g_mirror) g_mirror[off] = v; sq = fmaf(v, v, sq); };
  const int K = sec == 0 ? 64 : (sec == 1 ? in : 64);
  const bool fold = sec == 1 ? (n.use_fn != 0) : true;
  // the LayerNorm in front of the heads: base.mlp.fc2[0]'s for feed-forward nets, rnn.norm for recurrent ones
  const int gam_off = sec == 0 ? n.g.ln1_w : (sec == 1 ? n.g.fn_w : (n.recurrent ? n.g.rnn_ln_w : n.g.ln2_w[0]));
  const int bet_off = sec == 0 ? n.g.ln1_b : (sec == 1 ? n.g.fn_b : (n.recurrent ? n.g.rnn_ln_b : n.g.ln2_b[0]));
  float sg = 0.f, sb = 0.f;
  if (active && sec < 2) {
    const int ld = sec == 0 ? kHF : m.inF, one = sec == 0 ? kOne : in;
    const float* G = raw + (sec == 0 ? R.g2 : R.g1);
    const int w_off = sec == 0 ? n.g.fc2_w[0] : n.g.fc1_w, b_off = sec == 0 ? n.g.fc2_b[0] : n.g.fc1_b;
    if (k < K) {
      const float gam = fold ? p[gam_off + k] : 1.f, bet = fold ? p[bet_off + k] : 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int o = og * 4 + j;
        const float dw = G[o * ld + k], w = p[w_off + o * K + k], dbo = G[o * ld + one];
        put(w_off + o * K + k, fmaf(dbo, bet, dw * gam));     // b' = b + W beta depends on W as well
        sg = fmaf(dw, w, sg);
        sb = fmaf(dbo, w, sb);
      }
    }
    if (bx == 0 && tid < 64) put(b_off + tid, G[tid * ld + one]);
  } else if (active) {                                  // heads: raw gh[feature][a]; this unit owns 16 features
    if (k < 64) {
      const float gam = p[gam_off + k], bet = p[bet_off + k];
      for (int a = og; a < Atot; a += 16) {
        const float dw = raw[R.gh + k * m.NH + a], w = p[n.g.head_w + a * 64 + k], dba = raw[R.dbh + a];
        put(n.g.head_w + a * 64 + k, fmaf(dba, bet, dw * gam));
        sg = fmaf(dw, w, sg);
        sb = fmaf(dba, w, sb);
      }
    }
    if (bx == 0 && tid < Atot) put(n.g.head_b + tid, raw[R.dbh + tid]);
  }
  S.part_g[og][kx] = sg; S.part_b[og][kx] = sb;
  __syncthreads();
  if (active && fold && og == 0 && k < K) {
    float a = 0.f, c = 0.f;
#pragma unroll
    for (int q = 0; q < 16; ++q) { a += S.part_g[q][kx]; c += S.part_b[q][kx]; }
    put(gam_off + k, a);
    put(bet_off + k, c);
  }
  // sum of squares of everything this unit wrote
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  if ((tid & 31) == 0) S.sred[tid >> 5] = sq;
  __syncthreads();
  if (tid == 0 && active) {
    float t = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) t += S.sred[q];
    sumsq_part[by * grid_x + bx] = t;
  }
}

__global__ void __launch_bounds__(256)
tc_unfold_kernel(const NetDev n, const float* __restrict__ p, const float* __restrict__ raw, float* __restrict__ g,
                 float* __restrict__ sumsq_part) {
  __shared__ UnfoldScratch S;
  pdl_prologue();
  tc_unfold_unit(n, p, raw, g, sumsq_part, blockIdx.x, blockIdx.y, gridDim.x, threadIdx.x, true, S);
}

// element i of the folded tf32 weight image
__device__ __forceinline__ float pack_tc_element(const NetDev& n, const TcImage& m, const float* p, int i) {
  const int H = 64;
  {
    float v = 0.f;
    if (i < m.w2) {                                       // fc1: [inF/4][64][4]
      const int kc = i / 256, o = (i >> 2) & 63, k = kc * 4 + (i & 3);
      const float* W = p + n.g.fc1_w + o * n.in_dim;
      if (k < n.in_dim) v = W[k] * (n.use_fn ? p[n.g.fn_w + k] : 1.f);
      else if (k == n.in_dim) {
        v = p[n.g.fc1_b + o];
        if (n.use_fn) for (int j0 = 0; j0 < n.in_dim; ++j0) { const int j = (j0 + o) % n.in_dim; v = fmaf(W[j], p[n.g.fn_b + j], v); }
      }
    } else if (i < m.wh) {                                // fc2: [18][64][4], input LN = ln1
      const int t = i - m.w2, kc = t / 256, o = (t >> 2) & 63, k = kc * 4 + (t & 3);
      const float* W = p + n.g.fc2_w[0] + o * H;
      if (k < H) v = W[k] * p[n.g.ln1_w + k];
      else if (k == kOne) {
        v = p[n.g.fc2_b[0] + o];
        for (int j0 = 0; j0 < H; ++j0) { const int j = (j0 + o) & 63; v = fmaf(W[j], p[n.g.ln1_b + j], v); }
      }
    } else if (i < m.w2t) {                               // heads: [18][NH][4], input LN = ln2[0]
      const int t = i - m.wh, kc = t / (4 * m.NH), a = (t >> 2) % m.NH, k = kc * 4 + (t & 3);
      if (a < n.head_total) {
        const float* W = p + n.g.head_w + a * H;
        const int gw = n.recurrent ? n.g.rnn_ln_w : n.g.ln2_w[0], gb = n.recurrent ? n.g.rnn_ln_b : n.g.ln2_b[0];
        if (k < H) v = W[k] * p[gw + k];
        else if (k == kOne) {
          v = p[n.g.head_b + a];
          for (int j0 = 0; j0 < H; ++j0) { const int j = (j0 + a) & 63; v = fmaf(W[j], p[gb + j], v); }
        }
      }
    } else if (i < m.wht) {                               // fc2 transposed: element (row k, K-index o) = W2'[o][k]
      const int t = i - m.w2t, oc = t / 256, k = (t >> 2) & 63, o = oc * 4 + (t & 3);
      v = p[n.g.fc2_w[0] + o * H + k] * p[n.g.ln1_w + k];
    } else {                                              // heads transposed: (row k, K-index a) = Wh'[a][k]
      const int t = i - m.wht, ac = t / 256, k = (t >> 2) & 63, a = ac * 4 + (t & 3);
      if (a < n.head_total) v = p[n.g.head_w + a * H + k] * p[(n.recurrent ? n.g.rnn_ln_w : n.g.ln2_w[0]) + k];
    }
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v));
    return __uint_as_float(u);
  }
}
__global__ void __launch_bounds__(256) pack_tc_kernel(const NetDev n, const float* __restrict__ p, float* __restrict__ img) {
  const TcImage m = make_tc_image(n);
  pdl_prologue();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m.total; i += gridDim.x * blockDim.x) img[i] = pack_tc_element(n, m, p, i);
}

// ------------------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------------------
struct TcSmem { int img, p, x1t, x2t, ta, lg, dbh, xch, misc, total; };   // float offsets
__host__ __device__ inline TcSmem make_tc_smem(const TcImage& m) {
  TcSmem s;
  int o = 0;
  s.img = o; o += m.total;
  s.p = o; o += 32 * kS73 * 4;             // staging: K-major [<=18][128][4] tiles, or xhat0^T [32][inF+1][4]
  s.x1t = o; o += 32 * kS73 * 4;           // xhat1^T (+ constant-1 row 64, zero rows 65..71)
  s.x2t = o; o += 32 * kS65 * 4;           // xhat2^T
  s.ta = o; o += 32 * kS65 * 4;            // dL^T / dZ2^T / dZ1^T
  s.lg = o; o += m.NH * (kTM + 4);         // logits scratch for row_loss, transposed [j][132]
  s.dbh = o; o += 32;
  s.xch = o; o += 2 * 2 * 2 * kTM;         // row-pair exchange: [slot 2][warpgroup 2][128] float2
  s.misc = o; o += 16;                     // mbarriers (2 x 8 B) + tmem base
  s.total = o;
  return s;
}

// phase timestamps of CTA 0 / thread 0 (clock64), read back by mappo_debug_tc_timing(): where does a tile's
// latency go?  [0] start, [1] setup done, [2] S1 staged, [3] fc1 ready, [4] S3 done, [5] fc2 ready, [6] S5 done,
// [7] head ready, [8] S7 done, [9] dx2 ready, [10] S9 done, [11] dx1 ready, [12] S11 done, [13] G2 dumped (thread 0
// is in warpgroup 0, which dumps while the last G1 MMA runs), [14] G1 done, [15] end
__device__ long long g_tc_timing[16];
#define TC_STAMP(i) do { if (blockIdx.x == 0 && tid == 0) g_tc_timing[i] = clock64(); } while (0)


// LayerNorm + activation backward for one row: d = dL/dxhat (this thread's 32 columns) -> dZ in place.  xhat is re-read
// from the transposed tile (conflict-free 4-byte loads).  `pos`: bit f = the activation output of column f was > 0 in the forward
// pass -- the ReLU derivative must not be taken from the value reconstructed out of the tf32-rounded xhat (an inactive unit's
// exact 0 comes back as +-1e-4 |mu|, i.e. a coin flip).
__device__ __forceinline__ void ln_act_bwd32(float* d, const float* XT, int S, int r, int wg, PairXch& px, float mu, float rs,
                                             int act, uint32_t pos) {
  const float* base = XT + ((r >> 2) * S + wg * 32) * 4 + (r & 3);
  float xh[32];
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int f = 0; f < 32; ++f) { xh[f] = base[f * 4]; s1 += d[f]; s2 = fmaf(d[f], xh[f], s2); }
  const float2 t = px.sum(s1, s2);
  s1 = t.x * (1.f / 64.f); s2 = t.y * (1.f / 64.f);
  const float inv = 1.0f / rs;
#pragma unroll
  for (int f = 0; f < 32; ++f) {
    const float dA = rs * (d[f] - s1 - xh[f] * s2);
    const float da = act == ACT_RELU ? (((pos >> f) & 1u) ? 1.f : 0.f) : act_bwd(fmaf(xh[f], inv, mu), act);
    d[f] = to_tf32(dA * da);
  }
}

// MODE (recurrent nets run the base MLP and the heads on either side of the GRU sequence kernels of update_gru_tc.cu; planes are
// [position][64] fp32 workspaces indexed by the minibatch position p):
//   TC_FULL      the whole MLP net (feed-forward policies)
//   TC_BASE_FWD  S1..S5 only: xhat2 (pre-affine output of the last LayerNorm, tf32) -> plane_out                       no gradients
//   TC_BASE_BWD  S1..S5 recomputed, dL/dxhat2 read from plane_in instead of the head path, S9..S11 -> G2 / G1
//   TC_HEAD      row = plane_in[p] (GRU state h): LayerNorm -> heads -> loss -> dL/dh -> plane_out; Gh / dbh
enum { TC_FULL = 0, TC_BASE_FWD = 1, TC_BASE_BWD = 2, TC_HEAD = 3 };
template <int MODE>
__global__ void __launch_bounds__(kTCThreads, 1)
update_mlp_tc_kernel(const NetDev n, const float* __restrict__ params, const float* __restrict__ image, const BatchDev b,
                     const LossDev L, const double* __restrict__ norm_stats, const double* __restrict__ adv_stats,
                     const float* __restrict__ vn_state, float* __restrict__ grad_part, double* __restrict__ loss_out,
                     int n_tiles, uint32_t tmem_cols, const float* __restrict__ plane_in, float* __restrict__ plane_out) {
  extern __shared__ __align__(1024) float smem[];
  __shared__ double sred[2 * 32];
  pdl_prologue();                                            // (PDL: scheduled under the weight-pack kernel, released when it has finished)
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int r = tid & (kTM - 1), wg = tid >> 7;              // my row of the tile, my half of the hidden columns
  const TcImage im = make_tc_image(n);
  const TcSmem sm = make_tc_smem(im);
  float* sImg = smem + sm.img;
  float* P = smem + sm.p;
  float* X1T = smem + sm.x1t;
  float* X2T = smem + sm.x2t;
  float* TA = smem + sm.ta;
  float* lgT = smem + sm.lg;
  float* dbh = smem + sm.dbh;
  uint64_t* bar_w = reinterpret_cast<uint64_t*>(smem + sm.misc);
  uint64_t* bar_m = bar_w + 1;               // forward / dX accumulator ready
  uint64_t* bar_g = bar_w + 2;               // weight-gradient MMAs of the phase done (their operand tiles are free)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_w + 3);
  PairXch px{reinterpret_cast<float2*>(smem + sm.xch), wg, r, 1 + (warp & 3), 0};
  const int in = n.in_dim, inF = im.inF, NH = im.NH, Atot = n.head_total;
  const int S0 = inF + 1, SH = NH + 1;
  const int act = n.use_relu ? ACT_RELU : ACT_TANH;
  constexpr int LGLD = kTM + 4;

  TC_STAMP(0);
  // row index of my first tile: issued before the setup so that its latency hides behind barrier init / TMEM allocation
  auto row_of = [&](int tile) {
    const int q = tile * kTM + r;
    return (tile < n_tiles && q < b.n_rows) ? (b.rows ? b.rows[q] : q) : -1;
  };
  int gr_next = row_of(blockIdx.x);
  // ---- one-time setup: barriers, TMEM, weight image by TMA, constant rows of the transposed tiles ----
  if (tid == 0) {
    mbar_init(bar_w, 1);
    mbar_init(bar_m, 1);
    mbar_init(bar_g, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(tmem_slot, tmem_cols);
  for (int i = tid; i < 32; i += kTCThreads) dbh[i] = 0.f;
  if (wg == 0) {
    float* base = X1T + (r >> 2) * kS73 * 4 + (r & 3);              // constant-1 feature (row 64) and zero rows 65..71
#pragma unroll
    for (int f = 64; f < 72; ++f) base[f * 4] = (f == kOne) ? 1.f : 0.f;
  }
  if (wg == 0) reinterpret_cast<int*>(lgT)[r] = gr_next;          // row ids of the first tile (S1's rowid_s)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  if (tid == 0) {                          // the weight image arrives behind the first gather
    mbar_expect_tx(bar_w, (uint32_t)(im.total * sizeof(float)));
    tma_bulk_g2s(sImg, image, (uint32_t)(im.total * sizeof(float)), bar_w);
  }
  // TMEM columns: D fwd/bwd accumulator, Dh logits, G2 / G1 / Gh persistent weight-gradient accumulators
  const uint32_t cD = 0, cDh = 64, cG2 = 96, cG1 = 168, cGh = 240, cX0 = 272;     // cX0: parked xhat0aug (72 cols)
  const uint32_t lane_base = ((uint32_t)((warp & 3) * 32)) << 16;
  const uint32_t cMy = cD + 32 * wg;                   // my 32 columns of the 64-wide accumulator

  const LossConsts lc = make_loss_consts(n, L, norm_stats, adv_stats, vn_state);
  double acc[3] = {0.0, 0.0, 0.0};
  uint32_t phase = 0, phase_g = 0;
  bool first_tile = true, g1_pending = false, ids_published = true;
  const uint32_t aP = smem_u32(P), aX1T = smem_u32(X1T), aX2T = smem_u32(X2T), aTA = smem_u32(TA);
  const uint32_t aW1 = smem_u32(sImg + im.w1), aW2 = smem_u32(sImg + im.w2), aWh = smem_u32(sImg + im.wh);
  const uint32_t aW2T = smem_u32(sImg + im.w2t), aWhT = smem_u32(sImg + im.wht);
  constexpr uint32_t ROWB = kTM * 16;                  // chunk stride of a 128-row K-major staging tile

  // TC_HEAD / TC_BASE_BWD: this thread's 32 plane values of a tile travel in registers, fetched one tile (heads) or half a tile (base
  // backward) before their use, so the global-memory latency does not sit between two tiles
  float pref[32];
  auto fetch_plane_row = [&](int tile, bool ok) {
    const size_t pp = (size_t)tile * kTM + r;
    if (ok) { ld_pl16_pinned(plane_in, pp, wg * 8, pref); ld_pl16_pinned(plane_in, pp, wg * 8 + 4, pref + 16); }
    else {
#pragma unroll
      for (int i = 0; i < 32; ++i) pref[i] = 0.f;
    }
  };
  if (MODE == TC_HEAD) fetch_plane_row(blockIdx.x, gr_next >= 0);
  TC_STAMP(1);
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int p = tile * kTM + r;
    const int gr = gr_next;
    gr_next = row_of(tile + gridDim.x);
    if (MODE == TC_BASE_BWD) fetch_plane_row(tile, p < b.n_rows && gr >= 0);      // dL/dxhat2 of this tile, used in S9
    float mu0 = 0.f, rs0 = 1.f;
    const RowIn rin = load_row_in(n, b, (wg == 0 && (MODE == TC_FULL || MODE == TC_HEAD)) ? gr : -1);      // loss inputs (warpgroup 0 owns the loss): in flight
                                                                 // during the whole forward pass

    float mu1 = 0.f, rs1 = 1.f, mu2 = 0.f, rs2 = 1.f;
    uint32_t pos1 = 0u, pos2 = 0u;                              // activation output > 0, per column of this thread (ReLU backward)
    if (MODE != TC_HEAD) {
    // ---- S1: coalesced cooperative gather (a warp reads whole rows) -> shared staging -> my row in registers,
    //      feature LayerNorm, stage xhat0 (K-major in TA, + constant-1 feature), park it in TMEM ----
    {
      int* rowid_s = reinterpret_cast<int*>(lgT);                 // lgT is free until S7
      float* Rs = P;                                              // raw rows [128][RS], RS odd -> conflict-free row reads
      const int RS = in | 1;
      if (!ids_published) {                                       // (first pass: published before the setup barrier)
        if (wg == 0) rowid_s[r] = gr;
        __syncthreads();
      }
      ids_published = false;
      const float* base = n.is_critic ? b.share_obs : b.obs;
      // each of the 8 warps gathers 16 rows: 32 independent coalesced loads in flight per thread, then the stores
      {
        float v0[16], v1[16];
#pragma unroll
        for (int rr = 0; rr < 16; ++rr) {
          const int g0 = rowid_s[warp * 16 + rr];
          const float* rp = base + (size_t)(g0 < 0 ? 0 : g0) * in;
          v0[rr] = (lane < in && g0 >= 0) ? __ldg(rp + lane) : 0.f;
          v1[rr] = (lane + 32 < in && g0 >= 0) ? __ldg(rp + lane + 32) : 0.f;
        }
#pragma unroll
        for (int rr = 0; rr < 16; ++rr) {
          const int q = warp * 16 + rr;
          if (lane < in) Rs[q * RS + lane] = v0[rr];
          if (lane + 32 < in) Rs[q * RS + lane + 32] = v1[rr];
        }
      }
      __syncthreads();
      float x[64];
#pragma unroll
      for (int k = 0; k < 64; ++k) x[k] = k < in ? Rs[r * RS + k] : 0.f;
      if (n.use_fn && gr >= 0) {                                  // both threads of the row: same statistics
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;             // padding is zero; 4 chains instead of one
#pragma unroll
        for (int k = 0; k < 64; k += 4) { s0 += x[k]; s1 += x[k + 1]; s2 += x[k + 2]; s3 += x[k + 3]; }
        mu0 = ((s0 + s1) + (s2 + s3)) / (float)in;
        float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
#pragma unroll
        for (int k = 0; k < 64; k += 4) {
          const float d0 = x[k] - mu0, d1 = x[k + 1] - mu0, d2 = x[k + 2] - mu0, d3 = x[k + 3] - mu0;
          v0 = (k < in) ? fmaf(d0, d0, v0) : v0;
          v1 = (k + 1 < in) ? fmaf(d1, d1, v1) : v1;
          v2 = (k + 2 < in) ? fmaf(d2, d2, v2) : v2;
          v3 = (k + 3 < in) ? fmaf(d3, d3, v3) : v3;
        }
        rs0 = 1.0f / sqrtf(((v0 + v1) + (v2 + v3)) / (float)in + kLnEps);
      }
#pragma unroll
      for (int c8 = 0; c8 < 9; ++c8) {
        if (c8 * 8 < inF && (c8 & 1) == wg) {                     // 8-feature chunks alternate between the two threads
          float q[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int k = c8 * 8 + j;
            q[j] = (k == in) ? 1.f : ((k < in) ? to_tf32((x[k & 63] - mu0) * rs0) : 0.f);
          }
          reinterpret_cast<float4*>(TA)[(2 * c8) * kTM + r] = make_float4(q[0], q[1], q[2], q[3]);
          reinterpret_cast<float4*>(TA)[(2 * c8 + 1) * kTM + r] = make_float4(q[4], q[5], q[6], q[7]);
          tmem_st8(tmem + lane_base + cX0 + c8 * 8, q);        // parked for the fc1 weight gradient (S11)
        }
      }
      tmem_st_wait();
    }
    TC_STAMP(2);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      if (first_tile) mbar_wait(bar_w, 0);                      // weight image has landed
      const uint32_t id = make_idesc(128, 64, 0, 0);
      umma_seq(tmem + cD, aTA, 2 * ROWB, ROWB, aW1, 2 * 1024, 1024, id, inF / 8, false);
      umma_commit(bar_m);
    }
    // ---- S3: fc1 epilogue: activation, LayerNorm -> xhat1 (K-major staging + transposed copy) ----
    {
      float a[32];
      mbar_wait(bar_m, phase); phase ^= 1; TC_STAMP(3);
      tc_fence_after();
      tmem_ld16(tmem + lane_base + cMy, a);
      tmem_ld16(tmem + lane_base + cMy + 16, a + 16);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 32; ++i) { a[i] = act_fwd_tc(a[i], act); pos1 |= (a[i] > 0.f ? 1u : 0u) << i; }
      ln_stats_pair(a, px, mu1, rs1);
#pragma unroll
      for (int i = 0; i < 32; ++i) a[i] = to_tf32((a[i] - mu1) * rs1);
      put_kmajor32(P, r, wg, a, true);
      put_transposed32(X1T, kS73, r, wg, a);
    }
    TC_STAMP(4);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      const uint32_t id = make_idesc(128, 64, 0, 0);
      umma_seq(tmem + cD, aP, 2 * ROWB, ROWB, aW2, 2 * 1024, 1024, id, kHF / 8, false);
      umma_commit(bar_m);
    }
    // ---- S5: fc2 epilogue ----
    {
      float a[32];
      mbar_wait(bar_m, phase); phase ^= 1; TC_STAMP(5);
      tc_fence_after();
      tmem_ld16(tmem + lane_base + cMy, a);
      tmem_ld16(tmem + lane_base + cMy + 16, a + 16);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 32; ++i) { a[i] = act_fwd_tc(a[i], act); pos2 |= (a[i] > 0.f ? 1u : 0u) << i; }
      ln_stats_pair(a, px, mu2, rs2);
#pragma unroll
      for (int i = 0; i < 32; ++i) a[i] = to_tf32((a[i] - mu2) * rs2);
      if (MODE == TC_BASE_FWD) {                                  // the GRU's input rows; nothing else to do for this tile
        if (p < b.n_rows) { st_pl16(plane_out, (size_t)p, wg * 8, a); st_pl16(plane_out, (size_t)p, wg * 8 + 4, a + 16); }
        tc_fence_before();
        __syncthreads();
        continue;
      }
      if (MODE == TC_FULL) put_kmajor32(P, r, wg, a, true);
      put_transposed32(X2T, kS65, r, wg, a);
    }
    } else {
      // ---- TC_HEAD: the GRU state of this position -> LayerNorm (rnn.norm, rnn.py:79) -> xhat (K-major staging + transposed) ----
      float a[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) a[i] = pref[i];
      fetch_plane_row(tile + gridDim.x, gr_next >= 0);           // next tile's rows: in flight under this tile
      ln_stats_pair(a, px, mu2, rs2);
#pragma unroll
      for (int i = 0; i < 32; ++i) a[i] = to_tf32((a[i] - mu2) * rs2);
      put_kmajor32(P, r, wg, a, true);
      put_transposed32(X2T, kS65, r, wg, a);
    }
    if (MODE != TC_BASE_BWD) {
    TC_STAMP(6);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      if (MODE == TC_HEAD && first_tile) mbar_wait(bar_w, 0);   // weight image has landed
      const uint32_t id = make_idesc(128, NH, 0, 0);
      umma_seq(tmem + cDh, aP, 2 * ROWB, ROWB, aWh, 2 * NH * 16, NH * 16, id, kHF / 8, false);
      umma_commit(bar_m);
    }
    // ---- S7: heads, loss, d(loss)/d(logits): one thread per row (warpgroup 0) ----
    mbar_wait(bar_m, phase); phase ^= 1; TC_STAMP(7);
    tc_fence_after();
    if (wg == 0) {
      float lg[32];
      tmem_ld16(tmem + lane_base + cDh, lg);
      if (NH > 16) tmem_ld16(tmem + lane_base + cDh + 16, lg + 16);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) if (j < Atot) lgT[j * LGLD + r] = lg[j];
      row_loss_pre<LGLD>(n, b, L, lc, lgT, r, gr, p, rin, acc);    // thread-local: only column r is touched
      if (!b.eval_only) {
#pragma unroll
        for (int j = 0; j < 32; ++j) lg[j] = j < Atot ? to_tf32(lgT[j * LGLD + r]) : 0.f;
#pragma unroll
        for (int kc = 0; kc < 8; ++kc)
          if (kc * 4 < NH)
            reinterpret_cast<float4*>(P)[kc * kTM + r] = make_float4(lg[4 * kc], lg[4 * kc + 1], lg[4 * kc + 2], lg[4 * kc + 3]);
        float* tb = TA + (r >> 2) * SH * 4 + (r & 3);             // dL^T: [32][NH + 1][4]
#pragma unroll
        for (int j = 0; j < 32; ++j) if (j < NH) tb[j * 4] = lg[j];
        // head bias gradient: sum over the rows of this warp, one shared atomic per warp and output
        for (int j = 0; j < Atot; ++j) {
          float v = lg[j];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
          if (lane == 0) atomicAdd(dbh + j, v);
        }
      }
    }
    if (b.eval_only) { tc_fence_before(); __syncthreads(); continue; }
    TC_STAMP(8);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      // dxhat2 = dL Wh'       (M = 128 rows, N = 64 features, K = NH) first: S9 only needs this one ...
      const uint32_t idx = make_idesc(128, 64, 0, 0);
      umma_seq(tmem + cD, aP, 2 * ROWB, ROWB, aWhT, 2 * 1024, 1024, idx, NH / 8, false);
      umma_commit(bar_m);
      // ... Gh[k][a] += xhat2^T dL   (M = 64 features, N = NH, K = 128 rows; transposed tiles, K-major) runs behind the
      // first half of S9 and only gates the rewrite of TA
      const uint32_t idg = make_idesc(64, NH, 0, 0);
      umma_seq(tmem + cGh, aX2T, 2 * kS65 * 16, kS65 * 16, aTA, 2 * SH * 16, SH * 16, idg, kTM / 8, !first_tile);
      umma_commit(bar_g);
    }
    }   // MODE != TC_BASE_BWD
    if (MODE == TC_HEAD) {
      // ---- S9 (heads only): LayerNorm backward without an activation -> dL/dh of the head path, fp32, to the workspace ----
      float d[32];
      mbar_wait(bar_m, phase); phase ^= 1;
      tc_fence_after();
      tmem_ld16(tmem + lane_base + cMy, d);
      tmem_ld16(tmem + lane_base + cMy + 16, d + 16);
      tmem_ld_wait();
      {
        const float* base = X2T + ((r >> 2) * kS65 + wg * 32) * 4 + (r & 3);
        float xh[32];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int f = 0; f < 32; ++f) { xh[f] = base[f * 4]; s1 += d[f]; s2 = fmaf(d[f], xh[f], s2); }
        const float2 t = px.sum(s1, s2);
        s1 = t.x * (1.f / 64.f); s2 = t.y * (1.f / 64.f);
#pragma unroll
        for (int f = 0; f < 32; ++f) d[f] = rs2 * (d[f] - s1 - xh[f] * s2);
      }
      if (p < b.n_rows) { st_pl16(plane_out, (size_t)p, wg * 8, d); st_pl16(plane_out, (size_t)p, wg * 8 + 4, d + 16); }
      mbar_wait(bar_g, phase_g); phase_g ^= 1;             // Gh has consumed dL^T (TA) and xhat^T (X2T)
      tc_fence_after();
      first_tile = false;
      tc_fence_before();
      __syncthreads();
      continue;
    }
    // ---- S9: LayerNorm-2 + activation backward -> dZ2 (K-major staging + transposed) ----
    {
      float d[32];
      if (MODE == TC_BASE_BWD) {                           // dL/dxhat2 from the GRU input projection (update_gru_tc.cu)
#pragma unroll
        for (int i = 0; i < 32; ++i) d[i] = pref[i];
      } else {
        mbar_wait(bar_m, phase); phase ^= 1; TC_STAMP(9);
        tc_fence_after();
        tmem_ld16(tmem + lane_base + cMy, d);
        tmem_ld16(tmem + lane_base + cMy + 16, d + 16);
        tmem_ld_wait();
      }
      ln_act_bwd32(d, X2T, kS65, r, wg, px, mu2, rs2, act, pos2);
      put_kmajor32(P, r, wg, d, false);
      if (MODE != TC_BASE_BWD) {
        mbar_wait(bar_g, phase_g); phase_g ^= 1;           // Gh has consumed dL^T (TA)
        tc_fence_after();
      }
      put_transposed32(TA, kS65, r, wg, d);
    }
    TC_STAMP(10);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      // dxhat1 = dZ2 W2'             (M = 128, N = 64, K = 64) first ...
      const uint32_t idx = make_idesc(128, 64, 0, 0);
      umma_seq(tmem + cD, aP, 2 * ROWB, ROWB, aW2T, 2 * 1024, 1024, idx, 8, false);
      umma_commit(bar_m);
      // ... G2[o][k] += dZ2^T xhat1aug   (M = 64, N = 72, K = 128 rows) behind the first half of S11
      const uint32_t idg = make_idesc(64, kHF, 0, 0);
      umma_seq(tmem + cG2, aTA, 2 * kS65 * 16, kS65 * 16, aX1T, 2 * kS73 * 16, kS73 * 16, idg, kTM / 8, !first_tile);
      umma_commit(bar_g);
    }
    // ---- S11: LayerNorm-1 + activation backward -> dZ1^T; xhat0^T re-staged from its TMEM parking columns ----
    {
      float d[32];
      mbar_wait(bar_m, phase); phase ^= 1; TC_STAMP(11);
      tc_fence_after();
      tmem_ld16(tmem + lane_base + cMy, d);
      tmem_ld16(tmem + lane_base + cMy + 16, d + 16);
      tmem_ld_wait();
      ln_act_bwd32(d, X1T, kS73, r, wg, px, mu1, rs1, act, pos1);
      mbar_wait(bar_g, phase_g); phase_g ^= 1;             // G2 has consumed dZ2^T (TA)
      tc_fence_after();
      put_transposed32(TA, kS65, r, wg, d);
      float* pb = P + (r >> 2) * S0 * 4 + (r & 3);                // xhat0aug^T: [32][inF + 1][4]
#pragma unroll
      for (int c8 = 0; c8 < 9; ++c8) {
        if (c8 * 8 < inF && (c8 & 1) == wg) {
          float q[8];
          tmem_ld8(tmem + lane_base + cX0 + c8 * 8, q);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) pb[(c8 * 8 + j) * 4] = q[j];
        }
      }
    }
    TC_STAMP(12);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      // G1[o][k] += dZ1^T xhat0aug   (M = 64, N = inF, K = 128 rows)
      const uint32_t idg = make_idesc(64, inF, 0, 0);
      umma_seq(tmem + cG1, aTA, 2 * kS65 * 16, kS65 * 16, aP, 2 * S0 * 16, S0 * 16, idg, kTM / 8, !first_tile);
      umma_commit(bar_m);
    }
    first_tile = false;
    if (wg == 0 && tile + (int)gridDim.x >= n_tiles) { g1_pending = true; break; }   // last tile: G2 can be dumped now
    mbar_wait(bar_m, phase); phase ^= 1;                      // P / TA are rewritten by the next iteration
    tc_fence_after();
  }
  // ---- dump the raw (still folded) accumulators into this CTA's slot; they are summed over slots and unfolded once
  //      by mappo_update_finish (tc_unfold_kernel).  Warpgroup 0 dumps G2, warpgroup 1 dumps G1 and Gh. ----
  if (!b.eval_only && MODE != TC_BASE_FWD) {
    const TcRaw R = make_tc_raw(im);
    float* g = grad_part + (size_t)blockIdx.x * R.total;
    const bool has_tile = !first_tile && MODE != TC_HEAD;          // G2 / G1: not accumulated by the heads-only mode
    const bool has_head = !first_tile && MODE != TC_BASE_BWD;      // Gh: not accumulated by the base-backward mode
    const int o = (warp & 3) * 16 + lane;                 // accumulator row of this thread in the M = 64 layout
    const bool own = lane < 16;
    float v[72];
    if (wg == 0) {
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_ld16(tmem + lane_base + cG2 + c * 16, v + c * 16);
      tmem_ld8(tmem + lane_base + cG2 + 64, v + 64);
      tmem_ld_wait();
      if (own) {
#pragma unroll
        for (int q = 0; q < 18; ++q)
          reinterpret_cast<float4*>(g + R.g2 + o * kHF)[q] =
              has_tile ? make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_ld16(tmem + lane_base + cG1 + c * 16, v + c * 16);
      tmem_ld8(tmem + lane_base + cG1 + 64, v + 64);
      tmem_ld_wait();
      if (own) {
#pragma unroll
        for (int q = 0; q < 18; ++q)
          if (q * 4 < inF)
            reinterpret_cast<float4*>(g + R.g1 + o * inF)[q] =
                has_tile ? make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      tmem_ld16(tmem + lane_base + cGh, v);
      if (NH > 16) tmem_ld16(tmem + lane_base + cGh + 16, v + 16);
      tmem_ld_wait();
      if (own) {
#pragma unroll
        for (int q = 0; q < 8; ++q)
          if (q * 4 < NH)
            reinterpret_cast<float4*>(g + R.gh + o * NH)[q] =
                has_head ? make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    if (tid < NH) g[R.dbh + tid] = dbh[tid];
  }

  TC_STAMP(13);
  if (g1_pending) { mbar_wait(bar_m, phase); phase ^= 1; tc_fence_after(); }      // every MMA done before teardown
  TC_STAMP(14);
  // ---- loss scalars + teardown ----
  tc_fence_before();
  __syncthreads();
  if (MODE == TC_BASE_FWD || MODE == TC_BASE_BWD) {
    // no loss terms in these modes
  } else if (n.is_critic) {
    double one[1] = {acc[0]};
    block_accumulate<1>(one, loss_out + 0, sred, tid, kTCThreads);
  } else {
    double two[2] = {acc[0], acc[1]};
    block_accumulate<2>(two, loss_out + 1, sred, tid, kTCThreads);
    double rt[1] = {acc[2] / (lc.n_rows_d * (double)b.act_shape)};
    block_accumulate<1>(rt, loss_out + 5, sred, tid, kTCThreads);
  }
  if (warp == 0) tmem_dealloc(tmem, tmem_cols);
  TC_STAMP(15);
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
int debug_tc_timing(long long* out16) {
  return cudaMemcpyFromSymbol(out16, g_tc_timing, sizeof(long long) * 16) == cudaSuccess ? 0 : MAPPO_ERR_CUDA;
}

bool update_mlp_tc_supported(const NetDev& n) {
  return n.hid == 64 && n.layer_n == 1 && n.in_dim <= 63 && n.head_total <= 32 && !n.recurrent;
}

int64_t update_mlp_tc_workspace_floats(const NetDev& n) { return make_tc_image(n).total; }

int update_mlp_tc_slot_floats(const NetDev& n) { return make_tc_raw(make_tc_image(n)).total; }

// sum of the raw slots is in `raw_sum` -> flat gradient + sum(g^2) (one partial)
int update_mlp_tc_unfold_launch(const NetDev& n, const float* params, const float* raw_sum, float* grad,
                                float* sumsq_part, cudaStream_t st) {
  launch_pdl(tc_unfold_kernel, dim3(4, 3), dim3(256), 0, st, n, params, raw_sum, grad, sumsq_part);       // 12 partial sums of squares
  return check_launch("tc_unfold_kernel");
}

// ------------------------------------------------------------------------------------------------------------
// The whole optimiser tail of one net as ONE launch: slot sum -> unfold (+ sum g^2) -> [all-reduce over peer memory] ->
// clip + Adam -> folded image of the NEW weights for the next step's update kernel.
// One thread-block cluster of 8 CTAs x 1024 threads does the only wide part, the sum of the n_slots raw gradient slots
// (2.7 MB at c2), and delivers the result straight into the SHARED MEMORY of CTA 0 through distributed shared memory
// (st.shared::cluster); after one cluster barrier CTA 0 finishes alone out of its own shared memory -- the summed raw
// accumulators (43 KB), the gradient (42 KB) and the new parameters (42 KB) all fit -- so the unfold, the norm, Adam and the
// re-pack are separated by __syncthreads only, with no further global-memory hand-off.
// The arithmetic and every summation order are those of the kernels it replaces (grad_reduce_kernel's 8 x 4 partial sums per
// element, tc_unfold_unit, clip_adam_kernel<1>, pack_tc_element, p2p_allreduce_kernel).
// `stages`: bit 0 = slot sum + unfold (leaves grad + 12 partial sums of squares), bit 1 = clip + Adam + image (reading
// sumsq_part[0 .. n_part) when bit 0 did not run in the same launch), bit 2 = the data-parallel exchange between the two
// (only with both: 7) -- a multi-GPU optimiser step is then the update kernel plus THIS launch.
// ------------------------------------------------------------------------------------------------------------
constexpr int kTailCtas = 8, kTailThreads = 1024, kTailSubs = kTailThreads / 256, kTailUnits = kTailCtas * kTailSubs, kTailUnroll = 3;
struct TailArgs {
  NetDev n;
  const float* part; int n_slots;      // raw gradient slots [n_slots][R]
  float *p, *grad, *m, *v;             // flat parameters, gradient, Adam moments [P]
  float* sumsq_part; int n_part;       // partial sums of squares (stage 1 alone writes 12; stage 2 alone reads n_part)
  const float* lr_dev; int* step_dev; float eps, max_norm; int use_clip;
  double* norm_out; double* beta_pow;
  float* image;                        // folded tf32 weight image (NULL: not rebuilt)
  int stages;
  P2PArgs peers;                       // stage bit 2: symmetric buffers / signal pads of all ranks
  long long sym_offset_bytes;          // where the local gradient sits inside every rank's symmetric buffer
  uint32_t* round_dev;                 // {completed round, -, error flag, -} of this reducer
};
struct TailSmem { int raw, grad, par, total; };          // float offsets inside the dynamic shared memory
__host__ __device__ inline TailSmem make_tail_smem(const NetDev& n) {
  TailSmem t;
  const int R = make_tc_raw(make_tc_image(n)).total, P = n.g.total;
  t.raw = 0;
  t.grad = (R + 31) & ~31;
  t.par = t.grad + ((P + 31) & ~31);
  t.total = t.par + ((P + 31) & ~31);
  return t;
}

__global__ void __cluster_dims__(kTailCtas, 1, 1) __launch_bounds__(kTailThreads, 1) tc_tail_kernel(const TailArgs a) {
  extern __shared__ __align__(16) float tsm[];
  __shared__ float sacc[kTailSubs][kTailUnroll][8][33];
  __shared__ UnfoldScratch us[kTailSubs];
  __shared__ float s_sq[kTailUnits];
  __shared__ float s_total, s_coef, s_step_size, s_bc2_sqrt;
  __shared__ int s_step;
  __shared__ double s_p1, s_p2;
  __shared__ uint32_t s_round;
  const int tid = threadIdx.x, sub = tid >> 8, t = tid & 255;
  const int cta = (int)cluster_cta_rank();
  const int unit = cta * kTailSubs + sub;                        // 0 .. 31
  const TcImage im = make_tc_image(a.n);
  const TailSmem L = make_tail_smem(a.n);
  const int P = a.n.g.total;
  float* raw_s = tsm + L.raw;                                    // summed raw accumulators (valid in CTA 0)
  float* g_s = tsm + L.grad;                                     // the gradient Adam consumes
  float* p_s = tsm + L.par;                                      // parameters: the old ones for the unfold, the new ones for the re-pack
  constexpr int kPer = 11;                                       // parameters per thread of CTA 0 (P <= 11 K for every net of this path)

  // CTA 0: everything it will need from global memory is requested NOW, in flight underneath the slot sum
  float pr[kPer], mr[kPer], vr[kPer];
  int step_old = 0;
  double bp0 = 1.0, bp1 = 1.0, bp2 = -1.0;
  float lr = 0.f;
  if (cta == 0) {
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      const int i = tid + j * kTailThreads;
      pr[j] = i < P ? a.p[i] : 0.f;
    }
    if (tid == 0 && (a.stages & 2)) {
      step_old = *a.step_dev; lr = a.lr_dev[0];
      if (a.beta_pow) { bp0 = a.beta_pow[0]; bp1 = a.beta_pow[1]; bp2 = a.beta_pow[2]; }
    }
  }

  if (a.stages & 1) {
    // ---- slot sum (grad_reduce_kernel's order: warp sg adds slots sg, sg + 8, ... into 4 accumulators, then the 8 partials in turn)
    const int R = make_tc_raw(im).total, nvb = (R + 31) / 32;
    const int pi = t & 31, sg = t >> 5;
    const int n_it = (nvb + kTailUnits * kTailUnroll - 1) / (kTailUnits * kTailUnroll);
    for (int it = 0; it < n_it; ++it) {
#pragma unroll
      for (int u = 0; u < kTailUnroll; ++u) {
        const int vb = unit + kTailUnits * (it * kTailUnroll + u), i = vb * 32 + pi;
        float g0 = 0.f, g1 = 0.f, g2 = 0.f, g3 = 0.f;
        if (i < R) {
          if (a.n_slots <= 80) {
            // every slot value of this (element, slot group) is requested before the first add: ONE memory round trip instead of
            // one per loop iteration (the kernel is a chain of dependent loads: ncu showed 1.7 us of issue in 50 us).  The adds
            // keep grad_reduce_kernel's order (x + 0.f == x for the padded tail).
            float v[10];
#pragma unroll
            for (int q = 0; q < 10; ++q) {
              const int s = sg + 8 * q;
              v[q] = s < a.n_slots ? a.part[(size_t)s * R + i] : 0.f;
            }
            int qt = 0;                                    // first slot index of the sequential tail (indices stay compile time)
#pragma unroll
            for (int q0 = 0; q0 < 8; q0 += 4)
              if (qt == q0 && sg + 8 * q0 + 24 < a.n_slots) { g0 += v[q0]; g1 += v[q0 + 1]; g2 += v[q0 + 2]; g3 += v[q0 + 3]; qt = q0 + 4; }
#pragma unroll
            for (int q = 0; q < 10; ++q)
              if (q >= qt) g0 += v[q];
          } else {
            int s = sg;
            for (; s + 24 < a.n_slots; s += 32) {
              g0 += a.part[(size_t)s * R + i];
              g1 += a.part[(size_t)(s + 8) * R + i];
              g2 += a.part[(size_t)(s + 16) * R + i];
              g3 += a.part[(size_t)(s + 24) * R + i];
            }
            for (; s < a.n_slots; s += 8) g0 += a.part[(size_t)s * R + i];
          }
        }
        sacc[sub][u][sg][pi] = (g0 + g1) + (g2 + g3);
      }
      __syncthreads();
      if (sg == 0) {
#pragma unroll
        for (int u = 0; u < kTailUnroll; ++u) {
          const int vb = unit + kTailUnits * (it * kTailUnroll + u), i = vb * 32 + pi;
          float g = 0.f;
#pragma unroll
          for (int k = 0; k < 8; ++k) g += sacc[sub][u][k][pi];
          if (i < R) st_cluster_f32(raw_s + i, 0u, g);           // into CTA 0's shared memory
        }
      }
      __syncthreads();
    }
    cluster_sync_all();                                          // the DSMEM stores have landed in CTA 0
  }
  if (cta != 0) return;                                          // CTA 0 finishes alone (nobody touches the others' memory)
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const int i = tid + j * kTailThreads;
    if (i < P) p_s[i] = pr[j];
    mr[j] = ((a.stages & 2) && i < P) ? a.m[i] : 0.f;           // Adam moments: in flight underneath the unfold
    vr[j] = ((a.stages & 2) && i < P) ? a.v[i] : 0.f;
  }
  __syncthreads();

  int n_part = a.n_part;
  if (a.stages & 1) {
    // ---- unfold: the 12 (bx, by) units of tc_unfold_kernel's grid (4, 3), four at a time
    float* g_out = (a.stages & 4) ? reinterpret_cast<float*>(const_cast<char*>(static_cast<const char*>(a.peers.buf[a.peers.rank])) + a.sym_offset_bytes)
                                  : a.grad;
    for (int u0 = 0; u0 < 12; u0 += kTailSubs) {
      const int u = u0 + sub;
      tc_unfold_unit(a.n, p_s, raw_s, g_out, s_sq, u & 3, u >> 2, 4, t, u < 12, us[sub], g_s);
      __syncthreads();
    }
    n_part = 12;
    if (!(a.stages & 2) && tid < 12) a.sumsq_part[tid] = s_sq[tid];
  }
  if (a.stages & 4) {
    // ---- all-reduce over peer memory (p2p_allreduce_kernel<float>: arrive, wait, sum in rank order, per-block sum of squares)
    if (tid == 0) s_round = a.round_dev[0] + 1;
    __syncthreads();
    const uint32_t round = s_round;
    if (tid < a.peers.world) {
      __threadfence_system();                                     // the unfolded gradient is visible to the peers
      st_release_sys(a.peers.sig[tid] + a.peers.rank, round);
      const uint32_t* mine = a.peers.sig[a.peers.rank] + tid;
      const long long t0 = clock64();
      while ((int)(ld_acquire_sys(mine) - round) < 0) {
        if (clock64() - t0 > 8000000000LL) { atomicExch(a.round_dev + 2, 1u + (uint32_t)tid); break; }
      }
    }
    __syncthreads();
    // the stand-alone kernel's grid: `blocks` CTAs of 256 threads; sub-block s plays CTAs s, s + 4, ...
    const int n = P;
    int blocks = (n / 4 + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > kTailUnits) blocks = kTailUnits;
    for (int vb0 = 0; vb0 < blocks; vb0 += kTailSubs) {
      const int vb = vb0 + sub;
      float sq = 0.f;
      if (vb < blocks) {
        const int vt = vb * 256 + t, nt = blocks * 256;
        if ((n & 3) == 0 && (a.sym_offset_bytes & 15) == 0) {
          for (int i = vt; i < n / 4; i += nt) {
            float4 v[kMaxPeers];
#pragma unroll
            for (int q = 0; q < kMaxPeers; ++q)
              if (q < a.peers.world)
                v[q] = ld_peer4(reinterpret_cast<const float*>(static_cast<const char*>(a.peers.buf[q]) + a.sym_offset_bytes) + 4 * i);
            float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int q = 0; q < kMaxPeers; ++q)
              if (q < a.peers.world) { sum.x += v[q].x; sum.y += v[q].y; sum.z += v[q].z; sum.w += v[q].w; }
            reinterpret_cast<float4*>(a.grad)[i] = sum;
            reinterpret_cast<float4*>(g_s)[i] = sum;
            sq = fmaf(sum.x, sum.x, fmaf(sum.y, sum.y, fmaf(sum.z, sum.z, fmaf(sum.w, sum.w, sq))));
          }
        } else {
          for (int i = vt; i < n; i += nt) {
            float v[kMaxPeers];
#pragma unroll
            for (int q = 0; q < kMaxPeers; ++q)
              if (q < a.peers.world) v[q] = ld_peer<float>(reinterpret_cast<const float*>(static_cast<const char*>(a.peers.buf[q]) + a.sym_offset_bytes) + i);
            float sum = 0.f;
#pragma unroll
            for (int q = 0; q < kMaxPeers; ++q)
              if (q < a.peers.world) sum += v[q];
            a.grad[i] = sum;
            g_s[i] = sum;
            sq = fmaf(sum, sum, sq);
          }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
      if ((tid & 31) == 0) us[sub].sred[t >> 5] = sq;
      __syncthreads();
      if (t == 0 && vb < blocks) {
        float tot = 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) tot += us[sub].sred[q];
        s_sq[vb] = tot;
      }
      __syncthreads();
    }
    n_part = blocks;
    if (tid == 0) a.round_dev[0] = round;
  }
  if (!(a.stages & 2)) return;

  // ---- clip_grad_norm_ + Adam (clip_adam_kernel<1>: the scalar prologue in one warp, fixed order)
  const bool from_global = !(a.stages & 1);                       // stage 2 alone: gradient and partials come from global memory
  __syncthreads();
  if (tid < 32) {
    double x = 0.0;
    for (int i = tid; i < n_part; i += 32) x += (double)(from_global ? a.sumsq_part[i] : s_sq[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (tid == 0) {
      const float tot = (float)sqrt(x);
      const int st = step_old + 1;
      double p1, p2;
      if (a.beta_pow && bp2 == (double)(st - 1)) { p1 = bp0 * 0.9; p2 = bp1 * 0.999; }
      else { p1 = pow(0.9, (double)st); p2 = pow(0.999, (double)st); }
      s_p1 = p1; s_p2 = p2;
      const double bc1 = 1.0 - p1, bc2 = 1.0 - p2;
      s_total = tot;
      s_coef = a.use_clip ? fminf(a.max_norm / (tot + 1e-6f), 1.0f) : 1.f;
      s_step_size = (float)((double)lr / bc1);
      s_bc2_sqrt = (float)sqrt(bc2);
      s_step = st;
    }
  }
  __syncthreads();
  const float coef = s_coef, step_size = s_step_size, bc2_sqrt = s_bc2_sqrt;
  float gr[kPer];
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const int i = tid + j * kTailThreads;
    gr[j] = i < P ? (from_global ? a.grad[i] : g_s[i]) : 0.f;
  }
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const int i = tid + j * kTailThreads;
    if (i < P) {
      const float g = gr[j] * coef, m_in = mr[j], v_in = vr[j];
      const float mo = m_in + (g - m_in) * (float)(1.0 - 0.9);
      const float vo = v_in * 0.999f + (float)(1.0 - 0.999) * g * g;
      const float denom = sqrtf(vo) / bc2_sqrt + a.eps;
      const float pn = pr[j] - step_size * (mo / denom);
      a.p[i] = pn; p_s[i] = pn;
      a.m[i] = mo; a.v[i] = vo;
    }
  }
  if (tid == 0) {
    a.step_dev[0] = s_step;
    if (a.beta_pow) { a.beta_pow[0] = s_p1; a.beta_pow[1] = s_p2; a.beta_pow[2] = (double)s_step; }
    if (a.norm_out) *a.norm_out += (double)s_total;
  }
  __syncthreads();
  // ---- folded image of the new weights (pack_tc_kernel of the NEXT optimiser step), parameters read from shared memory
  if (a.image)
    for (int i = tid; i < im.total; i += kTailThreads) a.image[i] = pack_tc_element(a.n, im, p_s, i);
}

int update_mlp_tc_tail_launch(const NetDev& n, const float* part, int n_slots, float* raw_sum, float* params, float* grad, float* m,
                              float* v, float* sumsq_part, int n_part, const float* lr_dev, int* step_dev, float eps, float max_norm,
                              int use_clip, double* norm_out, double* beta_pow, float* image, int stages, cudaStream_t st,
                              const void* const* peer_bufs, void* const* peer_signals, int world, int rank, long long sym_offset_bytes,
                              uint32_t* round_dev) {
  if (!update_mlp_tc_supported(n)) { set_error("update_tail: the fused optimiser tail is built for the tcgen05 small-net path only"); return MAPPO_ERR_UNSUPPORTED; }
  if ((stages & 3) == 0 || ((stages & 1) && (!part || n_slots <= 0)) || ((stages & 2) && (!m || !v || !lr_dev || !step_dev)) ||
      ((stages & 3) == 2 && n_part <= 0)) { set_error("update_tail: bad arguments for stages %d", stages); return MAPPO_ERR_INVALID; }
  TailArgs a;
  (void)raw_sum;
  a.n = n; a.part = part; a.n_slots = n_slots; a.p = params; a.grad = grad; a.m = m; a.v = v;
  a.sumsq_part = sumsq_part; a.n_part = n_part; a.lr_dev = lr_dev; a.step_dev = step_dev; a.eps = eps; a.max_norm = max_norm;
  a.use_clip = use_clip; a.norm_out = norm_out; a.beta_pow = beta_pow; a.image = image; a.stages = stages;
  memset(&a.peers, 0, sizeof(a.peers));
  a.sym_offset_bytes = sym_offset_bytes; a.round_dev = round_dev;
  if (stages & 4) {
    if ((stages & 7) != 7) { set_error("update_tail: the exchange stage runs between stages 1 and 2 of the same launch (stages = 7)"); return MAPPO_ERR_INVALID; }
    if (!peer_bufs || !peer_signals || !round_dev || world < 1 || world > kMaxPeers || rank < 0 || rank >= world || (sym_offset_bytes & 3)) {
      set_error("update_tail: bad peer arguments (world %d, rank %d)", world, rank); return MAPPO_ERR_INVALID;
    }
    for (int q = 0; q < world; ++q) { a.peers.buf[q] = peer_bufs[q]; a.peers.sig[q] = static_cast<uint32_t*>(peer_signals[q]); }
    a.peers.world = world; a.peers.rank = rank;
  }
  if (n.g.total > 11 * kTailThreads) { set_error("update_tail: %d parameters exceed the kernel's register budget", n.g.total); return MAPPO_ERR_UNSUPPORTED; }
  const size_t bytes = (size_t)make_tail_smem(n).total * sizeof(float);
  static thread_local SmemConfig tail_cfg = {};
  size_t& configured = tail_cfg.slot();
  if (bytes > configured) {
    if (cudaFuncSetAttribute(tc_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
      return check_launch("tc_tail_kernel: cudaFuncSetAttribute");
    // same shared-memory carveout as the update kernel it alternates with on these SMs (no L1 / shared re-partitioning between them)
    cudaFuncSetAttribute(tc_tail_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    configured = bytes;
  }
  tc_tail_kernel<<<kTailCtas, kTailThreads, bytes, st>>>(a);
  return check_launch("tc_tail_kernel");
}

int update_mlp_tc_slots(const NetDev&, int n_rows, int sm_count) {
  const int n_tiles = (n_rows + kTM - 1) / kTM;
  return n_tiles < sm_count ? n_tiles : sm_count;
}

int update_mlp_tc_launch(const NetDev& n, const float* params, const BatchDev& b, const LossDev& L,
                         const double* norm_stats, const double* adv_stats, const float* vn_state, float* grad_part,
                         int n_slots, double* loss_out, float* image, cudaStream_t st, bool image_ready) {
  if (!update_mlp_tc_supported(n)) { set_error("update_mlp_tc: configuration not built for the tcgen05 path"); return MAPPO_ERR_UNSUPPORTED; }
  if (!image) { set_error("update_mlp_tc: weight-image workspace is NULL"); return MAPPO_ERR_INVALID; }
  if ((reinterpret_cast<uintptr_t>(image) & 15) != 0) { set_error("update_mlp_tc: workspace must be 16-byte aligned"); return MAPPO_ERR_INVALID; }
  const TcImage im = make_tc_image(n);
  const TcSmem sm = make_tc_smem(im);
  const size_t bytes = (size_t)sm.total * sizeof(float) + 1024;
  if (bytes > 227 * 1024) { set_error("update_mlp_tc: %zu B shared memory > 227 KB", bytes); return MAPPO_ERR_UNSUPPORTED; }
  if (!image_ready) {                  // (the fused optimiser tail of the previous step leaves the image of the current weights)
    launch_pdl(pack_tc_kernel, dim3((im.total + 255) / 256), dim3(256), 0, st, n, params, image);      // one element per thread
    const int rc = check_launch("pack_tc_kernel");
    if (rc) return rc;
  }
  static thread_local SmemConfig configured_dev = {};
  size_t& configured = configured_dev.slot();
  if (bytes > configured) {
    if (cudaFuncSetAttribute(update_mlp_tc_kernel<TC_FULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
      return check_launch("update_mlp_tc: cudaFuncSetAttribute");
    configured = bytes;
  }
  const int n_tiles = (b.n_rows + kTM - 1) / kTM;
  const uint32_t cols = 512u;          // accumulators [0,272) + parked xhat0 [272,344): one CTA per SM owns all of TMEM
  launch_pdl(update_mlp_tc_kernel<TC_FULL>, dim3(n_slots), dim3(kTCThreads), bytes, st, n, params, image, b, L, norm_stats, adv_stats, vn_state,
             grad_part, loss_out, n_tiles, cols, (const float*)nullptr, (float*)nullptr);
  return check_launch("update_mlp_tc_kernel");
}


// ---- recurrent nets (update_gru_tc.cu): the same kernel around the GRU sequence kernels ----
int update_mlp_tc_pack_launch(const NetDev& n, const float* params, float* image, cudaStream_t st) {
  const TcImage im = make_tc_image(n);
  launch_pdl(pack_tc_kernel, dim3((im.total + 255) / 256), dim3(256), 0, st, n, params, image);
  return check_launch("pack_tc_kernel");
}

template <int MODE>
static int mode_launch(const NetDev& n, const float* params, const float* image, const BatchDev& b, const LossDev& L,
                       const double* norm_stats, const double* adv_stats, const float* vn_state, float* grad_part, int n_ctas,
                       double* loss_out, const float* plane_in, float* plane_out, cudaStream_t st) {
  const TcImage im = make_tc_image(n);
  const TcSmem sm = make_tc_smem(im);
  const size_t bytes = (size_t)sm.total * sizeof(float) + 1024;
  if (bytes > 227 * 1024) { set_error("update_mlp_tc: %zu B shared memory > 227 KB", bytes); return MAPPO_ERR_UNSUPPORTED; }
  static thread_local SmemConfig configured_dev = {};
  size_t& configured = configured_dev.slot();
  if (bytes > configured) {
    if (cudaFuncSetAttribute(update_mlp_tc_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
      return check_launch("update_mlp_tc: cudaFuncSetAttribute");
    configured = bytes;
  }
  const int n_tiles = (b.n_rows + kTM - 1) / kTM;
  launch_pdl(update_mlp_tc_kernel<MODE>, dim3(n_ctas), dim3(kTCThreads), bytes, st, n, params, image, b, L, norm_stats, adv_stats, vn_state,
             grad_part, loss_out, n_tiles, 512u, plane_in, plane_out);
  return check_launch("update_mlp_tc_kernel<mode>");
}

int update_mlp_tc_mode_launch(int mode, const NetDev& n, const float* params, const float* image, const BatchDev& b, const LossDev& L,
                              const double* norm_stats, const double* adv_stats, const float* vn_state, float* grad_part, int n_ctas,
                              double* loss_out, const float* plane_in, float* plane_out, cudaStream_t st) {
  if (n.hid != 64 || n.layer_n != 1 || n.in_dim > 63 || n.head_total > 32) { set_error("update_mlp_tc: configuration not built"); return MAPPO_ERR_UNSUPPORTED; }
  switch (mode) {
    case TC_BASE_FWD: return mode_launch<TC_BASE_FWD>(n, params, image, b, L, norm_stats, adv_stats, vn_state, grad_part, n_ctas, loss_out, plane_in, plane_out, st);
    case TC_BASE_BWD: return mode_launch<TC_BASE_BWD>(n, params, image, b, L, norm_stats, adv_stats, vn_state, grad_part, n_ctas, loss_out, plane_in, plane_out, st);
    case TC_HEAD:     return mode_launch<TC_HEAD>(n, params, image, b, L, norm_stats, adv_stats, vn_state, grad_part, n_ctas, loss_out, plane_in, plane_out, st);
  }
  set_error("update_mlp_tc: bad mode %d", mode);
  return MAPPO_ERR_INVALID;
}

}  // namespace mappo
