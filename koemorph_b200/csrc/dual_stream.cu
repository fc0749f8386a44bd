// Dual-stream attention core on CUDA cores (precision 0: exact fp32 FMA), emotion stream and EMA scan.
//
// Replaces DualStreamCrossAttention.forward (reference src/model/dual_stream_attention.py:162-280),
// the eGeMAPS compression (src/features/opensmile_extractor.py:583-604) and apply_temporal_smoothing
// (src/model/simplified_dual_stream_model.py:341-368).
//
// One persistent CTA per SM walks over (clip, window) work items.  Per window, everything between the
// mel-power rows in HBM and the 52 output coefficients stays in shared memory / registers:
//   P0  window dB reference (max over the window's frame maxima), normalise rows -> A block
//   G1  z = Xn[80 x K] Wc^T + bc, LayerNorm          (K = 259 / 515, streamed in 64-row blocks)
//   G3  V = enc Wv^T + bv                            [80 x 256]
//   S   scores^T = enc Qk^T                          [80 x 224]; Qk folds (Wq q + bq)/sqrt(32) and Wk,
//                                                    the key bias adds a per-row constant that softmax drops
//   softmax over the 80 mel-channel tokens, P V per head, O -> h = relu(O Wa^T + ba), sigmoid(h w2 + b2)
//   fusion: out[idx] = clamp(coef[idx] * y), coef = 0.5 (softmax(mel_w/T) + softmax(emo_w/T)).
#include <algorithm>

#include "common.cuh"
#include "core_params.cuh"

namespace koe {

constexpr int kTok = KOE_N_MELS;         // 80 tokens (mel channels) per window
constexpr int kD = KOE_D_MODEL;          // 256
constexpr int kHQ = KOE_N_HEADS * KOE_N_MOUTH;  // 224 score rows
constexpr int kCoreThreads = 256;
constexpr int kKC = 16;                  // weight rows per cp.async stage
constexpr int kABlockRows = 64;          // rows of Xn staged per G1 block
constexpr int kEncStride = 81;           // encT[n][m] row stride (odd: conflict-free transposed stores)
constexpr int kVStride = kD;             // V[m][n]
constexpr int kSStride = 84;             // S[hq][t] row stride (float4-aligned)
constexpr int kOStride = 36;             // OT[k][q] row stride (float4-aligned)

// acc[TM][TN] += A[k][ty*TM + i] * B[k][tx + 32 j] for k < K.
// A lives in shared memory ([K][lda]); B is streamed from global ([ceil16(K)][32*TN], zero padded) through a
// two-stage cp.async ring.  Ends with a __syncthreads().
template <int TM, int TN, bool A_VEC2>
__device__ __forceinline__ void gemm_acc(const float* __restrict__ As, int lda, const float* __restrict__ Bg, int K,
                                         float* __restrict__ stage, float (&acc)[TM][TN], int tid) {
  constexpr int NC = 32 * TN;
  constexpr int F4 = kKC * NC / 4;
  const int tx = tid & 31, ty = tid >> 5;
  const int nchunks = (K + kKC - 1) / kKC;
  auto issue = [&](int c) {
    const float4* src = reinterpret_cast<const float4*>(Bg + (size_t)c * kKC * NC);
    float4* dst = reinterpret_cast<float4*>(stage + (c & 1) * kKC * NC);
#pragma unroll
    for (int i = 0; i < F4 / kCoreThreads; ++i) cp_async16(dst + tid + i * kCoreThreads, src + tid + i * kCoreThreads);
    cp_async_commit();
  };
  // packed fp32x2 accumulators: acc2[i][j] = (acc[i][2j], acc[i][2j+1]); one FFMA2 (broadcast a, pair of b) does the work
  // of two FFMAs in one issue slot -- same rounding per element, so the results are bit-identical to the scalar form
  static_assert(TN % 2 == 0, "TN must be even");
  float2 acc2[TM][TN / 2];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN / 2; ++j) acc2[i][j] = make_float2(acc[i][2 * j], acc[i][2 * j + 1]);
  issue(0);
  for (int c = 0; c < nchunks; ++c) {
    if (c + 1 < nchunks) {
      issue(c + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* bs = stage + (c & 1) * kKC * NC + tx;
    const float* as = As + (size_t)c * kKC * lda + ty * TM;
    const int kmax = min(kKC, K - c * kKC);
#pragma unroll 4
    for (int kk = 0; kk < kmax; ++kk) {
      float a[TM];
      float2 b[TN / 2];
      if constexpr (A_VEC2) {
#pragma unroll
        for (int i = 0; i < TM / 2; ++i) {
          const float2 v = *reinterpret_cast<const float2*>(as + kk * lda + 2 * i);
          a[2 * i] = v.x;
          a[2 * i + 1] = v.y;
        }
      } else {
#pragma unroll
        for (int i = 0; i < TM; ++i) a[i] = as[kk * lda + i];
      }
#pragma unroll
      for (int j = 0; j < TN / 2; ++j) b[j] = make_float2(bs[kk * NC + 64 * j], bs[kk * NC + 64 * j + 32]);
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN / 2; ++j) acc2[i][j] = __ffma2_rn(make_float2(a[i], a[i]), b[j], acc2[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN / 2; ++j) {
      acc[i][2 * j] = acc2[i][j].x;
      acc[i][2 * j + 1] = acc2[i][j].y;
    }
}

constexpr size_t kCoreSmemFloats = (size_t)kABlockRows * kTok      // A block
                                   + (size_t)kD * kEncStride       // encT, later S/P
                                   + (size_t)kTok * kVStride       // V, later OT
                                   + 2 * kKC * kD                  // weight stages
                                   + 64;                           // reductions
constexpr size_t kCoreSmem = kCoreSmemFloats * sizeof(float);

// one instantiation per CoreMode except Early; the window of a work item and the rows of its frames come from CoreRows<M>
template <CoreMode M>
__global__ void __launch_bounds__(kCoreThreads, 1) dual_stream_fp32_kernel(CoreParams p) {
  extern __shared__ __align__(16) float smem[];
  float* s_a = smem;                               // [64][80]
  float* s_enc = s_a + kABlockRows * kTok;         // [256][81]  (S: [224][84])
  float* s_v = s_enc + kD * kEncStride;            // [80][256]  (OT: [256][36])
  float* s_stage = s_v + kTok * kVStride;          // [2][16][256]
  float* s_red = s_stage + 2 * kKC * kD;           // [64]

  const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
  const koe_core_weights& W = p.w;
  const int T_launch = p.frames_per_window;
  const int n_items = p.n_clips * p.n_out;

  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const CoreWindow win = CoreRows<M>::template window<true>(p, item);
    const int T = CoreRows<M>::frames(win, T_launch);
    const bool prenorm = p.mel_long != nullptr;

    // ---- P0: dB reference of this window -------------------------------------------------------
    float ref_db = 0.0f;
    if (!prenorm) {
      float mx = -INFINITY;
      for (int k = tid; k < T; k += kCoreThreads) {
        const int v = win.plain_only ? 0 : CoreRows<M>::variant(p, win, T, k);
        mx = fmaxf(mx, p.fmax[v][CoreRows<M>::row(p, win, v, k)]);
      }
      mx = warp_max(mx);
      if (tx == 0) s_red[ty] = mx;
      __syncthreads();
      if (tid < 32) {
        float v = tid < 8 ? s_red[tid] : -INFINITY;
        v = warp_max(v);
        if (tid == 0) s_red[8] = v;
      }
      __syncthreads();
      ref_db = s_red[8];
    }

    // ---- G1: z = Xn Wc^T, K streamed in 64-row blocks -------------------------------------------
    float acc[10][8];
#pragma unroll
    for (int i = 0; i < 10; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;

    for (int kb = 0; kb < W.k_mel; kb += kABlockRows) {
      const int rows = min(kABlockRows, W.k_mel - kb);
      for (int idx = tid; idx < rows * (kTok / 4); idx += kCoreThreads) {
        const int r = idx / (kTok / 4), q = idx % (kTok / 4);
        const int t = kb + r;
        int k;  // window frame feeding row t, or -1 for zero padding
        if (t < p.mel_seq) {
          k = t < T ? t : -1;
        } else {
          const int s = t - p.mel_seq;
          k = T >= 3 ? T - 3 + s : (s < T ? s : -1);
        }
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (prenorm) {
          if (t >= p.mel_seq)
            v = __ldg(reinterpret_cast<const float4*>(p.mel_short + ((size_t)win.owner * 3 + (t - p.mel_seq)) * kTok) + q);
          else if (t < p.n_long)
            v = __ldg(reinterpret_cast<const float4*>(p.mel_long + ((size_t)win.owner * p.n_frames + t) * kTok) + q);
        } else if (k >= 0) {
          const int var = win.plain_only ? 0 : CoreRows<M>::variant(p, win, T, k);
          const float4 pw = __ldg(reinterpret_cast<const float4*>(p.power[var] + CoreRows<M>::row(p, win, var, k) * kTok) + q);
          v.x = normalise_db(pw.x, ref_db, true);
          v.y = normalise_db(pw.y, ref_db, true);
          v.z = normalise_db(pw.z, ref_db, true);
          v.w = normalise_db(pw.w, ref_db, true);
        }
        *reinterpret_cast<float4*>(s_a + r * kTok + 4 * q) = v;
      }
      __syncthreads();
      gemm_acc<10, 8, true>(s_a, kTok, W.wc_t + (size_t)kb * kD, rows, s_stage, acc, tid);
    }

    // ---- bias + LayerNorm over the 256 features of each token (one warp owns 10 whole tokens) ----
    {
      float bcv[8], gv[8], bv[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        bcv[j] = __ldg(W.bc + tx + 32 * j);
        gv[j] = __ldg(W.ln_g + tx + 32 * j);
        bv[j] = __ldg(W.ln_b + tx + 32 * j);
      }
#pragma unroll
      for (int i = 0; i < 10; ++i) {
        float s = 0.0f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc[i][j] += bcv[j];
          s += acc[i][j];
        }
        const float mean = warp_sum(s) * (1.0f / kD);
        float q = 0.0f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float d = acc[i][j] - mean;
          q = fmaf(d, d, q);
        }
        const float rstd = rsqrtf(warp_sum(q) * (1.0f / kD) + W.ln_eps);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          s_enc[(tx + 32 * j) * kEncStride + ty * 10 + i] = (acc[i][j] - mean) * rstd * gv[j] + bv[j];
      }
    }
    __syncthreads();

    // ---- G3: V = enc Wv^T + bv -> s_v[m][n] -----------------------------------------------------
#pragma unroll
    for (int i = 0; i < 10; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
    gemm_acc<10, 8, false>(s_enc, kEncStride, W.wv_t, kD, s_stage, acc, tid);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float bias = __ldg(W.bv + tx + 32 * j);
#pragma unroll
      for (int i = 0; i < 10; ++i) s_v[(ty * 10 + i) * kVStride + tx + 32 * j] = acc[i][j] + bias;
    }

    // ---- S^T = enc Qk^T (columns hq = h*28 + q; 224..255 are zero padding) ----------------------
#pragma unroll
    for (int i = 0; i < 10; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
    gemm_acc<10, 8, false>(s_enc, kEncStride, W.qk_t, kD, s_stage, acc, tid);
    // every warp is past its last read of s_enc (gemm_acc ends with a barrier): reuse it for S[hq][t]
    float* s_s = s_enc;
#pragma unroll
    for (int j = 0; j < 7; ++j)
#pragma unroll
      for (int i = 0; i < 10; ++i) s_s[(tx + 32 * j) * kSStride + ty * 10 + i] = acc[i][j];
    __syncthreads();

    // ---- softmax over the 80 tokens of each of the 224 rows (warp per row) ----------------------
    for (int r = ty; r < kHQ; r += 8) {
      float* row = s_s + r * kSStride;
      const float v0 = row[tx], v1 = row[tx + 32], v2 = tx < 16 ? row[tx + 64] : -INFINITY;
      const float m = warp_max(fmaxf(fmaxf(v0, v1), v2));
      const float e0 = expf(v0 - m), e1 = expf(v1 - m), e2 = tx < 16 ? expf(v2 - m) : 0.0f;
      const float inv = 1.0f / warp_sum(e0 + e1 + e2);
      row[tx] = e0 * inv;
      row[tx + 32] = e1 * inv;
      if (tx < 16) row[tx + 64] = e2 * inv;
    }
    __syncthreads();

    if (p.attn_out != nullptr) {  // head-averaged weights (nn.MultiheadAttention need_weights=True)
      float* dst = p.attn_out + (size_t)item * KOE_N_MOUTH * kTok;
      for (int idx = tid; idx < KOE_N_MOUTH * kTok; idx += kCoreThreads) {
        const int q = idx / kTok, t = idx % kTok;
        float s = 0.0f;
#pragma unroll
        for (int h = 0; h < KOE_N_HEADS; ++h) s += s_s[(h * KOE_N_MOUTH + q) * kSStride + t];
        dst[idx] = s * (1.0f / KOE_N_HEADS);
      }
    }

    // ---- O[h][q][d] = sum_t P[h*28+q][t] V[t][32 h + d]: warp = head, lane = d --------------------
    float o[KOE_N_MOUTH];
#pragma unroll
    for (int q = 0; q < KOE_N_MOUTH; ++q) o[q] = 0.0f;
    {
      const float* prow = s_s + (ty * KOE_N_MOUTH) * kSStride;
      const float* vcol = s_v + 32 * ty + tx;
      for (int t = 0; t < kTok; t += 4) {
        const float v0 = vcol[(t + 0) * kVStride], v1 = vcol[(t + 1) * kVStride];
        const float v2 = vcol[(t + 2) * kVStride], v3 = vcol[(t + 3) * kVStride];
#pragma unroll
        for (int q = 0; q < KOE_N_MOUTH; ++q) {
          const float4 pq = *reinterpret_cast<const float4*>(prow + q * kSStride + t);
          o[q] = fmaf(pq.x, v0, o[q]);
          o[q] = fmaf(pq.y, v1, o[q]);
          o[q] = fmaf(pq.z, v2, o[q]);
          o[q] = fmaf(pq.w, v3, o[q]);
        }
      }
    }
    __syncthreads();  // all reads of s_v done -> reuse as OT[k = 32 h + d][q]
    float* s_o = s_v;
#pragma unroll
    for (int q = 0; q < KOE_N_MOUTH; ++q) s_o[(32 * ty + tx) * kOStride + q] = o[q];
#pragma unroll
    for (int q = KOE_N_MOUTH; q < 32; ++q) s_o[(32 * ty + tx) * kOStride + q] = 0.0f;
    __syncthreads();

    // ---- decoder: h = relu(O Wa^T + ba) [28 x 128], logit = h . w2 + b2 --------------------------
    float hacc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) hacc[i][j] = 0.0f;
    gemm_acc<4, 4, true>(s_o, kOStride, W.wa_t, kD, s_stage, hacc, tid);
    {
      float part[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float ba = __ldg(W.ba + tx + 32 * j), w2 = __ldg(W.w2 + tx + 32 * j);
#pragma unroll
        for (int i = 0; i < 4; ++i) part[i] = fmaf(fmaxf(hacc[i][j] + ba, 0.0f), w2, part[i]);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) part[i] = warp_sum(part[i]);
      if (tx < 4) {
        const int q = ty * 4 + tx;
        if (q < KOE_N_MOUTH) {
          const float logit = (tx == 0 ? part[0] : tx == 1 ? part[1] : tx == 2 ? part[2] : part[3]) + W.b2;
          const float y = 1.0f / (1.0f + expf(-logit));
          const int idx = __ldg(W.mouth_idx + q);
          const size_t o_off = (size_t)item * KOE_N_BLENDSHAPES + idx;
          p.out[o_off] = fminf(fmaxf(__ldg(W.coef + idx) * y, 0.0f), 1.0f);
          if (p.sigmoid_out != nullptr) p.sigmoid_out[o_off] = y;
        }
      }
    }
    if (tid < KOE_N_EXPR && p.expr_sigmoid != nullptr) {  // (NULL: the fused forward's emotion kernel writes these)
      const float y = __ldg(p.expr_sigmoid + win.owner);
      const int idx = __ldg(W.expr_idx + tid);
      const size_t o_off = (size_t)item * KOE_N_BLENDSHAPES + idx;
      p.out[o_off] = fminf(fmaxf(__ldg(W.coef + idx) * y, 0.0f), 1.0f);
      if (p.sigmoid_out != nullptr) p.sigmoid_out[o_off] = y;
    }
    __syncthreads();
  }
}

constexpr int kEmoInMax = 272;

// ---- emotion stream (reference dual_stream_attention.py:234-240 with the 264 -> 256 compression folded in): two GEMVs
// around a LayerNorm per clip, x [emo_in] -> z [256] -> LayerNorm -> relu(h [128]) . w2 -> sigmoid.
// The expression blendshapes depend on the emotion stream ONLY and the mouth blendshapes on the mel stream only, so in the
// fused forward (csrc/session.cu) this kernel writes its 24 entries of every output row itself and the core skips them:
// the core does not wait for this kernel's results, and this kernel -- a few dozen CTAs, ~9 us each -- runs on the SMs
// that the frontend's CTAs leave first (their ends are spread over ~15 us), done about when the last of them is.
//   * weights arrive through a ring of 32 KiB stages, one cp.async.bulk (TMA) each, issued by a producer warp: 32 rows of
//     we1_t [emo_in][256], then 64 rows of we2_t [256][128]
//   * register tiles: a thread owns 4 output features x NC clips (NC / 2 packed FFMA2 per feature and weight row: one
//     16-byte weight load, NC / 4 broadcast 16-byte input loads); a warp is one K slice (rows k = slice mod 4 / 8) of 128
//     features, the slices' partial sums meet in shared memory in a fixed order
//   * everything else the CTA reads (inputs, biases, LayerNorm vectors, output constants) is requested at once at the
//     start: eight warps cannot hide one memory latency per phase
constexpr int kEt2Stage = 32768;
constexpr int kEt2Rows1 = kEt2Stage / (kD * 4);      // 32 rows of we1_t per stage
constexpr int kEt2Rows2 = kEt2Stage / (128 * 4);     // 64 rows of we2_t per stage
constexpr int kEt2Threads = 288;                     // 8 consumer warps + the producer warp
constexpr int kEt2XLoads = (kEmoInMax + 255) / 256;  // input values per thread per clip
template <int NC>
struct Et2 {
  static constexpr int kSlots = NC > 8 ? 3 : 4;
  static constexpr size_t kSmem = (size_t)kSlots * kEt2Stage + sizeof(float) * (kEmoInMax * NC   // x [k][clip]
                                                                               + 4 * NC * kD      // partial sums
                                                                               + kD * NC          // LayerNorm output [k][clip]
                                                                               + 5 * kD)          // be1, eln_g, eln_b, be2, w2
                                  + 8 * 2 * kSlots + 16;
};

template <int NP>  // NP = clips / 2: one packed accumulator per feature and clip pair
__device__ __forceinline__ void et2_row(const float4 w, const float4* __restrict__ x, float2 (&acc)[4][NP]) {
  const float wf[4] = {w.x, w.y, w.z, w.w};
  float2 x2[NP];
#pragma unroll
  for (int q = 0; q < NP / 2; ++q) {
    const float4 v = x[q];
    x2[2 * q] = make_float2(v.x, v.y), x2[2 * q + 1] = make_float2(v.z, v.w);
  }
#pragma unroll
  for (int f = 0; f < 4; ++f)
#pragma unroll
    for (int c = 0; c < NP; ++c) acc[f][c] = __ffma2_rn(make_float2(wf[f], wf[f]), x2[c], acc[f][c]);
}

__device__ __forceinline__ long long global_ns() {
  unsigned long long g;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
  return (long long)g;
}

// kVarlen: clip c's output rows are [row_base[c], row_base[c + 1]) (the packed variable-length forward) instead of n_out
// rows from c * n_out; a separate instantiation
template <int NC, bool kVarlen = false>
__global__ void __launch_bounds__(kEt2Threads, 1)
emotion_tiled_kernel(koe_core_weights W, const float* __restrict__ emo_in, int n_clips, float* __restrict__ expr_sigmoid,
                     float* __restrict__ out, float* __restrict__ sigmoid_out, int n_out, long long* dbg,
                     const int* __restrict__ row_base) {
  constexpr int kSlots = Et2<NC>::kSlots, NP = NC / 2;
  extern __shared__ __align__(128) unsigned char et2_smem[];
  unsigned char* s_ring = et2_smem;
  float* s_x = reinterpret_cast<float*>(et2_smem + kSlots * kEt2Stage);     // [emo_in_pad][NC]
  float* s_part = s_x + kEmoInMax * NC;                                      // [slice][clip][feature]
  float* s_zn = s_part + 4 * NC * kD;                                        // [256][NC]
  float* s_vec = s_zn + kD * NC;                                             // be1 | eln_g | eln_b | be2 (128) . w2 (128)
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_vec + 5 * kD);
  const uint32_t bar_full = smem_u32addr(s_bar), bar_empty = bar_full + 8 * kSlots;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c0 = blockIdx.x * NC;
  const int nc = min(NC, n_clips - c0);
  const int n1 = (W.emo_in_pad + kEt2Rows1 - 1) / kEt2Rows1, n2 = kD / kEt2Rows2;
  if (dbg != nullptr && tid == 0) dbg[3 * blockIdx.x] = global_ns();  // (scripts/chain_timeline.py)
  if (tid == 0) {
    for (int i = 0; i < kSlots; ++i) {
      mbarrier_init(bar_full + 8 * i, 1);
      mbarrier_init(bar_empty + 8 * i, 8);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  // Launched behind the frontend with the programmatic attribute: this kernel reads nothing the frontend writes (the
  // frontend released it after its own wait, so everything queued before THAT has completed).  The next kernel of the
  // stream (the core) may set itself up beside this one; it orders itself by its own griddepcontrol.wait.
  pdl_launch_dependents();

  if (warp == 8) {
    // ===================================================== weight producer =============================
    // The whole warp runs the loop and one lane issues: lanes that left it early would sit in the griddepcontrol.wait at
    // the end of the kernel, and that stalls the WARP -- the issuing lane with it -- until the previous kernel has
    // completed (measured: the weight stages arrived 11 us late, exactly when that kernel ended).
    uint32_t slot = 0, phase = 0;
    for (int c = 0; c < n1 + n2; ++c) {
      mbarrier_wait(bar_empty + 8 * slot, phase ^ 1);
      const float* src;
      uint32_t bytes;
      if (c < n1) {
        src = W.we1_t + (size_t)c * kEt2Rows1 * kD;
        bytes = (uint32_t)min(kEt2Rows1, W.emo_in_pad - c * kEt2Rows1) * kD * 4;
      } else {
        src = W.we2_t + (size_t)(c - n1) * kEt2Rows2 * 128;
        bytes = kEt2Stage;
      }
      if (lane == 0) {
        mbarrier_expect_tx(bar_full + 8 * slot, bytes);
        bulk_copy_g2s(smem_u32addr(s_ring + slot * kEt2Stage), src, bytes, bar_full + 8 * slot);
      }
      __syncwarp();
      if (++slot == kSlots) slot = 0, phase ^= 1;
    }
  } else {
    // ===================================================== consumers ===================================
    // inputs, clip-contiguous (x[k][0..NC): broadcast 16-byte loads per weight row; rows beyond emo_in read as zero)
    {
      float xv[NC][kEt2XLoads];
#pragma unroll
      for (int c = 0; c < NC; ++c)
#pragma unroll
        for (int j = 0; j < kEt2XLoads; ++j) {
          const int k = tid + 256 * j;
          xv[c][j] = (c < nc && k < W.emo_in) ? __ldg(emo_in + (size_t)(c0 + c) * W.emo_in + k) : 0.0f;
        }
      const float v0 = __ldg(W.be1 + tid), v1 = __ldg(W.eln_g + tid), v2 = __ldg(W.eln_b + tid);
      const float v3 = tid < 128 ? __ldg(W.be2 + tid) : __ldg(W.w2 + tid - 128);
#pragma unroll
      for (int j = 0; j < kEt2XLoads; ++j) {
        const int k = tid + 256 * j;
        if (k < W.emo_in_pad) {
#pragma unroll
          for (int q = 0; q < NC / 4; ++q)
            *reinterpret_cast<float4*>(s_x + k * NC + 4 * q) =
                make_float4(xv[4 * q][j], xv[4 * q + 1][j], xv[4 * q + 2][j], xv[4 * q + 3][j]);
        }
      }
      s_vec[tid] = v0, s_vec[kD + tid] = v1, s_vec[2 * kD + tid] = v2, s_vec[3 * kD + tid] = v3;
    }
    int o_idx = 0;
    float o_coef = 0.0f;
    if (lane < KOE_N_EXPR) {
      o_idx = __ldg(W.expr_idx + lane);
      o_coef = __ldg(W.coef + o_idx);
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    const float *s_be1 = s_vec, *s_g = s_vec + kD, *s_b = s_vec + 2 * kD, *s_be2 = s_vec + 3 * kD, *s_w2 = s_vec + 3 * kD + 128;
    uint32_t slot = 0, phase = 0;
    float2 acc[4][NP];
    // ---- layer 1: z = we1_t^T x.  warp = (K slice = warp >> 1, feature block = warp & 1); thread: features 4 fl .. 4 fl + 3
    {
      const int slice = warp >> 1, fl = 32 * (warp & 1) + lane;
#pragma unroll
      for (int f = 0; f < 4; ++f)
#pragma unroll
        for (int c = 0; c < NP; ++c) acc[f][c] = make_float2(0.0f, 0.0f);
      for (int ch = 0; ch < n1; ++ch) {
        mbarrier_wait(bar_full + 8 * slot, phase);
        const float4* wrow = reinterpret_cast<const float4*>(s_ring + slot * kEt2Stage) + fl;
        const int r0 = ch * kEt2Rows1, rows = min(kEt2Rows1, W.emo_in_pad - r0);
#pragma unroll
        for (int j = 0; j < kEt2Rows1 / 4; ++j) {
          const int r = slice + 4 * j;
          if (r < rows) et2_row<NP>(wrow[r * (kD / 4)], reinterpret_cast<const float4*>(s_x + (r0 + r) * NC), acc);
        }
        __syncwarp();
        if (lane == 0) mbarrier_arrive(bar_empty + 8 * slot);
        if (++slot == kSlots) slot = 0, phase ^= 1;
      }
      float* dst = s_part + (size_t)slice * NC * kD + 4 * fl;
#pragma unroll
      for (int c = 0; c < NP; ++c) {
        *reinterpret_cast<float4*>(dst + (2 * c) * kD) = make_float4(acc[0][c].x, acc[1][c].x, acc[2][c].x, acc[3][c].x);
        *reinterpret_cast<float4*>(dst + (2 * c + 1) * kD) = make_float4(acc[0][c].y, acc[1][c].y, acc[2][c].y, acc[3][c].y);
      }
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    // ---- bias, LayerNorm (two passes): a warp takes clips warp, warp + 8; lane: features lane + 32 j
    for (int c = warp; c < NC; c += 8) {
      float z[8];
      float sum = 0.0f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int f = lane + 32 * j;
        float v = s_be1[f];
#pragma unroll
        for (int sl = 0; sl < 4; ++sl) v += s_part[((size_t)sl * NC + c) * kD + f];
        z[j] = v;
        sum += v;
      }
      const float mean = warp_sum(sum) * (1.0f / kD);
      float sq = 0.0f;
#pragma unroll
      for (int j = 0; j < 8; ++j) sq = fmaf(z[j] - mean, z[j] - mean, sq);
      const float rstd = rsqrtf(warp_sum(sq) * (1.0f / kD) + W.ln_eps);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int f = lane + 32 * j;
        s_zn[f * NC + c] = (z[j] - mean) * rstd * s_g[f] + s_b[f];
      }
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    // ---- layer 2: h = we2_t^T zn.  warp = K slice (rows k = warp mod 8); thread: hidden features 4 lane .. 4 lane + 3
    {
#pragma unroll
      for (int f = 0; f < 4; ++f)
#pragma unroll
        for (int c = 0; c < NP; ++c) acc[f][c] = make_float2(0.0f, 0.0f);
      for (int ch = 0; ch < n2; ++ch) {
        mbarrier_wait(bar_full + 8 * slot, phase);
        const float4* wrow = reinterpret_cast<const float4*>(s_ring + slot * kEt2Stage) + lane;
#pragma unroll
        for (int j = 0; j < kEt2Rows2 / 8; ++j) {
          const int r = warp + 8 * j;
          et2_row<NP>(wrow[r * (128 / 4)], reinterpret_cast<const float4*>(s_zn + (ch * kEt2Rows2 + r) * NC), acc);
        }
        __syncwarp();
        if (lane == 0) mbarrier_arrive(bar_empty + 8 * slot);
        if (++slot == kSlots) slot = 0, phase ^= 1;
      }
      float* dst = s_part + (size_t)warp * NC * 128 + 4 * lane;   // [slice 8][clip][128]
#pragma unroll
      for (int c = 0; c < NP; ++c) {
        *reinterpret_cast<float4*>(dst + (2 * c) * 128) = make_float4(acc[0][c].x, acc[1][c].x, acc[2][c].x, acc[3][c].x);
        *reinterpret_cast<float4*>(dst + (2 * c + 1) * 128) = make_float4(acc[0][c].y, acc[1][c].y, acc[2][c].y, acc[3][c].y);
      }
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    // ---- relu, output layer, sigmoid; the clip's expression entries of every output row
    for (int c = warp; c < nc; c += 8) {
      float part = 0.0f;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int j = lane + 32 * q;
        float h = s_be2[j];
#pragma unroll
        for (int sl = 0; sl < 8; ++sl) h += s_part[((size_t)sl * NC + c) * 128 + j];
        part = fmaf(fmaxf(h, 0.0f), s_w2[j], part);
      }
      const float logit = warp_sum(part) + W.b2;
      const float y = 1.0f / (1.0f + expf(-logit));
      if (lane == 0 && expr_sigmoid != nullptr) expr_sigmoid[c0 + c] = y;
      if (out != nullptr && lane < KOE_N_EXPR) {
        const float v = fminf(fmaxf(o_coef * y, 0.0f), 1.0f);
        size_t o = (size_t)(c0 + c) * n_out * KOE_N_BLENDSHAPES + o_idx;
        int rows = n_out;
        if constexpr (kVarlen) {
          const int r0 = __ldg(row_base + c0 + c);
          o = (size_t)r0 * KOE_N_BLENDSHAPES + o_idx;
          rows = __ldg(row_base + c0 + c + 1) - r0;
        }
        for (int wi = 0; wi < rows; ++wi, o += KOE_N_BLENDSHAPES) {
          out[o] = v;
          if (sigmoid_out != nullptr) sigmoid_out[o] = y;
        }
      }
    }
  }
  // the kernel before this one (the frontend) must have completed before this one does: the core, queued next, waits on
  // THIS kernel only
  if (dbg != nullptr && tid == 0) dbg[3 * blockIdx.x + 1] = global_ns();
  pdl_wait();
  if (dbg != nullptr && tid == 0) dbg[3 * blockIdx.x + 2] = global_ns();
}

// ---- EMA scan: y_t = alpha x_t + (1 - alpha) y_{t-1}, warp-parallel over 32 frames per step --------
constexpr int kEmaTile = 32;
constexpr int kEmaStride = KOE_N_BLENDSHAPES + 1;

// one frame per clip (the streaming step): y = alpha x + (1 - alpha) state, or x itself for the first frame -- the same
// roundings as the scan kernel below for n_out == 1
__global__ void __launch_bounds__(256) ema_step_kernel(float* __restrict__ frames, int n, float alpha,
                                                       float* __restrict__ state, int has_state) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const float x = frames[i];
  const float y = (has_state && state != nullptr) ? fmaf(1.0f - alpha, state[i], alpha * x) : x;
  frames[i] = y;
  if (state != nullptr) state[i] = y;
}

// kVarlen: the segmented scan of a packed variable-length batch, clip b's frames are rows [row_base[b], row_base[b + 1])
// (tiles counted from each clip's first frame, as for a clip alone); a separate instantiation
template <bool kVarlen = false>
__global__ void __launch_bounds__(256) ema_scan_kernel(float* __restrict__ frames, int n_out, float alpha,
                                                       float* __restrict__ state, int has_state,
                                                       const int* __restrict__ row_base) {
  __shared__ float s_t[kEmaTile * kEmaStride];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* x = frames + (size_t)b * n_out * KOE_N_BLENDSHAPES;
  if constexpr (kVarlen) {
    x = frames + (size_t)__ldg(row_base + b) * KOE_N_BLENDSHAPES;
    n_out = __ldg(row_base + b + 1) - __ldg(row_base + b);
  }
  const float a = 1.0f - alpha;
  float apow[5];  // a^1, a^2, a^4, a^8, a^16
  apow[0] = a;
#pragma unroll
  for (int i = 1; i < 5; ++i) apow[i] = apow[i - 1] * apow[i - 1];
  const float a_lane = powf(a, (float)(lane + 1));
  // warp w owns coefficients j = w, w + 8, ...; carry[j-slot] is y_{t0 - 1}
  float carry[7];
#pragma unroll
  for (int s = 0; s < 7; ++s) {
    const int j = warp + 8 * s;
    carry[s] = (has_state && state != nullptr && j < KOE_N_BLENDSHAPES) ? state[(size_t)b * KOE_N_BLENDSHAPES + j] : 0.0f;
  }
  for (int t0 = 0; t0 < n_out; t0 += kEmaTile) {
    const int nt = min(kEmaTile, n_out - t0);
    for (int i = tid; i < nt * KOE_N_BLENDSHAPES; i += 256)
      s_t[(i / KOE_N_BLENDSHAPES) * kEmaStride + i % KOE_N_BLENDSHAPES] = x[(size_t)t0 * KOE_N_BLENDSHAPES + i];
    __syncthreads();
#pragma unroll
    for (int s = 0; s < 7; ++s) {
      const int j = warp + 8 * s;
      if (j < KOE_N_BLENDSHAPES) {
        float c = 0.0f;
        if (lane < nt) {
          const float v = s_t[lane * kEmaStride + j];
          // first frame of a fresh sequence passes through (reference :357-359)
          c = (t0 + lane == 0 && !has_state) ? v : alpha * v;
        }
#pragma unroll
        for (int i = 0; i < 5; ++i) {
          const float up = __shfl_up_sync(kFullMask, c, 1 << i);
          if (lane >= (1 << i)) c = fmaf(apow[i], up, c);
        }
        const float y = fmaf(a_lane, carry[s], c);
        if (lane < nt) s_t[lane * kEmaStride + j] = y;
        carry[s] = __shfl_sync(kFullMask, y, nt - 1);
      }
    }
    __syncthreads();
    for (int i = tid; i < nt * KOE_N_BLENDSHAPES; i += 256)
      x[(size_t)t0 * KOE_N_BLENDSHAPES + i] = s_t[(i / KOE_N_BLENDSHAPES) * kEmaStride + i % KOE_N_BLENDSHAPES];
    __syncthreads();
  }
  if (state != nullptr && lane == 0) {
#pragma unroll
    for (int s = 0; s < 7; ++s) {
      const int j = warp + 8 * s;
      if (j < KOE_N_BLENDSHAPES) state[(size_t)b * KOE_N_BLENDSHAPES + j] = carry[s];
    }
  }
}

int launch_dual_stream_tc(const CoreParams& p, CoreMode mode, cudaStream_t stream);  // dual_stream_tc.cu

}  // namespace koe

using namespace koe;

static int validate_weights(const koe_core_weights* w) {
  KOE_REQUIRE(w != nullptr, "koe_core_weights is NULL");
  KOE_REQUIRE(w->wc_t && w->bc && w->ln_g && w->ln_b && w->qk_t && w->wv_t && w->bv && w->wa_t && w->ba && w->w2 &&
                  w->coef && w->mouth_idx && w->expr_idx && w->we1_t && w->be1 && w->eln_g && w->eln_b && w->we2_t &&
                  w->be2,
              "koe_core_weights has a NULL field");
  KOE_REQUIRE(w->k_mel >= 4 && w->k_mel <= 4096 && w->k_mel_pad >= w->k_mel && w->k_mel_pad % 16 == 0,
              "koe_core_weights: bad k_mel/k_mel_pad");
  KOE_REQUIRE(w->emo_in > 0 && w->emo_in <= kEmoInMax && w->emo_in_pad >= w->emo_in, "koe_core_weights: bad emo_in");
  return KOE_OK;
}

static long long* g_tc_debug = nullptr;  // (koe_debug_set_tc_timestamps below)

// One launcher for the public entry (expr_sigmoid only, plain stream order: the producer of emo_in may be the kernel
// queued just before) and the fused forward (`after_frontend`: the caller guarantees that the kernel queued just before
// this one is the log-mel frontend, which writes nothing this kernel reads -- only then may it start beside that kernel's
// last CTAs; `out` != NULL: the expression entries of the n_out output rows of every clip are written here).
int koe::launch_emotion_stream(const koe_core_weights* w, const float* emo_in, int n_clips, float* expr_sigmoid, float* out,
                               float* sigmoid_out, int n_out, void* stream, bool after_frontend, const int* row_base) {
  if (int rc = validate_weights(w)) return rc;
  KOE_REQUIRE(n_clips >= 0 && n_out >= 1, "koe_emotion_stream: bad size");
  if (n_clips == 0) return KOE_OK;  // nothing to do: empty buffers may be NULL
  KOE_REQUIRE(emo_in != nullptr && (expr_sigmoid != nullptr || out != nullptr), "koe_emotion_stream: NULL argument");
  KOE_REQUIRE(w->emo_in_pad % 8 == 0 && w->emo_in_pad <= kEmoInMax, "koe_emotion_stream: emo_in_pad must be a multiple of 8");
  KOE_REQUIRE(((reinterpret_cast<uintptr_t>(w->we1_t) | reinterpret_cast<uintptr_t>(w->we2_t)) & 15) == 0,
              "koe_emotion_stream: weights must be 16-byte aligned");
  static bool configured[64] = {false};
  int dev = 0;
  KOE_CUDA(cudaGetDevice(&dev));
  KOE_REQUIRE(dev >= 0 && dev < 64, "device index too large");
  if (!configured[dev]) {
    KOE_CUDA(cudaFuncSetAttribute(emotion_tiled_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Et2<8>::kSmem));
    KOE_CUDA(cudaFuncSetAttribute(emotion_tiled_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Et2<16>::kSmem));
    KOE_CUDA(cudaFuncSetAttribute(emotion_tiled_kernel<8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)Et2<8>::kSmem));
    KOE_CUDA(cudaFuncSetAttribute(emotion_tiled_kernel<16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)Et2<16>::kSmem));
    configured[dev] = true;
  }
  // every CTA streams all the weights (0.4 MB).  Eight clips per CTA: 64 CTAs of ~9 us for 512 clips, which start on the
  // SMs the frontend's earliest CTAs leave and are done about when its last CTA is (step 207.9 -> 198.9 us against the
  // round-1 kernel, 4 clips per CTA and cp.async staging; sixteen clips per CTA, 32 CTAs of ~15 us: 204.6 us).  Sixteen only
  // where the weight traffic of eight would show (thousands of CTAs).
  const bool wide = n_clips > 2048;
  const dim3 grid(wide ? (n_clips + 15) / 16 : (n_clips + 7) / 8), block(kEt2Threads);
  const size_t smem = wide ? Et2<16>::kSmem : Et2<8>::kSmem;
  KOE_REQUIRE(row_base == nullptr || out != nullptr, "koe_emotion_stream: row_base without out");
  auto kernel = row_base != nullptr ? (wide ? emotion_tiled_kernel<16, true> : emotion_tiled_kernel<8, true>)
                                    : (wide ? emotion_tiled_kernel<16> : emotion_tiled_kernel<8>);
  long long* dbg = after_frontend && g_tc_debug != nullptr ? g_tc_debug + 128 + 2 * 148 : nullptr;
  if (after_frontend) {
    KOE_CUDA(launch_after_primary_starts(kernel, grid, block, smem, (cudaStream_t)stream, *w, emo_in, n_clips, expr_sigmoid, out,
                                         sigmoid_out, n_out, dbg, row_base));
  } else {
    kernel<<<grid, block, smem, (cudaStream_t)stream>>>(*w, emo_in, n_clips, expr_sigmoid, out, sigmoid_out, n_out, dbg,
                                                        row_base);
    KOE_CUDA(cudaGetLastError());
  }
  count_launch();
  return KOE_OK;
}

extern "C" int koe_emotion_stream(const koe_core_weights* w, const float* emo_in, int n_clips, float* expr_sigmoid,
                                  void* stream) {
  return koe::launch_emotion_stream(w, emo_in, n_clips, expr_sigmoid, nullptr, nullptr, 1, stream, /*after_frontend=*/false);
}

// ---- y = x W^T + b for a handful of rows: the 264 -> 256 eGeMAPS compression as a stand-alone call
// (OpenSMILEeGeMAPSExtractor.get_concatenated_features, src/features/opensmile_extractor.py:583-604; the batch path folds
// this layer into the emotion stream instead)
namespace koe {
__global__ void __launch_bounds__(256) affine_rows_kernel(const float* __restrict__ x, int n_in,
                                                          const float* __restrict__ w_t, const float* __restrict__ b,
                                                          int n_out, float* __restrict__ y) {
  extern __shared__ float s_x[];
  const int r = blockIdx.x;
  for (int i = threadIdx.x; i < n_in; i += blockDim.x) s_x[i] = x[(long long)r * n_in + i];
  __syncthreads();
  for (int o = threadIdx.x; o < n_out; o += blockDim.x) {
    float acc = 0.0f;
    for (int i = 0; i < n_in; ++i) acc = fmaf(s_x[i], w_t[(long long)i * n_out + o], acc);
    y[(long long)r * n_out + o] = acc + b[o];
  }
}
}  // namespace koe

extern "C" int koe_affine_rows(const float* x, int n_rows, int n_in, const float* w_t, const float* b, int n_out, float* y,
                               void* stream) {
  KOE_REQUIRE(n_rows >= 0 && n_in > 0 && n_in <= 8192 && n_out > 0, "koe_affine_rows: bad sizes");
  if (n_rows == 0) return KOE_OK;
  KOE_REQUIRE(x && w_t && b && y, "koe_affine_rows: NULL argument");
  koe::affine_rows_kernel<<<n_rows, 256, n_in * sizeof(float), (cudaStream_t)stream>>>(x, n_in, w_t, b, n_out, y);
  count_launch();
  KOE_CUDA(cudaGetLastError());
  return KOE_OK;
}

// bring-up / profiling hook (not in the public header; scripts/tc_timeline.py): a device buffer of 128 + 2 * gridDim
// 64-bit slots that the tensor-core kernel fills with phase timestamps of CTA 0 (clock64) and every CTA's start / end
// (globaltimer); NULL (the default) turns the stamps off
extern "C" void koe_debug_set_tc_timestamps(long long* device_buffer) { g_tc_debug = device_buffer; }

// sets the shared-memory size of the instantiation once per device, then launches it
template <CoreMode M>
static int launch_fp32(const CoreParams& p, cudaStream_t stream) {
  static bool configured[64] = {false};
  int dev = 0, sms = 0;
  KOE_CUDA(cudaGetDevice(&dev));
  KOE_REQUIRE(dev >= 0 && dev < 64, "device index too large");
  if (!configured[dev]) {
    KOE_CUDA(cudaFuncSetAttribute(dual_stream_fp32_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCoreSmem));
    configured[dev] = true;
  }
  KOE_CUDA(sm_count(&sms));
  dual_stream_fp32_kernel<M><<<std::min(p.n_clips * p.n_out, sms), kCoreThreads, kCoreSmem, stream>>>(p);
  count_launch();
  KOE_CUDA(cudaGetLastError());
  return KOE_OK;
}

static int launch_core(const CoreParams& p_in, CoreMode mode, int precision, cudaStream_t stream) {
  CoreParams p = p_in;
  p.dbg = g_tc_debug;
  if (precision == 2) return launch_dual_stream_tc(p, mode, stream);
  if (precision != 0)
    return fail(KOE_E_INVALID, "precision must be 0 (fp32) or 2 (bf16 operands, tcgen05), got %d", precision);
  switch (mode) {
    case CoreMode::Windows: return launch_fp32<CoreMode::Windows>(p, stream);
    case CoreMode::Pool: return launch_fp32<CoreMode::Pool>(p, stream);
    case CoreMode::Varlen: return launch_fp32<CoreMode::Varlen>(p, stream);
    case CoreMode::PoolHops: return launch_fp32<CoreMode::PoolHops>(p, stream);
    case CoreMode::Early: break;
  }
  return fail(KOE_E_INVALID, "early release needs the tensor-core core (precision 2)");
}

// The part every core entry fills alike: the weights (validated by the caller), the 1 + 2 n_edge mel-power / frame-max
// buffers -- each non-NULL, the power rows 16-byte aligned; power == NULL: none, the prenormalised features -- and the
// outputs; one window per clip, frames 1 apart, unless the entry says otherwise.  `what` names the entry in error messages.
static int core_params(const char* what, const koe_core_weights* w, const float* const* power, const float* const* frame_max,
                       int n_edge, const float* expr_sigmoid, float* out, float* sigmoid_out, float* attn_out,
                       CoreParams* p) {
  *p = CoreParams{};
  p->w = *w;
  for (int j = 0; power != nullptr && j < 1 + 2 * n_edge; ++j) {
    KOE_REQUIRE(power[j] != nullptr && frame_max[j] != nullptr, "%s: NULL power[%d] / frame_max[%d]", what, j, j);
    KOE_REQUIRE((reinterpret_cast<uintptr_t>(power[j]) & 15) == 0, "%s: power[%d] must be 16-byte aligned", what, j);
    p->power[j] = power[j], p->fmax[j] = frame_max[j];
  }
  p->n_edge = n_edge;
  p->n_out = 1;
  p->stride_frames = 1;
  p->mel_seq = w->k_mel - 3;
  p->expr_sigmoid = expr_sigmoid;
  p->out = out;
  p->sigmoid_out = sigmoid_out;
  p->attn_out = attn_out;
  return KOE_OK;
}

extern "C" int koe_dual_stream_windows(const koe_core_weights* w, const float* const* power,
                                       const float* const* frame_max, int n_edge, int n_clips, int n_frames,
                                       int n_out, int stride_frames, int frames_per_window,
                                       const float* expr_sigmoid, float* out, float* sigmoid_out, float* attn_out,
                                       int precision, void* stream) {
  return koe::launch_dual_stream_windows(w, power, frame_max, n_edge, n_clips, n_frames, n_out, stride_frames,
                                         frames_per_window, expr_sigmoid, out, sigmoid_out, attn_out, precision, stream,
                                         /*expr_by_emotion_kernel=*/false);
}

int koe::launch_dual_stream_windows(const koe_core_weights* w, const float* const* power, const float* const* frame_max,
                                    int n_edge, int n_clips, int n_frames, int n_out, int stride_frames,
                                    int frames_per_window, const float* expr_sigmoid, float* out, float* sigmoid_out,
                                    float* attn_out, int precision, void* stream, bool expr_by_emotion_kernel,
                                    unsigned* early_flag, unsigned early_target, int early_items, bool* early_applied) {
  if (early_applied != nullptr) *early_applied = false;
  if (int rc = validate_weights(w)) return rc;
  if (n_clips == 0 || n_out == 0) return KOE_OK;  // nothing to do: empty buffers may be NULL
  KOE_REQUIRE(power != nullptr && frame_max != nullptr && out != nullptr, "koe_dual_stream_windows: NULL argument");
  // the expression entries of `out` come from expr_sigmoid -- or, in the fused forward, from the emotion kernel itself
  KOE_REQUIRE((expr_sigmoid != nullptr) != expr_by_emotion_kernel, "koe_dual_stream_windows: NULL expr_sigmoid");
  KOE_REQUIRE(n_edge >= 0 && n_edge <= KOE_MAX_EDGE, "koe_dual_stream_windows: n_edge out of range");
  KOE_REQUIRE(n_clips >= 0 && n_out >= 0 && stride_frames >= 1 && frames_per_window >= 1,
              "koe_dual_stream_windows: bad sizes");
  KOE_REQUIRE(frames_per_window > 2 * n_edge, "koe_dual_stream_windows: window shorter than its edge frames");
  KOE_REQUIRE(n_out == 0 || (long long)(n_out - 1) * stride_frames + frames_per_window <= n_frames,
              "koe_dual_stream_windows: windows run past n_frames");
  KOE_REQUIRE((long long)n_clips * n_out < (1ll << 31), "koe_dual_stream_windows: too many windows");
  CoreParams p;
  if (int rc = core_params("koe_dual_stream_windows", w, power, frame_max, n_edge, expr_sigmoid, out, sigmoid_out, attn_out,
                           &p))
    return rc;
  p.n_clips = n_clips;
  p.n_frames = n_frames;
  p.n_out = n_out;
  p.stride_frames = stride_frames;
  p.frames_per_window = frames_per_window;
  CoreMode mode = CoreMode::Windows;
  if (early_flag != nullptr && early_target > 0 && early_items > 0 && precision == 2 && n_out == 1 && n_edge == 0 &&
      attn_out == nullptr && (w->k_mel == 259 || w->k_mel == 515)) {
    mode = CoreMode::Early;
    p.early_flag = early_flag;
    p.early_target = early_target;
    p.early_items = early_items;
  }
  const int rc = launch_core(p, mode, precision, (cudaStream_t)stream);
  if (rc == KOE_OK && early_applied != nullptr) *early_applied = mode == CoreMode::Early;
  return rc;
}

extern "C" int koe_dual_stream_ring_edges(const koe_core_weights* w, const float* const* power,
                                          const float* const* frame_max, int n_edge, int n_streams, int ring_frames,
                                          int ring_base, int frames_per_window, const float* expr_sigmoid, float* out,
                                          float* sigmoid_out, float* attn_out, int precision, void* stream) {
  if (int rc = validate_weights(w)) return rc;
  KOE_REQUIRE(power != nullptr && frame_max != nullptr && expr_sigmoid != nullptr && out != nullptr,
              "koe_dual_stream_ring: NULL argument");
  KOE_REQUIRE(n_edge >= 1 && n_edge <= KOE_MAX_EDGE, "koe_dual_stream_ring: n_edge out of range");
  KOE_REQUIRE(n_streams >= 0 && ring_base >= 0 && frames_per_window > 2 * n_edge && ring_frames >= frames_per_window - 1,
              "koe_dual_stream_ring: bad sizes (the ring must hold every plain frame of a window)");
  if (n_streams == 0) return KOE_OK;
  CoreParams p;
  if (int rc = core_params("koe_dual_stream_ring", w, power, frame_max, n_edge, expr_sigmoid, out, sigmoid_out, attn_out, &p))
    return rc;
  p.n_clips = n_streams;
  p.n_frames = ring_frames;
  p.frames_per_window = frames_per_window;
  p.ring_frames = ring_frames;
  p.ring_base = ring_base % ring_frames;
  return launch_core(p, CoreMode::Windows, precision, (cudaStream_t)stream);
}

int koe::launch_dual_stream_pool(const koe_core_weights* w, const float* const* power, const float* const* frame_max,
                                 int n_edge, int n_windows, int ring_frames, const int* slot, const int* base,
                                 const float* expr_sigmoid, float* out, int precision, void* stream) {
  if (int rc = validate_weights(w)) return rc;
  KOE_REQUIRE(power != nullptr && frame_max != nullptr && slot != nullptr && base != nullptr && expr_sigmoid != nullptr &&
                  out != nullptr,
              "stream pool core: NULL argument");
  KOE_REQUIRE(n_edge >= 1 && n_edge <= KOE_MAX_EDGE && n_windows >= 0 && ring_frames == w->k_mel - 3,
              "stream pool core: bad sizes");
  if (n_windows == 0) return KOE_OK;
  CoreParams p;
  if (int rc = core_params("stream pool core", w, power, frame_max, n_edge, expr_sigmoid, out, nullptr, nullptr, &p)) return rc;
  p.n_clips = n_windows;
  p.n_frames = ring_frames;
  p.frames_per_window = ring_frames + 1;
  p.ring_frames = ring_frames;
  p.pool_slot = slot;
  p.pool_base = base;
  return launch_core(p, CoreMode::Pool, precision, (cudaStream_t)stream);
}

int koe::launch_dual_stream_pool_hops(const koe_core_weights* w, const float* const* power, const float* const* frame_max,
                                      int n_edge, int n_windows, int ring_frames, const int* hop_end, const int* hop_slot,
                                      const int* hop_row, int hop_base_shift, const int* hop_frames,
                                      const float* expr_sigmoid, float* out, int precision, void* stream) {
  if (int rc = validate_weights(w)) return rc;
  KOE_REQUIRE(power != nullptr && frame_max != nullptr && hop_end != nullptr && hop_slot != nullptr && hop_row != nullptr &&
                  expr_sigmoid != nullptr && out != nullptr,
              "stream pool burst core: NULL argument");
  KOE_REQUIRE(n_edge >= 1 && n_edge <= KOE_MAX_EDGE && n_windows >= 0 && ring_frames >= w->k_mel - 3 &&
                  hop_base_shift >= 0 && hop_base_shift < ring_frames,
              "stream pool burst core: bad sizes");
  if (n_windows == 0) return KOE_OK;
  CoreParams p;
  if (int rc = core_params("stream pool burst core", w, power, frame_max, n_edge, expr_sigmoid, out, nullptr, nullptr, &p))
    return rc;
  p.n_clips = n_windows;
  p.n_frames = ring_frames;
  p.frames_per_window = w->k_mel - 2;
  p.ring_frames = ring_frames;
  p.hop_end = hop_end;
  p.hop_slot = hop_slot;
  p.hop_row = hop_row;
  p.hop_base_shift = hop_base_shift;
  p.hop_frames = hop_frames;
  return launch_core(p, CoreMode::PoolHops, precision, (cudaStream_t)stream);
}

int koe::launch_dual_stream_varlen(const koe_core_weights* w, const float* const* power, const float* const* frame_max,
                                   int n_edge, int n_rows, int n_frames, int stride_frames, int frames_per_window,
                                   int n_clips, const int* row_base, const int* frame_base, const int* edge_base,
                                   const int* lead_base, const int* plain_only, float* out, float* sigmoid_out,
                                   float* attn_out, int precision, void* stream) {
  if (int rc = validate_weights(w)) return rc;
  KOE_REQUIRE(power != nullptr && frame_max != nullptr && row_base != nullptr && frame_base != nullptr &&
                  edge_base != nullptr && plain_only != nullptr && out != nullptr,
              "varlen core: NULL argument");
  KOE_REQUIRE(n_edge >= 0 && n_edge <= KOE_MAX_EDGE && n_rows >= 0 && n_clips >= 0 && stride_frames >= 1 &&
                  frames_per_window > 2 * n_edge && frames_per_window == w->k_mel - 2,
              "varlen core: bad sizes");
  if (n_rows == 0) return KOE_OK;
  CoreParams p;
  if (int rc = core_params("varlen core", w, power, frame_max, n_edge, nullptr, out, sigmoid_out, attn_out, &p)) return rc;
  p.n_clips = n_rows;
  p.n_frames = n_frames;
  p.stride_frames = stride_frames;
  p.frames_per_window = frames_per_window;
  p.vl_row_base = row_base;
  p.vl_frame_base = frame_base;
  p.vl_plain_only = plain_only;
  p.vl_clips = n_clips;
  p.vl_edge_base = edge_base;
  p.vl_lead_base = lead_base;
  return launch_core(p, CoreMode::Varlen, precision, (cudaStream_t)stream);
}

int koe::launch_ema_scan_varlen(float* frames, int n_clips, const int* row_base, float alpha, void* stream) {
  KOE_REQUIRE(frames != nullptr && row_base != nullptr && n_clips >= 0, "varlen smoothing: bad argument");
  KOE_REQUIRE(alpha >= 0.0f && alpha <= 1.0f, "koe_ema_scan: alpha must be in [0, 1]");
  if (n_clips == 0) return KOE_OK;
  ema_scan_kernel<true><<<n_clips, 256, 0, (cudaStream_t)stream>>>(frames, 0, alpha, nullptr, 0, row_base);
  count_launch();
  KOE_CUDA(cudaGetLastError());
  return KOE_OK;
}

extern "C" int koe_dual_stream_ring(const koe_core_weights* w, const float* power_ring, const float* fmax_ring,
                                    const float* power_lo_ring, const float* fmax_lo_ring, const float* power_hi,
                                    const float* fmax_hi, int n_streams, int ring_frames, int ring_base,
                                    int frames_per_window, const float* expr_sigmoid, float* out, float* sigmoid_out,
                                    float* attn_out, int precision, void* stream) {
  const float* power[3] = {power_ring, power_lo_ring, power_hi};
  const float* fmax[3] = {fmax_ring, fmax_lo_ring, fmax_hi};
  return koe_dual_stream_ring_edges(w, power, fmax, 1, n_streams, ring_frames, ring_base, frames_per_window, expr_sigmoid,
                                    out, sigmoid_out, attn_out, precision, stream);
}

extern "C" int koe_dual_stream_features(const koe_core_weights* w, const float* mel_long, int n_long,
                                        const float* mel_short, int n_clips, const float* expr_sigmoid, float* out,
                                        float* sigmoid_out, float* attn_out, int precision, void* stream) {
  if (int rc = validate_weights(w)) return rc;
  KOE_REQUIRE(n_clips >= 0 && n_long >= 0, "koe_dual_stream_features: bad sizes");
  if (n_clips == 0) return KOE_OK;  // nothing to do: empty buffers may be NULL
  KOE_REQUIRE(mel_long != nullptr && mel_short != nullptr && expr_sigmoid != nullptr && out != nullptr,
              "koe_dual_stream_features: NULL argument");
  KOE_REQUIRE(((reinterpret_cast<uintptr_t>(mel_long) | reinterpret_cast<uintptr_t>(mel_short)) & 15) == 0,
              "koe_dual_stream_features: features must be 16-byte aligned");
  CoreParams p;
  if (int rc = core_params("koe_dual_stream_features", w, nullptr, nullptr, 0, expr_sigmoid, out, sigmoid_out, attn_out, &p))
    return rc;
  p.n_clips = n_clips;
  p.frames_per_window = 1;
  p.mel_long = mel_long;
  p.mel_short = mel_short;
  p.n_long = n_long < p.mel_seq ? n_long : p.mel_seq;
  // rows of a longer mel_long are still addressed with its true length
  p.n_frames = n_long;
  return launch_core(p, CoreMode::Windows, precision, (cudaStream_t)stream);
}

extern "C" int koe_ema_scan(float* frames, int n_clips, int n_out, float alpha, float* state, int has_state,
                            void* stream) {
  KOE_REQUIRE(frames != nullptr && n_clips >= 0 && n_out >= 0, "koe_ema_scan: bad argument");
  KOE_REQUIRE(alpha >= 0.0f && alpha <= 1.0f, "koe_ema_scan: alpha must be in [0, 1]");
  KOE_REQUIRE(!has_state || state != nullptr, "koe_ema_scan: has_state set but state is NULL");
  if (n_clips == 0 || n_out == 0) return KOE_OK;
  if (n_out == 1)
    ema_step_kernel<<<(n_clips * KOE_N_BLENDSHAPES + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        frames, n_clips * KOE_N_BLENDSHAPES, alpha, state, has_state);
  else
    ema_scan_kernel<<<n_clips, 256, 0, (cudaStream_t)stream>>>(frames, n_out, alpha, state, has_state, nullptr);
  count_launch();
  KOE_CUDA(cudaGetLastError());
  return KOE_OK;
}
