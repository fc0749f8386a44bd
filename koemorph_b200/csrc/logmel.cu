// Log-mel frontend for sm_100a: framing + periodic Hann + 1024-point FFT + |X|^2 + sparse Slaney
// filterbank, fused in one kernel; then a small dB-normalisation kernel.
//
// Replaces the per-clip librosa loop of SimplifiedDualStreamModel.extract_mel_features
// (reference src/model/simplified_dual_stream_model.py:184-229).
//
// Kernel design (see DESIGN.md section "K1"):
//   * one warp transforms TWO real frames of the same clip at once as one complex 1024-point FFT
//     (z = a + i b), decomposed 32 x 32: radix-2 DIT FFT of 32 points in registers, twiddle, 32x32 transpose
//     through a padded shared-memory tile, second 32-point FFT in registers.  Every complex value is one
//     64-bit register pair and every butterfly is written with the packed fp32x2 instructions of sm_100
//     (FADD2 / FMUL2 / FFMA2, whose operands take per-half negation and a half swap, so "times -i" is free
//     and a butterfly with a general twiddle is 3 instructions: x = a + w b as two FFMA2, y = 2a - x as one).
//   * after the second pass lane l holds Z[l + 32 r]; the conjugate-symmetric partner Z[1024 - k] lives in lane
//     (32 - l) & 31, so the two real spectra are separated with 32 warp shuffles and no further shared-memory
//     round trip; the pair (|A_k|^2, |B_k|^2) comes out of one FMUL2 + one FFMA2.
//   * 16 warps transform 16 pairs per iteration -> 32 power spectra, parked in the warps' transposition tiles with
//     bank-skewed bases.  The Slaney filterbank is then applied with lane = frame: the 506 weighted bins are split into
//     16 runs, every weight / bin index is a broadcast, every spectrum read is conflict-free and the control flow is
//     warp-uniform.  Results leave through a shared staging tile as coalesced rows of 80 mel values in dB.
//   * two organisations of that iteration (bit-identical results):
//       logmel_power_ws_kernel   the default bank's batch launches: 16 PRODUCER warps (loads, FFT, spectra) and 8 CONSUMER
//                                warps (mel phase, store phase) joined by mbarriers, registers split with setmaxnreg
//       logmel_power_kernel      16 identical warps with one __syncthreads and one mbarrier per iteration and a store phase
//                                staggered by warp class (generic banks, 512-point flavours, the streaming step's split output)
//   * frame pairs that touch the padding / a window edge / the end of the clip take masked or reflected loads and are
//     grouped by the launch order into iterations of their own: a masked pair costs its warp ~25 % more instructions.
//   * the default bank (sr 16000, 80 mels, 80..8000 Hz) runs the filterbank as straight-line FFMAs with immediate
//     weights unrolled from compile-time tables (melbank_default.inc); any other bank takes the looped variant.
#include <algorithm>
#include <cmath>
#include <mutex>
#include <type_traits>
#include <vector>

#include "common.cuh"

namespace koe {

constexpr int kFrameLen = 1024;
constexpr int kBins = 513;
constexpr int kWarps = 16;
constexpr int kThreads = kWarps * 32;
constexpr int kSlots = 2 * kWarps;      // frames per CTA iteration (= 32: one per lane in the filterbank phase)
constexpr int kRowF2 = 33;              // float2 per row of the transposition tile (padded: conflict-free both ways)
constexpr int kScratch = 2120;          // floats per warp tile: >= 2 * 32 * 33, == 8 (mod 32)
constexpr int kSecondFrame = 516;       // offset of the warp's second spectrum, == 4 (mod 32): with lane = frame the
                                        // bases of 8 consecutive frames are 16 bytes apart mod 128 -> LDS.128 conflict-free
constexpr int kMaxBins = 512;           // spectrum bins that carry filterbank weight (507 for 80..8000 Hz)
constexpr int kMaxGroups = 96;          // groups of consecutive bins feeding the same pair of adjacent filters
constexpr int kTileStride = 81;         // mel staging row stride (floats), odd: conflict-free across frames

struct FrontendTables {
  const float* hann;     // [1024]
  const float2* tw;      // [32][32] W_1024^(k1*n2)
  // Slaney filterbank, bin-major: a spectrum bin feeds at most two ADJACENT filters (fl, fl + 1)
  const float2* binw;    // [n_bins] 0.25 * (weight into filter fl, weight into filter fl + 1)
  const int4* groups;    // [n_groups] {first bin k, first entry of binw, number of bins, fl}: fl rises by one per group
  const int* runs;       // [kWarps + 1] group range of every warp in the filterbank phase
  int n_bins, n_groups;
  int log_mode;          // 0: 10 log10(max(p, 1e-10)) (librosa power_to_db, first term); 1: ln(p + log_eps) (stft.py:124)
  float log_eps;
};

struct LogmelParams {
  const float* audio;
  int64_t audio_stride;
  int n_clips, n_samples, hop, n_frames;
  int lo_rel, hi_rel;
  int frame_offset, frame_step;  // output row j is the frame centred on sample_offset + (frame_offset + j*frame_step)*hop
  int sample_offset;
  int pad_mode;                  // 0: samples outside the clip are zero; 1: reflected (numpy "reflect")
  float* power;
  float* frame_max;
  long long power_clip_stride, fmax_clip_stride;  // elements between consecutive clips' output blocks
  float* power_b;                // optional: odd frames 2j+1 go to power_b[clip][j] / frame_max_b[clip][j] instead
  float* frame_max_b;
  long long power_b_clip_stride, fmax_b_clip_stride;
  int edge_lo, edge_hi;          // leading / trailing frame pairs of a clip that need masked loads (launch order only)
  int mid_pairs;                 // interior pairs per clip (0: no edge grouping, every pair is located the slow way)
  int step_clips, step_pairs;    // gridDim.x * kWarps pairs, as whole clips of mid_pairs + a remainder
  int wait_at_end;               // launch chaining: this launch follows another frontend launch of the same forward (below)
  // early release of the core (csrc/session.cu): every consumer warp adds one to *early_flag (release) when its CTA has
  // stored the rows of all its iterations below early_iters -- the core's first rounds of windows need no more than that
  unsigned* early_flag;
  unsigned early_iters;
  // packed variable-length batch (FrontendMode::Varlen, VarlenLocator only): pair k of the launch is pair
  // k - vl_pair_base[c] of clip c, vl_length[c] samples at audio + vl_sample_off[c], rows vl_row_base[c] ..
  // vl_row_base[c + 1] - 1; n_clips / n_samples / n_frames / the clip strides are not used
  const long long* vl_sample_off;
  const int* vl_length;
  const int* vl_pair_base;
  const int* vl_row_base;
  int vl_clips;
  unsigned vl_pairs;
};

__host__ __device__ constexpr int bitrev5(int i) {
  return ((i & 1) << 4) | ((i & 2) << 2) | (i & 4) | ((i & 8) >> 2) | ((i & 16) >> 4);
}

// cos(2*pi*t/32) for t = 0..15 as literals so the unrolled butterflies use immediates
__device__ __forceinline__ float cos32(int t) {
  switch (t) {
    case 0: return 1.0f;
    case 1: return 0.98078528040323043f;
    case 2: return 0.92387953251128674f;
    case 3: return 0.83146961230254524f;
    case 4: return 0.70710678118654752f;
    case 5: return 0.55557023301960218f;
    case 6: return 0.38268343236508978f;
    case 7: return 0.19509032201612825f;
    case 8: return 0.0f;
    case 9: return -0.19509032201612825f;
    case 10: return -0.38268343236508978f;
    case 11: return -0.55557023301960218f;
    case 12: return -0.70710678118654752f;
    case 13: return -0.83146961230254524f;
    case 14: return -0.92387953251128674f;
    default: return -0.98078528040323043f;
  }
}

// ---- complex arithmetic on (re, im) register pairs with the packed fp32x2 pipe ----------------------------------
__device__ __forceinline__ float2 bcast(float s) { return make_float2(s, s); }
// a + w*b and a - w*b for a compile-time twiddle w = W_32^t = cos(2 pi t/32) - i sin(2 pi t/32)
__device__ __forceinline__ void butterfly(int t, float2& a, float2& b) {
  if (t == 0) {
    const float2 x = __fadd2_rn(a, b);
    b = __fadd2_rn(a, make_float2(-b.x, -b.y));
    a = x;
  } else if (t == 8) {  // w = -i: w*b = (b.y, -b.x)
    const float2 x = __fadd2_rn(a, make_float2(b.y, -b.x));
    b = __fadd2_rn(a, make_float2(-b.y, b.x));
    a = x;
  } else {
    const float wr = cos32(t);
    const float ws = cos32(t > 8 ? t - 8 : 8 - t);  // sin(2 pi t/32)
    // w*b = (wr b.x + ws b.y, wr b.y - ws b.x)
    float2 x = __ffma2_rn(b, bcast(wr), a);
    x = __ffma2_rn(make_float2(b.y, -b.x), bcast(ws), x);
    b = __ffma2_rn(a, bcast(2.0f), make_float2(-x.x, -x.y));
    a = x;
  }
}

// In-register radix-2 decimation-in-time FFT of 32 complex values (forward, e^{-i...}).
// On entry element i holds x[bitrev5(i)]; on return element k holds X[k].
__device__ __forceinline__ void fft32(float2 (&v)[32]) {
#pragma unroll
  for (int h = 1; h <= 16; h <<= 1) {
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      if ((i & h) == 0) butterfly((i & (h - 1)) * (16 / h), v[i], v[i + h]);
    }
  }
}

// Where a frame pair lives: clip, first frame (< 0: no pair), first sample of both frames, valid sample ranges.
__host__ __device__ __forceinline__ int imax(int a, int b) { return a > b ? a : b; }
__host__ __device__ __forceinline__ int imin(int a, int b) { return a < b ? a : b; }

struct PairInfo {
  int clip, frame;
  int fa_lo, fb_lo;            // first sample of frame A / frame B (may be negative)
  int lo_a, hi_a, lo_b, hi_b;  // samples outside [lo, hi) read as zero (or are reflected, pad_mode 1)
  bool interior, has_b;
};

// geometry of frame pair j (frames 2j, 2j + 1) of clip b
__host__ __device__ __forceinline__ PairInfo pair_geometry(const LogmelParams& p, int b, int j) {
  PairInfo pi;
  const int ga = 2 * j;
  pi.clip = b;
  pi.frame = ga;
  pi.has_b = ga + 1 < p.n_frames;
  const int fa = p.frame_offset + ga * p.frame_step, fb = fa + p.frame_step;  // frame indices in hops
  pi.lo_a = 0, pi.hi_a = p.n_samples, pi.lo_b = 0, pi.hi_b = p.n_samples;
  if (p.lo_rel != KOE_NO_EDGE) {
    pi.lo_a = imax(pi.lo_a, p.sample_offset + (fa + p.lo_rel) * p.hop);
    pi.lo_b = imax(pi.lo_b, p.sample_offset + (fb + p.lo_rel) * p.hop);
  }
  if (p.hi_rel != KOE_NO_EDGE) {
    pi.hi_a = imin(pi.hi_a, p.sample_offset + (fa + p.hi_rel) * p.hop);
    pi.hi_b = imin(pi.hi_b, p.sample_offset + (fb + p.hi_rel) * p.hop);
  }
  if (!pi.has_b) pi.hi_b = pi.lo_b;  // empty range: second frame reads as silence
  pi.fa_lo = p.sample_offset + fa * p.hop - kFrameLen / 2;
  pi.fb_lo = p.sample_offset + fb * p.hop - kFrameLen / 2;
  pi.interior = pi.fa_lo >= pi.lo_a && pi.fa_lo + kFrameLen <= pi.hi_a && pi.fb_lo >= pi.lo_b &&
                pi.fb_lo + kFrameLen <= pi.hi_b;
  return pi;
}

// Launch order of the pairs: every clip's leading edge pairs, then every clip's trailing edge pairs, then the interior ones
// clip by clip.  Edge pairs are the ones that touch the padding, a window edge or the end of the clip and take the masked
// loads (~25 % more instructions for that warp); grouped, they fill whole 16-warp iterations instead of holding 15
// interior warps at the barrier in every few iterations.  edge_lo / edge_hi are counted on the host (same geometry).
__device__ __forceinline__ PairInfo locate_pair(const LogmelParams& p, unsigned pair, unsigned total_pairs, unsigned ppc) {
  if (pair >= total_pairs) {
    PairInfo pi;
    pi.clip = 0;
    pi.frame = -1;
    pi.interior = false;
    return pi;
  }
  const unsigned mid = ppc - (unsigned)(p.edge_lo + p.edge_hi);
  const unsigned n_lo = (unsigned)p.n_clips * (unsigned)p.edge_lo, n_hi = (unsigned)p.n_clips * (unsigned)p.edge_hi;
  int b, j;
  if (p.edge_lo + p.edge_hi == 0 || (unsigned)(p.edge_lo + p.edge_hi) >= ppc) {
    b = (int)(pair / ppc);
    j = (int)(pair - (unsigned)b * ppc);
  } else if (pair < n_lo) {
    b = (int)(pair / (unsigned)p.edge_lo);
    j = (int)(pair - (unsigned)b * (unsigned)p.edge_lo);
  } else if (pair < n_lo + n_hi) {
    const unsigned r = pair - n_lo;
    b = (int)(r / (unsigned)p.edge_hi);
    j = (int)(ppc - (unsigned)p.edge_hi + (r - (unsigned)b * (unsigned)p.edge_hi));
  } else {
    const unsigned r = pair - n_lo - n_hi;
    b = (int)(r / mid);
    j = p.edge_lo + (int)(r - (unsigned)b * mid);
  }
  return pair_geometry(p, b, j);
}

// interior frames (all but the first / last of a clip): no masking.  v[bitrev5(n1)] = (a[32 n1 + lane], b[32 n1 + lane])
__device__ __forceinline__ void load_interior(const LogmelParams& p, const PairInfo& pi, int lane, float2 (&v)[32]) {
  const float* clip = p.audio + (long long)pi.clip * p.audio_stride;
  const float* __restrict__ pa = clip + pi.fa_lo + lane;
  const float* __restrict__ pb = clip + pi.fb_lo + lane;
#pragma unroll
  for (int n1 = 0; n1 < 32; ++n1) v[bitrev5(n1)] = make_float2(__ldcs(pa + 32 * n1), __ldcs(pb + 32 * n1));  // streaming: evict-first in L2
}

// frames that touch a clip / window edge (~2 pairs per clip): masked or reflected samples, loaded into the same registers
// one iteration ahead like the interior ones (an edge pair that fetched its samples at the start of its own transform held
// the other 15 warps of the iteration at the barrier for the length of 32 dependent global loads)
__device__ __forceinline__ void load_edge(const LogmelParams& p, const PairInfo& pi, int lane, float2 (&v)[32]) {
  const float* __restrict__ clip = p.audio + (long long)pi.clip * p.audio_stride;
  const int last = p.n_samples - 1;
  const bool reflect = p.pad_mode == 1;  // numpy "reflect" padding about the first / last sample (MelSlidingWindowExtractor default)
  const bool b_on = pi.hi_b > pi.lo_b;
  const int sa0 = pi.fa_lo + lane, sb0 = pi.fb_lo + lane;
#pragma unroll
  for (int n1 = 0; n1 < 32; ++n1) {
    int sa = sa0 + 32 * n1, sb = sb0 + 32 * n1;
    bool oka, okb;
    if (reflect) {
      sa = sa < 0 ? -sa : (sa > last ? 2 * last - sa : sa);
      sb = sb < 0 ? -sb : (sb > last ? 2 * last - sb : sb);
      oka = sa >= 0 && sa <= last;
      okb = b_on && sb >= 0 && sb <= last;
    } else {
      oka = sa >= pi.lo_a && sa < pi.hi_a;
      okb = sb >= pi.lo_b && sb < pi.hi_b;
    }
    v[bitrev5(n1)] = make_float2(oka ? __ldcs(clip + sa) : 0.0f, okb ? __ldcs(clip + sb) : 0.0f);
  }
}

__device__ __forceinline__ float ln_from_power(float p, float eps) { return 0.69314718055994531f * __log2f(p + eps); }
__device__ __forceinline__ float db_from_power(float p) {
  // 10 log10(max(p, amin)) = (10 log10 2) * log2(.): the argument is a normal number, MUFU.LG2 is within 2 ulp
  return 3.0102999566398120f * __log2f(fmaxf(p, kAmin));
}
// order-preserving map float -> int32, so that a warp maximum is one REDUX
__device__ __forceinline__ int float_order(float f) {
  const int i = __float_as_int(f);
  return i ^ ((i >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float order_float(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7fffffff)); }

// ---- filterbank phase, default bank: straight-line code from the compile-time tables ------------------------------
#include "melbank_default.inc"
// Bins [b0, b1) of run W for one spectrum (lane = frame): every bin feeds the falling half of filter g (-> tlo[g]) and
// the rising half of filter g + 1 (-> thi[g + 1]) with immediate weights (kDefBinWDev folds away after unrolling); two
// accumulator pairs alternate so that the FFMA chains are half as long.
template <int W>
__device__ __forceinline__ void mel_run_default(const float* __restrict__ spec, float* __restrict__ tlo,
                                                float* __restrict__ thi) {
  constexpr int b0 = kDefRunBinDev[W], b1 = kDefRunBinDev[W + 1];
  if (b0 >= b1) return;
  float lo0 = 0.0f, lo1 = 0.0f, hi0 = 0.0f, hi1 = 0.0f;
#pragma unroll
  for (int k4 = (b0 & ~3); k4 < b1; k4 += 4) {
    const float4 x4 = *reinterpret_cast<const float4*>(spec + k4);
    const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k4 + j;
      if (k >= b0 && k < b1) {
        if (k > b0 && kDefBinGroupDev[k] != kDefBinGroupDev[k - 1]) {  // next interval: retire the falling / rising halves
          tlo[kDefBinGroupDev[k - 1]] = lo0 + lo1;
          thi[kDefBinGroupDev[k - 1] + 1] = hi0 + hi1;
          lo0 = lo1 = hi0 = hi1 = 0.0f;
        }
        const float wl = kDefBinWDev[2 * (k - kDefFirstBin)], wh = kDefBinWDev[2 * (k - kDefFirstBin) + 1];
        if (k & 1) {
          lo1 = fmaf(wl, xs[j], lo1);
          hi1 = fmaf(wh, xs[j], hi1);
        } else {
          lo0 = fmaf(wl, xs[j], lo0);
          hi0 = fmaf(wh, xs[j], hi0);
        }
      }
    }
  }
  tlo[kDefBinGroupDev[b1 - 1]] = lo0 + lo1;
  thi[kDefBinGroupDev[b1 - 1] + 1] = hi0 + hi1;  // the rising half of "filter 80" lands in the spare column of the tile
}

__device__ __forceinline__ void mel_phase_default(int warp, const float* spec, float* tlo, float* thi) {
  switch (warp) {
    case 0: mel_run_default<0>(spec, tlo, thi); break;
    case 1: mel_run_default<1>(spec, tlo, thi); break;
    case 2: mel_run_default<2>(spec, tlo, thi); break;
    case 3: mel_run_default<3>(spec, tlo, thi); break;
    case 4: mel_run_default<4>(spec, tlo, thi); break;
    case 5: mel_run_default<5>(spec, tlo, thi); break;
    case 6: mel_run_default<6>(spec, tlo, thi); break;
    case 7: mel_run_default<7>(spec, tlo, thi); break;
    case 8: mel_run_default<8>(spec, tlo, thi); break;
    case 9: mel_run_default<9>(spec, tlo, thi); break;
    case 10: mel_run_default<10>(spec, tlo, thi); break;
    case 11: mel_run_default<11>(spec, tlo, thi); break;
    case 12: mel_run_default<12>(spec, tlo, thi); break;
    case 13: mel_run_default<13>(spec, tlo, thi); break;
    case 14: mel_run_default<14>(spec, tlo, thi); break;
    default: mel_run_default<15>(spec, tlo, thi); break;
  }
}

// generic bank (any other sample rate / band edges): warp-uniform loops over the group table
__device__ __forceinline__ void mel_phase_generic(int g, int gend, const int4* s_groups, const float2* s_binw,
                                                  const float* spec, float* tlo, float* thi) {
  for (; g < gend; ++g) {
    const int4 gi = s_groups[g];
    const float* x = spec + gi.x;
    const float2* w = s_binw + gi.y;
    float lo = 0.0f, hi = 0.0f;
    for (int i = 0; i < gi.z; ++i) {
      const float xv = x[i];
      const float2 wv = w[i];
      lo = fmaf(wv.x, xv, lo);
      hi = fmaf(wv.y, xv, hi);
    }
    tlo[gi.w] = lo;
    thi[gi.w + 1] = hi;
  }
}

// Launch chaining of the frontend kernels (programmatic dependent launch, common.cuh).  Both kernels are launched with
// the programmatic attribute: their CTAs take SMs as the previous kernel of the stream (the core / smoothing kernel of the
// previous forward, another frontend launch, the streaming step's tail shift) drains, and the prologue above -- tables
// into shared memory, barrier set-up: it reads nothing but the frontend's own immutable tables -- runs beside that
// kernel's tail.  Everything after this point reads the audio and writes the mel rows, so it waits for the previous
// kernel to complete first; only THEN are this kernel's own dependents released (the emotion stream, which reads nothing
// this kernel writes, takes each SM as this kernel's CTA leaves it): a dependent released before the wait could run
// while the kernel before this one is still reading the buffers that dependent writes.
//
// `wait_at_end` (the edge-variant launches of a forward, csrc/session.cu): the kernel before this one is another frontend
// launch of the same forward -- it writes other buffers and has itself waited for everything older -- so this launch
// neither reads nor writes anything that kernel touches and does not wait for it: its CTAs start on the SMs that kernel's
// earliest CTAs leave.  It still must not COMPLETE before that kernel has (what follows waits on the last kernel of the
// chain only), so the wait moves to the end.
__device__ __forceinline__ void pdl_prologue_done(const LogmelParams& p) {
  if (!p.wait_at_end) pdl_wait();
  pdl_launch_dependents();
}
__device__ __forceinline__ void pdl_epilogue(const LogmelParams& p) {
  if (p.wait_at_end) pdl_wait();
}

// ---- the per-pair pieces shared by the two kernel organisations below ------------------------------------------------
// window, first 32-point FFT, twiddles: registers only.  On entry v[bitrev5(n1)] = (a, b)[32 n1 + lane]; on return
// v[k1] = W_1024^(k1 lane) Y[k1] of column n2 = lane
__device__ __forceinline__ void fft_first_half(float2 (&v)[32], const float* s_hann, const float2* s_tw, int lane) {
#pragma unroll
  for (int n1 = 0; n1 < 32; ++n1) v[bitrev5(n1)] = __fmul2_rn(v[bitrev5(n1)], bcast(s_hann[32 * n1 + lane]));
  fft32(v);
#pragma unroll
  for (int k1 = 1; k1 < 32; ++k1) {
    const float2 w = s_tw[k1 * 32 + lane];  // W_1024^(k1 * n2)
    const float2 z = v[k1];
    float2 r = __fmul2_rn(z, bcast(w.x));
    v[k1] = __ffma2_rn(make_float2(-z.y, z.x), bcast(w.y), r);
  }
}

// 32x32 transposition through the warp's padded tile, second FFT, separation of the two real spectra: leaves
// 4 |A_k|^2 at xb[k] and 4 |B_k|^2 at xb[kSecondFrame + k], k = 0..512
__device__ __forceinline__ void fft_second_half(float2 (&v)[32], float* xb, int lane) {
  float2* xb2 = reinterpret_cast<float2*>(xb);
#pragma unroll
  for (int k1 = 0; k1 < 32; ++k1) xb2[k1 * kRowF2 + lane] = v[k1];
  __syncwarp();
#pragma unroll
  for (int n2 = 0; n2 < 32; ++n2) v[bitrev5(n2)] = xb2[lane * kRowF2 + n2];
  __syncwarp();
  fft32(v);  // v[k2] = Z[lane + 32 * k2]

  // separate the two real spectra: partner of k = lane + 32 r is 1024 - k = ((32-lane)&31) + 32 r'.
  // Lanes 1..31: partner register r' = 31 - r; lane 0: r' = 32 - r, which is the value it fetched (from itself) one
  // step earlier, and r = 0 is its own partner.  Four steps at a time: only 8 shuffle results are live at once.
  const int src = (32 - lane) & 31;
  float* pa = xb;
  float* pb = xb + kSecondFrame;
  float2 prev = v[0];
#pragma unroll
  for (int r0 = 0; r0 < 16; r0 += 4) {
    float2 q[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      q[j].x = __shfl_sync(kFullMask, v[31 - r0 - j].x, src);
      q[j].y = __shfl_sync(kFullMask, v[31 - r0 - j].y, src);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = r0 + j;
      const float2 z = v[r];
      const float2 c = lane == 0 ? prev : q[j];
      prev = q[j];
      // 2A = z + conj(c), 2iB = z - conj(c): (4|A|^2, 4|B|^2) = u*u + w*w, u = (z.x + c.x, z.x - c.x), w = (z.y - c.y, z.y + c.y)
      const float2 u = __fadd2_rn(bcast(z.x), make_float2(c.x, -c.x));
      const float2 w = __fadd2_rn(bcast(z.y), make_float2(-c.y, c.y));
      const float2 pw = __ffma2_rn(w, w, __fmul2_rn(u, u));
      pa[lane + 32 * r] = pw.x;
      pb[lane + 32 * r] = pw.y;
    }
    asm volatile("" ::: "memory");  // keep the compiler from hoisting the next group's shuffles (register pressure)
  }
  if (lane == 0) {  // Nyquist bin 512 = register 16, self-paired: A = z.x, B = z.y (x4 like the others)
    pa[512] = 4.0f * v[16].x * v[16].x;
    pb[512] = 4.0f * v[16].y * v[16].y;
  }
}

// store phase of one frame pair whose mel rows sit in tile rows (row, row + 1): dB, per-frame maxima, coalesced stores
template <bool kSplitB>
__device__ __forceinline__ void store_pair_rows(const FrontendTables& tab, const LogmelParams& p, int clip, int frame,
                                                bool has_b, const float* tiles, int row, int lane) {
  const float* tlo = tiles + row * kTileStride;
  const float* thi = tlo + kSlots * kTileStride;
  float* dst = p.power + (long long)clip * p.power_clip_stride + (long long)frame * KOE_N_MELS;
  // the 160 values of the two rows (row B follows row A in the clip's block), five per lane: j = lane + 32 q;
  // j < 80 -> frame A filter j, else frame B filter j - 80, which sits kTileStride - 80 = 1 float further in the tile
  float db[5];
#pragma unroll
  for (int qd = 0; qd < 5; ++qd) {
    const int j = lane + 32 * qd;
    const bool second = qd > 2 || (qd == 2 && lane >= KOE_N_MELS - 64);
    const int t = j + (second ? kTileStride - KOE_N_MELS : 0);
    const float pw = tlo[t] + thi[t];
    // stored in dB (the consumer only subtracts its reference and clamps), or as ln(p + eps) for the torchaudio flavour
    db[qd] = tab.log_mode == 0 ? db_from_power(pw) : ln_from_power(pw, tab.log_eps);
  }
  float mx_a = fmaxf(db[0], db[1]), mx_b = fmaxf(db[3], db[4]);
  if (lane < KOE_N_MELS - 64) mx_a = fmaxf(mx_a, db[2]); else mx_b = fmaxf(mx_b, db[2]);
  // row B follows row A, or goes to its own buffer (power_b: pair j of the clip -> row j there); dst_b is biased by
  // one row so that the same indices address it
  float* dst_b = dst;
  if constexpr (kSplitB)
    dst_b = p.power_b + (long long)clip * p.power_b_clip_stride + (long long)(frame >> 1) * KOE_N_MELS - KOE_N_MELS;
  dst[lane] = db[0];
  dst[lane + 32] = db[1];
  float* dst_mid = lane < KOE_N_MELS - 64 ? dst : dst_b;  // the third 32-value piece straddles the two rows
  if (has_b || lane < KOE_N_MELS - 64) dst_mid[lane + 64] = db[2];
  if (has_b) {
    dst_b[lane + 96] = db[3];
    dst_b[lane + 128] = db[4];
  }
  if (p.frame_max != nullptr) {
    const int ia = __reduce_max_sync(kFullMask, float_order(mx_a));
    const int ib = __reduce_max_sync(kFullMask, float_order(mx_b));
    float* fm = p.frame_max + (long long)clip * p.fmax_clip_stride + frame;
    float* fm_b = fm;
    if constexpr (kSplitB) fm_b = p.frame_max_b + (long long)clip * p.fmax_b_clip_stride + (frame >> 1) - 1;
    if (lane == 0) fm[0] = order_float(ia);
    if (lane == 1 && has_b) fm_b[1] = order_float(ib);
  }
}

// Pair of iteration `iter` (pairs iter * kWarps + warp) for one warp.  Interior pairs (all but the few per clip that touch
// an edge) come last in the launch order, clip by clip; successive calls advance by a constant number of pairs
// (gridDim.x * kWarps), so clip and pair are kept incrementally: no division in the loop.
struct PairLocator {
  int in_clip = -1, in_j = 0;  // interior position of the pair located last (-1: none yet)
  __device__ __forceinline__ static unsigned total_pairs(const LogmelParams& p) {
    return (unsigned)p.n_clips * ((unsigned)(p.n_frames + 1) >> 1);
  }
  __device__ __forceinline__ PairInfo locate(const LogmelParams& p, unsigned iter, unsigned n_iters, unsigned total_pairs,
                                             unsigned ppc, int warp) {
    const unsigned n_edge_pairs = p.mid_pairs > 0 ? (unsigned)p.n_clips * (unsigned)(p.edge_lo + p.edge_hi) : total_pairs;
    const unsigned pair = iter < n_iters ? iter * kWarps + warp : total_pairs;
    if (pair < n_edge_pairs || pair >= total_pairs) {
      in_clip = -1;
      return locate_pair(p, pair, total_pairs, ppc);
    }
    if (in_clip < 0) {
      const unsigned r = pair - n_edge_pairs;
      in_clip = (int)(r / (unsigned)p.mid_pairs);
      in_j = (int)(r - (unsigned)in_clip * (unsigned)p.mid_pairs);
    } else {
      in_clip += p.step_clips;
      in_j += p.step_pairs;
      if (in_j >= p.mid_pairs) in_j -= p.mid_pairs, ++in_clip;
    }
    PairInfo pi;
    pi.clip = in_clip;
    pi.frame = 2 * (p.edge_lo + in_j);
    pi.has_b = true;
    pi.interior = true;
    pi.fa_lo = p.sample_offset + (p.frame_offset + pi.frame * p.frame_step) * p.hop - kFrameLen / 2;
    pi.fb_lo = pi.fa_lo + p.frame_step * p.hop;
    return pi;
  }
  // the located pair's samples -> registers
  __device__ __forceinline__ void load(const LogmelParams& p, const PairInfo& pi, int lane, float2 (&v)[32]) const {
    if (pi.interior) load_interior(p, pi, lane, v);
    else if (pi.frame >= 0) load_edge(p, pi, lane, v);
  }
};

// The same for a packed variable-length batch: clips of their own lengths, pairs numbered clip by clip, each clip's pairs
// (2j, 2j + 1) formed from its own frames exactly as a launch over that clip alone forms them.  The clip of a pair comes
// from the pair-base table: it only moves forward (by gridDim.x * kWarps pairs per call), so one 32-wide probe of the
// table past the current clip finds it, with a binary search only when the probe falls short (tiny clips) and for the
// warp's first pair.  The pair's geometry is the one-clip geometry with the clip's own length and frame count (masked loads
// where the frames reach past either end of the clip: the neighbours' samples read as zeros); PairInfo.clip is 0 and
// PairInfo.frame the global output row, so that the store phase needs no change.
struct VarlenLocator {
  int clip = -1;
  const float* src = nullptr;  // the located clip's first sample
  int len = 0;                 // its length
  __device__ __forceinline__ static unsigned total_pairs(const LogmelParams& p) { return p.vl_pairs; }
  __device__ __forceinline__ PairInfo locate(const LogmelParams& p, unsigned iter, unsigned n_iters, unsigned total_pairs,
                                             unsigned, int warp) {
    const unsigned pair = iter < n_iters ? iter * kWarps + warp : total_pairs;
    PairInfo pi;
    if (pair >= total_pairs) {
      pi.clip = 0;
      pi.frame = -1;
      pi.interior = false;
      return pi;
    }
    const int* pb = p.vl_pair_base;
    int c = clip < 0 ? 0 : clip;  // pb[c] <= pair
    const int i = c + 1 + (int)(threadIdx.x & 31);
    const unsigned m = __ballot_sync(kFullMask, i >= p.vl_clips || (unsigned)__ldg(pb + i) > pair);  // (pb[n_clips] = total)
    if (m != 0) {
      c += __ffs(m) - 1;
    } else {  // pb[c + 32] <= pair < pb[n_clips]
      int lo = c + 32, hi = p.vl_clips;
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if ((unsigned)__ldg(pb + mid) <= pair) lo = mid;
        else hi = mid;
      }
      c = lo;
    }
    clip = c;
    LogmelParams q = p;
    q.n_samples = len = __ldg(p.vl_length + c);
    const int row0 = __ldg(p.vl_row_base + c);
    q.n_frames = __ldg(p.vl_row_base + c + 1) - row0;
    src = p.audio + __ldg(p.vl_sample_off + c);
    pi = pair_geometry(q, 0, (int)(pair - (unsigned)__ldg(pb + c)));
    pi.frame += row0;
    return pi;
  }
  __device__ __forceinline__ void load(const LogmelParams& p, const PairInfo& pi, int lane, float2 (&v)[32]) const {
    LogmelParams q = p;
    q.audio = src;
    q.n_samples = len;
    if (pi.interior) {
      load_interior(q, pi, lane, v);
    } else if (pi.frame >= 0) {
      // a clip shorter than its window leaves whole pairs past its end: they read nothing but the zeros the masked loads
      // would give
      const bool a_off = pi.fa_lo >= pi.hi_a || pi.fa_lo + kFrameLen <= pi.lo_a;
      const bool b_off = pi.hi_b <= pi.lo_b || pi.fb_lo >= pi.hi_b || pi.fb_lo + kFrameLen <= pi.lo_b;
      if (a_off && b_off) {
#pragma unroll
        for (int n1 = 0; n1 < 32; ++n1) v[n1] = make_float2(0.0f, 0.0f);
      } else {
        load_edge(q, pi, lane, v);
      }
    }
  }
};

// the same for a warp that expects to wait long (the consumers of the warp-specialised kernel wait for the producers most
// of the time): try_wait with a suspend-time hint, then sleep between polls -- a tight poll loop issued 30 % of all the
// kernel's instructions (ncu: BRA / SYNCS / YIELD / ISETP), taking issue slots from the producers on the same scheduler
__device__ __forceinline__ void bar_wait_parked(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  for (uint32_t spin = 0; !ok; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(20000u)
        : "memory");
    if (!ok) {
      __nanosleep(128);
      if (spin > (1u << 20)) __trap();
    }
  }
}

// kSplitB: the pairs' second frames go to their own buffer (LogmelParams::power_b; the streaming step) -- a separate
// instantiation so that the batch kernel carries none of it (the extra pointer arithmetic cost it 3 us of 179)
//
// Schedule of one iteration (16 frame pairs per CTA, one per warp):
//   F  window, first 32-point FFT, twiddles                          registers only
//   W  wait "mel phase of the previous iteration done" (mbarrier): nobody reads this warp's tile any more
//   T  transposition through the tile, second FFT, separation -> the pair's two power spectra in the tile
//   L  the next pair's audio -> registers (in flight during everything below)
//   B  __syncthreads: all 32 spectra of the iteration are in the tiles
//   M  mel phase: lane = frame, warp = run of bins -> mel tiles; arrive on the mbarrier
//   S  store phase of the PREVIOUS iteration's rows (the tiles hold them until the next B), placed per warp class
//      (warp / 4, one warp of every class on each scheduler): classes 0 and 2 before F, classes 1 and 3 after L.  The
//      classes then run the FFT a store phase apart, so that the FMA-bound and the shared-memory-bound stretches of
//      different warps overlap instead of all 16 warps queueing for the same pipe at the same time.
template <bool kDefaultBank, bool kSplitB>
__global__ void __launch_bounds__(kThreads, 1)
logmel_power_kernel(FrontendTables tab, LogmelParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_hann = reinterpret_cast<float*>(smem_raw);              // 1024
  float2* s_tw = reinterpret_cast<float2*>(s_hann + kFrameLen);    // 1024 float2
  float2* s_binw = s_tw + 1024;                                    // kMaxBins float2
  int4* s_groups = reinterpret_cast<int4*>(s_binw + kMaxBins);     // kMaxGroups
  int* s_runs = reinterpret_cast<int*>(s_groups + kMaxGroups);     // kWarps + 1 (+ pad to 32)
  float* s_tiles = reinterpret_cast<float*>(s_runs + 32);          // (tlo | thi), each kSlots * kTileStride
  float* s_scratch = s_tiles + 2 * kSlots * kTileStride;           // kWarps * kScratch, 16-byte aligned, bank 0
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_scratch + kWarps * kScratch);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  for (int i = tid; i < kFrameLen; i += kThreads) s_hann[i] = tab.hann[i];
  for (int i = tid; i < 1024; i += kThreads) s_tw[i] = tab.tw[i];
  for (int i = tid; i < tab.n_bins; i += kThreads) s_binw[i] = tab.binw[i];
  for (int i = tid; i < tab.n_groups; i += kThreads) s_groups[i] = tab.groups[i];
  if (tid <= kWarps) s_runs[tid] = tab.runs[tid];
  // cells that no group writes (filter 0's rising half; filters without a falling / rising group in sparse banks) stay 0
  for (int i = tid; i < 2 * kSlots * kTileStride; i += kThreads) s_tiles[i] = 0.0f;
  const uint32_t mel_done = smem_u32addr(s_bar);
  if (tid == 0) {
    mbarrier_init(mel_done, kWarps);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_prologue_done(p);

  const unsigned ppc = (unsigned)(p.n_frames + 1) >> 1;  // frame pairs per clip
  const unsigned total_pairs = PairLocator::total_pairs(p);
  const unsigned n_iters = (total_pairs + kWarps - 1) / kWarps;
  float* xb = s_scratch + warp * kScratch;
  const bool store_first = ((warp >> 2) & 1) == 0;  // S before F (classes 0, 2) or after L (classes 1, 3)

  auto store_rows = [&](int clip, int frame, bool has_b, const float* tiles) {  // warp w owns tile rows 2w, 2w + 1
    store_pair_rows<kSplitB>(tab, p, clip, frame, has_b, tiles, 2 * warp, lane);
  };
  PairLocator loc;
  auto locate = [&](unsigned iter) { return loc.locate(p, iter, n_iters, total_pairs, ppc, warp); };

  float2 v[32];
  unsigned it = blockIdx.x;
  PairInfo nxt = locate(it);
  loc.load(p, nxt, lane, v);
  int pend_clip = 0, pend_frame = -1;  // the pair whose mel rows wait in the tiles for their store phase
  bool pend_has_b = false;
  unsigned k = 0;                      // iterations done by this CTA: parity of the mbarrier phase / tile buffer

  for (; it < n_iters; it += gridDim.x, ++k) {
    // the mel tiles hold the previous iteration's rows until the next mel phase, i.e. until the __syncthreads below:
    // every store phase, early or late, comes before it
    const float* prev_tiles = s_tiles;
    if (store_first && pend_frame >= 0) {
      mbarrier_wait(mel_done, (k + 1) & 1);  // the previous mel phase, by every warp
      store_rows(pend_clip, pend_frame, pend_has_b, prev_tiles);
      pend_frame = -1;
    }
    // ------------------------------------------------------------------ FFT phase (per warp)
    const PairInfo cur = nxt;
    if (cur.frame >= 0) fft_first_half(v, s_hann, s_tw, lane);
    // the tile still holds this warp's spectra of the previous iteration until every warp has finished that mel phase
    if (k > 0) mbarrier_wait(mel_done, (k + 1) & 1);
    if (cur.frame >= 0) fft_second_half(v, xb, lane);
    // audio of the next iteration: in flight during the mel / store phases
    nxt = locate(it + gridDim.x);
    loc.load(p, nxt, lane, v);
    if (!store_first && pend_frame >= 0) {
      store_rows(pend_clip, pend_frame, pend_has_b, prev_tiles);
      pend_frame = -1;
    }
    __syncthreads();

    // ------------------------------------------------------------------ mel phase: lane = frame slot, warp = run of bins
    {
      float* tlo = s_tiles + lane * kTileStride;
      float* thi = tlo + kSlots * kTileStride;
      const float* spec = s_scratch + (lane >> 1) * kScratch + (lane & 1) * kSecondFrame;
      if (kDefaultBank)
        mel_phase_default(warp, spec, tlo, thi);
      else
        mel_phase_generic(s_runs[warp], s_runs[warp + 1], s_groups, s_binw, spec, tlo, thi);
    }
    __syncwarp();
    if (lane == 0) mbarrier_arrive(mel_done);
    pend_clip = cur.clip, pend_frame = cur.frame, pend_has_b = cur.has_b;
  }
  if (pend_frame >= 0) {
    mbarrier_wait(mel_done, (k + 1) & 1);
    store_rows(pend_clip, pend_frame, pend_has_b, s_tiles);
  }
  pdl_epilogue(p);
}

// ---- warp-specialised organisation (default bank, batch launches) ------------------------------------------------------
// 16 producer warps (one frame pair each per iteration: loads, FFT, spectra into their tile) never touch the mel or store
// phases and never meet at a CTA barrier; 8 consumer warps (two per scheduler) run the mel phase of iteration k -- lane =
// frame, two runs of bins each -- and the store phase while the producers are already in iteration k + 1.  The register
// file is split with setmaxnreg: launch at 80 registers x 768 threads, producers grow (to 96), consumers shrink (to 48).
// Handshakes (mbarriers): spec_ready (16 producer arrivals: the 32 spectra and pair descriptors of iteration k are in
// shared memory), spec_free (8 consumer arrivals: nobody reads the spectra of iteration k any more, the producers may
// overwrite their tiles with the next transposition); the consumers meet at a named barrier between mel and store phase.
constexpr int kWsProducers = kWarps;
constexpr int kWsConsumers = 8;
constexpr int kWsThreads = (kWsProducers + kWsConsumers) * 32;
constexpr int kWsLaunchRegs = (65536 / kWsThreads) & ~7;
constexpr int kWsProducerRegs = 96;
constexpr int kWsConsumerRegs = 48;
static_assert(kWsProducers * kWsProducerRegs + kWsConsumers * kWsConsumerRegs <=
                  (kWsProducers + kWsConsumers) * kWsLaunchRegs,
              "setmaxnreg redistributes the launch allocation");
static_assert(kWarps % kWsConsumers == 0, "whole runs per consumer");

// Locator: PairLocator (clips of one length) or VarlenLocator (the packed variable-length batch)
template <class Locator>
__global__ void __launch_bounds__(kWsThreads, 1)
logmel_power_ws_kernel(FrontendTables tab, LogmelParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_hann = reinterpret_cast<float*>(smem_raw);              // 1024
  float2* s_tw = reinterpret_cast<float2*>(s_hann + kFrameLen);    // 1024 float2
  float* s_tiles = reinterpret_cast<float*>(s_tw + 1024);          // 2 buffers x (tlo | thi), each kSlots * kTileStride
  float* s_scratch = s_tiles + 4 * kSlots * kTileStride;           // kWarps * kScratch, 16-byte aligned
  int4* s_pair = reinterpret_cast<int4*>(s_scratch + kWarps * kScratch);  // [2][kWarps] {clip, frame, has_b, -}
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_pair + 2 * kWarps);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < kFrameLen; i += kWsThreads) s_hann[i] = tab.hann[i];
  for (int i = tid; i < 1024; i += kWsThreads) s_tw[i] = tab.tw[i];
  for (int i = tid; i < 4 * kSlots * kTileStride; i += kWsThreads) s_tiles[i] = 0.0f;
  const uint32_t spec_ready = smem_u32addr(s_bar), spec_free = smem_u32addr(s_bar + 1);
  if (tid == 0) {
    mbarrier_init(spec_ready, kWsProducers);
    mbarrier_init(spec_free, kWsConsumers);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_prologue_done(p);

  const unsigned ppc = (unsigned)(p.n_frames + 1) >> 1;
  const unsigned total_pairs = Locator::total_pairs(p);
  const unsigned n_iters = (total_pairs + kWarps - 1) / kWarps;
  const unsigned first = blockIdx.x, stride = gridDim.x;
  const unsigned n_local = first < n_iters ? (n_iters - first + stride - 1) / stride : 0;

  if (warp < kWsProducers) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kWsProducerRegs));
    float* xb = s_scratch + warp * kScratch;
    Locator loc;
    float2 v[32];
    PairInfo nxt = loc.locate(p, first, n_iters, total_pairs, ppc, warp);
    loc.load(p, nxt, lane, v);
    for (unsigned k = 0; k < n_local; ++k) {
      const PairInfo cur = nxt;
      if (cur.frame >= 0) fft_first_half(v, s_hann, s_tw, lane);
      // the tile holds this warp's spectra of iteration k - 1 until every consumer has finished that mel phase
      if (k > 0) mbarrier_wait(spec_free, (k + 1) & 1);
      if (cur.frame >= 0) fft_second_half(v, xb, lane);
      if (lane == 0) s_pair[(k & 1) * kWarps + warp] = make_int4(cur.clip, cur.frame, cur.has_b ? 1 : 0, 0);
      __syncwarp();
      if (lane == 0) mbarrier_arrive(spec_ready);
      // audio of the next iteration (an L2 prefetch of these lines one iteration ahead changed nothing: 146.7 vs 146.3 us)
      nxt = loc.locate(p, k + 1 < n_local ? first + (k + 1) * stride : n_iters, n_iters, total_pairs, ppc, warp);
      loc.load(p, nxt, lane, v);
    }
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kWsConsumerRegs));
    const int c = warp - kWsProducers;
    for (unsigned k = 0; k < n_local; ++k) {
      float* tiles = s_tiles + (k & 1) * (2 * kSlots * kTileStride);
      bar_wait_parked(spec_ready, k & 1);
      {
        float* tlo = tiles + lane * kTileStride;
        float* thi = tlo + kSlots * kTileStride;
        const float* spec = s_scratch + (lane >> 1) * kScratch + (lane & 1) * kSecondFrame;
#pragma unroll 1
        for (int run = c * (kWarps / kWsConsumers); run < (c + 1) * (kWarps / kWsConsumers); ++run)
          mel_phase_default(run, spec, tlo, thi);
      }
      __syncwarp();
      if (lane == 0) mbarrier_arrive(spec_free);
      asm volatile("bar.sync 1, %0;" ::"n"(kWsConsumers * 32) : "memory");  // every run of this iteration is in the tiles
#pragma unroll 1
      for (int w = c * (kWarps / kWsConsumers); w < (c + 1) * (kWarps / kWsConsumers); ++w) {
        const int4 pi = s_pair[(k & 1) * kWarps + w];
        if (pi.y >= 0) store_pair_rows<false>(tab, p, pi.x, pi.y, pi.z != 0, tiles, 2 * w, lane);
      }
      if (p.early_flag != nullptr) {
        // this CTA's last iteration below the threshold: its rows (this warp's share, and in program order all earlier
        // ones) are stored -> release them to the core, which acquires the counter (8 arrivals per CTA)
        const unsigned it = first + k * stride;
        if (it < p.early_iters && it + stride >= p.early_iters) {
          __syncwarp();
          if (lane == 0) {
            __threadfence();
            atomicAdd(p.early_flag, 1u);
          }
        }
      }
    }
  }
  pdl_epilogue(p);
}

constexpr size_t kLogmelWsSmem = sizeof(float) * kFrameLen + sizeof(float2) * 1024 +
                                 sizeof(float) * (4 * kSlots * kTileStride + kWarps * kScratch) + sizeof(int4) * 2 * kWarps + 16;

constexpr size_t kLogmelSmem = sizeof(float) * kFrameLen + sizeof(float2) * 1024 + sizeof(float2) * kMaxBins +
                               sizeof(int4) * kMaxGroups + sizeof(int) * 32 +
                               sizeof(float) * (2 * kSlots * kTileStride + kWarps * kScratch) + 16;

// The grid is one CTA per SM (launch_logmel): that is all either kernel's shared memory admits (228 KB per SM on sm_100,
// 1 KB of it reserved per CTA).
constexpr size_t kSmemPerSm = 228 * 1024, kSmemReservedPerCta = 1024;
static_assert(2 * (kLogmelSmem + kSmemReservedPerCta) > kSmemPerSm, "logmel_power_kernel: more than one CTA per SM");
static_assert(2 * (kLogmelWsSmem + kSmemReservedPerCta) > kSmemPerSm, "logmel_power_ws_kernel: more than one CTA per SM");

// ---- dB normalisation: ref = clip max, clamp, rescale; emits long-term and last-3 short-term features
__global__ void logmel_normalise_kernel(const float* __restrict__ power, const float* __restrict__ frame_max,
                                        int n_frames, int db_only, float* __restrict__ long_term,
                                        float* __restrict__ short_term) {
  __shared__ float s_red[32];
  __shared__ float s_ref_db;
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* fm = frame_max + (long long)b * n_frames;
  float mx = -INFINITY;
  for (int g = tid; g < n_frames; g += blockDim.x) mx = fmaxf(mx, fm[g]);
  mx = warp_max(mx);
  if ((tid & 31) == 0) s_red[tid >> 5] = mx;
  __syncthreads();
  if (tid < 32) {
    float v = tid < (blockDim.x >> 5) ? s_red[tid] : -INFINITY;
    v = warp_max(v);
    if (tid == 0) s_ref_db = v;
  }
  __syncthreads();
  const float ref_db = s_ref_db;
  const float4* src = reinterpret_cast<const float4*>(power + (long long)b * n_frames * KOE_N_MELS);
  float4* dst = reinterpret_cast<float4*>(long_term + (long long)b * n_frames * KOE_N_MELS);
  const int n4 = n_frames * (KOE_N_MELS / 4);
  const bool rescale = db_only == 0;
  for (int i = tid; i < n4; i += blockDim.x) {
    float4 v = src[i];
    v.x = normalise_db(v.x, ref_db, rescale);
    v.y = normalise_db(v.y, ref_db, rescale);
    v.z = normalise_db(v.z, ref_db, rescale);
    v.w = normalise_db(v.w, ref_db, rescale);
    dst[i] = v;
  }
  if (short_term != nullptr) {
    // last three frames; clips shorter than 3 frames: rows [0, n_frames) then zeros (reference :206-212)
    float* st = short_term + (long long)b * 3 * KOE_N_MELS;
    for (int i = tid; i < 3 * KOE_N_MELS; i += blockDim.x) {
      const int row = i / KOE_N_MELS, m = i % KOE_N_MELS;
      const int g = n_frames >= 3 ? n_frames - 3 + row : row;
      float v = 0.0f;
      if (g < n_frames)
        v = normalise_db(power[((long long)b * n_frames + g) * KOE_N_MELS + m], ref_db, rescale);
      st[i] = v;
    }
  }
}

// ---- host side: HTK filterbank without normalisation (torchaudio.functional.melscale_fbanks(mel_scale="htk", norm=None),
// the bank of T.MelSpectrogram in the reference's src/features/stft.py:84-96), on the bins of an n_fft-point spectrum
static std::vector<float> htk_filterbank(int sr, int n_fft, int n_mels, double fmin, double fmax) {
  const int n_bins = 1 + n_fft / 2;
  auto to_mel = [](double f) { return 2595.0 * std::log10(1.0 + f / 700.0); };
  auto to_hz = [](double m) { return 700.0 * (std::pow(10.0, m / 2595.0) - 1.0); };
  std::vector<double> f_pts(n_mels + 2);
  const double m0 = to_mel(fmin), m1 = to_mel(fmax);
  for (int i = 0; i < n_mels + 2; ++i) f_pts[i] = to_hz(m0 + (m1 - m0) * i / (n_mels + 1));
  std::vector<float> fb((size_t)n_mels * n_bins, 0.0f);
  for (int m = 0; m < n_mels; ++m) {
    const double d0 = f_pts[m + 1] - f_pts[m], d1 = f_pts[m + 2] - f_pts[m + 1];
    for (int k = 0; k < n_bins; ++k) {
      const double f = (double)(sr / 2) * k / (n_bins - 1);  // all_freqs = linspace(0, sr // 2, n_freqs)
      const double down = (f - f_pts[m]) / d0, up = (f_pts[m + 2] - f) / d1;
      fb[(size_t)m * n_bins + k] = (float)std::fmax(0.0, std::fmin(down, up));
    }
  }
  return fb;
}

// ---- host side: Slaney filterbank (librosa.filters.mel restated, float64 then float32) -----------
static double hz_to_mel(double f) {
  const double f_sp = 200.0 / 3, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp;
  const double logstep = std::log(6.4) / 27.0;
  return f >= min_log_hz ? min_log_mel + std::log(f / min_log_hz) / logstep : f / f_sp;
}
static double mel_to_hz(double m) {
  const double f_sp = 200.0 / 3, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp;
  const double logstep = std::log(6.4) / 27.0;
  return m >= min_log_mel ? min_log_hz * std::exp(logstep * (m - min_log_mel)) : f_sp * m;
}

static std::vector<float> slaney_filterbank(int sr, int n_fft, int n_mels, double fmin, double fmax) {
  const int n_bins = 1 + n_fft / 2;
  std::vector<double> mel_f(n_mels + 2);
  const double m0 = hz_to_mel(fmin), m1 = hz_to_mel(fmax);
  for (int i = 0; i < n_mels + 2; ++i) {
    // numpy.linspace: start + i * step, last point pinned to stop
    const double step = (m1 - m0) / (n_mels + 1);
    mel_f[i] = mel_to_hz(i == n_mels + 1 ? m1 : m0 + i * step);
  }
  std::vector<float> fb((size_t)n_mels * n_bins, 0.0f);
  for (int m = 0; m < n_mels; ++m) {
    const double d0 = mel_f[m + 1] - mel_f[m], d1 = mel_f[m + 2] - mel_f[m + 1];
    const double enorm = 2.0 / (mel_f[m + 2] - mel_f[m]);
    for (int k = 0; k < n_bins; ++k) {
      const double f = (double)k * sr / n_fft;
      const double lower = -(mel_f[m] - f) / d0, upper = (mel_f[m + 2] - f) / d1;
      const double w = std::fmax(0.0, std::fmin(lower, upper));
      // librosa stores float32 weights, then multiplies the float32 array by the float64 norm
      const float w32 = (float)w;
      fb[(size_t)m * n_bins + k] = (float)((double)w32 * enorm);
    }
  }
  return fb;
}

}  // namespace koe

using namespace koe;

struct koe_frontend {
  int device = 0, sample_rate = 0, n_fft = 0, n_mels = 0;
  float fmin = 0, fmax = 0;
  int log_mode = 0;
  float log_eps = 0;
  float* d_hann = nullptr;
  float2* d_tw = nullptr;
  float2* d_binw = nullptr;
  int* d_tables = nullptr;  // groups[kMaxGroups] (int4) | runs[kWarps + 1 -> 32]
  int n_bins = 0, n_groups = 0;
  bool default_bank = false;  // structure == melbank_default.inc: the unrolled filterbank phase applies
  std::vector<float> fb_host;
};

extern "C" int koe_frontend_create(int device, int sample_rate, int n_fft, int n_mels, float fmin, float fmax,
                                   koe_frontend_t** out) {
  koe_frontend_config c;
  c.device = device;
  c.sample_rate = sample_rate;
  c.n_fft = n_fft;
  c.n_mels = n_mels;
  c.fmin = fmin;
  c.fmax = fmax;
  c.mel_scale = KOE_MEL_SLANEY;
  c.mel_norm = KOE_MEL_NORM_SLANEY;
  c.window_normalized = 0;
  c.log_mode = KOE_LOG_DB;
  c.log_eps = 0.0f;
  c.win_length = 0;
  return koe_frontend_create_ex(&c, out);
}

extern "C" int koe_frontend_create_ex(const koe_frontend_config* cfg, koe_frontend_t** out) {
  KOE_REQUIRE(out != nullptr && cfg != nullptr, "koe_frontend_create: NULL argument");
  const int device = cfg->device, sample_rate = cfg->sample_rate, n_fft = cfg->n_fft, n_mels = cfg->n_mels;
  const float fmin = cfg->fmin, fmax = cfg->fmax;
  if ((n_fft != KOE_N_FFT && n_fft != KOE_N_FFT / 2) || n_mels != KOE_N_MELS)
    return fail(KOE_E_UNSUPPORTED, "koe_frontend_create: only n_fft=1024 or 512 and n_mels=80 are implemented (got %d, %d)",
                n_fft, n_mels);
  KOE_REQUIRE(sample_rate > 0 && fmin >= 0 && fmax > fmin && fmax <= sample_rate / 2.0f,
              "koe_frontend_create: bad sample_rate/fmin/fmax");
  KOE_REQUIRE((cfg->mel_scale == KOE_MEL_SLANEY && cfg->mel_norm == KOE_MEL_NORM_SLANEY) ||
                  (cfg->mel_scale == KOE_MEL_HTK && cfg->mel_norm == KOE_MEL_NORM_NONE),
              "koe_frontend_create: implemented banks are slaney scale + slaney norm (librosa) and htk scale + no norm "
              "(torchaudio)");
  KOE_REQUIRE((cfg->log_mode == KOE_LOG_DB) || (cfg->log_mode == KOE_LOG_LN_EPS && cfg->log_eps > 0),
              "koe_frontend_create: bad log_mode / log_eps");
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0)
    return fail(KOE_E_NODEVICE, "koe_frontend_create: no CUDA device (this library has no CPU path)");
  KOE_REQUIRE(device >= 0 && device < n_dev, "koe_frontend_create: device %d out of range", device);
  int prev = 0;
  KOE_CUDA(cudaGetDevice(&prev));
  KOE_CUDA(cudaSetDevice(device));

  auto* fe = new koe_frontend();
  fe->device = device;
  fe->sample_rate = sample_rate;
  fe->n_fft = n_fft;
  fe->n_mels = n_mels;
  fe->fmin = fmin;
  fe->fmax = fmax;
  fe->log_mode = cfg->log_mode;
  fe->log_eps = cfg->log_eps;
  // The kernel always transforms 1024 samples.  A 512-point frame is the same frame zero-extended: its spectrum is the
  // even bins of the 1024-point one (X_1024[2k] = X_512[k] up to a phase), so the window table holds the 512-point window
  // in its middle and the bank puts its weights on the even bins.
  const int sub = KOE_N_FFT / n_fft;  // 1 or 2
  {
    const std::vector<float> native = cfg->mel_scale == KOE_MEL_HTK
                                          ? htk_filterbank(sample_rate, n_fft, n_mels, fmin, fmax)
                                          : slaney_filterbank(sample_rate, n_fft, n_mels, fmin, fmax);
    const int nb = 1 + n_fft / 2;
    fe->fb_host.assign((size_t)n_mels * kBins, 0.0f);
    for (int m = 0; m < n_mels; ++m)
      for (int k = 0; k < nb; ++k) fe->fb_host[(size_t)m * kBins + sub * k] = native[(size_t)m * nb + k];
  }
  // periodic Hann of n_fft points, centred in the 1024-sample frame; torchaudio's normalized=True ("window") divides the
  // STFT by sqrt(sum w^2), i.e. the power by sum w^2: folded into the sparse weights below
  const int win_length = cfg->win_length > 0 ? cfg->win_length : n_fft;
  if (win_length > n_fft || win_length < 2) {
    delete fe;
    cudaSetDevice(prev);
    return fail(KOE_E_INVALID, "koe_frontend_create: win_length %d must be in [2, n_fft = %d]", win_length, n_fft);
  }
  std::vector<float> hann(kFrameLen, 0.0f);
  double wsum2 = 0.0;
  for (int n = 0; n < win_length; ++n) {  // window of win_length points centred in the n_fft frame (pad_center)
    const double w = 0.5 - 0.5 * std::cos(2.0 * M_PI * n / win_length);
    hann[(kFrameLen - n_fft) / 2 + (n_fft - win_length) / 2 + n] = (float)w;
    wsum2 += (double)(float)w * (double)(float)w;
  }
  const float wscale = cfg->window_normalized ? (float)(0.25 / wsum2) : 0.25f;  // 0.25: the kernel leaves 4 |X|^2

  // bin-major sparse filterbank: every weighted bin feeds one filter or two adjacent ones (fl, fl + 1); consecutive bins
  // with the same fl form a group (the interval between two filter centres), and fl rises by one from group to group
  std::vector<float2> binw;
  std::vector<int> tables(4 * kMaxGroups + 32, 0);
  std::vector<unsigned char> bin_group(kBins, 255);
  int n_groups = 0;
  auto unsupported = [&](const char* why, int k) {
    delete fe;
    cudaSetDevice(prev);
    return fail(KOE_E_UNSUPPORTED, "koe_frontend_create: filterbank is not a bank of adjacent triangles (%s at bin %d)", why, k);
  };
  {
    int prev_k = -1, prev_fl = -1;
    for (int k = 0; k < kBins; ++k) {
      int first = -1, count = 0, last = -1;
      for (int m = 0; m < n_mels; ++m)
        if (fe->fb_host[(size_t)m * kBins + k] > 1e-12f) {  // (a band edge that falls on a bin leaves ~1e-17 there)
          if (first < 0) first = m;
          last = m;
          ++count;
        }
      if (count == 0) continue;
      if (count > 2 || last - first > 1) return unsupported("more than two / non-adjacent filters", k);
      // bins without weight inside the support (the odd bins of a 512-point bank) ride along in the current group
      for (int z = prev_k + 1; prev_k >= 0 && z < k; ++z) {
        if ((int)binw.size() >= kMaxBins) return unsupported("too many weighted bins", z);
        ++tables[4 * (n_groups - 1) + 2];
        binw.push_back(make_float2(0.0f, 0.0f));
      }
      if ((int)binw.size() >= kMaxBins) return unsupported("too many weighted bins", k);
      if (first != prev_fl) {
        if (first < prev_fl) return unsupported("filters out of order", k);
        if (n_groups >= kMaxGroups) return unsupported("too many groups", k);
        tables[4 * n_groups + 0] = k;
        tables[4 * n_groups + 1] = (int)binw.size();
        tables[4 * n_groups + 2] = 0;
        tables[4 * n_groups + 3] = first;
        ++n_groups;
      }
      ++tables[4 * (n_groups - 1) + 2];
      bin_group[k] = (unsigned char)first;
      binw.push_back(make_float2(wscale * fe->fb_host[(size_t)first * kBins + k],
                                 count == 2 ? wscale * fe->fb_host[(size_t)last * kBins + k] : 0.0f));
      prev_k = k;
      prev_fl = first;
    }
    if (n_groups == 0) return unsupported("empty bank", 0);
  }
  fe->n_bins = (int)binw.size();
  fe->n_groups = n_groups;
  // runs: contiguous group ranges, one per warp, balanced on bins + a per-group overhead (generic kernel only)
  {
    int* runs = tables.data() + 4 * kMaxGroups;
    auto cost = [&](int g) { return 3 + tables[4 * g + 2]; };
    long long total = 0;
    for (int g = 0; g < n_groups; ++g) total += cost(g);
    long long acc = 0;
    int r = 1;
    runs[0] = 0;
    for (int g = 0; g < n_groups && r < kWarps; ++g) {
      acc += cost(g);
      if (acc * kWarps >= total * r) runs[r++] = g + 1;
    }
    for (; r <= kWarps; ++r) runs[r] = n_groups;
  }
  // the unrolled filterbank phase applies when the bank has the structure of melbank_default.inc and its weights
  // (computed above from the run-time arguments) equal the baked-in ones to within one float32 ulp
  fe->default_bank = sub == 1 && win_length == n_fft && !cfg->window_normalized && fe->n_bins == kDefNumBins && tables[0] == kDefFirstBin &&
                     std::equal(bin_group.begin(), bin_group.end(), kDefBinGroup);
  for (int i = 0; fe->default_bank && i < kDefNumBins; ++i) {
    const float got[2] = {binw[i].x, binw[i].y}, want[2] = {kDefBinW[2 * i], kDefBinW[2 * i + 1]};
    for (int h = 0; h < 2; ++h)
      if (std::fabs(got[h] - want[h]) > 1.2e-7f * std::fabs(want[h])) fe->default_bank = false;
  }
  std::vector<float2> tw(1024);
  for (int k1 = 0; k1 < 32; ++k1)
    for (int n2 = 0; n2 < 32; ++n2) {
      const double a = -2.0 * M_PI * (double)(k1 * n2) / 1024.0;
      tw[k1 * 32 + n2] = make_float2((float)std::cos(a), (float)std::sin(a));
    }
  cudaError_t e = cudaSuccess;
  auto up = [&](void** dptr, const void* src, size_t bytes) {
    if (e != cudaSuccess) return;
    e = cudaMalloc(dptr, bytes);
    if (e == cudaSuccess) e = cudaMemcpy(*dptr, src, bytes, cudaMemcpyHostToDevice);
  };
  up((void**)&fe->d_hann, hann.data(), hann.size() * sizeof(float));
  up((void**)&fe->d_tw, tw.data(), tw.size() * sizeof(float2));
  binw.resize(kMaxBins, make_float2(0.f, 0.f));
  up((void**)&fe->d_binw, binw.data(), binw.size() * sizeof(float2));
  up((void**)&fe->d_tables, tables.data(), tables.size() * sizeof(int));
  cudaSetDevice(prev);
  if (e != cudaSuccess) {
    koe_frontend_destroy(fe);
    return fail((int)e, "koe_frontend_create: %s", cudaGetErrorString(e));
  }
  *out = fe;
  return KOE_OK;
}

extern "C" int koe_frontend_destroy(koe_frontend_t* fe) {
  if (fe == nullptr) return KOE_OK;
  cudaFree(fe->d_hann);
  cudaFree(fe->d_tw);
  cudaFree(fe->d_binw);
  cudaFree(fe->d_tables);
  delete fe;
  return KOE_OK;
}

extern "C" int koe_frontend_uses_unrolled_bank(const koe_frontend_t* fe) { return fe != nullptr && fe->default_bank ? 1 : 0; }

extern "C" int koe_frontend_filterbank_host(const koe_frontend_t* fe, float* fb_host) {
  KOE_REQUIRE(fe != nullptr && fb_host != nullptr, "koe_frontend_filterbank_host: NULL argument");
  std::copy(fe->fb_host.begin(), fe->fb_host.end(), fb_host);
  return KOE_OK;
}

extern "C" int koe_logmel_power_ex(const koe_frontend_t* fe, const koe_logmel_args* a, void* stream) {
  const FrontendMode mode = a != nullptr && a->power_b != nullptr ? FrontendMode::SplitPairs : FrontendMode::Frames;
  return koe::launch_logmel(fe, a, mode, /*follows_frontend_launch=*/false, stream);
}

namespace koe {
namespace {
// sets the shared-memory size of the instantiation once per device, then launches it behind the previous kernel
template <void (*Kernel)(FrontendTables, LogmelParams)>
int launch_instantiation(const FrontendTables& tab, const LogmelParams& p, int grid, int threads, size_t smem,
                         cudaStream_t stream) {
  static bool configured[64] = {false};
  int dev = 0;
  KOE_CUDA(cudaGetDevice(&dev));
  KOE_REQUIRE(dev >= 0 && dev < 64, "device index too large");
  if (!configured[dev]) {
    KOE_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured[dev] = true;
  }
  const cudaError_t e = launch_after_primary_starts(Kernel, dim3(grid), dim3(threads), smem, stream, tab, p);
  count_launch();
  KOE_CUDA(e);
  return KOE_OK;
}

// the instantiation of each (mode, bank): the warp-specialised kernel where it exists, the lock-step one elsewhere
int launch_power(FrontendMode mode, bool default_bank, const FrontendTables& tab, const LogmelParams& p, int grid,
                 cudaStream_t stream) {
  switch (mode) {
    case FrontendMode::Frames:
      if (default_bank)
        return launch_instantiation<logmel_power_ws_kernel<PairLocator>>(tab, p, grid, kWsThreads, kLogmelWsSmem, stream);
      return launch_instantiation<logmel_power_kernel<false, false>>(tab, p, grid, kThreads, kLogmelSmem, stream);
    case FrontendMode::SplitPairs:
      if (default_bank)
        return launch_instantiation<logmel_power_kernel<true, true>>(tab, p, grid, kThreads, kLogmelSmem, stream);
      return launch_instantiation<logmel_power_kernel<false, true>>(tab, p, grid, kThreads, kLogmelSmem, stream);
    case FrontendMode::Varlen:
      if (default_bank)
        return launch_instantiation<logmel_power_ws_kernel<VarlenLocator>>(tab, p, grid, kWsThreads, kLogmelWsSmem, stream);
      return fail(KOE_E_UNSUPPORTED, "packed variable-length batches are implemented for the default filterbank only");
  }
  return fail(KOE_E_INVALID, "koe_logmel_power: unknown frontend mode %d", (int)mode);
}

// the frontend's tables, and the launch parameters every mode takes from the arguments
void launch_setup(const koe_frontend_t* fe, const koe_logmel_args* a, bool follows_frontend_launch, FrontendTables* tab,
                  LogmelParams* p) {
  tab->hann = fe->d_hann;
  tab->tw = fe->d_tw;
  tab->binw = fe->d_binw;
  tab->groups = reinterpret_cast<const int4*>(fe->d_tables);
  tab->runs = fe->d_tables + 4 * kMaxGroups;
  tab->n_bins = fe->n_bins;
  tab->n_groups = fe->n_groups;
  tab->log_mode = fe->log_mode;
  tab->log_eps = fe->log_eps;
  *p = LogmelParams{};
  p->audio = a->audio;
  p->audio_stride = a->audio_stride;
  p->n_clips = a->n_clips;
  p->n_samples = a->n_samples;
  p->hop = a->hop;
  p->n_frames = a->n_frames;
  p->lo_rel = a->lo_rel_hops;
  p->hi_rel = a->hi_rel_hops;
  p->frame_offset = a->frame_offset;
  p->frame_step = a->frame_step;
  p->sample_offset = a->sample_offset;
  p->pad_mode = a->pad_mode;
  p->power = a->power;
  p->frame_max = a->frame_max;
  p->power_clip_stride = a->power_clip_stride;
  p->fmax_clip_stride = a->frame_max_clip_stride;
  p->power_b = a->power_b;
  p->power_b_clip_stride = a->power_b_clip_stride;
  p->frame_max_b = a->frame_max_b;
  p->fmax_b_clip_stride = a->frame_max_b_clip_stride;
  p->wait_at_end = follows_frontend_launch ? 1 : 0;
}
}  // namespace
}  // namespace koe

// `follows_frontend_launch`: the kernel queued just before this one on `stream` is another frontend launch of the same
// forward, writing other buffers (see pdl_prologue_done in the kernels)
int koe::launch_logmel(const koe_frontend_t* fe, const koe_logmel_args* a, FrontendMode mode, bool follows_frontend_launch,
                       void* stream, EarlyRelease* early, const VarlenTables* vl) {
  if (early != nullptr) early->target = 0;
  long long pairs = 0;
  if (mode == FrontendMode::Varlen) {
    KOE_REQUIRE(fe != nullptr && a != nullptr && vl != nullptr, "koe_logmel_power (varlen): NULL argument");
    if (vl->n_clips == 0 || vl->pairs == 0) return KOE_OK;
    KOE_REQUIRE(a->audio != nullptr && a->power != nullptr && a->frame_max != nullptr && vl->sample_off && vl->length &&
                    vl->pair_base && vl->row_base,
                "koe_logmel_power (varlen): NULL buffer");
    KOE_REQUIRE(a->hop > 0 && a->frame_offset >= 0 && a->frame_step >= 1, "koe_logmel_power (varlen): bad geometry");
    pairs = vl->pairs;
  } else {
    KOE_REQUIRE(fe != nullptr && a != nullptr, "koe_logmel_power: NULL argument");
    KOE_REQUIRE(a->n_clips >= 0 && a->n_samples >= 0 && a->n_frames >= 0, "koe_logmel_power: negative size");
    if (a->n_clips == 0 || a->n_frames == 0) return KOE_OK;  // nothing to do: empty buffers may be NULL
    KOE_REQUIRE(a->audio != nullptr && a->power != nullptr, "koe_logmel_power: NULL buffer");
    KOE_REQUIRE(a->hop > 0 && a->audio_stride >= a->n_samples, "koe_logmel_power: bad hop/stride");
    KOE_REQUIRE(a->frame_offset >= 0 && a->frame_step >= 1 && a->sample_offset >= 0,
                "koe_logmel_power: bad frame_offset/frame_step/sample_offset");
    KOE_REQUIRE((long long)a->sample_offset +
                        ((long long)a->frame_offset + (long long)(a->n_frames + 1) * a->frame_step + KOE_MAX_EDGE + 1) *
                            a->hop < (1ll << 31) && a->n_samples < (1 << 30),
                "koe_logmel_power: clip too long for 32-bit sample indices");
    KOE_REQUIRE(a->pad_mode == 0 || a->pad_mode == 1, "koe_logmel_power: pad_mode must be 0 (constant) or 1 (reflect)");
    KOE_REQUIRE(a->pad_mode == 0 || (a->lo_rel_hops == KOE_NO_EDGE && a->hi_rel_hops == KOE_NO_EDGE &&
                                     a->n_samples > KOE_N_FFT / 2),
                "koe_logmel_power: reflect padding needs n_samples > n_fft/2 and no window edges");
    KOE_REQUIRE(a->power_clip_stride >= (int64_t)a->n_frames * KOE_N_MELS && a->power_clip_stride % 4 == 0,
                "koe_logmel_power: bad power_clip_stride");
    KOE_REQUIRE(a->frame_max == nullptr || a->frame_max_clip_stride >= a->n_frames,
                "koe_logmel_power: bad frame_max_clip_stride");
    KOE_REQUIRE(a->power_b == nullptr || (a->frame_max == nullptr) == (a->frame_max_b == nullptr),
                "koe_logmel_power_ex: power_b needs frame_max_b whenever frame_max is given");
    pairs = (long long)a->n_clips * ((a->n_frames + 1) / 2);
  }
  KOE_REQUIRE(pairs < (1ll << 31) - kWarps, "koe_logmel_power: more than 2^31 frame pairs in one call");
  FrontendTables tab;
  LogmelParams p;
  launch_setup(fe, a, follows_frontend_launch, &tab, &p);
  int sms = 0;
  KOE_CUDA(sm_count(&sms));
  const long long n_blocks = (pairs + kWarps - 1) / kWarps;
  const int grid = (int)std::min<long long>(n_blocks, sms);
  if (mode == FrontendMode::Varlen) {
    p.vl_sample_off = vl->sample_off;
    p.vl_length = vl->length;
    p.vl_pair_base = vl->pair_base;
    p.vl_row_base = vl->row_base;
    p.vl_clips = vl->n_clips;
    p.vl_pairs = (unsigned)pairs;
    return launch_power(mode, fe->default_bank, tab, p, grid, (cudaStream_t)stream);
  }
  const int ppc = (p.n_frames + 1) / 2;
  while (p.edge_lo < ppc && !pair_geometry(p, 0, p.edge_lo).interior) ++p.edge_lo;
  while (p.edge_lo + p.edge_hi < ppc && !pair_geometry(p, 0, ppc - 1 - p.edge_hi).interior) ++p.edge_hi;
  if (p.edge_lo + p.edge_hi > 0 && p.edge_lo + p.edge_hi < ppc) {
    p.mid_pairs = ppc - p.edge_lo - p.edge_hi;
    const long long step = (long long)grid * kWarps;
    p.step_clips = (int)(step / p.mid_pairs);
    p.step_pairs = (int)(step % p.mid_pairs);
  }
  // Early release of the core: the clips [0, early->clips) are complete once every pair ahead of clip `early->clips` in
  // the launch order is stored -- all edge pairs (they come first) and the interior pairs of those clips -- i.e. once
  // every CTA has finished its iterations below early_iters.  Only the warp-specialised kernel signals; every CTA must own
  // an iteration below the threshold and one at or above it.
  if (early != nullptr && early->flag != nullptr && early->clips > 0 && early->clips < a->n_clips &&
      mode == FrontendMode::Frames && fe->default_bank) {
    const long long before = p.mid_pairs > 0
                                 ? (long long)a->n_clips * (p.edge_lo + p.edge_hi) + (long long)early->clips * p.mid_pairs
                                 : (long long)early->clips * ppc;
    const long long iters = (before + kWarps - 1) / kWarps;
    if (iters >= grid && iters + grid <= n_blocks) {
      p.early_flag = early->flag;
      p.early_iters = (unsigned)iters;
      early->target = (unsigned)grid * kWsConsumers;  // one arrival per consumer warp
    }
  }
  return launch_power(mode, fe->default_bank, tab, p, grid, (cudaStream_t)stream);
}

extern "C" int koe_logmel_power(const koe_frontend_t* fe, const float* audio, int64_t audio_stride, int n_clips,
                                int n_samples, int hop, int n_frames, int frame_offset, int frame_step,
                                int lo_rel_hops, int hi_rel_hops, float* power, float* frame_max, void* stream) {
  koe_logmel_args a = {};
  a.audio = audio;
  a.audio_stride = audio_stride;
  a.n_clips = n_clips;
  a.n_samples = n_samples;
  a.hop = hop;
  a.n_frames = n_frames;
  a.frame_offset = frame_offset;
  a.frame_step = frame_step;
  a.sample_offset = 0;
  a.lo_rel_hops = lo_rel_hops;
  a.hi_rel_hops = hi_rel_hops;
  a.pad_mode = 0;
  a.power = power;
  a.power_clip_stride = (int64_t)n_frames * KOE_N_MELS;
  a.frame_max = frame_max;
  a.frame_max_clip_stride = n_frames;
  return koe_logmel_power_ex(fe, &a, stream);
}

extern "C" int koe_logmel_normalise(const float* power, const float* frame_max, int n_clips, int n_frames,
                                    int db_only, float* long_term, float* short_term, void* stream) {
  KOE_REQUIRE(power != nullptr && frame_max != nullptr && long_term != nullptr,
              "koe_logmel_normalise: NULL argument");
  KOE_REQUIRE(n_clips >= 0 && n_frames >= 0, "koe_logmel_normalise: negative size");
  KOE_REQUIRE(((reinterpret_cast<uintptr_t>(power) | reinterpret_cast<uintptr_t>(long_term)) & 15) == 0,
              "koe_logmel_normalise: buffers must be 16-byte aligned");
  if (n_clips == 0) return KOE_OK;
  logmel_normalise_kernel<<<n_clips, 256, 0, (cudaStream_t)stream>>>(power, frame_max, n_frames, db_only, long_term,
                                                                      short_term);
  count_launch();
  KOE_CUDA(cudaGetLastError());
  return KOE_OK;
}

// ---- 16-bit PCM host format: what a WAV file holds; halves the PCIe bytes of the host-buffer path ----------------------
namespace koe {
// eight samples per thread per step: one 16-byte load, two 16-byte streaming stores
__global__ void __launch_bounds__(256) pcm16_to_float_kernel(const int16_t* __restrict__ pcm, long long n,
                                                              float* __restrict__ audio) {
  constexpr float kScale = 1.0f / 32768.0f;  // libsndfile's int16 -> float normalisation (sf.read(dtype="float32"))
  const long long n8 = n >> 3;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
    const int4 w = __ldcs(reinterpret_cast<const int4*>(pcm) + i);
    const int word[4] = {w.x, w.y, w.z, w.w};
    float f[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      f[2 * k] = (float)(short)(word[k] & 0xffff) * kScale;
      f[2 * k + 1] = (float)(word[k] >> 16) * kScale;
    }
    float4* dst = reinterpret_cast<float4*>(audio) + 2 * i;
    dst[0] = make_float4(f[0], f[1], f[2], f[3]);
    dst[1] = make_float4(f[4], f[5], f[6], f[7]);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 7)) audio[(n8 << 3) + threadIdx.x] = (float)pcm[(n8 << 3) + threadIdx.x] * kScale;
}
}  // namespace koe

extern "C" int koe_pcm16_to_float(const int16_t* pcm, int64_t n_samples, float* audio, void* stream) {
  KOE_REQUIRE(n_samples >= 0, "koe_pcm16_to_float: negative size");
  if (n_samples == 0) return KOE_OK;
  KOE_REQUIRE(pcm != nullptr && audio != nullptr, "koe_pcm16_to_float: NULL argument");
  KOE_REQUIRE(((reinterpret_cast<uintptr_t>(pcm) | reinterpret_cast<uintptr_t>(audio)) & 15) == 0,
              "koe_pcm16_to_float: buffers must be 16-byte aligned");
  int sms = 0;
  KOE_CUDA(koe::sm_count(&sms));
  const long long want = ((n_samples >> 3) + 255) / 256;
  const int grid = (int)std::max<long long>(1, std::min<long long>(want, (long long)sms * 8));
  koe::pcm16_to_float_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(pcm, (long long)n_samples, audio);
  koe::count_launch();
  KOE_CUDA(cudaGetLastError());
  return KOE_OK;
}
