// One streaming step as ONE native call: the hop-aligned sliding window of scripts/rt.py:465-519 /
// SimplifiedDualStreamModel.process_audio_frame_realtime (src/model/simplified_dual_stream_model.py:452-500) for many
// lock-step streams.  The Python driver used to issue the step as a tensor concatenation, three frontend calls, the core
// call and the smoothing call: six kernels but ~150 us of interpreter / ctypes / allocator time per hop, a third of the
// latency of 4096 streams and nearly all of it for a handful.  Here the five launches are queued back to back from C++.
//
// State per stream (all caller-owned device memory, see koe_stream_args): the last n_fft/2 + hop samples (two buffers,
// ping-pong: step n reads tail[n & 1] and writes tail[(n + 1) & 1]), rings of W plain (F) and "window starts here" (R)
// mel rows with their per-frame maxima, one "window ends here" row (L), the smoothing state.  SURVEY.md section 8
// note E: frame n is centred on sample n * hop; R[n] is the same frame with everything before its centre zeroed; L[n + 1]
// is centred on (n + 1) * hop with everything from there on zeroed.
#include <algorithm>
#include <map>
#include <mutex>
#include <utility>

#include "core_params.cuh"

namespace koe {

// new_tail[s] = [old_tail[s][hop:], hop_audio[s]]: one CTA per stream row (strided over the grid), no index division
__global__ void __launch_bounds__(256) stream_tail_shift_kernel(const float* __restrict__ old_tail,
                                                               const float* __restrict__ hop_audio, int n_streams,
                                                               int tail_len, int hop, float* __restrict__ new_tail) {
  const int keep = tail_len - hop;
  for (int s = blockIdx.x; s < n_streams; s += gridDim.x) {
    const float* o = old_tail + (long long)s * tail_len + hop;
    const float* x = hop_audio + (long long)s * hop;
    float* t = new_tail + (long long)s * tail_len;
    for (int k = threadIdx.x; k < keep; k += blockDim.x) t[k] = o[k];
    for (int k = threadIdx.x; k < hop; k += blockDim.x) t[keep + k] = __ldcs(x + k);
  }
}

// The tail ends at sample (n + 1) * hop.  The newest frame whose samples are all there is global frame g = n - lag,
// lag = n_edge - 1, centred `half` samples into the tail; the frames centred one hop further each are the window-end
// variants of the window that ends now: beyond the end of the tail the clip reads as zeros, which is exactly their mask.
int launch_hop_frontend(const koe_frontend_t* fe, const float* tail, int n_streams, int tail_len, int half, int hop,
                        int n_edge, const MelRows* rows, void* stream) {
  koe_logmel_args f = {};
  f.audio = tail;
  f.audio_stride = tail_len;
  f.n_clips = n_streams;
  f.n_samples = tail_len;
  f.hop = hop;
  f.frame_offset = 0;
  f.frame_step = 1;
  f.pad_mode = 0;
  f.sample_offset = half;
  f.lo_rel_hops = KOE_NO_EDGE, f.hi_rel_hops = KOE_NO_EDGE;
  auto to = [&f](const MelRows& r) {
    f.power = r.power, f.power_clip_stride = r.power_stride;
    f.frame_max = r.frame_max, f.frame_max_clip_stride = r.fmax_stride;
  };
  // plain frame g and the frame one hop later as ONE pair of one launch: at 30 fps that second frame is the window-end
  // variant L0 (centred on the tail's end), at 60 fps the last-but-one frame of the window (L1)
  const MelRows& second = rows[n_edge == 1 ? 2 : 4];
  f.n_frames = 2;
  to(rows[0]);
  f.power_b = second.power, f.power_b_clip_stride = second.power_stride;
  f.frame_max_b = second.frame_max, f.frame_max_b_clip_stride = second.fmax_stride;
  if (int rc = launch_logmel(fe, &f, FrontendMode::SplitPairs, /*follows_frontend_launch=*/false, stream)) return rc;
  f.power_b = nullptr, f.frame_max_b = nullptr;
  f.n_frames = 1;
  if (n_edge == 2) {  // the frame centred on the tail's end: the window's last frame
    f.frame_offset = 2;
    to(rows[2]);
    if (int rc = launch_logmel(fe, &f, FrontendMode::Frames, /*follows_frontend_launch=*/false, stream)) return rc;
    f.frame_offset = 0;
  }
  // window-start variants of frame g: nothing before its centre (first frame of the window that starts at g), and at
  // 60 fps nothing before the centre of frame g - 1 (second frame of the window that starts at g - 1)
  for (int m = 0; m < n_edge; ++m) {
    f.lo_rel_hops = -m;
    to(rows[1 + 2 * m]);
    if (int rc = launch_logmel(fe, &f, FrontendMode::Frames, /*follows_frontend_launch=*/false, stream)) return rc;
  }
  return KOE_OK;
}

}  // namespace koe

using namespace koe;

extern "C" int koe_stream_push(const koe_stream_args* a, int* emitted, void* stream_v) {
  KOE_REQUIRE(a != nullptr && emitted != nullptr, "koe_stream_push: NULL argument");
  KOE_REQUIRE(a->frontend != nullptr && a->weights != nullptr, "koe_stream_push: NULL frontend / weights");
  KOE_REQUIRE(a->n_streams >= 0 && a->hop > 0 && a->window_frames > 0 && a->half_fft > 0 && a->step >= 0,
              "koe_stream_push: bad geometry");
  // frames within n_fft/2 of a window edge see zeros beyond it: ceil(half / hop) frames per side (1 at 30 fps, 2 at 60 fps)
  const int n_edge = (a->half_fft + a->hop - 1) / a->hop;
  KOE_REQUIRE(n_edge >= 1 && n_edge <= KOE_MAX_EDGE, "koe_stream_push: hop %d needs %d edge frames per window side (max %d)",
              a->hop, n_edge, KOE_MAX_EDGE);
  KOE_REQUIRE(a->hop_audio && a->tail[0] && a->tail[1] && a->ring_f && a->fmax_f && a->ring_r && a->fmax_r && a->row_l &&
                  a->fmax_l && a->expr_sigmoid && a->out,
              "koe_stream_push: NULL buffer");
  KOE_REQUIRE(n_edge == 1 || (a->ring_r2 && a->fmax_r2 && a->row_l2 && a->fmax_l2),
              "koe_stream_push: hop < n_fft/2 needs the second edge buffers (ring_r2, row_l2)");
  *emitted = 0;
  if (a->n_streams == 0) return KOE_OK;
  cudaStream_t stream = (cudaStream_t)stream_v;
  const int S = a->n_streams, hop = a->hop, W = a->window_frames, half = a->half_fft, tail_len = half + n_edge * hop;
  const int64_t n = a->step;
  const float* old_tail = a->tail[n & 1];
  float* tail = a->tail[(n + 1) & 1];
  {
    int sms = 0;
    KOE_CUDA(sm_count(&sms));
    const int grid = std::min(S, sms * 8);
    stream_tail_shift_kernel<<<grid, 256, 0, stream>>>(old_tail, a->hop_audio, S, tail_len, hop, tail);
    count_launch();
    KOE_CUDA(cudaGetLastError());
  }
  // frame g = n - (n_edge - 1) goes to ring slot g mod W (plain and window-start variants), the window-end variants to the
  // stream's own row
  const int64_t g = n - (n_edge - 1);
  const int slot = (int)(((g % W) + W) % W);
  float* const power[1 + 2 * KOE_MAX_EDGE] = {a->ring_f, a->ring_r, a->row_l, a->ring_r2, a->row_l2};
  float* const fmax[1 + 2 * KOE_MAX_EDGE] = {a->fmax_f, a->fmax_r, a->fmax_l, a->fmax_r2, a->fmax_l2};
  MelRows rows[1 + 2 * KOE_MAX_EDGE] = {};
  for (int v = 0; v < 1 + 2 * n_edge; ++v) {
    if (v > 0 && v % 2 == 0)
      rows[v] = {power[v], fmax[v], KOE_N_MELS, 1};
    else
      rows[v] = {power[v] + (size_t)slot * KOE_N_MELS, fmax[v] + slot, (int64_t)W * KOE_N_MELS, W};
  }
  if (int rc = launch_hop_frontend(a->frontend, tail, S, tail_len, half, hop, n_edge, rows, stream)) return rc;
  if (n + 1 < W) return KOE_OK;  // the context is not full yet
  const int base = (int)((n + 1 - W) % W);  // ring slot of the first frame of the window that ends now
  if (int rc = koe_dual_stream_ring_edges(a->weights, power, fmax, n_edge, S, W, base, W + 1, a->expr_sigmoid, a->out,
                                          nullptr, nullptr, a->precision, stream))
    return rc;
  if (a->ema_state != nullptr)
    if (int rc = koe_ema_scan(a->out, S, 1, a->alpha, a->ema_state, a->has_state, stream)) return rc;
  *emitted = 1;
  return KOE_OK;
}

// ---- early release of the core ------------------------------------------------------------------------------------------
// With one window per clip the core's CTA b handles clips b, b + G, b + 2G, ... (G = its grid).  The frontend stores the
// clips in index order, so all but the last round of windows can be read long before the frontend's slowest CTA has
// finished -- and the core's CTAs become resident exactly then, as the frontend's first CTAs leave.  The frontend's
// consumer warps count up a flag when the first E = G * floor((n - 1) / G) clips are stored; the core acquires it instead
// of waiting for the whole frontend, and executes griddepcontrol.wait only before its last round (step 199.1 -> 191.9 us
// at most, measured with a probe that did not wait at all).  The flag and the core's exit counter live in two words per
// (device, stream), zero between forwards: the last core CTA out clears them.
namespace {
struct EarlyFlags {
  static constexpr int kPool = 64;   // word pairs per device, allocated (and zeroed) at the first use outside a capture
  std::mutex mu;
  std::map<std::pair<int, void*>, unsigned*> words;
  std::map<int, std::pair<unsigned*, int>> pool;   // device -> (block, pairs handed out)
  unsigned* get(void* stream) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    std::lock_guard<std::mutex> lock(mu);
    auto it = words.find({dev, stream});
    if (it != words.end()) return it->second;
    auto pl = pool.find(dev);
    if (pl == pool.end()) {
      // (no allocation inside a stream capture: a forward captured before any eager one takes the plain chain)
      cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
      if (cudaStreamIsCapturing((cudaStream_t)stream, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) return nullptr;
      unsigned* block = nullptr;
      if (cudaMalloc(&block, kPool * 2 * sizeof(unsigned)) != cudaSuccess) return nullptr;
      if (cudaMemset(block, 0, kPool * 2 * sizeof(unsigned)) != cudaSuccess) {
        cudaFree(block);
        return nullptr;
      }
      pl = pool.emplace(dev, std::make_pair(block, 0)).first;
    }
    if (pl->second.second >= kPool) return nullptr;   // more streams than pairs: those forwards take the plain chain
    unsigned* w = pl->second.first + 2 * pl->second.second++;
    words[{dev, stream}] = w;
    return w;
  }
};
EarlyFlags g_early;
}  // namespace

// ---- the batch forward as one native call (see koe_forward_windows in the header) ------------------------------------
extern "C" int koe_forward_windows(const koe_forward_args* a, void* stream) {
  KOE_REQUIRE(a != nullptr && a->frontend != nullptr && a->weights != nullptr, "koe_forward_windows: NULL argument");
  KOE_REQUIRE(a->audio && a->egemaps && a->power[0] && a->frame_max[0] && a->expr_sigmoid && a->out,
              "koe_forward_windows: NULL buffer");
  KOE_REQUIRE(a->n_clips >= 0 && a->n_samples >= 0 && a->hop > 0 && a->n_out >= 1 && a->stride_frames >= 1 &&
                  a->frames_per_window >= 1 && a->n_edge >= 0 && a->n_edge <= KOE_MAX_EDGE,
              "koe_forward_windows: bad geometry");
  KOE_REQUIRE((long long)(a->n_out - 1) * a->stride_frames + a->frames_per_window <= a->n_frames,
              "koe_forward_windows: windows run past n_frames");
  if (a->n_clips == 0) return KOE_OK;
  koe_logmel_args f = {};
  f.audio = a->audio;
  f.audio_stride = a->audio_stride;
  f.n_clips = a->n_clips;
  f.n_samples = a->n_samples;
  f.hop = a->hop;
  f.pad_mode = 0;
  f.sample_offset = 0;
  // every global frame once
  f.n_frames = a->n_frames;
  f.frame_offset = 0, f.frame_step = 1;
  f.lo_rel_hops = KOE_NO_EDGE, f.hi_rel_hops = KOE_NO_EDGE;
  f.power = a->power[0], f.power_clip_stride = (int64_t)a->n_frames * KOE_N_MELS;
  f.frame_max = a->frame_max[0], f.frame_max_clip_stride = a->n_frames;
  // early release of the core (above): one window per clip, tensor-core core, no attention output, more than one round
  static const bool early_off = getenv("KOE_NO_EARLY_CORE") != nullptr;  // experiment switch
  EarlyRelease early = {0, nullptr, 0};
  if (!early_off && a->n_out == 1 && a->n_edge == 0 && a->precision == 2 && a->attn_out == nullptr &&
      (a->weights->k_mel == 259 || a->weights->k_mel == 515)) {
    const int G = dual_stream_tc_grid(a->n_clips);
    if (G > 0 && a->n_clips > G) {
      early.clips = G * ((a->n_clips - 1) / G);
      early.flag = g_early.get(stream);
    }
  }
  if (int rc = launch_logmel(a->frontend, &f, FrontendMode::Frames, /*follows_frontend_launch=*/false, stream, &early))
    return rc;
  unsigned* const early_flag = early.target != 0 ? early.flag : nullptr;
  bool early_applied = false;
  // the frames within n_fft/2 of a window edge, once per window (SURVEY.md section 8 note E)
  for (int m = 0; m < a->n_edge; ++m) {
    KOE_REQUIRE(a->power[1 + 2 * m] && a->power[2 + 2 * m] && a->frame_max[1 + 2 * m] && a->frame_max[2 + 2 * m],
                "koe_forward_windows: NULL edge buffer");
    f.n_frames = a->n_out;
    f.frame_step = a->stride_frames;
    f.power_clip_stride = (int64_t)a->n_out * KOE_N_MELS, f.frame_max_clip_stride = a->n_out;
    // (these launches follow a frontend launch of this forward and touch none of its buffers: they do not wait for it)
    f.frame_offset = m, f.lo_rel_hops = -m, f.hi_rel_hops = KOE_NO_EDGE;
    f.power = a->power[1 + 2 * m], f.frame_max = a->frame_max[1 + 2 * m];
    if (int rc = launch_logmel(a->frontend, &f, FrontendMode::Frames, /*follows_frontend_launch=*/true, stream)) return rc;
    f.frame_offset = a->frames_per_window - 1 - m, f.lo_rel_hops = KOE_NO_EDGE, f.hi_rel_hops = m;
    f.power = a->power[2 + 2 * m], f.frame_max = a->frame_max[2 + 2 * m];
    if (int rc = launch_logmel(a->frontend, &f, FrontendMode::Frames, /*follows_frontend_launch=*/true, stream)) return rc;
  }
  // The mouth entries of every output row come from the mel stream (the core) and the expression entries from the emotion
  // stream alone, so the two kernels do not depend on each other's results: the emotion kernel writes its entries of `out`
  // itself and the core skips them.  The kernel queued last is a frontend launch; the emotion stream (which reads none of
  // its outputs) runs on the SMs the frontend's first CTAs leave, the core sets itself up behind both.
  if (int rc = launch_emotion_stream(a->weights, a->egemaps, a->n_clips, a->expr_sigmoid, a->out, a->sigmoid_out, a->n_out,
                                     stream, /*after_frontend=*/true)) {
    if (early_flag != nullptr) cudaMemsetAsync(early_flag, 0, 2 * sizeof(unsigned), (cudaStream_t)stream);
    return rc;
  }
  if (int rc = launch_dual_stream_windows(a->weights, a->power, a->frame_max, a->n_edge, a->n_clips, a->n_frames, a->n_out,
                                          a->stride_frames, a->frames_per_window, nullptr, a->out, a->sigmoid_out,
                                          a->attn_out, a->precision, stream, /*expr_by_emotion_kernel=*/true, early_flag,
                                          early.target, early.clips, &early_applied)) {
    if (early_flag != nullptr) cudaMemsetAsync(early_flag, 0, 2 * sizeof(unsigned), (cudaStream_t)stream);  // frontend counted, nobody clears
    return rc;
  }
  // (the frontend counted but the core took the plain kernel: the flag must not survive this forward)
  if (early_flag != nullptr && !early_applied) KOE_CUDA(cudaMemsetAsync(early_flag, 0, 2 * sizeof(unsigned), (cudaStream_t)stream));
  if (a->smooth && a->n_out > 1)
    if (int rc = koe_ema_scan(a->out, a->n_clips, a->n_out, a->alpha, nullptr, 0, stream)) return rc;
  return KOE_OK;
}

// ---- packed variable-length batch (see koe_forward_varlen and koe_forward_varlen_ex in the header) ----------------------
// Per-clip tables, int32 words (the int64 sample offsets first, so that they are 8-byte aligned):
//   sample_off [B] int64 | length [B] | frame_base [B + 1] | window_base [B + 1] | pair_base [B + 1] | edge_pair_base [B + 1]
//   | plain_only [B]
// and with KOE_VARLEN_WARMUP | row_base [B + 1] | lead_base [B + 1] | lead_pair_base [B + 1].
// pair_base counts the frame pairs of the plain launch (ceil(n_frames_c / 2) per clip), edge_pair_base those of each
// edge-variant launch (ceil(n_out_c / 2), none for a clip that reads its window from the plain rows).  Warm-up: clip c
// has K_c lead windows (the grid hops h <= min(W - 2, n_c - 1)) and its steady windows (n_out_c when n_c >= W, else
// none); row_base is the first output row, lead_base the first lead row of the window-end buffers, lead_pair_base counts
// the frame pairs of each lead-variant launch (ceil(K_c / 2)).  The plain and edge-variant launches and their tables are
// those of the plain call.
// Workspace (16-byte aligned regions): power[0] [F][80] | power[1 .. 2 n_edge] [N][80] each | frame_max[0] [F] |
// frame_max[1 .. 2 n_edge] [N] each | tables.  Warm-up: the window-end buffers power[2 + 2m] / frame_max[2 + 2m] hold the
// Sum K_c lead rows after their N steady rows (N = 0 when no clip uses steady edge variants), and there are as many
// variant buffers as the steady or the lead windows need.
namespace {
constexpr int kVarlenTableWords = 8;      // table words per clip (+ 4)
constexpr int kWarmupTableWords = 3;      // more with KOE_VARLEN_WARMUP (+ 3)

struct VarlenPlan {
  int n_edge = 0;            // edge variants per window side of the steady windows (0: no clip uses them)
  int lead_edge = 0;         // window-end variants of the lead windows (0: no clip has one)
  int max_out = 0;           // most output rows of one clip
  long long windows = 0, frames = 0, pairs = 0, edge_pairs = 0;
  long long rows = 0, leads = 0, lead_pairs = 0;  // output rows; warm-up: lead windows and their frame pairs per launch
  size_t off_power[1 + 2 * KOE_MAX_EDGE] = {}, off_fmax[1 + 2 * KOE_MAX_EDGE] = {}, off_tables = 0, bytes = 0;
  size_t table_words = 0;
};

size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

// Validates the lengths and geometry of `a`, sums up the per-clip geometry (the rules of SequentialDualStreamModel; with
// `warm`, the grid of KOE_VARLEN_WARMUP) and lays out the workspace; with tables != NULL also writes the per-clip tables.
int plan_varlen(const koe_forward_varlen_args* a, bool warm, VarlenPlan* pl, int32_t* tables) {
  KOE_REQUIRE(a != nullptr && pl != nullptr, "koe_forward_varlen: NULL argument");
  KOE_REQUIRE(a->n_clips >= 0 && (a->n_clips == 0 || a->lengths_host != nullptr), "koe_forward_varlen: bad n_clips / lengths");
  KOE_REQUIRE(a->n_clips < (1 << 26), "koe_forward_varlen: %d clips (at most 2^26)", a->n_clips);
  KOE_REQUIRE(a->hop > 0 && a->window_frames > 0 && a->stride_frames >= 1 && a->half_fft > 0,
              "koe_forward_varlen: bad geometry");
  const int B = a->n_clips, hop = a->hop, W = a->window_frames, stride = a->stride_frames;
  const int n_edge = (a->half_fft + hop - 1) / hop;
  KOE_REQUIRE(n_edge <= KOE_MAX_EDGE && W + 1 > 2 * n_edge,
              "koe_forward_varlen: hop %d needs %d edge frames per window side (max %d)", hop, n_edge, KOE_MAX_EDGE);
  const int r = (W - 1) % stride;  // the first hop of the output grid h = W - 1 (mod stride)
  int64_t* sample_off = nullptr;
  int32_t *length = nullptr, *frame_base = nullptr, *window_base = nullptr, *pair_base = nullptr, *edge_pair_base = nullptr,
          *plain_only = nullptr, *row_base = nullptr, *lead_base = nullptr, *lead_pair_base = nullptr;
  if (tables != nullptr) {
    sample_off = reinterpret_cast<int64_t*>(tables);
    length = tables + 2 * (size_t)B;
    frame_base = length + B;
    window_base = frame_base + B + 1;
    pair_base = window_base + B + 1;
    edge_pair_base = pair_base + B + 1;
    plain_only = edge_pair_base + B + 1;
    if (warm) {
      row_base = plain_only + B;
      lead_base = row_base + B + 1;
      lead_pair_base = lead_base + B + 1;
    }
  }
  *pl = VarlenPlan();
  long long samples = 0;
  bool any_edge = false;
  for (int c = 0; c < B; ++c) {
    if (tables != nullptr) {
      frame_base[c] = (int32_t)pl->frames;
      window_base[c] = (int32_t)pl->windows;
      pair_base[c] = (int32_t)pl->pairs;
      edge_pair_base[c] = (int32_t)pl->edge_pairs;
      if (warm) row_base[c] = (int32_t)pl->rows, lead_pair_base[c] = (int32_t)pl->lead_pairs;
    }
    const int64_t L = a->lengths_host[c];
    KOE_REQUIRE(L >= 0 && L < (1ll << 30), "koe_forward_varlen: length %lld of clip %d outside [0, 2^30)", (long long)L, c);
    // num_output_frames: max(1, floor((L // hop - W) / stride) + 1) -- a negative numerator gives 1 either way
    const long long rel = L / hop - W;
    const long long n_out = rel < 0 ? 1 : rel / stride + 1;
    const long long n_frames = (n_out - 1) * stride + W + 1;
    const bool plain = n_out == 1 && L <= (long long)W * hop;  // one window spanning the whole clip: no interior edges
    // warm-up: the grid hops r, r + stride, .. the clip completes; below W - 1 they are lead windows
    long long leads = 0, clip_rows = n_out;
    if (warm) {
      const long long last_lead = std::min<long long>(W - 2, L / hop - 1);
      leads = last_lead < r ? 0 : (last_lead - r) / stride + 1;
      clip_rows = leads + (rel < 0 ? 0 : n_out);
      KOE_REQUIRE(clip_rows > 0,
                  "koe_forward_varlen_ex: clip %d of %lld samples completes no hop of the output grid (hop %d, first "
                  "output at %d complete hops)", c, (long long)L, hop, r + 1);
    }
    any_edge = any_edge || !plain;
    if (tables != nullptr) {
      sample_off[c] = samples;
      length[c] = (int32_t)L;
      plain_only[c] = plain ? 1 : 0;
      if (warm) lead_base[c] = (int32_t)pl->leads;  // (+ the steady window-end rows, below)
    }
    samples += L;
    pl->windows += n_out;
    pl->frames += n_frames;
    pl->pairs += (n_frames + 1) / 2;
    pl->edge_pairs += plain ? 0 : (n_out + 1) / 2;
    pl->rows += clip_rows;
    pl->leads += leads;
    pl->lead_pairs += (leads + 1) / 2;
    pl->max_out = (int)std::max<long long>(pl->max_out, clip_rows);
    KOE_REQUIRE(pl->frames < (1ll << 31) - 32 && pl->windows < (1ll << 31) && pl->rows < (1ll << 31),
                "koe_forward_varlen: more than 2^31 frames or windows");
  }
  pl->n_edge = any_edge ? n_edge : 0;
  pl->lead_edge = pl->leads > 0 ? n_edge : 0;
  const long long steady_rows = pl->n_edge > 0 ? pl->windows : 0;  // rows of each steady edge-variant buffer
  KOE_REQUIRE(steady_rows + pl->leads < (1ll << 31), "koe_forward_varlen: more than 2^31 edge-variant rows");
  if (tables != nullptr) {
    frame_base[B] = (int32_t)pl->frames;
    window_base[B] = (int32_t)pl->windows;
    pair_base[B] = (int32_t)pl->pairs;
    edge_pair_base[B] = (int32_t)pl->edge_pairs;
    if (warm) {
      row_base[B] = (int32_t)pl->rows, lead_pair_base[B] = (int32_t)pl->lead_pairs;
      for (int c = 0; c < B; ++c) lead_base[c] += (int32_t)steady_rows;
      lead_base[B] = (int32_t)(steady_rows + pl->leads);
    }
  }
  const int n_var = 2 * std::max(pl->n_edge, pl->lead_edge);
  // (window-start variants 1, 3: steady rows only; window-end variants 2, 4: steady rows, then the lead rows)
  auto var_rows = [&](int j) { return (size_t)(steady_rows + (j % 2 == 0 ? pl->leads : 0)); };
  size_t off = 0;
  pl->off_power[0] = off, off += align16((size_t)pl->frames * KOE_N_MELS * sizeof(float));
  for (int j = 1; j <= n_var; ++j) pl->off_power[j] = off, off += align16(var_rows(j) * KOE_N_MELS * sizeof(float));
  pl->off_fmax[0] = off, off += align16((size_t)pl->frames * sizeof(float));
  for (int j = 1; j <= n_var; ++j) pl->off_fmax[j] = off, off += align16(var_rows(j) * sizeof(float));
  pl->table_words = (size_t)kVarlenTableWords * B + 4 + (warm ? (size_t)kWarmupTableWords * B + 3 : 0);
  pl->off_tables = off, off += align16(pl->table_words * sizeof(int32_t));
  pl->bytes = off;
  return KOE_OK;
}

int varlen_flags(int flags, const char* what) {
  KOE_REQUIRE((flags & ~KOE_VARLEN_WARMUP) == 0, "%s: unknown flags 0x%x", what, (unsigned)flags);
  return KOE_OK;
}
}  // namespace

extern "C" int koe_forward_varlen_size_ex(const koe_forward_varlen_args* a, int flags, int64_t* n_windows,
                                          int64_t* n_frames, int64_t* workspace_bytes) {
  KOE_REQUIRE(n_windows != nullptr && n_frames != nullptr && workspace_bytes != nullptr, "koe_forward_varlen_size: NULL argument");
  if (int rc = varlen_flags(flags, "koe_forward_varlen_size_ex")) return rc;
  VarlenPlan pl;
  if (int rc = plan_varlen(a, flags & KOE_VARLEN_WARMUP, &pl, nullptr)) return rc;
  *n_windows = pl.rows, *n_frames = pl.frames, *workspace_bytes = (int64_t)pl.bytes;
  return KOE_OK;
}

extern "C" int koe_forward_varlen_size(const koe_forward_varlen_args* a, int64_t* n_windows, int64_t* n_frames,
                                       int64_t* workspace_bytes) {
  return koe_forward_varlen_size_ex(a, 0, n_windows, n_frames, workspace_bytes);
}

extern "C" int koe_forward_varlen_ex(const koe_forward_varlen_args* a, int flags, void* stream) {
  if (int rc = varlen_flags(flags, "koe_forward_varlen_ex")) return rc;
  const bool warm = flags & KOE_VARLEN_WARMUP;
  VarlenPlan pl;
  if (int rc = plan_varlen(a, warm, &pl, nullptr)) return rc;
  if (a->n_clips == 0) return KOE_OK;
  KOE_REQUIRE(a->frontend != nullptr && a->weights != nullptr, "koe_forward_varlen: NULL frontend / weights");
  KOE_REQUIRE(a->weights->k_mel == a->window_frames + 3, "koe_forward_varlen: weights for k_mel %d, window_frames %d",
              a->weights->k_mel, a->window_frames);
  KOE_REQUIRE(a->audio && a->egemaps && a->workspace && a->out, "koe_forward_varlen: NULL buffer");
  KOE_REQUIRE((reinterpret_cast<uintptr_t>(a->workspace) & 15) == 0, "koe_forward_varlen: workspace must be 16-byte aligned");
  KOE_REQUIRE(a->workspace_bytes >= (int64_t)pl.bytes, "koe_forward_varlen: workspace of %lld bytes, %lld needed",
              (long long)a->workspace_bytes, (long long)pl.bytes);
  KOE_REQUIRE(!a->smooth || (a->alpha >= 0.0f && a->alpha <= 1.0f), "koe_forward_varlen: alpha must be in [0, 1]");
  KOE_REQUIRE(a->precision == 0 || a->precision == 2, "koe_forward_varlen: precision must be 0 or 2");
  if (!koe_frontend_uses_unrolled_bank(a->frontend))
    return fail(KOE_E_UNSUPPORTED, "koe_forward_varlen: implemented for the default filterbank only");
  if (int rc = check_capture(stream, "koe_forward_varlen")) return rc;
  const int B = a->n_clips;
  const int core_edge = std::max(pl.n_edge, pl.lead_edge);
  char* ws = static_cast<char*>(a->workspace);
  float* power[1 + 2 * KOE_MAX_EDGE] = {};
  float* fmax[1 + 2 * KOE_MAX_EDGE] = {};
  for (int j = 0; j <= 2 * core_edge; ++j)
    power[j] = reinterpret_cast<float*>(ws + pl.off_power[j]), fmax[j] = reinterpret_cast<float*>(ws + pl.off_fmax[j]);
  int32_t* dev_tables = reinterpret_cast<int32_t*>(ws + pl.off_tables);
  const size_t words = pl.table_words;
  TableStaging* stage = nullptr;
  if (int rc = acquire_table_staging(stream, words, &stage)) return rc;
  if (int rc = plan_varlen(a, warm, &pl, stage->host)) return rc;
  if (int rc = upload_tables(stage, dev_tables, words, (cudaStream_t)stream)) return rc;
  const long long* sample_off = reinterpret_cast<const long long*>(dev_tables);
  const int* length = dev_tables + 2 * (size_t)B;
  const int* frame_base = length + B;
  const int* window_base = frame_base + B + 1;
  const int* pair_base = window_base + B + 1;
  const int* edge_pair_base = pair_base + B + 1;
  const int* plain_only = edge_pair_base + B + 1;
  const int* row_base = warm ? plain_only + B : window_base;  // each clip's first output row
  const int* lead_base = row_base + B + 1;                    // (warm-up only)
  const int* lead_pair_base = lead_base + B + 1;
  const int T = a->window_frames + 1;

  koe_logmel_args f = {};
  f.audio = a->audio;
  f.hop = a->hop;
  f.frame_offset = 0, f.frame_step = 1;
  f.lo_rel_hops = KOE_NO_EDGE, f.hi_rel_hops = KOE_NO_EDGE;
  f.power = power[0], f.frame_max = fmax[0];
  // every clip's global frames, then the frames within n_fft/2 of a window edge once per window of the clips that use them
  const VarlenTables frames = {sample_off, length, pair_base, frame_base, B, pl.pairs};
  const VarlenTables edges = {sample_off, length, edge_pair_base, window_base, B, pl.edge_pairs};
  if (int rc = launch_logmel(a->frontend, &f, FrontendMode::Varlen, /*follows_frontend_launch=*/false, stream, nullptr,
                             &frames))
    return rc;
  for (int m = 0; m < pl.n_edge; ++m) {
    f.frame_step = a->stride_frames;
    f.frame_offset = m, f.lo_rel_hops = -m, f.hi_rel_hops = KOE_NO_EDGE;
    f.power = power[1 + 2 * m], f.frame_max = fmax[1 + 2 * m];
    if (int rc = launch_logmel(a->frontend, &f, FrontendMode::Varlen, /*follows_frontend_launch=*/true, stream, nullptr,
                               &edges))
      return rc;
    f.frame_offset = T - 1 - m, f.lo_rel_hops = KOE_NO_EDGE, f.hi_rel_hops = m;
    f.power = power[2 + 2 * m], f.frame_max = fmax[2 + 2 * m];
    if (int rc = launch_logmel(a->frontend, &f, FrontendMode::Varlen, /*follows_frontend_launch=*/true, stream, nullptr,
                               &edges))
      return rc;
  }
  // warm-up: the lead window at grid hop h = r + j * stride ends on the window-end variants m < n_edge, frame h + 1 - m
  // with zeros from sample (h + 1) * hop on -- frame j of a launch with frame_offset r + 1 - m
  if (pl.lead_edge > 0) {
    const VarlenTables leads = {sample_off, length, lead_pair_base, lead_base, B, pl.lead_pairs};
    const int r = (a->window_frames - 1) % a->stride_frames;
    for (int m = 0; m < pl.lead_edge; ++m) {
      f.frame_step = a->stride_frames;
      f.frame_offset = r + 1 - m, f.lo_rel_hops = KOE_NO_EDGE, f.hi_rel_hops = m;
      f.power = power[2 + 2 * m], f.frame_max = fmax[2 + 2 * m];
      if (int rc = launch_logmel(a->frontend, &f, FrontendMode::Varlen, /*follows_frontend_launch=*/true, stream, nullptr,
                                 &leads))
        return rc;
    }
  }
  // as in koe_forward_windows: the emotion kernel writes the expression entries of each clip's rows, the core the rest
  if (int rc = launch_emotion_stream(a->weights, a->egemaps, B, nullptr, a->out, a->sigmoid_out, 1, stream,
                                     /*after_frontend=*/true, row_base))
    return rc;
  const float* cpower[1 + 2 * KOE_MAX_EDGE] = {power[0], power[1], power[2], power[3], power[4]};
  const float* cfmax[1 + 2 * KOE_MAX_EDGE] = {fmax[0], fmax[1], fmax[2], fmax[3], fmax[4]};
  if (int rc = launch_dual_stream_varlen(a->weights, cpower, cfmax, core_edge, (int)pl.rows, (int)pl.frames,
                                         a->stride_frames, T, B, row_base, frame_base, window_base,
                                         warm ? lead_base : nullptr, plain_only, a->out, a->sigmoid_out, a->attn_out,
                                         a->precision, stream))
    return rc;
  if (a->smooth && pl.max_out > 1)
    if (int rc = launch_ema_scan_varlen(a->out, B, row_base, a->alpha, stream)) return rc;
  return KOE_OK;
}

extern "C" int koe_forward_varlen(const koe_forward_varlen_args* a, void* stream) { return koe_forward_varlen_ex(a, 0, stream); }
