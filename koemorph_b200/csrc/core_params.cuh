// Launch parameters shared by the CUDA-core and the tcgen05 implementations of the dual-stream core.
#pragma once
#include "common.cuh"

namespace koe {

struct CoreParams {
  koe_core_weights w;
  const float* power[1 + 2 * KOE_MAX_EDGE];
  const float* fmax[1 + 2 * KOE_MAX_EDGE];
  int n_edge, n_clips, n_frames, n_out, stride_frames, frames_per_window, mel_seq;
  const float* expr_sigmoid;
  float* out;
  float* sigmoid_out;
  float* attn_out;
  // prenormalised mode (koe_dual_stream_features): rows come from mel_long / mel_short as they are
  const float* mel_long;
  const float* mel_short;
  int n_long;
  // ring mode (koe_dual_stream_ring): plain and lo-edge rows are slots of per-stream rings, the hi-edge row is per stream
  int ring_frames, ring_base;
  // early release (csrc/session.cu): items [0, early_items) may be read once *early_flag >= early_target (acquire); the
  // rest after griddepcontrol.wait.  early_flag == NULL: everything after griddepcontrol.wait, at the start of the kernel.
  // early_flag[1] counts the CTAs that have finished; the last one clears both words for the next forward.
  unsigned* early_flag;
  unsigned early_target;
  int early_items;
  long long* dbg;  // optional phase timestamps of CTA 0 (bring-up / profiling only), NULL in production
  // stream pool (csrc/stream_pool.cu; CoreMode::Pool only): window w reads the rings, edge rows and expression value of
  // stream pool_slot[w] with ring base pool_base[w], and writes output row w
  const int* pool_slot;
  const int* pool_base;
  // packed variable-length batch (csrc/session.cu; CoreMode::Varlen only): n_clips counts output rows (n_out = 1), item
  // is the output row; clip c owns rows [vl_row_base[c], vl_row_base[c + 1]) and its plain rows start at
  // vl_frame_base[c]; vl_plain_only[c] != 0: the clip's windows read every frame from the plain rows
  const int* vl_row_base;
  const int* vl_frame_base;
  const int* vl_plain_only;
  int vl_clips;
  // stream-pool bursts (csrc/stream_pool.cu; CoreMode::PoolHops only): the hops of a koe_stream_pool_push_hops call are
  // staged in call order.  Window w completes at staged hop e = hop_end[w], a hop of stream slot hop_slot[e] whose newest
  // plain row went to ring row hop_row[e]; the window starts hop_base_shift rows after that (mod ring_frames), and its
  // window-end rows (variants 2, 4) are hop e's staged rows: row e * (1 + 2 n_edge) of power[2] / power[4]
  const int* hop_end;
  const int* hop_slot;
  const int* hop_row;
  int hop_base_shift;
  // a warm-up pool's burst (PoolHops): window w has hop_frames[w] frames, 2 .. frames_per_window; a window shorter than
  // frames_per_window starts at its stream's sample 0 and has no window-start variants.  NULL: every window has
  // frames_per_window frames.
  const int* hop_frames;
  // packed batch (Varlen): clip c's first vl_lead_base[c + 1] - vl_lead_base[c] rows are lead windows (warm-up), whose
  // window-end rows (variants 2, 4) are rows vl_lead_base[c] .. of power[2] / power[4]; vl_lead_base == NULL: none.  The
  // rest are the clip's windows, stride_frames apart, whose edge rows start at vl_edge_base[c].
  const int* vl_edge_base;
  const int* vl_lead_base;
};

// Which flavour of the core a launch runs.  Each is a separate instantiation of both kernels (the fp32 kernel has no
// Early), so that adding one leaves the code of the others as it was.
//   Windows  windows of clips, n_out per clip, stride_frames apart; also, by run-time fields of the same instantiation,
//            the streaming step's per-stream rings (ring_frames > 0) and prenormalised features (mel_long != NULL)
//   Early    Windows with one window per clip, released early by the frontend (the fused forward; early_flag)
//   Pool     a stream-pool push: window w reads the rings of stream pool_slot[w] from ring base pool_base[w]
//   Varlen   a packed variable-length batch: output row w belongs to the clip c with vl_row_base[c] <= w < vl_row_base[c + 1];
//            with warm-up the clip's lead windows come first -- the window at grid hop h < W - 1 is the clip's first
//            h + 2 frames, shaped as a PoolHops window below frames_per_window
//   PoolHops a stream-pool burst: window w reads the rings of stream hop_slot[hop_end[w]] (ring_frames rows each) and
//            the window-end rows that hop hop_end[w] staged; on a warm-up pool it has hop_frames[w] frames, and below
//            frames_per_window it is the stream's whole audio so far: plain rows, then the n_edge window-end rows, no
//            window-start rows
enum class CoreMode { Windows, Early, Pool, Varlen, PoolHops };

// frame k of a window: which buffer (variant) holds it (see koe_dual_stream_windows in the header)
__device__ __forceinline__ int window_variant(const CoreParams& p, int k) {
  if (k < p.n_edge) return 1 + 2 * k;
  if (k >= p.frames_per_window - p.n_edge) return 2 + 2 * (p.frames_per_window - 1 - k);
  return 0;
}

// varlen: the clip of output row `item` (row_base[c] <= item < row_base[c + 1]; every clip has a row).  Scalar binary
// search, or -- every lane of a warp calling with the same item -- a 32-ary search with one table load per lane and round.
template <bool kWarp>
__device__ __forceinline__ int varlen_clip(const CoreParams& p, int item) {
  const int* wb = p.vl_row_base;
  int lo = 0, n = p.vl_clips;  // the clip is in [lo, lo + n)
  if constexpr (kWarp) {
    while (n > 1) {
      const int step = (n + 31) >> 5;
      const int i = lo + (int)(threadIdx.x & 31) * step;
      const unsigned m = __ballot_sync(0xffffffffu, i < lo + n && __ldg(wb + i) <= item);  // lane 0 always
      const int k = 31 - __clz(m);
      lo += k * step;
      n = min(step, n - k * step);
    }
  } else {
    while (n > 1) {
      const int half = n >> 1;
      if (__ldg(wb + lo + half) <= item) lo += half, n -= half;
      else n = half;
    }
  }
  return lo;
}

// A window as the row addressing of mode M sees it; CoreRows<M> below is the only code that reads its fields.
struct CoreWindow {
  int owner;        // whose rows: the clip (Windows, Early; ring mode: the stream), the stream slot (Pool, PoolHops), or
                    // the window's first plain row (Varlen)
  int pos;          // where in them: the window within its clip (Windows, Early), the ring base (Pool, PoolHops), or the
                    // window's row in every edge-variant buffer it reads (Varlen)
  bool plain_only;  // Varlen: the clip has no edge variants, every frame comes from the plain rows
  int hop;          // PoolHops: the staged hop at which the window completes (its window-end rows)
  int frames;       // PoolHops, Varlen: the window's frame count
};

// The window resolver of each mode: work item `item` is output row `item` and reads the window window<kWarp>(p, item);
// frame k of it, variant v, is row row(p, w, v, k) of p.power[v] / p.fmax[v].
template <CoreMode M>
struct CoreRows {
  // every window carries its own frame count (CoreWindow::frames), from 2 to frames_per_window
  static constexpr bool kWindowFrames = M == CoreMode::Varlen || M == CoreMode::PoolHops;
  // kWarp: every lane of a converged warp calls with the same item (Varlen searches the clip with the whole warp)
  template <bool kWarp>
  static __device__ __forceinline__ CoreWindow window(const CoreParams& p, int item) {
    if constexpr (M == CoreMode::Pool) {
      return {p.pool_slot[item], p.pool_base[item], false};
    } else if constexpr (M == CoreMode::PoolHops) {
      const int e = p.hop_end[item], T = p.hop_frames != nullptr ? p.hop_frames[item] : p.frames_per_window;
      // frame 0 is T - 2 - lag rows before the hop's newest plain row: hop_base_shift + frames_per_window - T is that
      // distance mod ring_frames, and the sum stays below 2 ring_frames
      const int base = (p.hop_row[e] + p.hop_base_shift + p.frames_per_window - T) % p.ring_frames;
      return {p.hop_slot[e], base, false, e, T};
    } else if constexpr (M == CoreMode::Varlen) {
      const int c = varlen_clip<kWarp>(p, item);
      const int local = item - __ldg(p.vl_row_base + c);
      int lead0 = 0, leads = 0;
      if (p.vl_lead_base != nullptr) lead0 = __ldg(p.vl_lead_base + c), leads = __ldg(p.vl_lead_base + c + 1) - lead0;
      if (local < leads)  // grid hop h = r + local * stride, r = (W - 1) mod stride: T = h + 2 frames from the clip's frame 0
        return {__ldg(p.vl_frame_base + c), lead0 + local, false, 0,
                (p.frames_per_window - 2) % p.stride_frames + local * p.stride_frames + 2};
      const int j = local - leads;  // the clip's window j
      return {__ldg(p.vl_frame_base + c) + j * p.stride_frames, __ldg(p.vl_edge_base + c) + j,
              __ldg(p.vl_plain_only + c) != 0, 0, p.frames_per_window};
    } else {
      return {item / p.n_out, item % p.n_out, false};
    }
  }
  static __device__ __forceinline__ long long row(const CoreParams& p, const CoreWindow& w, int variant, int k) {
    if constexpr (M == CoreMode::Varlen) {
      return variant == 0 ? (long long)w.owner + k : (long long)w.pos;
    } else if constexpr (M == CoreMode::Pool) {
      return variant > 0 && (variant & 1) == 0 ? (long long)w.owner
                                               : (long long)w.owner * p.ring_frames + (w.pos + k) % p.ring_frames;
    } else if constexpr (M == CoreMode::PoolHops) {
      return variant > 0 && (variant & 1) == 0 ? (long long)w.hop * (1 + 2 * p.n_edge)
                                               : (long long)w.owner * p.ring_frames + (w.pos + k) % p.ring_frames;
    } else {
      if (p.ring_frames > 0)  // plain and lo-edge rows are ring slots of the global frame; a hi-edge row (variants 2, 4) is per stream
        return variant > 0 && (variant & 1) == 0 ? (long long)w.owner
                                                 : (long long)w.owner * p.ring_frames + (p.ring_base + k) % p.ring_frames;
      return variant == 0 ? (long long)w.owner * p.n_frames + (long long)w.pos * p.stride_frames + k
                          : (long long)w.owner * p.n_out + w.pos;
    }
  }
  // the window's frame count: T, the launch's frames_per_window, unless kWindowFrames
  static __device__ __forceinline__ int frames(const CoreWindow& w, int T) {
    if constexpr (kWindowFrames) return w.frames;
    return T;
  }
  // whether the window's first n_edge frames have window-start variants (see window_variant); not in a kWindowFrames
  // window shorter than frames_per_window: it starts at sample 0 of its stream or clip, and its plain rows see zeros
  // before that
  static __device__ __forceinline__ bool window_starts(const CoreParams& p, const CoreWindow& w) {
    if constexpr (kWindowFrames) return w.frames == p.frames_per_window;
    return true;
  }
  // frame k of window w with frames(w, T) = T: which buffer (variant) holds it
  static __device__ __forceinline__ int variant(const CoreParams& p, const CoreWindow& w, int T, int k) {
    if constexpr (kWindowFrames) {
      if (T < p.frames_per_window) return k >= T - p.n_edge ? 2 + 2 * (T - 1 - k) : 0;
    }
    return window_variant(p, k);
  }
  // ring modes (ring_frames > 0, n_out == 1): the ring slot of the window's frame 0
  static __device__ __forceinline__ int ring_base(const CoreParams& p, const CoreWindow& w) {
    return M == CoreMode::Pool || M == CoreMode::PoolHops ? w.pos : p.ring_base;
  }
  // ring modes: the stream whose ring and frame maxima window `item` reads (the L2 prefetch of the next window)
  static __device__ __forceinline__ int ring_stream(const CoreParams& p, int item) {
    if constexpr (M == CoreMode::PoolHops) return p.hop_slot[p.hop_end[item]];
    return M == CoreMode::Pool ? p.pool_slot[item] : item;
  }
  // the clip or stream whose expression value (expr_sigmoid) output row `item` takes
  static __device__ __forceinline__ int expr_row(const CoreParams& p, int item) {
    if constexpr (M == CoreMode::PoolHops) return p.hop_slot[p.hop_end[item]];
    return M == CoreMode::Pool ? p.pool_slot[item] : item / p.n_out;
  }
  // the L2 policy of a window's plain rows: `reread` where other windows read them again (the overlapping windows of a
  // sequence or of a varlen clip), else `once`
  static __device__ __forceinline__ uint64_t plain_rows_policy(const CoreParams& p, uint64_t reread, uint64_t once) {
    return M == CoreMode::Varlen || p.n_out > 1 ? reread : once;
  }
};

// emotion stream launch shared by the public entry and the fused forward (csrc/session.cu, which has it write the
// expression entries of `out`); the core launch that leaves those entries alone (expr_sigmoid == NULL); see dual_stream.cu
// (row_base != NULL: the packed variable-length forward, clip c's output rows are [row_base[c], row_base[c + 1]))
int launch_emotion_stream(const koe_core_weights* w, const float* emo_in, int n_clips, float* expr_sigmoid, float* out,
                          float* sigmoid_out, int n_out, void* stream, bool after_frontend, const int* row_base = nullptr);
int launch_dual_stream_windows(const koe_core_weights* w, const float* const* power, const float* const* frame_max, int n_edge,
                               int n_clips, int n_frames, int n_out, int stride_frames, int frames_per_window,
                               const float* expr_sigmoid, float* out, float* sigmoid_out, float* attn_out, int precision,
                               void* stream, bool expr_by_emotion_kernel, unsigned* early_flag = nullptr,
                               unsigned early_target = 0, int early_items = 0, bool* early_applied = nullptr);
// the core over the emitting windows of a stream-pool push (csrc/stream_pool.cu): window w is stream slot[w] (device
// table) with ring base base[w]; output row w
int launch_dual_stream_pool(const koe_core_weights* w, const float* const* power, const float* const* frame_max, int n_edge,
                            int n_windows, int ring_frames, const int* slot, const int* base, const float* expr_sigmoid,
                            float* out, int precision, void* stream);
// the core over the windows of a stream-pool burst (csrc/stream_pool.cu): window w completes at staged hop hop_end[w] (device
// tables as CoreParams::hop_*), rings of ring_frames rows, window-end rows power[2], power[4] at row hop * (1 + 2 n_edge);
// output row w; hop_frames != NULL (a warm-up pool): window w has hop_frames[w] frames (CoreParams::hop_frames)
int launch_dual_stream_pool_hops(const koe_core_weights* w, const float* const* power, const float* const* frame_max,
                                 int n_edge, int n_windows, int ring_frames, const int* hop_end, const int* hop_slot,
                                 const int* hop_row, int hop_base_shift, const int* hop_frames, const float* expr_sigmoid,
                                 float* out, int precision, void* stream);
// the core over the rows of a packed variable-length batch (csrc/session.cu): output row `item` of the n_rows belongs to
// the clip c with row_base[c] <= item < row_base[c + 1]; the clip's first lead_base[c + 1] - lead_base[c] rows are its
// lead windows (window-end rows power[2], power[4] from lead_base[c]; lead_base == NULL: none), the rest its windows j =
// 0, 1, .. with plain rows from frame_base[c] + j * stride_frames and edge rows at edge_base[c] + j unless plain_only[c];
// expression entries are written by the emotion kernel
int launch_dual_stream_varlen(const koe_core_weights* w, const float* const* power, const float* const* frame_max,
                              int n_edge, int n_rows, int n_frames, int stride_frames, int frames_per_window, int n_clips,
                              const int* row_base, const int* frame_base, const int* edge_base, const int* lead_base,
                              const int* plain_only, float* out, float* sigmoid_out, float* attn_out, int precision,
                              void* stream);
// segmented EMA of a packed variable-length batch: clip c's frames are rows [row_base[c], row_base[c + 1]) of `frames`
int launch_ema_scan_varlen(float* frames, int n_clips, const int* row_base, float alpha, void* stream);
// how many SMs' worth of CTAs the tensor-core core launches for n_items windows (the early-release split follows it)
int dual_stream_tc_grid(int n_items);

}  // namespace koe
