// Stream pool (koe_stream_pool_* in the header): koe_stream_push for streams that open, close and advance on their own
// clocks.  The kernels never needed lock-step -- every window is computed on its own and every per-stream state (audio
// tail, mel rings, smoothing state, expression value) is stored per stream -- only the addressing did: koe_stream_push
// derives one tail buffer, one ring slot and one ring base from one shared step counter.  Here the pool object keeps a
// clock per slot, and each push hands the kernels small tables built from those clocks:
//   pushing stream i:  slot, ring row (the slot of its newest complete frame), first hop or not
//   emitting stream w: slot, ring base, has smoothing state or not
// A push of n streams queues: the tail update (in place, per slot) with a compact copy of the tails, the frontend
// launches of koe_stream_push on the compact tails into compact staging rows, the scatter of those rows into each slot's
// rings, and -- when at least one stream emits -- the core over the emitting streams only and the smoothing.
//
// Stream n's frames are numbered from its own first hop: the newest complete frame after hop n is g = n - lag (lag =
// n_edge - 1) in ring row g mod R, and the window that ends after hop n starts at ring row (n + 1 - W) mod R -- the
// arithmetic of koe_stream_push, per stream.  R = ring_frames = W + max_hops - 1: W for a pool of koe_stream_pool_create.
//
// A burst (koe_stream_pool_push_hops) advances stream i by counts[i] hops in the same number of launches.  Its hops are
// staged in call order (stream by stream, hops in order); staged hop e gets its own compact tail -- the tail as it is right
// after that hop -- so the frontend runs on exactly the tails, and forms exactly the frame pairs, of one push per hop.  All
// rows of a burst are in the rings before the core reads the burst's first window; that window reaches back W + k - 1 - lag
// rows from the newest one, which is why the rings hold W + max_hops - 1.  Window-end rows are read by the one window that
// completes at their hop only, so the core reads them in the staging rows.  The smoothing runs each stream's frames of the
// call one after the other with the roundings of one push per hop (a scan would round differently).
//
// A warm-up pool (KOE_POOL_WARMUP) emits from every stream's hop 0: the frame at hop h < W - 1 is the forward of
// SimplifiedDualStreamModel on the h + 1 hops heard so far, T = h + 2 frames.  Those are frames 0 .. h + 1 of the
// stream's own clock, which the rings and the hop's staging already hold: plain rows F[0 .. h - lag] in ring rows
// 0 .. h - lag, and the hop's window-end rows for the last n_edge frames (they see zeros from sample (h + 1) hop on, as
// the prefix does).  Every frame before sample 0 reads zeros there too, because a stream's tail starts at zero, so the
// plain rows are the right first frames and no window-start variant is read.  A warm-up pool always runs the burst path
// (koe_stream_pool_push is koe_stream_pool_push_hops with counts of 1), with one more table column (each window's T) for
// the core, and from hop W - 1 on its windows are those of a pool without warm-up.
#include <algorithm>
#include <vector>

#include "core_params.cuh"

struct koe_stream_pool {
  int capacity, hop, window_frames, half_fft, n_edge, tail_len;
  int max_hops, ring_frames;      // hops one stream may advance per call; rows per ring, window_frames + max_hops - 1
  bool warmup;                    // KOE_POOL_WARMUP: every hop emits, from each stream's hop 0 on
  std::vector<unsigned char> open;
  std::vector<int64_t> hops;      // hops pushed since the slot was opened
  std::vector<int64_t> frames;    // frames emitted since the slot was opened
  std::vector<int32_t> row;       // ring row of the newest complete frame after the next hop, (hops - lag) mod R: kept as
                                  // a counter, so that a push of thousands of streams does no division on the host
  std::vector<uint32_t> listed;   // duplicate check: the call that last listed the slot
  uint32_t call = 0;
  std::vector<int32_t> ones;      // koe_stream_pool_push on a pool with max_hops > 1 or warm-up: counts of 1 ...
  std::vector<int64_t> emit_hop;  // ... and the emitting hops it does not return
};

namespace koe {

// pushing stream i: new_tail = [old_tail[hop:], hop_audio[i]] in slot push_slot[i]'s own tail (an opened slot's first
// hop reads the old tail as zeros: this is where a reused slot forgets its previous stream), copied to compact row i for
// the frontend.  One CTA per stream row: read, barrier, write.
__global__ void __launch_bounds__(256) pool_tail_kernel(float* __restrict__ tail, const float* __restrict__ hop_audio,
                                                         const int* __restrict__ push_slot, const int* __restrict__ push_first,
                                                         int n, int tail_len, int hop, float* __restrict__ compact) {
  extern __shared__ float s_tail[];
  const int keep = tail_len - hop;
  for (int i = blockIdx.x; i < n; i += gridDim.x) {
    float* t = tail + (long long)__ldg(push_slot + i) * tail_len;
    const bool first = __ldg(push_first + i) != 0;
    const float* x = hop_audio + (long long)i * hop;
    for (int k = threadIdx.x; k < keep; k += blockDim.x) s_tail[k] = first ? 0.0f : t[hop + k];
    for (int k = threadIdx.x; k < hop; k += blockDim.x) s_tail[keep + k] = __ldcs(x + k);
    __syncthreads();
    float* c = compact + (long long)i * tail_len;
    for (int k = threadIdx.x; k < tail_len; k += blockDim.x) {
      const float v = s_tail[k];
      t[k] = v;
      c[k] = v;
    }
    __syncthreads();
  }
}

struct PoolRings {
  float* power[1 + 2 * KOE_MAX_EDGE];  // plain ring, window-start ring 0, window-end row 0, window-start ring 1, window-end row 1
  float* fmax[1 + 2 * KOE_MAX_EDGE];
};

// staged row v of pushing stream i ([n][V][80], maxima [n][V]) -> ring row push_row[i] of slot push_slot[i] (plain and
// window-start variants) or the slot's own row (window-end variants)
__global__ void __launch_bounds__(256) pool_scatter_kernel(PoolRings r, const float* __restrict__ stage,
                                                            const float* __restrict__ stage_max,
                                                            const int* __restrict__ push_slot,
                                                            const int* __restrict__ push_row, int n, int n_var, int W) {
  constexpr int kQuads = KOE_N_MELS / 4;
  const int total = n * n_var * kQuads;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int q = idx % kQuads, iv = idx / kQuads, v = iv % n_var, i = iv / n_var;
    const long long s = __ldg(push_slot + i);
    const long long row = v > 0 && (v & 1) == 0 ? s : s * W + __ldg(push_row + i);
    reinterpret_cast<float4*>(r.power[v] + row * KOE_N_MELS)[q] = __ldcs(reinterpret_cast<const float4*>(stage) + (long long)iv * kQuads + q);
    if (q == 0) r.fmax[v][row] = __ldcs(stage_max + iv);
  }
}

// smoothing of the emitting streams: the roundings of ema_step_kernel (koe_ema_scan with n_out = 1), with stream
// emit_slot[w]'s state for output row w
__global__ void __launch_bounds__(256) pool_ema_kernel(float* __restrict__ frames, int k, float alpha,
                                                        float* __restrict__ state, const int* __restrict__ emit_slot,
                                                        const int* __restrict__ emit_has_state) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= k * KOE_N_BLENDSHAPES) return;
  const int w = i / KOE_N_BLENDSHAPES, j = i % KOE_N_BLENDSHAPES;
  float* st = state + (long long)__ldg(emit_slot + w) * KOE_N_BLENDSHAPES + j;
  const float x = frames[i];
  const float y = __ldg(emit_has_state + w) ? fmaf(1.0f - alpha, *st, alpha * x) : x;
  frames[i] = y;
  *st = y;
}

__global__ void __launch_bounds__(256) pool_expr_scatter_kernel(const float* __restrict__ compact, const int* __restrict__ slot,
                                                                 int n, float* __restrict__ expr_sigmoid) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < n) expr_sigmoid[__ldg(slot + i)] = compact[i];
}

// ---- bursts (koe_stream_pool_push_hops).  Staged hop e is hop j = e - first[i] of pushing stream i, first[i] <= e <
// first[i + 1] (first[n] = n_hops): hop_audio row e, compact tail e, staging rows e.

// pushing stream i: X = [its old tail (zeros on its first hop) | its hops]; compact tail e = the tail right after hop j,
// X[(j + 1) hop, (j + 1) hop + tail_len); the slot's own tail becomes the one after the stream's last hop.  One CTA per
// stream: the old tail's last tail_len - hop samples to shared memory, barrier, write.
__global__ void __launch_bounds__(256) pool_hops_tail_kernel(float* __restrict__ tail, const float* __restrict__ hop_audio,
                                                              const int* __restrict__ hop_slot, const int* __restrict__ first,
                                                              const int* __restrict__ fresh, int n, int n_hops, int tail_len,
                                                              int hop, float* __restrict__ compact) {
  extern __shared__ float s_old[];  // X[hop, tail_len)
  const int keep = tail_len - hop;
  for (int i = blockIdx.x; i < n; i += gridDim.x) {
    const int e0 = __ldg(first + i), e1 = i + 1 < n ? __ldg(first + i + 1) : n_hops;
    float* t = tail + (long long)__ldg(hop_slot + e0) * tail_len;
    const bool zero = __ldg(fresh + i) != 0;
    for (int k = threadIdx.x; k < keep; k += blockDim.x) s_old[k] = zero ? 0.0f : t[hop + k];
    __syncthreads();
    const float* x = hop_audio + (long long)e0 * hop;  // the stream's hops, back to back
    for (int e = e0; e < e1; ++e) {
      float* c = compact + (long long)e * tail_len;
      for (int k = threadIdx.x; k < tail_len; k += blockDim.x) {
        const int q = (e - e0) * hop + k;  // sample X[hop + q]
        const float v = q < keep ? s_old[q] : __ldg(x + (q - keep));
        c[k] = v;
        if (e == e1 - 1) t[k] = v;
      }
    }
    __syncthreads();
  }
}

// staged rows of hop e ([n_hops][V][80], maxima [n_hops][V]): the plain and window-start variants (0, 1, 3) -> ring row
// hop_row[e] of slot hop_slot[e]; the window-end variants stay in staging, where the core reads them
__global__ void __launch_bounds__(256) pool_hops_scatter_kernel(PoolRings r, const float* __restrict__ stage,
                                                                 const float* __restrict__ stage_max,
                                                                 const int* __restrict__ hop_slot,
                                                                 const int* __restrict__ hop_row, int n_hops, int n_edge,
                                                                 int ring_frames) {
  constexpr int kQuads = KOE_N_MELS / 4;
  const int n_ring = 1 + n_edge, V = 1 + 2 * n_edge;
  const int total = n_hops * n_ring * kQuads;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int q = idx % kQuads, im = idx / kQuads, m = im % n_ring, e = im / n_ring;
    const int v = m == 0 ? 0 : 2 * m - 1;
    const long long row = (long long)__ldg(hop_slot + e) * ring_frames + __ldg(hop_row + e);
    const long long src = (long long)e * V + v;
    reinterpret_cast<float4*>(r.power[v] + row * KOE_N_MELS)[q] = __ldcs(reinterpret_cast<const float4*>(stage) + src * kQuads + q);
    if (q == 0) r.fmax[v][row] = __ldcs(stage_max + src);
  }
}

// smoothing of a burst's frames: a stream's frames of the call are consecutive output rows; thread (w, j), w the first of
// them, runs them in order with the roundings of pool_ema_kernel -- exactly one push per hop.  has_state[w] == 0 only for
// a stream's first frame since it was opened.
__global__ void __launch_bounds__(256) pool_hops_ema_kernel(float* __restrict__ frames, int k, float alpha,
                                                             float* __restrict__ state, const int* __restrict__ hop_end,
                                                             const int* __restrict__ hop_slot,
                                                             const int* __restrict__ has_state) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= k * KOE_N_BLENDSHAPES) return;
  const int w = i / KOE_N_BLENDSHAPES, j = i % KOE_N_BLENDSHAPES;
  const int s = __ldg(hop_slot + __ldg(hop_end + w));
  if (w > 0 && __ldg(hop_slot + __ldg(hop_end + w - 1)) == s) return;  // not the stream's first frame of the call
  float* st = state + (long long)s * KOE_N_BLENDSHAPES + j;
  float y = *st;
  for (int r = w; r < k && (r == w || __ldg(hop_slot + __ldg(hop_end + r)) == s); ++r) {
    float* f = frames + (long long)r * KOE_N_BLENDSHAPES + j;
    const float x = *f;
    y = __ldg(has_state + r) ? fmaf(1.0f - alpha, y, alpha * x) : x;
    *f = y;
  }
  *st = y;
}

// ---- snapshots (koe_stream_pool_snapshot / koe_stream_pool_restore).  A record is a stream's whole state, in the layout
// of the header: rows [V_r][P][80], maxima [V_r][P], tail [tail_len], expression [1], smoothing row [52], zero padding to
// rec_floats (a multiple of 4).  Record row i of variant v is the stream's frame a + 1 - W + i (a: its hops), ring row
// row0 + i (mod R) of its slot; the first `skip` of them are frames < 0, which no window reads: zeros in the record, not
// written back.  Per stream i the tables hold [slot | row0 | skip].  CTA (x, y) copies part x of the records of streams
// y, y + gridDim.y, ...: the rows as float4s, kStateUnroll of them in flight per thread (all loads before any store), then
// the other fields as floats.
constexpr int kStateUnroll = 4;

struct PoolState {
  float* power[1 + KOE_MAX_EDGE];  // plain ring, window-start ring 0, window-start ring 1
  float* fmax[1 + KOE_MAX_EDGE];
  float* tail;
  float* expr;
  float* ema;  // or NULL
  // ring variant v's buffers, selected without indexing the parameter arrays (which would copy them to the stack)
  __device__ __forceinline__ float* ring(int v) const { return v == 0 ? power[0] : v == 1 ? power[1] : power[2]; }
  __device__ __forceinline__ float* ring_max(int v) const { return v == 0 ? fmax[0] : v == 1 ? fmax[1] : fmax[2]; }
};

__global__ void __launch_bounds__(256) pool_snapshot_kernel(PoolState b, const int* __restrict__ tab, int n, int n_ring,
                                                             int P, int R, int tail_len, int rec_floats,
                                                             float* __restrict__ records) {
  constexpr int kQuads = KOE_N_MELS / 4;
  const int quads = n_ring * P * kQuads, rows = n_ring * P;
  const int rest = rec_floats - rows * KOE_N_MELS;  // maxima, tail, expression, smoothing row, padding
  const int t0 = blockIdx.x * blockDim.x + threadIdx.x, dt = gridDim.x * blockDim.x;
  for (int i = blockIdx.y; i < n; i += gridDim.y) {
    const long long s = __ldg(tab + i);
    const int row0 = __ldg(tab + n + i), skip = __ldg(tab + 2 * n + i);
    float* rec = records + (long long)i * rec_floats;
    for (int u0 = t0; u0 < quads; u0 += kStateUnroll * dt) {
      float4 x[kStateUnroll];
#pragma unroll
      for (int k = 0; k < kStateUnroll; ++k) {
        const int u = u0 + k * dt;
        const int q = u % kQuads, vr = u / kQuads, r = vr % P, v = vr / P;
        x[k] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (u < quads && r >= skip) {
          const int rr = row0 + r < R ? row0 + r : row0 + r - R;
          x[k] = __ldcs(reinterpret_cast<const float4*>(b.ring(v) + (s * R + rr) * KOE_N_MELS) + q);
        }
      }
#pragma unroll
      for (int k = 0; k < kStateUnroll; ++k)
        if (u0 + k * dt < quads) __stcs(reinterpret_cast<float4*>(rec) + u0 + k * dt, x[k]);
    }
    float* tail_rec = rec + rows * KOE_N_MELS;
    for (int u = t0; u < rest; u += dt) {
      float x = 0.0f;
      if (u < rows) {
        const int r = u % P, v = u / P;
        const int rr = row0 + r < R ? row0 + r : row0 + r - R;
        if (r >= skip) x = __ldcs(b.ring_max(v) + s * R + rr);
      } else if (u < rows + tail_len) {
        x = __ldcs(b.tail + s * tail_len + (u - rows));
      } else if (u == rows + tail_len) {
        x = b.expr[s];
      } else if (u < rows + tail_len + 1 + KOE_N_BLENDSHAPES && b.ema != nullptr) {
        x = b.ema[s * KOE_N_BLENDSHAPES + (u - rows - tail_len - 1)];
      }
      __stcs(tail_rec + u, x);
    }
  }
}

// the inverse of pool_snapshot_kernel into the slots of the tables: the rows of frames >= 0, the maxima, the tail, the
// expression value and -- when b.ema is non-NULL -- the smoothing row
__global__ void __launch_bounds__(256) pool_restore_kernel(PoolState b, const int* __restrict__ tab, int n, int n_ring,
                                                            int P, int R, int tail_len, int rec_floats,
                                                            const float* __restrict__ records) {
  constexpr int kQuads = KOE_N_MELS / 4;
  const int quads = n_ring * P * kQuads, rows = n_ring * P;
  const int rest = rows + tail_len + 1 + KOE_N_BLENDSHAPES;
  const int t0 = blockIdx.x * blockDim.x + threadIdx.x, dt = gridDim.x * blockDim.x;
  for (int i = blockIdx.y; i < n; i += gridDim.y) {
    const long long s = __ldg(tab + i);
    const int row0 = __ldg(tab + n + i), skip = __ldg(tab + 2 * n + i);
    const float* rec = records + (long long)i * rec_floats;
    for (int u0 = t0; u0 < quads; u0 += kStateUnroll * dt) {
      float4 x[kStateUnroll];
#pragma unroll
      for (int k = 0; k < kStateUnroll; ++k) {
        x[k] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (u0 + k * dt < quads) x[k] = __ldcs(reinterpret_cast<const float4*>(rec) + u0 + k * dt);
      }
#pragma unroll
      for (int k = 0; k < kStateUnroll; ++k) {
        const int u = u0 + k * dt;
        const int q = u % kQuads, vr = u / kQuads, r = vr % P, v = vr / P;
        const int rr = row0 + r < R ? row0 + r : row0 + r - R;
        if (u < quads && r >= skip) reinterpret_cast<float4*>(b.ring(v) + (s * R + rr) * KOE_N_MELS)[q] = x[k];
      }
    }
    const float* tail_rec = rec + rows * KOE_N_MELS;
    for (int u = t0; u < rest; u += dt) {
      if (u < rows) {
        const int r = u % P, v = u / P;
        const int rr = row0 + r < R ? row0 + r : row0 + r - R;
        if (r >= skip) b.ring_max(v)[s * R + rr] = __ldcs(tail_rec + u);
      } else if (u < rows + tail_len) {
        b.tail[s * tail_len + (u - rows)] = __ldcs(tail_rec + u);
      } else if (u == rows + tail_len) {
        b.expr[s] = __ldcs(tail_rec + u);
      } else if (b.ema != nullptr) {
        b.ema[s * KOE_N_BLENDSHAPES + (u - rows - tail_len - 1)] = __ldcs(tail_rec + u);
      }
    }
  }
}

namespace {
// floats per snapshot record: rows and maxima of 1 + n_edge ring variants for the P = W - n_edge frames a later window
// can still read, the tail, the expression value and the smoothing row, rounded up to whole float4s
int64_t state_floats(const koe_stream_pool* p) {
  const int64_t P = p->window_frames - p->n_edge, rows = (int64_t)(1 + p->n_edge) * P;
  const int64_t f = rows * (KOE_N_MELS + 1) + p->tail_len + 1 + KOE_N_BLENDSHAPES;
  return (f + 3) / 4 * 4;
}

// the grid of both snapshot kernels: enough CTAs per stream for its rows at kStateUnroll float4s per thread (10 at
// 30 fps, 30 at 60 fps), streams over gridDim.y
dim3 state_grid(const koe_stream_pool* p, int n) {
  const int quads = (1 + p->n_edge) * (p->window_frames - p->n_edge) * (KOE_N_MELS / 4);
  const int per_cta = 256 * kStateUnroll;
  return dim3((unsigned)std::max(1, std::min((quads + per_cta - 1) / per_cta, 64)), (unsigned)std::min(n, 65535));
}

PoolState pool_state(const koe_stream_pool_args* a) {
  return PoolState{{a->ring_f, a->ring_r, a->ring_r2}, {a->fmax_f, a->fmax_r, a->fmax_r2}, a->tail, a->expr_sigmoid,
                   a->ema_state};
}

// every slot of slots[0, n) in range, open and listed once
int check_slots(koe_stream_pool* pool, const int32_t* slots, int n, const char* what) {
  KOE_REQUIRE(n >= 0 && n <= pool->capacity, "%s: %d streams for a pool of %d", what, n, pool->capacity);
  KOE_REQUIRE(n == 0 || slots != nullptr, "%s: NULL slots", what);
  if (++pool->call == 0) {  // (the stamp wrapped: forget every earlier call)
    std::fill(pool->listed.begin(), pool->listed.end(), 0u);
    pool->call = 1;
  }
  for (int i = 0; i < n; ++i) {
    const int s = slots[i];
    KOE_REQUIRE(s >= 0 && s < pool->capacity, "%s: slot %d out of range [0, %d)", what, s, pool->capacity);
    KOE_REQUIRE(pool->open[s], "%s: slot %d is not open", what, s);
    KOE_REQUIRE(pool->listed[s] != pool->call, "%s: slot %d listed twice", what, s);
    pool->listed[s] = pool->call;
  }
  return KOE_OK;
}

}  // namespace

}  // namespace koe

using namespace koe;

extern "C" int koe_stream_pool_create_ex2(int capacity, int hop, int window_frames, int half_fft, int max_hops, int flags,
                                          koe_stream_pool_t** out) {
  KOE_REQUIRE(out != nullptr, "koe_stream_pool_create: NULL argument");
  *out = nullptr;
  KOE_REQUIRE((flags & ~KOE_POOL_WARMUP) == 0, "koe_stream_pool_create: unknown flags 0x%x", (unsigned)flags);
  KOE_REQUIRE(capacity >= 1 && capacity <= (1 << 24) && hop > 0 && window_frames > 0 && half_fft > 0,
              "koe_stream_pool_create: bad geometry");
  KOE_REQUIRE(max_hops >= 1 && (int64_t)capacity * max_hops <= (1 << 24) && (int64_t)window_frames + max_hops - 1 <= INT32_MAX,
              "koe_stream_pool_create: max_hops %d for %d streams (need 1 <= max_hops, capacity * max_hops <= 2^24)",
              max_hops, capacity);
  const int n_edge = (half_fft + hop - 1) / hop;
  KOE_REQUIRE(n_edge >= 1 && n_edge <= KOE_MAX_EDGE && window_frames + 1 > 2 * n_edge,
              "koe_stream_pool_create: hop %d needs %d edge frames per window side (max %d)", hop, n_edge, KOE_MAX_EDGE);
  auto* p = new koe_stream_pool();
  p->capacity = capacity, p->hop = hop, p->window_frames = window_frames, p->half_fft = half_fft, p->n_edge = n_edge;
  p->tail_len = half_fft + n_edge * hop;
  p->max_hops = max_hops;
  p->ring_frames = window_frames + max_hops - 1;
  p->warmup = (flags & KOE_POOL_WARMUP) != 0;
  p->open.assign(capacity, 0);
  p->hops.assign(capacity, 0);
  p->frames.assign(capacity, 0);
  p->row.assign(capacity, 0);
  p->listed.assign(capacity, 0);
  if (max_hops > 1 || p->warmup) {
    p->ones.assign(capacity, 1);
    p->emit_hop.assign(capacity, 0);
  }
  *out = p;
  return KOE_OK;
}

extern "C" int koe_stream_pool_create_ex(int capacity, int hop, int window_frames, int half_fft, int max_hops,
                                         koe_stream_pool_t** out) {
  return koe_stream_pool_create_ex2(capacity, hop, window_frames, half_fft, max_hops, 0, out);
}

extern "C" int koe_stream_pool_create(int capacity, int hop, int window_frames, int half_fft, koe_stream_pool_t** out) {
  return koe_stream_pool_create_ex2(capacity, hop, window_frames, half_fft, 1, 0, out);
}

extern "C" int koe_stream_pool_destroy(koe_stream_pool_t* pool) {
  delete pool;
  return KOE_OK;
}

extern "C" int koe_stream_pool_open(koe_stream_pool_t* pool, int n, int32_t* slots_host) {
  KOE_REQUIRE(pool != nullptr && (n == 0 || slots_host != nullptr), "koe_stream_pool_open: NULL argument");
  KOE_REQUIRE(n >= 0, "koe_stream_pool_open: negative count");
  int free_slots = 0;
  for (int s = 0; s < pool->capacity; ++s) free_slots += pool->open[s] ? 0 : 1;
  KOE_REQUIRE(n <= free_slots, "koe_stream_pool_open: %d streams asked, %d of %d slots free", n, free_slots, pool->capacity);
  for (int s = 0, i = 0; i < n; ++s) {
    if (pool->open[s]) continue;
    pool->open[s] = 1;
    pool->hops[s] = 0;
    pool->frames[s] = 0;
    pool->row[s] = (pool->ring_frames - (pool->n_edge - 1)) % pool->ring_frames;
    slots_host[i++] = s;
  }
  return KOE_OK;
}

extern "C" int koe_stream_pool_close(koe_stream_pool_t* pool, int slot) {
  KOE_REQUIRE(pool != nullptr, "koe_stream_pool_close: NULL pool");
  KOE_REQUIRE(slot >= 0 && slot < pool->capacity, "koe_stream_pool_close: slot %d out of range [0, %d)", slot, pool->capacity);
  KOE_REQUIRE(pool->open[slot], "koe_stream_pool_close: slot %d is not open", slot);
  pool->open[slot] = 0;
  return KOE_OK;
}

extern "C" int koe_stream_pool_set_egemaps(koe_stream_pool_t* pool, const koe_stream_pool_args* a, const int32_t* slots_host,
                                           int n, const float* egemaps, void* stream) {
  KOE_REQUIRE(pool != nullptr && a != nullptr, "koe_stream_pool_set_egemaps: NULL argument");
  if (int rc = check_slots(pool, slots_host, n, "koe_stream_pool_set_egemaps")) return rc;
  if (n == 0) return KOE_OK;
  KOE_REQUIRE(a->weights != nullptr && egemaps != nullptr && a->expr_sigmoid != nullptr && a->expr_compact != nullptr &&
                  a->tables != nullptr,
              "koe_stream_pool_set_egemaps: NULL buffer");
  if (int rc = check_capture(stream, "koe_stream_pool_set_egemaps")) return rc;
  TableStaging* b = nullptr;
  if (int rc = acquire_table_staging(stream, (size_t)n, &b)) return rc;
  std::copy(slots_host, slots_host + n, b->host);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = upload_tables(b, a->tables, (size_t)n, st)) return rc;
  if (int rc = launch_emotion_stream(a->weights, egemaps, n, a->expr_compact, nullptr, nullptr, 1, stream, false)) return rc;
  pool_expr_scatter_kernel<<<(n + 255) / 256, 256, 0, st>>>(a->expr_compact, a->tables, n, a->expr_sigmoid);
  count_launch();
  KOE_CUDA(cudaGetLastError());
  return KOE_OK;
}

extern "C" int koe_stream_pool_push(koe_stream_pool_t* pool, const koe_stream_pool_args* a, const int32_t* slots_host, int n,
                                    int32_t* emitted_host, int* n_emitted, void* stream) {
  KOE_REQUIRE(pool != nullptr && a != nullptr && n_emitted != nullptr && emitted_host != nullptr,
              "koe_stream_pool_push: NULL argument");
  *n_emitted = 0;
  if (pool->max_hops > 1 || pool->warmup)  // rings of W + max_hops - 1 rows, or warm-up: a burst of one hop per stream
    return koe_stream_pool_push_hops(pool, a, slots_host, pool->ones.data(), n, emitted_host, pool->emit_hop.data(),
                                     n_emitted, stream);
  if (int rc = check_slots(pool, slots_host, n, "koe_stream_pool_push")) return rc;
  if (n == 0) return KOE_OK;
  const int W = pool->window_frames, n_edge = pool->n_edge, tail_len = pool->tail_len;
  const int hop = pool->hop, half = pool->half_fft, V = 1 + 2 * n_edge, lag = n_edge - 1;
  KOE_REQUIRE(a->frontend != nullptr && a->weights != nullptr, "koe_stream_pool_push: NULL frontend / weights");
  KOE_REQUIRE(a->weights->k_mel == W + 3, "koe_stream_pool_push: weights for k_mel %d, pool of window_frames %d",
              a->weights->k_mel, W);
  KOE_REQUIRE(a->hop_audio && a->tail && a->tail_compact && a->stage && a->stage_max && a->ring_f && a->fmax_f && a->ring_r &&
                  a->fmax_r && a->row_l && a->fmax_l && a->expr_sigmoid && a->out && a->tables,
              "koe_stream_pool_push: NULL buffer");
  KOE_REQUIRE(n_edge == 1 || (a->ring_r2 && a->fmax_r2 && a->row_l2 && a->fmax_l2),
              "koe_stream_pool_push: hop < n_fft/2 needs the second edge buffers (ring_r2, row_l2)");
  KOE_REQUIRE(a->ema_state == nullptr || (a->alpha >= 0.0f && a->alpha <= 1.0f), "koe_stream_pool_push: alpha must be in [0, 1]");
  if (int rc = check_capture(stream, "koe_stream_pool_push")) return rc;
  int sms = 0;
  KOE_CUDA(sm_count(&sms));
  cudaStream_t st = (cudaStream_t)stream;

  // ---- the per-call tables: [push slot | push ring row | push first hop][emit slot | emit ring base | emit has state]
  TableStaging* b = nullptr;
  if (int rc = acquire_table_staging(stream, 6 * (size_t)n, &b)) return rc;
  int32_t* h = b->host;
  int k = 0;
  for (int i = 0; i < n; ++i) {
    const int s = slots_host[i];
    const int64_t age = pool->hops[s];  // hops before this one
    h[i] = s;
    h[n + i] = pool->row[s];
    h[2 * n + i] = age == 0 ? 1 : 0;
    if (age + 1 >= W) emitted_host[k++] = s;  // this hop completes a window
  }
  // the emit columns are k long, laid out after the push columns; ring base (n + 1 - W) mod W = (row + lag + 1) mod W
  for (int w = 0; w < k; ++w) {
    const int s = emitted_host[w];
    const int base = pool->row[s] + lag + 1;
    h[3 * n + w] = s;
    h[3 * n + k + w] = base >= W ? base - W : base;
    h[3 * n + 2 * k + w] = pool->frames[s] > 0 ? 1 : 0;
  }
  const size_t ints = 3 * (size_t)n + 3 * (size_t)k;
  if (int rc = upload_tables(b, a->tables, ints, st)) return rc;
  const int* push_slot = a->tables;
  const int* push_row = a->tables + n;
  const int* push_first = a->tables + 2 * n;
  const int* emit_slot = a->tables + 3 * n;
  const int* emit_base = emit_slot + k;
  const int* emit_has = emit_slot + 2 * k;

  // ---- 1. tail update + compact copy
  {
    const int grid = std::min(n, sms * 8);
    pool_tail_kernel<<<grid, 256, tail_len * sizeof(float), st>>>(a->tail, a->hop_audio, push_slot, push_first, n, tail_len,
                                                                  hop, a->tail_compact);
    count_launch();
    KOE_CUDA(cudaGetLastError());
  }
  // ---- 2. the frontend launches of koe_stream_push, on the compact tails, into staging rows [n][V][80]
  MelRows stage[1 + 2 * KOE_MAX_EDGE] = {};
  for (int v = 0; v < V; ++v) stage[v] = {a->stage + (size_t)v * KOE_N_MELS, a->stage_max + v, (int64_t)V * KOE_N_MELS, V};
  if (int rc = launch_hop_frontend(a->frontend, a->tail_compact, n, tail_len, half, hop, n_edge, stage, stream)) return rc;
  // ---- 3. staging rows -> each slot's rings and window-end rows
  PoolRings r{};
  float* const power[1 + 2 * KOE_MAX_EDGE] = {a->ring_f, a->ring_r, a->row_l, a->ring_r2, a->row_l2};
  float* const fmax[1 + 2 * KOE_MAX_EDGE] = {a->fmax_f, a->fmax_r, a->fmax_l, a->fmax_r2, a->fmax_l2};
  for (int v = 0; v < V; ++v) r.power[v] = power[v], r.fmax[v] = fmax[v];
  {
    const int total = n * V * (KOE_N_MELS / 4);
    pool_scatter_kernel<<<std::min((total + 255) / 256, sms * 8), 256, 0, st>>>(
        r, a->stage, a->stage_max, push_slot, push_row, n, V, W);
    count_launch();
    KOE_CUDA(cudaGetLastError());
  }
  // ---- 4. the core over the emitting streams, 5. their smoothing
  if (k > 0) {
    const float* cpower[1 + 2 * KOE_MAX_EDGE] = {a->ring_f, a->ring_r, a->row_l, a->ring_r2, a->row_l2};
    const float* cfmax[1 + 2 * KOE_MAX_EDGE] = {a->fmax_f, a->fmax_r, a->fmax_l, a->fmax_r2, a->fmax_l2};
    if (int rc = launch_dual_stream_pool(a->weights, cpower, cfmax, n_edge, k, W, emit_slot, emit_base, a->expr_sigmoid,
                                         a->out, a->precision, stream))
      return rc;
    if (a->ema_state != nullptr) {
      pool_ema_kernel<<<(k * KOE_N_BLENDSHAPES + 255) / 256, 256, 0, st>>>(a->out, k, a->alpha, a->ema_state, emit_slot,
                                                                          emit_has);
      count_launch();
      KOE_CUDA(cudaGetLastError());
    }
  }
  // ---- the clocks advance once everything is queued
  for (int i = 0; i < n; ++i) {
    const int s = slots_host[i];
    if (++pool->hops[s] >= W) ++pool->frames[s];
    if (++pool->row[s] == W) pool->row[s] = 0;
  }
  *n_emitted = k;
  return KOE_OK;
}

extern "C" int koe_stream_pool_push_hops(koe_stream_pool_t* pool, const koe_stream_pool_args* a, const int32_t* slots_host,
                                         const int32_t* counts_host, int n, int32_t* emitted_slot_host,
                                         int64_t* emitted_hop_host, int* n_emitted, void* stream) {
  KOE_REQUIRE(pool != nullptr && a != nullptr && n_emitted != nullptr && emitted_slot_host != nullptr &&
                  emitted_hop_host != nullptr,
              "koe_stream_pool_push_hops: NULL argument");
  *n_emitted = 0;
  if (int rc = check_slots(pool, slots_host, n, "koe_stream_pool_push_hops")) return rc;
  if (n == 0) return KOE_OK;
  KOE_REQUIRE(counts_host != nullptr, "koe_stream_pool_push_hops: NULL counts");
  const int W = pool->window_frames, R = pool->ring_frames, H = pool->max_hops, n_edge = pool->n_edge;
  const int tail_len = pool->tail_len, hop = pool->hop, half = pool->half_fft, V = 1 + 2 * n_edge, lag = n_edge - 1;
  const bool warm = pool->warmup;
  // the windows a stream's c hops complete when it has pushed `age` hops before: at hops W - 1, W, ... -- or, warm-up,
  // at every hop
  auto completing = [&](int64_t age, int c) -> int {
    return warm ? c : (int)std::min<int64_t>(c, std::max<int64_t>(0, age + c - (W - 1)));
  };
  int n_hops = 0, k = 0;  // staged hops, windows that complete (<= capacity * max_hops <= 2^24)
  for (int i = 0; i < n; ++i) {
    const int c = counts_host[i];
    KOE_REQUIRE(c >= 1 && c <= H, "koe_stream_pool_push_hops: count %d for slot %d outside [1, %d]", c, slots_host[i], H);
    n_hops += c;
    k += completing(pool->hops[slots_host[i]], c);
  }
  KOE_REQUIRE(a->frontend != nullptr && a->weights != nullptr, "koe_stream_pool_push_hops: NULL frontend / weights");
  KOE_REQUIRE(a->weights->k_mel == W + 3, "koe_stream_pool_push_hops: weights for k_mel %d, pool of window_frames %d",
              a->weights->k_mel, W);
  KOE_REQUIRE(a->hop_audio && a->tail && a->tail_compact && a->stage && a->stage_max && a->ring_f && a->fmax_f && a->ring_r &&
                  a->fmax_r && a->expr_sigmoid && a->out && a->tables,
              "koe_stream_pool_push_hops: NULL buffer");
  KOE_REQUIRE(n_edge == 1 || (a->ring_r2 && a->fmax_r2), "koe_stream_pool_push_hops: hop < n_fft/2 needs ring_r2");
  KOE_REQUIRE(a->ema_state == nullptr || (a->alpha >= 0.0f && a->alpha <= 1.0f),
              "koe_stream_pool_push_hops: alpha must be in [0, 1]");
  if (int rc = check_capture(stream, "koe_stream_pool_push_hops")) return rc;
  int sms = 0;
  KOE_CUDA(sm_count(&sms));
  cudaStream_t st = (cudaStream_t)stream;

  // ---- the per-call tables: [hop slot | hop ring row] per staged hop, [first staged hop | first hop since open] per
  // pushing stream, [staged hop | has smoothing state] per window -- and on a warm-up pool [frames] per window;
  // 2 n_hops + 2 n + 2 k <= 6 capacity * max_hops, with the frames <= 7 capacity * max_hops
  TableStaging* b = nullptr;
  const size_t ints = 2 * (size_t)n_hops + 2 * (size_t)n + (warm ? 3 : 2) * (size_t)k;
  if (int rc = acquire_table_staging(stream, ints, &b)) return rc;
  int32_t* const h_slot = b->host;
  int32_t* const h_row = h_slot + n_hops;
  int32_t* const h_first = h_row + n_hops;
  int32_t* const h_fresh = h_first + n;
  int32_t* const h_end = h_fresh + n;
  int32_t* const h_has = h_end + k;
  int32_t* const h_frames = h_has + k;  // (warm-up pools only)
  for (int i = 0, e = 0, w = 0; i < n; ++i) {
    const int s = slots_host[i], c = counts_host[i];
    const int64_t age = pool->hops[s];  // hops before this call
    int64_t frames = pool->frames[s];
    int r = pool->row[s];
    h_first[i] = e;
    h_fresh[i] = age == 0 ? 1 : 0;
    for (int j = 0; j < c; ++j, ++e) {
      h_slot[e] = s;
      h_row[e] = r;
      if (++r == R) r = 0;
      if (warm || age + j + 1 >= W) {  // hop age + j completes a window
        if (warm) h_frames[w] = (int32_t)std::min<int64_t>(age + j + 2, W + 1);
        h_end[w] = e;
        h_has[w] = frames++ > 0 ? 1 : 0;
        emitted_slot_host[w] = s;
        emitted_hop_host[w++] = age + j;
      }
    }
  }
  if (int rc = upload_tables(b, a->tables, ints, st)) return rc;
  const int* hop_slot = a->tables;
  const int* hop_row = hop_slot + n_hops;
  const int* first = hop_row + n_hops;
  const int* fresh = first + n;
  const int* hop_end = fresh + n;
  const int* has_state = hop_end + k;
  const int* hop_frames = warm ? has_state + k : nullptr;

  // ---- 1. one compact tail per staged hop, each slot's tail after its last hop
  {
    const int grid = std::min(n, sms * 8);
    pool_hops_tail_kernel<<<grid, 256, (tail_len - hop) * sizeof(float), st>>>(a->tail, a->hop_audio, hop_slot, first, fresh,
                                                                               n, n_hops, tail_len, hop, a->tail_compact);
    count_launch();
    KOE_CUDA(cudaGetLastError());
  }
  // ---- 2. the frontend launches of koe_stream_push on the compact tails, into staging rows [n_hops][V][80]
  MelRows stage[1 + 2 * KOE_MAX_EDGE] = {};
  for (int v = 0; v < V; ++v) stage[v] = {a->stage + (size_t)v * KOE_N_MELS, a->stage_max + v, (int64_t)V * KOE_N_MELS, V};
  if (int rc = launch_hop_frontend(a->frontend, a->tail_compact, n_hops, tail_len, half, hop, n_edge, stage, stream)) return rc;
  // ---- 3. plain and window-start rows -> each slot's rings
  {
    PoolRings r{};
    float* const power[1 + 2 * KOE_MAX_EDGE] = {a->ring_f, a->ring_r, nullptr, a->ring_r2, nullptr};
    float* const fmax[1 + 2 * KOE_MAX_EDGE] = {a->fmax_f, a->fmax_r, nullptr, a->fmax_r2, nullptr};
    for (int v = 0; v < V; ++v) r.power[v] = power[v], r.fmax[v] = fmax[v];
    const int total = n_hops * (1 + n_edge) * (KOE_N_MELS / 4);
    pool_hops_scatter_kernel<<<std::min((total + 255) / 256, sms * 8), 256, 0, st>>>(r, a->stage, a->stage_max, hop_slot,
                                                                                    hop_row, n_hops, n_edge, R);
    count_launch();
    KOE_CUDA(cudaGetLastError());
  }
  // ---- 4. the core over the windows that complete, window-end rows from staging; 5. the smoothing
  if (k > 0) {
    const float* cpower[1 + 2 * KOE_MAX_EDGE] = {a->ring_f, a->ring_r, a->stage + 2 * KOE_N_MELS, a->ring_r2,
                                                 n_edge == 2 ? a->stage + 4 * KOE_N_MELS : nullptr};
    const float* cfmax[1 + 2 * KOE_MAX_EDGE] = {a->fmax_f, a->fmax_r, a->stage_max + 2, a->fmax_r2,
                                                n_edge == 2 ? a->stage_max + 4 : nullptr};
    // the window that completes at hop n starts at frame n + 1 - W = g + lag + 1 - W: ring row (row + lag + H) mod R (a
    // warm-up window at frame 0, which the core derives from its frame count)
    if (int rc = launch_dual_stream_pool_hops(a->weights, cpower, cfmax, n_edge, k, R, hop_end, hop_slot, hop_row, lag + H,
                                              hop_frames, a->expr_sigmoid, a->out, a->precision, stream))
      return rc;
    if (a->ema_state != nullptr) {
      pool_hops_ema_kernel<<<(k * KOE_N_BLENDSHAPES + 255) / 256, 256, 0, st>>>(a->out, k, a->alpha, a->ema_state, hop_end,
                                                                               hop_slot, has_state);
      count_launch();
      KOE_CUDA(cudaGetLastError());
    }
  }
  // ---- the clocks advance once everything is queued
  for (int i = 0; i < n; ++i) {
    const int s = slots_host[i], c = counts_host[i];
    pool->frames[s] += completing(pool->hops[s], c);
    pool->hops[s] += c;
    pool->row[s] += c;
    if (pool->row[s] >= R) pool->row[s] -= R;
  }
  *n_emitted = k;
  return KOE_OK;
}

extern "C" int koe_stream_pool_state_floats(const koe_stream_pool_t* pool) {
  KOE_REQUIRE(pool != nullptr, "koe_stream_pool_state_floats: NULL pool");
  const int64_t f = state_floats(pool);
  KOE_REQUIRE(f <= INT32_MAX, "koe_stream_pool_state_floats: %lld floats per record", (long long)f);
  return (int)f;
}

extern "C" int koe_stream_pool_snapshot(koe_stream_pool_t* pool, const koe_stream_pool_args* a, const int32_t* slots_host,
                                        int n, float* records, int64_t* hops_host, void* stream) {
  KOE_REQUIRE(pool != nullptr && a != nullptr, "koe_stream_pool_snapshot: NULL argument");
  if (int rc = check_slots(pool, slots_host, n, "koe_stream_pool_snapshot")) return rc;
  if (n == 0) return KOE_OK;
  KOE_REQUIRE(records != nullptr && hops_host != nullptr, "koe_stream_pool_snapshot: NULL records / hops");
  KOE_REQUIRE(((uintptr_t)records & 15) == 0, "koe_stream_pool_snapshot: records not 16-byte aligned");
  const int n_edge = pool->n_edge, R = pool->ring_frames, P = pool->window_frames - n_edge;
  KOE_REQUIRE(a->tail && a->ring_f && a->fmax_f && a->ring_r && a->fmax_r && a->expr_sigmoid && a->tables &&
                  (n_edge == 1 || (a->ring_r2 && a->fmax_r2)),
              "koe_stream_pool_snapshot: NULL buffer");
  const int rec = koe_stream_pool_state_floats(pool);
  if (rec < 0) return rec;
  if (int rc = check_capture(stream, "koe_stream_pool_snapshot")) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  // ---- [slot | ring row of the record's row 0 | leading rows of frames < 0] per stream
  TableStaging* b = nullptr;
  if (int rc = acquire_table_staging(stream, 3 * (size_t)n, &b)) return rc;
  for (int i = 0; i < n; ++i) {
    const int s = slots_host[i];
    const int r0 = pool->row[s] - P;  // row[s]: ring row of frame hops - lag = the record's row P
    b->host[i] = s;
    b->host[n + i] = r0 < 0 ? r0 + R : r0;
    b->host[2 * n + i] = (int)std::min<int64_t>(P, std::max<int64_t>(0, pool->window_frames - 1 - pool->hops[s]));
  }
  if (int rc = upload_tables(b, a->tables, 3 * (size_t)n, st)) return rc;
  pool_snapshot_kernel<<<state_grid(pool, n), 256, 0, st>>>(pool_state(a), a->tables, n, 1 + n_edge, P, R, pool->tail_len,
                                                            rec, records);
  count_launch();
  KOE_CUDA(cudaGetLastError());
  for (int i = 0; i < n; ++i) hops_host[i] = pool->hops[slots_host[i]];
  return KOE_OK;
}

extern "C" int koe_stream_pool_restore(koe_stream_pool_t* pool, const koe_stream_pool_args* a, const float* records,
                                       const int64_t* hops_host, int n, int32_t* slots_host, void* stream) {
  KOE_REQUIRE(pool != nullptr && a != nullptr, "koe_stream_pool_restore: NULL argument");
  KOE_REQUIRE(n >= 0, "koe_stream_pool_restore: negative count");
  if (n == 0) return KOE_OK;
  KOE_REQUIRE(records != nullptr && hops_host != nullptr && slots_host != nullptr,
              "koe_stream_pool_restore: NULL records / hops / slots");
  KOE_REQUIRE(((uintptr_t)records & 15) == 0, "koe_stream_pool_restore: records not 16-byte aligned");
  std::vector<int32_t> slots;  // the n lowest free slots, as koe_stream_pool_open takes them
  for (int s = 0; s < pool->capacity && (int)slots.size() < n; ++s)
    if (!pool->open[s]) slots.push_back(s);
  KOE_REQUIRE((int)slots.size() == n, "koe_stream_pool_restore: %d streams, %d of %d slots free", n, (int)slots.size(),
              pool->capacity);
  for (int i = 0; i < n; ++i)
    KOE_REQUIRE(hops_host[i] >= 0, "koe_stream_pool_restore: record %d has %lld hops", i, (long long)hops_host[i]);
  const int W = pool->window_frames, n_edge = pool->n_edge, R = pool->ring_frames, P = W - n_edge, lag = n_edge - 1;
  KOE_REQUIRE(a->tail && a->ring_f && a->fmax_f && a->ring_r && a->fmax_r && a->expr_sigmoid && a->tables &&
                  (n_edge == 1 || (a->ring_r2 && a->fmax_r2)),
              "koe_stream_pool_restore: NULL buffer");
  const int rec = koe_stream_pool_state_floats(pool);
  if (rec < 0) return rec;
  if (int rc = check_capture(stream, "koe_stream_pool_restore")) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  auto mod = [](int64_t x, int m) { return (int32_t)(((x % m) + m) % m); };
  TableStaging* b = nullptr;
  if (int rc = acquire_table_staging(stream, 3 * (size_t)n, &b)) return rc;
  for (int i = 0; i < n; ++i) {
    const int64_t h = hops_host[i];
    b->host[i] = slots[i];
    b->host[n + i] = mod(h + 1 - W, R);  // frame g lives in ring row g mod R in every pool
    b->host[2 * n + i] = (int)std::min<int64_t>(P, std::max<int64_t>(0, W - 1 - h));
  }
  if (int rc = upload_tables(b, a->tables, 3 * (size_t)n, st)) return rc;
  pool_restore_kernel<<<state_grid(pool, n), 256, 0, st>>>(pool_state(a), a->tables, n, 1 + n_edge, P, R, pool->tail_len,
                                                           rec, records);
  count_launch();
  KOE_CUDA(cudaGetLastError());
  // ---- the clocks, once the launch is queued: derived from the hops, as the pushes count them
  for (int i = 0; i < n; ++i) {
    const int s = slots[i];
    const int64_t h = hops_host[i];
    pool->open[s] = 1;
    pool->hops[s] = h;
    pool->frames[s] = pool->warmup ? h : std::max<int64_t>(0, h - W + 1);
    pool->row[s] = mod(h - lag, R);
    slots_host[i] = s;
  }
  return KOE_OK;
}
