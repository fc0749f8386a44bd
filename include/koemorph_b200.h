/*
 * koemorph_b200 -- C ABI of the B200 (sm_100a) audio -> ARKit-blendshape inference path.
 *
 * The reference (atsuki-ichikawa/KoeMorph) has no FFI / plugin / operator API for this path:
 * its boundary is the PyTorch nn.Module surface (SURVEY.md section 8b).  These entry points are
 * therefore what a binding for the path would bind; each one names the reference code it
 * replaces (paths relative to the reference root).  The Python host side in
 * koemorph_b200/ (a mirror of src/model and src/features) calls them through ctypes.
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless the name ends in _host;
 *   - every call is enqueued on `stream` (a cudaStream_t passed as void*) and returns immediately;
 *   - the caller owns every buffer; kernels borrow them for the stream-ordered duration of the call;
 *   - return value: 0 on success, a negative KOE_E_* code on misuse, a positive value is a cudaError_t;
 *     koe_last_error() returns a human-readable message for the calling thread;
 *   - there is no CPU fallback anywhere: without a CUDA device every call fails.
 */
#ifndef KOEMORPH_B200_H_
#define KOEMORPH_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KOE_OK 0
#define KOE_E_INVALID (-1)   /* bad argument (null pointer, size out of range, misaligned) */
#define KOE_E_UNSUPPORTED (-2) /* configuration outside what the kernels implement */
#define KOE_E_NODEVICE (-3)

#define KOE_N_MELS 80
#define KOE_N_FFT 1024
#define KOE_N_BLENDSHAPES 52
#define KOE_N_MOUTH 28
#define KOE_N_EXPR 24
#define KOE_D_MODEL 256
#define KOE_N_HEADS 8
#define KOE_NO_EDGE (-1000000) /* lo_rel_hops / hi_rel_hops: no window edge on that side */
#define KOE_MAX_EDGE 2         /* ceil((n_fft/2) / hop) for hop >= 256 */

const char* koe_last_error(void);
int koe_version(void);
/* sizeof of the public argument structs, for bindings that mirror them (ctypes, cgo, JNI): 0 koe_frontend_config,
 * 1 koe_logmel_args, 2 koe_core_weights, 3 koe_stream_args, 4 koe_forward_args, 5 koe_stream_pool_args,
 * 6 koe_forward_varlen_args; -1 for any other index */
int koe_sizeof_struct(int which);
/* number of kernels launched by this library in this process since load / since the last reset */
int64_t koe_launch_count(void);
void koe_reset_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Log-mel frontend.
 * Replaces: SimplifiedDualStreamModel.extract_mel_features, src/model/simplified_dual_stream_model.py:166-229
 * (librosa.feature.melspectrogram(n_fft=1024, hop, n_mels=80, fmin, fmax) + power_to_db(ref=max) + (x+80)/80)
 * and the librosa calls of MelSlidingWindowExtractor, src/features/mel_sliding_window.py:224-230,280-295.
 * ------------------------------------------------------------------------------------------ */
typedef struct koe_frontend koe_frontend_t; /* opaque: Hann window, FFT twiddles, sparse Slaney filterbank on one device */

int koe_frontend_create(int device, int sample_rate, int n_fft, int n_mels, float fmin, float fmax,
                        koe_frontend_t** out);

/*
 * General form: also the torchaudio flavour of the reference's MelSpectrogramExtractor (src/features/stft.py:23-142:
 * T.MelSpectrogram(n_fft=512, hop=sr/fps, mel_scale "htk", norm None, normalized=True, pad_mode "reflect") followed by
 * log(mel + eps)).  n_fft is 1024 or 512 (a 512-point frame is transformed as the middle of a zero-extended 1024-point
 * one); window_normalized divides the power by sum(window^2); log_mode selects what koe_logmel_power* store.
 */
#define KOE_MEL_SLANEY 0
#define KOE_MEL_HTK 1
#define KOE_MEL_NORM_NONE 0
#define KOE_MEL_NORM_SLANEY 1
#define KOE_LOG_DB 0     /* 10*log10(max(p, 1e-10)) */
#define KOE_LOG_LN_EPS 1 /* ln(p + log_eps) */
typedef struct {
  int32_t device, sample_rate, n_fft, n_mels;
  float fmin, fmax;
  int32_t mel_scale, mel_norm;
  int32_t window_normalized;
  int32_t log_mode;
  float log_eps;
  int32_t win_length; /* 0 = n_fft; else the periodic Hann of win_length <= n_fft points, centred in the n_fft frame
                         (librosa / torch.stft semantics of win_length < n_fft) */
} koe_frontend_config;
int koe_frontend_create_ex(const koe_frontend_config* cfg, koe_frontend_t** out);
int koe_frontend_destroy(koe_frontend_t* fe);
/* 1 when this frontend's filterbank has the structure of the path's default bank (sr 16000, 80 mels, 80..8000 Hz,
 * simplified_dual_stream_model.py:188-199) and runs the unrolled filterbank phase; 0: generic looped kernel */
int koe_frontend_uses_unrolled_bank(const koe_frontend_t* fe);
/* copy the dense (n_mels x (1+n_fft/2)) float32 filterbank to host memory (for parity tests) */
int koe_frontend_filterbank_host(const koe_frontend_t* fe, float* fb_host);

/*
 * Mel power, in dB, of n_frames frames of every clip.  Output row j is frame g = frame_offset + j*frame_step:
 * the 1024-sample periodic-Hann frame centred on sample g*hop (librosa center=True).  Samples outside
 * [0, n_samples) read as zero (librosa pad_mode="constant"); in addition, when lo_rel_hops != KOE_NO_EDGE
 * samples before (g + lo_rel_hops)*hop read as zero, and when hi_rel_hops != KOE_NO_EDGE samples at or
 * after (g + hi_rel_hops)*hop read as zero.  The edge variants are the first / last frames of the sliding
 * windows of SequentialDualStreamModel.forward (src/model/sequential_dual_stream_model.py:101-120):
 * a window starting at frame i sees frame i with lo_rel_hops=0 and frame i+W with hi_rel_hops=0.
 *   audio      [n_clips][audio_stride] float32
 *   power      [n_clips][n_frames][80] float32   10*log10(max(sum_k fb[m][k] * |X_g[k]|^2, 1e-10)): the first term of
 *                                                librosa.power_to_db, so that a consumer only subtracts its reference
 *   frame_max  [n_clips][n_frames]     float32   (max_m power[.,j,m]); may be NULL
 */
int koe_logmel_power(const koe_frontend_t* fe, const float* audio, int64_t audio_stride, int n_clips,
                     int n_samples, int hop, int n_frames, int frame_offset, int frame_step, int lo_rel_hops,
                     int hi_rel_hops, float* power, float* frame_max, void* stream);

/*
 * General form of koe_logmel_power for the streaming paths: frame j is centred on sample
 * sample_offset + (frame_offset + j*frame_step)*hop (the window-edge masks move with it); pad_mode 1 reflects the
 * clip about its first / last sample instead of zero padding (numpy "reflect", the default of
 * MelSlidingWindowExtractor, src/features/mel_sliding_window.py:178,291); the output blocks of consecutive clips are
 * power_clip_stride / frame_max_clip_stride elements apart, so rows can land directly in per-stream ring buffers.
 */
typedef struct {
  const float* audio;
  int64_t audio_stride;
  int32_t n_clips, n_samples, hop, n_frames;
  int32_t frame_offset, frame_step, sample_offset;
  int32_t lo_rel_hops, hi_rel_hops;
  int32_t pad_mode;
  float* power;
  int64_t power_clip_stride;
  float* frame_max;
  int64_t frame_max_clip_stride;
  /* optional second destination: when power_b != NULL the odd frames (2j + 1, the second frame of every pair the kernel
   * transforms together) are written to power_b[clip][j] / frame_max_b[clip][j] instead of row 2j + 1 of `power`.  The
   * streaming step uses it with n_frames = 2: the new plain frame goes into the stream's ring, the next hop's
   * "window ends here" frame (same launch, same transform) into its own row. */
  float* power_b;
  int64_t power_b_clip_stride;
  float* frame_max_b;
  int64_t frame_max_b_clip_stride;
} koe_logmel_args;
int koe_logmel_power_ex(const koe_frontend_t* fe, const koe_logmel_args* args, void* stream);

/*
 * 16-bit PCM -> float32 audio, sample / 32768: the normalisation libsndfile applies when the reference's loaders read a
 * WAV file as float (sf.read(path, dtype="float32"), src/data/io.py:71, src/data/sequential_dataset.py:99).  Lets a host
 * application hand the samples over as stored on disk, halving the PCIe bytes of the host-buffer path; the result is
 * bit-identical to converting on the host.  Both buffers 16-byte aligned, n_samples counts samples over all clips.
 */
int koe_pcm16_to_float(const int16_t* pcm, int64_t n_samples, float* audio, void* stream);

/*
 * Rest of power_to_db on koe_logmel_power's output (ref = max over the clip's n_frames frames, top_db=80), then (x+80)/80.
 * Writes the long-term features [n_clips][n_frames][80] and the short-term detail = last three frames
 * [n_clips][3][80] (zero rows when n_frames < 3: simplified_dual_stream_model.py:206-212).
 * db_only != 0 skips the (x+80)/80 rescale (MelSlidingWindowExtractor semantics, mel_sliding_window.py:295).
 */
int koe_logmel_normalise(const float* power, const float* frame_max, int n_clips, int n_frames, int db_only,
                         float* long_term, float* short_term, void* stream);

/* ------------------------------------------------------------------------------------------
 * Dual-stream attention core.
 * Replaces: DualStreamCrossAttention.forward, src/model/dual_stream_attention.py:162-280, and the
 * 264 -> 256 compression of OpenSMILEeGeMAPSExtractor.get_concatenated_features,
 * src/features/opensmile_extractor.py:583-604.
 * The host folds batch-invariant products once per weight update (koemorph_b200/model/folding.py);
 * all matrices below are row-major float32 and stored TRANSPOSED ([in][out]) for coalesced streaming.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t k_mel;     /* mel_sequence_length + 3: 259 (30 fps) or 515 (60 fps) */
  int32_t k_mel_pad; /* rows allocated in wc_t, multiple of 16, zero filled */
  int32_t emo_in;    /* 264 (compression folded in) or 256 (DualStreamCrossAttention standalone) */
  int32_t emo_in_pad;
  float b2;          /* blendshape_decoder.3.bias */
  float ln_eps;      /* 1e-5 */
  const float* wc_t;   /* [k_mel_pad][256]  mel_channel_encoder.weight^T                         (:211) */
  const float* bc;     /* [256] */
  const float* ln_g;   /* [256] mel_norm.weight                                                  (:212) */
  const float* ln_b;   /* [256] */
  const float* qk_t;   /* [256][256]: column h*28+q = ((Wq q_q + bq)_h / sqrt(32)) Wk_h; cols 224..255 zero (:225-230) */
  const float* wv_t;   /* [256][256] mel_attention.in_proj_weight[512:768]^T */
  const float* bv;     /* [256] */
  const float* wa_t;   /* [256][128] (decoder.0 . mel_output_proj . out_proj)^T                  (:231,248) */
  const float* ba;     /* [128] */
  const float* w2;     /* [128] blendshape_decoder.3.weight */
  const float* coef;   /* [52] 0.5*(softmax(mel_weights/T) + softmax(emotion_weights/T))         (:252-267) */
  const int32_t* mouth_idx; /* [28] */
  const int32_t* expr_idx;  /* [24] */
  const float* we1_t;  /* [emo_in_pad][256] (emotion_encoder . compression)^T                    (:216) */
  const float* be1;    /* [256] */
  const float* eln_g;  /* [256] emotion_norm */
  const float* eln_b;  /* [256] */
  const float* we2_t;  /* [256][128] (decoder.0 . emotion_output_proj . out_proj_e . Wv_e)^T     (:234-240,248) */
  const float* be2;    /* [128] */
  /* tcgen05 path (precision 2): the bf16 weight matrices pre-tiled into the UMMA no-swizzle K-major core-matrix
   * layout, as 16 KiB pipeline-stage images in consumption order (see csrc/dual_stream_tc.cu); NULL if absent */
  const void* tc_bf16;
  int32_t tc_stages;   /* number of 16 KiB stage images behind tc_bf16 */
  int32_t reserved_;
  /* tcgen05 path: the affine parts around the LayerNorm are folded into the pre-tiled weights (bc rides in the first GEMM
   * as weight row k_mel against a constant-one operand column; mel_norm.weight scales the columns of qk / wv; its bias
   * drops out of the scores (softmax-invariant) and moves into this value bias): tc_bv = wv . mel_norm.bias + bv, [256] */
  const float* tc_bv;
} koe_core_weights;

/*
 * Emotion stream: one key per clip, so softmax == 1 and all 24 expression queries give the same value
 * (dual_stream_attention.py:234-240).  emo_in [n_clips][w->emo_in] -> expr_sigmoid [n_clips].
 */
int koe_emotion_stream(const koe_core_weights* w, const float* emo_in, int n_clips, float* expr_sigmoid,
                       void* stream);

/*
 * y[r] = x[r] . w_t + b for n_rows rows: the stand-alone form of the 264 -> 256 eGeMAPS compression
 * (get_concatenated_features, src/features/opensmile_extractor.py:583-604), which SimplifiedDualStreamModel
 * .extract_emotion_features returns.  w_t is [n_in][n_out] (the nn.Linear weight transposed), row-major float32.
 */
int koe_affine_rows(const float* x, int n_rows, int n_in, const float* w_t, const float* b, int n_out, float* y,
                    void* stream);

/*
 * Windows of mel power -> blendshape frames.  Output frame i of clip b uses the window whose first frame
 * is g0 = i*stride_frames and that holds frames_per_window (T) frames; its frame k comes from
 *   power[1 + 2*k]       row (b, i)        lo-edge variant k      if k <  n_edge
 *   power[2 + 2*(T-1-k)] row (b, i)        hi-edge variant T-1-k  if k >= T - n_edge
 *   power[0]             row (b, g0 + k)   plain frames           otherwise.
 * i.e. power[0] is [n_clips][n_frames][80] over the clip's global frames, and every edge buffer is
 * [n_clips][n_out][80], one row per window (koe_logmel_power with frame_offset/frame_step = the window grid).
 * dB reference = max over the window's frames (librosa ref=np.max), -80 dB clamp, (x+80)/80,
 * long-term = first min(T, mel_seq) frames (zero padded to mel_seq), short-term = last 3 frames.
 *   frame_max[j]  same leading shape as power[j] without the 80
 *   expr_sigmoid  [n_clips] from koe_emotion_stream
 *   out           [n_clips][n_out][52]  final blendshapes (before temporal smoothing)
 *   sigmoid_out   [n_clips][n_out][52]  decoder output before the stream-weight fusion, or NULL
 *   attn_out      [n_clips][n_out][28][80] head-averaged mel attention weights, or NULL
 * precision: 0 = fp32 CUDA-core FMA; 2 = bf16 operands on tcgen05 with fp32 accumulation (1 is reserved and rejected).
 */
int koe_dual_stream_windows(const koe_core_weights* w, const float* const* power, const float* const* frame_max,
                            int n_edge, int n_clips, int n_frames, int n_out, int stride_frames,
                            int frames_per_window, const float* expr_sigmoid, float* out, float* sigmoid_out,
                            float* attn_out, int precision, void* stream);

/*
 * Same core on already-normalised features: the DualStreamCrossAttention.forward signature
 * (dual_stream_attention.py:162-168).  mel_long [n_clips][n_long][80] (zero padded / truncated to mel_seq),
 * mel_short [n_clips][3][80]; outputs as above with n_out = 1.
 */
int koe_dual_stream_features(const koe_core_weights* w, const float* mel_long, int n_long, const float* mel_short,
                             int n_clips, const float* expr_sigmoid, float* out, float* sigmoid_out,
                             float* attn_out, int precision, void* stream);

/*
 * Streaming step (rt.py-style sliding window, stride one hop, all streams in lockstep): one window per stream whose
 * frames live in per-stream rings of ring_frames mel rows.  Frame k of the window is
 *   k == 0                      lo-edge row:  power_lo_ring[s][(ring_base) % ring_frames]
 *   0 < k < frames_per_window-1 plain row:    power_ring  [s][(ring_base + k) % ring_frames]
 *   k == frames_per_window-1    hi-edge row:  power_hi    [s]
 * (30 fps geometry: hop >= n_fft/2, one edge frame per side).  Outputs as koe_dual_stream_windows with n_out = 1.
 */
int koe_dual_stream_ring(const koe_core_weights* w, const float* power_ring, const float* fmax_ring,
                         const float* power_lo_ring, const float* fmax_lo_ring, const float* power_hi,
                         const float* fmax_hi, int n_streams, int ring_frames, int ring_base, int frames_per_window,
                         const float* expr_sigmoid, float* out, float* sigmoid_out, float* attn_out, int precision,
                         void* stream);

/*
 * General form for hop < n_fft/2 (60 fps: hop 266, two edge frames per window side): power[0] / frame_max[0] the plain
 * ring, power[1 + 2m] the ring of lo-edge variant m (frame g with everything before (g - m) * hop zeroed, in the slot of
 * global frame g), power[2 + 2m] the per-stream row of hi-edge variant m (frame T-1-m of the window that ends now).
 */
int koe_dual_stream_ring_edges(const koe_core_weights* w, const float* const* power, const float* const* frame_max,
                               int n_edge, int n_streams, int ring_frames, int ring_base, int frames_per_window,
                               const float* expr_sigmoid, float* out, float* sigmoid_out, float* attn_out, int precision,
                               void* stream);

/*
 * One hop of every stream as ONE call (the real-time loop of scripts/rt.py:465-519 over
 * SimplifiedDualStreamModel.process_audio_frame_realtime, src/model/simplified_dual_stream_model.py:452-500, with the
 * sliding window of SequentialDualStreamModel.forward at stride 1): appends hop_audio to each stream's audio tail,
 * computes the new frames of the step (plain, window-start and window-end variants, SURVEY.md section 8 note E: three
 * at 30 fps, five at 60 fps where hop < n_fft/2) into the streams' rings, and -- once window_frames hops have been pushed --
 * runs koe_dual_stream_ring on the window that ends at the newest sample and smooths the result (koe_ema_scan with
 * n_out = 1).  Queues five kernels (seven at 60 fps); replaces the
 * Python driver's six separate calls (about 150 us of host time per hop).  All buffers are caller-owned device memory
 * and persist between calls; `step` counts the hops pushed before this one (0, 1, 2, ...) and selects the ping-pong tail
 * buffer (reads tail[step & 1], writes tail[(step + 1) & 1]) and the ring slot.  *emitted = 1 when `out` holds a frame.
 */
typedef struct {
  const koe_frontend_t* frontend;
  const koe_core_weights* weights;
  int32_t n_streams, hop, window_frames, half_fft; /* half_fft = n_fft / 2 (512) */
  const float* hop_audio;                          /* [n_streams][hop]: the next hop of every stream */
  float* tail[2];                                  /* [n_streams][half_fft + n_edge * hop] each, n_edge = ceil(half_fft / hop);
                                                      zero before the first hop */
  float* ring_f; float* fmax_f;                    /* [n_streams][window_frames][80], [n_streams][window_frames] */
  float* ring_r; float* fmax_r;                    /* same shapes: the window-start variants */
  float* row_l; float* fmax_l;                     /* [n_streams][80], [n_streams]: the window-end variant */
  /* hop < n_fft/2 (60 fps): the second edge frame of either side -- frame g with everything before (g - 1) * hop zeroed
   * (ring) and the last-but-one frame of the window that ends now (row); NULL when hop >= n_fft/2 */
  float* ring_r2; float* fmax_r2;
  float* row_l2; float* fmax_l2;
  const float* expr_sigmoid;                       /* [n_streams], from koe_emotion_stream */
  float* out;                                      /* [n_streams][52] */
  float* ema_state;                                /* [n_streams][52], or NULL: no temporal smoothing */
  float alpha;                                     /* sigmoid(smoothing_alpha) */
  int32_t has_state;                               /* 0 for the first emitted frame of a stream set */
  int32_t precision;
  int64_t step;
} koe_stream_args;
int koe_stream_push(const koe_stream_args* args, int* emitted, void* stream);

/*
 * Stream pool: up to `capacity` streams that open, close and advance on their own clocks (a real-time service whose users
 * connect, leave and send late packets).  Every stream of a pool computes exactly -- bit for bit -- what a one-stream
 * koe_stream_push computes when fed the same hops from the moment the stream was opened, whatever the other streams do
 * and whatever its slot held before: it emits from its own window_frames-th hop on, its first frame passes the
 * smoothing unchanged, and a reused slot carries no audio, mel rows or smoothing state over.
 *
 * The pool object (host memory) owns the clock policy: which slots are open, how many hops each stream has pushed and
 * how many frames it has emitted.  Its entry points return KOE_E_INVALID on misuse (slot out of range or not open, a
 * slot listed twice in one call, more streams than free slots) before anything is queued.  Device buffers are
 * caller-owned (koe_stream_pool_args, shapes below with C = capacity, H = max_hops (1 for koe_stream_pool_create),
 * R = window_frames + H - 1 ring rows, V = 1 + 2 * n_edge buffer variants: plain, window-start 0, window-end 0,
 * window-start 1, window-end 1).  The pushes upload their per-call tables (which stream, ring row and smoothing state
 * each pushed hop and each emitted frame belongs to) with one cudaMemcpyAsync from pinned staging that the library owns
 * per (device, stream); they cannot be captured into a CUDA graph.
 */
typedef struct koe_stream_pool koe_stream_pool_t;
typedef struct {
  const koe_frontend_t* frontend;
  const koe_core_weights* weights;
  const float* hop_audio;        /* [sum of counts][hop]: the pushed hops, stream by stream in call order */
  float* tail;                   /* [C][half_fft + n_edge * hop]: each slot's audio tail (any content when opened) */
  float* tail_compact;           /* [C * H][half_fft + n_edge * hop]: the tail after each pushed hop, in call order */
  float* stage;                  /* [C * H][V][80], */
  float* stage_max;              /* [C * H][V]: the new mel rows of each pushed hop, in call order */
  float* ring_f; float* fmax_f;  /* [C][R][80], [C][R] */
  float* ring_r; float* fmax_r;
  float* row_l; float* fmax_l;   /* [C][80], [C]: koe_stream_pool_push with H = 1 and no KOE_POOL_WARMUP only, else not
                                    read */
  float* ring_r2; float* fmax_r2; /* hop < n_fft/2 only, else NULL */
  float* row_l2; float* fmax_l2;  /* hop < n_fft/2, H = 1 and no KOE_POOL_WARMUP only, else NULL */
  float* expr_sigmoid;           /* [C] */
  float* expr_compact;           /* [C]: scratch of koe_stream_pool_set_egemaps */
  float* out;                    /* [C * H][52]: row r is the r-th frame emitted by the call */
  float* ema_state;              /* [C][52], or NULL: no temporal smoothing */
  int32_t* tables;               /* [6][C * H] int32 ([7][C * H] on a warm-up pool): the per-call tables */
  float alpha;                   /* sigmoid(smoothing_alpha) */
  int32_t precision;
} koe_stream_pool_args;
/* a pool whose streams advance by one hop per push: koe_stream_pool_create_ex with max_hops = 1 */
int koe_stream_pool_create(int capacity, int hop, int window_frames, int half_fft, koe_stream_pool_t** out);
/* a pool whose streams may advance by up to max_hops hops in one koe_stream_pool_push_hops (1 <= max_hops,
 * capacity * max_hops <= 2^24): its rings hold R = window_frames + max_hops - 1 rows, because every row of a burst is
 * written before the core reads the burst's first window */
int koe_stream_pool_create_ex(int capacity, int hop, int window_frames, int half_fft, int max_hops, koe_stream_pool_t** out);
/* koe_stream_pool_create_ex with a flags word (any other bit set: KOE_E_INVALID).  flags = 0 is koe_stream_pool_create_ex.
 *
 * KOE_POOL_WARMUP: a warm-up pool.  Every pushed hop of every open stream emits a frame, from the stream's hop 0 on,
 * instead of from its hop window_frames - 1 (W - 1): a new stream is animated after one hop instead of 8.5 s.
 *   - hops h >= W - 1: the unsmoothed frame is bit for bit the one a pool without the flag gives (the same rows,
 *     window-start variants included);
 *   - hops h < W - 1: the unsmoothed frame is SimplifiedDualStreamModel.forward on the stream's first (h + 1) * hop
 *     samples (up to the rounding of the frontend): T = h + 2 frames, frames 0 .. T - 1 - n_edge from the plain ring
 *     rows, the last n_edge from that hop's window-end rows, no window-start variants -- the long-term part is those
 *     frames zero-padded, the short-term detail their last three, the dB reference their maximum;
 *   - smoothing (ema_state != NULL) runs over every frame since the stream was opened: the hop-0 frame passes
 *     unchanged and every later one is smoothed onto the one before, so from hop W - 1 on the smoothed frames are the
 *     smoothing of this pool's own frames, not those of a pool without the flag.
 * koe_stream_pool_push on a warm-up pool is koe_stream_pool_push_hops with every count 1, whatever max_hops is; rings
 * keep R = W + max_hops - 1 rows, and the tables take [7][C * H] int32. */
#define KOE_POOL_WARMUP 1
int koe_stream_pool_create_ex2(int capacity, int hop, int window_frames, int half_fft, int max_hops, int flags,
                               koe_stream_pool_t** out);
int koe_stream_pool_destroy(koe_stream_pool_t* pool);
/* takes the n lowest free slots into slots_host[n]; their clocks start at zero (their expression input is unset until
 * koe_stream_pool_set_egemaps) */
int koe_stream_pool_open(koe_stream_pool_t* pool, int n, int32_t* slots_host);
int koe_stream_pool_close(koe_stream_pool_t* pool, int slot);
/* the emotion stream for n open streams: egemaps [n][weights->emo_in] -> expr_sigmoid[slots_host[i]] */
int koe_stream_pool_set_egemaps(koe_stream_pool_t* pool, const koe_stream_pool_args* args, const int32_t* slots_host, int n,
                                const float* egemaps, void* stream);
/* advances the n open streams slots_host[0..n) by one hop each.  *n_emitted streams emit a frame: their slots go to
 * emitted_host[0..*n_emitted) (capacity entries), in call order, and their frames to out rows 0..*n_emitted.  Queues the
 * tail update, the frontend launches of koe_stream_push on the pushing streams (2 at 30 fps, 4 at 60 fps), the scatter
 * into their rings and, when a stream emits, the core over the emitting streams and the smoothing: 6 kernels (8 at
 * 60 fps), 4 (6) when no stream emits, none for n = 0.  On a pool with max_hops > 1 or KOE_POOL_WARMUP this is
 * koe_stream_pool_push_hops with every count 1 (the same frames, the same number of kernels). */
int koe_stream_pool_push(koe_stream_pool_t* pool, const koe_stream_pool_args* args, const int32_t* slots_host, int n,
                         int32_t* emitted_host, int* n_emitted, void* stream);
/* advances the n open streams slots_host[0..n) by counts_host[i] hops each, 1 <= counts_host[i] <= max_hops (host
 * memory): hop_audio holds sum(counts) hops, stream 0's in order, then stream 1's, ...  Every frame is bit for bit the
 * frame that one koe_stream_pool_push per hop would give.  *n_emitted frames come out: row r of out is a frame of stream
 * emitted_slot_host[r], the one that completes at its hop emitted_hop_host[r] (counted from 0 since the stream was opened:
 * the first frame comes at hop window_frames - 1, or at hop 0 on a KOE_POOL_WARMUP pool); rows are grouped by stream in call order, hops ascending within a
 * stream (both host arrays take C * H entries).  All windows of a burst use the stream's expression value at the time of
 * the call: a koe_stream_pool_set_egemaps meant to take effect between two hops of a stream needs two calls.  Queues
 * the same kernels as koe_stream_pool_push, whatever the counts: a tail kernel that writes the tail after every pushed
 * hop, the frontend launches over all pushed hops, the scatter into the rings and, when a frame completes, the core over
 * all completing windows and the smoothing, which runs each stream's frames in order.  Misuse (a count outside
 * [1, max_hops], a slot out of range, not open or listed twice) returns KOE_E_INVALID before anything is queued. */
int koe_stream_pool_push_hops(koe_stream_pool_t* pool, const koe_stream_pool_args* args, const int32_t* slots_host,
                              const int32_t* counts_host, int n, int32_t* emitted_slot_host, int64_t* emitted_hop_host,
                              int* n_emitted, void* stream);

/*
 * Snapshots: a stream's whole state as one fixed-size float32 record, so that it can leave its slot -- into a pool of
 * another capacity or max_hops (a pool that grows), onto another GPU (load balancing, draining a GPU), or through host
 * memory (a restart of the serving process) -- and continue there bit for bit.
 *
 * koe_stream_pool_snapshot writes the records of the n open streams slots_host[0..n) to records[n][state_floats]
 * (caller-owned device memory, 16-byte aligned) and each stream's clock -- the hops pushed since it was opened -- to
 * hops_host[n].  The streams stay open and are not changed: their later frames are those they would have given without
 * the snapshot.  The record holds the state after every call queued before it on `stream`.
 * koe_stream_pool_restore takes the n lowest free slots (as koe_stream_pool_open) into slots_host[n], writes record i into
 * slot i and sets its clock to hops_host[i]; with hops_host[i] == 0 that is exactly an open.
 *
 * Equality: a stream snapshotted after a hops in pool A and restored into pool B, then pushed the same hops a, a + 1, ...
 * in B as in A -- any mix of koe_stream_pool_push and koe_stream_pool_push_hops -- gives bit for bit the frames (the
 * unsmoothed and the smoothed ones) and the hops the stream gives in A, when both pools run the same weights at the same
 * precision.  This holds whatever B's capacity and max_hops are and whatever B's slots held before.  A and B must have
 * the same hop, window_frames, half_fft and KOE_POOL_WARMUP flag: the record does not carry them, and a record of another
 * geometry is the caller's error (the Python layer, StreamSnapshot, refuses it).
 *
 * Only the hops travel; restore derives the rest as the pushes count them: frames = max(0, hops - W + 1) (hops on a
 * warm-up pool) and the ring row of frame g = g mod R_B.  The expression value and the smoothing row travel in the
 * record: no koe_stream_pool_set_egemaps is needed after a restore.  A snapshot with args->ema_state == NULL stores a
 * zero smoothing row; a restore with args->ema_state == NULL does not write one.
 *
 * Record layout, with W = window_frames, lag = n_edge - 1, a = the stream's hops, P = W - 1 - lag (the frames a later
 * window can still read: the window that completes at hop a starts at frame a + 1 - W, the newest complete frame is
 * a - 1 - lag) and V_r = 1 + n_edge ring variants (plain, window-start 0, at hop < n_fft/2 window-start 1):
 *   rows          [V_r][P][80]   variant v's row of frame a + 1 - W + i at row i (ring row (a + 1 - W + i) mod R)
 *   row maxima    [V_r][P]
 *   tail          [half_fft + n_edge * hop]
 *   expr_sigmoid  [1]
 *   ema_state     [52]
 *   zero padding  to a multiple of 4 floats (state_floats in all)
 * Rows of frames < 0 (a stream younger than W - 1 hops) are zeros and are not written back: no window reads them.
 * Window-end rows are not state (the pushes write and read them in one call).  30 fps: 42,408 floats (170 KB); 60 fps:
 * 125,028 floats (500 KB).
 *
 * Each call uploads a table of 3 n int32 through the pool's tables and queues one kernel; neither can be captured into a
 * CUDA graph.  Misuse returns KOE_E_INVALID before anything is queued and leaves every clock as it was: snapshot -- a slot
 * out of range, not open or listed twice, NULL records / hops; restore -- more records than free slots, a negative hops,
 * NULL records / hops / slots.  Of args only the rings (ring_f, ring_r, ring_r2 and their maxima), tail, expr_sigmoid,
 * ema_state and tables are used.  n = 0 is a no-op.
 */
/* floats per record for this pool's geometry (host only) */
int koe_stream_pool_state_floats(const koe_stream_pool_t* pool);
int koe_stream_pool_snapshot(koe_stream_pool_t* pool, const koe_stream_pool_args* args, const int32_t* slots_host, int n,
                             float* records, int64_t* hops_host, void* stream);
int koe_stream_pool_restore(koe_stream_pool_t* pool, const koe_stream_pool_args* args, const float* records,
                            const int64_t* hops_host, int n, int32_t* slots_host, void* stream);

/*
 * The whole forward of SequentialDualStreamModel.forward (src/model/sequential_dual_stream_model.py:63-167) -- or, with
 * n_out = 1 and n_edge = 0, of SimplifiedDualStreamModel.forward (src/model/simplified_dual_stream_model.py:370-415) --
 * as ONE call: koe_logmel_power on the clip's global frames, the 2 * n_edge edge-variant launches on the window grid,
 * the emotion stream, koe_dual_stream_windows and (smooth != 0, n_out > 1) koe_ema_scan, queued back to back on `stream`.
 * Because the call knows which kernel precedes which, every kernel is chained to the one before it with programmatic
 * dependent launch (it takes SMs as that kernel's CTAs leave them and orders itself with griddepcontrol.wait); the public
 * single-kernel entries above keep plain stream order.  The expression entries of `out` depend on the emotion stream only
 * and the mouth entries on the mel stream only, so here the emotion kernel writes its 24 entries of every output row
 * itself (and expr_sigmoid, as koe_emotion_stream would) and the core leaves them alone: neither waits for the other's
 * results.  With one window per clip (n_out = 1, n_edge = 0, precision 2, no attention output) and more clips than SMs,
 * the core does not wait for the whole frontend either: it starts every round of windows but its last on a release /
 * acquire flag that the frontend counts up once those clips are stored (two words per device and stream, owned by the
 * library, zero between calls).  Results are identical to the kernels run one after the other.
 * Window i of a clip starts at global frame i * stride_frames and holds
 * frames_per_window frames; n_frames >= (n_out - 1) * stride_frames + frames_per_window global frames are computed.
 * Workspace (caller-owned): power[0] / frame_max[0] [n_clips][n_frames][80] / [n_clips][n_frames]; for m < n_edge
 * power[1 + 2m], power[2 + 2m] [n_clips][n_out][80] (+ frame_max); expr_sigmoid [n_clips].
 */
typedef struct {
  const koe_frontend_t* frontend;
  const koe_core_weights* weights;
  const float* audio;      /* [n_clips][audio_stride] */
  int64_t audio_stride;
  int32_t n_clips, n_samples, hop;
  int32_t n_frames, frames_per_window, stride_frames, n_out, n_edge;
  const float* egemaps;    /* [n_clips][weights->emo_in] */
  float* power[1 + 2 * KOE_MAX_EDGE];
  float* frame_max[1 + 2 * KOE_MAX_EDGE];
  float* expr_sigmoid;
  float* out;              /* [n_clips][n_out][52] */
  float* sigmoid_out;      /* or NULL */
  float* attn_out;         /* or NULL */
  float alpha;             /* sigmoid(smoothing_alpha) */
  int32_t smooth;          /* != 0: EMA over the n_out frames of every clip (first frame passes through) */
  int32_t precision;
} koe_forward_args;
int koe_forward_windows(const koe_forward_args* args, void* stream);

/*
 * Packed variable-length batch: SequentialDualStreamModel.forward for clips of different lengths as ONE call.  The clips
 * lie back to back in `audio` (clip c = samples [sum of lengths_host[0..c), + lengths_host[c])); clip c gets
 *   n_out_c    = max(1, (L_c / hop - window_frames) / stride_frames + 1)   (floor division, as the model's num_output_frames)
 *   n_frames_c = (n_out_c - 1) * stride_frames + window_frames + 1 global frames,
 * and uses the window-edge variants (n_edge = ceil(half_fft / hop) per side) unless it is a single window that spans the
 * whole clip (n_out_c == 1 and L_c <= window_frames * hop): such a clip reads every frame of its window from the plain
 * rows, as koe_forward_windows does with n_edge = 0.  Output rows: clip c's frames are rows
 * [sum of n_out over clips < c, + n_out_c) of out / sigmoid_out / attn_out, each bit for bit what koe_forward_windows
 * computes for that clip alone (frame pairs of the frontend's complex FFT are formed within each clip, the smoothing
 * restarts at each clip's first frame).  The call derives the per-clip geometry from lengths_host, validates everything
 * (lengths in [0, 2^30), fewer than 2^31 frame pairs and windows, workspace large enough) and returns KOE_E_INVALID
 * before anything is queued.  It uploads its per-clip tables (sample offset, length, first frame, first window, first
 * frame pair, edge rule) with one cudaMemcpyAsync from pinned staging that the library owns per (device, stream), so it
 * cannot be captured into a CUDA graph.  Queues the kernels of koe_forward_windows, chained the same way (no early
 * release): frontend, 2 * n_edge edge-variant launches (none when no clip uses them), emotion stream, core and, when
 * smooth != 0 and some clip has more than one frame, the smoothing.  Only the default filterbank (sr 16000, 80 mels,
 * 80..8000 Hz) is implemented; other banks return KOE_E_UNSUPPORTED.  koe_forward_varlen_ex below adds the warm-up
 * frames: a frame at every hop of the output grid from the clip's first hop on.
 */
typedef struct {
  const koe_frontend_t* frontend;
  const koe_core_weights* weights;   /* k_mel == window_frames + 3 */
  const float* audio;                /* [sum of lengths] */
  const int64_t* lengths_host;       /* [n_clips] samples per clip, HOST memory */
  int32_t n_clips, hop, window_frames, stride_frames, half_fft; /* window_frames = mel_sequence_length; half_fft = 512 */
  int32_t smooth;                    /* != 0: EMA over each clip's frames (first frame passes through) */
  int32_t precision;
  float alpha;                       /* sigmoid(smoothing_alpha) */
  const float* egemaps;              /* [n_clips][weights->emo_in] */
  void* workspace;                   /* caller-owned device memory of koe_forward_varlen_size's workspace_bytes, 16-byte aligned */
  int64_t workspace_bytes;
  float* out;                        /* [n_windows][52] */
  float* sigmoid_out;                /* [n_windows][52], or NULL */
  float* attn_out;                   /* [n_windows][28][80], or NULL */
} koe_forward_varlen_args;
/* host only (no device work): total output rows, total global frames and the workspace koe_forward_varlen needs for
 * the lengths and geometry in args (the buffer and output fields are not read); KOE_E_INVALID on the same misuse.
 *
 * Workspace layout (what a caller may read back after the call; koe_forward_varlen_ex with the same flags).  With
 * n_edge = ceil(half_fft / hop), W = window_frames, s = stride_frames, n_out_c and n_frames_c as above, and prefix sums
 * over the clips before c: frame_base_c = sum n_frames, window_base_c = sum n_out, lead_base_c = sum K (K_c: the lead
 * windows of KOE_VARLEN_WARMUP below, 0 without the flag).  E = n_edge when some clip is not a plain single window or
 * (warm-up) some clip has a lead window, else 0; N = sum n_out over all clips when some clip is not a plain single
 * window, else 0.  Regions follow each other, each rounded up to a multiple of 16 bytes, in this order:
 *   power[0]           [sum n_frames][80]  clip c's global frame g at row frame_base_c + g (pad: frames past the clip
 *                                          read zeros)
 *   power[1 + 2m]      [N][80]             m < E: window-start variant m of window i of clip c at row window_base_c + i:
 *                                          frame i * s + m with everything before (i * s) * hop zeroed
 *   power[2 + 2m]      [N + sum K][80]     window-end variant m of window i at row window_base_c + i: frame
 *                                          i * s + W - m with everything from (i * s + W) * hop on zeroed; then the lead
 *                                          window at grid hop h = r + k * s (k < K_c) at row N + lead_base_c + k: frame
 *                                          h + 1 - m with everything from (h + 1) * hop on zeroed
 *   frame_max[0], frame_max[1 .. 2E]       the same rows without the 80: each row's largest band
 *   the per-clip tables the call uploads (not part of the interface)
 * Rows of a clip that reads its window from the plain rows are not written in power[1 .. 2E].  Within each launch the
 * frontend transforms a clip's rows 2j and 2j + 1 (of that buffer, counted from the clip's first row) as one pair. */
int koe_forward_varlen_size(const koe_forward_varlen_args* args, int64_t* n_windows, int64_t* n_frames,
                            int64_t* workspace_bytes);
int koe_forward_varlen(const koe_forward_varlen_args* args, void* stream);

/*
 * The same with a flags word; flags = 0 is koe_forward_varlen / koe_forward_varlen_size, any bit but KOE_VARLEN_WARMUP
 * returns KOE_E_INVALID.
 *
 * KOE_VARLEN_WARMUP: the frames a KOE_POOL_WARMUP stream pool would emit for each clip, in one call.  With W =
 * window_frames, s = stride_frames and n_c = L_c / hop complete hops, the output grid is the hops h = W - 1 (mod s) from
 * r = (W - 1) mod s on, and clip c gets one row per grid hop it completes: h = r, r + s, .. <= n_c - 1, ascending (rows
 * [sum of the rows of the clips < c, + those of clip c); n_windows of koe_forward_varlen_size_ex counts them).
 *   - Rows at h >= W - 1 are the windows of koe_forward_varlen (n_out_c of them when n_c >= W, else none), from the same
 *     frontend rows: bit for bit its rows when smooth = 0.  The padded single window of a clip with n_c < W is not a row.
 *   - Rows at h < W - 1 (lead windows) are SimplifiedDualStreamModel.forward on the clip's first (h + 1) * hop samples:
 *     T = h + 2 frames, the last n_edge of them window-end variants that see zeros from sample (h + 1) * hop on, no
 *     window-start variants; long-term part zero padded to mel_seq, short-term detail the last three frames, dB
 *     reference their maximum -- the frames of a warm-up pool at those hops.
 *   - smooth != 0: the EMA restarts at each clip's first row and runs over all of its rows, so rows from W - 1 on are
 *     the smoothing of this call's own rows (as a warm-up pool's frames differ from a plain pool's).
 *   - A clip that completes no grid hop (L_c < (r + 1) * hop) returns KOE_E_INVALID before anything is queued.
 * Launches: those of koe_forward_varlen (the plain and the 2 * n_edge steady edge-variant launches unchanged: the same
 * frames per clip, the same frame pairs), plus n_edge lead-variant frontend launches when some clip has a lead window
 * (any clip, when s < W), before the emotion stream; the core and the smoothing run over the rows above.  The workspace
 * grows by n_edge window-end buffers of one row per lead window.
 */
#define KOE_VARLEN_WARMUP 1
int koe_forward_varlen_size_ex(const koe_forward_varlen_args* args, int flags, int64_t* n_windows, int64_t* n_frames,
                               int64_t* workspace_bytes);
int koe_forward_varlen_ex(const koe_forward_varlen_args* args, int flags, void* stream);

/*
 * Learnable-alpha exponential smoothing along the frame axis, in place
 * (apply_temporal_smoothing, src/model/simplified_dual_stream_model.py:341-368):
 *   y_0 = x_0 (or alpha*x_0 + (1-alpha)*state when state != NULL and has_state != 0); y_t = alpha*x_t + (1-alpha)*y_{t-1}.
 * frames [n_clips][n_out][52]; state [n_clips][52] receives y_{n_out-1} when non-NULL.
 */
int koe_ema_scan(float* frames, int n_clips, int n_out, float alpha, float* state, int has_state, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KOEMORPH_B200_H_ */
