// tcgen05 / TMEM implementation of the dual-stream core (precision 2: bf16 operands, fp32 accumulation).
//
// Same arithmetic as dual_stream_fp32_kernel (reference src/model/dual_stream_attention.py:162-280) with
// every GEMM on the 5th-generation tensor cores:
//
//   phase  MMA (M=128, cta_group::1, kind::f16)                         accumulator (TMEM columns)
//   G1     z[tok 128(80) x 256]   = Xn[tok x 272] . Wc[256 x 272]^T      [0,256)
//   VT     vT[d 128 x tok 80]     = Wv_t[128 x 256] . enc[80 x 256]^T    [0,80) [80,160)       2 tiles
//   S      s[hq 128 x tok 80]     = Qk_t[128 x 256] . enc[80 x 256]^T    [256,336) [336,416)   2 tiles of 4 heads
//   PV     o[hq 128 x d 128]      = P_t[128 x 80] . vT_t[128 x 80]^T     [160,288) [288,416)   (diagonal 32x32 blocks used)
//   H1     h[q 128(28) x 128]     = O[q x 256] . Wa[128 x 256]^T         [288,416)
//
// Operands live in shared memory in the canonical UMMA *no-swizzle K-major* layout: 8-row x 16-byte core
// matrices, element (r, k) at (r/8)*SBO + (k/8)*128 + (r%8)*16 + (k%8)*2 bytes (measured at the M=128 floor of
// tcgen05.mma, scripts/microbench/umma_operand_layout_rate.cu).  Activations are written in that layout by the
// epilogue threads; weights are pre-tiled on the host into the same layout, 16 KiB per pipeline stage, so a producer
// moves one stage with a single cp.async.bulk (TMA bulk copy) that completes on an mbarrier.
//
// Roles (352 threads): warps 0-7 = SIMT (operand staging, TMEM epilogues; warps w and w + 4 own TMEM lanes
// 32 (w % 4) .. +31 and split every epilogue), warp 8 = weight producer (ring slots 0-3), warp 9 = TMEM allocator +
// MMA issuer (the whole warp runs the loop, one elected lane issues), warp 10 = mel-row producer (ring slots 4-5).
// Phases are serialised by mbarriers (mma_go: 256 SIMT arrivals; mma_done / vt_done: tcgen05.commit); both rings
// run ahead across phases and windows.  At 30 fps a window's timeline is
//   G1(i) [under the decoder tail of i-1] -> LayerNorm -> VT, S GEMMs [SIMT: stage window i+1, then the vT epilogue]
//   -> softmax -> PV -> O -> H1 -> decoder tail [G1(i+1) already running]
// (DESIGN.md section 4 has the measured cycle counts); at 60 fps the first GEMM's operand spans the region the S/VT
// GEMMs read, so the next window is staged after the decoder tail instead.
#include <cuda_bf16.h>

#include "common.cuh"
#include "core_params.cuh"

namespace koe {

namespace tc {

constexpr int kThreads = 352;   // warps 0-7 SIMT (two warpgroups), warp 8 weight producer, warp 9 MMA issuer, warp 10 mel-row producer
constexpr int kSimt = 256;
constexpr int kStageBytes = 16384;
constexpr int kRing = 6;             // 16 KiB stages: slots [0, kWRing) carry weights (consumer: the MMA warp), slots [kWRing, kRing)
constexpr int kWRing = 4;            // the windows' mel rows (consumer: the SIMT warps).  Two rings, two producers: a slow consumer of
                                     // one kind never holds up the other kind's stages, as it did when both shared one FIFO
constexpr int kTok = 80;
// Window geometry: K of the first GEMM = mel_sequence_length + 3 = 259 (30 fps) or 515 (60 fps)
template <int KMEL>
struct Geo {
  static constexpr int kKMel = KMEL;
  static constexpr int kKMelPad = (KMEL + 15) / 16 * 16;        // 272 / 528
  static constexpr int kA1Chunks = kKMelPad / 8;                // 34 / 66 16-byte K chunks per row
  static constexpr int kA1Sbo = kA1Chunks * 128 + 16;           // 4368 / 8464: row groups skewed by 16 B (shared-memory banks)
  static constexpr int kLongChunks = (KMEL - 3) / 8;            // 32 / 64 chunks of long-term frames, then the short-term chunk
  static constexpr int kStagesG1 = (kKMelPad + 31) / 32;        // 9 / 17 weight stages of [256 x 32]; the last is half full
  static constexpr int kStagesPerWindow = kStagesG1 + 20;       // + 5 x 4 stages of [128 x 64]
  // the first-GEMM operand of window i+1 is staged while the S/VT GEMMs of window i run; needs the operand to fit the X region
  static constexpr bool kStageAhead = KMEL == 259;
};
constexpr int kA1Sbo30 = Geo<259>::kA1Sbo;
constexpr int kESbo = 32 * 128;                   // enc / Oflat: K = 256 -> 32 chunks
constexpr int kPSbo = 10 * 128;                   // P / vT tiles: K = 80 -> 10 chunks
constexpr int kPTile = 16 * kPSbo;                // 20480
constexpr int kStagesTile = 4;
constexpr int kMelRows = 48;                      // mel rows (frames) per ring stage: 48 * 320 B = 15360 B, 6 K-chunks

// shared memory map (bytes)
constexpr int kOffBar = 0;                        // mbarriers + tmem base
constexpr int kOffConst = 256;                    // bc, ln_g, ln_b, bv (256 each), ba, w2 (128 each), LN partials (512)
constexpr int kOffX = kOffConst + 1792 * 4;       // A1 (43520): free from the end of the first GEMM, so at 30 fps the NEXT
                                                  // window's operand is staged here while the S/VT GEMMs of this one run
constexpr int kOffE = kOffX + (10 * kA1Sbo30 + 127) / 128 * 128;      // enc (40960) -> P tiles (40960) -> Oflat; at 60 fps the A1 operand (84480 B) spans X and E, which is
                                                  // free until the LayerNorm epilogue writes enc after the first GEMM
constexpr int kOffVT = kOffE + 10 * kESbo;        // vT tiles (40960)
constexpr int kOffRing = kOffVT + 2 * kPTile;
constexpr int kSmemBytes = kOffRing + kRing * kStageBytes;   // 229120
static_assert(kOffX % 128 == 0 && kOffE % 128 == 0 && kOffVT % 128 == 0 && kOffRing % 128 == 0, "alignment");
static_assert(kOffX + 16 * Geo<515>::kA1Sbo <= kSmemBytes && kOffE + 16 * kESbo <= kSmemBytes, "operand over-read stays inside");
static_assert(kOffX + 10 * Geo<515>::kA1Sbo <= kOffVT, "the 60 fps A1 operand ends where the vT tiles begin");

// TMEM column map
constexpr uint32_t kColD1 = 0, kColS = 256, kColVT = 0, kColO = 160;
// H sits clear of [0, 256): the next window's first GEMM runs while the decoder tail still reads it (O is consumed by then)
constexpr uint32_t kColH = 288;

// (dB - ref) clamped at -80 dB and rescaled to [0, 1], as normalise_db(., ., true) -- but the operand is rounded to bf16
// next (2^-9 relative), so the exact fp32 division of the reference is replaced by one FFMA (<= 1 ulp of fp32 away)
__device__ __forceinline__ float normalise_bf16(float db, float ref_db, bool) {
  return fmaf(fmaxf(db - ref_db, -kTopDb), 1.0f / 80.0f, 1.0f);
}

// ---- PTX wrappers ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// bounded spin: a protocol bug traps (error to the host) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  for (uint32_t spin = 0; !ok; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (!ok && spin > (1u << 22)) __trap();
  }
}
// L2 cache policies for the bulk copies: the weights are re-read by every window of every step (keep), a window's mel
// rows are read once (let them go first)
__device__ __forceinline__ uint64_t l2_policy_keep() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_stream() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void bulk_g2s_hint(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
// pull a 16-byte-aligned run of global memory into L2 (no destination in the SM, nothing to wait for)
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
// one lane of a converged warp
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets row (lane base + t)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// UMMA shared-memory descriptor, no swizzle, K-major: start>>4 | LBO>>4 << 16 | SBO>>4 << 32 | version 1 << 46
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((addr & 0x3FFFF) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         (1ull << 46);
}
// instruction descriptor: D=f32 (bit 4), A=B=bf16 (bits 7, 10), K-major both, N>>3 at 17, M>>4 at 24
__host__ __device__ constexpr uint32_t idesc_bf16(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ uint4 pack8_bf16(const float* v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
  __nv_bfloat162 c = __floats2bfloat162_rn(v[4], v[5]), d = __floats2bfloat162_rn(v[6], v[7]);
  uint4 o;
  o.x = *reinterpret_cast<uint32_t*>(&a);
  o.y = *reinterpret_cast<uint32_t*>(&b);
  o.z = *reinterpret_cast<uint32_t*>(&c);
  o.w = *reinterpret_cast<uint32_t*>(&d);
  return o;
}

__device__ __forceinline__ void stamp(long long* dbg, int slot) {
  if (dbg != nullptr) dbg[slot] = clock64();
}

__device__ __forceinline__ void simt_barrier() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// One instantiation per CoreMode; the window of a work item and the rows of its frames come from CoreRows<M>.  Early is
// the early-release flavour of the fused forward (see the wait below): as run-time branches its extra checks cost the
// kernel every other caller runs 4 % through register spills.
template <int KMEL, CoreMode M>
__global__ void __launch_bounds__(kThreads, 1) dual_stream_tc_kernel(CoreParams p) {
  using G = Geo<KMEL>;
  using Rows = CoreRows<M>;
  constexpr int kKMel = G::kKMel, kA1Chunks = G::kA1Chunks, kA1Sbo = G::kA1Sbo, kLongChunks = G::kLongChunks;
  constexpr int kStagesG1 = G::kStagesG1, kStagesPerWindow = G::kStagesPerWindow;
  constexpr bool kStageAhead = G::kStageAhead;
  extern __shared__ __align__(1024) unsigned char smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const koe_core_weights& W = p.w;
  // early release: a first look at the flag now, so that its L2 round trip runs beside the prologue (used below)
  unsigned early_seen = 0;
  if (M == CoreMode::Early && lane == 0) asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(early_seen) : "l"(p.early_flag) : "memory");
  long long* dk = (p.dbg != nullptr && blockIdx.x == 0 && tid == 0) ? p.dbg + 120 : nullptr;
  stamp(dk, 0);
  if (p.dbg != nullptr && tid == 0) {  // per-CTA wall-clock span (ns) for the launch-level picture
    unsigned long long g;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
    p.dbg[128 + 2 * blockIdx.x] = (long long)g;
  }

  // barriers: full[kRing], empty[kRing], mma_go, mma_done
  const uint32_t bar_full = sbase + kOffBar, bar_empty = bar_full + 8 * kRing;
  const uint32_t bar_go = bar_empty + 8 * kRing, bar_done = bar_go + 8;
  // the VT tiles' completion has its own barrier: the SIMT warps may still be staging the next window when both the VT
  // and the S tiles complete, and a waiter two phases behind on one barrier would never see its parity
  const uint32_t bar_vt = bar_done + 8;
  volatile uint32_t* s_tmem = reinterpret_cast<volatile uint32_t*>(smem + kOffBar + 8 * (2 * kRing + 3));
  float* s_red = reinterpret_cast<float*>(smem + kOffBar + 8 * (2 * kRing + 3) + 16);  // [8]
  float* s_const = reinterpret_cast<float*>(smem + kOffConst);
  const float* s_bv = s_const + 768;
  const float *s_ba = s_const + 1024, *s_w2 = s_const + 1152;
  float* s_ln = s_const + 1280;  // [stat 2][warpgroup 2][row 128]

  if (tid == 0) {
    for (int i = 0; i < kRing; ++i) {
      mbar_init(bar_full + 8 * i, 1);
      mbar_init(bar_empty + 8 * i, 1);
    }
    mbar_init(bar_go, kSimt);
    mbar_init(bar_done, 1);
    mbar_init(bar_vt, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < kSimt) {
    for (int i = tid; i < 256; i += kSimt) {
      s_const[768 + i] = W.tc_bv[i];  // (bc, mel_norm.weight / bias are folded into the pre-tiled weights)
    }
    if (tid < 128) {
      s_const[1024 + tid] = W.ba[tid];
      s_const[1152 + tid] = W.w2[tid];
    }
    // operand regions start as zeros so that never-written rows / K tails are finite
    uint4* z = reinterpret_cast<uint4*>(smem + kOffX);
    for (int i = tid; i < (kOffRing - kOffX) / 16; i += kSimt) z[i] = make_uint4(0, 0, 0, 0);
  }
  if (warp == 9) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(
        smem_u32((const void*)s_tmem)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *s_tmem;
  stamp(dk, 1);
  // everything above touched only this CTA's shared memory, TMEM and the weights; the mel rows, frame maxima and
  // emotion-stream outputs read below come from the previous kernels of the stream.  Early release (the fused forward,
  // one window per clip): the frontend's consumer warps count up *early_flag once the rows of the first early_items
  // clips are stored, which is long before its last CTA has finished -- this kernel's CTAs take SMs as the frontend's
  // CTAs leave them, and with the flag they start their first windows at once instead of idling until the frontend's
  // slowest CTA is done.  Acquire: one lane per warp polls, the warp barrier orders the other lanes behind it; the mel-row
  // producer adds a proxy fence (its reads are TMA copies).  Items from early_items on wait for griddepcontrol.wait.
  if constexpr (M == CoreMode::Early) {
    if (lane == 0) {
      unsigned seen = early_seen;
      for (uint32_t spin = 0; seen < p.early_target; ++spin) {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(p.early_flag) : "memory");
        if (seen < p.early_target) {
          __nanosleep(64);
          if (spin > (1u << 22)) __trap();
        }
      }
    }
    __syncwarp();
  } else {
    pdl_wait();
  }
  // (early_items is a multiple of the grid: a CTA's first item that the flag does not cover is early_items + blockIdx.x)
  const int first_late_item = M == CoreMode::Early ? p.early_items + (int)blockIdx.x : 0;
  // (no griddepcontrol.launch_dependents here: released early, the next forward's frontend CTAs take the SMs that this
  // kernel's last partial round of windows leaves idle and the step gets 11 us SLOWER -- measured, 198.6 vs 209.5 us)

  const int n_items = p.n_clips * p.n_out;
  const int T = p.frames_per_window;
  // mel power rows (linear buffer or per-stream ring; not prenormalised features) arrive by TMA
  const bool tma_mel = p.mel_long == nullptr;
  const int Tl = min(T, p.mel_seq);                              // long-term frames actually present
  const int n_mel_stages = tma_mel ? (Tl + kMelRows - 1) / kMelRows : 0;
  // the same for a window of wT = Rows::frames(win, T) frames: the launch's own unless every window has its own count
  // (Rows::kWindowFrames; the mel-row producer and the SIMT warps derive the stage count from the same window)
  auto long_frames = [&](int wT) { return Rows::kWindowFrames ? min(wT, p.mel_seq) : Tl; };
  auto mel_stages = [&](int wTl) {
    return Rows::kWindowFrames ? (tma_mel ? (wTl + kMelRows - 1) / kMelRows : 0) : n_mel_stages;
  };

  if (warp == 8) {
    // =========================================================== weight producer ========================
    if (lane == 0) {
      const unsigned char* src = reinterpret_cast<const unsigned char*>(W.tc_bf16);
      uint32_t slot = 0, phase = 0;
      const uint64_t pol_keep = l2_policy_keep();
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        long long* dp = (p.dbg != nullptr && blockIdx.x == 0 && item < 2 * (int)gridDim.x) ? p.dbg + 32 + 16 * (item / gridDim.x) : nullptr;
        for (int s = 0; s < kStagesPerWindow; ++s) {
          mbar_wait(bar_empty + 8 * slot, phase ^ 1);
          if (s >= kStagesPerWindow - 4) stamp(dp, s - (kStagesPerWindow - 4));
          if (s == 0) stamp(dp, 4);
          if (s == kStagesG1 - 1) stamp(dp, 5);
          if (s == kStagesG1) stamp(dp, 6);
          if (s == kStagesPerWindow - 5) stamp(dp, 7);
          mbar_expect_tx(bar_full + 8 * slot, kStageBytes);
          // the pre-tiled buffer holds [G1 | S tile 0, 1 | VT tile 0, 1 | H1]; the VT tiles are streamed before the S tiles
          // so that their epilogue runs while the S tiles are still on the tensor core
          const int ss = s < kStagesG1 || s >= kStagesG1 + 16 ? s : (s < kStagesG1 + 8 ? s + 8 : s - 8);
          bulk_g2s_hint(sbase + kOffRing + slot * kStageBytes, src + (size_t)ss * kStageBytes, kStageBytes,
                        bar_full + 8 * slot, pol_keep);
          if (++slot == kWRing) slot = 0, phase ^= 1;
        }
      }
    }
  } else if (warp == 10) {
    // =========================================================== mel-row producer =======================
    // a window's plain mel rows [0, Tl) are contiguous in HBM (linear buffer), or at most two runs per stage of a
    // stream's ring (row k is slot (ring_base + k) % ring_frames); the SIMT warps stage them as the first GEMM's operand
    if (lane == 0 && tma_mel) {
      uint32_t slot = kWRing, phase = 0;
      const uint64_t pol_keep = l2_policy_keep(), pol_stream = l2_policy_stream();
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        long long* dp = (p.dbg != nullptr && blockIdx.x == 0 && item < 2 * (int)gridDim.x) ? p.dbg + 32 + 16 * (item / gridDim.x) : nullptr;
        const CoreWindow win = Rows::template window<false>(p, item);
        const int wTl = long_frames(Rows::frames(win, T)), w_stages = mel_stages(wTl);
        if (M == CoreMode::Early && (item == (int)blockIdx.x || item == first_late_item)) {
          if (item == first_late_item) pdl_wait();
          asm volatile("fence.proxy.async.global;" ::: "memory");  // generic-proxy acquire / wait above -> TMA reads below
        }
        const float* base = p.ring_frames > 0 ? p.power[0] + (size_t)win.owner * p.ring_frames * kTok
                                              : p.power[0] + Rows::row(p, win, 0, 0) * kTok;
        // Ring mode (the streaming step): with thousands of streams the rings (82 KB each: 335 MB for 4096 streams) do not
        // stay in L2 from one hop to the next, and a window's six stages pass through two ring slots one HBM latency after
        // the other.  The NEXT window's ring and frame maxima are pulled into L2 now, a whole window ahead (4096 streams:
        // p50 0.4285 -> 0.4175 ms per hop; a steady window is 19.4 k cycles here against 17.6 k in the batch forward).
        if (p.ring_frames > 0 && item + (int)gridDim.x < n_items) {
          const int nb = Rows::ring_stream(p, item + gridDim.x);
          const char* ring = reinterpret_cast<const char*>(p.power[0] + (size_t)nb * p.ring_frames * kTok);
          const uint32_t ring_bytes = (uint32_t)p.ring_frames * kTok * 4;
          for (uint32_t off = 0; off < ring_bytes; off += 16384) bulk_prefetch_l2(ring + off, min(16384u, ring_bytes - off));
          const uint32_t fm_bytes = ((uint32_t)p.ring_frames * 4) & ~15u;
          if (fm_bytes > 0 && ((reinterpret_cast<uintptr_t>(p.fmax[0]) | ((size_t)nb * p.ring_frames * 4)) & 15) == 0)
            bulk_prefetch_l2(p.fmax[0] + (size_t)nb * p.ring_frames, fm_bytes);
        }
        for (int s = 0; s < w_stages; ++s) {
          const int n = min(kMelRows, wTl - kMelRows * s);
          const uint32_t bytes = (uint32_t)n * kTok * 4;
          const uint32_t dst = sbase + kOffRing + slot * kStageBytes;
          mbar_wait(bar_empty + 8 * slot, phase ^ 1);
          if (s == 0) stamp(dp, 8);
          if (s == w_stages - 1) stamp(dp, 9);
          mbar_expect_tx(bar_full + 8 * slot, bytes);
          if (p.ring_frames > 0) {
            const int r0 = (Rows::ring_base(p, win) + kMelRows * s) % p.ring_frames;
            const int n1 = min(n, p.ring_frames - r0);
            bulk_g2s_hint(dst, base + (size_t)r0 * kTok, (uint32_t)n1 * kTok * 4, bar_full + 8 * slot, pol_keep);
            if (n1 < n)
              bulk_g2s_hint(dst + (uint32_t)n1 * kTok * 4, base, (uint32_t)(n - n1) * kTok * 4, bar_full + 8 * slot, pol_keep);
          } else {
            bulk_g2s_hint(dst, base + (size_t)s * kMelRows * kTok, bytes, bar_full + 8 * slot,
                          Rows::plain_rows_policy(p, pol_keep, pol_stream));
          }
          if (++slot == kRing) slot = kWRing, phase ^= 1;
        }
      }
    }
  } else if (warp == 9) {
    // =========================================================== MMA issuer ============================
    // The whole warp runs the loop (waits, slot bookkeeping, descriptor arithmetic are warp-uniform, so they live in
    // uniform registers); one elected lane issues the tcgen05 instructions.  With a single active thread instead
    // (`if (lane == 0)`) every UTCHMMA / UTCBAR sits in its own elect-and-branch loop fed by R2UR moves and a stage of
    // four MMAs took ~490 cycles to issue against 225-256 cycles of tensor time (scripts/microbench/
    // umma_operand_layout_rate.cu: the no-swizzle K-major operands themselves run at the M=128 floor).
    {
      uint32_t slot = 0, phase = 0, go_phase = 0;
      const uint32_t ring = sbase + kOffRing;
      auto advance = [&]() {
        if (++slot == kWRing) slot = 0, phase ^= 1;
      };
      for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        long long* dm = (p.dbg != nullptr && lane == 0 && blockIdx.x == 0 && item < 2 * (int)gridDim.x) ? p.dbg + 64 + 16 * (item / gridDim.x) : nullptr;
        // ---- G1: 9 stages of [256 x 32] weights; the last stage carries K = 256..271 only
        mbar_wait(bar_go, go_phase), go_phase ^= 1;
        stamp(dm, 0);
        tc_fence_after();
        for (int s = 0; s < kStagesG1; ++s) {
          mbar_wait(bar_full + 8 * slot, phase);
          if (s < 3) stamp(dm, 12 + s);
          if (s == kStagesG1 - 1) stamp(dm, 15);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t a = smem_desc(sbase + kOffX + s * 512, 128, kA1Sbo);
            const uint64_t b = smem_desc(ring + slot * kStageBytes, 128, 4 * 128);
            tc_mma_bf16(tmem + kColD1, a, b, idesc_bf16(128, 256), s != 0);
            if (s != kStagesG1 - 1) tc_mma_bf16(tmem + kColD1, a + (256 >> 4), b + (256 >> 4), idesc_bf16(128, 256), 1);
            tc_commit(bar_empty + 8 * slot);
            if (s == kStagesG1 - 1) tc_commit(bar_done);
          }
          __syncwarp();
          advance();
        }
        stamp(dm, 1);
        // ---- VT (2 tiles), then S (2 tiles): A = weight stage [128 x 64], B = enc [80 x 256]
        mbar_wait(bar_go, go_phase), go_phase ^= 1;
        stamp(dm, 2);
        tc_fence_after();
        for (int js = 0; js < 4 * kStagesTile; ++js) {
          const int tile = js >> 2, s = js & 3;  // tiles 0, 1: VT; 2, 3: S
          const uint32_t d = tmem + (tile < 2 ? kColVT + 80 * tile : kColS + 80 * (tile - 2));
          mbar_wait(bar_full + 8 * slot, phase);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t a = smem_desc(ring + slot * kStageBytes, 128, 8 * 128);
            const uint64_t b = smem_desc(sbase + kOffE + s * 1024, 128, kESbo);
#pragma unroll
            for (int j = 0; j < 4; ++j)
              tc_mma_bf16(d, a + j * (256 >> 4), b + j * (256 >> 4), idesc_bf16(128, 80), (s | j) != 0);
            tc_commit(bar_empty + 8 * slot);
            if (js == 2 * kStagesTile - 1) tc_commit(bar_vt);
            if (js == 4 * kStagesTile - 1) tc_commit(bar_done);
          }
          __syncwarp();
          advance();
        }
        stamp(dm, 3);
        // ---- PV: A = P tile [128 x 80], B = vT tile [128 x 80]
        mbar_wait(bar_go, go_phase), go_phase ^= 1;
        stamp(dm, 4);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            const uint64_t a = smem_desc(sbase + kOffE + t * kPTile, 128, kPSbo);
            const uint64_t b = smem_desc(sbase + kOffVT + t * kPTile, 128, kPSbo);
#pragma unroll
            for (int j = 0; j < 5; ++j)
              tc_mma_bf16(tmem + kColO + 128 * t, a + j * (256 >> 4), b + j * (256 >> 4), idesc_bf16(128, 128), j != 0);
          }
          tc_commit(bar_done);
        }
        __syncwarp();
        stamp(dm, 5);
        // ---- H1: A = Oflat [128(28) x 256], B = weight stage [128 x 64]
        mbar_wait(bar_go, go_phase), go_phase ^= 1;
        stamp(dm, 6);
        tc_fence_after();
        for (int s = 0; s < kStagesTile; ++s) {
          mbar_wait(bar_full + 8 * slot, phase);
          stamp(dm, 8 + s);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t a = smem_desc(sbase + kOffE + s * 1024, 128, kESbo);
            const uint64_t b = smem_desc(ring + slot * kStageBytes, 128, 8 * 128);
#pragma unroll
            for (int j = 0; j < 4; ++j)
              tc_mma_bf16(tmem + kColH, a + j * (256 >> 4), b + j * (256 >> 4), idesc_bf16(128, 128), (s | j) != 0);
            tc_commit(bar_empty + 8 * slot);
            if (s == kStagesTile - 1) tc_commit(bar_done);
          }
          __syncwarp();
          advance();
        }
        stamp(dm, 7);
      }
    }
  } else {
    // =========================================================== SIMT warps 0-7 ========================
    // warpgroup wg = warp / 4; warps w and w + 4 both own TMEM lanes 32 (w % 4) .. +31, so the two warpgroups split
    // every epilogue between them (LayerNorm: column halves; softmax / vT / O: one tile of 4 heads each)
    uint32_t done_phase = 0, vt_phase = 0, slot = kWRing, phase = 0;  // (slot, phase): the mel-row ring
    const int wg = warp >> 2, wq = warp & 3;
    const int row = 32 * wq + lane;                                        // TMEM lane == accumulator row
    const uint32_t lane_taddr = tmem + ((uint32_t)(32 * wq) << 16);
    const bool prenorm = p.mel_long != nullptr;
    // first-GEMM operand of one window: dB reference, normalise, bf16, K-major core matrices in the X region
    // this thread's share of a window's per-frame maxima (its dB reference is their maximum): independent loads, issued
    // together; for the stage-ahead path they are requested one phase early so that their latency is never waited for
    auto frame_max_partial = [&](const int item) {
      float mx = -INFINITY;
      if (!prenorm) {
        const CoreWindow win = Rows::template window<true>(p, item);
        const int wT = Rows::frames(win, T);
        for (int k0 = tid; k0 < wT; k0 += 3 * kSimt) {
          float f[3];
#pragma unroll
          for (int u = 0; u < 3; ++u) {
            const int k = k0 + u * kSimt;
            f[u] = -INFINITY;
            if (k < wT) {
              const int v = win.plain_only ? 0 : Rows::variant(p, win, wT, k);
              f[u] = p.fmax[v][Rows::row(p, win, v, k)];
            }
          }
          mx = fmaxf(fmaxf(mx, f[0]), fmaxf(f[1], f[2]));
        }
      }
      return mx;
    };
    auto stage_window = [&](const int item, float mx, long long* ds) {
      const CoreWindow win = Rows::template window<true>(p, item);
      const int wT = Rows::frames(win, T), wTl = long_frames(wT), w_stages = mel_stages(wTl);
      // ---- window dB reference
      float ref_db = 0.0f;
      if (!prenorm) {
        mx = warp_max(mx);
        if (lane == 0) s_red[warp] = mx;
        simt_barrier();
        ref_db = fmaxf(fmaxf(fmaxf(s_red[0], s_red[1]), fmaxf(s_red[2], s_red[3])),
                       fmaxf(fmaxf(s_red[4], s_red[5]), fmaxf(s_red[6], s_red[7])));
        simt_barrier();
      }
      stamp(ds, 10);
      if (tma_mel) {
        // ---- A1 from the TMA-staged rows: Xn[channel j][time t] as bf16, one 16-byte store = 8 frames of a channel
        // rows that are not plain frames of this window (short-term detail, edge variants) are fetched directly, early
        float extra[5] = {0.f, 0.f, 0.f, 0.f, 0.f};       // [0..2] short-term frames T-3+s, [3] lo-edge frame 0, [4] hi-edge frame T-1
        if (tid < kTok) {
#pragma unroll
          for (int e = 0; e < 3; ++e) {
            const int k = wT >= 3 ? wT - 3 + e : (e < wT ? e : -1);
            if (k >= 0) {
              const int var = win.plain_only ? 0 : Rows::variant(p, win, wT, k);
              extra[e] = p.power[var][Rows::row(p, win, var, k) * kTok + tid];
            } else {
              extra[e] = -INFINITY;
            }
          }
          if (!win.plain_only && p.n_edge > 0) {
            if (Rows::window_starts(p, win)) extra[3] = __ldg(p.power[1] + Rows::row(p, win, 1, 0) * kTok + tid);
            if (wT - 1 < wTl) extra[4] = __ldg(p.power[2] + Rows::row(p, win, 2, wT - 1) * kTok + tid);
          }
        }
        for (int s = 0; s < w_stages; ++s) {
          mbar_wait(bar_full + 8 * slot, phase);
          const float* raw = reinterpret_cast<const float*>(smem + kOffRing + slot * kStageBytes);
          const int rows = min(kMelRows, wTl - kMelRows * s);
          const int chunks = (rows + 7) >> 3;
          if (rows == kMelRows) {
            // full stage: 6 chunks x 80 channels = 480 items of 8 frames; a thread's two items are loaded together
            static_assert(kMelRows * kTok / 8 <= 2 * kSimt, "two items per thread cover a stage");
            const int i0 = tid, i1 = tid + kSimt;
            const bool two = i1 < kMelRows * kTok / 8;
            const int c0 = i0 / kTok, j0 = i0 % kTok, c1 = two ? i1 / kTok : c0, j1 = two ? i1 % kTok : j0;
            float v0[8], v1[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              v0[e] = raw[(8 * c0 + e) * kTok + j0];
              v1[e] = raw[(8 * c1 + e) * kTok + j1];
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              v0[e] = normalise_bf16(v0[e], ref_db, true);
              v1[e] = normalise_bf16(v1[e], ref_db, true);
            }
            *reinterpret_cast<uint4*>(smem + kOffX + (j0 >> 3) * kA1Sbo + (6 * s + c0) * 128 + (j0 & 7) * 16) = pack8_bf16(v0);
            if (two)
              *reinterpret_cast<uint4*>(smem + kOffX + (j1 >> 3) * kA1Sbo + (6 * s + c1) * 128 + (j1 & 7) * 16) = pack8_bf16(v1);
          } else {
            for (int idx = tid; idx < chunks * kTok; idx += kSimt) {
              const int c = idx / kTok, j = idx % kTok;
              float v[8];
#pragma unroll
              for (int e = 0; e < 8; ++e)
                v[e] = 8 * c + e < rows ? normalise_bf16(raw[(8 * c + e) * kTok + j], ref_db, true) : 0.0f;
              *reinterpret_cast<uint4*>(smem + kOffX + (j >> 3) * kA1Sbo + (6 * s + c) * 128 + (j & 7) * 16) =
                  pack8_bf16(v);
            }
          }
          simt_barrier();                                   // every thread is done reading this ring slot
          if (s == 0) stamp(ds, 11);
          if (s == 2) stamp(ds, 12);
          if (s == w_stages - 1) stamp(ds, 13);
          if (tid == 0) mbar_arrive(bar_empty + 8 * slot);
          if (++slot == kRing) slot = kWRing, phase ^= 1;
        }
        if (tid < kTok) {
          const int j = tid;
          unsigned char* arow = smem + kOffX + (j >> 3) * kA1Sbo + (j & 7) * 16;
          // K chunks past the long-term frames: zeros up to frame 255, then [short-term x3, 0 x5], then zeros
          for (int c = (wTl + 7) >> 3; c < kLongChunks; ++c) *reinterpret_cast<uint4*>(arow + c * 128) = make_uint4(0, 0, 0, 0);
          float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int e = 0; e < 3; ++e) v[e] = normalise_bf16(extra[e], ref_db, true);
          v[3] = 1.0f;  // operand column k_mel: multiplies the encoder-bias row of the weights
          *reinterpret_cast<uint4*>(arow + kLongChunks * 128) = pack8_bf16(v);
          *reinterpret_cast<uint4*>(arow + (kLongChunks + 1) * 128) = make_uint4(0, 0, 0, 0);
          // edge frames inside the long-term range see zeros beyond the window edge: patch them in place
          // (frame m and frame T-1-m for m < n_edge: one per side at 30 fps, two at 60 fps)
          for (int m = 0; !win.plain_only && m < p.n_edge; ++m) {
            if (Rows::window_starts(p, win)) {
              const float lo = m == 0 ? extra[3] : __ldg(p.power[1 + 2 * m] + Rows::row(p, win, 1 + 2 * m, m) * kTok + j);
              *reinterpret_cast<__nv_bfloat16*>(arow + (m >> 3) * 128 + (m & 7) * 2) =
                  __float2bfloat16_rn(normalise_bf16(lo, ref_db, true));
            }
            const int k = wT - 1 - m;
            if (k < wTl) {
              const float x = m == 0 ? extra[4] : __ldg(p.power[2 + 2 * m] + Rows::row(p, win, 2 + 2 * m, k) * kTok + j);
              *reinterpret_cast<__nv_bfloat16*>(arow + (k >> 3) * 128 + (k & 7) * 2) =
                  __float2bfloat16_rn(normalise_bf16(x, ref_db, true));
            }
          }
        }
      } else {
      // ---- A1: Xn[channel j][time t] as bf16.  One item = 8 consecutive frames x 4 consecutive channels:
        // 8 independent 16-byte loads (frame rows are 320 B apart), then one 16-byte store per channel.
        // Two items are in flight per thread so that ~32 KB of loads per CTA hide the L2 latency.
        {
          constexpr int kQuads = kTok / 4;                 // 20 channel quads per frame
          constexpr int kItems = kA1Chunks * kQuads;       // 680
          auto load_item = [&](int idx, float4 (&r)[8]) {
            const int c = idx / kQuads, q = idx % kQuads;
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int t = 8 * c + e;
              float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
              // (this branch serves the prenormalised-features entry point only: raw mel power always comes through the
              // TMA mel ring above)
              if (t < kKMel) {
                if (t >= p.mel_seq)
                  x = __ldg(reinterpret_cast<const float4*>(p.mel_short + ((size_t)win.owner * 3 + (t - p.mel_seq)) * kTok) + q);
                else if (t < p.n_long)
                  x = __ldg(reinterpret_cast<const float4*>(p.mel_long + ((size_t)win.owner * p.n_frames + t) * kTok) + q);
              }
              r[e] = x;
            }
          };
          auto store_item = [&](int idx, const float4 (&r)[8]) {
            const int c = idx / kQuads, q = idx % kQuads;
            float v[4][8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              v[0][e] = r[e].x, v[1][e] = r[e].y, v[2][e] = r[e].z, v[3][e] = r[e].w;
              if (8 * c + e == kKMel)  // operand column k_mel: multiplies the encoder-bias row of the weights
                v[0][e] = v[1][e] = v[2][e] = v[3][e] = 1.0f;
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int j = 4 * q + i;
              *reinterpret_cast<uint4*>(smem + kOffX + (j >> 3) * kA1Sbo + c * 128 + (j & 7) * 16) = pack8_bf16(v[i]);
            }
          };
          for (int idx = tid; idx < kItems; idx += 2 * kSimt) {
            float4 r0[8], r1[8];
            const bool two = idx + kSimt < kItems;
            load_item(idx, r0);
            if (two) load_item(idx + kSimt, r1);
            store_item(idx, r0);
            if (two) store_item(idx + kSimt, r1);
          }
        }
      }
    };
    if (kStageAhead && (int)blockIdx.x < n_items) {
      stage_window(blockIdx.x, frame_max_partial(blockIdx.x), nullptr);
      fence_async_smem();
      mbar_arrive(bar_go);
      stamp(dk, 2);
    }
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int expr_row = Rows::expr_row(p, item);
      const bool has_next = item + (int)gridDim.x < n_items;
      long long* ds = (p.dbg != nullptr && blockIdx.x == 0 && tid == 0 && item < 2 * (int)gridDim.x) ? p.dbg + 16 * (item / gridDim.x) : nullptr;
      stamp(ds, 0);
      if (!kStageAhead) {
        if (M == CoreMode::Early && item == first_late_item) pdl_wait();  // (early release: this window's clip is not covered by the flag)
        stage_window(item, frame_max_partial(item), ds);
        fence_async_smem();
        mbar_arrive(bar_go);
      }
      stamp(ds, 1);
      // (early release: the next window is this CTA's first whose clip the flag does not cover -- it is read from here on)
      if (M == CoreMode::Early && has_next && item + (int)gridDim.x == first_late_item) pdl_wait();
      const float mx_next = kStageAhead && has_next ? frame_max_partial(item + gridDim.x) : -INFINITY;

      // ---- E1: bias + LayerNorm of token row tid -> enc (bf16, K-major) -------------------------------
      mbar_wait(bar_done, done_phase), done_phase ^= 1;
      stamp(ds, 2);
      tc_fence_after();
      {
        // warp-uniform guard: tcgen05.ld is warp-collective; the wq == 3 warps own only padding rows (96..127)
        const bool live = 32 * wq < kTok;
        const int cb = 128 * wg;                       // this warpgroup's half of the 256 features
        if (live) {
          float sa[4] = {0.f, 0.f, 0.f, 0.f}, qa[4] = {0.f, 0.f, 0.f, 0.f};  // four chains each (latency)
#pragma unroll
          for (int c0 = 0; c0 < 128; c0 += 32) {
            float v[32];
            tmem_ld32(lane_taddr + kColD1 + cb + c0, v);
#pragma unroll
            for (int i = 0; i < 32; ++i) {  // (the encoder bias came in through the GEMM)
              sa[i & 3] += v[i];
              qa[i & 3] = fmaf(v[i], v[i], qa[i & 3]);
            }
          }
          s_ln[wg * 128 + row] = (sa[0] + sa[1]) + (sa[2] + sa[3]);
          s_ln[256 + wg * 128 + row] = (qa[0] + qa[1]) + (qa[2] + qa[3]);
        }
        simt_barrier();
        if (live) {
          const float mean = (s_ln[row] + s_ln[128 + row]) * (1.0f / 256);
          const float var = fmaxf((s_ln[256 + row] + s_ln[384 + row]) * (1.0f / 256) - mean * mean, 0.0f);
          const float rstd = rsqrtf(var + W.ln_eps), shift = -mean * rstd;
          unsigned char* erow = smem + kOffE + (row >> 3) * kESbo + (row & 7) * 16;
          for (int c0 = 0; c0 < 128; c0 += 32) {
            float v[32];
            tmem_ld32(lane_taddr + kColD1 + cb + c0, v);
#pragma unroll
            for (int i = 0; i < 32; ++i)
              v[i] = fmaf(v[i], rstd, shift);  // normalised only: mel_norm.weight / bias live in the qk / wv weights
            if (row < kTok) {
#pragma unroll
              for (int q = 0; q < 4; ++q)
                *reinterpret_cast<uint4*>(erow + ((cb + c0) / 8 + q) * 128) = pack8_bf16(v + 8 * q);
            }
          }
        }
      }
      tc_fence_before();
      fence_async_smem();
      mbar_arrive(bar_go);
      stamp(ds, 3);
      if (kStageAhead) {
        // the S/VT GEMMs (weight-streaming bound, ~8 k cycles) need nothing from these warps: stage the next window now
        if (has_next) stage_window(item + gridDim.x, mx_next, ds);
      }

      // ---- E3 vT rows (+ bv) -> vT tiles, as soon as the VT tiles are done (the S tiles are still streaming) ----------
      mbar_wait(bar_vt, vt_phase), vt_phase ^= 1;
      tc_fence_after();
      {
        const int t = wg;
        float s[kTok];
        {
          float v[32];
          tmem_ld32(lane_taddr + kColVT + 80 * t, v);
#pragma unroll
          for (int i = 0; i < 32; ++i) s[i] = v[i];
          tmem_ld32(lane_taddr + kColVT + 80 * t + 32, v);
#pragma unroll
          for (int i = 0; i < 32; ++i) s[32 + i] = v[i];
          float u[16];
          tmem_ld16(lane_taddr + kColVT + 80 * t + 64, u);
#pragma unroll
          for (int i = 0; i < 16; ++i) s[64 + i] = u[i];
        }
        const float bias = s_bv[128 * t + row];
#pragma unroll
        for (int i = 0; i < kTok; ++i) s[i] += bias;
        unsigned char* vrow = smem + kOffVT + t * kPTile + (row >> 3) * kPSbo + (row & 7) * 16;
#pragma unroll
        for (int c = 0; c < 10; ++c) *reinterpret_cast<uint4*>(vrow + c * 128) = pack8_bf16(s + 8 * c);
      }
      // ---- E2 softmax rows -> P tiles (over enc, which the S GEMMs have now finished reading) -------------------
      mbar_wait(bar_done, done_phase), done_phase ^= 1;
      stamp(ds, 4);
      tc_fence_after();
      {
        const int t = wg;
        // row `row` of tile t is (head 4 t + wq, query lane); queries 28..31 are padding
        float s[kTok];
        {
          float v[32];
          tmem_ld32(lane_taddr + kColS + 80 * t, v);
#pragma unroll
          for (int i = 0; i < 32; ++i) s[i] = v[i];
          tmem_ld32(lane_taddr + kColS + 80 * t + 32, v);
#pragma unroll
          for (int i = 0; i < 32; ++i) s[32 + i] = v[i];
          float u[16];
          tmem_ld16(lane_taddr + kColS + 80 * t + 64, u);
#pragma unroll
          for (int i = 0; i < 16; ++i) s[64 + i] = u[i];
        }
        // four interleaved chains for the maximum and the sum: with two warps per scheduler an 80-long dependent chain is
        // pure latency
        float m4[4] = {s[0], s[1], s[2], s[3]};
#pragma unroll
        for (int i = 4; i < kTok; ++i) m4[i & 3] = fmaxf(m4[i & 3], s[i]);
        const float m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
        float sum4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int i = 0; i < kTok; ++i) {
          s[i] = __expf(s[i] - m);  // (the probabilities are rounded to bf16 next: MUFU.EX2 precision is ample)
          sum4[i & 3] += s[i];
        }
        const float sum = (sum4[0] + sum4[1]) + (sum4[2] + sum4[3]);
        const float inv = lane < KOE_N_MOUTH ? 1.0f / sum : 0.0f;
#pragma unroll
        for (int i = 0; i < kTok; ++i) s[i] *= inv;
        unsigned char* prow = smem + kOffE + t * kPTile + (row >> 3) * kPSbo + (row & 7) * 16;
#pragma unroll
        for (int c = 0; c < 10; ++c) *reinterpret_cast<uint4*>(prow + c * 128) = pack8_bf16(s + 8 * c);
        if (p.attn_out != nullptr && lane < KOE_N_MOUTH) {
          float* dst = p.attn_out + ((size_t)item * KOE_N_MOUTH + lane) * kTok;
#pragma unroll
          for (int i = 0; i < kTok; ++i) atomicAdd(dst + i, s[i] * (1.0f / KOE_N_HEADS));
        }
      }
      tc_fence_before();
      fence_async_smem();
      mbar_arrive(bar_go);
      stamp(ds, 5);

      // ---- E4: O[h][q][0..31] (diagonal block of tile t) -> Oflat row q, K = 32 h + d -------------------
      mbar_wait(bar_done, done_phase), done_phase ^= 1;
      stamp(ds, 6);
      tc_fence_after();
      {
        const int t = wg;
        float v[32];
        tmem_ld32(lane_taddr + kColO + 128 * t + 32 * wq, v);
        if (lane < KOE_N_MOUTH) {
          const int h = 4 * t + wq;
          unsigned char* orow = smem + kOffE + (lane >> 3) * kESbo + (lane & 7) * 16 + (4 * h) * 128;
#pragma unroll
          for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(orow + q * 128) = pack8_bf16(v + 8 * q);
        }
      }
      tc_fence_before();
      fence_async_smem();
      mbar_arrive(bar_go);
      stamp(ds, 7);

      // ---- E5: decoder tail on rows 0..27 + fusion -----------------------------------------------------
      mbar_wait(bar_done, done_phase), done_phase ^= 1;
      stamp(ds, 8);
      tc_fence_after();
      if (kStageAhead && has_next) {  // the next window's first GEMM (TMEM columns [0, 256)) runs under the decoder tail
        fence_async_smem();
        mbar_arrive(bar_go);
      }
      if (warp == 0) {
        float logit = 0.0f;
        for (int c0 = 0; c0 < 128; c0 += 32) {
          float v[32];
          tmem_ld32(lane_taddr + kColH + c0, v);
#pragma unroll
          for (int i = 0; i < 32; ++i) logit = fmaf(fmaxf(v[i] + s_ba[c0 + i], 0.0f), s_w2[c0 + i], logit);
        }
        if (lane < KOE_N_MOUTH) {
          const float y = 1.0f / (1.0f + expf(-(logit + W.b2)));
          const int idx = __ldg(W.mouth_idx + lane);
          const size_t o_off = (size_t)item * KOE_N_BLENDSHAPES + idx;
          p.out[o_off] = fminf(fmaxf(__ldg(W.coef + idx) * y, 0.0f), 1.0f);
          if (p.sigmoid_out != nullptr) p.sigmoid_out[o_off] = y;
        }
      } else if (warp == 1 && lane < KOE_N_EXPR && p.expr_sigmoid != nullptr) {  // (NULL: the emotion kernel writes these)
        const float y = __ldg(p.expr_sigmoid + expr_row);
        const int idx = __ldg(W.expr_idx + lane);
        const size_t o_off = (size_t)item * KOE_N_BLENDSHAPES + idx;
        p.out[o_off] = fminf(fmaxf(__ldg(W.coef + idx) * y, 0.0f), 1.0f);
        if (p.sigmoid_out != nullptr) p.sigmoid_out[o_off] = y;
      }
      stamp(ds, 9);
      tc_fence_before();
      simt_barrier();  // the next window's A1 staging overwrites the P tiles only after every row is consumed
    }
    stamp(dk, 3);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
  }
  if constexpr (M == CoreMode::Early) {
    // this kernel must not complete before the kernels ahead of it have (what follows waits on this kernel only); the
    // last CTA out clears the flag and the exit counter for the next forward on this stream
    pdl_wait();
    if (tid == 0 && atomicAdd(p.early_flag + 1, 1u) == gridDim.x - 1) {
      p.early_flag[0] = 0;
      p.early_flag[1] = 0;
    }
  }
  if (p.dbg != nullptr && tid == 0) {
    unsigned long long g;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
    p.dbg[129 + 2 * blockIdx.x] = (long long)g;
  }
}

}  // namespace tc

int dual_stream_tc_grid(int n_items) {
  int sms = 0;
  if (sm_count(&sms) != cudaSuccess) return 0;
  return std::min(n_items, sms);
}

// sets the shared-memory size of the instantiation once per device, then launches it behind the previous kernel
template <int KMEL, CoreMode M>
static int launch_tc(const CoreParams& p, int grid, cudaStream_t stream) {
  static bool configured[64] = {false};
  int dev = 0;
  KOE_CUDA(cudaGetDevice(&dev));
  KOE_REQUIRE(dev >= 0 && dev < 64, "device index too large");
  if (!configured[dev]) {
    KOE_CUDA(cudaFuncSetAttribute(tc::dual_stream_tc_kernel<KMEL, M>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  tc::kSmemBytes));
    configured[dev] = true;
  }
  KOE_CUDA(launch_after_primary_starts(tc::dual_stream_tc_kernel<KMEL, M>, dim3(grid), dim3(tc::kThreads), tc::kSmemBytes,
                                       stream, p));
  return KOE_OK;
}
template <CoreMode M>
static int launch_tc(const CoreParams& p, int grid, cudaStream_t stream) {
  return p.w.k_mel == 259 ? launch_tc<259, M>(p, grid, stream) : launch_tc<515, M>(p, grid, stream);
}

int launch_dual_stream_tc(const CoreParams& p, CoreMode mode, cudaStream_t stream) {
  if (p.w.k_mel != 259 && p.w.k_mel != 515)
    return fail(KOE_E_UNSUPPORTED, "tensor-core path is built for k_mel = 259 (30 fps) and 515 (60 fps); got %d", p.w.k_mel);
  const int need_stages = p.w.k_mel == 259 ? tc::Geo<259>::kStagesPerWindow : tc::Geo<515>::kStagesPerWindow;
  if (p.w.tc_bf16 == nullptr || p.w.tc_bv == nullptr || p.w.tc_stages != need_stages)
    return fail(KOE_E_INVALID, "tensor-core path: koe_core_weights.tc_bf16 is missing (%d stages, need %d)",
                p.w.tc_stages, need_stages);
  int sms = 0;
  KOE_CUDA(sm_count(&sms));
  const int grid = std::min(p.n_clips * p.n_out, sms);
  if (mode == CoreMode::Early)
    KOE_REQUIRE(p.n_out == 1 && p.early_items > 0 && p.early_items % grid == 0 && p.early_target > 0,
                "tensor-core path: bad early-release parameters");
  if (mode == CoreMode::Varlen)
    KOE_REQUIRE(p.n_out == 1 && p.ring_frames == 0 && p.expr_sigmoid == nullptr, "tensor-core path: bad varlen parameters");
  if (mode == CoreMode::Pool || mode == CoreMode::PoolHops)
    KOE_REQUIRE(p.n_out == 1 && p.ring_frames > 0 && p.attn_out == nullptr, "tensor-core path: bad stream-pool parameters");
  if (p.attn_out != nullptr)  // head-average is accumulated with atomics
    KOE_CUDA(cudaMemsetAsync(p.attn_out, 0, (size_t)p.n_clips * p.n_out * KOE_N_MOUTH * tc::kTok * sizeof(float),
                             stream));
  int rc = KOE_OK;
  switch (mode) {
    case CoreMode::Windows: rc = launch_tc<CoreMode::Windows>(p, grid, stream); break;
    case CoreMode::Early: rc = launch_tc<CoreMode::Early>(p, grid, stream); break;
    case CoreMode::Pool: rc = launch_tc<CoreMode::Pool>(p, grid, stream); break;
    case CoreMode::Varlen: rc = launch_tc<CoreMode::Varlen>(p, grid, stream); break;
    case CoreMode::PoolHops: rc = launch_tc<CoreMode::PoolHops>(p, grid, stream); break;
  }
  if (rc != KOE_OK) return rc;
  count_launch();
  KOE_CUDA(cudaGetLastError());
  return KOE_OK;
}

}  // namespace koe
