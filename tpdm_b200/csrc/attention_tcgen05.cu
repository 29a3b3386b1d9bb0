// tpdm_b200 -- joint text+image attention, softmax(Q K^T / sqrt(d)) V, on tcgen05 tensor cores (sm_100a).
//
// Replaces F.scaled_dot_product_attention inside diffusers' JointAttnProcessor2_0 as called from
// JointTransformerBlock (/root/reference/src/models/stable_diffusion_3/transformer_sd3.py:361-365): image tokens first,
// text tokens second, no mask, no dropout.  Q/K/V are read straight out of the token-major fused-QKV GEMM output
// [Bt][S][3*H*dp] through 4-D TMA tensor maps (no head permute, no concat copy); O is written token-major [Bt][S][H*dp]
// so the output projection consumes it as-is.
//
// One CTA = one 128-row query tile of one (batch, head); 384 threads; two CTAs co-resident per SM (dp = 64).
//   warp 0      TMA producer  (Q once, K/V tiles of 128 keys through a 2-stage smem ring)
//   warp 1      MMA issuer for S = Q K^T: one 128 x 128 score tile per K tile (SS, dp/16 instructions of N = 128)
//   warp 3      MMA issuer for O += P V (A = P from TMEM, B = V MN-major from smem, 8 instructions of N = dp)
//   warp 2      TMEM allocator
//   warps 4-11  softmax, two threads per query row: warps 4-7 take keys [0,64) of every tile, warps 8-11 keys [64,128) of the same
//               rows (a warp reaches the TMEM lanes 32 * (warp % 4) ..., so the pairs (4,8), (5,9), ... share rows).  Four softmax
//               warps per scheduler: with two the kernel was bound by the latency of each warp's own instruction stream.
// TMEM per CTA: S 128 fp32 columns, P 64 columns (128 keys of packed bf16), O dp columns -- ONE buffer each.  Overlap inside a
// CTA comes from releasing S as soon as its last chunk is in registers (Q K^T of the next tile then runs under the
// last quarter of this tile's exponentials and under P V), overlap on the SM from the second co-resident CTA.
//
// Why 128-key tiles (round 2; measurements in profiles/r02_*.txt):
//  * tools/microbench/mma_issue_rate.cu: an SS MMA of N = 64 cannot run faster than one per 48 cycles (its 6 KB of operands come
//    out of shared memory at 128 B/clk) although it holds the tensor pipe for 32, N = 128 runs at the pipe rate (64); issued
//    from inside `if (lane == 0)` -- as round 1 did -- every MMA additionally paid a waterfall loop (56-72 cycles in isolation,
//    115-180 next to busy warps: the round-1 timeline, tools/attn_trace.py, shows 539 cycles per 64 keys in the Q K^T issuer
//    alone).  N = 128 halves the instruction count and the MMAs are now issued by the converged warp (umma_*_elect).
//  * the same timeline showed ~625 of the 1460 cycles a softmax warp spent per 64 keys in mbarrier round trips, exposed TMEM
//    load latency and the P hand-over; with 128 keys per round trip that cost is halved, and the chunk loads are software
//    pipelined (the load of chunk c+1 is in flight while chunk c is exponentiated).
//  * tools/microbench/tmem_read_rate.cu: tcgen05.ld moves 490-1050 B/clk/SM, so reading S back in fp32 is NOT a floor (round 1
//    assumed 64 B/clk/SM); the floor of this kernel is the MUFU: 16 ex2 / clk / SM = 1024 cycles per 128 x 128 scores.
// Softmax: fp32, exp2 with log2(e)/sqrt(d) folded into one FFMA2, in two flavours (attn_cta<DP, kFast>):
//  * FAST (what every CTA runs first, on warps 4-11).  No maximum inside the key loop: the reference m_ref only has to keep
//    exp2(s - m_ref) inside the fp32 / bf16 exponent range.  It starts as the row maximum of the first key tile and is guarded by
//    the ROW SUM the loop computes anyway, at a checkpoint every 4th tile: a half whose partial sum has passed 2^24 proposes a
//    shift by floor(log2 l) through shared memory, and both halves of the row apply it at the next checkpoint (O and l rescaled
//    by that power of two; see `tile` in the fast branch of attn_cta).  A row the guard cannot keep in range (l > 2^64, inf, NaN,
//    or an argument > 127 reaching the polynomial, which would wrap instead of overflowing) flags the CTA.
//  * EXACT (a flagged CTA reruns its tile with it on warps 4-7 before it exits).  Reference maximum m_used raised lazily: every
//    32-column chunk computes its own maximum (FMNMX3 trees, issued under the MUFU work of the previous chunk) and only when that
//    exceeds m_used by more than 2^kRescaleThreshold does the row take the (rare, exact) path that moves the reference and
//    rescales what was accumulated under the old one -- O, l and the P chunks of this tile already stored.
// fp32 sums and bf16 P carry 8 exponent bits, so running far above the reference costs no precision, and the final 1/l cancels
// the reference.  Round-2 measurements (B200, S = 4429, H = 24, Bt = 2): exact 320-327 us, fast 276 us; cuDNN SDPA: 283 us;
// everything tried on the way (four softmax warps per CTA: 288-292 us) is in profiles/r02_attention_experiments.txt.
#include <cuda_bf16.h>

#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "host.h"

namespace tpdm {

namespace {

constexpr int kFastThreads = 384;   // 4 control warps + 8 softmax warps (the exact redo pass uses softmax warps 4-7 only)
constexpr int kQT = 128;   // query rows per CTA
constexpr int kKT = 128;   // keys per K/V smem tile = keys per S tile
constexpr int kChunk = 32; // S columns per tcgen05.ld of the exact softmax
constexpr int kKVStages = 2;
constexpr float kRescaleThreshold = 32.0f;  // log2 units
// Every kPolyEvery-th pair of exponentials is computed on the FMA/ALU pipes (Cody-Waite range reduction + cubic minimax
// polynomial, max relative error 7.5e-5 -- P is rounded to bf16 anyway) instead of MUFU.EX2.
// Measured on B200 with this kernel (S = 4429, H = 24, Bt = 2; profiles/r02_attention_experiments.txt): none -> 343 us, every 8th ->
// 328 us, every 4th -> 324 us, every 2nd -> 325 us.  (Round 1's 64-key kernel was latency bound and got SLOWER with it.)
// Packing P with integer adds + PRMT instead of F2FP (which shares the XU pipe with MUFU) was measured too: 358 us, rejected.
constexpr int kPolyEvery = 4;
// -DTPDM_ATTN_TRACE: clock64() time stamps of one CTA's fast pass: softmax warp 4 (role 0, 8 slots per key tile, STRACE) and the two
// MMA-issuing warps (roles 1 and 2, 4 slots per key tile), read back with tpdm_attn_trace_read (tools/attn_trace.py).  Diagnostic
// builds only.
#ifdef TPDM_ATTN_TRACE
__device__ long long g_attn_trace[3][2048];
#define ATRACE(role, idx)                                                                       \
  do {                                                                                          \
    if (trace_on && lane == 0 && (idx) < 2048) g_attn_trace[role][idx] = clock64();             \
  } while (0)
#define STRACE(e)                                                                               \
  do {                                                                                          \
    if (warp == 4) ATRACE(0, 8 * j + (e));                                                      \
  } while (0)
// CTA-level stamps of two CTAs (an early and a late one): [0] kernel entry, [1] past pdl_wait, [2] TMEM allocated, [3] first score
// tile ready, [4] last tile's P handed over, [5] O stored, [6] exit; [7] = %globaltimer at entry, [8] at exit
__device__ long long g_cta_trace[2][16];
#define CTRACE(idx)                                                                             \
  do {                                                                                          \
    if (ctr >= 0 && threadIdx.x == 128) g_cta_trace[ctr][idx] = clock64();                      \
  } while (0)
#else
#define ATRACE(role, idx)
#define STRACE(e)
#define CTRACE(idx)
#endif

__device__ unsigned long long g_redo_total;   // CTAs that took the exact pass since the library was loaded (tpdm_attention_redo_total)

template <int DP>
struct AttnSmem {
  static constexpr int kTile = kQT * DP * 2;  // bytes of one Q / K / V tile
  static constexpr int kQOff = 0;
  static constexpr int kKOff = kTile;
  static constexpr int kVOff = kKOff + kKVStages * kTile;
  static constexpr int kBarOff = kVOff + kKVStages * kTile;
  static constexpr int kTotal = kBarOff + 256 + 1024;
  static constexpr uint32_t kTmemCols = DP == 64 ? 256 : 512;
  static constexpr uint32_t kSCol = 0;     // S: 128 fp32 columns
  static constexpr uint32_t kPCol = 128;   // P: 64 columns (128 keys, packed bf16)
  static constexpr uint32_t kOCol = 192;   // O: DP columns
};

// mbarriers of one CTA, in the order they are laid out behind the tiles
template <int DP>
struct AttnBars {
  uint64_t *q_full, *k_full, *v_full, *k_empty, *v_empty, *s_full, *s_free, *p_full, *pv_done;
  uint32_t* tmem_slot;
  __device__ explicit AttnBars(uint8_t* smem) {
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + AttnSmem<DP>::kBarOff);
    q_full = bars + 0;
    k_full = bars + 1;                 // [kKVStages]
    v_full = k_full + kKVStages;       // [kKVStages]
    k_empty = v_full + kKVStages;      // [kKVStages]
    v_empty = k_empty + kKVStages;     // [kKVStages]
    s_full = v_empty + kKVStages;      // MMA -> softmax : S(j) written
    s_free = s_full + 1;               // softmax -> MMA : S(j) is in registers
    p_full = s_free + 1;               // [2] softmax -> MMA : keys [0,64) / [64,128) of P(j) written (and O rescaled if needed)
    pv_done = p_full + 2;              // MMA -> softmax : P(j) V accumulated (P may be overwritten, O may be touched)
    tmem_slot = reinterpret_cast<uint32_t*>(pv_done + 1);
  }
  static constexpr int kCount = 1 + 4 * kKVStages + 5;
  // one thread; `again`: the barriers carry the phases of a finished tile (before the exact redo pass) and are invalidated first;
  // s_free completes with one arrival per softmax warp
  __device__ void init(bool again, uint32_t s_free_count) const {
    if (again) {
      for (int i = 0; i < kCount; ++i) mbar_inval(q_full + i);
    }
    mbar_init(q_full, 1);
    for (int i = 0; i < kKVStages; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&k_empty[i], 1);
      mbar_init(&v_empty[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(s_free, s_free_count);
    mbar_init(&p_full[0], 4);
    mbar_init(&p_full[1], 4);
    mbar_init(pv_done, 1);
    fence_barrier_init();
  }
};

__device__ __forceinline__ uint8_t* attn_smem_base() {
  extern __shared__ uint8_t smem_raw[];
  return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
}

// (p0, p1) = 2^(x0, x1) through MUFU.EX2, or with `poly` on the FMA/ALU pipes: 2^x = 2^n * 2^f, n = rint(x) read from the mantissa
// of x + 1.5*2^23, f = x - n in [-0.5, 0.5].  Below -126 the clamp flushes the result to ~0; an argument above 127 would wrap the
// exponent instead of overflowing, so the callers keep x <= kRescaleThreshold (exact softmax) or check it (fast softmax: pmax).
// (An |x| check instead of the clamp was measured and rejected: profiles/r02_attention_experiments.txt.)
__device__ __forceinline__ void exp2_pair(const float x0, const float x1, const bool poly, float& p0, float& p1) {
  if (poly) {
    const uint64_t magic2 = pack_f32x2(12582912.f, 12582912.f), nmagic2 = pack_f32x2(-12582912.f, -12582912.f);
    const uint64_t mone2 = pack_f32x2(-1.f, -1.f);
    const uint64_t c0 = pack_f32x2(0.9999280572f, 0.9999280572f), c1 = pack_f32x2(0.6932609677f, 0.6932609677f),
                   c2 = pack_f32x2(0.2426111251f, 0.2426111251f), c3 = pack_f32x2(0.0551716499f, 0.0551716499f);
    const uint64_t xp = pack_f32x2(fmaxf(x0, -126.f), fmaxf(x1, -126.f));
    const uint64_t t = fadd2(xp, magic2);
    const uint64_t fr = ffma2(fadd2(t, nmagic2), mone2, xp);
    uint64_t pp = ffma2(c3, fr, c2);
    pp = ffma2(pp, fr, c1);
    pp = ffma2(pp, fr, c0);
    float t0, t1;
    unpack_f32x2(t, t0, t1);
    unpack_f32x2(pp, p0, p1);
    p0 = __int_as_float(__float_as_int(p0) + (__float_as_int(t0) << 23));
    p1 = __int_as_float(__float_as_int(p1) + (__float_as_int(t1) << 23));
  } else {
    p0 = exp2_approx(x0);
    p1 = exp2_approx(x1);
  }
}

// Epilogue: kCols columns of O (TMEM, from o_tmem on) times inv_l, as bf16 to out[0, kCols) of a token-major row; the TMEM loads are
// warp-wide, the stores only for rows < S (row_valid).
template <int kCols>
__device__ __forceinline__ void store_o(const uint32_t o_tmem, const float inv_l, __nv_bfloat16* out, const bool row_valid) {
#pragma unroll
  for (int c = 0; c < kCols / 32; ++c) {
    uint32_t o[32];
    tmem_ld_32x32(o_tmem + c * 32, o);
    tmem_wait_ld();
    if (row_valid) {
      uint4* dst = reinterpret_cast<uint4*>(out + c * 32);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        uint4 w;
        w.x = pack_bf16x2(__uint_as_float(o[8 * e + 0]) * inv_l, __uint_as_float(o[8 * e + 1]) * inv_l);
        w.y = pack_bf16x2(__uint_as_float(o[8 * e + 2]) * inv_l, __uint_as_float(o[8 * e + 3]) * inv_l);
        w.z = pack_bf16x2(__uint_as_float(o[8 * e + 4]) * inv_l, __uint_as_float(o[8 * e + 5]) * inv_l);
        w.w = pack_bf16x2(__uint_as_float(o[8 * e + 6]) * inv_l, __uint_as_float(o[8 * e + 7]) * inv_l);
        dst[e] = w;
      }
    }
  }
}

// One 128-row query tile (qt) of one (batch b, head h): the whole CTA, from initialised mbarriers and an allocated TMEM block to
// the stores of O.  kFast selects the guarded softmax without per-chunk maxima (redo_smem: set when the tile must be recomputed exactly).
template <int DP, bool kFast>
__device__ __forceinline__ void attn_cta(const AttnOp& A, uint8_t* smem, const int qt, const int h, const int b, int* redo_smem) {
  using L = AttnSmem<DP>;
  const AttnBars<DP> B(smem);
  uint64_t *const q_full = B.q_full, *const k_full = B.k_full, *const v_full = B.v_full, *const k_empty = B.k_empty,
                 *const v_empty = B.v_empty, *const s_full = B.s_full, *const s_free = B.s_free, *const p_full = B.p_full,
                 *const pv_done = B.pv_done;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q0 = qt * kQT;
  const int n_kv = (A.S + kKT - 1) / kKT;
#ifdef TPDM_ATTN_TRACE
  const int ctr = !kFast ? -1 : (qt == 5 && h == 3 && b == 0) ? 0 : (qt == 7 && h == 20 && b == 1) ? 1 : -1;   // see g_cta_trace
  const bool trace_on = ctr == 0;
#endif
  const uint32_t tmem_base = *B.tmem_slot;

  if (warp < 4) {
  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer
    if (lane == 0) {
      mbar_arrive_expect_tx(q_full, L::kTile);
#pragma unroll
      for (int hh = 0; hh < DP / 64; ++hh) tma_load_4d(smem + L::kQOff + hh * (kQT * 128), &A.tmQ, q_full, hh * 64, h, q0, b);
      int stage = 0;
      uint32_t phase = 0;
      for (int j = 0; j < n_kv; ++j) {
        mbar_wait_backoff(&k_empty[stage], phase ^ 1);
        mbar_arrive_expect_tx(&k_full[stage], L::kTile);
#pragma unroll
        for (int hh = 0; hh < DP / 64; ++hh)
          tma_load_4d(smem + L::kKOff + stage * L::kTile + hh * (kKT * 128), &A.tmK, &k_full[stage], hh * 64, h, j * kKT, b);
        mbar_wait_backoff(&v_empty[stage], phase ^ 1);
        mbar_arrive_expect_tx(&v_full[stage], L::kTile);
#pragma unroll
        for (int hh = 0; hh < DP / 64; ++hh)
          tma_load_4d(smem + L::kVOff + stage * L::kTile + hh * (kKT * 128), &A.tmV, &v_full[stage], hh * 64, h, j * kKT, b);
        if (++stage == kKVStages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer: S(j) = Q K(j)^T
    constexpr uint32_t idesc_qk = make_idesc_bf16(kQT, kKT, false);
    const uint32_t q_base = smem_u32(smem + L::kQOff);
    mbar_wait(q_full, 0);
    for (int j = 0; j < n_kv; ++j) {
      const int stage = j % kKVStages;
      ATRACE(1, 4 * j);
      mbar_wait(&k_full[stage], (j / kKVStages) & 1);
      if (j >= 1) mbar_wait_backoff(s_free, (j - 1) & 1);  // softmax(j-1) holds S(j-1) in registers
      tc_fence_after();
      ATRACE(1, 4 * j + 1);
      {
        // converged warp, one elected lane per instruction (umma_ss_elect in common.cuh): no waterfall loop around the MMAs
        const uint32_t k_base = smem_u32(smem + L::kKOff + stage * L::kTile);
        const uint64_t qdesc0 = make_smem_desc_sw128(q_base, 16, 1024), kdesc0 = make_smem_desc_sw128(k_base, 16, 1024);
#pragma unroll
        for (int ks = 0; ks < DP / 16; ++ks) {
          const uint32_t off = ((ks / 4) * (kQT * 128) + (ks % 4) * 32) >> 4;   // the start-address field counts 16-byte units
          umma_ss_elect(tmem_base + L::kSCol, qdesc0 + off, kdesc0 + off, idesc_qk, ks != 0 ? 1u : 0u);
        }
        // ONE commit per tile: the K stage is handed back to the TMA warp by the softmax warp that observes s_full
        umma_commit_elect(s_full);
      }
      ATRACE(1, 4 * j + 2);
      __syncwarp();
    }
  } else if (warp == 3) {
    // ---------------------------------------------------------------- MMA issuer: O += P(j) V(j)
    // Two issuing warps: every tcgen05.mma costs its issuing thread >= 56 cycles (mma_issue_rate.cu); all hand-offs between
    // the two instruction streams go through mbarriers (s_free / p_full / pv_done), none relies on a common issue order.
    constexpr uint32_t idesc_pv = make_idesc_bf16(kQT, DP, true);
    for (int j = 0; j < n_kv; ++j) {
      const int stage = j % kKVStages;
      ATRACE(2, 4 * j);
      // P(j) arrives in two halves of 64 keys: the first four MMAs run under the last quarter of the tile's exponentials, so only
      // four are left when the tile ends and P (single-buffered) is free again before the next tile's first chunk lands
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        mbar_wait_backoff(&p_full[half], j & 1);
        if (half == 0) mbar_wait(&v_full[stage], (j / kKVStages) & 1);
        tc_fence_after();
        if (half == 0) ATRACE(2, 4 * j + 1);
        {
          const uint32_t v_base = smem_u32(smem + L::kVOff + stage * L::kTile);
          // B = V tile, MN-major: 16 keys per MMA = 16 rows of 128 B; 64-wide d-groups are kKT*128 B apart (LBO)
          const uint64_t vdesc0 = make_smem_desc_sw128(v_base, kKT * 128, 1024);
#pragma unroll
          for (int k4 = 0; k4 < kKT / 32; ++k4) {
            const int ks = half * (kKT / 32) + k4;
            umma_ts_elect(tmem_base + L::kOCol, tmem_base + L::kPCol + ks * 8, vdesc0 + ks * (2048 >> 4), idesc_pv, (j | ks) != 0 ? 1u : 0u);
          }
          if (half == 1) umma_commit_elect(pv_done);   // the V stage is released by the softmax warp that observes pv_done
        }
        __syncwarp();
      }
      ATRACE(2, 4 * j + 2);
      __syncwarp();
    }
  }
  } else if (kFast) {
    // ---------------------------------------------------------------- fast softmax: warps 4-7 keys [0,64), warps 8-11 keys [64,128)
    // The reference m_ref only has to keep exp2(s - m_ref) inside the fp32 / bf16 exponent range; it does not have to be the maximum.
    // It starts as the row maximum of the first key tile and is then guarded by the ROW SUM, which the loop computes anyway (see
    // `tile`).  What the guard cannot repair -- a score more than ~2^64 above everything the row has seen (l > 2^64, inf or NaN at the
    // next check; or an argument > 127 reaching the polynomial) -- sets this CTA's redo flag, and the CTA then runs its tile a second
    // time with the exact softmax (per-chunk maxima, the branch below) before it exits.
    __shared__ float xch[2][kQT];
    __shared__ int bump[2][kQT];   // see `tile`: total reference shift (float bits, >= 0) in force from the tiles of one parity on
    const int q = warp & 3, half = (warp - 4) >> 2;
    const uint32_t lane_off = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t s_tmem = tmem_base + lane_off + L::kSCol + half * 64;
    const uint32_t p_tmem = tmem_base + lane_off + L::kPCol + half * 32;
    const uint32_t o_tmem = tmem_base + lane_off + L::kOCol + half * (DP / 2);
    const int rowi = q * 32 + lane;
    const float scale = A.scale_log2;
    const uint64_t scale2 = pack_f32x2(scale, scale);
    constexpr float kHard = 1.8446744073709552e19f, kPolyMax = 127.f;
    uint64_t la = pack_f32x2(0.f, 0.f), lb = pack_f32x2(0.f, 0.f);   // this half's row sum as four partial sums
    float pmax = -INFINITY;   // largest argument that went through the polynomial
    bool hard = false;
    float applied = 0.f;   // total shift applied to this thread's reference
    if (half == 0) {
      bump[0][q * 32 + lane] = 0;
      bump[1][q * 32 + lane] = 0;
    }
    auto mask16 = [&](const int c, uint32_t (&v)[16], const int valid) {   // keys >= S of the tail tile
      if (valid < kKT) {
#pragma unroll
        for (int e = 0; e < 16; ++e)
          if (half * 64 + c * 16 + e >= valid) v[e] = 0xff800000u;
      }
    };
    // reference = row maximum of the first key tile (both halves, exchanged through shared memory once)
    mbar_wait(s_full, 0);
    tc_fence_after();
    float m_ref;
    {
      const int valid0 = A.S < kKT ? A.S : kKT;
      float mx = -INFINITY;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t v[16];
        tmem_ld_32x16(s_tmem + c * 16, v);
        tmem_wait_ld();
        mask16(c, v, valid0);
#pragma unroll
        for (int e = 0; e < 16; e += 2) mx = fmax3(mx, __uint_as_float(v[e]), __uint_as_float(v[e + 1]));
      }
      xch[half][rowi] = mx * scale;
      asm volatile("bar.sync 1, 256;" ::: "memory");
      m_ref = fmaxf(xch[0][rowi], xch[1][rowi]);
      asm volatile("bar.sync 1, 256;" ::: "memory");   // xch is reused for the row sums
    }
    CTRACE(3);
    uint64_t negm2 = pack_f32x2(-m_ref, -m_ref);
    // exponentials of one 16-column chunk, packed to bf16
    auto exp16 = [&](const uint32_t (&v)[16], uint32_t (&pk)[8]) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float x0, x1, p0, p1;
        unpack_f32x2(ffma2(pack_f32x2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1])), scale2, negm2), x0, x1);
        const bool poly = i % kPolyEvery == kPolyEvery - 1;
        if (poly) pmax = fmax3(pmax, x0, x1);
        exp2_pair(x0, x1, poly, p0, p1);
        if (i & 1) lb = fadd2(lb, pack_f32x2(p0, p1));
        else la = fadd2(la, pack_f32x2(p0, p1));
        pk[i] = pack_bf16x2(p0, p1);
      }
    };
    auto row_sum = [&]() {
      float a0, a1, b0, b1;
      unpack_f32x2(la, a0, a1);
      unpack_f32x2(lb, b0, b1);
      return (a0 + a1) + (b0 + b1);
    };
    auto tile = [&](const int j, auto masked_tag) {
      constexpr bool kMasked = decltype(masked_tag)::value;
      const int valid = A.S - j * kKT;
      // Both halves of a row must move their reference at the SAME tile, so the guard runs at CHECKPOINTS (every 4th tile, the same
      // tiles for every thread) through two shared-memory slots per row that hold a TOTAL shift (float bits, only ever raised by
      // atomicMax: no slot needs clearing, and the larger of two simultaneous proposals wins for both halves).  At checkpoint c
      // a thread applies the total it finds in slot c & 1 -- the proposals of checkpoint c - 1 -- and, if its own partial sum has
      // passed 2^24, proposes applied + floor(log2 l) into slot (c + 1) & 1.  All of this sits BEHIND the wait for s_full(j): that
      // wait is ordered after every softmax warp's s_free arrivals of the earlier tiles, so the proposals of the last checkpoint
      // are visible and nobody still reads the slot that is written now.  A proposal takes effect 4 tiles later and up to 8 tiles
      // after the sum started to grow: the 2^40 between the proposal threshold and the exact-pass threshold cover that.  (A vote
      // per tile between the two halves costs the whole gain of the second four warps.)
      STRACE(0);
      hard = hard || pmax > kPolyMax;
      mbar_wait(s_full, j & 1);
      tc_fence_after();
      if (warp == 4 && lane == 0) mbar_arrive(&k_empty[j % kKVStages]);   // Q K(j)^T has completed: the K stage is free
      STRACE(1);
      uint32_t va[16], vb[16], pk[8];
      tmem_ld_32x16(s_tmem, va);
      tmem_ld_32x16(s_tmem + 16, vb);
      if ((j & 3) == 3) {
        const int c = j >> 2;
        const float lsum = row_sum();
        const float total = __int_as_float(bump[c & 1][rowi]);
        const bool over = !(lsum <= 16777216.f);
        hard = hard || !(lsum <= kHard);
        if (__any_sync(0xffffffffu, over || total > applied)) {   // rare; whole warp, rows without a shift use alpha = 1
          const float e = total > applied ? total - applied : 0.f;
          if (over && lsum <= kHard)   // the sum as it will stand after the shift applied right below
            atomicMax(&bump[(c + 1) & 1][rowi],
                      __float_as_int(fmaxf(total, applied) + fmaxf(static_cast<float>((__float_as_int(lsum) >> 23) - 127) - e, 0.f)));
          const float m_new = m_ref + e;
          const float alpha = exp2_approx(m_ref - m_new);
          m_ref = m_new;
          applied = fmaxf(total, applied);
          negm2 = pack_f32x2(-m_ref, -m_ref);
          mbar_wait(pv_done, (j - 1) & 1);   // every P V issued so far has drained: O may be touched
          tc_fence_after();
#pragma unroll 1
          for (int cc = 0; cc < DP / 32; ++cc) {   // this half's DP / 2 columns of O
            uint32_t o[16];
            tmem_ld_32x16(o_tmem + cc * 16, o);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st_32x16(o_tmem + cc * 16, o);
          }
          const uint64_t alpha2 = pack_f32x2(alpha, alpha);
          la = fmul2(la, alpha2);
          lb = fmul2(lb, alpha2);
        }
      }
      tmem_wait_ld();
      STRACE(2);
      if (kMasked) {
        mask16(0, va, valid);
        mask16(1, vb, valid);
      }
      exp16(va, pk);
      if (j > 0) {  // P is single-buffered: P(j-1) V must be done before P(j) lands
        mbar_wait(pv_done, (j - 1) & 1);
        tc_fence_after();
        if (warp == 4 && lane == 0) mbar_arrive(&v_empty[(j - 1) % kKVStages]);   // ... and its V stage is free
      }
      tmem_st_32x8(p_tmem, pk);
      tmem_ld_32x16(s_tmem + 32, va);
      STRACE(3);
      exp16(vb, pk);
      tmem_st_32x8(p_tmem + 8, pk);
      tmem_ld_32x16(s_tmem + 48, vb);
      tmem_wait_ld();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_free);   // this warp's half of S(j) is in registers (8 arrivals complete the phase)
      STRACE(4);
      if (kMasked) {
        mask16(2, va, valid);
        mask16(3, vb, valid);
      }
      exp16(va, pk);
      tmem_st_32x8(p_tmem + 16, pk);
      exp16(vb, pk);
      tmem_st_32x8(p_tmem + 24, pk);
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[half]);   // keys [0,64) from warps 4-7, keys [64,128) from warps 8-11: 4 arrivals each
      STRACE(5);
    };
    for (int j = 0; j < n_kv - 1; ++j) tile(j, std::false_type{});
    tile(n_kv - 1, std::true_type{});
    CTRACE(4);
    const float lh = row_sum();
    if (!(lh <= kHard) || pmax > kPolyMax) hard = true;
    if (hard) *redo_smem = 1;
    xch[half][rowi] = lh;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    const float inv_l = 1.0f / (xch[0][rowi] + xch[1][rowi]);
    mbar_wait(pv_done, (n_kv - 1) & 1);
    tc_fence_after();
    const int row = q0 + rowi;
    store_o<DP / 2>(o_tmem, inv_l,
                    A.out + (static_cast<long long>(b) * A.S + row) * (static_cast<long long>(A.H) * DP) + h * DP + half * (DP / 2), row < A.S);
  } else if (warp < 8) {
    // ---------------------------------------------------------------- exact softmax (the redo pass): warps 4-7, one thread per row
    const int q = warp & 3;
    const uint32_t lane_off = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t s_tmem = tmem_base + lane_off + L::kSCol;
    const uint32_t p_tmem = tmem_base + lane_off + L::kPCol;
    const uint32_t o_tmem = tmem_base + lane_off + L::kOCol;
    const float scale = A.scale_log2;
    const uint64_t scale2 = pack_f32x2(scale, scale);
    float m_used = -INFINITY;            // reference max of the running sums (log2 domain); may lag the true max by 2^kRescaleThreshold
    uint64_t l2 = pack_f32x2(0.f, 0.f);  // row sum as two partial sums

    // p = exp2(s * scale - m_used) for one half (16 columns) of a 32-column chunk, packed to bf16; accumulates the row sum.
    // x <= kRescaleThreshold by construction of m_used, so the polynomial pairs need no check.
    auto exp_half = [&](const uint32_t (&v)[32], uint32_t (&pk)[16], uint64_t negm2, const int half) {
#pragma unroll
      for (int ii = 0; ii < 8; ++ii) {
        const int i = half * 8 + ii;
        float x0, x1, p0, p1;
        unpack_f32x2(ffma2(pack_f32x2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1])), scale2, negm2), x0, x1);
        exp2_pair(x0, x1, i % kPolyEvery == kPolyEvery - 1, p0, p1);
        l2 = fadd2(l2, pack_f32x2(p0, p1));
        pk[i] = pack_bf16x2(p0, p1);
      }
    };
    // rare path: multiply everything accumulated under the old reference by alpha = 2^(m_old - m_new)
    auto rescale_o = [&](float alpha) {
#pragma unroll 1
      for (int c = 0; c < DP / 16; ++c) {
        uint32_t o[16];
        tmem_ld_32x16(o_tmem + c * 16, o);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
        tmem_st_32x16(o_tmem + c * 16, o);
      }
    };
    auto rescale_p_chunk = [&](int c, float alpha) {
      uint32_t pk[16];
      tmem_ld_32x16(p_tmem + c * 16, pk);
      tmem_wait_ld();
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float lo = __uint_as_float(pk[i] << 16) * alpha, hi = __uint_as_float(pk[i] & 0xffff0000u) * alpha;
        pk[i] = pack_bf16x2(lo, hi);
      }
      tmem_st_32x16(p_tmem + c * 16, pk);
    };
    // keys >= S of the masked tail tile (warp-uniform branch) get s = -inf, i.e. p = 0
    auto mask_chunk = [&](const int c, uint32_t (&v)[32], const int valid) {
      if (valid < kKT) {
#pragma unroll
        for (int e = 0; e < kChunk; ++e)
          if (c * kChunk + e >= valid) v[e] = 0xff800000u;
      }
    };
    // scaled maximum of one chunk: four independent FMNMX3 chains
    auto chunk_max = [&](const uint32_t (&v)[32]) {
      float m0 = __uint_as_float(v[0]), m1 = __uint_as_float(v[8]), m2 = __uint_as_float(v[16]), m3 = __uint_as_float(v[24]);
#pragma unroll
      for (int e = 1; e < 7; e += 2) {
        m0 = fmax3(m0, __uint_as_float(v[e]), __uint_as_float(v[e + 1]));
        m1 = fmax3(m1, __uint_as_float(v[8 + e]), __uint_as_float(v[8 + e + 1]));
        m2 = fmax3(m2, __uint_as_float(v[16 + e]), __uint_as_float(v[16 + e + 1]));
        m3 = fmax3(m3, __uint_as_float(v[24 + e]), __uint_as_float(v[24 + e + 1]));
      }
      m0 = fmax3(m0, __uint_as_float(v[7]), m1);
      m2 = fmax3(m2, __uint_as_float(v[15]), m3);
      return fmax3(m0, fmax3(m2, __uint_as_float(v[23]), __uint_as_float(v[31])), m0) * scale;
    };

    for (int j = 0; j < n_kv; ++j) {
      const int valid = A.S - j * kKT;  // keys valid in this tile (>= 1)
      mbar_wait(s_full, j & 1);
      tc_fence_after();
      if (warp == 4 && lane == 0) mbar_arrive(&k_empty[j % kKVStages]);   // Q K(j)^T has completed: the K stage is free
      uint32_t va[32], vb[32];
      tmem_ld_32x32(s_tmem, va);
      // rare path, entered by the whole warp when any row's chunk maximum runs more than 2^kRescaleThreshold above its reference
      // (always for the very first chunk, m_used = -inf): move the reference, rescale O, l and the P chunks [0, c) of this tile.
      // Nothing of this tile has been handed to the MMA warp yet (hand-over happens after the maximum of its last chunk is known).
      auto raise_reference = [&](const int c, const float mc) {
        const bool need = mc > m_used + kRescaleThreshold;
        const float alpha = need ? exp2_approx(m_used - mc) : 1.f;   // 0 when nothing has been accumulated yet
        if (need) m_used = mc;
        if (j > 0) {
          // O holds P V of every earlier tile: all of them must have drained (P(j-1) V is the newest issued) before O is touched
          mbar_wait(pv_done, (j - 1) & 1);
          tc_fence_after();
          rescale_o(alpha);
        }
        if (c > 0) {
          tmem_wait_st();   // the chunks of this tile stored so far
#pragma unroll 1
          for (int cc = 0; cc < c; ++cc) rescale_p_chunk(cc, alpha);
        }
        l2 = fmul2(l2, pack_f32x2(alpha, alpha));
      };
      // Software pipeline over the four chunks: on entry `cur` (chunk c) is in registers with its reference settled and the load
      // of `nxt` (chunk c+1) is in flight.  The wait for nxt and its maximum sit between the two halves of cur's exponentials,
      // i.e. in the shadow of the MUFU; the load of chunk c+2 is issued into cur's registers once they are dead.
      // (Measured and rejected, profiles/r02_attention_experiments.txt: the whole S tile in 128 registers with setmaxnreg 56 / 200,
      // S released at 10 % of the tile and P chunk 0 held in registers instead of waiting for P(j-1) V -- no wait on data left, yet
      // 375 us against 339 us: every mbarrier / tcgen05.wait placed between the halves of a chunk drains the warp's MUFU queue.)
      tmem_wait_ld();
      tmem_ld_32x32(s_tmem + kChunk, vb);
      mask_chunk(0, va, valid);
      {
        const float mc = chunk_max(va);
        if (__any_sync(0xffffffffu, mc > m_used + kRescaleThreshold)) raise_reference(0, mc);
      }
      auto do_chunk = [&](const int c, uint32_t (&cur)[32], uint32_t (&nxt)[32]) {
        constexpr int kLast = kKT / kChunk - 1;
        uint32_t pk[16];
        const uint64_t negm2 = pack_f32x2(-m_used, -m_used);
        exp_half(cur, pk, negm2, 0);
        float mnext = -INFINITY;
        if (c < kLast) {
          tmem_wait_ld();   // chunk c+1
          if (c + 1 == kLast) {
            // all of S(j) is in registers: Q K^T of the next tile may overwrite it
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(s_free);
          }
          mask_chunk(c + 1, nxt, valid);
          mnext = chunk_max(nxt);
        }
        exp_half(cur, pk, negm2, 1);
        if (c == 0 && j > 0) {  // P is single-buffered: P(j-1) V must be done before P(j) lands
          mbar_wait(pv_done, (j - 1) & 1);
          tc_fence_after();
          if (warp == 4 && lane == 0) mbar_arrive(&v_empty[(j - 1) % kKVStages]);   // ... and its V stage is free
        }
        tmem_st_32x16(p_tmem + c * 16, pk);
        if (c + 2 <= kLast) tmem_ld_32x32(s_tmem + (c + 2) * kChunk, cur);
        if (c < kLast && __any_sync(0xffffffffu, mnext > m_used + kRescaleThreshold)) raise_reference(c + 1, mnext);
        // Hand-over to the MMA warp: keys [0,64) once the reference of the WHOLE tile is settled (the maximum of the last chunk is
        // known after chunk 2, so a raise never has to touch P that is already being multiplied), keys [64,128) at the end
        if (c >= kLast - 1) {
          tmem_wait_st();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&p_full[c == kLast ? 1 : 0]);
        }
      };
      do_chunk(0, va, vb);
      do_chunk(1, vb, va);
      do_chunk(2, va, vb);
      do_chunk(3, vb, va);
    }
    float l_lo, l_hi;
    unpack_f32x2(l2, l_lo, l_hi);
    mbar_wait(pv_done, (n_kv - 1) & 1);
    tc_fence_after();
    const int row = q0 + q * 32 + lane;
    store_o<DP>(o_tmem, 1.0f / (l_lo + l_hi), A.out + (static_cast<long long>(b) * A.S + row) * (static_cast<long long>(A.H) * DP) + h * DP,
                row < A.S);
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
}

// Fast kernel: one CTA per (query tile, head, batch entry).  A CTA whose softmax warps met scores the row-sum guard cannot keep in
// range (see attn_cta) runs its tile a second time with the exact softmax (per-chunk maxima) before it exits -- same TMEM block,
// mbarriers re-initialised.  On ordinary activations no CTA does.
template <int DP>
__global__ void __launch_bounds__(kFastThreads, DP == 64 ? 2 : 1) joint_attention_fast_kernel(const __grid_constant__ AttnOp A) {
  using L = AttnSmem<DP>;
  pdl_launch_dependents();
  uint8_t* smem = attn_smem_base();
  const AttnBars<DP> B(smem);
  __shared__ int redo_smem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef TPDM_ATTN_TRACE
  const int ctr = (blockIdx.x == 5 && blockIdx.y == 3 && blockIdx.z == 0) ? 0 : (blockIdx.x == 7 && blockIdx.y == 20 && blockIdx.z == 1) ? 1 : -1;
  if (ctr >= 0 && threadIdx.x == 128) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_cta_trace[ctr][7] = t;
  }
#endif
  CTRACE(0);
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&A.tmQ);
    tma_prefetch_desc(&A.tmK);
    tma_prefetch_desc(&A.tmV);
  }
  if (warp == 1 && lane == 0) B.init(false, 8);
  if (threadIdx.x == 0) redo_smem = 0;
  pdl_wait();
  CTRACE(1);
  const int cta_id = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
  const bool idle = (A.skip != nullptr && *A.skip != 0) || (A.bmask != nullptr && A.bmask[blockIdx.z % A.bslots] == 0);
  if (idle) {   // a speculative step after the trajectory's end, or an emptied queue slot
    if (A.redo != nullptr && threadIdx.x == 0) A.redo[cta_id] = 0;
    return;
  }
  if (warp == 2) {
    tmem_alloc<L::kTmemCols>(B.tmem_slot);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  CTRACE(2);
  attn_cta<DP, true>(A, smem, blockIdx.x, blockIdx.y, blockIdx.z, &redo_smem);   // ends with a CTA-wide barrier
  CTRACE(5);
  const int redo = redo_smem;
  if (redo != 0) {
    if (threadIdx.x == 0) atomicAdd(&g_redo_total, 1ull);
    if (warp == 1 && lane == 0) B.init(true, 4);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    attn_cta<DP, false>(A, smem, blockIdx.x, blockIdx.y, blockIdx.z, nullptr);
  }
  if (A.redo != nullptr && threadIdx.x == 0) A.redo[cta_id] = redo;   // diagnostic: tpdm_attention_redo_count
  if (warp == 2) tmem_dealloc<L::kTmemCols>(*B.tmem_slot);
#ifdef TPDM_ATTN_TRACE
  CTRACE(6);
  if (ctr >= 0 && threadIdx.x == 128) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_cta_trace[ctr][8] = t;
  }
#endif
}

// Redo flags, one int per CTA: slices of one device buffer handed out round-robin at attn_op_init time (an op keeps its slice; after
// a wrap two ops may share one, which is harmless on one stream: every launch rewrites every flag of its grid).
constexpr size_t kRedoCapacity = size_t(1) << 20;
int* redo_slice(size_t n) {
  static int* buf = nullptr;
  static size_t cursor = 0;
  if (n > kRedoCapacity) return nullptr;
  if (buf == nullptr && cudaMalloc(&buf, kRedoCapacity * sizeof(int)) != cudaSuccess) {
    buf = nullptr;
    (void)cudaGetLastError();
    return nullptr;
  }
  if (cursor + n > kRedoCapacity) cursor = 0;
  int* p = buf + cursor;
  cursor += n;
  return p;
}

const int* g_last_redo = nullptr;   // slice and grid size of the last launch (tpdm_attention_redo_count; nullptr: no slice)
int g_last_redo_n = 0;

template <int DP>
int attn_launch_impl(const AttnOp& op, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    TPDM_CUDA_OK(cudaFuncSetAttribute(joint_attention_fast_kernel<DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttnSmem<DP>::kTotal));
    attr_set = true;
  }
  dim3 grid(op.q_tiles, op.H, op.Bt);
  g_last_redo = op.redo;
  g_last_redo_n = op.q_tiles * op.H * op.Bt;
  const double q_rows = op.q_tiles * kQT < op.S ? op.q_tiles * kQT : op.S;
  prof_begin(1, 4.0 * op.Bt * op.H * q_rows * op.S * op.head_dim, stream);
  TPDM_CUDA_OK(launch_pdl(joint_attention_fast_kernel<DP>, grid, dim3(kFastThreads), AttnSmem<DP>::kTotal, stream, op));
  prof_end(stream);
  count_launch();
  TPDM_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace

int attn_op_init(AttnOp* op, const void* qkv, int Bt, int S, int H, int dp, int head_dim, void* out) {
  *op = AttnOp{};
  TPDM_CHECK(dp == 64 || dp == 128, TPDM_ERR_SHAPE, "attention: padded head dim %d must be 64 or 128", dp);
  TPDM_CHECK(head_dim > 0 && head_dim <= dp, TPDM_ERR_SHAPE, "attention: head_dim %d exceeds padded %d", head_dim, dp);
  TPDM_CHECK(S > 0 && H > 0 && Bt > 0, TPDM_ERR_SHAPE, "attention: empty problem");
  op->S = S;
  op->H = H;
  op->Bt = Bt;
  op->dp = dp;
  op->head_dim = head_dim;
  op->q_tiles = (S + kQT - 1) / kQT;
  op->scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(head_dim));
  op->out = reinterpret_cast<__nv_bfloat16*>(out);
  op->redo = redo_slice(static_cast<size_t>(op->q_tiles) * H * Bt);
  const uint64_t row = static_cast<uint64_t>(3) * H * dp;  // elements per token in the fused qkv buffer
  uint64_t dims[4] = {static_cast<uint64_t>(dp), static_cast<uint64_t>(H), static_cast<uint64_t>(S), static_cast<uint64_t>(Bt)};
  uint64_t strides[3] = {static_cast<uint64_t>(dp) * 2, row * 2, row * S * 2};
  uint32_t box[4] = {64, 1, kQT, 1};
  const __nv_bfloat16* base = reinterpret_cast<const __nv_bfloat16*>(qkv);
  TPDM_TRY(encode_tmap_bf16(&op->tmQ, base, 4, dims, strides, box));
  TPDM_TRY(encode_tmap_bf16(&op->tmK, base + static_cast<size_t>(H) * dp, 4, dims, strides, box));
  TPDM_TRY(encode_tmap_bf16(&op->tmV, base + static_cast<size_t>(2) * H * dp, 4, dims, strides, box));
  return 0;
}

long long attn_redo_total() {
  unsigned long long v = 0;
  if (cudaDeviceSynchronize() != cudaSuccess) return -2;
  if (cudaMemcpyFromSymbol(&v, g_redo_total, sizeof(v)) != cudaSuccess) return -2;
  return static_cast<long long>(v);
}

int attn_redo_count() {
  if (g_last_redo == nullptr) return -1;
  static int* host = nullptr;
  static int host_n = 0;
  if (host_n < g_last_redo_n) {
    free(host);
    host = static_cast<int*>(malloc(sizeof(int) * g_last_redo_n));
    host_n = g_last_redo_n;
  }
  if (cudaDeviceSynchronize() != cudaSuccess) return -2;
  if (cudaMemcpy(host, g_last_redo, sizeof(int) * g_last_redo_n, cudaMemcpyDeviceToHost) != cudaSuccess) return -2;
  int n = 0;
  for (int i = 0; i < g_last_redo_n; ++i) n += host[i] != 0;
  return n;
}

#ifdef TPDM_ATTN_TRACE
extern "C" int tpdm_attn_cta_trace_read(long long* host) {
  return cudaMemcpyFromSymbol(host, g_cta_trace, sizeof(long long) * 32) == cudaSuccess ? 0 : -1;
}
extern "C" int tpdm_attn_trace_read(long long* host, int n) {
  return cudaMemcpyFromSymbol(host, g_attn_trace, sizeof(long long) * (n < 3 * 2048 ? n : 3 * 2048)) == cudaSuccess ? 0 : -1;
}
#endif

int attn_launch(const AttnOp* op_in, cudaStream_t stream) {
  AttnOp op_copy = *op_in;
  op_copy.skip = skip_flag();
  op_copy.bmask = batch_mask();
  op_copy.bslots = batch_mask_slots();
  const AttnOp* op = &op_copy;
  return op->dp == 64 ? attn_launch_impl<64>(*op, stream) : attn_launch_impl<128>(*op, stream);
}

}  // namespace tpdm
