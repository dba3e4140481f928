// KD — merged-token self-attention for sm_100a: QKV projection (tcgen05 GEMM, linear.cu) -> flash
// attention (this file) -> output projection (tcgen05 GEMM).
//
// Reference: `self.attn1(merged_tokens)` at vidtome/patch.py:157-162 = diffusers Attention; the math is
// restated in the reference at utils/pnp_utils.py:47-95: softmax(q k^T * scale) v per head.
//
// Flash-attention kernel, one CTA per (128-row query tile, head, sample), 192 threads, two CTAs per SM
// (256 TMEM columns, <= 97 KB of shared memory each):
//   warp 0      TMA producer: Q tile once, then K/V tiles of BKV keys through a ring, from the head-major padded
//               q/k/v buffers written by the projection epilogue (a tile = one contiguous run of cache lines).
//   warp 1      MMA issuer: S_j = Q K_j^T (A, B from shared memory, K-major; only ceil(d/16) K steps) into one of
//               TWO score buffers, and O += P_j V_j with A = P_j read from TENSOR MEMORY and B = V_j read MN-major
//               from shared memory (no transposed copy of V).  S_{j+1} is issued before P_j is awaited, so the
//               softmax warps never wait for the QK round trip.  The warp stays converged (elect.sync) so that
//               descriptor arithmetic runs on the uniform datapath: with head_dim 40 the MMAs are tiny and the
//               issue rate of this warp matters.
//   warps 2..5  softmax: one query row per thread; the row's 64 scores are read from TMEM ONCE into registers
//               (row max -> lazy reference max -> P = exp2(s*scale*log2e - m) as fp16 written over the consumed
//               score columns, fp32 row sum).  The reference max moves only when exceeded by 2^8; then O is
//               rescaled in TMEM (after P_{j-1} V_{j-1} has retired).  Finally O / l -> fp16.
// For head_dim 40 the kernel is bound by the exponential (MUFU.EX2, 16/clk/SM), not by the tensor pipe.
// TMEM (256 columns): S0/P0 [0,BKV) | S1/P1 [BKV,2 BKV) | O [2 BKV, 2 BKV + 16*KSTEPS); BKV = 96 keys per tile when
// that fits (head_dim <= 64), else 64.
#include <stdlib.h>
#include <type_traits>

#include "gemm_sm100.cuh"
#include "gemm_sm100_2cta.cuh"

extern "C" int vtm_linear_f16(const void*, const void*, const void*, int32_t, int32_t, int32_t, void*, int64_t,
                              void*);
extern "C" int vtm_linear_residual_f16(const void*, const void*, const void*, const void*, int64_t, int32_t, int32_t,
                                       int32_t, void*, int64_t, void*);

namespace vtm {
namespace {

// ---------------------------------------------------------------------------------------------------------
// QKV projection epilogue: writes q, k, v HEAD-MAJOR with rows padded to DP = 64 or 128 halfs (128 / 256 bytes):
//   qkvh[which][b][head][l][0..DP)   (which = 0 q, 1 k, 2 v; columns >= head_dim are written as zeros)
// so that a K or V tile of consecutive keys of one head is one contiguous run of full cache lines.  Reading
// q/k/v in place from the [B*L, 3C] GEMM output instead makes every key row an 80-byte slice at a 1920-byte
// pitch: ncu showed 112 M L2 requests of ~1.2 sectors each for one attention call, and the K/V feed — not the
// softmax — bounded the kernel (profiles/r01_attention_ncu_summary.md).
struct HeadSplitEpi {
  static constexpr uint32_t SCRATCH_PER_WARP = gemm::STAGE_STORE_BYTES;
  __half* qkvh;
  int M, C, H, d, L, DP, nb; // M = nb*L rows, C = H*d
  int dread;                 // columns of a padded row that the flash kernel reads: 16 x (its k-step count) <= DP
  int which0, n_proj;        // this GEMM produces projections which0 .. which0 + n_proj - 1 of (q, k, v); N = n_proj * C
  float qscale;              // q is written as fp16(q * qscale) (1 = plain; softmax scale * log2 e for the embedded reference)
  int kones;                 // also write 1.0 into padding column d of K (embedded reference, flash_attn_kernel EMB)
  long long which_stride;    // B*H*L*DP
  int row0;                  // first of the warp's 32 rows
  int b0, l0;                // (sample, position) of row0 + lane / 8, this lane's first row in the store phase
  uint32_t scratch;

  __device__ __forceinline__ void set_scratch(uint32_t a) { scratch = a; }
  // This epilogue, not the MMAs, bounds the projection GEMMs (K = 320 / 640: 0.7 us of MMA per tile): the first version
  // executed ~940 instructions per warp and 64-column chunk — per-element scale selects, per-store range checks and
  // sample-wrap loops, two integer divisions per chunk (ncu: 8.6 M warp instructions for 1288 tiles, tensor pipe 26 %).
  // Everything that is the same for the warp's 32 rows or the chunk's 64 columns is now decided once, warp-uniformly,
  // and the common case (rows of one sample, all in range; chunk inside one projection) runs without per-store tests.
  int bw, lw;                // (sample, position) of row0, the first of the warp's 32 rows (warp-uniform)
  float inv_c, inv_d;        // 1 / C, 1 / d (set by the host) for the exact small-integer divisions below
  __device__ __forceinline__ void begin(int m_tile, int, int row_in_tile) {
    row0 = m_tile * gemm::BM + (row_in_tile & ~31);
    bw = row0 / L;
    lw = row0 - bw * L;
    // this lane's first row in the store phase: row0 + lane / 8 (up to 3 rows further: several samples when L < 4)
    b0 = bw;
    l0 = lw + ((row_in_tile & 31) >> 3);
    while (l0 >= L) { l0 -= L; ++b0; }
  }
  // exact x / y for 0 <= x < 2^22 (x + 0.5 keeps the product away from the integer boundary)
  static __device__ __forceinline__ int div_small(int x, float inv_y) {
    return static_cast<int>((static_cast<float>(x) + 0.5f) * inv_y);
  }
  __device__ __forceinline__ void tile(uint32_t taddr, int col0, int ncols) {
    const int sub = threadIdx.x & 7;
    const bool rows_plain = lw + 31 < L && bw < nb;      // the warp's 32 rows exist and lie in one sample
#pragma unroll 1
    for (int cb = 0; cb < ncols; cb += 64) {
      uint32_t r[64];
      tmem_ld_32x32b_x64(taddr + cb, r);
      tmem_ld_wait();
      uint32_t pk[32];
      const int cfirst = col0 + cb;
      // q columns are written as fp16(q * qscale): decided per chunk (C is a multiple of 64 for every SD width)
      if (which0 == 0 && qscale != 1.f && cfirst + 64 <= C) {
        const uint64_t s2 = f32x2_pack(qscale, qscale);
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          float a, b;
          f32x2_unpack(f32x2_mul(f32x2_pack(__uint_as_float(r[2 * e]), __uint_as_float(r[2 * e + 1])), s2), a, b);
          pk[e] = pack_f16x2(a, b);
        }
      } else if (which0 == 0 && qscale != 1.f && cfirst < C) {
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const float sc = cfirst + 2 * e < C ? qscale : 1.f;
          pk[e] = pack_f16x2(__uint_as_float(r[2 * e]) * sc, __uint_as_float(r[2 * e + 1]) * sc);
        }
      } else {
#pragma unroll
        for (int e = 0; e < 32; ++e) pk[e] = pack_f16x2(__uint_as_float(r[2 * e]), __uint_as_float(r[2 * e + 1]));
      }
      // this lane's 8 columns in the store phase: the same for all of its rows
      const int n = cfirst + sub * 8;                        // groups of 8 columns never straddle a head (d % 8 == 0)
      const bool n_ok = n < n_proj * C && sub * 8 < ncols - cb;   // BN = 160: 16-column second chunk
      const int which = div_small(n, inv_c), c = n - which * C;
      const int head = div_small(c, inv_d), e0 = c - head * d;
      // columns [d, dread) are read by the flash kernel's last k-step(s) (dread = 16 x its k-step count): zeros — except
      // column d of V (and of K with `kones`), which holds 1.0 so that the P V MMA also produces the softmax denominator
      // (flash_attn_kernel, ONES).  The padding beyond dread (up to DP) is never read by an MMA — TMA copies it into
      // shared memory and nothing else touches it — so it is NOT written.
      const bool pads = e0 + 8 == d && d < dread;
      const uint4 pad0 = (which + which0 == 2 || (kones && which + which0 == 1)) ? make_uint4(0x00003C00u, 0, 0, 0)
                                                                                 : make_uint4(0, 0, 0, 0);
      // dst(b, l) = base + (b H L + l) DP: stepped by 4 rows per store (plus (H - 1) L DP when crossing a sample)
      __half* dst = qkvh + which * which_stride + static_cast<long long>(head) * L * DP + e0 +
                    (static_cast<long long>(b0) * H * L + l0) * DP;
      const long long row_step = 4ll * DP;
      // staged through shared memory (gemm::warp_store_rows64): eight lanes write 64 consecutive columns of one row
      if (rows_plain) {
        if (!n_ok) dst = nullptr;
        gemm::warp_store_rows64(scratch, pk, [&](int, int, const uint4& v) {
          if (dst) {
            *reinterpret_cast<uint4*>(dst) = v;
            if (pads) {
              *reinterpret_cast<uint4*>(dst + 8) = pad0;
              for (int pe = d + 8; pe < dread; pe += 8) *reinterpret_cast<uint4*>(dst + 8 + (pe - d)) = make_uint4(0, 0, 0, 0);
            }
            dst += row_step;
          }
        });
      } else {
        const long long sample_step = static_cast<long long>(H - 1) * L * DP;
        int bb = b0, ll = l0;
        gemm::warp_store_rows64(scratch, pk, [&](int, int, const uint4& v) {
          if (bb < nb && n_ok) {
            *reinterpret_cast<uint4*>(dst) = v;
            if (pads) {
              *reinterpret_cast<uint4*>(dst + 8) = pad0;
              for (int pe = d + 8; pe < dread; pe += 8) *reinterpret_cast<uint4*>(dst + 8 + (pe - d)) = make_uint4(0, 0, 0, 0);
            }
          }
          ll += 4;                                              // next row of this lane: 4 further down
          dst += row_step;
          while (ll >= L) { ll -= L; ++bb; dst += sample_step; }
        });
      }
    }
  }
  __device__ __forceinline__ void end(int, int, int) {}
};

// Columns of a head-major padded row that the flash kernels read for head_dim d: 16 x the k-step count of the instantiation
// launch_fa_any picks (3, 4, 5, 6 or 8).
inline int fa_columns_read(int d) {
  const int ks = (d + 15) / 16;
  return 16 * (ks <= 3 ? 3 : (ks <= 6 ? ks : 8));
}
#ifndef VTM_HEAD_PROJ_PAIR_DEFAULT
#define VTM_HEAD_PROJ_PAIR_DEFAULT 0
#endif
// x [nb * L, K] -> projections which0 .. which0 + n_proj - 1 of (q, k, v), head-major padded, at `out`
// ([n_proj][nb][H][L][DP]); w [n_proj * C, K].
int launch_head_proj(const void* x, const void* w, __half* out, int nb, int L, int K, int C, int H, int DP, int which0,
                     int n_proj, float qscale, int kones, cudaStream_t stream) {
  int sms = 0;
  int rc = gemm::device_sms(&sms);
  if (rc) return rc;
  const int M = nb * L, N = n_proj * C;
  HeadSplitEpi epi;
  epi.qkvh = out; epi.M = M; epi.C = C; epi.H = H; epi.d = C / H; epi.L = L; epi.DP = DP;
  epi.dread = fa_columns_read(C / H);
  epi.which0 = which0; epi.n_proj = n_proj; epi.qscale = qscale; epi.kones = kones;
  epi.which_stride = static_cast<long long>(nb) * H * L * DP; epi.row0 = 0; epi.scratch = 0; epi.b0 = 0; epi.l0 = 0; epi.nb = nb;
  epi.bw = 0; epi.lw = 0; epi.inv_c = 1.f / static_cast<float>(C); epi.inv_d = 1.f / static_cast<float>(C / H);
  CUtensorMap ta, tb;
  rc = make_tmap_3d_f16(&ta, x, K, M, 1, K, static_cast<uint64_t>(M) * K, gemm::BK, gemm::BM);
  if (rc) return rc;
  gemm::Work wk;
  // Wide projections (q, k, v together: N = 3 C) with a short K are bound by the L2 -> SM operand traffic of 128 x 128 tiles
  // (160 KB per 10.5 MFLOP at K = 320: the ds1 projection ran at 393 TFLOP/s); the CTA-pair mainloop fetches every B byte
  // once per PAIR of CTAs and uses 256-wide tiles, i.e. half the bytes per FLOP.
  const int pair_env = gemm::pair_override();
  if (pair_env != 0 && (pair_env == 1 || VTM_HEAD_PROJ_PAIR_DEFAULT) && N >= 768 && M >= 2048) {
    rc = make_tmap_3d_f16(&tb, w, K, N, 1, K, static_cast<uint64_t>(N) * K, gemm::BK, 128);
    if (rc) return rc;
    gemm::plan_2cta(&wk, M, N, K, 1, sms, 16);
    wk.n_fastest = 1;
    return gemm::launch_2cta<HeadSplitEpi>(ta, tb, wk, epi, sms, stream);
  }
  if (N % 160 == 0 && N % 256 != 0 && N < 960) {     // N = 320 / 640 (q projection of the cross-attention): exact 160-wide tiles
    rc = make_tmap_3d_f16(&tb, w, K, N, 1, K, static_cast<uint64_t>(N) * K, gemm::BK, 160);
    if (rc) return rc;
    wk.plan(M, N, K, 1, 160, sms, 16, 1);
    wk.n_fastest = 1;
    return gemm::launch<160, HeadSplitEpi>(ta, tb, wk, epi, sms, stream);
  }
  rc = make_tmap_3d_f16(&tb, w, K, N, 1, K, static_cast<uint64_t>(N) * K, gemm::BK, 128);
  if (rc) return rc;
  wk.plan(M, N, K, 1, 128, sms, 16, 1);
  wk.n_fastest = 1;
  return gemm::launch<128, HeadSplitEpi>(ta, tb, wk, epi, sms, stream);
}

int launch_qkv_heads(const void* x, const void* w_qkv, __half* qkvh, int B, int L, int C, int H, int DP, float qscale,
                     int kones, cudaStream_t stream) {
  return launch_head_proj(x, w_qkv, qkvh, B, L, C, C, H, DP, 0, 3, qscale, kones, stream);
}

#ifndef VTM_FA2_STAGGER_NS
#define VTM_FA2_STAGGER_NS 300
#endif
// per-SM start counter of the two-CTAs-per-SM kernel (a scheduling hint only: its parity decides which CTA staggers)
__device__ unsigned int vtm_fa_sm_slot[256];

constexpr int BQ = 128;    // query rows per CTA (UMMA M)
#ifndef VTM_FA_PAIRS_DEFAULT
#define VTM_FA_PAIRS_DEFAULT 0
#endif
constexpr int FA_THREADS = 192;        // TMA warp, MMA warp, four softmax warps
constexpr int FA_PAIR_THREADS = 320;   // ... eight softmax warps (flash_attn_kernel HALVES = 2)
constexpr uint32_t FA_PAIR_XCH_BYTES = 2048;   // [quadrant 4][slot 2][half 2][lane 32] floats
constexpr float RESCALE_LOG2 = 8.f;   // move the reference max only when exceeded by 2^8

struct FaParams {
  int L, H, d, C;     // L = number of keys per (sample, head)
  int Lq;             // number of queries per sample (== L for self-attention)
  float scale_log2;   // softmax scale * log2(e)
  __half* o;          // [B*L, C]
  // Work decomposition (see launch_fa): units [0, n_full) are whole (query tile, head, sample) problems; each of
  // the remaining tiles is cut into `splits` key ranges whose un-normalised results go to part_o / part_ml and
  // are merged by fa_combine_kernel.
  int n_qtiles, n_full, splits;
  int qk_shared;      // PnP injection (utils/pnp_utils.py:57-68,87-91): q and k of sample 0 for every sample, v per sample
  float* part_o;      // [tile - n_full][splits][BQ][DV_N]  fp32, relative to the part's reference max
  float2* part_ml;    // [tile - n_full][splits][BQ]        (reference max * scale_log2, denominator)
};

template <int KSTEPS>
struct FaCfg {
  static constexpr int ATOMS = (KSTEPS + 3) / 4;              // 64-wide head_dim blocks
  static constexpr int DV_N = 16 * KSTEPS;                    // UMMA N of P*V (head_dim rounded up to 16)
  // keys per tile: the largest multiple of 32 whose two score buffers fit next to O in 256 TMEM columns
  static constexpr int BKV = (2 * 96 + DV_N) <= 256 ? 96 : 64;
  static constexpr int STAGES = ATOMS == 1 ? 3 : 2;           // K/V ring depth
  static constexpr int MIN_CTAS = 2;                          // co-resident CTAs per SM
  static constexpr uint32_t Q_BYTES = ATOMS * BQ * 128;       // Q tile: ATOMS x [128 rows x 128 B]
  static constexpr uint32_t KV_ATOM = BKV * 128;              // one 64-wide block of a K or V tile
  static constexpr uint32_t TILE_BYTES = ATOMS * KV_ATOM;
  static constexpr uint32_t STAGE_BYTES = 2 * TILE_BYTES;     // K + V
  static constexpr uint32_t O_COL = 2 * BKV;
  static constexpr uint32_t TMEM_COLS = 256;                  // 2 x 64 score columns + up to 128 O columns
  static constexpr size_t SMEM_BYTES = 1024 + Q_BYTES + static_cast<size_t>(STAGES) * STAGE_BYTES + 256;
};

// Row maximum of this thread's BKV = 32*NCH scores, held in registers (read from TMEM exactly once: TMEM read
// bandwidth is shared with the MMAs, and a second pass over S would double it).  Four independent chains.
template <int NCH, bool TAIL>
__device__ __forceinline__ float fa_row_max(const uint32_t (&r)[NCH][32], int n_valid) {
  float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
#pragma unroll
  for (int ch = 0; ch < NCH; ++ch) {
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      const int col = ch * 32 + i;
      if (!TAIL) {
        if (i & 4) m1 = fmax3(m1, __uint_as_float(r[ch][i]), __uint_as_float(r[ch][i + 1])),
                   m3 = fmax3(m3, __uint_as_float(r[ch][i + 2]), __uint_as_float(r[ch][i + 3]));
        else       m0 = fmax3(m0, __uint_as_float(r[ch][i]), __uint_as_float(r[ch][i + 1])),
                   m2 = fmax3(m2, __uint_as_float(r[ch][i + 2]), __uint_as_float(r[ch][i + 3]));
      } else {
        if (col < n_valid) m0 = fmaxf(m0, __uint_as_float(r[ch][i]));
        if (col + 1 < n_valid) m1 = fmaxf(m1, __uint_as_float(r[ch][i + 1]));
        if (col + 2 < n_valid) m2 = fmaxf(m2, __uint_as_float(r[ch][i + 2]));
        if (col + 3 < n_valid) m3 = fmaxf(m3, __uint_as_float(r[ch][i + 3]));
      }
    }
  }
  return fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
}
// P = exp2(s*c - mc) for 32 scores -> 16 packed fp16 pairs; accumulates the fp32 row sum.  For small head_dim the
// kernel is bound by MUFU.EX2 (16/clk/SM) and by issue slots about equally, so (i) x = s*c - mc is one packed FFMA2 per
// PAIR of scores, and (ii) VTM_FA_POLY_NUM of every VTM_FA_POLY_DEN pairs are evaluated on the FMA/ALU pipes with the
// packed cubic (ex2_poly3_x2: 10 issue slots per pair against 2 MUFU) while the others go to MUFU: the two pipes run
// side by side (tools/ubench/fma2_pipe.cu: 16 FFMA2 + 8 MUFU take 74 cycles, 8 MUFU alone 65).  Per score and SMSP:
// MUFU 8 (1 - phi) cycles, issue 2.5 + 4 phi slots — balanced near phi = 0.45.  Swept on B200 (tools/sweep_fa_poly.py,
// ms for qkv + flash + out at B=2, L=10241, 8 heads x 40): see profiles/r02_attention_poly_sweep.md.
#ifndef VTM_FA_POLY_NUM
#define VTM_FA_POLY_NUM 3
#endif
#ifndef VTM_FA_POLY_DEN
#define VTM_FA_POLY_DEN 16
#endif
// with the embedded reference (MODE 1 / 2: no FFMA in front of the exponential) the balance moves towards the FMA pipe:
// swept 3 .. 10 of 16, flat minimum at 5 - 7 (profiles/r02_attention_embed_sweep*.jsonl)
#ifndef VTM_FA_POLY_NUM_EMB
#define VTM_FA_POLY_NUM_EMB 6
#endif
// MODE 0: x = s * c - mc (scores in raw units);  MODE 1: x = s (the scores already ARE the exponents: scale folded into
// q and the reference embedded in the QK product, see the EMB path of flash_attn_kernel);  MODE 2: x = s - mc.
template <bool TAIL, bool SUM, int MODE = 0>
__device__ __forceinline__ void fa_exp32(const uint32_t (&r)[32], uint32_t (&pk)[16], float c, float mc, int col0,
                                         int n_valid, float& sum0, float& sum1) {
  const uint64_t c2 = f32x2_pack(c, c), nmc2 = f32x2_pack(-mc, -mc);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const uint64_t s2 = f32x2_pack(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
    const uint64_t x2 = MODE == 0 ? f32x2_fma(s2, c2, nmc2) : (MODE == 1 ? s2 : f32x2_add(s2, nmc2));
    float p0, p1;
    // pair i goes to the polynomial when the running count floor((i+1) NUM / DEN) steps: an even spread
    constexpr int NUM = MODE == 0 ? VTM_FA_POLY_NUM : VTM_FA_POLY_NUM_EMB;
    if (((i + 1) * NUM) / VTM_FA_POLY_DEN != (i * NUM) / VTM_FA_POLY_DEN) {
      ex2_poly3_x2(x2, p0, p1);
    } else {
      float x0, x1;
      f32x2_unpack(x2, x0, x1);
      p0 = ex2_approx(x0);
      p1 = ex2_approx(x1);
    }
    if (TAIL) {
      if (col0 + 2 * i >= n_valid) p0 = 0.f;
      if (col0 + 2 * i + 1 >= n_valid) p1 = 0.f;
    }
    if (SUM) {
      sum0 += p0;
      sum1 += p1;
    }
    pk[i] = pack_f16x2(p0, p1);
  }
}

// The same for N raw exponents held in a plain register array (pair kernel below): MODE 1 (x = s) or 2 (x = s - mc);
// PAIR0 = index of the first pair in the thread's tile share, so that the polynomial pairs stay evenly spread.
template <int N, int PAIR0, bool TAIL, int MODE>
__device__ __forceinline__ void fa_exp_n(const uint32_t* r, uint32_t* pk, float mc, int n_valid) {
  const uint64_t nmc2 = f32x2_pack(-mc, -mc);
#pragma unroll
  for (int i = 0; i < N / 2; ++i) {
    const uint64_t s2 = f32x2_pack(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
    const uint64_t x2 = MODE == 1 ? s2 : f32x2_add(s2, nmc2);
    float p0, p1;
    const int g = PAIR0 + i;
    if (((g + 1) * VTM_FA_POLY_NUM_EMB) / VTM_FA_POLY_DEN != (g * VTM_FA_POLY_NUM_EMB) / VTM_FA_POLY_DEN) {
      ex2_poly3_x2(x2, p0, p1);
    } else {
      float x0, x1;
      f32x2_unpack(x2, x0, x1);
      p0 = ex2_approx(x0);
      p1 = ex2_approx(x1);
    }
    if (TAIL) {
      if (2 * (PAIR0 + i) >= n_valid) p0 = 0.f;
      if (2 * (PAIR0 + i) + 1 >= n_valid) p1 = 0.f;
    }
    pk[i] = pack_f16x2(p0, p1);
  }
}

// ONES: head_dim % 16 == 8 (40, the SD1.5 full-resolution blocks): column d of the padded V rows holds 1.0 and lies
// inside the P V MMA's N, so O[:, d] accumulates the row sums of P — the denominator comes out of the tensor core,
// follows every rescale of O automatically and is the sum of exactly the fp16 P values the numerator uses; the
// softmax warps drop one FADD per score.  Measured effect on time: -0.6 % at L=10241, none at L=21300 (same-box
// A/B against -DVTM_FA_NO_ONES) — the row sums were not what limits the softmax warps.
// EMB (requires ONES, i.e. head_dim % 16 == 8 and a spare column in the padded rows): the softmax scale * log2 e is folded
// into q by the projection epilogue, column d of every K row holds 1.0 and column d of a Q row holds MINUS the reference
// maximum of that query row, so that the tensor core delivers s' = exponent - reference directly: the softmax warps issue
// MUFU.EX2 on the accumulators as loaded, without the FFMA (and the dependency level) per score.  A thread owns its row's
// reference: it rewrites the 2-byte column in shared memory (swizzled address) when the reference moves — after the one
// QK MMA that may still be reading the tile has completed (s_full of the next tile) — and keeps track of which reference
// each tile's scores embed (QK runs one tile ahead, so a new reference takes effect two tiles later).
// HALVES == 2 (requires EMB): EIGHT softmax warps per CTA, two per 32-row TMEM quadrant, each taking one half of the tile's
// keys of the same rows — four softmax warps per scheduler instead of two to cover the fixed-latency dependencies that
// dominate the stall samples (profiles/r02_attention_kernel_study.md section 6).  With the denominator coming out of the P V MMA
// (ONES) and the reference embedded in the scores (EMB) the only thing the two warps of a row share is the decision "the
// reference moves" — one bar.red.or over the 64 threads per tile in the steady state, plus an exchange of the two half-row
// maxima through shared memory on the rare tiles where it does.  Each half writes its P into the first half of ITS OWN score
// columns (so no warp overwrites scores the other has not read yet); the P V MMAs take their A operand from the two pieces.
template <int KSTEPS, bool ONES, bool EMB = false, int HALVES = 1>
__global__ void __launch_bounds__(HALVES == 2 ? FA_PAIR_THREADS : FA_THREADS, FaCfg<KSTEPS>::MIN_CTAS)
flash_attn_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                  const __grid_constant__ CUtensorMap tm_v, const FaParams p) {
  using C = FaCfg<KSTEPS>;
  constexpr int STAGES = C::STAGES;
  constexpr int BKV = C::BKV;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sQ = smem_base;
  const uint32_t sKV = sQ + C::Q_BYTES;
  const uint32_t bar_base = sKV + STAGES * C::STAGE_BYTES;
  // 8-byte slots: q_full | k_full[S] | v_full[S] | kv_empty[S] | s_full[2] | p_full[2] | o_ready[2] | tmem ptr
  const uint32_t q_full = bar_base;
  auto k_full = [&](int s) { return bar_base + 8u * (1 + s); };
  auto v_full = [&](int s) { return bar_base + 8u * (1 + STAGES + s); };
  auto kv_empty = [&](int s) { return bar_base + 8u * (1 + 2 * STAGES + s); };
  auto s_full = [&](int i) { return bar_base + 8u * (1 + 3 * STAGES + i); };
  auto p_full = [&](int i) { return bar_base + 8u * (3 + 3 * STAGES + i); };
  // o_ready[i] completes when P_j V_j (j & 1 == i) has retired.  Two barriers so that a softmax warp may skip the
  // wait when it has nothing to rescale: the MMA warp is never more than one tile ahead, so the barrier consulted
  // is at most one completion ahead of the one asked for and the parity test stays unambiguous.
  auto o_ready = [&](int i) { return bar_base + 8u * (5 + 3 * STAGES + i); };
  const uint32_t tmem_ptr_addr = bar_base + 8u * (7 + 3 * STAGES);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // unit -> (tile, key range).  Whole tiles first, then the split ones: the split units fill the last, partial wave.
  int tile = blockIdx.x, part = 0, nparts = 1;
  if (tile >= p.n_full) {
    const int v = tile - p.n_full;
    tile = p.n_full + v / p.splits;
    part = v % p.splits;
    nparts = p.splits;
  }
  const int q0 = (tile % p.n_qtiles) * BQ;
  const int h = (tile / p.n_qtiles) % p.H;
  const int b = tile / (p.n_qtiles * p.H);
  const int bqk = p.qk_shared ? 0 : b;
  const int nkv_all = (p.L + BKV - 1) / BKV;
  const int j_lo = static_cast<int>(static_cast<long long>(part) * nkv_all / nparts);
  const int nkv = static_cast<int>(static_cast<long long>(part + 1) * nkv_all / nparts) - j_lo;   // >= 1

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_q);
    tma_prefetch_desc(&tm_k);
    tma_prefetch_desc(&tm_v);
    mbar_init(q_full, 1);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(k_full(s), 1);
      mbar_init(v_full(s), 1);
      mbar_init(kv_empty(s), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(s_full(i), 1);
      mbar_init(p_full(i), 4 * HALVES);  // one arrival per softmax warp
    }
    mbar_init(o_ready(0), 1);
    mbar_init(o_ready(1), 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_addr, C::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_ptr_addr));
  const uint32_t tmem_o = tmem_base + C::O_COL;

  if (warp == 0) {
    // ===================== TMA producer (whole warp converged; one elected lane issues) =====================
    if (elect_one()) {
      mbar_arrive_expect_tx(q_full, C::Q_BYTES);
      for (int a = 0; a < C::ATOMS; ++a) tma_load_3d(sQ + a * (BQ * 128), &tm_q, q_full, a * 64, q0, bqk * p.H + h);
    }
    for (int j = 0; j < nkv; ++j) {
      const int s = j % STAGES;
      const uint32_t ph = (j / STAGES) & 1u;
      mbar_wait(kv_empty(s), ph ^ 1u);
      const uint32_t sk = sKV + s * C::STAGE_BYTES;
      const uint32_t sv = sk + C::TILE_BYTES;
      if (elect_one()) {
        mbar_arrive_expect_tx(k_full(s), C::TILE_BYTES);
        for (int a = 0; a < C::ATOMS; ++a) tma_load_3d(sk + a * C::KV_ATOM, &tm_k, k_full(s), a * 64, (j_lo + j) * BKV, bqk * p.H + h);
        mbar_arrive_expect_tx(v_full(s), C::TILE_BYTES);
        for (int a = 0; a < C::ATOMS; ++a) tma_load_3d(sv + a * C::KV_ATOM, &tm_v, v_full(s), a * 64, (j_lo + j) * BKV, b * p.H + h);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp converged; one elected lane issues) =====================
    constexpr uint32_t idesc_qk = umma_idesc_f16(BQ, BKV);
    constexpr uint32_t idesc_pv = umma_idesc_f16_bmn(BQ, C::DV_N);
    auto issue_qk = [&](int j) {
      const int s = j % STAGES;
      mbar_wait(k_full(s), (j / STAGES) & 1u);
      tc_fence_after();
      const uint32_t sk = sKV + s * C::STAGE_BYTES;
      const uint32_t d_tmem = tmem_base + (j & 1) * BKV;
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < KSTEPS; ++ks) {
          const uint64_t adesc = umma_desc_sw128_kmajor(sQ + (ks >> 2) * (BQ * 128)) + 2u * (ks & 3);
          const uint64_t bdesc = umma_desc_sw128_kmajor(sk + (ks >> 2) * C::KV_ATOM) + 2u * (ks & 3);
          umma_f16(d_tmem, adesc, bdesc, idesc_qk, ks != 0 ? 1u : 0u);
        }
        umma_commit(s_full(j & 1));
      }
      __syncwarp();
    };
    mbar_wait(q_full, 0);
    issue_qk(0);
    for (int j = 0; j < nkv; ++j) {
      // Scores of the next tile first: they land in the other buffer, whose previous content (P_{j-1}) was
      // consumed by the P_{j-1} V_{j-1} MMAs issued before (tcgen05.mma executes in issue order).
      if (j + 1 < nkv) issue_qk(j + 1);
      const int s = j % STAGES;
      mbar_wait(v_full(s), (j / STAGES) & 1u);
      mbar_wait(p_full(j & 1), (j >> 1) & 1u);   // P_j in TMEM, O rescaled if needed
      tc_fence_after();
      const uint32_t sv = sKV + s * C::STAGE_BYTES + C::TILE_BYTES;
      const uint32_t p_tmem = tmem_base + (j & 1) * BKV;
      if (elect_one()) {
        const uint64_t vdesc = umma_desc_sw128_mnmajor(sv, C::KV_ATOM);
        // P of keys 16 t .. 16 t + 15: 8 packed columns; HALVES == 2: the second half of the keys starts at column BKV / 2
        auto p_col = [&](int t) -> uint32_t {
          return HALVES == 2 && t >= BKV / 32 ? static_cast<uint32_t>(BKV / 2 + 8 * (t - BKV / 32)) : 8u * t;
        };
        if (j == 0) {
#pragma unroll
          for (int t = 0; t < BKV / 16; ++t)
            umma_f16_ts(tmem_o, p_tmem + p_col(t), vdesc + 128u * t, idesc_pv, t != 0 ? 1u : 0u);
        } else {
#pragma unroll
          for (int t = 0; t < BKV / 16; ++t)
            umma_f16_ts(tmem_o, p_tmem + p_col(t), vdesc + 128u * t /* 16 rows x 128 B */, idesc_pv, 1u);
        }
        umma_commit(kv_empty(s));
        umma_commit(o_ready(j & 1));
      }
      __syncwarp();
    }
  } else {
    // ===================== softmax / correction / epilogue =====================
    const int quad = warp & 3;                                   // TMEM lane quadrant this warp may access
    const int half = HALVES == 2 ? ((warp - 2) >> 2) : 0;        // which half of a tile's keys (HALVES == 2)
    const int row = q0 + quad * 32 + lane;
    const uint32_t lane_field = static_cast<uint32_t>(quad * 32) << 16;
    const float c = p.scale_log2;
    float m_ref = -INFINITY;   // reference max (raw score units) used by the exponentials
    float l_run = 0.f;         // running denominator (same reference)
#if VTM_FA2_STAGGER_NS > 0
    // Two co-resident CTAs run the same instruction stream on equally long tiles and tend to stay in lock-step (both in
    // their MUFU phase, then both out of it).  Every second CTA that starts on an SM delays its softmax warps once by
    // about a third of a tile time so that the phases interleave.
    {
      uint32_t smid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      uint32_t slot = 0;
      if (lane == 0 && warp == 2) slot = atomicAdd(&vtm_fa_sm_slot[smid & 255u], 1u);
      // one draw per CTA, broadcast to the softmax warps through the (already initialised) tmem pointer slot + 4
      if (lane == 0 && warp == 2) asm volatile("st.shared.u32 [%0], %1;" ::"r"(tmem_ptr_addr + 4), "r"(slot) : "memory");
      bar_sync_named(2, 128 * HALVES);
      asm volatile("ld.shared.u32 %0, [%1];" : "=r"(slot) : "r"(tmem_ptr_addr + 4));
      if (slot & 1u) __nanosleep(VTM_FA2_STAGGER_NS);
    }
#endif
    if constexpr (EMB && HALVES == 2) {
      constexpr int HK = BKV / 2;          // keys per half tile
      constexpr int NB = HK - 32;          // scores beyond the first 32 of the half: 16 (BKV = 96) or 0 (BKV = 64)
      static_assert(NB == 0 || NB == 16, "half tiles of 32 or 48 keys");
      const int rit = quad * 32 + lane;
      const int dcol = p.d & 63, datom = p.d >> 6;
      const uint32_t q_ref_addr = sQ + datom * (BQ * 128) + rit * 128 + ((((2 * dcol) >> 4) ^ (rit & 7)) << 4) + ((2 * dcol) & 15);
      const uint32_t xch = bar_base + 256u + static_cast<uint32_t>(quad) * 512u;   // [slot][half][lane] floats of this quadrant
      const uint32_t bar_id = 3u + quad;   // named barrier of the two warps of this quadrant (0: __syncthreads, 2: stagger)
      float m_O = -INFINITY, e_tile0 = 0.f, e_tile1 = 0.f, e_q = 0.f;   // as in the HALVES == 1 loop; identical in both halves
      for (int j = 0; j < nkv; ++j) {
        mbar_wait(s_full(j & 1), (j >> 1) & 1u);
        tc_fence_after();
        const uint32_t s_addr = tmem_base + lane_field + (j & 1) * BKV + half * HK;   // my scores; my P goes to their first half
        const int n_tile = p.L - (j_lo + j) * BKV;
        const bool tail = n_tile < BKV;
        const int n_valid = n_tile - half * HK;        // existing keys of my half (<= 0: none)
        uint32_t ra[32], rb[NB > 0 ? NB : 1];
        const float e = (j & 1) ? e_tile1 : e_tile0;
        float mx;
        bool slow;
        if (j == 0 || tail) {
          tmem_ld_32x32b_x32(s_addr, ra);
          if constexpr (NB > 0) tmem_ld_32x32b_x16(s_addr + 32, rb);
          tmem_ld_wait();
          float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            if (!tail || i < n_valid) m0 = fmaxf(m0, __uint_as_float(ra[i]));
            if (!tail || i + 1 < n_valid) m1 = fmaxf(m1, __uint_as_float(ra[i + 1]));
          }
          if constexpr (NB > 0) {
#pragma unroll
            for (int i = 0; i < NB; i += 2) {
              if (!tail || 32 + i < n_valid) m0 = fmaxf(m0, __uint_as_float(rb[i]));
              if (!tail || 33 + i < n_valid) m1 = fmaxf(m1, __uint_as_float(rb[i + 1]));
            }
          }
          mx = fmaxf(m0, m1);
          slow = true;
        } else {
          // speculative, as in the HALVES == 1 loop: the scores are the exponents while the tile embeds O's reference and
          // no score of the ROW (both halves) exceeds it by more than 2^8
          float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
          tmem_ld_32x32b_x32(s_addr, ra);
          tmem_ld_wait();
          if constexpr (NB > 0) tmem_ld_32x32b_x16(s_addr + 32, rb);
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            m0 = fmax3(m0, __uint_as_float(ra[i]), __uint_as_float(ra[i + 1]));
            m1 = fmax3(m1, __uint_as_float(ra[i + 2]), __uint_as_float(ra[i + 3]));
            m2 = fmax3(m2, __uint_as_float(ra[i + 4]), __uint_as_float(ra[i + 5]));
            m3 = fmax3(m3, __uint_as_float(ra[i + 6]), __uint_as_float(ra[i + 7]));
          }
          {
            uint32_t pk[16];
            fa_exp_n<32, 0, false, 1>(ra, pk, 0.f, n_valid);
            tmem_st_32x32b_x16(s_addr, pk);
          }
          if constexpr (NB > 0) {
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < NB; i += 8) {
              m0 = fmax3(m0, __uint_as_float(rb[i]), __uint_as_float(rb[i + 1]));
              m1 = fmax3(m1, __uint_as_float(rb[i + 2]), __uint_as_float(rb[i + 3]));
              m2 = fmax3(m2, __uint_as_float(rb[i + 4]), __uint_as_float(rb[i + 5]));
              m3 = fmax3(m3, __uint_as_float(rb[i + 6]), __uint_as_float(rb[i + 7]));
            }
            uint32_t pk8[NB / 2];
            fa_exp_n<NB, 16, false, 1>(rb, pk8, 0.f, n_valid);
            tmem_st_32x32b_x8(s_addr + 16, pk8);
          }
          mx = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
          slow = bar_red_or(bar_id, 64, !(e == m_O && mx <= RESCALE_LOG2));   // over both warps of the quadrant
        }
        float alpha = 1.f;
        if (slow) {
          // the row maximum over both halves (slots alternate with j: a warp may enter its next slow tile before the other
          // has read this one's value; two tiles later the barrier of the tile in between orders them)
          const uint32_t slot = xch + static_cast<uint32_t>(j & 1) * 256u;
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(slot + (half * 32 + lane) * 4), "f"(mx) : "memory");
          bar_sync_named(bar_id, 64);
          float other;
          asm volatile("ld.shared.f32 %0, [%1];" : "=f"(other) : "r"(slot + ((half ^ 1) * 32 + lane) * 4) : "memory");
          mx = fmaxf(mx, other);
          const float abs_max = e + mx;
          float r_new = m_O;
          if (!(abs_max - m_O <= RESCALE_LOG2)) r_new = __half2float(__float2half_ru(abs_max));
          if (r_new != m_O) {
            alpha = ex2_approx(m_O - r_new);
            m_O = r_new;
          }
          const float delta = m_O - e;
          uint32_t pk[16];
          if (tail) fa_exp_n<32, 0, true, 2>(ra, pk, delta, n_valid);
          else fa_exp_n<32, 0, false, 2>(ra, pk, delta, n_valid);
          tmem_st_32x32b_x16(s_addr, pk);
          if constexpr (NB > 0) {
            uint32_t pk8[NB / 2];
            if (tail) fa_exp_n<NB, 16, true, 2>(rb, pk8, delta, n_valid);
            else fa_exp_n<NB, 16, false, 2>(rb, pk8, delta, n_valid);
            tmem_st_32x32b_x8(s_addr + 16, pk8);
          }
        }
        if (j > 0 && __any_sync(0xffffffffu, alpha != 1.f)) {     // same alpha in both halves: they share the O chunks
          mbar_wait(o_ready((j - 1) & 1), ((j - 1) >> 1) & 1u);
          tc_fence_after();
#pragma unroll
          for (int cb = 0; cb < C::DV_N; cb += 16) {
            if (((cb >> 4) & 1) != half) continue;
            uint32_t ro[16];
            tmem_ld_32x32b_x16(tmem_o + lane_field + cb, ro);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) ro[i] = __float_as_uint(__uint_as_float(ro[i]) * alpha);
            tmem_st_32x32b_x16(tmem_o + lane_field + cb, ro);
          }
        }
        if (j + 2 < nkv && __any_sync(0xffffffffu, e_q != m_O)) {
          if (half == 0) {                 // half 0 owns the row's reference column in shared memory
            mbar_wait(s_full((j + 1) & 1), ((j + 1) >> 1) & 1u);
            if (e_q != m_O) {
              const unsigned short neg = __half_as_ushort(__float2half_rn(-m_O));
              asm volatile("st.shared.u16 [%0], %1;" ::"r"(q_ref_addr), "h"(neg) : "memory");
            }
            fence_proxy_async_smem();
          }
          e_q = m_O;
        }
        if (j & 1) e_tile1 = e_q; else e_tile0 = e_q;
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full(j & 1));
      }
      m_ref = m_O;
    } else
    if constexpr (EMB) {
      static_assert(ONES, "the embedded reference uses the spare column of head_dim % 16 == 8");
      static_assert(HALVES == 1, "HALVES == 2 has its own loop above");
      const int rit = quad * 32 + lane;                                  // row in the Q tile
      const int dcol = p.d & 63, datom = p.d >> 6;                       // column d inside its 64-wide block
      const uint32_t q_ref_addr = sQ + datom * (BQ * 128) + rit * 128 + ((((2 * dcol) >> 4) ^ (rit & 7)) << 4) + ((2 * dcol) & 15);
      float m_O = -INFINITY;           // reference of O and of every P accumulated so far (log2 units, fp16-exact)
      float e_tile0 = 0.f, e_tile1 = 0.f;   // reference embedded in the scores of tile j (j even / odd)
      float e_q = 0.f;                 // reference currently in shared memory (embedded from tile j + 2 on)
      float dummy0 = 0.f, dummy1 = 0.f;
      // One key tile.  PLAIN = first tile of the unit (no reference yet) or its last one (possibly masked columns): row
      // maximum first, then the exponentials.  The steady-state tiles in between are instantiated separately so that their
      // loop body holds nothing but the speculative path and ONE warp-uniform branch around everything rare (reference
      // moved: recompute P, rescale O, republish the reference) — the instruction-fetch stalls after the taken branches of
      // the single-loop version were 7 % of the softmax warps' samples (profiles/r02_attention_kernel_study.md section 7).
      constexpr int NCH = BKV / 32;
      uint32_t r[NCH][32];             // the row's raw scores of the tile in flight (kept for the rare recomputation)
      float mx;
      // speculative path of a steady-state tile: the scores are the exponents as long as the tile embeds O's reference and
      // stays below 2^8.  Returns (warp-uniform) whether anything rare is due: reference moved, or a reference to publish.
      auto tile_fast = [&](const int j) -> bool {
        mbar_wait(s_full(j & 1), (j >> 1) & 1u);
        tc_fence_after();
        const uint32_t s_addr = tmem_base + lane_field + (j & 1) * BKV;
        const float e = (j & 1) ? e_tile1 : e_tile0;
        float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
        tmem_ld_32x32b_x32(s_addr, r[0]);
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) {
          tmem_ld_wait();
          if (ch + 1 < NCH) tmem_ld_32x32b_x32(s_addr + 32 * (ch + 1), r[ch + 1]);
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            m0 = fmax3(m0, __uint_as_float(r[ch][i]), __uint_as_float(r[ch][i + 1]));
            m1 = fmax3(m1, __uint_as_float(r[ch][i + 2]), __uint_as_float(r[ch][i + 3]));
            m2 = fmax3(m2, __uint_as_float(r[ch][i + 4]), __uint_as_float(r[ch][i + 5]));
            m3 = fmax3(m3, __uint_as_float(r[ch][i + 6]), __uint_as_float(r[ch][i + 7]));
          }
          uint32_t pk[16];
          fa_exp32<false, false, 1>(r[ch], pk, 0.f, 0.f, 32 * ch, 0, dummy0, dummy1);
          tmem_st_32x32b_x16(s_addr + 16 * ch, pk);
        }
        mx = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
        return __any_sync(0xffffffffu, !(e == m_O && mx <= RESCALE_LOG2) || e_q != m_O);
      };
      // first / last tile of the unit (no reference yet / possibly masked columns): all scores first, then their maximum
      auto tile_plain = [&](const int j) {
        mbar_wait(s_full(j & 1), (j >> 1) & 1u);
        tc_fence_after();
        const uint32_t s_addr = tmem_base + lane_field + (j & 1) * BKV;
        const int n_valid = p.L - (j_lo + j) * BKV;
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) tmem_ld_32x32b_x32(s_addr + 32 * ch, r[ch]);
        tmem_ld_wait();
        mx = n_valid < BKV ? fa_row_max<NCH, true>(r, n_valid) : fa_row_max<NCH, false>(r, n_valid);
      };
      // the rare work of a tile whose scores (r) and row maximum (mx) are in registers: settle the reference, recompute P
      // with it, rescale O, republish the reference for the tiles whose QK has not been issued yet
      auto tile_rare = [&](const int j) {
        const uint32_t s_addr = tmem_base + lane_field + (j & 1) * BKV;
        const int n_valid = p.L - (j_lo + j) * BKV;
        const bool tail = n_valid < BKV;
        const float e = (j & 1) ? e_tile1 : e_tile0;
        float alpha = 1.f;
        // keep O's reference unless the row maximum exceeds it by more than 2^8, then move it to the maximum (rounded UP
        // to fp16 so that it can be embedded exactly)
        const float abs_max = e + mx;
        float r_new = m_O;
        if (!(abs_max - m_O <= RESCALE_LOG2)) r_new = __half2float(__float2half_ru(abs_max));   // also the first tile (m_O = -inf)
        if (r_new != m_O) {
          alpha = ex2_approx(m_O - r_new);       // 0 on the first tile
          m_O = r_new;
        }
        const float delta = m_O - e;              // exponent = s' - delta
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) {
          uint32_t pk[16];
          if (tail) fa_exp32<true, false, 2>(r[ch], pk, 0.f, delta, 32 * ch, n_valid, dummy0, dummy1);
          else fa_exp32<false, false, 2>(r[ch], pk, 0.f, delta, 32 * ch, n_valid, dummy0, dummy1);
          tmem_st_32x32b_x16(s_addr + 16 * ch, pk);
        }
        if (j > 0 && __any_sync(0xffffffffu, alpha != 1.f)) {
          mbar_wait(o_ready((j - 1) & 1), ((j - 1) >> 1) & 1u);
          tc_fence_after();
#pragma unroll
          for (int cb = 0; cb < C::DV_N; cb += 16) {
            uint32_t ro[16];
            tmem_ld_32x32b_x16(tmem_o + lane_field + cb, ro);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) ro[i] = __float_as_uint(__uint_as_float(ro[i]) * alpha);
            tmem_st_32x32b_x16(tmem_o + lane_field + cb, ro);
          }
        }
        if (j + 2 < nkv && __any_sync(0xffffffffu, e_q != m_O)) {
          // QK of tile j + 1 (issued with the old column) may still be reading this Q tile: wait for its commit
          mbar_wait(s_full((j + 1) & 1), ((j + 1) >> 1) & 1u);
          if (e_q != m_O) {
            const unsigned short neg = __half_as_ushort(__float2half_rn(-m_O));
            asm volatile("st.shared.u16 [%0], %1;" ::"r"(q_ref_addr), "h"(neg) : "memory");
            e_q = m_O;
          }
          fence_proxy_async_smem();    // generic-proxy store -> visible to the tensor core's (async proxy) operand reads
        }
      };
      auto tile_done = [&](const int j) {
        if (j & 1) e_tile1 = e_q; else e_tile0 = e_q;     // what tile j + 2 will embed
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full(j & 1));
      };
      // The steady-state tiles run in a loop that holds nothing but the speculative path: a tile with rare work BREAKS out
      // of it, so that the rare code lies behind the loop instead of being jumped over once per tile (the softmax warps lost
      // 7 % of their samples to instruction fetch after taken branches, profiles/r02_attention_kernel_study.md section 7).
      tile_plain(0);
      tile_rare(0);
      tile_done(0);
      for (int j = 1; j + 1 < nkv;) {
        bool rare = false;
        for (; j + 1 < nkv; ++j) {
          rare = tile_fast(j);
          if (rare) break;
          tile_done(j);
        }
        if (!rare) break;
        tile_rare(j);
        tile_done(j);
        ++j;
      }
      if (nkv > 1) {
        tile_plain(nkv - 1);
        tile_rare(nkv - 1);
        tile_done(nkv - 1);
      }
      m_ref = m_O;      // log2 units already (see the partial-result store below)
    } else {
    // same structure as the EMB loop above: plain first / last tile, steady-state tiles in a loop that a tile with rare
    // work (reference moved) breaks out of
    constexpr int NCH = BKV / 32;
    uint32_t r[NCH][32];   // the row's scores, read from TMEM exactly once
    float alpha = 1.f, sum0 = 0.f, sum1 = 0.f;
    // ---- speculative path: the reference max moves only when exceeded by 2^RESCALE_LOG2, which is rare after the first
    //      tiles.  So the exponentials start chunk by chunk with the CURRENT reference while the row maximum is accumulated
    //      alongside (independent instruction streams; each TMEM load overlaps the previous chunk's MUFU work).  P stays
    //      <= 2^8 whenever the speculation holds.  Returns (warp-uniform) whether some row's reference moved.
    auto tile_fast = [&](const int j) -> bool {
      mbar_wait(s_full(j & 1), (j >> 1) & 1u);
      tc_fence_after();
      const uint32_t s_addr = tmem_base + lane_field + (j & 1) * BKV;
      alpha = 1.f; sum0 = 0.f; sum1 = 0.f;
      const float mc0 = m_ref * c;
      float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
      tmem_ld_32x32b_x32(s_addr, r[0]);
#pragma unroll
      for (int ch = 0; ch < NCH; ++ch) {
        tmem_ld_wait();
        if (ch + 1 < NCH) tmem_ld_32x32b_x32(s_addr + 32 * (ch + 1), r[ch + 1]);
#pragma unroll
        for (int i = 0; i < 32; i += 8) {   // FMNMX3: two scores per instruction, four independent chains
          m0 = fmax3(m0, __uint_as_float(r[ch][i]), __uint_as_float(r[ch][i + 1]));
          m1 = fmax3(m1, __uint_as_float(r[ch][i + 2]), __uint_as_float(r[ch][i + 3]));
          m2 = fmax3(m2, __uint_as_float(r[ch][i + 4]), __uint_as_float(r[ch][i + 5]));
          m3 = fmax3(m3, __uint_as_float(r[ch][i + 6]), __uint_as_float(r[ch][i + 7]));
        }
        uint32_t pk[16];
        fa_exp32<false, !ONES>(r[ch], pk, c, mc0, 32 * ch, 0, sum0, sum1);
        tmem_st_32x32b_x16(s_addr + 16 * ch, pk);
      }
      const float mx = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
      const bool moved = (mx - m_ref) * c > RESCALE_LOG2;
      if (moved) {
        alpha = ex2_approx((m_ref - mx) * c);
        m_ref = mx;
      }
      return __any_sync(0xffffffffu, moved);
    };
    // ---- plain path (first tile: no reference yet; last tile: masked columns): max first, then the reference
    auto tile_plain = [&](const int j) {
      mbar_wait(s_full(j & 1), (j >> 1) & 1u);
      tc_fence_after();
      const uint32_t s_addr = tmem_base + lane_field + (j & 1) * BKV;
      const int n_valid = p.L - (j_lo + j) * BKV;  // keys of this tile that exist
      alpha = 1.f;
#pragma unroll
      for (int ch = 0; ch < NCH; ++ch) tmem_ld_32x32b_x32(s_addr + 32 * ch, r[ch]);
      tmem_ld_wait();
      const float mx = n_valid < BKV ? fa_row_max<NCH, true>(r, n_valid) : fa_row_max<NCH, false>(r, n_valid);
      if ((mx - m_ref) * c > RESCALE_LOG2) {
        alpha = ex2_approx((m_ref - mx) * c);     // 0 on the first tile (m_ref = -inf)
        m_ref = mx;
      }
    };
    // ---- P from the kept scores with the settled reference; O rescaled where a reference moved (only after
    //      P_{j-1} V_{j-1} has retired)
    auto tile_rare = [&](const int j) {
      const uint32_t s_addr = tmem_base + lane_field + (j & 1) * BKV;
      const int n_valid = p.L - (j_lo + j) * BKV;
      const bool tail = n_valid < BKV;
      const float mc = m_ref * c;
      sum0 = 0.f;
      sum1 = 0.f;
#pragma unroll
      for (int ch = 0; ch < NCH; ++ch) {
        uint32_t pk[16];
        if (tail) fa_exp32<true, !ONES>(r[ch], pk, c, mc, 32 * ch, n_valid, sum0, sum1);
        else fa_exp32<false, !ONES>(r[ch], pk, c, mc, 32 * ch, n_valid, sum0, sum1);
        tmem_st_32x32b_x16(s_addr + 16 * ch, pk);
      }
      if (j > 0 && __any_sync(0xffffffffu, alpha != 1.f)) {
        mbar_wait(o_ready((j - 1) & 1), ((j - 1) >> 1) & 1u);
        tc_fence_after();
#pragma unroll
        for (int cb = 0; cb < C::DV_N; cb += 16) {
          uint32_t ro[16];
          tmem_ld_32x32b_x16(tmem_o + lane_field + cb, ro);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) ro[i] = __float_as_uint(__uint_as_float(ro[i]) * alpha);
          tmem_st_32x32b_x16(tmem_o + lane_field + cb, ro);
        }
      }
    };
    auto tile_done = [&](const int j) {
      if (!ONES) l_run = l_run * alpha + (sum0 + sum1);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full(j & 1));
    };
    tile_plain(0);
    tile_rare(0);
    tile_done(0);
    for (int j = 1; j + 1 < nkv;) {
      bool rare = false;
      for (; j + 1 < nkv; ++j) {
        rare = tile_fast(j);
        if (rare) break;
        tile_done(j);
      }
      if (!rare) break;
      tile_rare(j);
      tile_done(j);
      ++j;
    }
    if (nkv > 1) {
      tile_plain(nkv - 1);
      tile_rare(nkv - 1);
      tile_done(nkv - 1);
    }
    }
    mbar_wait(o_ready((nkv - 1) & 1), ((nkv - 1) >> 1) & 1u);
    tc_fence_after();
    if (ONES) {   // the denominator is column d of O
      uint32_t r[16];
      tmem_ld_32x32b_x16(tmem_o + lane_field + (p.d & ~15), r);
      tmem_ld_wait();
      l_run = __uint_as_float((p.d & 15) ? r[8] : r[0]);   // column d: d % 16 is 8, or 0 when a k-step was added for it
    }
    if (nparts == 1) {
      // ---- epilogue: O / l -> fp16 -> o[b, row, h*d : h*d + d]
      const float inv = 1.f / l_run;
      __half* orow = p.o + (static_cast<size_t>(b) * p.Lq + row) * p.C + h * p.d;
#pragma unroll
      for (int cb = 0; cb < C::DV_N; cb += 16) {
        if (HALVES == 2 && ((cb >> 4) & 1) != half) continue;     // the two warps of a row share the output chunks
        uint32_t r[16];
        tmem_ld_32x32b_x16(tmem_o + lane_field + cb, r);
        tmem_ld_wait();
        if (row < p.Lq) {
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            if (cb + g * 8 < p.d) {  // d % 8 == 0
              uint4 v;
              uint32_t* pv = reinterpret_cast<uint32_t*>(&v);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const __half2 hh = __floats2half2_rn(__uint_as_float(r[g * 8 + 2 * e]) * inv,
                                                     __uint_as_float(r[g * 8 + 2 * e + 1]) * inv);
                pv[e] = *reinterpret_cast<const uint32_t*>(&hh);
              }
              *reinterpret_cast<uint4*>(orow + cb + g * 8) = v;
            }
          }
        }
      }
    } else {
      // ---- split tile: un-normalised O, reference max and denominator of this key range
      const size_t prow = (static_cast<size_t>(tile - p.n_full) * nparts + part) * BQ + quad * 32 + lane;
      if (half == 0) p.part_ml[prow] = make_float2(EMB ? m_ref : m_ref * c, l_run);
      float* po = p.part_o + prow * C::DV_N;
#pragma unroll
      for (int cb = 0; cb < C::DV_N; cb += 16) {
        if (HALVES == 2 && ((cb >> 4) & 1) != half) continue;
        uint32_t r[16];
        tmem_ld_32x32b_x16(tmem_o + lane_field + cb, r);
        tmem_ld_wait();
#pragma unroll
        for (int g = 0; g < 4; ++g)
          *reinterpret_cast<uint4*>(po + cb + 4 * g) = make_uint4(r[4 * g], r[4 * g + 1], r[4 * g + 2], r[4 * g + 3]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// Merge the key-range partials of the split tiles: with M = max_p m_p and w_p = 2^(m_p - M),
//   o = sum_p w_p O_p / sum_p w_p l_p.   One thread per (row, 8 output columns).
__global__ void fa_combine_kernel(const FaParams p, int dv_n, int n_split_tiles) {
  const int groups = p.d / 8;
  const long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (t >= static_cast<long long>(n_split_tiles) * BQ * groups) return;
  const int g = static_cast<int>(t % groups);
  const int r = static_cast<int>((t / groups) % BQ);
  const int st = static_cast<int>(t / (static_cast<long long>(groups) * BQ));
  const int tile = p.n_full + st;
  const int row = (tile % p.n_qtiles) * BQ + r;
  if (row >= p.Lq) return;
  const int h = (tile / p.n_qtiles) % p.H;
  const int b = tile / (p.n_qtiles * p.H);
  const size_t prow0 = static_cast<size_t>(st) * p.splits * BQ + r;
  float M = -INFINITY;
  for (int s = 0; s < p.splits; ++s) M = fmaxf(M, p.part_ml[prow0 + static_cast<size_t>(s) * BQ].x);
  float l = 0.f, acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int s = 0; s < p.splits; ++s) {
    const size_t prow = prow0 + static_cast<size_t>(s) * BQ;
    const float2 ml = p.part_ml[prow];
    const float w = exp2f(ml.x - M);
    l = fmaf(w, ml.y, l);
    const float4* po = reinterpret_cast<const float4*>(p.part_o + prow * dv_n + g * 8);
    const float4 a0 = po[0], a1 = po[1];
    acc[0] = fmaf(w, a0.x, acc[0]); acc[1] = fmaf(w, a0.y, acc[1]);
    acc[2] = fmaf(w, a0.z, acc[2]); acc[3] = fmaf(w, a0.w, acc[3]);
    acc[4] = fmaf(w, a1.x, acc[4]); acc[5] = fmaf(w, a1.y, acc[5]);
    acc[6] = fmaf(w, a1.z, acc[6]); acc[7] = fmaf(w, a1.w, acc[7]);
  }
  const float inv = 1.f / l;
  uint4 v;
  uint32_t* pv = reinterpret_cast<uint32_t*>(&v);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const __half2 hh = __floats2half2_rn(acc[2 * e] * inv, acc[2 * e + 1] * inv);
    pv[e] = *reinterpret_cast<const uint32_t*>(&hh);
  }
  *reinterpret_cast<uint4*>(p.o + (static_cast<size_t>(b) * p.Lq + row) * p.C + h * p.d + g * 8) = v;
}

}  // namespace
}  // namespace vtm
#include "attention_groups.cuh"
namespace vtm {
namespace {

// Upper bound on split units (remainder tiles x splits); sizes the partial buffers in the workspace.
constexpr int FA_MAX_SPLIT_UNITS = 320;
constexpr int FA_MAX_SPLITS = 8;
constexpr size_t FA_PART_BYTES = static_cast<size_t>(FA_MAX_SPLIT_UNITS) * BQ * (128 * sizeof(float) + sizeof(float2));

// Which flash kernel: the two-CTAs-per-SM kernel above by default; VTM_FA_GROUPS=1 selects the grouped one
// (attention_groups.cuh: one CTA per SM, G softmax groups), which measured 4-7 % slower at the SD shapes
// (profiles/r02_attention_kernel_study.md).  Read once per process; immutable afterwards.
bool fa_use_groups() {
  static const int v = [] {
    const char* e = getenv("VTM_FA_GROUPS");
    return (e && e[0] == '1') ? 1 : 0;
  }();
  return v != 0;
}
// VTM_FA_PAIRS=0 keeps four softmax warps per CTA on the embedded-reference path (flash_attn_kernel HALVES = 1) for A/B runs.
bool fa_use_pairs() {
  static const int v = [] {
    const char* e = getenv("VTM_FA_PAIRS");
    return e ? (e[0] == '1' ? 1 : 0) : VTM_FA_PAIRS_DEFAULT;
  }();
  return v != 0;
}
int fa_forced_splits() {
  static const int v = [] {
    const char* e = getenv("VTM_FA_SPLITS");   // tuning override (tools/sweep_fa_splits.py)
    return e ? atoi(e) : 0;
  }();
  return v;
}

template <int KSTEPS, bool ONES>
int launch_fa_impl(const void* qh, const void* kh, const void* vh, __half* o, void* part_ws, int B, int Lq, int L, int C,
                   int H, int d, float scale, int qk_shared, int emb, cudaStream_t stream) {
  using Cf = FaCfg<KSTEPS>;
  using Cg = FaGCfg<KSTEPS>;
  const bool groups = fa_use_groups();
  const int bkv = groups ? Cg::BKV : Cf::BKV;
  CUtensorMap tq, tk, tv;
  const int DP = Cf::ATOMS * 64;                       // padded head_dim of the head-major q/k/v buffers
  const uint64_t BH = static_cast<uint64_t>(B) * H;
  int rc = make_tmap_3d_f16(&tq, qh, DP, Lq, BH, DP, static_cast<uint64_t>(Lq) * DP, 64, BQ);
  if (rc) return rc;
  rc = make_tmap_3d_f16(&tk, kh, DP, L, BH, DP, static_cast<uint64_t>(L) * DP, 64, bkv);
  if (rc) return rc;
  rc = make_tmap_3d_f16(&tv, vh, DP, L, BH, DP, static_cast<uint64_t>(L) * DP, 64, bkv);
  if (rc) return rc;
  int sms = 0, per_sm = 1;
  rc = gemm::device_sms(&sms);
  if (rc) return rc;
  // once per instantiation and device: shared-memory opt-in and occupancy (immutable afterwards)
  static int occ_tab[64];
  int dev = 0;
  rc = cuda_rc(cudaGetDevice(&dev));
  if (rc) return rc;
  int occ = (dev >= 0 && dev < 64) ? occ_tab[dev] : 0;
  if (occ == 0) {
    rc = cuda_rc(cudaFuncSetAttribute(flash_attn_kernel<KSTEPS, ONES>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(Cf::SMEM_BYTES)));
    if (rc) return rc;
    rc = cuda_rc(cudaFuncSetAttribute(flash_attn_groups_kernel<KSTEPS, ONES>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(Cg::SMEM_BYTES)));
    if (rc) return rc;
    if (ONES) {
      rc = cuda_rc(cudaFuncSetAttribute(flash_attn_kernel<KSTEPS, ONES, ONES>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(Cf::SMEM_BYTES)));
      if (rc) return rc;
    }
    if constexpr (ONES && KSTEPS == 3) {
      rc = cuda_rc(cudaFuncSetAttribute(flash_attn_kernel<KSTEPS, true, true, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(Cf::SMEM_BYTES + FA_PAIR_XCH_BYTES)));
      if (rc) return rc;
    }
    rc = cuda_rc(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, flash_attn_kernel<KSTEPS, ONES>, FA_THREADS,
                                                               Cf::SMEM_BYTES));
    if (rc) return rc;
    if (occ < 1) occ = 1;
    if (dev >= 0 && dev < 64) occ_tab[dev] = occ;
  }
  per_sm = groups ? 1 : (occ > 0 ? occ : 1);
  const int slots = sms * per_sm;

  FaParams p;
  p.L = L; p.Lq = Lq; p.H = H; p.d = d; p.C = C;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.o = o;
  p.qk_shared = qk_shared;
  p.n_qtiles = (Lq + BQ - 1) / BQ;
  // Every tile costs the same, so the grid runs in waves of `slots` CTAs and the last, partial wave leaves most of
  // the GPU idle for a whole tile time.  The tiles of that wave are cut into `splits` key ranges instead (chosen to
  // minimise the time of the remainder, ceil(R * S / slots) / S tile times) and merged by fa_combine_kernel.
  const long long tiles = static_cast<long long>(p.n_qtiles) * H * B;
  const int nkv = (L + bkv - 1) / bkv;
  const int rem = static_cast<int>(tiles % slots);
  int splits = 1;
  if (rem > 0) {
    // Time of the remainder in tile times.  The kernel is bound by per-SM throughput, so what counts is the
    // number of units the busiest SM gets, not CTA slots: sub-waves over `sms` x (1 / S + fixed cost of a unit,
    // about four key tiles).  Split only for a clear gain (the merge is one more launch).
    const double fixed = 4.0 / nkv;
    double best_t = 0.9;
    for (int sp = 2; sp <= FA_MAX_SPLITS && sp * 4 <= nkv && rem * sp <= FA_MAX_SPLIT_UNITS; ++sp) {
      const double t = static_cast<double>((static_cast<long long>(rem) * sp + sms - 1) / sms) * (1.0 / sp + fixed);
      if (t < best_t - 1e-9) { best_t = t; splits = sp; }
    }
  }
  if (const int sp = fa_forced_splits()) {
    if (sp >= 1 && sp <= FA_MAX_SPLITS && sp <= nkv && static_cast<long long>(rem) * sp <= FA_MAX_SPLIT_UNITS)
      splits = rem > 0 ? sp : 1;
  }
  p.splits = splits;
  p.n_full = static_cast<int>(splits > 1 ? tiles - rem : tiles);
  p.part_ml = static_cast<float2*>(part_ws);
  p.part_o = reinterpret_cast<float*>(static_cast<char*>(part_ws) +
                                      static_cast<size_t>(FA_MAX_SPLIT_UNITS) * BQ * sizeof(float2));
  const long long units = p.n_full + (tiles - p.n_full) * splits;
  bool launched = false;
  if constexpr (ONES && KSTEPS == 3) {
    if (!groups && emb && fa_use_pairs()) {
      flash_attn_kernel<KSTEPS, true, true, 2>
          <<<static_cast<unsigned>(units), FA_PAIR_THREADS, Cf::SMEM_BYTES + FA_PAIR_XCH_BYTES, stream>>>(tq, tk, tv, p);
      launched = true;
    }
  }
  if (launched) {
  } else if (groups)
    flash_attn_groups_kernel<KSTEPS, ONES><<<static_cast<unsigned>(units), Cg::THREADS, Cg::SMEM_BYTES, stream>>>(tq, tk, tv, p);
  else if (ONES && emb)
    flash_attn_kernel<KSTEPS, ONES, ONES><<<static_cast<unsigned>(units), FA_THREADS, Cf::SMEM_BYTES, stream>>>(tq, tk, tv, p);
  else
    flash_attn_kernel<KSTEPS, ONES><<<static_cast<unsigned>(units), FA_THREADS, Cf::SMEM_BYTES, stream>>>(tq, tk, tv, p);
  rc = launch_rc();
  if (rc || splits == 1) return rc;
  const long long work = static_cast<long long>(rem) * BQ * (d / 8);
  fa_combine_kernel<<<static_cast<unsigned>((work + 255) / 256), 256, 0, stream>>>(p, Cf::DV_N, rem);
  return launch_rc();
}

template <int KSTEPS>
int launch_fa(const void* qh, const void* kh, const void* vh, __half* o, void* part_ws, int B, int Lq, int L, int C, int H,
              int d, float scale, int qk_shared, int ones, int emb, cudaStream_t stream) {
#if !defined(VTM_FA_NO_ONES)   // A/B switch: keep the denominator in the softmax warps
  if (ones)
    return launch_fa_impl<KSTEPS, true>(qh, kh, vh, o, part_ws, B, Lq, L, C, H, d, scale, qk_shared, emb, stream);
#endif
  return launch_fa_impl<KSTEPS, false>(qh, kh, vh, o, part_ws, B, Lq, L, C, H, d, scale, qk_shared, 0, stream);
}

// The embedded-reference path (flash_attn_kernel EMB) is used when the head dimension leaves a spare column
// (head_dim % 16 == 8: the SD1.5 full-resolution blocks) and the 2-CTAs-per-SM kernel runs; VTM_FA_EMBED=0 switches
// it off (A/B measurements).  Read once per process.
// A spare column for the ones / reference trick exists when head_dim % 16 == 8 (inside the last k-step).  Buying one with an
// extra k-step when head_dim % 16 == 0 and the padded row is wider (48 -> 4 steps, 80 -> 6) was measured and is NOT taken:
// head_dim 80, L = 2561: 0.1159 ms with the extra step against 0.1127 ms without (profiles/r02_attention_embed_sweep3.jsonl).
int fa_ksteps_with_spare(int d, bool* spare) {
  *spare = d % 16 == 8;
  return (d + 15) / 16;
}
bool fa_use_embed(int d) {
  static const int v = [] {
    const char* e = getenv("VTM_FA_EMBED");
    return (e && e[0] == '0') ? 0 : 1;
  }();
#if defined(VTM_FA_NO_ONES)
  return false;
#endif
  bool spare = false;
  fa_ksteps_with_spare(d, &spare);
  return v != 0 && spare && !fa_use_groups();
}

int launch_fa_any(const void* qh, const void* kh, const void* vh, __half* o, void* part_ws, int B, int Lq, int L, int C,
                  int H, int d, float scale, int qk_shared, int emb, cudaStream_t stream) {
  bool spare = false;
  const int ks = fa_ksteps_with_spare(d, &spare);
  const int ones = spare ? 1 : 0;
  switch (ks) {
    case 1: case 2: case 3: return launch_fa<3>(qh, kh, vh, o, part_ws, B, Lq, L, C, H, d, scale, qk_shared, ones, emb, stream);
    case 4: return launch_fa<4>(qh, kh, vh, o, part_ws, B, Lq, L, C, H, d, scale, qk_shared, ones, emb, stream);
    case 5: return launch_fa<5>(qh, kh, vh, o, part_ws, B, Lq, L, C, H, d, scale, qk_shared, ones, emb, stream);
    case 6: return launch_fa<6>(qh, kh, vh, o, part_ws, B, Lq, L, C, H, d, scale, qk_shared, ones, emb, stream);
    default: return launch_fa<8>(qh, kh, vh, o, part_ws, B, Lq, L, C, H, d, scale, qk_shared, ones, emb, stream);
  }
}

}  // namespace
}  // namespace vtm

extern "C" size_t vtm_attention_workspace_bytes(int32_t B, int32_t L, int32_t C, int32_t heads) {
  (void)heads;
  if (B <= 0 || L <= 0 || C <= 0) return 0;
  if (heads <= 0 || C % heads != 0) return 0;
  const int d = C / heads;
  const size_t DP = d <= 64 ? 64 : 128;
  // q/k/v head-major [3][B][H][L][DP] + o [B*L, C], fp16; then the key-range partials of the split tiles
  return (static_cast<size_t>(3) * B * heads * L * DP + static_cast<size_t>(B) * L * C) * 2 + vtm::FA_PART_BYTES + 256;
}

extern "C" int vtm_attention_ex(const void* x_dev, const void* w_qkv_dev, const void* w_o_dev, const void* b_o_dev,
                                int32_t B, int32_t L, int32_t C, int32_t heads, float scale, int32_t flags, void* y_dev,
                                void* ws_dev, size_t ws_bytes, void* stream_) {
  using namespace vtm;
  if (!x_dev || !w_qkv_dev || !w_o_dev || !y_dev || !ws_dev) return VTM_E_NULL;
  if (B <= 0 || L <= 0 || C <= 0 || heads <= 0 || C % heads != 0) return VTM_E_SHAPE;
  const int d = C / heads;
  if (d % 8 != 0 || C % 8 != 0) return VTM_E_SHAPE;
  if (d > 128 || (flags & ~1) != 0) return VTM_E_UNSUPPORTED;
  if (ws_bytes < vtm_attention_workspace_bytes(B, L, C, heads)) return VTM_E_WS;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int DP = d <= 64 ? 64 : 128;
  __half* qkv = static_cast<__half*>(ws_dev);
  __half* o = qkv + static_cast<size_t>(3) * B * heads * L * DP;
  const int M = B * L;
  void* part_ws = reinterpret_cast<void*>(
      (reinterpret_cast<uintptr_t>(o + static_cast<size_t>(M) * C) + 255u) & ~static_cast<uintptr_t>(255u));
  const int emb = fa_use_embed(d) ? 1 : 0;
  int rc = launch_qkv_heads(x_dev, w_qkv_dev, qkv, B, L, C, heads, DP, emb ? scale * 1.4426950408889634f : 1.f, emb, stream);
  if (rc) return rc;
  const __half* kh = qkv + static_cast<size_t>(B) * heads * L * DP;
  const __half* vh = kh + static_cast<size_t>(B) * heads * L * DP;
  rc = launch_fa_any(qkv, kh, vh, o, part_ws, B, L, L, C, heads, d, scale, flags & 1, emb, stream);
  if (rc) return rc;
  return vtm_linear_f16(o, w_o_dev, b_o_dev, M, C, C, y_dev, C, stream_);
}

extern "C" int vtm_attention(const void* x_dev, const void* w_qkv_dev, const void* w_o_dev, const void* b_o_dev,
                             int32_t B, int32_t L, int32_t C, int32_t heads, float scale, void* y_dev,
                             void* ws_dev, size_t ws_bytes, void* stream_) {
  return vtm_attention_ex(x_dev, w_qkv_dev, w_o_dev, b_o_dev, B, L, C, heads, scale, 0, y_dev, ws_dev, ws_bytes, stream_);
}

// ------------------------------------------------------------------------------------------------------------------
// Cross-attention of the patched block (vidtome/patch.py:171-185: `self.attn2(norm2(h), encoder_hidden_states=ctx)` and
// the residual add) — diffusers Attention with K/V from the text context.
extern "C" size_t vtm_cross_attention_workspace_bytes(int32_t B, int32_t Lq, int32_t Lk, int32_t C, int32_t heads) {
  if (B <= 0 || Lq <= 0 || Lk <= 0 || C <= 0 || heads <= 0 || C % heads != 0) return 0;
  const int d = C / heads;
  const size_t DP = d <= 64 ? 64 : 128;
  return (static_cast<size_t>(B) * heads * (static_cast<size_t>(Lq) + 2 * static_cast<size_t>(Lk)) * DP +
          static_cast<size_t>(B) * Lq * C) * 2 + vtm::FA_PART_BYTES + 512;
}

extern "C" int vtm_cross_attention(const void* x_dev, const void* ctx_dev, const void* w_q_dev, const void* w_kv_dev,
                                   const void* w_o_dev, const void* b_o_dev, const void* resid_dev, int32_t B, int32_t Lq,
                                   int32_t Lk, int32_t C, int32_t Cctx, int32_t heads, float scale, void* y_dev,
                                   void* ws_dev, size_t ws_bytes, void* stream_) {
  using namespace vtm;
  if (!x_dev || !ctx_dev || !w_q_dev || !w_kv_dev || !w_o_dev || !y_dev || !ws_dev) return VTM_E_NULL;
  if (B <= 0 || Lq <= 0 || Lk <= 0 || C <= 0 || Cctx <= 0 || heads <= 0 || C % heads != 0) return VTM_E_SHAPE;
  const int d = C / heads;
  if (d % 8 != 0 || C % 8 != 0 || Cctx % 8 != 0) return VTM_E_SHAPE;
  if (d > 128) return VTM_E_UNSUPPORTED;
  if (ws_bytes < vtm_cross_attention_workspace_bytes(B, Lq, Lk, C, heads)) return VTM_E_WS;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int DP = d <= 64 ? 64 : 128;
  __half* qh = static_cast<__half*>(ws_dev);
  __half* kh = qh + static_cast<size_t>(B) * heads * Lq * DP;
  __half* vh = kh + static_cast<size_t>(B) * heads * Lk * DP;
  __half* o = vh + static_cast<size_t>(B) * heads * Lk * DP;
  void* part_ws = reinterpret_cast<void*>(
      (reinterpret_cast<uintptr_t>(o + static_cast<size_t>(B) * Lq * C) + 255u) & ~static_cast<uintptr_t>(255u));
  const int emb = fa_use_embed(d) ? 1 : 0;
  int rc = launch_head_proj(x_dev, w_q_dev, qh, B, Lq, C, C, heads, DP, 0, 1, emb ? scale * 1.4426950408889634f : 1.f, 0, stream);
  if (rc) return rc;
  rc = launch_head_proj(ctx_dev, w_kv_dev, kh, B, Lk, Cctx, C, heads, DP, 1, 2, 1.f, emb, stream);
  if (rc) return rc;
  rc = launch_fa_any(qh, kh, vh, o, part_ws, B, Lq, Lk, C, heads, d, scale, 0, emb, stream);
  if (rc) return rc;
  const int M = B * Lq;
  if (resid_dev) return vtm_linear_residual_f16(o, w_o_dev, b_o_dev, resid_dev, C, M, C, C, y_dev, C, stream_);
  return vtm_linear_f16(o, w_o_dev, b_o_dev, M, C, C, y_dev, C, stream_);
}
