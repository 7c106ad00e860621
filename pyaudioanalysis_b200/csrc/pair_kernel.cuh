// Warp-autonomous short-term kernel for windows N = 32 * R (R = 10, 15, 16, 20, 25, 30, 32: 320 / 480 / 512 / 640 / 800 / 960 /
// 1024 samples).
//
// One WARP owns a run of consecutive frames of one clip and processes them two at a time with no CTA-wide barrier:
//   * frames a = 2q and b = 2q + 1 ride through ONE complex FFT of length N: z[n] = sa (xa[n] - xa[0]) + i sb (xb[n] - xb[0])
//     (sa, sb: per-frame powers of two that bring both frames to unit level, so the float32 error of either spectrum is
//     relative to its OWN level).  n = 32 n1 + n2, k = k1 + R k2:  lane n2 runs the R-point transform over n1 in
//     registers (samples come straight from global memory, 2-byte coalesced loads), twiddles by W_N^(n2 k1), one
//     transpose through shared memory, lane k1 runs the 32-point transform over n2.  Z lands in shared memory in natural
//     order and |Xa[k]| = |Z[k] + conj Z[N-k]| / 2 sa,  |Xb[k]| = |Z[k] - conj Z[N-k]| / 2 sb  come out with lane = k mod 32
//     -- no post-twiddle, no packed-real butterfly.
//   * time-domain rows (zcr / energy / energy entropy) are accumulated per 32-sample row straight from the loaded
//     registers: sign masks by warp ballot, block energies by one multi-value butterfly reduction; with hop = N / 2 every
//     sample is visited once (the second halves of a and b are new, the rest is carried in a small ring).
//   * the spectral rows reuse the half-warp dense pass of fast_kernel.cuh (two frames per warp), the mel / chroma / DCT
//     contractions are shared-memory dot products over the two |X| rows; feature rows collect in an [8 x 34] tile per warp
//     and leave as 32-byte row segments.
// Work: every warp starts with an equal contiguous share of the launch's pair steps and takes it in chunks of a few pairs;
// a warp that runs dry steals the back half of somebody's remainder (sched.cuh).  A run starts one pair early (flux and the
// deltas need frame t - 1) and pairs are always (2q, 2q + 1), so results do not depend on how a clip was cut.
#pragma once
#include "common.cuh"
#include "dft_codelets.cuh"
#include <algorithm>
#include <cstring>
#include <utility>
#include "fast_kernel.cuh"
#include "sched.cuh"

namespace b200aa {

// Resident warps per SM.  Measured on B200 (1000 x 10 s @16 kHz, 800 / 400; profiles/ab_diet_r2.jsonl), CTAs x warps:
//   2 x 8 at 128 registers (round 2's first layout, 11.9 KB of shared memory per warp) 0.904 ms;  the 9.6 KB layout below:
//   2 x 8 (128 regs) 0.916   2 x 10 (96 regs; 3+3+2+2 warps per scheduler and CTA) 0.923   1 x 22 (80 regs, spills) 0.874
//   1 x 20 (96 regs, five warps per scheduler) 0.824  <- what the 800-sample window gets (22 warps would fit).  Warps per CTA
//   stay a multiple of four: a CTA's warps go round-robin to the four schedulers of the SM.  The shorter windows fit 24 warps
//   (80 registers, no spills to speak of): 640 / 320 0.868 -> 0.851 ms, 512 / 256 1.024 -> 0.984, 320 / 160 1.236 -> 1.191
//   (profiles/ab_solo_r2.jsonl); 960 and 1024 samples run 16 warps at 128 registers.
#ifndef B200AA_PAIR_MAXWARPS
#define B200AA_PAIR_MAXWARPS 24
#endif
constexpr int kPairMaxWarps = B200AA_PAIR_MAXWARPS;     // warps per CTA (each one autonomous); fewer for the longest windows (shared memory)
#ifndef B200AA_PAIR_MINBLOCKS
#define B200AA_PAIR_MINBLOCKS 1
#endif
constexpr int kPairMinBlocks = B200AA_PAIR_MINBLOCKS;   // one CTA per SM: the twiddle / mel / DCT / chroma tables exist once per SM
// the solo kernel's feature layout (solo_kernel.cuh): config 3 (64 x 60 s @44.1 kHz, 882 / 441) 2 x 8 warps 1.162 ms, 1 x 20 1.067,
// 1 x 24 (80 registers, no spills) 1.075; 400 / 160 on the bench batch 1.808 / 1.625 / 1.599
#ifndef B200AA_SOLO_MAXWARPS
#define B200AA_SOLO_MAXWARPS 24
#endif
#ifndef B200AA_SOLO_MINBLOCKS
#define B200AA_SOLO_MINBLOCKS 1
#endif
constexpr int kSoloMaxWarps = B200AA_SOLO_MAXWARPS, kSoloMinBlocks = B200AA_SOLO_MINBLOCKS;

template <int R>
struct PairShape {
    static constexpr int N = 32 * R, K = N / 2, Kp = DenseShape<K>::Kp, C = Kp / 32;
    static constexpr int JK = (K + 31) / 32;         // strided rows that hold real bins (k = lane + 32 j)
    // pass-1 outputs, row k1: quad m = n2 / 2 holds (re n2, re n2 + 1, im n2, im n2 + 1) -- re and im swap places in quads
    // 8..15 -- so that the second pass reads the (even, odd) FP32x2 operands of fft32_soa as one 16-byte word per quad.
    // Row stride LS = 68 floats (4 mod 32 words): the eight rows of a quarter-warp's 16-byte reads hit eight distinct bank
    // quads; the swap puts lanes n2 and n2 + 16 of pass 1's 4-byte stores on different banks.
    static constexpr int LS = 68;
    static constexpr int TZ = (R * LS / 2 > N + 2) ? R * LS / 2 : N + 2;   // float2 elements of the transform buffer
    static constexpr int Lt = N / 10;                // energy-entropy block length (ShortTermFeatures.py:41)
    static constexpr bool kShareable = (N % 160) == 0;    // half a frame = 5 whole blocks, rows split at lane 0 / 16 only
    // after the separation the transform buffer holds the |X| row of frame a (Kp floats) and, behind it, the mel scratch:
    // filter outputs, their log10, and the folded halves for the DCT ([f][0..19] sums, [f][20..39] differences), 2 x 40 each
    // (everything one step needs between the separation and the next transform lives in the transform buffer: a warp keeps
    // only the previous pair's |X| row, the feature tile and the block-energy ring beside it -- 9.6 KB for the 800-sample
    // window instead of 11.9 KB, i.e. 20-22 resident warps per SM instead of 16)
    static constexpr int MS0 = (Kp + 3) & ~3;
    static constexpr int RB0 = MS0 + 6 * B200AA_N_MEL;       // |X| row of frame b (Kp floats, 16-byte aligned)
    static constexpr int PT0 = RB0 + Kp;                     // spectral-entropy parts of the dense pass (2 x 32)
    static constexpr int CH0 = PT0 + 64;                     // raw chroma sums (2 x 12)
    static_assert(2 * TZ >= CH0 + 24, "|X| rows of both frames + mel scratch + parts + chroma fit the transform buffer");
    static_assert((RB0 % 4) == 0 && (LS % 4) == 0, "aligned |X| row, aligned pass-1 quads");
    static_assert(Lt >= 32, "a 32-sample row touches two blocks at most");
};

template <int R>
struct alignas(16) PairWarpMem {
    using S = PairShape<R>;
    float2 tz[S::TZ];                       // pass-1 outputs [k1][LS] (PairShape::LS)  ->  Z[k] (natural order, Z[N] = Z[0])  ->
                                            // |X| row of a | mel scratch | |X| row of b | entropy parts | chroma sums (PairShape::MS0 ...)
    alignas(16) float rowp[S::Kp];          // |X| row of the previous pair's frame b (the flux of frame a needs it)
    float fv[9 * kFvStride];                // feature rows: row 0 = the frame before the tile, rows 1..8 = the tile
    float blk[24];                          // block energies: a -> [0, 10), b -> [5, 15) (shared halves) or [10, 20); rests at 20, 21
};

// warps per CTA such that kPairMinBlocks CTAs fit the 227 KB of an SM (per CTA: kPairCtaCap of pair_launch_t, twiddles, lane
// constants, up to 6.5 KB of mel / DCT / chroma tables)
constexpr int kPairCtaCap = (kPairMinBlocks == 1 ? 227 : (kPairMinBlocks == 2 ? 113 : 228 / kPairMinBlocks - 1)) * 1024;
template <int R>
__host__ __device__ constexpr int pair_warps()
{
    constexpr int budget = kPairCtaCap - R * 32 * 8 - 256 - 6656;
    constexpr int w = budget / int(sizeof(PairWarpMem<R>));
    constexpr int c = w > kPairMaxWarps ? kPairMaxWarps : (w < 2 ? 2 : w);
    return c >= 4 ? (c & ~3) : c;           // whole rounds over the four schedulers
}

template <int R>
struct alignas(16) PairCtaMem {
    float2 tw[R * 32];                      // W_N^(k1 n2), [k1][n2]
    alignas(16) int dlane[16 * 4];          // per-lane constants of the dense pass
    PairWarpMem<R> w[pair_warps<R>()];
};

// constant tables of the pair kernel (int32 words, copied to shared memory once per CTA)
struct PairBlobLayout {
    int dct;        // [13 x 41] DCT rows (float)
    int mel_rec;    // [LQ][16] one record per (step q, lane): first bin | filter << 16 | flush << 24
    int mel_w;      // [LQ][16] float4: the four tap weights of the record (16-byte aligned)
    int chr;        // [CT][16] {bin, weight}: tap t of pitch class l (lanes 12..15: padding)
    int lq, ct;     // steps per lane
    int words;
};

struct PairParams {
    StParams st;
    const int *pblob;          // tables above
    PairBlobLayout pbl;
    const float2 *tw;          // [R][32] inter-pass twiddles
    StealParams sched;         // work distribution (sched.cuh): g = clip * sched.per_clip + pair
    float *dbg;                // optional dump of the |X| rows [clip][frame][K] (debugging)
};

template <int R>
inline size_t pair_smem_bytes(int blob_words) { return sizeof(PairCtaMem<R>) + sizeof(int) * size_t((blob_words + 3) & ~3); }

__device__ __forceinline__ float fsqrt_fast(float x)        // MUFU.SQRT (2 ulp, 0 -> 0)
{
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// ----------------------------------------------------------------------------------------------
// Dense spectral rows of two frames per warp (half-warp each): spectral_features_h of fast_kernel.cuh with the previous
// frame's row sum taken from where it already exists -- half 1 (frame b) receives half 0's (frame a's) sum by shuffle,
// half 0 the carried sum of the previous pair's b -- instead of re-reading the previous row.
// ----------------------------------------------------------------------------------------------
// per-lane constants: .x = bins of the lane's chunk that belong to the earlier entropy block, [.y, .z) = parts of block l
template <int K>
__device__ __forceinline__ int4 pair_lane_init(int l)
{
    constexpr int CB = 2 * (((K + 31) / 32) | 1), Lb = K / 10;
    const int k0 = l * CB;
    const int bnd = ((k0 + CB - 1) / Lb) * Lb;
    int4 d;
    d.x = bnd > k0 ? bnd - k0 : 0;
    int ps = 32, pe = 0;
    for (int q = 0; q < 16; ++q) {
        const int b0 = q * CB, bb = ((b0 + CB - 1) / Lb) * Lb, sp = bb > b0 ? bb - b0 : 0;
        if (sp > 0 && b0 >= l * Lb && b0 + sp <= (l + 1) * Lb) { ps = min(ps, 2 * q); pe = max(pe, 2 * q + 1); }
        if (b0 + sp >= l * Lb && b0 + CB <= (l + 1) * Lb) { ps = min(ps, 2 * q + 1); pe = max(pe, 2 * q + 2); }
    }
    if (l >= 10) { ps = 0; pe = 0; }
    d.y = ps; d.z = pe; d.w = 0;
    return d;
}

template <int K>
__device__ __forceinline__ void pair_spectral(const float *X, const float *Xp, float sxp_carried, bool own_prev, const int *dlp,
                                              float *parts, float *fv, int l, int half)
{
    constexpr int C2 = ((K + 31) / 32) | 1, CB = 2 * C2, Lb = K / 10;
    static_assert(CB < Lb, "one entropy block boundary per lane at most");
    const int k0 = l * CB;
    const int4 dlv = *reinterpret_cast<const int4 *>(dlp);        // {split (bins), ps, pe, -}
    const float2 *X2 = reinterpret_cast<const float2 *>(X) + l * C2;
    const float2 *Xp2 = reinterpret_cast<const float2 *>(Xp) + l * C2;
    float2 x2[C2];
#pragma unroll
    for (int j = 0; j < C2; ++j) x2[j] = X2[j];
    float sx = 0.f, s1 = 0.f, sb = 0.f;
    float2 plo2 = make_float2(0.f, 0.f), phi2 = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < C2; ++j) {
        const float t = x2[j].x + x2[j].y;
        sx += t;
        s1 = fmaf(float(2 * j + 1), t, s1);
        sb += x2[j].y;
        const float2 sq = __fmul2_rn(x2[j], x2[j]);
        if constexpr ((Lb % 2) == 0) {                   // block boundaries fall between (even, odd) bin pairs
            if (2 * j < dlv.x) plo2 = f2add(plo2, sq); else phi2 = f2add(phi2, sq);
        } else {                                         // power-of-two windows: a boundary may split a pair
            const float2 m = make_float2(2 * j < dlv.x ? 1.f : 0.f, 2 * j + 1 < dlv.x ? 1.f : 0.f);
            plo2 = __ffma2_rn(sq, m, plo2);
            phi2 = __ffma2_rn(sq, make_float2(1.f - m.x, 1.f - m.y), phi2);
        }
    }
    const float plo = plo2.x + plo2.y, phi = phi2.x + phi2.y, part = plo + phi;
    float sk = fmaf(float(k0), sx, s1 + sb);         // sum (k0 + i + 1) x_i
    parts[2 * l] = plo;
    parts[2 * l + 1] = phi;
    {   // two sums in 4 exchanges
        const bool up = l & 8;
        float keep = up ? sk : sx;
        const float give = up ? sx : sk;
        keep += __shfl_xor_sync(0xffffffffu, give, 8);
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, o);
        sx = __shfl_sync(0xffffffffu, keep, 0, 16);
        sk = __shfl_sync(0xffffffffu, keep, 8, 16);
    }
    // previous frame's row sum: frame b <- frame a (the other half, just computed), frame a <- carried (or itself)
    const float sx_a = __shfl_sync(0xffffffffu, sx, 0);
    const float sxp = half ? sx_a : (own_prev ? sx : sxp_carried);
    float incl = part;
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) {
        const float n = __shfl_up_sync(0xffffffffu, incl, o, 16);
        if (l >= o) incl += n;
    }
    const float sxx = __shfl_sync(0xffffffffu, incl, 15, 16);
    constexpr float invK = 1.f / float(K);
    const float cen = sx > 0.f ? fdiv(sk, sx) * invK : 0.f;
    const float nx = fdiv(1.f, sx + float(K) * B200AA_EPS);
    const float np_ = fdiv(1.f, sxp + float(K) * B200AA_EPS);
    const float thr = 0.90f * sxx - B200AA_EPS;
    float2 d2 = make_float2(float(k0 + 1) * invK - cen, float(k0 + 2) * invK - cen);
    const float2 dstep = make_float2(2.f * invK, 2.f * invK);
    const float2 nx2 = make_float2(nx, nx), mnp2 = make_float2(-np_, -np_);
    float2 sp2 = make_float2(0.f, 0.f), fl2 = make_float2(0.f, 0.f);
#ifdef B200AA_ROLLOFF_SEQ
    float run = incl - part, below = 0.f;       // (A/B reference: every lane walks its own chunk bin by bin)
#else
    // rolloff = number of bins whose cumulative energy stays <= thr.  The prefix over the lanes' chunks is monotone, so the
    // lanes before the crossing one count all their CB bins and only the crossing lane's chunk needs a bin-by-bin look: the
    // half-warp takes it together (one or two float2 of that chunk per lane, a 4-step scan) instead of CB dependent steps per lane.
    float below;
    {
        const unsigned under = __ballot_sync(0xffffffffu, incl <= thr);
        const int cl = __popc((under >> (16 * half)) & 0xffffu);      // chunks entirely under the threshold (< 16: the last prefix is sxx > thr)
        const float base = __shfl_sync(0xffffffffu, incl - part, cl, 16);      // cumulative energy before the crossing chunk
        constexpr int PER = (C2 + 15) / 16;                           // float2 elements of that chunk per lane (2 for the 1024-sample window)
        float2 sq[PER];
        float pre = 0.f;
#pragma unroll
        for (int t = 0; t < PER; ++t) {
            const int idx = l * PER + t;
            const float2 xc = idx < C2 ? reinterpret_cast<const float2 *>(X)[cl * C2 + idx] : make_float2(0.f, 0.f);
            sq[t] = __fmul2_rn(xc, xc);
            pre += sq[t].x + sq[t].y;
        }
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) {
            const float n = __shfl_up_sync(0xffffffffu, pre, o, 16);
            if (l >= o) pre += n;
        }
        const float prev = __shfl_up_sync(0xffffffffu, pre, 1, 16);
        float run = base + (l ? prev : 0.f);
        below = 0.f;
#pragma unroll
        for (int t = 0; t < PER; ++t) {
            const bool real = l * PER + t < C2;
            run += sq[t].x;
            below += (real && !(run > thr)) ? 1.f : 0.f;
            run += sq[t].y;
            below += (real && !(run > thr)) ? 1.f : 0.f;
        }
        if (l == 0) below += float(cl * CB);
    }
#endif
#pragma unroll
    for (int j = 0; j < C2; ++j) {
        sp2 = __ffma2_rn(__fmul2_rn(d2, d2), x2[j], sp2);
        d2 = f2add(d2, dstep);
        const float2 df = __ffma2_rn(x2[j], nx2, __fmul2_rn(Xp2[j], mnp2));
        fl2 = __ffma2_rn(df, df, fl2);
#ifdef B200AA_ROLLOFF_SEQ
        run = fmaf(x2[j].x, x2[j].x, run);
        below += run > thr ? 0.f : 1.f;
        run = fmaf(x2[j].y, x2[j].y, run);
        below += run > thr ? 0.f : 1.f;
#endif
    }
    const float sp = sp2.x + sp2.y, fl = fl2.x + fl2.y;
    __syncwarp();
    float e = 0.f;
    constexpr int MAXP = 2 * (Lb / CB + 2);
#pragma unroll
    for (int q = 0; q < MAXP; ++q) e += (dlv.y + q < dlv.z) ? parts[dlv.y + q] : 0.f;
    float ent = 0.f;
    if (l < 10) {
        const float sj = fdiv(e, sxx + B200AA_EPS);
        ent = -sj * flog2(sj + B200AA_EPS);
    }
    float q4;
    {   // four sums in 4 exchanges: lanes 0-3 spread, 4-7 flux, 8-11 rolloff count, 12-15 entropy
        const bool up8 = l & 8, up4 = l & 4;
        float k0_ = up8 ? below : sp, k1_ = up8 ? ent : fl;
        const float g0_ = up8 ? sp : below, g1_ = up8 ? fl : ent;
        k0_ += __shfl_xor_sync(0xffffffffu, g0_, 8);
        k1_ += __shfl_xor_sync(0xffffffffu, g1_, 8);
        float kk = up4 ? k1_ : k0_;
        const float gg = up4 ? k0_ : k1_;
        kk += __shfl_xor_sync(0xffffffffu, gg, 4);
        kk += __shfl_xor_sync(0xffffffffu, kk, 2);
        kk += __shfl_xor_sync(0xffffffffu, kk, 1);
        q4 = kk;
    }
    if (l == 0) {
        fv[3] = cen;
        fv[4] = sx > 0.f ? fsqrt_pos(fdiv(q4, sx)) : 0.f;
        fv[34] = sx;
        fv[35] = sxx;
    }
    if (l == 4) fv[6] = q4;
    if (l == 8) fv[7] = q4 >= float(K) ? 0.f : q4 * invK;
    if (l == 12) fv[5] = q4;
    __syncwarp();
}

// ----------------------------------------------------------------------------------------------
// Sum NV per-lane values over the warp with a halving butterfly: after the call v[0] of lane l holds the
// total of value number (l >> (5 - log2 P0)), P0 = the power of two >= NV (32, 16 or 8): NV + NV/2 + ... shuffles
// instead of 5 NV.
// ----------------------------------------------------------------------------------------------
template <int P, int NV, int D, int NA>
__device__ __forceinline__ void mr_halve(float (&v)[NA], int lane)
{
    if constexpr (P > 1) {
        constexpr int H = P / 2;
        const bool up = lane & D;
#pragma unroll
        for (int i = 0; i < H; ++i) {
            if (i < NV) {
                if (i + H < NV) {
                    const float keep = up ? v[i + H] : v[i], send = up ? v[i] : v[i + H];
                    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, D);
                } else {
                    v[i] += __shfl_xor_sync(0xffffffffu, v[i], D);
                }
            }
        }
        mr_halve<H, (NV < H ? NV : H), D / 2, NA>(v, lane);
    } else {
#pragma unroll
        for (int d = D; d >= 1; d >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], d);
    }
}
template <int NV>
struct MultiReduce {
    static constexpr int P0 = NV > 16 ? 32 : (NV > 8 ? 16 : 8);
    static constexpr int SH = NV > 16 ? 0 : (NV > 8 ? 1 : 2);       // value j ends up in lanes (l >> SH) == j
    __device__ static __forceinline__ void run(float (&v)[NV], int lane) { mr_halve<P0, NV, 16, NV>(v, lane); }
};

// ----------------------------------------------------------------------------------------------
// time-domain accumulation over the 32-sample rows of one frame (u[r] of lane l = sample 32 r + l, as the exact float
// M0 + x): per-lane sums of y^2 per energy-entropy block, and the number of sign flips from the ballot masks
//   FULL: all rows, blocks 0..9 (+ the samples beyond 10 blocks);  !FULL: the second half only (blocks 5..9)
// ----------------------------------------------------------------------------------------------
template <int R, bool FULL>
struct TdShape {
    using S = PairShape<R>;
    static constexpr int NREST = (S::N % 10) ? 1 : 0;
    static constexpr int NE = FULL ? 10 + NREST : 5;          // accumulators
    static constexpr int EB = FULL ? 0 : 5;                   // first block
    static constexpr int NFIRST = FULL ? 0 : S::N / 2;        // first sample covered
    static constexpr int ROW0 = NFIRST / 32, LANE0 = NFIRST % 32;
    static constexpr int ZROW0 = (!FULL && LANE0 == 0) ? ROW0 - 1 : ROW0;     // first row whose sign mask is needed
    static_assert(FULL || S::kShareable, "half-frame sharing needs whole blocks per half");
};

// Sign flips of the rows [ZROW0, R) from their ballot masks, one row per lane: lane r holds row r's mask m (0 in a lane
// that owns no row), takes row r - 1's by one shuffle and counts the pairs (n - 1, n), n >= max(1, NFIRST), of its row.
// Returns the lane's count plus, in bits 12.., the flip at sample NFIRST (the link between the halves; !FULL only).
// Whatever lane ZROW0 receives as its predecessor is masked out: its bit 0 is sample 0 (FULL) or precedes NFIRST.
template <int R, bool FULL>
__device__ __forceinline__ unsigned td_row_flips(unsigned m, int lane)
{
    using Td = TdShape<R, FULL>;
    const unsigned prev = __shfl_up_sync(0xffffffffu, m, 1);
    const int nstart = FULL ? 1 : Td::NFIRST, n0 = 32 * lane;
    const unsigned valid = lane < Td::ROW0 || lane >= R ? 0u
                         : (n0 >= nstart ? 0xffffffffu : (0xffffffffu << (nstart - n0)));
    const unsigned c = (m ^ __funnelshift_l(prev, m, 1)) & valid;
    unsigned v = __popc(c);
    if (!FULL && lane == Td::ROW0) v += ((c >> Td::LANE0) & 1u) << 12;
    return v;
}

template <int R, bool FULL, bool TWO>
__device__ __forceinline__ void td_frame(const float (&u)[R], float cm, const b200aa_clip_norm &nm, int lane,
                                         float *e /* [NE] */, int &flips, int &link)
{
    using S = PairShape<R>;
    using Td = TdShape<R, FULL>;
    constexpr int N = S::N, Lt = S::Lt;
    unsigned mP = 0u, mQ = 0u;          // row `lane`'s sign masks
#pragma unroll
    for (int r = Td::ZROW0; r < R; ++r) {
        const float d = u[r] - cm;
        // ---- sign masks: P = samples above the clip mean, Q = below (complementary unless a sample can equal the mean)
        const unsigned P = __ballot_sync(0xffffffffu, d > nm.lo);
        if (lane == r) mP = P;
        if (TWO) { const unsigned Q = __ballot_sync(0xffffffffu, d < nm.hi); if (lane == r) mQ = Q; }
        if (r >= Td::ROW0) {
            const int n0 = 32 * r;
            // ---- energy of the normalised samples into the row's block(s)
            // (fused multiply-adds, predicated: bit-identical to td_pair below, whichever of the two handles a frame)
            const float y = fmaf(nm.a, d, nm.bp);
            const bool live = !(r == Td::ROW0 && Td::LANE0 > 0) || lane >= Td::LANE0;
            const int b0 = (n0 / Lt) < 10 ? (n0 / Lt) : 10;
            const int end = b0 < 10 ? (b0 + 1) * Lt : N;
            const int thr = end - n0;                     // samples of this row that still belong to block b0
            const int i0 = b0 - Td::EB, i1 = (b0 + 1 < 10 ? b0 + 1 : 10) - Td::EB;
            if (thr >= 32) {
                if (i0 >= 0 && i0 < Td::NE) { if (live) e[i0] = fmaf(y, y, e[i0]); }
            } else {
                const bool first = lane < thr;
                if (i0 >= 0 && i0 < Td::NE) { if (live && first) e[i0] = fmaf(y, y, e[i0]); }
                if (i1 >= 0 && i1 < Td::NE) { if (live && !first) e[i1] = fmaf(y, y, e[i1]); }
            }
        }
    }
    unsigned v = td_row_flips<R, FULL>(mP, lane);
    if (TWO) v += td_row_flips<R, FULL>(mQ, lane);
    v = __reduce_add_sync(0xffffffffu, v);
    const int fl = int(v & 0xfffu), lk = int(v >> 12);
    // one-sided counting saw every change once; |s_n - s_(n-1)| is 2 for a sign change without a zero in between
    flips = TWO ? fl : 2 * fl;
    link = TWO ? lk : 2 * lk;
}

// The same accumulation for BOTH frames of a pair at once (they cover the same rows): u[r] = (sample of a, sample of b),
// e2[i] = (block sum of a, block sum of b) -- the arithmetic runs in FP32x2 instructions, only the sign masks stay per frame.
template <int R, bool FULL, bool TWO>
__device__ __forceinline__ void td_pair(const float2 (&u)[R], float cm, const b200aa_clip_norm &nm, int lane,
                                        float2 *e2 /* [NE] */, int &flips_a, int &link_a, int &flips_b, int &link_b)
{
    using S = PairShape<R>;
    using Td = TdShape<R, FULL>;
    constexpr int N = S::N, Lt = S::Lt;
    unsigned mPa = 0u, mQa = 0u, mPb = 0u, mQb = 0u;       // row `lane`'s sign masks
    const float2 ncm = make_float2(-cm, -cm), a2 = make_float2(nm.a, nm.a), bp2 = make_float2(nm.bp, nm.bp);
#pragma unroll
    for (int r = Td::ZROW0; r < R; ++r) {
        const float2 d = __fadd2_rn(u[r], ncm);
        const unsigned Pa = __ballot_sync(0xffffffffu, d.x > nm.lo), Pb = __ballot_sync(0xffffffffu, d.y > nm.lo);
        if (lane == r) { mPa = Pa; mPb = Pb; }
        if (TWO) {
            const unsigned Qa = __ballot_sync(0xffffffffu, d.x < nm.hi), Qb = __ballot_sync(0xffffffffu, d.y < nm.hi);
            if (lane == r) { mQa = Qa; mQb = Qb; }
        }
        if (r >= Td::ROW0) {
            const int n0 = 32 * r;
            const float2 y = __ffma2_rn(a2, d, bp2);
            const bool live = !(r == Td::ROW0 && Td::LANE0 > 0) || lane >= Td::LANE0;
            const int b0 = (n0 / Lt) < 10 ? (n0 / Lt) : 10;
            const int end = b0 < 10 ? (b0 + 1) * Lt : N;
            const int thr = end - n0;
            const int i0 = b0 - Td::EB, i1 = (b0 + 1 < 10 ? b0 + 1 : 10) - Td::EB;
            if (thr >= 32) {
                if (i0 >= 0 && i0 < Td::NE) { if (live) e2[i0] = __ffma2_rn(y, y, e2[i0]); }
            } else {
                const bool first = lane < thr;
                if (i0 >= 0 && i0 < Td::NE) { if (live && first) e2[i0] = __ffma2_rn(y, y, e2[i0]); }
                if (i1 >= 0 && i1 < Td::NE) { if (live && !first) e2[i1] = __ffma2_rn(y, y, e2[i1]); }
            }
        }
    }
    // both frames' counts in one reduction: a in bits 0..15, b in 16..31 (each field stays below 2^14)
    unsigned v = td_row_flips<R, FULL>(mPa, lane) + (td_row_flips<R, FULL>(mPb, lane) << 16);
    if (TWO) v += td_row_flips<R, FULL>(mQa, lane) + (td_row_flips<R, FULL>(mQb, lane) << 16);
    v = __reduce_add_sync(0xffffffffu, v);
    const int fa = int(v & 0xfffu), la = int((v >> 12) & 0xfu), fb = int((v >> 16) & 0xfffu), lb = int(v >> 28);
    flips_a = TWO ? fa : 2 * fa; link_a = TWO ? la : 2 * la;
    flips_b = TWO ? fb : 2 * fb; link_b = TWO ? lb : 2 * lb;
}

// power of two s with s * rms(x - x0) ~ 1 (E = sum y^2 of the frame, y = a (x - mean)); its inverse
__device__ __forceinline__ void frame_scale(float E, float inv_a2n, float &s, float &inv_s)
{
    const float t = E * inv_a2n;                                // mean square in sample units (>= 0)
    const int ex = (__float_as_int(t) >> 23) & 0xff;            // biased exponent
    int k = (127 - ex) >> 1;
    k = k < -30 ? -30 : (k > 40 ? 40 : k);
    s = __int_as_float((127 + k) << 23);
    inv_s = __int_as_float((127 - k) << 23);
}

// tables of the feature phases in shared memory
struct FeatTables {
    const float *dct;
    const int *mrec;
    const float4 *mw;
    const int2 *chr;
    int LQ, CT;
};

// ----------------------------------------------------------------------------------------------
// |X| rows of two frames (a: lanes 0-15, b: lanes 16-31) -> feature slots 3..33 of fva / fvb:
// spectral rows (pair_spectral), mel filters + log10, folded DCT-II, chroma.  Xprev = the row before frame a
// (frame a itself when there is none); frame b's predecessor is frame a.
// ----------------------------------------------------------------------------------------------
template <int K>
__device__ __forceinline__ void rows_to_features(const float *Xa, const float *Xb, const float *Xprev, bool fresh, float carried,
                                                 const int *dlane, float *parts, float *msraw, float *mslog, float *mfold, float *chr,
                                                 float *fva, float *fvb, const FeatTables &ft, int lane)
{
    const int half = lane >> 4, l16 = lane & 15;
    const unsigned FULLM = 0xffffffffu;
    {
        const float *X = half ? Xb : Xa;
        const float *Xp = half ? Xa : Xprev;
        pair_spectral<K>(X, Xp, carried, fresh, dlane + l16 * 4, parts + half * 32, half ? fvb : fva, l16, half);
    }
    // ---- mel filters: 16 lanes per frame, LQ steps of four taps each (whole filters per lane, balanced on the host);
    //      raw chroma sums: 12 lanes per frame, CT taps each
    {
        const float *X = half ? Xb : Xa;
        float acc = 0.f;
#pragma unroll 4
        for (int q = 0; q < ft.LQ; ++q) {
            const int rec = ft.mrec[q * 16 + l16];
            const float4 w = ft.mw[q * 16 + l16];
            const float *xp = X + (rec & 0xffff);
            acc = fmaf(xp[0], w.x, acc);
            acc = fmaf(xp[1], w.y, acc);
            acc = fmaf(xp[2], w.z, acc);
            acc = fmaf(xp[3], w.w, acc);
            if (rec & (1 << 24)) { msraw[half * B200AA_N_MEL + ((rec >> 16) & 0xff)] = acc; acc = 0.f; }
        }
        float ch = 0.f;
        for (int t = 0; t < ft.CT; ++t) {
            const int2 e = ft.chr[t * 16 + l16];
            const float v = X[e.x];
            ch = fmaf(v * v, __int_as_float(e.y), ch);
        }
        if (l16 < 12) chr[half * 12 + l16] = ch;
    }
    __syncwarp();
    // ---- log10, fold (m_n - k) +- (m_(39-n) - k) with k = m_0 (see flat_dct in fast_kernel.cuh), 13 x 20 DCT rows
#pragma unroll
    for (int t = lane; t < 2 * B200AA_N_MEL; t += 32) mslog[t] = 0.30102999566398120f * flog2(msraw[t] + B200AA_EPS);
    __syncwarp();
#pragma unroll
    for (int t = lane; t < 2 * B200AA_N_MEL; t += 32) {
        const int f = t >= B200AA_N_MEL ? 1 : 0, r = t - f * B200AA_N_MEL;
        const int kind = r >= 20 ? 1 : 0, n = r - 20 * kind;
        const float *m = mslog + f * B200AA_N_MEL;
        const float a = m[n], bq = m[39 - n], kap = m[0];
        mfold[t] = kind ? a - bq : (a - kap) + (bq - kap);
    }
    __syncwarp();
    {
        const int c = l16 < B200AA_N_MFCC ? l16 : 0;
        const float *src = mfold + half * B200AA_N_MEL + 20 * (c & 1);
        const float *row = ft.dct + c * 41;
        float acc = 0.f;
#pragma unroll
        for (int n = 0; n < 20; ++n) acc = fmaf(row[n], src[n], acc);
        if (c == 0) acc = fmaf(6.324555320336759f, mslog[half * B200AA_N_MEL], acc);      // sqrt(1/40) * 40 * k
        if (l16 < B200AA_N_MFCC) (half ? fvb : fva)[8 + c] = acc;
    }
    chroma_finalize_h(chr + half * 12, half ? fvb : fva, l16, true);
    __syncwarp();
    (void)FULLM;
}

// [<= 8 frames x n_out] tile of a warp -> global memory: lane -> (feature row f0 + 4 i, frame c): eight consecutive lanes
// write 32 consecutive bytes of one output row; deltas on the fly against the previous row (row 0 of fv = the frame
// before the tile)
__device__ __forceinline__ void tile_store(const float *fv, int tile_n, int tile_t0, float *out_clip, int64_t t_stride, int n_out, int lane)
{
    const int c = lane & 7, f0 = lane >> 3;
    if (c < tile_n) {
        float *const out_b = out_clip + tile_t0 + c;
        const float *cur_row = fv + (1 + c) * kFvStride, *prv_row = fv + c * kFvStride;
        const bool first = tile_t0 + c == 0;              // frame 0 of the clip: deltas are zero
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            const int f = f0 + 4 * i;
            if (f < B200AA_N_BASE) {
                const float v = cur_row[f];
                out_b[size_t(f) * t_stride] = v;
                if (n_out > B200AA_N_BASE) out_b[size_t(f + B200AA_N_BASE) * t_stride] = first ? 0.f : v - prv_row[f];
            }
        }
    }
}

// the pending rows of a warp's tile leave; row 0 of the tile buffer becomes the last row written (the deltas' predecessor)
__device__ __forceinline__ void tile_flush(float *fv, int &tile_n, int &tile_t0, float *out_clip, int64_t t_stride, int n_out, int lane)
{
    if (tile_n > 0) {
        tile_store(fv, tile_n, tile_t0, out_clip, t_stride, n_out, lane);
        __syncwarp();
        fv[lane] = fv[tile_n * kFvStride + lane];
        if (lane < 4) fv[32 + lane] = fv[tile_n * kFvStride + 32 + lane];     // incl. the row sum (slot 34)
        tile_t0 += tile_n;
        tile_n = 0;
        __syncwarp();
    }
}

// ----------------------------------------------------------------------------------------------
// kernel
// ----------------------------------------------------------------------------------------------
template <int R, bool SHARED>
__global__ void __launch_bounds__(32 * pair_warps<R>(), kPairMinBlocks) st_pair_kernel(const PairParams pp)
{
    using S = PairShape<R>;
    constexpr int N = S::N, K = S::K, Kp = S::Kp, C = S::C, JK = S::JK, LS = S::LS;
    static_assert(!SHARED || S::kShareable, "shared halves need N % 160 == 0");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PairCtaMem<R> &cm_ = *reinterpret_cast<PairCtaMem<R> *>(smem_raw);
    int *const blob_s = reinterpret_cast<int *>(smem_raw + sizeof(PairCtaMem<R>));
    const StParams &p = pp.st;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NTHR = 32 * pair_warps<R>();
    for (int i = tid; i < pp.pbl.words; i += NTHR) blob_s[i] = pp.pblob[i];
    for (int i = tid; i < R * 32; i += NTHR) cm_.tw[i] = pp.tw[i];
    if (tid < 16) *reinterpret_cast<int4 *>(cm_.dlane + tid * 4) = pair_lane_init<K>(tid);
    __syncthreads();
    const float *const t_dct = reinterpret_cast<const float *>(blob_s + pp.pbl.dct);
    const int *const t_mrec = blob_s + pp.pbl.mel_rec;
    const float4 *const t_mw = reinterpret_cast<const float4 *>(blob_s + pp.pbl.mel_w);
    const int2 *const t_chr = reinterpret_cast<const int2 *>(blob_s + pp.pbl.chr);
    const FeatTables ftab{t_dct, t_mrec, t_mw, t_chr, pp.pbl.lq, pp.pbl.ct};
    PairWarpMem<R> &wm = cm_.w[warp];
    float *const rowa = reinterpret_cast<float *>(wm.tz);
    // this lane's slots in a pass-1 row (lane = n2)
    const int t_re = 4 * (lane >> 1) + (lane & 1) + 2 * (lane >> 4), t_im = t_re ^ 2;
    float *const msraw = rowa + S::MS0, *const mslog = msraw + 2 * B200AA_N_MEL, *const mfold = mslog + 2 * B200AA_N_MEL;
    const int step = p.step;
    const int half = lane >> 4, l16 = lane & 15;
    const unsigned FULLM = 0xffffffffu;

    const unsigned wglob = blockIdx.x * unsigned(pair_warps<R>()) + unsigned(warp);
    if (lane == 0) sched_begin(pp.sched, wglob);
    __syncwarp();
    const int per_clip = int(pp.sched.per_clip);
    // ---- the run in progress (all of it warp-uniform: the chunk bounds come out of sched_next as lane-0 broadcasts)
    unsigned run_b = 0xffffffffu, run_q = 0xffffffffu;          // its clip and next pair; run_q = ~0: nothing carried
    int tile_n = 0, tile_t0 = 0;
    int zprev = 0;              // sign flips inside the first half of frame a (= second half of the previous b)
    // pending feature rows -> global memory (tile_flush: always inlined -- an out-of-line call in the step loop costs the
    // caller-saved registers)
#define B200AA_PAIR_FLUSH(clip_index) tile_flush(wm.fv, tile_n, tile_t0, p.out + size_t(clip_index) * p.n_out * p.t_stride, p.t_stride, p.n_out, lane)

    unsigned inc = pp.sched.chunk;      // pairs of the next claim (sched_claim adapts it)
    for (;;) {
        unsigned g0 = 0, g1 = 0;
        const int got = sched_next(pp.sched, blockIdx.x * unsigned(pair_warps<R>()) + unsigned(warp), lane, inc, g0, g1);
        if (got == 0) break;
        if (got == 2) continue;
        while (g0 < g1) {                                          // a chunk may run over the end of a clip
        const unsigned cb = g0 / unsigned(per_clip);
        const int q0 = int(g0 - cb * unsigned(per_clip));
        int qe = q0 + int(g1 - g0);
        qe = qe < per_clip ? qe : per_clip;
        const int64_t b = int64_t(cb);
        const bool cont = cb == run_b && unsigned(q0) == run_q;     // the run goes on: state carried, no halo
        if (!cont) B200AA_PAIR_FLUSH(run_b);                        // a new run: the previous one's tile leaves first
        // the clip's values (a handful of cached loads per chunk; kept local so that nothing but the run state is carried)
        const int64_t len = p.len ? p.len[b] : p.n_samples;
        const int T = int(len < N ? 0 : (len - N) / step + 1);
        const int NP = (T + 1) >> 1;                               // pairs of this clip
        const b200aa_clip_norm nm = p.norm[b];
        const bool is16 = p.dtype == B200AA_DTYPE_I16;
        const char *const clip = reinterpret_cast<const char *>(p.sig) + size_t(b) * p.clip_stride * (is16 ? 2 : 4);
        const float M0 = is16 ? 8421376.f : 0.f;                   // u = M0 + x exactly (2^23 + 2^15 trick for int16)
        const float cmv = M0 + nm.m;                                // u - cmv = x - m
        const bool two_sided = !(nm.hi > nm.lo);                    // a sample may equal the clip mean: count both masks
        const float inv_a2n = 1.f / (nm.a * nm.a * float(N));
        const float fscale = nm.a * (0.5f / float(K));
        bool fresh = !cont;         // no state carried from a previous pair: the run starts one pair early
        if (!cont) {
            tile_t0 = 2 * q0;
            zprev = 0;
        }
        g0 += unsigned(qe - q0);
        run_b = cb;
        run_q = 0xffffffffu;
        if (q0 >= NP) continue;                                    // ragged batch: beyond this clip's last pair
        const int q1 = qe < NP ? qe : NP;
        // samples: lane l holds samples 32 r + l of both frames of a pair, as exact floats M0 + x.
        // (Measured and rejected: issuing the loads of pair q + 1 in the middle of step q -- the 50 extra live registers
        // cost more in spills than the hidden latency gains, 0.94 vs 0.89 ms.)
        auto load_pair = [&](int qq, unsigned int (&wa)[R], unsigned int (&wb)[R]) {
            const int ta_ = 2 * qq, tb_ = (ta_ + 1 < T) ? ta_ + 1 : ta_;          // an odd tail pairs the last frame with itself
            if (is16) {
                const unsigned short *pa = reinterpret_cast<const unsigned short *>(clip) + size_t(ta_) * step + lane;
                const unsigned short *pb = reinterpret_cast<const unsigned short *>(clip) + size_t(tb_) * step + lane;
#pragma unroll
                for (int r = 0; r < R; ++r) { wa[r] = __ldg(pa + 32 * r); wb[r] = __ldg(pb + 32 * r); }
            } else {
                const unsigned int *pa = reinterpret_cast<const unsigned int *>(clip) + size_t(ta_) * step + lane;
                const unsigned int *pb = reinterpret_cast<const unsigned int *>(clip) + size_t(tb_) * step + lane;
#pragma unroll
                for (int r = 0; r < R; ++r) { wa[r] = __ldg(pa + 32 * r); wb[r] = __ldg(pb + 32 * r); }
            }
        };
        for (int q = q0 - ((fresh && q0 > 0) ? 1 : 0); q < q1; ++q) {
            const bool store = q >= q0;
            const int ta = 2 * q;
            const bool bvalid = ta + 1 < T;
            float2 uab[R];                      // (sample of a, sample of b) per row: FP32x2 operands
            {
                unsigned int wa[R], wb[R];
                load_pair(q, wa, wb);
                if (is16) {
#pragma unroll
                    for (int r = 0; r < R; ++r)
                        // wa / wb hold the 16-bit samples zero-extended: (x ^ 0x8000) | 0x4B000000 in one xor
                        uab[r] = make_float2(__uint_as_float(wa[r] ^ 0x4B008000u), __uint_as_float(wb[r] ^ 0x4B008000u));
                } else {
#pragma unroll
                    for (int r = 0; r < R; ++r) uab[r] = make_float2(__int_as_float(wa[r]), __int_as_float(wb[r]));
                }
            }
            const float u0a = __shfl_sync(FULLM, uab[0].x, 0), u0b = __shfl_sync(FULLM, uab[0].y, 0);   // first samples
            const int ra = store ? 1 + tile_n : 8, rb = store ? 2 + tile_n : 0;     // feature rows (a halo's b is "previous")
            float *const fva = wm.fv + ra * kFvStride, *const fvb = wm.fv + rb * kFvStride;

            // ---- time-domain rows
            const bool a_full = !SHARED || fresh;
            int fl_a, fl_b;
            {
                constexpr int NEF = TdShape<R, true>::NE, NREST = TdShape<R, true>::NREST;
                if constexpr (SHARED) { if (!a_full) {
                    // steady state: the second halves of a and b are new
                    float2 e2[5];
#pragma unroll
                    for (int i = 0; i < 5; ++i) e2[i] = make_float2(0.f, 0.f);
                    int fa_, la_, fb_, lb_;
                    if (two_sided) td_pair<R, false, true>(uab, cmv, nm, lane, e2, fa_, la_, fb_, lb_);
                    else td_pair<R, false, false>(uab, cmv, nm, lane, e2, fa_, la_, fb_, lb_);
                    float ev[10];
#pragma unroll
                    for (int i = 0; i < 5; ++i) { ev[i] = e2[i].x; ev[5 + i] = e2[i].y; }
                    if (lane < 5) wm.blk[lane] = wm.blk[10 + lane];                 // previous b's second half = a's first half
                    MultiReduce<10>::run(ev, lane);
                    __syncwarp();
                    if ((lane & 1) == 0 && (lane >> 1) < 10) wm.blk[5 + (lane >> 1)] = ev[0];
                    fl_a = zprev + fa_;                       // first half (carried) + link + second half
                    fl_b = (fa_ - la_) + fb_;
                    zprev = fb_ - lb_;
                } else {
                    // first step of a run: all of a, the second half of b
                    float ua[R], ub[R];
#pragma unroll
                    for (int r = 0; r < R; ++r) { ua[r] = uab[r].x; ub[r] = uab[r].y; }
                    float ev[NEF + 5];
#pragma unroll
                    for (int i = 0; i < NEF + 5; ++i) ev[i] = 0.f;
                    int fa_, la_, fb_, lb_;
                    if (two_sided) { td_frame<R, true, true>(ua, cmv, nm, lane, ev, fa_, la_); td_frame<R, false, true>(ub, cmv, nm, lane, ev + NEF, fb_, lb_); }
                    else { td_frame<R, true, false>(ua, cmv, nm, lane, ev, fa_, la_); td_frame<R, false, false>(ub, cmv, nm, lane, ev + NEF, fb_, lb_); }
                    // flips of a's second half alone: b's first half; recount from the shared-half helper
                    int fh_, lh_;
                    { float dump[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
                      if (two_sided) td_frame<R, false, true>(ua, cmv, nm, lane, dump, fh_, lh_); else td_frame<R, false, false>(ua, cmv, nm, lane, dump, fh_, lh_); }
                    MultiReduce<NEF + 5>::run(ev, lane);
                    __syncwarp();
                    {
                        constexpr int SH = MultiReduce<NEF + 5>::SH;
                        const int j = lane >> SH;
                        if ((lane & ((1 << SH) - 1)) == 0 && j < NEF + 5) wm.blk[j] = ev[0];       // a -> 0..9, b's new half -> 10..14
                    }
                    fl_a = fa_;
                    fl_b = (fh_ - lh_) + fb_;
                    zprev = fb_ - lb_;
                } } else {
                    // independent frames (any hop)
                    float2 e2[NEF];
#pragma unroll
                    for (int i = 0; i < NEF; ++i) e2[i] = make_float2(0.f, 0.f);
                    int la_, lb_;
                    if (two_sided) td_pair<R, true, true>(uab, cmv, nm, lane, e2, fl_a, la_, fl_b, lb_);
                    else td_pair<R, true, false>(uab, cmv, nm, lane, e2, fl_a, la_, fl_b, lb_);
                    float ev[2 * NEF];
#pragma unroll
                    for (int i = 0; i < NEF; ++i) { ev[i] = e2[i].x; ev[NEF + i] = e2[i].y; }
                    MultiReduce<2 * NEF>::run(ev, lane);
                    __syncwarp();
                    {
                        constexpr int SH = MultiReduce<2 * NEF>::SH;
                        const int j = lane >> SH;
                        if ((lane & ((1 << SH) - 1)) == 0 && j < 2 * NEF) {
                            const int f = j >= NEF ? 1 : 0, i = j - f * NEF;
                            wm.blk[i < 10 ? 10 * f + i : 20 + f] = ev[0];
                        }
                    }
                    (void)NREST;
                }
            }
            __syncwarp();
            float Ea, Eb;           // frame energies sum y^2 (warp-uniform)
            {
                constexpr int OB = SHARED ? 5 : 10;
                const bool own = l16 < 10;
                const float e = own ? wm.blk[half * OB + l16] : 0.f;
                float tot = half_sum(e);
                if (!SHARED && TdShape<R, true>::NREST) tot += wm.blk[20 + half];
                const float sj = fdiv(e, tot + B200AA_EPS);
                const float H = half_sum(own ? -sj * flog2(sj + B200AA_EPS) : 0.f);
                if (l16 == 0) {
                    float *fv = half ? fvb : fva;
                    fv[0] = float(half ? fl_b : fl_a) * 0.5f / float(N - 1);
                    fv[1] = tot / float(N);
                    fv[2] = H;
                }
                Ea = __shfl_sync(FULLM, tot, 0);
                Eb = __shfl_sync(FULLM, tot, 16);
            }

            // ---- pack the two frames into one complex sequence and transform: pass 1 (lane = n2, R points over n1)
            float sa, isa, sb, isb;
            frame_scale(Ea, inv_a2n, sa, isa);
            frame_scale(Eb, inv_a2n, sb, isb);
            bool a_flat, b_flat;        // every sample equals the frame's first one: the spectrum is exactly zero beyond DC
            {
                float2 z[R];
                const float2 s2 = make_float2(sa, sb), o2 = make_float2(-u0a * sa, -u0b * sb);
                float2 zz = make_float2(0.f, 0.f);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    z[r] = __ffma2_rn(uab[r], s2, o2);
                    zz = __ffma2_rn(z[r], z[r], zz);
                }
                // A constant frame must come out as exact zeros (the reference's float64 spectrum is ~1e-17 there, and
                // log10(. + eps) makes that visible): its partner would otherwise leak ~1e-7 of its own level into it
                a_flat = !__any_sync(FULLM, zz.x > 0.f);
                b_flat = !__any_sync(FULLM, zz.y > 0.f);
                fft_r<R>(z);
                rowa[t_re] = z[0].x; rowa[t_im] = z[0].y;
#pragma unroll
                for (int k1 = 1; k1 < R; ++k1) {
                    const float2 w = cmul(z[k1], cm_.tw[k1 * 32 + lane]);
                    rowa[k1 * LS + t_re] = w.x; rowa[k1 * LS + t_im] = w.y;
                }
            }
            __syncwarp();
            // ---- pass 2 (lane = k1, 32 points over n2, even / odd n2 side by side in FP32x2) -> Z[k1 + R k2] in natural order
            {
                float2 v[32];
                {
                    float2 re[16], im[16];
                    const int row = lane < R ? lane : 0;
                    const float4 *pq = reinterpret_cast<const float4 *>(rowa + row * LS);
#pragma unroll
                    for (int m = 0; m < 16; ++m) {
                        const float4 t = pq[m];
                        const float2 lo = make_float2(t.x, t.y), hi = make_float2(t.z, t.w);
                        re[m] = m < 8 ? lo : hi;
                        im[m] = m < 8 ? hi : lo;
                    }
                    fft32_soa(re, im, v);
                }
                __syncwarp();
                if (lane < R) {
#pragma unroll
                    for (int k2 = 0; k2 < 32; ++k2) wm.tz[lane + R * k2] = v[k2];
                    if (lane == 0) wm.tz[N] = v[0];
                }
            }
            __syncwarp();
            // ---- separate the two spectra: bins k = lane + 32 j
            float xa[C], xb[C];
            {
                const float fa = a_flat ? 0.f : fscale * isa, fb = b_flat ? 0.f : fscale * isb;
#pragma unroll
                for (int j = 0; j < C; ++j) {
                    const int k = lane + 32 * j;
                    xa[j] = 0.f; xb[j] = 0.f;
                    if (j < JK && k < K) {
                        const float2 zk = wm.tz[k], pk = wm.tz[N - k];
                        // Z + conj P = (zx + px, zy - py), Z - conj P = (zx - px, zy + py): one packed sum, one packed difference
                        const float2 sm_ = f2add(zk, pk), df_ = f2sub(zk, pk);
                        xa[j] = fsqrt_fast(fmaf(sm_.x, sm_.x, df_.y * df_.y)) * fa;
                        xb[j] = fsqrt_fast(fmaf(df_.x, df_.x, sm_.y * sm_.y)) * fb;
                    }
                }
                if (lane == 0) {
                    // DC: a sum(x - x0) + N (a (x0 - m) + bp), over K
                    const float2 z0 = wm.tz[0];
                    xa[0] = fabsf(fmaf(nm.a * isa, z0.x, float(N) * fmaf(nm.a, u0a - cmv, nm.bp))) / float(K);
                    xb[0] = fabsf(fmaf(nm.a * isb, z0.y, float(N) * fmaf(nm.a, u0b - cmv, nm.bp))) / float(K);
                }
            }
            __syncwarp();                    // every lane has read Z: the buffer becomes the |X| row of frame a
            float *const rowbn = rowa + S::RB0;
#pragma unroll
            for (int j = 0; j < C; ++j) { rowa[lane + 32 * j] = xa[j]; rowbn[lane + 32 * j] = xb[j]; }
            if (pp.dbg) {
#pragma unroll
                for (int j = 0; j < JK; ++j) {
                    const int k = lane + 32 * j;
                    if (k < K) {
                        pp.dbg[(size_t(b) * p.t_stride + ta) * K + k] = xa[j];
                        if (bvalid) pp.dbg[(size_t(b) * p.t_stride + ta + 1) * K + k] = xb[j];
                    }
                }
            }
            __syncwarp();
            // ---- spectral rows, mel / chroma / DCT: half-warp per frame over the two |X| rows
            rows_to_features<K>(rowa, rowbn, fresh ? rowa : wm.rowp, fresh, wm.fv[(ra - 1) * kFvStride + 34], cm_.dlane,
                                rowa + S::PT0, msraw, mslog, mfold, rowa + S::CH0, fva, fvb, ftab, lane);
            // frame b's row outlives the next transform beside the buffer (rows_to_features ends with a __syncwarp);
            // 16 bytes per lane and instruction: both rows are 16-byte aligned and Kp is a multiple of 32
#pragma unroll
            for (int j = 0; j < (Kp / 4 + 31) / 32; ++j) {
                const int i4 = lane + 32 * j;
                if (i4 < Kp / 4) reinterpret_cast<float4 *>(wm.rowp)[i4] = reinterpret_cast<const float4 *>(rowbn)[i4];
            }

            // ---- tile bookkeeping: full tiles leave at once, a partial one when the run ends
            if (store) {
                tile_n += bvalid ? 2 : 1;
                if (tile_n == 8) B200AA_PAIR_FLUSH(cb);
            }
            fresh = false;
            __syncwarp();                    // the copy above has read the buffer before the next step's pass 1 overwrites it
        }
        if (q1 < NP) run_q = unsigned(q1);
        else B200AA_PAIR_FLUSH(cb);          // end of the clip (an odd frame count leaves a partial tile)
        }
    }
    B200AA_PAIR_FLUSH(run_b);
#undef B200AA_PAIR_FLUSH
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
inline int pair_r_for_window(int window)
{
    switch (window) {
    case 320: return 10;
    case 480: return 15;
    case 512: return 16;
    case 640: return 20;
    case 800: return 25;
    case 960: return 30;
    case 1024: return 32;
    default: return 0;
    }
}

struct PairTables {
    float2 *d_tw = nullptr;
    int *d_pblob = nullptr;
    PairBlobLayout pbl{};
    int R = 0;
    void release()
    {
        if (d_tw) cudaFree(d_tw);
        if (d_pblob) cudaFree(d_pblob);
        d_tw = nullptr; d_pblob = nullptr;
    }
};

// Pair-kernel tables from the dense host tables (mel [40 x K], chroma [12 x K], dct [13 x 40], all float64):
//   mel: every filter is cut into groups of four consecutive taps (zero padded); whole filters are dealt to 16 lanes
//        (longest first, to the least loaded lane) and every lane walks its list in LQ steps, flushing a filter's sum
//        at the filter's last group;   chroma: per pitch class a list of (bin, weight) taps padded to CT entries.
inline void build_pair_blob(const std::vector<double> &mel, const std::vector<double> &chr, const std::vector<double> &dct, int K,
                            std::vector<int> &blob, PairBlobLayout &bl)
{
    struct Quad { int start, fid, last; float w[4]; };
    std::vector<std::vector<Quad>> per_filter(B200AA_N_MEL);
    for (int i = 0; i < B200AA_N_MEL; ++i) {
        int lo = -1, hi = -1;
        if (!mel.empty())
            for (int k = 0; k < K; ++k)
                if (mel[size_t(i) * K + k] != 0.0) { if (lo < 0) lo = k; hi = k; }
        if (lo < 0) { lo = 0; hi = -1; }                       // empty filter: one all-zero group (its log is log10(eps))
        const int nq = hi >= lo ? (hi - lo + 4) / 4 : 1;
        for (int q = 0; q < nq; ++q) {
            Quad qd{};
            const int s = lo + 4 * q;
            int s2 = s;
            if (s2 + 4 > K) s2 = K - 4 > 0 ? K - 4 : 0;        // keep the four reads inside the row
            qd.start = s2; qd.fid = i; qd.last = q == nq - 1;
            for (int j = 0; j < 4; ++j) {
                const int k = s2 + j;
                qd.w[j] = (k >= s && k < s + 4 && k <= hi && k < K) ? float(mel[size_t(i) * K + k]) : 0.f;
            }
            per_filter[i].push_back(qd);
        }
    }
    std::vector<int> order(B200AA_N_MEL);
    for (int i = 0; i < B200AA_N_MEL; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return per_filter[a].size() > per_filter[b].size(); });
    std::vector<std::vector<Quad>> lanes(16);
    for (int i : order) {
        int best = 0;
        for (int l = 1; l < 16; ++l) if (lanes[l].size() < lanes[best].size()) best = l;
        lanes[best].insert(lanes[best].end(), per_filter[i].begin(), per_filter[i].end());
    }
    size_t lq = 1;
    for (auto &l : lanes) lq = l.size() > lq ? l.size() : lq;
    // chroma taps
    std::vector<std::vector<std::pair<int, float>>> taps(12);
    size_t ct = 1;
    if (!chr.empty())
        for (int c = 0; c < 12; ++c) {
            for (int k = 0; k < K; ++k)
                if (chr[size_t(c) * K + k] != 0.0) taps[c].push_back({k, float(chr[size_t(c) * K + k])});
            ct = taps[c].size() > ct ? taps[c].size() : ct;
        }
    auto fbits = [](float f) { int w; std::memcpy(&w, &f, 4); return w; };
    blob.clear();
    bl.dct = 0;
    blob.resize(13 * 41 + 3, 0);
    for (int r = 0; r < 13; ++r)
        for (int n = 0; n < 40; ++n) blob[r * 41 + n] = fbits(float(dct[size_t(r) * 40 + n]));
    while (blob.size() % 4) blob.push_back(0);
    bl.mel_rec = (int)blob.size();
    for (size_t q = 0; q < lq; ++q)
        for (int l = 0; l < 16; ++l) {
            int rec = 0;                                        // padding step: bin 0, zero weights, no flush
            if (q < lanes[l].size()) rec = lanes[l][q].start | (lanes[l][q].fid << 16) | (lanes[l][q].last << 24);
            blob.push_back(rec);
        }
    bl.mel_w = (int)blob.size();                                // multiple of 4 words: 16-byte aligned
    for (size_t q = 0; q < lq; ++q)
        for (int l = 0; l < 16; ++l)
            for (int j = 0; j < 4; ++j) blob.push_back(q < lanes[l].size() ? fbits(lanes[l][q].w[j]) : 0);
    bl.chr = (int)blob.size();                                  // 8-byte aligned
    for (size_t t = 0; t < ct; ++t)
        for (int l = 0; l < 16; ++l) {
            const bool have = l < 12 && t < taps[l].size();
            blob.push_back(have ? taps[l][t].first : 0);
            blob.push_back(have ? fbits(taps[l][t].second) : 0);
        }
    while (blob.size() % 4) blob.push_back(0);
    bl.lq = (int)lq; bl.ct = (int)ct;
    bl.words = (int)blob.size();
}

inline int pair_plan_init(int window, const std::vector<int> &h_pblob, const PairBlobLayout &pbl, PairTables *pt)
{
    const int R = pair_r_for_window(window);
    pt->R = 0;
    if (!R) return B200AA_OK;
    if (getenv("B200AA_NO_PAIR")) return B200AA_OK;
    const int N = 32 * R;
    const double pi = 3.14159265358979323846264338327950288;
    std::vector<float2> tw(size_t(R) * 32);
    for (int k1 = 0; k1 < R; ++k1)
        for (int n2 = 0; n2 < 32; ++n2) {
            const double a = -2.0 * pi * double((k1 * n2) % N) / double(N);
            tw[size_t(k1) * 32 + n2] = make_float2(float(std::cos(a)), float(std::sin(a)));
        }
    if (cudaMalloc(&pt->d_tw, tw.size() * sizeof(float2)) != cudaSuccess) return B200AA_ERR_CUDA;
    if (cudaMemcpy(pt->d_tw, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess) return B200AA_ERR_CUDA;
    if (cudaMalloc(&pt->d_pblob, h_pblob.size() * sizeof(int)) != cudaSuccess) return B200AA_ERR_CUDA;
    if (cudaMemcpy(pt->d_pblob, h_pblob.data(), h_pblob.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) return B200AA_ERR_CUDA;
    pt->pbl = pbl;
    pt->R = R;
    return B200AA_OK;
}

#ifndef B200AA_LAYOUT_ONLY
template <int R, bool SHARED>
inline int pair_launch_t(const PairTables &pt, const StParams &p, int sm_count, int64_t T, unsigned long long *ranges, size_t ranges_cap,
                         float *dbg, cudaStream_t st)
{
    const size_t smem = pair_smem_bytes<R>(pt.pbl.words);
    if (smem > size_t(kPairCtaCap)) return B200AA_ERR_UNSUPPORTED;
    auto kern = st_pair_kernel<R, SHARED>;
    // always the cap, so concurrent launches of one instantiation cannot undercut each other
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kPairCtaCap) != cudaSuccess) return B200AA_ERR_CUDA;
    int occ = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 32 * pair_warps<R>(), smem) != cudaSuccess) return B200AA_ERR_CUDA;
    occ = occ < 1 ? 1 : occ;
    PairParams pp;
    pp.st = p;
    pp.tw = pt.d_tw;
    pp.pblob = pt.d_pblob;
    pp.pbl = pt.pbl;
    pp.dbg = dbg;
    const int64_t NP = (T + 1) / 2;                                  // pairs per (full-length) clip
    constexpr int kPairWarps = pair_warps<R>();
    const int64_t total = NP * p.n_clips;
    if (total <= 0) return B200AA_OK;                                // no clip has a frame
    if (total >= (int64_t(1) << 31)) return B200AA_ERR_UNSUPPORTED;
    // every resident warp gets an equal contiguous share (sched.cuh); small launches use as many warps as they have pairs
    int64_t grid = int64_t(sm_count) * occ;
    if (grid * kPairWarps > total) grid = (total + kPairWarps - 1) / kPairWarps;
    const int64_t n_warps = grid * kPairWarps;
    if (size_t(n_warps) * sizeof(unsigned long long) > ranges_cap) return B200AA_ERR_UNSUPPORTED;
    long chunk = 8, min_steal = 2;
    if (const char *ov = getenv("B200AA_PAIR_STEAL")) {              // tuning override: "chunk,min_steal"
        long a = 0, b2 = 0;
        if (sscanf(ov, "%ld,%ld", &a, &b2) == 2 && a > 0 && a <= 65536 && b2 > 1 && b2 <= 65536) { chunk = a; min_steal = b2; }
    }
    pp.sched.ranges = ranges;
    pp.sched.n_warps = unsigned(n_warps);
    pp.sched.total = unsigned(total);
    pp.sched.per_clip = unsigned(NP);
    pp.sched.chunk = unsigned(chunk);
    pp.sched.min_steal = unsigned(min_steal);
    pp.st.n_items = total;
    if (getenv("B200AA_DEBUG"))
        fprintf(stderr, "[b200aa] pair kernel R=%d shared=%d: smem %zu B, %d CTAs/SM x %d warps, grid %lld, %lld pairs (%lld per clip), chunk %ld, min steal %ld\n",
                R, int(SHARED), smem, occ, kPairWarps, (long long)grid, (long long)total, (long long)NP, chunk, min_steal);
    if (cudaMemsetAsync(ranges, 0, size_t(n_warps) * sizeof(unsigned long long), st) != cudaSuccess) return B200AA_ERR_CUDA;
    kern<<<(unsigned)grid, 32 * kPairWarps, smem, st>>>(pp);
    return cudaPeekAtLastError() == cudaSuccess ? B200AA_OK : B200AA_ERR_CUDA;
}

template <int R>
inline int pair_launch_r(const PairTables &pt, const StParams &p, int sm_count, int64_t T, unsigned long long *ranges, size_t ranges_cap,
                         float *dbg, cudaStream_t st)
{
    constexpr int N = 32 * R;
    if (PairShape<R>::kShareable && p.step == N / 2) return pair_launch_t<R, PairShape<R>::kShareable>(pt, p, sm_count, T, ranges, ranges_cap, dbg, st);
    return pair_launch_t<R, false>(pt, p, sm_count, T, ranges, ranges_cap, dbg, st);
}

// feature launch through the pair kernel; B200AA_ERR_UNSUPPORTED = let another kernel take it
inline int pair_launch_features(const PairTables &pt, const StParams &p, int sm_count, int64_t T, unsigned long long *ranges, size_t ranges_cap,
                                float *dbg, cudaStream_t st)
{
    // 2-byte (int16) / 4-byte (float) loads need nothing beyond natural alignment; frames must fit 32-bit indices
    switch (pt.R) {
    case 10: return pair_launch_r<10>(pt, p, sm_count, T, ranges, ranges_cap, dbg, st);
    case 15: return pair_launch_r<15>(pt, p, sm_count, T, ranges, ranges_cap, dbg, st);
    case 16: return pair_launch_r<16>(pt, p, sm_count, T, ranges, ranges_cap, dbg, st);
    case 32: return pair_launch_r<32>(pt, p, sm_count, T, ranges, ranges_cap, dbg, st);
    case 20: return pair_launch_r<20>(pt, p, sm_count, T, ranges, ranges_cap, dbg, st);
    case 25: return pair_launch_r<25>(pt, p, sm_count, T, ranges, ranges_cap, dbg, st);
    case 30: return pair_launch_r<30>(pt, p, sm_count, T, ranges, ranges_cap, dbg, st);
    default: return B200AA_ERR_UNSUPPORTED;
    }
}
#endif  // B200AA_LAYOUT_ONLY

}  // namespace b200aa
