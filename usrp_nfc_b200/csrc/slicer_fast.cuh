// slicer_fast.cuh -- the streaming slicer kernel (included by slicer.cu after exact_tile).
//
// Same contract as slicer_kernel (transition_sink.py:55-82 over one time segment per CTA, ring in shared
// memory), built for instruction count: per sample everything is float32 (eleven instructions, inline PTX with
// packed f32x2 adds and three-input min), the window sum is carried as a rigorous interval, and exact
// arithmetic is only done where a decision needs it.  Output is fixed-rate: two bits per sample (val != -1,
// val == 1) into a bitmap; extract.cu turns the bitmap into the ordered transition list in a data-parallel pass.
//
//  * A tile is NW*R chunks of 128 samples; warp w owns chunks [w*R, (w+1)*R) = R*128 contiguous samples, lane l
//    the samples 4l..4l+3 of each chunk (one 128-bit load, one 128-bit ring read, one 128-bit ring write).
//  * Per chunk the thresholds ss*lo/L and ss*hi/L are *guessed* (from the carried window sum and the previous
//    tile's drift) and every sample is classified by the guess.  The warp reduces (REDUX) per chunk: the
//    fixed-point sums of the admitted x - prev and |x - prev|, and the margins min |x - guess| to both guesses.
//  * After the first block barrier warp 0 scans the 32 chunk records (lane = chunk): the prefix of the sums gives
//    the window sum each chunk really saw (as an interval), hence the band the true thresholds lie in; the guess
//    is *proven* for a chunk when that band lies strictly inside (guess - margin, guess + margin): no sample is
//    between a guess and any value the true threshold can take.  Otherwise the tile is repeated once with the
//    measured thresholds as the guess; if a sample really sits inside the band, or a HIGH sample follows a LOW
//    sample closely enough for the hysteresis to matter, the tile is handed to exact_tile.  Warp 0 also prepares
//    the next tile's guesses; a second barrier publishes verdict and guesses.
//  * The window sum is carried as [ss_lo, ss_hi]: float rounding and fixed-point conversion errors are bounded
//    and added to the interval.  Where the exact value is needed (exact_tile, state snapshots, segment end) it
//    is recomputed as the sum of the ring in double (exact inside the audited exponent span, see slicer.cu).
#pragma once
#include <cstddef>

namespace nfc {

struct __align__(16) FastRec {  // one chunk of 128 samples
    int S;          // round(sum of admitted (x - prev) / q)
    int A;          // >= sum of admitted |x - prev| / q
    float mL, mH;   // cheap pass: min |x - guessed LOW threshold|, min |x - guessed HIGH threshold| (NaN: a sample is NaN, or
                    // a lane's sum does not fit the fixed point); precise pass: mL = smallest slack of any lane, in ss units
};
enum { FV_ACCEPT = 0, FV_REDO = 1, FV_SLOW = 2, FV_REDO_COARSE = 3, FV_VERIFY = 4 };
enum { FS_FAST = 0, FS_SLOW, FS_BAD, FS_UNC, FS_RESUM, FS_REDO, FS_ST2, FS_VER, FS_PIPE_T, FS_PIPE_IN, FS_PIPE_AB, FS_N };

static const int FAST_CH = 128;  // samples per chunk

__device__ __forceinline__ float redux_min_nan(float v) {
    float r;
    asm volatile("redux.sync.min.NaN.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float fmin_nan(float a, float b) {
    float r;
    asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ float redux_min(float v) {
    float r;
    asm volatile("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}

// Two samples of transition_sink.py:59-82 against guessed thresholds TL < TH (nTL2 / nTH2: {-TL,-TL}, {-TH,-TH}).
// NL / H: ballots of "not LOW" / "HIGH"; n: what the ring slot holds afterwards; s2: two running sums of n - prev
// (0 when not admitted), a: running sum of |n - prev|; mL / mH: running min of |x - TL| / |x - TH|, NaN-propagating.
__device__ __forceinline__ void classify_pair(float x0, float x1, float p0, float p1, float TL, float TH, unsigned long long nTL2,
                                              unsigned long long nTH2, float &mL, float &mH, unsigned long long &s2, float &a,
                                              unsigned &NL0, unsigned &NL1, unsigned &H0, unsigned &H1, float &n0, float &n1) {
    asm volatile(
        "{\n\t"
        ".reg .pred pnl0, ph0, pa0, pnl1, ph1, pa1;\n\t"
        ".reg .b64 xx, uu, vv, dd;\n\t"
        ".reg .f32 u0, u1, v0, v1, d0, d1;\n\t"
        "mov.b64 xx, {%10, %11};\n\t"
        "add.rn.f32x2 uu, xx, %16;\n\t"
        "add.rn.f32x2 vv, xx, %17;\n\t"
        "mov.b64 {u0, u1}, uu;\n\t"
        "mov.b64 {v0, v1}, vv;\n\t"
        "abs.f32 u0, u0;\n\t abs.f32 u1, u1;\n\t abs.f32 v0, v0;\n\t abs.f32 v1, v1;\n\t"
        "min.NaN.f32 %0, %0, u0, u1;\n\t"
        "min.NaN.f32 %1, %1, v0, v1;\n\t"
        "setp.gt.f32 pnl0, %10, %14;\n\t"
        "setp.gt.and.f32 ph0|pa0, %10, %15, pnl0;\n\t"  // ph: HIGH; pa: not LOW and not HIGH = admitted
        "vote.sync.ballot.b32 %4, pnl0, 0xffffffff;\n\t"
        "vote.sync.ballot.b32 %6, ph0, 0xffffffff;\n\t"
        "selp.f32 %8, %10, %12, pa0;\n\t"
        "setp.gt.f32 pnl1, %11, %14;\n\t"
        "setp.gt.and.f32 ph1|pa1, %11, %15, pnl1;\n\t"
        "vote.sync.ballot.b32 %5, pnl1, 0xffffffff;\n\t"
        "vote.sync.ballot.b32 %7, ph1, 0xffffffff;\n\t"
        "selp.f32 %9, %11, %13, pa1;\n\t"
        "sub.f32 d0, %8, %12;\n\t"
        "sub.f32 d1, %9, %13;\n\t"
        "mov.b64 dd, {d0, d1};\n\t"
        "add.rn.f32x2 %2, %2, dd;\n\t"
        "abs.f32 d0, d0;\n\t abs.f32 d1, d1;\n\t"
        "add.f32 %3, %3, d0;\n\t"
        "add.f32 %3, %3, d1;\n\t"
        "}"
        : "+f"(mL), "+f"(mH), "+l"(s2), "+f"(a), "=r"(NL0), "=r"(NL1), "=r"(H0), "=r"(H1), "=f"(n0), "=f"(n1)
        : "f"(x0), "f"(x1), "f"(p0), "f"(p1), "f"(TL), "f"(TH), "l"(nTL2), "l"(nTH2));
}

// block-uniform state of the streaming path, written by warps 0 and 1 (and thread 0), read by everyone after a barrier
struct __align__(16) FastUni {
    float q, invq, invqA, hwf;        // fixed-point step of the coming tile, half width of its ss interval (float, rounded up)
    float TLb, THb, tot_prev, a_est;  // thresholds at the interval's midpoint; last tile's drift; expected sum |x - prev| per tile
    double ss_lo, ss_hi;              // the window sum at the start of the coming tile lies in [ss_lo, ss_hi]
    float thr_min, thr_max;           // admitted samples of streamed tiles lie strictly between these
    int ok;                           // the coming tile may be streamed (ss > 0, step representable)
    int verdict;                      // warp 0: what the sums say
    int st2, cand_last_val, cand_newL, cand_newS;  // warp 1: hysteresis risk; the carries the tile would leave
    unsigned redo_mask;               // repeat: the chunks classified again, sample by sample (bit = chunk)
    int pad_[3];
    float gTL[32], gTH[32];           // guessed thresholds per chunk of the coming tile (or of the repeat), at the chunk's middle
    float gMid[32];                   // the guessed ss behind them (relative to the interval's midpoint)
    float gC0[32];                    // repeat: the measured ss at the chunk's first sample (relative to the midpoint) the guess assumes
    unsigned stats[FS_N];
};
static_assert(offsetof(FastUni, gTL) % 16 == 0 && offsetof(FastUni, gTH) % 16 == 0 && offsetof(FastUni, gMid) % 16 == 0 &&
                  offsetof(FastUni, gC0) % 16 == 0,
              "guess arrays are read with 128-bit loads");

// per-segment constants
struct __align__(16) FastPlan {
    int64_t tile0_pos;                // stream position of the first tile
    const char *xbase;                // input item of that position
    uint32_t *bm_base;                // bitmap word of that position's chunk
    int ntiles, t_int_lo, t_int_hi, t_strad, t_emit;  // tile indices relative to the first: see below
    int t_snap[4];                    // tiles before which a state snapshot is due (seam, three checkpoints), or -1
    int nb;                           // chunks a LOW sample can reach forward through the hysteresis
    float loLf, hiLf;
    float invLo, invHi;               // slightly less than 1 / loLf, 1 / hiLf
};

template <int NT, int R>
struct FastShared {
    static const int NW = NT / 32;
    static const int NC = NW * R;
    FastRec recs[32];
    uint32_t bm[NC * 8];  // the tile's bitmap words, chunk-major
    FastUni uni;
    FastPlan plan;
    double red[NW];
    double vtot[32];  // exact verification: sum of the admitted steps of each chunk
};

// The hysteresis of transition_sink.py:67-73 matters only where a HIGH sample comes within max_len + 1 samples after a LOW
// sample (cur_state == 2 holds it back: val != class there).  Lane = chunk of 128 samples of a tile (nl / hh: its "not LOW" /
// "HIGH" words; lanes beyond the tile hold no LOW and no HIGH sample); relC: the last LOW sample before the tile, relative
// to the tile's first sample (very negative: none in reach).  Exact to the sample for the first HIGH sample of a chunk
// against the nearest LOW sample before it; a chunk with a LOW sample behind its first HIGH sample counts as a risk.
__device__ __forceinline__ bool hysteresis_risk(const uint4 &nl, const uint4 &hh, bool hasL, bool hasH, int lane, int mx, int relC) {
    const unsigned NLw[4] = {nl.x, nl.y, nl.z, nl.w}, Hw[4] = {hh.x, hh.y, hh.z, hh.w};
    int firstH = 1 << 20, lastLany = -1;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        if (Hw[j]) firstH = min(firstH, ((__ffs(Hw[j]) - 1) << 2) | j);
        const unsigned lw = ~NLw[j];
        if (lw) lastLany = max(lastLany, ((31 - __clz(lw)) << 2) | j);
    }
    // the last LOW sample of the chunks before this one (or before the tile)
    int v = hasL ? lane * FAST_CH + lastLany : -(1 << 29);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(FULL, v, o);
        if (lane >= o) v = max(v, u);
    }
    int prevL = __shfl_up_sync(FULL, v, 1);
    if (lane == 0) prevL = -(1 << 29);
    prevL = max(prevL, relC);
    bool risk = false;
    if (hasH) {
        int nearest = prevL;
        if (hasL) {
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int cnt = (firstH - j + 3) >> 2;  // lanes l with 4l + j < firstH
                const unsigned m = cnt >= 32 ? FULL : (cnt <= 0 ? 0u : ((1u << cnt) - 1u));
                const unsigned lw = ~NLw[j] & m;
                if (lw) nearest = max(nearest, lane * FAST_CH + (((31 - __clz(lw)) << 2) | j));
            }
        }
        risk = (lane * FAST_CH + firstH - nearest <= mx + 1) || (hasL && lastLany > firstH);
    }
    return __any_sync(FULL, risk);
}

}  // namespace nfc
#include "slicer_pipe.cuh"
namespace nfc {

__device__ __forceinline__ uint32_t uniform_stats(const FastUni &u, int k) { return u.stats[k] > 0xffffu ? 0xffffu : u.stats[k]; }

// exact window sum = sum of the ring (any order: exact inside the audited exponent span)
template <int NT>
__device__ __noinline__ double ring_sum_exact(const float *ring, int L, double *red) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    cta_sync<NT>();  // all ring writes of earlier tiles have landed
    double part = 0.0;
    for (int i = tid * 4; i < L; i += NT * 4) {
        const float4 v = *reinterpret_cast<const float4 *>(ring + i);
        part += ((double)v.x + (double)v.y) + ((double)v.z + (double)v.w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(FULL, part, o);
    if (lane == 0) red[warp] = part;
    cta_sync<NT>();
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < NT / 32; i++) s += red[i];
    cta_sync<NT>();  // red may be reused
    return s;
}

// warp 0: constants and guessed thresholds of the coming tile from (ss_lo, ss_hi, tot_prev, a_est)
template <int NC>
__device__ __forceinline__ void fast_prepare(FastUni &u, double ss_lo, double ss_hi, float tot_prev, float a_est, double loL, double hiL,
                                             int lane) {
    const double ssm = 0.5 * (ss_lo + ss_hi);
    const float hwf = __double2float_ru(__dsub_ru(ss_hi, ssm)) + __double2float_ru(__dsub_ru(ssm, ss_lo));
    const float ssf = __double2float_rd(ssm);
    bool ok = ss_lo > 0.0 && ssf < 1.0e30f && ssf > 1.0e-30f;
    if (!(a_est > 0.0f)) a_est = ssf * 0x1p-7f;
    const unsigned ae = (__float_as_uint(a_est) >> 23) & 0xffu;  // fixed-point step: a power of two near a_est * 2^-31
    // (smaller tiles: a lane's share of the tile's steps is larger, the step coarser by as much)
    constexpr unsigned QEXP = NC >= 32 ? 30u : (NC >= 16 ? 29u : (NC >= 8 ? 28u : 27u));
    ok = ok && ae > 45u && ae < 250u;
    const float TLb = __double2float_rn(ssm * loL), THb = __double2float_rn(ssm * hiL);
    const float srel = ok ? __fdividef(tot_prev * (1.0f / NC), ssf) : 0.0f;  // predicted relative change of ss per chunk (a guess)
    const float f = fmaf(srel, (float)lane + 0.5f, 1.0f);
    u.gTL[lane] = TLb * f;
    u.gTH[lane] = THb * f;
    u.gMid[lane] = ssf * (f - 1.0f);
    __syncwarp();  // every lane has read the values of `u` its arguments were computed from
    if (lane == 0) {
        const unsigned qe = ok ? ae - QEXP : 127u;
        u.q = __uint_as_float(qe << 23);
        u.invq = __uint_as_float((254u - qe) << 23);
        u.invqA = u.invq * (1.0f + 0x1p-20f);
        u.hwf = hwf;
        u.TLb = TLb;
        u.THb = THb;
        u.tot_prev = tot_prev;
        u.a_est = a_est;
        u.ss_lo = ss_lo;
        u.ss_hi = ss_hi;
        u.ok = ok ? 1 : 0;
    }
}

// One chunk (row r of this warp) of phase 1.  PRECISE: the repeat pass, every sample against its own guessed ss.
template <bool PRECISE>
__device__ __forceinline__ void fast_row(const float4 x4, const float4 pv4, float thL, float thH, float invq, float invqA, float c0g,
                                         float TLb, float THb, float loLf, float hiLf, float invLo, float invHi, int lane, float (&n)[4], FastRec *rec,
                                         uint32_t *bmw) {
    unsigned NLm[4], Hm[4];
    unsigned long long s2 = 0ull;
    float a = 0.0f, mL = INFINITY, mH = INFINITY;
    const unsigned long long nTL2 = pack2(-thL, -thL), nTH2 = pack2(-thH, -thH);
    classify_pair(x4.x, x4.y, pv4.x, pv4.y, thL, thH, nTL2, nTH2, mL, mH, s2, a, NLm[0], NLm[1], Hm[0], Hm[1], n[0], n[1]);
    classify_pair(x4.z, x4.w, pv4.z, pv4.w, thL, thH, nTL2, nTH2, mL, mH, s2, a, NLm[2], NLm[3], Hm[2], Hm[3], n[2], n[3]);
    float sa, sb;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(sa), "=f"(sb) : "l"(s2));
    float ssum = sa + sb;
    if (PRECISE) {
        // steps before each lane under the classes just guessed ...
        float incA = ssum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float v = __shfl_up_sync(FULL, incA, o);
            if (lane >= o) incA += v;
        }
        float Pprev = incA - ssum;
        // ... give every sample its own guessed ss: (chunk start the repeat assumes) + (steps before it).  Classify again,
        // in order inside the lane; the margins are now against per-sample thresholds, in ss units.  The steps before a lane
        // were taken from the classes of the pass before: where samples hover around a threshold many of them change class,
        // and what the lanes' slack has to cover is how far that moved the prefix -- so go round (at most three times) with
        // the prefix of the classes just found until nothing moves any more.
        const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
        const float ps[4] = {pv4.x, pv4.y, pv4.z, pv4.w};
#pragma unroll 1
        for (int it = 0; it < 3; it++) {
            const float base = c0g + Pprev;
            const float tl0 = fmaf(base, loLf, TLb), th0 = fmaf(base, hiLf, THb);
            float run = 0.0f, wmin = INFINITY;
            a = 0.0f;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const float tl = fmaf(run, loLf, tl0), th = fmaf(run, hiLf, th0);
                const bool pnl = xs[j] > tl, ph = xs[j] > th;
                NLm[j] = __ballot_sync(FULL, pnl);
                Hm[j] = __ballot_sync(FULL, ph);
                const float nn = (pnl && !ph) ? xs[j] : ps[j];
                const float d = nn - ps[j];
                n[j] = nn;
                run += d;
                a += fabsf(d);
                wmin = fmin_nan(wmin, fmin_nan(fabsf(xs[j] - tl) * invLo, fabsf(xs[j] - th) * invHi));
            }
            ssum = run;
            float incB = ssum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const float v = __shfl_up_sync(FULL, incB, o);
                if (lane >= o) incB += v;
            }
            const float Pnew = incB - ssum;
            // slack of the lane, in ss units: margin less what this classification moved the steps before it by
            const float moved = fabsf(Pnew - Pprev);
            mL = wmin - moved * 1.001f;
            if (!__any_sync(FULL, moved != 0.0f)) break;  // self-consistent: the thresholds used are the ones these classes give
            Pprev = Pnew;
        }
        mH = INFINITY;
    }
    const float af = a * invqA;
    if (!(af < 33554432.0f)) mL = __int_as_float(0x7fc00000);  // a lane's sum does not fit 2^25 (or is NaN)
    const int si = __float2int_rn(ssum * invq);
    const int ai = __float2int_ru(fminf(af, 33554432.0f));
    const int S = __reduce_add_sync(FULL, si), A = __reduce_add_sync(FULL, ai);
    mL = redux_min_nan(mL);
    if (!PRECISE) mH = redux_min_nan(mH);
    if (lane == 0) {
        *reinterpret_cast<uint4 *>(rec) = make_uint4((unsigned)S, (unsigned)A, __float_as_uint(mL), __float_as_uint(mH));
        uint4 *bw = reinterpret_cast<uint4 *>(bmw);
        bw[0] = make_uint4(NLm[0], NLm[1], NLm[2], NLm[3]);
        bw[1] = make_uint4(Hm[0], Hm[1], Hm[2], Hm[3]);
    }
}

// KIND: InputKind of the segment's samples (compile-time: the load path has no branches).  PIPE: stages of the pipelined
// mode (slicer_pipe.cuh; 0 = synchronous loop only); the CTA then has two more warps than the NT worker threads.
template <int NT, int R, int MINB, int KIND, int PIPE>
__global__ void __launch_bounds__(NT + (PIPE ? 64 : 0), MINB) slicer_fast_kernel(const SegWork *__restrict__ works,
                                                                                 const SlicerParams *__restrict__ params) {
    constexpr int NW = NT / 32;
    constexpr int NC = NW * R;            // chunks per tile
    constexpr int WS = R * FAST_CH;       // samples per warp per tile
    constexpr int T = NW * WS;            // samples per tile
    constexpr int SUB = NT * 4;           // exact_tile row
    constexpr int XR = T / SUB;           // exact_tile rows per tile
    constexpr int ITEM = KIND == IN_IQ_F32 ? 8 : (KIND == IN_PCM_S16 ? 2 : 4);  // IN_SC16: 4 (I, Q int16)
    constexpr int tile_bytes = T * ITEM;
    static_assert(NC <= 32 && NC >= 4, "one lane per chunk record");
    static_assert(T % SUB == 0, "tile is a whole number of exact rows");
    static_assert(R == 4 || R == 2 || R == 1, "bitmap words of a warp are written by its first R * 8 lanes");
    static_assert(NW >= 4, "warps 0 and 1 share the verification, others write the bitmap, another keeps the carries");
    // Small windows (the reference's default: av_window = 2000 at 2 MS/s, transition_sink.py:12) take tiles of 512 samples:
    // four warps, one chunk each; the lanes of the verifying warps beyond the tile's chunks see empty chunks.
    constexpr int BM_FIRST = NW >= 8 ? NW - 4 : 2;  // warps BM_FIRST.. store the tile's bitmap words while warps 0 and 1 judge it
    constexpr int BM_WARPS = NW - BM_FIRST;
    constexpr int CARRY_THREAD = NT >= 256 ? 128 : 96;  // not in warp 0: that one has the longest way to the next barrier already
    extern __shared__ __align__(16) float ring[];
    __shared__ BlockShared<NT> sh;  // exact_tile's scratch
    __shared__ FastShared<NT, R> fs;
    __shared__ SegWork w_s;
    __shared__ SlicerParams p_s;
    __shared__ SegCarry c_s;
    constexpr bool PIPED = PIPE > 0 && KIND != IN_IQ_F32;
    constexpr int NT_ALL = NT + (PIPE ? 64 : 0);
    __shared__ PipeShared<NW, R, (PIPE > 0 ? PIPE : 1)> ps;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (PIPE > 0 && warp >= NW) {
        // judge and mapper of the pipelined mode: parked until the workers enter it (everything they read is set up by then)
        if (PIPED) pipe_aux_main<NW, R, (PIPE > 0 ? PIPE : 1), (KIND == IN_PCM_S16 ? 2 : 4)>(ps, fs.uni, fs.plan, p_s, c_s, ring, warp, lane);
        else pipe_aux_idle<NW>(ps);
        return;
    }
    const long long clk0 = clock64();
    if (threadIdx.x == 0) {
        w_s = works[blockIdx.x];
        p_s = params[w_s.param_idx];
    }
    if (threadIdx.x < FS_N) fs.uni.stats[threadIdx.x] = 0u;
    if (threadIdx.x == 0) ps.inited = 0;
    if (NC < 32 && threadIdx.x >= NC && threadIdx.x < 32) {  // chunks a smaller tile does not have: no steps, no samples near a guess
        FastRec e;
        e.S = 0; e.A = 0; e.mL = INFINITY; e.mH = INFINITY;
        fs.recs[threadIdx.x] = e;
        fs.vtot[threadIdx.x] = 0.0;
    }
    cta_sync<NT>();
    const SegWork &w = w_s;
    const SlicerParams &p = p_s;
    FastUni &uni = fs.uni;
    const FastPlan &plan = fs.plan;
    const int L = p.L;

    // ---- entry state (as slicer_kernel); the carry lives in shared memory (c_s), thread 0 / warps 0 and 1 maintain it
    {
        int emin = 1 << 30, emax = 0;
        if (threadIdx.x == 0) {
            sh.flags[0] = sh.flags[1] = sh.flags[2] = 0u;
            sh.emin = 1 << 30;
            sh.emax = 0;
        }
        double ss0;
        if (w.state_in) {
            const float *src = state_ring(w.state_in);
            for (int i = threadIdx.x; i < L; i += NT) {
                float v = src[i];
                ring[i] = v;
                exp_track(v, emin, emax);
            }
            ss0 = w.state_in->ss;
            cta_sync<NT>();
        } else {
            // Speculative start.  Any state will do (the seam check decides whether the segment stands); the closer to the
            // true one, the sooner it converges.  The true ring holds admitted samples only, so: the previous L samples,
            // with those a settled slicer would not have admitted (pauses, load modulation) replaced by the level of the rest.
            auto block_sum2 = [&](double a, double b, double &ra, double &rb) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    a += __shfl_xor_sync(FULL, a, o);
                    b += __shfl_xor_sync(FULL, b, o);
                }
                cta_sync<NT>();
                if (lane == 0) { sh.red[warp] = a; fs.red[warp] = b; }
                cta_sync<NT>();
                ra = 0.0; rb = 0.0;
                for (int i = 0; i < NW; i++) { ra += sh.red[i]; rb += fs.red[i]; }
            };
            double part = 0.0, cnt = 0.0;
            for (int i = threadIdx.x; i < L; i += NT) {
                const int64_t q = w.warm_begin - L + i;
                float v = load_one<KIND == IN_SC16>(w.in, q - w.in_pos0, p);
                ring[(int)(q % L)] = v;
                part += (double)v;
            }
            double tot, dummy;
            block_sum2(part, 0.0, tot, dummy);
            const float mean0 = (float)(tot / (double)L);
            part = 0.0;
            for (int i = threadIdx.x; i < L; i += NT) {
                const float v = ring[i];
                if (v > 0.5f * mean0 && v < 1.5f * mean0) { part += (double)v; cnt += 1.0; }
            }
            double tsum, tcnt;
            block_sum2(part, cnt, tsum, tcnt);
            const float mean1 = tcnt > 0.0 ? (float)(tsum / tcnt) : mean0;
            const float lo_v = (float)p.lo * mean1, hi_v = (float)p.hi * mean1;
            part = 0.0;
            for (int i = threadIdx.x; i < L; i += NT) {
                float v = ring[i];
                if (!(v >= lo_v && v <= hi_v) && mean1 > 0.0f) v = mean1;
                ring[i] = v;
                part += (double)v;
                exp_track(v, emin, emax);
            }
            block_sum2(part, 0.0, ss0, dummy);
        }
        emin = __reduce_min_sync(FULL, emin);
        emax = __reduce_max_sync(FULL, emax);
        if (lane == 0) { atomicMin(&sh.emin, emin); atomicMax(&sh.emax, emax); }
        if (threadIdx.x == 0) {
            SegCarry c;
            c.ss0 = ss0;
            c.lastL = w.state_in ? w.state_in->lastL : NO_POS;
            c.lrun_start = w.state_in ? w.state_in->lrun_start : NO_POS;
            c.last_val = w.state_in ? w.state_in->last_val : 0;
            c.seg_count = 0; c.scan_buf = 0; c.cnt_buf = 0; c.round_no = 0;
            c_s = c;
            uni.thr_min = 3.0e38f;
            uni.thr_max = 0.0f;
            // ---- the segment in tiles (indices relative to the first one)
            const bool fast_ok = ((L & 3) == 0) && L >= 2 * T && p.lo > 0.0 && p.hi > p.lo && w.bitmap != nullptr;
            FastPlan pl;
            const int64_t tile_first = w.warm_begin / T;
            pl.tile0_pos = tile_first * T;
            pl.xbase = reinterpret_cast<const char *>(w.in) + (pl.tile0_pos - w.in_pos0) * ITEM;
            pl.bm_base = w.bitmap ? w.bitmap + ((pl.tile0_pos - w.bm_pos0) >> 7) * 8 : nullptr;
            pl.ntiles = (w.end > w.warm_begin) ? (int)((w.end - 1) / T - tile_first) + 1 : 0;
            const int64_t lo_pos = max(w.warm_begin, w.in_begin), hi_pos = min(w.end, w.in_end);
            pl.t_int_lo = (int)((lo_pos + T - 1) / T - tile_first);             // first tile that is all inside
            pl.t_int_hi = hi_pos >= 0 ? (int)(hi_pos / T - tile_first) : 0;     // one past the last such tile
            if (!fast_ok) pl.t_int_hi = pl.t_int_lo;
            pl.t_strad = (w.begin % T) ? (int)(w.begin / T - tile_first) : -1;  // tile cut by `begin`
            pl.t_emit = (int)((w.begin + T - 1) / T - tile_first);              // tiles from here on are written
            pl.t_snap[0] = (w.seam_in && w.begin > w.warm_begin && (w.begin % T) == 0) ? (int)(w.begin / T - tile_first) : -1;
            for (int j = 0; j < 3; j++)
                pl.t_snap[j + 1] = (w.ckpt_state[j] && w.ckpt_pos[j] != INT64_MAX && (w.ckpt_pos[j] % T) == 0)
                                       ? (int)(w.ckpt_pos[j] / T - tile_first) : -1;
            pl.nb = (p.mx + FAST_CH) / FAST_CH;
            pl.loLf = (float)p.loL;
            pl.hiLf = (float)p.hiL;
            pl.invLo = (1.0f - 0x1p-20f) / pl.loLf;
            pl.invHi = (1.0f - 0x1p-20f) / pl.hiLf;
            fs.plan = pl;
        }
        if (warp == 0) fast_prepare<NC>(uni, ss0, ss0, 0.0f, -1.0f, p.loL, p.hiL, lane);
    }
    cta_sync<NT>();

    auto next_snap = [&](int after) -> int {
        int best = INT_MAX;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int ts = plan.t_snap[j];
            if (ts > after && ts < best) best = ts;
        }
        return best;
    };
    const int ntiles = plan.ntiles;
    const int64_t tile0_pos = plan.tile0_pos;

    const int slot_step = T % L;
    const int xoff = (warp * WS + lane * 4) * ITEM;  // this thread's first sample inside a tile of the input

    // Samples of the coming tile are copied asynchronously (cp.async) into this thread's four 16-byte slots of a
    // staging buffer behind the ring while the current tile is settled: no registers held, no scoreboard to wait on.
    // IQ input (32 KB per tile) does not fit beside the ring: loaded directly, the coming tile only prefetched into L2.
    constexpr bool STAGED = KIND != IN_IQ_F32;
    char *xbuf = reinterpret_cast<char *>(ring) + (((size_t)L * 4 + 15) / 16) * 16 + (size_t)threadIdx.x * (4 * ITEM);
    float4 xin[R];

    auto request_tile = [&](int t) {  // start the copy of tile t into the staging buffer
        const char *src = plan.xbase + (int64_t)t * tile_bytes + xoff;
        if (STAGED) {
            asm volatile("cp.async.wait_group 0;" ::: "memory");  // an earlier copy into the same slots must have landed
            const unsigned dst = (unsigned)__cvta_generic_to_shared(xbuf);
#pragma unroll
            for (int r = 0; r < R; r++) {
                if (ITEM == 4)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + r * (NT * 16)), "l"(src + r * FAST_CH * 4) : "memory");
                else
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + r * (NT * 8)), "l"(src + r * FAST_CH * 2) : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        } else {
#pragma unroll
            for (int r = 0; r < R; r++) asm volatile("prefetch.global.L2 [%0];" ::"l"(src + r * FAST_CH * ITEM));
#pragma unroll
            for (int r = 0; r < R; r++) asm volatile("prefetch.global.L2 [%0];" ::"l"(src + r * FAST_CH * ITEM + 16));
        }
    };
    auto staged_row = [&](int r) -> float4 {  // row r of the requested tile (after cp.async.wait_group 0), as envelope
        if (KIND == IN_PCM_S16) {
            const float pcm_scale = p.pcm_scale;
            const short4 sv = *reinterpret_cast<const short4 *>(xbuf + r * (NT * 8));
            return make_float4(env_real(__fdiv_rn((float)sv.x, pcm_scale)), env_real(__fdiv_rn((float)sv.y, pcm_scale)),
                               env_real(__fdiv_rn((float)sv.z, pcm_scale)), env_real(__fdiv_rn((float)sv.w, pcm_scale)));
        }
        float4 v = *reinterpret_cast<const float4 *>(xbuf + r * (NT * 16));
        if (KIND == IN_SC16) return env_sc16x4(v, p.pcm_scale);  // the 16 staged bytes are four short2
        if (KIND == IN_REAL_F32) { v.x = env_real(v.x); v.y = env_real(v.y); v.z = env_real(v.z); v.w = env_real(v.w); }
        return v;
    };
    auto load_tile = [&](int t) {
        const char *src = plan.xbase + (int64_t)t * tile_bytes + xoff;
        if (KIND == IN_ENVELOPE_F32 || KIND == IN_REAL_F32) {
#pragma unroll
            for (int r = 0; r < R; r++) xin[r] = ldg_stream4(reinterpret_cast<const float4 *>(src + r * FAST_CH * 4));
            if (KIND == IN_REAL_F32) {
#pragma unroll
                for (int r = 0; r < R; r++) {
                    xin[r].x = env_real(xin[r].x); xin[r].y = env_real(xin[r].y);
                    xin[r].z = env_real(xin[r].z); xin[r].w = env_real(xin[r].w);
                }
            }
        } else if (KIND == IN_IQ_F32) {
#pragma unroll
            for (int r = 0; r < R; r++) {
                const float4 *q = reinterpret_cast<const float4 *>(src + r * FAST_CH * 8);
                const float4 a = ldg_stream4(q), b = ldg_stream4(q + 1);
                xin[r] = make_float4(env_iq(a.x, a.y), env_iq(a.z, a.w), env_iq(b.x, b.y), env_iq(b.z, b.w));
            }
        } else if (KIND == IN_SC16) {
            const float pcm_scale = p.pcm_scale;
#pragma unroll
            for (int r = 0; r < R; r++) xin[r] = env_sc16x4(ldg_stream4(reinterpret_cast<const float4 *>(src + r * FAST_CH * 4)), pcm_scale);
        } else {  // IN_PCM_S16
            const float pcm_scale = p.pcm_scale;
#pragma unroll
            for (int r = 0; r < R; r++) {
                const short4 sv = __ldg(reinterpret_cast<const short4 *>(src + r * FAST_CH * 2));
                xin[r] = make_float4(env_real(__fdiv_rn((float)sv.x, pcm_scale)), env_real(__fdiv_rn((float)sv.y, pcm_scale)),
                                     env_real(__fdiv_rn((float)sv.z, pcm_scale)), env_real(__fdiv_rn((float)sv.w, pcm_scale)));
            }
        }
    };
    auto streamable = [&](int t) { return t >= plan.t_int_lo && t < plan.t_int_hi && t != plan.t_strad; };
    // the exact window sum into c_s.ss0 (and the interval collapsed onto it); ends with a barrier
    auto make_exact = [&]() {
        const double lo = uni.ss_lo, hi = uni.ss_hi;
        double s = lo;
        if (lo != hi) s = ring_sum_exact<NT>(ring, L, fs.red);
        else cta_sync<NT>();
        if (threadIdx.x == 0) {
            if (lo != hi) uni.stats[FS_RESUM]++;
            uni.ss_lo = uni.ss_hi = s;
            c_s.ss0 = s;
        }
        cta_sync<NT>();
    };
    auto snapshot = [&](SlicerHdr *dsth, int64_t pos) {
        make_exact();
        float *dst = state_ring(dsth);
        for (int i = threadIdx.x; i < L; i += NT) dst[i] = ring[i];
        if (threadIdx.x == 0) {
            SlicerHdr h;
            h.ss = c_s.ss0; h.pos = pos; h.lastL = c_s.lastL; h.lrun_start = c_s.lrun_start;
            h.last_val = c_s.last_val; h.emin = 0; h.emax = 0; h.status = 0; h.count = 0; h.pad = 0;
            *dsth = h;
        }
    };

    // phase 2b (warp 1): the class maps of the tile, lane = chunk: hysteresis risk and the carries the tile would leave
    auto maps_phase = [&](int t) {
            uint4 nl = make_uint4(FULL, FULL, FULL, FULL), hh = make_uint4(0u, 0u, 0u, 0u);
            if (NC == 32 || lane < NC) {
                nl = *reinterpret_cast<const uint4 *>(&fs.bm[lane * 8]);
                hh = *reinterpret_cast<const uint4 *>(&fs.bm[lane * 8 + 4]);
            }
            const bool hasL = (nl.x & nl.y & nl.z & nl.w) != FULL, hasH = (hh.x | hh.y | hh.z | hh.w) != 0u;
            const int firstc = (int)((nl.x & 1u) + (hh.x & 1u)), lastc = (int)((nl.w >> 31) + (hh.w >> 31));
            const unsigned Lmask = __ballot_sync(FULL, hasL), Hmask = __ballot_sync(FULL, hasH);
            const int64_t P0 = tile0_pos + (int64_t)t * T;
            // hysteresis can matter only if a HIGH sample comes within max_len + 1 samples after a LOW sample
            bool st2 = false;
            if (Hmask) {
                // cheap test by chunks first; only if it fires, to the sample
                const int nb = plan.nb;
                const int lo_c = max(lane - nb, 0);
                const unsigned win = (Lmask >> lo_c) & ((2u << (lane - lo_c)) - 1u);
                bool risk = hasH && win != 0u;
                const int64_t cl = c_s.lastL;
                if (hasH && cl != NO_POS && P0 + (int64_t)lane * FAST_CH - cl <= (int64_t)p.mx + 1) risk = true;
                if (__any_sync(FULL, risk)) {
                    const int relC = (cl != NO_POS && P0 - cl < (int64_t)(1 << 28)) ? (int)(cl - P0) : -(1 << 29);
                    st2 = hysteresis_risk(nl, hh, hasL, hasH, lane, p.mx, relC);
                }
            }
            // the carries the tile would leave: val of its last sample, last LOW sample and the start of its run
            int newL = -1, newS = -1;
            if (Lmask) {
                int prevlast = __shfl_up_sync(FULL, lastc, 1);
                if (lane == 0) prevlast = c_s.last_val + 1;  // class code of the sample before the tile
                int candL = -1, candS = -1;
                // only chunks whose LOW samples can still matter later: the run continues, or the tile ends soon
                if (hasL && (lastc == 0 || lane >= NC - plan.nb)) {
                    const unsigned NLw[4] = {nl.x, nl.y, nl.z, nl.w};
                    int bestL = -1, bestS = -1;
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const unsigned lw = ~NLw[j];
                        const unsigned pw = j == 0 ? ((NLw[3] << 1) & ~1u) : NLw[j - 1];  // predecessor not LOW
                        const unsigned sw = lw & pw;
                        if (lw) bestL = max(bestL, ((31 - __clz(lw)) << 2) | j);
                        if (sw) bestS = max(bestS, ((31 - __clz(sw)) << 2) | j);
                    }
                    candL = lane * FAST_CH + bestL;
                    if (bestS >= 0) candS = lane * FAST_CH + bestS;
                    if (firstc == 0 && prevlast != 0) candS = max(candS, lane * FAST_CH);  // a LOW run starts at the chunk's first sample
                }
                newL = __reduce_max_sync(FULL, candL);
                newS = __reduce_max_sync(FULL, candS);
            }
            const int lv_new = __shfl_sync(FULL, lastc, NC - 1) - 1;
            if (lane == 0) {
#ifdef NFC_ST2_DEBUG
                if (st2 && blockIdx.x == 312) printf("st2 seg %d tile %d P0 %lld L %08x H %08x lastL %lld\n", blockIdx.x, t, (long long)P0, Lmask, Hmask, (long long)c_s.lastL);
#endif
                uni.st2 = st2 ? 1 : 0;
                uni.cand_last_val = lv_new;
                uni.cand_newL = newL;
                uni.cand_newS = newS;
            }
    };

    // the tile's bitmap words to global memory.  Streamed tiles: by the last four warps while warps 0 and 1 judge the
    // tile (a tile that is repeated or settled another way simply overwrites them).
    auto bitmap_out = [&](int t, int first_warp) {  // between the two barriers of a pass
        if (t >= plan.t_emit) {
            uint32_t *dst = plan.bm_base + (size_t)t * (NC * 8);
            if (NC * 8 == BM_WARPS * 64) {  // two words per lane
                const int i = (warp - first_warp) * 64 + lane;
                dst[i] = fs.bm[i];
                dst[i + 32] = fs.bm[i + 32];
            } else {
                for (int i = (warp - first_warp) * 32 + lane; i < NC * 8; i += BM_WARPS * 32) dst[i] = fs.bm[i];
            }
        }
    };
    // ring update and carries of an accepted tile
    auto commit = [&](const float (&n)[R][4], int t, int slot) {
        int s0 = slot;
#pragma unroll
        for (int r = 0; r < R; r++) {
            *reinterpret_cast<float4 *>(ring + s0) = make_float4(n[r][0], n[r][1], n[r][2], n[r][3]);
            s0 += FAST_CH;
            if (s0 >= L) s0 -= L;
        }
        if (threadIdx.x == CARRY_THREAD) {
            uni.stats[FS_FAST]++;
            c_s.last_val = uni.cand_last_val;
            const int newL = uni.cand_newL, newS = uni.cand_newS;
            if (newL >= 0) {
                const int64_t P0 = tile0_pos + (int64_t)t * T;
                c_s.lastL = P0 + newL;
                if (newS >= 0) c_s.lrun_start = P0 + newS;
            }
        }
    };

    // The tile loop is split in two so that nothing but `t` lives across the rare paths (their calls and double
    // arithmetic would otherwise push the streamed loop's counters into local memory): an inner loop that only
    // streams, and a cold part around it that recomputes what it needs from `t`.
    enum { WHY_NONE = 0, WHY_SNAP, WHY_EXACT, WHY_VERIFY, WHY_PIPE };
    // pipelined mode: the window must span three tiles (ordering of the ring writes, slicer_pipe.cuh), bulk copies need
    // 16-byte aligned tiles; entered when a run of PIPE_MIN tiles can be streamed and the last PIPE_COOL tiles of the
    // synchronous loop were proven at the first attempt (bursts of tiles that need the precise passes stay with it)
    const int PIPE_MIN = g_pipe_tune[0], PIPE_COOL = g_pipe_tune[1];
    const int MEAS_MAX = g_pipe_tune[2];
    const int RESUM_BITS = g_pipe_tune[3];
    const double resum_eps = __longlong_as_double((long long)(1023 - (RESUM_BITS > 0 ? RESUM_BITS : 0)) << 52);  // 2^-RESUM_BITS
     // after a refused tile: sum the ring anew when the interval is wider than 2^-bits of the sum (0: never)  // passes with measured guesses before the exact fix-point takes a tile
    char *const stage0 = reinterpret_cast<char *>(ring) + (((size_t)L * 4 + 15) / 16) * 16;
    const bool pipe_can = PIPED && L >= 3 * T && ((reinterpret_cast<uintptr_t>(plan.xbase) & 15u) == 0u) && plan.bm_base != nullptr;
    int cool = 0, pipe_K = 0;
    long long pipe_cycles = 0;  // diagnostics: cycles spent inside pipelined runs (thread 0)
#ifdef NFC_CYCLES
    long long cyc[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};  // ... [8] after a pipelined run until the loop goes on, [9] loop top until the first pass / run, [10] commits  // tile passes (cycles, calls), ring sums after refused tiles, fix-point path, exact path, repeats (calls), segment set-up, snapshots
    cyc[6] = clock64() - clk0;
#define NFC_CYC(i, expr) do { const long long c0_ = clock64(); expr; cyc[i] += clock64() - c0_; } while (0)
#else
#define NFC_CYC(i, expr) do { expr; } while (0)
#endif
    int t = 0;
    while (t < ntiles) {
#ifdef NFC_CYCLES
        const long long c_top = clock64();
        bool top_open = true;
#endif
        const int t_entry = t;
        {
            bool snap = false;
#pragma unroll
            for (int j = 0; j < 4; j++) snap = snap || (t == plan.t_snap[j]);
            if (snap) {
#ifdef NFC_CYCLES
                const long long c_sn = clock64();
#endif
                if (t == plan.t_snap[0]) snapshot(w.seam_in, w.begin);
                for (int j = 1; j < 4; j++)
                    if (t == plan.t_snap[j]) snapshot(w.ckpt_state[j - 1], tile0_pos + (int64_t)t * T);
                // the interval collapsed: the coming tile's constants follow it
                if (warp == 0) {
                    const double lo = uni.ss_lo, hi = uni.ss_hi;
                    const float tp = uni.tot_prev, ae = uni.a_est;
                    __syncwarp();
                    fast_prepare<NC>(uni, lo, hi, tp, ae, p.loL, p.hiL, lane);
                }
                cta_sync<NT>();
#ifdef NFC_CYCLES
                cyc[7] += clock64() - c_sn;
#endif
            }
        }
        int why = WHY_NONE;
        {
            // ------------------------------------------------------------------------ streamed tiles
            // tiles [t, t_stop) can be streamed back to back: inside the segment, whole, no snapshot due
            int t_stop = min(next_snap(t), min(plan.t_int_hi, ntiles));
            if (plan.t_strad >= t) t_stop = min(t_stop, plan.t_strad);
            if (t < plan.t_int_lo) t_stop = t;
            // this kernel's slot of the thread's first sample of the tile (warp-contiguous layout)
            int slot_w = (int)((tile0_pos + (int64_t)t * T + (int64_t)warp * WS + (int64_t)lane * 4) % L);
            int have_x = 0;  // the tile's samples were requested during the previous tile
            float n[R][4];
            // one pass over tile t: classify against the guesses, sums and margins, verdict.  n_meas / n_coarse: repeats
            // of this tile so far with measured guesses / with a coarser fixed-point step
            auto tile_pass = [&](int x_ready, int n_meas, int n_coarse) -> int {
                int verdict;
                if (STAGED) {
                    if (!x_ready) request_tile(t);
                    asm volatile("cp.async.wait_group 0;" ::: "memory");
                } else {
                    load_tile(t);
                }
                x_ready = 0;
                const float invq = uni.invq, invqA = uni.invqA;
                const bool precise = n_meas > 0;  // a repeated tile is classified sample by sample against the measured sums
                // -------------------------------------------------------- phase 1: classify, sums, margins, maps
                {
                    int s0 = slot_w;
                    FastRec *rec = &fs.recs[warp * R];
                    uint32_t *bmw = &fs.bm[warp * R * 8];
                    if (!precise) {
#pragma unroll
                        for (int r = 0; r < R; r++) {
                            const float4 pv4 = *reinterpret_cast<const float4 *>(ring + s0);
                            fast_row<false>(STAGED ? staged_row(r) : xin[r], pv4, uni.gTL[warp * R + r], uni.gTH[warp * R + r], invq,
                                            invqA, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, lane, n[r], rec + r, bmw + r * 8);
                            s0 += FAST_CH;
                            if (s0 >= L) s0 -= L;
                        }
                    } else {
                        // only the chunks the verdict named: the others keep their records, maps and ring values
                        const float TLb = uni.TLb, THb = uni.THb;
                        const unsigned mine = uni.redo_mask >> (warp * R);
#pragma unroll
                        for (int r = 0; r < R; r++) {
                            if ((mine >> r) & 1u) {
                                const float4 pv4 = *reinterpret_cast<const float4 *>(ring + s0);
                                fast_row<true>(STAGED ? staged_row(r) : xin[r], pv4, uni.gTL[warp * R + r], uni.gTH[warp * R + r], invq,
                                               invqA, uni.gC0[warp * R + r], TLb, THb, plan.loLf, plan.hiLf, plan.invLo, plan.invHi,
                                               lane, n[r], rec + r, bmw + r * 8);
                            }
                            s0 += FAST_CH;
                            if (s0 >= L) s0 -= L;
                        }
                    }
                }
                // next tile's samples on their way while this one is settled -- unless the pipelined mode takes over with the
                // next tile (its own bulk copies fetch it; a copy requested here would only have to be waited for)
                if (t + 1 < t_stop && !(pipe_can && cool <= 1 && t_stop - (t + 1) >= PIPE_MIN)) {
                    request_tile(t + 1);
                    have_x = STAGED ? 1 : 0;
                }
                cta_sync<NT>();

                if (warp == 0) {
                    // ---------------------------------------------------- phase 2a (warp 0): the sums, lane = chunk
                    const uint4 r0 = *reinterpret_cast<const uint4 *>(&fs.recs[lane]);
                    const int S = (int)r0.x, A = (int)r0.y;
                    const float mL = __uint_as_float(r0.z), mH = __uint_as_float(r0.w);
                    const float q = uni.q, hwf = uni.hwf;
                    const float loLf = plan.loLf, hiLf = plan.hiLf;
                    // window sum at each chunk's first sample, relative to the midpoint of the tile's start interval
                    const float Sf = (float)S * q;
                    float inc = Sf;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const float v = __shfl_up_sync(FULL, inc, o);
                        if (lane >= o) inc += v;
                    }
                    const float c0 = inc - Sf;
                    // the tile's totals: exact sum of the chunk sums (they stay below 2^30), upper bound of the |step| sums
                    const long long totS = ((long long)__reduce_add_sync(FULL, S >> 8) << 8) + (long long)__reduce_add_sync(FULL, S & 0xff);
                    const float totA = (float)((unsigned)__reduce_add_sync(FULL, (A >> 6) + 1)) * 64.0f;
                    const bool nanm = !(mL == mL) || !(mH == mH);
                    const bool bad = __any_sync(FULL, nanm);
                    // error of the sums: conversion (half a step per lane and chunk), float rounding (2^-20 of |d|, also covers
                    // the float prefix above)
                    const float Ef = ((float)(16 * NC) + totA * 0x1p-20f) * q * 1.01f;
                    const float slack = (hwf + Ef) * 1.001f;
                    const float gl = uni.gTL[lane], gh = uni.gTH[lane];
                    bool fine;
                    // a repeat: chunks classified sample by sample (the mask of the last verdict) are judged by their lanes'
                    // slack, the others as in the first pass -- with the chunk starts as they are now
                    const bool lane_precise = precise && ((uni.redo_mask >> lane) & 1u);
                    if (lane_precise) {
                        // the lanes' slack must cover what the chunk's start is off the assumed one by, and the interval
                        const float need = (fabsf(c0 - uni.gC0[lane]) + slack) * (1.0f + 0x1p-18f) + uni.TLb * (0x1p-21f / loLf);
                        fine = (mL > need) && (gl > 0.0f);
                    } else {
                        // inside the chunk ss moves within [V, U] of its start: the sums of the negative / positive steps
                        const float U = 0.5f * (float)(A + S) * q, V = -0.5f * (float)(A - S) * q;
                        const float off = c0 - uni.gMid[lane];
                        const float dev = fmaxf(fabsf(off + U + slack), fabsf(off + V - slack));  // |ss - guessed ss| at any sample
                        const float rl = fmaf(dev, loLf, gl * 0x1p-19f), rh = fmaf(dev, hiLf, gh * 0x1p-19f);
                        // the guess is proven when no sample lies between it and any value the true threshold can take
                        fine = (mL > rl) && (mH > rh) && (gl - rl > 0.0f);
                    }
                    const unsigned failing = __ballot_sync(FULL, !fine);
                    const bool all_fine = failing == 0u;
                    if (!all_fine || bad) {
                        // first the failing chunks alone, then (if that does not settle it) every chunk
                        const bool redo = bad ? n_coarse < 3 : n_meas < MEAS_MAX;
                        const unsigned again = n_meas == 0 ? failing : FULL;
                        if (redo && !bad && ((again >> lane) & 1u)) {  // go round again with the measured window sums as the guess
                            const float mid = c0 + 0.5f * Sf;  // measured window sum at the chunk's middle
                            uni.gTL[lane] = fmaf(mid, loLf, uni.TLb);
                            uni.gTH[lane] = fmaf(mid, hiLf, uni.THb);
                            uni.gMid[lane] = mid;
                            uni.gC0[lane] = c0;
                        }
                        __syncwarp();  // every lane has read the step and the mask this pass was judged with
                        if (lane == 0) {
                            uni.redo_mask = again;
                            // a precise pass that cannot prove itself is checked sample by sample in exact arithmetic
                            int v = redo ? (bad ? FV_REDO_COARSE : FV_REDO) : ((precise && !bad) ? FV_VERIFY : FV_SLOW);
                            if (bad && redo) {  // a lane's sum did not fit: coarser fixed-point step
                                const float ae = uni.a_est * 16.0f;
                                const unsigned e = (__float_as_uint(ae) >> 23) & 0xffu;
                                constexpr unsigned QEXP = NC >= 32 ? 30u : (NC >= 16 ? 29u : (NC >= 8 ? 28u : 27u));
                                if (e > 45u && e < 250u) {
                                    uni.a_est = ae;
                                    uni.q = __uint_as_float((e - QEXP) << 23);
                                    uni.invq = __uint_as_float((254u - (e - QEXP)) << 23);
                                    uni.invqA = uni.invq * (1.0f + 0x1p-20f);
                                } else {
                                    v = FV_SLOW;
                                }
                            }
                            uni.verdict = v;
                            uni.stats[v == FV_SLOW ? FS_BAD : (v == FV_VERIFY ? FS_UNC : FS_REDO)]++;
                        }
                    } else {
                        // ---- the window sum after the tile and the coming tile's constants
                        const double delta = (double)totS * (double)q;  // exact
                        const double ss_lo = __dadd_rd(uni.ss_lo, __dadd_rd(delta, -(double)Ef));
                        const double ss_hi = __dadd_ru(uni.ss_hi, __dadd_ru(delta, (double)Ef));
                        const float a_new = fmaxf(fmaxf(totA * q, 0.25f * uni.a_est), uni.TLb * 0x1p-16f);  // follows the traffic, decays slowly
                        // admitted samples lie strictly between the guessed thresholds' surroundings: one binade of slack either way
                        const float tmin = redux_min(gl * 0.5f), tmax = -redux_min(-(gh * 2.0f));
                        if (lane == 0) {
                            uni.verdict = FV_ACCEPT;
                            uni.thr_min = fminf(uni.thr_min, tmin);
                            uni.thr_max = fmaxf(uni.thr_max, tmax);
                        }
                        fast_prepare<NC>(uni, ss_lo, ss_hi, (float)delta, a_new, p.loL, p.hiL, lane);
                    }
                } else if (warp == 1) {
                    maps_phase(t);
                } else if (warp >= BM_FIRST) {
                    bitmap_out(t, BM_FIRST);
                }
                cta_sync<NT>();
                verdict = uni.verdict;
                if (uni.st2 && verdict != FV_SLOW) {
                    verdict = FV_SLOW;
                    if (threadIdx.x == 0) uni.stats[FS_ST2]++;
                }
                return verdict;
            };
            for (;;) {
                if (t >= t_stop || !uni.ok) {
                    bool snap = false;
#pragma unroll
                    for (int j = 0; j < 4; j++) snap = snap || (t == plan.t_snap[j]);
                    why = (snap && t != t_entry) ? WHY_SNAP : WHY_EXACT;
                    break;
                }
                if (pipe_can && cool == 0 && t_stop - t >= PIPE_MIN) {
                    why = WHY_PIPE;
                    pipe_K = t_stop - t;
                    break;
                }
                const int x_ready = have_x;
                have_x = 0;
                int verdict;
#ifdef NFC_CYCLES
                if (top_open) { cyc[9] += clock64() - c_top; top_open = false; }
#endif
                NFC_CYC(0, verdict = tile_pass(x_ready, 0, 0));
#ifdef NFC_CYCLES
                cyc[1]++;
#endif
                if (verdict == FV_ACCEPT) {
                    if (cool > 0) cool--;
                } else {
                    cool = PIPE_COOL;
                }
                if (verdict != FV_ACCEPT) {
                    int n_meas = 0, n_coarse = 0;
                    for (;;) {
                        have_x = 0;  // the samples are needed for this tile again, or the exact path reloads
                        if (verdict == FV_REDO) {
                            n_meas++;
                        } else if (verdict == FV_REDO_COARSE) {  // other fixed-point step: every chunk's sums again
                            n_coarse++;
                            n_meas = 0;
                        } else {
                            break;
                        }
                        NFC_CYC(0, verdict = tile_pass(0, n_meas, n_coarse));
#ifdef NFC_CYCLES
                        cyc[1]++; cyc[5]++;
#endif
                        if (verdict == FV_ACCEPT) break;
                    }
                    if (verdict != FV_ACCEPT) {
                        why = verdict == FV_VERIFY ? WHY_VERIFY : WHY_EXACT;
                        break;
                    }
                }
                NFC_CYC(10, commit(n, t, slot_w));
                slot_w += slot_step;
                if (slot_w >= L) slot_w -= L;
                t++;
            }
        }
        if (t >= ntiles) break;
        if (why == WHY_SNAP) continue;
        if (PIPED && why == WHY_PIPE) {
            // ------------------------------------------------------------------------ pipelined run over tiles [t, t + pipe_K)
            asm volatile("cp.async.wait_group 0;" ::: "memory");  // a tile requested by the synchronous loop is dropped
#ifdef NFC_CYCLES
            if (top_open) { cyc[9] += clock64() - c_top; top_open = false; }
#endif
            const long long clk_p0 = clock64();
            if (threadIdx.x == 0) {
                ps.cmd = PIPE_CMD_ENTER;
                ps.t0 = t;
                ps.K = pipe_K;
                uni.stats[FS_PIPE_IN]++;
            }
            fence_proxy_async();  // the stages were written through the generic proxy so far
            named_bar_sync<PIPE_BAR_PARK, NT_ALL>();  // wakes judge and mapper
            named_bar_sync<PIPE_BAR_RUN, NT_ALL>();   // barriers and first guesses are set up
            const int done = pipe_worker<NW, R, (PIPE > 0 ? PIPE : 1), KIND>(ps, ring, stage0, plan, L, p.pcm_scale, warp, lane);
            named_bar_sync<PIPE_BAR_RUN, NT_ALL>();   // interval and carries are handed back
            if (threadIdx.x == 0) pipe_cycles += clock64() - clk_p0;
#ifdef NFC_CYCLES
            const long long c_post = clock64();
#endif
            t += done;
            if (done < pipe_K) {
                cool = PIPE_COOL > 1 ? PIPE_COOL : 1;  // at least the refused tile goes through the synchronous loop
                if (threadIdx.x == 0) uni.stats[FS_PIPE_AB]++;
                // A refused tile usually holds samples close to a threshold: what the precise pass can prove there is limited
                // by the width of the window sum's interval, which has grown with every streamed tile.  Summing the ring anew
                // (exact) is much cheaper than the exact fix-point a tile that cannot be proven falls back to.
                if (RESUM_BITS > 0) {
                    const double lo = uni.ss_lo, hi = uni.ss_hi;
                    if ((hi - lo) > hi * resum_eps) NFC_CYC(2, make_exact());  // block-uniform
                }
            }
            if (warp == 0) {  // the coming tile's constants for the synchronous loop
                const double lo = uni.ss_lo, hi = uni.ss_hi;
                const float tp = uni.tot_prev, ae = uni.a_est;
                __syncwarp();
                fast_prepare<NC>(uni, lo, hi, tp, ae, p.loL, p.hiL, lane);
            }
#ifdef NFC_CYCLES
            const long long c_bar = clock64();
#endif
            cta_sync<NT>();
#ifdef NFC_CYCLES
            cyc[11] += clock64() - c_bar;
            cyc[8] += clock64() - c_post;
#endif
            continue;
        }

        // ---------------------------------------------------------------------------- tile t the hard way (rare)
        bool done = false;
#ifdef NFC_CYCLES
        const long long c_hard = clock64();
        const int why_hard = why;
#endif
        if (why == WHY_VERIFY) {
            // ---------------------------------------------------------------- exact fix-point from the precise pass
            // Every sample's class is recomputed from its own exact window sum under the current classes, until
            // nothing changes: a self-consistent assignment is the sequential answer (the recurrence is causal).
            const int slot_w = (int)((tile0_pos + (int64_t)t * T + (int64_t)warp * WS + (int64_t)lane * 4) % L);
            make_exact();  // c_s.ss0: the exact window sum at the tile's first sample
            const double ss0 = c_s.ss0;
            load_tile(t);  // the staging buffer already holds the coming tile
            unsigned cls = 0u;  // two bits per sample: 0 LOW, 1 MID, 2 HIGH
#pragma unroll
            for (int r = 0; r < R; r++) {
                const uint4 nl = *reinterpret_cast<const uint4 *>(&fs.bm[(warp * R + r) * 8]);
                const uint4 hh = *reinterpret_cast<const uint4 *>(&fs.bm[(warp * R + r) * 8 + 4]);
                const unsigned nlw[4] = {nl.x, nl.y, nl.z, nl.w}, hw[4] = {hh.x, hh.y, hh.z, hh.w};
#pragma unroll
                for (int j = 0; j < 4; j++) cls |= (((nlw[j] >> lane) & 1u) + ((hw[j] >> lane) & 1u)) << (2 * (r * 4 + j));
            }
            bool settled = false;
            double total = 0.0;
            for (int it = 0; it < 8 && !settled; it++) {
                double lane_ex[R];
                int s0 = slot_w;
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const float4 pv4 = *reinterpret_cast<const float4 *>(ring + s0);
                    const float xs[4] = {xin[r].x, xin[r].y, xin[r].z, xin[r].w};
                    const float ps[4] = {pv4.x, pv4.y, pv4.z, pv4.w};
                    double tot = 0.0;
#pragma unroll
                    for (int j = 0; j < 4; j++)
                        if (((cls >> (2 * (r * 4 + j))) & 3u) == 1u) tot += (double)xs[j] - (double)ps[j];
                    double inc = tot;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const double v = __shfl_up_sync(FULL, inc, o);
                        if (lane >= o) inc += v;
                    }
                    lane_ex[r] = inc - tot;
                    if (lane == 31) fs.vtot[warp * R + r] = inc;
                    s0 += FAST_CH;
                    if (s0 >= L) s0 -= L;
                }
                cta_sync<NT>();
                const double ct = fs.vtot[lane];
                double cinc = ct;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const double v = __shfl_up_sync(FULL, cinc, o);
                    if (lane >= o) cinc += v;
                }
                const double chunk_ex = cinc - ct;
                total = __shfl_sync(FULL, cinc, NC - 1);
                unsigned ncls = 0u;
                s0 = slot_w;
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const float4 pv4 = *reinterpret_cast<const float4 *>(ring + s0);
                    const float xs[4] = {xin[r].x, xin[r].y, xin[r].z, xin[r].w};
                    const float ps[4] = {pv4.x, pv4.y, pv4.z, pv4.w};
                    double ssj = ss0 + __shfl_sync(FULL, chunk_ex, warp * R + r) + lane_ex[r];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        ncls |= (unsigned)(classify(xs[j], ssj, p) + 1) << (2 * (r * 4 + j));
                        if (((cls >> (2 * (r * 4 + j))) & 3u) == 1u) ssj += (double)xs[j] - (double)ps[j];
                    }
                    s0 += FAST_CH;
                    if (s0 >= L) s0 -= L;
                }
                const bool changed = ncls != cls;
                cls = ncls;
                settled = !cta_sync_or<NT>((int)changed);  // also: vtot may be written again
            }
            if (settled) {
                // ---- the tile's outputs from the settled classes
                float n[R][4];
                int s0 = slot_w;
                int emin = 1 << 30, emax = 0;  // the admitted samples enter the exactness audit
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const float4 pv4 = *reinterpret_cast<const float4 *>(ring + s0);
                    const float xs[4] = {xin[r].x, xin[r].y, xin[r].z, xin[r].w};
                    const float ps[4] = {pv4.x, pv4.y, pv4.z, pv4.w};
                    unsigned NLm[4], Hm[4];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const unsigned code = (cls >> (2 * (r * 4 + j))) & 3u;
                        NLm[j] = __ballot_sync(FULL, code != 0u);
                        Hm[j] = __ballot_sync(FULL, code == 2u);
                        n[r][j] = code == 1u ? xs[j] : ps[j];
                        if (code == 1u) exp_track(xs[j], emin, emax);
                    }
                    if (lane == 0) {
                        uint4 *bw = reinterpret_cast<uint4 *>(&fs.bm[(warp * R + r) * 8]);
                        bw[0] = make_uint4(NLm[0], NLm[1], NLm[2], NLm[3]);
                        bw[1] = make_uint4(Hm[0], Hm[1], Hm[2], Hm[3]);
                    }
                    s0 += FAST_CH;
                    if (s0 >= L) s0 -= L;
                }
                emin = __reduce_min_sync(FULL, emin);
                emax = __reduce_max_sync(FULL, emax);
                if (lane == 0) { atomicMin(&sh.emin, emin); atomicMax(&sh.emax, emax); }
                cta_sync<NT>();
                if (warp == 0) {
                    const float ae = uni.a_est;
                    __syncwarp();
                    fast_prepare<NC>(uni, ss0 + total, ss0 + total, (float)total, ae, p.loL, p.hiL, lane);
                } else if (warp == 1) {
                    maps_phase(t);
                }
                cta_sync<NT>();
                if (uni.st2) {  // a HIGH sample the hysteresis may hold back: val is not the class
                    if (threadIdx.x == 0) uni.stats[FS_ST2]++;
                } else {
                    // the words were rewritten from the settled classes: every warp stores its own (no barrier follows
                    // before the next tile's words are written, by lane 0 of the same warp)
                    if (t >= plan.t_emit && lane < R * 8)
                        plan.bm_base[(size_t)t * (NC * 8) + warp * (R * 8) + lane] = fs.bm[warp * (R * 8) + lane];
                    __syncwarp();
                    commit(n, t, slot_w);
                    done = true;
                }
            } else {
                if (threadIdx.x == 0) uni.stats[FS_VER]++;
            }
        }
        if (!done) {
            // ---------------------------------------------------------------- exact path, row by row
            make_exact();
            const double ss_before = c_s.ss0;
            const int64_t P0 = tile0_pos + (int64_t)t * T;
            const int slot_x = (int)((P0 + (int64_t)threadIdx.x * 4) % L);  // exact_tile's slot of this thread's first sample of a row
            cta_sync<NT>();
#pragma unroll 1
            for (int r = 0; r < XR; r++) {
                const int64_t Pr = P0 + (int64_t)r * SUB;
                if (Pr >= w.end || Pr + SUB <= w.warm_begin) continue;  // block-uniform
                int s0 = slot_x + r * SUB;
                while (s0 >= L) s0 -= L;
                exact_tile<NT, 4, true, KIND == IN_SC16>(&w_s, &p_s, ring, &sh, Pr, s0, &c_s);
            }
            if (warp == 0) {
                const double ss1 = c_s.ss0;
                const float ae = uni.a_est;
                __syncwarp();
                if (lane == 0) uni.stats[FS_SLOW]++;
                fast_prepare<NC>(uni, ss1, ss1, (float)(ss1 - ss_before), ae, p.loL, p.hiL, lane);
            }
            cta_sync<NT>();
        }
#ifdef NFC_CYCLES
        cyc[why_hard == WHY_VERIFY ? 3 : 4] += clock64() - c_hard;
#endif
        t++;
    }

    // ---- exit: exactness audit and final state
    if (PIPE > 0) {
        if (threadIdx.x == 0) ps.cmd = PIPE_CMD_QUIT;
        named_bar_sync<PIPE_BAR_PARK, NT_ALL>();
    }
    make_exact();
    if (threadIdx.x == 0 && uni.stats[FS_FAST]) {
        int emin = 1 << 30, emax = 0;
        exp_track(uni.thr_min, emin, emax);
        exp_track(uni.thr_max, emin, emax);
        atomicMin(&sh.emin, emin);
        atomicMax(&sh.emax, emax);
    }
    cta_sync<NT>();
    const int emin = sh.emin, emax = sh.emax;
    int status = SEG_OK;
    if (emax >= 255) status |= SEG_NOT_SANE;
    if (emax > 0 && emax - emin > p.span_limit) status |= SEG_INEXACT;

    if (w.state_out) {
        float *dst = state_ring(w.state_out);
        for (int i = threadIdx.x; i < L; i += NT) dst[i] = ring[i];
        if (threadIdx.x == 0) {
            SlicerHdr h;
            h.ss = c_s.ss0; h.pos = w.end; h.lastL = c_s.lastL; h.lrun_start = c_s.lrun_start;
            h.last_val = c_s.last_val; h.emin = emin; h.emax = emax; h.status = status;
            h.count = (uint32_t)((clock64() - clk0) >> 10);                      // diagnostics: kilocycles this segment took,
            h.pad = (uniform_stats(uni, FS_REDO) << 16) | uniform_stats(uni, FS_SLOW);  // repeated and exact-path tiles
            *w.state_out = h;
        }
    }
    if (threadIdx.x == 0) {
        if (w.trans_count) *w.trans_count = 0;
        if (w.status) *w.status = status;
        atomicAdd(&g_tile_stats[0], (unsigned long long)uni.stats[FS_FAST]);
        atomicAdd(&g_tile_stats[1], (unsigned long long)uni.stats[FS_SLOW]);
        atomicAdd(&g_tile_stats[2], (unsigned long long)uni.stats[FS_BAD]);
        atomicAdd(&g_tile_stats[3], (unsigned long long)uni.stats[FS_UNC]);
        atomicAdd(&g_tile_stats[4], (unsigned long long)uni.stats[FS_RESUM]);
        atomicAdd(&g_tile_stats[5], (unsigned long long)uni.stats[FS_REDO]);
        atomicAdd(&g_tile_stats[6], (unsigned long long)uni.stats[FS_ST2]);
        atomicAdd(&g_tile_stats[7], (unsigned long long)uni.stats[FS_VER]);
        atomicAdd(&g_tile_stats[8], (unsigned long long)c_s.round_no);
        atomicAdd(&g_tile_stats[11], (unsigned long long)uni.stats[FS_PIPE_T]);
        atomicAdd(&g_tile_stats[12], (unsigned long long)uni.stats[FS_PIPE_IN]);
        atomicAdd(&g_tile_stats[13], (unsigned long long)uni.stats[FS_PIPE_AB]);
        atomicAdd(&g_tile_stats[14], (unsigned long long)pipe_cycles);
        atomicAdd(&g_tile_stats[15], (unsigned long long)(clock64() - clk0));
#ifdef NFC_CYCLES
        for (int i = 0; i < 12; i++) atomicAdd(&g_cyc[i], (unsigned long long)cyc[i]);
#endif
    }
}

}  // namespace nfc
