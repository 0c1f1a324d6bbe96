// slicer.cu -- envelope + ratio classification + gated moving average + hysteresis, sm_100a.
//
// Replaces the per-sample loop of transition_sink.work_stable (transition_sink.py:55-82) and the
// envelope blocks in front of it (decoder.py:25-28, usrp_src.py:31).  Output: the positions where
// the slicer's `val` changes (runs.cu turns those into the reference's event list).
//
// Parallel formulation (validated on the CPU by tests/algomodel.py):
//  * One CTA walks one time segment tile by tile (T = NT*K samples).  The window sum obeys
//    ss[i+1] = ss[i] + admit[i] * (x[i] - ring[i mod L]) where admit depends on ss[i] itself.
//    Because the recurrence is causal, ANY self-consistent assignment of classes equals the
//    sequential answer: guess the classes with ss frozen at the tile start, prefix-sum the gated
//    deltas, re-classify every sample with its own exact ss, repeat until nothing changes.
//  * Sums are carried in double.  While every admitted sample lies within `span_limit` binades
//    all partial sums are exactly representable, so the result does not depend on summation order
//    and equals the reference's running `ss += cur - prev`.  The exponent range is tracked; a
//    segment that leaves it is flagged and redone by the strictly sequential kernel below.
//  * The reference's ratio test  RN64(x*L/ss) vs lo/hi  is decided by the sign of one FMA
//    (exact), with the real division only inside a 2^-50 relative band around the threshold.
//  * "ratio > hi is ignored while cur_state == 2" depends on cur_state only through the
//    distance to the last LOW sample (see vals_from_classes in tests/algomodel.py).
//  * Segments other than the first start cold (ring <- previous L samples, like the
//    reference's warm-up) `halo` samples early; the state they reach at their first emitted
//    sample is compared bit for bit with the predecessor's final state (seam_compare_kernel)
//    and the segment is redone from the true state when it differs.
#include <atomic>
#include <map>
#include <mutex>
#include <utility>
#include "common.cuh"
#include <cstdio>
#include <stdlib.h>

namespace nfc {

static const unsigned FULL = 0xffffffffu;
// tile counters (device-wide): 0 streamed, 1 exact path, 2 coarse-step retries exhausted, 3 exact fix-point pass, 4 ring resums,
// 5 repeated passes, 6 hysteresis risk, 7 fix-point pass gave up, 8 exact-path rounds, 11-15 pipelined mode and cycles (slicer_fast.cuh)
__device__ unsigned long long g_tile_stats[16];
#ifdef NFC_CYCLES
__device__ unsigned long long g_cyc[12];  // diagnostics build: see slicer_fast.cuh
#endif
// pipelined mode of the streaming kernel: shortest run worth entering (tiles), tiles the synchronous loop must prove at the
// first attempt before the pipeline is entered again (NFC_PIPE_MIN / NFC_PIPE_COOL set them per process, for experiments)
__device__ int g_pipe_tune[4] = {6, 3, 2, 18};  // NFC_PIPE_MIN, NFC_PIPE_COOL, NFC_MEAS_MAX, NFC_RESUM_BITS (slicer_fast.cuh)
enum { CLS_LOW = -1, CLS_MID = 0, CLS_HIGH = 1 };

// Barrier over the first NT threads of the CTA (named barrier 1).  The streaming kernel's CTAs carry two more warps
// (judge and mapper of the pipelined mode, slicer_pipe.cuh) that take no part in the segment's block-wide steps; for
// kernels whose CTAs have exactly NT threads this is __syncthreads().
template <int NT>
__device__ __forceinline__ void cta_sync() {
    asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");
}
template <int NT>
__device__ __forceinline__ int cta_sync_or(int pred) {
    int r;
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        "setp.ne.s32 p, %1, 0;\n\t"
        "bar.red.or.pred q, 1, %2, p;\n\t"
        "selp.s32 %0, 1, 0, q;\n\t"
        "}"
        : "=r"(r)
        : "r"(pred), "n"(NT)
        : "memory");
    return r;
}

// ---------------------------------------------------------------- sample loading / envelope
__device__ __forceinline__ float env_real(float s) { return __fmul_rn(s, s); }  // float_to_complex + mag^2, im = 0
__device__ __forceinline__ float env_iq(float re, float im) { return __fadd_rn(__fmul_rn(re, re), __fmul_rn(im, im)); }
// complex int16 (UHD's sc16): the IQ envelope of (I / scale, Q / scale), divided as int16 PCM is
__device__ __forceinline__ float env_sc16(short2 s, float scale) {
    return env_iq(__fdiv_rn((float)s.x, scale), __fdiv_rn((float)s.y, scale));
}
// four sc16 items read as one 16-byte vector (any 16-byte type): item j is word j, I in its low half
__device__ __forceinline__ float env_sc16_word(unsigned u, float scale) {
    return env_sc16(make_short2((short)(u & 0xffffu), (short)(u >> 16)), scale);
}
__device__ __forceinline__ float4 env_sc16x4(float4 v, float scale) {
    return make_float4(env_sc16_word(__float_as_uint(v.x), scale), env_sc16_word(__float_as_uint(v.y), scale),
                       env_sc16_word(__float_as_uint(v.z), scale), env_sc16_word(__float_as_uint(v.w), scale));
}

// SC16 = false: code for a kernel that is never launched on sc16 input (the streaming kernel of another kind), which then
// carries no sc16 branch at all
template <bool SC16 = true>
__device__ __forceinline__ float load_one(const void *in, int64_t idx, const SlicerParams &p) {
    if (SC16 && p.input_kind == IN_SC16) return env_sc16(__ldg(reinterpret_cast<const short2 *>(in) + idx), p.pcm_scale);
    switch (p.input_kind) {
        case IN_ENVELOPE_F32: return __ldg(reinterpret_cast<const float *>(in) + idx);
        case IN_REAL_F32: return env_real(__ldg(reinterpret_cast<const float *>(in) + idx));
        case IN_IQ_F32: {
            float2 c = __ldg(reinterpret_cast<const float2 *>(in) + idx);
            return env_iq(c.x, c.y);
        }
        default: {  // IN_PCM_S16
            float s = __fdiv_rn((float)__ldg(reinterpret_cast<const short *>(in) + idx), p.pcm_scale);
            return env_real(s);
        }
    }
}

// streaming 128-bit load: the sample stream is read exactly once
__device__ __forceinline__ float4 ldg_stream4(const float4 *ptr) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(ptr));
    return r;
}

template <int K, bool SC16 = true>
__device__ __forceinline__ void load_samples(const SegWork &w, const SlicerParams &p, int64_t p0, float (&x)[K]) {
    const int64_t i0 = p0 - w.in_pos0;
    if (K == 4 && p0 >= w.in_begin && p0 + 4 <= w.in_end) {
        if (p.input_kind == IN_ENVELOPE_F32 || p.input_kind == IN_REAL_F32) {
            float4 v = ldg_stream4(reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(w.in) + i0));
            x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
            if (p.input_kind == IN_REAL_F32) {
#pragma unroll
                for (int j = 0; j < K; j++) x[j] = env_real(x[j]);
            }
            return;
        }
        if (p.input_kind == IN_IQ_F32) {
            const float4 *q = reinterpret_cast<const float4 *>(reinterpret_cast<const float2 *>(w.in) + i0);
            float4 a = ldg_stream4(q), b = ldg_stream4(q + 1);
            x[0] = env_iq(a.x, a.y); x[1] = env_iq(a.z, a.w); x[2] = env_iq(b.x, b.y); x[3] = env_iq(b.z, b.w);
            return;
        }
        if (p.input_kind == IN_PCM_S16) {
            short4 s = __ldg(reinterpret_cast<const short4 *>(reinterpret_cast<const short *>(w.in) + i0));
            x[0] = env_real(__fdiv_rn((float)s.x, p.pcm_scale));
            x[1] = env_real(__fdiv_rn((float)s.y, p.pcm_scale));
            x[2] = env_real(__fdiv_rn((float)s.z, p.pcm_scale));
            x[3] = env_real(__fdiv_rn((float)s.w, p.pcm_scale));
            return;
        }
        if (SC16 && p.input_kind == IN_SC16) {
            const float4 v = env_sc16x4(ldg_stream4(reinterpret_cast<const float4 *>(reinterpret_cast<const short2 *>(w.in) + i0)),
                                        p.pcm_scale);
            x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
            return;
        }
    }
#pragma unroll
    for (int j = 0; j < K; j++) {
        int64_t q = p0 + j;
        x[j] = (q >= w.in_begin && q < w.in_end) ? load_one<SC16>(w.in, q - w.in_pos0, p) : 0.0f;
    }
}

// ---------------------------------------------------------------- the ratio test, exactly
// transition_sink.py:59-71:  ratio = bit*length/ss  (or the ss == 0 constants);  lo > ratio -> LOW;
// ratio > hi -> HIGH (before hysteresis); else MID.
__device__ __noinline__ int classify_div(double pr, double ss, double lo, double hi) {
    double ratio = __ddiv_rn(pr, ss);
    if (lo > ratio) return CLS_LOW;
    if (ratio > hi) return CLS_HIGH;
    return CLS_MID;
}

__device__ __forceinline__ int classify(float x, double ss, const SlicerParams &p) {
    if (ss == 0.0) return x == 0.0f ? p.cls_ss0_x0 : p.cls_ss0_xn;
    const double pr = (double)x * p.Ld;  // exact: 24-bit significand times an integer < 2^29
    if (!(ss > 0.0) || !(p.lo > 0.0) || !(p.hi > 0.0)) return classify_div(pr, ss, p.lo, p.hi);
    // sign(pr - lo*ss) is exact with one FMA; RN(pr/ss) can only disagree with it within half an ulp
    const double r = fma(-p.lo, ss, pr);
    if (r < 0.0) {
        if (r > -(p.lo * ss) * 0x1p-50) return classify_div(pr, ss, p.lo, p.hi);
        return CLS_LOW;
    }
    const double r2 = fma(-p.hi, ss, pr);
    if (r2 > 0.0) {
        if (r2 < (p.hi * ss) * 0x1p-50) return classify_div(pr, ss, p.lo, p.hi);
        return CLS_HIGH;
    }
    // r >= 0 and r2 <= 0: pr/ss in [lo, hi] exactly, and RN is monotonic
    return CLS_MID;
}

// hysteresis: is a HIGH-class sample at stream index i forced to val 0 (cur_state == 2)?
// b = last LOW sample before i, a = first sample of the LOW run containing b.
__device__ __forceinline__ bool st2_forced(int64_t i, int64_t b, int64_t a, int mx) {
    if (b == NO_POS || i - b > (int64_t)mx + 1) return false;
    const int64_t j = b - a;
    const bool tmo = j >= mx && (j % mx) == 0;  // b itself was a timeout sample: cur_state went back to 0
    return !tmo;
}

// ---------------------------------------------------------------- block-wide primitives
template <int NT>
struct BlockShared {
    static const int NW = NT / 32;
    double wsum[2][NW];
    int wcnt[2][NW];
    int wlastcls[NW];   // class of each warp's last sample (current round)
    int wmaxL[NW];      // tile-relative index of the last LOW sample per warp
    int wmaxS[NW];      // tile-relative index of the last LOW-run start per warp
    unsigned flags[3];
    int emin, emax;
    double red[NW];
};

// everything a segment carries from tile to tile (identical in all threads of the CTA)
struct SegCarry {
    double ss0;
    int64_t lastL, lrun_start;
    int last_val;
    uint32_t seg_count;
    unsigned round_no;
    int scan_buf, cnt_buf;
};

template <int NT>
__device__ __forceinline__ double block_excl_scan(double v, double &total, double (*wsum)[NT / 32], int buf) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        double n = __shfl_up_sync(FULL, inc, o);
        if (lane >= o) inc += n;
    }
    if (lane == 31) wsum[buf][warp] = inc;
    cta_sync<NT>();
    double wbase = 0.0, tot = 0.0;
#pragma unroll
    for (int w = 0; w < NT / 32; w++) {
        double s = wsum[buf][w];
        if (w < warp) wbase += s;
        tot += s;
    }
    total = tot;
    return wbase + (inc - v);
}

template <int NT>
__device__ __forceinline__ int block_excl_scan_int(int v, int &total, int (*wcnt)[NT / 32], int buf) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int n = __shfl_up_sync(FULL, inc, o);
        if (lane >= o) inc += n;
    }
    if (lane == 31) wcnt[buf][warp] = inc;
    cta_sync<NT>();
    int wbase = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < NT / 32; w++) {
        int s = wcnt[buf][w];
        if (w < warp) wbase += s;
        tot += s;
    }
    total = tot;
    return wbase + (inc - v);
}

__device__ __forceinline__ void exp_track(float x, int &emin, int &emax) {
    const unsigned ub = __float_as_uint(x);
    if (ub != 0u) {
        const int e = (int)(ub >> 23);  // sign bit set -> e >= 256 -> flagged not sane below
        emin = min(emin, max(e, 1));
        emax = max(emax, e);
    }
}

// ---------------------------------------------------------------- exact tile (fix-point over prefix sums)
// One tile of NT*K samples starting at stream index P0, classes decided with every sample's own exact ss.
// Always correct (inside the exactly-summable regime); several block barriers per tile.
template <int NT, int K, bool BM = false, bool SC16 = true>
__device__ __noinline__ void exact_tile(const SegWork *wp, const SlicerParams *pp, float *ring, BlockShared<NT> *shp,
                                        const int64_t P0, const int slot0, SegCarry *cs) {
    constexpr int NW = NT / 32;
    const SegWork &w = *wp;
    const SlicerParams &p = *pp;
    BlockShared<NT> &sh = *shp;
    const int L = p.L, mx = p.mx;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t p0 = P0 + (int64_t)tid * K;
    SegCarry c = *cs;  // shared -> registers (identical in all threads)
    int emin = 1 << 30, emax = 0;
    const double ss0 = c.ss0;
    const int64_t lastL = c.lastL, lrun_start = c.lrun_start;
    const int last_val = c.last_val;

    float x[K], prev[K];
    bool act[K];
    load_samples<K, SC16>(w, p, p0, x);
#pragma unroll
    for (int j = 0; j < K; j++) act[j] = (p0 + j >= w.warm_begin) && (p0 + j < w.end);

    int slot[K];
#pragma unroll
    for (int j = 0; j < K; j++) {
        int s = slot0 + j;
        slot[j] = s >= L ? s - L : s;
    }
    if (K == 4 && (L & 3) == 0) {
        float4 v = *reinterpret_cast<const float4 *>(ring + slot0);
        prev[0] = v.x; prev[1] = v.y; prev[2] = v.z; prev[3] = v.w;
    } else {
#pragma unroll
        for (int j = 0; j < K; j++) prev[j] = ring[slot[j]];
    }

    int cls[K];
    bool forced[K];
#pragma unroll
    for (int j = 0; j < K; j++) {
        cls[j] = act[j] ? classify(x[j], ss0, p) : CLS_MID;  // guess: ss frozen at the tile start
        forced[j] = false;
    }
    const bool carry_recent = lastL != NO_POS && (P0 - lastL) <= (int64_t)mx + 1;

    double total = 0.0;
    bool had_slow = false, anyL = false;
    for (;;) {
        const unsigned fb = c.round_no % 3u;
        if (tid == 0) sh.flags[(c.round_no + 1u) % 3u] = 0u;
        double pre[K];
        double run = 0.0;
#pragma unroll
        for (int j = 0; j < K; j++) {
            pre[j] = run;
            const bool admit = act[j] && (cls[j] == CLS_MID || (cls[j] == CLS_HIGH && forced[j]));
            if (admit) run += (double)x[j] - (double)prev[j];  // cur - prev (transition_sink.py:82)
        }
        const double base = block_excl_scan<NT>(run, total, sh.wsum, c.scan_buf);
        c.scan_buf ^= 1;

        unsigned f = 0u;
#pragma unroll
        for (int j = 0; j < K; j++) {
            if (act[j]) {
                const int cc = classify(x[j], ss0 + (base + pre[j]), p);
                if (cc != cls[j]) { f |= 1u; cls[j] = cc; }
                if (cc == CLS_HIGH) f |= 2u;
                if (cc == CLS_LOW) f |= 4u;
            }
        }
        f = __reduce_or_sync(FULL, f);
        if (lane == 0 && f) atomicOr(&sh.flags[fb], f);
        if (lane == 31) sh.wlastcls[warp] = act[K - 1] ? cls[K - 1] : 2;  // 2 = "no sample"
        cta_sync<NT>();
        unsigned flags = sh.flags[fb];
        c.round_no++;

        if ((flags & 2u) && ((flags & 4u) || carry_recent)) {
            // ---- hysteresis: distance from each HIGH sample to the last LOW sample / its run start
            int pc = __shfl_up_sync(FULL, cls[K - 1], 1);
            const bool pact = __shfl_up_sync(FULL, (int)act[K - 1], 1) != 0;
            if (lane == 0) {
                pc = CLS_MID;
                bool found = false;
                for (int ww = warp - 1; ww >= 0 && !found; ww--) {
                    int cc = sh.wlastcls[ww];
                    if (cc != 2) { pc = cc; found = true; }
                }
                if (!found) pc = (last_val == -1) ? CLS_LOW : CLS_MID;
            } else if (!pact) {
                pc = (last_val == -1) ? CLS_LOW : CLS_MID;  // inactive prefix of the first tile
            }
            int myL = -1, myS = -1;
            int preL[K], preS[K];
            {
                int c_prev = pc;
#pragma unroll
                for (int j = 0; j < K; j++) {
                    preL[j] = myL;
                    preS[j] = myS;
                    if (act[j]) {
                        if (cls[j] == CLS_LOW) {
                            if (c_prev != CLS_LOW) myS = tid * K + j;
                            myL = tid * K + j;
                        }
                        c_prev = cls[j];
                    }
                }
            }
            int incL = myL, incS = myS;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int a = __shfl_up_sync(FULL, incL, o), b = __shfl_up_sync(FULL, incS, o);
                if (lane >= o) { incL = max(incL, a); incS = max(incS, b); }
            }
            int exL = __shfl_up_sync(FULL, incL, 1), exS = __shfl_up_sync(FULL, incS, 1);
            if (lane == 0) { exL = -1; exS = -1; }
            if (lane == 31) { sh.wmaxL[warp] = incL; sh.wmaxS[warp] = incS; }
            cta_sync<NT>();
            for (int ww = 0; ww < warp; ww++) {
                exL = max(exL, sh.wmaxL[ww]);
                exS = max(exS, sh.wmaxS[ww]);
            }
            unsigned f2 = 0u;
#pragma unroll
            for (int j = 0; j < K; j++) {
                bool fo = false;
                if (act[j] && cls[j] == CLS_HIGH) {
                    const int bl = max(exL, preL[j]);
                    const int sl = max(exS, preS[j]);
                    const int64_t b = bl >= 0 ? P0 + bl : lastL;
                    const int64_t a = sl >= 0 ? P0 + sl : lrun_start;
                    fo = st2_forced(p0 + j, b, a, mx);
                }
                if (fo != forced[j]) { f2 = 1u; forced[j] = fo; }
            }
            const unsigned fb2 = c.round_no % 3u;
            if (tid == 0) sh.flags[(c.round_no + 1u) % 3u] = 0u;
            f2 = __reduce_or_sync(FULL, f2);
            if (lane == 0 && f2) atomicOr(&sh.flags[fb2], f2);
            cta_sync<NT>();
            flags |= sh.flags[fb2] & 1u;
            c.round_no++;
            had_slow = true;
        } else if (had_slow) {
            // `forced` flags are only ever set in the (block-uniform) branch above; once the tile no longer
            // needs it they are cleared, which changes `admit`, so vote for another round.
            unsigned f2 = 0u;
#pragma unroll
            for (int j = 0; j < K; j++) {
                if (forced[j]) { f2 = 1u; forced[j] = false; }
            }
            if (cta_sync_or<NT>((int)f2)) flags |= 1u;
            had_slow = false;
        }
        if (!(flags & 1u)) {  // converged: `total` belongs to the final classes
            anyL = (flags & 4u) != 0u;
            break;
        }
    }

    // ---- ring update (transition_sink.py:75-81) and exponent tracking
    float nv[K];
#pragma unroll
    for (int j = 0; j < K; j++) {
        const bool admit = act[j] && (cls[j] == CLS_MID || (cls[j] == CLS_HIGH && forced[j]));
        nv[j] = admit ? x[j] : prev[j];
        if (admit) exp_track(x[j], emin, emax);
    }
    if (K == 4 && (L & 3) == 0 && act[0] && act[K - 1]) {
        *reinterpret_cast<float4 *>(ring + slot0) = make_float4(nv[0], nv[1], nv[2], nv[3]);
    } else {
#pragma unroll
        for (int j = 0; j < K; j++)
            if (act[j]) ring[slot[j]] = nv[j];
    }

    // ---- vals and transitions
    int val[K];
#pragma unroll
    for (int j = 0; j < K; j++)
        val[j] = act[j] ? (cls[j] == CLS_LOW ? -1 : ((cls[j] == CLS_HIGH && !forced[j]) ? 1 : 0)) : 3;  // 3 = none
    int mylast = 3;
#pragma unroll
    for (int j = 0; j < K; j++)
        if (val[j] != 3) mylast = val[j];
    int pv;
    {
        const unsigned has = __ballot_sync(FULL, mylast != 3);
        const unsigned lower = has & ((1u << lane) - 1u);
        const int src = lower ? 31 - __clz(lower) : 0;
        const int got = __shfl_sync(FULL, mylast, src);
        pv = lower ? got : 3;
        int wl = __shfl_sync(FULL, mylast, has ? 31 - __clz(has) : 0);
        if (!has) wl = 3;
        if (lane == 0) sh.wlastcls[warp] = wl;  // reuse: last defined val of the warp (3 = none)
    }
    cta_sync<NT>();
    if (pv == 3) {
        pv = last_val;
        for (int ww = warp - 1; ww >= 0; ww--) {
            const int cc = sh.wlastcls[ww];
            if (cc != 3) { pv = cc; break; }
        }
    }
    int ntr = 0;
    unsigned trmask = 0u;
    int maxS = -1, maxL = -1;
    {
        int c_prev = pv;
#pragma unroll
        for (int j = 0; j < K; j++) {
            if (val[j] != 3) {
                if (val[j] != c_prev) {
                    if (p0 + j >= w.begin) { trmask |= 1u << j; ntr++; }
                    if (val[j] == -1) maxS = tid * K + j;
                }
                if (val[j] == -1) maxL = tid * K + j;
                c_prev = val[j];
            }
        }
    }
    if (anyL) {
        int mL = __reduce_max_sync(FULL, maxL), mS = __reduce_max_sync(FULL, maxS);
        if (lane == 0) { sh.wmaxL[warp] = mL; sh.wmaxS[warp] = mS; }
    }
    int tot_tr = 0;
    const int tr_base = block_excl_scan_int<NT>(ntr, tot_tr, sh.wcnt, c.cnt_buf);
    c.cnt_buf ^= 1;
    if (BM) {
        // bitmap output: this warp's 128 samples are one chunk (sample 4*lane + j <-> bit lane of word j)
        if (K == 4 && w.bitmap) {
            unsigned wv = 0u;
#pragma unroll
            for (int j = 0; j < K; j++) {
                // samples of the chunk outside [begin, end) are written as val == 0: a single stream masks them by position
                // (extract.cu), in a batch of captures they are the warm-up / padding around the capture
                const bool on = val[j] != 3 && (p0 + j >= w.begin);
                const unsigned bn = __ballot_sync(FULL, !on || val[j] != -1), bh = __ballot_sync(FULL, on && val[j] == 1);
                if (lane == j) wv = bn;
                if (lane == 4 + j) wv = bh;
            }
            const int64_t cfirst = P0 + (int64_t)warp * 128;
            if (lane < 8 && cfirst + 127 >= w.begin && cfirst < w.end) w.bitmap[((cfirst - w.bm_pos0) >> 7) * 8 + lane] = wv;
        }
    } else if (tot_tr) {
        uint32_t idx = c.seg_count + (uint32_t)tr_base;
#pragma unroll
        for (int j = 0; j < K; j++) {
            if (trmask & (1u << j)) {
                if (idx < w.trans_cap) w.trans[idx] = pack_trans((uint32_t)(p0 + j - w.slab_pos0), val[j]);
                idx++;
            }
        }
        c.seg_count += (uint32_t)tot_tr;
    }
    // ---- carries into the next tile
    c.ss0 = ss0 + total;
    if (anyL) {
        int mL = -1, mS = -1;
#pragma unroll
        for (int ww = 0; ww < NW; ww++) {
            mL = max(mL, sh.wmaxL[ww]);
            mS = max(mS, sh.wmaxS[ww]);
        }
        if (mL >= 0) {
            c.lastL = P0 + mL;
            if (mS >= 0) c.lrun_start = P0 + mS;
        }
    }
    {
        int lv = 3;
        for (int ww = NW - 1; ww >= 0; ww--) {
            const int cc = sh.wlastcls[ww];
            if (cc != 3) { lv = cc; break; }
        }
        if (lv != 3) c.last_val = lv;
    }
    emin = __reduce_min_sync(FULL, emin);
    emax = __reduce_max_sync(FULL, emax);
    if (lane == 0) {
        atomicMin(&sh.emin, emin);
        atomicMax(&sh.emax, emax);
    }
    if (tid == 0) *cs = c;
    cta_sync<NT>();  // carry, ring writes and shared scratch settle before the next tile reads them
}

// ---------------------------------------------------------------- the segment kernel
// First-generation kernel, for the windows the streaming kernel does not take (below 1024 samples or not a multiple of 4):
// one CTA walks one time segment in tiles of SLICER_NT samples, one sample per thread, each through exact_tile.
constexpr int SLICER_NT = 256;
__global__ void __launch_bounds__(SLICER_NT, 2) slicer_kernel(const SegWork *__restrict__ works,
                                                             const SlicerParams *__restrict__ params) {
    constexpr int NT = SLICER_NT, T = SLICER_NT;
    constexpr int NW = NT / 32;
    extern __shared__ __align__(16) float ring[];
    __shared__ BlockShared<NT> sh;

    // the work item and the parameters live in shared memory: one copy per CTA, no registers held
    __shared__ SegWork w_s;
    __shared__ SlicerParams p_s;
    __shared__ SegCarry c_s;
    if (threadIdx.x == 0) {
        w_s = works[blockIdx.x];
        p_s = params[w_s.param_idx];
    }
    __syncthreads();
    const SegWork &w = w_s;
    const SlicerParams &p = p_s;
    const int L = p.L;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // ---- entry state
    SegCarry c;
    int status = SEG_OK;
    int emin = 1 << 30, emax = 0;

    if (w.state_in) {
        const float *src = state_ring(w.state_in);
        for (int i = tid; i < L; i += NT) {
            float v = src[i];
            ring[i] = v;
            exp_track(v, emin, emax);
        }
        c.ss0 = w.state_in->ss;
        c.lastL = w.state_in->lastL;
        c.lrun_start = w.state_in->lrun_start;
        c.last_val = w.state_in->last_val;
    } else {
        // cold start: the previous L samples, unconditionally (transition_sink.py:118)
        double part = 0.0;
        for (int i = tid; i < L; i += NT) {
            const int64_t q = w.warm_begin - L + i;
            float v = load_one(w.in, q - w.in_pos0, p);
            ring[(int)(q % L)] = v;
            part += (double)v;
            exp_track(v, emin, emax);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(FULL, part, o);
        if (lane == 0) sh.red[warp] = part;
        __syncthreads();
        double s0 = 0.0;
        for (int i = 0; i < NW; i++) s0 += sh.red[i];
        c.ss0 = s0;
        c.lastL = NO_POS;
        c.lrun_start = NO_POS;
        c.last_val = 0;
    }
    if (tid == 0) {
        sh.flags[0] = sh.flags[1] = sh.flags[2] = 0u;
        sh.emin = 1 << 30;
        sh.emax = 0;
    }
    __syncthreads();
    c.seg_count = 0;
    c.scan_buf = 0;
    c.cnt_buf = 0;
    c.round_no = 0;
    unsigned n_exact = 0;

    const int64_t tile_first = w.warm_begin / T;
    const int64_t tile_last = (w.end > w.warm_begin) ? (w.end - 1) / T : tile_first - 1;
    int slot0 = (int)((tile_first * T + (int64_t)tid) % L);

    for (int64_t tile = tile_first; tile <= tile_last; tile++) {
        const int64_t P0 = tile * T;

        if (w.seam_in && P0 == w.begin && w.begin > w.warm_begin) {
            // snapshot of the speculative state at the first emitted sample
            float *dst = state_ring(w.seam_in);
            for (int i = tid; i < L; i += NT) dst[i] = ring[i];
            if (tid == 0) {
                SlicerHdr h;
                h.ss = c.ss0; h.pos = w.begin; h.lastL = c.lastL; h.lrun_start = c.lrun_start;
                h.last_val = c.last_val; h.emin = 0; h.emax = 0; h.status = 0; h.count = 0; h.pad = 0;
                *w.seam_in = h;
            }
        }

#pragma unroll
        for (int j = 0; j < 3; j++) {
            if (w.ckpt_state[j] && P0 == w.ckpt_pos[j]) {  // block-uniform
                float *dst = state_ring(w.ckpt_state[j]);
                for (int i = tid; i < L; i += NT) dst[i] = ring[i];
                if (tid == 0) {
                    SlicerHdr h;
                    h.ss = c.ss0; h.pos = P0; h.lastL = c.lastL; h.lrun_start = c.lrun_start;
                    h.last_val = c.last_val; h.emin = 0; h.emax = 0; h.status = 0; h.count = c.seg_count; h.pad = 0;
                    *w.ckpt_state[j] = h;
                }
            }
        }

        if (tid == 0) c_s = c;
        __syncthreads();
        exact_tile<NT, 1>(&w_s, &p_s, ring, &sh, P0, slot0, &c_s);
        c = c_s;
        n_exact++;
        slot0 += T % L;
        if (slot0 >= L) slot0 -= L;
    }

    // ---- exit: exactness audit and final state
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        emin = min(emin, __shfl_xor_sync(FULL, emin, o));
        emax = max(emax, __shfl_xor_sync(FULL, emax, o));
    }
    __syncthreads();
    if (lane == 0) { atomicMin(&sh.emin, emin); atomicMax(&sh.emax, emax); }
    __syncthreads();
    emin = sh.emin; emax = sh.emax;
    if (emax >= 255) status |= SEG_NOT_SANE;
    if (emax > 0 && emax - emin > p.span_limit) status |= SEG_INEXACT;
    if (c.seg_count > w.trans_cap) status |= SEG_OVERFLOW;

    if (w.state_out) {
        float *dst = state_ring(w.state_out);
        for (int i = tid; i < L; i += NT) dst[i] = ring[i];
        if (tid == 0) {
            SlicerHdr h;
            h.ss = c.ss0; h.pos = w.end; h.lastL = c.lastL; h.lrun_start = c.lrun_start;
            h.last_val = c.last_val; h.emin = emin; h.emax = emax; h.status = status; h.count = c.seg_count; h.pad = 0;
            *w.state_out = h;
        }
    }
    if (tid == 0 && w.trans_count) *w.trans_count = c.seg_count;
    if (tid == 0 && w.status) *w.status = status;
    if (tid == 0) {
        atomicAdd(&g_tile_stats[1], (unsigned long long)n_exact);
        atomicAdd(&g_tile_stats[8], (unsigned long long)c.round_no);
    }
}

}  // namespace nfc
#include "slicer_fast.cuh"
namespace nfc {

// ---------------------------------------------------------------- strictly sequential path
// The reference recurrence, literally, one thread per segment: used when av_window is smaller
// than a tile, when the exponent audit fails (inexact sums, negative or non-finite samples) and
// as the independent on-device cross-check of the parallel kernel.  `ss` is carried exactly as
// the reference carries it (ss += cur - prev in double, in order).
__global__ void slicer_serial_kernel(const SegWork *__restrict__ works, const SlicerParams *__restrict__ params,
                                     float *__restrict__ ring_scratch, size_t ring_stride) {
    if (threadIdx.x != 0) return;
    const SegWork w = works[blockIdx.x];
    const SlicerParams p = params[w.param_idx];
    const int L = p.L, mx = p.mx;
    float *ring = ring_scratch + (size_t)blockIdx.x * ring_stride;

    double ss;
    int64_t lastL, lrun_start;
    int last_val;
    if (w.state_in) {
        const float *src = state_ring(w.state_in);
        for (int i = 0; i < L; i++) ring[i] = src[i];
        ss = w.state_in->ss;
        lastL = w.state_in->lastL;
        lrun_start = w.state_in->lrun_start;
        last_val = w.state_in->last_val;
    } else {
        ss = 0.0;
        // slot order == stream order here only if warm_begin % L == 0; sum in stream order like sum(ar)
        for (int i = 0; i < L; i++) {
            const int64_t q = w.warm_begin - L + i;
            float v = load_one(w.in, q - w.in_pos0, p);
            ring[(int)(q % L)] = v;
            ss += (double)v;
        }
        lastL = NO_POS;
        lrun_start = NO_POS;
        last_val = 0;
    }
    uint32_t count = 0;
    int slot = (int)(w.warm_begin % L);
    for (int64_t q = w.warm_begin; q < w.end; q++) {
        if (w.seam_in && q == w.begin && w.begin > w.warm_begin) {
            float *dst = state_ring(w.seam_in);
            for (int i = 0; i < L; i++) dst[i] = ring[i];
            SlicerHdr h;
            h.ss = ss; h.pos = q; h.lastL = lastL; h.lrun_start = lrun_start;
            h.last_val = last_val; h.emin = 0; h.emax = 0; h.status = 0; h.count = 0; h.pad = 0;
            *w.seam_in = h;
        }
        const float x = load_one(w.in, q - w.in_pos0, p);
        const float prev = ring[slot];
        int c;
        if (ss == 0.0) c = x == 0.0f ? p.cls_ss0_x0 : p.cls_ss0_xn;
        else c = classify_div((double)x * p.Ld, ss, p.lo, p.hi);
        int val;
        if (c == CLS_LOW) {
            val = -1;
            if (last_val != -1) lrun_start = q;
            lastL = q;
        } else if (c == CLS_HIGH && !st2_forced(q, lastL, lrun_start, mx)) {
            val = 1;
        } else {
            val = 0;
            ring[slot] = x;
            ss += ((double)x - (double)prev);
        }
        if (val != last_val) {
            if (q >= w.begin) {
                if (count < w.trans_cap) w.trans[count] = pack_trans((uint32_t)(q - w.slab_pos0), val);
                count++;
            }
            last_val = val;
        }
        slot++;
        if (slot == L) slot = 0;
    }
    if (w.state_out) {
        float *dst = state_ring(w.state_out);
        for (int i = 0; i < L; i++) dst[i] = ring[i];
        SlicerHdr h;
        h.ss = ss; h.pos = w.end; h.lastL = lastL; h.lrun_start = lrun_start;
        h.last_val = last_val; h.emin = 0; h.emax = 0;
        h.status = count > w.trans_cap ? SEG_OVERFLOW : SEG_OK;
        h.count = count; h.pad = 0;
        *w.state_out = h;
    }
    if (w.trans_count) *w.trans_count = count;
    if (w.status) *w.status = count > w.trans_cap ? SEG_OVERFLOW : SEG_OK;
}

// ---------------------------------------------------------------- seam verification
// For seam k (between segment k-1 and k): does the state the predecessor really reached equal the
// state the successor assumed at its first emitted sample?  Bitwise on ring and ss; the hysteresis
// carry is compared in canonical form (only what can still influence the future).
__device__ __forceinline__ void canon_st2(const SlicerHdr &h, int mx, int &kind, int64_t &val) {
    if (h.last_val == -1) { kind = 1; val = h.lrun_start; return; }
    if (h.lastL == NO_POS) { kind = 0; val = 0; return; }
    const int64_t j = h.lastL - h.lrun_start;
    const bool tmo = j >= mx && (j % mx) == 0;
    const int64_t until = tmo ? h.lastL : h.lastL + mx + 1;
    if (until < h.pos) { kind = 0; val = 0; } else { kind = 2; val = until; }
}

__global__ void seam_compare_kernel(const SlicerHdr *const *__restrict__ truth, const SlicerHdr *const *__restrict__ assumed,
                                    const int *__restrict__ param_idx, const SlicerParams *__restrict__ params,
                                    int *__restrict__ mismatch) {
    const SlicerHdr *a = truth[blockIdx.x], *b = assumed[blockIdx.x];
    if (!a || !b) return;
    const SlicerParams p = params[param_idx[blockIdx.x]];
    int bad = 0;
    const uint32_t *ra = reinterpret_cast<const uint32_t *>(state_ring(a));
    const uint32_t *rb = reinterpret_cast<const uint32_t *>(state_ring(b));
    if ((((uintptr_t)ra | (uintptr_t)rb) & 15) == 0 && (p.L & 3) == 0) {  // 128-bit loads, two in flight per thread
        const uint4 *va = reinterpret_cast<const uint4 *>(ra), *vb = reinterpret_cast<const uint4 *>(rb);
        const int n4 = p.L >> 2;
        for (int i = threadIdx.x; i < n4; i += 2 * blockDim.x) {
            const int j = i + blockDim.x;
            const uint4 x0 = __ldg(va + i), y0 = __ldg(vb + i);
            uint4 x1 = x0, y1 = y0;
            if (j < n4) { x1 = __ldg(va + j); y1 = __ldg(vb + j); }
            bad |= (x0.x != y0.x) | (x0.y != y0.y) | (x0.z != y0.z) | (x0.w != y0.w) | (x1.x != y1.x) | (x1.y != y1.y) |
                   (x1.z != y1.z) | (x1.w != y1.w);
        }
    } else {
        for (int i = threadIdx.x; i < p.L; i += blockDim.x) bad |= (ra[i] != rb[i]);
    }
    if (threadIdx.x == 0) {
        if (__double_as_longlong(a->ss) != __double_as_longlong(b->ss)) bad = 1;
        if (a->last_val != b->last_val || a->pos != b->pos) bad = 1;
        int ka, kb;
        int64_t va, vb;
        canon_st2(*a, p.mx, ka, va);
        canon_st2(*b, p.mx, kb, vb);
        if (ka != kb || va != vb) bad = 1;
    }
    if (__syncthreads_or(bad) && threadIdx.x == 0) mismatch[blockIdx.x] = 1;
}

// ---------------------------------------------------------------- host launchers
bool slicer_streaming_ok(int L, int kind);
int slicer_streaming_tile(int L, int kind);
// tile of the kernel a window takes: segment boundaries and halos are whole tiles
int slicer_tile(int L, int kind) {
    if (slicer_streaming_ok(L, kind)) return slicer_streaming_tile(L, kind);
    return SLICER_NT;
}

static int raise_dynamic_smem(const void *fn, size_t smem);

// ---- variants of the streaming kernel.  Default: the pipelined one (slicer_pipe.cuh), two CTAs of 8 + 2 warps per SM with
// three stages of 4096 samples (NFC_SLICER_STAGES=2: two); windows too long for that (20 MS/s: 80 KB ring) take 16 + 2 warps,
// one CTA per SM.  NFC_SLICER_PIPE=0: the synchronous loop only (three CTAs of 8 warps per SM, round 1's kernel).
struct FastVariant {
    const void *fn;
    int threads;
    size_t smem;  // dynamic: the ring, then the stages (or the one staging buffer of the synchronous loop)
    int tile;     // samples per tile: segment boundaries and halos are whole tiles
};
static int env_int(const char *name, int dflt) {
    const char *v = getenv(name);
    return (v && v[0]) ? atoi(v) : dflt;
}
static size_t smem_optin_limit() {
    int dev = 0, lim = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    return (size_t)lim;
}
static const size_t FAST_STATIC_SMEM = 10 * 1024;  // upper bound of the kernels' static shared memory

// Windows below two tiles of 4096 samples (the reference's own default: av_window = 2000, transition_sink.py:12) take the
// same kernel with tiles of 512 samples: four worker warps, one chunk of 128 samples each.
static const int FAST_SMALL_MIN_L = 1024, FAST_BIG_MIN_L = 8192;
template <int KIND>
static FastVariant fast_variant(int L) {
    static const int pipe = env_int("NFC_SLICER_PIPE", 1), stages = env_int("NFC_SLICER_STAGES", 3);
    const size_t ring = ((size_t)L * 4 + 15) / 16 * 16;
    const size_t item = KIND == IN_IQ_F32 ? 8 : (KIND == IN_PCM_S16 ? 2 : 4);  // IN_SC16: 4, as the float kinds
    const size_t T = L >= FAST_BIG_MIN_L ? 4096 : 512;
    const size_t one = KIND == IN_IQ_F32 ? 0 : T * item;  // staging buffer of the synchronous loop (IQ tiles are not staged)
    // a stage of the pipelined mode (PipeStage): samples, undo log (4-byte items, sc16 included: the log overlays the samples)
    const size_t stg = KIND == IN_PCM_S16 ? T * 6 : T * 4;
    const size_t half = smem_optin_limit() / 2;               // two CTAs per SM
    FastVariant v;
    v.tile = (int)T;
    if (L < FAST_BIG_MIN_L) {
        if (pipe && KIND != IN_IQ_F32) {
            v.fn = (const void *)slicer_fast_kernel<128, 1, 5, KIND, 3>;
            v.threads = 192;
            v.smem = ring + 3 * stg;
        } else {
            v.fn = (const void *)slicer_fast_kernel<128, 1, 6, KIND, 0>;
            v.threads = 128;
            v.smem = ring + one;
        }
        return v;
    }
    if (pipe && KIND != IN_IQ_F32) {
        if (stages >= 3 && ring + 3 * stg + FAST_STATIC_SMEM <= half) {
            v.fn = (const void *)slicer_fast_kernel<256, 4, 2, KIND, 3>;
            v.threads = 320;
            v.smem = ring + 3 * stg;
        } else if (ring + 2 * stg + FAST_STATIC_SMEM <= half) {
            v.fn = (const void *)slicer_fast_kernel<256, 4, 2, KIND, 2>;
            v.threads = 320;
            v.smem = ring + 2 * stg;
        } else if (env_int("NFC_SLICER_HALF_TILE", 1) && ring + 3 * (stg / 2) + FAST_STATIC_SMEM <= half) {
            // a window too long for two CTAs with tiles of 4096 samples beside their rings (20 MS/s: 80 KB): tiles of 2048 samples
            // (two chunks per warp) keep two CTAs per SM
            v.fn = (const void *)slicer_fast_kernel<256, 2, 2, KIND, 3>;
            v.threads = 320;
            v.smem = ring + 3 * (stg / 2);
            v.tile = 2048;
        } else if (ring + 3 * stg + FAST_STATIC_SMEM <= smem_optin_limit()) {
            v.fn = (const void *)slicer_fast_kernel<512, 2, 1, KIND, 3>;
            v.threads = 576;
            v.smem = ring + 3 * stg;
        } else {  // a window that leaves no room for the stages beside its ring: the synchronous loop
            v.fn = (const void *)slicer_fast_kernel<256, 4, 3, KIND, 0>;
            v.threads = 256;
            v.smem = ring + one;
        }
    } else {
        v.fn = (const void *)slicer_fast_kernel<256, 4, 3, KIND, 0>;
        v.threads = 256;
        v.smem = ring + one;
    }
    return v;
}
static FastVariant fast_variant_of(int L, int kind) {
    switch (kind) {
        case IN_ENVELOPE_F32: return fast_variant<IN_ENVELOPE_F32>(L);
        case IN_REAL_F32: return fast_variant<IN_REAL_F32>(L);
        case IN_IQ_F32: return fast_variant<IN_IQ_F32>(L);
        case IN_SC16: return fast_variant<IN_SC16>(L);
        default: return fast_variant<IN_PCM_S16>(L);
    }
}

int slicer_streaming_tile(int L, int kind) { return fast_variant_of(L, kind).tile; }

// cudaFuncAttributeMaxDynamicSharedMemorySize of a kernel is only ever raised (streams with different windows share the
// kernels, and setting the attribute before every launch serialises the launching threads)
static int raise_dynamic_smem(const void *fn, size_t smem) {
    static std::mutex mu;
    static std::map<std::pair<const void *, int>, size_t> have;
    int dev = 0;
    NFC_CUDA_CHECK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    size_t &cur = have[std::make_pair(fn, dev)];
    if (cur < smem) {
        NFC_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cur = smem;
    }
    return 0;
}

// the streaming kernel takes windows that are a multiple of 4 from 1024 samples on, as long as the variant chosen for the
// window fits one CTA's shared memory: its dynamic part (ring and staging) and the kernel's static scratch
bool slicer_streaming_ok(int L, int kind) {
    if (L % 4 != 0 || L < FAST_SMALL_MIN_L) return false;
    const FastVariant v = fast_variant_of(L, kind);
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, v.fn) != cudaSuccess) return false;
    return v.smem + fa.sharedSizeBytes <= smem_optin_limit();
}

static int apply_pipe_tuning() {
    static std::mutex mu;
    static bool done[64] = {false};
    int dev = 0;
    NFC_CUDA_CHECK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    if (done[dev & 63]) return 0;
    done[dev & 63] = true;
    if (getenv("NFC_PIPE_MIN") || getenv("NFC_PIPE_COOL") || getenv("NFC_MEAS_MAX") || getenv("NFC_RESUM_BITS")) {
        int t[4] = {env_int("NFC_PIPE_MIN", 6), env_int("NFC_PIPE_COOL", 3), env_int("NFC_MEAS_MAX", 2), env_int("NFC_RESUM_BITS", 18)};
        if (t[0] < 3) t[0] = 3;
        if (t[1] < 0) t[1] = 0;
        if (t[2] < 1) t[2] = 1;
        NFC_CUDA_CHECK(cudaMemcpyToSymbol(g_pipe_tune, t, sizeof(t)));
    }
    return 0;
}

int launch_slicer_streaming(const SegWork *d_works, int n_works, const SlicerParams *d_params, int L, int kind, cudaStream_t stream) {
    if (n_works <= 0) return 0;
    if (apply_pipe_tuning()) return -1;
    const FastVariant v = fast_variant_of(L, kind);
    if (raise_dynamic_smem(v.fn, v.smem)) return -1;
    void *args[2] = {(void *)&d_works, (void *)&d_params};
    NFC_CUDA_CHECK(cudaLaunchKernel(v.fn, dim3((unsigned)n_works), dim3((unsigned)v.threads), args, v.smem, stream));
    return 0;
}

int launch_slicer(const SegWork *d_works, int n_works, const SlicerParams *d_params, int L, cudaStream_t stream) {
    if (n_works <= 0) return 0;
    const size_t smem = ((size_t)L * 4 + 15) / 16 * 16;
    if (raise_dynamic_smem((const void *)slicer_kernel, smem)) return -1;
    slicer_kernel<<<n_works, SLICER_NT, smem, stream>>>(d_works, d_params);
    NFC_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int slicer_tile_stats(unsigned long long *out4, bool reset) {
    NFC_CUDA_CHECK(cudaMemcpyFromSymbol(out4, g_tile_stats, sizeof(unsigned long long) * 16));
#ifdef NFC_CYCLES
    {
        unsigned long long c[12];
        NFC_CUDA_CHECK(cudaMemcpyFromSymbol(c, g_cyc, sizeof(c)));
        fprintf(stderr, "cycles: tile passes %llu in %llu calls (%llu repeats), ring sums after refused tiles %llu, fix-point path %llu, exact path %llu, segment set-up %llu, snapshots %llu, after pipelined runs %llu (its last barrier %llu), loop top %llu, commits %llu\n",
                c[0], c[1], c[5], c[2], c[3], c[4], c[6], c[7], c[8], c[11], c[9], c[10]);
        if (reset) {
            unsigned long long z[12] = {0};
            NFC_CUDA_CHECK(cudaMemcpyToSymbol(g_cyc, z, sizeof(z)));
        }
    }
#endif
    if (reset) {
        unsigned long long z[16] = {0};
        NFC_CUDA_CHECK(cudaMemcpyToSymbol(g_tile_stats, z, sizeof(z)));
    }
    return 0;
}

// CTAs of the slicer kernel that fit on the device at once (for sizing the number of segments)
int slicer_resident_ctas(int L, int kind) {
    int dev = 0, sms = 0, per = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaError_t e = cudaSuccess;
    const void *fn = (const void *)slicer_kernel;
    int threads = SLICER_NT;
    size_t dyn = ((size_t)L * 4 + 15) / 16 * 16;
    if (slicer_streaming_ok(L, kind)) {
        const FastVariant v = fast_variant_of(L, kind);
        fn = v.fn;
        threads = v.threads;
        dyn = v.smem;
    }
    if (raise_dynamic_smem(fn, dyn) == 0) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, fn, threads, dyn);
    if (e != cudaSuccess || per < 1) per = 1;
    return sms * per;
}

// ---------------------------------------------------------------- batches of independent captures
// The reference gives every capture its own transition_sink (transition_sink.py:12-34): the first av_window items fill the
// ring unconditionally, _sum is their left-to-right double sum (transition_sink.py:109-125).  One block per capture writes
// that state as a state block; the ring is laid out by stream position of the batch (capture c starts at c * pitch).
__global__ void __launch_bounds__(256) batch_warm_kernel(const char *__restrict__ items, int64_t stride_bytes, int64_t pitch,
                                                         const SlicerParams *__restrict__ params, char *__restrict__ states,
                                                         size_t state_bytes) {
    extern __shared__ float warm_s[];
    const int64_t c = blockIdx.x;
    const SlicerParams p = params[c];
    const int L = p.L;
    SlicerHdr *h = reinterpret_cast<SlicerHdr *>(states + (size_t)c * state_bytes);
    float *ring = state_ring(h);
    const int64_t B = c * pitch;
    const void *in = items + c * stride_bytes;
    for (int i = threadIdx.x; i < L; i += blockDim.x) {
        const float v = load_one(in, i, p);
        warm_s[i] = v;
        ring[(int)((B + i) % L)] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < L; i++) s += (double)warm_s[i];  // sum(ar), left to right (transition_sink.py:122)
        SlicerHdr hh;
        hh.ss = s;
        hh.pos = B + L;
        hh.lastL = NO_POS;
        hh.lrun_start = NO_POS;
        hh.last_val = 0;
        hh.emin = 0; hh.emax = 0; hh.status = 0; hh.count = 0; hh.pad = 0;
        *h = hh;
    }
}

// class bitmap of positions no segment writes (warm-ups, padding behind the captures): val == 0 everywhere
__global__ void bitmap_fill_kernel(uint4 *__restrict__ bm, size_t n_chunks) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_chunks) return;
    bm[2 * i] = make_uint4(FULL, FULL, FULL, FULL);
    bm[2 * i + 1] = make_uint4(0u, 0u, 0u, 0u);
}

int launch_batch_warm(const void *d_items, int64_t stride_bytes, int64_t pitch, int n_cap, int L, const SlicerParams *d_params,
                      void *d_states, size_t state_bytes, cudaStream_t stream) {
    if (n_cap <= 0) return 0;
    const size_t smem = (size_t)L * 4;
    if (raise_dynamic_smem((const void *)batch_warm_kernel, smem)) return -1;
    batch_warm_kernel<<<n_cap, 256, smem, stream>>>((const char *)d_items, stride_bytes, pitch, d_params, (char *)d_states, state_bytes);
    NFC_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_bitmap_fill(uint32_t *d_bm, size_t n_chunks, cudaStream_t stream) {
    if (!n_chunks) return 0;
    bitmap_fill_kernel<<<(unsigned)((n_chunks + 255) / 256), 256, 0, stream>>>(reinterpret_cast<uint4 *>(d_bm), n_chunks);
    NFC_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_slicer_serial(const SegWork *d_works, int n_works, const SlicerParams *d_params, float *d_ring_scratch,
                         size_t ring_stride, cudaStream_t stream) {
    if (n_works <= 0) return 0;
    slicer_serial_kernel<<<n_works, 32, 0, stream>>>(d_works, d_params, d_ring_scratch, ring_stride);
    NFC_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_seam_compare(const SlicerHdr *const *d_truth, const SlicerHdr *const *d_assumed, const int *d_param_idx,
                        const SlicerParams *d_params, int *d_mismatch, int n, cudaStream_t stream) {
    if (n <= 0) return 0;
    seam_compare_kernel<<<n, 256, 0, stream>>>(d_truth, d_assumed, d_param_idx, d_params, d_mismatch);
    NFC_CUDA_CHECK(cudaGetLastError());
    return 0;
}

}  // namespace nfc
