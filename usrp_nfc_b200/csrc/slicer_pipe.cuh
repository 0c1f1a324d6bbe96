// slicer_pipe.cuh -- the pipelined mode of the streaming slicer (included by slicer_fast.cuh).
//
// Same contract as the synchronous tile loop of slicer_fast_kernel (transition_sink.py:55-82, guessed thresholds that
// are proven afterwards), organised as a producer / consumer pipeline over mbarriers instead of two block barriers
// per tile:
//
//  * NW worker warps classify tile k against guessed thresholds (one guess per warp and tile: the warp's R*128
//    contiguous samples are one chunk), keep what the ring slots will hold in registers, publish one record per warp
//    (fixed-point sum of the admitted x - prev, max |x - prev|, the smallest distance of any sample to a guessed
//    threshold) and the tile's class bitmap, and only then wait for the verdict on tile k-1 and write its ring slots.
//    They never wait for tile k's own verdict before starting tile k+1.
//  * The judge warp (lane = chunk) turns the records of tile k into the window sum at every chunk start as an
//    interval, proves every chunk's guess (the band the true thresholds can lie in is strictly inside guess +- margin),
//    carries the interval on, publishes the guesses of tile k+2, and -- as soon as the workers are done reading a
//    stage -- has one lane issue the bulk copy (cp.async.bulk, completion on an mbarrier) of tile k+S into it.
//  * The mapper warp (lane = 128 samples) derives from the bitmap what the hysteresis needs: whether a HIGH sample
//    follows a LOW sample closely enough for cur_state == 2 to matter (then val != class and the tile is not ours),
//    and the carries (val of the last sample, last LOW sample, start of its run).
//  * Any tile that cannot be proven ends the pipelined run at that tile: nothing of it (or of the tile the workers
//    classified ahead) has been written to the ring, and the synchronous loop settles it (measured guesses, exact
//    fix-point, exact path) before the pipeline is entered again.
//
// Ordering of the ring: the slots tile k writes are read next by tiles >= k + L/T - 1.  A worker writes tile k-1's slots
// before it arrives on rec_full[k]; a worker starts tile k' after the verdict on k'-2, i.e. after every worker's
// arrival on rec_full[k'-2], i.e. after every write of tiles <= k'-3.  Hence L >= 3T is required (checked by the caller).
#pragma once

namespace nfc {

// ---------------------------------------------------------------- mbarrier / bulk copy (PTX)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *b, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_inval(unsigned long long *b) {
    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *b) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *b, unsigned bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(b)), "r"(bytes)
                 : "memory");
}
// Waits for the phase of the given parity to complete (each try_wait suspends the thread for a while).
// A wait that does not end -- a protocol error -- traps instead of hanging the device.
__device__ __forceinline__ void mbar_wait(unsigned long long *b, unsigned parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .u32 n;\n\t"
        "mov.u32 n, 0;\n\t"
        "PIPE_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra PIPE_DONE;\n\t"
        "add.u32 n, n, 1;\n\t"
        "setp.lt.u32 p, n, 0x100000;\n\t"
        "@p bra PIPE_WAIT;\n\t"
        "trap;\n\t"
        "PIPE_DONE:\n\t"
        "}" ::"r"(smem_u32(b)),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy (the TMA unit, no tensor map), completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------- packed float helpers (no `volatile`: free to schedule)
__device__ __forceinline__ void unpack2(unsigned long long v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long sub2(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// min(m, |a|, |b|), NaN if any operand is
__device__ __forceinline__ float min3nan_abs(float m, float a, float b) {
    float r;
    asm("{\n\t.reg .f32 aa, bb;\n\tabs.f32 aa, %2;\n\tabs.f32 bb, %3;\n\tmin.NaN.f32 %0, %1, aa, bb;\n\t}" : "=f"(r) : "f"(m), "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ float max3_abs(float m, float a, float b) {
    float r;
    asm("{\n\t.reg .f32 aa, bb;\n\tabs.f32 aa, %2;\n\tabs.f32 bb, %3;\n\tmax.f32 %0, %1, aa, bb;\n\t}" : "=f"(r) : "f"(m), "f"(a), "f"(b));
    return r;
}

// ---------------------------------------------------------------- shared state of the pipelined mode
struct __align__(16) PipeRec {  // one warp's chunk (R * 128 samples) of one tile
    int S;       // round(sum of admitted (x - prev) / q), summed over the lanes
    float amax;  // max |x - prev| over the admitted samples
    float m;     // min over the samples of the distance to the nearer guessed threshold (NaN: not usable)
    int pad;
};

enum { PIPE_CMD_ENTER = 1, PIPE_CMD_QUIT = 2 };
static const int PIPE_BAR_RUN = 2, PIPE_BAR_PARK = 3;  // named barriers over all threads of the CTA (workers + judge + mapper)
template <int ID, int N>
__device__ __forceinline__ void named_bar_sync() {
    asm volatile("bar.sync %0, %1;" ::"n"(ID), "n"(N) : "memory");
}

template <int NW, int R, int S>
struct __align__(16) PipeShared {
    unsigned long long x_full[S];  // stage s holds the samples of tile k, k % S == s
    unsigned long long rec_full[2];  // all workers have published tile k (k & 1), written tile k-1's ring slots, and are done reading tile k's stage
    unsigned long long verdict[2];   // judge and mapper have judged tile k (k & 1); the guesses of tile k+2 are published
    float4 G[2][NW];                 // per warp of tile k (k & 1): -centre and radius of the guessed thresholds, 1/q
    PipeRec recs[2][NW];
    uint32_t bm[2][NW * R * 8];      // the tile's bitmap words, chunk of 128 samples major (as FastShared::bm)
    int vfail[2], vst2[2];
    int cmd, t0, K, done;            // command to the parked warps; first tile and number of tiles of the run; tiles proven
    int inited, pad_[3];
};

// A stage: the tile's samples, overwritten in place by the undo log (what the ring slots held) while the tile is classified.
// 16-bit samples are narrower than the log's floats: their log follows the samples instead.
template <int NW, int R, int ITEM>
struct PipeStage {
    static const int T = NW * R * FAST_CH;
    static const int log_ofs = ITEM == 4 ? 0 : T * ITEM;
    static const int bytes = log_ofs + T * 4;
};

template <int NW, int R>
struct PipeConsts {
    static const int NC = NW * R;            // chunks of 128 samples per tile
    static const int CHS = R * FAST_CH;      // samples per warp and tile
    static const int T = NW * CHS;           // samples per tile
};

// ---------------------------------------------------------------- workers
// Two samples against the guessed thresholds centre -+ radius (ncg2 = {-centre, -centre}).
struct PipeAcc {
    unsigned long long s2;  // two running sums of n - prev
    float amax, m;
};
__device__ __forceinline__ void pipe_pair(float x0, float x1, float p0, float p1, unsigned long long ncg2, float rg, float nrg, PipeAcc &a,
                                          unsigned &NL0, unsigned &NL1, unsigned &H0, unsigned &H1, float &n0, float &n1) {
    float u0, u1;
    unpack2(add2(pack2(x0, x1), ncg2), u0, u1);
    const bool pnl0 = u0 > nrg, ph0 = u0 > rg, pnl1 = u1 > nrg, ph1 = u1 > rg;
    NL0 = __ballot_sync(FULL, pnl0);
    H0 = __ballot_sync(FULL, ph0);
    NL1 = __ballot_sync(FULL, pnl1);
    H1 = __ballot_sync(FULL, ph1);
    n0 = (pnl0 && !ph0) ? x0 : p0;  // transition_sink.py:75-81: only the MID branch admits the sample
    n1 = (pnl1 && !ph1) ? x1 : p1;
    a.m = min3nan_abs(a.m, fabsf(u0) - rg, fabsf(u1) - rg);
    const unsigned long long dd = sub2(pack2(n0, n1), pack2(p0, p1));
    a.s2 = add2(a.s2, dd);
    float d0, d1;
    unpack2(dd, d0, d1);
    a.amax = max3_abs(a.amax, d0, d1);
}

// Returns the number of tiles of the run that were proven (K when the whole run was); the ring holds exactly those.
// The ring slots are rewritten while a tile is classified; what they held goes to the tile's stage in place of the samples
// (an undo log), so that a refused tile -- and the tile classified ahead of its verdict -- can be taken back.
template <int NW, int R, int S, int KIND>
__device__ __noinline__ int pipe_worker(PipeShared<NW, R, S> &ps, float *ring, char *stage0, const FastPlan &plan, const int L,
                                        const float pcm_scale, const int warp, const int lane) {
    typedef PipeConsts<NW, R> C;
    constexpr int ITEM = KIND == IN_PCM_S16 ? 2 : 4;
    constexpr int stage_bytes = PipeStage<NW, R, ITEM>::bytes;
    constexpr int log_ofs = PipeStage<NW, R, ITEM>::log_ofs;
    const int t0 = ps.t0, K = ps.K;
    int slot_w = (int)((plan.tile0_pos + (int64_t)t0 * C::T + (int64_t)warp * C::CHS + (int64_t)lane * 4) % L);
    const int slot_step = C::T % L;
    char *const xs = stage0 + (warp * C::CHS + lane * 4) * ITEM;   // this thread's samples inside a stage
    char *const ls = stage0 + log_ofs + (warp * C::CHS + lane * 4) * 4;  // this thread's part of the undo log
    uint32_t *bm_g = plan.bm_base + (size_t)t0 * (C::NC * 8) + warp * (R * 8) + lane;
    const int emit_from = plan.t_emit - t0;  // tiles of the run from this one on are written to the bitmap

    auto undo = [&](int stage, int slot) {  // the ring slots of a tile as they were before it
        const char *lg = ls + stage * stage_bytes;
#pragma unroll
        for (int r = 0; r < R; r++) {
            *reinterpret_cast<float4 *>(ring + slot) = *reinterpret_cast<const float4 *>(lg + r * (FAST_CH * 4));
            slot += FAST_CH;
            if (slot >= L) slot -= L;
        }
    };

    int slot_prev = 0, st_prev = 0;
    int st = 0;
    unsigned xph = 0u;
    int k = 0;
#pragma unroll 1
    for (; k < K; k++) {
        const int b = k & 1;
        mbar_wait(&ps.x_full[st], xph);
        const float4 g = ps.G[b][warp];
        const unsigned long long ncg2 = pack2(g.x, g.x);
        const float rg = g.y, nrg = -g.y, invq = g.z;
        const char *xrow = xs + st * stage_bytes;
        char *lrow = ls + st * stage_bytes;
        uint32_t *bms = &ps.bm[b][warp * (R * 8)];
        PipeAcc a;
        a.s2 = 0ull;
        a.amax = 0.0f;
        a.m = INFINITY;
        // all loads of the tile first: the rows' dependency chains overlap (the compiler cannot move a load above a store
        // to shared memory that may alias it)
        float4 xv[R], pv[R];
        int sl[R];
        {
            int s0 = slot_w;
#pragma unroll
            for (int r = 0; r < R; r++) {
                sl[r] = s0;
                if (KIND == IN_PCM_S16) {
                    const short4 sv = *reinterpret_cast<const short4 *>(xrow + r * (FAST_CH * 2));
                    xv[r] = make_float4((float)sv.x, (float)sv.y, (float)sv.z, (float)sv.w);
                } else {
                    xv[r] = *reinterpret_cast<const float4 *>(xrow + r * (FAST_CH * 4));
                }
                pv[r] = *reinterpret_cast<const float4 *>(ring + s0);
                s0 += FAST_CH;
                if (s0 >= L) s0 -= L;
            }
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            float4 x4 = xv[r];
            if (KIND == IN_PCM_S16) {
                x4 = make_float4(env_real(__fdiv_rn(x4.x, pcm_scale)), env_real(__fdiv_rn(x4.y, pcm_scale)),
                                 env_real(__fdiv_rn(x4.z, pcm_scale)), env_real(__fdiv_rn(x4.w, pcm_scale)));
            } else if (KIND == IN_SC16) {
                x4 = env_sc16x4(x4, pcm_scale);  // loaded as 16 raw bytes: four short2
            } else if (KIND == IN_REAL_F32) {
                x4.x = env_real(x4.x); x4.y = env_real(x4.y); x4.z = env_real(x4.z); x4.w = env_real(x4.w);
            }
            const float4 p4 = pv[r];
            unsigned NL[4], H[4];
            float4 n4;
            pipe_pair(x4.x, x4.y, p4.x, p4.y, ncg2, rg, nrg, a, NL[0], NL[1], H[0], H[1], n4.x, n4.y);
            pipe_pair(x4.z, x4.w, p4.z, p4.w, ncg2, rg, nrg, a, NL[2], NL[3], H[2], H[3], n4.z, n4.w);
            *reinterpret_cast<float4 *>(ring + sl[r]) = n4;
            *reinterpret_cast<float4 *>(lrow + r * (FAST_CH * 4)) = p4;
            if (lane == 0) {
                uint4 *bw = reinterpret_cast<uint4 *>(bms + r * 8);
                bw[0] = make_uint4(NL[0], NL[1], NL[2], NL[3]);
                bw[1] = make_uint4(H[0], H[1], H[2], H[3]);
            }
        }
        // the warp's record
        float sa, sb;
        unpack2(a.s2, sa, sb);
        const float ssum = sa + sb;
        float m = a.m;
        if (!(fabsf(ssum) * invq < 4194304.0f)) m = __int_as_float(0x7fc00000);  // the lane's sum does not fit 2^22 steps (or is NaN)
        const int si = __float2int_rn(ssum * invq);
        const int Ssum = __reduce_add_sync(FULL, si);
        const unsigned amax_u = __reduce_max_sync(FULL, __float_as_uint(a.amax));  // amax >= 0: ordered like its bit pattern
        m = redux_min_nan(m);
        // the verdict on tile k-1: no tile is started two ahead of an open verdict (ring ordering, depth of the undo logs)
        if (k > 0) {
            mbar_wait(&ps.verdict[b ^ 1], (unsigned)((k - 1) >> 1) & 1u);
            const volatile int *vf = ps.vfail, *vs = ps.vst2;
            if (vf[b ^ 1] | vs[b ^ 1]) {
                undo(st, slot_w);
                undo(st_prev, slot_prev);
                return k - 1;
            }
        }
        if (lane == 0) {
            PipeRec rc;
            rc.S = Ssum;
            rc.amax = __uint_as_float(amax_u);
            rc.m = m;
            rc.pad = 0;
            ps.recs[b][warp] = rc;
        }
        __syncwarp();
        if (k >= emit_from && lane < R * 8) bm_g[(size_t)k * (C::NC * 8)] = bms[lane];
        if (lane == 0) mbar_arrive(&ps.rec_full[b]);
        slot_prev = slot_w;
        st_prev = st;
        slot_w += slot_step;
        if (slot_w >= L) slot_w -= L;
        if (++st == S) {
            st = 0;
            xph ^= 1u;
        }
    }
    // the last tile of the run
    mbar_wait(&ps.verdict[(K - 1) & 1], (unsigned)((K - 1) >> 1) & 1u);
    {
        const volatile int *vf = ps.vfail, *vs = ps.vst2;
        if (vf[(K - 1) & 1] | vs[(K - 1) & 1]) {
            undo(st_prev, slot_prev);
            return K - 1;
        }
    }
    return K;
}

// ---------------------------------------------------------------- judge
// fixed-point step: a power of two near a_est * 2^-27.  A lane's sum must stay below 2^22 steps (a_est / 32, a_est being an
// upper bound of the tile's sum of |x - prev| of late: 128 times the lane's share), so that the sums of a tile's chunks fit int32.
template <int NTHREADS>
__device__ __forceinline__ bool pipe_step(float a_est, float &q, float &invq) {
    const unsigned ae = (__float_as_uint(a_est) >> 23) & 0xffu;
    const bool ok = ae > 45u && ae < 250u;
    constexpr unsigned QEXP = NTHREADS >= 256 ? 27u : 24u;  // fewer threads: a lane's share of the tile's steps is larger
    const unsigned qe = ok ? ae - QEXP : 127u;
    q = __uint_as_float(qe << 23);
    invq = __uint_as_float((254u - qe) << 23);
    return ok;
}

// The judge is one warp with a serial job per tile: its instruction count and dependency chains bound how fast the
// workers may go.  Everything on the way to the verdict is float / int32 (the double-precision window sum is only touched
// after the verdict is out), per-parity values live in registers and are picked with selects.
//
//  * window sum at the tile's first sample: |true - ssm| <= hw (ssm double, hw float rounded up);
//  * the guesses of tile j+2 are published with the verdict on tile j (the workers start tile j+2 without waiting for
//    anything after that verdict).  They are made from ssm at the start of tile j (known before tile j's records arrive,
//    so its products with lo/L and hi/L are ready) and the drift of tile j (dr): the guessed window sum of chunk c is
//    gss = ssm_j + goff[c], goff[c] = dr * (2 + (c + 1/2) / NW); at tile j+2's start ssm - ssm_j is the drift of tiles j and
//    j+1 (d1 + d2), so (window sum at chunk c's first sample) - gss = (d1 + d2) - goff[c] + c0[c], c0 = exclusive prefix
//    of the chunk sums.  The first two tiles of a run are guessed from the window sum at its start.
template <int NW, int R, int S, int ITEM>
__device__ __noinline__ void pipe_judge(PipeShared<NW, R, S> &ps, FastUni &uni, const FastPlan &plan, const double loL, const double hiL,
                                        char *stage0, const int lane) {
    typedef PipeConsts<NW, R> C;
    constexpr unsigned stage_bytes = PipeStage<NW, R, ITEM>::bytes, tile_bytes = C::T * ITEM;
    const int t0 = ps.t0, K = ps.K;
    const char *src0 = plan.xbase + (int64_t)t0 * tile_bytes;
    int issued = 0;
    if (lane == 0) {
        if (ps.inited) {  // barriers of the previous run: nobody waits on them any more
            for (int s = 0; s < S; s++) mbar_inval(&ps.x_full[s]);
            for (int b = 0; b < 2; b++) {
                mbar_inval(&ps.rec_full[b]);
                mbar_inval(&ps.verdict[b]);
            }
        }
        ps.inited = 1;
        for (int s = 0; s < S; s++) mbar_init(&ps.x_full[s], 1);
        for (int b = 0; b < 2; b++) {
            mbar_init(&ps.rec_full[b], NW);
            mbar_init(&ps.verdict[b], 2);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async();
    }
    for (; issued < S && issued < K; issued++) {
        if (lane == 0) {
            mbar_expect_tx(&ps.x_full[issued], tile_bytes);
            bulk_g2s(stage0 + (size_t)issued * stage_bytes, src0 + (size_t)issued * tile_bytes, tile_bytes, &ps.x_full[issued]);
        }
    }
    // ---- state handed over by the synchronous loop
    const double ss_lo0 = uni.ss_lo, ss_hi0 = uni.ss_hi;
    double ssm = 0.5 * (ss_lo0 + ss_hi0);
    float hw = (__double2float_ru(__dsub_ru(ss_hi0, ssm)) + __double2float_ru(__dsub_ru(ssm, ss_lo0))) * 1.0001f;
    float drift = uni.tot_prev, a_est = uni.a_est;
    if (!(a_est > 0.0f)) a_est = __double2float_rd(ss_lo0) * 0x1p-7f;
    const float loLf = plan.loLf, hiLf = plan.hiLf, hiLs = plan.hiLf * (1.0f + 0x1p-20f);
    const bool act = lane < NW;
    const float fc = ((float)lane + 0.5f) * (1.0f / NW);  // the chunk's middle, in tiles
    float thr_min = 3.0e38f, thr_max = 0.0f;
    // per parity of the tile: guess offsets, guessed thresholds (LOW; HIGH * 2^-19), fixed-point step, guesses usable
    float goff0 = 0.0f, goff1 = 0.0f, gTL0 = 0.0f, gTL1 = 0.0f, gTHs0 = 0.0f, gTHs1 = 0.0f, q0 = 1.0f, q1 = 1.0f;
    bool ok0 = false, ok1 = false;
    // guesses of one tile from a window sum known now, whose products with lo/L and hi/L are TLm and THm: chunk c is taken
    // to see that window sum + dr * (ofs + fc)
    auto prepare = [&](int b, float TLm, float THm, float dr, float ofs, float a_e, bool sane) {
        float q, invq;
        const bool stepok = pipe_step<NW * 32>(a_e, q, invq);
        const float go = dr * (ofs + fc);
        const float TL = fmaf(go, loLf, TLm), TH = fmaf(go, hiLf, THm);
        const float cg = 0.5f * (TL + TH), rg = 0.5f * (TH - TL);
        if (act) ps.G[b][lane] = make_float4(-cg, rg, invq, 0.0f);
        const bool ok = __all_sync(FULL, !act || (TL > 0.0f && rg > 0.0f)) && stepok && sane;
        if (b) { goff1 = go; gTL1 = TL; gTHs1 = TH * 0x1p-19f; q1 = q; ok1 = ok; }
        else { goff0 = go; gTL0 = TL; gTHs0 = TH * 0x1p-19f; q0 = q; ok0 = ok; }
    };
    float TLm = __double2float_rn(ssm * loL), THm = __double2float_rn(ssm * hiL);  // of ssm at the start of the tile being judged
    bool sane;  // the window sum at the start of the tile being judged is positive and in range
    {
        const float ssf = __double2float_rd(ssm);
        sane = ssf - hw > 0.0f && ssf < 1.0e30f && ssf > 1.0e-30f;
        prepare(0, TLm, THm, drift, 0.0f, a_est, sane);
        prepare(1, TLm, THm, drift, 1.0f, a_est, sane);
    }
    float d1 = 0.0f, d2 = 0.0f;  // drifts of the two tiles before the one being judged (0 before the run's start)
    if (lane == 0) {
        ps.vfail[0] = ps.vfail[1] = 0;
        ps.vst2[0] = ps.vst2[1] = 0;
    }
    named_bar_sync<PIPE_BAR_RUN, (NW + 2) * 32>();  // barriers, guesses and flags are set up

    int k = 0, st = 0;
#pragma unroll 1
    for (; k < K; k++) {
        const int b = k & 1;
        const unsigned par = (unsigned)(k >> 1) & 1u;
        const float q = b ? q1 : q0, goff = b ? goff1 : goff0, gTL = b ? gTL1 : gTL0, gTHs = b ? gTHs1 : gTHs0;
        const bool okb = b ? ok1 : ok0;
        mbar_wait(&ps.rec_full[b], par);
        // ---------------------------------------------------------------- on the way to the verdict
        const PipeRec rc = ps.recs[b][act ? lane : 0];
        const int Si = act ? rc.S : 0;
        const float amax = act ? rc.amax : 0.0f;
        int inc = Si;
#pragma unroll
        for (int o = 1; o < NW; o <<= 1) {
            const int v = __shfl_up_sync(FULL, inc, o);
            if (lane >= o) inc += v;
        }
        const int c0i = inc - Si;                            // chunk sums below 2^27 steps each (lane sums below 2^22): no overflow
        const int toti = __shfl_sync(FULL, inc, NW - 1);
        const float c0f = (float)c0i * q, Sf = (float)Si * q;
        // upper bounds of the sums of |x - prev|: of the chunk, of the tile
        const float Ahat = amax * ((float)C::CHS * 1.0001f);
        const float totA = __uint_as_float(__reduce_max_sync(FULL, __float_as_uint(amax))) * ((float)C::T * 1.0002f);
        // error of the measured sums: conversion (half a step per lane and chunk), float rounding (2^-19 of |x - prev|)
        const float Ef = fmaf(totA, 0x1p-19f, (float)(16 * NW) * q) * 1.01f;
        const float dsince = k < 2 ? d1 : d1 + d2;  // ssm - (the window sum the guesses were made from)
        const float slack = (hw + Ef + (fabsf(d1) + fabsf(d2) + fabsf(goff) + fabsf(c0f)) * 0x1p-21f) * 1.001f;
        // inside the chunk the window sum moves within [V, U] of its start: the sums of the negative / positive steps
        const float U = fmaxf(0.5f * (Ahat + Sf), 0.0f) * (1.0f + 0x1p-20f), V = fminf(-0.5f * (Ahat - Sf), 0.0f) * (1.0f + 0x1p-20f);
        const float off = (dsince - goff) + c0f;
        const float dev = fmaxf(fabsf(off + (U + slack)), fabsf(off + (V - slack))) * (1.0f + 0x1p-20f);  // |window sum - guessed| at any sample
        // the guess is proven when no sample lies between it and any value the true threshold can take
        const float need = fmaf(dev, hiLs, gTHs);
        const bool fine = !act || ((rc.m > need) && (gTL - need > 0.0f));
        const bool accept = __all_sync(FULL, fine) && okb;
        // the guesses of tile k + 2, from the window sum at this tile's start: this tile's drift, as much again for tile k + 1
        const float dr = (float)toti * q;
        const float a_new = fmaxf(fmaxf(totA, 0.25f * a_est), __shfl_sync(FULL, gTL, 0) * 0x1p-16f);  // follows the traffic, decays slowly
        const float gTL_k = gTL, gTHs_k = gTHs;
        if (accept) prepare(b, TLm, THm, dr, 2.0f, a_new, sane);
        __syncwarp();
        if (lane == 0) {
            ps.vfail[b] = accept ? 0 : 1;
            mbar_arrive(&ps.verdict[b]);
        }
        // ---------------------------------------------------------------- the verdict is out
        // the window sum after the tile
        const double totd = (double)toti * (double)q;  // exact
        const double ssm2 = ssm + totd;
        const float ssf = __double2float_rd(ssm2);
        const float hw2 = hw + (Ef + ssf * 0x1p-50f + hw * 0x1p-22f) * 1.001f;
        const float TLm2 = __double2float_rn(ssm2 * loL), THm2 = __double2float_rn(ssm2 * hiL);
        mbar_wait(&ps.verdict[b], par);  // the mapper's say
        {
            const volatile int *vs = ps.vst2;
            if (!accept || vs[b]) break;
        }
        // admitted samples lie strictly between the guessed thresholds: one binade of slack either way (exponent audit)
        thr_min = fminf(thr_min, gTL_k * 0.5f);
        thr_max = fmaxf(thr_max, gTHs_k * 0x1p20f);
        ssm = ssm2;
        hw = hw2;
        TLm = TLm2;
        THm = THm2;
        sane = ssf - hw2 > 0.0f && ssf < 1.0e30f && ssf > 1.0e-30f;
        a_est = a_new;
        drift = dr;
        d2 = d1;
        d1 = dr;
        // tile k stands: its stage (the undo log by now) is free for tile k + S
        if (issued < K) {
            if (lane == 0) {
                // the workers' undo log (generic proxy) lies in this stage: it is ordered before this thread by the mbarriers,
                // the bulk copy (async proxy) behind it by the proxy fence
                fence_proxy_async();
                mbar_expect_tx(&ps.x_full[st], tile_bytes);
                bulk_g2s(stage0 + (size_t)st * stage_bytes, src0 + (size_t)issued * tile_bytes, tile_bytes, &ps.x_full[st]);
            }
            issued++;
        }
        if (++st == S) st = 0;
    }
    // ---- hand the state back: the interval after the last proven tile
    for (int j = max(issued - S, 0); j < issued; j++) mbar_wait(&ps.x_full[j % S], (unsigned)(j / S) & 1u);  // no copy in flight
    thr_min = redux_min(thr_min);
    thr_max = -redux_min(-thr_max);
    if (lane == 0) {
        if (k > 0) {
            uni.ss_lo = __dadd_rd(ssm, -(double)hw);
            uni.ss_hi = __dadd_ru(ssm, (double)hw);
            uni.tot_prev = drift;
            uni.a_est = a_est;
            uni.thr_min = fminf(uni.thr_min, thr_min);
            uni.thr_max = fmaxf(uni.thr_max, thr_max);
            uni.stats[FS_FAST] += (unsigned)k;
            uni.stats[FS_PIPE_T] += (unsigned)k;
        }
        ps.done = k;
    }
}

// ---------------------------------------------------------------- mapper
template <int NW, int R, int S>
__device__ __noinline__ void pipe_mapper(PipeShared<NW, R, S> &ps, SegCarry &cs, const FastPlan &plan, const int mx, const int lane) {
    typedef PipeConsts<NW, R> C;
    static_assert(C::NC <= 32, "one lane per chunk of 128 samples");
    const int t0 = ps.t0, K = ps.K;
    int64_t lastL = cs.lastL, lrun_start = cs.lrun_start;
    int last_val = cs.last_val;
    const bool act = lane < C::NC;
    named_bar_sync<PIPE_BAR_RUN, (NW + 2) * 32>();
    int k = 0;
#pragma unroll 1
    for (; k < K; k++) {
        const int b = k & 1;
        const unsigned par = (unsigned)(k >> 1) & 1u;
        mbar_wait(&ps.rec_full[b], par);
        uint4 nl = make_uint4(FULL, FULL, FULL, FULL), hh = make_uint4(0u, 0u, 0u, 0u);
        if (act) {
            nl = *reinterpret_cast<const uint4 *>(&ps.bm[b][lane * 8]);
            hh = *reinterpret_cast<const uint4 *>(&ps.bm[b][lane * 8 + 4]);
        }
        const bool hasL = (nl.x & nl.y & nl.z & nl.w) != FULL, hasH = (hh.x | hh.y | hh.z | hh.w) != 0u;
        const int firstc = (int)((nl.x & 1u) + (hh.x & 1u)), lastc = (int)((nl.w >> 31) + (hh.w >> 31));
        const unsigned Lmask = __ballot_sync(FULL, hasL), Hmask = __ballot_sync(FULL, hasH);
        const int64_t P0 = plan.tile0_pos + (int64_t)(t0 + k) * C::T;
        // hysteresis can matter only if a HIGH sample comes within max_len + 1 samples after a LOW sample
        bool st2 = false;
        if (Hmask) {
            // cheap test by chunks first; only if it fires, to the sample
            const int nb = plan.nb;
            const int lo_c = max(lane - nb, 0);
            const unsigned win = (Lmask >> lo_c) & ((2u << (lane - lo_c)) - 1u);
            bool risk = hasH && win != 0u;
            if (hasH && lastL != NO_POS && P0 + (int64_t)lane * FAST_CH - lastL <= (int64_t)mx + 1) risk = true;
            if (__any_sync(FULL, risk)) {
                const int relC = (lastL != NO_POS && P0 - lastL < (int64_t)(1 << 28)) ? (int)(lastL - P0) : -(1 << 29);
                st2 = hysteresis_risk(nl, hh, hasL, hasH, lane, mx, relC);
            }
        }
        // the carries the tile would leave: val of its last sample, last LOW sample and the start of its run
        int newL = -1, newS = -1;
        if (Lmask) {
            int prevlast = __shfl_up_sync(FULL, lastc, 1);
            if (lane == 0) prevlast = last_val + 1;  // class code of the sample before the tile
            int candL = -1, candS = -1;
            if (hasL && (lastc == 0 || lane >= C::NC - plan.nb)) {
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
        const int lv_new = __shfl_sync(FULL, lastc, C::NC - 1) - 1;
        if (lane == 0) {
            ps.vst2[b] = st2 ? 1 : 0;
            mbar_arrive(&ps.verdict[b]);
        }
        mbar_wait(&ps.verdict[b], par);  // the judge's say
        {
            const volatile int *vf = ps.vfail;
            if (st2 || vf[b]) break;
        }
        last_val = lv_new;
        if (newL >= 0) {
            lastL = P0 + newL;
            if (newS >= 0) lrun_start = P0 + newS;
        }
    }
    if (lane == 0) {
        cs.lastL = lastL;
        cs.lrun_start = lrun_start;
        cs.last_val = last_val;
    }
}

// IQ input has no pipelined mode (a tile of complex samples does not fit beside the ring twice): the extra warps only leave
template <int NW>
__device__ __forceinline__ void pipe_aux_idle_impl(volatile int *cmd) {
    for (;;) {
        named_bar_sync<PIPE_BAR_PARK, (NW + 2) * 32>();
        if (*cmd == PIPE_CMD_QUIT) return;
    }
}
template <int NW, class PS>
__device__ __forceinline__ void pipe_aux_idle(PS &ps) {
    pipe_aux_idle_impl<NW>(&ps.cmd);
}

// The two extra warps of a CTA: parked until the segment's workers enter the pipelined mode (or finish the segment).
template <int NW, int R, int S, int ITEM>
__device__ __forceinline__ void pipe_aux_main(PipeShared<NW, R, S> &ps, FastUni &uni, const FastPlan &plan, const SlicerParams &p, SegCarry &cs,
                                              float *ring, const int warp, const int lane) {
    for (;;) {
        named_bar_sync<PIPE_BAR_PARK, (NW + 2) * 32>();
        if (*(volatile int *)&ps.cmd == PIPE_CMD_QUIT) return;
        char *stage0 = reinterpret_cast<char *>(ring) + (((size_t)p.L * 4 + 15) / 16) * 16;  // the stages follow the ring
        if (warp == NW) pipe_judge<NW, R, S, ITEM>(ps, uni, plan, p.loL, p.hiL, stage0, lane);
        else pipe_mapper<NW, R, S>(ps, cs, plan, p.mx, lane);
        named_bar_sync<PIPE_BAR_RUN, (NW + 2) * 32>();  // the run is over, the state handed back
    }
}

}  // namespace nfc
