// linecode.cu -- events -> symbols -> frames: Manchester / modified-Miller decoding and framing.
//
// Replaces background.run's dispatch (background.py:30-52), manchester_decoder.process_transition
// (manchester.py:30-61), miller_decoder.process_transition (miller.py:153-197) and
// PacketProcessor.append_bit (packets.py:67-79).
//
// Both directions are finite transducers over the event stream:
//   reader machine R = miller state (16) x PacketProcessor._started (2)   fed by type-1 events
//   tag machine    G = manchester state (8) x _started (2)                fed by type-0 events
// (type -1 events and disabled directions are dropped, background.py:30-35).  The stream is cut
// into chunks of CHUNK events; pass A computes each chunk's transfer function (state at the chunk
// start -> state at its end) for every possible start state, an order-preserving scan composes
// them, and passes B/C re-run each chunk from its now known start state to count and to write
// symbols, frame bits and frame-closing records.  How many bits a frame holds (len(self._cur),
// packets.py:64) crosses chunks as a (has_emission, tail) pair combined by the same scan.
#include "common.cuh"
#include "scan.cuh"

#include <algorithm>

namespace nfc {

#ifndef NFC_LC_CHUNK
#define NFC_LC_CHUNK 64
#endif
static const int CHUNK = NFC_LC_CHUNK;
static const int LOOKBACK_LIMIT = 4096;  // events searched backwards for a reset before giving up
static const int RSTATES = 32, GSTATES = 16;

struct __align__(16) ChunkMap {
    uint8_t r[RSTATES];
    uint8_t g[GSTATES];
};
struct ComposeMap {  // (a then b)
    __device__ __forceinline__ ChunkMap operator()(const ChunkMap &a, const ChunkMap &b) const {
        ChunkMap c;
#pragma unroll
        for (int s = 0; s < RSTATES; s++) c.r[s] = b.r[a.r[s] & 31];
#pragma unroll
        for (int s = 0; s < GSTATES; s++) c.g[s] = b.g[a.g[s] & 15];
        return c;
    }
};

// Counts of a run of events.  nemit counts the frame closings that get a record: a frame that closes without a bit is not
// forwarded (packets.py:97) and gets none.  Whether the FIRST closing of a type in the run is such a frame can depend on the
// bits pending before the run: hasT bit 0 = the run closes a frame of type T (or a capture ends in it: nothing pending
// behind that), bit 1 = its first closing has no bit of the run before it and no capture end -- it is counted in nemit
// and is empty if and only if nothing is pending when the run begins (resolved when runs are combined, and against the
// slab's pending_in at last).
struct __align__(16) ChunkCnt {
    uint32_t nsym, nbit0, nbit1, nemit;
    uint32_t has0, tail0, has1, tail1;  // tailT: bits appended after the run's last closing (or all, if none)
};
struct CombineCnt {
    __device__ __forceinline__ ChunkCnt operator()(const ChunkCnt &a, const ChunkCnt &b) const {
        ChunkCnt c;
        c.nsym = a.nsym + b.nsym;
        c.nbit0 = a.nbit0 + b.nbit0;
        c.nbit1 = a.nbit1 + b.nbit1;
        c.nemit = a.nemit + b.nemit;
        if (a.has0 & 1) {
            if ((b.has0 & 2) && a.tail0 == 0) c.nemit--;  // b's first closing of type 0 is empty
            c.has0 = a.has0;
        } else {
            c.has0 = (b.has0 & 1) | (((b.has0 & 2) && a.tail0 == 0) ? 2u : 0u);
        }
        if (a.has1 & 1) {
            if ((b.has1 & 2) && a.tail1 == 0) c.nemit--;
            c.has1 = a.has1;
        } else {
            c.has1 = (b.has1 & 1) | (((b.has1 & 2) && a.tail1 == 0) ? 2u : 0u);
        }
        c.tail0 = (b.has0 & 1) ? b.tail0 : a.tail0 + b.tail0;
        c.tail1 = (b.has1 & 1) ? b.tail1 : a.tail1 + b.tail1;
        return c;
    }
};
// records before a run whose counts are pc, in a slab that begins with pending[] bits pending
__device__ __forceinline__ uint32_t resolved_records(const ChunkCnt &pc, const uint32_t *pending) {
    return pc.nemit - (((pc.has0 & 2) && pending[0] == 0) ? 1u : 0u) - (((pc.has1 & 2) && pending[1] == 0) ? 1u : 0u);
}

// The number of events of a slab is read from device memory (left there by the run kernels' scan), so that the host can
// queue the line-code kernels without waiting for it; cap sizes grids and buffers (more events than that: POST_OVF_EVENTS,
// raised by run_write_kernel, and the host does the slab again).
struct EvCount {
    const uint32_t *d_M;
    uint32_t cap;
    __device__ __forceinline__ uint32_t n() const { return min(*d_M, cap); }
};

struct TabView {
    const uint8_t *dcm, *dcg;       // duration classes (global)
    const TabEntry *tab;            // tables (one shared memory copy: Miller, then Manchester at goff)
    int goff;
    int use_reader, use_tag;
    // batches of captures (LineTables::batch_*); caps == nullptr: one stream
    const int64_t *caps;
    int64_t base;
    int n_caps, c0;
    uint32_t skip;
};

// Batches of captures: which capture an event belongs to, and whether it is one of the capture's own events.  Events come
// in position order, so a walk over events keeps a cursor in the capture table: one binary search where the walk begins,
// then a step to the next capture whenever an event passes its start.
struct CapCursor {
    int k;             // capture of the last event walked over (c0 - 1 before the slab's first event)
    uint32_t lo, hi;   // its own events: slab-relative positions [start + skip, start + length)
    uint32_t next;     // slab-relative start of capture k + 1
};
__device__ __forceinline__ uint32_t cap_rel(const TabView &tv, int64_t p) {  // batch position -> slab-relative (clamped)
    const int64_t r = p - tv.base;
    return r < 0 ? 0u : (r > (int64_t)0xffffffffu ? 0xffffffffu : (uint32_t)r);
}
__device__ __forceinline__ void cap_load(const TabView &tv, CapCursor &cc, int k) {
    const int64_t s = tv.caps[k], len = tv.caps[tv.n_caps + 1 + k];
    cc.k = k;
    cc.lo = cap_rel(tv, s + tv.skip);
    cc.hi = cap_rel(tv, s + len);
    cc.next = cap_rel(tv, tv.caps[k + 1]);
}
// the cursor at the capture of event i - 1 (before the slab's first capture when i == 0: a slab starts with a capture)
__device__ __forceinline__ void cap_seek(const TabView &tv, CapCursor &cc, const EventRec *__restrict__ ev, int64_t i) {
    if (i <= 0) {
        cc.k = tv.c0 - 1;
        cc.lo = cc.hi = cc.next = 0;
        return;
    }
    const int64_t p = tv.base + (int64_t)ev[i - 1].rel_pos;
    int lo = tv.c0, hi = tv.n_caps - 1;  // the last capture that starts at or before p (empty captures start where the next does)
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (tv.caps[mid] <= p) lo = mid;
        else hi = mid - 1;
    }
    cap_load(tv, cc, lo);
}
// moves the cursor to the capture of an event at rel_pos; true when that is another capture than the last event's
__device__ __forceinline__ bool cap_step(const TabView &tv, CapCursor &cc, uint32_t rel_pos, bool &inside) {
    bool changed = false;
    while (rel_pos >= cc.next && cc.k + 1 < tv.n_caps) {
        cap_load(tv, cc, cc.k + 1);
        changed = true;
    }
    inside = rel_pos >= cc.lo && rel_pos < cc.hi;
    return changed;
}

// one symbol into a PacketProcessor (packets.py:67-79); returns 1 when a frame is closed
template <class Sink>
__device__ __forceinline__ void framer_put(int &started, int o, int type, uint32_t pos, Sink &sink) {
    const int start_bit = type == 0 ? 1 : 0;  // packets.py:24-30
    sink.symbol(pos, type, o);
    if (o >= 2) {
        if (started) {
            sink.emission(pos, type);
            started = 0;
        }
    } else if (!started && o == start_bit) {
        started = 1;
    } else {
        sink.bit(type, o);
    }
}

// one event through the machine it belongs to; rs/gs are the R and G machine states.  One code path for both
// directions (table offset, state width and duration classes selected by the event's type): the lanes of a warp walk
// different chunks, so reader and tag events meet in every step and separate branches would both be executed.
template <class Sink>
__device__ __forceinline__ void step_event(const EventRec &ev, const TabView &tv, int &rs, int &gs, Sink &sink) {
    const bool is_r = ev.type == 1;
    if (!(is_r ? tv.use_reader != 0 : (ev.type == 0 && tv.use_tag != 0))) return;
    const uint8_t *dc = is_r ? tv.dcm : tv.dcg;
    const int nst = is_r ? MILLER_STATES : MANCH_STATES, sh = is_r ? 4 : 3;
    const int st = is_r ? rs : gs;
    const TabEntry e = tv.tab[(is_r ? 0 : tv.goff) + ((int)dc[ev.d] * 4 + (ev.v + 1)) * nst + (st & (nst - 1))];
    int started = st >> sh;
    const int n = tab_nout(e), type = is_r ? 1 : 0;
    if (n > 0) framer_put(started, tab_out0(e), type, ev.rel_pos, sink);
    if (n > 1 && is_r) framer_put(started, tab_out1(e), type, ev.rel_pos, sink);  // only the Miller decoder emits two symbols
    const int nx = (tab_next(e) & (nst - 1)) | (started << sh);
    rs = is_r ? nx : rs;
    gs = is_r ? gs : nx;
}

// the same for a stream that may be a batch of captures: a capture's first event finds everything as new
// (background.py:17-25, packets.py:63-65), events outside a capture's own range are ignored.  The kernels are instantiated
// for single streams (BATCH = false: no capture lookup in the event loops) and for batches.
template <bool BATCH, class Sink>
__device__ __forceinline__ void step_event_batch(const EventRec &ev, const TabView &tv, int &rs, int &gs, Sink &sink, CapCursor &cur) {
    if (BATCH) {
        bool inside;
        if (cap_step(tv, cur, ev.rel_pos, inside)) {
            rs = 0;
            gs = 0;
            sink.new_capture();
        }
        if (!inside) return;
    }
    step_event(ev, tv, rs, gs, sink);
}

// eight events at once (one 64-byte line): the loops below are chains of dependent loads otherwise.
// `base` is a multiple of 8; the event buffer is padded, so reading a little past n_ev is safe.
__device__ __forceinline__ void load8(const EventRec *__restrict__ ev, int64_t base, EventRec (&e)[8]) {
    // In 64-bit lanes, so that the single-stream kernels, which read no positions, still load 16 bytes at a time: with
    // 32-bit lanes the compiler drops the position words and issues eight 4-byte loads, which made the chains slower.
    const ulonglong2 *p = reinterpret_cast<const ulonglong2 *>(ev + base);
    const ulonglong2 q[4] = {__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3)};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const unsigned long long w[2] = {q[k].x, q[k].y};
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const unsigned hi = (unsigned)(w[h] >> 32);
            EventRec r;
            r.rel_pos = (unsigned)w[h];
            r.d = (uint16_t)(hi & 0xffffu);
            r.v = (int8_t)((hi >> 16) & 0xffu);
            r.type = (int8_t)(hi >> 24);
            e[2 * k + h] = r;
        }
    }
}

struct NullSink {
    __device__ __forceinline__ void symbol(uint32_t, int, int) {}
    __device__ __forceinline__ void emission(uint32_t, int) {}
    __device__ __forceinline__ void bit(int, int) {}
    __device__ __forceinline__ void new_capture() {}
};

__device__ __forceinline__ void load_tables(const LineTables &lt, TabEntry *sm, TabEntry *sg) {  // sg follows sm
    for (int i = threadIdx.x; i < lt.n_dclass_miller * 4 * MILLER_STATES; i += blockDim.x) sm[i] = lt.miller[i];
    for (int i = threadIdx.x; i < lt.n_dclass_manch * 4 * MANCH_STATES; i += blockDim.x) sg[i] = lt.manch[i];
    __syncthreads();
}

#define NFC_TABLE_SMEM                                              \
    __shared__ TabEntry s_tab[MAX_DCLASS * 4 * (MILLER_STATES + MANCH_STATES)]; \
    load_tables(lt, s_tab, s_tab + MAX_DCLASS * 4 * MILLER_STATES); \
    TabView tv;                                                     \
    tv.dcm = lt.dclass_miller; tv.dcg = lt.dclass_manch;            \
    tv.tab = s_tab; tv.goff = MAX_DCLASS * 4 * MILLER_STATES;        \
    tv.use_reader = lt.decode_reader; tv.use_tag = lt.decode_tag;   \
    tv.caps = lt.batch_tab; tv.base = lt.batch_base; tv.n_caps = (int)lt.batch_n; tv.c0 = (int)lt.batch_c0; tv.skip = lt.batch_skip;

// ---- pass A: transfer function of every chunk -------------------------------------------------
template <bool BATCH>
__global__ void chunk_map_kernel(const EventRec *__restrict__ ev, EvCount evc, LineTables lt,
                                 ChunkMap *__restrict__ maps, uint32_t cap_chunks) {
    NFC_TABLE_SMEM
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n_ev = evc.n();
    if (c >= cap_chunks) return;
    const uint32_t i0 = min(n_ev, c * CHUNK), i1 = min(n_ev, i0 + CHUNK);  // behind the last event: the identity
    uint8_t r[RSTATES], g[GSTATES];
    for (int s = 0; s < RSTATES; s++) r[s] = (uint8_t)s;
    for (int s = 0; s < GSTATES; s++) g[s] = (uint8_t)s;
    bool r_flat = false, g_flat = false;  // all start states already lead to the same state
    NullSink sink;
    CapCursor cur;
    if (BATCH) cap_seek(tv, cur, ev, (int64_t)i0);
    for (uint32_t i = i0; i < i1; i++) {
        const EventRec e = ev[i];
        if (BATCH) {
            bool inside;
            if (cap_step(tv, cur, e.rel_pos, inside)) {  // a new capture: every state leads to the initial one
                r[0] = 0; g[0] = 0;
                r_flat = g_flat = true;
            }
            if (!inside) continue;
        }
        if (e.type == 1 && tv.use_reader) {
            if (r_flat) {
                int rs = r[0], gs = 0;
                step_event(e, tv, rs, gs, sink);
                r[0] = (uint8_t)rs;
            } else {
                bool same = true;
                int first = 0;
                for (int s = 0; s < RSTATES; s++) {
                    int rs = r[s], gs = 0;
                    step_event(e, tv, rs, gs, sink);
                    r[s] = (uint8_t)rs;
                    if (s == 0) first = rs;
                    same = same && (rs == first);
                }
                r_flat = same;
            }
        } else if (e.type == 0 && tv.use_tag) {
            if (g_flat) {
                int rs = 0, gs = g[0];
                step_event(e, tv, rs, gs, sink);
                g[0] = (uint8_t)gs;
            } else {
                bool same = true;
                int first = 0;
                for (int s = 0; s < GSTATES; s++) {
                    int rs = 0, gs = g[s];
                    step_event(e, tv, rs, gs, sink);
                    g[s] = (uint8_t)gs;
                    if (s == 0) first = gs;
                    same = same && (gs == first);
                }
                g_flat = same;
            }
        }
    }
    ChunkMap m;
    for (int s = 0; s < RSTATES; s++) m.r[s] = r_flat ? r[0] : r[s];
    for (int s = 0; s < GSTATES; s++) m.g[s] = g_flat ? g[0] : g[s];
    maps[c] = m;
}

// ---- pass B: counts per chunk from the true start state -------------------------------------
struct CountSink {
    ChunkCnt c;
    __device__ __forceinline__ void symbol(uint32_t, int, int) { c.nsym++; }
    __device__ __forceinline__ void emission(uint32_t, int type) {
        uint32_t &has = type == 0 ? c.has0 : c.has1;
        uint32_t &tail = type == 0 ? c.tail0 : c.tail1;
        if (tail != 0) c.nemit++;                      // a frame with bits
        else if (!(has & 1)) { c.nemit++; has |= 2; }  // empty if nothing is pending before the chunk (ChunkCnt)
        has |= 1;                                      // (else: empty for certain -- no record)
        tail = 0;
    }
    __device__ __forceinline__ void bit(int type, int) {
        if (type == 0) { c.nbit0++; c.tail0++; } else { c.nbit1++; c.tail1++; }
    }
    __device__ __forceinline__ void new_capture() {  // the bits appended so far belong to no later frame
        c.has0 |= 1; c.tail0 = 0;
        c.has1 |= 1; c.tail1 = 0;
    }
};

// ---- frame-boundary search: the state at a chunk start from the nearest reset before it ------------
// An event whose duration is out of range resets its decoder whatever the state was (tables.cpp, reset_*).
// Pass 1 (chunk_summary_kernel): every chunk walks its own events once from an unknown state; after the first reset
// of a direction its state is known, and so is the state the chunk leaves behind.  summary[c] = R state | known << 5 |
// G state << 8 | known << 12.
// Pass 2 (chunk_start_kernel): a chunk looks back over the *summaries* for the nearest chunk that leaves a known state
// (per direction) and replays only the events between that chunk's end and its own start (none when it is the previous
// chunk).  start[c] = R state | G state << 8.  Chunks that find nothing within LOOKBACK_LIMIT events raise *unresolved
// (the host then takes the transfer-function scan below for the slab).
template <bool BATCH>
__global__ void chunk_summary_kernel(const EventRec *__restrict__ ev, EvCount evc, LineTables lt,
                                     uint16_t *__restrict__ summary) {
    NFC_TABLE_SMEM
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n_ev = evc.n(), n_chunks = (n_ev + CHUNK - 1) / CHUNK;
    if (c >= n_chunks) return;
    int rs = 0, gs = 0;
    bool kR = false, kG = false;
    NullSink sink;
    const uint32_t i0 = c * CHUNK, i1 = min(n_ev, i0 + CHUNK);
    CapCursor cur;
    if (BATCH) cap_seek(tv, cur, ev, (int64_t)i0);
    for (uint32_t i = i0; i < i1; i += 8) {
        EventRec e8[8];
        load8(ev, i, e8);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            if (i + k >= i1) continue;
            const EventRec e = e8[k];
            int dummy = 0;
            if (BATCH) {
                bool inside;
                if (cap_step(tv, cur, e.rel_pos, inside)) {  // a new capture: both machines are known to be in their initial state
                    rs = 0; kR = true;
                    gs = 0; kG = true;
                }
                if (!inside) continue;
            }
            if (e.type == 1 && tv.use_reader) {
                const uint8_t r = lt.reset_miller[(int)tv.dcm[e.d] * 4 + (e.v + 1)];
                if (r != 0xFF) { rs = r; kR = true; }
                else if (kR) step_event(e, tv, rs, dummy, sink);
            } else if (e.type == 0 && tv.use_tag) {
                const uint8_t r = lt.reset_manch[(int)tv.dcg[e.d] * 4 + (e.v + 1)];
                if (r != 0xFF) { gs = r; kG = true; }
                else if (kG) step_event(e, tv, dummy, gs, sink);
            }
        }
    }
    summary[c] = (uint16_t)((rs & 31) | (kR ? 32 : 0) | ((gs & 15) << 8) | (kG ? 4096 : 0));
}

template <bool BATCH>
__global__ void chunk_start_kernel(const EventRec *__restrict__ ev, EvCount evc, LineTables lt,
                                   const DecCarry *__restrict__ carry_in, const uint16_t *__restrict__ summary,
                                   uint16_t *__restrict__ start, uint32_t *__restrict__ flags) {
    NFC_TABLE_SMEM
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n_ev = evc.n(), n_chunks = (n_ev + CHUNK - 1) / CHUNK;
    if (c >= n_chunks) return;
    const DecCarry carry = *carry_in;
    int rs = (carry.miller_state & 15) | ((carry.started[1] & 1) << 4);
    int gs = (carry.manch_state & 7) | ((carry.started[0] & 1) << 3);
    const int64_t i0 = (int64_t)c * CHUNK;
    bool foundR = !tv.use_reader, foundG = !tv.use_tag;
    int64_t iR = -1, iG = -1;  // last event already accounted for (-1: replay from event 0 with the carry)
    int64_t cc = (int64_t)c - 1;
    const int64_t cmin = max((int64_t)0, (int64_t)c - LOOKBACK_LIMIT / CHUNK);
    for (; cc >= cmin && !(foundR && foundG); cc--) {
        const unsigned sm = summary[cc];
        if (!foundR && (sm & 32u)) { foundR = true; iR = (cc + 1) * CHUNK - 1; rs = (int)(sm & 31u); }
        if (!foundG && (sm & 4096u)) { foundG = true; iG = (cc + 1) * CHUNK - 1; gs = (int)((sm >> 8) & 15u); }
    }
    if (cc >= 0 && !(foundR && foundG)) {  // gave up before the first chunk: the carry cannot be used either
        atomicOr(flags, (uint32_t)POST_UNRESOLVED);
        start[c] = 0;
        return;
    }
    NullSink sink;
    // replay from the earliest point a still-unknown machine needs (a disabled direction needs nothing)
    const int64_t fromR = tv.use_reader ? iR + 1 : i0, fromG = tv.use_tag ? iG + 1 : i0;
    const int64_t from = fromR < fromG ? fromR : fromG;
    CapCursor cur;
    if (BATCH && from < i0) cap_seek(tv, cur, ev, from);
    for (int64_t base = from & ~(int64_t)7; base < i0; base += 8) {
        EventRec e8[8];
        load8(ev, base, e8);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int64_t kk = base + k;
            if (kk < from || kk >= i0) continue;
            const EventRec e = e8[k];
            int dummy_r = 0, dummy_g = 0;
            if (BATCH) {
                bool inside;
                if (cap_step(tv, cur, e.rel_pos, inside)) {  // a new capture behind the point a machine's state was known at: initial state
                    if (kk > iR) rs = 0;
                    if (kk > iG) gs = 0;
                }
                if (!inside) continue;
            }
            if (e.type == 1) {
                if (kk > iR) step_event(e, tv, rs, dummy_g, sink);
            } else if (e.type == 0) {
                if (kk > iG) step_event(e, tv, dummy_r, gs, sink);
            }
        }
    }
    start[c] = (uint16_t)(rs | (gs << 8));
}

// start states from the composed transfer functions (fallback path)
__global__ void chunk_start_from_maps_kernel(const ChunkMap *__restrict__ prefix, const DecCarry *__restrict__ carry_in,
                                             uint16_t *__restrict__ start, uint32_t n_chunks) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chunks) return;
    const DecCarry carry = *carry_in;
    const int rs0 = (carry.miller_state & 15) | ((carry.started[1] & 1) << 4);
    const int gs0 = (carry.manch_state & 7) | ((carry.started[0] & 1) << 3);
    start[c] = (uint16_t)(prefix[c].r[rs0] | (prefix[c].g[gs0] << 8));
}

template <bool BATCH>
__global__ void chunk_count_kernel(const EventRec *__restrict__ ev, EvCount evc, LineTables lt,
                                   const uint16_t *__restrict__ start, ChunkCnt *__restrict__ cnts, uint32_t cap_chunks) {
    NFC_TABLE_SMEM
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n_ev = evc.n(), n_chunks = (n_ev + CHUNK - 1) / CHUNK;
    if (c >= cap_chunks) return;
    CountSink sink;
    sink.c = ChunkCnt{0, 0, 0, 0, 0, 0, 0, 0};
    if (c >= n_chunks) {  // behind the slab's last event: nothing (the scan runs over the capacity)
        cnts[c] = sink.c;
        return;
    }
    int rs = start[c] & 31, gs = (start[c] >> 8) & 15;
    const uint32_t i0 = c * CHUNK, i1 = min(n_ev, i0 + CHUNK);
    CapCursor cur;
    if (BATCH) cap_seek(tv, cur, ev, (int64_t)i0);
    for (uint32_t i = i0; i < i1; i += 8) {
        EventRec e[8];
        load8(ev, i, e);
#pragma unroll
        for (int k = 0; k < 8; k++)
            if (i + k < i1) step_event_batch<BATCH>(e[k], tv, rs, gs, sink, cur);
    }
    cnts[c] = sink.c;
}

// ---- pass C: write symbols, frame bits and frame records --------------------------------
// A frame record is final as the device writes it (the layout of nfc_frame): closing position in stream coordinates, offset of
// the frame's first bit in the stream's bit arena of its type (all bits of a type in append order: bits_base[t] of them before
// this slab), length, type.  An empty frame (packets.py:97: not forwarded) gets no record (the counts of pass B leave it out:
// ChunkCnt) and is counted in *n_empty; the records go to their final place in host memory by DMA alone.
struct WriteSink {
    SymbolRec *sym;
    uint8_t *bits0, *bits1;
    FrameRec *fr;
    unsigned long long *fx;
    uint32_t *n_empty;
    int64_t a;
    unsigned long long base0, base1;
    uint32_t isym, ib0, ib1, iem;
    uint32_t pend0, pend1;
    uint32_t cap_sym, cap_b0, cap_b1, cap_em;
    __device__ __forceinline__ void symbol(uint32_t pos, int type, int o) {
        if (sym && isym < cap_sym) {
            SymbolRec s;
            s.rel_pos = pos; s.type = (int8_t)type; s.val = (int8_t)o; s.pad = 0;
            sym[isym] = s;
        }
        isym++;
    }
    __device__ __forceinline__ void emission(uint32_t pos, int type) {
        const uint32_t nbits = type == 0 ? pend0 : pend1;
        if (nbits == 0) {  // not forwarded (packets.py:97): no record -- the counts knew (ChunkCnt)
            atomicAdd(n_empty, 1u);
            return;
        }
        if (iem < cap_em) {
            FrameRec f;
            f.pos = a + (int64_t)pos;
            f.bit_off = (int64_t)((type == 0 ? base0 + ib0 : base1 + ib1) - nbits);  // frames of one type are back to back
            f.nbits = (int32_t)nbits;
            f.type = type;
            fr[iem] = f;
            fx[iem] = ((unsigned long long)f.pos << 24) | ((unsigned long long)nbits << 8) | (unsigned long long)type;
        }
        if ((((unsigned long long)(a + (int64_t)pos)) >> 40) || nbits >= 65536u) atomicOr(n_empty, 0x80000000u);  // does not fit the packed index
        iem++;
        if (type == 0) pend0 = 0; else pend1 = 0;
    }
    __device__ __forceinline__ void bit(int type, int o) {
        if (type == 0) { if (ib0 < cap_b0) bits0[ib0] = (uint8_t)o; ib0++; pend0++; }
        else { if (ib1 < cap_b1) bits1[ib1] = (uint8_t)o; ib1++; pend1++; }
    }
    __device__ __forceinline__ void new_capture() { pend0 = 0; pend1 = 0; }
};

struct LineOut {
    SymbolRec *sym;
    uint8_t *bits0, *bits1;
    FrameRec *fr;
    unsigned long long *fx;       // packed frame index beside the records: pos << 24 | nbits << 8 | type
    uint32_t cap_sym, cap_b0, cap_b1, cap_em;
    const uint32_t *pending_in;   // len(_cur) of each PacketProcessor at the slab start (device memory: [2])
    int64_t a;                    // stream position of the slab's first sample
    const unsigned long long *bits_in;  // bits of each type appended before this slab (device memory: [2]) ...
    unsigned long long *bits_out;       // ... and behind it
    uint32_t *n_empty;
    uint32_t *n_frames;                 // records written (the scan's total may count one more per type: ChunkCnt)
};

template <bool BATCH>
__global__ void chunk_write_kernel(const EventRec *__restrict__ ev, EvCount evc, LineTables lt,
                                   const uint16_t *__restrict__ start,
                                   const ChunkCnt *__restrict__ cnt_prefix, LineOut out, const DecCarry *__restrict__ carry_in,
                                   DecCarry *__restrict__ carry_out, uint32_t *__restrict__ pending_out) {
    NFC_TABLE_SMEM
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n_ev = evc.n(), n_chunks = (n_ev + CHUNK - 1) / CHUNK;
    if (n_chunks == 0 && c == 0) {  // a slab without events hands the carries on as they came
        *carry_out = *carry_in;
        pending_out[0] = out.pending_in[0];
        pending_out[1] = out.pending_in[1];
        out.bits_out[0] = out.bits_in[0];
        out.bits_out[1] = out.bits_in[1];
    }
    if (c >= n_chunks) return;
    int rs = start[c] & 31, gs = (start[c] >> 8) & 15;
    const ChunkCnt pc = cnt_prefix[c];
    WriteSink sink;
    sink.sym = out.sym; sink.bits0 = out.bits0; sink.bits1 = out.bits1; sink.fr = out.fr; sink.fx = out.fx;
    sink.n_empty = out.n_empty; sink.a = out.a; sink.base0 = out.bits_in[0]; sink.base1 = out.bits_in[1];
    sink.cap_sym = out.cap_sym; sink.cap_b0 = out.cap_b0; sink.cap_b1 = out.cap_b1; sink.cap_em = out.cap_em;
    sink.isym = pc.nsym; sink.ib0 = pc.nbit0; sink.ib1 = pc.nbit1; sink.iem = resolved_records(pc, out.pending_in);
    sink.pend0 = (pc.has0 & 1) ? pc.tail0 : out.pending_in[0] + pc.tail0;
    sink.pend1 = (pc.has1 & 1) ? pc.tail1 : out.pending_in[1] + pc.tail1;
    const uint32_t i0 = c * CHUNK, i1 = min(n_ev, i0 + CHUNK);
    CapCursor cur;
    if (BATCH) cap_seek(tv, cur, ev, (int64_t)i0);
    for (uint32_t i = i0; i < i1; i += 8) {
        EventRec e[8];
        load8(ev, i, e);
#pragma unroll
        for (int k = 0; k < 8; k++)
            if (i + k < i1) step_event_batch<BATCH>(e[k], tv, rs, gs, sink, cur);
    }
    if (c == n_chunks - 1) {
        DecCarry co;
        co.miller_state = rs & 15; co.started[1] = rs >> 4;
        co.manch_state = gs & 7; co.started[0] = gs >> 3;
        *carry_out = co;
        pending_out[0] = sink.pend0;
        pending_out[1] = sink.pend1;
        out.bits_out[0] = sink.base0 + sink.ib0;  // the last chunk's counters are the slab's totals
        out.bits_out[1] = sink.base1 + sink.ib1;
        *out.n_frames = sink.iem;
    }
}

// ---- host launchers ------------------------------------------------------------------------------
uint32_t linecode_chunks(uint32_t n_ev) { return (n_ev + CHUNK - 1) / CHUNK; }
size_t linecode_map_bytes() { return sizeof(ChunkMap); }
size_t linecode_cnt_bytes() { return sizeof(ChunkCnt); }
size_t linecode_emission_bytes() { return sizeof(FrameRec); }
size_t linecode_scratch_bytes(uint32_t n_chunks) {
    return scan_scratch_elems(n_chunks) * sizeof(ChunkMap) + scan_scratch_elems(n_chunks) * sizeof(ChunkCnt);
}

// Start states by frame-boundary search; POST_UNRESOLVED in *d_flags afterwards means the caller must use the scan path.
// d_M / cap_ev: see EvCount.  d_carry_in: the decoder state the slab before left on the device.
int launch_linecode_start(const EventRec *d_ev, const uint32_t *d_M, uint32_t cap_ev, const LineTables &lt, const DecCarry *d_carry_in,
                          uint16_t *d_summary, uint16_t *d_start, uint32_t *d_flags, cudaStream_t stream) {
    const uint32_t nc = std::max(1u, linecode_chunks(cap_ev));
    const EvCount evc{d_M, cap_ev};
    (lt.batch_tab ? chunk_summary_kernel<true> : chunk_summary_kernel<false>)<<<(nc + 127) / 128, 128, 0, stream>>>(d_ev, evc, lt, d_summary);
    NFC_CUDA_CHECK(cudaGetLastError());
    (lt.batch_tab ? chunk_start_kernel<true> : chunk_start_kernel<false>)<<<(nc + 127) / 128, 128, 0, stream>>>(d_ev, evc, lt, d_carry_in, d_summary, d_start, d_flags);
    NFC_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// Start states by composing chunk transfer functions (always applicable).
int launch_linecode_start_scan(const EventRec *d_ev, const uint32_t *d_M, uint32_t cap_ev, const LineTables &lt,
                               const DecCarry *d_carry_in, void *d_maps, void *d_prefix, void *d_scratch, uint16_t *d_start,
                               cudaStream_t stream) {
    const uint32_t nc = std::max(1u, linecode_chunks(cap_ev));
    ChunkMap *maps = (ChunkMap *)d_maps, *prefix = (ChunkMap *)d_prefix;
    const unsigned nb = (nc + 127) / 128;
    const EvCount evc{d_M, cap_ev};
    (lt.batch_tab ? chunk_map_kernel<true> : chunk_map_kernel<false>)<<<nb, 128, 0, stream>>>(d_ev, evc, lt, maps, nc);
    NFC_CUDA_CHECK(cudaGetLastError());
    ChunkMap ident;
    for (int s = 0; s < RSTATES; s++) ident.r[s] = (uint8_t)s;
    for (int s = 0; s < GSTATES; s++) ident.g[s] = (uint8_t)s;
    if (device_exclusive_scan<ChunkMap, ComposeMap>(maps, prefix, nc, ident, ComposeMap(), (ChunkMap *)d_scratch, nullptr, stream))
        return -1;
    chunk_start_from_maps_kernel<<<nb, 128, 0, stream>>>(prefix, d_carry_in, d_start, nc);
    NFC_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// Counts per chunk from the start states, scanned into d_cnt_prefix; totals in *d_total.
int launch_linecode_count(const EventRec *d_ev, const uint32_t *d_M, uint32_t cap_ev, const LineTables &lt, const uint16_t *d_start,
                          void *d_cnts, void *d_cnt_prefix, void *d_scratch, void *d_total, cudaStream_t stream) {
    const uint32_t nc = std::max(1u, linecode_chunks(cap_ev));
    ChunkCnt *cnts = (ChunkCnt *)d_cnts, *cprefix = (ChunkCnt *)d_cnt_prefix;
    const EvCount evc{d_M, cap_ev};
    (lt.batch_tab ? chunk_count_kernel<true> : chunk_count_kernel<false>)<<<(nc + 127) / 128, 128, 0, stream>>>(d_ev, evc, lt, d_start, cnts, nc);
    NFC_CUDA_CHECK(cudaGetLastError());
    ChunkCnt zero = {0, 0, 0, 0, 0, 0, 0, 0};
    return device_exclusive_scan<ChunkCnt, CombineCnt>(cnts, cprefix, nc, zero, CombineCnt(), (ChunkCnt *)d_scratch,
                                                       (ChunkCnt *)d_total, stream);
}

int launch_linecode_write(const EventRec *d_ev, const uint32_t *d_M, uint32_t cap_ev, const LineTables &lt, const uint16_t *d_start,
                          const void *d_cnt_prefix, SymbolRec *d_sym, uint32_t cap_sym, uint8_t *d_bits0, uint32_t cap_b0,
                          uint8_t *d_bits1, uint32_t cap_b1, void *d_frames, void *d_findex, uint32_t cap_em, int64_t a,
                          const void *d_bits_in, void *d_bits_out, uint32_t *d_n_empty, uint32_t *d_n_frames, const uint32_t *d_pending_in,
                          const DecCarry *d_carry_in, DecCarry *d_carry_out, uint32_t *d_pending_out, cudaStream_t stream) {
    const uint32_t nc = std::max(1u, linecode_chunks(cap_ev));
    LineOut out;
    out.sym = d_sym; out.bits0 = d_bits0; out.bits1 = d_bits1; out.fr = (FrameRec *)d_frames; out.fx = (unsigned long long *)d_findex;
    out.cap_sym = cap_sym; out.cap_b0 = cap_b0; out.cap_b1 = cap_b1; out.cap_em = cap_em;
    out.pending_in = d_pending_in;
    out.a = a;
    out.bits_in = (const unsigned long long *)d_bits_in;
    out.bits_out = (unsigned long long *)d_bits_out;
    out.n_empty = d_n_empty;
    out.n_frames = d_n_frames;
    const EvCount evc{d_M, cap_ev};
    (lt.batch_tab ? chunk_write_kernel<true> : chunk_write_kernel<false>)<<<(nc + 127) / 128, 128, 0, stream>>>(d_ev, evc, lt, d_start, (const ChunkCnt *)d_cnt_prefix, out,
                                                             d_carry_in, d_carry_out, d_pending_out);
    NFC_CUDA_CHECK(cudaGetLastError());
    return 0;
}

}  // namespace nfc
