// stream.cu -- host driver of one sample stream and the extern "C" boundary (include/usrp_nfc_b200.h).
//
// A push is cut into slabs; a slab into time segments (one CTA each, slicer.cu).  Segment 0 starts
// from the stream's true state, the others start cold `halo` samples early and are verified at the
// seam against their predecessor's final state, then redone from the true state if they differ.
// The ordered transitions of the slab go through runs.cu (events) and linecode.cu (symbols, frames);
// only records leave the device.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <thread>
#include <deque>
#include <vector>

#include "../../include/usrp_nfc_b200.h"
#include "common.cuh"
#include "tables.h"

namespace nfc {

// ---- launchers implemented in the kernel files
int launch_slicer(const SegWork *d_works, int n_works, const SlicerParams *d_params, int L, cudaStream_t);
bool slicer_streaming_ok(int L, int kind);
int launch_slicer_streaming(const SegWork *d_works, int n_works, const SlicerParams *d_params, int L, int kind, cudaStream_t);
int launch_extract_count(const uint32_t *d_bm, int64_t bm_pos0, int64_t a, int64_t b, const RunCarry *d_rc_in, int carry_from_bm,
                         uint32_t *d_block_counts, uint32_t *d_block_offsets, uint32_t *d_scan_scratch, uint32_t *d_total,
                         cudaStream_t stream);
int launch_extract_write(const uint32_t *d_bm, int64_t bm_pos0, int64_t a, int64_t b, const RunCarry *d_rc_in, int carry_from_bm,
                         const uint32_t *d_block_offsets, TransRec *d_out, uint32_t out_cap, cudaStream_t stream);
size_t extract_blocks(int64_t bm_pos0, int64_t a, int64_t b);
int launch_slicer_serial(const SegWork *d_works, int n_works, const SlicerParams *d_params, float *d_ring_scratch,
                         size_t ring_stride, cudaStream_t);
int launch_seam_compare(const SlicerHdr *const *d_truth, const SlicerHdr *const *d_assumed, const int *d_param_idx,
                        const SlicerParams *d_params, int *d_mismatch, int n, cudaStream_t);
int launch_gather_transitions(const SegWork *d_works, const uint32_t *d_counts, uint32_t *d_offsets, int n_segs,
                              TransRec *d_dense, cudaStream_t);
int launch_gather_pieces(const TransRec *const *d_src, const uint32_t *d_n, const uint32_t *d_off, int n_pieces,
                         TransRec *d_dense, cudaStream_t);
int launch_run_count(const TransRec *d_tr, const uint32_t *d_R, uint32_t cap_R, int64_t w0, int64_t w1, const RunCarry *d_rc_in,
                     int mx, int keep_dropped, uint32_t *d_counts, uint32_t *d_offsets, uint32_t *d_scratch, uint32_t *d_total,
                     uint32_t *d_flags, cudaStream_t stream);
int launch_run_write(const TransRec *d_tr, const uint32_t *d_R, uint32_t cap_R, int64_t w0, int64_t w1, const RunCarry *d_rc_in,
                     int mx, int keep_dropped, const uint32_t *d_offsets, EventRec *d_events, uint32_t cap, const uint32_t *d_M,
                     RunCarry *d_carry_out, uint32_t *d_flags, cudaStream_t stream);
uint32_t linecode_chunks(uint32_t n_ev);
size_t linecode_map_bytes();
size_t linecode_cnt_bytes();
size_t linecode_emission_bytes();
size_t linecode_scratch_bytes(uint32_t n_chunks);
int launch_linecode_start(const EventRec *d_ev, const uint32_t *d_M, uint32_t cap_ev, const LineTables &lt, const DecCarry *d_carry_in,
                          uint16_t *d_summary, uint16_t *d_start, uint32_t *d_flags, cudaStream_t stream);
int launch_linecode_start_scan(const EventRec *d_ev, const uint32_t *d_M, uint32_t cap_ev, const LineTables &lt,
                               const DecCarry *d_carry_in, void *d_maps, void *d_prefix, void *d_scratch, uint16_t *d_start,
                               cudaStream_t stream);
int launch_linecode_count(const EventRec *d_ev, const uint32_t *d_M, uint32_t cap_ev, const LineTables &lt, const uint16_t *d_start,
                          void *d_cnts, void *d_cnt_prefix, void *d_scratch, void *d_total, cudaStream_t stream);
int launch_linecode_write(const EventRec *d_ev, const uint32_t *d_M, uint32_t cap_ev, const LineTables &lt, const uint16_t *d_start,
                          const void *d_cnt_prefix, SymbolRec *d_sym, uint32_t cap_sym, uint8_t *d_bits0, uint32_t cap_b0,
                          uint8_t *d_bits1, uint32_t cap_b1, void *d_frames, void *d_findex, uint32_t cap_em, int64_t a,
                          const void *d_bits_in, void *d_bits_out, uint32_t *d_n_empty, uint32_t *d_n_frames, const uint32_t *d_pending_in,
                          const DecCarry *d_carry_in, DecCarry *d_carry_out, uint32_t *d_pending_out, cudaStream_t stream);
int slicer_tile(int L, int kind);
int slicer_resident_ctas(int L, int kind);
int slicer_tile_stats(unsigned long long *out4, bool reset);
int launch_batch_warm(const SegWork *d_works, int n_works, int L, const SlicerParams *d_params, cudaStream_t stream);
int launch_bitmap_fill(uint32_t *d_bm, size_t n_chunks, cudaStream_t stream);
int synth_render(void *dev_out, int64_t n, int64_t first_index, const int8_t *codes, const int64_t *lens, int64_t n_runs,
                 float carrier, float pause, float tag_high, float noise, float fade, double fade_period, uint64_t seed,
                 int as_envelope, cudaStream_t);

// ---- error reporting
static thread_local char g_err[512] = "";
void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        NFC_CUDA_CHECK(cudaMalloc(&p, want));
        cap = want;
        return 0;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T *as() const { return reinterpret_cast<T *>(p); }
};

static size_t item_bytes(int kind) {
    switch (kind) {
        case IN_IQ_F32: return 8;
        case IN_PCM_S16: return 2;
        case IN_SC16: return 4;  // I, Q: two int16
        default: return 4;
    }
}

static int ceil_log2(int v) {
    int l = 0;
    while ((1LL << l) < v) l++;
    return l;
}

static int classify_ratio_host(double ratio, double lo, double hi) {  // transition_sink.py:67-71
    if (lo > ratio) return -1;
    if (ratio > hi) return 1;
    return 0;
}

// The frame records of a stream in page-locked memory: the device writes them final (linecode.cu: WriteSink::emission), a
// slab's records are copied straight behind those of the slabs before.
struct FrameArena {
    nfc_frame *p = nullptr;
    size_t n = 0, cap = 0;
    size_t size() const { return n; }
    bool empty() const { return n == 0; }
    nfc_frame *data() { return p; }
    const nfc_frame &operator[](size_t i) const { return p[i]; }
    void clear() { n = 0; }
    int reserve(size_t need) {  // may move the arena: no copy into it in flight, nobody reading
        if (need <= cap) return 0;
        const size_t ncap = std::max(need + need / 2 + 4096, cap * 2);
        nfc_frame *q = nullptr;
        if (cudaMallocHost((void **)&q, ncap * sizeof(nfc_frame)) != cudaSuccess) return -1;
        if (n) memcpy(q, p, n * sizeof(nfc_frame));
        if (p) cudaFreeHost(p);
        p = q;
        cap = ncap;
        return 0;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        n = cap = 0;
    }
};
static_assert(sizeof(nfc_frame) == sizeof(FrameRec), "the device writes nfc_frame records");

// All frame bits of one type in the order they were appended (cpp.append_bit), in page-locked memory: a slab's bits are
// copied from the device straight to their final place behind the bits of the slabs before, frames refer to them by offset.
// [0, closed): bits of the frames handed out so far (up to the last frame closing); [closed, len): bits of a frame still open.
struct BitArena {
    uint8_t *p = nullptr;
    size_t cap = 0, len = 0, closed = 0;
    // May move the arena: the caller guarantees that no copy into it is in flight and that nobody reads it.
    int reserve(size_t need) {
        if (need <= cap) return 0;
        const size_t ncap = std::max(need + need / 2 + 65536, cap * 2);
        uint8_t *q = nullptr;
        if (cudaMallocHost((void **)&q, ncap) != cudaSuccess) return -1;
        if (len) memcpy(q, p, len);
        if (p) cudaFreeHost(p);
        p = q;
        cap = ncap;
        return 0;
    }
    void consume() {  // the frames were handed out: the open bits move to the front
        const size_t open = len - closed;
        if (open && closed) memmove(p, p + closed, open);
        len = open;
        closed = 0;
    }
    void clear() { len = closed = 0; }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = len = closed = 0;
    }
};

struct Stream {
    nfc_params prm;
    SlicerParams sp;
    HostTables ht;
    LineTables lt;
    double factor;
    cudaStream_t cs = nullptr;
    cudaStream_t cs2 = nullptr;  // device -> host copies of a slab's records, beside the next slab's slicer
    cudaStream_t cs3 = nullptr;  // host -> device copies of the next slab's samples, beside this slab's kernels
    cudaEvent_t ev_h[2] = {nullptr, nullptr};
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;  // around a launch of the streaming slicer kernel
    DevBuf staging2[2];
    // A slab's post-slicer chain (extraction -> runs -> line code) is queued on `cs` without waiting for any count: the
    // kernels read counts and carries from the slab's context block in device memory (ring of NCTX blocks, PostCtx) and from
    // the block of the slab before; buffers are sized from the slabs before.  The host looks at a slab's context (copied to
    // pinned memory behind its chain) one slab later -- the next chain is already queued by then -- and only then puts the
    // records on their way to the host.  A slab whose buffers turn out too small is done again with exact sizes.
    static const int NCTX = 4;
    cudaEvent_t ev_a[NCTX] = {}, ev_b[NCTX] = {}, ev_c[NCTX] = {};  // timing: slab begins, transitions ready, chain done
    // The three stages of a chain run on three streams: extraction on `cs` (behind the slicer), runs on csR, line code on csL;
    // stage X of slab k waits for the stage before it (event) and, being queued behind it, for stage X of slab k-1 -- so the
    // extraction of slab k+1 runs beside the runs of slab k and the line code of slab k-1.
    cudaStream_t csR = nullptr, csL = nullptr;
    cudaEvent_t evE[NCTX] = {}, evR[NCTX] = {}, evL[NCTX] = {};
    long long chain_first_seq = 0;   // slabs from this one on were queued since the streams were last idle (their events are valid)
    long long last_final_seq = -1;
    cudaEvent_t ev_ctx[NCTX] = {};   // the slab's context block has arrived in ctx_h
    cudaEvent_t ev_out[2] = {};      // the records of the slab that used output set i are on the host
    bool ev_out_set[2] = {false, false};
    DevBuf ctx_d;
    char *ctx_h = nullptr;           // pinned, NCTX blocks
    long long slab_seq = 0;
    struct Rates {                   // records per sample seen so far (maxima, slowly decaying): sizes the next slab's buffers
        bool have = false;
        double R = 0, M = 0, sym = 0, b0 = 0, b1 = 0, em = 0;
    } rates;

    // stream state
    int64_t pos = 0;
    bool stable = false;
    bool serial_mode = false;
    std::vector<float> warm;
    DevBuf state;   // current true state block (hdr + ring)
    RunCarry run_carry{0, 0, 0, 0};
    DecCarry dec_carry{0, 0, {0, 0}};
    uint32_t pending[2] = {0, 0};

    // tuning
    int64_t seg_len = 0, halo = 0, slab_len = 0;
    int force_serial = 0;

    // device scratch
    DevBuf params_d, tab_d, staging, works_d, states_d, trans_seg, seg_counts, seg_status,
        seam_ptrs, mismatch_d, run_counts, run_offsets, scan_scr, maps_d, prefix_d, cnts_d, cprefix_d,
        line_scr, serial_ring, start_d, ckpt_d, redo_states, redo_trans,
        redo_counts, pieces_d, bitmap_d, ex_counts, ex_offsets, ex_scr, summ_d;
    // outputs of a slab's chain, two sets: the records of slab k travel to the host while the chain of slab k+1 writes the other
    DevBuf events_d[2], sym_d[2], bits0_d[2], bits1_d[2], em_d[2], fx_d[2];  // em_d: frame records (FrameRec), fx_d: their packed index
    DevBuf trans_dense[2];  // transitions of slab k in [k & 1]: the extraction of slab k+1 runs beside the runs of slab k
    std::vector<DevBuf> kept_bufs;  // redo buffers whose contents are still referenced by transition pieces
    // results come back into one of three pinned buffers.  The carries of a slab (256 bytes) are copied first and are all
    // the next slab waits for; the records behind them are awaited by a worker thread, which turns them into the output
    // vectors while the device works on the following slabs (the threads form a chain: each joins its predecessor first).
    static const int NPIN = 3;
    void *pinned[NPIN] = {nullptr, nullptr, nullptr};
    size_t pinned_cap[NPIN] = {0, 0, 0};
    long long slabs_enqueued = 0;               // slabs whose records were put on their way
    std::atomic<long long> slabs_marshalled{0};  // slabs whose records are in the output vectors
    std::thread marshal_thr;
    // wait mode (nfc_stream_set_wait_mode): host threads sleep in the driver instead of spinning while they wait for this
    // stream -- for many streams driven by many host threads (batches of captures), where spinning threads outnumber the cores
    bool blocking_wait = false;
    cudaEvent_t ev_blk = nullptr;
    cudaError_t sync_cs() {
        if (!blocking_wait) return cudaStreamSynchronize(cs);
        const cudaError_t e = cudaEventRecord(ev_blk, cs);
        return e != cudaSuccess ? e : cudaEventSynchronize(ev_blk);
    }
    int set_wait_mode(bool blocking);
    std::atomic<int> marshal_err{0};
    // a slab whose chain is queued and whose context the host has not looked at yet
    struct SlabJob {
        long long seq = 0;
        int64_t a = 0, b = 0;
        uint32_t cap_R = 0, cap_M = 0, cap_sym = 0, cap_b0 = 0, cap_b1 = 0, cap_em = 0;
        bool exact = false;      // sizes were read while queuing: cannot overflow
        bool events_only = false;  // events from the caller (push_events): says nothing about records per sample
        bool from_bitmap = false;
        bool want_ev = false, want_sym = false, want_fr = false, have_line = false;
        double t0 = 0, t1 = 0, t2 = 0;
    };
    std::deque<SlabJob> jobs;
    cudaEvent_t ev_d[NPIN] = {nullptr, nullptr, nullptr};  // all records of the slab that used pinned[i] have arrived
    int post_chain(int64_t a, int64_t b, bool from_bitmap, uint32_t R_host, bool force_exact, double t0, double t1,
                   const EventRec *host_events = nullptr, uint32_t n_host_events = 0);
    int64_t push_events(const nfc_event *ev, int64_t n);
    int finalize_front();
    int finalize_all() {
        while (!jobs.empty())
            if (finalize_front()) return -1;
        return 0;
    }
    int marshal(const SlabJob &j, int pi, char *hp, size_t off_ev, size_t off_sym, uint32_t M, uint32_t nsym);

    // results
    std::vector<nfc_event> out_events;
    std::vector<nfc_symbol> out_symbols;
    FrameArena out_frames;               // bit_off is relative to fb[type].p
    cudaEvent_t ev_last_records = nullptr;  // the copy of the last finalized slab's records (a slab no worker thread waits for)
    bool have_last_records = false;
    int settle_frames();
    // packed frame offsets (pos << 24 | nbits << 8 | type) of out_frames in page-locked memory (nfc_stream_view_frame_index)
    uint64_t *findex = nullptr;
    size_t findex_n = 0, findex_cap = 0;
    bool findex_bad = false;
    bool findex_ext = false;  // the caller's memory (nfc_stream_set_frame_index_buffer): never reallocated
    bool findex_ext_locked = false;  // ... page-locked by this library for the time it is in use (cudaHostRegister), so that the copies into it stay asynchronous
    void findex_drop() {
        if (findex && findex_ext && findex_ext_locked) cudaHostUnregister(findex);
        if (findex && !findex_ext) cudaFreeHost(findex);
        findex = nullptr;
        findex_ext = findex_ext_locked = false;
        findex_cap = findex_n = 0;
    }
    int findex_reserve(size_t n) {  // worker thread or settled stream only
        if (n <= findex_cap) return 0;
        if (findex_ext) return -1;
        const size_t cap = std::max(n, findex_cap * 2 + 4096);
        uint64_t *p = nullptr;
        if (cudaMallocHost((void **)&p, cap * sizeof(uint64_t)) != cudaSuccess) return -1;
        if (findex_n) memcpy(p, findex, findex_n * sizeof(uint64_t));
        if (findex) cudaFreeHost(findex);
        findex = p;
        findex_cap = cap;
        return 0;
    }
    BitArena fb[2];                      // frame bits per type, frames back to back
    int resident_ctas = 0;
    size_t ev_head = 0, sym_head = 0, fr_head = 0;

    nfc_stats stats;

    int tile() const { return slicer_tile(sp.L, sp.input_kind); }
    // windows of 256 to 52000 samples take the streaming kernel (multiples of 4 from 1024 on) or the first-generation kernel;
    // the others take the sequential kernel: shorter ones than a tile, and longer ones, whose ring does not fit a CTA's shared
    // memory beside the kernels' own scratch
    bool parallel_ok() const { return sp.L >= 256 && sp.L <= 52000 && !force_serial && !serial_mode; }

    int init(const nfc_params *p);
    void destroy();
    int ensure_pinned(int idx, size_t bytes);
    int join_marshal();
    int finish_pending() { return finalize_all(); }
    int settle() { return finalize_all() || join_marshal() || settle_frames() ? -1 : 0; }
    int64_t push(const void *items, int64_t n, int mem, int *called_back);
    int64_t push_batch(const void *items, int mem, int64_t n_cap, int64_t cap_len, int64_t stride_items, const double *lo_vals,
                       const double *hi_vals, int64_t *pitch_out);
    int64_t push_batch_ragged(const void *const *items, int mem, int64_t n_cap, const int64_t *lengths, const double *lo_vals,
                              const double *hi_vals, int64_t *starts_out);
    // the segment ranges [start + L, start + length) of the batch the class bitmap was last filled for: positions no segment
    // of that batch wrote hold val == 0.  A batch whose segments are the same ranges, or a prefix of them, finds the rest of
    // its positions at val == 0 too; any other layout, and a single stream's slicer, write elsewhere (empty: fill again).
    std::vector<int64_t> batch_fill;
    DevBuf batch_states, batch_stage, batch_tab;
    std::vector<int64_t> batch_starts;  // host copy of the capture table's starts (a slab's first capture: post_chain)
    int finish_warmup();
    int process_slab(const void *d_in, int64_t in_pos0, int64_t in_begin, int64_t in_end, int64_t a, int64_t b, int64_t slicer_end);
    // the streaming kernel writes the class bitmap; the first-generation kernel (windows below 1024 samples or not a
    // multiple of 4) and the sequential kernel write transition lists
    enum class Slicer { streaming, first_gen, sequential };
    int run_slicer(Slicer kind, const void *d_in, int64_t in_pos0, int64_t in_begin, int64_t in_end, int64_t a, int64_t b,
                   uint32_t *R_out, bool *fell_back);
    int launch_streaming(const SegWork *d_works, int n_works);
    void add_kernel_time();
    int compare_states(const std::vector<const SlicerHdr *> &truth, const std::vector<const SlicerHdr *> &assumed, int n,
                       std::vector<int> &mism);
    // the class bitmap holds stream positions [bm_lo, bm_hi) (chunk 0 at bm_origin): the streaming slicer may run ahead of the
    // slab that is being turned into events
    int64_t bm_lo = 0, bm_hi = 0, bm_origin = 0;
    // slabs per launch of the streaming slicer on device-resident input (NFC_SUPER_SLAB, 1..8): segments twice as long halve
    // the share of the speculative starts; the slabs after the first take their transitions from the bitmap (extract_only)
    int64_t super_slab = 5;
    bool super_balance = true;  // NFC_SUPER_BALANCE=0: every launch but the last takes super_slab slabs
    bool streaming_ok() const { return parallel_ok() && slicer_streaming_ok(sp.L, sp.input_kind); }
};

int Stream::ensure_pinned(int idx, size_t bytes) {
    if (bytes <= pinned_cap[idx]) return 0;
    if (pinned[idx]) cudaFreeHost(pinned[idx]);
    pinned[idx] = nullptr;
    pinned_cap[idx] = 0;
    NFC_CUDA_CHECK(cudaMallocHost(&pinned[idx], bytes + bytes / 4 + 4096));
    pinned_cap[idx] = bytes + bytes / 4 + 4096;
    return 0;
}

// waits for the records of the previous slab to be in the output vectors
int Stream::join_marshal() {
    if (marshal_thr.joinable()) marshal_thr.join();
    if (const int err = marshal_err.exchange(0)) {
        set_error(err == 3 ? "more frames than the caller's frame index buffer holds (nfc_stream_set_frame_index_buffer)"
                           : (err == 2 ? "copying a slab's records to the host failed" : "internal: frame longer than the retained bits"));
        return -1;
    }
    return 0;
}

int Stream::init(const nfc_params *p) {
    prm = *p;
    memset(&stats, 0, sizeof(stats));
    if (!(p->samp_rate > 0) || p->av_window < 1 || p->max_len < 1 || p->max_len > 65535) {
        set_error("bad parameters: samp_rate=%g av_window=%d max_len=%d", p->samp_rate, p->av_window, p->max_len);
        return -1;
    }
    if (p->av_window >= (1 << 28)) {
        set_error("av_window too large");
        return -1;
    }
    NFC_CUDA_CHECK(cudaSetDevice(p->device));
    NFC_CUDA_CHECK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
    NFC_CUDA_CHECK(cudaStreamCreateWithFlags(&cs2, cudaStreamNonBlocking));
    NFC_CUDA_CHECK(cudaStreamCreateWithFlags(&cs3, cudaStreamNonBlocking));
    NFC_CUDA_CHECK(cudaStreamCreateWithFlags(&csR, cudaStreamNonBlocking));
    NFC_CUDA_CHECK(cudaStreamCreateWithFlags(&csL, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) NFC_CUDA_CHECK(cudaEventCreateWithFlags(&ev_h[i], cudaEventDisableTiming));
    NFC_CUDA_CHECK(cudaEventCreate(&ev_k0));
    NFC_CUDA_CHECK(cudaEventCreate(&ev_k1));
    for (int i = 0; i < NCTX; i++) {
        NFC_CUDA_CHECK(cudaEventCreate(&ev_a[i]));
        NFC_CUDA_CHECK(cudaEventCreate(&ev_b[i]));
        NFC_CUDA_CHECK(cudaEventCreate(&ev_c[i]));
        NFC_CUDA_CHECK(cudaEventCreateWithFlags(&ev_ctx[i], cudaEventDisableTiming));
        NFC_CUDA_CHECK(cudaEventCreateWithFlags(&evE[i], cudaEventDisableTiming));
        NFC_CUDA_CHECK(cudaEventCreateWithFlags(&evR[i], cudaEventDisableTiming));
        NFC_CUDA_CHECK(cudaEventCreateWithFlags(&evL[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < 2; i++) NFC_CUDA_CHECK(cudaEventCreateWithFlags(&ev_out[i], cudaEventDisableTiming));
    // the worker thread that turns a slab's records into the output vectors is off the critical path: it sleeps while it waits
    // (spinning waiters of eight ranks crowd the host's cores)
    for (int i = 0; i < NPIN; i++) NFC_CUDA_CHECK(cudaEventCreateWithFlags(&ev_d[i], cudaEventDisableTiming | cudaEventBlockingSync));
    NFC_CUDA_CHECK(cudaMallocHost((void **)&ctx_h, (size_t)NCTX * 256));
    if (ctx_d.ensure((size_t)NCTX * 256)) return -1;
    NFC_CUDA_CHECK(cudaMemset(ctx_d.p, 0, (size_t)NCTX * 256));
    factor = 1e6 / p->samp_rate;  // transition_sink.py:21
    sp.lo = p->lo_val;
    sp.hi = p->hi_val;
    sp.L = p->av_window;
    sp.Ld = (double)p->av_window;
    sp.mx = p->max_len;
    sp.loL = sp.lo / sp.Ld;
    sp.hiL = sp.hi / sp.Ld;
    sp.cls_ss0_x0 = classify_ratio_host(1.0, sp.lo, sp.hi);            // transition_sink.py:60-61
    sp.cls_ss0_xn = classify_ratio_host(sp.hi + 0.1, sp.lo, sp.hi);    // transition_sink.py:62-63
    sp.span_limit = std::max(0, 28 - ceil_log2(sp.L) - 1);
    sp.input_kind = p->input_kind;
    sp.pcm_scale = p->pcm_scale > 0 ? p->pcm_scale : 32767.0f;
    if (params_d.ensure(sizeof(SlicerParams))) return -1;
    NFC_CUDA_CHECK(cudaMemcpy(params_d.p, &sp, sizeof(sp), cudaMemcpyHostToDevice));

    if (!build_tables(sp.mx, factor, ht)) {
        set_error("line-code tables need more than %d duration classes", MAX_DCLASS);
        return -1;
    }
    const size_t dcm = ht.dclass_miller.size(), dcg = ht.dclass_manch.size();
    const size_t tm = ht.miller.size() * sizeof(TabEntry), tg = ht.manch.size() * sizeof(TabEntry);
    auto up = [](size_t v) { return (v + 255) / 256 * 256; };
    const size_t o1 = up(dcm), o2 = o1 + up(dcg), o3 = o2 + up(tm), o4 = o3 + up(tg), o5 = o4 + up(ht.reset_miller.size());
    if (tab_d.ensure(o5 + up(ht.reset_manch.size()))) return -1;
    char *base = tab_d.as<char>();
    NFC_CUDA_CHECK(cudaMemcpy(base, ht.dclass_miller.data(), dcm, cudaMemcpyHostToDevice));
    NFC_CUDA_CHECK(cudaMemcpy(base + o1, ht.dclass_manch.data(), dcg, cudaMemcpyHostToDevice));
    NFC_CUDA_CHECK(cudaMemcpy(base + o2, ht.miller.data(), tm, cudaMemcpyHostToDevice));
    NFC_CUDA_CHECK(cudaMemcpy(base + o3, ht.manch.data(), tg, cudaMemcpyHostToDevice));
    NFC_CUDA_CHECK(cudaMemcpy(base + o4, ht.reset_miller.data(), ht.reset_miller.size(), cudaMemcpyHostToDevice));
    NFC_CUDA_CHECK(cudaMemcpy(base + o5, ht.reset_manch.data(), ht.reset_manch.size(), cudaMemcpyHostToDevice));
    lt.dclass_miller = (const uint8_t *)base;
    lt.dclass_manch = (const uint8_t *)(base + o1);
    lt.miller = (const TabEntry *)(base + o2);
    lt.manch = (const TabEntry *)(base + o3);
    lt.reset_miller = (const uint8_t *)(base + o4);
    lt.reset_manch = (const uint8_t *)(base + o5);
    lt.n_dclass_miller = ht.n_dclass_miller;
    lt.n_dclass_manch = ht.n_dclass_manch;
    lt.decode_reader = p->decode_reader;
    lt.decode_tag = p->decode_tag;
    lt.batch_tab = nullptr;
    lt.batch_base = 0;
    lt.batch_n = lt.batch_c0 = lt.batch_skip = 0;

    warm.reserve((size_t)sp.L);
    if (state.ensure(state_block_bytes(sp.L))) return -1;
    resident_ctas = parallel_ok() ? slicer_resident_ctas(sp.L, sp.input_kind) : 1;
    if (const char *e = getenv("NFC_SUPER_SLAB")) super_slab = std::max(1, std::min(8, atoi(e)));
    if (const char *e = getenv("NFC_SUPER_BALANCE")) super_balance = atoi(e) != 0;
    return 0;
}

void Stream::destroy() {
    DevBuf *all[] = {&batch_states, &batch_stage, &batch_tab, &params_d, &tab_d, &staging, &works_d, &states_d, &trans_seg, &trans_dense[0], &trans_dense[1], &seg_counts,
                     &seg_status, &seam_ptrs, &mismatch_d, &run_counts, &run_offsets, &scan_scr, &maps_d,
                     &prefix_d, &cnts_d, &cprefix_d, &line_scr, &ctx_d, &events_d[0], &events_d[1], &sym_d[0], &sym_d[1], &bits0_d[0],
                     &bits0_d[1], &bits1_d[0], &bits1_d[1], &em_d[0], &em_d[1], &fx_d[0], &fx_d[1],
                     &serial_ring, &start_d, &ckpt_d, &redo_states, &redo_trans, &redo_counts, &pieces_d, &state, &bitmap_d,
                     &ex_counts, &ex_offsets, &ex_scr, &summ_d};
    finalize_all();
    if (marshal_thr.joinable()) marshal_thr.join();
    if (cs) cudaStreamSynchronize(cs);
    if (csR) cudaStreamSynchronize(csR);
    if (csL) cudaStreamSynchronize(csL);
    if (cs2) cudaStreamSynchronize(cs2);
    for (DevBuf *b : all) b->release();
    if (ctx_h) cudaFreeHost(ctx_h);
    ctx_h = nullptr;
    fb[0].release();
    fb[1].release();
    out_frames.release();
    findex_drop();
    for (int i = 0; i < NPIN; i++)
        if (pinned[i]) cudaFreeHost(pinned[i]);
    for (int i = 0; i < NCTX; i++) {
        if (ev_a[i]) cudaEventDestroy(ev_a[i]);
        if (ev_b[i]) cudaEventDestroy(ev_b[i]);
        if (ev_c[i]) cudaEventDestroy(ev_c[i]);
        if (ev_ctx[i]) cudaEventDestroy(ev_ctx[i]);
        if (evE[i]) cudaEventDestroy(evE[i]);
        if (evR[i]) cudaEventDestroy(evR[i]);
        if (evL[i]) cudaEventDestroy(evL[i]);
    }
    for (int i = 0; i < 2; i++)
        if (ev_out[i]) cudaEventDestroy(ev_out[i]);
    if (csR) cudaStreamDestroy(csR);
    if (csL) cudaStreamDestroy(csL);
    if (cs2) cudaStreamDestroy(cs2);
    if (cs3) cudaStreamDestroy(cs3);
    if (ev_k0) cudaEventDestroy(ev_k0);
    if (ev_k1) cudaEventDestroy(ev_k1);
    for (int i = 0; i < 2; i++) {
        if (ev_h[i]) cudaEventDestroy(ev_h[i]);
        staging2[i].release();
    }
    for (int i = 0; i < NPIN; i++)
        if (ev_d[i]) cudaEventDestroy(ev_d[i]);
    if (ev_blk) cudaEventDestroy(ev_blk);
    if (cs) cudaStreamDestroy(cs);
}

// host-side envelope of the few warm-up samples (same float operations as the device path)
static float host_env(const void *items, int64_t i, int kind, float pcm_scale) {
    switch (kind) {
        case IN_ENVELOPE_F32: return ((const float *)items)[i];
        case IN_REAL_F32: {
            volatile float s = ((const float *)items)[i];
            volatile float r = s * s;
            return r;
        }
        case IN_IQ_F32: {
            volatile float re = ((const float *)items)[2 * i], im = ((const float *)items)[2 * i + 1];
            volatile float a = re * re, b = im * im;
            volatile float r = a + b;
            return r;
        }
        case IN_SC16: {
            const int16_t *iq = (const int16_t *)items + 2 * i;
            volatile float re = (float)iq[0] / pcm_scale, im = (float)iq[1] / pcm_scale;
            volatile float a = re * re, b = im * im;
            volatile float r = a + b;
            return r;
        }
        default: {
            volatile float s = (float)((const int16_t *)items)[i] / pcm_scale;
            volatile float r = s * s;
            return r;
        }
    }
}

int Stream::set_wait_mode(bool blocking) {
    if (settle()) return -1;
    NFC_CUDA_CHECK(cudaSetDevice(prm.device));
    const unsigned flags = cudaEventDisableTiming | (blocking ? cudaEventBlockingSync : 0);
    for (int i = 0; i < NCTX; i++) {
        if (ev_ctx[i]) cudaEventDestroy(ev_ctx[i]);
        ev_ctx[i] = nullptr;
        NFC_CUDA_CHECK(cudaEventCreateWithFlags(&ev_ctx[i], flags));
    }
    if (blocking && !ev_blk) NFC_CUDA_CHECK(cudaEventCreateWithFlags(&ev_blk, cudaEventDisableTiming | cudaEventBlockingSync));
    blocking_wait = blocking;
    return 0;
}

int Stream::finish_warmup() {
    // transition_sink.py:121-124: _sum = sum(ar) (left to right, double), _dur = length % max
    double s = 0;
    for (int i = 0; i < sp.L; i++) s += (double)warm[(size_t)i];
    std::vector<char> blk(state_block_bytes(sp.L), 0);
    SlicerHdr *h = reinterpret_cast<SlicerHdr *>(blk.data());
    h->ss = s;
    h->pos = sp.L;
    h->lastL = NO_POS;
    h->lrun_start = NO_POS;
    h->last_val = 0;
    memcpy(state_ring(h), warm.data(), (size_t)sp.L * 4);
    NFC_CUDA_CHECK(cudaMemcpyAsync(state.p, blk.data(), blk.size(), cudaMemcpyHostToDevice, cs));
    NFC_CUDA_CHECK(sync_cs());  // blk is a local buffer
    run_carry.st = 0;
    run_carry.last_bit = 0;
    run_carry.dur = sp.L % sp.mx;
    stable = true;
    return 0;
}

int64_t Stream::push(const void *items, int64_t n, int mem, int *called_back) {
    if (called_back) *called_back = 0;
    batch_fill.clear();  // the slicer writes the class bitmap at this stream's positions
    if (n < 0) {
        set_error("negative item count");
        return -1;
    }
    NFC_CUDA_CHECK(cudaSetDevice(prm.device));
    const size_t ib = item_bytes(sp.input_kind);
    if (!stable) {  // transition_sink.py:109-125
        const int64_t need = sp.L - (int64_t)warm.size();
        const int64_t can = std::min(n, need);
        if (can > 0) {
            std::vector<char> tmp;
            const void *src = items;
            if (mem == NFC_MEM_DEVICE) {
                tmp.resize((size_t)can * ib);
                // on the stream's own CUDA stream: a copy on the default stream would queue behind other streams' work
                NFC_CUDA_CHECK(cudaMemcpyAsync(tmp.data(), items, (size_t)can * ib, cudaMemcpyDeviceToHost, cs));
                NFC_CUDA_CHECK(sync_cs());
                src = tmp.data();
            }
            for (int64_t i = 0; i < can; i++) warm.push_back(host_env(src, i, sp.input_kind, sp.pcm_scale));
        }
        pos += can;
        if (can == need && finish_warmup()) return -1;
        return can;
    }
    if (called_back) *called_back = 1;
    int64_t done = 0;
    // transition records hold positions relative to the slab in 30 bits
    const int64_t slab = slab_len > 0 ? std::min<int64_t>(slab_len, (int64_t)1 << 30) : (int64_t)1 << 28;
    // Host input goes through two staging buffers: the copy of slab k+1 (stream cs3) runs beside the kernels of slab k.
    const bool host_in = mem == NFC_MEM_HOST;
    auto stage_host = [&](int64_t off, int64_t m, int64_t a, int buf) -> int {
        const size_t padb = (size_t)(a - (a - (a & 3))) * ib;
        if (staging2[buf].ensure(padb + (size_t)m * ib + 64)) return -1;
        NFC_CUDA_CHECK(cudaMemcpyAsync(staging2[buf].as<char>() + padb, (const char *)items + (size_t)off * ib, (size_t)m * ib,
                                       cudaMemcpyHostToDevice, cs3));
        NFC_CUDA_CHECK(cudaEventRecord(ev_h[buf], cs3));
        stats.h2d_bytes += (int64_t)((size_t)m * ib);
        return 0;
    };
    int hbuf = 0;
    if (host_in && n > 0) {
        // the buffers may still be read by kernels of an earlier push: those are complete once the stream is idle
        NFC_CUDA_CHECK(sync_cs());
        if (stage_host(0, std::min(slab, n), pos, hbuf)) return -1;
    }
    while (done < n) {
        const int64_t m = std::min(slab, n - done);
        const int64_t a = pos, b = pos + m;
        const int64_t in_pos0 = a - (a & 3);
        const void *d_in = nullptr;
        int64_t in_begin = in_pos0;
        int64_t slicer_end = b;
        const char *src = (const char *)items + (size_t)done * ib;
        const size_t padb = (size_t)(a - in_pos0) * ib;
        if (host_in) {
            const int64_t m_next = std::min(slab, n - (done + m));
            // the other buffer was read by the slicer of the slab before this one, which has completed
            if (m_next > 0 && stage_host(done + m, m_next, b, hbuf ^ 1)) return -1;
            NFC_CUDA_CHECK(cudaStreamWaitEvent(cs, ev_h[hbuf], 0));
            d_in = staging2[hbuf].p;
            hbuf ^= 1;
        } else if ((((uintptr_t)src - padb) & 15) == 0) {
            d_in = src - padb;  // usable in place: item with stream index in_pos0 would sit 16-byte aligned
            in_begin = a;       // ... but nothing before the caller's pointer is read
            // device-resident input: the streaming slicer may run over several slabs at once (only positions relative to a
            // slab are limited to 30 bits, and the slicer writes none)
            // ... over equally many slabs per launch (ten slabs at four per launch go 4 + 3 + 3, not 4 + 4 + 2: the
            // segments of a short last launch would be short too)
            int64_t take = super_slab;
            if (super_balance) {
                const int64_t left = (n - done + slab - 1) / slab, launches = (left + super_slab - 1) / super_slab;
                take = (left + launches - 1) / launches;
            }
            slicer_end = std::min(pos + (n - done), a + take * slab);
        } else {
            if (staging.ensure(padb + (size_t)m * ib + 64)) return -1;
            NFC_CUDA_CHECK(cudaMemcpyAsync(staging.as<char>() + padb, src, (size_t)m * ib, cudaMemcpyDeviceToDevice, cs));
            d_in = staging.p;
        }
        if (process_slab(d_in, in_pos0, in_begin, std::max(b, slicer_end), a, b, slicer_end)) return -1;
        pos = b;
        done += m;
        stats.samples += m;
    }
    return n;
}

// A batch of independent captures in one pass (BASELINE.json configs[3]).  The reference gives every capture its own
// transition_sink (own warm-up, own lo_val / hi_val: transition_sink.py:12-34,109-125), background thread, decoders and
// PacketProcessors (decoder.py:29-33).  Here capture c owns the positions [starts[c], starts[c + 1]) of one position space
// (its length rounded up to tiles; nothing for a capture of at most av_window items, which the warm-up consumes whole); one
// launch of the streaming slicer runs one segment per capture from the capture's own warm-up state (computed on the
// device), and extraction / runs / line code walk the batch as one stream in which a capture's first event finds decoders
// and PacketProcessors as new (linecode.cu, through a device table of the captures' starts and lengths).  Frames come out
// with positions of that space: the capture is the last c with starts[c] <= pos, the index in it pos - starts[c].
// Returns n_cap, -1 on error, -3 when a capture leaves the exactly-summable regime (the caller decodes captures one by
// one then: nfc_stream_push takes the sequential path for such input).
int64_t Stream::push_batch_ragged(const void *const *items, int mem, int64_t n_cap, const int64_t *lengths, const double *lo_vals,
                                  const double *hi_vals, int64_t *starts_out) {
    NFC_CUDA_CHECK(cudaSetDevice(prm.device));
    const int L = sp.L;
    const int T = tile();
    const size_t ib = item_bytes(sp.input_kind);
    if (pos != 0 || stable || !warm.empty()) {
        set_error("push_batch: the stream has consumed samples; reset it first");
        return -1;
    }
    if (!streaming_ok()) {
        set_error("push_batch: needs the streaming slicer (av_window in [1024, 52000], a multiple of 4)");
        return -1;
    }
    // Any capture longer than L items is decoded on the device, however short its own range [L, length) is; there is no
    // bound of L + 2 max_len.  Its segment starts from the exact state of its warm-up (batch_warm_kernel), not from a
    // speculative start, so no seam, checkpoint or halo needs a minimum length.  Behind it lie val == 0 positions (padding,
    // then the next capture's warm-up of L > max_len + 1 samples), so every run open at its end times out and resets
    // cur_state (transition_sink.py:95-99) before the next capture's first own sample; the events at or past its length
    // are not the capture's and the line code ignores them.  L > max_len + 1 is what that needs.
    if (n_cap <= 0 || n_cap >= ((int64_t)1 << 31) || L <= sp.mx + 1) {
        set_error("push_batch: bad shape (captures %lld, av_window %d, max_len %d)", (long long)n_cap, L, sp.mx);
        return -1;
    }
    if (prm.outputs & NFC_OUT_DROPPED_EVENTS) {
        set_error("push_batch: type -1 events are not reproduced across capture boundaries (NFC_OUT_DROPPED_EVENTS)");
        return -1;
    }
    // ---- layout: starts[c + 1] = starts[c] + the capture's length rounded up to tiles (0 for at most L items)
    std::vector<int64_t> starts((size_t)n_cap + 1, 0);
    for (int64_t c = 0; c < n_cap; c++) {
        const int64_t len = lengths[c];
        if (len < 0 || (len > 0 && !items[c])) {
            set_error("push_batch: capture %lld: bad length %lld or null items", (long long)c, (long long)len);
            return -1;
        }
        const int64_t width = len > L ? (len + T - 1) / T * T : 0;
        if (width >= ((int64_t)1 << 30)) {
            set_error("push_batch: capture %lld too long for one slab (%lld items): decode it with nfc_stream_push", (long long)c,
                      (long long)len);
            return -1;
        }
        if (width && mem == NFC_MEM_DEVICE && ((uintptr_t)items[c] % 16) != 0) {
            set_error("push_batch: capture %lld: device items must start 16-byte aligned", (long long)c);
            return -1;
        }
        starts[(size_t)c + 1] = starts[(size_t)c] + width;
    }
    if (starts_out) memcpy(starts_out, starts.data(), sizeof(int64_t) * ((size_t)n_cap + 1));
    // ---- the captures' items on the device; host captures are staged into 16-byte aligned slots, one copy per run of
    // captures that lie exactly one behind the other in host memory (a contiguous 2-D batch is one copy).  Nothing between
    // two captures is read: that memory is not the caller's to give, and may not even be mapped.
    std::vector<const void *> d_in((size_t)n_cap, nullptr);
    if (mem == NFC_MEM_HOST) {
        struct Run { const char *h; size_t bytes, slot; };
        std::vector<Run> runs;
        std::vector<std::pair<size_t, size_t>> where((size_t)n_cap);  // (run, byte offset in it)
        size_t total_bytes = 0;
        const char *prev = nullptr;
        size_t prev_bytes = 0;
        for (int64_t c = 0; c < n_cap; c++) {
            if (starts[(size_t)c + 1] == starts[(size_t)c]) continue;  // no segment: its items are not read
            const char *h = (const char *)items[c];
            const size_t bytes = (size_t)lengths[c] * ib;
            const bool joins = prev && h == prev + prev_bytes && (size_t)(h - runs.back().h) % 16 == 0;
            if (!joins) {
                total_bytes = (total_bytes + 255) / 256 * 256;
                runs.push_back(Run{h, 0, total_bytes});
            }
            Run &r = runs.back();
            where[(size_t)c] = {runs.size() - 1, (size_t)(h - r.h)};
            const size_t end = (size_t)(h - r.h) + bytes;
            total_bytes += end - r.bytes;
            r.bytes = end;
            prev = h;
            prev_bytes = bytes;
        }
        if (batch_stage.ensure(total_bytes + 64)) return -1;
        for (const Run &r : runs) {
            NFC_CUDA_CHECK(cudaMemcpyAsync(batch_stage.as<char>() + r.slot, r.h, r.bytes, cudaMemcpyHostToDevice, cs));
            stats.h2d_bytes += (int64_t)r.bytes;
        }
        for (int64_t c = 0; c < n_cap; c++)
            if (starts[(size_t)c + 1] != starts[(size_t)c]) d_in[(size_t)c] = batch_stage.as<char>() + runs[where[(size_t)c].first].slot + where[(size_t)c].second;
    } else {
        for (int64_t c = 0; c < n_cap; c++) d_in[(size_t)c] = items[c];
    }
    // ---- per-capture parameters (transition_sink's lo_val / hi_val constructor arguments)
    std::vector<SlicerParams> ps((size_t)n_cap, sp);
    for (int64_t c = 0; c < n_cap; c++) {
        SlicerParams &q = ps[(size_t)c];
        if (lo_vals) q.lo = lo_vals[c];
        if (hi_vals) q.hi = hi_vals[c];
        q.loL = q.lo / q.Ld;
        q.hiL = q.hi / q.Ld;
        q.cls_ss0_x0 = classify_ratio_host(1.0, q.lo, q.hi);
        q.cls_ss0_xn = classify_ratio_host(q.hi + 0.1, q.lo, q.hi);
        if (!(q.lo > 0.0) || !(q.hi > q.lo)) {
            set_error("push_batch: capture %lld: thresholds must satisfy 0 < lo_val < hi_val", (long long)c);
            return -1;
        }
    }
    if (params_d.ensure(sizeof(SlicerParams) * (size_t)n_cap)) return -1;
    NFC_CUDA_CHECK(cudaMemcpyAsync(params_d.p, ps.data(), sizeof(SlicerParams) * (size_t)n_cap, cudaMemcpyHostToDevice, cs));
    // ---- the capture table of the line code: starts, then lengths (read by chains until the last slab is finalized)
    std::vector<int64_t> tab(starts);
    tab.insert(tab.end(), lengths, lengths + n_cap);
    if (batch_tab.ensure(sizeof(int64_t) * tab.size())) return -1;
    NFC_CUDA_CHECK(cudaMemcpyAsync(batch_tab.p, tab.data(), sizeof(int64_t) * tab.size(), cudaMemcpyHostToDevice, cs));
    // ---- bitmap, one segment per capture, warm-up states
    const size_t sblk = state_block_bytes(L);
    if (batch_states.ensure(sblk * (size_t)n_cap) || seg_status.ensure(sizeof(int32_t) * (size_t)n_cap) ||
        works_d.ensure(sizeof(SegWork) * (size_t)n_cap))
        return -1;
    const int64_t total = starts[(size_t)n_cap];
    const size_t n_chunks = (size_t)(total / 128);
    std::vector<int64_t> fill;  // the segment ranges, in capture order
    for (int64_t c = 0; c < n_cap; c++)
        if (starts[(size_t)c + 1] != starts[(size_t)c]) {
            fill.push_back(starts[(size_t)c] + L);
            fill.push_back(starts[(size_t)c] + lengths[c]);
        }
    const size_t bm_cap_before = bitmap_d.cap;
    if (bitmap_d.ensure((n_chunks + 64) * 32)) return -1;
    if (bitmap_d.cap != bm_cap_before || batch_fill.size() < fill.size() || batch_fill.empty() ||
        !std::equal(fill.begin(), fill.end(), batch_fill.begin())) {
        if (launch_bitmap_fill(bitmap_d.as<uint32_t>(), n_chunks, cs)) return -1;
        batch_fill = fill;
        stats.launches++;
    }
    // Captures take different times: the longer a capture, and the closer hi_val lies to the tag's HIGH level (the more of
    // its tiles need the precise passes), the longer its segment runs.  There are more segments than CTAs fit on the device
    // at once: the ones expected to take longest go first, so that the last wave is made of short ones.
    std::vector<int64_t> order;
    for (int64_t c = 0; c < n_cap; c++)
        if (starts[(size_t)c + 1] != starts[(size_t)c]) order.push_back(c);
    std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) {
        if (lengths[a] != lengths[b]) return lengths[a] > lengths[b];
        return hi_vals && hi_vals[a] > hi_vals[b];
    });
    const int n_works = (int)order.size();
    std::vector<SegWork> works((size_t)n_works);
    for (int k = 0; k < n_works; k++) {
        const int64_t c = order[(size_t)k];
        SegWork &w = works[(size_t)k];
        memset(&w, 0, sizeof(w));
        const int64_t B = starts[(size_t)c];
        w.in = d_in[(size_t)c];
        w.in_pos0 = B;
        w.in_begin = B;
        w.in_end = B + lengths[c];
        w.warm_begin = B + L;
        w.begin = B + L;
        w.end = B + lengths[c];
        w.slab_pos0 = 0;
        w.state_in = reinterpret_cast<const SlicerHdr *>(batch_states.as<char>() + sblk * (size_t)c);
        for (int j = 0; j < 3; j++) w.ckpt_pos[j] = INT64_MAX;
        w.status = seg_status.as<int32_t>() + c;
        w.param_idx = (int32_t)c;
        w.bitmap = bitmap_d.as<uint32_t>();
        w.bm_pos0 = 0;
    }
    std::vector<int32_t> status((size_t)n_cap, 0);
    if (n_works) {
        NFC_CUDA_CHECK(cudaMemcpyAsync(works_d.p, works.data(), sizeof(SegWork) * (size_t)n_works, cudaMemcpyHostToDevice, cs));
        if (launch_batch_warm(works_d.as<SegWork>(), n_works, L, params_d.as<SlicerParams>(), cs)) return -1;
        stats.launches++;
        if (launch_streaming(works_d.as<SegWork>(), n_works)) return -1;
        stats.launches++;
        stats.slicer_launches++;
        stats.segments += n_works;
        NFC_CUDA_CHECK(cudaMemcpyAsync(status.data(), seg_status.p, sizeof(int32_t) * (size_t)n_cap, cudaMemcpyDeviceToHost, cs));
    }
    NFC_CUDA_CHECK(sync_cs());
    if (n_works) add_kernel_time();
    for (int64_t c : order)
        if (status[(size_t)c] & (SEG_INEXACT | SEG_NOT_SANE)) {
            set_error("push_batch: capture %lld is outside the exactly-summable regime: decode the captures one by one", (long long)c);
            return -3;
        }
    // ---- extraction, runs, line code: slabs of whole captures
    stable = true;
    bm_lo = 0;
    bm_hi = total;
    bm_origin = 0;
    batch_starts = starts;
    lt.batch_tab = batch_tab.as<int64_t>();
    lt.batch_n = (uint32_t)n_cap;
    lt.batch_skip = (uint32_t)L;
    // slabs of whole captures, packed greedily up to slab_max positions; a wider capture is a slab of its own
    // (nfc_stream_set_tuning's slab_len shortens them: tests; more, shorter slabs were slower: 10.5 against 9.6 ms)
    const int64_t slab_max = slab_len > 0 ? std::min<int64_t>(slab_len, (int64_t)1 << 30) : (int64_t)1 << 30;
    int rc = 0;
    if (finish_pending()) rc = -1;
    // What a slab's chain inherits from the slab before (run carry, decoder state, the val before its first sample) does
    // not matter: a capture's warm-up flushes it, and its first event finds decoders and PacketProcessors as new.  So the
    // chains of the batch's slabs are queued back to back like those of one stream.
    run_carry = RunCarry{0, 0, L % sp.mx, 0};
    for (int64_t c0 = 0; c0 < n_cap && !rc;) {
        int64_t c1 = c0 + 1;
        while (c1 < n_cap && starts[(size_t)c1 + 1] - starts[(size_t)c0] <= slab_max) c1++;
        const int64_t a = starts[(size_t)c0], b = starts[(size_t)c1];
        if (b > a && process_slab(nullptr, a, a, b, a, b, b)) rc = -1;
        pos = b;
        for (int64_t c = c0; c < c1; c++) stats.samples += lengths[c];
        c0 = c1;
    }
    if (!rc && finish_pending()) rc = -1;
    lt.batch_tab = nullptr;
    lt.batch_n = 0;
    bm_lo = bm_hi = 0;
    // the parameter block of a single stream again
    cudaMemcpyAsync(params_d.p, &sp, sizeof(sp), cudaMemcpyHostToDevice, cs);
    if (sync_cs() != cudaSuccess && !rc) rc = -1;
    return rc ? rc : n_cap;
}

// Equally long captures at items + c * stride_items: the ragged batch with starts[c] = c * pitch.
int64_t Stream::push_batch(const void *items, int mem, int64_t n_cap, int64_t cap_len, int64_t stride_items, const double *lo_vals,
                           const double *hi_vals, int64_t *pitch_out) {
    const size_t ib = item_bytes(sp.input_kind);
    if (n_cap <= 0 || cap_len <= (int64_t)sp.L || stride_items < cap_len) {
        set_error("push_batch: bad shape (captures %lld, items %lld, stride %lld, av_window %d)", (long long)n_cap, (long long)cap_len,
                  (long long)stride_items, sp.L);
        return -1;
    }
    if (((size_t)stride_items * ib) % 16 != 0 || ((uintptr_t)items % 16) != 0) {
        set_error("push_batch: captures must start 16-byte aligned");
        return -1;
    }
    std::vector<const void *> ptrs((size_t)n_cap);
    for (int64_t c = 0; c < n_cap; c++) ptrs[(size_t)c] = (const char *)items + (size_t)c * (size_t)stride_items * ib;
    std::vector<int64_t> lengths((size_t)n_cap, cap_len), starts((size_t)n_cap + 1);
    const int64_t rc = push_batch_ragged(ptrs.data(), mem, n_cap, lengths.data(), lo_vals, hi_vals, starts.data());
    if (rc >= 0 && pitch_out) *pitch_out = starts[1];
    return rc;
}

// Launches the streaming slicer kernel between ev_k0 and ev_k1; add_kernel_time() counts its time once the stream has been
// synchronised.
int Stream::launch_streaming(const SegWork *d_works, int n_works) {
    NFC_CUDA_CHECK(cudaEventRecord(ev_k0, cs));
    if (launch_slicer_streaming(d_works, n_works, params_d.as<SlicerParams>(), sp.L, sp.input_kind, cs)) return -1;
    NFC_CUDA_CHECK(cudaEventRecord(ev_k1, cs));
    return 0;
}

void Stream::add_kernel_time() {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ev_k0, ev_k1) == cudaSuccess) {
        stats.slicer_kernel_ms += ms;
        stats.slicer_kernel_launches++;
    }
}

// Queues the bit-for-bit comparison of the states truth[q] and assumed[q], q < n (a pair with a nullptr is skipped);
// mism[q] is set once the stream has been synchronised.  seam_ptrs has room for truth.size() entries of each kind.
int Stream::compare_states(const std::vector<const SlicerHdr *> &truth, const std::vector<const SlicerHdr *> &assumed, int n,
                           std::vector<int> &mism) {
    const size_t room = truth.size();
    char *base = seam_ptrs.as<char>();
    NFC_CUDA_CHECK(cudaMemcpyAsync(base, truth.data(), sizeof(void *) * (size_t)n, cudaMemcpyHostToDevice, cs));
    NFC_CUDA_CHECK(cudaMemcpyAsync(base + sizeof(void *) * room, assumed.data(), sizeof(void *) * (size_t)n, cudaMemcpyHostToDevice, cs));
    NFC_CUDA_CHECK(cudaMemsetAsync(base + 2 * sizeof(void *) * room, 0, sizeof(int) * (size_t)n, cs));  // parameter set 0
    NFC_CUDA_CHECK(cudaMemsetAsync(mismatch_d.p, 0, sizeof(int) * (size_t)n, cs));
    if (launch_seam_compare((const SlicerHdr *const *)base, (const SlicerHdr *const *)(base + sizeof(void *) * room),
                            (const int *)(base + 2 * sizeof(void *) * room), params_d.as<SlicerParams>(), mismatch_d.as<int>(), n, cs))
        return -1;
    stats.launches++;
    NFC_CUDA_CHECK(cudaMemcpyAsync(mism.data(), mismatch_d.p, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, cs));
    return 0;
}

// NFC_SEGDEBUG: the cycles the streaming kernel spent on each segment (its final state's count, in thousands) and the
// tiles it redid or took slowly (pad), on stderr.
static int print_segment_cycles(const std::vector<SegWork> &works) {
    const int nseg = (int)works.size();
    double sum = 0;
    uint32_t mn = ~0u, mx = 0;
    std::vector<uint32_t> kc((size_t)nseg), rs((size_t)nseg);
    for (int k = 0; k < nseg; k++) {
        SlicerHdr h;
        NFC_CUDA_CHECK(cudaMemcpy(&h, works[(size_t)k].state_out, sizeof(SlicerHdr), cudaMemcpyDeviceToHost));
        kc[(size_t)k] = h.count; rs[(size_t)k] = h.pad;
        sum += h.count; mn = std::min(mn, h.count); mx = std::max(mx, h.count);
    }
    fprintf(stderr, "segments %d kcycles min %u avg %.0f max %u\n", nseg, mn, sum / nseg, mx);
    for (int k = 0; k < nseg; k += std::max(1, nseg / 24))
        fprintf(stderr, "  seg %d: %u kcyc, redo %u slow %u\n", k, kc[(size_t)k], rs[(size_t)k] >> 16, rs[(size_t)k] & 0xffff);
    // the slowest
    for (int q = 0; q < 6; q++) {
        int best = 0;
        for (int k = 1; k < nseg; k++) if (kc[(size_t)k] > kc[(size_t)best]) best = k;
        fprintf(stderr, "  slowest seg %d: %u kcyc, redo %u slow %u\n", best, kc[(size_t)best], rs[(size_t)best] >> 16, rs[(size_t)best] & 0xffff);
        kc[(size_t)best] = 0;
    }
    return 0;
}

// Runs one slicer kernel over [a, b) of a slab and leaves the slab's true final state in `state`.  The streaming kernel
// writes the class bitmap in place ([bm_lo, bm_hi) afterwards); the first-generation and the sequential kernel write
// transition lists per segment, gathered into trans_dense[slab_seq & 1] (*R_out transitions).  *fell_back: a parallel
// kernel left the exactly-summable regime, the caller redoes the slab with the sequential kernel.
int Stream::run_slicer(Slicer kind, const void *d_in, int64_t in_pos0, int64_t in_begin, int64_t in_end, int64_t a, int64_t b,
                       uint32_t *R_out, bool *fell_back) {
    // the slabs whose chains are still queued read the bitmap and trans_dense this slicer is about to overwrite; should one
    // of them have to be done again, its input must still be there: look at them first (their chains end within a fraction
    // of a millisecond)
    if (finalize_all()) return -1;
    bm_hi = bm_lo = 0;
    const bool bitmap = kind == Slicer::streaming;
    const int L = sp.L;
    const int T = tile();
    *fell_back = false;
    // ---- plan segments
    std::vector<int64_t> begins;  // first emitted sample of each segment
    begins.push_back(a);
    int64_t H = 0;
    if (kind != Slicer::sequential) {
        const int64_t Hs = halo > 0 ? halo : (int64_t)16 * L;
        H = (Hs + T - 1) / T * T;
        int64_t S = seg_len;
        if (S <= 0) {
            const int64_t n = b - a, res = std::max(1, resident_ctas);
            const int64_t s_min = 6 * H;
            int64_t s_max, k = 1;
            if (bitmap) {
                // one segment per resident CTA if that keeps them below s_max, else the fewest waves that do: the longer
                // the segments, the smaller the share of the speculative starts
                s_max = std::max<int64_t>((int64_t)4096 * L, s_min);
                k = std::max<int64_t>(1, (n + res * s_max - 1) / (res * s_max));
            } else {
                // as many segments as CTAs fit on the device at once (times k), each at least 6 halos long so that the
                // speculative halo costs little, at most 256 windows so that a redo stays cheap
                s_max = std::max<int64_t>((int64_t)256 * L, s_min);
                while (n / (res * (k + 1)) >= s_min) k++;
            }
            S = std::clamp(n / (res * k), s_min, s_max);
        }
        S = (S + T - 1) / T * T;
        int64_t b1 = a + std::max<int64_t>(S, (int64_t)L + H);
        b1 = (b1 + T - 1) / T * T;
        while (b1 + S / 2 <= b && b1 < b) {
            begins.push_back(b1);
            b1 += S;
        }
    }
    const int nseg = (int)begins.size();
    const size_t sblk = state_block_bytes(L);
    const int NCK = 3;
    // checkpoints of every speculative segment, at 1, 3 and 7 halos after its first emitted sample
    const int64_t ck_off[NCK] = {H, 3 * H, 7 * H};
    // state blocks: [seam_in k][state_out k] per segment; work items: the segments, behind them the redos of a repair round
    if (states_d.ensure(sblk * 2 * (size_t)nseg) || (nseg > 1 && ckpt_d.ensure(sblk * NCK * (size_t)nseg))) return -1;
    if (seg_status.ensure(sizeof(int32_t) * (size_t)nseg) || works_d.ensure(sizeof(SegWork) * (size_t)nseg * 2) ||
        mismatch_d.ensure(sizeof(int) * (size_t)nseg) || seam_ptrs.ensure((sizeof(void *) * 2 + sizeof(int)) * (size_t)nseg))
        return -1;
    if (!bitmap && seg_counts.ensure(sizeof(uint32_t) * (size_t)nseg)) return -1;
    if (kind == Slicer::sequential && serial_ring.ensure((size_t)L * 4 + 64)) return -1;
    // bitmap of the slab, chunk 0 at the tile boundary at or before a
    const int64_t bm_pos0 = a / T * T;
    if (bitmap && bitmap_d.ensure(((size_t)((b - bm_pos0 + 127) / 128) + 64) * 32)) return -1;
    auto seam_in = [&](int k) { return reinterpret_cast<SlicerHdr *>(states_d.as<char>() + sblk * (2 * (size_t)k)); };
    auto st_out = [&](int k) { return reinterpret_cast<SlicerHdr *>(states_d.as<char>() + sblk * (2 * (size_t)k + 1)); };
    auto ckpt = [&](int k, int j) { return reinterpret_cast<SlicerHdr *>(ckpt_d.as<char>() + sblk * ((size_t)k * NCK + (size_t)j)); };
    auto tmp_state = [&](int i) { return reinterpret_cast<SlicerHdr *>(redo_states.as<char>() + sblk * (size_t)i); };
    auto launch = [&](const SegWork *d_works, int n_works) -> int {
        if (kind == Slicer::streaming) {
            if (launch_streaming(d_works, n_works)) return -1;
        } else if (kind == Slicer::first_gen) {
            if (launch_slicer(d_works, n_works, params_d.as<SlicerParams>(), L, cs)) return -1;
        } else {
            if (launch_slicer_serial(d_works, n_works, params_d.as<SlicerParams>(), serial_ring.as<float>(), (size_t)L + 16, cs))
                return -1;
            stats.serial_segments += n_works;
        }
        stats.launches++;
        stats.slicer_launches++;
        return 0;
    };

    // transition lists: capacities per segment, raised when a launch overflows them
    std::vector<uint32_t> caps((size_t)nseg);
    for (int k = 0; k < nseg; k++) {
        const int64_t e = k + 1 < nseg ? begins[(size_t)k + 1] : b;
        caps[(size_t)k] = (uint32_t)std::min<int64_t>((e - begins[(size_t)k]) / 8 + 1024, (e - begins[(size_t)k]) + 16);
    }
    std::vector<SegWork> works((size_t)nseg);
    std::vector<uint32_t> counts((size_t)nseg);
    std::vector<int32_t> status((size_t)nseg);
    struct Piece {
        const TransRec *src;
        uint32_t n;
    };

    for (int attempt = 0; attempt < 4; attempt++) {
        std::vector<size_t> toff((size_t)nseg);
        if (!bitmap) {
            size_t total_cap = 0;
            for (int k = 0; k < nseg; k++) {
                toff[(size_t)k] = total_cap;
                total_cap += caps[(size_t)k];
            }
            if (trans_seg.ensure(total_cap * sizeof(TransRec) + 16)) return -1;
        }
        for (int k = 0; k < nseg; k++) {
            SegWork &w = works[(size_t)k];
            memset(&w, 0, sizeof(w));
            w.in = d_in;
            w.in_pos0 = in_pos0;
            w.in_begin = in_begin;
            w.in_end = in_end;
            w.begin = begins[(size_t)k];
            w.end = k + 1 < nseg ? begins[(size_t)k + 1] : b;
            w.warm_begin = k == 0 ? a : w.begin - H;
            w.slab_pos0 = a;
            w.state_in = k == 0 ? state.as<SlicerHdr>() : nullptr;
            w.seam_in = k == 0 ? nullptr : seam_in(k);
            for (int j = 0; j < NCK; j++) {
                const bool use = k > 0 && w.begin + ck_off[j] < w.end;
                w.ckpt_pos[j] = use ? w.begin + ck_off[j] : INT64_MAX;
                w.ckpt_state[j] = use ? ckpt(k, j) : nullptr;
            }
            w.state_out = st_out(k);
            w.status = seg_status.as<int32_t>() + k;
            if (bitmap) {
                w.bitmap = bitmap_d.as<uint32_t>();
                w.bm_pos0 = bm_pos0;
            } else {
                w.trans = trans_seg.as<TransRec>() + toff[(size_t)k];
                w.trans_cap = caps[(size_t)k];
                w.trans_count = seg_counts.as<uint32_t>() + k;
            }
        }
        NFC_CUDA_CHECK(cudaMemcpyAsync(works_d.p, works.data(), sizeof(SegWork) * (size_t)nseg, cudaMemcpyHostToDevice, cs));
        if (launch(works_d.as<SegWork>(), nseg)) return -1;
        stats.segments += nseg;

        // ---- seams: compare what each speculative segment assumed with what its predecessor reached
        std::vector<int> mism((size_t)nseg, 0);
        std::vector<const SlicerHdr *> truth((size_t)nseg, nullptr), assumed((size_t)nseg, nullptr);
        if (nseg > 1) {
            for (int k = 1; k < nseg; k++) {
                truth[(size_t)k] = st_out(k - 1);
                assumed[(size_t)k] = seam_in(k);
            }
            if (compare_states(truth, assumed, nseg, mism)) return -1;
        }
        if (!bitmap)
            NFC_CUDA_CHECK(cudaMemcpyAsync(counts.data(), seg_counts.p, sizeof(uint32_t) * (size_t)nseg, cudaMemcpyDeviceToHost, cs));
        NFC_CUDA_CHECK(cudaMemcpyAsync(status.data(), seg_status.p, sizeof(int32_t) * (size_t)nseg, cudaMemcpyDeviceToHost, cs));
        NFC_CUDA_CHECK(sync_cs());
        if (bitmap) add_kernel_time();
        int st_all = 0;
        bool over = false;
        for (int k = 0; k < nseg; k++) {
            st_all |= status[(size_t)k];
            if (counts[(size_t)k] > caps[(size_t)k]) {
                over = true;
                caps[(size_t)k] = counts[(size_t)k] + 16;
            }
        }
        if (kind != Slicer::sequential && (st_all & (SEG_INEXACT | SEG_NOT_SANE))) {
            *fell_back = true;
            return 0;
        }
        if (over) {
            stats.overflow_retries++;
            continue;
        }

        // ---- repair: a segment whose assumption was wrong is redone from its predecessor's true final state,
        // checkpoint by checkpoint, and stops as soon as it reproduces a checkpoint of the speculative run: from
        // there on the speculative output is the true output.  Only a redo that reaches the segment end changes the
        // segment's final state, and then the next seam is checked again.  A redo of the streaming kernel overwrites the
        // bitmap in place; the other kernels' redos write to redo_trans, and `pieces` says which stretches of which lists
        // make up each segment's transitions.
        std::vector<std::vector<Piece>> pieces((size_t)nseg);
        for (int k = 0; k < nseg && !bitmap; k++) pieces[(size_t)k].push_back(Piece{works[(size_t)k].trans, counts[(size_t)k]});
        std::vector<char> bad((size_t)nseg, 0);
        int nbad = 0;
        for (int k = 1; k < nseg; k++) {
            bad[(size_t)k] = mism[(size_t)k] ? 1 : 0;
            nbad += bad[(size_t)k];
        }
        for (int guard = 0; nbad > 0 && guard < nseg + 2; guard++) {
            // this round: the flagged segments whose predecessor is settled
            std::vector<int> ks;
            for (int k = 1; k < nseg; k++)
                if (bad[(size_t)k] && !bad[(size_t)k - 1]) ks.push_back(k);
            const int nr = (int)ks.size();
            stats.seam_mismatches += nr;
            size_t rcap_total = 0;
            std::vector<size_t> roff((size_t)nr);
            for (int i = 0; i < nr; i++) {
                roff[(size_t)i] = rcap_total;
                rcap_total += caps[(size_t)ks[(size_t)i]];
            }
            // redo_counts: the redos' transition counts, then their status
            if (redo_states.ensure(sblk * (size_t)nr) || redo_counts.ensure(sizeof(uint32_t) * 2 * (size_t)nr) ||
                (!bitmap && redo_trans.ensure(rcap_total * sizeof(TransRec) + 16)))
                return -1;
            std::vector<uint32_t> used((size_t)nr, 0);
            std::vector<int64_t> at((size_t)nr);
            std::vector<char> active((size_t)nr, 1);
            for (int i = 0; i < nr; i++) at[(size_t)i] = works[(size_t)ks[(size_t)i]].begin;
            for (int stage = 0; stage <= NCK; stage++) {
                std::vector<SegWork> redo;
                std::vector<int> who;
                for (int i = 0; i < nr; i++) {
                    if (!active[(size_t)i]) continue;
                    const int k = ks[(size_t)i];
                    const SegWork &ws = works[(size_t)k];
                    if (stage < NCK && !ws.ckpt_state[stage]) continue;  // no such checkpoint: a later stage runs on
                    SegWork w = ws;
                    w.warm_begin = w.begin = at[(size_t)i];
                    w.end = stage < NCK ? ws.ckpt_pos[stage] : ws.end;
                    w.state_in = at[(size_t)i] == ws.begin ? st_out(k - 1) : tmp_state(i);
                    w.seam_in = nullptr;
                    for (int j = 0; j < NCK; j++) { w.ckpt_pos[j] = INT64_MAX; w.ckpt_state[j] = nullptr; }
                    w.state_out = tmp_state(i);
                    w.status = reinterpret_cast<int32_t *>(redo_counts.as<uint32_t>() + nr + i);
                    if (!bitmap) {
                        w.trans = redo_trans.as<TransRec>() + roff[(size_t)i] + used[(size_t)i];
                        w.trans_cap = caps[(size_t)k] - std::min(caps[(size_t)k], used[(size_t)i]);
                        w.trans_count = redo_counts.as<uint32_t>() + i;
                    }
                    redo.push_back(w);
                    who.push_back(i);
                }
                if (redo.empty()) continue;
                SegWork *d_redo = works_d.as<SegWork>() + nseg;
                NFC_CUDA_CHECK(cudaMemcpyAsync(d_redo, redo.data(), sizeof(SegWork) * redo.size(), cudaMemcpyHostToDevice, cs));
                if (launch(d_redo, (int)redo.size())) return -1;
                // did each redo reproduce the checkpoint it stopped at?
                const int nw = (int)who.size();
                std::vector<SlicerHdr> ck_hdr((size_t)nw);
                for (int q = 0; q < nw; q++) {
                    const int i = who[(size_t)q], k = ks[(size_t)i];
                    truth[(size_t)q] = tmp_state(i);
                    assumed[(size_t)q] = stage < NCK ? works[(size_t)k].ckpt_state[stage] : tmp_state(i);
                    if (!bitmap && stage < NCK)
                        NFC_CUDA_CHECK(cudaMemcpyAsync(&ck_hdr[(size_t)q], works[(size_t)k].ckpt_state[stage], sizeof(SlicerHdr),
                                                       cudaMemcpyDeviceToHost, cs));
                }
                if (compare_states(truth, assumed, nw, mism)) return -1;
                std::vector<uint32_t> rc((size_t)nr * 2);
                NFC_CUDA_CHECK(cudaMemcpyAsync(rc.data(), redo_counts.p, sizeof(uint32_t) * 2 * (size_t)nr, cudaMemcpyDeviceToHost, cs));
                NFC_CUDA_CHECK(sync_cs());
                if (bitmap) add_kernel_time();
                for (int q = 0; q < nw; q++) {
                    const int i = who[(size_t)q], k = ks[(size_t)i];
                    if ((int32_t)rc[(size_t)nr + i] & (SEG_INEXACT | SEG_NOT_SANE)) {
                        *fell_back = true;
                        return 0;
                    }
                    if (!bitmap) {
                        const uint32_t got = rc[(size_t)i];
                        if (got > redo[(size_t)q].trans_cap) {
                            over = true;
                            caps[(size_t)k] = caps[(size_t)k] * 2 + got;
                        }
                        used[(size_t)i] += std::min(got, redo[(size_t)q].trans_cap);
                    }
                    at[(size_t)i] = redo[(size_t)q].end;
                    if (stage < NCK && !mism[(size_t)q]) {
                        // converged with the speculative run: keep its output from this checkpoint on
                        const uint32_t cc = ck_hdr[(size_t)q].count;
                        if (!bitmap)
                            pieces[(size_t)k] = {Piece{redo_trans.as<TransRec>() + roff[(size_t)i], used[(size_t)i]},
                                                 Piece{works[(size_t)k].trans + cc, counts[(size_t)k] - std::min(counts[(size_t)k], cc)}};
                        active[(size_t)i] = 0;
                        bad[(size_t)k] = 0;
                    } else if (stage == NCK || at[(size_t)i] >= works[(size_t)k].end) {
                        // redone to its end: new final state, next seam must be looked at again
                        if (!bitmap) pieces[(size_t)k] = {Piece{redo_trans.as<TransRec>() + roff[(size_t)i], used[(size_t)i]}};
                        NFC_CUDA_CHECK(cudaMemcpyAsync(st_out(k), tmp_state(i), sblk, cudaMemcpyDeviceToDevice, cs));
                        active[(size_t)i] = 0;
                        bad[(size_t)k] = 0;
                        if (k + 1 < nseg) bad[(size_t)k + 1] = 2;  // unknown: re-compare below
                    }
                }
                if (over) break;
            }
            if (over) break;
            // re-compare the seams behind segments that were redone to their end
            std::vector<int> unk;
            for (int k = 1; k < nseg; k++)
                if (bad[(size_t)k] == 2) unk.push_back(k);
            if (!unk.empty()) {
                for (size_t q = 0; q < unk.size(); q++) {
                    truth[q] = st_out(unk[q] - 1);
                    assumed[q] = seam_in(unk[q]);
                }
                if (compare_states(truth, assumed, (int)unk.size(), mism)) return -1;
                NFC_CUDA_CHECK(sync_cs());
                for (size_t q = 0; q < unk.size(); q++) bad[(size_t)unk[q]] = mism[q] ? 1 : 0;
            }
            nbad = 0;
            for (int k = 1; k < nseg; k++) nbad += bad[(size_t)k] ? 1 : 0;
            if (nbad > 0 && !bitmap) {
                // another round will overwrite redo_trans / redo_states: detach the buffers this round's pieces use
                kept_bufs.push_back(redo_trans);
                redo_trans = DevBuf();
            }
        }
        if (over) {
            stats.overflow_retries++;
            for (DevBuf &kb : kept_bufs) kb.release();
            kept_bufs.clear();
            continue;
        }
        if (nbad > 0) {
            set_error("seam repair did not settle");
            return -1;
        }
        if (bitmap && getenv("NFC_SEGDEBUG") && print_segment_cycles(works)) return -1;
        // the slab's final state becomes the stream's state
        NFC_CUDA_CHECK(cudaMemcpyAsync(state.p, st_out(nseg - 1), sblk, cudaMemcpyDeviceToDevice, cs));
        if (bitmap) {
            bm_lo = a;
            bm_hi = b;
            bm_origin = bm_pos0;
            return 0;
        }
        // ---- dense ordered transitions
        std::vector<const TransRec *> psrc;
        std::vector<uint32_t> pn, poff;
        size_t R = 0;
        for (int k = 0; k < nseg; k++)
            for (const Piece &pc : pieces[(size_t)k]) {
                psrc.push_back(pc.src);
                pn.push_back(pc.n);
                poff.push_back((uint32_t)R);
                R += pc.n;
            }
        const size_t np = psrc.size();
        DevBuf &td = trans_dense[slab_seq & 1];  // the chain of this slab (post_chain) reads the set of its sequence number
        if (td.ensure((R + 16) * sizeof(TransRec)) || pieces_d.ensure(np * (sizeof(void *) + 8) + 64)) return -1;
        char *pb = pieces_d.as<char>();
        NFC_CUDA_CHECK(cudaMemcpyAsync(pb, psrc.data(), np * sizeof(void *), cudaMemcpyHostToDevice, cs));
        NFC_CUDA_CHECK(cudaMemcpyAsync(pb + np * sizeof(void *), pn.data(), np * 4, cudaMemcpyHostToDevice, cs));
        NFC_CUDA_CHECK(cudaMemcpyAsync(pb + np * (sizeof(void *) + 4), poff.data(), np * 4, cudaMemcpyHostToDevice, cs));
        if (launch_gather_pieces((const TransRec *const *)pb, (const uint32_t *)(pb + np * sizeof(void *)),
                                 (const uint32_t *)(pb + np * (sizeof(void *) + 4)), (int)np, td.as<TransRec>(), cs))
            return -1;
        stats.launches++;
        NFC_CUDA_CHECK(sync_cs());  // pieces may live in buffers released below
        for (DevBuf &kb : kept_bufs) kb.release();
        kept_bufs.clear();
        *R_out = (uint32_t)R;
        return 0;
    }
    set_error("transition buffers kept overflowing");
    return -1;
}

static double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ---- a slab's context block in device memory (256 bytes; ring of NCTX): counts and flags of the slab's chain, and the
// carries it leaves for the next slab (the reference's cur_state / last_bit / dur, decoder and PacketProcessor state)
struct PostCtx {
    uint32_t M, R, flags, n_empty, n_frames, pad0[3];
    uint32_t tot[8];      // ChunkCnt: nsym, nbit0, nbit1, nemit, has0, tail0, has1, tail1
    RunCarry rc_out;
    DecCarry dc_out;
    uint32_t pend_out[2];
    uint32_t pad1[2];
    unsigned long long bits_out[2];  // bits of each type appended so far (offsets into the stream's bit arenas)
    uint32_t pad2[32];
};
static_assert(sizeof(PostCtx) == 256, "context blocks are 256 bytes apart");

// background.append (background.py:27-29): a list of transition_sink's events straight into the line-code stage.
int64_t Stream::push_events(const nfc_event *ev, int64_t n) {
    if (n < 0 || (n > 0 && !ev) || n >= ((int64_t)1 << 31)) {
        set_error("push_events: bad arguments");
        return -1;
    }
    NFC_CUDA_CHECK(cudaSetDevice(prm.device));
    if (finalize_all()) return -1;
    if (n == 0) return 0;
    const int64_t a = ev[0].pos;
    std::vector<EventRec> recs((size_t)n);
    int64_t prev = a;
    for (int64_t i = 0; i < n; i++) {
        const int64_t rel = ev[i].pos - a;
        if (ev[i].pos < prev || rel >= ((int64_t)1 << 32) || ev[i].d < 1 || ev[i].d > sp.mx || ev[i].v < -1 || ev[i].v > 2 ||
            ev[i].type < -1 || ev[i].type > 1) {
            set_error("push_events: event %lld out of range (positions ascend within 2^32, d in 1..max_len, v in -1..2, type in -1..1)",
                      (long long)i);
            return -1;
        }
        prev = ev[i].pos;
        EventRec r;
        r.rel_pos = (uint32_t)rel;
        r.d = (uint16_t)ev[i].d;
        r.v = ev[i].v;
        r.type = ev[i].type;
        recs[(size_t)i] = r;
    }
    const double t0 = now_ms();
    const int ci = (int)(slab_seq % NCTX);
    NFC_CUDA_CHECK(cudaEventRecord(ev_a[ci], cs));
    if (post_chain(a, a + 1, false, 0, false, t0, t0, recs.data(), (uint32_t)n)) return -1;
    if (finalize_all()) return -1;
    return n;
}

int Stream::process_slab(const void *d_in, int64_t in_pos0, int64_t in_begin, int64_t in_end, int64_t a, int64_t b,
                         int64_t slicer_end) {
    const double t0 = now_ms();
    const int ci = (int)(slab_seq % NCTX);
    NFC_CUDA_CHECK(cudaEventRecord(ev_a[ci], cs));
    uint32_t R = 0;
    bool fell_back = false, from_bitmap = false;
    if (streaming_ok() && a >= bm_lo && b <= bm_hi) {
        from_bitmap = true;  // the slicer ran over this slab together with the one before
    } else if (streaming_ok()) {
        if (run_slicer(Slicer::streaming, d_in, in_pos0, in_begin, in_end, a, std::max(b, slicer_end), &R, &fell_back)) return -1;
        from_bitmap = !fell_back;
    } else {
        const Slicer kind = parallel_ok() ? Slicer::first_gen : Slicer::sequential;
        if (run_slicer(kind, d_in, in_pos0, in_begin, in_end, a, b, &R, &fell_back)) return -1;
    }
    if (fell_back) {
        serial_mode = true;  // sums are no longer exactly representable: stay on the sequential kernel
        if (run_slicer(Slicer::sequential, d_in, in_pos0, in_begin, in_end, a, b, &R, &fell_back)) return -1;
    }
    return post_chain(a, b, from_bitmap, R, false, t0, now_ms());
}

// Queues extraction (from the bitmap; else the slicer left R_host transitions in trans_dense) -> runs -> line code of slab
// [a, b) and the copy of its context block to the host.  Sizes: from the slabs before; exact (read while queuing, with a
// synchronisation each) for the first slab of a stream and for a slab that is done again.
int Stream::post_chain(int64_t a, int64_t b, bool from_bitmap, uint32_t R_host, bool force_exact, double t0, double t1,
                       const EventRec *host_events, uint32_t n_host_events) {
    static const bool no_async = getenv("NFC_POST_SYNC") != nullptr;
    const int64_t n = b - a;
    SlabJob j;
    j.seq = slab_seq++;
    j.a = a; j.b = b;
    j.from_bitmap = from_bitmap;
    j.t0 = t0; j.t1 = t1;
    const int ci = (int)(j.seq % NCTX), pv = (int)((j.seq + NCTX - 1) % NCTX), oi = (int)(j.seq & 1);
    PostCtx *cx = ctx_d.as<PostCtx>() + ci, *cp = ctx_d.as<PostCtx>() + pv;
    if (force_exact) NFC_CUDA_CHECK(cudaEventRecord(ev_a[ci], cs));  // a slab done again: not through process_slab
    const bool fresh = jobs.empty();
    if (fresh) {
        // nothing is queued: the host's copy of the carries is the current one (reset, warm-up, set_state, the slab before)
        // and all three streams are idle
        PostCtx up;
        memset(&up, 0, sizeof(up));
        up.rc_out = run_carry;
        up.dc_out = dec_carry;
        up.pend_out[0] = pending[0];
        up.pend_out[1] = pending[1];
        up.bits_out[0] = fb[0].len;
        up.bits_out[1] = fb[1].len;
        NFC_CUDA_CHECK(cudaMemcpyAsync(cp, &up, sizeof(up), cudaMemcpyHostToDevice, cs));
        chain_first_seq = j.seq;
    }
    auto queued = [&](long long seq) { return seq >= chain_first_seq && seq >= 0; };  // its events were recorded since the streams idled
    NFC_CUDA_CHECK(cudaMemsetAsync(cx, 0, 64, cs));  // counts, flags, totals
    const bool want_line = (prm.outputs & (NFC_OUT_SYMBOLS | NFC_OUT_FRAMES)) != 0;
    const bool want_sym = (prm.outputs & NFC_OUT_SYMBOLS) != 0;
    const int keep_dropped = (prm.outputs & NFC_OUT_DROPPED_EVENTS) ? 1 : 0;
    j.exact = force_exact || no_async || !rates.have || !from_bitmap || host_events != nullptr;
    j.events_only = host_events != nullptr;
    auto cap_of = [&](double rate) -> uint32_t {
        const double c = rate * (double)n * 1.5 + 65536.0;
        return (uint32_t)std::min(c, 4.0e9);
    };
    auto sync_on = [&](cudaStream_t st) -> cudaError_t {
        if (!blocking_wait) return cudaStreamSynchronize(st);
        const cudaError_t e = cudaEventRecord(ev_blk, st);
        return e != cudaSuccess ? e : cudaEventSynchronize(ev_blk);
    };
    DevBuf &td = trans_dense[oi];

    // ---------------------------------------------------------------- extraction (cs, behind the slicer)
    if (from_bitmap) {
        // the transitions of slab k-2 (same set) have been read by its run kernels
        if (queued(j.seq - 2)) NFC_CUDA_CHECK(cudaStreamWaitEvent(cs, evR[(j.seq - 2) % NCTX], 0));
        const size_t nblk = extract_blocks(bm_origin, a, b);
        if (ex_counts.ensure((nblk + 16) * 4) || ex_offsets.ensure((nblk + 16) * 4) || ex_scr.ensure((nblk / 256 + 1024) * 4 * 4)) return -1;
        // the val before the slab's first sample: the slab before may still be in its run kernels -- its last val is in the
        // bitmap as well (the same launch of the slicer filled it); a fresh chain takes the carry just uploaded
        const int carry_from_bm = (!fresh && a > bm_lo) ? 1 : 0;
        if (!fresh && !carry_from_bm) NFC_CUDA_CHECK(cudaStreamWaitEvent(cs, evR[pv], 0));
        if (launch_extract_count(bitmap_d.as<uint32_t>(), bm_origin, a, b, &cp->rc_out, carry_from_bm, ex_counts.as<uint32_t>(),
                                 ex_offsets.as<uint32_t>(), ex_scr.as<uint32_t>(), &cx->R, cs))
            return -1;
        stats.launches += 4;
        if (j.exact) {
            uint32_t R = 0;
            NFC_CUDA_CHECK(cudaMemcpyAsync(&R, &cx->R, 4, cudaMemcpyDeviceToHost, cs));
            NFC_CUDA_CHECK(sync_on(cs));
            j.cap_R = R;
        } else {
            j.cap_R = cap_of(rates.R);
        }
        if (td.ensure(((size_t)j.cap_R + 16) * sizeof(TransRec))) return -1;
        if (launch_extract_write(bitmap_d.as<uint32_t>(), bm_origin, a, b, &cp->rc_out, carry_from_bm, ex_offsets.as<uint32_t>(),
                                 td.as<TransRec>(), j.cap_R, cs))
            return -1;
        stats.launches++;
    } else {
        j.cap_R = R_host;
        NFC_CUDA_CHECK(cudaMemcpyAsync(&cx->R, &R_host, 4, cudaMemcpyHostToDevice, cs));
    }
    NFC_CUDA_CHECK(cudaEventRecord(ev_b[ci], cs));
    NFC_CUDA_CHECK(cudaEventRecord(evE[ci], cs));

    // ---------------------------------------------------------------- runs -> events (csR)
    NFC_CUDA_CHECK(cudaStreamWaitEvent(csR, evE[ci], 0));
    if (queued(j.seq - 2)) NFC_CUDA_CHECK(cudaStreamWaitEvent(csR, evL[(j.seq - 2) % NCTX], 0));  // the events of slab k-2 have been decoded
    if (ev_out_set[oi]) NFC_CUDA_CHECK(cudaStreamWaitEvent(csR, ev_out[oi], 0));                  // ... and have left for the host
    if (host_events) {
        // the events come from the caller (nfc_stream_push_events): no runs to turn into events, the run carry passes through
        j.cap_M = n_host_events;
        if (events_d[oi].ensure(((size_t)j.cap_M + 16) * sizeof(EventRec))) return -1;
        if (n_host_events)
            NFC_CUDA_CHECK(cudaMemcpyAsync(events_d[oi].p, host_events, (size_t)n_host_events * sizeof(EventRec), cudaMemcpyHostToDevice, csR));
        NFC_CUDA_CHECK(cudaMemcpyAsync(&cx->M, &n_host_events, 4, cudaMemcpyHostToDevice, csR));
        NFC_CUDA_CHECK(cudaMemcpyAsync(&cx->rc_out, &cp->rc_out, sizeof(RunCarry), cudaMemcpyDeviceToDevice, csR));
        NFC_CUDA_CHECK(cudaStreamSynchronize(csR));  // host_events is the caller's memory
    } else {
    const size_t nrun = (size_t)j.cap_R + 1;
    if (run_counts.ensure(nrun * 4) || run_offsets.ensure(nrun * 4) || scan_scr.ensure((nrun / 256 + 1024) * 4 * 4)) return -1;
    if (launch_run_count(td.as<TransRec>(), &cx->R, j.cap_R, 0, n, &cp->rc_out, sp.mx, keep_dropped, run_counts.as<uint32_t>(),
                         run_offsets.as<uint32_t>(), scan_scr.as<uint32_t>(), &cx->M, &cx->flags, csR))
        return -1;
    stats.launches += 3;
    if (j.exact) {
        uint32_t M = 0;
        NFC_CUDA_CHECK(cudaMemcpyAsync(&M, &cx->M, 4, cudaMemcpyDeviceToHost, csR));
        NFC_CUDA_CHECK(sync_on(csR));
        j.cap_M = M;
    } else {
        j.cap_M = cap_of(rates.M);
    }
    if (events_d[oi].ensure(((size_t)j.cap_M + 16) * sizeof(EventRec))) return -1;
    if (launch_run_write(td.as<TransRec>(), &cx->R, j.cap_R, 0, n, &cp->rc_out, sp.mx, keep_dropped, run_offsets.as<uint32_t>(),
                         events_d[oi].as<EventRec>(), j.cap_M, &cx->M, &cx->rc_out, &cx->flags, csR))
        return -1;
    stats.launches++;
    }
    NFC_CUDA_CHECK(cudaEventRecord(evR[ci], csR));

    // ---------------------------------------------------------------- events -> symbols, frame bits, frame closings (csL)
    NFC_CUDA_CHECK(cudaStreamWaitEvent(csL, evR[ci], 0));
    if (ev_out_set[oi]) NFC_CUDA_CHECK(cudaStreamWaitEvent(csL, ev_out[oi], 0));  // the records of slab k-2 have left this output set
    j.have_line = want_line;
    LineTables slt = lt;  // a batch's slab: its first capture and position (also when the slab is done again later)
    if (slt.batch_tab) {
        slt.batch_base = a;
        slt.batch_c0 = (uint32_t)(std::lower_bound(batch_starts.begin(), batch_starts.end(), a) - batch_starts.begin());
    }
    if (want_line) {
        const uint32_t nc = std::max(1u, linecode_chunks(j.cap_M));
        if (start_d.ensure((size_t)nc * 2 + 64) || summ_d.ensure((size_t)nc * 2 + 64) || cnts_d.ensure((size_t)nc * linecode_cnt_bytes()) ||
            cprefix_d.ensure((size_t)nc * linecode_cnt_bytes()) || line_scr.ensure(linecode_scratch_bytes(nc) + 256))
            return -1;
        const EventRec *ev = events_d[oi].as<EventRec>();
        if (launch_linecode_start(ev, &cx->M, j.cap_M, slt, &cp->dc_out, summ_d.as<uint16_t>(), start_d.as<uint16_t>(), &cx->flags, csL)) return -1;
        if (launch_linecode_count(ev, &cx->M, j.cap_M, slt, start_d.as<uint16_t>(), cnts_d.p, cprefix_d.p, line_scr.p, cx->tot, csL)) return -1;
        stats.launches += 6;
        if (j.exact) {
            PostCtx hx;
            NFC_CUDA_CHECK(cudaMemcpyAsync(&hx, cx, 64, cudaMemcpyDeviceToHost, csL));
            NFC_CUDA_CHECK(sync_on(csL));
            if (hx.flags & POST_UNRESOLVED) {
                // some chunk saw no decoder reset within the search limit: compose chunk transfer functions instead
                stats.linecode_scan_fallbacks++;
                if (maps_d.ensure((size_t)nc * linecode_map_bytes()) || prefix_d.ensure((size_t)nc * linecode_map_bytes())) return -1;
                if (launch_linecode_start_scan(ev, &cx->M, j.cap_M, slt, &cp->dc_out, maps_d.p, prefix_d.p, line_scr.p, start_d.as<uint16_t>(), csL))
                    return -1;
                if (launch_linecode_count(ev, &cx->M, j.cap_M, slt, start_d.as<uint16_t>(), cnts_d.p, cprefix_d.p, line_scr.p, cx->tot, csL)) return -1;
                stats.launches += 9;
                NFC_CUDA_CHECK(cudaMemsetAsync(&cx->flags, 0, 4, csL));
                NFC_CUDA_CHECK(cudaMemcpyAsync(&hx, cx, 64, cudaMemcpyDeviceToHost, csL));
                NFC_CUDA_CHECK(sync_on(csL));
            }
            j.cap_sym = hx.tot[0]; j.cap_b0 = hx.tot[1]; j.cap_b1 = hx.tot[2]; j.cap_em = hx.tot[3];
        } else {
            j.cap_sym = cap_of(rates.sym); j.cap_b0 = cap_of(rates.b0); j.cap_b1 = cap_of(rates.b1); j.cap_em = cap_of(rates.em);
        }
        if ((want_sym && sym_d[oi].ensure(((size_t)j.cap_sym + 16) * sizeof(SymbolRec))) || bits0_d[oi].ensure((size_t)j.cap_b0 + 16) ||
            bits1_d[oi].ensure((size_t)j.cap_b1 + 16) || em_d[oi].ensure(((size_t)j.cap_em + 16) * linecode_emission_bytes()) ||
            fx_d[oi].ensure(((size_t)j.cap_em + 16) * 8))
            return -1;
        if (launch_linecode_write(ev, &cx->M, j.cap_M, slt, start_d.as<uint16_t>(), cprefix_d.p, want_sym ? sym_d[oi].as<SymbolRec>() : nullptr,
                                  want_sym ? j.cap_sym : 0, bits0_d[oi].as<uint8_t>(), j.cap_b0, bits1_d[oi].as<uint8_t>(), j.cap_b1, em_d[oi].p,
                                  fx_d[oi].p, j.cap_em, a, cp->bits_out, cx->bits_out, &cx->n_empty, &cx->n_frames, cp->pend_out, &cp->dc_out, &cx->dc_out,
                                  cx->pend_out, csL))
            return -1;
        stats.launches++;
    } else {
        // no decoder runs: its state passes through
        NFC_CUDA_CHECK(cudaMemcpyAsync(&cx->dc_out, &cp->dc_out, sizeof(DecCarry) + 8 + 8 + 16, cudaMemcpyDeviceToDevice, csL));  // dc_out .. bits_out
    }
    NFC_CUDA_CHECK(cudaEventRecord(ev_c[ci], csL));
    NFC_CUDA_CHECK(cudaMemcpyAsync(ctx_h + (size_t)ci * 256, cx, 256, cudaMemcpyDeviceToHost, csL));
    NFC_CUDA_CHECK(cudaEventRecord(ev_ctx[ci], csL));
    NFC_CUDA_CHECK(cudaEventRecord(evL[ci], csL));
    j.want_ev = (prm.outputs & NFC_OUT_EVENTS) != 0;
    j.want_sym = want_sym && want_line;
    j.want_fr = (prm.outputs & NFC_OUT_FRAMES) != 0 && want_line;
    j.t2 = now_ms();
    jobs.push_back(j);
    // the slab before this one: its chain has run (or is about to end) while this one was queued
    while (jobs.size() > 1)
        if (finalize_front()) return -1;
    return 0;
}

// Everything queued has been looked at: wait for the last frame records to arrive (slabs without event or symbol output have
// no worker thread that would).
int Stream::settle_frames() {
    if (have_last_records) {
        // the copy events sleep when waited for (worker threads wait on them); the caller's thread is about to read the
        // records and polls instead, unless the stream was told to keep its waits off the cores (nfc_stream_set_wait_mode):
        // waking up costs 0.25 ms, which a work()-sized call would pay every time
        cudaError_t e;
        if (blocking_wait) e = cudaEventSynchronize(ev_last_records);
        else
            while ((e = cudaEventQuery(ev_last_records)) == cudaErrorNotReady) {}
        NFC_CUDA_CHECK(e);
        have_last_records = false;
    }
    return 0;
}

// The context block of the oldest queued slab has arrived: take over its carries, put its records on their way to the
// host and hand them to the worker thread -- or, if a buffer was too small for it, do it (and whatever was queued behind
// it) again with exact sizes.
int Stream::finalize_front() {
    if (jobs.empty()) return 0;
    static const bool timing = getenv("NFC_TIMING") != nullptr;
    const SlabJob j = jobs.front();
    const int ci = (int)(j.seq % NCTX), oi = (int)(j.seq & 1);
    NFC_CUDA_CHECK(cudaEventSynchronize(ev_ctx[ci]));
    const double t3 = now_ms();
    PostCtx hx;
    memcpy(&hx, ctx_h + (size_t)ci * 256, sizeof(hx));
    bool bad = false;
    if (!j.exact) {
        bad = (hx.flags & (POST_OVF_TRANS | POST_OVF_EVENTS | POST_UNRESOLVED)) != 0 || hx.R > j.cap_R || hx.M > j.cap_M;
        if (j.have_line)
            bad = bad || (j.want_sym && hx.tot[0] > j.cap_sym) || hx.tot[1] > j.cap_b0 || hx.tot[2] > j.cap_b1 || hx.tot[3] > j.cap_em;
    } else if (hx.flags & (POST_OVF_TRANS | POST_OVF_EVENTS | POST_UNRESOLVED)) {
        set_error("internal: a slab sized exactly reports flags %u", hx.flags);
        return -1;
    }
    if (bad) {
        // sizes taken from the slabs before did not hold (or the frame-boundary search needs the scan): this slab and the
        // ones queued behind it (they started from its carries) again, sized exactly; their bitmap is still in place
        std::vector<SlabJob> again(jobs.begin(), jobs.end());
        jobs.clear();
        NFC_CUDA_CHECK(cudaStreamSynchronize(cs));
        NFC_CUDA_CHECK(cudaStreamSynchronize(csR));
        NFC_CUDA_CHECK(cudaStreamSynchronize(csL));
        stats.overflow_retries++;
        slab_seq = j.seq;
        for (const SlabJob &r : again) {
            if (!r.from_bitmap) {
                set_error("internal: a slab without bitmap cannot be done again");
                return -1;
            }
            if (post_chain(r.a, r.b, true, 0, true, r.t0, r.t1)) return -1;  // finalizes the one before it
        }
        return 0;
    }
    jobs.pop_front();
    const uint32_t M = hx.M, nsym = hx.tot[0], nbit0 = hx.tot[1], nbit1 = hx.tot[2];
    const uint32_t nemit = hx.n_frames;  // (tot[3] may count one frame per type more: an empty one, linecode.cu ChunkCnt)
    // ---- carries and sizes
    run_carry = hx.rc_out;
    dec_carry = hx.dc_out;
    pending[0] = hx.pend_out[0];
    pending[1] = hx.pend_out[1];
    if (!j.events_only) {
        const double n = (double)std::max<int64_t>(1, j.b - j.a);
        auto upd = [&](double &r, uint32_t v) { r = std::max(r * 0.98, (double)v / n); };
        upd(rates.R, hx.R); upd(rates.M, M); upd(rates.sym, nsym); upd(rates.b0, nbit0); upd(rates.b1, nbit1); upd(rates.em, nemit);
        rates.have = true;
    }
    float ms_ab = 0, ms_ac = 0, ms_cc = 0;
    cudaEventElapsedTime(&ms_ab, ev_a[ci], ev_b[ci]);
    cudaEventElapsedTime(&ms_ac, ev_a[ci], ev_c[ci]);
    // chains of consecutive slabs overlap: the device time this slab adds ends at its chain's end and begins at the end of
    // the chain before it, if that came later than this slab's own begin
    if (last_final_seq == j.seq - 1 && j.seq > chain_first_seq &&
        cudaEventElapsedTime(&ms_cc, ev_c[(j.seq + NCTX - 1) % NCTX], ev_c[ci]) == cudaSuccess && ms_cc > 0 && ms_cc < ms_ac)
        ms_ac = ms_cc;
    last_final_seq = j.seq;
    stats.slicer_ms += ms_ab;
    stats.kernel_ms += ms_ac;

    // ---- records back to the host (cs2; the chain has completed: the host has seen its context block)
    const bool want_ev = j.want_ev, want_sym = j.want_sym, want_fr = j.want_fr;
    size_t off_ev = 0, off_sym = 0, total = 0;
    auto place = [&](size_t bytes) {
        size_t o = total;
        total += (bytes + 63) / 64 * 64;
        return o;
    };
    place(64);
    if (want_ev) off_ev = place((size_t)M * sizeof(EventRec));
    if (want_sym) off_sym = place((size_t)nsym * sizeof(SymbolRec));
    const int pi = (int)(slabs_enqueued % NPIN);
    // the slab that used this buffer last (three slabs ago) must be in the output vectors: long done, normally
    while (slabs_marshalled.load(std::memory_order_acquire) < slabs_enqueued - (NPIN - 1)) std::this_thread::yield();
    if (ensure_pinned(pi, total)) return -1;
    char *hp = (char *)pinned[pi];
    if (want_fr) {
        // The slab's frame records, their packed index and the frame bits go straight behind those of the slabs before, in
        // page-locked memory; an arena that has to grow moves: no copy into it may be in flight then, and the worker threads
        // must be done with what they were given.
        const uint32_t nb[2] = {nbit0, nbit1};
        const size_t f0 = out_frames.size();
        const bool grow_any = fb[0].len + nb[0] > fb[0].cap || fb[1].len + nb[1] > fb[1].cap || f0 + nemit > out_frames.cap ||
                              f0 + nemit > findex_cap;
        if (grow_any) {
            if (join_marshal()) return -1;
            NFC_CUDA_CHECK(cudaStreamSynchronize(cs2));
            if (findex_n != f0) {
                set_error("internal: frame index out of step");
                return -1;
            }
            if (fb[0].reserve(fb[0].len + nb[0]) || fb[1].reserve(fb[1].len + nb[1]) || out_frames.reserve(f0 + nemit)) {
                set_error("out of page-locked memory for the frames of a slab");
                return -1;
            }
            if (findex_reserve(f0 + nemit)) {
                set_error(findex_ext ? "more frames than the caller's frame index buffer holds (nfc_stream_set_frame_index_buffer)"
                                     : "out of page-locked memory for the frame index");
                return -1;
            }
        }
        if (nemit) {
            NFC_CUDA_CHECK(cudaMemcpyAsync(out_frames.p + f0, em_d[oi].p, (size_t)nemit * sizeof(nfc_frame), cudaMemcpyDeviceToHost, cs2));
            NFC_CUDA_CHECK(cudaMemcpyAsync(findex + f0, fx_d[oi].p, (size_t)nemit * 8, cudaMemcpyDeviceToHost, cs2));
        }
        if (nbit0) NFC_CUDA_CHECK(cudaMemcpyAsync(fb[0].p + fb[0].len, bits0_d[oi].p, nbit0, cudaMemcpyDeviceToHost, cs2));
        if (nbit1) NFC_CUDA_CHECK(cudaMemcpyAsync(fb[1].p + fb[1].len, bits1_d[oi].p, nbit1, cudaMemcpyDeviceToHost, cs2));
        // bits up to the last closing of a type are handed out with the frames (the line-code totals know where that is)
        if (hx.tot[4] & 1) fb[0].closed = fb[0].len + nbit0 - hx.tot[5];
        if (hx.tot[6] & 1) fb[1].closed = fb[1].len + nbit1 - hx.tot[7];
        fb[0].len += nbit0;
        fb[1].len += nbit1;
        out_frames.n = f0 + nemit;
        findex_n = f0 + nemit;
        stats.empty_frames += hx.n_empty & 0x7fffffffu;
        if (hx.n_empty >> 31) findex_bad = true;  // a position or a length that the packed index cannot hold
        total += (size_t)nbit0 + nbit1 + (size_t)nemit * (sizeof(nfc_frame) + 8);
    }
    if (want_ev && M) NFC_CUDA_CHECK(cudaMemcpyAsync(hp + off_ev, events_d[oi].p, (size_t)M * sizeof(EventRec), cudaMemcpyDeviceToHost, cs2));
    if (want_sym && nsym)
        NFC_CUDA_CHECK(cudaMemcpyAsync(hp + off_sym, sym_d[oi].p, (size_t)nsym * sizeof(SymbolRec), cudaMemcpyDeviceToHost, cs2));
    NFC_CUDA_CHECK(cudaEventRecord(ev_d[pi], cs2));
    NFC_CUDA_CHECK(cudaEventRecord(ev_out[oi], cs2));
    ev_out_set[oi] = true;
    slabs_enqueued++;
    stats.d2h_bytes += (int64_t)total + 256;
    if (timing)
        fprintf(stderr, "slab %lld..%lld%s: slicer %.2f ms (dev %.2f), chain queued in %.2f (dev %.2f), context seen %.2f ms after queuing\n",
                (long long)j.a, (long long)j.b, j.exact ? " (exact sizes)" : "", j.t1 - j.t0, ms_ab, j.t2 - j.t1, ms_ac - ms_ab, t3 - j.t2);
    if (!want_ev && !want_sym) {  // nothing for a worker thread to do: the frames arrive where they belong by DMA
        ev_last_records = ev_d[pi];
        have_last_records = true;
        slabs_marshalled.fetch_add(1, std::memory_order_release);
        return 0;
    }
    return marshal(j, pi, hp, off_ev, off_sym, M, nsym);
}

// Event and symbol records of a slab -> output vectors (absolute positions) on a worker thread: it waits for its predecessor
// (the vectors are filled in slab order), then for the slab's records to arrive (the slab's frames, copied before them on the
// same stream, have arrived by then as well).
int Stream::marshal(const SlabJob &j, int pi, char *hp, size_t off_ev, size_t off_sym, uint32_t M, uint32_t nsym) {
    const int64_t a = j.a;
    const bool want_ev = j.want_ev, want_sym = j.want_sym;
    if (marshal_err.load()) return join_marshal();
    auto prev = std::make_shared<std::thread>(std::move(marshal_thr));
    const cudaEvent_t evd = ev_d[pi];
    const int dev = prm.device;
    marshal_thr = std::thread([this, prev, evd, dev, hp, off_ev, off_sym, M, nsym, a, want_ev, want_sym]() {
      if (prev->joinable()) prev->join();
      cudaSetDevice(dev);
      static const bool timing = getenv("NFC_TIMING") != nullptr;
      const double tm0 = timing ? now_ms() : 0.0;
      double tm1 = tm0;
      if (cudaEventSynchronize(evd) != cudaSuccess) marshal_err = 2;
      else [&]() {
        if (timing) tm1 = now_ms();
        auto grow = [](auto &v, size_t more) {  // geometric: an exact reserve per slab would copy the vector every slab
            if (v.capacity() < v.size() + more) v.reserve(std::max(v.size() + more, v.capacity() * 2));
        };
        // ---- marshal records (absolute positions)
        if (want_ev) {
            const EventRec *e = reinterpret_cast<const EventRec *>(hp + off_ev);
            grow(out_events, M);
            for (uint32_t i = 0; i < M; i++) {
                nfc_event o;
                o.pos = a + (int64_t)e[i].rel_pos;
                o.d = e[i].d;
                o.v = e[i].v;
                o.type = e[i].type;
                o.pad = 0;
                out_events.push_back(o);
            }
        }
        if (want_sym) {
            const SymbolRec *s = reinterpret_cast<const SymbolRec *>(hp + off_sym);
            grow(out_symbols, nsym);
            for (uint32_t i = 0; i < nsym; i++) {
                nfc_symbol o;
                o.pos = a + (int64_t)s[i].rel_pos;
                o.type = s[i].type;
                o.val = s[i].val;
                o.pad = 0;
                o.pad2 = 0;
                out_symbols.push_back(o);
            }
        }
      }();
      if (timing) fprintf(stderr, "  records of slab at %lld: waited %.2f ms for them, into the output vectors in %.2f ms\n", (long long)a, tm1 - tm0, now_ms() - tm1);
      slabs_marshalled.fetch_add(1, std::memory_order_release);
    });
    return 0;
}

}  // namespace nfc

// =================================================================================== extern "C"
using nfc::Stream;
struct nfc_stream {
    Stream s;
};

template <class T>
static int64_t drain_vec(std::vector<T> &v, size_t &head, T *out, int64_t cap) {
    const int64_t avail = (int64_t)(v.size() - head);
    if (cap <= 0 || !out) return avail;
    const int64_t n = std::min(avail, cap);
    memcpy(out, v.data() + head, (size_t)n * sizeof(T));
    head += (size_t)n;
    if (head == v.size()) {
        v.clear();
        head = 0;
    }
    return n;
}

extern "C" {

void nfc_default_params(nfc_params *p) {
    memset(p, 0, sizeof(*p));
    p->samp_rate = 2e6;
    p->lo_val = 0.1;
    p->hi_val = 1.1;
    p->av_window = 2000;
    p->max_len = 50;
    p->decode_reader = 1;
    p->decode_tag = 1;
    p->input_kind = NFC_IN_ENVELOPE_F32;
    p->outputs = NFC_OUT_EVENTS | NFC_OUT_SYMBOLS | NFC_OUT_FRAMES | NFC_OUT_DROPPED_EVENTS;
    p->device = 0;
    p->pcm_scale = 32767.0f;
}

int nfc_stream_create(const nfc_params *p, nfc_stream **out) {
    if (!p || !out) {
        nfc::set_error("null argument");
        return -1;
    }
    if (p->input_kind < NFC_IN_ENVELOPE_F32 || p->input_kind > NFC_IN_SC16) {
        nfc::set_error("unknown input_kind %d (NFC_IN_ENVELOPE_F32 .. NFC_IN_SC16: 0 .. 4)", (int)p->input_kind);
        return -1;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        nfc::set_error("no CUDA device: this library has no CPU path");
        return -1;
    }
    nfc_stream *h = new (std::nothrow) nfc_stream();
    if (!h) {
        nfc::set_error("out of memory");
        return -1;
    }
    if (h->s.init(p)) {
        h->s.destroy();
        delete h;
        return -1;
    }
    *out = h;
    return 0;
}

int nfc_stream_destroy(nfc_stream *h) {
    if (!h) return 0;
    cudaSetDevice(h->s.prm.device);
    h->s.destroy();
    delete h;
    return 0;
}

int nfc_stream_reset(nfc_stream *h) {
    if (!h) return -1;
    Stream &s = h->s;
    s.settle();
    s.pos = 0;
    s.stable = false;
    s.serial_mode = false;
    s.bm_lo = s.bm_hi = 0;
    s.warm.clear();
    s.run_carry = nfc::RunCarry{0, 0, 0, 0};
    s.dec_carry = nfc::DecCarry{0, 0, {0, 0}};
    s.pending[0] = s.pending[1] = 0;
    s.fb[0].clear();
    s.fb[1].clear();
    s.out_events.clear();
    s.out_symbols.clear();
    s.out_frames.clear();
    s.findex_n = 0;
    s.findex_bad = false;
    s.ev_head = s.sym_head = s.fr_head = 0;
    return 0;
}

int nfc_stream_set_thresholds(nfc_stream *h, double lo_val, double hi_val) {
    if (!h) return -1;
    Stream &s = h->s;
    if (s.settle()) return -1;
    if (s.pos != 0 || s.stable || !s.warm.empty()) {
        nfc::set_error("set_thresholds: the stream has consumed samples; reset it first");
        return -1;
    }
    cudaSetDevice(s.prm.device);
    s.prm.lo_val = lo_val;
    s.prm.hi_val = hi_val;
    s.sp.lo = lo_val;
    s.sp.hi = hi_val;
    s.sp.loL = s.sp.lo / s.sp.Ld;
    s.sp.hiL = s.sp.hi / s.sp.Ld;
    s.sp.cls_ss0_x0 = nfc::classify_ratio_host(1.0, s.sp.lo, s.sp.hi);
    s.sp.cls_ss0_xn = nfc::classify_ratio_host(s.sp.hi + 0.1, s.sp.lo, s.sp.hi);
    NFC_CUDA_CHECK(cudaMemcpyAsync(s.params_d.p, &s.sp, sizeof(s.sp), cudaMemcpyHostToDevice, s.cs));
    NFC_CUDA_CHECK(s.sync_cs());
    return 0;
}

int64_t nfc_stream_push(nfc_stream *h, const void *items, int64_t n, int mem, int *called_back) {
    if (!h || (n > 0 && !items)) {
        nfc::set_error("null argument");
        return -1;
    }
    return h->s.push(items, n, mem, called_back);
}

int64_t nfc_stream_push_batch(nfc_stream *h, const void *items, int mem, int64_t n_captures, int64_t items_per_capture,
                              int64_t stride_items, const double *lo_vals, const double *hi_vals, int64_t *pitch) {
    if (!h || !items) {
        nfc::set_error("null argument");
        return -1;
    }
    if (h->s.settle()) return -1;
    return h->s.push_batch(items, mem, n_captures, items_per_capture, stride_items, lo_vals, hi_vals, pitch);
}

int64_t nfc_stream_push_batch_ragged(nfc_stream *h, const void *const *items, int mem, int64_t n_captures, const int64_t *lengths,
                                     const double *lo_vals, const double *hi_vals, int64_t *starts) {
    if (!h || !items || !lengths || !starts) {
        nfc::set_error("null argument");
        return -1;
    }
    if (h->s.settle()) return -1;
    return h->s.push_batch_ragged(items, mem, n_captures, lengths, lo_vals, hi_vals, starts);
}

int64_t nfc_stream_push_events(nfc_stream *h, const nfc_event *ev, int64_t n) {
    if (!h) {
        nfc::set_error("null argument");
        return -1;
    }
    return h->s.push_events(ev, n);
}

int64_t nfc_stream_drain_events(nfc_stream *h, nfc_event *out, int64_t cap) {
    if (!h || h->s.settle()) return -1;
    return drain_vec(h->s.out_events, h->s.ev_head, out, cap);
}

int64_t nfc_stream_drain_symbols(nfc_stream *h, nfc_symbol *out, int64_t cap) {
    if (!h || h->s.settle()) return -1;
    return drain_vec(h->s.out_symbols, h->s.sym_head, out, cap);
}

int64_t nfc_stream_pending_frame_bits(nfc_stream *h) {
    if (!h || h->s.settle()) return -1;
    return (int64_t)(h->s.fb[0].closed + h->s.fb[1].closed);
}

int64_t nfc_stream_drain_frames(nfc_stream *h, nfc_frame *out, int64_t cap, uint8_t *bits, int64_t bits_cap) {
    if (!h || h->s.settle()) return -1;
    Stream &s = h->s;
    const int64_t avail = (int64_t)s.out_frames.size();
    if (cap <= 0 || !out) return avail;
    const int64_t nb0 = (int64_t)s.fb[0].closed, nb1 = (int64_t)s.fb[1].closed;
    if (cap < avail || bits_cap < nb0 + nb1 || (!bits && nb0 + nb1 > 0)) {
        nfc::set_error("drain_frames: buffers too small (%lld frames, %lld bits pending)", (long long)avail,
                       (long long)(nb0 + nb1));
        return -2;
    }
    // all pending frames at once: tag->reader bits first, then reader->tag bits (large drains: copied by helper threads)
    auto copy_frames = [&](int64_t i0, int64_t i1) {
        for (int64_t i = i0; i < i1; i++) {
            out[i] = s.out_frames[(size_t)i];
            if (out[i].type == 1) out[i].bit_off += nb0;
        }
    };
    if (nb0 + nb1 > (4 << 20)) {
        std::thread t0([&] { if (nb0) memcpy(bits, s.fb[0].p, (size_t)nb0); });
        std::thread t1([&] { if (nb1) memcpy(bits + nb0, s.fb[1].p, (size_t)nb1); });
        std::thread t2([&] { copy_frames(0, avail / 2); });
        copy_frames(avail / 2, avail);
        t0.join();
        t1.join();
        t2.join();
    } else {
        if (nb0) memcpy(bits, s.fb[0].p, (size_t)nb0);
        if (nb1) memcpy(bits + nb0, s.fb[1].p, (size_t)nb1);
        copy_frames(0, avail);
    }
    s.out_frames.clear();
    s.findex_n = 0;
    s.findex_bad = false;
    s.fb[0].consume();
    s.fb[1].consume();
    s.fr_head = 0;
    return avail;
}

int64_t nfc_stream_view_frames(nfc_stream *h, const nfc_frame **frames, const uint8_t **bits_tag, int64_t *n_bits_tag,
                               const uint8_t **bits_reader, int64_t *n_bits_reader) {
    if (!h || !frames || !bits_tag || !n_bits_tag || !bits_reader || !n_bits_reader) {
        nfc::set_error("null argument");
        return -1;
    }
    if (getenv("NFC_TIMING")) {
        const double t0 = nfc::now_ms();
        if (h->s.finish_pending()) return -1;
        const double t1 = nfc::now_ms();
        if (h->s.join_marshal()) return -1;
        fprintf(stderr, "view_frames: last slab's records %.2f ms, its marshalling %.2f ms\n", t1 - t0, nfc::now_ms() - t1);
    }
    if (h->s.settle()) return -1;
    Stream &s = h->s;
    *frames = s.out_frames.data();
    *bits_tag = s.fb[0].p;
    *n_bits_tag = (int64_t)s.fb[0].closed;
    *bits_reader = s.fb[1].p;
    *n_bits_reader = (int64_t)s.fb[1].closed;
    return (int64_t)s.out_frames.size();
}

int64_t nfc_stream_view_frame_index(nfc_stream *h, const uint64_t **index) {
    if (!h || !index) {
        nfc::set_error("null argument");
        return -1;
    }
    if (h->s.settle()) return -1;
    Stream &s = h->s;
    if (s.findex_bad || s.findex_n != s.out_frames.size()) {
        nfc::set_error("view_frame_index: a frame does not fit the packing (position >= 2^40 or more than 65535 bits)");
        return -1;
    }
    *index = s.findex;
    return (int64_t)s.findex_n;
}

int nfc_stream_set_frame_index_buffer(nfc_stream *h, uint64_t *buf, int64_t cap) {
    if (!h || (buf && cap <= 0)) {
        nfc::set_error("bad argument");
        return -1;
    }
    if (h->s.settle()) return -1;
    Stream &s = h->s;
    if (!s.out_frames.empty()) {
        nfc::set_error("set_frame_index_buffer: the stream holds frames; release them first");
        return -1;
    }
    cudaSetDevice(s.prm.device);
    s.findex_drop();
    s.findex = buf;
    s.findex_ext = buf != nullptr;
    s.findex_cap = buf ? (size_t)cap : 0;
    if (buf) {
        // memory that is page-locked already (or cannot be locked) is used as it is: the copies into it are then staged by the driver
        s.findex_ext_locked = cudaHostRegister(buf, (size_t)cap * 8, cudaHostRegisterPortable) == cudaSuccess;
        if (!s.findex_ext_locked) cudaGetLastError();
    }
    s.findex_n = 0;
    s.findex_bad = false;
    return 0;
}

int nfc_stream_release_frames(nfc_stream *h) {
    if (!h || h->s.settle()) return -1;
    Stream &s = h->s;
    s.out_frames.clear();
    s.findex_n = 0;
    s.findex_bad = false;
    s.fb[0].consume();
    s.fb[1].consume();
    s.fr_head = 0;
    return 0;
}

int nfc_stream_get_state(nfc_stream *h, nfc_state *st, float *ring, uint8_t *pending_bits) {
    if (!h || !st) {
        nfc::set_error("null argument");
        return -1;
    }
    if (h->s.settle()) return -1;
    Stream &s = h->s;
    memset(st, 0, sizeof(*st));
    st->pos = s.pos;
    st->stable = s.stable ? 1 : 0;
    st->serial_mode = s.serial_mode ? 1 : 0;
    st->lastL = nfc::NO_POS;
    st->lrun_start = nfc::NO_POS;
    if (s.stable) {
        cudaSetDevice(s.prm.device);
        std::vector<char> blk(nfc::state_block_bytes(s.sp.L));
        NFC_CUDA_CHECK(cudaMemcpy(blk.data(), s.state.p, blk.size(), cudaMemcpyDeviceToHost));
        const nfc::SlicerHdr *hd = reinterpret_cast<const nfc::SlicerHdr *>(blk.data());
        st->ss = hd->ss;
        st->lastL = hd->lastL;
        st->lrun_start = hd->lrun_start;
        st->index = (int32_t)(s.pos % s.sp.L);
        if (ring) memcpy(ring, nfc::state_ring(hd), (size_t)s.sp.L * 4);
        st->cur_state = s.run_carry.st;
        st->last_bit = s.run_carry.last_bit;
        st->dur = s.run_carry.dur;
    } else {
        st->dur = 1;  // transition_sink.py:22
        if (ring) {
            memset(ring, 0, (size_t)s.sp.L * 4);
            if (!s.warm.empty()) memcpy(ring, s.warm.data(), s.warm.size() * 4);
        }
    }
    st->miller_state = s.dec_carry.miller_state;
    st->manch_state = s.dec_carry.manch_state;
    for (int t = 0; t < 2; t++) {
        st->started[t] = s.dec_carry.started[t];
        st->pending[t] = (int32_t)s.pending[t];
    }
    if (pending_bits) {
        size_t o = 0;
        for (int t = 0; t < 2; t++) {
            const size_t open = s.fb[t].len - s.fb[t].closed;
            if (open) memcpy(pending_bits + o, s.fb[t].p + s.fb[t].closed, open);
            o += open;
        }
    }
    return 0;
}

int nfc_stream_set_state(nfc_stream *h, const nfc_state *st, const float *ring, const uint8_t *pending_bits) {
    if (!h || !st) {
        nfc::set_error("null argument");
        return -1;
    }
    Stream &s = h->s;
    s.bm_lo = s.bm_hi = 0;
    if (s.settle()) return -1;
    if (!st->stable || !ring) {
        nfc::set_error("set_state needs a stable state with its ring");
        return -1;
    }
    cudaSetDevice(s.prm.device);
    std::vector<char> blk(nfc::state_block_bytes(s.sp.L), 0);
    nfc::SlicerHdr *hd = reinterpret_cast<nfc::SlicerHdr *>(blk.data());
    hd->ss = st->ss;
    hd->pos = st->pos;
    if (st->lastL == INT64_MIN) {
        // hysteresis carry not supplied (a state saved from the reference's attributes): it is a function
        // of (cur_state, last_bit, dur) -- see vals_from_classes in tests/algomodel.py
        const int64_t P = st->pos;
        if (st->cur_state == 2 && st->last_bit == -1) {
            hd->lastL = P - 1;
            hd->lrun_start = P - st->dur;
        } else if (st->cur_state == 2) {
            hd->lastL = P - st->dur - 1;
            hd->lrun_start = hd->lastL;
        } else if (st->last_bit == -1) {  // timeout on the last LOW sample: cur_state back to 0, run continues
            hd->lastL = P - 1;
            hd->lrun_start = P - 1 - s.sp.mx;
        } else {
            hd->lastL = nfc::NO_POS;
            hd->lrun_start = nfc::NO_POS;
        }
    } else {
        hd->lastL = st->lastL;
        hd->lrun_start = st->lrun_start;
    }
    hd->last_val = st->last_bit;
    memcpy(nfc::state_ring(hd), ring, (size_t)s.sp.L * 4);
    NFC_CUDA_CHECK(cudaMemcpy(s.state.p, blk.data(), blk.size(), cudaMemcpyHostToDevice));
    s.pos = st->pos;
    s.stable = true;
    s.serial_mode = st->serial_mode != 0;
    s.run_carry.st = st->cur_state;
    s.run_carry.last_bit = st->last_bit;
    s.run_carry.dur = st->dur;
    s.dec_carry.miller_state = st->miller_state;
    s.dec_carry.manch_state = st->manch_state;
    size_t o = 0;
    for (int t = 0; t < 2; t++) {
        s.dec_carry.started[t] = st->started[t];
        s.pending[t] = (uint32_t)st->pending[t];
        // the open bits behind whatever has not been handed out yet
        s.fb[t].len = s.fb[t].closed;
        if (s.fb[t].reserve(s.fb[t].len + (size_t)st->pending[t] + 64)) {
            nfc::set_error("out of page-locked memory");
            return -1;
        }
        if (pending_bits) memcpy(s.fb[t].p + s.fb[t].len, pending_bits + o, (size_t)st->pending[t]);
        else memset(s.fb[t].p + s.fb[t].len, 0, (size_t)st->pending[t]);
        s.fb[t].len += (size_t)st->pending[t];
        o += (size_t)st->pending[t];
    }
    return 0;
}

int nfc_stream_set_wait_mode(nfc_stream *h, int blocking) {
    if (!h) return -1;
    return h->s.set_wait_mode(blocking != 0);
}

int nfc_stream_set_tuning(nfc_stream *h, int64_t seg_len, int64_t halo, int64_t slab_len, int force_serial) {
    if (!h) return -1;
    h->s.seg_len = seg_len;
    h->s.halo = halo;
    h->s.slab_len = slab_len;
    h->s.force_serial = force_serial;
    return 0;
}

int nfc_stream_get_stats(nfc_stream *h, nfc_stats *st) {
    if (!h || !st) return -1;
    h->s.finish_pending();
    cudaSetDevice(h->s.prm.device);
    unsigned long long ts[16] = {0};
    if (nfc::slicer_tile_stats(ts, false) == 0) {  // device-wide counters (all streams of this process)
        h->s.stats.fast_tiles = (int64_t)ts[0];
        h->s.stats.exact_tiles = (int64_t)ts[1];
        h->s.stats.repeated_passes = (int64_t)ts[5];
        h->s.stats.fixpoint_tiles = (int64_t)ts[3];
        h->s.stats.st2_tiles = (int64_t)ts[6];
        h->s.stats.unproven_tiles = (int64_t)(ts[2] + ts[7]);
        h->s.stats.ring_resums = (int64_t)ts[4];
        h->s.stats.exact_rounds = (int64_t)ts[8];
        h->s.stats.pipe_tiles = (int64_t)ts[11];
        h->s.stats.pipe_runs = (int64_t)ts[12];
        h->s.stats.pipe_aborts = (int64_t)ts[13];
        if (getenv("NFC_TIMING"))
            fprintf(stderr, "slicer segments: %llu cycles in all, %llu of them inside pipelined runs (%llu tiles of %llu)\n", ts[15], ts[14], ts[11], ts[0]);
    }
    *st = h->s.stats;
    return 0;
}

int nfc_stream_reset_stats(nfc_stream *h) {
    if (!h) return -1;
    memset(&h->s.stats, 0, sizeof(h->s.stats));
    unsigned long long ts[16];
    cudaSetDevice(h->s.prm.device);
    nfc::slicer_tile_stats(ts, true);
    return 0;
}

void *nfc_stream_cuda_stream(nfc_stream *h) { return h ? (void *)h->s.cs : nullptr; }

int nfc_build_tables(double samp_rate, int32_t max_len, int which, uint8_t *dclass, int32_t dclass_cap, uint16_t *table,
                     int32_t table_cap, int32_t *n_dclass) {
    nfc::HostTables t;
    if (!(samp_rate > 0) || max_len < 1 || !nfc::build_tables(max_len, 1e6 / samp_rate, t)) {
        nfc::set_error("cannot build line-code tables for samp_rate=%g max_len=%d", samp_rate, max_len);
        return -1;
    }
    const std::vector<uint8_t> &dc = which ? t.dclass_miller : t.dclass_manch;
    const std::vector<nfc::TabEntry> &tb = which ? t.miller : t.manch;
    if (n_dclass) *n_dclass = which ? t.n_dclass_miller : t.n_dclass_manch;
    if (dclass && dclass_cap >= (int32_t)dc.size()) memcpy(dclass, dc.data(), dc.size());
    if (table && table_cap >= (int32_t)tb.size()) memcpy(table, tb.data(), tb.size() * sizeof(uint16_t));
    return (int)tb.size();
}

int nfc_synth_render(void *dev_out, int64_t n, int64_t first_index, const int8_t *codes, const int64_t *lens,
                     int64_t n_runs, float carrier, float pause, float tag_high, float noise, float fade,
                     double fade_period, uint64_t seed, int as_envelope, int device) {
    if (cudaSetDevice(device) != cudaSuccess) {
        nfc::set_error("cudaSetDevice(%d) failed", device);
        return -1;
    }
    return nfc::synth_render(dev_out, n, first_index, codes, lens, n_runs, carrier, pause, tag_high, noise, fade, fade_period, seed,
                             as_envelope, nullptr);
}

const char *nfc_last_error(void) { return nfc::g_err; }
int nfc_abi_version(void) { return NFC_ABI_VERSION; }

int nfc_abi_sizeof(int which) {
    switch (which) {
        case 0: return (int)sizeof(nfc_params);
        case 1: return (int)sizeof(nfc_event);
        case 2: return (int)sizeof(nfc_symbol);
        case 3: return (int)sizeof(nfc_frame);
        case 4: return (int)sizeof(nfc_frame_tail);
        case 5: return (int)sizeof(nfc_state);
        case 6: return (int)sizeof(nfc_stats);
        default: return -1;
    }
}
int nfc_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

}  // extern "C"
