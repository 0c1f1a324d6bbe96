// common.cuh -- records, parameters and small device helpers shared by the kernels.
//
// Data flow (one slab of one stream; all buffers live in HBM):
//   samples --slicer.cu--> val transitions --runs.cu--> events --linecode.cu--> symbols --> frames
// The reference computes all of this in one per-sample Python loop plus two per-event FSMs
// (transition_sink.py:55-99, manchester.py:30-61, miller.py:153-197, packets.py:67-79).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace nfc {

// ---- records crossing kernel boundaries -------------------------------------------------
// A change of the slicer's `val` (transition_sink.py:67-77): packed (rel_pos << 2) | (val + 1),
// rel_pos relative to the slab's first sample.
typedef uint32_t TransRec;
__host__ __device__ inline TransRec pack_trans(uint32_t rel_pos, int val) { return (rel_pos << 2) | (uint32_t)(val + 1); }
__host__ __device__ inline uint32_t trans_pos(TransRec t) { return t >> 2; }
__host__ __device__ inline int trans_val(TransRec t) { return (int)(t & 3u) - 1; }

// One element of the list transition_sink passes to its callback (transition_sink.py:89-90,97).
struct __align__(8) EventRec {
    uint32_t rel_pos;  // sample (relative to the slab) whose processing emitted it
    uint16_t d;        // duration in samples, 1..max_len   (dur_us = d * factor)
    int8_t v;          // -1..2
    int8_t type;       // cur_state - 1: -1 dropped by background.py, 0 tag->reader, 1 reader->tag
};

// One cpp.append_bit(val, type) call (manchester.py:28, miller.py:151).
struct __align__(8) SymbolRec {
    uint32_t rel_pos;
    int8_t type;
    int8_t val;  // 0/1 or ErrorCode 2..7
    int16_t pad;
};

// One fsm.process_bits(bits, type) hand-off (packets.py:94-98).
struct __align__(8) FrameRec {
    int64_t pos;      // absolute stream index of the closing event
    int64_t bit_off;  // into the stream's frame-bit buffer (one byte per bit)
    int32_t nbits;
    int32_t type;
};

// ---- slicer parameters -------------------------------------------------------------------
enum InputKind { IN_ENVELOPE_F32 = 0, IN_REAL_F32 = 1, IN_IQ_F32 = 2, IN_PCM_S16 = 3, IN_SC16 = 4 };

struct SlicerParams {
    double lo, hi;   // lo_val, hi_val (transition_sink.py:32-33)
    double Ld;       // (double)av_window
    double loL, hiL; // lo / L and hi / L: sample-domain thresholds are ss * loL and ss * hiL
    int L;           // av_window (transition_sink.py:27)
    int mx;          // max_len   (transition_sink.py:20)
    int cls_ss0_x0;  // class when ss == 0 and bit == 0 (ratio = 1)        transition_sink.py:59-61
    int cls_ss0_xn;  // class when ss == 0 and bit != 0 (ratio = hi + 0.1) transition_sink.py:62-63
    int span_limit;  // max (emax - emin) of admitted exponents for which double sums are exact
    int input_kind;
    float pcm_scale; // divisor applied to int16 samples: PCM (blocks.wavfile_source) and sc16 I / Q
};

// Slicer state that crosses tiles, segments, slabs and pushes.  The ring itself (L floats) is
// stored right after the header in a state block.
struct SlicerHdr {
    double ss;           // _sum
    int64_t pos;         // stream index of the next sample
    int64_t lastL;       // stream index of the last LOW-class sample, or NO_POS
    int64_t lrun_start;  // first sample of the LOW run containing lastL
    int32_t last_val;    // val of the last processed sample (== _last_bit)
    int32_t emin, emax;  // biased exponent range of the ring contents / admitted samples
    int32_t status;      // SEG_* flags accumulated while producing this state
    uint32_t count;      // transitions the segment had written when this snapshot was taken
    uint32_t pad;
};
static const int64_t NO_POS = INT64_MIN / 4;

enum SegStatus {
    SEG_OK = 0,
    SEG_INEXACT = 1,    // exponent span exceeded: double sums may round -> needs the serial path
    SEG_NOT_SANE = 2,   // negative / non-finite sample admitted, or ss <= 0 where it matters
    SEG_OVERFLOW = 4,   // transition buffer too small
};

static inline size_t state_block_bytes(int L) { return ((sizeof(SlicerHdr) + (size_t)L * 4 + 255) / 256) * 256; }
__host__ __device__ inline float *state_ring(SlicerHdr *h) { return reinterpret_cast<float *>(h + 1); }
__host__ __device__ inline const float *state_ring(const SlicerHdr *h) { return reinterpret_cast<const float *>(h + 1); }

// One unit of slicer work: a time segment of one stream, processed tile by tile by one CTA.
struct SegWork {
    const void *in;      // sample buffer; in[0] has stream index in_pos0 (in_pos0 % 4 == 0, 16-byte aligned)
    int64_t in_pos0;
    int64_t in_begin;    // first stream index that may be read (>= in_pos0; pad items before it are not ours)
    int64_t in_end;      // stream index one past the last sample present in `in`
    int64_t warm_begin;  // first sample processed (== begin when starting from `state_in`)
    int64_t begin;       // first sample whose transitions are written
    int64_t end;         // one past the last sample processed
    int64_t slab_pos0;   // stream index that rel_pos = 0 refers to
    const SlicerHdr *state_in;  // exact state at warm_begin, or nullptr = cold start:
                                // ring <- samples [warm_begin - L, warm_begin) unconditionally,
                                // like the reference's warm-up (transition_sink.py:109-125)
    SlicerHdr *seam_in;   // snapshot at `begin` (cold starts only; may be nullptr)
    // checkpoints of a speculative segment: a redo from the true state stops at the first one it reproduces
    int64_t ckpt_pos[3];  // tile-aligned stream positions (unused entries: INT64_MAX)
    SlicerHdr *ckpt_state[3];
    SlicerHdr *state_out; // state at `end`
    TransRec *trans;      // output, in order
    uint32_t trans_cap;
    uint32_t *trans_count;
    int32_t *status;      // SegStatus flags of this run of the segment
    int32_t param_idx;    // into the SlicerParams array (batches of captures differ in hi_val, rates)
    int32_t pad;
    // bitmap output (streaming kernel): 8 words per chunk of 128 samples, chunk k covers stream positions
    // [bm_pos0 + 128k, bm_pos0 + 128k + 128); words 0-3: val != -1 of sample 4l+j at bit l of word j, words 4-7: val == 1
    uint32_t *bitmap;     // nullptr: transitions are written to `trans` instead
    int64_t bm_pos0;      // multiple of 128
};

// ---- a slab's post-slicer chain (extraction -> runs -> line code) queued without host round trips ----
// Flags the kernels raise in device memory when a buffer sized from the slabs before turns out too small (the host then
// does the slab again with exact sizes), or when the frame-boundary search finds no reset (scan fallback).
enum PostFlags { POST_OVF_TRANS = 1, POST_OVF_EVENTS = 2, POST_UNRESOLVED = 4 };

// ---- run -> event carry (the reference's cur_state / last_bit / dur at a window start) ----
struct RunCarry {
    int32_t st, last_bit, dur;
    int32_t pad;
};

// ---- line-code tables (built on the host by tables.cpp from the decoders' own rules) -------
static const int MILLER_STATES = 16;  // stage(4) x has_started(2) x prev(2)   miller.py:14-29
static const int MANCH_STATES = 8;    // prev_set(2) x prev in {-1,0,1,2}      manchester.py:23-25
static const int MAX_DCLASS = 24;     // distinct duration classes per decoder

// entry: bits 0-3 next state, 4-5 number of outputs, 6-8 out0, 9-11 out1
typedef uint16_t TabEntry;
__host__ __device__ inline int tab_next(TabEntry e) { return e & 15; }
__host__ __device__ inline int tab_nout(TabEntry e) { return (e >> 4) & 3; }
__host__ __device__ inline int tab_out0(TabEntry e) { return (e >> 6) & 7; }
__host__ __device__ inline int tab_out1(TabEntry e) { return (e >> 9) & 7; }

struct LineTables {
    // duration class of d samples (index d, 0..max_len), per decoder
    const uint8_t *dclass_miller;
    const uint8_t *dclass_manch;
    // [dclass][v + 1][state]
    const TabEntry *miller;
    const TabEntry *manch;
    // [dclass][v + 1]: 0xFF or the state every state of the machine is sent to (universal reset)
    const uint8_t *reset_miller;
    const uint8_t *reset_manch;
    int n_dclass_miller, n_dclass_manch;
    int decode_reader, decode_tag;
    // A batch of independent captures decoded as one event stream (every capture its own transition_sink, decoders and
    // PacketProcessors in the reference: transition_sink.py:12-34, background.py:17-25): capture k of a slab owns the
    // slab-relative positions [k * batch_pitch, (k + 1) * batch_pitch); only events at offsets [batch_skip, batch_len) of it
    // are the capture's (before: its warm-up, transition_sink.py:109-125; behind: padding), the others are ignored; the first
    // event of a capture finds both decoders and both PacketProcessors as new.  batch_pitch == 0: one stream.
    uint32_t batch_pitch, batch_skip, batch_len;
};

struct DecCarry {
    int32_t miller_state, manch_state;
    int32_t started[2];  // PacketProcessor._started per type (packets.py:63-65)
};

#define NFC_CUDA_CHECK(expr)                                                                 \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            nfc::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return -1;                                                                       \
        }                                                                                    \
    } while (0)

void set_error(const char *fmt, ...);

}  // namespace nfc
