/*
 * usrp_nfc_b200.h -- C ABI of the B200 sample-rate decode path of usrp_nfc.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++ or torch types.  Each entry
 * point names the reference interface it stands in for (paths relative to the reference's
 * code/ directory).  INTEGRATION.md shows the ctypes binding a maintainer of the reference adds.
 *
 * Conventions: every function returns 0 (or a non-negative count) on success and a negative
 * value on failure, never throws; nfc_last_error() describes the last failure on the calling
 * thread.  The caller owns every buffer it passes in.  One handle = one sample stream; a handle
 * is not thread-safe, distinct handles are independent.  All decoding runs on the GPU: there is
 * no CPU fallback, creation fails when no CUDA device is usable.
 */
#ifndef USRP_NFC_B200_H
#define USRP_NFC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NFC_ABI_VERSION 7

/* what a pushed item is */
enum {
    NFC_IN_ENVELOPE_F32 = 0, /* float32 |z|^2 -- transition_sink's in_sig (transition_sink.py:16)             */
    NFC_IN_REAL_F32 = 1,     /* float32 WAV samples; envelope = x*x on device (decoder.py:25-28)             */
    NFC_IN_IQ_F32 = 2,       /* complex64 from UHD; envelope = re^2+im^2 on device (usrp_src.py:31)          */
    NFC_IN_PCM_S16 = 3,      /* int16 PCM; /pcm_scale, then x*x on device (blocks.wavfile_source, unpinned)  */
    NFC_IN_SC16 = 4          /* complex int16 (UHD sc16: I then Q, 4 B); each /pcm_scale, then re^2+im^2 on device,
                              * exactly as NFC_IN_IQ_F32 for (I/pcm_scale, Q/pcm_scale) (usrp_src.py:31)          */
};
enum { NFC_MEM_HOST = 0, NFC_MEM_DEVICE = 1 };
/* which outputs a stream materialises */
enum { NFC_OUT_EVENTS = 1, NFC_OUT_SYMBOLS = 2, NFC_OUT_FRAMES = 4, NFC_OUT_DROPPED_EVENTS = 8 };

typedef struct nfc_stream nfc_stream;

/* Constructor parameters of transition_sink (transition_sink.py:12) and of background / decoder
 * (background.py:17-21, decoder.py:16): same names, meaning and defaults. */
typedef struct {
    double samp_rate; /* 2e6 */
    double lo_val;    /* 0.1 */
    double hi_val;    /* 1.1 (decoder.py picks 1.1 for uhd, 1.09 for WAV) */
    int32_t av_window; /* 2000, in samples */
    int32_t max_len;   /* 50, in samples   */
    int32_t decode_reader; /* background(reader=...) */
    int32_t decode_tag;    /* background(tag=...)    */
    int32_t input_kind;    /* NFC_IN_*; nfc_stream_create rejects any other value */
    int32_t outputs;       /* NFC_OUT_* bit mask; NFC_OUT_DROPPED_EVENTS keeps the type -1 events too */
    int32_t device;        /* CUDA device ordinal */
    float pcm_scale;       /* divisor for NFC_IN_PCM_S16 and NFC_IN_SC16, 32767 = GNU Radio's 16-bit WAV normalisation */
} nfc_params;

/* One element of the list handed to transition_sink's callback (transition_sink.py:89-90,97):
 * ((v, d*factor), type).  dur_us = d * (1e6 / samp_rate). */
typedef struct {
    int64_t pos;  /* stream index of the sample that emitted it */
    int32_t d;
    int8_t v;
    int8_t type;
    int16_t pad;
} nfc_event;

/* One CombinedPacketProcessor.append_bit(val, type) call (packets.py:94). */
typedef struct {
    int64_t pos;
    int8_t type;
    int8_t val;
    int16_t pad;
    int32_t pad2;
} nfc_symbol;

/* One fsm.process_bits(bits, packet_type) hand-off (packets.py:97-98). */
typedef struct {
    int64_t pos;     /* stream index of the event that closed the frame */
    int64_t bit_off; /* into the buffer filled by nfc_stream_drain_frames */
    int32_t nbits;
    int32_t type;    /* PacketType: 0 TAG_TO_READER, 1 READER_TO_TAG (packets.py:19-20) */
} nfc_frame;

/* Filled with the defaults of the reference's constructors. */
void nfc_default_params(nfc_params *p);

/* transition_sink.__init__ + background.__init__ (transition_sink.py:12-34, background.py:17-25). */
int nfc_stream_create(const nfc_params *p, nfc_stream **out);
int nfc_stream_destroy(nfc_stream *s);
/* Back to the state right after creation (a fresh transition_sink / background pair); keeps device buffers. */
int nfc_stream_reset(nfc_stream *s);
/* New thresholds for the next capture (transition_sink's lo_val / hi_val constructor arguments, transition_sink.py:12):
 * allowed only on a stream that has consumed nothing since its creation or last reset.  Batches of captures that differ
 * only in hi_val reuse one stream (and its device buffers) this way. */
int nfc_stream_set_thresholds(nfc_stream *s, double lo_val, double hi_val);

/* transition_sink.work (transition_sink.py:37-125): offers n items, returns how many were consumed.
 * Like the reference, the call that completes the warm-up consumes only the warm-up part and
 * reports *called_back = 0; afterwards every call consumes everything and reports 1 (the reference
 * invokes its callback exactly once per work_stable call, even with an empty list).  The samples are
 * copied (or fully processed) before the call returns.  mem = NFC_MEM_HOST or NFC_MEM_DEVICE.  Device items are read on
 * the handle's own CUDA stream: the work that produces them must have completed when the call is made. */
int64_t nfc_stream_push(nfc_stream *s, const void *items, int64_t n, int mem, int *called_back);

/* A batch of independent captures in one pass: n_captures captures of items_per_capture items each (of the stream's input
 * kind: an NFC_IN_SC16 capture holds items_per_capture sc16 items, 4 B each), capture c starting at items + c * stride_items.  In the reference every capture is its own decoder (decoder.py:16-33): its own
 * transition_sink with its own warm-up and lo_val / hi_val (transition_sink.py:12-34,109-125; lo_vals / hi_vals: one value
 * per capture, NULL = the stream's), its own background thread, Miller / Manchester decoders and PacketProcessors
 * (background.py:17-25).  The stream must be new or reset; its outputs afterwards are those of all captures, positions
 * in one space: capture = pos / *pitch, item index inside the capture = pos % *pitch (*pitch: items_per_capture rounded
 * up to whole tiles).  Events and symbols at indices below av_window or from items_per_capture on belong to no capture
 * (they flush the decoders between captures) and are to be skipped by the consumer; frames never carry such positions.
 * NFC_OUT_DROPPED_EVENTS is not available in this mode.  Needs av_window in [1024, 52000], a multiple of 4, and 16-byte
 * aligned captures.  Returns n_captures; -1 on error; -3 when some capture has to take the sequential path (negative or widely
 * spread samples): decode the captures one by one with nfc_stream_push then.  The stream takes no further items until reset. */
int64_t nfc_stream_push_batch(nfc_stream *s, const void *items, int mem, int64_t n_captures, int64_t items_per_capture,
                              int64_t stride_items, const double *lo_vals, const double *hi_vals, int64_t *pitch);

/* background.append(transitions) (background.py:27-29): the list transition_sink hands to its callback, fed directly -- the
 * decoders, PacketProcessors and everything behind them run on the device as for pushed samples; decoder and framer state
 * carry on from whatever was pushed before.  ev[i].pos: positions the symbols and frames are reported at (ascending, less
 * than 2^32 apart from ev[0].pos); d in 1..max_len.  Returns n, or -1. */
int64_t nfc_stream_push_events(nfc_stream *s, const nfc_event *ev, int64_t n);

/* Results accumulated since the last drain, in stream order.  Each call copies up to cap records
 * and removes them from the stream.  Pass cap = 0 to query the number available. */
int64_t nfc_stream_drain_events(nfc_stream *s, nfc_event *out, int64_t cap);
int64_t nfc_stream_drain_symbols(nfc_stream *s, nfc_symbol *out, int64_t cap);
/* All pending frames at once: records to out (bit_off relative to bits) and one byte per bit; returns -2 when
 * cap or bits_cap is too small (query first with cap = 0 and nfc_stream_pending_frame_bits). */
int64_t nfc_stream_drain_frames(nfc_stream *s, nfc_frame *out, int64_t cap, uint8_t *bits, int64_t bits_cap);
int64_t nfc_stream_pending_frame_bits(nfc_stream *s); /* bytes the next full drain needs */
/* Zero-copy variant for bulk consumers: pointers into the stream's own buffers, valid until the next push / drain / reset /
 * release on this stream.  frames[i].bit_off indexes bits_tag (type 0) or bits_reader (type 1).  Returns the frame count;
 * nfc_stream_release_frames discards what was viewed (like a drain). */
int64_t nfc_stream_view_frames(nfc_stream *s, const nfc_frame **frames, const uint8_t **bits_tag, int64_t *n_bits_tag,
                               const uint8_t **bits_reader, int64_t *n_bits_reader);
int nfc_stream_release_frames(nfc_stream *s);
/* The frame offsets alone, eight bytes per frame, in page-locked host memory: what a time shard sends to the rank that
 * merges the shards (the order contract of CombinedPacketProcessor.append_bit, packets.py:94-98: frames reach
 * fsm.process_bits in closing order).  index[i] = pos << 24 | nbits << 8 | type of frame i of nfc_stream_view_frames
 * (pos < 2^40, nbits < 2^16); maintained beside the frame records while slabs are decoded, so viewing it costs nothing.
 * Valid until the next push / drain / reset / release on this stream.  Returns the frame count, -1 on error (a frame that
 * does not fit the packing). */
int64_t nfc_stream_view_frame_index(nfc_stream *s, const uint64_t **index);
/* Keep the packed frame index in memory of the caller's (room for cap records; NULL: the stream's own buffer again) -- e.g. a
 * shared-memory segment that the process merging the time shards of one node maps, so that "gathering" the frame offsets
 * moves no data at all.  The stream must hold no frames (right after create / reset / release).  More frames than cap make
 * the push that produces them fail.  The device writes the index there by DMA: the library page-locks the buffer
 * (cudaHostRegister) for as long as it is set -- set NULL (or destroy the stream) before freeing or unmapping it. */
int nfc_stream_set_frame_index_buffer(nfc_stream *s, uint64_t *buf, int64_t cap);

/* What fsm.process_bits does to a frame before any protocol logic, for a batch of frames on the device:
 * fsm._fix_ending (fsm.py:51-66), fsm._check_parity (fsm.py:28-49), fsm._print_enc (fsm.py:114-131) and
 * utilities.CRC.check_crc with CRC_14443_A (utilities.py:26-46).  Crypto1 traffic must be decrypted before its parity
 * and CRC mean anything (fsm.py:133-160, host side); for plain traffic the verdicts are final. */
typedef struct {
    int32_t nbits;     /* length after _fix_ending: a multiple of 9 */
    int32_t nbytes;    /* nbits / 9: what _print_enc prints, what _check_parity returns when it accepts */
    int64_t byte_off;  /* of the frame's bytes in `bytes` / `parity_flags` */
    int8_t fix_flag;   /* 0, 1 = _fix_ending printed "EXTRA ERROR", 2 = "MANY MORE ERROR" */
    int8_t parity_ok;  /* 1: _check_parity returns a non-empty list; 0: process_bits prints PARITY ERROR (fsm.py:226-228) */
    int8_t crc_ok;     /* CRC.check_crc(bytes) for nbytes >= 2, else 0 */
    int8_t pad[5];
} nfc_frame_tail;
/* frames[i].bit_off indexes bits_tag (type 0) or bits_reader (type 1), as nfc_stream_view_frames returns them (pass the one
 * buffer of nfc_stream_drain_frames twice); all pointers are host memory.  bytes[k] / parity_flags[k]: the k-th byte of the
 * batch, LSB first, and 1 where _print_enc appends '!' (parity violated).  Returns the number of bytes written, < 0 on
 * error (bytes_cap too small: sum of (nbits + 1) / 9 always suffices). */
int64_t nfc_frames_tail(int device, const nfc_frame *frames, int64_t n_frames, const uint8_t *bits_tag, int64_t n_bits_tag,
                        const uint8_t *bits_reader, int64_t n_bits_reader, nfc_frame_tail *tails, uint8_t *bytes,
                        uint8_t *parity_flags, int64_t bytes_cap);

/* Implicit streaming state of the reference objects (transition_sink.py:20-34,102-106; decoder and
 * PacketProcessor attributes), for checkpointing and for stitching time-sharded captures. */
typedef struct {
    int64_t pos;           /* items consumed so far */
    double ss;             /* _sum */
    int32_t cur_state, last_bit, dur; /* _current_state, _last_bit, _dur */
    int32_t index;         /* _index */
    int32_t stable;        /* work is work_stable */
    int32_t miller_state, manch_state;
    int32_t started[2];    /* PacketProcessor._started per type */
    int32_t pending[2];    /* len(PacketProcessor._cur) per type */
    int32_t serial_mode;   /* 1 once the stream left the exactly-summable regime */
    int64_t lastL, lrun_start; /* position of the last LOW sample / start of its run (hysteresis carry);
                                * set lastL = INT64_MIN in set_state to have both derived from cur_state/last_bit/dur */
} nfc_state;
/* ring: av_window floats (the _ar list), may be NULL.  pending_bits: pending[0]+pending[1] bytes, may be NULL. */
int nfc_stream_get_state(nfc_stream *s, nfc_state *st, float *ring, uint8_t *pending_bits);
int nfc_stream_set_state(nfc_stream *s, const nfc_state *st, const float *ring, const uint8_t *pending_bits);

/* Execution knobs (not part of the reference's interface).  seg_len / halo in samples (rounded up to
 * tiles; 0 = automatic), slab_len = samples processed per kernel wave, force_serial = use the strictly
 * sequential kernel for everything (the on-device cross-check). */
int nfc_stream_set_tuning(nfc_stream *s, int64_t seg_len, int64_t halo, int64_t slab_len, int force_serial);
/* blocking != 0: host threads that wait for this stream's results sleep in the driver (blocking-sync events) instead of
 * spinning.  For many streams driven by many host threads -- one per independent capture, each its own transition_sink
 * (code/transition_sink.py:12-34) -- where spinning waiters would outnumber the cores; the default (0) has the lower latency. */
int nfc_stream_set_wait_mode(nfc_stream *s, int blocking);

/* Counters since creation: kernel time measured with CUDA events on the stream's CUDA stream. */
typedef struct {
    double kernel_ms;        /* device time spent in this library's kernels */
    double slicer_ms;        /* of which the slicer kernel */
    int64_t launches;        /* kernels launched */
    int64_t slicer_launches;
    int64_t samples;         /* items decoded on the device */
    int64_t segments, seam_mismatches, serial_segments, overflow_retries;
    int64_t linecode_scan_fallbacks; /* slabs where the frame-boundary search gave up and the scan path ran */
    int64_t h2d_bytes, d2h_bytes;
    /* slicer tiles by the way they were settled (device-wide counters: all streams of the process) */
    int64_t fast_tiles;       /* proven by the streaming path (including repeated and fix-point tiles) */
    int64_t exact_tiles;      /* handed to the exact path (segment edges, hysteresis-relevant HIGH samples, ...) */
    int64_t repeated_passes;  /* extra streaming passes: measured guesses, or a coarser fixed-point step */
    int64_t fixpoint_tiles;   /* tiles settled by the exact fix-point pass after the precise pass could not prove itself */
    int64_t st2_tiles;        /* tiles sent to the exact path because the hysteresis could matter */
    int64_t unproven_tiles;   /* tiles sent to the exact path because the streaming passes gave up */
    int64_t ring_resums;      /* exact recomputations of the window sum from the ring */
    int64_t exact_rounds;     /* fix-point rounds of the exact path (first-generation kernel) */
    double slicer_kernel_ms;  /* CUDA-event time of the streaming slicer kernel's launches alone */
    int64_t slicer_kernel_launches;
    /* the pipelined mode of the streaming kernel (device-wide counters, like the tile counters above) */
    int64_t pipe_tiles;       /* tiles proven while the workers ran ahead of the verdicts (subset of fast_tiles) */
    int64_t pipe_runs;        /* runs of consecutive tiles entered in that mode */
    int64_t pipe_aborts;      /* runs ended by a tile the pipelined mode could not prove (settled by the synchronous loop) */
    int64_t empty_frames;     /* frames closed without a bit: the reference does not forward them (packets.py:97), nor are they handed out */
} nfc_stats;
int nfc_stream_get_stats(nfc_stream *s, nfc_stats *st);
int nfc_stream_reset_stats(nfc_stream *s);
/* The CUDA stream (cudaStream_t) the handle launches on, for callers that time with their own events. */
void *nfc_stream_cuda_stream(nfc_stream *s);

/* The line-code tables the device uses (built on the host from the decoder rules, csrc/tables.cpp), for
 * inspection and host-side tests; needs no GPU.  dclass[d] for d = 0..max_len, then
 * table[dclass][v+1][state] entries (bits 0-3 next state, 4-5 number of outputs, 6-8 out0, 9-11 out1).
 * which: 0 Manchester (8 states), 1 Miller (16 states).  Returns the number of table entries. */
int nfc_build_tables(double samp_rate, int32_t max_len, int which, uint8_t *dclass, int32_t dclass_cap,
                     uint16_t *table, int32_t table_cap, int32_t *n_dclass);

/* Device-side synthetic traffic (binary_src.work, binary_src.py:64-103, rendered from a pulse schedule):
 * level codes 0 carrier / 1 reader pause / 2 tag high with run lengths in samples; the schedule repeats.
 * dev_out[k] is sample first_index + k of the endless capture (time shards render their own part). */
int nfc_synth_render(void *dev_out_f32, int64_t n, int64_t first_index, const int8_t *codes, const int64_t *lens,
                     int64_t n_runs, float carrier, float pause, float tag_high, float noise, float fade,
                     double fade_period, uint64_t seed, int as_envelope, int device);

const char *nfc_last_error(void);
int nfc_abi_version(void);
/* sizeof of the structs above as this library was compiled, for bindings to check their own layouts against:
 * which = 0 nfc_params, 1 nfc_event, 2 nfc_symbol, 3 nfc_frame, 4 nfc_frame_tail, 5 nfc_state, 6 nfc_stats; -1 otherwise */
int nfc_abi_sizeof(int which);
int nfc_device_count(void);

#ifdef __cplusplus
}
#endif
#endif
