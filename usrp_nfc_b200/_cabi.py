"""ctypes binding of the C ABI in include/usrp_nfc_b200.h.

The shared library holds the sm_100a kernels; there is no other implementation.  If it has not
been built (`python -c "import __graft_entry__ as g; g.build()"` or `make -C usrp_nfc_b200/csrc`)
importing this module fails loudly instead of falling back to anything.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# USRP_NFC_B200_LIB: another build of the same library (A/B measurements of kernel variants)
LIB_PATH = os.environ.get("USRP_NFC_B200_LIB") or os.path.join(_HERE, "libusrp_nfc_b200.so")

IN_ENVELOPE_F32, IN_REAL_F32, IN_IQ_F32, IN_PCM_S16, IN_SC16 = 0, 1, 2, 3, 4
MEM_HOST, MEM_DEVICE = 0, 1
OUT_EVENTS, OUT_SYMBOLS, OUT_FRAMES, OUT_DROPPED_EVENTS = 1, 2, 4, 8
OUT_ALL = OUT_EVENTS | OUT_SYMBOLS | OUT_FRAMES | OUT_DROPPED_EVENTS

EVENT_DTYPE = np.dtype([("pos", "<i8"), ("d", "<i4"), ("v", "i1"), ("type", "i1"), ("pad", "<i2")])
SYMBOL_DTYPE = np.dtype([("pos", "<i8"), ("type", "i1"), ("val", "i1"), ("pad", "<i2"), ("pad2", "<i4")])
FRAME_DTYPE = np.dtype([("pos", "<i8"), ("bit_off", "<i8"), ("nbits", "<i4"), ("type", "<i4")])
FRAME_TAIL_DTYPE = np.dtype([("nbits", "<i4"), ("nbytes", "<i4"), ("byte_off", "<i8"), ("fix_flag", "i1"), ("parity_ok", "i1"),
                             ("crc_ok", "i1"), ("pad", "i1", (5,))])


class Params(C.Structure):
    _fields_ = [("samp_rate", C.c_double), ("lo_val", C.c_double), ("hi_val", C.c_double),
                ("av_window", C.c_int32), ("max_len", C.c_int32), ("decode_reader", C.c_int32),
                ("decode_tag", C.c_int32), ("input_kind", C.c_int32), ("outputs", C.c_int32),
                ("device", C.c_int32), ("pcm_scale", C.c_float)]


class State(C.Structure):
    _fields_ = [("pos", C.c_int64), ("ss", C.c_double), ("cur_state", C.c_int32), ("last_bit", C.c_int32),
                ("dur", C.c_int32), ("index", C.c_int32), ("stable", C.c_int32), ("miller_state", C.c_int32),
                ("manch_state", C.c_int32), ("started", C.c_int32 * 2), ("pending", C.c_int32 * 2),
                ("serial_mode", C.c_int32), ("lastL", C.c_int64), ("lrun_start", C.c_int64)]


class Stats(C.Structure):
    _fields_ = [("kernel_ms", C.c_double), ("slicer_ms", C.c_double), ("launches", C.c_int64),
                ("slicer_launches", C.c_int64), ("samples", C.c_int64), ("segments", C.c_int64),
                ("seam_mismatches", C.c_int64), ("serial_segments", C.c_int64), ("overflow_retries", C.c_int64),
                ("linecode_scan_fallbacks", C.c_int64),
                ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("fast_tiles", C.c_int64),
                ("exact_tiles", C.c_int64), ("repeated_passes", C.c_int64), ("fixpoint_tiles", C.c_int64),
                ("st2_tiles", C.c_int64), ("unproven_tiles", C.c_int64), ("ring_resums", C.c_int64),
                ("exact_rounds", C.c_int64), ("slicer_kernel_ms", C.c_double), ("slicer_kernel_launches", C.c_int64),
                ("pipe_tiles", C.c_int64), ("pipe_runs", C.c_int64), ("pipe_aborts", C.c_int64),
                ("empty_frames", C.c_int64)]


# every symbol include/usrp_nfc_b200.h declares: (restype, argtypes)
SIGNATURES = {
    "nfc_default_params": (None, [C.POINTER(Params)]),
    "nfc_stream_create": (C.c_int, [C.POINTER(Params), C.POINTER(C.c_void_p)]),
    "nfc_stream_destroy": (C.c_int, [C.c_void_p]),
    "nfc_stream_reset": (C.c_int, [C.c_void_p]),
    "nfc_stream_set_thresholds": (C.c_int, [C.c_void_p, C.c_double, C.c_double]),
    "nfc_stream_push": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.POINTER(C.c_int)]),
    "nfc_stream_push_batch": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                          C.POINTER(C.c_int64)]),
    "nfc_stream_push_events": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int64]),
    "nfc_stream_drain_events": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int64]),
    "nfc_stream_drain_symbols": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int64]),
    "nfc_stream_drain_frames": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]),
    "nfc_stream_pending_frame_bits": (C.c_int64, [C.c_void_p]),
    "nfc_stream_view_frames": (C.c_int64, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_int64),
                                           C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "nfc_stream_release_frames": (C.c_int, [C.c_void_p]),
    "nfc_stream_view_frame_index": (C.c_int64, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "nfc_stream_set_frame_index_buffer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "nfc_stream_get_state": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_void_p, C.c_void_p]),
    "nfc_stream_set_state": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_void_p, C.c_void_p]),
    "nfc_stream_set_tuning": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int]),
    "nfc_stream_set_wait_mode": (C.c_int, [C.c_void_p, C.c_int]),
    "nfc_stream_get_stats": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "nfc_stream_reset_stats": (C.c_int, [C.c_void_p]),
    "nfc_stream_cuda_stream": (C.c_void_p, [C.c_void_p]),
    "nfc_build_tables": (C.c_int, [C.c_double, C.c_int32, C.c_int, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32,
                                   C.POINTER(C.c_int32)]),
    "nfc_synth_render": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_float,
                                   C.c_float, C.c_float, C.c_float, C.c_double, C.c_uint64, C.c_int, C.c_int]),
    "nfc_frames_tail": (C.c_int64, [C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_int64]),
    "nfc_last_error": (C.c_char_p, []),
    "nfc_abi_version": (C.c_int, []),
    "nfc_abi_sizeof": (C.c_int, [C.c_int]),
    "nfc_device_count": (C.c_int, []),
}

_lib = None


class NfcError(RuntimeError):
    pass


class BatchNeedsSequential(NfcError):
    """nfc_stream_push_batch returned -3: some capture has to take the sequential path; decode the captures one by one."""


def lib():
    """The loaded shared library.  Raises if it was not built: there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "usrp_nfc_b200: %s is missing. Build the CUDA library first (make -C usrp_nfc_b200/csrc, or "
                "__graft_entry__.build()); there is no CPU implementation to fall back to." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def last_error():
    return (lib().nfc_last_error() or b"").decode()


def _torch_dtype_name(input_kind):
    return {IN_ENVELOPE_F32: "float32", IN_REAL_F32: "float32", IN_IQ_F32: "complex64", IN_PCM_S16: "int16",
            IN_SC16: "int16"}[input_kind]


def _is_tensor(items):
    return hasattr(items, "data_ptr") and hasattr(items, "is_cuda")


def _check_sc16(items, ndim):
    """IN_SC16 items are int16 (I, Q) pairs: an int16 array or tensor of `ndim` dimensions whose last one is 2 (push: [n, 2],
    push_batch: [captures, items, 2]).  A file written by rx_samples_to_file is np.fromfile(path, np.int16).reshape(-1, 2).
    Returns the items (a numpy array as an ndarray); raises TypeError / ValueError for anything else."""
    if _is_tensor(items):
        dt = str(items.dtype).replace("torch.", "")
    else:
        if not isinstance(items, np.ndarray):
            raise TypeError("sc16 items are an int16 numpy array or tensor of shape [..., 2], got %s" % type(items).__name__)
        dt = str(items.dtype)
    if dt != "int16":
        raise TypeError("sc16 items are int16 (I, Q) pairs, got %s" % dt)
    shape = tuple(items.shape)
    if len(shape) != ndim or shape[-1] != 2:
        want = "[n, 2]" if ndim == 2 else "[captures, items, 2]"
        raise ValueError("sc16 items have shape %s (I, Q last), got %s" % (want, list(shape)))
    return items


def _ptr_and_mem(items, input_kind=None):
    """(address, item count, mem kind, keepalive) of a numpy array or a torch tensor.  A tensor must already hold items of the
    stream's input kind (one element = one item): the kernels read t.numel() items of that size behind the pointer.  IN_SC16:
    one item is a row of two int16 elements, so the count is the number of rows."""
    per_item = 2 if input_kind == IN_SC16 else 1
    if hasattr(items, "data_ptr") and hasattr(items, "is_cuda"):  # torch tensor
        if input_kind is not None:
            want = _torch_dtype_name(input_kind)
            if str(items.dtype).replace("torch.", "") != want:
                raise TypeError("stream input kind %d takes %s items, got a tensor of %s" % (input_kind, want, items.dtype))
        t = items.contiguous()
        if t.is_cuda:
            # the library reads device items on its own CUDA stream: whatever produced them on torch's stream must be done
            import torch
            torch.cuda.current_stream(t.device).synchronize()
        return t.data_ptr(), t.numel() // per_item, (MEM_DEVICE if t.is_cuda else MEM_HOST), t
    a = np.ascontiguousarray(items)
    return a.ctypes.data, a.size // per_item, MEM_HOST, a


_KIND_DTYPES = {IN_ENVELOPE_F32: np.float32, IN_REAL_F32: np.float32, IN_IQ_F32: np.complex64, IN_PCM_S16: np.int16,
                IN_SC16: np.int16}


class Stream(object):
    """One sample stream on one GPU (RAII over nfc_stream)."""

    def __init__(self, samp_rate, lo_val=0.1, hi_val=1.1, av_window=2000, max_len=50, reader=True, tag=True,
                 input_kind=IN_ENVELOPE_F32, outputs=OUT_ALL, device=0, pcm_scale=32767.0):
        L = lib()
        p = Params()
        L.nfc_default_params(C.byref(p))
        p.samp_rate, p.lo_val, p.hi_val = float(samp_rate), float(lo_val), float(hi_val)
        p.av_window, p.max_len = int(av_window), int(max_len)
        p.decode_reader, p.decode_tag = int(bool(reader)), int(bool(tag))
        p.input_kind, p.outputs, p.device, p.pcm_scale = int(input_kind), int(outputs), int(device), float(pcm_scale)
        self.params = p
        self.factor = 1e6 / float(samp_rate)  # transition_sink.py:21
        self.input_kind = int(input_kind)
        self._h = C.c_void_p()
        if L.nfc_stream_create(C.byref(p), C.byref(self._h)) != 0:
            self._h = None
            raise NfcError("nfc_stream_create: " + last_error())

    def close(self):
        if getattr(self, "_h", None) and lib is not None:
            lib().nfc_stream_destroy(self._h)
            self._h = None

    __del__ = close

    def set_thresholds(self, lo_val, hi_val):
        """lo_val / hi_val for the next capture; only on a freshly created or reset stream."""
        if lib().nfc_stream_set_thresholds(self._h, float(lo_val), float(hi_val)) != 0:
            raise NfcError(last_error())
        self.params.lo_val, self.params.hi_val = float(lo_val), float(hi_val)

    def push(self, items):
        """-> (consumed, called_back): transition_sink.work semantics (transition_sink.py:37-125).  IN_SC16: items is [n, 2]."""
        if self.input_kind == IN_SC16:
            _check_sc16(items, 2)
        elif not _is_tensor(items):
            items = np.ascontiguousarray(items, dtype=_KIND_DTYPES[self.input_kind])
        addr, n, mem, keep = _ptr_and_mem(items, self.input_kind)
        cb = C.c_int(0)
        used = lib().nfc_stream_push(self._h, addr, n, mem, C.byref(cb))
        del keep
        if used < 0:
            raise NfcError("nfc_stream_push: " + last_error())
        return int(used), bool(cb.value)

    def push_batch(self, items, lo_vals=None, hi_vals=None):
        """A batch of independent captures in one pass: items is a 2-D array / tensor [captures, items per capture] of the
        stream's input kind (every row its own transition_sink + decoders in the reference, decoder.py:16-33); lo_vals /
        hi_vals: per-capture thresholds.  Returns the pitch of the position space the results use (capture = pos // pitch,
        index inside the capture = pos % pitch).  Raises BatchNeedsSequential when a capture must take the sequential path.
        IN_SC16: items is 3-D, [captures, items per capture, 2] int16."""
        if self.input_kind == IN_SC16:
            _check_sc16(items, 3)
            if _is_tensor(items):
                keep = items if (items.stride(2) == 1 and items.stride(1) == 2 and items.stride(0) % 2 == 0) else items.contiguous()
                if keep.is_cuda:
                    import torch
                    torch.cuda.current_stream(keep.device).synchronize()  # the library reads the items on its own CUDA stream
                ncap, n, stride = int(keep.shape[0]), int(keep.shape[1]), int(keep.stride(0)) // 2
                addr, mem = keep.data_ptr(), (MEM_DEVICE if keep.is_cuda else MEM_HOST)
            else:
                keep = np.ascontiguousarray(items)
                ncap, n, stride = int(keep.shape[0]), int(keep.shape[1]), int(keep.shape[1])
                addr, mem = keep.ctypes.data, MEM_HOST
        elif _is_tensor(items):
            if items.dim() != 2:
                raise ValueError("push_batch takes a 2-D tensor")
            want = _torch_dtype_name(self.input_kind)
            if str(items.dtype).replace("torch.", "") != want:
                raise TypeError("stream input kind %d takes %s items, got a tensor of %s" % (self.input_kind, want, items.dtype))
            keep = items if items.stride(1) == 1 else items.contiguous()
            if keep.is_cuda:
                import torch
                torch.cuda.current_stream(keep.device).synchronize()  # the library reads the items on its own CUDA stream
            ncap, n, stride = int(keep.shape[0]), int(keep.shape[1]), int(keep.stride(0))
            addr, mem = keep.data_ptr(), (MEM_DEVICE if keep.is_cuda else MEM_HOST)
        else:
            keep = np.ascontiguousarray(items, dtype=_KIND_DTYPES[self.input_kind])
            if keep.ndim != 2:
                raise ValueError("push_batch takes a 2-D array")
            ncap, n, stride = int(keep.shape[0]), int(keep.shape[1]), int(keep.shape[1])
            addr, mem = keep.ctypes.data, MEM_HOST
        lo = None if lo_vals is None else np.ascontiguousarray(lo_vals, dtype=np.float64)
        hi = None if hi_vals is None else np.ascontiguousarray(hi_vals, dtype=np.float64)
        for v in (lo, hi):
            if v is not None and v.size != ncap:
                raise ValueError("one threshold per capture")
        pitch = C.c_int64(0)
        rc = lib().nfc_stream_push_batch(self._h, addr, mem, ncap, n, stride, None if lo is None else lo.ctypes.data,
                                         None if hi is None else hi.ctypes.data, C.byref(pitch))
        del keep
        if rc == -3:
            raise BatchNeedsSequential(last_error())
        if rc < 0:
            raise NfcError("nfc_stream_push_batch: " + last_error())
        return int(pitch.value)

    def push_events(self, events):
        """background.append (background.py:27-29): transition_sink's events (EVENT_DTYPE array: pos, d, v, type) straight
        into the decoders on the device."""
        ev = np.ascontiguousarray(events, dtype=EVENT_DTYPE)
        n = lib().nfc_stream_push_events(self._h, ev.ctypes.data, len(ev))
        if n < 0:
            raise NfcError("nfc_stream_push_events: " + last_error())
        return int(n)

    def push_all(self, items, chunk=None):
        """Feed everything, re-offering what a call did not consume (the GNU Radio scheduler's job)."""
        if self.input_kind == IN_SC16:
            n = len(_check_sc16(items, 2))  # rows of (I, Q)
        else:
            n = items.numel() if hasattr(items, "numel") else len(items)
        off = 0
        step = chunk or n
        while off < n:
            used, _ = self.push(items[off: off + step])
            off += used
            if used == 0:
                break
        return off

    def _drain(self, fn, dtype):
        n = fn(self._h, None, 0)
        if n < 0:
            raise NfcError(last_error())
        out = np.zeros(n, dtype=dtype)
        if n:
            got = fn(self._h, out.ctypes.data, n)
            if got < 0:
                raise NfcError(last_error())
            out = out[:got]
        return out

    def drain_events(self):
        return self._drain(lib().nfc_stream_drain_events, EVENT_DTYPE)

    def drain_symbols(self):
        return self._drain(lib().nfc_stream_drain_symbols, SYMBOL_DTYPE)

    def drain_frames(self):
        """-> (frame records, [uint8 bit array per frame]); what fsm.process_bits receives (packets.py:97-98)."""
        L = lib()
        n = L.nfc_stream_drain_frames(self._h, None, 0, None, 0)
        nb = L.nfc_stream_pending_frame_bits(self._h)
        if n < 0 or nb < 0:
            raise NfcError(last_error())
        fr = np.zeros(n, dtype=FRAME_DTYPE)
        bits = np.zeros(max(nb, 1), dtype=np.uint8)
        if n:
            got = L.nfc_stream_drain_frames(self._h, fr.ctypes.data, n, bits.ctypes.data, nb)
            if got < 0:
                raise NfcError(last_error())
            fr = fr[:got]
        return fr, [bits[f["bit_off"]: f["bit_off"] + f["nbits"]].copy() for f in fr]

    def drain_frames_flat(self, reuse=False):
        """-> (frame records, one uint8 array with all frame bits; record.bit_off indexes into it).
        reuse=True returns views of buffers owned by this object, valid until the next drain (no allocation per call)."""
        L = lib()
        n = L.nfc_stream_drain_frames(self._h, None, 0, None, 0)
        nb = L.nfc_stream_pending_frame_bits(self._h)
        if n < 0 or nb < 0:
            raise NfcError(last_error())
        if reuse:
            if getattr(self, "_fr_buf", None) is None or self._fr_buf.size < n:
                self._fr_buf = np.zeros(int(n * 1.25) + 16, dtype=FRAME_DTYPE)
            if getattr(self, "_bit_buf", None) is None or self._bit_buf.size < max(nb, 1):
                self._bit_buf = np.zeros(int(nb * 1.25) + 16, dtype=np.uint8)
            fr, bits = self._fr_buf[:n], self._bit_buf[:max(nb, 1)]
        else:
            fr = np.zeros(n, dtype=FRAME_DTYPE)
            bits = np.zeros(max(nb, 1), dtype=np.uint8)
        if n:
            got = L.nfc_stream_drain_frames(self._h, fr.ctypes.data, n, bits.ctypes.data, nb)
            if got < 0:
                raise NfcError(last_error())
            fr = fr[:got]
        return fr, bits[:nb]

    def view_frames(self):
        """Zero-copy bulk access: (frame records, tag->reader bits, reader->tag bits) as numpy views of the stream's own
        buffers; record.bit_off indexes the bit array of the record's type.  Valid until the next push / drain / reset /
        release_frames on this stream."""
        fp, b0, b1 = C.c_void_p(), C.c_void_p(), C.c_void_p()
        n0, n1 = C.c_int64(0), C.c_int64(0)
        n = lib().nfc_stream_view_frames(self._h, C.byref(fp), C.byref(b0), C.byref(n0), C.byref(b1), C.byref(n1))
        if n < 0:
            raise NfcError(last_error())

        def arr(ptr, count, dtype):
            if not count or not ptr.value:
                return np.zeros(0, dtype=dtype)
            buf = (C.c_char * (count * np.dtype(dtype).itemsize)).from_address(ptr.value)
            return np.frombuffer(buf, dtype=dtype, count=count)

        return arr(fp, n, FRAME_DTYPE), arr(b0, n0.value, np.uint8), arr(b1, n1.value, np.uint8)

    def view_frame_index(self):
        """The frame offsets alone (nfc_stream_view_frame_index): a uint64 numpy view of page-locked memory owned by the
        stream, one record per frame of view_frames: pos << 24 | nbits << 8 | type.  Valid like view_frames."""
        p = C.c_void_p()
        n = lib().nfc_stream_view_frame_index(self._h, C.byref(p))
        if n < 0:
            raise NfcError(last_error())
        if not n or not p.value:
            return np.zeros(0, dtype=np.uint64)
        buf = (C.c_char * (n * 8)).from_address(p.value)
        return np.frombuffer(buf, dtype=np.uint64, count=n)

    def set_frame_index_buffer(self, address, cap):
        """Keep the packed frame index in the caller's memory (address of room for cap uint64 records; None: the stream's
        own buffer again): nfc_stream_set_frame_index_buffer."""
        if lib().nfc_stream_set_frame_index_buffer(self._h, C.c_void_p(address) if address else None, int(cap)) != 0:
            raise NfcError(last_error())

    def release_frames(self):
        if lib().nfc_stream_release_frames(self._h) != 0:
            raise NfcError(last_error())

    def state(self):
        st = State()
        ring = np.zeros(self.params.av_window, dtype=np.float32)
        if lib().nfc_stream_get_state(self._h, C.byref(st), ring.ctypes.data, None) != 0:
            raise NfcError(last_error())
        npend = st.pending[0] + st.pending[1]
        pend = np.zeros(max(npend, 1), dtype=np.uint8)
        if lib().nfc_stream_get_state(self._h, C.byref(st), None, pend.ctypes.data) != 0:
            raise NfcError(last_error())
        return st, ring, pend[:npend]

    def set_state(self, st, ring, pending_bits=None):
        ring = np.ascontiguousarray(ring, dtype=np.float32)
        pb = None if pending_bits is None else np.ascontiguousarray(pending_bits, dtype=np.uint8)
        if lib().nfc_stream_set_state(self._h, C.byref(st), ring.ctypes.data, None if pb is None else pb.ctypes.data) != 0:
            raise NfcError(last_error())

    def reset(self):
        if lib().nfc_stream_reset(self._h) != 0:
            raise NfcError("nfc_stream_reset: " + last_error())

    def set_tuning(self, seg_len=0, halo=0, slab_len=0, force_serial=False):
        if lib().nfc_stream_set_tuning(self._h, int(seg_len), int(halo), int(slab_len), int(bool(force_serial))) != 0:
            raise NfcError("nfc_stream_set_tuning: " + last_error())

    def set_wait_mode(self, blocking=True):
        """Waiting host threads sleep instead of spinning (many streams on many threads: usrp_nfc_b200/batch.py)."""
        if lib().nfc_stream_set_wait_mode(self._h, int(bool(blocking))) != 0:
            raise NfcError(last_error())

    def stats(self):
        st = Stats()
        if lib().nfc_stream_get_stats(self._h, C.byref(st)) != 0:
            raise NfcError("nfc_stream_get_stats: " + last_error())
        return {k: getattr(st, k) for k, _ in Stats._fields_}

    def reset_stats(self):
        if lib().nfc_stream_reset_stats(self._h) != 0:
            raise NfcError("nfc_stream_reset_stats: " + last_error())

    def cuda_stream(self):
        return lib().nfc_stream_cuda_stream(self._h)


def frames_tail(frames, bits_tag, bits_reader=None, device=0):
    """fsm._fix_ending / _check_parity / _print_enc / CRC_A for a batch of frames on the device (csrc/frametail.cu).

    frames: FRAME_DTYPE records whose bit_off index bits_tag (type 0) / bits_reader (type 1); with bits_reader None both
    types index bits_tag (the single buffer of drain_frames_flat).  Returns (tails, bytes, parity_flags).
    """
    frames = np.ascontiguousarray(frames, dtype=FRAME_DTYPE)
    b0 = np.ascontiguousarray(bits_tag, dtype=np.uint8)
    b1 = b0 if bits_reader is None else np.ascontiguousarray(bits_reader, dtype=np.uint8)
    n = int(frames.size)
    tails = np.zeros(n, dtype=FRAME_TAIL_DTYPE)
    cap = int(((frames["nbits"].astype(np.int64) + 1) // 9).sum()) if n else 0
    by = np.zeros(max(cap, 1), dtype=np.uint8)
    fl = np.zeros(max(cap, 1), dtype=np.uint8)
    got = lib().nfc_frames_tail(int(device), frames.ctypes.data, n, b0.ctypes.data, b0.size, b1.ctypes.data, b1.size,
                                tails.ctypes.data, by.ctypes.data, fl.ctypes.data, cap)
    if got < 0:
        raise NfcError("nfc_frames_tail: " + last_error())
    return tails, by[:got], fl[:got]


def build_tables(samp_rate, max_len, which):
    """(dclass[d], table[dclass][v+1][state]) of the Manchester (which=0) or Miller (which=1) automaton."""
    nstates = 16 if which else 8
    ncls = C.c_int32(0)
    n = lib().nfc_build_tables(samp_rate, max_len, which, None, 0, None, 0, C.byref(ncls))
    if n < 0:
        raise NfcError(last_error())
    dcl = np.zeros(max_len + 1, dtype=np.uint8)
    tab = np.zeros(n, dtype=np.uint16)
    lib().nfc_build_tables(samp_rate, max_len, which, dcl.ctypes.data, dcl.size, tab.ctypes.data, tab.size, C.byref(ncls))
    return dcl, tab.reshape(ncls.value, 4, nstates)


def synth_render(dev_tensor, codes, lens, carrier=0.5, pause=0.02, tag_high=1.08, noise=0.003, fade=0.0,
                 fade_period=40000.0, seed=1, as_envelope=True, device=0, first_index=0):
    """Fill a float32 CUDA tensor with rendered traffic (csrc/synth.cu)."""
    codes = np.ascontiguousarray(codes, dtype=np.int8)
    lens = np.ascontiguousarray(lens, dtype=np.int64)
    rc = lib().nfc_synth_render(dev_tensor.data_ptr(), dev_tensor.numel(), int(first_index), codes.ctypes.data, lens.ctypes.data,
                                codes.size, carrier, pause, tag_high, noise, fade, float(fade_period), int(seed),
                                int(bool(as_envelope)), int(device))
    if rc != 0:
        raise NfcError("nfc_synth_render: " + last_error())
