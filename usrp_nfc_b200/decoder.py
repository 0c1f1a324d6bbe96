"""Drop-in replacement of the reference's decoder hier block (decoder.py:15-33) with the whole
sample-rate path fused on the GPU: envelope, slicer, Manchester/Miller decoding and framing.

decoder(src, dst, repeat, reader, tag, samp_rate, emulator) keeps the reference's signature.  Closed,
non-empty frames are handed to fsm.process_bits(bits, packet_type) in stream order, which is what
CombinedPacketProcessor.append_bit does (packets.py:94-98); with an emulator the fsm callback is
emulator.process_packet and emulator.set_encoder(fsm.process_outgoing) is called (packets.py:88-90).
The protocol FSM, Crypto1 and the emulators are the reference's own host code and stay unchanged: the
`fsm` module is imported from the reference checkout when it is on sys.path, or injected with `fsm=`.
"""
import wave

import numpy

from . import _cabi
from .grcompat import HAVE_GNURADIO, blocks, gr


class frame_sink(gr.sync_block):
    """The GPU end of the flowgraph: consumes items, forwards frames.  in_sig is float32 for the WAV
    path (raw samples, squared on the device), complex64 for UHD, int16 for 16-bit PCM and (int16, 2) for complex int16
    (UHD's sc16: one item is an I, Q pair; work() takes [n, 2] views)."""

    def __init__(self, samp_rate, on_frame, reader=True, tag=True, hi_val=1.1, lo_val=0.1, av_window=2000, max_len=50,
                 input_kind=_cabi.IN_REAL_F32, device=0, on_frame_bytes=None, coalesce=0):
        """coalesce: GNU Radio hands a sync block a few thousand items per work() call; a call costs about a millisecond of
        launches whatever its size.  With coalesce > 0 the items of successive calls are collected (every call still consumes
        all it is offered) and go to the device once at least that many are there: the same frames in the same order, at
        most `coalesce` items later.  0: every call is pushed as it comes."""
        in_type = {_cabi.IN_IQ_F32: numpy.complex64, _cabi.IN_PCM_S16: numpy.int16,
                   _cabi.IN_SC16: (numpy.int16, 2)}.get(input_kind, numpy.float32)
        gr.sync_block.__init__(self, name="nfc_frame_sink", in_sig=[in_type], out_sig=None)
        self._on_frame = on_frame
        self._on_frame_bytes = on_frame_bytes
        self._device = device
        self._coalesce = int(coalesce)
        self._held, self._held_n = [], 0
        self._stream = _cabi.Stream(samp_rate, lo_val, hi_val, av_window, max_len, reader=reader, tag=tag,
                                    input_kind=input_kind, outputs=_cabi.OUT_FRAMES, device=device)

    def work(self, input_items, output_items):
        items = input_items[0]
        if self._coalesce > 0:
            self._held.append(numpy.array(items, copy=True))  # the view is only valid during the call
            self._held_n += len(items)
            if self._held_n >= self._coalesce:
                self.flush()
            return len(items)
        consumed, _ = self._stream.push(items)
        self._forward()
        return consumed

    def flush(self):
        """Push what coalescing holds back (end of the source)."""
        if self._held_n:
            block = self._held[0] if len(self._held) == 1 else numpy.concatenate(self._held)
            self._held, self._held_n = [], 0
            self._stream.push_all(block)
            self._forward()

    def _forward(self):
        records, flat = self._stream.drain_frames_flat()
        if self._on_frame is not None:
            for rec in records:
                o = int(rec["bit_off"])
                self._on_frame(flat[o: o + int(rec["nbits"])].tolist(), int(rec["type"]))
        if self._on_frame_bytes is not None and len(records):
            # what fsm.process_bits computes first for every frame (_fix_ending, _check_parity / _print_enc, CRC_A), as
            # one device pass over the batch: on_frame_bytes(bytes, parity_flags, tail_record, packet_type)
            tails, by, fl = _cabi.frames_tail(records, flat, device=self._device)
            for rec, tl in zip(records, tails):
                o, n = int(tl["byte_off"]), int(tl["nbytes"])
                self._on_frame_bytes(by[o: o + n].tolist(), fl[o: o + n].tolist(), tl, int(rec["type"]))

    def stream(self):
        return self._stream


def read_wav(path, iq=False):
    """The samples of a 16-bit PCM WAV file as int16: channel 0 ([n]), or with iq=True a 2-channel file's (I, Q) pairs
    ([n, 2], channel 0 = I, channel 1 = Q: GNU Radio's two-channel wavfile_sink and most SDR recorders write baseband so)."""
    w = wave.open(path, "rb")
    try:
        if w.getsampwidth() != 2:
            raise ValueError("only 16-bit PCM WAV files are supported without GNU Radio")
        nch = w.getnchannels()
        if iq and nch != 2:
            raise ValueError("an IQ WAV file has two channels (I, Q), %s has %d" % (path, nch))
        data = numpy.frombuffer(w.readframes(w.getnframes()), dtype="<i2").astype(numpy.int16)
    finally:
        w.close()
    if iq:
        return data.reshape(-1, 2).copy()
    return data[::nch].copy()


def _load_fsm(fsm_module):
    if fsm_module is not None:
        return fsm_module
    try:
        import packets  # noqa: F401  the reference requires packets to be imported before fsm (packets.py:55)
        import fsm
        return fsm
    except Exception:
        return None


class decoder(gr.hier_block2):
    def __init__(self, src="uhd", dst=None, repeat=False, reader=True, tag=True, samp_rate=2e6, emulator=None,
                 fsm=None, on_frame=None, device=0, on_frame_bytes=None, iq=False, **sink_kwargs):
        """iq=True: src is complex int16 baseband (UHD's sc16), an [n, 2] int16 array or a 2-channel 16-bit WAV path
        (channels I, Q), decoded as NFC_IN_SC16 with the thresholds of src="uhd".  Without it an int16 array or a WAV
        file's channel 0 is real PCM."""
        gr.hier_block2.__init__(self, "decoder",
                                gr.io_signature(0, 0, 0),  # Input signature
                                gr.io_signature(0, 0, 0))  # Output signature
        fsm_mod = _load_fsm(fsm)
        if on_frame is not None:
            self._on_frame = on_frame
        elif fsm_mod is None and on_frame_bytes is not None:
            self._on_frame = None  # bytes only: the device does the frame tail, nobody wants the bit lists
        elif fsm_mod is not None:  # packets.py:81-92
            if emulator:
                self._fsm = fsm_mod.fsm(emulator.process_packet)
                emulator.set_encoder(self._fsm.process_outgoing)
            else:
                self._fsm = fsm_mod.fsm()
            self._on_frame = self._fsm.process_bits
        else:
            raise ImportError("decoder needs the reference's fsm module on sys.path, or fsm=/on_frame=")

        self._pcm = None
        iq = bool(iq) and not (isinstance(src, str) and src == "uhd")
        if isinstance(src, str) and src == "uhd":
            hi_val = 1.1  # decoder.py:23
            kind = _cabi.IN_IQ_F32
        elif iq:
            hi_val = 1.1  # baseband from the USRP, as src="uhd" (decoder.py:23)
            kind = _cabi.IN_SC16
        else:
            hi_val = 1.09  # decoder.py:29: may need to be set to 1.05 depending on antenna setup
            kind = _cabi.IN_REAL_F32
        hi_val = sink_kwargs.pop("hi_val", hi_val)
        if iq:
            if isinstance(src, numpy.ndarray):
                _cabi._check_sc16(src, 2)
            elif not isinstance(src, str):
                raise TypeError("iq=True takes an [n, 2] int16 array or a 2-channel 16-bit WAV path")
        elif not HAVE_GNURADIO and isinstance(src, str) and src != "uhd":
            kind = _cabi.IN_PCM_S16  # no wavfile_source here: read the PCM ourselves, normalise on the device
        elif isinstance(src, numpy.ndarray):
            kind = {numpy.dtype(numpy.int16): _cabi.IN_PCM_S16,
                    numpy.dtype(numpy.complex64): _cabi.IN_IQ_F32}.get(src.dtype, _cabi.IN_REAL_F32)
        self._trans = frame_sink(samp_rate, self._on_frame, reader=reader, tag=tag, hi_val=hi_val, input_kind=kind,
                                 device=device, on_frame_bytes=on_frame_bytes, **sink_kwargs)
        if HAVE_GNURADIO and isinstance(src, str) and not iq:  # pragma: no cover - needs GNU Radio
            if src == "uhd":
                # the source of usrp_src.py:19-30 itself, complex items: the reference's wrapper squares them on the host
                # (usrp_src.py:31-33) and has a float output, this sink takes IN_IQ_F32 and computes the envelope on the device
                from gnuradio import uhd
                self._src = uhd.usrp_source(device_addr="", stream_args=uhd.stream_args(cpu_format="fc32", channels=range(1)))
                self._src.set_samp_rate(samp_rate)
                self._src.set_center_freq(13.57e6, 0)  # usrp_src.py:14 defaults: freq, rx_gain
                self._src.set_gain(6.5, 0)
                self._src.set_antenna("RX", 0)
            else:
                self._src = blocks.wavfile_source(src, repeat)
            self.connect(self._src, self._trans)
        elif isinstance(src, numpy.ndarray):
            self._pcm = src
        elif isinstance(src, str) and src != "uhd":
            self._pcm = read_wav(src, iq=iq)
        else:
            raise RuntimeError("src='uhd' needs GNU Radio and UHD")

    def run(self, chunk=8192):
        """Without a GNU Radio scheduler: push the whole source through work() in `chunk`-item calls."""
        x = self._pcm
        off = 0
        while off < len(x):
            used = self._trans.work([x[off: off + chunk]], None)
            off += used
            if used == 0:
                break
        self._trans.flush()
        return off

    def stream(self):
        return self._trans.stream()
