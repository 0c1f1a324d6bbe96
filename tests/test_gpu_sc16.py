"""Complex int16 baseband (NFC_IN_SC16, UHD's sc16): one item is an (I, Q) pair of int16.  Its envelope is by definition
that of the complex64 item (I / pcm_scale, Q / pcm_scale) through NFC_IN_IQ_F32, so every decode here is compared twice:
with the oracle fed that envelope (computed in float32 on the host) and, bit for bit, with the IQ_F32 decode of the
complex64 conversion -- events, symbols, frames, frame bits and the final slicer state, ring included."""
import wave

import numpy as np
import pytest

from oracle import oracle
from tests import helpers as H
from usrp_nfc_b200 import _cabi, batch, synth

pytestmark = pytest.mark.gpu

SCALE = np.float32(32767.0)


def sc16_from_amplitude(a, seed):
    """I = rint(a cos phi), Q = rint(a sin phi) with a seeded uniform phase, clipped to int16: [n, 2]."""
    rng = np.random.default_rng(seed)
    phi = rng.uniform(0.0, 2.0 * np.pi, a.size)
    a = np.asarray(a, dtype=np.float64)
    iq = np.empty((a.size, 2), dtype=np.int16)
    iq[:, 0] = np.clip(np.rint(a * np.cos(phi)), -32768, 32767)
    iq[:, 1] = np.clip(np.rint(a * np.sin(phi)), -32768, 32767)
    return iq


def sc16_to_c64(iq, scale=SCALE):
    f = iq.astype(np.float32) / np.float32(scale)  # RN32(I / scale), RN32(Q / scale)
    return np.ascontiguousarray(f).view(np.complex64).reshape(-1)


def sc16_envelope(iq, scale=SCALE):
    """RN32(RN32(fi * fi) + RN32(fq * fq)), fi = RN32(I / scale): the definition of the sc16 envelope (no FMA)."""
    f = iq.astype(np.float32) / np.float32(scale)
    a = f[:, 0] * f[:, 0]
    b = f[:, 1] * f[:, 1]
    return (a + b).astype(np.float32)


def decode(x, rate, kind, chunk=None, tuning=None, **kw):
    s = _cabi.Stream(rate, input_kind=kind, **kw)
    if tuning:
        s.set_tuning(**tuning)
    s.reset_stats()  # the tile counters are device-wide: count this stream's decode only
    n = len(x)
    off, step = 0, chunk or max(n, 1)
    while off < n:
        used, _ = s.push(x[off: off + step])
        assert used > 0
        off += used
    out = dict(events=s.drain_events(), symbols=s.drain_symbols())
    out["frames"], out["frame_bits"] = s.drain_frames()
    out["state"], out["ring"], _ = s.state()
    out["stats"] = s.stats()
    s.close()
    return out


def check_against_oracle(got, want):
    H.assert_events_equal(got["events"], want["events"])
    H.assert_symbols_equal(got["symbols"], want["symbols"])
    assert len(got["frames"]) == len(want["frames"])
    for f in ("pos", "nbits", "type"):
        assert np.array_equal(got["frames"][f], want["frames"][f]), f
    for a, b in zip(got["frame_bits"], want["frame_bits"]):
        assert np.array_equal(a, b)


def check_identical(a, b):
    """Two decodes of the same envelope: identical records, frame bits and final state."""
    for k in ("events", "symbols", "frames"):
        assert a[k].tobytes() == b[k].tobytes(), k
    assert len(a["frame_bits"]) == len(b["frame_bits"])
    for x, y in zip(a["frame_bits"], b["frame_bits"]):
        assert np.array_equal(x, y)
    assert a["state"].pos == b["state"].pos and a["state"].ss == b["state"].ss
    assert a["state"].serial_mode == b["state"].serial_mode
    assert a["ring"].tobytes() == b["ring"].tobytes()


def check_sc16(iq, rate, chunk=None, tuning=None, min_frames=1, **kw):
    """iq decoded as sc16 equals the oracle and the IQ_F32 decode of its complex64 conversion; returns the sc16 decode."""
    want = oracle.decode_capture(sc16_envelope(iq), rate, **kw)
    got = decode(iq, rate, _cabi.IN_SC16, chunk=chunk, tuning=tuning, **kw)
    check_against_oracle(got, want)
    ref = decode(sc16_to_c64(iq), rate, _cabi.IN_IQ_F32, chunk=chunk, tuning=tuning, **kw)
    check_identical(got, ref)
    assert len(want["frames"]) >= min_frames
    got["iq_f32"] = ref
    return got


STORED = [
    ("surrogate_ultralight", 2e6, dict(hi_val=1.09)),  # tiles of 512 samples, pipelined
    ("rate_1356", 13.56e6, dict(hi_val=1.09, av_window=13560, max_len=339)),  # tiles of 4096, pipelined
    ("rate_2000", 20e6, dict(hi_val=1.09, av_window=20000, max_len=500)),  # tiles of 2048, pipelined
]


@pytest.mark.parametrize("name,rate,kw", STORED)
@pytest.mark.parametrize("chunk", [None, 8192, 3001])
def test_stored_captures_as_sc16(name, rate, kw, chunk):
    """Whole, in 8192-item calls, and in calls of an odd size (the warm-up ends inside a call, slabs start unaligned)."""
    iq = sc16_from_amplitude(H.load_case(name)["pcm"], 11)
    got = check_sc16(iq, rate, chunk=chunk, **kw)
    if chunk is None:
        # the pipelined mode of the streaming kernel ran on sc16 input (complex64 input never takes it)
        assert got["stats"]["pipe_tiles"] > 0, got["stats"]
        assert got["iq_f32"]["stats"]["pipe_tiles"] == 0


def _long_capture(rate, seed, sessions):
    p = synth.rate_params(rate)
    pcm = synth.capture(synth.load_sessions()["classic1k"], rate, seed, channel=synth.Channel(pause=0.03, tag_high=1.07, fade=0.05),
                        av_window=p["av_window"], sessions=sessions)
    return sc16_from_amplitude(pcm, seed + 1), p


@pytest.mark.parametrize("shift", [0, 1, 3])
def test_device_resident_sc16(shift):
    """A CUDA tensor [n, 2] of int16: read in place when 16-byte aligned, through the staging copy when it starts 1 or 3 items
    later.  Short segments and slabs: speculative segments, seam checks and several slabs per launch on sc16 input."""
    import torch
    rate = 13.56e6
    iq, p = _long_capture(rate, 500, 2)
    t = torch.from_numpy(np.concatenate([np.zeros((shift, 2), np.int16), iq])).cuda()[shift:]
    assert t.shape == (len(iq), 2) and (t.data_ptr() % 16 == 0) == (shift == 0)
    tuning = dict(seg_len=65536, halo=4 * p["av_window"], slab_len=1 << 19)
    want = oracle.decode_capture(sc16_envelope(iq), rate, hi_val=1.09, **p)
    got = decode(t, rate, _cabi.IN_SC16, tuning=tuning, hi_val=1.09, **p)
    check_against_oracle(got, want)
    ref = decode(torch.from_numpy(sc16_to_c64(iq)).cuda(), rate, _cabi.IN_IQ_F32, tuning=tuning, hi_val=1.09, **p)
    check_identical(got, ref)
    assert got["stats"]["segments"] >= 3 and len(want["frames"]) > 100
    assert got["stats"]["slicer_kernel_launches"] > 0


@pytest.mark.parametrize("L,tuning", [(1000, dict(seg_len=4096, halo=1024)), (1002, dict(seg_len=4096, halo=1024)),
                                      (2000, dict(force_serial=True))])
def test_other_kernels_on_sc16(L, tuning):
    """av_window 1000 / 1002: the first-generation kernel (a window that is a multiple of 4 and one that is not);
    force_serial: the sequential kernel."""
    iq = sc16_from_amplitude(H.load_case("surrogate_classic1k")["pcm"], 12)
    got = check_sc16(iq, 2e6, tuning=tuning, hi_val=1.09, av_window=L, max_len=50, min_frames=100)
    assert got["stats"]["slicer_kernel_launches"] == 0
    if tuning.get("force_serial"):
        assert got["stats"]["serial_segments"] > 0


def _corner_amplitude(L, mx, n, seed):
    """The corner-case stream of the longest-window test as an amplitude (envelope 0.25 <-> 16384): long pauses at envelope
    1e-3, spikes right after a pause, stretches hovering around the HIGH threshold, steps of the level."""
    rng = np.random.default_rng(seed)
    x = (0.25 * (1 + 0.01 * rng.standard_normal(n))).astype(np.float64)
    i = L + 10
    while i < n - 4 * mx - 10:
        kind = rng.integers(0, 5)
        ln = int(rng.choice([1, 2, mx - 1, mx, mx + 1, 2 * mx, 2 * mx + 1, 3 * mx + 1, 6, 700]))
        ln = min(ln, n - i - 1)
        if kind == 0:
            x[i:i + ln] = 1e-3
            i += ln
            if rng.random() < 0.7:
                k = int(rng.integers(0, mx + 4))
                x[i + k: i + k + int(rng.integers(1, 4))] = 0.4
        elif kind == 1:
            x[i:i + ln] = 0.3 * (1 + 0.01 * rng.standard_normal(ln))
            i += ln
        elif kind == 2:
            x[i:i + ln] = 0.2725 * (1 + 0.002 * rng.standard_normal(ln))
            i += ln
        elif kind == 3 and rng.random() < 0.05:
            x[i:] *= rng.choice([0.7, 1.4])
        i += int(rng.integers(1, 6 * mx))
    return np.sqrt(x) * 32768.0


@pytest.mark.parametrize("L,mx,streaming", [(1024, 50, True), (52000, 339, True), (51998, 339, False)])
def test_window_edges_on_sc16(L, mx, streaming):
    """1024: the shortest streaming window; 52000: the streaming kernel's synchronous loop at 4 B per item (the ring, the
    staging tile and the static scratch fill one CTA's shared memory); 51998: the first-generation kernel."""
    iq = sc16_from_amplitude(_corner_amplitude(L, mx, 1_500_000, L + mx), 13)
    got = check_sc16(iq, 13.56e6, tuning=dict(seg_len=262144, halo=4 * L), hi_val=1.09, av_window=L, max_len=mx, min_frames=0)
    st = got["stats"]
    assert not got["state"].serial_mode
    assert st["segments"] >= 3
    if streaming:
        assert st["slicer_kernel_launches"] > 0
    else:
        assert st["slicer_kernel_launches"] == 0 and st["serial_segments"] == 0


@pytest.mark.parametrize("rate,L,mx", [(2e6, 2000, 50), (13.56e6, 8192, 50), (13.56e6, 13560, 339)])
def test_degenerate_sc16_values(rate, L, mx):
    """Envelopes that are exactly 0 (I = Q = 0), full-scale pairs (-32768, -32768: envelope 2 (32768/32767)^2) and a long
    silence: the span audit and the fall-back to the sequential kernel decide the path, the result equals the oracle."""
    n = 400000
    a = 16384.0 * (1 + 0.01 * np.random.default_rng(5).standard_normal(n))
    iq = sc16_from_amplitude(a, 14)
    iq[30000:30040] = 0                 # a short run of zeros inside the carrier
    iq[50000:50003] = 0
    iq[60000:60010] = -32768            # full-scale pairs: HIGH
    iq[60500:60600:7] = -32768
    iq[70000:70200] = 0                 # a pause of zeros, then full scale right after it
    iq[70200:70203] = -32768
    iq[150000:260000] = 0               # long silence: the window sum reaches 0
    iq[300000:300001] = (1, 0)          # the smallest non-zero envelope, 1/32767^2
    for chunk in (None, 8192):
        check_sc16(iq, rate, chunk=chunk, hi_val=1.09, av_window=L, max_len=mx, min_frames=0)


def _uniform_sc16_captures(rate, n, n_items, seed0):
    sess = synth.load_sessions()
    p = synth.rate_params(rate)
    caps, his, los = [], [], []
    for i in range(n):
        name = "ultralight" if i % 3 == 0 else "classic1k"
        ch = synth.Channel(pause=0.02 + 0.005 * (i % 4), tag_high=1.06 + 0.01 * (i % 3), fade=0.02 * (i % 2))
        pcm = synth.capture(sess[name], rate, seed0 + i, channel=ch, av_window=p["av_window"], sessions=2)
        if i % 5 == 0:  # the capture starts inside the traffic
            pcm = pcm[p["av_window"] + 6000 + 997 * (i % 7):]
        reps = int(np.ceil(n_items / pcm.size))
        pcm = np.tile(pcm, reps)[:n_items] if reps > 1 else pcm[:n_items]
        caps.append(sc16_from_amplitude(pcm, seed0 + 100 + i))
        his.append([1.05, 1.06, 1.07, 1.08, 1.09, 1.10][i % 6])
        los.append([0.1, 0.08, 0.12][i % 3])
    return np.stack(caps), np.array(los), np.array(his), p


def _check_batch(x3d, rate, p, los, his, res):
    got = batch.split_captures(res, x3d.shape[0])
    total = 0
    for i, (fr, bits) in enumerate(got):
        want = oracle.decode_capture(sc16_envelope(x3d[i]), rate, lo_val=float(los[i]), hi_val=float(his[i]), **p)
        assert len(fr) == len(want["frames"]), (i, len(fr), len(want["frames"]))
        for f in ("pos", "nbits", "type"):
            assert np.array_equal(fr[f], want["frames"][f]), (i, f)
        for (pos, typ, b), wb in zip(batch.frames_as_lists(fr, bits), want["frame_bits"]):
            assert np.array_equal(b, wb), i
        total += len(fr)
    return total


def test_batch_of_sc16_captures():
    """push_batch with [captures, items, 2]: from host memory (numpy) and from the device (torch), per-capture thresholds;
    every capture equals the oracle's decode of that capture alone."""
    import torch
    rate, n, n_items = 13.56e6, 12, 262144 + 1000
    x3d, los, his, p = _uniform_sc16_captures(rate, n, n_items, 7300)
    assert x3d.shape == (n, n_items, 2) and x3d.dtype == np.int16
    res = batch.decode_batch_onepass(x3d, rate, p, lo_vals=los, hi_vals=his, kind=_cabi.IN_SC16)
    assert res["pitch"] is not None and res["pitch"] >= n_items
    assert _check_batch(x3d, rate, p, los, his, res) > 100
    st = res["stream"].stats()
    assert st["slicer_kernel_launches"] == 1
    xd = torch.from_numpy(x3d).cuda()
    res2 = batch.decode_batch_onepass(xd, rate, p, lo_vals=los[::-1].copy(), hi_vals=his[::-1].copy(), stream=res["stream"])
    assert res2["pitch"] == res["pitch"]
    assert _check_batch(x3d, rate, p, los[::-1], his[::-1], res2) > 100
    # a view of every other capture: the stride between captures is not the capture length
    xv = xd[::2]
    res3 = batch.decode_batch_onepass(xv, rate, p, lo_vals=los[::2].copy(), hi_vals=his[::2].copy(), stream=res["stream"])
    assert _check_batch(x3d[::2], rate, p, los[::2], his[::2], res3) > 50
    res["stream"].close()
    # the worker-thread batch path takes [n, 2] captures the same way
    got = batch.decode_batch([x3d[i] for i in range(3)], rate, [dict(hi_val=float(his[i]), lo_val=float(los[i]), **p) for i in range(3)],
                             kind=_cabi.IN_SC16, workers=2)
    for i, (fr, bits) in enumerate(got):
        want = oracle.decode_capture(sc16_envelope(x3d[i]), rate, lo_val=float(los[i]), hi_val=float(his[i]), **p)
        assert np.array_equal(fr["pos"], want["frames"]["pos"]), i


def _stream_frames(x, kind, hi_val, rate=2e6):
    s = _cabi.Stream(rate, hi_val=hi_val, input_kind=kind, outputs=_cabi.OUT_FRAMES)
    s.push_all(x)
    fr, bits = s.drain_frames()
    s.close()
    return [(int(f["type"]), b.tolist()) for f, b in zip(fr, bits)]


def _write_wav(path, iq):
    w = wave.open(str(path), "wb")
    w.setnchannels(2)
    w.setsampwidth(2)
    w.setframerate(2000000)
    w.writeframes(np.ascontiguousarray(iq).astype("<i2").tobytes())
    w.close()


def test_decoder_block_takes_sc16(tmp_path):
    """decoder(src=..., iq=True): an [n, 2] int16 array or a 2-channel 16-bit WAV file, the same frames as the Stream path
    (hi_val 1.1, as for src="uhd"); frame_sink's coalescing passes the [n, 2] items through; without iq=True a stereo WAV
    is still its channel 0 as PCM."""
    from usrp_nfc_b200.decoder import decoder, frame_sink
    case = H.load_case("surrogate_classic1k")
    iq = sc16_from_amplitude(case["pcm"], 15)
    want = _stream_frames(iq, _cabi.IN_SC16, 1.1)
    assert len(want) > 100

    def run(src, **kw):
        got = []
        d = decoder(src=src, samp_rate=2e6, on_frame=lambda bits, t: got.append((t, list(bits))), **kw)
        d.run()
        return got

    assert run(iq, iq=True) == want
    assert run(iq, iq=True, coalesce=50000) == want
    path = tmp_path / "iq.wav"
    _write_wav(path, iq)
    assert run(str(path), iq=True) == want
    # without iq=True: channel 0 of the same file, as real PCM with the WAV path's threshold
    assert run(str(path)) == _stream_frames(iq[:, 0].copy(), _cabi.IN_PCM_S16, 1.09)

    sink = frame_sink(2e6, None, input_kind=_cabi.IN_SC16)
    assert sink._in_sig == [(np.int16, 2)]
    assert sink.work([iq[:5000]], None) == 2000  # the warm-up part of the first call (av_window items)
    sink.stream().close()
