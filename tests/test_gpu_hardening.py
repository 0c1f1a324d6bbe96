"""The rare paths of the CUDA pipeline, forced and asserted as taken: the line-code scan fallback, the transition-buffer
overflow retry, seam mismatches and their repair, two live streams of different windows on one device, the synthesis kernel
against the host renderer.  Every case is compared with the oracle."""
import numpy as np
import pytest

from oracle import oracle
from usrp_nfc_b200 import _cabi, synth

from .test_gpu_parity import check_against_oracle, gpu_decode

pytestmark = pytest.mark.gpu


def test_line_code_scan_fallback_is_taken():
    """More than 4096 events without a single reader event: the frame-boundary search finds no known Miller state and the
    slab takes the transfer-function scan (linecode.cu: chunk_map_kernel + ChunkMap scan)."""
    rate = 2e6
    rng = np.random.default_rng(11)
    frames = [(synth.TAG_TO_READER, synth.bytes_to_bits(rng.integers(0, 256, 18).tolist())) for _ in range(60)]
    pcm = synth.capture(frames, rate, 12, channel=synth.Channel(tag_high=1.12), av_window=2000, tag_gap_us=(60.0, 90.0))
    x = synth.envelope(synth.pcm_to_float(pcm))
    want = oracle.decode_capture(x, rate, hi_val=1.09)
    assert len(want["events"]) > 6000 and not (want["events"]["type"] == 1).any()
    got = gpu_decode(x, rate, hi_val=1.09)
    check_against_oracle(got, want)
    assert got["stream"].stats()["linecode_scan_fallbacks"] > 0


def test_transition_buffer_overflow_is_retried():
    """A stretch where val changes with every sample: the segments' transition lists outgrow their first estimate
    (one per eight samples) and the launch is repeated with larger buffers.  (A window below 1024 samples: the
    first-generation kernel with transition lists; larger windows write the class bitmap.)"""
    rate = 2e6
    frames = synth.load_sessions()["ultralight"]
    pcm = synth.capture(frames, rate, 5, av_window=1000)
    x = synth.envelope(synth.pcm_to_float(pcm)).copy()
    lvl = float(np.median(x[:1000]))
    a = 2000 + 9000
    x[a: a + 20000: 2] = np.float32(lvl * 1.3)  # HIGH on every other sample, the carrier level between
    want = oracle.decode_capture(x, rate, hi_val=1.09, av_window=1000)
    got = gpu_decode(x, rate, hi_val=1.09, av_window=1000, tuning=dict(seg_len=8192, halo=4096))
    check_against_oracle(got, want)
    assert got["stream"].stats()["overflow_retries"] > 0


@pytest.mark.parametrize("av_window,seg_len,halo", [(2000, 4096, 1024), (1000, 1024, 256), (1002, 1024, 256)])
def test_seam_mismatches_are_found_and_repaired(av_window, seg_len, halo):
    """Short segments with a short halo: speculative starts inside frames do not converge in time, the seam check finds
    them and the repair restores the exact stream.  av_window 2000: the streaming kernel (class bitmap); 1000 and 1002:
    the first-generation kernel (transition lists, tiles of 256 samples: segments of four tiles with a halo of one), with a
    window that is a multiple of 4 and one that is not."""
    rate = 2e6
    frames = synth.load_sessions()["classic1k"]
    pcm = synth.capture(frames, rate, 77, channel=synth.Channel(pause=0.03, tag_high=1.07, fade=0.06), av_window=av_window)
    x = synth.envelope(synth.pcm_to_float(pcm))
    want = oracle.decode_capture(x, rate, hi_val=1.09, av_window=av_window)
    got = gpu_decode(x, rate, hi_val=1.09, av_window=av_window, tuning=dict(seg_len=seg_len, halo=halo))
    check_against_oracle(got, want)
    st = got["stream"].stats()
    assert st["segments"] > 20 and st["seam_mismatches"] > 0


def test_two_live_streams_of_different_windows_alternate():
    """Two envelope streams with different av_window >= 8192 on one device, pushed in turns: each launch of the streaming
    kernel needs its own amount of dynamic shared memory."""
    frames = synth.load_sessions()["ultralight"]
    streams = []
    for rate, L, mx in ((13.56e6, 13560, 339), (13.56e6, 9000, 339), (20e6, 20000, 500)):
        pcm = synth.capture(frames, rate, 8, av_window=L)
        x = synth.envelope(synth.pcm_to_float(pcm))
        streams.append((x, rate, L, mx, _cabi.Stream(rate, hi_val=1.09, av_window=L, max_len=mx)))
    offs = [0] * len(streams)
    for step in range(6):
        for k, (x, rate, L, mx, s) in enumerate(streams):
            n = x.size // 5 + 1
            if offs[k] < x.size:
                used, _ = s.push(x[offs[k]: offs[k] + n])
                offs[k] += used
    for k, (x, rate, L, mx, s) in enumerate(streams):
        while offs[k] < x.size:
            used, _ = s.push(x[offs[k]:])
            offs[k] += used
        want = oracle.decode_capture(x, rate, hi_val=1.09, av_window=L, max_len=mx)
        fr, bits = s.drain_frames()
        assert len(fr) == len(want["frames"]) and np.array_equal(fr["pos"], want["frames"]["pos"])
        for a, b in zip(bits, want["frame_bits"]):
            assert np.array_equal(a, b)
        assert s.stats()["fast_tiles"] > 0
        s.close()


def test_synthesis_kernel_renders_the_host_schedule():
    """synth_kernel (binary_src.work, binary_src.py:64-103, on the device) against the host renderer without noise and
    fade: identical 16-bit PCM, identical envelope."""
    import torch
    rate = 13.56e6
    rng = np.random.default_rng(3)
    frames = synth.load_sessions()["ultralight"]
    codes, lens = synth.schedule(frames, rate, rng, av_window=13560)
    ch = synth.Channel(carrier=0.5, pause=0.02, tag_high=1.08, noise=0.0, fade=0.0)
    pcm = synth.render(codes, lens, rate, np.random.default_rng(0), ch)
    n = int(lens.sum())
    for as_env in (False, True):
        x = torch.empty(n + 1000, dtype=torch.float32, device="cuda")  # the schedule repeats behind its end
        _cabi.synth_render(x, codes, lens, carrier=0.5, pause=0.02, tag_high=1.08, noise=0.0, fade=0.0, as_envelope=as_env)
        got = x.cpu().numpy()
        want = synth.pcm_to_float(pcm)
        if as_env:
            want = synth.envelope(want)
        assert np.array_equal(got[:n], want)
        assert np.array_equal(got[n:], want[:1000])
    # a time shard of the endless capture: first_index shifts the schedule
    y = torch.empty(5000, dtype=torch.float32, device="cuda")
    _cabi.synth_render(y, codes, lens, carrier=0.5, pause=0.02, tag_high=1.08, noise=0.0, fade=0.0, as_envelope=False, first_index=n - 1234)
    ref = synth.pcm_to_float(np.concatenate([pcm, pcm]))[n - 1234: n - 1234 + 5000]
    assert np.array_equal(y.cpu().numpy(), ref)


def test_queued_slab_chain_is_done_again_when_its_buffers_are_too_small():
    """Slabs after the first are queued with buffers sized from the slabs before (no host round trip per slab).  Calm
    slabs first, then a stretch where val changes with every sample: the chain of that slab finds its buffers too small,
    raises the flag in its context block, and the host does it (and the slab queued behind it) again with exact sizes."""
    rate, L, mx = 13.56e6, 13560, 339
    frames = synth.load_sessions()["ultralight"]
    pcm = synth.capture(frames, rate, 5, av_window=L, sessions=24)
    x = synth.envelope(synth.pcm_to_float(pcm)).copy()
    slab = 1 << 20
    assert x.size > 5 * slab
    lvl = float(np.median(x[:L]))
    a = 3 * slab + 70000
    x[a: a + 400000: 2] = np.float32(lvl * 1.3)  # HIGH on every other sample: 400k transitions in one slab
    want = oracle.decode_capture(x, rate, hi_val=1.09, av_window=L, max_len=mx)
    got = gpu_decode(x, rate, hi_val=1.09, av_window=L, max_len=mx, tuning=dict(slab_len=slab))
    check_against_oracle(got, want)
    st = got["stream"].stats()
    import os
    assert st["fast_tiles"] > 0
    assert st["overflow_retries"] > 0 or os.environ.get("NFC_POST_SYNC")  # (every slab is sized exactly then)


def test_frame_index_is_the_frames_in_eight_bytes():
    """nfc_stream_view_frame_index: one packed record per frame of view_frames (pos << 24 | nbits << 8 | type), kept in step
    with the frame records over several pushes, emptied by release."""
    from usrp_nfc_b200 import sharding
    rate = 13.56e6
    p = synth.rate_params(rate)
    frames = synth.load_sessions()["classic1k"]
    pcm = synth.capture(frames, rate, 9, av_window=p["av_window"], sessions=2)
    x = synth.envelope(synth.pcm_to_float(pcm))
    s = _cabi.Stream(rate, hi_val=1.09, outputs=_cabi.OUT_FRAMES, **p)
    s.set_tuning(slab_len=1 << 20)
    half = x.size // 2
    s.push_all(x[:half])
    s.push_all(x[half:])
    fr, b0, b1 = s.view_frames()
    idx = s.view_frame_index()
    assert len(fr) == len(idx) > 100
    back = sharding.unpack_records([idx], [0])
    assert np.array_equal(back["pos"], fr["pos"]) and np.array_equal(back["nbits"], fr["nbits"]) and np.array_equal(back["type"], fr["type"])
    assert np.array_equal(sharding.pack_records(fr), idx)
    s.release_frames()
    assert len(s.view_frame_index()) == 0 and len(s.view_frames()[0]) == 0
    s.close()


def test_frame_index_in_the_callers_memory():
    """nfc_stream_set_frame_index_buffer: the packed index is written into memory of the caller's (what the ranks of a node
    share); a buffer that is too small is reported, not overrun."""
    import ctypes
    rate = 2e6
    frames = synth.load_sessions()["ultralight"]
    x = synth.envelope(synth.pcm_to_float(synth.capture(frames, rate, 3)))
    buf = (ctypes.c_uint64 * 64)()
    guard = 0xdeadbeefdeadbeef
    for i in range(64):
        buf[i] = guard
    s = _cabi.Stream(rate, hi_val=1.09, outputs=_cabi.OUT_FRAMES)
    s.set_frame_index_buffer(ctypes.addressof(buf), 32)
    s.push_all(x)
    fr = s.view_frames()[0]
    idx = s.view_frame_index()
    assert len(fr) == len(frames) == len(idx) <= 32
    assert idx.ctypes.data == ctypes.addressof(buf) and all(buf[i] == guard for i in range(32, 64))
    assert np.array_equal(idx >> np.uint64(24), fr["pos"].astype(np.uint64))
    s.release_frames()
    s.reset()
    s.set_frame_index_buffer(ctypes.addressof(buf), 4)  # fewer records than the capture has frames
    with pytest.raises(_cabi.NfcError):
        s.push_all(x)
        s.view_frame_index()
    assert all(buf[i] == guard for i in range(32, 64))
    s.close()
