"""Batches of captures of different lengths in one device pass (nfc_stream_push_batch_ragged, Stream.push_batch_ragged,
batch.decode_batch_onepass with a list): every capture must equal the oracle's decode of that capture alone."""
import os

import numpy as np
import pytest

from oracle import oracle
from tests.test_gpu_sc16 import sc16_envelope, sc16_from_amplitude
from usrp_nfc_b200 import _cabi, batch, synth

pytestmark = pytest.mark.gpu

TILE = {13.56e6: 4096, 2e6: 512}  # the streaming slicer's tile at the rate's av_window


def _traffic(rate, i, seed0, n_items, pcm=False):
    """Session traffic of capture i cut to n_items: it ends wherever it falls, and every fifth capture starts inside it."""
    sess = synth.load_sessions()
    p = synth.rate_params(rate)
    name = "ultralight" if i % 3 == 0 else "classic1k"
    ch = synth.Channel(pause=0.02 + 0.005 * (i % 4), tag_high=1.06 + 0.01 * (i % 3), fade=0.02 * (i % 2))
    x = synth.capture(sess[name], rate, seed0 + i, channel=ch, av_window=p["av_window"], sessions=2)
    if not pcm:
        x = synth.envelope(synth.pcm_to_float(x))
    if i % 5 == 0:
        x = x[p["av_window"] + 6000 + 997 * (i % 7):]
    reps = int(np.ceil(max(n_items, 1) / x.size))
    return np.ascontiguousarray(np.tile(x, reps)[:n_items] if reps > 1 else x[:n_items])


def _thresholds(n):
    his = np.array([[1.05, 1.06, 1.07, 1.08, 1.09, 1.10][i % 6] for i in range(n)])
    los = np.array([[0.1, 0.08, 0.12][i % 3] for i in range(n)])
    return los, his


def _lengths(rate, n, seed, base=262144):
    """Seeded lengths from 0.3x to 3x of base, with the edge cases around the window at the front."""
    p = synth.rate_params(rate)
    L, mx = p["av_window"], p["max_len"]
    rng = np.random.default_rng(seed)
    lens = [int(v) for v in np.exp(rng.uniform(np.log(0.3 * base), np.log(3.0 * base), n))]
    edge = [L, L + 1, L + mx, L + 2 * mx, L + 2 * mx + 1, 7, 16 * TILE[rate], 16 * TILE[rate] + 1]
    lens[1:1 + len(edge)] = edge  # capture 0 stays a long one
    return lens


def _check_starts(starts, lens, rate):
    L, T = synth.rate_params(rate)["av_window"], TILE[rate]
    widths = [(-(-n // T) * T if n > L else 0) for n in lens]
    assert starts.dtype == np.int64
    assert starts.tolist() == [0] + np.cumsum(widths).tolist()


def _check(caps, rate, p, los, his, res, env=lambda x: x):
    got = batch.split_captures(res, len(caps))
    total = 0
    for i, (fr, bits) in enumerate(got):
        want = oracle.decode_capture(env(caps[i]), rate, lo_val=float(los[i]), hi_val=float(his[i]), **p)
        assert len(fr) == len(want["frames"]), (i, len(fr), len(want["frames"]))
        for f in ("pos", "nbits", "type"):
            assert np.array_equal(fr[f], want["frames"][f]), (i, f)
        for (pos, typ, b), wb in zip(batch.frames_as_lists(fr, bits), want["frame_bits"]):
            assert np.array_equal(b, wb), i
        total += len(fr)
    return total


@pytest.mark.parametrize("rate,n,seed", [(13.56e6, 40, 11000), (2e6, 30, 12000)])
def test_mixed_lengths_match_oracle(rate, n, seed):
    """Captures of 0.3x to 3x 262144 items with their own thresholds, tile multiples and not, one of at most av_window items,
    the lengths around av_window + 2 max_len, cut inside frames; one launch of the streaming slicer for all of them."""
    p = synth.rate_params(rate)
    lens = _lengths(rate, n, seed)
    caps = [_traffic(rate, i, seed, m) for i, m in enumerate(lens)]
    los, his = _thresholds(n)
    res = batch.decode_batch_onepass(caps, rate, p, lo_vals=los, hi_vals=his)
    assert res["pitch"] is None
    _check_starts(res["starts"], lens, rate)
    assert _check(caps, rate, p, los, his, res) > 100
    st = res["stream"].stats()
    assert st["slicer_kernel_launches"] == 1
    if rate == 13.56e6:
        assert st["pipe_tiles"] > 0 or os.environ.get("NFC_SLICER_PIPE") == "0"
    res["stream"].close()


def test_device_inputs_match_host_and_oracle():
    """Device captures as separate tensors, as 16-byte aligned slices of one flat tensor and as a misaligned slice (copied by
    the binding): the same frames as from host memory, and as the oracle's."""
    import torch
    rate, n, seed = 13.56e6, 10, 13000
    p = synth.rate_params(rate)
    lens = [400000, 13561, 170001, 262144, 13560, 90000, 500003, 250000, 131072, 333333]
    caps = [_traffic(rate, i, seed, m) for i, m in enumerate(lens)]
    los, his = _thresholds(n)
    s = _cabi.Stream(rate, outputs=_cabi.OUT_FRAMES, **p)
    host = batch.decode_batch_onepass(caps, rate, p, lo_vals=los, hi_vals=his, stream=s)
    want = batch.split_captures(host, n)
    assert sum(len(f) for f, _ in want) > 30

    def same(res):
        assert res["starts"].tolist() == host["starts"].tolist()
        for (fa, ba), (fb, bb) in zip(batch.split_captures(res, n), want):
            assert fa.tobytes() == fb.tobytes() and np.array_equal(ba, bb)

    same(batch.decode_batch_onepass([torch.from_numpy(c).cuda() for c in caps], rate, p, lo_vals=los, hi_vals=his, stream=s))
    offs = np.concatenate([[0], np.cumsum([(m + 3) // 4 * 4 for m in lens])])
    flat = np.zeros(int(offs[-1]) + 8, np.float32)
    for c, o in zip(caps, offs):
        flat[o: o + c.size] = c
    fd = torch.from_numpy(flat).cuda()
    same(batch.decode_batch_onepass([fd[int(o): int(o) + m] for o, m in zip(offs, lens)], rate, p, lo_vals=los, hi_vals=his,
                                    stream=s))
    # capture 3 one float further on: its address is not 16-byte aligned
    flat2 = flat.copy()
    o3 = int(offs[3]) + 1
    flat2[o3: o3 + lens[3]] = caps[3]
    fd2 = torch.from_numpy(flat2).cuda()
    views = [fd2[int(o): int(o) + m] for o, m in zip(offs, lens)]
    views[3] = fd2[o3: o3 + lens[3]]
    assert views[3].data_ptr() % 16 != 0
    same(batch.decode_batch_onepass(views, rate, p, lo_vals=los, hi_vals=his, stream=s))
    assert _check(caps, rate, p, los, his, host) > 30
    s.close()


def test_sc16_captures_of_different_lengths():
    import torch
    rate, n, seed = 13.56e6, 9, 14000
    p = synth.rate_params(rate)
    lens = [300001, 13560, 200000, 13561 + 2 * p["max_len"], 450000, 98304, 123457, 262144, 80000]
    caps = [sc16_from_amplitude(_traffic(rate, i, seed, m, pcm=True), seed + 100 + i) for i, m in enumerate(lens)]
    assert all(c.shape == (m, 2) and c.dtype == np.int16 for c, m in zip(caps, lens))
    los, his = _thresholds(n)
    res = batch.decode_batch_onepass(caps, rate, p, lo_vals=los, hi_vals=his, kind=_cabi.IN_SC16)
    _check_starts(res["starts"], lens, rate)
    assert _check(caps, rate, p, los, his, res, env=sc16_envelope) > 30
    res2 = batch.decode_batch_onepass([torch.from_numpy(c).cuda() for c in caps], rate, p, lo_vals=los, hi_vals=his,
                                      stream=res["stream"])
    assert _check(caps, rate, p, los, his, res2, env=sc16_envelope) > 30
    res["stream"].close()


def test_several_slabs_and_a_capture_wider_than_a_slab():
    rate, seed = 13.56e6, 15000
    p = synth.rate_params(rate)
    lens = [300000, 900001, 150000, 13560, 400000, 1200000, 20000, 13561, 610000, 250000, 5, 700000]
    caps = [_traffic(rate, i, seed, m) for i, m in enumerate(lens)]
    los, his = _thresholds(len(lens))
    s = _cabi.Stream(rate, outputs=_cabi.OUT_FRAMES, **p)
    s.set_tuning(slab_len=600000)  # 900001, 1200000, 610000 and 700000 items are wider: slabs of their own
    res = batch.decode_batch_onepass(caps, rate, p, lo_vals=los, hi_vals=his, stream=s)
    _check_starts(res["starts"], lens, rate)
    assert _check(caps, rate, p, los, his, res) > 50
    assert s.stats()["slicer_kernel_launches"] == 1
    s.close()


def test_sequential_fallback():
    rate, seed = 13.56e6, 16000
    p = synth.rate_params(rate)
    lens = [131072, 200001, 90000, 13560, 160000]
    caps = [_traffic(rate, i, seed, m) for i, m in enumerate(lens)]
    caps[2][5000] = -1.0  # a negative sample in the warm-up enters the ring: only the sequential path takes it
    los, his = _thresholds(len(lens))
    s = _cabi.Stream(rate, outputs=_cabi.OUT_FRAMES, **p)
    with pytest.raises(_cabi.BatchNeedsSequential):
        s.push_batch_ragged(caps, lo_vals=los, hi_vals=his)
    s.close()
    res = batch.decode_batch_onepass(caps, rate, p, lo_vals=los, hi_vals=his)
    assert res["per_capture"] is not None
    assert _check(caps, rate, p, los, his, res) > 10
    res["stream"].close()


def test_equal_lengths_through_both_entries():
    """A list of equally long captures lays out as the 2-D batch (starts[c] = c * pitch) and gives the same frame records and
    frame bits, byte for byte."""
    rate, n, m, seed = 13.56e6, 16, 262144 + 1000, 17000
    p = synth.rate_params(rate)
    caps = [_traffic(rate, i, seed, m) for i in range(n)]
    los, his = _thresholds(n)
    s = _cabi.Stream(rate, outputs=_cabi.OUT_FRAMES, **p)
    pitch = s.push_batch(np.stack(caps), lo_vals=los, hi_vals=his)
    fr0, b00, b01 = [np.array(v).copy() for v in s.view_frames()]
    s.release_frames()
    s.reset()
    starts = s.push_batch_ragged(caps, lo_vals=los, hi_vals=his)
    assert starts.tolist() == [c * pitch for c in range(n + 1)]
    fr1, b10, b11 = s.view_frames()
    assert len(fr0) > 100
    assert np.asarray(fr1).tobytes() == fr0.tobytes()
    assert np.array_equal(b10, b00) and np.array_equal(b11, b01)
    s.close()


def test_stream_reuse_equal_ragged_equal():
    """Equal-length, ragged and equal-length batches on one stream: the class bitmap outside each batch's segments must
    read as the warm-up / padding of that batch, never as a stale fill of the batch before."""
    rate, seed = 13.56e6, 18000
    p = synth.rate_params(rate)
    m = 262144 + 1000
    eq = np.stack([_traffic(rate, i, seed, m) for i in range(8)])
    lens = [150000, 13560, 700000, 262144 + 1000, 13561, 400000, 90001]
    rg = [_traffic(rate, i, seed + 50, n) for i, n in enumerate(lens)]
    los, his = _thresholds(8)
    s = _cabi.Stream(rate, outputs=_cabi.OUT_FRAMES, **p)
    for step in range(3):
        if step == 1:
            res = batch.decode_batch_onepass(rg, rate, p, lo_vals=los[:7], hi_vals=his[:7], stream=s)
            assert _check(rg, rate, p, los[:7], his[:7], res) > 30
        else:
            res = batch.decode_batch_onepass(eq, rate, p, lo_vals=los, hi_vals=his, stream=s)
            assert _check(list(eq), rate, p, los, his, res) > 30
        s.release_frames()
    s.close()


def test_host_captures_around_an_unmapped_hole():
    """Two host captures with an unmapped page range between them, passed in ascending address order: the library copies
    only the captures' own bytes (one copy each) and never the memory between them."""
    import ctypes
    import mmap
    rate, seed = 13.56e6, 19000
    p = synth.rate_params(rate)
    libc = ctypes.CDLL(None, use_errno=True)
    libc.mmap.restype = ctypes.c_void_p
    libc.mmap.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_long]
    libc.munmap.argtypes = [ctypes.c_void_p, ctypes.c_size_t]
    S = 200704 * 4  # bytes per region: a whole number of pages
    base = libc.mmap(None, 3 * S, mmap.PROT_READ | mmap.PROT_WRITE, mmap.MAP_PRIVATE | mmap.MAP_ANONYMOUS, -1, 0)
    assert base not in (None, ctypes.c_void_p(-1).value)
    try:
        assert libc.munmap(base + S, S) == 0  # the hole
        n = S // 4
        caps = [np.ctypeslib.as_array((ctypes.c_float * n).from_address(base + k * S)) for k in (0, 2)]
        for i, c in enumerate(caps):
            c[:] = _traffic(rate, i + 1, seed, n)
        los, his = _thresholds(2)
        s = _cabi.Stream(rate, outputs=_cabi.OUT_FRAMES, **p)
        res = batch.decode_batch_onepass(caps, rate, p, lo_vals=los, hi_vals=his, stream=s)
        assert s.stats()["h2d_bytes"] == 2 * S
        assert _check([c.copy() for c in caps], rate, p, los, his, res) > 5
        s.close()
    finally:
        libc.munmap(base, S)
        libc.munmap(base + 2 * S, S)
