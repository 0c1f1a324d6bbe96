"""Batches of captures of different lengths on the host: what the binding hands the library (one pointer and one length per
capture), what it refuses before the library is reached, and how split_captures assigns frames by the batch's starts.
No GPU needed."""
import ctypes
import os
import re

import numpy as np
import pytest

from usrp_nfc_b200 import _cabi, batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _StubLib(object):
    """Stands in for the library: records the pointers and lengths the binding passes and writes a layout."""

    def __init__(self, rc=None):
        self.calls = []
        self.rc = rc

    def nfc_stream_push_batch_ragged(self, h, items, mem, ncap, lengths, lo, hi, starts):
        ptrs = list(items)[:ncap]
        lens = list((ctypes.c_int64 * ncap).from_address(lengths))
        self.calls.append((ptrs, lens, mem))
        out = (ctypes.c_int64 * (ncap + 1)).from_address(starts)
        for c in range(ncap):
            out[c + 1] = out[c] + (0 if lens[c] <= 4 else -(-lens[c] // 8) * 8)
        return ncap if self.rc is None else self.rc

    def nfc_last_error(self):
        return b"stub"

    def nfc_stream_destroy(self, h):
        return 0


def _stream(monkeypatch, kind, rc=None):
    stub = _StubLib(rc)
    monkeypatch.setattr(_cabi, "lib", lambda: stub)
    s = object.__new__(_cabi.Stream)  # no device: the checks in front of the library only
    s._h = None
    s.input_kind = kind
    return s, stub


def test_symbol_in_header_and_binding():
    with open(os.path.join(ROOT, "include", "usrp_nfc_b200.h")) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    assert re.search(r"\bnfc_stream_push_batch_ragged\s*\(", text)
    assert "nfc_stream_push_batch_ragged" in _cabi.SIGNATURES


def test_one_pointer_and_length_per_capture(monkeypatch):
    s, stub = _stream(monkeypatch, _cabi.IN_ENVELOPE_F32)
    caps = [np.zeros(n, np.float32) for n in (3, 17, 0, 40)]
    starts = s.push_batch_ragged(caps)
    ptrs, lens, mem = stub.calls[-1]
    assert lens == [3, 17, 0, 40] and mem == _cabi.MEM_HOST
    assert ptrs[0] == caps[0].ctypes.data and ptrs[1] == caps[1].ctypes.data and ptrs[3] == caps[3].ctypes.data
    assert starts.dtype == np.int64 and starts.tolist() == [0, 0, 24, 24, 64]
    # other dtypes are converted like push_batch does; the lengths stay
    s.push_batch_ragged([np.arange(5, dtype=np.float64), [1.0, 2.0, 3.0]])
    assert stub.calls[-1][1] == [5, 3]


def test_sc16_captures_count_rows(monkeypatch):
    s, stub = _stream(monkeypatch, _cabi.IN_SC16)
    s.push_batch_ragged([np.zeros((9, 2), np.int16), np.zeros((64, 2), np.int16)[::2]])
    assert stub.calls[-1][1] == [9, 32]


@pytest.mark.parametrize("bad,exc", [
    ([np.zeros(16, np.int16)], ValueError),            # interleaved but flat
    ([np.zeros((16, 3), np.int16)], ValueError),
    ([np.zeros((2, 8, 2), np.int16)], ValueError),     # a 2-D batch as one capture
    ([np.zeros((16, 2), np.float32)], TypeError),
    ([np.zeros((16, 2), np.int16), [[0, 0]] * 4], TypeError),
])
def test_sc16_refuses_other_representations(monkeypatch, bad, exc):
    s, stub = _stream(monkeypatch, _cabi.IN_SC16)
    with pytest.raises(exc):
        s.push_batch_ragged(bad)
    assert stub.calls == []


def test_refuses_bad_shapes_and_dtypes(monkeypatch):
    torch = pytest.importorskip("torch")
    s, stub = _stream(monkeypatch, _cabi.IN_ENVELOPE_F32)
    for bad, exc in (([np.zeros((4, 4), np.float32)], ValueError), ([torch.zeros(8, dtype=torch.float64)], TypeError),
                     ([torch.zeros((2, 8))], ValueError), ([], ValueError)):
        with pytest.raises(exc):
            s.push_batch_ragged(bad)
    with pytest.raises(ValueError):
        s.push_batch_ragged([np.zeros(8, np.float32)] * 2, hi_vals=[1.1])
    assert stub.calls == []


class _FakeCuda(object):
    """A CUDA tensor as far as the binding looks at one (address, device, dtype, shape)."""

    def __init__(self, addr, n):
        self.addr, self.n, self.cloned = addr, n, False
        self.is_cuda = True
        self.dtype = "torch.float32"
        self.shape = (n,)
        self.device = "cuda:0"

    def dim(self):
        return 1

    def data_ptr(self):
        return self.addr

    def contiguous(self):
        return self

    def clone(self):
        c = _FakeCuda(4096 * 1024, self.n)
        c.cloned = True
        return c


def test_mixed_memory_refused(monkeypatch):
    s, stub = _stream(monkeypatch, _cabi.IN_ENVELOPE_F32)
    with pytest.raises(ValueError):
        s.push_batch_ragged([np.zeros(8, np.float32), _FakeCuda(1 << 20, 8)])
    assert stub.calls == []


def test_misaligned_device_capture_is_copied(monkeypatch):
    s, stub = _stream(monkeypatch, _cabi.IN_ENVELOPE_F32)
    synced = []

    class _Torch(object):
        class cuda(object):
            @staticmethod
            def current_stream(d):
                class _S(object):
                    def synchronize(self):
                        synced.append(d)
                return _S()

    monkeypatch.setitem(__import__("sys").modules, "torch", _Torch)
    aligned, odd = _FakeCuda(1 << 20, 100), _FakeCuda((1 << 20) + 4 * 101, 33)
    s.push_batch_ragged([aligned, odd])
    ptrs, lens, mem = stub.calls[-1]
    assert mem == _cabi.MEM_DEVICE and lens == [100, 33]
    assert ptrs[0] == aligned.addr and ptrs[1] == 4096 * 1024  # the copy, not the misaligned slice
    assert synced == ["cuda:0"]


def test_library_errors_surface(monkeypatch):
    s, _ = _stream(monkeypatch, _cabi.IN_ENVELOPE_F32, rc=-3)
    with pytest.raises(_cabi.BatchNeedsSequential):
        s.push_batch_ragged([np.zeros(8, np.float32)])
    s, _ = _stream(monkeypatch, _cabi.IN_ENVELOPE_F32, rc=-1)
    with pytest.raises(_cabi.NfcError):
        s.push_batch_ragged([np.zeros(8, np.float32)])


def _frames(rows):
    fr = np.zeros(len(rows), dtype=_cabi.FRAME_DTYPE)
    for i, (pos, off, nbits, typ) in enumerate(rows):
        fr[i] = (pos, off, nbits, typ)
    return fr


def test_split_captures_by_starts():
    # captures 1 and 3 own no positions (at most av_window items); capture 4 starts where capture 3 would
    starts = np.array([0, 4096, 4096, 12288, 12288, 16384], np.int64)
    bits_tag = np.arange(20, dtype=np.uint8) % 2
    bits_reader = (np.arange(30, dtype=np.uint8) // 3) % 2
    fr = _frames([(2500, 0, 4, 0), (4096 + 2100, 0, 7, 1), (4096 + 5000, 4, 3, 0), (12288 + 2001, 7, 9, 1),
                  (16383, 7, 2, 0)])
    res = dict(frames=fr, bits_tag=bits_tag, bits_reader=bits_reader, starts=starts, pitch=None)
    got = batch.split_captures(res, 5)
    assert [len(f) for f, _ in got] == [1, 0, 2, 0, 2]
    f0, b0 = got[0]
    assert f0["pos"].tolist() == [2500] and f0["bit_off"].tolist() == [0] and np.array_equal(b0, bits_tag[0:4])
    f2, b2 = got[2]
    assert f2["pos"].tolist() == [2100, 5000] and f2["bit_off"].tolist() == [0, 7] and f2["type"].tolist() == [1, 0]
    assert np.array_equal(b2, np.concatenate([bits_reader[0:7], bits_tag[4:7]]))
    f4, b4 = got[4]
    assert f4["pos"].tolist() == [2001, 4095] and f4["bit_off"].tolist() == [0, 9]
    assert np.array_equal(b4, np.concatenate([bits_reader[7:16], bits_tag[7:9]]))
    assert got[1][1].size == 0 and got[3][1].size == 0


def test_split_captures_equal_pitch_unchanged():
    """A 2-D batch's starts are c * pitch: the split is what pos // pitch gave."""
    pitch = 8192
    bits = np.ones(40, np.uint8)
    fr = _frames([(3000, 0, 5, 0), (pitch + 3000, 5, 5, 0), (3 * pitch + 8000, 10, 5, 0)])
    with_starts = batch.split_captures(dict(frames=fr, bits_tag=bits, bits_reader=bits, pitch=pitch,
                                            starts=np.arange(5, dtype=np.int64) * pitch), 4)
    pitch_only = batch.split_captures(dict(frames=fr, bits_tag=bits, bits_reader=bits, pitch=pitch), 4)
    for (fa, ba), (fb, bb) in zip(with_starts, pitch_only):
        assert fa.tobytes() == fb.tobytes() and np.array_equal(ba, bb)
    assert [len(f) for f, _ in with_starts] == [1, 1, 0, 1] and with_starts[3][0]["pos"][0] == 8000
