"""The sc16 input kind (complex int16, UHD's sc16) on the host: the enum value, the WAV reader and the binding's shape and dtype
checks, which must refuse bad input before the library is reached.  No GPU needed."""
import ctypes
import os
import re
import wave

import numpy as np
import pytest

from usrp_nfc_b200 import _cabi, decoder

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_enum_matches_binding():
    with open(os.path.join(ROOT, "include", "usrp_nfc_b200.h")) as f:
        text = f.read()
    kinds = dict((k, int(v)) for k, v in re.findall(r"\bNFC_IN_([A-Z0-9_]+)\s*=\s*(\d+)", text))
    assert kinds["SC16"] == _cabi.IN_SC16 == 4
    assert [kinds[k] for k in ("ENVELOPE_F32", "REAL_F32", "IQ_F32", "PCM_S16")] == [
        _cabi.IN_ENVELOPE_F32, _cabi.IN_REAL_F32, _cabi.IN_IQ_F32, _cabi.IN_PCM_S16]


def _write_wav(path, data, channels):
    w = wave.open(str(path), "wb")
    w.setnchannels(channels)
    w.setsampwidth(2)
    w.setframerate(2000000)
    w.writeframes(np.ascontiguousarray(data).astype("<i2").tobytes())
    w.close()


def test_wav_reader(tmp_path):
    rng = np.random.default_rng(1)
    iq = rng.integers(-32768, 32768, (1001, 2)).astype(np.int16)
    _write_wav(tmp_path / "iq.wav", iq, 2)
    got = decoder.read_wav(str(tmp_path / "iq.wav"), iq=True)
    assert got.dtype == np.int16 and got.shape == (1001, 2) and np.array_equal(got, iq)
    ch0 = decoder.read_wav(str(tmp_path / "iq.wav"))
    assert ch0.dtype == np.int16 and ch0.shape == (1001,) and np.array_equal(ch0, iq[:, 0])
    _write_wav(tmp_path / "mono.wav", iq[:, 1], 1)
    assert np.array_equal(decoder.read_wav(str(tmp_path / "mono.wav")), iq[:, 1])
    with pytest.raises(ValueError):
        decoder.read_wav(str(tmp_path / "mono.wav"), iq=True)


class _StubLib(object):
    """Stands in for the library: records the item counts and strides the binding passes."""

    def __init__(self):
        self.calls = []

    def nfc_stream_push(self, h, addr, n, mem, cb):
        self.calls.append(("push", n, mem))
        return n

    def nfc_stream_push_batch(self, h, addr, mem, ncap, n, stride, lo, hi, pitch):
        self.calls.append(("push_batch", ncap, n, stride, mem))
        return ncap

    def nfc_stream_destroy(self, h):
        return 0


@pytest.fixture
def sc16_stream(monkeypatch):
    stub = _StubLib()
    monkeypatch.setattr(_cabi, "lib", lambda: stub)
    s = object.__new__(_cabi.Stream)  # no device: the checks in front of the library only
    s._h = None
    s.input_kind = _cabi.IN_SC16
    return s, stub


@pytest.mark.parametrize("bad,exc", [
    (np.zeros(16, np.int16), ValueError),               # interleaved but flat
    (np.zeros((16, 3), np.int16), ValueError),
    (np.zeros((2, 8, 2), np.int16), ValueError),        # a batch handed to push
    (np.zeros((16, 2), np.float32), TypeError),
    (np.zeros((16, 2), np.int32), TypeError),
    (np.zeros(16, np.complex64), TypeError),
    ([[0, 0]] * 16, TypeError),
])
def test_push_refuses_other_representations(sc16_stream, bad, exc):
    s, stub = sc16_stream
    with pytest.raises(exc):
        s.push(bad)
    with pytest.raises(exc):
        s.push_all(bad)
    assert stub.calls == []


def test_push_counts_items_not_elements(sc16_stream):
    s, stub = sc16_stream
    assert s.push(np.zeros((37, 2), np.int16)) == (37, False)
    assert s.push(np.zeros((64, 2), np.int16)[::2]) == (32, False)  # a strided view is copied, still 32 items
    assert s.push_all(np.zeros((100, 2), np.int16), chunk=40) == 100
    assert [c[1] for c in stub.calls] == [37, 32, 40, 40, 20]


@pytest.mark.parametrize("bad,exc", [
    (np.zeros((4, 16), np.int16), ValueError),
    (np.zeros((4, 16, 3), np.int16), ValueError),
    (np.zeros((4, 16, 2), np.float32), TypeError),
    (np.zeros((4, 16, 2, 1), np.int16), ValueError),
])
def test_push_batch_refuses_other_representations(sc16_stream, bad, exc):
    s, stub = sc16_stream
    with pytest.raises(exc):
        s.push_batch(bad)
    assert stub.calls == []


def test_push_batch_shapes_and_strides(sc16_stream):
    s, stub = sc16_stream
    s.push_batch(np.zeros((3, 16, 2), np.int16))
    assert stub.calls[-1][1:4] == (3, 16, 16)
    torch = pytest.importorskip("torch")
    big = torch.zeros((3, 24, 2), dtype=torch.int16)
    s.push_batch(big[:, :16])  # captures 24 items apart
    assert stub.calls[-1][1:4] == (3, 16, 24)
    s.push_batch(big[::2, :16])
    assert stub.calls[-1][1:4] == (2, 16, 48)
    s.push_batch(torch.zeros((3, 2, 16), dtype=torch.int16).transpose(1, 2))  # I and Q not adjacent: made contiguous
    assert stub.calls[-1][1:4] == (3, 16, 16)
    for bad, exc in ((torch.zeros((3, 16), dtype=torch.int16), ValueError), (torch.zeros((3, 16, 2)), TypeError)):
        n = len(stub.calls)
        with pytest.raises(exc):
            s.push_batch(bad)
        assert len(stub.calls) == n


def test_push_takes_cpu_tensors(sc16_stream):
    torch = pytest.importorskip("torch")
    s, stub = sc16_stream
    assert s.push(torch.zeros((21, 2), dtype=torch.int16)) == (21, False)
    with pytest.raises(TypeError):
        s.push(torch.zeros((21, 2), dtype=torch.float32))
    with pytest.raises(ValueError):
        s.push(torch.zeros(42, dtype=torch.int16))
    assert [c[1] for c in stub.calls] == [21]


def test_create_rejects_unknown_input_kinds():
    p = _cabi.Params()
    L = _cabi.lib()
    L.nfc_default_params(ctypes.byref(p))
    h = ctypes.c_void_p()
    for kind in (-1, 5, 99):
        p.input_kind = kind
        assert L.nfc_stream_create(ctypes.byref(p), ctypes.byref(h)) == -1
        assert "input_kind" in _cabi.last_error()
        assert not h.value
