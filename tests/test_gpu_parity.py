"""Parity of the CUDA path (through the C ABI) with the oracle and the reference-derived fixtures.
Bit-exact on events, symbols and frames; the float envelope is compared where it is materialised."""
import json

import numpy as np
import pytest

from oracle import oracle
from tests import helpers as H
from usrp_nfc_b200 import _cabi, synth

pytestmark = pytest.mark.gpu

CAPTURES = [
    ("surrogate_classic1k", 2e6, dict(hi_val=1.09)),
    ("surrogate_ultralight", 2e6, dict(hi_val=1.09)),
    ("rate_1356", 13.56e6, dict(hi_val=1.09, av_window=13560, max_len=339)),
    ("rate_2000", 20e6, dict(hi_val=1.09, av_window=20000, max_len=500)),
]


def gpu_decode(x, rate, chunk=None, kind=_cabi.IN_ENVELOPE_F32, tuning=None, outputs=_cabi.OUT_ALL, **kw):
    s = _cabi.Stream(rate, input_kind=kind, outputs=outputs, **kw)
    if tuning:
        s.set_tuning(**tuning)
    n = len(x)
    off = 0
    step = chunk or max(n, 1)
    while off < n:
        used, _ = s.push(x[off: off + step])
        off += used
        assert used > 0
    ev, sym = s.drain_events(), s.drain_symbols()
    fr, bits = s.drain_frames()
    return dict(events=ev, symbols=sym, frames=fr, frame_bits=bits, stream=s)


def check_against_oracle(got, want):
    H.assert_events_equal(got["events"], want["events"])
    H.assert_symbols_equal(got["symbols"], want["symbols"])
    assert len(got["frames"]) == len(want["frames"])
    for f in ("pos", "nbits", "type"):
        assert np.array_equal(got["frames"][f], want["frames"][f]), f
    for a, b in zip(got["frame_bits"], want["frame_bits"]):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("name,rate,kw", CAPTURES)
@pytest.mark.parametrize("chunk", [None, 8192])
def test_capture_matches_reference(name, rate, kw, chunk):
    case = H.load_case(name)
    got = gpu_decode(H.case_input(case), rate, chunk=chunk, **kw)
    H.assert_events_equal(got["events"], case["ev"])
    H.assert_symbols_equal(got["symbols"], case["sym"])
    H.assert_frames_equal(got["frames"], got["frame_bits"], case)
    st, ring, _ = got["stream"].state()
    assert st.ss == float(case["state_ss"])
    assert (st.cur_state, st.dur, st.last_bit, st.index) == tuple(
        int(case["state_" + k]) for k in ("cur_state", "dur", "last_bit", "index"))
    assert np.array_equal(ring.astype(np.float64), case["state_ring"])
    assert not st.serial_mode


@pytest.mark.parametrize("name,rate,kw", CAPTURES[:3])
def test_capture_from_pcm_on_device_envelope(name, rate, kw):
    """int16 PCM in, normalise + square on the device (decoder.py:25-28 chain)."""
    case = H.load_case(name)
    got = gpu_decode(case["pcm"], rate, kind=_cabi.IN_PCM_S16, **kw)
    H.assert_events_equal(got["events"], case["ev"])
    H.assert_frames_equal(got["frames"], got["frame_bits"], case)
    real = gpu_decode(synth.pcm_to_float(case["pcm"]), rate, kind=_cabi.IN_REAL_F32, **kw)
    H.assert_events_equal(real["events"], case["ev"])
    # the float envelope itself (north star: 1e-5 relative; here it is bit-identical by construction)
    _, ring, _ = real["stream"].state()
    assert np.array_equal(ring.astype(np.float64), case["state_ring"])


@pytest.mark.parametrize("name,rate,kw", CAPTURES[:2])
def test_sequential_kernel_matches_reference(name, rate, kw):
    case = H.load_case(name)
    got = gpu_decode(H.case_input(case), rate, tuning=dict(force_serial=True), **kw)
    H.assert_events_equal(got["events"], case["ev"])
    H.assert_frames_equal(got["frames"], got["frame_bits"], case)
    assert got["stream"].stats()["serial_segments"] > 0


@pytest.mark.parametrize("seg,halo", [(8192, 2048), (16384, 16384), (65536, 32768)])
def test_segment_seams_and_repairs(seg, halo):
    """Small segments and short halos force speculative starts that do not converge: the seam
    check must catch them and the repair must restore the exact stream."""
    case = H.load_case("surrogate_classic1k")
    got = gpu_decode(H.case_input(case), 2e6, tuning=dict(seg_len=seg, halo=halo), hi_val=1.09)
    H.assert_events_equal(got["events"], case["ev"])
    H.assert_symbols_equal(got["symbols"], case["sym"])
    H.assert_frames_equal(got["frames"], got["frame_bits"], case)
    st = got["stream"].stats()
    assert st["segments"] > 4
    print("segments %d, seam mismatches repaired %d" % (st["segments"], st["seam_mismatches"]))


def test_slabs_and_chunked_pushes_agree():
    case = H.load_case("surrogate_classic1k")
    x = H.case_input(case)
    got = gpu_decode(x, 2e6, chunk=100003, tuning=dict(slab_len=30011, seg_len=8192, halo=4096), hi_val=1.09)
    H.assert_events_equal(got["events"], case["ev"])
    H.assert_frames_equal(got["frames"], got["frame_bits"], case)


def test_slicer_known_answers_small_windows():
    z = H.load_case("slicer_kat")
    meta = json.loads(bytes(z["meta"]).decode())
    for ci, m in enumerate(meta):
        x = z["x%d" % ci]
        s = _cabi.Stream(2e6, m["lo"], m["hi"], m["L"], m["mx"], outputs=_cabi.OUT_EVENTS | _cabi.OUT_DROPPED_EVENTS)
        off, k, evs, nb = 0, 0, [], []
        while off < x.size:
            n = m["chunks"][k % len(m["chunks"])]
            k += 1
            used, cb = s.push(x[off: off + n])
            if cb:
                ev = s.drain_events()
                evs.append(ev)
                nb.append(len(ev))
            off += used
        ev = np.concatenate(evs) if evs else np.zeros(0, _cabi.EVENT_DTYPE)
        assert nb == z["nb%d" % ci].tolist(), "case %d: per-callback batch sizes" % ci
        got = np.stack([ev["v"], ev["d"], ev["type"]], 1).astype(np.int32) if len(ev) else np.zeros((0, 3), np.int32)
        assert np.array_equal(got, z["ev%d" % ci]), "case %d: events" % ci
        st, ring, _ = s.state()
        assert bool(st.stable) == m["stable"]
        if m["stable"]:
            assert st.ss == m["ss"] or (np.isnan(st.ss) and np.isnan(m["ss"])), "case %d: ss" % ci
            assert (st.cur_state, st.dur, st.last_bit, st.index) == (m["cur_state"], m["dur"], m["last_bit"], m["index"]), ci
            assert np.array_equal(ring.astype(np.float64), z["ring%d" % ci], equal_nan=True), "case %d: ring" % ci


@pytest.mark.parametrize("L,mx", [(256, 7), (300, 50), (1024, 50), (1000, 33), (2002, 50), (4096, 13)])
def test_parallel_kernel_small_windows_and_corner_cases(L, mx):
    """Windows at the tile-size boundaries, windows that are not a multiple of 4 (scalar kernel),
    long pauses (timeouts inside a LOW run) and spikes right after a pause (hysteresis)."""
    rng = np.random.default_rng(L * 131 + mx)
    n = 60000
    x = (0.25 * (1 + 0.01 * rng.standard_normal(n))).astype(np.float32)
    i = L + 10
    while i < n - 4 * mx - 10:
        kind = rng.integers(0, 4)
        ln = int(rng.choice([1, 2, mx - 1, mx, mx + 1, 2 * mx, 2 * mx + 1, 3 * mx + 1, 6]))
        if kind == 0:
            x[i:i + ln] = 1e-4
            i += ln
            if rng.random() < 0.7:
                k = int(rng.integers(0, mx + 4))
                x[i + k: i + k + int(rng.integers(1, 4))] = 0.4
        elif kind == 1:
            x[i:i + ln] = 0.3 * (1 + 0.01 * rng.standard_normal(ln))
            i += ln
        elif kind == 2:
            x[i:i + ln] = 0.2725 * (1 + 0.002 * rng.standard_normal(ln))  # hovering around hi = 1.09
            i += ln
        i += int(rng.integers(1, 4 * mx))
    want = oracle.decode_capture(x, 2e6, hi_val=1.09, av_window=L, max_len=mx)
    got = gpu_decode(x, 2e6, hi_val=1.09, av_window=L, max_len=mx, tuning=dict(seg_len=8192, halo=4096))
    check_against_oracle(got, want)
    assert not got["stream"].state()[0].serial_mode


def test_inexact_sums_fall_back_to_sequential_kernel():
    """Samples spanning 40 binades: double sums round, order matters, only the sequential recurrence
    reproduces the reference.  The stream must notice and switch."""
    rng = np.random.default_rng(9)
    n = 20000
    x = (np.abs(rng.standard_normal(n)) * 10.0 ** rng.integers(-6, 6, n)).astype(np.float32)
    want = oracle.decode_capture(x, 2e6, av_window=512, max_len=20)
    got = gpu_decode(x, 2e6, av_window=512, max_len=20)
    check_against_oracle(got, want)
    assert got["stream"].state()[0].serial_mode


def test_zeros_and_negative_input():
    x = np.zeros(5000, np.float32)
    x[3000:] = 0.25
    x[4000:4010] = -1.0
    want = oracle.decode_capture(x, 2e6, av_window=256, max_len=10)
    got = gpu_decode(x, 2e6, av_window=256, max_len=10)
    check_against_oracle(got, want)


def test_empty_and_tiny_pushes():
    s = _cabi.Stream(2e6)
    assert s.push(np.zeros(0, np.float32)) == (0, False)
    assert s.push(np.ones(1999, np.float32)) == (1999, False)
    assert s.push(np.ones(10, np.float32)) == (1, False)
    assert s.push(np.zeros(0, np.float32)) == (0, True)
    assert len(s.drain_events()) == 0
    assert s.push(np.ones(3, np.float32)) == (3, True)


def test_state_roundtrip_between_handles():
    case = H.load_case("surrogate_classic1k")
    x = H.case_input(case)
    cut = 201234
    a = _cabi.Stream(2e6, hi_val=1.09)
    a.push_all(x[:cut])
    st, ring, pend = a.state()
    b = _cabi.Stream(2e6, hi_val=1.09)
    b.set_state(st, ring, pend)
    b.push_all(x[cut:])
    ev = np.concatenate([a.drain_events(), b.drain_events()])
    H.assert_events_equal(ev, case["ev"])
    fa, ba = a.drain_frames()
    fb, bb = b.drain_frames()
    H.assert_frames_equal(np.concatenate([fa, fb]), ba + bb, case)


def test_reader_only_and_tag_only():
    case = H.load_case("surrogate_ultralight")
    x = H.case_input(case)
    for reader, tag, keep in ((True, False, 1), (False, True, 0)):
        got = gpu_decode(x, 2e6, hi_val=1.09, reader=reader, tag=tag)
        want = case["sym"][case["sym"]["type"] == keep]
        H.assert_symbols_equal(got["symbols"], want)


def test_device_resident_input_torch():
    import torch
    case = H.load_case("rate_1356")
    x = torch.from_numpy(H.case_input(case)).cuda()
    got = gpu_decode(x, 13.56e6, hi_val=1.09, av_window=13560, max_len=339)
    H.assert_events_equal(got["events"], case["ev"])
    got2 = gpu_decode(x[3:], 13.56e6, hi_val=1.09, av_window=13560, max_len=339)  # misaligned device pointer
    want = oracle.decode_capture(H.case_input(case)[3:], 13.56e6, hi_val=1.09, av_window=13560, max_len=339)
    check_against_oracle(got2, want)


@pytest.mark.parametrize("rate,n_sessions", [(13.56e6, 3), (2e6, 6)])
def test_large_synthetic_stream(rate, n_sessions):
    p = synth.rate_params(rate)
    frames = synth.load_sessions()["classic1k"]
    pcm = synth.capture(frames, rate, 4242, channel=synth.Channel(pause=0.03, tag_high=1.07, fade=0.08),
                        av_window=p["av_window"], sessions=n_sessions)
    x = synth.envelope(synth.pcm_to_float(pcm))
    want = oracle.decode_capture(x, rate, hi_val=1.09, **p)
    got = gpu_decode(x, rate, hi_val=1.09, **p)
    check_against_oracle(got, want)
    assert len(want["frames"]) >= 200 * n_sessions
    print("samples %d frames %d stats %s" % (x.size, len(want["frames"]), got["stream"].stats()))


@pytest.mark.parametrize("n,seg_len,super_slab,slab_len", [(48_000_000, 0, 1, 1 << 23), (20_000_000, 1_200_000, 1, 1 << 23),
                                                            (20_000_000, 1_200_000, 2, 1 << 23), (20_000_000, 1_200_000, 4, 1 << 21)])
def test_bench_workload_matches_oracle(n, seg_len, super_slab, slab_len, monkeypatch):
    """The bench.py traffic (dense frames, 5 % fade: many samples close to the HIGH threshold, repeated tiles, exact-path
    tiles, seam repairs) rendered on the device, decoded by the streaming kernel and by the oracle.  super_slab = 2: the
    slicer runs over two slabs per launch, the second slab's transitions come from the bitmap it left; super_slab = 4 with
    ten slabs: launches over 4 + 3 + 3 slabs."""
    import torch
    import bench
    monkeypatch.setenv("NFC_SUPER_SLAB", str(super_slab))
    rate = 13.56e6
    codes, lens, p = bench.build_schedule(rate, 2024)
    x = torch.empty(n, dtype=torch.float32, device="cuda")
    _cabi.synth_render(x, codes, lens, carrier=0.5, pause=0.015, tag_high=1.07, noise=0.003, fade=0.05,
                       fade_period=round(rate * 0.02), seed=7, as_envelope=True, device=0, first_index=123456789)
    torch.cuda.synchronize()
    s = _cabi.Stream(rate, hi_val=1.09, outputs=_cabi.OUT_ALL, **p)
    if seg_len:
        s.set_tuning(seg_len=seg_len, halo=4 * p["av_window"], slab_len=slab_len)
    s.push_all(x)
    got = dict(events=s.drain_events(), symbols=s.drain_symbols())
    got["frames"], got["frame_bits"] = s.drain_frames()
    want = oracle.decode_capture(x.cpu().numpy(), rate, hi_val=1.09, **p)
    check_against_oracle(got, want)
    st = s.stats()
    assert st["fast_tiles"] > 0.9 * (n / 4096) * (0.5 if seg_len else 1)
    print("stats", st)


@pytest.mark.parametrize("name,rate,kw", [CAPTURES[1], CAPTURES[2]])
def test_iq_input_envelope_on_device(name, rate, kw):
    """Complex baseband input (usrp_src.py:31 complex_to_mag_squared): the envelope RN32(RN32(re^2) + RN32(im^2)) is formed on
    the device; the oracle gets the same envelope computed in float32 on the host."""
    case = H.load_case(name)
    amp = synth.pcm_to_float(case["pcm"])
    rng = np.random.default_rng(11)
    phase = rng.uniform(0, 2 * np.pi, amp.size).astype(np.float32)
    iq = np.empty((amp.size, 2), dtype=np.float32)
    iq[:, 0] = amp * np.cos(phase)
    iq[:, 1] = amp * np.sin(phase)
    env = (iq[:, 0] * iq[:, 0]).astype(np.float32) + (iq[:, 1] * iq[:, 1]).astype(np.float32)
    want = oracle.decode_capture(env.astype(np.float32), rate, **kw)
    got = gpu_decode(iq.view(np.complex64).reshape(-1), rate, kind=_cabi.IN_IQ_F32, **kw)
    check_against_oracle(got, want)
    assert len(want["frames"]) > 0


def test_sampled_window_parity_at_scale():
    """BASELINE-sized streams cannot be decoded by the oracle in test time.  Size-independent check (SURVEY.md 8(d)): decode
    1.5e9 samples on the GPU, then let the oracle decode a few windows cold-started 24 av_windows early (its state converges to
    the stream's long before the window begins) and compare every frame closing inside the windows."""
    import torch
    import bench
    rate = 13.56e6
    codes, lens, p = bench.build_schedule(rate, 2024)
    L = p["av_window"]
    n = 1_500_000_000
    x = torch.empty(n, dtype=torch.float32, device="cuda")
    _cabi.synth_render(x, codes, lens, carrier=0.5, pause=0.015, tag_high=1.07, noise=0.003, fade=0.05,
                       fade_period=round(rate * 0.02), seed=99, as_envelope=True, device=0, first_index=0)
    torch.cuda.synchronize()
    s = _cabi.Stream(rate, hi_val=1.09, outputs=_cabi.OUT_FRAMES, **p)
    s.set_tuning(slab_len=1 << 30)
    s.push_all(x)
    fr, bits = s.drain_frames_flat()
    assert len(fr) > 100000
    rng = np.random.default_rng(1)
    halo, wlen = 24 * L, 12_000_000
    for w0 in sorted(rng.integers(halo, n - wlen, 3).tolist()) + [1 << 30]:  # one window across the slab boundary
        w0 = int(w0)
        w1 = w0 + wlen
        want = oracle.decode_capture(x[w0 - halo - L: w1].cpu().numpy(), rate, hi_val=1.09, **p)
        base = w0 - halo - L
        wpos = want["frames"]["pos"] + base
        wsel = np.nonzero((wpos >= w0 + 100000) & (wpos < w1))[0]
        gsel = np.nonzero((fr["pos"] >= w0 + 100000) & (fr["pos"] < w1))[0]
        assert len(wsel) == len(gsel) and len(wsel) > 100, (w0, len(wsel), len(gsel))
        assert np.array_equal(wpos[wsel], fr["pos"][gsel])
        assert np.array_equal(want["frames"]["type"][wsel], fr["type"][gsel])
        assert np.array_equal(want["frames"]["nbits"][wsel], fr["nbits"][gsel])
        for i, j in zip(wsel[:: max(1, len(wsel) // 200)], gsel[:: max(1, len(gsel) // 200)]):
            g = fr[j]
            assert np.array_equal(want["frame_bits"][i], bits[g["bit_off"]: g["bit_off"] + g["nbits"]])


def _corner_stream(L, mx, n, seed):
    """Carrier with long pauses (timeouts inside a LOW run), spikes right after a pause (hysteresis), stretches hovering
    around the HIGH threshold (samples inside every guard band), strong steps of the level."""
    rng = np.random.default_rng(seed)
    x = (0.25 * (1 + 0.01 * rng.standard_normal(n))).astype(np.float32)
    i = L + 10
    while i < n - 4 * mx - 10:
        kind = rng.integers(0, 5)
        ln = int(rng.choice([1, 2, mx - 1, mx, mx + 1, 2 * mx, 2 * mx + 1, 3 * mx + 1, 6, 700]))
        ln = min(ln, n - i - 1)
        if kind == 0:
            x[i:i + ln] = 1e-4
            i += ln
            if rng.random() < 0.7:
                k = int(rng.integers(0, mx + 4))
                x[i + k: i + k + int(rng.integers(1, 4))] = 0.4
        elif kind == 1:
            x[i:i + ln] = 0.3 * (1 + 0.01 * rng.standard_normal(ln))
            i += ln
        elif kind == 2:
            x[i:i + ln] = 0.2725 * (1 + 0.002 * rng.standard_normal(ln))  # hovering around hi = 1.09
            i += ln
        elif kind == 3 and rng.random() < 0.05:
            x[i:] *= np.float32(rng.choice([0.7, 1.4]))  # the level steps: guesses are off, sums do not fit the fixed point
        i += int(rng.integers(1, 6 * mx))
    return x


@pytest.mark.parametrize("L,mx,tuning", [(8192, 50, None), (13560, 339, dict(seg_len=131072, halo=4 * 13560)),
                                         (8196, 7, dict(seg_len=65536, halo=32784)), (20000, 500, None)])
def test_streaming_kernel_corner_cases(L, mx, tuning):
    n = 700000
    x = _corner_stream(L, mx, n, L * 7 + mx)
    want = oracle.decode_capture(x, 13.56e6, hi_val=1.09, av_window=L, max_len=mx)
    got = gpu_decode(x, 13.56e6, hi_val=1.09, av_window=L, max_len=mx, tuning=tuning)
    check_against_oracle(got, want)
    st = got["stream"].stats()
    assert not got["stream"].state()[0].serial_mode
    assert st["fast_tiles"] > 0 and st["exact_tiles"] > 0
    print("stats", st)


@pytest.mark.parametrize("L,streaming", [(52000, True), (51456, True), (51998, False)])
def test_longest_parallel_windows(L, streaming):
    """The top of the parallel window range, several segments each: a multiple of 4 up to 52000 takes the streaming kernel
    (at 52000 the ring, the staging tile and the kernel's static scratch fill one CTA's shared memory), any other window
    the first-generation kernel."""
    mx = 339
    # pauses at 1e-3 rather than 1e-4: the first-generation kernel starts a segment from the raw previous L samples, and at
    # these windows its sums are exact only while those span at most 28 - 16 - 1 = 11 binades (else the sequential kernel)
    x = np.maximum(_corner_stream(L, mx, 1_500_000, L + mx), np.float32(1e-3))
    want = oracle.decode_capture(x, 13.56e6, hi_val=1.09, av_window=L, max_len=mx)
    got = gpu_decode(x, 13.56e6, hi_val=1.09, av_window=L, max_len=mx, tuning=dict(seg_len=262144, halo=4 * L))
    check_against_oracle(got, want)
    st = got["stream"].stats()
    assert not got["stream"].state()[0].serial_mode
    assert st["segments"] >= 3
    if streaming:
        assert st["slicer_kernel_launches"] > 0
    else:
        assert st["slicer_kernel_launches"] == 0 and st["serial_segments"] == 0


def test_streaming_kernel_degenerate_inputs():
    L, mx = 8192, 50
    # silence (ss == 0), then a carrier, negative samples, back to silence
    x = np.zeros(150000, np.float32)
    x[40000:100000] = 0.25
    x[60000:60010] = -1.0
    x[70000:70003] = 0.0
    want = oracle.decode_capture(x, 13.56e6, av_window=L, max_len=mx)
    got = gpu_decode(x, 13.56e6, av_window=L, max_len=mx)
    check_against_oracle(got, want)
    # thresholds the streaming path does not take (lo_val = 0, hi_val < lo_val): every tile through the exact path
    rng = np.random.default_rng(3)
    y = (0.25 * (1 + 0.05 * rng.standard_normal(120000))).astype(np.float32)
    y[50000:50040] = 1e-5
    for lo, hi in ((0.0, 1.05), (1.2, 1.1), (0.98, 1.02)):
        want = oracle.decode_capture(y, 13.56e6, lo_val=lo, hi_val=hi, av_window=L, max_len=mx)
        got = gpu_decode(y, 13.56e6, lo_val=lo, hi_val=hi, av_window=L, max_len=mx)
        check_against_oracle(got, want)


def test_streaming_kernel_falls_back_on_inexact_or_insane_samples():
    L, mx = 8192, 50
    rng = np.random.default_rng(9)
    n = 100000
    x = (np.abs(rng.standard_normal(n)) * 10.0 ** rng.integers(-6, 6, n)).astype(np.float32)  # 40 binades: sums round
    want = oracle.decode_capture(x, 13.56e6, av_window=L, max_len=mx)
    got = gpu_decode(x, 13.56e6, av_window=L, max_len=mx)
    check_against_oracle(got, want)
    assert got["stream"].state()[0].serial_mode
    z = (0.25 * (1 + 0.01 * rng.standard_normal(n))).astype(np.float32)
    z[50000] = np.inf
    z[60000:60004] = 1e-4
    want = oracle.decode_capture(z, 13.56e6, av_window=L, max_len=mx)
    got = gpu_decode(z, 13.56e6, av_window=L, max_len=mx)
    check_against_oracle(got, want)


def _empty_closings(symbols):
    """PacketProcessor.append_bit (packets.py:67-79) on a symbol list [(type, val, ...)]: how many frames close empty."""
    started, cur, empty = [False, False], [0, 0], 0
    for row in symbols:
        t, v = int(row[0]), int(row[1])
        if v != 0 and v != 1:
            if started[t]:
                empty += cur[t] == 0
                started[t], cur[t] = False, 0
        elif not started[t] and v == (1 if t == 0 else 0):  # PacketType.start_bit (packets.py:24-28)
            started[t] = True
        else:
            cur[t] += 1
    return empty


def test_decoder_kats_through_the_device_line_code():
    """The 40 known-answer event streams of the reference's decoders (tests/golden/decoder_kat.npz: miller_decoder,
    manchester_decoder and PacketProcessor driven on adversarial event lists) through nfc_stream_push_events -- the
    background.append boundary (background.py:27-29): symbols and frames of the device's line-code kernels, fed whole and in
    two parts (decoder and framer state carry over)."""
    z = H.load_case("decoder_kat")
    empties = 0
    for ci in range(40):
        evs = z["ev%d" % ci]
        ev = np.zeros(len(evs), dtype=_cabi.EVENT_DTYPE)
        ev["v"], ev["d"], ev["type"], ev["pos"] = evs[:, 0], evs[:, 1], evs[:, 2], np.arange(len(evs)) * 3 + 7
        for cut in (len(ev), len(ev) // 3):
            s = _cabi.Stream(2e6, outputs=_cabi.OUT_SYMBOLS | _cabi.OUT_FRAMES)
            s.push_events(ev[:cut])
            if cut < len(ev):
                s.push_events(ev[cut:])
            sym = s.drain_symbols()
            fr, bits = s.drain_frames()
            n_empty = s.stats()["empty_frames"]
            s.close()
            want = z["sym%d" % ci]
            # frames closed without a bit (packets.py:67-79: started, then a symbol that is no bit) are counted, not handed out
            assert n_empty == _empty_closings(want), (ci, cut)
            empties += n_empty
            assert len(sym) == len(want), (ci, cut)
            assert np.array_equal(sym["type"], want[:, 0]) and np.array_equal(sym["val"], want[:, 1]), (ci, cut)
            assert np.array_equal(fr["type"], z["ftype%d" % ci]) and np.array_equal(fr["nbits"], z["flen%d" % ci]), (ci, cut)
            got_bits = np.concatenate(bits) if len(bits) else np.zeros(0, dtype=np.uint8)
            assert np.array_equal(got_bits, z["fbits%d" % ci]), (ci, cut)
            # symbols are reported at the positions of the events that produced them
            assert set(sym["pos"].tolist()) <= set(ev["pos"].tolist())
    assert empties > 0  # the known answers do hold such closings


def test_push_events_rejects_what_transition_sink_cannot_emit():
    s = _cabi.Stream(2e6, outputs=_cabi.OUT_SYMBOLS)
    ev = np.zeros(3, dtype=_cabi.EVENT_DTYPE)
    ev["d"], ev["pos"] = [5, 51, 5], [0, 1, 2]
    with pytest.raises(_cabi.NfcError):
        s.push_events(ev)  # d beyond max_len
    ev["d"], ev["pos"] = [5, 5, 5], [5, 4, 6]
    with pytest.raises(_cabi.NfcError):
        s.push_events(ev)  # positions do not ascend
    s.close()
