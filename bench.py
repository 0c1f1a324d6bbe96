#!/usr/bin/env python
"""bench.py -- decoded Msamples/s of the usrp_nfc sample-rate path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores
    python bench.py --gpus 1 ... --dump-outputs DIR          # also write the last timed step's frames to DIR/*.npy

A step = one pass of the hot path (envelope -> slicer -> Manchester/Miller -> frames) over one synthetic
ISO 14443A capture that is already resident in HBM.  N=1 workload: BASELINE.json configs[2], 1e10 samples at
13.56 MS/s (av_window=13560, max_len=339, hi_val=1.09; SURVEY.md 8(d)).  N>1: weak scaling, every rank
decodes its own 1e10-sample time shard of one endless capture (no data-path collective; frame counts are
gathered).  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RATE = 13.56e6  # BASELINE.json configs[2]; --rate 20e6 gives configs[4] (time-sharded 20 MS/s capture)
HI_VAL = 1.09
# the reference's own Python loop (transition_sink.work_stable + decoders), measured per core in the build container where
# /root/reference can be imported (BASELINE.md 2); the GPU box has no /root/reference, so the arm below times the C port
PY_REF_NOTE = "the reference's Python 2 loop does 2.3-3.6 Msamples/s per core (BASELINE.md 2, SURVEY.md 6: 0.91 published); kind 'port' is its C restatement, ~60x faster per core"


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def build_schedule(rate, seed):
    """Pulse schedule of one period of dense traffic: 12 Classic + 4 Ultralight sessions with idle gaps."""
    from usrp_nfc_b200 import synth
    rng = np.random.default_rng(seed)
    sess = synth.load_sessions()
    p = synth.rate_params(rate)
    codes, lens = [], []
    order = ["classic1k"] * 3 + ["ultralight"]
    for i in range(16):
        lead = float(rng.uniform(1000.0, 5000.0))
        c, l = synth.schedule(sess[order[i % 4]], rate, rng, lead_us=lead, av_window=p["av_window"])
        codes.append(c)
        lens.append(l)
    return np.concatenate(codes), np.concatenate(lens), p


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs."""

    def __init__(self, index):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.rows, self._stop_evt, self.proc, self.first = index, [], threading.Event(), None, threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))
                self.first.set()
                if self._stop_evt.is_set():
                    break
        except Exception:
            pass
        self.first.set()

    def wait_running(self, timeout=3.0):
        """nvidia-smi needs ~0.1 s to start: the step is shorter than that, so the caller waits for the first row."""
        self.first.wait(timeout)

    def stop(self, t_load=None, t0=None, t1=None):
        """Rows inside the timed region [t0, t1] if there are any, else the rows since the load began (t_load: the warm-up steps
        in front of the timed region run the same work); `window` says which."""
        self._stop_evt.set()
        if self.proc:
            self.proc.terminate()
        rows = list(self.rows)
        timed = [r for t, r in rows if t0 is not None and t0 <= t <= t1]
        load = [r for t, r in rows if t_load is not None and t_load <= t <= t1]
        use, window = (timed, "timed region") if timed else ((load, "warm-up + timed region") if load else ([r for _, r in rows], "whole run"))
        sm, mx, reasons = [], 0, set()
        for r in use:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "window": window, "samples_timed": len(timed)}


def same_frames(ra, rb):
    """Two decodes of one capture: identical frame records (closing position, type, length) and identical frame bits."""
    (fa, a0, a1), (fb, b0, b1) = ra, rb
    if len(fa) != len(fb) or len(a0) != len(b0) or len(a1) != len(b1):
        return False
    return bool(np.array_equal(fa["pos"], fb["pos"]) and np.array_equal(fa["type"], fb["type"]) and
                np.array_equal(fa["nbits"], fb["nbits"]) and np.array_equal(a0, b0) and np.array_equal(a1, b1))


DUMP_FRAMES = 1 << 21  # --dump-outputs: frame records written whole up to this many, else a seeded sample of this many
DUMP_BITS = 1 << 21    # frame bits of each direction, likewise


def sample_index(n, k, seed):
    """Sorted indices of a fixed, seeded sample of k of n items (all n when n <= k)."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def dump_outputs(out_dir, frames):
    """What a caller of the timed decode receives, as out_dir/<name>.npy: the frame records (closing position in float64, type
    and length in float32) and the tag -> reader and reader -> tag frame bits (float32), each capped as above: at most 48 MiB.
    frames: (records, tag bits, reader bits) as view_frames returns them.  Two builds that decode alike write identical files."""
    fr, b0, b1 = frames
    i = sample_index(len(fr), DUMP_FRAMES, 1)
    out = {"frame_pos": fr["pos"][i].astype(np.float64), "frame_type": fr["type"][i].astype(np.float32),
           "frame_nbits": fr["nbits"][i].astype(np.float32),
           "bits_tag": b0[sample_index(len(b0), DUMP_BITS, 2)].astype(np.float32),
           "bits_reader": b1[sample_index(len(b1), DUMP_BITS, 3)].astype(np.float32)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def oracle_windows(x, frames, params, k, wlen=6_000_000):
    """k random windows of the device-resident capture x against the oracle (test infrastructure: the checker, not the
    thing measured).  frames: (records, tag bits, reader bits) of the CUDA decode of x as view_frames returns them."""
    from oracle import oracle
    fr, b0, b1 = frames
    L = params["av_window"]
    n = int(x.numel())
    halo = 24 * L
    rng = np.random.default_rng(7)
    starts = sorted(int(v) for v in rng.integers(halo + L, max(halo + L + 1, n - wlen), k))
    if n > (1 << 30) + wlen:
        starts[0] = (1 << 30) - wlen // 2  # one window across a slab boundary
    ok, nfr, nbits = True, 0, 0
    for w0 in starts:
        w1 = min(n, w0 + wlen)
        base = w0 - halo - L
        want = oracle.decode_capture(x[base:w1].cpu().numpy(), RATE, hi_val=HI_VAL, **params)
        wpos = want["frames"]["pos"] + base
        wsel = np.nonzero((wpos >= w0 + 100000) & (wpos < w1))[0]
        lo, hi = np.searchsorted(fr["pos"], [w0 + 100000, w1])
        g = fr[lo:hi]
        same = len(wsel) == len(g) and np.array_equal(wpos[wsel], g["pos"]) and np.array_equal(want["frames"]["type"][wsel], g["type"]) \
            and np.array_equal(want["frames"]["nbits"][wsel], g["nbits"])
        if same:
            for i, r in zip(wsel, g):
                bits = b0 if r["type"] == 0 else b1
                if not np.array_equal(want["frame_bits"][i], bits[r["bit_off"]: r["bit_off"] + r["nbits"]]):
                    same = False
                    break
                nbits += int(r["nbits"])
        ok = ok and bool(same)
        nfr += len(wsel)
    return {"windows": len(starts), "samples_each": wlen, "frames_compared": int(nfr), "frame_bits_compared": int(nbits),
            "identical": bool(ok), "starts": starts}


def cpu_baseline(x_host_pieces, params, threads):
    """The reference algorithm (oracle port, C) on the host cores: one independent piece per thread."""
    from oracle import oracle
    oracle.lib()
    res = [None] * len(x_host_pieces)

    def work(i):
        res[i] = oracle.chain_run(x_host_pieces[i], RATE, 0.1, HI_VAL, params["av_window"], params["max_len"])

    t0 = time.perf_counter()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(len(x_host_pieces))]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    n = sum(len(p) for p in x_host_pieces)
    return n / dt / 1e6, dt, res


def shm_room():
    """Free bytes in /dev/shm (a segment larger than that kills the process that touches it)."""
    try:
        st = os.statvfs("/dev/shm")
        return st.f_bavail * st.f_frsize
    except Exception:
        return 0


def chan_for(rate, args):
    """Amplitude model of SURVEY.md 8(d) at a sample rate (the fade period is 20 ms of samples)."""
    return dict(carrier=0.5, pause=0.015, tag_high=args.tag_high, noise=0.003, fade=args.fade, fade_period=round(rate * 0.02))


def step_frac(samples_per_gpu, ms, peak):
    """Whole-step fraction of the HBM roofline: 4 algorithmic bytes per sample over the step's wall time."""
    return 4.0 * samples_per_gpu / (ms * 1e-3) / 1e9 / peak if ms and ms > 0 else None


def leg_stream(torch, _cabi, rate, n, local_rank, args, peak, steps=2, warmup=2):
    """One device-resident capture of n samples at `rate` with that rate's parameters (SURVEY.md 8(d)) through one
    nfc_stream on this GPU: the N1 row (2 / 13.56 / 20 MS/s) beside the headline.  Own timing, roofline fractions, clocks."""
    codes, lens, params = build_schedule(rate, 2024)
    L = params["av_window"]
    n = int(n) - int(n) % (L * 4 // np.gcd(L, 4))
    x = torch.empty(n, dtype=torch.float32, device="cuda")
    _cabi.synth_render(x, codes, lens, seed=99, as_envelope=True, device=local_rank, first_index=0, **chan_for(rate, args))
    torch.cuda.synchronize()
    s = _cabi.Stream(rate, hi_val=HI_VAL, outputs=_cabi.OUT_FRAMES, device=local_rank, **params)
    s.set_tuning(slab_len=1 << 30)
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.wait_running()
    t_load = time.perf_counter()

    def step():
        s.reset()
        s.push_all(x)
        fr = s.view_frames()[0]
        k = len(fr)
        s.release_frames()
        return k
    for _ in range(warmup):
        step()
    s.reset_stats()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        frames = step()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    st = s.stats()
    clocks = sampler.stop(t_load, t0, t0 + wall)
    s.close()
    del x
    torch.cuda.empty_cache()
    ms = wall * 1e3 / steps
    kern = st["slicer_kernel_ms"] / steps
    return {"workload": "synthetic ISO 14443A reader+tag traffic, %.3g samples at %.2f MS/s on one GPU" % (n, rate / 1e6),
            "samp_rate": rate, **params, "hi_val": HI_VAL, "steps": steps, "warmup": warmup, "ms": ms,
            "value": n / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "frac": step_frac(n, ms, peak),
            "kernel_ms": kern, "kernel_frac": step_frac(n, kern, peak) if kern > 0 else None,
            "slicer_stage_ms": st["slicer_ms"] / steps, "device_ms": st["kernel_ms"] / steps, "frames": int(frames),
            "streaming_tiles": int(st["fast_tiles"]), "pipelined_tiles": int(st["pipe_tiles"]), "exact_tiles": int(st["exact_tiles"]),
            "tiles": {k: int(st[k]) for k in ("repeated_passes", "fixpoint_tiles", "st2_tiles", "unproven_tiles", "pipe_runs", "pipe_aborts", "segments")},
            "clocks": clocks}


def leg_batch(torch, _cabi, dist, rank, world, local_rank, args, peak, per_rank_captures, ns, rate, steps=2, warmup=2):
    """BASELINE.json configs[3] (C4): per_rank_captures independent captures per GPU (4096 over eight GPUs = 512 each), mixed
    Ultralight / Classic traffic, hi_val per capture from 1.05..1.10, decoded in one pass per GPU (nfc_stream_push_batch);
    frame records stay per rank, their counts are all-reduced.  Weak in N: value = all captures / max-over-ranks time."""
    from usrp_nfc_b200 import batch
    codes, lens, params = build_schedule(rate, 2024)
    chan = chan_for(rate, args)
    uniq = 8
    his = [1.05, 1.06, 1.07, 1.08, 1.09, 1.10]
    mine = [rank * per_rank_captures + k for k in range(per_rank_captures)]
    x2d = torch.empty((len(mine), ns), dtype=torch.float32, device="cuda")
    for u in range(uniq):
        _cabi.synth_render(x2d[u], codes, lens, seed=500 + u, as_envelope=True, device=local_rank, first_index=u * 7919 * 4096, **chan)
    for k, i in enumerate(mine):
        if k >= uniq:
            x2d[k].copy_(x2d[k % uniq])
    hv = np.array([his[i % len(his)] for i in mine], dtype=np.float64)
    torch.cuda.synchronize()
    state = {}

    def step():
        res = batch.decode_batch_onepass(x2d, rate, params, hi_vals=hv, device=local_rank, stream=state.get("s"))
        state["s"] = res["stream"]
        if res.get("per_capture") is not None:
            return sum(len(fr) for fr, _ in res["per_capture"])
        return len(res["frames"])
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.wait_running()
    t_load = time.perf_counter()
    for _ in range(warmup):
        frames = step()
    state["s"].reset_stats()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        frames = step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - t0
    st = state["s"].stats()
    clocks = sampler.stop(t_load, t0, t0 + wall) if rank == 0 else None
    t = torch.tensor([wall * 1e3 / steps, float(frames), st["slicer_kernel_ms"] / steps], dtype=torch.float64, device="cuda")
    if world > 1:
        mx, sm = t.clone(), t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms, frames, kern = float(mx[0]), int(sm[1]), float(mx[2])
    else:
        ms, frames, kern = float(t[0]), int(t[1]), float(t[2])
    state["s"].release_frames()
    state["s"].close()
    del x2d
    torch.cuda.empty_cache()
    n_rank = per_rank_captures * ns
    return {"workload": "batch of %d independent synthetic captures (%d per GPU) of %.3g samples at %.2f MS/s, mixed Ultralight / "
                        "Classic sessions, hi_val 1.05..1.10 per capture, one pass per GPU (nfc_stream_push_batch)" % (
                            per_rank_captures * world, per_rank_captures, ns, rate / 1e6),
            "samp_rate": rate, **params, "n_gpus": world, "scaling": "weak", "steps": steps, "warmup": warmup, "ms": ms,
            "value": world * n_rank / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "frac": step_frac(n_rank, ms, peak),
            "kernel_ms": kern, "kernel_frac": step_frac(n_rank, kern, peak) if kern > 0 else None, "frames": frames, "clocks": clocks}


def leg_c5(torch, _cabi, dist, rank, world, local_rank, args, peak, total, rate, piece, buf=None):
    """BASELINE.json configs[4] (C5): ONE capture of `total` samples at 20 MS/s, strong-scaled: time shards with a halo
    (sharding.plan), every rank decodes total / N samples.  The capture never exists as a whole: each rank renders its shard
    piece by piece (`piece` samples, one reused buffer: 1e11 samples are 400 GB) and pushes the piece into its stream, which
    carries the state on -- the slabbed regenerate-and-decode loop of SURVEY.md 7.7.  Rendering is not timed (the clock stops
    while a piece is rendered); seam verification (all_gather of the seam states), any repair and the gather of the frame
    offsets to rank 0 (fixed 8-byte records over NCCL) are."""
    from usrp_nfc_b200 import sharding
    codes, lens, params = build_schedule(rate, 2024)
    chan = chan_for(rate, args)
    L = params["av_window"]
    q = L * 4 // np.gcd(L, 4)
    total = int(total) - int(total) % (q * world)
    piece = int(piece) - int(piece) % q
    if buf is None or buf.numel() < piece:
        buf = torch.empty(piece, dtype=torch.float32, device="cuda")
    s = _cabi.Stream(rate, hi_val=HI_VAL, outputs=_cabi.OUT_FRAMES, device=local_rank, **params)
    clock = {"on": None, "sum": 0.0, "render": 0.0, "calls": 0}
    n_fetches = 1 + -(-(total // world) // piece)  # per pass and rank: the halo (rank 0: a barrier in its place), then the pieces

    def fetch(a, b):
        torch.cuda.synchronize()  # the decode of the piece before is still on the device: that is decode time, not rendering
        t = time.perf_counter()
        if clock["on"] is not None:
            clock["sum"] += t - clock["on"]
        _cabi.synth_render(buf[: b - a], codes, lens, seed=99, as_envelope=True, device=local_rank, first_index=a, **chan)
        torch.cuda.synchronize()
        clock["calls"] += 1
        if world > 1 and clock["calls"] <= n_fetches:  # (a shard that is decoded again after a seam mismatch fetches alone)
            dist.barrier()  # every rank has rendered: nobody's decode clock runs while it waits for another rank's rendering
        clock["on"] = time.perf_counter()
        clock["render"] += clock["on"] - t
        return buf[: b - a]
    s.set_tuning(slab_len=1 << 30)
    # warm-up: the whole pass once, untimed (device buffers and the host's output vectors reach their sizes)
    gstate = {}
    shared = None
    if world > 1:
        want_recs = int(total // world * 2.5e-4) + (1 << 16)
        shared = sharding.SharedFrameIndex(s, want_recs if shm_room() > 4 * world * want_recs * 8 else 0, dist)
        if rank == 0:
            clock["calls"] += 1
            dist.barrier()  # (pairs with the other ranks' halo fetch, see below)
    res = sharding.decode_time_sharded(s, fetch, total, L, _cabi.State, dist=dist if world > 1 else None, device="cuda",
                                       halo_windows=args.halo_windows, flat="view", piece=piece)
    sharding.gather_frame_records(s, res["pos_offset"], dist if world > 1 else None, device="cuda", state=gstate, shared=shared)
    s.release_frames()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.wait_running()
    s.reset_stats()
    clock["calls"] = 0
    if world > 1 and rank == 0:
        clock["calls"] += 1
        dist.barrier()  # the other ranks fetch (render) a halo first: the barrier of that fetch
    clock.update(on=time.perf_counter(), sum=0.0, render=0.0)
    t_begin = clock["on"]
    res = sharding.decode_time_sharded(s, fetch, total, L, _cabi.State, dist=dist if world > 1 else None, device="cuda",
                                       halo_windows=args.halo_windows, flat="view", piece=piece)
    index = sharding.gather_frame_records(s, res["pos_offset"], dist if world > 1 else None, device="cuda", state=gstate, shared=shared)
    torch.cuda.synchronize()
    t_end = time.perf_counter()
    clock["sum"] += t_end - clock["on"]
    st = s.stats()
    n_frames_rank = int(res["n_frames"])
    n_index = int(len(index)) if index is not None else 0
    via = "shared memory of the node (no copy)" if (shared is not None and shared.ok) else ("NCCL gather" if world > 1 else "local")
    index = None
    s.release_frames()
    if shared is not None:
        shared.close()
    s.close()
    clocks = sampler.stop(t_begin, t_begin, t_end) if rank == 0 else None
    t = torch.tensor([clock["sum"] * 1e3, clock["render"] * 1e3, float(res["repaired"]), st["slicer_kernel_ms"]], dtype=torch.float64, device="cuda")
    if world > 1:
        mx = t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        ms, render_ms, repaired, kern = float(mx[0]), float(mx[1]), int(mx[2]), float(mx[3])
    else:
        ms, render_ms, repaired, kern = float(t[0]), float(t[1]), int(t[2]), float(t[3])
    per_gpu = total // world
    return {"workload": "ONE synthetic capture of %.3g samples at %.2f MS/s, time shards of %.3g samples with a halo of %d av_windows, "
                        "rendered and decoded in pieces of %.3g samples (400 GB never resident)" % (
                            total, rate / 1e6, per_gpu, args.halo_windows, piece),
            "samp_rate": rate, **params, "n_gpus": world, "scaling": "strong", "steps": 1, "warmup": 1,
            "ms": ms, "value": total / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "frac": step_frac(per_gpu, ms, peak),
            "kernel_ms": kern, "kernel_frac": step_frac(per_gpu, kern, peak) if kern > 0 else None,
            "render_ms_untimed": render_ms, "frames": n_index if rank == 0 else n_frames_rank,
            "frame_offsets_gathered_bytes": n_index * 8, "gathered_via": via,
            "ranks_redone": repaired, "clocks": clocks}


def leg_work_calls(torch, _cabi, local_rank, args, n=16_000_000, chunk=8192):
    """The reference's real call pattern: GNU Radio hands the sink block about 8192 items per work() call
    (transition_sink.py:37-107 runs once per call).  A 2 MS/s capture as 16-bit PCM in host memory through
    usrp_nfc_b200.decoder.decoder (the drop-in block; frames counted by an on_frame callback) in calls of `chunk` items:
    every call pushed as it comes, and with the items of successive calls coalesced (frame_sink(coalesce=))."""
    from usrp_nfc_b200.decoder import decoder
    rate = 2e6
    codes, lens, params = build_schedule(rate, 2024)
    x = torch.empty(n, dtype=torch.float32, device="cuda")
    _cabi.synth_render(x, codes, lens, seed=99, as_envelope=False, device=local_rank, first_index=0, **chan_for(rate, args))
    pcm = torch.round(x * 32767.0).to(torch.int16).cpu().numpy()
    del x
    out = {"workload": "synthetic ISO 14443A traffic, %.3g samples at 2 MS/s, int16 PCM in host memory, through the decoder block in "
                       "work() calls of %d items" % (n, chunk), "samp_rate": rate, **params, "chunk": chunk}
    for name, co in (("per_call", 0), ("coalesce_262144", 262144)):
        cnt = [0]

        def on_frame(bits, t):
            cnt[0] += 1
        d = decoder(src=pcm, samp_rate=rate, on_frame=on_frame, device=local_rank, coalesce=co, hi_val=HI_VAL, **params)
        m = n if co else n // 8  # per-call pushes are slow: a shorter stretch
        d._pcm = pcm[:m]
        t0 = time.perf_counter()
        d.run(chunk=chunk)
        dt = time.perf_counter() - t0
        d.stream().close()
        out[name] = {"samples": m, "calls": (m + chunk - 1) // chunk, "s": dt, "value": m / dt / 1e6, "unit": "Msamples/s",
                     "ms_per_call": dt * 1e3 / ((m + chunk - 1) // chunk), "frames": cnt[0], "realtime_factor": m / dt / rate}
    return out


def bench_batch(args, rank, world, local_rank, codes, lens, params, chan, dist, torch, _cabi):
    """BASELINE.json configs[3]: a batch of independent captures (hi_val varies per capture) dealt round-robin to the ranks,
    several nfc_streams per GPU in flight (usrp_nfc_b200/batch.py).  Captures are resident in HBM; a step decodes the whole batch."""
    from usrp_nfc_b200 import batch
    ns = int(args.batch_samples)
    mine = batch.rank_share(args.batch, rank, world)
    uniq = 8  # distinct renderings kept in HBM; capture i uses rendering i % uniq with its own hi_val
    pool = []
    for u in range(uniq):
        x = torch.empty(ns, dtype=torch.float32, device="cuda")
        _cabi.synth_render(x, codes, lens, seed=500 + u, as_envelope=True, device=local_rank, first_index=u * 7919 * 4096, **chan)
        pool.append(x)
    torch.cuda.synchronize()
    his = [1.05, 1.06, 1.07, 1.08, 1.09, 1.10]
    plist = [dict(hi_val=his[i % len(his)], **params) for i in mine]
    tuning = dict(seg_len=0, halo=0, slab_len=1 << 28)
    state = {}
    if args.batch_legacy:
        caps = [pool[i % uniq] for i in mine]

        def step():
            res = batch.decode_batch(caps, RATE, plist, device=local_rank, workers=args.batch_workers, tuning=tuning,
                                     blocking_wait=not args.batch_spin)
            return sum(len(fr) for fr, _ in res)
    else:
        # one pass over the rank's share (nfc_stream_push_batch): the captures side by side in HBM, one threshold per capture
        x2d = torch.empty((len(mine), ns), dtype=torch.float32, device="cuda")
        for k, i in enumerate(mine):
            x2d[k].copy_(pool[i % uniq])
        hv = np.array([his[i % len(his)] for i in mine], dtype=np.float64)
        del pool
        torch.cuda.synchronize()

        def step():
            res = batch.decode_batch_onepass(x2d, RATE, params, hi_vals=hv, device=local_rank, stream=state.get("s"))
            state["s"] = res["stream"]
            if res.get("per_capture") is not None:
                return sum(len(fr) for fr, _ in res["per_capture"])
            return len(res["frames"])

    frames = 0
    for _ in range(args.warmup):
        frames = step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        frames = step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    t = torch.tensor([wall_ms, float(frames)], dtype=torch.float64, device="cuda")
    if world > 1:
        mx = t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        wall_ms, frames = float(mx[0]), int(sm[1])
    if rank == 0:
        line = {"metric": "decoded_msamples_per_s", "value": args.batch * ns / (wall_ms * 1e-3) / 1e6, "unit": "Msamples/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall_ms, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "batch of %d independent synthetic captures of %.3g samples at %.2f MS/s, hi_val 1.05..1.10 per capture, "
                                       "round-robin over %d GPU(s), %s" % (args.batch, ns, RATE / 1e6, world,
                                                                          ("%d streams in flight per GPU (%s waits)" % (args.batch_workers, "spinning" if args.batch_spin else "blocking"))
                                                                          if args.batch_legacy else "one pass per GPU (nfc_stream_push_batch)"),
                           "samp_rate": RATE, **params},
                "frames_per_step": int(frames)}
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


_STDOUT_FD = None


def quiet_stdout():
    """Everything libraries write to stdout while the bench runs (NCCL prints its version there) goes to stderr; the one JSON
    line is written to the real stdout by emit()."""
    global _STDOUT_FD
    if _STDOUT_FD is None:
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    if _STDOUT_FD is not None:
        os.dup2(_STDOUT_FD, 1)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--samples", type=float, default=1e10, help="samples per GPU per step")
    ap.add_argument("--e2e-samples", type=float, default=float(1 << 30))
    ap.add_argument("--cpu-piece", type=float, default=1.5e8, help="CPU-baseline samples per host thread")
    ap.add_argument("--slab", type=float, default=float(1 << 30))
    ap.add_argument("--seg-len", type=int, default=0)
    ap.add_argument("--halo", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-selfcheck", action="store_true", help="skip the untimed full-size self-check (second decode with another segmentation)")
    ap.add_argument("--rate", type=float, default=RATE, help="13.56e6 (configs[2]) or 20e6 (configs[4])")
    ap.add_argument("--halo-windows", type=int, default=16, help="speculative halo of a time shard, in av_windows")
    ap.add_argument("--batch", type=int, default=0, help="configs[3]: decode a batch of this many independent captures instead")
    ap.add_argument("--batch-samples", type=float, default=4e6, help="samples per capture of the batch")
    ap.add_argument("--batch-workers", type=int, default=8)
    ap.add_argument("--batch-spin", action="store_true", help="batch: spinning waits (the library's default for a single stream)")
    ap.add_argument("--batch-legacy", action="store_true", help="batch: one nfc_stream per capture on worker threads instead of one pass")
    ap.add_argument("--no-configs", action="store_true", help="skip the sub-runs of the other BASELINE.json configs (2 / 20 MS/s, batch, C5)")
    ap.add_argument("--c5-total", type=float, default=1e11, help="configs[4]: samples of the one strong-scaled 20 MS/s capture")
    ap.add_argument("--c5-piece", type=float, default=1e10, help="configs[4]: samples rendered and pushed at a time")
    ap.add_argument("--c4-per-gpu", type=int, default=512, help="configs[3] leg: captures per GPU (4096 over eight GPUs)")
    ap.add_argument("--parity-windows", type=int, default=4, help="windows of the timed capture decoded again by the oracle (untimed)")
    ap.add_argument("--wait", default="auto", choices=["auto", "spin", "blocking"],
                    help="how host threads wait for the device: blocking sleeps in the driver (auto = spin: at eight ranks "
                         "blocking waits were no faster)")
    ap.add_argument("--fade", type=float, default=0.05, help="channel: slow amplitude fade depth (experiments)")
    ap.add_argument("--tag-high", type=float, default=1.07, help="channel: tag load-modulation amplitude ratio (experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the frames of the last one to DIR/<name>.npy "
                                                          "(records and a seeded sample of the frame bits; inputs are seeded)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps < 1:
        ap.error("--steps: at least one timed step")
    if args.dump_outputs and (args.impl != "b200" or args.batch > 0 or world > 1):
        ap.error("--dump-outputs: the decode of one capture on one GPU only (no --batch, --impl reference or several ranks)")
    quiet_stdout()
    globals()["RATE"] = args.rate
    import torch
    import torch.distributed as dist

    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    codes, lens, params = build_schedule(RATE, 2024)
    period = int(lens.sum())
    chan = dict(carrier=0.5, pause=0.015, tag_high=args.tag_high, noise=0.003, fade=args.fade, fade_period=round(RATE * 0.02))
    workload = "synthetic ISO 14443A reader+tag traffic, %.3g samples at %.2f MS/s per GPU" % (args.samples, RATE / 1e6)
    config = {"workload": workload, "samp_rate": RATE, "hi_val": HI_VAL, "input": "float32 envelope resident in HBM",
              "l2": "input (%.1f GB per step) is far larger than L2; no flush needed" % (args.samples * 4 / 1e9),
              "schedule_period_samples": period, **params}

    # ------------------------------------------------------------------ reference arm (host cores)
    if args.impl == "reference":
        if rank != 0:
            return 0
        from usrp_nfc_b200 import synth
        threads = max(1, cores)
        piece = int(min(args.cpu_piece, (1 << 31) / threads))
        rng = np.random.default_rng(5)
        # same schedule, rendered on the host with the numpy generator (no GPU is used by this arm)
        reps = int(np.ceil((piece + params["av_window"]) / period))
        base = synth.render(np.tile(codes, reps), np.tile(lens, reps), RATE, rng,
                            synth.Channel(pause=chan["pause"], tag_high=chan["tag_high"], noise=chan["noise"],
                                          fade=chan["fade"], fade_period_us=20000.0))[:piece]
        x = synth.envelope(synth.pcm_to_float(base))
        pieces = [np.roll(x, 977 * i) for i in range(threads)]
        vals = []
        for i in range(args.warmup + args.steps):
            v, dt, _ = cpu_baseline(pieces, params, threads)
            if i >= args.warmup:
                vals.append((v, dt))
        v = float(np.mean([a for a, _ in vals]))
        ms = float(np.mean([b for _, b in vals])) * 1e3
        sample = "%d independent pieces of %d samples of the same schedule, one per host thread" % (threads, piece)
        line = {"impl": "reference", "metric": "decoded_msamples_per_s", "value": v, "unit": "Msamples/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config, "sample_note": "bounded CPU sample per step: " + sample,
                "cpu_baseline": {"value": v, "unit": "Msamples/s", "cores": threads, "kind": "port", "sample": sample,
                                 "python_reference": PY_REF_NOTE},
                "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit(line)
        return 0

    # ------------------------------------------------------------------ this repo's CUDA path
    from usrp_nfc_b200 import _cabi
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.batch > 0:
        return bench_batch(args, rank, world, local_rank, codes, lens, params, chan, dist, torch, _cabi)
    from usrp_nfc_b200 import sharding
    L = params["av_window"]
    n = int(args.samples)
    q = L * 4 // np.gcd(L, 4)
    n -= n % q  # shard boundaries are multiples of av_window and of 4 (sharding.plan)
    total = world * n
    bounds, halo = sharding.plan(total, world, L, args.halo_windows)
    begin, end = bounds[rank]
    base = max(0, begin - halo - L) if rank > 0 else 0
    # every rank renders its own time shard of one endless capture, plus the halo in front of it
    x = torch.empty(end - base, dtype=torch.float32, device="cuda")
    _cabi.synth_render(x, codes, lens, seed=99, as_envelope=True, device=local_rank, first_index=base, **chan)
    torch.cuda.synchronize()

    s = _cabi.Stream(RATE, hi_val=HI_VAL, outputs=_cabi.OUT_FRAMES, device=local_rank, **params)
    s.set_tuning(seg_len=args.seg_len, halo=args.halo, slab_len=int(args.slab))
    blocking = args.wait == "blocking"  # (A/B at eight ranks: spinning 31.1 ms per step, blocking 32.0)
    if blocking:
        s.set_wait_mode(True)
    host_waits = "blocking" if blocking else "spinning"  # (not part of `config`: the reference arm has no such thing)
    shard_info = {}
    gather_state = {}
    shared = None
    if world > 1:
        # the ranks of the node keep their packed frame indexes in shared memory that rank 0 maps (falls back to the NCCL
        # gather when /dev/shm has no room)
        want_recs = int(n * 2.5e-4) + (1 << 16)
        room = shm_room()
        shared = sharding.SharedFrameIndex(s, want_recs if room > 4 * world * want_recs * 8 else 0, dist)

    def step(keep=False):
        if world == 1:
            s.reset()
            s.push_all(x)
            fr, _, _ = s.view_frames()  # records and frame bits in host memory (zero-copy view of the library's buffers)
            nfr = len(fr)
            if not keep:  # (kept: dumped and released once the clock has stopped)
                s.release_frames()
            return nfr
        res = sharding.decode_time_sharded(s, lambda a, b: x[a - base: b - base], total, L, _cabi.State, dist=dist,
                                           device="cuda", halo_windows=args.halo_windows, flat="view")
        shard_info.update(repaired=res["repaired"], seam_ok=res["seam_ok"])
        nfr = res["n_frames"]
        tg = time.perf_counter()
        # the frame offsets of all shards on rank 0, in stream order (packets.py:94-98): fixed 8-byte records over NCCL
        index = sharding.gather_frame_records(s, res["pos_offset"], dist, device="cuda", state=gather_state, shared=shared)
        if index is not None:
            shard_info.update(gathered_frames=int(len(index)), gathered_bytes=int(len(index)) * 8, index=index,
                              gather_via="shared memory of the node (no copy)" if (shared is not None and shared.ok) else "NCCL gather")
        shard_info["phases_ms"] = dict(res["phases_ms"], gather_offsets=(time.perf_counter() - tg) * 1e3)
        s.release_frames()
        return nfr

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    frames = 0
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.wait_running()
    t_load = time.perf_counter()
    for _ in range(args.warmup):
        frames = step()
    s.reset_stats()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    for i in range(args.steps):
        frames = step(keep=bool(args.dump_outputs) and i == args.steps - 1)
    ev1.record()
    barrier()
    wall = time.perf_counter() - t0
    st = s.stats()
    clocks = sampler.stop(t_load, t0, t0 + wall) if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, s.view_frames())
        s.release_frames()
    # device time of the step on the library's own stream (CUDA events inside the library bracket every slab)
    dev_ms = st["kernel_ms"] / args.steps
    wall_ms = wall * 1e3 / args.steps
    t = torch.tensor([wall_ms, dev_ms, float(frames), float(st["launches"]), float(st["seam_mismatches"]),
                      st["slicer_ms"] / args.steps, st["slicer_kernel_ms"] / args.steps], dtype=torch.float64, device="cuda")
    per_rank = None
    if world > 1:
        allt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank = [{"wall_ms": float(a[0]), "device_ms": float(a[1]), "slicer_ms": float(a[5]), "frames": int(a[2]),
                     "seam_mismatches": int(a[4])} for a in allt]
        mx = t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        wall_ms, dev_ms, slicer_ms, kern_ms = float(mx[0]), float(mx[1]), float(mx[5]), float(mx[6])
        frames_total, launches, mism = int(sm[2]), int(sm[3]), int(sm[4])
    else:
        slicer_ms, kern_ms = float(t[5]), float(t[6])
        frames_total, launches, mism = frames, int(st["launches"]), int(st["seam_mismatches"])
    value = world * n / (wall_ms * 1e-3) / 1e6  # whole job, wall clock around the synchronous ABI calls (>= device time)
    repaired_ranks = 0
    if world > 1 and rank == 0 and shard_info.get("index") is not None:  # untimed: the gathered offsets are in stream order
        pos_all = shard_info.pop("index").positions()
        shard_info["in_order"] = bool((np.diff(pos_all) >= 0).all()) if len(pos_all) > 1 else True
    shard_info.pop("index", None)
    if world > 1:
        rp = torch.tensor([1.0 if shard_info.get("repaired") else 0.0], device="cuda")
        dist.all_reduce(rp)
        repaired_ranks = int(rp.item())

    # ---- full-size self-check (untimed).  The slicer's answer is unique (the recurrence is causal), so it may not depend
    # on how the capture was cut: decode once more with other slab and segment lengths (other speculative starts, seams,
    # edge tiles) and compare every frame record and every frame bit on the host.
    selfcheck = None
    if world == 1 and rank == 0 and not args.no_selfcheck:
        def grab(st_):
            st_.reset()
            st_.push_all(x)
            fr_v, b0_v, b1_v = st_.view_frames()
            out = (fr_v.copy(), b0_v.copy(), b1_v.copy())
            st_.release_frames()
            return out
        ra = grab(s)
        s2 = _cabi.Stream(RATE, hi_val=HI_VAL, outputs=_cabi.OUT_FRAMES, device=local_rank, **params)
        alt = dict(seg_len=1703936, halo=args.halo, slab_len=3 << 28)
        s2.set_tuning(**alt)
        rb = grab(s2)
        st2 = s2.stats()
        s2.close()
        selfcheck = {"property": "frames (closing position, type, length, bits) do not depend on the segmentation: default tuning "
                                 "against seg_len %d, slab_len %d" % (alt["seg_len"], alt["slab_len"]),
                     "identical": same_frames(ra, rb), "frames": int(len(ra[0])), "frame_bits": int(len(ra[1]) + len(ra[2])),
                     "segments_alt": int(st2["segments"]), "seam_mismatches_alt": int(st2["seam_mismatches"])}
        # ---- windows of the timed capture decoded by the oracle (untimed): cold-started 24 av_windows early, its state has
        # converged to the stream's long before the window begins; every frame closing inside the window must be the CUDA path's
        if args.parity_windows > 0:
            try:
                selfcheck["parity_windows"] = oracle_windows(x, ra, params, args.parity_windows)
            except Exception as exc:
                selfcheck["parity_windows"] = {"error": str(exc)[:200]}
        del ra, rb

    # ---- e2e: host (pinned) buffers through the same ABI call, H2D inside the timed region.  The host buffer holds what
    # the reference's source block reads from a recording: 16-bit PCM (decoder.py:25 wavfile_source); normalisation and
    # envelope run on the device (NFC_IN_PCM_S16).  Same capture, same frames as the float path.
    e2e = None
    ne = int(min(args.e2e_samples, n))
    try:
        # ---- the host -> device ceiling of this box, measured first: rank 0 alone, then all ranks at once (the e2e number
        # cannot exceed samples = bytes / 2 over these).  The GPUs of a node share PCIe roots unevenly (eight at once: 24 to
        # 35 GB/s each): every rank's host buffer is sized in proportion to the rate its GPU gets, so that the ranks finish
        # together (the job is as fast as its slowest rank); the sizes are in the line.
        h2d = {}
        per = [1.0] * world
        try:
            scratch = torch.empty(min(ne, 1 << 27), dtype=torch.int16, pin_memory=True)
            dev_buf = torch.empty_like(scratch, device="cuda")

            def copy_gbs():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                dev_buf.copy_(scratch, non_blocking=True)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(4):
                    dev_buf.copy_(scratch, non_blocking=True)
                e1.record()
                torch.cuda.synchronize()
                return 4 * scratch.numel() * 2 / (e0.elapsed_time(e1) * 1e-3) / 1e9
            if world > 1:
                dist.barrier()
                alone = copy_gbs() if rank == 0 else 0.0
                dist.barrier()
            else:
                alone = copy_gbs()
            mine_gbs = copy_gbs()
            tg = torch.tensor([mine_gbs, alone], dtype=torch.float64, device="cuda")
            if world > 1:
                allg = [torch.empty_like(tg) for _ in range(world)]
                dist.all_gather(allg, tg)
                per = [float(a[0]) for a in allg]
                alone = float(allg[0][1])
            else:
                per = [mine_gbs]
            h2d = {"one_gpu_alone_gbs": alone, "all_gpus_at_once_gbs_per_rank": per, "all_gpus_at_once_gbs_sum": float(sum(per)),
                   "e2e_ceiling_msamples_per_s": float(sum(per)) * 1e3 / 2.0,
                   "note": "pinned int16 host buffer -> device, torch copy, 4 repetitions of %d MB; all ranks copy at the same time" % (scratch.numel() * 2 >> 20)}
            del dev_buf, scratch
        except Exception as exc:
            h2d = {"error": str(exc)[:200]}
            per = [1.0] * world
        ne_r = ne
        if world > 1 and min(per) > 0:
            share = per[rank] / (sum(per) / world)
            ne_r = int(ne * min(max(share, 0.5), 1.6))
            ne_r -= ne_r % 4
        xa = torch.empty(ne_r, dtype=torch.float32, device="cuda")
        _cabi.synth_render(xa, codes, lens, seed=99, as_envelope=False, device=local_rank, first_index=base, **chan)
        pcm_d = torch.round(xa * 32767.0).to(torch.int16)
        del xa
        xh = torch.empty(ne_r, dtype=torch.int16, pin_memory=True)
        xh.copy_(pcm_d)
        del pcm_d
        torch.cuda.synchronize()
        se = _cabi.Stream(RATE, hi_val=HI_VAL, outputs=_cabi.OUT_FRAMES, device=local_rank, input_kind=_cabi.IN_PCM_S16, **params)
        se.set_tuning(seg_len=args.seg_len, halo=args.halo, slab_len=int(min(args.slab, 1 << 28)))
        xh_np = xh.numpy()
        for _ in range(2):
            se.reset()
            se.push_all(xh_np)
            se.view_frames()
            se.release_frames()
        se.reset_stats()
        barrier()
        t0 = time.perf_counter()
        esteps = max(2, min(args.steps, 5))
        for _ in range(esteps):
            se.reset()
            se.push_all(xh_np)
            fr_e = se.view_frames()[0]
            n_fr_e = len(fr_e)
            se.release_frames()
        barrier()
        e_wall = (time.perf_counter() - t0) / esteps
        est = se.stats()
        tt = torch.tensor([e_wall], dtype=torch.float64, device="cuda")
        tot = torch.tensor([float(ne_r), est["h2d_bytes"] / esteps, est["d2h_bytes"] / esteps, float(n_fr_e)], dtype=torch.float64, device="cuda")
        sizes = [ne_r]
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            alls = [torch.empty_like(tot) for _ in range(world)]
            dist.all_gather(alls, tot)
            sizes = [int(a[0]) for a in alls]
            tot = torch.stack(alls).sum(0)
        e2e = {"value": float(tot[0]) / float(tt[0]) / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": int(tot[1]), "d2h_bytes_per_step": int(tot[2]),
               "samples_per_step_per_gpu": sizes if world > 1 else ne_r, "samples_per_step": int(tot[0]),
               "ms_per_step": float(tt[0]) * 1e3, "frames_per_step": int(tot[3]),
               "host_buffer": "int16 PCM (pinned), what wavfile_source reads; normalised and squared on the device; bytes and frames "
                              "are the whole job's" + ("; buffer sizes in proportion to the host -> device rate every GPU gets" if world > 1 else ""),
               "h2d_ceiling": h2d}
        se.close()
        del xh
    except Exception as exc:  # pinned allocation can fail on small hosts
        e2e = {"value": None, "unit": "Msamples/s", "error": str(exc)[:200]}

    peak, peak_src = measured_peak_gbs()
    cpu_pieces = None
    if rank == 0 and not args.no_cpu_baseline:
        threads = max(1, cores)
        piece = int(min(args.cpu_piece, (1 << 31) / threads, n // max(1, threads)))
        piece -= piece % 4
        host = x[: piece * threads].cpu().numpy()
        cpu_pieces = [host[i * piece: (i + 1) * piece] for i in range(threads)]

    if shared is not None:
        shared.close()
    # ---- the other BASELINE.json configs, each with its own timing, roofline fractions and clocks (none of them enters `value`)
    configs = None
    if not args.no_configs:
        s.close()
        del x
        torch.cuda.empty_cache()
        configs = {}

        def leg(name, fn):
            try:
                configs[name] = fn()
            except Exception as exc:
                configs[name] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:300])}
        leg("c4_batch", lambda: leg_batch(torch, _cabi, dist, rank, world, local_rank, args, peak, args.c4_per_gpu,
                                          int(args.batch_samples), 13.56e6))
        leg("c5_one_capture_20MS_strong", lambda: leg_c5(torch, _cabi, dist, rank, world, local_rank, args, peak, args.c5_total,
                                                         20e6, min(args.c5_piece, args.c5_total / world)))
        if world == 1:
            leg("n1_2MS_reference_defaults", lambda: leg_stream(torch, _cabi, 2e6, 2e9, local_rank, args, peak))
            leg("n1_20MS", lambda: leg_stream(torch, _cabi, 20e6, 4e9, local_rank, args, peak))
            calm = argparse.Namespace(**dict(vars(args), fade=0.0))
            leg("n1_13.56MS_without_fade", lambda: leg_stream(torch, _cabi, 13.56e6, 4e9, local_rank, calm, peak))
            leg("work_calls_2MS", lambda: leg_work_calls(torch, _cabi, local_rank, args))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # the dominant kernel alone: CUDA events around every launch of the streaming slicer kernel, on the library's stream
    k_launches = max(1, st["slicer_kernel_launches"])
    alg_bytes_per_launch = 4.0 * n * args.steps / k_launches
    achieved = 4.0 * n / (kern_ms * 1e-3) / 1e9 if kern_ms > 0 else None
    traffic = None
    try:  # DRAM bytes per sample of the committed ncu --set full capture of this kernel, scaled to this run's launches
        with open(os.path.join(ROOT, "profiles", "slicer_traffic.json")) as f:
            tj = json.load(f)
        traffic = {"bytes_per_launch": tj["dram_bytes_per_sample"] * n * args.steps / k_launches,
                   "dram_bytes_per_sample": tj["dram_bytes_per_sample"], "source": tj["source"]}
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak if achieved else None, "traffic": traffic,
                "kernel": "nfc::slicer_fast_kernel<256,4,2,IN_ENVELOPE_F32,3> (pipelined mode: slicer_pipe.cuh)", "peak_source": peak_src,
                "algorithmic_bytes_per_sample": 4, "algorithmic_bytes_per_launch": alg_bytes_per_launch,
                "avg_launch_ms": kern_ms * args.steps / k_launches, "launches_per_step": k_launches / args.steps,
                "slicer_stage_ms_per_step": slicer_ms,
                "step_frac": step_frac(n, wall_ms, peak), "step_ms": wall_ms,
                "step_note": "step_frac = 4 B x samples per GPU / wall time of the whole step (slicer, extraction, runs, line code, "
                             "framing, records to the host" + (", seam verification, gather of the frame offsets)" if world > 1 else ")"),
                "note": "achieved = 4 B x samples / CUDA-event time of the streaming slicer kernel's launches per step; the slicer "
                        "stage (kernel, seam checks and repairs, bitmap -> transition extraction) is slicer_stage_ms_per_step"}

    cpu = None
    if cpu_pieces is not None:
        threads = len(cpu_pieces)
        v, dt, _ = cpu_baseline(cpu_pieces, params, threads)
        cpu = {"value": v, "unit": "Msamples/s", "cores": threads, "kind": "port",
               "sample": "%d consecutive pieces of %d samples of rank 0's capture, one per host thread, %.1f s" % (
                   threads, len(cpu_pieces[0]), dt),
               "python_reference": PY_REF_NOTE}

    line = {"metric": "decoded_msamples_per_s", "value": value, "unit": "Msamples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "sharding": {"kind": "time shards of one capture, halo %d av_windows, seam states all_gathered and verified, frame "
                                 "offsets gathered to rank 0 inside the timed step" % args.halo_windows,
                         "ranks_redone_last_step": repaired_ranks, "frame_offsets_gathered": shard_info.get("gathered_frames"),
                         "gathered_bytes_per_step": shard_info.get("gathered_bytes"), "gathered_in_stream_order": shard_info.get("in_order"),
                         "gathered_via": shard_info.get("gather_via"),
                         "rank0_phases_ms_last_step": shard_info.get("phases_ms")} if world > 1 else None,
            "per_rank": per_rank,
            "device_ms_per_step": dev_ms, "frames_per_step": frames_total, "seam_mismatches": mism,
            "selfcheck": selfcheck, "slicer_ms_per_step": slicer_ms, "tiles": {k: st[k] for k in ("fast_tiles", "exact_tiles", "repeated_passes", "fixpoint_tiles", "st2_tiles", "unproven_tiles", "ring_resums", "segments", "pipe_tiles", "pipe_runs", "pipe_aborts")},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "configs": configs,
            "host_waits": host_waits}
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
