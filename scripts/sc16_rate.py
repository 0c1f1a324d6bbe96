"""Decode rate of complex int16 (sc16) baseband against complex64 (fc32) and the float32 envelope, on one GPU.

The bench traffic (bench.build_schedule at 13.56 MS/s) is rendered on the device as an amplitude and turned into sc16 with
a seeded phase per sample: I = rint(32767 a cos phi), Q = rint(32767 a sin phi).  Its complex64 conversion holds
RN32(I / 32767), RN32(Q / 32767) (a table of all 65536 quotients computed on the host, so no reciprocal multiply can creep
in), and the envelope is RN32(RN32(fi^2) + RN32(fq^2)): the three inputs carry the same envelope by definition.

1. Device-resident: the three inputs are decoded in turn over several repetitions (step time, slicer kernel time,
   pipelined tiles and aborts of each).
2. From pinned host memory through nfc_stream_push: sc16 against fc32.
3. The frames, frame bits and final slicer state of the sc16 and IQ_F32 decodes must be identical.

Writes one JSON file (default profiles/sc16_rate.json) with the card's name and power limit read in the same run.
    python scripts/sc16_rate.py [--samples 4e9] [--host-samples 5e8] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm,driver_version",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock, driver = [v.strip() for v in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock, driver=driver)
    except Exception as exc:  # the numbers are worth nothing without the card: say so in the file
        return dict(error=repr(exc))


def make_inputs(torch, _cabi, bench, n, piece, seed):
    """sc16 [n, 2] int16, its complex64 conversion and the float32 envelope, all on the device."""
    rate = 13.56e6
    codes, lens, p = bench.build_schedule(rate, 2024)
    dev = "cuda"
    quot = torch.from_numpy(np.arange(-32768, 32768, dtype=np.float32) / np.float32(32767.0)).to(dev)  # RN32(k / 32767)
    sc = torch.empty((n, 2), dtype=torch.int16, device=dev)
    cf = torch.empty((n, 2), dtype=torch.float32, device=dev)
    env = torch.empty(n, dtype=torch.float32, device=dev)
    amp = torch.empty(piece, dtype=torch.float32, device=dev)
    g = torch.Generator(device=dev)
    for a in range(0, n, piece):
        m = min(piece, n - a)
        _cabi.synth_render(amp[:m], codes, lens, carrier=0.5, pause=0.015, tag_high=1.07, noise=0.003, fade=0.05,
                           fade_period=round(rate * 0.02), seed=99, as_envelope=False, device=0, first_index=a)
        torch.cuda.synchronize()
        g.manual_seed(seed + a)
        phi = torch.rand(m, generator=g, device=dev, dtype=torch.float32) * (2.0 * np.pi)
        r = amp[:m] * 32767.0
        sc[a:a + m, 0] = torch.round(r * torch.cos(phi)).clamp_(-32768, 32767).to(torch.int16)
        sc[a:a + m, 1] = torch.round(r * torch.sin(phi)).clamp_(-32768, 32767).to(torch.int16)
        del phi, r
        f = quot[sc[a:a + m].to(torch.int64) + 32768]
        cf[a:a + m] = f
        e = f[:, 0] * f[:, 0]
        e2 = f[:, 1] * f[:, 1]
        env[a:a + m] = e + e2  # separate kernels: RN32(RN32(fi^2) + RN32(fq^2)), no FMA
        del f, e, e2
    del amp
    torch.cuda.synchronize()
    return sc, torch.view_as_complex(cf), env, p


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=float, default=4e9, help="device-resident samples per decode")
    ap.add_argument("--host-samples", type=float, default=5e8, help="samples per decode from pinned host memory")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--piece", type=float, default=2 ** 28, help="samples rendered and converted at a time")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sc16_rate.json"))
    args = ap.parse_args()

    import torch
    import bench
    from usrp_nfc_b200 import _cabi
    if not torch.cuda.is_available():
        raise SystemExit("sc16_rate.py measures on a GPU; none is visible")
    info = gpu_info()
    rate = 13.56e6
    from usrp_nfc_b200 import synth
    L = synth.rate_params(rate)["av_window"]
    n = int(args.samples)
    n -= n % (L * 4 // np.gcd(L, 4))
    t_make = time.perf_counter()
    sc, c64, env, p = make_inputs(torch, _cabi, bench, n, int(args.piece), 1234)
    t_make = time.perf_counter() - t_make
    inputs = [("sc16", _cabi.IN_SC16, sc), ("iq_f32", _cabi.IN_IQ_F32, c64), ("envelope_f32", _cabi.IN_ENVELOPE_F32, env)]
    streams = {}
    for name, kind, _ in inputs:
        s = _cabi.Stream(rate, hi_val=1.09, outputs=_cabi.OUT_FRAMES, input_kind=kind, **p)
        s.set_tuning(slab_len=1 << 30)
        streams[name] = s

    def decode(name, x):
        s = streams[name]
        s.reset()
        s.reset_stats()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        s.push_all(x)
        k = len(s.view_frames()[0])
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        st = s.stats()
        return dict(ms=wall * 1e3, frames=k, slicer_kernel_ms=st["slicer_kernel_ms"], kernel_ms=st["kernel_ms"],
                    pipe_tiles=st["pipe_tiles"], pipe_runs=st["pipe_runs"], pipe_aborts=st["pipe_aborts"],
                    fast_tiles=st["fast_tiles"], exact_tiles=st["exact_tiles"], segments=st["segments"],
                    serial_segments=st["serial_segments"])

    for name, _, x in inputs:  # warm-up: modules, buffers
        decode(name, x)
        streams[name].release_frames()
    runs = {name: [] for name, _, _ in inputs}
    for r in range(args.reps):
        for name, _, x in (inputs if r % 2 == 0 else inputs[::-1]):
            runs[name].append(decode(name, x))
            streams[name].release_frames()
            print("rep %d %-13s %s" % (r, name, runs[name][-1]), flush=True)

    # ---- equality of the sc16 and IQ_F32 decodes at this size
    res = {}
    for name, _, x in inputs[:2]:
        s = streams[name]
        s.reset()
        s.push_all(x)
        fr, bits = s.drain_frames_flat()
        st, ring, pend = s.state()
        res[name] = (fr.copy(), bits.copy(), st, ring.copy(), pend.copy())
    a, b = res["sc16"], res["iq_f32"]
    equal = dict(frames=a[0].tobytes() == b[0].tobytes(), frame_bits=a[1].tobytes() == b[1].tobytes(),
                 ss=a[2].ss == b[2].ss, pos=a[2].pos == b[2].pos, ring=a[3].tobytes() == b[3].tobytes(),
                 pending_bits=a[4].tobytes() == b[4].tobytes(),
                 state=all(getattr(a[2], f) == getattr(b[2], f) for f, _ in _cabi.State._fields_ if f not in ("started", "pending")))
    n_frames = int(len(a[0]))
    del res, a, b

    # ---- from pinned host memory: sc16 against fc32 through nfc_stream_push (PCIe-bound)
    nh = min(int(args.host_samples), n)
    nh -= nh % (L * 4 // np.gcd(L, 4))
    host = {}
    host["sc16"] = torch.empty((nh, 2), dtype=torch.int16, pin_memory=True)
    host["sc16"].copy_(sc[:nh])
    host["iq_f32"] = torch.empty(nh, dtype=torch.complex64, pin_memory=True)
    host["iq_f32"].copy_(c64[:nh])
    torch.cuda.synchronize()
    del sc, c64, env, inputs
    torch.cuda.empty_cache()
    hruns = {k: [] for k in host}
    for k in host:
        decode(k, host[k])
        streams[k].release_frames()
    for r in range(args.reps):
        for k in (("sc16", "iq_f32") if r % 2 == 0 else ("iq_f32", "sc16")):
            d = decode(k, host[k])
            streams[k].release_frames()
            st = streams[k].stats()
            d["h2d_bytes"] = st["h2d_bytes"]
            hruns[k].append(d)
            print("host rep %d %-7s %s" % (r, k, d), flush=True)
    for s in streams.values():
        s.close()

    def summary(rs, count):
        ms = sorted(x["ms"] for x in rs)
        return dict(ms_min=ms[0], ms_max=ms[-1], gsamples_per_s_best=count / (ms[0] * 1e-3) / 1e9,
                    slicer_kernel_ms=[x["slicer_kernel_ms"] for x in rs], pipe_tiles=rs[-1]["pipe_tiles"],
                    pipe_aborts=rs[-1]["pipe_aborts"], fast_tiles=rs[-1]["fast_tiles"], exact_tiles=rs[-1]["exact_tiles"],
                    runs=rs)

    out = dict(
        what="sc16 vs complex64 vs float32 envelope, bench traffic at 13.56 MS/s (scripts/sc16_rate.py)",
        gpu=info, torch=torch.__version__, samples_device=n, samples_host=nh, reps=args.reps, seconds_to_make_inputs=t_make,
        params=p, hi_val=1.09, frames=n_frames,
        device_resident={name: summary(runs[name], n) for name in runs},
        from_pinned_host={k: summary(hruns[k], nh) for k in hruns},
        sc16_equals_iq_f32=equal)
    d = os.path.dirname(os.path.abspath(args.out))
    os.makedirs(d, exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1, default=float)
    print(json.dumps(dict(gpu=info, equal=equal, frames=n_frames,
                          device={k: (v["ms_min"], v["gsamples_per_s_best"], v["pipe_tiles"], v["pipe_aborts"])
                                  for k, v in out["device_resident"].items()},
                          host={k: (v["ms_min"], v["gsamples_per_s_best"]) for k, v in out["from_pinned_host"].items()})))
    if not all(equal.values()):
        raise SystemExit("sc16 and IQ_F32 decodes differ: %s" % equal)


if __name__ == "__main__":
    main()
