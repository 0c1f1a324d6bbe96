"""Decode rate of a batch of captures of different lengths on one GPU.

The bench traffic (bench.build_schedule at 13.56 MS/s, bench's default channel) is rendered once on the device and cut into
512 captures with seeded log-uniform lengths from 5e5 to 1.6e7 samples (about 2.3e9 in all), each starting 16-byte aligned.
hi_val cycles through 1.05..1.10 per capture as in bench.py's batch leg.  Compared, each after warm-up:

  (a) ragged: the captures in one pass (batch.decode_batch_onepass with the list, nfc_stream_push_batch_ragged);
  (b) per_capture: batch.decode_batch with 8 workers, one nfc_stream per capture at a time;
  (c) equal: nfc_stream_push_batch on 512 equally long captures with the same total, the reference rate.

Reports wall time per step, Gsamples/s and slicer kernel time (CUDA events inside the library; (b) runs its streams inside
decode_batch, whose kernel time is not collected).  (a) and (b) must give identical per-capture frame records and frame bits.  --equal-only runs
(c) alone and prints a digest of its frame records and bits (for comparing builds).

Writes one JSON file (default profiles/ragged_batch_rate.json) with the card's name and power limit read in the same run.
    python scripts/ragged_batch_rate.py [--captures 512] [--steps 5] [--warmup 2] [--out FILE] [--equal-only]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

RATE = 13.56e6
HIS = [1.05, 1.06, 1.07, 1.08, 1.09, 1.10]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm,driver_version",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock, driver = [v.strip() for v in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock, driver=driver)
    except Exception as exc:  # the numbers are worth nothing without the card: say so in the file
        return dict(error=repr(exc))


def layout(n_caps, seed, lo=5e5, hi=1.6e7):
    """Seeded log-uniform lengths and 16-byte aligned (multiple-of-4-sample) offsets into one flat buffer."""
    rng = np.random.default_rng(seed)
    lens = np.exp(rng.uniform(np.log(lo), np.log(hi), n_caps)).astype(np.int64)
    offs = np.zeros(n_caps + 1, np.int64)
    offs[1:] = np.cumsum((lens + 3) // 4 * 4)
    return lens, offs


def render(torch, _cabi, bench, n, piece):
    codes, lens, p = bench.build_schedule(RATE, 2024)
    x = torch.empty(n, dtype=torch.float32, device="cuda")
    for a in range(0, n, piece):
        m = min(piece, n - a)
        _cabi.synth_render(x[a:a + m], codes, lens, carrier=0.5, pause=0.015, tag_high=1.07, noise=0.003, fade=0.05,
                           fade_period=round(RATE * 0.02), seed=500, as_envelope=True, device=0, first_index=a)
    torch.cuda.synchronize()
    return x, p


def digest(fr, b0, b1):
    h = hashlib.sha256()
    for a in (fr, b0, b1):
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--captures", type=int, default=512)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workers", type=int, default=8)
    ap.add_argument("--piece", type=float, default=2 ** 28, help="samples rendered at a time")
    ap.add_argument("--equal-only", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ragged_batch_rate.json"))
    args = ap.parse_args()

    import torch
    import bench
    from usrp_nfc_b200 import _cabi, batch
    if not torch.cuda.is_available():
        raise SystemExit("ragged_batch_rate.py measures on a GPU; none is visible")
    info = gpu_info()
    n_caps = args.captures
    lens, offs = layout(n_caps, args.seed)
    total = int(lens.sum())
    t_make = time.perf_counter()
    flat, p = render(torch, _cabi, bench, int(offs[-1]), int(args.piece))
    t_make = time.perf_counter() - t_make
    his = np.array([HIS[i % len(HIS)] for i in range(n_caps)], dtype=np.float64)
    caps = [flat[int(o): int(o) + int(m)] for o, m in zip(offs[:-1], lens)]
    m_eq = total // n_caps // 4 * 4
    x2d = flat[:n_caps * m_eq].view(n_caps, m_eq)
    s = _cabi.Stream(RATE, outputs=_cabi.OUT_FRAMES, **p)

    def timed(fn, count):
        for _ in range(args.warmup):
            fn()
        s.reset_stats()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            out = fn()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / args.steps
        st = s.stats()
        return out, dict(ms_per_step=ms, gsamples_per_s=count / (ms * 1e-3) / 1e9,
                         slicer_kernel_ms_per_step=st["slicer_kernel_ms"] / args.steps,
                         slicer_kernel_launches=st["slicer_kernel_launches"], pipe_tiles=st["pipe_tiles"])

    def equal_step():
        return batch.decode_batch_onepass(x2d, RATE, p, hi_vals=his, stream=s)

    res_c, eq = timed(equal_step, n_caps * m_eq)
    fr, b0, b1 = res_c["stream"].view_frames()
    eq.update(samples=n_caps * m_eq, items_per_capture=m_eq, frames=int(len(fr)), digest=digest(fr, b0, b1))
    print("equal: %s" % json.dumps(eq), flush=True)
    s.release_frames()
    if args.equal_only:
        print(json.dumps(dict(gpu=info, equal=eq)))
        s.close()
        return

    def ragged_step():
        return batch.decode_batch_onepass(caps, RATE, p, hi_vals=his, stream=s)

    res_a, rg = timed(ragged_step, total)
    got_a = [(f.copy(), b.copy()) for f, b in batch.split_captures(res_a, n_caps)]
    rg.update(samples=total, frames=int(sum(len(f) for f, _ in got_a)))
    print("ragged: %s" % json.dumps(rg), flush=True)
    s.release_frames()

    plist = [dict(hi_val=float(h), **p) for h in his]

    def per_capture_step():
        return batch.decode_batch(caps, RATE, plist, workers=args.workers)

    got_b, pc = timed(per_capture_step, total)
    pc.update(samples=total, frames=int(sum(len(f) for f, _ in got_b)), slicer_kernel_ms_per_step=None,
              slicer_kernel_launches=None, pipe_tiles=None)
    print("per_capture: %s" % json.dumps(pc), flush=True)
    s.close()

    same = len(got_a) == len(got_b)
    differences = []
    for c, ((fa, ba), (fb, bb)) in enumerate(zip(got_a, got_b)):
        # records and each frame's bits (the per-capture bit arrays may differ in what follows the last frame: decode_batch
        # drains the bits a capture's unfinished frame had gathered too)
        if all(np.array_equal(fa[k], fb[k]) for k in ("pos", "nbits", "type")) and all(
                np.array_equal(x[2], y[2]) for x, y in zip(batch.frames_as_lists(fa, ba), batch.frames_as_lists(fb, bb))):
            continue
        same = False
        if len(differences) < 4:  # which of the two the oracle agrees with
            from oracle import oracle
            want = oracle.decode_capture(caps[c].cpu().numpy(), RATE, hi_val=float(his[c]), **p)["frames"]
            first = next((i for i in range(min(len(fa), len(fb))) if fa["pos"][i] != fb["pos"][i] or fa["nbits"][i] != fb["nbits"][i]),
                         min(len(fa), len(fb)))
            differences.append(dict(capture=c, length=int(lens[c]), frames_one_pass=len(fa), frames_per_capture=len(fb),
                                    frames_oracle=len(want), first_difference=int(first),
                                    pos_one_pass=fa["pos"][first:first + 3].tolist(), pos_per_capture=fb["pos"][first:first + 3].tolist(),
                                    one_pass_equals_oracle=bool(np.array_equal(fa["pos"], want["pos"]) and np.array_equal(fa["nbits"], want["nbits"])),
                                    per_capture_equals_oracle=bool(np.array_equal(fb["pos"], want["pos"]) and np.array_equal(fb["nbits"], want["nbits"]))))
            print("difference: %s" % json.dumps(differences[-1]), flush=True)

    out = dict(
        what="512 captures of log-uniform lengths (5e5..1.6e7 samples) of bench traffic at 13.56 MS/s, device-resident, one "
             "GPU (scripts/ragged_batch_rate.py)",
        gpu=info, torch=torch.__version__, captures=n_caps, samples=total, longest=int(lens.max()), shortest=int(lens.min()),
        steps=args.steps, warmup=args.warmup, seconds_to_render=t_make, params=p,
        ragged_one_pass=rg, per_capture_decode_batch=pc, equal_push_batch=eq,
        ragged_equals_per_capture=bool(same), differences=differences)
    d = os.path.dirname(os.path.abspath(args.out))
    os.makedirs(d, exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1, default=float)
    print(json.dumps(dict(gpu=info, same=bool(same), ragged=(rg["ms_per_step"], rg["gsamples_per_s"]),
                          per_capture=(pc["ms_per_step"], pc["gsamples_per_s"]), equal=(eq["ms_per_step"], eq["gsamples_per_s"]))))
    if not same:
        raise SystemExit("the one-pass and per-capture decodes differ")


if __name__ == "__main__":
    main()
