"""Batches of independent captures (SURVEY.md section 8(e), BASELINE.json configs[3]).

Every capture is its own `transition_sink` + decoders + packet processors in the reference (separate state,
its own `hi_val`), so a batch partitions trivially: captures are dealt round-robin to the ranks (one process per
GPU) and, inside a rank, to a few worker threads that each drive one `nfc_stream` at a time on its own CUDA
stream -- the kernels of different captures overlap on the device, the C ABI releases the GIL.  There is no
data-path collective; only frame counts / records are gathered.
"""
import threading

import numpy as np

from . import _cabi


def _decode_one(x, samp_rate, params, device, tuning, outputs, kind, cache, blocking=True):
    """One capture through one nfc_stream; a worker keeps one stream per window geometry and only changes its thresholds
    between captures (device buffers are not reallocated)."""
    key = tuple(sorted((k, v) for k, v in params.items() if k not in ("lo_val", "hi_val")))
    s = cache.get(key)
    if s is None:
        s = _cabi.Stream(samp_rate, device=device, outputs=outputs, input_kind=kind, **params)
        if tuning:
            s.set_tuning(**tuning)
        s.set_wait_mode(blocking)
        cache[key] = s
    else:
        s.reset()
        s.set_thresholds(params.get("lo_val", 0.1), params.get("hi_val", 1.1))
    s.push_all(x)
    fr, bits = s.drain_frames_flat()
    return fr, bits


def decode_batch(captures, samp_rate, params, device=0, workers=8, tuning=None, outputs=_cabi.OUT_FRAMES,
                 kind=_cabi.IN_ENVELOPE_F32, blocking_wait=True):
    """Decode independent captures on one GPU.

    captures: sequence of sample arrays (numpy, or CUDA tensors on `device`); params: one dict of Stream keyword
    arguments per capture (hi_val, av_window, max_len, ...) or a single dict for all.
    blocking_wait: the workers sleep while they wait for their stream (nfc_stream_set_wait_mode) instead of spinning --
    with spinning waits, the workers and each stream's marshalling thread outnumber the host cores.
    Returns a list of (frame records, flat frame bits) in capture order.
    """
    n = len(captures)
    plist = params if isinstance(params, (list, tuple)) else [params] * n
    out = [None] * n
    errors = []
    lock = threading.Lock()
    nxt = [0]

    def work():
        cache = {}
        try:
            _work(cache)
        finally:
            for st in cache.values():
                st.close()

    def _work(cache):
        while True:
            with lock:
                i = nxt[0]
                nxt[0] += 1
            if i >= n:
                return
            try:
                out[i] = _decode_one(captures[i], samp_rate, plist[i], device, tuning, outputs, kind, cache, blocking_wait)
            except Exception as exc:  # surfaced to the caller below
                errors.append((i, exc))
                return

    ths = [threading.Thread(target=work) for _ in range(max(1, min(workers, n)))]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    if errors:
        raise errors[0][1]
    return out


def decode_batch_onepass(captures, samp_rate, params, lo_vals=None, hi_vals=None, device=0, outputs=_cabi.OUT_FRAMES,
                         kind=_cabi.IN_ENVELOPE_F32, stream=None):
    """A batch of captures in one pass over the device (nfc_stream_push_batch / nfc_stream_push_batch_ragged): one launch
    of the slicer with one segment per capture, extraction / runs / line code over the whole batch, no host work per
    capture.

    captures: 2-D array or CUDA tensor [captures, items] of equally long captures, or a list of 1-D arrays or CUDA tensors
    of any lengths (all on the host or all on the device; IN_SC16: [items, 2] int16 each); params: the Stream keyword
    arguments all captures share (av_window, max_len, ...); lo_vals / hi_vals: one threshold per capture (transition_sink's
    constructor arguments, transition_sink.py:12).  stream: a Stream to reuse (it is reset).  Returns dict(starts, pitch,
    frames, bits_tag, bits_reader, stream): frame records with positions in the batch's position space (capture c owns
    [starts[c], starts[c + 1]), its item i is at starts[c] + i; pitch: the distance between captures of a 2-D batch, None for
    a list), bit_off into bits_tag (type 0) / bits_reader (type 1); views valid until the stream is used again.  Falls back
    to decode_batch when a capture needs the sequential path (the same results, capture by capture).

    Every capture is one segment on one CTA: a capture far longer than the rest bounds the batch's time at one CTA's rate."""
    s = stream
    if s is None:
        s = _cabi.Stream(samp_rate, device=device, outputs=outputs, input_kind=kind, **params)
    else:
        s.release_frames()
        s.reset()
    ragged = isinstance(captures, (list, tuple))
    try:
        if ragged:
            starts, pitch = s.push_batch_ragged(captures, lo_vals=lo_vals, hi_vals=hi_vals), None
        else:
            pitch = s.push_batch(captures, lo_vals=lo_vals, hi_vals=hi_vals)
            starts = np.arange(len(captures) + 1, dtype=np.int64) * pitch
    except _cabi.BatchNeedsSequential:
        n = len(captures)
        plist = []
        for i in range(n):
            p = dict(params)
            if lo_vals is not None:
                p["lo_val"] = float(lo_vals[i])
            if hi_vals is not None:
                p["hi_val"] = float(hi_vals[i])
            plist.append(p)
        res = decode_batch([captures[i] for i in range(n)], samp_rate, plist, device=device, outputs=outputs, kind=kind)
        return dict(starts=None, pitch=None, per_capture=res, stream=s)
    fr, b0, b1 = s.view_frames()
    return dict(starts=starts, pitch=pitch, frames=fr, bits_tag=b0, bits_reader=b1, stream=s)


def split_captures(res, n_captures):
    """Result of decode_batch_onepass -> [(frame records, flat frame bits)] per capture, as decode_batch returns them:
    positions relative to the capture, bit_off into the capture's own bit array."""
    if res.get("per_capture") is not None:
        return res["per_capture"]
    fr = res["frames"]
    starts = res.get("starts")
    if starts is None:
        starts = np.arange(n_captures + 1, dtype=np.int64) * res["pitch"]
    starts = np.asarray(starts, dtype=np.int64)
    cap = np.searchsorted(starts, fr["pos"], "right") - 1
    out = []
    for c in range(n_captures):
        sel = fr[cap == c].copy()
        bits = []
        off = 0
        for r in sel:
            src = res["bits_tag"] if r["type"] == 0 else res["bits_reader"]
            bits.append(np.array(src[int(r["bit_off"]): int(r["bit_off"]) + int(r["nbits"])], dtype=np.uint8))
            r["bit_off"] = off
            off += int(r["nbits"])
        sel["pos"] -= starts[c]
        out.append((sel, np.concatenate(bits) if bits else np.zeros(0, np.uint8)))
    return out


def rank_share(n_captures, rank, world):
    """Indices of the captures rank `rank` decodes (round-robin)."""
    return list(range(rank, n_captures, world))


def decode_batch_distributed(make_capture, n_captures, samp_rate, params_of, dist=None, group=None, device=0,
                             workers=8, tuning=None, kind=_cabi.IN_ENVELOPE_F32):
    """Round-robin a batch over the ranks.  make_capture(i) -> samples of capture i (called only for this rank's
    share), params_of(i) -> its Stream keyword arguments.  Returns dict(indices, results, n_frames_total)."""
    rank = dist.get_rank(group) if dist is not None else 0
    world = dist.get_world_size(group) if dist is not None else 1
    mine = rank_share(n_captures, rank, world)
    caps = [make_capture(i) for i in mine]
    res = decode_batch(caps, samp_rate, [params_of(i) for i in mine], device=device, workers=workers, tuning=tuning,
                       kind=kind)
    n_frames = sum(len(fr) for fr, _ in res)
    total = n_frames
    if dist is not None and world > 1:
        import torch
        dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
        t = torch.tensor([float(n_frames)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, group=group)
        total = int(t.item())
    return dict(indices=mine, results=res, n_frames=n_frames, n_frames_total=total)


def frames_as_lists(fr, bits):
    """(records, flat bits) -> [(pos, type, uint8 bit array)] like Stream.drain_frames."""
    return [(int(r["pos"]), int(r["type"]), np.array(bits[int(r["bit_off"]): int(r["bit_off"]) + int(r["nbits"])], dtype=np.uint8))
            for r in fr]
