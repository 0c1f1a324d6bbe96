"""Host logic of the batch driver (no GPU)."""
from usrp_nfc_b200 import batch


def test_rank_share_is_a_partition():
    for world in (1, 2, 3, 8):
        seen = sorted(i for r in range(world) for i in batch.rank_share(4096, r, world))
        assert seen == list(range(4096))
        sizes = [len(batch.rank_share(4096, r, world)) for r in range(world)]
        assert max(sizes) - min(sizes) <= 1


def test_bench_same_frames_compares_records_and_bits():
    """bench.py's full-size self-check compares two decodes field by field."""
    import numpy as np
    import bench
    from usrp_nfc_b200 import _cabi
    fr = np.zeros(3, dtype=_cabi.FRAME_DTYPE)
    fr["pos"], fr["nbits"], fr["type"], fr["bit_off"] = [10, 20, 30], [2, 1, 2], [0, 1, 0], [0, 0, 2]
    b0, b1 = np.array([1, 0, 1, 1], np.uint8), np.array([1], np.uint8)
    assert bench.same_frames((fr, b0, b1), (fr.copy(), b0.copy(), b1.copy()))
    other = fr.copy()
    other["pos"][1] += 1
    assert not bench.same_frames((fr, b0, b1), (other, b0, b1))
    flipped = b0.copy()
    flipped[2] ^= 1
    assert not bench.same_frames((fr, b0, b1), (fr, flipped, b1))
    assert not bench.same_frames((fr, b0, b1), (fr[:2], b0, b1))


def test_bench_dump_outputs_writes_the_frames_as_floats(tmp_path, monkeypatch):
    """bench.py --dump-outputs: records whole while they fit the cap, a fixed sample of the frame bits beyond it."""
    import numpy as np
    import bench
    from usrp_nfc_b200 import _cabi
    fr = np.zeros(3, dtype=_cabi.FRAME_DTYPE)
    fr["pos"], fr["nbits"], fr["type"] = [10, (1 << 40) + 3, 30], [2, 1, 2], [0, 1, 0]
    rng = np.random.default_rng(0)
    b0, b1 = rng.integers(0, 2, 5000).astype(np.uint8), np.array([1], np.uint8)
    monkeypatch.setattr(bench, "DUMP_BITS", 1000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), (fr, b0, b1))
    got = {p.stem: np.load(p) for p in (tmp_path / "a").iterdir()}
    assert sorted(got) == ["bits_reader", "bits_tag", "frame_nbits", "frame_pos", "frame_type"]
    assert got["frame_pos"].dtype == np.float64 and got["frame_pos"].tolist() == fr["pos"].tolist()
    assert got["frame_type"].dtype == got["frame_nbits"].dtype == np.float32
    assert got["frame_nbits"].tolist() == [2, 1, 2] and got["frame_type"].tolist() == [0, 1, 0]
    assert got["bits_reader"].tolist() == [1.0]
    idx = bench.sample_index(b0.size, 1000, 2)
    assert idx.size == 1000 and (np.diff(idx) > 0).all()
    assert got["bits_tag"].dtype == np.float32 and np.array_equal(got["bits_tag"], b0[idx])
    for name, a in got.items():
        assert np.array_equal(np.load(tmp_path / "b" / (name + ".npy")), a)
