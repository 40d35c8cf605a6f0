"""bench.py --dump-outputs: float32 arrays under DIR, at most DUMP_BYTES in all, the same seeded sample on every run. CPU only."""
import os

import numpy as np


def _dump(tmp_path, name, arrays):
    import bench
    d = str(tmp_path / name)
    bench.dump_outputs(d, arrays)
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_small_outputs_are_written_whole(tmp_path):
    st = (np.arange(1000) % 7 == 3).astype(np.uint8)
    got = _dump(tmp_path, "a", {"verify_status": st, "e2e_status": st})
    assert set(got) == {"verify_status", "e2e_status"}
    assert got["verify_status"].dtype == np.float32 and np.array_equal(got["verify_status"], st)


def test_planted_rejections_are_seeded_and_touch_only_their_items():
    import bench
    n = 5000
    rng = np.random.default_rng(0)
    pks = rng.integers(0, 256, size=n * 48, dtype=np.uint8)
    sigs = rng.integers(0, 256, size=n * 96, dtype=np.uint8)
    p, s, want = bench.plant_rejections(pks, sigs, n)
    p2, s2, want2 = bench.plant_rejections(pks, sigs, n)
    assert np.array_equal(p, p2) and np.array_equal(s, s2) and np.array_equal(want, want2)
    assert [int((want == st).sum()) for st in range(5)] == [n - 4 * 64, 64, 64, 64, 64]
    rows_p, rows_s = p.reshape(n, 48), s.reshape(n, 96)
    same = want == 0
    assert np.array_equal(rows_p[same], pks.reshape(n, 48)[same]) and np.array_equal(rows_s[same], sigs.reshape(n, 96)[same])
    i1, i2, i3, i4 = (np.nonzero(want == st)[0] for st in (1, 2, 3, 4))
    assert np.array_equal(rows_s[i1], sigs.reshape(n, 96)[(i1 + 1) % n])
    assert (rows_s[i2, 0] == 0xC0).all() and not rows_s[i2, 1:].any()
    assert (rows_p[i3, 0] == 0xC0).all() and not rows_p[i3, 1:].any()
    assert not rows_p[i4].any()
    assert not bench.plant_rejections(pks[:48 * 7], sigs[:96 * 7], 7)[2].any()   # too small to plant anything


def test_large_outputs_are_a_fixed_sample_within_the_budget(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 24_000)
    st = np.arange(10_000, dtype=np.uint32) % 251
    arrays = {"verify_status": st, "e2e_status": st, "strong_status": st}
    a, b = _dump(tmp_path, "a", arrays), _dump(tmp_path, "b", arrays)
    assert sum(v.nbytes for v in a.values()) <= 24_000
    for name in arrays:
        idx = a[name + "_index"]
        assert idx.dtype == np.float64 and a[name].dtype == np.float32 and idx.size > 0
        assert np.array_equal(a[name], st[idx.astype(np.int64)])
        assert np.array_equal(a[name], b[name]) and np.array_equal(idx, b[name + "_index"])
