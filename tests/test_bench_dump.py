"""bench.py --dump-outputs: the sample of a liftover's outputs is fixed by its seed, exact, and within its size budget."""
import numpy as np

import bench


def fake_views(n, mean_len, seed=1):
    rng = np.random.default_rng(seed)
    off = np.zeros(n + 1, np.uint64)
    off[1:] = np.cumsum(rng.integers(mean_len // 2, mean_len * 3 // 2, n))
    st = {k: rng.integers(0, 2**32, n, dtype=np.uint64).astype(np.uint32) for k in bench.STATS_U32}
    st.update({k: rng.random(n, dtype=np.float32) * 100 for k in bench.STATS_F32})
    return dict(n_out=n, n_pairs=n, paf_nbytes=int(off[-1]), line_off=off, paf_text=rng.integers(32, 127, int(off[-1]), dtype=np.uint8), stats=st)


def test_sample_is_seeded_exact_and_small():
    v = fake_views(300_000, 100)
    a, b = bench.sample_outputs(v, "c5"), bench.sample_outputs(v, "c5")
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert sum(x.nbytes for x in a.values()) < 32 << 20  # two workloads stay under 64 MB
    rows, off = a["c5_rows"].astype(np.int64), v["line_off"]
    assert len(rows) == bench.DUMP_ROWS and (np.diff(rows) > 0).all()
    assert np.array_equal(a["c5_line_len"], (off[rows + 1] - off[rows]).astype(np.float64))
    for k in bench.STATS_U32 + bench.STATS_F32:
        assert (a["c5_" + k] == v["stats"][k][rows]).all(), k
    assert a["c5_stats_totals"][0] == int(v["stats"]["equal"].sum(dtype=np.uint64))
    text = np.concatenate([v["paf_text"][int(off[r]):int(off[r + 1])] for r in a["c5_text_rows"].astype(np.int64)])
    assert np.array_equal(a["c5_text"], text.astype(np.float32)) and 0 < len(text) <= bench.DUMP_TEXT_BYTES


def test_sample_of_tiny_and_empty_outputs():
    assert len(bench.sample_outputs(fake_views(10, 50), "c4")["c4_rows"]) == 10
    empty = bench.sample_outputs(fake_views(0, 50), "c4")
    assert len(empty["c4_rows"]) == 0 and len(empty["c4_text"]) == 0 and empty["c4_counts"][0] == 0
