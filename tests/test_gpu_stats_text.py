"""rb_stats_text (PAF bytes in, the rows of `rb stats --paf [--qbed]` out, formatted on the device) on one-, two- and three-device
contexts against rb_stats on host-parsed records plus the host formatter, and against the oracle.  Two and three contexts on GPU 0
stand in for two and three GPUs (the split, the line fix-up, the per-device threads and the merge are the same code).  Needs a real
B200 (pytest -m gpu)."""
import gzip
import os
import re
import subprocess

import numpy as np
import pytest

import gen
import orc
from rustybam_b200 import bamstats, capi, hostlib
from rustybam_b200.capi import RbError
from test_gpu_inflate import bgzf

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STATS = ("equal", "diff", "ins", "del", "ins_events", "del_events", "matches", "id_by_matches", "id_by_events", "id_by_all")


@pytest.fixture(scope="module")
def ctxs():
    old = os.environ.get("RB_MULTI_MIN_BYTES")
    os.environ["RB_MULTI_MIN_BYTES"] = "0"  # (read when a context is created)
    try:
        cs = capi.Context(0), capi.Context(devices=[0, 0]), capi.Context(devices=[0, 0, 0])
    finally:
        if old is None:
            del os.environ["RB_MULTI_MIN_BYTES"]
        else:
            os.environ["RB_MULTI_MIN_BYTES"] = old
    yield cs
    for c in cs:
        c.close()


def n_lines(text: bytes) -> int:
    return text.count(b"\n") + (1 if text and not text.endswith(b"\n") else 0)


def shuffled(text, seed):
    lines = text.splitlines(keepends=True)
    rng = np.random.default_rng(seed)
    return b"".join(lines[i] for i in rng.permutation(len(lines)))


def same_stats(got, exp):
    assert got["n"] == exp["n"]
    for k in STATS:
        if exp[k].dtype == np.float32:
            assert np.array_equal(got[k].view(np.uint32), exp[k].view(np.uint32)), k
        else:
            assert np.array_equal(got[k], exp[k]), k


def check(ctxs, text, data=None, oracle=True, qbeds=(False, True)):
    """stats_text on every context == rb_stats on host-parsed records + the host formatter (== the oracle if asked)."""
    hp = hostlib.HostPaf.from_text(text)
    exp = ctxs[0].stats(hp) if hp.n_rec else None
    for qbed in qbeds:
        rows = hp.stats_text(exp, qbed=qbed, header=False) if hp.n_rec else b""
        if oracle:
            assert bamstats.print_cigar_stats_header(qbed).encode() + rows == orc.run_stats(text, qbed)
        offs = np.concatenate([[0], np.cumsum([len(r) for r in rows.splitlines(keepends=True)], dtype=np.uint64)]).astype(np.uint64)
        for c in ctxs:
            got = c.stats_text(text if data is None else data, qbed=qbed)
            assert got["n_out"] == hp.n_rec and got["paf_nbytes"] == len(rows)
            assert got["paf_text"] == rows
            assert np.array_equal(got["line_off"], offs)
            assert "q_st" not in got
            if exp is None:
                assert got["stats"]["n"] == 0
            else:
                same_stats(got["stats"], exp)
            info = got["paf_info"]
            assert info["n_rec"] == hp.n_rec and info["n_lines"] == n_lines(text) and info["skipped"] == n_lines(text) - hp.n_rec
    return hp


def test_fixture_plain_and_bgzf(ctxs):
    text = orc.golden_paf()
    check(ctxs, text)
    check(ctxs, text, data=bgzf(text, block=200))


def test_random_pafs_every_op_class(ctxs):
    for seed in (1, 2, 3):
        for kw in (dict(style="eqx"), dict(style="mixed"), dict(style="mixed", canonical=False, clips=True)):
            text, _ = gen.random_paf(seed, n_contigs=4, recs_per_contig=9, max_ops=300, **kw)
            for t in (text, shuffled(text, seed)):
                check(ctxs, t, oracle=seed == 1 and "clips" not in kw)


def test_lifted_rows(ctxs):
    """rb liftover's output is the common input of rb stats --paf: many short records, ids, `_TO.` suffixes of the indel strip."""
    for seed in (4, 5):
        text, contigs = gen.random_paf(seed, n_contigs=3, recs_per_contig=8, max_ops=400)
        for bed in (gen.tiling_bed(contigs, 17), gen.random_bed(seed, contigs, 60)):
            lifted = orc.run_liftover(text, bed)
            assert lifted.count(b"\n") > 100
            check(ctxs, lifted)


def test_identity_edge_values(ctxs):
    """Exact integers, exact ties that round up (16.007813), 0, and NaN: a record without a cg tag and empty spans."""
    lines = []
    for i, cg in enumerate(["2049=10751X", "1=1X", "10=", "3X", "1=2X", "7=1X1=3I", "1=99999X", "12345=1X", "999=1X2D5="]):
        t = sum(int(x) for x in re.findall(r"(\d+)[=XD]", cg))
        q = sum(int(x) for x in re.findall(r"(\d+)[=XI]", cg))
        lines.append(f"q{i}\t{q + 10}\t0\t{q}\t+\tchr1\t20000000\t{i * 200000}\t{i * 200000 + t}\t0\t0\t60\tcg:Z:{cg}\n".encode())
    lines.append(b"qn\t10\t5\t5\t-\tchr1\t20000000\t7\t7\t0\t0\t60\n")
    text = b"".join(lines)
    check(ctxs, text)
    rows = ctxs[0].stats_text(text)["paf_text"]
    assert b"\t16.007813\t" in rows and b"\t100\t" in rows and b"\tNaN\tNaN\tNaN\t" in rows


def test_long_names(ctxs):
    """Names of 1-3 KB (rows past k_emit's 2 KB limit), many of them in one block, and names of 20-30 KB: rows longer than
    k_stats_rows' staging area, among short ones."""
    text, _ = gen.random_paf(6, n_contigs=3, recs_per_contig=6, max_ops=40)
    rng = np.random.default_rng(6)
    out = []
    for k, ln in enumerate(text.splitlines(keepends=True)):
        f = ln.split(b"\t")
        if k % 3 == 0:
            f[0] = b"q" * int(rng.integers(1000, 3000))
        if k % 5 == 0:
            f[5] = b"t" * int(rng.integers(1000, 3000)) + f[5]
        out.append(b"\t".join(f))
    text = b"".join(out)
    check(ctxs, text)
    # a block's rows well past k_stats_rows' 20 KB staging area (400 rows of ~3 KB), and rows longer than the staging area itself
    # (names of 20-30 KB: written straight to global memory) between short ones
    big = b"".join(ln.replace(b"\t", b"N" * 3000 + b"\t", 1) for ln in text.splitlines(keepends=True) * 20)
    check(ctxs, big, oracle=False)
    huge = b"".join(ln.replace(b"\t", b"L" * int(rng.integers(20_000, 30_000)) + b"\t", 1) if k % 3 == 1 else ln
                    for k, ln in enumerate(text.splitlines(keepends=True) * 3))
    check(ctxs, huge, oracle=False)


def test_odd_shapes(ctxs):
    text, _ = gen.random_paf(7, n_contigs=2, recs_per_contig=5, max_ops=40)
    lines = text.splitlines(keepends=True)
    long_one, _ = gen.random_paf(8, n_contigs=1, recs_per_contig=1, max_ops=20000)
    check(ctxs, lines[0] + long_one + b"".join(lines[1:]))  # one line longer than all the others together
    check(ctxs, lines[0])                                    # fewer lines than devices
    check(ctxs, b"".join(lines[:2]))
    check(ctxs, text.rstrip(b"\n"))                          # no final newline
    check(ctxs, b"")                                         # empty input
    t = shuffled(text, 7)
    for block in (1, 7, 61, 200):                            # BGZF blocks that straddle lines and devices
        check(ctxs, t, data=bgzf(t, block=block), oracle=False)
    check(ctxs, t.rstrip(b"\n"), data=bgzf(t.rstrip(b"\n"), block=9), oracle=False)


def test_skipped_lines_are_summed(ctxs):
    text, _ = gen.random_paf(9, n_contigs=3, recs_per_contig=6, max_ops=60)
    skipped = b"q\t10\t0\t10\t+-\tt\t10\t0\t10\t10\t10\t60\tcg:Z:10M\n"
    t = b"".join(ln + (skipped if k % 4 == 1 else b"") for k, ln in enumerate(text.splitlines(keepends=True)))
    hp = check(ctxs, t)
    for c in ctxs:
        assert c.stats_text(t)["paf_info"]["skipped"] == n_lines(t) - hp.n_rec > 0


def range_of(pos, n, D):
    """The device whose byte range holds text offset `pos` (the PAF's n bytes are cut at n * d // D)."""
    return max(d for d in range(D) if n * d // D <= pos)


@pytest.mark.parametrize("bad,code,msg", [
    (b"a\tb\tc", capi.RB_ERR_REF_PAF_PARSE, "t.len() >= 12"),
    (b"", capi.RB_ERR_REF_PAF_PARSE, "t.len() >= 12"),
    (b"q\t10\t0\t10\t+\tt\t10\t0\t10\t10\t10\t60\tnotatag", capi.RB_ERR_REF_PAF_PARSE, "PAF_TAG"),
    (b"q\t10\t0\t1x\t+\tt\t10\t0\t10\t10\t10\t60\tcg:Z:10M5", capi.RB_ERR_REF_CIGAR_PARSE, "Unable to parse cigar"),
])
def test_panics_on_later_devices(ctxs, bad, code, msg):
    good, _ = gen.random_paf(10, n_contigs=2, recs_per_contig=8, max_ops=60)
    lines = good.splitlines(keepends=True)
    for c, D in ((ctxs[1], 2), (ctxs[2], 3)):
        for target in range(1, D):  # the bad line's first byte in the range of device `target`
            ks = [k for k in range(len(lines) + 1)
                  if range_of(len(b"".join(lines[:k])), len(good) + len(bad) + 1, D) == target]
            assert ks, (D, target)
            k = ks[len(ks) // 2]
            text = b"".join(lines[:k]) + bad + b"\n" + b"".join(lines[k:])
            for ctx in (ctxs[0], c):
                with pytest.raises(RbError) as e:
                    ctx.stats_text(text)
                assert e.value.code == code and f"line {k + 1}:" in str(e.value) and msg in str(e.value), str(e.value)
        assert c.stats_text(good)["paf_text"] == ctxs[0].stats_text(good)["paf_text"]  # the context still works


def test_integrity_panic_on_later_devices(ctxs):
    good, _ = gen.random_paf(11, n_contigs=2, recs_per_contig=10, max_ops=60)
    lines = good.splitlines(keepends=True)
    for j in (len(lines) // 2 + 1, len(lines) - 3):
        t = lines[j].split(b"\t")
        t[3] = str(int(t[3]) + 7).encode()  # query span no longer matches the CIGAR
        text = b"".join(lines[:j]) + b"\t".join(t) + b"".join(lines[j + 1:])
        with pytest.raises(RbError) as e1:
            ctxs[0].stats(hostlib.HostPaf.from_text(text))
        assert f"record {j}:" in str(e1.value)
        for c in ctxs:
            with pytest.raises(RbError) as e:
                c.stats_text(text)
            assert e.value.code == e1.value.code and str(e.value) == str(e1.value)


def test_refusals(ctxs):
    text = orc.golden_paf()
    for c in ctxs:
        for want in (capi.WANT_TEXT, capi.WANT_NUMERIC, capi.WANT_QBED, capi.WANT_STATS_TEXT | capi.WANT_TEXT):
            with pytest.raises(RbError) as e:
                c.stats_text(text, want=want)
            assert e.value.code == capi.RB_ERR_BAD_ARG
        with pytest.raises(RbError) as e:
            c.stats_text(gzip.compress(text))
        assert e.value.code == capi.RB_ERR_BAD_ARG and "plain gzip" in str(e.value)
        z = bytearray(bgzf(text, block=300))
        z[40] ^= 0xFF
        with pytest.raises(RbError) as e:
            c.stats_text(bytes(z))
        assert e.value.code == capi.RB_ERR_BAD_ARG


def test_counters_only(ctxs):
    text = orc.golden_paf()
    exp = ctxs[0].stats(hostlib.HostPaf.from_text(text))
    for c in ctxs:
        got = c.stats_text(text, want=0)
        assert got["n_out"] == exp["n"] and "paf_text" not in got
        same_stats(got["stats"], exp)


def test_contexts_reused_after_other_calls(ctxs):
    """rb_liftover on an interleaved PAF, rb_liftover_text and a failed call leave the scratch batches behind; rb_stats_text must
    not see any of it."""
    big, bc = gen.random_paf(12, n_contigs=4, recs_per_contig=12, max_ops=300)
    big = shuffled(big, 12)
    hb = hostlib.HostPaf.from_text(big)
    wb = hb.windows_from_bed_text(gen.tiling_bed(bc, 40))
    more, _ = gen.random_paf(13, n_contigs=5, recs_per_contig=20, max_ops=120)
    more = shuffled(more, 13)
    hm = hostlib.HostPaf.from_text(more)
    rows = hm.stats_text(ctxs[0].stats(hm), header=False)
    for c in ctxs:
        c.liftover(hb, wb, want=capi.WANT_TEXT | capi.WANT_NUMERIC, stats=True)
        assert c.stats_text(more)["paf_text"] == rows
        c.liftover_text(big, gen.tiling_bed(bc, 40), want=capi.WANT_STATS_TEXT, stats=False)
        assert c.stats_text(more)["paf_text"] == rows
        with pytest.raises(RbError):
            c.stats_text(more + b"x\ty\n")
        assert c.stats_text(more)["paf_text"] == rows
        same_stats(c.stats(hm), ctxs[0].stats(hm))


def test_c4_full_size(ctxs):
    """The synthetic C4 PAF (few long records) and its rows lifted at 1 kb windows (3 M short records), as text and as BGZF."""
    hp = hostlib.HostPaf.synth()
    text = hp.text()
    hp = hostlib.HostPaf.from_text(text)
    lifted = ctxs[0].liftover(hp, hp.tiling_windows(1000), want=capi.WANT_TEXT, stats=False)["paf_text"]
    for t in (text, lifted):
        h = hostlib.HostPaf.from_text(t)
        exp = ctxs[0].stats(h)
        rows = h.stats_text(exp, header=False)
        for c in (ctxs[0], ctxs[1]):
            for data in (t, bgzf(t, level=1)):
                got = c.stats_text(data)
                assert got["n_out"] == h.n_rec and got["paf_text"] == rows
                same_stats(got["stats"], exp)


# ---- CLI: RB_DEVICE_PARSE=1 rb [--gpus N] stats --paf [--qbed] ----
def run_rb(args, env_extra=None, stdin=None):
    rb = os.path.join(ROOT, "rustybam_b200", "rb")
    env = dict(os.environ, **(env_extra or {}))
    return subprocess.run([rb] + args, capture_output=True, env=env, input=stdin)


def gpu_count():
    import torch
    return torch.cuda.device_count()


def test_cli_equals_the_default(tmp_path):
    paf = orc.golden_paf()
    (tmp_path / "a.paf.gz").write_bytes(gzip.compress(paf))
    (tmp_path / "a.paf.bgz").write_bytes(bgzf(paf, block=500))
    (tmp_path / "a.paf").write_bytes(paf)
    (tmp_path / "bad.paf").write_bytes(paf + b"x\ty\n")
    gpus = [[]] + ([["--gpus", "2"]] if gpu_count() >= 2 else [])
    on = {"RB_DEVICE_PARSE": "1", "RB_MULTI_MIN_BYTES": "0"}
    for g in gpus:
        for qbed in ([], ["--qbed"]):
            for f in ("a.paf.gz", "a.paf.bgz", "a.paf", "bad.paf", "-"):
                args = g + ["stats", "--paf"] + qbed + [str(tmp_path / f) if f != "-" else "-"]
                stdin = paf if f == "-" else None
                want = run_rb(args, stdin=stdin)
                got = run_rb(args, on, stdin=stdin)
                assert got.returncode == want.returncode and got.stdout == want.stdout, (f, args, got.stderr[-500:])
                assert got.returncode == (101 if f == "bad.paf" else 0)
                if f != "bad.paf":
                    assert got.stdout == orc.run_stats(paf, bool(qbed))
