"""rb_liftover_text (PAF and BED bytes in, lifted rows out) on multi-device contexts against rb_liftover on host-parsed records on one
device and the oracle: every device parses, tokenises and lifts the lines of its own byte range of the PAF, and the rows are merged in
(contig, device) order.  Two and three contexts on GPU 0 stand in for two and three GPUs (the split, the line fix-up, the per-device
threads and the merge are the same code).  Needs a real B200 (pytest -m gpu)."""
import gzip
import os
import random
import subprocess

import numpy as np
import pytest

import gen
import orc
from rustybam_b200 import capi, hostlib
from rustybam_b200.capi import RbError
from test_gpu_inflate import bgzf

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NUM = ("line_off", "q_st", "q_en", "t_st", "t_en", "nmatch", "aln_len", "rec_idx", "win_idx")


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


def same_rows(got, exp):
    assert got["n_out"] == exp["n_out"] and got["n_pairs"] == exp["n_pairs"] and got["paf_nbytes"] == exp["paf_nbytes"]
    for k in ("paf_text",) + NUM:
        if k in exp:
            assert k in got, k
            if isinstance(exp[k], bytes):
                assert got[k] == exp[k], k
            else:
                assert np.array_equal(got[k], exp[k]), k
    if "stats" in exp:
        for k, v in exp["stats"].items():
            if k == "n":
                assert got["stats"][k] == v
            elif v.dtype == np.float32:
                assert np.array_equal(got["stats"][k].view(np.uint32), v.view(np.uint32)), k
            else:
                assert np.array_equal(got["stats"][k], v), k


def check(ctxs, text, bed, data=None, bed_data=None, oracle=False, modes=None):
    """liftover_text on every context == rb_liftover on host-parsed records on one device (== the oracle if asked)."""
    one = ctxs[0]
    hp = hostlib.HostPaf.from_text(text)
    hw = hp.windows_from_bed_text(bed)
    modes = modes or [(p, w, s) for p in (capi.POLICY_RIGHTMOST, capi.POLICY_EARLY_EXIT)
                      for w, s in ((capi.WANT_TEXT | capi.WANT_NUMERIC, True), (capi.WANT_STATS_TEXT, False), (capi.WANT_NUMERIC, True))]
    for policy, want, stats in modes:
        if hp.n_rec:
            exp = one.liftover(hp, hw, policy=policy, want=want, stats=stats)
        else:  # (no records: the one-device batch path is the reference)
            exp = one.liftover_text(text, bed, policy=policy, want=want, stats=stats)
            assert exp["n_out"] == 0
        if oracle and want & capi.WANT_TEXT and policy == capi.POLICY_RIGHTMOST:
            assert exp["paf_text"] == orc.run_liftover(text, bed)
        for c in ctxs:
            got = c.liftover_text(text if data is None else data, bed if bed_data is None else bed_data, policy=policy, want=want, stats=stats)
            same_rows(got, exp)
            assert got["paf_info"]["n_rec"] == hp.n_rec and got["paf_info"]["n_lines"] == n_lines(text)
            assert got["paf_info"]["skipped"] == n_lines(text) - hp.n_rec
            assert got["bed_info"]["n_win"] == hw.n_win
    return hp


def n_lines(text: bytes) -> int:
    return text.count(b"\n") + (1 if text and not text.endswith(b"\n") else 0)


def shuffled(text, seed):
    lines = text.splitlines(keepends=True)
    rng = np.random.default_rng(seed)
    return b"".join(lines[i] for i in rng.permutation(len(lines)))


def test_fixture_and_oracle(ctxs):
    text, bed = orc.golden_paf(), orc.golden_bed()
    check(ctxs, text, bed, oracle=True)
    check(ctxs, text, bed, data=bgzf(text, block=200), bed_data=bgzf(bed, block=150), oracle=True)


def test_grouped_interleaved_and_many_contigs(ctxs):
    for seed in (1, 2):
        text, contigs = gen.random_paf(seed, n_contigs=4, recs_per_contig=9, max_ops=300)
        for t in (text, shuffled(text, seed)):
            check(ctxs, t, gen.tiling_bed(contigs, 40), oracle=True)
            check(ctxs, t, gen.random_bed(seed, contigs, 30))
    text, contigs = gen.random_paf(3, n_contigs=320, recs_per_contig=2, max_ops=40)
    t = shuffled(text, 3)
    check(ctxs, t, gen.tiling_bed(contigs, 25), oracle=True, modes=[(capi.POLICY_RIGHTMOST, capi.WANT_TEXT | capi.WANT_NUMERIC, True)])


def test_bgzf_blocks_straddle_lines_and_devices(ctxs):
    text, contigs = gen.random_paf(4, n_contigs=3, recs_per_contig=6, max_ops=80)
    t = shuffled(text, 4)
    bed = gen.tiling_bed(contigs, 30)
    modes = [(capi.POLICY_RIGHTMOST, capi.WANT_TEXT | capi.WANT_NUMERIC, True)]
    for block in (1, 7, 61, 200):
        check(ctxs, t, bed, data=bgzf(t, block=block), modes=modes)
    check(ctxs, t, bed, bed_data=bgzf(bed, block=13), modes=modes)


def test_bed_kinds(ctxs):
    import test_gpu_bed_ingest as tb
    text, contigs = gen.random_paf(5, n_contigs=3, recs_per_contig=8, max_ops=200)
    t = shuffled(text, 5)
    modes = [(p, capi.WANT_TEXT | capi.WANT_NUMERIC, True) for p in (capi.POLICY_RIGHTMOST, capi.POLICY_EARLY_EXIT)]
    for bed in (gen.tiling_bed(contigs, 33), gen.random_bed(5, contigs, 40), tb.nested_bed(contigs)):
        check(ctxs, t, bed, modes=modes, oracle=True)
        rows = bed.splitlines(keepends=False)
        with_ids = b"".join(r.split(b"\t")[0] + b"\t" + b"\t".join(r.split(b"\t")[1:3]) + b"\tid%d\n" % k for k, r in enumerate(rows) if r)
        check(ctxs, t, with_ids, modes=modes)


def test_odd_shapes(ctxs):
    text, contigs = gen.random_paf(6, n_contigs=2, recs_per_contig=5, max_ops=40)
    bed = gen.tiling_bed(contigs, 20)
    lines = text.splitlines(keepends=True)
    long_one = gen.random_paf(7, n_contigs=1, recs_per_contig=1, max_ops=20000)
    modes = [(capi.POLICY_RIGHTMOST, capi.WANT_TEXT | capi.WANT_NUMERIC, True)]
    # one line longer than all the others together
    lt, lc = long_one
    check(ctxs, lines[0] + lt + b"".join(lines[1:]), gen.tiling_bed({**contigs, **lc}, 50), modes=modes)
    check(ctxs, lines[0], bed, modes=modes)                          # fewer lines than devices
    check(ctxs, b"".join(lines[:2]), bed, modes=modes)
    check(ctxs, text.rstrip(b"\n"), bed, modes=modes)                # no final newline
    check(ctxs, text.rstrip(b"\n"), bed, data=bgzf(text.rstrip(b"\n"), block=9), modes=modes)
    check(ctxs, b"", bed, modes=modes)                               # empty input
    check(ctxs, text, b"", modes=modes)


def test_skipped_lines_are_summed(ctxs):
    text, contigs = gen.random_paf(8, n_contigs=3, recs_per_contig=6, max_ops=60)
    skipped = b"q\t10\t0\t10\t+-\tt\t10\t0\t10\t10\t10\t60\tcg:Z:10M\n"
    lines = text.splitlines(keepends=True)
    t = b"".join(ln + (skipped if k % 4 == 1 else b"") for k, ln in enumerate(lines))
    hp = check(ctxs, t, gen.tiling_bed(contigs, 25), modes=[(capi.POLICY_RIGHTMOST, capi.WANT_TEXT, False)])
    for c in ctxs:
        info = c.liftover_text(t, gen.tiling_bed(contigs, 25), want=capi.WANT_TEXT, stats=False)["paf_info"]
        assert info["skipped"] == n_lines(t) - hp.n_rec > 0


def range_of(pos, n, D):
    """The device whose byte range holds text offset `pos` (rb_liftover_text cuts n bytes at n * d // D)."""
    return max(d for d in range(D) if n * d // D <= pos)


@pytest.mark.parametrize("bad,code,msg", [
    (b"a\tb\tc", capi.RB_ERR_REF_PAF_PARSE, "t.len() >= 12"),
    (b"", capi.RB_ERR_REF_PAF_PARSE, "t.len() >= 12"),
    (b"q\t10\t0\t10\t+\tt\t10\t0\t10\t10\t10\t60\tnotatag", capi.RB_ERR_REF_PAF_PARSE, "PAF_TAG"),
    (b"q\t10\t0\t1x\t+\tt\t10\t0\t10\t10\t10\t60\tcg:Z:10M5", capi.RB_ERR_REF_CIGAR_PARSE, "Unable to parse cigar"),
])
def test_panics_on_later_devices(ctxs, bad, code, msg):
    good, contigs = gen.random_paf(9, n_contigs=2, recs_per_contig=8, max_ops=60)
    bed = gen.tiling_bed(contigs, 25)
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
                    ctx.liftover_text(text, bed)
                assert e.value.code == code and f"line {k + 1}:" in str(e.value) and msg in str(e.value), str(e.value)
        same_rows(c.liftover_text(good, bed, stats=False), ctxs[0].liftover_text(good, bed, stats=False))  # the context still works


def test_lift_error_on_a_later_device(ctxs):
    good, contigs = gen.random_paf(10, n_contigs=2, recs_per_contig=10, max_ops=60)
    lines = good.splitlines(keepends=True)
    t = lines[-3].split(b"\t")
    t[3] = str(int(t[3]) + 7).encode()                  # target span no longer matches the CIGAR
    text = b"".join(lines[:-3]) + b"\t".join(t) + b"".join(lines[-2:])
    bed = gen.tiling_bed(contigs, 25)
    hp = hostlib.HostPaf.from_text(text)
    with pytest.raises(RbError) as e1:
        ctxs[0].liftover(hp, hp.windows_from_bed_text(bed))
    for c in ctxs:
        with pytest.raises(RbError) as e:
            c.liftover_text(text, bed)
        assert e.value.code == e1.value.code and str(e.value) == str(e1.value)


def test_refusals(ctxs):
    text, bed = orc.golden_paf(), orc.golden_bed()
    for c in ctxs:
        with pytest.raises(RbError) as e:
            c.liftover_text(text, bed, want=capi.WANT_TEXT | capi.WANT_QBED)
        assert e.value.code == capi.RB_ERR_BAD_ARG
        with pytest.raises(RbError) as e:
            c.liftover_text(gzip.compress(text), bed)
        assert e.value.code == capi.RB_ERR_BAD_ARG and "plain gzip" in str(e.value)
        z = bytearray(bgzf(text, block=300))
        z[40] ^= 0xFF
        with pytest.raises(RbError) as e:
            c.liftover_text(bytes(z), bed)
        assert e.value.code == capi.RB_ERR_BAD_ARG


def test_corrupt_block_on_a_later_device_is_numbered_in_the_file(ctxs):
    text, bed = orc.golden_paf(), orc.golden_bed()
    z = bytearray(bgzf(text, block=300))
    starts, pos = [], 0
    while pos < len(z):
        starts.append(pos)
        pos += int.from_bytes(z[pos + 16:pos + 18], "little") + 1
    j = len(starts) * 9 // 10      # (ISIZE-balanced cuts: the last device's blocks for two and three devices)
    end = starts[j + 1]
    z[end - 8] ^= 0xFF             # its CRC-32
    msgs = []
    for c in ctxs:
        with pytest.raises(RbError) as e:
            c.liftover_text(bytes(z), bed)
        assert e.value.code == capi.RB_ERR_BAD_ARG and f"block {j} " in str(e.value), str(e.value)
        msgs.append(str(e.value))
    assert len(set(msgs)) == 1, msgs


def test_contexts_reused_after_rb_liftover(ctxs):
    """rb_liftover on an interleaved PAF leaves the scratch batches of a multi-device context mapping rows to that call's records;
    rb_liftover_text afterwards must not see any of it, on the N-device path and on the one-device path of a small PAF."""
    big, bc = gen.random_paf(11, n_contigs=4, recs_per_contig=12, max_ops=300)
    big = shuffled(big, 11)
    hb = hostlib.HostPaf.from_text(big)
    wb = hb.windows_from_bed_text(gen.tiling_bed(bc, 40))
    old = os.environ.get("RB_MULTI_MIN_BYTES")
    small, sc = gen.random_paf(12, n_contigs=1, recs_per_contig=2, max_ops=20)
    assert len(small) < 2000 < hb.cigar_nbytes
    os.environ["RB_MULTI_MIN_BYTES"] = "2000"
    try:
        mid = capi.Context(devices=[0, 0])
    finally:
        if old is None:
            del os.environ["RB_MULTI_MIN_BYTES"]
        else:
            os.environ["RB_MULTI_MIN_BYTES"] = old
    more, mc = gen.random_paf(13, n_contigs=5, recs_per_contig=20, max_ops=120)
    more = shuffled(more, 13)
    want = capi.WANT_TEXT | capi.WANT_NUMERIC
    try:
        for c, text, contigs in ((mid, small, sc), (ctxs[1], more, mc), (ctxs[2], more, mc), (ctxs[1], small, sc)):
            ref = ctxs[0].liftover(hb, wb, want=want, stats=True)
            same_rows(c.liftover(hb, wb, want=want, stats=True), ref)   # leaves the scratch batches gathered from `big`
            bed = gen.tiling_bed(contigs, 30)
            hp = hostlib.HostPaf.from_text(text)
            exp = ctxs[0].liftover(hp, hp.windows_from_bed_text(bed), want=want, stats=True)
            same_rows(c.liftover_text(text, bed, want=want, stats=True), exp)
    finally:
        mid.close()


def test_c4_full_size_two_devices(ctxs):
    hp = hostlib.HostPaf.synth()
    text = hp.text()
    hp = hostlib.HostPaf.from_text(text)
    bed = hp.tiling_bed_text(10_000)
    exp = ctxs[0].liftover(hp, hp.windows_from_bed_text(bed), want=capi.WANT_TEXT | capi.WANT_NUMERIC, stats=True)
    for data in (text, bgzf(text)):
        same_rows(ctxs[1].liftover_text(data, bed, want=capi.WANT_TEXT | capi.WANT_NUMERIC, stats=True), exp)


# ---- CLI: RB_DEVICE_PARSE=1 rb --gpus 2 liftover ----
def run_rb(args, env_extra=None):
    rb = os.path.join(ROOT, "rustybam_b200", "rb")
    env = dict(os.environ, **(env_extra or {}))
    return subprocess.run([rb] + args, capture_output=True, env=env)


def gpu_count():
    import torch
    return torch.cuda.device_count()


def test_cli_two_gpus_equals_the_default(tmp_path):
    if gpu_count() < 2:
        pytest.skip("needs two GPUs")
    paf, bed = orc.golden_paf(), orc.golden_bed()
    (tmp_path / "a.bed").write_bytes(bed)
    (tmp_path / "a.paf.gz").write_bytes(gzip.compress(paf))
    (tmp_path / "a.paf.bgz").write_bytes(bgzf(paf, block=500))
    (tmp_path / "a.paf").write_bytes(paf)
    (tmp_path / "bad.paf").write_bytes(paf + b"x\ty\n")
    on = {"RB_DEVICE_PARSE": "1", "RB_MULTI_MIN_BYTES": "0"}
    for f in ("a.paf.gz", "a.paf.bgz", "a.paf", "bad.paf"):
        for args in (["liftover"], ["liftover", "--stats"], ["liftover", "--largest"]):
            args = ["--gpus", "2"] + args + ["--bed", str(tmp_path / "a.bed"), str(tmp_path / f)]
            want = run_rb(args)
            got = run_rb(args, on)
            assert got.returncode == want.returncode and got.stdout == want.stdout, (f, args, got.stderr[-500:])
            assert got.returncode == (101 if f == "bad.paf" else 0)
