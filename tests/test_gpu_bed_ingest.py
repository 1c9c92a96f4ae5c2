"""BED text parsed on the device (rb_batch_set_windows_bed) against the host packer rbh::Windows::pack_text: the batch's window tables
field for field (rb_batch_windows), the rb_bed_info counts, BGZF input, then liftover / stats rows of such a batch against
host-set windows and the oracle, full-size C4, and the `rb` CLI under RB_DEVICE_PARSE=1.  Needs a real B200 (pytest -m gpu)."""
import gzip
import os
import random
import re
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
AWKWARD = [b"#c\nchr1\t5\t9\tA\textra\nchr2\t1\t2\tB\textra\nchr3\t1\t2\n", b"chr1\t5\t9\r\nchr1\tx\t9\nchr1\t10\t12\n\n\nchrZ\t1\t2\nchr1\t1\t3\n",
           b"track name=x\nchr1\t1\t5\n", b"\r\r\nchr2\t+5\t9\nchr2\t 5\t9\nchr2\t5\t18446744073709551616\nchr2\t3\t99999999999999999999\n"
           b"chr2\t7\t8\nchr1\t0\t18446744073709551615", b"chr1\t1\t2\t\nchr1\t1\t2\t\tx\nchr1\t0\t5\t\n#x\nchr1\t0\t5\tid with spaces\n"]


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def host_windows(hw):
    c, n = hw.c, hw.n_win

    def a(p, cnt, dt):
        return np.ctypeslib.as_array(p, shape=(cnt,)).copy() if cnt else np.zeros(0, dt)
    res = dict(n_win=n, t_id=a(c.t_id, n, np.uint32), st=a(c.st, n, np.uint64), en=a(c.en, n, np.uint64), bed_row=a(c.bed_row, n, np.uint32),
               ids_off=None, ids=None)
    if c.ids_off:
        res["ids_off"] = a(c.ids_off, n + 1, np.uint64)
        nb = int(res["ids_off"][-1])
        res["ids"] = bytes(a(c.ids, nb, np.uint8)) if nb else b""
    return res


def same_windows(got, want):
    assert got["n_win"] == want["n_win"]
    for k in ("t_id", "st", "en", "bed_row"):
        assert np.array_equal(got[k], want[k]), k
    assert (got["ids_off"] is None) == (want["ids_off"] is None)
    if want["ids_off"] is not None:
        assert np.array_equal(got["ids_off"], want["ids_off"]) and got["ids"] == want["ids"]


def expected_info(text: bytes, want) -> dict:
    """rb_bed_info from the rules, restated plainly (bed_parse_core.cuh)."""
    lines = [ln for ln in re.split(rb"[\r\n]+", text) if ln]
    rows = [ln for ln in lines if not ln.startswith(b"#")]
    nf0 = rows[0].count(b"\t") + 1 if rows else 0

    def num(f):
        return bool(re.fullmatch(rb"[0-9]+", f)) and int(f) < (1 << 64)
    parsed = sum(1 for ln in rows if nf0 >= 3 and ln.count(b"\t") + 1 == nf0 and num(ln.split(b"\t")[1]) and num(ln.split(b"\t")[2]))
    t, en, row = want["t_id"], want["en"], want["bed_row"]
    same = t[1:] == t[:-1]
    general = bool(np.any(same & ((en[1:] < en[:-1]) | (row[1:] < row[:-1])))) if len(t) > 1 else False
    return dict(text_bytes=len(text), n_lines=len(lines), n_comments=len(lines) - len(rows), n_parsed=parsed, n_win=want["n_win"],
                n_fields=nf0, default_ids=int(nf0 <= 3), general=int(general))


def check_bed(ctx, b, hp, bed: bytes, data: bytes = None):
    """Device parse of `data` (default: the BED itself) into batch b == host packer on `bed`."""
    info = ctx.batch_set_windows_bed(b, bed if data is None else data)
    want = host_windows(hp.windows_from_bed_text(bed))
    same_windows(ctx.batch_windows(b), want)
    assert info == expected_info(bed, want)
    return info


def batches(ctx, text):
    """The same records as a device-parsed batch and as a host-packed one (both without windows)."""
    hp = hostlib.HostPaf.from_text(text)
    return hp, [ctx.upload_paf(text)[0], ctx.upload(hp)]


def nested_bed(contigs):
    rows = []
    for name, ln in contigs.items():
        rows += [(name, 0, ln), (name, 5, 40), (name, 20, 30), (name, 1, 2)]
    return gen.bed_text(rows, True)


def test_field_by_field(ctx):
    seen_general = 0
    for seed in range(4):
        text, contigs = gen.random_paf(seed, n_contigs=4, recs_per_contig=10, max_ops=200)
        hp, bs = batches(ctx, text)
        beds = [gen.random_bed(seed, contigs, 80), gen.random_bed(seed, contigs, 80, with_ids=False),
                gen.random_bed(seed, contigs, 80, sort=True), gen.random_bed(seed, contigs, 80, with_ids=False, sort=True),
                gen.tiling_bed(contigs, 17), gen.tiling_bed(contigs, 23, with_ids=True), nested_bed(contigs),
                b"", b"#only\n#comments\r\n", b"chr1\t0\t10\t" + b"x" * (1 << 20) + b"\nchr2\t3\t4\tshort\n"] + AWKWARD
        try:
            for b in bs:
                for bed in beds:
                    seen_general += check_bed(ctx, b, hp, bed)["general"]
        finally:
            for b in bs:
                ctx.batch_free(b)
    assert seen_general > 0


def test_set_windows_round_trip(ctx):
    text, contigs = gen.random_paf(5, n_contigs=3, recs_per_contig=8)
    hp, bs = batches(ctx, text)
    try:
        for bed in (gen.tiling_bed(contigs, 29, with_ids=True), gen.random_bed(5, contigs, 60), nested_bed(contigs)):
            hw = hp.windows_from_bed_text(bed)
            for b in bs:
                ctx.batch_set_windows(b, hw)
                same_windows(ctx.batch_windows(b), host_windows(hw))
    finally:
        for b in bs:
            ctx.batch_free(b)


def test_read_level_query_names(ctx):
    rng = np.random.default_rng(11)
    n = 1_000_000
    qlen = rng.integers(50, 150, n)
    rows = [b"read%d\t%d\t0\t%d\t+\tctg%d\t100000\t%d\t%d\t%d\t%d\t60\tcg:Z:%d=" % (i, ql, ql, i % 97, i % 1000, i % 1000 + ql, ql, ql, ql)
            for i, ql in enumerate(qlen.tolist())]
    text = b"\n".join(rows) + b"\n"
    picks = rng.integers(0, n + 50_000, 200_000)   # some names absent
    bed = b"".join(b"read%d\t%d\t%d\tr%d\n" % (k, k % 40, k % 40 + 10, k) for k in picks.tolist())
    bed += b"".join(b"ctg%d\t%d\t%d\tc\n" % (k % 99, k, k + 100) for k in range(5000))
    hp = hostlib.HostPaf.from_text(text)
    b, _ = ctx.upload_paf(text)
    try:
        info = check_bed(ctx, b, hp, bed)
        assert 150_000 < info["n_win"] < 200_000 + 5000
    finally:
        ctx.batch_free(b)


def test_bgzf_and_bad_input(ctx):
    text, contigs = gen.random_paf(7, n_contigs=4, recs_per_contig=10)
    hp, bs = batches(ctx, text)
    beds = [gen.random_bed(7, contigs, 3000), gen.tiling_bed(contigs, 3, with_ids=True), AWKWARD[1] * 200, b""]
    try:
        for b in bs:
            for bed in beds:
                for block in (60000, 777, 65280):      # lines straddle block boundaries
                    check_bed(ctx, b, hp, bed, bgzf(bed, block))
            bed = beds[0]
            z = bgzf(bed[:5000], 1000, eof=False) + bgzf(b"", eof=False) + bgzf(bed[5000:], 3000)
            check_bed(ctx, b, hp, bed, z)
            bad = bytearray(bgzf(bed, 20000))
            bad[len(bad) // 2] ^= 0x40
            for data in (bytes(bad), gzip.compress(bed)):
                check_bed(ctx, b, hp, bed)
                with pytest.raises(RbError) as e:
                    ctx.batch_set_windows_bed(b, data)
                assert e.value.code == capi.RB_ERR_BAD_ARG
                assert ctx.batch_windows(b)["n_win"] == 0
            check_bed(ctx, b, hp, bed)              # the context and the batch still work
    finally:
        for b in bs:
            ctx.batch_free(b)


def lift(ctx, b, policy, want, stats):
    ctx.batch_liftover(b, policy=policy, with_stats=stats, want=want)
    return ctx.batch_download_lift(b, want=capi.WANT_TEXT if want & capi.WANT_STATS_TEXT else want, stats=stats)


def same_rows(got, exp):
    for k in exp:
        if k == "stats":
            for s in exp[k]:
                assert np.array_equal(np.asarray(got[k][s]), np.asarray(exp[k][s])), s
        elif isinstance(exp[k], np.ndarray):
            assert np.array_equal(got[k], exp[k]), k
        else:
            assert got[k] == exp[k], k


def check_rows(ctx, text, bed):
    hp, bs = batches(ctx, text)
    hw = hp.windows_from_bed_text(bed)
    try:
        for b in bs:
            for policy in (capi.POLICY_RIGHTMOST, capi.POLICY_EARLY_EXIT):
                for want, stats in ((capi.WANT_TEXT | capi.WANT_NUMERIC, True), (capi.WANT_STATS_TEXT, False)):
                    ctx.batch_set_windows(b, hw)
                    exp = lift(ctx, b, policy, want, stats)
                    ctx.batch_set_windows_bed(b, bed)
                    same_rows(lift(ctx, b, policy, want, stats), exp)
                    ctx.batch_set_windows_bed(b, bed)        # twice: replaces
                    same_rows(lift(ctx, b, policy, want, stats), exp)
            ctx.batch_set_windows_bed(b, bed)
            ctx.batch_set_windows(b, hw)                      # host-set windows after device-parsed ones
            same_rows(lift(ctx, b, capi.POLICY_RIGHTMOST, capi.WANT_TEXT | capi.WANT_NUMERIC, True),
                      ctx.liftover(hp, hw, want=capi.WANT_TEXT | capi.WANT_NUMERIC, stats=True))
    finally:
        for b in bs:
            ctx.batch_free(b)


def test_rows_equal_host_set_windows_and_the_oracle(ctx):
    text, bed = orc.golden_paf(), orc.golden_bed()
    b, _ = ctx.upload_paf(text)
    try:
        ctx.batch_set_windows_bed(b, bed)
        assert lift(ctx, b, capi.POLICY_RIGHTMOST, capi.WANT_TEXT, False)["paf_text"] == orc.run_liftover(text, bed, threads=4)
    finally:
        ctx.batch_free(b)
    check_rows(ctx, text, bed)
    for seed in range(3):
        text, contigs = gen.random_paf(seed, n_contigs=3, recs_per_contig=12, max_ops=300)
        for bed in (gen.random_bed(seed, contigs, 60), gen.tiling_bed(contigs, 37), nested_bed(contigs)):
            check_rows(ctx, text, bed)
        b, _ = ctx.upload_paf(text)
        try:
            bed = gen.random_bed(seed, contigs, 40, sort=True)
            ctx.batch_set_windows_bed(b, bed)
            assert lift(ctx, b, capi.POLICY_RIGHTMOST, capi.WANT_TEXT, False)["paf_text"] == orc.run_liftover(text, bed, threads=4)
        finally:
            ctx.batch_free(b)


def test_c4_full_size(ctx):
    hp = hostlib.HostPaf.synth()
    bed = hp.tiling_bed_text(1000)
    rng = random.Random(5)
    rows = bed.splitlines()[:400_000]
    rng.shuffle(rows)
    shuffled = b"".join(r + b"\tid%d" % k + b"\r\n" for k, r in enumerate(rows))
    b = ctx.upload(hp)
    try:
        info = check_bed(ctx, b, hp, bed)
        assert info["n_win"] > 3_000_000 and info["general"] == 0
        got = lift(ctx, b, capi.POLICY_RIGHTMOST, capi.WANT_TEXT | capi.WANT_NUMERIC, True)
        ctx.batch_set_windows(b, hp.windows_from_bed_text(bed))
        same_rows(got, lift(ctx, b, capi.POLICY_RIGHTMOST, capi.WANT_TEXT | capi.WANT_NUMERIC, True))
        info = check_bed(ctx, b, hp, shuffled)
        assert info["n_win"] == 400_000 and info["default_ids"] == 0
        got = lift(ctx, b, capi.POLICY_RIGHTMOST, capi.WANT_TEXT | capi.WANT_NUMERIC, True)
        ctx.batch_set_windows(b, hp.windows_from_bed_text(shuffled))
        same_rows(got, lift(ctx, b, capi.POLICY_RIGHTMOST, capi.WANT_TEXT | capi.WANT_NUMERIC, True))
    finally:
        ctx.batch_free(b)


# ---- CLI: RB_DEVICE_PARSE=1 ----
def run_rb(args, env_extra=None):
    rb = os.path.join(ROOT, "rustybam_b200", "rb")
    env = dict(os.environ, **(env_extra or {}))
    return subprocess.run([rb] + args, capture_output=True, env=env)


def test_cli_device_bed_equals_the_default(tmp_path):
    cases = [(orc.golden_paf(), orc.golden_bed())]
    for seed in range(2):
        text, contigs = gen.random_paf(seed, n_contigs=3, recs_per_contig=12, max_ops=300)
        cases.append((text, gen.random_bed(seed, contigs, 80)))
        cases.append((text, gen.tiling_bed(contigs, 41, with_ids=False)))
    on = {"RB_DEVICE_PARSE": "1"}
    for k, (paf, bed) in enumerate(cases):
        (tmp_path / "a.paf").write_bytes(paf)
        (tmp_path / "a.bed").write_bytes(bed)
        (tmp_path / "a.bed.bgz").write_bytes(bgzf(bed, 1000))
        (tmp_path / "a.bed.gz").write_bytes(gzip.compress(bed))
        for bf in ("a.bed", "a.bed.bgz", "a.bed.gz"):
            for mode in ([], ["--stats"], ["--largest"]):
                args = ["liftover"] + mode + ["--bed", str(tmp_path / bf), str(tmp_path / "a.paf")]
                want = run_rb(args)
                got = run_rb(args, on)
                assert want.returncode == 0 and got.returncode == 0, (k, bf, mode, got.stderr[-500:])
                assert got.stdout == want.stdout, (k, bf, mode)
