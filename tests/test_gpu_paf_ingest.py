"""PAF text parsed on the device (rb_batch_upload_paf) against the host reader rbh::Paf::from_text: the batch's records field for
field, the name table, skipped lines, every panic with its line; BGZF input; then liftover / stats rows of such a batch against the
host-packed path and the oracle; and the `rb` CLI under RB_DEVICE_PARSE=1.  Needs a real B200 (pytest -m gpu)."""
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
COLS = ("q_len", "q_st", "q_en", "t_len", "t_st", "t_en", "mapq")


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def host_arrays(hp):
    c, n = hp.c, hp.n_rec

    def a(p, cnt, dt):
        return np.ctypeslib.as_array(p, shape=(cnt,)).copy() if cnt else np.zeros(0, dt)
    nn = int(c.n_names)
    off = a(c.names_off, nn + 1, np.uint64)
    blob = bytes(a(c.names, int(off[-1]), np.uint8)) if nn else b""
    res = dict(n_rec=n, cigar_off=a(c.cigar_off, n + 1, np.uint64), strand=a(c.strand, n, np.uint8), q_id=a(c.q_id, n, np.uint32),
               t_id=a(c.t_id, n, np.uint32), names=[blob[int(off[i]):int(off[i + 1])] for i in range(nn)],
               cigar=a(c.cigar, int(c.cigar_nbytes), np.uint8))
    for k in COLS:
        res[k] = a(getattr(c, k), n, np.uint64)
    return res


def n_lines(text: bytes) -> int:
    return text.count(b"\n") + (1 if text and not text.endswith(b"\n") else 0)


def same_records(got, want):
    assert got["n_rec"] == want["n_rec"]
    assert got["names"] == want["names"]
    for k in COLS + ("cigar_off", "strand", "q_id", "t_id", "cigar"):
        assert np.array_equal(got[k], want[k]), k


def check_text(ctx, text: bytes, data: bytes = None):
    """Device parse of `data` (default: the text itself) == host parse of `text`."""
    hp = hostlib.HostPaf.from_text(text)
    b, info = ctx.upload_paf(text if data is None else data)
    try:
        got = ctx.batch_records(b, with_cigar=True)
        want = host_arrays(hp)
        same_records(got, want)
        assert info["names"] == want["names"] and info["n_rec"] == hp.n_rec and info["skipped"] == hp.skipped
        assert info["n_lines"] == n_lines(text) and info["text_bytes"] == len(text) and info["cigar_bytes"] == hp.cigar_nbytes
    finally:
        ctx.batch_free(b)
    return hp


# ---- a corpus of mutated lines (the CPU test fuzzes the shared line core much harder; this is the GPU's share) ----
def mutated_lines(seed, n):
    rng = random.Random(seed)
    base = gen.random_paf(seed, n_contigs=4, recs_per_contig=max(1, n // 4), max_ops=60)[0].split(b"\n")
    out = []
    for ln in base:
        if not ln:
            continue
        t = ln.split(b"\t")
        k = rng.randrange(14)
        if k == 0:
            t[1] = b"+" + t[1]                                        # '+17'
        elif k == 1:
            t[2] = b"18446744073709551616"                            # u64 overflow: skipped
        elif k == 2:
            t[3] = b"00000000000000000000" + t[3]                     # 20+ digits, parses
        elif k == 3:
            t[4] = b"+-"                                              # 2-byte strand: skipped
        elif k == 4:
            t = t[:12] + [b"xx" + x for x in t[12:]]                  # prefixed cg: still the cg tag
        elif k == 5:
            t = t + [b"cg:Z:1M"]                                      # duplicated cg: the first wins
        elif k == 6:
            t = t[:12]                                                # no cg
        elif k == 7:
            t = t[:12] + [b"cg:Z:"] + t[12:]                          # empty cg: the later one replaces it
        sep = [b"\t", b" ", b"\x0c", b" \t", b"\t\x0c "][rng.randrange(5)] if rng.randrange(4) == 0 else b"\t"
        line = sep.join(t)
        if rng.randrange(6) == 0:
            line += b"\r"
        out.append(line)
    return out


def test_bundled_random_and_mutated(ctx):
    check_text(ctx, orc.golden_paf())
    for seed in range(6):
        check_text(ctx, gen.random_paf(seed, n_contigs=3, recs_per_contig=20, max_ops=400)[0])
        check_text(ctx, b"\n".join(mutated_lines(seed, 200)) + b"\n")
        check_text(ctx, b"\n".join(mutated_lines(seed + 100, 50)))   # no final newline


def test_edge_sizes(ctx):
    check_text(ctx, b"")                                   # empty input: no line
    rng = random.Random(3)
    ops = b"".join(b"%d%s" % (rng.randrange(1, 9), rng.choice([b"=", b"X", b"I", b"D"])) for _ in range(1_700_000))
    q = sum(int(x[:-1]) for x in [ops[i:i + 2] for i in range(0, len(ops), 2)] if x[-1:] in b"=XI")
    tl = sum(int(x[:-1]) for x in [ops[i:i + 2] for i in range(0, len(ops), 2)] if x[-1:] in b"=XD")
    assert len(ops) >= 3 << 20
    line = b"q\t%d\t0\t%d\t+\tt\t%d\t0\t%d\t0\t0\t60\tcs:Z::%s\tcg:Z:%s" % (q, q, tl, tl, b"7" * (1 << 20), ops)
    assert len(line) >= 4 << 20                            # a line of more than 4 MiB, two long tags
    small = gen.random_paf(1, n_contigs=2, recs_per_contig=5)[0]
    check_text(ctx, small + line + b"\n" + small)
    check_text(ctx, small + line)                           # ... as the unterminated last line


def test_read_level_paf_many_names(ctx):
    rng = np.random.default_rng(7)
    n = 1_000_000
    qlen = rng.integers(50, 150, n)
    rows = [b"read%d\t%d\t0\t%d\t%s\tctg%d\t100000\t%d\t%d\t%d\t%d\t60\tcg:Z:%d=" %
            (i, ql, ql, b"+-"[i & 1:(i & 1) + 1], i % 97, i % 1000, i % 1000 + ql, ql, ql, ql) for i, ql in enumerate(qlen.tolist())]
    text = b"\n".join(rows) + b"\n"
    check_text(ctx, text)


def test_bgzf_input_gives_the_same_batch(ctx):
    text = orc.golden_paf() + b"\n".join(mutated_lines(9, 300)) + b"\n"
    for block in (60000, 777, 65280):                       # lines straddle block boundaries
        check_text(ctx, text, bgzf(text, block))
    z = bgzf(text[:5000], 1000, eof=False) + bgzf(b"", eof=False) + bgzf(text[5000:], 3000)   # an empty block in the middle
    check_text(ctx, text, z)
    bad = bytearray(bgzf(text, 20000))
    bad[len(bad) // 2] ^= 0x40
    with pytest.raises(RbError) as e:
        ctx.upload_paf(bytes(bad))
    assert e.value.code == capi.RB_ERR_BAD_ARG
    import gzip
    with pytest.raises(RbError) as e:
        ctx.upload_paf(gzip.compress(text))                 # a plain gzip member is the caller's to inflate
    assert e.value.code == capi.RB_ERR_BAD_ARG
    check_text(ctx, text)                                   # the context still works


@pytest.mark.parametrize("bad,code,msg", [
    (b"a\tb\tc", capi.RB_ERR_REF_PAF_PARSE, "t.len() >= 12"),
    (b"", capi.RB_ERR_REF_PAF_PARSE, "t.len() >= 12"),                                   # an empty line
    (b"q\t10\t0\t10\t+\tt\t10\t0\t10\t10\t10\t60\tnotatag", capi.RB_ERR_REF_PAF_PARSE, "PAF_TAG"),
    (b"q\t10\t0\t1x\t+\tt\t10\t0\t10\t10\t10\t60\tcg:Z:10M5", capi.RB_ERR_REF_CIGAR_PARSE, "Unable to parse cigar"),
])
def test_panics_name_the_line(ctx, bad, code, msg):
    good = gen.random_paf(2, n_contigs=2, recs_per_contig=4)[0]
    skipped = b"q\t10\t0\t10\t+-\tt\t10\t0\t10\t10\t10\t60\tcg:Z:10M\n"    # a skipped line before the panic
    text = good + skipped + bad + b"\n" + good + b"a\tb\n"
    with pytest.raises(hostlib.HostPanic) as hpe:
        hostlib.HostPaf.from_text(text)
    assert msg in str(hpe.value)
    with pytest.raises(RbError) as e:
        ctx.upload_paf(text)
    assert e.value.code == code
    line = good.count(b"\n") + 2
    assert f"line {line}:" in str(e.value) and msg in str(e.value)


def lift_rows(ctx, b, wins, policy, want, stats):
    ctx.batch_set_windows(b, wins)
    ctx.batch_liftover(b, policy=policy, with_stats=stats, want=want)
    return ctx.batch_download_lift(b, want=capi.WANT_TEXT if want & capi.WANT_STATS_TEXT else want, stats=stats)


def check_rows(ctx, text, bed):
    hp = hostlib.HostPaf.from_text(text)
    hw = hp.windows_from_bed_text(bed)
    b, info = ctx.upload_paf(text)
    try:
        assert info["names"] == host_arrays(hp)["names"]
        for policy in (capi.POLICY_RIGHTMOST, capi.POLICY_EARLY_EXIT):
            for want, stats in ((capi.WANT_TEXT | capi.WANT_NUMERIC, True), (capi.WANT_STATS_TEXT, False)):
                got = lift_rows(ctx, b, hw, policy, want, stats)
                exp = ctx.liftover(hp, hw, policy=policy, want=want, stats=stats)
                for k in exp:
                    if k == "stats":
                        for s in exp[k]:
                            assert np.array_equal(np.asarray(got[k][s]), np.asarray(exp[k][s])), s
                    elif isinstance(exp[k], np.ndarray):
                        assert np.array_equal(got[k], exp[k]), k
                    else:
                        assert got[k] == exp[k], k
        ctx.batch_stats(b)
        st = ctx.batch_download_stats(b)
        exp = ctx.stats(hp)
        for k in exp:
            assert np.array_equal(np.asarray(st[k]), np.asarray(exp[k])), k
    finally:
        ctx.batch_free(b)
    return got


def test_c1_rows_equal_the_oracle(ctx):
    text, bed = orc.golden_paf(), orc.golden_bed()
    hp = hostlib.HostPaf.from_text(text)
    b, _ = ctx.upload_paf(text)
    try:
        got = lift_rows(ctx, b, hp.windows_from_bed_text(bed), capi.POLICY_RIGHTMOST, capi.WANT_TEXT, False)
        assert got["paf_text"] == orc.run_liftover(text, bed, threads=4)
    finally:
        ctx.batch_free(b)
    check_rows(ctx, text, bed)


def test_random_rows_equal_the_host_path(ctx):
    for seed in range(3):
        text, contigs = gen.random_paf(seed, n_contigs=3, recs_per_contig=12, max_ops=300)
        check_rows(ctx, text, gen.random_bed(seed, contigs, 60))
        check_rows(ctx, text, gen.tiling_bed(contigs, 37))


def test_c4_synthetic_full_size(ctx):
    text = hostlib.HostPaf.synth().text()
    hp = hostlib.HostPaf.from_text(text)  # (the generator's own name table is not in first-appearance order)
    hw = hp.tiling_windows(10_000)
    b, info = ctx.upload_paf(text)
    try:
        assert info["n_rec"] == hp.n_rec and info["cigar_bytes"] == hp.cigar_nbytes
        same_records(ctx.batch_records(b), host_arrays(hp))
        got = lift_rows(ctx, b, hw, capi.POLICY_RIGHTMOST, capi.WANT_TEXT | capi.WANT_NUMERIC, True)
        ref = ctx.upload(hp, hw)
        try:
            ctx.batch_liftover(ref, with_stats=True)
            exp = ctx.batch_download_lift(ref)
        finally:
            ctx.batch_free(ref)
        assert got["paf_text"] == exp["paf_text"] and np.array_equal(got["line_off"], exp["line_off"])
        for k in ("equal", "diff", "ins", "del", "id_by_all"):
            assert np.array_equal(got["stats"][k], exp["stats"][k]), k
    finally:
        ctx.batch_free(b)


# ---- CLI: RB_DEVICE_PARSE=1 ----
def run_rb(args, env_extra=None):
    rb = os.path.join(ROOT, "rustybam_b200", "rb")
    env = dict(os.environ, **(env_extra or {}))
    return subprocess.run([rb] + args, capture_output=True, env=env)


def test_cli_device_parse_equals_the_default(tmp_path):
    import gzip
    paf, bed = orc.golden_paf(), orc.golden_bed()
    (tmp_path / "a.bed").write_bytes(bed)
    (tmp_path / "a.paf.gz").write_bytes(gzip.compress(paf))
    (tmp_path / "a.paf.bgz").write_bytes(bgzf(paf))
    (tmp_path / "a.paf").write_bytes(paf)
    (tmp_path / "bad.paf").write_bytes(paf + b"x\ty\n")
    on = {"RB_DEVICE_PARSE": "1"}
    for f in ("a.paf.gz", "a.paf.bgz", "a.paf", "bad.paf"):
        for args in (["liftover", "--bed", str(tmp_path / "a.bed")], ["liftover", "--stats", "--bed", str(tmp_path / "a.bed")],
                     ["liftover", "--largest", "--bed", str(tmp_path / "a.bed")], ["stats", "--paf"]):
            want = run_rb(args + [str(tmp_path / f)])
            got = run_rb(args + [str(tmp_path / f)], on)
            assert got.returncode == want.returncode and got.stdout == want.stdout, (f, args, got.stderr[-500:])
            if f == "bad.paf":
                assert got.returncode == 101
            else:
                assert got.returncode == 0
