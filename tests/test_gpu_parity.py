"""Parity tests proper: the CUDA path through the C ABI (rbcuda.h) against the CPU oracle,
byte-for-byte.  Every test here needs a real B200 (pytest -m gpu)."""
import hashlib

import numpy as np
import pytest

import gen
import orc
from rustybam_b200 import bamstats, bed, capi, hostlib, liftover
from rustybam_b200.paf import Paf, ReferencePanic

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def lift_and_stats(ctx, paf_text, bed_text, policy=0):
    """(`rb liftover` bytes, `rb stats --paf` bytes of that output) from the GPU path."""
    paf = Paf.from_text(paf_text)
    rgns = bed.parse_bed_text(bed_text)
    res = liftover.trim_paf_by_rgns(ctx, rgns, paf, policy=policy, stats=True)
    lifted = res["paf_text"]
    # the fused per-row stats, printed with the lifted rows' own columns (what `| rb stats --paf` prints)
    out_paf = Paf.from_text(lifted)
    assert len(out_paf) == res["n_out"]
    stats_txt = (bamstats.print_cigar_stats_header() + bamstats.stats_rows(out_paf, res["stats"])).encode()
    return res, lifted, stats_txt


def check_against_oracle(ctx, paf_text, bed_text, policy=0):
    want = orc.run_liftover(paf_text, bed_text, policy=policy, threads=4)
    res, lifted, stats_txt = lift_and_stats(ctx, paf_text, bed_text, policy)
    assert lifted == want
    assert stats_txt == orc.run_stats(want)
    # numeric mirror agrees with the text
    rows = [ln.split(b"\t") for ln in lifted.splitlines()]
    assert [int(r[2]) for r in rows] == res["q_st"].tolist()
    assert [int(r[3]) for r in rows] == res["q_en"].tolist()
    assert [int(r[7]) for r in rows] == res["t_st"].tolist()
    assert [int(r[8]) for r in rows] == res["t_en"].tolist()
    assert [int(r[9]) for r in rows] == res["nmatch"].tolist()
    assert [int(r[10]) for r in rows] == res["aln_len"].tolist()
    off = res["line_off"]
    assert off[0] == 0 and off[-1] == len(lifted)
    assert all(lifted[int(o) - 1:int(o)] == b"\n" for o in off[1:])
    return res


# ---------------------------------------------------------------- config 1: bundled fixture
def test_c1_bundled_liftover_and_stats(ctx):
    res = check_against_oracle(ctx, orc.golden_paf(), orc.golden_bed())
    assert res["n_out"] == 12 and res["paf_nbytes"] == 508497
    assert hashlib.md5(res["paf_text"]).hexdigest() == "f009e11b3bc56a4967cf594f750123a9"


def test_c1_stats_of_input_paf(ctx):
    got = bamstats.run_stats(ctx, orc.golden_paf())
    assert got == orc.run_stats(orc.golden_paf())


@pytest.mark.parametrize("width", [100_000, 10_000])
def test_c1_tiling_windows(ctx, width):
    paf_text = orc.golden_paf()
    contigs = {}
    for ln in paf_text.splitlines():
        f = ln.split(b"\t")
        contigs[f[5].decode()] = int(f[6])
    bed_text = gen.tiling_bed(contigs, width)
    res = check_against_oracle(ctx, paf_text, bed_text)
    assert res["n_out"] == {100_000: 1657, 10_000: 14385}[width]


# ---------------------------------------------------------------- the reference's own vectors, through the C ABI
F_PAF = b"Q\t10\t2\t10\t+\tT\t40\t12\t20\t3\t9\t60\tcg:Z:4M1I1=1D2=\n"
R_PAF = b"Q\t10\t2\t10\t-\tT\t40\t12\t20\t3\t9\t60\tcg:Z:4M1I1=1D2=\n"


@pytest.mark.parametrize("policy", [0, 1])
def test_aln_pair_liftover_vectors(ctx, policy):
    # liftover.rs:233-325: (q_st, q_en) for six regions, + and - strand
    regions = [(14, 15), (14, 18), (12, 20), (12, 30), (5, 20), (5, 30)]
    sts = [4, 7, 4, 4, 2, 2, 2, 2, 2, 2, 2, 2]
    ens = [5, 8, 8, 8, 10, 10, 10, 10, 10, 10, 10, 10]
    bed_text = "".join(f"T\t{a}\t{b}\n" for a, b in regions).encode()
    idx = 0
    got = {}
    for name, text in (("f", F_PAF), ("r", R_PAF)):
        res = liftover.trim_paf_by_rgns(ctx, bed.parse_bed_text(bed_text), Paf.from_text(text), policy=policy)
        assert res["n_out"] == 6
        got[name] = res
    for k in range(6):
        for name in ("f", "r"):
            assert int(got[name]["q_st"][k]) == sts[idx] and int(got[name]["q_en"][k]) == ens[idx]
            idx += 1


def test_add_cigar_stats_vector(ctx):
    # bamstats.rs:287-295
    st = bamstats.stats_from_paf(ctx, Paf.from_text(b"Q\t20\t0\t20\t+\tT\t20\t0\t20\t0\t0\t60\tcg:Z:10=10X\n"))
    assert st["id_by_all"][0] == np.float32(50.0) and st["equal"][0] == 10 and st["diff"][0] == 10


def test_tokeniser_vs_reference_parser_doctest(ctx):
    # paf.rs:1007-1012 strings; checked through the stats counters + integrity check of the spans
    for cg, t, q in (("10M4D100I1102=", 10 + 4 + 1102, 10 + 100 + 1102), ("100000M20=5P10X4M", 100034, 100034)):
        line = f"Q\t{q}\t0\t{q}\t+\tT\t{t}\t0\t{t}\t0\t0\t60\tcg:Z:{cg}\n".encode()
        assert bamstats.run_stats(ctx, line) == orc.run_stats(line)


# ---------------------------------------------------------------- randomised parity, edge cases included
@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("policy", [0, 1])
def test_random_eqx_tiling(ctx, seed, policy):
    paf_text, contigs = gen.random_paf(seed, n_contigs=4, recs_per_contig=8)
    check_against_oracle(ctx, paf_text, gen.tiling_bed(contigs, 7 + seed), policy)


@pytest.mark.parametrize("seed", range(6))
def test_random_streaming_lift_mode(ctx, seed):
    # RB_LIFT_STREAM: window boundaries resolved inside the prefix scan (k_scan_lift + k_combine)
    ctx.set_lift_mode(capi.LIFT_STREAM)
    try:
        paf_text, contigs = gen.random_paf(400 + seed, n_contigs=4, recs_per_contig=8, style="all" if seed % 2 else "eqx",
                                           canonical=(seed < 4), allow_zero=(seed >= 4), clips=(seed % 3 == 0))
        check_against_oracle(ctx, paf_text, gen.tiling_bed(contigs, 5 + seed))
        check_against_oracle(ctx, paf_text, gen.random_bed(seed, contigs, 80, sort=True))
        check_against_oracle(ctx, orc.golden_paf(), gen.tiling_bed({"chr20": 66210247, "chr21": 45827691, "chr22": 51353906}, 10_000 + seed))
    finally:
        ctx.set_lift_mode(capi.LIFT_SEARCH)


@pytest.mark.parametrize("seed", range(6))
def test_random_sliced_calls(ctx, seed):
    # rb_liftover in slices (forced onto tiny inputs: >= 64 bytes of CIGAR per slice)
    ctx.set_slicing(64)
    try:
        paf_text, contigs = gen.random_paf(500 + seed, n_contigs=5, recs_per_contig=9, style="all" if seed % 2 else "eqx",
                                           canonical=(seed < 4), allow_zero=(seed >= 4), clips=(seed % 3 == 0), max_ops=200)
        if seed % 2 == 0:  # grouped by target: emission order == file order, slices are plain runs of the input
            paf_text = b"".join(sorted(paf_text.splitlines(keepends=True), key=lambda ln: ln.split(b"\t")[5]))
        # (odd seeds: contigs interleave in the file, every slice is gathered in emission order)
        check_against_oracle(ctx, paf_text, gen.tiling_bed(contigs, 5 + seed), seed % 2)
        check_against_oracle(ctx, paf_text, gen.random_bed(seed, contigs, 80, sort=True, with_ids=(seed % 2 == 0)))
        check_against_oracle(ctx, paf_text, gen.random_bed(seed, contigs, 40))  # general layout: falls back to one batch
        check_against_oracle(ctx, orc.golden_paf(), gen.tiling_bed({"chr20": 66210247, "chr21": 45827691, "chr22": 51353906}, 20_000 + seed))
    finally:
        ctx.set_slicing()


def test_sliced_call_fails_cleanly_when_a_late_slice_panics(ctx):
    # a record of the LAST contig has a leading deletion (remove_trailing_indels panics, Q9): the sliced call has
    # already downloaded earlier slices by then; it must fail like the single-batch call and leave the context usable
    paf_text, contigs = gen.random_paf(91, n_contigs=5, recs_per_contig=8, max_ops=200, lead_trail=False)
    lines = sorted(paf_text.splitlines(keepends=True), key=lambda ln: ln.split(b"\t")[5])
    bad = b"Qbad\t13\t0\t5\t+\t" + lines[-1].split(b"\t")[5] + b"\t100000\t10\t18\t0\t0\t60\tcg:Z:3D5=\n"
    paf_text = b"".join(lines) + bad
    bed_text = gen.tiling_bed(contigs, 9)
    with pytest.raises(orc.ReferencePanic):
        orc.run_liftover(paf_text, bed_text)
    ctx.set_slicing(64)
    try:
        with pytest.raises(ReferencePanic):
            liftover.run_liftover(ctx, paf_text, bed_text)
        good = b"".join(lines)
        assert liftover.run_liftover(ctx, good, bed_text) == orc.run_liftover(good, bed_text)
    finally:
        ctx.set_slicing()


def test_sliced_call_restarts_when_the_text_estimate_is_too_small(capfd, monkeypatch):
    # the pinned text buffer of a sliced call is sized from the first slice; here the first slice yields one short row
    # and the later ones whole records, so the estimate is far too small and the call must restart as a single batch
    paf_text, contigs = gen.random_paf(77, n_contigs=8, recs_per_contig=20, max_ops=400)
    paf_text = b"".join(sorted(paf_text.splitlines(keepends=True), key=lambda ln: ln.split(b"\t")[5]))
    names = sorted(contigs)
    first = [ln for ln in paf_text.splitlines() if ln.split(b"\t")[5].decode() == names[0]][0].split(b"\t")
    rows = [(names[0], int(first[7]) + 1, int(first[7]) + 3)] + [(nm, 0, contigs[nm] + 1000) for nm in names[1:]]
    bed_text = gen.bed_text(rows, with_ids=False)
    monkeypatch.setenv("RB_TRACE", "1")  # the library logs its slice decisions to stderr
    ctx = capi.Context(0)                # a fresh context: no large pinned block from an earlier call to fall into
    ctx.set_slicing(64)
    try:
        res = check_against_oracle(ctx, paf_text, bed_text)
    finally:
        ctx.close()
    assert res["n_out"] > 30
    assert "text estimate too small: falling back" in capfd.readouterr().err


@pytest.mark.parametrize("seed", range(6))
def test_random_unsorted_nested_bed_general_path(ctx, seed):
    # BED file order is never sorted by the reference (Q5); nested + duplicate rows
    paf_text, contigs = gen.random_paf(100 + seed, n_contigs=3, recs_per_contig=6)
    check_against_oracle(ctx, paf_text, gen.random_bed(seed, contigs, 60, with_ids=(seed % 2 == 0)), seed % 2)


@pytest.mark.parametrize("seed", range(4))
def test_random_sorted_overlapping_bed(ctx, seed):
    paf_text, contigs = gen.random_paf(200 + seed, n_contigs=3, recs_per_contig=6)
    check_against_oracle(ctx, paf_text, gen.random_bed(seed, contigs, 80, sort=True))


@pytest.mark.parametrize("seed", range(6))
def test_random_all_ops_noncanonical(ctx, seed):
    # M/N/P ops, zero-length ops, adjacent same-class ops (Q15 re-collapse), clips
    paf_text, contigs = gen.random_paf(300 + seed, style="all", canonical=False, allow_zero=True, clips=(seed % 2 == 0))
    check_against_oracle(ctx, paf_text, gen.tiling_bed(contigs, 11), seed % 2)
    assert bamstats.run_stats(ctx, paf_text) == orc.run_stats(paf_text)


def test_many_tiny_records_in_one_tile(ctx):
    paf_text, contigs = gen.random_paf(7, n_contigs=2, recs_per_contig=400, max_ops=3, lead_trail=False)
    check_against_oracle(ctx, paf_text, gen.tiling_bed(contigs, 50))
    assert bamstats.run_stats(ctx, paf_text) == orc.run_stats(paf_text)


def test_long_numbers_and_leading_zeros(ctx):
    cg = "0000000000000000000012=3X000004=1I0000000000000000000000000000000000007=268435455D5="
    t = 12 + 3 + 4 + 7 + 268435455 + 5
    q = 12 + 3 + 4 + 1 + 7 + 5
    line = f"Q\t{q}\t0\t{q}\t+\tT\t{t + 10}\t5\t{t + 5}\t0\t0\t60\tcg:Z:{cg}\n".encode()
    assert bamstats.run_stats(ctx, line) == orc.run_stats(line)
    check_against_oracle(ctx, line, b"T\t0\t20\nT\t10\t268435480\nT\t268435470\t268435999\n")


def test_empty_inputs(ctx):
    res = liftover.trim_paf_by_rgns(ctx, [], Paf.from_text(F_PAF))
    assert res["n_out"] == 0 and res["paf_text"] == b""
    res = liftover.trim_paf_by_rgns(ctx, bed.parse_bed_text(b"T\t0\t5\n"), Paf.from_text(F_PAF))  # no overlap
    assert res["n_out"] == 0
    res = liftover.trim_paf_by_rgns(ctx, bed.parse_bed_text(b"T\t0\t5\n"), Paf.from_text(b""))
    assert res["n_out"] == 0
    assert bamstats.run_stats(ctx, b"") == orc.run_stats(b"")


def test_record_without_cigar_and_zero_spans(ctx):
    line = b"Q\t10\t3\t3\t+\tT\t40\t12\t12\t0\t0\t60\ttp:A:P\n"
    assert bamstats.run_stats(ctx, line) == orc.run_stats(line)  # NaN identities


# ---------------------------------------------------------------- where the reference panics, the call fails loudly
@pytest.mark.parametrize("cg,t,q", [("3D5=", 8, 5), ("5Q", 5, 5), ("5=3", 5, 5), ("=5", 5, 5), ("5==", 5, 5), ("4294967296=", 5, 5),
                                    ("5=3H2=", 7, 7), ("2I3D", 3, 2)])
def test_reference_panics_liftover(ctx, cg, t, q):
    line = f"Q\t{q + 5}\t0\t{q}\t+\tT\t{t + 5}\t0\t{t}\t0\t0\t60\tcg:Z:{cg}\n".encode()
    with pytest.raises(orc.ReferencePanic):
        orc.run_liftover(line, b"T\t0\t100\n")
    with pytest.raises(ReferencePanic):
        liftover.run_liftover(ctx, line, b"T\t0\t100\n")


def test_integrity_panic(ctx):
    line = b"Q\t20\t0\t11\t+\tT\t20\t0\t10\t0\t0\t60\tcg:Z:10=\n"
    with pytest.raises(orc.ReferencePanic):
        orc.run_stats(line)
    with pytest.raises(ReferencePanic):
        bamstats.run_stats(ctx, line)


def test_after_an_error_the_context_still_works(ctx):
    with pytest.raises(ReferencePanic):
        bamstats.run_stats(ctx, b"Q\t20\t0\t11\t+\tT\t20\t0\t10\t0\t0\t60\tcg:Z:10=\n")
    assert bamstats.run_stats(ctx, F_PAF) == orc.run_stats(F_PAF)


def test_resident_batch_is_repeatable(ctx):
    paf_text, contigs = gen.random_paf(11, n_contigs=3, recs_per_contig=10)
    paf = Paf.from_text(paf_text)
    recs = paf.pack()
    wins = bed.pack_windows(bed.parse_bed_text(gen.tiling_bed(contigs, 9)), recs.name_index)
    b = ctx.upload(recs, wins)
    s1 = ctx.batch_liftover(b)
    s2 = ctx.batch_liftover(b)
    assert s1 == s2
    out = ctx.batch_download_lift(b)
    assert out["paf_text"] == orc.run_liftover(paf_text, gen.tiling_bed(contigs, 9))
    views, release = ctx.batch_download_lift_view(b)  # the same outputs, left in the library's pinned block
    assert views["paf_text"].tobytes() == out["paf_text"]
    for k in ("line_off", "q_st", "t_en", "rec_idx", "win_idx"):
        assert (views[k] == out[k]).all(), k
    for k in ("equal", "diff", "ins", "del", "ins_events", "del_events", "matches", "id_by_all"):
        assert (views["stats"][k] == out["stats"][k]).all(), k
    release()
    ctx.batch_free(b)


# ---------------------------------------------------------------- rb break-paf (SURVEY 8f.1): same kernels, windows from the record's own indels
def check_break_against_oracle(ctx, paf_text, max_size, policy=0):
    want = orc.run_break_paf(paf_text, max_size, policy)
    res = liftover.break_paf_on_indels(ctx, Paf.from_text(paf_text), max_size, policy=policy, stats=True)
    assert res["paf_text"] == want
    out_paf = Paf.from_text(res["paf_text"])
    assert len(out_paf) == res["n_out"]
    st = (bamstats.print_cigar_stats_header() + bamstats.stats_rows(out_paf, res["stats"])).encode()
    assert st == orc.run_stats(want)
    rows = [ln.split(b"\t") for ln in want.splitlines()]
    assert [int(r[7]) for r in rows] == res["t_st"].tolist() and [int(r[3]) for r in rows] == res["q_en"].tolist()
    return res


def test_break_paf_reference_doctest_vectors(ctx):
    # liftover.rs:169-181: every piece of 5=5I5= / 5=5D5= broken at indels > 0 has a target span of 5
    for line in (b"Q\t10\t0\t10\t+\tT\t15\t0\t15\t9\t15\t60\tcg:Z:5=5D5=\n", b"Q\t15\t0\t15\t+\tT\t10\t0\t10\t9\t15\t60\tcg:Z:5=5I5=\n",
                 b"Q\t15\t0\t15\t-\tT\t10\t0\t10\t9\t15\t60\tcg:Z:5=5I5=\n"):
        res = check_break_against_oracle(ctx, line, 0)
        assert res["n_out"] == 2 and ((res["t_en"] - res["t_st"]) == 5).all()


@pytest.mark.parametrize("max_size", [0, 2, 10, 100])
@pytest.mark.parametrize("seed", range(4))
def test_break_paf_random(ctx, seed, max_size):
    paf_text, _ = gen.random_paf(600 + seed, n_contigs=4, recs_per_contig=8, style="all" if seed % 2 else "eqx", canonical=(seed < 2),
                                 allow_zero=(seed >= 2), clips=(seed == 3), max_ops=200)
    check_break_against_oracle(ctx, paf_text, max_size, policy=seed % 2)


@pytest.mark.parametrize("max_size", [10, 100, 1000])
def test_break_paf_bundled_fixture(ctx, max_size):
    res = check_break_against_oracle(ctx, orc.golden_paf(), max_size)
    assert res["n_out"] == {10: 5998, 100: 2447, 1000: 553}[max_size]


def test_break_paf_panics_like_the_reference(ctx):
    line = b"Q\t13\t0\t5\t+\tT\t13\t0\t8\t0\t0\t60\tcg:Z:3D5=\n"
    with pytest.raises(orc.ReferencePanic):
        orc.run_break_paf(line, 1)
    with pytest.raises(ReferencePanic):
        liftover.run_break_paf(ctx, line, 1)
    assert liftover.run_break_paf(ctx, b"", 1) == b""


# ---------------------------------------------------------------- liftover --qbed / --largest (SURVEY 8f.2)
def query_bed(paf_text, seed, width):
    """BED rows in QUERY coordinates (tiling every query), for --qbed."""
    qlens = {}
    for ln in paf_text.splitlines():
        f = ln.split(b"\t")
        qlens[f[0].decode()] = int(f[1])
    return gen.tiling_bed(qlens, width)


@pytest.mark.parametrize("seed", range(6))
def test_liftover_qbed_random(ctx, seed):
    # paf_swap_query_and_target (paf.rs:1050-1094): I <-> D, op order reversed on '-' strands, then the same liftover
    # (= X I D only: N / S / H keep their meaning across the swap, so a record holding one fails check_integrity in the
    #  reference as well — see the next test)
    paf_text, contigs = gen.random_paf(700 + seed, n_contigs=4, recs_per_contig=8, style="eqx",
                                       canonical=(seed < 4), allow_zero=(seed >= 4), clips=False, lead_trail=False)
    bed_text = query_bed(paf_text, seed, 7 + seed)
    want = orc.run_liftover(paf_text, bed_text, qbed=True, policy=seed % 2, threads=2)
    got = liftover.run_liftover(ctx, paf_text, bed_text, policy=seed % 2, qbed=True)
    assert got == want and len(want) > 0
    ctx.set_slicing(64)  # and through the sliced pipeline
    try:
        assert liftover.run_liftover(ctx, paf_text, bed_text, policy=seed % 2, qbed=True) == want
    finally:
        ctx.set_slicing()


def test_liftover_qbed_soft_clips_panic_like_the_reference(ctx):
    # S consumes the query on both sides of the swap, so the swapped record's target span no longer matches its CIGAR
    for line in (b"Q\t30\t0\t13\t+\tT\t40\t5\t15\t0\t0\t60\tcg:Z:3S10=\n", b"Q\t30\t0\t10\t-\tT\t40\t5\t20\t0\t0\t60\tcg:Z:5=5N5=\n"):
        with pytest.raises(orc.ReferencePanic):
            orc.run_liftover(line, b"Q\t0\t30\n", qbed=True)
        with pytest.raises(ReferencePanic):
            liftover.run_liftover(ctx, line, b"Q\t0\t30\n", qbed=True)


def test_liftover_qbed_bundled_fixture(ctx):
    paf_text = orc.golden_paf()
    bed_text = query_bed(paf_text, 0, 200_000)
    want = orc.run_liftover(paf_text, bed_text, qbed=True, threads=4)
    assert liftover.run_liftover(ctx, paf_text, bed_text, qbed=True) == want and want.count(b"\n") > 100


# ---------------------------------------------------------------- rb invert (SURVEY 8f.2): whole records, query <-> target
def check_invert_against_oracle(ctx, paf_text):
    want = orc.run_invert(paf_text)
    res = liftover.paf_swap_query_and_target(ctx, Paf.from_text(paf_text))
    assert res["paf_text"] == want
    rows = [ln.split(b"\t") for ln in want.splitlines()]
    assert res["n_out"] == len(rows)
    assert [int(r[7]) for r in rows] == res["t_st"].tolist() and [int(r[3]) for r in rows] == res["q_en"].tolist()
    assert [int(r[9]) for r in rows] == res["nmatch"].tolist() and [int(r[10]) for r in rows] == res["aln_len"].tolist()
    assert res["rec_idx"].tolist() == list(range(len(rows)))
    return want


def test_invert_reference_vectors(ctx):
    # paf.rs:1050-1065 on make_fake_paf_rec (paf.rs:1096-1100) and the two strands of one record
    assert check_invert_against_oracle(ctx, b"Q\t10\t2\t10\t-\tT\t20\t12\t20\t3\t9\t60\tcg:Z:4M1I1D3=\n") == \
        b"T\t20\t12\t20\t-\tQ\t10\t2\t10\t7\t9\t60\tid:Z:\tcg:Z:3=1I1D4M\n"
    assert check_invert_against_oracle(ctx, b"Q\t10\t2\t10\t+\tT\t20\t12\t20\t3\t9\t60\tcg:Z:4M1I1D3=\n") == \
        b"T\t20\t12\t20\t+\tQ\t10\t2\t10\t7\t9\t60\tid:Z:\tcg:Z:4M1D1I3=\n"


@pytest.mark.parametrize("seed", range(8))
def test_invert_random(ctx, seed):
    # nothing is stripped or merged: leading / trailing indels, repeated classes, zero lengths, clips and N all pass through
    paf_text, _ = gen.random_paf(900 + seed, n_contigs=4, recs_per_contig=8, style="all" if seed % 2 else "eqx", canonical=(seed < 4),
                                 allow_zero=(seed >= 4), clips=(seed in (3, 7)), max_ops=300)
    want = check_invert_against_oracle(ctx, paf_text)
    if seed % 2:
        # N and S keep their side across the swap, so the inverted record no longer passes check_integrity when it is read
        # back: the reference panics on its own output, and so does the GPU path
        with pytest.raises(orc.ReferencePanic):
            orc.run_invert(want)
        with pytest.raises(ReferencePanic):
            liftover.run_invert(ctx, want)
        return
    # involution: inverting twice gives the records back (12 columns + cg; tags are dropped, nmatch / aln_len re-inferred)
    assert liftover.run_invert(ctx, want) == orc.run_invert(want)
    twice = liftover.run_invert(ctx, want).splitlines()
    for a, b in zip(paf_text.splitlines(), twice):
        fa, fb = a.split(b"\t"), b.split(b"\t")
        assert fa[:9] == fb[:9] and fa[11] == fb[11]


def test_invert_bundled_fixture(ctx):
    want = check_invert_against_oracle(ctx, orc.golden_paf())
    assert want.count(b"\n") == 249
    assert liftover.run_invert(ctx, b"") == b""


def test_invert_panics_like_the_reference(ctx):
    # check_integrity at load (paf.rs:70) is on the record as read: spans that do not match the CIGAR panic ...
    bad = b"Q\t30\t0\t13\t+\tT\t40\t5\t16\t0\t0\t60\tcg:Z:3S10=\n"
    with pytest.raises(orc.ReferencePanic):
        orc.run_invert(bad)
    with pytest.raises(ReferencePanic):
        liftover.run_invert(ctx, bad)
    # ... while S / N, which keep their side across the swap, are fine when the spans are right
    for ok in (b"Q\t30\t0\t13\t+\tT\t40\t5\t15\t0\t0\t60\tcg:Z:3S10=\n", b"Q\t30\t0\t10\t-\tT\t40\t5\t20\t0\t0\t60\tcg:Z:5=5N5=\n",
               b"Q\t30\t0\t12\t-\tT\t40\t5\t15\t0\t0\t60\tcg:Z:2I4=1X3D2=3I\n"):
        check_invert_against_oracle(ctx, ok)


@pytest.mark.parametrize("seed", range(4))
def test_liftover_largest(ctx, seed):
    paf_text, contigs = gen.random_paf(800 + seed, n_contigs=3, recs_per_contig=10)
    for bed_text in (gen.tiling_bed(contigs, 25), gen.random_bed(seed, contigs, 60, with_ids=True), gen.random_bed(seed, contigs, 60, with_ids=False)):
        want = orc.run_liftover(paf_text, bed_text, largest=True, threads=1)
        assert liftover.run_liftover(ctx, paf_text, bed_text, largest=True) == want


# ---------------------------------------------------------------- multi-device context behind the C ABI (SURVEY 8e)
def test_multi_device_context_equals_single_and_oracle(monkeypatch):
    """rb_ctx_create with several device ids: rb_liftover / rb_stats partition the records over the devices (contiguous runs
    of the emission order, liftover.rs:151-164) and merge the rows into one output.  Two contexts on GPU 0 stand in for two
    GPUs here (the partition, the per-device threads and the merge are the same code); results == one device == oracle."""
    monkeypatch.setenv("RB_MULTI_MIN_BYTES", "0")
    one, two, three = capi.Context(0), capi.Context(devices=[0, 0]), capi.Context(devices=[0, 0, 0])
    try:
        for seed in (11, 12, 13):
            paf_text, contigs = gen.random_paf(seed, n_contigs=4, recs_per_contig=9, max_ops=300)
            lines = paf_text.splitlines(keepends=True)
            rng = np.random.default_rng(seed)
            paf_text = b"".join(lines[i] for i in rng.permutation(len(lines)))  # contigs interleave: emission order != file order
            bed_text = gen.tiling_bed(contigs, 40)
            hp = hostlib.HostPaf.from_text(paf_text)
            wins = hp.windows_from_bed_text(bed_text)
            want = orc.run_liftover(paf_text, bed_text)
            a = one.liftover(hp, wins, want=capi.WANT_TEXT | capi.WANT_NUMERIC, stats=True)
            assert a["paf_text"] == want
            for ctx in (two, three):
                b = ctx.liftover(hp, wins, want=capi.WANT_TEXT | capi.WANT_NUMERIC, stats=True)
                assert b["paf_text"] == want and b["n_pairs"] == a["n_pairs"]
                for k in ("line_off", "q_st", "q_en", "t_st", "t_en", "nmatch", "aln_len", "rec_idx", "win_idx"):
                    assert (a[k] == b[k]).all(), k
                for k in ("equal", "diff", "ins", "del", "ins_events", "del_events", "matches"):
                    assert (a["stats"][k] == b["stats"][k]).all(), k
                assert (a["stats"]["id_by_all"].view(np.uint32) == b["stats"]["id_by_all"].view(np.uint32)).all()
                st1, st2 = one.stats(hp), ctx.stats(hp)
                for k in st1:
                    assert np.array_equal(st1[k], st2[k], equal_nan=True) if k != "n" else st1[k] == st2[k], k
            # forced slices: dealt round-robin to the devices, rows land in one block in emission order
            for ctx in (two, three):
                ctx.set_slicing(64)
                try:
                    b = ctx.liftover(hp, wins, want=capi.WANT_TEXT | capi.WANT_NUMERIC, stats=True)
                    st = ctx.liftover(hp, wins, want=capi.WANT_STATS_TEXT, stats=False)
                finally:
                    ctx.set_slicing()
                assert b["paf_text"] == want and (a["rec_idx"] == b["rec_idx"]).all() and (a["line_off"] == b["line_off"]).all()
                assert (a["stats"]["equal"] == b["stats"]["equal"]).all()
                assert bamstats.print_cigar_stats_header().encode() + st["paf_text"] == orc.run_stats(want)
        # a reference panic on one device's share fails the whole call with that record's error
        name, ln = next(iter(contigs.items()))
        bad = paf_text + b"Q\t10\t0\t5\t+\t" + name.encode() + b"\t" + str(ln).encode() + b"\t0\t8\t0\t0\t60\tcg:Z:3D5=\n"
        hb = hostlib.HostPaf.from_text(bad)
        with pytest.raises(capi.RbError) as e1:
            one.liftover(hb, hb.windows_from_bed_text(bed_text))
        with pytest.raises(capi.RbError) as e2:
            two.liftover(hb, hb.windows_from_bed_text(bed_text))
        assert e1.value.code == e2.value.code
    finally:
        for c in (one, two, three):
            c.close()


# ---------------------------------------------------------------- RB_WANT_STATS_TEXT: `rb liftover | rb stats --paf` rows formatted on the device
def _stats_header():
    return bamstats.print_cigar_stats_header().encode()


@pytest.mark.parametrize("policy", [orc.RIGHTMOST, orc.EARLY_EXIT])
def test_stats_text_mode_is_liftover_piped_into_stats(policy):
    """bamstats.rs:225-270 on the rows of liftover.rs:107-167: the device prints the stats TSV rows itself (f32 identities with
    Rust's shortest-round-trip Display digits) — byte-identical to the oracle's `rb liftover | rb stats --paf`."""
    ctx = capi.Context(0)
    try:
        cases = [(orc.golden_paf(), orc.golden_bed())]
        for seed in (21, 22, 23, 24):
            paf_text, contigs = gen.random_paf(seed, n_contigs=3, recs_per_contig=8, max_ops=250, style="eqx" if seed % 2 else "mixed")
            cases.append((paf_text, gen.tiling_bed(contigs, 30 + seed, with_ids=bool(seed & 2))))
            cases.append((paf_text, gen.random_bed(seed, contigs, 60)))
        for paf_text, bed_text in cases:
            hp = hostlib.HostPaf.from_text(paf_text)
            wins = hp.windows_from_bed_text(bed_text)
            want = orc.run_stats(orc.run_liftover(paf_text, bed_text, policy=policy))
            got = ctx.liftover(hp, wins, policy=policy, want=capi.WANT_STATS_TEXT, stats=True)
            assert _stats_header() + got["paf_text"] == want
            assert got["line_off"][-1] == len(got["paf_text"]) and got["n_out"] == want.count(b"\n") - 1
            # forced slices and the multi-device merge carry the same rows
            ctx.set_slicing(64)
            try:
                assert ctx.liftover(hp, wins, policy=policy, want=capi.WANT_STATS_TEXT, stats=False)["paf_text"] == got["paf_text"]
            finally:
                ctx.set_slicing()
        with pytest.raises(capi.RbError):
            ctx.liftover(hp, wins, want=capi.WANT_STATS_TEXT | capi.WANT_TEXT)
    finally:
        ctx.close()


def test_stats_text_identity_edge_values():
    """Identities that are exact integers, exact ties (round up, not to even), NaN (0 / 0 cannot happen for a lifted row, but
    100 * 0 / n = 0 does) and long fractions: rows whose CIGARs are built to hit them."""
    ctx = capi.Context(0)
    try:
        lines = []
        for i, cg in enumerate(["2049=10751X", "1=1X", "10=", "3X", "1=2X", "7=1X1=3I", "1=99999X", "12345=1X", "999=1X2D5="]):
            t = sum(int(x) for x in __import__("re").findall(r"(\d+)[=XD]", cg))
            q = sum(int(x) for x in __import__("re").findall(r"(\d+)[=XI]", cg))
            lines.append(f"q{i}\t{q + 10}\t0\t{q}\t+\tchr1\t20000000\t{i * 200000}\t{i * 200000 + t}\t0\t0\t60\tcg:Z:{cg}\n".encode())
        paf_text = b"".join(lines)
        bed_text = b"chr1\t0\t20000000\n"
        hp = hostlib.HostPaf.from_text(paf_text)
        got = ctx.liftover(hp, hp.windows_from_bed_text(bed_text), want=capi.WANT_STATS_TEXT, stats=False)
        want = orc.run_stats(orc.run_liftover(paf_text, bed_text))
        assert _stats_header() + got["paf_text"] == want
        assert b"\t16.007813\t" in got["paf_text"] and b"\t100\t" in got["paf_text"] and b"\t0\t0\t0\t0\t3\t" in got["paf_text"]
    finally:
        ctx.close()


def test_fused_tokeniser_scan_kernel_opt_in():
    """RB_TOKSCAN=1 (k_tok_scan: tokeniser + sample scan in one kernel, absolute sub-samples) gives the same bytes: the
    random / tiling / non-canonical / tiny-record / panic cases of this file once more in a process that has it switched on."""
    import os
    import subprocess
    import sys
    if os.environ.get("RB_TOKSCAN"):
        pytest.skip("already inside the RB_TOKSCAN=1 run")
    env = dict(os.environ, RB_TOKSCAN="1")
    sel = "c1_ or random_eqx or random_sliced or all_ops or tiny_records or long_numbers or reference_panics or integrity or break_paf_random"
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-m", "gpu", "-k", sel],
                       env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
