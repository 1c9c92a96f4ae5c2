#!/usr/bin/env python
"""bench.py — PAF liftover + stats hot path on B200 (the metric of BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--haps H] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload, the SAME FIXED JOB at every N ("scaling": "strong"): BASELINE.json's C5 — H = 94 synthetic haplotypes
vs the CHM13-like reference concatenated (haplotype-major file order), `rb liftover --bed <10 kb tiling windows>` + the
per-row `rb stats --paf` counters.  A step = one pass of the hot path over the whole job.
  value  lifted window-records/s with the inputs resident in HBM: one process per GPU, rank r holds the records of its
         target contigs (LPT over the contigs on their length ~ CIGAR bytes; no collective on the data path), CUDA events on
         the stream the library launches on, max over ranks.
  e2e    the same job through the reference-facing C-ABI call rb_liftover() with HOST buffers in and pinned host buffers
         out, copies inside the timed region.  N = 1: the call's sliced pipeline on one device.  N > 1: ONE call on an
         N-device rb_ctx made by rank 0 (partition in C++, one host thread per GPU, rows merged in emission order into one
         output — all inside the timed region); the per-rank form (every rank lifts its own shard) is reported beside it.
At N = 1 the line also carries "c4": BASELINE's C4 (one haplotype, 1 kb windows: the workload of round 1's headline) with its
own resident / e2e / per-kernel roofline numbers, and the rows of a few contigs of BOTH workloads are compared byte for byte
with the CPU oracle ("parity_checked_rows").
--dump-outputs DIR: what the last timed resident step of C4 and C5 computed (the PAF rows, their line offsets and the stats
counters), as a fixed, seeded sample of rows in DIR/<name>.npy, so that two builds can be compared output for output.  The
synthetic inputs depend only on the arguments.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "lifted window-records/s"
UNIT = "records/s"
CONTIG_LEN = [248387328, 242696752, 201105948, 193574945, 182045439, 172126628, 160567428, 146259331, 150617247, 134758134,
              135127769, 133324548, 113566686, 101161492, 99753195, 96330374, 84276897, 80542538, 61707364, 66210255, 45090682,
              51324926, 154259566, 62460029, 16569]
CONTIG_NAME = [f"chr{i}" for i in range(1, 23)] + ["chrX", "chrY", "chrM"]
C5_WINDOW, C4_WINDOW = 10_000, 1_000
REF_SAMPLE_CONTIGS = ["chr21", "chr22", "chrM"]  # --impl reference, per step: ~96 Mbp of one haplotype
CPU_BASELINE_CONTIGS = ["chr16", "chr17", "chr18", "chr19", "chr20", "chr21", "chr22", "chrM"]  # cpu_baseline: ~0.5 Gbp, one pass
C4_PARITY_CONTIGS = ["chr20", "chr21", "chr22", "chrM"]
DTYPE = "u32/u64 (+f32 identities)"
# --dump-outputs, per workload: rows drawn, and bytes of their text kept (4 B each as float32): ~22 MB, C4 + C5 under 64 MB
DUMP_ROWS, DUMP_TEXT_BYTES, DUMP_SEED = 65536, 4 << 20, 0
STATS_U32 = ("equal", "diff", "ins", "del", "ins_events", "del_events", "matches")
STATS_F32 = ("id_by_matches", "id_by_events", "id_by_all")


def workload_name(haps):
    return (f"C5: {haps} synthetic haplotypes vs CHM13-like concatenated (haplotype-major), rb liftover --bed <10 kb tiling windows> "
            "+ per-row rb stats --paf")


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        # median over the samples taken under load (an idle GPU between the timed loops parks its clock)
        busy = [x for x in sm if x >= 0.5 * (max(mx) if mx else 0)] or sm
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(self.rows)}


def lpt_contigs(world):
    """Target contigs -> ranks: longest-processing-time-first on the contig length (CIGAR bytes are proportional to it)."""
    loads, bins = [0] * world, [[] for _ in range(world)]
    for c in sorted(range(len(CONTIG_LEN)), key=lambda c: -CONTIG_LEN[c]):
        b = loads.index(min(loads))
        bins[b].append(c)
        loads[b] += CONTIG_LEN[c]
    return [sorted(b) for b in bins], max(loads) / (sum(loads) / world)


def sample_texts(paf, contig_names, window, first_run_only=True):
    """PAF + BED text of the records of `contig_names` (first haplotype only) and their record ranges in `paf`."""
    import numpy as np
    t_id = np.ctypeslib.as_array(paf.c.t_id, shape=(paf.n_rec,))
    texts, beds, ranges = [], [], []
    for nm in contig_names:
        tid = paf.find_name(nm)
        if tid < 0:
            continue
        r = np.flatnonzero(t_id == tid)
        cuts = np.flatnonzero(np.diff(r) != 1) + 1
        lo, hi = int(r[0]), int((r[cuts[0] - 1] if len(cuts) else r[-1])) + 1  # the first run = the first haplotype's records
        texts.append(paf.text(lo, hi))
        beds.append(paf.tiling_bed_text(window, tid))
        ranges.append((lo, hi))
    return b"".join(texts), b"".join(beds), ranges


def check_rows_against_oracle(views, paf, ranges, oracle_lifted, oracle_stats):
    """GPU rows of the records in `ranges` (consecutive runs, one per sampled contig, in the oracle's order) == the bytes the
    oracle printed for them (`rb liftover`) and the `rb stats --paf` rows of those bytes.  Returns the number of rows compared."""
    import numpy as np
    from rustybam_b200 import hostlib
    idx = views["rec_idx"]
    off = views["line_off"]
    got_text, got_rows = [], []
    for lo, hi in ranges:
        rows = np.flatnonzero((idx >= lo) & (idx < hi))
        if len(rows) == 0:
            continue
        assert rows[-1] - rows[0] + 1 == len(rows), "rows of one contig are one contiguous run"
        r0, r1 = int(rows[0]), int(rows[-1]) + 1
        got_text.append(views["paf_text"][int(off[r0]):int(off[r1])].tobytes())
        got_rows.append((r0, r1))
    lifted = b"".join(got_text)
    if lifted != oracle_lifted:
        raise SystemExit("PARITY FAILURE: lifted rows differ from the CPU oracle")
    st_text, hdr = [], None
    for (r0, r1), t in zip(got_rows, got_text):
        s = hostlib.HostPaf.from_text(t).stats_text(views["stats"], row0=r0, header=hdr is None)
        hdr = True
        st_text.append(s)
    if b"".join(st_text) != oracle_stats:
        raise SystemExit("PARITY FAILURE: fused stats rows differ from the CPU oracle")
    return sum(b - a for a, b in got_rows)


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the host cores.  The Rust binary cannot be
    built in this image (no cargo/rustc, no network), so this is the oracle port; each step = a bounded sample of the C5 job."""
    if rank != 0:
        return
    import orc
    from rustybam_b200 import build, hostlib
    build.build_host()
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
    threads = os.cpu_count() or 8  # `rb -t N`: every host core (the reference's default is -t 8, cli.rs:17-19)
    cont = [CONTIG_NAME.index(c) for c in REF_SAMPLE_CONTIGS]
    paf = hostlib.HostPaf.synth(scale=1.0, n_hap=1, threads=min(8, threads), contigs=cont)
    paf_text, bed_text, ranges = sample_texts(paf, REF_SAMPLE_CONTIGS, C5_WINDOW)
    nrec = sum(b - a for a, b in ranges)
    times, rows = [], 0
    for i in range(args.warmup + args.steps):
        r = orc.bench_pipeline(paf_text, bed_text, threads=threads)
        if i >= args.warmup:
            times.append(r["secs_liftover"] + r["secs_stats"])
        rows = r["rows"]
    sec = sum(times) / len(times)
    value = rows / sec
    sample = (f"one haplotype's records of {'+'.join(REF_SAMPLE_CONTIGS)} ({nrec} records, {len(paf_text) / 1e6:.1f} MB PAF text) x their 10 kb "
              f"windows -> {rows} rows per step; text -> text: PAF parse + liftover + print + stats re-parse + stats print; restated "
              "reference CPU path (oracle/), not the rb binary")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": workload_name(args.haps), "window_bp": C5_WINDOW, "sample_per_step": "+".join(REF_SAMPLE_CONTIGS) + " of one haplotype",
                       "host_cores": os.cpu_count(), "same_config": False,
                       "note": "a step of this arm is a 3 % sample of ONE of the job's haplotypes; the B200 arm times the whole job, and "
                               "also this very sample (its `same_sample` object) for a like-for-like ratio"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def bind_to_gpu_numa_node(index):
    """Host side of the e2e path: run this rank's threads (and so first-touch its page-locked buffers) on the NUMA
    node the GPU's PCIe root hangs off.  Returns (node, n_cpus, previous affinity) or None (single-node hosts: no-op)."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(index)  # CUDA's numbering (honours CUDA_VISIBLE_DEVICES), unlike NVML's
        path = f"/sys/bus/pci/devices/{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        before = os.sched_getaffinity(0)
        cpus &= before
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node, len(cpus), before
    except Exception:
        return None


class Pinner:
    """Page-locks the big host buffers of a packed PAF / window table (rb_host_register) for asynchronous DMA."""

    def __init__(self, lib):
        self.lib, self.addrs = lib, []

    def pin(self, paf, wins):
        ids_bytes = int(wins.c.ids_off[wins.n_win]) if wins.c.ids_off else 0  # 3-column BED: ids are formatted on the GPU
        for ptr, nbytes in ((paf.c.cigar, paf.cigar_nbytes), (wins.c.st, wins.n_win * 8), (wins.c.en, wins.n_win * 8),
                            (wins.c.ids, ids_bytes), (wins.c.ids_off, (wins.n_win + 1) * 8 if ids_bytes else 0),
                            (wins.c.bed_row, wins.n_win * 4), (wins.c.t_id, wins.n_win * 4)):
            addr = C.cast(ptr, C.c_void_p).value
            if addr and nbytes and self.lib.rb_host_register(C.c_void_p(addr), nbytes) == 0:
                self.addrs.append(addr)
        return ids_bytes

    def release(self):
        for a in self.addrs:
            self.lib.rb_host_unregister(C.c_void_p(a))
        self.addrs = []


def algorithmic_bytes(summ, n_win, n_rec):
    """SURVEY §8(d): compulsory bytes of one liftover(+fused stats) step, and per kernel given the layout of DESIGN §3."""
    n_ops, n_pairs, n_out = summ["n_ops"], summ["n_pairs"], summ["n_out"]
    out_bytes, cigar_bytes = summ["out_bytes"], summ["cigar_bytes"]
    # 1 sample + 3 sub-samples of 48 B per 32-op chunk; wide windows (more than 64 ops per pair): the sample only (rbcuda.cu, RB_SUBS)
    smp_bytes = (n_ops // 32) * 48 * (1 if (n_pairs and n_ops > 64 * n_pairs) else 4)
    per_kernel = {
        "k_tokenise": cigar_bytes + 4 * n_ops,                       # text in, one 4-byte op word out
        "k_samples": 4 * n_ops + smp_bytes,                          # op words in, samples out
        "k_scan_lift": 4 * n_ops + smp_bytes + 16 * n_win + 128 * n_pairs,
        "k_combine": n_pairs * (128 + 16 + 112 + 4),
        "k_lift": n_pairs * (16 + 112 + 4) + 4 * n_ops + smp_bytes,  # (only the blocks k_emit does not lift itself)
        # fused lift + line scan + serialiser: windows (16 B), every op word and sample block in; every output byte, the stats
        # row (40 B) and the line offset (8 B) out — no per-pair intermediate
        "k_emit": n_pairs * 16 + 4 * n_ops + smp_bytes + out_bytes + n_out * 48,
        "k_serialise": n_pairs * (112 + 8) + out_bytes + n_out * (40 + 8) + cigar_bytes,
        "k_scan_lines": n_pairs * (4 + 16),
    }
    whole = cigar_bytes + 8 * (n_rec + 1) + 49 * n_rec + 20 * n_win + out_bytes + 40 * n_out + 8 * (n_out + 1)
    return per_kernel, whole


def sample_outputs(views, prefix, share=1.0):
    """A fixed, seeded sample of one liftover's outputs as float arrays: the line offset, length and stats counters of
    `share` * DUMP_ROWS rows drawn without replacement (u32 / u64 values are exact in float64, the f32 identities stay f32),
    the text bytes of the first drawn rows that fit `share` * DUMP_TEXT_BYTES (as float32), the row count and byte total, and
    every counter summed over all rows."""
    import numpy as np
    n = views["n_out"]
    off, text, st = views["line_off"], views["paf_text"], views["stats"]
    drawn = np.random.default_rng(DUMP_SEED).choice(n, size=min(n, int(DUMP_ROWS * share)), replace=False)
    rows = np.sort(drawn)
    start, end = off[rows].astype(np.int64), off[rows + 1].astype(np.int64)
    out = {"counts": np.array([n, views["n_pairs"], views["paf_nbytes"]], dtype=np.float64),
           "rows": rows.astype(np.float64), "line_off": start.astype(np.float64), "line_len": (end - start).astype(np.float64),
           "stats_totals": np.array([st[k].sum(dtype=np.uint64) for k in STATS_U32], dtype=np.float64)}
    out.update({k: st[k][rows].astype(np.float64) for k in STATS_U32})
    out.update({k: st[k][rows].astype(np.float32) for k in STATS_F32})
    lens = (off[drawn + 1] - off[drawn]).astype(np.int64)
    text_rows = np.sort(drawn[:int(np.searchsorted(np.cumsum(lens), DUMP_TEXT_BYTES * share, side="right"))])
    out["text_rows"] = text_rows.astype(np.float64)
    out["text"] = np.concatenate([text[int(off[r]):int(off[r + 1])] for r in text_rows] or [np.zeros(0, np.uint8)]).astype(np.float32)
    return {f"{prefix}_{k}": v for k, v in out.items()}


def write_outputs(directory, arrays):
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def measure_resident(torch, ctx, stream, flush, paf, wins, steps, warmup, barrier, dump=None, dump_share=1.0):
    """W + K resident steps (inputs uploaded once), then a pass with CUDA events around every kernel.  dump: a name prefix
    under which the outputs of the last timed step are sampled (sample_outputs) into the result's "dump"."""
    from rustybam_b200 import capi
    b = ctx.upload(paf, wins)
    summ = None
    for _ in range(warmup):
        summ = ctx.batch_liftover(b, with_stats=True, want=capi.WANT_TEXT)
    barrier()
    step_ms = []
    for _ in range(steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        summ = ctx.batch_liftover(b, with_stats=True, want=capi.WANT_TEXT)
        e1.record(stream)
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
    barrier()
    dumped = None
    if dump:
        views, release = ctx.batch_download_lift_view(b, want=capi.WANT_TEXT, stats=True)
        dumped = sample_outputs(views, dump, dump_share)
        release()
        barrier()
    ctx.set_profiling(True)
    ctx.kernel_times(reset=True)
    n_prof = max(3, steps // 4)
    prof_ms = []
    for _ in range(n_prof):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ctx.batch_liftover(b, with_stats=True, want=capi.WANT_TEXT)
        e1.record(stream)
        e1.synchronize()
        prof_ms.append(e0.elapsed_time(e1))
    torch.cuda.synchronize()
    ktimes = ctx.kernel_times(reset=True)
    ctx.set_profiling(False)
    ctx.batch_free(b)
    return dict(ms=sum(step_ms) / len(step_ms), summ=summ, ktimes=ktimes, n_prof=n_prof, prof_ms=sum(prof_ms) / len(prof_ms), dump=dumped)


def measure_e2e(ctx, paf, wins, steps, warmup, barrier, stream=None, torch=None, flush=None, want=None):
    """rb_liftover() with host buffers in / pinned host buffers out, W + K calls.  Timed with CUDA events on the context's stream
    when it has one the bench can see (single device), else by the host clock around the blocking call (multi-device context:
    the call returns when every device's rows have landed in the merged output)."""
    from rustybam_b200 import capi
    want = capi.WANT_TEXT if want is None else want
    with_stats = want == capi.WANT_TEXT  # (the stats rows carry the counters as text: no numeric copy beside them)
    t0 = time.perf_counter()
    r = ctx.liftover(paf, wins, want=want, stats=with_stats, copy=False)
    first_ms = (time.perf_counter() - t0) * 1e3
    for _ in range(max(0, warmup - 1)):
        ctx.liftover(paf, wins, want=want, stats=with_stats, copy=False)
    barrier()
    ms = []
    for _ in range(steps):
        if flush is not None:
            flush.fill_(1)
        if stream is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            r = ctx.liftover(paf, wins, want=want, stats=with_stats, copy=False)
            e1.record(stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        else:
            if torch is not None:
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = ctx.liftover(paf, wins, want=want, stats=with_stats, copy=False)
            ms.append((time.perf_counter() - t0) * 1e3)
    barrier()
    return dict(ms=sum(ms) / len(ms), first_call_ms=first_ms, n_out=r["n_out"], out_bytes=r["paf_nbytes"], n_pairs=r["n_pairs"])


def copy_bytes(paf, wins, ids_bytes, n_out, out_bytes):
    h2d = paf.cigar_nbytes + paf.n_rec * (8 * 8 + 1 + 8) + wins.n_win * (8 + 8 + 4) + ((wins.n_win + 1) * 8 + ids_bytes if ids_bytes else 0)
    d2h = out_bytes + (n_out + 1) * 8 + n_out * 40
    return int(h2d), int(d2h)


def roofline_of(res, wins_n, n_rec, peak, peak_src, traffic_key):
    alg, whole = algorithmic_bytes(res["summ"], wins_n, n_rec)
    ktimes = res["ktimes"]
    total_k = sum(ms for _, ms in ktimes.values()) or 1.0
    if "k_emit" in ktimes and "k_lift" in ktimes and ktimes["k_lift"][1] < 0.25 * ktimes["k_emit"][1]:
        alg.pop("k_lift")  # k_emit lifted (nearly) every block itself: k_lift only saw the few it could not, its formula does not apply
    dom = max((k for k in ktimes if k in alg), key=lambda k: ktimes[k][1])
    launches, ms_sum = ktimes[dom]
    dom_ms = ms_sum / max(launches, 1)
    achieved = alg[dom] / (dom_ms * 1e-3) / 1e9
    # measured DRAM bytes per launch of that kernel (ncu --set full, profiles/traffic.json: one haplotype), scaled to this launch's CIGAR bytes
    traffic, step_traffic = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            t = json.load(open(tpath))
            scale = res["summ"]["cigar_bytes"] / t["cigar_bytes"]
            traffic = int(t[traffic_key][dom] * scale) if dom in t[traffic_key] else None
            step_traffic = int(t[traffic_key + "_step_total"] * scale)
        except Exception:
            traffic = None
    return {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": int(alg[dom]),
            "kernel_ms": dom_ms, "kernel_share_of_step": ms_sum / total_k, "step_ms_with_per_kernel_events": res["prof_ms"],
            "all_kernels_ms": {k: v[1] / max(v[0], 1) for k, v in ktimes.items()},
            "all_kernels_frac": {k: (alg[k] / (v[1] / max(v[0], 1) * 1e-3) / 1e9) / peak for k, v in ktimes.items() if k in alg},
            # SURVEY §8(d): the step's compulsory bytes (text in, windows, coordinates, every output byte, stats rows) over the
            # WHOLE resident step — intermediates are not counted
            "whole_step": {"algorithmic_bytes": int(whole), "ms": res["ms"], "achieved": whole / (res["ms"] * 1e-3) / 1e9,
                           "frac": whole / (res["ms"] * 1e-3) / 1e9 / peak, "dram_traffic": step_traffic,
                           "traffic_over_algorithmic": (step_traffic / whole) if step_traffic else None}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--haps", type=int, default=94, help="haplotypes of the fixed C5 job")
    ap.add_argument("--scale", type=float, default=1.0, help="genome scale (1.0 = ~3.1 Gbp, the BASELINE configs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--only-c4", action="store_true", help="only the C4 sub-bench (one haplotype, 1 kb windows): tuning runs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs samples the outputs of the B200 path; --impl reference has none to sample")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import numpy as np
    import torch
    import torch.distributed as dist
    from rustybam_b200 import build, capi, hostlib

    if rank == 0:
        build.build_all()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if not os.environ.get("RB_BENCH_NO_NUMA") else None
    cpu_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")  # host-side waits that must not occupy the GPUs
    ncpu = os.cpu_count() or 8

    lib = capi.load()
    ctx = capi.Context(local_rank)
    # a real (non-default) stream: the library launches on it and the CUDA events are recorded on it (handle 0 would mean
    # "use your own stream" in the C ABI, and events on torch's default stream would not bracket the kernels)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ctx.set_stream(stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > L2 (126 MB): written between timed steps

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    peak, peak_src = measured_peak()
    sampler = ClockSampler(local_rank)
    sampler.start()
    line = {}

    # =============================== C4 (N = 1 only): one haplotype, 1 kb windows ===============================
    c4 = None
    if world == 1:
        paf4 = hostlib.HostPaf.synth(scale=args.scale, n_hap=1, threads=ncpu)
        wins4 = paf4.tiling_windows(C4_WINDOW)
        pin4 = Pinner(lib)
        ids4 = pin4.pin(paf4, wins4)
        r4 = measure_resident(torch, ctx, stream, flush, paf4, wins4, args.steps, args.warmup, barrier, dump=args.dump_outputs and "c4")
        if args.dump_outputs:
            write_outputs(args.dump_outputs, r4["dump"])
        e4 = measure_e2e(ctx, paf4, wins4, args.steps, args.warmup, barrier, stream, torch, flush)
        h2d4, d2h4 = copy_bytes(paf4, wins4, ids4, e4["n_out"], e4["out_bytes"])
        t4 = measure_e2e(ctx, paf4, wins4, args.steps, args.warmup, barrier, stream, torch, flush, want=capi.WANT_STATS_TEXT)
        s4 = r4["summ"]
        c4 = {"workload": "C4: rb liftover --bed <1 kb tiling windows> over synthetic HG002-vs-CHM13-scale eqx PAF + per-row rb stats --paf",
              "value": s4["n_out"] / (r4["ms"] * 1e-3), "unit": UNIT, "ms_per_step": r4["ms"], "records": paf4.n_rec, "bed_rows": wins4.n_win,
              "pairs": s4["n_pairs"], "rows": s4["n_out"], "cigar_ops": s4["n_ops"], "cigar_bytes": s4["cigar_bytes"], "out_bytes": s4["out_bytes"],
              "cigar_gb_per_s": s4["cigar_bytes"] / (r4["ms"] * 1e-3) / 1e9,
              "e2e": {"value": e4["n_out"] / (e4["ms"] * 1e-3), "unit": UNIT, "ms_per_step": e4["ms"], "first_call_ms": e4["first_call_ms"],
                      "h2d_bytes_per_step": h2d4, "d2h_bytes_per_step": d2h4},
              # the pipeline's FINAL output (`rb liftover | rb stats --paf` rows, formatted on the device) instead of PAF rows + counters
              "e2e_stats_text": {"value": t4["n_out"] / (t4["ms"] * 1e-3), "unit": UNIT, "ms_per_step": t4["ms"], "h2d_bytes_per_step": h2d4,
                                 "d2h_bytes_per_step": int(t4["out_bytes"] + (t4["n_out"] + 1) * 8)},
              "gpu_launches_per_step": int(sum(v[0] for v in r4["ktimes"].values()) // r4["n_prof"]),
              "roofline": roofline_of(r4, wins4.n_win, paf4.n_rec, peak, peak_src, "c4")}
        if not args.no_cpu_baseline:  # rows of a few contigs of the full-size call against the CPU oracle, byte for byte
            import orc
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
            ptxt, btxt, ranges = sample_texts(paf4, C4_PARITY_CONTIGS, C4_WINDOW)
            want = orc.bench_pipeline_keep(ptxt, btxt, threads=ncpu)
            views, release = ctx.liftover_view(paf4, wins4, want=capi.WANT_TEXT | capi.WANT_NUMERIC, stats=True)
            c4["parity_checked_rows"] = check_rows_against_oracle(views, paf4, ranges, want["lifted"], want["stats"])
            release()
        pin4.release()
        wins4.close()
        paf4.close()
        if args.only_c4:
            line = dict(c4)
            line.update({"metric": METRIC, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "clocks": sampler.stop()})
            print(json.dumps(line))
            ctx.close()
            return

    # =============================== C5: the fixed job, this rank's contigs resident ===============================
    bins, balance = lpt_contigs(world)
    t0 = time.time()
    shard = hostlib.HostPaf.synth(scale=args.scale, n_hap=args.haps, threads=max(1, ncpu // world), contigs=bins[rank])
    wins = shard.tiling_windows(C5_WINDOW)
    gen_s = time.time() - t0
    pin = Pinner(lib)
    ids_bytes = pin.pin(shard, wins)
    res = measure_resident(torch, ctx, stream, flush, shard, wins, args.steps, args.warmup, barrier,
                           dump=args.dump_outputs and ("c5" if world == 1 else f"c5_rank{rank}"), dump_share=1.0 / world)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, res["dump"])
    # per-rank end to end: every rank lifts its own shard through rb_liftover (host buffers both ways)
    e2e_rank = measure_e2e(ctx, shard, wins, args.steps, args.warmup, barrier, stream, torch, flush)
    e2e_st = measure_e2e(ctx, shard, wins, args.steps, args.warmup, barrier, stream, torch, flush, want=capi.WANT_STATS_TEXT)
    summ = res["summ"]
    h2d, d2h = copy_bytes(shard, wins, ids_bytes, e2e_rank["n_out"], e2e_rank["out_bytes"])
    tot = torch.tensor([float(summ["n_out"]), float(summ["cigar_bytes"]), float(summ["out_bytes"]), float(summ["n_pairs"]),
                        float(summ["n_ops"]), float(h2d), float(d2h), float(shard.n_rec), float(wins.n_win)], dtype=torch.float64, device="cuda")
    tmax = torch.tensor([res["ms"], e2e_rank["ms"], e2e_rank["first_call_ms"], e2e_st["ms"]], dtype=torch.float64, device="cuda")
    st_bytes = torch.tensor([float(e2e_st["out_bytes"] + (e2e_st["n_out"] + 1) * 8)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(st_bytes, op=dist.ReduceOp.SUM)
    st_bytes = st_bytes.item()
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    tot, tmax = tot.tolist(), tmax.tolist()

    # ---- N > 1: the whole job through ONE rb_liftover call on an N-device context (rank 0; the other ranks step aside) ----
    multi = None
    if world > 1:
        pin.release()
        wins.close()
        shard.close()
        ctx.close()
        del flush
        torch.cuda.empty_cache()
        torch.cuda.synchronize()
        dist.barrier(group=cpu_group)  # every rank has released its GPU
        if rank == 0:
            t0 = time.time()
            full = hostlib.HostPaf.synth(scale=args.scale, n_hap=args.haps, threads=ncpu)
            fwins = full.tiling_windows(C5_WINDOW)
            gen_full_s = time.time() - t0
            pinf = Pinner(lib)
            idsf = pinf.pin(full, fwins)
            mctx = capi.Context(devices=list(range(world)))
            m = measure_e2e(mctx, full, fwins, args.steps, args.warmup, lambda: None, None, torch, None)
            mst = measure_e2e(mctx, full, fwins, args.steps, args.warmup, lambda: None, None, torch, None, want=capi.WANT_STATS_TEXT)
            hf, df = copy_bytes(full, fwins, idsf, m["n_out"], m["out_bytes"])
            multi = {"ms": m["ms"], "first_call_ms": m["first_call_ms"], "n_out": m["n_out"], "h2d": hf, "d2h": df, "gen_s": gen_full_s,
                     "records": full.n_rec, "st_ms": mst["ms"], "st_d2h": int(mst["out_bytes"] + (mst["n_out"] + 1) * 8)}
            if not args.no_cpu_baseline:  # the merged output of the N-device call against the oracle (first haplotype, a few contigs)
                import orc
                subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
                ptxt, btxt, ranges = sample_texts(full, REF_SAMPLE_CONTIGS, C5_WINDOW)
                want = orc.bench_pipeline_keep(ptxt, btxt, threads=ncpu)
                views, release = mctx.liftover_view(full, fwins, want=capi.WANT_TEXT | capi.WANT_NUMERIC, stats=True)
                multi["parity_checked_rows"] = check_rows_against_oracle(views, full, ranges, want["lifted"], want["stats"])
                release()
            pinf.release()
            mctx.close()
        dist.barrier(group=cpu_group)

    if rank == 0:
        clocks = sampler.stop()
        n_out_total = tot[0]
        e2e_ms = multi["ms"] if multi else tmax[1]
        e2e = {"value": n_out_total / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": int(multi["h2d"] if multi else tot[5]), "d2h_bytes_per_step": int(multi["d2h"] if multi else tot[6]),
               "cigar_gb_per_s": tot[1] / (e2e_ms * 1e-3) / 1e9, "first_call_ms": multi["first_call_ms"] if multi else tmax[2],
               "how": (f"ONE rb_liftover() call on a {world}-device rb_ctx from rank 0: partition (C++, contiguous runs of the emission order "
                       "balanced on CIGAR bytes), per-device uploads / kernels / downloads and the merge into one pinned output are all inside "
                       "the timed region (host clock around the blocking call)") if multi else
                      "rb_liftover() on one device: sliced pipeline, CUDA events on the library's stream around the call"}
        st_ms = multi["st_ms"] if multi else tmax[3]
        e2e["stats_text"] = {"value": n_out_total / (st_ms * 1e-3), "ms_per_step": st_ms, "d2h_bytes_per_step": int(multi["st_d2h"] if multi else st_bytes),
                             "how": "the same call with RB_WANT_STATS_TEXT: the pipeline's final output (`rb liftover | rb stats --paf` rows, formatted on "
                                    "the device) comes back instead of PAF rows + counters"}
        if multi:
            e2e["per_rank_form"] = {"value": n_out_total / (tmax[1] * 1e-3), "ms_per_step": tmax[1],
                                    "how": "every rank lifts its own contig shard through rb_liftover on its GPU; max over ranks; no merge"}
            if "parity_checked_rows" in multi:
                e2e["parity_checked_rows"] = multi["parity_checked_rows"]
        roof = roofline_of(res, wins.n_win if world == 1 else int(tot[8] / world), int(tot[7] / world) if world > 1 else shard.n_rec, peak, peak_src, "w10k")
        line = {
            "metric": METRIC, "value": n_out_total / (tmax[0] * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": tmax[0], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": workload_name(args.haps), "haplotypes": args.haps, "window_bp": C5_WINDOW, "scale": args.scale,
                       "records": int(tot[7]), "bed_rows_all_ranks": int(tot[8]), "pairs": int(tot[3]), "rows": int(tot[0]), "cigar_ops": int(tot[4]),
                       "cigar_bytes": int(tot[1]), "out_bytes": int(tot[2]),
                       "partition": "resident: target contigs over the ranks, LPT on contig length (~ CIGAR bytes), no collective; e2e (N > 1): "
                                    "contiguous runs of the emission order inside the C-ABI call, balanced on CIGAR bytes",
                       "lpt_balance": balance, "l2": "256 MiB buffer written between timed steps (L2 flush); inputs+outputs > L2"},
            "cigar_gb_per_s": tot[1] / (tmax[0] * 1e-3) / 1e9,
            "e2e": e2e,
            "gpu_launches": int(sum(v[0] for v in res["ktimes"].values()) // res["n_prof"]) * args.steps,
            "clocks": clocks,
            "roofline": roof,
            "gen_s": gen_s,
        }
        if c4 is not None:
            line["c4"] = c4
        line["numa"] = {"node": numa[0], "cpus": numa[1]} if numa else None
        if numa:
            os.sched_setaffinity(0, numa[2])  # the CPU baseline gets every host core back
        if not args.no_cpu_baseline:
            import orc
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
            cont = [CONTIG_NAME.index(c) for c in CPU_BASELINE_CONTIGS]
            one = hostlib.HostPaf.synth(scale=args.scale, n_hap=1, threads=ncpu, contigs=cont)
            ptxt, btxt, ranges = sample_texts(one, CPU_BASELINE_CONTIGS, C5_WINDOW)
            want = orc.bench_pipeline_keep(ptxt, btxt, threads=ncpu)
            sec = want["secs_liftover"] + want["secs_stats"]
            nrec = sum(b - a for a, b in ranges)
            line["cpu_baseline"] = {
                "value": want["rows"] / sec, "unit": UNIT, "cores": ncpu, "kind": "port", "host_cores": ncpu, "seconds": sec,
                "sample": f"one haplotype's records of {'+'.join(CPU_BASELINE_CONTIGS)} ({nrec} records, {len(ptxt) / 1e6:.0f} MB PAF text) x their 10 kb "
                          f"windows -> {want['rows']} rows; restated reference CPU path (oracle/), not the rb binary; text -> text (PAF parse + liftover + "
                          "print + stats re-parse + stats print)"}
            # the SAME sample on the GPU: (a) through rb_liftover from packed host buffers, (b) text -> text like the CPU arm
            sctx = capi.Context(0)
            swins = one.tiling_windows(C5_WINDOW)
            for _ in range(3):
                sctx.liftover(one, swins, want=capi.WANT_TEXT, stats=True, copy=False)
            t0 = time.perf_counter()
            for _ in range(5):
                sctx.liftover(one, swins, want=capi.WANT_TEXT, stats=True, copy=False)
            packed_ms = (time.perf_counter() - t0) / 5 * 1e3
            t2t = []
            for _ in range(3):
                t0 = time.perf_counter()
                hp = hostlib.HostPaf.from_text(ptxt)                       # host: parse the PAF text (all host threads)
                hw = hp.windows_from_bed_text(btxt)                        # host: parse + sort the BED rows
                views, release = sctx.liftover_view(hp, hw, want=capi.WANT_TEXT, stats=True)  # GPU: liftover + fused stats
                lifted = views["paf_text"].tobytes()
                st_text = hostlib.HostPaf.from_text(lifted).stats_text(views["stats"])  # host: the stats TSV rb stats --paf prints
                release()
                t2t.append((time.perf_counter() - t0) * 1e3)
            if lifted != want["lifted"] or st_text != want["stats"]:
                raise SystemExit("PARITY FAILURE: the sample's rows differ from the CPU oracle")
            line["same_sample"] = {"rows": int(want["rows"]), "cpu_ms": sec * 1e3, "gpu_packed_e2e_ms": packed_ms, "gpu_text_to_text_ms": min(t2t),
                                   "parity_checked_rows": int(want["rows"]),
                                   "note": "exactly the cpu_baseline sample on one B200: packed host buffers -> rb_liftover -> pinned host rows, and "
                                           "text -> text (host PAF/BED parse + GPU + host stats TSV formatting; single-threaded Python glue "
                                           "around the C++ host helpers)"}
            sctx.close()
        print(json.dumps(line))
    if world == 1:
        pin.release()
        ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
