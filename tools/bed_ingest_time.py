#!/usr/bin/env python
"""BED text -> the windows of a resident batch, three ways, on the batch of the synthetic C4 PAF (1 kb tiling: 3.1 M rows):
  host     rbh::Windows::pack_text on every host core + rb_batch_set_windows (the packed tables cross PCIe)
  text     rb_batch_set_windows_bed(text): the BED text crosses PCIe, it is parsed, sorted and packed on the device
  bgzf     rb_batch_set_windows_bed(BGZF bytes): inflated, then the same
for three BEDs: 3 columns sorted (bedtools makewindows), the same with a 4th id column, and the 3-column rows shuffled.
Host clock around each synchronised call, after a warm-up, best of --runs; per-kernel times from a separate profiled run.  Then
rb_batch_liftover (stats) + download after every path, rows compared byte for byte: exits 1 on a mismatch.  With --cli, one cold
`RB_TIMING=1 rb liftover --stats` run on C4 files with and without RB_DEVICE_PARSE=1.  Prints the device's name and power limit
and one JSON line per BED.
    python tools/bed_ingest_time.py [--runs R] [--cli] > profiles/rNN_bed_ingest.json"""
import json
import os
import random
import struct
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rustybam_b200 import capi, hostlib  # noqa: E402

runs = int(sys.argv[sys.argv.index("--runs") + 1]) if "--runs" in sys.argv else 5
BLK = 65280


def bgzf_block(text, off):
    chunk = text[off:off + BLK]
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    cdata = co.compress(chunk) + co.flush()
    return (b"\x1f\x8b\x08\x04" + b"\0" * 4 + b"\0\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, len(cdata) + 25) + cdata +
            struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))


def bgzf(text):
    with ThreadPoolExecutor(os.cpu_count() or 8) as ex:
        return b"".join(ex.map(lambda o: bgzf_block(text, o), range(0, len(text), BLK))) + bgzf_block(text, len(text))


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60)
        return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def best(fn, n):
    fn()  # warm-up
    t = []
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        t.append(time.perf_counter() - t0)
    return min(t)


def cli_timing(hp, bed):
    """One cold `rb liftover --stats` per mode on C4 files; the RB_TIMING phases of each."""
    rb = os.path.join(ROOT, "rustybam_b200", "rb")
    res = {}
    with tempfile.TemporaryDirectory() as d:
        paf_p, bed_p = os.path.join(d, "c4.paf"), os.path.join(d, "c4.bed")
        with open(paf_p, "wb") as f:
            f.write(hp.text())
        with open(bed_p, "wb") as f:
            f.write(bed)
        outs = {}
        for name, extra in (("default", {}), ("device_parse", {"RB_DEVICE_PARSE": "1"})):
            r = subprocess.run([rb, "liftover", "--stats", "--bed", bed_p, paf_p], capture_output=True, env=dict(os.environ, RB_TIMING="1", **extra))
            line = [ln for ln in r.stderr.decode().splitlines() if ln.startswith('{"rb_timing"')]
            res[name] = json.loads(line[-1])["rb_timing"] if r.returncode == 0 and line else {"error": r.stderr.decode()[-400:]}
            outs[name] = r.stdout
        res["stdout_equal"] = outs["default"] == outs["device_parse"] and len(outs["default"]) > 0
    return res


def main():
    hp = hostlib.HostPaf.synth(scale=1.0, n_hap=1, threads=os.cpu_count() or 8)
    tiling = hp.tiling_bed_text(1000)
    rows = tiling.splitlines()
    random.Random(3).shuffle(rows)
    beds = {"sorted3": tiling, "ids": b"".join(r + b"\tw%d\n" % k for k, r in enumerate(tiling.splitlines())),
            "shuffled3": b"\n".join(rows) + b"\n"}
    ctx = capi.Context(0)
    dev = device_info()
    print("device:", dev, file=sys.stderr)
    b = ctx.upload(hp)
    ok = True
    for bname, bed in beds.items():
        z = bgzf(bed)
        res = {"device": dev, "bed": bname, "bed_bytes": len(bed), "bgzf_bytes": len(z), "host_cores": os.cpu_count(), "runs": runs}

        def host_path():
            hw = hp.windows_from_bed_text(bed)
            ctx.batch_set_windows(b, hw)
            return hw
        res["host_pack_set_s"] = best(host_path, runs)
        t0 = time.perf_counter()
        hp.windows_from_bed_text(bed)
        res["host_pack_only_s"] = time.perf_counter() - t0
        res["device_text_s"] = best(lambda: ctx.batch_set_windows_bed(b, bed), runs)
        res["device_bgzf_s"] = best(lambda: ctx.batch_set_windows_bed(b, z), runs)
        info = ctx.batch_set_windows_bed(b, bed)
        res.update(n_win=info["n_win"], n_parsed=info["n_parsed"], general=info["general"], default_ids=info["default_ids"])
        ctx.set_profiling(True)
        for name, data in (("text", bed), ("bgzf", z)):
            ctx.kernel_times(reset=True)
            ctx.batch_set_windows_bed(b, data)
            res["kernels_" + name] = {k: round(v[1], 4) for k, v in ctx.kernel_times(reset=True).items()}
        ctx.set_profiling(False)
        rows_of = {}
        for name in ("host", "text", "bgzf"):
            if name == "host":
                hw = host_path()
            else:
                ctx.batch_set_windows_bed(b, bed if name == "text" else z)
            ctx.batch_liftover(b, with_stats=True)
            out = ctx.batch_download_lift(b)
            rows_of[name] = (out["paf_text"], out["line_off"].tobytes(), out["stats"]["equal"].tobytes(), out["stats"]["id_by_all"].tobytes())
        res["rows"] = len(rows_of["host"][1]) // 8 - 1
        res["rows_equal"] = rows_of["text"] == rows_of["host"] and rows_of["bgzf"] == rows_of["host"]
        ok = ok and res["rows_equal"]
        del hw
        print(json.dumps(res), flush=True)
    ctx.batch_free(b)
    ctx.close()
    if "--cli" in sys.argv:
        c = cli_timing(hp, tiling)
        ok = ok and c["stdout_equal"]
        print(json.dumps({"device": dev, "cli_liftover_stats_c4": c}), flush=True)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
