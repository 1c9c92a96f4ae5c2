#!/usr/bin/env python
"""PAF text -> a resident batch, three ways, on the synthetic C4 PAF (n_hap haplotypes):
  host     rbh::Paf::from_text on every host core + rb_batch_upload (the CIGAR bytes cross PCIe)
  text     rb_batch_upload_paf(text): the text crosses PCIe, lines are split and parsed on the device
  bgzf     rb_batch_upload_paf(BGZF bytes): inflated and parsed on the device
Host clock around each synchronised call, after a warm-up, best of --runs; per-kernel times from a separate profiled run.  Then
rb_batch_liftover (10 kb tiling windows, stats) + download on the batch of every path, rows compared byte for byte: exits 1 on a
mismatch.  Prints the device's name and power limit and one JSON line.
    python tools/paf_ingest_time.py [n_hap] [--runs R] > profiles/rNN_paf_ingest.json"""
import json
import os
import struct
import subprocess
import sys
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rustybam_b200 import capi, hostlib  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
n_hap = int(args[0]) if args else 1
runs = int(sys.argv[sys.argv.index("--runs") + 1]) if "--runs" in sys.argv else 5
BLK = 65280


def bgzf_block(text, off):
    chunk = text[off:off + BLK]
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    cdata = co.compress(chunk) + co.flush()
    return (b"\x1f\x8b\x08\x04" + b"\0" * 4 + b"\0\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, len(cdata) + 25) + cdata +
            struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))


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


def main():
    synth = hostlib.HostPaf.synth(scale=1.0, n_hap=n_hap, threads=os.cpu_count() or 8)
    text = synth.text()
    with ThreadPoolExecutor(os.cpu_count() or 8) as ex:
        z = b"".join(ex.map(lambda o: bgzf_block(text, o), range(0, len(text), BLK))) + bgzf_block(text, len(text))
    ctx = capi.Context(0)
    res = {"device": device_info(), "n_hap": n_hap, "text_bytes": len(text), "bgzf_bytes": len(z), "n_rec": synth.n_rec,
           "cigar_bytes": synth.cigar_nbytes, "host_cores": os.cpu_count(), "runs": runs}
    print("device:", res["device"], file=sys.stderr)

    def host_path():
        hp = hostlib.HostPaf.from_text(text)
        b = ctx.upload(hp)
        return hp, b

    def dev_path(data):
        return lambda: ctx.upload_paf(data)[0]

    def timed(make, n):
        held = []

        def once():
            b = make()
            held.append(b)
        s = best(once, n)
        for b in held:
            ctx.batch_free(b[1] if isinstance(b, tuple) else b)
        return s

    res["host_parse_upload_s"] = timed(host_path, runs)
    res["device_text_s"] = timed(dev_path(text), runs)
    res["device_bgzf_s"] = timed(dev_path(z), runs)
    for k in ("host_parse_upload", "device_text", "device_bgzf"):
        res[k + "_text_gb_per_s"] = len(text) / res[k + "_s"] / 1e9
    # per-kernel times: one profiled call of each device path
    ctx.set_profiling(True)
    for name, data in (("text", text), ("bgzf", z)):
        ctx.kernel_times(reset=True)
        b, _ = ctx.upload_paf(data)
        ctx.batch_free(b)
        res["kernels_" + name] = {k: round(v[1], 4) for k, v in ctx.kernel_times(reset=True).items()}
    ctx.set_profiling(False)
    # the rows of every path, byte for byte
    hp, hb = host_path()
    wins = hp.tiling_windows(10_000)
    rows = {}
    for name, b in (("host", hb), ("text", ctx.upload_paf(text)[0]), ("bgzf", ctx.upload_paf(z)[0])):
        ctx.batch_set_windows(b, wins)
        ctx.batch_liftover(b, with_stats=True)
        out = ctx.batch_download_lift(b)
        rows[name] = (out["paf_text"], out["line_off"].tobytes(), out["stats"]["equal"].tobytes(), out["stats"]["id_by_all"].tobytes())
        ctx.batch_free(b)
    res["rows"] = len(rows["host"][1]) // 8 - 1
    res["rows_bytes"] = len(rows["host"][0])
    res["rows_equal"] = rows["text"] == rows["host"] and rows["bgzf"] == rows["host"]
    ctx.close()
    print(json.dumps(res))
    return 0 if res["rows_equal"] else 1


if __name__ == "__main__":
    sys.exit(main())
