#!/usr/bin/env python
"""`rb stats --paf` from the file's bytes (rb_stats_text) against the host path, on two inputs:
  c4      the synthetic C4 PAF: few long records, parsing dominates
  lifted  its rows lifted at 1 kb tiling windows: millions of short records, formatting dominates
and three paths:
  host    rbh::Paf::from_text on every host core + rb_stats + the host formatter (hostlib stats_text)
  text    rb_stats_text(PAF text, RB_WANT_STATS_TEXT): parsed, counted and formatted on the device(s)
  bgzf    rb_stats_text(PAF as BGZF, ...): every device inflates its run of blocks, then the same
For every N from 1 to the visible device count: host clock around each synchronised call, after a warm-up, best of --runs; the rows of
the three paths compared byte for byte (exits 1 on a mismatch).  Kernel times (rb_ctx_set_profiling) of one text call on one device,
in a run of their own.  The CLI: `RB_TIMING=1 rb stats --paf` on the lifted rows, the default path against RB_DEVICE_PARSE=1, best of
--runs.  The device's name and power limit are read in the same run.  Writes <out>/r03d_stats_text_{c4,lifted}.json.
    python tools/stats_text_time.py [--runs R] [--out DIR]"""
import ctypes as C
import json
import os
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
out_dir = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(ROOT, "profiles")
BLK = 65280
RB = os.path.join(ROOT, "rustybam_b200", "rb")


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
        return q.stdout.strip().splitlines() if q.returncode == 0 and q.stdout.strip() else ["unknown"]
    except (OSError, subprocess.SubprocessError):
        return ["unknown"]


def best(fn, n):
    fn()  # warm-up
    t = []
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        t.append(time.perf_counter() - t0)
    return min(t)


def cli_time(path):
    """Best wall time and the rb_timing phases of `rb stats --paf path`, default path and RB_DEVICE_PARSE=1; their stdout compared."""
    res, outs = {}, {}
    for name, extra in (("default", {}), ("device_parse", {"RB_DEVICE_PARSE": "1"})):
        env = dict(os.environ, RB_TIMING="1", **extra)
        best_ms, phases = None, None
        for k in range(runs + 1):
            with tempfile.TemporaryFile() as f:
                t0 = time.perf_counter()
                p = subprocess.run([RB, "stats", "--paf", path], stdout=f, stderr=subprocess.PIPE, env=env)
                ms = (time.perf_counter() - t0) * 1e3
                if p.returncode != 0:
                    sys.exit(f"rb failed ({name}): {p.stderr[-500:]}")
                if k == 0:
                    f.seek(0)
                    outs[name] = f.read()
            if k and (best_ms is None or ms < best_ms):
                best_ms = ms
                line = [ln for ln in p.stderr.decode().splitlines() if ln.startswith("{\"rb_timing\"")]
                phases = json.loads(line[-1])["rb_timing"] if line else None
        res[name] = {"wall_ms": best_ms, "rb_timing": phases}
    res["stdout_identical"] = outs["default"] == outs["device_parse"]
    return res


def main():
    import torch
    n_dev = torch.cuda.device_count()
    if n_dev < 1:
        sys.exit("no CUDA device")
    dev = device_info()
    print("devices:", dev, file=sys.stderr)
    lib = capi.load()
    ok = True
    synth = hostlib.HostPaf.synth(scale=1.0, n_hap=1, threads=os.cpu_count() or 8)
    c4 = synth.text()
    ctx0 = capi.Context(0)
    hp = hostlib.HostPaf.from_text(c4)
    lifted = ctx0.liftover(hp, hp.tiling_windows(1000), want=capi.WANT_TEXT, stats=False)["paf_text"]
    hp.close()
    ctx0.close()
    os.makedirs(out_dir, exist_ok=True)
    for tag, text in (("c4", c4), ("lifted", lifted)):
        z = bgzf(text)
        res = {"devices": dev, "input": tag, "text_bytes": len(text), "bgzf_bytes": len(z), "host_cores": os.cpu_count(), "runs": runs,
               "clock": "host perf_counter around synchronised calls, warm-up + best of runs", "by_n": {}}

        def host_rows():
            h = hostlib.HostPaf.from_text(text)
            rows = h.stats_text(ctx.stats(h), header=False)
            h.close()
            return rows

        def device_rows(data):
            out = capi.RbLiftOut()
            ctx._check(lib.rb_stats_text(ctx.h, data, len(data), 0, capi.WANT_STATS_TEXT, C.byref(out), None, None))
            lib.rb_free_lift_out(ctx.h, C.byref(out))
        for n in range(1, max(n_dev, 2) + 1):
            if n > n_dev:
                res["by_n"][n] = "not measured (one GPU visible)"
                continue
            ctx = capi.Context(devices=list(range(n)))
            r = {"host_ms": best(host_rows, runs) * 1e3, "text_ms": best(lambda: device_rows(text), runs) * 1e3,
                 "bgzf_ms": best(lambda: device_rows(z), runs) * 1e3}
            want = host_rows()
            for name, data in (("text", text), ("bgzf", z)):
                same = ctx.stats_text(data)["paf_text"] == want
                r[name + "_rows_identical"] = bool(same)
                ok = ok and same
            r["n_rec"] = want.count(b"\n")
            r["out_bytes"] = len(want)
            if n == 1:  # kernel times in a run of their own
                ctx.set_profiling(True)
                ctx.kernel_times(reset=True)
                device_rows(text)
                r["kernels_ms"] = {k: round(v[1], 3) for k, v in sorted(ctx.kernel_times(reset=True).items(), key=lambda kv: -kv[1][1])}
                ctx.set_profiling(False)
            res["by_n"][n] = r
            print(f"{tag} N={n}: host {r['host_ms']:.1f} ms, text {r['text_ms']:.1f} ms, bgzf {r['bgzf_ms']:.1f} ms", file=sys.stderr)
            ctx.close()
        if tag == "lifted":
            with tempfile.NamedTemporaryFile(suffix=".paf") as f:
                f.write(text)
                f.flush()
                res["cli"] = cli_time(f.name)
                ok = ok and res["cli"]["stdout_identical"]
                print("cli:", res["cli"], file=sys.stderr)
        with open(os.path.join(out_dir, f"r03d_stats_text_{tag}.json"), "w") as f:
            f.write(json.dumps(res) + "\n")
    if not ok:
        print("MISMATCH between the paths' rows", file=sys.stderr)
        sys.exit(1)


if __name__ == "__main__":
    main()
