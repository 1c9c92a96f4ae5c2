#!/usr/bin/env python
"""`rb liftover` from the files' bytes on N devices, against the host-parse path on the same N-device context, on the synthetic C4 PAF
(n_hap haplotypes) with 10 kb tiling windows:
  host     rbh::Paf::from_text on every host core + the BED packed on the host + rb_liftover
  text     rb_liftover_text(PAF text, BED text): every device parses its byte range of the PAF
  bgzf     rb_liftover_text(PAF as BGZF, BED text): every device inflates its run of blocks, then the same
For every N from 1 to the visible device count: host clock around each synchronised call, after a warm-up, best of --runs; the rows
(text, line offsets) of the three paths compared byte for byte: exits 1 on a mismatch.  Prints the device's name and power limit and
one JSON line.
    python tools/text_liftover_time.py [n_hap] [--runs R] > profiles/rNN_text_liftover.json"""
import ctypes as C
import json
import os
import struct
import subprocess
import sys
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

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


def main():
    import torch
    n_dev = torch.cuda.device_count()
    if n_dev < 1:
        sys.exit("no CUDA device")
    synth = hostlib.HostPaf.synth(scale=1.0, n_hap=n_hap, threads=os.cpu_count() or 8)
    text = synth.text()
    bed = hostlib.HostPaf.from_text(text).tiling_bed_text(10_000)
    with ThreadPoolExecutor(os.cpu_count() or 8) as ex:
        z = b"".join(ex.map(lambda o: bgzf_block(text, o), range(0, len(text), BLK))) + bgzf_block(text, len(text))
    dev = device_info()
    res = {"devices": dev, "n_hap": n_hap, "text_bytes": len(text), "bgzf_bytes": len(z), "bed_bytes": len(bed), "n_rec": synth.n_rec,
           "window": 10_000, "host_cores": os.cpu_count(), "runs": runs, "by_n": {}}
    print("devices:", dev, file=sys.stderr)
    lib = capi.load()
    want = capi.WANT_TEXT
    ok = True
    for n in range(1, n_dev + 1):
        ctx = capi.Context(devices=list(range(n)))

        def host_path():
            hp = hostlib.HostPaf.from_text(text)
            hw = hp.windows_from_bed_text(bed)
            out = capi.RbLiftOut()
            ctx._check(lib.rb_liftover(ctx.h, C.byref(hp.c), C.byref(hw.c), capi.POLICY_RIGHTMOST, want, C.byref(out), None))
            lib.rb_free_lift_out(ctx.h, C.byref(out))
            hw.close()
            hp.close()

        def text_path(data):
            def run():
                out = capi.RbLiftOut()
                ctx._check(lib.rb_liftover_text(ctx.h, data, len(data), bed, len(bed), capi.POLICY_RIGHTMOST, want, C.byref(out), None, None, None))
                lib.rb_free_lift_out(ctx.h, C.byref(out))
            return run
        r = {"host_ms": best(host_path, runs) * 1e3, "text_ms": best(text_path(text), runs) * 1e3, "bgzf_ms": best(text_path(z), runs) * 1e3}
        hp = hostlib.HostPaf.from_text(text)
        exp = ctx.liftover(hp, hp.windows_from_bed_text(bed), want=want, stats=False)
        for name, data in (("text", text), ("bgzf", z)):
            got = ctx.liftover_text(data, bed, want=want, stats=False)
            same = got["paf_text"] == exp["paf_text"] and np.array_equal(got["line_off"], exp["line_off"])
            r[name + "_rows_identical"] = bool(same)
            ok = ok and same
        r["n_out"] = exp["n_out"]
        r["out_bytes"] = exp["paf_nbytes"]
        res["by_n"][n] = r
        print(f"N={n}: host {r['host_ms']:.1f} ms, text {r['text_ms']:.1f} ms, bgzf {r['bgzf_ms']:.1f} ms", file=sys.stderr)
        ctx.close()
    print(json.dumps(res))
    if not ok:
        print("MISMATCH between the paths' rows", file=sys.stderr)
        sys.exit(1)


if __name__ == "__main__":
    main()
