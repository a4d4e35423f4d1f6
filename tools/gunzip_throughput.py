#!/usr/bin/env python3
"""gzip inflate on the device (mp_gunzip_run) against zlib on one host thread, on a B200.

Workload: synthetic FASTQ (150-base reads, Illumina-like qualities that fall along the read), `gib` GiB of text (default 1), gzipped
in-process at levels 1, 6 and 9 as one member each.  For each level: zlib.decompress of the whole file on one thread (the rate of a
single gzread), and the library fed `piece` MiB per call (default 64) from page-locked memory with 256 MiB of page-locked output room
per call, twice, reporting the second pass (the first one loads the module and sizes the output buffer).  Rates are decompressed
bytes per second of wall clock: of the mp_gunzip_run calls alone (host-to-device and device-to-host copies included), and of the
whole loop with the caller's copy of every call's output; beside them the counters of the block search.
The driver loop on .fq.gz (bin/soap4, which inflates .gz read files with this library) is not timed by this tool.
Output: the card's name and power limit, then one line per measurement; `--out FILE` also writes those lines to FILE.
Usage: gunzip_throughput.py [gib] [--piece MiB] [--out FILE]"""
import os
import subprocess
import sys
import time
import zlib

import ctypes as C

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import megapath_b200 as mp  # noqa: E402

lines_out = []


def say(s):
    print(s, flush=True)
    lines_out.append(s)


def fastq_text(nbytes, seed=1, L=150):
    rng = np.random.default_rng(seed)
    per = 2 * L + 4 + 16
    n = nbytes // per + 1
    out = []
    lut = np.frombuffer(b"ACGT", np.uint8)
    for a in range(0, n, 200000):
        m = min(200000, n - a)
        seq = lut[rng.integers(0, 4, (m, L))]
        qual = (33 + np.clip(np.round(37 - np.abs(rng.normal(0, 3, (m, L))) - np.linspace(0, 8, L)), 2, 41)).astype(np.uint8)
        names = np.array([b"@r%010d/1\n" % (a + i) for i in range(m)])
        rec = np.concatenate([np.frombuffer(b"".join(names), np.uint8).reshape(m, -1), seq, np.full((m, 1), 10, np.uint8),
                              np.tile(np.frombuffer(b"+\n", np.uint8), (m, 1)), qual, np.full((m, 1), 10, np.uint8)], axis=1)
        out.append(rec.tobytes())
    return b"".join(out)[:nbytes]


def main():
    args = sys.argv[1:]
    out_path, piece = None, 64
    if "--out" in args:
        k = args.index("--out"); out_path = args[k + 1]; del args[k:k + 2]
    if "--piece" in args:
        k = args.index("--piece"); piece = int(args[k + 1]); del args[k:k + 2]
    gib = float(args[0]) if args else 1.0
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout.strip()
    say("card: %s" % card)
    text = fastq_text(int(gib * (1 << 30)))
    say("workload: %.2f GB of FASTQ text, calls of %d MiB" % (len(text) / 1e9, piece))
    ctx = mp.Context(0)
    L = mp.lib()
    for level in (1, 6, 9):
        t = time.time()
        co = zlib.compressobj(level, zlib.DEFLATED, 31)
        data = co.compress(text) + co.flush()
        tc = time.time() - t
        t = time.time()
        ref = zlib.decompress(data, 31)
        tz = time.time() - t
        assert ref == text
        del ref
        src = L.mp_host_alloc(len(data))
        assert src, "mp_host_alloc failed"
        C.memmove(src, data, len(data))
        out_cap = 256 << 20
        dst = L.mp_host_alloc(out_cap)
        got = bytearray(len(text) + out_cap)
        got_addr = C.addressof((C.c_char * len(got)).from_buffer(got))
        for rep in range(2):
            with ctx.gunzip_stream(piece << 20) as g:
                pos, at, agg, tlib = 0, 0, {}, 0.0
                used, produced, done = C.c_uint64(), C.c_uint64(), C.c_int()
                t = time.time()
                while True:
                    n = min(piece << 20, len(data) - pos)
                    t1 = time.time()
                    rc = L.mp_gunzip_run(g.h, C.c_void_p(src + pos), n, int(pos + n == len(data)), dst, out_cap,
                                         C.byref(used), C.byref(produced), C.byref(done))
                    tlib += time.time() - t1
                    assert rc == 0, L.mp_last_error()
                    C.memmove(got_addr + at, dst, produced.value)
                    at += produced.value
                    for k, v in g.stats().items():
                        agg[k] = agg.get(k, 0) + v
                    pos += used.value
                    if done.value:
                        break
                td = time.time() - t
        L.mp_host_free(src)
        L.mp_host_free(dst)
        assert at == len(text) and bytes(got[:at]) == text, "device output differs from zlib"
        say("level %d: %.1f MB compressed (ratio %.2f, compress %.0f s) | zlib 1 thread %.2f GB/s | library calls %.2f GB/s (%.1fx), "
            "with the caller's copies %.2f GB/s | chunks %d candidates %d false %d merged %d overflows %d rounds %d" %
            (level, len(data) / 1e6, len(text) / len(data), tc, len(text) / tz / 1e9, len(text) / tlib / 1e9, tz / tlib, len(text) / td / 1e9,
             agg["chunks"], agg["candidates"], agg["false_candidates"], agg["merged"], agg["overflows"], agg["rounds"]))
    ctx.close()
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            f.write("\n".join(lines_out) + "\n")


if __name__ == "__main__":
    main()
