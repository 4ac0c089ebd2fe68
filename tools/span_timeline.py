"""Device-side timeline of K1s (tokenize_span_kernel) from one launch to the next, at bench.py's C2 shapes.

    python tools/span_timeline.py [--launches 24] [--warmup 8] [--out FILE] [--lib TRACED_LIB | --build-only DIR]

Builds libbsq.so with -DBSQ_SPAN_TRACE into a scratch directory (never over bioseq_b200/libbsq.so; objects of the other
sources are reused from bioseq_b200/build/ when present), or uses --lib.  It then runs back-to-back C2 launches (PROTEIN
pbeos, 65 536 ragged rows of 50-1022 residues, P = 1024, the four rotating input / output sets of bench.py) on one
stream, each CTA recording %globaltimer (and clock64) at six events:

    entry -> griddepcontrol.wait returned -> tile 0's copy issued -> consumer warp 0 saw tile 0's full barrier
          -> consumer warp 0's first store issued -> exit (last consumer warp)

and prints, per launch after the first: the previous grid's last exit -> this grid's median / max wait release, wait
release -> tile 0 copy issued, copy issued -> first store, first store -> last exit (medians over the CTAs), the spread of
the CTAs' start times, how many CTAs started only after the previous grid had ended, and the tiles per CTA.
"""
import argparse
import ctypes as C
import importlib.util
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "bioseq_b200", "csrc")
WORDS = 16   # kSpanTraceWords
ENTRY, WAIT, COPY0, FULL0, STORE0, EXIT, SMID, TILES = range(8)
NSEQ, LO, HI, PADLEN, ROT = 65536, 50, 1022, 1024, 4


def load(name, rel):
    """A module of the package loaded by path: importing bioseq_b200 would map the untraced libbsq.so into the process."""
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, rel))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def build_traced(outdir):
    b = load("_bsq_build", os.path.join("bioseq_b200", "build.py"))
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(outdir, exist_ok=True)
    objs = []
    for src in b.LIB_SOURCES:
        stem = os.path.splitext(src)[0]
        shipped = os.path.join(ROOT, "bioseq_b200", "build", stem + ".o")
        if src != "bsq_span.cu" and os.path.exists(shipped) and not b._stale(shipped, [src]):
            objs.append(shipped)
            continue
        obj = os.path.join(outdir, stem + ".o")
        flags = ["-DBSQ_SPAN_TRACE"] if src == "bsq_span.cu" else []
        subprocess.check_call([nvcc] + b.NVCC_COMPILE + flags + ["-c", src, "-o", obj], cwd=CSRC)
        objs.append(obj)
    lib = os.path.join(outdir, "libbsq_trace.so")
    subprocess.check_call([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib] + objs + ["-lz"], cwd=CSRC)
    return lib


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        return "unknown"


def med(x):
    return float(statistics.median(x)) if len(x) else float("nan")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=24, help="traced launches after the warm-up (stats from the second on)")
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--lib", help="an already built traced library (see --build-only)")
    ap.add_argument("--build-only", metavar="DIR", help="build the traced library into DIR and exit")
    ap.add_argument("--out", help="also write the report here")
    args = ap.parse_args()
    if args.build_only:
        print(build_traced(args.build_only))
        return
    tmp = None
    lib_path = args.lib
    if lib_path is None:
        tmp = tempfile.mkdtemp(prefix="bsq_span_trace_")
        lib_path = build_traced(tmp)
    try:
        report = run(lib_path, args)
    finally:
        if tmp is not None:
            shutil.rmtree(tmp, ignore_errors=True)
    print(report)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(report + "\n")


def run(lib_path, args):
    import torch

    capi = load("_bsq_capi", os.path.join("bioseq_b200", "capi.py"))
    synth = load("_bsq_synth", os.path.join("bioseq_b200", "synth.py"))
    capi.LIB_PATH = lib_path
    L = capi.lib()
    L.bsq_span_trace_arm.restype, L.bsq_span_trace_arm.argtypes = None, [C.c_void_p]
    tok = capi.tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    torch.cuda.set_device(0)
    st = torch.cuda.current_stream().cuda_stream
    sets = []
    for r in range(ROT):
        buf, offs = synth.gen(102 + r, NSEQ, LO, HI, synth.AA20)
        sets.append((torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda(),
                     torch.empty((NSEQ, PADLEN), dtype=torch.uint8, device="cuda")))

    def launch(i):
        b, o, out = sets[i % ROT]
        capi.check(L.bsq_tokenize(0, st, b.data_ptr(), o.data_ptr(), NSEQ, PADLEN, C.byref(tok), 1, 0, out.data_ptr()))

    max_ctas = torch.cuda.get_device_properties(0).multi_processor_count * 8
    K = args.launches
    trace = torch.zeros((K, max_ctas, WORDS), dtype=torch.int64, device="cuda")
    for i in range(64):
        launch(i)
    torch.cuda.synchronize()
    # a spin kernel first, so that the host has queued every launch before the first one starts: the launches then run
    # back to back as in bench.py's timed loop
    torch.cuda._sleep(20_000_000)
    for i in range(args.warmup):
        launch(i)
    for k in range(K):
        L.bsq_span_trace_arm(trace[k].data_ptr())
        launch(args.warmup + k)
    L.bsq_span_trace_arm(None)
    torch.cuda.synchronize()
    tr = trace.cpu().numpy().view(np.uint64).astype(np.int64)

    lines = [f"# K1s launch hand-over timeline (tools/span_timeline.py), C2: {NSEQ} rows, P = {PADLEN}, {ROT} rotating sets",
             f"# device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power.limit, clocks.max.sm: {gpu_info()}",
             f"# warm-up {args.warmup} launches, {K} traced; times in us from %globaltimer unless marked cycles"]
    grids = []
    for k in range(K):
        g = tr[k]
        used = g[:, ENTRY] != 0
        grids.append(g[used])
    stamps = np.sort(np.concatenate([g[:, :EXIT + 1].ravel() for g in grids]))
    d = np.diff(stamps)
    d = d[d > 0]
    lines.append(f"# %globaltimer: smallest non-zero delta seen {int(d.min()) if d.size else -1} ns, "
                 f"{np.unique(stamps).size} distinct values over {stamps.size} stamps")
    lines.append(f"# CTAs per grid: {grids[0].shape[0]}")
    hdr = ("launch", "prev_exit->wait_med", "prev_exit->wait_max", "wait->copy0", "copy0->store0", "store0->last_exit",
           "start_spread", "late_ctas", "full0->store0_cyc", "wait->copy0_cyc", "tiles_min", "tiles_max", "period")
    lines.append(" ".join(f"{h:>18}" for h in hdr))
    rows = []
    for k in range(1, K):
        g, p = grids[k], grids[k - 1]
        prev_exit = p[:, EXIT].max()
        us = lambda x: x / 1e3  # noqa: E731
        row = (k, us(med(g[:, WAIT] - prev_exit)), us((g[:, WAIT] - prev_exit).max()), us(med(g[:, COPY0] - g[:, WAIT])),
               us(med(g[:, STORE0] - g[:, COPY0])), us(g[:, EXIT].max() - med(g[:, STORE0])),
               us(g[:, ENTRY].max() - g[:, ENTRY].min()), int((g[:, ENTRY] > prev_exit).sum()),
               med(g[:, 8 + STORE0] - g[:, 8 + FULL0]), med(g[:, 8 + COPY0] - g[:, 8 + WAIT]),
               int(g[:, TILES].min()), int(g[:, TILES].max()), us(g[:, EXIT].max() - prev_exit))
        rows.append(row)
        lines.append(" ".join(f"{v:>18.3f}" if isinstance(v, float) else f"{v:>18d}" for v in row))
    cols = list(zip(*rows))
    lines.append("median " + " ".join(f"{h}={med(c):.3f}" for h, c in zip(hdr[1:], cols[1:])))
    return "\n".join(lines)


if __name__ == "__main__":
    sys.exit(main())
