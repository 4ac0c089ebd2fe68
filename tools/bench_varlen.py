"""Padding-free tokens (K1v, bsq_tokenize_varlen) next to the padded kernel and to what users do without it.

    python tools/bench_varlen.py [--out profiles/r04_varlen_b200.json] [--launches 200] [--reps 3]

Per workload, three arms plus a copy reference, timed with CUDA events over `--launches` back-to-back launches that
rotate over 4 input/output sets (each workload's sets together are larger than the B200's 126 MB L2), and the arms
alternated `--reps` times in the same process:
  varlen       bsq_tokenize_varlen: tokens + int32 cu_seqlens, one kernel;
  padded       bsq_tokenize of the same batch, batch-first, P = 1024 (proteins; K1s) or max length + bos + eos (reads);
  padded_mask  what users do today: padded tokenize, a mask from the lengths, tokens[mask] (torch boolean indexing);
  memcpy       bsq_memcpy_d2d moving the varlen arm's algorithmic bytes (half of them read, half written).
Algorithmic bytes of the varlen arm: L residues + 8 (n + 1) offsets read, T * itemsize tokens + 4 (n + 1) cu_seqlens
written.  The varlen output is checked against padded[mask] once per workload.  GPU name and power limit are read in the
same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bioseq_b200 import capi  # noqa: E402
from bioseq_b200.synth import gen, AA20  # noqa: E402

ROT = 4

# name, (seed, n, lo, hi, alphabet), tokenizer (key, bos, eos, padchar), destchar, padded padlen (None: max + k)
WORKLOADS = [
    ("V2_pbeos_u8", (102, 65536, 50, 1022, AA20), ("PROTEIN", True, True, True), "B", 1024),
    ("V2x4_pbeos_u8", (102, 4 * 65536, 50, 1022, AA20), ("PROTEIN", True, True, True), "B", 1024),
    ("V2_pbeos_i32", (102, 65536, 50, 1022, AA20), ("PROTEIN", True, True, True), "i", 1024),
    ("V2_pbeos_i64", (102, 65536, 50, 1022, AA20), ("PROTEIN", True, True, True), "l", 1024),
    ("DNA150_k0_u8", (106, 262144, 150, 150, b"ACGT"), ("DNA", False, False, False), "B", None),
    ("DNA150_pbeos_u8", (106, 262144, 150, 150, b"ACGT"), ("DNA", True, True, True), "B", None),
    # rows of 10 000: one row boundary per 625 output vectors -- the per-tile chain without the element-by-element
    # boundary vectors, next to DNA150_pbeos (one boundary per ~10 vectors) at about the same bytes
    ("DNA10k_pbeos_u8", (107, 4096, 10000, 10000, b"ACGT"), ("DNA", True, True, True), "B", None),
]


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as e:  # the number stays unlabelled rather than the run failing
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"])
    return None


def time_launches(fn, launches):
    for i in range(8):
        fn(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(launches):
        fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1000.0 / launches  # us per launch


def run_workload(name, g, tk, destchar, padlen, launches, reps, peak):
    key, bos, eos, pad = tk
    tok = capi.tokenizer(key, eos=eos, bos=bos, padchar=pad)
    kind = capi.kind_of(destchar)
    itemsize = int(capi.lib().bsq_kind_size(kind))
    dtype = {1: torch.uint8, 4: torch.int32, 8: torch.int64}[itemsize]
    k = int(bos) + int(eos)
    buf, offs = gen(*g)
    n, L = offs.size - 1, int(offs[-1])
    lens = np.diff(offs)
    T = L + n * k
    P = padlen if padlen is not None else int(lens.max()) + k
    alg = L + 8 * (n + 1) + T * itemsize + 4 * (n + 1)
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    d_b0, d_o0 = torch.from_numpy(buf).to(dev), torch.from_numpy(offs).to(dev)
    sets = []
    for _ in range(ROT):
        sets.append({"b": d_b0.clone(), "o": d_o0.clone(), "tok": torch.empty(T, dtype=dtype, device=dev),
                     "cu": torch.empty(n + 1, dtype=torch.int32, device=dev),
                     "pad": torch.empty((n, P), dtype=dtype, device=dev),
                     "cpy": torch.empty(alg // 2 + 16, dtype=torch.uint8, device=dev)})
    mask = torch.arange(P, device=dev)[None, :] < (torch.from_numpy(lens).to(dev) + k)[:, None]

    def varlen(i):
        s = sets[i % ROT]
        capi.tokenize_varlen(0, st, s["b"], s["o"], n, tok, kind, s["tok"], s["cu"])

    def padded(i):
        s = sets[i % ROT]
        capi.tokenize(0, st, s["b"], s["o"], n, P, tok, True, kind, s["pad"])

    def padded_mask(i):
        padded(i)
        sets[i % ROT]["masked"] = sets[i % ROT]["pad"][mask]

    def memcpy(i):
        s, t = sets[i % ROT], sets[(i + 1) % ROT]
        capi.check(capi.lib().bsq_memcpy_d2d(0, st, s["cpy"].data_ptr(), t["cpy"].data_ptr(), alg // 2))

    # outputs at the timed size: varlen == padded[mask], cu_seqlens == the prefix sums
    varlen(0)
    padded_mask(0)
    torch.cuda.synchronize()
    want_cu = np.zeros(n + 1, np.int64)
    np.cumsum(lens + k, out=want_cu[1:])
    same = bool(torch.equal(sets[0]["tok"], sets[0]["masked"])) and np.array_equal(sets[0]["cu"].cpu().numpy(), want_cu)
    arms = {"varlen": varlen, "padded": padded, "padded_mask": padded_mask, "memcpy": memcpy}
    us = {a: [] for a in arms}
    for _ in range(reps):
        for a, fn in arms.items():
            us[a].append(time_launches(fn, launches))
    res = {"workload": name, "gen": list(g[:4]) + [g[4].decode()], "tokenizer": list(tk), "destchar": destchar, "n": n,
           "residues": L, "tokens": T, "itemsize": itemsize, "padded_padlen": P, "alg_bytes_varlen": alg,
           "alg_bytes_padded": L + 8 * (n + 1) + n * P * itemsize, "varlen_equals_padded_mask": same,
           "us_per_launch": {a: [round(x, 2) for x in v] for a, v in us.items()},
           "median_us": {a: round(statistics.median(v), 2) for a, v in us.items()}}
    m = res["median_us"]
    res["varlen_gbases_per_s"] = round(L / (m["varlen"] * 1e3), 1)
    res["varlen_gb_per_s"] = round(alg / (m["varlen"] * 1e3), 1)
    res["varlen_frac_of_inrun_copy"] = round(m["memcpy"] / m["varlen"], 3)
    if peak:
        res["varlen_frac_of_measured_peak"] = round(alg / (m["varlen"] * 1e3) / peak, 3)
    res["varlen_speedup_vs_padded"] = round(m["padded"] / m["varlen"], 2)
    res["varlen_speedup_vs_padded_mask"] = round(m["padded_mask"] / m["varlen"], 2)
    del sets
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_varlen_b200.json"))
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default="", help="comma-separated workload names")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_varlen.py needs a CUDA device")
    torch.cuda.set_device(0)
    peak = measured_peak()
    out = {"gpu": gpu_info(), "launches": a.launches, "reps": a.reps, "rotating_sets": ROT,
           "measured_peak_gbs": peak, "workloads": []}
    for name, g, tk, dc, P in WORKLOADS:
        if a.only and name not in a.only.split(","):
            continue
        r = run_workload(name, g, tk, dc, P, a.launches, a.reps, peak)
        print(json.dumps(r), flush=True)
        out["workloads"].append(r)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
