"""Cropping over-long sequences (K9, bsq_crop) next to a copy of the same bytes and to what users do without it.

    python tools/bench_crop.py [--out profiles/r06_crop_b200.json] [--launches 100] [--reps 3]

Per workload, arms timed with CUDA events over `--launches` back-to-back calls that rotate over 4 input/output sets
(each workload's sets together are larger than the B200's 126 MB L2), the arms alternated `--reps` times in the same
process:
  crop        one bsq_crop (random windows, starts not written): the kept bytes read once and written once;
  memcpy      bsq_memcpy_d2d (cudaMemcpyAsync device to device) of the kept bytes;
  crop_k1s    bsq_crop, then bsq_tokenize (K1s) of the cropped batch at padlen P, batch-first u8;
  torch_k1s   the torch recipe: starts from torch.rand, the window gather built with repeat_interleave + arange and
              one index, then the same bsq_tokenize.
At X1 also, host clock around a synchronised call, `--list-reps` times each, alternated:
  list_cropped  batch_tokenize_cropped on the Python list of items;
  list_slicing  Python slicing of every item to a random window, then Tokenizer.batch_tokenize(list).
Workloads (P = W + 2, PROTEIN with BOS / EOS / PAD):
  X1  65 536 protein sequences, lognormal lengths (median 300, sigma 1.0) clipped to [30, 34 000], W = 1022;
  X2  C2's inputs (65 536 sequences, uniform 50 .. 1022 residues), W = 510: most rows are cropped;
  X3  C2 with W = 1022: nothing is cropped (the cost of a pass that does no work).
The crop arm's output is compared once per workload with the torch recipe's windows drawn at the same starts.  GPU
name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bioseq_b200 import capi, cbioseq, consumers  # noqa: E402
from bioseq_b200.synth import gen, AA20  # noqa: E402
from bench_varlen import gpu_info, time_launches  # noqa: E402

ROT = 4


def lognormal_batch(seed, n, median, sigma, lo, hi):
    rng = np.random.default_rng(seed)
    lens = np.clip(np.round(rng.lognormal(np.log(median), sigma, size=n)), lo, hi).astype(np.int64)
    a = np.frombuffer(AA20, dtype=np.uint8)
    buf = a[rng.integers(0, len(a), size=int(lens.sum()))]
    offs = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    return np.ascontiguousarray(buf), offs


WORKLOADS = [
    ("X1_lognormal_W1022", lambda: lognormal_batch(106, 65536, 300, 1.0, 30, 34000), 1022),
    ("X2_C2_W510", lambda: gen(102, 65536, 50, 1022, AA20), 510),
    ("X3_C2_W1022_nothing_cropped", lambda: gen(102, 65536, 50, 1022, AA20), 1022),
]


def run_workload(name, make, W, launches, reps, list_reps):
    P = W + 2
    tok = capi.tokenizer("PROTEIN", eos=True, bos=True, padchar=True)
    buf, offs = make()
    n, L = offs.size - 1, int(offs[-1])
    lens = np.diff(offs)
    kept = np.minimum(lens, W)
    total = int(kept.sum())
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    d_b0, d_o0 = torch.from_numpy(buf).to(dev), torch.from_numpy(offs).to(dev)
    sets = []
    for _ in range(ROT):
        sets.append({"b": d_b0.clone(), "o": d_o0.clone(), "cb": torch.empty(max(total, 1), dtype=torch.uint8, device=dev),
                     "co": torch.empty(n + 1, dtype=torch.int64, device=dev),
                     "tok": torch.empty((n, P), dtype=torch.uint8, device=dev)})
    d_lens = torch.from_numpy(lens).to(dev)
    d_kept = torch.from_numpy(kept).to(dev)
    out_offs = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    out_offs[1:] = torch.cumsum(d_kept, 0)
    span = (d_lens - W + 1).clamp(min=1)
    ar = torch.arange(total, device=dev)
    rel = ar - torch.repeat_interleave(out_offs[:-1], d_kept, output_size=total)

    def crop(i):
        x = sets[i % ROT]
        capi.crop(0, st, x["b"], x["o"], n, W, True, i, 0, x["cb"], x["co"])

    def memcpy(i):
        a, b = sets[i % ROT], sets[(i + 1) % ROT]
        capi.check(capi.lib().bsq_memcpy_d2d(0, st, a["cb"].data_ptr(), b["cb"].data_ptr(), total))

    def crop_k1s(i):
        x = sets[i % ROT]
        capi.crop(0, st, x["b"], x["o"], n, W, True, i, 0, x["cb"], x["co"])
        capi.tokenize(0, st, x["cb"], x["co"], n, P, tok, True, capi.I8, x["tok"])

    def torch_window(x, starts):
        src = torch.repeat_interleave(x["o"][:-1] + starts, d_kept, output_size=total) + rel
        return x["b"][src]

    def torch_k1s(i):
        x = sets[i % ROT]
        starts = (torch.rand(n, device=dev, dtype=torch.float64) * span).long()
        cb = torch_window(x, starts)
        capi.tokenize(0, st, cb, out_offs, n, P, tok, True, capi.I8, x["tok"])

    # the crop's windows against the torch gather at the same starts
    starts = torch.empty(n, dtype=torch.int64, device=dev)
    capi.crop(0, st, sets[0]["b"], sets[0]["o"], n, W, True, 5, 0, sets[0]["cb"], sets[0]["co"], starts)
    torch.cuda.synchronize()
    consistent = bool(torch.equal(sets[0]["cb"][:total], torch_window(sets[0], starts)) and torch.equal(sets[0]["co"], out_offs))
    arms = {"crop": crop, "memcpy": memcpy, "crop_k1s": crop_k1s, "torch_k1s": torch_k1s}
    us = {a: [] for a in arms}
    for _ in range(reps):
        for a, fn in arms.items():
            us[a].append(time_launches(fn, launches))
    res = {"workload": name, "n": n, "residues": L, "crop_len": W, "padlen": P, "kept_bytes": total,
           "rows_cropped": int((lens > W).sum()), "median_len": float(np.median(lens)), "max_len": int(lens.max()),
           "crop_matches_torch_gather": consistent,
           "us_per_call": {a: [round(v, 2) for v in xs] for a, xs in us.items()},
           "median_us": {a: round(statistics.median(xs), 2) for a, xs in us.items()}}
    md = res["median_us"]
    res["crop_gb_per_s_read_plus_write"] = round(2 * total / (md["crop"] * 1e3), 1)
    res["crop_frac_of_inrun_copy"] = round(md["memcpy"] / md["crop"], 3)
    res["crop_k1s_speedup_vs_torch"] = round(md["torch_k1s"] / md["crop_k1s"], 2)
    if list_reps:
        res["list"] = run_list(buf, offs, W, P, list_reps)
    del sets
    torch.cuda.empty_cache()
    return res


def run_list(buf, offs, W, P, reps):
    tok = cbioseq.Tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    b = buf.tobytes()
    o = offs.tolist()
    items = [b[o[i]:o[i + 1]] for i in range(len(o) - 1)]
    rng = np.random.default_rng(0)

    def cropped(seed):
        return consumers.batch_tokenize_cropped(tok, items, P, seed=seed)

    def slicing(seed):
        out = []
        for s in items:
            if len(s) > W:
                j = int(rng.integers(0, len(s) - W + 1))
                s = s[j:j + W]
            out.append(s)
        return tok.batch_tokenize(out, padlen=P, batch_first=True, destchar="B")

    arms = {"list_cropped": cropped, "list_slicing": slicing}
    for fn in arms.values():
        fn(0)
    torch.cuda.synchronize()
    ms = {a: [] for a in arms}
    for r in range(reps):
        for a, fn in arms.items():
            t0 = time.perf_counter()
            fn(r + 1)
            torch.cuda.synchronize()
            ms[a].append((time.perf_counter() - t0) * 1e3)
    med = {a: round(statistics.median(v), 3) for a, v in ms.items()}
    return {"ms_per_call": {a: [round(x, 3) for x in v] for a, v in ms.items()}, "median_ms": med,
            "cropped_speedup_vs_slicing": round(med["list_slicing"] / med["list_cropped"], 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_crop_b200.json"))
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--list-reps", type=int, default=5)
    ap.add_argument("--only", default="", help="comma-separated workload names")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_crop.py needs a CUDA device")
    torch.cuda.set_device(0)
    out = {"gpu": gpu_info(), "launches": a.launches, "reps": a.reps, "rotating_sets": ROT, "workloads": []}
    for name, make, W in WORKLOADS:
        if a.only and name not in a.only.split(","):
            continue
        r = run_workload(name, make, W, a.launches, a.reps, a.list_reps if name.startswith("X1") else 0)
        print(json.dumps(r), flush=True)
        out["workloads"].append(r)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
