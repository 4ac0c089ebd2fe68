"""Reverse complement (K12, bsq_revcomp) next to a copy of the same bytes and to what users do without it.

    python tools/bench_revcomp.py [--out profiles/r09_revcomp_b200.json] [--launches 100] [--torch-launches 20] [--reps 3]

Per workload, arms timed with CUDA events over back-to-back calls that rotate over 4 input/output sets (each workload's
sets together are larger than the B200's 126 MB L2), the arms alternated `--reps` times in the same process:
  k12        one bsq_revcomp (out_offsets written, flip flags not): every residue read once, written once (twice with
             "both");
  memcpy     bsq_memcpy_d2d (cudaMemcpyAsync device to device) of the bytes k12 writes;
  torch      the torch recipe under k12's own flip flags: row ids by repeat_interleave, the mirrored int64 source index,
             one gather and a complement-LUT pass (`--torch-launches` calls);
At R1 also, with DNA `pbeos` tokens at padlen 152 (batch-first u8):
  k12_k1s    bsq_revcomp, then bsq_tokenize (K1s) of the flipped batch;
  torch_k1s  the torch recipe, then the same bsq_tokenize.
Workloads (DNA residues ACGTN):
  R1  262 144 x 150, random (rc_prob 0.5);
  R2  4 096 x 10 000, random;
  R3  32 x 4 000 000, always;
  R4  R1 with both (2n output sequences).
k12's output (bytes, offsets, flags) is compared once per workload with the torch recipe's.  Targets: >= 0.7 of the
in-run copy at R2 and R3, >= 0.6 at R1 and R4, >= 10x the torch recipe at R1 and R2.  GPU name and power limit are read
in the same run.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bioseq_b200 import capi  # noqa: E402
from bench_varlen import gpu_info, time_launches  # noqa: E402

ROT = 4
DNA5 = b"ACGTN"


def fixed_batch(seed, n, length):
    rng = np.random.default_rng(seed)
    a = np.frombuffer(DNA5, dtype=np.uint8)
    buf = a[rng.integers(0, len(a), size=n * length)]
    offs = np.arange(n + 1, dtype=np.int64) * length
    return np.ascontiguousarray(buf), offs


# name, (n, length), mode, copy target, torch-speedup target
WORKLOADS = [
    ("R1_dna_262144x150_random", (262_144, 150), capi.RC_RANDOM, 0.6, 10.0),
    ("R2_dna_4096x10000_random", (4_096, 10_000), capi.RC_RANDOM, 0.7, 10.0),
    ("R3_32x4000000_always", (32, 4_000_000), capi.RC_ALWAYS, 0.7, None),
    ("R4_dna_262144x150_both", (262_144, 150), capi.RC_BOTH, 0.6, None),
]


def run_workload(name, shape, mode, copy_target, torch_target, launches, torch_launches, reps, tokenize):
    n, length = shape
    buf, offs = fixed_batch(109, n, length)
    T = int(offs[-1])
    both = mode == capi.RC_BOTH
    nv, Tv = (2 * n, 2 * T) if both else (n, T)
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    P = length + 2
    tok = capi.tokenizer("DNA", eos=True, bos=True, padchar=True)
    d_b0, d_o0 = torch.from_numpy(buf).to(dev), torch.from_numpy(offs).to(dev)
    sets = []
    for _ in range(ROT):
        sets.append({"b": d_b0.clone(), "o": d_o0.clone(), "rb": torch.empty(Tv, dtype=torch.uint8, device=dev),
                     "ro": torch.empty(nv + 1, dtype=torch.int64, device=dev),
                     "tok": torch.empty((nv, P), dtype=torch.uint8, device=dev) if tokenize else None})
    del d_b0
    # the torch recipe's fixed inputs: per virtual row its length, source start and output start; k12's flags (seed 5)
    lens = torch.from_numpy(np.diff(offs)).to(dev)
    starts = d_o0[:-1]
    if both:
        lens, starts = torch.cat([lens, lens]), torch.cat([starts, starts])
    out_offs = torch.zeros(nv + 1, dtype=torch.int64, device=dev)
    out_offs[1:] = torch.cumsum(lens, 0)
    flags = torch.empty(nv, dtype=torch.uint8, device=dev)
    capi.revcomp(0, st, sets[0]["b"], sets[0]["o"], n, mode, 0.5, 5, 0, sets[0]["rb"], sets[0]["ro"], flags)
    flags = flags.bool()
    lut = torch.from_numpy(capi.revcomp_table()).to(dev)

    def torch_flip(x):
        row = torch.repeat_interleave(torch.arange(nv, device=dev), lens, output_size=Tv)
        j = torch.arange(Tv, device=dev) - out_offs[:-1][row]
        fr = flags[row]
        idx = starts[row] + torch.where(fr, lens[row] - 1 - j, j)
        g = x["b"][idx]
        return torch.where(fr, lut[g.long()], g)

    torch.cuda.synchronize()
    consistent = bool(torch.equal(sets[0]["rb"], torch_flip(sets[0])) and torch.equal(sets[0]["ro"], out_offs))

    def k12(i):
        x = sets[i % ROT]
        capi.revcomp(0, st, x["b"], x["o"], n, mode, 0.5, i, 0, x["rb"], x["ro"])

    def memcpy(i):
        a, b = sets[i % ROT], sets[(i + 1) % ROT]
        capi.check(capi.lib().bsq_memcpy_d2d(0, st, a["rb"].data_ptr(), b["rb"].data_ptr(), Tv))

    def torch_arm(i):
        torch_flip(sets[i % ROT])

    def k12_k1s(i):
        x = sets[i % ROT]
        capi.revcomp(0, st, x["b"], x["o"], n, mode, 0.5, i, 0, x["rb"], x["ro"])
        capi.tokenize(0, st, x["rb"], x["ro"], nv, P, tok, True, capi.I8, x["tok"])

    def torch_k1s(i):
        x = sets[i % ROT]
        capi.tokenize(0, st, torch_flip(x), out_offs, nv, P, tok, True, capi.I8, x["tok"])

    arms = {"k12": (k12, launches), "memcpy": (memcpy, launches), "torch": (torch_arm, torch_launches)}
    if tokenize:
        arms.update({"k12_k1s": (k12_k1s, launches), "torch_k1s": (torch_k1s, torch_launches)})
    us = {a: [] for a in arms}
    for _ in range(reps):
        for a, (fn, k) in arms.items():
            us[a].append(time_launches(fn, k))
    md = {a: round(statistics.median(xs), 2) for a, xs in us.items()}
    res = {"workload": name, "n": n, "length": length, "mode": {0: "always", 1: "random", 2: "both"}[mode], "bytes_written": Tv,
           "k12_matches_torch_recipe": consistent, "flipped_share": round(float(flags.float().mean()), 4),
           "us_per_call": {a: [round(v, 2) for v in xs] for a, xs in us.items()}, "median_us": md}
    res["k12_gb_per_s_read_plus_write"] = round((T + Tv) / (md["k12"] * 1e3), 1)
    res["k12_frac_of_inrun_copy"] = round(md["memcpy"] / md["k12"], 3)
    res["k12_speedup_vs_torch"] = round(md["torch"] / md["k12"], 2)
    targets = {"frac_of_copy": {"target": copy_target, "met": res["k12_frac_of_inrun_copy"] >= copy_target}}
    if torch_target is not None:
        targets["speedup_vs_torch"] = {"target": torch_target, "met": res["k12_speedup_vs_torch"] >= torch_target}
    res["targets"] = targets
    if tokenize:
        res["k12_k1s_speedup_vs_torch_k1s"] = round(md["torch_k1s"] / md["k12_k1s"], 2)
    del sets
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_revcomp_b200.json"))
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--torch-launches", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default="", help="comma-separated workload names")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_revcomp.py needs a CUDA device")
    torch.cuda.set_device(0)
    out = {"gpu": gpu_info(), "launches": a.launches, "torch_launches": a.torch_launches, "reps": a.reps, "rotating_sets": ROT,
           "workloads": []}
    for name, shape, mode, copy_target, torch_target in WORKLOADS:
        if a.only and name not in a.only.split(","):
            continue
        r = run_workload(name, shape, mode, copy_target, torch_target, a.launches, a.torch_launches, a.reps, name.startswith("R1"))
        print(json.dumps(r), flush=True)
        out["workloads"].append(r)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
