"""Translation (K14, bsq_translate) next to a copy with the same traffic and to what users do without it.

    python tools/bench_translate.py [--out profiles/r11_translate_b200.json] [--launches 100] [--torch-launches 10] [--reps 3]

Per workload, arms timed with CUDA events over back-to-back calls that rotate over 4 input/output sets (each workload's
sets together are larger than the B200's 126 MB L2), the arms alternated `--reps` times in the same process:
  k14        one bsq_translate (output bytes and offsets);
  memcpy     bsq_memcpy_d2d (cudaMemcpyAsync device to device) of (bytes read + bytes written) / 2: the same HBM traffic
             as k14's reads of the nucleotides plus its writes of the proteins, so the ratio is a ratio of bandwidths;
  torch      the torch recipe (`--torch-launches` calls): per frame, row ids by repeat_interleave, the int64 codon index
             (mirrored for reverse frames), three index_select gathers, the mask and complement look-ups as tensor gathers,
             the 12-bit index, a gather from the codon table and a scatter into sequence-major order.
At T3 also, with PROTEIN `pbeos` tokens at padlen 1024 (batch-first u8):
  k14_k1     bsq_translate, then bsq_tokenize of the proteins;
  torch_k1   the torch recipe, then the same bsq_tokenize.
Workloads:
  T1  DNA 262 144 x 150 (ACGT), six frames;
  T2  DNA 4 096 x 10 000, six frames;
  T3  65 536 coding sequences of 150..3 066 nucleotides (multiples of 3, uniform), frame +1, then the tokenizer;
  T4  T1 with 10 % IUPAC ambiguity codes (every code but ACGT), six frames: ambiguity has no slow path.
k14's output is compared once per workload with the torch recipe's.  Targets: k14 >= 0.5 of the in-run copy at T2;
>= 10x the torch recipe at T1, T2 and T4; T3 translate + tokenize >= 10x recipe + the same tokenize.  GPU name and power
limit are read in the same run.
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
SIX = (1, 2, 3, -1, -2, -3)
AMBIG = b"RYSWKMBDHVN"


def make_batch(seed, lens, ambiguity=0.0):
    rng = np.random.default_rng(seed)
    offs = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    T = int(offs[-1])
    buf = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, T)]
    if ambiguity > 0:
        pick = rng.random(T) < ambiguity
        buf[pick] = np.frombuffer(AMBIG, np.uint8)[rng.integers(0, len(AMBIG), int(pick.sum()))]
    return np.ascontiguousarray(buf), offs


def workloads():
    rng = np.random.default_rng(3)
    return [
        ("T1_dna_262144x150_six", lambda: make_batch(111, np.full(262_144, 150)), SIX, None, 0.0),
        ("T2_dna_4096x10000_six", lambda: make_batch(112, np.full(4_096, 10_000)), SIX, 0.5, 0.0),
        ("T3_cds_65536x150to3066_f1_tokenize", lambda: make_batch(113, 3 * rng.integers(50, 1023, 65_536)), (1,), None, 0.0),
        ("T4_dna_262144x150_six_iupac10", lambda: make_batch(114, np.full(262_144, 150), 0.1), SIX, None, 0.1),
    ]


def run_workload(name, make, frames, copy_target, launches, torch_launches, reps):
    buf, offs = make()
    n, F = len(offs) - 1, len(frames)
    T = int(offs[-1])
    tokenize = name.startswith("T3")
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    code = capi.genetic_code(1)
    total, _, longest = capi.translate_extent_host(offs, n, frames)
    P = 1024
    tok = capi.tokenizer("PROTEIN", eos=True, bos=True, padchar=True)
    d_b0, d_o0 = torch.from_numpy(buf).to(dev), torch.from_numpy(offs).to(dev)
    sets = []
    for _ in range(ROT):
        sets.append({"b": d_b0.clone(), "o": d_o0.clone(), "tb": torch.empty(total, dtype=torch.uint8, device=dev),
                     "to": torch.empty(n * F + 1, dtype=torch.int64, device=dev),
                     "tok": torch.empty((n * F, P), dtype=torch.uint8, device=dev) if tokenize else None})
    copy_bytes = (T + total) // 2
    cp = [torch.empty(copy_bytes, dtype=torch.uint8, device=dev) for _ in range(ROT)]
    # the torch recipe's fixed inputs (they depend on the lengths only): per frame its lengths and output row starts
    masks, codons = (torch.from_numpy(x).to(dev) for x in capi.translate_table(code))
    rev4 = torch.tensor([int(f"{m:04b}"[::-1], 2) for m in range(16)], dtype=torch.uint8, device=dev)
    cmasks = rev4[masks.long()]
    lens = d_o0[1:] - d_o0[:-1]
    starts = d_o0[:-1]
    per = [torch.clamp(lens - (abs(f) - 1), min=0) // 3 for f in frames]
    out_offs = torch.zeros(n * F + 1, dtype=torch.int64, device=dev)
    out_offs[1:] = torch.cumsum(torch.stack(per, 1).reshape(-1), 0)
    row_start = out_offs[:-1].view(n, F)
    plan = [(f, Lf, int(Lf.sum()), torch.cumsum(Lf, 0) - Lf, row_start[:, fi].contiguous()) for fi, (f, Lf) in enumerate(zip(frames, per))]

    def torch_translate(x):
        out = torch.empty(total, dtype=torch.uint8, device=dev)
        for f, Lf, m, first, dst0 in plan:
            row = torch.repeat_interleave(torch.arange(n, device=dev), Lf, output_size=m)
            t = torch.arange(m, device=dev) - first[row]
            k = abs(f)
            if f > 0:
                p = starts[row] + (k - 1) + 3 * t
                tbl, d = masks, 1
            else:
                p = starts[row] + lens[row] - k - 3 * t
                tbl, d = cmasks, -1
            m0 = tbl[x["b"].index_select(0, p).long()].long()
            m1 = tbl[x["b"].index_select(0, p + d).long()].long()
            m2 = tbl[x["b"].index_select(0, p + 2 * d).long()].long()
            out.index_put_((dst0[row] + t,), codons[(m0 << 8) | (m1 << 4) | m2])
        return out

    capi.translate(0, st, sets[0]["b"], sets[0]["o"], n, frames, code, sets[0]["tb"], sets[0]["to"])
    torch.cuda.synchronize()
    consistent = bool(torch.equal(sets[0]["tb"], torch_translate(sets[0])) and torch.equal(sets[0]["to"], out_offs))

    def k14(i):
        x = sets[i % ROT]
        capi.translate(0, st, x["b"], x["o"], n, frames, code, x["tb"], x["to"])

    def memcpy(i):
        capi.check(capi.lib().bsq_memcpy_d2d(0, st, cp[i % ROT].data_ptr(), cp[(i + 1) % ROT].data_ptr(), copy_bytes))

    def torch_arm(i):
        torch_translate(sets[i % ROT])

    def k14_k1(i):
        x = sets[i % ROT]
        capi.translate(0, st, x["b"], x["o"], n, frames, code, x["tb"], x["to"])
        capi.tokenize(0, st, x["tb"], x["to"], n * F, P, tok, True, capi.I8, x["tok"])

    def torch_k1(i):
        x = sets[i % ROT]
        capi.tokenize(0, st, torch_translate(x), out_offs, n * F, P, tok, True, capi.I8, x["tok"])

    arms = {"k14": (k14, launches), "memcpy": (memcpy, launches), "torch": (torch_arm, torch_launches)}
    if tokenize:
        arms.update({"k14_k1": (k14_k1, launches), "torch_k1": (torch_k1, torch_launches)})
    us = {a: [] for a in arms}
    for _ in range(reps):
        for a, (fn, k) in arms.items():
            us[a].append(time_launches(fn, k))
    md = {a: round(statistics.median(xs), 2) for a, xs in us.items()}
    res = {"workload": name, "n": n, "nucleotides": T, "frames": list(frames), "bytes_written": total, "longest_row": longest,
           "k14_matches_torch_recipe": consistent, "us_per_call": {a: [round(v, 2) for v in xs] for a, xs in us.items()},
           "median_us": md}
    res["k14_gb_per_s_read_plus_write"] = round((T + total) / (md["k14"] * 1e3), 1)
    res["k14_frac_of_inrun_copy"] = round(md["memcpy"] / md["k14"], 3)
    res["k14_speedup_vs_torch"] = round(md["torch"] / md["k14"], 2)
    targets = {}
    if copy_target is not None:
        targets["frac_of_copy"] = {"target": copy_target, "met": res["k14_frac_of_inrun_copy"] >= copy_target}
    if tokenize:
        res["k14_k1_speedup_vs_torch_k1"] = round(md["torch_k1"] / md["k14_k1"], 2)
        targets["e2e_speedup_vs_torch"] = {"target": 10.0, "met": res["k14_k1_speedup_vs_torch_k1"] >= 10.0}
    else:
        targets["speedup_vs_torch"] = {"target": 10.0, "met": res["k14_speedup_vs_torch"] >= 10.0}
    res["targets"] = targets
    del sets, cp
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_translate_b200.json"))
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--torch-launches", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default="", help="comma-separated workload names")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_translate.py needs a CUDA device")
    torch.cuda.set_device(0)
    out = {"gpu": gpu_info(), "launches": a.launches, "torch_launches": a.torch_launches, "reps": a.reps, "rotating_sets": ROT,
           "workloads": []}
    for name, make, frames, copy_target, _ in workloads():
        if a.only and name not in a.only.split(","):
            continue
        r = run_workload(name, make, frames, copy_target, a.launches, a.torch_launches, a.reps)
        print(json.dumps(r), flush=True)
        out["workloads"].append(r)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
