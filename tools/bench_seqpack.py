"""Sequence packing (K10, bsq_tokenize_seqpack) next to a copy of the same bytes and to the torch recipe it replaces.

    python tools/bench_seqpack.py [--out profiles/r07_seqpack_b200.json] [--launches 100] [--reps 3]

Per workload the batch is planned once on the host (bsq_seqpack_plan, best-fit decreasing into rows of L = 1024,
PROTEIN / DNA with BOS / EOS / PAD) and the device arms are timed with CUDA events over `--launches` back-to-back calls
that rotate over 4 input/output sets (each workload's sets together are larger than the B200's 126 MB L2), the arms
alternated `--reps` times in the same process:
  seqpack      one bsq_tokenize_seqpack: (R, L) u8 tokens + int32 position ids;
  seqpack_mlm  one bsq_tokenize_seqpack_mlm: (R, L) u8 inputs + int32 position ids + int64 labels;
  memcpy       bsq_memcpy_d2d (cudaMemcpyAsync device to device) of the bytes seqpack writes (R * L * 5);
  torch        the recipe without K10, on the same plan: K1v (bsq_tokenize_varlen) into a flat buffer, tokens.fill_(pad),
               a scatter to the planned positions (index from repeat_interleave of the starts), and position ids from
               arange - repeat_interleave of the segment starts.
On the host clock, `--plan-reps` times: the plan as batch_tokenize_seqpack makes it (a sizing call and a filling call).
Rows and fill are reported against padded rows (one per sequence).  K10's output is compared once per workload with
the torch recipe's.  GPU name and power limit are read in the same run.
Workloads:
  S1  X1: 65 536 protein sequences, lognormal lengths (median 300, sigma 1.0) clipped to [30, 34 000], cropped (head) to
      W = 1022 -- the crop benchmark's workload;
  S2  C2: 65 536 protein sequences, uniform 50 .. 1022 residues;
  S3  DNA: 262 144 reads of 150 bases (about 6 per row).
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

from bioseq_b200 import capi, consumers  # noqa: E402
from bioseq_b200.synth import gen, AA20  # noqa: E402
from bench_varlen import gpu_info, time_launches  # noqa: E402
from bench_crop import lognormal_batch  # noqa: E402

ROT = 4
L = 1024


def x1_cropped():
    buf, offs = lognormal_batch(106, 65536, 300, 1.0, 30, 34000)
    lens = np.minimum(np.diff(offs), L - 2)
    parts = [buf[offs[i]:offs[i] + lens[i]] for i in range(lens.size)]
    o = np.zeros(lens.size + 1, np.int64)
    np.cumsum(lens, out=o[1:])
    return np.ascontiguousarray(np.concatenate(parts)), o


WORKLOADS = [
    ("S1_X1_cropped_W1022", x1_cropped, "PROTEIN"),
    ("S2_C2", lambda: gen(102, 65536, 50, 1022, AA20), "PROTEIN"),
    ("S3_DNA_262144x150", lambda: gen(103, 262144, 150, 150, b"ACGT"), "DNA"),
]


def host_plan(offs, n, k, reps):
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        p = consumers._SeqPackPlan(offs, n, k, L, 0)
        ms.append((time.perf_counter() - t0) * 1e3)
    return p, ms


def run_workload(name, make, key, launches, reps, plan_reps):
    tok = capi.tokenizer(key, eos=True, bos=True, padchar=True)
    k = 2
    buf, offs = make()
    n = offs.size - 1
    lens = np.diff(offs)
    plan, plan_ms = host_plan(offs, n, k, plan_reps)
    R = plan.R
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    d_row_ptr, d_row_seq, d_starts, d_cu = plan.to_device(dev)
    d_b0, d_o0 = torch.from_numpy(buf).to(dev), torch.from_numpy(offs).to(dev)
    T = int(lens.sum()) + n * k
    sets = []
    for _ in range(ROT):
        sets.append({"b": d_b0.clone(), "o": d_o0.clone(), "tok": torch.empty((R, L), dtype=torch.uint8, device=dev),
                     "pos": torch.empty((R, L), dtype=torch.int32, device=dev),
                     "lab": torch.empty((R, L), dtype=torch.int64, device=dev),
                     "flat": torch.empty(T, dtype=torch.uint8, device=dev),
                     "cu": torch.empty(n + 1, dtype=torch.int32, device=dev)})
    mlm = consumers._mlm_desc(tok, "B", 0.15, 0.8, 0.1, None, -100, 1, 0)
    out_bytes = R * L * 5
    need = torch.from_numpy(lens + k).to(dev)
    seg_starts = d_cu[:-1].long()
    seg_lens = (d_cu[1:] - d_cu[:-1]).long()
    pad_id = int(tok.pad_id)

    def seqpack(i):
        x = sets[i % ROT]
        capi.tokenize_seqpack(0, st, x["b"], x["o"], tok, capi.I8, L, R, d_row_ptr, d_row_seq, x["tok"], x["pos"])

    def seqpack_mlm(i):
        x = sets[i % ROT]
        capi.tokenize_seqpack_mlm(0, st, x["b"], x["o"], tok, capi.I8, mlm, L, R, d_row_ptr, d_row_seq, x["tok"], x["pos"], x["lab"])

    def memcpy(i):
        a, b = sets[i % ROT], sets[(i + 1) % ROT]
        capi.check(capi.lib().bsq_memcpy_d2d(0, st, a["tok"].data_ptr(), b["tok"].data_ptr(), R * L))
        capi.check(capi.lib().bsq_memcpy_d2d(0, st, a["pos"].data_ptr(), b["pos"].data_ptr(), R * L * 4))

    def torch_recipe(i):
        x = sets[i % ROT]
        capi.tokenize_varlen(0, st, x["b"], x["o"], n, tok, capi.I8, x["flat"], x["cu"])
        cu = x["cu"].long()
        dest = torch.repeat_interleave(d_starts - cu[:-1], need, output_size=T) + torch.arange(T, device=dev)
        x["tok"].fill_(pad_id)
        x["tok"].view(-1)[dest] = x["flat"]
        x["pos"].view(-1).copy_(torch.arange(R * L, device=dev, dtype=torch.int32) -
                                torch.repeat_interleave(seg_starts, seg_lens, output_size=R * L).int())

    torch_recipe(0)
    want_tok, want_pos = sets[0]["tok"].clone(), sets[0]["pos"].clone()
    seqpack(0)
    torch.cuda.synchronize()
    consistent = bool(torch.equal(sets[0]["tok"], want_tok) and torch.equal(sets[0]["pos"], want_pos))
    arms = {"seqpack": seqpack, "seqpack_mlm": seqpack_mlm, "memcpy": memcpy, "torch": torch_recipe}
    us = {a: [] for a in arms}
    for _ in range(reps):
        for a, fn in arms.items():
            us[a].append(time_launches(fn, launches))
    res = {"workload": name, "n": n, "residues": int(lens.sum()), "row_len": L, "rows": R, "padded_rows": n,
           "fill": round(T / (R * L), 4), "padded_fill": round(T / (n * L), 4), "segments": plan.nseg,
           "seqpack_out_bytes": out_bytes, "seqpack_matches_torch": consistent,
           "plan_ms_host": [round(v, 3) for v in plan_ms], "plan_median_ms_host": round(statistics.median(plan_ms), 3),
           "us_per_call": {a: [round(v, 2) for v in xs] for a, xs in us.items()},
           "median_us": {a: round(statistics.median(xs), 2) for a, xs in us.items()}}
    md = res["median_us"]
    res["seqpack_gb_per_s_written"] = round(out_bytes / (md["seqpack"] * 1e3), 1)
    res["seqpack_frac_of_inrun_copy"] = round(md["memcpy"] / md["seqpack"], 3)
    res["seqpack_speedup_vs_torch"] = round(md["torch"] / md["seqpack"], 2)
    del sets
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_seqpack_b200.json"))
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--plan-reps", type=int, default=7)
    ap.add_argument("--only", default="", help="comma-separated workload names")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_seqpack.py needs a CUDA device")
    torch.cuda.set_device(0)
    out = {"gpu": gpu_info(), "launches": a.launches, "reps": a.reps, "rotating_sets": ROT, "workloads": []}
    for name, make, key in WORKLOADS:
        if a.only and name not in a.only.split(","):
            continue
        r = run_workload(name, make, key, a.launches, a.reps, a.plan_reps)
        print(json.dumps(r), flush=True)
        out["workloads"].append(r)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
