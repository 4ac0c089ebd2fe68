"""Masked-language-model batches (K8, bsq_tokenize_mlm / bsq_tokenize_varlen_mlm) next to what users do without them.

    python tools/bench_mlm.py [--out profiles/r05_mlm_b200.json] [--launches 100] [--reps 3]

Per workload, three arms timed with CUDA events over `--launches` back-to-back calls that rotate over 4 input/output
sets (each workload's sets together are larger than the B200's 126 MB L2), the arms alternated `--reps` times in the
same process:
  fused   one K8 launch: masked inputs + int64 labels (+ cu_seqlens), default fractions 0.15 / 0.8 / 0.1;
  torch   batch_tokenize (K1s, or K1v for the padding-free form) followed by the HuggingFace-collator recipe in torch:
          a residue mask from the lengths, torch.rand for the selection, labels by where, the 80 / 10 / 10 replacement
          with two more rand draws, randint and two index_puts, int64 casts;
  memcpy  bsq_memcpy_d2d moving the fused arm's algorithmic bytes (half of them read, half written).
Algorithmic bytes of the fused arm: L + 8 (n + 1) + n P (s + 8) padded, L + 8 (n + 1) + T (s + 8) + 4 (n + 1)
padding-free (s = input element size).  The fused output is checked for consistency once per workload (unselected
positions keep the token, selected ones carry it as their label).  GPU name and power limit are read in the same run.
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

from bioseq_b200 import capi, consumers  # noqa: E402
from bioseq_b200.synth import gen, AA20  # noqa: E402
from bench_varlen import gpu_info, measured_peak, time_launches  # noqa: E402

ROT = 4

# name, (seed, n, lo, hi, alphabet), tokenizer (key, bos, eos, padchar), destchar, padlen (None: padding-free)
WORKLOADS = [
    ("C2_padded_u8", (102, 65536, 50, 1022, AA20), ("PROTEIN", True, True, True), "B", 1024),
    ("C2x4_padded_u8", (102, 4 * 65536, 50, 1022, AA20), ("PROTEIN", True, True, True), "B", 1024),
    ("C2_varlen_u8", (102, 65536, 50, 1022, AA20), ("PROTEIN", True, True, True), "B", None),
    ("DNA150_varlen_pbeos_u8", (106, 262144, 150, 150, b"ACGT"), ("DNA", True, True, True), "B", None),
    ("C2_padded_i64", (102, 65536, 50, 1022, AA20), ("PROTEIN", True, True, True), "l", 1024),
]


def run_workload(name, g, tk, destchar, padlen, launches, reps, peak):
    key, bos, eos, pad = tk
    tok = capi.tokenizer(key, eos=eos, bos=bos, padchar=pad)
    kind = capi.kind_of(destchar)
    s = int(capi.lib().bsq_kind_size(kind))
    dtype = {1: torch.uint8, 8: torch.int64}[s]
    k = int(bos) + int(eos)
    varlen = padlen is None
    buf, offs = gen(*g)
    n, L = offs.size - 1, int(offs[-1])
    lens = np.diff(offs)
    T = L + n * k
    shape = (T,) if varlen else (n, padlen)
    alg = L + 8 * (n + 1) + (T * (s + 8) + 4 * (n + 1) if varlen else n * padlen * (s + 8))
    maskfrac, mask_prob, random_prob = 0.15, 0.8, 0.1
    mask_id = tok.alphabet_size
    m = capi.mlm_desc(1, 0, consumers._mlm_thresholds(maskfrac, mask_prob, random_prob), mask_id, -100)
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    d_b0, d_o0 = torch.from_numpy(buf).to(dev), torch.from_numpy(offs).to(dev)
    sets = []
    for _ in range(ROT):
        sets.append({"b": d_b0.clone(), "o": d_o0.clone(), "in": torch.empty(shape, dtype=dtype, device=dev),
                     "lab": torch.empty(shape, dtype=torch.int64, device=dev), "tok": torch.empty(shape, dtype=dtype, device=dev),
                     "cu": torch.empty(n + 1, dtype=torch.int32, device=dev),
                     "cpy": torch.empty(alg // 2 + 16, dtype=torch.uint8, device=dev)})
    # eligible positions, as a collator builds them from the lengths
    d_lens = torch.from_numpy(lens).to(dev)
    if varlen:
        row = torch.repeat_interleave(torch.arange(n, device=dev), d_lens + k)
        cu64 = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        cu64[1:] = torch.cumsum(d_lens + k, 0)
        col = torch.arange(T, device=dev) - cu64[row]
        residue = (col >= int(bos)) & (col < int(bos) + d_lens[row])
    else:
        cols = torch.arange(padlen, device=dev)[None, :]
        residue = (cols >= int(bos)) & (cols < int(bos) + d_lens[:, None])

    def fused(i):
        x = sets[i % ROT]
        if varlen:
            capi.tokenize_varlen_mlm(0, st, x["b"], x["o"], n, tok, kind, m, x["in"], x["lab"], x["cu"])
        else:
            capi.tokenize_mlm(0, st, x["b"], x["o"], n, padlen, tok, kind, m, x["in"], x["lab"])

    def torch_recipe(i):
        x = sets[i % ROT]
        if varlen:
            capi.tokenize_varlen(0, st, x["b"], x["o"], n, tok, kind, x["tok"], x["cu"])
        else:
            capi.tokenize(0, st, x["b"], x["o"], n, padlen, tok, True, kind, x["tok"])
        tokens = x["tok"]
        labels = tokens.long()
        selected = (torch.rand(shape, device=dev) < maskfrac) & residue
        labels = torch.where(selected, labels, torch.full_like(labels, -100))
        replaced = (torch.rand(shape, device=dev) < mask_prob) & selected
        inputs = tokens.clone()
        inputs[replaced] = mask_id
        randomized = (torch.rand(shape, device=dev) < random_prob / (1 - mask_prob)) & selected & ~replaced
        words = torch.randint(tok.nchars, shape, device=dev, dtype=dtype)
        inputs[randomized] = words[randomized]
        x["torch_out"] = (inputs, labels)

    def memcpy(i):
        a, b = sets[i % ROT], sets[(i + 1) % ROT]
        capi.check(capi.lib().bsq_memcpy_d2d(0, st, a["cpy"].data_ptr(), b["cpy"].data_ptr(), alg // 2))

    fused(0)
    if varlen:
        capi.tokenize_varlen(0, st, d_b0, d_o0, n, tok, kind, sets[1]["tok"], sets[1]["cu"])
    else:
        capi.tokenize(0, st, d_b0, d_o0, n, padlen, tok, True, kind, sets[1]["tok"])
    torch.cuda.synchronize()
    inp, lab, plain = sets[0]["in"], sets[0]["lab"], sets[1]["tok"]
    sel = lab != -100
    consistent = bool(torch.equal(inp[~sel], plain[~sel]) and torch.equal(lab[sel], plain[sel].long())
                      and not bool((sel & ~residue).any()))
    sel_share = float(sel.sum().item()) / float(residue.sum().item())
    arms = {"fused": fused, "torch": torch_recipe, "memcpy": memcpy}
    us = {a: [] for a in arms}
    for _ in range(reps):
        for a, fn in arms.items():
            us[a].append(time_launches(fn, launches if a != "torch" else max(10, launches // 5)))
    res = {"workload": name, "form": "varlen" if varlen else "padded", "gen": list(g[:4]) + [g[4].decode()],
           "tokenizer": list(tk), "destchar": destchar, "n": n, "residues": L, "positions": T if varlen else n * padlen,
           "padlen": padlen, "input_itemsize": s, "alg_bytes": alg, "fused_output_consistent": consistent,
           "selected_share_of_residues": round(sel_share, 5),
           "us_per_call": {a: [round(v, 2) for v in xs] for a, xs in us.items()},
           "median_us": {a: round(statistics.median(xs), 2) for a, xs in us.items()}}
    md = res["median_us"]
    res["fused_gb_per_s"] = round(alg / (md["fused"] * 1e3), 1)
    res["fused_frac_of_inrun_copy"] = round(md["memcpy"] / md["fused"], 3)
    if peak:
        res["fused_frac_of_measured_peak"] = round(alg / (md["fused"] * 1e3) / peak, 3)
    res["fused_speedup_vs_torch_recipe"] = round(md["torch"] / md["fused"], 2)
    del sets
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_mlm_b200.json"))
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default="", help="comma-separated workload names")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_mlm.py needs a CUDA device")
    torch.cuda.set_device(0)
    peak = measured_peak()
    out = {"gpu": gpu_info(), "launches": a.launches, "torch_launches": max(10, a.launches // 5), "reps": a.reps,
           "rotating_sets": ROT, "measured_peak_gbs": peak, "workloads": []}
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
