"""K-mer tokens (K11, bsq_tokenize_kmer / bsq_tokenize_kmer_varlen) next to a copy of the same bytes and to the torch
recipe users run without it.

    python tools/bench_kmer.py [--out profiles/r08_kmer_b200.json] [--launches 100] [--reps 3]

Per workload, three arms timed with CUDA events over `--launches` back-to-back launches (the torch recipe: `--launches`
/ 5) that rotate over 4 input/output sets -- each workload's sets together are larger than the B200's 126 MB L2, so
every pass reads from HBM -- and the arms alternated `--reps` times in the same process:
  k11      bsq_tokenize_kmer (padded) or bsq_tokenize_kmer_varlen (padding-free), int32 ids;
  memcpy   bsq_memcpy_d2d moving the k11 arm's algorithmic bytes (half of them read, half written): residues and offsets
           read, tokens (and cu_seqlens) written;
  torch    the recipe without K11 on the same device batch: batch_tokenize to int64 codes, a second LUT pass (the raw
           bytes through a BYTES tokenizer) for invalid residues, unfold(-1, k, s) and a multiply-sum against b ** arange,
           where for unk, the single-residue tail by gather, BOS / EOS / PAD by scatter, and for padding-free output
           out[mask] and a cumsum for cu_seqlens; int32 at the end.
The k11 output is asserted equal to the torch recipe's once per workload.  GPU name and power limit are read in the
same run.  Targets (goals, not measurements): k11 >= 5x the torch recipe everywhere, padded forms >= 0.5 of the copy.
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

from bioseq_b200 import capi, cbioseq  # noqa: E402
from bioseq_b200.synth import gen, AA20  # noqa: E402

ROT = 4
DNA150 = (106, 262144, 150, 150, b"ACGT")
DNA10K = (107, 4096, 10000, 10000, b"ACGT")
C2 = (102, 65536, 50, 1022, AA20)

# name, generator, key, k, stride, tail, padded padlen (None: padding-free)
WORKLOADS = [
    ("DNA150_dnabert_k6s1_padded", DNA150, "DNA", 6, 1, "drop", 147),
    ("DNA150_dnabert_k6s1_varlen", DNA150, "DNA", 6, 1, "drop", None),
    ("DNA150_nt_k6s6_padded", DNA150, "DNA", 6, 6, "single", 27),
    ("DNA150_nt_k6s6_varlen", DNA150, "DNA", 6, 6, "single", None),
    ("DNA10k_dnabert_k6s1_padded", DNA10K, "DNA", 6, 1, "drop", 9997),
    ("DNA10k_dnabert_k6s1_varlen", DNA10K, "DNA", 6, 1, "drop", None),
    ("DNA10k_nt_k6s6_padded", DNA10K, "DNA", 6, 6, "single", 1672),
    ("DNA10k_nt_k6s6_varlen", DNA10K, "DNA", 6, 6, "single", None),
    ("C2_protein_k3s1_padded1024", C2, "PROTEIN", 3, 1, "drop", 1024),
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


def time_launches(fn, launches):
    for i in range(4):
        fn(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(launches):
        fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1000.0 / launches  # us per launch


def torch_recipe(t_codes, t_bytes, lut, d_b, d_o, n, maxlen, lens, k, s, single, ids, P):
    """What a user writes without K11 (see the module docstring); returns padded (n, P) or (tokens, cu_seqlens)."""
    dev = d_b.device
    codes = t_codes.batch_tokenize_packed(d_b, d_o, padlen=maxlen, destchar="l", batch_first=True, check_lengths=False)       # (n, maxlen)
    bad = lut[t_bytes.batch_tokenize_packed(d_b, d_o, padlen=maxlen, destchar="l", batch_first=True, check_lengths=False)] < 0
    b = ids["b"]
    pw = b ** torch.arange(k - 1, -1, -1, device=dev, dtype=torch.int64)
    kid = (codes.unfold(-1, k, s) * pw).sum(-1)                                                          # (n, M)
    kid = torch.where(bad.unfold(-1, k, s).any(-1), ids["unk"], kid)
    m = torch.where(lens >= k, torch.div(lens - k, s, rounding_mode="floor") + 1, 0)
    covered = torch.where(m > 0, (m - 1) * s + k, 0)
    r = (lens - covered) if single else torch.zeros_like(lens)
    W = int(kid.shape[1] + (maxlen if single else 0))
    J = torch.arange(W, device=dev)[None, :]
    tok = torch.where(J < m[:, None], kid.gather(1, J.clamp(max=kid.shape[1] - 1).expand(n, -1)), ids["fill"])
    if single:
        ridx = (covered[:, None] + J - m[:, None]).clamp(0, maxlen - 1)
        sval = torch.where(bad.gather(1, ridx), ids["unk"], ids["nk"] + codes.gather(1, ridx))
        tok = torch.where((J >= m[:, None]) & (J < (m + r)[:, None]), sval, tok)
    T = m + r + 2
    width = max(P or 0, int(W) + 2)
    out = torch.full((n, width), ids["fill"], dtype=torch.int64, device=dev)
    out[:, 0] = ids["bos"]
    out[:, 1:1 + W] = tok
    out.scatter_(1, (T - 1)[:, None], ids["eos"])
    if P is not None:
        return out[:, :P].to(torch.int32)
    mask = torch.arange(width, device=dev)[None, :] < T[:, None]
    cu = torch.zeros(n + 1, dtype=torch.int32, device=dev)
    cu[1:] = torch.cumsum(T, 0).to(torch.int32)
    return out[mask].to(torch.int32), cu


def run_workload(name, g, key, k, s, tail, P, launches, reps):
    single = tail == "single"
    tok = capi.tokenizer(key, eos=True, bos=True, padchar=True)
    km = capi.kmer_desc(tok, k, s, capi.KMER_SINGLE if single else capi.KMER_DROP)
    buf, offs = gen(*g)
    n, L = offs.size - 1, int(offs[-1])
    lens = np.diff(offs)
    total, longest = capi.kmer_extent_host(offs, n, km)
    varlen = P is None
    assert varlen or longest <= P
    out_elems = total if varlen else n * P
    alg = L + 8 * (n + 1) + 4 * out_elems + (4 * (n + 1) if varlen else 0)
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    d_b0, d_o0 = torch.from_numpy(buf).to(dev), torch.from_numpy(offs).to(dev)
    sets = []
    for _ in range(ROT):
        sets.append({"b": d_b0.clone(), "o": d_o0.clone(), "out": torch.empty(out_elems, dtype=torch.int32, device=dev),
                     "cu": torch.empty(n + 1, dtype=torch.int32, device=dev),
                     "cpy": torch.empty(alg // 2 + 16, dtype=torch.uint8, device=dev)})

    def k11(i):
        x = sets[i % ROT]
        if varlen:
            capi.tokenize_kmer_varlen(0, st, x["b"], x["o"], n, tok, km, capi.I32, x["out"], x["cu"])
        else:
            capi.tokenize_kmer(0, st, x["b"], x["o"], n, P, tok, km, capi.I32, x["out"])

    def memcpy(i):
        x, y = sets[i % ROT], sets[(i + 1) % ROT]
        capi.check(capi.lib().bsq_memcpy_d2d(0, st, x["cpy"].data_ptr(), y["cpy"].data_ptr(), alg // 2))

    t_codes = cbioseq.Tokenizer(key)
    t_bytes = cbioseq.Tokenizer("BYTES")
    lut_np = np.array(tok.lut, np.int64)
    lut_np[0x80:] = -1
    lut = torch.from_numpy(lut_np).to(dev)
    d_lens = torch.from_numpy(lens).to(dev)
    ids = {"b": int(km.nchars), "nk": int(km.nkmers), "unk": int(km.unk_id), "bos": int(km.bos_id), "eos": int(km.eos_id),
           "fill": int(km.pad_id)}
    maxlen = int(lens.max())

    def recipe(i):
        x = sets[i % ROT]
        x["torch"] = torch_recipe(t_codes, t_bytes, lut, x["b"], x["o"], n, maxlen, d_lens, k, s, single, ids, P)

    k11(0)
    recipe(0)
    torch.cuda.synchronize()
    if varlen:
        same = bool(torch.equal(sets[0]["out"], sets[0]["torch"][0])) and bool(torch.equal(sets[0]["cu"], sets[0]["torch"][1]))
    else:
        same = bool(torch.equal(sets[0]["out"].view(n, P), sets[0]["torch"]))
    assert same, f"{name}: K11 differs from the torch recipe"
    for x in sets:
        x.pop("torch", None)
    arms = {"k11": (k11, launches), "memcpy": (memcpy, launches), "torch": (recipe, max(launches // 5, 4))}
    us = {a: [] for a in arms}
    for _ in range(reps):
        for a, (fn, nl) in arms.items():
            us[a].append(time_launches(fn, nl))
            for x in sets:
                x.pop("torch", None)
    med = {a: round(statistics.median(v), 2) for a, v in us.items()}
    res = {"workload": name, "gen": list(g[:4]) + [g[4].decode()], "tokenizer": [key, True, True, True], "k": k, "stride": s,
           "tail": tail, "form": "padding-free" if varlen else f"padded {P}", "destchar": "i", "n": n, "residues": L,
           "tokens_written": out_elems, "alg_bytes": alg, "k11_equals_torch_recipe": same,
           "us_per_launch": {a: [round(x, 2) for x in v] for a, v in us.items()}, "median_us": med,
           "k11_gb_per_s": round(alg / (med["k11"] * 1e3), 1), "k11_frac_of_inrun_copy": round(med["memcpy"] / med["k11"], 3),
           "k11_speedup_vs_torch": round(med["torch"] / med["k11"], 2)}
    res["targets"] = {"speedup_ge_5x": res["k11_speedup_vs_torch"] >= 5.0,
                      "padded_ge_0.5_copy": None if varlen else res["k11_frac_of_inrun_copy"] >= 0.5}
    del sets
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_kmer_b200.json"))
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default="", help="comma-separated workload names")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_kmer.py needs a CUDA device")
    torch.cuda.set_device(0)
    out = {"gpu": gpu_info(), "launches": a.launches, "reps": a.reps, "rotating_sets": ROT, "l2_note":
           "each workload's 4 rotating input/output sets exceed the 126 MB L2", "workloads": []}
    for name, g, key, k, s, tail, P in WORKLOADS:
        if a.only and name not in a.only.split(","):
            continue
        r = run_workload(name, g, key, k, s, tail, P, a.launches, a.reps)
        print(json.dumps(r), flush=True)
        out["workloads"].append(r)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
