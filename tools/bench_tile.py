"""Sliding-window tiling (K13a, bsq_tile) and stitching (K13b, bsq_untile_mean) next to a copy of the same bytes and to
what users do without them.

    python tools/bench_tile.py [--out profiles/r10_tile_b200.json] [--launches 50] [--torch-launches 10] [--reps 3]

Per workload, arms timed with CUDA events over back-to-back calls that rotate over 4 input/output sets (each workload's
sets together are larger than the B200's 126 MB L2), the arms alternated `--reps` times in the same process.
Tiling workloads (T*):
  k13a       one bsq_tile (out_offsets, seq_ptr, seq_index and starts written);
  memcpy     bsq_memcpy_d2d (cudaMemcpyAsync device to device) of the bytes k13a writes;
  torch      the torch recipe on the window table (given to it for free): window ids by repeat_interleave, an int64 source
             index, one gather;
  at T1 and T3 also, with DNA `pbeos` tokens at padlen W + 2 (batch-first u8):
  k13a_k1s   bsq_tile, then bsq_tokenize (K1s) of the windows; torch_k1s: the torch recipe, then the same bsq_tokenize.
Stitching workloads (U*):
  k13b       one bsq_untile_mean;
  memcpy     a copy of (bytes read + bytes written) / 2, i.e. the same HBM traffic as k13b's reads and writes;
  torch      the index_add_ recipe on precomputed int64 indices: a gather of the window rows, index_add_ of the values and
             of ones into float32 sums and counts, a division.  Its sums are unordered, so the outputs are compared
             with a tolerance.
Workloads:
  T1  16 x 8 000 000 DNA, W = 1 000, S = 500, END;
  T2  65 536 protein sequences, lognormal lengths (median 300, sigma 1.0, clipped to [30, 34 000]), W = 1 022, S = 511,
      SHORT;
  T3  4 096 x 10 000 DNA, W = S = 512, SHORT;
  T4  16 x 8 000 000 DNA, W = 131 072, S = 65 536, SHORT;
  U1  T1's windows, C = 1 float32, padded P = 1 002 (BOS at column 0);
  U2  64 x 100 000 DNA, W = 1 000, S = 500, C = 64 bf16, padding-free.
Each kernel's output is compared once per workload with the torch recipe's.  Targets: k13a >= 0.5 of the in-run copy and
>= 10x the torch recipe at T1, T3 and T4; k13b >= 0.5 of the copy and >= 5x the recipe.  GPU name and power limit are
read in the same run.
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
from bench_crop import lognormal_batch  # noqa: E402

ROT = 4
DNA5 = b"ACGTN"


def fixed_batch(seed, n, length):
    rng = np.random.default_rng(seed)
    a = np.frombuffer(DNA5, dtype=np.uint8)
    return np.ascontiguousarray(a[rng.integers(0, len(a), size=n * length)]), np.arange(n + 1, dtype=np.int64) * length


def t2_batch():
    return lognormal_batch(110, 65536, 300, 1.0, 30, 34000)


# name, batch, W, S, tail, tokenize
TILE_WORKLOADS = [
    ("T1_dna_16x8000000_W1000_S500_end", lambda: fixed_batch(110, 16, 8_000_000), 1000, 500, capi.TILE_END, True),
    ("T2_X1_protein_W1022_S511_short", t2_batch, 1022, 511, capi.TILE_SHORT, False),
    ("T3_dna_4096x10000_W512_S512_short", lambda: fixed_batch(111, 4096, 10_000), 512, 512, capi.TILE_SHORT, True),
    ("T4_dna_16x8000000_W131072_S65536_short", lambda: fixed_batch(112, 16, 8_000_000), 131_072, 65_536, capi.TILE_SHORT, False),
]
TILE_TARGETS = {"T1": (0.5, 10.0), "T3": (0.5, 10.0), "T4": (0.5, 10.0)}


def summarise(us, res, kernel, copy_target, torch_target):
    md = {a: round(statistics.median(xs), 2) for a, xs in us.items()}
    res["us_per_call"] = {a: [round(v, 2) for v in xs] for a, xs in us.items()}
    res["median_us"] = md
    res[f"{kernel}_frac_of_inrun_copy"] = round(md["memcpy"] / md[kernel], 3)
    res[f"{kernel}_speedup_vs_torch"] = round(md["torch"] / md[kernel], 2)
    if copy_target is not None:
        res["targets"] = {"frac_of_copy": {"target": copy_target, "met": res[f"{kernel}_frac_of_inrun_copy"] >= copy_target},
                          "speedup_vs_torch": {"target": torch_target, "met": res[f"{kernel}_speedup_vs_torch"] >= torch_target}}
    return md


def tile_tables(offs, W, S, tail):
    """Host window table (the torch recipe gets it for free): per window its source start, length and output start."""
    lens = np.diff(offs)
    starts, wl, seq = [], [], []
    for i, n in enumerate(lens):
        n = int(n)
        if n <= W:
            js = [(0, n)]
        elif tail == capi.TILE_DROP:
            js = [(j * S, W) for j in range((n - W) // S + 1)]
        else:
            m = -(-(n - W) // S) + 1
            js = [(j * S, min(W, n - j * S)) for j in range(m)]
            if tail == capi.TILE_END:
                js[-1] = (n - W, W)
        starts += [int(offs[i]) + s for s, _ in js]
        wl += [ln for _, ln in js]
        seq += [i] * len(js)
    wl = np.array(wl, np.int64)
    oo = np.zeros(wl.size + 1, np.int64)
    np.cumsum(wl, out=oo[1:])
    return np.array(starts, np.int64), wl, oo, np.array(seq, np.int64)


def run_tile(name, make, W, S, tail, tokenize, launches, torch_launches, reps):
    buf, offs = make()
    n = offs.size - 1
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    M, nbytes, longest = capi.tile_extent_host(offs, n, W, S, tail)
    src_start, wl, oo, _ = tile_tables(offs, W, S, tail)
    P = W + 2
    tok = capi.tokenizer("DNA", eos=True, bos=True, padchar=True)
    d_b0, d_o0 = torch.from_numpy(buf).to(dev), torch.from_numpy(offs).to(dev)
    sets = []
    for _ in range(ROT):
        x = {"b": d_b0.clone(), "o": d_o0.clone(), "tb": torch.empty(nbytes, dtype=torch.uint8, device=dev),
             "to": torch.empty(M + 1, dtype=torch.int64, device=dev), "sp": torch.empty(n + 1, dtype=torch.int64, device=dev),
             "si": torch.empty(M, dtype=torch.int64, device=dev), "st": torch.empty(M, dtype=torch.int64, device=dev)}
        if tokenize:
            x["tok"] = torch.empty((M, P), dtype=torch.uint8, device=dev)
        sets.append(x)
    del d_b0
    t_start, t_len = torch.from_numpy(src_start).to(dev), torch.from_numpy(wl).to(dev)
    t_oo = torch.from_numpy(oo).to(dev)

    def torch_tile(x):
        win = torch.repeat_interleave(torch.arange(M, device=dev), t_len, output_size=nbytes)
        idx = t_start[win] + torch.arange(nbytes, device=dev) - t_oo[:-1][win]
        return x["b"][idx]

    def k13a(i):
        x = sets[i % ROT]
        capi.tile(0, st, x["b"], x["o"], n, W, S, tail, x["tb"], x["to"], x["sp"], x["si"], x["st"])

    k13a(0)
    torch.cuda.synchronize()
    consistent = bool(torch.equal(sets[0]["tb"], torch_tile(sets[0])) and torch.equal(sets[0]["to"], t_oo))

    def memcpy(i):
        a, b = sets[i % ROT], sets[(i + 1) % ROT]
        capi.check(capi.lib().bsq_memcpy_d2d(0, st, a["tb"].data_ptr(), b["tb"].data_ptr(), nbytes))

    def torch_arm(i):
        torch_tile(sets[i % ROT])

    def k13a_k1s(i):
        k13a(i)
        x = sets[i % ROT]
        capi.tokenize(0, st, x["tb"], x["to"], M, P, tok, True, capi.I8, x["tok"])

    def torch_k1s(i):
        x = sets[i % ROT]
        capi.tokenize(0, st, torch_tile(x), t_oo, M, P, tok, True, capi.I8, x["tok"])

    arms = {"k13a": (k13a, launches), "memcpy": (memcpy, launches), "torch": (torch_arm, torch_launches)}
    if tokenize:
        arms.update({"k13a_k1s": (k13a_k1s, launches), "torch_k1s": (torch_k1s, torch_launches)})
    us = {a: [] for a in arms}
    for _ in range(reps):
        for a, (fn, k) in arms.items():
            us[a].append(time_launches(fn, k))
    res = {"workload": name, "n": n, "window": W, "stride": S, "tail": {0: "short", 1: "end", 2: "drop"}[tail], "windows": M,
           "bytes_read": int(offs[-1] - offs[0]), "bytes_written": nbytes, "k13a_matches_torch_recipe": consistent}
    copy_target, torch_target = TILE_TARGETS.get(name[:2], (None, None))
    md = summarise(us, res, "k13a", copy_target, torch_target)
    res["k13a_gb_per_s_written"] = round(nbytes / (md["k13a"] * 1e3), 1)
    if tokenize:
        res["k13a_k1s_speedup_vs_torch_k1s"] = round(md["torch_k1s"] / md["k13a_k1s"], 2)
    del sets
    torch.cuda.empty_cache()
    return res


def run_untile(name, make, W, S, tail, C, dtype, varlen, launches, torch_launches, reps):
    buf, offs = make()
    n = offs.size - 1
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    M, nbytes, _ = capi.tile_extent_host(offs, n, W, S, tail)
    src_start, wl, oo, seq = tile_tables(offs, W, S, tail)
    R = int(offs[-1] - offs[0])
    P = W + 2
    d_o = torch.from_numpy(offs).to(dev)
    seq_ptr = torch.from_numpy(np.searchsorted(seq, np.arange(n + 1)).astype(np.int64)).to(dev)
    if varlen:
        cu = torch.from_numpy(np.arange(M + 1, dtype=np.int64) * 2 + oo).to(dev)  # [BOS] residues [EOS] per window
        rows = int(cu[-1])
        cu32 = cu.int()
    else:
        rows = M * P
    esz = torch.empty(0, dtype=dtype).element_size()
    sets = []
    g = torch.Generator(device=dev).manual_seed(3)
    y0 = torch.randn((rows, C), generator=g, device=dev).to(dtype)
    for _ in range(ROT):
        sets.append({"y": y0.clone(), "out": torch.empty((R, C), dtype=torch.float32, device=dev)})
    del y0
    # the recipe's int64 indices: per window residue its row in y and its source row
    t_len = torch.from_numpy(wl).to(dev)
    win = torch.repeat_interleave(torch.arange(M, device=dev), t_len, output_size=nbytes)
    t = torch.arange(nbytes, device=dev) - torch.from_numpy(oo).to(dev)[:-1][win]
    ybase = cu[:-1][win] if varlen else win * P
    yrow = ybase + 1 + t
    srow = torch.from_numpy(src_start - int(offs[0])).to(dev)[win] + t
    del win, t, ybase
    dt = {torch.float32: capi.UNTILE_F32, torch.bfloat16: capi.UNTILE_BF16, torch.float16: capi.UNTILE_F16}[dtype]

    def k13b(i):
        x = sets[i % ROT]
        capi.untile_mean(0, st, dt, x["y"], C, 0 if varlen else P, cu32 if varlen else None, 1, d_o, n, W, S, tail, seq_ptr, M, 1,
                         None, x["out"])

    def torch_untile(x):
        s = torch.zeros((R, C), dtype=torch.float32, device=dev)
        c = torch.zeros(R, dtype=torch.float32, device=dev)
        s.index_add_(0, srow, x["y"][yrow].float())
        c.index_add_(0, srow, torch.ones(nbytes, dtype=torch.float32, device=dev))
        return s / c[:, None]

    k13b(0)
    torch.cuda.synchronize()
    diff = float((sets[0]["out"] - torch_untile(sets[0])).abs().max())
    read = nbytes * C * esz + (n + 1) * 16 + M * 8
    written = R * C * 4

    def memcpy(i):
        a, b = sets[i % ROT], sets[(i + 1) % ROT]
        capi.check(capi.lib().bsq_memcpy_d2d(0, st, a["y"].data_ptr(), b["y"].data_ptr(), (read + written) // 2))

    def torch_arm(i):
        torch_untile(sets[i % ROT])

    arms = {"k13b": (k13b, launches), "memcpy": (memcpy, launches), "torch": (torch_arm, torch_launches)}
    us = {a: [] for a in arms}
    for _ in range(reps):
        for a, (fn, k) in arms.items():
            us[a].append(time_launches(fn, k))
    res = {"workload": name, "n": n, "window": W, "stride": S, "channels": C, "dtype": str(dtype).replace("torch.", ""),
           "layout": "padding-free" if varlen else f"padded P={P}", "windows": M, "residues": R, "bytes_read": read,
           "bytes_written": written, "k13b_max_abs_diff_vs_torch_recipe": diff}
    md = summarise(us, res, "k13b", 0.5, 5.0)
    res["k13b_gb_per_s_read_plus_write"] = round((read + written) / (md["k13b"] * 1e3), 1)
    del sets
    torch.cuda.empty_cache()
    return res


UNTILE_WORKLOADS = [
    ("U1_T1_windows_C1_f32_padded", lambda: fixed_batch(110, 16, 8_000_000), 1000, 500, capi.TILE_END, 1, torch.float32, False),
    ("U2_dna_64x100000_W1000_S500_C64_bf16_varlen", lambda: fixed_batch(113, 64, 100_000), 1000, 500, capi.TILE_SHORT, 64,
     torch.bfloat16, True),
]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_tile_b200.json"))
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--torch-launches", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default="", help="comma-separated workload prefixes (T1, U2, ...)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_tile.py needs a CUDA device")
    torch.cuda.set_device(0)
    out = {"gpu": gpu_info(), "launches": a.launches, "torch_launches": a.torch_launches, "reps": a.reps, "rotating_sets": ROT,
           "workloads": []}
    only = [x for x in a.only.split(",") if x]
    for w in TILE_WORKLOADS + UNTILE_WORKLOADS:
        if only and not any(w[0].startswith(p) for p in only):
            continue
        r = (run_tile(*w, a.launches, a.torch_launches, a.reps) if w[0][0] == "T" else
             run_untile(*w, a.launches, a.torch_launches, a.reps))
        print(json.dumps(r), flush=True)
        out["workloads"].append(r)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
