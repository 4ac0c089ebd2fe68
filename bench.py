#!/usr/bin/env python
"""bench.py -- Gbases/s of the batch-tokenisation hot path on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch: BASELINE.json configs[1], PROTEIN
`pbeos` batch_tokenize (BOS+EOS+PAD), 65536 ragged sequences of 50..1022 residues, padlen 1024,
batch_first, 1-byte tokens -- per GPU (weak scaling: every rank owns its own shard of
sequences; the path has no collective).  Units are input residues ("bases").

  value     device-resident: packed residues + offsets already in HBM, one kernel launch per
            step through the C ABI (bsq_tokenize), CUDA events on the launching stream.  The
            batches rotate through ROT distinct input/output sets so every step reads and
            writes memory that is not in L2 (ROT x 103 MB > 126 MB).
  e2e       the same batch through the public Python API with HOST buffers
            (Tokenizer.batch_tokenize_packed on pinned numpy-visible memory): pipelined
            host->device copies + kernels + a device->host read of the last output row, per step.
  roofline  HBM-bound: algorithmic bytes per launch (residues + offsets + output, DESIGN.md
            section 4) / average launch duration, against MEASURED_PEAKS.json's copy bandwidth.
  cpu_baseline  (rank 0, N=1) the reference's own OpenMP tokenizer (oracle/_ref, built from
            /root/reference) on the same batch with all host threads; its output is also the
            parity check of the timed GPU batch.

--impl reference times only that CPU arm and prints the same JSON shape.

--dump-outputs DIR writes what the timed call returned in its last step: a fixed sample of DUMP_ROWS rows of the
(65536, 1024) token matrix as DIR/tokens.npy (float32; token ids are exact) and their indices as DIR/rows.npy
(float64).  The inputs are seeded, so two builds can be compared output for output.  The reference arm times the
batch of the GPU arm's last step (rotation index (K - 1) % 4), so the two arms' files can be compared as well.  With
N > 1 ranks every rank writes tokens_rank<r>.npy / rows_rank<r>.npy for its own shard, DUMP_ROWS // N rows each:
at most 33.6 MB in all, whatever N.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

NSEQ, LO, HI, PADLEN = 65536, 50, 1022, 1024
KEY, FLAGS = "PROTEIN", dict(bos=True, eos=True, padchar=True)
ROT = 4
DUMP_ROWS, DUMP_SEED = 8192, 2024      # 8192 x 1024 float32 = 33.6 MB over all ranks
WORKLOAD = ("configs[1]: PROTEIN pbeos batch_tokenize (BOS+EOS+PAD), 65536 ragged seqs len 50-1022, "
            "padlen 1024, batch_first, 1-byte tokens, per GPU")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


_SYNTH = None


def synth():
    """bioseq_b200/synth.py (pure numpy) loaded by path: the reference arm must not import the product package
    (that would map libbsq.so / the cbioseq extension into the process that times the reference)."""
    global _SYNTH
    if _SYNTH is None:
        import importlib.util
        spec = importlib.util.spec_from_file_location("_bsq_synth", os.path.join(ROOT, "bioseq_b200", "synth.py"))
        _SYNTH = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(_SYNTH)
    return _SYNTH


def make_batch(seed):
    sy = synth()
    return sy.gen(seed, NSEQ, LO, HI, sy.AA20)


def bench_config(world):
    """The one `config` object both arms print (the driver compares them field by field)."""
    return {"workload": WORKLOAD, "seqs_per_gpu": NSEQ, "padlen": PADLEN, "len_range": [LO, HI], "alphabet": "AA20 uniform",
            "tokenizer": "PROTEIN bos+eos+padchar", "batch_first": True, "dtype": "u8", "seed": 102,
            "l2": f"inputs+outputs rotate through {ROT} distinct 103 MB sets (> 126 MB L2)",
            "parallelism": f"{world} ranks, sequences sharded by index (byte-balanced ranges), no collective"}


def dump_rows(nseq, world):
    """The sorted row indices --dump-outputs keeps of one rank's batch: the same for every run with the same batch size
    and rank count.  Each of the `world` ranks keeps DUMP_ROWS // world rows, so the whole dump stays at DUMP_ROWS rows."""
    return np.sort(np.random.default_rng(DUMP_SEED).choice(nseq, size=min(nseq, DUMP_ROWS // world), replace=False))


def dump_outputs(d, rows, tokens, rank, world):
    os.makedirs(d, exist_ok=True)
    sfx = f"_rank{rank}" if world > 1 else ""
    np.save(os.path.join(d, f"tokens{sfx}.npy"), np.ascontiguousarray(tokens).view(np.uint8).astype(np.float32))
    np.save(os.path.join(d, f"rows{sfx}.npy"), rows.astype(np.float64))


def algorithmic_bytes(nbases, nseq, padlen, itemsize=1, ncols=1):
    """SURVEY.md 8(d): residues + offsets + every output byte once; no memset term."""
    return nbases + 8 * (nseq + 1) + padlen * nseq * ncols * itemsize


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed regions run."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        hi = [s for s, p in zip(sm, power) if p >= 0.5 * max(power)] or sm     # samples under load
        return {"sm_mhz": statistics.median(hi), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


def cpu_arm(buf, offs, steps, warmup, budget_s=20.0, opt="O3", nthreads=None):
    """The reference's CPU implementation on the host cores (oracle/_ref), else the C port."""
    as_list = synth().as_list
    from oracle.oracle import load_ref, OracleTokenizer
    nbases = int(offs[-1])
    R = load_ref(opt=opt)
    cores = nthreads or os.cpu_count() or 1
    if R is not None:
        tok = R.Tokenizer(KEY, **FLAGS)
        seqs = as_list(buf, offs)
        fn = lambda: tok.batch_tokenize(seqs, padlen=PADLEN, destchar="B", batch_first=True, nthreads=cores)  # noqa: E731
        kind, used = "reference", cores
        flags = "-O3 -march=x86-64-v3 -fopenmp" if opt == "O3" else "-O0 -fopenmp (the flags the reference ships with, setup.py:50-55)"
        how = f"oracle/_ref (reference src/tokenize.cpp, g++ {flags}), nthreads={cores}, list[bytes] input"
    else:
        tok = OracleTokenizer(KEY, **FLAGS)
        fn = lambda: tok.batch_tokenize((buf, offs), padlen=PADLEN, destchar="B", batch_first=True)  # noqa: E731
        kind, used = "port", 1
        how = "oracle/bsq_oracle.c (scalar C port), 1 thread, packed input"
    out = None
    for _ in range(max(1, warmup)):
        out = fn()
    times = []
    t_begin = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        out = fn()
        times.append(time.perf_counter() - t0)
        if budget_s is not None and time.perf_counter() - t_begin > budget_s:
            break
    total = sum(times)
    return {"value": nbases * len(times) / total / 1e9, "unit": "Gbases/s", "cores": used, "kind": kind,
            "sample": f"{len(times)} full passes over the {NSEQ}-sequence batch ({nbases} bases each); {how}",
            "ms_per_step": 1e3 * total / len(times), "best_ms": 1e3 * min(times)}, out


def native_so_loaded():
    """Shared objects of this repository mapped into the process right now (the driver records the same from outside)."""
    out = set()
    try:
        for ln in open("/proc/self/maps"):
            path = ln.rsplit(None, 1)[-1]
            if path.startswith(ROOT) and ".so" in os.path.basename(path):
                out.add(os.path.relpath(path, ROOT))
    except OSError:
        pass
    return sorted(out)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    buf, offs = make_batch(102 + (args.steps - 1) % ROT)   # the batch of the GPU arm's last timed step
    res, out = cpu_arm(buf, offs, args.steps, args.warmup, budget_s=None, opt=args.ref_opt, nthreads=args.ref_threads or None)
    if args.dump_outputs:
        rows = dump_rows(len(offs) - 1, 1)
        dump_outputs(args.dump_outputs, rows, np.ascontiguousarray(out)[rows], 0, 1)
    line = {"impl": "reference", "metric": "tokenize_throughput", "value": res["value"], "unit": "Gbases/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": bench_config(args.gpus), "note": "CPU arm: one host, all threads; not sharded over GPUs",
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": res["value"], "unit": "Gbases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "native_so_loaded": native_so_loaded()}
    print(json.dumps(line), flush=True)


def cpu_arm_subprocess(opt, nthreads, steps=3, warmup=1):
    """Another build / thread count of the reference, timed in its own process (the -O3 and -O0 builds both register
    the pybind11 type `Tokenizer`: only one of them can live in a process)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps), "--warmup", str(warmup),
           "--ref-opt", opt, "--ref-threads", str(nthreads)]
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env).stdout.strip().splitlines()
        d = json.loads(out[-1])
        return dict(d["cpu_baseline"], ms_per_step=d["ms_per_step"])
    except Exception as e:   # a missing -O0 build etc.: reported, not fatal
        return {"unavailable": repr(e)[:200]}


def rank_batches(rank, world):
    """This rank's ROT batches.  N = 1: BASELINE.json configs[1] as is (seed 102 + r).  N > 1: the N ranks' batches are
    one global batch of N x 65536 sequences (chunk c = gen(102 + 1000 c + r)), partitioned the way DESIGN.md section 6
    describes -- contiguous sequence ranges holding equal shares of the RESIDUES (bioseq_b200/shard.py, the same split
    as the C ABI's bsq_shard_bounds) -- so the byte-balanced partition is the one that is timed."""
    sy = synth()
    if world == 1:
        return [make_batch(102 + r) for r in range(ROT)], None
    import importlib.util
    spec = importlib.util.spec_from_file_location("_bsq_shard", os.path.join(ROOT, "bioseq_b200", "shard.py"))
    sh = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sh)
    sets, info = [], []
    for r in range(ROT):
        lens = np.concatenate([sy.gen_lens(102 + 1000 * c + r, NSEQ, LO, HI) for c in range(world)])
        goffs = np.zeros(lens.size + 1, dtype=np.int64)
        np.cumsum(lens, out=goffs[1:])
        bounds = sh.shard_bounds(goffs, world)
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        parts = []
        for c in range(lo // NSEQ, (hi - 1) // NSEQ + 1):
            cb, co = sy.gen(102 + 1000 * c + r, NSEQ, LO, HI, sy.AA20)
            i0, i1 = max(lo - c * NSEQ, 0), min(hi - c * NSEQ, NSEQ)
            parts.append(cb[co[i0]:co[i1]])
        buf = np.ascontiguousarray(np.concatenate(parts))
        offs = np.ascontiguousarray(goffs[lo:hi + 1] - goffs[lo])
        assert offs[-1] == buf.size
        sets.append((buf, offs))
        info.append({"first_seq": lo, "nseq": hi - lo, "bases": int(buf.size)})
    return sets, info


def run_ours(args):
    import torch
    import ctypes as C
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cpus = os.cpu_count() or 1
    # host threads per rank for the pack / bounce loops: the ranks of one box share its cores
    host_threads = max(1, (cpus * 3 // 4) // world)
    os.environ.setdefault("BSQ_POOL_CAP", str(host_threads))
    from bioseq_b200 import capi
    import bioseq_b200

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        # The path has no data-path collective: the ranks only meet at barriers and to reduce their timings.  Those
        # go over gloo (host tensors) while anything is being timed, and NCCL is brought up AFTER the timed sections for
        # the final reduction of the reported numbers: an initialised NCCL communicator makes every kernel launch of the
        # process ~1-2 us slower (measured on one GPU with a 1-rank group: 21.1 -> 22.0 us per 20 us launch, without PDL
        # 22.8 -> 24.9; gpurun_out/r02m), which is 5-10 % of this workload's step and has nothing to do with the path.
        import torch.distributed as dist
        dist.init_process_group("gloo")
    dev = local
    L = capi.lib()
    tok = capi.tokenizer(KEY, **FLAGS)
    ptok = bioseq_b200.Tokenizer(KEY, **FLAGS)

    # ---- inputs: ROT distinct batches per rank, resident in HBM ---------------------------------
    batches, shard_info = rank_batches(rank, world)
    sets = []
    for buf, offs in batches:
        n = len(offs) - 1
        sets.append({"buf": buf, "offs": offs, "n": n, "nbases": int(offs[-1]),
                     "d_bytes": torch.from_numpy(buf).cuda(), "d_offs": torch.from_numpy(offs).cuda(),
                     "out": torch.empty((n, PADLEN), dtype=torch.uint8, device="cuda")})
    st = torch.cuda.current_stream().cuda_stream
    for s in sets:
        capi.check_lengths_device(dev, st, s["d_offs"], s["n"], PADLEN, tok)
    calls = [(dev, st, s["d_bytes"].data_ptr(), s["d_offs"].data_ptr(), s["n"], PADLEN, C.byref(tok), 1, capi.I8,
              s["out"].data_ptr()) for s in sets]

    def step(i):
        rc = L.bsq_tokenize(*calls[i % ROT])
        if rc:
            capi.check(rc)

    sampler = ClockSampler(local)
    # clocks ramp from idle: keep the GPU busy for a moment before anything is timed
    t_end = time.perf_counter() + 0.5
    i = 0
    while time.perf_counter() < t_end:
        step(i); i += 1
    torch.cuda.synchronize()
    if rank == 0 and args.smi != "off":
        sampler.start()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: device-resident, exactly K steps ------------------------------------------------
    for i in range(args.warmup):
        step(i)
    barrier()
    L.bsq_launch_count_reset()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    t_host0 = time.perf_counter()
    for i in range(args.steps):
        step(i)
    host_us_per_launch = (time.perf_counter() - t_host0) / args.steps * 1e6   # host time to enqueue a step (the device must not wait for it)
    ev[1].record()
    barrier()
    launches = int(L.bsq_launch_count())
    ms_total = ev[0].elapsed_time(ev[1])
    bases_timed = sum(sets[i % ROT]["nbases"] for i in range(args.steps))
    alg_bytes = sum(algorithmic_bytes(sets[i % ROT]["nbases"], sets[i % ROT]["n"], PADLEN) for i in range(args.steps))
    dumped = None
    if args.dump_outputs:   # copied out now, written once every timed section is over
        final = sets[(args.steps - 1) % ROT]
        rows = dump_rows(final["n"], world)
        dumped = (rows, final["out"][torch.from_numpy(rows).cuda()].cpu().numpy())

    # ---- the same HBM traffic as a plain device-to-device copy, in the same run, rotated the same way -------------
    # (cudaMemcpyAsync of half the step's algorithmic bytes: reads n and writes n.)  What a 103 MB launch can reach at
    # all on this part -- launch ramp and tail included -- is this number, not the 2 GiB burst copy of MEASURED_PEAKS.
    half = int(alg_bytes / args.steps / 2) // 256 * 256
    half = min(half, min(s["out"].numel() for s in sets))
    cdst = [torch.empty(half, dtype=torch.uint8, device="cuda") for _ in range(ROT)]

    def copy_step(i):
        L.bsq_memcpy_d2d(dev, st, cdst[i % ROT].data_ptr(), sets[i % ROT]["out"].data_ptr(), half)
    for i in range(args.warmup):
        copy_step(i)
    barrier()
    ev[0].record()
    for i in range(args.steps):
        copy_step(i)
    ev[1].record()
    barrier()
    copy_us = ev[0].elapsed_time(ev[1]) / args.steps * 1e3
    del cdst

    clocks_early = None
    if args.smi == "value":
        # K steps last a few ms, less than one nvidia-smi sampling period: keep the very same launches going
        # (untimed) so that the sampler sees the clocks of this load, then stop it -- an nvidia-smi poller
        # stalls CUDA API calls of the host-side (e2e) sections on virtualised hosts (tools/e2e_probe2.py).
        t_end = time.perf_counter() + 1.2
        i = 0
        while time.perf_counter() < t_end:
            for _ in range(64):
                step(i); i += 1
            torch.cuda.synchronize()
        if rank == 0:
            clocks_early = sampler.stop()
            clocks_early["sampled_over"] = "warm-up, the K timed launches and 1.2 s of the same launches back to back (untimed)"
        barrier()

    # ---- e2e: the reference's own call -- Tokenizer.batch_tokenize(list[bytes]) -- with HOST items: item walk, pinned
    # pack, host->device copies and kernels inside the timed region, plus a device->host read of the last output row ----
    sections = set(args.sections.split(","))
    as_list = synth().as_list
    lists = [as_list(s["buf"], s["offs"]) for s in sets] if "e2e" in sections else None
    pinned = [(torch.from_numpy(s["buf"]).pin_memory(), torch.from_numpy(s["offs"]).pin_memory()) for s in sets]
    last = torch.empty(PADLEN, dtype=torch.uint8).pin_memory()

    def e2e_step(i):
        out = ptok.batch_tokenize(lists[i % ROT], padlen=PADLEN, destchar="B", batch_first=True, nthreads=host_threads)
        last.copy_(out[-1], non_blocking=True)
        return out

    def e2e_packed_step(i):
        hb, ho = pinned[i % ROT]
        out = ptok.batch_tokenize_packed(hb, ho, padlen=PADLEN, destchar="B", batch_first=True)
        last.copy_(out[-1], non_blocking=True)
        return out

    def timed_region(fn, nsteps, repeats):
        """`repeats` back-to-back repeats of the same nsteps-step region; the median repeat is reported (a host hiccup --
        page-locking, another tenant of the box -- inside one repeat would otherwise decide the number)."""
        reps, out = [], None
        for _ in range(repeats):
            barrier()
            t0 = time.perf_counter()
            for i in range(nsteps):
                out = fn(i)
            torch.cuda.synchronize()
            reps.append(time.perf_counter() - t0)
        return sorted(reps)[len(reps) // 2], reps, out

    e2e_steps = max(3, min(args.steps, 50)) if "e2e" in sections else 1
    e2e_s, e2e_repeats, e2e_ok, packed_s, packed_repeats, packed_ok = 1.0, [1.0], None, 1.0, [1.0], None
    if "e2e" in sections:
        for i in range(2 * ROT):   # every set goes through the link once before timing
            e2e_step(i)
        e2e_s, e2e_repeats, out = timed_region(e2e_step, e2e_steps, 5)
        e2e_ok = bool(torch.equal(out, sets[(e2e_steps - 1) % ROT]["out"]))
        for i in range(2 * ROT):
            e2e_packed_step(i)
        packed_s, packed_repeats, out = timed_region(e2e_packed_step, e2e_steps, 5)
        packed_ok = bool(torch.equal(out, sets[(e2e_steps - 1) % ROT]["out"]))
        del out
    barrier()
    # host link: every rank copies at the same moment (barrier-aligned); the sum over ranks is the roofline of the
    # e2e numbers (at N=8 well below N x the single-GPU rate)
    host_link = None
    if "e2e" in sections:
        barrier()
        host_link = measure_host_link(torch, barrier)
        hl = torch.tensor([host_link["h2d_gbs"]], dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(hl, op=dist.ReduceOp.SUM)
        host_link["h2d_gbs_all_ranks_concurrent"] = hl.tolist()[0]
        barrier()
        hm = torch.tensor([measure_host_memcpy(barrier, host_threads)], dtype=torch.float64)
        host_link["host_memcpy_gbs_this_rank"] = hm.tolist()[0]
        if dist is not None:
            dist.all_reduce(hm, op=dist.ReduceOp.SUM)
        host_link["host_memcpy_gbs_all_ranks_concurrent"] = hm.tolist()[0]
        host_link["host_memcpy_threads_per_rank"] = int(host_threads)
        barrier()
    lists = None
    e2e_bases = sum(sets[i % ROT]["nbases"] for i in range(e2e_steps))
    h2d = int(np.mean([s["nbases"] + 8 * (s["n"] + 1) for s in sets]))

    # ---- parity of the timed output on EVERY rank: the reference's own tokenizer on a sample of this rank's batch ----
    step(0)
    torch.cuda.synchronize()
    parity_rank = rank_parity(sets[0], as_list)

    # ---- C5 on every rank (configs[4]: sharded tokenize + one-hot with H2D staging) ----------
    c5 = None
    if "c5" in sections:
        barrier()
        c5 = c5_slice(torch, capi, L, dev, st, rank, barrier)
        barrier()
    c5f = None
    if "c5full" in sections or ("c5" in sections and world == 8 and args.c5full != "off") or args.c5full == "on":
        barrier()
        c5f = c5_full(torch, capi, L, dev, st, rank, world, barrier, host_threads, with_cpu=(rank == 0))
        barrier()

    # ---- reduce over ranks: max time ------------------------------------------------------------
    c5v = [c5["ms_h2d_inclusive"], c5["ms_device_resident"]] if c5 else [0.0, 0.0]
    c5s = [c5["bases"], c5["h2d_bytes"], c5["alg_bytes_device"], c5["bases_device"]] if c5 else [0.0] * 4
    c5fv = [c5f["ms_pass"], c5f["ms_pass_mapped"], c5f["ms_pass_registered"]] if c5f else [0.0, 0.0, 0.0]
    c5fs = [c5f["bases"], c5f["h2d_bytes"], float(c5f["parity"])] if c5f else [0.0, 0.0, 1.0]
    t = torch.tensor([ms_total, e2e_s * 1e3, packed_s * 1e3, copy_us] + c5v + c5fv, dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(bases_timed), float(e2e_bases), float(alg_bytes), float(launches)] + [float(x) for x in c5s] + c5fs[:2],
                       dtype=torch.float64, device="cuda")
    ok = torch.tensor([float(parity_rank["ok"]), float(e2e_ok is not False), float(packed_ok is not False), c5fs[2]], dtype=torch.float64, device="cuda")
    nccl_ranks = 1
    if dist is not None:
        # every timed section is over: NCCL (NVLink / NVSwitch) carries the reduction of the reported numbers
        barrier()
        pg = dist.new_group(backend="nccl", device_id=torch.device("cuda", local))
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=pg)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM, group=pg)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=pg)
        one = torch.ones(1, dtype=torch.float64, device="cuda")
        dist.all_reduce(one, op=dist.ReduceOp.SUM, group=pg)
        nccl_ranks = int(one.item())
    ms_total_max, e2e_ms_max, packed_ms_max, copy_us_max, c5_ms_h2d, c5_ms_dev, c5f_ms, c5f_ms_mapped, c5f_ms_reg = t.tolist()
    bases_all, e2e_bases_all, alg_all, launches_all, c5_bases, c5_h2d_bytes, c5_alg, c5_bases_dev, c5f_bases, c5f_h2d = tot.tolist()
    parity_all, e2e_all_ok, packed_all_ok, c5f_parity = [bool(x) for x in ok.tolist()]
    if not parity_all:
        raise SystemExit("bench.py: GPU output differs from the CPU reference on at least one rank -- refusing to report a number")

    extra = {}
    cpu = None
    parity = None
    if rank == 0:
        if "extra" in sections:
            extra = secondary_measurements(torch, capi, L, dev, st)
        if "frows" in sections:
            extra["f_rows"] = f_rows_measurements(torch, capi, L, dev, st)
        if "c4" in sections and world == 1:
            extra["c4_reduced_alphabets_1M_roundtrip"] = c4_measurements(torch, capi, L, dev, st, with_cpu="cpu" in sections)
        clocks = clocks_early if clocks_early is not None else sampler.stop()
        cpu_more = {}
        if world == 1 and "cpu" in sections:
            cpu, ref_out = cpu_arm(sets[0]["buf"], sets[0]["offs"], steps=10, warmup=1, budget_s=20.0)
            parity = bool(np.array_equal(np.ascontiguousarray(ref_out).view(np.uint8), sets[0]["out"].cpu().numpy()))
            if not parity:
                raise SystemExit("bench.py: GPU output differs from the CPU reference -- refusing to report a number")
            # SURVEY.md 8(d): the reference as shipped (-O0, setup.py:50-55) and the one-thread picture
            cpu_more["cpu_baseline_O0"] = cpu_arm_subprocess("O0", cpus)
            cpu_more["cpu_baseline_1thread"] = cpu_arm_subprocess("O3", 1)
        peak, peak_src = measured_peak()
        per_launch_ms = ms_total / launches if launches else float("nan")          # this rank's launches
        achieved = (alg_bytes / max(launches, 1)) / (per_launch_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                traffic = tj.get("tokenize_span_kernel")
                traffic_src = {k: tj.get(k) for k in ("captured_at_commit", "source", "note")}
            except Exception:
                traffic = None
        copy_bytes = 2 * half
        line = {
            "metric": "tokenize_throughput", "value": bases_all / (ms_total_max * 1e-3) / 1e9, "unit": "Gbases/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": bench_config(world), "ranks_seen_by_nccl": nccl_ranks,
            "bases_per_step_per_gpu": int(np.mean([s["nbases"] for s in sets])), "shard_of_rank0": shard_info,
            "e2e": {"value": e2e_bases_all / (e2e_ms_max * 1e-3) / 1e9, "unit": "Gbases/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": PADLEN, "steps": e2e_steps,
                    "api": f"Tokenizer.batch_tokenize(list[bytes], padlen=1024, batch_first=True, nthreads={host_threads}) -- the reference's own call (src/tokenize.cpp:82-98)",
                    "repeats_ms_per_step": [round(x * 1e3 / e2e_steps, 4) for x in e2e_repeats],
                    "matches_device_resident": e2e_all_ok, "host_threads_per_rank": host_threads, "host_cpus": cpus,
                    "packed_pinned_input": {"value": e2e_bases_all / (packed_ms_max * 1e-3) / 1e9, "unit": "Gbases/s",
                                            "api": "Tokenizer.batch_tokenize_packed(pinned bytes, pinned offsets) -- additive entry point, no per-item host work",
                                            "repeats_ms_per_step": [round(x * 1e3 / e2e_steps, 4) for x in packed_repeats],
                                            "matches_device_resident": packed_all_ok},
                    "host_link": None if host_link is None else dict(
                        host_link,
                        frac_list_api=(h2d * e2e_steps * world / (e2e_ms_max * 1e-3) / 1e9) / host_link["h2d_gbs_all_ranks_concurrent"],
                        frac_packed=(h2d * e2e_steps * world / (packed_ms_max * 1e-3) / 1e9) / host_link["h2d_gbs_all_ranks_concurrent"],
                        frac_list_api_of_host_memcpy=(h2d * e2e_steps * world / (e2e_ms_max * 1e-3) / 1e9) / host_link["host_memcpy_gbs_all_ranks_concurrent"],
                        note="frac = e2e H2D bytes/s over the pinned H2D rate of all ranks copying at once (best of 256 MiB copies and double-buffered 46 MB copies); "
                             "frac_list_api_of_host_memcpy = the same bytes/s over the host's own copy rate (all ranks' gather threads copying at once): "
                             "the list-of-items call gathers every residue from its Python object into the pinned pack, a host-memory-bound step")},
            "gpu_launches": int(launches_all), "native_so_loaded": native_so_loaded(),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel": "tokenize_span_kernel (K1s)",
                         "algorithmic_bytes_per_launch": int(alg_bytes / max(launches, 1)),
                         "launch_us": per_launch_ms * 1e3, "host_enqueue_us_per_launch": host_us_per_launch,
                         "copy_reference": {"what": "cudaMemcpyAsync device-to-device of the same traffic (read n + write n), same rotation, same run, max over ranks",
                                            "bytes": copy_bytes, "us": copy_us_max, "GB/s": copy_bytes / copy_us_max / 1e3,
                                            "frac_of_peak": copy_bytes / copy_us_max / 1e3 / peak,
                                            "kernel_us_over_copy_us": per_launch_ms * 1e3 / copy_us_max}},
            "cpu_baseline": cpu, "parity_vs_cpu_reference": parity, "parity_every_rank": dict(parity_rank, all_ranks_ok=parity_all),
            "clocks": clocks, "extra": extra,
        }
        line.update(cpu_more)
        if c5:
            hl = (host_link or {}).get("h2d_gbs_all_ranks_concurrent")
            line["c5_slice"] = {
                "workload": (f"configs[4] in bounded form, per GPU: {c5['nchunks']} chunks x {c5['chunk']} protein seqs (len 50-650), PROTEIN pbeos, "
                             f"padlen {c5['padlen']}: pinned H2D (double-buffered) + int8 tokens (B,P) + uint8 one-hot (P,B,23) into a ring of 2 buffers"),
                "n_gpus": world, "bases": int(c5_bases),
                "h2d_inclusive": {"Gbases/s": c5_bases / c5_ms_h2d / 1e6, "ms_per_pass": c5_ms_h2d,
                                  "h2d_GB/s_all_ranks": c5_h2d_bytes / c5_ms_h2d / 1e6,
                                  "frac_of_host_link": None if not hl else c5_h2d_bytes / c5_ms_h2d / 1e6 / hl},
                "device_resident": {"Gbases/s": c5_bases_dev / c5_ms_dev / 1e6, "ms_per_pass": c5_ms_dev, "GB/s_all_ranks": c5_alg / c5_ms_dev / 1e6,
                                    "frac_of_measured_hbm": c5_alg / c5_ms_dev / 1e6 / (peak * world)},
            }
        if c5f:
            hl = (host_link or {}).get("h2d_gbs_all_ranks_concurrent")
            line["c5_full"] = dict(c5f["report"], n_gpus=world, seqs_total=int(c5f["nseq"]) * world, bases_total=int(c5f_bases),
                                   ms_per_pass_max_over_ranks=c5f_ms, Gbases_per_s=c5f_bases / c5f_ms / 1e6,
                                   h2d_GBs_all_ranks=c5f_h2d / c5f_ms / 1e6,
                                   frac_of_host_link=None if not hl else c5f_h2d / c5f_ms / 1e6 / hl,
                                   mapped_file_pass={"ms_per_pass_max_over_ranks": c5f_ms_mapped, "Gbases_per_s": c5f_bases / c5f_ms_mapped / 1e6,
                                                     "h2d_GBs_all_ranks": c5f_h2d / c5f_ms_mapped / 1e6},
                                   registered_mapping_pass={"what": "FlatFile(prefault=2): the page-cache mapping page-locked in place (cudaHostRegister), direct DMA, no pinned copy of the file",
                                                            "registered_on_rank0": c5f["registered_ok"],
                                                            "ms_per_pass_max_over_ranks": c5f_ms_reg, "Gbases_per_s": c5f_bases / c5f_ms_reg / 1e6,
                                                            "h2d_GBs_all_ranks": c5f_h2d / c5f_ms_reg / 1e6},
                                   parity_sampled_chunk_every_rank=c5f_parity)
        print(json.dumps(line), flush=True)
    if dumped is not None:
        dump_outputs(args.dump_outputs, *dumped, rank, world)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def rank_parity(s, as_list, sample=4096):
    """The reference's own tokenizer (oracle/_ref; the C restatement if it is absent) on the first `sample` sequences of a
    batch, compared bit for bit with the GPU output of that batch."""
    from oracle.oracle import load_ref, OracleTokenizer
    m = min(sample, s["n"])
    offs = s["offs"][:m + 1]
    buf = s["buf"][:int(offs[-1])]
    R = load_ref()
    if R is not None:
        want = R.Tokenizer(KEY, **FLAGS).batch_tokenize(as_list(buf, offs), padlen=PADLEN, destchar="B", batch_first=True, nthreads=2)
        kind = "reference (oracle/_ref)"
    else:
        want = OracleTokenizer(KEY, **FLAGS).batch_tokenize((buf, offs), padlen=PADLEN, batch_first=True)
        kind = "port (oracle/bsq_oracle.c)"
    got = s["out"][:m].cpu().numpy()
    return {"ok": bool(np.array_equal(np.ascontiguousarray(want).view(np.uint8), got)), "rows_checked_per_rank": m, "checker": kind}


C4_KEYS = ("SEB6", "SEB8", "SEB10", "SEB14", "SEV10", "MURPHY", "LIA10", "LIB10", "DAYHOFF")


def c4_measurements(torch, capi, L, dev, st, with_cpu):
    """BASELINE.json configs[3]: reduced protein alphabets, tokenize + decode_tokens round trip, 1 M ragged
    sequences (SURVEY.md 8d C4: gen(104, 1e6, 50, 1024, AA20); pos tokenizers at padlen 1024, pbeos at 1026)."""
    import ctypes as C
    import bioseq_b200
    gen, AA20 = synth().gen, synth().AA20
    peak, _ = measured_peak()
    n = 1_000_000
    buf, offs = gen(104, n, 50, 1024, AA20)
    nbases = int(offs[-1])
    d_b, d_o = torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda()
    out = torch.empty(n * 1026, dtype=torch.uint8, device="cuda")
    res = {"nseq": n, "bases": nbases, "tokenize": {}, "decode": {}}
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for flavour, flags, padlen in (("pos", dict(padchar=True), 1024), ("pbeos", dict(bos=True, eos=True, padchar=True), 1026)):
        for key in C4_KEYS:
            tk = capi.tokenizer(key, **flags)
            call = (dev, st, d_b.data_ptr(), d_o.data_ptr(), n, padlen, C.byref(tk), 1, capi.I8, out.data_ptr())
            for _ in range(2):
                L.bsq_tokenize(*call)
            a.record()
            for _ in range(5):
                L.bsq_tokenize(*call)
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / 5
            nbytes = nbases + 8 * (n + 1) + n * padlen
            res["tokenize"][f"{key}_{flavour}"] = {"us_per_call": ms * 1e3, "Gbases/s": nbases / ms / 1e6,
                                                   "frac_of_measured_hbm": nbytes / ms / 1e6 / peak}
        # decode of the last alphabet's tokens: device part (validate + lengths + scan, then characters)
        toks = out[:n * padlen].view(n, padlen)
        d_ro = torch.empty(n + 1, dtype=torch.int64, device="cuda")
        d_tl = torch.empty(n, dtype=torch.int32, device="cuda")
        total = capi.decode_lengths(dev, st, toks, 1, n, padlen, padlen, 1, tk, d_ro, d_tl)
        d_ch = torch.empty(total, dtype=torch.uint8, device="cuda")
        tot = C.c_int64()

        def dec():
            L.bsq_decode_lengths(dev, st, toks.data_ptr(), 1, n, padlen, padlen, 1, C.byref(tk), d_ro.data_ptr(), d_tl.data_ptr(), C.byref(tot))
            L.bsq_decode_chars(dev, st, toks.data_ptr(), 1, n, padlen, padlen, 1, C.byref(tk), d_ro.data_ptr(), d_tl.data_ptr(), d_ch.data_ptr())
        dec()
        torch.cuda.synchronize()
        a.record()
        for _ in range(3):
            dec()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / 3
        nbytes = n * padlen + total + 8 * (n + 1)   # SURVEY.md 8(d)
        res["decode"][f"{key}_{flavour}_device"] = {"us_per_call": ms * 1e3, "Gtokens/s": n * padlen / ms / 1e6, "chars": int(total),
                                                    "GB/s": nbytes / ms / 1e6, "frac_of_measured_hbm": nbytes / ms / 1e6 / peak}
        # the public call on a slice of rows: device decode + D2H of the characters + Python str objects
        ptk = bioseq_b200.Tokenizer(key, **flags)
        rows = 32768
        ptk.decode_tokens(toks[:1024])
        t0 = time.perf_counter()
        strs = ptk.decode_tokens(toks[:rows])
        dt = time.perf_counter() - t0
        res["decode"][f"{key}_{flavour}_api_{rows}_rows"] = {"ms": dt * 1e3, "Gtokens/s": rows * padlen / dt / 1e9,
                                                             "chars": sum(map(len, strs))}
        if with_cpu:
            # checker + CPU baseline of the round trip: the reference's own tokenizer on the same rows
            as_list = synth().as_list
            from oracle.oracle import load_ref
            R = load_ref()
            if R is not None:
                m = 8192
                rt = R.Tokenizer(key, **flags)
                seqs = as_list(buf[:int(offs[m])], offs[:m + 1])
                t0 = time.perf_counter()
                rtoks = rt.batch_tokenize(seqs, padlen=padlen, destchar="B", batch_first=True, nthreads=os.cpu_count() or 1)
                t1 = time.perf_counter()
                rstrs = rt.decode_tokens(rtoks)
                t2 = time.perf_counter()
                ok = bool(np.array_equal(rtoks.view(np.uint8), toks[:m].cpu().numpy())) and rstrs == strs[:m]
                if not ok:
                    raise SystemExit(f"bench.py: C4 {key} {flavour}: GPU tokens/decoded strings differ from the CPU reference")
                res["decode"][f"{key}_{flavour}_cpu_reference_{m}_rows"] = {
                    "tokenize_ms": (t1 - t0) * 1e3, "decode_ms": (t2 - t1) * 1e3, "decode_Gtokens/s": m * padlen / (t2 - t1) / 1e9,
                    "parity": ok}
        del d_ch, d_ro
    return res


def c5_slice(torch, capi, L, dev, st, rank, barrier, nchunks=8, chunk=131072):
    """BASELINE.json configs[4], one GPU's share in bounded form: `nchunks` chunks of `chunk` protein sequences
    (lengths 50..650, seeds 105+chunk index as in SURVEY.md 8d C5), PROTEIN pbeos, padlen 652.  Each chunk goes
    pinned host -> device on a copy stream (double-buffered) and is tokenised (int8 (B,652)) and one-hot encoded
    (uint8 (652,B,23)) into a reused ring of two output buffers, like the full 8 M-sequences-per-GPU pass would."""
    import ctypes as C
    gen, AA20 = synth().gen, synth().AA20
    P, NC = 652, 23
    tk = capi.tokenizer(KEY, **FLAGS)
    host = []
    for c in range(nchunks):
        buf, offs = gen(105 + c + 1000 * rank, chunk, 50, 650, AA20)
        host.append((torch.from_numpy(buf).pin_memory(), torch.from_numpy(offs).pin_memory(), int(offs[-1])))
    maxb = max(h[2] for h in host)
    dbuf = [torch.empty(maxb + 64, dtype=torch.uint8, device="cuda") for _ in range(2)]
    doff = [torch.empty(chunk + 1, dtype=torch.int64, device="cuda") for _ in range(2)]
    toks = [torch.empty((chunk, P), dtype=torch.uint8, device="cuda") for _ in range(2)]
    oh = [torch.empty((P, chunk, NC), dtype=torch.uint8, device="cuda") for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    main = torch.cuda.current_stream()
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def one_pass(h2d):
        for c in range(nchunks):
            k = c % 2
            hb, ho, nb = host[c]
            if h2d:
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(consumed[k])
                    dbuf[k][:nb].copy_(hb, non_blocking=True)
                    doff[k].copy_(ho, non_blocking=True)
                    copied[k].record(copy_stream)
                main.wait_event(copied[k])
            L.bsq_tokenize(dev, st, dbuf[k].data_ptr(), doff[k].data_ptr(), chunk, P, C.byref(tk), 1, capi.I8, toks[k].data_ptr())
            L.bsq_onehot(dev, st, dbuf[k].data_ptr(), doff[k].data_ptr(), None, chunk, P, C.byref(tk), capi.I8, oh[k].data_ptr())
            consumed[k].record(main)

    for k in range(2):
        consumed[k].record(main)
    one_pass(True)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 2
    barrier()   # all ranks load the host links at the same moment (the data generation above takes seconds and drifts)
    t0 = time.perf_counter()
    a.record()
    for _ in range(reps):
        one_pass(True)
    b.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms_h2d = a.elapsed_time(b) / reps
    # device-resident share: the last two chunks are still in dbuf; re-run the kernels only
    a.record()
    for _ in range(reps):
        one_pass(False)
    b.record()
    torch.cuda.synchronize()
    ms_dev = a.elapsed_time(b) / reps
    # what the kernel-only pass actually read: chunks nchunks-2 / nchunks-1 alternate in the two device buffers
    bases = sum(h[2] for h in host)
    bases_dev = sum(host[nchunks - 2 + (c % 2)][2] for c in range(nchunks))
    alg = 2 * bases_dev + nchunks * (2 * 8 * (chunk + 1) + chunk * P + P * chunk * NC)
    return {"bases": bases, "ms_h2d_inclusive": max(ms_h2d, wall * 1e3 / reps), "ms_device_resident": ms_dev,
            "h2d_bytes": bases + nchunks * 8 * (chunk + 1), "alg_bytes_device": alg, "bases_device": bases_dev,
            "nchunks": nchunks, "chunk": chunk, "padlen": P}


def c5_full(torch, capi, L, dev, st, rank, world, barrier, host_threads, with_cpu, chunk=131072):
    """BASELINE.json configs[4] at its stated size: 64 M synthetic protein sequences over 8 GPUs = 8 M per GPU (lengths
    50..650, mean 350: 2.8 G residues per GPU; chunk seeds 105 + global chunk index as in SURVEY.md 8d C5), PROTEIN pbeos,
    padlen 652.  Every rank streams its share from a FlatFile -- the reference's on-disk packed layout (src/fxstats.cpp:50-59:
    u64 n | u64 offsets[n+1] | residues), consumed in bulk like FF2NP does (bioseq/loaders.py:11-26) -- in chunks of 131072
    sequences: mapped file -> pinned bounce ring -> device (two staging slots: the copy of chunk k+1 overlaps the kernels of
    chunk k), then int8 tokens (B, 652) and uint8 one-hot (652, B, 23) into a ring of two output buffers (the full one-hot
    would be 122 GB per GPU).  BSQ_C5_SEQS overrides the sequences per GPU (smoke runs)."""
    import ctypes as C
    import shutil
    import tempfile
    sy = synth()
    P, NC = 652, 23
    nseq = int(os.environ.get("BSQ_C5_SEQS", str(8 * 1024 * 1024)))
    nchunks = (nseq + chunk - 1) // chunk
    tk = capi.tokenizer(KEY, **FLAGS)
    root = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > (world + 1) * nseq * 400 else None
    td = tempfile.mkdtemp(prefix=f"bsq_c5_rank{rank}_", dir=root)
    path = os.path.join(td, "shard.ff")
    t0 = time.perf_counter()
    try:
        sizes = [min(chunk, nseq - c * chunk) for c in range(nchunks)]
        seeds = [105 + rank * nchunks + c for c in range(nchunks)]
        offs = np.zeros(nseq + 1, dtype=np.int64)
        pos = 0
        for c in range(nchunks):
            lens = sy.gen_lens(seeds[c], sizes[c], 50, 650)
            np.cumsum(lens, out=offs[pos + 1:pos + 1 + sizes[c]])
            offs[pos + 1:pos + 1 + sizes[c]] += offs[pos]
            pos += sizes[c]
        with open(path, "wb") as f:
            f.write(np.array([nseq], dtype=np.uint64).tobytes())
            f.write(offs.astype(np.uint64).tobytes())
            for c in range(nchunks):
                cb, co = sy.gen(seeds[c], sizes[c], 50, 650, sy.AA20)
                f.write(cb.tobytes())
        make_s = time.perf_counter() - t0
        stager = capi.Stager(dev)
        toks = [torch.empty((chunk, P), dtype=torch.uint8, device="cuda") for _ in range(2)]
        oh = [torch.empty((P, chunk, NC), dtype=torch.uint8, device="cuda") for _ in range(2)]
        ms, open_s = {}, {}
        registered_ok = None
        for mode, kw in (("pinned", dict(pinned=True)), ("registered", dict(prefault=2)), ("mapped", dict(prefault=True))):
            # pinned: the file is read into page-locked memory once (like loading a dataset), chunks DMA straight from it;
            # registered: the page-cache mapping itself is page-locked in place (cudaHostRegister), same direct DMA, no copy;
            # mapped: page-cache mapping, chunks bounce through the stager's pinned ring (pool threads, write-combining stores)
            t0 = time.perf_counter()
            ff = capi.FlatFile(path, **kw)
            open_s[mode] = time.perf_counter() - t0
            if mode == "registered":
                registered_ok = ff.pinned   # False: this platform cannot register a file mapping (the pass then equals "mapped")
            assert ff.nseqs == nseq
            fb, fo = ff.bytes_ptr, ff.offsets_ptr

            def run_chunk(c, k):
                n = sizes[c]
                db, do = stager.stage(st, fb, fo + 8 * c * chunk, n)
                L.bsq_tokenize(dev, st, db, do, n, P, C.byref(tk), 1, capi.I8, toks[k].data_ptr())
                rc = L.bsq_onehot(dev, st, db, do, None, n, P, C.byref(tk), capi.I8, oh[k].data_ptr())
                if rc:
                    capi.check(rc)
                stager.release(st)

            for c in range(min(2, nchunks)):   # warm-up: allocations, page-locking of the ring, kernels
                run_chunk(c, c % 2)
            torch.cuda.synchronize()
            barrier()
            t0 = time.perf_counter()
            for c in range(nchunks):
                run_chunk(c, c % 2)
            torch.cuda.synchronize()
            ms[mode] = (time.perf_counter() - t0) * 1e3
            if mode != "mapped":
                stager.sync_copies()
                ff.close()
        ms_pass = ms["pinned"]
        # parity: one sampled chunk per rank, its first rows against the reference's own tokenizer
        cs = (7 * rank + 3) % nchunks
        run_chunk(cs, 0)
        torch.cuda.synchronize()
        m = min(2048, sizes[cs])
        cb, co = sy.gen(seeds[cs], sizes[cs], 50, 650, sy.AA20)
        seqs = sy.as_list(cb[:int(co[m])], co[:m + 1])
        from oracle.oracle import load_ref, OracleTokenizer
        R = load_ref()
        if R is not None:
            rt = R.Tokenizer(KEY, **FLAGS)
            want_t = rt.batch_tokenize(seqs, padlen=P, destchar="B", batch_first=True, nthreads=2)
            want_o = rt.batch_onehot_encode(seqs, padlen=P, destchar="B", nthreads=2)
        else:
            ot = OracleTokenizer(KEY, **FLAGS)
            want_t = ot.batch_tokenize((cb[:int(co[m])], co[:m + 1]), padlen=P, batch_first=True)
            want_o = ot.batch_onehot_encode((cb[:int(co[m])], co[:m + 1]), padlen=P, destchar="B")
        ok = bool(np.array_equal(np.ascontiguousarray(want_t).view(np.uint8), toks[0][:m].cpu().numpy())) and \
            bool(np.array_equal(np.ascontiguousarray(want_o).view(np.uint8), oh[0][:, :m, :].contiguous().cpu().numpy()))
        cpu = None
        if with_cpu and R is not None:
            # CPU arm, extrapolated as SURVEY.md 8(d) prescribes: the reference on chunks that fit the host, scaled to 64 M
            rt = R.Tokenizer(KEY, **FLAGS)
            cores = os.cpu_count() or 1
            nseq_cpu = min(1 << 20, nseq)
            parts = [sy.gen(seeds[c], sizes[c], 50, 650, sy.AA20) for c in range((nseq_cpu + chunk - 1) // chunk)]
            big = [x for cb_, co_ in parts for x in sy.as_list(cb_, co_)][:nseq_cpu]
            bases_cpu = sum(map(len, big))
            rt.batch_tokenize(big[:8192], padlen=P, destchar="B", batch_first=True, nthreads=cores)
            tt = []
            for _ in range(2):
                t0 = time.perf_counter()
                rt.batch_tokenize(big, padlen=P, destchar="B", batch_first=True, nthreads=cores)
                tt.append(time.perf_counter() - t0)
            small = big[:65536]
            bases_small = sum(map(len, small))
            to = []
            for _ in range(2):
                t0 = time.perf_counter()
                rt.batch_onehot_encode(small, padlen=P, destchar="B", nthreads=cores)
                to.append(time.perf_counter() - t0)
            total_bases = 64 * (1 << 20) * 350.0
            s_tok, s_oh = min(tt) / bases_cpu * total_bases, min(to) / bases_small * total_bases
            cpu = {"kind": "reference", "cores": cores, "extrapolated": True,
                   "sample": f"oracle/_ref -O3: batch_tokenize on {nseq_cpu} sequences ({bases_cpu} bases, best of 2: {min(tt) * 1e3:.1f} ms) and "
                             f"batch_onehot_encode uint8 on 65536 sequences ({bases_small} bases, best of 2: {min(to) * 1e3:.1f} ms), nthreads={cores}, "
                             "list[bytes] input already in memory; scaled linearly to 64 M sequences x mean 350",
                   "tokenize_s_for_64M": s_tok, "onehot_s_for_64M": s_oh,
                   "Gbases/s_tokenize_plus_onehot": total_bases / (s_tok + s_oh) / 1e9}
        bases = int(offs[-1])
        report = {"workload": ("configs[4] at full size: 8 M synthetic protein sequences per GPU (len 50-650, mean 350) streamed from a FlatFile per rank "
                               f"in {nchunks} chunks of {chunk}: file held in page-locked memory -> device (2 staging slots; the mapped-file pass "
                               "bounces through the pinned ring instead), int8 tokens (B,652) + "
                               "uint8 one-hot (652,B,23) into a ring of 2 output buffers; PROTEIN pbeos"),
                  "seqs_per_gpu": nseq, "chunks_per_gpu": nchunks, "padlen": P, "file_bytes_per_gpu": os.path.getsize(path),
                  "file_dir": root or tempfile.gettempdir(), "file_make_s_rank0": make_s, "file_open_s_rank0": open_s, "cpu_baseline": cpu,
                  "device_bytes_written_per_gpu": nseq * P * (1 + NC)}
        stager.close()
        ff.close()
        return {"ms_pass": ms_pass, "ms_pass_mapped": ms["mapped"], "ms_pass_registered": ms["registered"], "registered_ok": registered_ok, "bases": bases, "h2d_bytes": bases + 8 * (nseq + nchunks), "parity": ok, "nseq": nseq, "report": report}
    finally:
        shutil.rmtree(td, ignore_errors=True)


def f_rows_measurements(torch, capi, L, dev, st):
    """SURVEY.md 8(f) rows built next to the hot path, each at the C2 batch (65536 ragged protein sequences, P = 1024)
    unless stated: K5 one-hot straight into the CNN's (B,C,L) float layout, K6 tokenize -> embedding rows, K7 BLOSUM62
    point mutations on the packed residues, and the FlatFile feeder (file -> GPU tokens, no per-sequence host work)."""
    import ctypes as C
    import tempfile
    import bioseq_b200
    gen, AA20 = synth().gen, synth().AA20
    peak, _ = measured_peak()
    res = {}

    def timed(fn, reps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    tk = capi.tokenizer(KEY, **FLAGS)
    ncols = tk.alphabet_size
    bufs = [gen(102 + r, NSEQ, LO, HI, AA20) for r in range(2)]
    dev_sets = [(torch.from_numpy(b).cuda(), torch.from_numpy(o).cuda(), int(o[-1])) for b, o in bufs]
    it = [0]

    def rot():
        it[0] += 1
        return dev_sets[it[0] % 2]

    # K5: (B, C, L) float32 one-hot, 16384 x 23 x 1024 x 4 B = 1.54 GB per call (write-bound)
    n5 = NSEQ // 4
    out5 = torch.empty((n5, ncols, PADLEN), dtype=torch.float32, device="cuda")
    def k5():
        d_b, d_o, _ = rot()
        capi.onehot_bcl(dev, st, d_b, d_o, None, n5, PADLEN, tk, capi.F32, out5)
    ms = timed(k5, 5)
    nb5 = int(bufs[0][1][n5])
    by = nb5 + 8 * (n5 + 1) + n5 * ncols * PADLEN * 4
    res["f4_onehot_bcl_f32_16384x23x1024"] = {"Gbases/s": nb5 / ms / 1e6, "GB/s": by / ms / 1e6, "frac_of_measured_hbm": by / ms / 1e6 / peak,
                                                "us_per_call": ms * 1e3}
    del out5
    # K6: tokenize -> embedding gather, D = 64 float32 (256 B rows), batch-first: 16384 x 1024 x 256 B = 4.3 GB per call
    D = 64
    w = torch.randn((ncols, D), dtype=torch.float32, device="cuda")
    out6 = torch.empty((n5, PADLEN, D), dtype=torch.float32, device="cuda")
    def k6():
        d_b, d_o, _ = rot()
        capi.embed(dev, st, d_b, d_o, n5, PADLEN, tk, True, w, ncols, D * 4, out6)
    ms = timed(k6, 5)
    by = nb5 + 8 * (n5 + 1) + n5 * PADLEN * D * 4
    res["f4_embed_f32_D64_16384x1024"] = {"Gbases/s": nb5 / ms / 1e6, "GB/s": by / ms / 1e6, "frac_of_measured_hbm": by / ms / 1e6 / peak,
                                           "us_per_call": ms * 1e3}
    del out6, w
    # K7: BLOSUM62 augmentation in place, one substitution per sequence (chain_len 1) and eight: touches one
    # 32-byte sector per substitution, so it is latency/launch-bound, not bandwidth-bound -- reported per sequence
    for chain in (1, 8):
        def k7():
            d_b, d_o, _ = rot()
            capi.augment_blosum62(dev, st, d_b, d_o, NSEQ, chain, 1.0, 1234, 0)
        ms = timed(k7, 20)
        res[f"f3_augment_blosum62_chain{chain}_65536_seqs"] = {"Gseqs/s": NSEQ / ms / 1e6, "us_per_call": ms * 1e3}
    # f1: FlatFile feeder.  The file is written once (FASTA -> flat file, the reference's FlatFile::make), then a whole
    # file goes file -> pinned copy / page cache -> GPU tokens through Tokenizer.batch_tokenize(FlatFile)
    ptok = bioseq_b200.Tokenizer(KEY, **FLAGS)
    buf, offs = bufs[0]
    with tempfile.TemporaryDirectory() as td:
        fa = os.path.join(td, "c2.fa")
        with open(fa, "wb") as f:
            for i in range(NSEQ):
                f.write(b">s\n")
                f.write(buf[offs[i]:offs[i + 1]].tobytes())
                f.write(b"\n")
        t0 = time.perf_counter()
        bioseq_b200.FlatFile(fa, fa + ".ff")
        make_s = time.perf_counter() - t0
        want = None
        for mode, kw in (("pinned", {"pinned": True}), ("mapped", {})):
            ff = bioseq_b200.FlatFile(fa + ".ff", **kw)
            for _ in range(5):
                o = ptok.batch_tokenize(ff, padlen=PADLEN, batch_first=True)
            torch.cuda.synchronize()
            reps, dts = 10, []
            for _ in range(3):   # three batches of calls, median batch reported (the mapped file's pages settle slowly on some hosts)
                t0 = time.perf_counter()
                for _ in range(reps):
                    o = ptok.batch_tokenize(ff, padlen=PADLEN, batch_first=True)
                torch.cuda.synchronize()
                dts.append((time.perf_counter() - t0) / reps)
            dt = sorted(dts)[1]
            if want is None:
                want = ptok.batch_tokenize_packed(torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda(), padlen=PADLEN, batch_first=True)  # (dev_sets were mutated by K7)
            res[f"f1_flatfile_{mode}_to_tokens_65536_seqs"] = {"Gbases/s": int(offs[-1]) / dt / 1e9, "ms_per_call": dt * 1e3,
                                                              "batches_ms_per_call": [round(x * 1e3, 3) for x in dts],
                                                              "matches_device_resident": bool(torch.equal(o, want))}
            del ff
        res["f1_flatfile_make_from_fasta"] = {"s": make_s, "MB/s": (int(offs[-1]) + 4 * NSEQ) / make_s / 1e6}
    return res


def measure_host_link(torch, barrier, nbytes=256 << 20, reps=5):
    """Pinned host->device copy rate of this rank's link with every rank copying at the same moment: the best of
    (a) back-to-back 256 MiB copies and (b) 46 MB copies alternating between two buffers on two streams (the shape of
    the staged pipelines) -- a denominator no measured section should exceed."""
    h = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    d.copy_(h, non_blocking=True)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best_big = 0.0
    for _ in range(2):
        barrier()
        a.record()
        for _ in range(reps):
            d.copy_(h, non_blocking=True)
        b.record()
        torch.cuda.synchronize()
        best_big = max(best_big, nbytes * reps / (a.elapsed_time(b) * 1e-3) / 1e9)
    m = 46 << 20
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    best_db = 0.0
    for _ in range(2):
        barrier()
        t0 = time.perf_counter()
        for k in range(16):
            with torch.cuda.stream(streams[k % 2]):
                d[(k % 2) * m:(k % 2 + 1) * m].copy_(h[(k % 4) * m:(k % 4 + 1) * m], non_blocking=True)
        torch.cuda.synchronize()
        best_db = max(best_db, 16 * m / (time.perf_counter() - t0) / 1e9)
    return {"h2d_gbs": max(best_big, best_db), "h2d_gbs_256MiB_copies": best_big, "h2d_gbs_double_buffered_46MB": best_db, "bytes": nbytes}


def measure_host_memcpy(barrier, nthreads, nbytes=256 << 20, reps=3):
    """Host-to-host copy rate of this rank with `nthreads` threads (numpy releases the GIL in copyto), every rank copying
    at the same moment: what the host's memory system gives the gather of the list-of-items call, which reads every
    residue from its Python object and writes it into the pinned pack while the DMA engine reads the previous pack."""
    import threading
    src = np.ones(nbytes, dtype=np.uint8)
    dst = np.empty(nbytes, dtype=np.uint8)
    dst[:] = 0
    nthreads = max(1, int(nthreads))
    cuts = [nbytes * k // nthreads for k in range(nthreads + 1)]
    best = 0.0
    for _ in range(reps):
        barrier()
        ts = [threading.Thread(target=np.copyto, args=(dst[cuts[k]:cuts[k + 1]], src[cuts[k]:cuts[k + 1]])) for k in range(nthreads)]
        t0 = time.perf_counter()
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        best = max(best, nbytes / (time.perf_counter() - t0) / 1e9)
    return best


def secondary_measurements(torch, capi, L, dev, st):
    """Other BASELINE.json configs, device-resident, reported under "extra" (not the headline)."""
    import ctypes as C
    gen = synth().gen
    peak, _ = measured_peak()
    res = {}

    profiling = os.environ.get("BSQ_BENCH_PROFILE") == "1"   # under ncu: one warm-up, one launch per case

    def timed(fn, reps):
        if profiling:
            reps = 1
        for _ in range(1 if profiling else 3):
            fn(0)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(reps):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    def report(name, ms, nbases, nbytes):
        res[name] = {"Gbases/s": nbases / ms / 1e6, "GB/s": nbytes / ms / 1e6, "frac_of_measured_hbm": nbytes / ms / 1e6 / peak,
                     "us_per_call": ms * 1e3}

    # C1: DNA 4096 x 1000, padlen 1024, batch-first; 8.3 MB per call, so stream 64 distinct batches
    tok = capi.tokenizer("DNA")
    nb = 64
    buf, offs = gen(101, 4096 * nb, 1000, 1000, b"ACGT")
    d_b, d_o = torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda()
    out = torch.empty((4096 * nb, 1024), dtype=torch.uint8, device="cuda")
    def c1(i):
        j = i % nb
        L.bsq_tokenize(dev, st, d_b.data_ptr(), d_o.data_ptr() + 8 * 4096 * j, 4096, 1024, C.byref(tok), 1, capi.I8,
                       out.data_ptr() + 4096 * 1024 * j)
    ms = timed(c1, 256)
    report("c1_dna_4096x1000_bf_u8_streamed", ms, 4096 * 1000, 4096 * 1000 + 8 * 4097 + 4096 * 1024)
    # the same 64 batches, 16 per launch (bsq_tokenize_many): what a caller with many small per-step batches uses
    import ctypes as C2
    groups = []
    for g in range(nb // 16):
        js = range(16 * g, 16 * g + 16)
        pb = (C2.c_void_p * 16)(*[d_b.data_ptr() for _ in js])
        po = (C2.c_void_p * 16)(*[d_o.data_ptr() + 8 * 4096 * j for j in js])
        ns = (C2.c_int64 * 16)(*[4096 for _ in js])
        pd = (C2.c_void_p * 16)(*[out.data_ptr() + 4096 * 1024 * j for j in js])
        groups.append((pb, po, ns, pd))
    def c1many(i):
        pb, po, ns, pd = groups[i % len(groups)]
        L.bsq_tokenize_many(dev, st, 16, pb, po, ns, 1024, C.byref(tok), 1, capi.I8, pd)
    ms = timed(c1many, 64) / 16
    report("c1_dna_4096x1000_bf_u8_many_16_per_launch", ms, 4096 * 1000, 4096 * 1000 + 8 * 4097 + 4096 * 1024)
    def c1big(i):
        L.bsq_tokenize(dev, st, d_b.data_ptr(), d_o.data_ptr(), 4096 * nb, 1024, C.byref(tok), 1, capi.I8, out.data_ptr())
    ms = timed(c1big, 10)
    report("c1x64_dna_262144x1000_bf_u8_one_launch", ms, 4096 * nb * 1000, 4096 * nb * (1000 + 8 + 1024))
    out_sf = torch.empty((1024, 4096 * nb), dtype=torch.uint8, device="cuda")
    def c1sf(i):
        L.bsq_tokenize(dev, st, d_b.data_ptr(), d_o.data_ptr(), 4096 * nb, 1024, C.byref(tok), 0, capi.I8, out_sf.data_ptr())
    ms = timed(c1sf, 10)
    report("c1x64_dna_seqfirst_u8_one_launch", ms, 4096 * nb * 1000, 4096 * nb * (1000 + 8 + 1024))
    del out, out_sf, d_b, d_o

    # C3: DNA one-hot float32 seq-first, 16384 x 4096 -> (4096, 16384, 4): 1.14 GB per call (> L2)
    buf, offs = gen(103, 16384, 4096, 4096, b"ACGT")
    d_b, d_o = torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda()
    out = torch.empty((4096, 16384, 4), dtype=torch.float32, device="cuda")
    def c3(i):
        L.bsq_onehot(dev, st, d_b.data_ptr(), d_o.data_ptr(), None, 16384, 4096, C.byref(tok), capi.F32, out.data_ptr())
    ms = timed(c3, 10)
    report("c3_dna_onehot_f32_16384x4096", ms, 16384 * 4096, 16384 * 4096 + 8 * 16385 + 4096 * 16384 * 16)
    del out, d_b, d_o

    # C2 variants: seq-first, unaligned padlen, protein one-hot u8, decode
    AA20 = synth().AA20
    ptk = capi.tokenizer(KEY, **FLAGS)
    buf, offs = gen(102, NSEQ * 4, LO, HI, AA20)
    nbases = int(offs[-1])
    n4 = NSEQ * 4
    d_b, d_o = torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda()
    for name, padlen, bf in (("c2x4_protein_bf_u8", 1024, 1), ("c2x4_protein_seqfirst_u8", 1024, 0), ("c2x4_protein_bf_u8_padlen1026", 1026, 1)):
        out = torch.empty(n4 * padlen, dtype=torch.uint8, device="cuda")
        def c2(i):
            L.bsq_tokenize(dev, st, d_b.data_ptr(), d_o.data_ptr(), n4, padlen, C.byref(ptk), bf, capi.I8, out.data_ptr())
        ms = timed(c2, 10)
        report(name, ms, nbases, nbases + 8 * (n4 + 1) + n4 * padlen)
    out32 = torch.empty(n4 * 1024, dtype=torch.int32, device="cuda")
    def c2i(i):
        L.bsq_tokenize(dev, st, d_b.data_ptr(), d_o.data_ptr(), n4, 1024, C.byref(ptk), 1, capi.I32, out32.data_ptr())
    ms = timed(c2i, 10)
    report("c2x4_protein_bf_i32", ms, nbases, nbases + 8 * (n4 + 1) + n4 * 1024 * 4)
    del out32
    oh = torch.empty((1024, NSEQ, 23), dtype=torch.uint8, device="cuda")
    nb1 = int(offs[NSEQ])
    def c2o(i):
        L.bsq_onehot(dev, st, d_b.data_ptr(), d_o.data_ptr(), None, NSEQ, 1024, C.byref(ptk), capi.I8, oh.data_ptr())
    ms = timed(c2o, 10)
    report("c2_protein_onehot_u8_C23", ms, nb1, nb1 + 8 * (NSEQ + 1) + 1024 * NSEQ * 23)
    del oh
    # decode of the batch-first tokens (device part only: lengths+scan, then characters)
    toks = out[:n4 * 1024].view(n4, 1024)
    L.bsq_tokenize(dev, st, d_b.data_ptr(), d_o.data_ptr(), n4, 1024, C.byref(ptk), 1, capi.I8, toks.data_ptr())
    d_ro = torch.empty(n4 + 1, dtype=torch.int64, device="cuda")
    d_tl = torch.empty(n4, dtype=torch.int32, device="cuda")
    total = capi.decode_lengths(dev, st, toks, 1, n4, 1024, 1024, 1, ptk, d_ro, d_tl)
    d_ch = torch.empty(total, dtype=torch.uint8, device="cuda")
    def dec(i):
        tot = C.c_int64()
        L.bsq_decode_lengths(dev, st, toks.data_ptr(), 1, n4, 1024, 1024, 1, C.byref(ptk), d_ro.data_ptr(), d_tl.data_ptr(), C.byref(tot))
        L.bsq_decode_chars(dev, st, toks.data_ptr(), 1, n4, 1024, 1024, 1, C.byref(ptk), d_ro.data_ptr(), d_tl.data_ptr(), d_ch.data_ptr())
    ms2 = timed(dec, 5)
    # the one-call form (bsq_decode_text: pass 2 enqueued behind pass 1, one host synchronisation) -- what
    # Tokenizer.decode_tokens runs; the buffer is the 3-characters-per-token guess the module makes
    d_big = torch.empty(3 * n4 * 1024, dtype=torch.uint8, device="cuda")
    def dec1(i):
        tot = C.c_int64()
        L.bsq_decode_text(dev, st, toks.data_ptr(), 1, n4, 1024, 1024, 1, C.byref(ptk), d_ro.data_ptr(), d_tl.data_ptr(), d_big.data_ptr(),
                          d_big.numel(), C.byref(tot))
        assert tot.value == total
    ms = timed(dec1, 5)
    nbytes = n4 * 1024 + total + 8 * (n4 + 1)   # SURVEY.md 8(d): B.P.s_in + sum(strlen) + 8 (B + 1): every token read once
    res["c2x4_decode_tokens_device"] = {"Gtokens/s": n4 * 1024 / ms / 1e6, "GB/s": nbytes / ms / 1e6, "frac_of_measured_hbm": nbytes / ms / 1e6 / peak,
                                        "us_per_call": ms * 1e3, "chars": int(total), "entry": "bsq_decode_text",
                                        "us_per_call_two_calls_lengths_then_chars": ms2 * 1e3}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--smi", default="value", choices=["value", "all", "off"],
                    help="nvidia-smi clock sampler: over the device-timed region only (default), the whole run, or off")
    ap.add_argument("--ref-opt", default="O3", choices=["O3", "O0"], help="reference arm: which build of oracle/_ref to time")
    ap.add_argument("--ref-threads", type=int, default=0, help="reference arm: nthreads (0 = all host cores)")
    ap.add_argument("--c5full", default="auto", choices=["auto", "on", "off"],
                    help="configs[4] at full size (8 M sequences per GPU streamed from a FlatFile): auto = only at --gpus 8")
    ap.add_argument("--sections", default="value,e2e,extra,frows,cpu,c4,c5",
                    help="comma list of measurement sections to run (profiling runs use --sections value)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the last timed step's tokens to DIR/*.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
