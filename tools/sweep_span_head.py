"""In-process A/B of K1s knobs (BSQ_TUNE=1), interleaved: per configuration the median us per launch of C2 (bench.py's
shapes and 4-set rotation, 200 launches per window) and of C2x4, P = 1026 and P = 652 (262 144 rows, 2 sets, 30 launches
per window), with every configuration's outputs checked bit for bit against the first one's.

    python tools/sweep_span_head.py [--rounds 3] [--root TREE] "" VT=1024 STAGES=3,CTAS=3 ...

Each argument is one configuration: comma-separated KEY=VALUE pairs for BSQ_SPAN_<KEY> (an empty string: the defaults).
--root: the built tree whose package is measured (default: this one), e.g. a build of another version for an A/B."""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

os.environ["BSQ_TUNE"] = "1"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if "--root" in sys.argv:
    ROOT = os.path.abspath(sys.argv[sys.argv.index("--root") + 1])
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from bioseq_b200 import capi  # noqa: E402
from bioseq_b200.synth import gen, AA20  # noqa: E402

CASES = (("c2", 65536, 4, 200, 1024, 1022), ("c2x4", 262144, 2, 30, 1024, 1022),
         ("c2x4_p1026", 262144, 2, 30, 1026, 1024), ("c5_p652", 262144, 2, 30, 652, 650))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--root", help="tree to measure (read before the imports)")
    ap.add_argument("configs", nargs="+")
    args = ap.parse_args()
    L = capi.lib()
    tok = capi.tokenizer("PROTEIN", bos=True, eos=True, padchar=True)
    st = torch.cuda.current_stream().cuda_stream
    peak = None
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak = json.load(f)["hbm_gbs"]
    except (OSError, KeyError, ValueError):
        pass
    cases = []
    for name, n, rot, reps, padlen, hi in CASES:
        sets = []
        for r in range(rot):
            buf, offs = gen(102 + r, n, 50, hi, AA20)
            sets.append((torch.from_numpy(buf).cuda(), torch.from_numpy(offs).cuda(),
                         torch.empty(n * padlen, dtype=torch.uint8, device="cuda"), int(offs[-1])))
        cases.append((name, n, rot, reps, padlen, sets))

    def apply(cfg):
        for k in [k for k in os.environ if k.startswith("BSQ_SPAN_")]:
            del os.environ[k]
        for kv in filter(None, cfg.split(",")):
            k, v = kv.split("=")
            os.environ["BSQ_SPAN_" + k] = v

    def launch(case, i):
        name, n, rot, reps, padlen, sets = case
        b, o, out, _ = sets[i % rot]
        rc = L.bsq_tokenize(0, st, b.data_ptr(), o.data_ptr(), n, padlen, C.byref(tok), 1, 0, out.data_ptr())
        assert rc == 0, capi.last_error()

    def window(case):
        reps = case[3]
        for i in range(8):
            launch(case, i)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(reps):
            launch(case, i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps * 1e3

    def outputs():
        res = []
        for case in cases:
            for i in range(case[2]):
                launch(case, i)
            torch.cuda.synchronize()
            res.append([s[2].clone() for s in case[5]])
        return res

    apply(args.configs[0])
    want = outputs()
    for cfg in args.configs[1:]:
        apply(cfg)
        got = outputs()
        same = all(torch.equal(x, y) for a, b in zip(want, got) for x, y in zip(a, b))
        print(f"outputs of [{cfg}] vs [{args.configs[0]}]: {'identical' if same else 'MISMATCH'}", flush=True)
        if not same:
            return 1
    del want
    times = {cfg: {c[0]: [] for c in cases} for cfg in args.configs}
    for r in range(args.rounds):
        for cfg in args.configs:
            apply(cfg)
            for case in cases:
                times[cfg][case[0]].append(window(case))
    for cfg in args.configs:
        parts = []
        for name, n, rot, reps, padlen, sets in cases:
            us = statistics.median(times[cfg][name])
            spread = f"{min(times[cfg][name]):.2f}-{max(times[cfg][name]):.2f}"
            frac = ""
            if peak:
                nb = sum(s[3] for s in sets) / rot
                frac = f" {(nb + 8 * (n + 1) + n * padlen) / us / 1e3 / peak:.3f}"
            parts.append(f"{name} {us:7.2f}us [{spread}]{frac}")
        print(f"[{cfg or 'defaults'}]".ljust(28), " | ".join(parts), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
