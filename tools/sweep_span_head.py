"""K1s timing of one build, in one process: the median us per launch of C2 (bench.py's shapes and 4-set rotation, 200
launches per window) and of C2x4, P = 1026 and P = 652 (262 144 rows, 2 sets, 30 launches per window).

    python tools/sweep_span_head.py [--rounds 3] [--root TREE]

--root: the built tree whose package is measured (default: this one), e.g. a build of another version for an A/B
(tools/span_handover_ab.sh alternates two builds this way)."""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

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

    times = {c[0]: [] for c in cases}
    for r in range(args.rounds):
        for case in cases:
            times[case[0]].append(window(case))
    parts = []
    for name, n, rot, reps, padlen, sets in cases:
        us = statistics.median(times[name])
        spread = f"{min(times[name]):.2f}-{max(times[name]):.2f}"
        frac = ""
        if peak:
            nb = sum(s[3] for s in sets) / rot
            frac = f" {(nb + 8 * (n + 1) + n * padlen) / us / 1e3 / peak:.3f}"
        parts.append(f"{name} {us:7.2f}us [{spread}]{frac}")
    print(" | ".join(parts), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
