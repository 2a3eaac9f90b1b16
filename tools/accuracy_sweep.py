"""Accuracy of every transform size the library accepts, against float64 DFTs (the checks of tests/test_gpu_sizes.py).

Prints the worst per-transform rel_l2 and per-slot figure max |got - ref| / rms(ref) per (family, kind, layout,
direction), then the worst of each size, so that a size far above its neighbours stands out.  This is the table of
profiles/r03_accuracy.txt, from which the TRIPWIRE bounds of tests/test_gpu_sizes.py are set.  It reports errors only,
no timings.

    python tools/accuracy_sweep.py [--max-log 28]
"""
import argparse
import math
import os
import subprocess
import sys
import traceback

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--max-log", type=int, default=28, help="largest size swept, log2 N")
    args = ap.parse_args()

    import torch

    import chowdsp_fft_b200 as cf
    from tests import test_gpu_sizes as t

    assert cf.device_available(), "needs a CUDA device"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    print(f"# device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit: {smi.stdout.strip() or 'n/a'}")
    records, failures, counts = [], [], {}
    for is_c in (True, False):
        for N in t.accepted_sizes(is_c):
            if N > 1 << args.max_log:
                continue
            fam = "mixed-radix" if N & (N - 1) else "power of two"
            counts[(fam, is_c)] = counts.get((fam, is_c), 0) + 1
            try:
                if N <= 1 << t.HOST_MAX_LOG_N:
                    t.sweep_host_size(cf, N, is_c, records)
                elif torch.cuda.mem_get_info()[0] >= t.closed_form_bytes(N, is_c):
                    t.sweep_closed_form_size(cf, N, is_c, records)
                else:
                    failures.append(f"{t.case_id(N, is_c)}: skipped, not enough free device memory")
            except Exception:
                failures.append(f"{t.case_id(N, is_c)}: {traceback.format_exc(limit=3)}")
    print("# sizes swept: " + ", ".join(f"{'c2c' if c else 'real'} {f}: {n}" for (f, c), n in sorted(counts.items())))
    if args.max_log == t.MAX_LOG_N:
        assert counts == {("mixed-radix", True): 69, ("mixed-radix", False): 69, ("power of two", True): 25, ("power of two", False): 24}, counts

    print("\n# worst per (family, kind, layout, direction); rel_l2 per transform, per-slot = max |got - ref| / rms(ref); "
          "'of contract' = rel_l2 / (1e-6 log2 N) at its worst")
    print(f"{'family':13s} {'kind':4s} {'layout':9s} {'direction':9s} {'checks':>6s} {'rel_l2':>9s} {'at N':>9s} {'per-slot':>9s} {'at N':>9s} "
          f"{'of contract':>11s}  tripwire")
    worst = {}
    for r in records:
        w = worst.setdefault(t.key(r), {"n": 0, "rel": (0.0, 0), "bin": (0.0, 0), "ratio": 0.0})
        w["n"] += 1
        w["rel"] = max(w["rel"], (r["rel_l2"], r["N"]))
        w["bin"] = max(w["bin"], (r["per_bin"], r["N"]))
        w["ratio"] = max(w["ratio"], r["rel_l2"] / (1e-6 * math.log2(r["N"])))
    for k in sorted(worst):
        w = worst[k]
        trip = t.TRIPWIRE.get(k)
        print(f"{k[0]:13s} {k[1]:4s} {k[2]:9s} {k[3]:9s} {w['n']:6d} {w['rel'][0]:9.3g} {w['rel'][1]:9d} {w['bin'][0]:9.3g} {w['bin'][1]:9d} "
              f"{w['ratio']:11.3f}  {'%.2g / %.2g' % trip if trip else '-'}")

    print("\n# worst per size over its layouts, widths, directions and kernels")
    per_size = {}
    for r in records:
        s = per_size.setdefault((r["kind"], r["N"]), [0.0, 0.0])
        s[0], s[1] = max(s[0], r["rel_l2"]), max(s[1], r["per_bin"])
    for (kind, N), (rel, pb) in sorted(per_size.items()):
        print(f"{kind:4s} {N:10d} {t.family(N, kind == 'c2c'):10s} rel_l2 {rel:9.3g} per-slot {pb:9.3g}")

    for f in failures:
        print("FAILED", f)
    return 1 if failures else 0


if __name__ == "__main__":
    sys.exit(main())
