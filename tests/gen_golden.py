"""Generates tests/golden/reference_vectors*.npz by RUNNING THE UNMODIFIED REFERENCE
(oracle/_ref/libchowdsp_fft_ref.so, built by oracle/Makefile from /root/reference).

The reference ships no golden vectors (its tests compare against pffft, which is not vendored,
SURVEY.md §8c), so these fixtures are the reference's own outputs on the reference tests' inputs
(test/test.cpp:23-27,82-85,142-148,193-197) and on seeded uniform noise.  Run from the repo root in
the build container:   python tests/gen_golden.py
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from oracle import oracle as o  # noqa: E402

CASES = [(N, is_c, avx) for N in (32, 64, 128, 256, 1024, 4096)
         for is_c in (False, True) for avx in (False, True)]


def main():
    ref = o.load_ref()
    assert ref is not None, "build oracle/_ref first (make -C oracle)"
    out = {}
    rng = np.random.default_rng(20240607)
    for N, is_c, avx in CASES:
        W = o.simd_width(N, is_c, avx)
        if W == 0 or (avx and W != 8):
            continue
        nfl = 2 * N if is_c else N
        tag = f"{'c' if is_c else 'r'}{N}w{W}"
        x = np.stack([o.ref_signal(N, is_c, 100.0), o.ref_signal(N, is_c, 200.0),
                      rng.uniform(-1, 1, nfl).astype(np.float32)])
        fo, _ = ref.transform(x, N, is_c, False, True, avx)
        fu, _ = ref.transform(x, N, is_c, False, False, avx)
        bo, _ = ref.transform(fo, N, is_c, True, True, avx)
        bu, _ = ref.transform(fu, N, is_c, True, False, avx)
        acc = rng.uniform(-1, 1, nfl).astype(np.float32)
        conv = ref.convolve(fu[0], fu[1], acc, N, is_c, 0.5 / N, avx)
        out[tag + "_x"] = x
        out[tag + "_fwd_ordered"] = fo
        out[tag + "_fwd_unordered"] = fu
        out[tag + "_bwd_ordered"] = bo
        out[tag + "_bwd_unordered"] = bu
        out[tag + "_conv_acc_in"] = acc
        out[tag + "_conv_out"] = conv
    # one file per width for the largest size keeps every file under 1 MB
    groups = {}
    for key, arr in out.items():
        N, W = key.split("_")[0][1:].split("w")
        name = "reference_vectors.npz" if int(N) < 4096 else f"reference_vectors_{N}w{W}.npz"
        groups.setdefault(name, {})[key] = arr
    for name, arrays in groups.items():
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name)
        np.savez_compressed(path, **arrays)
        print(path, os.path.getsize(path), "bytes,", len(arrays), "arrays")


if __name__ == "__main__":
    main()
