"""Every transform size the library accepts, against float64 DFTs: per transform and per bin.

fft_new_setup accepts three families of sizes, and each reaches different kernels: powers of two up to 2^14 complex
points run in one CTA (fft_kernels.cuh), longer powers of two in the multi-pass four-step (large_plan.h), and the
other 2^a 3^b 5^c sizes in mixq_kernel or mixed_kernel.  `accepted_sizes` enumerates every size the library accepts,
and the tests below sweep exactly that list:

* up to 2^24 points the reference is a float64 FFT on the host, compared slot by slot in both layouts, both SIMD
  widths and both directions; the backward direction is compared with the inverse DFT of the spectrum it is given,
  not with a round trip, which cannot see an error that the forward transform and the backward one undo together;
* beyond 2^24 points the host FFT is too slow to rerun, so the inputs have a DFT in closed form, evaluated in float64
  on the device with exact integer phases: a few impulses (every bin checked), a few nonzero bins (every sample
  checked), and uniform random data at sampled bins and samples.

Every transform of a batch is judged on its own, by rel_l2 = |got - ref| / |ref| and by the per-slot figure
max |got - ref| / rms(ref) (one slot = the real or the imaginary part of a bin or a sample).  rel_l2 must stay under
the contract 1e-6 log2 N, and both figures under TRIPWIRE: flat bounds, about twice the worst value measured on a B200
(profiles/r03_accuracy.txt, from tools/accuracy_sweep.py).  A bound that does not grow with N sees what the contract
misses at large N: a wrong twiddle, one wrong column of the four-step, a row scaled or strided wrongly.
"""
from __future__ import annotations

import math
from functools import lru_cache

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

MIXED_MAX_M = 12288   # mixed_kernels.cuh: kMixedMaxM, complex points of the mixed-radix kernels
MAX_LOG_N = 28        # large_plan.h: kMaxLargeLog, complex points of the longest transform
SINGLE_MAX_LOG_M = 14  # dispatch.h: kMaxLogM, complex points of the longest one-CTA transform
HOST_MAX_LOG_N = 24   # longer transforms are checked against closed forms on the device
GAP = 8               # floats between the rows of a batch: rows keep the 16-byte alignment of unordered spectra
SPARSE_TERMS = 6      # impulses of a sparse input, nonzero bins of a sparse spectrum
SAMPLED = 64          # bins / samples compared for random data beyond 2^24 points

# Flat bounds (rel_l2, per-slot figure) per (family, kind, layout, direction): about twice the worst value measured in
# profiles/r03_accuracy.txt (B200, 1000 W).  "large-sparse" / "large-random": the sizes beyond 2^24 points (closed forms).
TRIPWIRE = {
    ('single', 'c2c', 'ordered', 'forward'):                (3.1e-7, 2.0e-6),
    ('single', 'c2c', 'ordered', 'backward'):               (3.1e-7, 1.7e-6),
    ('single', 'c2c', 'unordered', 'forward'):              (3.1e-7, 2.0e-6),
    ('single', 'c2c', 'unordered', 'backward'):             (3.1e-7, 1.7e-6),
    ('single', 'real', 'ordered', 'forward'):               (3.3e-7, 1.9e-6),
    ('single', 'real', 'ordered', 'backward'):              (3.3e-7, 2.0e-6),
    ('single', 'real', 'unordered', 'forward'):             (3.3e-7, 1.9e-6),
    ('single', 'real', 'unordered', 'backward'):            (3.3e-7, 1.9e-6),
    ('multipass', 'c2c', 'ordered', 'forward'):             (4.3e-7, 3.4e-6),
    ('multipass', 'c2c', 'ordered', 'backward'):            (4.3e-7, 3.0e-6),
    ('multipass', 'c2c', 'unordered', 'forward'):           (4.3e-7, 3.4e-6),
    ('multipass', 'c2c', 'unordered', 'backward'):          (4.3e-7, 3.0e-6),
    ('multipass', 'real', 'ordered', 'forward'):            (4.4e-7, 3.2e-6),
    ('multipass', 'real', 'ordered', 'backward'):           (4.4e-7, 3.0e-6),
    ('multipass', 'real', 'unordered', 'forward'):          (4.4e-7, 3.2e-6),
    ('multipass', 'real', 'unordered', 'backward'):         (4.4e-7, 3.0e-6),
    ('mixq', 'c2c', 'ordered', 'forward'):                  (3.1e-7, 2.0e-6),
    ('mixq', 'c2c', 'ordered', 'backward'):                 (3.1e-7, 1.9e-6),
    ('mixq', 'c2c', 'unordered', 'forward'):                (3.1e-7, 2.0e-6),
    ('mixq', 'c2c', 'unordered', 'backward'):               (3.1e-7, 1.9e-6),
    ('mixq', 'real', 'ordered', 'forward'):                 (3.3e-7, 2.0e-6),
    ('mixq', 'real', 'ordered', 'backward'):                (3.3e-7, 1.9e-6),
    ('mixq', 'real', 'unordered', 'forward'):               (3.3e-7, 2.0e-6),
    ('mixq', 'real', 'unordered', 'backward'):              (3.3e-7, 1.9e-6),
    ('mixed', 'c2c', 'ordered', 'forward'):                 (3.1e-7, 1.8e-6),
    ('mixed', 'c2c', 'ordered', 'backward'):                (3.0e-7, 1.8e-6),
    ('mixed', 'c2c', 'unordered', 'forward'):               (3.1e-7, 1.8e-6),
    ('mixed', 'c2c', 'unordered', 'backward'):              (3.0e-7, 1.8e-6),
    ('mixed', 'real', 'ordered', 'forward'):                (3.2e-7, 2.2e-6),
    ('mixed', 'real', 'ordered', 'backward'):               (3.2e-7, 1.9e-6),
    ('mixed', 'real', 'unordered', 'forward'):              (3.2e-7, 2.2e-6),
    ('mixed', 'real', 'unordered', 'backward'):             (3.2e-7, 1.9e-6),
    ('large-sparse', 'c2c', 'ordered', 'forward'):          (4.3e-7, 3.0e-6),
    ('large-sparse', 'c2c', 'ordered', 'backward'):         (4.1e-7, 3.1e-6),
    ('large-sparse', 'c2c', 'unordered', 'forward'):        (4.3e-7, 3.0e-6),
    ('large-sparse', 'c2c', 'unordered', 'backward'):       (4.1e-7, 3.1e-6),
    ('large-sparse', 'real', 'ordered', 'forward'):         (4.1e-7, 3.2e-6),
    ('large-sparse', 'real', 'ordered', 'backward'):        (4.3e-7, 2.9e-6),
    ('large-sparse', 'real', 'unordered', 'forward'):       (4.1e-7, 3.2e-6),
    ('large-sparse', 'real', 'unordered', 'backward'):      (4.3e-7, 2.9e-6),
    ('large-random', 'c2c', 'ordered', 'forward'):          (5.0e-7, 1.8e-6),
    ('large-random', 'c2c', 'ordered', 'backward'):         (4.8e-7, 1.4e-6),
    ('large-random', 'c2c', 'unordered', 'forward'):        (5.6e-7, 1.7e-6),
    ('large-random', 'c2c', 'unordered', 'backward'):       (4.8e-7, 1.4e-6),
    ('large-random', 'real', 'ordered', 'forward'):         (4.9e-7, 1.7e-6),
    ('large-random', 'real', 'ordered', 'backward'):        (5.0e-7, 1.6e-6),
    ('large-random', 'real', 'unordered', 'forward'):       (4.8e-7, 1.8e-6),
    ('large-random', 'real', 'unordered', 'backward'):      (5.0e-7, 1.6e-6),
}


# --------------------------------------------------------------------------------------------------
# the sizes
# --------------------------------------------------------------------------------------------------
@lru_cache(maxsize=2)
def accepted_sizes(is_c: bool) -> tuple:
    """Every N fft_new_setup accepts for the kind: the powers of two from 16 (complex) / 32 (real) points to 2^28, and
    every other 2^a 3^b 5^c that is a multiple of 16 (complex) / 32 (real) with at most MIXED_MAX_M complex points."""
    unit = 16 if is_c else 32
    limit = MIXED_MAX_M if is_c else 2 * MIXED_MAX_M
    sizes = {1 << e for e in range(unit.bit_length() - 1, MAX_LOG_N + 1)}
    p3 = 1
    while unit * p3 <= limit:
        p5 = 1
        while unit * p3 * p5 <= limit:
            v = unit * p3 * p5
            while v <= limit:
                if p3 * p5 > 1:
                    sizes.add(v)
                v *= 2
            p5 *= 5
        p3 *= 3
    return tuple(sorted(sizes))


def complex_points(N: int, is_c: bool) -> int:
    return N if is_c else N // 2


def row_floats(N: int, is_c: bool) -> int:
    return 2 * N if is_c else N


def mixq_applies(M: int) -> bool:
    """mixq_kernels.cuh: mixq_applies -- M = Q 2^p with Q in {3, 5, 9, 15} and 16 <= 2^p <= 4096."""
    odd = M
    while odd % 2 == 0:
        odd //= 2
    return odd in (3, 5, 9, 15) and 16 <= M // odd <= 4096


def family(N: int, is_c: bool) -> str:
    M = complex_points(N, is_c)
    if N & (N - 1):
        return "mixq" if mixq_applies(M) else "mixed"
    return "single" if M <= 1 << SINGLE_MAX_LOG_M else "multipass"


def widths(N: int, is_c: bool) -> dict:
    """{W: use_avx} for every distinct unordered layout of the size (oracle.simd_width)."""
    from oracle import oracle as o

    out = {}
    for avx in (True, False):
        out.setdefault(o.simd_width(N, is_c, avx), avx)
    return out


def host_batch(N: int) -> int:
    """Odd batches give ragged CTAs (and, with the default 16 MiB L2 chunks, ragged chunks); two rows from 2^21 up."""
    return 11 if N <= 4096 else 5 if N <= 1 << 17 else 3 if N < 1 << 21 else 2


def row_scales(batch: int) -> np.ndarray:
    """A large and a small row next to unit rows: a per-row figure sees a row scaled or strided wrongly."""
    s = np.ones(batch)
    s[0], s[1] = 1e3, 1e-3
    return s


# --------------------------------------------------------------------------------------------------
# references
# --------------------------------------------------------------------------------------------------
def host_dft(x, N: int, is_c: bool, backward: bool) -> np.ndarray:
    """float64 transform of the rows of x in the library's ordered layout: interleaved complex, or packed real
    spectra (DC in float 0, Nyquist in float 1).  Backward is unscaled, like the library's."""
    import scipy.fft as sf

    x = np.asarray(x, np.float64)
    out = np.empty_like(x)
    if is_c:
        z = x[:, 0::2] + 1j * x[:, 1::2]
        Z = sf.ifft(z, axis=-1, norm="forward", workers=-1) if backward else sf.fft(z, axis=-1, workers=-1)
        out[:, 0::2], out[:, 1::2] = Z.real, Z.imag
    elif backward:
        X = np.empty((x.shape[0], N // 2 + 1), np.complex128)
        X[:, 0], X[:, -1] = x[:, 0], x[:, 1]
        X[:, 1:-1] = x[:, 2::2] + 1j * x[:, 3::2]
        out[:] = sf.irfft(X, n=N, axis=-1, norm="forward", workers=-1)
    else:
        X = sf.rfft(x, axis=-1, workers=-1)
        out[:, 0], out[:, 1] = X[:, 0].real, X[:, -1].real
        out[:, 2::2], out[:, 3::2] = X[:, 1:-1].real, X[:, 1:-1].imag
    return out


def unordered_slots(u, N: int, is_c: bool, W: int):
    """Ordered float slot held by unordered float slot u (int64 tensor): the closed form of oracle.np_unordered_map."""
    vec, lane = u // W, u % W
    k, is_im = vec // 2, vec % 2
    b, r = k // W, k % W
    if is_c:
        bins = r * (N // W) + b * W + lane
    else:
        Q = N // (2 * W)
        m = b * W + lane
        bins = r * Q + torch.where(r % 2 == 1, (Q - m) % Q, m)
    return 2 * bins + is_im


def dft_terms(src, val, N: int, is_c: bool, backward: bool):
    """The input of a transform as terms (index, weighted re, weighted im) of its DFT sum.  src: the float slots that
    hold val (every other slot zero), or None when val is the whole input; then the index is the term's position
    (returned as None) and the parts are views of val or float32 copies, so a 2^28-point input needs no float64 copy.
    Real backward inputs are packed spectra: DC and Nyquist count once, bins 1 .. N/2 - 1 twice (Hermitian symmetry)."""
    if src is None:
        if is_c:
            return None, val[0::2], val[1::2]
        if not backward:
            return None, val, torch.zeros_like(val)
        # terms k = 0 .. N/2: k = 0 is DC (float 0), k = N/2 Nyquist (float 1)
        a = torch.cat([val[0::2], val[1:2]])
        b = torch.cat([val[1::2], val[:1]])
        a[1:-1] *= 2
        b[1:-1] *= 2
        b[0] = b[-1] = 0
        return None, a, b
    src, val = src.to(torch.int64), val.to(torch.float64)
    if is_c:
        return src // 2, torch.where(src % 2 == 0, val, 0.0), torch.where(src % 2 == 1, val, 0.0)
    if not backward:
        return src, val, torch.zeros_like(val)
    re_in = (src % 2 == 0) | (src == 1)
    w = torch.where(src < 2, 1.0, 2.0).to(torch.float64)
    return torch.where(src == 1, N // 2, src // 2), torch.where(re_in, w * val, 0.0), torch.where(re_in, 0.0, w * val)


def dft_at(slots, src, val, N: int, is_c: bool, backward: bool, block: int = 1 << 24):
    """float64 values at the float slots `slots` of the ordered output of the transform of the input (src, val) (see
    dft_terms).  Phases come from exact integer arithmetic, (k n) mod N in int64, so they stay exact at 2^28 points.
    Tensors on any device; temporaries of about `block` elements."""
    sign = 1.0 if backward else -1.0
    i, wa, wb = dft_terms(src, val, N, is_c, backward)
    slots = slots.to(torch.int64)
    if is_c:  # complex sample / bin s // 2, real or imaginary part s % 2
        o, op = slots // 2, slots % 2
    elif not backward:  # bins, Nyquist in float 1
        o, op = torch.where(slots == 1, N // 2, slots // 2), torch.where(slots == 1, 0, slots % 2)
    else:  # real samples
        o, op = slots, torch.zeros_like(slots)
    ou, inv = torch.unique(o, return_inverse=True)
    re = torch.zeros(ou.shape[0], dtype=torch.float64, device=slots.device)
    im = torch.zeros_like(re)
    terms = wa.shape[0]
    rows = min(ou.shape[0], max(256, block // terms))
    cols = max(1, block // rows)
    for r0 in range(0, ou.shape[0], rows):
        orow = ou[r0:r0 + rows, None]
        for c0 in range(0, terms, cols):
            c1 = min(terms, c0 + cols)
            idx = torch.arange(c0, c1, device=slots.device) if i is None else i[c0:c1]
            ang = ((orow * idx[None, :]) % N).to(torch.float64) * (2.0 * math.pi / N)
            c, s = torch.cos(ang), torch.sin(ang)
            a, b = wa[c0:c1].to(torch.float64), wb[c0:c1].to(torch.float64)
            re[r0:r0 + rows] += c @ a - sign * (s @ b)
            im[r0:r0 + rows] += c @ b + sign * (s @ a)
    return torch.where(op == 0, re[inv], im[inv])


# --------------------------------------------------------------------------------------------------
# metrics
# --------------------------------------------------------------------------------------------------
def row_errors(got, ref):
    """Per row of got / ref (float64 arrays [rows, slots]): (rel_l2, max |got - ref| / rms(ref))."""
    d = np.asarray(got, np.float64) - ref
    nd, nr = np.linalg.norm(d, axis=1), np.linalg.norm(ref, axis=1)
    return nd / nr, np.abs(d).max(axis=1) / (nr / math.sqrt(ref.shape[1]))


def record(records, fam, is_c, ordered, backward, N, W, rel, per_bin):
    records.append(dict(family=fam, kind="c2c" if is_c else "real", layout="ordered" if ordered else "unordered",
                        direction="backward" if backward else "forward", N=N, W=W,
                        rel_l2=float(np.max(rel)), per_bin=float(np.max(per_bin))))


def key(r) -> tuple:
    return r["family"], r["kind"], r["layout"], r["direction"]


def check_records(records) -> None:
    bad = []
    for r in records:
        bound_rel, bound_bin = TRIPWIRE[key(r)]
        if not (r["rel_l2"] < 1e-6 * math.log2(r["N"]) and r["rel_l2"] < bound_rel and r["per_bin"] < bound_bin):
            bad.append(r)
    assert not bad, "\n".join(f"{key(r)} N={r['N']} W={r['W']}: rel_l2 {r['rel_l2']:.3g} (contract {1e-6 * math.log2(r['N']):.3g}, "
                              f"tripwire {TRIPWIRE[key(r)][0]:.3g}), per-slot {r['per_bin']:.3g} (tripwire {TRIPWIRE[key(r)][1]:.3g})"
                              for r in bad)


# --------------------------------------------------------------------------------------------------
# sizes up to 2^24: host float64 FFT
# --------------------------------------------------------------------------------------------------
def transform_rows(cf, setup, rows, backward: bool, ordered: bool) -> np.ndarray:
    """Rows [batch, nfl] through fft_transform_batched with row stride nfl + GAP; NaN in the gaps of the input and
    the output, and the output's gaps must still be NaN afterwards."""
    batch, nfl = rows.shape
    stride = nfl + GAP
    din = torch.full((batch, stride), float("nan"), device="cuda")
    din[:, :nfl] = torch.from_numpy(np.ascontiguousarray(rows, np.float32)).cuda()
    dout = torch.full((batch, stride), float("nan"), device="cuda")
    cf.fft_transform_batched(setup, din, dout, batch, stride, stride, cf.FFT_BACKWARD if backward else cf.FFT_FORWARD, ordered)
    torch.cuda.synchronize()
    out = dout.cpu().numpy()
    assert np.isnan(out[:, nfl:]).all(), "the transform wrote into the gap between rows"
    return out[:, :nfl]


def sweep_host_size(cf, N: int, is_c: bool, records: list) -> None:
    """Every layout, SIMD width and direction of one size against host_dft; for Q 2^p sizes both mixq_kernel and
    mixed_kernel (tuning hook mixq = 0).  Appends one record per (kernel, layout, width, direction)."""
    from oracle import oracle as o

    nfl = row_floats(N, is_c)
    batch = host_batch(N)
    rng = np.random.default_rng(2 * N + is_c)
    scale = row_scales(batch)[:, None]
    x = (rng.uniform(-1, 1, (batch, nfl)) * scale).astype(np.float32)
    spec = (rng.uniform(-1, 1, (batch, nfl)) * scale).astype(np.float32)
    ref_f, ref_b = host_dft(x, N, is_c, False), host_dft(spec, N, is_c, True)
    fam = family(N, is_c)
    ws = widths(N, is_c)
    W0 = next(iter(ws))  # the use_avx width; ordered data do not depend on it
    layouts = [(True, W0, ws[W0])] + [(False, W, avx) for W, avx in ws.items()]
    for hook in ((-1, 0) if fam == "mixq" else (-1,)):
        cf.set_tuning("mixq", hook)
        try:
            for ordered, W, avx in layouts:
                setup = cf.fft_new_setup(N, cf.FFT_COMPLEX if is_c else cf.FFT_REAL, avx)
                try:
                    perm = None if ordered else o.np_unordered_map(N, is_c, W)
                    for backward in (False, True):
                        src = spec if backward else x
                        got = transform_rows(cf, setup, src if ordered or not backward else src[:, perm], backward, ordered)
                        if fam in ("mixq", "mixed"):
                            assert ("mixq_kernel" in cf.last_kernel()) == (fam == "mixq" and hook != 0), (N, is_c, cf.last_kernel())
                        ref = ref_b if backward else (ref_f if ordered else ref_f[:, perm])
                        rel, per_bin = row_errors(got, ref)
                        record(records, fam if hook != 0 else "mixed", is_c, ordered, backward, N, W, rel, per_bin)
                finally:
                    cf.fft_destroy_setup(setup)
        finally:
            cf.set_tuning("mixq", -1)


# --------------------------------------------------------------------------------------------------
# sizes beyond 2^24: closed forms on the device
# --------------------------------------------------------------------------------------------------
def digits_index(d, logs, output_side: bool) -> int:
    """Complex index from the digits (d1, d2, d3) of the passes (log2 lengths logs = l1, l2, l3; l2 = 0: two passes).
    Input side n = n1 L2 L3 + n2 L3 + n3; output side k = k1 + L1 (k2 + L2 k3)."""
    l1, l2, l3 = logs
    if output_side:
        return d[0] + (d[1] << l1) + (d[2] << (l1 + l2))
    return (d[0] << (l2 + l3)) + (d[1] << l3) + d[2]


def sparse_indices(rng, logs, count: int) -> list:
    """Distinct input-side complex indices whose digits are all nonzero: every pass sees a nontrivial twiddle."""
    out = set()
    while len(out) < count:
        out.add(digits_index([int(rng.integers(1, 1 << l)) if l else 0 for l in logs], logs, False))
    return sorted(out)


def covering_indices(rng, logs, M: int, count: int) -> list:
    """Output-side complex indices: every bit of every digit set in one of them, each digit at 0 and at its largest
    value, the first, second, middle and last index, the rest uniform.  (A few dozen indices cannot take every value of
    a 512-value digit; the sparse inputs check every bin.)"""
    out = {0, 1, M // 2, M - 1}
    for j, l in enumerate(logs):
        if l == 0:
            continue
        for v in [1 << b for b in range(l)] + [(1 << l) - 1, 0]:
            d = [int(rng.integers(0, 1 << ll)) if ll else 0 for ll in logs]
            d[j] = v
            out.add(digits_index(d, logs, True))
    while len(out) < count:
        out.add(int(rng.integers(0, M)))
    return sorted(out)


def sparse_input(rng, logs, N: int, is_c: bool, backward: bool, device):
    """(float slots, float64 values) of a sparse input: SPARSE_TERMS impulses with random complex (complex plans) or real
    amplitudes, or, for the backward direction, as many nonzero bins (real plans: bins 1 .. N/2 - 1 plus DC and
    Nyquist).  Positions from sparse_indices; values are float32 numbers, so the float32 input holds them exactly."""
    idx = sparse_indices(rng, logs, SPARSE_TERMS)
    mag = rng.uniform(0.5, 1.0, len(idx))
    ph = rng.uniform(0, 2 * np.pi, len(idx))
    if is_c or backward:  # complex amplitudes: both floats of the sample / bin
        src = [2 * m + p for m in idx for p in (0, 1)]
        val = [v for a, f in zip(mag, ph) for v in (a * np.cos(f), a * np.sin(f))]
        if not is_c:
            src, val = [0, 1] + src, [0.7, -0.4] + val
    else:  # real impulses: the even or the odd float of complex index m
        src = [2 * m + int(rng.integers(0, 2)) for m in idx]
        val = list(mag * np.sign(ph - np.pi))
    return (torch.tensor(src, dtype=torch.int64, device=device),
            torch.tensor(val, dtype=torch.float32, device=device).double())


def gather_unordered(ordered, N: int, is_c: bool, W: int, block: int = 1 << 24):
    """The unordered layout of an ordered spectrum: slot u holds ordered slot map[u]."""
    out = torch.empty_like(ordered)
    for u0 in range(0, ordered.shape[0], block):
        u = torch.arange(u0, min(ordered.shape[0], u0 + block), device=ordered.device)
        out[u0:u0 + u.shape[0]] = ordered[unordered_slots(u, N, is_c, W)]
    return out


def full_errors(got, ref_at, block: int = 1 << 22):
    """(rel_l2, per-slot figure) of the device vector got against ref_at(slots), every slot, in blocks."""
    sd = sr = md = 0.0
    for u0 in range(0, got.shape[0], block):
        u = torch.arange(u0, min(got.shape[0], u0 + block), device=got.device)
        ref = ref_at(u)
        d = got[u0:u0 + u.shape[0]].double() - ref
        sd += float((d * d).sum())
        sr += float((ref * ref).sum())
        md = max(md, float(d.abs().max()))
    return math.sqrt(sd / sr), md / math.sqrt(sr / got.shape[0])


def sampled_errors(got, ref):
    d = got.double() - ref
    nr = float(ref.norm())
    return float(d.norm()) / nr, float(d.abs().max()) / (nr / math.sqrt(ref.shape[0]))


def sweep_closed_form_size(cf, N: int, is_c: bool, records: list) -> None:
    """One transform per call, ordered and every unordered width, both directions: a sparse input (every bin) and a
    sparse spectrum (every sample) against their closed forms, uniform random data at covering_indices."""
    nfl = row_floats(N, is_c)
    M = complex_points(N, is_c)
    dev = torch.device("cuda")
    rng = np.random.default_rng(N + is_c)
    gen = torch.Generator(device="cuda").manual_seed(N + is_c)
    ws = widths(N, is_c)
    W0 = next(iter(ws))  # the use_avx width; ordered data do not depend on it
    setups = {W: cf.fft_new_setup(N, cf.FFT_COMPLEX if is_c else cf.FFT_REAL, avx) for W, avx in ws.items()}
    try:
        logs = cf.fft_large_factors(setups[W0])
        assert sum(logs) == M.bit_length() - 1, logs

        def each_layout(inp, backward):
            """(ordered, W, output) for the ordered layout and every unordered width; inp is the ordered input."""
            for ordered, W in [(True, W0)] + [(False, W) for W in ws]:
                x = inp if ordered or not backward else gather_unordered(inp, N, is_c, W)
                out = torch.full_like(inp, float("nan"))
                cf.fft_transform_batched(setups[W], x, out, 1, nfl, nfl, cf.FFT_BACKWARD if backward else cf.FFT_FORWARD, ordered)
                torch.cuda.synchronize()
                del x
                yield ordered, W, out
                del out

        def ordered_slots(u, ordered, W, backward):
            """Ordered output slots held by the output slots u (a time-domain output has one layout)."""
            return u if ordered or backward else unordered_slots(u, N, is_c, W)

        for backward in (False, True):
            src, val = sparse_input(rng, logs, N, is_c, backward, dev)
            buf = torch.zeros(nfl, device=dev)
            buf[src] = val.float()
            for ordered, W, out in each_layout(buf, backward):
                rel, per_bin = full_errors(out, lambda u: dft_at(ordered_slots(u, ordered, W, backward), src, val, N, is_c, backward))
                record(records, "large-sparse", is_c, ordered, backward, N, W, [rel], [per_bin])
            del buf

        picks = covering_indices(rng, logs, M, SAMPLED)
        sampled = torch.tensor([2 * k + p for k in picks for p in (0, 1)], dtype=torch.int64, device=dev)
        for backward in (False, True):
            buf = torch.rand(nfl, device=dev, generator=gen) * 2 - 1
            refs = {}
            for ordered, W, out in each_layout(buf, backward):
                # unordered spectra: uniform unordered slots and the first and last one, each width its own
                key_ = None if ordered or backward else W
                if key_ not in refs:
                    u = sampled if key_ is None else torch.tensor(sorted({0, 1, nfl - 1} | {int(v) for v in rng.integers(0, nfl, 2 * SAMPLED)}), device=dev)
                    refs[key_] = u, dft_at(ordered_slots(u, ordered, W, backward), None, buf, N, is_c, backward)
                u, ref = refs[key_]
                rel, per_bin = sampled_errors(out[u], ref)
                record(records, "large-random", is_c, ordered, backward, N, W, [rel], [per_bin])
            del buf
    finally:
        for s in setups.values():
            cf.fft_destroy_setup(s)


def closed_form_bytes(N: int, is_c: bool) -> int:
    """Device memory sweep_closed_form_size needs: input, output, gathered input, the library's scratch, temporaries."""
    return 6 * row_floats(N, is_c) * 4 + (2 << 30)


# --------------------------------------------------------------------------------------------------
# tests
# --------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cf():
    import chowdsp_fft_b200 as m

    assert m.device_available(), "GPU tests need a CUDA device; there is no CPU fallback"
    return m


HOST_CASES = [(N, is_c) for is_c in (True, False) for N in accepted_sizes(is_c) if N <= 1 << HOST_MAX_LOG_N]
DEVICE_CASES = [(N, is_c) for is_c in (True, False) for N in accepted_sizes(is_c) if N > 1 << HOST_MAX_LOG_N]


def case_id(N, is_c):
    return f"{'c2c' if is_c else 'real'}-{N}"


def test_size_acceptance_matches_the_rule(cf, monkeypatch):
    """fft_new_setup accepts exactly accepted_sizes among every multiple of 16 up to 2^15, every power of two from 2^4
    to 2^29 and a few sizes that are not multiples of 16; both kinds, both use_avx values.  A rejection raises
    FFTError and leaves the context healthy; an acceptance reports the reference's SIMD width."""
    from oracle import oracle as o

    monkeypatch.setenv("CHOWDSP_FFT_B200_QUIET", "1")
    candidates = sorted(set(range(0, (1 << 15) + 1, 16)) | {1 << e for e in range(4, 30)} | {-16, 1, 8, 24, 40, 100, 120, 1000, 25000})
    for is_c in (True, False):
        want = set(accepted_sizes(is_c))
        assert want <= set(candidates)
        for avx in (True, False):
            got = set()
            for N in candidates:
                try:
                    s = cf.fft_new_setup(N, cf.FFT_COMPLEX if is_c else cf.FFT_REAL, avx)
                except cf.FFTError:
                    continue
                got.add(N)
                assert cf.fft_simd_width_bytes(s) == 4 * o.simd_width(N, is_c, avx), (N, is_c, avx)
                cf.fft_destroy_setup(s)
            assert got == want, (is_c, avx, sorted(got ^ want))
    x = torch.ones(64, device="cuda")
    s = cf.fft_new_setup(32, cf.FFT_COMPLEX)
    cf.fft_transform_batched(s, x, x, 1, 64, 64, cf.FFT_FORWARD, True)
    torch.cuda.synchronize()
    assert float(x[0]) == 32.0
    cf.fft_destroy_setup(s)


@pytest.mark.parametrize("N,is_c", HOST_CASES, ids=[case_id(*c) for c in HOST_CASES])
def test_sizes_against_host_dft(cf, N, is_c):
    records = []
    sweep_host_size(cf, N, is_c, records)
    check_records(records)


@pytest.mark.parametrize("N,is_c", DEVICE_CASES, ids=[case_id(*c) for c in DEVICE_CASES])
def test_large_sizes_against_closed_forms(cf, N, is_c):
    free, _ = torch.cuda.mem_get_info()
    if free < closed_form_bytes(N, is_c):
        pytest.skip(f"needs {closed_form_bytes(N, is_c) >> 30} GiB of free device memory")
    records = []
    sweep_closed_form_size(cf, N, is_c, records)
    check_records(records)
