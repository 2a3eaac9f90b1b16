"""Every kernel route of the transform dispatcher, against float64 and against single calls.

The kernel that runs a batch depends on more than the size: `enqueue_transform` (csrc/capi.cu) picks pipe_kernel,
fft_kernel, wpipe_kernel, fft_small_kernel, mixq_kernel, mixed_kernel or the multi-pass tile kernels from the batch
geometry (two-level batches, row strides, base alignment, batch size, overlapping frames), and host buffers are staged
in chunks that are routed one by one.  `expected_kernel` restates the dispatcher's rule for the default tuning; every
case below asserts that the kernel the library reports is the predicted one, and the last test that the sweep reached
every route.

Every row of every case is checked twice:
* against a float64 DFT (host_dft of tests/test_gpu_sizes.py), per row, under the contract 1e-6 log2 N and the
  TRIPWIRE bounds of its size family; rows are scaled 1e3 and 1e-3 next to unit rows, and every float outside the rows
  holds NaN before the call and must still hold it after;
* bit for bit against fft_transform / fft_transform_unordered called alone on that row at the same address, which is
  what include/chowdsp_fft_b200.h promises for every batched call (in-place batches: against the out-of-place result).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import pytest

from tests.test_gpu_sizes import TRIPWIRE, family, host_dft, mixq_applies, row_errors, row_scales, unordered_slots, widths

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

KINDS = ("C2C_FWD", "C2C_BWD", "R2C", "C2R")
CHUNK_BYTES = 32 << 20       # capi.cu: kChunkBytes, host staging granularity
SAMPLE = 12                  # rows of a long batch that get a single-call comparison besides the boundary rows

# the routes of the table in expected_kernel's docstring; test_every_route_was_reached checks that each was seen
ROUTES = ("pipe_kernel", "fft_kernel<13/14,32>", "wpipe_kernel", "fft_small_kernel", "fft_kernel", "mixq_kernel", "mixed_kernel",
          "tile_fft_kernel", "host staged", "host zero-copy")
REACHED: set = set()
SWEEPS_RUN: set = set()


# --------------------------------------------------------------------------------------------------
# the dispatcher's rule (default tuning)
# --------------------------------------------------------------------------------------------------
def radix_for(logM: int, is_c: bool) -> int:
    """capi.cu: radix_for with kRadix32Default -- 32 points per thread for complex 2^13 / 2^14, real 2^10 / 2^13 / 2^14."""
    return 32 if logM in ((13, 14) if is_c else (10, 13, 14)) else 16


def pipe_enabled(logM: int, kind: int, logW: int) -> bool:
    """capi.cu: pipe_enabled with kPipeDefault -- 2^13 / 2^14, ordered and 8-lane layouts, except ordered R2C / C2R at 2^13."""
    return logM in (13, 14) and logW in (0, 3) and not (logW == 0 and logM == 13 and kind in (2, 3))


def per_cta(logM: int, radix: int) -> int:
    """fft_kernels.cuh: Launch::PER_CTA -- transforms per CTA of fft_kernel (256 threads at least)."""
    T = (1 << logM) // radix
    return max(T, 256) // T


def pipe_ctas_per_sm(logM: int) -> int:
    """pipe_kernels.cuh: PipeGeo::CTAS_PER_SM -- two resident CTAs at 2^13, one at 2^14."""
    return 2 if logM == 13 else 1


@dataclass(frozen=True)
class Geometry:
    outer: int
    inner: int
    in_outer: int
    in_inner: int
    out_outer: int
    out_inner: int
    in_off: int = 0   # floats from a 16-byte boundary to the first input / output row
    out_off: int = 0
    inplace: bool = False

    @property
    def batch(self) -> int:
        return self.outer * self.inner

    def rows(self, side: str):
        """Float offset of every transform's row from the buffer base, in batch order."""
        o, i = np.divmod(np.arange(self.batch), self.inner)
        if side == "in":
            return self.in_off + o * self.in_outer + i * self.in_inner
        return self.out_off + o * self.out_outer + i * self.out_inner


def plain(batch: int, in_stride: int, out_stride: int, in_off: int = 0, out_off: int = 0, inplace: bool = False) -> Geometry:
    return Geometry(1, batch, 0, in_stride, 0, out_stride, in_off, out_off, inplace)


def expected_kernel(N: int, is_c: bool, backward: bool, ordered: bool, W: int, g: Geometry) -> tuple:
    """(route, kernel name prefix that last_kernel() reports) of a transform call under the default tuning:

    | route                | chosen when                                                                                    |
    | pipe_kernel          | complex 2^13 / 2^14 points, ordered or 8-lane, one-level batch, 16-byte aligned input rows     |
    | fft_kernel<13/14,32> | the same sizes otherwise (two-level batch, stride 2 mod 4, base 8 bytes off, 4-lane layout)    |
    | wpipe_kernel         | forward 2^10 complex points: overlapping frames, or unordered R2C 2048 with >= 4096 rows       |
    | fft_small_kernel     | dense one-level batches of 16 / 32 complex points, aligned                                     |
    | fft_kernel           | every other single-kernel size and geometry                                                    |
    | mixq / mixed / tile  | Q 2^p, other 2^a 3^b 5^c sizes, more than 2^14 points: one launch per outer index             |
    """
    fam = family(N, is_c)
    if fam == "mixq":
        return "mixq_kernel", "cfb::mixq_kernel<"
    if fam == "mixed":
        return "mixed_kernel", "cfb::mixed_kernel "
    if fam == "multipass":
        return "tile_fft_kernel", "cfb::tile_fft_kernel<"
    M = N if is_c else N // 2
    logM = M.bit_length() - 1
    row = 2 * M
    kind = (1 if backward else 0) if is_c else (3 if backward else 2)
    logW = 0 if ordered else (3 if W == 8 else 2)
    bstride = g.in_inner if g.outer == 1 else g.in_outer
    if pipe_enabled(logM, kind, logW) and (g.outer == 1 or g.inner == 1) and g.in_off % 4 == 0 and bstride % 4 == 0:
        return "pipe_kernel", f"cfb::pipe_kernel<{logM},{KINDS[kind]},{logW}>"
    frame_stride = g.in_inner if g.inner > 1 else g.in_outer
    frames = g.batch > 1 and 0 < frame_stride < row
    unord_real_2048 = not ordered and not is_c and logM == 10 and g.batch >= 4096
    if (logM == 10 and frames or unord_real_2048) and not backward and g.in_off % 4 == 0 and (g.inner == 1 or g.in_inner % 4 == 0) \
            and (g.outer == 1 or g.in_outer % 4 == 0):
        return "wpipe_kernel", f"cfb::wpipe_kernel<10,32,{KINDS[kind]},{logW}>"
    radix = radix_for(logM, is_c)
    al = 2 if ordered else 4
    if logM <= 5 and g.outer == 1 and g.in_inner == row and g.out_inner == row and g.in_off % al == 0 and g.out_off % al == 0:
        return "fft_small_kernel", f"cfb::fft_small_kernel<{logM},{radix},{KINDS[kind]},{logW}>"
    return ("fft_kernel<13/14,32>" if logM >= 13 else "fft_kernel"), f"cfb::fft_kernel<{logM},{radix},{KINDS[kind]},{logW}>"


# --------------------------------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cf():
    import chowdsp_fft_b200 as m

    assert m.device_available(), "GPU tests need a CUDA device; there is no CPU fallback"
    return m


def layouts(N: int, is_c: bool):
    """(ordered, W, use_avx) for the ordered layout and every unordered width of the size."""
    ws = widths(N, is_c)
    W0 = next(iter(ws))
    return [(True, W0, ws[W0])] + [(False, W, avx) for W, avx in ws.items()]


def unordered_perm(N: int, is_c: bool, W: int) -> np.ndarray:
    nfl = 2 * N if is_c else N
    return unordered_slots(torch.arange(nfl), N, is_c, W).numpy()


def data(N: int, is_c: bool, batch: int, seed: int):
    """(time-domain rows, ordered spectra): uniform in [-1, 1), scaled per row by row_scales."""
    nfl = 2 * N if is_c else N
    rng = np.random.default_rng(seed)
    scale = row_scales(max(batch, 2))[:batch, None]
    return ((rng.uniform(-1, 1, (batch, nfl)) * scale).astype(np.float32),
            (rng.uniform(-1, 1, (batch, nfl)) * scale).astype(np.float32))


def span(offs, nfl: int) -> int:
    return int(offs.max()) + nfl + 8


def sampled_rows(g: Geometry, sms: int) -> list:
    """Rows that get a single-call comparison: all of a short batch; of a long one the first and last, both sides of every
    persistent round of pipe_kernel, of every CTA of fft_kernel and of the 4096-row line, and a few random rows."""
    B = g.batch
    if B <= 64:
        return list(range(B))
    picks = {0, 1, B - 2, B - 1}
    for edge in [sms * k for k in (1, 2, 3, 4)] + [2 * sms * k for k in (1, 2, 3)] + [4095, 4096] + [8 * k for k in (1, 2)]:
        picks |= {e for e in (edge - 1, edge) if 0 <= e < B}
    picks |= set(np.random.default_rng(B).integers(0, B, SAMPLE).tolist())
    return sorted(picks)


def check_float64(got, ref, N: int, is_c: bool, ordered: bool, backward: bool, what: str) -> None:
    """Per row: rel_l2 under the contract 1e-6 log2 N and both figures under TRIPWIRE for the size's family."""
    key = (family(N, is_c), "c2c" if is_c else "real", "ordered" if ordered else "unordered", "backward" if backward else "forward")
    bound_rel, bound_bin = TRIPWIRE[key]
    rel, per_bin = row_errors(got, ref)
    bad = np.nonzero(~((rel < 1e-6 * math.log2(N)) & (rel < bound_rel) & (per_bin < bound_bin)))[0]
    assert bad.size == 0, f"{what}: rows {bad[:8].tolist()} rel_l2 {rel[bad[:8]]} per-slot {per_bin[bad[:8]]} (bounds {bound_rel}, {bound_bin})"


class Case:
    """One size / kind / layout / direction: the setup, the inputs and the float64 references of `batch` rows."""

    def __init__(self, cf, N: int, is_c: bool, ordered: bool, W: int, avx: bool, backward: bool, batch: int):
        self.cf, self.N, self.is_c, self.ordered, self.W, self.backward = cf, N, is_c, ordered, W, backward
        self.nfl = 2 * N if is_c else N
        self.setup = cf.fft_new_setup(N, cf.FFT_COMPLEX if is_c else cf.FFT_REAL, avx)
        x, spec = data(N, is_c, batch, 7 * N + 2 * is_c + backward)
        perm = None if ordered else unordered_perm(N, is_c, W)
        if backward:
            self.inp = spec if ordered else np.ascontiguousarray(spec[:, perm])
            self.ref = lambda rows: host_dft(spec[rows], N, is_c, True)
        else:
            self.inp = x
            self.ref = lambda rows: host_dft(x[rows], N, is_c, False) if ordered else host_dft(x[rows], N, is_c, False)[:, perm]
        self.direction = cf.FFT_BACKWARD if backward else cf.FFT_FORWARD

    def close(self):
        self.cf.fft_destroy_setup(self.setup)

    def single(self, in_ptr: int, out_ptr: int) -> None:
        f = self.cf.fft_transform if self.ordered else self.cf.fft_transform_unordered
        f(self.setup, in_ptr, out_ptr, 0, self.direction)

    def call(self, g: Geometry, in_ptr: int, out_ptr: int) -> None:
        cf = self.cf
        if g.outer == 1:
            cf.fft_transform_batched(self.setup, in_ptr, out_ptr, g.inner, g.in_inner, g.out_inner, self.direction, self.ordered)
        else:
            cf.fft_transform_strided(self.setup, in_ptr, out_ptr, g.outer, g.inner, g.in_outer, g.in_inner, g.out_outer, g.out_inner,
                                     self.direction, self.ordered)


def run_device(case: Case, g: Geometry, sms: int, inputs=None):
    """Runs the case on device buffers filled with NaN outside the rows; checks the reported kernel, the NaN floats,
    float64 per row and the single-call bits per sampled row.  Returns the output rows."""
    cf, nfl = case.cf, case.nfl
    inp = case.inp if inputs is None else inputs
    ioff, ooff = g.rows("in"), g.rows("out")
    if g.inplace:
        assert (ioff == ooff).all()
    buf_in = torch.full((span(ioff, nfl),), float("nan"), device="cuda")
    for r, o in enumerate(ioff):
        buf_in[o:o + nfl] = torch.from_numpy(inp[r]).cuda()  # overlapping frames: later rows rewrite the same samples
    buf_out = buf_in if g.inplace else torch.full((span(ooff, nfl),), float("nan"), device="cuda")
    frames = g.batch > 1 and not g.inplace and len(set(ioff.tolist())) == g.batch and np.diff(np.sort(ioff)).min() < nfl
    torch.cuda.synchronize()
    src = buf_in.clone() if not g.inplace else None
    case.call(g, buf_in.data_ptr() + 4 * g.in_off, buf_out.data_ptr() + 4 * g.out_off)
    torch.cuda.synchronize()
    route, want = expected_kernel(case.N, case.is_c, case.backward, case.ordered, case.W, g)
    got_kernel = cf.last_kernel()
    assert got_kernel.startswith(want), (case.N, case.is_c, case.ordered, case.W, case.backward, g, got_kernel, want)
    REACHED.add(route)
    out = buf_out.cpu().numpy()
    mask = np.ones(out.shape[0], bool)
    for o in ooff:
        mask[o:o + nfl] = False
    assert np.isnan(out[mask]).all(), f"{g}: the transform wrote outside its rows"
    rows = np.stack([out[o:o + nfl] for o in ooff])
    if frames:  # overlapping forward frames: the reference transforms the rows as they overlap in the buffer
        assert not case.backward
        held = buf_in.cpu().numpy()
        ref = host_dft(np.stack([held[o:o + nfl] for o in ioff]), case.N, case.is_c, False)
        ref = ref if case.ordered else ref[:, unordered_perm(case.N, case.is_c, case.W)]
    else:
        ref = case.ref(np.arange(g.batch))
    check_float64(rows, ref, case.N, case.is_c, case.ordered, case.backward, f"N={case.N} {g}")
    if src is not None:
        # bit contract: each sampled row alone at the same input address, into a buffer with the row's output alignment
        single = torch.full((nfl + 8,), float("nan"), device="cuda")
        mism = []
        for r in sampled_rows(g, sms):
            s_off = int(ooff[r]) % 4
            case.single(src.data_ptr() + 4 * int(ioff[r]), single.data_ptr() + 4 * s_off)
            one = single[s_off:s_off + nfl].cpu().numpy()
            if not np.array_equal(one.view(np.uint32), rows[r].view(np.uint32)):
                mism.append((r, int((one != rows[r]).sum())))
        assert not mism, f"N={case.N} {'c2c' if case.is_c else 'real'} ordered={case.ordered} W={case.W} backward={case.backward} {g} " \
                         f"via {got_kernel}: (row, differing floats) {mism[:8]} of {g.batch} rows differ from single calls"
    return rows


# --------------------------------------------------------------------------------------------------
# the sweep
# --------------------------------------------------------------------------------------------------
def geometries(N: int, is_c: bool, ordered: bool, backward: bool, sms: int) -> list:
    """The geometries of one size, kind, layout and direction that the alignment rule admits: unordered spectra need
    16-byte aligned rows, ordered data 8-byte aligned ones."""
    nfl = 2 * N if is_c else N
    M = N if is_c else N // 2
    logM = M.bit_length() - 1
    in_unord, out_unord = not ordered and backward, not ordered and not backward
    odd_in = 4 if in_unord else 2    # stride 2 mod 4 / base 8 bytes off, where the side may be
    odd_out = 4 if out_unord else 2
    off_in = 0 if in_unord else 2
    off_out = 0 if out_unord else 2
    gs = [plain(5, nfl, nfl), plain(5, nfl + 8, nfl + 12), plain(5, nfl + odd_in, nfl + odd_out),
          plain(3, nfl + 4, nfl + 4, off_in, off_out), plain(4, nfl, nfl, inplace=True), plain(1, nfl, nfl),
          Geometry(3, 5, 5 * (nfl + 4) + 12, nfl + 4, 5 * (nfl + 8) + 4, nfl + 8)]
    if family(N, is_c) != "single":
        return gs
    radix = radix_for(logM, is_c)
    pc = per_cta(logM, radix)
    gs += [plain(b, nfl, nfl) for b in (pc - 1, pc + 1) if b > 1 and b != 5]
    if logM in (13, 14):
        gs.append(plain(2 * sms * pipe_ctas_per_sm(logM) + 7, nfl, nfl))
    if logM <= 5:
        gs.append(plain(1000, nfl, nfl))  # dense batch of tiny transforms: fft_small_kernel across many CTAs
    if logM in (9, 10) and not is_c and not backward:
        gs.append(Geometry(2, 7, 6 * nfl + 4, nfl // 4, 7 * nfl, nfl))  # overlapping frames, hop N/4
    return gs


SINGLE = [(1 << e, True) for e in range(4, 15)] + [(1 << e, False) for e in range(5, 16)]
BEYOND = [(768, True), (400, True), (1536, False), (1 << 15, True), (1 << 17, True), (1 << 16, False)]
SWEEP = SINGLE + BEYOND


def case_id(N, is_c):
    return f"{'c2c' if is_c else 'real'}-{N}"


@pytest.mark.parametrize("N,is_c", SWEEP, ids=[case_id(*c) for c in SWEEP])
def test_routes_against_float64_and_single_calls(cf, N, is_c):
    """Every layout and direction of the size through every geometry of `geometries`."""
    assert mixq_applies(768) and not mixq_applies(400)  # the two non-power-of-two sizes reach both mixed-radix kernels
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    for ordered, W, avx in layouts(N, is_c):
        for backward in (False, True):
            gs = geometries(N, is_c, ordered, backward, sms)
            case = Case(cf, N, is_c, ordered, W, avx, backward, max(g.batch for g in gs))
            try:
                for g in gs:
                    rows = run_device(case, g, sms)
                    if g.inplace:  # in place: the bits of the out-of-place call
                        ref = run_device(case, plain(g.batch, g.in_inner, g.out_inner), sms)
                        assert np.array_equal(rows.view(np.uint32), ref.view(np.uint32)), f"N={N} in place differs from out of place"
            finally:
                case.close()
    SWEEPS_RUN.add((N, is_c))


def test_unordered_r2c_2048_across_4096_rows(cf):
    """Unordered R2C 2048 runs wpipe_kernel from 4096 rows on and fft_kernel below: 4095 and 4096 rows."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    N = 2048
    for W, avx in widths(N, False).items():
        case = Case(cf, N, False, False, W, avx, False, 4096)
        try:
            for b in (4095, 4096):
                run_device(case, plain(b, N, N), sms)
        finally:
            case.close()
    SWEEPS_RUN.add("4096")


# --------------------------------------------------------------------------------------------------
# host pointers
# --------------------------------------------------------------------------------------------------
def host_call(cf, case: Case, g: Geometry, kind: str):
    """The case on host buffers: 'pageable' (staged in chunks), 'pinned-zero-copy' (the kernel reads host memory),
    'pinned-staged' (pinned, but over the zero-copy limit).  Returns the output rows."""
    nfl = case.nfl
    ioff, ooff = g.rows("in"), g.rows("out")
    pin = kind != "pageable"
    hin = torch.full((span(ioff, nfl),), float("nan"), pin_memory=pin)
    hout = torch.full((span(ooff, nfl),), float("nan"), pin_memory=pin)
    for r, o in enumerate(ioff):
        hin[o:o + nfl] = torch.from_numpy(case.inp[r])
    nbytes = 4 * max(span(ioff, nfl), span(ooff, nfl))
    cf.set_tuning("zero_copy_kb", (nbytes >> 10) + 1 if kind == "pinned-zero-copy" else 0 if kind == "pinned-staged" else -1)
    try:
        case.call(g, hin.data_ptr() + 4 * g.in_off, hout.data_ptr() + 4 * g.out_off)
        torch.cuda.synchronize()
    finally:
        cf.set_tuning("zero_copy_kb", -1)
    out = hout.numpy()
    REACHED.add("host zero-copy" if kind == "pinned-zero-copy" and g.outer == 1 else "host staged")
    return np.stack([out[o:o + nfl] for o in ooff])


HOST_CASES = [
    # one-level: 4099 rows cross a 32 MiB chunk and the 4096-row line (first chunk wpipe_kernel, last chunk fft_kernel)
    ("r2c-2048-unordered-4099", 2048, False, False, False, plain(4099, 2048, 2048)),
    ("c2c-16384-plain", 16384, True, True, False, plain(3, 2 * 16384 + 4, 2 * 16384 + 8)),
    ("c2r-32768-unordered", 32768, False, False, True, plain(3, 32768, 32768)),
    # two-level: 52 channels of 5 rows, 51 per 32 MiB chunk, so the last chunk has one channel and runs pipe_kernel while
    # the device call and the other chunks run fft_kernel<14,32>
    ("c2c-16384-two-level", 16384, True, True, False, Geometry(52, 5, 5 * 32768, 32768, 5 * 32768, 32768)),
    ("c2c-16384-two-level-bwd", 16384, True, True, True, Geometry(52, 5, 5 * 32768, 32768, 5 * 32768, 32768)),
]


@pytest.mark.parametrize("name,N,is_c,ordered,backward,g", HOST_CASES, ids=[c[0] for c in HOST_CASES])
def test_host_pointers_equal_device_pointers(cf, name, N, is_c, ordered, backward, g):
    """Host buffers (pageable, pinned zero-copy, pinned staged) give the bits of the device-pointer call, whichever
    kernel each staged chunk is routed to."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    nfl = 2 * N if is_c else N
    if g.outer > 1:
        assert CHUNK_BYTES // (g.inner * nfl * 4) == g.outer - 1, "the last chunk must hold exactly one channel"
    W = 8
    avx = widths(N, is_c)[W] if not ordered else True
    case = Case(cf, N, is_c, ordered, W, avx, backward, g.batch)
    try:
        dev_rows = run_device(case, g, sms)
        kinds = ["pageable", "pinned-staged"] + (["pinned-zero-copy"] if g.outer == 1 else [])
        for kind in kinds:
            rows = host_call(cf, case, g, kind)
            diff = np.nonzero((rows.view(np.uint32) != dev_rows.view(np.uint32)).any(axis=1))[0]
            assert diff.size == 0, f"{name} {kind}: rows {diff[:8].tolist()} ({diff.size} of {g.batch}) differ from the device-pointer call"
    finally:
        case.close()
    SWEEPS_RUN.add(name)


def test_every_route_was_reached():
    """The sweep above reached every route of the dispatcher's table (run with the whole module)."""
    if len(SWEEPS_RUN) < len(SWEEP) + 1 + len(HOST_CASES):
        pytest.skip("only part of the module ran")
    missing = [r for r in ROUTES if r not in REACHED]
    assert not missing, f"routes never reached: {missing}; reached {sorted(REACHED)}"
