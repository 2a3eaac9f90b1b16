"""CPU checks of what tests/test_gpu_sizes.py trusts before it judges a kernel: the list of accepted sizes, the closed form
of the unordered layouts, and the float64 references (closed forms of sparse inputs, sampled DFTs of dense ones)
against numpy.fft."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import oracle as o  # noqa: E402
from tests.test_gpu_sizes import (MAX_LOG_N, MIXED_MAX_M, SPARSE_TERMS, accepted_sizes, covering_indices, dft_at,  # noqa: E402
                                  family, gather_unordered, host_dft, sparse_input, unordered_slots, widths)


def brute_force_sizes(is_c):
    """Trial division over every N up to 2^15 (every mixed-radix size is below 24577), powers of two above."""
    unit = 16 if is_c else 32
    out = []
    for N in range(1, 1 << 15):
        m = N
        for r in (2, 3, 5):
            while m % r == 0:
                m //= r
        if N & (N - 1) == 0:
            ok = N >= unit
        else:
            ok = m == 1 and N % unit == 0 and (N if is_c else N // 2) <= MIXED_MAX_M
        if ok:
            out.append(N)
    return out + [1 << e for e in range(15, MAX_LOG_N + 1)]


@pytest.mark.parametrize("is_c", [True, False])
def test_accepted_sizes_match_brute_force(is_c):
    sizes = accepted_sizes(is_c)
    assert list(sizes) == brute_force_sizes(is_c)
    pow2 = [N for N in sizes if N & (N - 1) == 0]
    mixed = [N for N in sizes if N & (N - 1)]
    assert len(pow2) == (25 if is_c else 24) and pow2[0] == (16 if is_c else 32) and pow2[-1] == 1 << 28
    assert len(mixed) == 69
    for N in sizes:  # every accepted size has a SIMD width in the reference's rule, and a family
        assert set(widths(N, is_c)) <= {4, 8} and 0 not in widths(N, is_c)
        assert family(N, is_c) in ("single", "multipass", "mixq", "mixed")
    assert {family(N, is_c) for N in mixed} == {"mixq", "mixed"}


@pytest.mark.parametrize("N,is_c,W", [(16, True, 4), (64, True, 8), (64, True, 4), (96, True, 4), (960, True, 8), (4096, True, 8),
                                      (32, False, 4), (128, False, 8), (480, False, 4), (1920, False, 8), (8192, False, 4)])
def test_unordered_slots_equal_the_oracle_map(N, is_c, W):
    nfl = 2 * N if is_c else N
    got = unordered_slots(torch.arange(nfl), N, is_c, W).numpy()
    assert np.array_equal(got, o.np_unordered_map(N, is_c, W))
    x = torch.from_numpy(np.random.default_rng(N).uniform(-1, 1, nfl))
    assert np.array_equal(gather_unordered(x, N, is_c, W, block=nfl // 3 + 1).numpy(), x.numpy()[o.np_unordered_map(N, is_c, W)])


# (N, is_c, log2 lengths of the passes): three- and two-pass shapes at sizes numpy transforms at once
SHAPES = [(1024, True, (3, 3, 4)), (4096, True, (6, 0, 6)), (2048, False, (3, 3, 4)), (512, False, (4, 0, 4))]


@pytest.mark.parametrize("N,is_c,logs", SHAPES)
@pytest.mark.parametrize("backward", [False, True])
def test_sparse_closed_forms_match_numpy(N, is_c, logs, backward):
    """dft_at on a sparse input == float64 numpy.fft, every slot, in the ordered layout and (forward) every unordered width."""
    rng = np.random.default_rng(N + backward)
    M = N if is_c else N // 2
    nfl = 2 * N if is_c else N
    src, val = sparse_input(rng, logs, N, is_c, backward, "cpu")
    m = (src // 2).numpy()
    if not (backward and not is_c):
        assert len(set(m)) == SPARSE_TERMS and m.min() > 0 and m.max() < M
    x = np.zeros(nfl)
    x[src.numpy()] = val.numpy()
    ref = host_dft(x[None], N, is_c, backward)[0]
    u = torch.arange(nfl)
    np.testing.assert_allclose(dft_at(u, src, val, N, is_c, backward, block=997).numpy(), ref, rtol=0, atol=1e-11)
    if not backward:
        for W in widths(N, is_c):
            got = dft_at(unordered_slots(u, N, is_c, W), src, val, N, is_c, backward).numpy()
            np.testing.assert_allclose(got, ref[o.np_unordered_map(N, is_c, W)], rtol=0, atol=1e-11)


@pytest.mark.parametrize("N,is_c,logs", SHAPES)
@pytest.mark.parametrize("backward", [False, True])
def test_sampled_dft_of_dense_input_matches_numpy(N, is_c, logs, backward):
    """dft_at on a dense float32 input == float64 numpy.fft at the covering indices (both floats of each), in blocks."""
    rng = np.random.default_rng(N + 7 + backward)
    M = N if is_c else N // 2
    nfl = 2 * N if is_c else N
    x = rng.uniform(-1, 1, nfl).astype(np.float32)
    picks = covering_indices(rng, logs, M, 48)
    for j, l in enumerate(logs):  # every bit of every output digit is set in some pick
        shift = sum(logs[:j])
        for b in range(l):
            assert any((k >> (shift + b)) & 1 for k in picks), (j, b)
    assert {0, 1, M // 2, M - 1} <= set(picks) and len(picks) == 48
    slots = torch.tensor([2 * k + p for k in picks for p in (0, 1)])
    got = dft_at(slots, None, torch.from_numpy(x), N, is_c, backward, block=4096).numpy()
    ref = host_dft(x[None], N, is_c, backward)[0][slots.numpy()]
    np.testing.assert_allclose(got, ref, rtol=0, atol=1e-10 * np.sqrt(N))
