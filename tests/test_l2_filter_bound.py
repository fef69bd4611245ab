"""The error bound behind the dot-product filter for L2 / L2 squared (DESIGN 3.1b, zebra_b200/csrc/zb_scan3_kernel.cuh METRIC 3):

    A = fma(-2, S, fl(n2(a) + n2(q)))      S, n2 = canonical 16-lane dot products (what simsimd's dot computes, lsh.rs:40)
    |A - D_c| <= Eq = ecoef * (n2(a) + n2(q)) + 1e-37,   ecoef = (4 chunks + 32) * 2^-24 * 1.01

where D_c is the EXACT canonical f32 value of sum (a - q)^2 (simsimd's l2sq, distance.rs:41) -- the value the reference
returns and the second pass recomputes.  Every list the two passes produce is exact only because this inequality holds for
every (row, query) whose norms are inside the limit, so it is checked here on the CPU with the oracle's arithmetic, on random
and on adversarial vectors: heavy cancellation (a ~ q, a == q, a == -q), scales from 1e-22 (squares underflow) to 1e15,
components of mixed magnitude, sparse vectors, dimensions that are not multiples of 16.  The kernel uses the LARGER bound with
the leaf's maximal norm in place of the row's, so the per-pair form tested here is the stricter statement."""
import numpy as np
import pytest

from oracle import zb_oracle as zo

F32 = np.float32
N2_LIMIT = F32(1e37)


def canonical_dots(a, b):
    return np.array([zo.dot(x, y) for x, y in zip(a, b)], dtype=F32)


def check_pairs(a, b):
    a = np.ascontiguousarray(a, F32)
    b = np.ascontiguousarray(b, F32)
    dim = a.shape[1]
    chunks = (dim + 15) // 16
    ecoef = F32(F32(4 * chunks + 32) * F32(2.0 ** -24) * F32(1.01))
    with np.errstate(over="ignore", invalid="ignore", under="ignore"):
        dc = zo.distance_bits_batch(zo.L2SQ, a, b).view(np.float64)          # exact canonical f32 sum, widened
        s = canonical_dots(a, b)
        na, nb = canonical_dots(a, a), canonical_dots(b, b)
        w = (na + nb).astype(F32)                                           # one f32 addition
        # fma(-2, S, W): -2 S is exact, the sum of two f32 values is exact in f64 unless they are > 2^29 apart (then the
        # smaller one is far below the result's half ulp and the double rounding cannot matter for an inequality with slack)
        A = (np.float64(-2.0) * s.astype(np.float64) + w.astype(np.float64)).astype(F32)
        usable = (w <= N2_LIMIT) & np.isfinite(A)
        eq = ecoef.astype(np.float64) * (na.astype(np.float64) + nb.astype(np.float64)) + 1e-37
        err = np.abs(A.astype(np.float64) - dc)
    assert usable.any()
    bad = usable & ~(err <= eq)
    assert not bad.any(), (dim, int(bad.sum()), float((err[bad] / eq[bad]).max()))
    # whatever the kernel treats as usable has a finite exact value too (nothing overflowed on the exact side)
    assert np.isfinite(dc[usable]).all()
    return float((err[usable] / eq[usable]).max())


@pytest.mark.parametrize("dim", [1, 7, 16, 48, 100, 384, 768, 1000, 1024, 1536, 2048, 3072, 4096, 4672])
def test_bound_on_random_and_cancelling_pairs(dim):
    """Up to 4672 dimensions: the widest row for which the fused kernel (and with it the filter) still fits in shared memory
    (test_scan3.py::test_tile_config_regimes)."""
    rng = np.random.default_rng(dim)
    worst = 0.0
    for scale in (1.0, 1e-3, 1e3, 1e-15, 1e15):
        n = 60
        a = (rng.standard_normal((n, dim)) * scale).astype(F32)
        far = (rng.standard_normal((n, dim)) * scale).astype(F32)
        near = (a + (rng.standard_normal((n, dim)) * scale * 1e-3).astype(F32)).astype(F32)     # D ~ 1e-6 |a|^2: A is all cancellation
        nearer = np.nextafter(a, F32(np.inf)).astype(F32)                                          # one ulp apart in every component
        worst = max(worst, check_pairs(a, far), check_pairs(a, near), check_pairs(a, nearer), check_pairs(a, a.copy()),
                    check_pairs(a, -a))
    assert worst < 1.0            # and in practice far below: the bound is a worst case, rounding errors add like a random walk


def test_bound_with_mixed_magnitudes_sparse_and_tiny_vectors():
    rng = np.random.default_rng(5)
    dim, n = 200, 80
    a = rng.standard_normal((n, dim)).astype(F32)
    b = rng.standard_normal((n, dim)).astype(F32)
    mag = (10.0 ** rng.integers(-6, 7, size=(n, dim))).astype(F32)
    check_pairs(a * mag, b * mag)                                   # components from 1e-6 to 1e6 inside one vector
    check_pairs(a * mag, b)                                         # ... against an ordinary one
    sparse = a * (rng.random((n, dim)) < 0.05)
    check_pairs(sparse, b * (rng.random((n, dim)) < 0.05))
    check_pairs(sparse, sparse.copy())
    tiny = (a * F32(1e-22)).astype(F32)                             # squares ~1e-44: subnormal or zero; covered by the 1e-37 term
    check_pairs(tiny, (b * F32(1e-22)).astype(F32))
    check_pairs(tiny, np.zeros_like(tiny))
    check_pairs((a * F32(1e-19)).astype(F32), (b * F32(1e-19)).astype(F32))   # squares around the smallest normal number
    big = (a * F32(5e16)).astype(F32)                               # |x|^2 ~ 5e35: just inside the 1e37 limit for the pair
    check_pairs(big, (b * F32(5e16)).astype(F32))


def test_rows_beyond_the_limit_are_what_the_kernel_excludes():
    """Norms whose sum exceeds 1e37 (or is not finite) are never scored through A: the kernel gives such rows key 0 and the
    visit is rescanned exactly.  Here: the predicate catches every pair whose exact value overflowed."""
    rng = np.random.default_rng(6)
    dim, n = 64, 200
    a = (rng.standard_normal((n, dim)) * 10.0 ** rng.uniform(17, 19.5, size=(n, 1))).astype(F32)
    b = (rng.standard_normal((n, dim)) * 10.0 ** rng.uniform(17, 19.5, size=(n, 1))).astype(F32)
    with np.errstate(over="ignore", invalid="ignore"):
        dc = zo.distance_bits_batch(zo.L2SQ, a, b).view(np.float64)
        w = (canonical_dots(a, a) + canonical_dots(b, b)).astype(F32)
    usable = w <= N2_LIMIT
    assert (~usable).any() and (~np.isfinite(dc)).any()
    assert np.isfinite(dc[usable]).all()
