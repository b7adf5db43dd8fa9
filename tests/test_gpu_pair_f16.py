"""The rank-64 pair kernel accumulates the Gramian with fp16 m16n8k16 MMAs on a hi/lo split scaled by a power of two
per 16-rating chunk.  fp16 covers only about 6e-8 .. 65504, so these cases put the scaled values far outside that
range: without the chunk scale they flush to zero or overflow.  One iteration against the oracle at rank 64.

Scaling every factor by 2^s and lambda by 2^2s is an exactly equivalent problem (the solution scales by 2^-s), so the
tolerance is the one of the unscaled problem."""
import numpy as np
import pytest

from pio_b200 import synth

pytestmark = pytest.mark.gpu

TOL = 1e-4


def frob_rel(a, b):
    a = a.astype(np.float64)
    b = b.astype(np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def one_iteration(native, oracle, nu, ni, u, i, r, implicit, s, lam=0.05, alpha=1.0):
    rank = 64
    u0 = np.ldexp(synth.synth_init_factors(nu, rank, 5, 0), s).astype(np.float32)
    i0 = np.ldexp(synth.synth_init_factors(ni, rank, 5, 1), s).astype(np.float32)
    lam_s = lam * 2.0 ** (2 * s)
    m = native.NativeALS(rank, nu, ni, lam=lam_s, implicit=implicit, alpha=alpha)
    m.set_ratings(u, i, r)
    m.set_init(u0, i0)
    m.run(1)
    g = m.get_factors()
    ph = m.phase_ms()
    assert ph["item_kernel"] == "pair" and ph["user_kernel"] == "pair", ph
    o = oracle.als_train(nu, ni, u, i, r, rank, 1, lam_s, implicit, alpha, u0, i0)
    assert (g[2] == o[2]).all() and (g[3] == o[3]).all()
    assert np.isfinite(g[0]).all() and np.isfinite(g[1]).all()
    return frob_rel(g[0], o[0]), frob_rel(g[1], o[1])


def uniform_ratings(nu, ni, nnz, seed, lo, hi, log=False):
    """Uniformly spread ratings: every user and item gets more ratings than the rank, so that the half-step whose
    regularisation the scaling shrinks (lambda * 2^2s against a Gramian of scale 2^-2s) stays positive definite."""
    rng = np.random.default_rng(seed)
    u = rng.integers(0, nu, nnz).astype(np.int32)
    i = rng.integers(0, ni, nnz).astype(np.int32)
    v = rng.uniform(lo, hi, nnz)
    return u, i, (np.power(10.0, v) if log else v).astype(np.float32)


@pytest.mark.parametrize("implicit", [True, False])
@pytest.mark.parametrize("s", [-20, 20])
def test_source_factors_scaled_by_powers_of_two(native, oracle, s, implicit):
    """(a) implicit and (c) explicit: every factor scaled by 2^-20 or 2^20 (products down to 2^-40 and up to 2^40)."""
    nu, ni, nnz = 1500, 300, 300000     # ~200 ratings per user, ~1000 per item
    u, i, r = uniform_ratings(nu, ni, nnz, 13, 1.0, 5.0)
    eu, ei = one_iteration(native, oracle, nu, ni, u, i, r, implicit, s)
    assert eu <= TOL and ei <= TOL, (eu, ei)


def test_implicit_confidences_up_to_1e6(native, oracle):
    """(b) ratings log-uniform in [1e4, 1e6] on factors scaled by 2^8: sqrt(c1) y reaches ~2^17, past the fp16 maximum."""
    nu, ni, nnz = 1500, 300, 300000
    u, i, r = uniform_ratings(nu, ni, nnz, 17, 4.0, 6.0, log=True)
    eu, ei = one_iteration(native, oracle, nu, ni, u, i, r, True, 8)
    assert eu <= TOL and ei <= TOL, (eu, ei)


def test_scaled_rows_longer_than_the_part_threshold(native, oracle):
    """(d) items of ~5000 ratings (cut into 512-rating parts, summed by the finish kernel) on factors scaled by 2^-20."""
    nu, ni, nnz = 20000, 200, 1000000
    u, i, r = uniform_ratings(nu, ni, nnz, 9, 1.0, 5.0)
    eu, ei = one_iteration(native, oracle, nu, ni, u, i, r, True, -20)
    assert eu <= TOL and ei <= TOL, (eu, ei)
