"""B^T y of a low-rank-corrected operator when the chunk sums span several steps of the fold (more chunks than one
shared-memory tile holds): the product A x + B S B^T x against scipy, and two runs bitwise equal."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dims,k", [((513, 513), 64), ((1025, 513), 17), ((33, 21), 1)])
def test_lrc_mult_many_chunks(dims, k):
    import oracle as orc
    import parmgmc_b200 as pmg
    ctx = pmg.Context(0, seed=1)
    rng = np.random.default_rng(11)
    A = orc.laplace(2, *dims, kappa=1.5)
    n = A.n
    B = np.zeros((n, k))
    for j in range(k):
        idx = rng.choice(n, size=min(n, 4096), replace=False)
        B[idx, j] = rng.uniform(0.2, 1.0, idx.size)
    S = rng.uniform(20.0, 200.0, k)
    mat = pmg.Mat.lrc(pmg.Mat.laplace(ctx, 2, *dims, kappa=1.5), B, S)
    x = rng.standard_normal(n)
    y1, y2 = mat.mult(x), mat.mult(x)
    ref = A.to_scipy() @ x + B @ (S * (B.T @ x))
    assert np.array_equal(y1, y2)
    assert np.abs(y1 - ref).max() / np.abs(ref).max() < 1e-13
    ctx.close()
