"""The Cholesky sampler above 4096 unknowns: the factor and L^-1 are formed on the device (cuSOLVER), the lower triangle of
L^-1 is packed into 64 x 64 tiles and every sample streams it twice.  References are float64 numpy / scipy dense factors,
the CPU oracle's V-cycle for the gamgmc case."""
import numpy as np
import pytest
import scipy.linalg as sla
import scipy.sparse as sp

from test_gpu_parity import _obs_matrix, oracle_mg

pytestmark = pytest.mark.gpu

SEED = 20260625
TOL = 1e-10


@pytest.fixture(scope="module")
def pmg():
    import parmgmc_b200 as m
    if m.device_count() == 0:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box")
    return m


@pytest.fixture(scope="module")
def ctx(pmg):
    c = pmg.Context(0, seed=0xCAFE)
    yield c
    c.close()


def relerr(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def from_scipy(pmg, ctx, M):
    M = sp.csr_matrix(M)
    M.sort_indices()
    return pmg.Mat.from_csr(ctx, M.indptr.astype(np.int64), M.indices.astype(np.int32), M.data)


def chol_pc(pmg, ctx, mat, opts=None):
    pc = pmg.PC(ctx, "cholsampler")
    pc.set_operator(mat)
    pc.set_options(opts or {})
    pc.setup()
    return pc


def ref_sample(Lw, b, z):
    """y = L^-T (L^-1 b + z), L the lower factor (src/pc_chols.c:284-287)."""
    v = sla.solve_triangular(Lw, b, lower=True) + z
    return sla.solve_triangular(Lw.T, v, lower=False)


def operator(orc, case):
    """65^2 grid (n = 4225, just above the 4096 of the host path) or a randomly permuted 80^2 grid (n = 6400)."""
    if case == "grid65":
        return orc.laplace(2, 65, 65, kappa=0.005).to_scipy()
    A = orc.laplace(2, 80, 80, kappa=0.005).to_scipy()
    p = np.random.default_rng(SEED).permutation(A.shape[0])
    return A[p][:, p].tocsr()


@pytest.mark.parametrize("case", ["grid65", "permuted80"])
def test_injected_tape_matches_dense_factor(pmg, ctx, orc, case):
    A = operator(orc, case)
    n = A.shape[0]
    pc = chol_pc(pmg, ctx, from_scipy(pmg, ctx, A))
    assert f"size {n}" in pc.view() and "device factor" in pc.view()
    Lw = np.linalg.cholesky(A.toarray())
    rng = np.random.default_rng(SEED)
    z, b = rng.standard_normal(4 * n), rng.standard_normal(n)
    pc.set_noise_tape(z)
    y = np.zeros(n)
    pc.apply_richardson(b, y, its=1)
    assert relerr(y, ref_sample(Lw, b, z[:n])) < TOL
    y3 = np.zeros(n)
    pc.apply_richardson(b, y3, its=3)  # cached forward product (src/pc_chols.c:306-336), last of three samples
    assert relerr(y3, ref_sample(Lw, b, z[3 * n:])) < TOL


@pytest.mark.parametrize("case", ["grid65", "permuted80"])
def test_noise_none_is_the_exact_solve(pmg, ctx, orc, case):
    A = operator(orc, case)
    n = A.shape[0]
    pc = chol_pc(pmg, ctx, from_scipy(pmg, ctx, A), {"-pc_b200_noise": "none"})
    b = np.random.default_rng(SEED).standard_normal(n)
    y = np.zeros(n)
    pc.apply_richardson(b, y, its=1)
    assert relerr(y, np.linalg.solve(A.toarray(), b)) < TOL


def test_chain_of_three_equals_three_single_samples_bitwise(pmg, ctx, orc):
    A = operator(orc, "grid65")
    n = A.shape[0]
    pc = chol_pc(pmg, ctx, from_scipy(pmg, ctx, A), {"-pc_b200_noise": "philox"})
    b = np.random.default_rng(SEED).standard_normal(n)

    def run(its_per_call, calls):
        ctx.set_seed(0x5EED)
        ctx.draw_counter = 0
        out = []
        pc.set_sample_callback(lambda it, ys: out.append(ys.copy()))
        y = np.zeros(n)
        for _ in range(calls):
            pc.apply_richardson(b, y, its=its_per_call)
        pc.set_sample_callback(None)
        return np.array(out)

    one = run(3, 1)
    assert one.shape == (3, n)
    assert np.array_equal(one, run(1, 3))
    assert np.array_equal(one, run(3, 1))  # the fold of the partial sums has a fixed order


def test_lrc_operator_factors_the_sum(pmg, ctx, orc):
    """MATLRC A + B diag(S) B^T, k = 5: the sum is assembled on the device before the factorisation (src/pc_chols.c:119-157)."""
    rng = np.random.default_rng(SEED)
    A = orc.laplace(2, 65, 65, kappa=0.05)
    n, k = A.n, 5
    B, S = _obs_matrix(rng, n, k), rng.uniform(0.5, 2.0, k)  # cond(A + B S B^T) about 4e3
    mat = pmg.Mat.lrc(pmg.Mat.from_csr(ctx, A.rowptr, A.col, A.val), B, S)
    pc = chol_pc(pmg, ctx, mat)
    Lw = np.linalg.cholesky(A.to_scipy().toarray() + B @ np.diag(S) @ B.T)
    z, b = rng.standard_normal(2 * n), rng.standard_normal(n)
    pc.set_noise_tape(z)
    y = np.zeros(n)
    pc.apply_richardson(b, y, its=2)
    assert relerr(y, ref_sample(Lw, b, z[n:])) < TOL


def test_gamgmc_with_a_4225_row_coarsest_level_matches_oracle(pmg, ctx, orc):
    dims, levels, kappa = (129, 129), 2, 0.01
    lap = pmg.Mat.laplace(ctx, 2, dims[0], dims[1], kappa=kappa)
    pc = pmg.PC(ctx, "gamgmc")
    pc.set_operator(lap)
    pc.set_options({"-gamgmc_pc_mg_levels": levels, "-pc_b200_coloring": "parity"})
    pc.setup()
    assert pc.gamgmc_level_info(0)[0] == 65 * 65
    assert "packed L^-1" in pc.view()
    omg = oracle_mg(orc, 2, dims + (1,), kappa, levels)
    rng = np.random.default_rng(SEED)
    its, per, n = 2, pc.noise_per_sample(), dims[0] * dims[1]
    z, b = rng.standard_normal(its * per), rng.standard_normal(n)
    pc.set_noise_tape(z)
    y = np.full(n, 0.5)
    pc.apply_richardson(b, y, its=its)
    ref = omg.richardson(orc.Noise.tape(z), b, np.full(n, 0.5), its)
    assert relerr(y, ref) < TOL, relerr(y, ref)


def test_woodbury_exact_posterior_above_4096(pmg, ctx, orc):
    """-pc_woodbury_sampler cholsampler -pc_woodbury_solver cholesky with n = 4225: per sample w = b + B (sqrt|S| z_k),
    x = L^-T (L^-1 w + z_n) with A = L L^T, y = x - G B^T x, G = C (S^-1 + B^T C)^-1, C = A^-1 B (src/woodbury.c);
    without noise this is the posterior mean (A + B S B^T)^-1 b."""
    rng = np.random.default_rng(SEED)
    A = orc.laplace(2, 65, 65, kappa=0.005)
    n, k = A.n, 5
    B, S = _obs_matrix(rng, n, k), rng.uniform(50.0, 200.0, k)
    Ad = A.to_scipy().toarray()
    P = Ad + B @ np.diag(S) @ B.T
    b = rng.standard_normal(n)

    def woodbury(noise):
        pc = pmg.PC(ctx, "woodbury")
        pc.set_operator(pmg.Mat.lrc(pmg.Mat.from_csr(ctx, A.rowptr, A.col, A.val), B, S))
        pc.set_options({"-pc_woodbury_sampler": "cholsampler", "-pc_woodbury_solver": "cholesky", "-pc_b200_noise": noise})
        pc.setup()
        return pc

    pc = woodbury("injected")
    its, per = 2, pc.noise_per_sample()
    assert per == k + n
    z = rng.standard_normal(its * per)
    pc.set_noise_tape(z)
    y = np.zeros(n)
    pc.apply_richardson(b, y, its=its)
    Lw = np.linalg.cholesky(Ad)
    Cm = np.linalg.solve(Ad, B)
    G = Cm @ np.linalg.inv(np.diag(1.0 / S) + B.T @ Cm)
    zl = z[per:]  # the last sample's draws: k first (src/woodbury.c:273), then the sampler's n
    x = ref_sample(Lw, b + B @ (np.sqrt(np.abs(S)) * zl[:k]), zl[k:])
    assert relerr(y, x - G @ (B.T @ x)) < TOL

    y0 = np.zeros(n)
    woodbury("none").apply_richardson(b, y0, its=1)
    assert relerr(y0, np.linalg.solve(P, b)) < TOL


def test_philox_sample_mean_and_variances(pmg, ctx, orc):
    """2000 exact samples of N(A^-1 b, A^-1) at n = 4225 (kappa = 0.05).  Mean: N (m - mu)^T A (m - mu) is chi^2 with n
    degrees of freedom (mean n, sd sqrt(2 n)); held to n +- 6 sqrt(2 n).  Variances: (N - 1) s_i^2 / sigma_i^2 is chi^2 with
    N - 1 degrees of freedom, so s_i^2 / sigma_i^2 is 1 with sd sqrt(2 / (N - 1)); every node is held to 1 +- 6.5 sd (a
    union bound over the 4225 nodes keeps a false failure below 1e-5) and their average to 1 +- 3 sd."""
    A = orc.laplace(2, 65, 65, kappa=0.05).to_scipy()
    n, N = A.shape[0], 2000
    pc = chol_pc(pmg, ctx, from_scipy(pmg, ctx, A), {"-pc_b200_noise": "philox"})
    b = np.random.default_rng(SEED).standard_normal(n)
    out = np.empty((N, n))

    def cb(it, ys):
        out[it] = ys

    ctx.set_seed(0xCAFE)
    pc.set_sample_callback(cb)
    pc.apply_richardson(b, np.zeros(n), its=N)
    pc.set_sample_callback(None)
    Ad = A.toarray()
    mu, var = np.linalg.solve(Ad, b), np.diag(np.linalg.inv(Ad))
    d = out.mean(0) - mu
    t = N * d @ (Ad @ d)
    assert abs(t - n) < 6.0 * np.sqrt(2.0 * n), t
    ratio = out.var(0, ddof=1) / var
    sd = np.sqrt(2.0 / (N - 1))
    assert np.abs(ratio - 1.0).max() < 6.5 * sd, np.abs(ratio - 1.0).max()
    assert abs(ratio.mean() - 1.0) < 3.0 * sd, ratio.mean()


def test_size_above_int32_index_range(pmg, ctx, orc):
    """n = 216^2 = 46656: n^2 > 2^31, so every matrix index is 64-bit; noise none gives A^-1 b."""
    A = orc.laplace(2, 216, 216, kappa=0.001)
    n = A.n
    assert n * n > 2**31
    mat = pmg.Mat.from_csr(ctx, A.rowptr, A.col, A.val)
    pc = chol_pc(pmg, ctx, mat, {"-pc_b200_noise": "none"})
    b = np.random.default_rng(SEED).standard_normal(n)
    y = np.zeros(n)
    pc.apply_richardson(b, y, its=1)
    assert np.linalg.norm(b - mat.mult(y)) / np.linalg.norm(b) <= 1e-10
    pc.close()


def test_errors_above_4096(pmg, ctx, orc):
    A = orc.laplace(2, 65, 65, kappa=0.005).to_scipy().tolil()
    A[4200, 4200] = -1.0  # indefinite: the leading minor of order 4201 fails
    pc = pmg.PC(ctx, "cholsampler")
    pc.set_operator(from_scipy(pmg, ctx, A))
    with pytest.raises(pmg.PMGError) as e:
        pc.setup()
    assert e.value.code == 5 and "4201" in str(e.value)

    pc = pmg.PC(ctx, "cholsampler")
    pc.set_operator(from_scipy(pmg, ctx, orc.laplace(2, 65, 65, kappa=0.005).to_scipy()))
    pc.set_option("-pc_cholsampler_b200_solve", "trsv")  # the one-CTA substitution holds n <= 4096
    with pytest.raises(pmg.PMGError) as e:
        pc.setup()
    assert e.value.code == 2

    n = 130000  # 12 n^2 bytes = 203 GB: refused before anything is allocated
    pc = pmg.PC(ctx, "cholsampler")
    pc.set_operator(from_scipy(pmg, ctx, sp.identity(n, format="csr")))
    with pytest.raises(pmg.PMGError) as e:
        pc.setup()
    assert e.value.code == 2 and str(n) in str(e.value)
