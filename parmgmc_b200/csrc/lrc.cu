// lrc.cu -- low-rank-corrected operators A + B diag(S) B^T (PETSc MATLRC, SURVEY Appendix A.6) for the sweep engine.
//
// Reference: MCSORSetUp's MATLRC branch (src/mc_sor.c:565-595), MCSORBuildLRCCorrection (src/mc_sor.c:480-544),
// MCSORPostSOR_LRC (src/mc_sor.c:101-112), PrepareRHS_LRC (src/pc_mcgibbs.c:130-140), the MATLRC branches of
// PCSORGibbsSample (src/pc_sorgibbs.c:84-101).
//
//   set-up    for each direction: C = M^-1 B (k deterministic sweeps from zero on the columns of B),
//             Bb = C (S^-1 + B^T C)^-1  (k x k solve on the host)
//   sample    w = b + sqrtdiag z + B (sqrt|S| eta),  eta ~ N(0, I_k);  sweep on A;  y -= Bb_dir (B^T y)
//
// B and Bb are dense n x k, column-major, k <= 64 (the benchmark problem has k = 17 observations,
// examples/benchmark/lshape.opts).  On the device the two tall-skinny products are a chunked, fixed-order reduction
// (B^T y: one CTA per 4096-row chunk, all k columns from one read of y; the last chunk to finish folds the chunk sums in
// chunk order) and a rank-k update; both are HBM-bound streams of B / Bb (2 n k 8 B per directional sweep, SURVEY a9).
//
// Distributed base (this rank holds n < nglobal rows, MPIAIJ with a row-distributed dense B in the reference): B, Bb and
// the vectors are this rank's rows.  Each rank folds its own B^T y into slot `rank` of an nranks x k buffer, the slots are
// all-gathered (k doubles per rank, on the compute stream, no host sync) and the update kernel sums them in rank order,
// so every rank applies the identical k-vector and two runs give the same bits.  The rank-order sum of per-rank sums
// rounds differently from one GPU's sum over all chunks: N GPUs agree with one to rounding, not bitwise.  Set-up reduces
// B^T C the same way (host, rank order).  The eta draws of PrepareRHS_LRC are one block keyed on j < k with row0 = 0, the
// same values on every rank, so the right-hand side needs no communication.
#include <cmath>

#include "common.hpp"
#include "philox.cuh"

int comm_allgatherv(pmg_ctx ctx, const double *send, double *recv, const int64_t *counts, const int64_t *displs, cudaStream_t stream); // comm.cu

namespace {
constexpr int LRC_MAX_K = 64, LRC_CHUNK = 4096, LRC_THREADS = 256, LRC_PER_THREAD = LRC_CHUNK / LRC_THREADS;
constexpr int LRC_FOLD_TILE = 2048, LRC_FOLD_PER_THREAD = LRC_FOLD_TILE / LRC_THREADS; // chunk sums staged per step of the fold

// partial[chunk * k + j] = sum over the chunk's rows of M[r + n j] * y[r]; the last chunk to finish folds the partials into
// out[j] in chunk order, starting from 0.0 (no floating-point atomics: the same bits on every run), and resets the ticket
__global__ void __launch_bounds__(LRC_THREADS) lrc_bty_partial_kernel(int64_t n, int k, const double *__restrict__ M, const double *__restrict__ y, double *__restrict__ partial, unsigned *__restrict__ ticket, double *__restrict__ out)
{
  __shared__ double red[LRC_THREADS / 32];
  const int64_t     r0 = (int64_t)blockIdx.x * LRC_CHUNK;
  double            yv[LRC_PER_THREAD];
#pragma unroll
  for (int q = 0; q < LRC_PER_THREAD; ++q) {
    const int64_t r = r0 + threadIdx.x + (int64_t)q * LRC_THREADS;
    yv[q]           = r < n ? y[r] : 0.0;
  }
  for (int j = 0; j < k; ++j) {
    const double *col = M + (size_t)j * n;
    double        acc = 0.0;
#pragma unroll
    for (int q = 0; q < LRC_PER_THREAD; ++q) {
      const int64_t r = r0 + threadIdx.x + (int64_t)q * LRC_THREADS;
      if (r < n) acc = fma(col[r], yv[q], acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double s = 0.0;
      for (int w = 0; w < LRC_THREADS / 32; ++w) s += red[w];
      partial[(size_t)blockIdx.x * k + j] = s;
    }
    __syncthreads();
  }
  __shared__ bool last;
  __threadfence(); // this chunk's partials are visible device-wide before it counts as done
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  // the fold: a dependent chain of nchunks additions per column; all threads stage the next tile of whole chunks while
  // threads 0 .. k-1 add up the current one
  __shared__ double stage[LRC_FOLD_TILE];
  const int     nchunks = (int)gridDim.x, per = LRC_FOLD_TILE / k;
  double        v[LRC_FOLD_PER_THREAD], s = 0.0;
  auto          load = [&](int c0) {
    const int64_t e0 = (int64_t)c0 * k, cnt = (int64_t)min(per, nchunks - c0) * k;
#pragma unroll
    for (int q = 0; q < LRC_FOLD_PER_THREAD; ++q) {
      const int e = threadIdx.x + q * LRC_THREADS;
      v[q]        = e < cnt ? __ldcg(partial + e0 + e) : 0.0;
    }
  };
  load(0);
  for (int c0 = 0; c0 < nchunks; c0 += per) {
    const int nc = min(per, nchunks - c0);
#pragma unroll
    for (int q = 0; q < LRC_FOLD_PER_THREAD; ++q) stage[threadIdx.x + q * LRC_THREADS] = v[q];
    __syncthreads();
    if (c0 + per < nchunks) load(c0 + per);
    if ((int)threadIdx.x < k)
      for (int c = 0; c < nc; ++c) s += stage[c * k + threadIdx.x];
    __syncthreads();
  }
  if ((int)threadIdx.x < k) out[threadIdx.x] = s;
  if (threadIdx.x == 0) *ticket = 0;
}

// t = (sum over ranks of their folded B^T y, in rank order) [* scale];  y[i] += sign * sum_j M[i + n j] t[j]
__global__ void __launch_bounds__(LRC_THREADS) lrc_rank_update_kernel(int64_t n, int k, const double *__restrict__ M, const double *__restrict__ all, int nranks, const double *__restrict__ scale, double sign, double *__restrict__ y)
{
  __shared__ double t[LRC_MAX_K];
  if ((int)threadIdx.x < k) {
    double s = all[threadIdx.x];
    for (int r = 1; r < nranks; ++r) s += all[(size_t)r * k + threadIdx.x];
    t[threadIdx.x] = scale ? __dmul_rn(s, scale[threadIdx.x]) : s;
  }
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double acc = 0.0;
  for (int j = 0; j < k; ++j) acc = fma(M[i + (size_t)j * n], t[j], acc);
  y[i] = fma(sign, acc, y[i]);
}

// out = b + B (sqrt|S| eta)   (PrepareRHS_LRC's extra term; the sweep kernel then adds sqrtdiag z)
__global__ void __launch_bounds__(LRC_THREADS) lrc_rhs_kernel(int64_t n, int k, const double *__restrict__ B, const double *__restrict__ sqrtS, NoiseArgs na, const double *__restrict__ b, double *__restrict__ out)
{
  __shared__ double w[LRC_MAX_K];
  if ((int)threadIdx.x < k) w[threadIdx.x] = na.mode == PMG_NOISE_NONE ? 0.0 : __dmul_rn(noise_value(na, threadIdx.x), sqrtS[threadIdx.x]);
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double acc = 0.0;
  for (int j = 0; j < k; ++j) acc = fma(B[i + (size_t)j * n], w[j], acc);
  out[i] = __dadd_rn(b ? b[i] : 0.0, acc);
}

// in-place inverse of a k x k matrix (row-major), Gauss-Jordan with partial pivoting; returns false when singular
bool host_invert(int k, std::vector<double> &a)
{
  std::vector<double> inv((size_t)k * k, 0.0);
  for (int i = 0; i < k; ++i) inv[(size_t)i * k + i] = 1.0;
  for (int c = 0; c < k; ++c) {
    int p = c;
    for (int r = c + 1; r < k; ++r)
      if (std::fabs(a[(size_t)r * k + c]) > std::fabs(a[(size_t)p * k + c])) p = r;
    if (a[(size_t)p * k + c] == 0.0) return false;
    if (p != c)
      for (int q = 0; q < k; ++q) {
        std::swap(a[(size_t)p * k + q], a[(size_t)c * k + q]);
        std::swap(inv[(size_t)p * k + q], inv[(size_t)c * k + q]);
      }
    const double d = 1.0 / a[(size_t)c * k + c];
    for (int q = 0; q < k; ++q) {
      a[(size_t)c * k + q] *= d;
      inv[(size_t)c * k + q] *= d;
    }
    for (int r = 0; r < k; ++r) {
      if (r == c) continue;
      const double f = a[(size_t)r * k + c];
      if (f == 0.0) continue;
      for (int q = 0; q < k; ++q) {
        a[(size_t)r * k + q] -= f * a[(size_t)c * k + q];
        inv[(size_t)r * k + q] -= f * inv[(size_t)c * k + q];
      }
    }
  }
  a = inv;
  return true;
}
} // namespace

int LrcData::init(pmg_ctx c, int64_t n_, bool dist_, int k_, const double *B_host, const double *S_host)
{
  ctx  = c;
  n    = n_;
  k    = k_;
  dist = dist_;
  if (dist) {
    // S is one replicated vector in the reference (SURVEY A.6): every rank must hold the same k and bitwise the same S.
    // Both are compared on every rank from the same gathered values, so a mismatch fails everywhere and no rank is left
    // waiting in a later collective.
    const int            nr = ctx->nranks;
    int64_t              mine = k;
    std::vector<int64_t> all((size_t)nr);
    PMG_TRY(comm_allgather_i64(ctx, &mine, 1, all.data()));
    for (int r = 0; r < nr; ++r)
      if (all[(size_t)r] != all[0]) PMG_FAIL(PMG_ERR_ARG, "low-rank term: rank %d passes %lld columns, rank 0 passes %lld (k must be the same on every rank)", r, (long long)all[(size_t)r], (long long)all[0]);
    if (k >= 1 && k <= LRC_MAX_K) {
      std::vector<int64_t> bits((size_t)k), every((size_t)nr * k);
      std::memcpy(bits.data(), S_host, sizeof(double) * (size_t)k);
      PMG_TRY(comm_allgather_i64(ctx, bits.data(), k, every.data()));
      for (int r = 1; r < nr; ++r)
        if (std::memcmp(every.data() + (size_t)r * k, every.data(), sizeof(int64_t) * (size_t)k) != 0) PMG_FAIL(PMG_ERR_ARG, "low-rank term: S on rank %d differs from S on rank 0 (S must be identical on every rank)", r);
    }
  }
  if (k < 1 || k > LRC_MAX_K) PMG_FAIL(PMG_ERR_SUP, "low-rank term with %d columns: 1 .. %d are supported", k, LRC_MAX_K);
  Bh.assign(B_host, B_host + (size_t)n * k);
  Sh.assign(S_host, S_host + k);
  std::vector<double> sq((size_t)k);
  for (int j = 0; j < k; ++j) {
    if (Sh[(size_t)j] == 0.0) PMG_FAIL(PMG_ERR_ARG, "low-rank term: S[%d] = 0 (S^-1 is needed, src/mc_sor.c:524)", j);
    sq[(size_t)j] = std::sqrt(std::fabs(Sh[(size_t)j])); // VecSqrtAbs, src/pc_mcgibbs.c:241
  }
  PMG_TRY(B.upload(Bh, ctx->stream));
  PMG_TRY(S.upload(Sh, ctx->stream));
  PMG_TRY(sqrtS.upload(sq, ctx->stream));
  nchunks = (int)((n + LRC_CHUNK - 1) / LRC_CHUNK);
  PMG_TRY(partial.alloc((size_t)nchunks * k));
  PMG_TRY(rhs.alloc((size_t)n));
  PMG_TRY(bty_all.alloc((size_t)(dist ? ctx->nranks : 1) * k));
  PMG_TRY(bty_all.zero(ctx->stream)); // a rank without rows contributes this zero slot
  PMG_TRY(ticket.alloc(1));
  PMG_TRY(ticket.zero(ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  built = false;
  return 0;
}

// MCSORBuildLRCCorrection (src/mc_sor.c:480-544) for both directions, with the deterministic sweep of `base` at omega_build
int LrcData::build(LevelOp *base, double omega_build)
{
  if (built && omega_build == omega_built && built_for == (const void *)base && built_version == base->layout_version) return 0;
  built_for     = base;
  built_version = base->layout_version;
  SweepCoeffs co;
  PMG_TRY(base->make_coeffs(omega_build, co));
  NoiseArgs      none{PMG_NOISE_NONE, nullptr, 0, 0, 0};
  DevBuf<double> C;
  PMG_TRY(C.alloc((size_t)n * k));
  std::vector<double> Ch((size_t)n * k);
  for (int d = 0; d < 2; ++d) {
    const int dir = d == 0 ? PMG_SOR_FORWARD_SWEEP : PMG_SOR_BACKWARD_SWEEP;
    PMG_TRY(C.zero(ctx->stream));
    for (int j = 0; j < k; ++j) PMG_TRY(base->sweep(dir, co, B.p + (size_t)j * n, C.p + (size_t)j * n, none)); // column j of M^-1 B
    PMG_CUDA(cudaMemcpyAsync(Ch.data(), C.p, Ch.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    PMG_TRY(correction_from(Ch, d == 0 ? Bb_f : Bb_b));
  }
  built       = true;
  omega_built = omega_build;
  return 0;
}

// out = C (S^-1 + B^T C)^-1 for a host copy of C = M^-1 B (n x k, column-major)
int LrcData::correction_from(const std::vector<double> &Ch, DevBuf<double> &out)
{
  std::vector<double> t((size_t)k * k, 0.0), bb((size_t)n * k); // t = S^-1 + B^T C
  for (int a = 0; a < k; ++a)
    for (int b2 = 0; b2 < k; ++b2) {
      const double *ba = Bh.data() + (size_t)a * n, *cb = Ch.data() + (size_t)b2 * n;
      double        s = 0.0;
      for (int64_t i = 0; i < n; ++i) s += ba[i] * cb[i];
      t[(size_t)a * k + b2] = s;
    }
  if (dist) { // every rank's k x k product over its rows, summed in rank order: every rank inverts the identical matrix
    const size_t         kk = (size_t)k * k;
    std::vector<int64_t> mine(kk), all(kk * (size_t)ctx->nranks);
    std::memcpy(mine.data(), t.data(), sizeof(double) * kk);
    PMG_TRY(comm_allgather_i64(ctx, mine.data(), (int)kk, all.data()));
    std::memcpy(t.data(), all.data(), sizeof(double) * kk);
    for (int r = 1; r < ctx->nranks; ++r)
      for (size_t e = 0; e < kk; ++e) {
        double v;
        std::memcpy(&v, all.data() + (size_t)r * kk + e, sizeof v);
        t[e] += v;
      }
  }
  for (int a = 0; a < k; ++a)
    for (int b2 = 0; b2 < k; ++b2) t[(size_t)a * k + b2] = t[(size_t)a * k + b2] + (a == b2 ? 1.0 / Sh[(size_t)a] : 0.0);
  if (!host_invert(k, t)) PMG_FAIL(PMG_ERR_NOT_SPD, "low-rank correction: S^-1 + B^T M^-1 B is singular");
  for (int j = 0; j < k; ++j)
    for (int64_t i = 0; i < n; ++i) {
      double s = 0.0;
      for (int q = 0; q < k; ++q) s += Ch[(size_t)q * n + i] * t[(size_t)q * k + j];
      bb[(size_t)j * n + i] = s;
    }
  PMG_TRY(out.upload(bb, ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// bty_all = B^T y of every rank (one slot per rank, gathered when the base is distributed)
int LrcData::bty(const double *y)
{
  const int me = dist ? ctx->rank : 0;
  if (nchunks) {
    lrc_bty_partial_kernel<<<(unsigned)nchunks, LRC_THREADS, 0, ctx->stream>>>(n, k, B.p, y, partial.p, ticket.p, bty_all.p + (size_t)me * k);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  if (!dist) return 0;
  std::vector<int64_t> counts((size_t)ctx->nranks, k), displs((size_t)ctx->nranks);
  for (int r = 0; r < ctx->nranks; ++r) displs[(size_t)r] = (int64_t)r * k;
  return comm_allgatherv(ctx, bty_all.p + (size_t)me * k, bty_all.p, counts.data(), displs.data(), ctx->stream);
}

int LrcData::rank_update(const double *M, const double *scale, double sign, double *y)
{
  if (n == 0) return 0;
  lrc_rank_update_kernel<<<(unsigned)((n + LRC_THREADS - 1) / LRC_THREADS), LRC_THREADS, 0, ctx->stream>>>(n, k, M, bty_all.p, dist ? ctx->nranks : 1, scale, sign, y);
  PMG_CUDA(cudaGetLastError());
  ctx->launches++;
  return 0;
}

int LrcData::prepare_rhs(const double *b, const NoiseArgs &na_eta, double *out)
{
  if (n == 0) return 0;
  lrc_rhs_kernel<<<(unsigned)((n + LRC_THREADS - 1) / LRC_THREADS), LRC_THREADS, 0, ctx->stream>>>(n, k, B.p, sqrtS.p, na_eta, b, out);
  PMG_CUDA(cudaGetLastError());
  ctx->launches++;
  return 0;
}

// MCSORPostSOR_LRC: y -= Bb_dir (B^T y)
int LrcData::post(int dir, double *y) { return post_with(dir == PMG_SOR_BACKWARD_SWEEP ? Bb_b.p : Bb_f.p, y); }
int LrcData::post_with(const double *M, double *y)
{
  PMG_TRY(bty(y));
  return rank_update(M, nullptr, -1.0, y);
}

// out += sign * B (S o (B^T x))
int LrcData::add_bsbt(const double *x, double sign, double *out)
{
  PMG_TRY(bty(x));
  return rank_update(B.p, S.p, sign, out);
}

// The operator A + B diag(S) B^T: everything that concerns the sweep is A's (MatLRCGetMats -> Asor, src/mc_sor.c:566);
// products and residuals include the low-rank term.
struct LrcOp final : LevelOp {
  LevelOp *base = nullptr; // borrowed, like the Mat inside a MATLRC
  LrcData  d;
  int64_t  n() const override { return base->n(); }
  int64_t  nglobal() const override { return base->nglobal(); }
  int64_t  row0() const override { return base->row0(); }
  bool     distributed() const override { return base->distributed(); }
  int      ncolors() const override { return base->ncolors(); }
  int      make_coeffs(double omega, SweepCoeffs &c) override { return base->make_coeffs(omega, c); }
  int      sweep(int dir, const SweepCoeffs &c, const double *b, double *y, const NoiseArgs &na) override { return base->sweep(dir, c, b, y, na); }
  int      residual(const double *b, const double *x, double *r) override
  {
    PMG_TRY(base->residual(b, x, r));
    return d.add_bsbt(x, -1.0, r);
  }
  int mult(const double *x, double *y) override
  {
    PMG_TRY(base->mult(x, y));
    return d.add_bsbt(x, 1.0, y);
  }
  const HostCsr *host_csr() override { return nullptr; } // the low-rank term is not part of any assembled form
  int            get_coloring(std::vector<int32_t> &c) override { return base->get_coloring(c); }
  int            set_coloring(int nc, const int32_t *c) override { return base->set_coloring(nc, c); }
  int            set_coloring_auto(int policy) override { return base->set_coloring_auto(policy); }
  void           describe(std::string &out) override
  {
    base->describe(out);
    out = "low-rank corrected (k = " + std::to_string(d.k) + ") " + out;
  }
  LrcData *lrc_data() override { return &d; }
  LevelOp *lrc_base() override { return base; }
  bool     structured(int &dim, int64_t dims[3]) const override { return base->structured(dim, dims); }
};

int make_lrc_op(pmg_ctx ctx, LevelOp *base, int k, const double *B_host, const double *S_host, std::unique_ptr<LevelOp> &op)
{
  if (base->lrc_data()) PMG_FAIL(PMG_ERR_SUP, "nested low-rank corrections are not supported");
  auto o  = std::make_unique<LrcOp>();
  o->ctx  = ctx;
  o->base = base;
  // distributed is a property of the base, not of the context: levels every rank holds in full never reduce across ranks
  PMG_TRY(o->d.init(ctx, base->n(), base->n() < base->nglobal(), k, B_host, S_host));
  op = std::move(o);
  return 0;
}
