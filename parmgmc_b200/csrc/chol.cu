// chol.cu -- dense Cholesky sampler on the device: the PCCHOLSAMPLER analogue for the coarsest level.
//
// Reference: src/pc_chols.c:173-195 (dense potrf "L" once), :220-260 (trsv "L","N" / "L","T"),
// :284-287 (v = L^-1 b; v += z; y = L^-T v  =>  y ~ N(A^-1 b, A^-1)), :306-336 (cached forward solve).
// The factor is computed once on the host at set-up (not on the per-sample path) and kept on the
// device as L and L^T (both column-major, so every per-step access is a coalesced column read).
// Two per-sample paths:
//   gemv (default)  W = L^-1 is formed once at set-up; a sample is two triangular matrix-vector products
//                   v = W b + z, y = W^T v, one warp per output entry over coalesced rows (W is kept row-major and
//                   column-major).  Fully parallel: a 289-unknown coarsest level costs a few microseconds instead
//                   of the ~0.26 ms of two sequential substitutions (profiles/r1_summary.md).  Agrees with the
//                   substitution to rounding (cond(L) eps).
//   trsv            (-pc_cholsampler_b200_solve trsv) one CTA does both triangular solves from shared memory; per
//                   unknown the accumulation order is reference-BLAS dtrsv's (forward k ascending, transposed k
//                   descending), so the result is bit-identical to the sequential substitution (src/pc_chols.c:231,253).
// Both hold n <= 4096.  Above that (any n whose factor fits the device) the set-up runs on the device instead: the operator
// is scattered into a dense work matrix, cuSOLVER factors it, cuBLAS triangular solves form W = L^-1 a panel at a time (both
// loaded at run time; cuSOLVER's trtri rejects n^2 >= 2^31), and the lower triangle of W is packed into 64 x 64 tiles.  A sample is the same two products, each one stream over the packed
// triangle (tri_rows_kernel, tri_cols_kernel), about 8 n^2 bytes per sample instead of two n x n copies.
#include <dlfcn.h>
#include <cusolverDn.h>

#include "common.hpp"
#include "philox.cuh"

namespace {
constexpr int CHOL_MAX_N   = 4096;
constexpr int CHOL_THREADS = 1024;
// packed triangle: tile (I, J), I >= J, at tile index I (I + 1) / 2 + J, each tile row-major and contiguous
constexpr int TB        = 64, TT = TB * TB;
constexpr int TRI_NT    = 256; // 8 warps, 8 tile rows each
constexpr int CHUNK_MAX = 16;  // tiles per chunk: a chunk's input segment is staged in shared memory
constexpr int PANEL_W   = 2048; // columns of U^-1 formed per triangular solve at set-up (a multiple of TB)

__device__ __forceinline__ int64_t tile_index(int64_t I, int64_t J) { return I * (I + 1) / 2 + J; }

// Last chunk of a panel to finish: fold the panel's partial sums in chunk order (no floating-point atomics, so two
// runs give the same bits), add the noise, write the panel's 64 outputs, reset the counter for the next launch.
__device__ __forceinline__ void fold_panel(const CholChunk &c, int64_t n, const double *part, unsigned *done, double *out, const NoiseArgs &na)
{
  __shared__ bool last;
  __threadfence(); // this thread's partials are visible device-wide before the chunk counts as done
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(done + c.panel, 1u) == (unsigned)(c.nq - 1);
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (threadIdx.x < TB) {
    const int64_t i = (int64_t)c.panel * TB + threadIdx.x;
    double        s = 0.0;
    for (int q = 0; q < c.nq; ++q) s += __ldcg(part + (int64_t)(c.q0 + q) * TB + threadIdx.x);
    if (i < n) out[i] = na.mode != PMG_NOISE_NONE ? __dadd_rn(s, noise_value(na, i)) : s;
  }
  if (threadIdx.x == 0) done[c.panel] = 0;
}

// out = W in (+ z): one CTA per chunk of a row panel I.  Warp w owns tile rows 8w .. 8w+7; lane l reads columns 2l, 2l+1
// of each row (512 contiguous bytes per warp and row) and keeps one running sum per row, reduced across the warp at the end.
__global__ void __launch_bounds__(TRI_NT) tri_rows_kernel(int64_t n, const double *__restrict__ tri, const CholChunk *__restrict__ list, const double *__restrict__ in, double *__restrict__ part, unsigned *__restrict__ done, double *__restrict__ out, NoiseArgs na)
{
  __shared__ __align__(16) double xs[CHUNK_MAX * TB];
  const CholChunk c    = list[blockIdx.x];
  const int       warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_launch_dependents();
  pdl_wait();
  for (int k = threadIdx.x; k < (c.t1 - c.t0) * TB; k += TRI_NT) {
    const int64_t g = (int64_t)c.t0 * TB + k;
    xs[k]           = g < n ? in[g] : 0.0;
  }
  __syncthreads();
  double         acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const double2 *tp     = reinterpret_cast<const double2 *>(tri + tile_index(c.panel, c.t0) * TT) + warp * 8 * (TB / 2) + lane;
  for (int j = 0; j < c.t1 - c.t0; ++j, tp += TT / 2) { // tiles (I, t0 .. t1-1) are consecutive
    const double2 x = reinterpret_cast<const double2 *>(xs + j * TB)[lane];
    double2       w[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) w[r] = __ldg(tp + r * (TB / 2));
#pragma unroll
    for (int r = 0; r < 8; ++r) acc[r] = fma(w[r].y, x.y, fma(w[r].x, x.x, acc[r]));
  }
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
  if (lane < 8) {
    double s = acc[0];
#pragma unroll
    for (int r = 1; r < 8; ++r) s = lane == r ? acc[r] : s;
    part[(int64_t)blockIdx.x * TB + warp * 8 + lane] = s;
  }
  fold_panel(c, n, part, done, out, na);
}

// out = W^T in: one CTA per chunk of a column panel J (tiles (t0 .. t1-1, J)).  Warp w reads tile rows 8w .. 8w+7; lane l
// owns columns 2l, 2l+1 of the panel and sums down its rows; the 8 warps' sums are added in warp order.
__global__ void __launch_bounds__(TRI_NT) tri_cols_kernel(int64_t n, const double *__restrict__ tri, const CholChunk *__restrict__ list, const double *__restrict__ in, double *__restrict__ part, unsigned *__restrict__ done, double *__restrict__ out)
{
  __shared__ __align__(16) double xs[CHUNK_MAX * TB];
  __shared__ double2              red[TRI_NT / 32][TB / 2];
  const CholChunk c    = list[blockIdx.x];
  const int       warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_launch_dependents();
  pdl_wait();
  for (int k = threadIdx.x; k < (c.t1 - c.t0) * TB; k += TRI_NT) {
    const int64_t g = (int64_t)c.t0 * TB + k;
    xs[k]           = g < n ? in[g] : 0.0;
  }
  __syncthreads();
  double2 acc = make_double2(0.0, 0.0);
  for (int I = c.t0; I < c.t1; ++I) {
    const double2 *tp = reinterpret_cast<const double2 *>(tri + tile_index(I, c.panel) * TT) + warp * 8 * (TB / 2) + lane;
    const double  *x  = xs + (I - c.t0) * TB + warp * 8;
    double2        w[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) w[r] = __ldg(tp + r * (TB / 2));
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      acc.x = fma(w[r].x, x[r], acc.x);
      acc.y = fma(w[r].y, x[r], acc.y);
    }
  }
  red[warp][lane] = acc;
  __syncthreads();
  if (threadIdx.x < TB) {
    const double *rd = reinterpret_cast<const double *>(&red[0][0]);
    double        s  = rd[threadIdx.x];
#pragma unroll
    for (int w = 1; w < TRI_NT / 32; ++w) s += rd[w * TB + threadIdx.x];
    part[(int64_t)blockIdx.x * TB + threadIdx.x] = s;
  }
  fold_panel(c, n, part, done, out, NoiseArgs{PMG_NOISE_NONE, nullptr, 0, 0, 0});
}

// ---- set-up on the device ----
// a[r + c n] = A(r, c) of the CSR operator (a zeroed)
__global__ void csr_to_dense_kernel(int64_t n, const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col, const double *__restrict__ val, double *__restrict__ a)
{
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  for (int64_t k = rowptr[r]; k < rowptr[r + 1]; ++k) a[r + (int64_t)col[k] * n] = val[k];
}
// a(r, c) += sum_j B(r, j) S_j B(c, j) for r <= c (the triangle potrf "U" reads), j ascending as the host assembly adds
__global__ void add_bsbt_dense_kernel(int64_t n, int k, const double *__restrict__ B, const double *__restrict__ S, double *__restrict__ a)
{
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t c = blockIdx.y; c < n; c += gridDim.y) {
    if (r > c) continue;
    double s = a[r + c * n];
    for (int j = 0; j < k; ++j) s = __dadd_rn(s, __dmul_rn(B[r + (int64_t)j * n], __dmul_rn(S[j], B[c + (int64_t)j * n])));
    a[r + c * n] = s;
  }
}
// x (m x w, column-major) = columns j0 .. j0+w-1 of the identity's leading m rows
__global__ void identity_panel_kernel(int64_t m, int64_t w, int64_t j0, double *__restrict__ x)
{
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < m * w) x[e] = e % m == j0 + e / m ? 1.0 : 0.0;
}
// x holds columns j0 .. j0+w-1 of U^-1 (A = U^T U), i.e. rows j0 .. of W = L^-1 = U^-T: W(i, j) = x[j + (i - j0) m].  One CTA
// per tile of the row panels I = j0 / 64 .. ; tile index t0 + blockIdx.x
__global__ void pack_panel_kernel(int64_t n, int64_t m, int64_t j0, int64_t t0, const double *__restrict__ x, double *__restrict__ tri)
{
  const int64_t t = t0 + blockIdx.x;
  int64_t       I = (int64_t)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
  while (I * (I + 1) / 2 > t) --I;
  while ((I + 1) * (I + 2) / 2 <= t) ++I;
  const int64_t J = t - I * (I + 1) / 2;
  for (int e = threadIdx.x; e < TT; e += blockDim.x) {
    const int64_t i = I * TB + e / TB, j = J * TB + e % TB;
    tri[t * TT + e] = i < n && j <= i ? x[j + (i - j0) * m] : 0.0;
  }
}

// ---- cuSOLVER (potrf) and cuBLAS (trsm), bound at run time ----
struct DenseApi {
  decltype(&cusolverDnCreate)            Create            = nullptr;
  decltype(&cusolverDnDestroy)           Destroy           = nullptr;
  decltype(&cusolverDnSetStream)         SetStream         = nullptr;
  decltype(&cusolverDnCreateParams)      CreateParams      = nullptr;
  decltype(&cusolverDnDestroyParams)     DestroyParams     = nullptr;
  decltype(&cusolverDnXpotrf_bufferSize) Xpotrf_bufferSize = nullptr;
  decltype(&cusolverDnXpotrf)            Xpotrf            = nullptr;
  decltype(&cublasCreate_v2)             BlasCreate        = nullptr;
  decltype(&cublasDestroy_v2)            BlasDestroy       = nullptr;
  decltype(&cublasSetStream_v2)          BlasSetStream     = nullptr;
  decltype(&cublasDtrsm_v2_64)           Dtrsm             = nullptr;
  bool                                   ok                = false;
};
DenseApi &dense_api()
{
  static DenseApi api = [] {
    DenseApi a;
    void    *hs = nullptr, *hb = nullptr;
    for (const char *nm : {"libcusolver.so.11", "libcusolver.so.12", "libcusolver.so"})
      if ((hs = dlopen(nm, RTLD_NOW | RTLD_GLOBAL))) break;
    for (const char *nm : {"libcublas.so.12", "libcublas.so.13", "libcublas.so"})
      if ((hb = dlopen(nm, RTLD_NOW | RTLD_GLOBAL))) break;
    if (!hs || !hb) return a;
#define PMG_SYM(h, field, name) a.field = (decltype(a.field))dlsym(h, name)
    PMG_SYM(hs, Create, "cusolverDnCreate"); PMG_SYM(hs, Destroy, "cusolverDnDestroy"); PMG_SYM(hs, SetStream, "cusolverDnSetStream");
    PMG_SYM(hs, CreateParams, "cusolverDnCreateParams"); PMG_SYM(hs, DestroyParams, "cusolverDnDestroyParams");
    PMG_SYM(hs, Xpotrf_bufferSize, "cusolverDnXpotrf_bufferSize"); PMG_SYM(hs, Xpotrf, "cusolverDnXpotrf");
    PMG_SYM(hb, BlasCreate, "cublasCreate_v2"); PMG_SYM(hb, BlasDestroy, "cublasDestroy_v2"); PMG_SYM(hb, BlasSetStream, "cublasSetStream_v2");
    PMG_SYM(hb, Dtrsm, "cublasDtrsm_v2_64");
#undef PMG_SYM
    a.ok = a.Create && a.Destroy && a.SetStream && a.CreateParams && a.DestroyParams && a.Xpotrf_bufferSize && a.Xpotrf && a.BlasCreate && a.BlasDestroy && a.BlasSetStream && a.Dtrsm;
    return a;
  }();
  return api;
}
struct DenseSession { // handles of one set-up, released on every return path
  cusolverDnHandle_t h = nullptr;
  cusolverDnParams_t p = nullptr;
  cublasHandle_t     b = nullptr;
  ~DenseSession()
  {
    if (p) dense_api().DestroyParams(p);
    if (h) dense_api().Destroy(h);
    if (b) dense_api().BlasDestroy(b);
  }
};
#define PMG_DENSE(call, lib)                                                                          \
  do {                                                                                                \
    const int s_ = (int)(call);                                                                       \
    if (s_ != 0) PMG_FAIL(PMG_ERR_CUDA, "%s:%d: %s error %d", __FILE__, __LINE__, lib, s_);           \
  } while (0)

// chunks of at most `len` tiles over panels 0 .. nt-1, panel p holding len_of(p) tiles starting at first_of(p)
template <class F0, class F1> void chunk_list(int64_t nt, int len, F0 first_of, F1 len_of, std::vector<CholChunk> &out)
{
  out.clear();
  for (int64_t p = 0; p < nt; ++p) {
    const int f = first_of(p), m = len_of(p), nq = (m + len - 1) / len, q0 = (int)out.size();
    for (int q = 0; q < nq; ++q) out.push_back(CholChunk{(int)p, f + q * len, f + std::min(m, (q + 1) * len), q0, nq});
  }
}

// s[0..n) holds the rhs on entry and the solution on exit.  blk is a 32x33 staging area for the diagonal
// block, so that the 32 dependent steps of a block read shared memory instead of waiting on L2 each time.
__device__ void trsv_forward(int n, const double *__restrict__ L, double *s, double (*blk)[33])
{
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int kb = 0; kb < n; kb += 32) {
    const int kmax = min(32, n - kb);
    {
      const int r = tid & 31, c = tid >> 5; // 1024 threads: one block entry each, column-major read is coalesced
      if (r < kmax && c < kmax) blk[r][c] = L[(kb + r) + (size_t)(kb + c) * n];
    }
    __syncthreads();
    if (warp == 0) {
      const int i  = kb + lane;
      double    si = i < n ? s[i] : 0.0;
      for (int k = 0; k < kmax; ++k) {
        double xk = 0.0;
        if (lane == k) xk = si / blk[k][k];
        xk = __shfl_sync(0xffffffffu, xk, k);
        if (lane == k) si = xk;
        else if (lane > k && i < n) si = fma(-blk[lane][k], xk, si);
      }
      if (i < n) s[i] = si;
    }
    __syncthreads();
    for (int i = kb + 32 + tid; i < n; i += blockDim.x) {
      double        si = s[i];
      const double *Lp = L + i + (size_t)kb * n;
#pragma unroll 8
      for (int k = 0; k < kmax; ++k) si = fma(-Lp[(size_t)k * n], s[kb + k], si);
      s[i] = si;
    }
    __syncthreads();
  }
}

// LT[i + k n] = L[k + i n]
__device__ void trsv_backward(int n, const double *__restrict__ L, const double *__restrict__ LT, double *s, double (*blk)[33])
{
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nb = (n + 31) / 32;
  (void)L;
  for (int b = nb - 1; b >= 0; --b) {
    const int kb = b * 32, kmax = min(32, n - kb);
    {
      const int r = tid & 31, c = tid >> 5;
      if (r < kmax && c < kmax) blk[r][c] = LT[(kb + r) + (size_t)(kb + c) * n]; // = L[kb+c, kb+r]
    }
    __syncthreads();
    if (warp == 0) {
      const int i  = kb + lane;
      double    si = i < n ? s[i] : 0.0;
      for (int k = kmax - 1; k >= 0; --k) {
        double xk = 0.0;
        if (lane == k) xk = si / blk[k][k];
        xk = __shfl_sync(0xffffffffu, xk, k);
        if (lane == k) si = xk;
        else if (lane < k) si = fma(-blk[lane][k], xk, si);
      }
      if (i < n) s[i] = si;
    }
    __syncthreads();
    for (int i = tid; i < kb; i += blockDim.x) {
      double        si = s[i];
      const double *Lp = LT + i + (size_t)kb * n;
#pragma unroll 8
      for (int k = kmax - 1; k >= 0; --k) si = fma(-Lp[(size_t)k * n], s[kb + k], si);
      s[i] = si;
    }
    __syncthreads();
  }
}

// mode bit 0: forward solve of `in`; bit 1: add noise and backward solve
__global__ void __launch_bounds__(CHOL_THREADS) chol_sample_kernel(int n, const double *__restrict__ L, const double *__restrict__ LT, const double *__restrict__ in, double *__restrict__ out, NoiseArgs na, int mode)
{
  __shared__ double s[CHOL_MAX_N];
  __shared__ double blk[32][33];
  for (int i = threadIdx.x; i < n; i += blockDim.x) s[i] = in[i];
  __syncthreads();
  if (mode & 1) trsv_forward(n, L, s, blk);
  if (mode & 2) {
    if (na.mode != PMG_NOISE_NONE)
      for (int i = threadIdx.x; i < n; i += blockDim.x) s[i] = __dadd_rn(s[i], noise_value(na, i));
    __syncthreads();
    trsv_backward(n, L, LT, s, blk);
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) out[i] = s[i];
}
// out[i] = sum_{k in [klo(i), khi(i))} M[i*n + k] in[k]  (+ z_i); LOWER: k <= i, else k >= i.  One warp per entry.
template <bool LOWER> __global__ void __launch_bounds__(256) tri_gemv_kernel(int n, const double *__restrict__ M, const double *__restrict__ in, double *__restrict__ out, NoiseArgs na)
{
  const int i    = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();
  if (i >= n) return;
  const int     k0 = LOWER ? 0 : i, k1 = LOWER ? i + 1 : n;
  const double *row = M + (size_t)i * n;
  // the factor is a launch constant: pull this warp's row towards L2 while the preceding kernel is still running
  for (int k = k0 + lane * 16; k < k1; k += 32 * 16) asm volatile("prefetch.global.L2 [%0];" ::"l"(row + k));
  pdl_wait();
  double        acc = 0.0;
  for (int k = k0 + lane; k < k1; k += 32) acc = fma(row[k], in[k], acc);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) out[i] = na.mode != PMG_NOISE_NONE ? __dadd_rn(acc, noise_value(na, i)) : acc;
}

__global__ void add_noise_kernel(int n, const double *__restrict__ v, double *__restrict__ out, NoiseArgs na)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __dadd_rn(v[i], noise_value(na, i));
}
} // namespace

double CholSampler::sample_bytes() const { return packed ? 2.0 * (double)tri.n * sizeof(double) : 16.0 * (double)n * (double)n; }

// n > 4096: factor and invert on the device, pack W = L^-1 (see the top of this file)
static int setup_packed(CholSampler &s, const HostCsr &a, const LrcData *lrc)
{
  pmg_ctx       ctx = s.ctx;
  const int64_t n = s.n, nt = (n + TB - 1) / TB, ntiles = nt * (nt + 1) / 2;
  // the work matrix, the packed triangle and one panel of U^-1 live side by side until the packing is done
  const double need = 8.0 * (double)n * (double)n + 8.0 * (double)TT * (double)ntiles + 8.0 * (double)n * PANEL_W + 12.0 * (double)a.nnz() + 8.0 * (double)(n + 1);
  size_t       free_b = 0, total_b = 0;
  PMG_CUDA(cudaMemGetInfo(&free_b, &total_b));
  if (need > (double)free_b)
    PMG_FAIL(PMG_ERR_SUP, "cholsampler: the dense factor of n = %lld needs %.0f bytes of device memory (n x n work matrix + packed triangle of L^-1); %zu are free", (long long)n, need, free_b);
  if (!dense_api().ok) PMG_FAIL(PMG_ERR_SUP, "cholsampler with n = %lld > %d factors on the device, and libcusolver / libcublas could not be loaded: %s", (long long)n, CHOL_MAX_N, dlerror());
  s.nt = nt;
  {
    DevBuf<double> work;
    PMG_TRY(work.alloc((size_t)(n * n)));
    PMG_TRY(work.zero(ctx->stream));
    {
      DevBuf<int64_t> rp;
      DevBuf<int32_t> cl;
      DevBuf<double>  vl;
      PMG_TRY(rp.upload(a.rowptr, ctx->stream));
      PMG_TRY(cl.upload(a.col, ctx->stream));
      PMG_TRY(vl.upload(a.val, ctx->stream));
      csr_to_dense_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(n, rp.p, cl.p, vl.p, work.p);
      PMG_CUDA(cudaGetLastError());
      PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    if (lrc) { // A + B diag(S) B^T (src/pc_chols.c:119-157), B and S already on the device
      add_bsbt_dense_kernel<<<dim3((unsigned)((n + 255) / 256), (unsigned)std::min<int64_t>(n, 4096)), 256, 0, ctx->stream>>>(n, lrc->k, lrc->B.p, lrc->S.p, work.p);
      PMG_CUDA(cudaGetLastError());
    }
    DenseSession ds;
    DenseApi    &api = dense_api();
    PMG_DENSE(api.Create(&ds.h), "cuSOLVER");
    PMG_DENSE(api.SetStream(ds.h, ctx->stream), "cuSOLVER");
    PMG_DENSE(api.CreateParams(&ds.p), "cuSOLVER");
    PMG_DENSE(api.BlasCreate(&ds.b), "cuBLAS");
    PMG_DENSE(api.BlasSetStream(ds.b, ctx->stream), "cuBLAS");
    // upper factor A = U^T U (L = U^T): the columns of U^-1 are the rows of W, so W's row panels come out contiguous
    size_t dw = 0, hw = 0;
    PMG_DENSE(api.Xpotrf_bufferSize(ds.h, ds.p, CUBLAS_FILL_MODE_UPPER, n, CUDA_R_64F, work.p, n, CUDA_R_64F, &dw, &hw), "cuSOLVER");
    {
      DevBuf<char>      dws;
      DevBuf<int>       dinfo;
      std::vector<char> hws(std::max<size_t>(hw, 1));
      PMG_TRY(dws.alloc(std::max<size_t>(dw, 1)));
      PMG_TRY(dinfo.alloc(1));
      int info = 0;
      PMG_DENSE(api.Xpotrf(ds.h, ds.p, CUBLAS_FILL_MODE_UPPER, n, CUDA_R_64F, work.p, n, CUDA_R_64F, dws.p, dw, hws.data(), hw, dinfo.p), "cuSOLVER");
      PMG_CUDA(cudaMemcpyAsync(&info, dinfo.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
      PMG_CUDA(cudaStreamSynchronize(ctx->stream));
      if (info > 0) PMG_FAIL(PMG_ERR_NOT_SPD, "Dense Cholesky failed: leading minor of order %d is not positive definite", info); // src/pc_chols.c:192
      if (info < 0) PMG_FAIL(PMG_ERR_CUDA, "cuSOLVER potrf: argument %d is invalid", -info);
    }
    // U^-1 panel by panel: columns j0 .. j0+w-1 solve U[0:m, 0:m] X = I[0:m, j0:j0+w] with m = j0 + w (U^-1 is upper
    // triangular), then go straight into their tiles
    PMG_TRY(s.tri.alloc((size_t)(ntiles * TT)));
    DevBuf<double> x;
    PMG_TRY(x.alloc((size_t)(n * PANEL_W)));
    const double one = 1.0;
    for (int64_t j0 = 0; j0 < n; j0 += PANEL_W) {
      const int64_t w = std::min<int64_t>(PANEL_W, n - j0), m = j0 + w;
      identity_panel_kernel<<<(unsigned)((m * w + 255) / 256), 256, 0, ctx->stream>>>(m, w, j0, x.p);
      PMG_CUDA(cudaGetLastError());
      PMG_DENSE(api.Dtrsm(ds.b, CUBLAS_SIDE_LEFT, CUBLAS_FILL_MODE_UPPER, CUBLAS_OP_N, CUBLAS_DIAG_NON_UNIT, m, w, &one, work.p, n, x.p, m), "cuBLAS");
      const int64_t I0 = j0 / TB, I1 = (m + TB - 1) / TB;
      pack_panel_kernel<<<(unsigned)(I1 * (I1 + 1) / 2 - I0 * (I0 + 1) / 2), 256, 0, ctx->stream>>>(n, m, j0, I0 * (I0 + 1) / 2, x.p, s.tri.p);
      PMG_CUDA(cudaGetLastError());
    }
    PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  } // work matrix freed
  // chunks: about 8 per SM in each product, at most CHUNK_MAX tiles
  const int           len = (int)std::max<int64_t>(1, std::min<int64_t>(CHUNK_MAX, ntiles / (8 * (int64_t)ctx->sm_count)));
  std::vector<CholChunk> rl, cl;
  chunk_list(nt, len, [](int64_t) { return 0; }, [](int64_t I) { return (int)I + 1; }, rl);                   // row panel I: J = 0 .. I
  chunk_list(nt, len, [](int64_t J) { return (int)J; }, [nt](int64_t J) { return (int)(nt - J); }, cl);       // column panel J: I = J .. nt-1
  PMG_TRY(s.rows.upload(rl, ctx->stream));
  PMG_TRY(s.cols.upload(cl, ctx->stream));
  PMG_TRY(s.part.alloc((size_t)TB * std::max(rl.size(), cl.size())));
  PMG_TRY(s.done.alloc((size_t)nt));
  PMG_TRY(s.done.zero(ctx->stream));
  PMG_TRY(s.tmp.alloc((size_t)n));
  s.packed = true;
  return 0;
}

int CholSampler::setup(pmg_ctx c, const HostCsr &a, const LrcData *lrc)
{
  ctx    = c;
  n      = a.n;
  packed = false;
  for (DevBuf<double> *d : {&L, &LT, &tri, &part}) d->release();
  if (n > CHOL_MAX_N && !use_gemv) PMG_FAIL(PMG_ERR_SUP, "coarsest operator has %lld rows; -pc_cholsampler_b200_solve trsv keeps the vector in one CTA's shared memory and handles up to %d", (long long)n, CHOL_MAX_N);
  if (n > CHOL_MAX_N) {
    PMG_TRY(setup_packed(*this, a, lrc));
    PMG_TRY(vcache.alloc((size_t)n));
    PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
  }
  std::vector<double> l((size_t)(n * n), 0.0), lt((size_t)(n * n), 0.0);
  for (int64_t r = 0; r < n; ++r)
    for (int64_t k = a.rowptr[r]; k < a.rowptr[r + 1]; ++k) l[(size_t)(r + (int64_t)a.col[k] * n)] = a.val[k];
  if (lrc) { // P = A + B diag(S) B^T, assembled densely (src/pc_chols.c:119-157 forms it as a sparse product)
    for (int j = 0; j < lrc->k; ++j) {
      const double *bj = lrc->Bh.data() + (size_t)j * n;
      const double  sj = lrc->Sh[(size_t)j];
      for (int64_t cc = 0; cc < n; ++cc) {
        const double f = sj * bj[cc];
        if (f == 0.0) continue;
        for (int64_t r = 0; r < n; ++r) l[(size_t)(r + cc * n)] += bj[r] * f;
      }
    }
  }
  const int info = host_potrf_lower(n, l);
  if (info) PMG_FAIL(PMG_ERR_NOT_SPD, "Dense Cholesky failed: leading minor of order %d is not positive definite", info); // src/pc_chols.c:192
  for (int64_t i = 0; i < n; ++i)
    for (int64_t k = 0; k < n; ++k) {
      if (k > i) l[(size_t)(i + k * n)] = 0.0; // strictly upper part of the potrf workspace is not referenced
      lt[(size_t)(i + k * n)] = k >= i ? l[(size_t)(k + i * n)] : 0.0;
    }
  if (use_gemv) { // W = L^-1 by forward substitution on the columns of the identity (column sweeps: contiguous)
    std::vector<double> w((size_t)(n * n), 0.0), wt((size_t)(n * n), 0.0);
    for (int64_t j = 0; j < n; ++j) {
      double *col = w.data() + (size_t)(j * n);
      col[j]      = 1.0;
      for (int64_t k = j; k < n; ++k) {
        const double x = col[k] / l[(size_t)(k + k * n)];
        col[k]         = x;
        const double *lk = l.data() + (size_t)(k * n);
        for (int64_t i = k + 1; i < n; ++i) col[i] = std::fma(-lk[i], x, col[i]);
      }
    }
    for (int64_t i = 0; i < n; ++i)
      for (int64_t k = 0; k <= i; ++k) wt[(size_t)(k + i * n)] = w[(size_t)(i + k * n)]; // wt = row-major W
    PMG_TRY(L.upload(wt, ctx->stream));  // "L"  slot: W row-major     (rows of W contiguous: v = W b)
    PMG_TRY(LT.upload(w, ctx->stream));  // "LT" slot: W column-major  (rows of W^T contiguous: y = W^T v)
    PMG_TRY(tmp.alloc((size_t)n));
  } else {
    PMG_TRY(L.upload(l, ctx->stream));
    PMG_TRY(LT.upload(lt, ctx->stream));
  }
  PMG_TRY(vcache.alloc((size_t)n));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

static int launch_chol(pmg_ctx ctx, int64_t n, const double *L, const double *LT, const double *in, double *out, const NoiseArgs &na, int mode)
{
  chol_sample_kernel<<<1, CHOL_THREADS, 0, ctx->stream>>>((int)n, L, LT, in, out, na, mode);
  PMG_CUDA(cudaGetLastError());
  ctx->launches++;
  return 0;
}

template <bool LOWER> static int launch_gemv(pmg_ctx ctx, int64_t n, const double *M, const double *in, double *out, const NoiseArgs &na)
{
  PMG_CUDA(launch_pdl(ctx->stream, tri_gemv_kernel<LOWER>, dim3((unsigned)((n * 32 + 255) / 256)), dim3(256), 0, (int)n, M, in, out, na));
  PMG_CUDA(cudaGetLastError());
  ctx->launches++;
  return 0;
}

static int launch_rows(const CholSampler &s, const double *in, double *out, const NoiseArgs &na)
{
  PMG_CUDA(launch_pdl(s.ctx->stream, tri_rows_kernel, dim3((unsigned)s.rows.n), dim3(TRI_NT), 0, s.n, (const double *)s.tri.p, (const CholChunk *)s.rows.p, in, s.part.p, s.done.p, out, na));
  s.ctx->launches++;
  return 0;
}
static int launch_cols(const CholSampler &s, const double *in, double *out)
{
  PMG_CUDA(launch_pdl(s.ctx->stream, tri_cols_kernel, dim3((unsigned)s.cols.n), dim3(TRI_NT), 0, s.n, (const double *)s.tri.p, (const CholChunk *)s.cols.p, in, s.part.p, s.done.p, out));
  s.ctx->launches++;
  return 0;
}

int CholSampler::sample(const double *b, double *y, const NoiseArgs &na)
{
  if (!use_gemv) return launch_chol(ctx, n, L.p, LT.p, b, y, na, 3);
  NoiseArgs none{PMG_NOISE_NONE, nullptr, 0, 0, 0};
  if (packed) {
    PMG_TRY(launch_rows(*this, b, tmp.p, na)); // v = W b + z
    return launch_cols(*this, tmp.p, y);        // y = W^T v
  }
  PMG_TRY(launch_gemv<true>(ctx, n, L.p, b, tmp.p, na)); // v = W b + z
  return launch_gemv<false>(ctx, n, LT.p, tmp.p, y, none); // y = W^T v
}
int CholSampler::forward(const double *b, double *v)
{
  NoiseArgs none{PMG_NOISE_NONE, nullptr, 0, 0, 0};
  if (!use_gemv) return launch_chol(ctx, n, L.p, LT.p, b, v, none, 1);
  if (packed) return launch_rows(*this, b, v, none);
  return launch_gemv<true>(ctx, n, L.p, b, v, none);
}
int CholSampler::backward_noise(const double *v, double *y, const NoiseArgs &na)
{
  if (!use_gemv) return launch_chol(ctx, n, L.p, LT.p, v, y, na, 2);
  NoiseArgs none{PMG_NOISE_NONE, nullptr, 0, 0, 0};
  if (na.mode != PMG_NOISE_NONE) {
    add_noise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>((int)n, v, tmp.p, na);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    v = tmp.p;
  }
  if (packed) return launch_cols(*this, v, y);
  return launch_gemv<false>(ctx, n, LT.p, v, y, none);
}
