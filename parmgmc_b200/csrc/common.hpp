// common.hpp -- internal types of the B200 sampling library (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h> // header-only; a no-op unless a profiler injects itself

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <utility>
#include <memory>
#include <string>
#include <vector>

#include "../../include/parmgmc_b200.h"

void pmg_set_error(const char *fmt, ...);

#define PMG_CUDA(call)                                                                         \
  do {                                                                                         \
    cudaError_t e_ = (call);                                                                   \
    if (e_ != cudaSuccess) {                                                                   \
      pmg_set_error("%s:%d: CUDA error: %s", __FILE__, __LINE__, cudaGetErrorString(e_));      \
      return PMG_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)

#define PMG_TRY(call)          \
  do {                         \
    int rc_ = (call);          \
    if (rc_) return rc_;       \
  } while (0)

#define PMG_FAIL(code, ...)    \
  do {                         \
    pmg_set_error(__VA_ARGS__); \
    return (code);             \
  } while (0)

// ---- programmatic dependent launch --------------------------------------------------------------------------------
// The kernels of a V-cycle are short and strictly ordered, so launch latency and each kernel's prologue (noise tables,
// mbarriers, work item) sit on the critical path.  A kernel launched with the programmatic-stream-serialization attribute
// may start while its predecessor is still running; it does its prologue, then blocks in pdl_wait() until the predecessor
// has completed and its writes are visible.  Everything a kernel reads or writes that another kernel of the stream
// touches must come after pdl_wait(); pdl_launch_dependents() at the top lets the successor be scheduled early in turn.
// Without the attribute both instructions are no-ops.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
template <class... KA, class... A> inline cudaError_t launch_pdl(cudaStream_t stream, void (*kern)(KA...), dim3 grid, dim3 block, size_t smem, A &&...args)
{
  static const bool off = std::getenv("PMG_NO_PDL") != nullptr;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim          = grid;
  cfg.blockDim         = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream           = stream;
  cudaLaunchAttribute at[1];
  at[0].id                                         = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs    = at;
  cfg.numAttrs = off ? 0 : 1;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<A>(args)...);
}
#endif

// device buffer
template <class T> struct DevBuf {
  T     *p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  DevBuf(DevBuf &&o) noexcept : p(o.p), n(o.n)
  {
    o.p = nullptr;
    o.n = 0;
  }
  DevBuf &operator=(DevBuf &&o) noexcept
  {
    if (this != &o) {
      release();
      p   = o.p;
      n   = o.n;
      o.p = nullptr;
      o.n = 0;
    }
    return *this;
  }
  ~DevBuf() { release(); }
  void release()
  {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  int alloc(size_t count)
  {
    if (count == n && p) return 0;
    release();
    if (count == 0) return 0;
    PMG_CUDA(cudaMalloc((void **)&p, count * sizeof(T)));
    n = count;
    return 0;
  }
  int zero(cudaStream_t s)
  {
    if (n) PMG_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), s));
    return 0;
  }
  int upload(const T *h, size_t count, cudaStream_t s)
  {
    PMG_TRY(alloc(count));
    if (count) PMG_CUDA(cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, s));
    return 0;
  }
  int upload(const std::vector<T> &h, cudaStream_t s) { return upload(h.data(), h.size(), s); }
};

struct pmg_ctx_s {
  int          device     = 0;
  cudaStream_t stream     = nullptr;
  bool         own_stream = false;
  int          sm_count   = 148;
  uint64_t     seed       = 0xCAFE; // examples/ex6.c:131
  uint64_t     draws      = 0;      // global draw (fill) counter: the "position" in the reference's single stream
  void        *nccl_comm  = nullptr;
  int          rank = 0, nranks = 1;
  cudaStream_t comm_stream = nullptr;
  // peer-memory halo exchange (comm.cu): this rank's mailbox, the neighbours' mailboxes mapped through CUDA IPC, and the
  // exchange counters per channel (0: compute stream, 1: communication stream) and side (0: rank-1, 1: rank+1)
  void              *p2p_base    = nullptr;
  void              *p2p_peer[2] = {nullptr, nullptr};
  unsigned long long p2p_seq[2][2] = {{0, 0}, {0, 0}}, p2p_ctas[2] = {0, 0};
  bool               p2p_ok = false;
  // measurement
  int64_t launches = 0, dof_updates = 0;
  // objects created on a context keep it alive: pmg_ctx_destroy only drops the caller's reference
  int refs = 1;
};
// The reference's two PetscLogEvents as NVTX ranges under the same names: "MulticolSOR" around MCSORApply
// (src/mc_sor.c:221,237) and "VecSetRandN" around the generator fill (src/parmgmc.c:76,114; here the fill is fused into the
// sweep kernels, so the range brackets the stand-alone fills only).
struct NvtxRange {
  explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange &) = delete;
  NvtxRange &operator=(const NvtxRange &) = delete;
};
void pmg_ctx_retain(pmg_ctx ctx);
void pmg_ctx_release(pmg_ctx ctx);
void comm_p2p_teardown(pmg_ctx ctx); // comm.cu

// One N(0,1) block: what a single VecSetRandomStandardNormal call (src/parmgmc.c:70-116) produces.
struct NoiseArgs {
  int           mode; // PMG_NOISE_*
  const double *tape; // device pointer to this block (injected mode), indexed by local row
  uint64_t      seed, call;
  int64_t       row0; // global index of local row 0
};

// The global noise stream of one top-level sampler call (SURVEY F7 / 8(c) tape contract).
struct NoiseStream {
  int            mode = PMG_NOISE_PHILOX;
  DevBuf<double> tape;
  int64_t        tape_len = 0, tape_pos = 0;
  NoiseStream   *parent = nullptr; // a sampler nested in another PC (PCWOODBURY) draws from the outer PC's stream
  // next block of n local rows
  int next(pmg_ctx ctx, int64_t n, int64_t row0, NoiseArgs &na)
  {
    if (parent) return parent->next(ctx, n, row0, na);
    na.mode = mode;
    na.tape = nullptr;
    na.seed = ctx->seed;
    na.call = ctx->draws;
    na.row0 = row0;
    if (mode == PMG_NOISE_INJECTED) {
      if (tape_pos + n > tape_len) PMG_FAIL(PMG_ERR_NOISE, "injected noise tape exhausted: need %lld more values at position %lld of %lld", (long long)n, (long long)tape_pos, (long long)tape_len);
      na.tape = tape.p + tape_pos;
      tape_pos += n;
    }
    if (mode != PMG_NOISE_NONE) ctx->draws++;
    return 0;
  }
};

// host CSR (set-up only)
struct HostCsr {
  int64_t              n = 0, m = 0;
  std::vector<int64_t> rowptr;
  std::vector<int32_t> col;
  std::vector<double>  val;
  int64_t nnz() const { return rowptr.empty() ? 0 : rowptr.back(); }
};

// omega-dependent per-row coefficients of a sweep (src/mc_sor.c:114-124, src/pc_mcgibbs.c:142-153)
struct SweepCoeffs {
  double         omega = -1;
  DevBuf<double> idiag, sqrtdiag; // layout is private to the operator that made them ...
  const void    *made_for = nullptr; // ... and to its sweep layout: the operator and its layout version at make_coeffs time
  uint64_t       made_version = 0;
};
uint64_t pmg_next_layout_version(); // process-wide counter: a new value whenever an operator is created or re-coloured

// Low-rank part of an operator A + B diag(S) B^T (MATLRC) and its sweep corrections (lrc.cu).  On a distributed base
// (this rank holds n < nglobal rows) B, Bb and the vectors are this rank's rows; B^T y is folded per rank, the nranks
// k-vectors are all-gathered and summed in rank order, so every rank applies the identical rank-k update.
struct LevelOp;
struct LrcData {
  pmg_ctx             ctx = nullptr;
  int64_t             n   = 0;
  int                 k   = 0, nchunks = 0;
  bool                dist = false;                        // the base is row-distributed: B^T y and B^T C are reduced across ranks
  std::vector<double> Bh, Sh;                             // host copies (set-up)
  DevBuf<double>      B, S, sqrtS, Bb_f, Bb_b, partial, rhs; // n x k column-major; k; k; n x k (forward / backward); chunk sums; n
  DevBuf<double>      bty_all;                            // nranks x k: slot r holds rank r's B^T y (slot 0 only on one rank)
  DevBuf<unsigned>    ticket;                             // chunks of the current B^T y finished (the last one folds and resets it)
  bool                built       = false;
  double              omega_built = 0;
  const void         *built_for = nullptr; // base operator and its layout version the corrections were built with
  uint64_t            built_version = 0;
  int init(pmg_ctx ctx, int64_t n, bool dist, int k, const double *B_host, const double *S_host); // collective when dist
  int build(LevelOp *base, double omega_build);                      // MCSORBuildLRCCorrection, both directions
  int prepare_rhs(const double *b, const NoiseArgs &na_eta, double *out); // out = b + B (sqrt|S| eta)
  int post(int dir, double *y);                                      // y -= Bb_dir (B^T y)
  int post_with(const double *M, double *y);                         // y -= M (B^T y), M dense n x k
  int correction_from(const std::vector<double> &C_host, DevBuf<double> &out); // out = C (S^-1 + B^T C)^-1 (src/mc_sor.c:513-535)
  int add_bsbt(const double *x, double sign, double *out);           // out += sign B (S o B^T x)
  int bty(const double *y);                                          // bty_all = every rank's B^T y (collective when dist)
  int rank_update(const double *M, const double *scale, double sign, double *y); // y += sign M (sum_r bty_all[r] [o scale])
};

// An operator on one level on one device.
struct LevelOp {
  pmg_ctx ctx = nullptr;
  // changes whenever the order / padding of the sweep rows changes (creation, set_coloring*): cached per-row coefficients
  // (SweepCoeffs, the low-rank corrections) are rebuilt when it differs from the one they were made for
  uint64_t layout_version = pmg_next_layout_version();
  // Row stride of this level's V-cycle vectors (b, x) when the cycle keeps them PITCHED (box2d.cuh: a Galerkin level between
  // two one-pass levels); 0: natural layout.  Set by the V-cycle set-up, read by the kernels that write / read the level's
  // vectors from the level above (fused restriction / prolongation).
  int64_t level_pitch = 0;
  virtual ~LevelOp() {}
  virtual int64_t n() const    = 0; // local rows
  virtual int64_t nglobal() const { return n(); }
  virtual int64_t row0() const { return 0; }
  virtual int     ncolors() const                                  = 0;
  virtual int     make_coeffs(double omega, SweepCoeffs &c)        = 0;
  // one directional multicolour sweep of src/mc_sor.c:241-296 on  w = b + sqrtdiag*z  (src/pc_mcgibbs.c:119-128),
  // w never materialised; dir is PMG_SOR_FORWARD_SWEEP or PMG_SOR_BACKWARD_SWEEP; b may be null (b = 0)
  virtual int sweep(int dir, const SweepCoeffs &c, const double *b, double *y, const NoiseArgs &na) = 0;
  virtual int residual(const double *b, const double *x, double *r) = 0; // r = b - A x
  virtual int mult(const double *x, double *y)                      = 0; // y = A x
  virtual const HostCsr *host_csr() { return nullptr; }             // assembled form for set-up, if any
  virtual int  get_coloring(std::vector<int32_t> &color) = 0;
  virtual int  set_coloring(int ncolors, const int32_t *color) = 0;
  virtual int  set_coloring_auto(int policy) = 0;
  virtual void describe(std::string &out) = 0;
  virtual bool structured(int &dim, int64_t dims[3]) const { (void)dim; (void)dims; return false; }
  virtual bool matrix_free() const { return false; } // true: hierarchy is built on the device (stencil_op.cu)
  virtual LrcData *lrc_data() { return nullptr; }    // non-null: the operator is A + B diag(S) B^T and sweeps run on A
  virtual LevelOp *lrc_base() { return nullptr; }    // ... and this is A
  // Fused single-pass sweep (stream2d.cuh), out of place:  xout = sweep_dir(guess) with guess = xin (or 0 when xin is
  // null) plus P xc when xc is given; when bc is given also bc = P^T (b - A xout).  `coarse` supplies the coarse geometry.
  virtual bool fused_ok() const { return false; }
  // Start refreshing the ghost units of the pitched vector v on the communication stream (ordered after everything queued
  // on the compute stream so far); the next fused_sweep whose iterate is v waits for it instead of exchanging itself.
  virtual int halo_begin(double *v) { (void)v; return 0; }
  virtual bool    distributed() const { return false; }  // this rank holds a slab of the level, not the whole level
  virtual int64_t level_first_row() const { return 0; } // first unit of the slowest dimension held by this level's V-cycle vectors
  virtual bool    box2_capable() const { return false; } // a Galerkin level that can run on the one-pass kernels once its vectors are pitched
  virtual int64_t box2_pitch() const { return 0; }
  virtual bool fused_mg_ok() const { return false; } // fused_sweep also does the prolongation / residual + restriction
  virtual bool fused_tape_ok() const { return true; } // fused_sweep can take an injected noise tape
  virtual bool fused_null_xin_ok() const { return true; } // fused_sweep accepts xin = NULL for a zero iterate
  virtual bool pitched_is_natural() const { return false; } // the pitched layout of the fused sweeps equals the natural one
  // slab-distributed finest level of the V-cycle: fused sweeps for the smoothing (one exchange of two ghost units per sweep
  // instead of one per colour), residual and transfers as separate kernels on the pitched vectors
  virtual bool fused_smooth_ok() const { return false; }
  virtual int  residual_pitched(const double *b, const double *x, double *r)
  {
    (void)b; (void)x; (void)r;
    pmg_set_error("pitched residual not available for this operator");
    return PMG_ERR_SUP;
  }
  // One directional sweep in a single out-of-place pass on the level's natural-layout vectors (box_stream.cuh)
  virtual bool stream_ok() const { return false; }
  virtual int  stream_sweep(int dir, const SweepCoeffs &c, const double *b, const double *xin, double *xout, const NoiseArgs &na)
  {
    (void)dir; (void)c; (void)b; (void)xin; (void)xout; (void)na;
    pmg_set_error("streaming sweep not available for this operator");
    return PMG_ERR_SUP;
  }
  // The fused sweeps work on PITCHED copies of the level's vectors (row stride rounded up so that every row starts on a
  // 32-byte boundary): fused_size() elements each; to/from_pitched convert between the natural layout of the API and it.
  virtual int64_t fused_size() const { return n(); }
  virtual int     to_pitched(const double *natural, double *pitched) { (void)natural; (void)pitched; return PMG_ERR_SUP; }
  virtual int     from_pitched(const double *pitched, double *natural) { (void)natural; (void)pitched; return PMG_ERR_SUP; }
  virtual int  fused_sweep(int dir, const SweepCoeffs &c, const double *b, const double *xin, double *xout, const NoiseArgs &na, LevelOp *coarse, const double *xc, double *bc)
  {
    (void)dir; (void)c; (void)b; (void)xin; (void)xout; (void)na; (void)coarse; (void)xc; (void)bc;
    pmg_set_error("fused sweep not available for this operator");
    return PMG_ERR_SUP;
  }
};

// per-sample statistics kept on the device (estimators.cu; examples/benchmark/main.cc:151-175, src/iact.c)
struct QoiState {
  pmg_ctx        ctx = nullptr;
  bool           on = false, welford = false;
  int64_t        n = 0, cap = 0, count = 0, nseen = 0;
  int            nchunks = 0;
  DevBuf<double> meas, trace, partial, mean, M2;
  int init(pmg_ctx ctx, int64_t n, const double *meas_host, int64_t capacity, bool with_mean_var);
  int accumulate(const double *y_dev);
};
int device_autocorrelation(pmg_ctx ctx, int64_t n, const double *x_host, double *acf_host);
int device_iact(pmg_ctx ctx, int64_t n, const double *x_host, double *tau, double *acf_or_null, int *valid);

// work list of the fused 3D sweep (stencil_op.cu), host only
void sweep3d_plan(int64_t n0, int64_t n1, int64_t n2, int64_t slo, int64_t shi, int bz, int nw, bool allow_narrow, int thin_planes, std::vector<int32_t> &out);
void sweep2d_plan(int64_t n0, int64_t n1, int64_t slo, int64_t shi, bool parallel, int by, bool restrict_mode, bool thin_on, std::vector<int32_t> &out, int &nohalo_count);

// grid transfer between level l (fine) and l-1 (coarse): SURVEY Appendix A.3
struct Transfer {
  virtual ~Transfer() {}
  virtual bool tail_ok() const { return false; } // matrix-free Q1 transfer between two whole grids on one device
  // b_c = P^T (b - A x) in one kernel, without storing the residual (same arithmetic as residual + restrict_to)
  virtual bool fused_residual_ok() const { return false; }
  virtual int  restrict_residual(const double *b_fine, const double *x_fine, double *b_coarse)
  {
    (void)b_fine; (void)x_fine; (void)b_coarse;
    pmg_set_error("fused residual + restriction not available for this transfer");
    return PMG_ERR_SUP;
  }
  // the same transfers with the FINE vector in the pitched layout of the fused sweeps (ghost units in place)
  virtual int restrict_pitched(double *r_fine_pitched, double *b_coarse)
  {
    (void)r_fine_pitched; (void)b_coarse;
    pmg_set_error("pitched restriction not available for this transfer");
    return PMG_ERR_SUP;
  }
  virtual int prolong_pitched(const double *x_coarse, double *x_fine_pitched)
  {
    (void)x_coarse; (void)x_fine_pitched;
    pmg_set_error("pitched prolongation not available for this transfer");
    return PMG_ERR_SUP;
  }
  // hooks of the fused transfers (the fine level's kernels write b_coarse / read x_coarse themselves): refresh what other ranks own
  virtual int fused_after_restrict(double *b_coarse) { (void)b_coarse; return 0; }
  virtual int fused_before_prolong(double *x_coarse) { (void)x_coarse; return 0; }
  virtual int restrict_to(const double *r_fine, double *b_coarse) = 0; // b_c = P^T r
  virtual int prolong_add(const double *x_coarse, double *x_fine) = 0; // x_f += P x_c
};

struct pmg_mat_s {
  pmg_ctx                  ctx = nullptr;
  std::unique_ptr<LevelOp> op;
  pmg_mat                  base = nullptr; // low-rank corrected operators borrow their base matrix (MatCreateLRC references A)
  explicit pmg_mat_s(pmg_ctx c) : ctx(c) { pmg_ctx_retain(c); }
  ~pmg_mat_s()
  {
    op.reset();
    pmg_ctx_release(ctx);
  }
};

int comm_exchange_v(pmg_ctx ctx, const double *send, const int64_t *send_off, double *recv, const int64_t *recv_off, cudaStream_t stream);
int comm_allgather_i64(pmg_ctx ctx, const int64_t *local_host, int count, int64_t *all_host);
// row-partitioned CSR operator: this rank's rows [row_start, row_start + n_local) with GLOBAL column indices (csr_op.cu)
int make_csr_dist_op(pmg_ctx ctx, int64_t n_global, int64_t row_start, int64_t n_local, const int64_t *rowptr, const int64_t *col_global, const double *val, std::unique_ptr<LevelOp> &op);
int make_lrc_op(pmg_ctx ctx, LevelOp *base, int k, const double *B_host, const double *S_host, std::unique_ptr<LevelOp> &op); // lrc.cu

// host-side sparse helpers (host_sparse.cpp)
void host_transpose(const HostCsr &a, HostCsr &t);
void host_matmul(const HostCsr &a, const HostCsr &b, HostCsr &c);
void host_q1_dims(int dim, const int64_t nf[3], int64_t nc[3]);
void host_q1_interp(int dim, const int64_t nf[3], const int64_t nc[3], HostCsr &p);
int  host_coloring_greedy(const HostCsr &a, std::vector<int32_t> &color);
int  host_coloring_levelset(const HostCsr &a, std::vector<int32_t> &color);
int64_t host_coloring_violations(const HostCsr &a, const std::vector<int32_t> &color);
int  host_potrf_lower(int64_t n, std::vector<double> &a);

// factories
int make_csr_op(pmg_ctx ctx, HostCsr &&a, std::unique_ptr<LevelOp> &op);
int make_csr_grid_op(pmg_ctx ctx, HostCsr &&a, int dim, const int64_t dims[3], std::unique_ptr<LevelOp> &op); // CSR with known grid
int make_csr_transfer(pmg_ctx ctx, const HostCsr &p, std::unique_ptr<Transfer> &t);

// dense Cholesky sampler (chol.cu): src/pc_chols.c
struct CholChunk { // a run of tiles [t0, t1) of one row panel (v = W b) or column panel (y = W^T v) of the packed triangle
  int panel, t0, t1, q0, nq; // partial sums of the panel: chunks q0 .. q0 + nq - 1 of the list
};
struct CholSampler {
  pmg_ctx        ctx = nullptr;
  int64_t        n   = 0;
  DevBuf<double> L, LT, vcache, tmp;
  bool           use_gemv = true; // false: sequential substitution in dtrsv's order (-pc_cholsampler_b200_solve trsv)
  // n > 4096: factor on the device, W = L^-1 kept as its lower triangle of 64 x 64 tiles (L / LT stay empty, and the
  // one-launch V-cycle tails, which read L / LT as full matrices, are never chosen)
  bool              packed = false;
  int64_t           nt     = 0; // tiles per dimension
  DevBuf<double>    tri, part;  // packed triangle; per-chunk partial sums
  DevBuf<CholChunk> rows, cols; // work lists of the two products
  DevBuf<unsigned>  done;       // per panel: chunks finished (the last one folds the partials and resets it)
  double sample_bytes() const;  // compulsory bytes of one sample (two triangular products)
  int setup(pmg_ctx ctx, const HostCsr &a, const LrcData *lrc = nullptr); // lrc: factor A + B diag(S) B^T (src/pc_chols.c:119-157)
  // y = L^-T (L^-1 b + z)
  int sample(const double *b, double *y, const NoiseArgs &na);
  int forward(const double *b, double *v);                      // v = L^-1 b
  int backward_noise(const double *v, double *y, const NoiseArgs &na); // y = L^-T (v + z)
};

// ---- the coarse tail of a V-cycle in ONE launch (stencil_op.cu grid_tail_kernel) ----------------------------------
// Levels 0 .. nlev-1 of a geometric hierarchy on one device: level 0 is the dense Cholesky sampler, levels >= 1 are
// stencil-array operators smoothed by colour sweeps.  One thread-block cluster runs pre-sampling, residual, restriction,
// the coarse sample, prolongation and post-sampling of all of them with cluster barriers in between, instead of ~11
// launches per level (profiles/: the small levels were pure launch latency).
struct TailNoise {
  uint64_t      call;
  const double *tape;
};
struct TailLevelSpec {
  LevelOp           *op     = nullptr;
  const SweepCoeffs *coeffs = nullptr;
  int                ndirs  = 0;
  int                dirs[8];
  double            *b = nullptr, *x = nullptr, *r = nullptr;
};
bool grid_tail_level_ok(LevelOp *op);
bool grid_tail_smem_fits(int nlev, LevelOp *const *ops, int64_t chol_n); // levels 0 .. nlev-1 fit the one-CTA shared-memory tail (tail2d.cuh)
int  grid_tail_cycle(pmg_ctx ctx, int nlev, const TailLevelSpec *lv, const CholSampler &chol, int noise_mode, uint64_t seed, const TailNoise *ns, int nns);

int launch_normal_fill(pmg_ctx ctx, const NoiseArgs &na, int64_t n, double *z_dev);
// Batched fill of the noise blocks of several 2D levels in ONE launch (csr_op.cu): segment s is the block `call` of an nx x ny
// level whose generator index space is padded to `pitch` columns (philox.cuh); the values land in natural layout (row stride nx)
// and are, bit for bit, the ones the sweep kernels would generate on the fly.
struct PrefillSeg {
  double  *dst;
  int      nx, ny, pitch;
  uint64_t call;
  int64_t  q0; // first quad of the segment in the launch's work list
};
constexpr int PREFILL_MAX = 24;
struct PrefillArgs {
  int        nseg;
  int64_t    total; // quads of all segments
  uint64_t   seed;
  PrefillSeg seg[PREFILL_MAX];
};
int launch_noise_prefill(pmg_ctx ctx, const PrefillArgs &a);
int launch_axpy(pmg_ctx ctx, int64_t n, double a, const double *x, double *y); // y += a x
