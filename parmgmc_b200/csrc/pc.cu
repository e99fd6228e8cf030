// pc.cu -- the C ABI: context, operators, MCSOR engine and the four sampler "PC" types.
//
// Mirrors the reference's plugin surface (SURVEY section 8(b)):
//   src/parmgmc.c      ParMGMCInitialize / global RNG / PCSetSampleCallback  -> pmg_ctx_*, pmg_pc_set_sample_callback
//   src/mc_sor.c       MCSOR*                                                 -> pmg_mcsor_*
//   src/pc_mcgibbs.c   PCMCGIBBS                                              -> pmg_pc type "mcgibbs"
//   src/pc_sorgibbs.c  PCSORGIBBS                                             -> pmg_pc type "sorgibbs"
//   src/pc_gamgmc.c    PCGAMGMC (+ PETSc PCMG cycle, SURVEY Appendix A.3)     -> pmg_pc type "gamgmc"
//   src/pc_chols.c     PCCHOLSAMPLER                                          -> pmg_pc type "cholsampler"
#include <cmath>
#include <cstdlib>
#include <atomic>
#include <map>

#include "common.hpp"

// ---------------------------------------------------------------------------------------------------
static thread_local std::string g_error;

uint64_t pmg_next_layout_version()
{
  static std::atomic<uint64_t> v{1};
  return v.fetch_add(1);
}

void pmg_set_error(const char *fmt, ...)
{
  char    buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_error = buf;
}

// Reports (and clears) a CUDA error left behind by an earlier call whose status nobody looked at, so that
// it is attributed to the right place instead of to the next kernel launch.
static void pmg_stale(const char *where)
{
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) fprintf(stderr, "[parmgmc_b200] stale CUDA error '%s' found on entry to %s\n", cudaGetErrorString(e), where);
}

int make_laplace_op(pmg_ctx ctx, int dim, int64_t nx, int64_t ny, int64_t nz, double kappa, int64_t slab_lo, int64_t slab_hi, std::unique_ptr<LevelOp> &op);
int build_structured_hierarchy(pmg_ctx ctx, LevelOp *fine, int nlevels, int64_t replicate_below, std::vector<std::unique_ptr<LevelOp>> &ops, std::vector<std::unique_ptr<Transfer>> &transfers);

void pmg_ctx_retain(pmg_ctx ctx) { ctx->refs++; }
void pmg_ctx_release(pmg_ctx ctx)
{
  if (--ctx->refs > 0) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->comm_stream) cudaStreamDestroy(ctx->comm_stream);
  comm_p2p_teardown(ctx);
  delete ctx;
}

extern "C" {

const char *pmg_version(void) { return "parmgmc_b200 0.1 (sm_100a)"; }
const char *pmg_last_error(void) { return g_error.c_str(); }

int pmg_device_count(int *count)
{
  pmg_stale("pmg_device_count");
  int         n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    cudaGetLastError();
    n = 0;
  }
  *count = n;
  return PMG_OK;
}

int pmg_ctx_create(int device, pmg_ctx *out)
{
  pmg_stale("pmg_ctx_create");
  int n = 0;
  pmg_device_count(&n);
  if (n == 0) PMG_FAIL(PMG_ERR_NO_DEVICE, "no CUDA device visible: parmgmc_b200 has no CPU fallback");
  if (device < 0 || device >= n) PMG_FAIL(PMG_ERR_ARG, "device %d out of range (0..%d)", device, n - 1);
  PMG_CUDA(cudaSetDevice(device));
  auto *ctx   = new pmg_ctx_s();
  ctx->device = device;
  PMG_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  ctx->own_stream = true;
  cudaDeviceProp prop;
  PMG_CUDA(cudaGetDeviceProperties(&prop, device));
  ctx->sm_count = prop.multiProcessorCount;
  *out          = ctx;
  return PMG_OK;
}

int pmg_ctx_destroy(pmg_ctx ctx)
{
  pmg_stale("pmg_ctx_destroy");
  if (ctx) pmg_ctx_release(ctx);
  return PMG_OK;
}

int pmg_ctx_set_stream(pmg_ctx ctx, void *s)
{
  pmg_stale("pmg_ctx_set_stream");
  if (ctx->own_stream && ctx->stream) {
    cudaStreamSynchronize(ctx->stream);
    cudaStreamDestroy(ctx->stream);
  }
  ctx->stream     = (cudaStream_t)s;
  ctx->own_stream = false;
  return PMG_OK;
}

int pmg_ctx_synchronize(pmg_ctx ctx)
{
  pmg_stale("pmg_ctx_synchronize");
  PMG_CUDA(cudaSetDevice(ctx->device));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return PMG_OK;
}

int pmg_ctx_set_seed(pmg_ctx ctx, uint64_t seed)
{
  pmg_stale("pmg_ctx_set_seed");
  ctx->seed  = seed;
  ctx->draws = 0;
  return PMG_OK;
}
int pmg_ctx_get_draw_counter(pmg_ctx ctx, uint64_t *d)
{
  pmg_stale("pmg_ctx_get_draw_counter");
  *d = ctx->draws;
  return PMG_OK;
}
int pmg_ctx_set_draw_counter(pmg_ctx ctx, uint64_t d)
{
  pmg_stale("pmg_ctx_set_draw_counter");
  ctx->draws = d;
  return PMG_OK;
}

// ---- operators --------------------------------------------------------------------------------------
int pmg_mat_create_csr(pmg_ctx ctx, int64_t n, const int64_t *rowptr, const int32_t *col, const double *val, pmg_mat *out)
{
  pmg_stale("pmg_mat_create_csr");
  if (!ctx || !rowptr || !col || !val || n <= 0) PMG_FAIL(PMG_ERR_ARG, "pmg_mat_create_csr: bad arguments");
  PMG_CUDA(cudaSetDevice(ctx->device));
  HostCsr a;
  a.n = a.m = n;
  a.rowptr.assign(rowptr, rowptr + n + 1);
  if (a.rowptr[0] != 0) PMG_FAIL(PMG_ERR_ARG, "rowptr[0] must be 0");
  a.col.assign(col, col + a.rowptr[n]);
  a.val.assign(val, val + a.rowptr[n]);
  auto m = std::make_unique<pmg_mat_s>(ctx);
  PMG_TRY(make_csr_op(ctx, std::move(a), m->op));
  *out = m.release();
  return PMG_OK;
}

int pmg_mat_create_csr_dist(pmg_ctx ctx, int64_t n_global, int64_t row_start, int64_t n_local, const int64_t *rowptr, const int64_t *col_global, const double *val, pmg_mat *out)
{
  pmg_stale("pmg_mat_create_csr_dist");
  if (!ctx || !rowptr || !col_global || !val || !out) PMG_FAIL(PMG_ERR_ARG, "pmg_mat_create_csr_dist: bad arguments");
  PMG_CUDA(cudaSetDevice(ctx->device));
  auto m = std::make_unique<pmg_mat_s>(ctx);
  PMG_TRY(make_csr_dist_op(ctx, n_global, row_start, n_local, rowptr, col_global, val, m->op));
  *out = m.release();
  return PMG_OK;
}

int pmg_mat_create_laplace(pmg_ctx ctx, int dim, int64_t nx, int64_t ny, int64_t nz, double kappa, int64_t slab_lo, int64_t slab_hi, pmg_mat *out)
{
  pmg_stale("pmg_mat_create_laplace");
  if (!ctx || (dim != 2 && dim != 3) || nx < 2 || ny < 1) PMG_FAIL(PMG_ERR_ARG, "pmg_mat_create_laplace: bad arguments");
  PMG_CUDA(cudaSetDevice(ctx->device));
  auto m = std::make_unique<pmg_mat_s>(ctx);
  PMG_TRY(make_laplace_op(ctx, dim, nx, ny, dim == 3 ? nz : 1, kappa, slab_lo, slab_hi, m->op));
  *out = m.release();
  return PMG_OK;
}

int pmg_mat_create_lrc(pmg_mat A, int k, const double *B_host, const double *S_host, pmg_mat *out)
{
  pmg_stale("pmg_mat_create_lrc");
  if (!A || !B_host || !S_host || !out || k < 1) PMG_FAIL(PMG_ERR_ARG, "pmg_mat_create_lrc: bad arguments");
  PMG_CUDA(cudaSetDevice(A->ctx->device));
  auto m  = std::make_unique<pmg_mat_s>(A->ctx);
  m->base = A;
  PMG_TRY(make_lrc_op(A->ctx, A->op.get(), k, B_host, S_host, m->op));
  *out = m.release();
  return PMG_OK;
}

int pmg_mat_destroy(pmg_mat m)
{
  pmg_stale("pmg_mat_destroy");
  if (m) {
    cudaSetDevice(m->ctx->device);
    delete m;
  }
  return PMG_OK;
}

int pmg_mat_get_size(pmg_mat m, int64_t *nl, int64_t *ng, int64_t *r0)
{
  pmg_stale("pmg_mat_get_size");
  if (nl) *nl = m->op->n();
  if (ng) *ng = m->op->nglobal();
  if (r0) *r0 = m->op->row0();
  return PMG_OK;
}

int pmg_mat_set_coloring(pmg_mat m, int ncolors, const int32_t *color)
{
  pmg_stale("pmg_mat_set_coloring");
  PMG_CUDA(cudaSetDevice(m->ctx->device));
  return m->op->set_coloring(ncolors, color);
}
int pmg_mat_set_coloring_auto(pmg_mat m, int policy)
{
  pmg_stale("pmg_mat_set_coloring_auto");
  PMG_CUDA(cudaSetDevice(m->ctx->device));
  return m->op->set_coloring_auto(policy);
}
int pmg_mat_get_coloring(pmg_mat m, int *ncolors, int32_t *color)
{
  pmg_stale("pmg_mat_get_coloring");
  if (ncolors) *ncolors = m->op->ncolors();
  if (color) {
    std::vector<int32_t> c;
    PMG_TRY(m->op->get_coloring(c));
    std::memcpy(color, c.data(), c.size() * sizeof(int32_t));
  }
  return PMG_OK;
}

int pmg_mat_mult(pmg_mat m, const double *x, double *y)
{
  pmg_stale("pmg_mat_mult");
  pmg_ctx ctx = m->ctx;
  PMG_CUDA(cudaSetDevice(ctx->device));
  const int64_t  n = m->op->n();
  DevBuf<double> dx, dy;
  PMG_TRY(dx.upload(x, (size_t)n, ctx->stream));
  PMG_TRY(dy.alloc((size_t)n));
  PMG_TRY(m->op->mult(dx.p, dy.p));
  PMG_CUDA(cudaMemcpyAsync(y, dy.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return PMG_OK;
}

} // extern "C"

// ---------------------------------------------------------------------------------------------------
// One Gibbs / SOR sampler on one operator: the body of PCApplyRichardson_MulticolorGibbs's loop
// (src/pc_mcgibbs.c:168-182) == PCSORGibbsSample (src/pc_sorgibbs.c:76-103) for omega = 1, forward.
struct GibbsCore {
  LevelOp    *op = nullptr;
  SweepCoeffs coeffs;
  double      omega = 1.0;
  int         type  = PMG_SOR_FORWARD_SWEEP;

  int ensure()
  {
    // omega_changed (src/pc_mcgibbs.c:165), or another operator / another colouring since the coefficients were made: they
    // are stored per padded sweep position of ONE matrix and colouring
    if (coeffs.omega != omega || coeffs.made_for != (const void *)op || coeffs.made_version != op->layout_version) {
      PMG_TRY(op->make_coeffs(omega, coeffs));
      coeffs.made_for     = op;
      coeffs.made_version = op->layout_version;
    }
    return 0;
  }
  // one directional sweep of an operator with a low-rank term: PrepareRHS_LRC (src/pc_mcgibbs.c:130-140: the k extra
  // draws come after the n of the sweep), MCSORApply on the base matrix, MCSORPostSOR_LRC (src/mc_sor.c:101-112)
  int sweep_lrc(LrcData *lrc, NoiseStream &ns, int dir, const double *b, double *y)
  {
    NoiseArgs na, na_eta;
    PMG_TRY(lrc->build(op, lrc_omega_build));
    PMG_TRY(ns.next(op->ctx, op->n(), op->row0(), na));
    PMG_TRY(ns.next(op->ctx, lrc->k, 0, na_eta));
    const double *rhs = b;
    if (na_eta.mode != PMG_NOISE_NONE) {
      PMG_TRY(lrc->prepare_rhs(b, na_eta, lrc->rhs.p));
      rhs = lrc->rhs.p;
    }
    PMG_TRY(op->sweep(dir, coeffs, rhs, y, na));
    return lrc->post(dir, y);
  }
  double lrc_omega_build = 1.0; // the reference builds Bb with a temporary MCSOR at its default omega (src/mc_sor.c:583-593)
  int sample(NoiseStream &ns, const double *b, double *y)
  {
    NvtxRange range("MulticolSOR");
    PMG_TRY(ensure());
    if (LrcData *lrc = op->lrc_data()) {
      if (type == PMG_SOR_SYMMETRIC_SWEEP) {
        PMG_TRY(sweep_lrc(lrc, ns, PMG_SOR_FORWARD_SWEEP, b, y));
        return sweep_lrc(lrc, ns, PMG_SOR_BACKWARD_SWEEP, b, y);
      }
      return sweep_lrc(lrc, ns, type == PMG_SOR_BACKWARD_SWEEP ? PMG_SOR_BACKWARD_SWEEP : PMG_SOR_FORWARD_SWEEP, b, y);
    }
    NoiseArgs na;
    if (type == PMG_SOR_SYMMETRIC_SWEEP) { // forward with fresh noise, then backward with fresh noise (:172-182)
      PMG_TRY(ns.next(op->ctx, op->n(), op->row0(), na));
      PMG_TRY(op->sweep(PMG_SOR_FORWARD_SWEEP, coeffs, b, y, na));
      PMG_TRY(ns.next(op->ctx, op->n(), op->row0(), na));
      PMG_TRY(op->sweep(PMG_SOR_BACKWARD_SWEEP, coeffs, b, y, na));
    } else {
      const int dir = type == PMG_SOR_BACKWARD_SWEEP ? PMG_SOR_BACKWARD_SWEEP : PMG_SOR_FORWARD_SWEEP;
      PMG_TRY(ns.next(op->ctx, op->n(), op->row0(), na));
      PMG_TRY(op->sweep(dir, coeffs, b, y, na));
    }
    return 0;
  }
  int64_t draws_per_sample() const { return (type == PMG_SOR_SYMMETRIC_SWEEP ? 2 : 1) * (op->n() + (op->lrc_data() ? op->lrc_data()->k : 0)); }
};

struct pmg_mcsor_s {
  pmg_ctx        ctx;
  pmg_mat        mat;
  explicit pmg_mcsor_s(pmg_ctx c) : ctx(c) { pmg_ctx_retain(c); }
  ~pmg_mcsor_s()
  {
    core.coeffs = SweepCoeffs();
    b.release();
    y.release();
    pmg_ctx_release(ctx);
  }
  GibbsCore      core;
  NoiseStream    none;
  DevBuf<double> b, y;
};

enum { KIND_SORGIBBS = 0, KIND_MCGIBBS = 1, KIND_CHOL = 2 };

struct LevelSampler {
  int         kind = KIND_SORGIBBS;
  int         its  = 1;
  GibbsCore   gibbs;
  CholSampler chol;
};

struct MgLevel {
  LevelOp                  *op = nullptr;
  std::unique_ptr<LevelOp>  owned;
  std::unique_ptr<LevelOp>  lrc_owned; // A_l + B_l diag(S) B_l^T around `owned` (MATLRC hierarchies)
  std::unique_ptr<Transfer> P; // between this level and the next coarser one
  HostCsr                   interp;
  bool                      has_interp = false;
  LevelSampler              smp;
  DevBuf<double>            b, x, r;
  DevBuf<double>            x2; // second iterate buffer of the fused (out-of-place) sweeps (pitched)
};

struct pmg_pc_s {
  pmg_ctx                            ctx = nullptr;
  std::string                        type;
  pmg_mat                            mat = nullptr;
  std::map<std::string, std::string> opts;
  bool                               is_setup = false;
  NoiseStream                        noise;
  pmg_sample_cb                      cb      = nullptr;
  void                              *cbctx   = nullptr;
  pmg_ctx_deleter                    deleter = nullptr;
  int64_t                            sample_index = 0;
  LevelSampler                       smp; // mcgibbs / sorgibbs / cholsampler
  // gamgmc
  int                  nlevels = 0;
  std::vector<MgLevel> lv;
  DevBuf<double>       w, work;
  bool                 direct_cycle = true; // cycle applied to (b, y) directly instead of y += MG(b - A y); same map, fewer passes
  // Opt-in (PMG_PREFILL=1; measured slower, see prefill_wanted): noise of the 9-point levels ahead of their sweeps (one device,
  // Philox).  ONE batched launch at the start of a sample writes the normals of all their sweeps (launch_noise_prefill: the
  // same values, bit for bit) and the sweeps read them as a tape.  The blocks a
  // sample draws, and their order, are fixed by the hierarchy: the first sample records (level, pre/post, sweep) -> offset of
  // the draw counter, the following ones use the record and check it draw by draw.
  struct NoisePrefill {
    struct Entry {
      int            level, post, s;
      int64_t        k; // draw counter of the block minus the draw counter at the start of the sample
      int            nx, ny, pitch;
      DevBuf<double> buf;
    };
    std::vector<Entry> entries;
    bool               recorded = false, recording = false, active = false;
    uint64_t           draws0 = 0;
    size_t             cursor = 0;
    void               reset() { entries.clear(); recorded = recording = active = false; cursor = 0; }
  } prefill;
  int                  tail_top     = -1;   // levels 0 .. tail_top of the direct cycle run in one launch (mg_tail); -1: none
  // PCWOODBURY (src/woodbury.c): a sampler on the base matrix A of a MATLRC operator + the correction G
  pmg_pc               wb_sampler = nullptr;
  DevBuf<double>       wb_G;
  QoiState             qoi; // device-side SaveSample (examples/benchmark/main.cc:151-175)
  DevBuf<double>       scratch;             // out-of-place partner of the iterate for the fused sweeps (pitched)
  DevBuf<double>       pit_y, pit_b;        // pitched copies of the caller's y and b (LevelOp::fused_size)
  // staging
  DevBuf<double> d_b, d_y;
  double        *h_pinned = nullptr;
  cudaEvent_t    ev0 = nullptr, ev1 = nullptr;
  double         last_ms = 0;
  int64_t        last_launches = 0, last_updates = 0;
  // per-kernel profile of the V-cycle (-pc_b200_profile): CUDA events around every labelled launch on the launching stream
  struct ProfRec {
    std::string label;
    double      bytes_min, bytes_survey; // compulsory traffic of the fused kernel; sum of SURVEY 8(d)'s per-unit figures it replaces
    cudaEvent_t e0, e1;
  };
  struct ProfSum {
    double  ms = 0, bytes_min = 0, bytes_survey = 0;
    int64_t launches = 0;
  };
  bool                           prof_on = false;
  std::vector<ProfRec>           prof_pending;
  std::map<std::string, ProfSum> prof_sum;
  std::vector<std::string>       prof_order;

  explicit pmg_pc_s(pmg_ctx c) : ctx(c) { pmg_ctx_retain(c); }
  ~pmg_pc_s()
  {
    delete wb_sampler;
    wb_G.release();
    if (deleter) deleter(cbctx);
    if (h_pinned) cudaFreeHost(h_pinned);
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    lv.clear();
    smp = LevelSampler();
    noise.tape.release();
    w.release(); work.release(); d_b.release(); d_y.release(); scratch.release(); pit_y.release(); pit_b.release();
    pmg_ctx_release(ctx);
  }
  bool        has(const std::string &k) const { return opts.count(k) != 0; }
  std::string get(const std::string &k, const std::string &d) const
  {
    auto it = opts.find(k);
    return it == opts.end() ? d : it->second;
  }
};

static bool opt_true(const std::string &v) { return v.empty() || v == "1" || v == "true" || v == "yes" || v == "on" || v == "TRUE"; }

// PCSetFromOptions_MulticolorGibbs (src/pc_mcgibbs.c:190-211) / _SORGibbs (src/pc_sorgibbs.c:264-278) for the
// sampler configured under `prefix` ("" for a stand-alone PC, "gamgmc_mg_levels_" / "gamgmc_mg_coarse_" inside MG)
// the mode of the stream a PC really draws from (a sampler nested in PCWOODBURY draws from the outer PC's stream)
static int noise_mode(pmg_pc pc)
{
  const NoiseStream *ns = &pc->noise;
  while (ns->parent) ns = ns->parent;
  return ns->mode;
}

// ---- per-kernel profile ----
static int prof_begin(pmg_pc pc, const std::string &label, double bytes_min, double bytes_survey)
{
  if (!pc->prof_on) return 0;
  pmg_pc_s::ProfRec r;
  r.label = label; r.bytes_min = bytes_min; r.bytes_survey = bytes_survey;
  PMG_CUDA(cudaEventCreate(&r.e0));
  PMG_CUDA(cudaEventCreate(&r.e1));
  PMG_CUDA(cudaEventRecord(r.e0, pc->ctx->stream));
  pc->prof_pending.push_back(r);
  return 0;
}
static int prof_end(pmg_pc pc)
{
  if (!pc->prof_on || pc->prof_pending.empty()) return 0;
  PMG_CUDA(cudaEventRecord(pc->prof_pending.back().e1, pc->ctx->stream));
  return 0;
}
static int prof_collect(pmg_pc pc)
{
  if (pc->prof_pending.empty()) return 0;
  PMG_CUDA(cudaStreamSynchronize(pc->ctx->stream));
  for (auto &r : pc->prof_pending) {
    float ms = 0;
    PMG_CUDA(cudaEventElapsedTime(&ms, r.e0, r.e1));
    if (!pc->prof_sum.count(r.label)) pc->prof_order.push_back(r.label);
    auto &a = pc->prof_sum[r.label];
    a.ms += ms; a.bytes_min += r.bytes_min; a.bytes_survey += r.bytes_survey; a.launches++;
    cudaEventDestroy(r.e0);
    cudaEventDestroy(r.e1);
  }
  pc->prof_pending.clear();
  return 0;
}

static int configure_sampler(pmg_pc pc, const std::string &prefix, const std::string &pctype, LevelSampler &s)
{
  if (pctype == "mcgibbs") {
    s.kind = KIND_MCGIBBS;
    if (pc->has(prefix + "pc_mcgibbs_omega")) s.gibbs.omega = std::atof(pc->get(prefix + "pc_mcgibbs_omega", "1").c_str());
    if (!(s.gibbs.omega > 0 && s.gibbs.omega < 2)) PMG_FAIL(PMG_ERR_ARG, "-%spc_mcgibbs_omega must be in (0,2)", prefix.c_str());
    if (pc->has(prefix + "pc_mcgibbs_forward") && opt_true(pc->get(prefix + "pc_mcgibbs_forward", ""))) s.gibbs.type = PMG_SOR_FORWARD_SWEEP;
    if (pc->has(prefix + "pc_mcgibbs_backward") && opt_true(pc->get(prefix + "pc_mcgibbs_backward", ""))) s.gibbs.type = PMG_SOR_BACKWARD_SWEEP;
    if (pc->has(prefix + "pc_mcgibbs_symmetric") && opt_true(pc->get(prefix + "pc_mcgibbs_symmetric", ""))) s.gibbs.type = PMG_SOR_SYMMETRIC_SWEEP;
  } else if (pctype == "sorgibbs") {
    s.kind        = KIND_SORGIBBS;
    s.gibbs.omega = 1.0; // no omega option (SURVEY F6)
    s.gibbs.type  = PMG_SOR_FORWARD_SWEEP; // forward and local_forward coincide on one device
  } else if (pctype == "cholsampler") {
    s.kind = KIND_CHOL;
    const std::string solve = pc->get(prefix + "pc_cholsampler_b200_solve", pc->get("pc_cholsampler_b200_solve", "gemv"));
    if (solve != "gemv" && solve != "trsv") PMG_FAIL(PMG_ERR_ARG, "-pc_cholsampler_b200_solve %s: expected gemv | trsv", solve.c_str());
    s.chol.use_gemv = solve == "gemv";
  } else PMG_FAIL(PMG_ERR_SUP, "sampler type '%s' is not supported (mcgibbs | sorgibbs | cholsampler)", pctype.c_str());
  return 0;
}

static int apply_coloring_policy(pmg_pc pc, LevelOp *op, bool is_user_mat)
{
  const std::string p = pc->get("pc_b200_coloring", "");
  if (p.empty() || p == "keep") return 0; // user matrices keep whatever colouring they carry
  (void)is_user_mat;
  if (p == "greedy") return op->set_coloring_auto(PMG_COLORING_GREEDY);
  if (p == "lexicographic") return op->set_coloring_auto(PMG_COLORING_LEXICOGRAPHIC);
  if (p == "parity") return op->set_coloring_auto(PMG_COLORING_PARITY);
  PMG_FAIL(PMG_ERR_ARG, "-pc_b200_coloring %s: expected greedy | lexicographic | parity | keep", p.c_str());
}

static int setup_level_sampler(pmg_ctx ctx, LevelSampler &s, LevelOp *op)
{
  if (s.kind == KIND_CHOL) {
    if (op->lrc_data() && op->lrc_data()->dist) PMG_FAIL(PMG_ERR_SUP, "cholsampler on a low-rank corrected operator with a row-distributed base is not supported: the exact sampler factors the whole operator on one device");
    const HostCsr *a = op->lrc_base() ? op->lrc_base()->host_csr() : op->host_csr();
    if (!a) PMG_FAIL(PMG_ERR_SUP, "cholsampler needs an assembled operator");
    return s.chol.setup(ctx, *a, op->lrc_data());
  }
  s.gibbs.op = op;
  return s.gibbs.ensure();
}

// KSP(richardson, max_it = its) around a level sampler.  Continues from x (the reference samplers ignore
// guesszero, src/pc_sorgibbs.c:94 / src/pc_mcgibbs.c:170).
static int run_level_sampler(pmg_pc pc, LevelSampler &s, const double *b, double *x)
{
  if (s.kind == KIND_CHOL) {
    NoiseArgs na;
    if (s.its == 1) { // src/pc_chols.c:303-304 -> PCApply_CholSampler :262-291
      PMG_TRY(pc->noise.next(pc->ctx, s.chol.n, 0, na));
      return s.chol.sample(b, x, na);
    }
    PMG_TRY(s.chol.forward(b, s.chol.vcache.p)); // forward solve cached (:306-336)
    for (int it = 0; it < s.its; ++it) {
      PMG_TRY(pc->noise.next(pc->ctx, s.chol.n, 0, na));
      PMG_TRY(s.chol.backward_noise(s.chol.vcache.p, x, na));
    }
    return 0;
  }
  for (int it = 0; it < s.its; ++it) PMG_TRY(s.gibbs.sample(pc->noise, b, x));
  return 0;
}

static int64_t sampler_draws(const LevelSampler &s)
{
  if (s.kind == KIND_CHOL) return s.its * s.chol.n;
  return s.its * s.gibbs.draws_per_sample();
}

// PCMGMCycle_Private, V-cycle (SURVEY Appendix A.3)
static int mg_cycle(pmg_pc pc, int l, const double *b, double *x)
{
  MgLevel &v = pc->lv[l];
  PMG_TRY(run_level_sampler(pc, v.smp, b, x));
  if (l == 0) return 0;
  MgLevel &c = pc->lv[l - 1];
  PMG_TRY(v.op->residual(b, x, v.r.p));
  PMG_TRY(v.P->restrict_to(v.r.p, c.b.p));
  PMG_TRY(c.x.zero(pc->ctx->stream));
  PMG_TRY(mg_cycle(pc, l - 1, c.b.p, c.x.p));
  PMG_TRY(v.P->prolong_add(c.x.p, x));
  return run_level_sampler(pc, v.smp, b, x);
}

// PCApply_MG: x = 0, one cycle
static int mg_apply(pmg_pc pc, const double *b, double *x)
{
  const int64_t n = pc->lv[pc->nlevels - 1].op->n();
  PMG_CUDA(cudaMemsetAsync(x, 0, (size_t)n * sizeof(double), pc->ctx->stream));
  return mg_cycle(pc, pc->nlevels - 1, b, x);
}

// the directional sweeps one level-KSP solve performs, with a fresh noise block each (src/pc_mcgibbs.c:168-182)
static int sweep_dirs(const LevelSampler &s, std::vector<int> &dirs)
{
  dirs.clear();
  for (int it = 0; it < s.its; ++it) {
    if (s.gibbs.type == PMG_SOR_SYMMETRIC_SWEEP) {
      dirs.push_back(PMG_SOR_FORWARD_SWEEP);
      dirs.push_back(PMG_SOR_BACKWARD_SWEEP);
    } else dirs.push_back(s.gibbs.type == PMG_SOR_BACKWARD_SWEEP ? PMG_SOR_BACKWARD_SWEEP : PMG_SOR_FORWARD_SWEEP);
  }
  return 0;
}

// The same V-cycle applied directly to (b, x): because every stage is affine in (b, x) and acts on the residual,
// cycle(b, x) == x + cycle(b - A x, 0) (SURVEY section 7, hard part 8), so the outer w = b - A y / y += work passes of
// src/pc_gamgmc.c:253-256 disappear.  Levels whose operator has a fused streaming sweep run pre-smoothing + residual +
// restriction in one pass over memory and prolongation + post-smoothing in another; on such a level b and x are the
// PITCHED vectors of LevelOp::fused_size() elements (only the finest level can be one: the caller converts).
static int mg_tail(pmg_pc pc, int lt);

// ---- noise of the 9-point levels ahead of their sweeps (pmg_pc_s::NoisePrefill) --------------------------------------------
static bool prefill_wanted(pmg_pc pc)
{
  // opt-in (PMG_PREFILL=1): measured SLOWER on B200 (4097^2: 0.474 against 0.445 ms per sample) -- the generator work is the same and
  // in the sweeps it rides in issue slots that the dependent FP64 chain leaves empty anyway, while the batched launch costs
  // ~25 us of its own; kept as a tested path because it turns any device-generated sample into a replayable tape
  return pc->noise.mode == PMG_NOISE_PHILOX && !pc->noise.parent && pc->ctx->nranks == 1 && std::getenv("PMG_PREFILL") != nullptr;
}
static int prefill_begin(pmg_pc pc)
{
  auto &pf = pc->prefill;
  pf.active = pf.recording = false;
  if (!prefill_wanted(pc)) return 0;
  pf.draws0 = pc->ctx->draws;
  pf.cursor = 0;
  if (!pf.recorded) {
    pf.entries.clear();
    pf.recording = true;
    return 0;
  }
  if (pf.entries.empty()) return 0;
  PrefillArgs a;
  std::memset(&a, 0, sizeof a);
  a.seed = pc->ctx->seed;
  for (auto &e : pf.entries) {
    PrefillSeg &sg = a.seg[a.nseg++];
    sg.dst = e.buf.p; sg.nx = e.nx; sg.ny = e.ny; sg.pitch = e.pitch;
    sg.call = pf.draws0 + (uint64_t)e.k;
    sg.q0   = a.total;
    a.total += (int64_t)(e.pitch >> 2) * e.ny;
  }
  PMG_TRY(prof_begin(pc, "noise of the 9-point levels (one launch)", 8.0 * (double)a.total * 4, 0.0));
  PMG_TRY(launch_noise_prefill(pc->ctx, a));
  PMG_TRY(prof_end(pc));
  pf.active = true;
  return 0;
}
// after noise.next() of sweep s (pre: post = 0, post-smoothing: 1) of level l: record the block, or hand the sweep its tape
static int prefill_hook(pmg_pc pc, int l, int post, int s, LevelOp *op, NoiseArgs &na)
{
  auto &pf = pc->prefill;
  if (pf.recording) {
    int     dim;
    int64_t dims[3];
    if (na.mode != PMG_NOISE_PHILOX || !op->level_pitch || !op->structured(dim, dims) || dim != 2 || (int)pf.entries.size() >= PREFILL_MAX) return 0;
    pmg_pc_s::NoisePrefill::Entry e;
    e.level = l; e.post = post; e.s = s;
    e.k  = (int64_t)(na.call - pf.draws0);
    e.nx = (int)dims[0]; e.ny = (int)dims[1]; e.pitch = (int)op->level_pitch;
    pf.entries.push_back(std::move(e));
    return 0;
  }
  if (!pf.active) return 0;
  if (pf.cursor < pf.entries.size()) {
    auto &e = pf.entries[pf.cursor];
    if (e.level == l && e.post == post && e.s == s && na.call == pf.draws0 + (uint64_t)e.k && na.mode == PMG_NOISE_PHILOX) {
      ++pf.cursor;
      na.mode = PMG_NOISE_INJECTED;
      na.tape = e.buf.p;
      return 0;
    }
  }
  PMG_FAIL(PMG_ERR_NOISE, "gamgmc: the noise blocks of this sample are not the recorded ones (level %d, %s sweep %d): the hierarchy changed without pmg_pc_setup", l, post ? "post" : "pre", s);
}
static int prefill_end(pmg_pc pc)
{
  auto &pf = pc->prefill;
  if (pf.recording) {
    pf.recording = false;
    for (auto &e : pf.entries) PMG_TRY(e.buf.alloc((size_t)e.nx * (size_t)e.ny));
    pf.recorded = true;
  } else if (pf.active && pf.cursor != pf.entries.size()) {
    pf.active = false;
    PMG_FAIL(PMG_ERR_NOISE, "gamgmc: %zu of the %zu prefilled noise blocks were not consumed", pf.entries.size() - pf.cursor, pf.entries.size());
  }
  pf.active = false;
  return 0;
}

static int mg_cycle_direct(pmg_pc pc, int l, const double *b, double *x, bool zero_guess)
{
  pmg_ctx  ctx = pc->ctx;
  MgLevel &v   = pc->lv[l];
  if (l == pc->tail_top && zero_guess && b == v.b.p && x == v.x.p) { // levels 0..l in one launch
    PMG_TRY(prof_begin(pc, "L0-L" + std::to_string(l) + " coarse tail (one launch)", 0, 0));
    PMG_TRY(mg_tail(pc, l));
    return prof_end(pc);
  }
  const bool fused = l > 0 && v.smp.kind != KIND_CHOL && v.op->fused_mg_ok() && v.x2.p && !(v.op->distributed() && pc->lv[l - 1].op->distributed() && !pc->lv[l - 1].op->level_pitch);
  // stencil-array levels: each directional sweep is one out-of-place pass (box_stream.cuh); the level's iterate
  // ping-pongs between v.x and v.x2, so the current one is always v.x.p
  const bool bstream = !fused && l > 0 && v.smp.kind != KIND_CHOL && v.x2.p && x == v.x.p && v.op->stream_ok() &&
                       (noise_mode(pc) != PMG_NOISE_INJECTED || v.op->fused_tape_ok());
  if (!fused && l > 0 && pc->lv[l - 1].op->level_pitch) PMG_FAIL(PMG_ERR_ORDER, "gamgmc: level %d keeps pitched vectors but level %d does not run the fused kernels (path switches must be set before pmg_pc_setup)", l - 1, l);
  if (bstream) {
    MgLevel         &c = pc->lv[l - 1];
    std::vector<int> dirs;
    sweep_dirs(v.smp, dirs);
    PMG_TRY(v.smp.gibbs.ensure());
    NoiseArgs na;
    auto      smooth = [&]() -> int {
      for (int d : dirs) {
        PMG_TRY(pc->noise.next(ctx, v.op->n(), v.op->row0(), na));
        { NvtxRange range("MulticolSOR"); PMG_TRY(v.op->stream_sweep(d, v.smp.gibbs.coeffs, b, v.x.p, v.x2.p, na)); }
        std::swap(v.x, v.x2);
      }
      return 0;
    };
    if (zero_guess) PMG_CUDA(cudaMemsetAsync(v.x.p, 0, (size_t)v.op->n() * sizeof(double), ctx->stream));
    PMG_TRY(smooth());
    if (v.P->fused_residual_ok() && !v.op->lrc_data()) PMG_TRY(v.P->restrict_residual(b, v.x.p, c.b.p));
    else {
      PMG_TRY(v.op->residual(b, v.x.p, v.r.p));
      PMG_TRY(v.P->restrict_to(v.r.p, c.b.p));
    }
    PMG_TRY(mg_cycle_direct(pc, l - 1, c.b.p, c.x.p, true));
    PMG_TRY(v.P->prolong_add(pc->lv[l - 1].x.p, v.x.p));
    return smooth();
  }
  // slab-distributed finest level: fused sweeps on the pitched vectors (one ghost exchange per sweep), pitched residual / transfers
  if (!fused && l > 0 && l == pc->nlevels - 1 && v.smp.kind != KIND_CHOL && v.op->fused_smooth_ok() && v.x2.p && x == pc->pit_y.p) {
    MgLevel         &c = pc->lv[l - 1];
    std::vector<int> dirs;
    sweep_dirs(v.smp, dirs);
    PMG_TRY(v.smp.gibbs.ensure());
    double   *cur = x, *oth = v.x2.p;
    NoiseArgs na;
    auto      smooth = [&]() -> int {
      for (int d : dirs) {
        PMG_TRY(pc->noise.next(ctx, v.op->n(), v.op->row0(), na));
        { NvtxRange range("MulticolSOR"); PMG_TRY(v.op->fused_sweep(d, v.smp.gibbs.coeffs, b, cur, oth, na, nullptr, nullptr, nullptr)); }
        std::swap(cur, oth);
      }
      return 0;
    };
    if (zero_guess) PMG_CUDA(cudaMemsetAsync(cur, 0, (size_t)v.op->fused_size() * sizeof(double), ctx->stream));
    PMG_TRY(smooth());
    PMG_TRY(v.op->residual_pitched(b, cur, v.r.p));
    PMG_TRY(v.P->restrict_pitched(v.r.p, c.b.p));
    PMG_TRY(mg_cycle_direct(pc, l - 1, c.b.p, c.x.p, true));
    PMG_TRY(v.P->prolong_pitched(c.x.p, cur));
    PMG_TRY(smooth());
    if (cur != x) PMG_CUDA(cudaMemcpyAsync(x, cur, (size_t)v.op->fused_size() * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    return 0;
  }
  if (!fused) {
    if (zero_guess) PMG_CUDA(cudaMemsetAsync(x, 0, (size_t)v.op->n() * sizeof(double), ctx->stream));
    if (l == 0 && v.smp.kind == KIND_CHOL) PMG_TRY(prof_begin(pc, "L0 dense Cholesky sample", v.smp.chol.sample_bytes(), v.smp.chol.sample_bytes()));
    PMG_TRY(run_level_sampler(pc, v.smp, b, x));
    if (l == 0) return prof_end(pc);
    MgLevel &c = pc->lv[l - 1];
    if (v.P->fused_residual_ok() && !v.op->lrc_data()) PMG_TRY(v.P->restrict_residual(b, x, c.b.p));
    else {
      PMG_TRY(v.op->residual(b, x, v.r.p));
      PMG_TRY(v.P->restrict_to(v.r.p, c.b.p));
    }
    PMG_TRY(mg_cycle_direct(pc, l - 1, c.b.p, c.x.p, true));
    PMG_TRY(v.P->prolong_add(pc->lv[l - 1].x.p, x));
    return run_level_sampler(pc, v.smp, b, x);
  }
  MgLevel         &c = pc->lv[l - 1];
  std::vector<int> dirs;
  sweep_dirs(v.smp, dirs);
  PMG_TRY(v.smp.gibbs.ensure());
  double   *cur = x, *oth = v.x2.p;
  NoiseArgs na;
  for (size_t s = 0; s < dirs.size(); ++s) { // pre-smoothing; the last sweep also forms the coarse right-hand side
    const bool last = s + 1 == dirs.size();
    PMG_TRY(pc->noise.next(ctx, v.op->n(), v.op->row0(), na));
    if (l < pc->nlevels - 1) PMG_TRY(prefill_hook(pc, l, 0, (int)s, v.op, na));
    const double *xin = (zero_guess && s == 0) ? nullptr : cur;
    if (!xin && !v.op->fused_null_xin_ok()) { // the 3D sweep reads its iterate through the TMA: hand it zeros
      PMG_CUDA(cudaMemsetAsync(cur, 0, (size_t)v.op->fused_size() * sizeof(double), ctx->stream));
      xin = cur;
    }
    if (pc->prof_on) {
      // bytes per DOF: compulsory traffic of this pass (b, x in unless zero, x out, b_c out) | SURVEY 8(d): K1 (24 at omega = 1, else 32) [+ K3 24 + K4 10]
      const double nn = (double)v.op->n(), k1 = v.smp.gibbs.omega == 1.0 ? 24.0 : 32.0;
      PMG_TRY(prof_begin(pc, "L" + std::to_string(l) + (last ? " pre-sample+residual+restrict" : " sweep"), nn * ((b ? 8 : 0) + (xin ? 8 : 0) + 8 + (last ? 2 : 0)), nn * (k1 + (last ? 34 : 0))));
    }
    { NvtxRange range("MulticolSOR"); PMG_TRY(v.op->fused_sweep(dirs[s], v.smp.gibbs.coeffs, b, xin, oth, na, c.op, nullptr, last ? c.b.p : nullptr)); }
    PMG_TRY(prof_end(pc));
    std::swap(cur, oth);
  }
  PMG_TRY(v.P->fused_after_restrict(c.b.p)); // slabs: ghost rows of the coarse right-hand side (or the gather of a replicated level)
  PMG_TRY(v.op->halo_begin(cur));            // slabs: the post-smoother's ghost rows travel (communication stream) while the coarse levels work
  PMG_TRY(mg_cycle_direct(pc, l - 1, c.b.p, c.x.p, true));
  PMG_TRY(v.P->fused_before_prolong(c.x.p));
  for (size_t s = 0; s < dirs.size(); ++s) { // post-smoothing; the first sweep starts from x + P x_c
    PMG_TRY(pc->noise.next(ctx, v.op->n(), v.op->row0(), na));
    if (l < pc->nlevels - 1) PMG_TRY(prefill_hook(pc, l, 1, (int)s, v.op, na));
    if (pc->prof_on) { // K5 (18) + K1
      const double nn = (double)v.op->n(), k1 = v.smp.gibbs.omega == 1.0 ? 24.0 : 32.0;
      PMG_TRY(prof_begin(pc, "L" + std::to_string(l) + (s == 0 ? " prolong+post-sample" : " sweep"), nn * ((b ? 8 : 0) + 8 + 8 + (s == 0 ? 2 : 0)), nn * (k1 + (s == 0 ? 18 : 0))));
    }
    { NvtxRange range("MulticolSOR"); PMG_TRY(v.op->fused_sweep(dirs[s], v.smp.gibbs.coeffs, b, cur, oth, na, c.op, s == 0 ? pc->lv[l - 1].x.p : nullptr, nullptr)); }
    PMG_TRY(prof_end(pc));
    std::swap(cur, oth);
  }
  if (cur != x) PMG_CUDA(cudaMemcpyAsync(x, cur, (size_t)v.op->fused_size() * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  return 0;
}

// Levels 0 .. lt of the V-cycle in one cluster launch (stencil_op.cu grid_tail_kernel).  The noise blocks are handed out
// here in the order the level-by-level path draws them, so counters, tapes and results do not depend on the choice.
static int mg_tail(pmg_pc pc, int lt)
{
  pmg_ctx                    ctx = pc->ctx;
  std::vector<TailLevelSpec> lv((size_t)lt + 1);
  std::vector<TailNoise>     ns;
  NoiseArgs                  na;
  for (int l = 0; l <= lt; ++l) {
    MgLevel &v = pc->lv[l];
    lv[l].op = v.op;
    lv[l].b = v.b.p; lv[l].x = v.x.p; lv[l].r = v.r.p;
    if (l == 0) continue;
    PMG_TRY(v.smp.gibbs.ensure());
    lv[l].coeffs = &v.smp.gibbs.coeffs;
    std::vector<int> dirs;
    sweep_dirs(v.smp, dirs);
    lv[l].ndirs = (int)dirs.size();
    for (size_t q = 0; q < dirs.size(); ++q) lv[l].dirs[q] = dirs[q];
  }
  for (int l = lt; l >= 1; --l)
    for (int q = 0; q < lv[l].ndirs; ++q) {
      PMG_TRY(pc->noise.next(ctx, pc->lv[l].op->n(), 0, na));
      ns.push_back(TailNoise{na.call, na.tape});
    }
  PMG_TRY(pc->noise.next(ctx, pc->lv[0].smp.chol.n, 0, na));
  ns.push_back(TailNoise{na.call, na.tape});
  for (int l = 1; l <= lt; ++l)
    for (int q = 0; q < lv[l].ndirs; ++q) {
      PMG_TRY(pc->noise.next(ctx, pc->lv[l].op->n(), 0, na));
      ns.push_back(TailNoise{na.call, na.tape});
    }
  return grid_tail_cycle(ctx, lt + 1, lv.data(), pc->lv[0].smp.chol, noise_mode(pc), ctx->seed, ns.data(), (int)ns.size());
}

static int gamgmc_setup(pmg_pc pc)
{
  pmg_ctx  ctx  = pc->ctx;
  pc->prefill.reset();
  LevelOp *top  = pc->mat->op.get();                      // what the user handed over (possibly A + B S B^T)
  LevelOp *fine = top->lrc_base() ? top->lrc_base() : top; // the hierarchy is built from the base matrix (src/pc_gamgmc.c:296-353)
  // -pc_gamgmc_mg_type (src/pc_gamgmc.c:364): only the geometric hierarchy can be built without PETSc's GAMG
  const std::string mgtype = pc->get("pc_gamgmc_mg_type", "mg");
  bool              user_p = false;
  for (auto &l : pc->lv) user_p |= l.has_interp;
  if (mgtype != "mg" && !user_p) PMG_FAIL(PMG_ERR_SUP, "-pc_gamgmc_mg_type %s: algebraic (GAMG) coarsening is PETSc-internal and not reproduced; use 'mg' on a structured operator or supply interpolations", mgtype.c_str());
  int L = pc->nlevels;
  if (pc->has("gamgmc_pc_mg_levels")) L = std::atoi(pc->get("gamgmc_pc_mg_levels", "0").c_str());
  int     dim = 0;
  int64_t dims[3] = {0, 0, 0};
  bool structured = fine->structured(dim, dims);
  if (!structured && pc->has("pc_b200_grid")) { // the grid of an assembled operator (what PCSetDM tells the reference, src/pc_gamgmc.c:290-294)
    long long g[3] = {1, 1, 1};
    const int k    = std::sscanf(pc->get("pc_b200_grid", "").c_str(), "%lld,%lld,%lld", &g[0], &g[1], &g[2]);
    if (k < 2 || g[0] * g[1] * g[2] != fine->n()) PMG_FAIL(PMG_ERR_ARG, "-pc_b200_grid nx,ny[,nz]: must multiply to the operator size %lld", (long long)fine->n());
    dim = k;
    for (int q = 0; q < 3; ++q) dims[q] = g[q];
    structured = true;
  }
  if (L <= 0) { // automatic depth: coarsen until the coarsest grid is at most 17 nodes per direction
    if (!structured) PMG_FAIL(PMG_ERR_ORDER, "gamgmc: set the number of levels (-gamgmc_pc_mg_levels / pmg_pc_gamgmc_set_levels)");
    L = 1;
    int64_t d[3] = {dims[0], dims[1], dims[2]};
    while (std::max(d[0], std::max(d[1], d[2])) > 17 && L < 30) {
      int64_t c[3];
      host_q1_dims(dim, d, c);
      std::memcpy(d, c, sizeof d);
      ++L;
    }
  }
  if (L < 1) PMG_FAIL(PMG_ERR_ARG, "gamgmc: need at least one level");
  std::vector<MgLevel> old = std::move(pc->lv);
  pc->lv.clear();
  pc->lv.resize((size_t)L);
  for (int l = 0; l < L && l < (int)old.size(); ++l)
    if (old[l].has_interp) {
      pc->lv[l].interp     = std::move(old[l].interp);
      pc->lv[l].has_interp = true;
    }
  pc->nlevels      = L;
  pc->lv[L - 1].op = fine;
  PMG_TRY(apply_coloring_policy(pc, fine, true));

  bool all_user = L > 1;
  for (int l = 1; l < L; ++l) all_user &= pc->lv[l].has_interp;
  if (L > 1 && !all_user && !structured) PMG_FAIL(PMG_ERR_SUP, "gamgmc: operator is not structured; supply an interpolation for every level 1..%d", L - 1);

  if (L > 1 && !all_user && structured && fine->matrix_free()) {
    // matrix-free structured hierarchy built on the device
    std::vector<std::unique_ptr<LevelOp>>  ops;
    std::vector<std::unique_ptr<Transfer>> trs;
    // levels of at most this many nodes (globally) are held in full by every rank instead of being split into slabs
    const int64_t repl = std::atoll(pc->get("pc_b200_replicate_below", "4194304").c_str());
    PMG_TRY(build_structured_hierarchy(ctx, fine, L, repl, ops, trs));
    for (int l = L - 1; l >= 1; --l) {
      pc->lv[l].P         = std::move(trs[(size_t)l]);
      pc->lv[l - 1].owned = std::move(ops[(size_t)l - 1]);
      pc->lv[l - 1].op    = pc->lv[l - 1].owned.get();
    }
  } else {
    // assembled hierarchy: Q1 interpolation (SURVEY A.4) unless supplied, Galerkin A_c = P^T A P
    int64_t d[3] = {dims[0], dims[1], dims[2]};
    for (int l = L - 1; l >= 1; --l) {
      MgLevel &v = pc->lv[l];
      const HostCsr *A = v.op->host_csr();
      if (!A) PMG_FAIL(PMG_ERR_SUP, "gamgmc: level %d has no assembled operator", l);
      bool grid_known = false;
      if (!v.has_interp) {
        int64_t c[3];
        host_q1_dims(dim, d, c);
        if (c[0] * c[1] * c[2] == d[0] * d[1] * d[2]) PMG_FAIL(PMG_ERR_ARG, "gamgmc: cannot coarsen a %lldx%lldx%lld grid further (level %d)", (long long)d[0], (long long)d[1], (long long)d[2], l);
        host_q1_interp(dim, d, c, v.interp);
        std::memcpy(d, c, sizeof d);
        grid_known = true;
      }
      if (v.interp.n != A->n) PMG_FAIL(PMG_ERR_ARG, "gamgmc: interpolation of level %d has %lld rows, operator has %lld", l, (long long)v.interp.n, (long long)A->n);
      HostCsr R, AP, Ac;
      host_transpose(v.interp, R);
      host_matmul(*A, v.interp, AP);
      host_matmul(R, AP, Ac);
      PMG_TRY(make_csr_transfer(ctx, v.interp, v.P));
      if (grid_known) PMG_TRY(make_csr_grid_op(ctx, std::move(Ac), dim, d, pc->lv[l - 1].owned));
      else PMG_TRY(make_csr_op(ctx, std::move(Ac), pc->lv[l - 1].owned));
      pc->lv[l - 1].op = pc->lv[l - 1].owned.get();
    }
  }
  if (LrcData *flrc = top->lrc_data()) {
    // PCGAMGMC_SetUpHierarchy's MATLRC branch (src/pc_gamgmc.c:157-196): B_{l-1} = P_l^T B_l, every level samples from and
    // computes residuals with A_l + B_l diag(S) B_l^T
    const int           k = flrc->k;
    std::vector<double> Bl = flrc->Bh, Bc;
    DevBuf<double>      dBl, dBc;
    pc->lv[L - 1].op = top;
    for (int l = L - 1; l >= 1; --l) {
      const int64_t nf = pc->lv[l].op->n(), nc = pc->lv[l - 1].op->n();
      PMG_TRY(dBl.upload(Bl, ctx->stream));
      PMG_TRY(dBc.alloc((size_t)nc * k));
      for (int j = 0; j < k; ++j) PMG_TRY(pc->lv[l].P->restrict_to(dBl.p + (size_t)j * nf, dBc.p + (size_t)j * nc));
      Bc.resize((size_t)nc * k);
      PMG_CUDA(cudaMemcpyAsync(Bc.data(), dBc.p, Bc.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
      PMG_CUDA(cudaStreamSynchronize(ctx->stream));
      PMG_TRY(make_lrc_op(ctx, pc->lv[l - 1].op, k, Bc.data(), flrc->Sh.data(), pc->lv[l - 1].lrc_owned));
      pc->lv[l - 1].op = pc->lv[l - 1].lrc_owned.get();
      Bl.swap(Bc);
    }
  }
  const std::string cyc = pc->get("pc_b200_cycle", "direct");
  if (cyc != "direct" && cyc != "literal") PMG_FAIL(PMG_ERR_ARG, "-pc_b200_cycle %s: expected direct | literal", cyc.c_str());
  pc->direct_cycle = cyc == "direct";
  const char   *tm_env   = std::getenv("PMG_TAIL_MAX");
  const int64_t tail_max = (int64_t)std::atof(pc->get("pc_b200_tail_max_n", tm_env ? tm_env : "1500").c_str());
  // Levels 0 .. tail_fit fit the one-CTA shared-memory tail (tail2d.cuh) whatever -pc_b200_tail_max_n says (which bounds the
  // cluster tail through global memory); only asked for when the tail's other conditions can hold and the size is not user-set
  int tail_fit = -1;
  if (pc->direct_cycle && L >= 3 && tail_max > 0 && !pc->has("pc_b200_tail_max_n") && !tm_env && pc->get("gamgmc_mg_coarse_pc_type", "cholsampler") == "cholsampler" &&
      std::atoi(pc->get("gamgmc_mg_coarse_ksp_max_it", "1").c_str()) == 1 && pc->get("gamgmc_mg_levels_pc_type", "sorgibbs") != "cholsampler") {
    std::vector<LevelOp *> ops;
    for (int l = 0; l < L - 1; ++l) {
      ops.push_back(pc->lv[l].op);
      // one SM runs the whole tail: beyond a 65 x 65 top level (profiles/r2_summary.md: +27 us) the one-pass kernels on all SMs are faster
      static const int64_t top_max = std::getenv("PMG_TAIL_SMEM_MAX") ? std::atoll(std::getenv("PMG_TAIL_SMEM_MAX")) : 4500;
      if (l >= 1 && !ops[l]->distributed() && ops[l]->n() <= top_max && grid_tail_smem_fits(l + 1, ops.data(), ops[0]->n())) tail_fit = l;
    }
  }
  auto tail_sized = [&](int l) { return pc->lv[l].op->n() <= tail_max || l <= tail_fit; };
  // Galerkin levels that run on the one-pass kernels (box2d.cuh) keep their vectors PITCHED: a chain of levels below a fused
  // finest level, down to the first level that is small enough for the one-launch tail (or cannot run the kernels)
  for (int l = 0; l < L - 1; ++l) pc->lv[l].op->level_pitch = 0;
  if (pc->direct_cycle && L > 2 && !top->lrc_data() && pc->get("gamgmc_mg_levels_pc_type", "sorgibbs") != "cholsampler") {
    bool chain = pc->lv[L - 1].op->fused_mg_ok();
    for (int l = L - 2; l >= 1 && chain; --l) {
      LevelOp *o = pc->lv[l].op;
      chain      = o->box2_capable() && (o->distributed() || !tail_sized(l));
      if (chain) o->level_pitch = o->box2_pitch();
    }
    // a slab level's fused transfers write / read the level below in place: that level must be pitched too (or held in full)
    for (int l = 1; l <= L - 2; ++l) {
      LevelOp *o = pc->lv[l].op, *c = pc->lv[l - 1].op;
      if (o->level_pitch && o->distributed() && c->distributed() && !c->level_pitch) o->level_pitch = 0;
    }
  }
  // samplers: defaults of src/pc_gamgmc.c:305-349 (levels: richardson + sorgibbs, 1 it; coarse: cholsampler)
  for (int l = 0; l < L; ++l) {
    MgLevel          &v      = pc->lv[l];
    const std::string prefix = l == 0 ? "gamgmc_mg_coarse_" : "gamgmc_mg_levels_";
    const std::string ptype  = pc->get(prefix + "pc_type", l == 0 ? "cholsampler" : "sorgibbs");
    PMG_TRY(configure_sampler(pc, prefix, ptype, v.smp));
    const std::string ksp = pc->get(prefix + "ksp_type", "richardson");
    if (ksp != "richardson" && ksp != "preonly") PMG_FAIL(PMG_ERR_SUP, "-%sksp_type %s: samplers run under richardson (or preonly)", prefix.c_str(), ksp.c_str());
    v.smp.its = ksp == "preonly" ? 1 : std::atoi(pc->get(prefix + "ksp_max_it", "1").c_str());
    if (v.smp.its < 1) PMG_FAIL(PMG_ERR_ARG, "-%sksp_max_it must be >= 1", prefix.c_str());
    if (l < L - 1) PMG_TRY(apply_coloring_policy(pc, v.op, false));
    PMG_TRY(setup_level_sampler(ctx, v.smp, v.op));
    const size_t n = (size_t)v.op->n();
    const bool   pitched_level = l < L - 1 && v.op->level_pitch != 0;
    if (pitched_level) { // pad columns are read as ordinary elements by the TMA and must stay zero
      const size_t fs = (size_t)v.op->fused_size();
      PMG_TRY(v.b.alloc(fs));
      PMG_TRY(v.x.alloc(fs));
      PMG_TRY(v.x2.alloc(fs));
      PMG_TRY(v.b.zero(ctx->stream));
      PMG_TRY(v.x.zero(ctx->stream));
      PMG_TRY(v.x2.zero(ctx->stream));
    } else if (l < L - 1) {
      PMG_TRY(v.b.alloc(n));
      PMG_TRY(v.x.alloc(n));
    }
    if (l > 0 && !pitched_level) PMG_TRY(v.r.alloc(n));
    if (l > 0 && l < L - 1 && !pitched_level && v.smp.kind != KIND_CHOL && v.op->stream_ok()) PMG_TRY(v.x2.alloc(n));
    if (l > 0 && l == L - 1 && (v.op->fused_mg_ok() || v.op->fused_smooth_ok()) && v.smp.kind != KIND_CHOL) {
      if (v.op->fused_smooth_ok()) { // the residual lives in the pitched layout too
        PMG_TRY(v.r.alloc((size_t)v.op->fused_size()));
        PMG_TRY(v.r.zero(ctx->stream));
      }
      PMG_TRY(v.x2.alloc((size_t)v.op->fused_size()));
      PMG_TRY(pc->pit_y.alloc((size_t)v.op->fused_size()));
      PMG_TRY(pc->pit_b.alloc((size_t)v.op->fused_size()));
      // the pad columns of the pitched vectors are read by the TMA as ordinary elements and must stay zero
      PMG_TRY(v.x2.zero(ctx->stream));
      PMG_TRY(pc->pit_y.zero(ctx->stream));
      PMG_TRY(pc->pit_b.zero(ctx->stream));
    }
  }
  // the coarse tail: the largest lt < L-1 such that levels 0..lt are whole-grid stencil-array levels on this device, level 0
  // is the dense gemv sampler with one iteration, and level lt has at most -pc_b200_tail_max_n nodes
  pc->tail_top = -1;
  {
    MgLevel      &c0       = pc->lv[0];
    if (pc->direct_cycle && L >= 3 && tail_max > 0 && c0.smp.kind == KIND_CHOL && c0.smp.its == 1 && c0.smp.chol.use_gemv && !c0.smp.chol.packed && grid_tail_level_ok(c0.op)) {
      int lt = 0;
      for (int l = 1; l < L - 1; ++l) {
        MgLevel &v = pc->lv[l];
        if (v.smp.kind == KIND_CHOL || !grid_tail_level_ok(v.op) || !v.P || !v.P->tail_ok() || !tail_sized(l) || v.smp.its * (v.smp.gibbs.type == PMG_SOR_SYMMETRIC_SWEEP ? 2 : 1) > 8) break;
        lt = l;
      }
      if (lt >= 1 && lt + 1 <= 10) pc->tail_top = lt;
    }
  }
  const size_t nf = (size_t)fine->n();
  PMG_TRY(pc->w.alloc(nf));
  PMG_TRY(pc->work.alloc(nf));
  return 0;
}

static int pc_alloc_staging(pmg_pc pc)
{
  const size_t n = (size_t)pc->mat->op->n();
  PMG_TRY(pc->d_b.alloc(n));
  PMG_TRY(pc->d_y.alloc(n));
  if (pc->h_pinned) cudaFreeHost(pc->h_pinned);
  pc->h_pinned = nullptr;
  PMG_CUDA(cudaMallocHost((void **)&pc->h_pinned, n * sizeof(double)));
  if (!pc->ev0) {
    PMG_CUDA(cudaEventCreate(&pc->ev0));
    PMG_CUDA(cudaEventCreate(&pc->ev1));
  }
  return 0;
}

static int pc_notify(pmg_pc pc, int64_t it, const double *y_dev)
{
  PMG_TRY(pc->qoi.accumulate(y_dev));
  if (!pc->cb) return 0;
  const int64_t n = pc->mat->op->n();
  PMG_CUDA(cudaMemcpyAsync(pc->h_pinned, y_dev, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, pc->ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(pc->ctx->stream)); // host-visible y before the callback fires (SURVEY 8(b) threading)
  if (pc->cb(it, pc->h_pinned, n, pc->cbctx)) PMG_FAIL(PMG_ERR_CALLBACK, "sample callback returned an error at sample %lld", (long long)it);
  return 0;
}

static int richardson_body(pmg_pc pc, const double *b, double *y, int64_t its, int guesszero);

static int richardson_dev(pmg_pc pc, const double *b, double *y, int64_t its, int guesszero)
{
  pmg_ctx ctx = pc->ctx;
  if (!pc->is_setup) PMG_FAIL(PMG_ERR_ORDER, "pmg_pc_setup has not been called");
  const int64_t l0 = ctx->launches, u0 = ctx->dof_updates;
  PMG_CUDA(cudaEventRecord(pc->ev0, ctx->stream));
  PMG_TRY(richardson_body(pc, b, y, its, guesszero));
  PMG_CUDA(cudaEventRecord(pc->ev1, ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  float ms = 0;
  PMG_CUDA(cudaEventElapsedTime(&ms, pc->ev0, pc->ev1));
  PMG_TRY(prof_collect(pc));
  pc->last_ms       = ms;
  pc->last_launches = ctx->launches - l0;
  pc->last_updates  = ctx->dof_updates - u0;
  return 0;
}

// the samples themselves, asynchronous on the context's stream
static int richardson_body(pmg_pc pc, const double *b, double *y, int64_t its, int guesszero)
{
  pmg_ctx ctx = pc->ctx;
  if (!pc->is_setup) PMG_FAIL(PMG_ERR_ORDER, "pmg_pc_setup has not been called");
  const int64_t n = pc->mat->op->n();
  if (pc->type == "woodbury") { // PCApplyRichardson_Woodbury, src/woodbury.c:259-286
    LrcData *lrc = pc->mat->op->lrc_data();
    NoiseArgs na_eta;
    for (int64_t it = 0; it < its; ++it) {
      PMG_TRY(pc->noise.next(ctx, lrc->k, 0, na_eta));              // wk ~ N(0, I_k), scaled by sqrt|S|
      PMG_TRY(lrc->prepare_rhs(b, na_eta, lrc->rhs.p));             // w = b + B wk
      PMG_TRY(richardson_body(pc->wb_sampler, lrc->rhs.p, y, 1, 0)); // one sample of the inner sampler on A
      PMG_TRY(lrc->post_with(pc->wb_G.p, y));                       // y -= G (B^T y)
      PMG_TRY(pc_notify(pc, it, y));
    }
    return 0;
  }
  if (pc->type == "gamgmc") { // src/pc_gamgmc.c:242-259
    LevelOp *A = pc->lv[pc->nlevels - 1].op;
    if (!b) {
      PMG_TRY(pc->d_b.zero(ctx->stream));
      b = pc->d_b.p;
    }
    const bool top_fused = pc->direct_cycle && pc->nlevels > 1 && pc->lv[pc->nlevels - 1].x2.p;
    if (top_fused) { // the finest level runs the fused streaming sweeps on pitched copies of b and y
      PMG_TRY(A->to_pitched(b, pc->pit_b.p));
      if (!guesszero) PMG_TRY(A->to_pitched(y, pc->pit_y.p));
    }
    for (int64_t it = 0; it < its; ++it) {
      if (top_fused) {
        PMG_TRY(prefill_begin(pc));
        PMG_TRY(mg_cycle_direct(pc, pc->nlevels - 1, pc->pit_b.p, pc->pit_y.p, it == 0 && guesszero));
        PMG_TRY(prefill_end(pc));
        if (pc->cb || pc->qoi.on || it + 1 == its) PMG_TRY(A->from_pitched(pc->pit_y.p, y));
      } else if (pc->direct_cycle) {
        PMG_TRY(mg_cycle_direct(pc, pc->nlevels - 1, b, y, it == 0 && guesszero));
      } else if (it == 0 && guesszero) {
        PMG_TRY(mg_apply(pc, b, y));
      } else {
        PMG_TRY(A->residual(b, y, pc->w.p));             // w = b - A y
        PMG_TRY(mg_apply(pc, pc->w.p, pc->work.p));      // work = MG(w)
        PMG_TRY(launch_axpy(ctx, n, 1.0, pc->work.p, y)); // y += work
      }
      PMG_TRY(pc_notify(pc, it, y));
    }
  } else if (pc->type == "cholsampler") { // src/pc_chols.c:293-342
    if (!b) {
      PMG_TRY(pc->d_b.zero(ctx->stream));
      b = pc->d_b.p;
    }
    NoiseArgs na;
    if (its == 1) {
      PMG_TRY(pc->noise.next(ctx, n, 0, na));
      PMG_TRY(pc->smp.chol.sample(b, y, na));
      PMG_TRY(pc_notify(pc, pc->sample_index++, y));
    } else {
      PMG_TRY(pc->smp.chol.forward(b, pc->smp.chol.vcache.p));
      for (int64_t it = 0; it < its; ++it) {
        PMG_TRY(pc->noise.next(ctx, n, 0, na));
        PMG_TRY(pc->smp.chol.backward_noise(pc->smp.chol.vcache.p, y, na));
        PMG_TRY(pc_notify(pc, pc->sample_index++, y));
      }
    }
  } else { // mcgibbs: src/pc_mcgibbs.c:167-184; sorgibbs: src/pc_sorgibbs.c:125-129 (running sample_index from 0)
    if (pc->type == "sorgibbs") pc->sample_index = 0;
    LevelOp *op = pc->smp.gibbs.op;
    if (op->fused_ok() && pc->scratch.p && (noise_mode(pc) != PMG_NOISE_INJECTED || op->fused_tape_ok())) { // one fused pass per directional sweep, ping-pong between y and scratch
      std::vector<int> dirs;
      LevelSampler     one;
      one.its        = 1;
      one.gibbs.type = pc->smp.gibbs.type;
      sweep_dirs(one, dirs);
      PMG_TRY(pc->smp.gibbs.ensure());
      // when the pitched layout IS the natural one (row length a multiple of 4, no ghost units) the sweeps run on the
      // caller's vectors directly: no layout copies, y and the scratch vector ping-pong
      const bool    direct = op->pitched_is_natural() && ((((uintptr_t)y) | ((uintptr_t)b)) & 31u) == 0;
      const double *pb = nullptr;
      if (b) {
        if (direct) pb = b;
        else {
          PMG_TRY(op->to_pitched(b, pc->pit_b.p));
          pb = pc->pit_b.p;
        }
      }
      if (!direct) PMG_TRY(op->to_pitched(y, pc->pit_y.p));
      double   *cur = direct ? y : pc->pit_y.p, *oth = pc->scratch.p;
      NoiseArgs na;
      for (int64_t it = 0; it < its; ++it) {
        for (int d : dirs) {
          PMG_TRY(pc->noise.next(ctx, n, op->row0(), na));
          { NvtxRange range("MulticolSOR"); PMG_TRY(op->fused_sweep(d, pc->smp.gibbs.coeffs, pb, cur, oth, na, nullptr, nullptr, nullptr)); }
          std::swap(cur, oth);
        }
        if (pc->cb || pc->qoi.on || it + 1 == its) {
          if (!direct) PMG_TRY(op->from_pitched(cur, y));
          else if (cur != y) PMG_CUDA(cudaMemcpyAsync(y, cur, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        }
        PMG_TRY(pc_notify(pc, pc->type == "sorgibbs" ? pc->sample_index++ : it, y));
      }
    } else {
      for (int64_t it = 0; it < its; ++it) {
        PMG_TRY(pc->smp.gibbs.sample(pc->noise, b, y));
        PMG_TRY(pc_notify(pc, pc->type == "sorgibbs" ? pc->sample_index++ : it, y));
      }
    }
  }
  return 0;
}

// PCSetUp_Woodbury + PCWoodburyBuildLRCCorrection (src/woodbury.c:21-86, :141-186): the operator must be a MATLRC; sampler and
// solver are PCs of this library on its base matrix A.  `-pc_woodbury_solver cholesky` is the exact dense solve (the
// cholsampler without noise); any sampler type can also serve as solver: its deterministic application from a zero guess
// (one V-cycle for gamgmc, one sweep for mcgibbs / sorgibbs).
static int woodbury_setup(pmg_pc pc)
{
  pmg_ctx  ctx = pc->ctx;
  LrcData *lrc = pc->mat->op->lrc_data();
  if (!lrc || !pc->mat->base) PMG_FAIL(PMG_ERR_SUP, "PCWoodbury only supports matrices of type LRC"); // src/woodbury.c:161
  if (lrc->dist) PMG_FAIL(PMG_ERR_SUP, "PCWoodbury on a low-rank corrected operator with a row-distributed base is not supported: its exact solver is a dense single-device solve");
  if (!pc->has("pc_woodbury_sampler") || !pc->has("pc_woodbury_solver")) PMG_FAIL(PMG_ERR_SUP, "Must provide sampler and solver"); // :149
  auto make_inner = [&](const std::string &which, pmg_pc *out) -> int {
    std::string type = pc->get("pc_woodbury_" + which, "");
    if (type == "cholesky" || type == "lu") type = "cholsampler";
    PMG_TRY(pmg_pc_create(ctx, type.c_str(), out));
    (*out)->mat = pc->mat->base;
    const std::string prefix = "pc_woodbury_" + which + "_";
    for (const auto &kv : pc->opts)
      if (kv.first.compare(0, prefix.size(), prefix) == 0) (*out)->opts[kv.first.substr(prefix.size())] = kv.second;
    return 0;
  };
  if (pc->wb_sampler) pmg_pc_destroy(pc->wb_sampler);
  pc->wb_sampler = nullptr;
  PMG_TRY(make_inner("sampler", &pc->wb_sampler));
  pc->wb_sampler->noise.parent = &pc->noise;
  PMG_TRY(pmg_pc_setup(pc->wb_sampler));
  pmg_pc solver = nullptr;
  PMG_TRY(make_inner("solver", &solver));
  solver->noise.mode = PMG_NOISE_NONE;
  solver->opts.erase("pc_b200_noise");
  int err = pmg_pc_setup(solver);
  // C = solver(B), column by column from a zero guess (PCApply, src/woodbury.c:40-52)
  const int64_t       n = lrc->n;
  DevBuf<double>      C;
  std::vector<double> Ch((size_t)n * lrc->k);
  if (!err) err = C.alloc((size_t)n * lrc->k);
  if (!err) err = C.zero(ctx->stream);
  for (int j = 0; j < lrc->k && !err; ++j) err = richardson_body(solver, lrc->B.p + (size_t)j * n, C.p + (size_t)j * n, 1, 1);
  if (!err && cudaMemcpyAsync(Ch.data(), C.p, Ch.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) err = PMG_ERR_CUDA;
  if (!err && cudaStreamSynchronize(ctx->stream) != cudaSuccess) err = PMG_ERR_CUDA;
  pmg_pc_destroy(solver); // the reference drops the solver after set-up too (src/woodbury.c:184)
  if (err) return err;
  return lrc->correction_from(Ch, pc->wb_G);
}

extern "C" {

// ---- MCSOR -------------------------------------------------------------------------------------------
int pmg_mcsor_create(pmg_mat mat, pmg_mcsor *out)
{
  pmg_stale("pmg_mcsor_create");
  if (!mat) PMG_FAIL(PMG_ERR_ARG, "pmg_mcsor_create: null operator");
  PMG_CUDA(cudaSetDevice(mat->ctx->device));
  auto mc       = std::make_unique<pmg_mcsor_s>(mat->ctx);
  mc->mat       = mat;
  mc->core.op   = mat->op.get();
  mc->none.mode = PMG_NOISE_NONE;
  const char *e = std::getenv("PMG_MC_SOR_OMEGA"); // -mc_sor_omega read at create (src/mc_sor.c:638)
  if (e) mc->core.omega = std::atof(e);
  PMG_TRY(mc->core.ensure());
  PMG_TRY(mc->b.alloc((size_t)mat->op->n()));
  PMG_TRY(mc->y.alloc((size_t)mat->op->n()));
  *out = mc.release();
  return PMG_OK;
}
int pmg_mcsor_destroy(pmg_mcsor mc)
{
  pmg_stale("pmg_mcsor_destroy");
  if (mc) {
    cudaSetDevice(mc->ctx->device);
    delete mc;
  }
  return PMG_OK;
}
int pmg_mcsor_set_omega(pmg_mcsor mc, double omega)
{
  pmg_stale("pmg_mcsor_set_omega");
  mc->core.omega = omega;
  return PMG_OK;
}
int pmg_mcsor_set_sweep_type(pmg_mcsor mc, int type)
{
  pmg_stale("pmg_mcsor_set_sweep_type");
  if (type != PMG_SOR_FORWARD_SWEEP && type != PMG_SOR_BACKWARD_SWEEP && type != PMG_SOR_SYMMETRIC_SWEEP) PMG_FAIL(PMG_ERR_SUP, "Only forward, backward and symmetric sweep supported"); // src/mc_sor.c:427
  mc->core.type = type;
  return PMG_OK;
}
int pmg_mcsor_get_sweep_type(pmg_mcsor mc, int *type)
{
  pmg_stale("pmg_mcsor_get_sweep_type");
  *type = mc->core.type;
  return PMG_OK;
}
int pmg_mcsor_get_num_colors(pmg_mcsor mc, int *n)
{
  pmg_stale("pmg_mcsor_get_num_colors");
  *n = mc->mat->op->ncolors();
  return PMG_OK;
}
int pmg_mcsor_apply_dev(pmg_mcsor mc, const double *b, double *y)
{
  pmg_stale("pmg_mcsor_apply_dev");
  PMG_CUDA(cudaSetDevice(mc->ctx->device));
  PMG_TRY(mc->core.sample(mc->none, b, y));
  PMG_CUDA(cudaStreamSynchronize(mc->ctx->stream));
  return PMG_OK;
}
int pmg_mcsor_apply(pmg_mcsor mc, const double *b, double *y)
{
  pmg_stale("pmg_mcsor_apply");
  pmg_ctx ctx = mc->mat->ctx;
  PMG_CUDA(cudaSetDevice(ctx->device));
  const size_t n = (size_t)mc->mat->op->n();
  PMG_CUDA(cudaMemcpyAsync(mc->b.p, b, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  PMG_CUDA(cudaMemcpyAsync(mc->y.p, y, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  PMG_TRY(mc->core.sample(mc->none, mc->b.p, mc->y.p));
  PMG_CUDA(cudaMemcpyAsync(y, mc->y.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return PMG_OK;
}

// ---- PC ------------------------------------------------------------------------------------------------
int pmg_pc_create(pmg_ctx ctx, const char *type, pmg_pc *out)
{
  pmg_stale("pmg_pc_create");
  if (!ctx || !type) PMG_FAIL(PMG_ERR_ARG, "pmg_pc_create: bad arguments");
  const std::string t = type;
  if (t != "mcgibbs" && t != "sorgibbs" && t != "gamgmc" && t != "cholsampler" && t != "woodbury") PMG_FAIL(PMG_ERR_SUP, "PC type '%s' is not provided by parmgmc_b200 (mcgibbs | sorgibbs | gamgmc | cholsampler | woodbury)", type);
  auto pc  = std::make_unique<pmg_pc_s>(ctx);
  pc->type = t;
  *out     = pc.release();
  return PMG_OK;
}

int pmg_pc_destroy(pmg_pc pc)
{
  pmg_stale("pmg_pc_destroy");
  if (pc) {
    cudaSetDevice(pc->ctx->device);
    delete pc;
  }
  return PMG_OK;
}

int pmg_pc_reset(pmg_pc pc)
{
  pmg_stale("pmg_pc_reset");
  PMG_CUDA(cudaSetDevice(pc->ctx->device));
  pc->lv.clear();
  pc->is_setup     = false;
  pc->sample_index = 0;
  pc->smp          = LevelSampler();
  if (pc->deleter) { // PCReset_* runs the deleter (src/pc_mcgibbs.c:113-116)
    pc->deleter(pc->cbctx);
    pc->deleter = nullptr;
  }
  return PMG_OK;
}

int pmg_pc_set_operator(pmg_pc pc, pmg_mat mat)
{
  pmg_stale("pmg_pc_set_operator");
  if (!mat) PMG_FAIL(PMG_ERR_ARG, "null operator");
  if (mat->ctx != pc->ctx) PMG_FAIL(PMG_ERR_ARG, "operator and PC live on different contexts");
  pc->mat      = mat;
  pc->is_setup = false;
  return PMG_OK;
}

int pmg_pc_set_option(pmg_pc pc, const char *key, const char *value)
{
  pmg_stale("pmg_pc_set_option");
  if (!key) PMG_FAIL(PMG_ERR_ARG, "null option key");
  std::string k = key;
  while (!k.empty() && k[0] == '-') k.erase(0, 1);
  if (k == "pc_b200_profile") { // measurement switch: does not invalidate the set-up
    pc->prof_on = opt_true(value ? value : "");
    return PMG_OK;
  }
  pc->opts[k]  = value ? value : "";
  pc->is_setup = false;
  return PMG_OK;
}

int pmg_pc_setup(pmg_pc pc)
{
  pmg_stale("pmg_pc_setup");
  if (!pc->mat) PMG_FAIL(PMG_ERR_ORDER, "pmg_pc_setup: no operator set");
  pmg_ctx ctx = pc->ctx;
  PMG_CUDA(cudaSetDevice(ctx->device));
  const std::string nm = pc->get("pc_b200_noise", "");
  if (nm == "philox") pc->noise.mode = PMG_NOISE_PHILOX;
  else if (nm == "injected") pc->noise.mode = PMG_NOISE_INJECTED;
  else if (nm == "none") pc->noise.mode = PMG_NOISE_NONE;
  else if (!nm.empty()) PMG_FAIL(PMG_ERR_ARG, "-pc_b200_noise %s: expected philox | injected | none", nm.c_str());
  if (pc->type == "woodbury") PMG_TRY(woodbury_setup(pc));
  else if (pc->type == "gamgmc") PMG_TRY(gamgmc_setup(pc));
  else {
    const double omega_keep = pc->smp.gibbs.omega;
    const int    type_keep  = pc->smp.gibbs.type;
    PMG_TRY(configure_sampler(pc, "", pc->type, pc->smp));
    if (pc->type == "mcgibbs") { // setters called before set-up survive unless an option overrides them
      if (!pc->has("pc_mcgibbs_omega")) pc->smp.gibbs.omega = omega_keep;
      if (!pc->has("pc_mcgibbs_forward") && !pc->has("pc_mcgibbs_backward") && !pc->has("pc_mcgibbs_symmetric")) pc->smp.gibbs.type = type_keep;
    }
    PMG_TRY(apply_coloring_policy(pc, pc->mat->op.get(), true));
    PMG_TRY(setup_level_sampler(ctx, pc->smp, pc->mat->op.get()));
    if (pc->smp.kind != KIND_CHOL && pc->mat->op->fused_ok()) {
      PMG_TRY(pc->scratch.alloc((size_t)pc->mat->op->fused_size()));
      PMG_TRY(pc->pit_y.alloc((size_t)pc->mat->op->fused_size()));
      PMG_TRY(pc->pit_b.alloc((size_t)pc->mat->op->fused_size()));
      // the pad columns of the pitched vectors are read by the TMA as ordinary elements and must stay zero
      PMG_TRY(pc->scratch.zero(ctx->stream));
      PMG_TRY(pc->pit_y.zero(ctx->stream));
      PMG_TRY(pc->pit_b.zero(ctx->stream));
    }
  }
  PMG_TRY(pc_alloc_staging(pc));
  pc->is_setup = true;
  return PMG_OK;
}

int pmg_pc_view(pmg_pc pc, char *buf, size_t len)
{
  pmg_stale("pmg_pc_view");
  std::string s = "PC type: " + pc->type + "\n";
  char        t[256];
  if (!pc->is_setup) s += "  (not set up)\n";
  else if (pc->type == "mcgibbs") { // PCView_MulticolorGibbs, src/pc_mcgibbs.c:257-266
    snprintf(t, sizeof t, "Number of colours: %d\n", pc->mat->op->ncolors());
    s += t;
  } else if (pc->type == "sorgibbs") { // PCView_SORGibbs, src/pc_sorgibbs.c:295-305
    s += "Sweep type: Forward\n";
    snprintf(t, sizeof t, "Number of colours: %d\n", pc->mat->op->ncolors());
    s += t;
  } else if (pc->type == "cholsampler") { // PCView_CholSampler, src/pc_chols.c:383-396
    const CholSampler &ch = pc->smp.chol;
    snprintf(t, sizeof t, "Dense Cholesky factor for sequential block of size %lld\n", (long long)ch.n);
    s += t;
    if (ch.packed) snprintf(t, sizeof t, "  device factor (cuSOLVER potrf, cuBLAS trsm); samples stream the lower triangle of L^-1 in %lld tiles of 64 x 64 (%.0f bytes per sample)\n", (long long)(ch.nt * (ch.nt + 1) / 2), ch.sample_bytes());
    else if (ch.use_gemv) snprintf(t, sizeof t, "  host factor; samples are two matrix-vector products with dense copies of L^-1\n");
    else snprintf(t, sizeof t, "  host factor; samples are two sequential triangular solves in one CTA\n");
    s += t;
  } else {
    snprintf(t, sizeof t, "MG: type is MULTIPLICATIVE, levels=%d cycles=v\n", pc->nlevels);
    s += t;
    for (int l = 0; l < pc->nlevels; ++l) {
      std::string d;
      pc->lv[l].op->describe(d);
      const LevelSampler &sm = pc->lv[l].smp;
      snprintf(t, sizeof t, "  level %d: %s; sampler %s, max_it %d\n", l, d.c_str(), sm.kind == KIND_CHOL ? (sm.chol.packed ? "cholsampler (device factor, packed L^-1)" : "cholsampler") : sm.kind == KIND_MCGIBBS ? "mcgibbs" : "sorgibbs", sm.its);
      s += t;
    }
  }
  if (buf && len) {
    std::strncpy(buf, s.c_str(), len - 1);
    buf[len - 1] = 0;
  }
  return PMG_OK;
}

int pmg_pc_apply_richardson_dev(pmg_pc pc, const double *b, double *y, int64_t its, int guesszero, int64_t *outits, int *reason)
{
  pmg_stale("pmg_pc_apply_richardson_dev");
  PMG_CUDA(cudaSetDevice(pc->ctx->device));
  PMG_TRY(richardson_dev(pc, b, y, its, guesszero));
  if (outits) *outits = its;
  if (reason) *reason = 4; // PCRICHARDSON_CONVERGED_ITS
  return PMG_OK;
}

int pmg_pc_apply_richardson(pmg_pc pc, const double *b, double *y, int64_t its, int guesszero, int64_t *outits, int *reason)
{
  pmg_stale("pmg_pc_apply_richardson");
  pmg_ctx ctx = pc->ctx;
  if (!pc->is_setup) PMG_FAIL(PMG_ERR_ORDER, "pmg_pc_setup has not been called");
  PMG_CUDA(cudaSetDevice(ctx->device));
  const size_t n = (size_t)pc->mat->op->n();
  if (b) PMG_CUDA(cudaMemcpyAsync(pc->d_b.p, b, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  PMG_CUDA(cudaMemcpyAsync(pc->d_y.p, y, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  PMG_TRY(richardson_dev(pc, b ? pc->d_b.p : nullptr, pc->d_y.p, its, guesszero));
  PMG_CUDA(cudaMemcpyAsync(y, pc->d_y.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  if (outits) *outits = its;
  if (reason) *reason = 4;
  return PMG_OK;
}

int pmg_pc_apply(pmg_pc pc, const double *x, double *y)
{
  pmg_stale("pmg_pc_apply");
  pmg_ctx ctx = pc->ctx;
  if (!pc->is_setup) PMG_FAIL(PMG_ERR_ORDER, "pmg_pc_setup has not been called");
  if (pc->type != "sorgibbs" && pc->type != "cholsampler") PMG_FAIL(PMG_ERR_SUP, "PCApply is only defined for sorgibbs and cholsampler (the reference sets ops->apply only there)");
  PMG_CUDA(cudaSetDevice(ctx->device));
  const size_t n = (size_t)pc->mat->op->n();
  PMG_CUDA(cudaMemcpyAsync(pc->d_b.p, x, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  if (pc->type == "sorgibbs") { // src/pc_sorgibbs.c:105-113: zero y, one sample, no callback
    PMG_TRY(pc->d_y.zero(ctx->stream));
    PMG_TRY(pc->smp.gibbs.sample(pc->noise, pc->d_b.p, pc->d_y.p));
  } else { // src/pc_chols.c:262-291 (+ notify)
    NoiseArgs na;
    PMG_TRY(pc->noise.next(ctx, (int64_t)n, 0, na));
    PMG_TRY(pc->smp.chol.sample(pc->d_b.p, pc->d_y.p, na));
    PMG_TRY(pc_notify(pc, pc->sample_index++, pc->d_y.p));
  }
  PMG_CUDA(cudaMemcpyAsync(y, pc->d_y.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return PMG_OK;
}

int pmg_pc_set_sample_callback(pmg_pc pc, pmg_sample_cb cb, void *cbctx, pmg_ctx_deleter deleter)
{
  pmg_stale("pmg_pc_set_sample_callback");
  if (pc->type == "gamgmc") { // src/pc_gamgmc.c:369-380: must pass a callback; NULL ctx/deleter are ignored, not cleared
    if (pc->cb && pc->deleter) pc->deleter(pc->cbctx);
    if (!cb) PMG_FAIL(PMG_ERR_SUP, "Must pass callback function");
    pc->cb = cb;
    if (cbctx) pc->cbctx = cbctx;
    if (deleter) pc->deleter = deleter;
    return PMG_OK;
  }
  if (pc->deleter) pc->deleter(pc->cbctx); // src/pc_mcgibbs.c:295-298
  pc->cb      = cb;
  pc->cbctx   = cbctx;
  pc->deleter = deleter;
  return PMG_OK;
}

int pmg_pc_mcgibbs_set_omega(pmg_pc pc, double omega)
{
  pmg_stale("pmg_pc_mcgibbs_set_omega");
  if (pc->type != "mcgibbs") PMG_FAIL(PMG_ERR_ARG, "not a mcgibbs PC");
  pc->smp.gibbs.omega = omega; // lazily rebuilt at the next sample (omega_changed, src/pc_mcgibbs.c:275-276)
  pc->opts.erase("pc_mcgibbs_omega");
  return PMG_OK;
}
int pmg_pc_mcgibbs_set_sweep_type(pmg_pc pc, int type)
{
  pmg_stale("pmg_pc_mcgibbs_set_sweep_type");
  if (pc->type != "mcgibbs") PMG_FAIL(PMG_ERR_ARG, "not a mcgibbs PC");
  if (type != PMG_SOR_FORWARD_SWEEP && type != PMG_SOR_BACKWARD_SWEEP && type != PMG_SOR_SYMMETRIC_SWEEP) PMG_FAIL(PMG_ERR_SUP, "Only forward, backward and symmetric sweep supported");
  pc->smp.gibbs.type = type;
  pc->opts.erase("pc_mcgibbs_forward");
  pc->opts.erase("pc_mcgibbs_backward");
  pc->opts.erase("pc_mcgibbs_symmetric");
  return PMG_OK;
}

int pmg_pc_gamgmc_set_levels(pmg_pc pc, int levels)
{
  pmg_stale("pmg_pc_gamgmc_set_levels");
  if (pc->type != "gamgmc") PMG_FAIL(PMG_ERR_ARG, "not a gamgmc PC");
  if (levels < 1) PMG_FAIL(PMG_ERR_ARG, "levels must be >= 1");
  pc->nlevels = levels;
  if ((int)pc->lv.size() < levels) pc->lv.resize((size_t)levels);
  pc->opts.erase("gamgmc_pc_mg_levels");
  pc->is_setup = false;
  return PMG_OK;
}
int pmg_pc_gamgmc_get_levels(pmg_pc pc, int *levels)
{
  pmg_stale("pmg_pc_gamgmc_get_levels");
  *levels = pc->nlevels;
  return PMG_OK;
}
int pmg_pc_gamgmc_set_interpolation(pmg_pc pc, int level, int64_t nf, int64_t nc, const int64_t *rowptr, const int32_t *col, const double *val)
{
  pmg_stale("pmg_pc_gamgmc_set_interpolation");
  if (pc->type != "gamgmc") PMG_FAIL(PMG_ERR_ARG, "not a gamgmc PC");
  if (level < 1) PMG_FAIL(PMG_ERR_ARG, "interpolation is defined for levels >= 1");
  if ((int)pc->lv.size() <= level) pc->lv.resize((size_t)level + 1);
  MgLevel &v = pc->lv[level];
  v.interp.n = nf;
  v.interp.m = nc;
  v.interp.rowptr.assign(rowptr, rowptr + nf + 1);
  v.interp.col.assign(col, col + rowptr[nf]);
  v.interp.val.assign(val, val + rowptr[nf]);
  v.has_interp = true;
  pc->is_setup = false;
  return PMG_OK;
}
int pmg_pc_gamgmc_get_level_info(pmg_pc pc, int level, int64_t *n, int64_t *nnz, int *ncolors)
{
  pmg_stale("pmg_pc_gamgmc_get_level_info");
  if (!pc->is_setup || level < 0 || level >= pc->nlevels) PMG_FAIL(PMG_ERR_ARG, "bad level");
  LevelOp *op = pc->lv[level].op;
  if (n) *n = op->n();
  if (nnz) *nnz = op->host_csr() ? op->host_csr()->nnz() : -1;
  if (ncolors) *ncolors = op->ncolors();
  return PMG_OK;
}
int pmg_pc_gamgmc_get_level_csr(pmg_pc pc, int level, int64_t *rowptr, int32_t *col, double *val)
{
  pmg_stale("pmg_pc_gamgmc_get_level_csr");
  if (!pc->is_setup || level < 0 || level >= pc->nlevels) PMG_FAIL(PMG_ERR_ARG, "bad level");
  const HostCsr *a = pc->lv[level].op->host_csr();
  if (!a) PMG_FAIL(PMG_ERR_SUP, "level %d is matrix-free", level);
  std::memcpy(rowptr, a->rowptr.data(), a->rowptr.size() * sizeof(int64_t));
  std::memcpy(col, a->col.data(), a->col.size() * sizeof(int32_t));
  std::memcpy(val, a->val.data(), a->val.size() * sizeof(double));
  return PMG_OK;
}

int pmg_pc_set_noise_mode(pmg_pc pc, int mode)
{
  pmg_stale("pmg_pc_set_noise_mode");
  if (mode != PMG_NOISE_PHILOX && mode != PMG_NOISE_INJECTED && mode != PMG_NOISE_NONE) PMG_FAIL(PMG_ERR_ARG, "bad noise mode");
  pc->noise.mode = mode;
  pc->opts.erase("pc_b200_noise");
  return PMG_OK;
}
int pmg_pc_set_noise_tape(pmg_pc pc, const double *z, int64_t len)
{
  pmg_stale("pmg_pc_set_noise_tape");
  PMG_CUDA(cudaSetDevice(pc->ctx->device));
  PMG_TRY(pc->noise.tape.upload(z, (size_t)len, pc->ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(pc->ctx->stream));
  pc->noise.tape_len = len;
  pc->noise.tape_pos = 0;
  pc->noise.mode     = PMG_NOISE_INJECTED;
  pc->opts.erase("pc_b200_noise");
  return PMG_OK;
}
int pmg_pc_noise_per_sample(pmg_pc pc, int64_t *doubles)
{
  pmg_stale("pmg_pc_noise_per_sample");
  if (!pc->is_setup) PMG_FAIL(PMG_ERR_ORDER, "pmg_pc_setup has not been called");
  int64_t d = 0;
  if (pc->type == "woodbury") {
    PMG_TRY(pmg_pc_noise_per_sample(pc->wb_sampler, &d));
    d += pc->mat->op->lrc_data()->k;
  } else if (pc->type == "gamgmc") {
    for (int l = 0; l < pc->nlevels; ++l) d += (l == 0 ? 1 : 2) * sampler_draws(pc->lv[l].smp);
  } else if (pc->type == "cholsampler") d = pc->smp.chol.n;
  else d = pc->smp.gibbs.draws_per_sample();
  *doubles = d;
  return PMG_OK;
}

// ---- statistics on the device (examples/benchmark/main.cc:151-175, src/iact.c) ----
int pmg_pc_set_qoi(pmg_pc pc, const double *meas_host, int64_t capacity, int est_mean_and_var)
{
  pmg_stale("pmg_pc_set_qoi");
  if (!pc->mat) PMG_FAIL(PMG_ERR_ORDER, "pmg_pc_set_qoi: no operator set");
  PMG_CUDA(cudaSetDevice(pc->ctx->device));
  if (!meas_host) { // switch off
    pc->qoi.on = false;
    return PMG_OK;
  }
  if (capacity < 1) PMG_FAIL(PMG_ERR_ARG, "pmg_pc_set_qoi: capacity must be positive");
  return pc->qoi.init(pc->ctx, pc->mat->op->n(), meas_host, capacity, est_mean_and_var != 0);
}
int pmg_pc_get_qoi(pmg_pc pc, double *qois_host, int64_t *count, int reset)
{
  pmg_stale("pmg_pc_get_qoi");
  if (!pc->qoi.on) PMG_FAIL(PMG_ERR_ORDER, "pmg_pc_get_qoi: no QOI registered");
  PMG_CUDA(cudaSetDevice(pc->ctx->device));
  if (qois_host && pc->qoi.count) PMG_CUDA(cudaMemcpyAsync(qois_host, pc->qoi.trace.p, sizeof(double) * (size_t)pc->qoi.count, cudaMemcpyDeviceToHost, pc->ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(pc->ctx->stream));
  if (count) *count = pc->qoi.count;
  if (reset) pc->qoi.count = 0;
  return PMG_OK;
}
int pmg_pc_get_mean_var(pmg_pc pc, double *mean_host, double *var_host, int64_t *nseen)
{
  pmg_stale("pmg_pc_get_mean_var");
  if (!pc->qoi.on || !pc->qoi.welford) PMG_FAIL(PMG_ERR_ORDER, "pmg_pc_get_mean_var: register the QOI with est_mean_and_var");
  PMG_CUDA(cudaSetDevice(pc->ctx->device));
  const size_t n = (size_t)pc->qoi.n;
  if (mean_host) PMG_CUDA(cudaMemcpyAsync(mean_host, pc->qoi.mean.p, sizeof(double) * n, cudaMemcpyDeviceToHost, pc->ctx->stream));
  if (var_host) PMG_CUDA(cudaMemcpyAsync(var_host, pc->qoi.M2.p, sizeof(double) * n, cudaMemcpyDeviceToHost, pc->ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(pc->ctx->stream));
  if (var_host && pc->qoi.nseen > 1)
    for (size_t i = 0; i < n; ++i) var_host[i] /= (double)(pc->qoi.nseen - 1); // sample variance from Welford's M2
  if (nseen) *nseen = pc->qoi.nseen;
  return PMG_OK;
}
int pmg_autocorrelation(pmg_ctx ctx, int64_t n, const double *x_host, double *acf_host)
{
  pmg_stale("pmg_autocorrelation");
  PMG_CUDA(cudaSetDevice(ctx->device));
  return device_autocorrelation(ctx, n, x_host, acf_host);
}
int pmg_iact(pmg_ctx ctx, int64_t n, const double *x_host, double *tau, double *acf_host_or_null, int *valid)
{
  pmg_stale("pmg_iact");
  PMG_CUDA(cudaSetDevice(ctx->device));
  return device_iact(ctx, n, x_host, tau, acf_host_or_null, valid);
}

// host-side work list of the fused 3D sweep: no device needed (tests/test_abi_cpu.py checks the tiling)
int pmg_plan_sweep3d(int64_t nx, int64_t ny, int64_t nz, int64_t slo, int64_t shi, int bz, int nw, int32_t *items, int64_t capacity, int64_t *count)
{
  if (nx < 1 || ny < 1 || nz < 1 || slo < 0 || shi > nz || slo >= shi || bz < 1 || nw < 3 || !count) PMG_FAIL(PMG_ERR_ARG, "pmg_plan_sweep3d: bad geometry");
  std::vector<int32_t> flat;
  sweep3d_plan(nx, ny, nz, slo, shi, bz, nw, true, 4, flat);
  *count = (int64_t)(flat.size() / 5);
  if (items) {
    if (capacity < *count) PMG_FAIL(PMG_ERR_ARG, "pmg_plan_sweep3d: %lld items, capacity %lld", (long long)*count, (long long)capacity);
    std::memcpy(items, flat.data(), flat.size() * sizeof(int32_t));
  }
  return PMG_OK;
}

int pmg_plan_sweep2d(int64_t nx, int64_t ny, int64_t slo, int64_t shi, int by, int restrict_mode, int overlap, int32_t *items, int64_t capacity, int64_t *count, int64_t *nohalo)
{
  if (nx < 8 || ny < 4 || slo < 0 || shi > ny || slo >= shi || by < 2 || (by & 1) || !count) PMG_FAIL(PMG_ERR_ARG, "pmg_plan_sweep2d: bad geometry");
  std::vector<int32_t> flat;
  int                  nh = 0;
  sweep2d_plan(nx, ny, slo, shi, slo > 0 || shi < ny, by, restrict_mode != 0, overlap != 0, flat, nh);
  *count = (int64_t)(flat.size() / 3);
  if (nohalo) *nohalo = nh;
  if (items) {
    if (capacity < *count) PMG_FAIL(PMG_ERR_ARG, "pmg_plan_sweep2d: %lld items, capacity %lld", (long long)*count, (long long)capacity);
    std::memcpy(items, flat.data(), flat.size() * sizeof(int32_t));
  }
  return PMG_OK;
}

int pmg_normal_fill(pmg_ctx ctx, uint64_t seed, uint64_t call, int64_t row0, int64_t n, double *z)
{
  pmg_stale("pmg_normal_fill");
  PMG_CUDA(cudaSetDevice(ctx->device));
  DevBuf<double> d;
  PMG_TRY(d.alloc((size_t)n));
  NoiseArgs na{PMG_NOISE_PHILOX, nullptr, seed, call, row0};
  NvtxRange range("VecSetRandN");
  PMG_TRY(launch_normal_fill(ctx, na, n, d.p));
  PMG_CUDA(cudaMemcpyAsync(z, d.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  PMG_CUDA(cudaStreamSynchronize(ctx->stream));
  return PMG_OK;
}

// Per-kernel profile of the V-cycle since the last reset, as JSON: [{"kernel": label, "launches": n, "ms": total,
// "bytes_min": compulsory bytes, "bytes_survey": SURVEY 8(d) bytes}, ...] in first-launch order.  Enabled with
// pmg_pc_set_option(pc, "-pc_b200_profile", "1") (may be switched at any time; events are recorded around every labelled launch).
int pmg_pc_profile(pmg_pc pc, char *buf, size_t len, int reset)
{
  pmg_stale("pmg_pc_profile");
  PMG_TRY(prof_collect(pc));
  std::string s = "[";
  char        t[512];
  bool        first = true;
  for (const auto &label : pc->prof_order) {
    const auto &a = pc->prof_sum[label];
    snprintf(t, sizeof t, "%s{\"kernel\": \"%s\", \"launches\": %lld, \"ms\": %.6f, \"bytes_min\": %.0f, \"bytes_survey\": %.0f}", first ? "" : ", ", label.c_str(), (long long)a.launches, a.ms, a.bytes_min, a.bytes_survey);
    s += t;
    first = false;
  }
  s += "]";
  if (buf && len) {
    std::strncpy(buf, s.c_str(), len - 1);
    buf[len - 1] = 0;
  }
  if (reset) {
    pc->prof_sum.clear();
    pc->prof_order.clear();
  }
  return PMG_OK;
}

int pmg_pc_last_stats(pmg_pc pc, double *ms, int64_t *launches, int64_t *updates)
{
  pmg_stale("pmg_pc_last_stats");
  if (ms) *ms = pc->last_ms;
  if (launches) *launches = pc->last_launches;
  if (updates) *updates = pc->last_updates;
  return PMG_OK;
}

// ---- multi-GPU plumbing is in comm.cu ---------------------------------------------------------------------

} // extern "C"
