/* parmgmc_b200.h -- C ABI of the B200-native sampling hot path of ParMGMC.
 *
 * This is the drop-in boundary: plain pointers and sizes, `extern "C"`, no torch / PETSc types.
 * A PETSc shim (shim/petsc/, INTEGRATION.md) registers the reference's PC types ("mcgibbs",
 * "sorgibbs", "gamgmc", "cholsampler") and forwards every PC op to the pmg_pc_* entry points
 * below; a non-PETSc C program can call them directly.  Citations are file:line under the
 * reference tree (nilsfriess/ParMGMC).
 *
 * Conventions
 *   - every function returns 0 on success or a PMG_ERR_* code; pmg_last_error() holds the message
 *     (the shim turns it into SETERRQ, reference convention: PetscErrorCode everywhere)
 *   - FP64 values, int32 column indices, int64 row offsets
 *   - `*_host` pointers are borrowed for the duration of the call only; `*_dev` pointers are device
 *     memory on the context's GPU
 *   - calls are blocking at return (host-visible results are coherent), like the reference
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     PMG_ERR_NO_DEVICE
 */
#ifndef PARMGMC_B200_H
#define PARMGMC_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define PMG_OK 0
#define PMG_ERR_ARG 1        /* PETSC_ERR_ARG_* */
#define PMG_ERR_SUP 2        /* PETSC_ERR_SUP, e.g. unsupported matrix / sweep type (src/mc_sor.c:427,568) */
#define PMG_ERR_NO_DEVICE 3  /* no CUDA device / extension cannot run */
#define PMG_ERR_CUDA 4       /* a CUDA runtime call failed */
#define PMG_ERR_NOT_SPD 5    /* PETSC_ERR_MAT_CH_ZRPVT (src/pc_chols.c:192) */
#define PMG_ERR_ORDER 6      /* object used before set-up */
#define PMG_ERR_NOISE 7      /* injected noise tape exhausted */
#define PMG_ERR_COLORING 8   /* colouring is not a valid distance-1 colouring */
#define PMG_ERR_COMM 9       /* NCCL failure */
#define PMG_ERR_CALLBACK 10  /* user callback returned non-zero */

/* PETSc MatSORType values, as passed to MCSORSetSweepType / PCMulticolorGibbsSetSweepType
 * (include/parmgmc/mc_sor.h:22, include/parmgmc/pc/pc_mcgibbs.h:18) */
#define PMG_SOR_FORWARD_SWEEP 1
#define PMG_SOR_BACKWARD_SWEEP 2
#define PMG_SOR_SYMMETRIC_SWEEP 3
#define PMG_SOR_LOCAL_FORWARD_SWEEP 4 /* -pc_sorgibbs_local_forward (src/pc_sorgibbs.c:274); == forward on one device */

/* colouring policies for pmg_mat_set_coloring_auto */
#define PMG_COLORING_GREEDY 0        /* first-fit distance-1 (stands in for MATCOLORINGJP, src/mc_sor.c:383-395) */
#define PMG_COLORING_LEXICOGRAPHIC 1 /* level sets: reproduces the 1-rank one-colour sweep (src/mc_sor.c:397-410) exactly */
#define PMG_COLORING_PARITY 2        /* structured grids: red-black (star stencil) / 2^d colours (box stencil) */

/* noise sources */
#define PMG_NOISE_PHILOX 0   /* counter-based Philox4x32-10 + Box-Muller, keyed (seed, draw#, global row) */
#define PMG_NOISE_INJECTED 1 /* z blocks supplied by the caller, consumed in call order (SURVEY 8(c) tape contract) */
#define PMG_NOISE_NONE 2     /* z = 0: deterministic SOR (MCSORApply semantics) */

typedef struct pmg_ctx_s   *pmg_ctx;
typedef struct pmg_mat_s   *pmg_mat;
typedef struct pmg_mcsor_s *pmg_mcsor;
typedef struct pmg_pc_s    *pmg_pc;

/* ---- library / context -------------------------------------------------------------------
 * replaces ParMGMCInitialize/Finalize (src/parmgmc.c:118-137) and the global RNG singleton
 * (src/parmgmc.c:38-68): the context owns the device, the stream and the noise state. */
const char *pmg_version(void);
const char *pmg_last_error(void);
int         pmg_device_count(int *count);
int         pmg_ctx_create(int device, pmg_ctx *ctx);
int         pmg_ctx_destroy(pmg_ctx ctx);
int         pmg_ctx_set_stream(pmg_ctx ctx, void *cuda_stream); /* run on a caller-owned cudaStream_t */
int         pmg_ctx_synchronize(pmg_ctx ctx);
/* PetscRandomSetSeed + PetscRandomSeed on the global stream (examples/benchmark/main.cc:228-236);
 * resets the draw counter */
int pmg_ctx_set_seed(pmg_ctx ctx, uint64_t seed);
int pmg_ctx_get_draw_counter(pmg_ctx ctx, uint64_t *draws);
int pmg_ctx_set_draw_counter(pmg_ctx ctx, uint64_t draws); /* (y, seed, draw counter) is a complete checkpoint */
/* one process per GPU; rank 0 creates the id and the host program broadcasts it (MPI_Bcast /
 * torch.distributed), replacing PETSc's communicator plumbing (src/mc_sor.c:169,203) */
int pmg_comm_unique_id(unsigned char id[128]);
int pmg_ctx_comm_init(pmg_ctx ctx, int rank, int nranks, const unsigned char id[128]);
int pmg_ctx_comm_rank(pmg_ctx ctx, int *rank, int *nranks);
/* 1: the ghost exchange of slab-partitioned grid operators (the per-colour VecScatter of src/mc_sor.c:318-319, :345-346) runs
 * through peer memory over NVLink (mailboxes mapped with CUDA IPC at pmg_ctx_comm_init); 0: through ncclSend / ncclRecv
 * (environment PMG_NO_P2P, or no peer access between the neighbours' devices) */
int pmg_ctx_comm_p2p(pmg_ctx ctx, int *enabled);

/* ---- operators -------------------------------------------------------------------------------
 * pmg_mat_create_csr: what the shim gets from MatSeqAIJGetCSRAndMemType (src/mc_sor.c:142,250);
 * values are copied to the device, the host arrays are not retained. */
int pmg_mat_create_csr(pmg_ctx ctx, int64_t n, const int64_t *rowptr_host, const int32_t *col_host, const double *val_host, pmg_mat *mat);
/* Matrix-free shifted Laplacian kappa^2 I + h^2 L of MatAssembleShiftedLaplaceFD (src/problems.c:14-75;
 * dim = 3 is the 7-point extension).  The grid is nx*ny*nz in natural order; this rank owns the
 * slab [slab_lo, slab_hi) of the slowest dimension (0, ny or nz for the whole grid). */
int pmg_mat_create_laplace(pmg_ctx ctx, int dim, int64_t nx, int64_t ny, int64_t nz, double kappa, int64_t slab_lo, int64_t slab_hi, pmg_mat *mat);
/* A row-partitioned operator, one call per rank (collective): this rank owns rows [row_start, row_start + n_local) of an
 * n_global x n_global matrix and passes them with GLOBAL column indices, as MatCreateMPIAIJWithArrays would.  The library
 * splits them into the diagonal block, the off-diagonal block and its column map exactly as the reference reads them
 * from MatMPIAIJGetSeqAIJ (src/mc_sor.c:308-310) and gathers the ghost values before every colour (src/mc_sor.c:318-319).
 * The colouring must be a distance-1 colouring of the GLOBAL graph (src/mc_sor.c:383-395): pmg_mat_set_coloring checks it
 * across ranks; the automatic one offsets a local greedy colouring by rank (parity) instead of PETSc's Jones-Plassmann. */
int pmg_mat_create_csr_dist(pmg_ctx ctx, int64_t n_global, int64_t row_start, int64_t n_local, const int64_t *rowptr_host, const int64_t *col_global_host, const double *val_host, pmg_mat *mat);
/* MatCreateLRC(A, B, S, NULL): the operator A + B diag(S) B^T with B dense n x k (column-major) and S of length k, as the
 * reference's samplers receive it through MatLRCGetMats (src/mc_sor.c:565-595, src/pc_mcgibbs.c:236-244,
 * src/pc_sorgibbs.c:204-223).  A is borrowed and must outlive the result; sweeps run on A and are followed by the
 * rank-k correction y -= Bb (B^T y) of MCSORPostSOR_LRC (src/mc_sor.c:101-112).
 * On a distributed A (this rank holds n_local < n_global rows: a slab of pmg_mat_create_laplace or pmg_mat_create_csr_dist)
 * the call is collective and B_host holds this rank's n_local rows, column-major with leading dimension n_local (n_local = 0
 * is allowed).  S must be bitwise identical on every rank and k the same: both are checked here, and a mismatch fails with
 * PMG_ERR_ARG on every rank.  B^T y is folded per rank, all-gathered and summed in rank order, so every rank applies the same
 * update and repeated runs give the same bits; the result agrees with one GPU to rounding, not bitwise.  A level that every
 * rank holds in full never reduces across ranks.  PCWOODBURY and a cholsampler on such an operator fail with PMG_ERR_SUP. */
int pmg_mat_create_lrc(pmg_mat A, int k, const double *B_host, const double *S_host, pmg_mat *mat);
int pmg_mat_destroy(pmg_mat mat);
int pmg_mat_get_size(pmg_mat mat, int64_t *n_local, int64_t *n_global, int64_t *row_start);
/* ISColoring of MCSORGetISColoring (src/mc_sor.c:92-99): explicit colours (validated) or a policy */
int pmg_mat_set_coloring(pmg_mat mat, int ncolors, const int32_t *color_of_row_host);
int pmg_mat_set_coloring_auto(pmg_mat mat, int policy);
int pmg_mat_get_coloring(pmg_mat mat, int *ncolors, int32_t *color_of_row_host_or_null);
/* y = A x on the device (MatMult, src/pc_gamgmc.c:253); host pointers */
int pmg_mat_mult(pmg_mat mat, const double *x_host, double *y_host);

/* ---- MCSOR: include/parmgmc/mc_sor.h:17-30 -----------------------------------------------------
 * MCSORCreate/SetUp/Destroy/Apply/SetOmega/SetSweepType/GetSweepType/GetNumColors. */
int pmg_mcsor_create(pmg_mat mat, pmg_mcsor *mc);          /* MCSORCreate + MCSORSetUp (src/mc_sor.c:553-642) */
int pmg_mcsor_destroy(pmg_mcsor mc);                       /* MCSORDestroy (src/mc_sor.c:60-90) */
int pmg_mcsor_set_omega(pmg_mcsor mc, double omega);       /* MCSORSetOmega (src/mc_sor.c:412-420) */
int pmg_mcsor_set_sweep_type(pmg_mcsor mc, int type);      /* MCSORSetSweepType (src/mc_sor.c:422-430); PMG_ERR_SUP otherwise */
int pmg_mcsor_get_sweep_type(pmg_mcsor mc, int *type);     /* MCSORGetSweepType (src/mc_sor.c:432-439) */
int pmg_mcsor_get_num_colors(pmg_mcsor mc, int *ncolors);  /* MCSORGetNumColors (src/mc_sor.c:607-616) */
int pmg_mcsor_apply(pmg_mcsor mc, const double *b_host, double *y_host); /* MCSORApply (src/mc_sor.c:216-239), in place on y */
int pmg_mcsor_apply_dev(pmg_mcsor mc, const double *b_dev, double *y_dev);

/* ---- samplers: the PC plugins of src/pc_mcgibbs.c, pc_sorgibbs.c, pc_gamgmc.c, pc_chols.c ---------
 * type is the reference's PC type string (include/parmgmc/parmgmc.h:26-31).  Options use the
 * reference's option keys (SURVEY Appendix C), e.g.
 *   pmg_pc_set_option(pc, "-pc_mcgibbs_omega", "1.2"); pmg_pc_set_option(pc, "-pc_mcgibbs_symmetric", "");
 *   pmg_pc_set_option(pc, "-gamgmc_pc_mg_levels", "10"); pmg_pc_set_option(pc, "-gamgmc_mg_levels_ksp_max_it", "2");
 * plus "-pc_b200_coloring greedy|lexicographic|parity", "-pc_b200_noise philox|injected|none",
 * "-pc_b200_cycle direct|literal" and "-pc_b200_grid nx,ny[,nz]" (grid of an assembled operator, what PCSetDM tells the
 * reference's geometric PCMG).
 * type "woodbury" (src/woodbury.c) needs a MATLRC operator (pmg_mat_create_lrc) and the options "-pc_woodbury_sampler
 * mcgibbs|sorgibbs|gamgmc|cholsampler" and "-pc_woodbury_solver cholesky|<sampler type>"; options of the two inner PCs are
 * passed with the prefixes "pc_woodbury_sampler_" / "pc_woodbury_solver_" (src/woodbury.c:189-252). */
typedef int (*pmg_sample_cb)(int64_t it, const double *y_host, int64_t n, void *ctx);
typedef int (*pmg_ctx_deleter)(void *ctx);

int pmg_pc_create(pmg_ctx ctx, const char *type, pmg_pc *pc);    /* PCCreate + PCSetType */
int pmg_pc_destroy(pmg_pc pc);                                   /* PCDestroy_* */
int pmg_pc_reset(pmg_pc pc);                                     /* PCReset_* */
int pmg_pc_set_operator(pmg_pc pc, pmg_mat mat);                 /* PCSetOperators; borrowed like src/mc_sor.c:630 */
int pmg_pc_set_option(pmg_pc pc, const char *key, const char *value); /* PCSetFromOptions_* */
int pmg_pc_setup(pmg_pc pc);                                     /* PCSetUp_* */
int pmg_pc_view(pmg_pc pc, char *buf, size_t buflen);            /* PCView_* */
/* PCApplyRichardson_*(pc,b,y,w,rtol,abstol,dtol,its,guesszero,outits,reason): `its` samples, the
 * chain continues from y (src/pc_mcgibbs.c:155-188, pc_sorgibbs.c:115-134, pc_gamgmc.c:227-264,
 * pc_chols.c:293-342).  Tolerances are ignored by every reference sampler and are not passed.
 * reason is always PCRICHARDSON_CONVERGED_ITS (= 4). b may be NULL (b = 0, prior sampling). */
int pmg_pc_apply_richardson(pmg_pc pc, const double *b_host, double *y_host, int64_t its, int guesszero, int64_t *outits, int *reason);
int pmg_pc_apply_richardson_dev(pmg_pc pc, const double *b_dev, double *y_dev, int64_t its, int guesszero, int64_t *outits, int *reason);
/* PCApply_SORGibbs (src/pc_sorgibbs.c:105-113: y = 0 then one sample) / PCApply_CholSampler
 * (src/pc_chols.c:262-291) */
int pmg_pc_apply(pmg_pc pc, const double *x_host, double *y_host);
/* PCSetSampleCallback (src/parmgmc.c:146-151): cb(it, y, ctx) after every sample, optional deleter
 * run on replace/destroy (src/pc_mcgibbs.c:290-303) */
int pmg_pc_set_sample_callback(pmg_pc pc, pmg_sample_cb cb, void *ctx, pmg_ctx_deleter deleter);
/* PCMulticolorGibbsSetOmega / SetSweepType (include/parmgmc/pc/pc_mcgibbs.h:17-18) */
int pmg_pc_mcgibbs_set_omega(pmg_pc pc, double omega);
int pmg_pc_mcgibbs_set_sweep_type(pmg_pc pc, int type);
/* PCGAMGMCSetLevels (include/parmgmc/pc/pc_gamgmc.h:16) and the PCMG calls a geometric user makes */
int pmg_pc_gamgmc_set_levels(pmg_pc pc, int levels);
int pmg_pc_gamgmc_get_levels(pmg_pc pc, int *levels); /* "PCMGGetLevels_C" (src/pc_gamgmc.c:413) */
int pmg_pc_gamgmc_set_interpolation(pmg_pc pc, int level, int64_t nf, int64_t nc, const int64_t *rowptr_host, const int32_t *col_host, const double *val_host); /* PCMGSetInterpolation */
int pmg_pc_gamgmc_get_level_info(pmg_pc pc, int level, int64_t *n, int64_t *nnz, int *ncolors);
int pmg_pc_gamgmc_get_level_csr(pmg_pc pc, int level, int64_t *rowptr_host, int32_t *col_host, double *val_host);
/* noise control: injected tape for deterministic parity runs (SURVEY 8(c)); total doubles the next
 * apply_richardson call(s) will consume can be queried */
int pmg_pc_set_noise_mode(pmg_pc pc, int mode);
int pmg_pc_set_noise_tape(pmg_pc pc, const double *z_host, int64_t len);
int pmg_pc_noise_per_sample(pmg_pc pc, int64_t *doubles);
/* fill z_host[0..n) with the device generator's N(0,1) draw for (seed, call, global rows row0..row0+n):
 * VecSetRandomStandardNormal (src/parmgmc.c:70-116) on the device */
/* ---- statistics kept on the device -------------------------------------------------------------
 * pmg_pc_set_qoi: what examples/benchmark/main.cc:151-175 (SaveSample) does in a host callback -- qoi[it] = <y, meas> after
 * every sample, optionally Welford's running mean / variance of the whole field -- as one kernel per sample, so that no
 * sample has to travel to the host.  meas_host = NULL switches it off.  pmg_iact / pmg_autocorrelation: IACT / Autocorrelation
 * of src/iact.c:17-92 (include/parmgmc/iact.h:14-15) with cuFFT in place of FFTW. */
int pmg_pc_set_qoi(pmg_pc pc, const double *meas_host, int64_t capacity, int est_mean_and_var);
int pmg_pc_get_qoi(pmg_pc pc, double *qois_host, int64_t *count, int reset);
int pmg_pc_get_mean_var(pmg_pc pc, double *mean_host, double *var_host, int64_t *nseen);
int pmg_autocorrelation(pmg_ctx ctx, int64_t n, const double *x_host, double *acf_host);
int pmg_iact(pmg_ctx ctx, int64_t n, const double *x_host, double *tau, double *acf_host_or_null, int *valid);

int pmg_normal_fill(pmg_ctx ctx, uint64_t seed, uint64_t call, int64_t row0, int64_t n, double *z_host);
/* host-side work list of the fused 3D sweep (csrc/sweep3d.cuh; the tiling that replaces the colour loops of src/mc_sor.c:257-285
 * on a 7-point grid operator): `count` items of five ints (strip of 120 columns, first row, first plane, end plane, narrow-strip flag).
 * Needs no device; the CPU tests check that the tiles cover the owned planes exactly once.  items = NULL only counts. */
int pmg_plan_sweep3d(int64_t nx, int64_t ny, int64_t nz, int64_t slo, int64_t shi, int bz, int nw, int32_t *items, int64_t capacity, int64_t *count);
/* the same for the fused 2D sweep (csrc/sweep2d.cuh): `count` items of three ints (strip of 120 columns, first row, end row) for the rows
 * [slo, shi) of an nx x ny grid in bands of `by` rows (fused residual + restriction variant: restrict_mode = 1).  The first `nohalo` tiles read
 * no ghost row; with overlap = 1 the others are 8-row bands next to the neighbouring slabs, which run behind the ghost exchange (the
 * per-colour scatter of src/mc_sor.c:318-319 overlapped with the interior rows). */
int pmg_plan_sweep2d(int64_t nx, int64_t ny, int64_t slo, int64_t shi, int by, int restrict_mode, int overlap, int32_t *items, int64_t capacity, int64_t *count, int64_t *nohalo);

/* ---- measurement hooks (bench.py) ----------------------------------------------------------------- */
/* average device time [ms] and launch count of the kernels the last apply_richardson* call issued */
int pmg_pc_last_stats(pmg_pc pc, double *ms_total, int64_t *launches, int64_t *dof_updates);
/* Per-kernel profile of the V-cycle (measurement aid; the analogue of the reference's PetscLogEvent pair MulticolSOR /
 * VecSetRandN, src/parmgmc.c:123-125, read with -log_view): after pmg_pc_set_option(pc, "-pc_b200_profile", "1") every
 * labelled launch of pmg_pc_apply_richardson* is bracketed by CUDA events; the totals come back as a JSON array. */
int pmg_pc_profile(pmg_pc pc, char *buf, size_t len, int reset);

#ifdef __cplusplus
}
#endif
#endif
