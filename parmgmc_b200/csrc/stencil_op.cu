// stencil_op.cu -- structured-grid operators: the matrix-free path.
//
//   LapOp   the shifted Laplacian kappa^2 I + h^2 L of MatAssembleShiftedLaplaceFD (reference
//           src/problems.c:14-75; dim 3 = the 7-point extension), never assembled: coefficients are
//           recomputed from the node's position.  Red-black colouring.
//   BoxOp   a 3^d-point operator stored as 3^d coefficient arrays in natural order (no column indices).
//           These are the Galerkin coarse operators A_c = P^T A P of the V-cycle (PETSc -pc_mg_galerkin,
//           src/pc_gamgmc.c:345-349).  2^d colours.  Nodes away from the boundary share one stencil, which is
//           detected at set-up and then read from kernel parameters instead of memory.
//   GridTransfer  matrix-free Q1 restriction / prolongation (PETSc DMDA interpolation, SURVEY Appendix A.4).
//
// Reference loops replaced: src/mc_sor.c:260-268 (+ noise, src/pc_mcgibbs.c:124-126) -> *_sweep_kernel;
// PCMG residual / MatRestrict / MatInterpolateAdd (SURVEY A.3) -> *_residual_kernel, restrict_kernel,
// prolong_kernel; MatPtAP -> galerkin_kernel.  Every kernel keeps the accumulation order of the assembled
// (CSR, ascending column) form, so results are bit-identical to the CSR path and to the oracle.
//
// Partitioning: the grid is split into slabs of the slowest dimension; a rank owns units [slo, shi) (a unit is
// a grid row in 2D, a plane in 3D) and sees one ghost unit on each side through separate ghost buffers.
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "common.hpp"
#include "philox.cuh"
#include "stream2d.cuh"
#include "sweep2d.cuh"
#include "sweep3d.cuh"
#include "sweep3d_ws.cuh"
#include "box_stream.cuh"
#include "box2d.cuh"
#include "box3d.cuh"
#include "tail2d.cuh"

void laplace_assemble(int dim, int64_t nx, int64_t ny, int64_t nz, double kappa, HostCsr &a);
int comm_halo_exchange(pmg_ctx ctx, const double *send_lo, double *recv_lo, const double *send_hi, double *recv_hi, size_t count_lo, size_t count_hi, cudaStream_t stream);
int comm_allgather_i64(pmg_ctx ctx, const int64_t *local_host, int count, int64_t *all_host);
int comm_allgatherv(pmg_ctx ctx, const double *send, double *recv, const int64_t *counts, const int64_t *displs, cudaStream_t stream);

// Work list of the fused 2D sweep (sweep2d.cuh), host only (also exported as pmg_plan_sweep2d for the CPU tests): items of three
// ints (strip of 120 output columns, first row, end row).  Bands of `by` rows (edge strips / bands at the grid boundary, which run the
// table-driven loop, 3/4 of that).  On a slab with the overlapped exchange (`thin_on`) the rows next to a NEIGHBOUR are bands of 8
// rows of their own: they are the only tiles that read ghost rows, and run on the communication stream right behind the exchange.
// Order: tiles that read no ghost row first (`nohalo` of them), the others last; within each group edge tiles before interior tiles.
void sweep2d_plan(int64_t n0, int64_t n1, int64_t slo, int64_t shi, bool parallel, int by, bool restrict_mode, bool thin_on, std::vector<int32_t> &out, int &nohalo_count)
{
  struct It { int32_t s, ja, jb; };
  const int       nstrips = (int)((n0 + sweep2d::STRIP_OUT - 1) / sweep2d::STRIP_OUT);
  std::vector<It> slow, fast;
  const int64_t   thin = 8;
  thin_on = thin_on && parallel && shi - slo >= 4 * thin;
  for (int s = 0; s < nstrips; ++s) {
    const int  c0 = s * sweep2d::STRIP_OUT - 4;
    const bool edge_strip = !(c0 >= 1 && c0 + 127 <= n0 - 2);
    int64_t    j = slo, end = shi;
    if (thin_on && slo > 0) {
      slow.push_back(It{s, (int32_t)j, (int32_t)(j + thin)});
      j += thin;
    }
    if (thin_on && shi < n1) end = shi - thin;
    while (j < end) {
      const int64_t jb_full = std::min<int64_t>(j + by, end);
      const int     lo = restrict_mode ? 4 : 2, hi = restrict_mode ? 2 : 0;
      const bool    interior = !edge_strip && j - lo >= 1 && jb_full + hi <= n1 - 2 && j - lo - 1 >= slo && jb_full + hi + 2 < shi; // sweep2d_kernel's test
      const int64_t h  = interior ? by : std::max(2, (by * 3 / 4) & ~1); // edge warps run the table-driven loop: shorter bands
      const int64_t jb = std::min<int64_t>(j + h, end);
      (interior ? fast : slow).push_back(It{s, (int32_t)j, (int32_t)jb});
      j = jb;
    }
    if (end < shi) slow.push_back(It{s, (int32_t)end, (int32_t)shi});
  }
  std::vector<It> all = slow;
  all.insert(all.end(), fast.begin(), fast.end());
  // a tile reads ghost rows when it reaches within lo / hi rows of a slab end that has a neighbour (rows beyond the GRID are not ghost rows)
  const int lo = restrict_mode ? 5 : 3, hi = restrict_mode ? 3 : 1;
  auto      nohalo = [&](const It &it) { return !parallel || ((it.ja - lo >= slo || slo == 0) && (it.jb + hi < shi || shi == n1)); };
  std::stable_partition(all.begin(), all.end(), nohalo);
  nohalo_count = 0;
  out.clear();
  for (const auto &it : all) {
    nohalo_count += nohalo(it) ? 1 : 0;
    out.push_back(it.s); out.push_back(it.ja); out.push_back(it.jb);
  }
}

// Work list of the fused 3D sweep (sweep3d.cuh), host only (also exported as pmg_plan_sweep3d for the CPU tests): items of
// five ints (strip, ya, ka, kb, narrow).  Strips of 120 output columns; tiles of nw - 2 output rows (narrow last strip of at
// most 56 columns: 2 nw - 2 rows, 16 lanes per grid row); bands along z: `thin` planes where a plane lacks a z neighbour (the
// table-driven tiles), equal bands of at most bz planes between.  Order: edge tiles, interior tiles, thin-band tiles.
void sweep3d_plan(int64_t n0, int64_t n1, int64_t n2, int64_t slo, int64_t shi, int bz, int nw, bool allow_narrow, int thin_planes, std::vector<int32_t> &out)
{
  constexpr int STRIP = sweep3d::STRIP_OUT;
  const int     nstrips = (int)((n0 + STRIP - 1) / STRIP), ty = nw - 2, ty16 = 2 * nw - 2;
  const int64_t last_w = n0 - (int64_t)(nstrips - 1) * STRIP; // columns of the last strip
  const bool    narrow = allow_narrow && last_w <= 56 && n1 >= ty16; // 14 output lanes of 4 columns
  std::vector<std::pair<int64_t, int64_t>> bands;
  {
    const int64_t thin = std::max(2, thin_planes);
    int64_t       lo = slo, hi = shi;
    const bool    edge_lo = slo < 2, edge_hi = shi > n2 - 2; // the slab holds the first / last planes of the grid
    if (shi - slo <= 2 * thin + 2) {
      for (int64_t k = lo; k < hi; k += bz) bands.push_back({k, std::min<int64_t>(k + bz, hi)});
    } else {
      if (edge_lo) { bands.push_back({lo, lo + thin}); lo += thin; }
      if (edge_hi) hi -= thin;
      const int64_t nb = (hi - lo + bz - 1) / bz;
      for (int64_t i = 0; i < nb; ++i) bands.push_back({lo + (hi - lo) * i / nb, lo + (hi - lo) * (i + 1) / nb});
      if (edge_hi) bands.push_back({hi, shi});
    }
  }
  std::vector<int32_t> slow, fast, small;
  for (const auto &bd : bands) {
    const int64_t k = bd.first, kb = bd.second;
    const bool    kin = k - 1 >= 1 && kb <= n2 - 2; // sweep3d_kernel's zconst test (the slab's tensors always hold planes k-2 and kb+1)
    const bool    thinband = kb - k < bz / 2;
    for (int s = 0; s < nstrips; ++s) {
      const bool nar  = narrow && kin && s == nstrips - 1;
      const int  step = nar ? ty16 : ty;
      for (int64_t ya = 0; ya < n1; ya += step) {
        const int  c0 = s * STRIP - 4;
        const bool interior = kin && !nar && c0 >= 1 && c0 + 127 <= n0 - 2 && ya - 1 >= 1 && ya + nw - 2 <= n1 - 2;
        std::vector<int32_t> &dst = thinband ? small : interior ? fast : slow;
        const int32_t         it[5] = {s, (int32_t)ya, (int32_t)k, (int32_t)kb, nar ? 1 : 0};
        dst.insert(dst.end(), it, it + 5);
      }
    }
  }
  out = slow;
  out.insert(out.end(), fast.begin(), fast.end());
  out.insert(out.end(), small.begin(), small.end());
}

namespace {

struct Geom {
  int     dim;
  int64_t n0, n1, n2; // global node counts (n2 = 1 in 2D)
  int64_t slo, shi;   // owned units of the slowest dimension
  int64_t unit;       // nodes per unit
  int64_t nl;         // owned nodes
  int64_t ld;         // row stride of the vectors the kernel indexes: n0 (natural layout) or the pitch of the fused sweeps (pitched())
  __host__ __device__ int64_t nslow() const { return dim == 2 ? n1 : n2; }
  __host__ __device__ int64_t row0() const { return unit * slo; }
};

Geom make_geom(int dim, const int64_t n[3], int64_t slo, int64_t shi)
{
  Geom g;
  g.dim  = dim;
  g.n0   = n[0];
  g.n1   = n[1];
  g.n2   = dim == 3 ? n[2] : 1;
  g.slo  = slo;
  g.shi  = shi;
  g.unit = dim == 2 ? g.n0 : g.n0 * g.n1;
  g.nl   = g.unit * (shi - slo);
  g.ld   = g.n0;
  return g;
}
// the same grid over PITCHED vectors (row stride `pitch`, no ghost units): for the kernels that index through ld / unit / nl
Geom pitched(Geom g, int64_t pitch)
{
  g.ld   = pitch;
  g.unit = g.dim == 2 ? pitch : pitch * g.n1;
  g.nl   = g.unit * (g.shi - g.slo);
  return g;
}

// value of vector entry at local index q, which may lie one unit below / above the owned range
__device__ __forceinline__ double ldg(const double *__restrict__ x, const double *__restrict__ glo, const double *__restrict__ ghi, int64_t q, const Geom &g)
{
  if (q < 0) return glo[q + g.unit];
  if (q >= g.nl) return ghi[q - g.nl];
  return x[q];
}

struct LapTab { // indexed by the number of existing neighbours
  double diag[7], idiag[7], sqrtdiag[7];
  double h;
};

// Launch geometry of the per-node kernels: x runs along the fastest grid dimension, y over grid rows, z over planes, so
// that no thread has to recover (i, j, k) from a linear index with 64-bit divisions (which used to cost more than the
// stencil itself).  Thread (tx, ty) of block (bx, by, bz): position tx + bx*blockDim.x in the row, row ty + by*blockDim.y.
struct Plan {
  dim3 grid, block;
};
static Plan plan3(int64_t ni, int64_t nrows, int64_t nplanes)
{
  // the block width (a multiple of 32, at most 256) that wastes the fewest threads on this row length: the grids of the
  // Q1 hierarchy have 2^k + 1 nodes per direction, which a power-of-two width covers at 50 % in the worst case
  unsigned bx = 32;
  int64_t  best = -1;
  for (unsigned c = 32; c <= 256; c += 32) {
    const int64_t slots = (ni + c - 1) / c * c;
    if (best < 0 || slots <= best) { best = slots; bx = c; }
  }
  const unsigned by = 256 / bx;
  Plan           p;
  p.block = dim3(bx, by, 1);
  p.grid  = dim3((unsigned)std::max<int64_t>(1, (ni + bx - 1) / bx), (unsigned)std::max<int64_t>(1, (nrows + by - 1) / by), (unsigned)std::max<int64_t>(1, nplanes));
  return p;
}
static bool plan_ok(const Plan &p) { return p.grid.y <= 65535u && p.grid.z <= 65535u; }
#define PMG_PLAN_CHECK(p) \
  if (!plan_ok(p)) PMG_FAIL(PMG_ERR_SUP, "grid too large for one launch (%u x %u x %u blocks)", (p).grid.x, (p).grid.y, (p).grid.z)

// node of this thread under plan3(n0, rows, planes): all owned nodes, natural order
template <int DIM> __device__ __forceinline__ bool node_of_thread(const Geom &g, int64_t &i, int64_t &j, int64_t &k, int64_t &idx)
{
  i                = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t rj = (int64_t)blockIdx.y * blockDim.y + threadIdx.y;
  if (i >= g.n0) return false;
  if (DIM == 2) {
    if (rj >= g.shi - g.slo) return false;
    j   = g.slo + rj;
    k   = 0;
    idx = i + g.ld * rj;
  } else {
    if (rj >= g.n1) return false;
    j   = rj;
    k   = g.slo + blockIdx.z;
    idx = i + g.ld * (rj + g.n1 * (int64_t)blockIdx.z);
  }
  return true;
}
template <int DIM> static Plan plan_nodes(const Geom &g) { return DIM == 2 ? plan3(g.n0, g.shi - g.slo, 1) : plan3(g.n0, g.n1, g.shi - g.slo); }

template <int DIM> __device__ __forceinline__ void decode(const Geom &g, int64_t idx, int64_t &i, int64_t &j, int64_t &k)
{
  i               = idx % g.n0;
  const int64_t r = idx / g.n0;
  if (DIM == 2) {
    j = g.slo + r;
    k = 0;
  } else {
    j = r % g.n1;
    k = g.slo + r / g.n1;
  }
}

// ---- TMA descriptors ---------------------------------------------------------------------------------
// cuTensorMapEncodeTiled through the runtime's driver entry point (no libcuda link dependency)
typedef CUresult (*pfn_tensor_map_encode_tiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static pfn_tensor_map_encode_tiled tensor_map_encoder()
{
  static pfn_tensor_map_encode_tiled fn = [] {
    void                           *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
    return (pfn_tensor_map_encode_tiled)p;
  }();
  return fn;
}
// FP64 tensor of `rank` dimensions (dims[0] fastest, strides in elements for dims 1..), box in elements; out-of-range
// coordinates read as zero
static int make_tensor_map(CUtensorMap &tm, const double *base, int rank, const int64_t *dims, const int64_t *strides, const int *box, bool swizzle32 = false)
{
  pfn_tensor_map_encode_tiled enc = tensor_map_encoder();
  if (!enc) PMG_FAIL(PMG_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  cuuint64_t gd[5], gs[5];
  cuuint32_t bx[5], es[5];
  for (int d = 0; d < rank; ++d) {
    gd[d] = (cuuint64_t)dims[d];
    bx[d] = (cuuint32_t)box[d];
    es[d] = 1;
    if (d > 0) gs[d - 1] = (cuuint64_t)strides[d] * sizeof(double);
  }
  const CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, (cuuint32_t)rank, (void *)base, gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) PMG_FAIL(PMG_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return 0;
}

// ---- LapOp kernels -----------------------------------------------------------------------------------
// one thread per node of the colour; nodes of a colour in a grid row are i = s, s+2, ...
template <int DIM> __global__ void __launch_bounds__(256) lap_sweep_kernel(Geom g, int color, LapTab tab, double omo, const double *__restrict__ b, double *__restrict__ x, const double *__restrict__ glo, const double *__restrict__ ghi, NoiseArgs na)
{
  const int64_t kk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t rj = (int64_t)blockIdx.y * blockDim.y + threadIdx.y; // 2D: local grid row; 3D: j
  int64_t       j, k, row;
  if (DIM == 2) {
    if (rj >= g.shi - g.slo) return;
    j   = g.slo + rj;
    k   = 0;
    row = rj;
  } else {
    if (rj >= g.n1) return;
    j   = rj;
    k   = g.slo + blockIdx.z;
    row = rj + g.n1 * blockIdx.z;
  }
  const int64_t i = 2 * kk + ((color + j + k) & 1);
  if (i >= g.n0) return;
  const int64_t idx = i + g.n0 * row;
  const bool    W = i > 0, E = i < g.n0 - 1, S = j > 0, N = j < g.n1 - 1, D = DIM == 3 && k > 0, U = DIM == 3 && k < g.n2 - 1;
  const int     deg = (int)W + (int)E + (int)S + (int)N + (int)D + (int)U;
  const double  h   = tab.h;
  const uint64_t nid = (uint64_t)(((DIM == 3 ? k * g.n1 : 0) + j) * ((g.n0 + 3) & ~(int64_t)3) + i); // padded index (philox.cuh)
  double         sum = noisy_rhs_id(na, idx, nid, tab.sqrtdiag[deg], b ? b[idx] : 0.0);
  // ascending column order of the assembled row: down, south, west | east, north, up; off-diagonal value -h
  if (DIM == 3) {
    if (D) sum = fma(h, ldg(x, glo, ghi, idx - g.unit, g), sum);
    if (S) sum = fma(h, x[idx - g.n0], sum);
  } else {
    if (S) sum = fma(h, ldg(x, glo, ghi, idx - g.n0, g), sum);
  }
  if (W) sum = fma(h, x[idx - 1], sum);
  if (E) sum = fma(h, x[idx + 1], sum);
  if (DIM == 3) {
    if (N) sum = fma(h, x[idx + g.n0], sum);
    if (U) sum = fma(h, ldg(x, glo, ghi, idx + g.unit, g), sum);
  } else {
    if (N) sum = fma(h, ldg(x, glo, ghi, idx + g.n0, g), sum);
  }
  const double t0 = __dmul_rn(omo, x[idx]);
  x[idx]          = fma(tab.idiag[deg], sum, t0);
}

// out = b - A x (residual) or A x (mult)
template <int DIM, bool RESIDUAL> __global__ void __launch_bounds__(256) lap_apply_kernel(Geom g, LapTab tab, const double *__restrict__ b, const double *__restrict__ x, const double *__restrict__ glo, const double *__restrict__ ghi, double *__restrict__ out)
{
  int64_t i, j, k, idx;
  if (!node_of_thread<DIM>(g, i, j, k, idx)) return;
  const bool   W = i > 0, E = i < g.n0 - 1, S = j > 0, N = j < g.n1 - 1, D = DIM == 3 && k > 0, U = DIM == 3 && k < g.n2 - 1;
  const int    deg = (int)W + (int)E + (int)S + (int)N + (int)D + (int)U;
  const double mh  = -tab.h;
  double       ax  = 0.0;
  if (DIM == 3) {
    if (D) ax = fma(mh, ldg(x, glo, ghi, idx - g.unit, g), ax);
    if (S) ax = fma(mh, x[idx - g.ld], ax);
  } else {
    if (S) ax = fma(mh, ldg(x, glo, ghi, idx - g.ld, g), ax);
  }
  if (W) ax = fma(mh, x[idx - 1], ax);
  ax = fma(tab.diag[deg], x[idx], ax);
  if (E) ax = fma(mh, x[idx + 1], ax);
  if (DIM == 3) {
    if (N) ax = fma(mh, x[idx + g.ld], ax);
    if (U) ax = fma(mh, ldg(x, glo, ghi, idx + g.unit, g), ax);
  } else {
    if (N) ax = fma(mh, ldg(x, glo, ghi, idx + g.ld, g), ax);
  }
  out[idx] = RESIDUAL ? __dsub_rn(b[idx], ax) : ax;
}

// ---- finest 3D level of the fused V-cycle: the same residual and prolongation on PITCHED vectors, four columns per thread
// (one 32-byte segment: 256-bit loads and stores, a quarter of the load instructions of the per-node kernels; the
// arithmetic per node is lap_apply_kernel<3, true>'s and prolong_kernel<3>'s, fma for fma).  Undistributed levels only.
__device__ __forceinline__ void ldg256(const double *p, double (&v)[4]) { asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]) : "l"(p)); }
__device__ __forceinline__ void ld256(const double *p, double (&v)[4]) { asm volatile("ld.global.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]) : "l"(p) : "memory"); }
__device__ __forceinline__ void stg256(double *p, const double (&v)[4]) { asm volatile("st.global.v4.f64 [%4], {%0,%1,%2,%3};" ::"d"(v[0]), "d"(v[1]), "d"(v[2]), "d"(v[3]), "l"(p) : "memory"); }
// thread -> (quad t of the row, row j, plane k)
__device__ __forceinline__ bool quad_of_thread(const Geom &g, int nq, int &t, int &j, int &k)
{
  const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= (unsigned)nq * (unsigned)g.n1) return false;
  j = (int)(q / (unsigned)nq);
  t = (int)(q - (unsigned)j * (unsigned)nq);
  k = (int)blockIdx.y;
  return true;
}
__global__ void __launch_bounds__(256) lap_residual3_pitched_kernel(Geom g, LapTab tab, const double *__restrict__ b, const double *__restrict__ x, double *__restrict__ out)
{
  const int nq = (int)(g.ld >> 2);
  int       t, j, kl;
  if (!quad_of_thread(g, nq, t, j, kl)) return; // kl: plane of the slab (the vectors start at the first owned plane, ghost planes in place around them)
  const int     k   = kl + (int)g.slo;
  const int64_t idx = 4 * (int64_t)t + g.ld * ((int64_t)j + g.n1 * (int64_t)kl);
  const bool    S = j > 0, N = j < g.n1 - 1, D = k > 0, U = k < g.n2 - 1;
  double        xc[4], xs[4] = {0, 0, 0, 0}, xn[4] = {0, 0, 0, 0}, xd[4] = {0, 0, 0, 0}, xu[4] = {0, 0, 0, 0}, bb[4], r[4];
  ldg256(x + idx, xc);
  ldg256(b + idx, bb);
  if (S) ldg256(x + idx - g.ld, xs);
  if (N) ldg256(x + idx + g.ld, xn);
  if (D) ldg256(x + idx - g.unit, xd);
  if (U) ldg256(x + idx + g.unit, xu);
  const int    i0 = 4 * t;
  const double xw = i0 > 0 ? __ldg(x + idx - 1) : 0.0, xe = i0 + 4 < g.n0 ? __ldg(x + idx + 4) : 0.0;
  const double mh = -tab.h;
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    const int  i = i0 + m;
    const bool W = i > 0, E = i < g.n0 - 1;
    const int  deg = (int)W + (int)E + (int)S + (int)N + (int)D + (int)U;
    double     ax  = 0.0;
    if (D) ax = fma(mh, xd[m], ax);
    if (S) ax = fma(mh, xs[m], ax);
    if (W) ax = fma(mh, m == 0 ? xw : xc[m == 0 ? 0 : m - 1], ax);
    ax = fma(tab.diag[deg], xc[m], ax);
    if (E) ax = fma(mh, m == 3 ? xe : xc[m == 3 ? 3 : m + 1], ax);
    if (N) ax = fma(mh, xn[m], ax);
    if (U) ax = fma(mh, xu[m], ax);
    r[m] = i < g.n0 ? __dsub_rn(bb[m], ax) : 0.0;
  }
  stg256(out + idx, r);
}
__global__ void __launch_bounds__(256) prolong3_pitched_kernel(Geom gf, Geom gc, const double *__restrict__ xc, const double *__restrict__ clo, const double *__restrict__ chi, double *__restrict__ xf)
{
  const int nq = (int)(gf.ld >> 2);
  int       t, j, kl;
  if (!quad_of_thread(gf, nq, t, j, kl)) return; // kl: plane of the fine slab; xc holds the coarse slab, clo / chi the coarse planes below / above it
  const int     k   = kl + (int)gf.slo;
  const int64_t idx = 4 * (int64_t)t + gf.ld * ((int64_t)j + gf.n1 * (int64_t)kl);
  double        s[4];
  ld256(xf + idx, s);
  const int cj = (j & 1) ? 2 : 1, ck = (k & 1) ? 2 : 1;
  const int J0 = j >> 1, K0 = k >> 1, I0 = 2 * t; // coarse columns I0, I0 + 1, I0 + 2 serve the four fine columns
  for (int c = 0; c < ck; ++c) { // prolong_kernel's order: K, then J, then I ascending
    const int K = K0 + c;
    if (K >= gc.n2) continue;
    for (int bq = 0; bq < cj; ++bq) {
      const int J = J0 + bq;
      if (J >= gc.n1) continue;
      const double *row = K < gc.slo ? clo + gc.ld * (int64_t)J : (K >= gc.shi ? chi + gc.ld * (int64_t)J : xc + gc.ld * ((int64_t)J + gc.n1 * (int64_t)(K - gc.slo)));
      const double  v0 = I0 < gc.n0 ? __ldg(row + I0) : 0.0, v1 = I0 + 1 < gc.n0 ? __ldg(row + I0 + 1) : 0.0, v2 = I0 + 2 < gc.n0 ? __ldg(row + I0 + 2) : 0.0;
      const double  we = (cj == 2 ? 0.5 : 1.0) * (ck == 2 ? 0.5 : 1.0), wo = 0.5 * (cj == 2 ? 0.5 : 1.0) * (ck == 2 ? 0.5 : 1.0); // even / odd fine column
      if (I0 < gc.n0) s[0] = fma(we, v0, s[0]);
      if (I0 < gc.n0) s[1] = fma(wo, v0, s[1]);
      if (I0 + 1 < gc.n0) s[1] = fma(wo, v1, s[1]);
      if (I0 + 1 < gc.n0) s[2] = fma(we, v1, s[2]);
      if (I0 + 1 < gc.n0) s[3] = fma(wo, v1, s[3]);
      if (I0 + 2 < gc.n0) s[3] = fma(wo, v2, s[3]);
    }
  }
#pragma unroll
  for (int m = 0; m < 4; ++m)
    if (4 * t + m >= gf.n0) s[m] = 0.0; // pad columns stay zero
  stg256(xf + idx, s);
}

// b_c = P^T r for a pitched fine residual: four coarse nodes per thread (fine columns 8t-1 .. 8t+7 of each of the 9 fine rows:
// two 256-bit loads and one scalar), restrict_kernel<3>'s accumulation order (k, j, i ascending) per coarse node
__global__ void __launch_bounds__(256) restrict3_pitched_kernel(Geom gf, Geom gc, const double *__restrict__ r, double *__restrict__ bc)
{
  const int      nqc = (int)((gc.n0 + 3) >> 2);
  const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= (unsigned)nqc * (unsigned)gc.n1) return;
  const int J = (int)(q / (unsigned)nqc), t = (int)(q - (unsigned)J * (unsigned)nqc), Kl = (int)blockIdx.y, K = Kl + (int)gc.slo; // Kl: plane of the coarse slab
  double    acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
  for (int dk = -1; dk <= 1; ++dk) {
    const int k = 2 * K + dk;
    if (k < 0 || k >= gf.n2) continue;
#pragma unroll
    for (int dj = -1; dj <= 1; ++dj) {
      const int j = 2 * J + dj;
      if (j < 0 || j >= gf.n1) continue;
      const double *row = r + gf.ld * ((int64_t)j + gf.n1 * (int64_t)(k - gf.slo)); // r starts at the first owned fine plane; planes slo-1 / shi are its ghost planes, in place
      const int     i0 = 8 * t; // fine column of the thread's first coarse node
      double        v[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}; // fine columns i0-1 .. i0+7; columns >= ld are not loaded
      if (i0 > 0) v[0] = __ldg(row + i0 - 1);
      {
        double a[4];
        ldg256(row + i0, a);
        v[1] = a[0]; v[2] = a[1]; v[3] = a[2]; v[4] = a[3];
      }
      if (i0 + 4 < gf.ld) {
        double a[4];
        ldg256(row + i0 + 4, a);
        v[5] = a[0]; v[6] = a[1]; v[7] = a[2]; v[8] = a[3];
      }
      const double wjk = (dj ? 0.5 : 1.0) * (dk ? 0.5 : 1.0);
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const int ic = i0 + 2 * m; // fine column of coarse node 4t + m
        if (ic - 1 >= 0 && ic - 1 < gf.n0) acc[m] = fma(0.5 * wjk, v[2 * m], acc[m]);
        if (ic < gf.n0) acc[m] = fma(wjk, v[2 * m + 1], acc[m]);
        if (ic + 1 < gf.n0) acc[m] = fma(0.5 * wjk, v[2 * m + 2], acc[m]);
      }
    }
  }
#pragma unroll
  for (int m = 0; m < 4; ++m)
    if (4 * t + m < gc.n0) bc[4 * t + m + gc.ld * ((int64_t)J + gc.n1 * (int64_t)Kl)] = acc[m];
}

// the four-columns-per-thread transfers above on a slab pair: pitched fine vectors (row stride a multiple of 4) with their ghost
// planes in place, coarse vectors in the natural layout with rows short enough for one launch
static bool pitched3_slab_ok(const Geom &gf, const Geom &gc)
{
  return gf.dim == 3 && (gf.ld & 3) == 0 && gf.shi > gf.slo && gc.shi > gc.slo && gc.shi - gc.slo <= 65535 && gf.shi - gf.slo <= 65535 && !std::getenv("PMG_NO_PITCHED3_SLAB");
}

// natural (row stride n0) <-> pitched (row stride pitch) copies of a 2D slab
template <bool TO_PITCHED> __global__ void __launch_bounds__(256) repitch_kernel(int64_t n0, int64_t rows, int64_t pitch, const double *__restrict__ src, double *__restrict__ dst)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, ry = (int64_t)blockIdx.y * blockDim.y + threadIdx.y;
  if (i >= n0 || ry >= rows) return;
  const int64_t r = ry + rows * (int64_t)blockIdx.z; // rows = grid rows per plane (2D: one plane)
  if (TO_PITCHED) dst[r * pitch + i] = src[r * n0 + i];
  else dst[r * n0 + i] = src[r * pitch + i];
}

// ---- BoxOp kernels -------------------------------------------------------------------------------------
struct BoxConst { // the shared interior stencil
  double c[27];
  double idiag, sqrtdiag;
  int    on, ring;
};

template <int DIM> __device__ __forceinline__ bool box_interior(const Geom &g, const BoxConst &bc, int64_t i, int64_t j, int64_t k)
{
  if (!bc.on) return false;
  const int64_t r = bc.ring;
  bool in = i >= r && i < g.n0 - r && j >= r && j < g.n1 - r;
  if (DIM == 3) in = in && k >= r && k < g.n2 - r;
  return in;
}

// sum_{s != centre, ascending} (sign) c_s x[q_s] accumulated into acc with fma; INCLUDE_CENTRE adds the diagonal in place
template <int DIM, bool NEG, bool INCLUDE_CENTRE, bool CG = false> // CG: x is read with ld.global.cg (written by other SMs in the same launch)
__device__ __forceinline__ double box_row(const Geom &g, const BoxConst &bc, const double *__restrict__ coef, int64_t stride, const double *__restrict__ x, const double *__restrict__ glo, const double *__restrict__ ghi, int64_t idx, int64_t i, int64_t j, int64_t k, double acc)
{
  constexpr int NST = DIM == 2 ? 9 : 27;
  const bool    interior = box_interior<DIM>(g, bc, i, j, k);
  if constexpr (DIM == 2) {
    // 9-point: all loads are issued before the first fma.  The accumulation is one dependent chain, and with loads and fmas
    // interleaved term by term a warp pays one memory latency per term (ncu: long-scoreboard stalls on the DFMAs; the
    // boundary lane of every grid row holds up its whole warp).  Same terms, same order.  Measured: 2D V-cycle -1 %; the
    // 27-point version of this (nine terms at a time) cost occupancy and was 4 % slower, so 3D keeps the interleaved loop.
    double v[9], c[9];
    bool   ex[9];
#pragma unroll
    for (int s = 0; s < 9; ++s) {
      const int     di = s % 3 - 1, dj = s / 3 - 1;
      const int64_t q = idx + di + g.n0 * dj;
      ex[s] = (INCLUDE_CENTRE || s != 4) && (interior || (i + di >= 0 && i + di < g.n0 && j + dj >= 0 && j + dj < g.n1));
      v[s]  = 0.0;
      c[s]  = 0.0;
      if (ex[s]) {
        v[s] = CG ? __ldcg(x + q) : ldg(x, glo, ghi, q, g);
        if (!interior) c[s] = coef[(int64_t)s * stride + idx];
      }
    }
#pragma unroll
    for (int s = 0; s < 9; ++s) {
      const double cc = interior ? bc.c[s] : c[s];
      if (ex[s]) acc = fma(NEG ? -cc : cc, v[s], acc); // structurally absent entries are skipped, not added as zeros
    }
    return acc;
  } else {
#pragma unroll
  for (int s = 0; s < NST; ++s) {
    if (!INCLUDE_CENTRE && s == NST / 2) continue;
    const int di = s % 3 - 1, dj = (s / 3) % 3 - 1, dk = DIM == 3 ? s / 9 - 1 : 0;
    const int64_t q = idx + di + g.n0 * dj + (DIM == 3 ? g.unit * dk : 0);
    double        c, v;
    if (interior) {
      c = bc.c[s];
      v = CG ? __ldcg(x + q) : ldg(x, glo, ghi, q, g);
    } else {
      const bool ex = i + di >= 0 && i + di < g.n0 && j + dj >= 0 && j + dj < g.n1 && (DIM == 2 || (k + dk >= 0 && k + dk < g.n2));
      if (!ex) continue; // structurally absent entry
      c = coef[(int64_t)s * stride + idx];
      v = CG ? __ldcg(x + q) : ldg(x, glo, ghi, q, g);
    }
    acc = fma(NEG ? -c : c, v, acc);
  }
  return acc;
  }
}

// node of this thread among the nodes of one colour, under box_colour_plan
template <int DIM> __device__ __forceinline__ bool box_colour_node(const Geom &g, int color, int64_t &idx, int64_t &i, int64_t &j, int64_t &k)
{
  const int     ci = color & 1, cj = (color >> 1) & 1, ck = (color >> 2) & 1;
  const int64_t tx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, ty = (int64_t)blockIdx.y * blockDim.y + threadIdx.y;
  i = 2 * tx + ci;
  if (i >= g.n0) return false;
  if (DIM == 2) {
    j = g.slo + ((cj ^ g.slo) & 1) + 2 * ty;
    if (j >= g.shi) return false;
    k   = 0;
    idx = i + g.n0 * (j - g.slo);
  } else {
    j = 2 * ty + cj;
    k = g.slo + ((ck ^ g.slo) & 1) + 2 * (int64_t)blockIdx.z;
    if (j >= g.n1 || k >= g.shi) return false;
    idx = i + g.n0 * (j + g.n1 * (k - g.slo));
  }
  return true;
}
template <int DIM> static Plan box_colour_plan(const Geom &g) { return DIM == 2 ? plan3((g.n0 + 1) / 2, (g.shi - g.slo + 1) / 2, 1) : plan3((g.n0 + 1) / 2, (g.n1 + 1) / 2, (g.shi - g.slo + 1) / 2); }

template <int DIM> __global__ void __launch_bounds__(256) box_sweep_kernel(Geom g, int color, const double *__restrict__ coef, int64_t stride, BoxConst bc, const double *__restrict__ idiag, const double *__restrict__ sqrtdiag, double omo, const double *__restrict__ b, double *__restrict__ x, const double *__restrict__ glo, const double *__restrict__ ghi, NoiseArgs na)
{
  int64_t idx, i, j, k;
  if (!box_colour_node<DIM>(g, color, idx, i, j, k)) return;
  const bool   interior = box_interior<DIM>(g, bc, i, j, k);
  const double   sq = interior ? bc.sqrtdiag : sqrtdiag[idx], id = interior ? bc.idiag : idiag[idx];
  const uint64_t nid = (uint64_t)(((DIM == 3 ? k * g.n1 : 0) + j) * ((g.n0 + 3) & ~(int64_t)3) + i); // padded index (philox.cuh)
  double         sum = noisy_rhs_id(na, idx, nid, sq, b ? b[idx] : 0.0);
  sum                = box_row<DIM, true, false>(g, bc, coef, stride, x, glo, ghi, idx, i, j, k, sum);
  const double t0  = __dmul_rn(omo, x[idx]);
  x[idx]           = fma(id, sum, t0);
}

// Two colours of the 27-point sweep that differ only in the x parity (c = ci + 2 cj + 4 ck and c + 1) live on the SAME grid rows,
// and no other row of their nine-row neighbourhood changes while they are swept.  One block per grid row stages the nine rows
// in shared memory (coalesced, each value fetched once for both colours), updates the nodes of the first colour, publishes them
// in the staged centre row, and updates the second colour from it: 4 launches per sweep instead of 8, unit-stride global loads
// instead of stride-2 gathers, and one Philox / Box-Muller call per node PAIR (columns 2t, 2t+1 are the cos / sin halves of one
// generator call, philox.cuh).  Arithmetic per node is box_sweep_kernel<3>'s, fma for fma.  Undistributed levels with rows of at
// most 512 nodes.
__global__ void __launch_bounds__(256) box_pair_sweep3_kernel(Geom g, int cjk, int backward, const double *__restrict__ coef, int64_t stride, BoxConst bc, const double *__restrict__ idiag, const double *__restrict__ sqrtdiag, double omo,
                                                              const double *__restrict__ b, double *__restrict__ x, NoiseArgs na)
{
  extern __shared__ double prow[]; // [9][n0 + 2]: row (dj + 1) + 3 (dk + 1), column i at index i + 1
  const int j = 2 * (int)blockIdx.x + (cjk & 1), k = 2 * (int)blockIdx.y + (cjk >> 1);
  if (j >= g.n1 || k >= g.n2) return;
  const int n0 = (int)g.n0, ldr = n0 + 2;
  { // all 18 loads of a thread are issued before the first store (2 blockDim.x >= n0: two elements per thread and row)
    const int i0 = threadIdx.x, i1 = threadIdx.x + blockDim.x;
    double    v[18];
#pragma unroll
    for (int r = 0; r < 9; ++r) {
      const int     jj = j + r % 3 - 1, kk = k + r / 3 - 1;
      const bool    ok = jj >= 0 && jj < g.n1 && kk >= 0 && kk < g.n2; // absent rows are never read
      const double *src = x + g.n0 * ((int64_t)(ok ? jj : j) + g.n1 * (int64_t)(ok ? kk : k));
      v[2 * r]     = i0 < n0 ? src[i0] : 0.0;
      v[2 * r + 1] = i1 < n0 ? src[i1] : 0.0;
    }
#pragma unroll
    for (int r = 0; r < 9; ++r) {
      if (i0 < n0) prow[r * ldr + 1 + i0] = v[2 * r];
      if (i1 < n0) prow[r * ldr + 1 + i1] = v[2 * r + 1];
    }
  }
  __syncthreads();
  const int     t = threadIdx.x;
  const int64_t row0 = g.n0 * ((int64_t)j + g.n1 * (int64_t)k);
  // the pair's two normals: one generator call (rows 4q, 4q+1 -> (w0, w1), rows 4q+2, 4q+3 -> (w2, w3); cos for the even row)
  double z0 = 0.0, z1 = 0.0;
  if (2 * t < n0) {
    if (na.mode == PMG_NOISE_INJECTED) {
      z0 = na.tape[row0 + 2 * t];
      if (2 * t + 1 < n0) z1 = na.tape[row0 + 2 * t + 1];
    } else if (na.mode == PMG_NOISE_PHILOX) {
      const uint64_t nid = (uint64_t)(((int64_t)k * g.n1 + j) * ((g.n0 + 3) & ~(int64_t)3) + 2 * t);
      uint32_t       w0, w1, w2, w3;
      philox4x32_10((uint32_t)(nid >> 2), (uint32_t)(nid >> 34), (uint32_t)na.call, (uint32_t)(na.call >> 32), (uint32_t)na.seed, (uint32_t)(na.seed >> 32), w0, w1, w2, w3);
      if (nid & 2) box_muller_32(w2, w3, z0, z1);
      else box_muller_32(w0, w1, z0, z1);
    }
  }
  auto node = [&](int p) {
    const int i = 2 * t + p;
    if (i >= n0) return;
    const int64_t idx = row0 + i;
    const bool    interior = box_interior<3>(g, bc, i, j, k);
    const double  sq = interior ? bc.sqrtdiag : sqrtdiag[idx], id = interior ? bc.idiag : idiag[idx];
    const double  bv = b ? b[idx] : 0.0;
    double        sum = na.mode == PMG_NOISE_NONE ? bv : __dadd_rn(__dmul_rn(p ? z1 : z0, sq), bv); // noisy_rhs_id
    if (interior) {
#pragma unroll
      for (int s = 0; s < 27; ++s) {
        if (s == 13) continue;
        const int di = s % 3 - 1, dj = (s / 3) % 3 - 1, dk = s / 9 - 1;
        sum          = fma(-bc.c[s], prow[((dj + 1) + 3 * (dk + 1)) * ldr + 1 + i + di], sum);
      }
    } else {
      // the one or two boundary nodes of an interior row sit in a warp whose other lanes wait for them: all coefficient loads
      // are issued before the first use (one memory latency instead of 26 dependent ones)
      double cf[27];
#pragma unroll
      for (int s = 0; s < 27; ++s) {
        const int  di = s % 3 - 1, dj = (s / 3) % 3 - 1, dk = s / 9 - 1;
        const bool ex = s != 13 && i + di >= 0 && i + di < n0 && j + dj >= 0 && j + dj < g.n1 && k + dk >= 0 && k + dk < g.n2;
        cf[s]         = ex ? coef[(int64_t)s * stride + idx] : 0.0;
      }
#pragma unroll
      for (int s = 0; s < 27; ++s) {
        if (s == 13) continue;
        const int  di = s % 3 - 1, dj = (s / 3) % 3 - 1, dk = s / 9 - 1;
        const bool ex = i + di >= 0 && i + di < n0 && j + dj >= 0 && j + dj < g.n1 && k + dk >= 0 && k + dk < g.n2;
        if (ex) sum = fma(-cf[s], prow[((dj + 1) + 3 * (dk + 1)) * ldr + 1 + i + di], sum); // structurally absent entries are skipped
      }
    }
    const double t0 = __dmul_rn(omo, prow[4 * ldr + 1 + i]);
    const double xn = fma(id, sum, t0);
    x[idx]                = xn;
    prow[4 * ldr + 1 + i] = xn;
  };
  node(backward ? 1 : 0);
  __syncthreads();
  node(backward ? 0 : 1);
}

template <int DIM, bool RESIDUAL> __global__ void __launch_bounds__(256) box_apply_kernel(Geom g, const double *__restrict__ coef, int64_t stride, BoxConst bc, const double *__restrict__ b, const double *__restrict__ x, const double *__restrict__ glo, const double *__restrict__ ghi, double *__restrict__ out)
{
  int64_t i, j, k, idx;
  if (!node_of_thread<DIM>(g, i, j, k, idx)) return;
  const double ax = box_row<DIM, false, true>(g, bc, coef, stride, x, glo, ghi, idx, i, j, k, 0.0);
  out[idx]        = RESIDUAL ? __dsub_rn(b[idx], ax) : ax;
}

template <int DIM> __global__ void box_coeffs_kernel(Geom g, const double *__restrict__ coef, int64_t stride, double omega, double f, double *__restrict__ idiag, double *__restrict__ sqrtdiag)
{
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= g.nl) return;
  const double d = coef[(int64_t)(DIM == 2 ? 4 : 13) * stride + idx];
  idiag[idx]     = __dmul_rn(__ddiv_rn(1.0, d), omega);
  sqrtdiag[idx]  = __dmul_rn(sqrt(fabs(d)), f);
}

// counts nodes of the interior (ring) whose stencil differs bitwise from the reference node's
template <int DIM> __global__ void box_uniform_kernel(Geom g, const double *__restrict__ coef, int64_t stride, int ring, int64_t ref_idx, unsigned long long *__restrict__ mismatches)
{
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= g.nl) return;
  int64_t i, j, k;
  decode<DIM>(g, idx, i, j, k);
  bool in = i >= ring && i < g.n0 - ring && j >= ring && j < g.n1 - ring;
  if (DIM == 3) in = in && k >= ring && k < g.n2 - ring;
  if (!in) return;
  constexpr int NST = DIM == 2 ? 9 : 27;
  bool          same = true;
  for (int s = 0; s < NST; ++s) same = same && (__double_as_longlong(coef[(int64_t)s * stride + idx]) == __double_as_longlong(coef[(int64_t)s * stride + ref_idx]));
  if (!same) atomicAdd(mismatches, 1ull);
}

// boundary classes of a 2D stencil-array level (box2d.cuh): class of a node = (row class, column class), each first /
// interior / last; counts the nodes whose nine coefficients differ bitwise from their class representative's
struct BoxClassTab {
  double c[9][9]; // [3 row class + column class][stencil entry]
};
__global__ void box_class_kernel(Geom g, const double *__restrict__ coef, int64_t stride, BoxClassTab t, unsigned long long *__restrict__ mismatches)
{
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= g.nl) return;
  const int64_t i = idx % g.n0, j = g.slo + idx / g.n0; // global row
  const int     cc = i == 0 ? 0 : (i == g.n0 - 1 ? 2 : 1), rc = j == 0 ? 0 : (j == g.n1 - 1 ? 2 : 1);
  bool          same = true;
  for (int s = 0; s < 9; ++s) same = same && (__double_as_longlong(coef[(int64_t)s * stride + idx]) == __double_as_longlong(t.c[3 * rc + cc][s]));
  if (!same) atomicAdd(mismatches, 1ull);
}

// the 3D analogue for the plane kernels (box3d.cuh): class = (x class, y class, z class); `raw` holds the 27 x 27 coefficients
struct BoxClass3Raw {
  double c[27][27]; // [cx + 3 cy + 9 cz][stencil entry]
};
__global__ void box_class3_gather_kernel(Geom g, const double *__restrict__ coef, int64_t stride, const int64_t *__restrict__ rep, double *__restrict__ out)
{
  const int q = blockIdx.x, s = threadIdx.x; // class q, entry s
  if (s < 27 && rep[q] >= 0) out[27 * q + s] = coef[(int64_t)s * stride + rep[q]];
}
__global__ void box_class3_check_kernel(Geom g, const double *__restrict__ coef, int64_t stride, const double *__restrict__ tab, unsigned long long *__restrict__ mismatches)
{
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= g.nl) return;
  int64_t i, j, k;
  decode<3>(g, idx, i, j, k);
  const int cx = i == 0 ? 0 : (i == g.n0 - 1 ? 2 : 1), cy = j == 0 ? 0 : (j == g.n1 - 1 ? 2 : 1), cz = k == 0 ? 0 : (k == g.n2 - 1 ? 2 : 1);
  const double *t = tab + 27 * (cx + 3 * cy + 9 * cz);
  bool          same = true;
  for (int s = 0; s < 27; ++s) {
    const int  di = s % 3 - 1, dj = (s / 3) % 3 - 1, dk = s / 9 - 1;
    const bool ex = i + di >= 0 && i + di < g.n0 && j + dj >= 0 && j + dj < g.n1 && k + dk >= 0 && k + dk < g.n2;
    // structurally absent entries are never read by the per-node kernels: the class table holds zeros for them
    same = same && (ex ? __double_as_longlong(coef[(int64_t)s * stride + idx]) == __double_as_longlong(t[s]) : true);
  }
  if (!same) atomicAdd(mismatches, 1ull);
}

// ---- Q1 transfers (SURVEY Appendix A.4) -------------------------------------------------------------------
// coarse node I sits on fine node 2I; nc = (nf + 1)/2 per direction
template <int DIM> __global__ void __launch_bounds__(256) restrict_kernel(Geom gf, Geom gc, const double *__restrict__ r, const double *__restrict__ rlo, const double *__restrict__ rhi, double *__restrict__ bc)
{
  int64_t I, J, K, idx;
  if (!node_of_thread<DIM>(gc, I, J, K, idx)) return;
  double acc = 0.0;
#pragma unroll
  for (int dk = (DIM == 3 ? -1 : 0); dk <= (DIM == 3 ? 1 : 0); ++dk)
#pragma unroll
    for (int dj = -1; dj <= 1; ++dj)
#pragma unroll
      for (int di = -1; di <= 1; ++di) { // ascending fine index = MatMultTranspose's accumulation order
        const int64_t i = 2 * I + di, j = 2 * J + dj, k = 2 * K + dk;
        if (i < 0 || i >= gf.n0 || j < 0 || j >= gf.n1 || k < 0 || k >= gf.n2) continue;
        const double  w = (di ? 0.5 : 1.0) * (dj ? 0.5 : 1.0) * (dk ? 0.5 : 1.0);
        const int64_t q = DIM == 2 ? i + gf.ld * (j - gf.slo) : i + gf.ld * (j + gf.n1 * (k - gf.slo));
        acc             = fma(w, ldg(r, rlo, rhi, q, gf), acc);
      }
  bc[idx] = acc;
}

template <int DIM> __global__ void __launch_bounds__(256) prolong_kernel(Geom gf, Geom gc, const double *__restrict__ xc, const double *__restrict__ clo, const double *__restrict__ chi, double *__restrict__ xf)
{
  int64_t i, j, k, idx;
  if (!node_of_thread<DIM>(gf, i, j, k, idx)) return;
  // per direction: even node -> one coarse parent (weight 1); odd node -> (p-1)/2 and (p+1)/2 (if it exists), weight 1/2
  const int     ci = (i & 1) ? 2 : 1, cj = (j & 1) ? 2 : 1, ck = (DIM == 3 && (k & 1)) ? 2 : 1;
  const int64_t I0 = i >> 1, J0 = j >> 1, K0 = k >> 1;
  double        s = xf[idx];
  for (int c = 0; c < ck; ++c) {
    const int64_t K = K0 + c;
    if (K >= gc.n2) continue;
    for (int bq = 0; bq < cj; ++bq) {
      const int64_t J = J0 + bq;
      if (J >= gc.n1) continue;
      for (int a = 0; a < ci; ++a) {
        const int64_t I = I0 + a;
        if (I >= gc.n0) continue;
        const double  w = (ci == 2 ? 0.5 : 1.0) * (cj == 2 ? 0.5 : 1.0) * (ck == 2 ? 0.5 : 1.0);
        const int64_t q = DIM == 2 ? I + gc.ld * (J - gc.slo) : I + gc.ld * (J + gc.n1 * (K - gc.slo));
        s               = fma(w, ldg(xc, clo, chi, q, gc), s);
      }
    }
  }
  xf[idx] = s;
}

// ---- the coarse tail of the V-cycle in one launch (common.hpp: grid_tail_cycle) ---------------------------------------
// Same node arithmetic as box_sweep_kernel / box_apply_kernel / restrict_kernel / prolong_kernel / tri_gemv_kernel, so the
// result is bit-identical to the launch-per-colour path.  Vectors that change during the launch are read with
// ld.global.cg (L2): the CTAs of the cluster sit on different SMs, whose L1s are not coherent.
struct TailLevelDev {
  Geom          g;
  BoxConst      bc; // with idiag / sqrtdiag of the level's omega
  const double *coef, *idiag, *sqrtdiag;
  double        omo;
  int           ndirs, dirs[8];
  double       *b, *x, *r;
};
constexpr int TAIL_MAX_LEVELS = 10, TAIL_MAX_NOISE = 2 * TAIL_MAX_LEVELS * 8 + 1;
struct TailArgs {
  int           nlev;
  TailLevelDev  lv[TAIL_MAX_LEVELS]; // lv[0]: geometry and vectors of the coarsest grid only
  int           nc;                  // coarsest: v = W b + z, x = W^T v (chol.cu, gemv form)
  const double *W, *WT;
  double       *tmp0;
  int           mode;
  uint64_t      seed;
  TailNoise     ns[TAIL_MAX_NOISE];
  int           cluster; // CTAs per cluster (== gridDim.x), 1: plain block barrier
};

__device__ __forceinline__ void tail_sync(int cluster)
{
  if (cluster > 1) asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
  else __syncthreads();
}

// One directional sweep.  The level's normals are generated first, four per Philox call (a node-at-a-time sweep would
// use one of the four values each call returns), into the level's residual vector, which is free during smoothing.
template <int DIM> __device__ __forceinline__ void tail_sweep(const TailLevelDev &L, int dir, const NoiseArgs &na, int gtid, int gsize, int cluster)
{
  const Geom &g  = L.g;
  const int   nc = DIM == 3 ? 8 : 4;
  double     *zb = L.r;
  if (na.mode == PMG_NOISE_PHILOX) {
    const int qrow = ((int)g.n0 + 3) >> 2, nrows = (int)(g.nl / g.n0), nq = qrow * nrows; // quads of the padded index space
    for (int q = gtid; q < nq; q += gsize) {
      const int row = q / qrow, qi = q - row * qrow;
      double    z[4];
      philox_normal_quad(na.seed, na.call, (uint64_t)q, z);
#pragma unroll
      for (int m = 0; m < 4; ++m)
        if (4 * qi + m < (int)g.n0) zb[(int64_t)row * g.n0 + 4 * qi + m] = z[m];
    }
    tail_sync(cluster);
  }
  for (int s = 0; s < nc; ++s) {
    const int c  = dir == PMG_SOR_FORWARD_SWEEP ? s : nc - 1 - s;
    const int ci = c & 1, cj = (c >> 1) & 1, ck = (c >> 2) & 1;
    const int ni = ((int)g.n0 - ci + 1) / 2, nj = ((int)g.n1 - cj + 1) / 2, nk = DIM == 3 ? ((int)g.n2 - ck + 1) / 2 : 1;
    const int total = ni * nj * nk;
    for (int t = gtid; t < total; t += gsize) {
      const int     tx = t % ni, u = t / ni, ty = u % nj, tz = u / nj;
      const int64_t i = 2 * tx + ci, j = 2 * ty + cj, k = DIM == 3 ? 2 * tz + ck : 0;
      const int64_t idx = i + g.n0 * (j + g.n1 * k);
      const bool    interior = box_interior<DIM>(g, L.bc, i, j, k);
      const double  sq = interior ? L.bc.sqrtdiag : L.sqrtdiag[idx], id = interior ? L.bc.idiag : L.idiag[idx];
      const double  bv = __ldcg(L.b + idx);
      double        sum = bv; // noisy_rhs: w = (z * sqrtdiag) + b
      if (na.mode == PMG_NOISE_PHILOX) sum = __dadd_rn(__dmul_rn(__ldcg(zb + idx), sq), bv);
      else if (na.mode == PMG_NOISE_INJECTED) sum = __dadd_rn(__dmul_rn(na.tape[idx], sq), bv);
      sum               = box_row<DIM, true, false, true>(g, L.bc, L.coef, g.nl, L.x, nullptr, nullptr, idx, i, j, k, sum);
      const double t0   = __dmul_rn(L.omo, __ldcg(L.x + idx));
      L.x[idx]          = fma(id, sum, t0);
    }
    tail_sync(cluster);
  }
}

template <int DIM> __global__ void __launch_bounds__(1024, 1) grid_tail_kernel(const __grid_constant__ TailArgs a)
{
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsize = gridDim.x * blockDim.x;
  const int cl   = a.cluster;
  int       kn   = 0; // cursor into the noise blocks, in the reference's consumption order (SURVEY 8(c) tape contract)
  { // PCMG zeroes the iterate of the level it enters
    const TailLevelDev &T = a.lv[a.nlev - 1];
    for (int t = gtid; t < (int)T.g.nl; t += gsize) T.x[t] = 0.0;
    tail_sync(cl);
  }
  for (int l = a.nlev - 1; l >= 1; --l) {
    const TailLevelDev &F = a.lv[l], &C = a.lv[l - 1];
    for (int d = 0; d < F.ndirs; ++d, ++kn) tail_sweep<DIM>(F, F.dirs[d], NoiseArgs{a.mode, a.ns[kn].tape, a.seed, a.ns[kn].call, 0}, gtid, gsize, cl);
    for (int t = gtid; t < (int)F.g.nl; t += gsize) { // r = b - A x
      const int     i = t % (int)F.g.n0, u = t / (int)F.g.n0, j = DIM == 3 ? u % (int)F.g.n1 : u, k = DIM == 3 ? u / (int)F.g.n1 : 0;
      const double  ax = box_row<DIM, false, true, true>(F.g, F.bc, F.coef, F.g.nl, F.x, nullptr, nullptr, t, i, j, k, 0.0);
      F.r[t]           = __dsub_rn(__ldcg(F.b + t), ax);
    }
    tail_sync(cl);
    for (int t = gtid; t < (int)C.g.nl; t += gsize) { // b_c = P^T r, x_c = 0
      const int I = t % (int)C.g.n0, u = t / (int)C.g.n0, J = DIM == 3 ? u % (int)C.g.n1 : u, K = DIM == 3 ? u / (int)C.g.n1 : 0;
      double    acc = 0.0;
#pragma unroll
      for (int dk = (DIM == 3 ? -1 : 0); dk <= (DIM == 3 ? 1 : 0); ++dk)
#pragma unroll
        for (int dj = -1; dj <= 1; ++dj)
#pragma unroll
          for (int di = -1; di <= 1; ++di) {
            const int i = 2 * I + di, j = 2 * J + dj, k = 2 * K + dk;
            if (i < 0 || i >= F.g.n0 || j < 0 || j >= F.g.n1 || k < 0 || k >= F.g.n2) continue;
            const double w = (di ? 0.5 : 1.0) * (dj ? 0.5 : 1.0) * (dk ? 0.5 : 1.0);
            acc            = fma(w, __ldcg(F.r + (i + F.g.n0 * (j + F.g.n1 * (int64_t)k))), acc);
          }
      C.b[t] = acc;
      C.x[t] = 0.0;
    }
    tail_sync(cl);
  }
  { // coarsest level: y = W^T (W b + z), one warp per entry (tri_gemv_kernel's order)
    const TailLevelDev &C = a.lv[0];
    const NoiseArgs     na{a.mode, a.ns[kn].tape, a.seed, a.ns[kn].call, 0};
    ++kn;
    const int lane = threadIdx.x & 31, gw = gtid >> 5, nw = gsize >> 5, n = a.nc;
    for (int i = gw; i < n; i += nw) {
      const double *row = a.W + (size_t)i * n;
      double        acc = 0.0;
      for (int k = lane; k < i + 1; k += 32) acc = fma(row[k], __ldcg(C.b + k), acc);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) a.tmp0[i] = na.mode != PMG_NOISE_NONE ? __dadd_rn(acc, noise_value(na, i)) : acc;
    }
    tail_sync(cl);
    for (int i = gw; i < n; i += nw) {
      const double *row = a.WT + (size_t)i * n;
      double        acc = 0.0;
      for (int k = i + lane; k < n; k += 32) acc = fma(row[k], __ldcg(a.tmp0 + k), acc);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) C.x[i] = acc;
    }
    tail_sync(cl);
  }
  for (int l = 1; l < a.nlev; ++l) {
    const TailLevelDev &F = a.lv[l], &C = a.lv[l - 1];
    for (int t = gtid; t < (int)F.g.nl; t += gsize) { // x_f += P x_c
      const int i = t % (int)F.g.n0, u = t / (int)F.g.n0, j = DIM == 3 ? u % (int)F.g.n1 : u, k = DIM == 3 ? u / (int)F.g.n1 : 0;
      const int ci = (i & 1) ? 2 : 1, cj = (j & 1) ? 2 : 1, ck = (DIM == 3 && (k & 1)) ? 2 : 1;
      const int I0 = i >> 1, J0 = j >> 1, K0 = k >> 1;
      double    sacc = __ldcg(F.x + t);
      for (int c = 0; c < ck; ++c) {
        const int K = K0 + c;
        if (K >= C.g.n2) continue;
        for (int bq = 0; bq < cj; ++bq) {
          const int J = J0 + bq;
          if (J >= C.g.n1) continue;
          for (int q = 0; q < ci; ++q) {
            const int I = I0 + q;
            if (I >= C.g.n0) continue;
            const double w = (ci == 2 ? 0.5 : 1.0) * (cj == 2 ? 0.5 : 1.0) * (ck == 2 ? 0.5 : 1.0);
            sacc           = fma(w, __ldcg(C.x + (I + C.g.n0 * (J + C.g.n1 * (int64_t)K))), sacc);
          }
        }
      }
      F.x[t] = sacc;
    }
    tail_sync(cl);
    for (int d = 0; d < F.ndirs; ++d, ++kn) tail_sweep<DIM>(F, F.dirs[d], NoiseArgs{a.mode, a.ns[kn].tape, a.seed, a.ns[kn].call, 0}, gtid, gsize, cl);
  }
}

// ---- Galerkin product on the grid: A_c = P^T (A P), same accumulation order as the row-by-row sparse product ----
template <int DIM> struct FineLap {
  Geom   g;
  LapTab tab;
  // entry A(p, p+d); p must exist
  __device__ double get(int64_t i, int64_t j, int64_t k, int di, int dj, int dk) const
  {
    const int nz = (di != 0) + (dj != 0) + (dk != 0);
    if (nz > 1) return 0.0;
    if (nz == 1) {
      const int64_t a = i + di, b = j + dj, c = k + dk;
      if (a < 0 || a >= g.n0 || b < 0 || b >= g.n1 || c < 0 || c >= g.n2) return 0.0;
      return -tab.h;
    }
    const int deg = (int)(i > 0) + (int)(i < g.n0 - 1) + (int)(j > 0) + (int)(j < g.n1 - 1) + (DIM == 3 ? (int)(k > 0) + (int)(k < g.n2 - 1) : 0);
    return tab.diag[deg];
  }
};
template <int DIM> struct FineBox {
  Geom          g;
  const double *coef, *clo, *chi; // owned coefficients and the ghost units' coefficients (stride g.unit)
  int64_t       stride;
  __device__ double get(int64_t i, int64_t j, int64_t k, int di, int dj, int dk) const
  {
    const int64_t a = i + di, b = j + dj, c = k + dk;
    if (a < 0 || a >= g.n0 || b < 0 || b >= g.n1 || c < 0 || c >= g.n2) return 0.0;
    const int     s   = (di + 1) + 3 * (dj + 1) + (DIM == 3 ? 9 * (dk + 1) : 0);
    const int64_t idx = DIM == 2 ? i + g.n0 * (j - g.slo) : i + g.n0 * (j + g.n1 * (k - g.slo));
    if (idx < 0) return clo[(int64_t)s * g.unit + idx + g.unit];
    if (idx >= g.nl) return chi[(int64_t)s * g.unit + idx - g.nl];
    return coef[(int64_t)s * stride + idx];
  }
};

// Q1 weight P(q, J) along one direction
__device__ __forceinline__ double q1w(int64_t q, int64_t J, int64_t nc)
{
  if (J < 0 || J >= nc) return 0.0;
  const int64_t d = q - 2 * J;
  return d == 0 ? 1.0 : (d == 1 || d == -1) ? 0.5 : 0.0;
}

template <int DIM, class Fine> __global__ void __launch_bounds__(128) galerkin_kernel(Fine A, Geom gc, double *__restrict__ coef_c, int64_t stride_c)
{
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= gc.nl) return;
  constexpr int NST = DIM == 2 ? 9 : 27;
  const Geom   &gf  = A.g;
  int64_t       I, J, K;
  decode<DIM>(gc, idx, I, J, K);
  double ac[NST];
  for (int s = 0; s < NST; ++s) ac[s] = 0.0;
  for (int ak = (DIM == 3 ? -1 : 0); ak <= (DIM == 3 ? 1 : 0); ++ak)
    for (int aj = -1; aj <= 1; ++aj)
      for (int ai = -1; ai <= 1; ++ai) { // fine rows p of R's row I, ascending
        const int64_t pi = 2 * I + ai, pj = 2 * J + aj, pk = 2 * K + ak;
        if (pi < 0 || pi >= gf.n0 || pj < 0 || pj >= gf.n1 || pk < 0 || pk >= gf.n2) continue;
        const double wp = (ai ? 0.5 : 1.0) * (aj ? 0.5 : 1.0) * (ak ? 0.5 : 1.0);
        double       ap[NST]; // (A P)(p, I + e)
        for (int s = 0; s < NST; ++s) ap[s] = 0.0;
        for (int dk = (DIM == 3 ? -1 : 0); dk <= (DIM == 3 ? 1 : 0); ++dk)
          for (int dj = -1; dj <= 1; ++dj)
            for (int di = -1; di <= 1; ++di) { // columns q of A's row p, ascending
              const double a = A.get(pi, pj, pk, di, dj, dk);
              if (a == 0.0) continue;
              const int64_t qi = pi + di, qj = pj + dj, qk = pk + dk;
              for (int ek = (DIM == 3 ? -1 : 0); ek <= (DIM == 3 ? 1 : 0); ++ek)
                for (int ej = -1; ej <= 1; ++ej)
                  for (int ei = -1; ei <= 1; ++ei) {
                    double w = q1w(qi, I + ei, gc.n0) * q1w(qj, J + ej, gc.n1);
                    if (DIM == 3) w *= q1w(qk, K + ek, gc.n2);
                    if (w == 0.0) continue;
                    const int e = (ei + 1) + 3 * (ej + 1) + (DIM == 3 ? 9 * (ek + 1) : 0);
                    ap[e]       = fma(a, w, ap[e]);
                  }
            }
        for (int e = 0; e < NST; ++e) ac[e] = fma(wp, ap[e], ac[e]);
      }
  for (int e = 0; e < NST; ++e) coef_c[(int64_t)e * stride_c + idx] = ac[e];
}

inline unsigned nblocks(int64_t n, int bs) { return (unsigned)((n + bs - 1) / bs); }

// ---- common base: geometry, ghosts, parity colouring -----------------------------------------------------
struct GridOp : LevelOp {
  Geom           g;
  DevBuf<double> ghost_lo, ghost_hi;
  bool           parallel = false;

  int64_t n() const override { return g.nl; }
  bool    distributed() const override { return parallel; }
  bool    matrix_free() const override { return true; }
  int64_t nglobal() const override { return g.n0 * g.n1 * g.n2; }
  int64_t row0() const override { return g.row0(); }
  bool    structured(int &dim, int64_t dims[3]) const override
  {
    dim     = g.dim;
    dims[0] = g.n0;
    dims[1] = g.n1;
    dims[2] = g.n2;
    return true;
  }
  int init_ghosts()
  {
    parallel = ctx->nranks > 1 && !(g.slo == 0 && g.shi == g.nslow()); // a whole-grid operator is a replica, not a slab
    if (parallel) {
      PMG_TRY(ghost_lo.alloc((size_t)g.unit));
      PMG_TRY(ghost_hi.alloc((size_t)g.unit));
      PMG_TRY(ghost_lo.zero(ctx->stream));
      PMG_TRY(ghost_hi.zero(ctx->stream));
      // the thinnest slab of the partition (every rank must take the same code path: the exchanges are collective)
      const int64_t        mine = g.shi - g.slo;
      std::vector<int64_t> all((size_t)ctx->nranks, 0);
      PMG_TRY(comm_allgather_i64(ctx, &mine, 1, all.data()));
      min_units = *std::min_element(all.begin(), all.end());
    }
    return 0;
  }
  int64_t min_units = (int64_t)1 << 40;
  // refresh the ghost units of x from the slab neighbours (replaces the per-colour VecScatter, src/mc_sor.c:318-319)
  int halo(const double *x)
  {
    if (!parallel) return 0;
    return comm_halo_exchange(ctx, x, ghost_lo.p, x + g.nl - g.unit, ghost_hi.p, (size_t)g.unit, (size_t)g.unit, ctx->stream);
  }
  // pitched layout of the fused sweeps (LapOp): geometry, offset of the owned part, ghost exchange in place
  virtual bool pitched_view(Geom &gp, int64_t &own_offset) const { (void)gp; (void)own_offset; return false; }
  virtual int  pitched_halo(double *pitched) { (void)pitched; return PMG_ERR_SUP; }
  // ---- halo exchange overlapped with the rows that do not need it (north_star: "exchanged over NVLink with NCCL send/recv,
  //      overlapped with interior rows"; the reference's scatter is blocking, src/mc_sor.c:318-319) ----
  // The exchange runs on the context's communication stream.  A sweep then launches the tiles that read no ghost unit,
  // waits for the exchange on the compute stream, and launches the tiles along the slab boundaries.
  cudaEvent_t   ev_ready = nullptr, ev_halo = nullptr;
  const double *halo_inflight = nullptr;
  virtual int   pitched_halo_on(double *pitched, cudaStream_t s) { (void)pitched; (void)s; return PMG_ERR_SUP; }
  // early exchange of the post-smoother's ghost rows (V-cycle): on unless PMG_NO_EARLY_HALO; split sweep launches: opt-in with
  // PMG_OVERLAP_SWEEP (3D; measured on 2 x B200 with NCCL, profiles/r2_summary.md: the exchange kernel only got CTAs when the interior
  // launch drained, and the boundary tiles were full-height bands launched after it, so the split cost more than it hid)
  static bool   overlap_on() { return std::getenv("PMG_NO_EARLY_HALO") == nullptr; }
  static bool   overlap_sweep_on() { return std::getenv("PMG_OVERLAP_SWEEP") != nullptr; }
  // 2D fused sweeps: on by default since the boundary rows are thin bands that run on the communication stream behind the exchange
  // (2 x B200, 4097 x 4096 per GPU: sweep 101.4 -> 97.2 us, V-cycle sample 0.568 -> 0.557 ms); PMG_NO_OVERLAP_SWEEP switches it off
  bool          overlap_sweep_here() const { return g.dim == 2 ? std::getenv("PMG_NO_OVERLAP_SWEEP") == nullptr : overlap_sweep_on(); }
  int halo_begin(double *v) override
  {
    if (!parallel || !overlap_on() || !ctx->comm_stream) return 0;
    if (!ev_ready) {
      PMG_CUDA(cudaEventCreateWithFlags(&ev_ready, cudaEventDisableTiming));
      PMG_CUDA(cudaEventCreateWithFlags(&ev_halo, cudaEventDisableTiming));
    }
    PMG_CUDA(cudaEventRecord(ev_ready, ctx->stream));
    PMG_CUDA(cudaStreamWaitEvent(ctx->comm_stream, ev_ready, 0));
    PMG_TRY(pitched_halo_on(v, ctx->comm_stream));
    PMG_CUDA(cudaEventRecord(ev_halo, ctx->comm_stream));
    halo_inflight = v;
    return 0;
  }
  int halo_wait() // the compute stream continues after the exchange
  {
    PMG_CUDA(cudaStreamWaitEvent(ctx->stream, ev_halo, 0));
    halo_inflight = nullptr;
    return 0;
  }
  ~GridOp() override
  {
    if (ev_ready) cudaEventDestroy(ev_ready);
    if (ev_halo) cudaEventDestroy(ev_halo);
  }
  virtual bool star() const = 0;
  int          ncolors() const override { return star() ? 2 : (g.dim == 3 ? 8 : 4); }
  int32_t      colour_of(int64_t i, int64_t j, int64_t k) const { return star() ? (int32_t)((i + j + k) & 1) : (int32_t)((i & 1) + 2 * (j & 1) + (g.dim == 3 ? 4 * (k & 1) : 0)); }
  int          get_coloring(std::vector<int32_t> &c) override
  {
    c.resize((size_t)g.nl);
    for (int64_t idx = 0; idx < g.nl; ++idx) {
      const int64_t i = idx % g.n0, r = idx / g.n0;
      const int64_t j = g.dim == 2 ? g.slo + r : r % g.n1, k = g.dim == 2 ? 0 : g.slo + r / g.n1;
      c[(size_t)idx]  = colour_of(i, j, k);
    }
    return 0;
  }
  int set_coloring(int nc, const int32_t *c) override
  {
    std::vector<int32_t> mine;
    get_coloring(mine);
    if (nc != ncolors() || !std::equal(mine.begin(), mine.end(), c)) PMG_FAIL(PMG_ERR_SUP, "matrix-free grid operators sweep in parity colouring only; assemble the operator (pmg_mat_create_csr) to inject another colouring");
    return 0;
  }
  int set_coloring_auto(int policy) override
  {
    if (policy == PMG_COLORING_PARITY) return 0;
    if (policy == PMG_COLORING_GREEDY) return 0; // first-fit in natural order on a star / box stencil IS the parity colouring
    PMG_FAIL(PMG_ERR_SUP, "matrix-free grid operators sweep in parity colouring only; assemble the operator (pmg_mat_create_csr) for the lexicographic order");
  }
};

struct LapOp final : GridOp {
  double  kappa = 1;
  LapTab  tab;
  HostCsr assembled;
  bool    star() const override { return true; }
  // assembled copy on demand (small grids only: dense coarsest factorisation when the hierarchy has one level, inspection)
  const HostCsr *host_csr() override
  {
    if (parallel) return nullptr;
    if (assembled.n == 0) laplace_assemble(g.dim, g.n0, g.n1, g.n2, kappa, assembled);
    return &assembled;
  }

  void fill_tab(double omega, LapTab &t) const
  {
    const double h = 1.0 / (double)((g.n0 - 1) * (g.n0 - 1)); // src/problems.c:24
    const double f = omega > 0 ? std::sqrt((2 - omega) / omega) : 0;
    t.h            = h;
    for (int deg = 0; deg < 7; ++deg) {
      double d = kappa * kappa;
      for (int q = 0; q < deg; ++q) d += h; // src/problems.c:31-58: one += per existing neighbour
      t.diag[deg]     = d;
      double inv      = 1.0 / d;
      t.idiag[deg]    = inv * omega;                     // src/mc_sor.c:119-121
      t.sqrtdiag[deg] = std::sqrt(std::fabs(d)) * f;     // src/pc_mcgibbs.c:148-150
    }
  }
  int make_coeffs(double omega, SweepCoeffs &c) override
  {
    if (!(omega > 0 && omega < 2)) PMG_FAIL(PMG_ERR_ARG, "omega must be in (0,2), got %g", omega);
    c.omega = omega; // the tables are rebuilt per launch from omega (a few flops on the host)
    return 0;
  }
  int sweep(int dir, const SweepCoeffs &co, const double *b, double *y, const NoiseArgs &na) override
  {
    LapTab t;
    fill_tab(co.omega, t);
    const Plan pl = g.dim == 2 ? plan3((g.n0 + 1) >> 1, g.shi - g.slo, 1) : plan3((g.n0 + 1) >> 1, g.n1, g.shi - g.slo);
    PMG_PLAN_CHECK(pl);
    for (int s = 0; s < 2; ++s) {
      const int c = dir == PMG_SOR_FORWARD_SWEEP ? s : 1 - s;
      PMG_TRY(halo(y));
      if (g.dim == 2) lap_sweep_kernel<2><<<pl.grid, pl.block, 0, ctx->stream>>>(g, c, t, 1.0 - co.omega, b, y, ghost_lo.p, ghost_hi.p, na);
      else lap_sweep_kernel<3><<<pl.grid, pl.block, 0, ctx->stream>>>(g, c, t, 1.0 - co.omega, b, y, ghost_lo.p, ghost_hi.p, na);
      PMG_CUDA(cudaGetLastError());
      ctx->launches++;
    }
    ctx->dof_updates += g.nl;
    return 0;
  }
  // ---- fused streaming path (stream2d.cuh): 2D, single device ----
  bool fused_ok() const override
  {
    if (std::getenv("PMG_NO_FUSED")) return false; // read per call: the tests switch paths inside one process
    if (parallel && (min_units < GH() || std::getenv("PMG_NO_FUSED_PARALLEL"))) return false; // the ghost units of a side come from ONE neighbour
    if (g.dim == 2) return g.n0 >= 8 && g.n1 >= 4 && g.n0 < (1 << 30) && g.n1 < (1 << 30);
    return g.n0 >= 8 && g.n1 >= 2 && g.n2 >= 2 && g.n0 < (1 << 20) && g.n1 < (1 << 20) && g.n2 < (1 << 20);
  }
  // the fused grid transfers run on slabs in 2D (ghost rows of the coarse vectors, common.hpp Transfer::fused_after_restrict)
  bool fused_mg_ok() const override { return fused_ok() && (g.dim == 2 ? (!parallel || !std::getenv("PMG_NO_FUSED_MG_PARALLEL")) : (!parallel && !std::getenv("PMG_NO_FUSED_MG3"))); }
  bool fused_null_xin_ok() const override { return g.dim == 2 && !parallel; }
  bool pitched_is_natural() const override { return !parallel && pitch() == g.n0; }
  bool fused_smooth_ok() const override { return parallel && fused_ok() && !std::getenv("PMG_NO_FUSED_SMOOTH"); }
  bool pitched_view(Geom &gp, int64_t &own_offset) const override
  {
    gp         = pitched(g, pitch());
    own_offset = GH() * unit_rows() * pitch();
    return true;
  }
  int pitched_halo(double *p) override { return fused_halo(p); }
  int pitched_halo_on(double *p, cudaStream_t s) override { return fused_halo(p, s); }
  int residual_pitched(const double *b, const double *x, double *r) override
  {
    PMG_TRY(fused_halo(const_cast<double *>(x)));
    Geom    gp;
    int64_t off;
    pitched_view(gp, off);
    const Plan pl = g.dim == 2 ? plan_nodes<2>(gp) : plan_nodes<3>(gp);
    PMG_PLAN_CHECK(pl);
    const double *xo = x + off;
    if (g.dim == 2) lap_apply_kernel<2, true><<<pl.grid, pl.block, 0, ctx->stream>>>(gp, tab, b + off, xo, xo - gp.unit, xo + gp.nl, r + off);
    else if (!std::getenv("PMG_NO_PITCHED3_SLAB")) // four columns per thread, ghost planes read in place (the per-node kernel costs 2x, profiles/r1_summary.md)
      lap_residual3_pitched_kernel<<<dim3((unsigned)(((pitch() >> 2) * g.n1 + 255) / 256), (unsigned)(g.shi - g.slo)), 256, 0, ctx->stream>>>(gp, tab, b + off, xo, r + off);
    else lap_apply_kernel<3, true><<<pl.grid, pl.block, 0, ctx->stream>>>(gp, tab, b + off, xo, xo - gp.unit, xo + gp.nl, r + off);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }
  bool fused_tape_ok() const override { return !parallel; } // the ghost units' noise is recomputed, which a tape of owned rows cannot supply
  // On a slab the pitched vectors carry GH ghost units (grid rows in 2D, planes in 3D) on either side: one fused sweep
  // updates both colours, so the boundary unit's second-colour update needs the neighbour's boundary unit AFTER its
  // first-colour update, which is recomputed here from two old ghost units (and the ghost unit of b; the noise is a
  // function of the global index).  One exchange of 2 units per sweep replaces the reference's per-colour scatters.
  // 2D: six ghost rows, what the pre-smoother with the fused residual + restriction reads beyond its band (sweep2d.cuh RESTRICT)
  int     GH() const { return parallel ? (g.dim == 2 ? 6 : 2) : 0; }
  int64_t unit_rows() const { return g.dim == 2 ? 1 : g.n1; }
  int     fused_halo(double *pitched, cudaStream_t s = nullptr)
  {
    if (!parallel) return 0;
    const int64_t U = unit_rows() * pitch(), nu = g.shi - g.slo;
    double       *own = pitched + GH() * U;
    return comm_halo_exchange(ctx, own, pitched, own + (nu - GH()) * U, own + nu * U, (size_t)(GH() * U), (size_t)(GH() * U), s ? s : ctx->stream);
  }
  // Work list of the streaming kernels.  Warps whose tile touches the physical boundary run the predicated loop, which
  // costs about 1.6x the interior loop per row (profiles/r1_summary.md), and the grid is a single wave, so those warps
  // get half-height bands: every warp then finishes at about the same time.  Bands start on even rows (the fused
  // restriction emits coarse row J from the band that owns fine row 2J).
  DevBuf<stream2d::Item> items[2]; // [restrict ? 1 : 0]
  int                    nitems[2] = {0, 0};
  int                    items_by  = 0;
  int build_items(int by)
  {
    using stream2d::Item;
    using stream2d::STRIP_OUT;
    const int nstrips = (int)((g.n0 + STRIP_OUT - 1) / STRIP_OUT);
    for (int r = 0; r < 2; ++r) {
      const int         lo_halo = r ? 4 : 2, hi_halo = r ? 4 : 2; // rows touched below ja / above jb (stream2d: jlo, jhi)
      std::vector<Item> slow, fast;
      for (int s = 0; s < nstrips; ++s) {
        const int  c0 = s * STRIP_OUT - 4;
        const bool edge_strip = !(c0 >= 1 && c0 + 127 <= g.n0 - 2);
        int64_t    j = g.slo;
        while (j < g.shi) {
          // would a full-height band starting here be interior?
          const int64_t jb_full = std::min<int64_t>(j + by, g.shi);
          const bool    interior = !edge_strip && j - lo_halo >= 1 && jb_full + hi_halo <= g.n1 - 2 && j - lo_halo >= g.slo && jb_full + hi_halo + 4 < g.shi;
          int64_t       h = interior ? by : std::max(2, (by / 2) & ~1);
          const int64_t jb = std::min<int64_t>(j + h, g.shi);
          (interior ? fast : slow).push_back(Item{s, (int)j, (int)jb});
          j = jb;
        }
      }
      slow.insert(slow.end(), fast.begin(), fast.end()); // predicated tiles first
      nitems[r] = (int)slow.size();
      PMG_TRY(items[r].upload(slow, ctx->stream));
    }
    PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    items_by = by;
    return 0;
  }

  int64_t pitch() const { return (g.n0 + 3) / 4 * 4; }
  int64_t slab_rows() const { return g.dim == 2 ? g.shi - g.slo : g.n1 * (g.shi - g.slo); }
  int64_t fused_size() const override { return pitch() * (slab_rows() + 2 * GH() * unit_rows()); }
  int     to_pitched(const double *natural, double *pitched) override
  {
    const Plan pl = g.dim == 2 ? plan3(g.n0, g.shi - g.slo, 1) : plan3(g.n0, g.n1, g.shi - g.slo);
    PMG_PLAN_CHECK(pl);
    repitch_kernel<true><<<pl.grid, pl.block, 0, ctx->stream>>>(g.n0, g.dim == 2 ? g.shi - g.slo : g.n1, pitch(), natural, pitched + GH() * unit_rows() * pitch());
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return fused_halo(pitched);
  }
  int from_pitched(const double *pitched, double *natural) override
  {
    const Plan pl = g.dim == 2 ? plan3(g.n0, g.shi - g.slo, 1) : plan3(g.n0, g.n1, g.shi - g.slo);
    PMG_PLAN_CHECK(pl);
    repitch_kernel<false><<<pl.grid, pl.block, 0, ctx->stream>>>(g.n0, g.dim == 2 ? g.shi - g.slo : g.n1, pitch(), pitched + GH() * unit_rows() * pitch(), natural);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }
  // b, xin, xout are pitched (fused_size() elements); xc / bc are the coarse level's natural-layout vectors
  // ---- 3D: stream3d.cuh ----
  DevBuf<sweep3d::Item> items3;
  DevBuf<double>        r_pitched; // residual of the fused 3D top level (fused_sweep with bc)
  int                   nitems3 = 0, nitems3_nohalo = 0, items3_bz = 0, items3_nw = 0;
  int build_items3(int bz, int NW3) // NW3 warps per CTA tile: NW3 - 2 output rows + 2 halo rows (narrow strips: 2 NW3 - 2 + 2)
  {
    static const bool narrow_env = std::getenv("PMG_SW3_NONARROW") == nullptr;
    static const int  thin_env   = std::getenv("PMG_SW3_THIN") ? std::atoi(std::getenv("PMG_SW3_THIN")) : 4;
    std::vector<int32_t> flat;
    sweep3d_plan(g.n0, g.n1, g.n2, g.slo, g.shi, bz, NW3, narrow_env, thin_env, flat);
    std::vector<sweep3d::Item> all(flat.size() / 5);
    for (size_t q = 0; q < all.size(); ++q) all[q] = sweep3d::Item{flat[5 * q], flat[5 * q + 1], flat[5 * q + 2], flat[5 * q + 3], flat[5 * q + 4]};
    // tiles that read no ghost plane first (they overlap the halo exchange), tiles along the slab boundaries last
    std::stable_partition(all.begin(), all.end(), [&](const sweep3d::Item &it) { return !parallel || (it.ka - 2 >= g.slo && it.kb + 1 < g.shi); });
    nitems3_nohalo = 0;
    for (const auto &it : all) nitems3_nohalo += (!parallel || (it.ka - 2 >= g.slo && it.kb + 1 < g.shi)) ? 1 : 0;
    nitems3 = (int)all.size();
    PMG_TRY(items3.upload(all, ctx->stream));
    PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    items3_bz = bz;
    items3_nw = NW3;
    return 0;
  }
  template <int NOISE, int NW, int SX, int SB, int MINB, bool WS = false> int launch3(sweep3d::Args &a, const double *b, const double *xin)
  {
    using namespace sweep3d;
    auto         kern = sweep3d_kernel<NOISE, NW, SX, SB, MINB, WS>;
    const size_t sm   = Smem<NW, SX, SB, WS>::total;
    static bool attr_set[16] = {false}; // per device: function attributes belong to the device's context
    if (!attr_set[ctx->device & 15]) {
      PMG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
      attr_set[ctx->device & 15] = true;
    }
    static const bool swz = std::getenv("PMG_SW3_PLAIN") == nullptr; // SWIZZLE_32B boxes: conflict-free shared-memory reads
    a.swizzle = swz ? 1 : 0;
    if (swz) {
      const int64_t dims[4] = {4, pitch() / 4, g.n1, g.shi - g.slo + 2 * GH()}, strides[4] = {1, 4, pitch(), pitch() * g.n1};
      const int     boxx[4] = {4, 32, NW + 2, 1}, boxb[4] = {4, 32, NW, 1};
      const int     boxx16[4] = {4, 16, 2 * NW + 2, 1}, boxb16[4] = {4, 16, 2 * NW, 1};
      PMG_TRY(make_tensor_map(a.tm_x, xin, 4, dims, strides, boxx, true));
      PMG_TRY(make_tensor_map(a.tm_b, b ? b : xin, 4, dims, strides, boxb, true));
      PMG_TRY(make_tensor_map(a.tm_x16, xin, 4, dims, strides, boxx16, true));
      PMG_TRY(make_tensor_map(a.tm_b16, b ? b : xin, 4, dims, strides, boxb16, true));
    } else {
      const int64_t dims[4] = {pitch(), g.n1, g.shi - g.slo + 2 * GH(), 1}, strides[4] = {1, pitch(), pitch() * g.n1, pitch() * g.n1 * (g.shi - g.slo + 2 * GH())};
      const int     boxx[4] = {128, NW + 2, 1, 1}, boxb[4] = {128, NW, 1, 1};
      const int     boxx16[4] = {64, 2 * NW + 2, 1, 1}, boxb16[4] = {64, 2 * NW, 1, 1};
      PMG_TRY(make_tensor_map(a.tm_x, xin, 4, dims, strides, boxx, false));
      PMG_TRY(make_tensor_map(a.tm_b, b ? b : xin, 4, dims, strides, boxb, false));
      PMG_TRY(make_tensor_map(a.tm_x16, xin, 4, dims, strides, boxx16, false));
      PMG_TRY(make_tensor_map(a.tm_b16, b ? b : xin, 4, dims, strides, boxb16, false));
    }
    static const int bz_env = std::getenv("PMG_SW3_BZ") ? std::atoi(std::getenv("PMG_SW3_BZ")) : 0;
    const int        bz     = bz_env > 0 ? bz_env : 64;
    if (items3_bz != bz || items3_nw != NW) PMG_TRY(build_items3(bz, NW));
    a.items = items3.p;
    if (split_launch && nitems3_nohalo > 0 && nitems3_nohalo < nitems3) { // interior tiles | wait for the halo | boundary tiles
      kern<<<(unsigned)nitems3_nohalo, NW * 32 * (WS ? 2 : 1), sm, ctx->stream>>>(a);
      PMG_TRY(halo_wait());
      a.items = items3.p + nitems3_nohalo;
      kern<<<(unsigned)(nitems3 - nitems3_nohalo), NW * 32 * (WS ? 2 : 1), sm, ctx->stream>>>(a);
      ctx->launches++;
    } else {
      if (split_launch) PMG_TRY(halo_wait());
      kern<<<(unsigned)nitems3, NW * 32 * (WS ? 2 : 1), sm, ctx->stream>>>(a);
    }
    split_launch = false;
    return 0;
  }
  bool split_launch = false; // set by the sweep that started its halo exchange on the communication stream
  // the persistent warp-specialised kernel (sweep3d_ws.cuh): device Philox noise, swizzled boxes; one CTA per SM draws tiles
  DevBuf<sweep3d::WsQueue> queue3;
  int launch3_ws(sweep3d::Args &a, const double *b, const double *xin)
  {
    using namespace sweep3d;
    constexpr int NW = WS_NW;
    auto          kern = sweep3d_ws_kernel;
    const size_t  sm   = Smem<NW, WS_SX, WS_SB, true>::total;
    PMG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    if (!queue3.p) {
      PMG_TRY(queue3.alloc(1));
      PMG_TRY(queue3.zero(ctx->stream));
    }
    a.swizzle = 1;
    const int64_t dims[4] = {4, pitch() / 4, g.n1, g.shi - g.slo + 2 * GH()}, strides[4] = {1, 4, pitch(), pitch() * g.n1};
    const int     boxx[4] = {4, 32, NW + 2, 1}, boxb[4] = {4, 32, NW, 1};
    const int     boxx16[4] = {4, 16, 2 * NW + 2, 1}, boxb16[4] = {4, 16, 2 * NW, 1};
    PMG_TRY(make_tensor_map(a.tm_x, xin, 4, dims, strides, boxx, true));
    PMG_TRY(make_tensor_map(a.tm_b, b ? b : xin, 4, dims, strides, boxb, true));
    PMG_TRY(make_tensor_map(a.tm_x16, xin, 4, dims, strides, boxx16, true));
    PMG_TRY(make_tensor_map(a.tm_b16, b ? b : xin, 4, dims, strides, boxb16, true));
    static const int bz_env = std::getenv("PMG_SW3_BZ") ? std::atoi(std::getenv("PMG_SW3_BZ")) : 0;
    const int        bz     = bz_env > 0 ? bz_env : 64;
    if (items3_bz != bz || items3_nw != NW) PMG_TRY(build_items3(bz, NW));
    a.queue = queue3.p;
    auto go = [&](const sweep3d::Item *items, int n) {
      a.items  = items;
      a.nitems = n;
      kern<<<(unsigned)std::min(n, ctx->sm_count), NW * 64, sm, ctx->stream>>>(a);
    };
    if (split_launch && nitems3_nohalo > 0 && nitems3_nohalo < nitems3) { // interior tiles | wait for the halo | boundary tiles
      go(items3.p, nitems3_nohalo);
      PMG_TRY(halo_wait());
      go(items3.p + nitems3_nohalo, nitems3 - nitems3_nohalo);
      ctx->launches++;
    } else {
      if (split_launch) PMG_TRY(halo_wait());
      go(items3.p, nitems3);
    }
    split_launch = false;
    return 0;
  }
  template <int NOISE> int launch3_cfg(int cfg, sweep3d::Args &a, const double *b, const double *xin)
  {
    static const bool plain = std::getenv("PMG_SW3_PLAIN") != nullptr;
    if (cfg == 7 && NOISE == sweep3d::NOISE_PHILOX && !plain) return launch3_ws(a, b, xin);
    switch (cfg) {
    case 1: return launch3<NOISE, 8, 3, 2, 2>(a, b, xin);  // 256 threads, 128 registers, 2 CTAs / SM
    case 2: return launch3<NOISE, 16, 4, 2, 1>(a, b, xin); // 512 threads, 128 registers, 1 CTA / SM
    default:
      if (NOISE == sweep3d::NOISE_PHILOX) return launch3<sweep3d::NOISE_PHILOX, 16, 4, 2, 1, true>(a, b, xin); // warp-specialised
      return launch3<NOISE, 16, 4, 2, 1>(a, b, xin);
    }
  }
  // ghost units of the sweep's iterate: already in flight (halo_begin by the caller), started here on the communication
  // stream (the launch is then split), or exchanged on the compute stream (no communicator stream / PMG_NO_OVERLAP)
  int start_halo(const double *xin)
  {
    split_launch = false;
    if (!parallel) return 0;
    if (halo_inflight == xin && xin) return halo_wait(); // exchanged ahead of time: one launch
    if (overlap_sweep_here() && overlap_on() && ctx->comm_stream) {
      PMG_TRY(halo_begin(const_cast<double *>(xin)));
      split_launch = true;
      return 0;
    }
    return fused_halo(const_cast<double *>(xin));
  }
  int fused_sweep3(int dir, const SweepCoeffs &co, const double *b, const double *xin, double *xout, const NoiseArgs &na)
  {
    using namespace sweep3d;
    if (!xin) PMG_FAIL(PMG_ERR_ARG, "fused 3D sweep needs an iterate");
    LapTab t;
    fill_tab(co.omega, t);
    const char      *cfg_str = std::getenv("PMG_SW3_CFG"); // read per call: the tests switch kernels inside one process
    const int        cfg_env = cfg_str ? std::atoi(cfg_str) : -1;
    // warp-specialised kernels for Philox on grids with >= 48 rows: 7 = persistent (sweep3d_ws.cuh), 6 = one CTA per tile.  Measured
    // on 512^3 (profiles/r2_summary.md): with a right-hand side both are bound by the memory system at the same time (6 is 0 - 2 %
    // ahead), without one (prior sampling, 16 B per update) the persistent kernel's shorter instruction stream is 16 % faster
    const int        cfg     = cfg_env >= 0 && cfg_env <= 7 ? cfg_env : (g.n1 >= 48 ? (b ? 6 : 7) : 1);
    Args a;
    a.nx = (int)g.n0; a.ny = (int)g.n1; a.nz = (int)g.n2; a.slo = (int)g.slo; a.shi = (int)g.shi;
    a.tlo = (int)g.slo - GH(); a.thi = (int)g.shi + GH();
    if (parallel && na.mode == PMG_NOISE_INJECTED) PMG_FAIL(PMG_ERR_SUP, "fused sweep on a slab cannot take an injected tape");
    PMG_TRY(start_halo(xin));
    a.pitch  = (int)pitch();
    a.pplane = (long long)pitch() * g.n1;
    a.flip   = dir == PMG_SOR_BACKWARD_SWEEP ? 1 : 0;
    a.has_b  = b ? 1 : 0;
    a.xout   = xout;
    a.tape   = na.tape;
    a.h = t.h; a.idiag = t.idiag[6]; a.sd = t.sqrtdiag[6]; a.omo = 1.0 - co.omega;
    for (int d = 0; d < 7; ++d) a.coef[d] = sweep2d::Coef{t.idiag[d], t.sqrtdiag[d], 1.0 - co.omega, 0.0};
    a.coef[7] = sweep2d::Coef{0.0, 0.0, 0.0, 0.0};
    philox_expand_keys(na.seed, a.pk);
    a.call_lo = (uint32_t)na.call; a.call_hi = (uint32_t)(na.call >> 32);
    if (na.mode == PMG_NOISE_NONE) PMG_TRY(launch3_cfg<NOISE_NONE>(cfg, a, b, xin));
    else if (na.mode == PMG_NOISE_INJECTED) PMG_TRY(launch3_cfg<NOISE_TAPE>(cfg, a, b, xin));
    else PMG_TRY(launch3_cfg<NOISE_PHILOX>(cfg, a, b, xin));
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    ctx->dof_updates += g.nl;
    return 0;
  }

  // ---- 2D plain sweep: sweep2d.cuh (TMA-fed) ----
  DevBuf<sweep2d::Item> items2;
  int                   nitems2 = 0, items2_cfg = -1;
  int build_items2(int by, std::vector<sweep2d::Item> &out, bool restrict_mode = false) const
  {
    std::vector<int32_t> flat;
    int                  nh = 0;
    sweep2d_plan(g.n0, g.n1, g.slo, g.shi, parallel, by, restrict_mode, parallel && overlap_sweep_here() && overlap_on(), flat, nh);
    out.resize(flat.size() / 3);
    for (size_t q = 0; q < out.size(); ++q) out[q] = sweep2d::Item{flat[3 * q], flat[3 * q + 1], flat[3 * q + 2]};
    (restrict_mode ? nohalo2r : nohalo2) = nh;
    return (int)out.size();
  }
  mutable int nohalo2 = 0, nohalo2r = 0;
  template <int NOISE, int WARPS, int STAGES, int MINB, bool RESTRICT = false> int launch2(const sweep2d::Args &a, int &slots)
  {
    using namespace sweep2d;
    auto          kern = sweep2d_kernel<NOISE, WARPS, STAGES, MINB, RESTRICT>;
    const size_t  sm   = smem_bytes<WARPS, STAGES>();
    static int    occ_dev[16] = {0}; // per device: function attributes belong to the device's context
    const int     dv = ctx->device & 15;
    if (!occ_dev[dv]) {
      int occ = 0;
      PMG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
      PMG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, WARPS * 32, sm));
      occ_dev[dv] = std::max(1, occ);
    }
    slots = occ_dev[dv] * WARPS * ctx->sm_count;
    if (a.nitems <= 0) return 0;
    const int nh = RESTRICT ? nohalo2r : nohalo2;
    if (split_launch && nh > 0 && nh < a.nitems) { // interior tiles | wait for the halo | boundary tiles
      sweep2d::Args a1 = a, a2 = a;
      a1.nitems = nh;
      a2.items  = a.items + nh;
      a2.nitems = a.nitems - nh;
      // the boundary tiles follow the exchange on the communication stream (thin bands: build_items2) beside the interior tiles on
      // the compute stream, which then waits for both
      kern<<<(unsigned)((a2.nitems + WARPS - 1) / WARPS), WARPS * 32, sm, ctx->comm_stream>>>(a2);
      PMG_CUDA(cudaEventRecord(ev_halo, ctx->comm_stream));
      PMG_CUDA(launch_pdl(ctx->stream, kern, dim3((unsigned)((a1.nitems + WARPS - 1) / WARPS)), dim3(WARPS * 32), sm, a1));
      PMG_TRY(halo_wait());
      ctx->launches++;
    } else {
      if (split_launch) PMG_TRY(halo_wait());
      PMG_CUDA(launch_pdl(ctx->stream, kern, dim3((unsigned)((a.nitems + WARPS - 1) / WARPS)), dim3(WARPS * 32), sm, a));
    }
    split_launch = false;
    return 0;
  }
  // the pre-smoother with the fused residual + restriction (sweep2d.cuh RESTRICT)
  template <int NOISE> int launch2r_cfg(int cfg, const sweep2d::Args &a, int &slots)
  {
    switch (cfg) {
    case 0: return launch2<NOISE, 8, 3, 2, true>(a, slots); // 128 registers, 16 warps / SM
    case 1: return launch2<NOISE, 4, 3, 3, true>(a, slots); // 168 registers, 12 warps / SM
    default: return launch2<NOISE, 8, 3, 1, true>(a, slots);
    }
  }
  int sweep2dr_launch(int cfg, const sweep2d::Args &a, int mode, int &slots)
  {
    if (mode == PMG_NOISE_NONE) return launch2r_cfg<sweep2d::NOISE_NONE>(cfg, a, slots);
    if (mode == PMG_NOISE_INJECTED) return launch2r_cfg<sweep2d::NOISE_TAPE>(cfg, a, slots);
    return launch2r_cfg<sweep2d::NOISE_PHILOX>(cfg, a, slots);
  }
  DevBuf<sweep2d::Item> items2r;
  int                   nitems2r = 0, items2r_cfg = -1;
  template <int NOISE> int launch2_cfg(int cfg, const sweep2d::Args &a, int &slots)
  {
    switch (cfg) {
    case 0: return launch2<NOISE, 4, 2, 4>(a, slots); // 128 registers, 16 warps / SM
    case 1: return launch2<NOISE, 4, 3, 4>(a, slots);
    case 2: return launch2<NOISE, 4, 2, 5>(a, slots); // 96 registers, 20 warps / SM
    case 3: return launch2<NOISE, 8, 2, 2>(a, slots);
    default: return launch2<NOISE, 8, 2, 3>(a, slots); // 80 registers, 24 warps / SM
    }
  }
  int sweep2d_launch(int cfg, const sweep2d::Args &a, int mode, int &slots)
  {
    if (mode == PMG_NOISE_NONE) return launch2_cfg<sweep2d::NOISE_NONE>(cfg, a, slots);
    if (mode == PMG_NOISE_INJECTED) return launch2_cfg<sweep2d::NOISE_TAPE>(cfg, a, slots);
    return launch2_cfg<sweep2d::NOISE_PHILOX>(cfg, a, slots);
  }
  int fused_sweep2_tma(int dir, const SweepCoeffs &co, const double *b, const double *xin, double *xout, const NoiseArgs &na, LevelOp *coarse = nullptr, const double *xc = nullptr, double *bc = nullptr)
  {
    using namespace sweep2d;
    LapTab t;
    fill_tab(co.omega, t);
    static const int cfg_env = std::getenv("PMG_SW2_CFG") ? std::atoi(std::getenv("PMG_SW2_CFG")) : 0;
    static const int by_env  = std::getenv("PMG_SW2_BY") ? std::atoi(std::getenv("PMG_SW2_BY")) : 0;
    const int        cfg     = std::getenv("PMG_SW2_CFG") && cfg_env >= 0 && cfg_env <= 4 ? cfg_env : 3;
    Args a;
    static const bool swz = std::getenv("PMG_SW2_SWIZZLE") != nullptr;
    a.swizzle = swz ? 1 : 0;
    if (swz) {
      const int64_t dims[3] = {4, pitch() / 4, g.shi - g.slo + 2 * GH()}, strides[3] = {1, 4, pitch()};
      const int     box[3]  = {4, 32, STAGE_ROWS};
      PMG_TRY(make_tensor_map(a.tm_x, xin, 3, dims, strides, box, true));
      PMG_TRY(make_tensor_map(a.tm_b, b ? b : xin, 3, dims, strides, box, true));
    } else { // pad columns are real (zero) elements in both views
      const int64_t dims[3] = {pitch(), g.shi - g.slo + 2 * GH(), 1}, strides[3] = {1, pitch(), pitch() * (g.shi - g.slo + 2 * GH())};
      const int     box[3]  = {128, STAGE_ROWS, 1};
      PMG_TRY(make_tensor_map(a.tm_x, xin, 3, dims, strides, box, false));
      PMG_TRY(make_tensor_map(a.tm_b, b ? b : xin, 3, dims, strides, box, false));
    }
    a.nx = (int)g.n0; a.ny = (int)g.n1; a.slo = (int)g.slo; a.shi = (int)g.shi;
    a.tlo = (int)g.slo - GH(); a.thi = (int)g.shi + GH();
    if (parallel && na.mode == PMG_NOISE_INJECTED) PMG_FAIL(PMG_ERR_SUP, "fused sweep on a slab cannot take an injected tape");
    PMG_TRY(start_halo(xin));
    a.pitch = (int)pitch();
    a.flip  = dir == PMG_SOR_BACKWARD_SWEEP ? 1 : 0;
    a.has_b = b ? 1 : 0;
    a.xout  = xout;
    a.xc = nullptr; a.bc = nullptr; a.cnx = a.cny = a.cpitch = a.ctlo = 0;
    if (xc || bc) { // prolongation / residual + restriction fused into the sweep: the coarse level is a whole grid on this device
      int     cd;
      int64_t cn[3];
      if (!coarse || !coarse->structured(cd, cn)) PMG_FAIL(PMG_ERR_SUP, "fused grid transfers need a structured coarse level");
      a.xc = xc; a.bc = bc; a.cnx = (int)cn[0]; a.cny = (int)cn[1];
      a.cpitch = (int)(coarse->level_pitch ? coarse->level_pitch : cn[0]);
      a.ctlo   = (int)coarse->level_first_row();
      if (parallel && !coarse->level_pitch && coarse->level_first_row() != 0) PMG_FAIL(PMG_ERR_SUP, "fused grid transfers on a slab need a pitched (or whole) coarse level");
    }
    a.tape  = na.tape;
    a.h = t.h; a.idiag = t.idiag[4]; a.sd = t.sqrtdiag[4]; a.omo = 1.0 - co.omega; a.diag = t.diag[4];
    for (int d = 0; d < 5; ++d) a.coef[d] = Coef{t.idiag[d], t.sqrtdiag[d], 1.0 - co.omega, t.diag[d]};
    a.coef[5] = Coef{0.0, 0.0, 0.0, 0.0};
    philox_expand_keys(na.seed, a.pk);
    a.call_lo = (uint32_t)na.call; a.call_hi = (uint32_t)(na.call >> 32);
    if (bc) { // pre-smoother + residual + restriction
      const int rcfg_env = std::getenv("PMG_SW2R_CFG") ? std::atoi(std::getenv("PMG_SW2R_CFG")) : 1; // 168 registers, 12 warps / SM measured fastest (profiles/r2_summary.md)
      static const int rby_env  = std::getenv("PMG_SW2R_BY") ? std::atoi(std::getenv("PMG_SW2R_BY")) : 0;
      if (items2r_cfg != rcfg_env) {
        a.items = nullptr; a.nitems = 0;
        int slots = 0;
        PMG_TRY(sweep2dr_launch(rcfg_env, a, na.mode, slots));
        std::vector<Item> list;
        const int         nstrips = (int)((g.n0 + STRIP_OUT - 1) / STRIP_OUT);
        int by = rby_env > 0 ? rby_env : std::max<int>(4, (int)(((g.shi - g.slo) * nstrips + slots - 1) / std::max(1, slots)));
        by += by & 1;
        while (build_items2(by, list, true) > slots - (parallel ? 8 : 0) && rby_env <= 0 && by < g.shi - g.slo) by += 2;
        nitems2r = (int)list.size();
        PMG_TRY(items2r.upload(list, ctx->stream));
        PMG_CUDA(cudaStreamSynchronize(ctx->stream));
        items2r_cfg = rcfg_env;
      }
      a.items = items2r.p; a.nitems = nitems2r;
      int slots = 0;
      PMG_TRY(sweep2dr_launch(rcfg_env, a, na.mode, slots));
      PMG_CUDA(cudaGetLastError());
      ctx->launches++;
      ctx->dof_updates += g.nl;
      return 0;
    }
    if (items2_cfg != cfg) { // size the bands so that the work list is one resident wave
      a.items = nullptr; a.nitems = 0;
      int slots = 0;
      PMG_TRY(sweep2d_launch(cfg, a, na.mode, slots));
      std::vector<Item> list;
      const int         nstrips = (int)((g.n0 + STRIP_OUT - 1) / STRIP_OUT);
      int by = by_env > 0 ? by_env : std::max<int>(2, (int)(((g.shi - g.slo) * nstrips + slots - 1) / std::max(1, slots)));
      by += by & 1;
      while (build_items2(by, list) > slots - (parallel ? 8 : 0) && by_env <= 0 && by < g.shi - g.slo) by += 2;
      nitems2 = (int)list.size();
      PMG_TRY(items2.upload(list, ctx->stream));
      PMG_CUDA(cudaStreamSynchronize(ctx->stream));
      items2_cfg = cfg;
    }
    a.items = items2.p; a.nitems = nitems2;
    int slots = 0;
    PMG_TRY(sweep2d_launch(cfg, a, na.mode, slots));
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    ctx->dof_updates += g.nl;
    return 0;
  }

  int fused_sweep(int dir, const SweepCoeffs &co, const double *b, const double *xin, double *xout, const NoiseArgs &na, LevelOp *coarse, const double *xc, double *bc) override
  {
    if (g.dim == 3) { // the transfers run as separate kernels on the pitched vectors (same arithmetic as the unfused V-cycle)
      if ((xc || bc) && (parallel || !coarse)) PMG_FAIL(PMG_ERR_SUP, "the 3D fused sweep with grid transfers needs an undistributed level pair");
      const Geom gp = pitched(g, pitch());
      if (xc) { // x_old = xin + P xc, in place (the caller's iterate buffer: it is dead after this sweep)
        const Geom &gc = static_cast<GridOp *>(coarse)->g;
        prolong3_pitched_kernel<<<dim3((unsigned)(((pitch() >> 2) * g.n1 + 255) / 256), (unsigned)g.n2), 256, 0, ctx->stream>>>(gp, gc, xc, nullptr, nullptr, const_cast<double *>(xin));
        PMG_CUDA(cudaGetLastError());
        ctx->launches++;
      }
      PMG_TRY(fused_sweep3(dir, co, b, xin, xout, na));
      if (bc) { // b_c = P^T (b - A xout)
        const Geom &gc = static_cast<GridOp *>(coarse)->g;
        if (!r_pitched.p) PMG_TRY(r_pitched.alloc((size_t)fused_size()));
        lap_residual3_pitched_kernel<<<dim3((unsigned)(((pitch() >> 2) * g.n1 + 255) / 256), (unsigned)g.n2), 256, 0, ctx->stream>>>(gp, tab, b, xout, r_pitched.p);
        restrict3_pitched_kernel<<<dim3((unsigned)((((gc.n0 + 3) >> 2) * gc.n1 + 255) / 256), (unsigned)gc.n2), 256, 0, ctx->stream>>>(gp, gc, r_pitched.p, bc);
        PMG_CUDA(cudaGetLastError());
        ctx->launches += 2;
      }
      return 0;
    }
    static const bool no_tma = std::getenv("PMG_NO_TMA") != nullptr;
    static const bool no_tma_prolong = std::getenv("PMG_NO_TMA_PROLONG") != nullptr;
    static const bool no_tma_restrict = std::getenv("PMG_NO_TMA_RESTRICT") != nullptr;
    if (xc && bc) PMG_FAIL(PMG_ERR_SUP, "fused sweep: prolongation and restriction in one pass are not combined");
    if (xin && !no_tma && (!xc || !no_tma_prolong) && (!bc || !no_tma_restrict)) return fused_sweep2_tma(dir, co, b, xin, xout, na, coarse, xc, bc);
    using namespace stream2d;
    LapTab t;
    fill_tab(co.omega, t);
    Args a;
    a.g = Geom2{(int)g.n0, (int)g.n1, (int)g.slo, (int)g.shi};
    a.gc = a.g;
    a.cpitch = a.g.nx;
    if (coarse) {
      int     cd;
      int64_t cn[3];
      coarse->structured(cd, cn);
      auto *cg = static_cast<GridOp *>(coarse);
      a.gc     = Geom2{(int)cn[0], (int)cn[1], (int)cg->g.slo, (int)cg->g.shi};
      a.cpitch = (int)(coarse->level_pitch ? coarse->level_pitch : cn[0]);
    }
    static const int by_env = std::getenv("PMG_STREAM_BY") ? std::atoi(std::getenv("PMG_STREAM_BY")) : 0;
    int by = by_env > 0 ? by_env : 64;
    by += by & 1;
    if (items_by != by) PMG_TRY(build_items(by));
    a.by      = by;
    a.pitch   = (int)pitch();
    a.items   = items[bc ? 1 : 0].p;
    a.nitems  = nitems[bc ? 1 : 0];
    a.nstrips = (int)((g.n0 + STRIP_OUT - 1) / STRIP_OUT);
    a.nbands  = (int)((g.shi - g.slo + by - 1) / by);
    a.flip    = dir == PMG_SOR_BACKWARD_SWEEP ? 1 : 0;
    a.xin = xin; a.b = b; a.xc = xc; a.xout = xout; a.bc = bc;
    for (int d = 0; d < 5; ++d) { a.tab.diag[d] = t.diag[d]; a.tab.idiag[d] = t.idiag[d]; a.tab.sqrtdiag[d] = t.sqrtdiag[d]; }
    a.tab.h   = t.h;
    a.tab.omo = 1.0 - co.omega;
    a.na      = na;
    const int64_t warps = a.nitems;
    const int     bs    = 128; // matches the kernels' __launch_bounds__
    const unsigned nb   = nblocks(warps * 32, bs);
    if (xc && bc) PMG_FAIL(PMG_ERR_SUP, "fused sweep: prolongation and restriction in one pass are not combined");
    if (bc) {
      if ((g.slo & 1) != 0) PMG_FAIL(PMG_ERR_SUP, "fused restriction needs an even first row");
      if (!xin) lap_stream_kernel<GUESS_ZERO, true><<<nb, bs, 0, ctx->stream>>>(a);
      else lap_stream_kernel<GUESS_LOAD, true><<<nb, bs, 0, ctx->stream>>>(a);
    } else if (xc) {
      if (!xin) PMG_FAIL(PMG_ERR_ARG, "fused prolongation needs a fine iterate");
      lap_stream_kernel<GUESS_PROLONG, false><<<nb, bs, 0, ctx->stream>>>(a);
    } else {
      if (!xin) lap_stream_kernel<GUESS_ZERO, false><<<nb, bs, 0, ctx->stream>>>(a);
      else lap_stream_kernel<GUESS_LOAD, false><<<nb, bs, 0, ctx->stream>>>(a);
    }
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    ctx->dof_updates += g.nl;
    return 0;
  }

  template <bool RES> int apply(const double *b, const double *x, double *out)
  {
    PMG_TRY(halo(x));
    const Plan pl = g.dim == 2 ? plan_nodes<2>(g) : plan_nodes<3>(g);
    PMG_PLAN_CHECK(pl);
    if (g.dim == 2) lap_apply_kernel<2, RES><<<pl.grid, pl.block, 0, ctx->stream>>>(g, tab, b, x, ghost_lo.p, ghost_hi.p, out);
    else lap_apply_kernel<3, RES><<<pl.grid, pl.block, 0, ctx->stream>>>(g, tab, b, x, ghost_lo.p, ghost_hi.p, out);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }
  int  residual(const double *b, const double *x, double *r) override { return apply<true>(b, x, r); }
  int  mult(const double *x, double *y) override { return apply<false>(nullptr, x, y); }
  void describe(std::string &out) override
  {
    char buf[256];
    snprintf(buf, sizeof buf, "matrix-free %d-point shifted Laplacian %lldx%lldx%lld (units %lld..%lld), kappa %g, red-black", g.dim == 2 ? 5 : 7, (long long)g.n0, (long long)g.n1, (long long)g.n2, (long long)g.slo, (long long)g.shi, kappa);
    out = buf;
  }
};

struct BoxOp final : GridOp {
  DevBuf<double> coef; // [3^d][nl]
  DevBuf<double> coef_lo, coef_hi; // ghost units of the coefficients (multi-GPU set-up)
  BoxConst       bc;
  HostCsr        assembled;
  bool           have_assembled = false;
  bool           star() const override { return false; }
  int            nst() const { return g.dim == 2 ? 9 : 27; }

  // ghost units of the coefficient arrays (needed by the next Galerkin product across a slab boundary)
  int exchange_coef_ghosts()
  {
    if (!parallel) return 0;
    PMG_TRY(coef_lo.alloc((size_t)nst() * g.unit));
    PMG_TRY(coef_hi.alloc((size_t)nst() * g.unit));
    PMG_TRY(coef_lo.zero(ctx->stream));
    PMG_TRY(coef_hi.zero(ctx->stream));
    for (int s = 0; s < nst(); ++s) {
      const double *a = coef.p + (size_t)s * g.nl;
      PMG_TRY(comm_halo_exchange(ctx, a, coef_lo.p + (size_t)s * g.unit, a + g.nl - g.unit, coef_hi.p + (size_t)s * g.unit, (size_t)g.unit, (size_t)g.unit, ctx->stream));
    }
    return 0;
  }

  int detect_interior()
  {
    bc.on = 0;
    for (int ring = 1; ring <= 2 && !bc.on; ++ring) {
      // reference node (ring, ring[, ring]) must be owned by this rank; otherwise use the first owned interior unit
      const int64_t ks = std::max<int64_t>(ring, g.slo);
      if (g.n0 <= 2 * ring || g.n1 <= 2 * ring || (g.dim == 3 && g.n2 <= 2 * ring)) break;
      if (ks >= std::min<int64_t>(g.shi, g.nslow() - ring)) break;
      const int64_t ref = g.dim == 2 ? ring + g.n0 * (ks - g.slo) : ring + g.n0 * (ring + g.n1 * (ks - g.slo));
      DevBuf<unsigned long long> cnt;
      PMG_TRY(cnt.alloc(1));
      PMG_TRY(cnt.zero(ctx->stream));
      if (g.dim == 2) box_uniform_kernel<2><<<nblocks(g.nl, 256), 256, 0, ctx->stream>>>(g, coef.p, g.nl, ring, ref, cnt.p);
      else box_uniform_kernel<3><<<nblocks(g.nl, 256), 256, 0, ctx->stream>>>(g, coef.p, g.nl, ring, ref, cnt.p);
      PMG_CUDA(cudaGetLastError());
      unsigned long long bad = 1;
      PMG_CUDA(cudaMemcpyAsync(&bad, cnt.p, sizeof bad, cudaMemcpyDeviceToHost, ctx->stream));
      PMG_CUDA(cudaStreamSynchronize(ctx->stream));
      if (bad == 0) {
        for (int s = 0; s < nst(); ++s) PMG_CUDA(cudaMemcpyAsync(&bc.c[s], coef.p + (size_t)s * g.nl + ref, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        PMG_CUDA(cudaStreamSynchronize(ctx->stream));
        bc.on   = 1;
        bc.ring = ring;
      }
    }
    // the interior stencil must be the same on every rank for the result to be partition independent: it is, because
    // it is a function of the (global) fine interior stencil only.
    return 0;
  }

  int make_coeffs(double omega, SweepCoeffs &c) override
  {
    if (!(omega > 0 && omega < 2)) PMG_FAIL(PMG_ERR_ARG, "omega must be in (0,2), got %g", omega);
    PMG_TRY(c.idiag.alloc((size_t)g.nl));
    PMG_TRY(c.sqrtdiag.alloc((size_t)g.nl));
    const double f = std::sqrt((2 - omega) / omega);
    if (g.dim == 2) box_coeffs_kernel<2><<<nblocks(g.nl, 256), 256, 0, ctx->stream>>>(g, coef.p, g.nl, omega, f, c.idiag.p, c.sqrtdiag.p);
    else box_coeffs_kernel<3><<<nblocks(g.nl, 256), 256, 0, ctx->stream>>>(g, coef.p, g.nl, omega, f, c.idiag.p, c.sqrtdiag.p);
    PMG_CUDA(cudaGetLastError());
    c.omega = omega;
    return 0;
  }
  int sweep(int dir, const SweepCoeffs &co, const double *b, double *y, const NoiseArgs &na) override
  {
    BoxConst k = bc;
    if (k.on) {
      const double d = k.c[nst() / 2];
      double     inv = 1.0 / d;
      k.idiag        = inv * co.omega;
      k.sqrtdiag     = std::sqrt(std::fabs(d)) * std::sqrt((2 - co.omega) / co.omega);
    }
    const int  nc = ncolors();
    if (box3_on()) return box3_sweep(dir, co, b, y, na); // four colours per launch, one CTA per plane (box3d.cuh)
    if (g.dim == 3 && !parallel && g.n0 <= 512 && (g.n2 + 1) / 2 <= 65535 && !std::getenv("PMG_NO_BOX_PAIR")) { // colour pairs (ci = 0, 1) in one launch
      const unsigned bx = (unsigned)((((g.n0 + 1) / 2) + 31) / 32 * 32);
      const dim3     grid((unsigned)((g.n1 + 1) / 2), (unsigned)((g.n2 + 1) / 2));
      const size_t   sm = (size_t)9 * (size_t)(g.n0 + 2) * sizeof(double);
      for (int s = 0; s < 4; ++s) {
        const int p = dir == PMG_SOR_FORWARD_SWEEP ? s : 3 - s;
        box_pair_sweep3_kernel<<<grid, bx, sm, ctx->stream>>>(g, p, dir == PMG_SOR_FORWARD_SWEEP ? 0 : 1, coef.p, g.nl, k, co.idiag.p, co.sqrtdiag.p, 1.0 - co.omega, b, y, na);
        PMG_CUDA(cudaGetLastError());
        ctx->launches++;
      }
      ctx->dof_updates += g.nl;
      return 0;
    }
    const Plan pl = g.dim == 2 ? box_colour_plan<2>(g) : box_colour_plan<3>(g);
    PMG_PLAN_CHECK(pl);
    // A colour lives on the units (grid rows / planes) of ONE parity of the slowest dimension, and everything it reads from a
    // ghost unit has the other parity: the ghosts need refreshing only when units of that other parity have been swept
    // since the last exchange -- twice per sweep instead of once per colour (src/mc_sor.c:318-319 scatters before every colour).
    bool dirty[2] = {true, true};
    for (int s = 0; s < nc; ++s) {
      const int c = dir == PMG_SOR_FORWARD_SWEEP ? s : nc - 1 - s;
      const int sp = g.dim == 2 ? (c >> 1) & 1 : (c >> 2) & 1;
      if (dirty[1 - sp]) {
        PMG_TRY(halo(y));
        dirty[0] = dirty[1] = false;
      }
      dirty[sp] = true;
      if (g.dim == 2) box_sweep_kernel<2><<<pl.grid, pl.block, 0, ctx->stream>>>(g, c, coef.p, g.nl, k, co.idiag.p, co.sqrtdiag.p, 1.0 - co.omega, b, y, ghost_lo.p, ghost_hi.p, na);
      else box_sweep_kernel<3><<<pl.grid, pl.block, 0, ctx->stream>>>(g, c, coef.p, g.nl, k, co.idiag.p, co.sqrtdiag.p, 1.0 - co.omega, b, y, ghost_lo.p, ghost_hi.p, na);
      PMG_CUDA(cudaGetLastError());
      ctx->launches++;
    }
    ctx->dof_updates += g.nl;
    return 0;
  }

  // ---- fused four-colour sweep in one pass (box_stream.cuh): 2D, one device ----
  DevBuf<boxstream::Item> sitems;
  int                     nsitems = 0;
  bool stream_ok() const override
  {
    if (std::getenv("PMG_NO_BOX_STREAM")) return false;
    const char   *mn    = std::getenv("PMG_BOX_STREAM_MIN"); // smaller levels are launch-latency bound either way
    const int64_t min_n = mn ? std::atoll(mn) : 20000;
    return !level_pitch && g.dim == 2 && !parallel && g.slo == 0 && g.shi == g.n1 && g.n0 >= 16 && g.n1 >= 8 && g.nl >= min_n && g.nl < ((int64_t)1 << 31);
  }
  int stream_sweep(int dir, const SweepCoeffs &co, const double *b, const double *xin, double *xout, const NoiseArgs &na) override
  {
    using namespace boxstream;
    constexpr int WARPS = 4;
    static const int mb_env = std::getenv("PMG_BOX_STREAM_MINB") ? std::atoi(std::getenv("PMG_BOX_STREAM_MINB")) : 4;
    auto          kern  = mb_env == 6 ? box_stream_kernel<WARPS, 6> : mb_env == 5 ? box_stream_kernel<WARPS, 5> : box_stream_kernel<WARPS, 4>; // replicated Box-Muller tables (TREP 2 / 4 / 8) measured: no gain here, the CTAs are short-lived
    if (!nsitems) { // one resident wave: bands sized from the kernel's occupancy
      int occ = 0;
      PMG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, WARPS * 32, 0));
      const int         slots   = std::max(1, occ) * WARPS * ctx->sm_count;
      const int         nstrips = (int)((g.n0 + STRIP_OUT - 1) / STRIP_OUT);
      static const int by_env = std::getenv("PMG_BOX_STREAM_BY") ? std::atoi(std::getenv("PMG_BOX_STREAM_BY")) : 0;
      int              by     = by_env > 0 ? by_env : 2; // short bands: the per-step dependency chain is long, parallelism hides it (profiles/r1_summary.md)
      by += by & 1;
      std::vector<Item> list;
      for (;; by += 2) {
        list.clear();
        for (int s = 0; s < nstrips; ++s)
          for (int64_t j = 0; j < g.n1; j += by) list.push_back(Item{s, (int)j, (int)std::min<int64_t>(j + by, g.n1)});
        if ((int)list.size() <= slots || by >= g.n1 || by_env > 0) break;
      }
      nsitems = (int)list.size();
      PMG_TRY(sitems.upload(list, ctx->stream));
      PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    Args a;
    a.nx = (int)g.n0; a.ny = (int)g.n1;
    a.items = sitems.p; a.nitems = nsitems;
    a.flip  = dir == PMG_SOR_BACKWARD_SWEEP ? 1 : 0;
    a.xin = xin; a.b = b; a.xout = xout;
    a.coef = coef.p; a.idiag = co.idiag.p; a.sqrtdiag = co.sqrtdiag.p;
    for (int s = 0; s < 9; ++s) a.c[s] = bc.c[s];
    a.has_const = bc.on; a.ring = bc.ring;
    a.idiag_c = a.sd_c = 0.0;
    if (bc.on) { // BoxOp::sweep's interior coefficients
      const double d   = bc.c[4];
      double       inv = 1.0 / d;
      a.idiag_c        = inv * co.omega;
      a.sd_c           = std::sqrt(std::fabs(d)) * std::sqrt((2 - co.omega) / co.omega);
    }
    a.omo  = 1.0 - co.omega;
    a.mode = na.mode; a.tape = na.tape;
    philox_expand_keys(na.seed, a.pk);
    a.call_lo = (uint32_t)na.call; a.call_hi = (uint32_t)(na.call >> 32);
    a.pitch4  = (int)((g.n0 + 3) & ~(int64_t)3);
    kern<<<(unsigned)((nsitems + WARPS - 1) / WARPS), WARPS * 32, 0, ctx->stream>>>(a);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    ctx->dof_updates += g.nl;
    return 0;
  }

  // ---- one-pass TMA kernels (box2d.cuh): 2D, one device, PITCHED level vectors (LevelOp::level_pitch) ----
  bool        classes_ok = false;
  BoxClassTab cls_tab;
  // class tables of the shared-memory tail whose top level this is (tail2d.cuh): device copy + the (level, omega) list it was built for
  DevBuf<box2d::Cls>                      tail_cls;
  std::vector<box2d::Cls>                 tail_cls_host;
  std::vector<std::pair<const void *, double>> tail_cls_key;
  // Every rank contributes the class representatives it owns (row class 0 lives on the first rank only, ...); the merged table is
  // verified against every owned node on every rank, and the verdict is the same everywhere (the kernels are collective on slabs).
  int         detect_classes()
  {
    classes_ok = false;
    const int64_t rows = g.shi - g.slo;
    if (g.dim != 2 || g.n0 < 3 || g.n1 < 3 || g.nl >= ((int64_t)1 << 31)) return 0;
    if (!parallel && (g.slo != 0 || g.shi != g.n1)) return 0;
    const int64_t ri[3] = {0, 1, g.n0 - 1}, rj[3] = {0, 1, g.n1 - 1};
    std::vector<int64_t> mine(90, 0); // 81 coefficients (bit patterns) + 9 "have it" flags
    for (int rc = 0; rc < 3; ++rc) {
      int64_t j = rj[rc];
      if (rc == 1 && !(j >= g.slo && j < g.shi)) { // any owned interior row serves as the interior representative
        j = std::max<int64_t>(g.slo, 1);
        if (j >= std::min<int64_t>(g.shi, g.n1 - 1)) j = -1;
      }
      if (j < g.slo || j >= g.shi || rows <= 0) continue;
      for (int cc = 0; cc < 3; ++cc) {
        for (int s = 0; s < 9; ++s) PMG_CUDA(cudaMemcpyAsync(&mine[(size_t)(9 * (3 * rc + cc) + s)], coef.p + (size_t)s * g.nl + (size_t)(ri[cc] + g.n0 * (j - g.slo)), sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        mine[(size_t)(81 + 3 * rc + cc)] = 1;
      }
    }
    PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    std::vector<int64_t> all((size_t)90 * ctx->nranks, 0);
    PMG_TRY(comm_allgather_i64(ctx, mine.data(), 90, all.data()));
    bool have_all = true;
    for (int q = 0; q < 9; ++q) {
      int src = -1;
      for (int r = 0; r < ctx->nranks && src < 0; ++r)
        if (all[(size_t)90 * r + 81 + q]) src = r;
      if (src < 0) { have_all = false; continue; }
      std::memcpy(cls_tab.c[q], &all[(size_t)90 * src + 9 * q], 9 * sizeof(double));
    }
    unsigned long long bad = have_all ? 0 : 1;
    if (have_all && g.nl > 0) {
      DevBuf<unsigned long long> cnt;
      PMG_TRY(cnt.alloc(1));
      PMG_TRY(cnt.zero(ctx->stream));
      box_class_kernel<<<nblocks(g.nl, 256), 256, 0, ctx->stream>>>(g, coef.p, g.nl, cls_tab, cnt.p);
      PMG_CUDA(cudaGetLastError());
      PMG_CUDA(cudaMemcpyAsync(&bad, cnt.p, sizeof bad, cudaMemcpyDeviceToHost, ctx->stream));
      PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    const int64_t        mybad = (int64_t)bad;
    std::vector<int64_t> allbad((size_t)ctx->nranks, 0);
    PMG_TRY(comm_allgather_i64(ctx, &mybad, 1, allbad.data()));
    classes_ok = true;
    for (int64_t v : allbad) classes_ok = classes_ok && v == 0;
    return 0;
  }
  // ---- plane kernels of the 27-point levels (box3d.cuh) ----
  bool                 classes3_ok = false;
  BoxClass3Raw         cls3_raw;
  DevBuf<box3d::Tab>   tab3_dev;
  double               tab3_omega = -1;
  // Every rank contributes the class representatives it owns; the merged table is verified against every owned node on every
  // rank and the verdict is the same everywhere (the sweeps are collective on slabs).
  int detect_classes3()
  {
    classes3_ok = false;
    tab3_omega  = -1;
    if (g.dim != 3 || g.n0 < 3 || g.n1 < 3 || g.n2 < 3 || g.n0 * g.n1 >= ((int64_t)1 << 30)) return 0;
    if (!parallel && (g.slo != 0 || g.shi != g.n2)) return 0;
    const int64_t ri[3] = {0, 1, g.n0 - 1}, rj[3] = {0, 1, g.n1 - 1}, rk[3] = {0, 1, g.n2 - 1};
    std::vector<int64_t> rep(27, -1);
    for (int cz = 0; cz < 3; ++cz) {
      int64_t k = rk[cz];
      if (cz == 1 && !(k >= g.slo && k < g.shi)) { // any owned interior plane serves as the interior representative
        k = std::max<int64_t>(g.slo, 1);
        if (k >= std::min<int64_t>(g.shi, g.n2 - 1)) k = -1;
      }
      if (k < g.slo || k >= g.shi) continue;
      for (int cy = 0; cy < 3; ++cy)
        for (int cx = 0; cx < 3; ++cx) rep[(size_t)(cx + 3 * cy + 9 * cz)] = ri[cx] + g.n0 * (rj[cy] + g.n1 * (k - g.slo));
    }
    DevBuf<int64_t> rep_dev;
    DevBuf<double>  raw_dev;
    PMG_TRY(rep_dev.upload(rep, ctx->stream));
    PMG_TRY(raw_dev.alloc(729));
    PMG_TRY(raw_dev.zero(ctx->stream));
    box_class3_gather_kernel<<<27, 32, 0, ctx->stream>>>(g, coef.p, g.nl, rep_dev.p, raw_dev.p);
    PMG_CUDA(cudaGetLastError());
    std::vector<int64_t> mine(729 + 27, 0); // coefficients (bit patterns) + "have it" flags
    PMG_CUDA(cudaMemcpyAsync(mine.data(), raw_dev.p, 729 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int q = 0; q < 27; ++q) mine[(size_t)(729 + q)] = rep[(size_t)q] >= 0 ? 1 : 0;
    std::vector<int64_t> all((size_t)756 * ctx->nranks, 0);
    PMG_TRY(comm_allgather_i64(ctx, mine.data(), 756, all.data()));
    bool have_all = true;
    for (int q = 0; q < 27; ++q) {
      int src = -1;
      for (int r = 0; r < ctx->nranks && src < 0; ++r)
        if (all[(size_t)756 * r + 729 + q]) src = r;
      if (src < 0) { have_all = false; continue; }
      std::memcpy(cls3_raw.c[q], &all[(size_t)756 * src + 27 * q], 27 * sizeof(double));
      const int cx = q % 3, cy = (q / 3) % 3, cz = q / 9; // entries towards a missing neighbour are never read: zero them
      for (int s = 0; s < 27; ++s) {
        const int di = s % 3 - 1, dj = (s / 3) % 3 - 1, dk = s / 9 - 1;
        if ((cx == 0 && di < 0) || (cx == 2 && di > 0) || (cy == 0 && dj < 0) || (cy == 2 && dj > 0) || (cz == 0 && dk < 0) || (cz == 2 && dk > 0)) cls3_raw.c[q][s] = 0.0;
      }
    }
    unsigned long long bad = have_all ? 0 : 1;
    if (have_all && g.nl > 0) {
      DevBuf<unsigned long long> cnt;
      PMG_TRY(cnt.alloc(1));
      PMG_TRY(cnt.zero(ctx->stream));
      PMG_CUDA(cudaMemcpyAsync(raw_dev.p, &cls3_raw.c[0][0], 729 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
      box_class3_check_kernel<<<nblocks(g.nl, 256), 256, 0, ctx->stream>>>(g, coef.p, g.nl, raw_dev.p, cnt.p);
      PMG_CUDA(cudaGetLastError());
      PMG_CUDA(cudaMemcpyAsync(&bad, cnt.p, sizeof bad, cudaMemcpyDeviceToHost, ctx->stream));
      PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    const int64_t        mybad = (int64_t)bad;
    std::vector<int64_t> allbad((size_t)ctx->nranks, 0);
    PMG_TRY(comm_allgather_i64(ctx, &mybad, 1, allbad.data()));
    classes3_ok = true;
    for (int64_t v : allbad) classes3_ok = classes3_ok && v == 0;
    return 0;
  }
  bool box3_on() const { return g.dim == 3 && classes3_ok && !std::getenv("PMG_NO_BOX3"); }
  // class table for this omega on the device (box_coeffs_kernel's idiag / sqrtdiag per class)
  int box3_args(double omega, box3d::Args &a)
  {
    if (tab3_omega != omega) {
      static box3d::Tab t; // host staging (set-up path, one stream)
      const double      f = std::sqrt((2 - omega) / omega);
      for (int q = 0; q < 27; ++q) {
        const double d = cls3_raw.c[q][13];
        for (int s = 0; s < 27; ++s) t.c[q].nc[s] = -cls3_raw.c[q][s];
        double inv   = 1.0 / d;
        t.c[q].idiag = inv * omega;
        t.c[q].sd    = std::sqrt(std::fabs(d)) * f;
        t.c[q].pad   = 0.0;
      }
      PMG_TRY(tab3_dev.alloc(1));
      PMG_CUDA(cudaMemcpyAsync(tab3_dev.p, &t, sizeof t, cudaMemcpyHostToDevice, ctx->stream));
      PMG_CUDA(cudaStreamSynchronize(ctx->stream));
      tab3_host  = t;
      tab3_omega = omega;
    }
    std::memset(&a, 0, sizeof a);
    a.n0 = (int)g.n0; a.n1 = (int)g.n1; a.n2 = (int)g.n2;
    a.slo = (int)g.slo; a.shi = (int)g.shi;
    a.pitch4 = (int)((g.n0 + 3) & ~(int64_t)3);
    a.omo    = 1.0 - omega;
    a.in     = tab3_host.c[13];
    a.tab    = tab3_dev.p;
    a.glo    = ghost_lo.p;
    a.ghi    = ghost_hi.p;
    return 0;
  }
  box3d::Tab tab3_host;
  static int box3_nt()
  {
    static const int nt = std::getenv("PMG_BOX3_NT") ? std::atoi(std::getenv("PMG_BOX3_NT")) : 512;
    return nt == 1024 ? 1024 : (nt == 256 ? 256 : 512);
  }
  int box3_sweep(int dir, const SweepCoeffs &co, const double *b, double *y, const NoiseArgs &na)
  {
    box3d::Args a;
    PMG_TRY(box3_args(co.omega, a));
    a.b = b;
    a.x = y;
    const int nt = box3_nt();
    const int np = (int)((g.n0 + 1) / 2);
    static const int r_env = std::getenv("PMG_BOX3_R") ? std::atoi(std::getenv("PMG_BOX3_R")) : 0;
    const int        dv = ctx->device & 15;
    // staged variant (rows of three planes in shared memory, de-interleaved by column parity): a thread owns two nodes, so a block
    // of R even rows keeps nt threads busy when R * ceil(np / 2) is about nt; R is bounded by the shared memory of one SM
    box3d::SmemGeom sg{0, 0};
    size_t          sm = 0;
    bool            staged = !std::getenv("PMG_BOX3_NO_SMEM") && g.n0 >= 5;
    if (staged) {
      sg.H  = (int)((((g.n0 + 1) / 2 + 1) & ~(int64_t)1) + 4);
      a.R   = r_env > 0 ? r_env : std::max(1, std::min(16, nt / ((np + 1) / 2)));
      auto need = [&](int R) { return sizeof(box3d::Tab) + ((size_t)(2 * R + 1) * a.pitch4 + (size_t)3 * (4 * R + 3) * 2 * sg.H) * sizeof(double); };
      while (a.R > 1 && need(a.R) > 224 * 1024) --a.R;
      sm     = need(a.R);
      sg.RR  = 4 * a.R + 3;
      staged = sm <= 224 * 1024;
    }
    if (staged) {
      auto kern = nt == 1024 ? box3d::box3_sweep_smem_kernel<1024> : (nt == 256 ? box3d::box3_sweep_smem_kernel<256> : box3d::box3_sweep_smem_kernel<512>);
      static size_t sms_set[16] = {0};
      if (sm > sms_set[dv]) {
        PMG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(sm, 48 * 1024)));
        sms_set[dv] = std::max<size_t>(sm, 48 * 1024);
      }
      bool dirty[2] = {true, true}; // ghost planes: see below
      for (int s = 0; s < 2; ++s) {
        const int kp = dir == PMG_SOR_FORWARD_SWEEP ? s : 1 - s;
        if (dirty[1 - kp]) {
          PMG_TRY(halo(y));
          dirty[0] = dirty[1] = false;
        }
        dirty[kp] = true;
        const int64_t first = g.slo + ((kp ^ g.slo) & 1);
        const int64_t np_k  = first < g.shi ? (g.shi - first + 1) / 2 : 0;
        if (np_k > 0) {
          kern<<<(unsigned)np_k, nt, sm, ctx->stream>>>(a, kp, dir == PMG_SOR_FORWARD_SWEEP ? 0 : 1, na, sg);
          PMG_CUDA(cudaGetLastError());
          ctx->launches++;
        }
      }
      ctx->dof_updates += g.nl;
      return 0;
    }
    a.R = r_env > 0 ? r_env : std::max(1, std::min(16, nt / np));
    sm  = sizeof(box3d::Tab) + (size_t)(2 * a.R + 1) * a.pitch4 * sizeof(double);
    if (sm > 200 * 1024) PMG_FAIL(PMG_ERR_SUP, "27-point plane sweep: grid rows of %lld nodes do not fit the shared-memory staging", (long long)g.n0);
    auto kern = nt == 1024 ? box3d::box3_sweep_kernel<1024> : (nt == 256 ? box3d::box3_sweep_kernel<256> : box3d::box3_sweep_kernel<512>);
    static size_t sm_set[16] = {0};
    if (sm > sm_set[dv]) {
      PMG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(sm, 48 * 1024)));
      sm_set[dv] = std::max<size_t>(sm, 48 * 1024);
    }
    // ghost planes have the other k parity than the boundary planes that read them: refresh them before a parity whose
    // neighbours have been swept since the last exchange -- twice per sweep (src/mc_sor.c:318-319 scatters before every colour)
    bool dirty[2] = {true, true};
    for (int s = 0; s < 2; ++s) {
      const int kp = dir == PMG_SOR_FORWARD_SWEEP ? s : 1 - s;
      if (dirty[1 - kp]) {
        PMG_TRY(halo(y));
        dirty[0] = dirty[1] = false;
      }
      dirty[kp] = true;
      const int64_t first = g.slo + ((kp ^ g.slo) & 1);
      const int64_t np_k  = first < g.shi ? (g.shi - first + 1) / 2 : 0;
      if (np_k > 0) {
        kern<<<(unsigned)np_k, nt, sm, ctx->stream>>>(a, kp, dir == PMG_SOR_FORWARD_SWEEP ? 0 : 1, na);
        PMG_CUDA(cudaGetLastError());
        ctx->launches++;
      }
    }
    ctx->dof_updates += g.nl;
    return 0;
  }
  template <bool RES> int box3_apply(const double *b, const double *x, double *out)
  {
    box3d::Args a;
    PMG_TRY(box3_args(tab3_omega > 0 ? tab3_omega : 1.0, a));
    a.x     = const_cast<double *>(x);
    a.out_b = b;
    a.out   = out;
    const int nt = box3_nt();
    auto      kern = nt == 1024 ? box3d::box3_apply_kernel<1024, RES> : (nt == 256 ? box3d::box3_apply_kernel<256, RES> : box3d::box3_apply_kernel<512, RES>);
    kern<<<(unsigned)(g.shi - g.slo), nt, sizeof(box3d::Tab), ctx->stream>>>(a);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }

  int64_t pitch() const { return (g.n0 + 3) / 4 * 4; }
  // a slab keeps four ghost rows per side in its pitched vectors: what one sweep with the fused residual + restriction (zero
  // iterate) or prolongation reads beyond its band (box2d.cuh band_range / band_steps)
  int     GHB() const { return parallel ? 4 : 0; }
  int64_t level_first_row() const override { return level_pitch ? g.slo - GHB() : (parallel ? g.slo : 0); }
  // the level can run on the one-pass kernels; whether it does is the V-cycle's decision (it must keep the vectors pitched)
  bool box2_capable() const override { return classes_ok && g.n0 >= 16 && g.n1 >= 8 && (!parallel || min_units >= GHB()) && !std::getenv("PMG_NO_BOX2") && !(parallel && std::getenv("PMG_NO_FUSED_MG_PARALLEL")); }
  int64_t box2_pitch() const override { return pitch(); }
  bool    fused_ok() const override { return level_pitch != 0; }
  bool    fused_mg_ok() const override { return level_pitch != 0; }
  bool    fused_tape_ok() const override { return !parallel; }
  int64_t fused_size() const override { return level_pitch ? level_pitch * (g.shi - g.slo + 2 * GHB()) : n(); }
  int     pitched_halo(double *v) override { return pitched_halo_on(v, ctx->stream); }
  int     pitched_halo_on(double *v, cudaStream_t s) override
  {
    if (!parallel) return 0;
    const int64_t U = level_pitch, nu = g.shi - g.slo, G = GHB();
    double       *own = v + G * U;
    return comm_halo_exchange(ctx, own, v, own + (nu - G) * U, own + nu * U, (size_t)(G * U), (size_t)(G * U), s);
  }
  int to_pitched(const double *natural, double *pitched) override
  {
    const Plan pl = plan3(g.n0, g.shi - g.slo, 1);
    PMG_PLAN_CHECK(pl);
    repitch_kernel<true><<<pl.grid, pl.block, 0, ctx->stream>>>(g.n0, g.shi - g.slo, pitch(), natural, pitched + GHB() * pitch());
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return pitched_halo(pitched);
  }
  int from_pitched(const double *pitched, double *natural) override
  {
    const Plan pl = plan3(g.n0, g.shi - g.slo, 1);
    PMG_PLAN_CHECK(pl);
    repitch_kernel<false><<<pl.grid, pl.block, 0, ctx->stream>>>(g.n0, g.shi - g.slo, pitch(), pitched + GHB() * pitch(), natural);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }
  DevBuf<box2d::Item> b2items[2]; // [MODE_RESTRICT ? 1 : 0]: the fused residual + restriction runs narrower strips
  int                 b2n[2] = {0, 0};
  template <int NOISE, int MODE, int PC> int launch_box2(box2d::Args &a)
  {
    using namespace box2d;
    constexpr int WARPS = 8, STAGES = 2, MINB = MODE == MODE_RESTRICT ? 1 : 2;
    auto          kern = box2d_kernel<NOISE, MODE, PC, WARPS, STAGES, MINB>;
    const size_t  sm   = smem_bytes<WARPS, STAGES>();
    static int    occ_dev[16] = {0}; // per device: function attributes belong to the device's context
    const int     dv = ctx->device & 15;
    if (!occ_dev[dv]) {
      PMG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
      int occ = 0;
      PMG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, WARPS * 32, sm));
      occ_dev[dv] = std::max(1, occ);
    }
    const int r = MODE == MODE_RESTRICT ? 1 : 0;
    if (!b2n[r]) { // about one resident wave of warps; bands start on even rows (the band that owns fine row 2J emits coarse row J)
      static const int by_env = std::getenv("PMG_BOX2_BY") ? std::atoi(std::getenv("PMG_BOX2_BY")) : 0;
      static const int by_min = std::getenv("PMG_BOX2_BY_MIN") ? std::atoi(std::getenv("PMG_BOX2_BY_MIN")) : 2; // short bands on small levels: a band step costs ~1.8 us of dependent FP64 latency (profiles/r2_summary.md)
      const int        slots   = occ_dev[dv] * WARPS * ctx->sm_count;
      const int        nstrips = (int)((g.n0 + Strip<MODE>::OUT - 1) / Strip<MODE>::OUT);
      int              by      = by_env > 0 ? by_env : std::max<int>(by_min, (int)(((g.shi - g.slo) * nstrips + slots - 1) / slots));
      by += by & 1;
      std::vector<Item> list;
      for (int64_t j = g.slo; j < g.shi; j += by)
        for (int st = 0; st < nstrips; ++st) list.push_back(Item{st, (int)j, (int)std::min<int64_t>(j + by, g.shi)});
      b2n[r] = (int)list.size();
      PMG_TRY(b2items[r].upload(list, ctx->stream));
      PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    a.items  = b2items[r].p;
    a.nitems = b2n[r];
    PMG_CUDA(launch_pdl(ctx->stream, kern, dim3((unsigned)((a.nitems + WARPS - 1) / WARPS)), dim3(WARPS * 32), sm, a));
    return 0;
  }
  template <int NOISE, int MODE> int launch_box2_dir(int dir, box2d::Args &a) { return dir == PMG_SOR_BACKWARD_SWEEP ? launch_box2<NOISE, MODE, 1>(a) : launch_box2<NOISE, MODE, 0>(a); }
  template <int MODE> int launch_box2_noise(int dir, int noise, box2d::Args &a) { return noise == PMG_NOISE_PHILOX ? launch_box2_dir<box2d::NOISE_PHILOX, MODE>(dir, a) : launch_box2_dir<box2d::NOISE_RT, MODE>(dir, a); }
  static void fill_class(box2d::Cls &k, const double (&c)[9], double omega)
  {
    const double d = c[4], f = std::sqrt((2 - omega) / omega);
    for (int s = 0, q = 0; s < 9; ++s)
      if (s != 4) k.nc[q++] = -c[s];
    double inv = 1.0 / d;
    k.idiag    = inv * omega;               // box_coeffs_kernel
    k.sd       = std::sqrt(std::fabs(d)) * f;
    k.omo      = 1.0 - omega;
    k.ndiag    = -d;
  }
  // b, xin, xout: this level's pitched vectors; xc / bc: the coarse level's vectors (row stride coarse->level_pitch or natural)
  int fused_sweep(int dir, const SweepCoeffs &co, const double *b, const double *xin, double *xout, const NoiseArgs &na, LevelOp *coarse, const double *xc, double *bc) override
  {
    using namespace box2d;
    if (!level_pitch) PMG_FAIL(PMG_ERR_ORDER, "one-pass sweep on a level whose vectors are not pitched");
    if (xc && bc) PMG_FAIL(PMG_ERR_SUP, "fused sweep: prolongation and restriction in one pass are not combined");
    if (xc && !xin) PMG_FAIL(PMG_ERR_ARG, "fused prolongation needs a fine iterate");
    if (parallel && na.mode == PMG_NOISE_INJECTED) PMG_FAIL(PMG_ERR_SUP, "one-pass sweep on a slab cannot take an injected tape");
    if (xin && parallel) { // replaces the per-colour VecScatter of src/mc_sor.c:318-319: one exchange per sweep, started by the
                           // V-cycle right after the pre-smoother where it can be (it then overlaps the whole coarse-grid correction)
      if (halo_inflight == xin) PMG_TRY(halo_wait());
      else PMG_TRY(pitched_halo(const_cast<double *>(xin)));
    }
    Args a;
    std::memset(&a, 0, sizeof a);
    const int64_t P = level_pitch, held = g.shi - g.slo + 2 * GHB();
    const int64_t dims[3] = {P, held, 1}, strides[3] = {1, P, P * held};
    const int     box[3]  = {128, 2, 1};
    const double *any = xin ? xin : (b ? b : xout);
    a.tlo = (int)(g.slo - GHB());
    PMG_TRY(make_tensor_map(a.tm_x, xin ? xin : any, 3, dims, strides, box, false));
    PMG_TRY(make_tensor_map(a.tm_b, b ? b : any, 3, dims, strides, box, false));
    a.nx = (int)g.n0; a.ny = (int)g.n1; a.pitch = (int)P;
    a.has_x = xin ? 1 : 0; a.has_b = b ? 1 : 0;
    a.xout = xout; a.xc = xc; a.bc = bc;
    if (xc || bc) {
      int     cd;
      int64_t cn[3];
      if (!coarse || !coarse->structured(cd, cn)) PMG_FAIL(PMG_ERR_SUP, "fused grid transfer needs a structured coarse level");
      a.cnx = (int)cn[0]; a.cny = (int)cn[1];
      a.cpitch = (int)(coarse->level_pitch ? coarse->level_pitch : cn[0]);
      a.ccols  = a.cpitch;
      a.ctlo   = (int)coarse->level_first_row();
      if (parallel && !coarse->level_pitch && coarse->level_first_row() != 0) PMG_FAIL(PMG_ERR_SUP, "fused grid transfers on a slab need a pitched (or whole) coarse level");
    }
    a.mode = na.mode; a.tape = na.tape;
    for (int q = 0; q < 16; ++q) {
      const int rc = q >> 2, cc = q & 3;
      if (rc < 3 && cc < 3) fill_class(a.cls[q], cls_tab.c[3 * rc + cc], co.omega);
    }
    a.in = a.cls[5];
    philox_expand_keys(na.seed, a.pk);
    a.call_lo = (uint32_t)na.call; a.call_hi = (uint32_t)(na.call >> 32);
    if (bc) PMG_TRY(launch_box2_noise<MODE_RESTRICT>(dir, na.mode, a));
    else if (xc) PMG_TRY(launch_box2_noise<MODE_PROLONG>(dir, na.mode, a));
    else PMG_TRY(launch_box2_noise<MODE_PLAIN>(dir, na.mode, a));
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    ctx->dof_updates += g.nl;
    return 0;
  }

  template <bool RES> int apply(const double *b, const double *x, double *out)
  {
    PMG_TRY(halo(x));
    if (box3_on() && g.n0 * g.n1 < ((int64_t)1 << 30)) return box3_apply<RES>(b, x, out);
    const Plan pl = g.dim == 2 ? plan_nodes<2>(g) : plan_nodes<3>(g);
    PMG_PLAN_CHECK(pl);
    if (g.dim == 2) box_apply_kernel<2, RES><<<pl.grid, pl.block, 0, ctx->stream>>>(g, coef.p, g.nl, bc, b, x, ghost_lo.p, ghost_hi.p, out);
    else box_apply_kernel<3, RES><<<pl.grid, pl.block, 0, ctx->stream>>>(g, coef.p, g.nl, bc, b, x, ghost_lo.p, ghost_hi.p, out);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }
  int residual(const double *b, const double *x, double *r) override { return apply<true>(b, x, r); }
  int mult(const double *x, double *y) override { return apply<false>(nullptr, x, y); }

  // assembled copy (existing neighbours only, ascending columns): for the dense coarsest factorisation and for inspection
  const HostCsr *host_csr() override
  {
    if (have_assembled) return &assembled;
    if (parallel) return nullptr;
    std::vector<double> h((size_t)nst() * g.nl);
    if (cudaMemcpyAsync(h.data(), coef.p, h.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) return nullptr;
    cudaStreamSynchronize(ctx->stream);
    HostCsr &a = assembled;
    a.n = a.m = g.nl;
    a.rowptr.assign((size_t)g.nl + 1, 0);
    a.col.clear();
    a.val.clear();
    for (int64_t idx = 0; idx < g.nl; ++idx) {
      const int64_t i = idx % g.n0, r = idx / g.n0, j = g.dim == 2 ? r : r % g.n1, k = g.dim == 2 ? 0 : r / g.n1;
      for (int s = 0; s < nst(); ++s) {
        const int     di = s % 3 - 1, dj = (s / 3) % 3 - 1, dk = g.dim == 3 ? s / 9 - 1 : 0;
        const int64_t a0 = i + di, a1 = j + dj, a2 = k + dk;
        if (a0 < 0 || a0 >= g.n0 || a1 < 0 || a1 >= g.n1 || a2 < 0 || a2 >= g.n2) continue;
        a.col.push_back((int32_t)(a0 + g.n0 * (a1 + g.n1 * a2)));
        a.val.push_back(h[(size_t)s * g.nl + idx]);
      }
      a.rowptr[(size_t)idx + 1] = (int64_t)a.col.size();
    }
    have_assembled = true;
    return &assembled;
  }
  void describe(std::string &out) override
  {
    char buf[256];
    snprintf(buf, sizeof buf, "%d-point stencil arrays %lldx%lldx%lld (units %lld..%lld), %d colours, interior stencil %s", nst(), (long long)g.n0, (long long)g.n1, (long long)g.n2, (long long)g.slo, (long long)g.shi, ncolors(), bc.on ? "shared (read from kernel parameters)" : "per node");
    out = buf;
    if (level_pitch) out += ", one-pass TMA kernels on pitched vectors";
  }
};

// b_c = P^T (b - A x) for a stencil-array fine level on one device: every coarse node recomputes the residuals of its (up
// to 3^d) fine nodes -- same box_row order and same ascending-fine-index accumulation as box_apply_kernel + restrict_kernel,
// so the result is bit-identical, but the residual is never written or read back (the level is L2-resident: the extra
// reads of x hit the cache).
template <int DIM> __global__ void __launch_bounds__(256) box_restrict_residual_kernel(Geom gf, Geom gc, const double *__restrict__ coef, BoxConst bc, const double *__restrict__ b, const double *__restrict__ x, double *__restrict__ bcoarse)
{
  int64_t I, J, K, idx;
  if (!node_of_thread<DIM>(gc, I, J, K, idx)) return;
  double acc = 0.0;
#pragma unroll
  for (int dk = (DIM == 3 ? -1 : 0); dk <= (DIM == 3 ? 1 : 0); ++dk)
#pragma unroll
    for (int dj = -1; dj <= 1; ++dj)
#pragma unroll
      for (int di = -1; di <= 1; ++di) {
        const int64_t i = 2 * I + di, j = 2 * J + dj, k = 2 * K + dk;
        if (i < 0 || i >= gf.n0 || j < 0 || j >= gf.n1 || k < 0 || k >= gf.n2) continue;
        const double  w  = (di ? 0.5 : 1.0) * (dj ? 0.5 : 1.0) * (dk ? 0.5 : 1.0);
        const int64_t q  = i + gf.n0 * (j + gf.n1 * k);
        const double  ax = box_row<DIM, false, true>(gf, bc, coef, gf.nl, x, nullptr, nullptr, q, i, j, k, 0.0);
        acc              = fma(w, __dsub_rn(b[q], ax), acc);
      }
  bcoarse[idx] = acc;
}

struct GridTransfer final : Transfer {
  pmg_ctx ctx;
  GridOp *fine, *coarse;
  // fused transfers on slabs: the kernels of the fine level write / read the coarse level's pitched vectors directly; the ghost
  // rows of those vectors are refreshed here (one grouped send / receive per call)
  int fused_after_restrict(double *b_coarse) override { return coarse->parallel && coarse->level_pitch ? coarse->pitched_halo(b_coarse) : 0; }
  int fused_before_prolong(double *x_coarse) override { return coarse->parallel && coarse->level_pitch ? coarse->pitched_halo(x_coarse) : 0; }
  bool    tail_ok() const override { return !fine->parallel && !coarse->parallel; }
  bool    fused_residual_ok() const override
  {
    // opt-in: bit-identical but not faster than residual + restriction on B200 (each fine residual is recomputed by up to
    // 2^d coarse nodes; measured 1.02 vs 1.01 ms per V-cycle sample, profiles/r1_summary.md)
    return std::getenv("PMG_FUSED_RESIDUAL") && !fine->parallel && !coarse->parallel && dynamic_cast<BoxOp *>(fine) != nullptr && fine->g.slo == 0 && fine->g.shi == fine->g.nslow();
  }
  int restrict_residual(const double *b, const double *x, double *bcoarse) override
  {
    auto       *bx = static_cast<BoxOp *>(fine);
    const Geom &gf = fine->g, &gc = coarse->g;
    const Plan  pl = gf.dim == 2 ? plan_nodes<2>(gc) : plan_nodes<3>(gc);
    PMG_PLAN_CHECK(pl);
    if (gf.dim == 2) box_restrict_residual_kernel<2><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, bx->coef.p, bx->bc, b, x, bcoarse);
    else box_restrict_residual_kernel<3><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, bx->coef.p, bx->bc, b, x, bcoarse);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }
  int restrict_to(const double *r, double *bcoarse) override
  {
    PMG_TRY(fine->halo(r));
    const Geom &gf = fine->g, &gc = coarse->g;
    const Plan pl = gf.dim == 2 ? plan_nodes<2>(gc) : plan_nodes<3>(gc);
    PMG_PLAN_CHECK(pl);
    if (gf.dim == 2) restrict_kernel<2><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, r, fine->ghost_lo.p, fine->ghost_hi.p, bcoarse);
    else restrict_kernel<3><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, r, fine->ghost_lo.p, fine->ghost_hi.p, bcoarse);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }
  int restrict_pitched(double *r, double *bcoarse) override
  {
    Geom    gf;
    int64_t off;
    if (!fine->pitched_view(gf, off)) PMG_FAIL(PMG_ERR_SUP, "the fine operator has no pitched layout");
    PMG_TRY(fine->pitched_halo(r));
    const Geom &gc = coarse->g;
    const Plan  pl = gf.dim == 2 ? plan_nodes<2>(gc) : plan_nodes<3>(gc);
    PMG_PLAN_CHECK(pl);
    const double *ro = r + off;
    if (gf.dim == 2) restrict_kernel<2><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, ro, ro - gf.unit, ro + gf.nl, bcoarse);
    else if (pitched3_slab_ok(gf, gc)) restrict3_pitched_kernel<<<dim3((unsigned)((((gc.n0 + 3) >> 2) * gc.n1 + 255) / 256), (unsigned)(gc.shi - gc.slo)), 256, 0, ctx->stream>>>(gf, gc, ro, bcoarse);
    else restrict_kernel<3><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, ro, ro - gf.unit, ro + gf.nl, bcoarse);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }
  int prolong_pitched(const double *xc, double *xf) override
  {
    Geom    gf;
    int64_t off;
    if (!fine->pitched_view(gf, off)) PMG_FAIL(PMG_ERR_SUP, "the fine operator has no pitched layout");
    PMG_TRY(coarse->halo(xc));
    const Geom &gc = coarse->g;
    const Plan  pl = gf.dim == 2 ? plan_nodes<2>(gf) : plan_nodes<3>(gf);
    PMG_PLAN_CHECK(pl);
    if (gf.dim == 2) prolong_kernel<2><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, xc, coarse->ghost_lo.p, coarse->ghost_hi.p, xf + off);
    else if (pitched3_slab_ok(gf, gc)) prolong3_pitched_kernel<<<dim3((unsigned)(((gf.ld >> 2) * gf.n1 + 255) / 256), (unsigned)(gf.shi - gf.slo)), 256, 0, ctx->stream>>>(gf, gc, xc, coarse->ghost_lo.p, coarse->ghost_hi.p, xf + off);
    else prolong_kernel<3><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, xc, coarse->ghost_lo.p, coarse->ghost_hi.p, xf + off);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }
  int prolong_add(const double *xc, double *xf) override
  {
    PMG_TRY(coarse->halo(xc));
    const Geom &gf = fine->g, &gc = coarse->g;
    const Plan pl = gf.dim == 2 ? plan_nodes<2>(gf) : plan_nodes<3>(gf);
    PMG_PLAN_CHECK(pl);
    if (gf.dim == 2) prolong_kernel<2><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, xc, coarse->ghost_lo.p, coarse->ghost_hi.p, xf);
    else prolong_kernel<3><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, xc, coarse->ghost_lo.p, coarse->ghost_hi.p, xf);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }
};

// Transfer between a slab-distributed fine level and a coarse level that every rank holds in full (the reference
// agglomerates its coarse levels on rank 0, src/pc_chols.c:38-47 / src/pc_gamgmc.c:210-222; replicating them instead
// costs the same wall time, needs no scatter on the way up and keeps every rank's noise counters in step).
struct ReplicatingTransfer final : Transfer {
  pmg_ctx              ctx;
  GridOp              *fine;
  Geom                 gc; // this rank's slab of the coarse grid (owner of fine unit 2J owns coarse unit J)
  std::vector<int64_t> counts, displs;
  DevBuf<double>       slab;
  GridOp              *coarse_full = nullptr;
  std::vector<int64_t> crows; // coarse units [cs[2r], cs[2r+1]) owned by rank r
  // fused transfers: every rank's kernel has written its coarse rows into the full vector; gather the others' in place
  int fused_after_restrict(double *b_coarse_full) override
  {
    const int64_t U = coarse_full->level_pitch ? coarse_full->level_pitch : gc.unit;
    std::vector<int64_t> cnt((size_t)ctx->nranks), dsp((size_t)ctx->nranks);
    for (int r = 0; r < ctx->nranks; ++r) {
      cnt[(size_t)r] = U * (crows[2 * (size_t)r + 1] - crows[2 * (size_t)r]);
      dsp[(size_t)r] = U * crows[2 * (size_t)r];
    }
    return comm_allgatherv(ctx, b_coarse_full + dsp[(size_t)ctx->rank], b_coarse_full, cnt.data(), dsp.data(), ctx->stream);
  }
  int restrict_to(const double *r, double *bcoarse_full) override
  {
    PMG_TRY(fine->halo(r));
    const Geom &gf = fine->g;
    if (gc.nl > 0) {
      const Plan pl = gf.dim == 2 ? plan_nodes<2>(gc) : plan_nodes<3>(gc);
      PMG_PLAN_CHECK(pl);
      if (gf.dim == 2) restrict_kernel<2><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, r, fine->ghost_lo.p, fine->ghost_hi.p, slab.p);
      else restrict_kernel<3><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, r, fine->ghost_lo.p, fine->ghost_hi.p, slab.p);
      PMG_CUDA(cudaGetLastError());
      ctx->launches++;
    }
    return comm_allgatherv(ctx, slab.p, bcoarse_full, counts.data(), displs.data(), ctx->stream);
  }
  int restrict_pitched(double *r, double *bcoarse_full) override
  {
    Geom    gf;
    int64_t off;
    if (!fine->pitched_view(gf, off)) PMG_FAIL(PMG_ERR_SUP, "the fine operator has no pitched layout");
    PMG_TRY(fine->pitched_halo(r));
    if (gc.nl > 0) {
      const Plan pl = gf.dim == 2 ? plan_nodes<2>(gc) : plan_nodes<3>(gc);
      PMG_PLAN_CHECK(pl);
      const double *ro = r + off;
      if (gf.dim == 2) restrict_kernel<2><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, ro, ro - gf.unit, ro + gf.nl, slab.p);
      else if (pitched3_slab_ok(gf, gc)) restrict3_pitched_kernel<<<dim3((unsigned)((((gc.n0 + 3) >> 2) * gc.n1 + 255) / 256), (unsigned)(gc.shi - gc.slo)), 256, 0, ctx->stream>>>(gf, gc, ro, slab.p);
      else restrict_kernel<3><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, ro, ro - gf.unit, ro + gf.nl, slab.p);
      PMG_CUDA(cudaGetLastError());
      ctx->launches++;
    }
    return comm_allgatherv(ctx, slab.p, bcoarse_full, counts.data(), displs.data(), ctx->stream);
  }
  int prolong_pitched(const double *xc_full, double *xf) override
  {
    Geom    gf;
    int64_t off;
    if (!fine->pitched_view(gf, off)) PMG_FAIL(PMG_ERR_SUP, "the fine operator has no pitched layout");
    const double *xc = xc_full + gc.row0(); // the neighbouring units are simply adjacent in the replica
    const Plan    pl = gf.dim == 2 ? plan_nodes<2>(gf) : plan_nodes<3>(gf);
    PMG_PLAN_CHECK(pl);
    if (gf.dim == 2) prolong_kernel<2><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, xc, xc - gc.unit, xc + gc.nl, xf + off);
    else if (pitched3_slab_ok(gf, gc)) prolong3_pitched_kernel<<<dim3((unsigned)(((gf.ld >> 2) * gf.n1 + 255) / 256), (unsigned)(gf.shi - gf.slo)), 256, 0, ctx->stream>>>(gf, gc, xc, xc - gc.unit, xc + gc.nl, xf + off);
    else prolong_kernel<3><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, xc, xc - gc.unit, xc + gc.nl, xf + off);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }
  int prolong_add(const double *xc_full, double *xf) override
  {
    const Geom   &gf = fine->g;
    const double *xc = xc_full + gc.row0(); // the neighbouring units are simply adjacent in the replica
    const Plan pl = gf.dim == 2 ? plan_nodes<2>(gf) : plan_nodes<3>(gf);
    PMG_PLAN_CHECK(pl);
    if (gf.dim == 2) prolong_kernel<2><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, xc, xc - gc.unit, xc + gc.nl, xf);
    else prolong_kernel<3><<<pl.grid, pl.block, 0, ctx->stream>>>(gf, gc, xc, xc - gc.unit, xc + gc.nl, xf);
    PMG_CUDA(cudaGetLastError());
    ctx->launches++;
    return 0;
  }
};

} // namespace

bool grid_tail_level_ok(LevelOp *op)
{
  auto *bx = dynamic_cast<BoxOp *>(op);
  return bx && !bx->parallel && bx->g.slo == 0 && bx->g.shi == bx->g.nslow() && bx->g.nl < (1 << 30);
}

// The same tail in ONE CTA with every level vector in shared memory (tail2d.cuh), when the levels are 2D, have boundary
// classes and fit; `done` tells whether it ran.
static int grid_tail_smem_cycle(pmg_ctx ctx, int nlev, const TailLevelSpec *lv, const CholSampler &chol, int noise_mode, uint64_t seed, const TailNoise *ns, int nns, bool &done)
{
  using namespace tail2d;
  done = false;
  if (std::getenv("PMG_NO_TAIL_SMEM") || nlev < 2 || nlev > MAX_LEVELS || nns > MAX_NOISE || chol.n > 512 || !chol.use_gemv) return 0;
  static Args a;
  a.nlev = nlev;
  const int top = nlev - 1;
  int64_t   off = 0, updates = 0;
  std::vector<std::pair<const void *, double>> key;
  for (int l = 0; l < nlev; ++l) {
    auto *bx = dynamic_cast<BoxOp *>(lv[l].op);
    if (!bx || bx->g.dim != 2 || bx->parallel || bx->g.slo != 0 || bx->g.shi != bx->g.n1 || (l > 0 && !bx->classes_ok)) return 0;
    Level &L = a.lv[l];
    L.n0 = (int)bx->g.n0; L.n1 = (int)bx->g.n1; L.n = (int)bx->g.nl;
    L.xoff = (int)off; off += L.n;
    if (l < top) { L.boff = (int)off; off += L.n; }
    else L.boff = -1;
    L.ndirs = 0;
    L.omo   = 0;
    if (l == 0) continue;
    if (lv[l].ndirs > 8) return 0;
    L.ndirs = lv[l].ndirs;
    for (int q = 0; q < L.ndirs; ++q) L.dirs[q] = lv[l].dirs[q];
    L.omo = 1.0 - lv[l].coeffs->omega;
    key.emplace_back((const void *)bx, lv[l].coeffs->omega);
    updates += 2 * (int64_t)L.ndirs * bx->g.nl;
  }
  if ((int64_t)a.lv[0].n != chol.n) return 0;
  a.tmpoff = (int)off; off += chol.n;
  a.zoff   = (int)off; off += a.lv[top].n;
  const size_t fixed = sizeof(fastnormal::SharedTables) + (size_t)9 * MAX_LEVELS * sizeof(box2d::Cls);
  if (fixed + (size_t)off * sizeof(double) > 224 * 1024) return 0;
  a.woff = a.wtoff = -1;
  if (fixed + (size_t)(off + 2 * chol.n * chol.n) * sizeof(double) <= 224 * 1024) { // the coarsest sampler's factors fit as well
    a.woff  = (int)off; off += chol.n * chol.n;
    a.wtoff = (int)off; off += chol.n * chol.n;
  }
  const size_t sm = fixed + (size_t)off * sizeof(double);
  auto *tb = dynamic_cast<BoxOp *>(lv[top].op);
  if (tb->tail_cls_key != key) {
    tb->tail_cls_host.assign((size_t)9 * nlev, box2d::Cls{});
    for (int l = 1; l < nlev; ++l) {
      auto *bx = dynamic_cast<BoxOp *>(lv[l].op);
      for (int q = 0; q < 9; ++q) BoxOp::fill_class(tb->tail_cls_host[(size_t)9 * l + q], bx->cls_tab.c[q], lv[l].coeffs->omega);
    }
    PMG_TRY(tb->tail_cls.upload(tb->tail_cls_host, ctx->stream));
    PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    tb->tail_cls_key = key;
  }
  a.cls  = tb->tail_cls.p;
  a.btop = lv[top].b;
  a.xtop = lv[top].x;
  a.nc = (int)chol.n; a.W = chol.L.p; a.WT = chol.LT.p;
  a.mode = noise_mode; a.seed = seed;
  for (int q = 0; q < nns; ++q) a.ns[q] = ns[q];
  static size_t sm_set[16] = {0};
  const int     dv = ctx->device & 15;
  if (sm > sm_set[dv]) {
    PMG_CUDA(cudaFuncSetAttribute(tail2d_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(sm, 48 * 1024)));
    sm_set[dv] = std::max<size_t>(sm, 48 * 1024);
  }
  PMG_CUDA(launch_pdl(ctx->stream, tail2d_kernel, dim3(1), dim3(NT), sm, a));
  ctx->launches++;
  ctx->dof_updates += updates;
  done = true;
  return 0;
}

// size / type test of the shared-memory tail for levels 0 .. nlev-1 (the V-cycle set-up asks before it lays the levels out)
bool grid_tail_smem_fits(int nlev, LevelOp *const *ops, int64_t chol_n)
{
  if (std::getenv("PMG_NO_TAIL_SMEM") || nlev < 2 || nlev > tail2d::MAX_LEVELS || chol_n > 512) return false;
  int64_t off = 0;
  for (int l = 0; l < nlev; ++l) {
    auto *bx = dynamic_cast<BoxOp *>(ops[l]);
    if (!bx || bx->g.dim != 2 || bx->parallel || bx->g.slo != 0 || bx->g.shi != bx->g.n1 || (l > 0 && !bx->classes_ok)) return false;
    off += (l < nlev - 1 ? 2 : 1) * bx->g.nl;
    if (l == 0 && bx->g.nl != chol_n) return false;
  }
  auto *tb = dynamic_cast<BoxOp *>(ops[nlev - 1]);
  off += chol_n + tb->g.nl;
  return sizeof(fastnormal::SharedTables) + (size_t)9 * tail2d::MAX_LEVELS * sizeof(box2d::Cls) + (size_t)off * sizeof(double) <= 224 * 1024;
}

int grid_tail_cycle(pmg_ctx ctx, int nlev, const TailLevelSpec *lv, const CholSampler &chol, int noise_mode, uint64_t seed, const TailNoise *ns, int nns)
{
  if (chol.packed) PMG_FAIL(PMG_ERR_SUP, "coarse tail: the coarsest sampler keeps L^-1 packed (n = %lld), the tail reads it as a full matrix", (long long)chol.n);
  {
    bool done = false;
    PMG_TRY(grid_tail_smem_cycle(ctx, nlev, lv, chol, noise_mode, seed, ns, nns, done));
    if (done) return 0;
  }
  if (nlev < 2 || nlev > TAIL_MAX_LEVELS || nns > TAIL_MAX_NOISE) PMG_FAIL(PMG_ERR_SUP, "coarse tail: %d levels / %d noise blocks exceed the kernel's tables", nlev, nns);
  static TailArgs a; // ~4 KB: filled per launch, passed by value
  a.nlev = nlev;
  int     dim = 2;
  int64_t updates = 0;
  for (int l = 0; l < nlev; ++l) {
    auto *bx = dynamic_cast<BoxOp *>(lv[l].op);
    if (!bx) PMG_FAIL(PMG_ERR_SUP, "coarse tail: level %d is not a stencil-array operator", l);
    dim             = bx->g.dim;
    TailLevelDev &d = a.lv[l];
    d.g             = bx->g;
    d.bc            = bx->bc;
    d.coef          = bx->coef.p;
    d.b = lv[l].b; d.x = lv[l].x; d.r = lv[l].r;
    d.ndirs = 0;
    if (l == 0) continue;
    const SweepCoeffs &co = *lv[l].coeffs;
    if (d.bc.on) { // BoxOp::sweep's interior coefficients
      const double dd  = d.bc.c[bx->nst() / 2];
      double       inv = 1.0 / dd;
      d.bc.idiag       = inv * co.omega;
      d.bc.sqrtdiag    = std::sqrt(std::fabs(dd)) * std::sqrt((2 - co.omega) / co.omega);
    }
    d.idiag = co.idiag.p; d.sqrtdiag = co.sqrtdiag.p;
    d.omo   = 1.0 - co.omega;
    d.ndirs = lv[l].ndirs;
    for (int q = 0; q < d.ndirs; ++q) d.dirs[q] = lv[l].dirs[q];
    updates += 2 * (int64_t)d.ndirs * bx->g.nl;
  }
  a.nc = (int)chol.n; a.W = chol.L.p; a.WT = chol.LT.p; a.tmp0 = chol.tmp.p;
  a.mode = noise_mode; a.seed = seed;
  for (int q = 0; q < nns; ++q) a.ns[q] = ns[q];
  // one cluster of up to 8 CTAs x 1024 threads; small tails run in fewer CTAs (a barrier between fewer SMs is cheaper)
  const int64_t big = a.lv[nlev - 1].g.nl;
  static int cl_max_dev[16] = {0}; // per device: 16 CTAs per cluster where the device allows it (non-portable size), else the portable 8
  int       &cl_max = cl_max_dev[ctx->device & 15];
  if (!cl_max) {
    cl_max = 8;
    bool ok = cudaFuncSetAttribute(grid_tail_kernel<2>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess && cudaFuncSetAttribute(grid_tail_kernel<3>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess;
    if (ok) {
      cudaLaunchConfig_t q = {};
      q.gridDim = dim3(16); q.blockDim = dim3(1024);
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = 16; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
      q.attrs = qa; q.numAttrs = 1;
      int nclusters = 0;
      if (cudaOccupancyMaxActiveClusters(&nclusters, grid_tail_kernel<2>, &q) == cudaSuccess && nclusters >= 1) cl_max = 16;
    }
    (void)cudaGetLastError();
  }
  int cl = big > 40000 ? cl_max : big > 9000 ? 8 : big > 2000 ? 4 : big > 500 ? 2 : 1;
  static const int cl_env = std::getenv("PMG_TAIL_CLUSTER") ? std::atoi(std::getenv("PMG_TAIL_CLUSTER")) : 0;
  if (cl_env >= 1 && cl_env <= cl_max) cl = cl_env;
  a.cluster = cl;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim  = dim3((unsigned)cl);
  cfg.blockDim = dim3(1024);
  cfg.stream   = ctx->stream;
  cudaLaunchAttribute at[1];
  at[0].id               = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)cl;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs    = at;
  cfg.numAttrs = 1;
  if (dim == 2) PMG_CUDA(cudaLaunchKernelEx(&cfg, grid_tail_kernel<2>, a));
  else PMG_CUDA(cudaLaunchKernelEx(&cfg, grid_tail_kernel<3>, a));
  PMG_CUDA(cudaGetLastError());
  ctx->launches++;
  ctx->dof_updates += updates;
  return 0;
}

int make_laplace_op(pmg_ctx ctx, int dim, int64_t nx, int64_t ny, int64_t nz, double kappa, int64_t slab_lo, int64_t slab_hi, std::unique_ptr<LevelOp> &op)
{
  const int64_t n[3]  = {nx, ny, dim == 3 ? nz : 1};
  const int64_t nslow = dim == 3 ? nz : ny;
  if (slab_hi == 0 && slab_lo == 0) slab_hi = nslow;
  if (slab_lo < 0 || slab_hi > nslow || slab_lo >= slab_hi) PMG_FAIL(PMG_ERR_ARG, "bad slab [%lld, %lld) of %lld", (long long)slab_lo, (long long)slab_hi, (long long)nslow);
  if ((slab_lo != 0 || slab_hi != nslow) && ctx->nranks == 1) PMG_FAIL(PMG_ERR_ARG, "a partial slab needs an initialised communicator (pmg_ctx_comm_init)");
  if (nx * ny * n[2] >= ((int64_t)1 << 40)) PMG_FAIL(PMG_ERR_ARG, "grid too large");
  auto o   = std::make_unique<LapOp>();
  o->ctx   = ctx;
  o->g     = make_geom(dim, n, slab_lo, slab_hi);
  o->kappa = kappa;
  o->fill_tab(1.0, o->tab);
  PMG_TRY(o->init_ghosts());
  op = std::move(o);
  return 0;
}

// Galerkin hierarchy below a matrix-free fine operator, built on the device (levels are numbered like PCMG: 0 = coarsest).
// With several ranks the upper levels stay slab-distributed; from the first level that is small (at most
// `replicate_below` nodes globally), too thin to split (a rank would own fewer than two units) or the coarsest, every rank
// holds the whole level.
int build_structured_hierarchy(pmg_ctx ctx, LevelOp *fine_op, int nlevels, int64_t replicate_below, std::vector<std::unique_ptr<LevelOp>> &ops, std::vector<std::unique_ptr<Transfer>> &transfers)
{
  auto *fine = dynamic_cast<GridOp *>(fine_op);
  if (!fine) PMG_FAIL(PMG_ERR_SUP, "not a grid operator");
  ops.clear();
  transfers.clear();
  ops.resize((size_t)nlevels);
  transfers.resize((size_t)nlevels);
  const int            R = ctx->nranks, me = ctx->rank;
  std::vector<int64_t> slabs((size_t)2 * R, 0);
  bool                 dist = fine->parallel;
  if (dist) {
    const int64_t mine[2] = {fine->g.slo, fine->g.shi};
    PMG_TRY(comm_allgather_i64(ctx, mine, 2, slabs.data()));
    for (int r = 0; r < R; ++r)
      if (slabs[2 * r] != (r ? slabs[2 * r - 1] : 0) || slabs[2 * r + 1] <= slabs[2 * r] || (r == R - 1 && slabs[2 * r + 1] != fine->g.nslow()))
        PMG_FAIL(PMG_ERR_ARG, "gamgmc: the slabs of the ranks must tile the grid in rank order (rank %d owns [%lld, %lld))", r, (long long)slabs[2 * r], (long long)slabs[2 * r + 1]);
    if (nlevels < 2) PMG_FAIL(PMG_ERR_SUP, "gamgmc on a distributed grid needs at least two levels (the coarsest level is replicated)");
  }
  std::vector<std::unique_ptr<BoxOp>> keep; // distributed shadows of replicated levels are only needed during set-up
  GridOp *cur = fine;
  for (int l = nlevels - 1; l >= 1; --l) {
    const Geom   &gf = cur->g;
    const int64_t nf[3] = {gf.n0, gf.n1, gf.n2};
    int64_t       nc[3];
    host_q1_dims(gf.dim, nf, nc);
    if (nc[0] * nc[1] * nc[2] == nf[0] * nf[1] * nf[2]) PMG_FAIL(PMG_ERR_ARG, "gamgmc: cannot coarsen a %lldx%lldx%lld grid further (level %d)", (long long)nf[0], (long long)nf[1], (long long)nf[2], l);
    int64_t clo = (gf.slo + 1) / 2, chi = (gf.shi + 1) / 2; // coarse unit J is owned by the owner of fine unit 2J
    bool    replicate = false;
    std::vector<int64_t> cs((size_t)2 * R, 0);
    if (dist) {
      int64_t minthick = INT64_MAX;
      for (int r = 0; r < R; ++r) {
        cs[2 * r]     = (slabs[2 * r] + 1) / 2;
        cs[2 * r + 1] = (slabs[2 * r + 1] + 1) / 2;
        minthick      = std::min(minthick, cs[2 * r + 1] - cs[2 * r]);
      }
      replicate = l - 1 == 0 || nc[0] * nc[1] * nc[2] <= replicate_below || minthick < 2;
    }
    auto c = std::make_unique<BoxOp>();
    c->ctx = ctx;
    c->g   = make_geom(gf.dim, nc, clo, chi);
    PMG_TRY(c->init_ghosts());
    PMG_TRY(c->coef.alloc((size_t)c->nst() * std::max<int64_t>(c->g.nl, 1)));
    const Geom &gc = c->g;
    if (gc.nl > 0) {
      if (auto *lap = dynamic_cast<LapOp *>(cur)) {
        if (gf.dim == 2) galerkin_kernel<2, FineLap<2>><<<nblocks(gc.nl, 128), 128, 0, ctx->stream>>>(FineLap<2>{gf, lap->tab}, gc, c->coef.p, gc.nl);
        else galerkin_kernel<3, FineLap<3>><<<nblocks(gc.nl, 128), 128, 0, ctx->stream>>>(FineLap<3>{gf, lap->tab}, gc, c->coef.p, gc.nl);
      } else {
        auto *box = static_cast<BoxOp *>(cur);
        if (gf.dim == 2) galerkin_kernel<2, FineBox<2>><<<nblocks(gc.nl, 128), 128, 0, ctx->stream>>>(FineBox<2>{gf, box->coef.p, box->coef_lo.p, box->coef_hi.p, gf.nl}, gc, c->coef.p, gc.nl);
        else galerkin_kernel<3, FineBox<3>><<<nblocks(gc.nl, 128), 128, 0, ctx->stream>>>(FineBox<3>{gf, box->coef.p, box->coef_lo.p, box->coef_hi.p, gf.nl}, gc, c->coef.p, gc.nl);
      }
      PMG_CUDA(cudaGetLastError());
    }
    PMG_CUDA(cudaStreamSynchronize(ctx->stream));
    if (!replicate) {
      PMG_TRY(c->exchange_coef_ghosts());
      PMG_TRY(c->detect_interior());
      PMG_TRY(c->detect_classes());
      PMG_TRY(c->detect_classes3());
      auto t    = std::make_unique<GridTransfer>();
      t->ctx    = ctx;
      t->fine   = cur;
      t->coarse = c.get();
      transfers[(size_t)l] = std::move(t);
      cur                  = c.get();
      ops[(size_t)l - 1]   = std::move(c);
      slabs                = cs;
    } else { // gather the coefficient arrays: from here down every rank holds whole levels
      auto full = std::make_unique<BoxOp>();
      full->ctx = ctx;
      full->g   = make_geom(gf.dim, nc, 0, gf.dim == 2 ? nc[1] : nc[2]);
      PMG_TRY(full->init_ghosts());
      PMG_TRY(full->coef.alloc((size_t)full->nst() * full->g.nl));
      auto t    = std::make_unique<ReplicatingTransfer>();
      t->ctx    = ctx;
      t->fine   = cur;
      t->gc     = gc;
      t->coarse_full = full.get();
      t->crows       = cs;
      t->counts.resize((size_t)R);
      t->displs.resize((size_t)R);
      for (int r = 0; r < R; ++r) {
        t->counts[(size_t)r] = gc.unit * (cs[2 * r + 1] - cs[2 * r]);
        t->displs[(size_t)r] = gc.unit * cs[2 * r];
      }
      PMG_TRY(t->slab.alloc((size_t)std::max<int64_t>(gc.nl, 1)));
      for (int s = 0; s < full->nst(); ++s) PMG_TRY(comm_allgatherv(ctx, c->coef.p + (size_t)s * gc.nl, full->coef.p + (size_t)s * full->g.nl, t->counts.data(), t->displs.data(), ctx->stream));
      PMG_CUDA(cudaStreamSynchronize(ctx->stream));
      PMG_TRY(full->detect_interior());
      PMG_TRY(full->detect_classes());
      PMG_TRY(full->detect_classes3());
      transfers[(size_t)l] = std::move(t);
      cur                  = full.get();
      ops[(size_t)l - 1]   = std::move(full);
      dist                 = false;
      (void)me;
    }
  }
  return 0;
}
