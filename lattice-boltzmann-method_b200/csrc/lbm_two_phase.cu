// lbm_two_phase.cu — kernels and step sequencing of the colour-gradient models
// (LBM_MODEL_MRTCG, LBM_MODEL_RK).  Arithmetic: lbm_two_phase.cuh.
//
// Steady state (the stored state is post-collision): ONE pass over the grid per time step,
//   k_tp_fused : a block owns a strip of columns and marches down a band of rows.  Per row it pulls
//              both lattices of row r+H (H = stencil half-width: 2 for the 5x5 differences of
//              MRTCG, 1 for the 3x3 ones of RK), computes the moments of that row — what the
//              drivers compute at the end of an iteration (mrtcg_rayleigh_taylor.cpp:472-477) —
//              into a shared-memory ring of 2H+2 rows, then collides row r from the ring (stencil
//              + own moments) and the re-pulled populations (an L1/L2 hit: the same block read them
//              H iterations earlier), and writes f_coll of both colours.
//              DRAM traffic per node: 144 R + 144 W + the strip/band halo re-reads (~3-6 %, mostly
//              L2 hits) — the moment planes never travel, which is below SURVEY §8(d)'s 352 B / 304 B
//              models (those assume a stored moment field).
//   The moment planes survive only where something other than the fused kernel needs them: listed
//   (table-driven) nodes and their 2-neighbourhood, the replicate padding, the two rows exchanged
//   across a slab cut.  k_tp_moments_nodes fills that thin region (O(X+Y) nodes) before the fused
//   kernel, which reads plane values there instead of recomputing.
// First step after an import (the stored state is post-stream and the caller supplied u): the
// two-pass pair k_tp_collide_interior<MODE_LOCAL> over the full moment planes.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <vector>

#include "lbm_internal.hpp"
#include "lbm_two_phase.cuh"
#include "lbm_async.cuh"

// (Tried and dropped on the fused kernel: L2 eviction-policy hints on its two reads and its stores, no gain - DESIGN §3.3;
// prefetch.global.L2 of the next iteration's second pull, -2 %.)

namespace lbm
{

struct TpKernel;   // an entry of tp_kernels / csf_kernels: the row-marching kernel of the step, chosen once per domain
struct CsfKernel;

struct TwoPhaseState
{
  MomGeom mg;
  double* mom = nullptr;  // M_COUNT planes
  TpParams p;
  int model = TP_MRTCG;
  // fused step: where the moment planes stay authoritative
  bool planes_full = false;            // planes hold the moments of every own node of the current state
  bool region_dirty = true;            // (re)build the lists below
  unsigned char* d_rowflag = nullptr;  // [Xl] 1 = every node of the row takes its moments from the planes
  int* d_region = nullptr;             // [n_region] local node ids x * Y + y the region kernel recomputes, by rows
  int n_region = 0;
  int n_region_lo = 0, n_region_hi = 0;  // how many of them lie in rows 0, 1 (the head of the list) and Xl-2, Xl-1 (its tail)
  bool ring_overlap = false;           // LBM_TP_OVERLAP=1: the ranks of a ring send their halos behind the interior bands (tp_steps_ring)
  int rows_per_block = 64;             // band height of the row-marching kernel (band_rows, once per rule set)
  const TpKernel* kernel = nullptr;    // TP_MRTCG / TP_RK: the row-marching kernel (LBM_TP_STAGED, LBM_TP_STASH, LBM_TP_NS, LBM_TP_PIPE)
  double* aux = nullptr;               // TP_CSF: A_COUNT planes in the moment-plane geometry (normal n, interfacial tension Fs)
  int rpb_override = 0;
  // TP_CSF single-pass variant
  bool csf_fused = true;               // the single-pass step (LBM_CSF_FUSED=0: three passes)
  const CsfKernel* csf_kernel = nullptr;  // its row-marching kernel (LBM_CSF_STAGED, LBM_CSF_PIPE)
  double* aux_next = nullptr;          // second aux set: a fused step reads Fs from aux and writes it here, then the two swap
  unsigned char* d_csf_flags = nullptr;  // [Xl] bit 0: moments of the whole row from the planes; bit 1: normals too
  int* d_csf_list4 = nullptr;          // interior-column nodes whose moments the pre-pass writes to the planes
  int* d_csf_list2 = nullptr;          // nodes (any column) whose normals the pre-pass writes to the planes
  int n_csf_list4 = 0, n_csf_list2 = 0;
  bool csf_lists_dirty = true;
};

static inline int cdiv(long long a, int b) { return (int)((a + b - 1) / b); }

constexpr int TPF_NT = 128;  // threads per block of the row-marching kernels = columns of a strip including its halo columns

// Rows per band of the row-marching kernels.  Tall bands amortise the warm-up rows above and below a band (their
// populations are read and their moments formed a second time) and the per-block set-up; short bands shorten the tail:
// the last blocks of the grid end at different times and nothing fills the SMs they leave.  Model, fitted to a sweep of
// the RK kernel at 4096^2 on the B200 (24 .. 128 rows: 0.867, 0.856, 0.857, 0.860, 0.870, 0.884, 0.908, 0.971 ms):
//     time ~ (blocks / resident) * d + 0.84 * d,   d = rows + 0.6 * warm-up rows + 1.5   (rows' worth of work per block)
// Round 1's rule (six waves' worth of blocks) and a first whole-waves rule both chose 51 .. 84 rows there; the minimum
// is at 32 .. 40.  Large grids (MRTCG 16384^2: 38 waves at 128 rows) are flat within 1 % and keep tall bands.
static int pick_band_rows(int Xl, int strips, int resident_blocks, int warmup_rows, int cap = 128)
{
  if (Xl <= 24) return std::max(Xl, 1);
  double best = 1e300;
  int best_rpb = std::min(cap, Xl);
  for (int rpb = std::min(cap, Xl); rpb >= 24; rpb--)
  {
    const double blocks = (double)strips * cdiv(Xl, rpb);
    const double d = rpb + 0.6 * warmup_rows + 1.5;
    const double t = blocks / std::max(resident_blocks, 1) * d + 0.84 * d;
    if (t < best * (1.0 - 1e-9))
    {
      best = t;
      best_rpb = rpb;
    }
  }
  return best_rpb;
}

// blocks of `kernel` (TPF_NT threads, `smem` dynamic bytes) the device keeps resident at once.  From the kernel's own
// resource use and the SM's limits rather than the occupancy calculator, whose answer depends on the shared-memory
// carve-out in force when it is asked (it said one block per SM for a kernel that runs two).
template <class K>
static int resident_blocks_of(const lbm_domain* d, K kernel, size_t smem)
{
  int sms = 0, smem_sm = 0, regs_sm = 0;
  cudaFuncAttributes fa{};
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, d->cfg.device) != cudaSuccess || sms < 1) sms = 148;
  if (cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, d->cfg.device) != cudaSuccess || smem_sm < 1) smem_sm = 233472;
  if (cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, d->cfg.device) != cudaSuccess || regs_sm < 1) regs_sm = 65536;
  int per_sm = 2;
  if (cudaFuncGetAttributes(&fa, (const void*)kernel) == cudaSuccess && fa.numRegs > 0)
  {
    const int regs_thread = (fa.numRegs + 7) / 8 * 8;  // allocation granularity
    const int by_regs = regs_sm / (regs_thread * TPF_NT);
    const int by_smem = (int)(smem_sm / (smem + fa.sharedSizeBytes + 1024));  // 1 KB per block is the system's
    per_sm = std::max(1, std::min({by_regs, by_smem, 16}));
  }
  cudaGetLastError();
  return per_sm * sms;
}

constexpr int TILE_X = 8, TILE_Y = 32, HALO = 2;
constexpr int SM_X = TILE_X + 2 * HALO, SM_Y = TILE_Y + 2 * HALO;

// ------------------------------------------------------------------------------------------------
// loaders
// ------------------------------------------------------------------------------------------------
template <int MODE>
__device__ __forceinline__ void tp_load_interior(const double* __restrict__ src, const SlabGeom& g, int x, int y, double (&f)[9])
{
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    if constexpr (MODE == MODE_LOCAL) f[q] = src[q * g.plane + node_off(g, x, y)];
    else f[q] = src[q * g.plane + node_off(g, x - CX(q), y - CY(q))];
  }
}

// Pull through a per-thread node pointer (src + node_off(g, x, y)) plus WARP-UNIFORM offsets
// q * plane - c_x * pitch - c_y: two integer instructions per access instead of a 64-bit index
// rebuilt per thread and per population.
__device__ __forceinline__ void tp_pull_at(const double* __restrict__ node, const SlabGeom& g, double (&f)[9])
{
#pragma unroll
  for (int q = 0; q < 9; q++) f[q] = __ldg(node + ((long long)q * g.plane - (long long)CX(q) * g.pitch - CY(q)));
}

template <int MODE>
__device__ __forceinline__ void tp_load_listed(const double* __restrict__ src, const SlabGeom& g, const BoundaryTable& t,
                                               int lattice, int i, int x, int y, double (&f)[9])
{
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    if constexpr (MODE == MODE_LOCAL) f[q] = src[q * g.plane + node_off(g, x, y)];
    else
    {
      const BcEntry e = t.ent[(long long)(lattice * 9 + q) * t.n + i];
      f[q] = e.coef * src[e.src] + e.cst;
    }
  }
}

// finite differences straight from the padded global planes (listed nodes, few of them)
template <int MODEL>
__device__ __forceinline__ void tp_stencil_global(const TpParams& p, const double* __restrict__ mom, const MomGeom& mg,
                                                  int x, int y, TpStencil& st)
{
  const long long o = mom_off(mg, x, y);
  const double* ph = mom + M_PH * mg.mplane;
  st.gx = st.gy = st.DxQx = st.DyQy = 0.0;
  if constexpr (MODEL == TP_RK)
  {
    // rk_static_droplet_test.cpp:52-62: "x" kernel differentiates along axis 1, "y" kernel along axis 0
#pragma unroll
    for (int a = -1; a <= 1; a++)
#pragma unroll
      for (int b = -1; b <= 1; b++)
      {
        const double v = ph[o + (long long)a * mg.pm + b];
        const double wa = a == 0 ? 1.0 / 9.0 : 1.0 / 36.0, wb = b == 0 ? 1.0 / 9.0 : 1.0 / 36.0;
        if (b != 0) st.gx += (3.0 * (wa * (double)b)) * v;
        if (a != 0) st.gy += (3.0 * (wb * (double)a)) * v;
      }
  }
  else
  {
    const double* RR = mom + M_RR * mg.mplane;
    const double* RB = mom + M_RB * mg.mplane;
    const double* UX = mom + M_UX * mg.mplane;
    const double* UY = mom + M_UY * mg.mplane;
#pragma unroll
    for (int a = -2; a <= 2; a++)
#pragma unroll
      for (int b = -2; b <= 2; b++)
      {
        if (a == 0 && b == 0) continue;
        const long long k = o + (long long)a * mg.pm + b;
        const double w = XI5(a, b);
        const double rr = RR[k], rb = RB[k], ux = UX[k], uy = UY[k], phv = ph[k];
        if (a != 0)
        {
          st.gx += (w * (double)a) * phv;
          st.DxQx += (w * (double)a) * ((p.cr * rr + p.cb * rb) * ux);
        }
        if (b != 0)
        {
          st.gy += (w * (double)b) * phv;
          st.DyQy += (w * (double)b) * ((p.cr * rr + p.cb * rb) * uy);
        }
      }
  }
}

// ------------------------------------------------------------------------------------------------
// collide, interior: block (TILE_Y, TILE_X) threads, one node per thread, columns 1 .. Y-2
// ------------------------------------------------------------------------------------------------
template <int MODEL, int MODE>
__global__ void __launch_bounds__(TILE_X* TILE_Y)
k_tp_collide_interior(const double* __restrict__ rsrc, const double* __restrict__ bsrc, double* __restrict__ rdst,
                      double* __restrict__ bdst, const SlabGeom g, const MomGeom mg, const double* __restrict__ mom,
                      const TpParams p, int row_begin, int row_end)
{
  constexpr int NF = MODEL == TP_MRTCG ? 3 : 1;
  __shared__ double sm[NF][SM_X][SM_Y + 1];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int x_t = row_begin + blockIdx.y * TILE_X, y_t = 1 + blockIdx.x * TILE_Y;  // tile origin
  // stage phase (and the four momentum fields Q_k = (1.8 alpha_k - 0.8) rho_k u) with the halo
  for (int n = ty * TILE_Y + tx; n < SM_X * SM_Y; n += TILE_X * TILE_Y)
  {
    const int i = n / SM_Y, j = n % SM_Y;
    int xs = x_t - HALO + i, ys = y_t - HALO + j;
    xs = min(xs, g.Xl + 1);
    ys = min(ys, g.Y + 1);
    const long long k = mom_off(mg, xs, ys);
    sm[0][i][j] = mom[M_PH * mg.mplane + k];
    if constexpr (MODEL == TP_MRTCG)
    {
      const double rr = mom[M_RR * mg.mplane + k], rb = mom[M_RB * mg.mplane + k];
      const double ux = mom[M_UX * mg.mplane + k], uy = mom[M_UY * mg.mplane + k];
      const double cq = p.cr * rr + p.cb * rb;
      sm[1][i][j] = cq * ux;
      sm[2][i][j] = cq * uy;
    }
  }
  __syncthreads();
  const int x = x_t + ty, y = y_t + tx;
  if (x >= row_end || y > g.Y - 2) return;

  TpStencil st;
  st.gx = st.gy = st.DxQx = st.DyQy = 0.0;
  const int ci = ty + HALO, cj = tx + HALO;
  if constexpr (MODEL == TP_RK)
  {
#pragma unroll
    for (int a = -1; a <= 1; a++)
#pragma unroll
      for (int b = -1; b <= 1; b++)
      {
        const double v = sm[0][ci + a][cj + b];
        const double wa = a == 0 ? 1.0 / 9.0 : 1.0 / 36.0, wb = b == 0 ? 1.0 / 9.0 : 1.0 / 36.0;
        if (b != 0) st.gx += (3.0 * (wa * (double)b)) * v;
        if (a != 0) st.gy += (3.0 * (wb * (double)a)) * v;
      }
  }
  else
  {
#pragma unroll
    for (int a = -2; a <= 2; a++)
#pragma unroll
      for (int b = -2; b <= 2; b++)
      {
        if (a == 0 && b == 0) continue;
        const double w = XI5(a, b);
        if (a != 0)
        {
          st.gx += (w * (double)a) * sm[0][ci + a][cj + b];
          st.DxQx += (w * (double)a) * sm[1][ci + a][cj + b];
        }
        if (b != 0)
        {
          st.gy += (w * (double)b) * sm[0][ci + a][cj + b];
          st.DyQy += (w * (double)b) * sm[2][ci + a][cj + b];
        }
      }
  }
  const long long km = mom_off(mg, x, y);
  const double rr = mom[M_RR * mg.mplane + km], rb = mom[M_RB * mg.mplane + km];
  const double ux = mom[M_UX * mg.mplane + km], uy = mom[M_UY * mg.mplane + km];
  const double ph = sm[0][ci][cj];

  double fr[9], fb[9];
  tp_load_interior<MODE>(rsrc, g, x, y, fr);
  tp_load_interior<MODE>(bsrc, g, x, y, fb);
  tp_collide<MODEL>(p, fr, fb, rr, rb, ux, uy, ph, st);
  const long long o = node_off(g, x, y);
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    rdst[q * g.plane + o] = fr[q];
    bdst[q * g.plane + o] = fb[q];
  }
}

// ------------------------------------------------------------------------------------------------
// fused step: moments of row r+H into a shared-memory ring, collision of row r out of it
// ------------------------------------------------------------------------------------------------

template <int MODEL>
struct TpFused
{
  static constexpr int H = MODEL == TP_MRTCG ? 2 : 1;   // stencil half-width
  static constexpr int NR = 2 * H + 2;                  // ring rows: 2H+1 live + the one being written
  // ring fields: phase, [Q_x, Q_y,] rho_r, rho_b, u_x, u_y
  static constexpr int NF = MODEL == TP_MRTCG ? 7 : 5;
  static constexpr int F_RR = NF - 4, F_RB = NF - 3, F_UX = NF - 2, F_UY = NF - 1;
  static constexpr int USEFUL = TPF_NT - 2 * H;         // columns a strip collides
  static constexpr size_t SMEM = sizeof(double) * NF * NR * TPF_NT;
};

// stencil at column t out of the ring; row_of(a) = element offset (slot * NT) of the ring row a rows from the centre
template <int MODEL, class RowOf>
__device__ __forceinline__ void tp_ring_stencil_at(const double* __restrict__ sm, RowOf row_of, int t, TpStencil& st)
{
  using C = TpFused<MODEL>;
  constexpr int NR = C::NR, NT = TPF_NT;
  auto S = [&](int f, int off, int col) -> double { return sm[f * NR * NT + off + col]; };
  st.gx = st.gy = st.DxQx = st.DyQy = 0.0;
  if constexpr (MODEL == TP_RK)
  {
#pragma unroll
    for (int a = -1; a <= 1; a++)
    {
      const int sa = row_of(a);
#pragma unroll
      for (int b = -1; b <= 1; b++)
      {
        const double v = S(0, sa, t + b);
        const double wa = a == 0 ? 1.0 / 9.0 : 1.0 / 36.0, wb = b == 0 ? 1.0 / 9.0 : 1.0 / 36.0;
        if (b != 0) st.gx += (3.0 * (wa * (double)b)) * v;
        if (a != 0) st.gy += (3.0 * (wb * (double)a)) * v;
      }
    }
  }
  else
  {
#pragma unroll
    for (int a = -2; a <= 2; a++)
    {
      const int sa = row_of(a);
#pragma unroll
      for (int b = -2; b <= 2; b++)
      {
        if (a == 0 && b == 0) continue;
        const double w = XI5(a, b);
        if (a != 0)
        {
          st.gx += (w * (double)a) * S(0, sa, t + b);
          st.DxQx += (w * (double)a) * S(1, sa, t + b);
        }
        if (b != 0)
        {
          st.gy += (w * (double)b) * S(0, sa, t + b);
          st.DyQy += (w * (double)b) * S(2, sa, t + b);
        }
      }
    }
  }
}

// stencil of row-slot sc, column t, out of the ring
template <int MODEL>
__device__ __forceinline__ void tp_ring_stencil(const double* __restrict__ sm, int sc, int t, TpStencil& st)
{
  constexpr int NR = TpFused<MODEL>::NR;
  // (a compare-and-wrap instead of the constant division measured 0 - 1.5 % slower)
  tp_ring_stencil_at<MODEL>(sm, [&](int a) { return ((sc + NR + a) % NR) * TPF_NT; }, t, st);
}

// grid: x = strips of USEFUL columns starting at column 1, y = bands of rows_per_block rows.
// Iteration r of the row loop:   A  issue the pulls of row r (both lattices)
//                                B  collide row r - LAG out of the ring (rows r-LAG-H .. r-LAG+H)
//                                C  moments of row r -> ring slot of r ;  __syncthreads
// PIPE = false: LAG = H and B runs after C and the barrier (collision of row r-H sees row r);
// PIPE = true : LAG = H + 1 and B runs between A and C, so the DRAM latency of A hides under the fp64
//               work of B (software pipelining, 36 more live registers).
// Resident blocks per SM the register allocation aims at.  Measured on B200 at 8192^2 (MRTCG, pipelined):
// 2 blocks (208 regs) 12.1 GLUPS, 3 blocks (168 regs, no spills) 12.9 GLUPS, 4 blocks (128 regs, spills) 8.0 GLUPS.
template <int MODEL, bool PIPE>
__global__ void __launch_bounds__(TPF_NT, MODEL == TP_MRTCG ? (PIPE ? 3 : 4) : 3)
k_tp_fused(const double* __restrict__ rsrc, const double* __restrict__ bsrc, double* __restrict__ rdst,
           double* __restrict__ bdst, const SlabGeom g, const MomGeom mg, const double* __restrict__ mom, const TpParams p,
           const unsigned char* __restrict__ rowflag, int rows_per_block, int band_lo, int band_jump)
{
  using C = TpFused<MODEL>;
  constexpr int H = C::H, NR = C::NR, NT = TPF_NT, LAG = PIPE ? H + 1 : H;
  extern __shared__ double sm[];  // [NF][NR][NT]
  auto S = [&](int f, int slot, int col) -> double& { return sm[(f * NR + slot) * NT + col]; };

  const int t = threadIdx.x;
  const int y = 1 + blockIdx.x * C::USEFUL - H + t;
  const int xb = ((int)blockIdx.y < band_lo ? (int)blockIdx.y : (int)blockIdx.y + band_jump) * rows_per_block;  // (0, 0): every band; see tp_launch_fused
  const int xe = min(xb + rows_per_block, g.Xl);
  const bool col_ok = y >= -2 && y <= g.Y + 1;           // inside the padded planes
  const bool col_plane = y < 1 || y > g.Y - 2;           // edge columns (listed nodes) and the padding
  const bool collider = t >= H && t < NT - H && y >= 1 && y <= g.Y - 2;

  // node pointers of (r, y) in both source lattices, advanced row by row
  const long long o0 = node_off(g, xb - H, y);
  const double* pr = rsrc + o0;
  const double* pb = bsrc + o0;
  const long long back = (long long)LAG * g.pitch;

  auto collide_row = [&](int sc) {
    // the second pull of this row (an L2 hit) first, so that its latency hides under the stencil arithmetic
    double fr[9], fb[9];
    tp_pull_at(pr - back, g, fr);
    tp_pull_at(pb - back, g, fb);
    TpStencil st;
    tp_ring_stencil<MODEL>(sm, sc, t, st);
    const double rr = S(C::F_RR, sc, t), rb = S(C::F_RB, sc, t);
    const double ux = S(C::F_UX, sc, t), uy = S(C::F_UY, sc, t), ph = S(0, sc, t);
    tp_collide<MODEL>(p, fr, fb, rr, rb, ux, uy, ph, st);
    double* wr = rdst + ((pr - back) - rsrc);
    double* wb = bdst + ((pr - back) - rsrc);
#pragma unroll
    for (int q = 0; q < 9; q++)
    {
      wr[(long long)q * g.plane] = fr[q];
      wb[(long long)q * g.plane] = fb[q];
    }
  };

  // the band's row flags once, in shared memory: a global load per iteration sat on the critical path of the
  // plane-or-pull decision (5 % of all stall samples in the ncu source view)
  __shared__ unsigned char sflag[128 + 2 * H + 2];
  for (int k = t; k < xe - xb + 2 * H; k += NT)
  {
    const int r = xb - H + k;
    sflag[k] = (r < 0 || r >= g.Xl) ? 1 : rowflag[r];
  }
  __syncthreads();

  int slot = 0;
  const int r_end = xe + LAG;
  for (int r = xb - H; r < r_end; r++, pr += g.pitch, pb += g.pitch)
  {
    const bool want = col_ok && r < xe + H;                                            // row r enters the ring
    const bool plane = col_plane || (want && sflag[r - (xb - H)]);
    double fr[9], fb[9];
    double rr, rb, ux, uy, ph;
    // ---- A: moments of node (r, y) of the post-stream state: from the planes, or pulled
    if (want)
    {
      if (plane)
      {
        const long long k = mom_off(mg, r, y);
        rr = mom[M_RR * mg.mplane + k];
        rb = mom[M_RB * mg.mplane + k];
        ux = mom[M_UX * mg.mplane + k];
        uy = mom[M_UY * mg.mplane + k];
        ph = mom[M_PH * mg.mplane + k];
      }
      else
      {
        tp_pull_at(pr, g, fr);
        tp_pull_at(pb, g, fb);
      }
    }
    // ---- B (pipelined): collision of row r - LAG
    if constexpr (PIPE)
    {
      if (r - LAG >= xb && collider) collide_row((slot + NR - LAG) % NR);
    }
    // ---- C: finish the moments, publish them
    if (want)
    {
      if (!plane) tp_moments<MODEL>(p, fr, fb, rr, rb, ux, uy, ph);
      S(0, slot, t) = ph;
      if constexpr (MODEL == TP_MRTCG)
      {
        const double cq = p.cr * rr + p.cb * rb;
        S(1, slot, t) = cq * ux;
        S(2, slot, t) = cq * uy;
      }
      S(C::F_RR, slot, t) = rr;
      S(C::F_RB, slot, t) = rb;
      S(C::F_UX, slot, t) = ux;
      S(C::F_UY, slot, t) = uy;
    }
    __syncthreads();
    // ---- B (plain): collision of row r - H, whose stencil rows are the last 2H+1 ring slots
    if constexpr (!PIPE)
    {
      if (r - LAG >= xb && collider) collide_row((slot + NR - LAG) % NR);
    }
    slot = slot + 1 == NR ? 0 : slot + 1;
  }
}

// ------------------------------------------------------------------------------------------------
// fused step with the population rows STAGED in shared memory by bulk asynchronous copies (lbm_async.cuh)
// ------------------------------------------------------------------------------------------------
// Same strips, bands, ring and plane rules as k_tp_fused, but nothing is pulled through registers and nothing is read
// twice: for every row r of the band (and its H warm-up rows on either side) one lane issues 18 bulk copies — population
// q of both lattices, source row r - c_x(q), the strip's column window widened by two columns on either side — into stage
// slot r mod NS, completed on that slot's mbarrier.  Iteration r waits for row r, forms its moments out of the slot (the
// +-1 column shift of the pull is an index offset), and collides row r - H out of ITS slot, which is still resident; the
// copies of rows r+1 .. r+NS-H-1 are in flight meanwhile, independent of what the fp64 work keeps in registers.
// rho_k, u of the H+1 rows between moments and collision stay in registers of the thread that formed them (same column).
//   DRAM: every population row segment once per band (+ 2H warm-up rows per band), results written once.
//   shared memory (MRTCG): NS x 18 x 132 doubles of stages + 3 x 6 x 128 of ring = 111 KB at NS = 5: two blocks per SM.
template <int MODEL, int NS>
struct TpStaged
{
  using F = TpFused<MODEL>;
  static constexpr int H = F::H, NR = F::NR;
  static constexpr int NF = MODEL == TP_MRTCG ? 3 : 1;       // ring fields: phase [, Q_x, Q_y]
  static constexpr int W = TPF_NT + 4;                        // staged columns per population row: even start <= ys - 1, end >= ys + 128
  static constexpr int ROW = 18 * W;                          // doubles per staged row
  static constexpr int USEFUL = F::USEFUL;
  static constexpr size_t RING_BYTES = sizeof(double) * NF * NR * TPF_NT;
  static constexpr size_t STAGE_BYTES = sizeof(double) * NS * ROW;
  static constexpr size_t SMEM = STAGE_BYTES + RING_BYTES + sizeof(uint64_t) * NS;
  static constexpr int TMEM_COLS = 128;                       // STASH: (H + 1) rows x 36 columns per thread, rounded up to a power of two
};

// STASH = false: a stage slot keeps its row until that row has been collided (H + 1 resident rows + the rows in flight:
//                NS >= H + 2; MRTCG at NS = 5: 111 KB per block, two blocks = 8 warps per SM, which is what bounds it —
//                ncu: DRAM traffic 293 B/node, the minimum, but 0.4 instructions per cycle and scheduler).
// STASH = true : the thread parks the 18 populations it has just read in TENSOR MEMORY (its own lane, 36 columns per
//                row, H + 1 rows) and takes them back H rows later for the collision; the stage slot is free as soon as the
//                moments are formed, so NS = 3 slots (57 KB) + ring: three or four blocks per SM.
template <int MODEL, int NS, int MINB, bool STASH>
__global__ void __launch_bounds__(TPF_NT, MINB)
k_tp_staged(const double* __restrict__ rsrc, const double* __restrict__ bsrc, double* __restrict__ rdst,
            double* __restrict__ bdst, const SlabGeom g, const MomGeom mg, const double* __restrict__ mom, const TpParams p,
            const unsigned char* __restrict__ rowflag, int rows_per_block, int band_lo, int band_jump)
{
  using C = TpStaged<MODEL, NS>;
  constexpr int H = C::H, NR = C::NR, NT = TPF_NT, W = C::W;
  constexpr int HOLD = STASH ? 0 : H;  // iterations a stage slot stays resident after its moments have been formed
  static_assert(NS >= HOLD + 2, "at least one row in flight");
  extern __shared__ double sm[];  // stages [NS][18][W] | ring [NF][NR][NT] | mbarriers [NS]
  double* stage = sm;
  double* ring = sm + NS * C::ROW;
  uint64_t* full = reinterpret_cast<uint64_t*>(ring + C::NF * NR * NT);

  const int t = threadIdx.x;
  const int ys = 1 + blockIdx.x * C::USEFUL - H;         // column of thread 0
  const int y = ys + t;
  const int xb = ((int)blockIdx.y < band_lo ? (int)blockIdx.y : (int)blockIdx.y + band_jump) * rows_per_block;  // (0, 0): every band; see tp_launch_fused
  const int xe = min(xb + rows_per_block, g.Xl);
  const int r0 = xb - H;                                 // first row of the march
  const int rs0 = max(r0, 0), rs1 = min(xe + H, g.Xl);   // rows whose populations are staged
  const bool col_ok = y >= -2 && y <= g.Y + 1;           // inside the padded planes
  const bool col_plane = y < 1 || y > g.Y - 2;           // edge columns (listed nodes) and the padding
  const bool collider = t >= H && t < NT - H && y >= 1 && y <= g.Y - 2;

  // staged column window [c0, c0 + W) clamped to the row; c0 even (16-byte aligned copies)
  const int c0 = (ys - 1) & ~1;                           // floor to even, also for negative ys - 1
  const int lo = max(c0, 0), hi = min(c0 + W, g.pitch);
  const unsigned seg_bytes = (unsigned)(hi - lo) * (unsigned)sizeof(double);
  const int my = t + (ys - c0);                          // this thread's column inside a staged segment (before the -c_y shift)

  __shared__ unsigned char sflag[128 + 2 * H + 2];
  __shared__ uint32_t tmem_slot;
  for (int k = t; k < xe - xb + 2 * H; k += NT)
  {
    const int r = r0 + k;
    sflag[k] = (r < 0 || r >= g.Xl) ? 1 : rowflag[r];
  }
  if (t == 0)
  {
    for (int s = 0; s < NS; s++) mbar_init(&full[s], 1);
    mbar_init_fence();
  }
  uint32_t tmem = 0;
  if constexpr (STASH) tmem = tmem_alloc<C::TMEM_COLS>(&tmem_slot);  // (contains the block barrier)
  else __syncthreads();

  // row rr of the march -> stage slot (rr - r0) % NS; every row of the march uses its slot's barrier once (rows without
  // populations — outside the slab — complete it with zero bytes), so the parity of a wait is ((rr - r0) / NS) & 1.
  // Lanes 0 .. 17 of warp 0 own one population row segment each: source pointer at row 0 and shared-memory offset once,
  // so that issuing a row costs that warp a dozen instructions (the other warps wait for it at the next barrier).
  const int lane_q = (t < 18 ? t : 0) % 9;
  const double* lane_src = (t < 9 ? rsrc : bsrc) + (long long)lane_q * g.plane + node_off(g, -CX(lane_q), lo);
  double* lane_dst = stage + (t < 18 ? t : 0) * W + (lo - c0);
  auto issue_row = [&](int rr, int slot) {
    if (t >= 32 || rr >= xe + H) return;
    const bool staged = rr >= rs0 && rr < rs1;
    if (t == 0) mbar_arrive_expect_tx(&full[slot], staged ? 18u * seg_bytes : 0u);
    __syncwarp();
    if (staged && t < 18) bulk_copy_g2s(lane_dst + (size_t)slot * C::ROW, lane_src + (long long)rr * g.pitch, seg_bytes, &full[slot]);
  };
  constexpr int AHEAD = NS - HOLD - (STASH ? 0 : 1);  // rows issued before the march starts = distance of the loop's refill rule
  for (int j = 0; j < AHEAD; j++) issue_row(r0 + j, j);
  __syncthreads();

  double mrr[H + 1], mrb[H + 1], mux[H + 1], muy[H + 1];  // rho_r, rho_b, u of rows r, r-1, .. r-H at this thread's column
#pragma unroll
  for (int k = 0; k <= H; k++) mrr[k] = mrb[k] = mux[k] = muy[k] = 0.0;

  // counters instead of k % NS, k / NS, k % (H + 1): slot and parity of row r, slot of the row to refill, tensor-memory slot
  int slot_ring = 0, sl = 0, sl_x = (NS - H % NS) % NS, sl_fill = AHEAD % NS, ts = 0;
  // rrow[j] = element offset of the ring row of row r - j: rotated once per iteration (2H register moves) instead of
  // one (slot mod NR) * NT per stencil row
  int rrow[2 * H + 1];
#pragma unroll
  for (int j = 0; j <= 2 * H; j++) rrow[j] = ((NR - j) % NR) * NT;
  unsigned par = 0;
  for (int r = r0; r < xe + H; r++)
  {
    const int k = r - r0;
    const double* st_r = stage + (size_t)sl * C::ROW;
    mbar_wait(&full[sl], par);
    // ---- A: moments of (r, y) -> ring, registers
#pragma unroll
    for (int j = H; j > 0; j--)
    {
      mrr[j] = mrr[j - 1];
      mrb[j] = mrb[j - 1];
      mux[j] = mux[j - 1];
      muy[j] = muy[j - 1];
    }
    double fr[9], fb[9];
    if constexpr (STASH)
    {
      // the previous rows' parks have landed (tcgen05.wait::st, a whole iteration after they were issued: nothing to wait
      // for in practice; measured alternatives: in front of the barrier the same, right before the collision's load -4 %).
      // A row is taken back H >= 1 iterations after its park, so every load has at least one such wait behind it.
      tmem_store_wait();
      // every thread takes its 18 populations out of the slot (rows outside the slab: stale shared memory, never used)
      // and parks them in its tensor-memory lane for the collision H rows later
#pragma unroll
      for (int q = 0; q < 9; q++)
      {
        fr[q] = st_r[q * W + my - CY(q)];
        fb[q] = st_r[(9 + q) * W + my - CY(q)];
      }
      tmem_store18(tmem + 36u * (unsigned)ts, fr, fb);
    }
    if (col_ok)
    {
      double rr_, rb_, ux_, uy_, ph_;
      if (col_plane || sflag[k])
      {
        const long long km = mom_off(mg, r, y);
        rr_ = mom[M_RR * mg.mplane + km];
        rb_ = mom[M_RB * mg.mplane + km];
        ux_ = mom[M_UX * mg.mplane + km];
        uy_ = mom[M_UY * mg.mplane + km];
        ph_ = mom[M_PH * mg.mplane + km];
      }
      else
      {
        if constexpr (!STASH)
        {
#pragma unroll
          for (int q = 0; q < 9; q++)
          {
            fr[q] = st_r[q * W + my - CY(q)];
            fb[q] = st_r[(9 + q) * W + my - CY(q)];
          }
        }
        tp_moments<MODEL>(p, fr, fb, rr_, rb_, ux_, uy_, ph_);
      }
      ring[rrow[0] + t] = ph_;
      if constexpr (MODEL == TP_MRTCG)
      {
        const double cq = p.cr * rr_ + p.cb * rb_;
        ring[NR * NT + rrow[0] + t] = cq * ux_;
        ring[2 * NR * NT + rrow[0] + t] = cq * uy_;
      }
      mrr[0] = rr_;
      mrb[0] = rb_;
      mux[0] = ux_;
      muy[0] = uy_;
    }
    // the collided row's populations are on their way back from tensor memory under the barrier
    [[maybe_unused]] uint32_t tr[36];
    if constexpr (STASH)
    {
      ts = ts == H ? 0 : ts + 1;  // now the slot of row r - H: (k - H) mod (H + 1) = (k + 1) mod (H + 1)
      tmem_load18_issue(tmem + 36u * (unsigned)ts, tr);
    }
    __syncthreads();
    // a slot is free now: the one this iteration read (STASH) / the one the previous iteration's collision read last
    issue_row(r + AHEAD, sl_fill);
    // ---- B: collision of row x = r - H out of tensor memory / its stage slot, and the ring rows x-H .. x+H
    const int x = r - H;
    if constexpr (STASH)
    {
      tmem_load_wait();
      tmem_unpack18(tr, fr, fb);
    }
    if (x >= xb && collider)
    {
      if constexpr (!STASH)
      {
        const double* st_x = stage + (size_t)sl_x * C::ROW;
#pragma unroll
        for (int q = 0; q < 9; q++)
        {
          fr[q] = st_x[q * W + my - CY(q)];
          fb[q] = st_x[(9 + q) * W + my - CY(q)];
        }
      }
      TpStencil st;
      tp_ring_stencil_at<MODEL>(ring, [&](int a) { return rrow[H - a]; }, t, st);  // row x + a = r - (H - a)
      tp_collide<MODEL>(p, fr, fb, mrr[H], mrb[H], mux[H], muy[H], ring[rrow[H] + t], st);
      double* wr = rdst + node_off(g, x, y);
      double* wb = bdst + node_off(g, x, y);
#pragma unroll
      for (int q = 0; q < 9; q++)
      {
        wr[(long long)q * g.plane] = fr[q];
        wb[(long long)q * g.plane] = fb[q];
      }
    }
    slot_ring = slot_ring + 1 == NR ? 0 : slot_ring + 1;
#pragma unroll
    for (int j = 2 * H; j > 0; j--) rrow[j] = rrow[j - 1];
    rrow[0] = slot_ring * NT;
    sl_x = sl_x + 1 == NS ? 0 : sl_x + 1;
    sl_fill = sl_fill + 1 == NS ? 0 : sl_fill + 1;
    if (++sl == NS)
    {
      sl = 0;
      par ^= 1u;
    }
  }
  if constexpr (STASH) tmem_free<C::TMEM_COLS>(tmem);
}

// moments of a short list of nodes (plain pull) into the planes: the region around listed nodes,
// the global edge rows and the rows next to a slab cut
template <int MODEL>
__global__ void __launch_bounds__(128)
k_tp_moments_nodes(const double* __restrict__ rsrc, const double* __restrict__ bsrc, const SlabGeom g, const MomGeom mg,
                   double* __restrict__ mom, const TpParams p, const int* __restrict__ nodes, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int x = nodes[i] / g.Y, y = nodes[i] % g.Y;
  double fr[9], fb[9];
  tp_load_interior<MODE_PULL>(rsrc, g, x, y, fr);
  tp_load_interior<MODE_PULL>(bsrc, g, x, y, fb);
  double rr, rb, ux, uy, ph;
  tp_moments<MODEL>(p, fr, fb, rr, rb, ux, uy, ph);
  const long long k = mom_off(mg, x, y);
  mom[M_RR * mg.mplane + k] = rr;
  mom[M_RB * mg.mplane + k] = rb;
  mom[M_UX * mg.mplane + k] = ux;
  mom[M_UY * mg.mplane + k] = uy;
  mom[M_PH * mg.mplane + k] = ph;
}

template <int MODEL, int MODE>
__global__ void __launch_bounds__(128)
k_tp_collide_listed(const double* __restrict__ rsrc, const double* __restrict__ bsrc, double* __restrict__ rdst,
                    double* __restrict__ bdst, const SlabGeom g, const MomGeom mg, const double* __restrict__ mom,
                    const TpParams p, const BoundaryTable t)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= t.n) return;
  const int x = t.x[i], y = t.y[i];
  TpStencil st;
  tp_stencil_global<MODEL>(p, mom, mg, x, y, st);
  const long long km = mom_off(mg, x, y);
  const double rr = mom[M_RR * mg.mplane + km], rb = mom[M_RB * mg.mplane + km];
  const double ux = mom[M_UX * mg.mplane + km], uy = mom[M_UY * mg.mplane + km], ph = mom[M_PH * mg.mplane + km];
  double fr[9], fb[9];
  tp_load_listed<MODE>(rsrc, g, t, 0, i, x, y, fr);
  tp_load_listed<MODE>(bsrc, g, t, 1, i, x, y, fb);
  tp_collide<MODEL>(p, fr, fb, rr, rb, ux, uy, ph, st);
  const long long o = node_off(g, x, y);
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    rdst[q * g.plane + o] = fr[q];
    bdst[q * g.plane + o] = fb[q];
  }
}

// ------------------------------------------------------------------------------------------------
// moments of the new post-stream state (and, with out_* set, its export in AoS)
// ------------------------------------------------------------------------------------------------
template <int MODEL, int MODE>
__global__ void __launch_bounds__(256)
k_tp_moments_interior(const double* __restrict__ rsrc, const double* __restrict__ bsrc, const SlabGeom g, const MomGeom mg,
                      double* __restrict__ mom, const TpParams p, double* __restrict__ out_r, double* __restrict__ out_b)
{
  const int y = 1 + blockIdx.x * blockDim.x + threadIdx.x;
  const int x = blockIdx.y;
  if (y > g.Y - 2) return;
  double fr[9], fb[9];
  tp_load_interior<MODE>(rsrc, g, x, y, fr);
  tp_load_interior<MODE>(bsrc, g, x, y, fb);
  if (out_r)
  {
    double* a = out_r + ((long long)x * g.Y + y) * 9;
    double* b = out_b + ((long long)x * g.Y + y) * 9;
#pragma unroll
    for (int q = 0; q < 9; q++)
    {
      a[q] = fr[q];
      b[q] = fb[q];
    }
    return;
  }
  double rr, rb, ux, uy, ph;
  tp_moments<MODEL>(p, fr, fb, rr, rb, ux, uy, ph);
  const long long k = mom_off(mg, x, y);
  mom[M_RR * mg.mplane + k] = rr;
  mom[M_RB * mg.mplane + k] = rb;
  mom[M_UX * mg.mplane + k] = ux;
  mom[M_UY * mg.mplane + k] = uy;
  mom[M_PH * mg.mplane + k] = ph;
}

template <int MODEL, int MODE>
__global__ void __launch_bounds__(128)
k_tp_moments_listed(const double* __restrict__ rsrc, const double* __restrict__ bsrc, const SlabGeom g, const MomGeom mg,
                    double* __restrict__ mom, const TpParams p, const BoundaryTable t, double* __restrict__ out_r,
                    double* __restrict__ out_b, int sel)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= t.n) return;
  const int x = t.x[i], y = t.y[i];
  // sel 1: only the rows next to a slab cut / the global edge (0, 1, Xl-2, Xl-1); sel 2: every other row (tp_pre_part)
  if (sel != 0 && ((x < 2 || x >= g.Xl - 2) != (sel == 1))) return;
  double fr[9], fb[9];
  tp_load_listed<MODE>(rsrc, g, t, 0, i, x, y, fr);
  tp_load_listed<MODE>(bsrc, g, t, 1, i, x, y, fb);
  if (out_r)
  {
    double* a = out_r + ((long long)x * g.Y + y) * 9;
    double* b = out_b + ((long long)x * g.Y + y) * 9;
#pragma unroll
    for (int q = 0; q < 9; q++)
    {
      a[q] = fr[q];
      b[q] = fb[q];
    }
    return;
  }
  double rr, rb, ux, uy, ph;
  tp_moments<MODEL>(p, fr, fb, rr, rb, ux, uy, ph);
  const long long k = mom_off(mg, x, y);
  mom[M_RR * mg.mplane + k] = rr;
  mom[M_RB * mg.mplane + k] = rb;
  mom[M_UX * mg.mplane + k] = ux;
  mom[M_UY * mg.mplane + k] = uy;
  mom[M_PH * mg.mplane + k] = ph;
}

// the region pass in ONE launch: blocks 0 .. ceil(n / 128) - 1 take the node list (plain pull), the others the listed nodes
// (pull through their rules).  The two sets are disjoint (tp_build_region).
template <int MODEL>
__global__ void __launch_bounds__(128)
k_tp_moments_region(const double* __restrict__ rsrc, const double* __restrict__ bsrc, const SlabGeom g, const MomGeom mg,
                    double* __restrict__ mom, const TpParams p, const int* __restrict__ nodes, int n, const BoundaryTable t)
{
  const int node_blocks = (n + 127) / 128;
  int x, y;
  double fr[9], fb[9];
  if ((int)blockIdx.x < node_blocks)
  {
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= n) return;
    x = nodes[i] / g.Y;
    y = nodes[i] % g.Y;
    tp_load_interior<MODE_PULL>(rsrc, g, x, y, fr);
    tp_load_interior<MODE_PULL>(bsrc, g, x, y, fb);
  }
  else
  {
    const int i = ((int)blockIdx.x - node_blocks) * 128 + threadIdx.x;
    if (i >= t.n) return;
    x = t.x[i];
    y = t.y[i];
    tp_load_listed<MODE_PULL>(rsrc, g, t, 0, i, x, y, fr);
    tp_load_listed<MODE_PULL>(bsrc, g, t, 1, i, x, y, fb);
  }
  double rr, rb, ux, uy, ph;
  tp_moments<MODEL>(p, fr, fb, rr, rb, ux, uy, ph);
  const long long k = mom_off(mg, x, y);
  mom[M_RR * mg.mplane + k] = rr;
  mom[M_RB * mg.mplane + k] = rb;
  mom[M_UX * mg.mplane + k] = ux;
  mom[M_UY * mg.mplane + k] = uy;
  mom[M_PH * mg.mplane + k] = ph;
}

// replicate padding of the moment planes: columns first (all owned rows), then rows (whole padded width)
__global__ void k_tp_pad_cols(double* __restrict__ mom, const SlabGeom g, const MomGeom mg, int nplanes, int x_begin, int x_end)
{
  const int x = x_begin + blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= g.Xl || x >= x_end) return;
  for (int f = 0; f < nplanes; f++)
  {
    double* pl = mom + f * mg.mplane;
    const double lo = pl[mom_off(mg, x, 0)], hi = pl[mom_off(mg, x, g.Y - 1)];
    pl[mom_off(mg, x, -1)] = lo;
    pl[mom_off(mg, x, -2)] = lo;
    pl[mom_off(mg, x, g.Y)] = hi;
    pl[mom_off(mg, x, g.Y + 1)] = hi;
  }
}

// lo_global / hi_global: this slab holds the global first / last row, where the padding replicates;
// elsewhere the two ghost rows come from the neighbouring slab (lbm_comm.cu)
__global__ void k_tp_pad_rows(double* __restrict__ mom, const SlabGeom g, const MomGeom mg, int lo_global, int hi_global, int nplanes)
{
  const int j = blockIdx.x * blockDim.x + threadIdx.x;  // padded column index 0 .. Y+3
  if (j >= g.Y + 4) return;
  const int y = j - 2;
  for (int f = 0; f < nplanes; f++)
  {
    double* pl = mom + f * mg.mplane;
    if (lo_global)
    {
      const double v = pl[mom_off(mg, 0, y)];
      pl[mom_off(mg, -1, y)] = v;
      pl[mom_off(mg, -2, y)] = v;
    }
    if (hi_global)
    {
      const double v = pl[mom_off(mg, g.Xl - 1, y)];
      pl[mom_off(mg, g.Xl, y)] = v;
      pl[mom_off(mg, g.Xl + 1, y)] = v;
    }
  }
}

// both paddings in one launch: threads 0 .. Xl-1 pad the columns of their row, threads Xl .. Xl+Y+3 the rows of their padded
// column (reading the edge rows at the column clamped into the grid: the value k_tp_pad_cols would have put there)
__global__ void k_tp_pad(double* __restrict__ mom, const SlabGeom g, const MomGeom mg, int lo_global, int hi_global, int nplanes)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < g.Xl)
  {
    for (int f = 0; f < nplanes; f++)
    {
      double* pl = mom + f * mg.mplane;
      const double lo = pl[mom_off(mg, i, 0)], hi = pl[mom_off(mg, i, g.Y - 1)];
      pl[mom_off(mg, i, -1)] = lo;
      pl[mom_off(mg, i, -2)] = lo;
      pl[mom_off(mg, i, g.Y)] = hi;
      pl[mom_off(mg, i, g.Y + 1)] = hi;
    }
    return;
  }
  const int j = i - g.Xl;
  if (j >= g.Y + 4) return;
  const int y = j - 2, yc = min(max(y, 0), g.Y - 1);
  for (int f = 0; f < nplanes; f++)
  {
    double* pl = mom + f * mg.mplane;
    if (lo_global)
    {
      const double v = pl[mom_off(mg, 0, yc)];
      pl[mom_off(mg, -1, y)] = v;
      pl[mom_off(mg, -2, y)] = v;
    }
    if (hi_global)
    {
      const double v = pl[mom_off(mg, g.Xl - 1, yc)];
      pl[mom_off(mg, g.Xl, y)] = v;
      pl[mom_off(mg, g.Xl + 1, y)] = v;
    }
  }
}

// initial state: adv_f = eq(rho_k, u) (mrtcg_rayleigh_taylor.cpp:409-410 ; rk_static_droplet_test.cpp:509-515)
template <int MODEL>
__global__ void k_tp_init(double* __restrict__ rbuf, double* __restrict__ bbuf, const SlabGeom g, const MomGeom mg,
                          double* __restrict__ mom, const TpParams p, const double* __restrict__ rho_r,
                          const double* __restrict__ rho_b, const double* __restrict__ u)
{
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (long long)g.Xl * g.Y) return;
  const int x = (int)(n / g.Y), y = (int)(n % g.Y);
  double rr = rho_r[n], rb = rho_b[n];
  const double ux = u[2 * n], uy = u[2 * n + 1];
  const double uu = ux * ux + uy * uy;
  double fr[9], fb[9];
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    fr[q] = tp_feq<MODEL>(q, rr, p.r_phi, p.r_eta, ux, uy, uu);
    fb[q] = tp_feq<MODEL>(q, rb, p.b_phi, p.b_eta, ux, uy, uu);
  }
  const long long o = node_off(g, x, y);
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    rbuf[q * g.plane + o] = fr[q];
    bbuf[q * g.plane + o] = fb[q];
  }
  if constexpr (MODEL == TP_RK)
  {
    // the RK driver re-reads the densities from the populations (rk_static_droplet_test.cpp:513-514)
    double jx, jy;
    moments(fr, rr, jx, jy);
    moments(fb, rb, jx, jy);
  }
  const long long k = mom_off(mg, x, y);
  mom[M_RR * mg.mplane + k] = rr;
  mom[M_RB * mg.mplane + k] = rb;
  mom[M_UX * mg.mplane + k] = ux;
  mom[M_UY * mg.mplane + k] = uy;
  mom[M_PH * mg.mplane + k] = phase_of(p, rr, rb);
}

// moments from imported populations (lbm_set_f on a two-phase domain)
template <int MODEL>
__global__ void k_tp_moments_local(const double* __restrict__ rbuf, const double* __restrict__ bbuf, const SlabGeom g,
                                   const MomGeom mg, double* __restrict__ mom, const TpParams p)
{
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (long long)g.Xl * g.Y) return;
  const int x = (int)(n / g.Y), y = (int)(n % g.Y);
  double fr[9], fb[9];
  tp_load_interior<MODE_LOCAL>(rbuf, g, x, y, fr);
  tp_load_interior<MODE_LOCAL>(bbuf, g, x, y, fb);
  double rr, rb, ux, uy, ph;
  tp_moments<MODEL>(p, fr, fb, rr, rb, ux, uy, ph);
  const long long k = mom_off(mg, x, y);
  mom[M_RR * mg.mplane + k] = rr;
  mom[M_RB * mg.mplane + k] = rb;
  mom[M_UX * mg.mplane + k] = ux;
  mom[M_UY * mg.mplane + k] = uy;
  mom[M_PH * mg.mplane + k] = ph;
}

__global__ void k_tp_read_moments(const double* __restrict__ mom, const SlabGeom g, const MomGeom mg, double* __restrict__ rho,
                                  double* __restrict__ u, double* __restrict__ ph, double* __restrict__ rr_out,
                                  double* __restrict__ rb_out)
{
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (long long)g.Xl * g.Y) return;
  const int x = (int)(n / g.Y), y = (int)(n % g.Y);
  const long long k = mom_off(mg, x, y);
  const double rr = mom[M_RR * mg.mplane + k], rb = mom[M_RB * mg.mplane + k];
  if (rho) rho[n] = rr + rb;
  if (u)
  {
    u[2 * n] = mom[M_UX * mg.mplane + k];
    u[2 * n + 1] = mom[M_UY * mg.mplane + k];
  }
  if (ph) ph[n] = mom[M_PH * mg.mplane + k];
  if (rr_out) rr_out[n] = rr;
  if (rb_out) rb_out[n] = rb;
}

__global__ void k_tp_write_u(double* __restrict__ mom, const SlabGeom g, const MomGeom mg, const double* __restrict__ u)
{
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (long long)g.Xl * g.Y) return;
  const int x = (int)(n / g.Y), y = (int)(n % g.Y);
  const long long k = mom_off(mg, x, y);
  mom[M_UX * mg.mplane + k] = u[2 * n];
  mom[M_UY * mg.mplane + k] = u[2 * n + 1];
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// f(std::integral_constant<int, MODEL>()) for the domain's model: TP_RK, or TP_MRTCG for the others (TP_CSF's export and
// import passes are MRTCG's: the export only pulls, and an import carries no interfacial tension)
template <class F>
static int with_model(const TwoPhaseState* tp, F&& f)
{
  if (tp->model == TP_RK) return f(std::integral_constant<int, TP_RK>());
  return f(std::integral_constant<int, TP_MRTCG>());
}

// The row-marching kernels a switch can select.  All instantiations of one family have the same parameters, so one table
// gives tp_create the attributes to set and the kernel to resolve, and the step its launch.
struct TpKernel
{
  int model;
  bool staged, stash;  // k_tp_staged (with the tensor-memory stash), or k_tp_fused
  int ns;              // k_tp_staged: stage slots
  bool pipe;           // k_tp_fused: the software-pipelined variant
  decltype(&k_tp_fused<TP_MRTCG, true>) kernel;
  size_t smem;
  int warmup_rows;     // band height: pick_band_rows with this many warm-up rows per band
};
template <int MODEL, bool PIPE>
static TpKernel tp_fused_kernel() { return {MODEL, false, false, 0, PIPE, k_tp_fused<MODEL, PIPE>, TpFused<MODEL>::SMEM, 2 * TpFused<MODEL>::H}; }
template <int MODEL, int NS, int MINB, bool STASH>
static TpKernel tp_staged_kernel() { return {MODEL, true, STASH, NS, false, k_tp_staged<MODEL, NS, MINB, STASH>, TpStaged<MODEL, NS>::SMEM, 2 * TpFused<MODEL>::H}; }
static const TpKernel tp_kernels[] = {
    tp_fused_kernel<TP_MRTCG, false>(), tp_fused_kernel<TP_MRTCG, true>(), tp_fused_kernel<TP_RK, false>(), tp_fused_kernel<TP_RK, true>(),
    tp_staged_kernel<TP_MRTCG, 4, 2, false>(), tp_staged_kernel<TP_MRTCG, 5, 2, false>(), tp_staged_kernel<TP_MRTCG, 6, 2, false>(),
    tp_staged_kernel<TP_RK, 3, 3, false>(), tp_staged_kernel<TP_RK, 4, 2, false>(), tp_staged_kernel<TP_RK, 5, 2, false>(), tp_staged_kernel<TP_RK, 6, 2, false>(),
    tp_staged_kernel<TP_MRTCG, 2, 4, true>(), tp_staged_kernel<TP_MRTCG, 3, 3, true>(), tp_staged_kernel<TP_MRTCG, 4, 2, true>(),
    tp_staged_kernel<TP_RK, 2, 4, true>(), tp_staged_kernel<TP_RK, 3, 3, true>(), tp_staged_kernel<TP_RK, 4, 2, true>()};

// the switches' kernel (LBM_TP_PIPE counts only when LBM_TP_STAGED=0)
static const TpKernel* tp_pick_kernel(int model, bool staged, bool stash, int stages, bool pipe)
{
  int ns = 0;
  if (staged)
  {
    // stage slots.  With the stash: the rows in flight only (2 .. 4).  Without it: H + 1 resident rows + the rows in flight
    // (H + 2 .. 6).  stages <= 0: the model's default
    const int H = model == TP_MRTCG ? TpFused<TP_MRTCG>::H : TpFused<TP_RK>::H;
    ns = stash ? std::clamp(stages > 0 ? stages : (model == TP_MRTCG ? 3 : 4), 2, 4) : std::clamp(stages > 0 ? stages : 5, H + 2, 6);
    pipe = false;
  }
  else stash = false;
  for (const TpKernel& k : tp_kernels)
    if (k.model == model && k.staged == staged && k.stash == stash && k.ns == ns && k.pipe == pipe) return &k;
  return nullptr;
}

// band height of a row-marching kernel, once per rule set: LBM_TP_RPB, else from the occupancy of the kernel that runs
// (warmup_rows = 0: 64 rows)
template <class K>
static int band_rows(lbm_domain* d, int strips, const K& k)
{
  TwoPhaseState* tp = d->tp;
  if (tp->rows_per_block <= 0)
    tp->rows_per_block = tp->rpb_override > 0 ? std::min(128, tp->rpb_override)  // the kernels stage <= 128 + 2H row flags
                         : k.warmup_rows > 0 ? pick_band_rows(d->g.Xl, strips, resident_blocks_of(d, k.kernel, k.smem), k.warmup_rows)
                                             : 64;
  return tp->rows_per_block;
}

double* tp_moment_planes(lbm_domain* d, int* pm, long long* mplane)
{
  *pm = d->tp->mg.pm;
  *mplane = d->tp->mg.mplane;
  return d->tp->mom;
}

int tp_destroy(lbm_domain* d)
{
  if (!d->tp) return LBM_OK;
  cudaFree(d->tp->mom);
  cudaFree(d->tp->aux);
  cudaFree(d->tp->aux_next);
  cudaFree(d->tp->d_csf_flags);
  cudaFree(d->tp->d_csf_list4);
  cudaFree(d->tp->d_csf_list2);
  cudaFree(d->tp->d_rowflag);
  cudaFree(d->tp->d_region);
  delete d->tp;
  d->tp = nullptr;
  return LBM_OK;
}

static BoundaryTable table_of(lbm_domain* d)
{
  BoundaryTable bt;
  bt.n = d->nb;
  bt.x = d->d_bx;
  bt.y = d->d_by;
  bt.ent = d->d_ent;
  bt.mom_cur = nullptr;
  bt.mom_prev = nullptr;
  return bt;
}

int tp_pad(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  const int lo = d->cfg.x0 == 0, hi = d->cfg.x1 == d->cfg.X;
  k_tp_pad<<<cdiv(d->g.Xl + d->g.Y + 4, 128), 128, 0, d->stream>>>(tp->mom, d->g, tp->mg, lo, hi, M_COUNT);
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

template <int MODEL, int MODE>
static int tp_launch_collide(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  const int s = d->cur, t = d->cur ^ 1;
  const int Yi = d->g.Y - 2;
  if (Yi > 0)
  {
    ProfScope ps(d, LBM_PROF_INTERIOR);
    dim3 grid(cdiv(Yi, TILE_Y), cdiv(d->g.Xl, TILE_X)), block(TILE_Y, TILE_X);
    k_tp_collide_interior<MODEL, MODE><<<grid, block, 0, d->stream>>>(d->buf[0][s], d->buf[1][s], d->buf[0][t], d->buf[1][t], d->g,
                                                                     tp->mg, tp->mom, tp->p, 0, d->g.Xl);
    d->launches++;
  }
  if (d->nb > 0)
  {
    ProfScope ps(d, LBM_PROF_BOUNDARY);
    k_tp_collide_listed<MODEL, MODE><<<cdiv(d->nb, 128), 128, 0, d->stream>>>(d->buf[0][s], d->buf[1][s], d->buf[0][t], d->buf[1][t],
                                                                             d->g, tp->mg, tp->mom, tp->p, table_of(d));
    d->launches++;
  }
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

// moments (out == nullptr) or AoS export (out set) of the post-stream state pulled from buffer `which`
template <int MODEL>
static int tp_launch_moments(lbm_domain* d, int which, double* out_r, double* out_b)
{
  TwoPhaseState* tp = d->tp;
  const int Yi = d->g.Y - 2;
  ProfScope ps(d, LBM_PROF_MOMENTS);
  if (Yi > 0)
  {
    dim3 grid(cdiv(Yi, 256), d->g.Xl);
    k_tp_moments_interior<MODEL, MODE_PULL><<<grid, 256, 0, d->stream>>>(d->buf[0][which], d->buf[1][which], d->g, tp->mg, tp->mom,
                                                                        tp->p, out_r, out_b);
    d->launches++;
  }
  if (d->nb > 0)
  {
    k_tp_moments_listed<MODEL, MODE_PULL><<<cdiv(d->nb, 128), 128, 0, d->stream>>>(d->buf[0][which], d->buf[1][which], d->g, tp->mg,
                                                                                  tp->mom, tp->p, table_of(d), out_r, out_b, 0);
    d->launches++;
  }
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

// rows whose moments stay in the planes, and the node list the region kernel recomputes every step
static int tp_build_region(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  if (!tp->region_dirty) return LBM_OK;
  const int Xl = d->g.Xl, Y = d->g.Y;
  std::vector<unsigned char> flag(Xl, 0);
  auto mark = [&](int x) { if (x >= 0 && x < Xl) flag[x] = 1; };
  // global edge rows feed the replicate padding, the rows next to a cut travel to the neighbour
  for (int x : {0, 1, Xl - 2, Xl - 1}) mark(x);
  // listed nodes read their 5x5 neighbourhood from the planes
  for (int x = 0; x < Xl && x < (int)d->row_has_listed.size(); x++)
    if (d->row_has_listed[x])
      for (int k = -2; k <= 2; k++) mark(x + k);
  // (listed nodes are left out: the listed half of k_tp_moments_region forms their moments through their rules, and the two
  // halves of that launch must not write the same cell)
  std::vector<int> nodes;
  auto add = [&](int id) { if (!std::binary_search(d->listed_ids.begin(), d->listed_ids.end(), id)) nodes.push_back(id); };
  for (int x = 0; x < Xl; x++)
  {
    if (flag[x])
    {
      for (int y = 1; y <= Y - 2; y++) add(x * Y + y);
      continue;
    }
    int last = 0;
    for (int y : {1, 2, Y - 3, Y - 2})
      if (y >= 1 && y <= Y - 2 && y > last)
      {
        add(x * Y + y);
        last = y;
      }
  }
  cudaFree(tp->d_rowflag);
  cudaFree(tp->d_region);
  tp->d_rowflag = nullptr;
  tp->d_region = nullptr;
  LBM_CUDA(cudaMalloc(&tp->d_rowflag, Xl));
  LBM_CUDA(cudaMemcpy(tp->d_rowflag, flag.data(), Xl, cudaMemcpyHostToDevice));
  tp->n_region = (int)nodes.size();
  tp->n_region_lo = tp->n_region_hi = 0;
  for (int id : nodes)
  {
    if (id / Y < 2) tp->n_region_lo++;
    else if (id / Y >= Xl - 2) tp->n_region_hi++;
  }
  if (tp->n_region > 0)
  {
    LBM_CUDA(cudaMalloc(&tp->d_region, sizeof(int) * nodes.size()));
    LBM_CUDA(cudaMemcpy(tp->d_region, nodes.data(), sizeof(int) * nodes.size(), cudaMemcpyHostToDevice));
  }
  tp->rows_per_block = 0;  // chosen at the next launch, from the occupancy of the kernel that runs (pick_band_rows)
  tp->region_dirty = false;
  return LBM_OK;
}

// which bands a launch of the fused kernel covers.  TP_BANDS_EDGE = band 0 and the last band (the last two when the last one
// has fewer than four rows): the rows whose results travel to the neighbouring ranks and whose stencils read the planes'
// halo rows; TP_BANDS_INTERIOR = the others; TP_BANDS_NONE only fixes the band height (tp->rows_per_block)
enum { TP_BANDS_ALL = 0, TP_BANDS_EDGE = 1, TP_BANDS_INTERIOR = 2, TP_BANDS_NONE = 3 };

static int tp_edge_bands_hi(const lbm_domain* d)
{
  const int rpb = d->tp->rows_per_block, nb = cdiv(d->g.Xl, rpb);
  return d->g.Xl - (nb - 1) * rpb < 4 ? 2 : 1;
}

template <int MODEL>
static int tp_launch_fused(lbm_domain* d, int part = TP_BANDS_ALL)
{
  TwoPhaseState* tp = d->tp;
  using C = TpFused<MODEL>;
  const int s = d->cur, t = d->cur ^ 1;
  const int Yi = d->g.Y - 2;
  if (Yi > 0)
  {
    const int strips = cdiv(Yi, C::USEFUL), rpb = band_rows(d, strips, *tp->kernel);
    if (part != TP_BANDS_NONE)
    {
      ProfScope ps(d, LBM_PROF_INTERIOR);
      // grid row j works on band j < band_lo ? j : j + band_jump
      const int nb = cdiv(d->g.Xl, rpb), k_hi = tp_edge_bands_hi(d);
      int ny = nb, band_lo = 0, band_jump = 0;
      if (part == TP_BANDS_EDGE) { ny = 1 + k_hi; band_lo = 1; band_jump = nb - k_hi - 1; }
      if (part == TP_BANDS_INTERIOR) { ny = nb - 1 - k_hi; band_jump = 1; }
      dim3 grid(strips, ny);
      auto k = tp->kernel->kernel;
      k<<<grid, TPF_NT, tp->kernel->smem, d->stream>>>(d->buf[0][s], d->buf[1][s], d->buf[0][t], d->buf[1][t], d->g, tp->mg, tp->mom, tp->p,
                                                      tp->d_rowflag, rpb, band_lo, band_jump);
      d->launches++;
    }
  }
  // listed nodes after the bands that hold them (a band writes every node of its rows' interior columns; with the bands split,
  // tp_ring_overlap_ok has checked that only the edge bands hold any)
  if (d->nb > 0 && part <= TP_BANDS_EDGE)
  {
    ProfScope ps(d, LBM_PROF_BOUNDARY);
    k_tp_collide_listed<MODEL, MODE_PULL><<<cdiv(d->nb, 128), 128, 0, d->stream>>>(d->buf[0][s], d->buf[1][s], d->buf[0][t],
                                                                                  d->buf[1][t], d->g, tp->mg, tp->mom, tp->p, table_of(d));
    d->launches++;
  }
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

// ---- the phases of one two-phase step.  lbm_step runs them back to back on one slab (NCCL halos inside);
//      lbm_step_group interleaves them across linked slabs.
// pre: the thin region of the moment planes that stays authoritative (listed nodes, their neighbourhood, edge and
//      cut rows) and its replicate padding, from the stored post-collision state
static int tp_phase_pre(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  LBM_TRY(tp_build_region(d));
  if (d->post_stream) return LBM_OK;  // first step after an import: the planes are full and hold the caller's u
  ProfScope ps(d, LBM_PROF_MOMENTS);
  const int s = d->cur;
  if (tp->n_region > 0 || d->nb > 0)
  {
    const int blocks = cdiv(tp->n_region, 128) + cdiv(d->nb, 128);
    with_model(tp, [&](auto M) {
      k_tp_moments_region<M><<<blocks, 128, 0, d->stream>>>(d->buf[0][s], d->buf[1][s], d->g, tp->mg, tp->mom, tp->p, tp->d_region, tp->n_region, table_of(d));
      return LBM_OK;
    });
    d->launches++;
  }
  LBM_TRY(tp_pad(d));
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

// main: collision of every node (fused kernel + listed nodes; two-pass MODE_LOCAL for a post-stream state)
static int tp_phase_main(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  LBM_TRY(with_model(tp, [&](auto M) { return d->post_stream ? tp_launch_collide<M, MODE_LOCAL>(d) : tp_launch_fused<M>(d); }));
  d->cur ^= 1;
  d->post_stream = false;
  tp->planes_full = false;
  return LBM_OK;
}

// ---- the ranks of a ring: both halo exchanges of a step behind the interior bands --------------------------------------
// tp_step on a ring is a chain: region moments -> moment-plane halo (NCCL) -> all bands -> ghost rows (NCCL), 0.3 - 0.4 ms of
// exposed exchange per step at 8192 x 16384 per GPU.  What crosses a cut is produced and consumed by the EDGE bands alone:
//   ghost rows of the new populations   <- rows 0, Xl-1 of this step             (edge bands + listed nodes)
//   moments of rows 0, 1, Xl-2, Xl-1    <- pull from rows -1 .. 2, Xl-3 .. Xl     (edge bands + those ghost rows)
//   moment-plane rows -2, -1, Xl, Xl+1  -> read by the stencils of rows 0, 1, Xl-2, Xl-1 of the NEXT step's edge bands
// so within one lbm_step(n) call the steps are run as
//   main stream:  region moments of rows 2 .. Xl-3 | wait side | edge bands, listed nodes | record | interior bands
//   side stream:  wait record | ghost rows | region moments of the four cut rows of the new state | moment-plane halo | record
// and the side chain of step i runs under the interior bands of step i; only the first step's cut rows are exchanged in line.
// Same kernels, same values: bit-identical to tp_step on the emulated rings and over NCCL on two B200s (tests/mp_nccl_check.py,
// bench.py's ring_parity force this path on).
// OFF by default (LBM_TP_OVERLAP=1 turns it on): measured on two B200s at 8192 x 16384 per GPU it is 0.4 - 1 % SLOWER than the
// in-line chain (7.55 ms in line; 7.63 overlapped; 7.58 with the side chain at the main stream's priority; 7.55 with
// NCCL_MAX_CTAS=1 - profiles/r02_ab_same_box.md).  The exchanges do leave the critical path (0.23 -> 0.10 ms outside the kernel)
// but NCCL's send/receive kernels are blocks of 512+ threads that need a nearly empty SM: beside a launch whose 128-thread
// blocks live for 0.1 ms and fill every SM they wait 0.5 - 1 ms for room and cost the interior bands 0.15 - 0.25 ms of
// throughput while they do.  What would make this pay is a transport without resident blocks (copy-engine peer copies
// between the ranks' buffers, which needs the ranks' allocations opened to each other) - the band split, the cut / rest
// split of the region pass and the event chain below are what such a transport plugs into.
enum { TP_PRE_ALL = 0, TP_PRE_CUT = 1, TP_PRE_REST = 2 };

// the authoritative thin region of the moment planes (tp_phase_pre) for the cut rows 0, 1, Xl-2, Xl-1 or for all the others
template <int MODEL>
static int tp_pre_part(lbm_domain* d, int part, cudaStream_t st)
{
  TwoPhaseState* tp = d->tp;
  ProfScope ps(d, LBM_PROF_MOMENTS, st);
  const int s = d->cur, Xl = d->g.Xl;
  auto nodes = [&](const int* list, int n) {
    if (n <= 0) return;
    k_tp_moments_nodes<MODEL><<<cdiv(n, 128), 128, 0, st>>>(d->buf[0][s], d->buf[1][s], d->g, tp->mg, tp->mom, tp->p, list, n);
    d->launches++;
  };
  if (part == TP_PRE_CUT)
  {
    nodes(tp->d_region, tp->n_region_lo);
    nodes(tp->d_region + (tp->n_region - tp->n_region_hi), tp->n_region_hi);
  }
  else
    nodes(tp->d_region + tp->n_region_lo, tp->n_region - tp->n_region_lo - tp->n_region_hi);
  if (d->nb > 0)
  {
    k_tp_moments_listed<MODEL, MODE_PULL><<<cdiv(d->nb, 128), 128, 0, st>>>(d->buf[0][s], d->buf[1][s], d->g, tp->mg, tp->mom, tp->p, table_of(d),
                                                                           nullptr, nullptr, part == TP_PRE_CUT ? 1 : 2);
    d->launches++;
  }
  if (part == TP_PRE_CUT)
  {
    k_tp_pad_cols<<<1, 128, 0, st>>>(tp->mom, d->g, tp->mg, M_COUNT, 0, 2);
    k_tp_pad_cols<<<1, 128, 0, st>>>(tp->mom, d->g, tp->mg, M_COUNT, Xl - 2, Xl);
    const int lo = d->cfg.x0 == 0, hi = d->cfg.x1 == d->cfg.X;  // the global edge replicates rows 0 / Xl-1 (padded width: after the columns)
    if (lo || hi) k_tp_pad_rows<<<cdiv(d->g.Y + 4, 128), 128, 0, st>>>(tp->mom, d->g, tp->mg, lo, hi, M_COUNT);
    d->launches += 2 + (lo || hi);
  }
  else
  {
    k_tp_pad_cols<<<cdiv(Xl - 4, 128), 128, 0, st>>>(tp->mom, d->g, tp->mg, M_COUNT, 2, Xl - 2);
    d->launches++;
  }
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

// can lbm_step run the remaining steps through tp_steps_ring?
bool tp_ring_overlap_ok(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  if (!tp || tp->model == TP_CSF || !tp->ring_overlap || !comm_active(d) || d->post_stream || d->g.Xl < 16 || d->g.Y < 3) return false;
  if (tp_build_region(d) != LBM_OK) return false;
  if (tp->rows_per_block <= 0) with_model(tp, [&](auto M) { return tp_launch_fused<M>(d, TP_BANDS_NONE); });
  const int rpb = tp->rows_per_block, nb = cdiv(d->g.Xl, rpb);
  if (rpb < 4 || nb < 4) return false;
  // a band overwrites the listed nodes of its rows' interior columns until the listed-node kernel has run: interior bands must hold none
  const int k_hi = tp_edge_bands_hi(d);
  for (int x = rpb; x < (nb - k_hi) * rpb && x < (int)d->row_has_listed.size(); x++)
    if (d->row_has_listed[x]) return false;
  return true;
}

template <int MODEL>
static int tp_steps_ring_t(lbm_domain* d, int n)
{
  TwoPhaseState* tp = d->tp;
  cudaStream_t side = d->side;
  // the first step's cut rows: in line
  LBM_TRY(tp_pre_part<MODEL>(d, TP_PRE_CUT, d->stream));
  {
    ProfScope ps(d, LBM_PROF_MOMENTS);
    LBM_TRY(comm_exchange_moments(d));
  }
  for (int i = 0; i < n; i++)
  {
    LBM_TRY(tp_pre_part<MODEL>(d, TP_PRE_REST, d->stream));
    if (i > 0) LBM_CUDA(cudaStreamWaitEvent(d->stream, d->ev_side, 0));  // ghost rows and cut-row moments of this state
    LBM_TRY(tp_launch_fused<MODEL>(d, TP_BANDS_EDGE));
    LBM_CUDA(cudaEventRecord(d->ev_early, d->stream));
    LBM_CUDA(cudaStreamWaitEvent(side, d->ev_early, 0));
    {
      // queued before the interior bands (its blocks find an idle GPU; measured the same as queued after them)
      ProfScope ps(d, LBM_PROF_GHOST, side);
      LBM_TRY(comm_exchange(d, d->cur ^ 1, side));
    }
    LBM_TRY(tp_launch_fused<MODEL>(d, TP_BANDS_INTERIOR));
    d->cur ^= 1;
    tp->planes_full = false;
    if (i + 1 < n)
    {
      LBM_TRY(tp_pre_part<MODEL>(d, TP_PRE_CUT, side));
      ProfScope ps(d, LBM_PROF_MOMENTS, side);
      int pm = 0;
      long long mplane = 0;
      LBM_TRY(comm_exchange_planes(d, tp_moment_planes(d, &pm, &mplane), M_COUNT, side));
    }
    LBM_CUDA(cudaEventRecord(d->ev_side, side));
  }
  LBM_CUDA(cudaStreamWaitEvent(d->stream, d->ev_side, 0));
  return LBM_OK;
}

int tp_steps_ring(lbm_domain* d, int n)
{
  return with_model(d->tp, [&](auto M) { return tp_steps_ring_t<M>(d, n); });
}

static int csf_fill_planes(lbm_domain* d);

// two rows of `nplanes` planes (moment-plane geometry) from the linked neighbours across every INTERNAL cut (the global
// edge replicates): the five moment planes, or the CSF model's normal field
static int tp_link_halo_planes(lbm_domain* d, double* TwoPhaseState::*field, int nplanes)
{
  TwoPhaseState* tp = d->tp;
  const int pm = tp->mg.pm, Xl = d->g.Xl;
  const size_t bytes = sizeof(double) * 2 * pm;
  for (int f = 0; f < nplanes; f++)
  {
    double* pl = tp->*field + (long long)f * tp->mg.mplane;
    if (d->cfg.x0 > 0 && d->link_lo)  // rows -2, -1 <- the lower slab's last two rows
    {
      lbm_domain* o = d->link_lo;
      const double* src = o->tp->*field + (long long)f * o->tp->mg.mplane + (long long)o->g.Xl * o->tp->mg.pm;
      if (o->cfg.device == d->cfg.device) LBM_CUDA(cudaMemcpyAsync(pl, src, bytes, cudaMemcpyDeviceToDevice, d->stream));
      else LBM_CUDA(cudaMemcpyPeerAsync(pl, d->cfg.device, src, o->cfg.device, bytes, d->stream));
      d->launches++;
    }
    if (d->cfg.x1 < d->cfg.X && d->link_hi)  // rows Xl, Xl+1 <- the upper slab's first two rows
    {
      lbm_domain* o = d->link_hi;
      const double* src = o->tp->*field + (long long)f * o->tp->mg.mplane + (long long)2 * o->tp->mg.pm;
      double* dst = pl + (long long)(Xl + 2) * pm;
      if (o->cfg.device == d->cfg.device) LBM_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, d->stream));
      else LBM_CUDA(cudaMemcpyPeerAsync(dst, d->cfg.device, src, o->cfg.device, bytes, d->stream));
      d->launches++;
    }
  }
  return LBM_OK;
}

// moments of every own node of the current state into the planes (diagnostics: lbm_get_moments /
// lbm_get_phase after fused steps).  No exchange: the halo cells are rebuilt by the next step.
static int tp_fill_planes(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  if (tp->planes_full || d->post_stream) return LBM_OK;
  if (tp->model == TP_CSF) return csf_fill_planes(d);
  LBM_TRY(with_model(tp, [&](auto M) { return tp_launch_moments<M>(d, d->cur, nullptr, nullptr); }));
  tp->planes_full = true;
  return LBM_OK;
}

int tp_commit(lbm_domain* d)
{
  for (const auto& so : d->ops)
    if (so.op.kind != LBM_BC_LINEAR)
    {
      set_error("two-phase models take LBM_BC_LINEAR rules only");
      return LBM_ERR_UNSUPPORTED;
    }
  d->tp->region_dirty = true;
  d->tp->csf_lists_dirty = true;
  return commit_boundary_tables(d);
}

// post-stream populations of both colours into d_aos[] (device, reference layout)
int tp_export(lbm_domain* d)
{
  const long long N = (long long)d->g.Xl * d->g.Y;
  if (d->post_stream)
  {
    for (int l = 0; l < 2; l++)
    {
      k_export_soa_to_aos<<<cdiv(N, 256), 256, 0, d->stream>>>(d->buf[l][d->cur], d->d_aos[l], d->g);
      d->launches++;
    }
    LBM_CUDA(cudaGetLastError());
    return LBM_OK;
  }
  // (with output pointers the pass only pulls: no model arithmetic)
  return with_model(d->tp, [&](auto M) { return tp_launch_moments<M>(d, d->cur, d->d_aos[0], d->d_aos[1]); });
}

int tp_stage_moments(lbm_domain* d, double* stage)
{
  const long long N = (long long)d->g.Xl * d->g.Y;
  LBM_TRY(tp_fill_planes(d));
  k_tp_read_moments<<<cdiv(N, 256), 256, 0, d->stream>>>(d->tp->mom, d->g, d->tp->mg, stage, stage + N, stage + 3 * N, stage + 4 * N,
                                                         stage + 5 * N);
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

// after lbm_set_f on a two-phase domain: rebuild the moment planes from the imported populations
int tp_refresh_moments(lbm_domain* d)
{
  const long long N = (long long)d->g.Xl * d->g.Y;
  with_model(d->tp, [&](auto M) {  // TP_CSF: an import carries no interfacial tension (u = j / rho + Fg / (2 rho))
    k_tp_moments_local<M><<<cdiv(N, 256), 256, 0, d->stream>>>(d->buf[0][d->cur], d->buf[1][d->cur], d->g, d->tp->mg, d->tp->mom, d->tp->p);
    return LBM_OK;
  });
  d->launches++;
  d->tp->planes_full = true;
  LBM_TRY(tp_pad(d));
  return comm_exchange_moments(d);
}

// ================================================================================================
// TP_CSF — test/mrt_rayleigh_taylor.cpp (SURVEY §8(f) rank 2).  First correct path: three passes per step over
// full moment planes (moments -> normals -> collision), stencils straight from the padded planes.
//   aux planes: A_NX, A_NY  n = -grad(phase) / (1e-20 + |grad|)  (padded like the moment planes: D differentiates them)
//               A_FX, A_FY  interfacial tension Fs = -sigma/2 K grad(phase), carried into the next step's velocity
// ================================================================================================
enum AuxPlane { A_NX = 0, A_NY = 1, A_FX = 2, A_FY = 3 };

// 5x5 isotropic differences of one padded plane at (x, y): dx along axis 0, dy along axis 1 (src/differential.hpp:9-40).
// This model divides by 1e-20 + |grad(phase)| (mrt_rayleigh_taylor.cpp:508): where the phase field is constant to
// machine precision the "normal" is the sign pattern of the ROUNDING RESIDUE of this sum, and the curvature of the
// rim nodes differentiates it.  To stay on the CPU reference there as far as that is possible at all, the sum runs in
// the order of a plain convolution loop (rows, then columns) with separately rounded products and additions — no
// fused multiply-add — like the oracle's orc_diff5; an exactly constant neighbourhood then leaves the same residue.
__device__ __forceinline__ void diff5_at(const double* __restrict__ pl, const MomGeom& mg, int x, int y, double& dx, double& dy)
{
  const long long o = mom_off(mg, x, y);
  dx = dy = 0.0;
#pragma unroll
  for (int a = -2; a <= 2; a++)
#pragma unroll
    for (int b = -2; b <= 2; b++)
    {
      if (a == 0 && b == 0) continue;
      const double v = pl[o + (long long)a * mg.pm + b];
      const double w = XI5(a, b);
      if (a != 0) dx = __dadd_rn(dx, __dmul_rn(w * (double)a, v));
      if (b != 0) dy = __dadd_rn(dy, __dmul_rn(w * (double)b, v));
    }
}

template <int MODE>
__global__ void __launch_bounds__(256)
k_csf_moments_interior(const double* __restrict__ rsrc, const double* __restrict__ bsrc, const SlabGeom g, const MomGeom mg,
                       double* __restrict__ mom, const double* __restrict__ aux, const TpParams p)
{
  const int y = 1 + blockIdx.x * blockDim.x + threadIdx.x;
  const int x = blockIdx.y;
  if (y > g.Y - 2) return;
  double fr[9], fb[9];
  tp_load_interior<MODE>(rsrc, g, x, y, fr);
  tp_load_interior<MODE>(bsrc, g, x, y, fb);
  const long long k = mom_off(mg, x, y);
  double rr, rb, ux, uy, ph;
  tp_moments<TP_CSF>(p, fr, fb, rr, rb, ux, uy, ph, aux[A_FX * mg.mplane + k], aux[A_FY * mg.mplane + k]);
  mom[M_RR * mg.mplane + k] = rr;
  mom[M_RB * mg.mplane + k] = rb;
  mom[M_UX * mg.mplane + k] = ux;
  mom[M_UY * mg.mplane + k] = uy;
  mom[M_PH * mg.mplane + k] = ph;
}

template <int MODE>
__global__ void __launch_bounds__(128)
k_csf_moments_listed(const double* __restrict__ rsrc, const double* __restrict__ bsrc, const SlabGeom g, const MomGeom mg,
                     double* __restrict__ mom, const double* __restrict__ aux, const TpParams p, const BoundaryTable t)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= t.n) return;
  const int x = t.x[i], y = t.y[i];
  double fr[9], fb[9];
  tp_load_listed<MODE>(rsrc, g, t, 0, i, x, y, fr);
  tp_load_listed<MODE>(bsrc, g, t, 1, i, x, y, fb);
  const long long k = mom_off(mg, x, y);
  double rr, rb, ux, uy, ph;
  tp_moments<TP_CSF>(p, fr, fb, rr, rb, ux, uy, ph, aux[A_FX * mg.mplane + k], aux[A_FY * mg.mplane + k]);
  mom[M_RR * mg.mplane + k] = rr;
  mom[M_RB * mg.mplane + k] = rb;
  mom[M_UX * mg.mplane + k] = ux;
  mom[M_UY * mg.mplane + k] = uy;
  mom[M_PH * mg.mplane + k] = ph;
}

// n = -grad(phase) / (1e-20 + |grad(phase)|)   (mrt_rayleigh_taylor.cpp:500-508)
__global__ void __launch_bounds__(256)
k_csf_normals(const double* __restrict__ mom, double* __restrict__ aux, const SlabGeom g, const MomGeom mg)
{
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (long long)g.Xl * g.Y) return;
  const int x = (int)(n / g.Y), y = (int)(n % g.Y);
  double gx, gy;
  diff5_at(mom + M_PH * mg.mplane, mg, x, y, gx, gy);
  const double inv = 1.0 / (1e-20 + sqrt(gx * gx + gy * gy));
  const long long k = mom_off(mg, x, y);
  aux[A_NX * mg.mplane + k] = -gx * inv;
  aux[A_NY * mg.mplane + k] = -gy * inv;
}

// collision of one node: stencils from the planes, curvature, interfacial tension (stored), tp_collide<TP_CSF>
__device__ __forceinline__ void csf_collide_node(const TpParams& p, const double* __restrict__ mom, const double* __restrict__ aux,
                                                 double* __restrict__ aux_out, const MomGeom& mg, int x, int y, double (&fr)[9],
                                                 double (&fb)[9])
{
  TpStencil st;
  tp_stencil_global<TP_MRTCG>(p, mom, mg, x, y, st);  // grad(phase), d/dx Q_x, d/dy Q_y
  double dx_nx, dy_nx, dx_ny, dy_ny;
  diff5_at(aux + A_NX * mg.mplane, mg, x, y, dx_nx, dy_nx);
  diff5_at(aux + A_NY * mg.mplane, mg, x, y, dx_ny, dy_ny);
  const long long k = mom_off(mg, x, y);
  const double nx = aux[A_NX * mg.mplane + k], ny = aux[A_NY * mg.mplane + k];
  // eval_local_curvature (:355-364); interf_tension = -0.5 sigma K grad (:510)
  const double K = nx * ny * (dy_nx + dx_ny) - (nx * nx) * dy_ny - (ny * ny) * dx_nx;
  st.Fsx = (-0.5 * p.sigma) * K * st.gx;
  st.Fsy = (-0.5 * p.sigma) * K * st.gy;
  aux_out[A_FX * mg.mplane + k] = st.Fsx;  // (aux_out == aux in the three-pass step: other planes of the same set)
  aux_out[A_FY * mg.mplane + k] = st.Fsy;
  const double rr = mom[M_RR * mg.mplane + k], rb = mom[M_RB * mg.mplane + k];
  const double ux = mom[M_UX * mg.mplane + k], uy = mom[M_UY * mg.mplane + k], ph = mom[M_PH * mg.mplane + k];
  tp_collide<TP_CSF>(p, fr, fb, rr, rb, ux, uy, ph, st);
}

// ---- collision pass, interior columns: 128-thread column strips marching down row bands like k_tp_fused, the nine
// fields a node's stencils and collision read (phase, Q_x, Q_y, n_x, n_y, rho_r, rho_b, u_x, u_y) staged row by row from
// the planes into a shared-memory ring of 2H+2 rows.  (Measured at 8192^2: 5.2 ms per step; a first version that took its 113
// stencil values per node straight from the planes through L1 needed 5.55 ms.  Like k_tp_fused the pass is bound by how many
// loads 12 warps of long fp64 chains keep in flight, not by the stencil reads.)
struct CsfRing
{
  static constexpr int H = 2, NR = 2 * H + 2, NF = 9;
  static constexpr int F_NX = 3, F_NY = 4, F_RR = 5, F_RB = 6, F_UX = 7, F_UY = 8;  // 0..2 = phase, Q_x, Q_y (tp_ring_stencil)
  static constexpr int USEFUL = TPF_NT - 2 * H;
  static constexpr size_t SMEM = sizeof(double) * NF * NR * TPF_NT;
};

// 5x5 differences of ring field f (the normal components).  Plain fused multiply-adds: unlike the gradient of the phase
// field in k_csf_normals, nothing divides by these sums, so their last bit does not matter.
__device__ __forceinline__ void csf_ring_diff5(const double* __restrict__ sm, int f, int sc, int t, double& dx, double& dy)
{
  constexpr int NR = CsfRing::NR, NT = TPF_NT;
  dx = dy = 0.0;
#pragma unroll
  for (int a = -2; a <= 2; a++)
  {
          const int sa = (sc + NR + a) % NR;  // (a compare-and-wrap instead of the constant division measured 0 - 1.5 % slower)
#pragma unroll
    for (int b = -2; b <= 2; b++)
    {
      if (a == 0 && b == 0) continue;
      const double v = sm[(f * NR + sa) * NT + t + b];
      const double w = XI5(a, b);
      if (a != 0) dx += (w * (double)a) * v;
      if (b != 0) dy += (w * (double)b) * v;
    }
  }
}

template <int MODE>
__global__ void __launch_bounds__(TPF_NT, 3)
k_csf_collide_ring(const double* __restrict__ rsrc, const double* __restrict__ bsrc, double* __restrict__ rdst,
                   double* __restrict__ bdst, const SlabGeom g, const MomGeom mg, const double* __restrict__ mom,
                   double* __restrict__ aux, const TpParams p, int rows_per_block)
{
  using C = CsfRing;
  constexpr int H = C::H, NR = C::NR, NT = TPF_NT;
  extern __shared__ double sm[];  // [NF][NR][NT]
  auto S = [&](int f, int slot, int col) -> double& { return sm[(f * NR + slot) * NT + col]; };
  const int t = threadIdx.x;
  const int y = 1 + blockIdx.x * C::USEFUL - H + t;
  const int xb = blockIdx.y * rows_per_block;
  const int xe = min(xb + rows_per_block, g.Xl);
  const bool col_ok = y >= -2 && y <= g.Y + 1;  // inside the padded planes
  const bool collider = t >= H && t < NT - H && y >= 1 && y <= g.Y - 2;
  int slot = 0;
  for (int r = xb - H; r < xe + H; r++)
  {
    if (col_ok)
    {
      const long long k = mom_off(mg, r, y);
      const double rr = mom[M_RR * mg.mplane + k], rb = mom[M_RB * mg.mplane + k];
      const double ux = mom[M_UX * mg.mplane + k], uy = mom[M_UY * mg.mplane + k];
      const double cq = p.cr * rr + p.cb * rb;
      S(0, slot, t) = mom[M_PH * mg.mplane + k];
      S(1, slot, t) = cq * ux;
      S(2, slot, t) = cq * uy;
      S(C::F_NX, slot, t) = aux[A_NX * mg.mplane + k];
      S(C::F_NY, slot, t) = aux[A_NY * mg.mplane + k];
      S(C::F_RR, slot, t) = rr;
      S(C::F_RB, slot, t) = rb;
      S(C::F_UX, slot, t) = ux;
      S(C::F_UY, slot, t) = uy;
    }
    __syncthreads();
    const int x = r - H;  // its stencil rows x-H .. x+H are the last 2H+1 slots
    if (x >= xb && collider)
    {
      const int sc = (slot + NR - H) % NR;
      double fr[9], fb[9];
      tp_load_interior<MODE>(rsrc, g, x, y, fr);
      tp_load_interior<MODE>(bsrc, g, x, y, fb);
      TpStencil st;
      tp_ring_stencil<TP_MRTCG>(sm, sc, t, st);  // grad(phase), d/dx Q_x, d/dy Q_y
      double dx_nx, dy_nx, dx_ny, dy_ny;
      csf_ring_diff5(sm, C::F_NX, sc, t, dx_nx, dy_nx);
      csf_ring_diff5(sm, C::F_NY, sc, t, dx_ny, dy_ny);
      const double nx = S(C::F_NX, sc, t), ny = S(C::F_NY, sc, t);
      const double K = nx * ny * (dy_nx + dx_ny) - (nx * nx) * dy_ny - (ny * ny) * dx_nx;  // eval_local_curvature (:355-364)
      st.Fsx = (-0.5 * p.sigma) * K * st.gx;                                              // interf_tension (:510)
      st.Fsy = (-0.5 * p.sigma) * K * st.gy;
      const long long k = mom_off(mg, x, y);
      aux[A_FX * mg.mplane + k] = st.Fsx;
      aux[A_FY * mg.mplane + k] = st.Fsy;
      tp_collide<TP_CSF>(p, fr, fb, S(C::F_RR, sc, t), S(C::F_RB, sc, t), S(C::F_UX, sc, t), S(C::F_UY, sc, t), S(0, sc, t), st);
      const long long o = node_off(g, x, y);
#pragma unroll
      for (int q = 0; q < 9; q++)
      {
        rdst[q * g.plane + o] = fr[q];
        bdst[q * g.plane + o] = fb[q];
      }
    }
    slot = slot + 1 == NR ? 0 : slot + 1;
    // no second barrier: the row written next iteration is the slot the oldest stencil row of THIS iteration's
    // collision occupied only after NR - (2H+1) = 1 more advance, i.e. slot (sc - H - 1) mod NR, which nobody reads now
  }
}

template <int MODE>
__global__ void __launch_bounds__(128)
k_csf_collide_listed(const double* __restrict__ rsrc, const double* __restrict__ bsrc, double* __restrict__ rdst,
                     double* __restrict__ bdst, const SlabGeom g, const MomGeom mg, const double* __restrict__ mom,
                     const double* __restrict__ aux, double* __restrict__ aux_out, const TpParams p, const BoundaryTable t)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= t.n) return;
  const int x = t.x[i], y = t.y[i];
  double fr[9], fb[9];
  tp_load_listed<MODE>(rsrc, g, t, 0, i, x, y, fr);
  tp_load_listed<MODE>(bsrc, g, t, 1, i, x, y, fb);
  csf_collide_node(p, mom, aux, aux_out, mg, x, y, fr, fb);
  const long long o = node_off(g, x, y);
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    rdst[q * g.plane + o] = fr[q];
    bdst[q * g.plane + o] = fb[q];
  }
}

// ================================================================================================
// TP_CSF in ONE pass over the populations (LBM_CSF_FUSED=1; monolithic domains).  Row-marching column strips like
// k_tp_fused, with two lags: the moments of row r enter a ring, the normal of row r-2 is formed from the ring's phase
// rows r-4 .. r, and row r-5 is collided from the moment rows r-7 .. r-3 and the normal rows r-7 .. r-3.  The
// populations are pulled twice (the second time out of L2, five rows later); nothing but the interfacial tension is
// written besides them: 320 B/node of DRAM traffic against the 584 B of the three-pass step.
//   planes stay authoritative (a pre-pass fills them) where the kernel cannot form a value itself:
//     moments  listed nodes, the padding, rows within 4 of a row with listed nodes or of the global edge rows 0..2
//     normals  listed nodes, the padding (replicated NORMALS, not normals of the replicated phase), rows within 2 of ...
//   Fs is double-buffered (aux -> aux_next): a neighbouring strip's halo still reads the previous step's value.
// ================================================================================================
struct CsfFused
{
  static constexpr int HC = 4;                 // halo columns per side: 2 for the curvature's normals + 2 for their phase
  static constexpr int NRM = 9, NRN = 6;       // ring rows: moments r-7 .. r + the one being written; normals r-7 .. r-2
  static constexpr int LAG_N = 2, LAG_C = 5;
  static constexpr int USEFUL = TPF_NT - 2 * HC;
  static constexpr size_t SMEM = sizeof(double) * (3 * NRM + 2 * NRN) * TPF_NT;
};

// pre-pass: moments of listed interior-column nodes' neighbourhoods (with the carried interfacial tension) into the planes
__global__ void __launch_bounds__(128)
k_csf_moments_nodes(const double* __restrict__ rsrc, const double* __restrict__ bsrc, const SlabGeom g, const MomGeom mg,
                    double* __restrict__ mom, const double* __restrict__ aux, const TpParams p, const int* __restrict__ nodes, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int x = nodes[i] / g.Y, y = nodes[i] % g.Y;
  double fr[9], fb[9];
  tp_load_interior<MODE_PULL>(rsrc, g, x, y, fr);
  tp_load_interior<MODE_PULL>(bsrc, g, x, y, fb);
  const long long k = mom_off(mg, x, y);
  double rr, rb, ux, uy, ph;
  tp_moments<TP_CSF>(p, fr, fb, rr, rb, ux, uy, ph, aux[A_FX * mg.mplane + k], aux[A_FY * mg.mplane + k]);
  mom[M_RR * mg.mplane + k] = rr;
  mom[M_RB * mg.mplane + k] = rb;
  mom[M_UX * mg.mplane + k] = ux;
  mom[M_UY * mg.mplane + k] = uy;
  mom[M_PH * mg.mplane + k] = ph;
}

// pre-pass: normals of a node list from the (padded) phase plane
__global__ void __launch_bounds__(128)
k_csf_normals_nodes(const double* __restrict__ mom, double* __restrict__ aux, const SlabGeom g, const MomGeom mg,
                    const int* __restrict__ nodes, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int x = nodes[i] / g.Y, y = nodes[i] % g.Y;
  double gx, gy;
  diff5_at(mom + M_PH * mg.mplane, mg, x, y, gx, gy);
  const double inv = 1.0 / (1e-20 + sqrt(gx * gx + gy * gy));
  const long long k = mom_off(mg, x, y);
  aux[A_NX * mg.mplane + k] = -gx * inv;
  aux[A_NY * mg.mplane + k] = -gy * inv;
}

// PIPE: the pulls of row r are issued first and finished (moments, ring) after the normal / collision work of the previous
// iteration, so their DRAM latency hides under that fp64 work (as in k_tp_fused); 36 more live registers, hence two
// resident blocks instead of three.  Which of the two is faster is a measurement (LBM_CSF_PIPE=1; default off).
template <bool PIPE>
__global__ void __launch_bounds__(TPF_NT, PIPE ? 2 : 3)
k_csf_fused(const double* __restrict__ rsrc, const double* __restrict__ bsrc, double* __restrict__ rdst, double* __restrict__ bdst,
            const SlabGeom g, const MomGeom mg, const double* __restrict__ mom, const double* __restrict__ aux,
            double* __restrict__ aux_out, const TpParams p, const unsigned char* __restrict__ rowflags, int rows_per_block)
{
  using C = CsfFused;
  constexpr int NT = TPF_NT, NRM = C::NRM, NRN = C::NRN, HC = C::HC;
  extern __shared__ double sm[];  // moments [3][NRM][NT] (phase, Q_x, Q_y), then normals [2][NRN][NT]
  double* smn = sm + 3 * NRM * NT;
  auto M = [&](int f, int slot, int col) -> double& { return sm[(f * NRM + slot) * NT + col]; };
  auto N = [&](int f, int slot, int col) -> double& { return smn[(f * NRN + slot) * NT + col]; };
  const int t = threadIdx.x;
  const int y = 1 + blockIdx.x * C::USEFUL - HC + t;
  const int xb = blockIdx.y * rows_per_block;
  const int xe = min(xb + rows_per_block, g.Xl);
  const bool col_ok = y >= -2 && y <= g.Y + 1;      // inside the padded planes
  const bool col_plane = y < 1 || y > g.Y - 2;      // listed edge columns and the padding
  const bool normal_thread = t >= 2 && t < NT - 2;  // has the phase of its columns y-2 .. y+2 in the ring
  const bool collider = t >= HC && t < NT - HC && y >= 1 && y <= g.Y - 2;
  __shared__ unsigned char sflag[128 + 16];  // flags of rows xb-4 .. xe+4 (outside the slab: everything from the planes)
  for (int k = t; k < xe - xb + 9; k += NT)
  {
    const int r = xb - 4 + k;
    sflag[k] = (r < 0 || r >= g.Xl) ? 3 : rowflags[r];
  }
  __syncthreads();
  auto flag_of = [&](int r) -> int { return sflag[r - (xb - 4)]; };

  // ---- B of iteration it: normal of (it - 2, y) -> normal ring
  auto stage_normal = [&](int it) {
    {
      const int rn = it - C::LAG_N;
      if (col_ok && rn >= xb - 2 && rn <= xe + 1 && rn >= -2 && rn <= g.Xl + 1)
      {
        double nx = 0.0, ny = 0.0;
        bool have = false;
        if (col_plane || (flag_of(rn) & 2))
        {
          const long long k = mom_off(mg, rn, y);
          nx = aux[A_NX * mg.mplane + k];
          ny = aux[A_NY * mg.mplane + k];
          have = true;
        }
        else if (normal_thread)
        {
          // the summation order of diff5_at (k_csf_normals): rows, then columns, separately rounded products and sums
          double gx = 0.0, gy = 0.0;
#pragma unroll
          for (int a = -2; a <= 2; a++)
          {
            const int sa = (rn + a + 4 * NRM) % NRM;
#pragma unroll
            for (int b = -2; b <= 2; b++)
            {
              if (a == 0 && b == 0) continue;
              const double v = M(0, sa, t + b);
              const double w = XI5(a, b);
              if (a != 0) gx = __dadd_rn(gx, __dmul_rn(w * (double)a, v));
              if (b != 0) gy = __dadd_rn(gy, __dmul_rn(w * (double)b, v));
            }
          }
          const double inv = 1.0 / (1e-20 + sqrt(gx * gx + gy * gy));
          nx = -gx * inv;
          ny = -gy * inv;
          have = true;
        }
        if (have)
        {
          const int slot = (rn + 4 * NRN) % NRN;
          N(0, slot, t) = nx;
          N(1, slot, t) = ny;
        }
      }
    }
  };
  // ---- C of iteration it: collision of (it - 5, y) from moment rows it-7 .. it-3 and normal rows it-7 .. it-3 (written before
  //      the barrier that precedes this stage)
  auto stage_collide = [&](int it) {
    {
      const int x = it - C::LAG_C;
      if (x >= xb && x < xe && collider)
      {
        double fr[9], fb[9];
        tp_pull_at(rsrc + node_off(g, x, y), g, fr);
        tp_pull_at(bsrc + node_off(g, x, y), g, fb);
        const long long k = mom_off(mg, x, y);
        double rr, rb, ux, uy, ph;
        // the same arithmetic on the same inputs as stage A / the pre-pass: identical values, no ring rows for them
        tp_moments<TP_CSF>(p, fr, fb, rr, rb, ux, uy, ph, aux[A_FX * mg.mplane + k], aux[A_FY * mg.mplane + k]);
        TpStencil st;
        st.gx = st.gy = st.DxQx = st.DyQy = 0.0;
        double dx_nx = 0.0, dy_nx = 0.0, dx_ny = 0.0, dy_ny = 0.0;
#pragma unroll
        for (int a = -2; a <= 2; a++)
        {
          const int sa = (x + a + 4 * NRM) % NRM;
#pragma unroll
          for (int b = -2; b <= 2; b++)
          {
            if (a == 0 && b == 0) continue;
            const double w = XI5(a, b);
            if (a != 0)
            {
              st.gx += (w * (double)a) * M(0, sa, t + b);
              st.DxQx += (w * (double)a) * M(1, sa, t + b);
            }
            if (b != 0)
            {
              st.gy += (w * (double)b) * M(0, sa, t + b);
              st.DyQy += (w * (double)b) * M(2, sa, t + b);
            }
          }
        }
#pragma unroll
        for (int a = -2; a <= 2; a++)
        {
          const int na = (x + a + 4 * NRN) % NRN;
#pragma unroll
          for (int b = -2; b <= 2; b++)
          {
            if (a == 0 && b == 0) continue;
            const double w = XI5(a, b);
            const double vx = N(0, na, t + b), vy = N(1, na, t + b);
            if (a != 0) { dx_nx += (w * (double)a) * vx; dx_ny += (w * (double)a) * vy; }
            if (b != 0) { dy_nx += (w * (double)b) * vx; dy_ny += (w * (double)b) * vy; }
          }
        }
        const int nc = (x + 4 * NRN) % NRN;
        const double nx = N(0, nc, t), ny = N(1, nc, t);
        const double K = nx * ny * (dy_nx + dx_ny) - (nx * nx) * dy_ny - (ny * ny) * dx_nx;  // eval_local_curvature (:355-364)
        st.Fsx = (-0.5 * p.sigma) * K * st.gx;                                              // interf_tension (:510)
        st.Fsy = (-0.5 * p.sigma) * K * st.gy;
        aux_out[A_FX * mg.mplane + k] = st.Fsx;
        aux_out[A_FY * mg.mplane + k] = st.Fsy;
        tp_collide<TP_CSF>(p, fr, fb, rr, rb, ux, uy, ph, st);
        const long long o = node_off(g, x, y);
#pragma unroll
        for (int q = 0; q < 9; q++)
        {
          rdst[q * g.plane + o] = fr[q];
          bdst[q * g.plane + o] = fb[q];
        }
      }
    }
  };
  for (int r = xb - 4; r <= xe + 4 + (PIPE ? 1 : 0); r++)
  {
    // ---- A: moments of (r, y) -> moment ring.  Loads first ...
    const bool want = col_ok && r >= -2 && r <= g.Xl + 1 && r <= xe + 4;
    const bool plane = want && (col_plane || (flag_of(r) & 1));
    double fr[9], fb[9];
    double rr, rb, ux, uy, ph, fsx = 0.0, fsy = 0.0;
    if (want)
    {
      const long long k = mom_off(mg, r, y);
      if (plane)
      {
        rr = mom[M_RR * mg.mplane + k];
        rb = mom[M_RB * mg.mplane + k];
        ux = mom[M_UX * mg.mplane + k];
        uy = mom[M_UY * mg.mplane + k];
        ph = mom[M_PH * mg.mplane + k];
      }
      else
      {
        tp_pull_at(rsrc + node_off(g, r, y), g, fr);
        tp_pull_at(bsrc + node_off(g, r, y), g, fb);
        fsx = aux[A_FX * mg.mplane + k];
        fsy = aux[A_FY * mg.mplane + k];
      }
    }
    // ... (pipelined) the previous iteration's normal and collision work while they are in flight ...
    if constexpr (PIPE)
    {
      if (r > xb - 4)
      {
        stage_normal(r - 1);
        stage_collide(r - 1);
      }
    }
    // ... then the moments, published
    if (want)
    {
      if (!plane) tp_moments<TP_CSF>(p, fr, fb, rr, rb, ux, uy, ph, fsx, fsy);
      const int slot = (r + 4 * NRM) % NRM;
      const double cq = p.cr * rr + p.cb * rb;
      M(0, slot, t) = ph;
      M(1, slot, t) = cq * ux;
      M(2, slot, t) = cq * uy;
    }
    __syncthreads();
    if constexpr (!PIPE)
    {
      stage_normal(r);
      stage_collide(r);
    }
    // no second barrier.  Plain: the next iteration writes moment slot (r+1) mod 9 = (r-8) mod 9 and, after ITS barrier, normal
    // slot (r-1) mod 6 = (r-7) mod 6 — the moment rows read above are r-7 .. r, the normal rows read after that barrier r-6 .. r-2.
    // Pipelined: the stages of iteration r-1 read moment rows r-8 .. r-1 and normal rows r-8 .. r-4 while this iteration writes
    // moment slot r mod 9 = (r-9) mod 9 and normal slot (r-3) mod 6 = (r-9) mod 6.
  }
}

// ------------------------------------------------------------------------------------------------
// The single pass with the population rows STAGED by bulk asynchronous copies and (STASH) parked in tensor memory —
// k_csf_fused's march, rings and plane rules; what changes is where the populations come from.  k_csf_fused pulls every
// row twice through registers, five rows apart, and on the B200 the second pull misses L2 (ncu: 322 B/node read against
// 160, long-scoreboard stalls on top).  Here every row is copied ONCE into a stage slot (18 bulk copies of the strip's
// column window per row, one mbarrier per slot), read out of it when its moments are formed, and kept for the collision
// five rows later
//   STASH = true : in the thread's own tensor-memory lane — 6 rows x 36 columns of populations + 5 rows x 8 columns of
//                  rho_r, rho_b, u (256 columns per block, two blocks per SM); the slot is free at once: NS = 3;
//   STASH = false: in the stage slot itself (6 resident rows + the rows in flight: NS = 7, 172 KB, one block per SM).
// Arithmetic per node exactly as k_csf_fused (same device functions, same summation order): the moments of the collided
// node are the ones formed when its row entered instead of a second evaluation of the same expression.
template <int NS>
struct CsfStaged
{
  using F = CsfFused;
  static constexpr int W = TPF_NT + 4, ROW = 20 * W;  // 18 population row segments + the carried interfacial tension (Fs_x, Fs_y)
  static constexpr size_t RING_BYTES = F::SMEM;
  static constexpr size_t SMEM = sizeof(double) * NS * ROW + RING_BYTES + sizeof(uint64_t) * NS;
  static constexpr int TMEM_COLS = 256, T_MOM = 6 * 36;  // columns: populations of 6 rows, then rho_r, rho_b, u_x, u_y of 5 rows
};

template <int NS, bool STASH>
__global__ void __launch_bounds__(TPF_NT, STASH ? 2 : 1)
k_csf_staged(const double* __restrict__ rsrc, const double* __restrict__ bsrc, double* __restrict__ rdst, double* __restrict__ bdst,
             const SlabGeom g, const MomGeom mg, const double* __restrict__ mom, const double* __restrict__ aux,
             double* __restrict__ aux_out, const TpParams p, const unsigned char* __restrict__ rowflags, int rows_per_block)
{
  using F = CsfFused;
  using C = CsfStaged<NS>;
  constexpr int NT = TPF_NT, NRM = F::NRM, NRN = F::NRN, HC = F::HC, W = C::W, LAG = F::LAG_C;
  constexpr int HOLD = STASH ? 0 : LAG;
  static_assert(NS >= HOLD + 2, "at least one row in flight");
  extern __shared__ double sm[];  // stages [NS][18][W] | moments ring [3][NRM][NT] | normals ring [2][NRN][NT] | mbarriers [NS]
  double* stage = sm;
  double* smm = sm + NS * C::ROW;
  double* smn = smm + 3 * NRM * NT;
  uint64_t* full = reinterpret_cast<uint64_t*>(smn + 2 * NRN * NT);
  auto M = [&](int f, int slot, int col) -> double& { return smm[(f * NRM + slot) * NT + col]; };
  auto N = [&](int f, int slot, int col) -> double& { return smn[(f * NRN + slot) * NT + col]; };
  const int t = threadIdx.x;
  const int ys = 1 + blockIdx.x * F::USEFUL - HC;
  const int y = ys + t;
  const int xb = blockIdx.y * rows_per_block;
  const int xe = min(xb + rows_per_block, g.Xl);
  const int r0 = xb - 4, r_end = xe + 4 + 1;          // rows r0 .. r_end - 1 are marched (the last iteration only collides)
  const int rs0 = max(r0, 0), rs1 = min(xe + 4, g.Xl); // rows whose populations are staged
  const bool col_ok = y >= -2 && y <= g.Y + 1;      // inside the padded planes
  const bool col_plane = y < 1 || y > g.Y - 2;      // listed edge columns and the padding
  const bool normal_thread = t >= 2 && t < NT - 2;  // has the phase of its columns y-2 .. y+2 in the ring
  const bool collider = t >= HC && t < NT - HC && y >= 1 && y <= g.Y - 2;
  const int c0 = (ys - 1) & ~1;
  const int lo = max(c0, 0), hi = min(c0 + W, g.pitch);
  const unsigned seg_bytes = (unsigned)(hi - lo) * (unsigned)sizeof(double);
  const int my = t + (ys - c0);

  __shared__ unsigned char sflag[128 + 16];  // flags of rows xb-4 .. xe+4 (outside the slab: everything from the planes)
  __shared__ uint32_t tmem_slot;
  for (int k = t; k < xe - xb + 9; k += NT)
  {
    const int r = r0 + k;
    sflag[k] = (r < 0 || r >= g.Xl) ? 3 : rowflags[r];
  }
  if (t == 0)
  {
    for (int s = 0; s < NS; s++) mbar_init(&full[s], 1);
    mbar_init_fence();
  }
  uint32_t tmem = 0;
  if constexpr (STASH) tmem = tmem_alloc<C::TMEM_COLS>(&tmem_slot);
  else __syncthreads();
  auto flag_of = [&](int r) -> int { return sflag[r - r0]; };

  // lanes 0 .. 17 of warp 0 own one population row segment each (source pointer at row 0, shared-memory offset); lanes 18, 19
  // the same column window of the carried interfacial tension's two planes (moment-plane geometry: two cells of padding)
  const int lane_q = (t < 18 ? t : 0) % 9;
  const int alo = max(c0 + 2, 0), ahi = min(c0 + 2 + W, mg.pm);   // plane columns [c0 + 2, c0 + 2 + W) hold grid columns [c0, c0 + W)
  const unsigned aux_bytes = (unsigned)(ahi - alo) * (unsigned)sizeof(double);
  const double* lane_src = t < 18 ? (t < 9 ? rsrc : bsrc) + (long long)lane_q * g.plane + node_off(g, -CX(lane_q), lo)
                                  : aux + (long long)(t == 18 ? A_FX : A_FY) * mg.mplane + 2LL * mg.pm + alo;  // (row 0 of the slab)
  double* lane_dst = stage + (t < 20 ? t : 0) * W + (t < 18 ? lo - c0 : alo - (c0 + 2));
  const long long lane_pitch = t < 18 ? g.pitch : mg.pm;
  const unsigned lane_bytes = t < 18 ? seg_bytes : aux_bytes;
  auto issue_row = [&](int rr, int slot) {
    if (t >= 32 || rr >= r_end) return;
    const bool staged = rr >= rs0 && rr < rs1;
    if (t == 0) mbar_arrive_expect_tx(&full[slot], staged ? 18u * seg_bytes + 2u * aux_bytes : 0u);
    __syncwarp();
    if (staged && t < 20) bulk_copy_g2s(lane_dst + (size_t)slot * C::ROW, lane_src + (long long)rr * lane_pitch, lane_bytes, &full[slot]);
  };
  constexpr int AHEAD = NS - HOLD - (STASH ? 0 : 1);  // rows issued before the march starts = distance of the loop's refill rule
  for (int j = 0; j < AHEAD; j++) issue_row(r0 + j, j);
  __syncthreads();

  // !STASH: rho_r, rho_b, u of rows r .. r-5 at this thread's column ride in registers
  double mrr[LAG + 1], mrb[LAG + 1], mux[LAG + 1], muy[LAG + 1];
#pragma unroll
  for (int k = 0; k <= LAG; k++) mrr[k] = mrb[k] = mux[k] = muy[k] = 0.0;

  // counters instead of k % NS, k / NS, k % 6, k % 5 and the ring slots' modulo arithmetic
  int sl = 0, sl_x = (NS - LAG % NS) % NS, sl_fill = AHEAD % NS, ts = 0, tm = 0;
  int ms = (r0 + 4 * NRM) % NRM;  // moment-ring slot of row r
  int ns = (r0 - F::LAG_N + 4 * NRN) % NRN;  // normal-ring slot of row r - 2
  unsigned par = 0;
  auto wrap = [](int v, int n) { return v < 0 ? v + n : (v >= n ? v - n : v); };  // v mod n for -n <= v < 2n
  for (int r = r0; r < r_end; r++)
  {
    const double* st_r = stage + (size_t)sl * C::ROW;
    mbar_wait(&full[sl], par);
    // ---- A: moments of (r, y) -> moment ring
    const bool want = col_ok && r >= -2 && r <= g.Xl + 1 && r <= xe + 3;  // (row xe + 4 only collides row xe - 1)
    const bool plane = want && (col_plane || (flag_of(r) & 1));
    double fr[9], fb[9];
    double rr = 0.0, rb = 0.0, ux = 0.0, uy = 0.0, ph = 0.0;
    if (STASH || (want && !plane))
    {
#pragma unroll
      for (int q = 0; q < 9; q++)
      {
        fr[q] = st_r[q * W + my - CY(q)];
        fb[q] = st_r[(9 + q) * W + my - CY(q)];
      }
    }
    if constexpr (STASH)
    {
      tmem_store_wait();  // the previous iterations' parks have landed (they are taken back five iterations after they were issued)
      tmem_store18(tmem + 36u * (unsigned)ts, fr, fb);
    }
    if (want)
    {
      const long long km = mom_off(mg, r, y);
      if (plane)
      {
        rr = mom[M_RR * mg.mplane + km];
        rb = mom[M_RB * mg.mplane + km];
        ux = mom[M_UX * mg.mplane + km];
        uy = mom[M_UY * mg.mplane + km];
        ph = mom[M_PH * mg.mplane + km];
      }
      else
        tp_moments<TP_CSF>(p, fr, fb, rr, rb, ux, uy, ph, st_r[18 * W + my], st_r[19 * W + my]);  // Fs of the previous step, staged with the row
      const double cq = p.cr * rr + p.cb * rb;
      M(0, ms, t) = ph;
      M(1, ms, t) = cq * ux;
      M(2, ms, t) = cq * uy;
    }
    if constexpr (!STASH)
    {
#pragma unroll
      for (int j = LAG; j > 0; j--)
      {
        mrr[j] = mrr[j - 1];
        mrb[j] = mrb[j - 1];
        mux[j] = mux[j - 1];
        muy[j] = muy[j - 1];
      }
      mrr[0] = rr; mrb[0] = rb; mux[0] = ux; muy[0] = uy;
    }
    __syncthreads();
    issue_row(r + AHEAD, sl_fill);
    // the collided row's populations start their way back from tensor memory under the normal's arithmetic
    [[maybe_unused]] uint32_t tr[36], tq[8];
    if constexpr (STASH)
    {
      tmem_load18_issue(tmem + 36u * (unsigned)(ts == 5 ? 0 : ts + 1), tr);       // row r - 5: slot (k - 5) mod 6 = (k + 1) mod 6
      tmem_load4_issue(tmem + (unsigned)C::T_MOM + 8u * (unsigned)tm, tq);        // and its moments: slot (k - 5) mod 5 = k mod 5
    }

    // ---- B: normal of (r - 2, y) -> normal ring
    {
      const int rn = r - F::LAG_N;
      if (col_ok && rn >= xb - 2 && rn <= xe + 1 && rn >= -2 && rn <= g.Xl + 1)
      {
        double nx = 0.0, ny = 0.0;
        bool have = false;
        if (col_plane || (flag_of(rn) & 2))
        {
          const long long kn = mom_off(mg, rn, y);
          nx = aux[A_NX * mg.mplane + kn];
          ny = aux[A_NY * mg.mplane + kn];
          have = true;
        }
        else if (normal_thread)
        {
          // the summation order of diff5_at (k_csf_normals): rows, then columns, separately rounded products and sums
          double gx = 0.0, gy = 0.0;
#pragma unroll
          for (int a = -2; a <= 2; a++)
          {
            const int sa = wrap(ms - F::LAG_N + a, NRM);  // moment row rn + a
#pragma unroll
            for (int b = -2; b <= 2; b++)
            {
              if (a == 0 && b == 0) continue;
              const double v = M(0, sa, t + b);
              const double w = XI5(a, b);
              if (a != 0) gx = __dadd_rn(gx, __dmul_rn(w * (double)a, v));
              if (b != 0) gy = __dadd_rn(gy, __dmul_rn(w * (double)b, v));
            }
          }
          const double inv = 1.0 / (1e-20 + sqrt(gx * gx + gy * gy));
          nx = -gx * inv;
          ny = -gy * inv;
          have = true;
        }
        if (have)
        {
          N(0, ns, t) = nx;
          N(1, ns, t) = ny;
        }
      }
    }
    // ---- C: collision of (r - 5, y) from moment rows r-7 .. r-3 and normal rows r-7 .. r-3 (written before this iteration's barrier)
    const int x = r - LAG;
    double crr, crb, cux, cuy;  // moments of the collided node, formed when its row entered
    if constexpr (STASH)
    {
      tmem_load_wait();
      tmem_unpack18(tr, fr, fb);
      tmem_unpack4(tq, crr, crb, cux, cuy);
    }
    else
    {
      crr = mrr[LAG]; crb = mrb[LAG]; cux = mux[LAG]; cuy = muy[LAG];
    }
    if (x >= xb && x < xe && collider)
    {
      if constexpr (!STASH)
      {
        const double* st_x = stage + (size_t)sl_x * C::ROW;
#pragma unroll
        for (int q = 0; q < 9; q++)
        {
          fr[q] = st_x[q * W + my - CY(q)];
          fb[q] = st_x[(9 + q) * W + my - CY(q)];
        }
      }
      const long long kx = mom_off(mg, x, y);
      TpStencil st;
      st.gx = st.gy = st.DxQx = st.DyQy = 0.0;
      double dx_nx = 0.0, dy_nx = 0.0, dx_ny = 0.0, dy_ny = 0.0;
#pragma unroll
      for (int a = -2; a <= 2; a++)
      {
        const int sa = wrap(ms - LAG + a, NRM);  // moment row x + a
#pragma unroll
        for (int b = -2; b <= 2; b++)
        {
          if (a == 0 && b == 0) continue;
          const double w = XI5(a, b);
          if (a != 0)
          {
            st.gx += (w * (double)a) * M(0, sa, t + b);
            st.DxQx += (w * (double)a) * M(1, sa, t + b);
          }
          if (b != 0)
          {
            st.gy += (w * (double)b) * M(0, sa, t + b);
            st.DyQy += (w * (double)b) * M(2, sa, t + b);
          }
        }
      }
#pragma unroll
      for (int a = -2; a <= 2; a++)
      {
        const int na = wrap(ns - (LAG - F::LAG_N) + a, NRN);  // normal row x + a
#pragma unroll
        for (int b = -2; b <= 2; b++)
        {
          if (a == 0 && b == 0) continue;
          const double w = XI5(a, b);
          const double vx = N(0, na, t + b), vy = N(1, na, t + b);
          if (a != 0) { dx_nx += (w * (double)a) * vx; dx_ny += (w * (double)a) * vy; }
          if (b != 0) { dy_nx += (w * (double)b) * vx; dy_ny += (w * (double)b) * vy; }
        }
      }
      const int nc = wrap(ns - (LAG - F::LAG_N), NRN);
      const double nx = N(0, nc, t), ny = N(1, nc, t);
      const double K = nx * ny * (dy_nx + dx_ny) - (nx * nx) * dy_ny - (ny * ny) * dx_nx;  // eval_local_curvature (:355-364)
      st.Fsx = (-0.5 * p.sigma) * K * st.gx;                                              // interf_tension (:510)
      st.Fsy = (-0.5 * p.sigma) * K * st.gy;
      aux_out[A_FX * mg.mplane + kx] = st.Fsx;
      aux_out[A_FY * mg.mplane + kx] = st.Fsy;
      tp_collide<TP_CSF>(p, fr, fb, crr, crb, cux, cuy, M(0, wrap(ms - LAG, NRM), t), st);
      const long long o = node_off(g, x, y);
#pragma unroll
      for (int q = 0; q < 9; q++)
      {
        rdst[q * g.plane + o] = fr[q];
        bdst[q * g.plane + o] = fb[q];
      }
    }
    // this row's moments take the tensor-memory slot the collided row's have just left
    if constexpr (STASH) tmem_store4(tmem + (unsigned)C::T_MOM + 8u * (unsigned)tm, rr, rb, ux, uy);
    ts = ts == 5 ? 0 : ts + 1;
    tm = tm == 4 ? 0 : tm + 1;
    ms = ms + 1 == NRM ? 0 : ms + 1;
    ns = ns + 1 == NRN ? 0 : ns + 1;
    sl_x = sl_x + 1 == NS ? 0 : sl_x + 1;
    sl_fill = sl_fill + 1 == NS ? 0 : sl_fill + 1;
    if (++sl == NS)
    {
      sl = 0;
      par ^= 1u;
    }
  }
  if constexpr (STASH) tmem_free<C::TMEM_COLS>(tmem);
}

// the single pass's row-marching kernels, as tp_kernels for MRTCG / RK
struct CsfKernel
{
  int staged;  // LBM_CSF_STAGED: 2 = k_csf_staged with the tensor-memory stash, 1 = without it, 0 (or any other value) = k_csf_fused
  bool pipe;   // k_csf_fused: the software-pipelined variant (LBM_CSF_PIPE)
  decltype(&k_csf_fused<false>) kernel;
  size_t smem;
  int warmup_rows;  // band height: pick_band_rows with this many warm-up rows per band, 0 = 64 rows
};
static const CsfKernel csf_kernels[] = {{0, false, k_csf_fused<false>, CsfFused::SMEM, 0},
                                        {0, true, k_csf_fused<true>, CsfFused::SMEM, 0},
                                        {1, false, k_csf_staged<7, false>, CsfStaged<7>::SMEM, 8},
                                        {2, false, k_csf_staged<3, true>, CsfStaged<3>::SMEM, 8}};

// the switches' kernel (LBM_CSF_PIPE counts only for k_csf_fused)
static const CsfKernel* csf_pick_kernel(int staged, bool pipe)
{
  if (staged != 1 && staged != 2) staged = 0;
  else pipe = false;
  for (const CsfKernel& k : csf_kernels)
    if (k.staged == staged && k.pipe == pipe) return &k;
  return nullptr;
}

// rho_r, rho_b, u (with the stored interfacial tension), phase of the current post-stream state into the planes
static int csf_fill_planes(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  ProfScope ps(d, LBM_PROF_MOMENTS);
  const int Yi = d->g.Y - 2, w = d->cur;
  if (Yi > 0)
  {
    dim3 grid(cdiv(Yi, 256), d->g.Xl);
    k_csf_moments_interior<MODE_PULL><<<grid, 256, 0, d->stream>>>(d->buf[0][w], d->buf[1][w], d->g, tp->mg, tp->mom, tp->aux, tp->p);
    d->launches++;
  }
  if (d->nb > 0)
  {
    k_csf_moments_listed<MODE_PULL><<<cdiv(d->nb, 128), 128, 0, d->stream>>>(d->buf[0][w], d->buf[1][w], d->g, tp->mg, tp->mom, tp->aux,
                                                                            tp->p, table_of(d));
    d->launches++;
  }
  LBM_CUDA(cudaGetLastError());
  tp->planes_full = true;
  return LBM_OK;
}

template <int MODE>
static int csf_launch_collide(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  const int s = d->cur, t = d->cur ^ 1, Yi = d->g.Y - 2;
  if (Yi > 0)
  {
    ProfScope ps(d, LBM_PROF_INTERIOR);
    const int rpb = tp->rpb_override > 0 ? tp->rpb_override : 64;
    dim3 grid(cdiv(Yi, CsfRing::USEFUL), cdiv(d->g.Xl, rpb));
    k_csf_collide_ring<MODE><<<grid, TPF_NT, CsfRing::SMEM, d->stream>>>(d->buf[0][s], d->buf[1][s], d->buf[0][t], d->buf[1][t], d->g,
                                                                        tp->mg, tp->mom, tp->aux, tp->p, rpb);
    d->launches++;
  }
  if (d->nb > 0)
  {
    ProfScope ps(d, LBM_PROF_BOUNDARY);
    k_csf_collide_listed<MODE><<<cdiv(d->nb, 128), 128, 0, d->stream>>>(d->buf[0][s], d->buf[1][s], d->buf[0][t], d->buf[1][t], d->g, tp->mg,
                                                                       tp->mom, tp->aux, tp->aux, tp->p, table_of(d));
    d->launches++;
  }
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

// The step in three phases; slabs put a two-row halo between them (normals differentiate the phase field, the
// curvature differentiates the normals: together the 4-row reach of SURVEY §8(f) rank 2):
//   moments   (pull)  rho_k, u (with the stored Fs), phase -> planes, columns padded      | halo: 5 moment planes
//   normals           global edge rows padded, n = -grad / (1e-20 + |grad|), columns padded | halo: n_x, n_y
//   collide           global edge rows of n padded, K, Fs, collision                        | ghost rows of the populations
static int csf_phase_moments(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  if (!d->post_stream && !tp->planes_full) LBM_TRY(csf_fill_planes(d));  // (post-stream state: the import's planes, the caller's u)
  ProfScope ps(d, LBM_PROF_MOMENTS);
  k_tp_pad_cols<<<cdiv(d->g.Xl, 128), 128, 0, d->stream>>>(tp->mom, d->g, tp->mg, M_COUNT, 0, d->g.Xl);
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

static int csf_phase_normals(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  ProfScope ps(d, LBM_PROF_MOMENTS);
  const int lo = d->cfg.x0 == 0, hi = d->cfg.x1 == d->cfg.X;
  k_tp_pad_rows<<<cdiv(d->g.Y + 4, 128), 128, 0, d->stream>>>(tp->mom, d->g, tp->mg, lo, hi, M_COUNT);
  const long long N = (long long)d->g.Xl * d->g.Y;
  k_csf_normals<<<cdiv(N, 256), 256, 0, d->stream>>>(tp->mom, tp->aux, d->g, tp->mg);
  k_tp_pad_cols<<<cdiv(d->g.Xl, 128), 128, 0, d->stream>>>(tp->aux, d->g, tp->mg, 2, 0, d->g.Xl);
  d->launches += 3;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

static int csf_phase_collide(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  {
    ProfScope ps(d, LBM_PROF_MOMENTS);
    const int lo = d->cfg.x0 == 0, hi = d->cfg.x1 == d->cfg.X;
    k_tp_pad_rows<<<cdiv(d->g.Y + 4, 128), 128, 0, d->stream>>>(tp->aux, d->g, tp->mg, lo, hi, 2);
    d->launches++;
  }
  if (d->post_stream) LBM_TRY(csf_launch_collide<MODE_LOCAL>(d));
  else LBM_TRY(csf_launch_collide<MODE_PULL>(d));
  d->cur ^= 1;
  d->post_stream = false;
  tp->planes_full = false;
  return LBM_OK;
}

// ---- single-pass step (LBM_CSF_FUSED=1)
// flags and node lists: which rows / nodes keep their moments and normals in the planes (see k_csf_fused)
static int csf_build_lists(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  if (!tp->csf_lists_dirty) return LBM_OK;
  const int Xl = d->g.Xl, Y = d->g.Y;
  std::vector<unsigned char> near2(Xl, 0), near4(Xl, 0);
  auto mark = [&](std::vector<unsigned char>& v, int x) { if (x >= 0 && x < Xl) v[x] = 1; };
  // the replicate padding of the normals copies rows 0 and Xl-1 (global edge), and rows 0, 1 / Xl-2, Xl-1 travel to the
  // neighbouring slab as its normal halo (ring): their own normals need the phase of two more rows each way
  for (int x : {0, 1, Xl - 2, Xl - 1}) mark(near2, x);
  for (int x : {0, 1, 2, 3, Xl - 4, Xl - 3, Xl - 2, Xl - 1}) mark(near4, x);
  // listed nodes differentiate the normals of their 5x5 neighbourhood, and those the phase of theirs
  for (int x = 0; x < Xl && x < (int)d->row_has_listed.size(); x++)
    if (d->row_has_listed[x])
      for (int k = -4; k <= 4; k++)
      {
        mark(near4, x + k);
        if (k >= -2 && k <= 2) mark(near2, x + k);
      }
  std::vector<unsigned char> flags(Xl);
  std::vector<int> list4, list2;
  for (int x = 0; x < Xl; x++)
  {
    flags[x] = (unsigned char)((near4[x] ? 1 : 0) | (near2[x] ? 2 : 0));
    for (int y = 1; y <= Y - 2; y++)
      if (near4[x] || y <= 4 || y >= Y - 5) list4.push_back(x * Y + y);   // the edge columns 0, Y-1 are listed nodes
    for (int y = 0; y <= Y - 1; y++)
      if (near2[x] || y <= 2 || y >= Y - 3) list2.push_back(x * Y + y);
  }
  cudaFree(tp->d_csf_flags); cudaFree(tp->d_csf_list4); cudaFree(tp->d_csf_list2);
  tp->d_csf_flags = nullptr; tp->d_csf_list4 = nullptr; tp->d_csf_list2 = nullptr;
  LBM_CUDA(cudaMalloc(&tp->d_csf_flags, Xl));
  LBM_CUDA(cudaMemcpy(tp->d_csf_flags, flags.data(), Xl, cudaMemcpyHostToDevice));
  tp->n_csf_list4 = (int)list4.size();
  tp->n_csf_list2 = (int)list2.size();
  LBM_CUDA(cudaMalloc(&tp->d_csf_list4, sizeof(int) * std::max<size_t>(list4.size(), 1)));
  LBM_CUDA(cudaMalloc(&tp->d_csf_list2, sizeof(int) * std::max<size_t>(list2.size(), 1)));
  LBM_CUDA(cudaMemcpy(tp->d_csf_list4, list4.data(), sizeof(int) * list4.size(), cudaMemcpyHostToDevice));
  LBM_CUDA(cudaMemcpy(tp->d_csf_list2, list2.data(), sizeof(int) * list2.size(), cudaMemcpyHostToDevice));
  tp->csf_lists_dirty = false;
  tp->rows_per_block = 0;
  return LBM_OK;
}

static bool csf_can_fuse(const lbm_domain* d)
{
  // monolithic domains and the slabs of an NCCL ring (two 2-row halos between the pre-pass stages, like the three-pass
  // step) or of a linked group (tp_step_group interleaves the same three stages)
  const bool whole = d->cfg.x0 == 0 && d->cfg.x1 == d->cfg.X, linked = d->link_lo || d->link_hi;
  return d->tp->csf_fused && !d->post_stream && (whole || comm_active(d) || linked) && d->g.Xl >= 8 && d->g.Y >= 12;
}

// the three stages of the single-pass step; between them the slabs of a ring / of a linked group swap two plane rows
static int csf_fused_moments(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  LBM_TRY(csf_build_lists(d));
  ProfScope ps(d, LBM_PROF_MOMENTS);
  const int s = d->cur;
  // pre-pass: the thin part of the planes that stays authoritative, from the stored post-collision state
  if (tp->n_csf_list4 > 0)
    k_csf_moments_nodes<<<cdiv(tp->n_csf_list4, 128), 128, 0, d->stream>>>(d->buf[0][s], d->buf[1][s], d->g, tp->mg, tp->mom, tp->aux,
                                                                          tp->p, tp->d_csf_list4, tp->n_csf_list4);
  if (d->nb > 0)
    k_csf_moments_listed<MODE_PULL><<<cdiv(d->nb, 128), 128, 0, d->stream>>>(d->buf[0][s], d->buf[1][s], d->g, tp->mg, tp->mom, tp->aux,
                                                                            tp->p, table_of(d));
  const int lo = d->cfg.x0 == 0, hi = d->cfg.x1 == d->cfg.X;  // replicate at the global edges only
  k_tp_pad_cols<<<cdiv(d->g.Xl, 128), 128, 0, d->stream>>>(tp->mom, d->g, tp->mg, M_COUNT, 0, d->g.Xl);
  k_tp_pad_rows<<<cdiv(d->g.Y + 4, 128), 128, 0, d->stream>>>(tp->mom, d->g, tp->mg, lo, hi, M_COUNT);
  d->launches += 4;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

static int csf_fused_normals(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  ProfScope ps(d, LBM_PROF_MOMENTS);
  const int lo = d->cfg.x0 == 0, hi = d->cfg.x1 == d->cfg.X;
  k_csf_normals_nodes<<<cdiv(tp->n_csf_list2, 128), 128, 0, d->stream>>>(tp->mom, tp->aux, d->g, tp->mg, tp->d_csf_list2, tp->n_csf_list2);
  k_tp_pad_cols<<<cdiv(d->g.Xl, 128), 128, 0, d->stream>>>(tp->aux, d->g, tp->mg, 2, 0, d->g.Xl);
  k_tp_pad_rows<<<cdiv(d->g.Y + 4, 128), 128, 0, d->stream>>>(tp->aux, d->g, tp->mg, lo, hi, 2);
  d->launches += 3;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

static int csf_fused_collide(lbm_domain* d)
{
  TwoPhaseState* tp = d->tp;
  const int s = d->cur, t = d->cur ^ 1, Yi = d->g.Y - 2;
  if (Yi > 0)
  {
    ProfScope ps(d, LBM_PROF_INTERIOR);
    const int strips = cdiv(Yi, CsfFused::USEFUL), rpb = band_rows(d, strips, *tp->csf_kernel);
    dim3 grid(strips, cdiv(d->g.Xl, rpb));
    auto k = tp->csf_kernel->kernel;
    k<<<grid, TPF_NT, tp->csf_kernel->smem, d->stream>>>(d->buf[0][s], d->buf[1][s], d->buf[0][t], d->buf[1][t], d->g, tp->mg, tp->mom, tp->aux,
                                                         tp->aux_next, tp->p, tp->d_csf_flags, rpb);
    d->launches++;
  }
  if (d->nb > 0)
  {
    ProfScope ps(d, LBM_PROF_BOUNDARY);
    k_csf_collide_listed<MODE_PULL><<<cdiv(d->nb, 128), 128, 0, d->stream>>>(d->buf[0][s], d->buf[1][s], d->buf[0][t], d->buf[1][t], d->g,
                                                                            tp->mg, tp->mom, tp->aux, tp->aux_next, tp->p, table_of(d));
    d->launches++;
  }
  LBM_CUDA(cudaGetLastError());
  d->cur ^= 1;
  d->post_stream = false;
  tp->planes_full = false;
  return LBM_OK;
}

// the interfacial tension just written is what the next step (and the getters) read.  Its own call: in a linked group a
// neighbour still copies this step's NORMAL rows out of `aux` after this slab's collision has been enqueued.
static void csf_fused_swap(lbm_domain* d) { std::swap(d->tp->aux, d->tp->aux_next); }

// ---- one two-phase step as three stages.  A stage takes two halo rows of `nplanes` planes of `halo` across every cut,
// then runs `phase`.  tp_step runs the stages back to back on one slab (NCCL halos); tp_step_group runs each stage on every
// linked slab before the next, ordering every cross-slab read by events on the slabs' streams: a stage waits for the
// neighbours' `wait` event, then records `done`.
//   MRTCG / RK:  pre (waits until the neighbours have finished reading this slab's plane rows in the step before) ->
//                moment halo (waits for the neighbours' pre) -> main
//   CSF:         moments -> moment halo (waits for the neighbours' moments), normals -> normal halo (waits for the
//                neighbours' normals), collide.  A slab's next moments pass comes after its wait for the neighbours'
//                collision (ev_stage, before the ghost rows), by which time they have finished copying rows out of its planes.
struct TpStage
{
  cudaEvent_t lbm_domain::*wait;  // (nullptr: none)
  double* TwoPhaseState::*halo;   // (nullptr: none)
  int nplanes;
  int (*phase)(lbm_domain*);      // (nullptr: none)
  cudaEvent_t lbm_domain::*done;
};
struct TpSchedule
{
  TpStage stage[3];
  bool swap_aux;               // single-pass CSF: the aux sets swap after the collision of every slab (csf_fused_swap)
  bool import_exchanged;       // MRTCG / RK: an import exchanges the planes it fills, so tp_step skips the halo of the
                               // step after it (and times the others as moments work)
};
static const TpSchedule tp_schedule_mrtcg_rk = {{{&lbm_domain::ev_packet, nullptr, 0, tp_phase_pre, &lbm_domain::ev_ready},
                                                 {&lbm_domain::ev_ready, &TwoPhaseState::mom, M_COUNT, nullptr, &lbm_domain::ev_packet},
                                                 {nullptr, nullptr, 0, tp_phase_main, &lbm_domain::ev_stage}},
                                                false, true};
static const TpSchedule tp_schedule_csf_fused = {{{nullptr, nullptr, 0, csf_fused_moments, &lbm_domain::ev_ready},
                                                  {&lbm_domain::ev_ready, &TwoPhaseState::mom, M_COUNT, csf_fused_normals, &lbm_domain::ev_packet},
                                                  {&lbm_domain::ev_packet, &TwoPhaseState::aux, 2, csf_fused_collide, &lbm_domain::ev_stage}},
                                                 true, false};
static const TpSchedule tp_schedule_csf_three = {{{nullptr, nullptr, 0, csf_phase_moments, &lbm_domain::ev_ready},
                                                  {&lbm_domain::ev_ready, &TwoPhaseState::mom, M_COUNT, csf_phase_normals, &lbm_domain::ev_packet},
                                                  {&lbm_domain::ev_packet, &TwoPhaseState::aux, 2, csf_phase_collide, &lbm_domain::ev_stage}},
                                                 false, false};

// the stages of the next step of slabs ds[0 .. n): the same for all of them (CSF: single pass on all slabs or none, since
// the halo rows a slab sends must be the ones its neighbour's stage expects)
static const TpSchedule& tp_schedule(lbm_domain* const* ds, int n)
{
  if (ds[0]->tp->model != TP_CSF) return tp_schedule_mrtcg_rk;
  bool fuse = true;
  for (int i = 0; i < n; i++) fuse = fuse && csf_can_fuse(ds[i]);
  return fuse ? tp_schedule_csf_fused : tp_schedule_csf_three;
}

int tp_step(lbm_domain* d)
{
  const TpSchedule& sc = tp_schedule(&d, 1);
  // a three-pass step out of an import does not swap the aux sets while it flips the population buffers: captured step
  // pairs (lbm_use_graph) hold the old pairing of the two.  (Never reached inside a capture: those start in steady state.)
  if (&sc == &tp_schedule_csf_three && d->tp->csf_fused && d->post_stream) drop_graphs(d);
  for (const TpStage& st : sc.stage)
  {
    // the halos: NCCL ring (rows 0, 1 / Xl-2, Xl-1 to the neighbours); nothing on a single slab
    if (st.halo && !sc.import_exchanged) LBM_TRY(comm_exchange_planes(d, d->tp->*st.halo, st.nplanes));
    else if (st.halo && !d->post_stream)
    {
      ProfScope ps(d, LBM_PROF_MOMENTS);
      LBM_TRY(comm_exchange_planes(d, d->tp->*st.halo, st.nplanes));
    }
    if (st.phase) LBM_TRY(st.phase(d));
  }
  if (sc.swap_aux) csf_fused_swap(d);
  // the next step pulls from the buffer just written: its ghost rows
  ProfScope ps(d, LBM_PROF_GHOST);
  if (comm_active(d)) return comm_exchange(d, d->cur, d->stream);
  return wrap_ghost_rows_local(d, d->cur, d->stream);
}

// linked two-phase slabs in lock step (lbm_step_group)
int tp_step_group(lbm_domain* const* ds, int n, int n_steps)
{
  const TpStage& first = tp_schedule(ds, n).stage[0];
  for (int i = 0; i < n; i++)
  {
    LBM_CUDA(on(ds[i]));
    LBM_CUDA(cudaEventRecord(ds[i]->ev_begin, ds[i]->stream));
    if (first.wait) LBM_CUDA(cudaEventRecord(ds[i]->*first.wait, ds[i]->stream));  // MRTCG / RK: "nobody is reading my planes"
  }
  for (int s = 0; s < n_steps; s++)
  {
    const TpSchedule& sc = tp_schedule(ds, n);
    for (const TpStage& st : sc.stage)
      for (int i = 0; i < n; i++)
      {
        lbm_domain* d = ds[i];
        LBM_CUDA(on(d));
        if (st.wait) LBM_TRY(wait_linked(d, d->stream, st.wait));
        if (st.halo) LBM_TRY(tp_link_halo_planes(d, st.halo, st.nplanes));
        if (st.phase) LBM_TRY(st.phase(d));
        LBM_CUDA(cudaEventRecord(d->*st.done, d->stream));
      }
    if (sc.swap_aux)
      for (int i = 0; i < n; i++) csf_fused_swap(ds[i]);
    for (int i = 0; i < n; i++)
    {
      lbm_domain* d = ds[i];
      LBM_CUDA(on(d));
      LBM_TRY(wait_linked(d, d->stream, &lbm_domain::ev_stage));
      ProfScope ps(d, LBM_PROF_GHOST);
      if (d->link_lo || d->link_hi) LBM_TRY(link_exchange(d, d->cur, d->stream));
      else LBM_TRY(wrap_ghost_rows_local(d, d->cur, d->stream));
    }
  }
  for (int i = 0; i < n; i++)
  {
    LBM_CUDA(on(ds[i]));
    LBM_CUDA(cudaEventRecord(ds[i]->ev_end, ds[i]->stream));
  }
  return LBM_OK;
}

// (here, below both kernel tables: the switches are read once, and every table entry gets its attributes)
int tp_create(lbm_domain* d)
{
  TwoPhaseState* tp = new TwoPhaseState();
  d->tp = tp;
  tp->model = d->cfg.model == LBM_MODEL_MRTCG ? TP_MRTCG : (d->cfg.model == LBM_MODEL_MRT_CSF ? TP_CSF : TP_RK);
  tp->mg.pm = ((d->g.Y + 4 + 15) / 16) * 16;
  tp->mg.mplane = (long long)(d->g.Xl + 4) * tp->mg.pm;
  const size_t bytes = sizeof(double) * M_COUNT * tp->mg.mplane;
  LBM_CUDA(cudaMalloc(&tp->mom, bytes));
  LBM_CUDA(cudaMemset(tp->mom, 0, bytes));
  TpParams& p = tp->p;
  const lbm_config& c = d->cfg;
  if (!(c.red.rho_0 > 0.0) || !(c.blue.rho_0 > 0.0) || !(c.delta > 0.0))
  {
    set_error("two-phase model: red/blue initial_density and delta must be positive");
    return LBM_ERR_INVALID;
  }
  tp_fill_params(c, (TpModel)tp->model, p);
  if (tp->model == TP_CSF)
  {
    const size_t ab = sizeof(double) * 4 * tp->mg.mplane;
    LBM_CUDA(cudaMalloc(&tp->aux, ab));
    LBM_CUDA(cudaMemset(tp->aux, 0, ab));
    int staged = 2;
    bool pipe = false;
    if (const char* e = getenv("LBM_CSF_FUSED")) tp->csf_fused = atoi(e) != 0;
    if (const char* e = getenv("LBM_CSF_PIPE")) pipe = atoi(e) != 0;
    if (const char* e = getenv("LBM_CSF_STAGED")) staged = atoi(e);
    tp->csf_kernel = csf_pick_kernel(staged, pipe);
    if (tp->csf_fused)
    {
      LBM_CUDA(cudaMalloc(&tp->aux_next, ab));
      LBM_CUDA(cudaMemset(tp->aux_next, 0, ab));
    }
  }
  else
  {
    // MRTCG (H = 2): the stash frees shared memory for a third block per SM (+17 %).  RK (H = 1) runs two blocks either way
    // and is 1 % faster with its two resident rows left in the stage slots
    bool pipe = true, staged = true, stash = tp->model == TP_MRTCG;
    int stages = 0;
    if (const char* e = getenv("LBM_TP_PIPE")) pipe = atoi(e) != 0;
    if (const char* e = getenv("LBM_TP_STAGED")) staged = atoi(e) != 0;
    if (const char* e = getenv("LBM_TP_NS")) stages = atoi(e);
    if (const char* e = getenv("LBM_TP_STASH")) stash = atoi(e) != 0;
    tp->kernel = tp_pick_kernel(tp->model, staged, stash, stages, pipe);
  }
  // every instantiation a switch can select, whichever this domain runs
  auto set_attributes = [](const auto& table) -> int {
    for (const auto& k : table)
    {
      LBM_CUDA(cudaFuncSetAttribute(k.kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem));
      if (k.staged) LBM_CUDA(cudaFuncSetAttribute(k.kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    }
    return LBM_OK;
  };
  LBM_TRY(set_attributes(tp_kernels));
  LBM_TRY(set_attributes(csf_kernels));
  LBM_CUDA(cudaFuncSetAttribute(k_csf_collide_ring<MODE_LOCAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CsfRing::SMEM));
  LBM_CUDA(cudaFuncSetAttribute(k_csf_collide_ring<MODE_PULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CsfRing::SMEM));
  if (const char* e = getenv("LBM_TP_RPB")) tp->rpb_override = atoi(e);
  if (const char* e = getenv("LBM_TP_OVERLAP")) tp->ring_overlap = atoi(e) != 0;  // (off by default: see tp_steps_ring)
  return LBM_OK;
}

// ================================================================================================
// Diagnostic fields of driver 17 (test/rk_static_droplet_test.cpp:546-600): interface normal with the driver's
// 0.1 max|grad| cut, local curvature, interfacial tension, eta, kappa, 1/tau, and the red colour's omega1 / omega2.
// Functions of the current post-stream state only; nothing here feeds the step (SURVEY §8(a) row a14).
// Planes in the moment-plane geometry: D_NX, D_NY (padded: the curvature differentiates them).
// ================================================================================================
// grad(phase) (the driver's swapped pair: [0] along axis 1, [1] along axis 0), its norm, and the global maximum of the
// norm: non-negative doubles order like their bit patterns, so one atomicMax on the bits per block does it
__global__ void __launch_bounds__(256)
k_rk_diag_grad(const double* __restrict__ mom, const SlabGeom g, const MomGeom mg, const TpParams p, double* __restrict__ grad,
               double* __restrict__ norm, unsigned long long* __restrict__ gmax_bits)
{
  __shared__ double smax[256];
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  double gn = 0.0;
  if (n < (long long)g.Xl * g.Y)
  {
    const int x = (int)(n / g.Y), y = (int)(n % g.Y);
    TpStencil st;
    tp_stencil_global<TP_RK>(p, mom, mg, x, y, st);
    gn = sqrt(st.gx * st.gx + st.gy * st.gy);
    grad[2 * n] = st.gx;
    grad[2 * n + 1] = st.gy;
    norm[n] = gn;
  }
  smax[threadIdx.x] = gn == gn ? gn : 0.0;  // a NaN does not take part (torch's max would propagate it; the cut is then moot)
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1)
  {
    if ((int)threadIdx.x < w) smax[threadIdx.x] = fmax(smax[threadIdx.x], smax[threadIdx.x + w]);
    __syncthreads();
  }
  if (threadIdx.x == 0) atomicMax(gmax_bits, (unsigned long long)__double_as_longlong(smax[0]));
}

// n = -normalize(grad where |grad| > 0.1 max|grad|, else 0), F::normalize's eps = 1e-12 (:559-567)
__global__ void __launch_bounds__(256)
k_rk_diag_normal(const double* __restrict__ grad, const double* __restrict__ norm, const SlabGeom g, const MomGeom mg,
                 const unsigned long long* __restrict__ gmax_bits, double* __restrict__ nplanes)
{
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (long long)g.Xl * g.Y) return;
  const int x = (int)(n / g.Y), y = (int)(n % g.Y);
  const double gmax = __longlong_as_double((long long)*gmax_bits);
  const bool cut = norm[n] <= 0.1 * gmax;
  const double cx = cut ? 0.0 : grad[2 * n], cy = cut ? 0.0 : grad[2 * n + 1];
  const double den = fmax(sqrt(cx * cx + cy * cy), 1e-12);
  const long long k = mom_off(mg, x, y);
  nplanes[k] = -(cx / den);
  nplanes[mg.mplane + k] = -(cy / den);
}

struct RkDiagOut  // device AoS buffers in the reference's tensor layouts; nullptr = not wanted
{
  double *K, *Fs, *eta, *kappa, *rparams, *omega1, *omega2, *omega3;
};

__global__ void __launch_bounds__(128)
k_rk_diag_final(const double* __restrict__ mom, const double* __restrict__ nplanes, const double* __restrict__ grad,
                const double* __restrict__ norm, const double* __restrict__ r_aos, const SlabGeom g, const MomGeom mg,
                const TpParams p, double sigma, RkDiagOut o)
{
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (long long)g.Xl * g.Y) return;
  const int x = (int)(n / g.Y), y = (int)(n % g.Y);
  const long long k = mom_off(mg, x, y);
  // eval_local_curvature (:440-446) with the driver's 3x3 kernels: x(.) along axis 1, y(.) along axis 0
  double x_nx = 0.0, y_nx = 0.0, x_ny = 0.0, y_ny = 0.0;
#pragma unroll
  for (int a = -1; a <= 1; a++)
#pragma unroll
    for (int b = -1; b <= 1; b++)
    {
      const double vx = nplanes[k + (long long)a * mg.pm + b], vy = nplanes[mg.mplane + k + (long long)a * mg.pm + b];
      const double wa = a == 0 ? 1.0 / 9.0 : 1.0 / 36.0, wb = b == 0 ? 1.0 / 9.0 : 1.0 / 36.0;
      if (b != 0) { x_nx += (3.0 * (wa * (double)b)) * vx; x_ny += (3.0 * (wa * (double)b)) * vy; }
      if (a != 0) { y_nx += (3.0 * (wb * (double)a)) * vx; y_ny += (3.0 * (wb * (double)a)) * vy; }
    }
  const double nx = nplanes[k], ny = nplanes[mg.mplane + k];
  const double K = nx * ny * (y_nx + x_ny) - (nx * nx) * y_ny - (ny * ny) * x_nx;
  const double gx = grad[2 * n], gy = grad[2 * n + 1], gn = norm[n];
  const double Fsx = 0.5 * sigma * K * gx, Fsy = 0.5 * sigma * K * gy;  // :572
  const double rr = mom[M_RR * mg.mplane + k], rb = mom[M_RB * mg.mplane + k];
  const double ux = mom[M_UX * mg.mplane + k], uy = mom[M_UY * mg.mplane + k], ph = mom[M_PH * mg.mplane + k];
  const double relax = 1.0 / relax_eval(p, ph);  // :587-589
  if (o.K) o.K[n] = K;
  if (o.Fs) { o.Fs[2 * n] = Fsx; o.Fs[2 * n + 1] = Fsy; }
  if (o.rparams) o.rparams[n] = relax;
  const double uu = ux * ux + uy * uy;
  const double kap = rr * rb / (rr + rb);
  const double ign2 = 1.0 / (1e-20 + gn * gn);
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    const double ex = (double)CX(q), ey = (double)CY(q);
    const double ue = ux * ex + uy * ey;
    // eval_eta (:398-413): ((ics2 (E - u) + ics2 (u.E) E) . Fs) W with ics2 = 3 in both terms, as written
    if (o.eta) o.eta[9 * n + q] = ((3.0 * (ex - ux) + 3.0 * (ue * ex)) * Fsx + (3.0 * (ey - uy) + 3.0 * (ue * ey)) * Fsy) * W(q);
    // eval_kappa (:415-438): rho_r rho_b / rho * ((-n) . E) W
    if (o.kappa) o.kappa[9 * n + q] = kap * (((-nx) * ex + (-ny) * ey) * W(q));
    const double o1 = relax * (tp_feq<TP_RK>(q, rr, p.r_phi, p.r_eta, ux, uy, uu) - r_aos[9 * n + q]);  // :255-262
    const double fe = gx * ex + gy * ey;
    const double o2 = ((0.5 * p.r_A) * gn) * (((fe * fe) * ign2) * W(q) - BQ(q));  // :239-245
    if (o.omega1) o.omega1[9 * n + q] = o1;
    if (o.omega2) o.omega2[9 * n + q] = o2;
    if (o.omega3) o.omega3[9 * n + q] = o1 + o2;  // :232-236
  }
}

}  // namespace lbm

using namespace lbm;

extern "C"
{

int lbm_get_phase(lbm_domain* d, double* phase, double* rho_r, double* rho_b)
{
  if (!d || !d->tp) { set_error("lbm_get_phase: not a two-phase domain"); return LBM_ERR_INVALID; }
  if (!d->have_state) { set_error("lbm_get_phase: no state"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_TRY(stage_fields(d, 0));
  const long long N = (long long)d->g.Xl * d->g.Y;
  const double* st = d->d_mom_out;
  if (phase) LBM_CUDA(cudaMemcpyAsync(phase, st + 3 * N, sizeof(double) * N, cudaMemcpyDeviceToHost, d->stream));
  if (rho_r) LBM_CUDA(cudaMemcpyAsync(rho_r, st + 4 * N, sizeof(double) * N, cudaMemcpyDeviceToHost, d->stream));
  if (rho_b) LBM_CUDA(cudaMemcpyAsync(rho_b, st + 5 * N, sizeof(double) * N, cudaMemcpyDeviceToHost, d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  return LBM_OK;
}

// interf_tension of the last step, {X,Y,2} (the driver snapshots it as gradx / grady, mrt_rayleigh_taylor.cpp:485-486)
int lbm_get_interfacial_tension(lbm_domain* d, double* Fs_aos)
{
  if (!d || !d->tp || d->tp->model != TP_CSF || !Fs_aos) { set_error("lbm_get_interfacial_tension: LBM_MODEL_MRT_CSF domains only"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  const MomGeom mg = d->tp->mg;
  const int Xl = d->g.Xl, Y = d->g.Y;
  std::vector<double> fx((size_t)mg.mplane), fy((size_t)mg.mplane);
  LBM_CUDA(cudaMemcpy(fx.data(), d->tp->aux + (long long)A_FX * mg.mplane, sizeof(double) * mg.mplane, cudaMemcpyDeviceToHost));
  LBM_CUDA(cudaMemcpy(fy.data(), d->tp->aux + (long long)A_FY * mg.mplane, sizeof(double) * mg.mplane, cudaMemcpyDeviceToHost));
  for (int x = 0; x < Xl; x++)
    for (int y = 0; y < Y; y++)
    {
      const size_t k = (size_t)(x + 2) * mg.pm + (y + 2);
      Fs_aos[2 * ((size_t)x * Y + y)] = fx[k];
      Fs_aos[2 * ((size_t)x * Y + y) + 1] = fy[k];
    }
  return LBM_OK;
}

int lbm_rk_diagnostics(lbm_domain* d, double sigma, const lbm_rk_diag* out)
{
  if (!d || !d->tp || d->tp->model != TP_RK || !out) { set_error("lbm_rk_diagnostics: LBM_MODEL_RK domains only"); return LBM_ERR_INVALID; }
  if (!d->have_state || !d->committed) { set_error("lbm_rk_diagnostics: no state or boundary rules not committed"); return LBM_ERR_INVALID; }
  const bool slab = d->cfg.x0 != 0 || d->cfg.x1 != d->cfg.X;
  if (slab && !comm_active(d))
  {
    // the normal's cut needs max|grad| over the whole grid and the curvature a halo of the normal planes: over the NCCL
    // ring both are exchanges (every rank calls this function); linked slabs of one process have no such collective
    set_error("lbm_rk_diagnostics: monolithic domains or the ranks of an lbm_comm_init ring only (this slab holds rows %d..%d of %d)",
              d->cfg.x0, d->cfg.x1, d->cfg.X);
    return LBM_ERR_UNSUPPORTED;
  }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  TwoPhaseState* tp = d->tp;
  const long long N = (long long)d->g.Xl * d->g.Y;
  const MomGeom mg = tp->mg;
  LBM_TRY(tp_fill_planes(d));
  LBM_TRY(tp_pad(d));
  LBM_TRY(comm_exchange_moments(d));  // ring: the two ghost rows of the moment planes at the cuts
  LBM_TRY(ensure_aos_scratch(d));
  LBM_TRY(tp_export(d));  // post-stream populations (adv_f) of both colours in the reference layout
  // one scratch allocation per call: this is a diagnostic path, not the time loop
  const size_t n_planes = 2 * (size_t)mg.mplane, n_nodes = (size_t)N * (2 + 1 + 1 + 2 + 9 + 9 + 1 + 27);
  double* scratch = nullptr;
  unsigned long long* gmax = nullptr;
  LBM_CUDA(cudaMalloc(&scratch, (n_planes + n_nodes) * sizeof(double)));
  if (cudaMalloc(&gmax, sizeof(unsigned long long)) != cudaSuccess) { cudaFree(scratch); set_error("lbm_rk_diagnostics: out of device memory"); return LBM_ERR_CUDA; }
  double* npl = scratch;
  double* grad = npl + n_planes;
  double* norm = grad + 2 * N;
  RkDiagOut o;
  o.K = norm + N; o.Fs = o.K + N; o.eta = o.Fs + 2 * N; o.kappa = o.eta + 9 * N; o.rparams = o.kappa + 9 * N;
  o.omega1 = o.rparams + N; o.omega2 = o.omega1 + 9 * N; o.omega3 = o.omega2 + 9 * N;
  int rc = LBM_OK;
  auto run = [&]() -> int {
    LBM_CUDA(cudaMemsetAsync(gmax, 0, sizeof(unsigned long long), d->stream));
    k_rk_diag_grad<<<cdiv(N, 256), 256, 0, d->stream>>>(tp->mom, d->g, mg, tp->p, grad, norm, gmax);
    LBM_TRY(comm_allreduce_max(d, reinterpret_cast<double*>(gmax)));  // grad_norm.max() over the whole grid (SURVEY §8(e))
    k_rk_diag_normal<<<cdiv(N, 256), 256, 0, d->stream>>>(grad, norm, d->g, mg, gmax, npl);
    k_tp_pad_cols<<<cdiv(d->g.Xl, 128), 128, 0, d->stream>>>(npl, d->g, mg, 2, 0, d->g.Xl);
    k_tp_pad_rows<<<cdiv(d->g.Y + 4, 128), 128, 0, d->stream>>>(npl, d->g, mg, d->cfg.x0 == 0, d->cfg.x1 == d->cfg.X, 2);
    LBM_TRY(comm_exchange_planes(d, npl, 2));  // the curvature differentiates the normal across the cuts
    k_rk_diag_final<<<cdiv(N, 128), 128, 0, d->stream>>>(tp->mom, npl, grad, norm, d->d_aos[0], d->g, mg, tp->p, sigma, o);
    d->launches += 5;
    LBM_CUDA(cudaGetLastError());
    auto back = [&](double* host, const double* dev, long long count) -> int {
      if (host) LBM_CUDA(cudaMemcpyAsync(host, dev, sizeof(double) * count, cudaMemcpyDeviceToHost, d->stream));
      return LBM_OK;
    };
    LBM_TRY(back(out->grad, grad, 2 * N));
    LBM_TRY(back(out->norm, norm, N));
    LBM_TRY(back(out->K, o.K, N));
    LBM_TRY(back(out->Fs, o.Fs, 2 * N));
    LBM_TRY(back(out->eta, o.eta, 9 * N));
    LBM_TRY(back(out->kappa, o.kappa, 9 * N));
    LBM_TRY(back(out->rparams, o.rparams, N));
    LBM_TRY(back(out->omega1, o.omega1, 9 * N));
    LBM_TRY(back(out->omega2, o.omega2, 9 * N));
    LBM_TRY(back(out->omega3, o.omega3, 9 * N));
    LBM_CUDA(cudaStreamSynchronize(d->stream));
    if (out->n || out->phase)
    {
      // the normal and the phase live in padded planes: unpad on the host
      std::vector<double> pl(out->n ? n_planes : 0), ph(out->phase ? (size_t)mg.mplane : 0);
      if (out->n) LBM_CUDA(cudaMemcpy(pl.data(), npl, sizeof(double) * n_planes, cudaMemcpyDeviceToHost));
      if (out->phase) LBM_CUDA(cudaMemcpy(ph.data(), tp->mom + (long long)M_PH * mg.mplane, sizeof(double) * mg.mplane, cudaMemcpyDeviceToHost));
      for (int x = 0; x < d->g.Xl; x++)
        for (int y = 0; y < d->g.Y; y++)
        {
          const size_t k = (size_t)(x + 2) * mg.pm + (y + 2), n = (size_t)x * d->g.Y + y;
          if (out->n) { out->n[2 * n] = pl[k]; out->n[2 * n + 1] = pl[(size_t)mg.mplane + k]; }
          if (out->phase) out->phase[n] = ph[k];
        }
    }
    return LBM_OK;
  };
  rc = run();
  cudaFree(scratch);
  cudaFree(gmax);
  return rc;
}

int lbm_set_u(lbm_domain* d, const double* u_aos)
{
  if (!d || !d->tp || !u_aos) { set_error("lbm_set_u: not a two-phase domain / null argument"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  const long long N = (long long)d->g.Xl * d->g.Y;
  double* tmp = nullptr;
  LBM_TRY(host_staging(d, &tmp));
  LBM_CUDA(cudaMemcpyAsync(tmp, u_aos, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, d->stream));
  k_tp_write_u<<<cdiv(N, 256), 256, 0, d->stream>>>(d->tp->mom, d->g, d->tp->mg, tmp);
  d->launches++;
  int s = tp_pad(d);
  if (s == LBM_OK) s = comm_exchange_moments(d);
  cudaStreamSynchronize(d->stream);
  return s;
}

int lbm_init_two_phase(lbm_domain* d, const double* rho_r, const double* rho_b, const double* u)
{
  if (!d || !d->tp || !rho_r || !rho_b || !u) { set_error("lbm_init_two_phase: not a two-phase domain / null argument"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  const long long N = (long long)d->g.Xl * d->g.Y;
  double* tmp = nullptr;
  LBM_TRY(host_staging(d, &tmp));  // [6][N] persistent staging: rho_r, rho_b, u use 4 N of it
  LBM_CUDA(cudaMemcpyAsync(tmp, rho_r, sizeof(double) * N, cudaMemcpyHostToDevice, d->stream));
  LBM_CUDA(cudaMemcpyAsync(tmp + N, rho_b, sizeof(double) * N, cudaMemcpyHostToDevice, d->stream));
  LBM_CUDA(cudaMemcpyAsync(tmp + 2 * N, u, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, d->stream));
  if (d->tp->aux) LBM_CUDA(cudaMemsetAsync(d->tp->aux, 0, sizeof(double) * 4 * d->tp->mg.mplane, d->stream));
  with_model(d->tp, [&](auto M) {
    k_tp_init<M><<<cdiv(N, 256), 256, 0, d->stream>>>(d->buf[0][d->cur], d->buf[1][d->cur], d->g, d->tp->mg, d->tp->mom, d->tp->p, tmp, tmp + N, tmp + 2 * N);
    return LBM_OK;
  });
  d->launches++;
  int s = tp_pad(d);
  if (s == LBM_OK) s = comm_exchange_moments(d);
  cudaStreamSynchronize(d->stream);
  if (s != LBM_OK) return s;
  d->post_stream = true;
  d->have_state = true;
  d->tp->planes_full = true;
  return LBM_OK;
}

}  // extern "C"
