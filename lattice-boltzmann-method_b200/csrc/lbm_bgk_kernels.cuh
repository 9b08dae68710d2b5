// lbm_bgk_kernels.cuh — fused collide+stream kernels of the single-phase family
// (LBM_MODEL_BGK, LBM_MODEL_BGK_ADE).
//
// Storage: SoA fp64, one plane per population, plane = (Xl+2) rows x pitch columns (ghost row
// below and above the slab), two buffers per lattice.  A step reads buffer `src` and writes
// buffer `dst`; what is stored between steps is the POST-COLLISION state f_coll, so that
//   f_adve(t+1)[q](x) = f_coll(t)[q](x - c_q)         (solver::advect, src/solver.cpp:76-131)
// is a pull with aligned 128-bit stores, and every boundary rule of the reference
// ("f_adve[...] = +-f_coll[...] (+ const)", e.g. test/horizontal_poiseuille_test.cpp:146-152)
// reads the same source buffer.
//
//   k_bgk_interior  : all rows, column pairs (y, y+1) with y even and 2 <= y, y+2 <= Y-1.
//                     No masks, no wrap logic, no boundary table: 9 x 128-bit loads, the +-1
//                     column shifts done with warp shuffles, 9 x 128-bit stores per thread.
//   k_bgk_boundary  : one thread per listed node (edge columns, every node some boundary rule
//                     touches, probe nodes); table-driven gather.  Runs after the interior kernel
//                     on the same stream and overwrites what that wrote for listed nodes.
//   k_fix_copy, k_pressure_pack/apply : pre-stream rules applied to the freshly written f_coll
//                     (zero-gradient copies, pressure-periodic rows).
//   k_bgk_interior_stats / k_bgk_boundary_stats : the same two kernels (STATS = true of their bodies bgk_interior /
//                     bgk_boundary) while a statistics record is on (lbm_stats_start): they also fold the moments their
//                     collision uses into the Welford accumulators of the time-averaged fields.
#pragma once
#include "lbm_device.cuh"

namespace lbm
{

// ------------------------------------------------------------------------------------------------
// boundary tables
// ------------------------------------------------------------------------------------------------
enum OpKind : int
{
  OP_LINEAR = 0,      // coef * src[src_idx] + cst
  OP_ABB_EXTRAP = 1,  // -src[src_idx] + abb(1.5 u[j1] - 0.5 u[j2])     (aux0 = j1, aux1 = j2, boundary-node indices)
  OP_ADE_INLET = 2    // -src[src_idx] + 2 geq(u_local + w_s, cst)       (second lattice only)
};

struct BcEntry
{
  long long src;  // linear offset into the lattice's source buffer (plane offset included)
  double coef;
  double cst;
  int kind;
  int sq;  // source population (needed by the ABB / ADE formulas)
  int aux0, aux1;
};

struct BoundaryTable
{
  int n;                  // listed nodes
  const int* x;           // local row
  const int* y;           // column
  const BcEntry* ent;     // [lattice][q][n]
  double* mom_cur;        // [n][4] rho, ux, uy, C written by this launch
  const double* mom_prev; // [n][4] of the previous collide
};

struct FixEntry
{
  long long dst;  // node offsets (no plane offset)
  long long src;
  int lattice;
  int pad;
};

// ------------------------------------------------------------------------------------------------
// time-averaged moments (lbm_stats_start)
// ------------------------------------------------------------------------------------------------
// Six planes of Xl x pitch doubles, node (x, y) at x * pitch + y: the running means of rho, ux, uy, then the Welford sums
// Mxx, Myy, Mxy of the products of the deviations.  Sample k (n = k + 1) updates them in an order NumPy restates,
//   d = v - mean;  mean += d * (1 / n);  M_ab += d_a * (v_b - mean_b)
// (raw sums of u^2 would lose the fluctuation's digits next to a steady mean).  1 / n is rounded once per step by
// k_stats_tick: an fp64 division in the step kernels would call its slow-path subroutine three times per node, and the
// calls cost the listed-node kernel a stack frame.  Every node is updated by exactly one launch of a step: listed nodes by
// k_bgk_boundary, every other node by k_bgk_interior.
struct StatsClock
{
  long long count;  // steps since lbm_stats_start
  double inv_n;     // 1 / n of this step's sample, 0 when the step is no sample
};

struct StatsArgs
{
  double* acc;              // plane k at acc + k * plane
  long long plane;          // Xl * pitch
  const StatsClock* clock;  // k_stats_tick advances it after all three launches of a step
  int words;                // 32-bit words per row of `listed`
  const unsigned* listed;   // early rows only: bit y of row x is set when (x, y) is a listed node; nullptr otherwise
};

// a = (mean rho, mean ux, mean uy, Mxx, Myy, Mxy) of one node
__device__ __forceinline__ void welford(double (&a)[6], double inv_n, double rho, double ux, double uy)
{
  const double dr = rho - a[0];
  a[0] = a[0] + dr * inv_n;
  const double dx = ux - a[1];
  a[1] = a[1] + dx * inv_n;
  const double dy = uy - a[2];
  a[2] = a[2] + dy * inv_n;
  a[3] = a[3] + dx * (ux - a[1]);
  a[4] = a[4] + dy * (uy - a[2]);
  a[5] = a[5] + dx * (uy - a[2]);
}

// one node (listed-node kernel)
__device__ __forceinline__ void stats_node(const StatsArgs& s, double inv_n, long long i, double rho, double ux, double uy)
{
  double a[6];
#pragma unroll
  for (int k = 0; k < 6; k++) a[k] = s.acc[k * s.plane + i];
  welford(a, inv_n, rho, ux, uy);
#pragma unroll
  for (int k = 0; k < 6; k++) s.acc[k * s.plane + i] = a[k];
}

// ------------------------------------------------------------------------------------------------
// interior kernel
// ------------------------------------------------------------------------------------------------
struct Pair
{
  double a, b;
};

__device__ __forceinline__ Pair ld_pair(const double* __restrict__ p)
{
  const double2 v = __ldg(reinterpret_cast<const double2*>(p));
  return Pair{v.x, v.y};
}

__device__ __forceinline__ void st_pair(double* __restrict__ p, double a, double b)
{
  *reinterpret_cast<double2*>(p) = make_double2(a, b);
}

// Loads the 9 populations of nodes (x,y) and (x,y+1) as they are after streaming.
// `base` points at plane 0 of the source buffer, `o` = node_off(x, y).
template <int MODE>
__device__ __forceinline__ void load_streamed_pair(const double* __restrict__ base, const SlabGeom& g, long long o,
                                                   bool active, bool last_active, int lane, double (&fa)[9],
                                                   double (&fb)[9])
{
  if constexpr (MODE == MODE_LOCAL)
  {
    if (active)
    {
#pragma unroll
      for (int q = 0; q < 9; q++)
      {
        const Pair v = ld_pair(base + q * g.plane + o);
        fa[q] = v.a;
        fb[q] = v.b;
      }
    }
  }
  else
  {
    // aligned pair of every population at its source row; edge scalars for the lanes whose
    // shuffle partner lies in another warp
    Pair v[9];
    double edge[9];
#pragma unroll
    for (int q = 0; q < 9; q++)
    {
      const double* row = base + q * g.plane + o - (long long)CX(q) * g.pitch;
      v[q] = Pair{0.0, 0.0};
      edge[q] = 0.0;
      if (active)
      {
        v[q] = ld_pair(row);
        if (CY(q) == 1 && lane == 0) edge[q] = __ldg(row - 1);
        if (CY(q) == -1 && (lane == 31 || last_active)) edge[q] = __ldg(row + 2);
      }
    }
#pragma unroll
    for (int q = 0; q < 9; q++)
    {
      if (CY(q) == 0)
      {
        fa[q] = v[q].a;
        fb[q] = v[q].b;
      }
      else if (CY(q) == 1)
      {
        // destination (y, y+1) <- source (y-1, y)
        double left = __shfl_up_sync(0xffffffffu, v[q].b, 1);
        if (lane == 0) left = edge[q];
        fa[q] = left;
        fb[q] = v[q].a;
      }
      else
      {
        // destination (y, y+1) <- source (y+1, y+2)
        double right = __shfl_down_sync(0xffffffffu, v[q].a, 1);
        if (lane == 31 || last_active) right = edge[q];
        fa[q] = v[q].b;
        fb[q] = right;
      }
    }
  }
}

// grid: x = ceil(npairs / blockDim.x), y = number of rows in `rows` (the launch's row list: the
// "early" rows whose results feed the ghost exchange / IBM pre-pass of the next step, or the bulk)
// No minimum-blocks argument: with one, ptxas sizes every instantiation for that occupancy — (128, 1) let the BGK+IBM
// kernel grow from 76 to 126 registers and cost the cylinder workload 8 %.  For the KBC instantiation (126 registers,
// 4 blocks/SM) forcing more resident blocks was measured at 8192^2: 5 blocks (spills 224 B) 31.4 GLUPS, 6 (404 B) 24.8,
// 8 (608 B) 18.4, against 35.9 as compiled here — that collision needs its registers.
template <int MODE, int EQ, int FORCE, bool ADE, bool STATS>
__device__ __forceinline__ void
bgk_interior(const double* __restrict__ fsrc, double* __restrict__ fdst, const double* __restrict__ gsrc,
             double* __restrict__ gdst, const SlabGeom g, const BgkParams p, const int* __restrict__ rows, int npairs,
             double* __restrict__ out_f, double* __restrict__ out_g, const StatsArgs st)
{
  static_assert(!(STATS && MODE == MODE_PULL_ONLY), "a pull-only pass is no step: nothing to sample");
  const int pi = blockIdx.x * blockDim.x + threadIdx.x;
  const int x = rows[blockIdx.y];
  const int lane = threadIdx.x & 31;
  const bool active = pi < npairs;
  const bool last_active = (pi == npairs - 1);
  const int y = 2 + 2 * pi;
  const long long o = node_off(g, x, y);

  double fa[9], fb[9];
  load_streamed_pair<MODE>(fsrc, g, o, active, last_active, lane, fa, fb);

  if constexpr (MODE == MODE_PULL_ONLY)
  {
    if (p.snap_rho != nullptr)
    {
      // snapshot: moments of the post-stream state straight from the pull (no AoS detour)
      if (active)
      {
        double ra, uxa, uya, rb, uxb, uyb;
        snapshot_moments<EQ, FORCE>(fa, p, ra, uxa, uya);
        snapshot_moments<EQ, FORCE>(fb, p, rb, uxb, uyb);
        const long long n = (long long)x * g.Y + y;
        p.snap_rho[n] = ra;
        p.snap_rho[n + 1] = rb;
        p.snap_u[2 * n] = uxa;
        p.snap_u[2 * n + 1] = uya;
        p.snap_u[2 * n + 2] = uxb;
        p.snap_u[2 * n + 3] = uyb;
      }
      return;
    }
    if (active)
    {
      double* oa = out_f + ((long long)x * g.Y + y) * 9;
#pragma unroll
      for (int q = 0; q < 9; q++)
      {
        oa[q] = fa[q];
        oa[9 + q] = fb[q];
      }
    }
    if constexpr (ADE)
    {
      double ga[9], gb[9];
      load_streamed_pair<MODE>(gsrc, g, o, active, last_active, lane, ga, gb);
      if (active)
      {
        double* og = out_g + ((long long)x * g.Y + y) * 9;
#pragma unroll
        for (int q = 0; q < 9; q++)
        {
          og[q] = ga[q];
          og[9 + q] = gb[q];
        }
      }
    }
    return;
  }
  else
  {
    double rho_a, ux_a, uy_a, rho_b, ux_b, uy_b;
    bool roi_a = false, roi_b = false;
    double Fxa = 0.0, Fya = 0.0, Fxb = 0.0, Fyb = 0.0;
    if constexpr (FORCE == FORCE_IBM || FORCE == FORCE_REGION)
    {
      const int xg = x + g.xg0;
      if (active && xg >= p.roi_r0 && xg < p.roi_r1)
      {
        const int rc = p.roi_c1 - p.roi_c0;
        const long long r = (long long)(xg - p.roi_r0) * rc;
        if (y >= p.roi_c0 && y < p.roi_c1)
        {
          roi_a = true;
          Fxa = p.Fx[r + (y - p.roi_c0)];
          Fya = p.Fy[r + (y - p.roi_c0)];
        }
        if (y + 1 >= p.roi_c0 && y + 1 < p.roi_c1)
        {
          roi_b = true;
          Fxb = p.Fx[r + (y + 1 - p.roi_c0)];
          Fyb = p.Fy[r + (y + 1 - p.roi_c0)];
        }
      }
    }
    bool given = false;
    if constexpr (EQ == EQ_KBC && MODE == MODE_LOCAL)
    {
      if (p.mom_in_rho != nullptr && active)  // the caller's m0, u for the first step (lbm_set_moments)
      {
        const long long n = (long long)x * p.Y + y;
        given = true;
        rho_a = p.mom_in_rho[n]; ux_a = p.mom_in_u[2 * n]; uy_a = p.mom_in_u[2 * n + 1];
        rho_b = p.mom_in_rho[n + 1]; ux_b = p.mom_in_u[2 * n + 2]; uy_b = p.mom_in_u[2 * n + 3];
      }
    }
    bgk_collide<EQ, FORCE>(fa, p, roi_a, Fxa, Fya, rho_a, ux_a, uy_a, given);
    bgk_collide<EQ, FORCE>(fb, p, roi_b, Fxb, Fyb, rho_b, ux_b, uy_b, given);
    if (active)
    {
#pragma unroll
      for (int q = 0; q < 9; q++) st_pair(fdst + q * g.plane + o, fa[q], fb[q]);
    }
    if constexpr (STATS)
    {
      const double inv_n = st.clock->inv_n;
      if (active && inv_n != 0.0)
      {
        // a listed node of an early row: k_bgk_boundary overwrites this collision and samples the node itself
        bool skip_a = false, skip_b = false;
        if (st.listed != nullptr)
        {
          const unsigned w = st.listed[(long long)x * st.words + (y >> 5)];  // y even: y and y + 1 share the word
          skip_a = (w >> (y & 31)) & 1u;
          skip_b = (w >> ((y + 1) & 31)) & 1u;
        }
        double* ps = st.acc + (o - g.pitch);  // (x, y) at x * pitch + y
        double a[6], b[6];
#pragma unroll
        for (int k = 0; k < 6; k++)
        {
          const double2 v = *reinterpret_cast<const double2*>(ps + k * st.plane);  // (read and written here: no __ldg)
          a[k] = v.x;
          b[k] = v.y;
        }
        welford(a, inv_n, rho_a, ux_a, uy_a);
        welford(b, inv_n, rho_b, ux_b, uy_b);
#pragma unroll
        for (int k = 0; k < 6; k++)
        {
          if (!skip_a && !skip_b) st_pair(ps + k * st.plane, a[k], b[k]);
          else if (!skip_a) ps[k * st.plane] = a[k];
          else if (!skip_b) ps[k * st.plane + 1] = b[k];
        }
      }
    }
    if constexpr (ADE)
    {
      double ga[9], gb[9];
      load_streamed_pair<MODE>(gsrc, g, o, active, last_active, lane, ga, gb);
      double Ca, Cb;
      ade_collide(ga, p.omega_g, ux_a, uy_a, p.w_s, Ca);
      ade_collide(gb, p.omega_g, ux_b, uy_b, p.w_s, Cb);
      if (active)
      {
#pragma unroll
        for (int q = 0; q < 9; q++) st_pair(gdst + q * g.plane + o, ga[q], gb[q]);
      }
    }
  }
}

template <int MODE, int EQ, int FORCE, bool ADE>
__global__ void __launch_bounds__(128)
k_bgk_interior(const double* __restrict__ fsrc, double* __restrict__ fdst, const double* __restrict__ gsrc,
               double* __restrict__ gdst, const SlabGeom g, const BgkParams p, const int* __restrict__ rows, int npairs,
               double* __restrict__ out_f, double* __restrict__ out_g)
{
  bgk_interior<MODE, EQ, FORCE, ADE, false>(fsrc, fdst, gsrc, gdst, g, p, rows, npairs, out_f, out_g, StatsArgs{});
}

// the step with a statistics record on (lbm_stats_start): an entry point of its own, so that the kernels without a record
// keep their names, parameters and machine code
template <int MODE, int EQ, int FORCE, bool ADE>
__global__ void __launch_bounds__(128)
k_bgk_interior_stats(const double* __restrict__ fsrc, double* __restrict__ fdst, const double* __restrict__ gsrc,
                     double* __restrict__ gdst, const SlabGeom g, const BgkParams p, const int* __restrict__ rows, int npairs,
                     const StatsArgs st)
{
  bgk_interior<MODE, EQ, FORCE, ADE, true>(fsrc, fdst, gsrc, gdst, g, p, rows, npairs, nullptr, nullptr, st);
}

// ------------------------------------------------------------------------------------------------
// boundary kernel: one thread per listed node
// ------------------------------------------------------------------------------------------------
template <int MODE, int EQ, int FORCE, bool ADE, bool STATS>
__device__ __forceinline__ void
bgk_boundary(const double* __restrict__ fsrc, double* __restrict__ fdst, const double* __restrict__ gsrc,
             double* __restrict__ gdst, const SlabGeom g, const BgkParams p, const BoundaryTable t,
             double* __restrict__ out_f, double* __restrict__ out_g, const StatsArgs st)
{
  static_assert(!(STATS && MODE == MODE_PULL_ONLY), "a pull-only pass is no step: nothing to sample");
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= t.n) return;
  const int x = t.x[i], y = t.y[i];
  const long long o = node_off(g, x, y);

  double f[9];
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    if constexpr (MODE == MODE_LOCAL) f[q] = fsrc[q * g.plane + o];
    else
    {
      const BcEntry e = t.ent[(long long)q * t.n + i];
      const double s = fsrc[e.src];
      if (e.kind == OP_LINEAR) f[q] = e.coef * s + e.cst;
      else  // OP_ABB_EXTRAP (test/rectangle_sedimentation_test.cpp:163-172)
      {
        const double uwx = 1.5 * t.mom_prev[4 * e.aux0 + 1] - 0.5 * t.mom_prev[4 * e.aux1 + 1];
        const double uwy = 1.5 * t.mom_prev[4 * e.aux0 + 2] - 0.5 * t.mom_prev[4 * e.aux1 + 2];
        double a = 0.0;
#pragma unroll
        for (int k = 1; k < 9; k++)
          if (k == e.sq) a = abb_term(k, uwx, uwy);
        f[q] = -s + a;
      }
    }
  }

  double rho, ux, uy;
  if constexpr (MODE == MODE_PULL_ONLY)
  {
    double jx, jy;
    moments(f, rho, jx, jy);
    // velocity of the NEW post-stream state, as rectangle_sedimentation_test.cpp:199-201 computes it
    ux = jx / rho;
    uy = jy / rho;
    if (p.snap_rho != nullptr)
    {
      double sr, sx, sy;
      snapshot_moments<EQ, FORCE>(f, p, sr, sx, sy);
      const long long n = (long long)x * g.Y + y;
      p.snap_rho[n] = sr;
      p.snap_u[2 * n] = sx;
      p.snap_u[2 * n + 1] = sy;
      return;
    }
    double* oa = out_f + ((long long)x * g.Y + y) * 9;
#pragma unroll
    for (int q = 0; q < 9; q++) oa[q] = f[q];
  }
  else
  {
    bool in_roi = false;
    double Fx = 0.0, Fy = 0.0;
    if constexpr (FORCE == FORCE_IBM || FORCE == FORCE_REGION)
    {
      const int xg = x + g.xg0;
      if (xg >= p.roi_r0 && xg < p.roi_r1 && y >= p.roi_c0 && y < p.roi_c1)
      {
        in_roi = true;
        const long long r = (long long)(xg - p.roi_r0) * (p.roi_c1 - p.roi_c0) + (y - p.roi_c0);
        Fx = p.Fx[r];
        Fy = p.Fy[r];
      }
    }
    double fpost[9];
#pragma unroll
    for (int q = 0; q < 9; q++) fpost[q] = f[q];
    bool given = false;
    if constexpr (EQ == EQ_KBC && MODE == MODE_LOCAL)
    {
      if (p.mom_in_rho != nullptr)
      {
        const long long n = (long long)x * p.Y + y;
        given = true;
        rho = p.mom_in_rho[n]; ux = p.mom_in_u[2 * n]; uy = p.mom_in_u[2 * n + 1];
      }
    }
    bgk_collide<EQ, FORCE>(fpost, p, in_roi, Fx, Fy, rho, ux, uy, given);
#pragma unroll
    for (int q = 0; q < 9; q++) fdst[q * g.plane + o] = fpost[q];
  }

  double C = 0.0;
  if constexpr (ADE)
  {
    // u of the node's new post-stream state feeds the ADE inlet rule (:204-218)
    double jx, jy, r2;
    moments(f, r2, jx, jy);
    const double unx = jx / r2, uny = jy / r2;
    double gq[9];
#pragma unroll
    for (int q = 0; q < 9; q++)
    {
      if constexpr (MODE == MODE_LOCAL) gq[q] = gsrc[q * g.plane + o];
      else
      {
        const BcEntry e = t.ent[(long long)(9 + q) * t.n + i];
        const double s = gsrc[e.src];
        if (e.kind == OP_LINEAR) gq[q] = e.coef * s + e.cst;
        else  // OP_ADE_INLET
        {
          const double ax = unx + p.w_s, ay = uny + p.w_s;
          const double aa = ax * ax + ay * ay;
          double ge = 0.0;
#pragma unroll
          for (int k = 1; k < 9; k++)
            if (k == e.sq) ge = feq_comp(k, 1.0, ax, ay, aa) * e.cst;
          gq[q] = -s + 2.0 * ge;
        }
      }
    }
    if constexpr (MODE == MODE_PULL_ONLY)
    {
      double* og = out_g + ((long long)x * g.Y + y) * 9;
#pragma unroll
      for (int q = 0; q < 9; q++) og[q] = gq[q];
    }
    else
    {
      ade_collide(gq, p.omega_g, ux, uy, p.w_s, C);
#pragma unroll
      for (int q = 0; q < 9; q++) gdst[q * g.plane + o] = gq[q];
    }
  }

  if constexpr (MODE != MODE_PULL_ONLY)
  {
    t.mom_cur[4 * i + 0] = rho;
    t.mom_cur[4 * i + 1] = ux;
    t.mom_cur[4 * i + 2] = uy;
    t.mom_cur[4 * i + 3] = C;
  }
  if constexpr (STATS)
  {
    const double inv_n = st.clock->inv_n;
    if (inv_n != 0.0) stats_node(st, inv_n, o - g.pitch, rho, ux, uy);  // (x, y) at x * pitch + y
  }
}

template <int MODE, int EQ, int FORCE, bool ADE>
__global__ void __launch_bounds__(128)
k_bgk_boundary(const double* __restrict__ fsrc, double* __restrict__ fdst, const double* __restrict__ gsrc,
               double* __restrict__ gdst, const SlabGeom g, const BgkParams p, const BoundaryTable t,
               double* __restrict__ out_f, double* __restrict__ out_g)
{
  bgk_boundary<MODE, EQ, FORCE, ADE, false>(fsrc, fdst, gsrc, gdst, g, p, t, out_f, out_g, StatsArgs{});
}

template <int MODE, int EQ, int FORCE, bool ADE>
__global__ void __launch_bounds__(128)
k_bgk_boundary_stats(const double* __restrict__ fsrc, double* __restrict__ fdst, const double* __restrict__ gsrc,
                     double* __restrict__ gdst, const SlabGeom g, const BgkParams p, const BoundaryTable t, const StatsArgs st)
{
  bgk_boundary<MODE, EQ, FORCE, ADE, true>(fsrc, fdst, gsrc, gdst, g, p, t, nullptr, nullptr, st);
}

// ------------------------------------------------------------------------------------------------
// pre-stream rules applied to the freshly written post-collision buffers
// ------------------------------------------------------------------------------------------------
// zero-gradient copies (test/rectangle_sedimentation_test.cpp:138-141): f_coll[dst, :] = f_coll[src, :]
static __global__ void __launch_bounds__(128)
k_fix_copy(double* __restrict__ f, double* __restrict__ gl, const SlabGeom g, const FixEntry* __restrict__ fix, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const FixEntry e = fix[i];
  double* b = e.lattice == 0 ? f : gl;
#pragma unroll
  for (int q = 0; q < 9; q++) b[q * g.plane + e.dst] = b[q * g.plane + e.src];
}

// Pressure-periodic rows (test/horizontal_poiseuille_test.cpp:25-45) in two halves, so that the source
// row may live on another slab (test/decompose_domain.cpp:50-73):
//   pack  (owner of the source row): packet[q][y] = f_coll[src_row, y, q], packet[9..11][y] = rho, ux, uy
//   apply (owner of the written row): f_coll[dst_row] = (feq(rho_bc, u) + f_coll[src]) - feq(rho, u)
static __global__ void __launch_bounds__(128)
k_pressure_pack(const double* __restrict__ f, const SlabGeom g, int src_lx, const int* __restrict__ src_bidx,
                const double* __restrict__ mom, double* __restrict__ packet, int y_lo, int y_hi)
{
  const int y = y_lo + blockIdx.x * blockDim.x + threadIdx.x;
  if (y >= y_hi) return;
  const long long o = node_off(g, src_lx, y);
#pragma unroll
  for (int q = 0; q < 9; q++) packet[q * g.Y + y] = f[q * g.plane + o];
  const int j = src_bidx[y];
  packet[9 * g.Y + y] = mom[4 * j + 0];
  packet[10 * g.Y + y] = mom[4 * j + 1];
  packet[11 * g.Y + y] = mom[4 * j + 2];
}

template <int EQ>
static __global__ void __launch_bounds__(128)
k_pressure_apply(double* __restrict__ f, const SlabGeom g, int dst_lx, const double* __restrict__ packet, double rho_bc,
                 int y_lo, int y_hi)
{
  const int y = y_lo + blockIdx.x * blockDim.x + threadIdx.x;
  if (y >= y_hi) return;
  const long long o = node_off(g, dst_lx, y);
  const double rho = packet[9 * g.Y + y], ux = packet[10 * g.Y + y], uy = packet[11 * g.Y + y];
  const double uu = ux * ux + uy * uy;
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    // the imposed-density term: the model's own equilibrium, except for the KBC driver, which takes
    // solver::incomp_equilibrium there and kbc.iequi_f^-1 for the subtracted one (test/ulbm_poiseuille.cpp:52-57,117)
    const double t = feq_any<EQ == EQ_KBC ? EQ_INCOMP : EQ>(q, rho_bc * 1.0, ux, uy, uu);
    f[q * g.plane + o] = (t + packet[q * g.Y + y]) - feq_any<EQ>(q, rho, ux, uy, uu);
  }
}

// pack + apply in one launch when the source row and the written row live on the same slab (the single-GPU case:
// two dependent tiny launches fewer on the side chain per pressure row)
template <int EQ>
static __global__ void __launch_bounds__(128)
k_pressure_local(double* __restrict__ f, const SlabGeom g, int src_lx, int dst_lx, const int* __restrict__ src_bidx,
                 const double* __restrict__ mom, double rho_bc, int y_lo, int y_hi)
{
  const int y = y_lo + blockIdx.x * blockDim.x + threadIdx.x;
  if (y >= y_hi) return;
  const long long os = node_off(g, src_lx, y), od = node_off(g, dst_lx, y);
  const int j = src_bidx[y];
  const double rho = mom[4 * j + 0], ux = mom[4 * j + 1], uy = mom[4 * j + 2];
  const double uu = ux * ux + uy * uy;
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    const double t = feq_any<EQ == EQ_KBC ? EQ_INCOMP : EQ>(q, rho_bc * 1.0, ux, uy, uu);
    f[q * g.plane + od] = (t + f[q * g.plane + os]) - feq_any<EQ>(q, rho, ux, uy, uu);
  }
}

// ghost rows of a single slab that is its own neighbour (periodic wrap of solver::advect along
// axis 0): row -1 <- row Xl-1 for c_x = +1 populations, row Xl <- row 0 for c_x = -1 populations.
// With all_q != 0 every population is copied (models whose boundary rules read a whole opposite row).
static __global__ void k_wrap_ghost_rows(double* __restrict__ f0, double* __restrict__ f1, const SlabGeom g, int all_q)
{
  const int y = blockIdx.x * blockDim.x + threadIdx.x;
  if (y >= g.pitch) return;
  double* __restrict__ f = blockIdx.y == 0 ? f0 : f1;  // grid row = lattice
  const long long lo = y, hi = (long long)(g.Xl + 1) * g.pitch + y;
  const long long first = (long long)g.pitch + y, last = (long long)g.Xl * g.pitch + y;
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    if (all_q || CX(q) == 1) f[q * g.plane + lo] = f[q * g.plane + last];
    if (all_q || CX(q) == -1) f[q * g.plane + hi] = f[q * g.plane + first];
  }
}

// ------------------------------------------------------------------------------------------------
// layout conversion and moments of a stored buffer
// ------------------------------------------------------------------------------------------------
// AoS {Xl,Y,9} -> SoA planes
static __global__ void k_import_aos(const double* __restrict__ aos, double* __restrict__ f, const SlabGeom g)
{
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (long long)g.Xl * g.Y) return;
  const int x = (int)(n / g.Y), y = (int)(n % g.Y);
  const long long o = node_off(g, x, y);
#pragma unroll
  for (int q = 0; q < 9; q++) f[q * g.plane + o] = aos[n * 9 + q];
}

// SoA planes -> AoS {Xl,Y,9}
static __global__ void k_export_soa_to_aos(const double* __restrict__ f, double* __restrict__ aos, const SlabGeom g)
{
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (long long)g.Xl * g.Y) return;
  const int x = (int)(n / g.Y), y = (int)(n % g.Y);
  const long long o = node_off(g, x, y);
#pragma unroll
  for (int q = 0; q < 9; q++) aos[n * 9 + q] = f[q * g.plane + o];
}

}  // namespace lbm
