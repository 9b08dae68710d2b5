// lbm_domain.cu — C ABI: domain life cycle, boundary compiler, state import/export and the
// step sequencing of the single-phase family.  See include/lbm_b200.h for the contract.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstring>
#include <map>

#include "lbm_internal.hpp"

namespace lbm
{

static thread_local std::string g_error;

void set_error(const char* fmt, ...)
{
  char b[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(b, sizeof(b), fmt, ap);
  va_end(ap);
  g_error = b;
}

static inline int cdiv(long long a, int b) { return (int)((a + b - 1) / b); }

ProfScope::ProfScope(lbm_domain* dom, int cls, cudaStream_t stream) : d(dom), st(stream ? stream : dom->stream)
{
  if (!d->profiling) return;
  if (d->prof_used == d->prof.size())
  {
    if (d->prof.size() >= 65536) return;  // stop recording rather than grow without bound
    ProfRec rec;
    rec.cls = cls;
    if (cudaEventCreate(&rec.a) != cudaSuccess || cudaEventCreate(&rec.b) != cudaSuccess) return;
    d->prof.push_back(rec);
  }
  idx = (long)d->prof_used++;
  d->prof[idx].cls = cls;
  cudaEventRecord(d->prof[idx].a, st);
}

ProfScope::~ProfScope()
{
  if (idx >= 0) cudaEventRecord(d->prof[idx].b, st);
}

// ------------------------------------------------------------------------------------------------
// small kernels used only by the import / export paths
// ------------------------------------------------------------------------------------------------
// moments of an AoS post-stream state, with the conventions of the model's driver
__global__ void k_moments_aos(const double* __restrict__ aos, long long n_nodes, int incompressible, double sx,
                              double sy, double* __restrict__ rho_out, double* __restrict__ u_out)
{
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_nodes) return;
  double f[9];
#pragma unroll
  for (int q = 0; q < 9; q++) f[q] = aos[n * 9 + q];
  double rho, jx, jy;
  moments(f, rho, jx, jy);
  if (rho_out) rho_out[n] = rho;
  if (u_out)
  {
    double ux = incompressible ? jx : jx / rho;
    double uy = incompressible ? jy : jy / rho;
    u_out[2 * n] = ux + sx;
    u_out[2 * n + 1] = uy + sy;
  }
}

// kind: lbm_equilibrium_kind
__global__ void k_init_equilibrium(double* __restrict__ f, const SlabGeom g, int kind,
                                   const double* __restrict__ rho, const double* __restrict__ u)
{
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (long long)g.Xl * g.Y) return;
  const int x = (int)(n / g.Y), y = (int)(n % g.Y);
  const long long o = node_off(g, x, y);
  const double r = rho[n], ux = u[2 * n], uy = u[2 * n + 1];
  const double uu = ux * ux + uy * uy;
  if (kind == LBM_EQ_KBC || kind == LBM_EQ_KBC_FRESH)
  {
    // kbc::eval_equilibrium (src/ulbm.cpp:246-262); FRESH: its members ux2, uy2 are still zero, as when
    // test/ulbm_double_shear_flow.cpp:97 builds the initial state
    double e[9];
    kbc_eq_coef(ux, uy, kind == LBM_EQ_KBC ? ux * ux : 0.0, kind == LBM_EQ_KBC ? uy * uy : 0.0, e);
#pragma unroll
    for (int q = 0; q < 9; q++) f[q * g.plane + o] = e[q] * r;
    return;
  }
#pragma unroll
  for (int q = 0; q < 9; q++)
    f[q * g.plane + o] = kind == LBM_EQ_INCOMPRESSIBLE ? feq_incomp(q, r, ux, uy) : feq_comp(q, r, ux, uy, uu);
}

// ------------------------------------------------------------------------------------------------
// kernel dispatch
// ------------------------------------------------------------------------------------------------
// what one launch of the fused kernels works on
struct LaunchArgs
{
  int s, t;             // source / destination buffer
  const int* rows;      // row list of the interior kernel (nullptr: no interior launch)
  int n_rows;
  bool listed;          // run the listed-node kernel
  int slot;             // IBM force-field slot to read
  cudaStream_t stream;
  double* snap_rho = nullptr;  // MODE_PULL_ONLY: write moments here instead of the AoS populations
  double* snap_u = nullptr;
  int prof_cls = LBM_PROF_INTERIOR;  // profiling class of the interior launch
  bool early = false;  // the early rows of a step: with a statistics record, the interior kernel skips the listed nodes
};

// Threads per block of the side chain's kernels (listed nodes, stages, ghost rows).  (32-thread blocks, so that a pending
// block of the high-priority side stream fits the hole any retiring bulk block leaves, were measured: no difference — the
// listed-node kernel takes 79 us beside the bulk launch of a 2700 x 2100 grid against 13 us alone either way.)
constexpr int SIDE_NT = 128;

template <int MODE, int EQ, int FORCE, bool ADE, bool STATS>
static int launch_bgk(lbm_domain* d, const LaunchArgs& a)
{
  BgkParams p;
  p.omega = d->cfg.omega;
  p.inv_omega = 1.0 / d->cfg.omega;
  p.omega_g = d->cfg.omega_g;
  p.Fg0 = d->cfg.Fg[0];
  p.Fg1 = d->cfg.Fg[1];
  p.w_s = d->cfg.w_s;
  p.roi_r0 = (int)d->ibm.r0; p.roi_r1 = (int)d->ibm.r1; p.roi_c0 = (int)d->ibm.c0; p.roi_c1 = (int)d->ibm.c1;
  p.Fx = d->ibm.d_Fx[a.slot];
  p.Fy = d->ibm.d_Fy[a.slot];
  p.ics2 = d->ics2;
  p.ics4 = d->ics4;
  p.mom_in_rho = (MODE == MODE_LOCAL && d->mom_in_valid) ? d->d_mom_in : nullptr;
  p.mom_in_u = p.mom_in_rho ? d->d_mom_in + (long long)d->g.Xl * d->g.Y : nullptr;
  p.Y = d->g.Y;
  p.snap_rho = a.snap_rho;
  p.snap_u = a.snap_u;
  StatsArgs st{};  // (STATS = false: unused)
  if constexpr (STATS)
  {
    st.acc = d->st.d_acc;
    st.plane = (long long)d->g.Xl * d->g.pitch;
    st.clock = d->st.d_clock;
    st.words = d->st.words;
    st.listed = a.early ? d->st.d_listed : nullptr;
  }
  if (a.rows && d->npairs > 0 && a.n_rows > 0)
  {
    ProfScope ps(d, a.prof_cls, a.stream);
    // block size among 64 / 96 / 128 that wastes the fewest threads in a row's last block (Y = 2100: 1048 pairs are
    // 8.2 blocks of 128 but 10.9 blocks of 96)
    int bs = 128;
    for (int c : {96, 64})
      if ((long long)cdiv(d->npairs, c) * c < (long long)cdiv(d->npairs, bs) * bs) bs = c;
    dim3 grid(cdiv(d->npairs, bs), a.n_rows);
    if constexpr (STATS)
      k_bgk_interior_stats<MODE, EQ, FORCE, ADE><<<grid, bs, 0, a.stream>>>(d->buf[0][a.s], d->buf[0][a.t], d->buf[1][a.s], d->buf[1][a.t],
                                                                            d->g, p, a.rows, d->npairs, st);
    else
      k_bgk_interior<MODE, EQ, FORCE, ADE><<<grid, bs, 0, a.stream>>>(d->buf[0][a.s], d->buf[0][a.t], d->buf[1][a.s], d->buf[1][a.t],
                                                                      d->g, p, a.rows, d->npairs, d->d_aos[0], d->d_aos[1]);
    d->launches++;
  }
  if (a.listed && d->nb > 0)
  {
    ProfScope ps(d, LBM_PROF_BOUNDARY, a.stream);
    BoundaryTable bt;
    bt.n = d->nb;
    bt.x = d->d_bx;
    bt.y = d->d_by;
    bt.ent = d->d_ent;
    bt.mom_prev = d->d_mom[d->mom_cur];
    bt.mom_cur = MODE == MODE_PULL_ONLY ? nullptr : d->d_mom[d->mom_cur ^ 1];
    if constexpr (STATS)
      k_bgk_boundary_stats<MODE, EQ, FORCE, ADE><<<cdiv(d->nb, SIDE_NT), SIDE_NT, 0, a.stream>>>(d->buf[0][a.s], d->buf[0][a.t], d->buf[1][a.s],
                                                                                          d->buf[1][a.t], d->g, p, bt, st);
    else
      k_bgk_boundary<MODE, EQ, FORCE, ADE><<<cdiv(d->nb, SIDE_NT), SIDE_NT, 0, a.stream>>>(d->buf[0][a.s], d->buf[0][a.t], d->buf[1][a.s],
                                                                                  d->buf[1][a.t], d->g, p, bt, d->d_aos[0], d->d_aos[1]);
    d->launches++;
  }
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

template <int MODE, bool STATS = false>
static int dispatch_bgk(lbm_domain* d, const LaunchArgs& a)
{
  const bool ade = d->cfg.model == LBM_MODEL_BGK_ADE;
  const int eq = d->cfg.equilibrium, fo = (d->cfg.force == LBM_FORCE_IBM && d->ibm.fixed) ? (int)FORCE_REGION : d->cfg.force;
  if (ade)
  {
    // with an immersed body (BASELINE configs[4] "with immersed-boundary coupling"): the cylinder driver's force term on the
    // fluid lattice, the ADE lattice advected by the same u
    if (fo == FORCE_IBM) return launch_bgk<MODE, EQ_COMP, FORCE_IBM, true, STATS>(d, a);
    return launch_bgk<MODE, EQ_COMP, FORCE_NONE, true, STATS>(d, a);
  }
  if (d->cfg.model == LBM_MODEL_KBC) return launch_bgk<MODE, EQ_KBC, FORCE_NONE, false, STATS>(d, a);
#define LBM_CASE(E, F) \
  if (eq == E && fo == F) return launch_bgk<MODE, E, F, false, STATS>(d, a);
  LBM_CASE(EQ_COMP, FORCE_NONE)
  LBM_CASE(EQ_COMP, FORCE_UNIFORM)
  LBM_CASE(EQ_COMP, FORCE_IBM)
  LBM_CASE(EQ_INCOMP, FORCE_NONE)
  LBM_CASE(EQ_INCOMP, FORCE_UNIFORM)
  LBM_CASE(EQ_INCOMP, FORCE_IBM)
  LBM_CASE(EQ_COMP, FORCE_REGION)
  LBM_CASE(EQ_INCOMP, FORCE_REGION)
#undef LBM_CASE
  set_error("unsupported equilibrium/force combination (%d, %d)", eq, fo);
  return LBM_ERR_INVALID;
}

// a step's launches: with a statistics record on, the STATS instantiations
static int dispatch_mode(lbm_domain* d, int mode, const LaunchArgs& a)
{
  if (d->st.on && mode == MODE_LOCAL) return dispatch_bgk<MODE_LOCAL, true>(d, a);
  if (d->st.on && mode == MODE_PULL) return dispatch_bgk<MODE_PULL, true>(d, a);
  if (mode == MODE_LOCAL) return dispatch_bgk<MODE_LOCAL>(d, a);
  if (mode == MODE_PULL) return dispatch_bgk<MODE_PULL>(d, a);
  return dispatch_bgk<MODE_PULL_ONLY>(d, a);
}

int wrap_ghost_rows_local(lbm_domain* d, int which, cudaStream_t st)
{
  // one launch for both lattices (grid row = lattice)
  k_wrap_ghost_rows<<<dim3(cdiv(d->g.pitch, SIDE_NT), d->nlat), SIDE_NT, 0, st>>>(d->buf[0][which], d->nlat > 1 ? d->buf[1][which] : nullptr, d->g,
                                                                                d->wrap_all_q ? 1 : 0);
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

// ------------------------------------------------------------------------------------------------
// One time step of the single-phase family.
//
//   main stream : [wait side chain of the previous step]  EARLY rows  ->  ev_early  ->  BULK rows
//   side stream : [wait ev_early] listed nodes -> pre-stream stages -> ghost rows of the new buffer
//                 (local wrap / NCCL ring) -> IBM pre-pass for the NEXT step -> ev_side
//   (no bulk rows at all: the early launch opens the side chain instead, see step_early)
//
// EARLY rows are the few rows whose results something else needs soon: the first and last row
// (ghost exchange), rows owning a listed node in an interior column or feeding a stage (the listed
// kernel and the stages overwrite / read them), and the immersed-boundary ROI rows (next pre-pass).
// Everything small therefore runs concurrently with the BULK launch, which is >95 % of the step.
// ------------------------------------------------------------------------------------------------
int step_rows(lbm_domain* d)
{
  if (!d->rows_dirty) return LBM_OK;
  const int Xl = d->g.Xl;
  std::vector<char> early(Xl, 0);
  early[0] = early[Xl - 1] = 1;
  for (int x = 0; x < Xl && x < (int)d->row_has_listed.size(); x++)
    if (d->row_has_listed[x]) early[x] = 1;
  if (d->ibm.enabled && !d->ibm.fixed)
    for (long gx = d->ibm.r0 - 1; gx < d->ibm.r1 + 1; gx++)
    {
      const long x = gx - d->cfg.x0;
      if (x >= 0 && x < Xl) early[x] = 1;
    }
  std::vector<int> all(Xl), e, b;
  for (int x = 0; x < Xl; x++)
  {
    all[x] = x;
    (early[x] ? e : b).push_back(x);
  }
  cudaFree(d->d_rows_all); cudaFree(d->d_rows_early); cudaFree(d->d_rows_bulk);
  d->d_rows_all = d->d_rows_early = d->d_rows_bulk = nullptr;
  LBM_CUDA(cudaMalloc(&d->d_rows_all, sizeof(int) * Xl));
  LBM_CUDA(cudaMalloc(&d->d_rows_early, sizeof(int) * std::max<size_t>(e.size(), 1)));
  LBM_CUDA(cudaMalloc(&d->d_rows_bulk, sizeof(int) * std::max<size_t>(b.size(), 1)));
  LBM_CUDA(cudaMemcpy(d->d_rows_all, all.data(), sizeof(int) * Xl, cudaMemcpyHostToDevice));
  LBM_CUDA(cudaMemcpy(d->d_rows_early, e.data(), sizeof(int) * e.size(), cudaMemcpyHostToDevice));
  LBM_CUDA(cudaMemcpy(d->d_rows_bulk, b.data(), sizeof(int) * b.size(), cudaMemcpyHostToDevice));
  d->n_early = (int)e.size();
  d->n_bulk = (int)b.size();
  d->rows_dirty = false;
  return LBM_OK;
}

// Side chain for a state that no step has prepared (first step after an import, or an export):
// ghost rows of buf[cur] and the IBM field the next step reads.
int step_prologue(lbm_domain* d, bool exchange_local, bool with_ibm)
{
  if (d->side_ready) return LBM_OK;
  const int mode = d->post_stream ? MODE_LOCAL : MODE_PULL;
  LBM_CUDA(cudaEventRecord(d->ev_ready, d->stream));
  LBM_CUDA(cudaStreamWaitEvent(d->side, d->ev_ready, 0));
  if (mode == MODE_PULL && exchange_local)
  {
    ProfScope ps(d, LBM_PROF_GHOST, d->side);
    if (comm_active(d)) LBM_TRY(comm_exchange(d, d->cur, d->side));
    else LBM_TRY(wrap_ghost_rows_local(d, d->cur, d->side));
  }
  if (with_ibm && uses_ibm(d))
  {
    ProfScope ps(d, LBM_PROF_IBM, d->side);
    LBM_TRY(ibm_prepass(d, mode, d->cur, d->ibm.next_slot, d->side));
  }
  LBM_CUDA(cudaEventRecord(d->ev_side, d->side));
  d->side_ready = with_ibm || !uses_ibm(d);  // (linked slabs: lbm_step_group finishes the immersed-boundary part)
  return LBM_OK;
}

// Early rows.  With a bulk launch to overlap: on the main stream, ahead of it (the side chain starts from ev_early and runs
// beside the bulk rows).  WITHOUT one — every row is an early row, e.g. the sedimentation driver, whose outlet stage reads
// every row — the step is a serial chain anyway, and the launch opens the side chain itself: one cross-stream hop per step
// instead of two, +5.7 % on the 4096 x 8192 sedimentation workload.  (Moving the early rows to the side stream in
// general was measured too: same speed at 8192^2, -5 % on the 2700 x 2100 Poiseuille grid, whose side chain is its
// critical path, and per-kernel times that no longer add up because the two launches share the SMs.)
int step_early(lbm_domain* d)
{
  LBM_TRY(step_rows(d));
  const int mode = d->post_stream ? MODE_LOCAL : MODE_PULL;
  if (!d->skip_side_wait) LBM_CUDA(cudaStreamWaitEvent(d->stream, d->ev_side, 0));  // main: the previous side chain
  d->skip_side_wait = false;
  d->early_on_side = d->n_bulk == 0;
  if (d->early_on_side)
  {
    LBM_CUDA(cudaEventRecord(d->ev_early, d->stream));
    LBM_CUDA(cudaStreamWaitEvent(d->side, d->ev_early, 0));
    LaunchArgs a{d->cur, d->cur ^ 1, d->d_rows_early, d->n_early, false, d->ibm.next_slot, d->side};
    a.prof_cls = LBM_PROF_EARLY;
    a.early = true;
    return dispatch_mode(d, mode, a);
  }
  LaunchArgs a{d->cur, d->cur ^ 1, d->d_rows_early, d->n_early, false, d->ibm.next_slot, d->stream};
  a.prof_cls = LBM_PROF_EARLY;
  a.early = true;
  LBM_TRY(dispatch_mode(d, mode, a));
  LBM_CUDA(cudaEventRecord(d->ev_early, d->stream));
  return LBM_OK;
}

int step_listed(lbm_domain* d)
{
  const int mode = d->post_stream ? MODE_LOCAL : MODE_PULL;
  if (!d->early_on_side) LBM_CUDA(cudaStreamWaitEvent(d->side, d->ev_early, 0));
  LaunchArgs a{d->cur, d->cur ^ 1, nullptr, 0, true, d->ibm.next_slot, d->side};
  return dispatch_mode(d, mode, a);
}

int stage_pack(lbm_domain* d, size_t k)
{
  Stage& sg = d->stages[k];
  if (sg.kind != 1 || !sg.own_src || sg.y_hi <= sg.y_lo) return LBM_OK;
  ProfScope ps(d, LBM_PROF_FIXUP, d->side);
  const int t = d->cur ^ 1;
  k_pressure_pack<<<cdiv(sg.y_hi - sg.y_lo, SIDE_NT), SIDE_NT, 0, d->side>>>(d->buf[0][t], d->g, sg.src_gx - d->cfg.x0, sg.d_src_bidx,
                                                                    d->d_mom[d->mom_cur ^ 1], sg.d_packet, sg.y_lo, sg.y_hi);
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

int stage_apply(lbm_domain* d, size_t k)
{
  Stage& sg = d->stages[k];
  const int t = d->cur ^ 1;
  ProfScope ps(d, LBM_PROF_FIXUP, d->side);
  if (sg.kind == 0)
  {
    if (sg.n == 0) return LBM_OK;
    k_fix_copy<<<cdiv(sg.n, SIDE_NT), SIDE_NT, 0, d->side>>>(d->buf[0][t], d->buf[1][t], d->g, sg.d_entries, sg.n);
    d->launches++;
  }
  else
  {
    if (!sg.own_dst || sg.y_hi <= sg.y_lo) return LBM_OK;
    const int lx = sg.dst_gx - d->cfg.x0, nblk = cdiv(sg.y_hi - sg.y_lo, SIDE_NT);
    if (d->cfg.model == LBM_MODEL_KBC)
      k_pressure_apply<EQ_KBC><<<nblk, SIDE_NT, 0, d->side>>>(d->buf[0][t], d->g, lx, sg.d_packet, sg.rho_bc, sg.y_lo, sg.y_hi);
    else if (d->cfg.equilibrium == EQ_INCOMP)
      k_pressure_apply<EQ_INCOMP><<<nblk, SIDE_NT, 0, d->side>>>(d->buf[0][t], d->g, lx, sg.d_packet, sg.rho_bc, sg.y_lo, sg.y_hi);
    else
      k_pressure_apply<EQ_COMP><<<nblk, SIDE_NT, 0, d->side>>>(d->buf[0][t], d->g, lx, sg.d_packet, sg.rho_bc, sg.y_lo, sg.y_hi);
    d->launches++;
  }
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

static int stage_local(lbm_domain* d, size_t k)
{
  Stage& sg = d->stages[k];
  if (sg.y_hi <= sg.y_lo) return LBM_OK;
  ProfScope ps(d, LBM_PROF_FIXUP, d->side);
  const int t = d->cur ^ 1, nblk = cdiv(sg.y_hi - sg.y_lo, SIDE_NT);
  const int src_lx = sg.src_gx - d->cfg.x0, dst_lx = sg.dst_gx - d->cfg.x0;
  double* f = d->buf[0][t];
  const double* mom = d->d_mom[d->mom_cur ^ 1];
  if (d->cfg.model == LBM_MODEL_KBC)
    k_pressure_local<EQ_KBC><<<nblk, SIDE_NT, 0, d->side>>>(f, d->g, src_lx, dst_lx, sg.d_src_bidx, mom, sg.rho_bc, sg.y_lo, sg.y_hi);
  else if (d->cfg.equilibrium == EQ_INCOMP)
    k_pressure_local<EQ_INCOMP><<<nblk, SIDE_NT, 0, d->side>>>(f, d->g, src_lx, dst_lx, sg.d_src_bidx, mom, sg.rho_bc, sg.y_lo, sg.y_hi);
  else
    k_pressure_local<EQ_COMP><<<nblk, SIDE_NT, 0, d->side>>>(f, d->g, src_lx, dst_lx, sg.d_src_bidx, mom, sg.rho_bc, sg.y_lo, sg.y_hi);
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

// ghost rows of the NEW buffer and the IBM field of the NEXT step, then ev_side
int step_side_tail(lbm_domain* d, bool exchange_local, bool with_ibm)
{
  const int t = d->cur ^ 1;
  if (exchange_local)
  {
    ProfScope ps(d, LBM_PROF_GHOST, d->side);
    if (comm_active(d)) LBM_TRY(comm_exchange(d, t, d->side));
    else LBM_TRY(wrap_ghost_rows_local(d, t, d->side));
  }
  if (with_ibm && uses_ibm(d))
  {
    ProfScope ps(d, LBM_PROF_IBM, d->side);
    LBM_TRY(ibm_prepass(d, MODE_PULL, t, d->ibm.next_slot ^ 1, d->side));
  }
  LBM_TRY(body_force_step(d));
  LBM_CUDA(cudaEventRecord(d->ev_side, d->side));
  return LBM_OK;
}

int step_bulk(lbm_domain* d)
{
  const int mode = d->post_stream ? MODE_LOCAL : MODE_PULL;
  LaunchArgs a{d->cur, d->cur ^ 1, d->d_rows_bulk, d->n_bulk, false, d->ibm.next_slot, d->stream};
  LBM_TRY(dispatch_mode(d, mode, a));
  LBM_TRY(stats_tick(d));
  d->cur ^= 1;
  d->mom_cur ^= 1;
  d->post_stream = false;
  d->mom_in_valid = false;
  d->ibm.used_slot = d->ibm.next_slot;
  d->ibm.next_slot ^= 1;
  d->side_ready = true;  // the side chain enqueued during this step prepared the new buffer
  return LBM_OK;
}

static int bgk_step_once(lbm_domain* d)
{
  bool remote_faces = false;
  for (const auto& fl : d->faces)
  {
    if (fl.peer_rank < 0)
    {
      set_error("lbm_step: this block is bound to others across a column face; advance the set with lbm_step_group");
      return LBM_ERR_INVALID;
    }
    remote_faces = true;
  }
  remote_faces = remote_faces || !d->serves.empty();
  if (comm_blocks(d) && !d->faces_remote_ready)
  {
    set_error("lbm_step: blocks bound across ranks: call lbm_comm_faces_commit (every rank) after the last lbm_link_face_rank");
    return LBM_ERR_INVALID;
  }
  if (uses_ibm(d) && d->ibm.split && !comm_active(d))
  {
    set_error("lbm_step: the immersed body crosses this slab's edge; advance the slabs with lbm_step_group or join them with lbm_comm_init");
    return LBM_ERR_INVALID;
  }
  if (d->link_lo || d->link_hi)
  {
    set_error("lbm_step: this slab is linked to neighbours; advance the set with lbm_step_group");
    return LBM_ERR_INVALID;
  }
  const bool unprepared = !d->side_ready;
  LBM_TRY(step_prologue(d, true, true));
  if (remote_faces && unprepared && !d->post_stream)
  {
    // a stored state no step has prepared (after an export): the face tails of the CURRENT buffers, like lbm_step_group
    LBM_TRY(faces_exchange_remote(d, false));
    LBM_CUDA(cudaEventRecord(d->ev_side, d->side));
  }
  LBM_TRY(step_early(d));
  LBM_TRY(step_listed(d));
  if (remote_faces) LBM_TRY(faces_exchange_remote(d, true));  // the edge columns just written feed the bound blocks' next step
  for (size_t k = 0; k < d->stages.size(); k++)
  {
    const Stage& sg = d->stages[k];
    if (sg.kind == 1 && sg.own_src && sg.own_dst && !comm_active(d))
    {
      LBM_TRY(stage_local(d, k));  // source and written row on this slab: one launch
      continue;
    }
    LBM_TRY(stage_pack(d, k));
    if (comm_active(d)) LBM_TRY(comm_stage_transfer(d, k, d->side));
    LBM_TRY(stage_apply(d, k));
  }
  LBM_TRY(step_side_tail(d, true, true));
  return step_bulk(d);
}

int ensure_aos_scratch(lbm_domain* d)
{
  const size_t bytes = (size_t)d->g.Xl * d->g.Y * 9 * sizeof(double);
  for (int l = 0; l < d->nlat; l++)
    if (!d->d_aos[l]) LBM_CUDA(cudaMalloc(&d->d_aos[l], bytes));
  return LBM_OK;
}

// post-stream populations of every lattice into d_aos[] (device, reference layout)
static int export_post_stream(lbm_domain* d)
{
  LBM_TRY(ensure_aos_scratch(d));
  if (d->tp) return tp_export(d);
  const long long N = (long long)d->g.Xl * d->g.Y;
  if (d->post_stream)
  {
    for (int l = 0; l < d->nlat; l++)
    {
      k_export_soa_to_aos<<<cdiv(N, 256), 256, 0, d->stream>>>(d->buf[l][d->cur], d->d_aos[l], d->g);
      d->launches++;
    }
    LBM_CUDA(cudaGetLastError());
    return LBM_OK;
  }
  // pull-only pass over every row: the ghost rows of buf[cur] must be in place
  LBM_TRY(step_rows(d));
  if (d->link_lo || d->link_hi) LBM_TRY(comm_link_refresh(d));
  else LBM_TRY(step_prologue(d, true, true));
  LBM_CUDA(cudaStreamWaitEvent(d->stream, d->ev_side, 0));
  LaunchArgs a{d->cur, d->cur ^ 1, d->d_rows_all, d->g.Xl, true, d->ibm.used_slot, d->stream};
  return dispatch_bgk<MODE_PULL_ONLY>(d, a);
}

// ------------------------------------------------------------------------------------------------
// boundary compiler
// ------------------------------------------------------------------------------------------------
static void resolve_slice(int b, int e, int n, int& lo, int& hi)
{
  // torch::indexing::Slice semantics for step 1
  long long bb = b, ee = (e == LBM_END) ? n : e;
  if (bb < 0) bb += n;
  if (ee < 0) ee += n;
  bb = std::max(0LL, std::min<long long>(bb, n));
  ee = std::max(0LL, std::min<long long>(ee, n));
  lo = (int)bb;
  hi = (int)std::max(bb, ee);
}

static int resolve_index(int v, int n) { return v < 0 ? v + n : v; }

struct SrcNode
{
  int gx, y;
  bool ok;
};

static SrcNode src_of(const lbm_bc_op& op, int gx, int y, int X, int Y)
{
  SrcNode s{gx, y, true};
  switch (op.src_mode)
  {
    case LBM_SRC_SAME_NODE: break;
    case LBM_SRC_SHIFT: s.gx = gx + op.src_a; s.y = y + op.src_b; break;
    case LBM_SRC_ROW: s.gx = resolve_index(op.src_a, X); break;
    case LBM_SRC_COL: s.y = resolve_index(op.src_a, Y); break;
    default: s.ok = false;
  }
  if (s.y < 0 || s.y >= Y || s.gx < 0 || s.gx >= X) s.ok = false;
  return s;
}

// global row -> local storage row (ghost rows -1 and Xl included); INT_MIN if not reachable
static int local_row(const lbm_domain* d, int gx)
{
  const int X = d->cfg.X, x0 = d->cfg.x0, x1 = d->cfg.x1;
  if (gx >= x0 - 1 && gx <= x1) return gx - x0;
  if (x0 == 0 && gx == X - 1) return -1;          // periodic image below row 0
  if (x1 == X && gx == 0) return x1 - x0;         // periodic image above the last row
  return INT_MIN;
}

void drop_graphs(lbm_domain* d)
{
  for (int k = 0; k < 2; k++)
    if (d->graph_exec[k])
    {
      cudaGraphExecDestroy(d->graph_exec[k]);
      d->graph_exec[k] = nullptr;
    }
}

static void release_compiled(lbm_domain* d)
{
  drop_graphs(d);
  if (d->bf.on && !d->bf.immersed) body_force_release(d);  // its links were checked against the rules being replaced
  cudaFree(d->d_bx); cudaFree(d->d_by); cudaFree(d->d_ent); cudaFree(d->d_mom[0]); cudaFree(d->d_mom[1]);
  d->d_bx = d->d_by = nullptr; d->d_ent = nullptr; d->d_mom[0] = d->d_mom[1] = nullptr;
  for (auto& sg : d->stages)
  {
    cudaFree(sg.d_entries);
    cudaFree(sg.d_src_bidx);
    cudaFree(sg.d_packet);
  }
  d->stages.clear();
  d->nb = 0;
  d->committed = false;
}

static bool is_post_stream(int kind)
{
  return kind == LBM_BC_LINEAR || kind == LBM_BC_ABB_FIXED || kind == LBM_BC_ABB_EXTRAPOLATED || kind == LBM_BC_ADE_INLET;
}

int commit_boundary_tables(lbm_domain* d)
{
  const int X = d->cfg.X, Y = d->cfg.Y, x0 = d->cfg.x0, Xl = d->g.Xl;
  const SlabGeom& g = d->g;
  const int y_int_begin = d->y_int_begin, y_int_end = d->y_int_end;  // columns owned by the interior kernel

  // ---- pass 1: which nodes need a table entry
  std::map<long long, int> index;  // local node id -> boundary index
  auto touch = [&](int lx, int y) {
    if (lx < 0 || lx >= Xl) return;
    index.emplace((long long)lx * Y + y, 0);
  };
  for (int lx = 0; lx < Xl; lx++)
    for (int y = 0; y < Y; y++)
      if (y < y_int_begin || y >= y_int_end) touch(lx, y);
  d->wrap_all_q = false;
  for (const auto& so : d->ops)
  {
    const lbm_bc_op& op = so.op;
    int xl, xh, yl, yh;
    resolve_slice(op.x_begin, op.x_end, X, xl, xh);
    resolve_slice(op.y_begin, op.y_end, Y, yl, yh);
    for (int gx = xl; gx < xh; gx++)
      for (int y = yl; y < yh; y++)
      {
        if (is_post_stream(op.kind)) touch(gx - x0, y);
        if (op.kind == LBM_BC_ABB_EXTRAPOLATED)
        {
          touch(gx - x0, Y - 1);
          touch(gx - x0, Y - 2);
        }
        if (op.kind == LBM_BC_PRESSURE_PERIODIC)
        {
          SrcNode s = src_of(op, gx, y, X, Y);
          if (s.ok) touch(s.gx - x0, s.y);
        }
        if (op.kind == LBM_BC_LINEAR && op.src_mode != LBM_SRC_SAME_NODE)
        {
          SrcNode s = src_of(op, gx, y, X, Y);
          if (s.ok && std::abs(s.gx - gx) > 1) d->wrap_all_q = true;  // reads across the periodic wrap
        }
      }
  }
  int nb = 0;
  for (auto& kv : index) kv.second = nb++;

  // ---- pass 2: default entries = periodic pull (solver::advect)
  std::vector<int> bx(nb), by(nb);
  std::vector<BcEntry> ent((size_t)d->nlat * 9 * nb);
  for (auto& kv : index)
  {
    const int i = kv.second, lx = (int)(kv.first / Y), y = (int)(kv.first % Y);
    bx[i] = lx;
    by[i] = y;
    for (int l = 0; l < d->nlat; l++)
      for (int q = 0; q < 9; q++)
      {
        int sy = y - CY(q);
        if (sy < 0) sy += Y;
        if (sy >= Y) sy -= Y;
        const int sx = lx - CX(q);  // ghost rows carry the wrap / the neighbour slab
        BcEntry e;
        e.src = (long long)q * g.plane + (long long)(sx + 1) * g.pitch + sy;
        e.coef = 1.0; e.cst = 0.0; e.kind = OP_LINEAR; e.sq = q; e.aux0 = e.aux1 = 0;
        ent[((size_t)l * 9 + q) * nb + i] = e;
      }
  }
  for (int l = 0; l < 2; l++) d->mask[l].assign(l < d->nlat ? (size_t)Xl * Y * 9 : 0, 0);

  // ---- pass 3: ops in order (later ops win, like the reference's successive assignments)
  struct HostStage
  {
    int kind = 0, dst_gx = 0, src_gx = 0, y_lo = 0, y_hi = 0;
    double rho_bc = 1.0;
    bool own_src = false, own_dst = false;
    std::vector<FixEntry> entries;
    std::vector<int> src_bidx;
  };
  std::vector<HostStage> host_stages;
  for (size_t k = 0; k < d->ops.size(); k++)
  {
    const lbm_bc_op& op = d->ops[k].op;
    int xl, xh, yl, yh;
    resolve_slice(op.x_begin, op.x_end, X, xl, xh);
    resolve_slice(op.y_begin, op.y_end, Y, yl, yh);
    const int lat_lo = op.lattice < 0 ? 0 : op.lattice, lat_hi = op.lattice < 0 ? d->nlat - 1 : op.lattice;
    if (lat_hi >= d->nlat) { set_error("bc op %zu: lattice %d does not exist in this model", k, op.lattice); return LBM_ERR_INVALID; }
    if (op.kind == LBM_BC_COPY_PRE)
    {
      HostStage hs;
      hs.kind = 0;
      for (int gx = xl; gx < xh; gx++)
      {
        if (gx < x0 || gx >= d->cfg.x1) continue;
        for (int y = yl; y < yh; y++)
        {
          SrcNode s = src_of(op, gx, y, X, Y);
          if (!s.ok) { set_error("bc op %zu: source node outside the grid", k); return LBM_ERR_INVALID; }
          if (s.gx < x0 || s.gx >= d->cfg.x1)
          {
            set_error("bc op %zu: copy source row %d is owned by another slab (not supported across slabs)", k, s.gx);
            return LBM_ERR_UNSUPPORTED;
          }
          for (int l = lat_lo; l <= lat_hi; l++)
          {
            FixEntry e;
            e.dst = (long long)(gx - x0 + 1) * g.pitch + y;
            e.src = (long long)(s.gx - x0 + 1) * g.pitch + s.y;
            e.lattice = l;
            e.pad = 0;
            hs.entries.push_back(e);
          }
        }
      }
      host_stages.push_back(std::move(hs));
      continue;
    }
    if (op.kind == LBM_BC_PRESSURE_PERIODIC)
    {
      if (xh - xl != 1 || op.src_mode != LBM_SRC_ROW)
      {
        set_error("bc op %zu: LBM_BC_PRESSURE_PERIODIC writes one row from one source row (LBM_SRC_ROW)", k);
        return LBM_ERR_INVALID;
      }
      HostStage hs;
      hs.kind = 1;
      hs.dst_gx = xl;
      hs.src_gx = resolve_index(op.src_a, X);
      if (hs.src_gx < 0 || hs.src_gx >= X) { set_error("bc op %zu: source row outside the grid", k); return LBM_ERR_INVALID; }
      hs.y_lo = yl; hs.y_hi = yh; hs.rho_bc = op.rho_bc;
      hs.own_dst = hs.dst_gx >= x0 && hs.dst_gx < d->cfg.x1;
      hs.own_src = hs.src_gx >= x0 && hs.src_gx < d->cfg.x1;
      if (hs.own_src)
      {
        hs.src_bidx.assign(Y, 0);
        for (int y = yl; y < yh; y++) hs.src_bidx[y] = index.at((long long)(hs.src_gx - x0) * Y + y);
      }
      host_stages.push_back(std::move(hs));
      continue;
    }
    if (!is_post_stream(op.kind)) { set_error("bc op %zu: unknown kind %d", k, op.kind); return LBM_ERR_INVALID; }
    if (op.kind == LBM_BC_ADE_INLET && (d->cfg.model != LBM_MODEL_BGK_ADE || op.lattice != 1))
    { set_error("bc op %zu: LBM_BC_ADE_INLET applies to lattice 1 of LBM_MODEL_BGK_ADE", k); return LBM_ERR_INVALID; }
    for (int gx = xl; gx < xh; gx++)
    {
      if (gx < x0 || gx >= d->cfg.x1) continue;
      const int lx = gx - x0;
      for (int y = yl; y < yh; y++)
      {
        const int i = index.at((long long)lx * Y + y);
        // population loop: LINEAR with dst_q = -1 copies all nine; ABB-type rules with src_q = -1 cover the 8 moving ones
        const bool abb_like = op.kind != LBM_BC_LINEAR;
        const int q_lo = abb_like ? (op.src_q < 0 ? 1 : op.src_q) : (op.dst_q < 0 ? 0 : op.dst_q);
        const int q_hi = abb_like ? (op.src_q < 0 ? 8 : op.src_q) : (op.dst_q < 0 ? 8 : op.dst_q);
        for (int qq = q_lo; qq <= q_hi; qq++)
        {
          int dq, sq;
          if (abb_like) { sq = qq; dq = OPP(qq); }
          else { dq = qq; sq = op.dst_q < 0 ? qq : op.src_q; }
          if (dq < 0 || dq > 8 || sq < 0 || sq > 8) { set_error("bc op %zu: population index out of range", k); return LBM_ERR_INVALID; }
          SrcNode s = src_of(op, gx, y, X, Y);
          if (!s.ok) { set_error("bc op %zu: source node outside the grid", k); return LBM_ERR_INVALID; }
          const int slx = local_row(d, s.gx);
          if (slx == INT_MIN)
          {
            set_error("bc op %zu: source row %d is not reachable from slab rows [%d,%d)", k, s.gx, x0, d->cfg.x1);
            return LBM_ERR_UNSUPPORTED;
          }
          for (int l = lat_lo; l <= lat_hi; l++)
          {
            BcEntry e;
            e.src = (long long)sq * g.plane + (long long)(slx + 1) * g.pitch + s.y;
            e.sq = sq; e.aux0 = e.aux1 = 0;
            switch (op.kind)
            {
              case LBM_BC_LINEAR: e.kind = OP_LINEAR; e.coef = op.coef; e.cst = op.cst; break;
              case LBM_BC_ABB_FIXED: e.kind = OP_LINEAR; e.coef = -1.0; e.cst = abb_term(sq, op.uw[0], op.uw[1]); break;
              case LBM_BC_ABB_EXTRAPOLATED:
                e.kind = OP_ABB_EXTRAP; e.coef = -1.0; e.cst = 0.0;
                e.aux0 = index.at((long long)lx * Y + (Y - 1));
                e.aux1 = index.at((long long)lx * Y + (Y - 2));
                break;
              case LBM_BC_ADE_INLET: e.kind = OP_ADE_INLET; e.coef = -1.0; e.cst = d->ops[k].per_row[gx]; break;
            }
            ent[((size_t)l * 9 + dq) * nb + i] = e;
            d->mask[l][((size_t)lx * Y + y) * 9 + dq] = (int32_t)(k + 1);
          }
        }
      }
    }
  }

  // ---- column-face bindings (lbm_link_face), after every op like "Bind the domains" at the end of the reference's loop
  // body (test/decompose_domain_loop.cpp:230-261): population q entering through the edge column on row rb + k comes
  // from row k - c_qx of the facing column; where that row is outside the bound range the wall rule stays
  for (size_t j = 0; j < d->faces.size(); j++)
  {
    const FaceLink& fl = d->faces[j];
    const int col = fl.side == 0 ? 0 : Y - 1;
    for (int k = 0; k < fl.n; k++)
    {
      const int i = index.at((long long)(fl.rb + k) * Y + col);
      for (int qi = 0; qi < 3; qi++)
      {
        const int q = face_q(fl.side, qi);
        const int ks = k - CX(q);
        if (ks < 0 || ks >= fl.n) continue;
        for (int l = 0; l < d->nlat; l++)
        {
          BcEntry e;
          e.src = face_tail_off(g, fl.side, qi, fl.rb + ks);
          e.coef = 1.0; e.cst = 0.0; e.kind = OP_LINEAR; e.sq = q; e.aux0 = e.aux1 = 0;
          ent[((size_t)l * 9 + q) * nb + i] = e;
          d->mask[l][((size_t)(fl.rb + k) * Y + col) * 9 + q] = (int32_t)(d->ops.size() + 1 + j);
        }
      }
    }
  }

  // rows the interior kernel must finish before the listed-node kernel / the stages touch them
  d->row_has_listed.assign(Xl, 0);
  d->listed_ids.clear();
  for (auto& kv : index)  // (ordered map: ascending ids)
  {
    const int lx = (int)(kv.first / Y), y = (int)(kv.first % Y);
    if (y >= y_int_begin && y < y_int_end) d->row_has_listed[lx] = 1;
    d->listed_ids.push_back((int)kv.first);
  }
  for (auto& hs : host_stages)
  {
    if (hs.kind == 1)
    {
      if (hs.own_dst) d->row_has_listed[hs.dst_gx - x0] = 1;
      if (hs.own_src) d->row_has_listed[hs.src_gx - x0] = 1;
    }
    for (auto& e : hs.entries)
    {
      d->row_has_listed[(int)(e.dst / g.pitch) - 1] = 1;
      d->row_has_listed[(int)(e.src / g.pitch) - 1] = 1;
    }
  }
  d->rows_dirty = true;
  d->side_ready = false;
  if (d->st.on) LBM_TRY(stats_listed_mask(d));

  // ---- upload
  d->nb = nb;
  if (nb > 0)
  {
    LBM_CUDA(cudaMalloc(&d->d_bx, sizeof(int) * nb));
    LBM_CUDA(cudaMalloc(&d->d_by, sizeof(int) * nb));
    LBM_CUDA(cudaMalloc(&d->d_ent, sizeof(BcEntry) * ent.size()));
    LBM_CUDA(cudaMalloc(&d->d_mom[0], sizeof(double) * 4 * nb));
    LBM_CUDA(cudaMalloc(&d->d_mom[1], sizeof(double) * 4 * nb));
    LBM_CUDA(cudaMemcpy(d->d_bx, bx.data(), sizeof(int) * nb, cudaMemcpyHostToDevice));
    LBM_CUDA(cudaMemcpy(d->d_by, by.data(), sizeof(int) * nb, cudaMemcpyHostToDevice));
    LBM_CUDA(cudaMemcpy(d->d_ent, ent.data(), sizeof(BcEntry) * ent.size(), cudaMemcpyHostToDevice));
    LBM_CUDA(cudaMemset(d->d_mom[0], 0, sizeof(double) * 4 * nb));
    LBM_CUDA(cudaMemset(d->d_mom[1], 0, sizeof(double) * 4 * nb));
  }
  for (auto& hs : host_stages)
  {
    Stage sg;
    sg.kind = hs.kind;
    sg.n = (int)hs.entries.size();
    sg.dst_gx = hs.dst_gx; sg.src_gx = hs.src_gx; sg.y_lo = hs.y_lo; sg.y_hi = hs.y_hi; sg.rho_bc = hs.rho_bc;
    sg.own_src = hs.own_src; sg.own_dst = hs.own_dst;
    if (sg.n > 0)
    {
      LBM_CUDA(cudaMalloc(&sg.d_entries, sizeof(FixEntry) * sg.n));
      LBM_CUDA(cudaMemcpy(sg.d_entries, hs.entries.data(), sizeof(FixEntry) * sg.n, cudaMemcpyHostToDevice));
    }
    if (hs.kind == 1 && (hs.own_src || hs.own_dst))
    {
      LBM_CUDA(cudaMalloc(&sg.d_packet, sizeof(double) * 12 * Y));
      LBM_CUDA(cudaMemset(sg.d_packet, 0, sizeof(double) * 12 * Y));
      if (hs.own_src)
      {
        LBM_CUDA(cudaMalloc(&sg.d_src_bidx, sizeof(int) * Y));
        LBM_CUDA(cudaMemcpy(sg.d_src_bidx, hs.src_bidx.data(), sizeof(int) * Y, cudaMemcpyHostToDevice));
      }
    }
    d->stages.push_back(sg);
  }
  d->committed = true;
  return LBM_OK;
}

// The staging buffer of the snapshot path doubles as the landing zone of host fields on their way in
// (cudaMalloc / cudaFree per call cost 30-600 ms at 136 MB on this box: measured, hence persistent).
int host_staging(lbm_domain* d, double** out)
{
  const long long N = (long long)d->g.Xl * d->g.Y;
  if (d->copy_pending)
  {
    if (cudaEventQuery(d->ev_copied) == cudaSuccess) d->copy_pending = false;
    else
    {
      // an asynchronous snapshot is still on its way to the host out of d_mom_out: the import takes a second staging area
      // (4 N doubles: the largest import, rho_r, rho_b, u) instead of waiting, so that its host->device copy runs beside the
      // snapshot's device->host copy — PCIe is full duplex.  Out of memory: wait after all.
      cudaGetLastError();
      if (d->stage_in_busy) LBM_CUDA(cudaStreamWaitEvent(d->stream, d->ev_stage_free, 0));  // (an lbm_init_equilibrium's kernel may still read it)
      if (!d->d_stage_in && cudaMalloc(&d->d_stage_in, 4 * N * sizeof(double)) != cudaSuccess)
      {
        cudaGetLastError();
        d->d_stage_in = nullptr;
        LBM_CUDA(cudaEventSynchronize(d->ev_copied));
        d->copy_pending = false;
      }
      else
      {
        *out = d->d_stage_in;
        return LBM_OK;
      }
    }
  }
  if (!d->d_mom_out) LBM_CUDA(cudaMalloc(&d->d_mom_out, 6 * N * sizeof(double)));
  *out = d->d_mom_out;
  return LBM_OK;
}

// rho, u (and for two-phase models phase, rho_r, rho_b) of the current state into the staging buffer,
// on the domain's stream.  A copy still draining the buffer (lbm_snapshot_async) is waited for first.
int stage_fields(lbm_domain* d, int lattice)
{
  const long long N = (long long)d->g.Xl * d->g.Y;
  if (!d->d_mom_out) LBM_CUDA(cudaMalloc(&d->d_mom_out, 6 * N * sizeof(double)));
  if (!d->copy)
  {
    LBM_CUDA(cudaStreamCreateWithFlags(&d->copy, cudaStreamNonBlocking));
    LBM_CUDA(cudaEventCreateWithFlags(&d->ev_staged, cudaEventDisableTiming));
    LBM_CUDA(cudaEventCreateWithFlags(&d->ev_copied, cudaEventDisableTiming));
  }
  if (d->copy_pending) LBM_CUDA(cudaStreamWaitEvent(d->stream, d->ev_copied, 0));
  if (d->tp) return tp_stage_moments(d, d->d_mom_out);
  if (lattice == 0 && !d->post_stream)
  {
    // straight from the stored post-collision state: one pull-only pass that writes rho, u (72 B read + 24 B written
    // per node; no AoS scratch)
    LBM_TRY(step_rows(d));
    if (d->link_lo || d->link_hi) LBM_TRY(comm_link_refresh(d));
    else LBM_TRY(step_prologue(d, true, true));
    LBM_CUDA(cudaStreamWaitEvent(d->stream, d->ev_side, 0));
    LaunchArgs a{d->cur, d->cur ^ 1, d->d_rows_all, d->g.Xl, true, d->ibm.used_slot, d->stream};
    a.snap_rho = d->d_mom_out;
    a.snap_u = d->d_mom_out + N;
    return dispatch_bgk<MODE_PULL_ONLY>(d, a);
  }
  LBM_TRY(export_post_stream(d));
  int incompressible = 0;
  double sx = 0.0, sy = 0.0;
  if (d->cfg.model == LBM_MODEL_BGK)
  {
    incompressible = d->cfg.equilibrium == LBM_EQ_INCOMPRESSIBLE;
    if (d->cfg.force == LBM_FORCE_UNIFORM) { sx = d->cfg.Fg[0]; sy = d->cfg.Fg[1]; }
  }
  k_moments_aos<<<cdiv(N, 256), 256, 0, d->stream>>>(d->d_aos[lattice], N, incompressible, sx, sy, d->d_mom_out, d->d_mom_out + N);
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

}  // namespace lbm

using namespace lbm;

// ================================================================================================
// C ABI
// ================================================================================================
extern "C"
{

const char* lbm_last_error(void) { return g_error.c_str(); }
const char* lbm_version(void) { return "lbm_b200 0.1 (sm_100a, fp64 SoA, pull)"; }

void lbm_config_default(lbm_config* c)
{
  std::memset(c, 0, sizeof(*c));
  c->model = LBM_MODEL_BGK;
  c->equilibrium = LBM_EQ_COMPRESSIBLE;
  c->force = LBM_FORCE_NONE;
  c->omega = 1.0;
  c->omega_g = 1.0;
  c->delta = 0.1;
  c->sigma = 0.1;
}

void lbm_bc_op_default(lbm_bc_op* op)
{
  std::memset(op, 0, sizeof(*op));
  op->kind = LBM_BC_LINEAR;
  op->x_end = LBM_END;
  op->y_end = LBM_END;
  op->coef = 1.0;
  op->src_mode = LBM_SRC_SAME_NODE;
}

int lbm_create(const lbm_config* cfg, lbm_domain** out)
{
  if (!cfg || !out) { set_error("lbm_create: null argument"); return LBM_ERR_INVALID; }
  *out = nullptr;
  if (cfg->X < 3 || cfg->Y < 3) { set_error("lbm_create: grid %dx%d too small (need >= 3x3)", cfg->X, cfg->Y); return LBM_ERR_INVALID; }
  if (cfg->x0 < 0 || cfg->x1 > cfg->X || cfg->x1 <= cfg->x0) { set_error("lbm_create: bad slab rows [%d,%d) of %d", cfg->x0, cfg->x1, cfg->X); return LBM_ERR_INVALID; }
  if (cfg->model < LBM_MODEL_BGK || cfg->model > LBM_MODEL_MRT_CSF) { set_error("lbm_create: unknown model %d", cfg->model); return LBM_ERR_INVALID; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
  {
    set_error("lbm_create: no CUDA device (this library has no CPU fallback)");
    return LBM_ERR_CUDA;
  }
  if (cfg->device < 0 || cfg->device >= ndev) { set_error("lbm_create: device %d of %d", cfg->device, ndev); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(cfg->device));
  lbm_domain* d = new lbm_domain();
  d->cfg = *cfg;
  d->g.Xl = cfg->x1 - cfg->x0;
  d->g.Y = cfg->Y;
  d->g.pitch = ((cfg->Y + 15) / 16) * 16;
  d->g.xg0 = cfg->x0;
  d->g.plane = (long long)(d->g.Xl + 2) * d->g.pitch;
  d->nlat = (cfg->model == LBM_MODEL_BGK || cfg->model == LBM_MODEL_KBC) ? 1 : 2;
  if (d->nlat == 1 || cfg->model == LBM_MODEL_BGK_ADE)
  {
    // two nodes per thread: pairs (y, y+1), y even, 2 <= y and y + 2 <= Y - 1
    d->npairs = cfg->Y >= 5 ? (cfg->Y - 3) / 2 : 0;
    d->y_int_begin = 2;
    d->y_int_end = 2 + 2 * d->npairs;
  }
  else
  {
    // one node per thread: columns 1 .. Y-2
    d->npairs = 0;
    d->y_int_begin = 1;
    d->y_int_end = cfg->Y - 1;
  }
  const size_t bytes = ((size_t)9 * d->g.plane + (size_t)6 * d->g.Xl) * sizeof(double);  // nine planes + the face tail
  for (int l = 0; l < d->nlat; l++)
    for (int b = 0; b < 2; b++)
    {
      cudaError_t e = cudaMalloc(&d->buf[l][b], bytes);
      if (e != cudaSuccess)
      {
        set_error("lbm_create: cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
        lbm_destroy(d);
        return LBM_ERR_CUDA;
      }
      cudaMemset(d->buf[l][b], 0, bytes);
    }
  // streams and events: a failure here goes through lbm_destroy like the allocation failures above (no leaked slab)
  auto make_streams_and_events = [&]() -> int {
    LBM_CUDA(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
    // the side chain is a string of tiny kernels: give it priority so it slips in between the
    // blocks of the bulk launch instead of queueing behind them
    int lo = 0, hi = 0;
    LBM_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    LBM_CUDA(cudaStreamCreateWithPriority(&d->side, cudaStreamNonBlocking, hi));
    LBM_CUDA(cudaEventCreate(&d->ev_begin));
    LBM_CUDA(cudaEventCreate(&d->ev_end));
    for (cudaEvent_t* e : {&d->ev_ready, &d->ev_early, &d->ev_side, &d->ev_stage, &d->ev_packet, &d->ev_ibm, &d->ev_ibm_got})
      LBM_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    return LBM_OK;
  };
  if (int s = make_streams_and_events(); s != LBM_OK) { lbm_destroy(d); return s; }
  if (cfg->model == LBM_MODEL_MRTCG || cfg->model == LBM_MODEL_RK || cfg->model == LBM_MODEL_MRT_CSF)
  {
    int s = tp_create(d);
    if (s != LBM_OK) { lbm_destroy(d); return s; }
  }
  *out = d;
  return LBM_OK;
}

int lbm_destroy(lbm_domain* d)
{
  if (!d) return LBM_OK;
  cudaSetDevice(d->cfg.device);
  if (d->stream) cudaStreamSynchronize(d->stream);
  if (d->side) cudaStreamSynchronize(d->side);
  release_compiled(d);
  stats_release(d);
  faces_release(d);
  ibm_release(d);
  tp_destroy(d);
  comm_release(d);
  for (int l = 0; l < 2; l++)
  {
    for (int b = 0; b < 2; b++) cudaFree(d->buf[l][b]);
    cudaFree(d->d_aos[l]);
  }
  cudaFree(d->d_mom_out);
  cudaFree(d->d_stage_in);
  if (d->copyin)
  {
    cudaStreamSynchronize(d->copyin);
    cudaEventDestroy(d->ev_h2d);
    cudaEventDestroy(d->ev_stage_free);
    cudaStreamDestroy(d->copyin);
  }
  cudaFree(d->d_mom_in);
  if (d->copy)
  {
    cudaStreamSynchronize(d->copy);
    cudaEventDestroy(d->ev_staged);
    cudaEventDestroy(d->ev_copied);
    cudaStreamDestroy(d->copy);
  }
  for (int k = 0; k < 2; k++)
    if (d->graph_exec[k]) cudaGraphExecDestroy(d->graph_exec[k]);
  for (auto& r : d->prof)
  {
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  if (d->ev_begin) cudaEventDestroy(d->ev_begin);
  if (d->ev_end) cudaEventDestroy(d->ev_end);
  for (cudaEvent_t e : {d->ev_ready, d->ev_early, d->ev_side, d->ev_stage, d->ev_packet, d->ev_ibm, d->ev_ibm_got})
    if (e) cudaEventDestroy(e);
  cudaFree(d->d_rows_all); cudaFree(d->d_rows_early); cudaFree(d->d_rows_bulk);
  if (d->side) cudaStreamDestroy(d->side);
  if (d->stream) cudaStreamDestroy(d->stream);
  delete d;
  return LBM_OK;
}

// ---------------------------------------------------------------- boundary description
int lbm_bc_clear(lbm_domain* d)
{
  if (!d) { set_error("null domain"); return LBM_ERR_INVALID; }
  d->ops.clear();
  cudaSetDevice(d->cfg.device);
  release_compiled(d);
  return LBM_OK;
}

int lbm_bc_add(lbm_domain* d, const lbm_bc_op* op)
{
  if (!d || !op) { set_error("lbm_bc_add: null argument"); return LBM_ERR_INVALID; }
  if (op->kind < LBM_BC_LINEAR || op->kind > LBM_BC_COPY_PRE) { set_error("lbm_bc_add: unknown kind %d", op->kind); return LBM_ERR_INVALID; }
  if (op->lattice < -1 || op->lattice > 1) { set_error("lbm_bc_add: lattice %d", op->lattice); return LBM_ERR_INVALID; }
  StoredOp so;
  so.op = *op;
  if (op->kind == LBM_BC_ADE_INLET)
  {
    if (!op->per_row) { set_error("lbm_bc_add: LBM_BC_ADE_INLET needs per_row (C_w[X])"); return LBM_ERR_INVALID; }
    so.per_row.assign(op->per_row, op->per_row + d->cfg.X);
  }
  so.op.per_row = nullptr;
  d->ops.push_back(std::move(so));
  d->committed = false;
  return LBM_OK;
}

int lbm_bc_commit(lbm_domain* d)
{
  if (!d) { set_error("null domain"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  release_compiled(d);
  if (d->tp) return tp_commit(d);
  return commit_boundary_tables(d);
}

int lbm_bc_get_mask(lbm_domain* d, int lattice, int32_t* mask)
{
  if (!d || !mask || lattice < 0 || lattice >= d->nlat) { set_error("lbm_bc_get_mask: bad argument"); return LBM_ERR_INVALID; }
  if (!d->committed) { set_error("lbm_bc_get_mask: call lbm_bc_commit first"); return LBM_ERR_INVALID; }
  std::memcpy(mask, d->mask[lattice].data(), d->mask[lattice].size() * sizeof(int32_t));
  return LBM_OK;
}

// ---------------------------------------------------------------- state
int lbm_set_f(lbm_domain* d, int lattice, const double* f_aos)
{
  if (!d || !f_aos || lattice < 0 || lattice >= d->nlat) { set_error("lbm_set_f: bad argument"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  const long long N = (long long)d->g.Xl * d->g.Y;
  if (!d->post_stream && d->have_state)
  {
    // the other lattice (if any) is stored post-collision: bring the whole state back to post-stream first
    if (d->nlat > 1)
    {
      LBM_TRY(export_post_stream(d));
      for (int l = 0; l < d->nlat; l++)
      {
        k_import_aos<<<cdiv(N, 256), 256, 0, d->stream>>>(d->d_aos[l], d->buf[l][d->cur], d->g);
        d->launches++;
      }
    }
    d->post_stream = true;
  }
  LBM_TRY(ensure_aos_scratch(d));
  LBM_CUDA(cudaMemcpyAsync(d->d_aos[lattice], f_aos, N * 9 * sizeof(double), cudaMemcpyHostToDevice, d->stream));
  k_import_aos<<<cdiv(N, 256), 256, 0, d->stream>>>(d->d_aos[lattice], d->buf[lattice][d->cur], d->g);
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  d->post_stream = true;
  d->have_state = true;
  d->side_ready = false;
  d->mom_in_valid = false;
  if (d->tp) LBM_TRY(tp_refresh_moments(d));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  return LBM_OK;
}

int lbm_get_f(lbm_domain* d, int lattice, double* f_aos)
{
  if (!d || !f_aos || lattice < 0 || lattice >= d->nlat) { set_error("lbm_get_f: bad argument"); return LBM_ERR_INVALID; }
  if (!d->have_state) { set_error("lbm_get_f: no state (call lbm_set_f / lbm_init_* first)"); return LBM_ERR_INVALID; }
  if (!d->committed) { set_error("lbm_get_f: call lbm_bc_commit first"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_TRY(export_post_stream(d));
  const long long N = (long long)d->g.Xl * d->g.Y;
  LBM_CUDA(cudaMemcpyAsync(f_aos, d->d_aos[lattice], N * 9 * sizeof(double), cudaMemcpyDeviceToHost, d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  return LBM_OK;
}

int lbm_get_moments(lbm_domain* d, int lattice, double* rho, double* u)
{
  if (!d || lattice < 0 || lattice >= d->nlat) { set_error("lbm_get_moments: bad argument"); return LBM_ERR_INVALID; }
  if (!d->have_state || !d->committed) { set_error("lbm_get_moments: no state or boundary rules not committed"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_TRY(stage_fields(d, lattice));
  const long long N = (long long)d->g.Xl * d->g.Y;
  if (rho) LBM_CUDA(cudaMemcpyAsync(rho, d->d_mom_out, N * sizeof(double), cudaMemcpyDeviceToHost, d->stream));
  if (u) LBM_CUDA(cudaMemcpyAsync(u, d->d_mom_out + N, 2 * N * sizeof(double), cudaMemcpyDeviceToHost, d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  return LBM_OK;
}

// Snapshot without stalling the time loop: the fields are staged on the domain's stream, the
// device->host copies run on a separate copy stream under the following steps.
int lbm_snapshot_async(lbm_domain* d, int lattice, double* rho, double* u, double* phase)
{
  if (!d || lattice < 0 || lattice >= d->nlat) { set_error("lbm_snapshot_async: bad argument"); return LBM_ERR_INVALID; }
  if (!d->have_state || !d->committed) { set_error("lbm_snapshot_async: no state or boundary rules not committed"); return LBM_ERR_INVALID; }
  if (phase && !d->tp) { set_error("lbm_snapshot_async: phase is a two-phase field"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_TRY(stage_fields(d, lattice));
  const long long N = (long long)d->g.Xl * d->g.Y;
  LBM_CUDA(cudaEventRecord(d->ev_staged, d->stream));
  LBM_CUDA(cudaStreamWaitEvent(d->copy, d->ev_staged, 0));
  if (rho) LBM_CUDA(cudaMemcpyAsync(rho, d->d_mom_out, N * sizeof(double), cudaMemcpyDeviceToHost, d->copy));
  if (u) LBM_CUDA(cudaMemcpyAsync(u, d->d_mom_out + N, 2 * N * sizeof(double), cudaMemcpyDeviceToHost, d->copy));
  if (phase) LBM_CUDA(cudaMemcpyAsync(phase, d->d_mom_out + 3 * N, N * sizeof(double), cudaMemcpyDeviceToHost, d->copy));
  LBM_CUDA(cudaEventRecord(d->ev_copied, d->copy));
  d->copy_pending = true;
  return LBM_OK;
}

int lbm_snapshot_wait(lbm_domain* d)
{
  if (!d) { set_error("null domain"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  if (d->copy_pending) LBM_CUDA(cudaEventSynchronize(d->ev_copied));
  d->copy_pending = false;
  return LBM_OK;
}

int lbm_init_equilibrium(lbm_domain* d, int lattice, int eq_kind, const double* rho, const double* u)
{
  if (!d || !rho || !u || lattice < 0 || lattice >= d->nlat) { set_error("lbm_init_equilibrium: bad argument"); return LBM_ERR_INVALID; }
  if (d->tp) { set_error("lbm_init_equilibrium: use lbm_init_two_phase for two-phase models"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  const long long N = (long long)d->g.Xl * d->g.Y;
  if (eq_kind < LBM_EQ_COMPRESSIBLE || eq_kind > LBM_EQ_KBC_FRESH) { set_error("lbm_init_equilibrium: unknown equilibrium kind %d", eq_kind); return LBM_ERR_INVALID; }
  // The host->device copy runs on its own stream into an import staging area, so that it overlaps whatever the domain's
  // stream is still doing (the previous run's steps, a snapshot's staging) — a driver that feeds one initial state after
  // the other keeps the copy engine, the SMs and the snapshot's device->host copy busy at once.  The call returns when the
  // HOST buffers have been consumed; the equilibrium kernel is ordered behind both the copy and the stream's earlier work.
  if (!d->copyin)
  {
    LBM_CUDA(cudaStreamCreateWithFlags(&d->copyin, cudaStreamNonBlocking));
    LBM_CUDA(cudaEventCreateWithFlags(&d->ev_h2d, cudaEventDisableTiming));
    LBM_CUDA(cudaEventCreateWithFlags(&d->ev_stage_free, cudaEventDisableTiming));
  }
  if (!d->d_stage_in) LBM_CUDA(cudaMalloc(&d->d_stage_in, 4 * N * sizeof(double)));
  double *d_rho = d->d_stage_in, *d_u = d->d_stage_in + N;
  if (d->stage_in_busy) LBM_CUDA(cudaStreamWaitEvent(d->copyin, d->ev_stage_free, 0));  // the previous import's kernel has read the area
  LBM_CUDA(cudaMemcpyAsync(d_rho, rho, N * sizeof(double), cudaMemcpyHostToDevice, d->copyin));
  LBM_CUDA(cudaMemcpyAsync(d_u, u, 2 * N * sizeof(double), cudaMemcpyHostToDevice, d->copyin));
  LBM_CUDA(cudaEventRecord(d->ev_h2d, d->copyin));
  LBM_CUDA(cudaStreamWaitEvent(d->stream, d->ev_h2d, 0));
  k_init_equilibrium<<<cdiv(N, 256), 256, 0, d->stream>>>(d->buf[lattice][d->cur], d->g, eq_kind, d_rho, d_u);
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  LBM_CUDA(cudaEventRecord(d->ev_stage_free, d->stream));
  d->stage_in_busy = true;
  LBM_CUDA(cudaEventSynchronize(d->ev_h2d));
  d->post_stream = true;
  d->have_state = true;
  d->side_ready = false;
  d->mom_in_valid = false;
  return LBM_OK;
}

// ulbm drivers keep m0 / m1 as members that the first collide() reads before they are recomputed from the
// populations (test/ulbm_poiseuille.cpp:93: adve_f = 0, m0 = 1, m1 = 0): the first step after an import
// takes these fields instead of the moments of the imported populations.
int lbm_set_moments(lbm_domain* d, const double* rho, const double* u)
{
  if (!d || !rho || !u) { set_error("lbm_set_moments: null argument"); return LBM_ERR_INVALID; }
  if (d->cfg.model != LBM_MODEL_KBC) { set_error("lbm_set_moments: only LBM_MODEL_KBC carries m0 / m1 into its first collision"); return LBM_ERR_UNSUPPORTED; }
  if (!d->have_state || !d->post_stream) { set_error("lbm_set_moments: import the populations first (lbm_set_f / lbm_init_equilibrium)"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  const long long N = (long long)d->g.Xl * d->g.Y;
  if (!d->d_mom_in) LBM_CUDA(cudaMalloc(&d->d_mom_in, 3 * N * sizeof(double)));
  LBM_CUDA(cudaMemcpyAsync(d->d_mom_in, rho, N * sizeof(double), cudaMemcpyHostToDevice, d->stream));
  LBM_CUDA(cudaMemcpyAsync(d->d_mom_in + N, u, 2 * N * sizeof(double), cudaMemcpyHostToDevice, d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  d->mom_in_valid = true;
  return LBM_OK;
}

// ---------------------------------------------------------------- stepping
static int step_once(lbm_domain* d)
{
  if (d->tp && (d->link_lo || d->link_hi))
  {
    set_error("lbm_step: this slab is linked to neighbours; advance the set with lbm_step_group");
    return LBM_ERR_INVALID;
  }
  return d->tp ? tp_step(d) : bgk_step_once(d);
}

// One steady-state step PAIR captured into a CUDA graph (a pair returns every A/B toggle — buffers,
// listed-node moments, IBM force slots — to where it started, so the graph replays as is).  For the
// launch-bound small grids: ~12 launches on two streams per step become one graph launch per two steps.
static int capture_pair(lbm_domain* d)
{
  const int k = d->cur;
  if (d->graph_exec[k]) return LBM_OK;
  const long long launches0 = d->launches;
  cudaGraph_t graph = nullptr;
  LBM_CUDA(cudaStreamBeginCapture(d->stream, cudaStreamCaptureModeThreadLocal));
  int s = LBM_OK;
  for (int i = 0; i < 2 && s == LBM_OK; i++)
  {
    d->skip_side_wait = (i == 0) && !d->tp;  // the side chain of the step before the pair is joined outside the graph
    s = step_once(d);
  }
  d->skip_side_wait = false;
  // join the side stream (captured through ev_early) back into the origin stream
  if (s == LBM_OK && !d->tp && cudaStreamWaitEvent(d->stream, d->ev_side, 0) != cudaSuccess) s = LBM_ERR_CUDA;
  cudaError_t e = cudaStreamEndCapture(d->stream, &graph);
  if (s != LBM_OK || e != cudaSuccess)
  {
    if (graph) cudaGraphDestroy(graph);
    if (s == LBM_OK) set_error("cudaStreamEndCapture failed: %s", cudaGetErrorString(e));
    cudaGetLastError();
    return s != LBM_OK ? s : LBM_ERR_CUDA;
  }
  e = cudaGraphInstantiate(&d->graph_exec[k], graph, 0);
  cudaGraphDestroy(graph);
  if (e != cudaSuccess) { set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(e)); return LBM_ERR_CUDA; }
  d->graph_launches[k] = d->launches - launches0;
  d->launches = launches0;  // nothing ran yet
  return LBM_OK;
}

static bool graph_eligible(const lbm_domain* d)
{
  return d->use_graph && !d->profiling && !comm_active(d) && !d->link_lo && !d->link_hi;
}

int lbm_step(lbm_domain* d, int n_steps)
{
  if (!d || n_steps < 0) { set_error("lbm_step: bad argument"); return LBM_ERR_INVALID; }
  if (!d->have_state) { set_error("lbm_step: no state (call lbm_set_f / lbm_init_* first)"); return LBM_ERR_INVALID; }
  if (!d->committed) { set_error("lbm_step: call lbm_bc_commit first"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaEventRecord(d->ev_begin, d->stream));
  int s = 0;
  if (graph_eligible(d) && n_steps >= 4)
  {
    // reach the steady state (post-collision storage, side chain prepared, row lists built) with plain steps
    while (s < n_steps && (d->post_stream || (!d->tp && !d->side_ready))) { LBM_TRY(step_once(d)); s++; }
    if (n_steps - s >= 2)
    {
      if (!d->tp)
      {
        // everything the side stream still owes the current buffer, joined outside the graph
        LBM_CUDA(cudaEventRecord(d->ev_ready, d->side));
        LBM_CUDA(cudaStreamWaitEvent(d->stream, d->ev_ready, 0));
      }
      LBM_TRY(capture_pair(d));
      const int k = d->cur;
      for (; n_steps - s >= 2; s += 2)
      {
        LBM_CUDA(cudaGraphLaunch(d->graph_exec[k], d->stream));
        d->launches += d->graph_launches[k];
      }
      // events last recorded inside the capture must not be waited on by plain steps: re-record them here
      if (!d->tp) LBM_CUDA(cudaEventRecord(d->ev_side, d->stream));
    }
  }
  if (d->tp && comm_active(d) && !(d->link_lo || d->link_hi))
  {
    // ring ranks: the first step after an import in line, the others with their halo exchanges behind the interior bands
    while (s < n_steps && d->post_stream) { LBM_TRY(step_once(d)); s++; }
    if (n_steps - s >= 2 && tp_ring_overlap_ok(d))
    {
      LBM_TRY(tp_steps_ring(d, n_steps - s));
      s = n_steps;
    }
  }
  for (; s < n_steps; s++) LBM_TRY(step_once(d));
  LBM_CUDA(cudaEventRecord(d->ev_end, d->stream));
  return LBM_OK;
}

int lbm_synchronize(lbm_domain* d)
{
  if (!d) { set_error("null domain"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  // the tail of the last step's side chain (ghost rows, the next step's IBM pre-pass) and a pending snapshot copy
  if (d->side) LBM_CUDA(cudaStreamSynchronize(d->side));
  if (d->copy) LBM_CUDA(cudaStreamSynchronize(d->copy));
  return LBM_OK;
}

int lbm_last_step_ms(lbm_domain* d, float* ms)
{
  if (!d || !ms) { set_error("lbm_last_step_ms: bad argument"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaEventSynchronize(d->ev_end));
  LBM_CUDA(cudaEventElapsedTime(ms, d->ev_begin, d->ev_end));
  return LBM_OK;
}

int lbm_kernel_launches(lbm_domain* d, long long* n)
{
  if (!d || !n) { set_error("lbm_kernel_launches: bad argument"); return LBM_ERR_INVALID; }
  *n = d->launches;
  return LBM_OK;
}

int lbm_get_stream(lbm_domain* d, void** stream)
{
  if (!d || !stream) { set_error("lbm_get_stream: bad argument"); return LBM_ERR_INVALID; }
  *stream = (void*)d->stream;
  return LBM_OK;
}

int lbm_use_graph(lbm_domain* d, int enable)
{
  if (!d) { set_error("null domain"); return LBM_ERR_INVALID; }
  d->use_graph = enable != 0;
  if (!d->use_graph)
  {
    cudaSetDevice(d->cfg.device);
    cudaStreamSynchronize(d->stream);
    drop_graphs(d);
  }
  return LBM_OK;
}

int lbm_profile_enable(lbm_domain* d, int enable)
{
  if (!d) { set_error("null domain"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  d->profiling = enable != 0;
  d->prof_used = 0;
  return LBM_OK;
}

int lbm_profile_read(lbm_domain* d, int cls, double* total_ms, long long* launches)
{
  if (!d || !total_ms || !launches || cls < 0 || cls >= LBM_PROF_CLASSES) { set_error("lbm_profile_read: bad argument"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  double sum = 0.0;
  long long n = 0;
  for (size_t i = 0; i < d->prof_used; i++)
  {
    if (d->prof[i].cls != cls) continue;
    float ms = 0.f;
    LBM_CUDA(cudaEventElapsedTime(&ms, d->prof[i].a, d->prof[i].b));
    sum += ms;
    n++;
  }
  *total_ms = sum;
  *launches = n;
  return LBM_OK;
}

int lbm_row_split(lbm_domain* d, int* n_early_rows, int* n_bulk_rows)
{
  if (!d || !n_early_rows || !n_bulk_rows) { set_error("lbm_row_split: null argument"); return LBM_ERR_INVALID; }
  if (d->tp) { set_error("lbm_row_split: the two-phase models march row bands, they have no early / bulk split"); return LBM_ERR_UNSUPPORTED; }
  if (!d->committed) { set_error("lbm_row_split: call lbm_bc_commit first"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_TRY(step_rows(d));
  *n_early_rows = d->n_early;
  *n_bulk_rows = d->n_bulk;
  return LBM_OK;
}

int lbm_decompose_rows(int X, int n_ranks, int rank, int* x0, int* x1)
{
  if (X <= 0 || n_ranks <= 0 || rank < 0 || rank >= n_ranks || !x0 || !x1) { set_error("lbm_decompose_rows: bad argument"); return LBM_ERR_INVALID; }
  // contiguous slabs along axis 0; the first X % n_ranks slabs get one extra row
  const int base = X / n_ranks, rem = X % n_ranks;
  *x0 = rank * base + std::min(rank, rem);
  *x1 = *x0 + base + (rank < rem ? 1 : 0);
  return LBM_OK;
}

}  // extern "C"

// lbm_body_force_record / _read / _stop and their kernels
#include "lbm_body_force.cuh"
// lbm_stats_start / _read / _stop and their kernels
#include "lbm_stats.cuh"
