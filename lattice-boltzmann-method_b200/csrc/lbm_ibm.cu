// lbm_ibm.cu — immersed boundary (multi-direct forcing) kept on the device.
//
// Replaces class ibm / struct marker (src/ibm.hpp:9-34, src/ibm.cpp:15-190).  The reference walks
// the markers sequentially and does ~8 tiny tensor ops per marker and forcing iteration.  Here:
//   k_ibm_gather : one thread per marker — interpolate u, rho over its 4x4 box, fj = -2 rho_j u_j
//   k_ibm_spread : one thread per ROI node — sum phi * fj over the markers that cover the node,
//                  IN MARKER ORDER (a node->markers list built once on the host), so the fp64
//                  summation order of the reference's sequential scatter is reproduced without
//                  atomics; then u += F_n / (2 rho), F += F_n.
// The Peskin 4-point weights are static and computed once on the host exactly like
// marker::set_box (src/ibm.cpp:21-57), including its pairing of the stencil's first row with the
// x distance and of k % 4 with the column offset of the box.
#include <algorithm>
#include <cmath>

#include "lbm_internal.hpp"

namespace lbm
{

static inline int cdiv(long long a, int b) { return (int)((a + b - 1) / b); }

// src/ibm.cpp:39-45
static double peskin(double r_)
{
  const double r = std::fabs(r_);
  if (r <= 1) return 0.125 * (3.0 - 2.0 * r + std::sqrt(1.0 + 4.0 * r - 4.0 * r * r));
  else if (r <= 2) return 0.125 * (5.0 - 2.0 * r - std::sqrt(-7.0 + 12.0 * r - 4.0 * r * r));
  return 0.0;
}

// moments of the ROI nodes from the stored populations (ROI nodes are interior: plain pull)
// Only the nodes some marker's 4x4 box covers are ever read (gather) or changed (spread), so the
// pre-pass runs over that short "active" list, not over the whole ROI rectangle.
template <int MODE, int EQ>
__global__ void k_ibm_roi_moments(const double* __restrict__ f, const SlabGeom g, int r0, int c0, int na, int RC,
                                  const int* __restrict__ active, double* __restrict__ u, double* __restrict__ rho)
{
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= na) return;  // active already points at this slab's part of the list
  const int n = active[a];
  const int i = n / RC, j = n % RC;
  const int x = r0 + i - g.xg0, y = c0 + j;
  double v[9];
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    if constexpr (MODE == MODE_LOCAL) v[q] = f[q * g.plane + node_off(g, x, y)];
    else v[q] = f[q * g.plane + node_off(g, x - CX(q), y - CY(q))];
  }
  double r, jx, jy;
  moments(v, r, jx, jy);
  rho[n] = r;
  u[2 * n] = EQ == EQ_COMP ? jx / r : jx;
  u[2 * n + 1] = EQ == EQ_COMP ? jy / r : jy;
}

// src/ibm.cpp:170-177
__global__ void k_ibm_gather(int nm, const int* __restrict__ mrow, const int* __restrict__ mcol,
                             const double* __restrict__ phi, int RC, const double* __restrict__ u,
                             const double* __restrict__ rho, double* __restrict__ fj)
{
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= nm) return;
  double ujx = 0.0, ujy = 0.0, rj = 0.0;
#pragma unroll
  for (int k = 0; k < 16; k++)
  {
    const int n = (mrow[m] + k / 4) * RC + (mcol[m] + k % 4);
    const double w = phi[16 * m + k];
    ujx += w * u[2 * n];
    ujy += w * u[2 * n + 1];
    rj += w * rho[n];
  }
  fj[2 * m] = -2.0 * rj * ujx;
  fj[2 * m + 1] = -2.0 * rj * ujy;
}

// src/ibm.cpp:180-186
__global__ void k_ibm_spread(int na, const int* __restrict__ active, const int* __restrict__ ptr,
                             const int* __restrict__ em, const double* __restrict__ ephi, const double* __restrict__ fj,
                             double* __restrict__ u, const double* __restrict__ rho, double* __restrict__ Fx,
                             double* __restrict__ Fy, int first)
{
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= na) return;
  const int n = active[a];
  double fx = 0.0, fy = 0.0;
  for (int e = ptr[a]; e < ptr[a + 1]; e++)
  {
    fx += ephi[e] * fj[2 * em[e]];
    fy += ephi[e] * fj[2 * em[e] + 1];
  }
  u[2 * n] += 0.5 * fx / rho[n];
  u[2 * n + 1] += 0.5 * fy / rho[n];
  Fx[n] = first ? fx : Fx[n] + fx;
  Fy[n] = first ? fy : Fy[n] + fy;
}

__global__ void k_ibm_load_roi(const double* __restrict__ u_aos, const double* __restrict__ rho_aos, int Y, int r0,
                               int c0, int RR, int RC, double* __restrict__ u, double* __restrict__ rho)
{
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= RR * RC) return;
  const long long gidx = (long long)(r0 + n / RC) * Y + (c0 + n % RC);
  u[2 * n] = u_aos[2 * gidx];
  u[2 * n + 1] = u_aos[2 * gidx + 1];
  rho[n] = rho_aos[gidx];
}

__global__ void k_ibm_pack_force(int nn, const double* __restrict__ Fx, const double* __restrict__ Fy,
                                 double* __restrict__ F_aos)
{
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= nn) return;
  F_aos[2 * n] = Fx[n];
  F_aos[2 * n + 1] = Fy[n];
}

int ibm_release(lbm_domain* d)
{
  IbmState& ib = d->ibm;
  if (d->bf.on && d->bf.immersed) body_force_release(d);  // it reads the active list and force fields freed here
  cudaFree(ib.d_active); cudaFree(ib.d_mrow); cudaFree(ib.d_mcol); cudaFree(ib.d_phi); cudaFree(ib.d_fj); cudaFree(ib.d_ptr);
  cudaFree(ib.d_ent_marker); cudaFree(ib.d_ent_phi); cudaFree(ib.d_u); cudaFree(ib.d_rho);
  for (int k = 0; k < 2; k++) { cudaFree(ib.d_Fx[k]); cudaFree(ib.d_Fy[k]); }
  ib = IbmState();
  return LBM_OK;
}

// the four forcing iterations n = 1 .. m_max-1 on the ROI copies (src/ibm.cpp:166-187)
int ibm_iterate(lbm_domain* d, int slot, cudaStream_t st)
{
  IbmState& ib = d->ibm;
  const int RC = (int)(ib.c1 - ib.c0), nn = (int)(ib.r1 - ib.r0) * RC;
  if (ib.m_max <= 1)
  {
    LBM_CUDA(cudaMemsetAsync(ib.d_Fx[slot], 0, sizeof(double) * nn, st));
    LBM_CUDA(cudaMemsetAsync(ib.d_Fy[slot], 0, sizeof(double) * nn, st));
  }
  for (int n = 1; n < ib.m_max; n++)
  {
    k_ibm_gather<<<cdiv(ib.n_markers, 128), 128, 0, st>>>(ib.n_markers, ib.d_mrow, ib.d_mcol, ib.d_phi, RC, ib.d_u, ib.d_rho, ib.d_fj);
    k_ibm_spread<<<cdiv(ib.n_active, 128), 128, 0, st>>>(ib.n_active, ib.d_active, ib.d_ptr, ib.d_ent_marker, ib.d_ent_phi, ib.d_fj,
                                                         ib.d_u, ib.d_rho, ib.d_Fx[slot], ib.d_Fy[slot], n == 1 ? 1 : 0);
    d->launches += 2;
  }
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

// u, rho of the active ROI nodes on this slab's rows, from buffer `which` (mode: how that buffer is to be read)
int ibm_roi_local(lbm_domain* d, int mode, int which, cudaStream_t st)
{
  IbmState& ib = d->ibm;
  const int RC = (int)(ib.c1 - ib.c0), na = ib.a_hi - ib.a_lo;
  if (na <= 0) return LBM_OK;
  const double* f = d->buf[0][which];
  const bool comp = d->cfg.equilibrium == LBM_EQ_COMPRESSIBLE;
#define LBM_ROI(M, E)                                                                                                         \
  k_ibm_roi_moments<M, E><<<cdiv(na, 128), 128, 0, st>>>(f, d->g, (int)ib.r0, (int)ib.c0, na, RC, ib.d_active + ib.a_lo, ib.d_u, ib.d_rho)
  if (mode == MODE_LOCAL) { if (comp) LBM_ROI(MODE_LOCAL, EQ_COMP); else LBM_ROI(MODE_LOCAL, EQ_INCOMP); }
  else { if (comp) LBM_ROI(MODE_PULL, EQ_COMP); else LBM_ROI(MODE_PULL, EQ_INCOMP); }
#undef LBM_ROI
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

// force field for the step that will read buffer `which`: one slab per process (lbm_step).  Linked slabs of one
// process go through lbm_step_group, which runs the three phases itself with event-ordered copies in between.
int ibm_prepass(lbm_domain* d, int mode, int which, int slot, cudaStream_t st)
{
  LBM_TRY(ibm_roi_local(d, mode, which, st));
  if (d->ibm.split)
  {
    if (!comm_active(d))
    {
      set_error("immersed boundary across a slab cut: advance the slabs with lbm_step_group or join them with lbm_comm_init");
      return LBM_ERR_INVALID;
    }
    LBM_TRY(comm_ibm_share(d, st));
  }
  return ibm_iterate(d, slot, st);
}

}  // namespace lbm

using namespace lbm;

extern "C"
{

int lbm_ibm_set_markers(lbm_domain* d, const double* xs, const double* ys, int n, int m_max)
{
  if (!d || !xs || !ys || n <= 0 || m_max < 1) { set_error("lbm_ibm_set_markers: bad argument"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  ibm_release(d);
  d->ibm_given = IbmGiven();
  d->ics2 = 1.0 / 3.0;  // cylinder_test.cpp:112-113
  d->ics4 = 1.0 / 9.0;
  IbmState& ib = d->ibm;
  // ROI: src/ibm.cpp:122-156
  long r_min = 1000000, r_max = 0, c_min = 1000000, c_max = 0;
  for (int i = 0; i < n; i++)
  {
    if (r_min > (int)(std::floor(xs[i]) - 2)) r_min = (int)(std::floor(xs[i]) - 2);
    if (r_max < (int)(std::floor(xs[i]) + 2)) r_max = (int)(std::floor(xs[i]) + 2);
    if (c_min > (int)(std::floor(ys[i]) - 2)) c_min = (int)(std::floor(ys[i]) - 2);
    if (c_max < (int)(std::floor(ys[i]) + 2)) c_max = (int)(std::floor(ys[i]) + 2);
  }
  ib.r0 = r_min; ib.r1 = r_max + 1; ib.c0 = c_min; ib.c1 = c_max + 1;
  ib.n_markers = n;
  {
    // FNV-1a over the coordinates as given: lbm_comm_check compares it across the ring
    unsigned long long h = 1469598103934665603ull;
    auto eat = [&](const double* a) {
      const unsigned char* b = reinterpret_cast<const unsigned char*>(a);
      for (size_t k = 0; k < sizeof(double) * (size_t)n; k++) { h ^= b[k]; h *= 1099511628211ull; }
    };
    eat(xs);
    eat(ys);
    d->ibm_given.n = n;
    d->ibm_given.r0 = ib.r0;
    d->ibm_given.r1 = ib.r1;
    d->ibm_given.hash = h;
  }
  ib.m_max = m_max;
  const int y_int_end = d->y_int_end;
  if (ib.r0 < 0 || ib.r1 > d->cfg.X || ib.c0 < d->y_int_begin || ib.c1 > y_int_end)
  {
    set_error("lbm_ibm_set_markers: ROI rows [%ld,%ld) cols [%ld,%ld) must lie inside the grid's rows [0,%d) and interior columns [2,%d)",
              ib.r0, ib.r1, ib.c0, ib.c1, d->cfg.X, y_int_end);
    ib = IbmState();
    d->ibm_given = IbmGiven();
    return LBM_ERR_UNSUPPORTED;
  }
  if (ib.r1 <= d->cfg.x0 || ib.r0 >= d->cfg.x1)
  {
    // the body lies on other slabs: nothing to do here (every slab may be handed the same marker list)
    ib = IbmState();
    d->rows_dirty = true;
    d->side_ready = false;
    drop_graphs(d);
    return LBM_OK;
  }
  ib.split = ib.r0 < d->cfg.x0 || ib.r1 > d->cfg.x1;
  ib.row_lo = (int)(std::max<long>(ib.r0, d->cfg.x0) - ib.r0);
  ib.row_hi = (int)(std::min<long>(ib.r1, d->cfg.x1) - ib.r0);
  const int RR = (int)(ib.r1 - ib.r0), RC = (int)(ib.c1 - ib.c0), nn = RR * RC;
  std::vector<int> mrow(n), mcol(n);
  std::vector<double> phi((size_t)n * 16);
  std::vector<std::vector<std::pair<int, double>>> cover(nn);
  for (int i = 0; i < n; i++)
  {
    const double x = xs[i] - (double)ib.r0, y = ys[i] - (double)ib.c0;  // marker(x_m - r_off, y_m - c_off), src/ibm.cpp:101
    mrow[i] = (int)((long)std::floor(x) - 1);
    mcol[i] = (int)((long)std::floor(y) - 1);
    for (int k = 0; k < 16; k++)
    {
      const double sx = x - ((double)(k % 4) + std::floor(x) - 1.0);
      const double sy = y - ((double)(k / 4) + std::floor(y) - 1.0);
      phi[(size_t)i * 16 + k] = peskin(sx) * peskin(sy);
      const int node = (mrow[i] + k / 4) * RC + (mcol[i] + k % 4);
      cover[node].push_back({i, phi[(size_t)i * 16 + k]});  // markers arrive in increasing order
    }
  }
  std::vector<int> ptr, em, active;
  std::vector<double> ephi;
  for (int node = 0; node < nn; node++)
  {
    if (cover[node].empty()) continue;
    active.push_back(node);
    ptr.push_back((int)em.size());
    for (auto& c : cover[node]) { em.push_back(c.first); ephi.push_back(c.second); }
  }
  ptr.push_back((int)em.size());
  ib.n_active = (int)active.size();
  // the active list is sorted by node id (row-major), so the nodes on this slab's rows are one contiguous range
  ib.a_lo = (int)(std::lower_bound(active.begin(), active.end(), ib.row_lo * RC) - active.begin());
  ib.a_hi = (int)(std::lower_bound(active.begin(), active.end(), ib.row_hi * RC) - active.begin());
  LBM_CUDA(cudaMalloc(&ib.d_mrow, sizeof(int) * n));
  LBM_CUDA(cudaMalloc(&ib.d_mcol, sizeof(int) * n));
  LBM_CUDA(cudaMalloc(&ib.d_phi, sizeof(double) * n * 16));
  LBM_CUDA(cudaMalloc(&ib.d_fj, sizeof(double) * n * 2));
  LBM_CUDA(cudaMalloc(&ib.d_ptr, sizeof(int) * ptr.size()));
  LBM_CUDA(cudaMalloc(&ib.d_active, sizeof(int) * std::max<size_t>(active.size(), 1)));
  LBM_CUDA(cudaMemcpy(ib.d_active, active.data(), sizeof(int) * active.size(), cudaMemcpyHostToDevice));
  LBM_CUDA(cudaMalloc(&ib.d_ent_marker, sizeof(int) * std::max<size_t>(em.size(), 1)));
  LBM_CUDA(cudaMalloc(&ib.d_ent_phi, sizeof(double) * std::max<size_t>(em.size(), 1)));
  LBM_CUDA(cudaMalloc(&ib.d_u, sizeof(double) * nn * 2));
  LBM_CUDA(cudaMalloc(&ib.d_rho, sizeof(double) * nn));
  LBM_CUDA(cudaMemset(ib.d_u, 0, sizeof(double) * nn * 2));
  LBM_CUDA(cudaMemset(ib.d_rho, 0, sizeof(double) * nn));
  for (int k = 0; k < 2; k++)
  {
    LBM_CUDA(cudaMalloc(&ib.d_Fx[k], sizeof(double) * nn));
    LBM_CUDA(cudaMalloc(&ib.d_Fy[k], sizeof(double) * nn));
    LBM_CUDA(cudaMemset(ib.d_Fx[k], 0, sizeof(double) * nn));
    LBM_CUDA(cudaMemset(ib.d_Fy[k], 0, sizeof(double) * nn));
  }
  LBM_CUDA(cudaMemcpy(ib.d_mrow, mrow.data(), sizeof(int) * n, cudaMemcpyHostToDevice));
  LBM_CUDA(cudaMemcpy(ib.d_mcol, mcol.data(), sizeof(int) * n, cudaMemcpyHostToDevice));
  LBM_CUDA(cudaMemcpy(ib.d_phi, phi.data(), sizeof(double) * n * 16, cudaMemcpyHostToDevice));
  LBM_CUDA(cudaMemcpy(ib.d_ptr, ptr.data(), sizeof(int) * ptr.size(), cudaMemcpyHostToDevice));
  LBM_CUDA(cudaMemcpy(ib.d_ent_marker, em.data(), sizeof(int) * em.size(), cudaMemcpyHostToDevice));
  LBM_CUDA(cudaMemcpy(ib.d_ent_phi, ephi.data(), sizeof(double) * ephi.size(), cudaMemcpyHostToDevice));
  ib.enabled = true;
  d->rows_dirty = true;
  d->side_ready = false;
  drop_graphs(d);
  return LBM_OK;
}

// torch::indexing::Slice(b, e) over n entries (negative = from the end, LBM_END = None, clamped)
static void clamp_slice(int b, int e, int n, long& lo, long& hi)
{
  lo = b < 0 ? b + n : b;
  hi = e == LBM_END ? n : (e < 0 ? e + n : e);
  lo = std::min<long>(std::max<long>(lo, 0), n);
  hi = std::min<long>(std::max<long>(hi, lo), n);
}

int lbm_set_force_region(lbm_domain* d, int x_begin, int x_end, int y_begin, int y_end, double Fx, double Fy, double ics2, double ics4)
{
  if (!d) { set_error("lbm_set_force_region: null domain"); return LBM_ERR_INVALID; }
  if (d->cfg.force != LBM_FORCE_IBM || d->tp || d->cfg.model == LBM_MODEL_KBC)
  {
    set_error("lbm_set_force_region: the region force uses the force-field slot of the BGK kernels (create the domain with force = LBM_FORCE_IBM)");
    return LBM_ERR_INVALID;
  }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->side));
  ibm_release(d);
  IbmState& ib = d->ibm;
  clamp_slice(x_begin, x_end, d->cfg.X, ib.r0, ib.r1);
  clamp_slice(y_begin, y_end, d->cfg.Y, ib.c0, ib.c1);
  const size_t nn = (size_t)(ib.r1 - ib.r0) * (size_t)(ib.c1 - ib.c0);
  if (nn == 0) { ib = IbmState(); return LBM_OK; }
  std::vector<double> hx(nn, Fx), hy(nn, Fy);
  for (int k = 0; k < 2; k++)
  {
    LBM_CUDA(cudaMalloc(&ib.d_Fx[k], sizeof(double) * nn));
    LBM_CUDA(cudaMalloc(&ib.d_Fy[k], sizeof(double) * nn));
    LBM_CUDA(cudaMemcpy(ib.d_Fx[k], hx.data(), sizeof(double) * nn, cudaMemcpyHostToDevice));
    LBM_CUDA(cudaMemcpy(ib.d_Fy[k], hy.data(), sizeof(double) * nn, cudaMemcpyHostToDevice));
  }
  ib.fixed = true;
  ib.enabled = true;
  d->ics2 = ics2;
  d->ics4 = ics4;
  d->rows_dirty = true;
  d->side_ready = false;
  drop_graphs(d);
  return LBM_OK;
}

int lbm_ibm_get_roi(lbm_domain* d, long* roi)
{
  if (!d || !roi || !d->ibm.enabled) { set_error("lbm_ibm_get_roi: no immersed boundary"); return LBM_ERR_INVALID; }
  roi[0] = d->ibm.r0; roi[1] = d->ibm.r1; roi[2] = d->ibm.c0; roi[3] = d->ibm.c1;
  return LBM_OK;
}

static int ibm_download_force(lbm_domain* d, double* F_aos, int slot)
{
  IbmState& ib = d->ibm;
  const int nn = (int)((ib.r1 - ib.r0) * (ib.c1 - ib.c0));
  double* tmp = nullptr;
  LBM_CUDA(cudaMalloc(&tmp, sizeof(double) * 2 * nn));
  k_ibm_pack_force<<<cdiv(nn, 128), 128, 0, d->stream>>>(nn, ib.d_Fx[slot], ib.d_Fy[slot], tmp);
  d->launches++;
  LBM_CUDA(cudaMemcpyAsync(F_aos, tmp, sizeof(double) * 2 * nn, cudaMemcpyDeviceToHost, d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  cudaFree(tmp);
  return LBM_OK;
}

int lbm_ibm_get_force(lbm_domain* d, double* F_aos)
{
  if (!d || !F_aos || !d->ibm.enabled) { set_error("lbm_ibm_get_force: no immersed boundary"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  // the field the last step read; the side stream may already be filling the other slot
  return ibm_download_force(d, F_aos, d->ibm.used_slot);
}

int lbm_ibm_force(lbm_domain* d, const double* u_aos, const double* rho_aos, double* F_aos)
{
  if (!d || !u_aos || !rho_aos || !F_aos || !d->ibm.enabled) { set_error("lbm_ibm_force: bad argument or no immersed boundary"); return LBM_ERR_INVALID; }
  if (d->cfg.x0 != 0 || d->cfg.x1 != d->cfg.X) { set_error("lbm_ibm_force: stand-alone call needs a single-slab domain"); return LBM_ERR_UNSUPPORTED; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  IbmState& ib = d->ibm;
  const long long N = (long long)d->cfg.X * d->cfg.Y;
  const int RR = (int)(ib.r1 - ib.r0), RC = (int)(ib.c1 - ib.c0), nn = RR * RC;
  double *du = nullptr, *dr = nullptr;
  LBM_CUDA(cudaMalloc(&du, sizeof(double) * 2 * N));
  LBM_CUDA(cudaMalloc(&dr, sizeof(double) * N));
  LBM_CUDA(cudaMemcpyAsync(du, u_aos, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, d->stream));
  LBM_CUDA(cudaMemcpyAsync(dr, rho_aos, sizeof(double) * N, cudaMemcpyHostToDevice, d->stream));
  k_ibm_load_roi<<<cdiv(nn, 128), 128, 0, d->stream>>>(du, dr, d->cfg.Y, (int)ib.r0, (int)ib.c0, RR, RC, ib.d_u, ib.d_rho);
  d->launches++;
  // scratch use of the slot no enqueued step reads; the side stream must be idle first
  LBM_CUDA(cudaStreamSynchronize(d->side));
  const int slot = d->ibm.next_slot ^ 1;
  LBM_TRY(ibm_iterate(d, slot, d->stream));
  int s = ibm_download_force(d, F_aos, slot);
  cudaFree(du);
  cudaFree(dr);
  return s;
}

}  // extern "C"
