// lbm_body_force.cuh — the force the fluid on this slab's rows exerts on one body, recorded on the device once per step.
//
// Replaces the offline force sum of the reference's cylinder driver (test/cylinder_test.cpp:112 accumulates F_s, which the
// driver snapshots and a script sums): a per-step drag / lift series without a host round trip.
//   bounce-back body (lbm_bc_add_solid): momentum exchange over the links (n, q) with n fluid on this slab's rows and
//                     n - c_q solid,  F = sum 2 c_opp(q) f_coll(t)[n, opp(q)]
//   immersed body (lbm_ibm_set_markers): F = -sum F_euler over the active ROI nodes on this slab's rows
//
//   k_body_force_links / k_body_force_roi : one link / node per thread, a fixed-shape block reduction -> per-block partials
//   k_body_force_finish                   : one block sums the partials in a fixed order into ring[count % capacity] and
//                                           advances the device-side step counter
// No floating-point atomics: the record is bit-identical from run to run, with or without a CUDA graph.
//
// Compiled as part of lbm_domain.cu's translation unit (included once, at its end), so that every build of csrc/ — the
// library, `make NOFMA=1` and the emulated device of tests/cpu_emu — carries these kernels and entry points.
#pragma once
#include <algorithm>

#include "lbm_internal.hpp"

namespace lbm
{

constexpr int BF_NT = 256;  // threads per block of the three kernels

static inline int bf_blocks(int n) { return (n + BF_NT - 1) / BF_NT; }

// sum of (x, y) over the block, tree-shaped: the same additions in the same order on every launch
template <int NT>
__device__ __forceinline__ void block_sum2(double& x, double& y)
{
  __shared__ double sx[NT], sy[NT];
  const int t = threadIdx.x;
  sx[t] = x;
  sy[t] = y;
  __syncthreads();
#pragma unroll
  for (int s = NT / 2; s > 0; s >>= 1)
  {
    if (t < s)
    {
      sx[t] += sx[t + s];
      sy[t] += sy[t + s];
    }
    __syncthreads();
  }
  x = sx[0];
  y = sy[0];
}

// link = (offset of f[opp(q)] at the fluid node in a lattice buffer) << 4 | q
template <int NT>
__global__ void __launch_bounds__(NT) k_body_force_links(const double* __restrict__ f, const long long* __restrict__ link, int n,
                                                         double* __restrict__ part)
{
  const int i = blockIdx.x * NT + threadIdx.x;
  double x = 0.0, y = 0.0;
  if (i < n)
  {
    const long long e = link[i];
    const int q = (int)(e & 15);
    const double v = 2.0 * f[e >> 4];
    x = (double)CX(OPP(q)) * v;
    y = (double)CY(OPP(q)) * v;
  }
  block_sum2<NT>(x, y);
  if (threadIdx.x == 0)
  {
    part[2 * blockIdx.x] = x;
    part[2 * blockIdx.x + 1] = y;
  }
}

template <int NT>
__global__ void __launch_bounds__(NT) k_body_force_roi(const double* __restrict__ Fx, const double* __restrict__ Fy,
                                                       const int* __restrict__ active, int n, double* __restrict__ part)
{
  const int i = blockIdx.x * NT + threadIdx.x;
  double x = 0.0, y = 0.0;
  if (i < n)
  {
    const int a = active[i];
    x = -Fx[a];
    y = -Fy[a];
  }
  block_sum2<NT>(x, y);
  if (threadIdx.x == 0)
  {
    part[2 * blockIdx.x] = x;
    part[2 * blockIdx.x + 1] = y;
  }
}

template <int NT>
__global__ void __launch_bounds__(NT) k_body_force_finish(const double* __restrict__ part, int nblk, double* __restrict__ ring,
                                                          long long* __restrict__ count, int capacity)
{
  double x = 0.0, y = 0.0;
  for (int b = threadIdx.x; b < nblk; b += NT)
  {
    x += part[2 * b];
    y += part[2 * b + 1];
  }
  block_sum2<NT>(x, y);
  if (threadIdx.x == 0)
  {
    const long long c = *count;
    ring[2 * (c % capacity)] = x;
    ring[2 * (c % capacity) + 1] = y;
    *count = c + 1;
  }
}

void body_force_release(lbm_domain* d)
{
  BodyForce& bf = d->bf;
  cudaFree(bf.d_link);
  cudaFree(bf.d_part);
  cudaFree(bf.d_ring);
  cudaFree(bf.d_count);
  bf = BodyForce();
}

// Side stream, after the listed-node kernel and the pre-stream stages of the step: buf[cur ^ 1] then holds f_coll(t) at every
// link's fluid node (a listed node: the bulk launch running beside the side chain does not write it), and ibm.next_slot is
// the force field this step's collision adds.  The next step joins the side chain before it writes either.
int body_force_step(lbm_domain* d)
{
  BodyForce& bf = d->bf;
  if (!bf.on) return LBM_OK;
  const int nblk = bf_blocks(bf.n);
  if (nblk > 0)
  {
    if (bf.immersed)
    {
      const IbmState& ib = d->ibm;
      k_body_force_roi<BF_NT><<<nblk, BF_NT, 0, d->side>>>(ib.d_Fx[ib.next_slot], ib.d_Fy[ib.next_slot], ib.d_active + ib.a_lo, bf.n,
                                                           bf.d_part);
    }
    else
      k_body_force_links<BF_NT><<<nblk, BF_NT, 0, d->side>>>(d->buf[0][d->cur ^ 1], bf.d_link, bf.n, bf.d_part);
    d->launches++;
  }
  k_body_force_finish<BF_NT><<<1, BF_NT, 0, d->side>>>(bf.d_part, nblk, bf.d_ring, bf.d_count, bf.capacity);
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

// the momentum-exchange links of this slab's rows, sorted by (node, q); each must be a plain bounce-back rule of lattice 0
static int bounce_back_links(lbm_domain* d, const unsigned char* solid, std::vector<long long>& links)
{
  const int X = d->cfg.X, Y = d->cfg.Y, x0 = d->cfg.x0;
  const std::vector<int32_t>& mask = d->mask[0];
  for (int lx = 0; lx < d->g.Xl; lx++)
  {
    const int gx = x0 + lx;
    for (int y = 0; y < Y; y++)
    {
      if (solid[(size_t)gx * Y + y]) continue;
      for (int q = 1; q < 9; q++)
      {
        const int sx = (gx - CX(q) + X) % X, sy = (y - CY(q) + Y) % Y;  // periodic, like lbm_bc_add_solid
        if (!solid[(size_t)sx * Y + sy]) continue;
        const int k = mask[((size_t)lx * Y + y) * 9 + q] - 1;
        bool ok = k >= 0 && k < (int)d->ops.size();
        if (ok)
        {
          const lbm_bc_op& op = d->ops[k].op;
          ok = op.kind == LBM_BC_LINEAR && op.src_mode == LBM_SRC_SAME_NODE && op.dst_q == q && op.src_q == OPP(q) && op.coef == 1.0 &&
               op.cst == 0.0;
        }
        if (!ok)
        {
          set_error("lbm_body_force_record: link (%d, %d, q = %d) into the body is not owned by a bounce-back rule f_adve[n, q] = "
                    "f_coll[n, opp(q)] (owner: %s %d); add the body with lbm_bc_add_solid after the other rules",
                    gx, y, q, k < 0 ? "no rule" : (k < (int)d->ops.size() ? "rule" : "column-face binding"), k);
          return LBM_ERR_INVALID;
        }
        const long long off = (long long)OPP(q) * d->g.plane + (long long)(lx + 1) * d->g.pitch + y;
        links.push_back(off << 4 | q);
      }
    }
  }
  return LBM_OK;
}

}  // namespace lbm

using namespace lbm;

extern "C"
{

int lbm_body_force_record(lbm_domain* d, const unsigned char* solid, int X, int Y, int capacity)
{
  if (!d) { set_error("lbm_body_force_record: null domain"); return LBM_ERR_INVALID; }
  if (d->tp) { set_error("lbm_body_force_record: the two-phase models have no body force record (single-phase family only)"); return LBM_ERR_UNSUPPORTED; }
  if (capacity < 1) { set_error("lbm_body_force_record: capacity %d (need >= 1)", capacity); return LBM_ERR_INVALID; }
  if (!d->committed) { set_error("lbm_body_force_record: call lbm_bc_commit first"); return LBM_ERR_INVALID; }
  if (solid && (X != d->cfg.X || Y != d->cfg.Y))
  {
    set_error("lbm_body_force_record: mask %dx%d is not the domain's global grid %dx%d", X, Y, d->cfg.X, d->cfg.Y);
    return LBM_ERR_INVALID;
  }
  if (!solid && (d->cfg.force != LBM_FORCE_IBM || d->ibm_given.n == 0 || d->ibm.fixed))
  {
    set_error("lbm_body_force_record: no solid mask and no immersed body (lbm_ibm_set_markers on a domain with force = LBM_FORCE_IBM)");
    return LBM_ERR_INVALID;
  }
  std::vector<long long> links;
  if (solid) LBM_TRY(bounce_back_links(d, solid, links));
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->side));
  body_force_release(d);
  drop_graphs(d);
  BodyForce& bf = d->bf;
  bf.immersed = !solid;
  bf.capacity = capacity;
  // a slab that owns none of the immersed body's ROI rows records zeros
  bf.n = solid ? (int)links.size() : (d->ibm.enabled ? d->ibm.a_hi - d->ibm.a_lo : 0);
  const int nblk = std::max(bf_blocks(bf.n), 1);
  auto alloc = [&]() -> int {
    if (solid && bf.n > 0)
    {
      LBM_CUDA(cudaMalloc(&bf.d_link, sizeof(long long) * bf.n));
      LBM_CUDA(cudaMemcpy(bf.d_link, links.data(), sizeof(long long) * bf.n, cudaMemcpyHostToDevice));
    }
    LBM_CUDA(cudaMalloc(&bf.d_part, sizeof(double) * 2 * nblk));
    LBM_CUDA(cudaMalloc(&bf.d_ring, sizeof(double) * 2 * capacity));
    LBM_CUDA(cudaMalloc(&bf.d_count, sizeof(long long)));
    LBM_CUDA(cudaMemset(bf.d_ring, 0, sizeof(double) * 2 * capacity));
    LBM_CUDA(cudaMemset(bf.d_count, 0, sizeof(long long)));
    return LBM_OK;
  };
  if (int s = alloc(); s != LBM_OK)
  {
    body_force_release(d);
    return s;
  }
  bf.on = true;
  return LBM_OK;
}

int lbm_body_force_read(lbm_domain* d, double* F, int max_steps, int* n_steps, long long* first_step)
{
  if (!d || !n_steps || !first_step || max_steps < 0 || (!F && max_steps > 0)) { set_error("lbm_body_force_read: bad argument"); return LBM_ERR_INVALID; }
  const BodyForce& bf = d->bf;
  if (!bf.on) { set_error("lbm_body_force_read: nothing is being recorded (call lbm_body_force_record first)"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaStreamSynchronize(d->side));
  long long count = 0;
  std::vector<double> ring(2 * (size_t)bf.capacity);
  LBM_CUDA(cudaMemcpyAsync(&count, bf.d_count, sizeof(long long), cudaMemcpyDeviceToHost, d->stream));
  LBM_CUDA(cudaMemcpyAsync(ring.data(), bf.d_ring, sizeof(double) * ring.size(), cudaMemcpyDeviceToHost, d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  const long long n = std::min<long long>(std::min<long long>(count, bf.capacity), max_steps);
  const long long first = count - n;
  for (long long k = 0; k < n; k++)
  {
    const size_t slot = (size_t)((first + k) % bf.capacity);
    F[2 * k] = ring[2 * slot];
    F[2 * k + 1] = ring[2 * slot + 1];
  }
  *n_steps = (int)n;
  *first_step = first;
  return LBM_OK;
}

int lbm_body_force_stop(lbm_domain* d)
{
  if (!d) { set_error("lbm_body_force_stop: null domain"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->side));
  body_force_release(d);
  drop_graphs(d);
  return LBM_OK;
}

}  // extern "C"
