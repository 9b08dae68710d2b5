// lbm_stats.cuh — time-averaged flow fields accumulated on the device: mean density, mean velocity and the velocity
// covariance <u'u'>, <v'v'>, <u'v'> of the moments each step's collision uses.
//
// Replaces the offline averaging of snapshots (the reference's drivers torch::save rho / u for post-processing): a copy of
// rho and u per step would move 24 B/node to the host, where the step itself moves 144 B/node on the device.  The moments
// are already in registers inside k_bgk_interior / k_bgk_boundary, so their STATS instantiations fold them into six
// Welford planes (lbm_bgk_kernels.cuh, StatsArgs) with no second pass over the populations.
//
//   k_stats_tick : one thread, main stream, after the step's side chain: advances the device-side clock (step count and
//                  1 / n of the next step's sample, 0 for no sample) that the three launches of a step (early and bulk
//                  rows on the main stream, listed nodes on the side stream) read, so that replayed CUDA graphs sample the
//                  right steps
//   k_stats_read : planes -> rho_mean {Xl,Y}, u_mean {Xl,Y,2}, u_cov {Xl,Y,3} = M / n in the host staging buffer
//
// Compiled as part of lbm_domain.cu's translation unit (included once, at its end), like lbm_body_force.cuh.
#pragma once
#include "lbm_internal.hpp"

namespace lbm
{

// the clock of the next step: step k is a sample when k % every == 0, sample n = k / every + 1
static __global__ void k_stats_tick(StatsClock* __restrict__ clock, int every)
{
  const long long k = clock->count + 1;
  clock->count = k;
  clock->inv_n = k % every == 0 ? 1.0 / (double)(k / every + 1) : 0.0;
}

static __global__ void k_stats_read(const double* __restrict__ acc, long long plane, const SlabGeom g, double n,
                                    double* __restrict__ rho, double* __restrict__ u, double* __restrict__ cov)
{
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= (long long)g.Xl * g.Y) return;
  const long long i = (k / g.Y) * g.pitch + k % g.Y;
  rho[k] = acc[i];
  u[2 * k] = acc[plane + i];
  u[2 * k + 1] = acc[2 * plane + i];
#pragma unroll
  for (int c = 0; c < 3; c++) cov[3 * k + c] = acc[(3 + c) * plane + i] / n;
}

void stats_release(lbm_domain* d)
{
  Stats& s = d->st;
  cudaFree(s.d_acc);
  cudaFree(s.d_clock);
  cudaFree(s.d_listed);
  s = Stats();
}

// The listed nodes in interior columns lie on early rows (step_rows), where the interior kernel computes a collision that
// k_bgk_boundary then overwrites; the early launch reads this mask to leave their accumulators to the listed kernel.
// Bulk rows hold no such node, so the bulk launch and the listed kernel — concurrent on two streams — update disjoint nodes.
int stats_listed_mask(lbm_domain* d)
{
  Stats& s = d->st;
  std::vector<unsigned> bits((size_t)d->g.Xl * s.words, 0u);
  for (int id : d->listed_ids)
  {
    const int x = id / d->g.Y, y = id % d->g.Y;
    if (y >= d->y_int_begin && y < d->y_int_end) bits[(size_t)x * s.words + (y >> 5)] |= 1u << (y & 31);
  }
  if (!s.d_listed) LBM_CUDA(cudaMalloc(&s.d_listed, sizeof(unsigned) * bits.size()));
  LBM_CUDA(cudaMemcpy(s.d_listed, bits.data(), sizeof(unsigned) * bits.size(), cudaMemcpyHostToDevice));
  return LBM_OK;
}

// After the bulk rows of a step: the early and bulk launches are on the main stream already, the listed nodes on the side
// stream end before ev_side.  The next step waits for ev_side before its early rows anyway, so this adds no serialisation.
int stats_tick(lbm_domain* d)
{
  if (!d->st.on) return LBM_OK;
  LBM_CUDA(cudaStreamWaitEvent(d->stream, d->ev_side, 0));
  k_stats_tick<<<1, 1, 0, d->stream>>>(d->st.d_clock, d->st.every);
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  return LBM_OK;
}

}  // namespace lbm

using namespace lbm;

extern "C"
{

int lbm_stats_start(lbm_domain* d, int every)
{
  if (!d) { set_error("lbm_stats_start: null domain"); return LBM_ERR_INVALID; }
  if (d->tp) { set_error("lbm_stats_start: the two-phase models have no statistics record (single-phase family only)"); return LBM_ERR_UNSUPPORTED; }
  if (every < 1) { set_error("lbm_stats_start: every = %d (need >= 1)", every); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->side));
  stats_release(d);
  drop_graphs(d);  // the captured step pairs launch the kernels without the record
  Stats& s = d->st;
  s.every = every;
  s.words = (d->g.Y + 31) / 32;
  auto alloc = [&]() -> int {
    const size_t acc = sizeof(double) * 6 * (size_t)d->g.Xl * d->g.pitch;
    LBM_CUDA(cudaMalloc(&s.d_acc, acc));
    LBM_CUDA(cudaMalloc(&s.d_clock, sizeof(StatsClock)));
    LBM_CUDA(cudaMemset(s.d_acc, 0, acc));
    const StatsClock first{0, 1.0};  // step 0 is sample n = 1
    LBM_CUDA(cudaMemcpy(s.d_clock, &first, sizeof(StatsClock), cudaMemcpyHostToDevice));
    return stats_listed_mask(d);
  };
  if (int r = alloc(); r != LBM_OK)
  {
    stats_release(d);
    return r;
  }
  s.on = true;
  return LBM_OK;
}

int lbm_stats_read(lbm_domain* d, double* rho_mean, double* u_mean, double* u_cov, long long* n_samples)
{
  if (!d || !n_samples) { set_error("lbm_stats_read: null argument"); return LBM_ERR_INVALID; }
  const Stats& s = d->st;
  if (!s.on) { set_error("lbm_stats_read: nothing is being accumulated (call lbm_stats_start first)"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaStreamSynchronize(d->side));  // listed nodes of the last step
  StatsClock clock{};
  LBM_CUDA(cudaMemcpyAsync(&clock, s.d_clock, sizeof(StatsClock), cudaMemcpyDeviceToHost, d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  const long long n = (clock.count + s.every - 1) / s.every;  // steps k < count with k % every == 0
  *n_samples = n;
  if (n == 0) return LBM_OK;
  const long long N = (long long)d->g.Xl * d->g.Y;
  if (!d->d_mom_out) LBM_CUDA(cudaMalloc(&d->d_mom_out, 6 * N * sizeof(double)));
  if (d->copy_pending) LBM_CUDA(cudaStreamWaitEvent(d->stream, d->ev_copied, 0));  // an lbm_snapshot_async still drains it
  double* out = d->d_mom_out;
  k_stats_read<<<(unsigned)((N + 255) / 256), 256, 0, d->stream>>>(s.d_acc, (long long)d->g.Xl * d->g.pitch, d->g, (double)n, out,
                                                                   out + N, out + 3 * N);
  d->launches++;
  LBM_CUDA(cudaGetLastError());
  if (rho_mean) LBM_CUDA(cudaMemcpyAsync(rho_mean, out, N * sizeof(double), cudaMemcpyDeviceToHost, d->stream));
  if (u_mean) LBM_CUDA(cudaMemcpyAsync(u_mean, out + N, 2 * N * sizeof(double), cudaMemcpyDeviceToHost, d->stream));
  if (u_cov) LBM_CUDA(cudaMemcpyAsync(u_cov, out + 3 * N, 3 * N * sizeof(double), cudaMemcpyDeviceToHost, d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  return LBM_OK;
}

int lbm_stats_stop(lbm_domain* d)
{
  if (!d) { set_error("lbm_stats_stop: null domain"); return LBM_ERR_INVALID; }
  if (!d->st.on) { set_error("lbm_stats_stop: nothing is being accumulated (call lbm_stats_start first)"); return LBM_ERR_INVALID; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaStreamSynchronize(d->stream));
  LBM_CUDA(cudaStreamSynchronize(d->side));
  stats_release(d);
  drop_graphs(d);
  return LBM_OK;
}

}  // extern "C"
