// lbm_comm.cu — slabs along axis 0 on several GPUs (SURVEY §8e; test/decompose_domain.cpp:181-187).
//
// What crosses a cut, per lattice and per step: the three populations of the boundary row that head
// for the neighbour — c_x = +1 {1,5,8} upwards, c_x = -1 {3,6,7} downwards — copied into the
// neighbour's ghost row, where the pull then finds them with the +-1 column shift of the diagonal
// directions exactly as the reference's "bind" block writes them.  The slabs form a ring, which is
// the periodic wrap of solver::advect.  Two-phase models also exchange two rows of the five moment
// planes for the 5x5 differences (no wrap: the global edge replicates).  Pressure-periodic rows whose
// source row lives on another slab travel as a 12 x Y packet (lbm_bgk_kernels.cuh).
//
// Two transports:
//   NCCL   one process per GPU (torchrun): ncclSend/ncclRecv grouped per step on the slab's side
//          stream, overlapping the interior rows.  libnccl is dlopen'ed so that single-GPU use has
//          no NCCL dependency.
//   link   several slabs inside one process (same or different devices): cudaMemcpyPeerAsync between
//          the slabs' streams, driven by lbm_step_group.  This is also how the decomposition is
//          tested on a single GPU.
#include <dlfcn.h>

#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>

#include "lbm_internal.hpp"

namespace lbm
{

// ---- the few NCCL declarations used (ABI-stable since NCCL 2.7)
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { ncclFloat64 = 8 };

struct NcclApi
{
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

static NcclApi g_nccl;

static int load_nccl()
{
  static std::mutex mu;  // several host threads (one per GPU) may create their communicators at once
  std::lock_guard<std::mutex> lock(mu);
  if (g_nccl.handle) return LBM_OK;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  // LBM_NCCL_LIB: path of the NCCL build to bind instead (a site's own libnccl; tests/cpu_emu points it at its stand-in)
  if (const char* path = std::getenv("LBM_NCCL_LIB"))
  {
    h = dlopen(path, RTLD_NOW | RTLD_LOCAL);
    if (!h)
    {
      set_error("cannot load LBM_NCCL_LIB=%s: %s", path, dlerror());
      return LBM_ERR_COMM;
    }
  }
  for (const char* n : names)
  {
    if (h) break;
    h = dlopen(n, RTLD_NOW | RTLD_NOLOAD);  // the copy the host process (e.g. torch) already loaded
  }
  for (const char* n : names)
  {
    if (h) break;
    h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
  }
  if (!h)
  {
    set_error("cannot load libnccl.so.2: %s", dlerror());
    return LBM_ERR_COMM;
  }
  NcclApi a;
  a.handle = h;
#define LBM_SYM(field, name)                                                  \
  a.field = reinterpret_cast<decltype(a.field)>(dlsym(h, name));              \
  if (!a.field) { set_error("libnccl lacks %s", name); return LBM_ERR_COMM; }
  LBM_SYM(GetUniqueId, "ncclGetUniqueId")
  LBM_SYM(CommInitRank, "ncclCommInitRank")
  LBM_SYM(CommDestroy, "ncclCommDestroy")
  LBM_SYM(Send, "ncclSend")
  LBM_SYM(Recv, "ncclRecv")
  LBM_SYM(GroupStart, "ncclGroupStart")
  LBM_SYM(GroupEnd, "ncclGroupEnd")
  LBM_SYM(GetErrorString, "ncclGetErrorString")
#undef LBM_SYM
  g_nccl = a;
  return LBM_OK;
}

// A failed Send / Recv inside a ncclGroupStart / ncclGroupEnd bracket must not leave this thread's group open (every
// later NCCL call would nest into it and never launch: a hang instead of LBM_ERR_COMM), so the bracket depth is
// tracked and closed on the error path.
static thread_local int t_group_depth = 0;

#define LBM_NCCL(call)                                                                         \
  do                                                                                           \
  {                                                                                            \
    ncclResult_t r__ = (call);                                                                 \
    if (r__ != 0)                                                                              \
    {                                                                                          \
      set_error("%s failed: %s", #call, g_nccl.GetErrorString ? g_nccl.GetErrorString(r__) : "?"); \
      for (; t_group_depth > 0; t_group_depth--) g_nccl.GroupEnd();                            \
      return LBM_ERR_COMM;                                                                     \
    }                                                                                          \
  } while (0)
#define LBM_NCCL_GROUP_BEGIN()        \
  do                                  \
  {                                   \
    LBM_NCCL(g_nccl.GroupStart());    \
    t_group_depth++;                  \
  } while (0)
#define LBM_NCCL_GROUP_END()          \
  do                                  \
  {                                   \
    t_group_depth--;                  \
    LBM_NCCL(g_nccl.GroupEnd());      \
  } while (0)

// the NCCL communicator of a ring, shared by every domain of this process that joined it (lbm_comm_init creates it,
// lbm_comm_share hands it on: a driver that advances several fields on the same slabs, or a bench that runs one workload
// after the other, pays ncclCommInitRank — seconds on eight ranks — once)
struct CommHandle
{
  ncclComm_t comm = nullptr;
  ~CommHandle()
  {
    if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(comm);
  }
};

struct CommState
{
  std::shared_ptr<CommHandle> handle;
  ncclComm_t comm = nullptr;  // = handle->comm
  int n_ranks = 1, rank = 0;
  bool blocks = false;        // lbm_comm_init_blocks: independent blocks bound across column faces, not the slabs of one grid
};

bool comm_active(const lbm_domain* d) { return d->comm != nullptr && d->comm->n_ranks > 1 && !d->comm->blocks; }
bool comm_blocks(const lbm_domain* d) { return d->comm != nullptr && d->comm->blocks; }

int comm_release(lbm_domain* d)
{
  if (!d->comm) return LBM_OK;
  delete d->comm;  // the communicator goes with its last holder
  d->comm = nullptr;
  return LBM_OK;
}

// rank that owns global row gx under lbm_decompose_rows
static int owner_of(int X, int n_ranks, int gx)
{
  const int base = X / n_ranks, rem = X % n_ranks;
  const int split = rem * (base + 1);
  if (gx < split) return gx / (base + 1);
  return rem + (gx - split) / base;
}

// population ghost rows of buffer `which` of every lattice, on stream st
int comm_exchange(lbm_domain* d, int which, cudaStream_t st)
{
  CommState* c = d->comm;
  const int up = (c->rank + 1) % c->n_ranks, dn = (c->rank + c->n_ranks - 1) % c->n_ranks;
  const SlabGeom& g = d->g;
  const size_t n = (size_t)g.pitch;
  LBM_NCCL_GROUP_BEGIN();
  for (int l = 0; l < d->nlat; l++)
  {
    double* f = d->buf[l][which];
    for (int q = 0; q < 9; q++)
    {
      double* plane = f + (long long)q * g.plane;
      double* ghost_lo = plane;                                   // storage row 0      = row -1
      double* first = plane + (long long)g.pitch;                 // storage row 1      = row 0
      double* last = plane + (long long)g.Xl * g.pitch;           // storage row Xl     = row Xl-1
      double* ghost_hi = plane + (long long)(g.Xl + 1) * g.pitch; // storage row Xl + 1 = row Xl
      if (d->wrap_all_q || CX(q) == 1)
      {
        LBM_NCCL(g_nccl.Send(last, n, ncclFloat64, up, c->comm, st));
        LBM_NCCL(g_nccl.Recv(ghost_lo, n, ncclFloat64, dn, c->comm, st));
      }
      if (d->wrap_all_q || CX(q) == -1)
      {
        LBM_NCCL(g_nccl.Send(first, n, ncclFloat64, dn, c->comm, st));
        LBM_NCCL(g_nccl.Recv(ghost_hi, n, ncclFloat64, up, c->comm, st));
      }
    }
  }
  LBM_NCCL_GROUP_END();
  d->launches++;
  return LBM_OK;
}

// two ghost rows of `nplanes` planes in the moment-plane geometry across every INTERNAL cut (the global edge replicates)
int comm_exchange_planes(lbm_domain* d, double* base, int nplanes, cudaStream_t st)
{
  if (!d->tp || !comm_active(d)) return LBM_OK;
  if (!st) st = d->stream;
  CommState* c = d->comm;
  int pm = 0;
  long long mplane = 0;
  tp_moment_planes(d, &pm, &mplane);
  const int Xl = d->g.Xl;
  const size_t n = (size_t)2 * pm;
  const bool has_dn = d->cfg.x0 > 0, has_up = d->cfg.x1 < d->cfg.X;
  LBM_NCCL_GROUP_BEGIN();
  for (int f = 0; f < nplanes; f++)
  {
    double* pl = base + (long long)f * mplane;
    // storage row r holds slab row r - 2
    if (has_up)
    {
      LBM_NCCL(g_nccl.Send(pl + (long long)Xl * pm, n, ncclFloat64, c->rank + 1, c->comm, st));        // rows Xl-2, Xl-1
      LBM_NCCL(g_nccl.Recv(pl + (long long)(Xl + 2) * pm, n, ncclFloat64, c->rank + 1, c->comm, st));  // rows Xl, Xl+1
    }
    if (has_dn)
    {
      LBM_NCCL(g_nccl.Send(pl + (long long)2 * pm, n, ncclFloat64, c->rank - 1, c->comm, st));  // rows 0, 1
      LBM_NCCL(g_nccl.Recv(pl, n, ncclFloat64, c->rank - 1, c->comm, st));                      // rows -2, -1
    }
  }
  LBM_NCCL_GROUP_END();
  d->launches++;
  return LBM_OK;
}

// max over the ring of one non-negative double held on the device: every rank hands its value to every other, the
// reduction runs on the host.  Diagnostic paths only (lbm_rk_diagnostics: the normal's cut at 0.1 max|grad|).
int comm_allreduce_max(lbm_domain* d, double* dev_value)
{
  if (!comm_active(d)) return LBM_OK;
  CommState* c = d->comm;
  const int P = c->n_ranks;
  double* all = nullptr;
  LBM_CUDA(cudaMalloc(&all, sizeof(double) * P));
  auto run = [&]() -> int {
    LBM_CUDA(cudaMemcpyAsync(all + c->rank, dev_value, sizeof(double), cudaMemcpyDeviceToDevice, d->stream));
    LBM_NCCL_GROUP_BEGIN();
    for (int k = 0; k < P; k++)
    {
      if (k == c->rank) continue;
      LBM_NCCL(g_nccl.Send(dev_value, 1, ncclFloat64, k, c->comm, d->stream));
      LBM_NCCL(g_nccl.Recv(all + k, 1, ncclFloat64, k, c->comm, d->stream));
    }
    LBM_NCCL_GROUP_END();
    std::vector<double> host(P);
    LBM_CUDA(cudaMemcpyAsync(host.data(), all, sizeof(double) * P, cudaMemcpyDeviceToHost, d->stream));
    LBM_CUDA(cudaStreamSynchronize(d->stream));
    double m = 0.0;
    for (double v : host) m = v > m ? v : m;
    LBM_CUDA(cudaMemcpyAsync(dev_value, &m, sizeof(double), cudaMemcpyHostToDevice, d->stream));
    LBM_CUDA(cudaStreamSynchronize(d->stream));
    return LBM_OK;
  };
  const int rc = run();
  cudaFree(all);
  return rc;
}

int comm_exchange_moments(lbm_domain* d)
{
  if (!d->tp) return LBM_OK;
  int pm = 0;
  long long mplane = 0;
  return comm_exchange_planes(d, tp_moment_planes(d, &pm, &mplane), 5);
}

// Immersed boundary across slab cuts: the moments of the active ROI nodes, one contiguous row segment per slab that owns
// ROI rows, swapped between all of those slabs (usually two).  Every rank derives the same list from lbm_decompose_rows.
int comm_ibm_share(lbm_domain* d, cudaStream_t st)
{
  CommState* c = d->comm;
  IbmState& ib = d->ibm;
  const int RC = (int)(ib.c1 - ib.c0);
  LBM_NCCL_GROUP_BEGIN();
  for (int k = 0; k < c->n_ranks; k++)
  {
    if (k == c->rank) continue;
    int kx0 = 0, kx1 = 0;
    lbm_decompose_rows(d->cfg.X, c->n_ranks, k, &kx0, &kx1);
    const long lo = std::max<long>(ib.r0, kx0) - ib.r0, hi = std::min<long>(ib.r1, kx1) - ib.r0;
    if (hi <= lo) continue;  // rank k owns no ROI row
    const size_t mine = (size_t)(ib.row_hi - ib.row_lo) * RC, theirs = (size_t)(hi - lo) * RC;
    LBM_NCCL(g_nccl.Send(ib.d_rho + (size_t)ib.row_lo * RC, mine, ncclFloat64, k, c->comm, st));
    LBM_NCCL(g_nccl.Send(ib.d_u + 2 * (size_t)ib.row_lo * RC, 2 * mine, ncclFloat64, k, c->comm, st));
    LBM_NCCL(g_nccl.Recv(ib.d_rho + (size_t)lo * RC, theirs, ncclFloat64, k, c->comm, st));
    LBM_NCCL(g_nccl.Recv(ib.d_u + 2 * (size_t)lo * RC, 2 * theirs, ncclFloat64, k, c->comm, st));
  }
  LBM_NCCL_GROUP_END();
  d->launches++;
  return LBM_OK;
}

// pressure packet of stage k: from the rank that owns the source row to the rank that owns the written row
int comm_stage_transfer(lbm_domain* d, size_t k, cudaStream_t st)
{
  Stage& sg = d->stages[k];
  if (sg.kind != 1) return LBM_OK;
  CommState* c = d->comm;
  const int src_rank = owner_of(d->cfg.X, c->n_ranks, sg.src_gx), dst_rank = owner_of(d->cfg.X, c->n_ranks, sg.dst_gx);
  if (src_rank == dst_rank) return LBM_OK;
  const size_t n = (size_t)12 * d->g.Y;
  if (c->rank == src_rank) LBM_NCCL(g_nccl.Send(sg.d_packet, n, ncclFloat64, dst_rank, c->comm, st));
  if (c->rank == dst_rank) LBM_NCCL(g_nccl.Recv(sg.d_packet, n, ncclFloat64, src_rank, c->comm, st));
  if (c->rank == src_rank || c->rank == dst_rank) d->launches++;
  return LBM_OK;
}

// ------------------------------------------------------------------------------------------------
// link transport: slabs of one process
// ------------------------------------------------------------------------------------------------
static int copy_rows(lbm_domain* dst, double* dptr, lbm_domain* src, const double* sptr, size_t count, cudaStream_t st)
{
  if (dst->cfg.device == src->cfg.device)
    LBM_CUDA(cudaMemcpyAsync(dptr, sptr, count * sizeof(double), cudaMemcpyDeviceToDevice, st));
  else
    LBM_CUDA(cudaMemcpyPeerAsync(dptr, dst->cfg.device, sptr, src->cfg.device, count * sizeof(double), st));
  dst->launches++;
  return LBM_OK;
}

// Ghost rows of buffer `which` of slab d from the same buffer index of its linked neighbours, on
// stream st.  The caller has made st wait for the neighbours' rows to be final.
int link_exchange(lbm_domain* d, int which, cudaStream_t st)
{
  const SlabGeom& g = d->g;
  for (int l = 0; l < d->nlat; l++)
    for (int q = 0; q < 9; q++)
    {
      double* plane = d->buf[l][which] + (long long)q * g.plane;
      if (d->link_lo && (d->wrap_all_q || CX(q) == 1))
      {
        lbm_domain* s = d->link_lo;
        const double* last = s->buf[l][which] + (long long)q * s->g.plane + (long long)s->g.Xl * s->g.pitch;
        LBM_TRY(copy_rows(d, plane, s, last, g.pitch, st));
      }
      if (d->link_hi && (d->wrap_all_q || CX(q) == -1))
      {
        lbm_domain* s = d->link_hi;
        const double* first = s->buf[l][which] + (long long)q * s->g.plane + (long long)s->g.pitch;
        LBM_TRY(copy_rows(d, plane + (long long)(g.Xl + 1) * g.pitch, s, first, g.pitch, st));
      }
    }
  return LBM_OK;
}

// Linked slab outside lbm_step_group (export right after an import): bring the ghost rows of
// buf[cur] in from the neighbours' current buffers and signal ev_side.
int comm_link_refresh(lbm_domain* d)
{
  if (d->side_ready) return LBM_OK;
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  LBM_CUDA(cudaEventRecord(d->ev_ready, d->stream));
  LBM_CUDA(cudaStreamWaitEvent(d->side, d->ev_ready, 0));
  if (!d->post_stream)
  {
    for (lbm_domain* o : {d->link_lo, d->link_hi})
    {
      if (!o || o == d) continue;
      if (o->cur != d->cur || o->post_stream)
      {
        set_error("linked slabs are out of step (advance them together with lbm_step_group)");
        return LBM_ERR_INVALID;
      }
      LBM_CUDA(cudaSetDevice(o->cfg.device));
      LBM_CUDA(cudaEventRecord(o->ev_ready, o->stream));
      LBM_CUDA(cudaSetDevice(d->cfg.device));
      LBM_CUDA(cudaStreamWaitEvent(d->side, o->ev_ready, 0));
      LBM_CUDA(cudaStreamWaitEvent(d->side, o->ev_side, 0));
    }
    LBM_TRY(link_exchange(d, d->cur, d->side));
  }
  LBM_TRY(step_prologue(d, false, !d->ibm.split));  // IBM field if any, then ev_side (on the same side stream)
  return LBM_OK;
}

// packet[lattice][qi][k] = f_coll(lattice)[row0 + k, col, face_q(side, qi)]
__global__ void k_face_pack(const double* __restrict__ f0, const double* __restrict__ f1, const SlabGeom g, int col, int row0,
                            int n, int side, int nlat, double* __restrict__ packet)
{
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= nlat * 3 * n) return;
  const int k = idx % n, qi = (idx / n) % 3, l = idx / (3 * n);
  const double* f = l == 0 ? f0 : f1;
  packet[idx] = f[(long long)face_q(side, qi) * g.plane + node_off(g, row0 + k, col)];
}

int faces_release(lbm_domain* d)
{
  for (auto& fl : d->faces)
  {
    cudaSetDevice(fl.other_device);
    cudaFree(fl.d_packet);
    if (fl.ev) cudaEventDestroy(fl.ev);
  }
  d->faces.clear();
  cudaSetDevice(d->cfg.device);
  for (auto& sv : d->serves) cudaFree(sv.d_packet);
  d->serves.clear();
  d->faces_remote_ready = false;
  return LBM_OK;
}

// Bound column faces between blocks on DIFFERENT ranks (lbm_link_face_rank): on the side stream, behind the listed-node
// kernel that wrote the edge columns of buffer `w` — pack the rows remote readers asked for, then one NCCL group: send the
// packets, receive this block's face tails straight into place (3 x nlat contiguous pieces per link).  Between two ranks
// sends and receives match in order: the reader enumerates its links to that peer by index, the server the same links out
// of the reader's descriptors (lbm_comm_faces_commit), each link as [lattice][qi].
int faces_exchange_remote(lbm_domain* d, bool new_buffer)
{
  if (!comm_blocks(d)) return LBM_OK;
  CommState* c = d->comm;
  const int w = new_buffer ? d->cur ^ 1 : d->cur;
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  for (auto& sv : d->serves)
  {
    const int total = d->nlat * 3 * sv.n;
    k_face_pack<<<(total + 127) / 128, 128, 0, d->side>>>(d->buf[0][w], d->buf[1][w], d->g, sv.reader_side == 0 ? d->g.Y - 1 : 0, sv.rb, sv.n,
                                                         sv.reader_side, d->nlat, sv.d_packet);
    d->launches++;
  }
  LBM_CUDA(cudaGetLastError());
  ProfScope ps(d, LBM_PROF_GHOST, d->side);
  LBM_NCCL_GROUP_BEGIN();
  for (auto& sv : d->serves)
    for (int l = 0; l < d->nlat; l++)
      for (int qi = 0; qi < 3; qi++)
        LBM_NCCL(g_nccl.Send(sv.d_packet + (size_t)(l * 3 + qi) * sv.n, (size_t)sv.n, ncclFloat64, sv.peer_rank, c->comm, d->side));
  for (auto& fl : d->faces)
  {
    if (fl.peer_rank < 0) continue;
    for (int l = 0; l < d->nlat; l++)
      for (int qi = 0; qi < 3; qi++)
        LBM_NCCL(g_nccl.Recv(d->buf[l][w] + face_tail_off(d->g, fl.side, qi, fl.rb), (size_t)fl.n, ncclFloat64, fl.peer_rank, c->comm, d->side));
  }
  LBM_NCCL_GROUP_END();
  d->launches++;
  return LBM_OK;
}

}  // namespace lbm

using namespace lbm;

extern "C"
{

int lbm_comm_unique_id(char id[LBM_UNIQUE_ID_BYTES])
{
  if (!id) { set_error("lbm_comm_unique_id: null argument"); return LBM_ERR_INVALID; }
  LBM_TRY(load_nccl());
  ncclUniqueId u;
  LBM_NCCL(g_nccl.GetUniqueId(&u));
  static_assert(sizeof(u) == LBM_UNIQUE_ID_BYTES, "ncclUniqueId is 128 bytes");
  std::memcpy(id, &u, sizeof(u));
  return LBM_OK;
}

int lbm_comm_init(lbm_domain* d, const char id[LBM_UNIQUE_ID_BYTES], int n_ranks, int rank)
{
  if (!d || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) { set_error("lbm_comm_init: bad argument"); return LBM_ERR_INVALID; }
  int x0 = 0, x1 = 0;
  LBM_TRY(lbm_decompose_rows(d->cfg.X, n_ranks, rank, &x0, &x1));
  if (x0 != d->cfg.x0 || x1 != d->cfg.x1)
  {
    set_error("lbm_comm_init: rank %d of %d must own rows [%d,%d) (lbm_decompose_rows), the domain has [%d,%d)", rank, n_ranks,
              x0, x1, d->cfg.x0, d->cfg.x1);
    return LBM_ERR_INVALID;
  }
  if (d->tp && d->have_state)
  {
    // the two-phase imports (lbm_init_two_phase, lbm_set_f, lbm_set_u) swap the moment-plane halos of the cuts when they
    // run; a ring joined afterwards would take its first step with replicate-padded halos at every cut
    set_error("lbm_comm_init: a two-phase domain joins the ring BEFORE its state is imported (lbm_init_two_phase / lbm_set_f / lbm_set_u)");
    return LBM_ERR_INVALID;
  }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  comm_release(d);
  LBM_TRY(load_nccl());
  CommState* c = new CommState();
  c->n_ranks = n_ranks;
  c->rank = rank;
  c->handle = std::make_shared<CommHandle>();
  ncclUniqueId u;
  std::memcpy(&u, id, sizeof(u));
  ncclResult_t r = g_nccl.CommInitRank(&c->handle->comm, n_ranks, u, rank);
  if (r != 0)
  {
    set_error("ncclCommInitRank failed: %s", g_nccl.GetErrorString(r));
    c->handle->comm = nullptr;
    delete c;
    return LBM_ERR_COMM;
  }
  c->comm = c->handle->comm;
  d->comm = c;
  d->side_ready = false;
  return LBM_OK;
}

// d joins the ring `member` already belongs to, on the same communicator.  Same conditions as lbm_comm_init: d owns the
// rows lbm_decompose_rows gives this rank, and a two-phase domain joins before its state is imported.  Both domains live
// on the same device; they may be stepped one after the other, not concurrently from several host threads.
int lbm_comm_share(lbm_domain* d, lbm_domain* member)
{
  if (!d || !member || !member->comm || !member->comm->handle) { set_error("lbm_comm_share: the second domain has not joined a ring"); return LBM_ERR_INVALID; }
  if (d->cfg.device != member->cfg.device) { set_error("lbm_comm_share: the two domains live on different devices"); return LBM_ERR_INVALID; }
  const int n_ranks = member->comm->n_ranks, rank = member->comm->rank;
  int x0 = 0, x1 = 0;
  LBM_TRY(lbm_decompose_rows(d->cfg.X, n_ranks, rank, &x0, &x1));
  if (x0 != d->cfg.x0 || x1 != d->cfg.x1)
  {
    set_error("lbm_comm_share: rank %d of %d must own rows [%d,%d) (lbm_decompose_rows), the domain has [%d,%d)", rank, n_ranks, x0, x1,
              d->cfg.x0, d->cfg.x1);
    return LBM_ERR_INVALID;
  }
  if (d->tp && d->have_state)
  {
    set_error("lbm_comm_share: a two-phase domain joins the ring BEFORE its state is imported (lbm_init_two_phase / lbm_set_f / lbm_set_u)");
    return LBM_ERR_INVALID;
  }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  comm_release(d);
  CommState* c = new CommState();
  c->n_ranks = n_ranks;
  c->rank = rank;
  c->handle = member->comm->handle;
  c->comm = c->handle->comm;
  d->comm = c;
  d->side_ready = false;
  return LBM_OK;
}

// Collective over the ring: every rank calls it once its setup is complete (rules committed, markers set), before the
// first lbm_step.  Each rank hands every other rank a ten-number record of what it was set up with; a difference that
// would make the ring wait for a message nobody sends (an immersed body whose ROI rows a slab owns but whose marker list
// that slab was never given; different grids, models or force modes) comes back as LBM_ERR_COMM on every rank instead.
int lbm_comm_check(lbm_domain* d)
{
  if (!d) { set_error("lbm_comm_check: null domain"); return LBM_ERR_INVALID; }
  if (!comm_active(d)) return LBM_OK;
  CommState* c = d->comm;
  constexpr int NREC = 10;
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  const int P = c->n_ranks;
  std::vector<double> rec((size_t)P * NREC, 0.0);
  double* mine = rec.data() + (size_t)c->rank * NREC;
  mine[0] = d->cfg.X; mine[1] = d->cfg.Y; mine[2] = d->cfg.model; mine[3] = d->cfg.force; mine[4] = d->cfg.equilibrium;
  mine[5] = d->ibm_given.n; mine[6] = (double)d->ibm_given.r0; mine[7] = (double)d->ibm_given.r1;
  mine[8] = (double)(d->ibm_given.hash >> 32); mine[9] = (double)(d->ibm_given.hash & 0xffffffffull);  // exact in fp64
  double* dev = nullptr;
  LBM_CUDA(cudaMalloc(&dev, sizeof(double) * rec.size()));
  auto exchange = [&]() -> int {
    LBM_CUDA(cudaMemcpyAsync(dev + (size_t)c->rank * NREC, mine, sizeof(double) * NREC, cudaMemcpyHostToDevice, d->stream));
    LBM_NCCL_GROUP_BEGIN();
    for (int k = 0; k < P; k++)
    {
      if (k == c->rank) continue;
      LBM_NCCL(g_nccl.Send(dev + (size_t)c->rank * NREC, NREC, ncclFloat64, k, c->comm, d->stream));
      LBM_NCCL(g_nccl.Recv(dev + (size_t)k * NREC, NREC, ncclFloat64, k, c->comm, d->stream));
    }
    LBM_NCCL_GROUP_END();
    LBM_CUDA(cudaMemcpyAsync(rec.data(), dev, sizeof(double) * rec.size(), cudaMemcpyDeviceToHost, d->stream));
    LBM_CUDA(cudaStreamSynchronize(d->stream));
    return LBM_OK;
  };
  const int rc = exchange();
  cudaFree(dev);
  if (rc != LBM_OK) return rc;
  const char* names[5] = {"X", "Y", "model", "force", "equilibrium"};
  for (int k = 0; k < P; k++)
  {
    const double* r = rec.data() + (size_t)k * NREC;
    for (int f = 0; f < 5; f++)
      if (r[f] != rec[f])
      {
        set_error("lbm_comm_check: rank %d was created with %s = %g, rank 0 with %g", k, names[f], r[f], rec[f]);
        return LBM_ERR_COMM;
      }
  }
  // every slab that owns rows of some rank's ROI must hold that very marker list
  for (int k = 0; k < P; k++)
  {
    const double* r = rec.data() + (size_t)k * NREC;
    if (r[5] == 0.0) continue;
    for (int j = 0; j < P; j++)
    {
      int jx0 = 0, jx1 = 0;
      lbm_decompose_rows(d->cfg.X, P, j, &jx0, &jx1);
      if ((double)jx1 <= r[6] || (double)jx0 >= r[7]) continue;  // rank j owns none of these ROI rows
      const double* q = rec.data() + (size_t)j * NREC;
      if (q[5] != r[5] || q[8] != r[8] || q[9] != r[9])
      {
        set_error("lbm_comm_check: the immersed body rank %d was given (%d markers, ROI rows [%d,%d)) crosses the slab of rank %d, "
                  "which was given %s: hand lbm_ibm_set_markers the same list on every rank of the ring",
                  k, (int)r[5], (int)r[6], (int)r[7], j, q[5] == 0.0 ? "no markers" : "a different list");
        return LBM_ERR_COMM;
      }
    }
  }
  return LBM_OK;
}

int lbm_link_neighbours(lbm_domain* d, lbm_domain* lower, lbm_domain* upper)
{
  if (!d) { set_error("lbm_link_neighbours: null domain"); return LBM_ERR_INVALID; }
  for (lbm_domain* o : {lower, upper})
  {
    if (!o) continue;
    if (o->cfg.Y != d->cfg.Y || o->cfg.X != d->cfg.X || o->nlat != d->nlat)
    {
      set_error("lbm_link_neighbours: slabs of different grids / models");
      return LBM_ERR_INVALID;
    }
    if (o->cfg.device != d->cfg.device)
    {
      int can = 0;
      LBM_CUDA(cudaDeviceCanAccessPeer(&can, d->cfg.device, o->cfg.device));
      if (can)
      {
        LBM_CUDA(cudaSetDevice(d->cfg.device));
        cudaError_t e = cudaDeviceEnablePeerAccess(o->cfg.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) LBM_CUDA(e);
        cudaGetLastError();
      }
    }
  }
  d->link_lo = lower;
  d->link_hi = upper;
  d->side_ready = false;
  drop_graphs(d);
  return LBM_OK;
}

int lbm_link_face(lbm_domain* d, int side, int row_begin, int n_rows, lbm_domain* other, int other_row_begin)
{
  if (!d || !other || (side != 0 && side != 1) || n_rows < 1) { set_error("lbm_link_face: bad argument"); return LBM_ERR_INVALID; }
  if (d->tp || other->tp || d->nlat != other->nlat)
  {
    set_error("lbm_link_face: column faces are built for the single-phase models (the two-phase moment planes have no column halo)");
    return LBM_ERR_UNSUPPORTED;
  }
  if (d->cfg.x0 != 0 || d->cfg.x1 != d->cfg.X || other->cfg.x0 != 0 || other->cfg.x1 != other->cfg.X)
  {
    set_error("lbm_link_face: a block bound across a column face must own all of its rows (no row slabs)");
    return LBM_ERR_UNSUPPORTED;
  }
  if (row_begin < 0 || row_begin + n_rows > d->cfg.X || other_row_begin < 0 || other_row_begin + n_rows > other->cfg.X)
  {
    set_error("lbm_link_face: rows [%d,%d) / [%d,%d) outside the blocks", row_begin, row_begin + n_rows, other_row_begin, other_row_begin + n_rows);
    return LBM_ERR_INVALID;
  }
  for (const auto& fl : d->faces)
    if (fl.side == side && row_begin < fl.rb + fl.n && fl.rb < row_begin + n_rows)
    {
      set_error("lbm_link_face: rows [%d,%d) of side %d are already bound", row_begin, row_begin + n_rows, side);
      return LBM_ERR_INVALID;
    }
  FaceLink fl;
  fl.side = side; fl.rb = row_begin; fl.n = n_rows; fl.orb = other_row_begin; fl.other = other;
  fl.other_device = other->cfg.device;
  LBM_CUDA(cudaSetDevice(other->cfg.device));
  LBM_CUDA(cudaMalloc(&fl.d_packet, sizeof(double) * d->nlat * 3 * n_rows));
  LBM_CUDA(cudaEventCreateWithFlags(&fl.ev, cudaEventDisableTiming));
  if (other->cfg.device != d->cfg.device)
  {
    int can = 0;
    LBM_CUDA(cudaDeviceCanAccessPeer(&can, d->cfg.device, other->cfg.device));
    if (can)
    {
      LBM_CUDA(cudaSetDevice(d->cfg.device));
      cudaError_t e = cudaDeviceEnablePeerAccess(other->cfg.device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) LBM_CUDA(e);
      cudaGetLastError();
    }
  }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  d->faces.push_back(fl);
  d->committed = false;  // the edge-column programs change: lbm_bc_commit again
  d->side_ready = false;
  drop_graphs(d);
  return LBM_OK;
}

// ---- the same binding between blocks on different ranks.  One process per block: lbm_comm_init_blocks makes the
// communicator (no slab ring: the blocks are independent grids), lbm_link_face_rank declares what THIS block reads, and
// lbm_comm_faces_commit — collective — lets every rank learn which of its rows the others read.
int lbm_comm_init_blocks(lbm_domain* d, const char id[LBM_UNIQUE_ID_BYTES], int n_ranks, int rank)
{
  if (!d || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) { set_error("lbm_comm_init_blocks: bad argument"); return LBM_ERR_INVALID; }
  if (d->tp) { set_error("lbm_comm_init_blocks: column faces are built for the single-phase models"); return LBM_ERR_UNSUPPORTED; }
  if (d->cfg.x0 != 0 || d->cfg.x1 != d->cfg.X) { set_error("lbm_comm_init_blocks: a block owns all of its rows (no row slabs)"); return LBM_ERR_UNSUPPORTED; }
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  comm_release(d);
  LBM_TRY(load_nccl());
  CommState* c = new CommState();
  c->n_ranks = n_ranks;
  c->rank = rank;
  c->blocks = true;
  c->handle = std::make_shared<CommHandle>();
  ncclUniqueId u;
  std::memcpy(&u, id, sizeof(u));
  ncclResult_t r = g_nccl.CommInitRank(&c->handle->comm, n_ranks, u, rank);
  if (r != 0)
  {
    set_error("ncclCommInitRank failed: %s", g_nccl.GetErrorString(r));
    c->handle->comm = nullptr;
    delete c;
    return LBM_ERR_COMM;
  }
  c->comm = c->handle->comm;
  d->comm = c;
  d->side_ready = false;
  return LBM_OK;
}

int lbm_link_face_rank(lbm_domain* d, int side, int row_begin, int n_rows, int peer_rank, int peer_row_begin)
{
  if (!d || (side != 0 && side != 1) || n_rows < 1 || peer_row_begin < 0) { set_error("lbm_link_face_rank: bad argument"); return LBM_ERR_INVALID; }
  if (!comm_blocks(d)) { set_error("lbm_link_face_rank: call lbm_comm_init_blocks first"); return LBM_ERR_INVALID; }
  if (peer_rank < 0 || peer_rank >= d->comm->n_ranks || peer_rank == d->comm->rank)
  {
    set_error("lbm_link_face_rank: peer rank %d of %d (this is rank %d; bind blocks of one process with lbm_link_face)", peer_rank, d->comm->n_ranks,
              d->comm->rank);
    return LBM_ERR_INVALID;
  }
  if (row_begin < 0 || row_begin + n_rows > d->cfg.X) { set_error("lbm_link_face_rank: rows [%d,%d) outside the block", row_begin, row_begin + n_rows); return LBM_ERR_INVALID; }
  for (const auto& fl : d->faces)
    if (fl.side == side && row_begin < fl.rb + fl.n && fl.rb < row_begin + n_rows)
    {
      set_error("lbm_link_face_rank: rows [%d,%d) of side %d are already bound", row_begin, row_begin + n_rows, side);
      return LBM_ERR_INVALID;
    }
  FaceLink fl;
  fl.side = side; fl.rb = row_begin; fl.n = n_rows; fl.orb = peer_row_begin; fl.other = nullptr; fl.peer_rank = peer_rank;
  fl.other_device = d->cfg.device;
  d->faces.push_back(fl);
  d->committed = false;  // the edge-column programs change: lbm_bc_commit again
  d->side_ready = false;
  d->faces_remote_ready = false;
  drop_graphs(d);
  return LBM_OK;
}

// Collective over the block communicator, after every rank's lbm_link_face_rank calls: each rank hands every other its list
// of remote links (side, rows, the peer's rows); a rank finds the links that name it and from now on packs and sends those
// rows of its facing edge column every step.  Checks that the rows exist on the serving block.
int lbm_comm_faces_commit(lbm_domain* d)
{
  if (!d) { set_error("lbm_comm_faces_commit: null domain"); return LBM_ERR_INVALID; }
  if (!comm_blocks(d)) { set_error("lbm_comm_faces_commit: call lbm_comm_init_blocks first"); return LBM_ERR_INVALID; }
  CommState* c = d->comm;
  constexpr int MAXF = 16, NREC = 1 + 5 * MAXF;  // count, then (side, rb, n, orb, peer) per link
  const int P = c->n_ranks;
  LBM_CUDA(cudaSetDevice(d->cfg.device));
  std::vector<double> rec((size_t)P * NREC, 0.0);
  double* mine = rec.data() + (size_t)c->rank * NREC;
  int nf = 0;
  for (const auto& fl : d->faces)
  {
    if (fl.peer_rank < 0) continue;
    if (nf == MAXF) { set_error("lbm_comm_faces_commit: more than %d remote links on one block", MAXF); return LBM_ERR_UNSUPPORTED; }
    double* r = mine + 1 + 5 * nf++;
    r[0] = fl.side; r[1] = fl.rb; r[2] = fl.n; r[3] = fl.orb; r[4] = fl.peer_rank;
  }
  mine[0] = nf;
  double* dev = nullptr;
  LBM_CUDA(cudaMalloc(&dev, sizeof(double) * rec.size()));
  auto exchange = [&]() -> int {
    LBM_CUDA(cudaMemcpyAsync(dev + (size_t)c->rank * NREC, mine, sizeof(double) * NREC, cudaMemcpyHostToDevice, d->stream));
    LBM_NCCL_GROUP_BEGIN();
    for (int k = 0; k < P; k++)
    {
      if (k == c->rank) continue;
      LBM_NCCL(g_nccl.Send(dev + (size_t)c->rank * NREC, NREC, ncclFloat64, k, c->comm, d->stream));
      LBM_NCCL(g_nccl.Recv(dev + (size_t)k * NREC, NREC, ncclFloat64, k, c->comm, d->stream));
    }
    LBM_NCCL_GROUP_END();
    LBM_CUDA(cudaMemcpyAsync(rec.data(), dev, sizeof(double) * rec.size(), cudaMemcpyDeviceToHost, d->stream));
    LBM_CUDA(cudaStreamSynchronize(d->stream));
    return LBM_OK;
  };
  const int rc = exchange();
  cudaFree(dev);
  if (rc != LBM_OK) return rc;
  for (auto& sv : d->serves) cudaFree(sv.d_packet);
  d->serves.clear();
  for (int k = 0; k < P; k++)  // readers in rank order, their links in index order: the order both sides send / receive in
  {
    if (k == c->rank) continue;
    const double* r = rec.data() + (size_t)k * NREC;
    for (int j = 0; j < (int)r[0]; j++)
    {
      const double* q = r + 1 + 5 * j;
      if ((int)q[4] != c->rank) continue;
      FaceServe sv;
      sv.reader_side = (int)q[0]; sv.n = (int)q[2]; sv.rb = (int)q[3]; sv.peer_rank = k;
      if (sv.rb < 0 || sv.rb + sv.n > d->cfg.X)
      {
        set_error("lbm_comm_faces_commit: rank %d binds rows [%d,%d) of this block, which has %d rows", k, sv.rb, sv.rb + sv.n, d->cfg.X);
        return LBM_ERR_COMM;
      }
      LBM_CUDA(cudaMalloc(&sv.d_packet, sizeof(double) * d->nlat * 3 * sv.n));
      d->serves.push_back(sv);
    }
  }
  d->faces_remote_ready = true;
  d->side_ready = false;
  return LBM_OK;
}


// Face tails of every bound block: the facing edge columns of the other blocks (written by their listed-node kernels on
// their side streams) packed there, copied here on this block's side stream ahead of its next listed-node kernel.
// new_buffer: the buffers being written by the step in flight (cur ^ 1) rather than the current ones.
static int group_faces(lbm_domain* const* ds, int n, bool new_buffer)
{
  for (int i = 0; i < n; i++)
  {
    lbm_domain* d = ds[i];
    for (auto& fl : d->faces)
    {
      if (fl.peer_rank >= 0) continue;  // a block on another rank: faces_exchange_remote
      lbm_domain* o = fl.other;
      bool member = false;
      for (int j = 0; j < n; j++) member = member || ds[j] == o;
      if (!member || !o->have_state) { set_error("lbm_step_group: a block is bound to a block outside the group"); return LBM_ERR_INVALID; }
      const int ow = new_buffer ? o->cur ^ 1 : o->cur, dw = new_buffer ? d->cur ^ 1 : d->cur;
      LBM_CUDA(on(o));
      LBM_CUDA(cudaStreamWaitEvent(o->side, d->ev_side, 0));  // the copy out of this packet one step ago
      const int total = d->nlat * 3 * fl.n;
      k_face_pack<<<(total + 127) / 128, 128, 0, o->side>>>(o->buf[0][ow], o->buf[1][ow], o->g, fl.side == 0 ? o->g.Y - 1 : 0, fl.orb,
                                                           fl.n, fl.side, d->nlat, fl.d_packet);
      o->launches++;
      LBM_CUDA(cudaGetLastError());
      LBM_CUDA(cudaEventRecord(fl.ev, o->side));
      LBM_CUDA(on(d));
      LBM_CUDA(cudaStreamWaitEvent(d->side, fl.ev, 0));
      ProfScope ps(d, LBM_PROF_GHOST, d->side);
      for (int l = 0; l < d->nlat; l++)
        for (int qi = 0; qi < 3; qi++)
          LBM_TRY(copy_rows(d, d->buf[l][dw] + face_tail_off(d->g, fl.side, qi, fl.rb), o, fl.d_packet + (size_t)(l * 3 + qi) * fl.n,
                            (size_t)fl.n, d->side));
    }
  }
  return LBM_OK;
}

// Immersed-boundary pre-pass of linked slabs: (a) every slab computes the moments of the active ROI nodes on its own rows
// from buffer `which`; (b) slabs that share a body copy each other's row segments; (c) each runs the forcing
// iterations into its slot and signals ev_side.  use_next: the pre-pass belongs to the step after the one being
// enqueued (side tail) rather than to this one (prologue).
static int group_ibm(lbm_domain* const* ds, int n, bool tail)
{
  for (int i = 0; i < n; i++)
  {
    lbm_domain* d = ds[i];
    if (!uses_ibm(d) || (!tail && d->side_ready)) continue;
    LBM_CUDA(on(d));
    if (d->ibm.split)  // the other owners may still be copying the segment of the pre-pass before
      for (int j = 0; j < n; j++)
        if (j != i && uses_ibm(ds[j]) && ds[j]->ibm.split) LBM_CUDA(cudaStreamWaitEvent(d->side, ds[j]->ev_side, 0));
    ProfScope ps(d, LBM_PROF_IBM, d->side);
    const int mode = tail ? MODE_PULL : (d->post_stream ? MODE_LOCAL : MODE_PULL);
    LBM_TRY(ibm_roi_local(d, mode, tail ? d->cur ^ 1 : d->cur, d->side));
    LBM_CUDA(cudaEventRecord(d->ev_ibm, d->side));
  }
  for (int i = 0; i < n; i++)
  {
    lbm_domain* d = ds[i];
    if (!uses_ibm(d) || (!tail && d->side_ready)) continue;
    LBM_CUDA(on(d));
    ProfScope ps(d, LBM_PROF_IBM, d->side);
    if (d->ibm.split)
    {
      const size_t RC = (size_t)(d->ibm.c1 - d->ibm.c0);
      for (int j = 0; j < n; j++)
      {
        lbm_domain* o = ds[j];
        if (j == i || !uses_ibm(o) || o->ibm.row_hi <= o->ibm.row_lo) continue;
        if (o->ibm.r0 != d->ibm.r0 || o->ibm.r1 != d->ibm.r1 || o->ibm.n_markers != d->ibm.n_markers)
        {
          set_error("lbm_step_group: slabs %d and %d carry different immersed bodies (hand every slab the same marker list)", i, j);
          return LBM_ERR_INVALID;
        }
        LBM_CUDA(cudaStreamWaitEvent(d->side, o->ev_ibm, 0));
        const size_t lo = (size_t)o->ibm.row_lo * RC, cnt = (size_t)(o->ibm.row_hi - o->ibm.row_lo) * RC;
        LBM_TRY(copy_rows(d, d->ibm.d_rho + lo, o, o->ibm.d_rho + lo, cnt, d->side));
        LBM_TRY(copy_rows(d, d->ibm.d_u + 2 * lo, o, o->ibm.d_u + 2 * lo, 2 * cnt, d->side));
      }
    }
    LBM_CUDA(cudaEventRecord(d->ev_ibm_got, d->side));
  }
  // (c) the forcing iterations update the ROI velocities in place: not before every co-owner has taken its copy
  for (int i = 0; i < n; i++)
  {
    lbm_domain* d = ds[i];
    if (!uses_ibm(d) || (!tail && d->side_ready)) continue;
    LBM_CUDA(on(d));
    ProfScope ps(d, LBM_PROF_IBM, d->side);
    if (d->ibm.split)
      for (int j = 0; j < n; j++)
        if (j != i && uses_ibm(ds[j]) && ds[j]->ibm.split) LBM_CUDA(cudaStreamWaitEvent(d->side, ds[j]->ev_ibm_got, 0));
    LBM_TRY(ibm_iterate(d, tail ? d->ibm.next_slot ^ 1 : d->ibm.next_slot, d->side));
    LBM_CUDA(cudaEventRecord(d->ev_side, d->side));
  }
  return LBM_OK;
}

// Advance a set of linked slabs in lock step: the phases of one step (lbm_domain.cu) interleaved
// across the slabs, with the ghost rows and pressure packets copied between the slabs' side streams.
int lbm_step_group(lbm_domain* const* ds, int n, int n_steps)
{
  if (!ds || n < 1 || n_steps < 0) { set_error("lbm_step_group: bad argument"); return LBM_ERR_INVALID; }
  for (int i = 0; i < n; i++)
  {
    if (!ds[i] || !ds[i]->have_state || !ds[i]->committed) { set_error("lbm_step_group: slab %d has no state / uncommitted rules", i); return LBM_ERR_INVALID; }
    if ((ds[i]->tp != nullptr) != (ds[0]->tp != nullptr)) { set_error("lbm_step_group: slabs of different models"); return LBM_ERR_INVALID; }
    if (ds[i]->stages.size() != ds[0]->stages.size()) { set_error("lbm_step_group: slabs carry different rule lists"); return LBM_ERR_INVALID; }
    if (ds[i]->cur != ds[0]->cur || ds[i]->post_stream != ds[0]->post_stream) { set_error("lbm_step_group: slabs are out of step"); return LBM_ERR_INVALID; }
  }
  for (int i = 0; i < n; i++)
    for (const auto& fl : ds[i]->faces)
    {
      bool member = fl.peer_rank >= 0;  // (blocks on other ranks are not advanced by a group)
      for (int j = 0; j < n; j++) member = member || ds[j] == fl.other;
      if (!member) { set_error("lbm_step_group: block %d is bound across a column face to a block outside the group", i); return LBM_ERR_INVALID; }
    }
  if (ds[0]->tp) return tp_step_group(ds, n, n_steps);
  for (int i = 0; i < n; i++)
  {
    LBM_CUDA(on(ds[i]));
    LBM_CUDA(cudaEventRecord(ds[i]->ev_begin, ds[i]->stream));
  }
  for (int s = 0; s < n_steps; s++)
  {
    // ---- state nobody prepared yet (first step): ghost rows from the neighbours + IBM field
    bool any = false;
    for (int i = 0; i < n; i++) any = any || !ds[i]->side_ready;
    if (any)
    {
      for (int i = 0; i < n; i++)
      {
        LBM_CUDA(on(ds[i]));
        LBM_CUDA(cudaEventRecord(ds[i]->ev_ready, ds[i]->stream));
      }
      for (int i = 0; i < n; i++)
      {
        lbm_domain* d = ds[i];
        if (d->side_ready) continue;
        LBM_CUDA(on(d));
        if (!d->post_stream)
        {
          for (lbm_domain* o : {d->link_lo, d->link_hi})
            if (o) LBM_CUDA(cudaStreamWaitEvent(d->side, o->ev_ready, 0));
          LBM_CUDA(cudaStreamWaitEvent(d->side, d->ev_ready, 0));
          ProfScope ps(d, LBM_PROF_GHOST, d->side);
          if (d->link_lo || d->link_hi) LBM_TRY(link_exchange(d, d->cur, d->side));
          else LBM_TRY(wrap_ghost_rows_local(d, d->cur, d->side));
        }
        LBM_TRY(step_prologue(d, false, false));
      }
      if (!ds[0]->post_stream)
      {
        LBM_TRY(group_faces(ds, n, false));
        for (int i = 0; i < n; i++)
          if (!ds[i]->faces.empty()) { LBM_CUDA(on(ds[i])); LBM_CUDA(cudaEventRecord(ds[i]->ev_side, ds[i]->side)); }
      }
      LBM_TRY(group_ibm(ds, n, false));
      for (int i = 0; i < n; i++) ds[i]->side_ready = true;
    }
    // ---- early rows, listed nodes
    for (int i = 0; i < n; i++) { LBM_CUDA(on(ds[i])); LBM_TRY(step_early(ds[i])); }
    for (int i = 0; i < n; i++) { LBM_CUDA(on(ds[i])); LBM_TRY(step_listed(ds[i])); }
    LBM_TRY(group_faces(ds, n, true));  // the edge columns just written feed the bound blocks' next step
    // ---- pre-stream stages, packets handed from the source owner to the writer
    for (size_t k = 0; k < ds[0]->stages.size(); k++)
    {
      lbm_domain *src = nullptr, *dst = nullptr;
      for (int i = 0; i < n; i++)
      {
        LBM_CUDA(on(ds[i]));
        LBM_TRY(stage_pack(ds[i], k));
        if (ds[i]->stages[k].kind == 1 && ds[i]->stages[k].own_src) src = ds[i];
        if (ds[i]->stages[k].kind == 1 && ds[i]->stages[k].own_dst) dst = ds[i];
      }
      if (src && dst && src != dst)
      {
        LBM_CUDA(on(src));
        LBM_CUDA(cudaEventRecord(src->ev_packet, src->side));
        LBM_CUDA(on(dst));
        LBM_CUDA(cudaStreamWaitEvent(dst->side, src->ev_packet, 0));
        LBM_TRY(copy_rows(dst, dst->stages[k].d_packet, src, src->stages[k].d_packet, (size_t)12 * dst->g.Y, dst->side));
      }
      for (int i = 0; i < n; i++) { LBM_CUDA(on(ds[i])); LBM_TRY(stage_apply(ds[i], k)); }
    }
    for (int i = 0; i < n; i++) { LBM_CUDA(on(ds[i])); LBM_CUDA(cudaEventRecord(ds[i]->ev_stage, ds[i]->side)); }
    // ---- ghost rows of the new buffers, next IBM field
    for (int i = 0; i < n; i++)
    {
      lbm_domain* d = ds[i];
      LBM_CUDA(on(d));
      LBM_TRY(wait_linked(d, d->side, &lbm_domain::ev_stage));
      {
        ProfScope ps(d, LBM_PROF_GHOST, d->side);
        if (d->link_lo || d->link_hi) LBM_TRY(link_exchange(d, d->cur ^ 1, d->side));
        else LBM_TRY(wrap_ghost_rows_local(d, d->cur ^ 1, d->side));
      }
      LBM_TRY(step_side_tail(d, false, false));
    }
    LBM_TRY(group_ibm(ds, n, true));
    // ---- bulk rows
    for (int i = 0; i < n; i++) { LBM_CUDA(on(ds[i])); LBM_TRY(step_bulk(ds[i])); }
  }
  for (int i = 0; i < n; i++)
  {
    LBM_CUDA(on(ds[i]));
    LBM_CUDA(cudaEventRecord(ds[i]->ev_end, ds[i]->stream));
  }
  return LBM_OK;
}

}  // extern "C"
