// lbm_internal.hpp — host-side state of one slab (the opaque lbm_domain of include/lbm_b200.h).
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/lbm_b200.h"
#include "lbm_bgk_kernels.cuh"

namespace lbm
{

void set_error(const char* fmt, ...);

#define LBM_CUDA(call)                                                                         \
  do                                                                                           \
  {                                                                                            \
    cudaError_t e__ = (call);                                                                  \
    if (e__ != cudaSuccess)                                                                    \
    {                                                                                          \
      lbm::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
      return LBM_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)

#define LBM_TRY(call)              \
  do                               \
  {                                \
    int s__ = (call);              \
    if (s__ != LBM_OK) return s__; \
  } while (0)

struct StoredOp
{
  lbm_bc_op op;
  std::vector<double> per_row;
};

// One pre-stream rule, in the order the rules were added.  Every slab builds the same list (the
// rules are global), so stage k of one slab pairs with stage k of every other slab.
struct Stage
{
  int kind = 0;  // 0 = copy group (local), 1 = pressure-periodic row
  // copy group
  int n = 0;
  FixEntry* d_entries = nullptr;
  // pressure row
  int dst_gx = 0, src_gx = 0, y_lo = 0, y_hi = 0;
  double rho_bc = 1.0;
  bool own_src = false, own_dst = false;
  int* d_src_bidx = nullptr;  // [Y] boundary-node index of the source-row nodes (owner of the source row)
  double* d_packet = nullptr; // [12][Y] packed by the source owner; the writer reads it (its own copy when remote)
};

struct IbmState
{
  bool enabled = false;
  int n_markers = 0, m_max = 5;
  long r0 = 0, r1 = 0, c0 = 0, c1 = 0;  // global ROI [r0,r1) x [c0,c1)
  // markers
  int* d_mrow = nullptr;   // box start row / col in ROI coordinates
  int* d_mcol = nullptr;
  double* d_phi = nullptr; // [n][16]
  double* d_fj = nullptr;  // [n][2]
  // nodes covered by some marker box ("active"), and for each its (marker, weight) list in marker order
  int n_active = 0;
  int* d_active = nullptr; // [n_active] ROI-local node ids
  int* d_ptr = nullptr;    // [n_active + 1]
  int* d_ent_marker = nullptr;
  double* d_ent_phi = nullptr;
  // ROI fields
  double* d_u = nullptr;   // [roi][2]
  double* d_rho = nullptr; // [roi]
  double* d_Fx[2] = {nullptr, nullptr};  // [roi], double-buffered: the pre-pass of step t+1 runs while
  double* d_Fy[2] = {nullptr, nullptr};  // the bulk rows of step t still read the field of step t
  // A body whose ROI rows cross a slab cut: every slab that owns ROI rows keeps the WHOLE solve (markers, lists, ROI
  // fields); it computes the moments of the active nodes on its own rows, the slabs swap those row segments, and each
  // runs the (tiny) forcing iterations redundantly — identical arithmetic, so the force field is the same on all of them.
  // lbm_set_force_region: the field is a constant the caller gave (no markers, no pre-pass)
  bool fixed = false;
  bool split = false;
  int row_lo = 0, row_hi = 0;  // ROI-local rows owned by this slab
  int a_lo = 0, a_hi = 0;      // range of the active list that lies on those rows
  int next_slot = 0;  // slot the next step reads (filled by the last pre-pass)
  int used_slot = 0;  // slot the last enqueued step read (lbm_ibm_get_force)
};

// the marker list as lbm_ibm_set_markers was handed it (kept on slabs that own none of its ROI rows too): what
// lbm_comm_check compares across the ring
struct IbmGiven
{
  int n = 0;
  long r0 = 0, r1 = 0;
  unsigned long long hash = 0;
};

// lbm_body_force_record: the force on one body, summed on the device once per step into a ring (lbm_body_force.cuh)
struct BodyForce
{
  bool on = false;
  bool immersed = false;          // the immersed body's force field; otherwise the bounce-back links of a solid mask
  int capacity = 0;               // steps the ring keeps
  int n = 0;                      // links, or active ROI nodes on this slab's rows
  long long* d_link = nullptr;    // [n] (offset of f[opp(q)] at the link's fluid node in a lattice buffer) << 4 | q, by (node, q)
  double* d_part = nullptr;       // [blocks][2] per-block partial sums
  double* d_ring = nullptr;       // [capacity][2]
  long long* d_count = nullptr;   // steps recorded so far (advanced by the kernel, so graph replays count too)
};

// lbm_stats_start: time-averaged moments, accumulated by the STATS instantiations of the step kernels (lbm_stats.cuh)
struct Stats
{
  bool on = false;
  int every = 1;
  double* d_acc = nullptr;       // [6][Xl][pitch]: mean rho, mean ux, mean uy, Mxx, Myy, Mxy (StatsArgs)
  StatsClock* d_clock = nullptr; // steps since lbm_stats_start and 1 / n of the next sample (advanced on the device, so
                                 // graph replays count too)
  unsigned* d_listed = nullptr;  // [Xl][words]: one bit per listed node in an interior column, rebuilt by lbm_bc_commit
  int words = 0;
};

struct ProfRec
{
  cudaEvent_t a, b;
  int cls;
};

struct TwoPhaseState;  // lbm_two_phase.cu
struct CommState;      // lbm_comm.cu

}  // namespace lbm

namespace lbm
{
// test/decompose_domain_loop.cpp:232-261, one direction of one face: rows [rb, rb + n) of this block's edge column
// `side` (0 = first column: populations 2, 5, 6 enter; 1 = last column: 4, 7, 8) are fed by rows [orb, orb + n) of the
// facing edge column of `other`
struct FaceLink
{
  int side = 0, rb = 0, n = 0, orb = 0;
  lbm_domain* other = nullptr;  // the facing block in this process (lbm_link_face) ...
  int peer_rank = -1;           // ... or the rank that owns it (lbm_link_face_rank): its column arrives over NCCL
  int other_device = 0;        // kept separately: `other` may be destroyed before this block is
  double* d_packet = nullptr;  // [lattice][3][n] on other's device
  cudaEvent_t ev = nullptr;    // packet packed (other's side stream)
};
// what this block packs and sends so that a block on another rank can read it through ITS face link (the mirror image of
// that rank's FaceLink, derived from the descriptors the ranks exchange in lbm_comm_faces_commit)
struct FaceServe
{
  int reader_side = 0;         // the READER's side: 0 = it reads our last column (populations 2, 5, 6), 1 = our first (4, 7, 8)
  int rb = 0, n = 0;           // our rows
  int peer_rank = 0;
  double* d_packet = nullptr;  // [lattice][3][n]
};
// the three populations that enter through the first (side 0: c_y = +1) / last (side 1: c_y = -1) column
__host__ __device__ inline int face_q(int side, int qi) { return side == 0 ? (qi == 0 ? 2 : (qi == 1 ? 5 : 6)) : (qi == 0 ? 4 : (qi == 1 ? 7 : 8)); }
inline long long face_tail_off(const SlabGeom& g, int side, int qi, int row) { return 9 * g.plane + (long long)(side * 3 + qi) * g.Xl + row; }
}  // namespace lbm

struct lbm_domain
{
  lbm_config cfg;
  lbm::SlabGeom g;
  int nlat = 1;
  double* buf[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};  // [lattice][buffer]
  int cur = 0;              // buffer holding the current state
  bool post_stream = true;  // true: buf[cur] = f_adve (just imported); false: buf[cur] = f_coll
  bool have_state = false;
  int npairs = 0;           // interior column pairs per row (single-phase kernels)
  int y_int_begin = 2;      // columns [y_int_begin, y_int_end) belong to the interior kernel,
  int y_int_end = 2;        // every other column is a listed (table-driven) node
  cudaStream_t stream = nullptr;
  cudaStream_t side = nullptr;      // IBM pre-pass / ghost exchange, overlapped with the interior rows
  cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
  cudaEvent_t ev_ready = nullptr;   // everything enqueued so far on the main stream
  cudaEvent_t ev_early = nullptr;   // early rows of the step written (main stream)
  cudaEvent_t ev_side = nullptr;    // side chain done: listed nodes, stages, ghost rows, next IBM field
  cudaEvent_t ev_stage = nullptr;   // listed nodes + stages done (side stream), linked slabs
  cudaEvent_t ev_ibm_got = nullptr; // ... and the co-owners' segments copied in
  cudaEvent_t ev_ibm = nullptr;     // moments of this slab's active ROI nodes done (side stream), linked slabs sharing a body
  cudaEvent_t ev_packet = nullptr;  // pressure packet packed (side stream), linked slabs
  bool side_ready = false;          // ghost rows of buf[cur] and the IBM field for the next step are (being) prepared
  // row lists of the interior kernel
  bool rows_dirty = true;
  int n_early = 0, n_bulk = 0;
  bool early_on_side = false;  // this step's early rows were launched on the side stream (no bulk rows to overlap)
  int *d_rows_all = nullptr, *d_rows_early = nullptr, *d_rows_bulk = nullptr;
  std::vector<char> row_has_listed;  // row owns a listed node in an interior column, or feeds a stage
  std::vector<int> listed_ids;       // local node ids x * Y + y of the listed nodes, ascending (commit_boundary_tables)
  float last_ms = 0.f;
  long long launches = 0;

  // boundary description and its compiled form
  std::vector<lbm::StoredOp> ops;
  bool committed = false;
  int nb = 0;
  int *d_bx = nullptr, *d_by = nullptr;
  lbm::BcEntry* d_ent = nullptr;
  double* d_mom[2] = {nullptr, nullptr};
  int mom_cur = 0;
  std::vector<lbm::Stage> stages;
  std::vector<int32_t> mask[2];
  bool wrap_all_q = false;  // some rule reads a whole row across the periodic wrap

  // scratch for export
  double* d_aos[2] = {nullptr, nullptr};
  double* d_mom_in = nullptr;   // LBM_MODEL_KBC: caller's rho {Xl,Y}, u {Xl,Y,2} for the first step (lbm_set_moments)
  bool mom_in_valid = false;
  // snapshot staging: [6][Xl*Y] rho, u (2), phase, rho_r, rho_b — filled on `stream`, drained either on `stream`
  // (lbm_get_moments / lbm_get_phase) or on `copy` while later steps run (lbm_snapshot_async)
  double* d_mom_out = nullptr;
  double* d_stage_in = nullptr;  // import staging area (lbm_init_equilibrium always; the other imports while an async snapshot still reads d_mom_out)
  cudaStream_t copyin = nullptr;  // host->device copies of lbm_init_equilibrium, beside the domain's stream
  cudaEvent_t ev_h2d = nullptr, ev_stage_free = nullptr;
  bool stage_in_busy = false;
  cudaStream_t copy = nullptr;
  cudaEvent_t ev_staged = nullptr, ev_copied = nullptr;
  bool copy_pending = false;

  lbm::IbmState ibm;
  lbm::IbmGiven ibm_given;
  lbm::BodyForce bf;
  lbm::Stats st;
  double ics2 = 1.0 / 3.0, ics4 = 1.0 / 9.0;  // source-term constants (lbm_set_force_region overrides them)
  // column-face bindings to other blocks (lbm_link_face): the populations entering through an edge column are read
  // from a tail appended to every lattice buffer, [side][3 populations][Xl] behind the nine planes
  std::vector<lbm::FaceLink> faces;
  std::vector<lbm::FaceServe> serves;   // remote readers of this block's edge columns (lbm_comm_faces_commit)
  bool faces_remote_ready = false;       // the descriptors have been exchanged since the last lbm_link_face_rank
  lbm::TwoPhaseState* tp = nullptr;
  lbm::CommState* comm = nullptr;
  lbm_domain *link_lo = nullptr, *link_hi = nullptr;

  // optional per-kernel-class timing
  bool profiling = false;
  std::vector<lbm::ProfRec> prof;
  size_t prof_used = 0;

  // CUDA graph of one steady-state step pair
  bool use_graph = false;
  cudaGraphExec_t graph_exec[2] = {nullptr, nullptr};  // keyed by the buffer the pair starts from
  long long graph_launches[2] = {0, 0};                // kernels one replay launches
  bool skip_side_wait = false;                         // first step of a captured pair
};

namespace lbm
{
// drivers of linked slabs: make the slab's device current, and let `st` wait for event `ev` of each linked neighbour
// (a slab linked to itself waits for nothing)
inline cudaError_t on(const lbm_domain* d) { return cudaSetDevice(d->cfg.device); }
inline int wait_linked(const lbm_domain* d, cudaStream_t st, cudaEvent_t lbm_domain::*ev)
{
  for (const lbm_domain* o : {d->link_lo, d->link_hi})
    if (o && o != d) LBM_CUDA(cudaStreamWaitEvent(st, o->*ev, 0));
  return LBM_OK;
}
// the immersed body's pre-pass runs every step (markers, not a fixed region force)
inline bool uses_ibm(const lbm_domain* d) { return d->ibm.enabled && !d->ibm.fixed && d->cfg.force == LBM_FORCE_IBM; }
// lbm_domain.cu
int ensure_aos_scratch(lbm_domain* d);
void drop_graphs(lbm_domain* d);
// persistent [6][Xl*Y] device staging for host fields on their way in or out (waits for a pending snapshot copy)
int host_staging(lbm_domain* d, double** out);  // captured step pairs hold device pointers: drop them when tables / markers change
// brackets a group of launches of one class with events when profiling is on
struct ProfScope
{
  lbm_domain* d;
  cudaStream_t st;
  long idx = -1;
  ProfScope(lbm_domain* dom, int cls, cudaStream_t stream = nullptr);
  ~ProfScope();
};
int commit_boundary_tables(lbm_domain* d);
// step phases (lbm_domain.cu); lbm_comm.cu interleaves them across linked slabs
int step_rows(lbm_domain* d);                            // (re)build the early / bulk row lists
int step_early(lbm_domain* d);                           // main: wait side chain, early rows, record ev_early
int step_listed(lbm_domain* d);                          // side: wait ev_early, listed-node kernel
int stage_pack(lbm_domain* d, size_t k);                 // side: source half of stage k
int stage_apply(lbm_domain* d, size_t k);                // side: writer half of stage k
int step_side_tail(lbm_domain* d, bool exchange_local, bool with_ibm);  // side: ghost rows of the new buffer, next IBM field, ev_side
int step_bulk(lbm_domain* d);                            // main: bulk rows, then the buffer swap
int step_prologue(lbm_domain* d, bool exchange_local, bool with_ibm);   // side chain for a state no step has prepared yet
int wrap_ghost_rows_local(lbm_domain* d, int which, cudaStream_t st);
// lbm_ibm.cu
int ibm_release(lbm_domain* d);
int ibm_prepass(lbm_domain* d, int mode, int which, int slot, cudaStream_t st);
int ibm_roi_local(lbm_domain* d, int mode, int which, cudaStream_t st);  // moments of the active ROI nodes on this slab's rows
int ibm_iterate(lbm_domain* d, int slot, cudaStream_t st);               // forcing iterations on the complete ROI fields
int comm_ibm_share(lbm_domain* d, cudaStream_t st);
int faces_release(lbm_domain* d);                      // NCCL: ROI row segments between the slabs that own ROI rows
// lbm_body_force.cuh (compiled inside lbm_domain.cu)
void body_force_release(lbm_domain* d);
int body_force_step(lbm_domain* d);  // side: the force of the step being enqueued into the ring (no-op when not recording)
// lbm_stats.cuh (compiled inside lbm_domain.cu)
void stats_release(lbm_domain* d);
int stats_listed_mask(lbm_domain* d);  // (re)build the listed-node bit mask from listed_ids
int stats_tick(lbm_domain* d);         // main, after the bulk rows: wait for the side chain, advance the sample counter
// lbm_two_phase.cu
int tp_create(lbm_domain* d);
int tp_destroy(lbm_domain* d);
int tp_step(lbm_domain* d);
bool tp_ring_overlap_ok(lbm_domain* d);   // ring rank in the steady state whose halos can travel behind the interior bands
int tp_steps_ring(lbm_domain* d, int n);  // n such steps (both exchanges on the side stream; joined into d->stream at the end)
int tp_step_group(lbm_domain* const* ds, int n, int n_steps);  // linked two-phase slabs in lock step
int tp_commit(lbm_domain* d);
int tp_export(lbm_domain* d);
int tp_stage_moments(lbm_domain* d, double* stage);  // planes -> [6][N] staging (rho, u, phase, rho_r, rho_b)
int stage_fields(lbm_domain* d, int lattice);        // lbm_domain.cu: fills d->d_mom_out on d->stream
int tp_refresh_moments(lbm_domain* d);
// lbm_comm.cu
int comm_release(lbm_domain* d);
bool comm_active(const lbm_domain* d);
int link_exchange(lbm_domain* d, int which, cudaStream_t st);  // ghost rows from linked neighbours
int comm_exchange(lbm_domain* d, int which, cudaStream_t st);  // population ghost rows over NCCL
int comm_exchange_planes(lbm_domain* d, double* base, int nplanes, cudaStream_t st = nullptr);  // 2 ghost rows of planes in the moment-plane geometry
int comm_allreduce_max(lbm_domain* d, double* dev_value);  // ring-wide max of one non-negative device double (diagnostics)
int comm_exchange_moments(lbm_domain* d);  // two-phase: 2 ghost rows of the moment planes at slab cuts
int comm_stage_transfer(lbm_domain* d, size_t k, cudaStream_t st);  // pressure packet of stage k between ranks
bool comm_blocks(const lbm_domain* d);                              // member of a block communicator (lbm_comm_init_blocks): no slab ring
int faces_exchange_remote(lbm_domain* d, bool new_buffer);           // side stream: pack what remote readers need, send / receive the face tails
int comm_link_refresh(lbm_domain* d);                               // linked slabs: ghost rows of buf[cur] outside lbm_step_group
double* tp_moment_planes(lbm_domain* d, int* pm, long long* mplane);
}  // namespace lbm
