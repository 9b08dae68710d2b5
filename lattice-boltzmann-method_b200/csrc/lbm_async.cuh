// lbm_async.cuh — bulk asynchronous global -> shared copies (cp.async.bulk, the 1-D form of TMA) completed on mbarriers.
//
// The row-marching two-phase kernels stage whole population rows of their strip in shared memory this way: one lane
// issues a kilobyte-sized copy per population row segment, the copy engine moves it without passing through registers,
// and the block waits on the stage's mbarrier when it gets to that row — so several rows per block are in flight at any
// time, whatever the register allocation of the fp64 work.  SASS: UBLKCP (copy), SYNCS (mbarrier).
//
// Requirements of cp.async.bulk: source, destination and size are multiples of 16 bytes.
#pragma once
#include <cstdint>
#if defined(LBM_CPU_EMU)
#include <cstdio>
#include <cstdlib>
#include <cstring>
#endif

namespace lbm
{

#if !defined(LBM_CPU_EMU)

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}

// makes the initialised barriers visible to the async proxy (the copy engine); follow with __syncthreads()
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

// one arrival that also announces `bytes` of copy traffic the phase has to see before it completes
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, unsigned bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}

__device__ __forceinline__ void bulk_copy_g2s(void* dst_smem, const void* src_gmem, unsigned bytes, uint64_t* bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}

// blocks until the phase with the given parity has completed (0 for the first use of a barrier, then alternating)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity)
{
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "LBM_MBAR_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra LBM_MBAR_DONE;\n"
      "bra LBM_MBAR_WAIT;\n"
      "LBM_MBAR_DONE:\n"
      "}\n" ::"r"(smem_addr(bar)),
      "r"(parity)
      : "memory");
}

// ---- tensor memory (TMEM, 512 columns x 128 lanes x 32 bit per SM) as a per-thread stash.  No tensor-core work runs in
// these kernels; TMEM is idle capacity next to the 227 KB of shared memory, and a thread of a 128-thread block can park
// values in "its" lane (lane = threadIdx.x; a warp reaches the 32 lanes of its own sub-partition, warp_id % 4) and take them
// back a few rows later: tcgen05.st / tcgen05.ld in the 32x32b shape move N consecutive 32-bit columns of the thread's own
// lane.  SASS: STTM / LDTM.  All tcgen05 instructions here are warp-collective (.sync.aligned): every thread of the
// warp executes them, outside divergent code.
template <int COLS>
__device__ __forceinline__ uint32_t tmem_alloc(uint32_t* smem_slot)
{
  static_assert(COLS == 32 || COLS == 64 || COLS == 128 || COLS == 256 || COLS == 512, "TMEM allocations are powers of two >= 32 columns");
  if (threadIdx.x < 32)
  {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(smem_slot)), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  // this thread's lane: the warp's sub-partition base in the lane field (bits 31..16)
  return *smem_slot + (((threadIdx.x >> 5) & 3u) << 21);
}

template <int COLS>
__device__ __forceinline__ void tmem_free(uint32_t base)
{
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base & 0x0000ffffu), "n"(COLS) : "memory");
}

// 18 doubles (both colours' populations of one node) = 36 columns at `taddr` (thread-lane address + column offset)
__device__ __forceinline__ void tmem_store18(uint32_t taddr, const double (&a)[9], const double (&b)[9])
{
  uint32_t r[36];
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    r[2 * q] = (uint32_t)__double2loint(a[q]);
    r[2 * q + 1] = (uint32_t)__double2hiint(a[q]);
    r[18 + 2 * q] = (uint32_t)__double2loint(b[q]);
    r[18 + 2 * q + 1] = (uint32_t)__double2hiint(b[q]);
  }
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, "
      "%21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
      "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]),
      "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr + 32u), "r"(r[32]), "r"(r[33]), "r"(r[34]), "r"(r[35])
               : "memory");
}

__device__ __forceinline__ void tmem_store_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// the load in two halves, so that its latency can pass under other work: issue (the destination registers are written
// asynchronously), later wait, then read the registers
__device__ __forceinline__ void tmem_load18_issue(uint32_t taddr, uint32_t (&r)[36])
{
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, "
      "%21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
        "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
        "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]) : "r"(taddr + 32u) : "memory");
}
__device__ __forceinline__ void tmem_load_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_unpack18(uint32_t (&r)[36], double (&a)[9], double (&b)[9])
{
  // the registers pass through an empty volatile statement first: nothing may read them ahead of the wait above
#pragma unroll
  for (int c = 0; c < 36; c++) asm volatile("" : "+r"(r[c])::"memory");
#pragma unroll
  for (int q = 0; q < 9; q++)
  {
    a[q] = __hiloint2double((int)r[2 * q + 1], (int)r[2 * q]);
    b[q] = __hiloint2double((int)r[18 + 2 * q + 1], (int)r[18 + 2 * q]);
  }
}
__device__ __forceinline__ void tmem_load18(uint32_t taddr, double (&a)[9], double (&b)[9])
{
  uint32_t r[36];
  tmem_load18_issue(taddr, r);
  tmem_load_wait();
  tmem_unpack18(r, a, b);
}

// four doubles = 8 columns
__device__ __forceinline__ void tmem_store4(uint32_t taddr, double a, double b, double c, double d)
{
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(__double2loint(a)),
               "r"(__double2hiint(a)), "r"(__double2loint(b)), "r"(__double2hiint(b)), "r"(__double2loint(c)), "r"(__double2hiint(c)),
               "r"(__double2loint(d)), "r"(__double2hiint(d))
               : "memory");
}
__device__ __forceinline__ void tmem_load4_issue(uint32_t taddr, uint32_t (&r)[8])
{
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
// after tmem_load_wait()
__device__ __forceinline__ void tmem_unpack4(uint32_t (&r)[8], double& a, double& b, double& c, double& d)
{
#pragma unroll
  for (int k = 0; k < 8; k++) asm volatile("" : "+r"(r[k])::"memory");
  a = __hiloint2double((int)r[1], (int)r[0]);
  b = __hiloint2double((int)r[3], (int)r[2]);
  c = __hiloint2double((int)r[5], (int)r[4]);
  d = __hiloint2double((int)r[7], (int)r[6]);
}

#else  // ---- tests/cpu_emu: a copy lands when it is issued; a wait on a phase nobody completed is a kernel bug and aborts

inline void emu_async_fail(const char* what)
{
  std::fprintf(stderr, "cuda_emu: %s\n", what);
  std::abort();
}

struct EmuMbar
{
  int32_t tx;
  int16_t pending, phase;
};
static_assert(sizeof(EmuMbar) == sizeof(uint64_t), "the emulated barrier lives in the kernel's 8-byte slot");

inline void emu_mbar_settle(EmuMbar* b, unsigned count_reset)
{
  if (b->pending == 0 && b->tx == 0)
  {
    b->phase ^= 1;
    b->pending = (int16_t)count_reset;
  }
}
inline void mbar_init(uint64_t* bar, unsigned count)
{
  EmuMbar* b = (EmuMbar*)bar;
  b->tx = 0;
  b->pending = (int16_t)count;
  b->phase = 0;
}
inline void mbar_init_fence() {}
inline void mbar_arrive_expect_tx(uint64_t* bar, unsigned bytes)
{
  EmuMbar* b = (EmuMbar*)bar;
  b->tx += (int32_t)bytes;
  b->pending--;
  emu_mbar_settle(b, 1);
}
inline void bulk_copy_g2s(void* dst_smem, const void* src_gmem, unsigned bytes, uint64_t* bar)
{
  if (bytes % 16 || (uintptr_t)src_gmem % 16 || (uintptr_t)dst_smem % 16) emu_async_fail("bulk_copy_g2s: source, destination and size must be multiples of 16 bytes");
  std::memcpy(dst_smem, src_gmem, bytes);
  EmuMbar* b = (EmuMbar*)bar;
  b->tx -= (int32_t)bytes;
  emu_mbar_settle(b, 1);
}
inline void mbar_wait(uint64_t* bar, unsigned parity)
{
  const volatile EmuMbar* b = (const volatile EmuMbar*)bar;
  // phase p completed  <=>  the barrier's current phase bit differs from p.  Poll like the device does, handing the host
  // thread to the block's other fibers; a phase nobody ever completes is a kernel bug and aborts instead of spinning for ever
  for (long spins = 0; (unsigned)b->phase == (parity & 1u); spins++)
  {
    if (spins > (1L << 22)) emu_async_fail("mbar_wait: the awaited phase is never completed (no thread of the block issues the copy)");
    emu::spin_yield();
  }
}

// tensor memory: one 512-column lane per thread of the block (static thread_local like __shared__: one block at a time per host thread)
inline uint32_t (*emu_tmem())[512]
{
  static thread_local uint32_t lanes[128][512];
  return lanes;
}
template <int COLS>
inline uint32_t tmem_alloc(uint32_t*)
{
  __syncthreads();
  return 0u;
}
template <int COLS>
inline void tmem_free(uint32_t) { __syncthreads(); }
inline void tmem_store18(uint32_t taddr, const double (&a)[9], const double (&b)[9])
{
  if (taddr + 36u > 512u || threadIdx.x >= 128u) emu_async_fail("tmem_store18: outside the thread's 512 columns");
  uint32_t* c = emu_tmem()[threadIdx.x] + taddr;
  std::memcpy(c, a, 72);
  std::memcpy(c + 18, b, 72);
}
inline void tmem_store_wait() {}
inline void tmem_load18(uint32_t taddr, double (&a)[9], double (&b)[9])
{
  if (taddr + 36u > 512u || threadIdx.x >= 128u) emu_async_fail("tmem_load18: outside the thread's 512 columns");
  const uint32_t* c = emu_tmem()[threadIdx.x] + taddr;
  std::memcpy(a, c, 72);
  std::memcpy(b, c + 18, 72);
}

inline void tmem_load18_issue(uint32_t taddr, uint32_t (&r)[36])
{
  if (taddr + 36u > 512u || threadIdx.x >= 128u) emu_async_fail("tmem_load18_issue: outside the thread's 512 columns");
  std::memcpy(r, emu_tmem()[threadIdx.x] + taddr, 144);
}
inline void tmem_load_wait() {}
inline void tmem_unpack18(uint32_t (&r)[36], double (&a)[9], double (&b)[9])
{
  std::memcpy(a, r, 72);
  std::memcpy(b, r + 18, 72);
}
inline void tmem_store4(uint32_t taddr, double a, double b, double c, double d)
{
  if (taddr + 8u > 512u || threadIdx.x >= 128u) emu_async_fail("tmem_store4: outside the thread's 512 columns");
  const double v[4] = {a, b, c, d};
  std::memcpy(emu_tmem()[threadIdx.x] + taddr, v, 32);
}
inline void tmem_load4_issue(uint32_t taddr, uint32_t (&r)[8])
{
  if (taddr + 8u > 512u || threadIdx.x >= 128u) emu_async_fail("tmem_load4_issue: outside the thread's 512 columns");
  std::memcpy(r, emu_tmem()[threadIdx.x] + taddr, 32);
}
inline void tmem_unpack4(uint32_t (&r)[8], double& a, double& b, double& c, double& d)
{
  double v[4];
  std::memcpy(v, r, 32);
  a = v[0]; b = v[1]; c = v[2]; d = v[3];
}

#endif

}  // namespace lbm
