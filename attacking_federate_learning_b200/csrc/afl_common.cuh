// Shared device/host helpers for the sm_100a kernels: error plumbing, PTX wrappers for mbarrier,
// TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM alloc / ld / commit) and small warp utilities.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/afl_b200.h"

#ifndef AFL_BAR_TIMEOUT_LOG2
#define AFL_BAR_TIMEOUT_LOG2 32
#endif

namespace afl {

// ------------------------------------------------------------------------------------------------
// host-side error plumbing
// ------------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);
void count_launch(int n = 1);

#define AFL_CUDA(call)                                                        \
  do {                                                                        \
    cudaError_t _e = (call);                                                  \
    if (_e != cudaSuccess) return ::afl::cuda_fail(_e, #call, __FILE__, __LINE__); \
  } while (0)

#define AFL_LAUNCH_CHECK(name)                                                \
  do {                                                                        \
    ::afl::count_launch();                                                    \
    cudaError_t _e = cudaGetLastError();                                      \
    if (_e != cudaSuccess) return ::afl::cuda_fail(_e, name, __FILE__, __LINE__); \
  } while (0)

constexpr int kMaxDevices = 64;
int current_device();      // ordinal of the current device (0 when no device is visible)
int sm_count();            // SM count of the CURRENT device

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device: remember it per (kernel, device).
template <typename K>
static inline cudaError_t ensure_dyn_smem(K kernel, int bytes, int (&done)[kMaxDevices]) {
  const int dev = current_device();
  if (done[dev] >= bytes) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) done[dev] = bytes;
  return e;
}

// Optional tail of gram_to_sqdist_kernel (csrc/xgpu.cu): the LAST block to finish also publishes this rank's epoch
// flag to every peer, which saves a launch per multi-GPU Krum step.
constexpr int kMaxWorld = 16;
struct PubHook {
  unsigned long long* flag[kMaxWorld];   // flags block of every rank (peer-mapped)
  int world, rank;
  unsigned long long epoch;
  unsigned int* counter;                 // zero-initialised, reset by the last block
};

// Optional CUDA-event bracket around a kernel launch (active only after afl_profile_enable(1)).
struct ProfScope {
  ProfScope(const char* name, cudaStream_t stream);
  ~ProfScope();
  const char* name_; cudaStream_t stream_; void* rec_;
};

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

#ifdef __CUDACC__
// ------------------------------------------------------------------------------------------------
// small device utilities
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Streaming (read-once) global loads: bypass L1 allocation.
__device__ __forceinline__ float4 ldg_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ float bf16_bits_to_f32(uint32_t b16) { return __uint_as_float(b16 << 16); }

// ------------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must trap (launch error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > (1ll << AFL_BAR_TIMEOUT_LOG2)) {  // ~2 s by default: no legitimate wait is longer than one pipeline step
      printf("afl: mbarrier timeout block %d thread %d bar %u parity %u\n", (int)blockIdx.x, (int)threadIdx.x,
             smem_u32(bar), parity);
      __trap();
    }
  }
}

// Warp-level wait: one lane spins, the others sleep at the warp barrier and then observe the (already
// completed) phase with a single probe each, which gives every lane its own acquire.
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity) {
  if ((threadIdx.x & 31) == 0) mbar_wait(bar, parity);
  __syncwarp();
  mbar_wait(bar, parity);          // completes on the first probe; bounded like every other wait
}

// Explicit shared-space 16-byte accesses (a hand-aligned pointer into dynamic shared memory loses its
// address space and would otherwise compile to slow generic LD.E / ST.E).
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const float4& v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// Named barriers (ids 1..15; 0 is __syncthreads): producers bar.arrive, the consumer warp bar.sync.
// (aligned barriers: the whole warp must execute them convergently, hence the __syncwarp)
__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t nthreads) {
  __syncwarp();
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  __syncwarp();
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Fast-path wait: one probe by every lane (an already-completed phase costs a single try_wait); only if
// the phase is still pending does lane 0 spin while the others sleep at the warp barrier.
__device__ __forceinline__ void mbar_wait_fast(uint64_t* bar, uint32_t parity) {
  if (__all_sync(0xffffffffu, mbar_try_wait(bar, parity))) return;
  mbar_wait_warp(bar, parity);
}

// generic-proxy writes (st.shared) -> visible to the async proxy (TMA / tcgen05 operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------
// TMA
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tiled load, completes `bytes` on the mbarrier.  c0 = innermost (column) coord, c1 = row coord.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0,
                                            int c1, uint64_t cache_policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1),
        "l"(cache_policy)
      : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t policy_evict_normal() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}

// 16-byte asynchronous global->shared copy (LDGSTS), zero-filling bytes past src_bytes, and an
// mbarrier arrival that fires when all of this thread's earlier cp.async have landed.
__device__ __forceinline__ void cp_async_16(uint32_t smem_addr, const void* gptr, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_addr), "l"(gptr), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]^T, TF32 inputs, fp32 accumulate, issued by ONE thread.
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 16 consecutive fp32 columns -> 16 registers per thread (thread t <-> TMEM lane base+t).
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor: K-major operand, 128-byte swizzle, rows of exactly 128 bytes,
// 8-row groups 1024 bytes apart (layout written by a TMA box {32 fp32, rows} with SWIZZLE_128B).
// Fields (cute::UMMA::SmemDescriptor): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) |
// version=1 [46,48) | layout_type=2 (SWIZZLE_128B) [61,64).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;             // LBO (ignored for swizzled K-major), canonical 1
  d |= static_cast<uint64_t>(1024 >> 4) << 32;     // SBO = 1024 B between 8-row core-matrix groups
  d |= static_cast<uint64_t>(1) << 46;             // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;             // SWIZZLE_128B
  return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 (1) [4,6) | a_format TF32 (2)
// [7,10) | b_format TF32 (2) [10,13) | a/b K-major (0) | n>>3 [17,23) | m>>4 [24,29).
__host__ __device__ __forceinline__ uint32_t umma_idesc_tf32(uint32_t m, uint32_t n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}
// c_format F32 (1) [4,6) | a_format BF16 (1) [7,10) | b_format BF16 (1) [10,13) | K-major | n>>3 | m>>4
__host__ __device__ __forceinline__ uint32_t umma_idesc_bf16(uint32_t m, uint32_t n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}
// K-major, SWIZZLE_128B, 128-byte rows, 8-row groups `sbo` bytes apart.
__device__ __forceinline__ uint64_t umma_desc_sw128_sbo(uint32_t smem_addr, uint32_t sbo) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(sbo >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T, BF16 inputs, fp32 accumulate, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 8 consecutive fp32 columns -> 8 registers per thread.
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr) : "memory");
}

// ------------------------------------------------------------------------------------------------
// bf16x2 operands, converted in place (gram_bf16.cu, gram_pair.cu)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16x2_rn(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ void sts64(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.b32 [%0], {%1,%2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}
// Per-lane constants of bf16x2_convert_units: a half warp owns one 256-byte fp32 row (16 lanes x 16 bytes), the warp
// reads 2 rows per LDS.128 and an 8-row unit (2 KB) with 4 of them.  The lane with fp32 chunk c16 owns bf16 bytes
// [8 c16, 8 c16 + 8) of the 128-byte bf16 row, i.e. half of 16-byte chunk c16/2, which SWIZZLE_128B places at chunk
// (c16/2) ^ (row & 7).  dst_off[u]: destination of row 2u + rsub inside the unit's atom.
__device__ __forceinline__ void bf16x2_lane_offsets(uint32_t& src_lane, uint32_t (&dst_off)[4]) {
  const int rsub = lane_id() >> 4, c16 = lane_id() & 15;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const uint32_t row8 = static_cast<uint32_t>(2 * u + rsub);
    dst_off[u] = row8 * 128u + ((static_cast<uint32_t>(c16 >> 1) ^ row8) << 4) + (static_cast<uint32_t>(c16 & 1) << 3);
  }
  src_lane = static_cast<uint32_t>(rsub) * 256u + static_cast<uint32_t>(c16) * 16u;
}
// Rewrites `units` 8-row units of fp32 (2 KB each, 256-byte rows of 64 columns, from `base`) IN PLACE: unit u
// becomes one SWIZZLE_128B core-matrix atom of b1 at base + 2048 u followed by one of b2 at base + 2048 u + 1024,
// with g - c = b1 + b2 + r, |r| <= 2^-17 |g - c| (both roundings to nearest); c = this lane's 4 columns of the
// centre.  A unit's output only overwrites that unit's own input, which the warp has already loaded.
__device__ __forceinline__ void bf16x2_convert_units(uint32_t base, int units, uint32_t src_lane,
                                                     const uint32_t (&dst_off)[4], float4 cen) {
  float4 v[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) v[u] = lds128(base + src_lane + static_cast<uint32_t>(u) * 512u);
#pragma unroll 1
  for (int unit = 0; unit < units; ++unit) {
    uint32_t h[4][2], l[4][2];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float x0 = v[u].x - cen.x, x1 = v[u].y - cen.y, x2 = v[u].z - cen.z, x3 = v[u].w - cen.w;
      h[u][0] = pack_bf16x2_rn(x0, x1);
      h[u][1] = pack_bf16x2_rn(x2, x3);
      l[u][0] = pack_bf16x2_rn(x0 - __uint_as_float(h[u][0] << 16), x1 - __uint_as_float(h[u][0] & 0xFFFF0000u));
      l[u][1] = pack_bf16x2_rn(x2 - __uint_as_float(h[u][1] << 16), x3 - __uint_as_float(h[u][1] & 0xFFFF0000u));
    }
    const uint32_t ub = base + static_cast<uint32_t>(unit) * 2048u;
    if (unit + 1 < units) {                               // next unit's loads before this unit's stores
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = lds128(ub + 2048u + src_lane + static_cast<uint32_t>(u) * 512u);
    }
    __syncwarp();                                         // every lane has read this unit before anyone overwrites it
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      sts64(ub + dst_off[u], h[u][0], h[u][1]);
      sts64(ub + 1024u + dst_off[u], l[u][0], l[u][1]);
    }
  }
}

// Centre of the bf16x2 Gram kernels: mean of the LAST `rows` clients (cref = first of those rows, pitch ld) over
// this lane's 4 consecutive columns starting at `col`.  Distances are translation invariant, so any centre is
// correct; a centre close to the clients' common component keeps ||g - c||^2 (which the dropped-term and
// accumulation biases scale with) of the order of the distances themselves.  Ids >= f are honest (main.py:28).
constexpr int kGramCenterRows = 8;
__device__ __forceinline__ float4 gram_center(const float* cref, int rows, int64_t ld, int64_t col, int64_t d) {
  // always kGramCenterRows loads, all issued before the first add (a runtime trip count would serialise 8 dependent
  // L2 round trips per k-block); with fewer clients the last row is simply counted more than once - any centre is valid
  float4 t[kGramCenterRows];
  if (col + 3 < d) {
#pragma unroll
    for (int r = 0; r < kGramCenterRows; ++r)
      t[r] = __ldg(reinterpret_cast<const float4*>(cref + static_cast<int64_t>(r < rows ? r : rows - 1) * ld + col));
  } else {
#pragma unroll
    for (int r = 0; r < kGramCenterRows; ++r) {
      const float* q = cref + static_cast<int64_t>(r < rows ? r : rows - 1) * ld + col;
      t[r] = make_float4(col < d ? __ldg(q) : 0.f, col + 1 < d ? __ldg(q + 1) : 0.f, col + 2 < d ? __ldg(q + 2) : 0.f, 0.f);
    }
  }
  float cx = 0.f, cy = 0.f, cz = 0.f, cw = 0.f;
#pragma unroll
  for (int r = 0; r < kGramCenterRows; ++r) { cx += t[r].x; cy += t[r].y; cz += t[r].z; cw += t[r].w; }
  const float inv = 1.0f / static_cast<float>(kGramCenterRows);
  return make_float4(cx * inv, cy * inv, cz * inv, cw * inv);
}


template <int kRegs>
__device__ __forceinline__ void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegs));
}
template <int kRegs>
__device__ __forceinline__ void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegs));
}
#endif  // __CUDACC__

}  // namespace afl
