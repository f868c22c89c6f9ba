// Gram kernel for the streaming regime (64 <= N_pad <= 112 clients, large D): the kernel that serves
// Krum at "N = 100, D = 11.2 M" (reference: defences.py:16-21).
//
// Why a second kernel: a tcgen05.mma microbenchmark (tools/mma_bench.cu) gives t = 43 + N/2 cycles for
// M = 128, for BOTH kind::tf32 (K = 8) and kind::f16 (K = 16).  At N = 2*112 the split-TF32 kernel of
// gram.cu needs >= 620 tensor cycles per 32 columns, more than the ~550 cycles HBM needs for them, while
// bf16 operands need 310.  Here:
//
//   * TMA (cp.async.bulk.tensor.2d, no swizzle, zero OOB fill) streams one k-block {64 fp32 columns x N_pad
//     rows} per instruction into a 7-slot ring (slot = k-block % 7; rows N..N_pad-1 are zero fill).
//     tools/tma_bench.cu measured a fixed ~450 ns per 2-D box per SM whatever its size, so 128-byte-wide
//     boxes cap at 3.8 TB/s chip-wide while 256-byte-wide boxes reach the HBM bound;
//   * 4 converter warps (warp w takes k-blocks w, w+4, ...) rewrite the slot IN PLACE
//     (bf16x2_convert_units, shared with gram_pair.cu): every 8-row unit u (2 KB of fp32) becomes one
//     SWIZZLE_128B core-matrix atom of b1 at slot + 2048 u followed by one of b2 at slot + 2048 u + 1024,
//     g - c = b1 + b2 + r (both roundings to nearest, |r| <= 2^-17 |g - c|), c = the mean of the last 8
//     clients' rows of the same k-block, read from the slot before its first store.  Without a second
//     staging buffer the ring holds 7 k-blocks in flight instead of 4: a slot lives for TMA latency +
//     conversion + MMA, and the ring depth, not HBM, paced the 4-slot version (Little's law);
//   * S ~= b1 b1^T + b1 b2^T + (b1 b2^T)^T: ONE tcgen05.mma.kind::f16 (K = 16) per 16 columns.  A = b1
//     (M = 128, 8-row groups 2048 bytes apart from the slot base; rows >= N_pad reach past the slot and
//     land in result rows nobody reads) and B = the whole slot with 8-row groups 1024 bytes apart, i.e.
//     N = 2*N_pad rows b1 unit 0, b2 unit 0, b1 unit 1, ...: result column 16 u + r holds b1 b1^T of client
//     8 u + r, column 16 u + 8 + r holds b1 b2^T.  Dropped terms (b2 b2^T, r) are ~2^-17 relative per
//     product; b2 b2^T is positive on every squared distance and shows up as a uniform ~-1.3e-6 scale of d2;
//   * the MMA commit of a k-block returns its slot to the TMA producer.  Two MMA issuer warps alternate
//     k-blocks strictly (named barriers 8 and 9), so every CTA accumulates in k-block order; TMEM
//     accumulators are double-buffered and drained every `flush` k-blocks by 8 epilogue warps into fp32
//     registers, K is interleaved over the CTAs into private partial slots that gram_reduce_kernel sums in a
//     fixed order in float64 (bit-reproducible; identical rows give exact zeros and identical table rows).
//
// Warp roles (512 threads): warp 0 TMA producer, warps 1,3 MMA issue, warp 2 TMEM alloc, warps 4-7
// converters, warps 8-15 epilogue (warp group a drains the 8-column groups 2u + a).
#include "afl_common.cuh"

namespace afl {
namespace gram {

constexpr int kB16Threads = 512;
constexpr int kB16Slots = 7;         // ring slots, one k-block [N_pad x 64 fp32] each (slot = k-block % 7)
constexpr int kB16Cols = 64;         // fp32 columns per k-block = 128 bytes of bf16 per row
constexpr int kB16ASpan = 16 * 2048; // bytes the A operand (128 rows, 2 KB per 8-row group) spans from its slot base
constexpr int kB16PartElems = 2 * 128 * 128;

struct B16Params {
  int n, nb;            // clients, padded to a multiple of 16 (64..112)
  int splits;           // CTAs; CTA c owns k-blocks c, c+splits, ...
  int kblocks;          // ceil(d / 64)
  int flush;            // k-blocks per TMEM accumulation chain (even)
  float* parts;         // [splits][2][128][128]
  int center;           // subtract the mean of the last clients' rows while converting (translation invariance)
};

__global__ void __launch_bounds__(kB16Threads, 1)
gram_bf16x2_kernel(const __grid_constant__ CUtensorMap tmap, const B16Params p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t raw_full[kB16Slots], slot_free[kB16Slots], acc_full[2], acc_empty[2], first_issued[2];
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wg = warp >> 2;
  const int split = blockIdx.x;
  const int nkb = (p.kblocks - split + p.splits - 1) / p.splits;      // k-blocks split, split+splits, ...
  const int ngroups = (nkb + p.flush - 1) / p.flush;
  const uint32_t slot_bytes = static_cast<uint32_t>(p.nb) * 256u;     // one fp32 k-block [nb x 64], row-major
  const uint32_t ring = smem_u32(smem);

  if (threadIdx.x == 0) {
    for (int s = 0; s < kB16Slots; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&slot_free[s], 1); }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 2);
      mbar_init(&acc_empty[b], 8);
      mbar_init(&first_issued[b], 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(&tmem_base_smem, 512);
    tmem_relinquish();
  }
  if (warp == 0 && lane == 0) tma_prefetch_desc(&tmap);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // tmem_base_smem is read where it is used: kept live through the converters' 112 registers it would spill

  if (wg == 0) {
    setmaxnreg_dec<64>();
    if (warp == 0) {
      // ===================== TMA producer: one box [nb x 64 fp32] per k-block =====================
      if (lane == 0) {
        const uint64_t pol = policy_evict_first();
        int s = 0;
        uint32_t ph = 0;
        for (int i = 0; i < nkb; ++i) {
          mbar_wait(&slot_free[s], ph ^ 1);
          mbar_arrive_expect_tx(&raw_full[s], slot_bytes);
          tma_load_2d(smem + static_cast<size_t>(s) * slot_bytes, &tmap, &raw_full[s], (split + i * p.splits) * kB16Cols, 0, pol);
          if (++s == kB16Slots) { s = 0; ph ^= 1; }
        }
      }
    } else if (warp == 1 || warp == 3) {
      // ===================== MMA issuers (alternating k-blocks) =====================
      const int j = (warp == 3) ? 1 : 0;
      const uint32_t idesc = umma_idesc_bf16(128, 2 * p.nb);
      const uint32_t tmem_base = tmem_base_smem;
      for (int g = 0; g < ngroups; ++g) {
        const int b = g & 1;
        const uint32_t gph = (g >> 1) & 1;
        const int it_begin = g * p.flush, it_end = min(it_begin + p.flush, nkb);
        const uint32_t d_acc = tmem_base + static_cast<uint32_t>(b * 256);
        int it = it_begin + j;
        // issuer 1 waits for issuer 0's first MMA of the group even when it has no k-block in it (odd tail): its
        // acc_full commit must not land in the barrier's previous phase
        if (j == 0) mbar_wait_fast(&acc_empty[b], gph ^ 1);
        else mbar_wait_fast(&first_issued[b], gph);
        tc_fence_after();
        for (; it < it_end; it += 2) {
          const int s = it % kB16Slots;
          named_bar_sync(1 + s, 32 + 32);                // the converter warp of k-block `it` has written and fenced slot s
          // Strict alternation: k-block `it` is issued only after k-block it-1 has been, so the accumulation order is
          // the k-block order (reproducible run to run).  Barrier 8: issuer 0 -> 1, barrier 9: issuer 1 -> 0.
          if (it > 0) named_bar_sync(j == 0 ? 9u : 8u, 32 + 32);
          tc_fence_after();
          const uint32_t slot = ring + static_cast<uint32_t>(s) * slot_bytes;
          const uint64_t da = umma_desc_sw128_sbo(slot, 2048u);   // A = b1 atoms: rows 0..127
          const uint64_t db = umma_desc_sw128_sbo(slot, 1024u);   // B = b1, b2 atoms alternating: rows 0..2nb-1
          if (elect_one()) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)               // 4 x K=16 bf16 = 64 columns; +32 bytes per step
              umma_bf16(d_acc, da + static_cast<uint64_t>(ks * 2), db + static_cast<uint64_t>(ks * 2), idesc,
                        (it != it_begin) || (ks != 0));
            umma_commit(&slot_free[s]);
            if (it == it_begin) mbar_arrive(&first_issued[b]);
          }
          __syncwarp();
          if (it + 1 < nkb) named_bar_arrive(j == 0 ? 8u : 9u, 32 + 32);
        }
        if (elect_one()) umma_commit(&acc_full[b]);
        __syncwarp();
      }
    }
  } else if (wg == 1) {
    setmaxnreg_dec<112>();
    // ===================== converters: fp32 k-block -> b1 / b2 atoms, in place =====================
    const int w4 = warp - 4;
    uint32_t src_lane, dst_off[4];
    bf16x2_lane_offsets(src_lane, dst_off);
    const int units = p.nb >> 3;
    // centre = mean of the last 8 clients over this lane's 4 columns; their rows are part of the k-block that TMA
    // just delivered, so they are read from shared memory (8 broadcast LDS.128 per k-block) - no extra L2 traffic
    const int crow0 = p.n >= kGramCenterRows ? p.n - kGramCenterRows : 0;
    const uint32_t cen_off = static_cast<uint32_t>(lane & 15) * 16u;
    for (int kb = w4; kb < nkb; kb += 4) {
      const int s = kb % kB16Slots;
      const uint32_t ph = static_cast<uint32_t>(kb / kB16Slots) & 1u;
      // k-block kb - 7 (another converter's) may still be in flight: the copies of two TMA boxes complete in no
      // defined order, and while raw_full[s] is still in kb - 7's phase a wait for kb's parity would see the phase
      // before it as complete.  kb - 7's MMA commit (the producer's own wait before loading kb) closes that window.
      if (kb >= kB16Slots) mbar_wait_fast(&slot_free[s], ph ^ 1u);
      mbar_wait_fast(&raw_full[s], ph);
      const uint32_t slot = ring + static_cast<uint32_t>(s) * slot_bytes;
      float4 cen = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p.center) {                                     // before the first store: the last rows are overwritten last
        float4 t[kGramCenterRows];
#pragma unroll
        for (int r = 0; r < kGramCenterRows; ++r) {
          const int row = crow0 + r < p.n ? crow0 + r : p.n - 1;
          t[r] = lds128(slot + static_cast<uint32_t>(row) * 256u + cen_off);
        }
#pragma unroll
        for (int r = 0; r < kGramCenterRows; ++r) { cen.x += t[r].x; cen.y += t[r].y; cen.z += t[r].z; cen.w += t[r].w; }
        cen.x *= 0.125f; cen.y *= 0.125f; cen.z *= 0.125f; cen.w *= 0.125f;
      }
      bf16x2_convert_units(slot, units, src_lane, dst_off, cen);
      fence_proxy_async_smem();
      named_bar_arrive(1 + s, 32 + 32);
    }
  } else {
    setmaxnreg_inc<168>();
    // ===================== epilogue: drain TMEM chains into fp32 registers =====================
    const int q = warp & 3;             // TMEM lane quadrant this warp may access
    const int a = (warp - 8) >> 2;      // 0: b1*b1^T (8-column groups 2u), 1: b1*b2^T (groups 2u + 1)
    const uint32_t tmem_base = tmem_base_smem;
    float run[112];
#pragma unroll
    for (int i = 0; i < 112; ++i) run[i] = 0.f;
    for (int g = 0; g < ngroups; ++g) {
      const int b = g & 1;
      mbar_wait_fast(&acc_full[b], (g >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(b * 256 + a * 8);
#pragma unroll
      for (int u = 0; u < 14; u += 2) {                   // clients 8u .. 8u + 15 (nb is a multiple of 16)
        if (u * 8 < p.nb) {
          uint32_t v0[8], v1[8];
          tmem_ld_32x32b_x8(taddr + u * 16, v0);
          tmem_ld_32x32b_x8(taddr + u * 16 + 16, v1);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            run[u * 8 + i] += __uint_as_float(v0[i]);
            run[u * 8 + 8 + i] += __uint_as_float(v1[i]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[b]);
    }
    float* out = p.parts + static_cast<size_t>(split) * kB16PartElems + static_cast<size_t>(a) * 128 * 128 +
                 static_cast<size_t>(q * 32 + lane) * 128;
#pragma unroll
    for (int c = 0; c < 112; c += 4)
      if (c < p.nb) *reinterpret_cast<float4*>(out + c) = make_float4(run[c], run[c + 1], run[c + 2], run[c + 3]);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base_smem, 512);
  }
}

bool bf16x2_eligible(int n, int64_t d) {
  const int nb = (n + 15) & ~15;
  return nb >= 64 && nb <= 112 && d >= 32768;
}

int bf16x2_splits(int64_t d) {
  const int64_t kblocks = (d + kB16Cols - 1) / kB16Cols;
  int s = sm_count();
  if (const char* e = getenv("AFL_GRAM_SPLITS")) if (atoi(e) > 0) s = atoi(e);
  if (s > kblocks) s = static_cast<int>(kblocks);
  return s < 1 ? 1 : s;
}

typedef CUresult (*EncodeTiledFn2)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// parts must hold bf16x2_splits(d) * 2*128*128 floats (gram_reduce_kernel only reads rows/columns < n).
int launch_bf16x2(const float* G, int n, int64_t d, int64_t ld, float* parts, int splits, int flush, int center,
                  cudaStream_t stream) {
  static EncodeTiledFn2 enc = nullptr;
  if (!enc) {
    void* fp = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess) { set_error("cuTensorMapEncodeTiled entry point not found"); return AFL_ERR_CUDA; }
    enc = reinterpret_cast<EncodeTiledFn2>(fp);
  }
  B16Params p{};
  p.n = n; p.nb = (n + 15) & ~15;
  p.kblocks = static_cast<int>((d + kB16Cols - 1) / kB16Cols);
  p.flush = flush < 2 ? 2 : (flush & ~1);
  p.splits = splits;
  p.parts = parts;
  p.center = center ? 1 : 0;
  CUtensorMap tmap;
  const cuuint64_t gdim[2] = {static_cast<cuuint64_t>(d), static_cast<cuuint64_t>(n)};
  const cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * sizeof(float)};
  const cuuint32_t box[2] = {kB16Cols, static_cast<cuuint32_t>(p.nb)};   // rows n..nb-1: zero fill
  const cuuint32_t estride[2] = {1, 1};
  CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(G), gdim, gstride, box, estride,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed: %d", static_cast<int>(r)); return AFL_ERR_CUDA; }
  // the last slot's A operand reads kB16ASpan bytes from its base: keep that inside the allocation (+1 KB alignment)
  const size_t slot_bytes = static_cast<size_t>(p.nb) * 256;
  const size_t smem = (kB16Slots - 1) * slot_bytes + kB16ASpan + 1024;
  static int smem_attr_done[kMaxDevices] = {0};
  AFL_CUDA(ensure_dyn_smem(gram_bf16x2_kernel, 226 * 1024, smem_attr_done));
  {
    ProfScope ps("gram_bf16x2", stream);
    gram_bf16x2_kernel<<<splits, kB16Threads, smem, stream>>>(tmap, p);
  }
  AFL_LAUNCH_CHECK("gram_bf16x2_kernel");
  return AFL_OK;
}

}  // namespace gram
}  // namespace afl
