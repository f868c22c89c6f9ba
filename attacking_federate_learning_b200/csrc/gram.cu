// Pairwise squared distances of the N client rows (reference: defences.py:16-21
// `_krum_create_distances`, the dominant cost of Krum and Bulyan).
//
// tcgen05 path (fp32 input, 16-byte aligned rows):
//   d2_ij = s_ii + s_jj - 2 s_ij with S = G G^T computed on the 5th-gen tensor cores.
//   * Operand tiles [128 rows x 32 fp32] are fetched by TMA (SWIZZLE_128B, rows past N zero-filled)
//     into a multi-stage shared-memory ring.
//   * fp32 is split as g = hi + lo, hi = the TF32 the tensor core sees (top 10 mantissa bits), lo =
//     RN_tf32(g - hi).  S ~= hi hi^T + hi lo^T + (hi lo^T)^T: two MMAs per k-step instead of three
//     (the third product is the transpose of the second and is added in the reduce kernel).  The
//     dropped lo*lo^T term is <= 2^-20 relative.  The "split" warps compute lo from the TMA tile with
//     CUDA cores and store it in the same swizzled layout (same byte offsets), so it needs no address
//     math and feeds tcgen05.mma directly.
//   * One elected thread issues tcgen05.mma.kind::tf32 (M=128, N=16..128, K=8); accumulators live in
//     TMEM, double-buffered: every `flush` k-blocks the accumulator is drained by the epilogue warps
//     (tcgen05.ld) into fp32 registers (round-to-nearest adds) while the MMA continues on the other
//     buffer.  This bounds the length of the tensor core's internal accumulation chain.
//   * K (the parameter dimension) is split over CTAs; every CTA writes its partial tile to its own
//     workspace slot and `reduce` sums the slots in a fixed order in float64 -> bit-reproducible and
//     identical rows give bit-identical table rows (Krum's [1,0,2,...] tie-break relies on this).
//
// SIMT path (any pitch, fp32 or bf16): direct sum of squared fp32 differences, float64 accumulation.
// Used for misaligned pitches and as an independent check of the tensor path in the tests.
#include "afl_common.cuh"

namespace afl {
namespace gram {

constexpr int kBK = 32;                      // fp32 columns per k-block = 128 B = one swizzle row
constexpr int kTileRows = 128;               // UMMA M, and the largest UMMA N used
constexpr int kTileBytes = kTileRows * 128;  // 16 KB
constexpr int kThreads = 512;                // 4 warpgroups
constexpr int kTmemCols = 512;
#ifndef AFL_SPLIT_RN
#define AFL_SPLIT_RN 0
#endif

constexpr int kPartElems = 2 * kTileRows * kTileRows;  // per (pair, split): [2][128][128] fp32

struct Params {
  int n;
  int tiles;          // T = ceil(n / 128); pairs = T*T
  int splits;         // K-splits
  int kblocks;        // ceil(d / 32)
  int flush;          // k-blocks per TMEM accumulation chain
  int stages;
  int stage_bytes;    // 32 KB (T == 1: [A][LO]) or 48 KB ([A][B][LO])
  int single_pass;
  int dbg;            // measurement only: 1 = split work but narrow (hi*hi) MMA, 2 = no split work but wide MMA
  int rewrite_hi;
  float* parts;       // [pairs][splits][2][128][128]
  int box_rows;       // rows per TMA box (<= 128; rows past it are never written and only feed ignored outputs)
  int kchunk_log2;    // k-blocks per contiguous K chunk owned by one split (1 << kchunk_log2)
  int loader;         // 0: TMA boxes, 1: cp.async (LDGSTS) rows written in the same swizzled layout
  const float* G;     // matrix base and pitch (elements) for the cp.async loader
  int64_t ld, d;
  long long* trace;   // debug: [2 CTAs][kTraceLen][kTraceEv] clock64 timestamps, or null
};
constexpr int kTraceLen = 512;
constexpr int kTraceEv = 16;

__device__ __forceinline__ float tf32_trunc(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }
// round-to-nearest (ties away) to TF32 precision = cvt.rna.tf32.f32, done on the integer pipe
__device__ __forceinline__ float tf32_rna(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}

__device__ __forceinline__ void trace_ev(const Params& p, int it, int ev) {
  if (p.trace && it < kTraceLen && (blockIdx.x == 0 || blockIdx.x == 77))
    p.trace[((blockIdx.x == 0 ? 0 : 1) * kTraceLen + it) * kTraceEv + ev] = clock64();
}

__global__ void __launch_bounds__(kThreads, 1)
gram_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap, const Params p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-byte alignment is required by SWIZZLE_128B; the dynamic smem base is only 16 B aligned by
  // contract, so align by hand (the host adds 1 KB of slack).
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  __shared__ __align__(8) uint64_t full_bar[16], empty_bar[16], acc_full[2], acc_empty[2], first_issued[2];
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int wg = warp >> 2;

  const int pairs = p.tiles * p.tiles;
  const int pair = blockIdx.x % pairs;
  const int split = blockIdx.x / pairs;
  const int ti = pair / p.tiles, tj = pair % p.tiles;
  const bool has_b = (ti != tj);
  const int rows_j = min(kTileRows, p.n - tj * kTileRows);
  const int nb = (rows_j + 15) & ~15;  // UMMA N
  // K assignment: k-blocks are grouped in chunks of kChunk (512 contiguous bytes per row); split s owns
  // chunks s, s+splits, s+2*splits, ...  At any moment the CTAs of one tile pair therefore read a
  // contiguous band of every row (DRAM pages are consumed whole) instead of 128-byte pieces that are
  // megabytes apart.
  const int kChunk = 1 << p.kchunk_log2;
  const int nchunks_total = (p.kblocks + kChunk - 1) >> p.kchunk_log2;
  const int my_chunks = split < nchunks_total ? (nchunks_total - split + p.splits - 1) / p.splits : 0;
  int nkb = my_chunks * kChunk;
  if (my_chunks > 0 && split + (my_chunks - 1) * p.splits == nchunks_total - 1)
    nkb -= nchunks_total * kChunk - p.kblocks;          // the globally last chunk may be short
  const int ngroups = (nkb + p.flush - 1) / p.flush;
  const uint32_t off_b = kTileBytes;
  // lo tile sits directly behind the nb valid rows of the B-side tile, so that raw||lo is ONE K-major
  // operand of 2*nb rows (rows nb..127 of that tile are TMA zero fill and may be overwritten)
  const uint32_t off_lo = (has_b ? off_b : 0u) + static_cast<uint32_t>(nb) * 128u;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], p.loader ? 32 : 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 2);        // one tcgen05.commit from each of the two MMA issuer warps
      mbar_init(&acc_empty[b], 8);
      mbar_init(&first_issued[b], 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(&tmem_base_smem, kTmemCols);
    tmem_relinquish();
  }
  if (warp == 0 && lane == 0) tma_prefetch_desc(&tmap);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  if (wg == 0) {
    setmaxnreg_dec<64>();
    if (p.loader == 1 && (warp == 0 || warp == 2)) {
      // ===================== cp.async producers: two warps, alternating stages =====================
      // Lane l copies 16-byte chunk (l & 7) of row 4*i + (l >> 3); the destination is the position a TMA
      // box with SWIZZLE_128B would have used: row*128 + ((chunk ^ (row & 7)) << 4).
      const int j = (warp == 2) ? 1 : 0;
      const int rows_i = min(kTileRows, p.n - ti * kTileRows);
      const int sub = lane >> 3, c16 = lane & 7;
      int s = j;
      uint32_t ph = 0;
      for (int it = j; it < nkb; it += 2) {
        mbar_wait_warp(&empty_bar[s], ph ^ 1);
        if (lane == 0) trace_ev(p, it, 1);
        const int col = ((split + (it >> p.kchunk_log2) * p.splits) * kChunk + (it & (kChunk - 1))) * kBK + c16 * 4;
        const int64_t remain = p.d - col;
        const uint32_t nbytes = remain >= 4 ? 16u : (remain > 0 ? static_cast<uint32_t>(remain) * 4u : 0u);
        const uint32_t st = smem_u32(smem) + static_cast<uint32_t>(s) * static_cast<uint32_t>(p.stage_bytes);
        const float* gcol = p.G + (remain > 0 ? col : 0);
#pragma unroll 5
        for (int r = sub; r < rows_i; r += 4)
          cp_async_16(st + r * 128 + ((c16 ^ (r & 7)) << 4), gcol + static_cast<int64_t>(ti * kTileRows + r) * p.ld, nbytes);
        if (has_b) {
#pragma unroll 5
          for (int r = sub; r < rows_j; r += 4)
            cp_async_16(st + off_b + r * 128 + ((c16 ^ (r & 7)) << 4),
                        gcol + static_cast<int64_t>(tj * kTileRows + r) * p.ld, nbytes);
        }
        cp_async_mbar_arrive_noinc(&full_bar[s]);
        s += 2;
        if (s >= p.stages) { s -= p.stages; ph ^= 1; }
      }
    } else if (warp == 0) {
      // ===================== TMA producer =====================
      if (p.loader == 1) {
      } else
      if (lane == 0) {
        const uint64_t pol = (p.tiles == 1) ? policy_evict_first() : policy_evict_normal();
        int s = 0;
        uint32_t ph = 0;
        int chunk_col = split * kChunk * kBK, in_chunk = 0;
        for (int it = 0; it < nkb; ++it) {
          trace_ev(p, it, 0);
          mbar_wait(&empty_bar[s], ph ^ 1);
          trace_ev(p, it, 1);
          uint8_t* st = smem + static_cast<size_t>(s) * p.stage_bytes;
          mbar_arrive_expect_tx(&full_bar[s], static_cast<uint32_t>(p.box_rows) * 128u * (has_b ? 2u : 1u));
          const int col = chunk_col + in_chunk * kBK;
          tma_load_2d(st, &tmap, &full_bar[s], col, ti * kTileRows, pol);
          if (has_b) tma_load_2d(st + off_b, &tmap, &full_bar[s], col, tj * kTileRows, pol);
          if (++in_chunk == kChunk) { in_chunk = 0; chunk_col += p.splits * kChunk * kBK; }
          if (++s == p.stages) { s = 0; ph ^= 1; }
        }
      }
    } else if (warp == 1 || warp == 3) {
      // ===================== MMA issuers: two warps, alternating k-blocks =====================
      // An issuing thread is blocked while its UTCHMMAs drain into the tensor queue (~one k-block of
      // tensor time) and then needs several hundred cycles of barrier latency before it can issue
      // again; with two issuers one waits while the other issues.  Each warp runs its loop
      // convergently and one elected lane issues (issuing from a divergent `if (lane == 0)` makes
      // the compiler wrap every UTCHMMA in an ELECT/retry loop).  Both issuers accumulate into the
      // same TMEM buffer; the overwrite (accumulate = 0) MMA of a group is always issuer 0's first,
      // and issuer 1 does not start a group before that MMA has been issued (`first_issued`).
      const int j = (warp == 3) ? 1 : 0;
      const bool wide = p.dbg == 2 || (!p.single_pass && p.dbg != 1);
      const uint32_t idesc = umma_idesc_tf32(kTileRows, wide ? 2 * nb : nb);
      int s = j;
      for (int g = 0; g < ngroups; ++g) {
        const int b = g & 1;
        const uint32_t gph = (g >> 1) & 1;
        const int it_begin = g * p.flush, it_end = min(it_begin + p.flush, nkb);
        const uint32_t d_acc = tmem_base + static_cast<uint32_t>(b * 256);
        int it = it_begin + j;                          // flush is even: parity of `it` == issuer id
        // issuer 1 waits for issuer 0's first MMA of the group even when it has no k-block in it (odd tail): its
        // acc_full commit must not land in the barrier's previous phase
        if (j == 0) mbar_wait_fast(&acc_empty[b], gph ^ 1);
        else mbar_wait_fast(&first_issued[b], gph);
        tc_fence_after();
        for (; it < it_end; it += 2) {
          if (lane == 0) trace_ev(p, it, 11);
          named_bar_sync(1 + s, 32 + 32);               // the split warp owning stage s is done (implies TMA landed)
          if (lane == 0) trace_ev(p, it, 12);
          tc_fence_after();
          const uint32_t st = smem_u32(smem) + static_cast<uint32_t>(s) * static_cast<uint32_t>(p.stage_bytes);
          const uint64_t da = umma_desc_sw128(st);
          const uint64_t db = umma_desc_sw128(st + (has_b ? off_b : 0));
          if (elect_one()) {
            trace_ev(p, it, 4);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint64_t adv = static_cast<uint64_t>(ks * 2);  // 32 bytes (8 tf32) >> 4
              umma_tf32(d_acc, da + adv, db + adv, idesc, (it != it_begin) || (ks != 0));   // [hi*hi^T | hi*lo^T]
            }
            umma_commit(&empty_bar[s]);
            if (it == it_begin) mbar_arrive(&first_issued[b]);
            trace_ev(p, it, 5);
          }
          __syncwarp();
          s += 2;
          if (s >= p.stages) s -= p.stages;
        }
        if (elect_one()) umma_commit(&acc_full[b]);     // arrives once this issuer's MMAs of the group are done
        __syncwarp();
      }
    }
  } else if (wg == 1) {
    setmaxnreg_dec<96>();
    // ===================== split warps: lo = g - hi, one warp per stage (4 stages in parallel) =====================
    // hi = what the tensor core keeps of an fp32 operand (top 10 mantissa bits); lo is the exact residual,
    // stored at the same swizzled byte offsets in the sibling tile (the tensor core truncates it to 11 bits).
    const int w4 = warp - 4;
    const int nchunks_b = nb * 8;                         // 16-byte chunks of the B-side tile (rows < nb)
    int s = w4;
    uint32_t ph = 0;
    for (int it = w4; it < nkb; it += 4) {
      mbar_wait_fast(&full_bar[s], ph);
      if (lane == 0) trace_ev(p, it, 2);
      uint8_t* st = smem + static_cast<size_t>(s) * p.stage_bytes;
      if (!p.single_pass && p.dbg != 2) {
        const uint32_t src = smem_u32(st + (has_b ? off_b : 0)) + static_cast<uint32_t>(lane) * 16u;
        const uint32_t dst = smem_u32(st + off_lo) + static_cast<uint32_t>(lane) * 16u;
#pragma unroll 1
        for (int c0 = 0; c0 < nchunks_b; c0 += 8 * 32) {
          float4 v[8];
#pragma unroll
          for (int u = 0; u < 8; ++u)                     // all loads first: 8 LDS.128 in flight per thread
            if (c0 + u * 32 + lane < nchunks_b) v[u] = lds128(src + (c0 + u * 32) * 16);
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            if (c0 + u * 32 + lane < nchunks_b) {
              float4 l;
#if AFL_SPLIT_RN
              l.x = tf32_rna(v[u].x - tf32_trunc(v[u].x)); l.y = tf32_rna(v[u].y - tf32_trunc(v[u].y));
              l.z = tf32_rna(v[u].z - tf32_trunc(v[u].z)); l.w = tf32_rna(v[u].w - tf32_trunc(v[u].w));
#else
              l.x = v[u].x - tf32_trunc(v[u].x); l.y = v[u].y - tf32_trunc(v[u].y);
              l.z = v[u].z - tf32_trunc(v[u].z); l.w = v[u].w - tf32_trunc(v[u].w);
#endif
              sts128(dst + (c0 + u * 32) * 16, l);
            }
          }
        }
        fence_proxy_async_smem();
      }
      if (p.single_pass && p.loader == 1) fence_proxy_async_smem();   // cp.async data -> async proxy
      named_bar_arrive(1 + s, 32 + 32);
      if (lane == 0) trace_ev(p, it, 3);
      s += 4;
      if (s >= p.stages) { s -= p.stages; ph ^= 1; }
    }
  } else {
    setmaxnreg_inc<176>();
    // ===================== epilogue: drain TMEM chains into fp32 registers =====================
    const int q = warp & 3;             // TMEM lane quadrant this warp may access
    const int a = (warp - 8) >> 2;      // 0: hi*hi^T accumulator, 1: hi*lo^T accumulator
    float run[kTileRows];
#pragma unroll
    for (int i = 0; i < kTileRows; ++i) run[i] = 0.f;
    const bool active = !(a == 1 && p.single_pass);
    for (int g = 0; g < ngroups; ++g) {
      const int b = g & 1;
      mbar_wait_fast(&acc_full[b], (g >> 1) & 1);
      tc_fence_after();
      if (warp == 8 && lane == 0) trace_ev(p, g, 6);
      if (active) {
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                               static_cast<uint32_t>(b * 256 + a * nb);
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
          if (c * 16 < nb) {
            uint32_t v0[16], v1[16];
            tmem_ld_32x32b_x16(taddr + c * 16, v0);
            tmem_ld_32x32b_x16(taddr + c * 16 + 16, v1);   // columns past nb hold stale data; ignored
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              run[c * 16 + i] += __uint_as_float(v0[i]);
              run[c * 16 + 16 + i] += __uint_as_float(v1[i]);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[b]);
      if (warp == 8 && lane == 0) trace_ev(p, g, 7);
    }
    float* out = p.parts + (static_cast<size_t>(pair) * p.splits + split) * kPartElems +
                 static_cast<size_t>(a) * kTileRows * kTileRows + static_cast<size_t>(q * 32 + lane) * kTileRows;
#pragma unroll
    for (int c = 0; c < kTileRows; c += 4) {
      float4 v = make_float4(run[c], run[c + 1], run[c + 2], run[c + 3]);
      if (c >= nb || !active) v = make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(out + c) = v;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// Split reduction.  parts[pair][split][a][128][128] -> HX[a][n][n] (float64), a = 0: sum of hi*hi^T,
// a = 1: sum of hi*lo^T.  One block per (row i, accumulator a); threadIdx.x walks the columns (coalesced),
// threadIdx.y owns a fixed, contiguous range of splits; the kSy partial sums are then added in a fixed
// order, so the result is bit-reproducible and rows that were identical on input stay identical.
constexpr int kSy = 8;
__global__ void __launch_bounds__(128 * kSy)
gram_reduce_kernel(const float* __restrict__ parts, int n, int tiles, int splits, double* __restrict__ HX) {
  __shared__ double sh[kSy][128];
  const int i = blockIdx.x, a = blockIdx.y, tj = blockIdx.z;
  const int jj = threadIdx.x, sy = threadIdx.y;
  const int j = tj * kTileRows + jj;
  const int ti = i >> 7, ii = i & 127;
  const float* base = parts + static_cast<size_t>(ti * tiles + tj) * splits * kPartElems +
                      static_cast<size_t>(a) * kTileRows * kTileRows + ii * kTileRows + jj;
  const int s0 = splits * sy / kSy, s1 = splits * (sy + 1) / kSy;
  double acc = 0.0;
  if (j < n)
    for (int s = s0; s < s1; ++s) acc += static_cast<double>(base[static_cast<size_t>(s) * kPartElems]);
  sh[sy][jj] = acc;
  __syncthreads();
  if (sy == 0 && j < n) {
    double t = sh[0][jj];
#pragma unroll
    for (int y = 1; y < kSy; ++y) t += sh[y][jj];
    HX[(static_cast<size_t>(a) * n + i) * n + j] = t;
  }
}

// d2_ij = s_ii + s_jj - 2 s_ij with s_ij = hh_ij + (x_ij + x_ji); x_ij + x_ji is commutative, so s (and d2)
// are exactly symmetric, and identical rows give exact zeros.  hook.counter != null: the last block to finish also
// publishes this rank's epoch flag to every peer (csrc/xgpu.cu), which saves a launch per multi-GPU Krum step.
__global__ void gram_to_sqdist_kernel(const double* __restrict__ HX, int n, double* __restrict__ d2, const PubHook hook) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y;
  if (j < n) {
    const double* H = HX;
    const double* X = HX + static_cast<size_t>(n) * n;
    double v = 0.0;
    if (i != j) {
      const int lo = min(i, j), hi = max(i, j);
      const size_t ll = static_cast<size_t>(lo) * n + lo, hh = static_cast<size_t>(hi) * n + hi;
      const size_t lh = static_cast<size_t>(lo) * n + hi, hl = static_cast<size_t>(hi) * n + lo;
      const double s_ll = H[ll] + (X[ll] + X[ll]);
      const double s_hh = H[hh] + (X[hh] + X[hh]);
      const double s_lh = H[lh] + (X[lh] + X[hl]);
      v = (s_ll + s_hh) - 2.0 * s_lh;
    }
    d2[static_cast<size_t>(i) * n + j] = v;
  }
  if (!hook.counter) return;
  __shared__ int s_last;
  __threadfence_system();                                  // this block's rows, before its count
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(hook.counter, 1u) == gridDim.x * gridDim.y - 1u) ? 1 : 0;
  __syncthreads();
  if (!s_last) return;
  if (threadIdx.x == 0) *hook.counter = 0u;
  if (threadIdx.x < hook.world) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(hook.flag[threadIdx.x] + hook.rank), "l"(hook.epoch) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// SIMT difference kernel: block = 16x16 threads, tile = 32 x 32 client pairs, k-chunks of 32.
// ------------------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float load_elem(const T* p);
template <> __device__ __forceinline__ float load_elem<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float load_elem<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}

template <typename T>
__global__ void __launch_bounds__(256)
sqdist_simt_kernel(const T* __restrict__ G, int n, int64_t d, int64_t ld, int splits, double* __restrict__ part) {
  __shared__ float As[32][33], Bs[32][33];
  const int tiles = (n + 31) / 32;
  const int ti = blockIdx.x / tiles, tj = blockIdx.x % tiles;
  if (tj > ti) return;                                  // lower triangle (incl. diagonal tiles)
  const int split = blockIdx.y;
  const int64_t chunks = (d + 31) / 32;
  const int64_t c0 = chunks * split / splits, c1 = chunks * (split + 1) / splits;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  double acc[2][2] = {{0, 0}, {0, 0}};
  for (int64_t c = c0; c < c1; ++c) {
    const int64_t col0 = c * 32;
    for (int e = threadIdx.x; e < 32 * 32; e += 256) {
      const int r = e >> 5, k = e & 31;
      const int64_t col = col0 + k;
      const int ra = ti * 32 + r, rb = tj * 32 + r;
      As[r][k] = (ra < n && col < d) ? load_elem<T>(G + static_cast<int64_t>(ra) * ld + col) : 0.f;
      Bs[r][k] = (rb < n && col < d) ? load_elem<T>(G + static_cast<int64_t>(rb) * ld + col) : 0.f;
    }
    __syncthreads();
    float part32[2][2] = {{0, 0}, {0, 0}};
#pragma unroll 8
    for (int k = 0; k < 32; ++k) {
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          const float df = As[ty * 2 + u][k] - Bs[tx * 2 + v][k];   // fl32(g_i - g_j), as the reference
          part32[u][v] = fmaf(df, df, part32[u][v]);
        }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int v = 0; v < 2; ++v) acc[u][v] += static_cast<double>(part32[u][v]);
    __syncthreads();
  }
#pragma unroll
  for (int u = 0; u < 2; ++u)
#pragma unroll
    for (int v = 0; v < 2; ++v) {
      const int i = ti * 32 + ty * 2 + u, j = tj * 32 + tx * 2 + v;
      if (i < n && j < n && j < i) part[(static_cast<size_t>(split) * n + i) * n + j] = acc[u][v];
    }
}

__global__ void sqdist_simt_reduce_kernel(const double* __restrict__ part, int n, int splits,
                                          double* __restrict__ d2) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y;
  if (j >= n) return;
  double v = 0.0;
  if (i != j) {
    const int hi = max(i, j), lo = min(i, j);
    for (int s = 0; s < splits; ++s) v += part[(static_cast<size_t>(s) * n + hi) * n + lo];
  }
  d2[static_cast<size_t>(i) * n + j] = v;
}

__global__ void sqdist_to_dist_kernel(const double* __restrict__ d2, int n, float* __restrict__ dist) {
  const size_t e = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= static_cast<size_t>(n) * n) return;
  const int i = static_cast<int>(e / n), j = static_cast<int>(e % n);
  const double v = d2[e];
  dist[e] = (i == j) ? 0.f : static_cast<float>(sqrt(v > 0.0 ? v : 0.0));
}

// streaming bf16x2 kernel (gram_bf16.cu)
bool bf16x2_eligible(int n, int64_t d);
int bf16x2_splits(int64_t d);
int launch_bf16x2(const float* G, int n, int64_t d, int64_t ld, float* parts, int splits, int flush, int center, cudaStream_t stream);
// tile-pair bf16x2 kernel for N > 128 (gram_pair.cu)
int pair_splits(int n, int64_t d);
size_t pair_parts_bytes(int n, int64_t d);
size_t pair_center_bytes(int64_t d);
int launch_pair(const void* G, int dtype, int n, int64_t d, int64_t ld, float* parts, double* S, float* cvec, double* d2_out,
                int flush, int center, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

struct Plan {
  bool tensor;
  bool bf16;          // streaming bf16x2 kernel (gram_bf16.cu) instead of the TMA + split-TF32 kernel
  bool pair;          // lower-triangular tile-pair bf16x2 kernel (gram_pair.cu), N > 128
  int tiles, splits, stages, stage_bytes, flush, kchunk_log2;
  int simt_splits;
  size_t parts_bytes, s_bytes, total;
};

static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return (v && *v) ? atoi(v) : dflt;
}

static bool tensor_eligible(const void* G, int n, int64_t d, int64_t ld, int dtype) {
  const int64_t per16 = dtype == AFL_F32 ? 4 : 8;           // elements per 16 bytes: TMA needs 16-byte aligned rows
  return (dtype == AFL_F32 || dtype == AFL_BF16) && (ld % per16 == 0) && (reinterpret_cast<uintptr_t>(G) % 16 == 0) && n >= 1 &&
         d >= 1 && n <= 4096 && d < (int64_t(1) << 31) - 64;
}

static Plan make_plan(const void* G, int n, int64_t d, int64_t ld, int dtype, int flags) {
  Plan pl{};
  pl.tensor = !(flags & AFL_GRAM_FORCE_SIMT) && tensor_eligible(G, n, d, ld, dtype);
  const int sms = sm_count();
  if (pl.tensor) {
    pl.tiles = (n + kTileRows - 1) / kTileRows;
    const char* kenv = getenv("AFL_GRAM_KERNEL");
    // Streaming shapes (64 <= N_pad <= 112, D >= 32768) default to the bf16x2 kernel (gram_bf16.cu: twice the
    // tensor headroom and a loader that is not capped by the TMA box rate); AFL_GRAM_TF32X2 or
    // AFL_GRAM_KERNEL=tf32 keeps the TMA + split-TF32 kernel (smaller uniform bias, ~0.9e-6 vs ~3.2e-6).
    pl.bf16 = bf16x2_eligible(n, d) && !(flags & (AFL_GRAM_SINGLE_PASS | AFL_GRAM_TF32X2)) &&
              !(kenv && kenv[0] == 't');
    const int pairs = pl.tiles * pl.tiles;
    int kc_log2 = env_int("AFL_GRAM_KCHUNK_LOG2", 0);
    if (kc_log2 < 0 || kc_log2 > 4) kc_log2 = 0;
    pl.kchunk_log2 = kc_log2;
    const int kChunk = 1 << kc_log2;
    const int kblocks = (static_cast<int>((d + kBK - 1) / kBK) + kChunk - 1) / kChunk;   // in chunks
    // choose K-splits so that pairs*splits fills an integer number of waves as well as possible
    int best = 1; double best_eff = -1.0;
    for (int w = 1; w <= 4; ++w) {
      int s = (sms * w) / pairs; if (s < 1) s = 1;
      if (s > kblocks) s = kblocks;
      const int ctas = pairs * s;
      const double eff = static_cast<double>(ctas) / (static_cast<double>((ctas + sms - 1) / sms) * sms);
      if (eff > best_eff + 1e-9) { best_eff = eff; best = s; }
      if (s == kblocks) break;
    }
    pl.splits = env_int("AFL_GRAM_SPLITS", best);
    if (pl.splits > kblocks) pl.splits = kblocks;
    if (pl.splits < 1) pl.splits = 1;
    if (pl.tiles == 1) {
      // single tile: a stage is exactly raw(nb rows) || lo(nb rows); the ring is as deep as shared memory allows
      const int nb = (n + 15) & ~15;
      pl.stage_bytes = 2 * nb * 128;
      // the A operand always spans 128 rows from the stage base: keep that inside the allocation
      const int slack = (2 * nb < kTileRows) ? (kTileRows - 2 * nb) * 128 : 0;
      int st = (225 * 1024 - slack) / pl.stage_bytes;
      if (st > 14) st = 14;                            // named barrier ids 1..15
      if (st > 12) st = 12;
      st &= ~3;                                        // multiple of 4: split warp w owns stages w, w+4, ...
      pl.stages = env_int("AFL_GRAM_STAGES", st);
      if (pl.stages > st) pl.stages = st;
      if (pl.stages < 4) pl.stages = 4;
      pl.stages &= ~3;
    } else {
      pl.stage_bytes = 3 * kTileBytes;
      pl.stages = 4;
    }
    pl.flush = env_int("AFL_GRAM_FLUSH", 4);
    if (pl.flush < 2) pl.flush = 2;
    pl.flush &= ~1;                                     // even: the two issuers alternate k-blocks
    if (pl.bf16) pl.splits = bf16x2_splits(d);
    pl.parts_bytes = static_cast<size_t>(pairs) * pl.splits * kPartElems * sizeof(float);
    // N > 128: the triangular bf16x2 tile-pair kernel (AFL_GRAM_TF32X2 / AFL_GRAM_KERNEL=tf32 keeps the round-1
    // all-ordered-pairs split-TF32 kernel for comparison)
    pl.pair = (n > kTileRows && !(flags & (AFL_GRAM_SINGLE_PASS | AFL_GRAM_TF32X2)) && !(kenv && kenv[0] == 't')) ||
              dtype == AFL_BF16;      // bf16 matrices: TMA delivers ready-made operand tiles to the pair kernel (any n)
    if (dtype == AFL_BF16) pl.bf16 = false;
    if (pl.pair) { pl.splits = pair_splits(n, d); pl.parts_bytes = pair_parts_bytes(n, d); }
    pl.s_bytes = align_up(2 * static_cast<size_t>(n) * n * sizeof(double), 256);
    pl.total = pl.parts_bytes + pl.s_bytes + (pl.pair ? pair_center_bytes(d) : 0);
  } else {
    const int t32 = (n + 31) / 32;
    int64_t chunks = (d + 31) / 32;
    int s = (sms * 8) / (t32 * (t32 + 1) / 2); if (s < 1) s = 1;
    if (s > chunks) s = static_cast<int>(chunks);
    if (s > 1024) s = 1024;
    pl.simt_splits = s;
    pl.total = static_cast<size_t>(s) * n * n * sizeof(double);
  }
  pl.total = align_up(pl.total, 256);
  return pl;
}

size_t workspace_bytes(int n, int64_t d, int dtype, int flags) {
  // Upper bound that holds for either path (the pointer alignment is unknown here).
  Plan a = make_plan(reinterpret_cast<const void*>(16), n, d, 8, dtype, flags & ~AFL_GRAM_FORCE_SIMT);
  Plan b = make_plan(reinterpret_cast<const void*>(16), n, d, 8, dtype, flags | AFL_GRAM_FORCE_SIMT);
  return (a.total > b.total ? a.total : b.total) + 256;
}

int sqdist_partial_ex(const void* G, int n, int64_t d, int64_t ld, int dtype, double* d2_out, void* ws, size_t ws_bytes,
                      int flags, cudaStream_t stream, const PubHook* hook, bool* hook_done);
int sqdist_partial(const void* G, int n, int64_t d, int64_t ld, int dtype, double* d2_out, void* ws, size_t ws_bytes,
                   int flags, cudaStream_t stream) {
  return sqdist_partial_ex(G, n, d, ld, dtype, d2_out, ws, ws_bytes, flags, stream, nullptr, nullptr);
}
// hook != null: the caller (csrc/xgpu.cu) wants its epoch flag published once d2_out is complete; *hook_done tells
// whether gram_to_sqdist_kernel did it (single-tile bf16x2 path) or the caller still has to launch its publish kernel.
int sqdist_partial_ex(const void* G, int n, int64_t d, int64_t ld, int dtype, double* d2_out, void* ws, size_t ws_bytes,
                      int flags, cudaStream_t stream, const PubHook* hook, bool* hook_done) {
  if (hook_done) *hook_done = false;
  if (!G || !d2_out || n < 1 || d < 1 || ld < d) { set_error("afl_sqdist_partial: bad argument"); return AFL_ERR_BAD_ARG; }
  if (dtype != AFL_F32 && dtype != AFL_BF16) { set_error("afl_sqdist_partial: dtype"); return AFL_ERR_UNSUPPORTED; }
  Plan pl = make_plan(G, n, d, ld, dtype, flags);
  if ((flags & AFL_GRAM_FORCE_TCGEN05) && !pl.tensor) {
    set_error("afl_sqdist_partial: tcgen05 path needs fp32, 16-byte aligned base and pitch %% 4 == 0, n <= 4096");
    return AFL_ERR_UNSUPPORTED;
  }
  if (!ws || ws_bytes < pl.total || (reinterpret_cast<uintptr_t>(ws) % 256) != 0) {
    set_error("afl_sqdist_partial: workspace too small or misaligned (%zu < %zu)", ws_bytes, pl.total);
    return AFL_ERR_WORKSPACE;
  }
  const dim3 rblock(128), rgrid((n + 127) / 128, n);
  // translation invariance: operands are converted as g - (last client's row) unless switched off
  const int center = !(flags & AFL_GRAM_NO_CENTER) && env_int("AFL_GRAM_CENTER", 1) != 0;
  if (pl.tensor) {
    if (pl.pair) {
      float* parts = static_cast<float*>(ws);
      double* S = reinterpret_cast<double*>(static_cast<uint8_t*>(ws) + pl.parts_bytes);
      float* cvec = reinterpret_cast<float*>(static_cast<uint8_t*>(ws) + pl.parts_bytes + pl.s_bytes);
      return launch_pair(G, dtype, n, d, ld, parts, S, cvec, d2_out, pl.flush, center, stream);
    }
    if (pl.bf16) {
      float* parts = static_cast<float*>(ws);
      double* S = reinterpret_cast<double*>(static_cast<uint8_t*>(ws) + pl.parts_bytes);
      int rc = launch_bf16x2(static_cast<const float*>(G), n, d, ld, parts, pl.splits, pl.flush, center, stream);
      if (rc) return rc;
      gram_reduce_kernel<<<dim3(n, 2, 1), dim3(128, kSy), 0, stream>>>(parts, n, 1, pl.splits, S);
      AFL_LAUNCH_CHECK("gram_reduce_kernel");
      const bool pub = hook && hook->counter;
      PubHook h{};
      if (pub && hook->world > 1) h = *hook;           // a single rank has no flag to publish
      gram_to_sqdist_kernel<<<rgrid, rblock, 0, stream>>>(S, n, d2_out, h);
      AFL_LAUNCH_CHECK("gram_to_sqdist_kernel");
      if (hook_done) *hook_done = pub;
      return AFL_OK;
    }
    EncodeTiledFn enc = encode_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled entry point not found"); return AFL_ERR_CUDA; }
    CUtensorMap tmap;
    const cuuint64_t gdim[2] = {static_cast<cuuint64_t>(d), static_cast<cuuint64_t>(n)};
    const cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * sizeof(float)};
    int box_rows = kTileRows;
    if (pl.tiles == 1) box_rows = (n + 15) & ~15;     // rows n..nb-1 are TMA zero fill; nothing past nb is written
    if (box_rows < 8 || box_rows > kTileRows || pl.tiles > 1) box_rows = kTileRows;
    const cuuint32_t box[2] = {kBK, static_cast<cuuint32_t>(box_rows)};
    const cuuint32_t estride[2] = {1, 1};
    CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(G), gdim, gstride, box, estride,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed: %d", static_cast<int>(r)); return AFL_ERR_CUDA; }
    Params p{};
    p.n = n; p.tiles = pl.tiles; p.splits = pl.splits; p.kblocks = static_cast<int>((d + kBK - 1) / kBK);
    p.flush = pl.flush; p.stages = pl.stages; p.stage_bytes = pl.stage_bytes;
    p.single_pass = (flags & AFL_GRAM_SINGLE_PASS) ? 1 : 0;
    p.box_rows = box_rows;
    p.dbg = env_int("AFL_GRAM_DBG", 0);
    p.kchunk_log2 = pl.kchunk_log2;
    p.loader = env_int("AFL_GRAM_LOADER", 0) ? 1 : 0;
    p.G = static_cast<const float*>(G); p.ld = ld; p.d = d;
    p.rewrite_hi = 0;   // AFL_GRAM_REWRITE_HI is accepted but ignored: kind::tf32 was measured to truncate
    p.parts = static_cast<float*>(ws);
    double* S = reinterpret_cast<double*>(static_cast<uint8_t*>(ws) + pl.parts_bytes);
    const size_t smem = static_cast<size_t>(pl.stages) * pl.stage_bytes + 1024 +
                        ((pl.tiles == 1 && pl.stage_bytes < kTileBytes) ? (kTileBytes - pl.stage_bytes) : 0);
  static int smem_attr_done[kMaxDevices] = {0};
  AFL_CUDA(ensure_dyn_smem(gram_tcgen05_kernel, 226 * 1024, smem_attr_done));
    const char* trace_path = getenv("AFL_GRAM_TRACE");      // debug aid: dump per-role clock64 timestamps
    if (trace_path && *trace_path) {
      AFL_CUDA(cudaMalloc(&p.trace, sizeof(long long) * 2 * kTraceLen * kTraceEv));
      AFL_CUDA(cudaMemsetAsync(p.trace, 0, sizeof(long long) * 2 * kTraceLen * kTraceEv, stream));
    }
    {
      ProfScope ps("gram_tcgen05", stream);
      gram_tcgen05_kernel<<<pl.tiles * pl.tiles * pl.splits, kThreads, smem, stream>>>(tmap, p);
    }
    if (p.trace) {
      static long long host_trace[2 * kTraceLen * kTraceEv];
      AFL_CUDA(cudaStreamSynchronize(stream));
      AFL_CUDA(cudaMemcpy(host_trace, p.trace, sizeof(host_trace), cudaMemcpyDeviceToHost));
      cudaFree(p.trace);
      if (FILE* f = fopen(trace_path, "w")) {
        for (int c = 0; c < 2; ++c)
          for (int i = 0; i < kTraceLen; ++i) {
            fprintf(f, "%d %d", c, i);
            for (int e = 0; e < kTraceEv; ++e) fprintf(f, " %lld", host_trace[(c * kTraceLen + i) * kTraceEv + e]);
            fprintf(f, "\n");
          }
        fclose(f);
      }
    }
    AFL_LAUNCH_CHECK("gram_tcgen05_kernel");
    gram_reduce_kernel<<<dim3(n, 2, pl.tiles), dim3(128, kSy), 0, stream>>>(p.parts, n, pl.tiles, pl.splits, S);
    AFL_LAUNCH_CHECK("gram_reduce_kernel");
    gram_to_sqdist_kernel<<<rgrid, rblock, 0, stream>>>(S, n, d2_out, PubHook{});
    AFL_LAUNCH_CHECK("gram_to_sqdist_kernel");
  } else {
    const int t32 = (n + 31) / 32;
    double* part = static_cast<double*>(ws);
    const dim3 grid(t32 * t32, pl.simt_splits);
    {
      ProfScope ps("sqdist_simt", stream);
      if (dtype == AFL_F32)
        sqdist_simt_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(G), n, d, ld, pl.simt_splits, part);
      else
        sqdist_simt_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(G), n, d, ld,
                                                                     pl.simt_splits, part);
    }
    AFL_LAUNCH_CHECK("sqdist_simt_kernel");
    sqdist_simt_reduce_kernel<<<rgrid, rblock, 0, stream>>>(part, n, pl.simt_splits, d2_out);
    AFL_LAUNCH_CHECK("sqdist_simt_reduce_kernel");
  }
  return AFL_OK;
}

int sqdist_to_dist(const double* d2, int n, float* dist, cudaStream_t stream) {
  if (!d2 || !dist || n < 1) { set_error("afl_sqdist_to_dist: bad argument"); return AFL_ERR_BAD_ARG; }
  const size_t total = static_cast<size_t>(n) * n;
  sqdist_to_dist_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(d2, n, dist);
  AFL_LAUNCH_CHECK("sqdist_to_dist_kernel");
  return AFL_OK;
}

}  // namespace gram
}  // namespace afl
