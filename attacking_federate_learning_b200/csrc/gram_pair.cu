// Gram kernel for N > 128 clients (Bulyan N = 500, ALIE -> Krum / Bulyan N = 1000; reference:
// defences.py:16-21): lower-triangular 128 x 128 tile pairs, bf16x2 operands converted IN PLACE.
//
//   * The N x N table is cut into T = ceil(N/128) row tiles; only the T(T+1)/2 pairs (I >= J) are computed
//     (the round-1 kernel computed all T^2 ordered pairs).  CTA = (pair, K split); split s owns the 64-column
//     k-blocks s, s+S, s+2S, ... and writes its partial [hh | X] tile to a private slot, which
//     pair_reduce_kernel sums in a fixed order in float64 (bit-reproducible).
//   * One TMA box {64 fp32 columns x 128 rows} (32 KB, no swizzle, OOB rows/columns zero-filled) per tile and
//     k-block lands in a 7-slot shared-memory ring (tools/tma_bench.cu: ~450 ns per box per SM whatever it
//     holds, so boxes must be this large).  A converter warp then rewrites the slot IN PLACE: every 8-row unit
//     (2 KB of fp32) becomes one SWIZZLE_128B core-matrix atom of b1 (1 KB) followed by one of b2 (1 KB), with
//     g - c = b1 + b2 + r, |r| <= 2^-17 |g - c| (both roundings to nearest), c = the mean of the LAST 8 clients' rows
//     (translation invariance of the distances: the cancellation error of d2 = s_ii + s_jj - 2 s_ij then
//     scales with the distances to an honest client - main.py:28 makes ids >= f honest - instead of with
//     ||g||^2).  A unit's output only overwrites that unit's own input, which the warp has already loaded, so
//     there is no second staging buffer: 7 x 32 KB of shared memory hold 3.5 k-blocks in flight.
//   * Operands are K-major with an 8-row-group stride (SBO) of 2048 bytes: b1 tile at slot + 0, b2 tile at
//     slot + 1024.  Per 16 columns three tcgen05.mma.kind::f16 (M = 128, N = 128, K = 16):
//         hh += b1_I b1_J^T        X += b1_I b2_J^T        X += b2_I b1_J^T
//     EVERY pair - diagonal ones too - issues exactly this sequence on the same K partition, so two clients
//     with identical rows get bit-identical s_ii, s_jj and s_ij wherever their tiles are, and their distance
//     is exactly 0 (ALIE makes rows 0..f-1 one array, f = 240 spans two tiles at N = 1000; Krum's
//     [1, 0, 2, ...] tie-break depends on it).  S_ij = hh + X for i >= j, mirrored.
//   * TMEM: two accumulator buffers of 256 columns ([hh | X]), drained every `flush` k-blocks by 8 epilogue
//     warps into fp32 registers (the tensor core truncates while accumulating; chains stay short).
//
// Warp roles (512 threads): warp 0 TMA producer, warps 1,3 MMA issue (alternating k-blocks), warp 2 TMEM
// alloc, warps 4-7 converters (warp w owns boxes w, w+4, ...), warps 8-15 epilogue.
// bounded waits trap after 2^35 cycles (~18 s) here: profiler replays with patched SASS run this kernel >100x slower
#define AFL_BAR_TIMEOUT_LOG2 35
#include "afl_common.cuh"

namespace afl {
namespace gram {

constexpr int kPThreads = 512;
// J tile by cp.async (LDGSTS) from warp 2 instead of a second TMA box per k-block: measured 2.3x SLOWER than two TMA
// boxes (r02 run E: 6.2 ms vs 2.7 ms at N = 1000, D = 524,288), kept behind this switch for the record.
constexpr bool kJByCpAsync = false;
constexpr int kPSlots = kJByCpAsync ? 6 : 7;   // 32 KB slots: one box = one tile's k-block
constexpr int kPSlotBytes = 128 * 256;       // 128 rows x 64 fp32
constexpr int kPCols = 64;                   // columns per k-block
constexpr int kPPartElems = 2 * 128 * 128;   // [hh | X] per (pair, split)

struct PairParams {
  int n, tiles, pairs, splits;
  int kblocks;          // ceil(d / 64)
  int flush;            // k-blocks per TMEM accumulation chain (even)
  int center;           // subtract the last client's row while converting
  const float* cref;    // first of the last cref_rows rows
  int cref_rows; int64_t cref_ld;
  const float* cvec;    // precomputed centre (mean of those rows), padded with zeros to a multiple of 64 columns
  int64_t d;
  float* parts;         // [pairs][splits][2][128][128]
  const float* G;       // matrix base and pitch (elements): the J tile is loaded with cp.async (LDGSTS), not TMA
  int64_t ld;
  int in_bf16;          // bf16 client matrix: TMA delivers ready-made SWIZZLE_128B operand tiles (b1 = g exactly, no b2,
                        // no converter pass, no centring), one MMA per 16 columns
};

__global__ void __launch_bounds__(kPThreads, 1)
gram_pair_kernel(const __grid_constant__ CUtensorMap tmap, const PairParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t raw_full[kPSlots], slot_free[kPSlots], acc_full[2], acc_empty[2], first_issued[2];
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wg = warp >> 2;
  const int pair = blockIdx.x % p.pairs;
  const int split = blockIdx.x / p.pairs;
  int ti = 0;
  while ((ti + 1) * (ti + 2) / 2 <= pair) ++ti;           // pair = ti (ti + 1) / 2 + tj, tj <= ti
  const int tj = pair - ti * (ti + 1) / 2;
  const bool has_b = ti != tj;
  const int nbx = has_b ? 2 : 1;                            // TMA boxes (= ring slots) per k-block
  const int nkb = split < p.kblocks ? (p.kblocks - split + p.splits - 1) / p.splits : 0;
  const int nboxes = nkb * nbx;
  const int ngroups = (nkb + p.flush - 1) / p.flush;
  const uint32_t ring = smem_u32(smem);
  // Box b of this CTA (b = k-block * nbx + which) lives in ring slot slot_of(b).  Off-diagonal pairs keep the I tile
  // (TMA, one expect_tx arrival) in even slots and the J tile (cp.async, one arrival per lane) in odd slots: the TMA
  // unit then moves ONE box per k-block (it needs ~450-600 ns per box whatever the box holds, more than the ~680 ns of
  // tensor work per k-block would leave for two), the other 32 KB go through the LSU path.
  auto slot_of = [&](int b) -> int { return (kJByCpAsync && has_b) ? ((b >> 1) % 3) * 2 + (b & 1) : b % kPSlots; };
  auto phase_of = [&](int b) -> uint32_t { return static_cast<uint32_t>((kJByCpAsync && has_b) ? ((b >> 1) / 3) : (b / kPSlots)) & 1u; };

  if (threadIdx.x == 0) {
    for (int s = 0; s < kPSlots; ++s) { mbar_init(&raw_full[s], (kJByCpAsync && has_b && (s & 1)) ? 32 : 1); mbar_init(&slot_free[s], 1); }
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
  const uint32_t tmem_base = tmem_base_smem;

  if (wg == 0) {
    setmaxnreg_dec<64>();
    if (warp == 0) {
      // ===================== TMA producer: one box {64 cols x 128 rows} per (tile, k-block) =====================
      if (lane == 0) {
        const uint64_t pol = policy_evict_normal();       // every row tile is read by T CTAs: keep it in L2
        for (int i = 0; i < nkb; ++i) {
          for (int t = 0; t < ((kJByCpAsync || !has_b) ? 1 : 2); ++t) {
            const int b = i * nbx + t;
            const int s = slot_of(b);
            mbar_wait(&slot_free[s], phase_of(b) ^ 1u);
            mbar_arrive_expect_tx(&raw_full[s], p.in_bf16 ? kPSlotBytes / 2 : kPSlotBytes);
            tma_load_2d(smem + static_cast<size_t>(s) * kPSlotBytes, &tmap, &raw_full[s], (split + i * p.splits) * kPCols,
                        (t == 0 ? ti : tj) * 128, pol);
          }
        }
      }
    } else if (warp == 2) {
      // ===================== J-tile producer: cp.async (LDGSTS), 16 bytes per lane, zero fill past d =====================
      if (kJByCpAsync && has_b) {
        const float* gj = p.G + static_cast<int64_t>(tj) * 128 * p.ld;    // tj < ti: the J tile always has 128 rows
        for (int i = 0; i < nkb; ++i) {
          const int b = 2 * i + 1;
          const int s = slot_of(b);
          mbar_wait_warp(&slot_free[s], phase_of(b) ^ 1u);
          const int64_t col = static_cast<int64_t>(split + i * p.splits) * kPCols;
          const uint32_t dst = ring + static_cast<uint32_t>(s) * kPSlotBytes;
#pragma unroll 8
          for (int it = 0; it < 64; ++it) {                // a warp instruction copies 2 rows x 256 bytes
            const int q = it * 32 + lane, row = q >> 4, c = q & 15;
            const int64_t cc = col + 4 * c, rem = p.d - cc;
            const uint32_t nbytes = rem >= 4 ? 16u : (rem > 0 ? static_cast<uint32_t>(rem) * 4u : 0u);
            const float* src = nbytes ? gj + static_cast<int64_t>(row) * p.ld + cc : p.G;
            cp_async_16(dst + static_cast<uint32_t>(row) * 256u + static_cast<uint32_t>(c) * 16u, src, nbytes);
          }
          cp_async_mbar_arrive_noinc(&raw_full[s]);
        }
      }
    } else if (warp == 1 || warp == 3) {
      // ===================== MMA issuers (alternating k-blocks) =====================
      const int j = (warp == 3) ? 1 : 0;
      const uint32_t idesc = umma_idesc_bf16(128, 128);
      for (int g = 0; g < ngroups; ++g) {
        const int b = g & 1;
        const uint32_t gph = (g >> 1) & 1;
        const int it_begin = g * p.flush, it_end = min(it_begin + p.flush, nkb);
        const uint32_t d_hh = tmem_base + static_cast<uint32_t>(b * 256);
        const uint32_t d_x = d_hh + 128u;
        int it = it_begin + j;
        // issuer 0 owns the group's first k-block and waits for the epilogue to have drained this buffer; issuer 1
        // waits for that first MMA to be issued EVEN IF it has no k-block in this group (odd tail), so that its
        // acc_full commit can never land in the previous phase of the barrier
        if (j == 0) mbar_wait_fast(&acc_empty[b], gph ^ 1);
        else mbar_wait_fast(&first_issued[b], gph);
        tc_fence_after();
        for (; it < it_end; it += 2) {
          const int s_i = slot_of(it * nbx);
          const int s_j = has_b ? slot_of(it * nbx + 1) : s_i;
          if (p.in_bf16) {                                // TMA wrote the operand tiles themselves
            mbar_wait_fast(&raw_full[s_i], phase_of(it * nbx));
            if (has_b) mbar_wait_fast(&raw_full[s_j], phase_of(it * nbx + 1));
          } else {
            named_bar_sync(1 + s_i, 32 + 32);            // the converter warp of that box has written and fenced it
            if (has_b) named_bar_sync(1 + s_j, 32 + 32);
          }
          // Strict alternation of the two issuers: k-block `it` is issued only after k-block it-1 has been, so every
          // CTA accumulates its k-blocks in the same order and identical rows get bit-identical sums in every tile
          // pair (and the table is reproducible run to run).  Barrier 8: issuer 0 -> 1, barrier 9: issuer 1 -> 0.
          if (it > 0) named_bar_sync(j == 0 ? 9u : 8u, 32 + 32);
          tc_fence_after();
          const uint32_t a_i = ring + static_cast<uint32_t>(s_i) * kPSlotBytes;
          const uint32_t a_j = ring + static_cast<uint32_t>(s_j) * kPSlotBytes;
          const uint32_t sbo = p.in_bf16 ? 1024u : 2048u;
          const uint64_t d_b1i = umma_desc_sw128_sbo(a_i, sbo), d_b2i = umma_desc_sw128_sbo(a_i + 1024u, 2048u);
          const uint64_t d_b1j = umma_desc_sw128_sbo(a_j, sbo), d_b2j = umma_desc_sw128_sbo(a_j + 1024u, 2048u);
          if (elect_one()) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {             // 4 x K=16 bf16 = 64 columns; +32 bytes per step
              const uint64_t adv = static_cast<uint64_t>(ks * 2);
              const uint32_t acc = (it != it_begin) || (ks != 0);
              umma_bf16(d_hh, d_b1i + adv, d_b1j + adv, idesc, acc);       // hh += b1_I b1_J^T
              if (!p.in_bf16) {
                umma_bf16(d_x, d_b1i + adv, d_b2j + adv, idesc, acc);      // X  += b1_I b2_J^T
                umma_bf16(d_x, d_b2i + adv, d_b1j + adv, idesc, 1u);       // X  += b2_I b1_J^T
              }
            }
            umma_commit(&slot_free[s_i]);
            if (has_b) umma_commit(&slot_free[s_j]);
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
    setmaxnreg_dec<96>();
    // ===================== converters: fp32 box -> b1 / b2 atoms, in place (bf16x2_convert_units) =====================
    const int w4 = warp - 4;
    const int c16 = lane & 15;
    uint32_t src_lane, dst_off[4];
    bf16x2_lane_offsets(src_lane, dst_off);
    float4 cen = make_float4(0.f, 0.f, 0.f, 0.f);
    auto load_center = [&](int box) -> float4 {
      if (!(p.center && box < nboxes)) return make_float4(0.f, 0.f, 0.f, 0.f);
      const int64_t col = static_cast<int64_t>(split + (box / nbx) * p.splits) * kPCols + c16 * 4;
      return __ldg(reinterpret_cast<const float4*>(p.cvec + col));     // one load per box (measured: 8 row loads cost 12 %)
    };
    cen = load_center(w4);
    for (int box = w4; box < (p.in_bf16 ? 0 : nboxes); box += 4) {
      const int s = slot_of(box);
      const uint32_t ph = phase_of(box);
      const float4 cnext = load_center(box + 4);          // in flight while this box is converted
      // the slot's previous box (another converter's) may still be in flight: wait for its MMA commit first, or the
      // raw_full wait below could see that box's phase as this one's (see gram_bf16.cu)
      if (box >= kPSlots) mbar_wait_fast(&slot_free[s], ph ^ 1u);
      mbar_wait_fast(&raw_full[s], ph);
      bf16x2_convert_units(ring + static_cast<uint32_t>(s) * kPSlotBytes, 16, src_lane, dst_off, cen);
      cen = cnext;
      fence_proxy_async_smem();
      named_bar_arrive(1 + s, 32 + 32);
    }
  } else {
    setmaxnreg_inc<176>();
    // ===================== epilogue: drain TMEM chains into fp32 registers =====================
    const int q = warp & 3;             // TMEM lane quadrant this warp may access
    const int a = (warp - 8) >> 2;      // 0: hh columns, 1: X columns
    float run[128];
#pragma unroll
    for (int i = 0; i < 128; ++i) run[i] = 0.f;
    for (int g = 0; g < ngroups; ++g) {
      const int b = g & 1;
      mbar_wait_fast(&acc_full[b], (g >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(b * 256 + a * 128);
#pragma unroll
      for (int c = 0; c < ((p.in_bf16 && a == 1) ? 0 : 8); c += 2) {
        uint32_t v0[16], v1[16];
        tmem_ld_32x32b_x16(taddr + c * 16, v0);
        tmem_ld_32x32b_x16(taddr + c * 16 + 16, v1);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          run[c * 16 + i] += __uint_as_float(v0[i]);
          run[c * 16 + 16 + i] += __uint_as_float(v1[i]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[b]);
    }
    float* out = p.parts + (static_cast<size_t>(pair) * p.splits + split) * kPPartElems +
                 static_cast<size_t>(a) * 128 * 128 + static_cast<size_t>(q * 32 + lane) * 128;
#pragma unroll
    for (int c = 0; c < 128; c += 4) *reinterpret_cast<float4*>(out + c) = make_float4(run[c], run[c + 1], run[c + 2], run[c + 3]);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// Split reduction of the lower-triangular tile pairs: S[i][j] (i >= j, float64) = sum_s hh + sum_s X, splits in
// a fixed order (threadIdx.y owns a contiguous range, the kPSy partial sums are added in order).
constexpr int kPSy = 8;
__global__ void __launch_bounds__(128 * kPSy)
pair_reduce_kernel(const float* __restrict__ parts, int n, int splits, double* __restrict__ S) {
  __shared__ double sh[2][kPSy][128];
  const int i = blockIdx.x, tj = blockIdx.y;
  const int ti = i >> 7, ii = i & 127;
  if (tj > ti) return;
  const int jj = threadIdx.x, sy = threadIdx.y;
  const int j = tj * 128 + jj;
  const int pair = ti * (ti + 1) / 2 + tj;
  const float* base = parts + static_cast<size_t>(pair) * splits * kPPartElems + ii * 128 + jj;
  const int s0 = splits * sy / kPSy, s1 = splits * (sy + 1) / kPSy;
  double hh = 0.0, xx = 0.0;
  if (j <= i && j < n)
    for (int s = s0; s < s1; ++s) {
      hh += static_cast<double>(base[static_cast<size_t>(s) * kPPartElems]);
      xx += static_cast<double>(base[static_cast<size_t>(s) * kPPartElems + 128 * 128]);
    }
  sh[0][sy][jj] = hh;
  sh[1][sy][jj] = xx;
  __syncthreads();
  if (sy == 0 && j <= i && j < n) {
    double th = sh[0][0][jj], tx = sh[1][0][jj];
#pragma unroll
    for (int y = 1; y < kPSy; ++y) { th += sh[0][y][jj]; tx += sh[1][y][jj]; }
    S[static_cast<size_t>(i) * n + j] = th + tx;
  }
}

// d2_ij = (S_hh + S_ll) - 2 S_hl with h = max(i, j), l = min(i, j): exactly symmetric, zero diagonal, and exactly
// zero between clients whose rows are identical.
__global__ void pair_to_sqdist_kernel(const double* __restrict__ S, int n, double* __restrict__ d2) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y;
  if (j >= n) return;
  double v = 0.0;
  if (i != j) {
    const int lo = min(i, j), hi = max(i, j);
    v = (S[static_cast<size_t>(hi) * n + hi] + S[static_cast<size_t>(lo) * n + lo]) - 2.0 * S[static_cast<size_t>(hi) * n + lo];
  }
  d2[static_cast<size_t>(i) * n + j] = v;
}

// centre vector: mean of the last `rows` clients, zero past d (the k-blocks are 64 columns wide)
__global__ void __launch_bounds__(256)
pair_center_kernel(const float* __restrict__ cref, int rows, int64_t ld, int64_t d, int64_t d_pad, float* __restrict__ cvec) {
  const int64_t col = (static_cast<int64_t>(blockIdx.x) * 256 + threadIdx.x) * 4;
  if (col >= d_pad) return;
  const float4 c = gram_center(cref, rows, ld, col, d);
  *reinterpret_cast<float4*>(cvec + col) = c;
}

typedef CUresult (*EncodeTiledFn3)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int pair_splits(int n, int64_t d) {
  const int tiles = (n + 127) / 128, pairs = tiles * (tiles + 1) / 2;
  const int64_t kblocks = (d + kPCols - 1) / kPCols;
  int s = sm_count() / pairs;
  if (const char* e = getenv("AFL_GRAM_SPLITS")) if (atoi(e) > 0) s = atoi(e);
  if (s > kblocks) s = static_cast<int>(kblocks);
  return s < 1 ? 1 : s;
}
size_t pair_center_bytes(int64_t d) { return align_up(static_cast<size_t>((d + kPCols - 1) / kPCols * kPCols) * sizeof(float), 256); }
size_t pair_parts_bytes(int n, int64_t d) {
  const int tiles = (n + 127) / 128, pairs = tiles * (tiles + 1) / 2;
  return static_cast<size_t>(pairs) * pair_splits(n, d) * kPPartElems * sizeof(float);
}

// G: fp32 [n, d] (pitch multiple of 4 elements) or bf16 (pitch multiple of 8), 16-byte aligned.
// parts: pair_parts_bytes(); S: n*n doubles.
int launch_pair(const void* Gv, int dtype, int n, int64_t d, int64_t ld, float* parts, double* S, float* cvec, double* d2_out,
                int flush, int center, cudaStream_t stream) {
  const float* G = static_cast<const float*>(Gv);
  const bool bf16 = dtype == AFL_BF16;
  static EncodeTiledFn3 enc = nullptr;
  if (!enc) {
    void* fp = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess) { set_error("cuTensorMapEncodeTiled entry point not found"); return AFL_ERR_CUDA; }
    enc = reinterpret_cast<EncodeTiledFn3>(fp);
  }
  PairParams p{};
  p.n = n; p.tiles = (n + 127) / 128; p.pairs = p.tiles * (p.tiles + 1) / 2;
  p.splits = pair_splits(n, d);
  p.kblocks = static_cast<int>((d + kPCols - 1) / kPCols);
  p.flush = flush < 2 ? 2 : (flush & ~1);
  p.center = (center && !bf16) ? 1 : 0;
  p.in_bf16 = bf16 ? 1 : 0;
  p.cref_rows = n < kGramCenterRows ? n : kGramCenterRows;
  p.cref = G + static_cast<int64_t>(n - p.cref_rows) * ld;
  p.cref_ld = ld;
  p.d = d;
  p.parts = parts;
  p.G = G; p.ld = ld;
  p.cvec = cvec;
  if (p.center) {
    const int64_t d_pad = (d + kPCols - 1) / kPCols * kPCols;
    pair_center_kernel<<<static_cast<unsigned>((d_pad / 4 + 255) / 256), 256, 0, stream>>>(p.cref, p.cref_rows, ld, d, d_pad, cvec);
    AFL_LAUNCH_CHECK("pair_center_kernel");
  }
  CUtensorMap tmap;
  const cuuint64_t gdim[2] = {static_cast<cuuint64_t>(d), static_cast<cuuint64_t>(n)};
  const cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * (bf16 ? 2 : 4)};
  const cuuint32_t box[2] = {kPCols, 128};
  const cuuint32_t estride[2] = {1, 1};
  CUresult r = enc(&tmap, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(Gv), gdim,
                   gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE, bf16 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed: %d", static_cast<int>(r)); return AFL_ERR_CUDA; }
  const size_t smem = static_cast<size_t>(kPSlots) * kPSlotBytes + 1024;
  static int smem_attr_done[kMaxDevices] = {0};
  AFL_CUDA(ensure_dyn_smem(gram_pair_kernel, static_cast<int>(smem), smem_attr_done));
  {
    ProfScope ps("gram_pair", stream);
    gram_pair_kernel<<<p.pairs * p.splits, kPThreads, smem, stream>>>(tmap, p);
  }
  AFL_LAUNCH_CHECK("gram_pair_kernel");
  pair_reduce_kernel<<<dim3(n, p.tiles), dim3(128, kPSy), 0, stream>>>(parts, n, p.splits, S);
  AFL_LAUNCH_CHECK("pair_reduce_kernel");
  pair_to_sqdist_kernel<<<dim3((n + 127) / 128, n), 128, 0, stream>>>(S, n, d2_out);
  AFL_LAUNCH_CHECK("pair_to_sqdist_kernel");
  return AFL_OK;
}

}  // namespace gram
}  // namespace afl
