// match.cu — exhaustive putative matching of 128-D uint8 SIFT descriptors on sm_100a.
//
// Replaces (reference, /root/reference/src/openMVG):
//   matching_image_collection/Matcher_Regions.cpp:32-107   pair loop (BRUTE_FORCE_L2)
//   matching/regions_matcher.hpp:162-207                   MatchDistanceRatio
//   matching/matcher_brute_force.hpp:100-200               2-NN scan (L2<uint8_t>, metric.hpp:55-93)
//   matching/matching_filters.hpp:38-60                    NNdistanceRatio
//
// Design (DESIGN.md §MATCH):
//   |q - b|^2 = |q|^2 + |b|^2 - 2 q.b.   q.b for a 128-query x 256-database tile is ONE dense
//   u8 x u8 -> s32 contraction with K = 128: four tcgen05.mma.kind::i8 (M128 N256 K32) fed by TMA
//   (128-byte rows, SWIZZLE_128B), accumulators in TMEM (2 x 256 columns, double buffered).
//   Epilogue (8 warps): key = 512*dot + ckey[b], ckey[b] = -256*|b|^2 + (b / G)  — one IMAD gives
//   ((2 q.b - |b|^2) << 8) | group(b); the running MAX of the key over a 32-column chunk is one
//   max per element, and a top-2 over chunk maxima costs 3 ops per 32 elements.  The kernel thus
//   emits, per query, the exact best key (=> exact d1 and the 32..G-row group holding the nearest
//   neighbour) and the best key of any OTHER chunk (=> an upper bound ub2 >= d2 that is exact
//   whenever the second neighbour lies outside the best chunk).  A finalize kernel re-scans the one
//   group exactly (dp4a) only for queries that can still pass the ratio test with ub2, recovers
//   (i1, d2) exactly, applies  float(d1) < fratio*float(d2)  and compacts in ascending query order.
//   All integer arithmetic is exact, so the output is bit-identical to the reference.
#include "common.cuh"
#include <cub/device/device_radix_sort.cuh>

#include <cuda.h>
#include <algorithm>
#include <climits>
#include <cstring>
#include <vector>

namespace omvg {

constexpr int TILE_Q = 128;      // UMMA M  (queries  -> TMEM lanes)
constexpr int TILE_DB = 256;     // UMMA N  (database -> TMEM columns)
constexpr int ROW_PAD = 256;     // every image starts at a multiple of this many arena rows
constexpr int A_STAGES = 2, B_STAGES = 4;
constexpr int A_BYTES = TILE_Q * OMVG_DESC_LEN;                 // 16 KB
constexpr int B_BYTES = TILE_DB * OMVG_DESC_LEN;                // 32 KB
constexpr int CK_BYTES = TILE_DB * 4;                           //  1 KB of packed keys
constexpr int B_STAGE_BYTES = B_BYTES + CK_BYTES;
constexpr int SMEM_BYTES = A_STAGES * A_BYTES + B_STAGES * B_STAGE_BYTES + 1024 /*align slack*/ + 2048 /*merge*/ + 256 /*barriers*/;
constexpr int TC_THREADS = 320;  // warp0 TMA, warp1 MMA, warps 2-5 / 6-9 epilogue for even / odd tiles
constexpr int KEY_MIN = INT_MIN;

struct Unit { uint32_t q_row, db_row, n_db_tiles, out_off; };   // one (pair, 128-query tile); n_db_tiles = tiles | (rows per group / 32) << 20
constexpr uint32_t UNIT_TILES_MASK = 0xFFFFFu;

// --------------------------------------------------------------------------------- prep kernel
// norm[r] = |row r|^2 ; ckey[r] = -256*norm + (local_row / G) for real rows, INT_MIN for padding.
__global__ void prep_rows_kernel(const uint8_t *__restrict__ desc, const uint32_t *__restrict__ img_row0,
                                 const uint32_t *__restrict__ img_count, const uint32_t *__restrict__ img_group,
                                 const uint32_t *__restrict__ row_img, int32_t *__restrict__ norm,
                                 int32_t *__restrict__ ckey, uint32_t total_rows) {
  const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;   // 8 threads per row, 16 B each
  const uint32_t sub = threadIdx.x & 7;
  if (gw >= total_rows) return;
  const uint4 v = reinterpret_cast<const uint4 *>(desc + (size_t)gw * OMVG_DESC_LEN)[sub];
  uint32_t s = __dp4a(v.x, v.x, 0u); s = __dp4a(v.y, v.y, s); s = __dp4a(v.z, v.z, s); s = __dp4a(v.w, v.w, s);
  s += __shfl_xor_sync(0xffffffffu, s, 1); s += __shfl_xor_sync(0xffffffffu, s, 2); s += __shfl_xor_sync(0xffffffffu, s, 4);
  if (sub == 0) {
    const uint32_t img = row_img[gw >> 8];                      // ROW_PAD == 256 rows per slot
    const uint32_t local = gw - img_row0[img];
    norm[gw] = (int32_t)s;
    ckey[gw] = local < img_count[img] ? (int32_t)(-(int32_t)(s << 8) + (int32_t)(local / img_group[img])) : KEY_MIN;
  }
}

// --------------------------------------------------------------------------------- tcgen05 kernel
__device__ __forceinline__ void tmem_ld_wait_dep(int32_t (&r)[32]) {
  // tcgen05.wait::ld, with the 32 registers as in/out operands so that no use of them can be
  // scheduled above the wait.
  asm volatile("tcgen05.wait::ld.sync.aligned;"
    : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
      "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
      "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
      "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
    :: "memory");
}

__device__ __forceinline__ int4 lds128(uint32_t saddr) {
  int4 v;
  asm("ld.shared.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
  return v;
}

__device__ __forceinline__ void chunk_update(const int32_t (&r)[32], uint32_t ck, int &k1, int &k2) {
  // four independent max chains (ILP) instead of one 16-deep dependent chain
  int g0 = KEY_MIN, g1 = KEY_MIN, g2 = KEY_MIN, g3 = KEY_MIN;
  #pragma unroll
  for (int j = 0; j < 8; j += 2) {
    const int4 c = lds128(ck + 16 * j);                          // LDS.128, same address for all lanes (broadcast)
    const int4 d = lds128(ck + 16 * j + 16);
    g0 = max(max(g0, r[4 * j + 0] * 512 + c.x), r[4 * j + 1] * 512 + c.y);
    g1 = max(max(g1, r[4 * j + 2] * 512 + c.z), r[4 * j + 3] * 512 + c.w);
    g2 = max(max(g2, r[4 * j + 4] * 512 + d.x), r[4 * j + 5] * 512 + d.y);
    g3 = max(max(g3, r[4 * j + 6] * 512 + d.z), r[4 * j + 7] * 512 + d.w);
  }
  const int gm = max(max(g0, g1), max(g2, g3));
  k2 = max(k2, min(k1, gm));
  k1 = max(k1, gm);
}

__global__ void __launch_bounds__(TC_THREADS, 1)
match_tc_kernel(const __grid_constant__ CUtensorMap tmap, const int32_t *__restrict__ ckey,
                const Unit *__restrict__ units, uint32_t n_units, int2 *__restrict__ k12) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t *a_smem = smem;                                        // [A_STAGES][16 KB]
  uint8_t *b_smem = smem + A_STAGES * A_BYTES;                   // [B_STAGES][32 KB + 1 KB]
  int2 *merge = reinterpret_cast<int2 *>(b_smem + B_STAGES * B_STAGE_BYTES);   // [2][128]
  uint64_t *bars = reinterpret_cast<uint64_t *>(merge + 2 * TILE_Q);
  uint64_t *full_a = bars, *empty_a = bars + 2, *full_b = bars + 4, *empty_b = bars + 8;
  uint64_t *tmem_full = bars + 12, *tmem_empty = bars + 14;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 16);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap);
    for (int i = 0; i < A_STAGES; ++i) { mbar_init(&full_a[i], 1); mbar_init(&empty_a[i], 1); }
    for (int i = 0; i < B_STAGES; ++i) { mbar_init(&full_b[i], 1); mbar_init(&empty_b[i], 1 + 4); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 4); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================================================================== TMA producer
    if (lane == 0) {
      uint32_t g = 0, ul = 0;
      for (uint32_t u = blockIdx.x; u < n_units; u += gridDim.x, ++ul) {
        const Unit un = units[u];
        const uint32_t as = ul & 1;
        mbar_wait(&empty_a[as], ((ul >> 1) & 1) ^ 1);
        mbar_arrive_expect_tx(&full_a[as], A_BYTES);
        tma_load_2d(a_smem + as * A_BYTES, &tmap, 0, (int)un.q_row, &full_a[as]);
        for (uint32_t t = 0; t < (un.n_db_tiles & UNIT_TILES_MASK); ++t, ++g) {
          const uint32_t st = g % B_STAGES;
          mbar_wait(&empty_b[st], ((g / B_STAGES) & 1) ^ 1);
          mbar_arrive_expect_tx(&full_b[st], B_STAGE_BYTES);
          uint8_t *dst = b_smem + st * B_STAGE_BYTES;
          const uint32_t row = un.db_row + t * TILE_DB;
          tma_load_2d(dst, &tmap, 0, (int)row, &full_b[st]);
          tma_load_2d(dst + A_BYTES, &tmap, 0, (int)(row + 128), &full_b[st]);
          bulk_load_1d(dst + B_BYTES, ckey + row, CK_BYTES, &full_b[st]);
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_u8(TILE_Q, TILE_DB);
      uint32_t g = 0, ul = 0;
      for (uint32_t u = blockIdx.x; u < n_units; u += gridDim.x, ++ul) {
        const uint32_t n_tiles = units[u].n_db_tiles & UNIT_TILES_MASK;
        const uint32_t as = ul & 1;
        mbar_wait(&full_a[as], (ul >> 1) & 1);
        const uint32_t a_addr = smem_u32(a_smem + as * A_BYTES);
        for (uint32_t t = 0; t < n_tiles; ++t, ++g) {
          const uint32_t st = g % B_STAGES, acc = g & 1;
          mbar_wait(&full_b[st], (g / B_STAGES) & 1);
          mbar_wait(&tmem_empty[acc], ((g >> 1) & 1) ^ 1);
          tc_fence_after();
          const uint32_t b_addr = smem_u32(b_smem + st * B_STAGE_BYTES);
          const uint32_t d = tmem_base + acc * TILE_DB;
          #pragma unroll
          for (int k = 0; k < OMVG_DESC_LEN / 32; ++k)
            umma_i8(d, make_kmajor_sw128_desc(a_addr + k * 32), make_kmajor_sw128_desc(b_addr + k * 32), idesc, k > 0);
          tc_commit(&empty_b[st]);
          tc_commit(&tmem_full[acc]);
        }
        tc_commit(&empty_a[as]);
      }
    }
  } else {
    // ===================================================================== epilogue (8 warps)
    const uint32_t wg = (warp - 2) >> 2;                 // 0: even tiles / acc 0, 1: odd tiles / acc 1
    const uint32_t quarter = warp & 3;                   // TMEM lane quarter this warp may access
    const uint32_t row_in_tile = quarter * 32 + lane;
    uint32_t g = 0, ul = 0;
    for (uint32_t u = blockIdx.x; u < n_units; u += gridDim.x, ++ul) {
      const Unit un = units[u];
      int k1 = KEY_MIN, k2 = KEY_MIN;
      for (uint32_t t = 0; t < (un.n_db_tiles & UNIT_TILES_MASK); ++t, ++g) {
        if ((g & 1) != wg) continue;
        const uint32_t st = g % B_STAGES, acc = wg;
        mbar_wait(&full_b[st], (g / B_STAGES) & 1);      // packed keys of this tile are in smem
        mbar_wait(&tmem_full[acc], (g >> 1) & 1);        // accumulator complete
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((quarter * 32) << 16) + acc * TILE_DB;
        const uint32_t ck = smem_u32(b_smem + st * B_STAGE_BYTES + B_BYTES);
        int32_t ra[32], rb[32];
        tmem_ld_32x32(taddr, ra);
        #pragma unroll
        for (int c = 0; c < TILE_DB / 32; c += 2) {
          tmem_ld_wait_dep(ra);
          tmem_ld_32x32(taddr + (c + 1) * 32, rb);
          chunk_update(ra, ck + c * 128, k1, k2);
          tmem_ld_wait_dep(rb);
          if (c + 2 < TILE_DB / 32) tmem_ld_32x32(taddr + (c + 2) * 32, ra);
          chunk_update(rb, ck + (c + 1) * 128, k1, k2);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) { mbar_arrive(&tmem_empty[acc]); mbar_arrive(&empty_b[st]); }
      }
      // merge the two warpgroups' partial top-2 (disjoint chunks) and store
      int2 *mb = merge + (ul & 1) * TILE_Q;
      if (wg == 1) mb[row_in_tile] = make_int2(k1, k2);
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (wg == 0) {
        const int2 o = mb[row_in_tile];
        const int K1 = max(k1, o.x);
        const int K2 = max(min(k1, o.x), max(k2, o.y));
        k12[(size_t)un.out_off + row_in_tile] = make_int2(K1, K2);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, 512);
}


// --------------------------------------------------------------------------------- tcgen05 kernel, fifth K-slice
// The shipped kernel (match_dig2_kernel below).  match_tc_kernel above spends 1 IMAD per accumulator on
// key = 512*dot + ckey[column]; here the per-column constant rides in the MMA instead: a fifth K=32 slice multiplies a
// CONSTANT A tile (weights 1, 255 x 15, 1, 255 x 15 in every row) with 32 signed "digits" per database row (u8 x s8,
// its own instruction descriptor) so that the accumulator is   acc = q.b - h(b) + c0(image),  h = ceil(|b|^2 / 2).
// The epilogue is then a pure running max (VIMNMX3: half an instruction per accumulator) and ONE key per 32-column
// chunk, key = 256 * max + group.  What is lost is the parity of |b|^2:  2 q.b - |b|^2 = 2 acc - 2 c0 + p, p in
// {0, 1}; the finalize kernel works with the two-sided bound and falls back to an exact scan of the whole database
// image in the (rare) cases where the one unit matters — see match_finalize_kernel<true>.  Padding rows carry the
// most negative digit vector (DIG_PAD), strictly below every real column, and zero descriptors.
// Digit range: v = c0 - h must lie in [DIG_VMIN, DIG_VMAX]; omvg_match_prepare picks c0 per image and uses this
// kernel only if every image fits (|b|^2 spread <= 3.9 M inside an image: always true for SIFT, whose |b|^2 is
// ~2.6e5); otherwise match_tc_kernel runs.
constexpr int DIG_LEN = 32;
constexpr int DG_BYTES = TILE_DB * DIG_LEN;                      //  8 KB of digits per database tile
constexpr int B5_STAGE_BYTES = B_BYTES + DG_BYTES;               // 40 KB
constexpr int ACONST_BYTES = TILE_Q * DIG_LEN;                   //  4 KB
constexpr int DIG_PAD = -128 * 2 - 128 * 255 * 30;               // -979456: all 32 digits = -128
constexpr int DIG_VMIN = -979328, DIG_VMAX = 971676;             // v = d0 + 255 M, d0 in [-128, 126], M in [-3840, 3810]
constexpr int DIG_SPREAD_MAX = DIG_VMAX - DIG_VMIN;              // 1 951 004 (in units of h)

// per-image min / max of h = ceil(|row|^2 / 2) over the real rows (one block per image)
__global__ void prep_minmax_kernel(const int32_t *__restrict__ norm, const uint32_t *__restrict__ img_row0,
                                   const uint32_t *__restrict__ img_count, int2 *__restrict__ out) {
  __shared__ int smin[8], smax[8];
  const uint32_t img = blockIdx.x, r0 = img_row0[img], n = img_count[img];
  int lo = INT_MAX, hi = INT_MIN;
  for (uint32_t r = threadIdx.x; r < n; r += blockDim.x) { const int h = (norm[r0 + r] + 1) >> 1; lo = min(lo, h); hi = max(hi, h); }
  #pragma unroll
  for (int off = 16; off > 0; off >>= 1) { lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, off)); hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, off)); }
  if ((threadIdx.x & 31) == 0) { smin[threadIdx.x >> 5] = lo; smax[threadIdx.x >> 5] = hi; }
  __syncthreads();
  if (threadIdx.x == 0) { for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { lo = min(lo, smin[w]); hi = max(hi, smax[w]); } out[img] = make_int2(lo, hi); }
}

// digits of v = c0 - h for real rows, all -128 for padding rows.  Byte 0 and byte 16 have weight 1, the others 255.
__global__ void prep_digits_kernel(const int32_t *__restrict__ norm, const uint32_t *__restrict__ img_row0,
                                   const uint32_t *__restrict__ img_count, const uint32_t *__restrict__ row_img,
                                   const int32_t *__restrict__ img_c0, uint4 *__restrict__ dig, uint32_t total_rows) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= total_rows) return;
  const uint32_t img = row_img[r >> 8], local = r - img_row0[img];
  uint32_t w[8];
  if (local < img_count[img]) {
    const int v = img_c0[img] - ((norm[r] + 1) >> 1);
    int M = (v + 128) / 255; if ((v + 128) - M * 255 < 0) --M;                // floor division
    const int d0 = v - 255 * M;                                               // [-128, 126]
    int qd = M / 30; if (M - qd * 30 < 0) --qd;
    const int rem = M - qd * 30;                                              // [0, 29]
    #pragma unroll
    for (int i = 0; i < 8; ++i) {
      uint32_t word = 0;
      #pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int pos = 4 * i + b;
        int d;
        if (pos == 0) d = d0; else if (pos == 16) d = 0;
        else { const int k = pos < 16 ? pos - 1 : pos - 2; d = qd + (k < rem ? 1 : 0); }
        word |= (uint32_t)(d & 255) << (8 * b);
      }
      w[i] = word;
    }
  } else {
    #pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = 0x80808080u;
  }
  dig[2 * (size_t)r] = make_uint4(w[0], w[1], w[2], w[3]);
  dig[2 * (size_t)r + 1] = make_uint4(w[4], w[5], w[6], w[7]);
}

__device__ __forceinline__ void chunk_max(const int32_t (&r)[32], int gid, int &k1, int &k2) {
  int g0 = max(max(r[0], r[1]), r[2]), g1 = max(max(r[8], r[9]), r[10]), g2 = max(max(r[16], r[17]), r[18]), g3 = max(max(r[24], r[25]), r[26]);
  g0 = max(max(g0, r[3]), r[4]); g1 = max(max(g1, r[11]), r[12]); g2 = max(max(g2, r[19]), r[20]); g3 = max(max(g3, r[27]), r[28]);
  g0 = max(max(g0, r[5]), r[6]); g1 = max(max(g1, r[13]), r[14]); g2 = max(max(g2, r[21]), r[22]); g3 = max(max(g3, r[29]), r[30]);
  const int gm = max(max(max(g0, r[7]), max(g1, r[15])), max(max(g2, r[23]), max(g3, r[31])));
  const int key = gm * 256 + gid;
  k2 = max(k2, min(k1, key));
  k1 = max(k1, key);
}

// K-major operand tile of 32-byte rows under the 32-byte swizzle (TMA SWIZZLE_32B): 8-row x 32-B atoms, SBO 256 B.
__device__ __forceinline__ uint64_t make_kmajor_sw32_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(256 >> 4) << 32;                     // SBO
  d |= (uint64_t)1 << 46;                              // descriptor version (Blackwell)
  d |= (uint64_t)6 << 61;                              // SWIZZLE_32B
  return d;
}

// --------------------------------------------------------------------------------- two query tiles per database tile
// Streaming the whole database image through a CTA once per 128 queries costs 40 KB per 640 tensor cycles and SM =
// 18 TB/s of L2 -> SM traffic at full rate, which the L2 does not deliver (such a TMA + MMA skeleton WITHOUT any
// epilogue runs at 61-69 % tensor pipe).  So one CTA keeps TWO query tiles (256 queries) resident and multiplies both
// with every database tile it loads: accumulator 0 = queries 0-127, accumulator 1 = queries 128-255, which are at the
// same time the two halves of the TMEM double buffer (the epilogue of accumulator 0 runs under the MMAs of accumulator
// 1 and vice versa).  NSPLIT = 2 epilogue warps per TMEM lane quarter and accumulator, each draining half the columns.
constexpr int A2_BYTES = 2 * A_BYTES;                            // 32 KB: two query tiles
constexpr int B2_STAGES = 3;
constexpr int NSPLIT = 2;
constexpr int DIG2_THREADS = 64 + 256 * NSPLIT;                  // TMA warp, MMA warp, 8 * NSPLIT epilogue warps
constexpr int DIG2_SMEM_BYTES = A_STAGES * A2_BYTES + B2_STAGES * B5_STAGE_BYTES + ACONST_BYTES + 1024 /*align slack*/ + 2 * 2 * TILE_Q * 8 /*merge*/ + 256 /*barriers*/;
constexpr uint32_t UNIT_TWO = 0x80000000u;                       // Unit.n_db_tiles bit 31: the super-tile has a second query tile

__global__ void __launch_bounds__(DIG2_THREADS, 1)
match_dig2_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_dig,
                  const Unit *__restrict__ units, uint32_t n_units, int2 *__restrict__ k12) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t *a_smem = smem;                                        // [A_STAGES][2 x 16 KB]
  uint8_t *b_smem = smem + A_STAGES * A2_BYTES;                  // [B2_STAGES][32 KB descriptors + 8 KB digits]
  uint8_t *aconst = b_smem + B2_STAGES * B5_STAGE_BYTES;         // [128][32 B] constant weights
  int2 *merge = reinterpret_cast<int2 *>(aconst + ACONST_BYTES); // [2 accumulators][2][128]
  uint64_t *bars = reinterpret_cast<uint64_t *>(merge + 2 * 2 * TILE_Q);
  uint64_t *full_a = bars, *empty_a = bars + 2, *full_b = bars + 4, *empty_b = bars + 8;
  uint64_t *tmem_full = bars + 12, *tmem_empty = bars + 14;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 16);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap); prefetch_tmap(&tmap_dig);
    for (int i = 0; i < A_STAGES; ++i) { mbar_init(&full_a[i], 1); mbar_init(&empty_a[i], 1); }
    for (int i = 0; i < B2_STAGES; ++i) { mbar_init(&full_b[i], 1); mbar_init(&empty_b[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 4 * NSPLIT); }
    fence_barrier_init();
  }
  for (int i = threadIdx.x; i < ACONST_BYTES / 16; i += blockDim.x)
    reinterpret_cast<uint4 *>(aconst)[i] = make_uint4(0xFFFFFF01u, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
  fence_proxy_async();
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================================================================== TMA producer
    if (lane == 0) {
      uint32_t g = 0, ul = 0;
      for (uint32_t u = blockIdx.x; u < n_units; u += gridDim.x, ++ul) {
        const Unit un = units[u];
        const uint32_t as = ul & 1, n_tiles = un.n_db_tiles & UNIT_TILES_MASK;
        const bool two = (un.n_db_tiles & UNIT_TWO) != 0;
        mbar_wait(&empty_a[as], ((ul >> 1) & 1) ^ 1);
        mbar_arrive_expect_tx(&full_a[as], two ? A2_BYTES : A_BYTES);
        tma_load_2d(a_smem + as * A2_BYTES, &tmap, 0, (int)un.q_row, &full_a[as]);
        if (two) tma_load_2d(a_smem + as * A2_BYTES + A_BYTES, &tmap, 0, (int)(un.q_row + TILE_Q), &full_a[as]);
        for (uint32_t t = 0; t < n_tiles; ++t, ++g) {
          const uint32_t st = g % B2_STAGES;
          mbar_wait(&empty_b[st], ((g / B2_STAGES) & 1) ^ 1);
          mbar_arrive_expect_tx(&full_b[st], B5_STAGE_BYTES);
          uint8_t *dst = b_smem + st * B5_STAGE_BYTES;
          const uint32_t row = un.db_row + t * TILE_DB;
          tma_load_2d(dst, &tmap, 0, (int)row, &full_b[st]);
          tma_load_2d(dst + A_BYTES, &tmap, 0, (int)(row + 128), &full_b[st]);
          tma_load_2d(dst + B_BYTES, &tmap_dig, 0, (int)row, &full_b[st]);
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_u8(TILE_Q, TILE_DB);
      constexpr uint32_t idesc5 = idesc | (1u << 10);             // B operand signed: u8 weights x s8 digits
      const uint64_t ac_desc = make_kmajor_sw32_desc(smem_u32(aconst));
      uint32_t g = 0, ul = 0, cnt[2] = {0, 0};                    // cnt[h]: accumulations issued into accumulator h
      for (uint32_t u = blockIdx.x; u < n_units; u += gridDim.x, ++ul) {
        const uint32_t ndt = units[u].n_db_tiles;
        const uint32_t n_tiles = ndt & UNIT_TILES_MASK, nh = (ndt & UNIT_TWO) ? 2u : 1u;
        const uint32_t as = ul & 1;
        mbar_wait(&full_a[as], (ul >> 1) & 1);
        const uint32_t a_addr = smem_u32(a_smem + as * A2_BYTES);
        for (uint32_t t = 0; t < n_tiles; ++t, ++g) {
          const uint32_t st = g % B2_STAGES;
          mbar_wait(&full_b[st], (g / B2_STAGES) & 1);
          const uint32_t b_addr = smem_u32(b_smem + st * B5_STAGE_BYTES);
          const uint64_t dg_desc = make_kmajor_sw32_desc(b_addr + B_BYTES);
          for (uint32_t h = 0; h < nh; ++h) {
            mbar_wait(&tmem_empty[h], (cnt[h] & 1) ^ 1);
            tc_fence_after();
            const uint32_t d = tmem_base + h * TILE_DB;
            #pragma unroll
            for (int k = 0; k < OMVG_DESC_LEN / 32; ++k)
              umma_i8(d, make_kmajor_sw128_desc(a_addr + h * A_BYTES + k * 32), make_kmajor_sw128_desc(b_addr + k * 32), idesc, k > 0);
            umma_i8(d, ac_desc, dg_desc, idesc5, 1);
            tc_commit(&tmem_full[h]);
            ++cnt[h];
          }
          tc_commit(&empty_b[st]);
        }
        tc_commit(&empty_a[as]);
      }
    }
  } else {
    // ===================================================================== epilogue (8 * NSPLIT warps)
    const uint32_t e = warp - 2;
    const uint32_t wg = e / (4 * NSPLIT);                 // accumulator = query tile (0: rows 0-127, 1: rows 128-255)
    const uint32_t part = (e % (4 * NSPLIT)) >> 2;        // which 256/NSPLIT-column part of the accumulator
    const uint32_t quarter = warp & 3;                    // TMEM lane quarter this warp may access
    const uint32_t row_in_tile = quarter * 32 + lane;
    constexpr uint32_t NCH = 8 / NSPLIT;                  // 32-column chunks per warp and tile
    const uint32_t c0 = part * NCH;
    uint32_t cnt = 0, um = 0;                             // accumulations consumed from this accumulator; units merged
    for (uint32_t u = blockIdx.x; u < n_units; u += gridDim.x) {
      const Unit un = units[u];
      if (wg == 1 && !(un.n_db_tiles & UNIT_TWO)) continue;
      const uint32_t n_tiles = un.n_db_tiles & UNIT_TILES_MASK, gdiv = (un.n_db_tiles >> 20) & 0x7FFu;
      int k1 = KEY_MIN, k2 = KEY_MIN;
      for (uint32_t t = 0; t < n_tiles; ++t, ++cnt) {
        mbar_wait(&tmem_full[wg], cnt & 1);               // accumulator complete
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((quarter * 32) << 16) + wg * TILE_DB + c0 * 32;
        const uint32_t chunk0 = t * 8 + c0;
        int32_t ra[32], rb[32];
        tmem_ld_32x32(taddr, ra);
        #pragma unroll
        for (uint32_t c = 0; c < NCH; c += 2) {
          tmem_ld_wait_dep(ra);
          tmem_ld_32x32(taddr + (c + 1) * 32, rb);
          chunk_max(ra, (int)(gdiv <= 1 ? chunk0 + c : (chunk0 + c) / gdiv), k1, k2);
          tmem_ld_wait_dep(rb);
          if (c + 2 < NCH) tmem_ld_32x32(taddr + (c + 2) * 32, ra);
          else {                                             // every column of the accumulator is in registers: hand it back
            tc_fence_before();                               // to the MMA warp before the arithmetic of the last chunk
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[wg]);
          }
          chunk_max(rb, (int)(gdiv <= 1 ? chunk0 + c + 1 : (chunk0 + c + 1) / gdiv), k1, k2);
        }
      }
      // merge the two column parts of this accumulator
      int2 *mb = merge + (wg * 2 + (um & 1)) * TILE_Q; ++um;
      if (part) mb[row_in_tile] = make_int2(k1, k2);
      if (wg == 0) asm volatile("bar.sync 1, 256;" ::: "memory"); else asm volatile("bar.sync 2, 256;" ::: "memory");
      if (part == 0) { const int2 o = mb[row_in_tile]; const int lo = min(k1, o.x); k1 = max(k1, o.x); k2 = max(lo, max(k2, o.y)); }
      if (part == 0) k12[(size_t)un.out_off + wg * TILE_Q + row_in_tile] = make_int2(k1, k2);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, 512);
}


// --------------------------------------------------------------------------------- finalize
struct PairInfo { uint32_t db_row0, db_count, db_group, q_row0, q_count; uint32_t unit0; uint64_t out_off; int32_t db_c0; int32_t pad_; };

// expand the per-pair table into the (pair, 128-query tile) work units on the device (one block per pair)
// q_tiles = 1 (match_tc_kernel): one unit per 128 queries; q_tiles = 2 (match_dig2_kernel): one unit per 256 queries,
// UNIT_TWO set when the second query tile holds real rows
__global__ void expand_units_kernel(const PairInfo *__restrict__ pairs, Unit *__restrict__ units, uint32_t q_tiles) {
  const PairInfo P = pairs[blockIdx.x];
  const uint32_t rows = TILE_Q * q_tiles;
  const uint32_t qt = (P.q_count + rows - 1) / rows, dt = (P.db_count + TILE_DB - 1) / TILE_DB;
  for (uint32_t t = threadIdx.x; t < qt; t += blockDim.x) {
    uint32_t flags = 0;
    if (q_tiles == 2 && P.q_count - t * rows > TILE_Q) flags = UNIT_TWO;
    units[P.unit0 + t] = Unit{P.q_row0 + t * rows, P.db_row0, dt | ((P.db_group / 32) << 20) | flags, (uint32_t)(P.out_off + t * rows)};
  }
}

// exact top-2 of one query inside rows [r0, r1) of the database; whole warp cooperates.
__device__ __forceinline__ void warp_rescan(const uint8_t *__restrict__ desc, const int32_t *__restrict__ norm,
                                            uint32_t q_row, uint32_t r0, uint32_t r1, uint32_t db_row0,
                                            int lane, int &bd1, uint32_t &bi1, int &bd2) {
  const uint32_t qword = reinterpret_cast<const uint32_t *>(desc + (size_t)q_row * OMVG_DESC_LEN)[lane];
  const int qn = norm[q_row];
  int d1 = INT_MAX, d2 = INT_MAX; uint32_t i1 = 0xffffffffu;
  for (uint32_t base = r0; base < r1; base += 32) {              // uniform trip count for the shuffles
    const uint32_t r = base + lane;
    const bool ok = r < r1;
    const uint4 *rp = reinterpret_cast<const uint4 *>(desc + (size_t)(ok ? r : r0) * OMVG_DESC_LEN);
    uint32_t dot = 0;
    #pragma unroll
    for (int k = 0; k < 8; ++k) {
      const uint4 v = rp[k];
      dot = __dp4a(v.x, __shfl_sync(0xffffffffu, qword, 4 * k + 0), dot);
      dot = __dp4a(v.y, __shfl_sync(0xffffffffu, qword, 4 * k + 1), dot);
      dot = __dp4a(v.z, __shfl_sync(0xffffffffu, qword, 4 * k + 2), dot);
      dot = __dp4a(v.w, __shfl_sync(0xffffffffu, qword, 4 * k + 3), dot);
    }
    if (ok) {
      const int d = qn + norm[r] - 2 * (int)dot;
      if (d < d1) { d2 = d1; d1 = d; i1 = r - db_row0; } else if (d < d2) d2 = d;
    }
  }
  #pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const int od1 = __shfl_xor_sync(0xffffffffu, d1, off), od2 = __shfl_xor_sync(0xffffffffu, d2, off);
    const uint32_t oi1 = __shfl_xor_sync(0xffffffffu, i1, off);
    if (od1 < d1 || (od1 == d1 && oi1 < i1)) { d2 = min(od2, d1); d1 = od1; i1 = oi1; }
    else d2 = min(d2, od1);
  }
  bd1 = d1; bi1 = i1; bd2 = d2;
}

constexpr int FIN_THREADS = 256;
// DIG = false: keys of match_tc_kernel (exact d1, exact bound ub2).
// DIG = true : keys of match_dig2_kernel.  A = key >> 8 is the chunk maximum of acc = q.b - h + c0, so the best column
// of that chunk has distance  D - 1 or D,  D = |q|^2 - 2 A + 2 c0  (parity of |b|^2 unknown).  Then
//   * A1 > A2: the nearest neighbour lies in the chunk (group) of A1 — every other column has acc <= A2 <= A1 - 1, i.e.
//     distance >= D1 + 1; its exact distance and index come from the group re-scan as before.
//   * A1 == A2: two chunks tie to within the parity -> exact scan of the whole database image for this query.
//   * the best column outside the group bounds d2 from above by D2 and the truth is D2 - 1 or D2; if the ratio test
//     gives the same answer for both, that is the answer, otherwise -> exact scan of the whole image.
//   * candidates are pre-filtered with the weakest case (d1 >= D1 - 1, d2 <= D2); float() and the multiplication by a
//     non-negative constant are monotone, so nothing that could pass is dropped.
// Chunks that hold only padding have A == DIG_PAD (never reached by a real column): "no second chunk".
template <bool DIG>
__global__ void __launch_bounds__(FIN_THREADS)
match_finalize_kernel(const uint8_t *__restrict__ desc, const int32_t *__restrict__ norm,
                      const PairInfo *__restrict__ pairs, int2 *__restrict__ k12, uint32_t *__restrict__ counts,
                      float fratio) {
  __shared__ uint32_t warp_tot[FIN_THREADS / 32];
  __shared__ uint32_t running;
  const PairInfo P = pairs[blockIdx.x];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) running = 0;
  __syncthreads();
  int2 *io = k12 + P.out_off;
  for (uint32_t q0 = 0; q0 < P.q_count; q0 += FIN_THREADS) {
    const uint32_t q = q0 + threadIdx.x;
    const bool valid = q < P.q_count;
    int ub2 = 0, lo2 = 0; uint32_t g1 = 0; bool cand = false, full = false;
    if (valid) {
      const int2 K = io[q];
      const int qn = norm[P.q_row0 + q];
      g1 = (uint32_t)(K.x & 255);
      if (!DIG) {
        const int d1 = qn - (K.x >> 8);
        ub2 = (K.y == KEY_MIN) ? INT_MAX : qn - (K.y >> 8);
        lo2 = ub2;
        cand = __int2float_rn(d1) < __fmul_rn(fratio, __int2float_rn(ub2));
      } else {
        const int A1 = K.x >> 8, A2 = K.y >> 8;
        const int D1 = qn - 2 * A1 + 2 * P.db_c0;
        const bool none2 = A2 <= DIG_PAD;
        ub2 = none2 ? INT_MAX : qn - 2 * A2 + 2 * P.db_c0;
        lo2 = none2 ? INT_MAX : ub2 - 1;
        cand = __int2float_rn(max(D1 - 1, 0)) < __fmul_rn(fratio, __int2float_rn(ub2));
        full = cand && !none2 && A1 == A2;
      }
    }
    bool keep = false; uint32_t idx = 0;
    uint32_t m = __ballot_sync(0xffffffffu, cand && !full);
    while (m) {
      const int src = __ffs(m) - 1; m &= m - 1;
      const uint32_t qq = __shfl_sync(0xffffffffu, q, src);
      const uint32_t gg = __shfl_sync(0xffffffffu, g1, src);
      const uint32_t r0 = P.db_row0 + gg * P.db_group;
      const uint32_t r1 = min(r0 + P.db_group, P.db_row0 + P.db_count);
      int bd1, bd2; uint32_t bi1;
      warp_rescan(desc, norm, P.q_row0 + qq, r0, r1, P.db_row0, lane, bd1, bi1, bd2);
      if (lane == src) {
        const bool k_hi = __int2float_rn(bd1) < __fmul_rn(fratio, __int2float_rn(min(ub2, bd2)));   // matching_filters.hpp:57
        const bool k_lo = __int2float_rn(bd1) < __fmul_rn(fratio, __int2float_rn(min(lo2, bd2)));
        if (k_hi == k_lo) keep = k_hi; else full = true;
        idx = bi1;
      }
    }
    if (DIG) {                                          // exact scan of the whole database image (rare)
      m = __ballot_sync(0xffffffffu, full);
      while (m) {
        const int src = __ffs(m) - 1; m &= m - 1;
        const uint32_t qq = __shfl_sync(0xffffffffu, q, src);
        int bd1, bd2; uint32_t bi1;
        warp_rescan(desc, norm, P.q_row0 + qq, P.db_row0, P.db_row0 + P.db_count, P.db_row0, lane, bd1, bi1, bd2);
        if (lane == src) { keep = __int2float_rn(bd1) < __fmul_rn(fratio, __int2float_rn(bd2)); idx = bi1; }
      }
    }
    // ordered compaction (ascending q): block exclusive scan of keep
    const uint32_t bal = __ballot_sync(0xffffffffu, keep);
    const uint32_t in_warp = __popc(bal & ((1u << lane) - 1));
    if (lane == 0) warp_tot[warp] = __popc(bal);
    __syncthreads();                                   // all reads of io[q0..] done, warp totals visible
    uint32_t before = running;
    for (int w = 0; w < warp; ++w) before += warp_tot[w];
    if (keep) reinterpret_cast<uint2 *>(io)[before + in_warp] = make_uint2(idx, q);
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t t = 0; for (int w = 0; w < FIN_THREADS / 32; ++w) t += warp_tot[w]; running += t; }
    __syncthreads();
  }
  if (threadIdx.x == 0) counts[blockIdx.x] = running;
}

// exclusive scan of per-pair counts of one batch, offset by *total_io (running total over batches)
__global__ void scan_counts_kernel(const uint32_t *__restrict__ counts, uint32_t n, uint64_t *__restrict__ offsets,
                                   uint64_t *__restrict__ total_io) {
  __shared__ uint64_t wsum[32];
  __shared__ uint64_t carry;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry = *total_io;
  __syncthreads();
  for (uint32_t base = 0; base < n; base += blockDim.x) {
    const uint32_t i = base + threadIdx.x;
    uint64_t v = i < n ? counts[i] : 0, x = v;
    #pragma unroll
    for (int off = 1; off < 32; off <<= 1) { const uint64_t y = __shfl_up_sync(0xffffffffu, x, off); if (lane >= off) x += y; }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    uint64_t pre = carry;
    for (int w = 0; w < warp; ++w) pre += wsum[w];
    if (i < n) offsets[i] = pre + x - v;
    __syncthreads();
    if (threadIdx.x == 0) { uint64_t t = 0; for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += wsum[w]; carry += t; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { offsets[n] = carry; *total_io = carry; }
}

__global__ void compact_kernel(const int2 *__restrict__ k12, const PairInfo *__restrict__ pairs,
                               const uint32_t *__restrict__ counts, const uint64_t *__restrict__ offsets,
                               uint2 *__restrict__ out) {
  const uint32_t p = blockIdx.x, n = counts[p];
  const uint2 *src = reinterpret_cast<const uint2 *>(k12 + pairs[p].out_off);
  uint2 *dst = out + offsets[p];
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
}

// --------------------------------------------------------------------------------- SIMT validation
// Exact 2-NN by brute force with dp4a; one block per query.  Tests only.
__global__ void __launch_bounds__(128)
top2_simt_kernel(const uint8_t *__restrict__ desc, const int32_t *__restrict__ norm, uint32_t db_row0,
                 uint32_t db_count, uint32_t q_row0, int32_t *__restrict__ od1, uint32_t *__restrict__ oi1,
                 int32_t *__restrict__ od2) {
  __shared__ uint32_t qs[32];
  __shared__ int sd1[128], sd2[128]; __shared__ uint32_t si1[128];
  const uint32_t q = blockIdx.x;
  if (threadIdx.x < 32) qs[threadIdx.x] = reinterpret_cast<const uint32_t *>(desc + (size_t)(q_row0 + q) * OMVG_DESC_LEN)[threadIdx.x];
  __syncthreads();
  const int qn = norm[q_row0 + q];
  int d1 = INT_MAX, d2 = INT_MAX; uint32_t i1 = 0xffffffffu;
  for (uint32_t r = threadIdx.x; r < db_count; r += blockDim.x) {
    const uint4 *rp = reinterpret_cast<const uint4 *>(desc + (size_t)(db_row0 + r) * OMVG_DESC_LEN);
    uint32_t dot = 0;
    #pragma unroll
    for (int k = 0; k < 8; ++k) { const uint4 v = rp[k];
      dot = __dp4a(v.x, qs[4 * k], dot); dot = __dp4a(v.y, qs[4 * k + 1], dot);
      dot = __dp4a(v.z, qs[4 * k + 2], dot); dot = __dp4a(v.w, qs[4 * k + 3], dot); }
    const int d = qn + norm[db_row0 + r] - 2 * (int)dot;
    if (d < d1) { d2 = d1; d1 = d; i1 = r; } else if (d < d2) d2 = d;
  }
  sd1[threadIdx.x] = d1; sd2[threadIdx.x] = d2; si1[threadIdx.x] = i1;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int t = 1; t < 128; ++t) {
      const int a1 = sd1[t], a2 = sd2[t]; const uint32_t ai = si1[t];
      if (a1 < d1 || (a1 == d1 && ai < i1)) { d2 = min(a2, d1); d1 = a1; i1 = ai; } else d2 = min(d2, a1);
    }
    od1[q] = d1; oi1[q] = i1; od2[q] = d2;
  }
}

__global__ void decode_k12_kernel(const int2 *__restrict__ k12, const int32_t *__restrict__ norm, uint32_t q_row0,
                                  uint32_t n, int32_t *d1, uint32_t *g1, int32_t *ub2) {
  const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n) return;
  const int2 K = k12[q]; const int qn = norm[q_row0 + q];
  d1[q] = qn - (K.x >> 8); g1[q] = (uint32_t)(K.x & 255);
  ub2[q] = (K.y == KEY_MIN) ? INT_MAX : qn - (K.y >> 8);
}


// ================================================================================= cascade hashing (M9 / N2)
// openMVG's default matcher for scalar descriptors (matching/cascade_hasher.hpp, Cascade_Hashing_Matcher_Regions.cpp):
// 128-bit sign code + 6 x 10-bit bucket ids per descriptor, candidates = union of the query's 6 buckets in the
// database image, first 10 by (Hamming, insertion order), exact L2 on those, top-2 by (distance, id), ratio test.
// Everything after the hashing is exact integer work; the hashing is a float mat-vec whose summation order is
// fixed here (k ascending, separate multiply and add); the CPU checker used by the tests mirrors it.
constexpr int CH_GROUPS = 6, CH_BITS = 10, CH_NB = 1 << CH_BITS, CH_OUT = OMVG_DESC_LEN + CH_GROUPS * CH_BITS, CH_TOP = 10;
constexpr int CH_HASH_THREADS = 192, CH_HASH_ROWS = 16;

// integer column sums of one image (exact): the float means are formed on the host from them
__global__ void cascade_colsum_kernel(const uint8_t *__restrict__ desc, const uint32_t *__restrict__ img_row0, const uint32_t *__restrict__ img_count,
                                      unsigned long long *__restrict__ sums) {
  const uint32_t img = blockIdx.x, k = threadIdx.x;
  const uint8_t *base = desc + (size_t)img_row0[img] * OMVG_DESC_LEN;
  unsigned long long s = 0;
  for (uint32_t r = 0; r < img_count[img]; ++r) s += base[(size_t)r * OMVG_DESC_LEN + k];
  sums[(size_t)img * OMVG_DESC_LEN + k] = s;
}

// code bit j = (P_j . (d - zm) > 0), bucket id of group g = 10 such signs of S_g, MSB first (cascade_hasher.hpp:203-232)
__global__ void __launch_bounds__(CH_HASH_THREADS) cascade_hash_kernel(const uint8_t *__restrict__ desc, uint32_t total_rows, const float *__restrict__ zm,
                                                                       const float *__restrict__ proj /*[188][128]: primary then secondary*/,
                                                                       uint4 *__restrict__ code, uint4 *__restrict__ bid) {
  __shared__ float sd[CH_HASH_ROWS][OMVG_DESC_LEN];
  __shared__ uint32_t sbid[CH_HASH_ROWS][8];
  __shared__ uint32_t scode[CH_HASH_ROWS][4];
  const uint32_t row0 = blockIdx.x * CH_HASH_ROWS, t = threadIdx.x;
  for (uint32_t idx = t; idx < CH_HASH_ROWS * OMVG_DESC_LEN; idx += CH_HASH_THREADS) {
    const uint32_t r = idx >> 7, k = idx & 127;
    sd[r][k] = row0 + r < total_rows ? __fsub_rn((float)desc[(size_t)(row0 + r) * OMVG_DESC_LEN + k], zm[k]) : 0.0f;
  }
  if (t < CH_HASH_ROWS * 8) sbid[t >> 3][t & 7] = 0;
  __syncthreads();
  if (t < CH_OUT) {
    const float *pr = proj + (size_t)t * OMVG_DESC_LEN;
    float acc[CH_HASH_ROWS];
    #pragma unroll
    for (int r = 0; r < CH_HASH_ROWS; ++r) acc[r] = 0.0f;
    for (int k = 0; k < OMVG_DESC_LEN; ++k) {
      const float pv = pr[k];
      #pragma unroll
      for (int r = 0; r < CH_HASH_ROWS; ++r) acc[r] = __fadd_rn(acc[r], __fmul_rn(pv, sd[r][k]));
    }
    #pragma unroll
    for (int r = 0; r < CH_HASH_ROWS; ++r) {
      const bool bit = acc[r] > 0.0f;
      if (t < OMVG_DESC_LEN) { const uint32_t w = __ballot_sync(0xffffffffu, bit); if ((t & 31) == 0) scode[r][t >> 5] = w; }
      else if (bit) { const int u = t - OMVG_DESC_LEN, g = u / CH_BITS, b = u % CH_BITS; atomicOr(&sbid[r][g], 1u << (CH_BITS - 1 - b)); }
    }
  }
  __syncthreads();
  if (t < CH_HASH_ROWS && row0 + t < total_rows) {
    code[row0 + t] = make_uint4(scode[t][0], scode[t][1], scode[t][2], scode[t][3]);
    bid[row0 + t] = make_uint4(sbid[t][0] | (sbid[t][1] << 16), sbid[t][2] | (sbid[t][3] << 16), sbid[t][4] | (sbid[t][5] << 16), 0u);
  }
}

// sort keys (segment = image*6 + group | bucket | local id) for the bucket tables
__global__ void cascade_keys_kernel(const uint4 *__restrict__ bid, const uint32_t *__restrict__ img_row0, const uint32_t *__restrict__ img_count,
                                    const uint32_t *__restrict__ img_real0, uint32_t n_images, unsigned long long *__restrict__ keys) {
  const uint32_t img = blockIdx.y;
  for (uint32_t local = blockIdx.x * blockDim.x + threadIdx.x; local < img_count[img]; local += gridDim.x * blockDim.x) {
    const uint4 b = bid[img_row0[img] + local];
    const uint32_t ids[6] = {b.x & 0xffffu, b.x >> 16, b.y & 0xffffu, b.y >> 16, b.z & 0xffffu, b.z >> 16};
    #pragma unroll
    for (int g = 0; g < CH_GROUPS; ++g)
      keys[(size_t)CH_GROUPS * (img_real0[img] + local) + g] = ((unsigned long long)(img * CH_GROUPS + g) << 34) | ((unsigned long long)ids[g] << 24) | local;
  }
}
// bucket starts from the sorted keys (bucket index = key >> 24, dense: segment * 1024 + bucket id) and item ids
__global__ void cascade_starts_kernel(const unsigned long long *__restrict__ keys, uint64_t n, uint32_t n_buckets, uint32_t *__restrict__ start, uint32_t *__restrict__ items) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t > n) return;
  const long long lo = t == 0 ? -1 : (long long)(keys[t - 1] >> 24), hi = t == n ? (long long)n_buckets : (long long)(keys[t] >> 24);
  for (long long k = lo + 1; k <= hi; ++k) start[k] = (uint32_t)t;
  if (t < n) items[t] = (uint32_t)(keys[t] & 0xffffffull);
}

// one warp per query (4 queries per warp); writes out[out_off + q].x = matched database id or -1
__global__ void __launch_bounds__(256) cascade_query_kernel(const uint8_t *__restrict__ desc, const int32_t *__restrict__ norm, const uint4 *__restrict__ code,
                                                            const uint4 *__restrict__ bid, const uint32_t *__restrict__ bstart, const uint32_t *__restrict__ bitems,
                                                            const PairInfo *__restrict__ pairs, int2 *__restrict__ out, float fratio) {
  const PairInfo P = pairs[blockIdx.y];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int qq = 0; qq < 4; ++qq) {
    const uint32_t q = blockIdx.x * 32 + warp * 4 + qq;
    if (q >= P.q_count) return;
    const uint32_t qrow = P.q_row0 + q;
    const uint4 qc = code[qrow], qb4 = bid[qrow];
    const uint32_t qb[6] = {qb4.x & 0xffffu, qb4.x >> 16, qb4.y & 0xffffu, qb4.y >> 16, qb4.z & 0xffffu, qb4.z >> 16};
    uint32_t s[6], len[6], tot = 0;
    #pragma unroll
    for (int g = 0; g < CH_GROUPS; ++g) { const uint32_t b = (P.db_group * CH_GROUPS + g) * CH_NB + qb[g]; s[g] = bstart[b]; len[g] = bstart[b + 1] - s[g]; tot += len[g]; }
    int result = -1;
    if (tot > 2) {                                              // "not at least NN candidates" counts duplicates (:301-304)
      // first CH_TOP unique candidates by (Hamming, position in the concatenated bucket lists): CH_TOP selection rounds
      // over the (short) lists; a candidate is a duplicate iff it already sat in the query's bucket of an earlier group
      uint32_t last = 0, my_sel = 0; int nsel = 0;
      if (tot <= 128) {
        // common case: every candidate's (Hamming, position | id) key is formed ONCE into 4 registers per lane, then
        // CH_TOP rounds of warp-min pick the winners (the streaming form below re-reads the lists every round)
        unsigned long long kk[4];
        #pragma unroll
        for (int i = 0; i < 4; ++i) {
          kk[i] = 0xffffffffffffffffull;
          uint32_t pp = lane + 32 * i;
          if (pp < tot) {
            const uint32_t pos = pp; int g = 0; uint32_t sg = 0;
            bool found = false;
            #pragma unroll
            for (int g2 = 0; g2 < CH_GROUPS; ++g2) if (!found) { if (pp < len[g2]) { g = g2; sg = s[g2]; found = true; } else pp -= len[g2]; }
            const uint32_t id = bitems[sg + pp], row = P.db_row0 + id;
            const uint4 cb = bid[row];
            const uint32_t cbv[6] = {cb.x & 0xffffu, cb.x >> 16, cb.y & 0xffffu, cb.y >> 16, cb.z & 0xffffu, cb.z >> 16};
            bool dup = false;
            #pragma unroll
            for (int g2 = 0; g2 < CH_GROUPS; ++g2) if (g2 < g && cbv[g2] == qb[g2]) dup = true;
            if (!dup) {
              const uint4 cc = code[row];
              const uint32_t ham = __popc(cc.x ^ qc.x) + __popc(cc.y ^ qc.y) + __popc(cc.z ^ qc.z) + __popc(cc.w ^ qc.w);
              kk[i] = ((unsigned long long)((ham << 24) | pos) << 32) | id;
            }
          }
        }
        for (int r = 0; r < CH_TOP; ++r) {
          unsigned long long m = min(min(kk[0], kk[1]), min(kk[2], kk[3]));
          #pragma unroll
          for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
          if (m == 0xffffffffffffffffull) break;
          #pragma unroll
          for (int i = 0; i < 4; ++i) if (kk[i] == m) kk[i] = 0xffffffffffffffffull;
          if (lane == r) my_sel = (uint32_t)(m & 0xffffffffull);
          ++nsel;
        }
      } else
      for (int r = 0; r < CH_TOP; ++r) {
        uint32_t best = 0xffffffffu, base = 0;
        #pragma unroll
        for (int g = 0; g < CH_GROUPS; ++g) {
          for (uint32_t off0 = 0; off0 < len[g]; off0 += 32) {
            const uint32_t off = off0 + lane;
            if (off < len[g]) {
              const uint32_t row = P.db_row0 + bitems[s[g] + off];
              const uint4 cb = bid[row];
              const uint32_t cbv[6] = {cb.x & 0xffffu, cb.x >> 16, cb.y & 0xffffu, cb.y >> 16, cb.z & 0xffffu, cb.z >> 16};
              bool dup = false;
              #pragma unroll
              for (int g2 = 0; g2 < CH_GROUPS; ++g2) if (g2 < g && cbv[g2] == qb[g2]) dup = true;
              if (!dup) {
                const uint4 cc = code[row];
                const uint32_t ham = __popc(cc.x ^ qc.x) + __popc(cc.y ^ qc.y) + __popc(cc.z ^ qc.z) + __popc(cc.w ^ qc.w);
                const uint32_t key = ((ham << 24) | (base + off)) + 1u;
                if (key > last && key < best) best = key;
              }
            }
          }
          base += len[g];
        }
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
        if (best == 0xffffffffu) break;
        last = best;
        uint32_t pos = (best - 1u) & 0xffffffu, id = 0; bool found = false;
        #pragma unroll
        for (int g = 0; g < CH_GROUPS; ++g) if (!found) { if (pos < len[g]) { id = bitems[s[g] + pos]; found = true; } else pos -= len[g]; }
        if (lane == r) my_sel = id;
        ++nsel;
      }
      if (nsel >= 2) {
        // exact L2 of the selected candidates: d = |q|^2 + |c|^2 - 2 q.c  (integers)
        const uint32_t qv = reinterpret_cast<const uint32_t *>(desc + (size_t)qrow * OMVG_DESC_LEN)[lane];
        const int qn = norm[qrow];
        unsigned long long mine = 0xffffffffffffffffull;
        for (int r = 0; r < nsel; ++r) {
          const uint32_t id = __shfl_sync(0xffffffffu, my_sel, r), row = P.db_row0 + id;
          uint32_t dot = __dp4a(qv, reinterpret_cast<const uint32_t *>(desc + (size_t)row * OMVG_DESC_LEN)[lane], 0u);
          #pragma unroll
          for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
          const int d = qn + norm[row] - 2 * (int)dot;
          if (lane == r) mine = ((unsigned long long)(uint32_t)d << 32) | id;
        }
        // top-2 of (distance, id) in lexicographic order (std::partial_sort of pair<dist,int>, :352-355)
        unsigned long long b1 = mine;
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) b1 = min(b1, __shfl_xor_sync(0xffffffffu, b1, o));
        unsigned long long b2 = mine == b1 ? 0xffffffffffffffffull : mine;
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) b2 = min(b2, __shfl_xor_sync(0xffffffffu, b2, o));
        const int d1 = (int)(b1 >> 32), d2 = (int)(b2 >> 32);
        if (__int2float_rn(d1) < __fmul_rn(fratio, __int2float_rn(d2))) result = (int)(uint32_t)(b1 & 0xffffffffull);   // matching_filters.hpp:57
      }
    }
    if (lane == 0) out[P.out_off + q].x = result;
  }
}

// ordered compaction of one pair's results: (database id, query id) for the kept queries, ascending query
__global__ void __launch_bounds__(FIN_THREADS) cascade_compact_kernel(const PairInfo *__restrict__ pairs, int2 *__restrict__ k12, uint32_t *__restrict__ counts) {
  __shared__ uint32_t warp_tot[FIN_THREADS / 32];
  __shared__ uint32_t running;
  const PairInfo P = pairs[blockIdx.x];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) running = 0;
  __syncthreads();
  int2 *io = k12 + P.out_off;
  for (uint32_t q0 = 0; q0 < P.q_count; q0 += FIN_THREADS) {
    const uint32_t q = q0 + threadIdx.x;
    const int v = q < P.q_count ? io[q].x : -1;
    const bool keep = v >= 0;
    const uint32_t bal = __ballot_sync(0xffffffffu, keep);
    const uint32_t in_warp = __popc(bal & ((1u << lane) - 1));
    if (lane == 0) warp_tot[warp] = __popc(bal);
    __syncthreads();
    uint32_t before = running;
    for (int w = 0; w < warp; ++w) before += warp_tot[w];
    if (keep) reinterpret_cast<uint2 *>(io)[before + in_warp] = make_uint2((uint32_t)v, q);
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t t = 0; for (int w = 0; w < FIN_THREADS / 32; ++w) t += warp_tot[w]; running += t; }
    __syncthreads();
  }
  if (threadIdx.x == 0) counts[blockIdx.x] = running;
}

}  // namespace omvg

// ===================================================================================== host side
using namespace omvg;

struct omvg_match_ctx {
  int device = 0, n_sms = 0;
  cudaStream_t stream = nullptr;
  uint32_t n_images = 0, total_rows = 0;
  std::vector<uint32_t> counts, row0, group;
  uint8_t *d_desc = nullptr; int32_t *d_norm = nullptr, *d_ckey = nullptr;
  uint32_t *d_img_row0 = nullptr, *d_img_count = nullptr, *d_img_group = nullptr, *d_row_img = nullptr;
  bool uploaded = false, prepared = false;
  CUtensorMap tmap, tmap_dig;   // descriptors: 128-row boxes; digits: 256-row boxes (one database tile)
  // fifth-slice kernel (match_dig2_kernel): 32 signed digits per arena row, per-image offset c0, eligibility
  uint4 *d_dig = nullptr; int32_t *d_img_c0 = nullptr; int2 *d_hmm = nullptr; std::vector<int32_t> c0; bool use_dig = false;
  // run state
  int2 *d_k12 = nullptr; size_t k12_cap = 0;           // in int2 elements
  Unit *d_units = nullptr; size_t units_cap = 0;
  PairInfo *d_pairs = nullptr; uint32_t *d_counts = nullptr; size_t pairs_cap = 0;
  uint64_t *d_offsets = nullptr; size_t offsets_cap = 0;   // n_pairs + 1 (global)
  uint64_t *d_total = nullptr;
  uint2 *d_out = nullptr; size_t out_cap = 0;
  uint64_t n_pairs_last = 0, total_last = 0; bool have_result = false;
  uint64_t *h_offsets = nullptr; size_t h_offsets_cap = 0; uint32_t *h_ij = nullptr; size_t h_ij_cap = 0;
  uint64_t launches = 0;
  double tc_ms = 0; uint64_t tc_launches = 0; std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
  std::vector<cudaEvent_t> ev_pool;
  size_t k12_budget_bytes = size_t(2) << 30;
  // cascade hashing state (omvg_match_cascade_prepare)
  uint4 *d_code = nullptr, *d_bid = nullptr; uint32_t *d_bstart = nullptr, *d_bitems = nullptr; float *d_proj = nullptr, *d_zm = nullptr;
  bool cascade_ready = false; std::vector<float> h_zm;
};

namespace {

typedef CUresult (*encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_tmap(omvg_match_ctx *c) {
  void *fn = nullptr; cudaDriverEntryPointQueryResult qres;
  OMVG_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (!fn || qres != cudaDriverEntryPointSuccess) return fail(OMVG_E_CUDA, "cuTensorMapEncodeTiled not available");
  const cuuint64_t dims[2] = {OMVG_DESC_LEN, c->total_rows};
  const cuuint64_t strides[1] = {OMVG_DESC_LEN};
  const cuuint32_t box[2] = {OMVG_DESC_LEN, 128};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = ((encode_tiled_fn)fn)(&c->tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, c->d_desc, dims, strides, box, estr,
                                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(OMVG_E_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  const cuuint64_t ddims[2] = {DIG_LEN, c->total_rows};
  const cuuint64_t dstrides[1] = {DIG_LEN};
  const cuuint32_t dbox[2] = {DIG_LEN, TILE_DB};
  const CUresult r2 = ((encode_tiled_fn)fn)(&c->tmap_dig, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, c->d_dig, ddims, dstrides, dbox, estr,
                                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B,
                                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r2 != CUDA_SUCCESS) return fail(OMVG_E_CUDA, "cuTensorMapEncodeTiled (digits) failed (%d)", (int)r2);
  return OMVG_OK;
}

void free_images(omvg_match_ctx *c) {
  cudaFree(c->d_code); cudaFree(c->d_bid); cudaFree(c->d_bstart); cudaFree(c->d_bitems); cudaFree(c->d_proj); cudaFree(c->d_zm);
  c->d_code = c->d_bid = nullptr; c->d_bstart = c->d_bitems = nullptr; c->d_proj = c->d_zm = nullptr; c->cascade_ready = false;
  cudaFree(c->d_desc); cudaFree(c->d_norm); cudaFree(c->d_ckey); cudaFree(c->d_img_row0); cudaFree(c->d_img_count);
  cudaFree(c->d_img_group); cudaFree(c->d_row_img); cudaFree(c->d_dig); cudaFree(c->d_img_c0); cudaFree(c->d_hmm);
  c->d_dig = nullptr; c->d_img_c0 = nullptr; c->d_hmm = nullptr; c->use_dig = false;
  c->d_desc = nullptr; c->d_norm = c->d_ckey = nullptr; c->d_img_row0 = c->d_img_count = c->d_img_group = c->d_row_img = nullptr;
}

template <typename T> int ensure(T *&p, size_t &cap, size_t need) {
  if (need <= cap) return OMVG_OK;
  if (p) cudaFree(p);
  p = nullptr; cap = 0;
  OMVG_CUDA(cudaMalloc(&p, need * sizeof(T)));
  cap = need; return OMVG_OK;
}

int drain_timers(omvg_match_ctx *c) {
  for (auto &pr : c->pending) {
    float ms = 0; OMVG_CUDA(cudaEventSynchronize(pr.second)); OMVG_CUDA(cudaEventElapsedTime(&ms, pr.first, pr.second));
    c->tc_ms += ms; c->ev_pool.push_back(pr.first); c->ev_pool.push_back(pr.second);
  }
  c->pending.clear(); return OMVG_OK;
}
cudaEvent_t get_event(omvg_match_ctx *c) {
  if (!c->ev_pool.empty()) { cudaEvent_t e = c->ev_pool.back(); c->ev_pool.pop_back(); return e; }
  cudaEvent_t e; cudaEventCreate(&e); return e;
}

// one batch of pairs: tensor-core kernel + finalize + scan + compact
int run_batch(omvg_match_ctx *c, const uint32_t *pi, const uint32_t *pj, uint64_t p0, uint64_t p1, float fratio,
              std::vector<Unit> &units, std::vector<PairInfo> &pinfo) {
  units.clear(); pinfo.clear();
  size_t out = 0, n_units = 0;
  const uint32_t q_tiles = c->use_dig ? 2 : 1;            // query tiles per unit: match_dig2_kernel takes two
  for (uint64_t p = p0; p < p1; ++p) {
    const uint32_t I = pi[p], J = pj[p];
    PairInfo P{}; P.db_row0 = c->row0[I]; P.db_count = c->counts[I]; P.db_group = c->group[I]; P.db_c0 = c->c0.empty() ? 0 : c->c0[I];
    P.q_row0 = c->row0[J]; P.q_count = c->counts[J]; P.out_off = out;
    // Matcher_Regions.cpp:65-69,85-90 (empty regions) and matcher_brute_force.hpp:108-113 (NN > rows)
    const bool active = P.db_count >= 2 && P.q_count >= 1;
    if (!active) P.q_count = 0;
    pinfo.push_back(P);
    if (!active) continue;
    const uint32_t qt = (P.q_count + TILE_Q - 1) / TILE_Q;
    pinfo.back().unit0 = (uint32_t)n_units; n_units += (qt + q_tiles - 1) / q_tiles;
    out += size_t(qt) * TILE_Q;
  }
  if (out > 0xffffffffull) return fail(OMVG_E_ARG, "batch too large");
  const uint32_t nb = (uint32_t)(p1 - p0);
  int rc;
  if ((rc = ensure(c->d_k12, c->k12_cap, std::max<size_t>(out, 1)))) return rc;
  if ((rc = ensure(c->d_units, c->units_cap, std::max<size_t>(n_units, 1)))) return rc;
  if (nb > c->pairs_cap) {
    if (c->d_pairs) cudaFree(c->d_pairs); if (c->d_counts) cudaFree(c->d_counts);
    c->d_pairs = nullptr; c->d_counts = nullptr; c->pairs_cap = 0;
    OMVG_CUDA(cudaMalloc(&c->d_pairs, nb * sizeof(PairInfo))); OMVG_CUDA(cudaMalloc(&c->d_counts, nb * sizeof(uint32_t)));
    c->pairs_cap = nb;
  }
  OMVG_CUDA(cudaMemcpyAsync(c->d_pairs, pinfo.data(), nb * sizeof(PairInfo), cudaMemcpyHostToDevice, c->stream));
  if (n_units) {
    expand_units_kernel<<<nb, 64, 0, c->stream>>>(c->d_pairs, c->d_units, q_tiles); OMVG_CUDA(cudaGetLastError()); c->launches++;
    const uint32_t grid = (uint32_t)std::min<size_t>(n_units, (size_t)c->n_sms);
    cudaEvent_t e0 = get_event(c), e1 = get_event(c);
    OMVG_CUDA(cudaEventRecord(e0, c->stream));
    if (c->use_dig) match_dig2_kernel<<<grid, DIG2_THREADS, DIG2_SMEM_BYTES, c->stream>>>(c->tmap, c->tmap_dig, c->d_units, (uint32_t)n_units, c->d_k12);
    else match_tc_kernel<<<grid, TC_THREADS, SMEM_BYTES, c->stream>>>(c->tmap, c->d_ckey, c->d_units, (uint32_t)n_units, c->d_k12);
    OMVG_CUDA(cudaGetLastError());
    OMVG_CUDA(cudaEventRecord(e1, c->stream));
    c->pending.emplace_back(e0, e1); c->tc_launches++; c->launches++;
  }
  if (c->use_dig) match_finalize_kernel<true><<<nb, FIN_THREADS, 0, c->stream>>>(c->d_desc, c->d_norm, c->d_pairs, c->d_k12, c->d_counts, fratio);
  else match_finalize_kernel<false><<<nb, FIN_THREADS, 0, c->stream>>>(c->d_desc, c->d_norm, c->d_pairs, c->d_k12, c->d_counts, fratio);
  OMVG_CUDA(cudaGetLastError());
  scan_counts_kernel<<<1, 1024, 0, c->stream>>>(c->d_counts, nb, c->d_offsets + p0, c->d_total);
  OMVG_CUDA(cudaGetLastError());
  c->launches += 2;
  // size the global output buffer: needs the running total (one small sync per batch)
  uint64_t total = 0;
  OMVG_CUDA(cudaMemcpyAsync(&total, c->d_total, sizeof total, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  if (total > c->out_cap) {
    const size_t ncap = std::max<size_t>(total, c->out_cap * 2 + 1024);
    uint2 *n = nullptr; OMVG_CUDA(cudaMalloc(&n, ncap * sizeof(uint2)));
    if (c->d_out && c->total_last) OMVG_CUDA(cudaMemcpyAsync(n, c->d_out, c->total_last * sizeof(uint2), cudaMemcpyDeviceToDevice, c->stream));
    OMVG_CUDA(cudaStreamSynchronize(c->stream));
    if (c->d_out) cudaFree(c->d_out);
    c->d_out = n; c->out_cap = ncap;
  }
  compact_kernel<<<nb, 128, 0, c->stream>>>(c->d_k12, c->d_pairs, c->d_counts, c->d_offsets + p0, c->d_out);
  OMVG_CUDA(cudaGetLastError());
  c->launches++;
  c->total_last = total;
  return OMVG_OK;
}

}  // namespace

extern "C" {

int omvg_version(void) { return 100; }
const char *omvg_last_error(void) { return last_error().c_str(); }
int omvg_device_count(void) {
  int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  int ok = 0; for (int d = 0; d < n; ++d) { cudaDeviceProp p; if (cudaGetDeviceProperties(&p, d) == cudaSuccess && p.major == 10) ++ok; }
  return ok;
}

int omvg_match_create(omvg_match_ctx **out, int device) {
  if (!out) return fail(OMVG_E_ARG, "null ctx");
  int n = 0; OMVG_CUDA(cudaGetDeviceCount(&n));
  if (device < 0 || device >= n) return fail(OMVG_E_CUDA, "no CUDA device %d (found %d)", device, n);
  int cc_major = 0, cc_minor = 0, n_sms = 0;
  OMVG_CUDA(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, device));
  OMVG_CUDA(cudaDeviceGetAttribute(&cc_minor, cudaDevAttrComputeCapabilityMinor, device));
  OMVG_CUDA(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, device));
  if (cc_major != 10) return fail(OMVG_E_CUDA, "device %d is sm_%d%d; this library is sm_100a only", device, cc_major, cc_minor);
  OMVG_CUDA(cudaSetDevice(device));
  omvg_match_ctx *c = new omvg_match_ctx; c->device = device; c->n_sms = n_sms;
  OMVG_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  OMVG_CUDA(cudaFuncSetAttribute(match_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  OMVG_CUDA(cudaFuncSetAttribute(match_dig2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DIG2_SMEM_BYTES));
  OMVG_CUDA(cudaMalloc(&c->d_total, sizeof(uint64_t)));
  if (const char *e = getenv("OMVG_MATCH_K12_MB")) c->k12_budget_bytes = size_t(atol(e)) << 20;
  *out = c; return OMVG_OK;
}

int omvg_match_destroy(omvg_match_ctx *c) {
  if (!c) return OMVG_OK;
  cudaSetDevice(c->device); cudaStreamSynchronize(c->stream);
  drain_timers(c); for (auto e : c->ev_pool) cudaEventDestroy(e);
  free_images(c);
  cudaFree(c->d_k12); cudaFree(c->d_units); cudaFree(c->d_pairs); cudaFree(c->d_counts); cudaFree(c->d_offsets);
  cudaFree(c->d_total); cudaFree(c->d_out);
  if (c->h_offsets) cudaFreeHost(c->h_offsets); if (c->h_ij) cudaFreeHost(c->h_ij);
  cudaStreamDestroy(c->stream);
  delete c; return OMVG_OK;
}

int omvg_match_set_images(omvg_match_ctx *c, uint32_t n_images, const uint32_t *counts) {
  if (!c || (!counts && n_images)) return fail(OMVG_E_ARG, "bad arguments");
  OMVG_CUDA(cudaSetDevice(c->device));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  free_images(c);
  c->n_images = n_images; c->counts.assign(counts, counts + n_images); c->row0.resize(n_images); c->group.resize(n_images);
  uint64_t rows = 0; std::vector<uint32_t> row_img;
  for (uint32_t k = 0; k < n_images; ++k) {
    c->row0[k] = (uint32_t)rows;
    const uint32_t padded = (counts[k] + ROW_PAD - 1) / ROW_PAD * ROW_PAD;
    c->group[k] = 32 * std::max<uint32_t>(1, (counts[k] + 8191) / 8192);      // rows/group <= 256 groups
    for (uint32_t s = 0; s < padded / ROW_PAD; ++s) row_img.push_back(k);
    rows += padded;
    if (rows + 2 * ROW_PAD > 0xffffffffull) return fail(OMVG_E_ARG, "collection too large (%llu rows)", (unsigned long long)rows);
  }
  rows += ROW_PAD;                                      // tail slot: TMA boxes never leave the arena
  row_img.push_back(n_images ? n_images - 1 : 0);
  c->total_rows = (uint32_t)rows;
  OMVG_CUDA(cudaMalloc(&c->d_desc, rows * OMVG_DESC_LEN));
  OMVG_CUDA(cudaMemsetAsync(c->d_desc, 0, rows * OMVG_DESC_LEN, c->stream));
  OMVG_CUDA(cudaMalloc(&c->d_norm, rows * 4)); OMVG_CUDA(cudaMalloc(&c->d_ckey, rows * 4));
  OMVG_CUDA(cudaMalloc(&c->d_dig, rows * DIG_LEN)); OMVG_CUDA(cudaMalloc(&c->d_img_c0, std::max(1u, n_images) * 4)); OMVG_CUDA(cudaMalloc(&c->d_hmm, std::max(1u, n_images) * sizeof(int2)));
  OMVG_CUDA(cudaMalloc(&c->d_img_row0, std::max(1u, n_images) * 4)); OMVG_CUDA(cudaMalloc(&c->d_img_count, std::max(1u, n_images) * 4));
  OMVG_CUDA(cudaMalloc(&c->d_img_group, std::max(1u, n_images) * 4)); OMVG_CUDA(cudaMalloc(&c->d_row_img, row_img.size() * 4));
  if (n_images) {
    OMVG_CUDA(cudaMemcpyAsync(c->d_img_row0, c->row0.data(), n_images * 4, cudaMemcpyHostToDevice, c->stream));
    OMVG_CUDA(cudaMemcpyAsync(c->d_img_count, c->counts.data(), n_images * 4, cudaMemcpyHostToDevice, c->stream));
    OMVG_CUDA(cudaMemcpyAsync(c->d_img_group, c->group.data(), n_images * 4, cudaMemcpyHostToDevice, c->stream));
  }
  OMVG_CUDA(cudaMemcpyAsync(c->d_row_img, row_img.data(), row_img.size() * 4, cudaMemcpyHostToDevice, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  c->uploaded = false; c->prepared = false; c->have_result = false;
  return make_tmap(c);
}

int omvg_match_upload_host(omvg_match_ctx *c, uint32_t image, const uint8_t *desc) {
  if (!c || image >= c->n_images || (!desc && c->counts[image])) return fail(OMVG_E_ARG, "bad image %u", image);
  OMVG_CUDA(cudaSetDevice(c->device));
  if (c->counts[image])
    OMVG_CUDA(cudaMemcpyAsync(c->d_desc + (size_t)c->row0[image] * OMVG_DESC_LEN, desc, (size_t)c->counts[image] * OMVG_DESC_LEN,
                              cudaMemcpyHostToDevice, c->stream));
  c->uploaded = true; c->prepared = false; c->cascade_ready = false; return OMVG_OK;
}

int omvg_match_upload_device(omvg_match_ctx *c, uint32_t image, const void *desc_dev) {
  if (!c || image >= c->n_images || (!desc_dev && c->counts[image])) return fail(OMVG_E_ARG, "bad image %u", image);
  OMVG_CUDA(cudaSetDevice(c->device));
  if (c->counts[image])
    OMVG_CUDA(cudaMemcpyAsync(c->d_desc + (size_t)c->row0[image] * OMVG_DESC_LEN, desc_dev, (size_t)c->counts[image] * OMVG_DESC_LEN,
                              cudaMemcpyDeviceToDevice, c->stream));
  c->uploaded = true; c->prepared = false; c->cascade_ready = false; return OMVG_OK;
}

int omvg_match_upload_device_packed(omvg_match_ctx *c, const void *desc_dev) {
  if (!c || !desc_dev) return fail(OMVG_E_ARG, "bad arguments");
  size_t off = 0;
  for (uint32_t k = 0; k < c->n_images; ++k) {
    const int rc = omvg_match_upload_device(c, k, static_cast<const uint8_t *>(desc_dev) + off);
    if (rc) return rc;
    off += (size_t)c->counts[k] * OMVG_DESC_LEN;
  }
  c->uploaded = true; return OMVG_OK;
}

int omvg_match_prepare(omvg_match_ctx *c) {
  if (!c || !c->d_desc) return fail(OMVG_E_STATE, "set_images first");
  OMVG_CUDA(cudaSetDevice(c->device));
  const uint32_t threads = 256, rows_per_block = threads / 8;
  prep_rows_kernel<<<(c->total_rows + rows_per_block - 1) / rows_per_block, threads, 0, c->stream>>>(
      c->d_desc, c->d_img_row0, c->d_img_count, c->d_img_group, c->d_row_img, c->d_norm, c->d_ckey, c->total_rows);
  OMVG_CUDA(cudaGetLastError());
  c->launches++;
  // fifth-slice kernel: per-image range of h = ceil(|b|^2 / 2) -> offset c0 and eligibility (one small read-back)
  c->c0.assign(c->n_images, 0); c->use_dig = false;
  const bool force_tc4 = getenv("OMVG_MATCH_TC4") != nullptr;         // A/B: the round-1 kernel (IMAD epilogue)
  if (c->n_images && !force_tc4) {
    prep_minmax_kernel<<<c->n_images, 256, 0, c->stream>>>(c->d_norm, c->d_img_row0, c->d_img_count, c->d_hmm); OMVG_CUDA(cudaGetLastError());
    std::vector<int2> hmm(c->n_images);
    OMVG_CUDA(cudaMemcpyAsync(hmm.data(), c->d_hmm, c->n_images * sizeof(int2), cudaMemcpyDeviceToHost, c->stream));
    OMVG_CUDA(cudaStreamSynchronize(c->stream));
    bool ok = true;
    for (uint32_t k = 0; k < c->n_images; ++k) {
      if (!c->counts[k]) continue;
      if ((long long)hmm[k].y - hmm[k].x > DIG_SPREAD_MAX || c->group[k] / 32 >= 2048) { ok = false; break; }
      c->c0[k] = std::max(0, hmm[k].y + DIG_VMIN);                           // v = c0 - h in [DIG_VMIN, DIG_VMAX]
    }
    if (ok) {
      OMVG_CUDA(cudaMemcpyAsync(c->d_img_c0, c->c0.data(), c->n_images * 4, cudaMemcpyHostToDevice, c->stream));
      prep_digits_kernel<<<(c->total_rows + 255) / 256, 256, 0, c->stream>>>(c->d_norm, c->d_img_row0, c->d_img_count, c->d_row_img, c->d_img_c0, c->d_dig, c->total_rows);
      OMVG_CUDA(cudaGetLastError());
      OMVG_CUDA(cudaStreamSynchronize(c->stream));                            // c->c0 (host vector) is read by the copy above
      c->launches += 2; c->use_dig = true;
    }
  }
  c->prepared = true; c->cascade_ready = false; return OMVG_OK;
}

int omvg_match_run(omvg_match_ctx *c, const uint32_t *pair_i, const uint32_t *pair_j, uint64_t n_pairs, float dist_ratio) {
  if (!c || ((!pair_i || !pair_j) && n_pairs)) return fail(OMVG_E_ARG, "bad arguments");
  if (!c->prepared) return fail(OMVG_E_STATE, "omvg_match_prepare must follow the uploads");
  if (!(dist_ratio >= 0.f)) return fail(OMVG_E_ARG, "dist_ratio must be >= 0");
  OMVG_CUDA(cudaSetDevice(c->device));
  for (uint64_t p = 0; p < n_pairs; ++p)
    if (pair_i[p] >= c->n_images || pair_j[p] >= c->n_images) return fail(OMVG_E_ARG, "pair %llu out of range", (unsigned long long)p);
  const float fratio = dist_ratio * dist_ratio;                   // numeric.h:56 Square<float>, regions_matcher.hpp:196
  if (n_pairs + 1 > c->offsets_cap) {
    if (c->d_offsets) cudaFree(c->d_offsets);
    c->d_offsets = nullptr; c->offsets_cap = 0;
    OMVG_CUDA(cudaMalloc(&c->d_offsets, (n_pairs + 1) * sizeof(uint64_t))); c->offsets_cap = n_pairs + 1;
  }
  OMVG_CUDA(cudaMemsetAsync(c->d_total, 0, sizeof(uint64_t), c->stream));
  OMVG_CUDA(cudaMemsetAsync(c->d_offsets, 0, sizeof(uint64_t), c->stream));
  c->total_last = 0; c->n_pairs_last = n_pairs; c->have_result = false;
  std::vector<Unit> units; std::vector<PairInfo> pinfo;
  const size_t budget = c->k12_budget_bytes / sizeof(int2);
  uint64_t p0 = 0;
  while (p0 < n_pairs) {
    size_t acc = 0; uint64_t p1 = p0;
    while (p1 < n_pairs) {
      const size_t need = size_t((c->counts[pair_j[p1]] + TILE_Q - 1) / TILE_Q) * TILE_Q;
      if (p1 > p0 && (acc + need > budget || p1 - p0 >= (1u << 20))) break;
      acc += need; ++p1;
    }
    const int rc = run_batch(c, pair_i, pair_j, p0, p1, fratio, units, pinfo);
    if (rc) return rc;
    p0 = p1;
  }
  c->have_result = true; return OMVG_OK;
}

int omvg_match_sync(omvg_match_ctx *c) {
  if (!c) return fail(OMVG_E_ARG, "null ctx");
  OMVG_CUDA(cudaSetDevice(c->device)); OMVG_CUDA(cudaStreamSynchronize(c->stream));
  return drain_timers(c);
}

int omvg_match_fetch(omvg_match_ctx *c, const uint64_t **offsets, const uint32_t **ij, uint64_t *n_matches) {
  if (!c || !offsets || !ij || !n_matches) return fail(OMVG_E_ARG, "bad arguments");
  if (!c->have_result) return fail(OMVG_E_STATE, "no result: call omvg_match_run");
  OMVG_CUDA(cudaSetDevice(c->device));
  const size_t no = c->n_pairs_last + 1;
  if (no > c->h_offsets_cap) { if (c->h_offsets) cudaFreeHost(c->h_offsets); c->h_offsets = nullptr; c->h_offsets_cap = 0;
    OMVG_CUDA(cudaMallocHost(&c->h_offsets, no * sizeof(uint64_t))); c->h_offsets_cap = no; }
  OMVG_CUDA(cudaMemcpyAsync(c->h_offsets, c->d_offsets, no * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
  if (c->n_pairs_last == 0) { OMVG_CUDA(cudaStreamSynchronize(c->stream)); c->h_offsets[0] = 0; }
  const size_t nm = c->total_last;
  if (nm > c->h_ij_cap || !c->h_ij) { if (c->h_ij) cudaFreeHost(c->h_ij); c->h_ij = nullptr; c->h_ij_cap = 0;
    OMVG_CUDA(cudaMallocHost(&c->h_ij, std::max<size_t>(nm, 1) * 2 * sizeof(uint32_t))); c->h_ij_cap = std::max<size_t>(nm, 1); }
  if (nm) OMVG_CUDA(cudaMemcpyAsync(c->h_ij, c->d_out, nm * sizeof(uint2), cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  drain_timers(c);
  *offsets = c->h_offsets; *ij = c->h_ij; *n_matches = nm;
  return OMVG_OK;
}

uint64_t omvg_match_launch_count(const omvg_match_ctx *c) { return c ? c->launches : 0; }
int omvg_match_kernel_variant(const omvg_match_ctx *c) { return (!c || !c->prepared) ? 0 : (c->use_dig ? 5 : 4); }

int omvg_match_kernel_time(omvg_match_ctx *c, double *ms, uint64_t *launches, int reset) {
  if (!c) return fail(OMVG_E_ARG, "null ctx");
  OMVG_CUDA(cudaSetDevice(c->device)); OMVG_CUDA(cudaStreamSynchronize(c->stream));
  const int rc = drain_timers(c); if (rc) return rc;
  if (ms) *ms = c->tc_ms; if (launches) *launches = c->tc_launches;
  if (reset) { c->tc_ms = 0; c->tc_launches = 0; }
  return OMVG_OK;
}

// ---- cascade hashing ---------------------------------------------------------------------------------------
// Hash every image (zero-mean vector over the USED images, Cascade_Hashing_Matcher_Regions.cpp:78-105), build the
// 6 x 1024 bucket tables of every image with one radix sort.  Needs omvg_match_prepare (row norms).
int omvg_match_cascade_prepare(omvg_match_ctx *c, const float *primary, const float *secondary, const uint8_t *used) {
  if (!c || !primary || !secondary) return fail(OMVG_E_ARG, "bad arguments");
  if (!c->prepared) return fail(OMVG_E_STATE, "omvg_match_prepare must come first");
  OMVG_CUDA(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  const uint32_t ni = c->n_images;
  for (uint32_t k = 0; k < ni; ++k) if (c->counts[k] >= (1u << 24)) return fail(OMVG_E_UNSUPPORTED, "image %u has more than 2^24 descriptors", k);
  // zero-mean descriptor: exact integer column sums on the device, the two float reductions on the host
  // (float(sum)/float(n) per image; sequential float sum over the used images, / n_used: cascade_hasher.hpp:166-176)
  unsigned long long *d_sums = nullptr; OMVG_CUDA(cudaMalloc(&d_sums, std::max<size_t>(1, ni) * OMVG_DESC_LEN * sizeof(unsigned long long)));
  if (ni) { cascade_colsum_kernel<<<ni, OMVG_DESC_LEN, 0, st>>>(c->d_desc, c->d_img_row0, c->d_img_count, d_sums); OMVG_CUDA(cudaGetLastError()); c->launches++; }
  std::vector<unsigned long long> sums((size_t)ni * OMVG_DESC_LEN);
  if (ni) OMVG_CUDA(cudaMemcpyAsync(sums.data(), d_sums, sums.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  OMVG_CUDA(cudaStreamSynchronize(st)); cudaFree(d_sums);
  c->h_zm.assign(OMVG_DESC_LEN, 0.0f);
  uint32_t n_used = 0; for (uint32_t k = 0; k < ni; ++k) if (!used || used[k]) ++n_used;
  for (int col = 0; col < OMVG_DESC_LEN; ++col) {
    float acc = 0.0f;
    for (uint32_t k = 0; k < ni; ++k) { if (used && !used[k]) continue;
      const float m = c->counts[k] ? (float)sums[(size_t)k * OMVG_DESC_LEN + col] / (float)c->counts[k] : 0.0f; acc = acc + m; }
    c->h_zm[col] = n_used ? acc / (float)n_used : 0.0f;
  }
  if (!c->d_proj) OMVG_CUDA(cudaMalloc(&c->d_proj, (size_t)CH_OUT * OMVG_DESC_LEN * sizeof(float)));
  if (!c->d_zm) OMVG_CUDA(cudaMalloc(&c->d_zm, OMVG_DESC_LEN * sizeof(float)));
  OMVG_CUDA(cudaMemcpyAsync(c->d_proj, primary, (size_t)OMVG_DESC_LEN * OMVG_DESC_LEN * sizeof(float), cudaMemcpyHostToDevice, st));
  OMVG_CUDA(cudaMemcpyAsync(c->d_proj + (size_t)OMVG_DESC_LEN * OMVG_DESC_LEN, secondary, (size_t)CH_GROUPS * CH_BITS * OMVG_DESC_LEN * sizeof(float), cudaMemcpyHostToDevice, st));
  OMVG_CUDA(cudaMemcpyAsync(c->d_zm, c->h_zm.data(), OMVG_DESC_LEN * sizeof(float), cudaMemcpyHostToDevice, st));
  if (!c->d_code) { OMVG_CUDA(cudaMalloc(&c->d_code, (size_t)c->total_rows * sizeof(uint4))); OMVG_CUDA(cudaMalloc(&c->d_bid, (size_t)c->total_rows * sizeof(uint4))); }
  cascade_hash_kernel<<<(c->total_rows + CH_HASH_ROWS - 1) / CH_HASH_ROWS, CH_HASH_THREADS, 0, st>>>(c->d_desc, c->total_rows, c->d_zm, c->d_proj, c->d_code, c->d_bid);
  OMVG_CUDA(cudaGetLastError()); c->launches++;
  // bucket tables
  std::vector<uint32_t> real0(ni + 1, 0); for (uint32_t k = 0; k < ni; ++k) real0[k + 1] = real0[k] + c->counts[k];
  const uint64_t n_real = real0[ni], n_keys = n_real * CH_GROUPS; const uint32_t n_buckets = ni * CH_GROUPS * CH_NB;
  if (n_keys >= (1ull << 31)) return fail(OMVG_E_UNSUPPORTED, "collection too large for the bucket tables (%llu keys; CUB radix sort takes int counts)", (unsigned long long)n_keys);
  cudaFree(c->d_bstart); cudaFree(c->d_bitems); c->d_bstart = c->d_bitems = nullptr;
  OMVG_CUDA(cudaMalloc(&c->d_bstart, ((size_t)n_buckets + 1) * sizeof(uint32_t))); OMVG_CUDA(cudaMalloc(&c->d_bitems, std::max<uint64_t>(1, n_keys) * sizeof(uint32_t)));
  uint32_t *d_real0 = nullptr; unsigned long long *d_keys = nullptr, *d_keys2 = nullptr; void *d_tmp = nullptr;
  struct Scratch { uint32_t *&a; unsigned long long *&b, *&c; void *&d; ~Scratch() { cudaFree(a); cudaFree(b); cudaFree(c); cudaFree(d); } } scratch{d_real0, d_keys, d_keys2, d_tmp};   // freed on every exit
  OMVG_CUDA(cudaMalloc(&d_real0, (ni + 1) * sizeof(uint32_t)));
  OMVG_CUDA(cudaMemcpyAsync(d_real0, real0.data(), (ni + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  OMVG_CUDA(cudaMalloc(&d_keys, std::max<uint64_t>(1, n_keys) * 8)); OMVG_CUDA(cudaMalloc(&d_keys2, std::max<uint64_t>(1, n_keys) * 8));
  if (n_keys) {
    cascade_keys_kernel<<<dim3(32, ni), 256, 0, st>>>(c->d_bid, c->d_img_row0, c->d_img_count, d_real0, ni, d_keys); OMVG_CUDA(cudaGetLastError());
    int seg_bits = 1; while ((1ull << seg_bits) < (unsigned long long)ni * CH_GROUPS) ++seg_bits;
    size_t tb = 0; OMVG_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tb, d_keys, d_keys2, (int)n_keys, 0, 34 + seg_bits, st));
    OMVG_CUDA(cudaMalloc(&d_tmp, tb));
    OMVG_CUDA(cub::DeviceRadixSort::SortKeys(d_tmp, tb, d_keys, d_keys2, (int)n_keys, 0, 34 + seg_bits, st));
    c->launches += 2;
  }
  cascade_starts_kernel<<<(unsigned)((n_keys + 256) / 256), 256, 0, st>>>(d_keys2, n_keys, n_buckets, c->d_bstart, c->d_bitems); OMVG_CUDA(cudaGetLastError());
  c->launches++;
  OMVG_CUDA(cudaStreamSynchronize(st));
  c->cascade_ready = true; return OMVG_OK;
}

// Cascade_Hashing_Matcher_Regions.cpp:110-189 for a list of pairs (I = database, J = queries).  The result is read
// with omvg_match_fetch: CSR rows of (i, j) in ascending j (the caller sorts by (i, j) as IndMatch::getDeduplicated does).
int omvg_match_cascade_run(omvg_match_ctx *c, const uint32_t *pair_i, const uint32_t *pair_j, uint64_t n_pairs, float dist_ratio) {
  if (!c || ((!pair_i || !pair_j) && n_pairs)) return fail(OMVG_E_ARG, "bad arguments");
  if (!c->cascade_ready) return fail(OMVG_E_STATE, "omvg_match_cascade_prepare first");
  if (!(dist_ratio >= 0.f)) return fail(OMVG_E_ARG, "dist_ratio must be >= 0");
  OMVG_CUDA(cudaSetDevice(c->device));
  for (uint64_t p = 0; p < n_pairs; ++p)
    if (pair_i[p] >= c->n_images || pair_j[p] >= c->n_images) return fail(OMVG_E_ARG, "pair %llu out of range", (unsigned long long)p);
  const float fratio = dist_ratio * dist_ratio;
  if (n_pairs + 1 > c->offsets_cap) {
    if (c->d_offsets) cudaFree(c->d_offsets);
    c->d_offsets = nullptr; c->offsets_cap = 0;
    OMVG_CUDA(cudaMalloc(&c->d_offsets, (n_pairs + 1) * sizeof(uint64_t))); c->offsets_cap = n_pairs + 1;
  }
  OMVG_CUDA(cudaMemsetAsync(c->d_total, 0, sizeof(uint64_t), c->stream));
  OMVG_CUDA(cudaMemsetAsync(c->d_offsets, 0, sizeof(uint64_t), c->stream));
  c->total_last = 0; c->n_pairs_last = n_pairs; c->have_result = false;
  std::vector<PairInfo> pinfo;
  const size_t budget = c->k12_budget_bytes / sizeof(int2);
  uint64_t p0 = 0;
  while (p0 < n_pairs) {
    pinfo.clear(); size_t out = 0; uint64_t p1 = p0; uint32_t maxq = 0;
    while (p1 < n_pairs && p1 - p0 < 65535) {
      const uint32_t I = pair_i[p1], J = pair_j[p1];
      if (p1 > p0 && out + c->counts[J] > budget) break;
      PairInfo P{}; P.db_row0 = c->row0[I]; P.db_count = c->counts[I]; P.db_group = I; P.q_row0 = c->row0[J]; P.q_count = c->counts[J]; P.out_off = out;
      if (P.db_count == 0) P.q_count = 0;                      // empty database image: nothing (:120-124)
      out += P.q_count; maxq = std::max(maxq, P.q_count); pinfo.push_back(P); ++p1;
    }
    const uint32_t nb = (uint32_t)(p1 - p0);
    int rc;
    if ((rc = ensure(c->d_k12, c->k12_cap, std::max<size_t>(out, 1)))) return rc;
    if (nb > c->pairs_cap) {
      if (c->d_pairs) cudaFree(c->d_pairs); if (c->d_counts) cudaFree(c->d_counts);
      c->d_pairs = nullptr; c->d_counts = nullptr; c->pairs_cap = 0;
      OMVG_CUDA(cudaMalloc(&c->d_pairs, nb * sizeof(PairInfo))); OMVG_CUDA(cudaMalloc(&c->d_counts, nb * sizeof(uint32_t)));
      c->pairs_cap = nb;
    }
    OMVG_CUDA(cudaMemcpyAsync(c->d_pairs, pinfo.data(), nb * sizeof(PairInfo), cudaMemcpyHostToDevice, c->stream));
    if (maxq) {
      cudaEvent_t e0 = get_event(c), e1 = get_event(c);
      OMVG_CUDA(cudaEventRecord(e0, c->stream));
      cascade_query_kernel<<<dim3((maxq + 31) / 32, nb), 256, 0, c->stream>>>(c->d_desc, c->d_norm, c->d_code, c->d_bid, c->d_bstart, c->d_bitems, c->d_pairs, c->d_k12, fratio);
      OMVG_CUDA(cudaGetLastError());
      OMVG_CUDA(cudaEventRecord(e1, c->stream));
      c->pending.emplace_back(e0, e1); c->tc_launches++; c->launches++;
    }
    cascade_compact_kernel<<<nb, FIN_THREADS, 0, c->stream>>>(c->d_pairs, c->d_k12, c->d_counts); OMVG_CUDA(cudaGetLastError());
    scan_counts_kernel<<<1, 1024, 0, c->stream>>>(c->d_counts, nb, c->d_offsets + p0, c->d_total); OMVG_CUDA(cudaGetLastError());
    c->launches += 2;
    uint64_t total = 0;
    OMVG_CUDA(cudaMemcpyAsync(&total, c->d_total, sizeof total, cudaMemcpyDeviceToHost, c->stream));
    OMVG_CUDA(cudaStreamSynchronize(c->stream));
    if (total > c->out_cap) {
      const size_t ncap = std::max<size_t>(total, c->out_cap * 2 + 1024);
      uint2 *n = nullptr; OMVG_CUDA(cudaMalloc(&n, ncap * sizeof(uint2)));
      if (c->d_out && c->total_last) OMVG_CUDA(cudaMemcpyAsync(n, c->d_out, c->total_last * sizeof(uint2), cudaMemcpyDeviceToDevice, c->stream));
      OMVG_CUDA(cudaStreamSynchronize(c->stream));
      if (c->d_out) cudaFree(c->d_out);
      c->d_out = n; c->out_cap = ncap;
    }
    compact_kernel<<<nb, 128, 0, c->stream>>>(c->d_k12, c->d_pairs, c->d_counts, c->d_offsets + p0, c->d_out); OMVG_CUDA(cudaGetLastError());
    c->launches++; c->total_last = total;
    p0 = p1;
  }
  c->have_result = true; return OMVG_OK;
}

// Validation aid (tests only): hash codes [count][4], bucket ids [count][6] and the zero-mean vector [128].
int omvg_match_cascade_debug_hash(omvg_match_ctx *c, uint32_t image, uint32_t *codes, uint16_t *bids, float *zero_mean) {
  if (!c || image >= c->n_images) return fail(OMVG_E_ARG, "bad arguments");
  if (!c->cascade_ready) return fail(OMVG_E_STATE, "omvg_match_cascade_prepare first");
  OMVG_CUDA(cudaSetDevice(c->device));
  const uint32_t n = c->counts[image];
  std::vector<uint4> hc(n), hb(n);
  if (n) { OMVG_CUDA(cudaMemcpyAsync(hc.data(), c->d_code + c->row0[image], n * sizeof(uint4), cudaMemcpyDeviceToHost, c->stream));
           OMVG_CUDA(cudaMemcpyAsync(hb.data(), c->d_bid + c->row0[image], n * sizeof(uint4), cudaMemcpyDeviceToHost, c->stream)); }
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  for (uint32_t r = 0; r < n; ++r) {
    if (codes) { codes[4 * r] = hc[r].x; codes[4 * r + 1] = hc[r].y; codes[4 * r + 2] = hc[r].z; codes[4 * r + 3] = hc[r].w; }
    if (bids) { bids[6 * r] = hb[r].x & 0xffff; bids[6 * r + 1] = hb[r].x >> 16; bids[6 * r + 2] = hb[r].y & 0xffff; bids[6 * r + 3] = hb[r].y >> 16; bids[6 * r + 4] = hb[r].z & 0xffff; bids[6 * r + 5] = hb[r].z >> 16; }
  }
  if (zero_mean) for (int k = 0; k < OMVG_DESC_LEN; ++k) zero_mean[k] = c->h_zm[k];
  return OMVG_OK;
}

int omvg_match_debug_top2_simt(omvg_match_ctx *c, uint32_t I, uint32_t J, int32_t *d1, uint32_t *i1, int32_t *d2) {
  if (!c || I >= c->n_images || J >= c->n_images) return fail(OMVG_E_ARG, "bad image");
  if (!c->prepared) return fail(OMVG_E_STATE, "prepare first");
  OMVG_CUDA(cudaSetDevice(c->device));
  const uint32_t nq = c->counts[J];
  if (nq == 0 || c->counts[I] < 2) return fail(OMVG_E_ARG, "need >=2 database rows and >=1 query");
  int32_t *dd1, *dd2; uint32_t *di1;
  OMVG_CUDA(cudaMalloc(&dd1, nq * 4)); OMVG_CUDA(cudaMalloc(&dd2, nq * 4)); OMVG_CUDA(cudaMalloc(&di1, nq * 4));
  top2_simt_kernel<<<nq, 128, 0, c->stream>>>(c->d_desc, c->d_norm, c->row0[I], c->counts[I], c->row0[J], dd1, di1, dd2);
  OMVG_CUDA(cudaGetLastError()); c->launches++;
  OMVG_CUDA(cudaMemcpyAsync(d1, dd1, nq * 4, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(i1, di1, nq * 4, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(d2, dd2, nq * 4, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  cudaFree(dd1); cudaFree(dd2); cudaFree(di1);
  return OMVG_OK;
}

int omvg_match_debug_top2_tc(omvg_match_ctx *c, uint32_t I, uint32_t J, int32_t *d1, uint32_t *g1, int32_t *ub2) {
  if (!c || I >= c->n_images || J >= c->n_images) return fail(OMVG_E_ARG, "bad image");
  if (!c->prepared) return fail(OMVG_E_STATE, "prepare first");
  OMVG_CUDA(cudaSetDevice(c->device));
  const uint32_t nq = c->counts[J], ndb = c->counts[I];
  if (nq == 0 || ndb < 2) return fail(OMVG_E_ARG, "need >=2 database rows and >=1 query");
  const uint32_t qt = (nq + TILE_Q - 1) / TILE_Q, dt = (ndb + TILE_DB - 1) / TILE_DB;
  std::vector<Unit> units;
  for (uint32_t t = 0; t < qt; ++t) units.push_back(Unit{c->row0[J] + t * TILE_Q, c->row0[I], dt, t * TILE_Q});
  int rc;
  if ((rc = ensure(c->d_k12, c->k12_cap, size_t(qt) * TILE_Q))) return rc;
  if ((rc = ensure(c->d_units, c->units_cap, units.size()))) return rc;
  OMVG_CUDA(cudaMemcpyAsync(c->d_units, units.data(), units.size() * sizeof(Unit), cudaMemcpyHostToDevice, c->stream));
  match_tc_kernel<<<std::min<uint32_t>(qt, c->n_sms), TC_THREADS, SMEM_BYTES, c->stream>>>(c->tmap, c->d_ckey, c->d_units, qt, c->d_k12);
  OMVG_CUDA(cudaGetLastError()); c->launches++;
  int32_t *dd1, *dd2; uint32_t *dg1;
  OMVG_CUDA(cudaMalloc(&dd1, nq * 4)); OMVG_CUDA(cudaMalloc(&dd2, nq * 4)); OMVG_CUDA(cudaMalloc(&dg1, nq * 4));
  decode_k12_kernel<<<(nq + 255) / 256, 256, 0, c->stream>>>(c->d_k12, c->d_norm, c->row0[J], nq, dd1, dg1, dd2);
  OMVG_CUDA(cudaGetLastError()); c->launches++;
  OMVG_CUDA(cudaMemcpyAsync(d1, dd1, nq * 4, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(g1, dg1, nq * 4, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaMemcpyAsync(ub2, dd2, nq * 4, cudaMemcpyDeviceToHost, c->stream));
  OMVG_CUDA(cudaStreamSynchronize(c->stream));
  cudaFree(dd1); cudaFree(dd2); cudaFree(dg1);
  c->have_result = false;
  return OMVG_OK;
}

}  // extern "C"
