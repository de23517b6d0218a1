// Tensor-core engine of the brute-force Hamming matcher (step 2 of the SOS front-end; same contract as the XOR+POPC
// engine in hamming.cu, which it replaces for large problems: FeatureMatcher.match on cv2.BFMatcher(NORM_HAMMING),
// reference omnistereo/camera_models.py:402-446).
//
// Hamming distance is a contraction: with the 256 descriptor bits mapped to signs s = +-1,
//     <s_q, s_t> = 256 - 2 d(q, t),
// so the all-pairs distance matrix of a (query, train) segment is an integer GEMM with K = 256.  Here it runs on the
// 5th-generation tensor cores (tcgen05.mma kind::i8, int32 accumulators in tensor memory: exact), and the part that bounds
// the POPC engine — ~26 integer instructions per descriptor pair — shrinks to reading the accumulator back and ONE max:
//
//   * operands are +-16 instead of +-1, so the accumulator holds 256 * <s_q, s_t>;
//   * 32 extra K columns carry bookkeeping through the same MMA: the query side holds the constants (16, 1, 127 x 30),
//     the train side (-(u >> 4), -(u & 15), pad x 30) with u = row of the train descriptor inside its 128-row tile and
//     pad = -128 for the padding rows of a ragged last tile, 0 otherwise.  The accumulator therefore is
//         acc = 256 * <s_q, s_t> - u - 487680 * [padding row]
//     i.e. ALREADY the packed sort key: max(acc) over a tile = smallest distance, ties to the lowest train row (OpenCV's
//     order), padding rows lose against everything — no index arithmetic, no masking in the epilogue;
//   * the epilogue thread that owns query row r (TMEM lane r) reads its 128 accumulators with tcgen05.ld and keeps the
//     running maximum (3-input integer max: half an instruction per pair); top-2 costs 3 instructions per pair.
//
// Data flow per work item (256 query rows x a range of train tiles; one CTA per SM at a time, warp-specialised):
//   expand kernel : descriptors -> "tile-ready" int8 images in global memory, 128 rows x 288 bytes per tile, stored in the
//                   canonical K-major no-swizzle UMMA layout (8-row x 16-byte core matrices), so that a tile is ONE
//                   contiguous 36 KB block
//   warp 0        : cp.async.bulk (TMA engine, mbarrier complete_tx) of the two query tiles, then a 4-stage ring of
//                   train tiles
//   warps 1, 3    : one lane of each issues 9 tcgen05.mma (M128 N128 K32) per train tile, one warp per query tile, into a double-buffered TMEM
//                   accumulator (2 buffers x 2 query tiles x 128 columns = all 512 columns); tcgen05.commit releases the
//                   shared-memory stage and publishes the accumulator
//   warp 2        : tensor-memory allocation
//   warps 4..11   : epilogue, one thread per (query tile, row)
// The per-split partial keys use the POPC engine's format and are merged by the same hamming_merge_kernel.
#include <cuda_bf16.h>

#include "sos_common.cuh"
#include "tc_common.cuh"

namespace sos_hamming_mma {

constexpr int TILE = 128;                        // rows per expanded tile = UMMA M = UMMA N
constexpr int KB = 288;                          // bytes of K per row: 256 sign bytes + 32 bookkeeping bytes
constexpr int CHUNKS = KB / 16;                  // 18 core-matrix columns
constexpr int GROUP_BYTES = CHUNKS * 128;        // one 8-row group: 18 core matrices of 8 x 16 bytes
constexpr int TILE_BYTES = (TILE / 8) * GROUP_BYTES;  // 36864
constexpr int THREADS = 384;
constexpr int smem_bytes(int stages) { return (2 + stages) * TILE_BYTES + 256; }
constexpr int PAD_DROP = 30 * 127 * 128;         // what the 30 pad columns subtract from a padding row's accumulator
constexpr int KEY_IDX_BITS = 22;                 // must match hamming.cu
constexpr uint32_t KEY_NONE = 0xFFFFFFFFu;
constexpr int ITEM_SPLIT_BITS = 6, ITEM_TILE_BITS = 10;   // item = seg << 16 | tile << 6 | split (hamming.cu)

// ---- expansion ------------------------------------------------------------------------------------------------------
// four descriptor bits -> four int8 values: bit 0 -> +16, bit 1 -> -16
__device__ __forceinline__ uint32_t expand4(uint32_t nib) {
  const uint32_t spread = (nib * 0x00204081u) & 0x01010101u;   // bit i -> LSB of byte i (the shifted copies never overlap)
  return 0x10101010u ^ (spread * 0xE0u);
}

// role 0: query rows (A operand), role 1: train rows (B operand).  Tile t of segment s lives at
// out + (s * tiles_per_seg + t) * TILE_BYTES; byte (row r, k) of a tile at (r / 8) * GROUP_BYTES + (k / 16) * 128 + (r % 8) * 16 + k % 16.
// One launch expands both roles (blockIdx.z); the nine 16-byte units of a thread are independent, so the loop is unrolled
// and all descriptor loads are in flight before the first store (the rolled loop was latency bound: 4 x 27 us per step).
struct ExpandArgs {
  const uint32_t* desc[2];
  const int32_t *start[2], *len[2];
  int max_rows[2], tiles_per_seg[2];
  uint8_t* out[2];
};

__global__ void __launch_bounds__(256)
expand_kernel(const ExpandArgs a) {
  const int role = blockIdx.z, seg = blockIdx.y, tile = blockIdx.x;
  if (tile >= a.tiles_per_seg[role]) return;
  const int n = min(a.len[role][seg], a.max_rows[role]);
  const int row0 = tile * TILE;
  if (row0 >= n) return;
  const uint32_t* d = a.desc[role] + (size_t)a.start[role][seg] * 8;
  uint8_t* tbase = a.out[role] + ((size_t)seg * a.tiles_per_seg[role] + tile) * TILE_BYTES;
  constexpr int UNITS = TILE * CHUNKS / 256;   // 9
  uint32_t bits[UNITS];
#pragma unroll
  for (int it = 0; it < UNITS; ++it) {
    const int u = threadIdx.x + it * 256;
    const int r8 = u & 7, chunk = (u >> 3) % CHUNKS, rg = u / (8 * CHUNKS);
    const int row = row0 + rg * 8 + r8;
    bits[it] = (chunk < 16 && row < n) ? (__ldg(d + (size_t)row * 8 + (chunk >> 1)) >> ((chunk & 1) * 16)) & 0xFFFFu : 0u;
  }
#pragma unroll
  for (int it = 0; it < UNITS; ++it) {
    const int u = threadIdx.x + it * 256;
    const int r8 = u & 7, chunk = (u >> 3) % CHUNKS, rg = u / (8 * CHUNKS);
    const int r = rg * 8 + r8, row = row0 + r;
    const bool valid = row < n;
    uint4 v;
    if (chunk < 16) {
      v.x = expand4(bits[it] & 15u);
      v.y = expand4((bits[it] >> 4) & 15u);
      v.z = expand4((bits[it] >> 8) & 15u);
      v.w = expand4(bits[it] >> 12);
      if (!valid) v = make_uint4(0u, 0u, 0u, 0u);          // padding rows: <s_q, s_t> = 0
    } else if (role == 0) {
      v = make_uint4(0x7F7F7F7Fu, 0x7F7F7F7Fu, 0x7F7F7F7Fu, 0x7F7F7F7Fu);
      if (chunk == 16) v.x = 0x7F7F0110u;                  // bytes (16, 1, 127, 127)
    } else {
      const uint32_t pad = valid ? 0u : 0x80808080u;       // -128 in every pad column of a padding row
      v = make_uint4(pad, pad, pad, pad);
      if (chunk == 16) {
        const uint32_t hi = (uint32_t)(-(r >> 4)) & 0xFFu, lo = (uint32_t)(-(r & 15)) & 0xFFu;
        v.x = (pad & 0xFFFF0000u) | (lo << 8) | hi;
      }
    }
    *(uint4*)(tbase + (size_t)rg * GROUP_BYTES + chunk * 128 + r8 * 16) = v;
  }
}

using namespace sos_tc;
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr) { return sos_tc::smem_desc(addr, (uint32_t)GROUP_BYTES); }
// instruction descriptor: D = S32 (2 << 4), A = B = signed int8 (1 << 7, 1 << 10), both K-major, N = 128, M = 128
constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TILE >> 3) << 17) | ((uint32_t)(TILE >> 4) << 24);
// the float-descriptor L2 engine: D = F32 (1 << 4), A = B = BF16 (1 << 7, 1 << 10), both K-major, N = 128, M = 128
constexpr uint32_t IDESC_L2 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TILE >> 3) << 17) | ((uint32_t)(TILE >> 4) << 24);

template <bool TOP2>
__device__ __forceinline__ void reduce32(const int (&v)[32], int& m0, int& m1) {
  if (TOP2) {
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      m1 = max(m1, min(m0, v[i]));
      m0 = max(m0, v[i]);
    }
  } else {
    int a = m0;
#pragma unroll
    for (int i = 0; i < 32; i += 2) a = __vimax3_s32(a, v[i], v[i + 1]);
    m0 = a;
  }
}

// accumulator of (query row, train row u of tile `tile`) -> the POPC engine's key (distance << 22 | train row of the segment)
__device__ __forceinline__ uint32_t acc_to_key(int acc, int tile) {
  const int dot = (acc + 255) >> 8;              // acc = 256 * dot - u with 0 <= u < 128
  if (dot < -256) return KEY_NONE;               // padding row (or no train row at all)
  const int u = 256 * dot - acc;
  return ((uint32_t)((256 - dot) >> 1) << KEY_IDX_BITS) | (uint32_t)(tile * TILE + u);
}

// ---- float-descriptor L2 engine: epilogue pieces ------------------------------------------------------------------------
// accumulator (float32, an exact integer) = 2 <q, t> - |t|^2 of (query row, train row u); the largest one is the nearest
// neighbour.  key = acc * 128 + (127 - u): max(key) = largest accumulator, ties to the lowest train row.
constexpr int L2_PAD_BELOW = -12000000;   // valid accumulators are >= -128 * 255^2 = -8323200; padding rows sit at -16.7 M
template <bool TOP2>
__device__ __forceinline__ void reduce32_l2(const int (&v)[32], int col0, int& m0, int& m1) {
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int k = __float2int_rn(__int_as_float(v[i])) * 128 + (127 - (col0 + i));
    if (TOP2) m1 = max(m1, min(m0, k));
    m0 = max(m0, k);
  }
}
constexpr unsigned long long KEY64_NONE = ~0ull;
// key of the tile -> (squared distance << 32 | train row of the segment); nq = |q|^2 of this thread's query row
__device__ __forceinline__ unsigned long long l2_key(int key, int tile, int nq) {
  const int acc = key >> 7;                          // floor: key = acc * 128 + low, 0 <= low < 128
  if (acc < L2_PAD_BELOW) return KEY64_NONE;
  const int u = 127 - (key & 127);
  return ((unsigned long long)(uint32_t)(nq - acc) << 32) | (unsigned long long)(uint32_t)(tile * TILE + u);
}

// ---- general float-descriptor L2 engine (KIND_L2F): epilogue pieces -------------------------------------------------------
// The accumulator approximates 2 <q, t> - |t|^2 (float32, not exact: see the band derivation above l2f_expand_kernel).  Each
// epilogue thread keeps the K = 3 (2 for 1-NN) largest accumulators of its query row in descending order, ties to the lowest
// train row: columns and tiles arrive in increasing train-row order and a value only moves past a STRICTLY smaller one.
// `!(v <= m[K-1])` also catches NaN and +inf: such a row is flagged (`bad`) and its keys are never used.
// row0 = train row (of the segment) of v[0]; rows >= nt are the padding of a ragged last tile (accumulator 0): skipped.
template <int K>
__device__ __forceinline__ void reduce32_l2f(const int (&v)[32], int row0, int nt, float (&m)[3], int (&c)[3], int& bad) {
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const float x = __int_as_float(v[i]);
    if (!(x <= m[K - 1])) {
      if (!(x < INFINITY)) bad = 1;
      else if (row0 + i < nt) {
        const int col = row0 + i;
        if (x > m[0]) {
          if (K == 3) { m[2] = m[1]; c[2] = c[1]; }
          m[1] = m[0]; c[1] = c[0]; m[0] = x; c[0] = col;
        } else if (K == 3 && x > m[1]) {
          m[2] = m[1]; c[2] = c[1]; m[1] = x; c[1] = col;
        } else {
          m[K - 1] = x; c[K - 1] = col;
        }
      }
    }
  }
}
// (accumulator, train row of the segment) -> 64-bit key, smaller = larger accumulator, ties to the lowest row
__device__ __forceinline__ unsigned long long l2f_key(float acc, int row) {
  const uint32_t b = __float_as_uint(acc);
  const uint32_t ord = (b & 0x80000000u) ? ~b : (b | 0x80000000u);   // ascending with acc
  return ((unsigned long long)~ord << 32) | (uint32_t)row;
}

struct Args {
  const int32_t* a_norm;   // KIND_L2: |q|^2 per expanded query row [n_seg, q_tiles_per_seg * 128]
  const uint8_t *a_exp, *b_exp;
  const int32_t *q_len, *t_len;
  int max_nq, max_nt, splits, q_tiles_per_seg, t_tiles_per_seg;
  const uint32_t* items;
  const int32_t* n_items;
  void* partial;           // uint2 (Hamming keys), ulonglong2 (L2 keys) or 2 x ulonglong2 (L2F: 3 keys, flag) per
                           // (segment, query row, split)
  int dim, nsub;           // KIND_L2F: descriptor length; 288-byte sub-tiles per 128-row tile (1: dim <= 64, 2: dim <= 128)
};

// Work item -> (segment, first query row, split, train tiles [tile_begin, tile_begin + n_iter))
struct Item {
  int seg, q_tile, split, nq, tile_begin, n_iter;
};
__device__ __forceinline__ Item decode_item(const Args& a, uint32_t item) {
  Item it;
  it.seg = (int)(item >> 16);
  it.q_tile = (int)((item >> ITEM_SPLIT_BITS) & ((1u << ITEM_TILE_BITS) - 1u));   // 256 query rows
  it.split = (int)(item & ((1u << ITEM_SPLIT_BITS) - 1u));
  it.nq = min(a.q_len[it.seg], a.max_nq);
  const int nt = min(a.t_len[it.seg], a.max_nt);
  const int t_tiles = (nt + TILE - 1) / TILE;
  const int chunk_tiles = (t_tiles + a.splits - 1) / a.splits;
  it.tile_begin = min(t_tiles, it.split * chunk_tiles);
  it.n_iter = min(t_tiles, it.tile_begin + chunk_tiles) - it.tile_begin;
  return it;
}

// A CTA walks the work list with stride gridDim.x (launched either with one CTA per item, or PERSISTENT with one CTA per SM:
// see the host side).  Barriers, the tensor-memory allocation and the three pipelines (train-tile ring, accumulator double
// buffer, query tiles) live across items, so in the persistent shape the tensor pipe only idles while the next item's query
// tiles land (the train tiles of the next item are already streaming into the ring by then).  The roles agree on every
// counter because they walk the same items in the same order:
//   t  = train tiles consumed so far by this CTA -> ring stage t % STAGES, accumulator buffer t & 1
//   ic = items with work so far                  -> phase of the query-tile barriers
template <bool TOP2, int STAGES, int KIND>
__global__ void __launch_bounds__(THREADS, 1) mma_kernel(Args a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int n_items = *a.n_items;
  if ((int)blockIdx.x >= n_items) return;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint8_t* sA = smem;
  uint8_t* sB = smem + 2 * TILE_BYTES;
  uint64_t* bars = (uint64_t*)(smem + (2 + STAGES) * TILE_BYTES);
  // bars: FULL + s (train stage landed), EMPTY + s (stage consumed), TFULL + b (accumulator complete), TEMPTY + b
  // (accumulator drained), AFULL (query tiles landed), AEMPTY (query tiles no longer read by the tensor core)
  constexpr int FULL = 0, EMPTY = STAGES, TFULL = 2 * STAGES, TEMPTY = 2 * STAGES + 2, AFULL = 2 * STAGES + 4, AEMPTY = 2 * STAGES + 5;
  uint32_t* tmem_slot = (uint32_t*)(bars + AEMPTY + 1);
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };

  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(BAR(FULL + i), 1); mbar_init(BAR(EMPTY + i), 2); }   // EMPTY, TFULL, AEMPTY: one commit per MMA warp
    mbar_init(BAR(TFULL), 2); mbar_init(BAR(TFULL + 1), 2);
    mbar_init(BAR(TEMPTY), 8); mbar_init(BAR(TEMPTY + 1), 8);
    mbar_init(BAR(AFULL), 1); mbar_init(BAR(AEMPTY), 2);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (KIND == KIND_L2F && warp == 0) {
    // producer of the general float engine: a 128-row tile is nsub 288-byte sub-tiles (36 KB each); the two query tiles of
    // an item take 2 nsub of the six 36 KB buffers, the ring of train sub-tiles the remaining 6 - 2 nsub
    const int nsub = a.nsub, ns = STAGES + 2 - 2 * nsub;
    uint32_t r = 0, ic = 0;
    for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
      const Item it = decode_item(a, a.items[w]);
      if (it.n_iter <= 0) continue;
      const uint8_t* gb = a.b_exp + ((size_t)it.seg * a.t_tiles_per_seg + it.tile_begin) * nsub * TILE_BYTES;
      uint8_t* sB2 = smem + 2 * nsub * TILE_BYTES;
      auto load_b = [&](int k) {                 // k-th sub-tile of this item
        const uint32_t s = r % ns;
        mbar_wait(BAR(EMPTY + s), ((r / ns) & 1) ^ 1);
        if (elect_one()) {
          mbar_expect_tx(BAR(FULL + s), TILE_BYTES);
          const uint32_t dst = smem_u32(sB2) + s * TILE_BYTES;
#pragma unroll
          for (int p = 0; p < 4; ++p)
            bulk_g2s(dst + p * (TILE_BYTES / 4), gb + (size_t)k * TILE_BYTES + (size_t)p * (TILE_BYTES / 4), TILE_BYTES / 4, BAR(FULL + s));
        }
        __syncwarp();
        ++r;
      };
      const int n_sub = it.n_iter * nsub, pre = min(n_sub, ns);
      for (int k = 0; k < pre; ++k) load_b(k);
      mbar_wait(BAR(AEMPTY), (ic & 1) ^ 1);
      const uint8_t* ga = a.a_exp + ((size_t)it.seg * a.q_tiles_per_seg + (size_t)it.q_tile * 2) * nsub * TILE_BYTES;
      if (elect_one()) {
        mbar_expect_tx(BAR(AFULL), 2u * nsub * TILE_BYTES);
        for (int p = 0; p < 8 * nsub; ++p) bulk_g2s(smem_u32(sA) + p * (TILE_BYTES / 4), ga + (size_t)p * (TILE_BYTES / 4), TILE_BYTES / 4, BAR(AFULL));
      }
      __syncwarp();
      ++ic;
      for (int k = pre; k < n_sub; ++k) load_b(k);
    }
  } else if (KIND == KIND_L2F && (warp == 1 || warp == 3)) {
    // MMA issuers of the general float engine.  Sub-tile j of a row holds [hi (64) | mid (64) | 16 more] bf16 of the values
    // 64 j .. 64 j + 63; the products hi*hi, hi*mid and mid*hi of each 16-value block come from the same two tiles at
    // different K offsets (descriptor + 16 per 256 bytes), and sub-tile 0 adds the |t|^2 columns: for dim = 64 that is
    // 4 x 3 + 1 = 13 instructions per tile pair, for dim = 128 25, against the integer engine's 9.
    const int qt = warp == 1 ? 0 : 1, nsub = a.nsub, ns = STAGES + 2 - 2 * nsub;
    uint8_t* sB2 = smem + 2 * nsub * TILE_BYTES;
    uint32_t t = 0, r = 0, ic = 0;
    for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
      const Item it = decode_item(a, a.items[w]);
      if (it.n_iter <= 0) continue;
      mbar_wait(BAR(AFULL), ic & 1);
      ++ic;
      for (int k = 0; k < it.n_iter; ++k, ++t) {
        const uint32_t b = t & 1;
        mbar_wait(BAR(TEMPTY + b), ((t >> 1) & 1) ^ 1);
        for (int j = 0; j < nsub; ++j, ++r) {
          const uint32_t s = r % ns;
          mbar_wait(BAR(FULL + s), (r / ns) & 1);
          tc_fence_after();
          const uint64_t da = smem_desc(smem_u32(sA) + (qt * nsub + j) * TILE_BYTES);
          const uint64_t db = smem_desc(smem_u32(sB2) + s * TILE_BYTES);
          const int nk = (min(64, a.dim - 64 * j) + 15) >> 4;
          const uint32_t d = tmem + (b * 2 + qt) * TILE;
          if (elect_one()) {
            if (j == 0) tc_mma<KIND>(d, da + 128u, db + 128u, IDESC_L2, 0u);     // 1 x (-|t|^2 pieces)
            for (int kk = 0; kk < nk; ++kk) {
              tc_mma<KIND>(d, da + (uint64_t)(16 * kk), db + (uint64_t)(16 * kk), IDESC_L2, 1u);            // hi * hi
              tc_mma<KIND>(d, da + (uint64_t)(16 * kk), db + (uint64_t)(16 * (4 + kk)), IDESC_L2, 1u);      // hi * mid
              tc_mma<KIND>(d, da + (uint64_t)(16 * (4 + kk)), db + (uint64_t)(16 * kk), IDESC_L2, 1u);      // mid * hi
            }
            tc_commit(BAR(EMPTY + s));
            if (j == nsub - 1) tc_commit(BAR(TFULL + b));
          }
          __syncwarp();
        }
      }
      if (elect_one()) tc_commit(BAR(AEMPTY));
      __syncwarp();
    }
  } else if (warp == 0) {
    // producer: the whole (converged) warp walks the items, the elected lane issues the copies (tc_common.cuh: elect_one)
    uint32_t t = 0, ic = 0;
    for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
      const Item it = decode_item(a, a.items[w]);
      if (it.n_iter <= 0) continue;
      const uint8_t* gb = a.b_exp + ((size_t)it.seg * a.t_tiles_per_seg + it.tile_begin) * TILE_BYTES;
      auto load_b = [&](int k) {
        const uint32_t s = t % STAGES;
        mbar_wait(BAR(EMPTY + s), ((t / STAGES) & 1) ^ 1);
        if (elect_one()) {
          mbar_expect_tx(BAR(FULL + s), TILE_BYTES);
          const uint32_t dst = smem_u32(sB) + s * TILE_BYTES;
#pragma unroll
          for (int p = 0; p < 4; ++p)
            bulk_g2s(dst + p * (TILE_BYTES / 4), gb + (size_t)k * TILE_BYTES + (size_t)p * (TILE_BYTES / 4), TILE_BYTES / 4, BAR(FULL + s));
        }
        __syncwarp();
        ++t;
      };
      // the first train tiles of this item go into the ring as soon as stages free up, i.e. while the previous item is still
      // being multiplied; only then wait for the tensor core to be done with the previous item's query tiles and fetch ours
      const int pre = min(it.n_iter, STAGES);
      for (int k = 0; k < pre; ++k) load_b(k);
      mbar_wait(BAR(AEMPTY), (ic & 1) ^ 1);
      const uint8_t* ga = a.a_exp + ((size_t)it.seg * a.q_tiles_per_seg + (size_t)it.q_tile * 2) * TILE_BYTES;
      if (elect_one()) {
        mbar_expect_tx(BAR(AFULL), 2u * TILE_BYTES);
#pragma unroll
        for (int p = 0; p < 8; ++p) bulk_g2s(smem_u32(sA) + p * (TILE_BYTES / 4), ga + (size_t)p * (TILE_BYTES / 4), TILE_BYTES / 4, BAR(AFULL));
      }
      __syncwarp();
      ++ic;
      for (int k = pre; k < it.n_iter; ++k) load_b(k);
    }
  } else if (warp == 1 || warp == 3) {
    // MMA issuers: converged warps, elected lane — issued from `if (lane == 0)` every tcgen05.mma was wrapped in an
    // elect / broadcast loop of ~13 instructions and the issuing thread, not the tensor pipe, set the pace.  Two of them (on
    // different sub-partitions), one per query tile = accumulator: the issue loop of a single warp sharing its scheduler
    // with busy epilogue warps was still slower than the tensor pipe (found on the score engine, score_mma.cuh).
    const int qt = warp == 1 ? 0 : 1;
    const uint64_t da = smem_desc(smem_u32(sA) + qt * TILE_BYTES);
    uint32_t t = 0, ic = 0;
    for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
      const Item it = decode_item(a, a.items[w]);
      if (it.n_iter <= 0) continue;
      mbar_wait(BAR(AFULL), ic & 1);
      ++ic;
      for (int k = 0; k < it.n_iter; ++k, ++t) {
        const uint32_t s = t % STAGES, b = t & 1;
        mbar_wait(BAR(TEMPTY + b), ((t >> 1) & 1) ^ 1);    // the epilogue has drained this accumulator buffer
        mbar_wait(BAR(FULL + s), (t / STAGES) & 1);        // the train tile has landed
        tc_fence_after();
        const uint64_t db = smem_desc(smem_u32(sB) + s * TILE_BYTES);
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < KB / 32; ++kk)
            tc_mma<KIND>(tmem + (b * 2 + qt) * TILE, da + (uint64_t)(16 * kk), db + (uint64_t)(16 * kk), KIND == KIND_L2 ? IDESC_L2 : IDESC, kk > 0);
          tc_commit(BAR(EMPTY + s));    // shared-memory stage free once both warps' MMAs have read it
          tc_commit(BAR(TFULL + b));    // this query tile's accumulator complete
        }
        __syncwarp();
      }
      if (elect_one()) tc_commit(BAR(AEMPTY));         // every MMA of this item has read the query tiles
      __syncwarp();
    }
  } else if (warp >= 4) {
    const int g = (warp - 4) >> 2, quarter = warp & 3;   // a warp may only touch the TMEM lanes of its quarter
    uint32_t t = 0;
    for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
      const Item it = decode_item(a, a.items[w]);
      const int row = it.q_tile * 256 + g * TILE + quarter * 32 + lane;
      uint32_t k0 = KEY_NONE, k1 = KEY_NONE;
      unsigned long long w0 = KEY64_NONE, w1 = KEY64_NONE;
      float fm[3] = {-INFINITY, -INFINITY, -INFINITY};   // KIND_L2F: running top-K over the item, train rows fc
      int fc[3] = {-1, -1, -1}, fbad = 0;
      const int nt_seg = KIND == KIND_L2F ? min(a.t_len[it.seg], a.max_nt) : 0;
      int nq_norm = 0;
      if (KIND == KIND_L2 && it.n_iter > 0) nq_norm = a.a_norm[(size_t)it.seg * a.q_tiles_per_seg * TILE + row];
      for (int k = 0; k < it.n_iter; ++k, ++t) {
        const uint32_t b = t & 1;
        mbar_wait(BAR(TFULL + b), (t >> 1) & 1);
        tc_fence_after();
        const uint32_t taddr = tmem + ((uint32_t)(quarter * 32) << 16) + (b * 2 + g) * TILE;
        int m0 = INT_MIN, m1 = INT_MIN;
        int va[32], vb[32];
        auto reduce = [&](const int (&v)[32], int col0) {
          if (KIND == KIND_L2F) reduce32_l2f<TOP2 ? 3 : 2>(v, (it.tile_begin + k) * TILE + col0, nt_seg, fm, fc, fbad);
          else if (KIND == KIND_L2) reduce32_l2<TOP2>(v, col0, m0, m1);
          else reduce32<TOP2>(v, m0, m1);
        };
        tmem_ld32(taddr, va);
        tmem_ld_wait(va);
        tmem_ld32(taddr + 32, vb);          // in flight while va is reduced
        reduce(va, 0);
        tmem_ld_wait(vb);
        tmem_ld32(taddr + 64, va);
        reduce(vb, 32);
        tmem_ld_wait(va);
        tmem_ld32(taddr + 96, vb);
        reduce(va, 64);
        tmem_ld_wait(vb);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(BAR(TEMPTY + b));     // buffer b may be overwritten
        reduce(vb, 96);
        const int tile = it.tile_begin + k;
        if (KIND == KIND_L2) {
          const unsigned long long key0 = l2_key(m0, tile, nq_norm);
          if (TOP2) {
            const unsigned long long key1 = m1 == INT_MIN ? KEY64_NONE : l2_key(m1, tile, nq_norm);
            w1 = min(w1, max(w0, key0));
            w0 = min(w0, key0);
            w1 = min(w1, key1);
          } else {
            w0 = min(w0, key0);
          }
        } else if (KIND == KIND_HAMMING) {          // (KIND_L2F: the running top-K is already up to date)
          const uint32_t key0 = acc_to_key(m0, tile);
          if (TOP2) {
            const uint32_t key1 = acc_to_key(m1, tile);
            k1 = min(k1, max(k0, key0));                    // merge two sorted pairs
            k0 = min(k0, key0);
            k1 = min(k1, key1);
          } else {
            k0 = min(k0, key0);
          }
        }
      }
      // (no train rows in this split: the keys stay "none")
      if (row < it.nq) {
        const size_t o = ((size_t)it.seg * a.max_nq + row) * a.splits + it.split;
        if (KIND == KIND_L2F) {
          unsigned long long f[3];
#pragma unroll
          for (int i = 0; i < 3; ++i) f[i] = fc[i] < 0 ? KEY64_NONE : l2f_key(fm[i], fc[i]);
          ((ulonglong2*)a.partial)[2 * o] = make_ulonglong2(f[0], f[1]);
          ((ulonglong2*)a.partial)[2 * o + 1] = make_ulonglong2(TOP2 ? f[2] : KEY64_NONE, (unsigned long long)fbad);
        } else if (KIND == KIND_L2) ((ulonglong2*)a.partial)[o] = make_ulonglong2(w0, w1);
        else ((uint2*)a.partial)[o] = make_uint2(k0, k1);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
}

// ---- float-descriptor L2 engine: expansion ---------------------------------------------------------------------------
// Float descriptors whose values are integers in [0, 255] (what cv2's SIFT returns) are exactly representable in bfloat16,
// their dot products (< 2^24) exactly in the float32 accumulator: |q - t|^2 = |q|^2 + |t|^2 - 2 <q, t> comes out of the
// tensor core as an exact integer.  A tile has the Hamming engine's geometry: 144 bf16 = 288 bytes per row; elements 0..127
// hold 2 q (query role) or t (train role), elements 128..130 carry the norm: (1, 256, 65536) against minus the base-256
// digits of |t|^2, so that the accumulator is 2 <q, t> - |t|^2; padding rows get the digits (255, 255, 255).
// One block per tile; every warp first sums the squares of 16 rows.  flag[0] is set when a value is not an integer in [0, 255].
__global__ void __launch_bounds__(256)
expand_l2_kernel(const float* __restrict__ desc, int dim, const int32_t* __restrict__ start, const int32_t* __restrict__ len,
                 int max_rows, int tiles_per_seg, int role, uint8_t* __restrict__ out, int32_t* __restrict__ norms,
                 int32_t* __restrict__ flag) {
  __shared__ int snorm[TILE];
  const int seg = blockIdx.y, tile = blockIdx.x;
  const int n = min(len[seg], max_rows);
  const int row0 = tile * TILE;
  if (row0 >= n) return;
  const float* d = desc + (size_t)start[seg] * dim;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  bool bad = false;
  for (int r = warp; r < TILE; r += 8) {
    const int row = row0 + r;
    int acc = 0;
    if (row < n)
      for (int k = lane; k < dim; k += 32) {
        const float v = __ldg(d + (size_t)row * dim + k);
        const int iv = (int)v;
        bad |= !(v >= 0.f && v <= 255.f && (float)iv == v);
        acc += iv * iv;
      }
    acc = __reduce_add_sync(0xFFFFFFFFu, acc);
    if (lane == 0) snorm[r] = row < n ? acc : -1;
  }
  if (bad) atomicOr(flag, 1);
  __syncthreads();
  uint8_t* tbase = out + ((size_t)seg * tiles_per_seg + tile) * TILE_BYTES;
  if (role == 0 && norms)
    for (int r = threadIdx.x; r < TILE; r += 256) norms[((size_t)seg * tiles_per_seg + tile) * TILE + r] = max(snorm[r], 0);
  const float scale = role == 0 ? 2.f : 1.f;
  for (int u = threadIdx.x; u < TILE * CHUNKS; u += 256) {
    const int r8 = u & 7, chunk = (u >> 3) % CHUNKS, rg = u / (8 * CHUNKS);
    const int r = rg * 8 + r8, row = row0 + r;
    const bool valid = row < n;
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    if (chunk < 16) {                       // elements 8 chunk .. 8 chunk + 7
      if (valid) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int k = chunk * 8 + e;
          const float v = k < dim ? scale * __ldg(d + (size_t)row * dim + k) : 0.f;
          w[e >> 1] |= (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v)) << (16 * (e & 1));
        }
      }
    } else if (chunk == 16) {               // elements 128 .. 135: the norm digits
      float e0, e1, e2;
      if (role == 0) { e0 = 1.f; e1 = 256.f; e2 = 65536.f; }
      else {
        const int nt = valid ? snorm[r] : 0xFFFFFF;
        e0 = -(float)(nt & 255); e1 = -(float)((nt >> 8) & 255); e2 = -(float)((nt >> 16) & 255);
      }
      w[0] = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(e0)) | ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(e1)) << 16);
      w[1] = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(e2));
    }
    *(uint4*)(tbase + (size_t)rg * GROUP_BYTES + chunk * 128 + r8 * 16) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// ---- general float-descriptor L2 engine (sos_l2f_top2): expansion, band, decision -------------------------------------
// Contract: d^2(q, t) = sum_k (double(q_k) - double(t_k))^2 in float64, k = 0 .. dim-1 in order, no FMA; the two smallest,
// ties to the lowest train row; distance = float32(sqrt(d^2)).  The tensor cores only rank: every float32 value x is split
// into hi = bf16(x) and mid = bf16(x - hi) (x - hi is exact in float32); the query side carries 2 q (exact), and the GEMM forms
// hi*hi + hi*mid + mid*hi per component plus 1 x (-|t|^2 in three bfloat16 pieces), so that the float32 accumulator is
//     a(q, t) ~ 2 <q, t> - |t|^2 = |q|^2 - d^2(q, t)          (larger = nearer).
// Pieces below 2^-126 (bfloat16 subnormals) are set to 0 by the expansion, so the tensor core never sees a subnormal operand.
//
// Band: |a - (|q|^2 - d2_ref)| <= B_q, with M = the segment's largest |t| and u = 2^-24 (derivation; terms of |q| M, M^2,
// |q|^2, |q| + M and a constant):
//   * split: x = hi + mid + lo with |mid| <= 2^-8 (1 + 2^-8) |x| and |lo| <= 2^-16 |x|; the dropped products hi*lo, mid*mid,
//     lo*hi (and three of order 2^-24) are below 3.02 * 2^-16 |q_k| |t_k|; times 2 (the query carries 2 q) and summed with
//     Cauchy-Schwarz: 6.05 * 2^-16 |q| M = 9.23e-5 |q| M;
//   * flushed pieces: each value loses at most 2^-125 more, i.e. 2.01 * 2^-125 sqrt(dim) (2 |q| + M) <= 2^-120.5 (|q| + M);
//   * |t|^2 (summed in float64) minus its three bfloat16 pieces: <= 1.0002 * 2^-24 M^2 + 3 * 2^-126;
//   * accumulation — the HARDWARE ASSUMPTION of score_mma.cuh, not documented by NVIDIA: each tcgen05.mma kind::f16 adds the
//     exact sum of its 16 products to the float32 accumulator and rounds once, to nearest (e = u) or toward zero (e = 2u);
//     every partial sum is at most T = sum |terms| <= 2.032 |q| M + 1.004 M^2, and there are m <= 25 instructions
//     (3 ceil(dim / 16) + 1): m e T <= 6.05e-6 |q| M + 2.99e-6 M^2 toward zero (half that to nearest); products and
//     roundings that land below 2^-126 may be flushed: <= (3 dim + 28) 2^-126 < 2^-117;
//   * the float64 reference itself: |d2_ref - d^2| <= 131 * 2^-53 d^2 <= 1.5e-14 (|q| + M)^2, and |q|^2 (float64, any
//     order) is off by <= 1.5e-14 |q|^2.
// Worst case, toward zero: 9.83e-5 |q| M + 3.05e-6 M^2 + 4.5e-14 |q|^2 + 2^-120.5 (|q| + M) + 2^-117 (to nearest 9.52e-5 |q| M
// + 1.56e-6 M^2); the constants below hold it with 2 % / 24 % / 55 % / 80 % / 50 % to spare, and the 2 % also covers the
// float64 roundings of the test itself.  tests/test_l2f_split_cpu.py checks a NumPy model of this arithmetic against the band.
// Overflow: with T < 2^126 and |q| < 2^125 no product, piece or partial sum can leave the float32 range; otherwise the
// query is uncertain.  A query is CERTAIN when a1 - a2 > 2 B_q (and, for the second neighbour, a2 - a3 > 2 B_q) over its three
// largest accumulators: then the float64 reference orders those rows the same way, and only the winners' d^2 are computed
// in float64.  Every other query is re-decided by a float64 brute force over its segment (l2f_redecide_kernel).
constexpr double L2F_C_QT = 1e-4, L2F_C_TT = 4e-6, L2F_C_QQ = 1e-13;
constexpr double L2F_C_LIN = 3.4694469519536142e-36 /* 2^-118 */, L2F_C_ABS = 1.3877787807814457e-35 /* 2^-116 */;

__device__ __forceinline__ float l2f_flush(float v) { return fabsf(v) < 1.17549435e-38f ? 0.f : v; }
__device__ __forceinline__ float l2f_bf16(float v) { return l2f_flush(__bfloat162float(__float2bfloat16_rn(v))); }

// One block per (tile, segment); role 0: query rows (A operand, 2 q), role 1: train rows (B operand).  Tile t of segment s is
// nsub consecutive 36 KB sub-tiles at out + ((s * tiles_per_seg + t) * nsub + j) * TILE_BYTES, each in the canonical layout of
// expand_kernel: 144 bf16 per row = [hi of values 64 j .. 64 j + 63 | their mid | 16 columns]; the 16 columns of sub-tile 0
// are (1, 1, 1, 0 ...) for queries and (-n1, -n2, -n3, 0 ...) for train rows, |t|^2 ~ n1 + n2 + n3.  Padding rows are zero.
// norm2: role 0: |q|^2 per expanded query row [n_seg, tiles_per_seg * 128]; role 1: max |t|^2 of the segment, as the bits of a
// non-negative double (atomicMax).  flag[0] is set when a value is NaN or +-Inf.
__global__ void __launch_bounds__(256)
l2f_expand_kernel(const float* __restrict__ desc, int dim, const int32_t* __restrict__ start, const int32_t* __restrict__ len,
                  int max_rows, int tiles_per_seg, int nsub, int role, uint8_t* __restrict__ out, double* __restrict__ norm2,
                  int32_t* __restrict__ flag) {
  __shared__ double snorm[TILE];
  const int seg = blockIdx.y, tile = blockIdx.x;
  const int n = min(len[seg], max_rows);
  const int row0 = tile * TILE;
  if (row0 >= n) return;
  const float* d = desc + (size_t)start[seg] * dim;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  bool bad = false;
  for (int r = warp; r < TILE; r += 8) {
    const int row = row0 + r;
    double acc = 0.0;
    if (row < n)
      for (int k = lane; k < dim; k += 32) {
        const float v = __ldg(d + (size_t)row * dim + k);
        bad |= !(fabsf(v) <= 3.40282347e38f);
        acc += (double)v * (double)v;
      }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, off);
    if (lane == 0) snorm[r] = acc;
  }
  if (bad) atomicOr(flag, 1);
  __syncthreads();
  if (role == 0) {
    for (int r = threadIdx.x; r < TILE; r += 256) norm2[((size_t)seg * tiles_per_seg + tile) * TILE + r] = snorm[r];
  } else if (warp == 0) {
    double m = fmax(fmax(snorm[lane], snorm[lane + 32]), fmax(snorm[lane + 64], snorm[lane + 96]));
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = fmax(m, __shfl_xor_sync(0xFFFFFFFFu, m, off));
    if (lane == 0) atomicMax((unsigned long long*)norm2 + seg, (unsigned long long)__double_as_longlong(m));
  }
  const float scale = role == 0 ? 2.f : 1.f;
  for (int j = 0; j < nsub; ++j) {
    uint8_t* tbase = out + (((size_t)seg * tiles_per_seg + tile) * nsub + j) * TILE_BYTES;
    for (int u = threadIdx.x; u < TILE * CHUNKS; u += 256) {
      const int r8 = u & 7, chunk = (u >> 3) % CHUNKS, rg = u / (8 * CHUNKS);
      const int r = rg * 8 + r8, row = row0 + r;
      uint32_t w[4] = {0u, 0u, 0u, 0u};
      if (row < n && chunk < 16) {            // hi (chunks 0..7) or mid (8..15) of values 64 j + 8 (chunk % 8) + 0..7
        const int k0 = 64 * j + (chunk & 7) * 8;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int k = k0 + e;
          const float x = k < dim ? __ldg(d + (size_t)row * dim + k) : 0.f;
          const float hi = l2f_bf16(x);
          const float p = chunk < 8 ? hi : l2f_bf16(x - hi);
          w[e >> 1] |= (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(scale * p)) << (16 * (e & 1));
        }
      } else if (row < n && chunk == 16 && j == 0) {
        float e0 = 1.f, e1 = 1.f, e2 = 1.f;
        if (role == 1) {
          const double nt = snorm[r];
          const float n1 = l2f_bf16((float)nt);
          const double r1 = nt - (double)n1;
          const float n2 = l2f_bf16((float)r1);
          const float n3 = l2f_bf16((float)(r1 - (double)n2));
          e0 = -n1; e1 = -n2; e2 = -n3;
        }
        w[0] = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(e0)) | ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(e1)) << 16);
        w[1] = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(e2));
      }
      *(uint4*)(tbase + (size_t)rg * GROUP_BYTES + chunk * 128 + r8 * 16) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  }
}

// the float64 reference distance, in index order and without FMA (the contract of sos_l2f_top2)
__device__ __forceinline__ double l2f_d2(const float* __restrict__ q, const float* __restrict__ t, int dim) {
  double s = 0.0;
  for (int k = 0; k < dim; ++k) {
    const double x = __dsub_rn((double)q[k], (double)t[k]);
    s = __dadd_rn(s, __dmul_rn(x, x));
  }
  return s;
}
__device__ __forceinline__ float l2f_dist(double d2) { return __double2float_rn(__dsqrt_rn(d2)); }

__device__ __forceinline__ float l2f_acc(unsigned long long key) {
  const uint32_t ord = ~(uint32_t)(key >> 32);
  return __uint_as_float((ord & 0x80000000u) ? (ord & 0x7FFFFFFFu) : ~ord);
}

// One thread per query row: merge the per-split top-K keys, then decide (see the band derivation above).  Certain queries get
// their winners' float64 distances here; the others are appended to `list` for l2f_redecide_kernel.
__global__ void __launch_bounds__(256)
l2f_decide_kernel(const ulonglong2* __restrict__ partial, const float* __restrict__ q, const float* __restrict__ t, int dim,
                  const int32_t* __restrict__ q_start, const int32_t* __restrict__ q_len, const int32_t* __restrict__ t_start,
                  const int32_t* __restrict__ t_len, int max_nq, int max_nt, int splits, int q_rows_per_seg,
                  const double* __restrict__ qnorm2, const double* __restrict__ tmax2, int32_t* __restrict__ idx0,
                  float* __restrict__ d0, int32_t* __restrict__ idx1, float* __restrict__ d1, int2* __restrict__ list,
                  int32_t* __restrict__ list_n, int32_t* __restrict__ stats) {
  const int seg = blockIdx.y;
  const int nq = min(q_len[seg], max_nq), row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= nq) return;
  const bool top2 = idx1 != nullptr || d1 != nullptr;
  const int K = top2 ? 3 : 2;
  const int nt = min(t_len[seg], max_nt), g = q_start[seg] + row;
  unsigned long long w[3] = {KEY64_NONE, KEY64_NONE, KEY64_NONE}, bad = 0;
  const ulonglong2* p = partial + ((size_t)seg * max_nq + row) * splits * 2;
  for (int s = 0; s < splits; ++s) {
    const ulonglong2 a = p[2 * s], b = p[2 * s + 1];
    bad |= b.y;
    const unsigned long long k3[3] = {a.x, a.y, b.x};
    for (int i = 0; i < K; ++i) {
      const unsigned long long k = k3[i];
      if (k < w[0]) { w[2] = w[1]; w[1] = w[0]; w[0] = k; }
      else if (k < w[1]) { w[2] = w[1]; w[1] = k; }
      else if (k < w[2]) w[2] = k;
    }
  }
  int found = 0;
  double acc[3];
  for (int i = 0; i < 3; ++i) {
    found += (i < K && w[i] != KEY64_NONE) ? 1 : 0;
    acc[i] = (i < K && w[i] != KEY64_NONE) ? (double)l2f_acc(w[i]) : -INFINITY;
  }
  if (nt == 0) {
    idx0[g] = -1; d0[g] = -1.f;
    if (idx1) idx1[g] = -1;
    if (d1) d1[g] = -1.f;
    return;
  }
  const double qn2 = qnorm2[(size_t)seg * q_rows_per_seg + row], m2 = tmax2[seg];
  const double qn = sqrt(qn2), mt = sqrt(m2);
  const double band = L2F_C_QT * qn * mt + L2F_C_TT * m2 + L2F_C_QQ * qn2 + L2F_C_LIN * (qn + mt) + L2F_C_ABS;
  bool certain = bad == 0 && found >= min(nt, K) && qn < 0x1p125 && 2.1 * qn * mt + 1.1 * m2 < 0x1p126;
  certain = certain && acc[0] - acc[1] > 2.0 * band && (!top2 || acc[1] - acc[2] > 2.0 * band);
  if (!certain) {
    list[atomicAdd(list_n, 1)] = make_int2(seg, row);
    return;
  }
  const float* qr = q + (size_t)g * dim;
  const float* tb = t + (size_t)t_start[seg] * dim;
  double worst = 0.0;
  const int r0 = (int)(uint32_t)w[0];
  const double e0 = l2f_d2(qr, tb + (size_t)r0 * dim, dim);
  worst = fabs((qn2 - acc[0]) - e0) / band;
  idx0[g] = r0; d0[g] = l2f_dist(e0);
  if (top2) {
    int r1 = -1;
    float dist1 = -1.f;
    if (w[1] != KEY64_NONE) {
      r1 = (int)(uint32_t)w[1];
      const double e1 = l2f_d2(qr, tb + (size_t)r1 * dim, dim);
      worst = fmax(worst, fabs((qn2 - acc[1]) - e1) / band);
      dist1 = l2f_dist(e1);
    }
    if (idx1) idx1[g] = r1;
    if (d1) d1[g] = dist1;
  }
  if (stats) atomicMax(stats + SOS_L2F_STAT_BAND_PPM, (int)fmin(worst * 1e6, 2147483647.0));
}

// Float64 brute force for the queries l2f_decide_kernel could not decide: one block per listed query (grid-stride over the
// device-side count, the grid is sized from the host bound), each thread scans train rows tid, tid + 256, ... in the reference
// order, then the block merges the per-thread top-2 by (d^2, row).
constexpr int RD_THREADS = 256;
__device__ __forceinline__ bool l2f_before(double da, int ra, double db, int rb) { return da < db || (da == db && ra < rb); }
__device__ __forceinline__ void l2f_insert(double d, int r, double (&bd)[2], int (&br)[2]) {
  if (r < 0) return;
  if (br[0] < 0 || l2f_before(d, r, bd[0], br[0])) { bd[1] = bd[0]; br[1] = br[0]; bd[0] = d; br[0] = r; }
  else if (br[1] < 0 || l2f_before(d, r, bd[1], br[1])) { bd[1] = d; br[1] = r; }
}

__global__ void __launch_bounds__(RD_THREADS)
l2f_redecide_kernel(const float* __restrict__ q, const float* __restrict__ t, int dim, const int32_t* __restrict__ q_start,
                    const int32_t* __restrict__ t_start, const int32_t* __restrict__ t_len, int max_nt,
                    const int2* __restrict__ list, const int32_t* __restrict__ list_n, int32_t* __restrict__ idx0,
                    float* __restrict__ d0, int32_t* __restrict__ idx1, float* __restrict__ d1, int32_t* __restrict__ stats) {
  __shared__ float sq[128];
  __shared__ double wd[RD_THREADS / 32][2];
  __shared__ int wr[RD_THREADS / 32][2];
  const int n = *list_n, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (stats && blockIdx.x == 0 && tid == 0) stats[SOS_L2F_STAT_REDECIDED] = n;
  for (int e = blockIdx.x; e < n; e += gridDim.x) {
    const int2 it = list[e];
    const int g = q_start[it.x] + it.y, nt = min(t_len[it.x], max_nt);
    const float* tb = t + (size_t)t_start[it.x] * dim;
    __syncthreads();                                   // the previous entry is done with sq / wd / wr
    for (int k = tid; k < dim; k += RD_THREADS) sq[k] = q[(size_t)g * dim + k];
    __syncthreads();
    double bd[2] = {0.0, 0.0};
    int br[2] = {-1, -1};
    for (int j = tid; j < nt; j += RD_THREADS) l2f_insert(l2f_d2(sq, tb + (size_t)j * dim, dim), j, bd, br);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      double od[2];
      int orr[2];
      for (int i = 0; i < 2; ++i) { od[i] = __shfl_xor_sync(0xFFFFFFFFu, bd[i], off); orr[i] = __shfl_xor_sync(0xFFFFFFFFu, br[i], off); }
      l2f_insert(od[0], orr[0], bd, br);
      l2f_insert(od[1], orr[1], bd, br);
    }
    if (lane == 0) { wd[warp][0] = bd[0]; wd[warp][1] = bd[1]; wr[warp][0] = br[0]; wr[warp][1] = br[1]; }
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < RD_THREADS / 32; ++w) { l2f_insert(wd[w][0], wr[w][0], bd, br); l2f_insert(wd[w][1], wr[w][1], bd, br); }
      idx0[g] = br[0]; d0[g] = br[0] < 0 ? -1.f : l2f_dist(bd[0]);
      if (idx1) idx1[g] = br[1];
      if (d1) d1[g] = br[1] < 0 ? -1.f : l2f_dist(bd[1]);
    }
  }
}

}  // namespace sos_hamming_mma

// Host side, called by sos_hamming_top2 (hamming.cu).  `ws` holds the partial keys + work items (already planned);
// `exp` is scratch for the expanded tiles.
size_t sos_hamming_mma_scratch_bytes(int n_seg, int max_nq, int max_nt) {
  using namespace sos_hamming_mma;
  const size_t qt = (size_t)((max_nq + 255) / 256) * 2, tt = (size_t)((max_nt + TILE - 1) / TILE);
  return (size_t)n_seg * (qt + tt) * TILE_BYTES + 256;
}

int sos_hamming_mma_launch(sos_ctx* ctx, const uint32_t* q, const uint32_t* t, const int32_t* q_start,
                           const int32_t* q_len, const int32_t* t_start, const int32_t* t_len, int n_seg, int max_nq,
                           int max_nt, int splits, const uint32_t* items, const int32_t* n_items, unsigned max_items,
                           bool top2, void* exp, uint2* partial) {
  using namespace sos_hamming_mma;
  const int qt = ((max_nq + 255) / 256) * 2, tt = (max_nt + TILE - 1) / TILE;
  uint8_t* a_exp = (uint8_t*)exp;
  uint8_t* b_exp = a_exp + (size_t)n_seg * qt * TILE_BYTES;
  if (qt > 0 || tt > 0) {
    ExpandArgs e;
    e.desc[0] = q; e.desc[1] = t; e.start[0] = q_start; e.start[1] = t_start; e.len[0] = q_len; e.len[1] = t_len;
    e.max_rows[0] = max_nq; e.max_rows[1] = max_nt; e.tiles_per_seg[0] = qt; e.tiles_per_seg[1] = tt;
    e.out[0] = a_exp; e.out[1] = b_exp;
    expand_kernel<<<dim3(qt > tt ? qt : tt, n_seg, 2), 256, 0, ctx->stream>>>(e);
    SOS_LAUNCHED_AS(ctx, "hamming_expand_kernel");
  }
  Args a;
  a.a_exp = a_exp; a.b_exp = b_exp; a.q_len = q_len; a.t_len = t_len;
  a.max_nq = max_nq; a.max_nt = max_nt; a.splits = splits; a.q_tiles_per_seg = qt; a.t_tiles_per_seg = tt;
  a.items = items; a.n_items = n_items; a.partial = partial;
  a.a_norm = nullptr;
  // ring depth 4 (221 KB of shared memory); 3 stages measured the same (profiles/r02/score_variants_and_ring_depth_ab.log)
  constexpr int ST = 4;
  static bool attr_set[64][2] = {};     // per device: the opt-in to > 48 KB of dynamic shared memory
  const int dev = ctx->device & 63, v = top2 ? 1 : 0;
  if (!attr_set[dev][v]) {
    if (top2) SOS_CUDA(cudaFuncSetAttribute(mma_kernel<true, ST, KIND_HAMMING>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(ST)));
    else SOS_CUDA(cudaFuncSetAttribute(mma_kernel<false, ST, KIND_HAMMING>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(ST)));
    attr_set[dev][v] = true;
  }
  // One kernel, two launch shapes.  Short items (stereo buckets: a handful of train tiles each) run PERSISTENT — one CTA per
  // SM walks the work list, so barriers, tensor memory and the pipelines survive from item to item (measured: 0.083 ->
  // 0.076 ms on the 384 C2 buckets).  Long items (temporal matching: ~36 train tiles each) get one CTA per item and leave
  // the balancing to the hardware scheduler: the fixed striding of the persistent shape loses more to unequal SMs than the
  // per-item set-up costs (0.285 vs 0.300 ms; profiles/r02/hamming_ab_persistent.log).
  const bool persistent = max_nt <= 2048;
  const unsigned grid = (persistent && max_items > (unsigned)ctx->sm_count) ? (unsigned)ctx->sm_count : max_items;
  if (top2) mma_kernel<true, ST, KIND_HAMMING><<<grid, THREADS, smem_bytes(ST), ctx->stream>>>(a);
  else mma_kernel<false, ST, KIND_HAMMING><<<grid, THREADS, smem_bytes(ST), ctx->stream>>>(a);
  SOS_LAUNCHED_AS(ctx, "hamming_mma_kernel");
  return SOS_OK;
}

// The float-descriptor L2 engine (sos_l2_top2 in hamming.cu).  `exp` = expanded tiles followed by the query norms.
size_t sos_l2_mma_scratch_bytes(int n_seg, int max_nq, int max_nt) {
  using namespace sos_hamming_mma;
  const size_t qt = (size_t)((max_nq + 255) / 256) * 2;
  return sos_hamming_mma_scratch_bytes(n_seg, max_nq, max_nt) + (size_t)n_seg * qt * TILE * sizeof(int32_t) + 256;
}

int sos_l2_mma_launch(sos_ctx* ctx, const float* q, const float* t, int dim, const int32_t* q_start, const int32_t* q_len,
                      const int32_t* t_start, const int32_t* t_len, int n_seg, int max_nq, int max_nt, int splits,
                      const uint32_t* items, const int32_t* n_items, unsigned max_items, bool top2, void* exp,
                      ulonglong2* partial, int32_t* flag) {
  using namespace sos_hamming_mma;
  const int qt = ((max_nq + 255) / 256) * 2, tt = (max_nt + TILE - 1) / TILE;
  uint8_t* a_exp = (uint8_t*)exp;
  uint8_t* b_exp = a_exp + (size_t)n_seg * qt * TILE_BYTES;
  int32_t* norms = (int32_t*)(b_exp + sos_align_up((size_t)n_seg * tt * TILE_BYTES, 256));
  if (qt > 0) {
    expand_l2_kernel<<<dim3(qt, n_seg), 256, 0, ctx->stream>>>(q, dim, q_start, q_len, max_nq, qt, 0, a_exp, norms, flag);
    SOS_LAUNCHED_AS(ctx, "l2_expand_kernel");
  }
  if (tt > 0) {
    expand_l2_kernel<<<dim3(tt, n_seg), 256, 0, ctx->stream>>>(t, dim, t_start, t_len, max_nt, tt, 1, b_exp, nullptr, flag);
    SOS_LAUNCHED_AS(ctx, "l2_expand_kernel");
  }
  Args a;
  a.a_norm = norms;
  a.a_exp = a_exp; a.b_exp = b_exp; a.q_len = q_len; a.t_len = t_len;
  a.max_nq = max_nq; a.max_nt = max_nt; a.splits = splits; a.q_tiles_per_seg = qt; a.t_tiles_per_seg = tt;
  a.items = items; a.n_items = n_items; a.partial = partial;
  constexpr int ST = 4;
  static bool attr_set[64][2] = {};
  const int dev = ctx->device & 63, v = top2 ? 1 : 0;
  if (!attr_set[dev][v]) {
    if (top2) SOS_CUDA(cudaFuncSetAttribute(mma_kernel<true, ST, KIND_L2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(ST)));
    else SOS_CUDA(cudaFuncSetAttribute(mma_kernel<false, ST, KIND_L2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(ST)));
    attr_set[dev][v] = true;
  }
  const bool persistent = max_nt <= 2048;
  const unsigned grid = (persistent && max_items > (unsigned)ctx->sm_count) ? (unsigned)ctx->sm_count : max_items;
  if (top2) mma_kernel<true, ST, KIND_L2><<<grid, THREADS, smem_bytes(ST), ctx->stream>>>(a);
  else mma_kernel<false, ST, KIND_L2><<<grid, THREADS, smem_bytes(ST), ctx->stream>>>(a);
  SOS_LAUNCHED_AS(ctx, "l2_mma_kernel");
  return SOS_OK;
}

// The general float-descriptor L2 engine (sos_l2f_top2 in hamming.cu): expansion, GEMM, decision and float64 re-decision.
// Scratch: partial keys (2 x ulonglong2 per query row and split) | list of undecided queries | its count | |q|^2 per expanded
// query row | max |t|^2 per segment | expanded query tiles | expanded train tiles.
static size_t l2f_align(size_t b) { return sos_align_up(b, 256); }
size_t sos_l2f_scratch_bytes(int n_seg, int max_nq, int max_nt, int dim, int splits) {
  using namespace sos_hamming_mma;
  const size_t qt = (size_t)((max_nq + 255) / 256) * 2, tt = (size_t)((max_nt + TILE - 1) / TILE), nsub = dim > 64 ? 2 : 1;
  const size_t rows = (size_t)max_nq * n_seg;
  return l2f_align(rows * splits * 2 * sizeof(ulonglong2)) + l2f_align(rows * sizeof(int2)) + 256 +
         l2f_align((size_t)n_seg * qt * TILE * sizeof(double)) + l2f_align((size_t)n_seg * sizeof(double)) +
         (size_t)n_seg * (qt + tt) * nsub * TILE_BYTES;
}

int sos_l2f_launch(sos_ctx* ctx, const float* q, const float* t, int dim, const int32_t* q_start, const int32_t* q_len,
                   const int32_t* t_start, const int32_t* t_len, int n_seg, int max_nq, int max_nt, int splits,
                   const uint32_t* items, const int32_t* n_items, unsigned max_items, bool top2, void* scratch,
                   int32_t* idx0, float* d0, int32_t* idx1, float* d1, int32_t* flag, int32_t* stats) {
  using namespace sos_hamming_mma;
  const int qt = ((max_nq + 255) / 256) * 2, tt = (max_nt + TILE - 1) / TILE, nsub = dim > 64 ? 2 : 1;
  const size_t rows = (size_t)max_nq * n_seg;
  char* p = (char*)scratch;
  ulonglong2* partial = (ulonglong2*)p;            p += l2f_align(rows * splits * 2 * sizeof(ulonglong2));
  int2* list = (int2*)p;                           p += l2f_align(rows * sizeof(int2));
  int32_t* list_n = (int32_t*)p;                   p += 256;
  double* qnorm2 = (double*)p;                     p += l2f_align((size_t)n_seg * qt * TILE * sizeof(double));
  double* tmax2 = (double*)p;                      p += l2f_align((size_t)n_seg * sizeof(double));
  uint8_t* a_exp = (uint8_t*)p;
  uint8_t* b_exp = a_exp + (size_t)n_seg * qt * nsub * TILE_BYTES;
  SOS_CUDA(cudaMemsetAsync(list_n, 0, sizeof(int32_t), ctx->stream));
  SOS_CUDA(cudaMemsetAsync(tmax2, 0, (size_t)n_seg * sizeof(double), ctx->stream));
  if (stats) SOS_CUDA(cudaMemsetAsync(stats, 0, SOS_L2F_STATS * sizeof(int32_t), ctx->stream));
  if (qt > 0) {
    l2f_expand_kernel<<<dim3(qt, n_seg), 256, 0, ctx->stream>>>(q, dim, q_start, q_len, max_nq, qt, nsub, 0, a_exp, qnorm2, flag);
    SOS_LAUNCHED_AS(ctx, "l2f_expand_kernel");
  }
  if (tt > 0) {
    l2f_expand_kernel<<<dim3(tt, n_seg), 256, 0, ctx->stream>>>(t, dim, t_start, t_len, max_nt, tt, nsub, 1, b_exp, tmax2, flag);
    SOS_LAUNCHED_AS(ctx, "l2f_expand_kernel");
  }
  Args a;
  a.a_norm = nullptr;
  a.dim = dim; a.nsub = nsub;
  a.a_exp = a_exp; a.b_exp = b_exp; a.q_len = q_len; a.t_len = t_len;
  a.max_nq = max_nq; a.max_nt = max_nt; a.splits = splits; a.q_tiles_per_seg = qt; a.t_tiles_per_seg = tt;
  a.items = items; a.n_items = n_items; a.partial = partial;
  // six 36 KB buffers: 2 nsub for the query tiles, the rest a ring of train sub-tiles (4 for dim <= 64, 2 above)
  constexpr int ST = 4;
  static bool attr_set[64][2] = {};
  const int dev = ctx->device & 63, v = top2 ? 1 : 0;
  if (!attr_set[dev][v]) {
    if (top2) SOS_CUDA(cudaFuncSetAttribute(mma_kernel<true, ST, KIND_L2F>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(ST)));
    else SOS_CUDA(cudaFuncSetAttribute(mma_kernel<false, ST, KIND_L2F>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(ST)));
    attr_set[dev][v] = true;
  }
  const bool persistent = max_nt <= 2048;
  const unsigned grid = (persistent && max_items > (unsigned)ctx->sm_count) ? (unsigned)ctx->sm_count : max_items;
  if (top2) mma_kernel<true, ST, KIND_L2F><<<grid, THREADS, smem_bytes(ST), ctx->stream>>>(a);
  else mma_kernel<false, ST, KIND_L2F><<<grid, THREADS, smem_bytes(ST), ctx->stream>>>(a);
  SOS_LAUNCHED_AS(ctx, "l2f_mma_kernel");
  dim3 mgrid((max_nq + 255) / 256, n_seg);
  l2f_decide_kernel<<<mgrid, 256, 0, ctx->stream>>>(partial, q, t, dim, q_start, q_len, t_start, t_len, max_nq, max_nt, splits,
                                                    qt * TILE, qnorm2, tmax2, idx0, d0, idx1, d1, list, list_n, stats);
  SOS_LAUNCHED_AS(ctx, "l2f_decide_kernel");
  const size_t rd_grid = rows < (size_t)(8 * ctx->sm_count) ? rows : (size_t)(8 * ctx->sm_count);
  l2f_redecide_kernel<<<(unsigned)rd_grid, RD_THREADS, 0, ctx->stream>>>(q, t, dim, q_start, t_start, t_len, max_nt, list,
                                                                        list_n, idx0, d0, idx1, d1, stats);
  SOS_LAUNCHED_AS(ctx, "l2f_redecide_kernel");
  return SOS_OK;
}
