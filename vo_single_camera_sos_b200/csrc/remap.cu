// Step 1 of the SOS front-end: LUT panoramic remap of the two mirror views.
//
// Replaces cv2.remap(INTER_LINEAR, BORDER_CONSTANT) as called by Panorama.get_panoramic_image (reference
// omnistereo/panorama.py:258-321) on the masked omni images of OmniStereoModel.get_fully_masked_images
// (camera_models.py:2932-3025).  The arithmetic is OpenCV's fixed-point bilinear path, restated:
//   sx = cvRound(32*x) (round-half-even; NaN / overflow -> INT_MIN), x0 = sat_s16(sx >> 5), ax = sx & 31
//   weights  w = {(32-ay)(32-ax), (32-ay)ax, ay(32-ax), ay*ax} * 32   (Q15, sum == 32768 exactly)
//   dst = (w00*p00 + w01*p01 + w10*p10 + w11*p11 + 16384) >> 15,  taps outside the image = border value.
// The mirror mask is folded into the packed LUT (one validity bit per tap): a masked-out source pixel reads
// as the background colour, so the masked omni images are never materialised.
//
// HBM-bound: per panorama pixel 8 B of LUT in, `ch` bytes out, and the source annulus is read about once.
// Layout: block = 8 warps = 8 panorama rows x 128 columns, a thread owns 4 consecutive pixels, so LUT reads
// are 2 x LDG.128 per thread, stores are 4*ch contiguous bytes per thread, and neighbouring rows/columns of
// the tile hit the same source cache lines in L1.
#include "sos_common.cuh"

namespace {

constexpr int RM_PX = 4;              // pixels per thread
constexpr int RM_TILE_COLS = 32 * RM_PX;
constexpr int RM_TILE_ROWS = 8;

__device__ __forceinline__ int cv_round_q5(float x) {
  // cv::remap: cvRound(x * INTER_TAB_SIZE) via cvtps2dq: round-half-even, "integer indefinite" otherwise
  const float xs = x * 32.0f;
  if (!(fabsf(xs) < 2147483648.0f)) return INT_MIN;
  return __float2int_rn(xs);
}

template <typename T>
__global__ void __launch_bounds__(256)
lut_pack_kernel(const T* __restrict__ map_x, const T* __restrict__ map_y, int n, const uint8_t* __restrict__ mask,
                int src_h, int src_w, uint64_t* __restrict__ lut) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int sx = cv_round_q5((float)map_x[i]);  // float64 -> float32 cast of panorama.py:291-292
  const int sy = cv_round_q5((float)map_y[i]);
  const int x0 = max(-32768, min(32767, sx >> 5));
  const int y0 = max(-32768, min(32767, sy >> 5));
  const uint32_t ax = (uint32_t)sx & 31u, ay = (uint32_t)sy & 31u;
  uint32_t inside = 0, live = 0;
#pragma unroll
  for (int tap = 0; tap < 4; ++tap) {
    const int x = x0 + (tap & 1), y = y0 + (tap >> 1);
    if (x >= 0 && x < src_w && y >= 0 && y < src_h) {
      inside |= 1u << tap;
      if (mask == nullptr || mask[(size_t)y * src_w + x] != 0) live |= 1u << tap;
    }
  }
  // bit 56: all four taps usable AND the 16 bytes from tap 2 of a 3-channel frame lie inside it; gates remap3b_kernel's
  // fast taps, whose three aligned 32-bit loads per tap row end at most 12 bytes past the tap
  uint32_t wide3 = 0;
  if (live == 15u) {
    const long long p1 = (((long long)y0 + 1) * src_w + x0) * 3;
    wide3 = (p1 + 16 <= (long long)src_h * src_w * 3) ? 1u : 0u;
  }
  const uint64_t lo = (uint32_t)(x0 & 0xFFFF) | ((uint32_t)(y0 & 0xFFFF) << 16);
  const uint64_t hi = ax | (ay << 5) | (inside << 16) | (live << 20) | (wide3 << 24);
  lut[i] = lo | (hi << 32);
}

template <int CH>
__device__ __forceinline__ void load_tap(const uint8_t* __restrict__ p, uint32_t w, uint32_t* acc) {
#pragma unroll
  for (int c = 0; c < CH; ++c) acc[c] += w * (uint32_t)__ldg(p + c);
}

// One output pixel: returns CH bytes in out[].
template <int CH>
__device__ __forceinline__ void remap_pixel(const uint8_t* __restrict__ src, int src_w, uint64_t e, const uint32_t* border,
                                            const uint32_t* bg, uint32_t* out) {
  const int x0 = (int)(int16_t)(e & 0xFFFF);
  const int y0 = (int)(int16_t)((e >> 16) & 0xFFFF);
  const uint32_t hi = (uint32_t)(e >> 32);
  const uint32_t ax = hi & 31u, ay = (hi >> 5) & 31u;
  const uint32_t inside = (hi >> 16) & 15u, live = (hi >> 20) & 15u;
  if (inside == 0) {  // all four taps outside: Q15 weights sum to 32768, so the result is the border value
#pragma unroll
    for (int c = 0; c < CH; ++c) out[c] = border[c];
    return;
  }
  const uint32_t w[4] = {(32u - ay) * (32u - ax) * 32u, (32u - ay) * ax * 32u, ay * (32u - ax) * 32u, ay * ax * 32u};
  uint32_t acc[CH];
#pragma unroll
  for (int c = 0; c < CH; ++c) acc[c] = 16384u;
  const uint8_t* p = src + ((size_t)y0 * src_w + x0) * CH;
  if (live == 15u) {
    load_tap<CH>(p, w[0], acc);
    load_tap<CH>(p + CH, w[1], acc);
    load_tap<CH>(p + (size_t)src_w * CH, w[2], acc);
    load_tap<CH>(p + (size_t)src_w * CH + CH, w[3], acc);
  } else {
#pragma unroll
    for (int tap = 0; tap < 4; ++tap) {
      if (w[tap] == 0) continue;
      if (live & (1u << tap)) {
        load_tap<CH>(p + ((size_t)(tap >> 1) * src_w + (tap & 1)) * CH, w[tap], acc);
      } else {
        const uint32_t* v = (inside & (1u << tap)) ? bg : border;
#pragma unroll
        for (int c = 0; c < CH; ++c) acc[c] += w[tap] * v[c];
      }
    }
  }
#pragma unroll
  for (int c = 0; c < CH; ++c) out[c] = acc[c] >> 15;
}

struct RemapConst {
  uint32_t border[4];
  uint32_t bg[4];
};

template <int CH>
__global__ void __launch_bounds__(256)
remap_kernel(const uint8_t* __restrict__ src, int src_h, int src_w, const uint64_t* __restrict__ lut, int views, int rows,
             int cols, RemapConst k, uint8_t* __restrict__ dst) {
  const int lane_col = blockIdx.x * RM_TILE_COLS + (threadIdx.x & 31) * RM_PX;
  const int row = blockIdx.y * RM_TILE_ROWS + (threadIdx.x >> 5);
  if (row >= rows || lane_col >= cols) return;
  const int img = blockIdx.z;  // batch * views + view
  const int view = img % views, b = img / views;
  const uint8_t* s = src + (size_t)b * src_h * src_w * CH;
  const size_t px0 = (size_t)row * cols + lane_col;
  const uint64_t* l = lut + (size_t)view * rows * cols + px0;
  uint8_t* d = dst + ((size_t)img * rows * cols + px0) * CH;

  const int n = min(RM_PX, cols - lane_col);
  uint64_t e[RM_PX];
  if (n == RM_PX && (((uintptr_t)l) & 15) == 0) {
    const ulonglong2 a = __ldg((const ulonglong2*)l), c = __ldg((const ulonglong2*)l + 1);
    e[0] = a.x; e[1] = a.y; e[2] = c.x; e[3] = c.y;
  } else {
#pragma unroll
    for (int i = 0; i < RM_PX; ++i) e[i] = (i < n) ? __ldg(l + i) : 0ull;
  }
  uint32_t o[RM_PX][CH];
#pragma unroll
  for (int i = 0; i < RM_PX; ++i) {
    if (i < n) remap_pixel<CH>(s, src_w, e[i], k.border, k.bg, o[i]);
  }
  if (n == RM_PX && (((uintptr_t)d) & 3) == 0) {
    // RM_PX * CH bytes = CH 32-bit words
    uint32_t words[CH];
#pragma unroll
    for (int wd = 0; wd < CH; ++wd) {
      uint32_t v = 0;
#pragma unroll
      for (int bt = 0; bt < 4; ++bt) {
        const int flat = wd * 4 + bt;
        v |= o[flat / CH][flat % CH] << (8 * bt);
      }
      words[wd] = v;
    }
    if (CH == 4 && (((uintptr_t)d) & 15) == 0) {
      *(uint4*)d = make_uint4(words[0], words[1], words[2 % CH], words[3 % CH]);
    } else {
#pragma unroll
      for (int wd = 0; wd < CH; ++wd) ((uint32_t*)d)[wd] = words[wd];
    }
  } else {
    for (int i = 0; i < n; ++i)
#pragma unroll
      for (int c = 0; c < CH; ++c) d[i * CH + c] = (uint8_t)o[i][c];
  }
}


// ---- lane mapping of the 3-channel kernel -----------------------------------------------------------------------------
// A warp-wide gather costs one L1 wavefront per distinct 128-byte line it touches.  32 consecutive pixels of ONE panorama
// row follow an arc in the omni image that crosses ~14 source rows (top mirror at C2) -> ~14 wavefronts per tap load; a
// lane-per-pixel-along-the-row kernel is bound by exactly that (l1tex data-pipe 87 % busy, DRAM 11 %).  Mapping the 32 lanes onto a compact
// 4-row x 8-column panorama patch halves the distinct lines (measured on the C2 LUT: 13.7 -> 6.1 top, 4.5 -> 1.9 bottom).
// Warp tile = 4 rows x 32 columns in 4 passes (lane l: row l / 8, column 8 * pass + l % 8); the 4 x 96 output bytes are
// staged in shared memory and written as 16-byte vectors.
constexpr int RP_ROWS = 4;                 // rows per warp tile
constexpr int RP_COLS = 32;                // columns per warp tile
constexpr int RP_WARPS_X = 4, RP_WARPS_Y = 2;

// ---- batch-looped kernel with TMA-staged LUT tiles (the default 3-channel path) --------------------------------------------
// The LUT depends on (view, row, col) only, so a block that owns one 8 x 128 LUT tile serves that tile for EVERY frame of
// its share of the batch: the tile is fetched once (8 KB, one cp.async.bulk row copy per panorama row, completion on an
// mbarrier), each lane decodes its four entries ONCE into registers (32-bit source offset, alignment shift, weights), and
// the per-frame loop is nothing but 16 tap loads, the alignment funnel, dp4a arithmetic and the staged store:
//   * ~45 instructions per pixel and frame instead of ~100 (ncu, round 1: a per-frame 4 x 8-patch kernel was issue bound
//     and spent more than half of its instructions on LUT decode, 64-bit address arithmetic, per-warp prologue and branches);
//   * all 16 loads of a lane are in flight before the first use: no LUT-load -> tap-load dependency in the loop;
//   * rows outside the mirror's field of view (38 % of the C2 panorama: whole rows of the LUT are "dead") never touch the
//     source image: the warp stages the border colour once and only stores;
//   * lanes that are neither fast nor dead (image edge, mirror-mask edge: ~1 % of the 4 x 8 patches) are fixed up by the
//     generic per-tap path inside a warp-uniform branch.
// Vertical interpolation first: one PRMT gathers (row 0, row 1) bytes of the left and right tap of a channel, dp4a with the
// weights (32 - ay, ay, 0, 0) / (0, 0, 32 - ay, ay) gives vL and vR, then (wl * vL + ax * vR + 512) >> 10 — the same integer
// as cv::remap's (sum_i w_i p_i + 16384) >> 15 because the Q15 weights are 32 * (6-bit x 6-bit products).
// Requires a 4-byte aligned source whose rows are a multiple of 4 bytes (src_w % 4 == 0), so that the alignment of a tap
// address is the same for every frame and both rows; other shapes take remap_kernel<3>.
constexpr int RB_TILE_ROWS = RP_ROWS * RP_WARPS_Y;   // 8
constexpr int RB_TILE_COLS = RP_COLS * RP_WARPS_X;   // 128
constexpr int RB_NP = RP_COLS / 8;                   // passes per lane

__device__ inline uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__global__ void __launch_bounds__(RP_WARPS_X * RP_WARPS_Y * 32, 3)
remap3b_kernel(const uint8_t* __restrict__ src, int batch, int frames_per_block, int src_h, int src_w,
               const uint64_t* __restrict__ lut, int views, int rows, int cols, RemapConst k, uint8_t* __restrict__ dst) {
  __shared__ __align__(128) uint64_t slut[RB_TILE_ROWS][RB_TILE_COLS];
  __shared__ __align__(16) uint8_t sout[RP_WARPS_X * RP_WARPS_Y][RP_ROWS][RP_COLS * 3];
  __shared__ __align__(8) uint64_t mbar;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int view = blockIdx.z % views;
  const int b_begin = (blockIdx.z / views) * frames_per_block, b_end = min(batch, b_begin + frames_per_block);
  const int row_t0 = blockIdx.y * RB_TILE_ROWS, col_t0 = blockIdx.x * RB_TILE_COLS;
  const uint64_t* ltile = lut + ((size_t)view * rows + row_t0) * cols + col_t0;
  // bulk copies need 16-byte aligned addresses and sizes: full tiles of an even-width, 16-byte aligned LUT
  const bool bulk = (col_t0 + RB_TILE_COLS <= cols) && (row_t0 + RB_TILE_ROWS <= rows) && ((cols & 1) == 0) &&
                    ((((uintptr_t)lut) & 15) == 0);
  if (bulk) {
    const uint32_t bar = smem_addr(&mbar);
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)sizeof(slut)) : "memory");
#pragma unroll
      for (int r = 0; r < RB_TILE_ROWS; ++r)
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         smem_addr(&slut[r][0])),
                     "l"(ltile + (size_t)r * cols), "r"((uint32_t)(RB_TILE_COLS * sizeof(uint64_t))), "r"(bar)
                     : "memory");
    }
    uint32_t done = 0;
    for (int spin = 0; spin < (1 << 22) && !done; ++spin)   // try_wait sleeps in hardware; the bound only guards a lost copy
      asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
                   : "=r"(done) : "r"(bar) : "memory");
    if (!done) __trap();
  } else {
    for (int i = tid; i < RB_TILE_ROWS * RB_TILE_COLS; i += blockDim.x) {
      const int r = i / RB_TILE_COLS, c = i % RB_TILE_COLS;
      slut[r][c] = (row_t0 + r < rows && col_t0 + c < cols) ? __ldg(ltile + (size_t)r * cols + c) : 0ull;
    }
    __syncthreads();
  }

  const int wy = warp / RP_WARPS_X, wx = warp % RP_WARPS_X;
  const int col0 = col_t0 + wx * RP_COLS, row0 = row_t0 + wy * RP_ROWS;
  if (row0 >= rows || col0 >= cols) return;   // whole warps leave together; only __syncwarp below
  const int npx = min(RP_COLS, cols - col0), nrows = min(RP_ROWS, rows - row0);
  const int r = lane >> 3, cc = lane & 7;
  const uint32_t row_bytes = (uint32_t)src_w * 3u;
  const size_t img_bytes = (size_t)src_h * row_bytes;
  // decode once.  Bit p of fastm / deadm / slowm classifies this lane's pixel of pass p:
  //   fast: all four taps usable, wide loads stay inside the image    dead: no tap inside the image -> border colour
  //   slow: everything else (image edge, mirror-mask edge)            -> generic per-tap path, per frame
  uint32_t off[RB_NP], sh[RB_NP], wl[RB_NP], ax[RB_NP], wya[RB_NP];
  uint32_t fastm = 0, deadm = 0, slowm = 0;
#pragma unroll
  for (int pass = 0; pass < RB_NP; ++pass) {
    const int c = pass * 8 + cc;
    const uint64_t e = slut[wy * RP_ROWS + r][wx * RP_COLS + c];
    const uint32_t lo = (uint32_t)e, hi = (uint32_t)(e >> 32);
    const bool live = r < nrows && c < npx;
    const bool w = live && (hi & (1u << 24));
    const bool dd = live && !w && ((hi >> 16) & 0xFu) == 0;
    fastm |= (w ? 1u : 0u) << pass;
    deadm |= (dd ? 1u : 0u) << pass;
    slowm |= ((live && !w && !dd) ? 1u : 0u) << pass;
    // fast entries have 0 <= x0, y0 (all taps inside the image): plain unsigned arithmetic
    const uint32_t o = w ? ((lo >> 16) * (uint32_t)src_w + (lo & 0xFFFFu)) * 3u : 0u;   // other lanes read (and discard) the first bytes of the frame
    off[pass] = o & ~3u;
    sh[pass] = (o & 3u) * 8u;
    ax[pass] = hi & 31u;
    wl[pass] = 32u - ax[pass];
    const uint32_t ay = (hi >> 5) & 31u;
    wya[pass] = (32u - ay) | (ay << 8);
  }
  const bool any_fast = __any_sync(0xFFFFFFFFu, fastm != 0u);
  const bool any_slow = __any_sync(0xFFFFFFFFu, slowm != 0u);
  uint8_t* so = sout[warp][r];
  // dead pixels are the same in every frame (the fast path below never stores to them)
#pragma unroll
  for (int pass = 0; pass < RB_NP; ++pass)
    if ((deadm >> pass) & 1u) {
      const int c = pass * 8 + cc;
      so[c * 3 + 0] = (uint8_t)k.border[0];
      so[c * 3 + 1] = (uint8_t)k.border[1];
      so[c * 3 + 2] = (uint8_t)k.border[2];
    }
  __syncwarp();
  const int nbytes = npx * 3;
  const size_t drow = (size_t)cols * 3;
  const int r2 = lane / 6, ch = lane - r2 * 6;
  const uint8_t* s = src + (size_t)b_begin * img_bytes;
  uint8_t* d0 = dst + ((((size_t)b_begin * views + view) * rows + row0) * cols + col0) * 3;
  const size_t dframe = (size_t)views * rows * cols * 3;
  const bool vec_out = nbytes == RP_COLS * 3 && ((((uintptr_t)d0) | drow | dframe) & 15) == 0;
  for (int b = b_begin; b < b_end; ++b, s += img_bytes, d0 += dframe) {
    if (any_fast) {
      // all tap loads of the frame first (unconditional: 24 independent loads per lane), then arithmetic.  The six bytes of a
      // tap pair sit in the 12-byte window at the 4-byte aligned address below them: three 32-bit loads per row.  (Two 64-bit
      // loads + selects were measured slower, 0.460 vs 0.403 ms: the kernel is bound by the L1 data pipe, which spends one
      // wavefront per distinct 128-byte line of a request and two for 64-bit accesses — ncu l1tex__data_pipe_lsu_wavefronts 83 %.)
      uint32_t ta[RB_NP][2][3];
#pragma unroll
      for (int pass = 0; pass < RB_NP; ++pass) {
#pragma unroll
        for (int row = 0; row < 2; ++row) {
          const uint32_t* p = (const uint32_t*)(s + off[pass] + (row ? row_bytes : 0u));
          ta[pass][row][0] = __ldg(p);
          ta[pass][row][1] = __ldg(p + 1);
          // the six bytes reach into the third word only when they start at byte 3 of the window (a quarter of the taps): the
          // predicated load touches fewer distinct lines per request, and wavefronts per line are what the L1 pipe counts
          ta[pass][row][2] = sh[pass] == 24u ? __ldg(p + 2) : 0u;
        }
      }
#pragma unroll
      for (int pass = 0; pass < RB_NP; ++pass) {
        const int c = pass * 8 + cc;
        const uint32_t lo0 = __funnelshift_r(ta[pass][0][0], ta[pass][0][1], sh[pass]), hi0 = __funnelshift_r(ta[pass][0][1], ta[pass][0][2], sh[pass]);
        const uint32_t lo1 = __funnelshift_r(ta[pass][1][0], ta[pass][1][1], sh[pass]), hi1 = __funnelshift_r(ta[pass][1][1], ta[pass][1][2], sh[pass]);
        // (row 0, row 1) byte pairs: q0 = channel 0 left | right, q1 = channel 1 left | channel 2 left, q2 = channel 1 right | channel 2 right
        const uint32_t q0 = __byte_perm(lo0, lo1, 0x7340), q1 = __byte_perm(lo0, lo1, 0x6251), q2 = __byte_perm(hi0, hi1, 0x5140);
        const uint32_t wa = wya[pass], wb = wya[pass] << 16;
        const uint32_t v0l = __dp4a(q0, wa, 0u), v0r = __dp4a(q0, wb, 0u);
        const uint32_t v1l = __dp4a(q1, wa, 0u), v2l = __dp4a(q1, wb, 0u);
        const uint32_t v1r = __dp4a(q2, wa, 0u), v2r = __dp4a(q2, wb, 0u);
        const uint32_t o0 = (wl[pass] * v0l + (ax[pass] * v0r + 512u)) >> 10;
        const uint32_t o1 = (wl[pass] * v1l + (ax[pass] * v1r + 512u)) >> 10;
        const uint32_t o2 = (wl[pass] * v2l + (ax[pass] * v2r + 512u)) >> 10;
        if ((fastm >> pass) & 1u) {
          so[c * 3 + 0] = (uint8_t)o0;
          so[c * 3 + 1] = (uint8_t)o1;
          so[c * 3 + 2] = (uint8_t)o2;
        }
      }
    }
    if (any_slow) {
#pragma unroll 1
      for (int pass = 0; pass < RB_NP; ++pass)
        if ((slowm >> pass) & 1u) {
          const int c = pass * 8 + cc;
          uint32_t o[3];
          remap_pixel<3>(s, src_w, slut[wy * RP_ROWS + r][wx * RP_COLS + c], k.border, k.bg, o);
          so[c * 3 + 0] = (uint8_t)o[0];
          so[c * 3 + 1] = (uint8_t)o[1];
          so[c * 3 + 2] = (uint8_t)o[2];
        }
    }
    __syncwarp();
    if (vec_out) {
      if (lane < 24 && r2 < nrows) ((uint4*)(d0 + r2 * drow))[ch] = ((const uint4*)sout[warp][r2])[ch];
    } else {
      for (int rr = 0; rr < nrows; ++rr)
        for (int i = lane; i < nbytes; i += 32) d0[rr * drow + i] = sout[warp][rr][i];
    }
    __syncwarp();
  }
}

}  // namespace

template <typename T>
static int lut_pack_impl(sos_ctx* ctx, const T* map_x, const T* map_y, int rows, int cols, const uint8_t* mask,
                         int src_h, int src_w, sos_lut_entry* lut) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(rows >= 0 && cols >= 0 && src_h > 0 && src_w > 0, "bad size");
  SOS_CHECK_ARG(src_h <= 32767 && src_w <= 32767, "source image larger than 32767 (int16 coordinates)");
  const long long n = (long long)rows * cols;
  if (n == 0) return SOS_OK;
  SOS_CHECK_ARG(n < (1ll << 31), "panorama too large");
  SOS_CHECK_ARG(map_x && map_y && lut, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  lut_pack_kernel<T><<<sos_div_up((int)n, 256), 256, 0, ctx->stream>>>(map_x, map_y, (int)n, mask, src_h, src_w, lut);
  SOS_LAUNCHED_AS(ctx, "lut_pack_kernel");
  return SOS_OK;
}

extern "C" int sos_lut_pack_f32(sos_ctx* ctx, const float* map_x, const float* map_y, int rows, int cols,
                                const uint8_t* mask, int src_h, int src_w, sos_lut_entry* lut) {
  return lut_pack_impl<float>(ctx, map_x, map_y, rows, cols, mask, src_h, src_w, lut);
}

extern "C" int sos_lut_pack_f64(sos_ctx* ctx, const double* map_x, const double* map_y, int rows, int cols,
                                const uint8_t* mask, int src_h, int src_w, sos_lut_entry* lut) {
  return lut_pack_impl<double>(ctx, map_x, map_y, rows, cols, mask, src_h, src_w, lut);
}

extern "C" int sos_remap_u8(sos_ctx* ctx, const uint8_t* src, int batch, int src_h, int src_w, int channels,
                            const sos_lut_entry* lut, int views, int rows, int cols, const uint8_t* border,
                            const uint8_t* background, uint8_t* dst) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(channels == 1 || channels == 3 || channels == 4, "channels must be 1, 3 or 4");
  SOS_CHECK_ARG(batch >= 0 && views >= 0 && rows >= 0 && cols >= 0 && src_h > 0 && src_w > 0, "bad size");
  if (batch == 0 || views == 0 || rows == 0 || cols == 0) return SOS_OK;
  SOS_CHECK_ARG((long long)batch * views <= 65535, "batch*views exceeds 65535");
  SOS_CHECK_ARG(src && lut && dst, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  RemapConst k;
  for (int c = 0; c < 4; ++c) {
    k.border[c] = (border && c < channels) ? border[c] : 0;
    k.bg[c] = (background && c < channels) ? background[c] : 0;
  }
  // Batch-looped blocks with TMA-staged LUT tiles (remap3b_kernel) need tap addresses whose alignment is the same in every
  // frame and row (4-byte aligned source, src_w % 4 == 0) and 32-bit offsets inside a frame.  Every other 3-channel call,
  // and every 1- or 4-channel call, takes the generic kernel.  tests/test_gpu_remap.py runs every case on both.
  if (channels == 3 && ((uintptr_t)src & 3) == 0 && (src_w % 4) == 0 && (size_t)src_h * src_w * 3 < (1ull << 32)) {
    const int tiles = sos_div_up(cols, RB_TILE_COLS) * sos_div_up(rows, RB_TILE_ROWS) * views;
    // enough blocks for ~5 waves of 3 blocks per SM; every block decodes its LUT tile once for its share of the batch
    const int want_blocks = ctx->sm_count * 3 * 5;
    int splits = (want_blocks + tiles - 1) / tiles;
    splits = splits < 1 ? 1 : (splits > batch ? batch : splits);
    const int fpb = sos_div_up(batch, splits);
    splits = sos_div_up(batch, fpb);
    SOS_CHECK_ARG((long long)views * splits <= 65535, "views * batch splits exceeds 65535");
    dim3 gb(sos_div_up(cols, RB_TILE_COLS), sos_div_up(rows, RB_TILE_ROWS), views * splits);
    remap3b_kernel<<<gb, RP_WARPS_X * RP_WARPS_Y * 32, 0, ctx->stream>>>(src, batch, fpb, src_h, src_w, lut, views, rows, cols, k, dst);
    SOS_LAUNCHED_AS(ctx, "remap3b_kernel");
    return SOS_OK;
  }
  dim3 grid(sos_div_up(cols, RM_TILE_COLS), sos_div_up(rows, RM_TILE_ROWS), batch * views);
  if (channels == 1) remap_kernel<1><<<grid, 256, 0, ctx->stream>>>(src, src_h, src_w, lut, views, rows, cols, k, dst);
  else if (channels == 3) remap_kernel<3><<<grid, 256, 0, ctx->stream>>>(src, src_h, src_w, lut, views, rows, cols, k, dst);
  else remap_kernel<4><<<grid, 256, 0, ctx->stream>>>(src, src_h, src_w, lut, views, rows, cols, k, dst);
  SOS_LAUNCHED_AS(ctx, "remap_kernel");
  return SOS_OK;
}
