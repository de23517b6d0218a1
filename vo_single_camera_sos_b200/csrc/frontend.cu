// The batched, GPU-resident SOS front-end: one "step" takes B new frames (omni image + per-view ORB features) and
// produces B frame-pair poses (frame i-1 -> frame i; the last frame of a step is carried over as the reference of the
// next step).  It chains the five hot-path steps exactly as StereoPanoramicFrame.establish_stereo_correspondences
// (reference omnistereo/pose_est_tools.py:320-402) and TrackerStereoSE3.track_frame (pose_est_tools.py:736-847) do,
// but for all frames of the batch at once and without ever returning to the host: every data-dependent size (matches
// per bucket, triangulated points per frame, correspondences per pair) stays in device memory and is read by the next
// kernel.  The kernel chain is captured once into a CUDA graph and replayed per step.
//
//   remap (2 views)                                           panorama.py:258-321, camera_models.py:3107-3120
//   stereo Hamming match per azimuthal bucket, bottom = query  camera_models.py:3027-3101
//   sort by distance + pixel gate (|du| <= 2.5, dv >= 1)        camera_models.py:444, common_cv.py:167-188
//   lift + midpoint triangulation + range gate + compaction    pose_est_tools.py:344-397
//   temporal Hamming match top<->top, bottom<->bottom           pose_est_tools.py:741-749, 211-269
//   stack correspondences (top first, then bottom)             pose_est_tools.py:752-778
//   RANSAC over seeded Arun hypotheses (+ inlier refit)        pose_est_tools.py:785, 830
//
// The RGB-D front-end (sos_frontend_create_rgbd) runs the same stage B on one view and a central camera, after a store
// stage of its own (rgbd_store_kernel): RGBDFrame.establish_keypoints (pose_est_tools.py:600-623) and
// TrackerRGBDSE3.track_frame (pose_est_tools.py:880-958).
#include <string.h>

#include <vector>

#include <algorithm>
#include <climits>

#include "rgbd.cuh"
#include "sos_common.cuh"

namespace {

struct Buf {
  void* p = nullptr;
  size_t bytes = 0;
};

// One thread per frame: the (query = bottom, train = top) segment of every azimuthal bucket.  Offsets are clamped to the
// frame's feature capacity F and a bucket's rows to max_bucket (the per-segment capacity of the matching scratch and of
// the candidate-pair arrays); what the clamps drop is counted in overflow[b] so that the caller can see it (the
// reference has no such cap: size max_feat_per_bucket for the detector's per-bucket budget, pose_est_tools.py:862).
__global__ void stereo_segments_kernel(const int32_t* __restrict__ boff_top, const int32_t* __restrict__ boff_bot, int B,
                                       int nb, int F, int max_bucket, int32_t* __restrict__ q_start,
                                       int32_t* __restrict__ q_len, int32_t* __restrict__ t_start,
                                       int32_t* __restrict__ t_len, int32_t* __restrict__ overflow) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int32_t* ot = boff_top + (size_t)b * (nb + 1);
  const int32_t* ob = boff_bot + (size_t)b * (nb + 1);
  int dropped = 0;
  for (int k = 0; k < nb; ++k) {
    const int s = b * nb + k;
    const int q0 = min(max(ob[k], 0), F), q1 = min(max(ob[k + 1], q0), F);
    const int t0 = min(max(ot[k], 0), F), t1 = min(max(ot[k + 1], t0), F);
    const int nq = min(q1 - q0, max_bucket), nt = min(t1 - t0, max_bucket);
    dropped += max(0, ob[k + 1] - ob[k]) - nq + max(0, ot[k + 1] - ot[k]) - nt;
    q_start[s] = b * F + q0;  // bottom view = query (camera_models.py:3042)
    q_len[s] = nq;
    t_start[s] = b * F + t0;  // top view = train
    t_len[s] = nt;
  }
  overflow[b] = dropped;
}

// desc_c[(view*(B+1) + slot)*cap + k] = desc_view[src_view[slot*cap + k]] for the B new slots (1..B)
__global__ void gather_desc_kernel(const uint4* __restrict__ desc_top, const uint4* __restrict__ desc_bot,
                                   const int32_t* __restrict__ src_top, const int32_t* __restrict__ src_bot,
                                   const int32_t* __restrict__ n, int B, int cap, uint4* __restrict__ desc_c) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const int slot = blockIdx.y + 1;
  const int view = blockIdx.z;
  if (k >= n[slot]) return;
  const size_t row = (size_t)slot * cap + k;
  const int src = view == 0 ? src_top[row] : src_bot[row];
  const uint4* d = (view == 0 ? desc_top : desc_bot) + (size_t)src * 2;
  uint4* o = desc_c + ((size_t)(view * (B + 1) + slot) * cap + k) * 2;
  o[0] = __ldg(d);
  o[1] = __ldg(d + 1);
}

// Pair i tracks store slot i + 1 against its reference slot: slot i (consecutive frames) or ref_slot[i] (keyframe mode:
// the slot of the tracking reference, pose_est_tools.py:1489; -1 = pair switched off).  One segment per view and pair.
__global__ void temporal_segments_kernel(const int32_t* __restrict__ n, const int32_t* __restrict__ ref_slot, int B, int cap,
                                         int views, int32_t* __restrict__ q_start, int32_t* __restrict__ q_len,
                                         int32_t* __restrict__ t_start, int32_t* __restrict__ t_len) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= views * B) return;
  const int view = s / B, i = s % B;
  const int r = ref_slot ? ref_slot[i] : i;
  const bool on = r >= 0 && r <= B && r != i + 1;
  q_start[s] = (view * (B + 1) + i + 1) * cap;  // query = current frame (pose_est_tools.py:215)
  q_len[s] = on ? n[i + 1] : 0;
  t_start[s] = (view * (B + 1) + (on ? r : 0)) * cap;  // train = reference frame
  t_len[s] = on ? n[r] : 0;
}

// Stack the temporal matches of both views into one correspondence list per frame pair (pose_est_tools.py:752-778); with
// one view (RGB-D, pose_est_tools.py:912-914) the list is that view's matches and cam is NULL (central camera).
__global__ void __launch_bounds__(256)
assemble_kernel(const int32_t* __restrict__ m_q, const int32_t* __restrict__ m_t, const int32_t* __restrict__ m_count,
                const int32_t* __restrict__ q_start, int B, int cap, int views, const float* __restrict__ xyz,
                const float* __restrict__ b_top, const float* __restrict__ b_bot, float* __restrict__ p_ref,
                float* __restrict__ p_cur, float* __restrict__ f_cur, uint8_t* __restrict__ cam,
                int32_t* __restrict__ n_corr, int32_t* __restrict__ n_corr_top) {
  const int i = blockIdx.y;  // frame pair; blockIdx.x: 256 rows of its list (one block per pair left 116 of 148 SMs idle)
  const int c_top = m_count[i], c_bot = views == 2 ? m_count[B + i] : 0;
  const int total = c_top + c_bot;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    n_corr[i] = total;
    n_corr_top[i] = c_top;
  }
  const int cap2 = views * cap;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < total; k += gridDim.x * blockDim.x) {
    const int view = k < c_top ? 0 : 1;
    const int s = view * B + i;
    const int kk = view == 0 ? k : k - c_top;
    const int base = view * (B + 1) * cap;        // descriptor-store rows of this view start here
    const int rq = m_q[q_start[s] + kk] - base;   // store row of the current-frame correspondence
    const int rt = m_t[q_start[s] + kk] - base;   // store row of the reference-frame correspondence
    const size_t o = ((size_t)i * cap2 + k) * 3;
    const float* bq = (view == 0 ? b_top : b_bot) + (size_t)rq * 3;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      p_ref[o + d] = xyz[(size_t)rt * 3 + d];
      p_cur[o + d] = xyz[(size_t)rq * 3 + d];
      f_cur[o + d] = bq[d];
    }
    if (cam) cam[(size_t)i * cap2 + k] = (uint8_t)view;
  }
}

// Store slot `from` -> slot 0 (the tracking reference of what follows).  views == 1: uv_bot and b_bot are not read.
__global__ void carry_over_kernel(int B, int from, int cap, int views, float* __restrict__ uv_top, float* __restrict__ uv_bot,
                                  float* __restrict__ b_top, float* __restrict__ b_bot, float* __restrict__ xyz,
                                  uint32_t* __restrict__ desc_c, int32_t* __restrict__ n) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const int cnt = n[from];
  if (k == 0) n[0] = cnt;
  if (k >= cnt) return;
  const size_t src = (size_t)from * cap + k, dst = k;
  ((float2*)uv_top)[dst] = ((const float2*)uv_top)[src];
  if (views == 2) ((float2*)uv_bot)[dst] = ((const float2*)uv_bot)[src];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    b_top[3 * dst + c] = b_top[3 * src + c];
    if (views == 2) b_bot[3 * dst + c] = b_bot[3 * src + c];
    xyz[3 * dst + c] = xyz[3 * src + c];
  }
  for (int view = 0; view < views; ++view) {
    uint4* base = (uint4*)(desc_c + (size_t)view * (B + 1) * cap * 8);
    base[2 * dst] = base[2 * src];
    base[2 * dst + 1] = base[2 * src + 1];
  }
}

// Per source row: which 64-byte blocks any live panorama pixel may read (both tap rows, plus the slack of the wide loads).
// blocks[row * words + w] is a bitmap over blocks 64 w .. 64 w + 63 of that row.
__global__ void lut_row_blocks_kernel(const sos_lut_entry* __restrict__ lut, size_t n, int src_h, int src_w, int ch, int words,
                                      unsigned long long* __restrict__ blocks) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t e = lut[i];
  if (((e >> 48) & 0xF) == 0) return;   // no tap inside the image: nothing is read
  const int x0 = (int)(int16_t)(e & 0xFFFF), y0 = (int)(int16_t)((e >> 16) & 0xFFFF);
  const int lo = max(0, x0 * ch - 16), hi = min(src_w * ch, (x0 + 2) * ch + 24);
  if (hi <= lo) return;
  for (int y = y0; y <= y0 + 1; ++y)
    if (y >= 0 && y < src_h)
      for (int b = lo >> 6; b <= (hi - 1) >> 6; ++b) atomicOr(&blocks[(size_t)y * words + (b >> 6)], 1ull << (b & 63));
}

__global__ void stats_kernel(const int32_t* __restrict__ n, const int32_t* __restrict__ n_corr,
                             const int32_t* __restrict__ best_count, const int32_t* __restrict__ best_hyp, int B,
                             int32_t* __restrict__ stats) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  stats[4 * i + 0] = n[i + 1];       // triangulated stereo correspondences of the new frame
  stats[4 * i + 1] = n_corr[i];      // temporal correspondences handed to RANSAC
  stats[4 * i + 2] = best_count[i];  // RANSAC inliers
  stats[4 * i + 3] = best_hyp[i];
}

// Images-in step: the corners of one (frame, view) -> the bucketed feature rows sos_frontend_step reads, as
// FeatureFront.detect (features.py) builds them.  One block per (frame, view); the nb * N slots (bucket-major, strongest
// first) are scanned in tiles of the block: slot j of bucket k is kept iff j < count[k] and ORB kept it (border rule); kept
// slot number p becomes feature row p if p < F.  Bucket offsets are the prefix sums of kept slots clamped to F; rows past
// the last are zeroed.  A bucket whose selection refused its candidate list (count < 0) contributes nothing.
// stats [B, 2, 4]: corners accepted, corners kept by ORB, rows dropped by the F clamp, refused masks.
constexpr int DP_THREADS = 1024;

__global__ void __launch_bounds__(DP_THREADS)
detect_pack_kernel(const float2* __restrict__ xy, const int32_t* __restrict__ count, const uint8_t* __restrict__ keep,
                   const uint4* __restrict__ desc, int B, int nb, int N, int F, float2* __restrict__ px_top,
                   uint4* __restrict__ desc_top, int32_t* __restrict__ boff_top, float2* __restrict__ px_bot,
                   uint4* __restrict__ desc_bot, int32_t* __restrict__ boff_bot, int32_t* __restrict__ stats) {
  __shared__ int s_warp[DP_THREADS / 32];
  __shared__ int s_bucket[32];
  const int b = blockIdx.x, view = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t list0 = ((size_t)view * B + b) * nb;               // xy / count / keep / desc are [2, B, nb, N, ...]
  float2* px = (view == 0 ? px_top : px_bot) + (size_t)b * F;
  uint4* ds = (view == 0 ? desc_top : desc_bot) + (size_t)b * F * 2;
  int32_t* boff = (view == 0 ? boff_top : boff_bot) + (size_t)b * (nb + 1);
  if (threadIdx.x < 32) s_bucket[threadIdx.x] = 0;
  __syncthreads();
  const int total_slots = nb * N;
  int base = 0;
  for (int i0 = 0; i0 < total_slots; i0 += DP_THREADS) {
    const int i = i0 + threadIdx.x;
    bool kept = false;
    int k = 0;
    if (i < total_slots) {
      k = i / N;
      kept = (i - k * N) < count[list0 + k] && keep[list0 * N + i] != 0;
    }
    const unsigned vote = __ballot_sync(0xFFFFFFFFu, kept);
    if (lane == 0) s_warp[warp] = __popc(vote);
    __syncthreads();
    int before = 0, tile = 0;
    for (int w = 0; w < DP_THREADS / 32; ++w) {
      const int c = s_warp[w];
      if (w < warp) before += c;
      tile += c;
    }
    if (kept) {
      atomicAdd(&s_bucket[k], 1);
      const int pos = base + before + __popc(vote & ((1u << lane) - 1u));
      if (pos < F) {
        px[pos] = xy[list0 * N + i];
        const uint4* src = desc + (list0 * N + i) * 2;
        ds[2 * pos] = src[0];
        ds[2 * pos + 1] = src[1];
      }
    }
    base += tile;
    __syncthreads();
  }
  for (int r = base + threadIdx.x; r < F; r += DP_THREADS) {
    px[r] = make_float2(0.f, 0.f);
    ds[2 * r] = make_uint4(0u, 0u, 0u, 0u);
    ds[2 * r + 1] = make_uint4(0u, 0u, 0u, 0u);
  }
  if (threadIdx.x == 0) {
    int acc = 0, accepted = 0, refused = 0;
    boff[0] = 0;
    for (int k = 0; k < nb; ++k) {
      const int c = count[list0 + k];
      accepted += max(c, 0);
      refused += c < 0;
      acc += s_bucket[k];
      boff[k + 1] = min(acc, F);
    }
    int32_t* st = stats + ((size_t)b * 2 + view) * 4;
    st[0] = accepted;
    st[1] = base;
    st[2] = max(0, base - F);
    st[3] = refused;
  }
}

// RGB-D step, store stage (RGBDFrame.establish_keypoints, pose_est_tools.py:600-623): one block per frame b.  Keypoint row
// k < n_kp[b] (clamped to [0, cap]) is looked up at its truncated pixel (astype(np.uint), :612) and back-projected by
// rgbd_point, the arithmetic of sos_rgbd_backproject; a pixel outside the map (or a NaN coordinate) drops the keypoint.
// The valid rows are compacted in row order (kpts[valid], :618-623) into store slot b + 1, tiles of the block as in
// detect_pack_kernel: float keypoint coordinates (what the |du| gate reads), xyz, bearing, descriptor, input row; n[b + 1].
constexpr int RS_THREADS = 1024;

__global__ void __launch_bounds__(RS_THREADS)
rgbd_store_kernel(RgbdP c, const float* __restrict__ depth, int h, int w, const float2* __restrict__ px,
                  const uint4* __restrict__ desc, const int32_t* __restrict__ n_kp, int cap, double zmin, double zmax,
                  float2* __restrict__ uv, float* __restrict__ bearing, float* __restrict__ xyz, uint4* __restrict__ desc_c,
                  int32_t* __restrict__ src, int32_t* __restrict__ n) {
  __shared__ int s_warp[RS_THREADS / 32];
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rows = min(max(n_kp[b], 0), cap);
  const float* dmap = depth + (size_t)b * h * w;
  const size_t in0 = (size_t)b * cap, out0 = (size_t)(b + 1) * cap;
  int base = 0;
  for (int k0 = 0; k0 < rows; k0 += RS_THREADS) {
    const int k = k0 + threadIdx.x;
    float2 q = make_float2(0.f, 0.f);
    float p[3], f[3];
    bool ok = false;
    if (k < rows) {
      q = px[in0 + k];
      const float tx = truncf(q.x), ty = truncf(q.y);
      if (tx >= 0.f && tx < (float)w && ty >= 0.f && ty < (float)h)   // false for NaN; keeps the int conversion in range
        ok = rgbd_point(c, dmap, h, w, (int)tx, (int)ty, zmin, zmax, p, f);
    }
    const unsigned vote = __ballot_sync(0xFFFFFFFFu, ok);
    if (lane == 0) s_warp[warp] = __popc(vote);
    __syncthreads();
    int before = 0, tile = 0;
    for (int wi = 0; wi < RS_THREADS / 32; ++wi) {
      const int cnt = s_warp[wi];
      if (wi < warp) before += cnt;
      tile += cnt;
    }
    if (ok) {
      const size_t o = out0 + base + before + __popc(vote & ((1u << lane) - 1u));
      uv[o] = q;
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        xyz[3 * o + d] = p[d];
        bearing[3 * o + d] = f[d];
      }
      desc_c[2 * o] = desc[2 * (in0 + k)];
      desc_c[2 * o + 1] = desc[2 * (in0 + k) + 1];
      src[o] = k;
    }
    base += tile;
    __syncthreads();
  }
  if (threadIdx.x == 0) n[b + 1] = base;
}

}  // namespace

// The inputs of one step, which are also the key of its captured graph: a feature step (omni, px_top, desc_top, boff_top,
// px_bot, desc_bot, boff_bot), an images-in step (omni; the feature pointers are the front-end's own buffers) or an RGB-D
// step (depth, px, desc, n_kp).
enum StepKind { STEP_FEATURES = 0, STEP_IMAGES = 1, STEP_RGBD = 2 };
struct StepIn {
  const void* p[7];
  intptr_t kind;
};

struct sos_frontend {
  sos_ctx* ctx = nullptr;     // private (own scratch arena)
  sos_ctx* parent = nullptr;  // the caller's context (launch accounting)
  sos_frontend_config cfg;     // RGB-D: the fields stage B reads (batch, cap = max_kp, RANSAC and refinement, keyframe_mode)
  bool rgbd = false;           // made by sos_frontend_create_rgbd
  int views = 2;               // 2 (SOS) or 1 (RGB-D)
  sos_rgbd_frontend_config rgbd_cfg;
  const sos_lut_entry* lut = nullptr;
  const uint32_t* hyp = nullptr;
  // device state
  sos_frontend_buffers d;
  std::vector<void*> owned;
  // staging for the host API (double buffered)
  static constexpr int DEPTH = 2;
  struct Stage {
    uint8_t* omni = nullptr;      // RGB-D: depth maps (float32); px_top / desc_top hold the keypoints
    int32_t* n_kp = nullptr;      // RGB-D
    float *px_top = nullptr, *px_bot = nullptr;
    uint32_t *desc_top = nullptr, *desc_bot = nullptr;
    int32_t *boff_top = nullptr, *boff_bot = nullptr;
    float* h_poses = nullptr;     // pinned
    int32_t* h_stats = nullptr;   // pinned
    cudaEvent_t copied = nullptr, done = nullptr;
    bool in_flight = false;
  } stage[DEPTH];
  cudaStream_t copy_stream = nullptr;
  // host API: only the bytes of the omni image that some LUT entry can read are uploaded, in bands of rows
  struct Band {
    int row0, nrows, x0_bytes, width_bytes;
  };
  std::vector<Band> bands;
  int64_t omni_bytes_per_frame = 0;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;  // fences against the caller's stream
  // the remap is a branch of its own in the step (nothing later in the step reads the panoramas): it fills the SMs while the
  // many small, latency-bound kernels of the matching / RANSAC chain run
  cudaStream_t remap_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  bool remap_forked = false;
  int next_stage = 0;
  // graph cache keyed on the inputs of a step
  struct GraphEntry {
    StepIn key;
    cudaGraphExec_t exec = nullptr;
    int launches = 0;
    const void* arena = nullptr;   // fe->ctx->arena at capture
  };
  std::vector<GraphEntry> graphs;
  bool use_graph = true;
  // images-in step (sos_frontend_set_detector): front-end-owned buffers, allocated by the first set_detector
  struct Detector {
    bool on = false;
    sos_detect_config cfg;
    int32_t overlap[2] = {0, 0};         // masks of the view share pixels (read back once, when they are packed)
    uint8_t *med = nullptr, *gray = nullptr;   // [B, 2, rows, cols, 3] median output, [B, 2, rows, cols] gray
    uint8_t* blur = nullptr;             // [B, 2, rows, cols] ORB's blurred gray (in the arena it could regrow
                                         // the arena that the feature steps' graphs hold)
    uint32_t* mask_bits[2] = {nullptr, nullptr};
    int32_t* flags = nullptr;            // [2] overlap flags of the mask packing
    // GFT scratch, shared by the two views (they run one after the other)
    float* eig = nullptr;                // [B, rows, cols]
    uint32_t* max_bits = nullptr;        // [B * nb]
    int32_t* cand = nullptr;             // [B * nb] candidates per list
    unsigned long long* keys = nullptr;  // [B * nb * SOS_GFT_CAP]
    int32_t* rank = nullptr;             // [B, rows, cols], all -1: cleared once, the selection leaves it so
    float* xy = nullptr;                 // [2, B, nb, N, 2]  corners, N = corners_per_bucket
    int32_t* count = nullptr;            // [2, B, nb]
    int32_t* kp_image = nullptr;         // [2, B, nb, N] image of each corner in gray (2 b + view)
    uint32_t* kp_desc = nullptr;         // [2, B, nb, N, 8]
    uint8_t* kp_keep = nullptr;          // [2, B, nb, N]
    sos_frontend_features f;             // packed features + detect_stats
  } det;
};

namespace {

template <typename T>
int fe_alloc(sos_frontend* fe, T** out, size_t count) {
  void* p = nullptr;
  const size_t bytes = sos_align_up(count * sizeof(T) + 256, 256);
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) {
    sos_set_error("sos_frontend: cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    return SOS_ERR_NOMEM;
  }
  cudaMemsetAsync(p, 0, bytes, fe->ctx->stream);
  fe->owned.push_back(p);
  *out = (T*)p;
  return SOS_OK;
}

// Images-in step, ahead of stage A: remap, then the feature front of FeatureFront.detect (features.py) on the panoramas —
// 11 x 11 median and BGR2GRAY over both views at once, Shi-Tomasi per view, ORB description over both views — and
// detect_pack_kernel into the feature arrays stage A reads.  Nothing is read back: a candidate list over the selection's
// capacity yields no corners (counted in detect_stats) instead of failing the step.
int enqueue_detect(sos_frontend* fe, const uint8_t* omni) {
  sos_ctx* ctx = fe->ctx;
  const sos_frontend_config& c = fe->cfg;
  sos_frontend::Detector& dt = fe->det;
  const int B = c.batch, nb = c.n_buckets, N = dt.cfg.corners_per_bucket, H = c.pano_rows, W = c.pano_cols;
  int rc = sos_remap_u8(ctx, omni, B, c.src_h, c.src_w, c.channels, fe->lut, 2, H, W, c.border, c.background, fe->d.pano);
  if (rc) return rc;
  const uint8_t* bgr = fe->d.pano;
  if (dt.cfg.median) {
    rc = sos_median_blur_11(ctx, fe->d.pano, 2 * B, H, W, 3, dt.med);
    if (rc) return rc;
    bgr = dt.med;
  }
  rc = sos_bgr_to_gray(ctx, bgr, (size_t)2 * B * H * W, dt.gray);
  if (rc) return rc;
  const size_t plane = (size_t)H * W;
  for (int view = 0; view < 2; ++view) {
    sos_gft_work w;
    w.mask_bits = dt.mask_bits[view];
    w.eig = dt.eig;
    w.max_bits = dt.max_bits;
    w.counts = dt.cand;
    w.keys = dt.keys;
    w.rank_img = dt.rank;
    float* xy = dt.xy + (size_t)view * B * nb * N * 2;
    int32_t* count = dt.count + (size_t)view * B * nb;
    // the gray image of view v of frame b is plane 2 b + v
    rc = sos_gft_candidates(ctx, w, dt.gray + view * plane, 2 * plane, B, H, W, nb, dt.cfg.quality_level);
    // the counts are not known here: every block gets the shared memory of a full list (62 registers x 1024 threads leave
    // room for one block per SM whatever the shared memory, so smaller lists would not share an SM anyway)
    if (!rc) rc = sos_gft_select(ctx, w, B, H, W, nb, N, dt.cfg.min_distance, dt.overlap[view] != 0, SOS_GFT_CAP, xy, count);
    if (rc) return rc;
  }
  rc = sos_orb_describe_into(ctx, dt.gray, 2 * B, H, W, dt.xy, nullptr, dt.kp_image, 2 * B * nb * N, dt.kp_desc, dt.kp_keep,
                             dt.blur);
  if (rc) return rc;
  const sos_frontend_features& f = dt.f;
  detect_pack_kernel<<<dim3(B, 2), DP_THREADS, 0, ctx->stream>>>((const float2*)dt.xy, dt.count, dt.kp_keep,
                                                                 (const uint4*)dt.kp_desc, B, nb, N, c.max_feat_per_view,
                                                                 (float2*)f.px_top, (uint4*)f.desc_top, f.boff_top,
                                                                 (float2*)f.px_bot, (uint4*)f.desc_bot, f.boff_bot,
                                                                 f.detect_stats);
  SOS_LAUNCHED_AS(ctx, "detect_pack_kernel");
  return SOS_OK;
}

// Stage A of a step (remap, stereo matching, lifting + triangulation into store slots 1..B), enqueued on ctx->stream.
// images: the panoramas were already made by enqueue_detect.
int enqueue_stage_a(sos_frontend* fe, const uint8_t* omni, const float* px_top, const uint32_t* desc_top,
                 const int32_t* boff_top, const float* px_bot, const uint32_t* desc_bot, const int32_t* boff_bot, bool images) {
  sos_ctx* ctx = fe->ctx;
  const sos_frontend_config& c = fe->cfg;
  sos_frontend_buffers& d = fe->d;
  const int B = c.batch, nb = c.n_buckets, F = c.max_feat_per_view, cap = c.cap;
  int rc;
  // step 1, as a parallel branch (fork here, join at the end of the step).  Round 1 measured no gain from this — then the
  // chain was three long kernels that filled the GPU; now a fifth of the step is small launches that leave most SMs idle.
  // Per-kernel profiling runs keep it in line so that every kernel is timed alone.  In an images-in step the remap feeds
  // the detection and has already run.
  fe->remap_forked = fe->remap_stream != nullptr && !ctx->prof && !images;
  if (fe->remap_forked) {
    SOS_CUDA(cudaEventRecord(fe->ev_fork, ctx->stream));
    SOS_CUDA(cudaStreamWaitEvent(fe->remap_stream, fe->ev_fork, 0));
    cudaStream_t main_stream = ctx->stream;
    ctx->stream = fe->remap_stream;
    rc = sos_remap_u8(ctx, omni, B, c.src_h, c.src_w, c.channels, fe->lut, 2, c.pano_rows, c.pano_cols, c.border,
                      c.background, d.pano);
    ctx->stream = main_stream;
    if (rc) return rc;
    SOS_CUDA(cudaEventRecord(fe->ev_join, fe->remap_stream));
  } else if (!images) {
    rc = sos_remap_u8(ctx, omni, B, c.src_h, c.src_w, c.channels, fe->lut, 2, c.pano_rows, c.pano_cols, c.border,
                      c.background, d.pano);
    if (rc) return rc;
  }
  // step 2a: stereo matching per bucket
  const int S = B * nb;
  stereo_segments_kernel<<<sos_div_up(B, 128), 128, 0, ctx->stream>>>(boff_top, boff_bot, B, nb, F, c.max_feat_per_bucket,
                                                                       d.st_q_start, d.st_q_len, d.st_t_start, d.st_t_len,
                                                                       d.overflow);
  SOS_LAUNCHED_AS(ctx, "stereo_segments_kernel");
  rc = sos_hamming_top2(ctx, desc_bot, desc_top, d.st_q_start, d.st_q_len, d.st_t_start, d.st_t_len, S,
                        c.max_feat_per_bucket, c.max_feat_per_bucket, d.st_idx0, d.st_d0, nullptr, nullptr);
  if (rc) return rc;
  rc = sos_match_select(ctx, SOS_MATCH_NN, 0.75, d.st_idx0, d.st_d0, nullptr, nullptr, d.st_q_start, d.st_q_len,
                        d.st_t_start, S, px_bot, px_top, c.stereo_max_du, c.stereo_min_dv, d.st_pair_q, d.st_pair_t,
                        d.st_pair_d, d.st_pair_count);
  if (rc) return rc;
  // steps 3+4 into store slots 1..B
  rc = sos_stereo_lift_triangulate(ctx, c.pano_top, c.pano_bot, px_top, px_bot, d.st_pair_q, d.st_pair_t, d.st_pair_count,
                                   d.st_q_start, B, nb, c.max_feat_per_bucket, B * F, c.f_top, c.f_bot, c.min_range,
                                   c.max_range, c.homogeneous_norm, cap,
                                   d.uv_top + (size_t)cap * 2, d.uv_bot + (size_t)cap * 2, d.b_top + (size_t)cap * 3,
                                   d.b_bot + (size_t)cap * 3, d.xyz + (size_t)cap * 3, d.src_top + cap, d.src_bot + cap,
                                   d.n + 1);
  if (rc) return rc;
  {
    dim3 grid(sos_div_up(cap, 128), B, 2);
    gather_desc_kernel<<<grid, 128, 0, ctx->stream>>>((const uint4*)desc_top, (const uint4*)desc_bot, d.src_top, d.src_bot,
                                                      d.n, B, cap, (uint4*)d.desc_c);
    SOS_LAUNCHED_AS(ctx, "gather_desc_kernel");
  }
  return SOS_OK;
}

// Stage B: temporal matching against the reference slots, RANSAC, refinement.  Re-runnable on its own (sos_frontend_retrack).
// SOS: two views and the two-mirror rig; RGB-D: one view and a central camera (rig NULL, pyopengv.absolute_pose_ransac).
int enqueue_stage_b(sos_frontend* fe) {
  sos_ctx* ctx = fe->ctx;
  const sos_frontend_config& c = fe->cfg;
  sos_frontend_buffers& d = fe->d;
  const int B = c.batch, cap = c.cap, V = fe->views, stride = V * cap;
  const double* rig = V == 2 ? c.rig : nullptr;
  const int n_cams = V == 2 ? 2 : 0;
  int rc;
  // step 2b: temporal matching, V views x B pairs
  temporal_segments_kernel<<<sos_div_up(V * B, 128), 128, 0, ctx->stream>>>(d.n, c.keyframe_mode ? d.ref_slot : nullptr, B, cap,
                                                                            V, d.tm_q_start, d.tm_q_len, d.tm_t_start, d.tm_t_len);
  SOS_LAUNCHED_AS(ctx, "temporal_segments_kernel");
  rc = sos_hamming_top2(ctx, d.desc_c, d.desc_c, d.tm_q_start, d.tm_q_len, d.tm_t_start, d.tm_t_len, V * B, cap, cap,
                        d.tm_idx0, d.tm_d0, nullptr, nullptr);
  if (rc) return rc;
  // pixel gate on u only (pose_est_tools.py:245-247): coordinates of the compacted store, all views in one array
  rc = sos_match_select(ctx, SOS_MATCH_NN, 0.75, d.tm_idx0, d.tm_d0, nullptr, nullptr, d.tm_q_start, d.tm_q_len,
                        d.tm_t_start, V * B, d.uv_c, d.uv_c, c.temporal_max_du, -1.0, d.tm_pair_q, d.tm_pair_t, d.tm_pair_d,
                        d.tm_pair_count);
  if (rc) return rc;
  assemble_kernel<<<dim3(sos_div_up(stride, 256), B), 256, 0, ctx->stream>>>(d.tm_pair_q, d.tm_pair_t, d.tm_pair_count, d.tm_q_start, B, cap, V, d.xyz, d.b_top,
                                              d.b_bot, d.p_ref, d.p_cur, d.f_cur, d.cam, d.n_corr, d.n_corr_top);
  SOS_LAUNCHED_AS(ctx, "assemble_kernel");
  // step 5
  rc = c.solver == SOS_SOLVER_P3P
           ? sos_ransac_p3p(ctx, d.p_ref, d.f_cur, d.cam, d.n_corr, B, stride, rig, n_cams, fe->hyp, c.n_hyp, 0, c.ransac_threshold,
                            d.ransac_pose, d.best_hyp, d.best_count, d.inlier_mask, nullptr, nullptr)
           : sos_ransac_p3d(ctx, d.p_ref, d.p_cur, d.f_cur, d.cam, d.n_corr, B, stride, rig, n_cams, fe->hyp, c.n_hyp, 0,
                            c.score_mode, c.ransac_threshold, d.ransac_pose, d.best_hyp, d.best_count, d.inlier_mask, nullptr,
                            nullptr);
  if (rc) return rc;
  if (c.refit == SOS_REFINE_LM) {
    rc = sos_refine_pose(ctx, d.p_ref, d.f_cur, d.cam, d.inlier_mask, d.n_corr, B, stride, rig, n_cams, d.ransac_pose,
                         c.refine_iters > 0 ? c.refine_iters : 20, 0, d.pose, nullptr, d.refine_stats);
    if (rc) return rc;
  } else if (c.refit == SOS_REFINE_ARUN) {
    rc = sos_refit_inliers(ctx, d.p_ref, d.p_cur, d.inlier_mask, d.n_corr, B, stride, d.pose, d.n_refit);
    if (rc) return rc;
  } else {
    SOS_CUDA(cudaMemcpyAsync(d.pose, d.ransac_pose, (size_t)B * 12 * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
  }
  stats_kernel<<<sos_div_up(B, 128), 128, 0, ctx->stream>>>(d.n, d.n_corr, d.best_count, d.best_hyp, B, d.stats);
  SOS_LAUNCHED_AS(ctx, "stats_kernel");
  return SOS_OK;
}

int enqueue_carry(sos_frontend* fe, int from) {
  sos_ctx* ctx = fe->ctx;
  sos_frontend_buffers& d = fe->d;
  carry_over_kernel<<<sos_div_up(fe->cfg.cap, 256), 256, 0, ctx->stream>>>(fe->cfg.batch, from, fe->cfg.cap, fe->views, d.uv_top, d.uv_bot,
                                                                            d.b_top, d.b_bot, d.xyz, d.desc_c, d.n);
  SOS_LAUNCHED_AS(ctx, "carry_over_kernel");
  return SOS_OK;
}

// The kernel chain of one step.  Consecutive mode ends by carrying the last frame over as the reference of the next
// step (slot B -> slot 0, one kernel instead of 8 copy nodes); in keyframe mode the caller promotes a slot itself.
// images: the features are detected on the step's panoramas first (the px / desc / boff pointers are fe->det.f's).
int enqueue_step(sos_frontend* fe, const uint8_t* omni, const float* px_top, const uint32_t* desc_top,
                 const int32_t* boff_top, const float* px_bot, const uint32_t* desc_bot, const int32_t* boff_bot, bool images) {
  int rc = images ? enqueue_detect(fe, omni) : SOS_OK;
  if (rc == SOS_OK) rc = enqueue_stage_a(fe, omni, px_top, desc_top, boff_top, px_bot, desc_bot, boff_bot, images);
  if (rc == SOS_OK) rc = enqueue_stage_b(fe);
  if (rc == SOS_OK && !fe->cfg.keyframe_mode) rc = enqueue_carry(fe, fe->cfg.batch);
  if (fe->remap_forked) {   // join the remap branch (also on an error path: a capture must not end with an open fork)
    fe->remap_forked = false;
    SOS_CUDA(cudaStreamWaitEvent(fe->ctx->stream, fe->ev_join, 0));
  }
  return rc;
}

// RGB-D step: store stage into slots 1..B, stage B, and in consecutive mode the carry-over of slot B.
int enqueue_rgbd_step(sos_frontend* fe, const float* depth, const float* px, const uint32_t* desc, const int32_t* n_kp) {
  sos_ctx* ctx = fe->ctx;
  const sos_rgbd_frontend_config& r = fe->rgbd_cfg;
  sos_frontend_buffers& d = fe->d;
  RgbdP cam;
  for (int i = 0; i < SOS_RGBD_NPARAMS; ++i) cam.v[i] = r.cam[i];
  rgbd_store_kernel<<<r.batch, RS_THREADS, 0, ctx->stream>>>(cam, depth, r.height, r.width, (const float2*)px, (const uint4*)desc,
                                                              n_kp, r.max_kp, r.min_z, r.max_z, (float2*)d.uv_c, d.b_top, d.xyz,
                                                              (uint4*)d.desc_c, d.src_top, d.n);
  SOS_LAUNCHED_AS(ctx, "rgbd_store_kernel");
  int rc = enqueue_stage_b(fe);
  if (rc == SOS_OK && !fe->cfg.keyframe_mode) rc = enqueue_carry(fe, fe->cfg.batch);
  return rc;
}

int enqueue_any(sos_frontend* fe, const StepIn& in) {
  const void* const* p = in.p;
  if (in.kind == STEP_RGBD)
    return enqueue_rgbd_step(fe, (const float*)p[0], (const float*)p[1], (const uint32_t*)p[2], (const int32_t*)p[3]);
  return enqueue_step(fe, (const uint8_t*)p[0], (const float*)p[1], (const uint32_t*)p[2], (const int32_t*)p[3],
                      (const float*)p[4], (const uint32_t*)p[5], (const int32_t*)p[6], in.kind == STEP_IMAGES);
}

StepIn sos_step_in(const uint8_t* omni, const float* px_top, const uint32_t* desc_top, const int32_t* boff_top,
                   const float* px_bot, const uint32_t* desc_bot, const int32_t* boff_bot, bool images) {
  StepIn in;
  memset(&in, 0, sizeof(in));
  const void* ptrs[7] = {omni, px_top, desc_top, boff_top, px_bot, desc_bot, boff_bot};
  memcpy(in.p, ptrs, sizeof(ptrs));
  in.kind = images ? STEP_IMAGES : STEP_FEATURES;
  return in;
}

StepIn rgbd_step_in(const float* depth, const float* px, const uint32_t* desc, const int32_t* n_kp) {
  StepIn in;
  memset(&in, 0, sizeof(in));
  in.p[0] = depth; in.p[1] = px; in.p[2] = desc; in.p[3] = n_kp;
  in.kind = STEP_RGBD;
  return in;
}

// Eager run, or the captured graph of these inputs (captured after one eager run).  An images-in step's feature pointers
// are replaced by fe->det.f's.
int run_step(sos_frontend* fe, StepIn key) {
  sos_ctx* ctx = fe->ctx;
  if (key.kind == STEP_IMAGES) {
    const sos_frontend_features& f = fe->det.f;
    const void* ptrs[6] = {f.px_top, f.desc_top, f.boff_top, f.px_bot, f.desc_bot, f.boff_bot};
    memcpy(key.p + 1, ptrs, sizeof(ptrs));
  }
  if (!fe->use_graph || ctx->prof) return enqueue_any(fe, key);
  // a graph holds the scratch arena's address: one captured before an eager run regrew the arena must not be replayed
  for (size_t i = 0; i < fe->graphs.size();) {
    if (fe->graphs[i].arena != ctx->arena) {
      cudaGraphExecDestroy(fe->graphs[i].exec);
      fe->graphs.erase(fe->graphs.begin() + i);
    } else {
      ++i;
    }
  }
  for (auto& g : fe->graphs) {
    if (memcmp(&g.key, &key, sizeof(key)) == 0) {
      SOS_CUDA(cudaGraphLaunch(g.exec, ctx->stream));
      ctx->launches += g.launches;
      return SOS_OK;
    }
  }
  // first time with these buffers: run once eagerly (sizes the scratch arena), then capture
  const int64_t before = ctx->launches;
  int rc = enqueue_any(fe, key);
  if (rc) return rc;
  const int launches = (int)(ctx->launches - before);
  fe->d.launches_per_step = launches;
  SOS_CUDA(cudaStreamSynchronize(ctx->stream));
  // the eager run advanced the carried state; capturing does not execute anything
  cudaGraph_t graph = nullptr;
  SOS_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
  const int64_t l0 = ctx->launches;
  rc = enqueue_any(fe, key);
  ctx->launches = l0;
  cudaError_t e = cudaStreamEndCapture(ctx->stream, &graph);
  if (rc) {
    if (graph) cudaGraphDestroy(graph);
    return rc;
  }
  if (e != cudaSuccess) {
    sos_set_error("sos_frontend: graph capture failed: %s", cudaGetErrorString(e));
    return SOS_ERR_CUDA;
  }
  sos_frontend::GraphEntry ge;
  ge.key = key;
  ge.launches = launches;
  ge.arena = ctx->arena;   // the capture refuses to grow the arena, so this is the address the graph holds
  SOS_CUDA(cudaGraphInstantiate(&ge.exec, graph, 0));
  cudaGraphDestroy(graph);
  if (fe->graphs.size() >= 8) {
    cudaGraphExecDestroy(fe->graphs.front().exec);
    fe->graphs.erase(fe->graphs.begin());
  }
  fe->graphs.push_back(ge);
  return SOS_OK;
}

}  // namespace

namespace {
// A front-end without buffers: private context (same device, but its own scratch arena — the arena address is baked into
// the captured graphs, so no other caller may regrow it), its own compute stream (the caller's may be the legacy default
// stream, which cannot be captured; every step is fenced against the caller's current stream with events, so the caller
// sees ordinary stream semantics) and, for SOS, the remap branch.  On failure everything made so far is destroyed.
int fe_open(sos_ctx* ctx, bool remap_branch, sos_frontend** out) {
  SOS_CUDA(cudaSetDevice(ctx->device));
  sos_frontend* fe = new sos_frontend();
  fe->ctx = new sos_ctx();
  fe->ctx->device = ctx->device;
#define FE_CUDA(call)                                                                               \
  do {                                                                                              \
    cudaError_t e__ = (call);                                                                       \
    if (e__ != cudaSuccess) {                                                                       \
      sos_set_error("sos_frontend_create: %s failed: %s", #call, cudaGetErrorString(e__));          \
      sos_frontend_destroy(fe);                                                                     \
      return SOS_ERR_CUDA;                                                                          \
    }                                                                                               \
  } while (0)
  int prio_lo = 0, prio_hi = 0;   // (numerically lower = higher priority)
  FE_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  FE_CUDA(cudaStreamCreateWithPriority(&fe->ctx->stream, cudaStreamNonBlocking, prio_hi));
  fe->ctx->own_stream = true;
  FE_CUDA(cudaEventCreateWithFlags(&fe->ev_in, cudaEventDisableTiming));
  FE_CUDA(cudaEventCreateWithFlags(&fe->ev_out, cudaEventDisableTiming));
  if (remap_branch) {
    // lowest priority for the remap branch: the chain's kernels take the SMs they can use first, the remap's blocks fill
    // what is left (measured: 1.321 -> 1.303 ms per C2 step; shorter remap blocks to free SMs sooner were slower)
    FE_CUDA(cudaStreamCreateWithPriority(&fe->remap_stream, cudaStreamNonBlocking, prio_lo));
    FE_CUDA(cudaEventCreateWithFlags(&fe->ev_fork, cudaEventDisableTiming));
    FE_CUDA(cudaEventCreateWithFlags(&fe->ev_join, cudaEventDisableTiming));
  }
#undef FE_CUDA
  fe->ctx->sm_count = ctx->sm_count;
  fe->parent = ctx;
  memset(&fe->d, 0, sizeof(fe->d));
  *out = fe;
  return SOS_OK;
}

// The zero fills of fe_alloc were queued on the private stream: finish them before anybody can look at the buffers.
int fe_finish(sos_frontend* fe, sos_ctx* ctx, int rc, sos_frontend** out) {
  if (rc == SOS_OK) {
    cudaError_t e = cudaStreamSynchronize(fe->ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
      sos_set_error("sos_frontend_create: cudaStreamSynchronize failed: %s", cudaGetErrorString(e));
      rc = SOS_ERR_CUDA;
    }
  }
  if (rc != SOS_OK) {
    sos_frontend_destroy(fe);
    return rc;
  }
  *out = fe;
  return SOS_OK;
}
}  // namespace

extern "C" int sos_frontend_create(sos_ctx* ctx, const sos_frontend_config* cfg, const sos_lut_entry* lut,
                                   const uint32_t* hyp, sos_frontend** out) {
  SOS_CHECK_ARG(ctx && cfg && lut && hyp && out, "NULL argument");
  SOS_CHECK_ARG(cfg->batch > 0 && cfg->batch <= 4096, "batch out of range");
  SOS_CHECK_ARG(cfg->channels == 1 || cfg->channels == 3 || cfg->channels == 4, "channels must be 1, 3 or 4");
  SOS_CHECK_ARG(cfg->n_buckets > 0 && cfg->max_feat_per_view > 0 && cfg->max_feat_per_bucket > 0 && cfg->cap > 0, "bad capacity");
  SOS_CHECK_ARG(cfg->n_hyp >= 0, "negative n_hyp");
  SOS_CHECK_ARG(cfg->solver == SOS_SOLVER_ARUN || cfg->solver == SOS_SOLVER_P3P, "unknown solver");
  SOS_CHECK_ARG(cfg->solver != SOS_SOLVER_P3P || cfg->score_mode == SOS_SCORE_BEARING, "the bearing-only solver scores bearings");
  sos_frontend* fe = nullptr;
  int rc = fe_open(ctx, true, &fe);
  if (rc) return rc;
  fe->cfg = *cfg;
  fe->lut = lut;
  fe->hyp = hyp;
  const sos_frontend_config& c = fe->cfg;
  const size_t B = c.batch, F = c.max_feat_per_view, cap = c.cap, S = B * c.n_buckets, slots = B + 1;
  sos_frontend_buffers& d = fe->d;
#define FE_ALLOC(field, count) \
  if (rc == SOS_OK) rc = fe_alloc(fe, &d.field, (count))
  FE_ALLOC(pano, B * 2 * c.pano_rows * c.pano_cols * c.channels);
  FE_ALLOC(st_q_start, S); FE_ALLOC(st_q_len, S); FE_ALLOC(st_t_start, S); FE_ALLOC(st_t_len, S);
  FE_ALLOC(st_idx0, B * F); FE_ALLOC(st_d0, B * F);
  FE_ALLOC(st_pair_q, B * F); FE_ALLOC(st_pair_t, B * F); FE_ALLOC(st_pair_d, B * F); FE_ALLOC(st_pair_count, S);
  // compacted per-frame store: uv_c holds both views back to back so that descriptor-store rows index it directly
  FE_ALLOC(uv_c, 2 * slots * cap * 2);
  d.uv_top = d.uv_c;
  d.uv_bot = d.uv_c + slots * cap * 2;
  FE_ALLOC(b_top, slots * cap * 3); FE_ALLOC(b_bot, slots * cap * 3); FE_ALLOC(xyz, slots * cap * 3);
  FE_ALLOC(src_top, slots * cap); FE_ALLOC(src_bot, slots * cap); FE_ALLOC(n, slots);
  FE_ALLOC(desc_c, 2 * slots * cap * 8);
  FE_ALLOC(tm_q_start, 2 * B); FE_ALLOC(tm_q_len, 2 * B); FE_ALLOC(tm_t_start, 2 * B); FE_ALLOC(tm_t_len, 2 * B);
  FE_ALLOC(tm_idx0, 2 * slots * cap); FE_ALLOC(tm_d0, 2 * slots * cap);
  FE_ALLOC(tm_pair_q, 2 * slots * cap); FE_ALLOC(tm_pair_t, 2 * slots * cap); FE_ALLOC(tm_pair_d, 2 * slots * cap);
  FE_ALLOC(tm_pair_count, 2 * B);
  FE_ALLOC(p_ref, B * 2 * cap * 3); FE_ALLOC(p_cur, B * 2 * cap * 3); FE_ALLOC(f_cur, B * 2 * cap * 3);
  FE_ALLOC(cam, B * 2 * cap); FE_ALLOC(n_corr, B); FE_ALLOC(n_corr_top, B);
  FE_ALLOC(ransac_pose, B * 12); FE_ALLOC(pose, B * 12); FE_ALLOC(best_hyp, B); FE_ALLOC(best_count, B);
  FE_ALLOC(n_refit, B); FE_ALLOC(inlier_mask, B * 2 * cap); FE_ALLOC(stats, B * 4); FE_ALLOC(refine_stats, B * 4); FE_ALLOC(ref_slot, B); FE_ALLOC(overflow, B);
#undef FE_ALLOC
  d.batch = c.batch;
  d.cap = c.cap;
  d.views = 2;
  return fe_finish(fe, ctx, rc, out);
}

extern "C" int sos_frontend_create_rgbd(sos_ctx* ctx, const sos_rgbd_frontend_config* cfg, const uint32_t* hyp,
                                        sos_frontend** out) {
  SOS_CHECK_ARG(ctx && cfg && hyp && out, "NULL argument");
  SOS_CHECK_ARG(cfg->batch > 0 && cfg->batch <= 4096, "batch out of range");
  SOS_CHECK_ARG(cfg->height > 0 && cfg->width > 0 && (long long)cfg->height * cfg->width < (1ll << 31), "bad depth map size");
  SOS_CHECK_ARG(cfg->max_kp > 0 && (long long)(cfg->batch + 1) * cfg->max_kp < (1ll << 31), "bad max_kp");
  SOS_CHECK_ARG(cfg->n_hyp >= 0, "negative n_hyp");
  SOS_CHECK_ARG(cfg->solver == SOS_SOLVER_ARUN || cfg->solver == SOS_SOLVER_P3P, "unknown solver");
  SOS_CHECK_ARG(cfg->refit == SOS_REFINE_NONE || cfg->refit == SOS_REFINE_ARUN || cfg->refit == SOS_REFINE_LM, "unknown refit");
  sos_frontend* fe = nullptr;
  int rc = fe_open(ctx, false, &fe);
  if (rc) return rc;
  fe->rgbd = true;
  fe->views = 1;
  fe->rgbd_cfg = *cfg;
  fe->hyp = hyp;
  // what stage B, the keyframe calls and the host path read
  sos_frontend_config& c = fe->cfg;
  memset(&c, 0, sizeof(c));
  c.batch = cfg->batch;
  c.cap = cfg->max_kp;
  c.n_hyp = cfg->n_hyp;
  c.score_mode = SOS_SCORE_BEARING;
  c.refit = cfg->refit;
  c.refine_iters = cfg->refine_iters;
  c.keyframe_mode = cfg->keyframe_mode;
  c.solver = cfg->solver;
  c.ransac_threshold = cfg->ransac_threshold;
  c.temporal_max_du = cfg->temporal_max_du;
  const size_t B = c.batch, cap = c.cap, slots = B + 1;
  sos_frontend_buffers& d = fe->d;
#define FE_ALLOC(field, count) \
  if (rc == SOS_OK) rc = fe_alloc(fe, &d.field, (count))
  FE_ALLOC(uv_c, slots * cap * 2);
  d.uv_top = d.uv_c;
  FE_ALLOC(b_top, slots * cap * 3); FE_ALLOC(xyz, slots * cap * 3); FE_ALLOC(src_top, slots * cap); FE_ALLOC(n, slots);
  FE_ALLOC(desc_c, slots * cap * 8);
  FE_ALLOC(tm_q_start, B); FE_ALLOC(tm_q_len, B); FE_ALLOC(tm_t_start, B); FE_ALLOC(tm_t_len, B);
  FE_ALLOC(tm_idx0, slots * cap); FE_ALLOC(tm_d0, slots * cap);
  FE_ALLOC(tm_pair_q, slots * cap); FE_ALLOC(tm_pair_t, slots * cap); FE_ALLOC(tm_pair_d, slots * cap);
  FE_ALLOC(tm_pair_count, B);
  FE_ALLOC(p_ref, B * cap * 3); FE_ALLOC(p_cur, B * cap * 3); FE_ALLOC(f_cur, B * cap * 3);
  FE_ALLOC(n_corr, B); FE_ALLOC(n_corr_top, B);
  FE_ALLOC(ransac_pose, B * 12); FE_ALLOC(pose, B * 12); FE_ALLOC(best_hyp, B); FE_ALLOC(best_count, B);
  FE_ALLOC(n_refit, B); FE_ALLOC(inlier_mask, B * cap); FE_ALLOC(stats, B * 4); FE_ALLOC(refine_stats, B * 4); FE_ALLOC(ref_slot, B);
#undef FE_ALLOC
  d.batch = c.batch;
  d.cap = c.cap;
  d.views = 1;
  return fe_finish(fe, ctx, rc, out);
}

extern "C" int sos_frontend_destroy(sos_frontend* fe) {
  if (!fe) return SOS_OK;
  cudaSetDevice(fe->ctx->device);
  if (fe->ctx->stream) cudaStreamSynchronize(fe->ctx->stream);
  if (fe->copy_stream) cudaStreamSynchronize(fe->copy_stream);
  if (fe->remap_stream) cudaStreamSynchronize(fe->remap_stream);
  for (auto& g : fe->graphs) cudaGraphExecDestroy(g.exec);
  for (void* p : fe->owned) cudaFree(p);
  for (auto& s : fe->stage) {
    if (s.h_poses) cudaFreeHost(s.h_poses);
    if (s.h_stats) cudaFreeHost(s.h_stats);
    if (s.copied) cudaEventDestroy(s.copied);
    if (s.done) cudaEventDestroy(s.done);
  }
  if (fe->copy_stream) cudaStreamDestroy(fe->copy_stream);
  if (fe->ev_in) cudaEventDestroy(fe->ev_in);
  if (fe->ev_out) cudaEventDestroy(fe->ev_out);
  if (fe->ev_fork) cudaEventDestroy(fe->ev_fork);
  if (fe->ev_join) cudaEventDestroy(fe->ev_join);
  if (fe->remap_stream) cudaStreamDestroy(fe->remap_stream);
  if (fe->ctx->own_stream && fe->ctx->stream) cudaStreamDestroy(fe->ctx->stream);
  if (fe->ctx->arena) cudaFree(fe->ctx->arena);
  delete fe->ctx;
  delete fe;
  return SOS_OK;
}

extern "C" int sos_frontend_reset(sos_frontend* fe) {
  SOS_CHECK_ARG(fe, "fe is NULL");
  SOS_CUDA(cudaMemsetAsync(fe->d.n, 0, sizeof(int32_t) * (fe->cfg.batch + 1), fe->ctx->stream));
  SOS_CUDA(cudaStreamSynchronize(fe->ctx->stream));
  return SOS_OK;
}

extern "C" int sos_frontend_set_graph(sos_frontend* fe, int enabled) {
  SOS_CHECK_ARG(fe, "fe is NULL");
  fe->use_graph = enabled != 0;
  return SOS_OK;
}

namespace {
struct Fence {  // order the front-end's own stream after / before the caller's stream
  sos_frontend* fe;
  explicit Fence(sos_frontend* f) : fe(f) {
    cudaEventRecord(fe->ev_in, fe->parent->stream);
    cudaStreamWaitEvent(fe->ctx->stream, fe->ev_in, 0);
  }
  ~Fence() {
    cudaEventRecord(fe->ev_out, fe->ctx->stream);
    cudaStreamWaitEvent(fe->parent->stream, fe->ev_out, 0);
  }
};
}  // namespace

extern "C" int sos_frontend_set_ref_slots(sos_frontend* fe, const int32_t* ref_slots) {
  SOS_CHECK_ARG(fe && ref_slots, "NULL argument");
  SOS_CHECK_ARG(fe->cfg.keyframe_mode, "reference slots are only used in keyframe mode");
  for (int i = 0; i < fe->cfg.batch; ++i)
    SOS_CHECK_ARG(ref_slots[i] >= -1 && ref_slots[i] <= fe->cfg.batch && ref_slots[i] != i + 1, "reference slot out of range");
  SOS_CUDA(cudaSetDevice(fe->ctx->device));
  Fence fence(fe);
  SOS_CUDA(cudaMemcpyAsync(fe->d.ref_slot, ref_slots, sizeof(int32_t) * fe->cfg.batch, cudaMemcpyHostToDevice, fe->ctx->stream));
  SOS_CUDA(cudaStreamSynchronize(fe->ctx->stream));  // ref_slots may be pageable / reused by the caller
  return SOS_OK;
}

extern "C" int sos_frontend_promote(sos_frontend* fe, int slot) {
  SOS_CHECK_ARG(fe, "fe is NULL");
  SOS_CHECK_ARG(slot >= 1 && slot <= fe->cfg.batch, "slot out of range");
  SOS_CUDA(cudaSetDevice(fe->ctx->device));
  Fence fence(fe);
  const int64_t before = fe->ctx->launches;
  const int rc = enqueue_carry(fe, slot);
  fe->parent->launches += fe->ctx->launches - before;
  return rc;
}

extern "C" int sos_frontend_retrack(sos_frontend* fe) {
  SOS_CHECK_ARG(fe, "fe is NULL");
  SOS_CUDA(cudaSetDevice(fe->ctx->device));
  Fence fence(fe);
  const int64_t before = fe->ctx->launches;
  const int rc = enqueue_stage_b(fe);
  fe->parent->launches += fe->ctx->launches - before;
  return rc;
}

extern "C" int sos_frontend_profile_begin(sos_frontend* fe) {
  SOS_CHECK_ARG(fe, "fe is NULL");
  return sos_ctx_profile_begin(fe->ctx);  // run_step launches eagerly while profiling: events cannot be captured
}

extern "C" int sos_frontend_profile_end(sos_frontend* fe, char* names, size_t names_cap, float* ms, int max_n, int* n_out) {
  SOS_CHECK_ARG(fe, "fe is NULL");
  return sos_ctx_profile_end(fe->ctx, names, names_cap, ms, max_n, n_out);
}

extern "C" int sos_frontend_get_buffers(sos_frontend* fe, sos_frontend_buffers* out) {
  SOS_CHECK_ARG(fe && out, "NULL argument");
  *out = fe->d;
  return SOS_OK;
}

#define SOS_CHECK_SOS(fe) SOS_CHECK_ARG(!(fe)->rgbd, "not available on an RGB-D front-end")
#define SOS_CHECK_RGBD(fe) SOS_CHECK_ARG((fe)->rgbd, "needs an RGB-D front-end (sos_frontend_create_rgbd)")

namespace {
int step_device(sos_frontend* fe, const StepIn& in) {
  SOS_CUDA(cudaSetDevice(fe->ctx->device));
  // inputs were produced on the caller's stream; results must be visible to it afterwards
  SOS_CUDA(cudaEventRecord(fe->ev_in, fe->parent->stream));
  SOS_CUDA(cudaStreamWaitEvent(fe->ctx->stream, fe->ev_in, 0));
  const int64_t before = fe->ctx->launches;
  const int rc = run_step(fe, in);
  fe->parent->launches += fe->ctx->launches - before;
  if (rc) return rc;
  SOS_CUDA(cudaEventRecord(fe->ev_out, fe->ctx->stream));
  SOS_CUDA(cudaStreamWaitEvent(fe->parent->stream, fe->ev_out, 0));
  return SOS_OK;
}
}  // namespace

extern "C" int sos_frontend_step(sos_frontend* fe, const uint8_t* omni, const float* px_top, const uint32_t* desc_top,
                                 const int32_t* bucket_off_top, const float* px_bot, const uint32_t* desc_bot,
                                 const int32_t* bucket_off_bot) {
  SOS_CHECK_ARG(fe, "fe is NULL");
  SOS_CHECK_SOS(fe);
  SOS_CHECK_ARG(omni && px_top && desc_top && bucket_off_top && px_bot && desc_bot && bucket_off_bot, "NULL input");
  return step_device(fe, sos_step_in(omni, px_top, desc_top, bucket_off_top, px_bot, desc_bot, bucket_off_bot, false));
}

extern "C" int sos_frontend_step_rgbd(sos_frontend* fe, const float* depth, const float* px, const uint32_t* desc,
                                      const int32_t* n_kp) {
  SOS_CHECK_ARG(fe, "fe is NULL");
  SOS_CHECK_RGBD(fe);
  SOS_CHECK_ARG(depth && px && desc && n_kp, "NULL input");
  return step_device(fe, rgbd_step_in(depth, px, desc, n_kp));
}

extern "C" int sos_frontend_set_detector(sos_frontend* fe, const sos_detect_config* dcfg, const uint8_t* masks_top,
                                         const uint8_t* masks_bot) {
  SOS_CHECK_ARG(fe && dcfg, "NULL argument");
  SOS_CHECK_SOS(fe);
  SOS_CHECK_ARG(masks_top && masks_bot, "NULL masks");
  const sos_frontend_config& c = fe->cfg;
  if (c.channels != 3 || c.n_buckets > 32) {
    sos_set_error("sos_frontend_set_detector: the feature front needs 3-channel images and at most 32 buckets (channels %d, "
                  "n_buckets %d)", c.channels, c.n_buckets);
    return SOS_ERR_UNSUPPORTED;
  }
  SOS_CHECK_ARG(dcfg->corners_per_bucket >= 1 && dcfg->corners_per_bucket <= c.max_feat_per_bucket,
                "corners_per_bucket must lie in [1, max_feat_per_bucket]");
  SOS_CHECK_ARG(dcfg->median == 0 || dcfg->median == 1, "median must be 0 or 1");
  SOS_CHECK_ARG(dcfg->quality_level > 0.0 && dcfg->min_distance >= 0.0 && dcfg->min_distance < 64.0,
                "bad quality level / minimum distance");
  SOS_CHECK_ARG(c.pano_rows > 62 && c.pano_cols > 62 && (size_t)c.pano_rows * c.pano_cols < (1ull << 31),
                "panorama smaller than ORB's border or too large");
  SOS_CHECK_ARG((long long)c.batch * c.n_buckets <= 65535, "too many (frame, bucket) lists");
  SOS_CHECK_ARG(2ll * c.batch * c.n_buckets * c.max_feat_per_bucket < (1ll << 31), "too many corner slots");
  SOS_CUDA(cudaSetDevice(fe->ctx->device));
  Fence fence(fe);   // the masks may have been written on the caller's stream
  sos_frontend::Detector& dt = fe->det;
  const size_t B = c.batch, nb = c.n_buckets, Nmax = c.max_feat_per_bucket, F = c.max_feat_per_view;
  const size_t plane = (size_t)c.pano_rows * c.pano_cols;
  if (!dt.med) {
    int rc = SOS_OK;
    sos_frontend_features& f = dt.f;
#define DT_ALLOC(ptr, count) \
    if (rc == SOS_OK) rc = fe_alloc(fe, &(ptr), (count))
    DT_ALLOC(dt.med, B * 2 * plane * 3); DT_ALLOC(dt.gray, B * 2 * plane); DT_ALLOC(dt.blur, B * 2 * plane);
    DT_ALLOC(dt.mask_bits[0], plane); DT_ALLOC(dt.mask_bits[1], plane); DT_ALLOC(dt.flags, 2);
    DT_ALLOC(dt.eig, B * plane); DT_ALLOC(dt.max_bits, B * nb); DT_ALLOC(dt.cand, B * nb);
    DT_ALLOC(dt.keys, B * nb * SOS_GFT_CAP); DT_ALLOC(dt.rank, B * plane);
    DT_ALLOC(dt.xy, 2 * B * nb * Nmax * 2); DT_ALLOC(dt.count, 2 * B * nb); DT_ALLOC(dt.kp_image, 2 * B * nb * Nmax);
    DT_ALLOC(dt.kp_desc, 2 * B * nb * Nmax * 8); DT_ALLOC(dt.kp_keep, 2 * B * nb * Nmax);
    DT_ALLOC(f.px_top, B * F * 2); DT_ALLOC(f.desc_top, B * F * 8); DT_ALLOC(f.boff_top, B * (nb + 1));
    DT_ALLOC(f.px_bot, B * F * 2); DT_ALLOC(f.desc_bot, B * F * 8); DT_ALLOC(f.boff_bot, B * (nb + 1));
    DT_ALLOC(f.detect_stats, B * 2 * 4);
#undef DT_ALLOC
    if (rc) return rc;
    // the selection leaves every rank-image entry it sets back at -1, so one clear serves every later step
    SOS_CUDA(cudaMemsetAsync(dt.rank, 0xFF, B * plane * sizeof(int32_t), fe->ctx->stream));
  }
  // corner slot (view, b, k, j) is described on gray plane 2 b + view
  const size_t N = dcfg->corners_per_bucket;
  std::vector<int32_t> img(2 * B * nb * N);
  for (size_t i = 0; i < img.size(); ++i) {
    const size_t vb = i / (nb * N);
    img[i] = (int32_t)(2 * (vb % B) + vb / B);
  }
  SOS_CUDA(cudaMemcpyAsync(dt.kp_image, img.data(), img.size() * sizeof(int32_t), cudaMemcpyHostToDevice, fe->ctx->stream));
  for (int view = 0; view < 2; ++view) {
    const int rc = sos_gft_pack_masks(fe->ctx, view == 0 ? masks_top : masks_bot, c.pano_rows, c.pano_cols, c.n_buckets,
                                      dt.mask_bits[view], dt.flags + view);
    if (rc) return rc;
  }
  SOS_CUDA(cudaMemcpyAsync(dt.overlap, dt.flags, sizeof(dt.overlap), cudaMemcpyDeviceToHost, fe->ctx->stream));
  SOS_CUDA(cudaStreamSynchronize(fe->ctx->stream));
  dt.cfg = *dcfg;
  dt.on = true;
  // captured images-in steps bake the previous detector's parameters in
  for (size_t i = 0; i < fe->graphs.size();) {
    if (fe->graphs[i].key.kind == STEP_IMAGES) {
      cudaGraphExecDestroy(fe->graphs[i].exec);
      fe->graphs.erase(fe->graphs.begin() + i);
    } else {
      ++i;
    }
  }
  return SOS_OK;
}

extern "C" int sos_frontend_step_images(sos_frontend* fe, const uint8_t* omni) {
  SOS_CHECK_ARG(fe && omni, "NULL argument");
  SOS_CHECK_SOS(fe);
  SOS_CHECK_ARG(fe->det.on, "no detector: call sos_frontend_set_detector first");
  return step_device(fe, sos_step_in(omni, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, true));
}

extern "C" int sos_frontend_get_features(sos_frontend* fe, sos_frontend_features* out) {
  SOS_CHECK_ARG(fe && out, "NULL argument");
  SOS_CHECK_SOS(fe);
  SOS_CHECK_ARG(fe->det.on, "no detector: call sos_frontend_set_detector first");
  *out = fe->det.f;
  return SOS_OK;
}

static int ensure_staging(sos_frontend* fe) {
  if (fe->copy_stream) return SOS_OK;
  const sos_frontend_config& c = fe->cfg;
  const size_t B = c.batch, F = c.max_feat_per_view;
  SOS_CUDA(cudaStreamCreateWithFlags(&fe->copy_stream, cudaStreamNonBlocking));
  if (fe->rgbd) {   // whole depth maps, keypoints, descriptors and counts
    const sos_rgbd_frontend_config& r = fe->rgbd_cfg;
    for (auto& s : fe->stage) {
      int rc = fe_alloc(fe, &s.omni, B * r.height * r.width * sizeof(float));
      if (!rc) rc = fe_alloc(fe, &s.px_top, B * r.max_kp * 2);
      if (!rc) rc = fe_alloc(fe, &s.desc_top, B * r.max_kp * 8);
      if (!rc) rc = fe_alloc(fe, &s.n_kp, B);
      if (rc) return rc;
      SOS_CUDA(cudaMallocHost((void**)&s.h_poses, B * 12 * sizeof(float)));
      SOS_CUDA(cudaMallocHost((void**)&s.h_stats, B * 4 * sizeof(int32_t)));
      SOS_CUDA(cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming));
      SOS_CUDA(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
    }
    SOS_CUDA(cudaStreamSynchronize(fe->ctx->stream));
    return SOS_OK;
  }
  for (auto& s : fe->stage) {
    int rc = fe_alloc(fe, &s.omni, B * c.src_h * c.src_w * c.channels);
    if (!rc) rc = fe_alloc(fe, &s.px_top, B * F * 2);
    if (!rc) rc = fe_alloc(fe, &s.px_bot, B * F * 2);
    if (!rc) rc = fe_alloc(fe, &s.desc_top, B * F * 8);
    if (!rc) rc = fe_alloc(fe, &s.desc_bot, B * F * 8);
    if (!rc) rc = fe_alloc(fe, &s.boff_top, B * (c.n_buckets + 1));
    if (!rc) rc = fe_alloc(fe, &s.boff_bot, B * (c.n_buckets + 1));
    if (rc) return rc;
    SOS_CUDA(cudaMallocHost((void**)&s.h_poses, B * 12 * sizeof(float)));
    SOS_CUDA(cudaMallocHost((void**)&s.h_stats, B * 4 * sizeof(int32_t)));
    SOS_CUDA(cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming));
    SOS_CUDA(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
  }
  SOS_CUDA(cudaStreamSynchronize(fe->ctx->stream));
  // which bytes of an omni image can the remap read?  Per source row a bitmap of the 64-byte blocks some LUT entry touches;
  // rows are grouped into bands of 64, and every run of used blocks of a band (runs closer than 1 KB are merged) becomes one
  // strided copy: the two mirror annuli are uploaded, the corners of the frame and the hole in the middle are not.
  fe->bands.clear();
  fe->omni_bytes_per_frame = (int64_t)c.src_h * c.src_w * c.channels;
  const char* full = getenv("SOS_FULL_UPLOAD");   // A/B switch (tests run both): upload whole images
  if (full == nullptr || full[0] == '0') {
    const int pitch = c.src_w * c.channels;
    const int n_blocks = (pitch + 63) / 64, words = (n_blocks + 63) / 64;
    unsigned long long* dblk = nullptr;
    int rc = fe_alloc(fe, &dblk, (size_t)c.src_h * words);
    if (rc) return rc;
    const size_t n = (size_t)2 * c.pano_rows * c.pano_cols;
    lut_row_blocks_kernel<<<(unsigned)((n + 255) / 256), 256, 0, fe->ctx->stream>>>(fe->lut, n, c.src_h, c.src_w, c.channels, words, dblk);
    SOS_CUDA(cudaStreamSynchronize(fe->ctx->stream));
    std::vector<unsigned long long> blk((size_t)c.src_h * words);
    SOS_CUDA(cudaMemcpy(blk.data(), dblk, blk.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    const int band_rows = 64, merge_gap = 16;   // C2 rig: 32 copies, 0.74 of the image (32-row bands: 62 copies, 0.73)
    int64_t total = 0;
    std::vector<sos_frontend::Band> bands;
    std::vector<unsigned long long> acc(words);
    for (int r0 = 0; r0 < c.src_h; r0 += band_rows) {
      const int nr = std::min(band_rows, c.src_h - r0);
      std::fill(acc.begin(), acc.end(), 0ull);
      for (int r = r0; r < r0 + nr; ++r)
        for (int w = 0; w < words; ++w) acc[w] |= blk[(size_t)r * words + w];
      int run_lo = -1, run_hi = -1;   // current run of used blocks [run_lo, run_hi]
      auto flush = [&]() {
        if (run_lo < 0) return;
        const int x0 = run_lo * 64, x1 = std::min(pitch, (run_hi + 1) * 64);
        bands.push_back({r0, nr, x0, x1 - x0});
        total += (int64_t)nr * (x1 - x0);
        run_lo = run_hi = -1;
      };
      for (int b = 0; b < n_blocks; ++b) {
        if (!((acc[b >> 6] >> (b & 63)) & 1ull)) continue;
        if (run_lo >= 0 && b - run_hi > merge_gap) flush();
        if (run_lo < 0) run_lo = b;
        run_hi = b;
      }
      flush();
    }
    if (total < fe->omni_bytes_per_frame * 97 / 100) {   // otherwise one plain copy is cheaper than the band copies
      fe->bands = bands;
      fe->omni_bytes_per_frame = total;
    }
  }
  return SOS_OK;
}

extern "C" int sos_frontend_host_bytes(sos_frontend* fe, int64_t* h2d_bytes_per_step, int64_t* d2h_bytes_per_step) {
  SOS_CHECK_ARG(fe, "fe is NULL");
  SOS_CUDA(cudaSetDevice(fe->ctx->device));
  const int rc = ensure_staging(fe);
  if (rc) return rc;
  const sos_frontend_config& c = fe->cfg;
  const int64_t B = c.batch, F = c.max_feat_per_view;
  if (h2d_bytes_per_step && fe->rgbd) {
    const sos_rgbd_frontend_config& r = fe->rgbd_cfg;
    *h2d_bytes_per_step = B * ((int64_t)r.height * r.width * 4 + (int64_t)r.max_kp * (2 * 4 + 32) + 4);
  } else if (h2d_bytes_per_step) {
    *h2d_bytes_per_step = B * (fe->omni_bytes_per_frame + 2 * F * 2 * 4 + 2 * F * 32 + 2 * (c.n_buckets + 1) * 4);
  }
  if (d2h_bytes_per_step) *d2h_bytes_per_step = B * (12 * 4 + 4 * 4);
  return SOS_OK;
}

namespace {
// H2D of one step's inputs on the copy stream (so that it overlaps the kernels of the previous step), the step, and the
// D2H of poses and stats.  in: HOST pointers; images-in step: only the omni images are uploaded and the features are
// detected on the device; RGB-D step: whole depth maps, then keypoints, descriptors and counts.
int submit(sos_frontend* fe, const StepIn& in, int* ticket) {
  SOS_CUDA(cudaSetDevice(fe->ctx->device));
  int rc = ensure_staging(fe);
  if (rc) return rc;
  const int k = fe->next_stage;
  sos_frontend::Stage& s = fe->stage[k];
  if (s.in_flight) {
    sos_set_error("sos_frontend_submit_host: both staging slots are in flight; call sos_frontend_wait_host first");
    return SOS_ERR_INVALID;
  }
  const sos_frontend_config& c = fe->cfg;
  const size_t B = c.batch, F = c.max_feat_per_view;
  cudaStream_t cs = fe->copy_stream;
  const bool images = in.kind == STEP_IMAGES;
  const uint8_t* omni = (const uint8_t*)in.p[0];
  const float *px_top = (const float*)in.p[1], *px_bot = (const float*)in.p[4];
  const uint32_t *desc_top = (const uint32_t*)in.p[2], *desc_bot = (const uint32_t*)in.p[5];
  const int32_t *bucket_off_top = (const int32_t*)in.p[3], *bucket_off_bot = (const int32_t*)in.p[6];
  StepIn dev;
  if (in.kind == STEP_RGBD) {
    const sos_rgbd_frontend_config& r = fe->rgbd_cfg;
    SOS_CUDA(cudaMemcpyAsync(s.omni, in.p[0], B * r.height * r.width * sizeof(float), cudaMemcpyHostToDevice, cs));
    SOS_CUDA(cudaMemcpyAsync(s.px_top, in.p[1], B * r.max_kp * 2 * sizeof(float), cudaMemcpyHostToDevice, cs));
    SOS_CUDA(cudaMemcpyAsync(s.desc_top, in.p[2], B * r.max_kp * 32, cudaMemcpyHostToDevice, cs));
    SOS_CUDA(cudaMemcpyAsync(s.n_kp, in.p[3], B * sizeof(int32_t), cudaMemcpyHostToDevice, cs));
    dev = rgbd_step_in((const float*)s.omni, s.px_top, s.desc_top, s.n_kp);
  } else if (fe->bands.empty()) {
    SOS_CUDA(cudaMemcpyAsync(s.omni, omni, B * c.src_h * c.src_w * c.channels, cudaMemcpyHostToDevice, cs));
  } else {
    // one strided copy per band of rows, covering that band in every frame of the batch (depth = frames)
    const size_t pitch = (size_t)c.src_w * c.channels;
    for (const auto& bd : fe->bands) {
      cudaMemcpy3DParms p = {};
      p.srcPtr = make_cudaPitchedPtr((void*)omni, pitch, pitch, c.src_h);
      p.dstPtr = make_cudaPitchedPtr((void*)s.omni, pitch, pitch, c.src_h);
      p.srcPos = make_cudaPos(bd.x0_bytes, bd.row0, 0);
      p.dstPos = make_cudaPos(bd.x0_bytes, bd.row0, 0);
      p.extent = make_cudaExtent(bd.width_bytes, bd.nrows, B);
      p.kind = cudaMemcpyHostToDevice;
      SOS_CUDA(cudaMemcpy3DAsync(&p, cs));
    }
  }
  if (in.kind == STEP_FEATURES) {
    SOS_CUDA(cudaMemcpyAsync(s.px_top, px_top, B * F * 2 * sizeof(float), cudaMemcpyHostToDevice, cs));
    SOS_CUDA(cudaMemcpyAsync(s.px_bot, px_bot, B * F * 2 * sizeof(float), cudaMemcpyHostToDevice, cs));
    SOS_CUDA(cudaMemcpyAsync(s.desc_top, desc_top, B * F * 32, cudaMemcpyHostToDevice, cs));
    SOS_CUDA(cudaMemcpyAsync(s.desc_bot, desc_bot, B * F * 32, cudaMemcpyHostToDevice, cs));
    SOS_CUDA(cudaMemcpyAsync(s.boff_top, bucket_off_top, B * (c.n_buckets + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, cs));
    SOS_CUDA(cudaMemcpyAsync(s.boff_bot, bucket_off_bot, B * (c.n_buckets + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, cs));
  }
  if (in.kind != STEP_RGBD) dev = sos_step_in(s.omni, s.px_top, s.desc_top, s.boff_top, s.px_bot, s.desc_bot, s.boff_bot, images);
  SOS_CUDA(cudaEventRecord(s.copied, cs));
  SOS_CUDA(cudaStreamWaitEvent(fe->ctx->stream, s.copied, 0));
  const int64_t before = fe->ctx->launches;
  rc = run_step(fe, dev);
  fe->parent->launches += fe->ctx->launches - before;
  if (rc) return rc;
  SOS_CUDA(cudaMemcpyAsync(s.h_poses, fe->d.pose, B * 12 * sizeof(float), cudaMemcpyDeviceToHost, fe->ctx->stream));
  SOS_CUDA(cudaMemcpyAsync(s.h_stats, fe->d.stats, B * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, fe->ctx->stream));
  SOS_CUDA(cudaEventRecord(s.done, fe->ctx->stream));
  // slot reuse is safe: sos_frontend_wait_host(ticket) must return before this slot is submitted to again
  s.in_flight = true;
  *ticket = k;
  fe->next_stage = (k + 1) % sos_frontend::DEPTH;
  return SOS_OK;
}
}  // namespace

extern "C" int sos_frontend_submit_host(sos_frontend* fe, const uint8_t* omni, const float* px_top,
                                        const uint32_t* desc_top, const int32_t* bucket_off_top, const float* px_bot,
                                        const uint32_t* desc_bot, const int32_t* bucket_off_bot, int* ticket) {
  SOS_CHECK_ARG(fe && ticket, "NULL argument");
  SOS_CHECK_SOS(fe);
  SOS_CHECK_ARG(omni && px_top && desc_top && bucket_off_top && px_bot && desc_bot && bucket_off_bot, "NULL input");
  return submit(fe, sos_step_in(omni, px_top, desc_top, bucket_off_top, px_bot, desc_bot, bucket_off_bot, false), ticket);
}

extern "C" int sos_frontend_submit_host_rgbd(sos_frontend* fe, const float* depth, const float* px, const uint32_t* desc,
                                             const int32_t* n_kp, int* ticket) {
  SOS_CHECK_ARG(fe && ticket, "NULL argument");
  SOS_CHECK_RGBD(fe);
  SOS_CHECK_ARG(depth && px && desc && n_kp, "NULL input");
  for (int b = 0; b < fe->cfg.batch; ++b) SOS_CHECK_ARG(n_kp[b] >= 0 && n_kp[b] <= fe->rgbd_cfg.max_kp, "n_kp outside [0, max_kp]");
  return submit(fe, rgbd_step_in(depth, px, desc, n_kp), ticket);
}

extern "C" int sos_frontend_submit_host_images(sos_frontend* fe, const uint8_t* omni, int* ticket) {
  SOS_CHECK_ARG(fe && ticket && omni, "NULL argument");
  SOS_CHECK_SOS(fe);
  SOS_CHECK_ARG(fe->det.on, "no detector: call sos_frontend_set_detector first");
  return submit(fe, sos_step_in(omni, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, true), ticket);
}

extern "C" int sos_frontend_wait_host(sos_frontend* fe, int ticket, float* poses, int32_t* stats) {
  SOS_CHECK_ARG(fe, "fe is NULL");
  SOS_CHECK_ARG(ticket >= 0 && ticket < sos_frontend::DEPTH && fe->stage[ticket].in_flight, "unknown ticket");
  sos_frontend::Stage& s = fe->stage[ticket];
  SOS_CUDA(cudaEventSynchronize(s.done));
  const size_t B = fe->cfg.batch;
  if (poses) memcpy(poses, s.h_poses, B * 12 * sizeof(float));
  if (stats) memcpy(stats, s.h_stats, B * 4 * sizeof(int32_t));
  s.in_flight = false;
  return SOS_OK;
}

extern "C" int sos_frontend_step_host(sos_frontend* fe, const uint8_t* omni, const float* px_top, const uint32_t* desc_top,
                                      const int32_t* bucket_off_top, const float* px_bot, const uint32_t* desc_bot,
                                      const int32_t* bucket_off_bot, float* poses, int32_t* stats) {
  int ticket = -1;
  int rc = sos_frontend_submit_host(fe, omni, px_top, desc_top, bucket_off_top, px_bot, desc_bot, bucket_off_bot, &ticket);
  if (rc) return rc;
  return sos_frontend_wait_host(fe, ticket, poses, stats);
}
