/*
 * sosfront.h — C-ABI of libsosfront.so, the B200 (sm_100a) SOS visual-odometry front-end.
 *
 * This is the drop-in boundary for the per-frame hot path of ubuntuslave/vo_single_camera_sos.
 * The reference is pure Python and has no FFI of its own; every entry point below replaces one
 * call the reference makes into NumPy / OpenCV / OpenGV on that path.  The "replaces:" line of
 * each function cites the reference call site (paths relative to the reference root).
 *
 * Conventions
 *   - every function returns an int status: SOS_OK (0) or a negative SOS_ERR_* code; the message
 *     of the last failure on the calling thread is returned by sos_last_error().  Nothing throws,
 *     nothing calls exit().
 *   - all array arguments are plain pointers to C-contiguous (row-major) memory.  Unless a
 *     function name ends in _host, array pointers are DEVICE pointers and the call is asynchronous
 *     on the context's stream.  *_host functions take HOST pointers, stage through the context's
 *     device buffers (H2D, kernels, D2H) and return after the results are in host memory.
 *   - scalar / small struct parameters (sizes, thresholds, GUM parameter vectors, foci) are always
 *     passed by value or as HOST pointers.
 *   - the caller owns every input and output buffer.  Scratch memory lives in the context and only
 *     grows (sos_ctx_reserve pre-sizes it, which is required before CUDA-graph capture).
 *   - a sos_ctx is bound to one device and one stream and must be used by one thread at a time
 *     (the reference calls arrive on its VO thread, pose_est_tools.py:1725-1727).
 */
#ifndef SOSFRONT_H_
#define SOSFRONT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SOS_OK 0
#define SOS_ERR_INVALID (-1)     /* bad argument */
#define SOS_ERR_CUDA (-2)        /* CUDA runtime / launch failure */
#define SOS_ERR_NOMEM (-3)       /* allocation failure */
#define SOS_ERR_UNSUPPORTED (-4) /* valid request this build cannot serve */
#define SOS_ERR_CAPTURE (-5)     /* would have to allocate while the stream is being captured */

#define SOS_ABI_VERSION 1

typedef struct sos_ctx sos_ctx;

/* ------------------------------------------------------------------------------------------------
 * Context, stream and memory plumbing
 * ---------------------------------------------------------------------------------------------- */
int sos_abi_version(void);
const char* sos_last_error(void);
int sos_device_count(int* count);
int sos_ctx_create(int device, sos_ctx** out);
int sos_ctx_destroy(sos_ctx* ctx);
/* Borrow an externally owned cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream) instead of the stream the
 * context created for itself; NULL selects the legacy default stream. */
int sos_ctx_set_stream(sos_ctx* ctx, void* cuda_stream);
void* sos_ctx_get_stream(sos_ctx* ctx);
int sos_ctx_sync(sos_ctx* ctx);
/* Make sure the context scratch arena holds at least `bytes`. */
int sos_ctx_reserve(sos_ctx* ctx, size_t bytes);
/* Number of kernel launches issued through this context since creation (for bench.py's gpu_launches). */
int64_t sos_ctx_launch_count(sos_ctx* ctx);
/* Per-launch device timing for bench.py's roofline numbers: between begin and end every kernel launched through the
 * context is followed by a CUDA event on the context's stream.  end() synchronises and returns, for launch k, the
 * elapsed time since the previous launch's event in ms[k] and the launching entry point's name (one per line) in names. */
int sos_ctx_profile_begin(sos_ctx* ctx);
int sos_ctx_profile_end(sos_ctx* ctx, char* names, size_t names_cap, float* ms, int max_n, int* n_out);

int sos_malloc(sos_ctx* ctx, size_t bytes, void** dptr);
int sos_free(sos_ctx* ctx, void* dptr);
int sos_malloc_host(size_t bytes, void** hptr); /* pinned */
int sos_free_host(void* hptr);
int sos_memcpy_h2d(sos_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes); /* async on ctx stream */
int sos_memcpy_d2h(sos_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes); /* async on ctx stream */
int sos_memset(sos_ctx* ctx, void* dst_dev, int value, size_t bytes);

/* ------------------------------------------------------------------------------------------------
 * Step 1 — panoramic remap (SURVEY §8a F1, F2, F3)
 * ---------------------------------------------------------------------------------------------- */

/* Packed fixed-point LUT entry (one uint64 per panorama pixel), the device form of what
 * cv2.convertMaps(CV_16SC2) produces (panorama.py:482) plus the folded mirror mask:
 *   bits  0..15  x0  (int16)  = sat_s16(cvRound(32*map_x) >> 5)
 *   bits 16..31  y0  (int16)  = sat_s16(cvRound(32*map_y) >> 5)
 *   bits 32..36  ax  = cvRound(32*map_x) & 31        bits 37..41  ay = cvRound(32*map_y) & 31
 *   bits 48..51  tap i lies inside the source image  (i = 0:(y0,x0) 1:(y0,x0+1) 2:(y0+1,x0) 3:(y0+1,x0+1))
 *   bits 52..55  tap i is inside AND its mask byte is non-zero (mask == NULL: same as inside)
 *   bit  56      all four taps usable and the 16 bytes from tap 2 of a 3-channel frame lie inside it: gates the
 *                fast taps of remap3b_kernel (aligned 32-bit window loads)
 * NaN / |32*x| >= 2^31 map to INT_MIN exactly as cvtps2dq does inside cv::remap. */
typedef uint64_t sos_lut_entry;

/* replaces: the per-frame float64->float32 cast + the float->fixed conversion inside cv2.remap
 * (panorama.py:291-298) and the mirror mask of get_fully_masked_images (camera_models.py:2932-3010).
 * map_x/map_y: [rows*cols]; mask: [src_h*src_w] uint8 or NULL; lut: [rows*cols]. */
int sos_lut_pack_f32(sos_ctx* ctx, const float* map_x, const float* map_y, int rows, int cols,
                     const uint8_t* mask, int src_h, int src_w, sos_lut_entry* lut);
int sos_lut_pack_f64(sos_ctx* ctx, const double* map_x, const double* map_y, int rows, int cols,
                     const uint8_t* mask, int src_h, int src_w, sos_lut_entry* lut);

/* replaces: cv2.remap(src, map_x32, map_y32, INTER_LINEAR, dst, BORDER_CONSTANT, border) in
 * Panorama.get_panoramic_image (panorama.py:293-298), for `views` LUTs at once (top and bottom
 * mirror, camera_models.py:3119-3120), with `dst = mask ? src : background` of
 * get_fully_masked_images applied at tap fetch.  Bit-exact with cv2.remap (Q5 coords, Q15 weights).
 *   src  [batch, src_h, src_w, channels] uint8      lut [views, rows, cols]
 *   dst  [batch, views, rows, cols, channels] uint8  border/background: HOST pointers to `channels` bytes
 * channels in {1,3,4}. */
int sos_remap_u8(sos_ctx* ctx, const uint8_t* src, int batch, int src_h, int src_w, int channels,
                 const sos_lut_entry* lut, int views, int rows, int cols, const uint8_t* border,
                 const uint8_t* background, uint8_t* dst);

/* GUM parameter vector (HOST doubles), gum.py:48-140 Parameters + gum.py:361-383 set_model_params. */
enum {
  SOS_GUM_XI1 = 0, SOS_GUM_XI2, SOS_GUM_XI3, /* Cp_wrt_M */
  SOS_GUM_K1, SOS_GUM_K2, SOS_GUM_K3,        /* forward radial distortion */
  SOS_GUM_GAMMA1, SOS_GUM_GAMMA2, SOS_GUM_ALPHA_C, SOS_GUM_U0, SOS_GUM_V0,
  SOS_GUM_L1, SOS_GUM_L2, SOS_GUM_L3,        /* inverse radial model (gum.py:2689-2694) */
  SOS_GUM_P1, SOS_GUM_P2,                    /* tangential terms of the Heikkila inverse (gum.py:2713-2725) */
  SOS_GUM_PLANE_K,                           /* z of the normalised projection plane wrt [M] (gum.py:379-382) */
  SOS_GUM_USE_DISTORTION,                    /* 0/1 */
  SOS_GUM_NPARAMS
};

/* replaces: GUM.get_pixel_from_3D_point_wrt_M (gum.py:2512-2551): points wrt [M] -> pixels.
 * pts [n,3] float64 -> uv [n,2] float64. */
int sos_gum_project(sos_ctx* ctx, const double* gum, const double* pts, int n, double* uv);

/* replaces: Panorama._generate_LUTs (panorama.py:414-492): forward-project the cylinder grid.
 * psi(c) = reversed linspace(0,2pi,cols,endpoint=False) and theta(r) = atan2(linspace(h_max,h_min,rows,
 * endpoint=False), 1) are rounded to float32 as the reference does (panorama.py:431,441); rows whose
 * theta lies outside [elev_lo, elev_hi] get NaN.  map_x/map_y: [rows*cols] float64. */
int sos_lut_build(sos_ctx* ctx, const double* gum, int rows, int cols, double cyl_height_max,
                  double cyl_height_min, double elev_lo, double elev_hi, double* map_x, double* map_y);

/* ------------------------------------------------------------------------------------------------
 * Step 2 — brute-force Hamming matching of 256-bit descriptors (SURVEY §8a F4, F5, F6)
 * ---------------------------------------------------------------------------------------------- */

/* replaces: cv2.BFMatcher(NORM_HAMMING).match / .knnMatch(k=2) (camera_models.py:402,421,442), for n_seg
 * independent (query, train) segment pairs in one launch (azimuthal buckets camera_models.py:3038, views, frames).
 *   q, t [*, 8] uint32 (row = one 32-byte ORB descriptor), 16-byte aligned
 *   segment s compares query rows [q_start[s], q_start[s]+q_len[s]) with train rows [t_start[s], t_start[s]+t_len[s]);
 *   q_start, q_len, t_start, t_len [n_seg] int32 live on the DEVICE (lengths may be produced by earlier kernels);
 *   max_nq / max_nt: HOST upper bounds of any q_len / t_len (they size the grid; longer segments are truncated)
 *   idx0, idx1 [*] int32, indexed like q: best / second-best train row RELATIVE to t_start[s] (-1: none)
 *   d0, d1     [*] int32: their Hamming distances (-1: none)
 * Order is (distance, train index): ties go to the lowest train index, as OpenCV does.
 * idx1/d1 may be NULL (1-NN only). */
int sos_hamming_top2(sos_ctx* ctx, const uint32_t* q, const uint32_t* t, const int32_t* q_start,
                     const int32_t* q_len, const int32_t* t_start, const int32_t* t_len, int n_seg, int max_nq,
                     int max_nt, int32_t* idx0, int32_t* d0, int32_t* idx1, int32_t* d1);

/* replaces: cv2.BFMatcher(NORM_HAMMING).radiusMatch(queryDescriptors, trainDescriptors, maxDistance), the
 * use_radius_match branch of FeatureMatcher.match (camera_models.py:409-412): every train row t with
 * hamming(q, t) <= max_distance, per query in train-index order.  Two passes over the same arguments:
 *   pass 1: count int32 [nq] receives the number of rows per query (offset, out_t, out_d NULL);
 *   pass 2: offset int64 [nq] (exclusive prefix sum of count) says where query r writes its out_t / out_d entries. */
int sos_hamming_radius(sos_ctx* ctx, const uint32_t* q, int nq, const uint32_t* t, int nt, int max_distance,
                       int32_t* count, const int64_t* offset, int32_t* out_t, int32_t* out_d);

/* replaces: cv2.BFMatcher() (NORM_L2) .match / .knnMatch(k = 2) on float descriptors — the SIFT / SURF branch of
 * FeatureMatcher (camera_models.py:397-399, 417-442).  The optional float-descriptor variant of the matcher, a real GEMM:
 * |q - t|^2 = |q|^2 + |t|^2 - 2 <q, t> on the tensor cores (tcgen05.mma kind::f16, bfloat16 operands, float32
 * accumulators in tensor memory).  EXACT for descriptors whose values are integers in [0, 255] — what cv2's SIFT
 * returns — because those are exact in bfloat16 and every partial sum stays below 2^24: distances equal cv2's
 * sqrt(float32 sum of squared differences) bit for bit, ties go to the lowest train row.  Other values are refused:
 * not_integer_flag[0] (DEVICE int32) is set non-zero and the outputs are meaningless.
 *   q, t [*, dim] float32 rows, dim <= 128; segments as in sos_hamming_top2
 *   idx0, idx1 int32 (train row relative to t_start[s], -1: none); d0, d1 float32 L2 distances (-1: none);
 *   idx1 / d1 may be NULL. */
int sos_l2_top2(sos_ctx* ctx, const float* q, const float* t, int dim, const int32_t* q_start, const int32_t* q_len,
                const int32_t* t_start, const int32_t* t_len, int n_seg, int max_nq, int max_nt, int32_t* idx0,
                float* d0, int32_t* idx1, float* d1, int32_t* not_integer_flag);

/* replaces: cv2.BFMatcher() (NORM_L2) .match / .knnMatch(k = 2) on ANY finite float descriptors (SURF, KAZE, RootSIFT, ...) —
 * the SIFT / SURF branch of FeatureMatcher (camera_models.py:397-399, 417-442) when the values are not integers in [0, 255].
 * Results are those of a float64 reference with a fixed evaluation order, bit for bit:
 *   d^2(q, t) = sum_k (double(q_k) - double(t_k))^2, summed for k = 0 .. dim-1 in order, without fused multiply-add;
 *   the two smallest d^2 per query, ties to the lowest train row; distance = float32(sqrt(d^2)) rounded from double.
 * On integer-valued inputs this equals cv2 (and sos_l2_top2).  On other inputs cv2's float32 SIMD sum is build-dependent;
 * its distances may differ from these by an ulp.
 * The tensor cores rank the candidates (each value split into two bfloat16 pieces, float32 accumulators); a query whose
 * nearest rows are closer together than a derived error band, or whose magnitudes could leave the float32 range, is
 * re-decided by a float64 brute force over its segment, so the result never depends on the band.
 *   q, t [*, dim] float32 rows, 1 <= dim <= 128; segments, idx0 / idx1 / d0 / d1 as in sos_l2_top2 (idx1 / d1 may be NULL)
 *   nonfinite_flag: DEVICE int32 [1], set non-zero when a value is NaN or +-Inf (the outputs are then meaningless)
 *   stats (may be NULL): DEVICE int32 [SOS_L2F_STATS], zeroed by the call, indices SOS_L2F_STAT_*. */
#define SOS_L2F_STATS 2
#define SOS_L2F_STAT_REDECIDED 0   /* queries re-decided by the float64 brute force */
#define SOS_L2F_STAT_BAND_PPM 1    /* largest |approximate - float64 d^2| / band over the winners decided from the GEMM, ppm */
int sos_l2f_top2(sos_ctx* ctx, const float* q, const float* t, int dim, const int32_t* q_start, const int32_t* q_len,
                 const int32_t* t_start, const int32_t* t_len, int n_seg, int max_nq, int max_nt, int32_t* idx0,
                 float* d0, int32_t* idx1, float* d1, int32_t* nonfinite_flag, int32_t* stats);

#define SOS_MATCH_NN 0    /* 1-NN, the reference default (k_best = 1, pose_est_tools.py:686) */
#define SOS_MATCH_RATIO 1 /* keep m0 iff d0 < ratio * d1 (camera_models.py:421-436) */
#define SOS_MATCH_CROSS 2 /* mutual nearest neighbours (BFMatcher crossCheck, camera_models.py:401) */

/* replaces: the tail of FeatureMatcher.match — sorted(matches, key=distance) (camera_models.py:444) —
 * followed by filter_pixel_correspondences (common_cv.py:167-188) as applied by
 * match_features_panoramic_top_bottom (camera_models.py:3086) and match_features_frame_to_frame
 * (pose_est_tools.py:245-247).  Per segment: select by `mode`, order stably by (distance, query index),
 * then keep pairs with |u_t - u_q| <= max_du (if max_du > 0) and v_t - v_q >= min_dv (if min_dv >= 0),
 * evaluated in float64 on the float32 pixel coordinates.
 *   rev_idx0: best query row (relative to q_start[s]) per train row, indexed like t (SOS_MATCH_CROSS only, else NULL)
 *   px_q, px_t [*,2] float32 (u,v), indexed like q / t, or NULL when no gate is requested
 *   out_q, out_t, out_d: segment s writes its pairs to rows q_start[s] + k, k < out_count[s]; out_q / out_t hold
 *   ABSOLUTE rows (q_start[s] + query, t_start[s] + train);  out_count [n_seg]: pairs kept per segment. */
int sos_match_select(sos_ctx* ctx, int mode, double ratio, const int32_t* idx0, const int32_t* d0,
                     const int32_t* d1, const int32_t* rev_idx0, const int32_t* q_start,
                     const int32_t* q_len, const int32_t* t_start, int n_seg, const float* px_q,
                     const float* px_t, double max_du, double min_dv, int32_t* out_q,
                     int32_t* out_t, int32_t* out_d, int32_t* out_count);

/* replaces: filter_pixel_correspondences (common_cv.py:167-188) as a stand-alone call on n already paired points:
 * valid[i] = (max_du <= 0 || |top[i].u - bot[i].u| <= max_du) && (min_dv < 0 || top[i].v - bot[i].v >= min_dv).
 * pts_top, pts_bot [n,2] float64 (the reference hands it float64 coordinates); valid [n] uint8. */
int sos_pixel_gate(sos_ctx* ctx, const double* pts_top, const double* pts_bot, int n, double max_du, double min_dv,
                   uint8_t* valid);

/* ------------------------------------------------------------------------------------------------
 * Steps 3+4 — lifting and midpoint triangulation (SURVEY §8a F7-F11), RGB-D back-projection (F12)
 * ---------------------------------------------------------------------------------------------- */

/* Panorama geometry (HOST doubles): cols, rows, pixel_size, cyl_height_max, cyl_circumference, cyl_radius */
enum { SOS_PANO_COLS = 0, SOS_PANO_ROWS, SOS_PANO_PIXEL_SIZE, SOS_PANO_HEIGHT_MAX, SOS_PANO_CIRCUMFERENCE,
       SOS_PANO_RADIUS, SOS_PANO_NPARAMS };

/* replaces: Panorama.get_direction_angles_from_pixel_pano(use_LUTs=False) (panorama.py:616-666) +
 * GUM.get_3D_point_from_angles_wrt_focus (gum.py:2564 -> camera_models.py:1031-1065).
 * uv [n,2] float32 -> az, el [n] float32, bearing [n,3] float32 (NaN outside the panorama). Any output may be NULL. */
int sos_lift_pano(sos_ctx* ctx, const double* pano, const float* uv, int n, float* az, float* el, float* bearing);
/* Same with float64 in and out (the reference's dtype; used by the per-call Python mirror). */
int sos_lift_pano_f64(sos_ctx* ctx, const double* pano, const double* uv, int n, double* az, double* el, double* bearing);

/* replaces: GUM.lift_pixel_to_unit_sphere_wrt_focus (gum.py:2673-2940, new_method branch) and
 * OmniCamModel.get_direction_angles_from_pixel (camera_models.py:1183-1194).
 * uv [n,2] float64 omni-image pixels -> sphere [n,3] float64, az/el [n] float64 (may be NULL). */
int sos_lift_gum(sos_ctx* ctx, const double* gum, const double* uv, int n, double* sphere, double* az, double* el);

/* replaces: OmniStereoModel.get_triangulated_point_from_direction_angles(use_midpoint_triangulation=True)
 * (camera_models.py:3323-3364 -> 2420-2490) + filter_panoramic_points_due_to_range (camera_models.py:3299-3321).
 * az/el of the top (1) and bottom (2) rays [n] float32; f1, f2: HOST foci [3] in frame [C].
 * xyz [n,3] float32; valid [n] uint8 (may be NULL) = (rmin <= norm <= rmax), rmin/rmax <= 0 disabling that bound.
 * homogeneous_norm != 0 reproduces the reference's frame code, which hands the N x 4 HOMOGENEOUS array to the range
 * filter (pose_est_tools.py:365-372) so that norm = sqrt(x^2 + y^2 + z^2 + 1). */
int sos_triangulate_midpoint(sos_ctx* ctx, const float* az1, const float* el1, const float* az2,
                             const float* el2, int n, const double* f1, const double* f2, double rmin,
                             double rmax, int homogeneous_norm, float* xyz, uint8_t* valid);
/* replaces: OmniCamModel.map_angles_to_unit_sphere (camera_models.py:1031-1065) as a stand-alone call: az, el [n]
 * float64 -> sphere [n,3] float64, NaN-propagating. */
int sos_angles_to_sphere_f64(sos_ctx* ctx, const double* az, const double* el, int n, double* sphere);
/* replaces: filter_panoramic_points_due_to_range (camera_models.py:3299-3321) as a stand-alone call: xyz [n,3] float64. */
int sos_range_gate_f64(sos_ctx* ctx, const double* xyz, int n, double rmin, double rmax, int homogeneous_norm,
                       uint8_t* valid);
int sos_triangulate_midpoint_f64(sos_ctx* ctx, const double* az1, const double* el1, const double* az2,
                                 const double* el2, int n, const double* f1, const double* f2, double rmin,
                                 double rmax, int homogeneous_norm, double* xyz, uint8_t* valid);

/* Fused steps 3+4 over matched pairs, driven by DEVICE-side counts (no host sync), as
 * StereoPanoramicFrame.establish_stereo_correspondences does after matching (pose_est_tools.py:344-397).
 * Frame f owns segments [f*segs_per_frame, (f+1)*segs_per_frame) (its azimuthal buckets, in order).  For segment s
 * and k < pair_count[s], pair (q,t) = (pair_q[seg_off[s]+k], pair_t[seg_off[s]+k]) with q a bottom-view feature
 * row and t a top-view feature row (both GLOBAL rows into px_bot / px_top [*,2] float32): lift both pixels (F7,F8),
 * triangulate (F10), range-gate (F11) and append the survivors, in order, to the compacted per-frame
 * correspondence store (T1, camera_models.py:291-362), rows [f*cap_per_frame, f*cap_per_frame + out_n[f]):
 *   out_uv_top/out_uv_bot [*,2], out_b_top/out_b_bot [*,3] (unit bearings), out_xyz [*,3] float32,
 *   out_src_top/out_src_bot [*] int32 (feature rows, for descriptor gathers), out_n [n_frames] int32. */
int sos_stereo_lift_triangulate(sos_ctx* ctx, const double* pano_top, const double* pano_bot, const float* px_top,
                                const float* px_bot, const int32_t* pair_q, const int32_t* pair_t,
                                const int32_t* pair_count, const int32_t* seg_off, int n_frames, int segs_per_frame,
                                int max_pairs_per_seg /* HOST bound of any pair_count */, int pair_rows /* rows of pair_q */,
                                const double* f1, const double* f2, double rmin, double rmax, int homogeneous_norm,
                                int cap_per_frame, float* out_uv_top, float* out_uv_bot, float* out_b_top,
                                float* out_b_bot, float* out_xyz, int32_t* out_src_top, int32_t* out_src_bot,
                                int32_t* out_n);

/* RGB-D intrinsics (HOST doubles): fx, fy, cx, cy, focal_length_m, depth_is_Z(0/1) — camera_models.py:752-779 */
enum { SOS_RGBD_FX = 0, SOS_RGBD_FY, SOS_RGBD_CX, SOS_RGBD_CY, SOS_RGBD_FOCAL_M, SOS_RGBD_DEPTH_IS_Z, SOS_RGBD_NPARAMS };

/* replaces: RGBDCamModel.get_depth_Z over the whole map (camera_models.py:781-799). depth/z [h,w] float32. */
int sos_rgbd_depth_to_z(sos_ctx* ctx, const double* cam, const float* depth, int batch, int h, int w, float* z);

/* replaces: RGBDCamModel.get_XYZ at keypoints (camera_models.py:835-860), get_normalized_points
 * (camera_models.py:203-212) and the NaN / Z-range gate of RGBDFrame.establish_keypoints
 * (pose_est_tools.py:612-620).  depth [batch,h,w] float32; u,v [batch,n] int32 pixel indices;
 * xyz, bearing [batch,n,3] float32 (NaN where depth == 0); valid [batch,n] uint8 = !NaN && zmin <= Z <= zmax. */
int sos_rgbd_backproject(sos_ctx* ctx, const double* cam, const float* depth, int batch, int h, int w,
                         const int32_t* u, const int32_t* v, int n, double zmin, double zmax, float* xyz,
                         float* bearing, uint8_t* valid);

/* ------------------------------------------------------------------------------------------------
 * Step 5 — batched RANSAC for rigid 3D-3D registration (SURVEY §8a R1, R2)
 * ---------------------------------------------------------------------------------------------- */

#define SOS_SOLVER_ARUN 0
#define SOS_SOLVER_P3P 1
#define SOS_SCORE_EUCLID 0  /* |p_ref - (R p_cur + t)| < thr */
#define SOS_SCORE_BEARING 1 /* 1 - f . normalize(Rc^T (R^T (p_ref - t) - tc)) < thr  (pose_est_tools.py:150-203, 181-185) */

/* replaces: transformations.superimposition_matrix(v0, v1, scale=False, usesvd=True)
 * (transformations.py:982-1030 -> 874-980) for n_sets independent point sets of k points each.
 * v0, v1 [n_sets, k, 3] float64 -> M [n_sets, 12] float64 (row-major 3x4 [R|t], v1 ~ R v0 + t);
 * with_scale != 0 adds Umeyama's uniform scale (scale=True, transformations.py:971-975): v1 ~ s R v0 + t, M = [sR|t];
 * ok [n_sets] uint8 = 0 for degenerate (rank < 2) sets. */
int sos_arun_batch(sos_ctx* ctx, const double* v0, const double* v1, int n_sets, int k, int with_scale, double* M,
                   uint8_t* ok);

/* One RANSAC problem per `problem` (frame pair).  The correspondences of problem b are rows
 * [b*cap, b*cap + n[b]) of the arrays below, n DEVICE int32 [n_problems].
 *   p_ref [*,3] float32  3D points in the reference frame (pose_est_tools.py:753-756)
 *   p_cur [*,3] float32  3D points of the same landmarks in the current frame (Arun hypotheses; EUCLID score)
 *   f_cur [*,3] float32  unit bearings in the current frame (BEARING score; may be NULL for EUCLID)
 *   cam   [*]   uint8    camera index of each bearing (0 top, 1 bottom; NULL = central)
 *   rig   HOST doubles [n_cams*12]: per camera row-major 3x4 [Rc|tc] (pose_est_tools.py:852-859), NULL = identity
 * Hypotheses: hyp [n_hyp,3] uint32 DEVICE, shared by all problems; sample j of hypothesis h is row
 * floor(hyp[h][j] * n / 2^32) (size-independent, so the oracle draws the same triples); a hypothesis with a
 * repeated row or a degenerate (collinear) triple scores -1.  Best = highest inlier count, lowest h on ties
 * (OpenGV's strict '>' update).
 * Outputs: best_pose [n_problems,12] float32 (row-major [R|t] of the current frame wrt the reference frame,
 * p_ref ~ R p_cur + t, what pyopengv.absolute_pose_*_ransac returns, pose_est_tools.py:785,915),
 * best_hyp, best_count [n_problems] int32, inlier_mask [n_problems*cap] uint8,
 * best_key [n_problems] uint64 = (count+1) << 32 | (0xFFFFFFFF - (hyp_offset + h)) for cross-GPU max-reduce
 * (may be NULL), all_counts [n_problems, n_hyp] int32 (may be NULL): every hypothesis' inlier count, negative for a
 * rejected sample.
 * Scoring runs in float32 (bfloat16-split GEMMs on the tensor cores; SOS_SCORE_ENGINE=fma selects the FP32-pipe kernel)
 * with a rounding-error guard band; pairs inside the band are re-decided in float64 with
 * the reference's formula, so counts and inlier sets equal the float64 result. */
int sos_ransac_p3d(sos_ctx* ctx, const float* p_ref, const float* p_cur, const float* f_cur, const uint8_t* cam,
                   const int32_t* n, int n_problems, int cap, const double* rig, int n_cams, const uint32_t* hyp,
                   int n_hyp, int hyp_offset, int score_mode, double threshold, float* best_pose,
                   int32_t* best_hyp, int32_t* best_count, uint8_t* inlier_mask, uint64_t* best_key,
                   int32_t* all_counts);

/* Diagnostics of the score engines, two optional outputs (at least one must be given).
 * sn (may be NULL): sos_ransac_p3d forced onto the tensor-core engine (csrc/score_mma.cuh), which additionally stores what the
 * tensor cores accumulated for every (hypothesis, correspondence) pair: sn [n_problems, n_hyp, ceil(cap/128)*128, 2] float32.
 * SOS_SCORE_BEARING: (s, N') with s = f . x and N' = |x|^2 + 1.52 max_cam |b|^2, x = Rc^T (R^T (p - t) - tc)
 * (pose_est_tools.py:150-203, 181-185); SOS_SCORE_EUCLID: (s', n2) with s' = |q|^2 - 2 q . x and n2 = |x|^2, q = p_cur, so
 * that s' + n2 = |x - q|^2.  The parity tests bound their error against float64 with it.  With sn NULL the engine is the one
 * sos_ransac_p3d picks (SOS_SCORE_ENGINE).
 * stats (may be NULL): DEVICE int32 [SOS_SCORE_STATS], zeroed by the call, then filled with how much work went through the
 * deferred float64 path of the engine that ran (indices SOS_STAT_*; the other engine's entries stay 0).  Tensor-core engine,
 * per work item (problem x 128 hypotheses x a range of correspondence tiles): 32-pair chunks with uncertain pairs, queued in
 * shared memory up to 1536 per item and decided by the scoring thread itself past that; pairs expanded from the queue, in
 * rounds of at most 2048.  FP32-pipe kernel, per block: (32-correspondence batch, hypothesis) entries with an uncertain pair,
 * queued up to 2048 per block; a block past that re-decides its whole range in float64.
 * Counts equal those of sos_ransac_p3d on the same engine. */
#define SOS_SCORE_STATS 8
#define SOS_STAT_TC_ITEMS 0              /* tensor-core work items that ran */
#define SOS_STAT_TC_CHUNKS 1             /* chunks with uncertain pairs, summed over items */
#define SOS_STAT_TC_CHUNKS_MAX 2         /* largest number of such chunks in one item */
#define SOS_STAT_TC_CHUNKS_IN_THREAD 3   /* chunks past the 1536 queue entries of their item, decided in-thread */
#define SOS_STAT_TC_PAIRS 4              /* pairs expanded from the queues and re-decided, summed */
#define SOS_STAT_TC_ROUNDS_MAX 5         /* largest number of expansion rounds (<= 2048 pairs each) in one item */
#define SOS_STAT_FMA_ENTRIES 6           /* FP32 kernel: queue entries, summed over blocks, overflowing ones included */
#define SOS_STAT_FMA_OVERFLOW_BLOCKS 7   /* FP32 kernel: blocks whose queue overflowed */
int sos_ransac_score_probe(sos_ctx* ctx, const float* p_ref, const float* p_cur, const float* f_cur, const uint8_t* cam,
                           const int32_t* n, int n_problems, int cap, const double* rig, int n_cams, const uint32_t* hyp,
                           int n_hyp, int score_mode, double threshold, float* best_pose, int32_t* best_hyp,
                           int32_t* best_count, int32_t* all_counts, float* sn, int32_t* stats);

/* replaces: pyopengv.absolute_pose_noncentral_ransac(bearings, cam_idx, points, cam_offsets, cam_rotations, thr, iters)
 * (pose_est_tools.py:785) and pyopengv.absolute_pose_ransac(bearings, points, algo, thr, iters) (pose_est_tools.py:915)
 * WITH THE ARGUMENTS THE REFERENCE PASSES: bearings of the current frame and 3D points of the reference frame only.
 * Same layout, scoring (bearing residual), first-maximum rule and outputs as sos_ransac_p3d, but
 *   hyp [n_hyp,4] uint32: rows 0-2 are the minimal sample, row 3 picks among its solutions (OpenGV's sample size for its
 *   three-point solvers); a hypothesis with a repeated row, a collinear triple or no solution scores negative.
 * Minimal solver: depths along the three rays with |X_i - X_j| = |P_i - P_j| — Grunert's three-point problem for a common
 * origin (quartic, closed form), then Newton on the three distance equations with each ray's own origin for a non-central
 * rig (rig / cam as in sos_ransac_p3d; NULL = central) — and the pose of the two congruent triangles.  It solves the problem
 * OpenGV's KNEIP / GP3P solvers solve, not by OpenGV's code (absent from the reference tree): parity with OpenGV unpinned. */
int sos_ransac_p3p(sos_ctx* ctx, const float* p_ref, const float* f_cur, const uint8_t* cam, const int32_t* n,
                   int n_problems, int cap, const double* rig, int n_cams, const uint32_t* hyp, int n_hyp,
                   int hyp_offset, double threshold, float* best_pose, int32_t* best_hyp, int32_t* best_count,
                   uint8_t* inlier_mask, uint64_t* best_key, int32_t* all_counts);

/* Re-derive pose and inlier mask of hypothesis `hyp_index[b]` (DEVICE int32, GLOBAL index, i.e. the winner
 * of the cross-GPU reduce, SURVEY §8e) without scoring the others. */
int sos_ransac_p3d_eval(sos_ctx* ctx, const float* p_ref, const float* p_cur, const float* f_cur, const uint8_t* cam,
                        const int32_t* n, int n_problems, int cap, const double* rig, int n_cams,
                        const uint32_t* hyp_row /* [n_problems,3] uint32: the winning triples */, int score_mode,
                        double threshold, float* pose, int32_t* count, uint8_t* inlier_mask);

/* Arun refit on the inlier set (stands in for pyopengv.*_optimize_nonlinear, pose_est_tools.py:830,937; an
 * approximation — see DESIGN.md).  pose [n_problems,12] float32. */
int sos_refit_inliers(sos_ctx* ctx, const float* p_ref, const float* p_cur, const uint8_t* inlier_mask,
                      const int32_t* n, int n_problems, int cap, float* pose, int32_t* n_used);

/* ------------------------------------------------------------------------------------------------
 * Feature description on the panoramas (SURVEY §8f N3, description half)
 * ---------------------------------------------------------------------------------------------- */

/* replaces: cv2.medianBlur(pano_img, 11) (camera_models.py:1708-1709 with median_win_size = 11, pose_est_tools.py:297):
 * exact per-channel median of the 11 x 11 window, BORDER_REPLICATE.  src, dst uint8 [n_images, height, width, channels],
 * channels 1 or 3, not in place.  Bit-exact. */
int sos_median_blur_11(sos_ctx* ctx, const uint8_t* src, int n_images, int height, int width, int channels, uint8_t* dst);

/* replaces: the pair cv2.medianBlur(pano_img, 11) + cv2.cvtColor(pano_img, cv2.COLOR_BGR2GRAY) (camera_models.py:1708-1711)
 * in one pass: src uint8 [n_images, height, width, 3] -> gray [n_images, height, width]; dst_bgr (the blurred colour image,
 * same shape as src) may be NULL when only the gray image is consumed.  Bit-exact with the two OpenCV calls. */
int sos_median_blur_11_gray(sos_ctx* ctx, const uint8_t* src, int n_images, int height, int width, uint8_t* dst_bgr,
                            uint8_t* gray);

/* replaces: cv2.cvtColor(pano_img, cv2.COLOR_BGR2GRAY) (camera_models.py:1711).  Bit-exact with OpenCV 4.x (15-bit fixed point). */
int sos_bgr_to_gray(sos_ctx* ctx, const uint8_t* bgr, size_t n_pixels, uint8_t* gray);

/* The blur inside cv2.ORB.compute: separable 7-tap Gaussian of sigma 2, BORDER_REFLECT_101, exact arithmetic rounded
 * once (not cv2.GaussianBlur's fixed-point path; identified and pinned by scripts/derive_orb_pattern.py).
 * gray, blurred: uint8 [n_images, height, width]; not in place. */
int sos_orb_blur(sos_ctx* ctx, const uint8_t* gray, int n_images, int height, int width, uint8_t* blurred);

/* replaces: cv2.ORB_create(nfeatures).compute(image = gray panorama, keypoints) (camera_models.py:1683, 1766) for
 * keypoints of octave 0 (what cv2.KeyPoint_convert and single-scale detectors produce).  Bit-exact with OpenCV 4.13.
 *   kp_xy        float32 [n, 2] pixel coordinates          kp_angle_deg float32 [n] or NULL (= -1, KeyPoint_convert's angle)
 *   kp_image     int32 [n] image index or NULL (= 0)       desc uint32 [n, 8] (256 bits, OpenCV byte order)
 *   keep         uint8 [n] (nullable): 0 where OpenCV drops the keypoint (closer than 31 px to the border; desc = 0) */
int sos_orb_describe(sos_ctx* ctx, const uint8_t* gray, int n_images, int height, int width, const float* kp_xy,
                     const float* kp_angle_deg, const int32_t* kp_image, int n, uint32_t* desc, uint8_t* keep);

/* replaces: cv2.cornerMinEigenVal(gray, blockSize = 3, ksize = 3) — the corner measure inside goodFeaturesToTrack.
 * gray uint8 [n_images, height, width] -> eig float32 [n_images, height, width].  Same float32 arithmetic as OpenCV 4.13
 * (written out at the top of csrc/gft.cu; the Sobel rows are smoothed in cv2's tap order).  Bit-equal to cv2 except in
 * its SIMD tail columns (the last <= 16 of a row) and, on sharp images, at a few pixels where cv2's sliding-window box
 * sums round differently (at most half a unit in the last place of the image's largest measure). */
int sos_corner_min_eigenval(sos_ctx* ctx, const uint8_t* gray, int n_images, int height, int width, float* eig);

/* replaces: cv2.goodFeaturesToTrack(image = gray, maxCorners, qualityLevel, minDistance, mask = masks[m],
 * useHarrisDetector = False) for every (image, mask) pair (camera_models.py:1737, one call per azimuthal mask).
 *   masks     uint8 [n_masks, height, width], shared by all images; NULL with n_masks = 1 = no mask
 *   out_xy    float32 [n_images, n_masks, max_corners, 2] corner (x, y), strongest first
 *   out_count int32 [n_images, n_masks]
 *   eig_out   float32 [n_images, height, width] (nullable) receives the corner measure
 * max_corners must be >= 1 (cv2's maxCorners <= 0, "no limit", has no fixed output size).  More than 16384 local maxima
 * above the quality threshold in one (image, mask) cannot be ranked reproducibly: the call then fails with
 * SOS_ERR_INVALID, whatever the number of masks.  The call reads the candidate counts back, so it returns only after the
 * candidate stage has run on ctx's stream. */
int sos_gft_detect(sos_ctx* ctx, const uint8_t* gray, const uint8_t* masks, int n_images, int height, int width,
                   int n_masks, int max_corners, double quality_level, double min_distance, float* out_xy,
                   int32_t* out_count, float* eig_out);

/* Dense triangulation of panoramic disparity maps into point clouds (SURVEY §8f N4).
 * replaces: OmniStereoModel.resolve_pano_correspondences_from_disparity_map (camera_models.py:2492-2538) + the lifting and
 *           midpoint triangulation of triangulate_from_depth_map (camera_models.py:2567-2685, own midpoint method).
 * disparity float32 [n_maps, rows, cols] is linked to the TOP panorama: pixel (u, v) matches (u, v - d) in the bottom
 * panorama.  A pixel is valid iff roi_col0 <= u < roi_col1 (negative = whole width), d != 0, min_disparity <= d <=
 * max_disparity (0 = the ROI-masked map's maximum) and v - d <= lowest_reference_row.
 * xyz float32 [n_maps, rows, cols, 3] wrt [C] (NaN where invalid); valid uint8 [n_maps, rows, cols] (nullable). */
int sos_dense_triangulate(sos_ctx* ctx, const double* pano_top, const double* pano_bot, const float* disparity,
                          int n_maps, int rows, int cols, double min_disparity, double max_disparity,
                          double lowest_reference_row, int roi_col0, int roi_col1, const double* f1,
                          const double* f2, float* xyz, uint8_t* valid);

/* Non-linear pose refinement on the inlier set (SURVEY §8f N1).
 * replaces: pyopengv.absolute_pose_noncentral_optimize_nonlinear (pose_est_tools.py:830) and
 *           pyopengv.absolute_pose_optimize_nonlinear (pose_est_tools.py:937; n_cams = 0 -> central camera).
 * Levenberg-Marquardt in float64 on sum_i r_i^2, r_i = 1 - f_i . normalize(Rc^T (R^T (p_i - t) - tc)) — OpenGV's
 * published residual, the same one the bearing score uses (pose_est_tools.py:150-203) — starting from pose_in.
 * One thread-block cluster per problem (cluster_size CTAs, 0 = choose from cap, at most 8).
 * inlier_mask NULL = use all n[b] rows.  pose_out float32 [n_problems,12] and/or pose_out64 float64 [n_problems,12]
 * (either may be NULL, not both); stats (nullable) float64 [n_problems,4] = initial cost, final cost, cost
 * evaluations, rows used.  Fewer than 6 usable rows -> pose_in is passed through. */
int sos_refine_pose(sos_ctx* ctx, const float* p_ref, const float* f_cur, const uint8_t* cam,
                    const uint8_t* inlier_mask, const int32_t* n, int n_problems, int cap, const double* rig,
                    int n_cams, const float* pose_in, int max_iters, int cluster_size, float* pose_out,
                    double* pose_out64, double* stats);

/* ------------------------------------------------------------------------------------------------
 * The batched, GPU-resident front-end: B new frames in, B frame-pair poses out (SURVEY §8a T1, §8e)
 * ---------------------------------------------------------------------------------------------- */

/* One step chains the five hot-path steps for a batch of frames exactly as
 * StereoPanoramicFrame.establish_stereo_correspondences (pose_est_tools.py:320-402) and
 * TrackerStereoSE3.track_frame (pose_est_tools.py:736-847) do for one frame; defaults in pose_est_tools.py:284-308,
 * 672-707, 862-878.  Feature detection is upstream of the hot path (SURVEY §2 row 5): features arrive as input. */
/* sos_frontend_config.refit */
enum {
  SOS_REFINE_NONE = 0, /* pose = RANSAC model */
  SOS_REFINE_ARUN = 1, /* Arun refit on the inliers (sos_refit_inliers) */
  SOS_REFINE_LM = 2    /* Levenberg-Marquardt on the bearing residual (sos_refine_pose), as the reference does with OpenGV */
};

typedef struct sos_frontend_config {
  int32_t batch;               /* frames per step; pair i = (frame i-1, frame i), frame -1 = last frame of the previous step */
  int32_t src_h, src_w, channels;
  int32_t pano_rows, pano_cols;
  int32_t n_buckets;           /* azimuthal buckets per view (12, pose_est_tools.py:871) */
  int32_t max_feat_per_view;   /* rows reserved per frame and view in the feature arrays */
  int32_t max_feat_per_bucket; /* upper bound of any bucket's feature count */
  int32_t cap;                 /* capacity of triangulated stereo correspondences per frame */
  int32_t n_hyp;               /* RANSAC hypotheses (210 in the reference, pose_est_tools.py:709-720) */
  int32_t score_mode;          /* SOS_SCORE_* */
  int32_t homogeneous_norm;    /* 1 = range gate on the homogeneous norm as the reference does (pose_est_tools.py:365-372) */
  int32_t refit;               /* SOS_REFINE_*: what turns the RANSAC pose into the output pose */
  int32_t refine_iters;        /* SOS_REFINE_LM: maximum cost evaluations (0 = 20) */
  int32_t keyframe_mode;       /* 0: pair i = (slot i, slot i+1), the last frame is carried over automatically (throughput mode);
                                  1: pair i = (slot ref_slot[i], slot i+1) and slot 0 only changes through sos_frontend_promote —
                                     the reference's keyframe tracking (pose_est_tools.py:1489, 1553-1566), SURVEY §8f N2 */
  int32_t solver;              /* SOS_SOLVER_ARUN: 3D-3D hypotheses, hyp [n_hyp,3] (sos_ransac_p3d);
                                  SOS_SOLVER_P3P: bearing-only hypotheses, hyp [n_hyp,4], bearing score (sos_ransac_p3p) */
  double ransac_threshold;     /* 1 - cos(5 deg) for SOS_SCORE_BEARING (pose_est_tools.py:675-676) */
  double stereo_max_du, stereo_min_dv; /* 2.5, 1 (pose_est_tools.py:298-304) */
  double temporal_max_du;      /* 0.125 * 0.5 * cols (pose_est_tools.py:866) */
  double min_range, max_range; /* 0.5 m, 7 m in model units (pose_est_tools.py:306-308) */
  double pano_top[SOS_PANO_NPARAMS], pano_bot[SOS_PANO_NPARAMS];
  double f_top[3], f_bot[3];   /* mirror foci in [C] */
  double rig[24];              /* 2 x row-major 3x4 [Rc|tc] (pose_est_tools.py:852-859) */
  uint8_t border[4], background[4];
} sos_frontend_config;

/* Device buffers of the front-end, exposed for parity tests and for consumers that keep working on the device.
 * "store" arrays hold batch+1 slots of `cap` rows: slot 0 = carried reference frame, slot i+1 = frame i of the step. */
typedef struct sos_frontend_buffers {
  uint8_t* pano;                                   /* [batch, 2, rows, cols, ch] */
  int32_t *st_q_start, *st_q_len, *st_t_start, *st_t_len; /* stereo segments [batch*n_buckets] */
  int32_t *st_idx0, *st_d0;                        /* [batch*max_feat] indexed like the bottom-view features */
  int32_t *st_pair_q, *st_pair_t, *st_pair_d, *st_pair_count;
  float *uv_c, *uv_top, *uv_bot;                   /* store [2][slots*cap][2]; uv_top / uv_bot alias its halves */
  float *b_top, *b_bot, *xyz;                      /* store [slots*cap][3] */
  int32_t *src_top, *src_bot, *n;                  /* store [slots*cap], n [slots] */
  uint32_t* desc_c;                                /* store [2][slots*cap][8] */
  int32_t *tm_q_start, *tm_q_len, *tm_t_start, *tm_t_len; /* temporal segments [2*batch]: view-major */
  int32_t *tm_idx0, *tm_d0, *tm_pair_q, *tm_pair_t, *tm_pair_d, *tm_pair_count;
  float *p_ref, *p_cur, *f_cur;                    /* [batch, 2*cap, 3] */
  uint8_t* cam;                                    /* [batch, 2*cap] */
  int32_t *n_corr, *n_corr_top;                    /* [batch] */
  float *ransac_pose, *pose;                       /* [batch, 12]; pose = refit (or a copy of ransac_pose) */
  int32_t *best_hyp, *best_count, *n_refit;        /* [batch] */
  uint8_t* inlier_mask;                            /* [batch, 2*cap] */
  int32_t* stats;                                  /* [batch, 4]: n_stereo, n_correspondences, n_inliers, best_hyp */
  double* refine_stats;                            /* [batch, 4] of sos_refine_pose (SOS_REFINE_LM only) */
  int32_t* ref_slot;                               /* [batch] reference slot of pair i (keyframe_mode only) */
  int32_t* overflow;                               /* [batch] feature rows of frame i the capacity clamps dropped in the
                                                      last step (bucket > max_feat_per_bucket, offsets > max_feat_per_view);
                                                      0 everywhere unless the configuration is too small for the input */
  int32_t batch, cap, launches_per_step;
} sos_frontend_buffers;

typedef struct sos_frontend sos_frontend;

/* lut [2, pano_rows, pano_cols] (top, bottom) and hyp [n_hyp, 3] are DEVICE arrays that must outlive the front-end.
 * The front-end computes on a private stream; every call (step, submit_host, set_ref_slots, promote, retrack) is fenced
 * with events against the stream the context holds AT THAT CALL (sos_ctx_set_stream), so callers see plain stream order. */
int sos_frontend_create(sos_ctx* ctx, const sos_frontend_config* cfg, const sos_lut_entry* lut, const uint32_t* hyp,
                        sos_frontend** out);
int sos_frontend_destroy(sos_frontend* fe);
int sos_frontend_reset(sos_frontend* fe);                /* forget the carried reference frame */
int sos_frontend_set_graph(sos_frontend* fe, int enabled); /* CUDA-graph replay (default) or eager launches */

/* Keyframe mode (sos_frontend_config.keyframe_mode = 1), the device side of the reference's VO loop
 * (pose_est_tools.py:1481-1566): a step tracks every frame of the batch against a reference slot, normally the current
 * keyframe in slot 0; when the host's keyframe policy promotes frame j, the frames after j are re-tracked against it
 * without repeating remap / stereo matching / triangulation.
 *   set_ref_slots: HOST int32 [batch]; ref_slots[i] in [0, batch] is the store slot pair i tracks against (slot i+1 is
 *                  the frame itself and not allowed), -1 switches pair i off.  Initially all 0.
 *   promote:       copy store slot `slot` (1..batch) into slot 0.
 *   retrack:       re-run temporal matching + RANSAC + refinement of the current store with the current ref_slots. */
int sos_frontend_set_ref_slots(sos_frontend* fe, const int32_t* ref_slots);
int sos_frontend_promote(sos_frontend* fe, int slot);
int sos_frontend_retrack(sos_frontend* fe);
int sos_frontend_get_buffers(sos_frontend* fe, sos_frontend_buffers* out);
/* Same as sos_ctx_profile_begin/_end for the front-end's own launches (steps run eagerly while profiling). */
int sos_frontend_profile_begin(sos_frontend* fe);
int sos_frontend_profile_end(sos_frontend* fe, char* names, size_t names_cap, float* ms, int max_n, int* n_out);

/* One step on DEVICE-resident inputs (asynchronous):
 *   omni [batch, src_h, src_w, channels] uint8
 *   px_top, px_bot [batch, max_feat_per_view, 2] float32 panorama pixel coordinates of the features of each view
 *   desc_top, desc_bot [batch, max_feat_per_view, 8] uint32
 *   bucket_off_top, bucket_off_bot [batch, n_buckets+1] int32: bucket k of frame b holds feature rows
 *   [off[b][k], off[b][k+1]) of that frame. */
int sos_frontend_step(sos_frontend* fe, const uint8_t* omni, const float* px_top, const uint32_t* desc_top,
                      const int32_t* bucket_off_top, const float* px_bot, const uint32_t* desc_bot,
                      const int32_t* bucket_off_bot);

/* The same step on HOST buffers (pinned for full copy bandwidth): H2D on a copy stream, kernels, D2H of
 * poses [batch,12] float32 and stats [batch,4] int32.  submit/wait overlap the copies of step k+1 with the kernels of
 * step k (two staging slots); step_host = submit + wait. */
int sos_frontend_submit_host(sos_frontend* fe, const uint8_t* omni, const float* px_top, const uint32_t* desc_top,
                             const int32_t* bucket_off_top, const float* px_bot, const uint32_t* desc_bot,
                             const int32_t* bucket_off_bot, int* ticket);
int sos_frontend_wait_host(sos_frontend* fe, int ticket, float* poses, int32_t* stats);
/* Bytes one submit/wait pair moves over PCIe.  Of every omni image only the bytes some LUT entry can read (both tap rows
 * of every live panorama pixel plus the slack of the vector loads) are uploaded, as one strided copy per band of 64 rows
 * covering all frames of the batch; the rest of the staging image is never read by the remap. */
int sos_frontend_host_bytes(sos_frontend* fe, int64_t* h2d_bytes_per_step, int64_t* d2h_bytes_per_step);
int sos_frontend_step_host(sos_frontend* fe, const uint8_t* omni, const float* px_top, const uint32_t* desc_top,
                           const int32_t* bucket_off_top, const float* px_bot, const uint32_t* desc_bot,
                           const int32_t* bucket_off_bot, float* poses, int32_t* stats);

/* ------------------------------------------------------------------------------------------------
 * Roofline denominators measured in-process (integer POPC pipe, FP32 FMA pipe) — bench.py only.
 * ---------------------------------------------------------------------------------------------- */
int sos_peak_popc(sos_ctx* ctx, double* tera_popc_per_s);
int sos_peak_ffma(sos_ctx* ctx, double* tflops);
int sos_peak_dfma(sos_ctx* ctx, double* tflops); /* float64 FMA pipe (dense triangulation, LM refinement) */
int sos_peak_ffma2(sos_ctx* ctx, double* tflops); /* packed fma.rn.f32x2 (the form the RANSAC score kernel issues) */
int sos_peak_tmem_read(sos_ctx* ctx, double* tera_bytes_per_s); /* tcgen05.ld bandwidth: epilogue bound of the tensor-core
                                                                    Hamming engine */

#ifdef __cplusplus
}
#endif
#endif /* SOSFRONT_H_ */
