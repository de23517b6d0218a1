// Steps 3+4 of the SOS front-end: pixel -> direction angles -> unit-sphere bearings -> midpoint triangulation,
// the GUM forward projection / panorama LUT generation, and the RGB-D back-projection used by demo_vo_rgbd.py.
//
// All of these are elementwise and bandwidth / latency bound (53 B per stereo correspondence, SURVEY §8d), so the
// arithmetic is done in float64 registers at no measurable cost on B200 while inputs and outputs stay float32
// where the hot path stores them (pixel coordinates are float32 cv2.KeyPoint.pt values, so nothing is lost on input).
#include <math_constants.h>

#include "rgbd.cuh"
#include "sos_common.cuh"

namespace {

struct GumP {
  double v[SOS_GUM_NPARAMS];
};
struct PanoP {
  double v[SOS_PANO_NPARAMS];
};
struct Vec3 {
  double x, y, z;
};

// ---- F7: panorama pixel -> (azimuth, elevation), panorama.py:616-642 ---------------------------------------
__device__ __forceinline__ void pano_pixel_to_angles(const PanoP& p, double u, double v, double& az, double& el) {
  const double cols = p.v[SOS_PANO_COLS], rows = p.v[SOS_PANO_ROWS], ps = p.v[SOS_PANO_PIXEL_SIZE];
  az = (0.0 <= u && u < cols) ? p.v[SOS_PANO_CIRCUMFERENCE] - ps * u : CUDART_NAN;              // panorama.py:638
  el = (0.0 <= v && v < rows) ? atan2(p.v[SOS_PANO_HEIGHT_MAX] - ps * v, p.v[SOS_PANO_RADIUS]) : CUDART_NAN;  // :619
}

// ---- F8: angles -> unit sphere, camera_models.py:1031-1065 ----------------------------------------------------
__device__ __forceinline__ Vec3 angles_to_sphere(double az, double el) {
  double se, ce, sa, ca;
  sincos(el, &se, &ce);
  sincos(az, &sa, &ca);
  return {ce * ca, ce * sa, se};
}

// ---- F10: midpoint of the common perpendicular, camera_models.py:2420-2490, 3323-3364 -------------------------
__device__ __forceinline__ Vec3 triangulate_midpoint(double az1, double el1, double az2, double el2, Vec3 f1, Vec3 f2) {
  // rays on the unit cylinder (camera_models.py:3333-3340): v = (cos az, sin az, tan el)
  double s1, c1, s2, c2;
  sincos(az1, &s1, &c1);
  sincos(az2, &s2, &c2);
  const Vec3 v1 = {c1, s1, tan(el1)}, v2 = {c2, s2, tan(el2)};
  Vec3 n = {v1.y * v2.z - v1.z * v2.y, v1.z * v2.x - v1.x * v2.z, v1.x * v2.y - v1.y * v2.x};
  const double mag = sqrt(n.x * n.x + n.y * n.y + n.z * n.z);
  n.x /= mag; n.y /= mag; n.z /= mag;
  // solve [v1 | -v2 | n] (l1, l2, lp)^T = f2 - f1 by Cramer's rule (np.linalg.solve at camera_models.py:2483)
  const Vec3 b = {f2.x - f1.x, f2.y - f1.y, f2.z - f1.z};
  const Vec3 a = v1, c = n;
  const Vec3 m = {-v2.x, -v2.y, -v2.z};
  auto det3 = [](Vec3 p, Vec3 q, Vec3 r) {
    return p.x * (q.y * r.z - q.z * r.y) - q.x * (p.y * r.z - p.z * r.y) + r.x * (p.y * q.z - p.z * q.y);
  };
  const double D = det3(a, m, c);
  const double l1 = det3(b, m, c) / D;
  const double lp = det3(a, m, b) / D;
  const Vec3 g1 = {f1.x + l1 * v1.x, f1.y + l1 * v1.y, f1.z + l1 * v1.z};
  return {g1.x + 0.5 * lp * n.x, g1.y + 0.5 * lp * n.y, g1.z + 0.5 * lp * n.z};
}

// ---- F11: range gate, camera_models.py:3299-3321 ---------------------------------------------------------------
// The reference passes the HOMOGENEOUS N x 4 array (pose_est_tools.py:365-372), so its norm is sqrt(x^2+y^2+z^2+1);
// `homo` selects that behaviour.
__device__ __forceinline__ bool range_ok(Vec3 p, double rmin, double rmax, int homo) {
  const double nrm = sqrt(p.x * p.x + p.y * p.y + p.z * p.z + (homo ? 1.0 : 0.0));
  bool ok = true;
  if (rmin > 0.0) ok = ok && (nrm >= rmin);
  if (rmax > 0.0) ok = ok && (nrm <= rmax);
  if (rmin > 0.0 || rmax > 0.0) return ok;
  return true;
}

// T = float: the storage type of the batched hot path; T = double: the reference's own dtype, used by the per-call
// Python mirror (omnistereo.panorama / camera_models) so that chained calls lose nothing between kernels.
template <typename T>
__global__ void lift_pano_kernel(PanoP p, const T* __restrict__ uv, int n, T* __restrict__ az_out,
                                 T* __restrict__ el_out, T* __restrict__ bearing) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double az, el;
  pano_pixel_to_angles(p, (double)uv[2 * i], (double)uv[2 * i + 1], az, el);
  if (az_out) az_out[i] = (T)az;
  if (el_out) el_out[i] = (T)el;
  if (bearing) {
    const Vec3 s = angles_to_sphere(az, el);
    bearing[3 * i + 0] = (T)s.x;
    bearing[3 * i + 1] = (T)s.y;
    bearing[3 * i + 2] = (T)s.z;
  }
}

template <typename T>
__global__ void triangulate_kernel(const T* __restrict__ az1, const T* __restrict__ el1,
                                   const T* __restrict__ az2, const T* __restrict__ el2, int n, Vec3 f1, Vec3 f2,
                                   double rmin, double rmax, int homo, T* __restrict__ xyz,
                                   uint8_t* __restrict__ valid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Vec3 P = triangulate_midpoint((double)az1[i], (double)el1[i], (double)az2[i], (double)el2[i], f1, f2);
  xyz[3 * i + 0] = (T)P.x;
  xyz[3 * i + 1] = (T)P.y;
  xyz[3 * i + 2] = (T)P.z;
  if (valid) valid[i] = range_ok(P, rmin, rmax, homo) ? 1 : 0;
}

// ---- fused steps 3+4 with ordered compaction -------------------------------------------------------------------
// Two kernels: (A) one thread per matched pair does the float64 geometry (fully parallel over all frames and buckets)
// and parks bearings / xyz / keep flag in scratch; (B) one block per frame walks its segments in order and appends the
// survivors to the frame's store (block-wide ballot scan), which is pure data movement.
struct StereoArgs {
  PanoP pano_top, pano_bot;
  const float2 *px_top, *px_bot;
  const int32_t *pair_q, *pair_t, *pair_count, *seg_off;
  int segs_per_frame;
  Vec3 f1, f2;
  double rmin, rmax;
  int homo;
  int cap;
  float* tmp;        // [pair_rows, 9]: b_top, b_bot, xyz
  uint8_t* tmp_keep; // [pair_rows]
  int32_t* seg_keep; // [n_segments]: survivors per segment (zeroed before the geometry kernel)
  float2 *out_uv_top, *out_uv_bot;
  float *out_b_top, *out_b_bot, *out_xyz;
  int32_t *out_src_top, *out_src_bot, *out_n;
};

__global__ void __launch_bounds__(256) stereo_geometry_kernel(StereoArgs a) {
  const int s = blockIdx.y;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= a.pair_count[s]) return;
  const int row = a.seg_off[s] + k;
  const int rq = a.pair_q[row];  // bottom-view feature row (query, camera_models.py:3042)
  const int rt = a.pair_t[row];  // top-view feature row (train)
  const float2 mt = a.px_top[rt], mb = a.px_bot[rq];
  double az1, el1, az2, el2;
  pano_pixel_to_angles(a.pano_top, (double)mt.x, (double)mt.y, az1, el1);
  pano_pixel_to_angles(a.pano_bot, (double)mb.x, (double)mb.y, az2, el2);
  const Vec3 bt = angles_to_sphere(az1, el1), bb = angles_to_sphere(az2, el2);
  const Vec3 P = triangulate_midpoint(az1, el1, az2, el2, a.f1, a.f2);
  float* t = a.tmp + (size_t)row * 9;
  t[0] = (float)bt.x; t[1] = (float)bt.y; t[2] = (float)bt.z;
  t[3] = (float)bb.x; t[4] = (float)bb.y; t[5] = (float)bb.z;
  t[6] = (float)P.x; t[7] = (float)P.y; t[8] = (float)P.z;
  const bool keep = range_ok(P, a.rmin, a.rmax, a.homo);
  a.tmp_keep[row] = keep ? 1 : 0;
  const unsigned vote = __ballot_sync(__activemask(), keep);
  if (keep && (threadIdx.x & 31) == (__ffs(vote) - 1)) atomicAdd(&a.seg_keep[s], __popc(vote));
}

constexpr int ST_THREADS = 1024;

// One block per SEGMENT: its survivors start after those of the earlier segments of the same frame.
__global__ void __launch_bounds__(ST_THREADS) stereo_compact_kernel(StereoArgs a) {
  __shared__ int warp_sums[ST_THREADS / 32];
  const int s = blockIdx.x;
  const int frame = s / a.segs_per_frame;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int base = 0;
  for (int e = frame * a.segs_per_frame; e < s; ++e) base += a.seg_keep[e];
  if (s == (frame + 1) * a.segs_per_frame - 1 && tid == 0) a.out_n[frame] = min(base + a.seg_keep[s], a.cap);
  const int off = a.seg_off[s];
  const int cnt = a.pair_count[s];
  for (int k0 = 0; k0 < cnt; k0 += ST_THREADS) {
    const int k = k0 + tid;
    const bool keep = (k < cnt) && a.tmp_keep[off + k] != 0;
    const unsigned vote = __ballot_sync(0xFFFFFFFFu, keep);
    if (lane == 0) warp_sums[warp] = __popc(vote);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < ST_THREADS / 32; ++w) {
      const int c = warp_sums[w];
      if (w < warp) before += c;
      total += c;
    }
    if (keep) {
      const int pos = base + before + __popc(vote & ((1u << lane) - 1u));
      if (pos < a.cap) {
        const size_t o = (size_t)frame * a.cap + pos;
        const int row = off + k;
        const int rq = a.pair_q[row], rt = a.pair_t[row];
        const float* t = a.tmp + (size_t)row * 9;
        a.out_uv_top[o] = a.px_top[rt];
        a.out_uv_bot[o] = a.px_bot[rq];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          a.out_b_top[3 * o + c] = t[c];
          a.out_b_bot[3 * o + c] = t[3 + c];
          a.out_xyz[3 * o + c] = t[6 + c];
        }
        a.out_src_top[o] = rt;
        a.out_src_bot[o] = rq;
      }
    }
    base += total;
    __syncthreads();
  }
}

// ---- N4: dense triangulation of a panoramic disparity map (camera_models.py:2492-2538, 2567-2685) -----------------
// One thread per panorama pixel: 4 B in, 13 B out — meant to be an HBM-bound streaming kernel, so the float64 work per
// pixel is kept to ~40 FMAs and one reciprocal:
//   * rays on the unit cylinder are v = (cos az, sin az, tan el) with tan(el) = tan(atan2(h, r)) = h / r: no atan/tan;
//   * cos/sin of the azimuth depend on the column only: a per-column table (built by dense_column_table_kernel);
//   * with w = v1 x v2 and b = f2 - f1 the 3x3 solve of triangulate_midpoint() collapses to
//       P = f1 + ((b x v2).w / |w|^2) v1 + 0.5 (w.b / |w|^2) w        (n = w/|w|, det[v1,-v2,n] = -|w|).
//   Everything that depends on the column only is tabulated too (w.z, (b x v2).z, b.z sin az2, b.z cos az2).
__global__ void dense_column_table_kernel(PanoP pano_top, PanoP pano_bot, Vec3 b, int cols, double4* __restrict__ table) {
  const int u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= cols) return;
  double az1, az2, el;
  pano_pixel_to_angles(pano_top, (double)u, 0.0, az1, el);
  pano_pixel_to_angles(pano_bot, (double)u, 0.0, az2, el);
  double c1, s1, c2, s2;
  sincos(az1, &s1, &c1);
  sincos(az2, &s2, &c2);
  table[2 * u + 0] = make_double4(c1, s1, c2, s2);
  table[2 * u + 1] = make_double4(c1 * s2 - s1 * c2, b.x * s2 - b.y * c2, b.z * s2, b.z * c2);   // w.z, (b x v2).z, ...
}

constexpr int DT_ROWS = 16;   // rows per block: the column terms live in registers and are reused for all of them

__global__ void __launch_bounds__(256)
dense_triangulate_kernel(PanoP pano_top, PanoP pano_bot, const double4* __restrict__ table,
                         const float* __restrict__ disparity, int rows, int cols, int n_maps,
                         double min_disp, const float* __restrict__ max_disp_dev, double max_disp_host, double lowest_row,
                         int roi0, int roi1, Vec3 f1, Vec3 f2, double inv_r_top, double inv_r_bot, float* __restrict__ xyz,
                         uint8_t* __restrict__ valid) {
  // grid = (column blocks, row chunks, maps); thread = one panorama column, looping over DT_ROWS rows
  __shared__ float sxyz[3 * 256];   // a row segment's 256 x 3 floats leave as three fully coalesced store instructions
  const int u = blockIdx.x * blockDim.x + threadIdx.x, map = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool inside = u < cols;
  const int uc = inside ? u : cols - 1;
  const double4 cs = table[2 * uc], ct = table[2 * uc + 1];
  const Vec3 b = {f2.x - f1.x, f2.y - f1.y, f2.z - f1.z};
  const double dmax = max_disp_dev ? (double)max_disp_dev[map] : max_disp_host;  // :2507-2508 (0 -> the map's maximum)
  const bool in_roi = inside && u >= roi0 && u < roi1;                            // :2500-2503
  const int u0 = blockIdx.x * blockDim.x;
  const int nfl = 3 * min((int)blockDim.x, cols - u0);
  const int v0 = blockIdx.y * DT_ROWS;
  const int v_end = min(rows, v0 + DT_ROWS);
  float dreg[DT_ROWS];   // all disparities of the block's rows are in flight before the first one is used
#pragma unroll
  for (int k = 0; k < DT_ROWS; ++k)
    dreg[k] = (in_roi && v0 + k < rows) ? __ldg(disparity + ((size_t)map * rows + v0 + k) * cols + uc) : 0.f;
#pragma unroll
  for (int k = 0; k < DT_ROWS; ++k) {
    const int v = v0 + k;
    if (v >= v_end) break;
    const size_t i = ((size_t)map * rows + v) * cols + uc;
    const double d = (double)dreg[k];
    const bool ok = d != 0.0 && min_disp <= d && d <= dmax && ((double)v - d) <= lowest_row;   // :2511-2525
    float o0 = CUDART_NAN_F, o1 = CUDART_NAN_F, o2 = CUDART_NAN_F;
    const double vb = (double)v - d;                                               // :2529: bottom pixel (u, v - d)
    if (ok && 0.0 <= vb && vb < pano_bot.v[SOS_PANO_ROWS] && (double)v < pano_top.v[SOS_PANO_ROWS]) {
      const double t1 = (pano_top.v[SOS_PANO_HEIGHT_MAX] - pano_top.v[SOS_PANO_PIXEL_SIZE] * (double)v) * inv_r_top;
      const double t2 = (pano_bot.v[SOS_PANO_HEIGHT_MAX] - pano_bot.v[SOS_PANO_PIXEL_SIZE] * vb) * inv_r_bot;
      const Vec3 w = {cs.y * t2 - t1 * cs.w, t1 * cs.z - cs.x * t2, ct.x};      // v1 x v2
      const Vec3 bv = {b.y * t2 - ct.z, ct.w - b.x * t2, ct.y};                  // b x v2
      const double inv = 1.0 / (w.x * w.x + w.y * w.y + w.z * w.z);
      const double l1 = (bv.x * w.x + bv.y * w.y + bv.z * w.z) * inv;
      const double hp = 0.5 * (w.x * b.x + w.y * b.y + w.z * b.z) * inv;
      o0 = (float)(f1.x + l1 * cs.x + hp * w.x);
      o1 = (float)(f1.y + l1 * cs.y + hp * w.y);
      o2 = (float)(f1.z + l1 * t1 + hp * w.z);
    }
    // each warp stages its 32 x 3 floats and writes them as three coalesced 128-byte stores: no block-wide barrier
    float* sw = sxyz + 96 * warp;
    sw[3 * lane + 0] = o0;
    sw[3 * lane + 1] = o1;
    sw[3 * lane + 2] = o2;
    if (valid && inside) valid[i] = ok ? 1 : 0;
    __syncwarp();
    float* dst = xyz + 3 * (((size_t)map * rows + v) * cols + u0 + 32 * warp);
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      const int j = q * 32 + lane;
      if (96 * warp + j < nfl) dst[j] = sw[j];
    }
    __syncwarp();
  }
}

// per-map maximum of the ROI-masked disparity (max_disparity = 0 in the reference means "the map's maximum")
__global__ void __launch_bounds__(1024)
disparity_max_kernel(const float* __restrict__ disparity, int rows, int cols, int roi0, int roi1, float* __restrict__ out) {
  __shared__ float red[32];
  const size_t per_map = (size_t)rows * cols;
  const float* d = disparity + (size_t)blockIdx.x * per_map;
  float m = 0.f;   // the ROI mask writes zeros, so the maximum is never below 0 (camera_models.py:2500-2503)
  bool any_outside = roi0 > 0 || roi1 < cols;
  if (!any_outside) m = -CUDART_INF_F;
  for (size_t k = threadIdx.x; k < per_map; k += blockDim.x) {
    const int u = (int)(k % cols);
    if (u >= roi0 && u < roi1) m = fmaxf(m, d[k]);
  }
  for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, off));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    m = red[threadIdx.x];
    for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, off));
    if (threadIdx.x == 0) out[blockIdx.x] = m;
  }
}

// ---- F3: GUM forward projection, gum.py:2512-2562, 1368-1385, 2942-2959 ----------------------------------------
__device__ __forceinline__ void gum_project(const GumP& g, Vec3 P, double& u, double& v) {
  const double nrm = sqrt(P.x * P.x + P.y * P.y + P.z * P.z);
  const double qx = P.x / nrm - g.v[SOS_GUM_XI1], qy = P.y / nrm - g.v[SOS_GUM_XI2], qz = P.z / nrm - g.v[SOS_GUM_XI3];
  const double az = fabs(qz);
  double x = qx / az, y = qy / az;
  if (g.v[SOS_GUM_USE_DISTORTION] != 0.0) {
    const double r2 = x * x + y * y;
    const double f = 1.0 + g.v[SOS_GUM_K1] * r2 + g.v[SOS_GUM_K2] * r2 * r2 + g.v[SOS_GUM_K3] * r2 * r2 * r2;
    x *= f;
    y *= f;
  }
  u = g.v[SOS_GUM_GAMMA1] * x + g.v[SOS_GUM_GAMMA1] * g.v[SOS_GUM_ALPHA_C] * y + g.v[SOS_GUM_U0];
  v = g.v[SOS_GUM_GAMMA2] * y + g.v[SOS_GUM_V0];
}

__global__ void gum_project_kernel(GumP g, const double* __restrict__ pts, int n, double* __restrict__ uv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double u, v;
  gum_project(g, {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]}, u, v);
  uv[2 * i] = u;
  uv[2 * i + 1] = v;
}

__global__ void lut_build_kernel(GumP g, int rows, int cols, double h_max, double h_min, double elev_lo, double elev_hi,
                                 double* __restrict__ map_x, double* __restrict__ map_y) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y;
  if (c >= cols) return;
  // panorama.py:429-441: psi = reversed linspace(0, 2pi, cols, endpoint=False), theta = atan2(linspace(h_max, h_min,
  // rows, endpoint=False), 1) validated against the mirror's own elevation band; both rounded to float32.
  const double psi_step = (2.0 * CUDART_PI) / (double)cols;
  const double psi = (double)(float)((double)(cols - 1 - c) * psi_step);
  const double h = h_max + (double)r * ((h_min - h_max) / (double)rows);
  double theta = atan2(h, 1.0);
  if (!(elev_lo <= theta && theta <= elev_hi)) theta = CUDART_NAN;
  theta = (double)(float)theta;
  const Vec3 s = angles_to_sphere(psi, theta);
  double u, v;
  gum_project(g, s, u, v);
  map_x[(size_t)r * cols + c] = u;
  map_y[(size_t)r * cols + c] = v;
}

// ---- F9: GUM omni-pixel -> unit sphere, gum.py:2653-2762, camera_models.py:135-187 -----------------------------
__global__ void lift_gum_kernel(GumP g, const double* __restrict__ uv, int n, double* __restrict__ sphere,
                                double* __restrict__ az, double* __restrict__ el) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double u = uv[2 * i], v = uv[2 * i + 1];
  const double g1 = g.v[SOS_GUM_GAMMA1], g2 = g.v[SOS_GUM_GAMMA2], ac = g.v[SOS_GUM_ALPHA_C];
  const double u0 = g.v[SOS_GUM_U0], v0 = g.v[SOS_GUM_V0];
  // inverse camera matrix, gum.py:136-140
  const double ik11 = 1.0 / g1, ik12 = -ac / g2, ik13 = ac * v0 / g2 - u0 / g1, ik22 = 1.0 / g2, ik23 = -v0 / g2;
  const double xd = ik11 * u + ik12 * v + ik13, yd = ik22 * v + ik23;
  double xu = xd, yu = yd;
  if (g.v[SOS_GUM_USE_DISTORTION] != 0.0) {
    if (g.v[SOS_GUM_L1] != 0.0) {  // gum.py:2689-2694: multiplicative inverse radial model
      const double r2 = xd * xd + yd * yd;
      const double f = 1.0 + g.v[SOS_GUM_L1] * r2 + g.v[SOS_GUM_L2] * r2 * r2 + g.v[SOS_GUM_L3] * r2 * r2 * r2;
      xu = xd * f;
      yu = yd * f;
    } else {  // gum.py:2713-2725: Heikkila closed form (k3 unused there)
      const double k1 = g.v[SOS_GUM_K1], k2 = g.v[SOS_GUM_K2], p1 = g.v[SOS_GUM_P1], p2 = g.v[SOS_GUM_P2];
      const double x2 = xd * xd, y2 = yd * yd, xy = xd * yd, r2 = x2 + y2, r4 = r2 * r2;
      const double rad = k1 * r2 + k2 * r4;
      const double dx = xd * rad + p2 * (r2 + 2.0 * x2) + 2.0 * p1 * xy;
      const double dy = yd * rad + p1 * (r2 + 2.0 * y2) + 2.0 * p2 * xy;
      const double inv = 1.0 / (1.0 + 4.0 * k1 * r2 + 6.0 * k2 * r4 + 8.0 * p1 * yd + 8.0 * p2 * xd);
      xu = xd - inv * dx;
      yu = yd - inv * dy;
    }
  }
  // point on the normalised plane wrt [M] and the line from it with direction (p - Cp): gum.py:2748-2752
  const double cx = g.v[SOS_GUM_XI1], cy = g.v[SOS_GUM_XI2], cz = g.v[SOS_GUM_XI3];
  const double px = cx + xu, py = cy + yu, pz = g.v[SOS_GUM_PLANE_K];
  const double vx = px - cx, vy = py - cy, vz = pz - cz;
  // unit-sphere intersection, first root (camera_models.py:165-186, gum.py:2762)
  const double A = vx * vx + vy * vy + vz * vz;
  const double B = 2.0 * (vx * px + vy * py + vz * pz);
  const double Cc = px * px + py * py + pz * pz - 1.0;
  const double t = (-B + sqrt(B * B - 4.0 * A * Cc)) / (2.0 * A);
  const double sx = px + t * vx, sy = py + t * vy, sz = pz + t * vz;
  if (sphere) {
    sphere[3 * i] = sx;
    sphere[3 * i + 1] = sy;
    sphere[3 * i + 2] = sz;
  }
  if (az) az[i] = atan2(sy, sx);  // camera_models.py:1191-1193
  if (el) el[i] = asin(sz);
}

// ---- F12: RGB-D, camera_models.py:781-799, 835-860, 203-212; pose_est_tools.py:612-620 (rgbd.cuh) -------------

// One thread per pixel position, looping over the frames: the double-precision square root of the radial model depends on
// (x, y) only, so it is taken once per thread and the per-frame work is one multiply and one divide (first version: sqrt and
// divide per element, 0.36 ms for 256 VGA frames = 0.27 of the HBM roofline, FP64-pipe bound).
constexpr int RGBD_Z_SLICES = 8;

__global__ void rgbd_depth_to_z_kernel(RgbdP c, const float* __restrict__ depth, int batch, int h, int w, float* __restrict__ z) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= w) return;
  const bool is_z = c.v[SOS_RGBD_DEPTH_IS_Z] != 0.0;
  const double f = c.v[SOS_RGBD_FOCAL_M];
  const double xi = (f / c.v[SOS_RGBD_FX]) * ((double)x - c.v[SOS_RGBD_CX]);
  const double yi = (f / c.v[SOS_RGBD_FY]) * ((double)y - c.v[SOS_RGBD_CY]);
  const double den = sqrt(xi * xi + yi * yi + f * f);
  const size_t plane = (size_t)h * w, o0 = (size_t)y * w + x;
  for (int b = blockIdx.z; b < batch; b += gridDim.z) {
    const float d = depth[b * plane + o0];
    z[b * plane + o0] = is_z ? d : (float)(f * (double)d / den);     // same operations as rgbd_depth_z
  }
}

__global__ void rgbd_backproject_kernel(RgbdP c, const float* __restrict__ depth, int h, int w,
                                        const int32_t* __restrict__ us, const int32_t* __restrict__ vs, int n, double zmin,
                                        double zmax, float* __restrict__ xyz, float* __restrict__ bearing,
                                        uint8_t* __restrict__ valid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int b = blockIdx.y;
  const size_t o = (size_t)b * n + i;
  float p[3], f[3];
  const bool ok = rgbd_point(c, depth + (size_t)b * h * w, h, w, us[o], vs[o], zmin, zmax, p, f);
  xyz[3 * o] = p[0]; xyz[3 * o + 1] = p[1]; xyz[3 * o + 2] = p[2];
  if (bearing) {
    bearing[3 * o] = f[0]; bearing[3 * o + 1] = f[1]; bearing[3 * o + 2] = f[2];
  }
  if (valid) valid[o] = ok ? 1 : 0;
}

static GumP load_gum(const double* g) {
  GumP p;
  for (int i = 0; i < SOS_GUM_NPARAMS; ++i) p.v[i] = g[i];
  return p;
}
static PanoP load_pano(const double* g) {
  PanoP p;
  for (int i = 0; i < SOS_PANO_NPARAMS; ++i) p.v[i] = g[i];
  return p;
}

}  // namespace

template <typename T>
static int lift_pano_impl(sos_ctx* ctx, const double* pano, const T* uv, int n, T* az, T* el, T* bearing) {
  SOS_CHECK_ARG(ctx && pano, "NULL argument");
  SOS_CHECK_ARG(n >= 0, "negative size");
  if (n == 0) return SOS_OK;
  SOS_CHECK_ARG(uv, "uv is NULL");
  SOS_CUDA(cudaSetDevice(ctx->device));
  lift_pano_kernel<T><<<sos_div_up(n, 256), 256, 0, ctx->stream>>>(load_pano(pano), uv, n, az, el, bearing);
  SOS_LAUNCHED_AS(ctx, "lift_pano_kernel");
  return SOS_OK;
}

extern "C" int sos_lift_pano(sos_ctx* ctx, const double* pano, const float* uv, int n, float* az, float* el,
                             float* bearing) {
  return lift_pano_impl<float>(ctx, pano, uv, n, az, el, bearing);
}

extern "C" int sos_lift_pano_f64(sos_ctx* ctx, const double* pano, const double* uv, int n, double* az, double* el,
                                 double* bearing) {
  return lift_pano_impl<double>(ctx, pano, uv, n, az, el, bearing);
}

template <typename T>
static int triangulate_impl(sos_ctx* ctx, const T* az1, const T* el1, const T* az2, const T* el2, int n, const double* f1,
                            const double* f2, double rmin, double rmax, int homogeneous_norm, T* xyz, uint8_t* valid) {
  SOS_CHECK_ARG(ctx && f1 && f2, "NULL argument");
  SOS_CHECK_ARG(n >= 0, "negative size");
  if (n == 0) return SOS_OK;
  SOS_CHECK_ARG(az1 && el1 && az2 && el2 && xyz, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  triangulate_kernel<T><<<sos_div_up(n, 256), 256, 0, ctx->stream>>>(az1, el1, az2, el2, n, {f1[0], f1[1], f1[2]},
                                                                    {f2[0], f2[1], f2[2]}, rmin, rmax, homogeneous_norm,
                                                                    xyz, valid);
  SOS_LAUNCHED_AS(ctx, "triangulate_kernel");
  return SOS_OK;
}

extern "C" int sos_triangulate_midpoint(sos_ctx* ctx, const float* az1, const float* el1, const float* az2,
                                        const float* el2, int n, const double* f1, const double* f2, double rmin,
                                        double rmax, int homogeneous_norm, float* xyz, uint8_t* valid) {
  return triangulate_impl<float>(ctx, az1, el1, az2, el2, n, f1, f2, rmin, rmax, homogeneous_norm, xyz, valid);
}

extern "C" int sos_triangulate_midpoint_f64(sos_ctx* ctx, const double* az1, const double* el1, const double* az2,
                                            const double* el2, int n, const double* f1, const double* f2, double rmin,
                                            double rmax, int homogeneous_norm, double* xyz, uint8_t* valid) {
  return triangulate_impl<double>(ctx, az1, el1, az2, el2, n, f1, f2, rmin, rmax, homogeneous_norm, xyz, valid);
}

extern "C" int sos_stereo_lift_triangulate(sos_ctx* ctx, const double* pano_top, const double* pano_bot,
                                           const float* px_top, const float* px_bot, const int32_t* pair_q,
                                           const int32_t* pair_t, const int32_t* pair_count, const int32_t* seg_off,
                                           int n_frames, int segs_per_frame, int max_pairs_per_seg, int pair_rows,
                                           const double* f1, const double* f2, double rmin, double rmax,
                                           int homogeneous_norm, int cap_per_frame,
                                           float* out_uv_top, float* out_uv_bot, float* out_b_top, float* out_b_bot,
                                           float* out_xyz, int32_t* out_src_top, int32_t* out_src_bot, int32_t* out_n) {
  SOS_CHECK_ARG(ctx && pano_top && pano_bot && f1 && f2, "NULL argument");
  SOS_CHECK_ARG(n_frames >= 0 && segs_per_frame >= 0 && cap_per_frame >= 0 && max_pairs_per_seg >= 0 && pair_rows >= 0,
                "negative size");
  SOS_CHECK_ARG((long long)n_frames * segs_per_frame <= 65535, "too many segments");
  if (n_frames == 0) return SOS_OK;
  SOS_CHECK_ARG(px_top && px_bot && pair_q && pair_t && pair_count && seg_off, "NULL input array");
  SOS_CHECK_ARG(out_uv_top && out_uv_bot && out_b_top && out_b_bot && out_xyz && out_src_top && out_src_bot && out_n,
                "NULL output array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  StereoArgs a;
  a.pano_top = load_pano(pano_top);
  a.pano_bot = load_pano(pano_bot);
  a.px_top = (const float2*)px_top; a.px_bot = (const float2*)px_bot;
  a.pair_q = pair_q; a.pair_t = pair_t; a.pair_count = pair_count; a.seg_off = seg_off;
  a.segs_per_frame = segs_per_frame;
  a.f1 = {f1[0], f1[1], f1[2]}; a.f2 = {f2[0], f2[1], f2[2]};
  a.rmin = rmin; a.rmax = rmax; a.homo = homogeneous_norm; a.cap = cap_per_frame;
  a.out_uv_top = (float2*)out_uv_top; a.out_uv_bot = (float2*)out_uv_bot;
  a.out_b_top = out_b_top; a.out_b_bot = out_b_bot; a.out_xyz = out_xyz;
  a.out_src_top = out_src_top; a.out_src_bot = out_src_bot; a.out_n = out_n;
  void* ws = nullptr;
  const size_t tmp_bytes = sos_align_up((size_t)pair_rows * 9 * sizeof(float), 256);
  const int n_segs = n_frames * segs_per_frame;
  const size_t keep_bytes = sos_align_up((size_t)pair_rows + 1, 256);
  const int rc = sos_arena_get(ctx, tmp_bytes + keep_bytes + (size_t)(n_segs + 1) * sizeof(int32_t) + 256, &ws);
  if (rc != SOS_OK) return rc;
  a.tmp = (float*)ws;
  a.tmp_keep = (uint8_t*)ws + tmp_bytes;
  a.seg_keep = (int32_t*)((uint8_t*)ws + tmp_bytes + keep_bytes);
  if (n_segs == 0) {
    SOS_CUDA(cudaMemsetAsync(out_n, 0, (size_t)n_frames * sizeof(int32_t), ctx->stream));
    return SOS_OK;
  }
  SOS_CUDA(cudaMemsetAsync(a.seg_keep, 0, (size_t)n_segs * sizeof(int32_t), ctx->stream));
  if (max_pairs_per_seg > 0) {
    dim3 grid(sos_div_up(max_pairs_per_seg, 256), n_segs);
    stereo_geometry_kernel<<<grid, 256, 0, ctx->stream>>>(a);
    SOS_LAUNCHED_AS(ctx, "stereo_geometry_kernel");
  }
  stereo_compact_kernel<<<n_segs, ST_THREADS, 0, ctx->stream>>>(a);
  SOS_LAUNCHED_AS(ctx, "stereo_compact_kernel");
  return SOS_OK;
}

extern "C" int sos_gum_project(sos_ctx* ctx, const double* gum, const double* pts, int n, double* uv) {
  SOS_CHECK_ARG(ctx && gum, "NULL argument");
  SOS_CHECK_ARG(n >= 0, "negative size");
  if (n == 0) return SOS_OK;
  SOS_CHECK_ARG(pts && uv, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  gum_project_kernel<<<sos_div_up(n, 256), 256, 0, ctx->stream>>>(load_gum(gum), pts, n, uv);
  SOS_LAUNCHED_AS(ctx, "gum_project_kernel");
  return SOS_OK;
}

extern "C" int sos_lut_build(sos_ctx* ctx, const double* gum, int rows, int cols, double cyl_height_max,
                             double cyl_height_min, double elev_lo, double elev_hi, double* map_x, double* map_y) {
  SOS_CHECK_ARG(ctx && gum, "NULL argument");
  SOS_CHECK_ARG(rows >= 0 && cols >= 0 && rows <= 65535, "bad size");
  if (rows == 0 || cols == 0) return SOS_OK;
  SOS_CHECK_ARG(map_x && map_y, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  dim3 grid(sos_div_up(cols, 256), rows);
  lut_build_kernel<<<grid, 256, 0, ctx->stream>>>(load_gum(gum), rows, cols, cyl_height_max, cyl_height_min, elev_lo,
                                                  elev_hi, map_x, map_y);
  SOS_LAUNCHED_AS(ctx, "lut_build_kernel");
  return SOS_OK;
}

extern "C" int sos_lift_gum(sos_ctx* ctx, const double* gum, const double* uv, int n, double* sphere, double* az,
                            double* el) {
  SOS_CHECK_ARG(ctx && gum, "NULL argument");
  SOS_CHECK_ARG(n >= 0, "negative size");
  if (n == 0) return SOS_OK;
  SOS_CHECK_ARG(uv, "uv is NULL");
  SOS_CUDA(cudaSetDevice(ctx->device));
  lift_gum_kernel<<<sos_div_up(n, 256), 256, 0, ctx->stream>>>(load_gum(gum), uv, n, sphere, az, el);
  SOS_LAUNCHED_AS(ctx, "lift_gum_kernel");
  return SOS_OK;
}

extern "C" int sos_rgbd_depth_to_z(sos_ctx* ctx, const double* cam, const float* depth, int batch, int h, int w,
                                   float* z) {
  SOS_CHECK_ARG(ctx && cam, "NULL argument");
  SOS_CHECK_ARG(batch >= 0 && h >= 0 && w >= 0 && h <= 65535 && batch <= 65535, "bad size");
  if (batch == 0 || h == 0 || w == 0) return SOS_OK;
  SOS_CHECK_ARG(depth && z, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  RgbdP c;
  for (int i = 0; i < SOS_RGBD_NPARAMS; ++i) c.v[i] = cam[i];
  dim3 grid(sos_div_up(w, 128), h, batch < RGBD_Z_SLICES ? batch : RGBD_Z_SLICES);
  rgbd_depth_to_z_kernel<<<grid, 128, 0, ctx->stream>>>(c, depth, batch, h, w, z);
  SOS_LAUNCHED_AS(ctx, "rgbd_depth_to_z_kernel");
  return SOS_OK;
}

extern "C" int sos_rgbd_backproject(sos_ctx* ctx, const double* cam, const float* depth, int batch, int h, int w,
                                    const int32_t* u, const int32_t* v, int n, double zmin, double zmax, float* xyz,
                                    float* bearing, uint8_t* valid) {
  SOS_CHECK_ARG(ctx && cam, "NULL argument");
  SOS_CHECK_ARG(batch >= 0 && h > 0 && w > 0 && n >= 0 && batch <= 65535, "bad size");
  if (batch == 0 || n == 0) return SOS_OK;
  SOS_CHECK_ARG(depth && u && v && xyz, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  RgbdP c;
  for (int i = 0; i < SOS_RGBD_NPARAMS; ++i) c.v[i] = cam[i];
  dim3 grid(sos_div_up(n, 256), batch);
  rgbd_backproject_kernel<<<grid, 256, 0, ctx->stream>>>(c, depth, h, w, u, v, n, zmin, zmax, xyz, bearing, valid);
  SOS_LAUNCHED_AS(ctx, "rgbd_backproject_kernel");
  return SOS_OK;
}

// ---- stand-alone F8 and F11 for the per-call Python mirror (float64, the reference's dtype) ---------------------
namespace {
__global__ void angles_to_sphere_kernel(const double* __restrict__ az, const double* __restrict__ el, int n,
                                        double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Vec3 s = angles_to_sphere(az[i], el[i]);  // NaN elevation / azimuth propagate as in camera_models.py:1046-1053
  out[3 * i] = s.x;
  out[3 * i + 1] = s.y;
  out[3 * i + 2] = s.z;
}

__global__ void range_gate_kernel(const double* __restrict__ xyz, int n, double rmin, double rmax, int homo,
                                  uint8_t* __restrict__ valid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  valid[i] = range_ok({xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]}, rmin, rmax, homo) ? 1 : 0;
}
}  // namespace

extern "C" int sos_angles_to_sphere_f64(sos_ctx* ctx, const double* az, const double* el, int n, double* sphere) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n >= 0, "negative size");
  if (n == 0) return SOS_OK;
  SOS_CHECK_ARG(az && el && sphere, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  angles_to_sphere_kernel<<<sos_div_up(n, 256), 256, 0, ctx->stream>>>(az, el, n, sphere);
  SOS_LAUNCHED_AS(ctx, "angles_to_sphere_kernel");
  return SOS_OK;
}

extern "C" int sos_range_gate_f64(sos_ctx* ctx, const double* xyz, int n, double rmin, double rmax, int homogeneous_norm,
                                  uint8_t* valid) {
  SOS_CHECK_ARG(ctx, "ctx is NULL");
  SOS_CHECK_ARG(n >= 0, "negative size");
  if (n == 0) return SOS_OK;
  SOS_CHECK_ARG(xyz && valid, "NULL array");
  SOS_CUDA(cudaSetDevice(ctx->device));
  range_gate_kernel<<<sos_div_up(n, 256), 256, 0, ctx->stream>>>(xyz, n, rmin, rmax, homogeneous_norm, valid);
  SOS_LAUNCHED_AS(ctx, "range_gate_kernel");
  return SOS_OK;
}

extern "C" int sos_dense_triangulate(sos_ctx* ctx, const double* pano_top, const double* pano_bot, const float* disparity,
                                     int n_maps, int rows, int cols, double min_disparity, double max_disparity,
                                     double lowest_reference_row, int roi_col0, int roi_col1, const double* f1,
                                     const double* f2, float* xyz, uint8_t* valid) {
  SOS_CHECK_ARG(ctx && pano_top && pano_bot && f1 && f2, "NULL argument");
  SOS_CHECK_ARG(n_maps >= 0 && rows >= 0 && cols >= 0, "negative size");
  if (n_maps == 0 || rows == 0 || cols == 0) return SOS_OK;
  SOS_CHECK_ARG(disparity && xyz, "NULL array");
  SOS_CHECK_ARG(n_maps <= 65535, "too many maps");
  SOS_CUDA(cudaSetDevice(ctx->device));
  if (roi_col0 < 0 || roi_col1 < 0) { roi_col0 = 0; roi_col1 = cols; }
  roi_col1 = roi_col1 < cols ? roi_col1 : cols;
  float* dmax = nullptr;
  void* ws = nullptr;
  const size_t table_bytes = sos_align_up((size_t)cols * 2 * sizeof(double4), 256);
  const int rc = sos_arena_get(ctx, table_bytes + sos_align_up((size_t)n_maps * sizeof(float), 256), &ws);
  if (rc != SOS_OK) return rc;
  double4* table = (double4*)ws;
  dense_column_table_kernel<<<sos_div_up(cols, 256), 256, 0, ctx->stream>>>(
      load_pano(pano_top), load_pano(pano_bot), {f2[0] - f1[0], f2[1] - f1[1], f2[2] - f1[2]}, cols, table);
  SOS_LAUNCHED_AS(ctx, "dense_column_table_kernel");
  if (max_disparity == 0.0) {
    dmax = (float*)((uint8_t*)ws + table_bytes);
    disparity_max_kernel<<<n_maps, 1024, 0, ctx->stream>>>(disparity, rows, cols, roi_col0, roi_col1, dmax);
    SOS_LAUNCHED_AS(ctx, "disparity_max_kernel");
  }
  SOS_CHECK_ARG(rows <= 65535, "more than 65535 panorama rows");
  dense_triangulate_kernel<<<dim3(sos_div_up(cols, 256), sos_div_up(rows, DT_ROWS), n_maps), 256, 0, ctx->stream>>>(
      load_pano(pano_top), load_pano(pano_bot), table, disparity, rows, cols, n_maps, min_disparity, dmax, max_disparity,
      lowest_reference_row, roi_col0, roi_col1, {f1[0], f1[1], f1[2]}, {f2[0], f2[1], f2[2]},
      1.0 / pano_top[SOS_PANO_RADIUS], 1.0 / pano_bot[SOS_PANO_RADIUS], xyz, valid);
  SOS_LAUNCHED_AS(ctx, "dense_triangulate_kernel");
  return SOS_OK;
}
