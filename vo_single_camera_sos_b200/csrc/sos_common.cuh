// Shared plumbing of libsosfront.so: the context object, error reporting and launch helpers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "sosfront.h"

struct sos_prof_mark {
  const char* name;  // __func__ of the C-ABI entry point that launched the kernel (static storage)
  cudaEvent_t ev;    // recorded right after the launch
};

struct sos_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  void* arena = nullptr;  // grow-only scratch
  size_t arena_bytes = 0;
  int64_t launches = 0;
  int sm_count = 148;
  bool prof = false;      // per-launch CUDA-event timing (sos_ctx_profile_begin / _end)
  std::vector<sos_prof_mark> marks;
};

void sos_set_error(const char* fmt, ...);
void sos_prof_mark_launch(sos_ctx* ctx, const char* name);

#define SOS_CHECK_ARG(cond, msg)                                  \
  do {                                                            \
    if (!(cond)) {                                                \
      sos_set_error("%s: invalid argument: %s", __func__, msg);   \
      return SOS_ERR_INVALID;                                     \
    }                                                             \
  } while (0)

#define SOS_CUDA(call)                                                                     \
  do {                                                                                     \
    cudaError_t e__ = (call);                                                              \
    if (e__ != cudaSuccess) {                                                              \
      sos_set_error("%s: %s failed: %s", __func__, #call, cudaGetErrorString(e__));        \
      return SOS_ERR_CUDA;                                                                 \
    }                                                                                      \
  } while (0)

// Call after every kernel launch: counts it and surfaces launch-configuration errors.  The profiling mark carries the
// kernel's name (SOS_LAUNCHED_AS) or, by default, the entry point that launched it.
#define SOS_LAUNCHED(ctx) SOS_LAUNCHED_AS(ctx, __func__)
#define SOS_LAUNCHED_AS(ctx, mark_name)                                                    \
  do {                                                                                     \
    (ctx)->launches++;                                                                     \
    if ((ctx)->prof) sos_prof_mark_launch((ctx), (mark_name));                             \
    cudaError_t e__ = cudaPeekAtLastError();                                               \
    if (e__ != cudaSuccess) {                                                              \
      (void)cudaGetLastError();                                                            \
      sos_set_error("%s: kernel launch failed: %s", __func__, cudaGetErrorString(e__));    \
      return SOS_ERR_CUDA;                                                                 \
    }                                                                                      \
  } while (0)

// Scratch arena: returns a pointer to at least `bytes` of device memory (256-byte aligned).
int sos_arena_get(sos_ctx* ctx, size_t bytes, void** out);

// Shi-Tomasi detection (csrc/gft.cu) on caller-owned buffers: the kernel sequence of sos_gft_detect, shared with the
// front-end's images-in step, which cannot read the candidate counts back.
constexpr int SOS_GFT_CAP = 16384;   // candidates per (image, mask) list the selection can rank
struct sos_gft_work {
  const uint32_t* mask_bits;   // [H*W] one bit per mask (sos_gft_pack_masks)
  float* eig;                  // [n_images, H, W]
  uint32_t* max_bits;          // [n_images * n_masks]
  int32_t* counts;             // [n_images * n_masks] candidates per list (> SOS_GFT_CAP: the list is refused)
  unsigned long long* keys;    // [n_images * n_masks * SOS_GFT_CAP]
  int32_t* rank_img;           // [n_images, H, W]: all -1 on entry, and the selection leaves it so
};
// masks uint8 [n_masks, H, W] (NULL = one mask covering everything) -> bits; *overlap = 1 if a pixel is in two masks
int sos_gft_pack_masks(sos_ctx* ctx, const uint8_t* masks, int height, int width, int n_masks, uint32_t* bits, int32_t* overlap);
// corner measure, mask maxima and candidate lists; image i of the batch starts at gray + i * img_stride
int sos_gft_candidates(sos_ctx* ctx, const sos_gft_work& w, const uint8_t* gray, size_t img_stride, int n_images, int height,
                       int width, int n_masks, double quality_level);
// strongest-first minimum-distance selection with shared memory for np2 sorted keys (np2 >= every list's count, or
// SOS_GFT_CAP); a list of more than SOS_GFT_CAP candidates gets out_count = -count and no corners.  overlap: the masks share
// pixels (one launch per mask).
int sos_gft_select(sos_ctx* ctx, const sos_gft_work& w, int n_images, int height, int width, int n_masks, int max_corners,
                   double min_distance, bool overlap, int np2, float* out_xy, int32_t* out_count);

// sos_orb_describe (csrc/orb.cu) with the blurred image in a caller-owned buffer blurred [n_images, H, W] instead of the
// scratch arena (arguments already checked by the caller)
int sos_orb_describe_into(sos_ctx* ctx, const uint8_t* gray, int n_images, int height, int width, const float* kp_xy,
                          const float* kp_angle_deg, const int32_t* kp_image, int n, uint32_t* desc, uint8_t* keep,
                          uint8_t* blurred);

static inline int sos_div_up(int a, int b) { return (a + b - 1) / b; }
static inline size_t sos_align_up(size_t a, size_t b) { return (a + b - 1) / b * b; }
