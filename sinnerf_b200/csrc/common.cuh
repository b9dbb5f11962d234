// common.cuh -- shared host/device definitions for libsinnerf_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>

#include "../../include/sinnerf_b200.h"

namespace snb {

// ------------------------------------------------------------------ errors (host)
void set_error(const std::string& msg);
int fail(int code, const char* fmt, ...);
int check_launch(const char* what);

// ------------------------------------------------------------------ per-device launch state (host)
// The library may be driven on several GPUs from one process (one device current per call): SM counts and
// the opt-in dynamic-shared-memory attribute are per DEVICE, so both are cached per device ordinal.
constexpr int kMaxDevices = 64;
int current_device();   // ordinal of the current CUDA device
int sm_count();         // its SM count (cached per ordinal)
struct SmemOptIn {      // one zero-initialised static per kernel instantiation
  int bytes[kMaxDevices];
};
template <class Kernel>
inline int ensure_smem(Kernel kernel, SmemOptIn& st, int bytes, const char* what) {
  const int dev = current_device() & (kMaxDevices - 1);
  if (st.bytes[dev] >= bytes) return SNB_OK;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return fail(SNB_ERR_CUDA, "cudaFuncSetAttribute(%s): %s", what, cudaGetErrorString(e));
  st.bytes[dev] = bytes;
  return SNB_OK;
}

#define SNB_REQUIRE(cond, ...)                           \
  do {                                                   \
    if (!(cond)) return ::snb::fail(SNB_ERR_INVALID, __VA_ARGS__); \
  } while (0)

// ------------------------------------------------------------------ field MLP shape
// NeRF(D=8, W=256, in_xyz=63, in_dir=27, skips=[4])  (reference models/nerf.py:47-103)
constexpr int kWidth = 256;
constexpr int kHalf = 128;
constexpr int kXyzCh = 63, kXyzPad = 64;
constexpr int kDirCh = 27, kDirPad = 32;
constexpr int kNumGemm = 10;  // 8 trunk layers, bottleneck ("final"), direction layer

// GEMM l computes  out[N_l] = act(W_l[K_l] . in + b_l); K is the PADDED, CONCAT-SPLIT depth:
//   l=0      : [enc(64)]                 l=4 : [enc(64) | hidden(256)]   (skip, nerf.py:132-133)
//   l=9 (dir): [bottleneck(256) | dir(32)]   (nerf.py:142)
__host__ __device__ constexpr int gemm_k(int l) {
  return l == 0 ? 64 : (l == 4 ? 320 : (l == 9 ? 288 : 256));
}
__host__ __device__ constexpr int gemm_n(int l) { return l == 9 ? kHalf : kWidth; }
// column of the nn.Linear weight a padded k maps to, or -1 for a zero pad row
__host__ __device__ constexpr int gemm_src_col(int l, int k) {
  return l == 0 ? (k < 63 ? k : -1)
                : (l == 4 ? (k < 63 ? k : (k == 63 ? -1 : k - 1)) : (l == 9 ? (k < 283 ? k : -1) : k));
}
// index of layer l's weight / bias in the 24-pointer state-dict order
__host__ __device__ constexpr int param_weight_index(int l) { return 2 * l; }  // l = 0..9 (8 = final, 9 = dir)
constexpr int kSigmaW = 20, kSigmaB = 21, kRgbW = 22, kRgbB = 23;

// ------------------------------------------------------------------ packed image header
struct PackedHeader {
  uint32_t magic;      // 'SNBW'
  int32_t precision;   // SNB_PREC_*
  int32_t new_activation;
  int32_t reserved0;   // unused; keeps the fields below at their offsets (tests read `dirty` as word 4)
  // snb_refresh_weights: a position-dependent 64-bit checksum of the 24 fp32 parameter tensors the image was
  // packed from.  The check kernel recomputes it on the device and sets `dirty`; the pack kernels of a
  // refresh return immediately when it is 0 -- no host round trip, and in-place updates that bypass
  // autograd's version counter (`p.data.copy_`, reference utils/optimizers.py:98,180,268) are still seen.
  int32_t dirty;
  uint32_t blocks_done;          // scratch of the check kernel (self-resetting)
  unsigned long long checksum;
  unsigned long long partial;    // scratch of the check kernel (self-resetting)
  int32_t reserved[54];
};
static_assert(sizeof(PackedHeader) == 256, "header is 256 B so payloads stay 256-B aligned");
constexpr uint32_t kMagic = 0x57424e53u;

// element counts of the 24 parameter tensors in state-dict order (weight, bias per layer)
__host__ __device__ constexpr int param_numel(int i) {
  // weights: l0 256x63, l1-3 256x256, l4 256x319, l5-7 256x256, final 256x256, dir 128x283, sigma 1x256, rgb 3x128
  return (i & 1) ? (i < 18 ? 256 : (i == 19 ? 128 : (i == 21 ? 1 : 3)))
                 : (i == 0 ? 256 * 63 : (i == 8 ? 256 * 319 : (i < 18 ? 256 * 256 : (i == 18 ? 128 * 283 : (i == 20 ? 256 : 384)))));
}
struct ParamPtrs {
  const float* p[SNB_N_PARAM_TENSORS];
};
// enqueues the check kernel: header.dirty = (image was not packed from exactly these values / this mode)
int launch_params_check(const ParamPtrs& pp, int precision, int new_activation, void* image, cudaStream_t st);

// ------------------------------------------------------------------ fp32 (FFMA) image
// floats after the header:
//   Wt_l  [K_l][N_l]  (K-major: one K row = N_l contiguous outputs)   l = 0..9
//   bias_l [N_l]                                                      l = 0..9
//   sigma_w[256], sigma_b[4], rgb_w[3][128], rgb_b[4]
struct Fp32Layout {
  int w[kNumGemm];
  int b[kNumGemm];
  int sigma_w, sigma_b, rgb_w, rgb_b, total;
};
__host__ __device__ constexpr Fp32Layout make_fp32_layout() {
  Fp32Layout L{};
  int off = 0;
  for (int l = 0; l < kNumGemm; ++l) {
    L.w[l] = off;
    off += gemm_k(l) * gemm_n(l);
  }
  for (int l = 0; l < kNumGemm; ++l) {
    L.b[l] = off;
    off += gemm_n(l);
  }
  L.sigma_w = off; off += kWidth;
  L.sigma_b = off; off += 4;
  L.rgb_w = off;   off += 3 * kHalf;
  L.rgb_b = off;   off += 4;
  L.total = off;
  return L;
}

// ------------------------------------------------------------------ device helpers
__device__ __forceinline__ float shifted_softplus_f(float x) {
  // reference models/activations.py:23-35
  float s = x - 1.0f;
  return log1pf(expf(-fabsf(s))) + (s >= 0.0f ? s : 0.0f);
}
__device__ __forceinline__ float widened_sigmoid_f(float x) {
  // reference models/activations.py:8-20
  return 0.5f * (1.0f + 1.002f * tanhf(0.5f * x));
}
__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

}  // namespace snb
