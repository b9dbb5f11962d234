// field_bwd.cu -- backward of the field MLP over fp32 saved activations (reference: autograd through
// models/nerf.py:105-148): the driver that walks the layers, the head kernel and the folded bottleneck.
// The two GEMMs of every layer run on tensor cores (wgrad_tc.cu, dgrad_tc.cu).
//
// Per render pass, given g_raw (P,4) = dL/d[r,g,b,sigma] from composite_bwd:
//   heads     : rgb head + its activation, direction-layer activation, sigma head  (head_bwd_kernel)
//   dir layer : W' = Wd[:, :256] Wf (fold_weights_kernel); dW', db' by one wgrad against h8; the chain
//               rule back to Wd, Wf, bf, bd is three P-independent products (unfold_grads_kernel)
//   per layer : dW_l += dY_l^T X_l, db_l += sum dY_l                               (wgrad_tc_kernel)
//               dX_l  = dY_l W_l  (x ReLU mask of the saved input, + sigma term at h8)  (dgrad_tc_kernel)
// walking dir layer -> layers 8..1.  Nothing flows into rays, z or across sample_pdf (the reference
// detaches it, models/rendering.py:311-313).
//
// Activations are plain (P, C) row-major fp32 tensors.  The wgrad of a layer also leaves the sign bits
// [X > 0] of its input in ws_m; the dgrad of the same layer reads them as its ReLU mask.
#include "common.cuh"

namespace snb {

// ------------------------------------------------------------------------------------------
// heads: one warp walks points; lanes own 4 of the 128 direction-layer units and 8 of the 256
// trunk units.  dS = (W_rgb^T g_pre_rgb) * act'(G);  dW_rgb, db_rgb, dW_sigma, db_sigma.
// ------------------------------------------------------------------------------------------
struct HeadArgs {
  const float* g_raw;   // (P,4)
  const float* raw;     // (P,4) forward output [rgb (post-activation), sigma]
  const float* G;       // (P,128) direction layer output
  const float* H8;      // (P,256)
  const float* Wr;      // (3,128)
  int new_activation;
  float* dS;            // (P,128)
  float* dWr; float* dbr; float* dWs; float* dbs;
  long long P;
};

__global__ void __launch_bounds__(256) head_bwd_kernel(HeadArgs a) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  float wr[3][4];
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int j = 0; j < 4; ++j) wr[c][j] = a.Wr[c * 128 + lane * 4 + j];
  float awr[3][4] = {}, abr[3] = {0.f, 0.f, 0.f}, aws[8] = {}, abs_ = 0.f;
  // 4 points per warp iteration: all their loads are issued before any is used (the kernel is a pure
  // HBM stream, 2 KB per point; one point at a time left it latency-bound)
  constexpr int kU = 4;
  for (long long pb = warp * kU; pb < a.P; pb += nwarps * kU) {
    float4 g[kU], o[kU], gv[kU], h0[kU], h1[kU];
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const long long p = pb + u < a.P ? pb + u : a.P - 1;      // tail: re-read the last point, contribute nothing
      g[u] = reinterpret_cast<const float4*>(a.g_raw)[p];
      o[u] = reinterpret_cast<const float4*>(a.raw)[p];
      gv[u] = *reinterpret_cast<const float4*>(a.G + p * 128 + lane * 4);
      h0[u] = *reinterpret_cast<const float4*>(a.H8 + p * 256 + lane * 8);
      h1[u] = *reinterpret_cast<const float4*>(a.H8 + p * 256 + lane * 8 + 4);
    }
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      if (pb + u >= a.P) break;
      const long long p = pb + u;
      float gp[3];
      const float gin[3] = {g[u].x, g[u].y, g[u].z}, out[3] = {o[u].x, o[u].y, o[u].z};
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        if (a.new_activation) {
          // y = 0.5 (1 + 1.002 tanh(x/2))  ->  dy/dx = 0.2505 (1 - tanh^2)
          const float t = (2.0f * out[c] - 1.0f) * (1.0f / 1.002f);
          gp[c] = gin[c] * 0.2505f * (1.0f - t * t);
        } else {
          gp[c] = gin[c] * out[c] * (1.0f - out[c]);
        }
      }
      const float gg[4] = {gv[u].x, gv[u].y, gv[u].z, gv[u].w};
      float ds[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float dg = wr[0][j] * gp[0] + wr[1][j] * gp[1] + wr[2][j] * gp[2];
        // softplus'(s) = sigmoid(s) = 1 - exp(-softplus(s));  ReLU' = [g > 0]
        const float der = a.new_activation ? (1.0f - expf(-gg[j])) : (gg[j] > 0.f ? 1.0f : 0.f);
        ds[j] = dg * der;
#pragma unroll
        for (int c = 0; c < 3; ++c) awr[c][j] = fmaf(gp[c], gg[j], awr[c][j]);
      }
      *reinterpret_cast<float4*>(a.dS + p * 128 + lane * 4) = make_float4(ds[0], ds[1], ds[2], ds[3]);
      const float hv[8] = {h0[u].x, h0[u].y, h0[u].z, h0[u].w, h1[u].x, h1[u].y, h1[u].z, h1[u].w};
#pragma unroll
      for (int j = 0; j < 8; ++j) aws[j] = fmaf(g[u].w, hv[j], aws[j]);
      if (lane == 0) { abr[0] += gp[0]; abr[1] += gp[1]; abr[2] += gp[2]; abs_ += g[u].w; }
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int j = 0; j < 4; ++j) atomicAdd(a.dWr + c * 128 + lane * 4 + j, awr[c][j]);
#pragma unroll
  for (int j = 0; j < 8; ++j) atomicAdd(a.dWs + lane * 8 + j, aws[j]);
  if (lane == 0) {
    atomicAdd(a.dbr + 0, abr[0]); atomicAdd(a.dbr + 1, abr[1]); atomicAdd(a.dbr + 2, abr[2]);
    atomicAdd(a.dbs, abs_);
  }
}

// ------------------------------------------------------------------------------------------
// host: the whole MLP backward of one render pass
// ------------------------------------------------------------------------------------------
// wgrad_tc.cu: dW[:, col_off + k] += dY^T X, db += sum dY on tensor cores (bf16 hi/lo split, fp32 accumulate in
// TMEM); x_pos_bits (nullable) receives [X > 0] for the dgrad of the same layer
int run_wgrad_tc(const float* dY, int N, const float* X, int ldx, int K, float* dW, int ldw, int col_off, float* db,
                 uint32_t* x_pos_bits, long long P, cudaStream_t st);
// dgrad_tc.cu: dX = (dY W[:, col_off:] + extra evec) x [mask_bits] on tensor cores (CTA pairs, W^T resident in
// shared memory)
int run_dgrad_tc(const float* dY, int N, const float* W, int ldw, int col_off, const uint32_t* mask_bits,
                 const float* extra, int extra_stride, const float* evec, float* dX, long long P, cudaStream_t st);

// params / grads: 24 device pointers in state-dict order (SNB_N_PARAM_TENSORS); grads are accumulated into.
// ------------------------------------------------------------------------------------------
// The bottleneck ("xyz_encoding_final", nerf.py:140) has no activation, so the direction layer sees
//   s = Wd[:, :256] (Wf h8 + bf) + Wd[:, 256:] dir + bd = W' h8 + Wd[:, 256:] dir + b',  W' = Wd[:, :256] Wf
// -- the forward kernels use exactly that (field_tc.cu folds W' at pack time), and so does the
// backward: one wgrad against h8 gives dW' (128 x 256) and db' (128), and the chain rule through the
// product is three tiny matrix products that do not depend on the number of points:
//   dWd[:, :256] += dW' Wf^T + db' (x) bf     dWf += Wd[:, :256]^T dW'     dbf += Wd[:, :256]^T db'     dbd += db'
// No per-point bottleneck activations, no P-sized wgrad / dgrad for that layer.
// ------------------------------------------------------------------------------------------
constexpr int kFoldW = 0, kFoldDW = kHalf * kWidth, kFoldDB = 2 * kHalf * kWidth;   // offsets into ws_w (floats)

__global__ void fold_weights_kernel(const float* __restrict__ Wd, const float* __restrict__ Wf, float* __restrict__ ws) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < kHalf * kWidth; e += gridDim.x * blockDim.x) {
    const int n = e / kWidth, k = e - n * kWidth;
    float acc = 0.f;
    for (int j = 0; j < kWidth; ++j) acc = fmaf(Wd[n * 283 + j], Wf[j * kWidth + k], acc);
    ws[kFoldW + e] = acc;
    ws[kFoldDW + e] = 0.f;
    if (e < kHalf) ws[kFoldDB + e] = 0.f;
  }
}

__global__ void unfold_grads_kernel(const float* __restrict__ Wd, const float* __restrict__ Wf, const float* __restrict__ bf,
                                    const float* __restrict__ ws, float* __restrict__ dWd, float* __restrict__ dbd,
                                    float* __restrict__ dWf, float* __restrict__ dbf) {
  const float* dWp = ws + kFoldDW;
  const float* dbp = ws + kFoldDB;
  const int n_a = kHalf * kWidth, n_b = kWidth * kWidth;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n_a + n_b + kWidth + kHalf; e += gridDim.x * blockDim.x) {
    if (e < n_a) {                       // dWd[n][j] += sum_k dW'[n][k] Wf[j][k] + db'[n] bf[j]
      const int n = e / kWidth, j = e - n * kWidth;
      float acc = dbp[n] * bf[j];
      for (int k = 0; k < kWidth; ++k) acc = fmaf(dWp[n * kWidth + k], Wf[j * kWidth + k], acc);
      dWd[n * 283 + j] += acc;
    } else if (e < n_a + n_b) {          // dWf[j][k] += sum_n Wd[n][j] dW'[n][k]
      const int f = e - n_a, j = f / kWidth, k = f - j * kWidth;
      float acc = 0.f;
      for (int n = 0; n < kHalf; ++n) acc = fmaf(Wd[n * 283 + j], dWp[n * kWidth + k], acc);
      dWf[f] += acc;
    } else if (e < n_a + n_b + kWidth) { // dbf[j] += sum_n Wd[n][j] db'[n]
      const int j = e - n_a - n_b;
      float acc = 0.f;
      for (int n = 0; n < kHalf; ++n) acc = fmaf(Wd[n * 283 + j], dbp[n], acc);
      dbf[j] += acc;
    } else {
      const int n = e - n_a - n_b - kWidth;
      dbd[n] += dbp[n];
    }
  }
}

// launch wrappers shared with the 16-bit backward (bwd16.cu)
int launch_fold_weights(const float* Wd, const float* Wf, float* ws, cudaStream_t st) {
  fold_weights_kernel<<<128, 256, 0, st>>>(Wd, Wf, ws);
  return check_launch("fold_weights_kernel");
}
int launch_unfold_grads(const float* Wd, const float* Wf, const float* bf, const float* ws, float* dWd, float* dbd,
                        float* dWf, float* dbf, cudaStream_t st) {
  unfold_grads_kernel<<<392, 256, 0, st>>>(Wd, Wf, bf, ws, dWd, dbd, dWf, dbf);
  return check_launch("unfold_grads_kernel");
}

int field_backward_fp32(const float* const* params, float* const* grads, int new_activation, const float* g_raw,
                        const float* raw, const float* save_enc, const float* save_dir, const float* save_h,
                        const float* save_g, int64_t n_points, float* ws_a, float* ws_b, float* ws_s, float* ws_w,
                        uint32_t* ws_m, cudaStream_t st) {
  const long long P = n_points;
  if (P == 0) return SNB_OK;
  auto H = [&](int l) { return save_h + (size_t)l * P * kWidth; };   // l = 0..7: h1..h8
  int rc;
  // heads
  {
    HeadArgs a{g_raw, raw, save_g, H(7), params[kRgbW], new_activation, ws_s,
               grads[kRgbW], grads[kRgbB], grads[kSigmaW], grads[kSigmaB], P};
    const int grid = sm_count() * 4;
    head_bwd_kernel<<<grid, 256, 0, st>>>(a);
    if ((rc = check_launch("head_bwd_kernel"))) return rc;
  }
  // direction layer with the bottleneck folded in: X = [h8 (through W') | dir]
  if ((rc = launch_fold_weights(params[18], params[16], ws_w, st))) return rc;
  if ((rc = run_wgrad_tc(ws_s, 128, H(7), 256, 256, ws_w + kFoldDW, 256, 0, ws_w + kFoldDB, ws_m, P, st))) return rc;
  if ((rc = run_wgrad_tc(ws_s, 128, save_dir, kDirPad, kDirCh, grads[18], 283, 256, nullptr, nullptr, P, st))) return rc;
  if ((rc = launch_unfold_grads(params[18], params[16], params[17], ws_w, grads[18], grads[19], grads[16], grads[17], st))) return rc;
  // into h8: through W', plus the sigma head's term; ReLU mask of h8
  if ((rc = run_dgrad_tc(ws_s, 128, ws_w + kFoldW, 256, 0, ws_m, g_raw + 3, 4, params[kSigmaW], ws_b, P, st))) return rc;
  // trunk layers 8..2 (index l = 7..1): dY lives in cur, dX goes to nxt
  float* cur = ws_b;
  float* nxt = ws_a;
  for (int l = 7; l >= 1; --l) {
    const int ldw = l == 4 ? 319 : 256;
    if (l == 4) {
      if ((rc = run_wgrad_tc(cur, 256, save_enc, kXyzPad, kXyzCh, grads[2 * l], ldw, 0, grads[2 * l + 1], nullptr, P, st))) return rc;
      if ((rc = run_wgrad_tc(cur, 256, H(l - 1), 256, 256, grads[2 * l], ldw, kXyzCh, nullptr, ws_m, P, st))) return rc;
      if ((rc = run_dgrad_tc(cur, 256, params[2 * l], ldw, kXyzCh, ws_m, nullptr, 0, nullptr, nxt, P, st))) return rc;
    } else {
      if ((rc = run_wgrad_tc(cur, 256, H(l - 1), 256, 256, grads[2 * l], ldw, 0, grads[2 * l + 1], ws_m, P, st))) return rc;
      if ((rc = run_dgrad_tc(cur, 256, params[2 * l], ldw, 0, ws_m, nullptr, 0, nullptr, nxt, P, st))) return rc;
    }
    float* t = cur; cur = nxt; nxt = t;
  }
  // layer 1: weights only
  return run_wgrad_tc(cur, 256, save_enc, kXyzPad, kXyzCh, grads[0], 63, 0, grads[1], nullptr, P, st);
}

}  // namespace snb
