// bwd16.cu -- backward of the field MLP over 16-bit saved activations (act16.cuh): the driver that walks the
// layers, the head kernel, the scale bookkeeping.  Same mathematics as field_bwd.cu (reference: autograd
// through models/nerf.py:105-148, bottleneck folded into the direction layer); the two GEMMs of every layer are
// wgrad16.cu / dgrad16.cu.
//
// Per render pass, given g_raw (P,4) = dL/d[r,g,b,sigma] (fp32, from the compositing backward):
//   prepare   : zero the running maxima, W' = Wd[:, :256] Wf, max column L1 norms of every weight matrix a
//               dgrad multiplies by (the growth bound behind each layer's power-of-two gradient scale)
//   heads     : rgb head + its activation, direction-layer activation -> dS (fp16 T32, scaled), the head-gradient
//               cells hg = [g_pre_rgb(3), g_sigma | their fp16 rounding residuals] (fp16 T32, scaled), db_rgb, db_sigma
//                                                                                                    (head_bwd16_kernel)
//   dir layer : dW', db' = wgrad16(dS, h8) with the sigma-head rows riding on the same X operand (dW_sigma = hg[3]^T h8);
//               dWd[:, 256:] = wgrad16(dS, dir);  dW_rgb = hg[0..2]^T g;  unfold through W'
//   layers    : dH_{l-1} = dgrad16(dH_l, W_l) * mask(h_l);  dW_l, db_l = wgrad16(dH_l, h_l)          l = 8 .. 1
// HBM per point: ~2.5 KB per 256-wide layer (fp32 version: ~5 KB), 4.5 KB of saved activations (8.9 KB).
#include <cuda_fp16.h>

#include "act16.cuh"
#include "common.cuh"

namespace snb {

// field_bwd.cu
int launch_fold_weights(const float* Wd, const float* Wf, float* ws, cudaStream_t st);
int launch_unfold_grads(const float* Wd, const float* Wf, const float* bf, const float* ws, float* dWd, float* dbd,
                        float* dWf, float* dbf, cudaStream_t st);
// wgrad16.cu / dgrad16.cu
int run_wgrad16(const void* dY, int FA, const void* X, int FB, int K, float* dW, int ldw, int col_off, float* db,
                const float* scale, const void* hg, float* const* dH, const float* scale2, long long n_points_pad,
                cudaStream_t st);
int run_dgrad16(const void* dY, const void* dY_lo, int N, const float* W, int ldw, int col_off, const uint32_t* mask,
                const float* extra, int extra_stride, const float* evec, void* dX, void* dX_lo, float* state, int st_amax_in,
                int st_scale_in, int st_l1, int st_amax_out, int st_scale_out, long long P, cudaStream_t st);

namespace {

constexpr int kFoldW = 0, kFoldDW = kHalf * kWidth, kFoldDB = 2 * kHalf * kWidth;   // offsets into the fold scratch (floats)

// ------------------------------------------------------------------------------------------
// max |g_raw| when the compositing backward did not provide it (stand-alone use of the C ABI)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) amax_kernel(const float4* __restrict__ g, long long n, uint32_t* __restrict__ out) {
  float m = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = g[i];
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_uint(m == m ? fminf(m, 3.0e38f) : 3.0e38f));
}

// ------------------------------------------------------------------------------------------
// prepare: block b computes one of the bound ingredients.  Blocks 0..7: max column L1 norm of the matrix the
// dgrad of "stage b" multiplies by (b = 0: W' from the fold scratch; b = l: W_l[:, col_off : col_off + 256], l = 1..7);
// block 8: max |w_sigma| and max_j sum_c |W_rgb[c][j]|; also takes over an externally computed max |g_raw|.
// ------------------------------------------------------------------------------------------
struct PrepArgs {
  const float* W[8]; int rows[8]; int ldw[8]; int col_off[8];
  const float* w_sigma; const float* w_rgb;
  const uint32_t* g_amax;      // nullable
  float* state;
};
__global__ void __launch_bounds__(256) bwd16_prepare_kernel(PrepArgs a) {
  __shared__ float red[8];
  const int b = blockIdx.x, tid = threadIdx.x;
  float v = 0.f;
  if (b < 8) {
    const float* W = a.W[b];
    for (int n = 0; n < a.rows[b]; ++n) v += fabsf(W[(size_t)n * a.ldw[b] + a.col_off[b] + tid]);   // column tid
  } else {
    v = fabsf(a.w_sigma[tid]);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, off));
  if ((tid & 31) == 0) red[tid >> 5] = v;
  __syncthreads();
  if (tid == 0) {
    float m = 0.f;
    for (int i = 0; i < 8; ++i) m = fmaxf(m, red[i]);
    if (b == 0) a.state[ST_L1_FOLD] = m;
    else if (b < 8) a.state[ST_L1_L0 + b] = m;
    else {
      a.state[ST_EVEC_MAX] = m;
      float wr = 0.f;
      for (int j = 0; j < kHalf; ++j) wr = fmaxf(wr, fabsf(a.w_rgb[j]) + fabsf(a.w_rgb[kHalf + j]) + fabsf(a.w_rgb[2 * kHalf + j]));
      a.state[ST_WR_L1] = wr;
      if (a.g_amax != nullptr) reinterpret_cast<uint32_t*>(a.state)[ST_AMAX_G] = *a.g_amax;
    }
  }
}

// ------------------------------------------------------------------------------------------
// heads: a warp walks 32-point tiles, lane = point.  Reads g_raw / raw (float4 per point, coalesced) and the 16
// cells of the direction layer's output g; writes the 16 cells of dS and the head-gradient cell.
//   g_pre_rgb_c = g_rgb_c * act_rgb'(out_c);   dS_j = (sum_c W_rgb[c][j] g_pre_rgb_c) * act_dir'(g_j)
// ------------------------------------------------------------------------------------------
struct Head16Args {
  const float4* g_raw;       // (P,)
  const float4* raw;         // (P,) forward output [rgb (post-activation), sigma]
  const unsigned char* G;    // (Ppad,128) fp16 T32
  const float* Wr;           // (3,128)
  int new_activation;
  unsigned char* dS;         // (Ppad,128) fp16 T32, scaled by state[ST_SCALE_DS]
  unsigned char* dS_lo;      // residual plane (nullable)
  unsigned char* hg;         // (Ppad,8) fp16 T32, scaled by state[ST_SCALE_HG]
  float* dbr; float* dbs;
  float* state;
  long long P, ppad;
};

__global__ void __launch_bounds__(256) head_bwd16_kernel(Head16Args a) {
  __shared__ float4 wr[kHalf];       // [j] = (Wr[0][j], Wr[1][j], Wr[2][j], 0)
  const int tid = threadIdx.x, lane = tid & 31;
  for (int j = tid; j < kHalf; j += blockDim.x) wr[j] = make_float4(a.Wr[j], a.Wr[kHalf + j], a.Wr[2 * kHalf + j], 0.f);
  __syncthreads();
  // scales: |hg| <= max |g_raw| (activation derivatives <= 0.2505 / 1);  |dS_j| <= 0.2505 max_j sum_c |Wr[c][j]| max |g_raw|
  const float amax_g = __uint_as_float(reinterpret_cast<const uint32_t*>(a.state)[ST_AMAX_G]);
  const float s_hg = pow2_scale(amax_g, kA16Target);
  const float s_ds = pow2_scale(0.2505f * a.state[ST_WR_L1] * amax_g, kA16Target);
  if (blockIdx.x == 0 && tid == 0) { a.state[ST_SCALE_HG] = s_hg; a.state[ST_SCALE_DS] = s_ds; }
  const long long warp = ((long long)blockIdx.x * blockDim.x + tid) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  float abr0 = 0.f, abr1 = 0.f, abr2 = 0.f, abs_ = 0.f, amax = 0.f;
  for (long long tile = warp; tile * 32 < a.ppad; tile += nwarps) {
    const long long p = tile * 32 + lane;
    const bool live = p < a.P;
    float gp[3] = {0.f, 0.f, 0.f}, gs = 0.f;
    if (live) {
      const float4 g = a.g_raw[p], o = a.raw[p];
      const float gin[3] = {g.x, g.y, g.z}, out[3] = {o.x, o.y, o.z};
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
      gs = g.w;
      abr0 += gp[0]; abr1 += gp[1]; abr2 += gp[2]; abs_ += gs;
    }
    {
      // head-gradient cell: features 0..3 = fp16 hi of [g_pre_rgb(3), g_sigma] * s_hg, features 4..7 = the rounding
      // residuals (the cell has the room): the head rows of wgrad16 add rows r and r + 4, i.e. 22-bit head gradients
      const float hv[4] = {gp[0] * s_hg, gp[1] * s_hg, gp[2] * s_hg, gs * s_hg};
      const uint32_t h01 = pack_half2_sat(hv[0], hv[1]), h23 = pack_half2_sat(hv[2], hv[3]);
      const float2 f01 = __half22float2(*reinterpret_cast<const __half2*>(&h01)), f23 = __half22float2(*reinterpret_cast<const __half2*>(&h23));
      *reinterpret_cast<uint4*>(a.hg + a16_cell(p, 0, 8)) =
          make_uint4(h01, h23, pack_half2_sat(hv[0] - f01.x, hv[1] - f01.y), pack_half2_sat(hv[2] - f23.x, hv[3] - f23.y));
    }
#pragma unroll 4
    for (int f8 = 0; f8 < 16; ++f8) {
      const uint4 c = live ? __ldg(reinterpret_cast<const uint4*>(a.G + a16_cell(p, f8, kHalf))) : make_uint4(0u, 0u, 0u, 0u);
      const uint32_t w[4] = {c.x, c.y, c.z, c.w};
      uint32_t o[4], ol[4];
#pragma unroll
      for (int j2 = 0; j2 < 4; ++j2) {
        const float2 gg = __half22float2(*reinterpret_cast<const __half2*>(&w[j2]));
        const float gv[2] = {gg.x, gg.y};
        float ds[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const float4 wj = wr[f8 * 8 + 2 * j2 + e];
          const float dg = wj.x * gp[0] + wj.y * gp[1] + wj.z * gp[2];
          // softplus'(s) = sigmoid(s) = 1 - exp(-softplus(s));  ReLU' = [g > 0]
          const float der = a.new_activation ? (1.0f - __expf(-gv[e])) : (gv[e] > 0.f ? 1.0f : 0.f);
          ds[e] = dg * der * s_ds;
          amax = fmaxf(amax, fabsf(ds[e]));
        }
        o[j2] = pack_half2_sat(ds[0], ds[1]);
        const float2 hv = __half22float2(*reinterpret_cast<const __half2*>(&o[j2]));
        ol[j2] = pack_half2_sat(ds[0] - hv.x, ds[1] - hv.y);
      }
      *reinterpret_cast<uint4*>(a.dS + a16_cell(p, f8, kHalf)) = make_uint4(o[0], o[1], o[2], o[3]);
      if (a.dS_lo != nullptr) *reinterpret_cast<uint4*>(a.dS_lo + a16_cell(p, f8, kHalf)) = make_uint4(ol[0], ol[1], ol[2], ol[3]);
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    abr0 += __shfl_xor_sync(0xffffffffu, abr0, off); abr1 += __shfl_xor_sync(0xffffffffu, abr1, off);
    abr2 += __shfl_xor_sync(0xffffffffu, abr2, off); abs_ += __shfl_xor_sync(0xffffffffu, abs_, off);
    amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, off));
  }
  if (lane == 0) {
    atomicAdd(a.dbr + 0, abr0); atomicAdd(a.dbr + 1, abr1); atomicAdd(a.dbr + 2, abr2);
    atomicAdd(a.dbs, abs_);
    if (amax > 0.f)
      atomicMax(reinterpret_cast<uint32_t*>(a.state) + ST_AMAX_DS, __float_as_uint(amax == amax ? fminf(amax, 65504.f) : 65504.f));
  }
}

}  // namespace

size_t act16_bytes(long long n_points) { return make_act16_layout(n_points).total; }
size_t bwd16_workspace_bytes(long long n_points) { return make_bwd16_layout(n_points).total; }

int field_backward16(const float* const* params, float* const* grads, int new_activation, const float* g_raw,
                     const float* raw, const void* act16, long long P, void* ws, const float* g_amax, cudaStream_t st) {
  if (P == 0) return SNB_OK;
  const long long ppad = a16_pad(P);
  const Act16Layout A = make_act16_layout(P);
  const Bwd16Layout B = make_bwd16_layout(P);
  const unsigned char* act = reinterpret_cast<const unsigned char*>(act16);
  unsigned char* w = reinterpret_cast<unsigned char*>(ws);
  float* fold = reinterpret_cast<float*>(w + B.fold);
  float* state = reinterpret_cast<float*>(w + B.state);
  const uint32_t* mask = reinterpret_cast<const uint32_t*>(act + A.mask);
  auto H = [&](int l) { return act + A.h[l]; };                          // l = 0..7: h1..h8
  auto M = [&](int l) { return mask + (size_t)l * 8 * (size_t)ppad; };   // ReLU mask of h_{l+1}
  // The gradient chain carries its fp16 rounding residual (a second plane) from dS down to dH_4; below that the
  // chain is hi-only: a weight gradient then sees at most 4 chained 11-bit roundings (measured <= 4e-4 rel-L2, parity
  // bar 1e-3) and the four lowest hops move 1 KB per point instead of 2.  DESIGN.md section 4.3 lists the measured
  // alternatives.
  constexpr int lo_floor = 4;                      // dH_l has a residual plane for l >= lo_floor
  int rc;
  if (cudaMemsetAsync(state, 0, kBwdStateFloats * sizeof(float), st) != cudaSuccess)
    return fail(SNB_ERR_CUDA, "field_backward16: cudaMemsetAsync failed");
  if (g_amax == nullptr) {
    amax_kernel<<<sm_count() * 4, 256, 0, st>>>(reinterpret_cast<const float4*>(g_raw), P, reinterpret_cast<uint32_t*>(state) + ST_AMAX_G);
    if ((rc = check_launch("amax_kernel"))) return rc;
  }
  if ((rc = launch_fold_weights(params[18], params[16], fold, st))) return rc;
  {
    PrepArgs a{};
    a.W[0] = fold + kFoldW; a.rows[0] = kHalf; a.ldw[0] = kWidth; a.col_off[0] = 0;
    for (int l = 1; l < 8; ++l) {
      a.W[l] = params[2 * l]; a.rows[l] = kWidth; a.ldw[l] = l == 4 ? 319 : 256; a.col_off[l] = l == 4 ? kXyzCh : 0;
    }
    a.w_sigma = params[kSigmaW]; a.w_rgb = params[kRgbW];
    a.g_amax = reinterpret_cast<const uint32_t*>(g_amax);
    a.state = state;
    bwd16_prepare_kernel<<<9, 256, 0, st>>>(a);
    if ((rc = check_launch("bwd16_prepare_kernel"))) return rc;
  }
  {
    Head16Args a{reinterpret_cast<const float4*>(g_raw), reinterpret_cast<const float4*>(raw), act + A.g, params[kRgbW],
                 new_activation, w + B.ds, w + B.ds_lo, w + B.hg, grads[kRgbB], grads[kSigmaB], state, P, ppad};
    long long tiles = ppad / 32, blocks = (tiles + 7) / 8;
    if (blocks > sm_count() * 4) blocks = sm_count() * 4;
    head_bwd16_kernel<<<(unsigned)blocks, 256, 0, st>>>(a);
    if ((rc = check_launch("head_bwd16_kernel"))) return rc;
  }
  const float* sc_ds = state + ST_SCALE_DS;
  const float* sc_hg = state + ST_SCALE_HG;
  // direction layer (bottleneck folded in): X = [h8 (through W') | dir]; the sigma head's weights ride on the h8 pass
  {
    float* dH[8] = {nullptr, nullptr, nullptr, grads[kSigmaW], nullptr, nullptr, nullptr, nullptr};
    if ((rc = run_wgrad16(w + B.ds, 128, H(7), 256, 256, fold + kFoldDW, 256, 0, fold + kFoldDB, sc_ds, w + B.hg, dH, sc_hg, ppad, st)))
      return rc;
  }
  if ((rc = run_wgrad16(w + B.ds, 128, act + A.dir, kDirPad, kDirCh, grads[18], 283, 256, nullptr, sc_ds, nullptr, nullptr, nullptr, ppad, st)))
    return rc;
  {
    float* dH[8] = {grads[kRgbW], grads[kRgbW] + kHalf, grads[kRgbW] + 2 * kHalf, nullptr, nullptr, nullptr, nullptr, nullptr};
    if ((rc = run_wgrad16(nullptr, 0, act + A.g, 128, 128, nullptr, 0, 0, nullptr, sc_ds, w + B.hg, dH, sc_hg, ppad, st))) return rc;
  }
  if ((rc = launch_unfold_grads(params[18], params[16], params[17], fold, grads[18], grads[19], grads[16], grads[17], st))) return rc;
  // into h8: through W', plus the sigma head's term; ReLU mask of h8
  unsigned char* cur = w + B.dya;
  unsigned char* nxt = w + B.dyb;
  unsigned char* cur_lo = w + B.dya_lo;
  unsigned char* nxt_lo = w + B.dyb_lo;
  if ((rc = run_dgrad16(w + B.ds, w + B.ds_lo, 128, fold + kFoldW, 256, 0, M(7), g_raw + 3, 4, params[kSigmaW], cur,
                        cur_lo, state, ST_AMAX_DS, ST_SCALE_DS, ST_L1_FOLD, ST_AMAX_H0 + 7, ST_SCALE_H0 + 7, P, st)))
    return rc;
  for (int l = 7; l >= 1; --l) {
    const int ldw = l == 4 ? 319 : 256;
    const float* sc = state + ST_SCALE_H0 + l;
    if (l == 4) {
      if ((rc = run_wgrad16(cur, 256, act + A.enc, kXyzPad, kXyzCh, grads[2 * l], ldw, 0, grads[2 * l + 1], sc, nullptr, nullptr, nullptr, ppad, st))) return rc;
      if ((rc = run_wgrad16(cur, 256, H(l - 1), 256, 256, grads[2 * l], ldw, kXyzCh, nullptr, sc, nullptr, nullptr, nullptr, ppad, st))) return rc;
    } else {
      if ((rc = run_wgrad16(cur, 256, H(l - 1), 256, 256, grads[2 * l], ldw, 0, grads[2 * l + 1], sc, nullptr, nullptr, nullptr, ppad, st))) return rc;
    }
    const bool lo_in = l >= lo_floor, lo_out = l - 1 >= lo_floor;
    if ((rc = run_dgrad16(cur, lo_in ? cur_lo : nullptr, 256, params[2 * l], ldw, l == 4 ? kXyzCh : 0, M(l - 1), nullptr, 0, nullptr,
                          nxt, lo_out ? nxt_lo : nullptr, state, ST_AMAX_H0 + l, ST_SCALE_H0 + l, ST_L1_L0 + l, ST_AMAX_H0 + l - 1,
                          ST_SCALE_H0 + l - 1, P, st)))
      return rc;
    unsigned char* t = cur; cur = nxt; nxt = t;
    t = cur_lo; cur_lo = nxt_lo; nxt_lo = t;
  }
  // layer 1: weights only
  return run_wgrad16(cur, 256, act + A.enc, kXyzPad, kXyzCh, grads[0], 63, 0, grads[1], state + ST_SCALE_H0, nullptr, nullptr, nullptr, ppad, st);
}

}  // namespace snb
