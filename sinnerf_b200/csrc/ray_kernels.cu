// ray_kernels.cu -- the HBM-bound per-ray stages of render_rays as warp-level kernels:
//   sample_coarse   models/rendering.py:264-282   (stratified depths)
//   embed           models/nerf.py:24-41          (stand-alone Embedding.forward)
//   composite_fwd   models/rendering.py:215-248   (sigma -> alpha -> transmittance -> rgb/depth)
//   sample_pdf      models/rendering.py:15-61     (inverse-CDF sampling)
//   importance_merge models/rendering.py:310-315  (z_mid + sample_pdf + sorted union)
// Mapping: one warp per ray, samples strided over lanes, shuffles for the scans.
// All of these are bound by HBM traffic; algorithmic bytes are listed per kernel.
#include "common.cuh"

namespace snb {

constexpr unsigned kFull = 0xffffffffu;

// ---------------------------------------------------------------------------------------
// sample_coarse: 32 B/ray in, 4*S B/ray out (+4*S in for perturb_u)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float z_at(float near, float far, float t, int use_disp) {
  // near*(1-t) + far*t with every product and sum rounded separately, as torch evaluates it
  const float omt = __fsub_rn(1.0f, t);
  if (!use_disp) return __fadd_rn(__fmul_rn(near, omt), __fmul_rn(far, t));
  const float a = __fmul_rn(__fdiv_rn(1.0f, near), omt);
  const float b = __fmul_rn(__fdiv_rn(1.0f, far), t);
  return __fdiv_rn(1.0f, __fadd_rn(a, b));
}

__global__ void sample_coarse_kernel(const float* __restrict__ rays, const float* __restrict__ z_steps,
                                     const float* __restrict__ perturb_u, float perturb, int use_disp,
                                     long long n_rays, int S, float* __restrict__ z_out) {
  const long long total = n_rays * S;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    const long long ray = e / S;
    const int i = (int)(e - ray * S);
    const float near = rays[ray * 8 + 6], far = rays[ray * 8 + 7];
    float z = z_at(near, far, z_steps[i], use_disp);
    if (perturb > 0.f) {
      // rendering.py:274-282: lower=[z0, mid...], upper=[mid..., z_last]
      const float zl = i > 0 ? z_at(near, far, z_steps[i - 1], use_disp) : z;
      const float zr = i < S - 1 ? z_at(near, far, z_steps[i + 1], use_disp) : z;
      const float lower = i > 0 ? __fmul_rn(0.5f, __fadd_rn(zl, z)) : z;
      const float upper = i < S - 1 ? __fmul_rn(0.5f, __fadd_rn(z, zr)) : z;
      const float pr = __fmul_rn(perturb, perturb_u[e]);
      z = __fadd_rn(lower, __fmul_rn(__fsub_rn(upper, lower), pr));
    }
    z_out[e] = z;
  }
}

// ---------------------------------------------------------------------------------------
// generate_rays (SURVEY.md 8f-1): rays of a pinhole camera straight into the (N,8) layout, replacing
//   get_ray_directions        datasets/ray_utils.py:73-91   d = [(i-W/2)/f, -(j-H/2)/f, -1]
//   get_ray_directions_dtu    datasets/dtu_proj.py:17-34    d = [(i-cx)/fx, (j-cy)/fy, 1]
//   get_rays                  datasets/ray_utils.py:94-120  d_world = d @ c2w[:, :3].T, o = c2w[:, 3]
//   + torch.cat([o, d, near, far])                          datasets/llff.py style assembly
// for a strided window of the pixel grid (the ray patches of *_ray_patch_* datasets).
// 0 B in, 32 B/ray out.
// ---------------------------------------------------------------------------------------
struct RayGenArgs {
  float c2w[12];     // row-major (3,4)
  float fx, fy, cx, cy;
  float near, far;
  int opencv;        // 0: blender/LLFF convention (-y up, -z forward), 1: DTU / OpenCV (+z forward)
  int row0, col0, rows, cols, stride;
  float* rays;
};
__global__ void generate_rays_kernel(RayGenArgs a) {
  const long long n = (long long)a.rows * a.cols;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(e / a.cols), c = (int)(e - (long long)r * a.cols);
    const float i = (float)(a.col0 + c * a.stride), j = (float)(a.row0 + r * a.stride);
    float dx, dy, dz;
    if (a.opencv) { dx = __fdiv_rn(i - a.cx, a.fx); dy = __fdiv_rn(j - a.cy, a.fy); dz = 1.0f; }
    else { dx = __fdiv_rn(i - a.cx, a.fx); dy = -__fdiv_rn(j - a.cy, a.fy); dz = -1.0f; }
    float4 lo, hi;
    lo.x = a.c2w[3]; lo.y = a.c2w[7]; lo.z = a.c2w[11];
    lo.w = fmaf(dz, a.c2w[2], fmaf(dy, a.c2w[1], dx * a.c2w[0]));
    hi.x = fmaf(dz, a.c2w[6], fmaf(dy, a.c2w[5], dx * a.c2w[4]));
    hi.y = fmaf(dz, a.c2w[10], fmaf(dy, a.c2w[9], dx * a.c2w[8]));
    hi.z = a.near; hi.w = a.far;
    reinterpret_cast<float4*>(a.rays)[2 * e] = lo;
    reinterpret_cast<float4*>(a.rays)[2 * e + 1] = hi;
  }
}

// ---------------------------------------------------------------------------------------
// embed: 4*C B in, 4*C*(2L+1) B out per row (264 B/point for C=3, L=10).
// A block computes 128 rows into smem (one sincosf per (row, freq, channel)), then streams
// the dense [128][C*(2L+1)] tile out with 128-bit stores.
// ---------------------------------------------------------------------------------------
constexpr int kEmbedRows = 128;
__global__ void __launch_bounds__(256) embed_kernel(const float* __restrict__ x, long long n, int C, int L,
                                                    float* __restrict__ out) {
  extern __shared__ float tile[];  // [kEmbedRows][W]
  const int W = C * (2 * L + 1);
  const long long nblocks = (n + kEmbedRows - 1) / kEmbedRows;
  for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
    const long long r0 = blk * kEmbedRows;
    const int rows = (int)((n - r0) < kEmbedRows ? (n - r0) : kEmbedRows);
    const int items = rows * C * (L + 1);
    for (int it = threadIdx.x; it < items; it += blockDim.x) {
      const int r = it / (C * (L + 1));
      const int rem = it - r * (C * (L + 1));
      const int f = rem / C, c = rem - f * C;  // f == 0: identity block; f >= 1: frequency f-1
      const float v = x[(r0 + r) * C + c];
      if (f == 0) {
        tile[r * W + c] = v;
      } else {
        float sn, cs;
        sincosf(v * (float)(1 << (f - 1)), &sn, &cs);
        tile[r * W + C + (f - 1) * 2 * C + c] = sn;
        tile[r * W + C + (f - 1) * 2 * C + C + c] = cs;
      }
    }
    __syncthreads();
    const long long base = r0 * W;  // float offset; 128*W*4 B per block keeps 16-B alignment
    const int nflt = rows * W;
    if ((base & 3) == 0) {
      const int nvec = nflt >> 2;
      float4* o4 = reinterpret_cast<float4*>(out + base);
      const float4* t4 = reinterpret_cast<const float4*>(tile);
      for (int v = threadIdx.x; v < nvec; v += blockDim.x) o4[v] = t4[v];
      for (int v = (nvec << 2) + threadIdx.x; v < nflt; v += blockDim.x) out[base + v] = tile[v];
    } else {
      for (int v = threadIdx.x; v < nflt; v += blockDim.x) out[base + v] = tile[v];
    }
    __syncthreads();
  }
}

// C == 3 with a compile-time number of frequencies (the two embeddings SinNeRF uses): no integer
// divisions, one sincosf per (row, frequency, coordinate).
template <int L>
__global__ void __launch_bounds__(256) embed3_kernel(const float* __restrict__ x, long long n, float* __restrict__ out) {
  constexpr int W = 3 * (2 * L + 1);
  __shared__ __align__(16) float tile[kEmbedRows * W];
  const long long nblocks = (n + kEmbedRows - 1) / kEmbedRows;
  for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
    const long long r0 = blk * kEmbedRows;
    const int rows = (int)((n - r0) < kEmbedRows ? (n - r0) : kEmbedRows);
    // item = (frequency slot f in 0..L, row r): thread handles one row's three coordinates at slot f
    for (int it = threadIdx.x; it < (L + 1) * kEmbedRows; it += 256) {
      const int f = it >> 7, r = it & (kEmbedRows - 1);
      if (r >= rows) continue;
      const float vx = x[(r0 + r) * 3], vy = x[(r0 + r) * 3 + 1], vz = x[(r0 + r) * 3 + 2];
      float* t = tile + r * W;
      if (f == 0) {
        t[0] = vx; t[1] = vy; t[2] = vz;
      } else {
        const float sc = (float)(1 << (f - 1));
        float s0, c0, s1, c1, s2, c2;
        sincosf(vx * sc, &s0, &c0); sincosf(vy * sc, &s1, &c1); sincosf(vz * sc, &s2, &c2);
        float* o = t + 3 + (f - 1) * 6;
        o[0] = s0; o[1] = s1; o[2] = s2; o[3] = c0; o[4] = c1; o[5] = c2;
      }
    }
    __syncthreads();
    const long long base = r0 * W;          // kEmbedRows * W * 4 B per block keeps 16-byte alignment
    const int nflt = rows * W, nvec = nflt >> 2;
    float4* o4 = reinterpret_cast<float4*>(out + base);
    const float4* t4 = reinterpret_cast<const float4*>(tile);
    for (int v = threadIdx.x; v < nvec; v += 256) o4[v] = t4[v];
    for (int v = (nvec << 2) + threadIdx.x; v < nflt; v += 256) out[base + v] = tile[v];
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------
// composite_fwd: read 16 B (rgb sigma) + 4 B (z) [+4 B noise] per point, write 4 B (w) per
// point, + 32 B in (ray) and 16 B out (rgb, depth) per ray  ->  24 B/point + 48 B/ray.
// One warp per ray; 32 samples per step; inclusive product scan by shuffles, carried across
// steps; the exclusive product is the scan shifted by one lane.
// ---------------------------------------------------------------------------------------
// Per-ray training losses folded into the compositing (SURVEY.md 8f-3; reference losses.py:12-22 MSELoss,
// models/sinnerf.py:32-42 SL1Loss, consumed at models/sinnerf.py:310-319):
//   loss[0] = sum_ray wr[ray] * sum_c (rgb_c - target_rgb_c)^2      (wr = 1 / (3 N) gives nn.MSELoss 'mean')
//   loss[1] = sum_ray wd[ray] * smooth_l1(depth - target_depth)     (wd = 1 / N gives nn.SmoothL1Loss 'mean', beta 1)
// Reduction: warp partials -> block partial (fixed order) -> ws; the last block to finish adds the block
// partials in index order, so the value is deterministic for a given grid.
struct LossSpec {
  const float* trgb;     // (N,3) nullable
  const float* tdepth;   // (N,)  nullable
  const float* wr;       // (N,) nullable -> wr0
  const float* wd;       // (N,) nullable -> wd0
  float wr0, wd0;
};
// [r, g, b, depth] rows of the rays into frame buffers that may live on other GPUs (include/sinnerf_b200.h: SnbPixelScatter)
struct PixelScatter {
  float4* dst[SNB_MAX_PIXEL_DST];
  int n;
  long long off;
};
__device__ __forceinline__ void scatter_pixel(const PixelScatter& ps, long long ray, float r, float g, float b, float d) {
  const float4 px = make_float4(r, g, b, d);
  for (int i = 0; i < ps.n; ++i) ps.dst[i][ps.off + ray] = px;   // plain stores: P2P-mapped or multicast addresses
}
__device__ __forceinline__ float smooth_l1(float x) { const float a = fabsf(x); return a < 1.0f ? 0.5f * x * x : a - 0.5f; }
__device__ __forceinline__ float smooth_l1_grad(float x) { return fabsf(x) < 1.0f ? x : (x > 0.f ? 1.0f : -1.0f); }

__global__ void __launch_bounds__(256) composite_fwd_kernel(
    const float* __restrict__ raw, int raw_channels, const float* __restrict__ z_vals,
    const float* __restrict__ rays, const float* __restrict__ noise, float noise_std, int white_back,
    long long n_rays, int S, float* __restrict__ rgb_out, float* __restrict__ depth_out,
    float* __restrict__ w_out, LossSpec ls, float* __restrict__ loss_out, float* __restrict__ loss_ws, PixelScatter ps) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  float loss_rgb = 0.f, loss_depth = 0.f;      // lane 0: this warp's share of the two loss sums
  for (long long ray = warp; ray < n_rays; ray += nwarps) {
    const float dx = rays[ray * 8 + 3], dy = rays[ray * 8 + 4], dz = rays[ray * 8 + 5];
    const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);  // torch.norm(dir_, dim=-1)
    const float* zr = z_vals + ray * S;
    float carry = 1.0f;  // product of (1 - alpha + 1e-10) over all earlier samples
    float ar = 0.f, ag = 0.f, ab = 0.f, ad = 0.f, aw = 0.f;
    for (int base = 0; base < S; base += 32) {
      const int i = base + lane;
      const bool valid = i < S;
      float sigma = 0.f, cr = 0.f, cg = 0.f, cb = 0.f, z = 0.f, delta = 0.f;
      if (valid) {
        if (raw_channels == 4) {
          const float4 v = reinterpret_cast<const float4*>(raw)[ray * S + i];
          cr = v.x; cg = v.y; cb = v.z; sigma = v.w;
        } else {
          sigma = raw[ray * S + i];
        }
        z = zr[i];
        delta = (i + 1 < S) ? __fsub_rn(zr[i + 1], z) : 1e10f;
        delta = __fmul_rn(delta, dnorm);
        if (noise != nullptr) sigma = __fadd_rn(sigma, __fmul_rn(noise[ray * S + i], noise_std));
      }
      // alpha = 1 - exp(-delta * relu(sigma))
      const float alpha = valid ? __fsub_rn(1.0f, expf(-__fmul_rn(delta, fmaxf(sigma, 0.f)))) : 0.f;
      const float t = valid ? __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f) : 1.0f;
      float scan = t;  // inclusive product scan over the 32 lanes
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const float up = __shfl_up_sync(kFull, scan, off);
        if (lane >= off) scan *= up;
      }
      float excl = __shfl_up_sync(kFull, scan, 1);
      if (lane == 0) excl = 1.0f;
      const float T = carry * excl;
      const float w = alpha * T;
      carry *= __shfl_sync(kFull, scan, 31);
      if (valid) {
        w_out[ray * S + i] = w;
        ar = fmaf(w, cr, ar); ag = fmaf(w, cg, ag); ab = fmaf(w, cb, ab);
        ad = fmaf(w, z, ad);
        aw += w;
      }
    }
    if (rgb_out != nullptr || depth_out != nullptr) {
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        ar += __shfl_xor_sync(kFull, ar, off);
        ag += __shfl_xor_sync(kFull, ag, off);
        ab += __shfl_xor_sync(kFull, ab, off);
        ad += __shfl_xor_sync(kFull, ad, off);
        aw += __shfl_xor_sync(kFull, aw, off);
      }
      if (lane == 0) {
        if (rgb_out != nullptr) {
          if (white_back) {  // rgb + 1 - weights_sum  (rendering.py:245-246)
            ar = __fsub_rn(__fadd_rn(ar, 1.0f), aw);
            ag = __fsub_rn(__fadd_rn(ag, 1.0f), aw);
            ab = __fsub_rn(__fadd_rn(ab, 1.0f), aw);
          }
          rgb_out[ray * 3 + 0] = ar; rgb_out[ray * 3 + 1] = ag; rgb_out[ray * 3 + 2] = ab;
          if (ls.trgb != nullptr) {
            const float e0 = ar - ls.trgb[ray * 3], e1 = ag - ls.trgb[ray * 3 + 1], e2 = ab - ls.trgb[ray * 3 + 2];
            loss_rgb = fmaf(ls.wr != nullptr ? ls.wr[ray] : ls.wr0, e0 * e0 + e1 * e1 + e2 * e2, loss_rgb);
          }
        }
        if (depth_out != nullptr) {
          depth_out[ray] = ad;
          if (ls.tdepth != nullptr)
            loss_depth = fmaf(ls.wd != nullptr ? ls.wd[ray] : ls.wd0, smooth_l1(ad - ls.tdepth[ray]), loss_depth);
        }
        if (ps.n > 0) scatter_pixel(ps, ray, ar, ag, ab, ad);
      }
    }
  }
  if (loss_out != nullptr) {
    __shared__ float part[8][2];
    __shared__ bool last;
    if (lane == 0) { part[threadIdx.x >> 5][0] = loss_rgb; part[threadIdx.x >> 5][1] = loss_depth; }
    __syncthreads();
    unsigned int* ticket = reinterpret_cast<unsigned int*>(loss_ws);
    float* partials = loss_ws + 4;
    if (threadIdx.x == 0) {
      float a = 0.f, b = 0.f;
      for (int i = 0; i < 8; ++i) { a += part[i][0]; b += part[i][1]; }
      partials[2 * blockIdx.x] = a; partials[2 * blockIdx.x + 1] = b;
      __threadfence();
      last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last && threadIdx.x < 32) {
      __threadfence();
      // fixed-order sum: lane l adds blocks l, l+32, ...; then a fixed shuffle tree
      float a = 0.f, b = 0.f;
      for (unsigned int i = lane; i < gridDim.x; i += 32) {
        a += __ldcg(partials + 2 * i); b += __ldcg(partials + 2 * i + 1);
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) { a += __shfl_xor_sync(kFull, a, off); b += __shfl_xor_sync(kFull, b, off); }
      if (lane == 0) { loss_out[0] = a; loss_out[1] = b; *ticket = 0u; }
    }
  }
}

// ---------------------------------------------------------------------------------------
// composite_bwd: closed-form backward of the compositing (SURVEY.md 8a-7; checked against
// autograd through the oracle in tests/test_gpu_backward.py).  One warp per ray; alpha, T, w are
// recomputed from sigma and z (nothing saved by the forward), the suffix sum
// sum_{k>i} gw_k w_k is a reverse warp scan.
//   gw_i     = g_rgb . c_i + g_depth z_i + g_w_i - [white_back] sum_c g_rgb_c
//   galpha_i = gw_i T_i - (sum_{k>i} gw_k w_k) / (1 - alpha_i + 1e-10)
//   gsigma_i = galpha_i delta_i exp(-delta_i relu(s_i)) [s_i > 0],   s_i = sigma_i + noise_i
//   gc_i     = g_rgb w_i
// Algorithmic bytes: 16+4(+4) in, 16 out per point (+4 if g_w is given).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) composite_bwd_kernel(
    const float* __restrict__ raw, const float* __restrict__ z_vals, const float* __restrict__ rays,
    const float* __restrict__ noise, float noise_std, int white_back, const float* __restrict__ g_rgb,
    const float* __restrict__ g_depth, const float* __restrict__ g_w, long long n_rays, int S,
    float* __restrict__ g_raw, LossSpec ls, const float* __restrict__ out_rgb, const float* __restrict__ out_depth,
    const float* __restrict__ g_loss, unsigned int* __restrict__ g_amax) {
  extern __shared__ float sm[];   // per warp: alpha[S], T[S], gwv[S] (= gw_i * w_i, then its suffix sums)
  float amax = 0.f;               // max |g_raw| written by this thread (for the 16-bit backward's scaling)
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  float* sa = sm + (size_t)wib * 3 * S;
  float* sT = sa + S;
  float* sg = sT + S;
  const long long warp = (long long)blockIdx.x * (blockDim.x >> 5) + wib;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long ray = warp; ray < n_rays; ray += nwarps) {
    const float dx = rays[ray * 8 + 3], dy = rays[ray * 8 + 4], dz = rays[ray * 8 + 5];
    const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
    const float* zr = z_vals + ray * S;
    float gr = 0.f, gg = 0.f, gb = 0.f, gd = 0.f;
    if (g_rgb != nullptr) { gr = g_rgb[ray * 3]; gg = g_rgb[ray * 3 + 1]; gb = g_rgb[ray * 3 + 2]; }
    if (g_depth != nullptr) gd = g_depth[ray];
    // fused losses: d loss[0] / d rgb_c = 2 wr (rgb_c - t_c), d loss[1] / d depth = wd smooth_l1'(depth - t)
    if (ls.trgb != nullptr) {
      const float k = 2.0f * (ls.wr != nullptr ? ls.wr[ray] : ls.wr0) * (g_loss != nullptr ? g_loss[0] : 1.0f);
      gr = fmaf(k, out_rgb[ray * 3] - ls.trgb[ray * 3], gr);
      gg = fmaf(k, out_rgb[ray * 3 + 1] - ls.trgb[ray * 3 + 1], gg);
      gb = fmaf(k, out_rgb[ray * 3 + 2] - ls.trgb[ray * 3 + 2], gb);
    }
    if (ls.tdepth != nullptr) {
      const float k = (ls.wd != nullptr ? ls.wd[ray] : ls.wd0) * (g_loss != nullptr ? g_loss[1] : 1.0f);
      gd = fmaf(k, smooth_l1_grad(out_depth[ray] - ls.tdepth[ray]), gd);
    }
    const float gwb = white_back ? (gr + gg + gb) : 0.f;
    // forward recompute + gw_i w_i
    float carry = 1.0f;
    for (int base = 0; base < S; base += 32) {
      const int i = base + lane;
      const bool valid = i < S;
      float alpha = 0.f, t = 1.0f, gw = 0.f;
      if (valid) {
        const float4 v = reinterpret_cast<const float4*>(raw)[ray * S + i];
        const float z = zr[i];
        float delta = (i + 1 < S) ? __fsub_rn(zr[i + 1], z) : 1e10f;
        delta = __fmul_rn(delta, dnorm);
        float sgm = v.w;
        if (noise != nullptr) sgm = __fadd_rn(sgm, __fmul_rn(noise[ray * S + i], noise_std));
        alpha = __fsub_rn(1.0f, expf(-__fmul_rn(delta, fmaxf(sgm, 0.f))));
        t = __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f);
        gw = gr * v.x + gg * v.y + gb * v.z + gd * z - gwb;
        if (g_w != nullptr) gw += g_w[ray * S + i];
      }
      float scan = t;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const float up = __shfl_up_sync(kFull, scan, off);
        if (lane >= off) scan *= up;
      }
      float excl = __shfl_up_sync(kFull, scan, 1);
      if (lane == 0) excl = 1.0f;
      const float T = carry * excl;
      carry *= __shfl_sync(kFull, scan, 31);
      if (valid) { sa[i] = alpha; sT[i] = T; sg[i] = gw * alpha * T; }
    }
    __syncwarp();
    // exclusive suffix sums of gw_k w_k, walking the 32-sample groups backwards
    float tail = 0.f;
    for (int base = ((S - 1) / 32) * 32; base >= 0; base -= 32) {
      const int i = base + lane;
      const float v = i < S ? sg[i] : 0.f;
      float scan = v;  // inclusive suffix scan inside the group
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const float dn = __shfl_down_sync(kFull, scan, off);
        if (lane + off < 32) scan += dn;
      }
      const float group_total = __shfl_sync(kFull, scan, 0);
      if (i < S) sg[i] = tail + scan - v;   // sum over k > i
      tail += group_total;
    }
    __syncwarp();
    for (int i = lane; i < S; i += 32) {
      const float4 v = reinterpret_cast<const float4*>(raw)[ray * S + i];
      const float z = zr[i];
      float delta = (i + 1 < S) ? __fsub_rn(zr[i + 1], z) : 1e10f;
      delta = __fmul_rn(delta, dnorm);
      float sgm = v.w;
      if (noise != nullptr) sgm = __fadd_rn(sgm, __fmul_rn(noise[ray * S + i], noise_std));
      const float alpha = sa[i], T = sT[i];
      const float w = alpha * T;
      float gw = gr * v.x + gg * v.y + gb * v.z + gd * z - gwb;
      if (g_w != nullptr) gw += g_w[ray * S + i];
      const float galpha = gw * T - sg[i] / (__fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f));
      const float e = expf(-__fmul_rn(delta, fmaxf(sgm, 0.f)));
      const float gsig = sgm > 0.f ? galpha * delta * e : 0.f;
      reinterpret_cast<float4*>(g_raw)[ray * S + i] = make_float4(gr * w, gg * w, gb * w, gsig);
      amax = fmaxf(fmaxf(amax, fabsf(gsig)), fmaxf(fmaxf(fabsf(gr * w), fabsf(gg * w)), fabsf(gb * w)));
    }
    __syncwarp();
  }
  if (g_amax != nullptr) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) amax = fmaxf(amax, __shfl_xor_sync(kFull, amax, off));
    // non-negative floats order like their bit patterns; NaN / inf gradients saturate the statistic
    if (lane == 0 && amax > 0.f) atomicMax(g_amax, __float_as_uint(amax == amax ? fminf(amax, 3.0e38f) : 3.0e38f));
  }
}

// ---------------------------------------------------------------------------------------
// Four-samples-per-thread compositing (round 2): the fast path for S % 4 == 0, S <= 128 (the 64 / 128-sample passes
// of every BASELINE config).  The warp-per-ray kernels above issue ~5.5 instructions per sample and lane (353 warp
// instructions per 64-sample ray, ncu) and are issue-bound at ~2.7 TB/s; here a thread owns FOUR consecutive samples
// -- one 16-byte load each of z / noise / g_w, four of raw, one 16-byte store of the weights (four of g_raw) --
// multiplies its four (1 - alpha) factors serially, and only the per-thread products go through the shuffle scan.
// The S/4 threads of a ray form an aligned group of L = 8, 16 or 32 lanes, 32 / L rays per warp pass, so the scan has
// log2(L) steps per four samples instead of five per sample, and 32 / L times the bytes are in flight per warp.
// Element-wise arithmetic (separately rounded delta, alpha, the 1e-10) is the warp-per-ray kernels'.
// ---------------------------------------------------------------------------------------
struct Quad {                 // what a thread derives for its four samples
  float alpha[4], T[4], e[4], delta[4], sg[4];
};
template <int L>
__device__ __forceinline__ void composite_quad(const float4 zq, const float znext, const bool last, const float dnorm,
                                               const float4 sig, const bool has_noise, const float4 nz,
                                               const float noise_std, const bool act, const int sl, Quad& q) {
  const float zz[5] = {zq.x, zq.y, zq.z, zq.w, znext};
  const float ss[4] = {sig.x, sig.y, sig.z, sig.w};
  const float nn[4] = {nz.x, nz.y, nz.z, nz.w};
  float t[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    float d = (k == 3 && last) ? 1e10f : __fsub_rn(zz[k + 1], zz[k]);
    d = __fmul_rn(d, dnorm);
    float sg = ss[k];
    if (has_noise) sg = __fadd_rn(sg, __fmul_rn(nn[k], noise_std));
    const float e = act ? expf(-__fmul_rn(d, fmaxf(sg, 0.f))) : 1.0f;
    const float a = act ? __fsub_rn(1.0f, e) : 0.f;
    q.delta[k] = d; q.sg[k] = sg; q.e[k] = e; q.alpha[k] = a;
    t[k] = act ? __fadd_rn(__fsub_rn(1.0f, a), 1e-10f) : 1.0f;
  }
  const float p0 = t[0], p1 = p0 * t[1], p2 = p1 * t[2], p3 = p2 * t[3];
  float scan = p3;            // inclusive product scan of the per-thread products over the ray's lane group
#pragma unroll
  for (int off = 1; off < L; off <<= 1) {
    const float up = __shfl_up_sync(kFull, scan, off, L);
    if (sl >= off) scan *= up;
  }
  float excl = __shfl_up_sync(kFull, scan, 1, L);
  if (sl == 0) excl = 1.0f;
  q.T[0] = excl; q.T[1] = excl * p0; q.T[2] = excl * p1; q.T[3] = excl * p2;
}

template <int L>
__global__ void __launch_bounds__(256) composite_fwd4_kernel(
    const float* __restrict__ raw, int raw_channels, const float* __restrict__ z_vals,
    const float* __restrict__ rays, const float* __restrict__ noise, float noise_std, int white_back,
    long long n_rays, int S, float* __restrict__ rgb_out, float* __restrict__ depth_out,
    float* __restrict__ w_out, LossSpec ls, float* __restrict__ loss_out, float* __restrict__ loss_ws, PixelScatter ps) {
  constexpr int kRpw = 32 / L;
  const int lane = threadIdx.x & 31, sl = lane & (L - 1), sub = lane / L;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const long long ngroups = (n_rays + kRpw - 1) / kRpw;
  const int nq = S >> 2;
  const bool last = sl == nq - 1;
  float loss_rgb = 0.f, loss_depth = 0.f;      // lanes with sl == 0: their rays' share of the two loss sums
  for (long long g = warp; g < ngroups; g += nwarps) {
    const long long ray = g * kRpw + sub;
    const bool act = ray < n_rays && sl < nq;
    float4 zq = make_float4(0.f, 0.f, 0.f, 0.f), sig = zq, nz = zq, c[4] = {zq, zq, zq, zq};
    float dnorm = 0.f;
    if (act) {
      const long long p0 = ray * S + 4 * sl;
      zq = *reinterpret_cast<const float4*>(z_vals + p0);
      if (raw_channels == 4) {
#pragma unroll
        for (int k = 0; k < 4; ++k) c[k] = reinterpret_cast<const float4*>(raw)[p0 + k];
        sig = make_float4(c[0].w, c[1].w, c[2].w, c[3].w);
      } else {
        sig = *reinterpret_cast<const float4*>(raw + p0);
      }
      if (noise != nullptr) nz = *reinterpret_cast<const float4*>(noise + p0);
      const float dx = rays[ray * 8 + 3], dy = rays[ray * 8 + 4], dz = rays[ray * 8 + 5];
      dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
    }
    const float znext = __shfl_down_sync(kFull, zq.x, 1);
    Quad q;
    composite_quad<L>(zq, znext, last, dnorm, sig, noise != nullptr, nz, noise_std, act, sl, q);
    const float zz[4] = {zq.x, zq.y, zq.z, zq.w};
    float w[4], ar = 0.f, ag = 0.f, ab = 0.f, ad = 0.f, aw = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      w[k] = q.alpha[k] * q.T[k];
      ar = fmaf(w[k], c[k].x, ar); ag = fmaf(w[k], c[k].y, ag); ab = fmaf(w[k], c[k].z, ab);
      ad = fmaf(w[k], zz[k], ad);
      aw += w[k];
    }
    if (act) *reinterpret_cast<float4*>(w_out + ray * S + 4 * sl) = make_float4(w[0], w[1], w[2], w[3]);
    if (rgb_out != nullptr || depth_out != nullptr) {
#pragma unroll
      for (int off = L / 2; off > 0; off >>= 1) {
        ar += __shfl_xor_sync(kFull, ar, off);
        ag += __shfl_xor_sync(kFull, ag, off);
        ab += __shfl_xor_sync(kFull, ab, off);
        ad += __shfl_xor_sync(kFull, ad, off);
        aw += __shfl_xor_sync(kFull, aw, off);
      }
      if (sl == 0 && ray < n_rays) {
        if (rgb_out != nullptr) {
          if (white_back) {  // rgb + 1 - weights_sum  (rendering.py:245-246)
            ar = __fsub_rn(__fadd_rn(ar, 1.0f), aw);
            ag = __fsub_rn(__fadd_rn(ag, 1.0f), aw);
            ab = __fsub_rn(__fadd_rn(ab, 1.0f), aw);
          }
          rgb_out[ray * 3 + 0] = ar; rgb_out[ray * 3 + 1] = ag; rgb_out[ray * 3 + 2] = ab;
          if (ls.trgb != nullptr) {
            const float e0 = ar - ls.trgb[ray * 3], e1 = ag - ls.trgb[ray * 3 + 1], e2 = ab - ls.trgb[ray * 3 + 2];
            loss_rgb = fmaf(ls.wr != nullptr ? ls.wr[ray] : ls.wr0, e0 * e0 + e1 * e1 + e2 * e2, loss_rgb);
          }
        }
        if (depth_out != nullptr) {
          depth_out[ray] = ad;
          if (ls.tdepth != nullptr)
            loss_depth = fmaf(ls.wd != nullptr ? ls.wd[ray] : ls.wd0, smooth_l1(ad - ls.tdepth[ray]), loss_depth);
        }
        if (ps.n > 0) scatter_pixel(ps, ray, ar, ag, ab, ad);
      }
    }
  }
  if (loss_out != nullptr) {
    // same two-level fixed-order reduction as composite_fwd_kernel; the warp's share first (lanes with sl != 0 hold 0)
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      loss_rgb += __shfl_xor_sync(kFull, loss_rgb, off);
      loss_depth += __shfl_xor_sync(kFull, loss_depth, off);
    }
    __shared__ float part[8][2];
    __shared__ bool last_block;
    if (lane == 0) { part[threadIdx.x >> 5][0] = loss_rgb; part[threadIdx.x >> 5][1] = loss_depth; }
    __syncthreads();
    unsigned int* ticket = reinterpret_cast<unsigned int*>(loss_ws);
    float* partials = loss_ws + 4;
    if (threadIdx.x == 0) {
      float a = 0.f, b = 0.f;
      for (int i = 0; i < 8; ++i) { a += part[i][0]; b += part[i][1]; }
      partials[2 * blockIdx.x] = a; partials[2 * blockIdx.x + 1] = b;
      __threadfence();
      last_block = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last_block && threadIdx.x < 32) {
      __threadfence();
      float a = 0.f, b = 0.f;
      for (unsigned int i = lane; i < gridDim.x; i += 32) {
        a += __ldcg(partials + 2 * i); b += __ldcg(partials + 2 * i + 1);
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) { a += __shfl_xor_sync(kFull, a, off); b += __shfl_xor_sync(kFull, b, off); }
      if (lane == 0) { loss_out[0] = a; loss_out[1] = b; *ticket = 0u; }
    }
  }
}

// Backward in the same mapping: everything of a thread's four samples stays in registers (the warp-per-ray kernel
// parks alpha / T / gw w in shared memory and reads raw twice), the suffix sums sum_{k>i} gw_k w_k are a serial sum
// inside the thread plus a log2(L)-step shuffle scan of the per-thread totals.
template <int L>
__global__ void __launch_bounds__(256) composite_bwd4_kernel(
    const float* __restrict__ raw, const float* __restrict__ z_vals, const float* __restrict__ rays,
    const float* __restrict__ noise, float noise_std, int white_back, const float* __restrict__ g_rgb,
    const float* __restrict__ g_depth, const float* __restrict__ g_w, long long n_rays, int S,
    float* __restrict__ g_raw, LossSpec ls, const float* __restrict__ out_rgb, const float* __restrict__ out_depth,
    const float* __restrict__ g_loss, unsigned int* __restrict__ g_amax) {
  constexpr int kRpw = 32 / L;
  const int lane = threadIdx.x & 31, sl = lane & (L - 1), sub = lane / L;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const long long ngroups = (n_rays + kRpw - 1) / kRpw;
  const int nq = S >> 2;
  const bool last = sl == nq - 1;
  float amax = 0.f;               // max |g_raw| written by this thread (for the 16-bit backward's scaling)
  for (long long g = warp; g < ngroups; g += nwarps) {
    const long long ray = g * kRpw + sub;
    const bool act = ray < n_rays && sl < nq;
    float4 zq = make_float4(0.f, 0.f, 0.f, 0.f), nz = zq, gwq = zq, c[4] = {zq, zq, zq, zq};
    float dnorm = 0.f, gr = 0.f, gg = 0.f, gb = 0.f, gd = 0.f;
    const long long p0 = ray * S + 4 * sl;
    if (act) {
      zq = *reinterpret_cast<const float4*>(z_vals + p0);
#pragma unroll
      for (int k = 0; k < 4; ++k) c[k] = reinterpret_cast<const float4*>(raw)[p0 + k];
      if (noise != nullptr) nz = *reinterpret_cast<const float4*>(noise + p0);
      if (g_w != nullptr) gwq = *reinterpret_cast<const float4*>(g_w + p0);
      const float dx = rays[ray * 8 + 3], dy = rays[ray * 8 + 4], dz = rays[ray * 8 + 5];
      dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
      if (g_rgb != nullptr) { gr = g_rgb[ray * 3]; gg = g_rgb[ray * 3 + 1]; gb = g_rgb[ray * 3 + 2]; }
      if (g_depth != nullptr) gd = g_depth[ray];
      // fused losses: d loss[0] / d rgb_c = 2 wr (rgb_c - t_c), d loss[1] / d depth = wd smooth_l1'(depth - t)
      if (ls.trgb != nullptr) {
        const float k = 2.0f * (ls.wr != nullptr ? ls.wr[ray] : ls.wr0) * (g_loss != nullptr ? g_loss[0] : 1.0f);
        gr = fmaf(k, out_rgb[ray * 3] - ls.trgb[ray * 3], gr);
        gg = fmaf(k, out_rgb[ray * 3 + 1] - ls.trgb[ray * 3 + 1], gg);
        gb = fmaf(k, out_rgb[ray * 3 + 2] - ls.trgb[ray * 3 + 2], gb);
      }
      if (ls.tdepth != nullptr) {
        const float k = (ls.wd != nullptr ? ls.wd[ray] : ls.wd0) * (g_loss != nullptr ? g_loss[1] : 1.0f);
        gd = fmaf(k, smooth_l1_grad(out_depth[ray] - ls.tdepth[ray]), gd);
      }
    }
    const float gwb = white_back ? (gr + gg + gb) : 0.f;
    const float znext = __shfl_down_sync(kFull, zq.x, 1);
    Quad q;
    composite_quad<L>(zq, znext, last, dnorm, make_float4(c[0].w, c[1].w, c[2].w, c[3].w), noise != nullptr, nz,
                      noise_std, act, sl, q);
    const float zz[4] = {zq.x, zq.y, zq.z, zq.w};
    const float gwv[4] = {gwq.x, gwq.y, gwq.z, gwq.w};
    float gw[4], v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      gw[k] = gr * c[k].x + gg * c[k].y + gb * c[k].z + gd * zz[k] - gwb;
      if (g_w != nullptr) gw[k] += gwv[k];
      v[k] = act ? gw[k] * q.alpha[k] * q.T[k] : 0.f;     // gw_k w_k
    }
    // exclusive suffix sums: inside the thread, then over the later threads of the ray
    const float s2 = v[3], s1 = v[3] + v[2], s0 = s1 + v[1], tot = s0 + v[0];
    float scan = tot;
#pragma unroll
    for (int off = 1; off < L; off <<= 1) {
      const float dn = __shfl_down_sync(kFull, scan, off, L);
      if (sl + off < L) scan += dn;
    }
    float tail = __shfl_down_sync(kFull, scan, 1, L);
    if (sl == L - 1) tail = 0.f;
    const float suf[4] = {tail + s0, tail + s1, tail + s2, tail};
    if (act) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float w = q.alpha[k] * q.T[k];
        const float galpha = gw[k] * q.T[k] - suf[k] / (__fadd_rn(__fsub_rn(1.0f, q.alpha[k]), 1e-10f));
        const float gsig = q.sg[k] > 0.f ? galpha * q.delta[k] * q.e[k] : 0.f;
        reinterpret_cast<float4*>(g_raw)[p0 + k] = make_float4(gr * w, gg * w, gb * w, gsig);
        amax = fmaxf(fmaxf(amax, fabsf(gsig)), fmaxf(fmaxf(fabsf(gr * w), fabsf(gg * w)), fabsf(gb * w)));
      }
    }
  }
  if (g_amax != nullptr) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) amax = fmaxf(amax, __shfl_xor_sync(kFull, amax, off));
    // non-negative floats order like their bit patterns; NaN / inf gradients saturate the statistic
    if (lane == 0 && amax > 0.f) atomicMax(g_amax, __float_as_uint(amax == amax ? fminf(amax, 3.0e38f) : 3.0e38f));
  }
}

// ---------------------------------------------------------------------------------------
// inverse-CDF sampling.  One warp per ray; cdf (M+1 floats) and, for the merged variant, the
// S+Ni depths live in the warp's slice of shared memory.
//   sample_pdf:       in 4*(M + M+1) B/ray (+4*Ni u), out 4*Ni B/ray
//   importance_merge: in 8*S B/ray (z, w), out 4*(S+Ni) B/ray
// ---------------------------------------------------------------------------------------
// Build cdf[0..M] in smem from weights w[0..M-1] (row pointer), eps as in rendering.py:29-36.
__device__ __forceinline__ void warp_build_cdf(const float* __restrict__ w, int M, float eps, float* cdf,
                                               int lane) {
  float sum = 0.f;
  for (int i = lane; i < M; i += 32) sum += __fadd_rn(w[i], eps);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(kFull, sum, off);
  float carry = 0.f;
  if (lane == 0) cdf[0] = 0.f;
  for (int base = 0; base < M; base += 32) {
    const int i = base + lane;
    float v = i < M ? __fdiv_rn(__fadd_rn(w[i], eps), sum) : 0.f;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const float up = __shfl_up_sync(kFull, v, off);
      if (lane >= off) v += up;
    }
    if (i < M) cdf[i + 1] = carry + v;
    carry += __shfl_sync(kFull, v, 31);
  }
  __syncwarp();
}

// One inverse-CDF sample.  bin(j) returns bins[j].  rendering.py:46-61.
template <class BinFn>
__device__ __forceinline__ float invert_cdf(const float* cdf, int M, float u, float eps, BinFn bin) {
  // idx = #{ j in [0,M] : cdf[j] <= u }   (searchsorted right=True)
  int lo = 0, hi = M + 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (cdf[mid] <= u) lo = mid + 1; else hi = mid;
  }
  const int below = lo - 1 < 0 ? 0 : lo - 1;
  const int above = lo > M ? M : lo;
  const float c0 = cdf[below], c1 = cdf[above];
  const float b0 = bin(below), b1 = bin(above);
  float denom = __fsub_rn(c1, c0);
  if (denom < eps) denom = 1.0f;
  // bins_g0 + (u - cdf_g0) / denom * (bins_g1 - bins_g0)
  return __fadd_rn(b0, __fmul_rn(__fdiv_rn(__fsub_rn(u, c0), denom), __fsub_rn(b1, b0)));
}

__global__ void __launch_bounds__(128) sample_pdf_kernel(
    const float* __restrict__ bins, long long bins_stride, const float* __restrict__ weights,
    long long w_stride, const float* __restrict__ u, long long u_stride, long long n_rays, int M, int Ni,
    float eps, float* __restrict__ out) {
  extern __shared__ float sm[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  float* cdf = sm + wib * (M + 1);
  const long long warp = (long long)blockIdx.x * (blockDim.x >> 5) + wib;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long ray = warp; ray < n_rays; ray += nwarps) {
    warp_build_cdf(weights + ray * w_stride, M, eps, cdf, lane);
    const float* b = bins + ray * bins_stride;
    for (int j = lane; j < Ni; j += 32) {
      const float uj = u[ray * u_stride + j];
      out[ray * Ni + j] = invert_cdf(cdf, M, uj, eps, [&](int k) { return b[k]; });
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(128) importance_merge_kernel(
    const float* __restrict__ z_coarse, const float* __restrict__ w_coarse, const float* __restrict__ u,
    long long u_stride, long long n_rays, int S, int Ni, float eps, float* __restrict__ z_fine,
    float* __restrict__ z_new_out) {
  extern __shared__ float sm[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int M = S - 2, F = S + Ni;
  const int per_warp = (S - 1) + F;   // cdf (M+1 = S-1) + merged depths
  float* cdf = sm + wib * per_warp;
  float* zs = cdf + (S - 1);
  const long long warp = (long long)blockIdx.x * (blockDim.x >> 5) + wib;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long ray = warp; ray < n_rays; ray += nwarps) {
    const float* zc = z_coarse + ray * S;
    for (int i = lane; i < S; i += 32) zs[i] = zc[i];
    warp_build_cdf(w_coarse + ray * S + 1, M, eps, cdf, lane);  // weights[:, 1:-1]
    for (int j = lane; j < Ni; j += 32) {
      const float uj = u[ray * u_stride + j];
      // bins = z_mid = 0.5*(z[k] + z[k+1])   (rendering.py:310)
      const float zn = invert_cdf(cdf, M, uj, eps,
                                  [&](int k) { return __fmul_rn(0.5f, __fadd_rn(zs[k], zs[k + 1])); });
      zs[S + j] = zn;
      if (z_new_out != nullptr) z_new_out[ray * Ni + j] = zn;
    }
    __syncwarp();
    // sorted union (torch.sort(cat([z, z_new]))).  The coarse depths are sorted whenever near <= far and
    // everything is finite; the new ones are rank-sorted first (random u: any order; det u: already monotone
    // up to an ulp at bin edges).  Then every element's position is its own index plus a binary-search count
    // in the other list (ties: coarse first).  O(Ni^2 + F log F) instead of the O(F^2) all-pairs rank.
    float* zn = zs + S;
    {
      // precondition of the merge: coarse row ascending, no NaN anywhere.  Rays with near > far, or NaN / inf
      // depths (near = 0 with use_disp), take the general path: an all-pairs rank sort of the S + Ni values
      // with torch.sort's order (ascending, NaN last) -- every slot of z_fine is written in either case.
      bool ok = true;
      for (int i = lane; i < F; i += 32) {
        const float v = zs[i];
        if (v != v) ok = false;
        if (i + 1 < S && !(v <= zs[i + 1])) ok = false;
      }
      if (!__all_sync(kFull, ok)) {
        for (int e = lane; e < F; e += 32) {
          const float v = zs[e];
          const bool vn = v != v;
          int r = 0;
          for (int k = 0; k < F; ++k) {
            const float o = zs[k];
            const bool on = o != o;
            const bool less = vn ? !on : (o < v);
            const bool same = vn ? on : (o == v);
            r += less || (same && k < e);
          }
          z_fine[ray * F + r] = v;
        }
        __syncwarp();
        continue;
      }
    }
    // deterministic u (inference): the new depths come out ascending -- nothing to sort (this check replaces the
    // O(Ni^2) rank sort that made the kernel 354 us per 160k-ray frame in round 1)
    bool new_sorted = true;
    for (int j = lane; j + 1 < Ni; j += 32) new_sorted &= zn[j] <= zn[j + 1];
    if (!__all_sync(kFull, new_sorted)) {
      float mine[8];                       // Ni <= 256
      int rk[8];
      int cnt = 0;
      for (int j = lane; j < Ni; j += 32, ++cnt) {
        const float v = zn[j];
        int r = 0;
        for (int k = 0; k < Ni; ++k) { const float o = zn[k]; r += (o < v) || (o == v && k < j); }
        mine[cnt] = v; rk[cnt] = r;
      }
      __syncwarp();
      for (int c = 0; c < cnt; ++c) zn[rk[c]] = mine[c];
      __syncwarp();
    }
    for (int i = lane; i < S; i += 32) {           // coarse element: + #{new < z}
      const float v = zs[i];
      int lo = 0, hi = Ni;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (zn[mid] < v) lo = mid + 1; else hi = mid; }
      z_fine[ray * F + i + lo] = v;
    }
    for (int j = lane; j < Ni; j += 32) {          // new element: + #{coarse <= z}
      const float v = zn[j];
      int lo = 0, hi = S;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (zs[mid] <= v) lo = mid + 1; else hi = mid; }
      z_fine[ray * F + j + lo] = v;
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------
// weight packing (fp32 image)
// ---------------------------------------------------------------------------------------
// ---------------------------------------------------------------------------------------
// params_check: 64-bit position-dependent checksum of the 24 parameter tensors vs the one stored in the
// image header (snb_refresh_weights).  2.4 MB of L2/HBM reads, one launch; the last block to finish
// compares, sets header.dirty and resets the scratch fields.
// ---------------------------------------------------------------------------------------
// Grid: 148 blocks x 1024 threads, four words per thread.  (Round 2 launched 64 x 256 -- 36 words per thread, 29 us
// per model, i.e. 58 us of the 900 us configs[2] patch render, profiles/r02b_timeline_patch_bf16_before.txt; 582 x 256
// blocks took 16 us: two same-address atomics per block serialise at ~13 ns each.)
constexpr int kCheckBlocks = 148, kCheckThreads = 1024;
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
  x ^= x >> 27; x *= 0x94d049bb133111ebull;
  return x ^ (x >> 31);
}
__global__ void __launch_bounds__(kCheckThreads) params_check_kernel(ParamPtrs pp, int precision, int new_activation,
                                                                     PackedHeader* hdr) {
  // flat index g over the concatenated tensors (the position the checksum mixes in): every thread owns g = gid + k T,
  // k = 0..3 -- four INDEPENDENT loads in flight.  (A loop over the 24 tensors with an inner grid-stride loop serialised
  // 24 load latencies per thread: 17 us per model on an idle GPU, 3.8 % of the configs[2] patch render.)
  __shared__ int s_off[SNB_N_PARAM_TENSORS + 1];
  if (threadIdx.x == 0) {
    int o = 0;
    for (int t = 0; t < SNB_N_PARAM_TENSORS; ++t) { s_off[t] = o; o += param_numel(t); }
    s_off[SNB_N_PARAM_TENSORS] = o;
  }
  __syncthreads();
  const int total = s_off[SNB_N_PARAM_TENSORS], stride = gridDim.x * blockDim.x;
  unsigned int w[4];
  int gi[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x + k * stride;
    gi[k] = g < total ? g : -1;
    w[k] = 0u;
    if (g < total) {
      int t = 0;                                   // tensor of element g: branch-free search over the 25 offsets
#pragma unroll
      for (int step = 16; step > 0; step >>= 1)
        if (t + step < SNB_N_PARAM_TENSORS && s_off[t + step] <= g) t += step;
      w[k] = __ldg(reinterpret_cast<const unsigned int*>(pp.p[t]) + (g - s_off[t]));
    }
  }
  unsigned long long h = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (gi[k] >= 0) h += mix64(((unsigned long long)gi[k] << 32) ^ (unsigned long long)w[k] ^ 0x9e3779b97f4a7c15ull);
  for (int g = blockIdx.x * blockDim.x + threadIdx.x + 4 * stride; g < total; g += stride) {   // (grids smaller than total / 4)
    int t = 0;
    for (int step = 16; step > 0; step >>= 1)
      if (t + step < SNB_N_PARAM_TENSORS && s_off[t + step] <= g) t += step;
    h += mix64(((unsigned long long)g << 32) ^ (unsigned long long)__ldg(reinterpret_cast<const unsigned int*>(pp.p[t]) + (g - s_off[t])) ^
               0x9e3779b97f4a7c15ull);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) h += __shfl_xor_sync(kFull, h, off);
  __shared__ unsigned long long part[kCheckThreads / 32];
  __shared__ bool last;
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = h;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long b = 0;
    for (int i = 0; i < kCheckThreads / 32; ++i) b += part[i];
    atomicAdd(&hdr->partial, b);
    __threadfence();
    last = atomicAdd(&hdr->blocks_done, 1u) == gridDim.x - 1;
    if (last) {
      __threadfence();
      const unsigned long long total = atomicAdd(&hdr->partial, 0ull);
      hdr->dirty = (hdr->magic != kMagic || hdr->precision != precision || hdr->new_activation != new_activation ||
                    hdr->checksum != total) ? 1 : 0;
      hdr->checksum = total;
      hdr->partial = 0ull;
      hdr->blocks_done = 0u;
    }
  }
}

int launch_params_check(const ParamPtrs& pp, int precision, int new_activation, void* image, cudaStream_t st) {
  params_check_kernel<<<kCheckBlocks, kCheckThreads, 0, st>>>(pp, precision, new_activation, reinterpret_cast<PackedHeader*>(image));
  return check_launch("params_check_kernel");
}

// only_if_dirty: part of a refresh -- return at once unless the check kernel flagged the image stale
__global__ void pack_fp32_kernel(ParamPtrs pp, int new_activation, unsigned char* image, int only_if_dirty) {
  constexpr Fp32Layout L = make_fp32_layout();
  PackedHeader* hdr = reinterpret_cast<PackedHeader*>(image);
  if (only_if_dirty && !hdr->dirty) return;
  float* W = reinterpret_cast<float*>(image + sizeof(PackedHeader));
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    hdr->magic = kMagic;
    hdr->precision = SNB_PREC_FP32;
    hdr->new_activation = new_activation;
  }
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < L.total; e += gridDim.x * blockDim.x) {
    float v = 0.f;
    if (e < L.b[0]) {
      int l = 0;
      while (l + 1 < kNumGemm && e >= L.w[l + 1]) ++l;
      const int rel = e - L.w[l];
      const int N = gemm_n(l);
      const int k = rel / N, n = rel - k * N;
      const int col = gemm_src_col(l, k);
      const int src_k = l == 0 ? 63 : (l == 4 ? 319 : (l == 9 ? 283 : 256));
      if (col >= 0) v = pp.p[param_weight_index(l)][n * src_k + col];
    } else if (e < L.sigma_w) {
      int l = 0;
      while (l + 1 < kNumGemm && e >= L.b[l + 1]) ++l;
      v = pp.p[param_weight_index(l) + 1][e - L.b[l]];
    } else if (e < L.sigma_b) {
      v = pp.p[kSigmaW][e - L.sigma_w];
    } else if (e < L.rgb_w) {
      v = (e == L.sigma_b) ? pp.p[kSigmaB][0] : 0.f;
    } else if (e < L.rgb_b) {
      v = pp.p[kRgbW][e - L.rgb_w];
    } else {
      v = (e - L.rgb_b < 3) ? pp.p[kRgbB][e - L.rgb_b] : 0.f;
    }
    W[e] = v;
  }
}

// ---------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------
static int grid_for(long long work_items, int per_block, int cap_blocks) {
  long long b = (work_items + per_block - 1) / per_block;
  if (b < 1) b = 1;
  return (int)(b < cap_blocks ? b : cap_blocks);
}
static int device_sms() { return sm_count(); }

int launch_sample_coarse(const float* rays, const float* z_steps, const float* perturb_u, float perturb,
                         int use_disp, int64_t n_rays, int S, float* z, cudaStream_t st) {
  if (n_rays == 0) return SNB_OK;
  const int grid = grid_for(n_rays * S, 256, device_sms() * 8);
  sample_coarse_kernel<<<grid, 256, 0, st>>>(rays, z_steps, perturb_u, perturb, use_disp, n_rays, S, z);
  return check_launch("sample_coarse_kernel");
}

int launch_generate_rays(const float* c2w_host, float fx, float fy, float cx, float cy, float near, float far,
                         int opencv, int row0, int col0, int rows, int cols, int stride, float* rays,
                         cudaStream_t st) {
  RayGenArgs a;
  for (int i = 0; i < 12; ++i) a.c2w[i] = c2w_host[i];
  a.fx = fx; a.fy = fy; a.cx = cx; a.cy = cy; a.near = near; a.far = far; a.opencv = opencv;
  a.row0 = row0; a.col0 = col0; a.rows = rows; a.cols = cols; a.stride = stride; a.rays = rays;
  const long long n = (long long)rows * cols;
  if (n == 0) return SNB_OK;
  generate_rays_kernel<<<grid_for(n, 256, device_sms() * 8), 256, 0, st>>>(a);
  return check_launch("generate_rays_kernel");
}

int launch_embed(const float* x, int64_t n, int C, int L, float* out, cudaStream_t st) {
  if (n == 0) return SNB_OK;
  if (C == 3 && (L == SNB_XYZ_FREQS || L == SNB_DIR_FREQS) && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
    const int grid3 = grid_for(n, kEmbedRows, device_sms() * 6);
    if (L == SNB_XYZ_FREQS) embed3_kernel<SNB_XYZ_FREQS><<<grid3, 256, 0, st>>>(x, n, out);
    else embed3_kernel<SNB_DIR_FREQS><<<grid3, 256, 0, st>>>(x, n, out);
    return check_launch("embed3_kernel");
  }
  const size_t smem = (size_t)kEmbedRows * C * (2 * L + 1) * sizeof(float);
  if (smem > 200 * 1024) return fail(SNB_ERR_UNSUPPORTED, "snb_embed: C*(2L+1) too large for the smem tile");
  static SmemOptIn optin;
  if (smem > 48 * 1024)
    if (int rc = ensure_smem(embed_kernel, optin, (int)smem, "embed")) return rc;
  const int grid = grid_for(n, kEmbedRows, device_sms() * 4);
  embed_kernel<<<grid, 256, smem, st>>>(x, n, C, L, out);
  return check_launch("embed_kernel");
}

// the four-samples-per-thread kernels need rows of whole 16-byte quads: S % 4 == 0 (and at most 32 threads per ray)
// and 16-byte aligned per-sample tensors; everything else takes the warp-per-ray kernels
static bool composite_quad_ok(int S, const void* raw, const void* z, const void* a, const void* b) {
  auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return S >= 4 && S <= 128 && (S & 3) == 0 && al(raw) && al(z) && al(a) && al(b);
}

static LossSpec make_loss_spec(const SnbLossSpec* l) {
  LossSpec ls{};
  if (l != nullptr) {
    ls.trgb = l->target_rgb; ls.tdepth = l->target_depth; ls.wr = l->rgb_weight; ls.wd = l->depth_weight;
    ls.wr0 = l->rgb_weight0; ls.wd0 = l->depth_weight0;
  }
  return ls;
}

int launch_composite(const float* raw, int raw_channels, const float* z, const float* rays, const float* noise,
                     float noise_std, int white_back, int64_t n_rays, int S, float* rgb, float* depth,
                     float* w, const SnbLossSpec* loss, float* loss_out, float* loss_ws, const SnbPixelScatter* scatter,
                     cudaStream_t st) {
  PixelScatter ps{};
  if (scatter != nullptr) {
    ps.n = scatter->n_dst;
    ps.off = scatter->row_offset;
    for (int i = 0; i < ps.n; ++i) ps.dst[i] = reinterpret_cast<float4*>(scatter->dst[i]);
  }
  if (n_rays == 0) {
    if (loss_out != nullptr) return cudaMemsetAsync(loss_out, 0, 2 * sizeof(float), st) == cudaSuccess
                                        ? SNB_OK : fail(SNB_ERR_CUDA, "cudaMemsetAsync(loss)");
    return SNB_OK;
  }
  if (composite_quad_ok(S, raw, z, noise, w)) {
    // four samples per thread: the ray's S/4 threads in a lane group of L = 8 / 16 / 32, 32 / L rays per warp pass
    const int L = S <= 32 ? 8 : (S <= 64 ? 16 : 32);
    int grid = grid_for(n_rays, 8 * (32 / L), device_sms() * 8);
    if (loss_out != nullptr && grid > (SNB_LOSS_WS_FLOATS - 4) / 2) grid = (SNB_LOSS_WS_FLOATS - 4) / 2;
    const LossSpec ls = make_loss_spec(loss);
    if (L == 8) composite_fwd4_kernel<8><<<grid, 256, 0, st>>>(raw, raw_channels, z, rays, noise, noise_std, white_back, n_rays, S, rgb, depth, w, ls, loss_out, loss_ws, ps);
    else if (L == 16) composite_fwd4_kernel<16><<<grid, 256, 0, st>>>(raw, raw_channels, z, rays, noise, noise_std, white_back, n_rays, S, rgb, depth, w, ls, loss_out, loss_ws, ps);
    else composite_fwd4_kernel<32><<<grid, 256, 0, st>>>(raw, raw_channels, z, rays, noise, noise_std, white_back, n_rays, S, rgb, depth, w, ls, loss_out, loss_ws, ps);
    return check_launch("composite_fwd4_kernel");
  }
  int grid = grid_for(n_rays, 8, device_sms() * 8);
  if (loss_out != nullptr && grid > (SNB_LOSS_WS_FLOATS - 4) / 2) grid = (SNB_LOSS_WS_FLOATS - 4) / 2;
  composite_fwd_kernel<<<grid, 256, 0, st>>>(raw, raw_channels, z, rays, noise, noise_std, white_back, n_rays,
                                             S, rgb, depth, w, make_loss_spec(loss), loss_out, loss_ws, ps);
  return check_launch("composite_fwd_kernel");
}

int launch_composite_bwd(const float* raw, const float* z, const float* rays, const float* noise, float noise_std,
                          int white_back, const float* g_rgb, const float* g_depth, const float* g_w, int64_t n_rays,
                          int S, float* g_raw, const SnbLossSpec* loss, const float* out_rgb, const float* out_depth,
                          const float* g_loss, float* g_amax, cudaStream_t st) {
  if (n_rays == 0) return SNB_OK;
  if (composite_quad_ok(S, raw, z, noise, g_w) && (reinterpret_cast<uintptr_t>(g_raw) & 15) == 0) {
    const int L = S <= 32 ? 8 : (S <= 64 ? 16 : 32);
    const int grid = grid_for(n_rays, 8 * (32 / L), device_sms() * 6);
    const LossSpec ls = make_loss_spec(loss);
    unsigned int* am = reinterpret_cast<unsigned int*>(g_amax);
    if (L == 8) composite_bwd4_kernel<8><<<grid, 256, 0, st>>>(raw, z, rays, noise, noise_std, white_back, g_rgb, g_depth, g_w, n_rays, S, g_raw, ls, out_rgb, out_depth, g_loss, am);
    else if (L == 16) composite_bwd4_kernel<16><<<grid, 256, 0, st>>>(raw, z, rays, noise, noise_std, white_back, g_rgb, g_depth, g_w, n_rays, S, g_raw, ls, out_rgb, out_depth, g_loss, am);
    else composite_bwd4_kernel<32><<<grid, 256, 0, st>>>(raw, z, rays, noise, noise_std, white_back, g_rgb, g_depth, g_w, n_rays, S, g_raw, ls, out_rgb, out_depth, g_loss, am);
    return check_launch("composite_bwd4_kernel");
  }
  const size_t smem = (size_t)8 * 3 * S * sizeof(float);
  if (smem > 96 * 1024) return fail(SNB_ERR_UNSUPPORTED, "snb_composite_backward: too many samples per ray (%d)", S);
  static SmemOptIn optin;
  if (smem > 48 * 1024)
    if (int rc = ensure_smem(composite_bwd_kernel, optin, (int)smem, "composite_bwd")) return rc;
  const int grid = grid_for(n_rays, 8, device_sms() * 8);
  composite_bwd_kernel<<<grid, 256, smem, st>>>(raw, z, rays, noise, noise_std, white_back, g_rgb, g_depth, g_w,
                                                n_rays, S, g_raw, make_loss_spec(loss), out_rgb, out_depth, g_loss,
                                                reinterpret_cast<unsigned int*>(g_amax));
  return check_launch("composite_bwd_kernel");
}

int launch_sample_pdf(const float* bins, int64_t bins_stride, const float* weights, int64_t w_stride,
                      const float* u, int64_t u_stride, int64_t n_rays, int M, int Ni, float eps, float* out,
                      cudaStream_t st) {
  if (n_rays == 0) return SNB_OK;
  const size_t smem = (size_t)4 * (M + 1) * sizeof(float);
  if (smem > 48 * 1024) return fail(SNB_ERR_UNSUPPORTED, "snb_sample_pdf: too many bins (%d)", M);
  const int grid = grid_for(n_rays, 4, device_sms() * 16);
  sample_pdf_kernel<<<grid, 128, smem, st>>>(bins, bins_stride, weights, w_stride, u, u_stride, n_rays, M, Ni,
                                             eps, out);
  return check_launch("sample_pdf_kernel");
}

int launch_importance_merge(const float* z_coarse, const float* w_coarse, const float* u, int64_t u_stride,
                            int64_t n_rays, int S, int Ni, float eps, float* z_fine, float* z_new,
                            cudaStream_t st) {
  if (n_rays == 0) return SNB_OK;
  if (Ni > 256) return fail(SNB_ERR_UNSUPPORTED, "snb_importance_merge: N_importance > 256 (%d)", Ni);
  const size_t smem = (size_t)4 * ((S - 1) + (S + Ni)) * sizeof(float);
  if (smem > 48 * 1024) return fail(SNB_ERR_UNSUPPORTED, "snb_importance_merge: S+Ni too large");
  const int grid = grid_for(n_rays, 4, device_sms() * 16);
  importance_merge_kernel<<<grid, 128, smem, st>>>(z_coarse, w_coarse, u, u_stride, n_rays, S, Ni, eps, z_fine,
                                                   z_new);
  return check_launch("importance_merge_kernel");
}

int launch_pack_fp32(const float* const* params, int new_activation, void* image, int only_if_dirty, cudaStream_t st) {
  ParamPtrs pp;
  for (int i = 0; i < SNB_N_PARAM_TENSORS; ++i) pp.p[i] = params[i];
  pack_fp32_kernel<<<device_sms() * 2, 256, 0, st>>>(pp, new_activation, reinterpret_cast<unsigned char*>(image), only_if_dirty);
  return check_launch("pack_fp32_kernel");
}

}  // namespace snb
