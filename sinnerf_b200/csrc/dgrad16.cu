// dgrad16.cu -- input gradients of one nn.Linear from / to 16-bit T32 tensors (act16.cuh), CTA pairs.
//
//   dX[p][k] = ( sum_n dY[p][n] W[n][col_off + k]  +  extra[p] evec[k] ) * [mask[p][k]]        k < 256
//
// (reference: autograd through models/nerf.py:105-148.)  Same mapping as dgrad_tc.cu -- a CTA pair owns 256
// points, tcgen05.mma.cta_group::2 with M = 256 / N = 128, halves a | b with their own accumulators, W^T
// resident in shared memory, A in TMEM refilled by eight loader warps in K quarters -- but the operands are
// already 16-bit in HBM:
//   * dY (Ppad, N) fp16 in the T32 layout, stored as true * s_in: lane = point, an 8-feature cell is 16 bytes,
//     32 lanes = 512 contiguous bytes: the loaders do LDG.128 -> tcgen05.st, no conversion, no transposition;
//   * the gradient CHAIN (dgrad -> dgrad) is carried as fp16 hi + lo planes (22 bits), so rounding does not
//     accumulate over the 8 layers; the wgrad of each layer reads only the hi plane -- its error is ONE fp16
//     rounding of that layer's gradient, whatever the depth (measured: hi-only chains reached 1.1e-3 on the first
//     layer's weights, hi + lo 2e-4; the parity bar is 1e-3).  field_backward16 carries hi + lo down to dH_4 and
//     runs the lower hops hi-only (kLoIn / kLoOut = false);
//   * W^T as fp16 hi + lo; products hi*hi + lo*hi + hi*lo (2 without the lo plane);
//   * the epilogue multiplies by the power-of-two ratio s_out / s_in, adds the sigma head's rank-1 term,
//     applies the ReLU mask (bit words the forward wrote, 32 B per point), rounds to fp16 and writes cells of
//     the output T32 tensor -- 4 x 512 contiguous bytes per warp and 32 columns; it also raises the running
//     max |dX * s_out| that the NEXT layer's scale is derived from.
//   * s_out = the largest power of two with  (max |dY| / s_in) * (max column L1 norm of W) [+ max |extra| max |evec|]
//     * s_out <= 2^14: a rigorous bound, so the fp16 stores cannot overflow; chosen identically by every CTA
//     from three device scalars (no host round trip).
// HBM per point and layer: 4 N + 32 B in, 1 KB out with the lo plane (the fp32 version moved the same bytes but
// spent its warps converting them, and its wgrad read 2 KB where wgrad16 reads 1 KB); 2 N + 32 in, 512 B out without.
#include <cuda_fp16.h>

#include "act16.cuh"

#include "common.cuh"
#include "umma.cuh"

namespace snb {
using namespace umma;

namespace {

constexpr int kDgTile = 128;                 // points per CTA (MMA M = 256 across the pair)
constexpr int kDgConvWarps = 8, kDgEpiWarps = 4;      // loaders: two warps per TMEM lane quadrant
constexpr int kDgMmaWarp = kDgConvWarps + kDgEpiWarps;
constexpr int kDgThreads = (kDgMmaWarp + 1) * 32;
constexpr uint32_t kDgColD = 0, kDgColA = 256, kDgColAlo = 384;

struct Dgrad16Args {
  const unsigned char* dY;         // (Ppad, NRED) fp16 T32, stored as true * state[st_scale_in]
  const unsigned char* dY_lo;      // same shape: fp16(true * s - hi) (kLo)
  const float* W; int ldw; int col_off;   // nn.Linear weight (NRED, ldw); inputs [col_off, col_off + 256)
  const uint32_t* mask;            // (8 words, Ppad) nullable: bit c of word w = [input[p][32 w + c] > 0]
  const float* extra; int extra_stride;   // nullable per-point scalar (true units)
  const float* evec;               // (256), with extra
  unsigned char* dX;               // (Ppad, 256) fp16 T32, stored as true * state[st_scale_out]
  unsigned char* dX_lo;            // residual plane (kLo)
  float* state;                    // Bwd16 state words (act16.cuh)
  int st_amax_in, st_scale_in, st_l1, st_amax_out, st_scale_out;
  long long P, ppad;
};

template <int NRED>
struct Dg16Smem {
  // W^T planes: [half a|b][hi|lo][k8 = n / 8][64 rows = this CTA's in-features of the half][8 n]
  static constexpr int kPlaneBytes = (NRED / 8) * 64 * 16;
  alignas(1024) unsigned char b[2][2][kPlaneBytes];
  alignas(16) float evec[256];
  uint64_t q_ready[4], q_free[4], d_full[2], d_drained[2];
  uint32_t tmem_base;
};

__device__ __forceinline__ void f16_split_pair(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(x0, x1);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  const float2 b = __half22float2(h);
  const __half2 l = __floats2half2_rn(x0 - b.x, x1 - b.y);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

// kLoIn: dY comes with its residual plane (3 products); kLoOut: dX is written with its residual plane
template <int NRED, bool kLoIn, bool kLoOut>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kDgThreads, 1) dgrad16_kernel(Dgrad16Args a) {
  constexpr bool kLo = kLoIn;
  using S = Dg16Smem<NRED>;
  constexpr int kQ = NRED / 64;               // K quarters (64 reduction columns each)
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  S& s = *reinterpret_cast<S*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const long long ntiles = (a.P + kDgTile - 1) / kDgTile;
  const long long n_pairs = gridDim.x / 2, pair = blockIdx.x / 2;
  const long long n_slots = ((ntiles + 1) / 2 + n_pairs - 1) / n_pairs;   // both CTAs run the same count

  // ---------------- one-time setup: barriers, TMEM, resident W^T
  if (tid == 0) {
    for (int q = 0; q < 4; ++q) { mbar_init(&s.q_ready[q], kDgConvWarps * 32 * 2); mbar_init(&s.q_free[q], 1); }
    for (int h = 0; h < 2; ++h) { mbar_init(&s.d_full[h], 1); mbar_init(&s.d_drained[h], kDgEpiWarps * 32 * 2); }
    fence_mbar_init();
  }
  if (warp == kDgMmaWarp) tmem_alloc_pair(&s.tmem_base);
  for (int i = tid; i < 256; i += kDgThreads) s.evec[i] = a.evec != nullptr ? a.evec[i] : 0.f;
  // task = (half, n8 block, row): 8 consecutive reduction rows n of one input column k
  for (int t = tid; t < 2 * (NRED / 8) * 64; t += kDgThreads) {
    const int row = t & 63, n8 = (t >> 6) % (NRED / 8), half = t / (64 * (NRED / 8));
    const int k = half * 128 + (int)rank * 64 + row;
    uint32_t h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float w0 = __ldg(a.W + (size_t)(n8 * 8 + 2 * j) * a.ldw + a.col_off + k);
      const float w1 = __ldg(a.W + (size_t)(n8 * 8 + 2 * j + 1) * a.ldw + a.col_off + k);
      f16_split_pair(w0, w1, h[j], l[j]);
    }
    const int off = n8 * (64 * 16) + row * 16;
    *reinterpret_cast<uint4*>(s.b[half][0] + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(s.b[half][1] + off) = make_uint4(l[0], l[1], l[2], l[3]);
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tbase = s.tmem_base;
  // output scale: every thread of every CTA derives the same power of two from three device scalars
  const float s_in = a.state[a.st_scale_in];
  float bound = __uint_as_float(reinterpret_cast<const uint32_t*>(a.state)[a.st_amax_in]) / s_in * a.state[a.st_l1];
  if (a.extra != nullptr)
    bound += __uint_as_float(reinterpret_cast<const uint32_t*>(a.state)[ST_AMAX_G]) * a.state[ST_EVEC_MAX];
  const float s_out = pow2_scale(bound, kA16Target);
  const float ratio = s_out / s_in;
  if (blockIdx.x == 0 && tid == 0) a.state[a.st_scale_out] = s_out;
  auto tile_of = [&](long long slot) { return (pair + slot * n_pairs) * 2 + rank; };
  // hand-offs to the MMA issuer, which lives in the leader CTA
  auto signal = [&](uint64_t* bar) { if (!leader) mbar_arrive_remote(bar, 0); else mbar_arrive(bar); };

  if (warp == kDgMmaWarp) {
    // ======================= MMA issuer (leader CTA, one elected lane) =======================
    if (leader && elect_one()) {
      const uint32_t idesc = make_idesc(kFmtF16, 2 * kDgTile, 128);
      const uint64_t desc0 = make_smem_desc(0, 64 * 16, 128);
      const uint32_t b_hi32 = (uint32_t)(desc0 >> 32);
      constexpr uint32_t kStepB = (2 * 64 * 16) >> 4;      // one K16 step, in 16-byte units
      for (long long slot = 0; slot < n_slots; ++slot) {
        const uint32_t par = (uint32_t)slot & 1, prev = par ^ 1;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint32_t d = tbase + kDgColD + h * 128;
          const uint32_t bh = (uint32_t)desc0 + (smem_u32(s.b[h][0]) >> 4), bl = (uint32_t)desc0 + (smem_u32(s.b[h][1]) >> 4);
#pragma unroll
          for (int q = 0; q < kQ; ++q) {
            if (h == 0) mbar_wait(&s.q_ready[q], par);
            if (q == 0 && slot > 0) mbar_wait(&s.d_drained[h], prev);
            tc_fence_after();
#pragma unroll
            for (int ks = q * 4; ks < q * 4 + 4; ++ks) {
              const uint32_t a_t = tbase + kDgColA + ks * 8;
              mma2_ts_lohi(d, a_t, bh + ks * kStepB, b_hi32, idesc, ks > 0 ? 1u : 0u);
              if (kLo) mma2_ts_lohi(d, tbase + kDgColAlo + ks * 8, bh + ks * kStepB, b_hi32, idesc, 1u);
              mma2_ts_lohi(d, a_t, bl + ks * kStepB, b_hi32, idesc, 1u);
            }
            if (h == 1) mma2_commit(&s.q_free[q]);      // both halves have consumed A quarter q
          }
          mma2_commit(&s.d_full[h]);
        }
      }
    }
    __syncwarp();
  } else if (warp < kDgConvWarps) {
    // ======================= loaders: dY cells (HBM, fp16 T32) -> A (TMEM) ========
    // A unit = 32 features (4 cells of 16 B) of one point.  The two warps of a quadrant take the two halves of
    // every K quarter; lane = point, so each LDG.128 of the warp covers 512 contiguous bytes.  The next unit's
    // loads are issued before the current one is stored (HBM latency ~1.3k cycles).
    const int quad = warp & 3, sub = warp >> 2;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const long long n_units = n_slots * kQ;
    struct Unit { uint4 h[4]; uint4 l[kLo ? 4 : 1]; };
    auto load_unit = [&](long long u, Unit& v) {
      const long long slot = u / kQ;
      const int q = (int)(u - slot * kQ);
      const long long pt = tile_of(slot) * kDgTile + quad * 32 + lane;
      const bool ok = u < n_units && pt < a.ppad;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const size_t off = a16_cell(pt, q * 8 + sub * 4 + c, NRED);
        v.h[c] = ok ? __ldg(reinterpret_cast<const uint4*>(a.dY + off)) : make_uint4(0u, 0u, 0u, 0u);
        if (kLo) v.l[c] = ok ? __ldg(reinterpret_cast<const uint4*>(a.dY_lo + off)) : make_uint4(0u, 0u, 0u, 0u);
      }
    };
    auto store_unit = [&](long long u, const Unit& v) {
      const long long slot = u / kQ;
      const int q = (int)(u - slot * kQ);
      uint32_t w[16];
#pragma unroll
      for (int c = 0; c < 4; ++c) { w[4 * c] = v.h[c].x; w[4 * c + 1] = v.h[c].y; w[4 * c + 2] = v.h[c].z; w[4 * c + 3] = v.h[c].w; }
      if (slot > 0) { mbar_wait(&s.q_free[q], (uint32_t)(slot - 1) & 1); tc_fence_after(); }
      tmem_st16(tbase + lane_base + kDgColA + q * 32 + sub * 16, w);
      if (kLo) {
#pragma unroll
        for (int c = 0; c < 4; ++c) { w[4 * c] = v.l[c].x; w[4 * c + 1] = v.l[c].y; w[4 * c + 2] = v.l[c].z; w[4 * c + 3] = v.l[c].w; }
        tmem_st16(tbase + lane_base + kDgColAlo + q * 32 + sub * 16, w);
      }
      tmem_wait_st();
      tc_fence_before();
      signal(&s.q_ready[q]);
    };
    {
      Unit x, y, z;
      load_unit(0, x);
      load_unit(1, y);
      for (long long u = 0; u < n_units; u += 3) {      // three units in flight per thread
        load_unit(u + 2, z);
        store_unit(u, x);
        load_unit(u + 3, x);
        if (u + 1 < n_units) store_unit(u + 1, y);
        load_unit(u + 4, y);
        if (u + 2 < n_units) store_unit(u + 2, z);
      }
    }
  } else {
    // ======================= epilogue: D (TMEM) -> scale, (+ sigma term), mask, fp16 -> dX cells (HBM) ===========
    const int quad = warp & 3;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    float amax = 0.f;
    for (long long slot = 0; slot < n_slots; ++slot) {
      const long long pt = tile_of(slot) * kDgTile + quad * 32 + lane;
      const bool live = pt < a.P, inbuf = pt < a.ppad;
      const float ex = (live && a.extra != nullptr) ? a.extra[pt * a.extra_stride] * s_out : 0.f;
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        uint32_t mw[4] = {~0u, ~0u, ~0u, ~0u};
        if (live && a.mask != nullptr) {
#pragma unroll
          for (int g = 0; g < 4; ++g) mw[g] = __ldg(a.mask + (size_t)(h * 4 + g) * (size_t)a.ppad + pt);
        }
        mbar_wait(&s.d_full[h], (uint32_t)slot & 1);
        tc_fence_after();
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const int c0 = h * 128 + g * 32;
          uint32_t v[32];
          tmem_ld32(tbase + lane_base + kDgColD + c0, v);
          tmem_wait_ld();
          if (g == 3) { tc_fence_before(); signal(&s.d_drained[h]); }   // half h is in registers
          uint32_t o[16], ol[kLoOut ? 16 : 1];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float2 e = *reinterpret_cast<const float2*>(s.evec + c0 + 2 * j);
            float x0 = fmaf(ex, e.x, __uint_as_float(v[2 * j]) * ratio);
            float x1 = fmaf(ex, e.y, __uint_as_float(v[2 * j + 1]) * ratio);
            x0 = (mw[g] >> (2 * j)) & 1u ? x0 : 0.f;
            x1 = (mw[g] >> (2 * j + 1)) & 1u ? x1 : 0.f;
            amax = fmaxf(amax, fmaxf(fabsf(x0), fabsf(x1)));
            o[j] = pack_half2_sat(x0, x1);
            if (kLoOut) {
              const float2 hv = __half22float2(*reinterpret_cast<const __half2*>(&o[j]));
              ol[j] = pack_half2_sat(x0 - hv.x, x1 - hv.y);
            }
          }
          if (inbuf) {
#pragma unroll
            for (int c = 0; c < 4; ++c)
              *reinterpret_cast<uint4*>(a.dX + a16_cell(pt, (c0 >> 3) + c, 256)) = make_uint4(o[4 * c], o[4 * c + 1], o[4 * c + 2], o[4 * c + 3]);
            if (kLoOut) {
#pragma unroll
              for (int c = 0; c < 4; ++c)
                *reinterpret_cast<uint4*>(a.dX_lo + a16_cell(pt, (c0 >> 3) + c, 256)) = make_uint4(ol[4 * c], ol[4 * c + 1], ol[4 * c + 2], ol[4 * c + 3]);
            }
          }
        }
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, off));
    if (lane == 0 && amax > 0.f)
      atomicMax(reinterpret_cast<uint32_t*>(a.state) + a.st_amax_out, __float_as_uint(amax == amax ? fminf(amax, 65504.f) : 65504.f));
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();     // neither CTA leaves (or frees TMEM) while its peer may still touch it
  if (warp == kDgMmaWarp) tmem_dealloc_pair(tbase);
}

template <int NRED, bool kLoIn, bool kLoOut>
int launch_dgrad16(const Dgrad16Args& a, cudaStream_t st) {
  static SmemOptIn optin;
  const int smem = (int)sizeof(Dg16Smem<NRED>) + 1024;
  if (int rc = ensure_smem(dgrad16_kernel<NRED, kLoIn, kLoOut>, optin, smem, "dgrad16")) return rc;
  const int sms = sm_count();
  const long long ntiles = (a.P + kDgTile - 1) / kDgTile;
  long long pairs = (ntiles + 1) / 2;
  if (pairs > sms / 2) pairs = sms / 2;
  dgrad16_kernel<NRED, kLoIn, kLoOut><<<(unsigned)(2 * pairs), kDgThreads, smem, st>>>(a);
  return check_launch("dgrad16_kernel");
}

}  // namespace

// dY (Ppad, N) -> dX (Ppad, 256), fp16 T32 hi (+ lo) planes; scales and running maxima live in `state` (act16.cuh).
// dY_lo / dX_lo NULL = that tensor has no residual plane (hi-only).
int run_dgrad16(const void* dY, const void* dY_lo, int N, const float* W, int ldw, int col_off, const uint32_t* mask,
                const float* extra, int extra_stride, const float* evec, void* dX, void* dX_lo, float* state, int st_amax_in,
                int st_scale_in, int st_l1, int st_amax_out, int st_scale_out, long long P, cudaStream_t st) {
  if (P == 0) return SNB_OK;
  Dgrad16Args a{reinterpret_cast<const unsigned char*>(dY), reinterpret_cast<const unsigned char*>(dY_lo), W, ldw, col_off, mask,
                extra, extra_stride, evec, reinterpret_cast<unsigned char*>(dX), reinterpret_cast<unsigned char*>(dX_lo), state,
                st_amax_in, st_scale_in, st_l1, st_amax_out, st_scale_out, P, a16_pad(P)};
  const bool li = dY_lo != nullptr, lo = dX_lo != nullptr;
  if (N == 256) {
    if (li && lo) return launch_dgrad16<256, true, true>(a, st);
    if (li) return launch_dgrad16<256, true, false>(a, st);
    if (!lo) return launch_dgrad16<256, false, false>(a, st);
  }
  if (N == 128 && li && lo) return launch_dgrad16<128, true, true>(a, st);
  if (!li && lo) return fail(SNB_ERR_INVALID, "run_dgrad16: a residual plane cannot be produced from a hi-only input chain");
  return fail(SNB_ERR_INVALID, "run_dgrad16: no kernel for reduction length %d with residual planes in / out = %d / %d", N, li, lo);
}

}  // namespace snb
