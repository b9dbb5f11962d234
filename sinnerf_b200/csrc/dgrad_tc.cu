// dgrad_tc.cu -- input gradients of one nn.Linear on 5th-gen tensor cores (CTA pairs).
//
//   dX[p][k] = ( sum_n dY[p][n] W[n][col_off + k]  +  extra[p] evec[k] ) * [mask[p][k] > 0]        k < 256
//
// (reference: autograd through models/nerf.py:105-148; the layer walk that calls it is in
// field_bwd.cu.)  dY (P, N) with N = 256 or 128, mask = sign bits of the saved post-ReLU input of
// the layer (32 B per point, emitted by the wgrad kernel that reads that input anyway), extra/evec =
// the sigma head's rank-1 term at h8.  dY and dX are plain row-major fp32.
//
// Mapping (the forward field kernel's, with HBM as the producer of A):
//   * a CTA pair owns 256 points; tcgen05.mma.cta_group::2, M = 256, N = 128 per instruction, so the
//     256 outputs are two halves a | b with their own TMEM accumulators: the epilogue of a runs
//     under the MMAs of b, the epilogue of b under the next tile's a;
//   * W^T (bf16 hi + lo, K-major canonical layout) is converted ONCE per CTA and stays resident
//     in shared memory (128 KB: each CTA of the pair holds 64 of a half's 128 rows) -- no weight
//     streaming at all;
//   * the A operand lives in TMEM as bf16 hi | lo planes; eight converter warps (two per lane
//     quadrant) read their point's dY row from HBM 32 columns at a time, split and tcgen05.st it.  Quarters form a ring with the MMA issuer: quarter q of the next tile is
//     refilled as soon as this tile's half b has consumed it, so HBM loads stay in flight while
//     the tensor pipe works;
//   * bf16 3-product split (hi*hi + lo*hi + hi*lo), fp32 accumulate: gradients need fp32's range.
//
// HBM per point and layer: dY 4N + 32 B of mask in, dX 1 KB out (2 KB at N = 256): the kernel is
// HBM-bound (~0.08 us per 256-point tile at 6.5 TB/s against 6144 tensor cycles); see DESIGN.md.
#include <cuda_bf16.h>

#include "common.cuh"
#include "umma.cuh"

namespace snb {
using namespace umma;

namespace {

constexpr int kDgTile = 128;                 // points per CTA (MMA M = 256 across the pair)
constexpr int kDgConvWarps = 8, kDgEpiWarps = 4;      // converters: two warps per TMEM lane quadrant
constexpr int kDgMmaWarp = kDgConvWarps + kDgEpiWarps;
constexpr int kDgThreads = (kDgMmaWarp + 1) * 32;
constexpr uint32_t kDgColD = 0, kDgColAhi = 256, kDgColAlo = 384;

struct DgradTcArgs {
  const float* dY;                 // (P, NRED)
  const float* W; int ldw; int col_off;   // nn.Linear weight (NRED, ldw); inputs [col_off, col_off + 256)
  const uint32_t* mask_bits;       // (P,8) nullable: bit c of word w = [input[p][32 w + c] > 0] (wgrad_tc emits it)
  const float* extra; int extra_stride;   // nullable per-point scalar
  const float* evec;               // (256), with extra
  float* dX;                       // (P,256)
  long long P;
};

template <int NRED>
struct DgSmem {
  // W^T planes: [half a|b][hi|lo][k8 = n / 8][64 rows = this CTA's in-features of the half][8 n]
  static constexpr int kPlaneBytes = (NRED / 8) * 64 * 16;
  alignas(1024) unsigned char b[2][2][kPlaneBytes];
  alignas(16) float evec[256];
  // per-warp 32 x 32 transposition tiles (row stride 36 words: conflict-free 128-bit accesses both ways).
  // HBM is read and written with rows-of-128-bytes per quarter warp (4 lines per instruction); the
  // thread = point-row view TMEM wants is produced here, not by 32-lines-per-instruction global accesses.
  alignas(16) float cstage[kDgConvWarps][32][36];
  alignas(16) float estage[kDgEpiWarps][32][36];
  uint64_t q_ready[4], q_free[4], d_full[2], d_drained[2];
  uint32_t tmem_base;
};

__device__ __forceinline__ void bf16_split_pair(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  const float b0 = __uint_as_float(hi << 16), b1 = __uint_as_float(hi & 0xffff0000u);
  const __nv_bfloat162 l = __floats2bfloat162_rn(x0 - b0, x1 - b1);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

template <int NRED>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kDgThreads, 1) dgrad_tc_kernel(DgradTcArgs a) {
  using S = DgSmem<NRED>;
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
      bf16_split_pair(w0, w1, h[j], l[j]);
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
  auto tile_of = [&](long long slot) { return (pair + slot * n_pairs) * 2 + rank; };
  // hand-offs to the MMA issuer, which lives in the leader CTA
  auto signal = [&](uint64_t* bar) { if (!leader) mbar_arrive_remote(bar, 0); else mbar_arrive(bar); };

  if (warp == kDgMmaWarp) {
    // ======================= MMA issuer (leader CTA, one elected lane) =======================
    if (leader && elect_one()) {
      const uint32_t idesc = make_idesc(kFmtBF16, 2 * kDgTile, 128);
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
              const uint32_t a_hi = tbase + kDgColAhi + ks * 8, a_lo = tbase + kDgColAlo + ks * 8;
              mma2_ts_lohi(d, a_hi, bh + ks * kStepB, b_hi32, idesc, ks > 0 ? 1u : 0u);
              mma2_ts_lohi(d, a_lo, bh + ks * kStepB, b_hi32, idesc, 1u);
              mma2_ts_lohi(d, a_hi, bl + ks * kStepB, b_hi32, idesc, 1u);
            }
            if (h == 1) mma2_commit(&s.q_free[q]);      // both halves have consumed A quarter q
          }
          mma2_commit(&s.d_full[h]);
        }
      }
    }
    __syncwarp();
  } else if (warp < kDgConvWarps) {
    // ======================= converters: dY rows (HBM) -> bf16 hi | lo planes of A (TMEM) ========
    // A unit = 32 columns of one point row (128 B).  The two warps of a quadrant take the two
    // halves of every K quarter; the next unit's loads are issued before the current one is split
    // and stored, so every thread keeps 128-256 B in flight (HBM latency ~1.3k cycles).
    const int quad = warp & 3, sub = warp >> 2;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const long long n_units = n_slots * kQ;
    // lane l of a load/store instruction handles 16 bytes of row (l >> 3) + 4 i, chunk l & 7
    const int rib0 = lane >> 3, chunk = lane & 7;
    auto load_unit = [&](long long u, float4 (&v)[8]) {
      const long long slot = u / kQ;
      const int q = (int)(u - slot * kQ);
      const long long pt0 = tile_of(slot) * kDgTile + quad * 32;      // first row of this warp's block
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const long long pt = pt0 + rib0 + 4 * i;
        v[i] = (u < n_units && pt < a.P)
                   ? __ldg(reinterpret_cast<const float4*>(a.dY + pt * NRED + q * 64 + sub * 32) + chunk)
                   : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    auto store_unit = [&](long long u, const float4 (&v)[8]) {
      const long long slot = u / kQ;
      const int q = (int)(u - slot * kQ);
      float (*st)[36] = s.cstage[warp];
      __syncwarp();                                   // the previous unit's row reads are done
#pragma unroll
      for (int i = 0; i < 8; ++i) *reinterpret_cast<float4*>(&st[rib0 + 4 * i][chunk * 4]) = v[i];
      __syncwarp();
      uint32_t hi[16], lo[16];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 x = *reinterpret_cast<const float4*>(&st[lane][j * 4]);     // this thread's point row
        bf16_split_pair(x.x, x.y, hi[2 * j], lo[2 * j]);
        bf16_split_pair(x.z, x.w, hi[2 * j + 1], lo[2 * j + 1]);
      }
      if (slot > 0) { mbar_wait(&s.q_free[q], (uint32_t)(slot - 1) & 1); tc_fence_after(); }
      tmem_st16(tbase + lane_base + kDgColAhi + q * 32 + sub * 16, hi);
      tmem_st16(tbase + lane_base + kDgColAlo + q * 32 + sub * 16, lo);
      tmem_wait_st();
      tc_fence_before();
      signal(&s.q_ready[q]);
    };
    {
      float4 x[8], y[8];
      load_unit(0, x);
      for (long long u = 0; u < n_units; u += 2) {
        load_unit(u + 1, y);
        store_unit(u, x);
        load_unit(u + 2, x);
        if (u + 1 < n_units) store_unit(u + 1, y);
      }
    }
  } else {
    // ======================= epilogue: D (TMEM) -> (+ sigma term) * mask -> dX (HBM) ===========
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const int rib0 = lane >> 3, chunk = lane & 7;
    float (*st)[36] = s.estage[warp - kDgConvWarps];
    for (long long slot = 0; slot < n_slots; ++slot) {
      const long long pt0 = tile_of(slot) * kDgTile + quad * 32;
      const long long pt = pt0 + lane;
      const bool live = pt < a.P;
      const float ex = (live && a.extra != nullptr) ? a.extra[pt * a.extra_stride] : 0.f;
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        uint4 mb = make_uint4(~0u, ~0u, ~0u, ~0u);
        if (live && a.mask_bits != nullptr) mb = __ldg(reinterpret_cast<const uint4*>(a.mask_bits + pt * 8) + h);
        const uint32_t mw[4] = {mb.x, mb.y, mb.z, mb.w};
        mbar_wait(&s.d_full[h], (uint32_t)slot & 1);
        tc_fence_after();
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const int c0 = h * 128 + g * 32;
          uint32_t v[32];
          tmem_ld32(tbase + lane_base + kDgColD + c0, v);
          tmem_wait_ld();
          if (g == 3) { tc_fence_before(); signal(&s.d_drained[h]); }   // half h is in registers
          __syncwarp();                                   // the previous group's tile has been written out
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 e = *reinterpret_cast<const float4*>(s.evec + c0 + 4 * j);
            float4 o;
            o.x = (mw[g] >> (4 * j)) & 1u ? fmaf(ex, e.x, __uint_as_float(v[4 * j])) : 0.f;
            o.y = (mw[g] >> (4 * j + 1)) & 1u ? fmaf(ex, e.y, __uint_as_float(v[4 * j + 1])) : 0.f;
            o.z = (mw[g] >> (4 * j + 2)) & 1u ? fmaf(ex, e.z, __uint_as_float(v[4 * j + 2])) : 0.f;
            o.w = (mw[g] >> (4 * j + 3)) & 1u ? fmaf(ex, e.w, __uint_as_float(v[4 * j + 3])) : 0.f;
            *reinterpret_cast<float4*>(&st[lane][j * 4]) = o;
          }
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const long long pr = pt0 + rib0 + 4 * i;
            if (pr < a.P)
              *(reinterpret_cast<float4*>(a.dX + pr * 256 + c0) + chunk) = *reinterpret_cast<const float4*>(&st[rib0 + 4 * i][chunk * 4]);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();     // neither CTA leaves (or frees TMEM) while its peer may still touch it
  if (warp == kDgMmaWarp) tmem_dealloc_pair(tbase);
}

template <int NRED>
int launch_dgrad_tc(const DgradTcArgs& a, cudaStream_t st) {
  static SmemOptIn optin;
  const int smem = (int)sizeof(DgSmem<NRED>) + 1024;
  if (int rc = ensure_smem(dgrad_tc_kernel<NRED>, optin, smem, "dgrad_tc")) return rc;
  const int sms = sm_count();
  const long long ntiles = (a.P + kDgTile - 1) / kDgTile;
  long long pairs = (ntiles + 1) / 2;
  if (pairs > sms / 2) pairs = sms / 2;
  dgrad_tc_kernel<NRED><<<(unsigned)(2 * pairs), kDgThreads, smem, st>>>(a);
  return check_launch("dgrad_tc_kernel");
}

}  // namespace

// run_dgrad (field_bwd.cu) on tensor cores; the ReLU mask arrives as the bit matrix run_wgrad_tc emitted
int run_dgrad_tc(const float* dY, int N, const float* W, int ldw, int col_off, const uint32_t* mask_bits,
                 const float* extra, int extra_stride, const float* evec, float* dX, long long P, cudaStream_t st) {
  if (P == 0) return SNB_OK;
  DgradTcArgs a{dY, W, ldw, col_off, mask_bits, extra, extra_stride, evec, dX, P};
  if (N == 256) return launch_dgrad_tc<256>(a, st);
  if (N == 128) return launch_dgrad_tc<128>(a, st);
  return fail(SNB_ERR_INVALID, "run_dgrad_tc: unsupported reduction length %d", N);
}

}  // namespace snb
