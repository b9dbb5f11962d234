// wgrad_tc.cu -- weight gradients of one nn.Linear on 5th-gen tensor cores.
//
//   dW[n][col_off + k] += sum_p dY[p][n] * X[p][k]      db[n] += sum_p dY[p][n]
//
// (reference: autograd of `nn.Linear` inside models/nerf.py:105-148; the layer walk that calls it
// is in field_bwd.cu.)  dY (P, N) and X (P, ldx) are the plain row-major
// fp32 tensors the training forward / the dgrad chain leave in HBM.
//
// As an MMA the reduction runs over POINTS:  D[m = out feature][n' = in feature] += A[m][p] B[n'][p],
// so both operands are needed "points-major" -- the transpose of how they sit in HBM -- and as bf16
// hi + lo planes (gradients span fp32's exponent range; the 3-product split  x*w ~ xh*wh + xl*wh +
// xh*wl  keeps ~16 mantissa bits per operand, the gradient parity bar is 1e-3 per tensor).
//
// A CTA owns a slice of points and ALL out features, so every byte of dY and X is read from HBM
// exactly once (2 KB per point for a 256x256 layer):
//   producer  (1 elected thread)  16 points of dY and of X are two contiguous runs in HBM: two
//             cp.async.bulk copies per batch into a 4-deep raw fp32 ring (mbarrier complete_tx);
//   converters (8 warps)          a thread owns one feature and 8 consecutive points: 8 conflict-free
//             LDS from the raw tile, split, one 16-byte row of the K-major (SWIZZLE_NONE) core-matrix
//             layout for the hi plane and one for the lo plane -- the transpose costs nothing extra;
//             also the bias gradient (column sums) and, for the dgrad that follows, [X > 0] as one
//             32-bit word per point and 32 features (a warp ballot);
//   issuer    (1 elected thread)  tcgen05.mma SS, M = 128 per out-feature block, N = Kpad, K = 16
//             points, 3 products, into TMEM accumulators that live for the whole slice (up to
//             2 x 256 = all 512 columns);
//   epilogue  TMEM -> smem -> coalesced fp32 atomics (split-P reduction across CTAs).
// Roofline: HBM, 4 (N + K) bytes per point; shared-memory traffic (TMA in, LDS, STS, MMA operand
// reads: ~10.5 KB per point) is the second limit, the tensor pipe (3 x 160 cycles per 16 points and
// out-feature block) the third; see DESIGN.md.
#include <cuda_bf16.h>

#include "common.cuh"
#include "umma.cuh"

namespace snb {
using namespace umma;

namespace {

constexpr int kWgBatch = 16;             // points per batch = one MMA K step
constexpr int kWgConvWarps = 8;
constexpr int kWgMmaWarp = kWgConvWarps, kWgLoadWarp = kWgConvWarps + 1;
constexpr int kWgThreads = (kWgConvWarps + 2) * 32;
constexpr int kWgRawStages = 4, kWgPlaneBufs = 2;

// KP: in features padded to an MMA N (256 / 64 / 32); NM: 128-row out-feature blocks (N = 128 NM); LDX: X row length
template <int KP, int NM, int LDX>
struct WgGeo {
  static constexpr int kN = 128 * NM;
  static constexpr int kRawDyBytes = kWgBatch * kN * 4;
  static constexpr int kRawXBytes = kWgBatch * LDX * 4;
  static constexpr int kRawBytes = kRawDyBytes + kRawXBytes;
  static constexpr int kAPlane = 2 * 128 * 16;               // one out-feature block, one of {hi, lo}: [k8 2][128][8]
  static constexpr int kBPlane = 2 * KP * 16;                // one of {hi, lo} of X^T: [k8 2][KP][8]
  static constexpr int kPlanesBytes = 2 * NM * kAPlane + 2 * kBPlane;
  static constexpr int kRingBytes = kWgRawStages * kRawBytes + kWgPlaneBufs * kPlanesBytes;
  static constexpr int kOutLd = KP + 4;
  static constexpr int kOutBytes = 128 * kOutLd * 4;         // epilogue staging (one block at a time), aliases the ring
  static constexpr int kSmemBytes = (kRingBytes > kOutBytes ? kRingBytes : kOutBytes) + 1024;
  static constexpr int kTmemColsRaw = NM * KP;
  static constexpr int kTmemCols = kTmemColsRaw < 32 ? 32 : kTmemColsRaw;
  static_assert((kTmemCols & (kTmemCols - 1)) == 0 && kTmemCols <= 512, "TMEM columns");
  static_assert(kSmemBytes <= 227 * 1024, "shared memory");
};

struct WgradTcArgs {
  const float* dY;                   // (P, N) contiguous rows
  const float* X;                    // (P, LDX) contiguous rows
  int K;                             // valid columns of X (<= KP)
  float* dW; int ldw; int col_off;   // dW (N, ldw): the block lands at columns [col_off, col_off + K)
  float* db;                         // nullable
  uint32_t* x_pos_bits;              // nullable, KP = 256 only: (P, 8) words, bit c of word w = [X[p][32 w + c] > 0]
  long long P;
  long long rows_per_split;          // multiple of kWgBatch
};

// 8 consecutive points of one feature column -> one 16-byte row of the hi plane and of the lo plane
__device__ __forceinline__ void split8_store(const float (&v)[8], unsigned char* hi_dst, unsigned char* lo_dst) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __nv_bfloat162 hh = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
    h[j] = *reinterpret_cast<const uint32_t*>(&hh);
    const float b0 = __uint_as_float(h[j] << 16), b1 = __uint_as_float(h[j] & 0xffff0000u);
    const __nv_bfloat162 ll = __floats2bfloat162_rn(v[2 * j] - b0, v[2 * j + 1] - b1);
    l[j] = *reinterpret_cast<const uint32_t*>(&ll);
  }
  *reinterpret_cast<uint4*>(hi_dst) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4*>(lo_dst) = make_uint4(l[0], l[1], l[2], l[3]);
}

template <int KP, int NM, int LDX>
__global__ void __launch_bounds__(kWgThreads, 1) wgrad_tc_kernel(WgradTcArgs a) {
  using G = WgGeo<KP, NM, LDX>;
  constexpr int kN = G::kN;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* ring = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  unsigned char* planes0 = ring + kWgRawStages * G::kRawBytes;
  __shared__ uint64_t raw_full[kWgRawStages], raw_empty[kWgRawStages], pl_full[kWgPlaneBufs], pl_empty[kWgPlaneBufs], d_full;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long r_begin = (long long)blockIdx.x * a.rows_per_split;
  const long long r_end = r_begin + a.rows_per_split < a.P ? r_begin + a.rows_per_split : a.P;
  const int n_batches = r_end > r_begin ? (int)((r_end - r_begin + kWgBatch - 1) / kWgBatch) : 0;

  if (tid == 0) {
    for (int i = 0; i < kWgRawStages; ++i) { mbar_init(&raw_full[i], 1); mbar_init(&raw_empty[i], kWgConvWarps * 32); }
    for (int i = 0; i < kWgPlaneBufs; ++i) { mbar_init(&pl_full[i], kWgConvWarps * 32); mbar_init(&pl_empty[i], 1); }
    mbar_init(&d_full, 1);
    fence_mbar_init();
  }
  if (warp == kWgMmaWarp) tmem_alloc<G::kTmemCols>(&tmem_base_s);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = tmem_base_s;

  if (warp == kWgLoadWarp) {
    // ======================= producer: HBM -> raw fp32 ring (bulk copies) =======================
    if (elect_one()) {
      for (int bi = 0; bi < n_batches; ++bi) {
        const int rs = bi % kWgRawStages;
        mbar_wait(&raw_empty[rs], ((bi / kWgRawStages) & 1) ^ 1);
        const long long p0 = r_begin + (long long)bi * kWgBatch;
        const uint32_t rows = (uint32_t)(r_end - p0 < kWgBatch ? r_end - p0 : kWgBatch);
        unsigned char* dst = ring + (size_t)rs * G::kRawBytes;
        mbar_arrive_expect_tx(&raw_full[rs], rows * (uint32_t)(kN * 4 + LDX * 4));
        bulk_g2s(dst, a.dY + (size_t)p0 * kN, rows * kN * 4, &raw_full[rs]);
        bulk_g2s(dst + G::kRawDyBytes, a.X + (size_t)p0 * LDX, rows * LDX * 4, &raw_full[rs]);
      }
    }
    __syncwarp();
  } else if (warp == kWgMmaWarp) {
    // ======================= MMA issuer =======================
    if (elect_one()) {
      const uint32_t idesc = make_idesc(kFmtBF16, 128, KP);
      for (int bi = 0; bi < n_batches; ++bi) {
        const int pb = bi % kWgPlaneBufs;
        mbar_wait(&pl_full[pb], (bi / kWgPlaneBufs) & 1);
        tc_fence_after();
        const uint32_t base = smem_u32(planes0 + (size_t)pb * G::kPlanesBytes);
        const uint32_t b_base = base + 2 * NM * G::kAPlane;
        const uint64_t b_hi = make_smem_desc(b_base, KP * 16, 128);
        const uint64_t b_lo = make_smem_desc(b_base + G::kBPlane, KP * 16, 128);
#pragma unroll
        for (int mb = 0; mb < NM; ++mb) {
          const uint64_t a_hi = make_smem_desc(base + mb * G::kAPlane, 128 * 16, 128);
          const uint64_t a_lo = make_smem_desc(base + (NM + mb) * G::kAPlane, 128 * 16, 128);
          const uint32_t d = tbase + mb * KP;
          mma_ss(d, a_hi, b_hi, idesc, bi > 0 ? 1u : 0u);
          mma_ss(d, a_lo, b_hi, idesc, 1u);
          mma_ss(d, a_hi, b_lo, idesc, 1u);
        }
        mma_commit(&pl_empty[pb]);
      }
      mma_commit(&d_full);
    }
    __syncwarp();
  } else {
    // ======================= converters: raw fp32 tile -> bf16 hi | lo planes, points-major =====
    // group = (feature, k8 block): 8 consecutive points of one feature.  dY^T has kN x 2 groups per
    // batch, X^T has KP x 2; group g of a thread = index tid + 256 g -> feature idx % F, k8 idx / F.
    constexpr int kGa = (kN * 2) / 256, kGb = (KP * 2 + 255) / 256;
    float bias_acc[kGa];
#pragma unroll
    for (int g = 0; g < kGa; ++g) bias_acc[g] = 0.f;
    for (int bi = 0; bi < n_batches; ++bi) {
      const int rs = bi % kWgRawStages, pb = bi % kWgPlaneBufs;
      const long long p0 = r_begin + (long long)bi * kWgBatch;
      const int rows = (int)(r_end - p0 < kWgBatch ? r_end - p0 : kWgBatch);
      mbar_wait(&raw_full[rs], (bi / kWgRawStages) & 1);
      const float* raw_dy = reinterpret_cast<const float*>(ring + (size_t)rs * G::kRawBytes);
      const float* raw_x = reinterpret_cast<const float*>(ring + (size_t)rs * G::kRawBytes + G::kRawDyBytes);
      float va[kGa][8], vb[kGb][8];
#pragma unroll
      for (int g = 0; g < kGa; ++g) {
        const int idx = tid + 256 * g, f = idx % kN, j = idx / kN;
#pragma unroll
        for (int r = 0; r < 8; ++r) va[g][r] = (j * 8 + r < rows) ? raw_dy[(j * 8 + r) * kN + f] : 0.f;
      }
#pragma unroll
      for (int g = 0; g < kGb; ++g) {
        const int idx = tid + 256 * g, f = idx % KP, j = idx / KP;
#pragma unroll
        for (int r = 0; r < 8; ++r) vb[g][r] = (j < 2 && j * 8 + r < rows && f < a.K) ? raw_x[(j * 8 + r) * LDX + f] : 0.f;
      }
      mbar_arrive(&raw_empty[rs]);                 // the raw tile is in registers
      mbar_wait(&pl_empty[pb], ((bi / kWgPlaneBufs) & 1) ^ 1);
      unsigned char* pl = planes0 + (size_t)pb * G::kPlanesBytes;
#pragma unroll
      for (int g = 0; g < kGa; ++g) {
        const int idx = tid + 256 * g, f = idx % kN, j = idx / kN;
#pragma unroll
        for (int r = 0; r < 8; ++r) bias_acc[g] += va[g][r];
        const int mb = f >> 7, off = j * (128 * 16) + (f & 127) * 16;
        split8_store(va[g], pl + mb * G::kAPlane + off, pl + (NM + mb) * G::kAPlane + off);
      }
#pragma unroll
      for (int g = 0; g < kGb; ++g) {
        const int idx = tid + 256 * g, f = idx % KP, j = idx / KP;
        if (j < 2) {
          const int off = j * (KP * 16) + f * 16;
          split8_store(vb[g], pl + 2 * NM * G::kAPlane + off, pl + 2 * NM * G::kAPlane + G::kBPlane + off);
        }
        if (KP == 256 && a.x_pos_bits != nullptr) {
          // the ReLU mask the following dgrad needs, as a by-product: a warp holds 32 consecutive features
          // of the same 8 points, so one ballot per point is that point's mask word
          uint32_t mine = 0;
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            const uint32_t w = __ballot_sync(0xffffffffu, vb[g][r] > 0.f);
            if (lane == r) mine = w;
          }
          if (lane < 8 && j * 8 + lane < rows) a.x_pos_bits[(p0 + j * 8 + lane) * 8 + (f >> 5)] = mine;
        }
      }
      fence_proxy_async_smem();     // generic-proxy smem writes -> visible to tcgen05.mma
      mbar_arrive(&pl_full[pb]);
    }
    if (a.db != nullptr && n_batches > 0) {
#pragma unroll
      for (int g = 0; g < kGa; ++g) atomicAdd(a.db + (tid + 256 * g) % kN, bias_acc[g]);
    }

    // ======================= epilogue: TMEM -> smem -> atomics, one out-feature block at a time ==
    if (n_batches > 0) {
      mbar_wait(&d_full, 0);
      tc_fence_after();
      float* out = reinterpret_cast<float*>(ring);       // [128][KP + 4]; every copy and MMA has retired
      constexpr int kLd = G::kOutLd;
#pragma unroll 1
      for (int mb = 0; mb < NM; ++mb) {
        if (warp < 4) {
          const int row = warp * 32 + lane;
#pragma unroll 1
          for (int c0 = 0; c0 < KP; c0 += 32) {
            uint32_t v[32];
            tmem_ld32(tbase + ((uint32_t)(warp * 32) << 16) + mb * KP + c0, v);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              *reinterpret_cast<float4*>(out + row * kLd + c0 + j) =
                  make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
          }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kWgConvWarps * 32) : "memory");
        if (KP % 4 == 0 && a.K == KP && ((a.ldw | a.col_off) & 3) == 0 && (reinterpret_cast<uintptr_t>(a.dW) & 15) == 0) {
          // 16-byte vector reductions (red.global.add.v4.f32): a quarter of the L2 atomic operations
          for (int e = tid; e < 128 * (KP / 4); e += kWgConvWarps * 32) {
            const int m = e / (KP / 4), k = (e - m * (KP / 4)) * 4;
            const float4 v = *reinterpret_cast<const float4*>(out + m * kLd + k);
            float* dst = a.dW + (size_t)(mb * 128 + m) * a.ldw + a.col_off + k;
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                         : "memory");
          }
        } else {
          for (int e = tid; e < 128 * KP; e += kWgConvWarps * 32) {
            const int m = e / KP, k = e - m * KP;
            if (k < a.K) atomicAdd(a.dW + (size_t)(mb * 128 + m) * a.ldw + a.col_off + k, out[m * kLd + k]);
          }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kWgConvWarps * 32) : "memory");
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kWgMmaWarp) tmem_dealloc<G::kTmemCols>(tbase);
}

int wg_sms() { return sm_count(); }

template <int KP, int NM, int LDX>
int launch_wgrad_tc(WgradTcArgs a, cudaStream_t st) {
  using G = WgGeo<KP, NM, LDX>;
  static SmemOptIn optin;
  if (int rc = ensure_smem(wgrad_tc_kernel<KP, NM, LDX>, optin, G::kSmemBytes, "wgrad_tc")) return rc;
  int splits = wg_sms();
  long long rows = (a.P + splits - 1) / splits;
  rows = (rows + kWgBatch - 1) / kWgBatch * kWgBatch;
  splits = (int)((a.P + rows - 1) / rows);
  a.rows_per_split = rows;
  wgrad_tc_kernel<KP, NM, LDX><<<splits, kWgThreads, G::kSmemBytes, st>>>(a);
  return check_launch("wgrad_tc_kernel");
}

}  // namespace

// run_wgrad (field_bwd.cu) on tensor cores: same accumulate-into semantics; optionally also emits the
// sign bits of X (the ReLU mask of the layer's input) for the dgrad that follows.  dY is (P, N) with
// N = 128 or 256, X is (P, ldx) with (K, ldx) one of (256, 256), (63, 64), (27, 32).
int run_wgrad_tc(const float* dY, int N, const float* X, int ldx, int K, float* dW, int ldw, int col_off, float* db,
                 uint32_t* x_pos_bits, long long P, cudaStream_t st) {
  if (P == 0) return SNB_OK;
  if (x_pos_bits != nullptr && K != 256) return fail(SNB_ERR_INVALID, "run_wgrad_tc: mask bits need K = 256");
  if ((reinterpret_cast<uintptr_t>(dY) | reinterpret_cast<uintptr_t>(X)) & 15)
    return fail(SNB_ERR_INVALID, "run_wgrad_tc: dY and X must be 16-byte aligned");
  WgradTcArgs a{dY, X, K, dW, ldw, col_off, db, x_pos_bits, P, 0};
  if (N == 256 && ldx == 256 && K == 256) return launch_wgrad_tc<256, 2, 256>(a, st);
  if (N == 128 && ldx == 256 && K == 256) return launch_wgrad_tc<256, 1, 256>(a, st);
  if (N == 256 && ldx == 64 && K <= 64) return launch_wgrad_tc<64, 2, 64>(a, st);
  if (N == 128 && ldx == 32 && K <= 32) return launch_wgrad_tc<32, 1, 32>(a, st);
  return fail(SNB_ERR_INVALID, "run_wgrad_tc: unsupported shape N=%d K=%d ldx=%d", N, K, ldx);
}

}  // namespace snb
