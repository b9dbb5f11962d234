// field_tc.cu -- the fused field pass on 5th-gen tensor cores (tcgen05 / TMEM / bulk TMA).
//
// Same contract as field_simt.cu (points o+d*z, both positional encodings, the 12-layer MLP,
// [r,g,b,sigma] out; reference models/rendering.py:184-212,284-285 + models/nerf.py:24-41,
// 105-148), but every 256-wide layer is a chain of tcgen05.mma instructions:
//
//   * persistent CTA PAIRS (cluster of 2, cta_group::2): every MMA is M = 256 -- 128 points of
//     the even CTA's tile and 128 of the odd CTA's -- and each CTA stages only HALF of every
//     weight chunk.  Measured reason: an SM ingests ~28 B/clk from L2, and a 1-CTA design needs
//     2.3 MB of weights per 128-point tile, i.e. 84k cycles of ingest against 56k cycles of MMA;
//     the pair halves the bytes per SM (probes/umma2_probe.cu validated the 2-CTA forms);
//   * accumulator D (128 x 256 fp32) in TMEM columns [0,256);
//   * the NEXT layer's A operand never touches shared memory or HBM: the epilogue warps read
//     D with tcgen05.ld, add bias, apply ReLU, split the fp32 value into a 16-bit hi part and a
//     16-bit lo part and write both back to TMEM columns [256,384) / [384,512) with tcgen05.st;
//     the MMAs read A straight from TMEM (".ts" operand form);
//   * weights stream from L2 through a 5-stage smem ring of 32 KB chunk shares (per CTA: 64 output
//     rows x 128 K x {hi,lo}) with cp.async.bulk (1-D TMA) + mbarrier complete_tx; the packed image is laid
//     out in exactly the order the MMA warp consumes it, in the SWIZZLE_NONE K-major canonical
//     core-matrix layout, so one share is one contiguous run of copies;
//   * one elect.sync-elected lane runs the whole MMA-issuer role over a schedule unrolled at compile
//     time (35 chunks per tile; every wait, operand offset and commit is an immediate): the tensor
//     queue is 20+ instructions deep and an MMA costs ~10 issue cycles (probes/umma_issue_probe.cu),
//     so a lean issuer stays ahead of the pipe; a table-driven loop (~200 instructions per chunk) did not;
//   * fp32 parity (SNB_PREC_F16X3 / BF16X3): x*w ~= xh*wh + xl*wh + xh*wl, three MMAs per K
//     step with fp32 accumulation -- 22 (fp16) or 16 (bf16) significand bits per operand;
//     SNB_PREC_BF16 is the single product;
//   * positional encodings (63->64, 27->32 columns) are computed by the epilogue warps into
//     shared memory in the canonical layout and consumed by ".ss" MMAs at layers 1, 5 (skip)
//     and the direction layer, so neither concat exists;
//   * sigma (256->1) and rgb (128->3) heads are fp32 dot products inside the epilogue;
//   * the bottleneck layer (256->256, no activation, nerf.py:140) is folded into the direction layer at
//     pack time: Wd[:, :256] (Wf h + bf) = (Wd[:, :256] Wf) h + Wd[:, :256] bf -- one 256-wide layer
//     (11 % of the MMA work) less per point, same function up to fp32 rounding.
//
// Schedule inside a layer (N = 256 split in halves a|b, K = 256 in halves 0|1):
//     (a,k0) (a,k1) -> D_a full | (b,k0) -> A[k0] free | (b,k1) -> D_b full
// Epilogue a (reads D_a, writes the next layer's A[k0]) overlaps both b phases -- it only has to
// hold its stores until (b,k0), the last reader of A[k0], has retired; epilogue b overlaps the
// next layer's (a,k0).  Measured with the clock64 trace (tools/trace_field.py): an epilogue half
// costs ~1400 cycles against 1536 per MMA phase, so the older interleaved order stalled ~1000
// cycles per layer.
//
// kTrain (snb_field_forward_train): the same kernel also writes the embeddings and every layer's
// post-activation output (fp32, row-major) for the backward; those stores go through per-warp
// shared-memory transposition tiles so that they leave as 64-byte runs, and the weight ring shrinks
// to 3 stages to make room.
//
// Roofline: tensor pipe.  Executed MMA FLOPs are 3x the algorithmic 1 186 816 FLOP/point in the
// split modes.  HBM traffic: 4 B/point in (z) + 16 B/point out; weights (2.3 MB per tile pass)
// are L2 hits.
#include <stdlib.h>

#include <type_traits>
#include <utility>

#include "act16.cuh"
#include "common.cuh"
#include "umma.cuh"

namespace snb {
using namespace umma;

// ------------------------------------------------------------------ geometry
constexpr int kTile = 128;             // points per CTA tile (an MMA spans both tiles of the pair: M = 256)
constexpr int kNh = 128;               // output columns per MMA (N); a 256-wide layer is two halves
constexpr int kEpiWarps = 16;          // warps 0..15: prologue / epilogue (4 per TMEM lane quadrant)
constexpr int kMmaWarp = 16, kLoadWarp = 17;
constexpr int kEncWarp0 = 18, kEncWarps = 2;   // positional encodings of the NEXT slot, off the epilogue warps' critical path
constexpr int kThreads = (kEncWarp0 + kEncWarps) * 32;   // 640: <= 102 registers per thread (96 used)
constexpr uint32_t kColD = 0, kColAhi = 256, kColAlo = 384;

// weight chunks: a chunk is 128 output rows x (16 * steps) of K, steps <= kMaxSteps; each CTA of the
// pair holds kRowsB = 64 of those rows
constexpr int kKc = 128;                                    // K per full chunk
constexpr int kRowsB = kNh / 2;
constexpr int kMaxSteps = kKc / 16;
constexpr uint32_t kStepBytes = kRowsB * 16 * 2;            // one K16 step of one of {hi, lo} of a CTA's share
constexpr uint32_t kPartBytesMax = kStepBytes * kMaxSteps;

enum { SRC_ENC = 0, SRC_HID = 1, SRC_DIR = 2 };
// WAIT_A0..A3: the previous layer's epilogue has stored output columns [64q, 64q+64) (= this layer's K
// quarter q) into the A operand -- and the threads that own those columns have read them out of the
// accumulator.  An MMA with accumulate = 0 overwrites all 128 columns of its half, so the first chunk on
// half a waits for A0 AND A1 (both column quarters of D_a drained), not just for the quarter whose data it
// consumes first; half b's first chunk comes after (a,k1), which has waited for A2 and A3.
enum { WAIT_NONE = 0, WAIT_ENC = 1, WAIT_DIR = 2, WAIT_A0 = 4, WAIT_A1 = 5, WAIT_A2 = 6, WAIT_A3 = 7 };
enum { COMMIT_NONE = 0, COMMIT_D0 = 1, COMMIT_D1 = 2, COMMIT_AFREE = 4 };   // bit flags

struct alignas(16) Chunk {
  uint8_t layer;     // 0..9 (8 = bottleneck, 9 = direction layer)
  uint8_t half;      // output columns [128*half, +128)
  uint8_t src;       // SRC_*: where the A operand of this chunk lives
  uint8_t a16;       // K offset of the chunk inside that source, in K16 steps
  uint8_t w16;       // K offset in the layer's padded weight K space (gemm_k), in K16 steps
  uint8_t steps;     // K16 steps in this chunk
  uint8_t first;     // first chunk of this (layer, half): accumulate = 0
  uint8_t wait;      // WAIT_* before the first step
  uint8_t wait_mid;  // WAIT_* before step `mid` (a chunk that spans two K quarters)
  uint8_t mid;       // first step of the second part (== steps when there is no second part)
  uint8_t commit;    // COMMIT_* flags after issuing
  uint8_t wait2;     // second WAIT_* before the first step (a chunk that overwrites accumulator half a)
  uint16_t off;      // K16 steps of all earlier chunks: byte offset in the image = off * step bytes
  uint16_t pad2;
};
constexpr int kMaxChunks = 160;
struct ChunkTable {
  Chunk c[kMaxChunks];
  int n_total;       // chunks per tile, full head
  int n_sigma_only;  // chunks per tile through layer 8
  int steps_total;   // sum of steps
};

// order inside a layer: half a (enc, hid k 0..255) -> D_a | half b (enc, hid k 0..127) -> A[k0] free |
// (hid k 128..255) -> D_b
__host__ __device__ constexpr ChunkTable make_chunk_table() {
  ChunkTable t{};
  int n = 0, off = 0;
  for (int l = 0; l < kNumGemm; ++l) {
    if (l == 8) continue;   // bottleneck: folded into the direction layer's weights (pack_tc_kernel)
    const bool has_enc = (l == 0 || l == 4);
    const bool has_hid = (l != 0);
    const int n_halves = l == 9 ? 1 : 2;
    for (int half = 0; half < n_halves; ++half) {
      bool first = true;
      // segments of this (layer, half): [enc 64] [hid 256] [dir 32]
      for (int seg = 0; seg < 3; ++seg) {
        const int src = seg == 0 ? SRC_ENC : (seg == 1 ? SRC_HID : SRC_DIR);
        const int klen = seg == 0 ? (has_enc ? kXyzPad : 0) : (seg == 1 ? (has_hid ? kWidth : 0) : (l == 9 ? kDirPad : 0));
        const int wbase = seg == 0 ? 0 : (seg == 1 ? (has_enc ? kXyzPad : 0) : kWidth);   // padded weight K offset
        for (int k0 = 0; k0 < klen; k0 += kKc) {
          const int kc = klen - k0 < kKc ? klen - k0 : kKc;
          Chunk c{};
          c.layer = l; c.half = half; c.src = src; c.a16 = k0 / 16; c.w16 = (wbase + k0) / 16; c.steps = kc / 16;
          c.first = first; c.mid = c.steps; c.off = off;
          int w = WAIT_NONE, w2 = WAIT_NONE, wm = WAIT_NONE;
          if (src == SRC_ENC && half == 0) {
            w = (l == 0) ? WAIT_ENC : WAIT_A0;                 // skip layer: D_a drained = both of its quarters
            if (l != 0) w2 = WAIT_A1;
          }
          if (src == SRC_DIR) w = WAIT_DIR;
          if (src == SRC_HID && half == 0) {
            // half a consumes K quarters 2 and 3 as the previous layer's epilogue delivers them; quarters 0
            // and 1 are both needed before the first (accumulator-overwriting) MMA of the half
            if (k0 == 0) {
              if (!has_enc) { w = WAIT_A0; w2 = WAIT_A1; }
            } else {
              if (k0 % 64 == 0) w = WAIT_A0 + k0 / 64;
              if (kc > 64) { wm = WAIT_A0 + k0 / 64 + 1; c.mid = (64 - k0 % 64) / 16; }
            }
          }
          c.wait = w; c.wait2 = w2; c.wait_mid = wm;
          const bool last_of_half = (seg == 2) || (seg == 1 && k0 + kc == klen && l != 9) || (seg == 0 && !has_hid && k0 + kc == klen);
          if (last_of_half) c.commit = half == 0 ? COMMIT_D0 : COMMIT_D1;
          // the last reader of A[k 0..127] in this layer: half b's chunk ending at K = 128
          if (half == 1 && seg == 1 && k0 + kc == 128) c.commit |= COMMIT_AFREE;
          if (half == 1 && !has_hid && last_of_half) c.commit |= COMMIT_AFREE;
          t.c[n++] = c;
          off += c.steps;
          first = false;
        }
      }
    }
    if (l == 7) t.n_sigma_only = n;
  }
  t.n_total = n;
  t.steps_total = off;
  return t;
}
__constant__ ChunkTable c_chunks = make_chunk_table();
static constexpr ChunkTable h_chunks = make_chunk_table();
static_assert(h_chunks.n_total == 35 && h_chunks.n_sigma_only == 32, "chunk schedule (K128)");
static_assert(h_chunks.steps_total == 258, "K16 steps per tile");

// number of waits on barrier code `code` (WAIT_*) in chunks [0, ci) -- plus chunk ci's own `wait` when
// the question is about its mid-chunk wait.  a_ready[q] completes once per layer epilogue, 8 per
// slot, so (prior_waits & 1) is the parity to wait for.
// stage: 0 = the chunk's first pre-wait, 1 = its second pre-wait, 2 = its mid-chunk wait
__host__ __device__ constexpr int prior_waits(const ChunkTable& t, int ci, int code, int stage) {
  int n = 0;
  for (int i = 0; i < ci; ++i) n += (t.c[i].wait == code) + (t.c[i].wait2 == code) + (t.c[i].wait_mid == code);
  if (stage >= 1) n += t.c[ci].wait == code;
  if (stage >= 2) n += t.c[ci].wait2 == code;
  return n;
}
__host__ __device__ constexpr bool wait_counts_ok(const ChunkTable& t) {
  for (int q = 0; q < 4; ++q) {
    if (prior_waits(t, t.n_total, WAIT_A0 + q, 0) != 8) return false;       // layers 1..7 and the dir layer
    if (prior_waits(t, t.n_sigma_only, WAIT_A0 + q, 0) != 7) return false;  // + the explicit drain of layer 8's
  }
  return prior_waits(t, t.n_total, WAIT_ENC, 0) == 1 && prior_waits(t, t.n_total, WAIT_DIR, 0) == 1;
}
static_assert(wait_counts_ok(h_chunks), "static wait parities");

template <class F, int... I>
__device__ __forceinline__ void static_for_impl(F&& f, std::integer_sequence<int, I...>) {
  (f(std::integral_constant<int, I>{}), ...);
}
template <int N, class F>
__device__ __forceinline__ void static_for(F&& f) { static_for_impl(f, std::make_integer_sequence<int, N>{}); }

// ------------------------------------------------------------------ packed image
// [PackedHeader 256 B][consts: biases + head weights, fp32][chunk 0][chunk 1]...
struct ConstLayout {
  int b[kNumGemm];
  int sigma_w, sigma_b, rgb_w, rgb_b, total;
};
__host__ __device__ constexpr ConstLayout make_const_layout() {
  ConstLayout L{};
  int off = 0;
  for (int l = 0; l < kNumGemm; ++l) { L.b[l] = off; off += gemm_n(l); }
  L.sigma_w = off; off += kWidth;
  L.sigma_b = off; off += 4;
  L.rgb_w = off; off += 3 * kHalf;
  L.rgb_b = off; off += 4;
  L.total = (off + 63) & ~63;
  return L;
}
constexpr int kConstFloats = make_const_layout().total;
constexpr size_t kConstBytes = (size_t)kConstFloats * 4;

__host__ __device__ constexpr bool prec_split(int precision) { return precision != SNB_PREC_BF16; }
// image bytes of one K16 step of a chunk (all CTAs' shares, hi and lo): 128 rows x 16 K x 2 B (x2)
__host__ __device__ constexpr uint32_t step_image_bytes(int precision) {
  return (uint32_t)(kNh * 16 * 2 * (prec_split(precision) ? 2 : 1));
}
// scratch at the end of the image: W' = Wd[:, :256] Wf (128 x 256) and b' = bd + Wd[:, :256] bf (128)
constexpr size_t kFusedFloats = (size_t)kHalf * kWidth + kHalf;
__host__ __device__ constexpr size_t chunks_bytes(int precision) {
  return (size_t)make_chunk_table().steps_total * step_image_bytes(precision);
}
size_t tc_packed_bytes(int precision) {
  return sizeof(PackedHeader) + kConstBytes + chunks_bytes(precision) + kFusedFloats * sizeof(float);
}

// 16-bit conversions -------------------------------------------------------------------
template <bool kBf16>
__device__ __forceinline__ uint16_t cvt16(float x) {
  if (kBf16) return __bfloat16_as_ushort(__float2bfloat16_rn(x));
  return __half_as_ushort(__float2half_rn(x));
}
template <bool kBf16>
__device__ __forceinline__ float up16(uint16_t h) {
  if (kBf16) return __bfloat162float(__ushort_as_bfloat16(h));
  return __half2float(__ushort_as_half(h));
}
// x -> (hi, lo) with hi + lo ~= x.  fp16 saturates at +-65504 instead of overflowing to inf.
template <bool kBf16>
__device__ __forceinline__ void split16(float x, uint16_t& hi, uint16_t& lo) {
  if (!kBf16) x = fminf(fmaxf(x, -65504.f), 65504.f);
  hi = cvt16<kBf16>(x);
  lo = cvt16<kBf16>(x - up16<kBf16>(hi));
}

// Two values at once, with the packed converts (F2FP.*.PACK_AB, full-rate pipe) instead of four
// scalar F2F (quarter-rate MIO pipe): hi = pack(x0, x1); lo = pack(x0 - up(hi.x), x1 - up(hi.y)).
template <bool kBf16, bool kSplit, bool kNonNeg = false>
__device__ __forceinline__ void split_pair(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  if (kBf16) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    if (kSplit) {
      const float b0 = __uint_as_float(hi << 16), b1 = __uint_as_float(hi & 0xffff0000u);
      const __nv_bfloat162 l = __floats2bfloat162_rn(x0 - b0, x1 - b1);
      lo = *reinterpret_cast<const uint32_t*>(&l);
    } else {
      lo = 0;
    }
  } else {
    if (kNonNeg) { x0 = fminf(x0, 65504.f); x1 = fminf(x1, 65504.f); }   // ReLU output: one-sided
    else { x0 = fminf(fmaxf(x0, -65504.f), 65504.f); x1 = fminf(fmaxf(x1, -65504.f), 65504.f); }
    const __half2 h = __floats2half2_rn(x0, x1);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    if (kSplit) {
      const float2 b = __half22float2(h);
      const __half2 l = __floats2half2_rn(x0 - b.x, x1 - b.y);
      lo = *reinterpret_cast<const uint32_t*>(&l);
    } else {
      lo = 0;
    }
  }
}

// ReLU + split of two PRE-activation values with no separate max / clamp instructions: the packed converts
// carry .relu and .satfinite themselves.  hi = relu(x) rounded TOWARD ZERO, so the residual x - hi is >= 0
// whenever x >= 0 and negative only when x < 0 (hi = 0) -- then lo = rn(relu(residual)) is 0, as it must be.
// (Truncation leaves a residual of up to one ulp of hi instead of half: hi + lo still carries 21 (fp16) /
// 15 (bf16) significand bits.)  4 + 2 instructions per pair instead of 8 + 2.
template <bool kBf16, bool kSplit>
__device__ __forceinline__ void split_pair_relu(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  if (kBf16) {
    if (kSplit) asm("cvt.rz.relu.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
    else asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
    if (kSplit) {
      const float r0 = x0 - __uint_as_float(hi << 16), r1 = x1 - __uint_as_float(hi & 0xffff0000u);
      asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(r1), "f"(r0));
    } else {
      lo = 0;
    }
  } else {
    if (kSplit) asm("cvt.rz.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
    else asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
    if (kSplit) {
      const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&hi));
      const float r0 = x0 - b.x, r1 = x1 - b.y;
      asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(r1), "f"(r0));
    } else {
      lo = 0;
    }
  }
}

// softplus(x - 1) with the hardware ex2 / lg2 approximations (abs error ~1e-7 on an O(1..200)
// value; the accurate expf/log1pf pair cost the dir-layer epilogue ~10k cycles per tile).
// `s` is already shifted (x - 1): 4 FP32 ops + 2 MUFU.
__device__ __forceinline__ float softplus_fast(float s) {
  float t;                                                             // exp(-|s|) in (0, 1]
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(-1.4426950408889634f * fabsf(s)));
  return fmaf(__log2f(1.0f + t), 0.6931471805599453f, fmaxf(s, 0.0f));   // max(s,0) + log1p(t)  (lg2.approx)
}

// sin / cos for the positional encoding of the single-product bf16 mode: two-constant Cody-Waite reduction to
// [-pi, pi] and the MUFU approximations (abs error ~1e-6 for |x| up to ~1e4 -- three orders below bf16's 2^-9
// rounding of the encoded value), ~8 instructions instead of sincosf's ~50.  In that mode an MMA phase is only 512
// cycles and the encoding, done by the epilogue warps between layers, was on the critical path: 8.8k of a 32k-cycle
// slot (profiles/r02_trace_bf16_before_fast_trig.txt).  The fp32-parity modes keep the accurate sincosf.
__device__ __forceinline__ void sincos_fast(float x, float* sn, float* cs) {
  const float k = rintf(x * 0.15915494309189535f);
  float r = fmaf(k, -6.2831854820251465f, x);
  r = fmaf(k, 1.7484555e-7f, r);
  *sn = __sinf(r);
  *cs = __cosf(r);
}

// ------------------------------------------------------------------ pack kernel
// W'[n][k] = sum_j Wd[n][j] Wf[j][k],  b'[n] = bd[n] + sum_j Wd[n][j] bf[j]   (double accumulation)
__global__ void fuse_bottleneck_kernel(ParamPtrs pp, float* fused, const PackedHeader* hdr, int only_if_dirty) {
  if (only_if_dirty && !hdr->dirty) return;
  const float* Wd = pp.p[18];   // (128, 283)
  const float* Wf = pp.p[16];   // (256, 256)
  const float* bf = pp.p[17];
  const float* bd = pp.p[19];
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < kHalf * (kWidth + 1); e += gridDim.x * blockDim.x) {
    const int n = e / (kWidth + 1), k = e - n * (kWidth + 1);
    double acc = k == kWidth ? (double)bd[n] : 0.0;
    for (int j = 0; j < kWidth; ++j) acc += (double)Wd[n * 283 + j] * (double)(k == kWidth ? bf[j] : Wf[j * kWidth + k]);
    if (k == kWidth) fused[kHalf * kWidth + n] = (float)acc;
    else fused[n * kWidth + k] = (float)acc;
  }
}

template <bool kBf16, bool kSplit>
__global__ void pack_tc_kernel(ParamPtrs pp, int precision, int new_activation, unsigned char* image, int only_if_dirty) {
  constexpr ConstLayout CL = make_const_layout();
  const ChunkTable& tab = c_chunks;
  PackedHeader* hdr = reinterpret_cast<PackedHeader*>(image);
  if (only_if_dirty && !hdr->dirty) return;
  float* cst = reinterpret_cast<float*>(image + sizeof(PackedHeader));
  unsigned char* chunks = image + sizeof(PackedHeader) + kConstBytes;
  const float* fused = reinterpret_cast<const float*>(chunks + chunks_bytes(precision));   // fuse_bottleneck_kernel
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
  if (gtid == 0) {
    hdr->magic = kMagic;
    hdr->precision = precision;
    hdr->new_activation = new_activation;
  }
  for (int e = gtid; e < kConstFloats; e += gsz) {
    float v = 0.f;
    if (e < CL.sigma_w) {
      int l = 0;
      while (l + 1 < kNumGemm && e >= CL.b[l + 1]) ++l;
      v = l == 9 ? fused[kHalf * kWidth + (e - CL.b[l])] : pp.p[param_weight_index(l) + 1][e - CL.b[l]];
    } else if (e < CL.sigma_b) v = pp.p[kSigmaW][e - CL.sigma_w];
    else if (e == CL.sigma_b) v = pp.p[kSigmaB][0];
    else if (e >= CL.rgb_w && e < CL.rgb_b) v = pp.p[kRgbW][e - CL.rgb_w];
    else if (e >= CL.rgb_b && e < CL.rgb_b + 3) v = pp.p[kRgbB][e - CL.rgb_b];
    cst[e] = v;
  }
  // chunk image: [CTA 0 share: hi | lo][CTA 1 share: hi | lo]; each of hi / lo is the canonical
  // (SWIZZLE_NONE, K-major) block [k8][kRowsB rows][8 elements] of the chunk's 16*steps K columns
  constexpr int kParts = kSplit ? 2 : 1;
  const int total = tab.steps_total * kNh * 16;
  for (int e = gtid; e < total; e += gsz) {
    const int gstep = e / (kNh * 16), rem = e - gstep * (kNh * 16);
    const int r = rem >> 4, k16 = rem & 15;
    int ci = 0;
    while (ci + 1 < tab.n_total && gstep >= tab.c[ci + 1].off) ++ci;
    const Chunk c = tab.c[ci];
    const int kk = (gstep - c.off) * 16 + k16;       // K index inside the chunk
    const int l = c.layer;
    const int n = c.half * kNh + r;
    const int kpad = c.w16 * 16 + kk;
    const int col = kpad < gemm_k(l) ? gemm_src_col(l, kpad) : -1;
    const int src_k = l == 0 ? 63 : (l == 4 ? 319 : (l == 9 ? 283 : 256));
    float w = col >= 0 ? pp.p[param_weight_index(l)][n * src_k + col] : 0.f;
    if (l == 9 && kpad < kWidth) w = fused[n * kWidth + kpad];     // direction layer sees h8 through W'
    const int owner = r / kRowsB, rr = r - owner * kRowsB;
    const uint32_t part = kStepBytes * c.steps;                   // bytes of one of {hi, lo} of a share
    unsigned char* base = chunks + (size_t)c.off * (kStepBytes * kParts * 2) + (size_t)owner * part * kParts;
    const uint32_t off = (uint32_t)(kk >> 3) * (kRowsB * 16) + rr * 16 + (kk & 7) * 2;
    if (kSplit) {
      uint16_t hi, lo;
      split16<kBf16>(w, hi, lo);
      *reinterpret_cast<uint16_t*>(base + off) = hi;
      *reinterpret_cast<uint16_t*>(base + part + off) = lo;
    } else {
      *reinterpret_cast<uint16_t*>(base + off) = cvt16<kBf16>(w);
    }
  }
}

int launch_pack_tc(const float* const* params, int precision, int new_activation, void* image, int only_if_dirty,
                   cudaStream_t st) {
  auto pack = precision == SNB_PREC_F16X3    ? pack_tc_kernel<false, true>
              : precision == SNB_PREC_BF16X3 ? pack_tc_kernel<true, true>
              : precision == SNB_PREC_BF16   ? pack_tc_kernel<true, false>
                                             : nullptr;
  if (!pack) return fail(SNB_ERR_INVALID, "launch_pack_tc: precision %d is not a tensor-core mode", precision);
  ParamPtrs pp;
  for (int i = 0; i < SNB_N_PARAM_TENSORS; ++i) pp.p[i] = params[i];
  unsigned char* img = reinterpret_cast<unsigned char*>(image);
  float* fused = reinterpret_cast<float*>(img + sizeof(PackedHeader) + kConstBytes + chunks_bytes(precision));
  fuse_bottleneck_kernel<<<148, 256, 0, st>>>(pp, fused, reinterpret_cast<const PackedHeader*>(img), only_if_dirty);
  if (int rc = check_launch("fuse_bottleneck_kernel")) return rc;
  pack<<<296, 256, 0, st>>>(pp, precision, new_activation, img, only_if_dirty);
  return check_launch("pack_tc_kernel");
}

// ------------------------------------------------------------------ shared memory
// kTrain: 0 = inference, 1 = training forward keeping fp32 row-major activations (snb_field_forward_train),
//         2 = training forward keeping fp16 activations in the T32 layout + ReLU mask words (act16.cuh)
template <bool kSplit, int kTrain>
struct TcSmem {
  static constexpr int kParts = kSplit ? 2 : 1;
  static constexpr uint32_t kStageBytes = kPartBytesMax * kParts;   // this CTA's share of a full chunk
  // up to 160 KB of weights in flight; the training forward gives 64 KB of that to the store tiles below
  static constexpr int kStagesRaw = ((kTrain == 1 ? 96 : 160) * 1024) / kStageBytes;
  static constexpr int kStages = kStagesRaw > 16 ? 16 : kStagesRaw;
  alignas(1024) unsigned char ring[kStages][kStageBytes];
  alignas(128) unsigned char enc[kParts][kTile * kXyzPad * 2];   // canonical [k8][row][8] hi (, lo)
  alignas(128) unsigned char dir[kParts][kTile * kDirPad * 2];
  alignas(16) float cst[kConstFloats];
  float sigp[4][kTile];           // sigma head partial sums per 32-column group; [0] ends up holding sigma
  // rgb head partial sums [4][3][kTile].  The split modes have no room for them and alias dir[0] (idle by then); the
  // single-product mode has, which lets the encoder warps write the next dir embedding without waiting for rgb_done
  float rgbp_own[kSplit ? 1 : 12 * kTile];
  // training forward: per-warp 32 x 16 transposition tiles (row stride 20 words: conflict-free 128-bit
  // accesses) so the activations leave as 64 contiguous bytes per 4 lanes instead of 16 bytes per lane
  // at a 1 KB stride -- 8 lines per store instruction instead of 32
  alignas(16) float store_tile[kTrain == 1 ? kEpiWarps : 1][kTrain == 1 ? 32 : 1][20];
  uint64_t full[16], empty[16];
  // (the rgb head's partial sums alias dir[0], idle by then: float [4][3][kTile])
  uint64_t d_full[2], a_ready[4], a_free, enc_ready, dir_ready, d_drained;
  uint64_t enc_free, dir_free;    // MMA -> encoder warps: the last MMA reading enc / dir of this slot has retired
  uint64_t rgb_done;              // epilogue -> encoder warps: the rgb partial sums parked in dir[0] have been consumed
  uint64_t d_full_dir;            // single-product mode: the direction layer's own "accumulator full" (without the d_drained
                                  // hand-shake d_full[0] would see two completions -- the direction layer and the next
                                  // layer 1 -- that no consumer observation separates)
  uint32_t tmem_base;
};

struct TcParams {
  const unsigned char* image;
  const float* rays;
  const float* z;
  int n_samples;
  const float* x;          // embedded input rows (standalone NeRF.forward)
  long long x_stride;
  long long n_points;
  int sigma_only;
  float* out;
  // training forward (kTrain): what the backward needs, row-major fp32 (snb_field_forward_train)
  float* save_enc;         // (P,64)
  float* save_dir;         // (P,32)
  float* save_h;           // (8,P,256)
  float* save_g;           // (P,128)
  // training forward, 16-bit storage (kTrain == 2): sections of the act16 buffer (act16.cuh)
  unsigned char* a_enc;    // (Ppad,64)  fp16 T32
  unsigned char* a_dir;    // (Ppad,32)
  unsigned char* a_h;      // 8 x (Ppad,256)
  unsigned char* a_g;      // (Ppad,128)
  uint32_t* a_mask;        // (8, 8, Ppad)
  long long ppad;
  int debug;   // SNB_TC_DEBUG; only bit 8 is read: record the clock64 trace below
};

// ---- debug trace (SNB_TC_DEBUG & 8): clock64 stamps of one slot of cluster 0's leader CTA
constexpr int kTraceLen = 2048;
__device__ long long g_trace[kTraceLen];
__device__ __forceinline__ void trace(bool on, int idx) { if (on && idx < kTraceLen) g_trace[idx] = clock64(); }

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 512;" ::: "memory"); }

template <bool kBf16, bool kSplit, bool kEmbedded, int kTrain>
__global__ void __launch_bounds__(kThreads, 1) field_tc_kernel(TcParams p) {
  static_assert(!(kTrain != 0 && kEmbedded), "the training forward is the fused (rays, z) entry only");
  using Smem = TcSmem<kSplit, kTrain>;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  Smem& s = *reinterpret_cast<Smem*>(smem_raw);
  constexpr ConstLayout CL = make_const_layout();
  constexpr uint32_t kStageBytes = Smem::kStageBytes;
  constexpr int kStages = Smem::kStages;
  constexpr int kParts = Smem::kParts;
  static_assert(kStages <= 16, "barrier arrays");
  const ChunkTable& tab = c_chunks;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const PackedHeader* hdr = reinterpret_cast<const PackedHeader*>(p.image);
  const int new_activation = hdr->new_activation;
  const float* g_cst = reinterpret_cast<const float*>(p.image + sizeof(PackedHeader));
  const unsigned char* g_chunks = p.image + sizeof(PackedHeader) + kConstBytes;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  // tile slots: pair g handles tile (g + i * n_pairs) * 2 + rank.  Both CTAs of a pair run the same
  // number of slots; slots past the end compute on zeros, store nothing.
  const long long ntiles = (p.n_points + kTile - 1) / kTile;
  const long long n_pairs = gridDim.x / 2, pair = blockIdx.x / 2;
  const long long n_slots = ((ntiles + 1) / 2 + n_pairs - 1) / n_pairs;
  const int n_layers_epi = 8;   // trunk layers with a TMEM->TMEM epilogue (the bottleneck is folded away)
  const int n_chunks = p.sigma_only ? tab.n_sigma_only : tab.n_total;
  // Deferred direction-layer epilogue (round 2, single-product mode).  The 128 softplus + rgb head of a tile are
  // MUFU-bound (~2.8k cycles for the 16 epilogue warps) and used to run between the direction layer and the NEXT tile's
  // layer-1 epilogue: the tensor pipe idled ~2.9k of a 26k-cycle slot at every slot boundary
  // (profiles/r02b_trace_bf16_before_deferral.txt, chunk 2).  The single-product mode never uses the A-lo columns
  // [384,512) of TMEM, so there the direction layer accumulates into THEM and the result simply stays: no drain, no
  // d_drained hand-shake, the next tile's layer 1 starts at once, and the epilogue warps work the pre-activations off in
  // four 8-column pieces (one tcgen05.ld each) in the windows where they wait for the next accumulator anyway -- after
  // the second epilogue half of layers 1..4 of the next slot (slot 24.4k cycles, r02b_trace_bf16_deferred_dir_epilogue.txt).
  // The split modes keep the in-place epilogue: TMEM is exactly full there, and a variant that parked the drained values
  // in local memory shortened the slot by 4 % in cycles and not at all in time -- that kernel runs at the 1 kW power cap
  // and the clock gave the cycles back (profiles/r02b_field_variants_ab.txt, r02b_trace_f16x3_deferred_experiment.txt).
  constexpr bool kDirTmem = !kSplit && kTrain != 1;      // (the legacy fp32-storage training forward keeps the old order)
  constexpr int kDirPieces = kDirTmem ? 4 : 1;

  // ---------------- one-time setup
  for (int i = tid; i < kConstFloats; i += kThreads) s.cst[i] = g_cst[i];
  if (tid == 0) {
    // full: this CTA's loader (+ the peer's relay, at the leader); a_ready / enc_ready live at the
    // leader and count the epilogue threads of both CTAs
    for (int i = 0; i < kStages; ++i) { mbar_init(&s.full[i], leader ? 2 : 1); mbar_init(&s.empty[i], 1); }
    mbar_init(&s.d_full[0], 1); mbar_init(&s.d_full[1], 1); mbar_init(&s.a_free, 1);
    for (int i = 0; i < 4; ++i) mbar_init(&s.a_ready[i], kEpiWarps * 16 * 2);   // the two warps-of-four that own the quarter
    mbar_init(&s.enc_ready, kEncWarps * 32 * 2);
    mbar_init(&s.dir_ready, kEncWarps * 32 * 2);
    mbar_init(&s.d_drained, kEpiWarps * 32 * 2);
    mbar_init(&s.enc_free, 1);
    mbar_init(&s.dir_free, 1);
    mbar_init(&s.rgb_done, kEpiWarps);
    mbar_init(&s.d_full_dir, 1);
    fence_mbar_init();
  }
  if (warp == kMmaWarp) tmem_alloc_pair(&s.tmem_base);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // the peer's barriers exist before anyone signals them
  tc_fence_after();
  const uint32_t tbase = s.tmem_base;

  // ---- helpers shared by the encoder and the epilogue warps
  auto tile_of = [&](long long slot) { return (pair + slot * n_pairs) * 2 + cta_rank; };
  // hand-off to the MMA issuer, which lives in the leader CTA
  auto signal = [&](uint64_t* bar) { if (!leader) mbar_arrive_remote(bar, 0); else mbar_arrive(bar); };
  // 16-bit storage: 8 consecutive features of one point -> one 16-byte cell of a T32 tensor
  auto store_cell16 = [&](unsigned char* base, long long pt, int f8, int F, const float (&v)[8]) {
    if (pt >= p.ppad) return;
    const bool live = pt < p.n_points;
    uint4 c;
    c.x = live ? pack_half2_sat(v[0], v[1]) : 0u; c.y = live ? pack_half2_sat(v[2], v[3]) : 0u;
    c.z = live ? pack_half2_sat(v[4], v[5]) : 0u; c.w = live ? pack_half2_sat(v[6], v[7]) : 0u;
    *reinterpret_cast<uint4*>(base + a16_cell(pt, f8, F)) = c;
  };
  // 8 consecutive channels (one 16-byte core-matrix row of tile row `r`) -> hi (and lo) vector stores, canonical layout
  auto put8 = [&](unsigned char* hi_base, unsigned char* lo_base, int k8, int r, const float (&v)[8]) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) split_pair<kBf16, kSplit>(v[2 * j], v[2 * j + 1], h[j], l[j]);
    const uint32_t off = (uint32_t)k8 * (kTile * 16) + r * 16;
    *reinterpret_cast<uint4*>(hi_base + off) = make_uint4(h[0], h[1], h[2], h[3]);
    if (kSplit) *reinterpret_cast<uint4*>(lo_base + off) = make_uint4(l[0], l[1], l[2], l[3]);
  };

  if (warp == kLoadWarp) {
    // ======================= weight loader (one elected lane) =======================
    // streams this CTA's share of every chunk, in schedule order, through the ring
    if (elect_one()) {
      uint32_t it = 0;
      for (long long slot = 0; slot < n_slots; ++slot) {
        for (int ci = 0; ci < n_chunks; ++ci, ++it) {
          const uint32_t st = it % kStages, ph = (it / kStages) & 1;
          mbar_wait(&s.empty[st], ph ^ 1);
          const Chunk c = tab.c[ci];
          const uint32_t share = kStepBytes * kParts * c.steps;         // this CTA's bytes of the chunk
          const unsigned char* src = g_chunks + (size_t)c.off * (kStepBytes * kParts * 2) + (size_t)cta_rank * share;
          mbar_arrive_expect_tx(&s.full[st], share);
          for (uint32_t o = 0; o < share; o += 16384)
            bulk_g2s(s.ring[st] + o, src + o, share - o < 16384 ? share - o : 16384, &s.full[st]);
        }
      }
    }
  } else if (warp == kMmaWarp && !leader) {
    // ======================= relay (odd CTA of a pair) =======================
    // tells the leader when this CTA's share of a chunk has landed
    if (elect_one()) {
      uint32_t it = 0;
      for (long long slot = 0; slot < n_slots; ++slot) {
        for (int ci = 0; ci < n_chunks; ++ci, ++it) {
          const uint32_t st = it % kStages, ph = (it / kStages) & 1;
          mbar_wait(&s.full[st], ph);
          mbar_arrive_remote(&s.full[st], 0);
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ======================= MMA issuer (leader CTA) =======================
    // One elected lane runs the whole role.  The chunk schedule is unrolled at compile time
    // (static_for over the constexpr table): every wait, operand offset, accumulate flag and
    // commit of a chunk is an immediate, so a chunk costs a few dozen instructions besides its
    // MMAs.  (Measured: the table-driven loop spent ~200 instructions / ~1000 cycles per chunk,
    // more than the 515 cycles the tensor pipe needs for a bf16 chunk -- the issuer, not the
    // pipe, set the pace; profiles/r01_timing_experiments.txt v11.)
    if (elect_one()) {
      constexpr ChunkTable T = make_chunk_table();
      const uint32_t idesc = make_idesc(kBf16 ? kFmtBF16 : kFmtF16, 2 * kTile, kNh);   // M = both tiles of the pair
      const uint32_t enc_hi = smem_u32(s.enc[0]), dir_hi = smem_u32(s.dir[0]);
      const uint32_t enc_lo = smem_u32(s.enc[kSplit ? 1 : 0]), dir_lo = smem_u32(s.dir[kSplit ? 1 : 0]);
      // descriptors as (lo, hi) words: only the 14-bit start-address field in the low word moves
      const uint64_t desc_b0 = make_smem_desc(0, kRowsB * 16, 128);
      const uint64_t desc_a0 = make_smem_desc(0, kTile * 16, 128);
      const uint32_t bd_hi32 = (uint32_t)(desc_b0 >> 32), ad_hi32 = (uint32_t)(desc_a0 >> 32);
      const uint32_t b_ring0 = (uint32_t)desc_b0 + (smem_u32(s.ring[0]) >> 4);
      const uint32_t a_enc_hi = (uint32_t)desc_a0 + (enc_hi >> 4), a_enc_lo = (uint32_t)desc_a0 + (enc_lo >> 4);
      const uint32_t a_dir_hi = (uint32_t)desc_a0 + (dir_hi >> 4), a_dir_lo = (uint32_t)desc_a0 + (dir_lo >> 4);
      constexpr uint32_t kStepB = (2 * kRowsB * 16) >> 4;        // one K16 step inside a chunk, in 16-B units
      constexpr uint32_t kStepA = (2 * kTile * 16) >> 4;
      uint32_t st = 0, ph_full = 0;            // ring position: stage and the parity of its `full` barrier
      for (long long slot = 0; slot < n_slots; ++slot) {
        const uint32_t slot_par = (uint32_t)slot & 1;    // enc_ready / dir_ready / d_drained complete once per slot
        const bool tr = (p.debug & 8) && blockIdx.x == 0 && slot == 3;
        static_for<T.n_total>([&](auto tag) {
          constexpr int CI = decltype(tag)::value;
          constexpr Chunk c = T.c[CI];
          if (CI >= T.n_sigma_only && p.sigma_only) return;
          trace(tr, CI * 4 + 0);
          // a_ready[q] completes 8 times per slot (static_assert below): the parity of each wait is static
          auto wait_code = [&](auto code_tag, auto stage_tag) {
            constexpr int w = decltype(code_tag)::value;
            if (w == WAIT_ENC) mbar_wait(&s.enc_ready, slot_par);
            else if (w == WAIT_DIR) mbar_wait(&s.dir_ready, slot_par);
            else if (w >= WAIT_A0) mbar_wait(&s.a_ready[w - WAIT_A0], prior_waits(T, CI, w, decltype(stage_tag)::value) & 1);
          };
          wait_code(std::integral_constant<int, c.wait>{}, std::integral_constant<int, 0>{});
          wait_code(std::integral_constant<int, c.wait2>{}, std::integral_constant<int, 1>{});
          trace(tr, CI * 4 + 1);
          mbar_wait(&s.full[st], ph_full);
          tc_fence_after();
          trace(tr, CI * 4 + 2);
          const uint32_t d = tbase + (c.layer == 9 ? (kDirTmem ? kColAlo : kColD) : kColD + c.half * kNh);
          const uint32_t bh = b_ring0 + st * (kStageBytes >> 4);           // W_hi block
          const uint32_t bl = bh + ((kStepBytes * c.steps) >> 4);           // W_lo block
          // K16 steps [kLo, kHi) of this chunk
          auto issue_range = [&](auto lo_tag, auto hi_tag) {
            constexpr int kLo = decltype(lo_tag)::value, kHi = decltype(hi_tag)::value;
            if (c.src == SRC_HID) {
              const uint32_t a_hi = tbase + kColAhi + (uint32_t)c.a16 * 8;
              const uint32_t a_lo = tbase + kColAlo + (uint32_t)c.a16 * 8;
#pragma unroll
              for (int ks = kLo; ks < kHi; ++ks) {
                const uint32_t acc = (ks == 0 && c.first) ? 0u : 1u;
                mma2_ts_lohi(d, a_hi + ks * 8, bh + ks * kStepB, bd_hi32, idesc, acc);
                if (kSplit) {
                  mma2_ts_lohi(d, a_lo + ks * 8, bh + ks * kStepB, bd_hi32, idesc, 1);
                  mma2_ts_lohi(d, a_hi + ks * 8, bl + ks * kStepB, bd_hi32, idesc, 1);
                }
              }
            } else {
              constexpr uint32_t a_off = ((uint32_t)c.a16 * 2 * (kTile * 16)) >> 4;
              const uint32_t ah = (c.src == SRC_ENC ? a_enc_hi : a_dir_hi) + a_off;
              const uint32_t al = (c.src == SRC_ENC ? a_enc_lo : a_dir_lo) + a_off;
#pragma unroll
              for (int ks = kLo; ks < kHi; ++ks) {
                const uint32_t acc = (ks == 0 && c.first) ? 0u : 1u;
                mma2_ss_lohi(d, ah + ks * kStepA, ad_hi32, bh + ks * kStepB, bd_hi32, idesc, acc);
                if (kSplit) {
                  mma2_ss_lohi(d, al + ks * kStepA, ad_hi32, bh + ks * kStepB, bd_hi32, idesc, 1);
                  mma2_ss_lohi(d, ah + ks * kStepA, ad_hi32, bl + ks * kStepB, bd_hi32, idesc, 1);
                }
              }
            }
          };
          using I0 = std::integral_constant<int, 0>;
          using IM = std::integral_constant<int, c.mid>;
          using IS = std::integral_constant<int, c.steps>;
          issue_range(I0{}, IM{});
          trace(tr, 512 + CI * 4 + 0);
          if (c.mid < c.steps) {            // the chunk spans two K quarters: the second arrives later
            wait_code(std::integral_constant<int, c.wait_mid>{}, std::integral_constant<int, 2>{});
            tc_fence_after();
            issue_range(IM{}, IS{});
            trace(tr, 512 + CI * 4 + 1);
          }
          mma2_commit(&s.empty[st]);   // ring slot free (in both CTAs of the pair) once these MMAs retire
          trace(tr, 512 + CI * 4 + 2);
          if (c.commit & COMMIT_AFREE) mma2_commit(&s.a_free);
          if (c.commit & COMMIT_D0) mma2_commit((c.layer == 9 && kDirTmem) ? &s.d_full_dir : &s.d_full[0]);
          if (c.commit & COMMIT_D1) mma2_commit(&s.d_full[1]);
          if (c.src == SRC_ENC && c.layer == 4 && c.half == 1) mma2_commit(&s.enc_free);   // last reader of enc in this slot
          if (c.src == SRC_DIR) mma2_commit(&s.dir_free);
          trace(tr, 512 + CI * 4 + 3);
          if (++st == kStages) { st = 0; ph_full ^= 1; }
          trace(tr, CI * 4 + 3);
        });
        if (p.sigma_only) {
          // layer 8's epilogue arrives on a_ready[0..3] with nobody waiting: consume the phases
#pragma unroll
          for (int q = 0; q < 4; ++q) mbar_wait(&s.a_ready[q], prior_waits(T, T.n_sigma_only, WAIT_A0 + q, 0) & 1);
        } else if (!kDirTmem) {
          // the next slot's layer 1 overwrites D[0,128): wait until the dir-layer epilogue has read it
          // (kDirTmem: the direction layer has its own accumulator; its next overwrite is ordered behind the
          // a_ready waits of the next slot's layer 8, which every epilogue thread signals after its last piece)
          mbar_wait(&s.d_drained, slot_par);
        }
      }
    }
    __syncwarp();
  } else if (warp >= kEncWarp0) {
    // ======================= encoder warps: positional encodings of the NEXT slot =======================
    // 64 threads, two tile rows each.  In round 1 the epilogue warps did this in their idle windows; in the
    // single-product bf16 mode (512-cycle MMA phases) those windows do not exist and the encodings -- global loads of
    // the ray and depth, a 64-bit division, 30 sin/cos pairs -- sat on the layer-to-layer critical path: ~8k of a
    // 30k-cycle slot (profiles/r02_trace_bf16_fast_trig.txt).  Here they run beside everything else: xyz for slot s+1
    // as soon as the skip layer of slot s has consumed enc (enc_free), dir as soon as the direction layer has (dir_free).
    const int e = (warp - kEncWarp0) * 32 + lane;
    auto encode_rows = [&](long long slot, bool xyz) {
#pragma unroll 1
      for (int rr = 0; rr < kTile / (kEncWarps * 32); ++rr) {
        const int r = e + rr * (kEncWarps * 32);
        const long long pt = tile_of(slot) * kTile + r;
        const bool live = pt < p.n_points;
        float x[3] = {0.f, 0.f, 0.f};
        const float* xr = nullptr;
        if (kEmbedded) {
          xr = p.x + pt * p.x_stride;
        } else if (live) {
          const long long ray = pt / p.n_samples;
          const float4 r0 = *reinterpret_cast<const float4*>(p.rays + ray * 8);
          const float4 r1 = *reinterpret_cast<const float4*>(p.rays + ray * 8 + 4);
          if (xyz) {
            const float zz = p.z[pt];
            x[0] = __fadd_rn(r0.x, __fmul_rn(r0.w, zz));   // rendering.py:284-285 rounding
            x[1] = __fadd_rn(r0.y, __fmul_rn(r1.x, zz));
            x[2] = __fadd_rn(r0.z, __fmul_rn(r1.y, zz));
          } else {
            x[0] = r0.w; x[1] = r1.x; x[2] = r1.y;          // ray direction (not normalised, rendering.py:261)
          }
        }
        // all channels of the row in registers, one sin / cos pair per (frequency, coordinate): static indices only
        auto emit = [&](auto ktag, const float (&v8)[8]) {
          constexpr int k8 = decltype(ktag)::value;
          if (!kEmbedded) {
            if (kTrain == 1 && live) {
              float4* dst = reinterpret_cast<float4*>((xyz ? p.save_enc + pt * kXyzPad : p.save_dir + pt * kDirPad) + k8 * 8);
              dst[0] = make_float4(v8[0], v8[1], v8[2], v8[3]); dst[1] = make_float4(v8[4], v8[5], v8[6], v8[7]);
            }
            if (kTrain == 2) store_cell16(xyz ? p.a_enc : p.a_dir, pt, k8, xyz ? kXyzPad : kDirPad, v8);
          }
          if (xyz) put8(s.enc[0], s.enc[kSplit ? 1 : 0], k8, r, v8);
          else put8(s.dir[0], s.dir[kSplit ? 1 : 0], k8, r, v8);
        };
        auto encode_all = [&](auto ltag) {
          constexpr int L = decltype(ltag)::value;            // 10 (xyz, 63 -> 64 channels) or 4 (dir, 27 -> 32)
          constexpr int kCh = 3 * (2 * L + 1), kPad = (kCh + 7) / 8 * 8;
          float v[kPad];
#pragma unroll
          for (int j = 0; j < kPad; ++j) v[j] = 0.f;
          if (kEmbedded) {
            const int nin = p.sigma_only ? kXyzCh : kXyzCh + kDirCh;
#pragma unroll
            for (int j = 0; j < kCh; ++j) {
              const int col = L == SNB_XYZ_FREQS ? j : kXyzCh + j;
              v[j] = (live && col < nin) ? xr[col] : 0.f;
            }
          } else {
            v[0] = x[0]; v[1] = x[1]; v[2] = x[2];
#pragma unroll
            for (int f = 0; f < L; ++f)
#pragma unroll
              for (int c = 0; c < 3; ++c) {
                float sn, cs;
                if (kSplit) sincosf(x[c] * (float)(1 << f), &sn, &cs);
                else sincos_fast(x[c] * (float)(1 << f), &sn, &cs);
                v[3 + 6 * f + c] = sn;
                v[3 + 6 * f + 3 + c] = cs;
              }
          }
          static_for<kPad / 8>([&](auto ktag) {
            constexpr int k8 = decltype(ktag)::value;
            const float v8[8] = {v[8 * k8], v[8 * k8 + 1], v[8 * k8 + 2], v[8 * k8 + 3], v[8 * k8 + 4], v[8 * k8 + 5], v[8 * k8 + 6], v[8 * k8 + 7]};
            emit(ktag, v8);
          });
        };
        if (xyz) encode_all(std::integral_constant<int, SNB_XYZ_FREQS>{});
        else encode_all(std::integral_constant<int, SNB_DIR_FREQS>{});
      }
      fence_proxy_async_smem();     // generic-proxy smem writes -> visible to tcgen05.mma
      signal(xyz ? &s.enc_ready : &s.dir_ready);
    };
    if (n_slots > 0) {
      encode_rows(0, true);
      if (!p.sigma_only) encode_rows(0, false);
    }
    for (long long slot = 0; slot + 1 < n_slots; ++slot) {
      mbar_wait(&s.enc_free, (uint32_t)slot & 1);
      encode_rows(slot + 1, true);
      if (!p.sigma_only) {
        mbar_wait(&s.dir_free, (uint32_t)slot & 1);
        if (kSplit) mbar_wait(&s.rgb_done, (uint32_t)slot & 1);    // the rgb partial sums alias dir[0] there
        encode_rows(slot + 1, false);
      }
    }
  } else {
    // ======================= prologue / epilogue warps =======================
    const int quad = warp & 3, ch = warp >> 2;       // TMEM lane quadrant, 32-column group (0..3) of a 128-column half
    const int row = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    uint32_t ph_d = 0, ph_free = 0;       // ph_d: bit h = parity of d_full[h]
    // training forward: 16 consecutive columns of this warp's 32 rows -> global, through the warp's tile.
    // `x4[k]` = this thread's row, columns [4k, 4k+4); dst_block = address of (first row of the block, first column)
    auto store_block16 = [&](const float4 (&x4)[4], float* dst_block, long long ld, long long pt_block0) {
      float (*tile)[20] = s.store_tile[kTrain == 1 ? warp : 0];
      __syncwarp();
#pragma unroll
      for (int k = 0; k < 4; ++k) *reinterpret_cast<float4*>(&tile[lane][4 * k]) = x4[k];
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = (lane >> 2) + 8 * i, c = lane & 3;
        if (pt_block0 + r < p.n_points)
          *reinterpret_cast<float4*>(dst_block + r * ld + 4 * c) = *reinterpret_cast<const float4*>(&tile[r][4 * c]);
      }
    };

    // ---------------- direction-layer epilogue (shifted softplus / ReLU, rgb head), in pieces
    constexpr int kJ4 = 8 / kDirPieces;          // groups of four columns per piece (this thread owns 32 columns)
    const int cdir0 = ch * 32;
    // rgb partial sums go through the dir-embedding buffer: its last readers (the dir-layer MMAs of the tile the sums
    // belong to) have retired, and the encoder warps write the next dir embedding only after rgb_done
    float* rgbp = kSplit ? reinterpret_cast<float*>(s.dir[0]) : s.rgbp_own;     // [4][3][kTile]
    // piece `pc` of the tile whose row of this thread is point `dpt`; `vreg` = the 32 drained values (in-place epilogue)
    auto dir_piece = [&](int pc, long long dpt, const uint32_t* vreg) {
      const int col0 = cdir0 + pc * (4 * kJ4);
      const float4* b4 = reinterpret_cast<const float4*>(s.cst + CL.b[9] + col0);
      const float4* w0 = reinterpret_cast<const float4*>(s.cst + CL.rgb_w + col0);
      const float4* w1 = reinterpret_cast<const float4*>(s.cst + CL.rgb_w + kHalf + col0);
      const float4* w2 = reinterpret_cast<const float4*>(s.cst + CL.rgb_w + 2 * kHalf + col0);
      float a0 = 0.f, a1 = 0.f, a2 = 0.f;
      if (pc > 0) { a0 = rgbp[(ch * 3 + 0) * kTile + row]; a1 = rgbp[(ch * 3 + 1) * kTile + row]; a2 = rgbp[(ch * 3 + 2) * kTile + row]; }
      uint32_t t8[kDirTmem ? 8 : 1];
      if constexpr (kDirTmem) {
        static_assert(!kDirTmem || kJ4 == 2, "a piece is one 8-column tcgen05.ld");
        tmem_ld8(tbase + lane_base + kColAlo + col0, t8);
        tmem_wait_ld();
      }
      uint32_t g16[kTrain == 2 ? 2 * kJ4 : 1];   // this piece's direction-layer outputs as fp16 pairs
      float4 keep[4];
      const float sh = new_activation ? 1.0f : 0.0f;   // shifted softplus: fold the -1 into the bias
#pragma unroll
      for (int jj = 0; jj < kJ4; ++jj) {
        const float4 bb = b4[jj], r0 = w0[jj], r1 = w1[jj], r2 = w2[jj];
        float x[4];
        if constexpr (kDirTmem) {
#pragma unroll
          for (int e = 0; e < 4; ++e) x[e] = __uint_as_float(t8[4 * jj + e]);
        } else {
#pragma unroll
          for (int e = 0; e < 4; ++e) x[e] = __uint_as_float(vreg[4 * jj + e]);
        }
        x[0] += bb.x - sh; x[1] += bb.y - sh; x[2] += bb.z - sh; x[3] += bb.w - sh;
        if (new_activation) {
#pragma unroll
          for (int e = 0; e < 4; ++e) x[e] = softplus_fast(x[e]);
        } else {
#pragma unroll
          for (int e = 0; e < 4; ++e) x[e] = fmaxf(x[e], 0.f);
        }
        if (kTrain == 1) {
          keep[jj & 3] = make_float4(x[0], x[1], x[2], x[3]);
          if ((jj & 3) == 3) store_block16(keep, p.save_g + (dpt - lane) * kHalf + cdir0 + (jj >> 2) * 16, kHalf, dpt - lane);
        }
        if (kTrain == 2) { g16[2 * jj] = pack_half2_sat(x[0], x[1]); g16[2 * jj + 1] = pack_half2_sat(x[2], x[3]); }
        a0 = fmaf(x[0], r0.x, a0); a0 = fmaf(x[1], r0.y, a0); a0 = fmaf(x[2], r0.z, a0); a0 = fmaf(x[3], r0.w, a0);
        a1 = fmaf(x[0], r1.x, a1); a1 = fmaf(x[1], r1.y, a1); a1 = fmaf(x[2], r1.z, a1); a1 = fmaf(x[3], r1.w, a1);
        a2 = fmaf(x[0], r2.x, a2); a2 = fmaf(x[1], r2.y, a2); a2 = fmaf(x[2], r2.z, a2); a2 = fmaf(x[3], r2.w, a2);
      }
      if (kTrain == 2 && dpt < p.ppad) {
        const bool live = dpt < p.n_points;
#pragma unroll
        for (int c = 0; c < kJ4 / 2; ++c)
          *reinterpret_cast<uint4*>(p.a_g + a16_cell(dpt, (col0 >> 3) + c, kHalf)) =
              live ? make_uint4(g16[4 * c], g16[4 * c + 1], g16[4 * c + 2], g16[4 * c + 3]) : make_uint4(0u, 0u, 0u, 0u);
      }
      rgbp[(ch * 3 + 0) * kTile + row] = a0; rgbp[(ch * 3 + 1) * kTile + row] = a1; rgbp[(ch * 3 + 2) * kTile + row] = a2;
    };
    // rgb head (nerf.py:144) + the tile's [r, g, b, sigma] rows
    auto dir_finish = [&](long long dpt) {
      epi_bar_sync();
      if (ch == 0 && dpt < p.n_points) {
        float c[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const float x = ((rgbp[k * kTile + row] + rgbp[(3 + k) * kTile + row]) +
                           (rgbp[(6 + k) * kTile + row] + rgbp[(9 + k) * kTile + row])) + s.cst[CL.rgb_b + k];
          c[k] = new_activation ? widened_sigmoid_f(x) : sigmoid_f(x);
        }
        reinterpret_cast<float4*>(p.out)[dpt] = make_float4(c[0], c[1], c[2], s.sigp[0][row]);
      }
      epi_bar_sync();
      if (lane == 0) mbar_arrive(&s.rgb_done);
    };
    bool pending = false;      // the previous slot's direction-layer epilogue is still owed (kDirTmem)

    for (long long slot = 0; slot < n_slots; ++slot) {
      const long long pt_slot = tile_of(slot) * kTile + row;
      float sig_part = 0.f;
      // ---------------- trunk epilogues: D (TMEM) -> act -> A (TMEM)
      const long long pt = pt_slot;
      for (int l = 0; l < n_layers_epi; ++l) {
        const float* bias = s.cst + CL.b[l];
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
          const bool tr = (p.debug & 8) && blockIdx.x == 0 && slot == 3 && tid == 0;
          const int tb = 1024 + (l * 2 + h) * 8;
          trace(tr, tb + 0);
          mbar_wait(&s.d_full[h], (ph_d >> h) & 1); ph_d ^= 1u << h;
          tc_fence_after();
          trace(tr, tb + 1);
          const int q = ch >> 1;                       // the 64-column quarter this thread's group belongs to
          const int c0 = h * kNh + ch * 32;            // output columns == next layer's k
          uint32_t v[32];
          tmem_ld32(tbase + lane_base + kColD + c0, v);
          tmem_wait_ld();
          trace(tr, tb + 2);
          // bias + activation + hi/lo split, in place: v[2j] = hi pair j, v[2j+1] = lo pair j
          uint32_t mask_word = 0;        // kTrain == 2: [value > 0] of this thread's 32 columns, stored after the hand-off
          auto finish_group = [&](auto sigma_tag) {
            constexpr bool kSigma = decltype(sigma_tag)::value;
            const float2* b2 = reinterpret_cast<const float2*>(bias + c0);
            const float2* w2 = reinterpret_cast<const float2*>(s.cst + CL.sigma_w + c0);
            const long long pt_block0 = pt - lane;      // first row of this warp's 32-row block
            float* save_blk = kTrain == 1 ? p.save_h + ((size_t)l * p.n_points + pt_block0) * kWidth + c0 : nullptr;
            float4 keep[4];
            uint32_t h16[kTrain == 2 ? 16 : 1];      // this thread's 32 post-ReLU values as fp16 pairs
            uint32_t mword = 0;                      // [value > 0] of the 32 columns (the fp32 test the reference's ReLU makes)
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
              float x[4];
              if (!kSigma && kTrain == 0) {
                // nobody needs the fp32 post-activation value: ReLU and the fp16 range guard ride on the converts
                // one 16-byte bias load and two packed fp32x2 adds (FADD2) per four columns
                const float4 bb = *reinterpret_cast<const float4*>(b2 + j);
                const float2 x01 = __fadd2_rn(make_float2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1])), make_float2(bb.x, bb.y));
                const float2 x23 = __fadd2_rn(make_float2(__uint_as_float(v[2 * j + 2]), __uint_as_float(v[2 * j + 3])), make_float2(bb.z, bb.w));
                split_pair_relu<kBf16, kSplit>(x01.x, x01.y, v[2 * j], v[2 * j + 1]);
                split_pair_relu<kBf16, kSplit>(x23.x, x23.y, v[2 * j + 2], v[2 * j + 3]);
                continue;
              }
              if (kTrain == 2 && !kSigma) {
                // same sums, one 16-byte bias load and two packed adds per four columns (the training forward's epilogue is
                // ~2.5x the inference one in instructions -- rn hi words, ReLU mask bits, activation stores -- and sets its pace)
                const float4 bb = *reinterpret_cast<const float4*>(b2 + j);
                const float2 x01 = __fadd2_rn(make_float2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1])), make_float2(bb.x, bb.y));
                const float2 x23 = __fadd2_rn(make_float2(__uint_as_float(v[2 * j + 2]), __uint_as_float(v[2 * j + 3])), make_float2(bb.z, bb.w));
                x[0] = x01.x; x[1] = x01.y; x[2] = x23.x; x[3] = x23.y;
#pragma unroll
                for (int e = 0; e < 4; ++e) x[e] = fmaxf(x[e], 0.f);
              } else {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                  const float2 bb = b2[j + e];
                  x[2 * e] = __uint_as_float(v[2 * (j + e)]) + bb.x;
                  x[2 * e + 1] = __uint_as_float(v[2 * (j + e) + 1]) + bb.y;
                  x[2 * e] = fmaxf(x[2 * e], 0.f); x[2 * e + 1] = fmaxf(x[2 * e + 1], 0.f);
                  if (kSigma) {
                    const float2 ww = w2[j + e];
                    sig_part = fmaf(x[2 * e], ww.x, sig_part); sig_part = fmaf(x[2 * e + 1], ww.y, sig_part);
                  }
                }
              }
              if (kTrain == 1) {
                keep[(j >> 1) & 3] = make_float4(x[0], x[1], x[2], x[3]);
                if (((j >> 1) & 3) == 3) store_block16(keep, save_blk + (j >> 3) * 16, kWidth, pt_block0);
              }
              split_pair<kBf16, kSplit, true>(x[0], x[1], v[2 * j], v[2 * j + 1]);
              split_pair<kBf16, kSplit, true>(x[2], x[3], v[2 * j + 2], v[2 * j + 3]);
              if (kTrain == 2) {
                // fp16 modes: the hi word of the split IS rn_fp16(value) (saturated); bf16 modes convert separately
                h16[j] = kBf16 ? pack_half2_sat(x[0], x[1]) : v[2 * j];
                h16[j + 1] = kBf16 ? pack_half2_sat(x[2], x[3]) : v[2 * j + 2];
                // [x > 0] of the post-ReLU value (x >= +0; fmaxf(-0, +0) is +0): bits(x) + 0x7fffffff has its top bit set
                // iff bits(x) != 0, and a funnel shift moves that bit in -- 2 instructions per column instead of 3 (compare,
                // select, or).  Columns enter in ascending order, so the word is built bit-reversed (one BREV below).
#pragma unroll
                for (int e = 0; e < 4; ++e) mword = __funnelshift_l(__float_as_uint(x[e]) + 0x7fffffffu, mword, 1);
              }
            }
            if (kTrain == 2) mword = __brev(mword);
            if (kTrain == 2 && kBf16 && pt < p.ppad) {
              const bool live = pt < p.n_points;
              unsigned char* hb = p.a_h + (size_t)l * (size_t)p.ppad * (kWidth * 2);
#pragma unroll
              for (int c = 0; c < 4; ++c)
                *reinterpret_cast<uint4*>(hb + a16_cell(pt, (c0 >> 3) + c, kWidth)) =
                    live ? make_uint4(h16[4 * c], h16[4 * c + 1], h16[4 * c + 2], h16[4 * c + 3]) : make_uint4(0u, 0u, 0u, 0u);
            }
            mask_word = mword;
          };
          if (l == 7) finish_group(std::true_type{});
          else finish_group(std::false_type{});
          // half a's results go to A[k 0..127], which this layer's (b,k0) MMAs still read: the math above
          // overlaps both b phases, the stores wait until those MMAs have retired (a_free); half b's
          // target A[k 128..255] is idle
          if (h == 0) { mbar_wait(&s.a_free, ph_free); ph_free ^= 1; tc_fence_after(); }
          {
            uint32_t phi[16], plo[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) { phi[j] = v[2 * j]; plo[j] = v[2 * j + 1]; }
            tmem_st16(tbase + lane_base + kColAhi + (c0 >> 1), phi);
            if (kSplit) tmem_st16(tbase + lane_base + kColAlo + (c0 >> 1), plo);
            tmem_wait_st();
            tc_fence_before();
            signal(&s.a_ready[h * 2 + q]);
            trace(tr, tb + 3 + q);
            if (kTrain == 2 && pt < p.ppad) {
              // what the backward reads -- off the layer-to-layer critical path, after the hand-off.  fp16 modes: the saved
              // activation IS the hi word just stored to TMEM (rn_fp16 of the saturated value); bf16 modes stored theirs above
              const bool live = pt < p.n_points;
              if (!kBf16) {
                unsigned char* hb = p.a_h + (size_t)l * (size_t)p.ppad * (kWidth * 2);
#pragma unroll
                for (int c = 0; c < 4; ++c)
                  *reinterpret_cast<uint4*>(hb + a16_cell(pt, (c0 >> 3) + c, kWidth)) =
                      live ? make_uint4(phi[4 * c], phi[4 * c + 1], phi[4 * c + 2], phi[4 * c + 3]) : make_uint4(0u, 0u, 0u, 0u);
              }
              p.a_mask[a16_mask_index(l, c0 >> 5, pt, p.ppad)] = live ? mask_word : 0u;
            }
          }
        }
        // ---- background work in the idle window before this layer's next accumulator half is ready
        if (kDirTmem && pending && l < kDirPieces) {
          // the previous tile's direction-layer epilogue, one piece per layer; sigp[0] still holds that tile's sigma
          // (rewritten at l == 7 of this slot)
          const bool trp = (p.debug & 8) && blockIdx.x == 0 && slot == 4 && tid == 0;
          const long long dpt = tile_of(slot - 1) * kTile + row;
          if (l == 0) trace(trp, 1024 + 18 * 8 + 5);
          dir_piece(l, dpt, nullptr);
          if (l == kDirPieces - 1) {
            trace(trp, 1024 + 18 * 8 + 3);
            dir_finish(dpt);
            pending = false;
            trace(trp, 1024 + 18 * 8 + 4);
          }
        }
        if (l == 7) {
          // sigma head (nerf.py:136): combine the two column halves of each row
          s.sigp[ch][row] = sig_part;
          epi_bar_sync();
          if (ch == 0) {
            const float sg = ((s.sigp[0][row] + s.sigp[1][row]) + (s.sigp[2][row] + s.sigp[3][row])) + s.cst[CL.sigma_b];
            s.sigp[0][row] = sg;         // keep for the final float4
            if (p.sigma_only && pt < p.n_points) p.out[pt] = sg;
          }
          epi_bar_sync();
        }
      }
      if (p.sigma_only) continue;

      // ---------------- direction layer: accumulator full -> (drain) -> epilogue now or in the next slot
      {
        const bool tr = (p.debug & 8) && blockIdx.x == 0 && slot == 3 && tid == 0;
        const int tb = 1024 + 18 * 8;
        trace(tr, tb + 0);
        if (kDirTmem) { mbar_wait(&s.d_full_dir, (uint32_t)slot & 1); }
        else { mbar_wait(&s.d_full[0], ph_d & 1); ph_d ^= 1u; }
        tc_fence_after();
        trace(tr, tb + 1);
        if (kDirTmem) {
          pending = true;            // the accumulator is columns [384,512): nothing to drain
        } else {
          uint32_t v[32];
          tmem_ld32(tbase + lane_base + kColD + cdir0, v);
          tmem_wait_ld();
          tc_fence_before();
          signal(&s.d_drained);      // D[0,128) is in registers: the next slot's layer 1 may overwrite it
          trace(tr, tb + 2);
          dir_piece(0, pt_slot, v);
          trace(tr, tb + 3);
          dir_finish(pt_slot);
          trace(tr, tb + 4);
        }
        if (kDirTmem) trace(tr, tb + 2);
      }
    }
    if (kDirTmem && pending) {     // the last slot's direction-layer epilogue
      const long long dpt = tile_of(n_slots - 1) * kTile + row;
#pragma unroll 1
      for (int pc = 0; pc < kDirPieces; ++pc) dir_piece(pc, dpt, nullptr);
      dir_finish(dpt);
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // neither CTA leaves (or frees TMEM) while its peer may still touch it
  if (warp == kMmaWarp) tmem_dealloc_pair(tbase);
}

// ------------------------------------------------------------------ host
template <bool kBf16, bool kSplit, bool kEmbedded, int kTrain>
static int launch_tc(const TcParams& p, cudaStream_t st) {
  static SmemOptIn optin;
  const long long ntiles = (p.n_points + kTile - 1) / kTile;
  if (ntiles == 0) return SNB_OK;       // an empty pass is a no-op: no CUDA call at all
  const size_t smem = sizeof(TcSmem<kSplit, kTrain>) + 1024;
  auto kern = field_tc_kernel<kBf16, kSplit, kEmbedded, kTrain>;
  if (int rc = ensure_smem(kern, optin, (int)smem, "field_tc")) return rc;
  const int sms = sm_count();
  long long pairs = (ntiles + 1) / 2;
  if (pairs > sms / 2) pairs = sms / 2;
  static const int debug = getenv("SNB_TC_DEBUG") ? atoi(getenv("SNB_TC_DEBUG")) : 0;
  TcParams pd = p;
  pd.debug = debug;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(pairs * 2));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, pd);
  if (e != cudaSuccess) return fail(SNB_ERR_CUDA, "field_tc_kernel launch: %s", cudaGetErrorString(e));
  return check_launch("field_tc_kernel");
}

template <bool kEmbedded, int kTrain>
static int dispatch_tc(int precision, const TcParams& p, cudaStream_t st) {
  switch (precision) {
    case SNB_PREC_F16X3: return launch_tc<false, true, kEmbedded, kTrain>(p, st);
    case SNB_PREC_BF16X3: return launch_tc<true, true, kEmbedded, kTrain>(p, st);
    case SNB_PREC_BF16: return launch_tc<true, false, kEmbedded, kTrain>(p, st);
  }
  return fail(SNB_ERR_INVALID, "precision %d is not a tensor-core mode", precision);
}

int field_forward_tc(const void* packed, int precision, const float* rays, const float* z, int64_t n_rays,
                     int n_samples, int sigma_only, float* raw, cudaStream_t st) {
  TcParams p{};
  p.image = reinterpret_cast<const unsigned char*>(packed);
  p.rays = rays; p.z = z; p.n_samples = n_samples;
  p.n_points = (long long)n_rays * n_samples;
  p.sigma_only = sigma_only;
  p.out = raw;
  return dispatch_tc<false, 0>(precision, p, st);
}

int field_forward_train_tc(const void* packed, int precision, const float* rays, const float* z, int64_t n_rays,
                           int n_samples, float* raw, float* save_enc, float* save_dir, float* save_h, float* save_g,
                           cudaStream_t st) {
  TcParams p{};
  p.image = reinterpret_cast<const unsigned char*>(packed);
  p.rays = rays; p.z = z; p.n_samples = n_samples;
  p.n_points = (long long)n_rays * n_samples;
  p.out = raw;
  p.save_enc = save_enc; p.save_dir = save_dir; p.save_h = save_h; p.save_g = save_g;
  return dispatch_tc<false, 1>(precision, p, st);
}

// training forward with 16-bit activation storage (act16.cuh): `act16` = one buffer of make_act16_layout(P).total bytes
int field_forward_train16_tc(const void* packed, int precision, const float* rays, const float* z, int64_t n_rays,
                             int n_samples, float* raw, void* act16, cudaStream_t st) {
  TcParams p{};
  p.image = reinterpret_cast<const unsigned char*>(packed);
  p.rays = rays; p.z = z; p.n_samples = n_samples;
  p.n_points = (long long)n_rays * n_samples;
  p.out = raw;
  const Act16Layout L = make_act16_layout(p.n_points);
  unsigned char* b = reinterpret_cast<unsigned char*>(act16);
  p.a_enc = b + L.enc; p.a_dir = b + L.dir; p.a_h = b + L.h[0]; p.a_g = b + L.g;
  p.a_mask = reinterpret_cast<uint32_t*>(b + L.mask);
  p.ppad = a16_pad(p.n_points);
  return dispatch_tc<false, 2>(precision, p, st);
}

int mlp_forward_tc(const void* packed, int precision, const float* x, int64_t x_stride, int64_t n_points,
                   int sigma_only, float* out, cudaStream_t st) {
  TcParams p{};
  p.image = reinterpret_cast<const unsigned char*>(packed);
  p.x = x; p.x_stride = x_stride;
  p.n_points = n_points;
  p.sigma_only = sigma_only;
  p.out = out;
  return dispatch_tc<true, 0>(precision, p, st);
}

}  // namespace snb

// debug-only export (not part of the public header): copy the device trace buffer to the host
extern "C" int snb_debug_trace(long long* host_out, int n) {
  if (n > snb::kTraceLen) n = snb::kTraceLen;
  return cudaMemcpyFromSymbol(host_out, snb::g_trace, sizeof(long long) * n) == cudaSuccess ? 0 : -2;
}
