// SuperPoint key-point extractor for sm_100a (SURVEY 8f N4): the producer of the matcher's query descriptors.
// Replaces SuperPoint.forward (reference src/models/extractors/SuperPoint/superpoint.py:140-197) behind the C ABI
// opb_sp_* of include/onepose_b200.h.
//
// Data layout: an activation of c channels over an h x w grid lives as fp16-split planes [rows, c], one ROW PER PIXEL of
// a (h+2) x (w+2) grid with a ZERO BORDER (row of image b, pixel (y, x): b*P + (y+1)*(w+2) + (x+1); P = the grid padded to
// a multiple of 256 rows).  A 3x3 convolution is then an implicit GEMM on the tcgen05 core (gemm_tc.cu, EPI_CONV):
//     out[p, :] = sum_tap  A[p + dy*(w+2) + dx, :] . W_tap^T          9 row-shifted TMA loads of the SAME matrix,
// no im2col buffer; the epilogue adds the bias, applies ReLU and writes zeros on border / padding rows, so that its output is
// again a valid zero-bordered input.  Arithmetic: the same 3-pass fp16-split product as the matcher (fp32 semantics; the
// reference network is fp32).  Everything that is not a GEMM (first layer with one input channel, 2x2 pooling, 65-way softmax
// + pixel shuffle, NMS, ordered key-point compaction, top-k, bilinear descriptor sampling) is a plain bandwidth-bound kernel.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/onepose_b200.h"
#include "common.cuh"
#include "gemm_common.cuh"
#include "gemm_tc.cuh"
#include "host_util.cuh"

namespace opb {
namespace {

constexpr int kNmsTile = 32;
constexpr int kSelChunk = 2048;          // pixels per block of the key-point compaction (256 threads x 8 consecutive pixels)

// ------------------------------------------------------------------------------------------------------------------
// conv1a: 1 -> 64 channels, 3x3, ReLU (superpoint.py:111,142).  K = 9 is no tensor-core shape: thread = (pixel row, 8 output
// channels); writes the zero-bordered planes of the first GEMM layer.  img fp32 [B, H, W].
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sp_conv1a(const float* __restrict__ img, int H, int W, int ppad, const float* __restrict__ w,
                                                 const float* __restrict__ bias, __half* __restrict__ ohi, __half* __restrict__ olo) {
  griddep_sync();
  // grid (chunks of 256 grid pixels, image); thread = (pixel, 4-channel group g): g is fixed per thread (256 % 16 == 0), so its
  // 4 x 9 weights and 4 biases live in registers; 16 lanes = one 128-byte plane row per store instruction.  All index math is
  // 32-bit (a 64-bit division per pixel made the first version of this kernel instruction-bound).
  const int g = threadIdx.x & 15;
  float wr[4][9], br[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    br[e] = __ldg(bias + g * 4 + e);
#pragma unroll
    for (int k = 0; k < 9; ++k) wr[e][k] = __ldg(w + (g * 4 + e) * 9 + k);
  }
  const int b = blockIdx.y;
  const float* im = img + (size_t)b * H * W;
  const unsigned w2 = (unsigned)(W + 2);
  const size_t row_base = (size_t)b * ppad;
#pragma unroll 4
  for (int it = 0; it < 16; ++it) {
    const unsigned q = blockIdx.x * 256u + it * 16u + (threadIdx.x >> 4);
    if (q >= (unsigned)ppad) break;
    const unsigned yq = q / w2;
    const int y = (int)yq - 1, x = (int)(q - yq * w2) - 1;       // image coordinates
    uint2 oh = make_uint2(0, 0), ol = make_uint2(0, 0);
    if (y >= 0 && y < H && x >= 0 && x < W) {
      float in[9];
      if (y >= 1 && y < H - 1 && x >= 1 && x < W - 1) {           // interior (99 % of the pixels): nine unconditional loads
        const float* c = im + (y - 1) * W + (x - 1);
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) in[ky * 3 + kx] = __ldg(c + ky * W + kx);
      } else {
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) {
            const int yy = y + ky - 1, xx = x + kx - 1;
            in[ky * 3 + kx] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? __ldg(im + yy * W + xx) : 0.f;
          }
      }
      float v[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < 9; ++k) acc = fmaf(wr[e][k], in[k], acc);
        v[e] = fmaxf(acc + br[e], 0.f) * kPre;
      }
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const float2 sc = make_float2(v[2 * e], v[2 * e + 1]);
        const __half2 h2 = __float22half2_rn(sc);
        const float2 back = __half22float2(h2);
        reinterpret_cast<__half2*>(&oh)[e] = h2;
        reinterpret_cast<__half2*>(&ol)[e] = __float22half2_rn(make_float2(sc.x - back.x, sc.y - back.y));
      }
    }
    reinterpret_cast<uint2*>(ohi)[(row_base + q) * 16 + g] = oh;
    reinterpret_cast<uint2*>(olo)[(row_base + q) * 16 + g] = ol;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// 2x2 / stride-2 max pooling (superpoint.py:108,144) on fp16-split planes: thread = (output pixel row, 8 channels).  The
// maximum is taken on hi + lo (exact in fp32) and the winning (hi, lo) pair is copied, so pooling is exact on the split values.
// Output: zero-bordered grid of (hin/2) x (win/2), every row written (border / padding rows as zero).
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sp_pool2x2(const __half* __restrict__ ihi, const __half* __restrict__ ilo, int C, int hin, int win, int ppad_in,
                                                  __half* __restrict__ ohi, __half* __restrict__ olo, int ppad_out, long long rows_out) {
  griddep_sync();
  const int gpr = C / 8;                               // 8-channel groups per row
  const long long t = (long long)blockIdx.x * 256 + threadIdx.x;
  const long long row = t / gpr;
  const int g = (int)(t - row * gpr);
  if (row >= rows_out) return;
  const int ho = hin / 2, wo = win / 2;
  const int b = (int)(row / ppad_out), q = (int)(row - (long long)b * ppad_out);
  const int y = q / (wo + 2) - 1, x = q % (wo + 2) - 1;
  uint4 oh = make_uint4(0, 0, 0, 0), ol = make_uint4(0, 0, 0, 0);
  if (y >= 0 && y < ho && x >= 0 && x < wo) {
    float best[8];
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      const long long r = (long long)b * ppad_in + (long long)(2 * y + (d >> 1) + 1) * (win + 2) + (2 * x + (d & 1) + 1);
      const uint4 h = __ldg(reinterpret_cast<const uint4*>(ihi) + r * gpr + g);
      const uint4 l = __ldg(reinterpret_cast<const uint4*>(ilo) + r * gpr + g);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const __half hh = reinterpret_cast<const __half*>(&h)[e], ll = reinterpret_cast<const __half*>(&l)[e];
        const float val = __half2float(hh) + __half2float(ll);
        if (d == 0 || val > best[e]) {
          best[e] = val;
          reinterpret_cast<__half*>(&oh)[e] = hh;
          reinterpret_cast<__half*>(&ol)[e] = ll;
        }
      }
    }
  }
  reinterpret_cast<uint4*>(ohi)[row * gpr + g] = oh;
  reinterpret_cast<uint4*>(olo)[row * gpr + g] = ol;
}

// ------------------------------------------------------------------------------------------------------------------
// Dense scores (superpoint.py:156-160): softmax over the 65 logits of a coarse cell, dustbin dropped, the 64 probabilities
// laid out as the cell's 8 x 8 pixels.  Warp per cell; logits fp32 [rows, 128] (65 valid).  scores fp32 [B, 8h, 8w].
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sp_scores(const float* __restrict__ logits, int h, int w, int ppad, int B, float* __restrict__ scores) {
  griddep_sync();
  const long long cell = ((long long)blockIdx.x * 256 + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (cell >= (long long)B * h * w) return;
  const int b = (int)(cell / (h * w)), rem = (int)(cell - (long long)b * h * w);
  const int y = rem / w, x = rem - y * w;
  const float* src = logits + ((long long)b * ppad + (long long)(y + 1) * (w + 2) + (x + 1)) * 128;
  const float v0 = src[lane], v1 = src[lane + 32], v2 = lane == 0 ? src[64] : -INFINITY;
  float mx = fmaxf(fmaxf(v0, v1), v2);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  const float e0 = expf(v0 - mx), e1 = expf(v1 - mx), e2 = lane == 0 ? expf(v2 - mx) : 0.f;
  const float sum = warp_sum(e0 + e1 + e2);
  const int W = 8 * w;
  float* dst = scores + ((long long)b * 8 * h + 8 * y) * W + 8 * x;
  dst[(long long)(lane >> 3) * W + (lane & 7)] = e0 / sum;              // channel c -> pixel (c / 8, c % 8) of the cell
  dst[(long long)((lane + 32) >> 3) * W + (lane & 7)] = e1 / sum;
}

// ------------------------------------------------------------------------------------------------------------------
// simple_nms (superpoint.py:47-61), radius r, as ONE tiled pass: a 32 x 32 output tile needs the scores of a halo of 5 r
// pixels (max-pool of the scores: r; each of the two suppression rounds: mask pool r + pool of the suppressed scores r).
// Positions outside the image do not exist for torch's max_pool2d (implicit -inf padding): -inf scores / zero mask here.
// Separable running maximum over shrinking valid regions; shared memory: 6 float planes of (32 + 10 r)^2.
// ------------------------------------------------------------------------------------------------------------------
// Work distribution inside the tile: one warp per row of the region, lanes over columns -- no integer divisions (the first
// version indexed a flattened range with / and % per element and was instruction-bound).
#define SP_FOR_REGION(lo_, hi_, ...)                                                           \
  for (int y = (lo_) + (int)(threadIdx.x >> 5); y < (hi_); y += (int)(blockDim.x >> 5))          \
    for (int x = (lo_) + (int)(threadIdx.x & 31); x < (hi_); x += 32) { __VA_ARGS__ }

__device__ __forceinline__ void pool_sep(const float* in, float* tmp, float* out, int D, int margin, int r) {
  // out = max over the (2r+1)^2 window of `in`, valid on [margin + r, D - margin - r)^2 given `in` valid on [margin, D - margin)^2
  const int lo = margin, hi = D - margin;
  for (int y = lo + (int)(threadIdx.x >> 5); y < hi; y += (int)(blockDim.x >> 5))
    for (int x = lo + r + (int)(threadIdx.x & 31); x < hi - r; x += 32) {
      const float* p = in + y * D + x;
      float m = p[-r];
      for (int d = -r + 1; d <= r; ++d) m = fmaxf(m, p[d]);
      tmp[y * D + x] = m;
    }
  __syncthreads();
  SP_FOR_REGION(lo + r, hi - r, {
    const float* p = tmp + y * D + x;
    float m = p[-r * D];
    for (int d = -r + 1; d <= r; ++d) m = fmaxf(m, p[d * D]);
    out[y * D + x] = m;
  })
  __syncthreads();
}

__global__ void __launch_bounds__(512) sp_nms(const float* __restrict__ scores, int H, int W, int r, float* __restrict__ out) {
  extern __shared__ float nms_smem[];
  const int halo = 5 * r, D = kNmsTile + 2 * halo, DD = D * D;
  float* S = nms_smem;            // scores (-inf outside the image)
  float* T = S + DD;              // scratch of the separable pool
  float* P = T + DD;              // pooled scores
  float* Mk = P + DD;             // max_mask as 0 / 1
  float* Sup = Mk + DD;           // pooled mask (> 0: suppressed)
  float* SS = Sup + DD;           // supp_scores
  griddep_sync();
  const int b = blockIdx.z;
  const int y0 = blockIdx.y * kNmsTile - halo, x0 = blockIdx.x * kNmsTile - halo;
  const float* src = scores + (size_t)b * H * W;
  SP_FOR_REGION(0, D, {
    const int gy = y0 + y, gx = x0 + x;
    S[y * D + x] = (gy >= 0 && gy < H && gx >= 0 && gx < W) ? src[gy * W + gx] : -INFINITY;
    Mk[y * D + x] = 0.f;
  })
  __syncthreads();
  pool_sep(S, T, P, D, 0, r);                                   // valid on margin r
  int margin = r;
  SP_FOR_REGION(margin, D - margin, {
    const int k = y * D + x;
    Mk[k] = (S[k] == P[k] && S[k] != -INFINITY) ? 1.f : 0.f;    // max_mask = scores == max_pool(scores)
  })
  __syncthreads();
  for (int it = 0; it < 2; ++it) {
    pool_sep(Mk, T, Sup, D, margin, r);                         // supp_mask = max_pool(max_mask.float()) > 0
    margin += r;
    SP_FOR_REGION(margin, D - margin, {
      const int k = y * D + x;
      SS[k] = S[k] == -INFINITY ? -INFINITY : (Sup[k] > 0.f ? 0.f : S[k]);     // supp_scores = where(supp_mask, 0, scores)
    })
    __syncthreads();
    pool_sep(SS, T, P, D, margin, r);
    margin += r;
    SP_FOR_REGION(margin, D - margin, {
      const int k = y * D + x;
      if (!(Sup[k] > 0.f) && SS[k] == P[k] && S[k] != -INFINITY) Mk[k] = 1.f;   // max_mask |= new_max_mask & ~supp_mask
    })
    __syncthreads();
  }
  float* dst = out + (size_t)b * H * W;
  SP_FOR_REGION(halo, halo + kNmsTile, {
    const int gy = y0 + y, gx = x0 + x;
    if (gy < H && gx < W) {
      const int k = y * D + x;
      dst[gy * W + gx] = Mk[k] == 1.f ? S[k] : 0.f;             // torch.where(max_mask, scores, zeros)
    }
  })
}
#undef SP_FOR_REGION

// ------------------------------------------------------------------------------------------------------------------
// Key-point selection (superpoint.py:163-174): pixels with nms score > threshold, inside the border margin, in row-major
// order (torch.nonzero).  Two passes over 2048-pixel chunks: per-chunk counts, then an ordered compaction.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool sp_keep(float s, int pix, int H, int W, float thr, int border) {
  const int y = pix / W, x = pix - y * W;
  return s > thr && y >= border && y < H - border && x >= border && x < W - border;
}

__global__ void __launch_bounds__(256) sp_count(const float* __restrict__ nms, int H, int W, float thr, int border, int* __restrict__ blk_counts) {
  __shared__ int wsum[8];
  griddep_sync();
  const int b = blockIdx.y, HW = H * W;
  const int p0 = blockIdx.x * kSelChunk + threadIdx.x * 8;
  int c = 0;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int p = p0 + e;
    if (p < HW && sp_keep(nms[(long long)b * HW + p], p, H, W, thr, border)) ++c;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int i = 0; i < 8; ++i) s += wsum[i];
    blk_counts[b * gridDim.x + blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(256) sp_compact(const float* __restrict__ nms, int H, int W, float thr, int border, const int* __restrict__ blk_counts,
                                                  int* __restrict__ cand_idx, float* __restrict__ cand_score, int* __restrict__ totals) {
  __shared__ int wsum[8];
  __shared__ int base_s;
  griddep_sync();
  const int b = blockIdx.y, HW = H * W;
  if (threadIdx.x < 32) {                                       // chunks in front of this one
    int s = 0;
    for (int i = threadIdx.x; i < (int)blockIdx.x; i += 32) s += blk_counts[b * gridDim.x + i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (threadIdx.x == 0) base_s = s;
  }
  const int p0 = blockIdx.x * kSelChunk + threadIdx.x * 8;
  float sv[8];
  unsigned keep = 0;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int p = p0 + e;
    sv[e] = p < HW ? nms[(long long)b * HW + p] : 0.f;
    if (p < HW && sp_keep(sv[e], p, H, W, thr, border)) keep |= 1u << e;
  }
  const int c = __popc(keep);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int incl = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  if (lane == 31) wsum[wid] = incl;
  __syncthreads();
  int off = base_s + incl - c;
  for (int i = 0; i < wid; ++i) off += wsum[i];
#pragma unroll
  for (int e = 0; e < 8; ++e)
    if (keep & (1u << e)) {
      cand_idx[(long long)b * HW + off] = p0 + e;
      cand_score[(long long)b * HW + off] = sv[e];
      ++off;
    }
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 255) totals[b] = off;
}

// Emission: all candidates in row-major order, or -- if there are more than k -- the k highest scores in descending order
// (torch.topk, superpoint.py:72-76; equal scores: lower pixel index first).  Rank by counting: candidate i goes to position
// #{j : key_j > key_i}; O(n^2) comparisons on at most a few 10^4 candidates.  Key points are (x, y) floats (superpoint.py:177).
__global__ void __launch_bounds__(256) sp_emit(const int* __restrict__ cand_idx, const float* __restrict__ cand_score, const int* __restrict__ totals, int HW,
                                               int W, int k, int cap, float* __restrict__ kpts, float* __restrict__ kscores, int* __restrict__ counts) {
  // key = (score bits, ~pixel index): scores are positive floats (> threshold >= 0 is not required: the sign bit is flipped
  // into an order-preserving unsigned), so one 64-bit compare orders by (score descending, index ascending)
  __shared__ unsigned long long tk[1024];
  griddep_sync();
  const int b = blockIdx.y;
  const int total = totals[b];
  const int sel = (k >= 0 && total > k) ? k : total;
  const int n_out = sel < cap ? sel : cap;
  if (blockIdx.x == 0 && threadIdx.x == 0) counts[b] = n_out;
  const int i0 = blockIdx.x * 256;
  if (i0 >= total) return;
  const int i = i0 + threadIdx.x;
  const bool live = i < total;
  const float si = live ? cand_score[(long long)b * HW + i] : 0.f;
  const int pi = live ? cand_idx[(long long)b * HW + i] : 0;
  auto make_key = [](float s, int p) {
    unsigned u = __float_as_uint(s);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);               // monotone float -> unsigned
    return ((unsigned long long)u << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)p);
  };
  int pos = i;
  if (k >= 0 && total > k) {
    const unsigned long long ki = make_key(si, pi);
    int rank = 0;
    for (int j0 = 0; j0 < total; j0 += 1024) {
      __syncthreads();
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + u * 256 + threadIdx.x;
        tk[u * 256 + threadIdx.x] = j < total ? make_key(cand_score[(long long)b * HW + j], cand_idx[(long long)b * HW + j]) : 0ull;
      }
      __syncthreads();
      const int lim = min(1024, total - j0);
      int t = 0;
      for (; t + 4 <= lim; t += 4) {                               // broadcast reads: two keys per 16-byte load
        const ulonglong2 a = *reinterpret_cast<const ulonglong2*>(&tk[t]);
        const ulonglong2 c = *reinterpret_cast<const ulonglong2*>(&tk[t + 2]);
        rank += (a.x > ki) + (a.y > ki) + (c.x > ki) + (c.y > ki);
      }
      for (; t < lim; ++t) rank += tk[t] > ki;
    }
    pos = rank;
  }
  if (live && pos < n_out) {
    const int y = pi / W, x = pi - y * W;
    kpts[((long long)b * cap + pos) * 2 + 0] = (float)x;
    kpts[((long long)b * cap + pos) * 2 + 1] = (float)y;
    kscores[(long long)b * cap + pos] = si;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// sample_descriptors (superpoint.py:79-92): the dense descriptors are L2-normalised per coarse cell (:181), sampled bilinearly
// at the key points (grid_sample, zero padding) and normalised again.  Warp per key point, lane = 8 channels; the four
// neighbour cells are normalised on the fly (the dense normalised map is never written).  ddesc fp32 [rows, 256] in the
// zero-bordered grid of the coarse stage; out fp32 [B, 256, cap] (channel-first like the reference's [256, n]).
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sp_sample(const float* __restrict__ ddesc, int h, int w, int ppad, const float* __restrict__ kpts,
                                                 const int* __restrict__ counts, int cap, int align_corners, float* __restrict__ out) {
  griddep_sync();
  const int b = blockIdx.y;
  const int i = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= counts[b]) return;
  const float kx = kpts[((long long)b * cap + i) * 2], ky = kpts[((long long)b * cap + i) * 2 + 1];
  const float s = 8.f;
  // keypoints - s/2 + 0.5;  / (w*s - s/2 - 0.5);  *2 - 1   -- the reference's own fp32 operation order
  float gx = (kx - s / 2 + 0.5f) / (w * s - s / 2 - 0.5f);
  float gy = (ky - s / 2 + 0.5f) / (h * s - s / 2 - 0.5f);
  gx = gx * 2.f - 1.f;
  gy = gy * 2.f - 1.f;
  // grid_sample un-normalisation (ATen grid_sampler_unnormalize)
  const float ix = align_corners ? ((gx + 1.f) / 2.f) * (w - 1) : ((gx + 1.f) * w - 1.f) / 2.f;
  const float iy = align_corners ? ((gy + 1.f) / 2.f) * (h - 1) : ((gy + 1.f) * h - 1.f) / 2.f;
  const float fx = floorf(ix), fy = floorf(iy);
  const int x0 = (int)fx, y0 = (int)fy;
  const float wx1 = ix - fx, wy1 = iy - fy, wx0 = 1.f - wx1, wy0 = 1.f - wy1;     // ATen: nw = (ix_se - ix) * (iy_se - iy), ...
  const float wgt[4] = {wx0 * wy0, wx1 * wy0, wx0 * wy1, wx1 * wy1};
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int d = 0; d < 4; ++d) {
    const int yy = y0 + (d >> 1), xx = x0 + (d & 1);
    if (yy < 0 || yy >= h || xx < 0 || xx >= w) continue;       // warp-uniform: zero padding
    const float4* src = reinterpret_cast<const float4*>(ddesc + ((long long)b * ppad + (long long)(yy + 1) * (w + 2) + (xx + 1)) * 256) + lane * 2;
    const float4 a = __ldg(src), c = __ldg(src + 1);
    const float v[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
    float ss = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) ss = fmaf(v[e], v[e], ss);
    ss = warp_sum(ss);
    const float inv = 1.f / fmaxf(sqrtf(ss), 1e-12f);          // F.normalize(p=2, dim=1, eps=1e-12)
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = fmaf(v[e] * inv, wgt[d], acc[e]);
  }
  float ss = 0.f;
#pragma unroll
  for (int e = 0; e < 8; ++e) ss = fmaf(acc[e], acc[e], ss);
  ss = warp_sum(ss);
  const float inv = 1.f / fmaxf(sqrtf(ss), 1e-12f);
#pragma unroll
  for (int e = 0; e < 8; ++e) out[((long long)b * 256 + lane * 8 + e) * cap + i] = acc[e] * inv;
}

__global__ void sp_counts_out(const int* __restrict__ totals, int k, int n, int* __restrict__ counts) {
  griddep_sync();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) counts[i] = (k >= 0 && totals[i] > k) ? k : totals[i];
}

__global__ void sp_join_planes(const __half* __restrict__ hi, const __half* __restrict__ lo, float* __restrict__ out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = join_f32(hi[i], lo[i]);
}

}  // namespace
}  // namespace opb

using namespace opb;

struct SpConv {
  PlaneBuf w;        // [cout, taps * cin]
  DevBuf b;          // [cout]
  int cin = 0, cout = 0, bn = 0, taps = 0;
};

struct opb_superpoint : HostState {
  opb_sp_config cfg{};
  bool ready = false;
  DevBuf w1a, b1a;                 // fp32 [64][9], [64]
  SpConv c1b, c2a, c2b, c3a, c3b, c4a, c4b, cPD, cPb, cDb;
  // workspace
  int ws_B = 0, ws_H = 0, ws_W = 0;
  PlaneBuf arena[2];               // ping-pong activations
  DevBuf logits, ddesc, scores, nms, cand_idx, cand_score, blk_counts, totals;
  int last_B = 0, last_H = 0, last_W = 0;
  int stop_after = -1;             // test hook: leave the encoder after layer i (opb_sp_debug_set_stop)
  int dbg_arena = 0, dbg_c = 0;
  long long dbg_rows = 0;
};

namespace {

// Pack one or two conv layers [cout, cin, k, k] (k = 3 or 1) that share their input into the B operand [cout_total (padded to
// cout_pad), taps*cin] with reduction index tap*cin + c (tap = ky*3 + kx), plus the bias.
int sp_pack(opb_superpoint* h, SpConv& L, const std::vector<std::string>& names, int cin, const std::vector<int>& couts, int ksz, int cout_pad, int bn) {
  const int taps = ksz * ksz;
  const size_t K = (size_t)taps * cin;
  std::vector<double> w((size_t)cout_pad * K, 0.0);
  std::vector<float> b(cout_pad, 0.f);
  int row0 = 0;
  for (size_t li = 0; li < names.size(); ++li) {
    const int cout = couts[li];
    const std::vector<float> *ww, *bb;
    if (int rc = find_w(h, names[li] + ".weight", (size_t)cout * cin * taps, ww)) return rc;
    if (int rc = find_w(h, names[li] + ".bias", (size_t)cout, bb)) return rc;
    for (int n = 0; n < cout; ++n) {
      for (int c = 0; c < cin; ++c)
        for (int t = 0; t < taps; ++t) w[(size_t)(row0 + n) * K + (size_t)t * cin + c] = (*ww)[((size_t)n * cin + c) * taps + t];
      b[row0 + n] = (*bb)[n];
    }
    row0 += cout;
  }
  L.cin = cin; L.cout = cout_pad; L.bn = bn; L.taps = taps;
  if (int rc = upload_planes(h, L.w, w)) return rc;
  return upload_f32(h, L.b, b);
}

struct Stage {
  int h, w, ppad;
  long long rows(int B) const { return (long long)B * ppad; }
};
Stage stage_of(int H, int W, int s) {
  Stage g;
  g.h = H >> s; g.w = W >> s;
  g.ppad = round_up((g.h + 2) * (g.w + 2), 256);
  return g;
}

int sp_ensure_workspace(opb_superpoint* h, int B, int H, int W) {
  if (B <= h->ws_B && H * W <= h->ws_H * h->ws_W && h->ws_H == H && h->ws_W == W) return 0;
  const int Bc = B > h->ws_B ? B : h->ws_B;
  const Stage s0 = stage_of(H, W, 0), s3 = stage_of(H, W, 3);
  const size_t elems = (size_t)Bc * s0.ppad * 64;           // the largest activation: 64 channels at full resolution
  const size_t head = (size_t)Bc * s3.ppad * 512;
  for (int i = 0; i < 2; ++i) CK(h, h->arena[i].ensure(elems > head ? elems : head));
  CK(h, h->logits.ensure((size_t)Bc * s3.ppad * 128 * sizeof(float)));
  CK(h, h->ddesc.ensure((size_t)Bc * s3.ppad * 256 * sizeof(float)));
  const size_t HW = (size_t)H * W;
  CK(h, h->scores.ensure(Bc * HW * sizeof(float)));
  CK(h, h->nms.ensure(Bc * HW * sizeof(float)));
  CK(h, h->cand_idx.ensure(Bc * HW * sizeof(int)));
  CK(h, h->cand_score.ensure(Bc * HW * sizeof(float)));
  CK(h, h->blk_counts.ensure((size_t)Bc * ((HW + kSelChunk - 1) / kSelChunk) * sizeof(int)));
  CK(h, h->totals.ensure((size_t)Bc * sizeof(int)));
  CK(h, cudaDeviceSynchronize());
  h->ws_B = Bc; h->ws_H = H; h->ws_W = W;
  return 0;
}

int sp_run_conv(opb_superpoint* h, const SpConv& L, const PlaneBuf& in, int in_ld, size_t in_off, const PlaneBuf* outp, float* outf, int out_ld,
                const Stage& g, int B, int relu, cudaStream_t st, const char* name) {
  GemmProblem p{};
  p.a1 = in.c(in_ld, in_off);
  p.b1 = L.w.c(L.taps * L.cin);
  p.K1 = L.taps * L.cin;
  p.rows = (int)g.rows(B);
  p.n_out = L.cout;
  p.bn = L.bn;
  p.batch = 1;
  p.bias = L.b.as<float>();
  if (outp) {
    p.epi = EPI_CONV;
    p.out = outp->m(out_ld);
    p.cv_w2 = g.w + 2; p.cv_h = g.h; p.cv_w = g.w; p.cv_ppad = g.ppad; p.relu = relu;
    if (L.taps == 9) {
      p.taps = 9; p.kb_per_tap = L.cin / 64;
      for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx) p.tap_off[ky * 3 + kx] = (ky - 1) * (g.w + 2) + (kx - 1);
    } else {
      p.taps = 1; p.kb_per_tap = L.cin / 64; p.tap_off[0] = 0;
    }
  } else {
    p.epi = EPI_F32;
    p.c = outf;
    p.ldc = out_ld;
  }
  // algorithmic FLOPs: interior pixels only
  return run_gemm(h, p, st, 2.0 * B * g.h * g.w * (double)L.cout * L.taps * L.cin, name);
}

}  // namespace

extern "C" {

int opb_sp_create(const opb_sp_config* cfg, opb_superpoint** out) {
  if (!cfg || !out) return fail(nullptr, OPB_E_INVALID, "null argument");
  if (cfg->descriptor_dim != 256) return fail(nullptr, OPB_E_INVALID, "descriptor_dim %d: only 256 is supported", cfg->descriptor_dim);
  if (cfg->max_keypoints == 0 || cfg->max_keypoints < -1) return fail(nullptr, OPB_E_INVALID, "\"max_keypoints\" must be positive or \"-1\"");
  if (cfg->nms_radius < 0 || cfg->nms_radius > 6) return fail(nullptr, OPB_E_NOT_IMPLEMENTED, "nms_radius %d: the tiled NMS supports 0..6", cfg->nms_radius);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= cfg->device) return fail(nullptr, OPB_E_CUDA, "no CUDA device %d", cfg->device);
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, cfg->device);
  if (prop.major != 10) return fail(nullptr, OPB_E_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", cfg->device, prop.major, prop.minor);
  if (cudaSetDevice(cfg->device) != cudaSuccess) return fail(nullptr, OPB_E_CUDA, "cudaSetDevice failed");
  auto* h = new opb_superpoint();
  h->cfg = *cfg;
  h->device = cfg->device;
  *out = h;
  return OPB_OK;
}

void opb_sp_destroy(opb_superpoint* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  for (SpConv* L : {&h->c1b, &h->c2a, &h->c2b, &h->c3a, &h->c3b, &h->c4a, &h->c4b, &h->cPD, &h->cPb, &h->cDb}) { L->w.release(); L->b.release(); }
  h->w1a.release(); h->b1a.release();
  h->arena[0].release(); h->arena[1].release();
  for (DevBuf* d : {&h->logits, &h->ddesc, &h->scores, &h->nms, &h->cand_idx, &h->cand_score, &h->blk_counts, &h->totals}) d->release();
  delete h;
}

const char* opb_sp_last_error(const opb_superpoint* h) { return h ? h->err.c_str() : g_last_error.c_str(); }

int opb_sp_load_weight(opb_superpoint* h, const char* name, const float* data, size_t n_elems) {
  ENTER(h);
  if (!name || !data) return fail(h, OPB_E_INVALID, "opb_sp_load_weight: null argument");
  h->host_w[name].assign(data, data + n_elems);
  h->ready = false;
  return OPB_OK;
}

int opb_sp_finalize_weights(opb_superpoint* h) {
  ENTER(h);
  const std::vector<float> *w1, *b1;
  if (int rc = find_w(h, "conv1a.weight", 64 * 9, w1)) return rc;
  if (int rc = find_w(h, "conv1a.bias", 64, b1)) return rc;
  if (int rc = upload_f32(h, h->w1a, *w1)) return rc;
  if (int rc = upload_f32(h, h->b1a, *b1)) return rc;
  if (int rc = sp_pack(h, h->c1b, {"conv1b"}, 64, {64}, 3, 64, 64)) return rc;
  if (int rc = sp_pack(h, h->c2a, {"conv2a"}, 64, {64}, 3, 64, 64)) return rc;
  if (int rc = sp_pack(h, h->c2b, {"conv2b"}, 64, {64}, 3, 64, 64)) return rc;
  if (int rc = sp_pack(h, h->c3a, {"conv3a"}, 64, {128}, 3, 128, 128)) return rc;
  if (int rc = sp_pack(h, h->c3b, {"conv3b"}, 128, {128}, 3, 128, 128)) return rc;
  if (int rc = sp_pack(h, h->c4a, {"conv4a"}, 128, {128}, 3, 128, 128)) return rc;
  if (int rc = sp_pack(h, h->c4b, {"conv4b"}, 128, {128}, 3, 128, 128)) return rc;
  // the two heads' 3x3 layers read the same tensor: ONE GEMM with 512 output channels [convPa | convDa]
  // (128-wide column tiles although C_out = 512 / 256: the narrow tiles keep the correction passes in their own accumulator)
  if (int rc = sp_pack(h, h->cPD, {"convPa", "convDa"}, 128, {256, 256}, 3, 512, 128)) return rc;
  if (int rc = sp_pack(h, h->cPb, {"convPb"}, 256, {65}, 1, 128, 128)) return rc;
  if (int rc = sp_pack(h, h->cDb, {"convDb"}, 256, {256}, 1, 256, 128)) return rc;
  CK(h, cudaDeviceSynchronize());
  h->ready = true;
  return OPB_OK;
}

int opb_sp_detect(opb_superpoint* h, const float* image, int32_t B, int32_t H, int32_t W, int32_t* counts, void* stream) {
  ENTER(h);
  if (!image || B <= 0 || H <= 0 || W <= 0) return fail(h, OPB_E_INVALID, "bad argument");
  if (!h->ready) return fail(h, OPB_E_STATE, "weights not finalized");
  if (H % 8 || W % 8) return fail(h, OPB_E_INVALID, "image size %dx%d: height and width must be multiples of 8 (three 2x2 poolings)", H, W);
  if ((long long)B * stage_of(H, W, 0).ppad > 0x7fffff00LL) return fail(h, OPB_E_INVALID, "batch too large for 32-bit row indices");
  if (int rc = sp_ensure_workspace(h, B, H, W)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  begin_call(h, st);
  const Stage s0 = stage_of(H, W, 0), s1 = stage_of(H, W, 1), s2 = stage_of(H, W, 2), s3 = stage_of(H, W, 3);
  PlaneBuf& A = h->arena[0];
  PlaneBuf& Bf = h->arena[1];
  auto blocks = [](long long threads) { return dim3((unsigned)((threads + 255) / 256)); };
  // test hook (opb_sp_debug_set_stop): leave after encoder step `idx`, remembering where its activation lives
  auto stopped = [&](int idx, int arena_idx, int C, const Stage& g) {
    h->dbg_arena = arena_idx; h->dbg_c = C; h->dbg_rows = g.rows(B);
    h->last_B = B; h->last_H = H; h->last_W = W;
    return h->stop_after == idx;
  };
  // ---- shared encoder (superpoint.py:142-152)
  LAUNCH(h, st, "sp_conv1a", sp_conv1a, dim3((s0.ppad + 255) / 256, B), dim3(256), 0, st, image, (int)H, (int)W, s0.ppad, (const float*)h->w1a.as<float>(),
         (const float*)h->b1a.as<float>(), A.hi.as<__half>(), A.lo.as<__half>());
  if (stopped(0, 0, 64, s0)) return OPB_OK;
  if (int rc = sp_run_conv(h, h->c1b, A, 64, 0, &Bf, nullptr, 64, s0, B, 1, st, "conv1b")) return rc;
  if (stopped(1, 1, 64, s0)) return OPB_OK;
  LAUNCH(h, st, "sp_pool2x2", sp_pool2x2, blocks(s1.rows(B) * 8), dim3(256), 0, st, (const __half*)Bf.hi.as<__half>(), (const __half*)Bf.lo.as<__half>(), 64,
         s0.h, s0.w, s0.ppad, A.hi.as<__half>(), A.lo.as<__half>(), s1.ppad, s1.rows(B));
  if (stopped(2, 0, 64, s1)) return OPB_OK;
  if (int rc = sp_run_conv(h, h->c2a, A, 64, 0, &Bf, nullptr, 64, s1, B, 1, st, "conv2a")) return rc;
  if (stopped(3, 1, 64, s1)) return OPB_OK;
  if (int rc = sp_run_conv(h, h->c2b, Bf, 64, 0, &A, nullptr, 64, s1, B, 1, st, "conv2b")) return rc;
  if (stopped(4, 0, 64, s1)) return OPB_OK;
  LAUNCH(h, st, "sp_pool2x2", sp_pool2x2, blocks(s2.rows(B) * 8), dim3(256), 0, st, (const __half*)A.hi.as<__half>(), (const __half*)A.lo.as<__half>(), 64,
         s1.h, s1.w, s1.ppad, Bf.hi.as<__half>(), Bf.lo.as<__half>(), s2.ppad, s2.rows(B));
  if (stopped(5, 1, 64, s2)) return OPB_OK;
  if (int rc = sp_run_conv(h, h->c3a, Bf, 64, 0, &A, nullptr, 128, s2, B, 1, st, "conv3a")) return rc;
  if (stopped(6, 0, 128, s2)) return OPB_OK;
  if (int rc = sp_run_conv(h, h->c3b, A, 128, 0, &Bf, nullptr, 128, s2, B, 1, st, "conv3b")) return rc;
  if (stopped(7, 1, 128, s2)) return OPB_OK;
  LAUNCH(h, st, "sp_pool2x2", sp_pool2x2, blocks(s3.rows(B) * 16), dim3(256), 0, st, (const __half*)Bf.hi.as<__half>(), (const __half*)Bf.lo.as<__half>(), 128,
         s2.h, s2.w, s2.ppad, A.hi.as<__half>(), A.lo.as<__half>(), s3.ppad, s3.rows(B));
  if (stopped(8, 0, 128, s3)) return OPB_OK;
  if (int rc = sp_run_conv(h, h->c4a, A, 128, 0, &Bf, nullptr, 128, s3, B, 1, st, "conv4a")) return rc;
  if (stopped(9, 1, 128, s3)) return OPB_OK;
  if (int rc = sp_run_conv(h, h->c4b, Bf, 128, 0, &A, nullptr, 128, s3, B, 1, st, "conv4b")) return rc;
  if (stopped(10, 0, 128, s3)) return OPB_OK;
  // ---- heads (superpoint.py:155-156, :180-181): [convPa | convDa] in one GEMM, then the two 1x1 layers as plain GEMMs
  if (int rc = sp_run_conv(h, h->cPD, A, 128, 0, &Bf, nullptr, 512, s3, B, 1, st, "convPa|convDa")) return rc;
  if (stopped(11, 1, 512, s3)) return OPB_OK;
  if (int rc = sp_run_conv(h, h->cPb, Bf, 512, 0, nullptr, h->logits.as<float>(), 128, s3, B, 0, st, "convPb")) return rc;
  if (int rc = sp_run_conv(h, h->cDb, Bf, 512, 256, nullptr, h->ddesc.as<float>(), 256, s3, B, 0, st, "convDb")) return rc;
  // ---- dense scores, NMS, key-point selection (superpoint.py:157-174)
  LAUNCH(h, st, "sp_scores", sp_scores, blocks((long long)B * s3.h * s3.w * 32), dim3(256), 0, st, (const float*)h->logits.as<float>(), s3.h, s3.w, s3.ppad, (int)B,
         h->scores.as<float>());
  {
    const int r = h->cfg.nms_radius, D = kNmsTile + 10 * r;
    const size_t smem = (size_t)6 * D * D * sizeof(float);
    CK(h, ensure_smem_attr((const void*)sp_nms, (int)smem));
    LAUNCH(h, st, "sp_nms", sp_nms, dim3((W + kNmsTile - 1) / kNmsTile, (H + kNmsTile - 1) / kNmsTile, B), dim3(512), smem, st,
           (const float*)h->scores.as<float>(), (int)H, (int)W, r, h->nms.as<float>());
  }
  const int HW = H * W, nchunks = (HW + kSelChunk - 1) / kSelChunk;
  LAUNCH(h, st, "sp_count", sp_count, dim3(nchunks, B), dim3(256), 0, st, (const float*)h->nms.as<float>(), (int)H, (int)W, h->cfg.keypoint_threshold,
         h->cfg.remove_borders, h->blk_counts.as<int>());
  LAUNCH(h, st, "sp_compact", sp_compact, dim3(nchunks, B), dim3(256), 0, st, (const float*)h->nms.as<float>(), (int)H, (int)W, h->cfg.keypoint_threshold,
         h->cfg.remove_borders, (const int*)h->blk_counts.as<int>(), h->cand_idx.as<int>(), h->cand_score.as<float>(), h->totals.as<int>());
  h->last_B = B; h->last_H = H; h->last_W = W;
  if (counts)     // number of key points opb_sp_describe will emit: min(total, max_keypoints)
    LAUNCH(h, st, "sp_counts_out", sp_counts_out, dim3((B + 127) / 128), dim3(128), 0, st, (const int*)h->totals.as<int>(), h->cfg.max_keypoints, (int)B, counts);
  return OPB_OK;
}

int opb_sp_describe(opb_superpoint* h, float* keypoints, float* scores, float* descriptors, int32_t* counts, int32_t cap, void* stream) {
  ENTER(h);
  if (!keypoints || !scores || !counts || cap <= 0) return fail(h, OPB_E_INVALID, "bad argument");
  if (!h->last_B) return fail(h, OPB_E_STATE, "opb_sp_describe without a preceding opb_sp_detect");
  cudaStream_t st = (cudaStream_t)stream;
  const int B = h->last_B, H = h->last_H, W = h->last_W, HW = H * W;
  const Stage s3 = stage_of(H, W, 3);
  LAUNCH(h, st, "sp_emit", sp_emit, dim3((HW + 255) / 256, B), dim3(256), 0, st, (const int*)h->cand_idx.as<int>(), (const float*)h->cand_score.as<float>(),
         (const int*)h->totals.as<int>(), HW, W, h->cfg.max_keypoints, (int)cap, keypoints, scores, counts);
  if (descriptors)
    LAUNCH(h, st, "sp_sample", sp_sample, dim3(((long long)cap * 32 + 255) / 256, B), dim3(256), 0, st, (const float*)h->ddesc.as<float>(), s3.h, s3.w, s3.ppad,
           (const float*)keypoints, (const int*)counts, (int)cap, h->cfg.align_corners, descriptors);
  return OPB_OK;
}

int opb_sp_forward(opb_superpoint* h, const float* image, int32_t B, int32_t H, int32_t W, float* keypoints, float* scores, float* descriptors,
                   int32_t* counts, int32_t cap, void* stream) {
  if (int rc = opb_sp_detect(h, image, B, H, W, nullptr, stream)) return rc;
  return opb_sp_describe(h, keypoints, scores, descriptors, counts, cap, stream);
}

int opb_sp_last_launch_count(const opb_superpoint* h) { return h ? h->launches : 0; }

int opb_sp_set_profiling(opb_superpoint* h, int32_t enable) {
  ENTER(h);
  h->profiling = enable != 0;
  return OPB_OK;
}

int opb_sp_get_profile(opb_superpoint* h, int32_t index, char* name, size_t name_cap, double* ms, double* flops) {
  ENTER(h);
  if (index < 0 || (size_t)index >= h->ev_name.size())                 // past the end: the caller's loop over the entries stops here
    return fail(h, OPB_E_INVALID, "opb_sp_get_profile: no entry %d (%zu launches logged)", index, h->ev_name.size());
  CK(h, cudaEventSynchronize(h->ev[index + 1]));
  float t = 0.f;
  if (int rc = entry_ms(h, index, &t)) return rc;
  if (ms) *ms = t;
  if (flops) *flops = h->ev_flops[index];
  if (name && name_cap) { strncpy(name, h->ev_name[index].c_str(), name_cap - 1); name[name_cap - 1] = 0; }
  return OPB_OK;
}

int opb_debug_set_conv_halo(int32_t mode) {
  if (mode < 0 || mode > 1) return fail(nullptr, OPB_E_INVALID, "%s: mode %d is not 0 or 1", __func__, mode);
  set_conv_halo_mode(mode);
  return OPB_OK;
}

int opb_sp_debug_set_stop(opb_superpoint* h, int32_t layer) {
  ENTER(h);
  h->stop_after = layer;
  return OPB_OK;
}

int opb_sp_debug_read(opb_superpoint* h, int32_t which, float* out, size_t capacity_elems, int64_t* n_elems, void* stream) {
  ENTER(h);
  if (!out || !h->last_B) return fail(h, OPB_E_INVALID, "opb_sp_debug_read: null output or no preceding opb_sp_detect");
  cudaStream_t st = (cudaStream_t)stream;
  const int B = h->last_B, H = h->last_H, W = h->last_W;
  const Stage s3 = stage_of(H, W, 3);
  size_t n = 0;
  const void* src = nullptr;
  switch (which) {
    case 0: n = (size_t)B * H * W; src = h->scores.p; break;                       // dense scores [B, H, W]
    case 1: n = (size_t)B * H * W; src = h->nms.p; break;                          // after NMS
    case 2: n = (size_t)B * s3.ppad * 128; src = h->logits.p; break;               // convPb output rows [B*P3, 128] (65 valid)
    case 3: n = (size_t)B * s3.ppad * 256; src = h->ddesc.p; break;                // convDb output rows [B*P3, 256]
    case 4: {                                                                      // activation planes of the last layer run (stop hook)
      n = (size_t)h->dbg_rows * h->dbg_c;
      if (n_elems) *n_elems = (int64_t)n;
      if (n > capacity_elems) return fail(h, OPB_E_INVALID, "opb_sp_debug_read: capacity %zu < %zu", capacity_elems, n);
      const PlaneBuf& a = h->arena[h->dbg_arena];
      sp_join_planes<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(a.hi.as<__half>(), a.lo.as<__half>(), out, (long long)n);
      return launch_status(h, __func__);
    }
    default: return fail(h, OPB_E_INVALID, "opb_sp_debug_read: unknown buffer %d", which);
  }
  if (n_elems) *n_elems = (int64_t)n;
  if (n > capacity_elems) return fail(h, OPB_E_INVALID, "opb_sp_debug_read: capacity %zu < %zu", capacity_elems, n);
  CK(h, cudaMemcpyAsync(out, src, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return OPB_OK;
}

}  // extern "C"
