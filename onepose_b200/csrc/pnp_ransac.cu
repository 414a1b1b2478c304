// Batched RANSAC-PnP on the GPU: the consumer of the matcher's 2D-3D correspondences
// (reference src/utils/eval_utils.py:18-42: cv2.solvePnPRansac(pts_3d, pts_2d, K, 0, reprojectionError=5,
//  iterationsCount=10000, flags=SOLVEPNP_EPNP) per frame on the host -- the step that dominates per-frame latency once
//  matching takes ~1 ms; SURVEY 8f N3).
//
// The reference delegates the arithmetic to OpenCV; parity for this row is the pose itself (the reference's own metric is the
// cm-degree error, src/evaluators/cmd_evaluator.py), not bits: OpenCV draws its minimal samples from its own RNG.  Algorithm:
//   hypotheses  one thread per minimal sample: 3 correspondences -> P3P (Grunert's quartic, coefficients as in Haralick et al.
//               1994; closed-form quartic roots + Newton polish) -> up to 4 poses, each scored by its inlier count over ALL
//               correspondences of the frame (reprojection error < threshold, point in front of the camera), fp64;
//   selection   per frame: hypothesis with the most inliers (lowest index wins ties: deterministic);
//   refinement  Gauss-Newton on the reprojection error of the inlier set (6 DoF, left rotation update), inlier set re-evaluated
//               between rounds (local optimisation) -- what OpenCV's final EPnP refit on the inliers approximates.
// One launch handles B frames (ragged correspondence lists, offsets[B+1]); everything stays on the device.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/onepose_b200.h"
#include "host_util.cuh"

namespace opb {
namespace {

struct Pose {
  double R[9];   // row-major, world -> camera
  double t[3];
};

__device__ __forceinline__ uint64_t mix64(uint64_t z) {   // splitmix64 finaliser
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// largest real root of z^3 + a2 z^2 + a1 z + a0
__device__ double cubic_largest_real(double a2, double a1, double a0) {
  const double q = (3.0 * a1 - a2 * a2) / 9.0, r = (9.0 * a2 * a1 - 27.0 * a0 - 2.0 * a2 * a2 * a2) / 54.0;
  const double D = q * q * q + r * r;
  if (D >= 0.0) {
    const double sD = sqrt(D);
    return cbrt(r + sD) + cbrt(r - sD) - a2 / 3.0;
  }
  const double th = acos(fmax(-1.0, fmin(1.0, r / sqrt(-q * q * q))));
  return 2.0 * sqrt(-q) * cos(th / 3.0) - a2 / 3.0;
}

// real roots of A4 x^4 + ... + A0 (Ferrari via the resolvent cubic), polished by two Newton steps; returns their number
__device__ int quartic_real_roots(double A4, double A3, double A2, double A1, double A0, double* x) {
  if (fabs(A4) < 1e-300) return 0;
  const double a = A3 / A4, b = A2 / A4, c = A1 / A4, d = A0 / A4;
  const double p = b - 3.0 * a * a / 8.0, q = c - a * b / 2.0 + a * a * a / 8.0;
  const double r = d - a * c / 4.0 + a * a * b / 16.0 - 3.0 * a * a * a * a / 256.0;
  double y[4];
  int n = 0;
  if (fabs(q) < 1e-14 * fmax(1.0, pow(fabs(p), 1.5))) {        // biquadratic
    const double disc = p * p - 4.0 * r;
    if (disc >= 0.0) {
      const double w[2] = {(-p + sqrt(disc)) / 2.0, (-p - sqrt(disc)) / 2.0};
      for (int k = 0; k < 2; ++k)
        if (w[k] >= 0.0) { y[n++] = sqrt(w[k]); y[n++] = -sqrt(w[k]); }
    }
  } else {
    const double z = cubic_largest_real(2.0 * p, p * p - 4.0 * r, -q * q);
    if (z <= 0.0) return 0;
    const double s = sqrt(z);
    for (int k = 0; k < 2; ++k) {
      const double sg = k ? -1.0 : 1.0;
      const double B = sg * s, C = (p + z - sg * q / s) / 2.0;   // y^2 + B y + C = 0
      const double disc = B * B - 4.0 * C;
      if (disc >= 0.0) { const double sd = sqrt(disc); y[n++] = (-B + sd) / 2.0; y[n++] = (-B - sd) / 2.0; }
    }
  }
  for (int k = 0; k < n; ++k) {
    double v = y[k] - a / 4.0;
    for (int it = 0; it < 2; ++it) {
      const double f = (((A4 * v + A3) * v + A2) * v + A1) * v + A0, df = ((4.0 * A4 * v + 3.0 * A3) * v + 2.0 * A2) * v + A1;
      if (df != 0.0) v -= f / df;
    }
    x[k] = v;
  }
  return n;
}

__device__ __forceinline__ void cross3(const double* a, const double* b, double* c) {
  c[0] = a[1] * b[2] - a[2] * b[1]; c[1] = a[2] * b[0] - a[0] * b[2]; c[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ __forceinline__ bool normalize3(double* a) {
  const double n = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
  if (!(n > 1e-12)) return false;
  a[0] /= n; a[1] /= n; a[2] /= n;
  return true;
}
// orthonormal frame of a triangle: columns e1 = (Q1-Q0)^, e3 = (e1 x (Q2-Q0))^, e2 = e3 x e1; F row-major [3][3] with columns e1,e2,e3
__device__ bool tri_frame(const double Q[3][3], double F[9]) {
  double e1[3] = {Q[1][0] - Q[0][0], Q[1][1] - Q[0][1], Q[1][2] - Q[0][2]};
  double d2[3] = {Q[2][0] - Q[0][0], Q[2][1] - Q[0][1], Q[2][2] - Q[0][2]};
  double e3[3], e2[3];
  if (!normalize3(e1)) return false;
  cross3(e1, d2, e3);
  if (!normalize3(e3)) return false;
  cross3(e3, e1, e2);
  for (int i = 0; i < 3; ++i) { F[i * 3 + 0] = e1[i]; F[i * 3 + 1] = e2[i]; F[i * 3 + 2] = e3[i]; }
  return true;
}

// P3P: world points P[3], unit bearings j[3] (camera frame) -> up to 4 poses
__device__ int p3p(const double P[3][3], const double j[3][3], Pose* out) {
  auto dist2 = [&](int a, int b) {
    const double dx = P[a][0] - P[b][0], dy = P[a][1] - P[b][1], dz = P[a][2] - P[b][2];
    return dx * dx + dy * dy + dz * dz;
  };
  auto dot = [&](int a, int b) { return j[a][0] * j[b][0] + j[a][1] * j[b][1] + j[a][2] * j[b][2]; };
  const double a2 = dist2(1, 2), b2 = dist2(0, 2), c2 = dist2(0, 1);
  if (!(a2 > 1e-18 && b2 > 1e-18 && c2 > 1e-18)) return 0;
  const double ca = dot(1, 2), cb = dot(0, 2), cg = dot(0, 1);
  const double p = (a2 - c2) / b2, q = (a2 + c2) / b2;
  const double A4 = (p - 1.0) * (p - 1.0) - 4.0 * c2 / b2 * ca * ca;
  const double A3 = 4.0 * (p * (1.0 - p) * cb - (1.0 - q) * ca * cg + 2.0 * c2 / b2 * ca * ca * cb);
  const double A2 = 2.0 * (p * p - 1.0 + 2.0 * p * p * cb * cb + 2.0 * ((b2 - c2) / b2) * ca * ca - 4.0 * q * ca * cb * cg + 2.0 * ((b2 - a2) / b2) * cg * cg);
  const double A1 = 4.0 * (-p * (1.0 + p) * cb + 2.0 * a2 / b2 * cg * cg * cb - (1.0 - q) * ca * cg);
  const double A0 = (1.0 + p) * (1.0 + p) - 4.0 * a2 / b2 * cg * cg;
  double v[4];
  const int nr = quartic_real_roots(A4, A3, A2, A1, A0, v);
  double FP[9];
  if (!tri_frame(P, FP)) return 0;
  int ns = 0;
  for (int k = 0; k < nr; ++k) {
    if (!(v[k] > 0.0)) continue;
    const double den = 2.0 * (cg - v[k] * ca);
    if (fabs(den) < 1e-12) continue;
    const double u = ((-1.0 + p) * v[k] * v[k] - 2.0 * p * cb * v[k] + 1.0 + p) / den;
    if (!(u > 0.0)) continue;
    const double s1sq = c2 / (1.0 + u * u - 2.0 * u * cg);
    if (!(s1sq > 0.0)) continue;
    const double s[3] = {sqrt(s1sq), u * sqrt(s1sq), v[k] * sqrt(s1sq)};
    double X[3][3];
    for (int i = 0; i < 3; ++i)
      for (int d = 0; d < 3; ++d) X[i][d] = s[i] * j[i][d];
    double FX[9];
    if (!tri_frame(X, FX)) continue;
    Pose& o = out[ns];
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) o.R[r * 3 + c] = FX[r * 3 + 0] * FP[c * 3 + 0] + FX[r * 3 + 1] * FP[c * 3 + 1] + FX[r * 3 + 2] * FP[c * 3 + 2];   // FX . FP^T
    for (int r = 0; r < 3; ++r) o.t[r] = X[0][r] - (o.R[r * 3 + 0] * P[0][0] + o.R[r * 3 + 1] * P[0][1] + o.R[r * 3 + 2] * P[0][2]);
    ++ns;
  }
  return ns;
}

__device__ __forceinline__ bool reproj_inlier(const Pose& T, const double* Kc /*fx,fy,cx,cy*/, const double* p3, const double* p2, double thr2) {
  const double x = T.R[0] * p3[0] + T.R[1] * p3[1] + T.R[2] * p3[2] + T.t[0];
  const double y = T.R[3] * p3[0] + T.R[4] * p3[1] + T.R[5] * p3[2] + T.t[1];
  const double z = T.R[6] * p3[0] + T.R[7] * p3[1] + T.R[8] * p3[2] + T.t[2];
  if (!(z > 1e-9)) return false;
  const double du = Kc[0] * x / z + Kc[2] - p2[0], dv = Kc[1] * y / z + Kc[3] - p2[1];
  return du * du + dv * dv < thr2;
}

// hyp: [B][H] {count, pose(12)} as 13 doubles
constexpr int kHypStride = 13;

__global__ void __launch_bounds__(128) pnp_hypotheses(const double* __restrict__ Kmat /*[B][9]*/, const double* __restrict__ pts2d, const double* __restrict__ pts3d,
                                                      const int* __restrict__ offsets, int H, double thr2, unsigned long long seed,
                                                      double* __restrict__ hyp) {
  const int b = blockIdx.y;
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= H) return;
  const int o0 = offsets[b], n = offsets[b + 1] - o0;
  double* out = hyp + ((size_t)b * H + h) * kHypStride;
  out[0] = 0.0;
  if (n < 4) return;
  const double* K = Kmat + (size_t)b * 9;
  const double Kc[4] = {K[0], K[4], K[2], K[5]};
  // three distinct correspondences
  uint64_t r = mix64(seed ^ ((uint64_t)b << 40) ^ (uint64_t)h);
  int idx[3];
  idx[0] = (int)(r % (uint64_t)n);
  r = mix64(r);
  idx[1] = (int)(r % (uint64_t)(n - 1));
  if (idx[1] >= idx[0]) ++idx[1];
  r = mix64(r);
  idx[2] = (int)(r % (uint64_t)(n - 2));
  { const int lo = min(idx[0], idx[1]), hi = max(idx[0], idx[1]); if (idx[2] >= lo) ++idx[2]; if (idx[2] >= hi) ++idx[2]; }
  double P[3][3], j[3][3];
  for (int k = 0; k < 3; ++k) {
    const double* p3 = pts3d + (size_t)(o0 + idx[k]) * 3;
    const double* p2 = pts2d + (size_t)(o0 + idx[k]) * 2;
    P[k][0] = p3[0]; P[k][1] = p3[1]; P[k][2] = p3[2];
    j[k][0] = (p2[0] - Kc[2]) / Kc[0]; j[k][1] = (p2[1] - Kc[3]) / Kc[1]; j[k][2] = 1.0;
    normalize3(j[k]);
  }
  Pose sol[4];
  const int ns = p3p(P, j, sol);
  int best = -1, best_cnt = 0;
  for (int s = 0; s < ns; ++s) {
    int cnt = 0;
    for (int i = 0; i < n; ++i) cnt += reproj_inlier(sol[s], Kc, pts3d + (size_t)(o0 + i) * 3, pts2d + (size_t)(o0 + i) * 2, thr2) ? 1 : 0;
    if (cnt > best_cnt) { best_cnt = cnt; best = s; }
  }
  if (best < 0) return;
  out[0] = (double)best_cnt;
  for (int k = 0; k < 9; ++k) out[1 + k] = sol[best].R[k];
  for (int k = 0; k < 3; ++k) out[10 + k] = sol[best].t[k];
}

__device__ void rodrigues_left(const double* w, Pose& T) {   // T <- exp([w]x) . T (rotation and translation), small-angle safe
  const double th2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2], th = sqrt(th2);
  const double A = th > 1e-8 ? sin(th) / th : 1.0 - th2 / 6.0, Bc = th > 1e-8 ? (1.0 - cos(th)) / th2 : 0.5 - th2 / 24.0;
  double E[9];
  const double W[9] = {0, -w[2], w[1], w[2], 0, -w[0], -w[1], w[0], 0};
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) {
      double w2 = 0;
      for (int k = 0; k < 3; ++k) w2 += W[r * 3 + k] * W[k * 3 + c];
      E[r * 3 + c] = (r == c ? 1.0 : 0.0) + A * W[r * 3 + c] + Bc * w2;
    }
  double Rn[9], tn[3];
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) Rn[r * 3 + c] = E[r * 3 + 0] * T.R[c] + E[r * 3 + 1] * T.R[3 + c] + E[r * 3 + 2] * T.R[6 + c];
    tn[r] = E[r * 3 + 0] * T.t[0] + E[r * 3 + 1] * T.t[1] + E[r * 3 + 2] * T.t[2];
  }
  for (int k = 0; k < 9; ++k) T.R[k] = Rn[k];
  for (int k = 0; k < 3; ++k) T.t[k] = tn[k];
}

// one block per frame: arg-max over hypotheses, local optimisation, outputs
constexpr int kRefineThreads = 256;
__global__ void __launch_bounds__(kRefineThreads) pnp_select_refine(const double* __restrict__ Kmat, const double* __restrict__ pts2d, const double* __restrict__ pts3d,
                                                                     const int* __restrict__ offsets, int H, double thr2, const double* __restrict__ hyp,
                                                                     double* __restrict__ pose_out /*[B][12]*/, int* __restrict__ inlier_mask,
                                                                     int* __restrict__ n_inliers /*[B]*/) {
  __shared__ unsigned long long best_key[kRefineThreads];
  __shared__ double red[27][kRefineThreads / 32];
  __shared__ Pose T;
  __shared__ double delta[6];
  __shared__ int ok;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int o0 = offsets[b], n = offsets[b + 1] - o0;
  const double* K = Kmat + (size_t)b * 9;
  const double Kc[4] = {K[0], K[4], K[2], K[5]};
  // ---- best hypothesis: max count, lowest index
  unsigned long long key = 0ull;
  for (int h = tid; h < H; h += kRefineThreads) {
    const unsigned long long c = (unsigned long long)hyp[((size_t)b * H + h) * kHypStride];
    const unsigned long long k = (c << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)h);
    key = k > key ? k : key;
  }
  best_key[tid] = key;
  __syncthreads();
  for (int s = kRefineThreads / 2; s > 0; s >>= 1) {
    if (tid < s && best_key[tid + s] > best_key[tid]) best_key[tid] = best_key[tid + s];
    __syncthreads();
  }
  const unsigned long long bk = best_key[0];
  const int best_cnt = (int)(bk >> 32), best_h = (int)(0xFFFFFFFFu - (unsigned)(bk & 0xFFFFFFFFull));
  if (tid == 0) {
    ok = best_cnt >= 4 ? 1 : 0;
    if (ok) {
      const double* src = hyp + ((size_t)b * H + best_h) * kHypStride;
      for (int k = 0; k < 9; ++k) T.R[k] = src[1 + k];
      for (int k = 0; k < 3; ++k) T.t[k] = src[10 + k];
    }
  }
  __syncthreads();
  if (!ok) {                                       // no model: identity pose, no inliers (the reference's except-branch result)
    if (tid < 12) pose_out[(size_t)b * 12 + tid] = (tid == 0 || tid == 5 || tid == 10) ? 1.0 : 0.0;
    for (int i = tid; i < n; i += kRefineThreads) inlier_mask[o0 + i] = 0;
    if (tid == 0) n_inliers[b] = 0;
    return;
  }
  // ---- Gauss-Newton on the inliers of the current pose; the inlier set is re-evaluated every round
  for (int it = 0; it < 10; ++it) {
    double acc[27];
#pragma unroll
    for (int k = 0; k < 27; ++k) acc[k] = 0.0;
    const Pose Tl = T;
    for (int i = tid; i < n; i += kRefineThreads) {
      const double* p3 = pts3d + (size_t)(o0 + i) * 3;
      const double* p2 = pts2d + (size_t)(o0 + i) * 2;
      if (!reproj_inlier(Tl, Kc, p3, p2, thr2)) continue;
      const double x = Tl.R[0] * p3[0] + Tl.R[1] * p3[1] + Tl.R[2] * p3[2] + Tl.t[0];
      const double y = Tl.R[3] * p3[0] + Tl.R[4] * p3[1] + Tl.R[5] * p3[2] + Tl.t[1];
      const double z = Tl.R[6] * p3[0] + Tl.R[7] * p3[1] + Tl.R[8] * p3[2] + Tl.t[2];
      const double iz = 1.0 / z;
      const double ru = Kc[0] * x * iz + Kc[2] - p2[0], rv = Kc[1] * y * iz + Kc[3] - p2[1];
      // d(proj)/dX, X' = exp(w) X + dt  =>  dX/dw = -[X]x, dX/dt = I
      const double jux = Kc[0] * iz, juz = -Kc[0] * x * iz * iz, jvy = Kc[1] * iz, jvz = -Kc[1] * y * iz * iz;
      double Ju[6], Jv[6];
      Ju[0] = juz * y;            Ju[1] = jux * z - juz * x;  Ju[2] = -jux * y;           // rotation part: row . (-[X]x)
      Jv[0] = -jvy * z + jvz * y; Jv[1] = -jvz * x;           Jv[2] = jvy * x;
      Ju[3] = jux; Ju[4] = 0.0; Ju[5] = juz;
      Jv[3] = 0.0; Jv[4] = jvy; Jv[5] = jvz;
      int k = 0;
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int c = r; c < 6; ++c) acc[k++] += Ju[r] * Ju[c] + Jv[r] * Jv[c];
#pragma unroll
      for (int r = 0; r < 6; ++r) acc[21 + r] += Ju[r] * ru + Jv[r] * rv;
    }
#pragma unroll
    for (int k = 0; k < 27; ++k) {
      double v = acc[k];
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) red[k][warp] = v;
    }
    __syncthreads();
    if (tid == 0) {
      double A[6][6], g[6];
      int k = 0;
      for (int r = 0; r < 6; ++r)
        for (int c = r; c < 6; ++c) {
          double v = 0;
          for (int w = 0; w < kRefineThreads / 32; ++w) v += red[k][w];
          A[r][c] = A[c][r] = v;
          ++k;
        }
      for (int r = 0; r < 6; ++r) {
        double v = 0;
        for (int w = 0; w < kRefineThreads / 32; ++w) v += red[21 + r][w];
        g[r] = -v;
      }
      for (int r = 0; r < 6; ++r) A[r][r] *= 1.0 + 1e-9;      // tiny damping against rank deficiency
      // Cholesky solve A d = g
      bool good = true;
      double Lm[6][6] = {};
      for (int r = 0; r < 6 && good; ++r)
        for (int c = 0; c <= r; ++c) {
          double s = A[r][c];
          for (int m = 0; m < c; ++m) s -= Lm[r][m] * Lm[c][m];
          if (r == c) { if (!(s > 1e-300)) { good = false; break; } Lm[r][r] = sqrt(s); }
          else Lm[r][c] = s / Lm[c][c];
        }
      double yv[6], d[6] = {0, 0, 0, 0, 0, 0};
      if (good) {
        for (int r = 0; r < 6; ++r) { double s = g[r]; for (int m = 0; m < r; ++m) s -= Lm[r][m] * yv[m]; yv[r] = s / Lm[r][r]; }
        for (int r = 5; r >= 0; --r) { double s = yv[r]; for (int m = r + 1; m < 6; ++m) s -= Lm[m][r] * d[m]; d[r] = s / Lm[r][r]; }
      }
      for (int r = 0; r < 6; ++r) delta[r] = d[r];
      rodrigues_left(d, T);
      T.t[0] += d[3]; T.t[1] += d[4]; T.t[2] += d[5];
    }
    __syncthreads();
    const double step = fabs(delta[0]) + fabs(delta[1]) + fabs(delta[2]) + fabs(delta[3]) + fabs(delta[4]) + fabs(delta[5]);
    if (step < 1e-12) break;
  }
  // ---- outputs
  int cnt = 0;
  for (int i = tid; i < n; i += kRefineThreads) {
    const int in = reproj_inlier(T, Kc, pts3d + (size_t)(o0 + i) * 3, pts2d + (size_t)(o0 + i) * 2, thr2) ? 1 : 0;
    inlier_mask[o0 + i] = in;
    cnt += in;
  }
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  __shared__ int cnt_w[kRefineThreads / 32];
  if (lane == 0) cnt_w[warp] = cnt;
  __syncthreads();
  if (tid == 0) {
    int c = 0;
    for (int w = 0; w < kRefineThreads / 32; ++w) c += cnt_w[w];
    n_inliers[b] = c;
    for (int r = 0; r < 3; ++r) {
      for (int k = 0; k < 3; ++k) pose_out[(size_t)b * 12 + r * 4 + k] = T.R[r * 3 + k];
      pose_out[(size_t)b * 12 + r * 4 + 3] = T.t[r];
    }
  }
}

}  // namespace
}  // namespace opb

extern "C" int opb_ransac_pnp(const double* K, const double* pts2d, const double* pts3d, const int32_t* offsets, int32_t B, int32_t hypotheses,
                              double reproj_error, uint64_t seed, double* workspace, double* pose_out, int32_t* inlier_mask, int32_t* n_inliers,
                              void* stream) {
  if (!K || !pts2d || !pts3d || !offsets || !workspace || !pose_out || !inlier_mask || !n_inliers || B <= 0 || hypotheses <= 0 || !(reproj_error > 0.0))
    return opb::fail(nullptr, OPB_E_INVALID, "%s: bad argument (B=%d, hypotheses=%d, reproj_error=%g)", __func__, B, hypotheses, reproj_error);
  cudaStream_t st = (cudaStream_t)stream;
  const double thr2 = reproj_error * reproj_error;
  opb::pnp_hypotheses<<<dim3((unsigned)((hypotheses + 127) / 128), (unsigned)B), 128, 0, st>>>(K, pts2d, pts3d, offsets, hypotheses, thr2,
                                                                                               (unsigned long long)seed, workspace);
  opb::pnp_select_refine<<<(unsigned)B, opb::kRefineThreads, 0, st>>>(K, pts2d, pts3d, offsets, hypotheses, thr2, workspace, pose_out, inlier_mask, n_inliers);
  return opb::launch_status(nullptr, __func__);
}
