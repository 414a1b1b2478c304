// C ABI of the B200-native GATsSPG matcher (see include/onepose_b200.h).
// Host-side state: packed weights, per-object constants, chunk workspace, launch sequence.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/onepose_b200.h"
#include "common.cuh"
#include "gemm_common.cuh"
#include "gemm_tc.cuh"
#include "host_util.cuh"
#include "kernels_aux.cuh"
#include "kv_state_tc.cuh"

namespace opb {

constexpr int kDefaultChunk = 32;   // frames pushed through the GNN together (measured: 4 -> 1340, 8 -> 1650, 16 -> 2390, 32 -> 2550 frames/s)
constexpr int kQPassFrames = 16;    // granularity of the query-side layer-1 pass when the queries stream in from the host

static bool g_pdl = true;
static int g_ws_fill = -1;     // >= 0: byte value written into every fresh allocation that the algorithm does not require to be zero
int ws_fill_byte() { return g_ws_fill; }
bool pdl_enabled() { return g_pdl; }
void set_pdl_enabled(bool on) { g_pdl = on; }

struct AttnLayerW {       // one AttentionPropagation (reference GATs_SuperGlue.py:104-113)
  PlaneBuf wqkv;          // [768,256]  rows: Q | K | V, head-contiguous output channels
  DevBuf bqkv;            // [768]
  PlaneBuf w0a;           // [512,256]  mlp.0.weight[:, :256]
  PlaneBuf w0m;           // [512,256]  mlp.0.weight[:, 256:] @ merge.weight (head-contiguous inputs): A operand of the G-fold GEMM
  DevBuf b0f;             // [512] = mlp.0.weight[:,256:] @ merge.bias + mlp.0.bias
  PlaneBuf w1;            // [256,512]  mlp.3.weight
  DevBuf b1;              // [256]
};

}  // namespace opb

using namespace opb;

struct opb_matcher : HostState {
  opb_config cfg{};
  bool weights_ready = false;
  bool object_ready = false;
  int num_sms = 148;
  // packed weights
  AttnLayerW attn[8];
  DevBuf wa2, wa3;        // [4][256] each (GATs: W a[:256], W a[256:])
  PlaneBuf wlin;          // [4][256][256]: W^T of the GATs layers (with_linear_transform only)
  PlaneBuf wf;            // final_proj [256,256]
  DevBuf bf;
  PlaneBuf eye;           // [256,256] identity, fp16-split (residual as an identity K-block of the mlp.3 GEMM)
  // per-object constants
  int M = 0, Lf = 0, m_pad = 0;
  DevBuf leaves;          // fp32 [M*Lf, 256] point-major
  PlaneBuf db;            // [m_pad, 256]
  DevBuf s2;              // [4][M*Lf]
  PlaneBuf xo;            // [m_pad, 256]: 3D-point state entering layer 2 (object prologue), valid while prologue_ready
  bool prologue_ready = false;
  // workspace (chunk)
  int chunk_frames = 0;   // user override
  int ws_frames = 0, ws_N = 0;
  bool hoist = true;      // evaluate the frame-invariant layers once per object (object_prologue)
  int identity_diag = 1;  // residual identity K-block as N = 64 MMAs on the diagonal blocks (opb_debug_set_identity_diag)
  int kv_two_pass = 1;    // k,v projection as A_hi.(B_hi + B_lo): its output is one fp16 plane, the A_lo term is below that rounding
  PlaneBuf x, qp, pn, g, xq, bd, lin_a, lin_b;
  DevBuf kvt;             // fp16 [rows, 512]
  DevBuf hid, kvpart, kmean, statpart, mu, rstd, rowsum_part, colsum_part, rowsum, colsum, rowbest, colbest;
  DevBuf range_flag;
  int* range_host = nullptr;                    // pinned copy of the flag, written at the end of every opb_forward
  cudaEvent_t range_ev = nullptr;
  bool range_pending = false;
  cudaStream_t last_stream = nullptr;
  // host-call staging
  DevBuf st_q, st_m0, st_m1, st_s0, st_s1, st_conf, st_len;
  cudaStream_t copy_stream = nullptr;          // opb_forward_host: H2D of chunk i+1 overlaps the compute of chunk i
  std::vector<cudaEvent_t> h2d_ev;              // one per piece; consumed by the chunk loop of opb_forward
  int h2d_pending = 0;
  Layout last_layout{};
  int last_launches = 0;
};

namespace opb {

// Profile name of a GEMM launch: "gemm epi<epilogue> n<N> k<K> <what>" (bench.py selects launches by its prefix), formatted
// only when profiling.
static int matcher_gemm(opb_matcher* m, const GemmProblem& p, cudaStream_t st, double flops, const char* what) {
  char tag[96];
  if (m->profiling) snprintf(tag, sizeof tag, "gemm epi%d n%d k%d %s", p.epi, p.n_out, p.K1 + p.K2, what);
  return run_gemm(m, p, st, flops, m->profiling ? tag : what);
}

static int ensure_workspace(opb_matcher* m, int frames, int N) {
  if (frames <= m->ws_frames && N <= m->ws_N) return 0;
  frames = frames > m->ws_frames ? frames : m->ws_frames;
  N = N > m->ws_N ? N : m->ws_N;
  const int n_pad = round_up(N, kSegPad);
  const size_t R = (size_t)n_pad + m->m_pad;
  const size_t rows = R * frames;
  const size_t S = 2 * (size_t)frames;
  CK(m, m->x.ensure(rows * kD));
  CK(m, m->qp.ensure(rows * kD));
  CK(m, m->pn.ensure(rows * kD));
  CK(m, m->g.ensure(S * 512 * kD));
  CK(m, m->bd.ensure(S * kD * kD, true));          // block-diagonal state operand: off-diagonal blocks stay zero for the buffer's lifetime
  CK(m, m->xq.ensure((size_t)frames * n_pad * kD));
  CK(m, m->kvt.ensure(rows * 512 * sizeof(__half)));
  CK(m, m->hid.ensure(rows * 512 * sizeof(float)));
  CK(m, m->kvpart.ensure(rows / 256 * kHeads * kKVPartial * sizeof(float)));
  CK(m, m->kmean.ensure(S * kD * sizeof(float)));
  CK(m, m->statpart.ensure(rows / 32 * 512 * 2 * sizeof(float)));
  CK(m, m->mu.ensure(S * 512 * sizeof(float)));
  CK(m, m->rstd.ensure(S * 512 * sizeof(float)));
  CK(m, m->rowsum.ensure((size_t)frames * n_pad * sizeof(float)));
  CK(m, m->rowsum_part.ensure((size_t)frames * (m->m_pad / 256) * 2 * n_pad * sizeof(float)));
  CK(m, m->colsum_part.ensure((size_t)frames * (n_pad / 32) * m->m_pad * sizeof(float)));
  CK(m, m->colsum.ensure((size_t)frames * m->m_pad * sizeof(float)));
  CK(m, m->rowbest.ensure((size_t)frames * n_pad * sizeof(unsigned long long)));
  CK(m, m->colbest.ensure((size_t)frames * m->m_pad * sizeof(unsigned long long)));
  CK(m, m->range_flag.ensure(sizeof(int), true));
  if (m->cfg.with_linear_transform) {
    CK(m, m->lin_a.ensure((size_t)frames * m->m_pad * kD));
    CK(m, m->lin_b.ensure((size_t)frames * m->m_pad * kD));
  }
  // (re)allocation fills ran on the legacy stream: order them against the caller's (possibly non-blocking) stream once
  CK(m, cudaDeviceSynchronize());
  m->ws_frames = frames;
  m->ws_N = N;
  return 0;
}

// One GATs layer on the 3D-point segments of `x` (layout L).
static int run_gats(opb_matcher* m, const Layout& L, XView x, int gi, cudaStream_t st) {
  const long long warps = (long long)L.M * L.B;
  if (warps == 0) return 0;
  const bool lin = m->cfg.with_linear_transform != 0;
  GatsOut out{lin ? m->lin_a.hi.as<__half>() : x.hi, lin ? m->lin_a.lo.as<__half>() : x.lo, lin ? 1 : 0};
  const float* s2 = m->s2.as<float>() + (size_t)gi * m->M * m->Lf;
  const float* wa3 = m->wa3.as<float>() + gi * kD;
  if (m->Lf == 8) {   // leaves loaded once per point and reused across 8 frames of the chunk (any B: one code path, frame-independent results)
    const long long w8 = (long long)L.M * ((L.B + kGatsFramesPerWarp - 1) / kGatsFramesPerWarp);
    LAUNCH(m, st, "gats_aggregate", gats_aggregate_frames8, dim3((unsigned)((w8 * 32 + 255) / 256)), dim3(256), 0, st, (const __half*)x.hi,
           (const __half*)x.lo, L, (const float*)m->leaves.as<float>(), s2, wa3, (int)m->cfg.include_self, (int)m->cfg.additional, 0.2f, out);
  } else {
    LAUNCH(m, st, "gats_aggregate", gats_aggregate, dim3((unsigned)((warps * 32 + 255) / 256)), dim3(256), 0, st, (const __half*)x.hi,
           (const __half*)x.lo, L, (const float*)m->leaves.as<float>(), m->Lf, s2, wa3, (int)m->cfg.include_self, (int)m->cfg.additional, 0.2f,
           out);
  }
  if (!lin) return 0;
  // with_linear_transform (GATs.py:56-57,64-65): t = pre . W on the tensor cores over the compact 3D rows, then ELU (+ h3)
  Layout Lc{};
  Lc.B = L.B; Lc.N = 0; Lc.M = L.M; Lc.n_pad = 0; Lc.m_pad = L.m_pad; Lc.R = L.m_pad;
  GemmProblem p{};
  p.L = Lc; p.batch = 1; p.rows = Lc.rows();
  p.a1 = m->lin_a.c(kD); p.K1 = kD; p.b1 = m->wlin.c(kD, (size_t)gi * kD * kD); p.n_out = kD;
  p.epi = EPI_BIAS_PLANES; p.out = m->lin_b.m(kD);
  if (int rc = matcher_gemm(m, p, st, 2.0 * L.B * (double)L.M * kD * kD, "gats.W")) return rc;
  const long long n = (long long)L.B * L.M * 32;
  LAUNCH(m, st, "gats_lin_finish", gats_lin_finish, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, (const __half*)m->lin_b.hi.as<__half>(),
         (const __half*)m->lin_b.lo.as<__half>(), x.hi, x.lo, L, (int)(m->cfg.include_self && m->cfg.additional));
  return 0;
}

// One AttentionPropagation layer (reference GATs_SuperGlue.py:55-64, :104-113) on every segment of `x`:
// both sides of all frames in ONE set of 8 launches (the layer's weights are shared by the two sides).
static int run_attn_layer(opb_matcher* m, const Layout& L, XView x, AttnLayerW& W, int cross, cudaStream_t st) {
  const int rows = L.rows();
  const int S = L.segs();
  const double valid_rows = (double)L.B * (L.N + L.M);
  // (1) k,v projection (:96-99), rows [256, 768) of the packed weight; epilogue: elu+1 on K, pad rows zeroed, ONE fp16 plane
  //     kvt[rows, 512] = fp16(64 * [elu1(K) | V]) -- the single-pass operands of the state kernel
  GemmProblem pk{};
  pk.L = L; pk.batch = 1; pk.rows = rows;
  pk.a1 = x.c(kD); pk.K1 = kD; pk.b1 = W.wqkv.c(kD, (size_t)256 * kD); pk.n_out = 512;
  pk.bias = W.bqkv.as<float>() + 256;
  pk.epi = EPI_QKV; pk.out = Planes{m->kvt.as<__half>(), m->kvt.as<__half>(), 512};
  pk.a_hi_only = m->kv_two_pass;
  if (int rc = matcher_gemm(m, pk, st, 2.0 * valid_rows * 512 * kD, "kv_proj")) return rc;
  // (2) linear-attention state of every segment (:71-78): per-row-group partial states on the tensor cores ...
  const KvGroups G = kv_groups_for(L, m->num_sms);
  if (launch_kv_state_h(m->kvt.as<__half>(), L, G, m->kvpart.as<float>(), st)) return fail(m, OPB_E_CUDA, "kv_state_h launch failed");
  log_launch(m, st, "kv_state_h", 0.0);
  // ... reduced per segment into Kmean and the block-diagonal operand of the G fold (indexed by DESTINATION segment)
  LAUNCH(m, st, "kv_state_reduce", kv_state_reduce, dim3(S * kHeads, (kKVPartial + 255) / 256), dim3(256), 0, st, (const float*)m->kvpart.as<float>(), L,
         G, cross, m->kmean.as<float>(), m->bd.hi.as<__half>(), m->bd.lo.as<__half>());
  // (3) q projection; epilogue: elu+1 and the per-head normaliser with the SOURCE segment's K mean -> Q' planes (:78-79)
  GemmProblem pq{};
  pq.L = L; pq.batch = 1; pq.rows = rows;
  pq.a1 = x.c(kD); pq.K1 = kD; pq.b1 = W.wqkv.c(kD); pq.n_out = 256; pq.bias = W.bqkv.as<float>();
  pq.epi = EPI_QSCALE; pq.kmean = m->kmean.as<float>(); pq.cross = cross; pq.out = m->qp.m(kD);
  if (int rc = matcher_gemm(m, pq, st, 2.0 * valid_rows * 256 * kD, "q_proj")) return rc;
  // (4) dynamic weight G[s] = W0m . blockdiag(KVmean_src(s))^T  -- merge and the message half of mlp.0 folded into one
  //     per-segment [512, 256] weight (4 x 64x64x512 MACs per segment), as a batched tcgen05 GEMM over the segments
  GemmProblem pg{};
  pg.batch = S; pg.rows = 512; pg.n_out = kD; pg.K1 = kD;
  pg.a1 = W.w0m.c(kD); pg.a_batch_rows = 0;
  pg.b1 = m->bd.c(kD); pg.b_batch_rows = kD;
  pg.epi = EPI_BIAS_PLANES; pg.out = m->g.m(kD);
  if (int rc = matcher_gemm(m, pg, st, 2.0 * S * 512.0 * kD * kDh, "g_fold")) return rc;
  // (5) hidden = mlp.0([x ; message]) = [x | Q'] . [W0a | G_seg]^T + b   (:101,:113,:122); epilogue also emits the InstanceNorm
  //     partial sums (:126)
  GemmProblem p2{};
  p2.L = L; p2.batch = 1; p2.rows = rows;
  p2.a1 = x.c(kD); p2.K1 = kD; p2.b1 = W.w0a.c(kD);
  p2.a2 = m->qp.c(kD); p2.K2 = kD; p2.b2 = m->g.c(kD); p2.b2_per_seg = 1;
  p2.n_out = 512; p2.bias = W.b0f.as<float>(); p2.c = m->hid.as<float>(); p2.ldc = 512;
  p2.epi = EPI_F32_STATS; p2.statpart = m->statpart.as<float>();
  if (int rc = matcher_gemm(m, p2, st, 2.0 * valid_rows * 512 * 512, "mlp0")) return rc;
  // (6) InstanceNorm statistics per segment (:126)
  LAUNCH(m, st, "in_stats_final", in_stats_final, dim3(S, 16), dim3(32, kStatSlices), 0, st, (const float*)m->statpart.as<float>(), L, m->mu.as<float>(),
         m->rstd.as<float>());
  // (7) x <- x + mlp.3(ReLU(IN(hidden)))  (:122, :59/:64): the converters form hn inside the GEMM, the residual is an identity K-block
  GemmProblem p3{};
  p3.L = L; p3.batch = 1; p3.rows = rows;
  p3.K1 = 512; p3.b1 = W.w1.c(512); p3.n_out = 256; p3.bias = W.b1.as<float>();
  p3.epi = EPI_BIAS_PLANES; p3.out = x.m(kD);
  p3.a2 = x.c(kD); p3.K2 = kD; p3.b2 = m->eye.c(kD); p3.b2_lo_zero = 1; p3.b2_identity = m->identity_diag;
  p3.a_conv = 1; p3.a_raw = m->hid.as<float>(); p3.a_raw_ld = 512; p3.mu = m->mu.as<float>(); p3.rstd = m->rstd.as<float>();
  return matcher_gemm(m, p3, st, 2.0 * valid_rows * 256 * 512, "mlp3");
}

// Object prologue: GNN layers 0 (GATs) and the 3D side of layer 1 (self-attention) depend only on the per-object
// constants (reference GATs_SuperGlue.py:50-54 and :60-64 with src1 = desc3d_db), not on the query frame.  They are
// evaluated ONCE PER OBJECT -- on a single copy of the object's rows, by the first opb_forward after opb_set_object /
// opb_finalize_weights (it needs the chunk workspace) -- and shared by every frame of every later call, like the leaf
// logits s2.  Result: m->xo = 3D-point state entering layer 2.
static int object_prologue(opb_matcher* m, cudaStream_t st) {
  Layout Lo{};
  Lo.B = 1; Lo.N = 0; Lo.M = m->M; Lo.n_pad = 0; Lo.m_pad = m->m_pad; Lo.R = m->m_pad;
  LAUNCH(m, st, "assemble_layout", assemble_layout, dim3(148 * 2, 1), dim3(256), 0, st, (const __half*)nullptr, (const __half*)nullptr,
         (const __half*)m->db.hi.as<__half>(), (const __half*)m->db.lo.as<__half>(), m->xo.hi.as<__half>(), m->xo.lo.as<__half>(), Lo);
  if (int rc = run_gats(m, Lo, m->xo.view(), 0, st)) return rc;
  return run_attn_layer(m, Lo, m->xo.view(), m->attn[0], /*cross=*/0, st);
}

// GNN + tail for `fb` frames starting at frame f0 of the call.
static int forward_chunk(opb_matcher* m, const float* q_cf, const int* nlen, int N, int fb, int64_t* m0, int64_t* m1, float* s0, float* s1,
                         float* conf, cudaStream_t st, int piece, int h2d_first) {
  Layout L{};
  L.B = fb; L.N = N; L.M = m->M; L.n_pad = round_up(N, kSegPad); L.m_pad = m->m_pad; L.R = L.n_pad + L.m_pad;
  L.nlen = nlen;
  m->last_layout = L;
  const int rows = L.rows();
  const double valid_rows = (double)fb * (N + L.M);
  __half *xh = m->x.hi.as<__half>(), *xl = m->x.lo.as<__half>();

  int first_layer = 0;
  if (m->hoist) {
    // layer 1 (self) for the query side only, on a compact [fb*n_pad, 256] buffer; layer 0 does not touch queries.
    // In sub-batches of `piece` frames: with host input (opb_forward_host) each sub-batch starts as soon as ITS descriptors
    // have landed, so the H2D copy of the rest runs under this pass
    for (int p0 = 0, si = 0; p0 < fb; p0 += piece, ++si) {
      const int sb = std::min(piece, fb - p0);
      if (h2d_first + si < m->h2d_pending) CK(m, cudaStreamWaitEvent(st, m->h2d_ev[h2d_first + si], 0));
      Layout Lq{};
      Lq.B = sb; Lq.N = N; Lq.M = 0; Lq.n_pad = L.n_pad; Lq.m_pad = 0; Lq.R = L.n_pad;
      Lq.nlen = nlen ? nlen + p0 : nullptr;
      XView xq = m->xq.view((size_t)p0 * L.n_pad);
      LAUNCH(m, st, "transpose_cf_to_rows", transpose_cf_to_rows<0>, dim3(L.n_pad / 32, sb), dim3(32, 8), 0, st, q_cf + (size_t)p0 * kD * N, N, N,
             (long long)kD * N, Lq.nlen, L.n_pad, xq.hi, xq.lo, (float*)nullptr, (long long)Lq.R, 0);
      if (int rc = run_attn_layer(m, Lq, xq, m->attn[0], 0, st)) return rc;
    }
    // assemble the full layout: query rows from xq, 3D rows from the object prologue
    LAUNCH(m, st, "assemble_layout", assemble_layout, dim3(148 * 2, fb), dim3(256), 0, st, (const __half*)m->xq.hi.as<__half>(),
           (const __half*)m->xq.lo.as<__half>(), (const __half*)m->xo.hi.as<__half>(), (const __half*)m->xo.lo.as<__half>(), xh, xl, L);
    first_layer = 2;
  } else {
    // inputs: query descriptors [fb,256,N] channel-first -> q segments; object rows -> d segments
    LAUNCH(m, st, "transpose_cf_to_rows", transpose_cf_to_rows<0>, dim3(L.n_pad / 32, fb), dim3(32, 8), 0, st, q_cf, N, N, (long long)kD * N, nlen,
           L.n_pad, xh, xl, (float*)nullptr, (long long)L.R, 0);
    LAUNCH(m, st, "assemble_layout", assemble_layout, dim3(148 * 2, fb), dim3(256), 0, st, (const __half*)nullptr, (const __half*)nullptr,
           (const __half*)m->db.hi.as<__half>(), (const __half*)m->db.lo.as<__half>(), xh, xl, L);
  }

  for (int layer = first_layer; layer < 12; ++layer) {
    if (layer % 3 == 0) {
      if (int rc = run_gats(m, L, m->x.view(), layer / 3, st)) return rc;
    } else {
      const int attn_idx = (layer / 3) * 2 + (layer % 3) - 1;
      if (int rc = run_attn_layer(m, L, m->x.view(), m->attn[attn_idx], (layer % 3 == 2) ? 1 : 0, st)) return rc;
    }
  }

  LAUNCH(m, st, "range_check", range_check, dim3((unsigned)(((long long)rows * kD / 8 + 255) / 256)), dim3(256), 0, st, (const __half*)xh,
         (long long)rows * kD / 8, m->range_flag.as<int>());

  // ---- tail (GATs_SuperGlue.py:209-237) ----
  GemmProblem pf{};
  pf.L = L; pf.batch = 1; pf.rows = rows;
  pf.a1 = m->x.c(kD); pf.K1 = kD; pf.b1 = m->wf.c(kD); pf.n_out = 256;
  pf.bias = m->bf.as<float>();
  pf.epi = EPI_L2NORM; pf.out = m->pn.m(kD);       // F.normalize fused into the final_proj epilogue (:209-213)
  if (int rc = matcher_gemm(m, pf, st, 2.0 * valid_rows * kD * kD, "final_proj")) return rc;
  // dual softmax + arg-max as two passes of the batched score GEMM (one batch = one frame); the cos matrix is never stored
  const int n_parts = (L.m_pad / 256) * 2, q_groups = L.n_pad / 32;
  GemmProblem ps{};
  ps.L = L; ps.batch = fb; ps.rows = L.n_pad; ps.n_out = L.m_pad;
  ps.a1 = m->pn.c(kD); ps.K1 = kD; ps.b1 = m->pn.c(kD, (size_t)L.n_pad * kD);
  ps.a_batch_rows = L.R; ps.b_batch_rows = L.R;
  ps.inv_scale = 1.f / m->cfg.scale_factor;
  ps.epi = EPI_SCORE_SUMS; ps.rowsum_part = m->rowsum_part.as<float>(); ps.colsum_part = m->colsum_part.as<float>();
  if (int rc = matcher_gemm(m, ps, st, 2.0 * fb * (double)N * L.M * kD, "score_sums")) return rc;
  LAUNCH(m, st, "score_sums_finalize", score_sums_finalize, dim3((L.n_pad + L.m_pad + 255) / 256, fb), dim3(256), 0, st,
         (const float*)m->rowsum_part.as<float>(), (const float*)m->colsum_part.as<float>(), L, n_parts, q_groups, m->rowsum.as<float>(),
         m->colsum.as<float>(), m->rowbest.as<unsigned long long>(), m->colbest.as<unsigned long long>());
  ps.epi = EPI_SCORE_CONF; ps.inv_rowsum = m->rowsum.as<float>(); ps.inv_colsum = m->colsum.as<float>();
  ps.conf = conf; ps.rowbest = m->rowbest.as<unsigned long long>(); ps.colbest = m->colbest.as<unsigned long long>();
  if (int rc = matcher_gemm(m, ps, st, 0.0, "score_conf")) return rc;      // recomputation: its FLOPs are not algorithmic
  LAUNCH(m, st, "mutual_match", mutual_match, dim3(fb), dim3(256), 0, st, (const unsigned long long*)m->rowbest.as<unsigned long long>(),
         (const unsigned long long*)m->colbest.as<unsigned long long>(), L, m->cfg.match_threshold, (const int*)m->range_flag.as<int>(),
         reinterpret_cast<long long*>(m0), reinterpret_cast<long long*>(m1), s0, s1);
  return 0;
}

static int chunk_of(const opb_matcher* m, int B) {
  int chunk = m->chunk_frames > 0 ? m->chunk_frames : kDefaultChunk;
  return chunk > B ? B : chunk;
}

}  // namespace opb

// =========================================================================================
extern "C" {

int opb_create(const opb_config* cfg, opb_matcher** out) {
  if (!cfg || !out) return fail(nullptr, OPB_E_INVALID, "null argument");
  if (cfg->descriptor_dim != kD || cfg->num_heads != kHeads)
    return fail(nullptr, OPB_E_INVALID, "only descriptor_dim=256, num_heads=4 are supported (got %d, %d)", cfg->descriptor_dim, cfg->num_heads);
  if (!(cfg->scale_factor > 0.f)) return fail(nullptr, OPB_E_INVALID, "scale_factor must be > 0");
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0)
    return fail(nullptr, OPB_E_CUDA, "no CUDA device: %s (this library has no CPU path)", cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= n_dev) return fail(nullptr, OPB_E_INVALID, "device %d out of range", cfg->device);
  e = cudaSetDevice(cfg->device);
  if (e != cudaSuccess) return fail(nullptr, OPB_E_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, cfg->device);
  if (prop.major != 10) return fail(nullptr, OPB_E_CUDA, "device is sm_%d%d; this library is built for sm_100a only", prop.major, prop.minor);
  auto* m = new opb_matcher();
  m->cfg = *cfg;
  m->device = cfg->device;
  m->num_sms = prop.multiProcessorCount;
  if (cudaMallocHost(&m->range_host, sizeof(int)) != cudaSuccess || cudaEventCreateWithFlags(&m->range_ev, cudaEventDisableTiming) != cudaSuccess) {
    delete m;
    return fail(nullptr, OPB_E_CUDA, "pinned flag / event allocation failed");
  }
  *m->range_host = 0;
  *out = m;
  return OPB_OK;
}

void opb_destroy(opb_matcher* m) {
  if (!m) return;
  cudaSetDevice(m->device);
  cudaDeviceSynchronize();
  for (auto& a : m->attn) { a.wqkv.release(); a.bqkv.release(); a.w0a.release(); a.w0m.release(); a.b0f.release(); a.w1.release(); a.b1.release(); }
  DevBuf* bufs[] = {&m->wa2, &m->wa3, &m->bf, &m->leaves, &m->s2, &m->kvt, &m->hid, &m->kvpart, &m->kmean, &m->statpart,
                    &m->mu, &m->rstd, &m->rowsum_part, &m->colsum_part, &m->rowsum, &m->colsum, &m->rowbest, &m->colbest, &m->range_flag,
                    &m->st_q, &m->st_m0, &m->st_m1, &m->st_s0, &m->st_s1, &m->st_conf, &m->st_len};
  for (auto* b : bufs) b->release();
  PlaneBuf* pb[] = {&m->wf, &m->wlin, &m->db, &m->xo, &m->x, &m->qp, &m->pn, &m->g, &m->xq, &m->bd, &m->lin_a, &m->lin_b, &m->eye};
  for (auto* b : pb) b->release();
  for (auto e : m->h2d_ev) cudaEventDestroy(e);
  if (m->copy_stream) cudaStreamDestroy(m->copy_stream);
  if (m->range_ev) cudaEventDestroy(m->range_ev);
  if (m->range_host) cudaFreeHost(m->range_host);
  delete m;
}

const char* opb_last_error(const opb_matcher* m) { return m ? m->err.c_str() : g_last_error.c_str(); }

int opb_load_weight(opb_matcher* m, const char* name, const float* data, size_t n) {
  ENTER(m);
  if (!name || !data) return fail(m, OPB_E_INVALID, "opb_load_weight: null argument");
  m->host_w[name] = std::vector<float>(data, data + n);
  m->weights_ready = false;
  return OPB_OK;
}

int opb_finalize_weights(opb_matcher* m) {
  ENTER(m);
  // head-contiguous channel order: new c' = h*64 + d  <-  reference c = d*4 + h (GATs_SuperGlue.py:97)
  int perm[kD];
  for (int h = 0; h < kHeads; ++h)
    for (int d = 0; d < kDh; ++d) perm[h * kDh + d] = d * kHeads + h;
  std::vector<double> wa2(4 * kD), wa3(4 * kD);
  int ai = 0;
  for (int layer = 0; layer < 12; ++layer) {
    const std::string p = "gnn.layers." + std::to_string(layer);
    if (layer % 3 == 0) {
      const std::vector<float> *W, *a;
      if (int rc = find_w(m, p + ".W", kD * kD, W)) return rc;
      if (int rc = find_w(m, p + ".a", 2 * kD, a)) return rc;
      const int gi = layer / 3;
      for (int c = 0; c < kD; ++c) {  // h @ W @ a[:256] = h . (W a[:256])   (GATs.py:40,78-80)
        double s2 = 0, s3 = 0;
        for (int o = 0; o < kD; ++o) {
          s2 += (double)(*W)[c * kD + o] * (double)(*a)[o];
          s3 += (double)(*W)[c * kD + o] * (double)(*a)[kD + o];
        }
        wa2[gi * kD + c] = s2;
        wa3[gi * kD + c] = s3;
      }
      if (m->cfg.with_linear_transform) {     // B operand of  t = pre . W :  B[o][c] = W[c][o]
        std::vector<double> wt((size_t)kD * kD);
        for (int c = 0; c < kD; ++c)
          for (int o = 0; o < kD; ++o) wt[(size_t)o * kD + c] = (*W)[(size_t)c * kD + o];
        if (int rc = upload_planes(m, m->wlin, wt, (size_t)gi * kD * kD, (size_t)4 * kD * kD)) return rc;
      }
      continue;
    }
    AttnLayerW& A = m->attn[ai++];
    const std::vector<float>*Wp[3], *bp[3], *Wm, *bm, *W0, *b0, *W1, *b1;
    for (int j = 0; j < 3; ++j) {
      if (int rc = find_w(m, p + ".attn.proj." + std::to_string(j) + ".weight", kD * kD, Wp[j])) return rc;
      if (int rc = find_w(m, p + ".attn.proj." + std::to_string(j) + ".bias", kD, bp[j])) return rc;
    }
    if (int rc = find_w(m, p + ".attn.merge.weight", kD * kD, Wm)) return rc;
    if (int rc = find_w(m, p + ".attn.merge.bias", kD, bm)) return rc;
    if (int rc = find_w(m, p + ".mlp.0.weight", 512 * 512, W0)) return rc;
    if (int rc = find_w(m, p + ".mlp.0.bias", 512, b0)) return rc;
    if (int rc = find_w(m, p + ".mlp.3.weight", kD * 512, W1)) return rc;
    if (int rc = find_w(m, p + ".mlp.3.bias", kD, b1)) return rc;
    std::vector<double> wqkv(768 * kD), bqkv(768);
    for (int j = 0; j < 3; ++j)
      for (int c = 0; c < kD; ++c) {
        for (int k = 0; k < kD; ++k) wqkv[((size_t)j * kD + c) * kD + k] = (*Wp[j])[(size_t)perm[c] * kD + k];
        bqkv[j * kD + c] = (*bp[j])[perm[c]];
      }
    std::vector<double> w0a(512 * kD), w0m(512 * kD), b0f(512);
    for (int c = 0; c < 512; ++c) {
      for (int k = 0; k < kD; ++k) w0a[(size_t)c * kD + k] = (*W0)[(size_t)c * 512 + k];
      double bacc = (*b0)[c];
      for (int o = 0; o < kD; ++o) bacc += (double)(*W0)[(size_t)c * 512 + kD + o] * (double)(*bm)[o];
      b0f[c] = bacc;
      for (int k = 0; k < kD; ++k) {  // message channel k (head-contiguous) = reference channel perm[k]
        double acc = 0;
        for (int o = 0; o < kD; ++o) acc += (double)(*W0)[(size_t)c * 512 + kD + o] * (double)(*Wm)[(size_t)o * kD + perm[k]];
        w0m[(size_t)c * kD + k] = acc;
      }
    }
    if (int rc = upload_planes(m, A.wqkv, wqkv)) return rc;
    if (int rc = upload_f32(m, A.bqkv, bqkv)) return rc;
    if (int rc = upload_planes(m, A.w0a, w0a)) return rc;
    if (int rc = upload_planes(m, A.w0m, w0m)) return rc;
    if (int rc = upload_f32(m, A.b0f, b0f)) return rc;
    if (int rc = upload_planes(m, A.w1, std::vector<double>(W1->begin(), W1->end()))) return rc;
    if (int rc = upload_f32(m, A.b1, *b1)) return rc;
  }
  const std::vector<float> *Wf, *bfv;
  if (int rc = find_w(m, "final_proj.weight", kD * kD, Wf)) return rc;
  if (int rc = find_w(m, "final_proj.bias", kD, bfv)) return rc;
  if (int rc = upload_planes(m, m->wf, std::vector<double>(Wf->begin(), Wf->end()))) return rc;
  {
    std::vector<double> eye((size_t)kD * kD, 0.0);
    for (int i = 0; i < kD; ++i) eye[(size_t)i * kD + i] = 1.0;
    if (int rc = upload_planes(m, m->eye, eye)) return rc;
  }
  if (int rc = upload_f32(m, m->bf, *bfv)) return rc;
  if (int rc = upload_f32(m, m->wa2, wa2)) return rc;
  if (int rc = upload_f32(m, m->wa3, wa3)) return rc;
  CK(m, cudaDeviceSynchronize());
  m->weights_ready = true;
  m->object_ready = false;  // s2 and the prologue depend on the weights
  m->prologue_ready = false;
  return OPB_OK;
}

int opb_set_object(opb_matcher* m, const float* desc3d_db, const float* desc2d_db, int32_t M, int32_t Lf, void* stream) {
  ENTER(m);
  if (!m->weights_ready) return fail(m, OPB_E_STATE, "opb_set_object before opb_finalize_weights");
  if (!desc3d_db || !desc2d_db || M <= 0 || Lf <= 0 || Lf > 32)
    return fail(m, OPB_E_INVALID, "set_object: need M > 0 and 1 <= num_leaf <= 32 (got M=%d, L=%d)", M, Lf);
  cudaStream_t st = (cudaStream_t)stream;
  const int m_pad = round_up(M, kSegPad);
  if (m_pad != m->m_pad) { m->ws_frames = 0; m->ws_N = 0; }  // workspace depends on m_pad
  m->M = M; m->Lf = Lf; m->m_pad = m_pad;
  const long long n_leaf_rows = (long long)M * Lf;
  m->leaves.grew = m->db.hi.grew = m->db.lo.grew = m->s2.grew = m->xo.hi.grew = false;
  m->prologue_ready = false;
  CK(m, m->leaves.ensure((size_t)n_leaf_rows * kD * sizeof(float)));
  CK(m, m->db.ensure((size_t)m_pad * kD));
  CK(m, m->s2.ensure((size_t)4 * n_leaf_rows * sizeof(float)));
  CK(m, m->xo.ensure((size_t)m_pad * kD));
  if (m->leaves.grew || m->db.hi.grew || m->s2.grew || m->xo.hi.grew) CK(m, cudaDeviceSynchronize());   // frees of the old buffers vs work in flight
  launch_k(transpose_cf_to_rows<1>, dim3((unsigned)((n_leaf_rows + 31) / 32), 1), dim3(32, 8), 0, st, desc2d_db, (int)n_leaf_rows, (int)n_leaf_rows, 0ll,
           (const int*)nullptr, (int)n_leaf_rows, (__half*)nullptr, (__half*)nullptr, m->leaves.as<float>(), 0ll, 0);
  // rows [M, m_pad) of the object planes are written as zero by the transpose (MODE 0 pads to rows_out)
  launch_k(transpose_cf_to_rows<0>, dim3(m_pad / 32, 1), dim3(32, 8), 0, st, desc3d_db, (int)M, (int)M, 0ll, (const int*)nullptr, m_pad,
           m->db.hi.as<__half>(), m->db.lo.as<__half>(), (float*)nullptr, 0ll, 0);
  launch_k(gats_leaf_logits, dim3(148 * 4), dim3(256), 0, st, (const float*)m->leaves.as<float>(), n_leaf_rows, (const float*)m->wa2.as<float>(),
           m->s2.as<float>());
  CK(m, cudaGetLastError());
  m->object_ready = true;
  return OPB_OK;
}

int opb_reserve_workspace(opb_matcher* m, int32_t frames, int32_t N) {
  ENTER(m);
  if (frames <= 0 || N <= 0) return fail(m, OPB_E_INVALID, "opb_reserve_workspace: bad argument (frames=%d, N=%d)", frames, N);
  if (!m->object_ready) return fail(m, OPB_E_STATE, "opb_reserve_workspace needs an object (the workspace depends on M)");
  return ensure_workspace(m, chunk_of(m, frames), N);
}

int opb_set_hoist(opb_matcher* m, int32_t enable) {
  ENTER(m);
  m->hoist = enable != 0;
  return OPB_OK;
}

int opb_set_chunk_frames(opb_matcher* m, int32_t frames) {
  ENTER(m);
  if (frames < 0) return fail(m, OPB_E_INVALID, "opb_set_chunk_frames: frames %d < 0", frames);
  m->chunk_frames = frames;
  return OPB_OK;
}

int opb_forward(opb_matcher* m, const float* q, const int32_t* n2d_lengths, int32_t B, int32_t N, int64_t* m0, int64_t* m1, float* s0, float* s1,
                float* conf, void* stream) {
  ENTER(m);
  if (!m->weights_ready || !m->object_ready) return fail(m, OPB_E_STATE, "opb_forward needs weights and an object (finalize_weights, set_object)");
  if (!q || !m0 || !m1 || !s0 || !s1 || B <= 0 || N <= 0) return fail(m, OPB_E_INVALID, "opb_forward: bad argument (B=%d, N=%d)", B, N);
  cudaStream_t st = (cudaStream_t)stream;
  const int chunk = chunk_of(m, B);
  if (int rc = ensure_workspace(m, chunk, N)) return rc;   // no-op once opb_reserve_workspace / an earlier call has sized it
  begin_call(m, st);
  if (m->hoist && !m->prologue_ready) {
    if (int rc = object_prologue(m, st)) return rc;
    m->prologue_ready = true;
  }
  // granularity of the query-side layer-1 pass: the host-copy pieces when the queries stream in from the host, else the chunk
  const int piece = m->h2d_pending > 0 ? std::min(chunk, kQPassFrames) : chunk;
  const int ppc = (chunk + piece - 1) / piece;              // pieces per chunk
  for (int f0 = 0, ci = 0; f0 < B; f0 += chunk, ++ci) {
    const int fb = std::min(chunk, B - f0);
    if (!m->hoist)                                          // per-frame evaluation consumes the whole chunk at once
      for (int si = 0; si * piece < fb; ++si)
        if (ci * ppc + si < m->h2d_pending) CK(m, cudaStreamWaitEvent(st, m->h2d_ev[ci * ppc + si], 0));
    int rc = forward_chunk(m, q + (size_t)f0 * kD * N, n2d_lengths ? n2d_lengths + f0 : nullptr, N, fb, m0 + (size_t)f0 * N, m1 + (size_t)f0 * m->M,
                           s0 + (size_t)f0 * N, s1 + (size_t)f0 * m->M, conf ? conf + (size_t)f0 * N * m->M : nullptr, st, piece, ci * ppc);
    if (rc) return rc;
  }
  // deferred range report: the flag travels to pinned host memory behind the call; opb_poll_range() reads it without blocking
  CK(m, cudaMemcpyAsync(m->range_host, m->range_flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(m, cudaEventRecord(m->range_ev, st));
  m->range_pending = true;
  m->last_stream = st;
  end_call(m, st);
  m->last_launches = m->launches;
  return OPB_OK;
}

int opb_set_profiling(opb_matcher* m, int32_t enable) {
  ENTER(m);
  m->profiling = enable != 0;
  return OPB_OK;
}

int opb_get_profile(opb_matcher* m, double* gemm_ms, double* gemm_flops, int32_t* gemm_launches, double* total_ms) {
  if (!m) return fail(nullptr, OPB_E_STATE, "opb_get_profile: null handle");
  ENTER(m);
  if (!m->ev_end) return fail(m, OPB_E_STATE, "opb_get_profile: no profiled call");
  CK(m, cudaEventSynchronize(m->ev_end));
  double ms = 0, fl = 0;
  int n_gemm = 0;
  std::map<std::string, std::pair<double, std::pair<double, int>>> agg;
  for (size_t i = 0; i < m->ev_flops.size(); ++i) {
    float t = 0;
    if (int rc = entry_ms(m, i, &t)) return rc;
    if (m->ev_name[i].compare(0, 4, "gemm") == 0) { ms += t; fl += m->ev_flops[i]; ++n_gemm; }
    auto& a = agg[m->ev_name[i]];
    a.first += t; a.second.first += m->ev_flops[i]; a.second.second++;
  }
  float tot = 0;
  CK(m, cudaEventElapsedTime(&tot, m->ev[0], m->ev_end));
  if (getenv("OPB_PROFILE_DUMP")) {   // measurement aid only: prints the table, selects nothing
    fprintf(stderr, "[opb profile] forward %.3f ms, GEMM %.3f ms in %d launches\n", tot, ms, n_gemm);
    for (auto& kv : agg)
      fprintf(stderr, "[opb profile] %-36s %4d launches %8.3f ms %5.1f%%  %7.1f TFLOP/s algorithmic\n", kv.first.c_str(), kv.second.second.second,
              kv.second.first, 100.0 * kv.second.first / tot, kv.second.second.first / (kv.second.first * 1e-3) / 1e12);
  }
  if (gemm_ms) *gemm_ms = ms;
  if (gemm_flops) *gemm_flops = fl;
  if (gemm_launches) *gemm_launches = (int32_t)n_gemm;
  if (total_ms) *total_ms = tot;
  return OPB_OK;
}

int opb_get_profile_entry(opb_matcher* m, const char* prefix, double* ms_out, double* flops_out, int32_t* launches_out) {
  if (!m) return fail(nullptr, OPB_E_STATE, "opb_get_profile_entry: null handle");
  ENTER(m);
  if (!prefix || !m->ev_end) return fail(m, OPB_E_STATE, "opb_get_profile_entry: no prefix or no profiled call");
  CK(m, cudaEventSynchronize(m->ev_end));
  double ms = 0, fl = 0;
  int n = 0;
  const size_t pl = strlen(prefix);
  for (size_t i = 0; i < m->ev_flops.size(); ++i) {
    if (m->ev_name[i].compare(0, pl, prefix) != 0) continue;
    float t = 0;
    if (int rc = entry_ms(m, i, &t)) return rc;
    ms += t; fl += m->ev_flops[i]; ++n;
  }
  if (ms_out) *ms_out = ms;
  if (flops_out) *flops_out = fl;
  if (launches_out) *launches_out = n;
  return OPB_OK;
}

int opb_forward_host(opb_matcher* m, const float* qh, const int32_t* n2d_lengths_host, int32_t B, int32_t N, int64_t* m0h, int64_t* m1h, float* s0h,
                     float* s1h, float* confh, int32_t materialize_conf, void* stream) {
  ENTER(m);
  if (!m->object_ready) return fail(m, OPB_E_STATE, "opb_forward_host needs an object");
  if (!qh || !m0h || !m1h || !s0h || !s1h || B <= 0 || N <= 0) return fail(m, OPB_E_INVALID, "opb_forward_host: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t M = m->M;
  const bool want_conf = confh != nullptr || materialize_conf != 0;
  DevBuf* stg[] = {&m->st_q, &m->st_m0, &m->st_m1, &m->st_s0, &m->st_s1, &m->st_conf, &m->st_len};
  for (auto* b : stg) b->grew = false;
  CK(m, m->st_q.ensure((size_t)B * kD * N * sizeof(float)));
  CK(m, m->st_m0.ensure((size_t)B * N * sizeof(int64_t)));
  CK(m, m->st_m1.ensure((size_t)B * M * sizeof(int64_t)));
  CK(m, m->st_s0.ensure((size_t)B * N * sizeof(float)));
  CK(m, m->st_s1.ensure((size_t)B * M * sizeof(float)));
  if (want_conf) CK(m, m->st_conf.ensure((size_t)B * N * M * sizeof(float)));
  if (n2d_lengths_host) CK(m, m->st_len.ensure((size_t)B * sizeof(int32_t)));
  // H2D per piece on a side stream: the copy of piece i+1 runs under the compute of piece i
  const int chunk = chunk_of(m, B);
  if (!m->copy_stream) CK(m, cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
  const int piece = std::min(chunk, kQPassFrames);
  const int ppc = (chunk + piece - 1) / piece;
  const int n_chunks = (B + chunk - 1) / chunk;
  const int n_ev = n_chunks * ppc;
  while ((int)m->h2d_ev.size() < n_ev + 1) {
    cudaEvent_t e;
    CK(m, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    m->h2d_ev.push_back(e);
  }
  CK(m, cudaEventRecord(m->h2d_ev[n_ev], st));                           // staging buffer reuse: wait for earlier work on `st`
  CK(m, cudaStreamWaitEvent(m->copy_stream, m->h2d_ev[n_ev], 0));
  if (n2d_lengths_host) CK(m, cudaMemcpyAsync(m->st_len.p, n2d_lengths_host, (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, m->copy_stream));
  for (int ci = 0; ci < n_chunks; ++ci) {
    const int c0 = ci * chunk, cb = std::min(chunk, B - c0);
    for (int si = 0; si < ppc; ++si) {
      const int f0 = c0 + si * piece, fb = std::min(piece, c0 + cb - f0);
      if (fb > 0) {
        const size_t off = (size_t)f0 * kD * N;
        CK(m, cudaMemcpyAsync(m->st_q.as<float>() + off, qh + off, (size_t)fb * kD * N * sizeof(float), cudaMemcpyHostToDevice, m->copy_stream));
      }
      CK(m, cudaEventRecord(m->h2d_ev[ci * ppc + si], m->copy_stream));
    }
  }
  m->h2d_pending = n_ev;
  const int frc = opb_forward(m, m->st_q.as<float>(), n2d_lengths_host ? m->st_len.as<int32_t>() : nullptr, B, N, m->st_m0.as<int64_t>(),
                              m->st_m1.as<int64_t>(), m->st_s0.as<float>(), m->st_s1.as<float>(), want_conf ? m->st_conf.as<float>() : nullptr, stream);
  m->h2d_pending = 0;
  if (frc) return frc;
  CK(m, cudaMemcpyAsync(m0h, m->st_m0.p, (size_t)B * N * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  CK(m, cudaMemcpyAsync(m1h, m->st_m1.p, (size_t)B * M * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  CK(m, cudaMemcpyAsync(s0h, m->st_s0.p, (size_t)B * N * sizeof(float), cudaMemcpyDeviceToHost, st));
  CK(m, cudaMemcpyAsync(s1h, m->st_s1.p, (size_t)B * M * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (confh) CK(m, cudaMemcpyAsync(confh, m->st_conf.p, (size_t)B * N * M * sizeof(float), cudaMemcpyDeviceToHost, st));
  CK(m, cudaStreamSynchronize(st));
  return opb_check_range(m, stream);
}

// Consume the range flag.  After a synchronisation of the stream the pinned copy written behind the last opb_forward is current.
static int consume_range_flag(opb_matcher* m) {
  m->range_pending = false;
  if (*m->range_host == 0) return OPB_OK;
  *m->range_host = 0;
  CK(m, cudaMemsetAsync(m->range_flag.p, 0, sizeof(int), m->last_stream));
  return fail(m, OPB_E_RANGE, "an activation left the fp16-split operand range (|x| >= 1023) or became NaN: the matches of that call were "
                              "reported as -1 (no match)");
}

int opb_check_range(opb_matcher* m, void* stream) {
  if (!m || !m->range_flag.p || !m->range_pending) return OPB_OK;
  (void)stream;
  CK(m, cudaSetDevice(m->device));
  CK(m, cudaEventSynchronize(m->range_ev));
  return consume_range_flag(m);
}

int opb_poll_range(opb_matcher* m) {
  if (!m || !m->range_pending) return OPB_OK;
  CK(m, cudaSetDevice(m->device));
  const cudaError_t q = cudaEventQuery(m->range_ev);
  if (q == cudaErrorNotReady) return OPB_OK;               // the call is still running: report on a later poll / check
  if (q != cudaSuccess) return fail(m, OPB_E_CUDA, "cudaEventQuery: %s", cudaGetErrorString(q));
  return consume_range_flag(m);
}

int opb_last_launch_count(const opb_matcher* m) { return m ? m->last_launches : 0; }

// ---- adjacent producers ------------------------------------------------------------------
static int scan_offsets(const int64_t* seg_len, int32_t M, long long** offs, cudaStream_t st, const char* fn) {
  const cudaError_t e = cudaMallocAsync(offs, (size_t)M * sizeof(long long), st);
  if (e != cudaSuccess) return fail(nullptr, OPB_E_CUDA, "%s: cudaMallocAsync failed: %s", fn, cudaGetErrorString(e));
  exclusive_scan_i64<<<1, 1024, 0, st>>>(reinterpret_cast<const long long*>(seg_len), *offs, M);
  return OPB_OK;
}

int opb_segmented_mean_f64(const double* desc, const int64_t* seg_len, int32_t M, int32_t D, double* out, void* stream) {
  if (!desc || !seg_len || !out || M <= 0 || D <= 0) return fail(nullptr, OPB_E_INVALID, "%s: bad argument (M=%d, D=%d)", __func__, M, D);
  cudaStream_t st = (cudaStream_t)stream;
  long long* offs = nullptr;
  if (int rc = scan_offsets(seg_len, M, &offs, st, __func__)) return rc;
  segmented_mean_f64<<<(unsigned)(((long long)M * 32 + 255) / 256), 256, 0, st>>>(desc, reinterpret_cast<const long long*>(seg_len), offs, M, D, out);
  cudaFreeAsync(offs, st);
  return launch_status(nullptr, __func__);
}

int opb_segmented_mean_scores_f64(const double* scores, const int64_t* seg_len, int32_t M, double* out, void* stream) {
  if (!scores || !seg_len || !out || M <= 0) return fail(nullptr, OPB_E_INVALID, "%s: bad argument (M=%d)", __func__, M);
  cudaStream_t st = (cudaStream_t)stream;
  long long* offs = nullptr;
  if (int rc = scan_offsets(seg_len, M, &offs, st, __func__)) return rc;
  segmented_mean_scores_f64<<<(unsigned)((M + 127) / 128), 128, 0, st>>>(scores, reinterpret_cast<const long long*>(seg_len), offs, M, out);
  cudaFreeAsync(offs, st);
  return launch_status(nullptr, __func__);
}

int opb_gather_features3d(const float* desc, const float* scores, int32_t dim, int64_t n_src, const int64_t* idx, int64_t n_idx, float* desc_out,
                          float* scores_out, int64_t n_out, void* stream) {
  if (!desc || !desc_out || dim <= 0 || n_src < 0 || n_out <= 0 || n_idx < 0 || n_idx > n_out)
    return fail(nullptr, OPB_E_INVALID, "%s: bad argument (dim=%d, n_src=%lld, n_idx=%lld, n_out=%lld)", __func__, dim, (long long)n_src,
                (long long)n_idx, (long long)n_out);
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned gx = (unsigned)((n_out + 255) / 256);
  gather_columns_f32<<<dim3(gx, (unsigned)dim), 256, 0, st>>>(desc, dim, (long long)n_src, reinterpret_cast<const long long*>(idx), (long long)n_idx,
                                                              desc_out, (long long)n_out);
  if (scores && scores_out)
    gather_scores_f32<<<gx, 256, 0, st>>>(scores, (long long)n_src, reinterpret_cast<const long long*>(idx), (long long)n_idx, scores_out, (long long)n_out);
  return launch_status(nullptr, __func__);
}

// ---- test hooks ---------------------------------------------------------------------------
int opb_debug_set_kv_passes(opb_matcher* m, int32_t passes) {
  ENTER(m);
  if (passes != 2 && passes != 3) return fail(m, OPB_E_INVALID, "opb_debug_set_kv_passes: passes %d is not 2 or 3", passes);
  m->kv_two_pass = passes == 2 ? 1 : 0;
  m->prologue_ready = false;
  return OPB_OK;
}

int opb_debug_set_identity_diag(opb_matcher* m, int32_t enable) {
  ENTER(m);
  m->identity_diag = enable ? 1 : 0;
  m->prologue_ready = false;
  return OPB_OK;
}

int opb_debug_set_ws_fill(int32_t byte) {
  g_ws_fill = byte < 0 ? -1 : (byte & 0xFF);
  return OPB_OK;
}

int opb_debug_set_pdl(int32_t enable) {
  set_pdl_enabled(enable != 0);
  return OPB_OK;
}

// Status of a GEMM launch of a debug hook: launch_gemm_* return -1 for a rejected problem, -2 for a CUDA error.
static int gemm_status(int rc, const char* fn) {
  if (rc == 0) return OPB_OK;
  return fail(nullptr, rc == -1 ? OPB_E_INVALID : OPB_E_CUDA, "%s: GEMM launch failed (rc=%d)", fn, rc);
}

static GemmProblem plain_problem(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, float* c, int32_t rows, int32_t n_out, int32_t K) {
  GemmProblem p{};
  p.a1 = CPlanes{(const __half*)a_hi, (const __half*)a_lo, K};
  p.b1 = CPlanes{(const __half*)b_hi, (const __half*)b_lo, K};
  p.K1 = K; p.K2 = 0; p.rows = rows; p.n_out = n_out; p.batch = 1; p.c = c; p.ldc = n_out;
  return p;
}

int opb_debug_gemm(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, float* c, int32_t rows, int32_t n_out, int32_t K,
                   int32_t backend, void* stream) {
  GemmProblem p = plain_problem(a_hi, a_lo, b_hi, b_lo, c, rows, n_out, K);
  return gemm_status(backend == 1 ? launch_gemm_simt(p, (cudaStream_t)stream) : launch_gemm_tc(p, (cudaStream_t)stream), __func__);
}

int opb_debug_gemm_timeline(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, float* c, int32_t rows, int32_t n_out,
                            int32_t K, long long* timeline, void* stream) {
  GemmProblem p = plain_problem(a_hi, a_lo, b_hi, b_lo, c, rows, n_out, K);
  return gemm_status(launch_gemm_tc(p, (cudaStream_t)stream, timeline), __func__);
}

int opb_debug_gemm_aconv(const float* a_raw, const void* b_hi, const void* b_lo, void* x_hi, void* x_lo, const float* mu, const float* rstd,
                         const float* bias, const void* eye_hi, const void* eye_lo, int32_t rows, long long* timeline, void* stream) {
  // the mlp.3 problem of one segment: x[rows,256] = [ReLU((a_raw - mu) * rstd) | x] . [B | I]^T + bias, converters on
  if (!eye_hi || !eye_lo) return fail(nullptr, OPB_E_INVALID, "%s: null identity planes", __func__);
  GemmProblem p{};
  p.b1 = CPlanes{(const __half*)b_hi, (const __half*)b_lo, 512};
  p.K1 = 512; p.rows = rows; p.n_out = 256; p.batch = 1; p.bias = bias;
  p.L.B = 1; p.L.N = rows; p.L.M = 0; p.L.n_pad = rows; p.L.m_pad = 0; p.L.R = rows;
  p.epi = EPI_BIAS_PLANES; p.out = Planes{(__half*)x_hi, (__half*)x_lo, kD};
  p.a2 = CPlanes{(const __half*)x_hi, (const __half*)x_lo, kD}; p.K2 = kD; p.b2 = CPlanes{(const __half*)eye_hi, (const __half*)eye_lo, kD};
  p.b2_lo_zero = 1; p.b2_identity = 1;
  p.a_conv = 1; p.a_raw = a_raw; p.a_raw_ld = 512; p.mu = mu; p.rstd = rstd;
  return gemm_status(launch_gemm_tc(p, (cudaStream_t)stream, timeline), __func__);
}

int opb_debug_kv_state_h(const void* kvh, int32_t frames, int32_t n, int32_t m_pts, int32_t slabs_per_group, float* partial, int32_t* n_groups,
                         void* stream) {
  Layout L{};
  L.B = frames; L.N = n; L.M = m_pts; L.n_pad = (n + kSegPad - 1) / kSegPad * kSegPad; L.m_pad = (m_pts + kSegPad - 1) / kSegPad * kSegPad;
  L.R = L.n_pad + L.m_pad;
  KvGroups G = kv_groups_for(L, 148);
  if (slabs_per_group > 0) {
    G.slabs = slabs_per_group;
    G.gq = (L.n_pad / 256 + G.slabs - 1) / G.slabs;
    G.gd = (L.m_pad / 256 + G.slabs - 1) / G.slabs;
  }
  if (n_groups) *n_groups = frames * (G.gq + G.gd);
  if (!partial) return OPB_OK;                    // size query
  if (launch_kv_state_h((const __half*)kvh, L, G, partial, (cudaStream_t)stream)) return fail(nullptr, OPB_E_CUDA, "%s: launch failed", __func__);
  return OPB_OK;
}

int opb_debug_split(const float* x, void* hi, void* lo, size_t n, void* stream) {
  split_planes<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, (__half*)hi, (__half*)lo, (long long)n);
  return launch_status(nullptr, __func__);
}

int opb_debug_read(opb_matcher* m, int32_t which, float* out, size_t cap, int64_t* rows, void* stream) {
  ENTER(m);
  if (!out) return fail(m, OPB_E_INVALID, "debug_read: null output");
  const Layout& L = m->last_layout;
  if (which == 0) {
    size_t n = (size_t)L.rows() * kD;
    if (rows) *rows = L.rows();
    if (n > cap) return fail(m, OPB_E_INVALID, "debug_read: capacity %zu < %zu", cap, n);
    join_planes<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(m->x.hi.as<__half>(), m->x.lo.as<__half>(), out, (long long)n);
    return launch_status(m, __func__);
  }
  return fail(m, OPB_E_INVALID, "debug_read: unknown buffer %d", which);
}

}  // extern "C"
