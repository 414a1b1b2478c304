/*
 * onepose_b200 -- C ABI of the B200-native GATsSPG 2D-3D matcher.
 *
 * The reference (zju3dv/OnePose) is pure Python and has no FFI; the boundary it
 * exposes for this path is `GATsSuperGlue.forward(data) -> (pred, conf_matrix)`
 * (reference src/models/GATsSPG_architectures/GATs_SuperGlue.py:179-241), reached
 * through `LitModelGATsSPG.forward` (src/models/GATsSPG_lightning_model.py:36-37)
 * from inference.py:146.  Each entry point below names the reference code it
 * replaces.  All signatures are plain C: pointers, sizes, a cudaStream_t passed
 * as void*.  No torch types.  Every function returns 0 on success or a negative
 * OPB_E_* code; opb_last_error() gives the message.  No exceptions cross the ABI.
 *
 * Pointer ownership: inputs are borrowed and never written; outputs are caller
 * allocated (device memory unless the name says _host).
 */
#ifndef ONEPOSE_B200_H_
#define ONEPOSE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OPB_OK 0
#define OPB_E_INVALID (-1)      /* bad argument / unsupported configuration        */
#define OPB_E_CUDA (-2)         /* CUDA runtime / driver error                      */
#define OPB_E_STATE (-3)        /* call order violated (weights / object missing)   */
#define OPB_E_RANGE (-4)        /* activation left the fp16-split operand range     */
#define OPB_E_NOT_IMPLEMENTED (-5)

typedef struct opb_matcher opb_matcher; /* opaque */

/* Hyper-parameters = the `hparams` mapping of GATsSuperGlue.__init__
 * (GATs_SuperGlue.py:145-177; released values configs/experiment/train_GATsSPG.yaml:44-60). */
typedef struct opb_config {
  int32_t descriptor_dim;        /* 256 (only value supported)                         */
  int32_t num_heads;             /* 4   (GATs_SuperGlue.py:43)                          */
  float scale_factor;            /* 0.07 (GATs_SuperGlue.py:217)                        */
  float match_threshold;         /* 0.2  (GATs_SuperGlue.py:227)                        */
  int32_t include_self;          /* GATs.py:48                                          */
  int32_t additional;            /* GATs.py:61                                          */
  int32_t with_linear_transform; /* GATs.py:56-57,64-65                                 */
  int32_t device;                /* CUDA device ordinal                                 */
} opb_config;

/* Replaces GATsSuperGlue.__init__ (GATs_SuperGlue.py:145-177). */
int opb_create(const opb_config* cfg, opb_matcher** out);
void opb_destroy(opb_matcher* m);
const char* opb_last_error(const opb_matcher* m); /* m may be NULL: message of this thread's last failed call that had no handle */

/* Replaces nn.Module.load_state_dict for the keys of GATs_SuperGlue.py (SURVEY 2.1):
 * `name` is the reference state-dict key ("gnn.layers.1.attn.proj.0.weight", ...),
 * `data` a HOST fp32 array in the reference's own layout.  Dead parameters
 * (kenc_*, bin_score) are accepted and ignored.  opb_finalize_weights() packs
 * (head permutation, merge->mlp.0 folding, W.a folding, fp16 hi/lo split) and uploads. */
int opb_load_weight(opb_matcher* m, const char* name, const float* data, size_t n_elems);
int opb_finalize_weights(opb_matcher* m);

/* Per-object constants = the tensors inference.py:113-130 builds once per sequence
 * and pack_data (inference.py:80-94) re-uploads every frame:
 *   desc3d_db  device fp32 [256, M]    (descriptors3d_db, channel-first)
 *   desc2d_db  device fp32 [256, M*L]  (descriptors2d_db, column i*L+j = leaf j of point i; GATs.py:46) */
int opb_set_object(opb_matcher* m, const float* desc3d_db, const float* desc2d_db,
                   int32_t M, int32_t L, void* stream);

/* Size the chunk workspace for calls of up to `frames` frames of up to N query points each (SURVEY 8b: no allocation on the
 * hot path beyond a workspace sized with the object).  Optional: opb_forward grows the workspace itself on first use / when a
 * call exceeds what was reserved (a one-time cudaMalloc + device synchronisation). */
int opb_reserve_workspace(opb_matcher* m, int32_t frames, int32_t N);

/* Replaces GATsSuperGlue.forward (GATs_SuperGlue.py:179-241) for B query frames of
 * the current object.  desc2d_query: device fp32 [B, 256, N] (channel-first, as in
 * the reference).  n2d_lengths: device int32 [B] = valid query points of each frame (SuperPoint yields a different count per
 * frame, src/sfm/extract_features.py:19-24; columns >= n2d_lengths[b] of frame b are ignored) or NULL = N everywhere.
 * Outputs (device): matches0 int64 [B,N], matches1 int64 [B,M], mscores0 fp32 [B,N], mscores1 fp32 [B,M]; conf fp32 [B,N,M]
 * or NULL to skip materialising the confidence matrix.  Entries of a frame beyond its length are -1 / 0.
 * Asynchronous on `stream`; no host synchronisation. */
int opb_forward(opb_matcher* m, const float* desc2d_query, const int32_t* n2d_lengths, int32_t B, int32_t N,
                int64_t* matches0, int64_t* matches1, float* mscores0, float* mscores1,
                float* conf, void* stream);

/* Same call with HOST buffers (pinned or pageable): H2D of the query descriptors (and lengths, may be NULL),
 * forward, D2H of matches/scores; returns after the stream has been synchronised.  The confidence matrix is
 * materialised on the device if conf_host is non-NULL (then also copied back) or materialize_conf != 0
 * (the reference always computes it; inference.py:146 discards it).  This is the end-to-end leg bench.py times. */
int opb_forward_host(opb_matcher* m, const float* desc2d_query_host, const int32_t* n2d_lengths_host, int32_t B, int32_t N,
                     int64_t* matches0_host, int64_t* matches1_host, float* mscores0_host,
                     float* mscores1_host, float* conf_host, int32_t materialize_conf, void* stream);

/* Range guard of the fp16-split operand format (|x| < 1023 per plane element).  A call that produced an activation outside the
 * range (or a NaN) reports "no match" (-1 / 0) for every point on the device, and the error is delivered to the host lazily:
 *   opb_poll_range   never blocks: OPB_E_RANGE if a finished earlier call raised the flag, OPB_OK otherwise (also while
 *                    the last call is still running);
 *   opb_check_range  waits for the last opb_forward and reports.  opb_forward_host calls it itself.
 * Reporting clears the flag. */
int opb_check_range(opb_matcher* m, void* stream);
int opb_poll_range(opb_matcher* m);

/* Number of kernels opb_forward launched in its last call (bench.py "gpu_launches"). */
int opb_last_launch_count(const opb_matcher* m);

/* Measurement hook for bench.py: with profiling on, every launch of opb_forward is followed by a CUDA event on the launch
 * stream.  opb_get_profile() synchronises and returns the summed GEMM time, the ALGORITHMIC FLOPs those launches performed
 * (2*valid_rows*n_out*K, each logical MMA counted once although it executes as 3 fp16 passes), their count, and the time of the
 * whole forward (first to last kernel).  Profiling perturbs timing slightly: never on in timed runs. */
int opb_set_profiling(opb_matcher* m, int32_t enable);
int opb_get_profile(opb_matcher* m, double* gemm_ms, double* gemm_flops, int32_t* gemm_launches, double* total_ms);
/* Same for the launches whose profile name starts with `prefix` ("gemm epi1 " = the mlp.0 GEMM, "kv_state", ...). */
int opb_get_profile_entry(opb_matcher* m, const char* prefix, double* ms, double* flops, int32_t* launches);

/* GNN layers 0 (GATs) and the 3D side of layer 1 (self) depend only on the per-object constants; by default they
 * are evaluated once per opb_forward call and shared by its frames.  enable = 0 evaluates them per frame like the
 * reference does (same results up to fp32 rounding; used by the tests). */
int opb_set_hoist(opb_matcher* m, int32_t enable);

/* Frames processed together through the GNN (workspace-size knob); 0 = default (32). */
int opb_set_chunk_frames(opb_matcher* m, int32_t frames);

/* ---- adjacent producers: the per-object feature files the path consumes (SURVEY 8f N2) ---- */
/* mean_descriptors (reference src/sfm/postprocess/feature_process.py:297-305, fp64):
 * desc device f64 [sum(seg_len), D], seg_len device int64 [M] -> out device f64 [M, D]. */
int opb_segmented_mean_f64(const double* desc, const int64_t* seg_len, int32_t M, int32_t D,
                           double* out, void* stream);
/* mean_scores (feature_process.py:308-317, fp64): scores device f64 [sum(seg_len)] -> out device f64 [M]
 * (numpy's pairwise summation order reproduced, bit-identical). */
int opb_segmented_mean_scores_f64(const double* scores, const int64_t* seg_len, int32_t M, double* out, void* stream);
/* Column gather of pad_features3d_random / build_features3d_leaves (reference src/utils/data_utils.py:143-205):
 * desc device fp32 [dim, n_src] (channel-first), scores device fp32 [n_src] (may be NULL), idx device int64 [n_idx] = source
 * column of each output column (n_src = the all-ones / zero-score dustbin; NULL = identity) -> desc_out [dim, n_out],
 * scores_out [n_out]; output columns >= n_idx are all-ones / zero padding. */
int opb_gather_features3d(const float* desc, const float* scores, int32_t dim, int64_t n_src, const int64_t* idx, int64_t n_idx,
                          float* desc_out, float* scores_out, int64_t n_out, void* stream);

/* ---- adjacent consumer: object pose from the matched correspondences (SURVEY 8f N3) ----
 * Replaces the per-frame cv2.solvePnPRansac(..., reprojectionError=5, iterationsCount=10000, flags=SOLVEPNP_EPNP) of
 * ransac_PnP (reference src/utils/eval_utils.py:18-42) for B frames in one call, on the device:
 *   K          device f64 [B, 9]   row-major camera matrices
 *   pts2d      device f64 [total, 2], pts3d device f64 [total, 3]  matched key points of all frames, concatenated
 *   offsets    device int32 [B+1]  frame b owns correspondences [offsets[b], offsets[b+1])
 *   hypotheses minimal samples per frame (P3P), reproj_error in pixels, seed of the sample generator (results are a
 *              deterministic function of it)
 *   workspace  device f64 [B * hypotheses * 13]
 * Outputs (device): pose f64 [B, 12] = row-major [R | t] (world -> camera), inlier_mask int32 [total], n_inliers int32 [B].
 * A frame with fewer than 4 correspondences or no model gets the identity pose and no inliers (the reference's cv2.error
 * branch).  Parity with the reference is on the pose (cm / degree), not on bits: OpenCV draws its own samples. */
int opb_ransac_pnp(const double* K, const double* pts2d, const double* pts3d, const int32_t* offsets, int32_t B, int32_t hypotheses,
                   double reproj_error, uint64_t seed, double* workspace, double* pose_out, int32_t* inlier_mask, int32_t* n_inliers,
                   void* stream);

/* ---- adjacent producer: SuperPoint key-point extractor (SURVEY 8f N4) ----
 * Replaces SuperPoint.forward (reference src/models/extractors/SuperPoint/superpoint.py:140-197): shared VGG-style encoder
 * (:142-152), score head + 65-way softmax + 8x8 pixel shuffle (:155-160), simple_nms (:47-61, :161), threshold / border /
 * top-k key-point selection (:163-174), descriptor head (:180-181) and bilinear descriptor sampling (:79-92, :184-185).
 * Its outputs are the `keypoints2d` / `descriptors2d_query` tensors inference.py:80-94 packs for the matcher; with a fixed
 * capacity (max_keypoints >= 0) they stay on the device: descriptors [B, 256, cap] + counts [B] are exactly the
 * `desc2d_query` / `n2d_lengths` arguments of opb_forward. */
typedef struct opb_superpoint opb_superpoint; /* opaque */

/* = the `config` mapping of SuperPoint.__init__ merged over its default_config (superpoint.py:97-103).  Note that the released
 * inference configuration (src/sfm/extract_features.py:19-24) spells the threshold key 'keypoints_threshold', so the default
 * 0.005 is what the reference runs with; nms_radius 3, max_keypoints 4096. */
typedef struct opb_sp_config {
  int32_t descriptor_dim;     /* 256 (only value supported)                                                    */
  int32_t nms_radius;         /* 0..6                                                                          */
  float keypoint_threshold;   /* superpoint.py:164                                                             */
  int32_t max_keypoints;      /* > 0, or -1 = keep all (superpoint.py:133-135 raises for 0 and < -1)            */
  int32_t remove_borders;     /* superpoint.py:64-69                                                           */
  int32_t align_corners;      /* grid_sample flag: 1 under the reference's pinned torch 1.8 (superpoint.py:86)  */
  int32_t device;
} opb_sp_config;

int opb_sp_create(const opb_sp_config* cfg, opb_superpoint** out);
void opb_sp_destroy(opb_superpoint* h);
const char* opb_sp_last_error(const opb_superpoint* h); /* h may be NULL: message of this thread's last failed call that had no handle */
/* Reference state-dict keys ("conv1a.weight", "conv1a.bias", ... "convDb.bias"; superpoint.py:111-126), HOST fp32 arrays in
 * the reference's own [C_out, C_in, kh, kw] layout.  opb_sp_finalize_weights packs them (tap-major reduction index, the two
 * heads' 3x3 layers side by side, fp16 hi/lo split) and uploads. */
int opb_sp_load_weight(opb_superpoint* h, const char* name, const float* data, size_t n_elems);
int opb_sp_finalize_weights(opb_superpoint* h);
/* First half of forward(): image device fp32 [B, 1, H, W] (H, W multiples of 8) -> internal candidate lists.
 * counts (device int32 [B], may be NULL) receives the number of key points opb_sp_describe will emit for each image
 * (= min(#candidates, max_keypoints)); a caller that needs exactly-sized outputs reads it (the reference synchronises at the
 * same point: torch.nonzero, superpoint.py:163-165) and passes cap = max(counts). */
int opb_sp_detect(opb_superpoint* h, const float* image, int32_t B, int32_t H, int32_t W, int32_t* counts, void* stream);
/* Second half: key points (x, y) fp32 [B, cap, 2], scores fp32 [B, cap], descriptors fp32 [B, 256, cap] (channel-first like the
 * reference's [256, n]; may be NULL), counts int32 [B]; entries >= counts[b] are not written.  Order: row-major (torch.nonzero)
 * or, when an image has more than max_keypoints candidates, descending score (torch.topk). */
int opb_sp_describe(opb_superpoint* h, float* keypoints, float* scores, float* descriptors, int32_t* counts, int32_t cap, void* stream);
/* Both halves with a caller-chosen capacity, no host synchronisation (cap >= max_keypoints makes it exact). */
int opb_sp_forward(opb_superpoint* h, const float* image, int32_t B, int32_t H, int32_t W, float* keypoints, float* scores,
                   float* descriptors, int32_t* counts, int32_t cap, void* stream);
int opb_sp_last_launch_count(const opb_superpoint* h);
/* bench.py hooks: with profiling on, an event follows every launch of opb_sp_detect / opb_sp_describe; entry i = launch i
 * (name, milliseconds, algorithmic FLOPs of a convolution: 2 * interior pixels * C_out * 9 * C_in). */
int opb_sp_set_profiling(opb_superpoint* h, int32_t enable);
int opb_sp_get_profile(opb_superpoint* h, int32_t index, char* name, size_t name_cap, double* ms, double* flops);
/* test hooks: stop the encoder after step i (0 conv1a, 1 conv1b, 2 pool, 3 conv2a, 4 conv2b, 5 pool, 6 conv3a, 7 conv3b, 8 pool,
 * 9 conv4a, 10 conv4b, 11 [convPa|convDa]; -1 = run everything) and read internal tensors as fp32: which = 0 dense scores
 * [B,H,W], 1 scores after NMS, 2 convPb output rows [B*P, 128], 3 convDb output rows [B*P, 256], 4 the activation of the last
 * step run, rows of the zero-bordered pixel grid [B*P, C]. */
int opb_sp_debug_set_stop(opb_superpoint* h, int32_t layer);
/* 3x3 convolutions on the 64- / 128-wide column tiles: 1 (default) = halo boxes (one (128 + 2)-row A box per kernel row and
 * 64-channel block serves the three horizontal taps through row-offset UMMA descriptors: a third of the L2 -> shared-memory
 * traffic), 0 = nine row-shifted boxes per tile.  Same operand bytes (bit-identical results with 64 input channels; a different
 * accumulation order of the same products with 128); A/B switch for tests/ and tools/. */
int opb_debug_set_conv_halo(int32_t mode);
int opb_sp_debug_read(opb_superpoint* h, int32_t which, float* out, size_t capacity_elems, int64_t* n_elems, void* stream);

/* ---- test hooks (used by tests/ and tools/ only; stable but not part of the drop-in surface) ---- */
/* Programmatic dependent launch on (default) / off for every launch of the library (A/B measurements). */
int opb_debug_set_pdl(int32_t enable);
/* byte >= 0: every workspace / object buffer allocated from now on is filled with `byte` (0xFF = NaN patterns) unless the
 * algorithm requires it to start as zero; -1: off.  Proves that no result depends on uninitialised memory. */
int opb_debug_set_ws_fill(int32_t byte);
/* Tensor-core passes of the k,v projection: 2 (default: A_hi.(B_hi + B_lo); its output is rounded to one fp16 plane anyway) or
 * 3 (the full split product), for the precision A/B in tests/ and tools/. */
int opb_debug_set_kv_passes(opb_matcher* m, int32_t passes);
/* Residual of a layer = identity K-block of its mlp.3 GEMM.  1 (default): k-block j runs as N = 64 MMAs on accumulator columns
 * [64 j, 64 j + 64) against the 64 x 64 diagonal block of I (a quarter of the tensor work); 0: full-width MMAs against I.
 * Bit-identical results (the skipped products are exact zeros); A/B switch for tests/ and tools/. */
int opb_debug_set_identity_diag(opb_matcher* m, int32_t enable);
/* C[rows, n_out] (fp32, ld = n_out) = A . B^T with fp16-split operands.  a_hi/a_lo [rows, K], b_hi/b_lo [n_out, K];
 * rows % 256 == 0, K % 64 == 0, n_out % 256 == 0.  backend 0 = the tcgen05 core, 1 = SIMT fp32 FFMA cross-check
 * (rows, n_out % 128 == 0, K % 16 == 0). */
int opb_debug_gemm(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo,
                   float* c, int32_t rows, int32_t n_out, int32_t K, int32_t backend, void* stream);
/* Same through the tcgen05 core with a per-CTA clock64 timeline (device int64 [n_ctas][64]); tuning aid. */
int opb_debug_gemm_timeline(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo,
                            float* c, int32_t rows, int32_t n_out, int32_t K, long long* timeline, void* stream);
/* The fp16 linear-attention state kernel on a caller-supplied plane kvh [frames*(n_pad+m_pad), 512] (pad rows must be
 * zero); slabs_per_group = 0: the library's own choice; *n_groups = number of partial states; partial [n_groups][4][64*64+64]
 * (NULL: size query only). */
int opb_debug_kv_state_h(const void* kvh, int32_t frames, int32_t n, int32_t m_pts, int32_t slabs_per_group, float* partial,
                         int32_t* n_groups, void* stream);
/* The mlp.3 GEMM of one segment with the A-operand converters on: x = [ReLU((a_raw - mu) * rstd) | x] . [B | I]^T + bias;
 * a_raw fp32 [rows,512], B planes [256,512], x planes [rows,256] updated in place, mu/rstd [512], eye planes [256,256]. */
int opb_debug_gemm_aconv(const float* a_raw, const void* b_hi, const void* b_lo, void* x_hi, void* x_lo, const float* mu,
                         const float* rstd, const float* bias, const void* eye_hi, const void* eye_lo, int32_t rows,
                         long long* timeline, void* stream);
/* fp32 [rows, cols] -> fp16-split planes: hi = fp16(64 x), lo = fp16(64 x - hi). */
int opb_debug_split(const float* x, void* hi, void* lo, size_t n, void* stream);
/* Copy an internal activation buffer of the last forward to `out` (device fp32):
 * which = 0: X [B*(n_pad+m_pad), 256] reconstructed from its planes. Returns rows via *rows. */
int opb_debug_read(opb_matcher* m, int32_t which, float* out, size_t capacity_elems, int64_t* rows, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ONEPOSE_B200_H_ */
