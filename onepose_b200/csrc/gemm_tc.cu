// tcgen05 / TMA GEMM core for sm_100a -- persistent, warp-specialised, 2-CTA UMMA, TMEM double-buffered.
//
//   C[128 x 256 tile] = sum_k A_tile . B_tile^T     A, B: fp16-split planes (hi, lo; common.cuh), K-major
//
// Each logical product runs as THREE tensor-core passes into ONE fp32 TMEM accumulator
//     D += A_hi.B_hi + A_hi.B_lo + A_lo.B_hi            (x 2^-12 in the epilogue)
// which reproduces fp32 products to ~2^-22 relative (tools/precision_ladder.py); the reference
// computes in fp32 (GATs_SuperGlue.py:191-193) and the contract is 1e-4 abs on conf.
//
// Persistent grid (one CTA per SM), static round-robin tile schedule (n-tile fastest so CTAs that share an A row-tile run
// together).  A CTA pair (cluster of 2, tcgen05 cta_group::2) works on two adjacent row tiles; each CTA keeps its own A tile
// and HALF of the B tile in shared memory -- the shared-memory port, not the tensor pipe, limited the 1-CTA form.  384 threads:
//   warp 0     TMA producer   cp.async.bulk.tensor 2D, SWIZZLE_128B boxes -> 3-stage smem ring (64 KB per stage)
//   warp 1     MMA issuer     one lane of the leader CTA: tcgen05.mma kind::f16, tcgen05.commit -> mbarriers of both CTAs
//   warp 2     TMEM owner     512 columns = 2 accumulator buffers x 256 (epilogue of tile i overlaps the main loop of tile i+1)
//   warps 4-11 epilogue       two groups of 4 warps (each group = the 4 TMEM lane quarters) splitting the tile's columns:
//                             tcgen05.ld -> registers -> fused op -> swizzled smem staging -> TMA store
// Converter variant (ACV_NORM_RELU, 512 threads): warps 4-7 = one epilogue group, warps 8-15 = A-operand converters that turn a
// raw fp32 tile landed by TMA into the (hi, lo) planes in place; setmaxnreg rebalances the registers.
// Every kernel starts with griddepcontrol.wait after its on-chip set-up (programmatic dependent launch: the set-up of launch
// i+1 overlaps the tail of launch i).
#include <cuda.h>

#include <cstdlib>

#include <map>
#include <mutex>
#include <tuple>

#include "gemm_tc.cuh"
#include "host_util.cuh"

namespace opb {
namespace {

constexpr int BM = 128, BN = 256, BK = 64;
constexpr int UMMA_K = 16;
constexpr int kStagesFull = 3;
constexpr int kABytes = BM * BK * 2;             // one plane of this CTA's A tile (16 KB)
constexpr int kBBytes = (BN / 2) * BK * 2;       // one plane of this CTA's HALF of the B tile (16 KB)
constexpr int kStageBytesFull = 2 * kABytes + 2 * kBBytes;
constexpr int kStagingBytes = 16384;             // one 128-row x 128-B swizzled epilogue buffer
constexpr int kNumStaging = 2;
constexpr int kExtraBytes = 1024;                // per-tile scratch of the score epilogue (inverse column sums of the tile)
constexpr int kSmemBytes = kStagesFull * kStageBytesFull + kNumStaging * kStagingBytes + 1024 /*align*/ + 256 /*barriers*/ + kExtraBytes;
constexpr uint32_t kSBO = 8 * BK * 2;            // bytes between 8-row groups of a K-major SWIZZLE_128B operand
constexpr int kTmemCols = 512;
// warps 0-3: TMA / MMA / TMEM / spare.  Plain variants: warps 4-11 = two epilogue groups of 4 warps (384 threads).
// Converter variant: warps 4-7 = one epilogue group, warps 8-15 = eight A-operand converter warps (512 threads, 128 registers
// per thread at launch; the converters hand 24 registers each to the epilogue group via setmaxnreg).
constexpr int threads_of(int acv) { return acv ? 512 : 384; }
constexpr int kConvWarps = 8;
constexpr int kConvRegs = 104, kEpiRegsAcv = 176;   // 128 + 176 + 2 x 104 = 512 = 4 warpgroups x 128
constexpr uint32_t kSpinLimit = 1u << 22;        // bounded waits: trap instead of hanging the GPU

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > kSpinLimit) __trap();
  }
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c_inner, int c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c_inner), "r"(c_outer)
      : "memory");
}
// 2-CTA (cta_group::2) forms
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* map, uint64_t* leader_bar, int c_inner, int c_outer) {
  // data lands in THIS CTA's smem; the transaction bytes are credited to the leader CTA's mbarrier (peer bit cleared)
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(map), "r"(smem_u32(leader_bar) & 0xFEFFFFFFu), "r"(c_inner), "r"(c_outer)
      : "memory");
}
__device__ __forceinline__ void tc_mma_f16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
__device__ __forceinline__ void tc_commit_2sm(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta_rank) {
  asm volatile(
      "{\n\t.reg .b32 remAddr32;\n\t"
      "mapa.shared::cluster.u32 remAddr32, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [remAddr32];\n\t}" ::"r"(smem_u32(bar)),
      "r"(cta_rank)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c_inner, int c_outer) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map), "r"(smem_u32(smem_src)),
               "r"(c_inner), "r"(c_outer)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map), "r"(smem_u32(smem_src)),
               "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) { asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
template <uint32_t R>
__device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(R)); }
template <uint32_t R>
__device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(R)); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_id(int id) { asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory"); }   // the 4 warps of one epilogue group

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 "version 1"):
//   start address >> 4 | LBO (unused for swizzled K-major; 1) | SBO = bytes between 8-row groups | swizzle mode
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(kSBO >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;                        // SWIZZLE_128B
  return d;
}
// Same for an operand whose first row is row `r0` of the box that was landed at `smem_addr` (1024-byte aligned): the start
// address simply moves by r0 * 128 bytes.  The swizzle XOR is a function of the ABSOLUTE shared-memory address bits (the
// hardware un-swizzles exactly what TMA wrote), so a row-offset start needs nothing else -- measured on B200: with the
// descriptor's "matrix base offset" field (bits 49-51) left at 0 the results are bit-identical to separately loaded boxes,
// with base offset = r0 they are garbage.  Used by the halo convolution: one 130-row box serves the three horizontal taps.
__device__ __forceinline__ uint64_t make_desc_rowoff(uint32_t smem_addr, uint32_t r0) { return make_desc(smem_addr + r0 * 128u); }
// kind::f16 instruction descriptor (built per column-tile width inside the kernel): D=f32, A=B=f16, both K-major, M = 256 across
// the CTA pair, N = BN

// byte offset of 16-byte chunk j of row r inside a 128-row x 128-B SWIZZLE_128B staging buffer
__device__ __forceinline__ uint32_t stg_off(int r, int j) { return (uint32_t)(r * 128 + ((j ^ (r & 7)) << 4)); }
// same for a 128-row x 64-B SWIZZLE_64B buffer (16-byte chunk j in 0..3): Swizzle<2,4,3> = address bits [4,6) ^= bits [7,9)
__device__ __forceinline__ uint32_t stg64_off(int r, int j) { return (uint32_t)(r * 64 + ((j ^ ((r >> 1) & 3)) << 4)); }

struct TcParams {
  int K1, K2;            // reduction split (multiples of BK)
  int b2_per_seg;
  int b2_lo_zero;        // skip the A_hi . B_lo pass of the K2 block (identity K-block: B_lo == 0)
  int b2_identity;       // K2 block = identity: diagonal 64 x 64 blocks as N = 64 MMAs (GemmProblem::b2_identity)
  int n_out;
  int m_tiles, n_tiles, batch;
  long long a_batch_rows, b_batch_rows;
  int c_batch_rows;      // output rows per batch (C is [batch*rows, ldc])
  int seg_rows;          // rows are rows of the activation layout L (segment-aware masking); 0: plain matrix
  Layout L;
  const float* bias;
  long long* tl;         // optional timeline buffer (debug)
  // fused epilogues
  const float* kmean;    // EPI_QSCALE
  int cross;
  float* statpart;       // EPI_F32_STATS
  // A-operand converters (ACV)
  const float* mu;       // ACV_NORM_RELU: [S][512]
  const float* rstd;
  // EPI_SCORE_*
  float inv_scale;
  float* rowsum_part;
  float* colsum_part;
  const float* inv_rowsum;
  const float* inv_colsum;
  float* conf;
  int conf_tma;          // 1: conf goes out through the 3-D tensor map (M % 4 == 0), 0: plain stores from the staged chunk
  unsigned long long* rowbest;
  unsigned long long* colbest;
  // implicit-GEMM convolution (GemmProblem::taps) and the EPI_CONV geometry
  int taps, kb_per_tap;
  int tap_off[9];
  int cv_w2, cv_h, cv_w, cv_ppad, relu;
  int halo;              // 3x3 convolution with one (BM + 2)-row A box per (kernel row, 64-channel block)
};

struct Maps {
  CUtensorMap a1h, a1l, a2h, a2l, b1h, b1l, b2h, b2l;   // loads
  CUtensorMap out_f32;                                    // store: fp32 [rows, ldc], box 32 x 128 (SWIZZLE_128B)
  CUtensorMap out_hi, out_lo;                             // store: fp16-split planes, box 32 x 128 (SWIZZLE_64B)
  CUtensorMap a_raw;                                      // load: fp32 source of a converted A operand, box 32 x 128 (SWIZZLE_128B)
                                                          // (halo convolution: a1h / a1l have boxes of BM + 2 rows)
};

// A-operand conversion: instead of fp16-split planes prepared by a separate kernel, the TMA producer lands the RAW fp32
// tile (128 rows x 64 columns = exactly the 32 KB of the stage's A_hi + A_lo planes) and eight converter warps rewrite it
// IN PLACE as the (hi, lo) planes the UMMA descriptors expect -- the pointwise op between two GEMMs runs on data that is
// already on the SM, and its 4 KB/row HBM round trip disappears:
//   ACV_NORM_RELU  A  = ReLU((hid - mu_seg) * rstd_seg)          mlp.3 reads mlp.0's fp32 output (GATs_SuperGlue.py:126-127)
enum { ACV_NONE = 0, ACV_NORM_RELU = 1 };

// HI: the A operand enters with its hi plane only (k,v projection, GemmProblem::a_hi_only): the stage shrinks to A_hi + B_hi + B_lo =
// 48 KB and the ring deepens to FOUR stages in the same 192 KB -- with two passes a k-block is only ~1k cycles of MMA, and three
// stages cannot cover the ~4k-cycle turn-around of a stage (load issue -> data landed) any more.
// BN_: column-tile width (256 for every matcher GEMM; 64 / 128 for the narrow convolution layers of the extractor: the B half-tile
// shrinks to BN_/2 rows per CTA and the ring deepens to four stages).
template <int EPI, int ACV = ACV_NONE, bool HI = false, int BN_ = 256>
__global__ void __launch_bounds__(threads_of(ACV), 1) gemm_tc_kernel(const __grid_constant__ Maps maps, TcParams p) {
  constexpr int BN = BN_;
  constexpr int kBBytes = (BN / 2) * BK * 2;
  constexpr int kStageBytesFull = 2 * kABytes + 2 * kBBytes;
  constexpr uint32_t kIdesc2 = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);
  constexpr uint32_t kIdesc64 = (1u << 4) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);   // N = 64 (identity K-block)
  constexpr int kDiagBBytes = 32 * BK * 2;         // this CTA's half (32 rows) of a 64 x 64 diagonal block of the identity
  static_assert(BN_ == 256 || (BN_ == 64 || BN_ == 128) && ACV == ACV_NONE && !HI && (EPI == EPI_CONV || EPI == EPI_F32), "narrow tiles: conv / fp32 epilogues only");
  constexpr int kStages = (HI || BN_ != 256) ? 4 : kStagesFull;
  constexpr int kStageBytes = HI ? kABytes + 2 * kBBytes : kStageBytesFull;
  constexpr int kBOff = HI ? kABytes : 2 * kABytes;      // offset of the B planes inside a stage
  static_assert(!HI || ACV == ACV_NONE, "converters need the full stage");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  // halo convolution (EPI_CONV, TcParams::halo): a stage = one (kernel row, 64-channel block) group = A_hi / A_lo boxes of BM + 2
  // rows (the three horizontal taps read it at row offsets 0 / 1 / 2) + the B half-tiles of the three taps
  constexpr int kHaloRows = BM + 2;
  constexpr int kHaloABytes = (kHaloRows * 128 + 1023) / 1024 * 1024;         // 17408
  constexpr int kHaloStageBytes = 2 * kHaloABytes + 6 * kBBytes;
  constexpr int kHaloStages = (EPI == EPI_CONV && BN_ != 256) ? (BN_ == 64 ? 3 : 2) : 0;
  constexpr int kRingBytes = kStages * kStageBytes > kHaloStages * kHaloStageBytes ? kStages * kStageBytes : kHaloStages * kHaloStageBytes;
  static_assert(kRingBytes <= kStagesFull * (2 * kABytes + 2 * (256 / 2) * BK * 2), "ring exceeds the shared-memory budget");
  const bool halo = EPI == EPI_CONV && kHaloStages > 0 && p.halo != 0;
  // Split accumulators (narrow tiles only: a 256-column buffer holds 256 / BN accumulators).  The fp32 TMEM accumulator is
  // TRUNCATED on every MMA, a bias toward zero that grows with the number of accumulate steps at full magnitude.  The two
  // correction passes (A_hi.B_lo, A_lo.B_hi: 2^-11 of the main term) get an accumulator of their own, and with 64-wide tiles the
  // main term is further split by kernel row; the epilogue adds the partial sums in registers with round-to-nearest.
  constexpr bool kSplitAcc = BN_ != 256;
  constexpr int kBufCols = kSplitAcc ? 256 : BN;                 // TMEM columns per accumulator buffer
  constexpr int kMainAcc = BN_ == 64 ? 3 : 1;                    // accumulators of the A_hi.B_hi term (3: one per kernel row of a 3x3 convolution)
  // accumulator slots of a buffer: 0 = main[0], 1 = corrections, 2.. = main[1..] (written by 3x3 convolutions only)
  const int n_main = (kMainAcc > 1 && EPI == EPI_CONV && p.taps == 9) ? kMainAcc : 1;
  constexpr int kHaloStagesDiv = kHaloStages ? kHaloStages : 1;  // (modulus of the halo ring; never used when there is none)
  uint8_t* staging = smem + kRingBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(staging + kNumStaging * kStagingBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full_bar = empty_bar + kStages;     // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;      // [2]
  uint64_t* raw_bar = tmem_empty_bar + 2;            // [kStages] raw fp32 A tile has landed (ACV)
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(raw_bar + kStages);
  float* extra = reinterpret_cast<float*>(staging + kNumStaging * kStagingBytes + 256);   // kExtraBytes of per-tile scratch

  // Epilogue groups: the TMEM -> registers -> staging -> TMA-store chain of one 32-column chunk is a serial latency chain
  // (tcgen05.ld, two named barriers, proxy fence), so ONE group of 4 warps drains a 128 x 256 tile in ~8.5k cycles no matter
  // how little it computes.  Two groups (each: 4 warps = the 4 TMEM lane quarters) split the tile's columns and overlap
  // their chains.  With A-operand converters, warps 8-15 convert and one group drains the accumulator.
  constexpr int kEpiGroups = ACV == ACV_NONE ? 2 : 1;
  constexpr int kColsPerGroup = BN / kEpiGroups;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb1 = p.K1 / BK, nkb = (p.K1 + p.K2) / BK;
  // work unit = 2 adjacent row tiles x one n-tile; this CTA takes row tile (2*mgroup + crank)
  const int crank = (int)cluster_ctarank();
  const int units_per_batch = (p.m_tiles / 2) * p.n_tiles;
  const int total_units = units_per_batch * p.batch;
  const int unit0 = blockIdx.x / 2, unit_step = gridDim.x / 2;
  long long* tl = p.tl ? p.tl + (long long)blockIdx.x * 64 : nullptr;
  if (tl && threadIdx.x == 0) tl[0] = clock64();

  if (threadIdx.x == 0) {
    // full: the TMA transaction arrive (+ with converters: one arrive per converter warp of BOTH CTAs, on the leader)
    for (int s = 0; s < kStages; ++s) { mbar_init(&full_bar[s], ACV ? 1 + 2 * kConvWarps : 1); mbar_init(&empty_bar[s], 1); mbar_init(&raw_bar[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full_bar[b], 1); mbar_init(&tmem_empty_bar[b], 8 * kEpiGroups); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&maps.a1h); prefetch_tmap(&maps.a1l); prefetch_tmap(&maps.b1h); prefetch_tmap(&maps.b1l);
    if (p.K2) { prefetch_tmap(&maps.a2h); prefetch_tmap(&maps.a2l); prefetch_tmap(&maps.b2h); prefetch_tmap(&maps.b2l); }
    if (ACV) prefetch_tmap(&maps.a_raw);
    if (EPI == EPI_F32 || EPI == EPI_F32_STATS || EPI == EPI_SCORE_CONF) prefetch_tmap(&maps.out_f32);
    if (EPI == EPI_QKV || EPI == EPI_QSCALE || EPI == EPI_L2NORM || EPI == EPI_BIAS_PLANES || EPI == EPI_CONV) { prefetch_tmap(&maps.out_hi); prefetch_tmap(&maps.out_lo); }
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_slot)), "n"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                  // peer barriers are initialised before any remote arrive / 2-CTA load can land
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;
  griddep_sync();                      // results of the previous launch are visible from here on; let the next launch set up
  if (tl && threadIdx.x == 0) tl[1] = clock64();

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t it = 0;   // k-block counter across all tiles of this CTA
      constexpr int kBRowsLoad = BN / 2;
      for (int u = unit0; u < total_units; u += unit_step) {
        const int z = u / units_per_batch, rem = u - z * units_per_batch;
        const int m_tile = (rem / p.n_tiles) * 2 + crank, n_tile = rem % p.n_tiles;
        const int row0 = m_tile * BM;
        const int a_row = (int)(z * p.a_batch_rows) + row0;
        const int b_row1 = (int)(z * p.b_batch_rows) + n_tile * BN + crank * kBRowsLoad;
        const int seg = p.b2_per_seg ? p.L.seg_of_row(row0) : 0;     // the pair's row tiles share a segment (segments are 256-row aligned)
        const int b_row2 = (p.b2_per_seg ? seg * p.n_out : 0) + n_tile * BN + crank * kBRowsLoad;
        if (halo) {
          const int ngroups = 3 * p.kb_per_tap;
          for (int g = 0; g < ngroups; ++g, ++it) {
            const int s = it % kHaloStagesDiv;
            mbar_wait(&empty_bar[s], ((it / kHaloStagesDiv) & 1) ^ 1);
            uint8_t* st = smem + s * kHaloStageBytes;
            if (crank == 0) mbar_expect_tx(&full_bar[s], 2 * (2 * kHaloRows * 128 + 6 * kBBytes));
            const int dy = g / p.kb_per_tap, cb = g - dy * p.kb_per_tap;
            const int arow = a_row + (dy - 1) * p.cv_w2 - 1;          // first row of the box: tap (dy, dx = 0); may be < 0 (zero fill)
            tma_load_2d_2sm(st, &maps.a1h, &full_bar[s], cb * BK, arow);
            tma_load_2d_2sm(st + kHaloABytes, &maps.a1l, &full_bar[s], cb * BK, arow);
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) {
              const int kcb = ((dy * 3 + dx) * p.kb_per_tap + cb) * BK;
              tma_load_2d_2sm(st + 2 * kHaloABytes + dx * 2 * kBBytes, &maps.b1h, &full_bar[s], kcb, b_row1);
              tma_load_2d_2sm(st + 2 * kHaloABytes + dx * 2 * kBBytes + kBBytes, &maps.b1l, &full_bar[s], kcb, b_row1);
            }
          }
          continue;
        }
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % kStages;
          mbar_wait(&empty_bar[s], ((it / kStages) & 1) ^ 1);
          uint8_t* st = smem + s * kStageBytes;
          const bool first = kb < nkb1;
          const bool conv = ACV == ACV_NORM_RELU && first;           // this k-block's A tile comes in raw
          const bool diag = BN_ == 256 && !first && p.b2_identity;     // identity K-block: B = one 64 x 64 diagonal block, hi plane only
          if (crank == 0)                                               // leader arms for both CTAs' loads
            mbar_expect_tx(&full_bar[s], conv ? 4 * kBBytes : (diag ? 2 * (2 * kABytes + kDiagBBytes) : 2 * kStageBytes));
          int kc = (first ? kb * BK : (kb - nkb1) * BK);
          int arow = a_row, kcb = kc;                                   // A rows / B columns of this k-block
          if (EPI == EPI_CONV && p.taps) {                              // implicit-GEMM convolution: tap t = row-shifted A, B columns follow kb
            const int t = kb / p.kb_per_tap;
            kcb = kb * BK;
            kc = (kb - t * p.kb_per_tap) * BK;
            arow = a_row + p.tap_off[t];                                // may leave [0, rows): the tensor map zero-fills
          }
          const CUtensorMap* mah = first ? &maps.a1h : &maps.a2h;
          const CUtensorMap* mal = first ? &maps.a1l : &maps.a2l;
          const CUtensorMap* mbh = first ? &maps.b1h : &maps.b2h;
          const CUtensorMap* mbl = first ? &maps.b1l : &maps.b2l;
          const int brow = first ? b_row1 : b_row2;
          if (conv) {
            // raw fp32 [128 x 64] = two 32-column boxes, landing where the hi / lo planes will be written
            mbar_expect_tx(&raw_bar[s], 2 * kABytes);
            tma_load_2d(st, &maps.a_raw, &raw_bar[s], kc, a_row);
            tma_load_2d(st + kABytes, &maps.a_raw, &raw_bar[s], kc + 32, a_row);
          } else {
            tma_load_2d_2sm(st, mah, &full_bar[s], kc, arow);
            if (!HI) tma_load_2d_2sm(st + kABytes, mal, &full_bar[s], kc, arow);
          }
          if (diag) {                                                   // rows [kc + 32 crank, +32) x columns [kc, kc + 64) of I (box: 32 rows)
            tma_load_2d_2sm(st + kBOff, mbh, &full_bar[s], kc, kc + crank * 32);
            continue;
          }
          tma_load_2d_2sm(st + kBOff, mbh, &full_bar[s], kcb, brow);
          tma_load_2d_2sm(st + kBOff + kBBytes, mbl, &full_bar[s], kcb, brow);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (the leader CTA issues for the pair) =====================
    if (lane == 0 && crank == 0) {
      uint32_t it = 0, tc = 0;
      for (int u = unit0; u < total_units; u += unit_step, ++tc) {
        const uint32_t buf = tc & 1;
        mbar_wait(&tmem_empty_bar[buf], ((tc >> 1) & 1) ^ 1);     // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d = tmem_base + buf * kBufCols;
        uint32_t started = 0;                                       // split accumulators already written in this tile
        auto acc_of = [&](int a, uint32_t& flag) {                   // TMEM address of split accumulator a; flag = accumulate?
          flag = (started >> a) & 1u;
          started |= 1u << a;
          return d + (uint32_t)(a * BN);
        };
        if (halo) {
          const int ngroups = 3 * p.kb_per_tap;
          for (int g = 0; g < ngroups; ++g, ++it) {
            const int s = it % kHaloStagesDiv;
            mbar_wait(&full_bar[s], (it / kHaloStagesDiv) & 1);
            tc_fence_after();
            const uint32_t sa_h = smem_u32(smem + s * kHaloStageBytes), sa_l = sa_h + kHaloABytes;
            const int am = (g / p.kb_per_tap) % n_main;             // kernel row -> main accumulator
            uint32_t fm, fc;
            const uint32_t dm = acc_of(am ? am + 1 : 0, fm), dc = acc_of(1, fc);
            // (issuing the group's main term first and the corrections afterwards, or keeping a single main accumulator, measured
            // the same time: tools/conv_halo_ab.py)
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) {
              const uint32_t sb_h = sa_h + 2 * kHaloABytes + dx * 2 * kBBytes, sb_l = sb_h + kBBytes;
#pragma unroll
              for (int k = 0; k < BK / UMMA_K; ++k) {
                const uint32_t koff = k * UMMA_K * 2;
                const uint64_t ah = make_desc_rowoff(sa_h + koff, dx), al = make_desc_rowoff(sa_l + koff, dx);
                const uint64_t bh = make_desc(sb_h + koff), bl = make_desc(sb_l + koff);
                tc_mma_f16_2sm(dm, ah, bh, kIdesc2, (dx | k) ? 1u : fm);
                tc_mma_f16_2sm(dc, ah, bl, kIdesc2, (dx | k) ? 1u : fc);
                tc_mma_f16_2sm(dc, al, bh, kIdesc2, 1u);
              }
            }
            tc_commit_2sm(&empty_bar[s], (uint16_t)0x3);
          }
          tc_commit_2sm(&tmem_full_bar[buf], (uint16_t)0x3);
          continue;
        }
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % kStages;
          mbar_wait(&full_bar[s], (it / kStages) & 1);
          if (tl && tc == 1 && kb < 16) tl[20 + kb] = clock64();
          tc_fence_after();
          const uint32_t sa_h = smem_u32(smem + s * kStageBytes);
          const uint32_t sa_l = sa_h + kABytes, sb_h = sa_h + kBOff, sb_l = sb_h + kBBytes;
          const bool skip_lo = p.b2_lo_zero && kb >= nkb1;          // B_lo == 0: the A_hi.B_lo pass adds exact zeros
          if (BN_ == 256 && kb >= nkb1 && p.b2_identity) {
            // identity K-block j: only output columns [64 j, 64 j + 64) receive anything -> N = 64 MMAs on that slice of the
            // accumulator (the other 192 columns of a full-width MMA would add exact zeros)
            const uint32_t dj = d + (uint32_t)(kb - nkb1) * 64u;
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              const uint32_t koff = k * UMMA_K * 2;
              const uint64_t bh = make_desc(sb_h + koff);
              tc_mma_f16_2sm(dj, make_desc(sa_h + koff), bh, kIdesc64, 1u);
              tc_mma_f16_2sm(dj, make_desc(sa_l + koff), bh, kIdesc64, 1u);
            }
            tc_commit_2sm(&empty_bar[s], (uint16_t)0x3);
            continue;
          }
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint32_t koff = k * UMMA_K * 2;   // bytes inside the swizzle row
            const uint64_t ah = make_desc(sa_h + koff), al = make_desc(sa_l + koff);
            const uint64_t bh = make_desc(sb_h + koff), bl = make_desc(sb_l + koff);
            if (kSplitAcc) {                                        // narrow tiles: never HI / skip_lo (launch_gemm_tc)
              uint32_t fm, fc;
              const int dy = (EPI == EPI_CONV && p.taps == 9) ? kb / (3 * p.kb_per_tap) : 0;
              const int am = dy % n_main;
              const uint32_t dm = acc_of(am ? am + 1 : 0, fm), dc = acc_of(1, fc);
              tc_mma_f16_2sm(dm, ah, bh, kIdesc2, fm);
              tc_mma_f16_2sm(dc, ah, bl, kIdesc2, fc);
              tc_mma_f16_2sm(dc, al, bh, kIdesc2, 1u);
              continue;
            }
            tc_mma_f16_2sm(d, ah, bh, kIdesc2, (uint32_t)((kb | k) != 0));
            if (!skip_lo) tc_mma_f16_2sm(d, ah, bl, kIdesc2, 1u);
            if (!HI) tc_mma_f16_2sm(d, al, bh, kIdesc2, 1u);
          }
          tc_commit_2sm(&empty_bar[s], (uint16_t)0x3);              // frees the stage in both CTAs
        }
        tc_commit_2sm(&tmem_full_bar[buf], (uint16_t)0x3);          // accumulator halves complete in both CTAs
      }
    }
  } else if (ACV != ACV_NONE && warp >= 8) {
    // ===================== A-operand converters (warps 8-15): raw fp32 tile -> (hi, lo) planes, in place =====================
    // Warp cw owns rows [16 cw, 16 cw + 16) of the tile: it reads exactly the smem bytes it later overwrites (row r of the raw
    // boxes and row r of the planes are the same two 128-byte slots), so a __syncwarp between the read and the write phase is
    // the only ordering needed.  Lane = (row 4i + lane/8, 8-column group c = lane%8): reads raw chunks 2c', 2c'+1 of box c/4,
    // writes chunk c of both planes -- every shared-memory instruction touches each bank group exactly once per wavefront.
    reg_dec<kConvRegs>();
    constexpr int kLPR = BK / 8;                     // lanes per row = 8-column groups per k-block
    constexpr int kRPI = 32 / kLPR;                  // rows per shared-memory instruction
    constexpr int kRowIters = BM / kConvWarps / kRPI;
    const int cw = warp - 8;
    const int c = lane % kLPR, rsub = lane / kLPR;
    // proxy fence + plain (remote) arrive on the leader's barrier -- the pattern CUTLASS's 2-SM transform warps use.  A
    // .release.cluster arrive compiles to MEMBAR.ALL.GPU and costs ~4k cycles per k-block (measured).
    auto conv_arrive = [crank](uint64_t* bar) {
      if (crank != 0) mbar_arrive_remote(bar, 0);
      else mbar_arrive(bar);
    };
    uint32_t it = 0, raw_phase = 0, tidx = 0;
    for (int u = unit0; u < total_units; u += unit_step, ++tidx) {
      const int z = u / units_per_batch, rem = u - z * units_per_batch;
      const int m_tile = (rem / p.n_tiles) * 2 + crank;
      const int row0 = m_tile * BM;
      const int seg = p.L.seg_of_row(row0);
      (void)z;
      for (int kb = 0; kb < nkb; ++kb, ++it) {
        const int s = it % kStages;
        const bool conv = kb < nkb1;
        if (!conv) {
          // plain TMA k-block: nothing to convert, but the barrier's arrival count is fixed -- arrive once the stage's
          // previous use has been consumed (so the arrival lands in the right phase)
          mbar_wait(&empty_bar[s], ((it / kStages) & 1) ^ 1);
          __syncwarp();
          if (lane == 0) conv_arrive(&full_bar[s]);
          continue;
        }
        const uint32_t st = smem_u32(smem) + s * kStageBytes;
        const uint32_t rawbox = st + ((2 * c) >> 3) * (BM * 128);
        const int kcol = kb * BK + 8 * c;            // first of this lane's 8 source columns
        float pa[8], pb[8];                          // per-column parameters: (-64 mu rstd, 64 rstd)
        {
          const float* base_a = p.mu + (long long)seg * 512 + kcol;
          const float4 a0 = __ldg(reinterpret_cast<const float4*>(base_a)), a1 = __ldg(reinterpret_cast<const float4*>(base_a) + 1);
          pa[0] = a0.x; pa[1] = a0.y; pa[2] = a0.z; pa[3] = a0.w; pa[4] = a1.x; pa[5] = a1.y; pa[6] = a1.z; pa[7] = a1.w;
          const float* base_b = p.rstd + (long long)seg * 512 + kcol;
          const float4 b0 = __ldg(reinterpret_cast<const float4*>(base_b)), b1 = __ldg(reinterpret_cast<const float4*>(base_b) + 1);
          pb[0] = b0.x; pb[1] = b0.y; pb[2] = b0.z; pb[3] = b0.w; pb[4] = b1.x; pb[5] = b1.y; pb[6] = b1.z; pb[7] = b1.w;
          // 64 * ReLU((h - mu) * rstd) = max(h * (64 rstd) - 64 mu rstd, 0): one FFMA + one FMNMX per element, pre-scale included
#pragma unroll
          for (int j = 0; j < 8; ++j) { pb[j] *= kPre; pa[j] = -pa[j] * pb[j]; }
        }
        mbar_wait(&raw_bar[s], (raw_phase >> s) & 1);
        raw_phase ^= 1u << s;
        if (tl && cw == 0 && lane == 0 && tidx == 1 && kb < 8) tl[3 + 2 * kb] = clock64();
        float4 ra[kRowIters], rb[kRowIters];
#pragma unroll
        for (int i = 0; i < kRowIters; ++i) {
          const int r = cw * (BM / kConvWarps) + kRPI * i + rsub;
          ra[i] = lds128(rawbox + r * 128 + ((((2 * c) & 7) ^ (r & 7)) << 4));
          rb[i] = lds128(rawbox + r * 128 + ((((2 * c + 1) & 7) ^ (r & 7)) << 4));
        }
        __syncwarp();                      // every lane holds its raw values before any lane overwrites them
#pragma unroll
        for (int i = 0; i < kRowIters; ++i) {
          const int r = cw * (BM / kConvWarps) + kRPI * i + rsub;
          float v[8] = {ra[i].x, ra[i].y, ra[i].z, ra[i].w, rb[i].x, rb[i].y, rb[i].z, rb[i].w};
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = fmaxf(fmaf(v[j], pb[j], pa[j]), 0.f);     // already x 2^6
          uint4 oh, ol;
#pragma unroll
          for (int j = 0; j < 4; ++j) {    // same rounding as split_f32, two elements per conversion instruction
            const float2 sc = make_float2(v[2 * j], v[2 * j + 1]);
            const __half2 h2 = __float22half2_rn(sc);
            const float2 back = __half22float2(h2);
            const __half2 l2 = __float22half2_rn(make_float2(sc.x - back.x, sc.y - back.y));
            reinterpret_cast<__half2*>(&oh)[j] = h2;
            reinterpret_cast<__half2*>(&ol)[j] = l2;
          }
          sts128(st + stg_off(r, c), oh);
          sts128(st + kABytes + stg_off(r, c), ol);
        }
        fence_async_smem();                // generic-proxy writes -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) conv_arrive(&full_bar[s]);
        if (tl && cw == 0 && lane == 0 && tidx == 1 && kb < 8) tl[4 + 2 * kb] = clock64();
      }
    }
  } else if (warp >= 4 && warp < 4 + 4 * kEpiGroups) {
    // ===================== epilogue: TMEM -> registers -> staging smem -> TMA store =====================
    if (ACV != ACV_NONE) reg_inc<kEpiRegsAcv>();
    const int grp = (warp - 4) >> 2;                // epilogue group: columns [grp*kColsPerGroup, +kColsPerGroup) of every tile
    const int q = (warp - 4) & 3;                   // TMEM lane quarter == warp_id % 4
    const int r_in_tile = q * 32 + lane;
    const int t_in_grp = threadIdx.x - 128 - grp * 128;
    const bool leader = t_in_grp == 0;
    const int c_begin = grp * kColsPerGroup, c_end = c_begin + kColsPerGroup;
    auto epi_bar = [grp]() { epi_bar_id(1 + grp); };
    // staging: one group -> two buffers used alternately; two groups -> one buffer each (the other group's chain overlaps)
    auto stage_sel = [grp](uint32_t ctr) { return kEpiGroups == 2 ? (uint32_t)grp : (ctr & 1u); };
    auto stage_wait = [leader]() {
      if (leader) {
        if (kEpiGroups == 2) tma_store_wait_read<0>();
        else tma_store_wait_read<1>();
      }
    };
    uint32_t tc = 0, chunk_ctr = 0;
    for (int u = unit0; u < total_units; u += unit_step, ++tc) {
      const int z = u / units_per_batch, rem = u - z * units_per_batch;
      const int m_tile = (rem / p.n_tiles) * 2 + crank, n_tile = rem % p.n_tiles;
      const uint32_t buf = tc & 1;
      mbar_wait(&tmem_full_bar[buf], (tc >> 1) & 1);
      if (tl && threadIdx.x == 128 && tc < 8) tl[40 + 2 * tc] = clock64();
      tc_fence_after();
      const uint32_t lane_base = tmem_base + buf * kBufCols + ((uint32_t)(q * 32) << 16);
      // 32 accumulator columns starting at c: one tcgen05.ld, or (split accumulators) the round-to-nearest sum of the partials
      auto load_acc = [&](int c, uint32_t (&v)[32]) {
        tmem_ld32(lane_base + c, v);
        tmem_ld_wait();
        if (kSplitAcc) {
#pragma unroll
          for (int a = 1; a <= kMainAcc; ++a) {
            if (a > n_main) break;
            uint32_t t[32];
            tmem_ld32(lane_base + a * BN + c, t);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(t[j]));
          }
        }
      };
      const int out_row0 = z * p.c_batch_rows + m_tile * BM;
      const int row0 = m_tile * BM;                               // within the batch
      int n_valid = BM;                                           // valid rows of this tile (segment-aware launches)
      int seg = 0;
      if (p.seg_rows) {
        seg = p.L.seg_of_row(row0);
        n_valid = p.L.seg_valid(seg) - (row0 - p.L.seg_start(seg));
      }
      if (EPI == EPI_F32 || EPI == EPI_F32_STATS) {
        // ---- fp32 tile out through swizzled staging + TMA store, 32 columns per chunk
#pragma unroll 1
        for (int c0 = c_begin; c0 < c_end; c0 += 32, ++chunk_ctr) {
          uint32_t v[32];
          load_acc(c0, v);
          const int col0 = n_tile * BN + c0;
          uint8_t* sb = staging + stage_sel(chunk_ctr) * kStagingBytes;
          stage_wait();                             // the store that last read this buffer is done with it
          epi_bar();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float4 o;
            o.x = __uint_as_float(v[4 * j + 0]) * kProdInv;
            o.y = __uint_as_float(v[4 * j + 1]) * kProdInv;
            o.z = __uint_as_float(v[4 * j + 2]) * kProdInv;
            o.w = __uint_as_float(v[4 * j + 3]) * kProdInv;
            if (p.bias) {
              const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + 4 * j));
              o.x += bb.x; o.y += bb.y; o.z += bb.z; o.w += bb.w;
            }
            *reinterpret_cast<float4*>(sb + stg_off(r_in_tile, j)) = o;
          }
          fence_async_smem();
          epi_bar();
          if (leader) {
            tma_store_2d(&maps.out_f32, sb, col0, out_row0);
            tma_store_commit();
          }
          if (EPI == EPI_F32_STATS) {
            // InstanceNorm partial sums straight from the staged tile: thread = (32-row quarter, column)
            const int t = t_in_grp, qq = t >> 5, cc = t & 31;
            float sum = 0.f, sq = 0.f;
            const int r_end = min(32, n_valid - qq * 32);
            for (int i = 0; i < r_end; ++i) {
              const int r = qq * 32 + i;
              const float x = *reinterpret_cast<const float*>(sb + stg_off(r, cc >> 2) + (cc & 3) * 4);
              sum += x;
              sq = fmaf(x, x, sq);
            }
            float2* dst = reinterpret_cast<float2*>(p.statpart) + ((long long)(out_row0 / 32 + qq) * p.n_out + col0 + cc);
            *dst = make_float2(sum, sq);
          }
        }
      } else if (EPI == EPI_QKV) {
        // ---- [K | V] tiles of the k,v projection -> one fp16 plane (x 2^6), 64 columns per chunk (128-byte staging rows).
        // elu+1 on K (GATs_SuperGlue.py:71-72); pad rows are zeroed so the state kernel needs no row masks.
        const bool is_k = n_tile == 0;
        const bool row_ok = r_in_tile < n_valid;
#pragma unroll 1
        for (int c0 = c_begin; c0 < c_end; c0 += 64, ++chunk_ctr) {
          uint32_t v0[32], v1[32];
          tmem_ld32(lane_base + c0, v0);
          tmem_ld32(lane_base + c0 + 32, v1);
          tmem_ld_wait();
          const int col0 = n_tile * BN + c0;
          uint8_t* sb = staging + stage_sel(chunk_ctr) * kStagingBytes;
          stage_wait();
          epi_bar();
#pragma unroll
          for (int j8 = 0; j8 < 8; ++j8) {
            const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + j8 * 8));
            const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + j8 * 8 + 4));
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
            float x[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int jj = j8 * 8 + e;
              x[e] = fmaf(__uint_as_float(jj < 32 ? v0[jj & 31] : v1[jj & 31]), kProdInv, bb[e]);
              if (is_k) x[e] = elu1_fast(x[e]);
              x[e] = row_ok ? x[e] * kPre : 0.f;
            }
            uint4 o;
#pragma unroll
            for (int e = 0; e < 4; ++e) reinterpret_cast<__half2*>(&o)[e] = __float22half2_rn(make_float2(x[2 * e], x[2 * e + 1]));
            *reinterpret_cast<uint4*>(sb + stg_off(r_in_tile, j8)) = o;
          }
          fence_async_smem();
          epi_bar();
          if (leader) {
            tma_store_2d(&maps.out_hi, sb, col0, out_row0);
            tma_store_commit();
          }
        }
      } else if (EPI == EPI_SCORE_SUMS) {
        // ---- dual-softmax tail, pass 1 (reference GATs_SuperGlue.py:217-218).  Unit-norm operands: cos <= 1, so with the
        // fixed shift  e = exp((cos - 1)/scale)  softmax(s,1)*softmax(s,2) = e^2 / (colsum*rowsum)  needs no running max.
        // Nothing is stored but the partial sums: row sums per (tile half, row) in registers; column sums over the warp's 32
        // rows by a transposing butterfly (31 shuffles per 32 x 32 block, no shared memory, no barriers).
        const int Nz = p.L.n_of(z), M = p.L.M;
        const int row = row0 + r_in_tile;                          // query index inside frame z
        const bool row_ok = row < Nz;
        const float ea = kProdInv * p.inv_scale * 1.4426950408889634f, eb = -p.inv_scale * 1.4426950408889634f;
        float rs = 0.f;
#pragma unroll 1
        for (int c0 = c_begin; c0 < c_end; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(lane_base + c0, v);
          tmem_ld_wait();
          const int col0 = n_tile * BN + c0;
          float e[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const bool ok = row_ok && (col0 + j) < M;
            e[j] = ok ? ex2_fast(fmaf(__uint_as_float(v[j]), ea, eb)) : 0.f;
            rs += e[j];
          }
          // after the butterfly lane l holds the sum over the warp's 32 rows of column col0 + l
#pragma unroll
          for (int off = 16; off >= 1; off >>= 1) {
            const bool up = (lane & off) != 0;
#pragma unroll
            for (int i = 0; i < off; ++i) {
              const float keep = up ? e[i + off] : e[i];
              const float send = up ? e[i] : e[i + off];
              e[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
            }
          }
          p.colsum_part[((long long)z * (p.m_tiles * 4) + m_tile * 4 + q) * p.L.m_pad + col0 + lane] = e[0];
        }
        p.rowsum_part[((long long)z * (p.n_tiles * 2) + n_tile * 2 + grp) * p.L.n_pad + row] = rs;
      } else if (EPI == EPI_SCORE_CONF) {
        // ---- dual-softmax tail, pass 2: conf = (e / rowsum) * (e / colsum) recomputed from the accumulator (the cos matrix is
        // never materialised), optional conf store, packed row / column arg-max (reference :218-220).  The 32-column chunk is
        // staged once in shared memory: it feeds the TMA store of conf and the per-column scan of the arg-max.
        const int Nz = p.L.n_of(z), M = p.L.M;
        const int row = row0 + r_in_tile;
        const bool row_ok = row < Nz;
        const float ea = kProdInv * p.inv_scale * 1.4426950408889634f, eb = -p.inv_scale * 1.4426950408889634f;
        const int t = t_in_grp, qq = t >> 5, cc = t & 31;          // column-scan role: (32-row quarter, column)
        const float irs = row_ok ? __ldg(p.inv_rowsum + (long long)z * p.L.n_pad + row) : 0.f;
        float* ics = extra + grp * kColsPerGroup;                   // this tile half's inverse column sums
        epi_bar();                                                  // every thread of the group is done with the previous tile's values
        ics[t] = __ldg(p.inv_colsum + (long long)z * p.L.m_pad + n_tile * BN + c_begin + t);
        epi_bar();
        // running row arg-max as (value, column): columns are visited in ascending order and only a STRICTLY larger value
        // replaces the best, so the first maximum wins like torch.max; packed once per tile for the 64-bit atomicMax
        float rbest_v = 0.f;
        int rbest_c = -1;
        const bool store_plain = p.conf != nullptr && !p.conf_tma;
#pragma unroll 1
        for (int c0 = c_begin; c0 < c_end; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(lane_base + c0, v);
          tmem_ld_wait();
          const int col0 = n_tile * BN + c0;
          uint8_t* sb = staging + grp * kStagingBytes;
          float o[32];
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const float4 ic4 = *reinterpret_cast<const float4*>(ics + (c0 - c_begin) + 4 * j4);   // broadcast read
            const float icv[4] = {ic4.x, ic4.y, ic4.z, ic4.w};
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
              const int j = 4 * j4 + jj;
              const bool ok = row_ok && (col0 + j) < M;
              const float e = ok ? ex2_fast(fmaf(__uint_as_float(v[j]), ea, eb)) : 0.f;
              const float c = (e * irs) * (e * icv[jj]);
              o[j] = c;
              if (c > rbest_v) { rbest_v = c; rbest_c = col0 + j; }
            }
          }
          if (p.conf_tma && leader) tma_store_wait_read<0>();       // the store that last read this group's buffer is done with it
          epi_bar();                                                // ... and every thread has finished scanning the previous chunk
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<float4*>(sb + stg_off(r_in_tile, j)) = make_float4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
          if (p.conf_tma) fence_async_smem();
          epi_bar();
          if (p.conf_tma && leader) {
            tma_store_3d(&maps.out_f32, sb, col0, row0, z);         // rows >= N and columns >= M are clipped by the tensor map
            tma_store_commit();
          }
          // column scan over the staged 128 x 32 chunk: thread (qq, cc) = rows [32 qq, +32) of column col0 + cc.  Fully unrolled
          // (invalid rows hold 0 and can never win): 32 independent shared-memory loads in flight instead of a latency chain.
          const int col = col0 + cc;
          if (col < M) {
            const int r_first = row0 + qq * 32;
            float cbest_v = 0.f;
            int cbest_r = -1;
            float cv[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) cv[i] = *reinterpret_cast<const float*>(sb + stg_off(qq * 32 + i, cc >> 2) + (cc & 3) * 4);
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (cv[i] > cbest_v) { cbest_v = cv[i]; cbest_r = r_first + i; }
            if (store_plain) {                                      // 32 consecutive columns of one row per warp instruction; rows
              float* crow = p.conf + ((long long)z * p.L.N + r_first) * M + col;       // [Nz, N) of a ragged frame are written as 0
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (r_first + i < p.L.N) crow[(long long)i * M] = cv[i];
            }
            if (cbest_r >= 0)
              atomicMax(p.colbest + (long long)z * M + col,
                        ((unsigned long long)__float_as_uint(cbest_v) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)cbest_r));
          }
        }
        if (rbest_c >= 0)
          atomicMax(p.rowbest + (long long)z * p.L.N + row,
                    ((unsigned long long)__float_as_uint(rbest_v) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)rbest_c));
      } else if (EPI == EPI_CONV) {
        // ---- convolution layer out: planes = [ReLU](acc + bias) on interior pixels, zero on the grid's border and padding rows
        // (the output is the next layer's zero-bordered input), 32 columns per chunk
        const long long grow = (long long)out_row0 + r_in_tile;
        const int qpix = (int)(grow % p.cv_ppad);
        const int yy = qpix / p.cv_w2, xx = qpix - yy * p.cv_w2;
        const bool row_ok = yy >= 1 && yy <= p.cv_h && xx >= 1 && xx <= p.cv_w;
#pragma unroll 1
        for (int c0 = c_begin; c0 < c_end; c0 += 32, ++chunk_ctr) {
          uint32_t v[32];
          load_acc(c0, v);
          const int col0 = n_tile * BN + c0;
          uint8_t* sh = staging + stage_sel(chunk_ctr) * 8192;
          uint8_t* sl = staging + kStagingBytes + stage_sel(chunk_ctr) * 8192;
          stage_wait();
          epi_bar();
#pragma unroll
          for (int j8 = 0; j8 < 4; ++j8) {
            const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + j8 * 8));
            const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + j8 * 8 + 4));
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
            uint4 oh, ol;
#pragma unroll
            for (int e = 0; e < 4; ++e) {    // same rounding as split_f32, two elements per conversion instruction
              float2 sc = make_float2(fmaf(__uint_as_float(v[j8 * 8 + 2 * e]), kPreInv, bb[2 * e] * kPre),
                                      fmaf(__uint_as_float(v[j8 * 8 + 2 * e + 1]), kPreInv, bb[2 * e + 1] * kPre));
              if (p.relu) sc = make_float2(fmaxf(sc.x, 0.f), fmaxf(sc.y, 0.f));
              if (!row_ok) sc = make_float2(0.f, 0.f);
              const __half2 h2 = __float22half2_rn(sc);
              const float2 back = __half22float2(h2);
              reinterpret_cast<__half2*>(&oh)[e] = h2;
              reinterpret_cast<__half2*>(&ol)[e] = __float22half2_rn(make_float2(sc.x - back.x, sc.y - back.y));
            }
            *reinterpret_cast<uint4*>(sh + stg64_off(r_in_tile, j8)) = oh;
            *reinterpret_cast<uint4*>(sl + stg64_off(r_in_tile, j8)) = ol;
          }
          fence_async_smem();
          epi_bar();
          if (leader) {
            tma_store_2d(&maps.out_hi, sh, col0, out_row0);
            tma_store_2d(&maps.out_lo, sl, col0, out_row0);
            tma_store_commit();
          }
        }
      } else if (EPI == EPI_BIAS_PLANES) {
        // ---- out planes = acc + bias, 32 columns per chunk (a residual, if any, already sits in the accumulator: identity
        // K-block); rows past the segment's valid count are written as zero so that padding never accumulates state
        const bool row_ok = r_in_tile < n_valid;
#pragma unroll 1
        for (int c0 = c_begin; c0 < c_end; c0 += 32, ++chunk_ctr) {
          uint32_t v[32];
          tmem_ld32(lane_base + c0, v);
          tmem_ld_wait();
          const int col0 = n_tile * BN + c0;
          uint8_t* sh = staging + stage_sel(chunk_ctr) * 8192;
          uint8_t* sl = staging + kStagingBytes + stage_sel(chunk_ctr) * 8192;
          stage_wait();
          epi_bar();
#pragma unroll
          for (int j8 = 0; j8 < 4; ++j8) {
            float bb[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (p.bias) {
              const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + j8 * 8));
              const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + j8 * 8 + 4));
              bb[0] = b0.x; bb[1] = b0.y; bb[2] = b0.z; bb[3] = b0.w; bb[4] = b1.x; bb[5] = b1.y; bb[6] = b1.z; bb[7] = b1.w;
            }
            uint4 oh, ol;
#pragma unroll
            for (int e = 0; e < 4; ++e) {    // same rounding as split_f32, two elements per conversion instruction
              float2 sc = make_float2(fmaf(__uint_as_float(v[j8 * 8 + 2 * e]), kPreInv, bb[2 * e] * kPre),
                                      fmaf(__uint_as_float(v[j8 * 8 + 2 * e + 1]), kPreInv, bb[2 * e + 1] * kPre));
              if (!row_ok) sc = make_float2(0.f, 0.f);
              const __half2 h2 = __float22half2_rn(sc);
              const float2 back = __half22float2(h2);
              reinterpret_cast<__half2*>(&oh)[e] = h2;
              reinterpret_cast<__half2*>(&ol)[e] = __float22half2_rn(make_float2(sc.x - back.x, sc.y - back.y));
            }
            *reinterpret_cast<uint4*>(sh + stg64_off(r_in_tile, j8)) = oh;
            *reinterpret_cast<uint4*>(sl + stg64_off(r_in_tile, j8)) = ol;
          }
          fence_async_smem();
          epi_bar();
          if (leader) {
            tma_store_2d(&maps.out_hi, sh, col0, out_row0);
            tma_store_2d(&maps.out_lo, sl, col0, out_row0);
            tma_store_commit();
          }
        }
      } else {
        // ---- planes out (row-major, 64 columns per chunk): EPI_QSCALE / EPI_L2NORM
        float inv_norm = 1.f;
        if (EPI == EPI_L2NORM) {                    // F.normalize: first pass over the accumulator for the row norm
          float ssp[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
          for (int c0 = 0; c0 < BN; c0 += 32) {
            uint32_t v[32];
            tmem_ld32(lane_base + c0, v);
            tmem_ld_wait();
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + c0) + j4);
              const float bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float x = fmaf(__uint_as_float(v[4 * j4 + e]), kProdInv, bv[e]);
                ssp[e] = fmaf(x, x, ssp[e]);
              }
            }
          }
          inv_norm = 1.f / fmaxf(sqrtf((ssp[0] + ssp[1]) + (ssp[2] + ssp[3])), 1e-12f);
        }
        int src = 0;
        float eps_m = 0.f;
        if (EPI == EPI_QSCALE) {
          src = p.L.src_seg(seg, p.cross);
          eps_m = 1e-6f / (float)max(p.L.seg_valid(src), 1);
        }
#pragma unroll 1
        for (int c0 = c_begin; c0 < c_end; c0 += 64) {
          uint32_t v0[32], v1[32];
          tmem_ld32(lane_base + c0, v0);
          tmem_ld32(lane_base + c0 + 32, v1);
          tmem_ld_wait();
          const int col0 = n_tile * BN + c0;
          float x[64];
          // warp-uniform parameter reads as 16-byte loads: 16 instead of 64 load instructions per chunk and thread
          const float4* bias4 = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
          for (int j4 = 0; j4 < 16; ++j4) {
            const float4 bb = __ldg(bias4 + j4);
            const float bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int j = 4 * j4 + e;
              x[j] = fmaf(__uint_as_float(j < 32 ? v0[j & 31] : v1[j & 31]), kProdInv, bv[e]);
            }
          }
          if (EPI == EPI_QSCALE) {
            // one 64-column chunk = one head (head-contiguous channels); the row's head dot product is thread-local
            const float4* km4 = reinterpret_cast<const float4*>(p.kmean + (long long)src * kD + col0);
            float dotp[4] = {0.f, 0.f, 0.f, 0.f};          // four independent chains instead of one 64-long dependent FFMA chain
#pragma unroll
            for (int j4 = 0; j4 < 16; ++j4) {
              const float4 kk = __ldg(km4 + j4);
              const float kv4[4] = {kk.x, kk.y, kk.z, kk.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int j = 4 * j4 + e;
                x[j] = elu1_fast(x[j]);
                dotp[e] = fmaf(x[j], kv4[e], dotp[e]);
              }
            }
            const float dot = (dotp[0] + dotp[1]) + (dotp[2] + dotp[3]);
            const float zf = 1.f / (dot + eps_m);
#pragma unroll
            for (int j = 0; j < 64; ++j) x[j] *= zf;
          } else {  // EPI_L2NORM
#pragma unroll
            for (int j = 0; j < 64; ++j) x[j] *= inv_norm;
          }
          // two 32-column sub-chunks; each has its own (hi, lo) pair of 8 KB SWIZZLE_64B staging buffers, so the TMA
          // store of one sub-chunk drains while the next is being written (same 32 KB of staging as the fp32 path)
#pragma unroll
          for (int sc = 0; sc < 2; ++sc, ++chunk_ctr) {
            uint8_t* sh = staging + stage_sel(chunk_ctr) * 8192;
            uint8_t* sl = staging + kStagingBytes + stage_sel(chunk_ctr) * 8192;
            stage_wait();
            epi_bar();
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) {
              uint4 oh, ol;
#pragma unroll
              for (int e = 0; e < 4; ++e) {    // same rounding as split_f32, two elements per conversion instruction
                const float2 sc2 = make_float2(x[sc * 32 + j8 * 8 + 2 * e] * kPre, x[sc * 32 + j8 * 8 + 2 * e + 1] * kPre);
                const __half2 h2 = __float22half2_rn(sc2);
                const float2 back = __half22float2(h2);
                reinterpret_cast<__half2*>(&oh)[e] = h2;
                reinterpret_cast<__half2*>(&ol)[e] = __float22half2_rn(make_float2(sc2.x - back.x, sc2.y - back.y));
              }
              *reinterpret_cast<uint4*>(sh + stg64_off(r_in_tile, j8)) = oh;
              *reinterpret_cast<uint4*>(sl + stg64_off(r_in_tile, j8)) = ol;
            }
            fence_async_smem();
            epi_bar();
            if (leader) {
              tma_store_2d(&maps.out_hi, sh, col0 + sc * 32, out_row0);
              tma_store_2d(&maps.out_lo, sl, col0 + sc * 32, out_row0);
              tma_store_commit();
            }
          }
        }
      }
      // all TMEM reads of this tile are complete (wait::ld above): hand the accumulator back
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (crank != 0) mbar_arrive_remote(&tmem_empty_bar[buf], 0);   // the leader's MMA warp waits for both CTAs
        else mbar_arrive(&tmem_empty_bar[buf]);
      }
      if (tl && threadIdx.x == 128 && tc < 8) tl[41 + 2 * tc] = clock64();
    }
    if (leader) tma_store_wait_all();
  }
  __syncthreads();
  cluster_sync_all();                  // no CTA leaves while its peer may still land loads in it / arrive on its barriers
  if (tl && threadIdx.x == 0) { tl[2] = clock64(); unsigned sm; asm("mov.u32 %0, %%smid;" : "=r"(sm)); tl[63] = sm; }
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols) : "memory");
  }
}

// ------------------------------------------------------------------ host: tensor maps
using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                              const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn get_encode() {
  static EncodeFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn>(f);
  });
  return fn;
}

// 2D row-major tensor [rows, ld] (cols used: `cols`), box = box_cols x box_rows.  Swizzle follows the box row
// width (128 B -> SWIZZLE_128B, 64 B -> SWIZZLE_64B, anything else -> none).  Cached per (ptr, shape, box, dtype).
bool make_map(CUtensorMap* out, const void* ptr, long long rows, long long cols, long long ld, int box_cols, int box_rows, bool f32) {
  const size_t esize = f32 ? 4 : 2;
  const size_t row_bytes = box_cols * esize;
  const CUtensorMapSwizzle swz = row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE);
  static std::map<std::tuple<const void*, long long, long long, long long, int, int, bool>, CUtensorMap> cache;
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  auto key = std::make_tuple(ptr, rows, cols, ld, box_cols, box_rows, f32);
  auto it = cache.find(key);
  if (it != cache.end()) { *out = it->second; return true; }
  EncodeFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * esize};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return false;
  if (cache.size() > 4096) cache.clear();
  cache[key] = *out;
  return true;
}

// conf [B][N][M] fp32 as a 3-D tensor (box 32 x 128 x 1, SWIZZLE_128B): a 128-row tile that hangs over the end of a
// frame (rows >= N) or of a row (columns >= M) is clipped by the hardware.  Needs M % 4 == 0 (16-byte global strides)
// and a 16-byte aligned base.
bool make_map3(CUtensorMap* out, const float* ptr, int M, int N, int B) {
  EncodeFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t dims[3] = {(cuuint64_t)M, (cuuint64_t)N, (cuuint64_t)B};
  cuuint64_t strides[2] = {(cuuint64_t)M * 4, (cuuint64_t)M * N * 4};
  cuuint32_t box[3] = {32, (cuuint32_t)BM, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int g_conv_halo = 1;      // 0: nine row-shifted boxes per tile; 1: halo boxes (default)
int conv_halo_mode() { return g_conv_halo; }

// SM count of the current device, cached per device.
int num_sms() {
  static std::mutex mu;
  static std::map<int, int> n;
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lock(mu);
  int& sms = n[dev];
  if (!sms) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms;
}

template <int EPI, int ACV = ACV_NONE, bool HI = false, int BN_ = 256>
cudaError_t launch_variant(const cudaLaunchConfig_t& cfg, const Maps& mp, const TcParams& tp) {
  auto* kern = gemm_tc_kernel<EPI, ACV, HI, BN_>;
  if (cudaError_t e = ensure_smem_attr((const void*)kern, kSmemBytes)) return e;
  return cudaLaunchKernelEx(&cfg, kern, mp, tp);
}

}  // namespace

void set_conv_halo_mode(int mode) { g_conv_halo = mode ? 1 : 0; }

bool make_tensor_map_2d(CUtensorMap* out, const void* ptr, long long rows, long long cols, long long ld, int box_cols, int box_rows, bool f32) {
  return make_map(out, ptr, rows, cols, ld, box_cols, box_rows, f32);
}

int launch_gemm_tc(const GemmProblem& p, cudaStream_t stream, long long* timeline) {
  const int bn = p.bn ? p.bn : BN;                 // column-tile width
  if (bn != BN && !((bn == 64 || bn == 128) && (p.epi == EPI_CONV || p.epi == EPI_F32) && !p.K2 && !p.a_conv && !p.a_hi_only)) return -1;
  if (p.rows % (2 * BM) || p.n_out % bn || p.K1 % BK || p.K2 % BK || p.K1 <= 0 || p.batch <= 0) return -1;
  if ((p.epi == EPI_QSCALE || p.epi == EPI_L2NORM || p.epi == EPI_BIAS_PLANES) && p.n_out != BN) return -1;
  if (p.taps && (p.epi != EPI_CONV || p.taps > 9 || p.kb_per_tap <= 0 || p.taps * p.kb_per_tap * BK != p.K1 || p.K2 || p.batch != 1)) return -1;
  if (p.epi == EPI_CONV && (!p.bias || !p.out.hi || !p.out.lo || p.cv_ppad <= 0 || p.cv_w2 <= 0 || p.batch != 1)) return -1;
  if (p.a_hi_only && (p.a_conv || p.K2 || p.epi != EPI_QKV)) return -1;
  if (p.a_conv && (p.a_conv != ACV_NORM_RELU || p.batch != 1 || !p.a_raw || p.epi != EPI_BIAS_PLANES || p.b2_per_seg || !p.mu || !p.rstd)) return -1;
  const bool f32_out = p.epi == EPI_F32 || p.epi == EPI_F32_STATS;
  // halo convolution: 3x3 taps in row-major order with unit horizontal steps, narrow column tiles (the 256-wide tile has no room
  // for two halo stages and is not L2-bound)
  int halo = (p.epi == EPI_CONV && p.taps == 9 && bn != BN) ? conv_halo_mode() : 0;
  for (int t = 0; t < 9 && halo; ++t)
    if (p.tap_off[t] != (t / 3 - 1) * p.cv_w2 + (t % 3 - 1)) halo = 0;
  if (p.epi == EPI_QKV && (p.n_out != 2 * BN || p.batch != 1 || !p.out.hi || !p.bias)) return -1;
  if ((p.epi == EPI_QSCALE || p.epi == EPI_L2NORM) && !p.bias) return -1;
  const bool score = p.epi == EPI_SCORE_SUMS || p.epi == EPI_SCORE_CONF;
  int conf_tma = 0;
  if (f32_out && (p.ldc % 4 || !p.c)) return -1;
  const long long a_rows = (long long)(p.batch - 1) * p.a_batch_rows + p.rows;
  const long long b1_rows = (long long)(p.batch - 1) * p.b_batch_rows + p.n_out;
  const long long b2_rows = p.b2_per_seg ? (long long)p.L.segs() * p.n_out : p.n_out;
  Maps mp;
  bool ok = make_map(&mp.b1h, p.b1.hi, b1_rows, p.K1, p.b1.ld, BK, bn / 2, false) && make_map(&mp.b1l, p.b1.lo, b1_rows, p.K1, p.b1.ld, BK, bn / 2, false);
  if (p.a_conv) { mp.a1h = mp.b1h; mp.a1l = mp.b1l; }     // every A1 tile comes in raw: the plane maps are never used
  else {
    const long long a_cols = p.taps ? (long long)p.kb_per_tap * BK : p.K1;      // convolution: A has C_in columns, the taps shift its rows
    const int a_box_rows = halo ? BM + 2 : BM;                                   // halo convolution: one box serves the three horizontal taps
    ok = ok && make_map(&mp.a1h, p.a1.hi, a_rows, a_cols, p.a1.ld, BK, a_box_rows, false) && make_map(&mp.a1l, p.a1.lo, a_rows, a_cols, p.a1.ld, BK, a_box_rows, false);
  }
  if (ok && p.a_conv) ok = make_map(&mp.a_raw, p.a_raw, a_rows, p.K1, p.a_raw_ld, 32, BM, true);
  else mp.a_raw = mp.b1h;
  if (ok && p.K2) {
    ok = make_map(&mp.b2h, p.b2.hi, b2_rows, p.K2, p.b2.ld, BK, p.b2_identity ? 32 : BN / 2, false) && make_map(&mp.b2l, p.b2.lo, b2_rows, p.K2, p.b2.ld, BK, BN / 2, false) &&
         make_map(&mp.a2h, p.a2.hi, a_rows, p.K2, p.a2.ld, BK, BM, false) && make_map(&mp.a2l, p.a2.lo, a_rows, p.K2, p.a2.ld, BK, BM, false);
  } else if (ok) {
    mp.a2h = mp.a1h; mp.a2l = mp.a1l; mp.b2h = mp.b1h; mp.b2l = mp.b1l;
  }
  const long long out_rows = (long long)p.batch * p.rows;
  if (f32_out) {
    ok = ok && make_map(&mp.out_f32, p.c, out_rows, p.n_out, p.ldc, 32, BM, true);
    mp.out_hi = mp.out_f32; mp.out_lo = mp.out_f32;
  } else if (p.epi == EPI_QKV) {
    ok = ok && make_map(&mp.out_hi, p.out.hi, out_rows, 2 * BN, p.out.ld, 64, BM, false);
    mp.out_f32 = mp.out_hi;
    mp.out_lo = mp.out_hi;
  } else if (score) {
    mp.out_f32 = mp.b1h; mp.out_hi = mp.b1h; mp.out_lo = mp.b1h;
    if (p.epi == EPI_SCORE_CONF && p.conf && p.L.M % 4 == 0 && (reinterpret_cast<uintptr_t>(p.conf) & 15) == 0)
      conf_tma = make_map3(&mp.out_f32, p.conf, p.L.M, p.L.N, p.batch) ? 1 : 0;
  } else {
    ok = ok && make_map(&mp.out_hi, p.out.hi, out_rows, p.n_out, p.out.ld, 32, BM, false) && make_map(&mp.out_lo, p.out.lo, out_rows, p.n_out, p.out.ld, 32, BM, false);
    mp.out_f32 = mp.out_hi;
  }
  if (!ok) return -2;
  TcParams tp{};
  tp.K1 = p.K1; tp.K2 = p.K2; tp.b2_per_seg = p.b2_per_seg; tp.b2_lo_zero = p.b2_lo_zero; tp.n_out = p.n_out;
  tp.b2_identity = p.b2_identity;
  if (p.b2_identity && (!p.b2_lo_zero || p.b2_per_seg || p.K2 != p.n_out || p.n_out != BN || p.K1 <= 0 || bn != BN)) return -1;
  tp.m_tiles = p.rows / BM; tp.n_tiles = p.n_out / bn; tp.batch = p.batch;
  tp.taps = p.taps; tp.kb_per_tap = p.kb_per_tap;
  for (int t = 0; t < 9; ++t) tp.tap_off[t] = p.tap_off[t];
  tp.cv_w2 = p.cv_w2; tp.cv_h = p.cv_h; tp.cv_w = p.cv_w; tp.cv_ppad = p.cv_ppad; tp.relu = p.relu; tp.halo = halo;
  tp.a_batch_rows = p.a_batch_rows; tp.b_batch_rows = p.b_batch_rows; tp.c_batch_rows = p.rows;
  tp.seg_rows = (p.batch == 1 && p.L.R > 0 && p.L.rows() == p.rows) ? 1 : 0;
  tp.L = p.L; tp.bias = p.bias; tp.tl = timeline;
  tp.inv_scale = p.inv_scale; tp.rowsum_part = p.rowsum_part; tp.colsum_part = p.colsum_part; tp.inv_rowsum = p.inv_rowsum;
  tp.inv_colsum = p.inv_colsum; tp.conf = p.conf; tp.conf_tma = conf_tma; tp.rowbest = p.rowbest; tp.colbest = p.colbest;
  tp.mu = p.mu; tp.rstd = p.rstd;
  tp.kmean = p.kmean; tp.cross = p.cross; tp.statpart = p.statpart;
  if ((p.epi == EPI_QSCALE || p.b2_per_seg || p.epi == EPI_QKV || p.epi == EPI_F32_STATS || p.a_conv) && !tp.seg_rows) return -1;
  const int total_units = (tp.m_tiles / 2) * tp.n_tiles * tp.batch;
  const int sms = num_sms();
  const int grid = total_units * 2 < sms ? total_units * 2 : (sms / 2) * 2;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(threads_of(p.a_conv));
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 2 : 1;
  cudaError_t le;
  if (p.a_conv) {
    le = launch_variant<EPI_BIAS_PLANES, ACV_NORM_RELU>(cfg, mp, tp);
  } else {
    switch (p.epi) {
      case EPI_F32:
        le = bn == 64 ? launch_variant<EPI_F32, ACV_NONE, false, 64>(cfg, mp, tp)
                      : bn == 128 ? launch_variant<EPI_F32, ACV_NONE, false, 128>(cfg, mp, tp) : launch_variant<EPI_F32>(cfg, mp, tp);
        break;
      case EPI_CONV:
        le = bn == 64 ? launch_variant<EPI_CONV, ACV_NONE, false, 64>(cfg, mp, tp)
                      : bn == 128 ? launch_variant<EPI_CONV, ACV_NONE, false, 128>(cfg, mp, tp) : launch_variant<EPI_CONV>(cfg, mp, tp);
        break;
      case EPI_F32_STATS: le = launch_variant<EPI_F32_STATS>(cfg, mp, tp); break;
      case EPI_QSCALE: le = launch_variant<EPI_QSCALE>(cfg, mp, tp); break;
      case EPI_L2NORM: le = launch_variant<EPI_L2NORM>(cfg, mp, tp); break;
      case EPI_SCORE_SUMS: le = launch_variant<EPI_SCORE_SUMS>(cfg, mp, tp); break;
      case EPI_SCORE_CONF: le = launch_variant<EPI_SCORE_CONF>(cfg, mp, tp); break;
      case EPI_QKV: le = p.a_hi_only ? launch_variant<EPI_QKV, ACV_NONE, true>(cfg, mp, tp) : launch_variant<EPI_QKV>(cfg, mp, tp); break;
      case EPI_BIAS_PLANES: le = launch_variant<EPI_BIAS_PLANES>(cfg, mp, tp); break;
      default: return -1;
    }
  }
  if (le != cudaSuccess) return -2;
  return 0;
}

}  // namespace opb
