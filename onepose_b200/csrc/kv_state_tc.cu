// Linear-attention state on the 5th-gen tensor cores.
//
//   per segment s, head h:   KV[h][d][q] = sum_rows elu1(K[r,h,d]) * V[r,h,q],   Ksum[h][d] = sum_rows elu1(K[r,h,d])
//   (reference GATs_SuperGlue.py:71-78; the 1/m of :75 is applied by kv_state_reduce)
//
// The k,v projection epilogue (EPI_QKV) leaves  kvh[rows, 512] = fp16(64 * [elu1(K) | V])  with pad rows zero, so the state
// is ONE tensor-core pass over operands that TMA lands directly in the UMMA MN-major SWIZZLE_128B layout (reduction index =
// row).  Rounding K and V to fp16 perturbs each product by <= 2^-11 relative with zero mean; the state is a MEAN over the
// segment's rows, so the perturbation of the mean is ~2^-12/sqrt(rows) -- measured end to end in tools/kv_precision.py
// (cosine error unchanged at 7e-7 down to 16-row segments).
#include <cuda.h>

#include "common.cuh"
#include "gemm_tc.cuh"
#include "host_util.cuh"
#include "kv_state_tc.cuh"

namespace opb {
namespace {

constexpr uint32_t kSpin = 1u << 22;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0, ok = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (ok) break;
    if (++spins > kSpin) __trap();
  }
}
// kind::f16, D = f32, A = B = f16, A and B MN-major, M = 128, N = 128
constexpr uint32_t kIdesc = (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);

__device__ __forceinline__ void mma(uint32_t tmem_d, uint64_t a, uint64_t b, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(a), "l"(b), "r"(kIdesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
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

// One CTA per ROW GROUP = `slabs_per_group` consecutive 256-row slabs of one segment (groups never straddle a segment; the
// host picks the group size so that the grid is about two CTAs per SM -- fewer, larger groups mean fewer partial states to
// write and re-read).  192 threads, 2 CTAs per SM:
//   warp 0     TMA producer: 32-row stages = 8 boxes of 64 channels x 32 rows (4 K blocks, 4 V blocks), 3-stage ring
//   warp 1     TMEM owner + MMA issuer: per stage 2 head pairs x 2 k-steps of 16 rows, M = N = 128, accumulating over the group
//   warps 2-5  K column sums from the staged tile (the K mean of the attention normaliser), then the epilogue
constexpr int kHRows = 32;                                 // rows per stage
constexpr int kHStages = 3;
constexpr int kHBlockBytes = kHRows * 128;                 // one 64-channel x 32-row box = 4 KB (LBO between channel blocks)
constexpr int kHStageBytes = 8 * kHBlockBytes;             // 32 KB
constexpr int kHSmemBytes = kHStages * kHStageBytes + 1024 + 128;

__device__ __forceinline__ uint64_t make_desc_mn_h(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(kHBlockBytes >> 4) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* map, uint64_t* bar, int c_inner, int c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_dst),
      "l"(map), "r"(smem_u32(bar)), "r"(c_inner), "r"(c_outer)
      : "memory");
}

__global__ void __launch_bounds__(192, 2) kv_state_h_kernel(const __grid_constant__ CUtensorMap kv_map, Layout L, KvGroups G, float* __restrict__ partial) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kHStages * kHStageBytes);   // [3] stage landed
  uint64_t* empty_bar = full_bar + kHStages;                                          // [3] stage consumed (MMAs retired + sums read)
  uint64_t* done_bar = empty_bar + kHStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // row group -> (frame, side, group index inside the segment)
  const int per_frame = G.gq + G.gd;
  const int b = blockIdx.x / per_frame, g = blockIdx.x - b * per_frame;
  const int side = g >= G.gq ? 1 : 0, gi = side ? g - G.gq : g;
  const int seg = 2 * b + side;
  const int group_rows = G.slabs * 256;
  const int row0 = L.seg_start(seg) + gi * group_rows;
  float* out = partial + (long long)blockIdx.x * kHeads * (kDh * kDh + kDh);
  griddep_sync();                                          // kvh of the preceding GEMM is visible from here on
  const int n_valid = min(group_rows, L.seg_valid(seg) - gi * group_rows);
  if (n_valid <= 0) {                                      // group entirely in the padding: never read by the reduction, defined anyway
    for (int i = tid; i < kHeads * (kDh * kDh + kDh); i += 192) out[i] = 0.f;
    return;
  }
  const int n_stages = (n_valid + kHRows - 1) / kHRows;    // rows past n_valid inside the last stage are zero (EPI_QKV zeroes pad rows)
  if (tid == 0) {
    for (int s = 0; s < kHStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 5); }
    mbar_init(done_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&kv_map) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(256) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int s = 0; s < n_stages; ++s) {
        const int buf = s % kHStages;
        if (s >= kHStages) mbar_wait(&empty_bar[buf], ((s / kHStages) - 1) & 1);
        mbar_expect_tx(&full_bar[buf], kHStageBytes);
        const uint32_t st = smem_u32(smem) + buf * kHStageBytes;
#pragma unroll
        for (int blk = 0; blk < 8; ++blk) tma_load_2d(st + blk * kHBlockBytes, &kv_map, &full_bar[buf], blk * 64, row0 + s * kHRows);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < n_stages; ++s) {
        const int buf = s % kHStages;
        mbar_wait(&full_bar[buf], (s / kHStages) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t kb = smem_u32(smem) + buf * kHStageBytes, vb = kb + 4 * kHBlockBytes;
#pragma unroll
        for (int pair = 0; pair < 2; ++pair) {
          const uint32_t d = tmem_base + pair * 128;
          const uint32_t po = pair * 2 * kHBlockBytes;
#pragma unroll
          for (int k = 0; k < kHRows / 16; ++k)
            mma(d, make_desc_mn_h(kb + po + k * 2048), make_desc_mn_h(vb + po + k * 2048), (uint32_t)((s | k) != 0));
        }
        commit(&empty_bar[buf]);
        if (s == n_stages - 1) commit(done_bar);
      }
    }
  } else {
    // ---- K column sums: thread = (8-channel chunk j of the 256 K channels, row group g of 4)
    const int t = tid - 64;
    const int j = t & 31, g = t >> 5;
    float ks[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int s = 0; s < n_stages; ++s) {
      const int buf = s % kHStages;
      mbar_wait(&full_bar[buf], (s / kHStages) & 1);
      const uint32_t base = smem_u32(smem) + buf * kHStageBytes + (j >> 3) * kHBlockBytes;
#pragma unroll
      for (int i = 0; i < kHRows / 4; ++i) {
        const int r = g + 4 * i;
        uint4 v;
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(base + r * 128 + (((j & 7) ^ (r & 7)) << 4)));
        const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = __half22float2(h[e]);
          ks[2 * e] += f.x;
          ks[2 * e + 1] += f.y;
        }
      }
      // The arrive releases the stage to the TMA producer and must not overtake the loads above: ptxas sinks the FADDs that
      // consume them below the arrive, so nothing in issue order guarantees they have returned.  Without the fence the K sums
      // picked up rows of the NEXT use of the stage (seen as run-to-run differences of the K mean).
      __threadfence_block();
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[buf]);
    }
    // ---- epilogue: diagonal head blocks of the two accumulators (this warp's TMEM lane quarter = warp % 4)
    mbar_wait(done_bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int quarter = warp & 3;
    const int lane_row = quarter * 32 + lane;      // accumulator row = K channel within the head pair
    const int hl = lane_row >> 6, d = lane_row & 63;
#pragma unroll 1
    for (int pair = 0; pair < 2; ++pair) {
      const int h = pair * 2 + hl;
      float* o = out + (long long)h * (kDh * kDh + kDh) + d * kDh;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t v[32];
        tmem_ld32(tmem_base + pair * 128 + hl * 64 + half * 32 + ((uint32_t)(quarter * 32) << 16), v);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int q = 0; q < 32; q += 4)
          *reinterpret_cast<float4*>(o + half * 32 + q) = make_float4(__uint_as_float(v[q]) * kProdInv, __uint_as_float(v[q + 1]) * kProdInv,
                                                                      __uint_as_float(v[q + 2]) * kProdInv, __uint_as_float(v[q + 3]) * kProdInv);
      }
    }
    // K sums: combine the 4 row groups through the (now idle) stage memory
    float* red = reinterpret_cast<float*>(smem);
    asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
    for (int e = 0; e < 8; ++e) red[g * 256 + j * 8 + e] = ks[e];
    asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
    for (int c = t; c < 256; c += 128)
      out[(long long)(c >> 6) * (kDh * kDh + kDh) + kDh * kDh + (c & 63)] = (red[c] + red[256 + c] + red[512 + c] + red[768 + c]) * kPreInv;
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(256) : "memory");
  }
}

}  // namespace

}  // namespace opb

namespace opb {
KvGroups kv_groups_for(const Layout& L, int num_sms) {
  const int total_slabs = L.rows() / 256;
  int slabs = total_slabs / (2 * num_sms);                 // about two CTAs per SM (the kernel's occupancy)
  slabs = slabs < 1 ? 1 : (slabs > 8 ? 8 : slabs);
  KvGroups G;
  G.slabs = slabs;
  G.gq = (L.n_pad / 256 + slabs - 1) / slabs;
  G.gd = (L.m_pad / 256 + slabs - 1) / slabs;
  return G;
}

int launch_kv_state_h(const __half* kvh, const Layout& L, const KvGroups& G, float* partial, cudaStream_t stream) {
  if (ensure_smem_attr((const void*)kv_state_h_kernel, kHSmemBytes) != cudaSuccess) return -2;
  CUtensorMap map;
  if (!make_tensor_map_2d(&map, kvh, L.rows(), 512, 512, 64, kHRows, false)) return -2;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(L.B * (G.gq + G.gd)));
  cfg.blockDim = dim3(192);
  cfg.dynamicSmemBytes = kHSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kv_state_h_kernel, map, L, G, partial) == cudaSuccess ? 0 : -2;
}
}  // namespace opb
