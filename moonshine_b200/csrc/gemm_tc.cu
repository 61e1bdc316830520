// Grouped "NT" GEMM on the 5th-gen tensor cores (tcgen05 + TMEM), fp32 in / fp32
// out, with the bf16x3 split that keeps the result within ~1e-5 of fp32:
//     a = a_hi + a_lo (both bf16),  a*w ~= a_hi*w_hi + a_hi*w_lo + a_lo*w_hi
// (DESIGN.md section 2: single bf16 / tf32 passes miss the 1e-3 logit bar).
//
// Same GemmParams interface and epilogue as gemm_simt.cu, so every strided /
// grouped / ragged view of the encoder (conv windows, per-head attention
// operands, swapped-orientation K^T / V^T projections) runs unchanged.
//
// CTA = 128x128 output tile, 288 threads, 2 CTAs per SM:
//   warps 0-3  load A rows, warps 4-7 load W rows: coalesced LDG.128 of fp32,
//              split to bf16 hi / lo in registers, STS into the K-major
//              SWIZZLE_64B layout tcgen05 expects, fence.proxy.async, arrive;
//   warp 8     one lane issues 6 tcgen05.mma (M128 N128 K16, kind::f16) per
//              32-wide K block (3 split products x 2 k-steps), accumulators in
//              TMEM; tcgen05.commit releases smem stages / signals the epilogue;
//   warps 0-3  epilogue: tcgen05.ld 32x32b from TMEM, shared epilogue, stores.
// The fp32 source cannot go through TMA (the split has to happen in registers);
// the second resident CTA hides one CTA's epilogue behind the other's mainloop.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.h"
#include "gemm_epilogue.cuh"
#include "kernels.h"

namespace msb {

namespace {

constexpr int TM = 128, TN = 128, TK = 32;
constexpr int kStages = 1;                     // bf16 operand stages (UMMA-ready)
constexpr int kRawStages = 2;                  // fp32 staging ring filled by cp.async
constexpr int kLoaders = 256;
constexpr int kThreadsTC = kLoaders + 32;
constexpr int kTileBytes = TM * TK * 2;        // one bf16 plane of one operand: 8 KB
constexpr int kStageBytesTC = 4 * kTileBytes;  // A_hi, A_lo, W_hi, W_lo
constexpr int kRawBytes = 2 * TM * TK * 4;     // A and W fp32 tiles of one K block: 32 KB
constexpr int kTmemCols = 128;
constexpr long long kSpinLimitTC = 4000000000LL;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ unsigned int g_gemm_tc_error = 0;  // watchdog flag (see gemm_tc_error_async)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t a = smem_u32(bar);
  uint32_t done = 0;
  const long long t0 = clock64();
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(a), "r"(parity)
        : "memory");
    if (done) break;
    if (clock64() - t0 > kSpinLimitTC) {  // poison instead of trapping the context: the host raises after its next synchronise
      atomicExch(&g_gemm_tc_error, 1u);
      break;
    }
  }
}

// K-major SWIZZLE_64B shared-memory matrix descriptor (sm_100 UMMA):
// start address >> 4, LBO = 1 (unused for swizzled K-major), SBO = 8 rows * 64 B,
// version 1, layout type 4 (SWIZZLE_64B).
__device__ __forceinline__ uint64_t make_desc_sw64(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;
  return d;
}
// kind::f16 instruction descriptor: D = F32, A = B = BF16, both K-major, N = 128, M = 128.
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(kIdesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// One lane of a converged warp (tcgen05.mma wants uniform-register operands: issued under elect.sync inside
// warp-uniform control flow it is a few instructions; from a divergent `if (tid == X)` the compiler wraps every
// MMA in an ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall loop, ~95 ns per MMA measured on B200).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ uint32_t uniform_u32(uint32_t v) { return __shfl_sync(0xffffffffu, v, 0); }

// Splits 4 floats into bf16 hi / lo quads (8 bytes each).
__device__ __forceinline__ void split4(const float4 v, uint2& hi, uint2& lo) {
  const __nv_bfloat162 h01 = __floats2bfloat162_rn(v.x, v.y);
  const __nv_bfloat162 h23 = __floats2bfloat162_rn(v.z, v.w);
  const float2 f01 = __bfloat1622float2(h01);
  const float2 f23 = __bfloat1622float2(h23);
  const __nv_bfloat162 l01 = __floats2bfloat162_rn(v.x - f01.x, v.y - f01.y);
  const __nv_bfloat162 l23 = __floats2bfloat162_rn(v.z - f23.x, v.w - f23.y);
  hi.x = *reinterpret_cast<const uint32_t*>(&h01);
  hi.y = *reinterpret_cast<const uint32_t*>(&h23);
  lo.x = *reinterpret_cast<const uint32_t*>(&l01);
  lo.y = *reinterpret_cast<const uint32_t*>(&l23);
}

__global__ void __launch_bounds__(kThreadsTC, 2) gemm_tc_kernel(const __grid_constant__ GemmParams p) {
  const int z = blockIdx.z;
  const int Mz = p.Mz ? p.Mz[z] : p.M;
  const int Nz = p.Nz ? p.Nz[z] : p.N;
  const int Kz = p.Kz ? p.Kz[z] : p.K;
  const int m0 = blockIdx.y * TM;
  const int n0 = blockIdx.x * TN;
  if (m0 >= Mz || n0 >= Nz) return;  // uniform per CTA

  extern __shared__ __align__(16) unsigned char smem_raw[];
  // SWIZZLE_64B atoms repeat every 512 B: align the stage ring to 1 KB by hand
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ __align__(8) uint64_t full_bar[kStages];
  __shared__ __align__(8) uint64_t empty_bar[kStages];
  __shared__ __align__(8) uint64_t accum_bar;
  __shared__ uint32_t tmem_base_smem;

  const int tid = threadIdx.x;
  const int warp = (int)uniform_u32((uint32_t)(threadIdx.x >> 5));  // provably warp-uniform

  if (tid == 0) {
    for (int s = 0; s < kStages; s++) {
      mbar_init(&full_bar[s], kLoaders);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&accum_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)),
                 "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_smem;

  const int nk = (Kz + TK - 1) / TK;

  if (warp < 8) {
    // ============================ loaders ============================
    const bool is_w = tid >= 128;
    const int lt = tid & 127;
    const int q = lt & 7;        // float4 index inside the 32-float K block
    const int rsub = lt >> 3;    // 0..15
    const float* __restrict__ src = is_w ? p.W + (p.offW ? p.offW[z] : (int64_t)z * p.strideW)
                                         : p.A + (p.offA ? p.offA[z] : (int64_t)z * p.strideA);
    const int ld = is_w ? p.ldw : p.lda;
    const int row0 = is_w ? n0 : m0;
    const int rows_valid = is_w ? Nz : Mz;
    // Each thread owns 8 fixed 16-byte chunks (row i*16+rsub, float4 q) of its operand tile:
    // it cp.asyncs them into the raw fp32 ring, later reads the same chunks back, splits them
    // to bf16 hi/lo and stores them K-major SWIZZLE_64B (row pitch 64 B, 16-byte chunk
    // c = q >> 1 stored at c ^ ((r >> 1) & 3)).  No cross-thread hazards on the raw ring.
    unsigned char* raw_base = smem + (size_t)kStages * kStageBytesTC + (is_w ? TM * TK * 4 : 0);
    auto issue = [&](int kb) {
      const int k = kb * TK + q * 4;
      unsigned char* dst = raw_base + (size_t)(kb % kRawStages) * kRawBytes;
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int rl = i * 16 + rsub;
        const int r = row0 + rl;
        if (r < rows_valid && k < Kz) {
          const uint32_t d = smem_u32(dst + rl * 128 + q * 16);
          const float* g = src + (int64_t)r * ld + k;
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(g) : "memory");
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    issue(0);
    if (nk > 1) issue(1); else asm volatile("cp.async.commit_group;" ::: "memory");
    for (int kb = 0; kb < nk; kb++) {
      const int s = kb % kStages;
      const uint32_t ph = (uint32_t)((kb / kStages) & 1);
      const int k = kb * TK + q * 4;
      asm volatile("cp.async.wait_group 1;" ::: "memory");   // this thread's chunks of block kb landed
      const unsigned char* rsrc = raw_base + (size_t)(kb % kRawStages) * kRawBytes;
      float4 v[8];
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int rl = i * 16 + rsub;
        const int r = row0 + rl;
        if (r < rows_valid && k < Kz) {
          v[i] = *reinterpret_cast<const float4*>(rsrc + rl * 128 + q * 16);
          if (k + 3 >= Kz) {  // K tail inside the float4: row padding must not contribute
            if (k + 1 >= Kz) v[i].y = 0.f;
            if (k + 2 >= Kz) v[i].z = 0.f;
            if (k + 3 >= Kz) v[i].w = 0.f;
          }
        } else {
          v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      uint2 hi[8], lo[8];
#pragma unroll
      for (int i = 0; i < 8; i++) split4(v[i], hi[i], lo[i]);
      // the reads above have been consumed: refill the raw slot just drained
      if (kb + kRawStages < nk) issue(kb + kRawStages);
      else asm volatile("cp.async.commit_group;" ::: "memory");
      mbar_wait(&empty_bar[s], ph ^ 1u);  // MMAs that read this bf16 stage have completed
      unsigned char* stage = smem + (size_t)s * kStageBytesTC + (is_w ? 2 * kTileBytes : 0);
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int r = i * 16 + rsub;
        const uint32_t off = (uint32_t)r * 64u + ((((uint32_t)q >> 1) ^ (((uint32_t)r >> 1) & 3u)) << 4) + ((uint32_t)q & 1u) * 8u;
        *reinterpret_cast<uint2*>(stage + off) = hi[i];
        *reinterpret_cast<uint2*>(stage + kTileBytes + off) = lo[i];
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> async proxy (UMMA)
      mbar_arrive(&full_bar[s]);
    }
  } else {
    // ============================ MMA issuer (warp 8, one elected lane) ============================
    const uint32_t tm = uniform_u32(tmem_base);
    for (int kb = 0; kb < nk; kb++) {
      const int s = kb % kStages;
      const uint32_t ph = (uint32_t)((kb / kStages) & 1);
      mbar_wait(&full_bar[s], ph);
      __syncwarp();
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t a_hi = uniform_u32(smem_u32(smem + (size_t)s * kStageBytesTC));
      const uint32_t a_lo = a_hi + kTileBytes;
      const uint32_t w_hi = a_hi + 2 * kTileBytes;
      const uint32_t w_lo = a_hi + 3 * kTileBytes;
      if (elect_one()) {
#pragma unroll
        for (int j = 0; j < TK / 16; j++) {
          const uint32_t ko = (uint32_t)j * 32u;  // 16 bf16 = 32 bytes along K inside the swizzle atom
          const uint64_t dah = make_desc_sw64(a_hi + ko), dal = make_desc_sw64(a_lo + ko);
          const uint64_t dwh = make_desc_sw64(w_hi + ko), dwl = make_desc_sw64(w_lo + ko);
          umma_bf16(tm, dal, dwh, (kb | j) ? 1u : 0u);  // small terms first
          umma_bf16(tm, dah, dwl, 1u);
          umma_bf16(tm, dah, dwh, 1u);
        }
        umma_commit(&empty_bar[s]);  // frees the smem stage when these MMAs retire
      }
      __syncwarp();
    }
    if (elect_one()) umma_commit(&accum_bar);  // accumulator complete
    __syncwarp();
  }

  // ============================ epilogue (warps 0-7) ============================
  // TMEM -> registers -> shared (row pitch 132 floats, conflict-free) -> coalesced row-wise
  // stores: 16 lanes cover 64 contiguous columns of one output row.  The staging area reuses
  // the operand ring, which is idle once the accumulator barrier has fired.
  if (warp < 8) {
    mbar_wait(&accum_bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int64_t c_base = p.offC ? p.offC[z] : (int64_t)z * p.strideC;
    const int lane = tid & 31;
    const int wq = warp & 3;                     // TMEM lane quarter this warp may access
    const int chalf = warp >> 2;                 // warps 0-3: columns 0-63, warps 4-7: 64-127
    constexpr int kPitch = 132;
    float* stage = reinterpret_cast<float*>(smem);   // [128][132] floats = 67.6 KB <= 96 KB ring
#pragma unroll 1
    for (int cb = chalf * 2; cb < chalf * 2 + 2; cb++) {
      if (n0 + cb * 32 >= Nz) break;            // uniform
      uint32_t r[32];
      const uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(cb * 32);
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
          "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
          "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
          : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
            "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
            "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
            "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
          : "r"(taddr)
          : "memory");
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      float* dst = stage + (wq * 32 + lane) * kPitch + cb * 32;
#pragma unroll
      for (int g = 0; g < 8; g++)
        *reinterpret_cast<float4*>(dst + g * 4) = make_float4(__uint_as_float(r[g * 4 + 0]), __uint_as_float(r[g * 4 + 1]),
                                                              __uint_as_float(r[g * 4 + 2]), __uint_as_float(r[g * 4 + 3]));
    }
    __syncwarp();
    // this warp staged rows [wq*32, wq*32+32) x columns [chalf*64, chalf*64+64): drain them row-wise
    const int n4 = lane & 15;
    const int n = n0 + chalf * 64 + n4 * 4;
#pragma unroll 4
    for (int it = 0; it < 16; it++) {
      const int rl = wq * 32 + it * 2 + (lane >> 4);
      const int m = m0 + rl;
      if (m < Mz && n < Nz) {
        const RowCtx rc = epilogue_row(p, c_base, m);
        const float4 a = *reinterpret_cast<const float4*>(stage + rl * kPitch + chalf * 64 + n4 * 4);
        const float acc[4] = {a.x, a.y, a.z, a.w};
        epilogue_store4(p, rc, n, Nz, acc);
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 8) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

}  // namespace

void launch_gemm_tc(const GemmParams& p, cudaStream_t stream) {
  if (p.M <= 0 || p.N <= 0 || p.groups <= 0) return;
  static SmemAttrCache cache;
  const size_t smem = (size_t)kStages * kStageBytesTC + (size_t)kRawStages * kRawBytes + 1024;
  if (cache.needs(smem))
    CUDA_CHECK(cudaFuncSetAttribute(gemm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((p.N + TN - 1) / TN, (p.M + TM - 1) / TM, p.groups);
  gemm_tc_kernel<<<grid, kThreadsTC, smem, stream>>>(p);
}

void launch_gemm(const GemmParams& p, cudaStream_t stream) {
  static const bool use_simt = [] {
    const char* e = std::getenv("MOONSHINE_B200_GEMM");
    return e && std::string(e) == "simt";
  }();
  if (use_simt) launch_gemm_simt(p, stream);
  else launch_gemm_tc(p, stream);
}

void gemm_tc_error_async(unsigned int* pinned_dst, cudaStream_t stream) {
  CUDA_CHECK(cudaMemcpyFromSymbolAsync(pinned_dst, g_gemm_tc_error, sizeof(unsigned int), 0, cudaMemcpyDeviceToHost, stream));
}
void gemm_tc_clear_error(cudaStream_t stream) {
  const unsigned int zero = 0;
  CUDA_CHECK(cudaMemcpyToSymbolAsync(g_gemm_tc_error, &zero, sizeof(unsigned int), 0, cudaMemcpyHostToDevice, stream));
}

}  // namespace msb
