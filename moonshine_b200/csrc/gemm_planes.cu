// Encoder dense layers on tcgen05 with BOTH operands pre-split: C[M, N] = A[M, K] . W[N, K]^T at fp32 accuracy
// (bf16x3: hi.hi + hi.lo + lo.hi, fp32 accumulation in TMEM), where A and W already lie in HBM as bf16 hi/lo planes
// in the exact UMMA K-major SWIZZLE_64B shared-memory image of a 128-row x 32-k tile:
//
//     tile (row tile rt, k-block kb) at byte ((rt * K/32) + kb) * 16384 :  [hi plane 128 x 64 B | lo plane 128 x 64 B],
//     16-byte chunk c of row r stored at chunk position c ^ ((r >> 1) & 3)
//
// so one cp.async.bulk per operand lands an MMA-ready stage and no thread ever converts anything in the main loop
// (gemm_tc.cu stages fp32 and splits it with 8 warps per stage: that conversion is its ceiling).  The weights are split
// once at load (Model::build_weights); activations are written in this form by their producers -- the LayerNorm kernel,
// this kernel's own epilogue (fc1 + GELU feeding fc2) and a small row converter for the attention output.
//
// CTA = one 128 x 128 output tile, 4 warps, 2 CTAs per SM (3 stages of 32 KB each, 128 TMEM columns each):
//   warp 0 lane 0   bulk copies of the A tiles        } a single thread sustains one bulk copy per ~0.45 us whatever its
//   warp 1 lane 0   bulk copies of the W tiles        } size (measured, profiles/r2d_ring_bandwidth_hbm_vs_l2.txt): two issuers
//   warp 2          six tcgen05.mma (M128 N128 K16) per k-block, tcgen05.commit hands the stage back
//   warps 0-3       epilogue: tcgen05.ld 32 columns at a time (thread = output row), bias / GELU / interleaved RoPE /
//                   residual accumulate, fp32 rows and / or hi-lo planes for the next GEMM
// Reference arithmetic: the encoder's q/k/o projections and MLP (HF MoonshineEncoderLayer; the ORT graphs the reference
// runs, core/moonshine-model.cpp:185-262, hold the same fp32 contractions).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <string>

#include "common.h"
#include "kernels.h"

namespace msb {
namespace {

constexpr int kStages = 3;
constexpr int kTile = kPlaneTileBytes;       // one operand tile: hi 8 KB | lo 8 KB
constexpr int kStage = 2 * kTile;            // A tile | W tile
constexpr long long kSpin = 4000000000LL;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t a, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(a), "r"(parity)
      : "memory");
  return done != 0;
}
// A wait that runs out of patience (a lost copy) poisons the launch instead of trapping the context: the flag makes every
// later wait of the grid return at once, the kernel drains with garbage, and the host turns the flag into an exception
// after its next synchronise (gemm_planes_take_error) -- the device context stays usable.
__device__ unsigned int g_planes_error = 0;
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t a = smem_u32(bar);
  if (mbar_try(a, parity)) return;
  const long long t0 = clock64();
  unsigned polls = 0;
  while (!mbar_try(a, parity)) {
    if ((++polls & 63u) == 0u) {
      if (*reinterpret_cast<volatile unsigned int*>(&g_planes_error) != 0u) return;
      if (clock64() - t0 > kSpin) { atomicExch(&g_planes_error, 1u); return; }
    }
  }
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ uint64_t make_desc_sw64(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;             // LBO (unused for swizzled K-major)
  d |= (uint64_t)(512 >> 4) << 32;    // SBO: 8 rows * 64 B
  d |= (uint64_t)1 << 46;             // descriptor version (sm_100)
  d |= (uint64_t)4 << 61;             // SWIZZLE_64B
  return d;
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
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
// D fp32, A/B bf16 K-major, M = 128, N = 128
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);

__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 ah = __float2bfloat16_rn(a), bh = __float2bfloat16_rn(b);
  const __nv_bfloat16 al = __float2bfloat16_rn(a - __bfloat162float(ah));
  const __nv_bfloat16 bl = __float2bfloat16_rn(b - __bfloat162float(bh));
  hi = (uint32_t)__bfloat16_as_ushort(ah) | ((uint32_t)__bfloat16_as_ushort(bh) << 16);
  lo = (uint32_t)__bfloat16_as_ushort(al) | ((uint32_t)__bfloat16_as_ushort(bl) << 16);
}
// 32 consecutive k values of row `row` -> the row's 64 hi bytes and 64 lo bytes of tile (row / 128, kb)
__device__ __forceinline__ void store_plane_row(unsigned char* planes, int nkb, int64_t row, int kb, const float* v) {
  const int r = (int)(row & 127);
  unsigned char* tile = planes + ((row >> 7) * nkb + kb) * (int64_t)kTile + r * 64;
  const int sw = (r >> 1) & 3;
#pragma unroll
  for (int c = 0; c < 4; c++) {
    uint4 hi, lo;
    split_bf16x2(v[c * 8 + 0], v[c * 8 + 1], hi.x, lo.x);
    split_bf16x2(v[c * 8 + 2], v[c * 8 + 3], hi.y, lo.y);
    split_bf16x2(v[c * 8 + 4], v[c * 8 + 5], hi.z, lo.z);
    split_bf16x2(v[c * 8 + 6], v[c * 8 + 7], hi.w, lo.w);
    *reinterpret_cast<uint4*>(tile + ((c ^ sw) << 4)) = hi;
    *reinterpret_cast<uint4*>(tile + (kTile / 2) + ((c ^ sw) << 4)) = lo;
  }
}
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

// one output row's 32 columns [n0, n0 + 32): bias / GELU / RoPE / residual accumulate, then whichever outputs are wanted.
// (The epilogue is the critical resource of these short-K products -- 128 x 128 x 13 k-blocks of MMAs take ~3 us, a naive
// epilogue longer -- so column -> (layer, head, dim) maps run on counters: one division per 32 columns, not per column.)
__device__ __forceinline__ void epilogue_chunk(const GemmPlanesParams& p, int64_t m, int pos, int n0, float* v) {
  const int ncols = min(32, p.N - n0);  // multiple of 4 (N % 4 == 0)
  if (p.Hk != nullptr) {  // decoder cross K (time-contiguous) | V (head rows), fp16
    if (n0 < p.n_split) {
      const int64_t base = __ldg(p.hk_row + m);
      if (base >= 0) {
        int l = n0 / p.Dm, r = n0 - l * p.Dm;
#pragma unroll
        for (int j = 0; j < 32; j++) {
          if (j < ncols) p.Hk[base + (int64_t)l * p.SL + (int64_t)r * p.Tpadm] = __float2half_rn(v[j]);
          if (++r == p.Dm) { r = 0; l++; }
        }
      }
    } else {
      const int64_t base = __ldg(p.hv_row + m);
      if (base >= 0) {
        const int n = n0 - p.n_split;
        int l = n / p.Dm, r = n - l * p.Dm, h = r / p.hdm, d = r - h * p.hdm;
        const int64_t hs = (int64_t)p.Tpadm * p.hdm;
#pragma unroll
        for (int j = 0; j < 32; j++) {
          if (j < ncols) p.Hv[base + (int64_t)l * p.SL + (int64_t)h * hs + d] = __float2half_rn(v[j]);
          if (++d == p.hdm) {
            d = 0;
            if ((++h) * p.hdm == p.Dm) { h = 0; l++; }
          }
        }
      }
    }
    return;
  }
  if (p.Vt != nullptr && n0 >= p.n_split) {
    // transposed store: lanes of a warp hold consecutive rows = consecutive t of one utterance (mostly), so every
    // column is one coalesced 128-byte line
    const int64_t base = __ldg(p.vt_row + m);
    if (base >= 0) {
      float* dst = p.Vt + base + (int64_t)(n0 - p.n_split) * p.vt_ld;
#pragma unroll
      for (int j = 0; j < 32; j++)
        if (j < ncols) dst[(int64_t)j * p.vt_ld] = v[j];
    }
    return;
  }
  if (p.bias != nullptr) {
#pragma unroll
    for (int j = 0; j < 32; j++)
      if (j < ncols) v[j] += __ldg(p.bias + n0 + j);
  }
  if (p.act == 1) {
#pragma unroll
    for (int j = 0; j < 32; j++) v[j] = gelu_erf(v[j]);
  }
  if (p.pos != nullptr && n0 < p.rope_cols) {
    // interleaved pairs (2i, 2i + 1) of the first rot_dim dims of every head; 32-column trips never split a pair
    const int half_rot = p.rot_dim >> 1;
    const float* cs_row = p.rope_cos + (int64_t)pos * half_rot;
    const float* sn_row = p.rope_sin + (int64_t)pos * half_rot;
    int d = n0 % p.head_dim;
#pragma unroll
    for (int j = 0; j < 32; j += 2) {
      if (j < ncols && n0 + j < p.rope_cols && d < p.rot_dim) {
        const float cs = __ldg(cs_row + (d >> 1)), sn = __ldg(sn_row + (d >> 1));
        const float x0 = v[j], x1 = v[j + 1];
        v[j] = x0 * cs - x1 * sn;
        v[j + 1] = x1 * cs + x0 * sn;
      }
      d += 2;
      if (d >= p.head_dim) d -= p.head_dim;
    }
  }
  if (p.C != nullptr) {
    float* dst = p.C + m * p.ldc + n0;
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      if (j < ncols) {
        float4 o = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        if (p.accumulate) {
          const float4 old = *reinterpret_cast<const float4*>(dst + j);
          o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w;
        }
        *reinterpret_cast<float4*>(dst + j) = o;
        if (p.accumulate) { v[j] = o.x; v[j + 1] = o.y; v[j + 2] = o.z; v[j + 3] = o.w; }
      }
    }
  }
  if (p.P != nullptr) {  // N % 32 == 0 (checked by the launcher)
    const int nkb_out = p.N >> 5;
    if (p.p_taps <= 1) {
      store_plane_row(p.P, nkb_out, m, n0 >> 5, v);
    } else {
      // the output IS the next convolution's im2col operand: row r of that operand is p_taps consecutive output rows
      // starting at p_stride * r, so output row m is tap k of row (m - k) / p_stride for every k congruent to m
      for (int k = (int)(m % p.p_stride); k < p.p_taps; k += p.p_stride)
        if (m >= k) store_plane_row(p.P, nkb_out * p.p_taps, (m - k) / p.p_stride, (k * p.N + n0) >> 5, v);
    }
  }
}

__global__ void __launch_bounds__(128, 2) gemm_planes_kernel(const __grid_constant__ GemmPlanesParams p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);           // [kStages]
  uint64_t* empty = full + kStages;                              // [kStages]
  uint64_t* acc_bar = empty + kStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_bar + 1);
  unsigned char* ring = smem + 1024;
  const int warp = (int)uniform_u32(threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int nkb = p.K >> 5;
  const int nt = blockIdx.x, mt = blockIdx.y;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; s++) {
      mbar_init(&full[s], 2);   // one arrive.expect_tx per producer
      mbar_init(&empty[s], 1);  // the MMA warp's commit
    }
    mbar_init(acc_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(128) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;

  if (warp < 2) {
    // ---- producers: warp 0 streams the A tiles of row tile mt, warp 1 the W tiles of row tile nt ----
    // (the whole warp walks the loop, one elected lane issues: a copy issued under `if (lane == 0)` gets a waterfall loop)
    const unsigned char* src = (warp == 0 ? p.A + (int64_t)mt * nkb * kTile : p.W + (int64_t)nt * nkb * kTile);
    unsigned char* dst0 = ring + (warp == 0 ? 0 : kTile);
    int s = 0;
    uint32_t par = 0;
    for (int kb = 0; kb < nkb; kb++) {
      mbar_wait(&empty[s], par ^ 1u);
      __syncwarp();
      if (elect_one()) {
        mbar_expect_tx(&full[s], kTile);
        bulk_g2s(dst0 + s * kStage, src + (int64_t)kb * kTile, kTile, &full[s]);
      }
      __syncwarp();
      if (++s == kStages) { s = 0; par ^= 1u; }
    }
  } else if (warp == 2) {
    // ---- MMA issue: per k-block 2 k16 steps x (hi.hi, hi.lo, lo.hi) into one 128-column accumulator ----
    int s = 0;
    uint32_t par = 0;
    for (int kb = 0; kb < nkb; kb++) {
      mbar_wait(&full[s], par);
      __syncwarp();
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t a = uniform_u32(smem_u32(ring + s * kStage));
      const uint32_t w = a + kTile;
      const uint32_t ebar = uniform_u32(smem_u32(&empty[s]));
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < 2; ks++) {
          const uint32_t ko = (uint32_t)ks * 32u;
          const uint64_t ahi = make_desc_sw64(a + ko), alo = make_desc_sw64(a + kTile / 2 + ko);
          const uint64_t whi = make_desc_sw64(w + ko), wlo = make_desc_sw64(w + kTile / 2 + ko);
          umma_bf16(tmem, alo, whi, kIdesc, (kb | ks) ? 1u : 0u);   // small terms first
          umma_bf16(tmem, ahi, wlo, kIdesc, 1u);
          umma_bf16(tmem, ahi, whi, kIdesc, 1u);
        }
        umma_commit(ebar);
      }
      __syncwarp();
      if (++s == kStages) { s = 0; par ^= 1u; }
    }
    const uint32_t abar = uniform_u32(smem_u32(acc_bar));
    if (elect_one()) umma_commit(abar);
    __syncwarp();
  }

  // ---- epilogue: all four warps; thread = output row (TMEM lane), 32 columns per trip ----
  mbar_wait(acc_bar, 0);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const int64_t m = (int64_t)mt * 128 + warp * 32 + lane;
  const bool row_ok = m < p.M;
  int pos = 0;
  if (p.pos != nullptr && row_ok) pos = p.pos[m];
#pragma unroll 1
  for (int c = 0; c < 4; c++) {
    const int n0 = nt * 128 + c * 32;
    if (n0 >= p.N) break;  // uniform
    float v[32];
    {
      uint32_t r[32];
      const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)(c * 32);
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
          "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
          "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
          : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
            "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
            "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
            "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
          : "r"(taddr));
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int j = 0; j < 32; j++) v[j] = __uint_as_float(r[j]);
    }
    if (!row_ok) continue;
    epilogue_chunk(p, m, pos, n0, v);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(128) : "memory");
  }
}

// ---- tcgen05.ld of 32 accumulator columns of this warp's 32 rows ----
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int j = 0; j < 32; j++) v[j] = __uint_as_float(r[j]);
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Persistent variant (default): one CTA per SM walks 128 x 256 macro tiles (one A tile against TWO adjacent W tiles, so
// the activations cross L2 -> SM once per 256 output columns), stages of TWO k-blocks (32 KB bulk copies: a copy costs
// ~0.45 us of its issuing thread whatever its size and an SM sustains ~4 copies / us, so 16 KB copies starve the tensor
// core), and TWO 256-column TMEM accumulators so the epilogue of tile i overlaps the main loop of tile i + 1.
//   warp 0 / 1 / 3   bulk copies of A / W0 / W1          warp 2   MMA issue          warps 4-11   epilogue (2 per lane quarter)
constexpr int kStages2 = 2;
constexpr int kStage2 = 6 * kTile;  // 2 k-blocks x (A | W0 | W1)
__global__ void __launch_bounds__(384, 1) gemm_planes_persistent_kernel(const __grid_constant__ GemmPlanesParams p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);   // [2] 3 arrivals (A, W0, W1) + bytes
  uint64_t* empty = full + kStages2;                     // [2] the MMA warp's commit
  uint64_t* acc_full = empty + kStages2;                 // [2] accumulator b complete
  uint64_t* acc_empty = acc_full + 2;                    // [2] accumulator b drained (8 epilogue warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  unsigned char* ring = smem + 1024;
  const int warp = (int)uniform_u32(threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int nkb = p.K >> 5, nst = (nkb + 1) >> 1;
  const int n_tiles = (p.N + 127) >> 7, n_macro = (n_tiles + 1) >> 1, m_tiles = (p.M + 127) >> 7;
  const int total = n_macro * m_tiles;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages2; s++) {
      mbar_init(&full[s], 3);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; b++) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], 8);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;

  if (warp == 0 || warp == 1 || warp == 3) {
    // ---- producers: operand `which` (0 = A, 1 = W0, 2 = W1) of every stage of every tile of this CTA ----
    const int which = warp == 0 ? 0 : (warp == 1 ? 1 : 2);
    int s = 0;
    uint32_t par = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
      const int mt = tile / n_macro, nm = tile - mt * n_macro;
      const int rt = which == 0 ? mt : 2 * nm + (which - 1);      // row tile of the operand
      const bool present = which == 0 || rt < n_tiles;            // the last macro tile may hold one W tile only
      const unsigned char* src = (which == 0 ? p.A : p.W) + (int64_t)rt * nkb * kTile;
      for (int st = 0; st < nst; st++) {
        const uint32_t bytes = (uint32_t)min(2, nkb - 2 * st) * kTile;
        mbar_wait(&empty[s], par ^ 1u);
        __syncwarp();
        if (elect_one()) {
          if (present) {
            mbar_expect_tx(&full[s], bytes);
            bulk_g2s(ring + s * kStage2 + which * 2 * kTile, src + (int64_t)st * 2 * kTile, bytes, &full[s]);
          } else {
            mbar_arrive(&full[s]);
          }
        }
        __syncwarp();
        if (++s == kStages2) { s = 0; par ^= 1u; }
      }
    }
  } else if (warp == 2) {
    // ---- MMA issue ----
    int s = 0;
    uint32_t par = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, it++) {
      const int mt = tile / n_macro, nm = tile - mt * n_macro;
      const bool two = 2 * nm + 1 < n_tiles;
      const int b = it & 1;
      mbar_wait(&acc_empty[b], ((uint32_t)(it >> 1) & 1u) ^ 1u);  // drained by the epilogue two tiles ago
      __syncwarp();
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t acc = tmem + (uint32_t)(b * 256);
      (void)mt;
      for (int st = 0; st < nst; st++) {
        const int nq = min(2, nkb - 2 * st);
        mbar_wait(&full[s], par);
        __syncwarp();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t base = uniform_u32(smem_u32(ring + s * kStage2));
        const uint32_t ebar = uniform_u32(smem_u32(&empty[s]));
        if (elect_one()) {
          for (int q = 0; q < nq; q++) {
            const uint32_t a = base + (uint32_t)(q * kTile), w0 = base + (uint32_t)((2 + q) * kTile), w1 = base + (uint32_t)((4 + q) * kTile);
#pragma unroll
            for (int ks = 0; ks < 2; ks++) {
              const uint32_t ko = (uint32_t)ks * 32u;
              const uint32_t first = (st | q | ks) ? 1u : 0u;
              const uint64_t ahi = make_desc_sw64(a + ko), alo = make_desc_sw64(a + kTile / 2 + ko);
              umma_bf16(acc, alo, make_desc_sw64(w0 + ko), kIdesc, first);
              umma_bf16(acc, ahi, make_desc_sw64(w0 + kTile / 2 + ko), kIdesc, 1u);
              umma_bf16(acc, ahi, make_desc_sw64(w0 + ko), kIdesc, 1u);
              if (two) {
                umma_bf16(acc + 128, alo, make_desc_sw64(w1 + ko), kIdesc, first);
                umma_bf16(acc + 128, ahi, make_desc_sw64(w1 + kTile / 2 + ko), kIdesc, 1u);
                umma_bf16(acc + 128, ahi, make_desc_sw64(w1 + ko), kIdesc, 1u);
              }
            }
          }
          umma_commit(ebar);
        }
        __syncwarp();
        if (++s == kStages2) { s = 0; par ^= 1u; }
      }
      const uint32_t abar = uniform_u32(smem_u32(&acc_full[b]));
      if (elect_one()) umma_commit(abar);
      __syncwarp();
    }
  } else {
    // ---- epilogue warps 4-11: TMEM lanes 32 (warp % 4) .. + 31, column half (warp - 4) / 4 of the macro tile ----
    const int ew = (warp - 4) & 3, half = (warp - 4) >> 2;
    int it = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, it++) {
      const int mt = tile / n_macro, nm = tile - mt * n_macro;
      const int b = it & 1;
      mbar_wait(&acc_full[b], (uint32_t)(it >> 1) & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const int64_t m = (int64_t)mt * 128 + ew * 32 + lane;
      const bool row_ok = m < p.M;
      int pos = 0;
      if (p.pos != nullptr && row_ok) pos = p.pos[m];
#pragma unroll 1
      for (int c = half * 4; c < half * 4 + 4; c++) {
        const int n0 = nm * 256 + c * 32;
        if (n0 >= p.N) break;  // uniform
        float v[32];
        tmem_ld32(tmem + ((uint32_t)(ew * 32) << 16) + (uint32_t)(b * 256 + c * 32), v);
        if (row_ok) epilogue_chunk(p, m, pos, n0, v);
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[b]);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
  }
}

// one warp per row: LayerNorm (gamma only) -> fp32 row (optional) + hi/lo planes
constexpr int kLnMax = 16;  // D <= 512
__global__ void layernorm_planes_kernel(const float* __restrict__ x, float* __restrict__ y, unsigned char* __restrict__ planes,
                                        const float* __restrict__ gamma, int64_t rows, int D) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* xr = x + row * D;
  float v[kLnMax];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMax; i++) {
    const int c = lane + i * 32;
    v[i] = c < D ? xr[c] : 0.f;
    s += v[i];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / D;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMax; i++) {
    const int c = lane + i * 32;
    const float d = c < D ? v[i] - mean : 0.f;
    q += d * d;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = rsqrtf(q / D + 1e-5f);
  const int nkb = D >> 5, r = (int)(row & 127), sw = (r >> 1) & 3;
  unsigned char* tile0 = planes + (row >> 7) * nkb * (int64_t)kTile + r * 64;
#pragma unroll
  for (int i = 0; i < kLnMax; i++) {
    const int c = lane + i * 32;  // k-block i, element `lane` of it
    if (c < D) {
      const float o = (v[i] - mean) * rstd * gamma[c];
      if (y != nullptr) y[row * D + c] = o;
      const __nv_bfloat16 h = __float2bfloat16_rn(o);
      const __nv_bfloat16 l = __float2bfloat16_rn(o - __bfloat162float(h));
      unsigned char* t = tile0 + (int64_t)i * kTile + ((((lane >> 3) ^ sw) << 4) | ((lane & 7) << 1));
      *reinterpret_cast<__nv_bfloat16*>(t) = h;
      *reinterpret_cast<__nv_bfloat16*>(t + kTile / 2) = l;
    }
  }
}

// GroupNorm(1 group) apply of the conv1 output, written straight as the plane tiles of conv2's im2col operand: operand row
// r2 = h1 rows 3 r2 .. 3 r2 + 6 (7 taps x D channels), so element (r1, c) is tap k of row (r1 - k) / 3 for k = r1 % 3, + 3, + 6.
// thread = 8 channels of one h1 row.  (reference arithmetic: HF MoonshineEncoder.groupnorm -> conv2, HF:566-572)
__global__ void groupnorm_im2col_planes_kernel(const float* __restrict__ h1, const int* __restrict__ t1, const int64_t* __restrict__ off1,
                                               const double* __restrict__ gn_partial, int nblk, const float* __restrict__ gamma,
                                               const float* __restrict__ beta, int D, unsigned char* __restrict__ planes) {
  __shared__ float stat[2];
  const int b = blockIdx.y;
  if (threadIdx.x == 0) {
    double a = 0.0, q = 0.0;
    for (int i = 0; i < nblk; i++) {
      a += gn_partial[((int64_t)b * nblk + i) * 2];
      q += gn_partial[((int64_t)b * nblk + i) * 2 + 1];
    }
    const double n = (double)t1[b] * D;
    const double mean = n > 0 ? a / n : 0.0;
    double var = n > 0 ? q / n - mean * mean : 0.0;
    if (var < 0) var = 0;
    stat[0] = (float)mean;
    stat[1] = (float)(1.0 / sqrt(var + 1e-5));
  }
  __syncthreads();
  const float mean = stat[0], rstd = stat[1];
  const int D8 = D >> 3, nkb = (7 * D) >> 5;
  const int64_t total = (int64_t)t1[b] * D8, row0 = off1[b];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = i / D8;
    const int c8 = (int)(i - t * D8);
    const int64_t r1 = row0 + t;
    const float* src = h1 + r1 * D + c8 * 8;
    const float4 a = *reinterpret_cast<const float4*>(src), c = *reinterpret_cast<const float4*>(src + 4);
    const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + c8 * 8)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + c8 * 8 + 4));
    const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta + c8 * 8)), b1 = __ldg(reinterpret_cast<const float4*>(beta + c8 * 8 + 4));
    uint4 hi, lo;
    split_bf16x2((a.x - mean) * rstd * g0.x + b0.x, (a.y - mean) * rstd * g0.y + b0.y, hi.x, lo.x);
    split_bf16x2((a.z - mean) * rstd * g0.z + b0.z, (a.w - mean) * rstd * g0.w + b0.w, hi.y, lo.y);
    split_bf16x2((c.x - mean) * rstd * g1.x + b1.x, (c.y - mean) * rstd * g1.y + b1.y, hi.z, lo.z);
    split_bf16x2((c.z - mean) * rstd * g1.z + b1.z, (c.w - mean) * rstd * g1.w + b1.w, hi.w, lo.w);
    for (int k = (int)(r1 % 3); k < 7; k += 3) {
      if (r1 < k) continue;
      const int64_t r2 = (r1 - k) / 3;
      const int kk = k * D + c8 * 8, r = (int)(r2 & 127);
      unsigned char* tdst = planes + ((r2 >> 7) * nkb + (kk >> 5)) * (int64_t)kTile + r * 64 + ((((kk & 31) >> 3) ^ ((r >> 1) & 3)) << 4);
      *reinterpret_cast<uint4*>(tdst) = hi;
      *reinterpret_cast<uint4*>(tdst + kTile / 2) = lo;
    }
  }
}

// fp32 rows -> planes (thread = one row's 8-element chunk)
__global__ void rows_to_planes_kernel(const float* __restrict__ src, int64_t ld, int64_t rows, int K, unsigned char* __restrict__ planes) {
  const int k8n = K >> 3;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * k8n) return;
  const int64_t row = i / k8n;
  const int k8 = (int)(i - row * k8n);
  const float4 a = *reinterpret_cast<const float4*>(src + row * ld + k8 * 8);
  const float4 b = *reinterpret_cast<const float4*>(src + row * ld + k8 * 8 + 4);
  uint4 hi, lo;
  split_bf16x2(a.x, a.y, hi.x, lo.x);
  split_bf16x2(a.z, a.w, hi.y, lo.y);
  split_bf16x2(b.x, b.y, hi.z, lo.z);
  split_bf16x2(b.z, b.w, hi.w, lo.w);
  const int r = (int)(row & 127), kb = k8 >> 2, c = k8 & 3;
  unsigned char* t = planes + ((row >> 7) * (K >> 5) + kb) * (int64_t)kTile + r * 64 + ((c ^ ((r >> 1) & 3)) << 4);
  *reinterpret_cast<uint4*>(t) = hi;
  *reinterpret_cast<uint4*>(t + kTile / 2) = lo;
}

}  // namespace

bool gemm_planes_supported(const GemmPlanesParams& p) {
  return p.M > 0 && p.N > 0 && p.K >= 32 && p.K % 32 == 0 && p.N % 4 == 0 && (p.P == nullptr || p.N % 32 == 0) &&
         (p.Vt == nullptr || (p.n_split % 32 == 0 && p.vt_row != nullptr && p.P == nullptr)) &&
         (p.Hk == nullptr || (p.Hv != nullptr && p.hk_row != nullptr && p.hv_row != nullptr && p.n_split % 32 == 0 && p.Vt == nullptr)) &&
         (p.p_taps <= 1 || (p.P != nullptr && p.p_stride >= 1 && p.p_stride <= p.p_taps)) &&
         (p.pos == nullptr || (p.head_dim % 2 == 0 && p.rot_dim % 2 == 0)) && (p.C == nullptr || p.ldc % 4 == 0);
}

void launch_gemm_planes(const GemmPlanesParams& p, cudaStream_t stream) {
  if (!gemm_planes_supported(p)) throw std::runtime_error("gemm_planes: unsupported shape");
  // Two mappings.  `tiles`: one 128 x 128 tile per CTA, 2 CTAs per SM -- best when a launch is only a few waves (tiny/32:
  // 105 row tiles).  `persistent`: 128 x 256 macro tiles, epilogue overlapped -- best from ~8 macro tiles per SM on
  // (base/256 encoder stage 27.2 -> 24.6 ms, base-streaming/64 7.0 -> 6.4; tiny/32 2.35 vs 2.49 the other way).
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  static int sm_count[64] = {0};
  if (dev >= 0 && dev < 64) {
    if (sm_count[dev] == 0) cudaDeviceGetAttribute(&sm_count[dev], cudaDevAttrMultiProcessorCount, dev);
    sms = sm_count[dev] > 0 ? sm_count[dev] : 148;
  }
  const int n_macro = ((p.N + 127) / 128 + 1) / 2, m_tiles = (p.M + 127) / 128;
  const int64_t total = (int64_t)n_macro * m_tiles;
  const bool tiles = p.variant == 1 || (p.variant == 0 && total < 8 * (int64_t)sms);
  if (tiles) {
    const size_t smem = 1024 + (size_t)kStages * kStage;
    static SmemAttrCache cache;
    if (cache.needs(smem)) CUDA_CHECK(cudaFuncSetAttribute(gemm_planes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((p.N + 127) / 128, (p.M + 127) / 128);
    gemm_planes_kernel<<<grid, 128, smem, stream>>>(p);
  } else {
    const size_t smem = 1024 + (size_t)kStages2 * kStage2;
    static SmemAttrCache cache;
    if (cache.needs(smem)) CUDA_CHECK(cudaFuncSetAttribute(gemm_planes_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gemm_planes_persistent_kernel<<<(unsigned)std::min<int64_t>(total, sms), 384, smem, stream>>>(p);
  }
  CUDA_CHECK(cudaGetLastError());
}

void gemm_planes_error_async(unsigned int* pinned_dst, cudaStream_t stream) {
  CUDA_CHECK(cudaMemcpyFromSymbolAsync(pinned_dst, g_planes_error, sizeof(unsigned int), 0, cudaMemcpyDeviceToHost, stream));
}
void gemm_planes_clear_error(cudaStream_t stream) {
  const unsigned int zero = 0;
  CUDA_CHECK(cudaMemcpyToSymbolAsync(g_planes_error, &zero, sizeof(unsigned int), 0, cudaMemcpyHostToDevice, stream));
}

void launch_layernorm_planes(const float* x, float* y, unsigned char* planes, const float* gamma, int64_t rows, int D,
                             cudaStream_t stream) {
  if (rows == 0) return;
  if (D % 32 != 0 || D > 32 * kLnMax) throw std::runtime_error("layernorm_planes: D must be a multiple of 32, <= 512");
  const int warps = 8;
  layernorm_planes_kernel<<<(unsigned)((rows + warps - 1) / warps), warps * 32, 0, stream>>>(x, y, planes, gamma, rows, D);
}

void launch_groupnorm_im2col_planes(const float* h1, const int* t1, const int64_t* off1, const double* gn_partial, int nblk,
                                    const float* gamma, const float* beta, int D, int B, int max_t1, unsigned char* planes,
                                    cudaStream_t stream) {
  if (B == 0 || max_t1 == 0) return;
  if (D % 32 != 0) throw std::runtime_error("groupnorm_im2col_planes: D must be a multiple of 32");
  const int64_t per = (int64_t)max_t1 * (D / 8);
  dim3 grid((unsigned)std::min<int64_t>((per + 255) / 256, 148 * 4), B);
  groupnorm_im2col_planes_kernel<<<grid, 256, 0, stream>>>(h1, t1, off1, gn_partial, nblk, gamma, beta, D, planes);
}

void launch_rows_to_planes(const float* src, int64_t ld, int64_t rows, int K, unsigned char* planes, cudaStream_t stream) {
  if (rows == 0) return;
  if (K % 32 != 0 || ld % 4 != 0) throw std::runtime_error("rows_to_planes: K must be a multiple of 32");
  const int64_t n = rows * (K >> 3);
  rows_to_planes_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(src, ld, rows, K, planes);
}

}  // namespace msb
