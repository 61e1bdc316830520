// Persistent decoder-step kernel, v2: operand streaming + tensor cores.
//
// Same phase structure and arithmetic order as decoder_step.cu (3 grid barriers
// per layer, deterministic partial sums), but every operand that does not
// depend on this step's activations -- all weights, the fp16 cross K/V cache,
// the self K/V cache up to position step-1 -- is brought into shared memory
// by two PRODUCER WARPS through a ring of TMA bulk copies
// (cp.async.bulk.shared::cluster.global + mbarrier complete_tx).  The producers
// walk the same (phase, item, operand, chunk) sequence as the 8 consumer warps
// but never wait for the grid barriers, so the HBM/L2 stream runs ahead of the
// dependency chain and the consumers only ever touch shared memory, plus the
// small activation / partial-sum exchanges through L2.
//
// Tensor-core phases (tcgen05 + TMEM, bf16x3 split, fp32 accumulate):
//   * logits: the head matrix arrives as pre-swizzled bf16 hi / lo A-operand planes; one thread issues
//     M=128 (vocab rows) x N<=64 (utterances) MMAs, tcgen05.commit hands ring stages back, the argmax is
//     taken in the TMEM epilogue (redux.sync + ballot);
//   * layer GEMVs of tiles with >= 8 utterances (QKV, cross-Q, FC1, FC2): same scheme with N = 16.
// Everything else (attention over the caches, LayerNorm, small-tile GEMVs) runs on the SIMT pipes from the ring.
// A two-utterance tile gives each utterance its own half of the CTA in the cross-attention phase.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.h"
#include "kernels.h"

namespace msb {

namespace {

constexpr int kConsumers = 256;
constexpr int kProducers = 2;                 // producer warps: the SM overlaps at most ~2 bulk copies, and only
                                              // when different warps issue them (scripts/ring_bw.py: 74 -> 140 GB/s)
constexpr int kThreads2 = kConsumers + 32 * kProducers;
constexpr int kWarpsC = kConsumers / 32;
constexpr int kStageBytes = 32768;
constexpr long long kSpinLimit = 4000000000LL;  // ~2 s of SM cycles: trap instead of hanging

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ void csync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

__device__ __forceinline__ unsigned ld_acquire(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// Consumer-side grid barrier (the producer warp never takes part).
__device__ __forceinline__ void grid_barrier(unsigned* bar, unsigned target) {
  csync();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(bar, 1u);
    const long long t0 = clock64();
    while ((int)(ld_acquire(bar) - target) < 0) {
      if (clock64() - t0 > kSpinLimit) __trap();
    }
    __threadfence();
  }
  csync();
}

// ---- mbarrier / bulk-copy primitives (PTX) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
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
    if (clock64() - t0 > kSpinLimit) __trap();
  }
}
// Same wait for threads that are NOT on the critical path (everyone but the MMA-issuing lane while a tensor-core
// phase runs): back off between polls so the spinning warps do not eat the issue slots of the one thread that
// feeds the tensor core.
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
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
    __nanosleep(64);
    if (clock64() - t0 > kSpinLimit) __trap();
  }
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---- the operand ring ----
// ---- tcgen05 helpers (UMMA descriptors, issue, commit) ----
__device__ __forceinline__ uint64_t make_desc_sw64(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;             // LBO (unused for swizzled K-major)
  d |= (uint64_t)(512 >> 4) << 32;    // SBO: 8 rows * 64 B
  d |= (uint64_t)1 << 46;             // descriptor version (sm_100)
  d |= (uint64_t)4 << 61;             // SWIZZLE_64B
  return d;
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// (a, b) -> packed bf16 pairs: hi = round-to-nearest bf16, lo = bf16 of the remainder (a in the low half)
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 ah = __float2bfloat16_rn(a), bh = __float2bfloat16_rn(b);
  const __nv_bfloat16 al = __float2bfloat16_rn(a - __bfloat162float(ah));
  const __nv_bfloat16 bl = __float2bfloat16_rn(b - __bfloat162float(bh));
  hi = (uint32_t)__bfloat16_as_ushort(ah) | ((uint32_t)__bfloat16_as_ushort(bh) << 16);
  lo = (uint32_t)__bfloat16_as_ushort(al) | ((uint32_t)__bfloat16_as_ushort(bl) << 16);
}

struct Ring {
  uint64_t* full;
  uint64_t* empty;
  char* data;
  int ns;
  // cursor over the chunk sequence (thread-local, uniform): stage index and pass parity are tracked
  // incrementally -- `idx % ns` / `idx / ns` with a runtime ns cost two integer divisions per chunk on the
  // critical path of every GEMV
  int st;        // stage of the next chunk
  uint32_t par;  // parity of the pass over the ring the next chunk belongs to
  int turn;      // producers: chunks until this lane's next turn (0 = issue this one)
  int who;       // producers: lane's slot among the kProducers issuing warps
  __device__ __forceinline__ void reset(int who_) {
    st = 0; par = 0; who = who_; turn = who_;
  }
  __device__ __forceinline__ int stage() const { return st; }
  __device__ __forceinline__ uint32_t parity() const { return par; }
  __device__ __forceinline__ void advance() {
    if (++st == ns) { st = 0; par ^= 1u; }
  }
  __device__ __forceinline__ void advance_by(int n) {
    for (int i = 0; i < n; i++) advance();
  }
  // consumers (all 256 threads call both)
  __device__ __forceinline__ const char* acquire() {
    mbar_wait(&full[st], par);
    return data + (size_t)st * kStageBytes;
  }
  // every consumer WARP releases the stage once its lanes are done reading it
  // (empty barriers count kWarpsC arrivals): no CTA-wide sync per chunk.
  __device__ __forceinline__ void release() {
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(&empty[st]);
    advance();
  }
  // producers (one lane per producer warp; every producer walks the whole sequence and issues its share)
  __device__ __forceinline__ void produce(const void* src, uint32_t bytes) {
    if (turn == 0) {
      mbar_wait(&empty[st], par ^ 1u);
      mbar_expect_tx(&full[st], bytes);
      bulk_g2s(data + (size_t)st * kStageBytes, src, bytes, &full[st]);
      turn = kProducers;
    }
    turn--;
    advance();
  }
};

// rows of a [K][N] fp32 k-major block per ring chunk
__device__ __forceinline__ int rows_per_chunk_f32(int K, int N) {
  int r = kStageBytes / (N * 4);
  return r < 1 ? 1 : (r > K ? K : r);
}
// rows of a fp16 [rows][cols] block per chunk; even row count keeps 16-byte granularity
__device__ __forceinline__ int rows_per_chunk_f16(int rows, int cols) {
  int r = (kStageBytes / (cols * 2)) & ~1;
  if (r < 2) r = 2;
  return r > rows ? rows : r;
}

struct SmemLayout2 {
  int hs, xs, act, att, red, ps, sc, flags, argv, argi, active, bars, ring, rope, bias, xp;  // byte offsets
  int actw, attw, total, ns, xg_bytes;
};

__host__ __device__ inline SmemLayout2 smem_layout2(int NBmax, int B, int D, int hd, int IC, int Tpad,
                                                    int Smax, int smem_limit) {
  SmemLayout2 L;
  L.actw = max(3 * hd, 2 * IC);
  L.attw = max(hd, IC);
  int o = 0;
  auto take = [&](int bytes) { int r = o; o += (bytes + 15) / 16 * 16; return r; };
  L.hs = take(NBmax * D * 4);
  L.xs = take(NBmax * D * 4);
  L.act = take(NBmax * L.actw * 4);
  L.att = take(NBmax * L.attw * 4);
  // split-K scratch only for small tiles (NB <= 4); larger tiles use the row-split mapping
  int red = (NBmax <= 4 ? 1024 * NBmax : 0) * 4;
  if (red < (32 + 1024) * 4) red = (32 + 1024) * 4;
  L.red = take(red);
  // the logits phase aliases [0, xg_bytes) with the bf16 hi/lo planes of its x tile
  // (nx utterances x D x 4 bytes, nx = min(64, round_up(B, 16)) but at most ~80 KB)
  {
    int nx = (B + 15) & ~15;
    if (nx > 64) nx = 64;
    while (nx > 16 && nx * D * 4 > 80 * 1024) nx -= 16;
    L.xg_bytes = nx * D * 4;
    if (o < L.xg_bytes) o = (L.xg_bytes + 15) / 16 * 16;
  }
  L.ps = take(2 * Tpad * 4);  // one probability row per half-CTA group (phase_cross)
  L.sc = take(kWarpsC * (Smax + 4) * 4);
  L.flags = take(64 * 4);
  L.argv = take(kWarpsC * 64 * 4);
  L.argi = take(kWarpsC * 64 * 4);
  L.rope = take(128 * 4);
  L.bias = take(2 * IC * 4);
  L.active = take(B);
  L.bars = take((2 * 16 + 2) * 8);  // ring full/empty, accumulator barrier, TMEM base
  o = (o + 1023) / 1024 * 1024;
  L.xp = take(((D + 31) / 32) * 2048);  // GEMV activation planes: 16 rows x (hi | lo) x 64 B per 32-wide k-block
  o = (o + 1023) / 1024 * 1024;  // SWIZZLE_64B operand chunks need 512-byte aligned stages
  L.ring = o;
  int ns = (smem_limit - o) / kStageBytes;
  if (ns > 16) ns = 16;
  L.ns = ns;
  L.total = o + ns * kStageBytes;
  return L;
}

constexpr int kProfSlots = 512;
struct Ctx {
  const float* rope;         // smem: cos[0..64) | sin[64..128) of this step's position
  float* bias;               // smem: staged FC1 bias chunk (2 * IC floats)
  unsigned char* xp;         // smem: bf16 hi/lo planes of a GEMV's activation tile (16 rows, K-major SW64)
  float* xg;                 // smem: bf16 hi/lo planes of the logits x tile (aliases hs..red)
  int nx;                    // utterances per logits pass (multiple of 16, <= 64)
  uint32_t tmem;             // TMEM base (128 columns)
  uint64_t* acc_bar;         // accumulator-ready mbarrier
  int acc_phase;
  unsigned long long* prof;  // optional [grid][kProfSlots] globaltimer stamps (thread 0)
  int prof_n;
  float *hs, *xs, *act, *att, *red, *ps, *sc, *argv;
  int *flags, *argi;
  const unsigned char* active;  // [B] 1 = utterance still decoding at kernel start
  int actw, attw;
};

__device__ __forceinline__ void prof_mark(Ctx& c, int tag) {
  if (c.prof != nullptr && threadIdx.x == 0 && c.prof_n < kProfSlots) {
    // SM cycle counter (cheap, ~20 cycles; %globaltimer costs hundreds and perturbs sub-microsecond stages);
    // reported as nanoseconds at the nominal 1.965 GHz -- stamps are only compared within one CTA
    const unsigned long long t = (unsigned long long)((double)clock64() * (1.0 / 1.965));
    c.prof[(size_t)blockIdx.x * kProfSlots + c.prof_n] = (t << 8) | (unsigned)tag;
    c.prof_n++;
  }
}

// ------------------------------------------------------------------------
// GEMMs over ring-staged weights.  Weight block Wt[K][N] (k-major, fp32) arrives
// in chunks of whole rows.  out[b][n] = sum_k x[b][k] * Wt[k][n] (+ bias[n]).
// ------------------------------------------------------------------------
// (a) split-K mapping for small row tiles: threads = (k-slice s, float4 n4).
template <int NB>
__device__ __forceinline__ void gemm_ring_splitk(Ring& ring, const float* x, int ldx, int K, int N,
                                                 const float* __restrict__ bias, float* red,
                                                 float* out, int ldo, Ctx* pc = nullptr) {
  const int N4 = N >> 2;
  int S = kConsumers / N4;
  if (S > K) S = K;
  const int t = threadIdx.x;
  const int n4 = t % N4, s = t / N4;
  const bool on = s < S;
  float acc[NB][4];
#pragma unroll
  for (int b = 0; b < NB; b++) acc[b][0] = acc[b][1] = acc[b][2] = acc[b][3] = 0.f;
  const int rpc = rows_per_chunk_f32(K, N);
  for (int k0 = 0; k0 < K; k0 += rpc) {
    const int rows = min(rpc, K - k0);
    const float4* W = reinterpret_cast<const float4*>(ring.acquire());
    if (pc) prof_mark(*pc, 42);
    if (on) {
      // 4 rows per trip, every shared-memory load issued before the first FMA: with two warps per
      // scheduler the loop is latency-bound unless the loads of several rows are in flight together
      for (int r = s; r < rows; r += 4 * S) {
        float4 w[4];
        float xv[4][NB];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int rr = r + u * S;
          const bool ok = rr < rows;
          w[u] = ok ? W[rr * N4 + n4] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int b = 0; b < NB; b++) xv[u][b] = ok ? x[b * ldx + k0 + rr] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
#pragma unroll
          for (int b = 0; b < NB; b++) {
            acc[b][0] = fmaf(xv[u][b], w[u].x, acc[b][0]);
            acc[b][1] = fmaf(xv[u][b], w[u].y, acc[b][1]);
            acc[b][2] = fmaf(xv[u][b], w[u].z, acc[b][2]);
            acc[b][3] = fmaf(xv[u][b], w[u].w, acc[b][3]);
          }
        }
      }
    }
    ring.release();
    if (pc) prof_mark(*pc, 40);
  }
  if (on) {
#pragma unroll
    for (int b = 0; b < NB; b++)
      *reinterpret_cast<float4*>(&red[(s * NB + b) * N + n4 * 4]) =
          make_float4(acc[b][0], acc[b][1], acc[b][2], acc[b][3]);
  }
  csync();
  if (pc) prof_mark(*pc, 41);
  for (int i = threadIdx.x; i < NB * N; i += kConsumers) {
    const int b = i / N, n = i - b * N;
    float v = bias ? bias[n] : 0.f;
    for (int s2 = 0; s2 < S; s2++) v += red[(s2 * NB + b) * N + n];
    out[b * ldo + n] = v;
  }
  csync();
}

// (b) row-split mapping for larger tiles: threads = (row group g, float4 n4);
// each thread owns up to MAXR rows of the tile for its 4 features, full K.
template <int NB, int MAXR>
__device__ __forceinline__ void gemm_ring_rows(Ring& ring, const float* x, int ldx, int K, int N,
                                               const float* __restrict__ bias, float* out, int ldo) {
  const int N4 = N >> 2;
  const int G = kConsumers / N4;
  const int t = threadIdx.x;
  const int n4 = t % N4, g = t / N4;
  const bool on = g < G && g < NB;
  float acc[MAXR][4];
#pragma unroll
  for (int r = 0; r < MAXR; r++) acc[r][0] = acc[r][1] = acc[r][2] = acc[r][3] = 0.f;
  const int rpc = rows_per_chunk_f32(K, N);
  for (int k0 = 0; k0 < K; k0 += rpc) {
    const int rows = min(rpc, K - k0);
    const float4* W = reinterpret_cast<const float4*>(ring.acquire());
    if (on) {
#pragma unroll 2
      for (int r = 0; r < rows; r++) {
        const float4 w = W[r * N4 + n4];
        const int k = k0 + r;
#pragma unroll
        for (int j = 0; j < MAXR; j++) {
          const int b = g + j * G;
          if (b < NB) {
            const float xv = x[b * ldx + k];
            acc[j][0] = fmaf(xv, w.x, acc[j][0]);
            acc[j][1] = fmaf(xv, w.y, acc[j][1]);
            acc[j][2] = fmaf(xv, w.z, acc[j][2]);
            acc[j][3] = fmaf(xv, w.w, acc[j][3]);
          }
        }
      }
    }
    ring.release();
  }
  if (on) {
    float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (bias) bv = reinterpret_cast<const float4*>(bias)[n4];
#pragma unroll
    for (int j = 0; j < MAXR; j++) {
      const int b = g + j * G;
      if (b < NB)
        *reinterpret_cast<float4*>(&out[b * ldo + n4 * 4]) =
            make_float4(acc[j][0] + bv.x, acc[j][1] + bv.y, acc[j][2] + bv.z, acc[j][3] + bv.w);
    }
  }
  csync();
}

// (c) tensor-core mapping (tcgen05): the weight block arrives as bf16 hi / lo A-operand planes (m-tiles of <= 128
// output features, k-blocks of 32), the activation rows are split to B-operand planes in shared memory (N = 16
// utterance columns, zero rows beyond NB), one thread issues the MMAs (3 split products per k16 step) into 16
// TMEM columns per m-tile and tcgen05.commit hands each ring stage back to the producers.  Epilogue: one
// tcgen05.ld per (warp, m-tile) gives every thread its feature's 16 utterance values.
__device__ __forceinline__ int plane_rows(int N, int mt) { return (min(128, N - mt * 128) + 7) & ~7; }
// k-blocks per ring chunk.  An M = 128 MMA reads 128 rows of the A plane it is pointed at even when the tile
// has fewer (the extra output rows are ignored), so the LAST plane of a chunk must still end inside the stage:
// (n - 1) * Rp * 128 + Rp * 64 + 128 * 64 <= kStageBytes.
__device__ __forceinline__ int plane_kb_per_chunk(int Rp) {
  const int n = (kStageBytes - 128 * 64 - Rp * 64) / (Rp * 128) + 1;
  return n < 1 ? 1 : n;
}

template <int NB>
__device__ __forceinline__ void gemm_ring_mma(Ring& ring, Ctx& c, const float* x, int ldx, int K, int N,
                                              const float* __restrict__ bias, float* out, int ldo) {
  static_assert(NB <= 16, "the activation tile is one N = 16 operand");
  const int nkb = (K + 31) >> 5, n_mt = (N + 127) >> 7;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* xp = c.xp;  // [kb][hi 16 x 64 B | lo 16 x 64 B]
  // ---- activation planes: item = (row r < 16, 16-byte chunk of 8 k) ----
  const int chunks = nkb * 4;
  for (int i = threadIdx.x; i < 16 * chunks; i += kConsumers) {
    const int r = i / chunks, c8 = i - r * chunks;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; e++) v[e] = 0.f;
    if (r < NB) {
      const float* src = x + r * ldx + c8 * 8;
      if (c8 * 8 < K) {
        const float4 a = *reinterpret_cast<const float4*>(src);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
      }
      if (c8 * 8 + 4 < K) {
        const float4 b4 = *reinterpret_cast<const float4*>(src + 4);
        v[4] = b4.x; v[5] = b4.y; v[6] = b4.z; v[7] = b4.w;
      }
    }
    uint4 hi, lo;
    split_bf16x2(v[0], v[1], hi.x, lo.x);
    split_bf16x2(v[2], v[3], hi.y, lo.y);
    split_bf16x2(v[4], v[5], hi.z, lo.z);
    split_bf16x2(v[6], v[7], hi.w, lo.w);
    const int kb = c8 >> 2, cc = c8 & 3;
    unsigned char* base = xp + (size_t)kb * 2048 + (size_t)r * 64 + ((cc ^ ((r >> 1) & 3)) << 4);
    *reinterpret_cast<uint4*>(base) = hi;
    *reinterpret_cast<uint4*>(base + 1024) = lo;
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  csync();
  // ---- MMA issue (thread 0); everyone else only moves its ring cursor ----
  constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(16 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  if (threadIdx.x == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    for (int mt = 0; mt < n_mt; mt++) {
      const int Rp = plane_rows(N, mt), kbc = plane_kb_per_chunk(Rp);
      // three accumulators per m-tile, one per split product: back-to-back MMAs into ONE accumulator serialise
      // on its latency when N is this small, independent chains overlap (summed in the epilogue)
      const uint32_t tmem_d = c.tmem + (uint32_t)(mt * 48);
      for (int kb0 = 0; kb0 < nkb; kb0 += kbc) {
        const int n = min(kbc, nkb - kb0);
        mbar_wait(&ring.full[ring.stage()], ring.parity());
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t a_base = smem_u32(ring.data + (size_t)ring.stage() * kStageBytes);
        for (int q = 0; q < n; q++) {
          const int kb = kb0 + q;
          const uint32_t a_hi = a_base + (uint32_t)(q * Rp * 128), a_lo = a_hi + (uint32_t)(Rp * 64);
          const uint32_t b_hi = smem_u32(xp + (size_t)kb * 2048), b_lo = b_hi + 1024u;
#pragma unroll
          for (int ks = 0; ks < 2; ks++) {
            if (kb * 32 + ks * 16 >= K) break;  // nothing but zero padding beyond K
            const uint32_t ko = (uint32_t)ks * 32u;
            const uint32_t acc = (kb | ks) ? 1u : 0u;
            umma_bf16(tmem_d, make_desc_sw64(a_lo + ko), make_desc_sw64(b_hi + ko), idesc, acc);
            umma_bf16(tmem_d + 16, make_desc_sw64(a_hi + ko), make_desc_sw64(b_lo + ko), idesc, acc);
            umma_bf16(tmem_d + 32, make_desc_sw64(a_hi + ko), make_desc_sw64(b_hi + ko), idesc, acc);
          }
        }
        umma_commit(&ring.empty[ring.stage()]);  // warp 0's arrival: the stage is free once the MMAs have read it
        ring.advance();
      }
    }
    umma_commit(c.acc_bar);
  } else {
    // The empty barriers count one arrival per consumer warp.  Warp 0's is the commit above; lane 0 of every
    // other warp gives its own as soon as the chunk has landed (waiting for `full` keeps an arrival from
    // slipping into the stage's previous round), which keeps 7 barrier operations off the issuing thread.
    int total = 0;
    for (int mt = 0; mt < n_mt; mt++) {
      const int kbc = plane_kb_per_chunk(plane_rows(N, mt));
      total += (nkb + kbc - 1) / kbc;
    }
    if (lane == 0 && warp != 0) {
      for (int i = 0; i < total; i++) {
        mbar_wait_relaxed(&ring.full[ring.stage()], ring.parity());
        mbar_arrive(&ring.empty[ring.stage()]);
        ring.advance();
      }
    } else {
      ring.advance_by(total);
    }
  }
  // lanes 1..31 of every warp park here (no polling) until their lane 0 is through its loop: in warp 0 that
  // keeps the divergent waiters from taking every other issue slot of the MMA-issuing thread
  __syncwarp();
  // ---- epilogue: TMEM -> out[b][n] (+ bias) ----
  mbar_wait_relaxed(c.acc_bar, (uint32_t)(c.acc_phase & 1));
  c.acc_phase++;
  __syncwarp();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  for (int mt = warp >> 2; mt < n_mt; mt += 2) {  // warps 0-3 take the even m-tiles, 4-7 the odd ones
    uint32_t r[3][16];
#pragma unroll
    for (int pr = 0; pr < 3; pr++) {
      const uint32_t taddr = c.tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(mt * 48 + pr * 16);
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
          "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
          : "=r"(r[pr][0]), "=r"(r[pr][1]), "=r"(r[pr][2]), "=r"(r[pr][3]), "=r"(r[pr][4]), "=r"(r[pr][5]),
            "=r"(r[pr][6]), "=r"(r[pr][7]), "=r"(r[pr][8]), "=r"(r[pr][9]), "=r"(r[pr][10]), "=r"(r[pr][11]),
            "=r"(r[pr][12]), "=r"(r[pr][13]), "=r"(r[pr][14]), "=r"(r[pr][15])
          : "r"(taddr)
          : "memory");
    }
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    const int n = mt * 128 + (warp & 3) * 32 + lane;
    if (n < N) {
      const float bv = bias ? bias[n] : 0.f;
#pragma unroll
      for (int b = 0; b < NB; b++)  // small cross terms first, then the hi*hi product
        out[b * ldo + n] = ((__uint_as_float(r[0][b]) + __uint_as_float(r[1][b])) + __uint_as_float(r[2][b])) + bv;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  csync();
}

// Which GEMVs take the tensor-core path: measured on B200, the single issuing thread plus the plane conversion
// cost ~2 us per call, which only pays off once the SIMT mapping is compute-heavy (tiles of >= 8 utterances)
// and the block has K >= 64 (QKV, cross-Q, FC1, FC2; not the K = head_dim output projections).  Producers and consumers apply the same rule.
__device__ __forceinline__ bool gemv_on_tensor_cores(int NB, int K) {
  return NB >= 8 && K >= 64;
}

template <int NB>
__device__ __forceinline__ void gemm_ring(Ring& ring, Ctx& c, const float* x, int ldx, int K, int N,
                                          const float* __restrict__ bias, float* out, int ldo) {
  if (gemv_on_tensor_cores(NB, K)) {
    gemm_ring_mma<NB>(ring, c, x, ldx, K, N, bias, out, ldo);
    return;
  }
  if constexpr (NB <= 4) {
    gemm_ring_splitk<NB>(ring, x, ldx, K, N, bias, c.red, out, ldo, &c);
  } else {
    // rows per thread = ceil(NB / G), G = 256 / (N/4) >= 2 for every N <= 512
    const int G = kConsumers / (N >> 2);
    if (NB <= G) gemm_ring_rows<NB, 1>(ring, x, ldx, K, N, bias, out, ldo);
    else if (NB <= 2 * G) gemm_ring_rows<NB, 2>(ring, x, ldx, K, N, bias, out, ldo);
    else if (NB <= 4 * G) gemm_ring_rows<NB, 4>(ring, x, ldx, K, N, bias, out, ldo);
    else gemm_ring_rows<NB, (NB + 1) / 2>(ring, x, ldx, K, N, bias, out, ldo);
  }
}

// producer side of a plane-packed [N][K] block: whole k-blocks of one m-tile per chunk
__device__ __forceinline__ void produce_block_planes(Ring& ring, const unsigned char* P, int N, int K) {
  const int nkb = (K + 31) >> 5, n_mt = (N + 127) >> 7;
  size_t off = 0;
  for (int mt = 0; mt < n_mt; mt++) {
    const int Rp = plane_rows(N, mt), kbc = plane_kb_per_chunk(Rp);
    for (int kb0 = 0; kb0 < nkb; kb0 += kbc) {
      const int n = min(kbc, nkb - kb0);
      ring.produce(P + off + (size_t)kb0 * Rp * 128, (uint32_t)(n * Rp * 128));
    }
    off += (size_t)Rp * nkb * 128;
  }
}
__device__ __forceinline__ size_t plane_block_bytes(int N, int K) {
  const int nkb = (K + 31) >> 5, n_mt = (N + 127) >> 7;
  size_t rows = 0;
  for (int mt = 0; mt < n_mt; mt++) rows += (size_t)plane_rows(N, mt);
  return rows * nkb * 128;
}

// producer side of a [K][N] fp32 block
__device__ __forceinline__ void produce_block_f32(Ring& ring, const float* Wt, int K, int N) {
  const int rpc = rows_per_chunk_f32(K, N);
  for (int k0 = 0; k0 < K; k0 += rpc) {
    const int rows = min(rpc, K - k0);
    ring.produce(Wt + (size_t)k0 * N, (uint32_t)rows * N * 4);
  }
}
__device__ __forceinline__ void produce_block_f16(Ring& ring, const __half* M, int rows, int cols) {
  const int rpc = rows_per_chunk_f16(rows, cols);
  for (int r0 = 0; r0 < rows; r0 += rpc) {
    const int n = min(rpc, rows - r0);
    ring.produce(M + (size_t)r0 * cols, (uint32_t)n * cols * 2);
  }
}

// LayerNorm WITHOUT the affine weight: gamma is folded into the rows of the
// following weight block at load time (Model::build_weights), so the dependency
// chain holds no global load here.
__device__ __forceinline__ void layernorm_rows(const float* hs, float* xs, int nb, int D) {
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int b = w; b < nb; b += kWarpsC) {
    const float* h = hs + b * D;
    float s = 0.f;
    for (int c = lane; c < D; c += 32) s += h[c];
    const float mean = warp_sum(s) / D;
    float q = 0.f;
    for (int c = lane; c < D; c += 32) {
      const float d = h[c] - mean;
      q += d * d;
    }
    const float rstd = rsqrtf(warp_sum(q) / D + 1e-5f);
    for (int c = lane; c < D; c += 32) xs[b * D + c] = (h[c] - mean) * rstd;
  }
  csync();
}

__device__ __forceinline__ int resolve_token_warp(const DecoderParams& p, int b, int parity) {
  const int lane = threadIdx.x & 31;
  float bv = -INFINITY;
  int bi = 0x7fffffff;
  const float* cv = p.cand_val + (int64_t)parity * p.n_vchunk * p.B;
  const int* ci = p.cand_idx + (int64_t)parity * p.n_vchunk * p.B;
  for (int c = lane; c < p.n_vchunk; c += 32) {
    const float v = cv[(int64_t)c * p.B + b];
    const int i = ci[(int64_t)c * p.B + b];
    if (v > bv || (v == bv && i < bi)) { bv = v; bi = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  if (bi == 0x7fffffff) bi = 0;
  return bi;
}

// Step prologue for an utterance that was active at kernel start (whole warp).
// Records the token emitted by the previous step; an utterance that finishes
// now (EOS consumed / max_len reached) is flagged done for LATER launches but
// still flows through this launch (its results are ignored), so that the
// producer warp and the consumers agree on the work list without talking.
__device__ __forceinline__ int step_prologue_warp(const DecoderParams& p, int b, bool writer) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)b * (p.Smax + 1);
  int tok_in;
  bool finished;
  if (p.step == 0) {
    tok_in = p.forced ? p.forced[row] : p.tokens[row];
    finished = p.max_len[b] <= 0;
  } else {
    const int emitted = resolve_token_warp(p, b, (p.step - 1) & 1);
    tok_in = p.forced ? p.forced[row + p.step] : emitted;
    finished = (tok_in == 2) || (p.step >= p.max_len[b]);
    if (writer && lane == 0) {
      p.tokens[row + p.step] = emitted;
      p.n_tokens[b] = p.step + 1;
    }
  }
  if (finished && writer && lane == 0) p.done[b] = 1;
  if (tok_in < 0 || tok_in >= p.V) tok_in = 0;
  return tok_in;
}

__device__ __forceinline__ void load_flags(const DecoderParams& p, const Ctx& c, int NB, int b0,
                                           bool with_enc_len = false) {
  if (threadIdx.x < NB) {
    const int b = b0 + threadIdx.x;
    c.flags[threadIdx.x] = (b < p.B) ? (c.active[b] ? 0 : 1) : 1;
    if (with_enc_len) c.flags[32 + threadIdx.x] = (b < p.B) ? p.enc_len[b] : 0;
  }
  csync();
}

__device__ __forceinline__ bool tile_active(const DecoderParams& p, const unsigned char* active, int NB,
                                            int b0) {
  bool any = false;
  for (int b = 0; b < NB; b++) any |= (b0 + b < p.B) && active[b0 + b];
  return any;
}

__device__ __forceinline__ void resolve_rows(const DecoderParams& p, const Ctx& c, int NB, int b0,
                                             const float* hrd, float* hwr, const float* part,
                                             int nparts, const float* __restrict__ bias, bool store) {
  const int D4 = p.D >> 2;
  for (int i = threadIdx.x; i < NB * D4; i += kConsumers) {
    const int b = i / D4, c4 = i - b * D4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!c.flags[b]) {
      const int64_t r = (int64_t)(b0 + b) * D4 + c4;
      v = reinterpret_cast<const float4*>(hrd)[r];
      const float4* pp = reinterpret_cast<const float4*>(part) + r;
      const int64_t pstride = (int64_t)p.B * D4;
      int j = 0;
      for (; j + 8 <= nparts; j += 8) {  // 8 independent loads in flight, summed in order
        float4 q[8];
#pragma unroll
        for (int u = 0; u < 8; u++) q[u] = pp[(int64_t)(j + u) * pstride];
#pragma unroll
        for (int u = 0; u < 8; u++) { v.x += q[u].x; v.y += q[u].y; v.z += q[u].z; v.w += q[u].w; }
      }
      for (; j < nparts; j++) {
        const float4 q = pp[(int64_t)j * pstride];
        v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
      }
      if (bias) {
        const float4 q = reinterpret_cast<const float4*>(bias)[c4];
        v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
      }
      if (store) reinterpret_cast<float4*>(hwr)[r] = v;
    }
    reinterpret_cast<float4*>(c.hs)[b * D4 + c4] = v;
  }
  csync();
}

__device__ __forceinline__ void store_partial(const DecoderParams& p, const Ctx& c, int NB, int b0,
                                              float* part_slice) {
  const int D4 = p.D >> 2;
  for (int i = threadIdx.x; i < NB * D4; i += kConsumers) {
    const int b = i / D4, c4 = i - b * D4;
    if (!c.flags[b])
      reinterpret_cast<float4*>(part_slice)[(int64_t)(b0 + b) * D4 + c4] =
          reinterpret_cast<const float4*>(c.hs)[b * D4 + c4];
  }
  csync();
}

// ============================== phase A =================================
__device__ __forceinline__ void produce_self(const DecoderParams& p, int l, int item, int NB, Ring& ring,
                                             const unsigned char* active) {
  const int H = p.H, hd = p.hd, D = p.D;
  const int h = item % H, b0 = (item / H) * NB;
  if (!tile_active(p, active, NB, b0)) return;
  const DecLayerWeights& w = p.layers[l];
  if (gemv_on_tensor_cores(NB, D)) produce_block_planes(ring, w.wqkvP + (size_t)h * plane_block_bytes(3 * hd, D), 3 * hd, D);
  else produce_block_f32(ring, w.wqkv + (int64_t)h * D * 3 * hd, D, 3 * hd);
  if (p.step > 0) {
    for (int b = 0; b < NB; b++) {
      if (b0 + b >= p.B || !active[b0 + b]) continue;
      const int64_t bh = ((int64_t)l * p.B + (b0 + b)) * H + h;
      produce_block_f32(ring, p.ks + bh * hd * p.Smax, hd, p.Smax);   // K^T [hd][Smax]
      produce_block_f32(ring, p.vs + bh * p.Smax * hd, p.step, hd);   // V rows [0, step)
    }
  }
  if (gemv_on_tensor_cores(NB, hd)) produce_block_planes(ring, w.woP + (size_t)h * plane_block_bytes(D, hd), D, hd);
  else produce_block_f32(ring, w.wo + (int64_t)h * hd * D, hd, D);
}

template <int NB>
__device__ void phase_self(const DecoderParams& p, int l, int item, Ctx& c, Ring& ring,
                           const float* hrd, float* hwr, const float* partC, float* partA) {
  const int D = p.D, hd = p.hd, H = p.H;
  const int h = item % H;
  const int b0 = (item / H) * NB;
  if (!tile_active(p, c.active, NB, b0)) return;
  const DecLayerWeights& w = p.layers[l];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int actw = c.actw, attw = c.attw;

  load_flags(p, c, NB, b0);
  if (l == 0) {
    for (int b = warp; b < NB; b += kWarpsC) {
      int tok = 0;
      if (!c.flags[b]) tok = step_prologue_warp(p, b0 + b, h == 0);
      if (lane == 0) c.flags[32 + b] = tok;
    }
    csync();
    const int D4 = D >> 2;
    for (int i = threadIdx.x; i < NB * D4; i += kConsumers) {
      const int b = i / D4, c4 = i - b * D4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (!c.flags[b]) {
        v = reinterpret_cast<const float4*>(p.embed)[(int64_t)c.flags[32 + b] * D4 + c4];
        if (h == 0) reinterpret_cast<float4*>(hwr)[(int64_t)(b0 + b) * D4 + c4] = v;
      }
      reinterpret_cast<float4*>(c.hs)[b * D4 + c4] = v;
    }
    csync();
  } else {
    resolve_rows(p, c, NB, b0, hrd, hwr, partC, p.n_chunk, p.layers[l - 1].b2, h == 0);
  }
  prof_mark(c, 1);
  layernorm_rows(c.hs, c.xs, NB, D);
  prof_mark(c, 2);
  gemm_ring<NB>(ring, c, c.xs, D, D, 3 * hd, nullptr, c.act, actw);
  prof_mark(c, 3);

  {  // RoPE (interleaved pairs) on q and k at position `step`
    const int half_rot = p.rot_dim >> 1;
    for (int i = threadIdx.x; i < NB * 2 * half_rot; i += kConsumers) {
      const int b = i / (2 * half_rot);
      const int r = i - b * 2 * half_rot;
      const int which = r / half_rot;
      const int pr = r - which * half_rot;
      const float cs = c.rope[pr];
      const float sn = c.rope[64 + pr];
      float* v = c.act + b * actw + which * hd + 2 * pr;
      const float x0 = v[0], x1 = v[1];
      v[0] = x0 * cs - x1 * sn;
      v[1] = x1 * cs + x0 * sn;
    }
  }
  csync();
  for (int i = threadIdx.x; i < NB * hd; i += kConsumers) {  // KV append
    const int b = i / hd, d = i - b * hd;
    if (!c.flags[b]) {
      const int64_t bh = ((int64_t)l * p.B + (b0 + b)) * H + h;
      p.ks[(bh * hd + d) * p.Smax + p.step] = c.act[b * actw + hd + d];
      p.vs[(bh * p.Smax + p.step) * hd + d] = c.act[b * actw + 2 * hd + d];
    }
  }
  // causal self-attention: ONE WARP per utterance (round-robin), warp-level syncs only.
  // Cache chunks arrive in utterance order; every warp acquires / releases every chunk (the
  // ring is CTA-wide) but only the owner warp computes on it, so utterances overlap.
  const float scale = rsqrtf((float)hd);
  {
    float* sc = c.sc + warp * (p.Smax + 4);
    int owner = 0;
    for (int b = 0; b < NB; b++) {
      if (c.flags[b]) continue;  // uniform
      const bool mine = (owner == warp);
      owner = (owner + 1) & (kWarpsC - 1);
      const float* q = c.act + b * actw;
      const float* kcur = q + hd;
      const float* vcur = q + 2 * hd;
      // scores: lane owns key positions t = lane, lane+32, ...
      if (mine)
        for (int t = lane; t <= p.step; t += 32) sc[t] = 0.f;
      if (p.step > 0) {
        const int rpc = rows_per_chunk_f32(hd, p.Smax);
        for (int d0 = 0; d0 < hd; d0 += rpc) {
          const int nd = min(rpc, hd - d0);
          const float* Kc = reinterpret_cast<const float*>(ring.acquire());
          if (mine) {
            for (int t = lane; t < p.step; t += 32) {
              float s = sc[t];
              for (int d = 0; d < nd; d++) s = fmaf(q[d0 + d], Kc[d * p.Smax + t], s);
              sc[t] = s;
            }
          }
          ring.release();
        }
      }
      float inv = 0.f;
      if (mine) {
        float s = 0.f;
        for (int d = lane; d < hd; d += 32) s = fmaf(q[d], kcur[d], s);
        s = warp_sum(s);
        if (lane == 0) sc[p.step] = s;
        __syncwarp();
        float mx = -INFINITY;
        for (int t = lane; t <= p.step; t += 32) mx = fmaxf(mx, sc[t] * scale);
        mx = warp_max(mx);
        float sum = 0.f;
        for (int t = lane; t <= p.step; t += 32) {
          const float e = expf(sc[t] * scale - mx);
          sc[t] = e;
          sum += e;
        }
        inv = 1.0f / warp_sum(sum);
        __syncwarp();
      }
      float o0 = 0.f, o1 = 0.f;  // lane owns dims d = lane, lane + 32 (hd <= 64)
      if (p.step > 0) {
        const int rpc = rows_per_chunk_f32(p.step, hd);
        for (int r0 = 0; r0 < p.step; r0 += rpc) {
          const int nr = min(rpc, p.step - r0);
          const float* Vc = reinterpret_cast<const float*>(ring.acquire());
          if (mine) {
            for (int t = 0; t < nr; t++) {
              const float pt = sc[r0 + t];
              if (lane < hd) o0 = fmaf(pt, Vc[t * hd + lane], o0);
              if (lane + 32 < hd) o1 = fmaf(pt, Vc[t * hd + lane + 32], o1);
            }
          }
          ring.release();
        }
      }
      if (mine) {
        const float pl = sc[p.step];
        if (lane < hd) c.att[b * attw + lane] = fmaf(pl, vcur[lane], o0) * inv;
        if (lane + 32 < hd) c.att[b * attw + lane + 32] = fmaf(pl, vcur[lane + 32], o1) * inv;
      }
    }
  }
  csync();
  prof_mark(c, 4);
  gemm_ring<NB>(ring, c, c.att, attw, hd, D, nullptr, c.hs, D);
  prof_mark(c, 5);
  store_partial(p, c, NB, b0, partA + (int64_t)h * p.B * D);
  prof_mark(c, 6);
}

// ============================== phase B =================================
__device__ __forceinline__ void produce_cross(const DecoderParams& p, int l, int item, int NB, Ring& ring,
                                              const unsigned char* active) {
  const int H = p.H, hd = p.hd, D = p.D;
  const int h = item % H, b0 = (item / H) * NB;
  if (!tile_active(p, active, NB, b0)) return;
  const DecLayerWeights& w = p.layers[l];
  if (gemv_on_tensor_cores(NB, D)) produce_block_planes(ring, w.wqcP + (size_t)h * plane_block_bytes(hd, D), hd, D);
  else produce_block_f32(ring, w.wqc + (int64_t)h * D * hd, D, hd);
  for (int b = 0; b < NB; b++) {
    if (b0 + b >= p.B || !active[b0 + b]) continue;
    const int64_t bh = ((int64_t)l * p.B + (b0 + b)) * H + h;
    produce_block_f16(ring, p.kc + bh * hd * p.Tpad, hd, p.Tpad);   // K^T [hd][Tpad]
    produce_block_f16(ring, p.vc + bh * p.Tpad * hd, p.Tpad, hd);   // V   [Tpad][hd]
  }
  if (gemv_on_tensor_cores(NB, hd)) produce_block_planes(ring, w.wocP + (size_t)h * plane_block_bytes(D, hd), D, hd);
  else produce_block_f32(ring, w.woc + (int64_t)h * hd * D, hd, D);
}

template <int NB>
__device__ void phase_cross(const DecoderParams& p, int l, int item, Ctx& c, Ring& ring,
                            const float* hrd, float* hwr, const float* partA, float* partB) {
  const int D = p.D, hd = p.hd, H = p.H;
  const int h = item % H;
  const int b0 = (item / H) * NB;
  if (!tile_active(p, c.active, NB, b0)) return;
  const DecLayerWeights& w = p.layers[l];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int actw = c.actw, attw = c.attw;

  load_flags(p, c, NB, b0, true);
  resolve_rows(p, c, NB, b0, hrd, hwr, partA, H, nullptr, h == 0);
  prof_mark(c, 11);
  layernorm_rows(c.hs, c.xs, NB, D);
  prof_mark(c, 12);
  gemm_ring<NB>(ring, c, c.xs, D, D, hd, nullptr, c.act, actw);
  prof_mark(c, 13);

  const float scale = rsqrtf((float)hd);
  const int Tpad = p.Tpad;
  const int tpr = hd >> 2;           // threads per V row (4 halves = 8 bytes each)
  // Thread groups.  A tile of two utterances gives each utterance its own half of the CTA (4 warps, own named
  // barrier and scratch): the two attentions run side by side instead of back to back -- one utterance keeps only
  // ~T/4 of 256 threads busy in the score pass anyway.  Otherwise the whole CTA walks the utterances in turn.
  const bool halves = (NB == 2) && (Tpad <= 512);
  const int half = halves ? (int)(threadIdx.x >> 7) : 0;
  const int gtid = halves ? (int)(threadIdx.x & 127) : (int)threadIdx.x;
  const int gthreads = halves ? 128 : kConsumers;
  const int gwarps = gthreads >> 5;
  const int gwarp = gtid >> 5;
  auto gsync = [&]() {
    if (halves) {
      if (half == 0) asm volatile("bar.sync 2, 128;" ::: "memory");
      else asm volatile("bar.sync 3, 128;" ::: "memory");
    } else {
      csync();
    }
  };
  const int G = gthreads / tpr;      // V rows per pass
  float* ps = c.ps + (halves ? half * Tpad : 0);
  float* red_max = c.red + half * 8;        // [<= 8] warp maxima
  float* red_sum = c.red + 16 + half * 8;   // [<= 8] warp sums
  float* pv = c.red + 32 + half * 512;      // [G][hd] PV partials (G * hd <= 1024, <= 512 per half)
  for (int b = 0; b < NB; b++) {
    if (c.flags[b]) continue;  // uniform
    const bool mine = !halves || (b == half);  // every thread walks every chunk; only the owner group computes
    const int T = c.flags[32 + b];   // encoder length, staged by load_flags
    const float* q = c.act + b * actw;
    // ---- scores over K^T chunks (rows = head dims); group thread j owns t = 4j .. 4j+3 ----
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    const int t4 = gtid * 4;
    {
      const int rpc = rows_per_chunk_f16(hd, Tpad);
      for (int d0 = 0; d0 < hd; d0 += rpc) {
        const int nd = min(rpc, hd - d0);
        const __half* Kc = reinterpret_cast<const __half*>(ring.acquire());
        if (mine && t4 < Tpad) {
#pragma unroll 4
          for (int d = 0; d < nd; d++) {
            const uint2 u = *reinterpret_cast<const uint2*>(Kc + d * Tpad + t4);
            const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
            const float2 f1 = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
            const float qd = q[d0 + d];
            s0 = fmaf(qd, f0.x, s0);
            s1 = fmaf(qd, f0.y, s1);
            s2 = fmaf(qd, f1.x, s2);
            s3 = fmaf(qd, f1.y, s3);
          }
        }
        ring.release();
      }
    }
    float inv = 0.f;
    if (mine) {
      float lmax = -INFINITY;
      if (t4 < Tpad) {
        s0 = (t4 + 0 < T) ? s0 * scale : -INFINITY;
        s1 = (t4 + 1 < T) ? s1 * scale : -INFINITY;
        s2 = (t4 + 2 < T) ? s2 * scale : -INFINITY;
        s3 = (t4 + 3 < T) ? s3 * scale : -INFINITY;
        lmax = fmaxf(fmaxf(s0, s1), fmaxf(s2, s3));
      }
      lmax = warp_max(lmax);
      if (lane == 0) red_max[gwarp] = lmax;
      gsync();                                   // (1) maxima visible; previous utterance fully done
      float mx = red_max[0];
      for (int i = 1; i < gwarps; i++) mx = fmaxf(mx, red_max[i]);
      float lsum = 0.f;
      if (t4 < Tpad) {
        s0 = (t4 + 0 < T) ? expf(s0 - mx) : 0.f;
        s1 = (t4 + 1 < T) ? expf(s1 - mx) : 0.f;
        s2 = (t4 + 2 < T) ? expf(s2 - mx) : 0.f;
        s3 = (t4 + 3 < T) ? expf(s3 - mx) : 0.f;
        *reinterpret_cast<float4*>(&ps[t4]) = make_float4(s0, s1, s2, s3);
        lsum = (s0 + s1) + (s2 + s3);
      }
      lsum = warp_sum(lsum);
      if (lane == 0) red_sum[gwarp] = lsum;
      gsync();                                   // (2) probabilities and sums visible
      float tot = 0.f;
      for (int i = 0; i < gwarps; i++) tot += red_sum[i];
      inv = 1.0f / tot;
      if (p.xattn_out != nullptr && t4 < Tpad) {  // word timestamps: export this (utterance, layer, head, step) row
        float* dst = p.xattn_out +
                     (((((int64_t)(b0 + b) * p.L + l) * H + h) * p.xattn_steps + p.step) * Tpad + t4);
        *reinterpret_cast<float4*>(dst) = make_float4(s0 * inv, s1 * inv, s2 * inv, s3 * inv);
      }
    }
    // ---- PV over V chunks (rows = time); group thread (g, dq) owns 4 dims of rows g, g+G, ... ----
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    const int g = gtid / tpr, dq = gtid - g * tpr;
    {
      const int rpc = rows_per_chunk_f16(Tpad, hd);
      for (int r0 = 0; r0 < Tpad; r0 += rpc) {
        const int nr = min(rpc, Tpad - r0);
        const __half* Vc = reinterpret_cast<const __half*>(ring.acquire());
        if (mine && g < G) {
          const int tend = min(nr, T - r0);
#pragma unroll 4
          for (int t = g; t < tend; t += G) {
            const uint2 u = *reinterpret_cast<const uint2*>(Vc + t * hd + dq * 4);
            const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
            const float2 f1 = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
            const float pt = ps[r0 + t];
            a0 = fmaf(pt, f0.x, a0);
            a1 = fmaf(pt, f0.y, a1);
            a2 = fmaf(pt, f1.x, a2);
            a3 = fmaf(pt, f1.y, a3);
          }
        }
        ring.release();
      }
    }
    if (mine) {
      if (g < G) *reinterpret_cast<float4*>(&pv[g * hd + dq * 4]) = make_float4(a0, a1, a2, a3);
      gsync();                                   // (3) PV partials visible
      if (gtid < hd) {
        float o = 0.f;
        for (int gg = 0; gg < G; gg++) o += pv[gg * hd + gtid];
        c.att[b * attw + gtid] = o * inv;
      }
    }
    // no sync here: the next utterance only overwrites red_max before its sync (1), ps after
    // it and pv after its sync (2) -- by then every thread of the group has left this reduction.
  }
  csync();
  prof_mark(c, 14);
  gemm_ring<NB>(ring, c, c.att, attw, hd, D, nullptr, c.hs, D);
  prof_mark(c, 15);
  store_partial(p, c, NB, b0, partB + (int64_t)h * p.B * D);
  prof_mark(c, 16);
}

// ============================== phase C =================================
__device__ __forceinline__ void produce_mlp(const DecoderParams& p, int l, int item, int NB, Ring& ring,
                                            const unsigned char* active) {
  const int D = p.D, IC = p.IC;
  const int ch = item % p.n_chunk, b0 = (item / p.n_chunk) * NB;
  if (!tile_active(p, active, NB, b0)) return;
  const DecLayerWeights& w = p.layers[l];
  if (gemv_on_tensor_cores(NB, D)) produce_block_planes(ring, w.w1P + (size_t)ch * plane_block_bytes(2 * IC, D), 2 * IC, D);
  else produce_block_f32(ring, w.w1 + (int64_t)ch * D * 2 * IC, D, 2 * IC);
  if (gemv_on_tensor_cores(NB, IC)) produce_block_planes(ring, w.w2P + (size_t)ch * plane_block_bytes(D, IC), D, IC);
  else produce_block_f32(ring, w.w2 + (int64_t)ch * IC * D, IC, D);
}

template <int NB>
__device__ void phase_mlp(const DecoderParams& p, int l, int item, Ctx& c, Ring& ring,
                          const float* hrd, float* hwr, const float* partB, float* partC) {
  const int D = p.D, IC = p.IC;
  const int ch = item % p.n_chunk;
  const int b0 = (item / p.n_chunk) * NB;
  if (!tile_active(p, c.active, NB, b0)) return;
  const DecLayerWeights& w = p.layers[l];
  const int actw = c.actw, attw = c.attw;
  for (int i = threadIdx.x; i < 2 * IC; i += kConsumers) c.bias[i] = w.b1[(int64_t)ch * 2 * IC + i];
  load_flags(p, c, NB, b0);
  resolve_rows(p, c, NB, b0, hrd, hwr, partB, p.H, nullptr, ch == 0);
  prof_mark(c, 21);
  layernorm_rows(c.hs, c.xs, NB, D);
  prof_mark(c, 22);
  gemm_ring<NB>(ring, c, c.xs, D, D, 2 * IC, c.bias, c.act, actw);
  prof_mark(c, 23);
  for (int i = threadIdx.x; i < NB * IC; i += kConsumers) {
    const int b = i / IC, j = i - b * IC;
    const float up = c.act[b * actw + j];
    const float gate = c.act[b * actw + IC + j];
    c.att[b * attw + j] = gate / (1.0f + expf(-gate)) * up;  // silu(gate) * up
  }
  csync();
  gemm_ring<NB>(ring, c, c.att, attw, IC, D, nullptr, c.hs, D);
  prof_mark(c, 25);
  store_partial(p, c, NB, b0, partC + (int64_t)ch * p.B * D);
  prof_mark(c, 26);
}

// ============================== phase F =================================
template <int NB>
__device__ void phase_final_ln(const DecoderParams& p, int item, Ctx& c, const float* hrd,
                               const float* partC) {
  const int D = p.D;
  const int b0 = item * NB;
  load_flags(p, c, NB, b0);
  resolve_rows(p, c, NB, b0, hrd, nullptr, partC, p.n_chunk, p.layers[p.L - 1].b2, false);
  layernorm_rows(c.hs, c.xs, NB, D);
  for (int i = threadIdx.x; i < NB * D; i += kConsumers) {
    const int b = i / D;
    if (b0 + b < p.B) p.xfin[(int64_t)(b0 + b) * D + (i - b * D)] = c.xs[i];
  }
  csync();
}

// ============================== phase G =================================
// Tied-embedding logits on tcgen05.  The CTA's vocab slab arrives through the ring ALREADY in the
// tensor core's operand format (bf16 hi/lo planes, K-major SWIZZLE_64B, built once at load time),
// so the only consumer of those stages is the MMA itself: thread 0 issues
//   D[128 vocab rows][Nx utterances] += A(slab chunk) * B(x planes)^T      (kind::f16, bf16x3)
// into TMEM and tcgen05.commit releases the ring stage when the MMAs have read it.  The x tile
// (final-LN rows of up to 64 utterances) is split to bf16 planes in shared memory once per pass.
// Epilogue: tcgen05.ld gives each thread one vocab row x Nx utterances; the per-utterance argmax is
// reduced across the CTA and only (value, index) candidates leave the SM.
__device__ __forceinline__ int logits_rows_per_pass(int B, int D, int xg_bytes) {
  int nx = (xg_bytes / (D * 4)) & ~15;
  if (nx > 64) nx = 64;
  const int b16 = (B + 15) & ~15;
  return nx < b16 ? nx : b16;
}

// chunk = up to two 32-wide k-blocks of one m-tile: [kb][hi R x 64 B | lo R x 64 B]
__device__ __forceinline__ void produce_logits(const DecoderParams& p, int item, Ring& ring, int nx) {
  const int D = p.D, VC = p.vchunk;
  const int n_mt = (VC + 127) >> 7, nkb = D >> 5;
  const unsigned char* slab = reinterpret_cast<const unsigned char*>(p.embP) + (size_t)item * VC * D * 4;
  for (int b0 = 0; b0 < p.B; b0 += nx) {
    size_t mt_off = 0;
    for (int mt = 0; mt < n_mt; mt++) {
      const int R = min(128, VC - mt * 128);
      for (int kb = 0; kb < nkb; kb += 2) {
        const int n = min(2, nkb - kb);
        ring.produce(slab + mt_off + (size_t)kb * R * 128, (uint32_t)(n * R * 128));
      }
      mt_off += (size_t)R * D * 4;
    }
  }
}

__device__ void phase_logits(const DecoderParams& p, int item, Ctx& c, Ring& ring) {
  const int D = p.D, V = p.V, VC = p.vchunk;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_mt = (VC + 127) >> 7, nkb = D >> 5;
  const int nx = c.nx;
  const int parity = p.step & 1;
  unsigned char* xp = reinterpret_cast<unsigned char*>(c.xg);  // [kb][hi nx x 64 B | lo nx x 64 B]
  const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(nx >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  for (int b0 = 0; b0 < p.B; b0 += nx) {
    const int nb = min(nx, p.B - b0);
    // ---- x planes: thread handles (row, 16-byte chunk of 8 k); loads batched 4 deep ----
    const int k8n = D >> 3, nitems = nx * k8n;
    for (int i0 = threadIdx.x; i0 < nitems; i0 += 4 * kConsumers) {
      float4 va[4], vb[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int i = i0 + u * kConsumers;
        const int r = i / k8n, k8 = i - r * k8n;
        va[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        vb[u] = va[u];
        if (i < nitems && r < nb) {
          va[u] = *reinterpret_cast<const float4*>(p.xfin + (int64_t)(b0 + r) * D + k8 * 8);
          vb[u] = *reinterpret_cast<const float4*>(p.xfin + (int64_t)(b0 + r) * D + k8 * 8 + 4);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int i = i0 + u * kConsumers;
        if (i >= nitems) break;
        const int r = i / k8n, k8 = i - r * k8n;
        uint4 hi, lo;
        split_bf16x2(va[u].x, va[u].y, hi.x, lo.x);
        split_bf16x2(va[u].z, va[u].w, hi.y, lo.y);
        split_bf16x2(vb[u].x, vb[u].y, hi.z, lo.z);
        split_bf16x2(vb[u].z, vb[u].w, hi.w, lo.w);
        const int kb = k8 >> 2, cc = k8 & 3;
        unsigned char* base = xp + (size_t)kb * nx * 128 + (size_t)r * 64 + ((cc ^ ((r >> 1) & 3)) << 4);
        *reinterpret_cast<uint4*>(base) = hi;
        *reinterpret_cast<uint4*>(base + nx * 64) = lo;
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    csync();
    prof_mark(c, 35);
    // ---- MMA issue (one thread); everyone else just advances its ring cursor ----
    int nchunks = 0;
    for (int mt = 0; mt < n_mt; mt++) nchunks += (nkb + 1) >> 1;
    if (threadIdx.x == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      for (int mt = 0; mt < n_mt; mt++) {
        const int R = min(128, VC - mt * 128);
        const uint32_t tmem_d = c.tmem + (uint32_t)(mt * nx);
        for (int kb = 0; kb < nkb; kb += 2) {
          const int n = min(2, nkb - kb);
          mbar_wait(&ring.full[ring.stage()], ring.parity());
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t a_base = smem_u32(ring.data + (size_t)ring.stage() * kStageBytes);
          for (int q = 0; q < n; q++) {
            const uint32_t a_hi = a_base + (uint32_t)(q * R * 128), a_lo = a_hi + (uint32_t)(R * 64);
            const uint32_t b_hi = smem_u32(xp + (size_t)(kb + q) * nx * 128), b_lo = b_hi + (uint32_t)(nx * 64);
#pragma unroll
            for (int jj = 0; jj < 2; jj++) {
              const uint32_t ko = (uint32_t)jj * 32u;
              const uint32_t first = (kb | q | jj) ? 1u : 0u;
              umma_bf16(tmem_d, make_desc_sw64(a_lo + ko), make_desc_sw64(b_hi + ko), idesc, first);
              umma_bf16(tmem_d, make_desc_sw64(a_hi + ko), make_desc_sw64(b_lo + ko), idesc, 1u);
              umma_bf16(tmem_d, make_desc_sw64(a_hi + ko), make_desc_sw64(b_hi + ko), idesc, 1u);
            }
          }
          // the stage is free once these MMAs have read it (the empty barrier counts one arrival per warp)
          umma_commit(&ring.empty[ring.stage()]);  // warp 0's arrival; the other warps give theirs below
          ring.advance();
        }
      }
      umma_commit(c.acc_bar);
      prof_mark(c, 36);
    } else if (lane == 0) {
      // lane 0 of warps 1-7: this warp's arrival on every stage, given once the chunk has landed
      for (int i = 0; i < nchunks; i++) {
        mbar_wait_relaxed(&ring.full[ring.stage()], ring.parity());
        mbar_arrive(&ring.empty[ring.stage()]);
        ring.advance();
      }
    } else {
      ring.advance_by(nchunks);
    }
    __syncwarp();  // other lanes park here instead of polling beside the issuing thread
    // ---- epilogue: TMEM -> registers, logits dump (optional), per-utterance argmax ----
    mbar_wait_relaxed(c.acc_bar, (uint32_t)(c.acc_phase & 1));
    c.acc_phase++;
    __syncwarp();
    prof_mark(c, 37);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int mt_w = warp >> 2;                      // warps 0-3: m-tile 0, warps 4-7: m-tile 1
    const int vrow = mt_w * 128 + (warp & 3) * 32 + lane;
    const int v = item * VC + vrow;
    const bool vok = (mt_w < n_mt) && (vrow < VC) && (v < V);
    for (int cb = 0; cb < nx; cb += 16) {
      uint32_t r[16];
      if (mt_w < n_mt) {  // warp-uniform
        const uint32_t taddr = c.tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(mt_w * nx + cb);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
              "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
            : "r"(taddr)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      }
#pragma unroll
      for (int e = 0; e < 16; e++) {
        const int b = cb + e;
        const float val = __uint_as_float(r[e]);
        if (vok && p.logits_out && b < nb) p.logits_out[(int64_t)(b0 + b) * V + v] = val;
        // order-preserving float -> uint key (NaN and masked rows -> 0, never win); one redux gives the
        // warp max, the lowest lane holding it is the first (smallest) vocab index
        uint32_t key = r[e];
        key = (key & 0x80000000u) ? ~key : (key | 0x80000000u);
        if (!vok || val != val) key = 0u;
        const uint32_t mx = __reduce_max_sync(0xffffffffu, key);
        const uint32_t who = __ballot_sync(0xffffffffu, key == mx);
        if (lane == 0) {
          c.argv[warp * 64 + b] = __uint_as_float(mx);
          c.argi[warp * 64 + b] = mx ? item * VC + mt_w * 128 + (warp & 3) * 32 + (__ffs(who) - 1) : 0x7fffffff;
        }
      }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    csync();
    prof_mark(c, 38);
    if (threadIdx.x < nb) {
      const int b = threadIdx.x;
      uint32_t bk = 0u;
      int bi = 0x7fffffff;
      for (int w2 = 0; w2 < kWarpsC; w2++) {
        const uint32_t ok = __float_as_uint(c.argv[w2 * 64 + b]);
        const int oi = c.argi[w2 * 64 + b];
        if (ok > bk || (ok == bk && oi < bi)) { bk = ok; bi = oi; }
      }
      // key -> float (0 = no candidate)
      const float bv = bk == 0u ? -INFINITY : __uint_as_float((bk & 0x80000000u) ? (bk & 0x7fffffffu) : ~bk);
      p.cand_val[((int64_t)parity * p.n_vchunk + item) * p.B + b0 + b] = bv;
      p.cand_idx[((int64_t)parity * p.n_vchunk + item) * p.B + b0 + b] = bi;
    }
    csync();
  }
}

template <int NB, int NBM>
__global__ void __launch_bounds__(kThreads2, 1)
decoder_step2_kernel(const __grid_constant__ DecoderParams p) {
  if (*p.n_active == 0) return;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  constexpr int NBmax = NB > NBM ? NB : NBM;
  const SmemLayout2 L = smem_layout2(NBmax, p.B, p.D, p.hd, p.IC, p.Tpad, p.Smax, p.smem_limit);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + L.bars);
  unsigned char* active = smem_raw + L.active;
  Ring ring;
  ring.full = bars;
  ring.empty = bars + 16;
  ring.data = reinterpret_cast<char*>(smem_raw + L.ring);
  ring.ns = L.ns;
  ring.reset((threadIdx.x - kConsumers) >> 5);  // `who` is meaningful for the producer lanes only

  // snapshot of the done flags: the work list of this launch
  for (int b = threadIdx.x; b < p.B; b += kThreads2) active[b] = p.done[b] ? 0 : 1;
  uint32_t& tmem_base_smem = *reinterpret_cast<uint32_t*>(bars + 33);
  if (threadIdx.x == 0) {
    for (int i = 0; i < L.ns; i++) {
      mbar_init(&ring.full[i], 1);
      mbar_init(&ring.empty[i], kWarpsC);
    }
    mbar_init(bars + 32, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x < 32) {  // warp 0 owns the TMEM allocation (256 columns: logits 2 m-tiles x <= 64 utterances; GEMVs 3 x 16 per m-tile)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)),
                 "r"(256)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_smem;

  const unsigned G = gridDim.x;
  const int n_bt = (p.B + NB - 1) / NB;
  const int n_btm = (p.B + NBM - 1) / NBM;

  if (threadIdx.x >= kConsumers) {
    // ======================= producer warps (one lane each) =======================
    if ((threadIdx.x & 31) == 0) {
      for (int l = 0; l < p.L; l++) {
        for (int it = blockIdx.x; it < n_bt * p.H; it += G) produce_self(p, l, it, NB, ring, active);
        for (int it = blockIdx.x; it < n_bt * p.H; it += G) produce_cross(p, l, it, NB, ring, active);
        for (int it = blockIdx.x; it < n_btm * p.n_chunk; it += G) produce_mlp(p, l, it, NBM, ring, active);
      }
      const int nx = logits_rows_per_pass(p.B, p.D, L.xg_bytes);
      for (int it = blockIdx.x; it < p.n_vchunk; it += G) produce_logits(p, it, ring, nx);
    }
    return;
  }

  // ========================= consumers =========================
  Ctx c;
  c.hs = reinterpret_cast<float*>(smem_raw + L.hs);
  c.xs = reinterpret_cast<float*>(smem_raw + L.xs);
  c.act = reinterpret_cast<float*>(smem_raw + L.act);
  c.att = reinterpret_cast<float*>(smem_raw + L.att);
  c.red = reinterpret_cast<float*>(smem_raw + L.red);
  c.ps = reinterpret_cast<float*>(smem_raw + L.ps);
  c.sc = reinterpret_cast<float*>(smem_raw + L.sc);
  c.flags = reinterpret_cast<int*>(smem_raw + L.flags);
  c.argv = reinterpret_cast<float*>(smem_raw + L.argv);
  c.argi = reinterpret_cast<int*>(smem_raw + L.argi);
  c.active = active;
  c.actw = L.actw;
  c.attw = L.attw;
  {
    float* rope = reinterpret_cast<float*>(smem_raw + L.rope);
    const int half_rot = p.rot_dim >> 1;  // <= 64
    for (int i = threadIdx.x; i < half_rot; i += kConsumers) {
      rope[i] = p.rope_cos[(int64_t)p.step * half_rot + i];
      rope[64 + i] = p.rope_sin[(int64_t)p.step * half_rot + i];
    }
    c.rope = rope;
    c.bias = reinterpret_cast<float*>(smem_raw + L.bias);
    c.xg = reinterpret_cast<float*>(smem_raw);
    c.nx = logits_rows_per_pass(p.B, p.D, L.xg_bytes);
    c.tmem = tmem_base;
    c.xp = smem_raw + L.xp;
    c.acc_bar = bars + 32;
    c.acc_phase = 0;
  }
  c.prof = reinterpret_cast<unsigned long long*>(p.prof);
  c.prof_n = 0;
  prof_mark(c, 0);

  unsigned nbar = p.barrier[1];
  const int64_t BD = (int64_t)p.B * p.D;
  float* partA = p.part;
  float* partB = p.part + (int64_t)p.H * BD;
  float* partC = p.part + (int64_t)2 * p.H * BD;
  int ph = 0;
  for (int l = 0; l < p.L; l++) {
    {
      const float* hrd = p.hbuf + (int64_t)(ph & 1) * BD;
      float* hwr = p.hbuf + (int64_t)((ph + 1) & 1) * BD;
      for (int it = blockIdx.x; it < n_bt * p.H; it += G)
        phase_self<NB>(p, l, it, c, ring, hrd, hwr, partC, partA);
      prof_mark(c, 7);
      grid_barrier(p.barrier, (++nbar) * G);
      prof_mark(c, 8);
      ph++;
    }
    {
      const float* hrd = p.hbuf + (int64_t)(ph & 1) * BD;
      float* hwr = p.hbuf + (int64_t)((ph + 1) & 1) * BD;
      for (int it = blockIdx.x; it < n_bt * p.H; it += G)
        phase_cross<NB>(p, l, it, c, ring, hrd, hwr, partA, partB);
      prof_mark(c, 17);
      grid_barrier(p.barrier, (++nbar) * G);
      prof_mark(c, 18);
      ph++;
    }
    {
      const float* hrd = p.hbuf + (int64_t)(ph & 1) * BD;
      float* hwr = p.hbuf + (int64_t)((ph + 1) & 1) * BD;
      for (int it = blockIdx.x; it < n_btm * p.n_chunk; it += G)
        phase_mlp<NBM>(p, l, it, c, ring, hrd, hwr, partB, partC);
      prof_mark(c, 27);
      grid_barrier(p.barrier, (++nbar) * G);
      prof_mark(c, 28);
      ph++;
    }
  }
  {
    const float* hrd = p.hbuf + (int64_t)(ph & 1) * BD;
    for (int it = blockIdx.x; it < p.B; it += G) phase_final_ln<1>(p, it, c, hrd, partC);
    prof_mark(c, 31);
    grid_barrier(p.barrier, (++nbar) * G);
    prof_mark(c, 32);
  }
  for (int it = blockIdx.x; it < p.n_vchunk; it += G) phase_logits(p, it, c, ring);
  prof_mark(c, 33);
  grid_barrier(p.barrier, (++nbar) * G);
  prof_mark(c, 34);
  if (blockIdx.x == 0) {
    int* cnt = c.flags;
    if (threadIdx.x == 0) *cnt = 0;
    csync();
    int n = 0;
    for (int b = threadIdx.x; b < p.B; b += kConsumers) n += p.done[b] ? 0 : 1;
    if (n) atomicAdd(cnt, n);
    csync();
    if (threadIdx.x == 0) {
      *p.n_active = *cnt;
      p.barrier[1] = nbar;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  csync();
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256) : "memory");
  }
}

template <int NB, int NBM>
void launch_variant2(const DecoderParams& p, int grid, size_t smem, cudaStream_t stream) {
  auto kern = decoder_step2_kernel<NB, NBM>;
  static SmemAttrCache cache;  // one per template instantiation
  if (cache.needs(smem)) CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  void* args[] = {const_cast<DecoderParams*>(&p)};
  CUDA_CHECK(cudaLaunchCooperativeKernel((void*)kern, dim3(grid), dim3(kThreads2), args, smem, stream));
}

}  // namespace

size_t decoder_step2_smem_bytes(const DecoderParams& p) {
  int nb, nbm;
  decoder_tiles_for_batch(p.B, nb, nbm);
  const SmemLayout2 L = smem_layout2(nb > nbm ? nb : nbm, p.B, p.D, p.hd, p.IC, p.Tpad, p.Smax, p.smem_limit);
  if (L.ns < 2) throw std::runtime_error("decoder v2: not enough shared memory for the operand ring");
  return (size_t)L.total;
}

void launch_decoder_step2(const DecoderParams& p, int grid, cudaStream_t stream) {
  int nb, nbm;
  decoder_tiles_for_batch(p.B, nb, nbm);
  const size_t smem = decoder_step2_smem_bytes(p);
  if (nb == 1 && nbm == 1) launch_variant2<1, 1>(p, grid, smem, stream);
  else if (nb == 1) launch_variant2<1, 2>(p, grid, smem, stream);
  else if (nb == 2) launch_variant2<2, 4>(p, grid, smem, stream);
  else if (nb == 4) launch_variant2<4, 8>(p, grid, smem, stream);
  else if (nb == 8) launch_variant2<8, 16>(p, grid, smem, stream);
  else launch_variant2<16, 16>(p, grid, smem, stream);
}

}  // namespace msb
