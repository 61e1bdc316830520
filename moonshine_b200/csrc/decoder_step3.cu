// Persistent decoder-step kernel, v3: weight-stationary tensor-core jobs + dataflow counters.
//
// One launch = one greedy token for the whole batch (reference loop: core/moonshine-model.cpp:380-517,
// core/moonshine-streaming-model.cpp:867-1082).  The step is a static program of PHASES, each a list of JOBS that
// are dealt to the 148 persistent CTAs by a fixed rule (job j of a phase runs on CTA (first + j % ncta) % grid):
//
//   per layer   SELF   (head h, tile of nb_self utterances): resolve the previous block's partial sums + LayerNorm
//                      -> q|k|v of head h on tcgen05 -> RoPE, K/V append, causal self-attention (one warp per
//                      utterance) -> per-head partial output projection
//               CROSS  (head h, tile of nb_cross utterances): resolve the 8 head partials + LayerNorm -> cross q of
//                      head h on tcgen05 -> attention over the fp16 cross K/V -> attc[b][h*hd ..]
//               OC     (128 output features, group of nx utterances): attc . Woc^T        on tcgen05
//               FC1    (128 interleaved value|gate rows, group): LN(h + OC) . W1^T, SiLU gate in the TMEM epilogue
//               FC2    (128 output features, k-slice, group): act . W2^T partials         on tcgen05
//   once        FINAL  (8 utterances): last residual + final LayerNorm rows
//               LOGITS (vocab chunk): tied head on tcgen05 + argmax in the TMEM epilogue
//
// Every dense contraction has the UTTERANCES as the MMA N operand (16 ... 64 columns) and 128 weight rows as M, so
// each weight byte crosses L2 -> SM once per group of utterances instead of once per pair of utterances (v2), and
// the weights arrive as pre-split bf16 hi/lo planes in UMMA K-major SWIZZLE_64B order through the same TMA
// bulk-copy ring as before (two producer warps that never wait for anything but ring space, so they run ahead of
// the dependency chain -- a GEMM CTA has its next weight tile in shared memory before its inputs exist).
//
// There is no grid-wide barrier: a phase's jobs wait until the completion counter of the previous phase reaches
// its job count (one ld.acquire poll by one thread), and signal their own counter with one release-add.  CTAs
// without a job in a phase walk straight on to the wait of their next job.  Counters grow monotonically over the
// launches of one decode (target = (epoch + 1) * jobs); the epoch lives in device memory and is advanced by CTA 0
// once the last phase is complete.  A wait that exceeds ~2 s raises an error flag in device memory and every wait
// in the grid falls through, so a logic error ends as a clean host-side exception, not as a hung context.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.h"
#include "kernels.h"

namespace msb {

namespace {

constexpr int kConsumers = 256;
constexpr int kProducers = 2;
constexpr int kThreads3 = kConsumers + 32 * kProducers;
constexpr int kWarpsC = kConsumers / 32;
constexpr int kStageBytes = 32768;
constexpr int kMaxNB = 16;                       // utterances per attention job (one N = 16 MMA operand)
constexpr int kMaxPairs = 8;                     // float2 per lane of a LayerNorm row: D <= 512
constexpr long long kSpinLimit = 4000000000LL;   // ~2 s of SM cycles
constexpr int kPlaneBatch = 6;                   // (row, 8-input) items a thread keeps in flight in planes_from_rows
constexpr int kBiasEntries = 512;                // per-utterance bias entries that may fall into one vocab chunk per pass

enum { PH_SELF = 0, PH_CROSS, PH_OC, PH_FC1, PH_FC2, PH_FINAL, PH_LOGITS, PH_KINDS };
constexpr int kPhasesPerLayer = 5;

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
// Data another CTA produced during this launch.  The consumer's dependency wait is an ld.acquire.gpu poll, which
// ptxas turns into LDG.STRONG.GPU + CCTL.IVALL: the SM's L1 holds nothing stale once the wait is over, so these are
// ordinary (weak, L1-allocating) loads the compiler may batch freely.  (ld.global.cg would compile to ORDERED
// LDG.STRONG.GPU loads: measured 2.4-2.9 us for one row's 10-30 loads.)
template <typename T>
__device__ __forceinline__ T ld_fresh(const T* p) { return *p; }
__device__ __forceinline__ bool poisoned(const unsigned* err) { return *reinterpret_cast<const volatile unsigned*>(err) != 0u; }

// ---- mbarrier / bulk-copy primitives (PTX) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
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
// A wait that runs out of patience poisons the grid (error flag) instead of trapping the context.  Only the first try is
// inlined: the kernel is several times the 128 KB instruction cache, and every inlined spin loop made that worse.
__device__ __noinline__ void mbar_wait_slow(uint32_t a, uint32_t parity, unsigned* err, int nap) {
  const long long t0 = clock64();
  unsigned polls = 0;
  while (!mbar_try(a, parity)) {
    if (nap) __nanosleep(32);
    if ((++polls & 15u) == 0u) {
      if (poisoned(err)) return;
      if (clock64() - t0 > kSpinLimit) { atomicExch(err, 1u); return; }
    }
  }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, unsigned* err) {
  const uint32_t a = smem_u32(bar);
  if (mbar_try(a, parity)) return;
  mbar_wait_slow(a, parity, err, 0);
}
// Same wait for threads that are NOT on the critical path: back off between polls.
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity, unsigned* err) {
  const uint32_t a = smem_u32(bar);
  if (mbar_try(a, parity)) return;
  mbar_wait_slow(a, parity, err, 1);
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

__device__ __forceinline__ void bulk_g2s_hint(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void l2_prefetch(const void* src, uint32_t bytes) {  // bytes: multiple of 16
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
// ---- tcgen05 helpers ----
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
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// One lane of a converged warp.  tcgen05.mma takes its operands from UNIFORM registers: issued under elect.sync
// inside warp-uniform control flow, with operands the compiler can prove uniform (shuffle broadcasts), it is a
// handful of instructions; issued from a divergent `if (threadIdx.x == 0)` the compiler wraps EVERY MMA in a
// waterfall loop (ELECT / 5x R2UR.BROADCAST / BRA.U.ANY), measured ~95 ns per MMA on B200.
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
__device__ __forceinline__ uint32_t idesc_bf16(int n) {  // D fp32, A/B bf16 K-major, M = 128, N = n
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
// (a, b) -> packed bf16 pairs: hi = round-to-nearest bf16, lo = bf16 of the remainder (a in the low half)
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 ah = __float2bfloat16_rn(a), bh = __float2bfloat16_rn(b);
  const __nv_bfloat16 al = __float2bfloat16_rn(a - __bfloat162float(ah));
  const __nv_bfloat16 bl = __float2bfloat16_rn(b - __bfloat162float(bh));
  hi = (uint32_t)__bfloat16_as_ushort(ah) | ((uint32_t)__bfloat16_as_ushort(bh) << 16);
  lo = (uint32_t)__bfloat16_as_ushort(al) | ((uint32_t)__bfloat16_as_ushort(bl) << 16);
}

// ---- the operand ring (TMA bulk copies, 32 KB stages) ----
struct Ring {
  uint64_t* full;
  uint64_t* empty;
  char* data;
  unsigned* err;
  int ns;
  int st;        // stage of the next chunk
  uint32_t par;  // parity of the pass over the ring the next chunk belongs to
  int turn;      // producers: chunks until this lane's next turn (0 = issue this one)
  __device__ __forceinline__ void reset(int who) { st = 0; par = 0; turn = who; }
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
    mbar_wait(&full[st], par, err);
    return data + (size_t)st * kStageBytes;
  }
  // every consumer WARP releases the stage once its lanes are done reading it (empty barriers count kWarpsC arrivals)
  __device__ __forceinline__ void release() {
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(&empty[st]);
    advance();
  }
  // producers (one lane per producer warp; every producer walks the whole sequence and issues its share)
  __device__ __forceinline__ void produce(const void* src, uint32_t bytes, uint64_t policy = 0) {
    if (turn == 0) {
      mbar_wait(&empty[st], par ^ 1u, err);
      mbar_expect_tx(&full[st], bytes);
      if (policy) bulk_g2s_hint(data + (size_t)st * kStageBytes, src, bytes, &full[st], policy);
      else bulk_g2s(data + (size_t)st * kStageBytes, src, bytes, &full[st]);
      turn = kProducers;
    }
    turn--;
    advance();
  }
};

__device__ __forceinline__ int rows_per_chunk_f32(int K, int N) {
  int r = kStageBytes / (N * 4);
  return r < 1 ? 1 : (r > K ? K : r);
}
__device__ __forceinline__ int rows_per_chunk_f16(int rows, int cols) {
  int r = (kStageBytes / (cols * 2)) & ~1;
  if (r < 2) r = 2;
  return r > rows ? rows : r;
}
// plane-packed [N][K] blocks: m-tiles of <= 128 rows (padded to 8), k-blocks of 32, [hi | lo] per k-block
__host__ __device__ __forceinline__ int plane_rows(int N, int mt) {
  const int r = N - mt * 128;
  return ((r < 128 ? r : 128) + 7) & ~7;
}
// k-blocks per ring chunk: an M = 128 MMA reads 128 rows of the plane it is pointed at even when the tile has
// fewer, so the LAST plane of a chunk must still end inside the stage.
__host__ __device__ __forceinline__ int plane_kb_per_chunk(int Rp) {
  const int n = (kStageBytes - 128 * 64 - Rp * 64) / (Rp * 128) + 1;
  return n < 1 ? 1 : n;
}
__host__ __device__ __forceinline__ size_t plane_block_bytes(int N, int K) {
  const int nkb = (K + 31) >> 5, n_mt = (N + 127) >> 7;
  size_t rows = 0;
  for (int mt = 0; mt < n_mt; mt++) rows += (size_t)plane_rows(N, mt);
  return rows * nkb * 128;
}
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
__device__ __forceinline__ void produce_block_f32(Ring& ring, const float* Wt, int K, int N) {
  const int rpc = rows_per_chunk_f32(K, N);
  for (int k0 = 0; k0 < K; k0 += rpc) {
    const int rows = min(rpc, K - k0);
    ring.produce(Wt + (size_t)k0 * N, (uint32_t)rows * N * 4);
  }
}
__device__ __forceinline__ void produce_block_f16(Ring& ring, const __half* M, int rows, int cols, uint64_t policy = 0) {
  const int rpc = rows_per_chunk_f16(rows, cols);
  for (int r0 = 0; r0 < rows; r0 += rpc) {
    const int n = min(rpc, rows - r0);
    ring.produce(M + (size_t)r0 * cols, (uint32_t)n * cols * 2, policy);
  }
}

// ---- shared memory layout ----
struct SmemLayout3 {
  int bars, active, flags, rope, argv, argi, sbias, rowflag, ent_key, ent_val, ent_n, scratch, ring;  // byte offsets
  int xp, act, att, sc, ps, red;                             // attention-job scratch (inside `scratch`)
  int actw, attw, nxl, ns, total;
};
__host__ __device__ inline int logits_rows_for(int B, int D) {
  int nx = (B + 15) & ~15;
  if (nx > 64) nx = 64;
  while (nx > 16 && nx * D * 4 > 80 * 1024) nx -= 16;
  return nx;
}
__host__ __device__ inline SmemLayout3 smem_layout3(int B, int D, int hd, int Kc, int nx, int Tpad, int Smax, int smem_limit) {
  SmemLayout3 L;
  int o = 0;
  auto take = [&](int bytes) { int r = o; o += (bytes + 15) / 16 * 16; return r; };
  L.bars = take((2 * 16 + 2) * 8);  // ring full / empty, accumulator barrier, TMEM base
  L.active = take(B);
  L.flags = take(64 * 4);
  L.rope = take(128 * 4);
  L.argv = take(kWarpsC * 64 * 4);
  L.argi = take(kWarpsC * 64 * 4);
  L.sbias = take(384 * 4);            // logit bias: static bonuses of this CTA's vocab chunk (<= 3 m-tiles),
  L.rowflag = take(384);              // rows with a per-utterance entry,
  L.ent_key = take(kBiasEntries * 4); // (row << 8 | utterance column) of each entry that falls into the chunk,
  L.ent_val = take(kBiasEntries * 4); // its bonus,
  L.ent_n = take(16);                 // and their count
  o = (o + 1023) / 1024 * 1024;
  L.scratch = o;
  L.actw = 3 * hd;
  L.attw = hd;
  // attention jobs
  L.xp = take(((D + 31) / 32) * 2048);  // x planes of a 16-utterance tile: [kb][hi 16 x 64 B | lo 16 x 64 B]
  L.act = take(kMaxNB * L.actw * 4);
  L.att = take(kMaxNB * L.attw * 4);
  L.sc = take(kWarpsC * (Smax + 4) * 4);
  L.ps = take(2 * Tpad * 4);
  L.red = take((32 + 1024) * 4);
  const int attn_end = o;
  // GEMM jobs and the logits phase alias the same region with their x planes (nx utterances x K x (hi + lo))
  const int kmax = ((D > Kc ? D : Kc) + 31) / 32 * 32;
  L.nxl = logits_rows_for(B, D);
  int xg = nx * kmax * 4;
  if (L.nxl * D * 4 > xg) xg = L.nxl * D * 4;
  if (L.scratch + xg > attn_end) o = L.scratch + xg;
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
  unsigned* err;
  const float* rope;         // smem: cos[0..64) | sin[64..128) of this step's position
  unsigned char* xp;         // smem: x planes of an attention job (16 rows)
  unsigned char* xg;         // smem: x planes of a GEMM job / logits pass (aliases the attention scratch)
  uint32_t tmem;             // TMEM base (256 columns)
  uint64_t* acc_bar;         // accumulator-ready mbarrier
  int acc_phase;
  unsigned long long* prof;  // optional [grid][kProfSlots] stamps (thread 0)
  int prof_n;
  float *act, *att, *red, *ps, *sc, *argv;
  int *flags, *argi;
  float *sbias, *ent_val;       // logit bias tables (logits phase)
  unsigned char* rowflag;
  int *ent_key, *ent_n;
  const unsigned char* active;  // [B] 1 = utterance still decoding at kernel start
  int actw, attw;
};

__device__ __forceinline__ void prof_mark(Ctx& c, int tag) {
  if (c.prof != nullptr && threadIdx.x == 0 && c.prof_n < kProfSlots) {
    const unsigned long long t = (unsigned long long)((double)clock64() * (1.0 / 1.965));
    c.prof[(size_t)blockIdx.x * kProfSlots + c.prof_n] = (t << 8) | (unsigned)tag;
    c.prof_n++;
  }
}

// byte offset of bf16 element (row r, input k) inside the hi plane of an activation tile of NXp rows
__device__ __forceinline__ uint32_t plane_off(int NXp, int r, int k) {
  return (uint32_t)((k >> 5) * NXp * 128 + r * 64 + ((((k >> 3) & 3) ^ ((r >> 1) & 3)) << 4) + (k & 7) * 2);
}

// ------------------------------------------------------------------------------------------------
// Row prologue, ONE WARP PER ROW: v = h + sum_j part_j (+ bias), optional store of the new residual row,
// LayerNorm without affine (gamma lives in the next weight block), result handed out as (k, x_k, x_k+1) pairs.
// Every input was written by other CTAs during this launch: read through L2 (ld.global.cg).
// ------------------------------------------------------------------------------------------------
struct RowVals {
  float2 v[kMaxPairs];
};
__device__ __forceinline__ void row_resolve(RowVals& rv, int D, const float* hrow, const float* part_row, int64_t pstride,
                                            int nparts, const float* __restrict__ bias) {
  // ld.global.cg compiles to an ORDERED load (LDG.STRONG.GPU) that the compiler never hoists over the adds of the
  // previous array, and one L2 round trip costs ~0.65 us here: stage up to 4 arrays (20-28 loads per lane) in
  // registers before the first add, so a row costs 1-2 round trips instead of one per array.  Sum order unchanged.
  const int lane = threadIdx.x & 31;
  float2 q[4][kMaxPairs];
#pragma unroll
  for (int i = 0; i < kMaxPairs; i++) {
    const int k = 2 * lane + 64 * i;
    rv.v[i] = (k < D) ? ld_fresh(reinterpret_cast<const float2*>(hrow + k)) : make_float2(0.f, 0.f);
  }
  for (int j0 = 0; j0 < nparts; j0 += 4) {
#pragma unroll
    for (int u = 0; u < 4; u++) {
#pragma unroll
      for (int i = 0; i < kMaxPairs; i++) {
        const int k = 2 * lane + 64 * i;
        q[u][i] = (j0 + u < nparts && k < D) ? ld_fresh(reinterpret_cast<const float2*>(part_row + (int64_t)(j0 + u) * pstride + k))
                                             : make_float2(0.f, 0.f);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      if (j0 + u < nparts) {
#pragma unroll
        for (int i = 0; i < kMaxPairs; i++) {
          rv.v[i].x += q[u][i].x;
          rv.v[i].y += q[u][i].y;
        }
      }
    }
  }
  if (bias != nullptr) {
#pragma unroll
    for (int i = 0; i < kMaxPairs; i++) {
      const int k = 2 * lane + 64 * i;
      if (k < D) {
        const float2 b2 = __ldg(reinterpret_cast<const float2*>(bias + k));
        rv.v[i].x += b2.x;
        rv.v[i].y += b2.y;
      }
    }
  }
}
__device__ __forceinline__ void row_store(const RowVals& rv, int D, float* dst) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < kMaxPairs; i++) {
    const int k = 2 * lane + 64 * i;
    if (k < D) *reinterpret_cast<float2*>(dst + k) = rv.v[i];
  }
}
__device__ __forceinline__ void row_layernorm(RowVals& rv, int D) {
  const int lane = threadIdx.x & 31;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxPairs; i++)
    if (2 * lane + 64 * i < D) s += rv.v[i].x + rv.v[i].y;
  const float mean = warp_sum(s) / D;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxPairs; i++)
    if (2 * lane + 64 * i < D) {
      const float dx = rv.v[i].x - mean, dy = rv.v[i].y - mean;
      q += dx * dx + dy * dy;
    }
  const float rstd = rsqrtf(warp_sum(q) / D + 1e-5f);
#pragma unroll
  for (int i = 0; i < kMaxPairs; i++) {
    rv.v[i].x = (rv.v[i].x - mean) * rstd;
    rv.v[i].y = (rv.v[i].y - mean) * rstd;
  }
}
// row r of an activation tile (NXp rows) <- bf16 hi / lo planes of the row values (zero row when !valid)
__device__ __forceinline__ void row_to_planes(const RowVals& rv, int D, unsigned char* planes, int NXp, int r, bool valid) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < kMaxPairs; i++) {
    const int k = 2 * lane + 64 * i;
    if (k < D) {
      uint32_t hi = 0u, lo = 0u;
      if (valid) split_bf16x2(rv.v[i].x, rv.v[i].y, hi, lo);
      unsigned char* at = planes + plane_off(NXp, r, k);
      *reinterpret_cast<uint32_t*>(at) = hi;
      *reinterpret_cast<uint32_t*>(at + NXp * 64) = lo;
    }
  }
}

// Activation tile from a plain fp32 matrix: rows [g0, g0 + nb) x columns [k0, k0 + K) of src (row stride ld) ->
// planes of NXp rows (rows >= nb and inactive rows are zero).  Item = (row, 8 inputs); loads batched 6 deep (one L2
// round trip for a 32 x 288 tile).
__device__ __forceinline__ void planes_from_rows(unsigned char* planes, int NXp, const float* src, int64_t ld, int g0, int nb,
                                                 int k0, int K, const unsigned char* active) {
  const int k8n = (K + 31) / 32 * 4;  // 8-wide chunks per row, whole k-blocks
  const int nitems = NXp * k8n;
  for (int i0 = threadIdx.x; i0 < nitems; i0 += kPlaneBatch * kConsumers) {
    float4 va[kPlaneBatch], vb[kPlaneBatch];
#pragma unroll
    for (int u = 0; u < kPlaneBatch; u++) {
      const int i = i0 + u * kConsumers;
      const int r = i / k8n, k8 = i - r * k8n;
      va[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      vb[u] = va[u];
      if (i < nitems && r < nb && active[g0 + r]) {
        const float* s = src + (int64_t)(g0 + r) * ld + k0 + k8 * 8;
        if (k8 * 8 < K) va[u] = ld_fresh(reinterpret_cast<const float4*>(s));
        if (k8 * 8 + 4 < K) vb[u] = ld_fresh(reinterpret_cast<const float4*>(s + 4));
      }
    }
#pragma unroll
    for (int u = 0; u < kPlaneBatch; u++) {
      const int i = i0 + u * kConsumers;
      if (i >= nitems) break;
      const int r = i / k8n, k8 = i - r * k8n;
      uint4 hi, lo;
      split_bf16x2(va[u].x, va[u].y, hi.x, lo.x);
      split_bf16x2(va[u].z, va[u].w, hi.y, lo.y);
      split_bf16x2(vb[u].x, vb[u].y, hi.z, lo.z);
      split_bf16x2(vb[u].z, vb[u].w, hi.w, lo.w);
      unsigned char* at = planes + plane_off(NXp, r, k8 * 8);
      *reinterpret_cast<uint4*>(at) = hi;
      *reinterpret_cast<uint4*>(at + NXp * 64) = lo;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Tensor-core block:  out[n][b] = sum_k W[n][k] * x[b][k]   for a plane-packed weight block of N rows (<= 256).
// A chunks come through the ring, the x planes (NXp rows, K inputs) lie in shared memory.  One thread issues
// 3 split products per k16 step into three accumulators (independent chains; summed in the epilogue);
// tcgen05.commit hands each ring stage back.  Epilogue: f(n, cb, v[16]) with v = the 16 utterance columns
// cb .. cb+15 of output row n.  Called by all 256 consumer threads.
// ------------------------------------------------------------------------------------------------
template <typename F>
__device__ __forceinline__ void gemm_block(Ring& ring, Ctx& c, const unsigned char* xplanes, int NXp, int K, int N, F f) {
  const int nkb = (K + 31) >> 5, n_mt = (N + 127) >> 7;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // x planes (generic-proxy stores) -> tensor core
  csync();
  prof_mark(c, 63);
  // Two MMAs per k16 step instead of three: the hi and lo planes of the x tile lie back to back ([hi NXp rows |
  // lo NXp rows], same 64-byte row pitch), so ONE instruction with N = 2 NXp multiplies the weight's hi plane with
  // both -- columns [0, NXp) = hi.hi, [NXp, 2 NXp) = hi.lo -- and a second with N = NXp adds lo.hi in columns
  // [2 NXp, 3 NXp).  A small tcgen05.mma costs ~43 ns whatever N is, so this is a third off the GEMV.
  const uint32_t idesc = idesc_bf16(NXp), idesc2 = idesc_bf16(2 * NXp);
  const int warp_u = (int)uniform_u32((uint32_t)warp);
  if (warp_u == 0) {
    // the whole of warp 0 walks the chunk list in lock step; one elected lane issues the MMAs and the commits
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t xb = uniform_u32(smem_u32(xplanes));
    const uint32_t tm = uniform_u32(c.tmem);
    for (int mt = 0; mt < n_mt; mt++) {
      const int Rp = plane_rows(N, mt), kbc = plane_kb_per_chunk(Rp);
      const uint32_t tmem_d = tm + (uint32_t)(mt * 3 * NXp);
      for (int kb0 = 0; kb0 < nkb; kb0 += kbc) {
        const int n = min(kbc, nkb - kb0);
        mbar_wait(&ring.full[ring.stage()], ring.parity(), c.err);
        __syncwarp();
        if (kb0 == 0 && mt == 0) prof_mark(c, 74);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t a_base = uniform_u32(smem_u32(ring.data + (size_t)ring.stage() * kStageBytes));
        const uint32_t empty_bar = uniform_u32(smem_u32(&ring.empty[ring.stage()]));
        if (elect_one()) {
          // not unrolled: the kernel's code already overflows the instruction cache (DESIGN.md 4.2)
#pragma unroll 1
          for (int q = 0; q < n; q++) {
            const int kb = kb0 + q;
            const uint32_t a_hi = a_base + (uint32_t)(q * Rp * 128), a_lo = a_hi + (uint32_t)(Rp * 64);
            const uint32_t b_hi = xb + (uint32_t)(kb * NXp * 128);
#pragma unroll
            for (int ks = 0; ks < 2; ks++) {
              if (kb * 32 + ks * 16 >= K) break;  // nothing but zero padding beyond K
              const uint32_t ko = (uint32_t)ks * 32u;
              const uint32_t acc = (kb | ks) ? 1u : 0u;
              umma_bf16(tmem_d, make_desc_sw64(a_hi + ko), make_desc_sw64(b_hi + ko), idesc2, acc);
              umma_bf16(tmem_d + 2 * NXp, make_desc_sw64(a_lo + ko), make_desc_sw64(b_hi + ko), idesc, acc);
            }
          }
          // warp 0's arrival on the stage: it is free once the MMAs have read it
          asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(empty_bar) : "memory");
        }
        __syncwarp();
        ring.advance();
      }
    }
    if (elect_one()) umma_commit(c.acc_bar);
    __syncwarp();
    prof_mark(c, 64);
  } else {
    // the empty barriers count one arrival per consumer warp: lane 0 of warps 1-7 gives its own as soon as the
    // chunk has landed (waiting for `full` keeps an arrival from slipping into the stage's previous round)
    int total = 0;
    for (int mt = 0; mt < n_mt; mt++) {
      const int kbc = plane_kb_per_chunk(plane_rows(N, mt));
      total += (nkb + kbc - 1) / kbc;
    }
    if (lane == 0) {
      for (int i = 0; i < total; i++) {
        mbar_wait_relaxed(&ring.full[ring.stage()], ring.parity(), c.err);
        mbar_arrive(&ring.empty[ring.stage()]);
        ring.advance();
      }
    } else {
      ring.advance_by(total);
    }
  }
  __syncwarp();  // lanes 1..31 park here instead of polling beside their lane 0
  mbar_wait_relaxed(c.acc_bar, (uint32_t)(c.acc_phase & 1), c.err);
  c.acc_phase++;
  __syncwarp();
  prof_mark(c, 65);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const int ncb = NXp >> 4;
  for (int u = warp >> 2; u < n_mt * ncb; u += 2) {  // warps 0-3 take the even (m-tile, column block) units, 4-7 the odd
    const int mt = u / ncb, cb = (u - mt * ncb) * 16;
    uint32_t r[3][16];
#pragma unroll
    for (int pr = 0; pr < 3; pr++) {
      const uint32_t taddr = c.tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(mt * 3 * NXp + pr * NXp + cb);
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
    float v[16];
#pragma unroll
    for (int e = 0; e < 16; e++)  // small cross terms (hi.lo, lo.hi) first, then the hi * hi product
      v[e] = (__uint_as_float(r[1][e]) + __uint_as_float(r[2][e])) + __uint_as_float(r[0][e]);
    f(mt * 128 + (warp & 3) * 32 + lane, cb, v);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  csync();
}

// ------------------------------------------------------------------------------------------------
// token bookkeeping (unchanged rules: start id, EOS, max_len; lowest index wins ties)
// ------------------------------------------------------------------------------------------------
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
// Step prologue of an utterance that was active at kernel start (whole warp).  Records the id emitted by the
// previous step; an utterance that finishes NOW is marked done from the next launch on (done[b] = step + 1, so
// every CTA's snapshot of this launch still counts it active whatever the timing) and still flows through.
__device__ __forceinline__ int step_prologue_warp(const DecoderParams& p, int b, bool writer) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)b * (p.Smax + 1);
  int tok_in;
  bool finished;
  if (p.row_tok) return min(max(__ldg(p.row_tok + b), 0), p.V - 1);  // explicit rows: the host-side plan kernel keeps the books
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
  if (finished && writer && lane == 0) p.done[b] = p.step + 1;
  if (tok_in < 0 || tok_in >= p.V) tok_in = 0;
  return tok_in;
}

// explicit rows (see DecoderParams): position, utterance and in-launch predecessors of row b
__device__ __forceinline__ int row_position(const DecoderParams& p, int b) { return p.row_pos ? __ldg(p.row_pos + b) : p.step; }
__device__ __forceinline__ int row_utterance(const DecoderParams& p, int b) { return p.row_utt ? __ldg(p.row_utt + b) : b; }
__device__ __forceinline__ int row_inlaunch(const DecoderParams& p, int b) { return p.row_nin ? __ldg(p.row_nin + b) : 0; }
__device__ __forceinline__ int cache_utts(const DecoderParams& p) { return p.row_utt ? p.B_utt : p.B; }

__device__ __forceinline__ bool tile_active(const DecoderParams& p, const unsigned char* active, int nb, int b0) {
  bool any = false;
  for (int b = 0; b < nb; b++) any |= (b0 + b < p.B) && active[b0 + b];
  return any;
}
// flags[r] = 1 when row r of the tile carries no live utterance
__device__ __forceinline__ void load_flags(const DecoderParams& p, const Ctx& c, int nb, int b0, bool with_enc_len) {
  if (threadIdx.x < kMaxNB) {
    const int b = b0 + threadIdx.x;
    const bool live = threadIdx.x < nb && b < p.B && c.active[b];
    c.flags[threadIdx.x] = live ? 0 : 1;
    if (with_enc_len) c.flags[32 + threadIdx.x] = live ? p.enc_len[row_utterance(p, b)] : 0;
  }
  csync();
}

// partial-sum areas inside p.part: [0, H) head partials of the self block | [H, H + KS) fc2 k-slices | [H + KS] OC
__device__ __forceinline__ float* part_self(const DecoderParams& p) { return p.part; }
__device__ __forceinline__ float* part_fc2(const DecoderParams& p) { return p.part + (int64_t)p.H * p.B * p.D; }
__device__ __forceinline__ float* part_oc(const DecoderParams& p) { return p.part + (int64_t)(p.H + p.ffn_ksplit) * p.B * p.D; }

// ============================== SELF =================================
__device__ __forceinline__ void produce_self(const DecoderParams& p, int l, int job, Ring& ring, const unsigned char* active) {
  const int H = p.H, hd = p.hd, D = p.D, nb = p.nb_self;
  const int h = job % H, b0 = (job / H) * nb;
  if (!tile_active(p, active, nb, b0)) return;
  const DecLayerWeights& w = p.layers[l];
  produce_block_planes(ring, w.wqkvP + (size_t)h * plane_block_bytes(3 * hd, D), 3 * hd, D);
  // The self K/V prefix is read straight from global by the warp that owns the utterance (a few KB per item,
  // written by earlier launches -- walking it through the CTA-wide ring serialised the 8 warps).  It has left L2
  // since (one step streams more than L2 holds): ask L2 for it now, a phase ahead of its use.
  if (p.step > 0 && ring.turn == 0 && p.row_pos == nullptr) {
    for (int b = 0; b < nb; b++) {
      if (b0 + b >= p.B || !active[b0 + b]) continue;
      const int64_t bh = ((int64_t)l * cache_utts(p) + row_utterance(p, b0 + b)) * H + h;
      const float* kt = p.ks + bh * hd * p.Smax;
      const float* vr = p.vs + bh * p.Smax * hd;
      const uint32_t kbytes = (uint32_t)(hd * p.Smax * 4), vbytes = (uint32_t)((p.step * hd * 4 + 15) & ~15);
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(kt), "r"(kbytes) : "memory");
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(vr), "r"(vbytes) : "memory");
    }
  }
  produce_block_f32(ring, w.wo + (int64_t)h * hd * D, hd, D);
}

// per-head partial output projection: dst[b0 + b][:] = att[b][0:hd] . Wo_h[hd][D] (k-major fp32 rows through the ring);
// thread = (row group g, 4 output features), NJ rows per thread
template <int NJ>
__device__ __forceinline__ void o_partial(const DecoderParams& p, Ctx& c, Ring& ring, int nb, int b0, float* dst) {
  const int D = p.D, hd = p.hd, attw = c.attw;
  const int D4 = D >> 2;
  const int G = kConsumers / D4;
  const int n4 = threadIdx.x % D4, g = threadIdx.x / D4;
  const bool on = g < G;
  float acc[NJ][4];
#pragma unroll
  for (int j = 0; j < NJ; j++) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
  const int rpc = rows_per_chunk_f32(hd, D);
  for (int k0 = 0; k0 < hd; k0 += rpc) {
    const int rows = min(rpc, hd - k0);
    const float4* W = reinterpret_cast<const float4*>(ring.acquire());
    prof_mark(c, 69);
    if (on) {
#pragma unroll 4
      for (int r = 0; r < rows; r++) {
        const float4 w4 = W[r * D4 + n4];
#pragma unroll
        for (int j = 0; j < NJ; j++) {
          const int b = g + j * G;
          const float xv = b < nb ? c.att[b * attw + k0 + r] : 0.f;
          acc[j][0] = fmaf(xv, w4.x, acc[j][0]);
          acc[j][1] = fmaf(xv, w4.y, acc[j][1]);
          acc[j][2] = fmaf(xv, w4.z, acc[j][2]);
          acc[j][3] = fmaf(xv, w4.w, acc[j][3]);
        }
      }
    }
    ring.release();
  }
  if (on) {
#pragma unroll
    for (int j = 0; j < NJ; j++) {
      const int b = g + j * G;
      if (b < nb && !c.flags[b])
        *reinterpret_cast<float4*>(dst + (int64_t)(b0 + b) * D + n4 * 4) = make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
    }
  }
}

__device__ void job_self(const DecoderParams& p, int l, int job, Ctx& c, Ring& ring, const float* hrd, float* hwr) {
  const int D = p.D, hd = p.hd, H = p.H, nb = p.nb_self;
  const int h = job % H;
  const int b0 = (job / H) * nb;
  if (!tile_active(p, c.active, nb, b0)) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int actw = c.actw, attw = c.attw;
  load_flags(p, c, nb, b0, false);
  prof_mark(c, 60);
  // ---- prologue, one warp per row: token / embedding (layer 0) or residual resolve, LayerNorm, x planes ----
  for (int r = warp; r < kMaxNB; r += kWarpsC) {
    RowVals rv;
    const bool live = !c.flags[r];
    if (live) {
      const int b = b0 + r;
      if (l == 0) {
        const int tok = step_prologue_warp(p, b, h == 0);
#pragma unroll
        for (int i = 0; i < kMaxPairs; i++) {
          const int k = 2 * lane + 64 * i;
          rv.v[i] = (k < D) ? __ldg(reinterpret_cast<const float2*>(p.embed + (int64_t)tok * D + k)) : make_float2(0.f, 0.f);
        }
      } else {
        row_resolve(rv, D, hrd + (int64_t)b * D, part_fc2(p) + (int64_t)b * D, (int64_t)p.B * D, p.ffn_ksplit,
                    p.layers[l - 1].b2);
      }
      prof_mark(c, 61);
      if (h == 0) row_store(rv, D, hwr + (int64_t)b * D);
      row_layernorm(rv, D);
      prof_mark(c, 62);
    }
    row_to_planes(rv, D, c.xp, 16, r, live);
  }
  prof_mark(c, 1);
  // ---- q | k | v of head h for the tile ----
  gemm_block(ring, c, c.xp, 16, D, 3 * hd, [&](int n, int cb, const float* v) {
    if (n < 3 * hd) {
#pragma unroll
      for (int e = 0; e < 16; e++) c.act[e * actw + n] = v[e];
    }
  });
  prof_mark(c, 2);
  {  // RoPE (interleaved pairs) on q and k at position `step`
    const int half_rot = p.rot_dim >> 1;
    for (int i = threadIdx.x; i < nb * 2 * half_rot; i += kConsumers) {
      const int b = i / (2 * half_rot);
      const int r = i - b * 2 * half_rot;
      const int which = r / half_rot;
      const int pr = r - which * half_rot;
      float cs = c.rope[pr], sn = c.rope[64 + pr];
      if (p.row_pos && b0 + b < p.B) {  // explicit rows: every row has its own position
        const int64_t at = (int64_t)__ldg(p.row_pos + b0 + b) * half_rot + pr;
        cs = __ldg(p.rope_cos + at);
        sn = __ldg(p.rope_sin + at);
      }
      float* v = c.act + b * actw + which * hd + 2 * pr;
      const float x0 = v[0], x1 = v[1];
      v[0] = x0 * cs - x1 * sn;
      v[1] = x1 * cs + x0 * sn;
    }
  }
  csync();
  for (int i = threadIdx.x; i < nb * hd; i += kConsumers) {  // K/V append at position `step`
    const int b = i / hd, d = i - b * hd;
    if (!c.flags[b]) {
      const int64_t bh = ((int64_t)l * cache_utts(p) + row_utterance(p, b0 + b)) * H + h;
      const int pos = row_position(p, b0 + b);
      p.ks[(bh * hd + d) * p.Smax + pos] = c.act[b * actw + hd + d];
      p.vs[(bh * p.Smax + pos) * hd + d] = c.act[b * actw + 2 * hd + d];
    }
  }
  // causal self-attention: ONE WARP per utterance (round-robin), warp-level syncs only.  The cached prefix
  // (positions < step, written by earlier launches) comes straight from global memory: lane t reads K^T[d][t]
  // (coalesced over t), lane d reads V[t][d] (coalesced over d); position `step` comes from shared memory.
  const float scale = rsqrtf((float)hd);
  {
    float* sc = c.sc + warp * (p.Smax + 4);
    int owner = 0;
    for (int b = 0; b < nb; b++) {
      if (c.flags[b]) continue;  // uniform
      const bool mine = (owner == warp);
      owner = (owner + 1) & (kWarpsC - 1);
      if (!mine) continue;
      const float* q = c.act + b * actw;
      // keys: cached positions [0, base) from global memory (written by earlier launches), then the rows of this launch
      // that precede the row inside its utterance (explicit rows: nin of them, straight from shared memory) and itself
      const int pos = row_position(p, b0 + b), nin = min(row_inlaunch(p, b0 + b), b), base = pos - nin;
      const int64_t bh = ((int64_t)l * cache_utts(p) + row_utterance(p, b0 + b)) * H + h;
      const float* Kt = p.ks + bh * hd * p.Smax;
      const float* Vr = p.vs + bh * p.Smax * hd;
      float mx = -INFINITY;
      // scores: two key positions per lane, 32 head dims per trip = 64 independent loads in flight per lane (the
      // chain is memory-latency bound: the prefix was written by earlier launches and has left L2 since)
      for (int t0 = 0; t0 < base; t0 += 64) {
        const int ta = t0 + lane, tb = t0 + 32 + lane;
        const bool va = ta < base, vb = tb < base;
        float sa = 0.f, sb = 0.f;
#pragma unroll 1
        for (int d0 = 0; d0 < hd; d0 += 32) {  // 64 loads in flight per lane: hd <= 64 is two round trips, not six
          float ka[32], kb[32];
#pragma unroll
          for (int u = 0; u < 32; u++) {
            const bool in = d0 + u < hd;
            ka[u] = (va && in) ? __ldg(Kt + (int64_t)(d0 + u) * p.Smax + ta) : 0.f;
            kb[u] = (vb && in) ? __ldg(Kt + (int64_t)(d0 + u) * p.Smax + tb) : 0.f;
          }
#pragma unroll
          for (int u = 0; u < 32; u++) {
            const float qd = d0 + u < hd ? q[d0 + u] : 0.f;
            sa = fmaf(qd, ka[u], sa);
            sb = fmaf(qd, kb[u], sb);
          }
        }
        if (va) { sa *= scale; sc[ta] = sa; mx = fmaxf(mx, sa); }
        if (vb) { sb *= scale; sc[tb] = sb; mx = fmaxf(mx, sb); }
      }
      for (int j = 0; j <= nin; j++) {
        const float* kj = c.act + (b - nin + j) * actw + hd;
        float s = 0.f;
        for (int d = lane; d < hd; d += 32) s = fmaf(q[d], kj[d], s);
        s = warp_sum(s) * scale;
        if (lane == 0) sc[base + j] = s;
        mx = fmaxf(mx, s);
      }
      mx = warp_max(mx);
      __syncwarp();
      prof_mark(c, 66);
      float sum = 0.f;
      for (int t = lane; t <= pos; t += 32) {
        const float e = expf(sc[t] - mx);
        sc[t] = e;
        sum += e;
      }
      const float inv = 1.0f / warp_sum(sum);
      __syncwarp();
      prof_mark(c, 67);
      float o0 = 0.f, o1 = 0.f;  // lane owns dims d = lane, lane + 32 (hd <= 64)
      {
        const bool has0 = lane < hd, has1 = lane + 32 < hd;
        int t = 0;
#pragma unroll 1
        for (; t + 16 <= base; t += 16) {  // 16 rows (32 loads) per trip
          float v0[16], v1[16];
#pragma unroll
          for (int u = 0; u < 16; u++) {
            v0[u] = has0 ? __ldg(Vr + (int64_t)(t + u) * hd + lane) : 0.f;
            v1[u] = has1 ? __ldg(Vr + (int64_t)(t + u) * hd + lane + 32) : 0.f;
          }
#pragma unroll
          for (int u = 0; u < 16; u++) {
            const float pt = sc[t + u];
            o0 = fmaf(pt, v0[u], o0);
            o1 = fmaf(pt, v1[u], o1);
          }
        }
#pragma unroll 1
        for (; t + 8 <= base; t += 8) {  // 8 rows (16 loads) per trip
          float v0[8], v1[8];
#pragma unroll
          for (int u = 0; u < 8; u++) {
            v0[u] = has0 ? __ldg(Vr + (int64_t)(t + u) * hd + lane) : 0.f;
            v1[u] = has1 ? __ldg(Vr + (int64_t)(t + u) * hd + lane + 32) : 0.f;
          }
#pragma unroll
          for (int u = 0; u < 8; u++) {
            const float pt = sc[t + u];
            o0 = fmaf(pt, v0[u], o0);
            o1 = fmaf(pt, v1[u], o1);
          }
        }
        for (; t < base; t++) {
          const float pt = sc[t];
          if (has0) o0 = fmaf(pt, __ldg(Vr + (int64_t)t * hd + lane), o0);
          if (has1) o1 = fmaf(pt, __ldg(Vr + (int64_t)t * hd + lane + 32), o1);
        }
      }
      for (int j = 0; j <= nin; j++) {
        const float* vj = c.act + (b - nin + j) * actw + 2 * hd;
        const float pl = sc[base + j];
        if (lane < hd) o0 = fmaf(pl, vj[lane], o0);
        if (lane + 32 < hd) o1 = fmaf(pl, vj[lane + 32], o1);
      }
      if (lane < hd) c.att[b * attw + lane] = o0 * inv;
      if (lane + 32 < hd) c.att[b * attw + lane + 32] = o1 * inv;
    }
  }
  prof_mark(c, 68);
  csync();
  prof_mark(c, 3);
  // ---- per-head partial output projection (fp32 SIMT, K = hd): thread = (row group g, 4 features) ----
  {
    const int G = kConsumers / (D >> 2);  // >= 2 for D <= 512
    const int nj = (nb + G - 1) / G;      // rows per thread
    float* dst = part_self(p) + (int64_t)h * p.B * D;
    if (nj <= 1) o_partial<1>(p, c, ring, nb, b0, dst);
    else if (nj <= 2) o_partial<2>(p, c, ring, nb, b0, dst);
    else if (nj <= 4) o_partial<4>(p, c, ring, nb, b0, dst);
    else o_partial<8>(p, c, ring, nb, b0, dst);
  }
  csync();
  prof_mark(c, 4);
}

// ============================== CROSS =================================
__device__ __forceinline__ void produce_cross(const DecoderParams& p, int l, int job, Ring& ring, const unsigned char* active) {
  const int H = p.H, hd = p.hd, D = p.D, nb = p.nb_cross;
  const int h = job % H, b0 = (job / H) * nb;
  if (!tile_active(p, active, nb, b0)) return;
  const DecLayerWeights& w = p.layers[l];
  // The cross K/V stream carries an L2 evict-first hint: the 191 MB a base/256 layer streams must not push the weight
  // planes out of L2 (measured 1677 -> 1582 us/step; an L2 prefetch window ahead of the ring and next-phase weight
  // prefetches were built and measured neutral or negative, profiles/r2e_prefetch_ab.txt, and removed again).
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  produce_block_planes(ring, w.wqcP + (size_t)h * plane_block_bytes(hd, D), hd, D);
  for (int b = 0; b < nb; b++) {
    if (b0 + b >= p.B || !active[b0 + b]) continue;
    const int64_t bh = ((int64_t)l * cache_utts(p) + row_utterance(p, b0 + b)) * H + h;
    produce_block_f16(ring, p.kc + bh * hd * p.Tpad, hd, p.Tpad, pol);   // K^T [hd][Tpad]
    produce_block_f16(ring, p.vc + bh * p.Tpad * hd, p.Tpad, hd, pol);   // V   [Tpad][hd]
  }
}

__device__ void job_cross(const DecoderParams& p, int l, int job, Ctx& c, Ring& ring, const float* hrd, float* hwr) {
  const int D = p.D, hd = p.hd, H = p.H, nb = p.nb_cross;
  const int h = job % H;
  const int b0 = (job / H) * nb;
  if (!tile_active(p, c.active, nb, b0)) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int actw = c.actw;
  load_flags(p, c, nb, b0, true);
  for (int r = warp; r < kMaxNB; r += kWarpsC) {
    RowVals rv;
    const bool live = !c.flags[r];
    if (live) {
      const int b = b0 + r;
      row_resolve(rv, D, hrd + (int64_t)b * D, part_self(p) + (int64_t)b * D, (int64_t)p.B * D, H, nullptr);
      if (h == 0) row_store(rv, D, hwr + (int64_t)b * D);
      row_layernorm(rv, D);
    }
    row_to_planes(rv, D, c.xp, 16, r, live);
  }
  prof_mark(c, 11);
  gemm_block(ring, c, c.xp, 16, D, hd, [&](int n, int cb, const float* v) {
    if (n < hd) {
#pragma unroll
      for (int e = 0; e < 16; e++) c.act[e * actw + n] = v[e];
    }
  });
  prof_mark(c, 12);

  const float scale = rsqrtf((float)hd);
  const int Tpad = p.Tpad;
  const int tpr = hd >> 2;           // threads per V row (4 halves = 8 bytes each)
  // Tiles with an even number of utterances give the two halves of the CTA (4 warps each, own named barrier and scratch)
  // alternate utterances: while one half is in the softmax / PV of utterance b the other is already in the scores of
  // b + 1 -- the 112 threads that own 4 keys each are all a 448-key utterance can use in the scores pass anyway.
  // Otherwise (one utterance per tile) the whole CTA walks it.
  const bool halves = (nb >= 2) && ((nb & 1) == 0) && (Tpad <= 512);
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
  for (int b = 0; b < nb; b++) {
    if (c.flags[b]) continue;  // uniform
    const bool mine = !halves || ((b & 1) == half);  // every thread walks every chunk; only the owner group computes
    const int T = c.flags[32 + b];
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
    prof_mark(c, 70);
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
        float* dst = p.xattn_out + (((((int64_t)(b0 + b) * p.L + l) * H + h) * p.xattn_steps + p.step) * Tpad + t4);
        *reinterpret_cast<float4*>(dst) = make_float4(s0 * inv, s1 * inv, s2 * inv, s3 * inv);
      }
    }
    prof_mark(c, 71);
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
    prof_mark(c, 72);
    if (mine) {
      if (g < G) *reinterpret_cast<float4*>(&pv[g * hd + dq * 4]) = make_float4(a0, a1, a2, a3);
      gsync();                                   // (3) PV partials visible
      if (gtid < hd) {
        float o = 0.f;
        for (int gg = 0; gg < G; gg++) o += pv[gg * hd + gtid];
        p.attc[(int64_t)(b0 + b) * D + h * hd + gtid] = o * inv;
      }
    }
    // no sync here: the next utterance only overwrites red_max before its sync (1), ps after it and pv after
    // its sync (2) -- by then every thread of the group has left this reduction.
  }
  csync();
  prof_mark(c, 13);
}

// ============================== GEMM jobs (OC, FC1, FC2) =================================
// job -> (m-tile mt, k-slice ks, utterance group g0 .. g0 + nb)
struct GemmJob {
  int mt, ks, g0, nb;
};
__device__ __forceinline__ int n_groups(const DecoderParams& p) { return (p.B + p.nx - 1) / p.nx; }
__device__ __forceinline__ GemmJob gemm_job(const DecoderParams& p, int kind, int job) {
  const int ng = n_groups(p);
  GemmJob j;
  const int gi = job % ng;
  int rest = job / ng;
  j.g0 = gi * p.nx;
  j.nb = min(p.nx, p.B - j.g0);
  j.ks = 0;
  if (kind == PH_FC2) {
    j.ks = rest % p.ffn_ksplit;
    rest /= p.ffn_ksplit;
  }
  j.mt = rest;
  return j;
}
__device__ __forceinline__ bool group_active(const unsigned char* active, int g0, int nb) {
  bool any = false;
  for (int b = 0; b < nb; b++) any |= active[g0 + b] != 0;
  return any;
}
// weight tile of a GEMM job: pointer, rows N of the tile, inputs K
__device__ __forceinline__ const unsigned char* gemm_tile(const DecoderParams& p, int kind, int l, const GemmJob& j, int& N, int& K) {
  const DecLayerWeights& w = p.layers[l];
  if (kind == PH_OC) {
    K = p.D;
    N = min(128, p.D - j.mt * 128);
    return w.wocF + (size_t)j.mt * 128 * ((K + 31) >> 5) * 128;
  }
  if (kind == PH_FC1) {
    K = p.D;
    N = min(128, 2 * p.I - j.mt * 128);
    return w.w1iF + (size_t)j.mt * 128 * ((K + 31) >> 5) * 128;
  }
  K = p.I / p.ffn_ksplit;
  N = min(128, p.D - j.mt * 128);
  return w.w2kF + (size_t)j.ks * plane_block_bytes(p.D, K) + (size_t)j.mt * 128 * ((K + 31) >> 5) * 128;
}
__device__ __forceinline__ void produce_gemm(const DecoderParams& p, int kind, int l, int job, Ring& ring, const unsigned char* active) {
  const GemmJob j = gemm_job(p, kind, job);
  if (!group_active(active, j.g0, j.nb)) return;
  int N, K;
  const unsigned char* P = gemm_tile(p, kind, l, j, N, K);
  produce_block_planes(ring, P, N, K);
}

__device__ void job_gemm(const DecoderParams& p, int kind, int l, int job, Ctx& c, Ring& ring, const float* hrd, float* hwr) {
  const GemmJob j = gemm_job(p, kind, job);
  if (!group_active(c.active, j.g0, j.nb)) return;
  int N, K;
  (void)gemm_tile(p, kind, l, j, N, K);
  const int D = p.D;
  const int NXp = (j.nb + 15) & ~15;
  const int warp = threadIdx.x >> 5;
  // ---- x planes ----
  if (kind == PH_FC1) {
    // LN(h + OC) per row, one warp per row, two rows of a warp in flight (the loads of both are issued before
    // either reduction); the first m-tile's job of the group keeps the new residual
    for (int r0 = warp; r0 < NXp; r0 += 2 * kWarpsC) {
      RowVals rv[2];
      bool live[2];
#pragma unroll
      for (int u = 0; u < 2; u++) {
        const int r = r0 + u * kWarpsC;
        live[u] = r < j.nb && c.active[j.g0 + r];
        if (live[u]) {
          const int b = j.g0 + r;
          row_resolve(rv[u], D, hrd + (int64_t)b * D, part_oc(p) + (int64_t)b * D, 0, 1, nullptr);
        }
      }
      prof_mark(c, 73);
#pragma unroll
      for (int u = 0; u < 2; u++) {
        const int r = r0 + u * kWarpsC;
        if (live[u]) {
          if (j.mt == 0) row_store(rv[u], D, hwr + (int64_t)(j.g0 + r) * D);
          row_layernorm(rv[u], D);
        }
        if (r < NXp) row_to_planes(rv[u], D, c.xg, NXp, r, live[u]);
      }
    }
  } else if (kind == PH_OC) {
    planes_from_rows(c.xg, NXp, p.attc, D, j.g0, j.nb, 0, K, c.active);
  } else {
    planes_from_rows(c.xg, NXp, p.act, p.I, j.g0, j.nb, j.ks * K, K, c.active);
  }
  prof_mark(c, 20 + kind);
  // ---- tensor core + epilogue ----
  if (kind == PH_FC1) {
    // rows interleaved (value, gate): even lanes hold the value of feature (n >> 1), odd lanes its gate
    const float* b1i = p.layers[l].b1i;
    float* act = p.act;
    const int I = p.I;
    gemm_block(ring, c, c.xg, NXp, K, N, [&](int nloc, int cb, const float* v) {
      const int n = j.mt * 128 + nloc;
      const float bias = (nloc < N) ? __ldg(b1i + n) : 0.f;
#pragma unroll
      for (int e = 0; e < 16; e++) {
        const float mine = v[e] + bias;
        const float other = __shfl_xor_sync(0xffffffffu, mine, 1);
        if (!(nloc & 1) && nloc < N && cb + e < j.nb) {
          const float gate = other;
          act[(int64_t)(j.g0 + cb + e) * I + (n >> 1)] = gate / (1.0f + expf(-gate)) * mine;  // silu(gate) * value
        }
      }
    });
  } else {
    float* out = (kind == PH_OC) ? part_oc(p) : part_fc2(p) + (int64_t)j.ks * p.B * D;
    gemm_block(ring, c, c.xg, NXp, K, N, [&](int nloc, int cb, const float* v) {
      if (nloc < N) {
        const int n = j.mt * 128 + nloc;
#pragma unroll
        for (int e = 0; e < 16; e++)
          if (cb + e < j.nb) out[(int64_t)(j.g0 + cb + e) * D + n] = v[e];
      }
    });
  }
  prof_mark(c, 30 + kind);
}

// ============================== FINAL =================================
// 8 utterances per job, one warp each: last residual resolve + final LayerNorm (gamma folded into the head matrix)
__device__ void job_final(const DecoderParams& p, int job, Ctx& c, const float* hrd) {
  const int D = p.D, warp = threadIdx.x >> 5;
  const int b = job * kWarpsC + warp;
  if (b < p.B && c.active[b]) {
    RowVals rv;
    row_resolve(rv, D, hrd + (int64_t)b * D, part_fc2(p) + (int64_t)b * D, (int64_t)p.B * D, p.ffn_ksplit, p.layers[p.L - 1].b2);
    row_layernorm(rv, D);
    row_store(rv, D, p.xfin + (int64_t)b * D);
  }
  csync();
}

// ============================== LOGITS =================================
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

__device__ void job_logits(const DecoderParams& p, int item, Ctx& c, Ring& ring, int nx) {
  const int D = p.D, V = p.V, VC = p.vchunk;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_mt = (VC + 127) >> 7, nkb = D >> 5;
  const int parity = p.step & 1;
  unsigned char* xp = c.xg;  // [kb][hi nx x 64 B | lo nx x 64 B]
  const uint32_t idesc = idesc_bf16(nx);
  for (int b0 = 0; b0 < p.B; b0 += nx) {
    const int nb = min(nx, p.B - b0);
    planes_from_rows(xp, nx, p.xfin, D, b0, nb, 0, D, c.active);
    const bool biased = p.bias_static != nullptr || p.bias_dyn_n != nullptr;
    if (biased) {
      // bonuses that land in this CTA's vocab chunk: the shared ones as a dense slice, the per-utterance ones as
      // (row, utterance column, bonus) entries
      for (int i = threadIdx.x; i < 384; i += kConsumers) {
        const int v = item * VC + i;
        c.sbias[i] = (p.bias_static != nullptr && i < VC && v < V) ? __ldg(p.bias_static + v) : 0.f;
        c.rowflag[i] = 0;
      }
      if (threadIdx.x == 0) *c.ent_n = 0;
      csync();
      if (p.bias_dyn_n != nullptr) {
        const int cap = p.bias_dyn_cap;
        for (int idx = threadIdx.x; idx < nb * cap; idx += kConsumers) {
          const int b = idx / cap, k = idx - b * cap;
          if (k < p.bias_dyn_n[b0 + b]) {
            const int loc = p.bias_dyn_ids[(int64_t)(b0 + b) * cap + k] - item * VC;
            if (loc >= 0 && loc < VC) {
              const int slot = atomicAdd(c.ent_n, 1);
              if (slot >= kBiasEntries) atomicExch(c.err, 2u);  // table overflow: fail the decode, never drop a bonus
              if (slot < kBiasEntries) {
                c.ent_key[slot] = (loc << 9) | b;
                c.ent_val[slot] = p.bias_dyn_val[(int64_t)(b0 + b) * cap + k];
                c.rowflag[loc] = 1;
              }
            }
          }
        }
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    csync();
    prof_mark(c, 35);
    int nchunks = 0;
    for (int mt = 0; mt < n_mt; mt++) nchunks += (nkb + 1) >> 1;
    const int warp_u = (int)uniform_u32((uint32_t)warp);
    if (warp_u == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t xb = uniform_u32(smem_u32(xp));
      const uint32_t tm = uniform_u32(c.tmem);
      for (int mt = 0; mt < n_mt; mt++) {
        const int R = min(128, VC - mt * 128);
        const uint32_t tmem_d = tm + (uint32_t)(mt * nx);
        for (int kb = 0; kb < nkb; kb += 2) {
          const int n = min(2, nkb - kb);
          mbar_wait(&ring.full[ring.stage()], ring.parity(), c.err);
          __syncwarp();
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t a_base = uniform_u32(smem_u32(ring.data + (size_t)ring.stage() * kStageBytes));
          const uint32_t empty_bar = uniform_u32(smem_u32(&ring.empty[ring.stage()]));
          if (elect_one()) {
            for (int q = 0; q < n; q++) {
              const uint32_t a_hi = a_base + (uint32_t)(q * R * 128), a_lo = a_hi + (uint32_t)(R * 64);
              const uint32_t b_hi = xb + (uint32_t)((kb + q) * nx * 128), b_lo = b_hi + (uint32_t)(nx * 64);
#pragma unroll
              for (int jj = 0; jj < 2; jj++) {
                const uint32_t ko = (uint32_t)jj * 32u;
                const uint32_t first = (kb | q | jj) ? 1u : 0u;
                umma_bf16(tmem_d, make_desc_sw64(a_lo + ko), make_desc_sw64(b_hi + ko), idesc, first);
                umma_bf16(tmem_d, make_desc_sw64(a_hi + ko), make_desc_sw64(b_lo + ko), idesc, 1u);
                umma_bf16(tmem_d, make_desc_sw64(a_hi + ko), make_desc_sw64(b_hi + ko), idesc, 1u);
              }
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(empty_bar) : "memory");
          }
          __syncwarp();
          ring.advance();
        }
      }
      if (elect_one()) umma_commit(c.acc_bar);
      __syncwarp();
      prof_mark(c, 36);
    } else if (lane == 0) {
      for (int i = 0; i < nchunks; i++) {
        mbar_wait_relaxed(&ring.full[ring.stage()], ring.parity(), c.err);
        mbar_arrive(&ring.empty[ring.stage()]);
        ring.advance();
      }
    } else {
      ring.advance_by(nchunks);
    }
    __syncwarp();
    mbar_wait_relaxed(c.acc_bar, (uint32_t)(c.acc_phase & 1), c.err);
    c.acc_phase++;
    __syncwarp();
    prof_mark(c, 37);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // running best (key, index) of this warp per utterance column; warps 0-3 take m-tiles 0, 2, warps 4-7 m-tile 1
    for (int b = lane; b < 64; b += 32) { c.argv[warp * 64 + b] = 0.f; c.argi[warp * 64 + b] = 0x7fffffff; }
    __syncwarp();
    for (int mt_w = warp >> 2; mt_w < n_mt; mt_w += 2) {
      const int vrow = mt_w * 128 + (warp & 3) * 32 + lane;
      const int v = item * VC + vrow;
      const bool vok = (vrow < VC) && (v < V);
      for (int cb = 0; cb < nx; cb += 16) {
        uint32_t r[16];
        {
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
        if (biased && vok) {
          const float sb = c.sbias[vrow];
#pragma unroll
          for (int e = 0; e < 16; e++) r[e] = __float_as_uint(__uint_as_float(r[e]) + sb);
          if (c.rowflag[vrow]) {  // rare: some utterance's active key-term path continues with this token
            const int n_ent = min(*c.ent_n, kBiasEntries);
            for (int s2 = 0; s2 < n_ent; s2++) {
              const int key = c.ent_key[s2];
              const int col = (key & 511) - cb;
              if ((key >> 9) == vrow && col >= 0 && col < 16) {
                const float add = c.ent_val[s2];
#pragma unroll
                for (int e = 0; e < 16; e++)
                  if (e == col) r[e] = __float_as_uint(__uint_as_float(r[e]) + add);
              }
            }
          }
        }
#pragma unroll
        for (int e = 0; e < 16; e++) {
          const int b = cb + e;
          const float val = __uint_as_float(r[e]);
          if (vok && p.logits_out && b < nb) p.logits_out[(int64_t)(b0 + b) * V + v] = val;
          // order-preserving float -> uint key (NaN and masked rows -> 0, never win); one redux gives the warp max,
          // the lowest lane holding it is the first (smallest) vocab index
          uint32_t key = r[e];
          key = (key & 0x80000000u) ? ~key : (key | 0x80000000u);
          if (!vok || val != val) key = 0u;
          const uint32_t mx = __reduce_max_sync(0xffffffffu, key);
          const uint32_t who = __ballot_sync(0xffffffffu, key == mx);
          if (lane == 0 && mx != 0u) {
            const int idx = item * VC + mt_w * 128 + (warp & 3) * 32 + (__ffs(who) - 1);
            const uint32_t cur_key = __float_as_uint(c.argv[warp * 64 + b]);
            if (mx > cur_key || (mx == cur_key && idx < c.argi[warp * 64 + b])) {
              c.argv[warp * 64 + b] = __uint_as_float(mx);
              c.argi[warp * 64 + b] = idx;
            }
          }
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
      const float bv = bk == 0u ? -INFINITY : __uint_as_float((bk & 0x80000000u) ? (bk & 0x7fffffffu) : ~bk);
      p.cand_val[((int64_t)parity * p.n_vchunk + item) * p.B + b0 + b] = bv;
      p.cand_idx[((int64_t)parity * p.n_vchunk + item) * p.B + b0 + b] = bi;
    }
    csync();
  }
}

// ------------------------------------------------------------------------------------------------
// program walk (identical for producers and consumers)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int phase_jobs(const DecoderParams& p, int kind) {
  const int ng = (p.B + p.nx - 1) / p.nx;
  switch (kind) {
    case PH_SELF: return p.H * ((p.B + p.nb_self - 1) / p.nb_self);
    case PH_CROSS: return p.H * ((p.B + p.nb_cross - 1) / p.nb_cross);
    case PH_OC: return ((p.D + 127) >> 7) * ng;
    case PH_FC1: return ((2 * p.I + 127) >> 7) * ng;
    case PH_FC2: return ((p.D + 127) >> 7) * p.ffn_ksplit * ng;
    case PH_FINAL: return (p.B + kWarpsC - 1) / kWarpsC;
    default: return p.n_vchunk;
  }
}
// first job of this CTA in a phase of `kind` (or >= njobs) and the stride between its jobs
__device__ __forceinline__ void my_jobs(const DecoderParams& p, int kind, int njobs, int& j0, int& stride) {
  const int G = (int)gridDim.x;
  int ncta = p.job_ncta[kind];
  if (ncta > G) ncta = G;
  const int rel = ((int)blockIdx.x - p.job_first[kind] % G + G) % G;
  stride = ncta;
  j0 = rel < ncta ? rel : njobs;
}

__global__ void __launch_bounds__(kThreads3, 1) decoder_step3_kernel(const __grid_constant__ DecoderParams p) {
  if (*p.n_active == 0) return;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  const int Kc = p.I / p.ffn_ksplit;
  const SmemLayout3 L = smem_layout3(p.B, p.D, p.hd, Kc, p.nx, p.Tpad, p.Smax, p.smem_limit);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + L.bars);
  unsigned char* active = smem_raw + L.active;
  unsigned* err = p.sync3 + 1;
  Ring ring;
  ring.full = bars;
  ring.empty = bars + 16;
  ring.data = reinterpret_cast<char*>(smem_raw + L.ring);
  ring.err = err;
  ring.ns = L.ns;
  ring.reset((threadIdx.x - kConsumers) >> 5);  // meaningful for the producer lanes only

  // work list of this launch: utterances not finished BEFORE this step (done[b] = step at which it finished + 1)
  for (int b = threadIdx.x; b < p.B; b += kThreads3) {
    if (p.row_tok) {  // explicit rows: the plan kernel decided which rows run
      active[b] = p.row_tok[b] >= 0 ? 1 : 0;
    } else {
      const int d = p.done[b];
      active[b] = (d == 0 || d > p.step) ? 1 : 0;
    }
  }
  const unsigned epoch = *reinterpret_cast<const volatile unsigned*>(p.sync3);
  uint32_t& tmem_base_smem = *reinterpret_cast<uint32_t*>(bars + 33);
  if (threadIdx.x == 0) {
    for (int i = 0; i < L.ns; i++) {
      mbar_init(&ring.full[i], 1);
      mbar_init(&ring.empty[i], kWarpsC);
    }
    mbar_init(bars + 32, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x < 32) {  // warp 0 owns the TMEM allocation (256 columns: 3 accumulators x <= 64 utterances)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "r"(256) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_smem;
  const int n_phases = p.L * kPhasesPerLayer + 2;

  if (threadIdx.x >= kConsumers) {
    // ======================= producer warps (one lane each) =======================
    if ((threadIdx.x & 31) == 0) {
      for (int pi = 0; pi < n_phases; pi++) {
        const int l = pi / kPhasesPerLayer;
        const int kind = l < p.L ? pi - l * kPhasesPerLayer : PH_FINAL + (pi - p.L * kPhasesPerLayer);
        if (kind == PH_FINAL) continue;  // no ring traffic
        const int njobs = phase_jobs(p, kind);
        int j0, stride;
        my_jobs(p, kind, njobs, j0, stride);
        for (int j = j0; j < njobs; j += stride) {
          if (kind == PH_SELF) produce_self(p, l, j, ring, active);
          else if (kind == PH_CROSS) produce_cross(p, l, j, ring, active);
          else if (kind == PH_LOGITS) produce_logits(p, j, ring, L.nxl);
          else produce_gemm(p, kind, l, j, ring, active);
        }
      }
    }
    return;
  }

  // ========================= consumers =========================
  Ctx c;
  c.err = err;
  c.xp = smem_raw + L.xp;
  c.xg = smem_raw + L.scratch;
  c.act = reinterpret_cast<float*>(smem_raw + L.act);
  c.att = reinterpret_cast<float*>(smem_raw + L.att);
  c.red = reinterpret_cast<float*>(smem_raw + L.red);
  c.ps = reinterpret_cast<float*>(smem_raw + L.ps);
  c.sc = reinterpret_cast<float*>(smem_raw + L.sc);
  c.flags = reinterpret_cast<int*>(smem_raw + L.flags);
  c.argv = reinterpret_cast<float*>(smem_raw + L.argv);
  c.argi = reinterpret_cast<int*>(smem_raw + L.argi);
  c.sbias = reinterpret_cast<float*>(smem_raw + L.sbias);
  c.rowflag = smem_raw + L.rowflag;
  c.ent_key = reinterpret_cast<int*>(smem_raw + L.ent_key);
  c.ent_val = reinterpret_cast<float*>(smem_raw + L.ent_val);
  c.ent_n = reinterpret_cast<int*>(smem_raw + L.ent_n);
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
  }
  c.tmem = tmem_base;
  c.acc_bar = bars + 32;
  c.acc_phase = 0;
  c.prof = reinterpret_cast<unsigned long long*>(p.prof);
  c.prof_n = 0;
  prof_mark(c, 0);
  csync();

  const int64_t BD = (int64_t)p.B * p.D;
  unsigned* counters = p.sync3 + 32;  // one 128-byte line per phase
  int ph = 0;                          // residual ping-pong: phases with an LN prologue read hbuf[ph & 1], write the other
  for (int pi = 0; pi < n_phases; pi++) {
    const int l = pi / kPhasesPerLayer;
    const int kind = l < p.L ? pi - l * kPhasesPerLayer : PH_FINAL + (pi - p.L * kPhasesPerLayer);
    const float* hrd = p.hbuf + (int64_t)(ph & 1) * BD;
    float* hwr = p.hbuf + (int64_t)((ph + 1) & 1) * BD;
    if (kind == PH_SELF || kind == PH_CROSS || kind == PH_FC1) ph++;
    const int njobs = phase_jobs(p, kind);
    int j0, stride;
    my_jobs(p, kind, njobs, j0, stride);
    if (j0 >= njobs) continue;
    if (pi > 0) {  // every job of the previous phase has signalled
      if (threadIdx.x == 0) {
        const int lk = (pi - 1) / kPhasesPerLayer;
        const int pk = lk < p.L ? (pi - 1) - lk * kPhasesPerLayer : PH_FINAL + ((pi - 1) - p.L * kPhasesPerLayer);
        const unsigned target = (epoch + 1u) * (unsigned)phase_jobs(p, pk);
        const unsigned* cnt = counters + (size_t)(pi - 1) * 32;
        const long long t0 = clock64();
        unsigned polls = 0;
        while ((int)(ld_acquire(cnt) - target) < 0) {
          if ((++polls & 15u) == 0u) {
            if (poisoned(err)) break;
            if (clock64() - t0 > kSpinLimit) { atomicExch(err, 1u); break; }
          }
        }
      }
      csync();
    }
    prof_mark(c, 40 + kind);
    for (int j = j0; j < njobs; j += stride) {
      if (kind == PH_SELF) job_self(p, l, j, c, ring, hrd, hwr);
      else if (kind == PH_CROSS) job_cross(p, l, j, c, ring, hrd, hwr);
      else if (kind == PH_FINAL) job_final(p, j, c, hrd);
      else if (kind == PH_LOGITS) job_logits(p, j, c, ring, L.nxl);
      else job_gemm(p, kind, l, j, c, ring, hrd, hwr);
      // every job ends with a CTA barrier behind its last global store: one release-add publishes them
      if (threadIdx.x == 0)
        asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(counters + (size_t)pi * 32), "r"(1u) : "memory");
    }
    prof_mark(c, 50 + kind);
  }
  if (blockIdx.x == 0) {
    // the step is over when every logits job has signalled; then count what is left and open the next epoch
    if (threadIdx.x == 0) {
      const unsigned target = (epoch + 1u) * (unsigned)phase_jobs(p, PH_LOGITS);
      const unsigned* cnt = counters + (size_t)(n_phases - 1) * 32;
      const long long t0 = clock64();
      unsigned polls = 0;
      while ((int)(ld_acquire(cnt) - target) < 0) {
        if ((++polls & 15u) == 0u) {
          if (poisoned(err)) break;
          if (clock64() - t0 > kSpinLimit) { atomicExch(err, 1u); break; }
        }
      }
    }
    csync();
    int* cnt = c.flags;
    if (threadIdx.x == 0) *cnt = 0;
    csync();
    int n = 0;
    if (p.row_tok == nullptr)
      for (int b = threadIdx.x; b < p.B; b += kConsumers) n += __ldcg(p.done + b) ? 0 : 1;
    if (n) atomicAdd(cnt, n);
    csync();
    if (threadIdx.x == 0) {
      if (p.row_tok == nullptr) *p.n_active = *cnt;  // explicit rows: the plan kernel counts
      p.sync3[0] = epoch + 1u;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  csync();
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256) : "memory");
  }
}

__global__ void decoder_resolve_kernel(const __grid_constant__ DecoderParams p, int* out) {
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (b >= p.B) return;
  const int tok = resolve_token_warp(p, b, p.step & 1);
  if ((threadIdx.x & 31) == 0) out[b] = tok;
}

// Plan of explicit-row launch k of a verify-then-continue decode (reference: decode_full,
// core/moonshine-streaming-model.cpp:1192-1397, batched and chunked: n rows per utterance per launch instead of the
// whole draft in one decoder run).  One warp per utterance: resolves the argmax of the rows launch k-1 ran for it,
// books the emitted ids exactly like the greedy loop would (ids, EOS / budget stop), advances the utterance
//   VERIFY  inputs [BOS, draft...] at positions pos .. pos+n-1 (row i also attends the i rows before it); an emitted
//           id that equals the next draft id keeps verifying, anything else (or the end of the draft) -> AR
//   AR      one row: the last emitted id at its own position (utterances diverge at different positions)
//   DONE    EOS emitted or the budget reached
// and writes the rows of launch k.  Rows behind a rejected draft id computed K/V for positions the utterance re-writes
// before it ever reads them (position p is appended by the row at p before any row attends it), so nothing is reset.
__global__ void decoder_verify_plan_kernel(const __grid_constant__ DecoderParams p, VerifyState s, int k, int n, int bos, int eos) {
  __shared__ int alive;
  if (threadIdx.x == 0) alive = 0;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  int* row_tok = const_cast<int*>(p.row_tok);
  int* row_pos = const_cast<int*>(p.row_pos);
  int* row_nin = const_cast<int*>(p.row_nin);
  int* row_utt = const_cast<int*>(p.row_utt);
  for (int u = warp; u < p.B_utt; u += nw) {
    int mode = s.mode[u], pos = s.pos[u], cur = s.cur[u];
    const int prevn = s.prev_n[u], m = s.draft_len[u], maxlen = p.max_len[u];
    const int* d = s.draft + (int64_t)u * s.draft_stride;
    const int64_t trow = (int64_t)u * (p.Smax + 1);
    if (k == 0) {
      mode = maxlen > 0 ? (m > 0 ? 0 : 1) : 2;
      pos = 0;
      cur = bos;
    } else if (mode != 2) {
      for (int i = 0; i < prevn; i++) {
        const int e = resolve_token_warp(p, u * n + i, (k - 1) & 1);
        const int t = pos + i;
        if (lane == 0) {
          p.tokens[trow + t + 1] = e;
          p.n_tokens[u] = t + 2;
        }
        if (e == eos || t + 1 >= maxlen) { mode = 2; break; }
        const bool accepted = mode == 0 && t < m && e == d[t];
        if (accepted && i + 1 < prevn) continue;
        if (!accepted) { mode = 1; cur = e; }
        pos = t + 1;
        break;
      }
    }
    int rows = 0;
    if (mode == 0) rows = min(n, min(m + 1 - pos, maxlen - pos));
    else if (mode == 1) rows = 1;
    if (lane < n) {
      const int r = u * n + lane;
      const bool on = lane < rows;
      const int at = pos + lane;
      row_tok[r] = !on ? -1 : (mode == 1 ? cur : (at == 0 ? bos : d[at - 1]));
      row_pos[r] = on ? at : 0;
      row_nin[r] = on && mode == 0 ? lane : 0;
      row_utt[r] = u;
    }
    if (lane == 0) {
      s.mode[u] = mode; s.pos[u] = pos; s.cur[u] = cur; s.prev_n[u] = rows;
      if (mode != 2) atomicAdd(&alive, 1);
      else p.done[u] = 1;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) *p.n_active = alive;
}

// Splice from explicit rows back into the lockstep loop: the argmax candidates of "step - 1" are seeded so that the next
// lockstep launch resolves utterance b's previous id to cur[b] (lowest index wins among equal values, every other chunk
// carries -inf).
__global__ void decoder_seed_candidates_kernel(const __grid_constant__ DecoderParams p, const int* cur, int parity) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n_vchunk * p.B) return;
  const int c = i / p.B, b = i - c * p.B;
  float* cv = p.cand_val + (int64_t)parity * p.n_vchunk * p.B;
  int* ci = p.cand_idx + (int64_t)parity * p.n_vchunk * p.B;
  cv[i] = c == 0 ? 0.f : -INFINITY;
  ci[i] = c == 0 ? cur[b] : 0x7fffffff;
}

}  // namespace

void launch_decoder_seed_candidates(const DecoderParams& p, const int* cur, int parity, cudaStream_t stream) {
  const int n = p.n_vchunk * p.B;
  decoder_seed_candidates_kernel<<<(n + 255) / 256, 256, 0, stream>>>(p, cur, parity);
}

void launch_decoder_verify_plan(const DecoderParams& p, const VerifyState& s, int k, int n, int bos, int eos, cudaStream_t stream) {
  if (n < 1 || n > 16) throw std::runtime_error("decoder v3: 1..16 rows per utterance");
  decoder_verify_plan_kernel<<<1, 1024, 0, stream>>>(p, s, k, n, bos, eos);
}

void launch_decoder_resolve(const DecoderParams& p, int* out, cudaStream_t stream) {
  const int warps_per_block = 4;
  const int blocks = (p.B + warps_per_block - 1) / warps_per_block;
  decoder_resolve_kernel<<<blocks, warps_per_block * 32, 0, stream>>>(p, out);
}

bool decoder_step3_supported(const DecoderParams& p) {
  return p.D % 32 == 0 && p.D <= 64 * kMaxPairs && p.hd <= 64 && p.hd % 4 == 0 && p.rot_dim <= 128 && p.Tpad <= 1024 &&
         p.L * kPhasesPerLayer + 2 <= 64 && p.layers[0].wocF != nullptr;
}

void decoder_step3_plan(DecoderParams& p, int grid) {
  const int B = p.B;
  // attention tiles: enough jobs to occupy ~128 CTAs, at most 16 utterances (one N = 16 operand)
  auto pick = [&](int want_jobs) {
    int nb = 1;
    while (nb < kMaxNB && p.H * ((B + nb - 1) / nb) > want_jobs) nb *= 2;
    return nb;
  };
  p.nb_cross = pick(128);
  p.nb_self = std::max(pick(128), std::min(8, p.nb_cross * 4));
  if (p.nb_self > kMaxNB) p.nb_self = kMaxNB;
  if (p.row_group > 1) {  // explicit rows: the rows of one utterance slot share a self-attention tile
    if (p.row_group > kMaxNB || (kMaxNB % p.row_group) != 0) throw std::runtime_error("decoder v3: row group must divide 16");
    while (p.nb_self % p.row_group) p.nb_self *= 2;
  }
  // GEMM groups: 32 utterances (measured: 64 / 48 / 32 -> 1470 / 1471 / 1419 us per step at base/256, 767 -> 734 at
  // base-streaming/64: smaller groups mean more jobs per phase and shorter resolve prologues), fewer when the x planes of
  // the widest input would not fit 80 KB
  const int Kc = p.I / p.ffn_ksplit;
  const int kmax = (std::max(p.D, Kc) + 31) / 32 * 32;
  p.nx = std::min(32, (B + 15) & ~15);
  while (p.nx > 16 && p.nx * kmax * 4 > 80 * 1024) p.nx -= 16;
  // CTA assignment.  Small batches leave CTAs beyond the attention jobs: they become the GEMM engines (their
  // weight tiles sit in shared memory before the attention phases end).  Large batches spread every phase.
  const int ng = (B + p.nx - 1) / p.nx;
  const int n_attn = std::max(p.H * ((B + p.nb_self - 1) / p.nb_self), p.H * ((B + p.nb_cross - 1) / p.nb_cross));
  const int attn_ctas = std::min(grid, n_attn);
  const int spare = grid - attn_ctas;
  for (int k = 0; k < 8; k++) { p.job_first[k] = 0; p.job_ncta[k] = grid; }
  const int jobs_gemm[3] = {((p.D + 127) / 128) * ng, ((2 * p.I + 127) / 128) * ng, ((p.D + 127) / 128) * p.ffn_ksplit * ng};
  int off = 0;
  for (int k = 0; k < 3; k++) {
    const int kind = PH_OC + k;
    if (spare >= 8 && jobs_gemm[k] <= spare) {
      p.job_first[kind] = attn_ctas + (spare > jobs_gemm[k] ? off % (spare - std::min(spare, jobs_gemm[k]) + 1) : 0);
      p.job_ncta[kind] = std::min(spare - (p.job_first[kind] - attn_ctas), std::max(1, jobs_gemm[k]));
      off += jobs_gemm[k];
    } else {
      p.job_first[kind] = (37 * (k + 1)) % grid;
      p.job_ncta[kind] = grid;
    }
  }
  p.job_first[PH_FINAL] = spare > 0 ? attn_ctas : 0;
  p.job_ncta[PH_FINAL] = spare > 0 ? spare : grid;
}

size_t decoder_step3_smem_bytes(const DecoderParams& p) {
  const SmemLayout3 L = smem_layout3(p.B, p.D, p.hd, p.I / p.ffn_ksplit, p.nx, p.Tpad, p.Smax, p.smem_limit);
  if (L.ns < 2) throw std::runtime_error("decoder v3: not enough shared memory for the operand ring");
  return (size_t)L.total;
}

void launch_decoder_step3(const DecoderParams& p, int grid, cudaStream_t stream) {
  const size_t smem = decoder_step3_smem_bytes(p);
  auto kern = decoder_step3_kernel;
  static SmemAttrCache cache;
  if (cache.needs(smem)) CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  void* args[] = {const_cast<DecoderParams*>(&p)};
  CUDA_CHECK(cudaLaunchCooperativeKernel((void*)kern, dim3(grid), dim3(kThreads3), args, smem, stream));
}

}  // namespace msb
