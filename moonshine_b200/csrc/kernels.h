// Kernel launch interface (host-callable) for the Moonshine B200 runtime.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdint>

namespace msb {

// ---------------------------------------------------------------------------
// Grouped "NT" GEMM:  C_z[m, n] = epi( alpha * sum_k A_z[m, k] * W_z[n, k] )
// A rows have stride lda, W rows stride ldw (both K-contiguous, multiples of 4
// floats, 16-byte aligned bases).  Per-group dims/offsets are optional device
// arrays; without them group z uses z * stride{A,W,C} and the uniform M/N/K.
// ---------------------------------------------------------------------------
struct GemmParams {
  const float* A = nullptr;
  const float* W = nullptr;
  void* C = nullptr;
  int M = 0, N = 0, K = 0;
  int lda = 0, ldw = 0;
  int groups = 1;
  int64_t strideA = 0, strideW = 0, strideC = 0;
  const int64_t* offA = nullptr;
  const int64_t* offW = nullptr;
  const int64_t* offC = nullptr;
  const int* Mz = nullptr;
  const int* Nz = nullptr;
  const int* Kz = nullptr;
  // epilogue
  float alpha = 1.0f;
  const float* bias = nullptr;  // indexed by n (or by m when bias_on_m)
  int bias_on_m = 0;
  int act = 0;                  // 0 = none, 1 = exact-erf GELU, 2 = SiLU
  int accumulate = 0;           // C += result (fp32 output only)
  int out_half = 0;             // store __half instead of float
  // output addressing: addr = offC + rowoff(m) + coloff(n)
  //   rowoff(m) = rm1 ? (m / rm1) * rs1 + ((m % rm1) / rm2) * rs2 + (m % rm2) * rs : m * rs
  //   coloff(n) = cm1 ? (n / cm1) * cs1 + ((n % cm1) / cm2) * cs2 + (n % cm2)      : n
  int64_t rs = 0;
  int rm1 = 0, rm2 = 1;
  int64_t rs1 = 0, rs2 = 0;
  int cm1 = 0, cm2 = 1;
  int64_t cs1 = 0, cs2 = 0;
  // optional interleaved-pair RoPE on columns n < rope_cols (per-row position)
  const int* pos = nullptr;        // [M]
  const float* rope_cos = nullptr; // [max_pos][rot_dim / 2]
  const float* rope_sin = nullptr;
  int rope_cols = 0, head_dim = 1, rot_dim = 0;
};
// Dispatches to the tcgen05 bf16x3 kernel (default) or the fp32 SIMT kernel
// (MOONSHINE_B200_GEMM=simt).
void launch_gemm(const GemmParams& p, cudaStream_t stream);
void launch_gemm_simt(const GemmParams& p, cudaStream_t stream);
void launch_gemm_tc(const GemmParams& p, cudaStream_t stream);

// ---------------------------------------------------------------------------
// Plane-fed GEMM (gemm_planes.cu): both operands pre-split to bf16 hi/lo planes in UMMA tile order, fed by bulk copies.
// Plane layout of an [R][K] operand (K % 32 == 0): tile (rt = r / 128, kb = k / 32) at ((rt * K/32) + kb) * kPlaneTileBytes,
// [hi 128 rows x 64 B | lo 128 rows x 64 B], chunk c of row r at position c ^ ((r >> 1) & 3).  Rows beyond R are padding
// (weights: zeros written at load; activations: whatever is there -- they only reach output rows that are never stored).
// ---------------------------------------------------------------------------
constexpr int kPlaneTileBytes = 16384;
inline size_t plane_tiles_bytes(int64_t rows, int K) { return (size_t)((rows + 127) / 128) * (size_t)(K / 32) * kPlaneTileBytes; }
struct GemmPlanesParams {
  const unsigned char* A = nullptr;  // planes of the activations [M][K]
  const unsigned char* W = nullptr;  // planes of the weights [N][K]
  int M = 0, N = 0, K = 0;
  float* C = nullptr;                // fp32 output rows (row stride ldc), may be null when only planes are wanted
  int64_t ldc = 0;
  unsigned char* P = nullptr;        // optional: the output as planes of an [M][N] operand (input of the next GEMM)
  int variant = 0;                   // 0 = pick by launch size, 1 = one 128 x 128 tile per CTA, 2 = persistent 128 x 256 macro tiles
  int p_taps = 1, p_stride = 1;      // > 1 taps: P is the im2col operand of a following convolution (row r = p_taps output rows from p_stride * r)
  const float* bias = nullptr;       // [N]
  int act = 0;                       // 1 = exact-erf GELU
  int accumulate = 0;                // C += result
  const int* pos = nullptr;          // interleaved-pair RoPE on columns n < rope_cols (per-row position), like GemmParams
  const float* rope_cos = nullptr;
  const float* rope_sin = nullptr;
  int rope_cols = 0, head_dim = 1, rot_dim = 0;
  // optional column split: columns n >= n_split (a multiple of 32) are stored TRANSPOSED instead, Vt[vt_row[m] + (n - n_split) * vt_ld]
  // (rows with vt_row[m] < 0 are skipped) -- the encoder's V^T_b[e][t] next to its Q | K rows
  // optional fp16 cross-K/V outputs of the decoder (replaces C / P): columns n < n_split = (l, h, d) of K, stored time-
  // contiguous Hk[hk_row[m] + (n / Dm) * SL + (n % Dm) * Tpadm]; columns >= n_split = (l, h, d) of V,
  // Hv[hv_row[m] + (n' / Dm) * SL + ((n' % Dm) / hdm) * Tpadm * hdm + n' % hdm]; rows with a negative base are skipped
  __half* Hk = nullptr;
  __half* Hv = nullptr;
  const int64_t* hk_row = nullptr;
  const int64_t* hv_row = nullptr;
  int64_t SL = 0;
  int Dm = 1, hdm = 1, Tpadm = 0;
  int n_split = 0;
  float* Vt = nullptr;
  const int64_t* vt_row = nullptr;
  int64_t vt_ld = 0;
};
bool gemm_planes_supported(const GemmPlanesParams& p);
void launch_gemm_planes(const GemmPlanesParams& p, cudaStream_t stream);
// watchdog flag of the plane-fed kernels (a wait that timed out): copy it to pinned memory in stream order / reset it
void gemm_planes_error_async(unsigned int* pinned_dst, cudaStream_t stream);
void gemm_planes_clear_error(cudaStream_t stream);
void gemm_tc_error_async(unsigned int* pinned_dst, cudaStream_t stream);
void gemm_tc_clear_error(cudaStream_t stream);
void attention_tc_error_async(unsigned int* pinned_dst, cudaStream_t stream);
void attention_tc_clear_error(cudaStream_t stream);
// y (optional fp32 rows) and planes of LayerNorm(x) * gamma
void launch_layernorm_planes(const float* x, float* y, unsigned char* planes, const float* gamma, int64_t rows, int D,
                             cudaStream_t stream);
// GroupNorm apply of the conv1 rows written as the plane tiles of conv2's im2col operand [tot1 / 3][7 * D]
void launch_groupnorm_im2col_planes(const float* h1, const int* t1, const int64_t* off1, const double* gn_partial, int nblk,
                                    const float* gamma, const float* beta, int D, int B, int max_t1, unsigned char* planes,
                                    cudaStream_t stream);
void launch_rows_to_planes(const float* src, int64_t ld, int64_t rows, int K, unsigned char* planes, cudaStream_t stream);

// ---------------------------------------------------------------------------
// Frontend
// ---------------------------------------------------------------------------
// conv1 (1 -> D, k=127, s=64, no bias) + tanh, channel-last output rows
// off1[b] + t, plus per-utterance GroupNorm(1 group) statistics.
void launch_conv1_tanh(const float* pcm, int64_t pcm_stride, const int* n_samples, const int* t1,
                       const int64_t* off1, const float* w1t /*[127][D]*/, float* h1, int D,
                       int B, int max_t1, double* gn_partial /*[B][nblk][2]*/, int* nblk_out,
                       cudaStream_t stream);
int conv1_blocks_per_utt(int max_t1);
// (x - mean) * rstd * gamma[c] + beta[c], in place, using the partial sums.
void launch_groupnorm_apply(float* h1, const int* t1, const int64_t* off1, const double* gn_partial,
                            int nblk, const float* gamma, const float* beta, int D, int B,
                            int max_t1, cudaStream_t stream);

// ---------------------------------------------------------------------------
// Row-wise ops
// ---------------------------------------------------------------------------
// y = (x - mean) / sqrt(var + 1e-5) * gamma   (nn.LayerNorm(D, bias=False))
void launch_layernorm(const float* x, float* y, const float* gamma, int64_t rows, int D,
                      cudaStream_t stream);
// In-place softmax over the first n_z columns of each row of group z's
// [m_z, ld] score matrix; columns [n_z, ld) are zeroed.
// win_past >= 0 restricts row m to columns m - win_past .. m + win_future (inclusive, the streaming
// encoder's sliding window); columns outside get probability 0.
void launch_softmax_rows(float* S, const int64_t* offS, const int* Mz, const int* Nz, int ld,
                         int groups, int max_m, cudaStream_t stream, int win_past = -1, int win_future = 0);

// ---------------------------------------------------------------------------
// Fused encoder self-attention (attention_tc.cu): per group z = (utterance, head)
//   out_z[m, 0:hd] = softmax_k(scale * Q_z[m] . K_z[k]) V_z[k]      m, k < T_z
// Q_z / K_z rows live in one array with row stride ldqk, V_z is given transposed ([hd][ldv], keys contiguous).
// win_past >= 0 restricts query m to keys m - win_past .. m + win_future (inclusive).
// ---------------------------------------------------------------------------
struct AttnParams {
  const float* qk = nullptr;
  const float* vt = nullptr;
  float* out = nullptr;
  const int64_t* offQ = nullptr;
  const int64_t* offK = nullptr;
  const int64_t* offV = nullptr;
  const int64_t* offO = nullptr;
  const int* Tz = nullptr;
  int ldqk = 0, ldv = 0, ldo = 0, hd = 0;
  float scale = 1.0f;
  int win_past = -1, win_future = 0;
};
// true when every query tile's key range fits the kernel's TMEM budget (448 score columns)
bool attention_tc_supported(int max_t, int hd, int win_past, int win_future);
void launch_attention_tc(const AttnParams& p, int groups, int max_t, cudaStream_t stream);

// ---------------------------------------------------------------------------
// Streaming frontend / adapter
// ---------------------------------------------------------------------------
// Per 80-sample frame: CMVN ((x - mean) / sqrt(mean((x - mean)^2) + 1e-6)), then asinh(k * x).
// Frame f of utterance b is read at pcm + b * stride + f * 80 and written to out row
// row0[b] + f (80 floats per row).
void launch_stream_frames(const float* pcm, int64_t pcm_stride, const int* n_frames, const int64_t* row0,
                          float k, float* out, int B, int max_frames, cudaStream_t stream);
// y[r] = x[r] + table[pos[r]]  (rows of width D)
void launch_add_rows_by_index(const float* x, const float* table, const int* pos, float* y, int64_t rows,
                              int D, cudaStream_t stream);
void launch_gelu_inplace(float* x, int64_t n, cudaStream_t stream);

// ---------------------------------------------------------------------------
// Decoder (persistent, one launch per greedy token)
// ---------------------------------------------------------------------------
struct DecLayerWeights {
  const float* ln1;    // [D]
  const float* wqkv;   // [H][D][3*hd]  k-major per head: (q | k | v) columns
  const float* wo;     // [H][hd][D]    rows of o_proj^T belonging to head h
  const float* ln2;
  const float* wqc;    // [H][D][hd]
  const float* woc;    // [H][hd][D]
  const float* ln3;
  const float* w1;     // [n_chunk][D][2*IC]  (up | gate) columns of the chunk
  const float* b1;     // [n_chunk][2*IC]
  const float* w2;     // [n_chunk][IC][D]
  const float* b2;     // [D]
  // The same blocks as tensor-core operands for the v2 kernel (decoder_plane_bytes(N, K) bytes per block):
  // bf16 hi / lo planes in UMMA K-major SWIZZLE_64B order, [m-tile of <= 128 output features][k-block of 32]
  // [hi | lo][rows padded to 8][32 bf16] -- a ring stage receives whole k-blocks by one bulk copy.
  const unsigned char* wqkvP;  // [H] blocks N = 3*hd, K = D
  const unsigned char* woP;    // [H] blocks N = D,    K = hd
  const unsigned char* wqcP;   // [H] blocks N = hd,   K = D
  const unsigned char* wocP;   // [H] blocks N = D,    K = hd
  const unsigned char* w1P;    // [n_chunk] blocks N = 2*IC, K = D
  const unsigned char* w2P;    // [n_chunk] blocks N = D,    K = IC
  // v3 kernel (weight-stationary GEMM jobs): whole matrices as plane-packed m-tiles of 128 output features
  const unsigned char* wocF;   // one block N = D, K = D           (cross-attention output projection)
  const unsigned char* w1iF;   // one block N = 2*I, K = D         rows interleaved: 2j = value j, 2j+1 = gate j
  const float* b1i;            // [2*I] fc1 bias in the same interleaved order
  const unsigned char* w2kF;   // [ffn_ksplit] blocks N = D, K = I / ffn_ksplit  (k-slices of fc2)
  // v4 kernel (cluster-resident layers): fp32 k-major slices per cluster rank r (CS ranks)
  const float* c4_wo;          // [CS][D][dsp]      output features r*D/CS .. of the self-attention output projection
  const float* c4_woc;         // [CS][D][dsp]      the same for the cross-attention output projection
  const float* c4_w1;          // [CS][D][2*I/CS]   fc1 columns of the rank's FFN slice, (value j, gate j) interleaved, x ln3 gamma
  const float* c4_b1;          // [CS][2*I/CS]
  const float* c4_w2;          // [CS][I/CS][D]     fc2 rows (inputs) of the rank's FFN slice
};
// bytes of one plane-packed [N][K] block
inline size_t decoder_plane_bytes(int N, int K) {
  const int nkb = (K + 31) / 32;
  size_t rows = 0;
  for (int n0 = 0; n0 < N; n0 += 128) rows += (size_t)(((N - n0 < 128 ? N - n0 : 128) + 7) & ~7);
  return rows * nkb * 128;
}

constexpr int kMaxDecLayers = 8;

struct DecoderParams {
  int B, D, H, hd, I, V, L, rot_dim;
  int step;               // decode position of the token being consumed
  int Tpad;               // cross K/V time padding (multiple of 8)
  int Smax;               // self K/V capacity (positions)
  int IC;                 // FFN columns per MLP work item (divides I)
  int n_chunk;            // I / IC
  int n_vchunk;           // vocab chunks in the logits phase
  int vchunk;             // vocab entries per chunk
  DecLayerWeights layers[kMaxDecLayers];
  const float* embed;     // [V][D]   (gather)
  const float* embT;      // [D][V]   (tied logits head, k-major)
  const void* embP;       // v2-v4 logits slab: bf16 hi/lo planes in UMMA K-major SWIZZLE_64B order,
                          // [n_vchunk][m-tile][k-block of 32][plane][rows][32] (see Model::build_weights)
  int smem_limit;         // opt-in shared memory per CTA (v2-v4 shared-memory layouts)
  void* prof;             // optional [grid][512] u64 timestamps (v2-v4 kernels, debugging)
  const float* final_ln;  // [D]
  const float* rope_cos;  // [Smax][rot/2]
  const float* rope_sin;
  const int* enc_len;     // [B] cross length T_b
  const int* max_len;     // [B] max decode steps per utterance
  const __half* kc;       // [L][B][H][hd][Tpad]   cross K, d-major
  const __half* vc;       // [L][B][H][Tpad][hd]   cross V
  float* ks;              // [L][B][H][hd][Smax]   self K, d-major
  float* vs;              // [L][B][H][Smax][hd]   self V
  float* hbuf;            // [2][B][D]  residual stream (ping-pong)
  float* part;            // [2H + n_chunk][B][D] partial sums (A | B | C)
  float* xfin;            // [B][D] final-LN rows feeding the logits phase
  float* cand_val;        // [2][n_vchunk][B]  per-chunk argmax candidates (ping-pong by step parity)
  int* cand_idx;          // [2][n_vchunk][B]
  int* tokens;            // [B][Smax + 1] emitted ids (index 0 = start token)
  int* n_tokens;          // [B] ids emitted so far (incl. start token)
  int* done;              // [B]
  int* n_active;          // [1] utterances still decoding (updated at step start)
  float* logits_out;      // optional [B][V] dump of this step's logits (parity/debug)
  const int* forced;      // optional [B][Smax + 1] teacher-forced ids
  float* xattn_out;       // optional [B][L][H][xattn_steps][Tpad] cross-attention probabilities (word timestamps)
  int xattn_steps;
  unsigned int* barrier;  // [2] grid barrier state
  // ---- v3 kernel ----
  int nb_self, nb_cross;  // utterances per attention job
  int nx;                 // utterances per GEMM job (multiple of 16, <= 64)
  int ffn_ksplit;         // k-slices of fc2 (partial sums resolved by the next consumer)
  int job_first[8], job_ncta[8];  // per phase kind: job j runs on CTA (first + j % ncta) % grid
  float* attc;            // [B][D] cross-attention output (all heads), input of the output projection
  float* act;             // [B][I] silu(gate) * value
  unsigned int* sync3;    // [kSync3Words] epoch, error flag, one completion counter per phase (own 128-byte line)
  // sparse logit bonuses added in the logits epilogue before the fused argmax (key-term biasing,
  // reference: ContextBiaser::apply, core/context-biaser.cpp:88-132); all null = no biasing
  int c4_cs, c4_nc, c4_u;     // v4: cluster size, clusters, utterances per cluster
  // ---- explicit rows (v3 only; multi-token verify and per-utterance positions; reference: run_decoder_with_cross_kv
  // fed n > 1 tokens by decode_tokens / decode_full, core/moonshine-streaming-model.cpp:1136-1190, 1192-1397).  A row is
  // one (utterance, position) pair; rows of one utterance are consecutive, ascending in position, and never straddle a
  // self-attention tile.  All null = row b is utterance b at position `step` (the lockstep greedy loop).
  const int* row_tok;         // [B] input id of the row; < 0: the row idles this launch
  const int* row_pos;         // [B] decode position (RoPE, K/V append slot, attention length - 1)
  const int* row_nin;         // [B] how many rows directly before this one belong to the same utterance in THIS launch
  const int* row_utt;         // [B] utterance of the row (self / cross caches, encoder length)
  int B_utt;                  // utterances behind the caches (= B when the row arrays are null)
  int row_group;              // rows per utterance slot (self-attention tiles hold a multiple of it)
  const float* bias_static;   // [V] bonus shared by every utterance and step (the trie root's children)
  const int* bias_dyn_n;      // [B] per-utterance entries of this step
  const int* bias_dyn_ids;    // [B][bias_dyn_cap] token ids
  const float* bias_dyn_val;  // [B][bias_dyn_cap] bonus ON TOP of bias_static[id]
  int bias_dyn_cap;
};
constexpr int kSync3Words = 32 + 32 * 64;
void launch_decoder_step3(const DecoderParams& p, int grid, cudaStream_t stream);
// explicit-row decoding (v3): per-utterance state of a verify-then-continue decode, all device pointers
struct VerifyState {
  int* mode;             // [B_utt] 0 verifying the draft, 1 auto-regressive, 2 done
  int* pos;              // [B_utt] next position to feed
  int* cur;              // [B_utt] next input id in auto-regressive mode
  int* prev_n;           // [B_utt] rows the previous launch ran for the utterance
  const int* draft;      // [B_utt][draft_stride] draft ids (no BOS / EOS)
  const int* draft_len;  // [B_utt]
  int draft_stride;
};
// books launch k-1 and writes the rows of launch k (p: explicit-row parameters, p.B = B_utt * n rows)
// seeds the argmax candidates of parity `parity` so that the lockstep kernels resolve utterance b's previous id to cur[b]
void launch_decoder_seed_candidates(const DecoderParams& p, const int* cur, int parity, cudaStream_t stream);
void launch_decoder_verify_plan(const DecoderParams& p, const VerifyState& s, int k, int n, int bos, int eos, cudaStream_t stream);
size_t decoder_step3_smem_bytes(const DecoderParams& p);
// fills nb_self / nb_cross / nx / job_first / job_ncta for batch size p.B on a grid of `grid` CTAs
void decoder_step3_plan(DecoderParams& p, int grid);
bool decoder_step3_supported(const DecoderParams& p);
// v4: cluster-resident layers for small batches (<= 8 utterances per cluster of 16 or 8 CTAs)
int decoder_step4_cluster_size(int device, int heads, size_t smem_hint, int* clusters);  // 16, 8 or 0 (none)
bool decoder_step4_supported(const DecoderParams& p);
void decoder_step4_plan(DecoderParams& p);
size_t decoder_step4_smem_bytes(const DecoderParams& p);
void launch_decoder_step4(const DecoderParams& p, cudaStream_t stream);
// out[b] = id emitted by the step that was just launched (p.step), resolved from its argmax candidates with the
// reference's lowest-index tie rule; the next launch's prologue resolves the same value on its own.
void launch_decoder_resolve(const DecoderParams& p, int* out, cudaStream_t stream);
void launch_decoder_step(const DecoderParams& p, int grid, cudaStream_t stream);
// v2: operands streamed through a TMA-bulk smem ring by a producer warp.
void launch_decoder_step2(const DecoderParams& p, int grid, cudaStream_t stream);
size_t decoder_step2_smem_bytes(const DecoderParams& p);
void decoder_tiles_for_batch(int B, int& nb_attn, int& nb_mlp);
size_t decoder_step_smem_bytes(const DecoderParams& p);
// Resolves the last step's argmax into tokens[] (the step kernel resolves the
// previous step's candidates in its prologue).
void launch_decoder_finalize(const DecoderParams& p, cudaStream_t stream);

// Microbenchmark (ring_bench.cu): ms for every CTA of `grid` to stream bytes_per_cta through a bulk-copy ring.
float ring_bandwidth_test(int64_t bytes_per_cta, int stage_bytes, int stages, int nsub, int shared_src, int grid);

}  // namespace msb
