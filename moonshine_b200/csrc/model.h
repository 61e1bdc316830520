// Device-side Moonshine model: weights in HBM + batched encoder / greedy
// decoder.  This is the B200 replacement of the reference's MoonshineModel
// (core/moonshine-model.{h,cpp}): same contract per utterance (PCM in ->
// token ids out, start token 1, EOS 2 appended, at most
// ceil(seconds * max_tokens_per_second) generated ids), but for a ragged
// batch of utterances at once.
#pragma once
#include <cstdint>
#include <memory>
#include <utility>
#include <vector>

#include "common.h"
#include "kernels.h"
#include "weights.h"

namespace msb {

struct DebugCapture {
  // Filled when non-null / true.
  std::vector<float>* encoder_out = nullptr;     // packed [sum T_b][D]
  std::vector<int>* encoder_frames = nullptr;    // T_b
  std::vector<float>* logits = nullptr;          // [steps][B][V]
  int logits_steps = 0;                          // capture the first N steps
  const int32_t* forced = nullptr;               // [B][forced_stride] teacher-forced ids (incl. start)
  int forced_stride = 0;
  bool skip_decode = false;
  int rows_per_launch = 0;                       // > 1 with `forced`: teacher-forced MULTI-token decoder runs (decode_tokens,
                                                 // moonshine-streaming-model.cpp:1136-1190): this many positions per launch
};

// Streaming architectures: what the host bookkeeping (Transcriber, mirroring
// core/transcriber.cpp:1331-1395) decided for each segment of the batch.  n_samples[b] passed beside it
// is the number of ANALYSED samples (whole 1280-sample chunks).
struct StreamPlan {
  const int* emitted = nullptr;     // [B] encoder features that form the decoder memory (<= analysed / 320)
  const int* max_tokens = nullptr;  // [B] decode budget
  // Speculative drafts (reference: decode_full's speculative_tokens, moonshine-streaming-model.cpp:1192-1197): the ids
  // of the previous decode of the same open segment, no BOS / EOS.  Verified kVerifyRows positions per launch on the
  // explicit-row decoder; the result equals the greedy decode id for id.  Null / length 0 = plain greedy.
  const int* const* draft = nullptr;  // [B] host pointers
  const int* draft_len = nullptr;     // [B]
};
constexpr int kVerifyRows = 8;  // draft positions verified per utterance per launch

// Decoder cross-attention of one utterance, as align_words consumes it: [layers * heads][steps][frames]
// (layer-major), steps = decoder runs = generated ids, frames = encoder memory length.
struct CrossAttention {
  int heads_total = 0, steps = 0, frames = 0;
  std::vector<float> prob;
};

// Host-side logit hook (key-term biasing; reference: ContextBiaser applied between decode_step and the argmax,
// core/transcriber.cpp:1440-1470).  When one is given, decoding is stepped from the host: every launch dumps
// the step's logits, the hook edits them, the host takes the first-max argmax and feeds the id to the next
// launch through the teacher-forcing input.
struct LogitHook {
  virtual ~LogitHook() = default;
  virtual void apply(int utterance, float* logits, int vocab) = 0;  // before the argmax of every step
  virtual void advance(int utterance, int token) = 0;               // after a non-EOS id was emitted
  // Sparse form, used by the on-device path (v3 kernel: the bonuses are added in the logits epilogue before the
  // fused argmax, nothing but B token ids crosses PCIe per step).  shared_bonus: the bonuses that hold for every
  // utterance at every step as a dense [vocab] array (nullptr = this hook has no sparse form: host-stepped path);
  // step_bonus: this step's extra bonuses of one utterance, ON TOP of the shared ones, as (token id, bonus).
  virtual const std::vector<float>* shared_bonus(int vocab) { (void)vocab; return nullptr; }
  virtual void step_bonus(int utterance, std::vector<std::pair<int32_t, float>>& out) { (void)utterance; out.clear(); }
};

struct StageTimes {
  float frontend_ms = 0, encoder_ms = 0, cross_kv_ms = 0, decode_ms = 0;
  int decode_steps = 0;
  int decode_launches = 0;
  int kernel_launches = 0;
  int decoder_version = 0;   // step kernel that ran: 1, 2, 3 (weight-stationary jobs) or 4 (cluster-resident layers)
};

class Model {
 public:
  Model(const Dims& dims, const WeightFile& weights, int device);
  // Replica on another device: the packed weight blob is copied device-to-device (cudaMemcpyPeer: NVLink when the
  // devices are peers) instead of being rebuilt and uploaded from the host -- the one weight broadcast of SURVEY 8(e).
  Model(const Model& src, int device);
  ~Model();

  const Dims& dims() const { return d_; }
  int device() const { return device_; }
  cudaStream_t stream() const { return stream_; }

  // Host PCM (16 kHz mono float).  Copies to the device inside the call.
  void transcribe(const float* const* pcm, const uint64_t* n_samples, int B,
                  float max_tokens_per_second, std::vector<std::vector<int32_t>>& tokens,
                  DebugCapture* dbg = nullptr, const StreamPlan* plan = nullptr,
                  std::vector<CrossAttention>* xattn = nullptr, LogitHook* hook = nullptr);
  // Device-resident PCM: row b at d_pcm + b * stride.
  void transcribe_device(const float* d_pcm, int64_t stride, const uint64_t* n_samples, int B,
                         float max_tokens_per_second, std::vector<std::vector<int32_t>>& tokens,
                         DebugCapture* dbg = nullptr, const StreamPlan* plan = nullptr);
  // Streaming bookkeeping for a one-shot call on a complete segment of n samples
  // (core/transcriber.cpp:1331-1390): analysed samples, emitted features, greedy token budget.
  void one_shot_stream_plan(uint64_t n_samples, float max_tokens_per_second, uint64_t& analysed, int& emitted,
                            int& max_tokens) const;

  // reference rule: core/moonshine-model.cpp:347-349
  static int max_len_for(uint64_t n_samples, float max_tokens_per_second);

  const StageTimes& last_times() const { return times_; }
  void set_timing(bool on) { timing_ = on; }
  // parity hook: plan-less calls on a streaming model act as a NON-final update (look-ahead held back)
  void set_debug_stream_partial(bool on) { debug_stream_partial_ = on; }
  // speculative drafts for the next transcribe() whose plan carries none (moonshine_b200_decode_with_drafts)
  void set_debug_drafts(const int* const* draft, const int* len) { dbg_draft_ = draft; dbg_draft_len_ = len; }
  size_t weight_bytes() const { return wblob_.bytes(); }

 private:
  struct EncLayer {
    const float *ln1, *wqk, *wv, *wo, *ln2, *w1, *b1, *w2, *b2;
    const unsigned char *wqkP, *woP, *w1P, *w2P;  // the dense weights as bf16 hi/lo plane tiles (gemm_planes.cu), or null
  };
  bool enc_planes_ = false;  // encoder dense layers on the plane-fed tcgen05 GEMM
  void build_weights(const WeightFile& wf);
  void ensure_rope(int max_pos);
  struct AutoPlan {
    std::vector<uint64_t> analysed;
    std::vector<int> emitted, max_tokens;
    StreamPlan plan;
  };
  // plan-less call on a streaming model: one-shot bookkeeping per utterance
  const StreamPlan* auto_plan(const uint64_t*& n_samples, int B, float max_tps, AutoPlan& ap) const;
  void run(const float* d_pcm, int64_t stride, const uint64_t* n_samples, int B, float max_tps,
           std::vector<std::vector<int32_t>>& tokens, DebugCapture* dbg, const StreamPlan* plan,
           std::vector<CrossAttention>* xattn = nullptr, LogitHook* hook = nullptr);

  Dims d_;
  int device_ = 0;
  int sm_count_ = 0;
  cudaStream_t stream_ = nullptr;
  bool timing_ = false;
  bool debug_stream_partial_ = false;
  bool stream_dirty_ = false;  // a run() left work on the stream without the closing synchronise (exception path)
  StageTimes times_;
  cudaEvent_t ev_[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};

  // weights
  DeviceBuffer<float> wblob_;
  const float *w1t_ = nullptr, *gn_w_ = nullptr, *gn_b_ = nullptr;
  const float *conv2_w_ = nullptr, *conv2_b_ = nullptr, *conv3_w_ = nullptr, *conv3_b_ = nullptr;
  std::vector<EncLayer> enc_;
  const float* enc_final_ln_ = nullptr;
  // streaming frontend / adapter (null for the classic architectures)
  const float *s_lin_w_ = nullptr, *s_c1_w_ = nullptr, *s_c1_b_ = nullptr, *s_c2_w_ = nullptr, *s_c2_b_ = nullptr;
  const float *pos_emb_ = nullptr, *proj_w_ = nullptr;
  float s_k_ = 1.0f;  // exp(log_k) of the asinh compression
  const float *wk_all_ = nullptr, *wv_all_ = nullptr;
  DecoderParams dec_{};  // weight pointers + dims prefilled
  int ffn_chunk_ = 64;
  int vchunk_ = 0, n_vchunk_ = 0, smem_optin_ = 0;
  int ffn_ksplit_ = 1;
  int c4_cs_ = 0;   // cluster size of the v4 decoder kernel (0: not used)
  int c4_nc_ = 0;   // co-resident clusters of that size

  // rope tables (grow-only)
  DeviceBuffer<float> rope_cos_, rope_sin_;
  int rope_positions_ = 0;

  // workspaces (grow-only)
  DeviceBuffer<float> pcm_dev_, h1_, h2_, x_, ln_, qk_, vt_, scores_, attn_, mid_, enc_out_, frames_;
  DeviceBuffer<float> lnP_, attnP_, midP_, a2P_, a3P_, encP_;  // activations as plane tiles (byte buffers; sized in floats)
  const unsigned char* conv2P_ = nullptr;  // conv2 / conv3 weights as plane tiles (classic frontend)
  const unsigned char* conv3P_ = nullptr;
  const unsigned char* wkvP_ = nullptr;    // stacked cross K | V projections of every decoder layer as plane tiles
  DeviceBuffer<double> gn_partial_;
  DeviceBuffer<__half> kc_, vc_;
  DeviceBuffer<float> ks_, vs_, hbuf_, part_, xfin_, cand_val_, logits_dbg_, xattn_dev_;
  DeviceBuffer<int> cand_idx_, tokens_dev_, ntok_dev_, done_dev_, forced_dev_;
  DeviceBuffer<int> meta_i32_;       // packed int32 metadata
  DeviceBuffer<int64_t> meta_i64_;   // packed int64 metadata
  DeviceBuffer<unsigned int> barrier_, sync3_;
  DeviceBuffer<float> attc_, act_, bias_static_dev_, bias_val_dev_;
  DeviceBuffer<int> bias_n_dev_, bias_ids_dev_, step_tok_dev_;
  PinnedBuffer<int> pin_bias_i32_;
  PinnedBuffer<float> pin_bias_f32_;
  DeviceBuffer<int> nactive_;
  DeviceBuffer<int> rows_dev_, vstate_dev_, draft_dev_;  // explicit-row decoding (speculative verify)
  DeviceBuffer<float> logits_rows_;                      // [rows][V] logits of one explicit-row launch (decode_tokens)
  const int* const* dbg_draft_ = nullptr;                // drafts for the NEXT run() when its plan carries none (test entry)
  const int* dbg_draft_len_ = nullptr;
  PinnedBuffer<int> pin_i32_;
  PinnedBuffer<int64_t> pin_i64_;
  PinnedBuffer<float> pin_pcm_;
  PinnedBuffer<int> pin_tokens_;
  PinnedBuffer<float> pin_logits_;
};

}  // namespace msb
