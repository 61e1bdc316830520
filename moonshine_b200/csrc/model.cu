// Host orchestration of the batched encoder and the greedy decoder.
#include "model.h"

#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include <algorithm>
#include <cmath>
#include <chrono>
#include <cstring>

namespace msb {

namespace {

// Appends tensors to one host blob (256-byte aligned) that is uploaded once.
struct BlobBuilder {
  std::vector<float> data;
  size_t add(size_t count) {
    size_t off = (data.size() + 63) / 64 * 64;
    data.resize(off + count, 0.f);
    return off;
  }
  size_t add_copy(const float* src, size_t count) {
    size_t off = add(count);
    std::memcpy(data.data() + off, src, count * sizeof(float));
    return off;
  }
};

int round_up(int x, int m) { return (x + m - 1) / m * m; }

uint16_t bf16_round(float x) {
  uint32_t u;
  std::memcpy(&u, &x, 4);
  if ((u & 0x7f800000u) == 0x7f800000u) return (uint16_t)(u >> 16);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
float bf16_value(uint16_t h) {
  const uint32_t u = (uint32_t)h << 16;
  float f;
  std::memcpy(&f, &u, 4);
  return f;
}

// Packs W[n][k] (n < N output features, k < K inputs; `get(n, k)`) as the tcgen05 A operand the v2 decoder
// streams: per m-tile of <= 128 features and k-block of 32 inputs a bf16 hi plane and a bf16 lo plane,
// [rows padded to 8][64 B], 16-byte chunk c of row r at position c ^ ((r >> 1) & 3) (K-major SWIZZLE_64B).
template <typename Get>
size_t pack_planes(BlobBuilder& bb, int N, int K, Get get) {
  const size_t bytes = decoder_plane_bytes(N, K);
  const size_t off = bb.add((bytes + 3) / 4);
  uint16_t* P = reinterpret_cast<uint16_t*>(&bb.data[off]);
  const int nkb = (K + 31) / 32;
  size_t o = 0;  // in uint16 units
  for (int n0 = 0; n0 < N; n0 += 128) {
    const int R = std::min(128, N - n0), Rp = (R + 7) & ~7;
    for (int kb = 0; kb < nkb; kb++) {
      uint16_t* hi = P + o;
      uint16_t* lo = hi + (size_t)Rp * 32;
      for (int r = 0; r < R; r++)
        for (int kk = 0; kk < 32; kk++) {
          const int k = kb * 32 + kk;
          const float x = k < K ? get(n0 + r, k) : 0.f;
          const uint16_t h = bf16_round(x);
          const uint16_t l = bf16_round(x - bf16_value(h));
          const size_t at = (size_t)r * 32 + (size_t)(((kk >> 3) ^ ((r >> 1) & 3)) * 8 + (kk & 7));
          hi[at] = h;
          lo[at] = l;
        }
      o += (size_t)Rp * 64;
    }
  }
  return off;
}

// W[n][k] as full 128-row plane tiles (gemm_planes.cu: tile (n / 128, k / 32) = [hi 8 KB | lo 8 KB], zero-padded rows)
template <typename Get>
size_t pack_tile_planes(BlobBuilder& bb, int N, int K, Get get) {
  const size_t bytes = plane_tiles_bytes(N, K);
  const size_t off = bb.add(bytes / 4);
  uint16_t* P = reinterpret_cast<uint16_t*>(&bb.data[off]);
  std::memset(P, 0, bytes);
  const int nkb = K / 32;
  for (int n = 0; n < N; n++) {
    const int r = n & 127;
    for (int kb = 0; kb < nkb; kb++) {
      uint16_t* hi = P + ((size_t)(n >> 7) * nkb + kb) * (kPlaneTileBytes / 2);
      uint16_t* lo = hi + kPlaneTileBytes / 4;
      for (int kk = 0; kk < 32; kk++) {
        const float x = get(n, kb * 32 + kk);
        const uint16_t h = bf16_round(x);
        const uint16_t l = bf16_round(x - bf16_value(h));
        const size_t at = (size_t)r * 32 + (size_t)(((kk >> 3) ^ ((r >> 1) & 3)) * 8 + (kk & 7));
        hi[at] = h;
        lo[at] = l;
      }
    }
  }
  return off;
}

}  // namespace

int Model::max_len_for(uint64_t n_samples, float max_tokens_per_second) {
  // `const float audio_duration = size / 16000.0f; ceil(duration * tps)`
  const float audio_duration = (float)n_samples / 16000.0f;
  return (int)std::ceil(audio_duration * max_tokens_per_second);
}

Model::Model(const Dims& dims, const WeightFile& weights, int device) : d_(dims), device_(device) {
  CUDA_CHECK(cudaSetDevice(device_));
  cudaDeviceProp prop;
  CUDA_CHECK(cudaGetDeviceProperties(&prop, device_));
  if (prop.major < 10) {
    throw std::runtime_error(format("moonshine-b200 requires an sm_100a GPU, found sm_%d%d (%s)",
                                    prop.major, prop.minor, prop.name));
  }
  sm_count_ = prop.multiProcessorCount;
  CUDA_CHECK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  for (auto& e : ev_) CUDA_CHECK(cudaEventCreate(&e));
  if (d_.dec_layers > kMaxDecLayers) throw std::runtime_error("too many decoder layers");
  CUDA_CHECK(cudaDeviceGetAttribute(&smem_optin_, cudaDevAttrMaxSharedMemoryPerBlockOptin, device_));
  {
    // v4 (cluster-resident layers) serves small batches of small models: every cluster streams all layer weights,
    // so they have to stay L2-resident next to the streamed cross K/V
    const double layer_mb = (double)d_.dec_layers * (4.0 * d_.dim * d_.dim + 3.0 * d_.dim * d_.ffn) * 4.0 / 1e6;
    c4_cs_ = 0;
    if (layer_mb <= 48.0 && d_.dim % 32 == 0)
      c4_cs_ = decoder_step4_cluster_size(device_, d_.heads, (size_t)smem_optin_, &c4_nc_);
    if (c4_cs_ > 0 && (d_.dim % c4_cs_ || d_.ffn % c4_cs_ || ((2 * d_.ffn / c4_cs_) % 4) || c4_cs_ % d_.heads)) c4_cs_ = 0;
  }
  {
    // vocab chunks of the logits phase: one per CTA of the kernel that will run it (128 with clusters, else one per SM)
    const int ctas = c4_cs_ > 0 ? c4_cs_ * c4_nc_ : sm_count_;
    int per = (d_.vocab + ctas - 1) / ctas;
    per = round_up(std::max(per, 32), 32);
    if (per > 384) per = 384;   // <= 3 m-tiles of 128 vocab rows per chunk
    vchunk_ = per;
    n_vchunk_ = (d_.vocab + per - 1) / per;
  }
  build_weights(weights);
  barrier_.reserve(2);
  CUDA_CHECK(cudaMemsetAsync(barrier_.ptr, 0, 2 * sizeof(unsigned), stream_));
  nactive_.reserve(1);
  CUDA_CHECK(cudaStreamSynchronize(stream_));
}

Model::Model(const Model& src, int device) : d_(src.d_), device_(device) {
  CUDA_CHECK(cudaSetDevice(device_));
  cudaDeviceProp prop;
  CUDA_CHECK(cudaGetDeviceProperties(&prop, device_));
  if (prop.major < 10) throw std::runtime_error(format("moonshine-b200 requires an sm_100a GPU, device %d is sm_%d%d", device_, prop.major, prop.minor));
  sm_count_ = prop.multiProcessorCount;
  CUDA_CHECK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  for (auto& e : ev_) CUDA_CHECK(cudaEventCreate(&e));
  CUDA_CHECK(cudaDeviceGetAttribute(&smem_optin_, cudaDevAttrMaxSharedMemoryPerBlockOptin, device_));
  ffn_chunk_ = src.ffn_chunk_; ffn_ksplit_ = src.ffn_ksplit_; vchunk_ = src.vchunk_; n_vchunk_ = src.n_vchunk_;
  s_k_ = src.s_k_;
  c4_cs_ = src.c4_cs_; c4_nc_ = src.c4_nc_;
  if (c4_cs_ > 0) {  // the weight layouts follow the source's cluster shape: this device must host it too
    int nc = 0;
    const int cs = decoder_step4_cluster_size(device_, d_.heads, (size_t)smem_optin_, &nc);
    if (cs != c4_cs_ || nc < c4_nc_) throw std::runtime_error("replica device cannot host the source device's cluster shape");
  }
  if (sm_count_ != src.sm_count_ && c4_cs_ == 0) throw std::runtime_error("replica device has a different SM count");
  // the one weight transfer: device to device
  wblob_.reserve(src.wblob_.count);
  int can = 0;
  if (device_ != src.device_ && cudaDeviceCanAccessPeer(&can, device_, src.device_) == cudaSuccess && can) {
    cudaDeviceEnablePeerAccess(src.device_, 0);  // already-enabled is fine
    cudaGetLastError();
  }
  CUDA_CHECK(cudaMemcpyPeerAsync(wblob_.ptr, device_, src.wblob_.ptr, src.device_, src.wblob_.bytes(), stream_));
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  // every weight pointer is an offset into the blob: rebase
  const char* ob = reinterpret_cast<const char*>(src.wblob_.ptr);
  const char* nb = reinterpret_cast<const char*>(wblob_.ptr);
  auto rb = [&](const float* q) -> const float* {
    return q == nullptr ? nullptr : reinterpret_cast<const float*>(nb + (reinterpret_cast<const char*>(q) - ob));
  };
  auto rbb = [&](const unsigned char* q) -> const unsigned char* {
    return q == nullptr ? nullptr : reinterpret_cast<const unsigned char*>(nb + (reinterpret_cast<const char*>(q) - ob));
  };
  w1t_ = rb(src.w1t_); gn_w_ = rb(src.gn_w_); gn_b_ = rb(src.gn_b_);
  conv2_w_ = rb(src.conv2_w_); conv2_b_ = rb(src.conv2_b_); conv3_w_ = rb(src.conv3_w_); conv3_b_ = rb(src.conv3_b_);
  conv2P_ = rbb(src.conv2P_); conv3P_ = rbb(src.conv3P_); wkvP_ = rbb(src.wkvP_);
  enc_final_ln_ = rb(src.enc_final_ln_);
  s_lin_w_ = rb(src.s_lin_w_); s_c1_w_ = rb(src.s_c1_w_); s_c1_b_ = rb(src.s_c1_b_); s_c2_w_ = rb(src.s_c2_w_); s_c2_b_ = rb(src.s_c2_b_);
  pos_emb_ = rb(src.pos_emb_); proj_w_ = rb(src.proj_w_);
  wk_all_ = rb(src.wk_all_); wv_all_ = rb(src.wv_all_);
  enc_ = src.enc_;
  for (EncLayer& e : enc_) {
    e.ln1 = rb(e.ln1); e.wqk = rb(e.wqk); e.wv = rb(e.wv); e.wo = rb(e.wo); e.ln2 = rb(e.ln2);
    e.w1 = rb(e.w1); e.b1 = rb(e.b1); e.w2 = rb(e.w2); e.b2 = rb(e.b2);
    e.wqkP = rbb(e.wqkP); e.woP = rbb(e.woP); e.w1P = rbb(e.w1P); e.w2P = rbb(e.w2P);
  }
  enc_planes_ = src.enc_planes_;
  dec_ = src.dec_;
  dec_.embed = rb(src.dec_.embed); dec_.embT = rb(src.dec_.embT); dec_.final_ln = rb(src.dec_.final_ln);
  dec_.embP = rbb(reinterpret_cast<const unsigned char*>(src.dec_.embP));
  dec_.smem_limit = smem_optin_;
  for (int l = 0; l < d_.dec_layers; l++) {
    DecLayerWeights& w = dec_.layers[l];
    const DecLayerWeights& o = src.dec_.layers[l];
    w.ln1 = rb(o.ln1); w.wqkv = rb(o.wqkv); w.wo = rb(o.wo); w.ln2 = rb(o.ln2); w.wqc = rb(o.wqc); w.woc = rb(o.woc);
    w.ln3 = rb(o.ln3); w.w1 = rb(o.w1); w.b1 = rb(o.b1); w.w2 = rb(o.w2); w.b2 = rb(o.b2);
    w.wqkvP = rbb(o.wqkvP); w.woP = rbb(o.woP); w.wqcP = rbb(o.wqcP); w.wocP = rbb(o.wocP); w.w1P = rbb(o.w1P); w.w2P = rbb(o.w2P);
    w.wocF = rbb(o.wocF); w.w1iF = rbb(o.w1iF); w.b1i = rb(o.b1i); w.w2kF = rbb(o.w2kF);
    w.c4_wo = rb(o.c4_wo); w.c4_woc = rb(o.c4_woc); w.c4_w1 = rb(o.c4_w1); w.c4_b1 = rb(o.c4_b1); w.c4_w2 = rb(o.c4_w2);
  }
  barrier_.reserve(2);
  CUDA_CHECK(cudaMemsetAsync(barrier_.ptr, 0, 2 * sizeof(unsigned), stream_));
  nactive_.reserve(1);
  CUDA_CHECK(cudaStreamSynchronize(stream_));
}

Model::~Model() {
  cudaSetDevice(device_);
  if (stream_) cudaStreamSynchronize(stream_);
  for (auto& e : ev_)
    if (e) cudaEventDestroy(e);
  if (stream_) cudaStreamDestroy(stream_);
}

void Model::build_weights(const WeightFile& wf) {
  const int D = d_.dim, I = d_.ffn, H = d_.heads, hd = d_.head_dim, V = d_.vocab;
  if (H * hd != D) throw std::runtime_error("heads * head_dim must equal the hidden size");
  if (D % 4 || hd % 4 || I % 4) throw std::runtime_error("dims must be multiples of 4");
  ffn_chunk_ = (I % 64 == 0) ? 64 : (I % 32 == 0) ? 32 : 16;
  if (I % ffn_chunk_) throw std::runtime_error("ffn size must be a multiple of 16");
  const int IC = ffn_chunk_, n_chunk = I / IC;

  BlobBuilder bb;
  const std::string e = "model.encoder.";
  const int E = d_.streaming ? d_.enc_dim : D;      // encoder hidden size
  const int EI = d_.streaming ? d_.enc_ffn : I;
  if (E % 4 || EI % 4 || E % H || (E / H) % 4) throw std::runtime_error("encoder dims must be multiples of 4");
  size_t o_w1t = 0, o_gnw = 0, o_gnb = 0, o_c2 = 0, o_c2b = 0, o_c3 = 0, o_c3b = 0, o_encln = 0, o_conv2P = 0, o_conv3P = 0;
  size_t o_slin = 0, o_sc1 = 0, o_sc1b = 0, o_sc2 = 0, o_sc2b = 0, o_pos = 0, o_proj = 0;
  struct EncOff { size_t ln1, wqk, wv, wo, ln2, w1, b1, w2, b2, wqkP = 0, woP = 0, w1P = 0, w2P = 0; };
  std::vector<EncOff> eo(d_.enc_layers);
  if (!d_.streaming) {
  // conv1 [D][1][127] -> [127][D]
  o_w1t = bb.add((size_t)127 * D);
  {
    const float* w = wf.get(e + "conv1.weight", {D, 1, 127}).data;
    for (int c = 0; c < D; c++)
      for (int j = 0; j < 127; j++) bb.data[o_w1t + (size_t)j * D + c] = w[(size_t)c * 127 + j];
  }
  o_gnw = bb.add_copy(wf.get(e + "groupnorm.weight", {D}).data, D);
  o_gnb = bb.add_copy(wf.get(e + "groupnorm.bias", {D}).data, D);
  // conv2 [2D][D][7] -> [2D][7*D] with K index = k*D + c (channel-last windows)
  o_c2 = bb.add((size_t)2 * D * 7 * D);
  {
    const float* w = wf.get(e + "conv2.weight", {2 * D, D, 7}).data;
    for (int o = 0; o < 2 * D; o++)
      for (int c = 0; c < D; c++)
        for (int k = 0; k < 7; k++)
          bb.data[o_c2 + ((size_t)o * 7 + k) * D + c] = w[((size_t)o * D + c) * 7 + k];
  }
  o_c2b = bb.add_copy(wf.get(e + "conv2.bias", {2 * D}).data, 2 * D);
  o_c3 = bb.add((size_t)D * 3 * 2 * D);
  {
    const float* w = wf.get(e + "conv3.weight", {D, 2 * D, 3}).data;
    for (int o = 0; o < D; o++)
      for (int c = 0; c < 2 * D; c++)
        for (int k = 0; k < 3; k++)
          bb.data[o_c3 + ((size_t)o * 3 + k) * 2 * D + c] = w[((size_t)o * 2 * D + c) * 3 + k];
  }
  o_c3b = bb.add_copy(wf.get(e + "conv3.bias", {D}).data, D);

  for (int l = 0; l < d_.enc_layers; l++) {
    const std::string p = e + "layers." + std::to_string(l) + ".";
    eo[l].ln1 = bb.add_copy(wf.get(p + "input_layernorm.weight", {D}).data, D);
    eo[l].wqk = bb.add((size_t)2 * D * D);
    std::memcpy(&bb.data[eo[l].wqk], wf.get(p + "self_attn.q_proj.weight", {D, D}).data, sizeof(float) * D * D);
    std::memcpy(&bb.data[eo[l].wqk + (size_t)D * D], wf.get(p + "self_attn.k_proj.weight", {D, D}).data, sizeof(float) * D * D);
    eo[l].wv = bb.add_copy(wf.get(p + "self_attn.v_proj.weight", {D, D}).data, (size_t)D * D);
    eo[l].wo = bb.add_copy(wf.get(p + "self_attn.o_proj.weight", {D, D}).data, (size_t)D * D);
    eo[l].ln2 = bb.add_copy(wf.get(p + "post_attention_layernorm.weight", {D}).data, D);
    eo[l].w1 = bb.add_copy(wf.get(p + "mlp.fc1.weight", {I, D}).data, (size_t)I * D);
    eo[l].b1 = bb.add_copy(wf.get(p + "mlp.fc1.bias", {I}).data, I);
    eo[l].w2 = bb.add_copy(wf.get(p + "mlp.fc2.weight", {D, I}).data, (size_t)D * I);
    eo[l].b2 = bb.add_copy(wf.get(p + "mlp.fc2.bias", {D}).data, D);
  }
  o_encln = bb.add_copy(wf.get(e + "layer_norm.weight", {D}).data, D);

  } else {
    // ---- streaming frontend (HF MoonshineStreamingEncoderEmbedder / lora/export.py:53-97) ----
    const std::string em = e + "embedder.";
    s_k_ = std::exp(wf.get(em + "comp.log_k").data[0]);
    o_slin = bb.add_copy(wf.get(em + "linear.weight", {E, 80}).data, (size_t)E * 80);
    // causal convs [C_out][C_in][5] -> [C_out][5 * C_in] with K index = k * C_in + c (channel-last windows)
    auto relayout_conv = [&](const std::string& name, int co, int ci) {
      const float* w = wf.get(name, {co, ci, 5}).data;
      size_t o = bb.add((size_t)co * 5 * ci);
      for (int oc = 0; oc < co; oc++)
        for (int c = 0; c < ci; c++)
          for (int k = 0; k < 5; k++) bb.data[o + ((size_t)oc * 5 + k) * ci + c] = w[((size_t)oc * ci + c) * 5 + k];
      return o;
    };
    o_sc1 = relayout_conv(em + "conv1.weight", 2 * E, E);
    o_sc1b = bb.add_copy(wf.get(em + "conv1.bias", {2 * E}).data, 2 * E);
    o_sc2 = relayout_conv(em + "conv2.weight", E, 2 * E);
    o_sc2b = bb.add_copy(wf.get(em + "conv2.bias", {E}).data, E);
    // unit-offset LayerNorm: y = LN(x) * (gamma + 1)  (HF MoonshineStreamingLayerNorm)
    auto add_gamma1 = [&](const std::string& name) {
      const float* g = wf.get(name, {E}).data;
      size_t o = bb.add(E);
      for (int k = 0; k < E; k++) bb.data[o + k] = g[k] + 1.0f;
      return o;
    };
    for (int l = 0; l < d_.enc_layers; l++) {
      const std::string p = e + "layers." + std::to_string(l) + ".";
      eo[l].ln1 = add_gamma1(p + "input_layernorm.gamma");
      eo[l].wqk = bb.add((size_t)2 * E * E);
      std::memcpy(&bb.data[eo[l].wqk], wf.get(p + "self_attn.q_proj.weight", {E, E}).data, sizeof(float) * E * E);
      std::memcpy(&bb.data[eo[l].wqk + (size_t)E * E], wf.get(p + "self_attn.k_proj.weight", {E, E}).data, sizeof(float) * E * E);
      eo[l].wv = bb.add_copy(wf.get(p + "self_attn.v_proj.weight", {E, E}).data, (size_t)E * E);
      eo[l].wo = bb.add_copy(wf.get(p + "self_attn.o_proj.weight", {E, E}).data, (size_t)E * E);
      eo[l].ln2 = add_gamma1(p + "post_attention_layernorm.gamma");
      eo[l].w1 = bb.add_copy(wf.get(p + "mlp.fc1.weight", {EI, E}).data, (size_t)EI * E);
      eo[l].b1 = bb.add_copy(wf.get(p + "mlp.fc1.bias", {EI}).data, EI);
      eo[l].w2 = bb.add_copy(wf.get(p + "mlp.fc2.weight", {E, EI}).data, (size_t)E * EI);
      eo[l].b2 = bb.add_copy(wf.get(p + "mlp.fc2.bias", {E}).data, E);
    }
    o_encln = add_gamma1(e + "final_norm.gamma");
    // adapter (lora/export.py:130-144): position table + optional projection E -> D
    o_pos = bb.add_copy(wf.get("model.decoder.pos_emb.weight", {d_.max_pos_emb, E}).data, (size_t)d_.max_pos_emb * E);
    if (E != D) o_proj = bb.add_copy(wf.get("model.decoder.proj.weight", {D, E}).data, (size_t)D * E);
  }

  // Encoder dense weights once more as bf16 hi/lo plane tiles: the plane-fed tcgen05 GEMM (gemm_planes.cu) streams them
  // with bulk copies, MMA-ready (same bytes as the fp32 copy, which the unfused / odd-shape paths keep using).
  {
    const int Ee = d_.streaming ? d_.enc_dim : D, EIe = d_.streaming ? d_.enc_ffn : I;
    enc_planes_ = Ee % 32 == 0 && EIe % 32 == 0 && Ee <= 512;
    // (the decoder's stacked cross K | V projections [2 L D][D] are packed after the decoder weights are laid out)
    if (enc_planes_ && !d_.streaming) {  // conv2 [2D][7D] and conv3 [D][6D] (tap-major K, as the fp32 copies)
      const size_t c2 = o_c2, c3 = o_c3;
      o_conv2P = pack_tile_planes(bb, 2 * D, 7 * D, [&](int n, int k) { return bb.data[c2 + (size_t)n * 7 * D + k]; });
      o_conv3P = pack_tile_planes(bb, D, 6 * D, [&](int n, int k) { return bb.data[c3 + (size_t)n * 6 * D + k]; });
    }
    if (enc_planes_) {
      for (int l = 0; l < d_.enc_layers; l++) {
        const size_t wqk = eo[l].wqk, wo = eo[l].wo, w1 = eo[l].w1, w2 = eo[l].w2;
        const size_t wv = eo[l].wv;  // q | k | v rows in one block: one GEMM makes all three
        eo[l].wqkP = pack_tile_planes(bb, 3 * Ee, Ee, [&](int n, int k) {
          return n < 2 * Ee ? bb.data[wqk + (size_t)n * Ee + k] : bb.data[wv + (size_t)(n - 2 * Ee) * Ee + k];
        });
        eo[l].woP = pack_tile_planes(bb, Ee, Ee, [&](int n, int k) { return bb.data[wo + (size_t)n * Ee + k]; });
        eo[l].w1P = pack_tile_planes(bb, EIe, Ee, [&](int n, int k) { return bb.data[w1 + (size_t)n * Ee + k]; });
        eo[l].w2P = pack_tile_planes(bb, Ee, EIe, [&](int n, int k) { return bb.data[w2 + (size_t)n * EIe + k]; });
      }
    }
  }

  // ---- decoder ----
  const std::string dd = "model.decoder.";
  const float* emb_in = wf.get(dd + "embed_tokens.weight", {V, D}).data;   // token embedding
  size_t o_emb = bb.add_copy(emb_in, (size_t)V * D);
  // logits head: the embedding when tied, else proj_out (lora/export.py:206-211)
  const float* emb = (d_.streaming && !d_.tied) ? wf.get("proj_out.weight", {V, D}).data : emb_in;
  // LayerNorm weights are folded into the rows (k index) of the weight block that consumes the
  // normalised activations, so the decoder kernels normalise without an affine step:
  // LN(x) W = ((x - mu) * rstd) (diag(gamma) W).
  const float* gfin = wf.get(dd + "norm.weight", {D}).data;
  size_t o_ones = bb.add(D);
  for (int k = 0; k < D; k++) bb.data[o_ones + k] = 1.0f;
  size_t o_embT = bb.add((size_t)D * V);
  for (int v = 0; v < V; v++)
    for (int k = 0; k < D; k++) bb.data[o_embT + (size_t)k * V + v] = emb[(size_t)v * D + k] * gfin[k];
  // Logits slab for the tcgen05 logits phase: (embedding * final-LN gamma) split into bf16 hi/lo
  // planes, laid out exactly as the UMMA K-major SWIZZLE_64B shared-memory tiles the kernel issues
  // MMAs on: [vocab chunk][m-tile of <=128 rows][k-block of 32][plane hi|lo][row][32 bf16], the 16-byte
  // chunk c of row r stored at position c ^ ((r >> 1) & 3).  A ring stage receives it by one bulk copy.
  const bool dec_tc_layouts = D % 32 == 0;  // the tensor-core decoders (v2, v3, v4) need whole 32-wide k-blocks
  const int n_mt = (vchunk_ + 127) / 128;
  const size_t slab_halfs = (size_t)n_vchunk_ * vchunk_ * D * 2;  // hi + lo
  size_t o_embP = bb.add((slab_halfs + 1) / 2);
  if (dec_tc_layouts) {
    uint16_t* P = reinterpret_cast<uint16_t*>(&bb.data[o_embP]);
    auto bf16_rn = [](float x) -> uint16_t {
      uint32_t u; std::memcpy(&u, &x, 4);
      if ((u & 0x7f800000u) == 0x7f800000u) return (uint16_t)(u >> 16);
      u += 0x7fffu + ((u >> 16) & 1u);
      return (uint16_t)(u >> 16);
    };
    auto bf16_to_f = [](uint16_t h) -> float { uint32_t u = (uint32_t)h << 16; float f; std::memcpy(&f, &u, 4); return f; };
    const int nkb = D / 32;
    for (int ch = 0; ch < n_vchunk_; ch++) {
      size_t chunk_base = (size_t)ch * vchunk_ * D * 2;
      size_t mt_base = chunk_base;
      for (int mt = 0; mt < n_mt; mt++) {
        const int R = std::min(128, vchunk_ - mt * 128);
        for (int kb = 0; kb < nkb; kb++) {
          uint16_t* hi = P + mt_base + (size_t)kb * 2 * R * 32;
          uint16_t* lo = hi + (size_t)R * 32;
          for (int r = 0; r < R; r++) {
            const int v = ch * vchunk_ + mt * 128 + r;
            for (int kk = 0; kk < 32; kk++) {
              const int k = kb * 32 + kk;
              const float x = v < V ? emb[(size_t)v * D + k] * gfin[k] : 0.f;
              const uint16_t h = bf16_rn(x);
              const uint16_t l = bf16_rn(x - bf16_to_f(h));
              const int c = kk >> 3, e = kk & 7;
              const size_t off = (size_t)r * 32 + (size_t)((c ^ ((r >> 1) & 3)) * 8 + e);
              hi[off] = h;
              lo[off] = l;
            }
          }
        }
        mt_base += (size_t)R * D * 2;
      }
    }
  }
  size_t o_decln = o_ones;
  size_t o_wk_all = bb.add((size_t)d_.dec_layers * D * D);
  size_t o_wv_all = bb.add((size_t)d_.dec_layers * D * D);
  struct DecOff { size_t ln1, wqkv, wo, ln2, wqc, woc, ln3, w1, b1, w2, b2, wqkvP, woP, wqcP, wocP, w1P, w2P, wocF, w1iF, b1i, w2kF,
                  c4_wo, c4_woc, c4_w1, c4_b1, c4_w2; };
  // fc2 k-slices of the v3 kernel: the smallest split whose slice is no wider than max(D, 256) inputs
  ffn_ksplit_ = 1;
  for (int k = 1; k <= 16; k++)
    if (I % k == 0 && (I / k) % 8 == 0 && I / k <= std::max(D, 256)) { ffn_ksplit_ = k; break; }
  const int KS = ffn_ksplit_, Kc = I / KS;
  std::vector<DecOff> dof(d_.dec_layers);
  for (int l = 0; l < d_.dec_layers; l++) {
    const std::string p = dd + "layers." + std::to_string(l) + ".";
    const float* q = wf.get(p + "self_attn.q_proj.weight", {D, D}).data;
    const float* k = wf.get(p + "self_attn.k_proj.weight", {D, D}).data;
    const float* v = wf.get(p + "self_attn.v_proj.weight", {D, D}).data;
    const float* o = wf.get(p + "self_attn.o_proj.weight", {D, D}).data;
    const float* qc = wf.get(p + "encoder_attn.q_proj.weight", {D, D}).data;
    const float* kc = wf.get(p + "encoder_attn.k_proj.weight", {D, D}).data;
    const float* vc = wf.get(p + "encoder_attn.v_proj.weight", {D, D}).data;
    const float* oc = wf.get(p + "encoder_attn.o_proj.weight", {D, D}).data;
    const float* f1 = wf.get(p + "mlp.fc1.weight", {2 * I, D}).data;
    const float* f1b = wf.get(p + "mlp.fc1.bias", {2 * I}).data;
    const float* f2 = wf.get(p + "mlp.fc2.weight", {D, I}).data;
    const float* g1 = wf.get(p + "input_layernorm.weight", {D}).data;
    const float* g2 = wf.get(p + "post_attention_layernorm.weight", {D}).data;
    const float* g3 = wf.get(p + "final_layernorm.weight", {D}).data;
    dof[l].ln1 = dof[l].ln2 = dof[l].ln3 = o_ones;
    dof[l].b2 = bb.add_copy(wf.get(p + "mlp.fc2.bias", {D}).data, D);
    // per-head k-major blocks
    dof[l].wqkv = bb.add((size_t)H * D * 3 * hd);
    dof[l].wo = bb.add((size_t)H * hd * D);
    dof[l].wqc = bb.add((size_t)H * D * hd);
    dof[l].woc = bb.add((size_t)H * hd * D);
    for (int h = 0; h < H; h++) {
      float* wqkv = &bb.data[dof[l].wqkv + (size_t)h * D * 3 * hd];
      float* wqc = &bb.data[dof[l].wqc + (size_t)h * D * hd];
      for (int kk = 0; kk < D; kk++)
        for (int n = 0; n < hd; n++) {
          const size_t src = (size_t)(h * hd + n) * D + kk;
          wqkv[(size_t)kk * 3 * hd + n] = q[src] * g1[kk];
          wqkv[(size_t)kk * 3 * hd + hd + n] = k[src] * g1[kk];
          wqkv[(size_t)kk * 3 * hd + 2 * hd + n] = v[src] * g1[kk];
          wqc[(size_t)kk * hd + n] = qc[src] * g2[kk];
        }
      float* wo = &bb.data[dof[l].wo + (size_t)h * hd * D];
      float* woc = &bb.data[dof[l].woc + (size_t)h * hd * D];
      for (int kk = 0; kk < hd; kk++)
        for (int n = 0; n < D; n++) {
          wo[(size_t)kk * D + n] = o[(size_t)n * D + h * hd + kk];
          woc[(size_t)kk * D + n] = oc[(size_t)n * D + h * hd + kk];
        }
    }
    // MLP chunks: fc1 rows [0, I) are the value ("up"), [I, 2I) the gate
    dof[l].w1 = bb.add((size_t)n_chunk * D * 2 * IC);
    dof[l].b1 = bb.add((size_t)n_chunk * 2 * IC);
    dof[l].w2 = bb.add((size_t)n_chunk * IC * D);
    for (int c = 0; c < n_chunk; c++) {
      float* w1 = &bb.data[dof[l].w1 + (size_t)c * D * 2 * IC];
      float* b1 = &bb.data[dof[l].b1 + (size_t)c * 2 * IC];
      float* w2 = &bb.data[dof[l].w2 + (size_t)c * IC * D];
      for (int n = 0; n < IC; n++) {
        b1[n] = f1b[c * IC + n];
        b1[IC + n] = f1b[I + c * IC + n];
        for (int kk = 0; kk < D; kk++) {
          w1[(size_t)kk * 2 * IC + n] = f1[(size_t)(c * IC + n) * D + kk] * g3[kk];
          w1[(size_t)kk * 2 * IC + IC + n] = f1[(size_t)(I + c * IC + n) * D + kk] * g3[kk];
        }
      }
      for (int kk = 0; kk < IC; kk++)
        for (int n = 0; n < D; n++) w2[(size_t)kk * D + n] = f2[(size_t)n * I + c * IC + kk];
    }
    // tensor-core copies of the same blocks (v2 kernel); LayerNorm gammas folded in exactly as above
    if (dec_tc_layouts) {
      // blocks of one kind are laid out back to back (block h at base + h * decoder_plane_bytes(N, K))
      for (int h = 0; h < H; h++) {
        const size_t a = pack_planes(bb, 3 * hd, D, [&](int n, int kk) {
          const float* src = n < hd ? q : (n < 2 * hd ? k : v);
          return src[(size_t)(h * hd + n % hd) * D + kk] * g1[kk];
        });
        if (h == 0) dof[l].wqkvP = a;
      }
      for (int h = 0; h < H; h++) {
        const size_t a = pack_planes(bb, D, hd, [&](int n, int kk) { return o[(size_t)n * D + h * hd + kk]; });
        if (h == 0) dof[l].woP = a;
      }
      for (int h = 0; h < H; h++) {
        const size_t a = pack_planes(bb, hd, D, [&](int n, int kk) { return qc[(size_t)(h * hd + n) * D + kk] * g2[kk]; });
        if (h == 0) dof[l].wqcP = a;
      }
      for (int h = 0; h < H; h++) {
        const size_t a = pack_planes(bb, D, hd, [&](int n, int kk) { return oc[(size_t)n * D + h * hd + kk]; });
        if (h == 0) dof[l].wocP = a;
      }
      for (int c = 0; c < n_chunk; c++) {
        const size_t a = pack_planes(bb, 2 * IC, D, [&](int n, int kk) {
          const int row = n < IC ? c * IC + n : I + c * IC + (n - IC);   // value ("up") columns, then gate
          return f1[(size_t)row * D + kk] * g3[kk];
        });
        if (c == 0) dof[l].w1P = a;
      }
      for (int c = 0; c < n_chunk; c++) {
        const size_t a = pack_planes(bb, D, IC, [&](int n, int kk) { return f2[(size_t)n * I + c * IC + kk]; });
        if (c == 0) dof[l].w2P = a;
      }
    }
    // v3 kernel: whole matrices as 128-row m-tiles (weight-stationary GEMM jobs)
    if (dec_tc_layouts) {
      dof[l].wocF = pack_planes(bb, D, D, [&](int n, int kk) { return oc[(size_t)n * D + kk]; });
      // fc1 rows interleaved (2j = value j, 2j+1 = gate j): the SiLU gate pairs adjacent TMEM lanes
      dof[l].w1iF = pack_planes(bb, 2 * I, D, [&](int n, int kk) {
        const int row = (n & 1) ? I + (n >> 1) : (n >> 1);
        return f1[(size_t)row * D + kk] * g3[kk];
      });
      dof[l].b1i = bb.add((size_t)2 * I);
      for (int n = 0; n < 2 * I; n++) bb.data[dof[l].b1i + n] = f1b[(n & 1) ? I + (n >> 1) : (n >> 1)];
      for (int ks = 0; ks < KS; ks++) {
        const size_t a = pack_planes(bb, D, Kc, [&](int n, int kk) { return f2[(size_t)n * I + ks * Kc + kk]; });
        if (ks == 0) dof[l].w2kF = a;
      }
    }
    // v4 kernel: fp32 k-major slices per cluster rank
    if (c4_cs_ > 0) {
      const int CS = c4_cs_, ds = D / CS, dsp = (ds + 3) & ~3, is = I / CS;
      dof[l].c4_wo = bb.add((size_t)CS * D * dsp);
      dof[l].c4_woc = bb.add((size_t)CS * D * dsp);
      dof[l].c4_w1 = bb.add((size_t)CS * D * 2 * is);
      dof[l].c4_b1 = bb.add((size_t)CS * 2 * is);
      dof[l].c4_w2 = bb.add((size_t)CS * is * D);
      for (int r = 0; r < CS; r++) {
        float* wo_s = &bb.data[dof[l].c4_wo + (size_t)r * D * dsp];
        float* woc_s = &bb.data[dof[l].c4_woc + (size_t)r * D * dsp];
        for (int kk = 0; kk < D; kk++)
          for (int j = 0; j < ds; j++) {
            wo_s[(size_t)kk * dsp + j] = o[(size_t)(r * ds + j) * D + kk];
            woc_s[(size_t)kk * dsp + j] = oc[(size_t)(r * ds + j) * D + kk];
          }
        float* w1_s = &bb.data[dof[l].c4_w1 + (size_t)r * D * 2 * is];
        float* b1_s = &bb.data[dof[l].c4_b1 + (size_t)r * 2 * is];
        float* w2_s = &bb.data[dof[l].c4_w2 + (size_t)r * is * D];
        for (int j = 0; j < is; j++) {
          const int f = r * is + j;                 // FFN feature of this rank
          b1_s[2 * j] = f1b[f];                     // value ("up")
          b1_s[2 * j + 1] = f1b[I + f];             // gate
          for (int kk = 0; kk < D; kk++) {
            w1_s[(size_t)kk * 2 * is + 2 * j] = f1[(size_t)f * D + kk] * g3[kk];
            w1_s[(size_t)kk * 2 * is + 2 * j + 1] = f1[(size_t)(I + f) * D + kk] * g3[kk];
          }
          for (int n = 0; n < D; n++) w2_s[(size_t)j * D + n] = f2[(size_t)n * I + f];
        }
      }
    }
    std::memcpy(&bb.data[o_wk_all + (size_t)l * D * D], kc, sizeof(float) * D * D);
    std::memcpy(&bb.data[o_wv_all + (size_t)l * D * D], vc, sizeof(float) * D * D);
  }
  size_t o_wkvP = 0;
  if (enc_planes_ && D % 32 == 0) {  // every layer's cross K then every layer's cross V projection as plane tiles: ONE product
    const int LD = d_.dec_layers * D;
    o_wkvP = pack_tile_planes(bb, 2 * LD, D, [&](int n, int k) {
      return n < LD ? bb.data[o_wk_all + (size_t)n * D + k] : bb.data[o_wv_all + (size_t)(n - LD) * D + k];
    });
  }

  wblob_.reserve(bb.data.size());
  CUDA_CHECK(cudaMemcpyAsync(wblob_.ptr, bb.data.data(), bb.data.size() * sizeof(float),
                             cudaMemcpyHostToDevice, stream_));
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  const float* base = wblob_.ptr;
  if (!d_.streaming) {
    w1t_ = base + o_w1t; gn_w_ = base + o_gnw; gn_b_ = base + o_gnb;
    conv2_w_ = base + o_c2; conv2_b_ = base + o_c2b; conv3_w_ = base + o_c3; conv3_b_ = base + o_c3b;
    if (enc_planes_) {
      conv2P_ = reinterpret_cast<const unsigned char*>(base) + o_conv2P * 4;
      conv3P_ = reinterpret_cast<const unsigned char*>(base) + o_conv3P * 4;
    }
  } else {
    s_lin_w_ = base + o_slin; s_c1_w_ = base + o_sc1; s_c1_b_ = base + o_sc1b;
    s_c2_w_ = base + o_sc2; s_c2_b_ = base + o_sc2b;
    pos_emb_ = base + o_pos;
    proj_w_ = (E != D) ? base + o_proj : nullptr;
  }
  enc_.resize(d_.enc_layers);
  for (int l = 0; l < d_.enc_layers; l++) {
    enc_[l] = {base + eo[l].ln1, base + eo[l].wqk, base + eo[l].wv, base + eo[l].wo, base + eo[l].ln2,
               base + eo[l].w1, base + eo[l].b1, base + eo[l].w2, base + eo[l].b2, nullptr, nullptr, nullptr, nullptr};
    if (enc_planes_) {
      const unsigned char* bytes = reinterpret_cast<const unsigned char*>(base);
      enc_[l].wqkP = bytes + eo[l].wqkP * 4; enc_[l].woP = bytes + eo[l].woP * 4;
      enc_[l].w1P = bytes + eo[l].w1P * 4; enc_[l].w2P = bytes + eo[l].w2P * 4;
    }
  }
  enc_final_ln_ = base + o_encln;
  wk_all_ = base + o_wk_all;
  wv_all_ = base + o_wv_all;
  wkvP_ = (enc_planes_ && D % 32 == 0) ? reinterpret_cast<const unsigned char*>(base) + o_wkvP * 4 : nullptr;
  std::memset(&dec_, 0, sizeof(dec_));
  dec_.D = D; dec_.H = H; dec_.hd = hd; dec_.I = I; dec_.V = V; dec_.L = d_.dec_layers;
  dec_.rot_dim = d_.rot_dim; dec_.IC = IC; dec_.n_chunk = n_chunk; dec_.ffn_ksplit = ffn_ksplit_;
  dec_.c4_cs = c4_cs_; dec_.c4_nc = c4_nc_;
  dec_.embed = base + o_emb; dec_.embT = base + o_embT; dec_.final_ln = base + o_decln;
  dec_.embP = base + o_embP; dec_.vchunk = vchunk_; dec_.n_vchunk = n_vchunk_; dec_.smem_limit = smem_optin_;
  for (int l = 0; l < d_.dec_layers; l++) {
    DecLayerWeights& w = dec_.layers[l];
    w.ln1 = base + dof[l].ln1; w.wqkv = base + dof[l].wqkv; w.wo = base + dof[l].wo;
    w.ln2 = base + dof[l].ln2; w.wqc = base + dof[l].wqc; w.woc = base + dof[l].woc;
    const unsigned char* bytes = reinterpret_cast<const unsigned char*>(base);
    w.wqkvP = bytes + dof[l].wqkvP * 4; w.woP = bytes + dof[l].woP * 4; w.wqcP = bytes + dof[l].wqcP * 4;
    w.wocP = bytes + dof[l].wocP * 4; w.w1P = bytes + dof[l].w1P * 4; w.w2P = bytes + dof[l].w2P * 4;
    w.wocF = dec_tc_layouts ? bytes + dof[l].wocF * 4 : nullptr; w.w1iF = bytes + dof[l].w1iF * 4;
    w.b1i = base + dof[l].b1i; w.w2kF = bytes + dof[l].w2kF * 4;
    if (c4_cs_ > 0) {
      w.c4_wo = base + dof[l].c4_wo; w.c4_woc = base + dof[l].c4_woc; w.c4_w1 = base + dof[l].c4_w1;
      w.c4_b1 = base + dof[l].c4_b1; w.c4_w2 = base + dof[l].c4_w2;
    }
    w.ln3 = base + dof[l].ln3; w.w1 = base + dof[l].w1; w.b1 = base + dof[l].b1;
    w.w2 = base + dof[l].w2; w.b2 = base + dof[l].b2;
  }
}

void Model::ensure_rope(int max_pos) {
  if (max_pos <= rope_positions_) return;
  const int n = round_up(std::max(max_pos, 1024), 256);
  const int half = d_.rot_dim / 2;
  std::vector<float> c((size_t)n * half), s((size_t)n * half);
  for (int j = 0; j < half; j++) {
    // HF: inv_freq = 1 / theta ** (arange(0, dim, 2) / dim), dim = int(hd * factor)
    const float inv_freq = (float)(1.0 / std::pow((double)d_.rope_theta, (2.0 * j) / (double)d_.rope_den));
    for (int pos = 0; pos < n; pos++) {
      const float ang = (float)pos * inv_freq;  // fp32 product like HF
      c[(size_t)pos * half + j] = (float)std::cos((double)ang);
      s[(size_t)pos * half + j] = (float)std::sin((double)ang);
    }
  }
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  rope_cos_.reserve(c.size());
  rope_sin_.reserve(s.size());
  CUDA_CHECK(cudaMemcpy(rope_cos_.ptr, c.data(), c.size() * sizeof(float), cudaMemcpyHostToDevice));
  CUDA_CHECK(cudaMemcpy(rope_sin_.ptr, s.data(), s.size() * sizeof(float), cudaMemcpyHostToDevice));
  rope_positions_ = n;
}

void Model::one_shot_stream_plan(uint64_t n_samples, float max_tps, uint64_t& analysed, int& emitted,
                                 int& max_tokens) const {
  analysed = n_samples / 1280 * 1280;         // whole chunks only (core/transcriber.cpp:1342-1343)
  emitted = (int)(analysed / 320);            // is_final: every analysed feature is emitted
  const float dur = (float)n_samples / 16000.0f;
  max_tokens = std::min((int)std::ceil(dur * max_tps), 256);  // core/transcriber.cpp:1386-1390
}

const StreamPlan* Model::auto_plan(const uint64_t*& n_samples, int B, float max_tps, AutoPlan& ap) const {
  ap.analysed.resize(B); ap.emitted.resize(B); ap.max_tokens.resize(B);
  for (int b = 0; b < B; b++) {
    one_shot_stream_plan(n_samples[b], max_tps, ap.analysed[b], ap.emitted[b], ap.max_tokens[b]);
    if (debug_stream_partial_) ap.emitted[b] = std::max(0, ap.emitted[b] - d_.lookahead());
    if (ap.emitted[b] < 1) {
      throw std::runtime_error(format("Audio segment of %llu samples gives the streaming encoder no memory",
                                      (unsigned long long)n_samples[b]));
    }
  }
  ap.plan.emitted = ap.emitted.data();
  ap.plan.max_tokens = ap.max_tokens.data();
  n_samples = ap.analysed.data();
  return &ap.plan;
}

// Staging copy with non-temporal stores: a DMA engine reading lines that are still dirty in the CPU caches has to snoop
// them out (measured here: 20 MB staged by 16 cores then copied host-to-device at ~9 GB/s instead of the 54 GB/s the same
// link gives for data that sits in DRAM); streaming stores put the staged audio straight into memory.  dst 16-byte aligned.
static void stream_copy(float* dst, const float* src, size_t n) {
#if defined(__SSE2__)
  size_t i = 0;
  if ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
    for (; i + 16 <= n; i += 16) {
      const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i));
      const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i + 4));
      const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i + 8));
      const __m128i d = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i + 12));
      _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i), a);
      _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i + 4), b);
      _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i + 8), c);
      _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i + 12), d);
    }
    _mm_sfence();
  }
  if (i < n) std::memcpy(dst + i, src + i, (n - i) * sizeof(float));
#else
  std::memcpy(dst, src, n * sizeof(float));
#endif
}

void Model::transcribe(const float* const* pcm, const uint64_t* n_samples, int B, float max_tps,
                       std::vector<std::vector<int32_t>>& tokens, DebugCapture* dbg, const StreamPlan* plan,
                       std::vector<CrossAttention>* xattn, LogitHook* hook) {
  CUDA_CHECK(cudaSetDevice(device_));
  tokens.clear();
  if (B <= 0) return;
  AutoPlan ap;
  if (d_.streaming && plan == nullptr) plan = auto_plan(n_samples, B, max_tps, ap);
  uint64_t max_n = 0;
  for (int b = 0; b < B; b++) max_n = std::max(max_n, n_samples[b]);
  const int64_t stride = (int64_t)((max_n + 3) / 4 * 4);
  pin_pcm_.reserve((size_t)B * stride);
  pcm_dev_.reserve((size_t)B * stride);
  const auto t0 = std::chrono::steady_clock::now();
  for (int b = 0; b < B; b++)
    if (pcm[b] == nullptr && n_samples[b] > 0) throw std::runtime_error("Audio data is nullptr");
  // Stage through pinned memory, then ONE host-to-device DMA.  Large batches stage on the persistent worker pool (one
  // memcpy thread moves ~5 GB/s, PCIe 5 x16 ~50); the DMA waits for all of it, since a copy engine reading lines other
  // cores are still writing is slow.
  {
    const size_t total_bytes = (size_t)B * stride * sizeof(float);
    if (total_bytes < ((size_t)2 << 20) || B < 2) {
      for (int b = 0; b < B; b++) std::memcpy(pin_pcm_.ptr + (size_t)b * stride, pcm[b], n_samples[b] * sizeof(float));
    } else {
      const int n_slices = std::min(B, 16);
      const int per = (B + n_slices - 1) / n_slices;
      WorkerPool::instance().parallel_for(n_slices, [&](int i) {
        const int lo = i * per, hi = std::min(B, lo + per);
        for (int b = lo; b < hi; b++) stream_copy(pin_pcm_.ptr + (size_t)b * stride, pcm[b], (size_t)n_samples[b]);
      });
    }
    CUDA_CHECK(cudaMemcpyAsync(pcm_dev_.ptr, pin_pcm_.ptr, total_bytes, cudaMemcpyHostToDevice, stream_));
  }
  const auto t1 = std::chrono::steady_clock::now();
  run(pcm_dev_.ptr, stride, n_samples, B, max_tps, tokens, dbg, plan, xattn, hook);
  if (std::getenv("MOONSHINE_B200_HOST_PROF")) {
    const auto t2 = std::chrono::steady_clock::now();
    MSB_LOGF("host profile: staging memcpy %.2f ms, h2d+run %.2f ms",
             std::chrono::duration<double, std::milli>(t1 - t0).count(),
             std::chrono::duration<double, std::milli>(t2 - t1).count());
  }
}

void Model::transcribe_device(const float* d_pcm, int64_t stride, const uint64_t* n_samples, int B,
                              float max_tps, std::vector<std::vector<int32_t>>& tokens,
                              DebugCapture* dbg, const StreamPlan* plan) {
  CUDA_CHECK(cudaSetDevice(device_));
  tokens.clear();
  if (B <= 0) return;
  AutoPlan ap;
  if (d_.streaming && plan == nullptr) plan = auto_plan(n_samples, B, max_tps, ap);
  run(d_pcm, stride, n_samples, B, max_tps, tokens, dbg, plan);
}

void Model::run(const float* d_pcm, int64_t stride, const uint64_t* n_samples, int B, float max_tps,
                std::vector<std::vector<int32_t>>& tokens, DebugCapture* dbg, const StreamPlan* plan,
                std::vector<CrossAttention>* xattn, LogitHook* hook) {
  const int D = d_.dim, I = d_.ffn, H = d_.heads, hd = d_.head_dim, V = d_.vocab;
  const int L = d_.dec_layers;
  times_ = StageTimes();
  int launches = 0;
  // MOONSHINE_B200_DEBUG_SYNC=<bitmask>: synchronise + check after stages
  // (1 setup, 2 frontend, 4 encoder layers, 8 cross K/V, 16 decoder steps, 32 finalize).
  static const int debug_sync = std::getenv("MOONSHINE_B200_DEBUG_SYNC") ? std::atoi(std::getenv("MOONSHINE_B200_DEBUG_SYNC")) : 0;
  auto stage = [&](const char* name, int idx = -1, int bit = 0) {
    if (!(debug_sync & bit)) return;
    cudaError_t e = cudaStreamSynchronize(stream_);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
      throw std::runtime_error(format("CUDA error %s after stage %s[%d] (B=%d): %s", cudaGetErrorName(e),
                                      name, idx, B, cudaGetErrorString(e)));
    }
  };

  // ---------------- plan ----------------
  // Row layouts.  Classic: conv1 rows off1[b] + t (T1 padded to 6 so that conv2 / conv3 are plain strided
  // GEMMs over the packed array), encoder rows r3[b] = off1[b] / 6.  Streaming: hidden frames at rows
  // hrow[b] + 4 + f and conv1 outputs at yrow[b] + 4 + j -- the 4 rows in front of each utterance stay
  // zero and are the causal left padding of the two k=5, s=2 convolutions -- encoder rows r3[b].
  const bool S = d_.streaming;
  const int E = S ? d_.enc_dim : D, EI = S ? d_.enc_ffn : I, ehd = E / H;
  if (S && plan == nullptr) throw std::runtime_error("streaming architectures need a StreamPlan");
  std::vector<int> T1(B), T2(B), T3(B), Tm(B), mlen(B), nsamp(B), Fn(B), C1(B);
  std::vector<int64_t> off1(B), hrow(B), yrow(B), r3v(B);
  int64_t tot1 = 0, tot_h = 0, tot_y = 0, tot3 = 0;
  int maxT1 = 0, maxT3 = 0, max_steps = 0, maxF = 0, maxC1 = 0;
  for (int b = 0; b < B; b++) {
    if (n_samples[b] == 0) throw std::runtime_error("Audio data is nullptr or empty");
    if (n_samples[b] > (uint64_t)INT32_MAX) throw std::runtime_error("Audio segment too long");
    nsamp[b] = (int)n_samples[b];
    if (!S) {
      frontend_lengths((int64_t)n_samples[b], T1[b], T2[b], T3[b]);
      if (T3[b] < 1) {
        throw std::runtime_error(format("Audio segment of %llu samples is too short for the encoder",
                                        (unsigned long long)n_samples[b]));
      }
      off1[b] = tot1;
      r3v[b] = tot1 / 6;
      tot1 += round_up(T1[b], 6);
      Tm[b] = T3[b];
      mlen[b] = max_len_for(n_samples[b], max_tps);
    } else {
      Fn[b] = nsamp[b] / 80;                       // whole 80-sample frames
      C1[b] = Fn[b] >= 1 ? (Fn[b] - 1) / 2 + 1 : 0;  // causal k=5, s=2: floor((F + 4 - 5) / 2) + 1
      T3[b] = C1[b] >= 1 ? (C1[b] - 1) / 2 + 1 : 0;
      Tm[b] = plan->emitted[b];
      mlen[b] = plan->max_tokens[b];
      if (Tm[b] < 1 || Tm[b] > T3[b])
        throw std::runtime_error(format("streaming segment %d: %d memory frames requested, %d analysed", b, Tm[b], T3[b]));
      if (T3[b] > d_.max_pos_emb) throw std::runtime_error("streaming segment longer than the adapter position table");
      if (mlen[b] > d_.max_seq_len) mlen[b] = d_.max_seq_len;
      hrow[b] = tot_h; tot_h += 4 + Fn[b];
      yrow[b] = tot_y; tot_y += 4 + C1[b];
      r3v[b] = tot3; tot3 += round_up(T3[b], 4);
      maxF = std::max(maxF, Fn[b]);
      maxC1 = std::max(maxC1, C1[b]);
    }
    maxT1 = std::max(maxT1, T1[b]);
    maxT3 = std::max(maxT3, T3[b]);
    max_steps = std::max(max_steps, mlen[b]);
  }
  const int64_t tot2 = tot1 / 3;
  if (!S) tot3 = tot1 / 6;
  const int Tp = round_up(maxT3, 4);      // encoder score / V^T row stride
  const int Tpad = round_up(maxT3, 8);    // decoder cross K/V time padding
  const int Smax = round_up(std::max(max_steps, 1) + 1, 4);
  const int BH = B * H;
  ensure_rope(std::max(maxT3, Smax) + 1);

  // ---------------- metadata upload ----------------
  // int32: nsamp[B] T1[B] T3[B] mlen[B] pos[tot3] MzT[BH] DzB[B] Tm[B] Fn[B] C1[B]
  // int64: off1[B] offQ[BH] offK[BH] offS[BH] offVh[BH] offO[BH] offXb[B] offVt[B] offKc[B] offVc[B]
  //        offMem[B] frRow[B] c1A[B] c1C[B] c2A[B] c2C[B]
  const size_t n_i32 = (size_t)4 * B + tot3 + BH + B + 3 * B;
  const size_t n_i64 = (size_t)B + 5 * BH + 4 * B + 6 * B + 3 * (size_t)tot3;  // + vtRow | kcRow | vcRow [tot3]: output address of every packed row (-1: skip)
  pin_i32_.reserve(n_i32);
  pin_i64_.reserve(n_i64);
  meta_i32_.reserve(n_i32);
  meta_i64_.reserve(n_i64);
  static const bool host_prof = std::getenv("MOONSHINE_B200_HOST_PROF") != nullptr;
  const auto hp0 = std::chrono::steady_clock::now();
  // The pinned metadata below is rewritten by every call.  A call that ran to its end has synchronised the stream (its
  // results were read back), so nothing can still be reading it; only a call that left early (exception) forces a wait.
  // Not waiting here lets the metadata build and the first launches overlap this call's own audio DMA.
  if (stream_dirty_) CUDA_CHECK(cudaStreamSynchronize(stream_));
  stream_dirty_ = true;
  const auto hp1 = std::chrono::steady_clock::now();
  int* pi = pin_i32_.ptr;
  int64_t* pl = pin_i64_.ptr;
  int *h_ns = pi, *h_t1 = pi + B, *h_t3 = pi + 2 * B, *h_ml = pi + 3 * B, *h_pos = pi + 4 * B;
  int* h_mzt = h_pos + tot3;
  int* h_dzb = h_mzt + BH;
  int *h_tm = h_dzb + B, *h_fn = h_tm + B, *h_c1 = h_fn + B;
  int64_t *h_off1 = pl, *h_offq = pl + B, *h_offk = h_offq + BH, *h_offs = h_offk + BH,
          *h_offvh = h_offs + BH, *h_offo = h_offvh + BH, *h_offxb = h_offo + BH,
          *h_offvt = h_offxb + B, *h_offkc = h_offvt + B, *h_offvc = h_offkc + B;
  int64_t *h_offmem = h_offvc + B, *h_frrow = h_offmem + B, *h_c1a = h_frrow + B, *h_c1c = h_c1a + B,
          *h_c2a = h_c1c + B, *h_c2c = h_c2a + B;
  int64_t* h_vtrow = h_c2c + B;
  int64_t *h_kcrow = h_vtrow + tot3, *h_vcrow = h_kcrow + tot3;
  for (int64_t r = 0; r < 3 * tot3; r++) h_vtrow[r] = -1;
  std::memset(h_pos, 0, sizeof(int) * tot3);
  for (int b = 0; b < B; b++) {
    h_ns[b] = nsamp[b]; h_t1[b] = T1[b]; h_t3[b] = T3[b]; h_ml[b] = mlen[b];
    h_tm[b] = Tm[b]; h_fn[b] = Fn[b]; h_c1[b] = C1[b];
    h_off1[b] = off1[b];
    const int64_t r3 = r3v[b];
    for (int t = 0; t < T3[b]; t++) {
      h_pos[r3 + t] = t;
      h_vtrow[r3 + t] = (int64_t)b * E * Tp + t;
      if (t < Tm[b]) {  // decoder memory rows: cross K^T [L][B][H][hd][Tpad] / V [L][B][H][Tpad][hd]
        h_kcrow[r3 + t] = (int64_t)b * H * hd * Tpad + t;
        h_vcrow[r3 + t] = (int64_t)b * H * Tpad * hd + (int64_t)t * hd;
      }
    }
    h_dzb[b] = E;
    h_offxb[b] = r3 * E;
    h_offmem[b] = r3 * D;
    h_offvt[b] = (int64_t)b * E * Tp;
    h_offkc[b] = (int64_t)b * H * hd * Tpad;
    h_offvc[b] = (int64_t)b * H * Tpad * hd;
    h_frrow[b] = hrow[b] + 4;
    h_c1a[b] = hrow[b] * E;
    h_c1c[b] = (yrow[b] + 4) * 2 * E;
    h_c2a[b] = yrow[b] * 2 * E;
    h_c2c[b] = r3 * E;
    for (int h = 0; h < H; h++) {
      const int z = b * H + h;
      h_mzt[z] = T3[b];
      h_offq[z] = r3 * 2 * E + (int64_t)h * ehd;
      h_offk[z] = r3 * 2 * E + E + (int64_t)h * ehd;
      h_offs[z] = (int64_t)z * maxT3 * Tp;
      h_offvh[z] = (int64_t)b * E * Tp + (int64_t)h * ehd * Tp;
      h_offo[z] = r3 * E + (int64_t)h * ehd;
    }
  }
  CUDA_CHECK(cudaMemcpyAsync(meta_i32_.ptr, pi, n_i32 * sizeof(int), cudaMemcpyHostToDevice, stream_));
  CUDA_CHECK(cudaMemcpyAsync(meta_i64_.ptr, pl, n_i64 * sizeof(int64_t), cudaMemcpyHostToDevice, stream_));
  const int* d_ns = meta_i32_.ptr;
  const int *d_t1 = d_ns + B, *d_t3 = d_ns + 2 * B, *d_ml = d_ns + 3 * B, *d_pos = d_ns + 4 * B;
  const int* d_mzt = d_pos + tot3;
  const int *d_tm = d_mzt + BH + B, *d_fn = d_tm + B, *d_c1 = d_fn + B;
  const int64_t* d_off1 = meta_i64_.ptr;
  const int64_t *d_offq = d_off1 + B, *d_offk = d_offq + BH, *d_offs = d_offk + BH,
                *d_offvh = d_offs + BH, *d_offo = d_offvh + BH, *d_offxb = d_offo + BH,
                *d_offvt = d_offxb + B, *d_offkc = d_offvt + B, *d_offvc = d_offkc + B;
  const int64_t *d_offmem = d_offvc + B, *d_frrow = d_offmem + B, *d_c1a = d_frrow + B, *d_c1c = d_c1a + B,
                *d_c2a = d_c1c + B, *d_c2c = d_c2a + B;
  const int64_t* d_vtrow = d_c2c + B;
  const int64_t *d_kcrow = d_vtrow + tot3, *d_vcrow = d_kcrow + tot3;

  // ---------------- workspaces ----------------
  auto reserve_zero = [&](DeviceBuffer<float>& buf, size_t n) {
    if (n > buf.count) {
      buf.reserve(n);
      CUDA_CHECK(cudaMemsetAsync(buf.ptr, 0, buf.bytes(), stream_));
    }
  };
  const bool conv_planes = !S && enc_planes_ && conv2P_ != nullptr;
  if (!S) {
    reserve_zero(h1_, (size_t)(tot1 + 8) * D);
    if (conv_planes) {  // im2col operands of conv2 / conv3 as plane tiles (written by GroupNorm-apply / conv2's epilogue)
      reserve_zero(a2P_, plane_tiles_bytes(tot2, 7 * D) / 4);
      reserve_zero(a3P_, plane_tiles_bytes(tot3, 6 * D) / 4);
    } else {
      reserve_zero(h2_, (size_t)(tot2 + 4) * 2 * D);
    }
  } else {
    reserve_zero(frames_, (size_t)(tot_h + 8) * 80);
    reserve_zero(h1_, (size_t)(tot_h + 8) * E);
    reserve_zero(h2_, (size_t)(tot_y + 8) * 2 * E);
    // the 4 rows in front of every utterance are the convolutions' zero padding
    CUDA_CHECK(cudaMemsetAsync(frames_.ptr, 0, (size_t)tot_h * 80 * sizeof(float), stream_));
    CUDA_CHECK(cudaMemsetAsync(h2_.ptr, 0, (size_t)tot_y * 2 * E * sizeof(float), stream_));
  }
  reserve_zero(x_, (size_t)tot3 * E);
  reserve_zero(ln_, (size_t)tot3 * E);
  reserve_zero(qk_, (size_t)tot3 * 2 * E);
  reserve_zero(vt_, (size_t)B * E * Tp);
  {
    // only the unfused attention path materialises scores in HBM
    bool need_scores = false;
    for (int l = 0; l < d_.enc_layers; l++)
      need_scores = need_scores || !attention_tc_supported(maxT3, ehd, S ? d_.win_past[l] : -1, S ? d_.win_future[l] : 0);
    if (need_scores) reserve_zero(scores_, (size_t)BH * maxT3 * Tp);
  }
  reserve_zero(attn_, (size_t)tot3 * E);
  if (enc_planes_) {  // activations as bf16 hi/lo plane tiles (same bytes as fp32 rows, rounded up to 128-row tiles)
    reserve_zero(lnP_, plane_tiles_bytes(tot3, E) / 4);
    reserve_zero(attnP_, plane_tiles_bytes(tot3, E) / 4);
    reserve_zero(midP_, plane_tiles_bytes(tot3, EI) / 4);
  } else {
    reserve_zero(mid_, (size_t)tot3 * EI);
  }
  reserve_zero(enc_out_, (size_t)tot3 * std::max(D, E));
  const int nblk = S ? 0 : conv1_blocks_per_utt(maxT1);
  if (!S) gn_partial_.reserve((size_t)B * nblk * 2);
  // V^T padding columns must stay finite: re-zero when the layout changes
  CUDA_CHECK(cudaMemsetAsync(vt_.ptr, 0, (size_t)B * E * Tp * sizeof(float), stream_));

  stage("setup", -1, 1);
  const auto hp2 = std::chrono::steady_clock::now();
  if (timing_) CUDA_CHECK(cudaEventRecord(ev_[0], stream_));
  // ---------------- frontend ----------------
  if (!S) {
    launch_conv1_tanh(d_pcm, stride, d_ns, d_t1, d_off1, w1t_, h1_.ptr, D, B, maxT1, gn_partial_.ptr,
                      nullptr, stream_);
    stage("conv1", -1, 2);
    if (conv_planes) {
      // GroupNorm-apply writes conv2's im2col operand as plane tiles; conv2 (+bias+GELU) writes conv3's the same way in
      // its epilogue; both convolutions are then plain plane-fed products -- no fp32 intermediate is stored at all.
      unsigned char* a2 = reinterpret_cast<unsigned char*>(a2P_.ptr);
      unsigned char* a3 = reinterpret_cast<unsigned char*>(a3P_.ptr);
      launch_groupnorm_im2col_planes(h1_.ptr, d_t1, d_off1, gn_partial_.ptr, nblk, gn_w_, gn_b_, D, B, maxT1, a2, stream_);
      stage("groupnorm", -1, 2);
      GemmPlanesParams c2;
      c2.A = a2; c2.W = conv2P_; c2.M = (int)tot2; c2.N = 2 * D; c2.K = 7 * D; c2.bias = conv2_b_; c2.act = 1;
      c2.P = a3; c2.p_taps = 3; c2.p_stride = 2;
      launch_gemm_planes(c2, stream_);
      stage("conv2", -1, 2);
      GemmPlanesParams c3;
      c3.A = a3; c3.W = conv3P_; c3.M = (int)tot3; c3.N = D; c3.K = 6 * D; c3.bias = conv3_b_; c3.act = 1;
      c3.C = x_.ptr; c3.ldc = D;
      launch_gemm_planes(c3, stream_);
      stage("conv3", -1, 2);
      launches += 4;
    } else {
    launch_groupnorm_apply(h1_.ptr, d_t1, d_off1, gn_partial_.ptr, nblk, gn_w_, gn_b_, D, B, maxT1, stream_);
    stage("groupnorm", -1, 2);
    launches += 2;
    // conv2 as a GEMM over overlapping row windows of the channel-last h1:
    // output row r reads h1 rows 3r .. 3r+6 (7*D contiguous floats).
    GemmParams g;
    g.A = h1_.ptr; g.lda = 3 * D; g.W = conv2_w_; g.ldw = 7 * D; g.C = h2_.ptr; g.rs = 2 * D;
    g.M = (int)tot2; g.N = 2 * D; g.K = 7 * D; g.bias = conv2_b_; g.act = 1;
    launch_gemm(g, stream_);
    GemmParams g3;
    g3.A = h2_.ptr; g3.lda = 2 * 2 * D; g3.W = conv3_w_; g3.ldw = 3 * 2 * D; g3.C = x_.ptr; g3.rs = D;
    g3.M = (int)tot3; g3.N = D; g3.K = 3 * 2 * D; g3.bias = conv3_b_; g3.act = 1;
    stage("conv2", -1, 2);
    launch_gemm(g3, stream_);
    stage("conv3", -1, 2);
    launches += 2;
    }
  } else {
    // frames -> CMVN -> asinh (one warp per frame), then Linear(80 -> E) + SiLU as one GEMM over every
    // row of the padded layout: padding rows of `frames_` are zero and the linear has no bias, so the
    // padding rows of the hidden array come out as exact zeros.
    launch_stream_frames(d_pcm, stride, d_fn, d_frrow, s_k_, frames_.ptr, B, maxF, stream_);
    stage("stream_frames", -1, 2);
    GemmParams g;
    g.A = frames_.ptr; g.lda = 80; g.W = s_lin_w_; g.ldw = 80; g.C = h1_.ptr; g.rs = E;
    g.M = (int)tot_h; g.N = E; g.K = 80; g.act = 2;
    launch_gemm(g, stream_);
    stage("stream_linear", -1, 2);
    // causal conv1 (E -> 2E, k=5, s=2) + SiLU: output j of utterance b reads hidden rows hrow[b] + 2j ..
    // + 4 (5 * E contiguous floats); grouped per utterance so the padding rows of the output stay zero.
    GemmParams c1;
    c1.A = h1_.ptr; c1.lda = 2 * E; c1.offA = d_c1a; c1.W = s_c1_w_; c1.ldw = 5 * E; c1.strideW = 0;
    c1.C = h2_.ptr; c1.offC = d_c1c; c1.rs = 2 * E;
    c1.groups = B; c1.M = maxC1; c1.N = 2 * E; c1.K = 5 * E; c1.Mz = d_c1; c1.bias = s_c1_b_; c1.act = 2;
    launch_gemm(c1, stream_);
    stage("stream_conv1", -1, 2);
    GemmParams c2;
    c2.A = h2_.ptr; c2.lda = 2 * 2 * E; c2.offA = d_c2a; c2.W = s_c2_w_; c2.ldw = 5 * 2 * E; c2.strideW = 0;
    c2.C = x_.ptr; c2.offC = d_c2c; c2.rs = E;
    c2.groups = B; c2.M = maxT3; c2.N = E; c2.K = 5 * 2 * E; c2.Mz = d_t3; c2.bias = s_c2_b_;
    launch_gemm(c2, stream_);
    stage("stream_conv2", -1, 2);
    launches += 4;
  }
  if (timing_) CUDA_CHECK(cudaEventRecord(ev_[1], stream_));

  // ---------------- encoder layers ----------------
  const float scale = 1.0f / std::sqrt((float)ehd);
  for (int l = 0; l < d_.enc_layers; l++) {
    const EncLayer& w = enc_[l];
    unsigned char* lnP = reinterpret_cast<unsigned char*>(lnP_.ptr);
    unsigned char* attnP = reinterpret_cast<unsigned char*>(attnP_.ptr);
    unsigned char* midP = reinterpret_cast<unsigned char*>(midP_.ptr);
    if (enc_planes_) launch_layernorm_planes(x_.ptr, nullptr, lnP, w.ln1, tot3, E, stream_);
    else launch_layernorm(x_.ptr, ln_.ptr, w.ln1, tot3, E, stream_);
    if (enc_planes_) {
      // Q | K | V in ONE product, both operands as pre-split planes (bulk copies feed the tensor core directly): columns
      // < 2E land in the Q|K rows (with RoPE), columns >= 2E are stored transposed, V^T_b[e][t], as the attention wants them
      GemmPlanesParams g;
      g.A = lnP; g.W = w.wqkP; g.M = (int)tot3; g.N = 3 * E; g.K = E; g.C = qk_.ptr; g.ldc = 2 * E;
      g.n_split = 2 * E; g.Vt = vt_.ptr; g.vt_row = d_vtrow; g.vt_ld = Tp;
      if (!S) {
        g.pos = d_pos; g.rope_cos = rope_cos_.ptr; g.rope_sin = rope_sin_.ptr;
        g.rope_cols = 2 * E; g.head_dim = ehd; g.rot_dim = d_.rot_dim;
      }
      launch_gemm_planes(g, stream_);
    } else {  // Q|K projection (classic: with fused interleaved RoPE; the streaming encoder has no positions)
      GemmParams g;
      g.A = ln_.ptr; g.lda = E; g.W = w.wqk; g.ldw = E; g.C = qk_.ptr; g.rs = 2 * E;
      g.M = (int)tot3; g.N = 2 * E; g.K = E;
      if (!S) {
        g.pos = d_pos; g.rope_cos = rope_cos_.ptr; g.rope_sin = rope_sin_.ptr;
        g.rope_cols = 2 * E; g.head_dim = ehd; g.rot_dim = d_.rot_dim;
      }
      launch_gemm(g, stream_);
    }
    if (!enc_planes_) {  // V^T_b[E, T_b] = Wv * ln_b^T  (swapped orientation, per utterance)
      GemmParams g;
      g.A = w.wv; g.lda = E; g.strideA = 0; g.W = ln_.ptr; g.ldw = E; g.offW = d_offxb;
      g.C = vt_.ptr; g.offC = d_offvt; g.rs = Tp;
      g.groups = B; g.M = E; g.N = maxT3; g.K = E; g.Nz = d_t3;
      launch_gemm(g, stream_);
    }
    const int wp = S ? d_.win_past[l] : -1, wf = S ? d_.win_future[l] : 0;
    if (attention_tc_supported(maxT3, ehd, wp, wf)) {
      // softmax(scale * Q K^T [window]) V in one tcgen05 kernel; scores stay in TMEM
      AttnParams a;
      a.qk = qk_.ptr; a.vt = vt_.ptr; a.out = attn_.ptr;
      a.offQ = d_offq; a.offK = d_offk; a.offV = d_offvh; a.offO = d_offo; a.Tz = d_mzt;
      a.ldqk = 2 * E; a.ldv = Tp; a.ldo = E; a.hd = ehd; a.scale = scale; a.win_past = wp; a.win_future = wf;
      launch_attention_tc(a, BH, maxT3, stream_);
      launches -= 2;
    } else {
      {  // S_z = scale * Q_z K_z^T
        GemmParams g;
        g.A = qk_.ptr; g.lda = 2 * E; g.offA = d_offq; g.W = qk_.ptr; g.ldw = 2 * E; g.offW = d_offk;
        g.C = scores_.ptr; g.offC = d_offs; g.rs = Tp;
        g.groups = BH; g.M = maxT3; g.N = maxT3; g.K = ehd; g.Mz = d_mzt; g.Nz = d_mzt;
        g.alpha = scale;
        launch_gemm(g, stream_);
      }
      if (S) launch_softmax_rows(scores_.ptr, d_offs, d_mzt, d_mzt, Tp, BH, maxT3, stream_, d_.win_past[l], d_.win_future[l]);
      else launch_softmax_rows(scores_.ptr, d_offs, d_mzt, d_mzt, Tp, BH, maxT3, stream_);
      {  // O_z = P_z V_z
        GemmParams g;
        g.A = scores_.ptr; g.lda = Tp; g.offA = d_offs; g.W = vt_.ptr; g.ldw = Tp; g.offW = d_offvh;
        g.C = attn_.ptr; g.offC = d_offo; g.rs = E;
        g.groups = BH; g.M = maxT3; g.N = ehd; g.K = maxT3; g.Mz = d_mzt; g.Kz = d_mzt;
        launch_gemm(g, stream_);
      }
    }
    if (enc_planes_) {
      launch_rows_to_planes(attn_.ptr, E, tot3, E, attnP, stream_);
      GemmPlanesParams o;  // x += attn Wo^T
      o.A = attnP; o.W = w.woP; o.M = (int)tot3; o.N = E; o.K = E; o.C = x_.ptr; o.ldc = E; o.accumulate = 1;
      launch_gemm_planes(o, stream_);
      launch_layernorm_planes(x_.ptr, nullptr, lnP, w.ln2, tot3, E, stream_);
      GemmPlanesParams f1;  // gelu(ln W1^T + b1), written straight as the planes fc2 reads
      f1.A = lnP; f1.W = w.w1P; f1.M = (int)tot3; f1.N = EI; f1.K = E; f1.P = midP; f1.bias = w.b1; f1.act = 1;
      launch_gemm_planes(f1, stream_);
      GemmPlanesParams f2;  // x += mid W2^T + b2
      f2.A = midP; f2.W = w.w2P; f2.M = (int)tot3; f2.N = E; f2.K = EI; f2.C = x_.ptr; f2.ldc = E; f2.bias = w.b2; f2.accumulate = 1;
      launch_gemm_planes(f2, stream_);
      launches += 1;
    } else {
    {  // x += attn Wo^T
      GemmParams g;
      g.A = attn_.ptr; g.lda = E; g.W = w.wo; g.ldw = E; g.C = x_.ptr; g.rs = E;
      g.M = (int)tot3; g.N = E; g.K = E; g.accumulate = 1;
      launch_gemm(g, stream_);
    }
    launch_layernorm(x_.ptr, ln_.ptr, w.ln2, tot3, E, stream_);
    {
      GemmParams g;
      g.A = ln_.ptr; g.lda = E; g.W = w.w1; g.ldw = E; g.C = mid_.ptr; g.rs = EI;
      g.M = (int)tot3; g.N = EI; g.K = E; g.bias = w.b1; g.act = 1;
      launch_gemm(g, stream_);
      GemmParams g2;
      g2.A = mid_.ptr; g2.lda = EI; g2.W = w.w2; g2.ldw = EI; g2.C = x_.ptr; g2.rs = E;
      g2.M = (int)tot3; g2.N = E; g2.K = EI; g2.bias = w.b2; g2.accumulate = 1;
      launch_gemm(g2, stream_);
    }
    }
    launches += 10;
    stage("encoder_layer", l, 4);
  }
  if (!S) {
    launch_layernorm(x_.ptr, enc_out_.ptr, enc_final_ln_, tot3, D, stream_);
    launches += 1;
  } else {
    // final unit-offset norm, then the adapter: memory = proj(encoded + pos_emb[frame index])
    // (lora/export.py:130-144; every segment is encoded from its first frame, so the offset is 0)
    launch_layernorm(x_.ptr, ln_.ptr, enc_final_ln_, tot3, E, stream_);
    if (proj_w_ == nullptr) {
      launch_add_rows_by_index(ln_.ptr, pos_emb_, d_pos, enc_out_.ptr, tot3, E, stream_);
    } else {
      launch_add_rows_by_index(ln_.ptr, pos_emb_, d_pos, attn_.ptr, tot3, E, stream_);
      GemmParams g;
      g.A = attn_.ptr; g.lda = E; g.W = proj_w_; g.ldw = E; g.C = enc_out_.ptr; g.rs = D;
      g.M = (int)tot3; g.N = D; g.K = E;
      launch_gemm(g, stream_);
      launches += 1;
    }
    launches += 2;
    stage("adapter", -1, 4);
  }
  if (timing_) CUDA_CHECK(cudaEventRecord(ev_[2], stream_));

  if (dbg && dbg->encoder_out) {
    dbg->encoder_out->clear();
    if (dbg->encoder_frames) dbg->encoder_frames->assign(Tm.begin(), Tm.end());
    std::vector<float> all((size_t)tot3 * D);
    CUDA_CHECK(cudaMemcpyAsync(all.data(), enc_out_.ptr, all.size() * sizeof(float), cudaMemcpyDeviceToHost, stream_));
    CUDA_CHECK(cudaStreamSynchronize(stream_));
    for (int b = 0; b < B; b++) {
      const float* src = all.data() + (size_t)r3v[b] * D;
      dbg->encoder_out->insert(dbg->encoder_out->end(), src, src + (size_t)Tm[b] * D);
    }
  }
  if (dbg && dbg->skip_decode) {
    tokens.assign(B, std::vector<int32_t>());
    CUDA_CHECK(cudaStreamSynchronize(stream_));
    stream_dirty_ = false;
    return;
  }

  // ---------------- cross K/V (fp16, layouts of the step kernel) ----------------
  const size_t kv_elems = (size_t)L * B * H * hd * Tpad;
  if (kv_elems > kc_.count) {
    kc_.reserve(kv_elems);
    vc_.reserve(kv_elems);
  }
  CUDA_CHECK(cudaMemsetAsync(kc_.ptr, 0, kv_elems * sizeof(__half), stream_));
  if (wkvP_ != nullptr) {
    // one plane-fed product for every layer's cross K and V: memory rows x [Wk_0 .. Wk_L-1 | Wv_0 .. Wv_L-1]^T, the
    // epilogue stores fp16 straight into the step kernels' layouts (K time-contiguous, V as head rows)
    reserve_zero(encP_, plane_tiles_bytes(tot3, D) / 4);
    unsigned char* encP = reinterpret_cast<unsigned char*>(encP_.ptr);
    launch_rows_to_planes(enc_out_.ptr, D, tot3, D, encP, stream_);
    GemmPlanesParams g;
    g.A = encP; g.W = wkvP_; g.M = (int)tot3; g.N = 2 * L * D; g.K = D;
    g.Hk = kc_.ptr; g.Hv = vc_.ptr; g.hk_row = d_kcrow; g.hv_row = d_vcrow; g.n_split = L * D;
    g.SL = (int64_t)B * H * hd * Tpad; g.Dm = D; g.hdm = hd; g.Tpadm = Tpad;
    launch_gemm_planes(g, stream_);
    launches += 2;
    stage("cross_kv", -1, 8);
  } else {
    GemmParams g;  // K^T: rows (l, h, d), cols t
    g.A = wk_all_; g.lda = D; g.W = enc_out_.ptr; g.ldw = D; g.offW = d_offmem;
    g.C = kc_.ptr; g.offC = d_offkc; g.out_half = 1;
    g.groups = B; g.M = L * D; g.N = maxT3; g.K = D; g.Nz = d_tm;
    g.rm1 = D; g.rs1 = (int64_t)B * H * hd * Tpad; g.rm2 = hd; g.rs2 = (int64_t)hd * Tpad; g.rs = Tpad;
    launch_gemm(g, stream_);
    GemmParams v;  // V: rows t, cols (l, h, d)
    v.A = enc_out_.ptr; v.lda = D; v.offA = d_offmem; v.W = wv_all_; v.ldw = D;
    v.C = vc_.ptr; v.offC = d_offvc; v.out_half = 1;
    v.groups = B; v.M = maxT3; v.N = L * D; v.K = D; v.Mz = d_tm;
    v.rs = hd; v.cm1 = D; v.cs1 = (int64_t)B * H * Tpad * hd; v.cm2 = hd; v.cs2 = (int64_t)Tpad * hd;
    launch_gemm(v, stream_);
    launches += 2;
    stage("cross_kv", -1, 8);
  }
  const auto hp3 = std::chrono::steady_clock::now();
  if (timing_) CUDA_CHECK(cudaEventRecord(ev_[3], stream_));

  // ---------------- greedy decode ----------------
  DecoderParams p = dec_;
  p.B = B; p.Tpad = Tpad; p.Smax = Smax;
  const size_t self_elems = (size_t)L * B * H * hd * Smax;
  ks_.reserve(self_elems);
  vs_.reserve(self_elems);
  hbuf_.reserve((size_t)2 * B * D);
  part_.reserve((size_t)std::max(2 * H + p.n_chunk, H + p.ffn_ksplit + 1) * B * D);
  attc_.reserve((size_t)B * D);
  act_.reserve((size_t)B * I);
  sync3_.reserve(kSync3Words);
  CUDA_CHECK(cudaMemsetAsync(sync3_.ptr, 0, kSync3Words * sizeof(unsigned), stream_));
  p.attc = attc_.ptr; p.act = act_.ptr; p.sync3 = sync3_.ptr;
  xfin_.reserve((size_t)B * D);
  cand_val_.reserve((size_t)2 * p.n_vchunk * B);
  cand_idx_.reserve((size_t)2 * p.n_vchunk * B);
  tokens_dev_.reserve((size_t)B * (Smax + 1));
  ntok_dev_.reserve(B);
  done_dev_.reserve(B);
  pin_tokens_.reserve((size_t)B * (Smax + 1) + 2 * (size_t)B + 4);
  {
    int* ht = pin_tokens_.ptr;
    int* hn = ht + (size_t)B * (Smax + 1);
    int* hact = hn + B;
    int active = 0;
    for (int b = 0; b < B; b++) {
      for (int t = 0; t <= Smax; t++) ht[(size_t)b * (Smax + 1) + t] = 0;
      ht[(size_t)b * (Smax + 1)] = d_.bos;
      hn[b] = 1;
      if (mlen[b] > 0) active++;
    }
    *hact = active;
    CUDA_CHECK(cudaMemcpyAsync(tokens_dev_.ptr, ht, (size_t)B * (Smax + 1) * sizeof(int), cudaMemcpyHostToDevice, stream_));
    CUDA_CHECK(cudaMemcpyAsync(ntok_dev_.ptr, hn, B * sizeof(int), cudaMemcpyHostToDevice, stream_));
    CUDA_CHECK(cudaMemcpyAsync(nactive_.ptr, hact, sizeof(int), cudaMemcpyHostToDevice, stream_));
    CUDA_CHECK(cudaMemsetAsync(done_dev_.ptr, 0, B * sizeof(int), stream_));
  }
  p.rope_cos = rope_cos_.ptr; p.rope_sin = rope_sin_.ptr;
  p.enc_len = d_tm; p.max_len = d_ml;
  p.kc = kc_.ptr; p.vc = vc_.ptr; p.ks = ks_.ptr; p.vs = vs_.ptr;
  p.hbuf = hbuf_.ptr; p.part = part_.ptr; p.xfin = xfin_.ptr;
  p.cand_val = cand_val_.ptr; p.cand_idx = cand_idx_.ptr;
  p.tokens = tokens_dev_.ptr; p.n_tokens = ntok_dev_.ptr; p.done = done_dev_.ptr;
  p.n_active = nactive_.ptr; p.barrier = barrier_.ptr;
  p.logits_out = nullptr; p.forced = nullptr;
  int dbg_steps = 0;
  if (dbg && dbg->forced) {
    std::vector<int> f((size_t)B * (Smax + 1), 0);
    for (int b = 0; b < B; b++)
      for (int t = 0; t <= Smax && t < dbg->forced_stride; t++)
        f[(size_t)b * (Smax + 1) + t] = dbg->forced[(size_t)b * dbg->forced_stride + t];
    forced_dev_.reserve(f.size());
    CUDA_CHECK(cudaMemcpy(forced_dev_.ptr, f.data(), f.size() * sizeof(int), cudaMemcpyHostToDevice));
    p.forced = forced_dev_.ptr;
  }
  if (dbg && dbg->logits && dbg->logits_steps > 0) {
    dbg_steps = std::min(dbg->logits_steps, max_steps);
    logits_dbg_.reserve((size_t)dbg_steps * B * V);
    CUDA_CHECK(cudaMemsetAsync(logits_dbg_.ptr, 0, (size_t)dbg_steps * B * V * sizeof(float), stream_));
  }
  const int grid = sm_count_;
  p.xattn_out = nullptr;
  p.xattn_steps = 0;
  // v2 streams operands through the smem ring; its cross-attention maps one thread to 4 key positions, so encoder
  // memories longer than 1024 frames take the v1 kernel.  v3 and v4 share that limit and keep a LayerNorm row in
  // registers, so they stop at D = 512: v2 serves the wider models.
  const bool use_v3 = decoder_step3_supported(p);
  const bool use_v4 = use_v3 && c4_cs_ > 0 && decoder_step4_supported(p);
  const bool use_v2 = !use_v3 && D % 32 == 0 && Tpad <= 1024 && hd <= 64 && d_.rot_dim <= 128;
  if (use_v4) decoder_step4_plan(p);
  else if (use_v3) decoder_step3_plan(p, grid);
  if (std::getenv("MOONSHINE_B200_VERBOSE"))
    MSB_LOGF("decoder kernel: %s (B=%d, cluster size %d)", use_v4 ? "v4" : use_v3 ? "v3" : use_v2 ? "v2" : "v1", B, c4_cs_);
  auto launch_step = [&]() {
    if (use_v4) launch_decoder_step4(p, stream_);
    else if (use_v3) launch_decoder_step3(p, grid, stream_);
    else if (use_v2) launch_decoder_step2(p, grid, stream_);
    else launch_decoder_step(p, grid, stream_);
  };
  static const int prof_step = std::getenv("MOONSHINE_B200_PROF") ? std::atoi(std::getenv("MOONSHINE_B200_PROF")) : -1;
  DeviceBuffer<unsigned long long> prof_buf;
  if (prof_step >= 0) {
    prof_buf.reserve((size_t)grid * 512);
    CUDA_CHECK(cudaMemsetAsync(prof_buf.ptr, 0, prof_buf.bytes(), stream_));
  }
  if (xattn != nullptr) {
    xattn->clear();
    if (!use_v2 && !use_v3)
      throw std::runtime_error("word_timestamps: the cross-attention export needs at most 1024 encoder frames, "
                               "head_dim <= 64, rotary dimension <= 128 and a hidden size that is a multiple of 32");
    p.xattn_steps = std::max(max_steps, 1);
    const size_t n = (size_t)B * L * H * p.xattn_steps * Tpad;
    xattn_dev_.reserve(n);
    CUDA_CHECK(cudaMemsetAsync(xattn_dev_.ptr, 0, n * sizeof(float), stream_));
    p.xattn_out = xattn_dev_.ptr;
  }
  std::vector<std::vector<int32_t>> hooked_tokens;  // filled by the host-stepped loop
  int steps_launched = max_steps;
  // explicit rows: every per-row buffer grows to R rows (the caches stay per utterance)
  auto widen = [&](DecoderParams& q, int n) {
    const int R = B * n;
    q.B = R; q.B_utt = B; q.row_group = n;
    hbuf_.reserve((size_t)2 * R * D);
    part_.reserve((size_t)std::max(2 * H + q.n_chunk, H + q.ffn_ksplit + 1) * R * D);
    attc_.reserve((size_t)R * D);
    act_.reserve((size_t)R * I);
    xfin_.reserve((size_t)R * D);
    cand_val_.reserve((size_t)2 * q.n_vchunk * R);
    cand_idx_.reserve((size_t)2 * q.n_vchunk * R);
    rows_dev_.reserve((size_t)4 * R);
    q.hbuf = hbuf_.ptr; q.part = part_.ptr; q.attc = attc_.ptr; q.act = act_.ptr; q.xfin = xfin_.ptr;
    q.cand_val = cand_val_.ptr; q.cand_idx = cand_idx_.ptr;
    q.row_tok = rows_dev_.ptr; q.row_pos = rows_dev_.ptr + R; q.row_nin = rows_dev_.ptr + 2 * R; q.row_utt = rows_dev_.ptr + 3 * R;
    q.logits_out = nullptr; q.xattn_out = nullptr; q.forced = nullptr; q.prof = nullptr;
    decoder_step3_plan(q, grid);
    return R;
  };
  const bool multi = dbg && dbg->forced && dbg->rows_per_launch > 1 && use_v3 && hook == nullptr && xattn == nullptr && max_steps > 0;
  bool any_draft = false;
  const int* const* drafts = (plan && plan->draft && plan->draft_len) ? plan->draft : dbg_draft_;
  const int* draft_lens = (plan && plan->draft && plan->draft_len) ? plan->draft_len : dbg_draft_len_;
  dbg_draft_ = nullptr;
  dbg_draft_len_ = nullptr;
  if (drafts && draft_lens)
    for (int b = 0; b < B; b++) any_draft |= drafts[b] != nullptr && draft_lens[b] > 0;
  const bool verify = any_draft && hook == nullptr && xattn == nullptr && dbg == nullptr && use_v3 && max_steps > 0 &&
                      B * kVerifyRows <= 4096;
  bool spliced = false;  // verify finished in the lockstep loop (which needs its finalize launch)
  if (multi) {
    // ---- teacher-forced multi-token decoder runs (decode_tokens, moonshine-streaming-model.cpp:1136-1190): n consecutive
    // positions of every utterance per launch, row i attending the cache and rows 0..i of its own launch; logits of
    // every position come back in the [steps][B][V] layout of the single-token dump ----
    int n = 2;
    while (n < dbg->rows_per_launch && n < 16) n *= 2;
    DecoderParams q = p;
    const int R = widen(q, n);
    logits_rows_.reserve((size_t)R * V);
    q.logits_out = logits_rows_.ptr;
    std::vector<int> rows((size_t)4 * R);
    int k = 0;
    for (int t0 = 0; t0 < max_steps; t0 += n, k++) {
      for (int b = 0; b < B; b++)
        for (int i = 0; i < n; i++) {
          const int r = b * n + i, t = t0 + i;
          const bool on = t < mlen[b] && t < dbg->forced_stride;
          rows[r] = on ? dbg->forced[(size_t)b * dbg->forced_stride + t] : -1;
          rows[(size_t)R + r] = on ? t : 0;
          rows[(size_t)2 * R + r] = on ? i : 0;
          rows[(size_t)3 * R + r] = b;
        }
      CUDA_CHECK(cudaMemcpyAsync(rows_dev_.ptr, rows.data(), rows.size() * sizeof(int), cudaMemcpyHostToDevice, stream_));
      q.step = k;
      launch_decoder_step3(q, grid, stream_);
      for (int b = 0; b < B; b++)
        for (int i = 0; i < n; i++) {
          const int t = t0 + i;
          if (t < dbg_steps && rows[(size_t)b * n + i] >= 0)
            CUDA_CHECK(cudaMemcpyAsync(logits_dbg_.ptr + ((size_t)t * B + b) * V, logits_rows_.ptr + (size_t)(b * n + i) * V,
                                       (size_t)V * sizeof(float), cudaMemcpyDeviceToDevice, stream_));
        }
      CUDA_CHECK(cudaStreamSynchronize(stream_));  // `rows` is reused by the next launch
    }
    steps_launched = k;
  } else if (verify) {
    // ---- verify-then-continue on explicit rows (decode_full, moonshine-streaming-model.cpp:1192-1397) ----
    // kVerifyRows consecutive draft positions of every utterance per launch; the plan kernel between two launches books
    // the emitted ids and moves each utterance on (verify -> auto-regressive -> done).  An accepted draft of m ids
    // costs ceil((m + 1) / kVerifyRows) launches instead of m + 1.
    const int n = kVerifyRows;
    DecoderParams q = p;
    widen(q, n);
    vstate_dev_.reserve((size_t)4 * B);
    const int dstride = Smax + 1;
    draft_dev_.reserve((size_t)B * dstride + B);
    std::vector<int> hd_((size_t)B * dstride + B, 0);
    int m_max = 0;
    for (int b = 0; b < B; b++) {
      const int m = drafts[b] ? std::min(std::max(draft_lens[b], 0), Smax - 1) : 0;
      for (int i = 0; i < m; i++) hd_[(size_t)b * dstride + i] = drafts[b][i];
      hd_[(size_t)B * dstride + b] = m;
      m_max = std::max(m_max, m);
    }
    CUDA_CHECK(cudaMemcpyAsync(draft_dev_.ptr, hd_.data(), hd_.size() * sizeof(int), cudaMemcpyHostToDevice, stream_));
    CUDA_CHECK(cudaMemsetAsync(vstate_dev_.ptr, 0, (size_t)4 * B * sizeof(int), stream_));
    VerifyState st;
    st.mode = vstate_dev_.ptr; st.pos = vstate_dev_.ptr + B; st.cur = vstate_dev_.ptr + 2 * B; st.prev_n = vstate_dev_.ptr + 3 * B;
    st.draft = draft_dev_.ptr; st.draft_len = draft_dev_.ptr + (size_t)B * dstride; st.draft_stride = dstride;
    int k = 0;
    auto run_steps = [&](int count) {
      for (int i = 0; i < count; i++, k++) {
        q.step = k;
        launch_decoder_step3(q, grid, stream_);
        launch_decoder_verify_plan(q, st, k + 1, n, d_.bos, d_.eos, stream_);
      }
    };
    launch_decoder_verify_plan(q, st, 0, n, d_.bos, d_.eos, stream_);
    run_steps(std::min((m_max + 1 + n - 1) / n, max_steps));
    // every draft is now either verified to its end or rejected: what is left is one id per launch and utterance
    int* hn = pin_tokens_.ptr + (size_t)B * (Smax + 1);
    while (true) {
      CUDA_CHECK(cudaMemcpyAsync(hn, ntok_dev_.ptr, B * sizeof(int), cudaMemcpyDeviceToHost, stream_));
      CUDA_CHECK(cudaMemcpyAsync(hn + B, vstate_dev_.ptr, B * sizeof(int), cudaMemcpyDeviceToHost, stream_));  // modes
      CUDA_CHECK(cudaStreamSynchronize(stream_));
      int rem = 0, pos_lo = 1 << 30, pos_hi = -1;
      bool all_ar = true;
      for (int b = 0; b < B; b++)
        if (hn[B + b] != 2) {
          rem = std::max(rem, mlen[b] - (hn[b] - 1));
          pos_lo = std::min(pos_lo, hn[b] - 1);
          pos_hi = std::max(pos_hi, hn[b] - 1);
          all_ar &= hn[B + b] == 1;
        }
      if (rem <= 0) break;
      if (all_ar && pos_lo == pos_hi && pos_lo >= 1) {
        // Every live utterance waits at the same position (always so for a single stream): the tail is the ordinary
        // lockstep loop on the kernel that is fastest for this batch (cluster-resident layers for small ones).  The
        // caches are position-indexed and shared by both row models; only the "previous id" hand-over is seeded.
        p.hbuf = hbuf_.ptr; p.part = part_.ptr; p.attc = attc_.ptr; p.act = act_.ptr; p.xfin = xfin_.ptr;
        p.cand_val = cand_val_.ptr; p.cand_idx = cand_idx_.ptr;
        // the phase counters are cumulative per launch shape ((epoch + 1) * jobs): a new shape starts a new epoch count
        CUDA_CHECK(cudaMemsetAsync(sync3_.ptr, 0, sizeof(unsigned), stream_));
        CUDA_CHECK(cudaMemsetAsync(sync3_.ptr + 32, 0, (kSync3Words - 32) * sizeof(unsigned), stream_));
        launch_decoder_seed_candidates(p, st.cur, (pos_lo - 1) & 1, stream_);
        for (int t = pos_lo; t < max_steps; t++, k++) {
          p.step = t;
          p.prof = nullptr;
          p.logits_out = nullptr;
          launch_step();
        }
        spliced = true;
        break;
      }
      run_steps(std::min(rem, 16));  // bounded bursts: an EOS ends the tail early, the next read sees it
    }
    steps_launched = k;
  } else if (hook == nullptr) {
    for (int t = 0; t < max_steps; t++) {
      p.step = t;
      p.prof = (t == prof_step) ? (void*)prof_buf.ptr : nullptr;
      p.logits_out = (t < dbg_steps) ? logits_dbg_.ptr + (size_t)t * B * V : nullptr;
      launch_step();
      stage("decoder_step", t, 16);
    }
  } else if (use_v3 && hook->shared_bonus(V) != nullptr) {
    // On-device biasing (reference: ContextBiaser between decode_step and the argmax, core/transcriber.cpp:1440-1470).
    // The host only walks the trie: per step it uploads each utterance's few (token, bonus) pairs, the kernel adds
    // them (and the shared root bonuses) in the logits epilogue before its fused argmax, and B token ids come back
    // to advance the walks.  No logits cross PCIe.
    const std::vector<float>& shared = *hook->shared_bonus(V);
    const int cap = 256;
    bias_static_dev_.reserve((size_t)V);
    CUDA_CHECK(cudaMemcpyAsync(bias_static_dev_.ptr, shared.data(), (size_t)V * sizeof(float), cudaMemcpyHostToDevice, stream_));
    bias_n_dev_.reserve(B); bias_ids_dev_.reserve((size_t)B * cap); bias_val_dev_.reserve((size_t)B * cap);
    step_tok_dev_.reserve(B);
    pin_bias_i32_.reserve((size_t)B + (size_t)B * cap + B);
    pin_bias_f32_.reserve((size_t)B * cap);
    int* h_n = pin_bias_i32_.ptr;
    int* h_ids = h_n + B;
    int* h_tok = h_ids + (size_t)B * cap;
    float* h_val = pin_bias_f32_.ptr;
    p.bias_static = bias_static_dev_.ptr;
    p.bias_dyn_n = bias_n_dev_.ptr; p.bias_dyn_ids = bias_ids_dev_.ptr; p.bias_dyn_val = bias_val_dev_.ptr;
    p.bias_dyn_cap = cap;
    std::vector<char> finished(B, 0);
    hooked_tokens.assign(B, std::vector<int32_t>{(int32_t)d_.bos});
    int remaining = 0;
    for (int b = 0; b < B; b++) {
      finished[b] = mlen[b] <= 0;
      remaining += finished[b] ? 0 : 1;
    }
    std::vector<std::pair<int32_t, float>> pairs;
    steps_launched = 0;
    for (int t = 0; t < max_steps && remaining > 0; t++) {
      for (int b = 0; b < B; b++) {
        h_n[b] = 0;
        if (finished[b]) continue;
        hook->step_bonus(b, pairs);
        if ((int)pairs.size() > cap) throw std::runtime_error("key-term biasing: more than 256 active continuations for one utterance");
        h_n[b] = (int)pairs.size();
        for (size_t k = 0; k < pairs.size(); k++) {
          h_ids[(size_t)b * cap + k] = pairs[k].first;
          h_val[(size_t)b * cap + k] = pairs[k].second;
        }
      }
      CUDA_CHECK(cudaMemcpyAsync(bias_n_dev_.ptr, h_n, B * sizeof(int), cudaMemcpyHostToDevice, stream_));
      CUDA_CHECK(cudaMemcpyAsync(bias_ids_dev_.ptr, h_ids, (size_t)B * cap * sizeof(int), cudaMemcpyHostToDevice, stream_));
      CUDA_CHECK(cudaMemcpyAsync(bias_val_dev_.ptr, h_val, (size_t)B * cap * sizeof(float), cudaMemcpyHostToDevice, stream_));
      p.step = t;
      p.prof = nullptr;
      p.logits_out = (t < dbg_steps) ? logits_dbg_.ptr + (size_t)t * B * V : nullptr;
      launch_step();
      launch_decoder_resolve(p, step_tok_dev_.ptr, stream_);
      steps_launched++;
      CUDA_CHECK(cudaMemcpyAsync(h_tok, step_tok_dev_.ptr, B * sizeof(int), cudaMemcpyDeviceToHost, stream_));
      CUDA_CHECK(cudaStreamSynchronize(stream_));
      for (int b = 0; b < B; b++) {
        if (finished[b]) continue;
        const int tok = h_tok[b];
        hooked_tokens[b].push_back(tok);
        if (tok == d_.eos || t + 1 >= mlen[b]) {
          finished[b] = 1;
          remaining--;
        }
        if (tok != d_.eos) hook->advance(b, tok);
      }
    }
    p.logits_out = nullptr;
    p.bias_static = nullptr; p.bias_dyn_n = nullptr; p.bias_dyn_ids = nullptr; p.bias_dyn_val = nullptr;
  } else {
    // Host-stepped greedy loop: logits of step t come back, the hook edits them, the host's first-max argmax
    // picks the id, and the id enters step t + 1 through the teacher-forcing input (the kernel's own EOS /
    // budget bookkeeping then follows the host's choice).
    const size_t fstride = (size_t)Smax + 1;
    std::vector<int> fhost((size_t)B * fstride, 0);
    for (int b = 0; b < B; b++) fhost[(size_t)b * fstride] = d_.bos;
    forced_dev_.reserve(fhost.size());
    CUDA_CHECK(cudaMemcpyAsync(forced_dev_.ptr, fhost.data(), fhost.size() * sizeof(int), cudaMemcpyHostToDevice, stream_));
    logits_dbg_.reserve((size_t)B * V);
    pin_logits_.reserve((size_t)B * V);
    std::vector<int> col(B, 0);
    std::vector<char> finished(B, 0);
    hooked_tokens.assign(B, std::vector<int32_t>{(int32_t)d_.bos});
    p.forced = forced_dev_.ptr;
    p.logits_out = logits_dbg_.ptr;
    int remaining = 0;
    for (int b = 0; b < B; b++) {
      finished[b] = mlen[b] <= 0;
      remaining += finished[b] ? 0 : 1;
    }
    steps_launched = 0;
    for (int t = 0; t < max_steps && remaining > 0; t++) {
      p.step = t;
      p.prof = nullptr;
      launch_step();
      steps_launched++;
      CUDA_CHECK(cudaMemcpyAsync(pin_logits_.ptr, logits_dbg_.ptr, (size_t)B * V * sizeof(float),
                                 cudaMemcpyDeviceToHost, stream_));
      CUDA_CHECK(cudaStreamSynchronize(stream_));
      for (int b = 0; b < B; b++) {
        col[b] = 0;
        if (finished[b]) continue;
        float* lg = pin_logits_.ptr + (size_t)b * V;
        hook->apply(b, lg, V);
        int best = 0;
        float best_v = lg[0];
        for (int v = 1; v < V; v++)
          if (lg[v] > best_v) { best_v = lg[v]; best = v; }
        hooked_tokens[b].push_back(best);
        col[b] = best;
        if (best == d_.eos || t + 1 >= mlen[b]) {
          finished[b] = 1;
          remaining--;
        }
        if (best != d_.eos) hook->advance(b, best);
      }
      if (t + 1 <= Smax)
        CUDA_CHECK(cudaMemcpy2DAsync(forced_dev_.ptr + (t + 1), fstride * sizeof(int), col.data(), sizeof(int),
                                     sizeof(int), (size_t)B, cudaMemcpyHostToDevice, stream_));
      CUDA_CHECK(cudaStreamSynchronize(stream_));  // `col` is reused next step
    }
    p.logits_out = nullptr;
  }
  if (prof_step >= 0) {
    std::vector<unsigned long long> h((size_t)grid * 512);
    CUDA_CHECK(cudaStreamSynchronize(stream_));
    CUDA_CHECK(cudaMemcpy(h.data(), prof_buf.ptr, h.size() * 8, cudaMemcpyDeviceToHost));
    for (int cta : {0, 1, 31, 77, 127, 128, 131, 140, 147}) {
      if (cta >= grid) continue;
      fprintf(stderr, "PROF cta %d:", cta);
      for (int i = 0; i < 512 && h[(size_t)cta * 512 + i]; i++)
        fprintf(stderr, " %u:%llu", (unsigned)(h[(size_t)cta * 512 + i] & 255), (h[(size_t)cta * 512 + i] >> 8) - (h[(size_t)cta * 512] >> 8));
      fprintf(stderr, "\n");
    }
  }
  if ((!verify || spliced) && !multi) {
    p.step = max_steps;
    launch_decoder_finalize(p, stream_);
    stage("decoder_finalize", -1, 32);
  }
  times_.decode_steps = steps_launched;
  times_.decode_launches = steps_launched + 1;
  times_.decoder_version = use_v4 ? 4 : use_v3 ? 3 : use_v2 ? 2 : 1;
  launches += steps_launched + 1;
  const auto hp4 = std::chrono::steady_clock::now();
  if (timing_) CUDA_CHECK(cudaEventRecord(ev_[4], stream_));

  // ---------------- results ----------------
  int* ht = pin_tokens_.ptr;
  int* hn = ht + (size_t)B * (Smax + 1);
  CUDA_CHECK(cudaMemcpyAsync(ht, tokens_dev_.ptr, (size_t)B * (Smax + 1) * sizeof(int), cudaMemcpyDeviceToHost, stream_));
  CUDA_CHECK(cudaMemcpyAsync(hn, ntok_dev_.ptr, B * sizeof(int), cudaMemcpyDeviceToHost, stream_));
  unsigned* h_err = reinterpret_cast<unsigned*>(hn + B + 1);  // spare word behind the counts and the n_active staging word
  *h_err = 0u;
  if (use_v3) CUDA_CHECK(cudaMemcpyAsync(h_err, sync3_.ptr + 1, sizeof(unsigned), cudaMemcpyDeviceToHost, stream_));
  // watchdog flags of the tcgen05 kernels outside the decoder step (plane-fed GEMM, fp32-staged GEMM, fused attention): a
  // wait that ran out of patience poisons its launch instead of trapping the context; raised here, after the synchronise
  unsigned* h_wd = reinterpret_cast<unsigned*>(hn + 2 * B + 1);
  h_wd[0] = h_wd[1] = h_wd[2] = 0u;
  gemm_planes_error_async(h_wd, stream_);
  gemm_tc_error_async(h_wd + 1, stream_);
  attention_tc_error_async(h_wd + 2, stream_);
  CUDA_CHECK(cudaStreamSynchronize(stream_));
  stream_dirty_ = false;
  if (h_wd[0] | h_wd[1] | h_wd[2]) {
    const unsigned which = h_wd[0] ? 0u : (h_wd[1] ? 1u : 2u);
    gemm_planes_clear_error(stream_);
    gemm_tc_clear_error(stream_);
    attention_tc_clear_error(stream_);
    CUDA_CHECK(cudaStreamSynchronize(stream_));
    static const char* names[3] = {"plane-fed GEMM", "fp32-staged GEMM", "fused attention"};
    throw std::runtime_error(std::string(names[which]) + " watchdog: a wait inside the kernel exceeded its limit "
                             "(results discarded; the device context is intact)");
  }
  if (host_prof) {
    const auto hp5 = std::chrono::steady_clock::now();
    auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    MSB_LOGF("host profile: run(): entry sync %.2f ms, metadata + workspaces %.2f, enqueue frontend..cross-kv %.2f, enqueue decode %.2f, wait for the GPU %.2f",
             ms(hp0, hp1), ms(hp1, hp2), ms(hp2, hp3), ms(hp3, hp4), ms(hp4, hp5));
  }
  if (*h_err != 0u)
    throw std::runtime_error("decoder step watchdog: a wait inside the persistent kernel exceeded its limit "
                             "(results discarded; the device context is intact)");
  tokens.assign(B, std::vector<int32_t>());
  for (int b = 0; b < B; b++) {
    const int n = std::min(hn[b], Smax + 1);
    tokens[b].assign(ht + (size_t)b * (Smax + 1), ht + (size_t)b * (Smax + 1) + n);
  }
  if (hook != nullptr) tokens = hooked_tokens;  // the device list holds its own (unhooked) argmax
  if (xattn != nullptr && p.xattn_out != nullptr) {
    // [B][L][H][S][Tpad] on the device -> per utterance [L * H][steps_b][T_b]
    const size_t per_utt = (size_t)L * H * p.xattn_steps * Tpad;
    std::vector<float> host(per_utt);
    xattn->resize(B);
    for (int b = 0; b < B; b++) {
      CrossAttention& xa = (*xattn)[b];
      xa.heads_total = L * H;
      xa.steps = std::max((int)tokens[b].size() - 1, 0);
      xa.frames = Tm[b];
      xa.prob.assign((size_t)xa.heads_total * xa.steps * xa.frames, 0.f);
      if (xa.steps == 0) continue;
      CUDA_CHECK(cudaMemcpy(host.data(), xattn_dev_.ptr + (size_t)b * per_utt, per_utt * sizeof(float),
                            cudaMemcpyDeviceToHost));
      for (int lh = 0; lh < xa.heads_total; lh++)
        for (int s2 = 0; s2 < xa.steps; s2++)
          std::memcpy(&xa.prob[((size_t)lh * xa.steps + s2) * xa.frames],
                      &host[((size_t)lh * p.xattn_steps + s2) * Tpad], (size_t)xa.frames * sizeof(float));
    }
  }
  if (dbg && dbg->logits && dbg_steps > 0) {
    dbg->logits->resize((size_t)dbg_steps * B * V);
    CUDA_CHECK(cudaMemcpy(dbg->logits->data(), logits_dbg_.ptr, dbg->logits->size() * sizeof(float), cudaMemcpyDeviceToHost));
    dbg->logits_steps = dbg_steps;
  }
  times_.kernel_launches = launches;
  if (timing_) {
    cudaEventElapsedTime(&times_.frontend_ms, ev_[0], ev_[1]);
    cudaEventElapsedTime(&times_.encoder_ms, ev_[1], ev_[2]);
    cudaEventElapsedTime(&times_.cross_kv_ms, ev_[2], ev_[3]);
    cudaEventElapsedTime(&times_.decode_ms, ev_[3], ev_[4]);
  }
}

}  // namespace msb
