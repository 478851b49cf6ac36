// Host launch API of the non-GEMM sm_100a kernels (plain CUDA; the torch binding lives in bindings.cpp).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace b200 {

// ---- elementwise.cu
cudaError_t rmsnorm_launch(const void* x, long long ld_x, const void* w, const void* residual, long long ld_res,
                           void* out, long long ld_out, int rows, int H, float eps, bool gemma, cudaStream_t s, uint32_t* signal_flag = nullptr,
                           uint32_t signal_value = 0, unsigned int* done_counter = nullptr);
cudaError_t rope_launch(void* x, long long ld_t, long long ld_h, int heads, const int* positions, const float* inv_freq,
                        int rot_off, int rot_dim, bool interleaved, float mscale, int T, cudaStream_t s);
cudaError_t embed_launch(const long long* ids, const void* table, const void* scales, const void* biases, int bits, int group,
                         void* out, int H, float scale, int T, cudaStream_t s);
cudaError_t kv_write_launch(const void* k, long long k_ld_t, long long k_ld_h, const void* v, long long v_ld_t,
                            long long v_ld_h, void* kpool, void* vpool, const int* slots, int heads, int dk, int dv,
                            int page, int T, cudaStream_t s);
cudaError_t kv_write_mla_launch(const void* kv, long long kv_ld_t, const void* kpe, long long pe_ld_t, void* kpool,
                                void* vpool, const int* slots, int heads, int nope, int rd, int vd, int page, int T,
                                cudaStream_t s);
cudaError_t mla_rope_kv_launch(void* q, long long q_ld_t, long long q_ld_h, const void* kpe, long long pe_ld_t, const void* kv,
                               long long kv_ld_t, void* kpool, void* vpool, const int* slots, const int* positions,
                               const float* inv_freq, float mscale, int heads, int nope, int rd, int vd, int page, int T,
                               cudaStream_t s);

// bf16 [rows, K] -> MXFP8: e4m3 bytes [rows, K] + ue8m0 scales [rows, K / 32] (one per 32 K-values)
cudaError_t quant_mxfp8_launch(const void* x, long long ld_x, void* q, void* sf, long long rows, int K, cudaStream_t s);

// ---- attention.cu
struct PagedAttnArgs {
  const void* q; long long q_ld_t, q_ld_h;       // bf16 [T, q_heads, dk]
  const void* kpool; const void* vpool;          // bf16 [pages, kv_heads, page, dk|dv]
  const int* block_tables; int max_blocks;       // int32 [num_seqs, max_blocks]
  const int* positions;                          // int32 [T]   causal limit = position + 1
  const int* token_seq;                          // int32 [T]   sequence (block-table row) of each token
  int T, q_heads, kv_heads, dk_, dv_, page;
  float scale, softcap;
  int nsplit;                                    // KV splits (1 = write output directly)
  void* out; long long o_ld_t;                   // bf16 [T, q_heads * dv]
  float* part_acc; float* part_ml;               // split workspaces: [T*Hq*nsplit*dv], [T*Hq*nsplit*2]
};
cudaError_t paged_attention_launch(const PagedAttnArgs& a, cudaStream_t s);

// ---- attention_prefill.cu (tensor-core causal flash attention for prefill chunks)
struct FlashPrefillArgs {
  const void* q; long long q_ld_t, q_ld_h;
  const void* kpool; const void* vpool;
  const int* block_tables; int max_blocks;
  const int* cu_seqlens; const int* context_lens;
  int num_seqs, max_tiles, q_heads, kv_heads, dk_, dv_, page;
  float scale;
  void* out; long long o_ld_t;
};
bool flash_prefill_supported(int dk, int dv);
cudaError_t flash_prefill_launch(const FlashPrefillArgs& a, cudaStream_t s);

// ---- mla_decode.cu (absorbed-latent MLA: tcgen05 decode attention over the cached 576-dim latent, + its prologue)
cudaError_t mla_absorbed_prologue_launch(void* q, long long q_ld_t, const void* ckv, long long ckv_ld_t, const void* kpe,
                                         long long pe_ld_t, const void* norm_w, float eps, void* pool, const int* slots,
                                         const int* positions, const float* inv_freq, float mscale, int T, cudaStream_t s);
size_t mla_decode_workspace_floats(int B, int nsplit);
// q: bf16 [B, 16, 576] (head stride 576, token stride q_ld_t); pool: bf16 [num_pages, 1, 64, 576]; out: bf16 [B, 16, 512]
cudaError_t mla_decode_launch(const void* q, long long q_ld_t, int B, const void* pool, long long num_pages, int page,
                              const int* block_tables, int max_blocks, const int* context_lens, int max_ctx, float scale,
                              int nsplit, float* workspace, void* out, long long o_ld_t, long long* dbg, cudaStream_t s);

// ---- expert-parallel peer tables (ep.cu, and the router's fused dispatch in moe.cu)
constexpr int kEpMaxWorld = 16;
struct EpPeerTable {
  unsigned long long p[kEpMaxWorld];
};
// Fused router + expert-parallel dispatch (see ep.cu): the router CTA of a token reserves the slots of its top-k pairs
// in the owners' expert-major receive buffers (remote atomics), stores the (normalised) row there and takes part in the
// publication protocol of ep_dispatch_scatter_kernel — one kernel instead of norm + route + dispatch.
struct RouteEP {
  int enabled = 0, experts_per_rank = 0, world = 0, my_rank = 0, cap_e = 0;
  EpPeerTable recv_x, recv_dst, recv_cnt, recv_seq, my_ret;
  uint32_t* send_seq = nullptr;
  unsigned int* done_counter = nullptr;
  uint32_t* ret_expected = nullptr;
};

// ---- moe.cu
// router: fp32 softmax(x W^T) -> top-k (optionally group limited) -> weights * scaling (or normalised)
// `extra`: always-on experts appended after the routed ones (ids E .. E+extra-1, weight 1); idx / wts rows are top_k + extra wide
cudaError_t moe_route_launch(const void* x, long long ld_x, const void* gate_w, int T, int H, int E, int top_k,
                             int n_group, int topk_group, float scaling, bool norm_topk, int extra, int* idx, float* wts,
                             int* sc_counts, int sc_stride, int* sc_pair_row, void* sc_x, const void* norm_w, float norm_eps,
                             cudaStream_t s, const RouteEP* ep = nullptr, void* normed_out = nullptr, long long ld_normed = 0);
// (normed_out: also store the normalised row — the shared-expert branch of an expert-parallel block consumes it)
// (norm_w != nullptr: `x` is the un-normalised residual stream; the router normalises the row in shared memory first — the fused
//  pre-MoE RMSNorm — so logits and scattered expert inputs equal what a separate norm kernel would have produced)
// (sc_*: scatter mode for decode batches — every (token, k) pair claims slot `atomicAdd(sc_counts[e])` of expert e's fixed-stride
//  segment, its row index goes to sc_pair_row and the token row is copied to sc_x[row]: no separate permutation kernels)
// permutation: counts/offsets per expert, destination row of every (token, k) pair, gathered rows
cudaError_t moe_permute_launch(const int* idx, int T, int top_k, int E, int* expert_offsets /*E+1*/, int* pair_row /*T*k*/,
                               int* counters /*E scratch*/, const void* x, long long ld_x, void* x_perm, int H,
                               cudaStream_t s);
// y[t] = sum_k w[t,k] * y_perm[pair_row[t,k]] (+ residual[t]); out may be a peer pointer; optional release flag
cudaError_t moe_combine_launch(const void* y_perm, const int* pair_row, const float* wts, const void* residual,
                               long long ld_res, void* out, long long ld_out, int T, int top_k, int H,
                               uint32_t* signal_flag, uint32_t signal_value, unsigned int* done_counter, int* zero_counts,
                               int n_zero, const void* norm_w, float norm_eps, void* normed, long long ld_normed, cudaStream_t s);
// (norm_w != nullptr: additionally writes normed = rmsnorm(out) * norm_w — the next layer's input norm fused into the combine)

// ---- sampler.cu
cudaError_t apply_penalties_launch(float* logits, int B, int V, const int* rep_ctx, int C, const float* penalty,
                                   const int* bias_idx, const float* bias_val, int NB, cudaStream_t s);
// tokens/logprob per row; temperature==0 -> argmax, top_p in (0,1) -> nucleus; Philox-style counter RNG
// row_rng (optional, device): per-row [seed, step] pairs that override the scalars (graph-replay safe);
// tag_src/tag_dst (optional): 16 bytes copied verbatim next to the results (scheduler step id)
cudaError_t sample_launch(const float* logits, int B, int V, const float* temperature, const float* top_p,
                          unsigned long long seed, unsigned long long step, const unsigned long long* row_rng, long long* tokens,
                          float* logprobs, int top_k, long long* top_ids, float* top_lp, const void* tag_src, void* tag_dst,
                          cudaStream_t s);

// ---- p2p.cu
cudaError_t wait_flag_launch(const uint32_t* flag, uint32_t expected, uint32_t* error_flag, cudaStream_t s);
// error_host (optional): mapped pinned host word set on a timeout, so the host can poll for failures without a device sync
cudaError_t wait_flag_counter_launch(const uint32_t* flag, uint32_t* local_counter, uint32_t* error_flag, uint32_t* error_host,
                                     cudaStream_t s);
cudaError_t set_flag_launch(uint32_t* flag, uint32_t value, cudaStream_t s);
cudaError_t copy_signal_launch(const void* src, void* dst, size_t bytes, uint32_t* flag, uint32_t value,
                               unsigned int* done_counter, cudaStream_t s);
cudaError_t advance_meta_launch(int* positions, int* context_lens, int* slots, const int* block_tables, int max_blocks,
                                int page, int B, cudaStream_t s);

// ---- launch.h: the next kernel launched by this host thread gets plain (non-programmatic) dependencies
void pdl_skip_next();

// ---- ep.cu (expert-parallel all-to-all over peer memory)
// dispatch: sender-side slot reservation into each destination's expert-major receive buffer
cudaError_t ep_dispatch_scatter_launch(const void* x, long long ld_x, const int* idx, int npairs, int top_k, int H, int experts_per_rank,
                                       int world, int my_rank, int cap_e, const unsigned long long* recv_x,
                                       const unsigned long long* recv_dst, const unsigned long long* recv_cnt,
                                       const unsigned long long* recv_seq, const unsigned long long* my_ret, uint32_t* send_seq,
                                       unsigned int* done_counter, uint32_t* ret_expected, cudaStream_t s);
cudaError_t ep_combine_launch(const uint32_t* flag, const uint32_t* expected_ptr, uint32_t* error_flag, const float* ret_y,
                              const float* wts, const void* residual, long long ld_res, void* out, long long ld_out, int T, int top_k,
                              int H, cudaStream_t s, const void* norm_w = nullptr, float norm_eps = 0.f,
                              void* normed = nullptr, long long ld_normed = 0);

}  // namespace b200
