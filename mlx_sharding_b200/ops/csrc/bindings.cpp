// PyTorch bindings for the sm_100a kernels.  Everything launches on the current torch CUDA stream so
// the ops compose with torch.cuda.CUDAGraph capture; scratch buffers are process-lifetime (never freed,
// never moved once handed to a kernel) so captured graphs stay valid.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include <string>
#include <vector>

#include "gemm_tcgen05.h"
#include "kernels.h"

namespace py = pybind11;
using torch::Tensor;

namespace {

#define CUDA_OK(expr)                                                                             \
  do {                                                                                            \
    cudaError_t e__ = (expr);                                                                     \
    TORCH_CHECK(e__ == cudaSuccess, #expr, " failed: ", cudaGetErrorString(e__));                 \
  } while (0)

// number of kernels launched by this module (bench.py reports it as gpu_launches)
int64_t g_launches = 0;
#define LAUNCH_OK(expr) \
  do {                   \
    CUDA_OK(expr);       \
    ++g_launches;        \
  } while (0)

cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

void check_bf16(const Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
  TORCH_CHECK(t.scalar_type() == torch::kBFloat16, name, " must be bfloat16");
}
void check_rows(const Tensor& t, const char* name) {
  TORCH_CHECK(t.dim() == 2 && t.stride(1) == 1, name, " must be 2-D with a contiguous last dim");
}
// Operands the kernels read or write as 16-byte vectors (uint4 / float4) row by row: the first element of the view must be 16-byte
// aligned and so must every row start.  The address comes from the storage, not data_ptr(), which is null for a tensor with no
// rows, so a zero-row view is judged by where its rows would begin.  A single row never uses its row stride.
void check_vec16(const Tensor& t, const char* name) {
  const auto addr = reinterpret_cast<uintptr_t>(t.storage().data()) + static_cast<uintptr_t>(t.storage_offset() * t.element_size());
  TORCH_CHECK(addr % 16 == 0, name, " must start on a 16-byte boundary (a column offset that is not a multiple of ",
              16 / t.element_size(), " elements?)");
  TORCH_CHECK(t.size(0) == 1 || t.stride(0) % (16 / t.element_size()) == 0, name, " row stride must be a multiple of ",
              16 / t.element_size(), " elements (16 bytes)");
}

// ---- persistent scratch -----------------------------------------------------------------------------------------
struct Scratch {
  std::vector<Tensor> keep;  // every buffer ever handed out stays alive (graph safety)
  Tensor ws;                 // fp32 split-K / attention-split workspace
  Tensor counters;           // uint32 tile tickets (self-resetting) + done counters
  Tensor get_ws(int64_t floats, const torch::Device& dev) {
    if (!ws.defined() || ws.numel() < floats) {
      int64_t n = std::max<int64_t>(floats, 16 << 20);
      ws = torch::empty({n}, torch::dtype(torch::kFloat32).device(dev));
      keep.push_back(ws);
    }
    return ws;
  }
  Tensor get_counters(const torch::Device& dev) {
    if (!counters.defined()) {
      counters = torch::zeros({1 << 16}, torch::dtype(torch::kInt32).device(dev));
      keep.push_back(counters);
    }
    return counters;
  }
};
Scratch& scratch() {
  static Scratch s;
  return s;
}

int sm_count() {
  static int n = 0;
  if (n == 0) n = at::cuda::getCurrentDeviceProperties()->multiProcessorCount;
  return n;
}

// Token tile of the grouped (MoE) GEMMs: ~2x the average rows per expert but never below 64 — measured on B200
// (profiles/results.md, DeepSeek-V2-Lite decode): tiles of 16 / 32 tokens are *slower* than 64 even when experts hold ~6
// rows, and 256-token tiles lose to 64 / 128 at 24 rows per expert.  MLXB200_GROUPED_BN=<n> overrides (tuning).
int grouped_bn(int64_t max_rows, int64_t R, int64_t E) {
  static const int forced = [] { const char* e = std::getenv("MLXB200_GROUPED_BN"); return e ? std::atoi(e) : 0; }();
  if (forced > 0) return b200::gemm_pick_bn((int)std::min<int64_t>(max_rows, forced));
  return b200::gemm_pick_bn((int)std::min<int64_t>(max_rows, std::max<int64_t>(64, 2 * ((R + E - 1) / E))));
}

int auto_splits(int rows, int n, int k, bool grouped) {
  if (grouped || rows > 256) return 1;
  const int tiles = (n + 127) / 128;
  const int kb = (k + 63) / 64;
  int s = 1;
  // fill ~one wave of SMs while keeping >= 8 k-blocks per split (measured: profiles/splitk_sweep.md) ...
  while (tiles * (s * 2) <= sm_count() && kb / (s * 2) >= 8 && s < 4) s *= 2;
  // ... and for long reductions over few feature tiles (the folded MLA output projection: 16 tiles x 128 k-blocks) go to the
  // full portable cluster of 8 splits: 64 CTAs stream at ~100 GB/s each, so the kernel is per-SM-bandwidth bound below that
  static const bool split8 = [] { const char* e = std::getenv("MLXB200_SPLIT8"); return e != nullptr && e[0] == '1'; }();  // measured slower (0.12 ms / step): opt-in
  if (split8 && s == 4 && tiles * 8 <= sm_count() && kb / 8 >= 16) s = 8;
  return s;
}

// ---- GEMM -------------------------------------------------------------------------------------------------------
Tensor linear(const Tensor& x, const Tensor& w, const c10::optional<Tensor>& w2, const c10::optional<Tensor>& residual,
              const c10::optional<Tensor>& bias, int64_t act, double softcap, bool out_fp32, const c10::optional<Tensor>& out_,
              int64_t splits, int64_t signal_flag_ptr, int64_t signal_value) {
  check_bf16(x, "x"); check_bf16(w, "w"); check_rows(x, "x"); check_rows(w, "w");
  const c10::cuda::CUDAGuard guard(x.device());
  const int64_t T = x.size(0), K = x.size(1), N = w.size(0);
  TORCH_CHECK(w.size(1) == K, "x/w inner dims differ");
  Tensor out = out_.has_value() ? *out_ : torch::empty({T, N}, x.options().dtype(out_fp32 ? torch::kFloat32 : torch::kBFloat16));
  TORCH_CHECK(out.dim() == 2 && out.stride(1) == 1 && out.size(0) >= T && out.size(1) == N, "bad out tensor");
  check_vec16(out, "out");
  if (residual.has_value()) { check_bf16(*residual, "residual"); check_rows(*residual, "residual"); check_vec16(*residual, "residual"); }
  if (T == 0) return out;
  b200::GemmArgs a;
  a.x = x.data_ptr(); a.x_rows = T; a.ld_x = x.stride(0);
  a.w = w.data_ptr(); a.ld_w = w.stride(0);
  if (w2.has_value()) { check_bf16(*w2, "w2"); TORCH_CHECK(w2->sizes() == w.sizes() && w2->stride(0) == w.stride(0)); a.w2 = w2->data_ptr(); }
  a.m = (int)T; a.n = (int)N; a.k = (int)K; a.max_rows = (int)T;
  a.out = out.data_ptr(); a.ld_out = out.stride(0); a.out_fp32 = out.scalar_type() == torch::kFloat32;
  if (residual.has_value()) { a.residual = residual->data_ptr(); a.ld_res = residual->stride(0); }
  if (bias.has_value()) { check_bf16(*bias, "bias"); a.bias = bias->data_ptr(); }
  a.act = (int)act; a.softcap = (float)softcap;
  int sp = splits > 0 ? (int)splits : auto_splits((int)T, (int)N, (int)K, false);
  a.splits = sp;
  auto& sc = scratch();
  Tensor ctr = sc.get_counters(x.device());
  if (sp > 1) {
    const int bn = b200::gemm_pick_bn((int)T);
    Tensor ws = sc.get_ws((int64_t)b200::gemm_workspace_floats(a, bn, sp), x.device());
    a.workspace = ws.data_ptr<float>();
    a.tile_counters = reinterpret_cast<unsigned int*>(ctr.data_ptr<int>());
  }
  if (signal_flag_ptr != 0) {
    a.signal_flag = reinterpret_cast<uint32_t*>(signal_flag_ptr);
    a.signal_value = (uint32_t)signal_value;
    a.done_counter = reinterpret_cast<unsigned int*>(ctr.data_ptr<int>()) + 65535;
  }
  LAUNCH_OK(b200::gemm_launch(a, cur_stream()));
  return out;
}

Tensor grouped_linear(const Tensor& x, const Tensor& w, const c10::optional<Tensor>& w2, const Tensor& expert_offsets,
                      int64_t max_rows, int64_t act, bool out_fp32, const c10::optional<Tensor>& row_dst,
                      const c10::optional<Tensor>& signal_peers, const c10::optional<Tensor>& done_counter, int64_t expected_rows,
                      int64_t expert_stride, int64_t ep_arrive_ptr, const c10::optional<Tensor>& ep_seq, int64_t ep_error_ptr,
                      int64_t ep_world, bool ep_zero_other) {
  check_bf16(x, "x"); check_bf16(w, "w"); check_rows(x, "x");
  TORCH_CHECK(w.dim() == 3 && w.is_contiguous(), "w must be contiguous [E, N, K]");
  const c10::cuda::CUDAGuard guard(x.device());
  const int64_t R = x.size(0), K = x.size(1), E = w.size(0), N = w.size(1);
  // expert_stride > 0 (scatter layout): expert e owns rows [e * stride, e * stride + expert_offsets[e]) and the array holds COUNTS
  TORCH_CHECK(w.size(2) == K && expert_offsets.scalar_type() == torch::kInt32 &&
              (expert_stride > 0 ? (expert_offsets.numel() >= E && R >= E * expert_stride) : expert_offsets.numel() == E + 1));
  TORCH_CHECK(ep_arrive_ptr == 0 || (expert_stride > 0 && ep_seq.has_value() && expert_offsets.numel() >= 2 * E),
              "EP arrival wait needs the scatter layout with parity-double-buffered counts");
  // EP return path (parallel/ep.py): every output row goes to the address in row_dst[row] (the source rank's return buffer, peer
  // memory) and all `signal_peers` flags are bumped once every tile is stored — the un-fused return kernel disappears
  const bool ep_ret = row_dst.has_value();
  Tensor out = torch::empty({ep_ret ? 0 : R, N}, x.options().dtype(out_fp32 ? torch::kFloat32 : torch::kBFloat16));
  if (R == 0) return out;
  b200::GemmArgs a;
  a.x = x.data_ptr(); a.x_rows = R; a.ld_x = x.stride(0);
  a.w = w.data_ptr(); a.ld_w = K;
  if (w2.has_value()) { check_bf16(*w2, "w2"); TORCH_CHECK(w2->is_contiguous() && w2->sizes() == w.sizes()); a.w2 = w2->data_ptr(); }
  a.m = (int)R; a.n = (int)N; a.k = (int)K; a.max_rows = (int)std::min<int64_t>(max_rows, R);
  a.num_experts = (int)E; a.expert_offsets = expert_offsets.data_ptr<int>(); a.expert_stride = (int)expert_stride;
  if (ep_arrive_ptr != 0) {
    a.ep_arrive = reinterpret_cast<const unsigned long long*>(ep_arrive_ptr);
    a.ep_seq = reinterpret_cast<const uint32_t*>(ep_seq->data_ptr<int>());
    a.ep_error = reinterpret_cast<uint32_t*>(ep_error_ptr);
    a.ep_world = (int)ep_world; a.ep_zero_other = ep_zero_other;
  }
  if (ep_ret) {
    TORCH_CHECK(signal_peers.has_value() && done_counter.has_value() && row_dst->scalar_type() == torch::kInt64 &&
                signal_peers->scalar_type() == torch::kInt64 && row_dst->numel() >= R && row_dst->is_contiguous(), "bad EP return arguments");
    a.row_dst = reinterpret_cast<const unsigned long long*>(row_dst->data_ptr<int64_t>());
    a.signal_peers = reinterpret_cast<const unsigned long long*>(signal_peers->data_ptr<int64_t>());
    a.num_signal_peers = (int)signal_peers->numel();
    a.done_counter = reinterpret_cast<unsigned int*>(done_counter->data_ptr<int>());
  }
  // token tile sized for ~2x the average rows per expert (not the worst case): less padding in the MMA N dimension and
  // smaller token-tile loads; experts with more rows simply take further tiles of the persistent tile list
  // expected_rows (>0): the caller's estimate of the rows actually present when x is an over-sized buffer (EP receive side)
  a.bn = grouped_bn(a.max_rows, expected_rows > 0 ? expected_rows : R, E);
  a.out = out.data_ptr(); a.ld_out = N; a.out_fp32 = out_fp32; a.act = (int)act; a.splits = 1;
  LAUNCH_OK(b200::gemm_launch(a, cur_stream()));
  return out;
}

// ---- quantised GEMM (in-kernel MLX affine dequant) ---------------------------------------------------------------
struct QW { const Tensor& wq; const Tensor& st; const Tensor& bt; };
void check_q(const Tensor& wq, const Tensor& st, const Tensor& bt, int64_t rows, int64_t K, int64_t bits, int64_t group) {
  TORCH_CHECK(wq.is_cuda() && wq.scalar_type() == torch::kInt32 && wq.is_contiguous(), "packed weight must be contiguous int32");
  TORCH_CHECK(wq.numel() == rows * K * bits / 32, "packed weight size mismatch");
  check_bf16(st, "scales_t"); check_bf16(bt, "biases_t");
  TORCH_CHECK(st.is_contiguous() && bt.is_contiguous() && st.numel() == rows * (K / group) && bt.numel() == st.numel(), "scales_t/biases_t must be [K/g, rows]");
}
Tensor linear_q(const Tensor& x, const Tensor& wq, const Tensor& scales_t, const Tensor& biases_t, const c10::optional<Tensor>& wq2,
                const c10::optional<Tensor>& scales2_t, const c10::optional<Tensor>& biases2_t, int64_t bits, int64_t group, int64_t N,
                const c10::optional<Tensor>& residual, const c10::optional<Tensor>& bias, int64_t act, double softcap, bool out_fp32,
                const c10::optional<Tensor>& out_, int64_t splits, int64_t signal_flag_ptr, int64_t signal_value) {
  check_bf16(x, "x"); check_rows(x, "x");
  const c10::cuda::CUDAGuard guard(x.device());
  const int64_t T = x.size(0), K = x.size(1);
  check_q(wq, scales_t, biases_t, N, K, bits, group);
  Tensor out = out_.has_value() ? *out_ : torch::empty({T, N}, x.options().dtype(out_fp32 ? torch::kFloat32 : torch::kBFloat16));
  TORCH_CHECK(out.dim() == 2 && out.stride(1) == 1 && out.size(0) >= T && out.size(1) == N, "bad out tensor");
  check_vec16(out, "out");
  if (residual.has_value()) { check_bf16(*residual, "residual"); check_rows(*residual, "residual"); check_vec16(*residual, "residual"); }
  if (T == 0) return out;
  b200::GemmArgs a;
  a.x = x.data_ptr(); a.x_rows = T; a.ld_x = x.stride(0);
  a.w = wq.data_ptr(); a.q_scales_t = scales_t.data_ptr(); a.q_biases_t = biases_t.data_ptr();
  a.q_bits = (int)bits; a.q_group = (int)group;
  if (wq2.has_value()) {
    check_q(*wq2, *scales2_t, *biases2_t, N, K, bits, group);
    a.w2 = wq2->data_ptr(); a.q_scales2_t = scales2_t->data_ptr(); a.q_biases2_t = biases2_t->data_ptr();
  }
  a.m = (int)T; a.n = (int)N; a.k = (int)K; a.max_rows = (int)T;
  a.out = out.data_ptr(); a.ld_out = out.stride(0); a.out_fp32 = out.scalar_type() == torch::kFloat32;
  if (residual.has_value()) { a.residual = residual->data_ptr(); a.ld_res = residual->stride(0); }
  if (bias.has_value()) { check_bf16(*bias, "bias"); a.bias = bias->data_ptr(); }
  a.act = (int)act; a.softcap = (float)softcap;
  // quantised weights: 3.5x fewer bytes per tile, so batches of >= 64 tokens use the persistent kernel un-split; tiny decode
  // batches are latency-bound per tile like the bf16 path and take the same split-K heuristic (MLXB200_Q_SPLITK=0 disables)
  static const bool q_splitk = [] { const char* e = std::getenv("MLXB200_Q_SPLITK"); return !(e && e[0] == '0'); }();
  int sp = splits > 0 ? (int)splits : ((q_splitk && T <= 32) ? auto_splits((int)T, (int)N, (int)K, false) : 1);
  a.splits = sp;
  auto& sc = scratch();
  Tensor ctr = sc.get_counters(x.device());
  if (sp > 1) {
    const int bn = b200::gemm_pick_bn((int)T);
    Tensor ws = sc.get_ws((int64_t)b200::gemm_workspace_floats(a, bn, sp), x.device());
    a.workspace = ws.data_ptr<float>();
    a.tile_counters = reinterpret_cast<unsigned int*>(ctr.data_ptr<int>());
  }
  if (signal_flag_ptr != 0) {
    a.signal_flag = reinterpret_cast<uint32_t*>(signal_flag_ptr);
    a.signal_value = (uint32_t)signal_value;
    a.done_counter = reinterpret_cast<unsigned int*>(ctr.data_ptr<int>()) + 65535;
  }
  LAUNCH_OK(b200::gemm_q_launch(a, cur_stream()));
  return out;
}

Tensor grouped_linear_q(const Tensor& x, const Tensor& wq, const Tensor& scales_t, const Tensor& biases_t, const c10::optional<Tensor>& wq2,
                        const c10::optional<Tensor>& scales2_t, const c10::optional<Tensor>& biases2_t, int64_t bits, int64_t group,
                        int64_t E, int64_t N, const Tensor& expert_offsets, int64_t max_rows, int64_t act, bool out_fp32) {
  check_bf16(x, "x"); check_rows(x, "x");
  const c10::cuda::CUDAGuard guard(x.device());
  const int64_t R = x.size(0), K = x.size(1);
  check_q(wq, scales_t, biases_t, E * N, K, bits, group);
  TORCH_CHECK(expert_offsets.numel() == E + 1 && expert_offsets.scalar_type() == torch::kInt32);
  Tensor out = torch::empty({R, N}, x.options().dtype(out_fp32 ? torch::kFloat32 : torch::kBFloat16));
  if (R == 0) return out;
  b200::GemmArgs a;
  a.x = x.data_ptr(); a.x_rows = R; a.ld_x = x.stride(0);
  a.w = wq.data_ptr(); a.q_scales_t = scales_t.data_ptr(); a.q_biases_t = biases_t.data_ptr();
  a.q_bits = (int)bits; a.q_group = (int)group;
  if (wq2.has_value()) {
    check_q(*wq2, *scales2_t, *biases2_t, E * N, K, bits, group);
    a.w2 = wq2->data_ptr(); a.q_scales2_t = scales2_t->data_ptr(); a.q_biases2_t = biases2_t->data_ptr();
  }
  a.m = (int)R; a.n = (int)N; a.k = (int)K; a.max_rows = (int)std::min<int64_t>(max_rows, R);
  a.num_experts = (int)E; a.expert_offsets = expert_offsets.data_ptr<int>();
  // token tile sized for ~2x the average rows per expert (not the worst case): less padding in the MMA N dimension and
  // smaller token-tile loads; experts with more rows simply take further tiles of the persistent tile list
  a.bn = grouped_bn(a.max_rows, R, E);
  a.out = out.data_ptr(); a.ld_out = N; a.out_fp32 = out_fp32; a.act = (int)act; a.splits = 1;
  LAUNCH_OK(b200::gemm_q_launch(a, cur_stream()));
  return out;
}
bool gemm_q_supported(int64_t bits, int64_t group, int64_t k) { return b200::gemm_q_supported((int)bits, (int)group, (int)k); }

// ---- elementwise ------------------------------------------------------------------------------------------------
Tensor rmsnorm(const Tensor& x, const Tensor& w, double eps, bool gemma, const c10::optional<Tensor>& residual,
               const c10::optional<Tensor>& out_, int64_t signal_flag_ptr, int64_t signal_value) {
  check_bf16(x, "x"); check_bf16(w, "w"); check_rows(x, "x");
  const c10::cuda::CUDAGuard guard(x.device());
  Tensor out = out_.has_value() ? *out_ : torch::empty({x.size(0), x.size(1)}, x.options());
  TORCH_CHECK(out.scalar_type() == torch::kBFloat16 && out.stride(1) == 1 && out.size(0) >= x.size(0) && out.size(1) == x.size(1), "bad out tensor");
  check_vec16(x, "x"); check_vec16(out, "out");
  unsigned int* done = nullptr;
  if (signal_flag_ptr != 0) done = reinterpret_cast<unsigned int*>(scratch().get_counters(x.device()).data_ptr<int>()) + 65532;
  const void* res = nullptr; long long ldr = 0;
  if (residual.has_value()) {
    check_bf16(*residual, "residual"); check_rows(*residual, "residual"); check_vec16(*residual, "residual");
    res = residual->data_ptr(); ldr = residual->stride(0);
  }
  LAUNCH_OK(b200::rmsnorm_launch(x.data_ptr(), x.stride(0), w.data_ptr(), res, ldr, out.data_ptr(), out.stride(0), (int)x.size(0),
                               (int)x.size(1), (float)eps, gemma, cur_stream(), reinterpret_cast<uint32_t*>(signal_flag_ptr),
                               (uint32_t)signal_value, done));
  return out;
}

void rope_(Tensor x, const Tensor& positions, const Tensor& inv_freq, int64_t rot_off, int64_t rot_dim, bool interleaved, double mscale) {
  check_bf16(x, "x");
  TORCH_CHECK(x.dim() == 3 && x.stride(2) == 1, "x must be [T, heads, D] with contiguous D");
  TORCH_CHECK(positions.scalar_type() == torch::kInt32 && inv_freq.scalar_type() == torch::kFloat32 && inv_freq.is_cuda());
  const c10::cuda::CUDAGuard guard(x.device());
  LAUNCH_OK(b200::rope_launch(x.data_ptr(), x.stride(0), x.stride(1), (int)x.size(1), positions.data_ptr<int>(), inv_freq.data_ptr<float>(),
                            (int)rot_off, (int)rot_dim, interleaved, (float)mscale, (int)x.size(0), cur_stream()));
}

Tensor embed(const Tensor& ids, const Tensor& table, const c10::optional<Tensor>& scales, const c10::optional<Tensor>& biases,
             int64_t bits, int64_t group, double scale) {
  TORCH_CHECK(ids.is_cuda() && ids.scalar_type() == torch::kInt64 && ids.is_contiguous(), "ids must be contiguous int64 CUDA");
  const c10::cuda::CUDAGuard guard(ids.device());
  const int64_t T = ids.numel();
  int64_t H;
  if (bits == 0) { check_bf16(table, "table"); H = table.size(1); }
  else { TORCH_CHECK(table.scalar_type() == torch::kInt32 && scales.has_value() && biases.has_value()); check_bf16(*scales, "scales"); check_bf16(*biases, "biases"); H = table.size(1) * (32 / bits); }
  TORCH_CHECK(table.is_contiguous());
  Tensor out = torch::empty({T, H}, torch::dtype(torch::kBFloat16).device(ids.device()));
  LAUNCH_OK(b200::embed_launch(reinterpret_cast<const long long*>(ids.data_ptr<int64_t>()), table.data_ptr(),
                             scales.has_value() ? scales->data_ptr() : nullptr, biases.has_value() ? biases->data_ptr() : nullptr,
                             (int)bits, (int)group, out.data_ptr(), (int)H, (float)scale, (int)T, cur_stream()));
  return out;
}

void kv_write(const Tensor& k, const Tensor& v, Tensor kpool, Tensor vpool, const Tensor& slots) {
  check_bf16(k, "k"); check_bf16(v, "v"); check_bf16(kpool, "kpool"); check_bf16(vpool, "vpool");
  TORCH_CHECK(k.dim() == 3 && v.dim() == 3 && k.stride(2) == 1 && v.stride(2) == 1 && kpool.is_contiguous() && vpool.is_contiguous());
  TORCH_CHECK(slots.scalar_type() == torch::kInt32);
  const c10::cuda::CUDAGuard guard(k.device());
  LAUNCH_OK(b200::kv_write_launch(k.data_ptr(), k.stride(0), k.stride(1), v.data_ptr(), v.stride(0), v.stride(1), kpool.data_ptr(),
                                vpool.data_ptr(), slots.data_ptr<int>(), (int)k.size(1), (int)k.size(2), (int)v.size(2),
                                (int)kpool.size(2), (int)k.size(0), cur_stream()));
}

void kv_write_mla(const Tensor& kv, const Tensor& kpe, Tensor kpool, Tensor vpool, const Tensor& slots, int64_t nope, int64_t vd) {
  check_bf16(kv, "kv"); check_bf16(kpe, "kpe");
  TORCH_CHECK(kv.dim() == 3 && kv.stride(2) == 1 && kv.stride(1) == kv.size(2) && kpe.dim() == 2 && kpe.stride(1) == 1);
  TORCH_CHECK(kpool.is_contiguous() && vpool.is_contiguous() && slots.scalar_type() == torch::kInt32);
  const c10::cuda::CUDAGuard guard(kv.device());
  LAUNCH_OK(b200::kv_write_mla_launch(kv.data_ptr(), kv.stride(0), kpe.data_ptr(), kpe.stride(0), kpool.data_ptr(), vpool.data_ptr(),
                                    slots.data_ptr<int>(), (int)kv.size(1), (int)nope, (int)kpe.size(1), (int)vd, (int)kpool.size(2),
                                    (int)kv.size(0), cur_stream()));
}

void mla_rope_kv_write(Tensor q, const Tensor& kpe, const Tensor& kv, Tensor kpool, Tensor vpool, const Tensor& slots,
                       const Tensor& positions, const Tensor& inv_freq, double mscale, int64_t nope, int64_t vd) {
  check_bf16(q, "q"); check_bf16(kpe, "kpe"); check_bf16(kv, "kv");
  TORCH_CHECK(q.dim() == 3 && q.stride(2) == 1 && kpe.dim() == 2 && kpe.stride(1) == 1);
  TORCH_CHECK(kv.dim() == 3 && kv.stride(2) == 1 && kv.stride(1) == kv.size(2) && kpool.is_contiguous() && vpool.is_contiguous());
  TORCH_CHECK(slots.scalar_type() == torch::kInt32 && positions.scalar_type() == torch::kInt32 && inv_freq.scalar_type() == torch::kFloat32);
  const c10::cuda::CUDAGuard guard(q.device());
  LAUNCH_OK(b200::mla_rope_kv_launch(q.data_ptr(), q.stride(0), q.stride(1), kpe.data_ptr(), kpe.stride(0), kv.data_ptr(), kv.stride(0),
                                     kpool.data_ptr(), vpool.data_ptr(), slots.data_ptr<int>(), positions.data_ptr<int>(),
                                     inv_freq.data_ptr<float>(), (float)mscale, (int)q.size(1), (int)nope, (int)kpe.size(1), (int)vd,
                                     (int)kpool.size(2), (int)q.size(0), cur_stream()));
}

// ---- MXFP8 (block-scaled fp8) -----------------------------------------------------------------------------------
std::vector<Tensor> quant_mxfp8(const Tensor& x) {
  check_bf16(x, "x"); check_rows(x, "x");
  const c10::cuda::CUDAGuard guard(x.device());
  const int64_t R = x.size(0), K = x.size(1);
  TORCH_CHECK(K % 128 == 0, "MXFP8 GEMM operands need K % 128 == 0");
  Tensor q = torch::empty({R, K}, x.options().dtype(torch::kUInt8));
  Tensor sf = torch::empty({R, K / 32}, x.options().dtype(torch::kUInt8));
  LAUNCH_OK(b200::quant_mxfp8_launch(x.data_ptr(), x.stride(0), q.data_ptr(), sf.data_ptr(), R, (int)K, cur_stream()));
  return {q, sf};
}

// Y = (xq * xsf) (wq * wsf)^T on the tensor cores (kind::mxf8f6f4.block_scale).  Dense: wq [N, K]; grouped: wq [E, N, K] with
// expert_offsets (offsets, or per-expert counts when expert_stride > 0) exactly like grouped_linear.
Tensor linear_fp8(const Tensor& xq, const Tensor& xsf, const Tensor& wq, const Tensor& wsf, const c10::optional<Tensor>& w2q,
                  const c10::optional<Tensor>& w2sf, const c10::optional<Tensor>& expert_offsets, int64_t max_rows,
                  const c10::optional<Tensor>& residual, int64_t act, bool out_fp32, int64_t expected_rows, int64_t expert_stride) {
  auto u8 = [](const Tensor& t, const char* n) { TORCH_CHECK(t.is_cuda() && t.scalar_type() == torch::kUInt8 && t.is_contiguous(), n, " must be contiguous uint8"); };
  u8(xq, "xq"); u8(xsf, "xsf"); u8(wq, "wq"); u8(wsf, "wsf");
  const c10::cuda::CUDAGuard guard(xq.device());
  const bool grouped = expert_offsets.has_value();
  const int64_t R = xq.size(0), K = xq.size(1), N = wq.size(-2), E = grouped ? wq.size(0) : 0;
  TORCH_CHECK(wq.size(-1) == K && K % 128 == 0 && N % 128 == 0 && xsf.numel() == R * (K / 32) && wsf.numel() == wq.numel() / 32,
              "MXFP8 GEMM: K % 128 == 0, N % 128 == 0, one scale per 32 K-values");
  Tensor out = torch::empty({R, N}, xq.options().dtype(out_fp32 ? torch::kFloat32 : torch::kBFloat16));
  if (R == 0) return out;
  b200::GemmArgs a;
  a.x = xq.data_ptr(); a.x_rows = R; a.ld_x = K; a.x_sf = xsf.data_ptr();
  a.w = wq.data_ptr(); a.ld_w = K; a.w_sf = wsf.data_ptr();
  if (w2q.has_value()) { u8(*w2q, "w2q"); u8(*w2sf, "w2sf"); TORCH_CHECK(w2q->sizes() == wq.sizes()); a.w2 = w2q->data_ptr(); a.w2_sf = w2sf->data_ptr(); }
  a.m = (int)R; a.n = (int)N; a.k = (int)K;
  a.max_rows = (int)std::min<int64_t>(grouped ? max_rows : R, R);
  if (grouped) {
    TORCH_CHECK(expert_offsets->scalar_type() == torch::kInt32 && (expert_stride > 0 ? expert_offsets->numel() >= E : expert_offsets->numel() == E + 1));
    a.num_experts = (int)E; a.expert_offsets = expert_offsets->data_ptr<int>(); a.expert_stride = (int)expert_stride;
    a.bn = grouped_bn(a.max_rows, expected_rows > 0 ? expected_rows : R, E);
  }
  if (residual.has_value()) { check_bf16(*residual, "residual"); check_rows(*residual, "residual"); a.residual = residual->data_ptr(); a.ld_res = residual->stride(0); }
  a.out = out.data_ptr(); a.ld_out = N; a.out_fp32 = out_fp32; a.act = (int)act;
  LAUNCH_OK(b200::gemm_fp8_launch(a, cur_stream()));
  return out;
}

// ---- attention --------------------------------------------------------------------------------------------------
Tensor paged_attention(const Tensor& q, const Tensor& kpool, const Tensor& vpool, const Tensor& block_tables, const Tensor& positions,
                       const Tensor& token_seq, double scale, double softcap, int64_t max_ctx) {
  check_bf16(q, "q"); check_bf16(kpool, "kpool"); check_bf16(vpool, "vpool");
  TORCH_CHECK(q.dim() == 3 && q.stride(2) == 1 && kpool.is_contiguous() && vpool.is_contiguous());
  TORCH_CHECK(block_tables.scalar_type() == torch::kInt32 && block_tables.is_contiguous() && positions.scalar_type() == torch::kInt32 &&
              token_seq.scalar_type() == torch::kInt32);
  const c10::cuda::CUDAGuard guard(q.device());
  const int T = (int)q.size(0), Hq = (int)q.size(1), Hk = (int)kpool.size(1), dv = (int)vpool.size(3);
  Tensor out = torch::empty({T, Hq, dv}, q.options());
  if (T == 0) return out;
  b200::PagedAttnArgs a;
  a.q = q.data_ptr(); a.q_ld_t = q.stride(0); a.q_ld_h = q.stride(1);
  a.kpool = kpool.data_ptr(); a.vpool = vpool.data_ptr();
  a.block_tables = block_tables.data_ptr<int>(); a.max_blocks = (int)block_tables.size(1);
  a.positions = positions.data_ptr<int>(); a.token_seq = token_seq.data_ptr<int>();
  a.T = T; a.q_heads = Hq; a.kv_heads = Hk; a.dk_ = (int)kpool.size(3); a.dv_ = dv; a.page = (int)kpool.size(2);
  a.scale = (float)scale; a.softcap = (float)softcap;
  // split the KV range until ~2 waves of CTAs exist, keeping >= 256 positions per split
  int nsplit = 1;
  const int ctas = T * Hk;
  while (ctas * nsplit < 2 * sm_count() && max_ctx / (nsplit * 2) >= 256 && nsplit < 32) nsplit *= 2;
  a.nsplit = nsplit;
  a.out = out.data_ptr(); a.o_ld_t = (long long)Hq * dv;
  a.part_acc = nullptr; a.part_ml = nullptr;
  if (nsplit > 1) {
    const int64_t n_acc = (int64_t)T * Hq * nsplit * dv, n_ml = (int64_t)T * Hq * nsplit * 2;
    Tensor ws = scratch().get_ws(n_acc + n_ml, q.device());
    a.part_acc = ws.data_ptr<float>();
    a.part_ml = ws.data_ptr<float>() + n_acc;
  }
  LAUNCH_OK(b200::paged_attention_launch(a, cur_stream()));
  if (nsplit > 1) ++g_launches;  // + LSE combine kernel
  return out;
}

Tensor flash_prefill(const Tensor& q, const Tensor& kpool, const Tensor& vpool, const Tensor& block_tables, const Tensor& cu_seqlens,
                     const Tensor& context_lens, double scale, int64_t num_tokens) {
  check_bf16(q, "q"); check_bf16(kpool, "kpool"); check_bf16(vpool, "vpool");
  TORCH_CHECK(q.dim() == 3 && q.stride(2) == 1 && kpool.is_contiguous() && vpool.is_contiguous());
  TORCH_CHECK(block_tables.scalar_type() == torch::kInt32 && block_tables.is_contiguous() && cu_seqlens.scalar_type() == torch::kInt32 &&
              context_lens.scalar_type() == torch::kInt32);
  const c10::cuda::CUDAGuard guard(q.device());
  const int T = (int)q.size(0), Hq = (int)q.size(1), dv = (int)vpool.size(3);
  Tensor out = torch::empty({T, Hq, dv}, q.options());
  if (T == 0) return out;
  b200::FlashPrefillArgs a;
  a.q = q.data_ptr(); a.q_ld_t = q.stride(0); a.q_ld_h = q.stride(1);
  a.kpool = kpool.data_ptr(); a.vpool = vpool.data_ptr();
  a.block_tables = block_tables.data_ptr<int>(); a.max_blocks = (int)block_tables.size(1);
  a.cu_seqlens = cu_seqlens.data_ptr<int>(); a.context_lens = context_lens.data_ptr<int>();
  a.num_seqs = (int)context_lens.numel(); a.max_tiles = (int)((num_tokens + 63) / 64 + a.num_seqs);
  a.q_heads = Hq; a.kv_heads = (int)kpool.size(1); a.dk_ = (int)kpool.size(3); a.dv_ = dv; a.page = (int)kpool.size(2);
  a.scale = (float)scale; a.out = out.data_ptr(); a.o_ld_t = (long long)Hq * dv;
  LAUNCH_OK(b200::flash_prefill_launch(a, cur_stream()));
  return out;
}
bool flash_prefill_supported(int64_t dk, int64_t dv) { return b200::flash_prefill_supported((int)dk, (int)dv); }

// ---- absorbed-latent MLA ----------------------------------------------------------------------------------------
void mla_absorbed_prologue(Tensor q, const Tensor& ckv, const Tensor& kpe, const Tensor& norm_w, double eps, Tensor pool,
                           const Tensor& slots, const Tensor& positions, const Tensor& inv_freq, double mscale) {
  check_bf16(q, "q"); check_bf16(ckv, "ckv"); check_bf16(kpe, "kpe"); check_bf16(norm_w, "norm_w"); check_bf16(pool, "pool");
  TORCH_CHECK(q.dim() == 3 && q.size(1) == 16 && q.size(2) == 576 && q.stride(2) == 1 && q.stride(1) == 576, "q must be [T,16,576] with packed heads");
  TORCH_CHECK(ckv.dim() == 2 && ckv.size(1) == 512 && ckv.stride(1) == 1 && kpe.dim() == 2 && kpe.size(1) == 64 && kpe.stride(1) == 1);
  TORCH_CHECK(pool.is_contiguous() && pool.size(-1) == 576 && norm_w.is_contiguous() && norm_w.numel() == 512);
  TORCH_CHECK(slots.scalar_type() == torch::kInt32 && positions.scalar_type() == torch::kInt32 && inv_freq.scalar_type() == torch::kFloat32 &&
              inv_freq.numel() == 32);
  const c10::cuda::CUDAGuard guard(q.device());
  LAUNCH_OK(b200::mla_absorbed_prologue_launch(q.data_ptr(), q.stride(0), ckv.data_ptr(), ckv.stride(0), kpe.data_ptr(), kpe.stride(0),
                                               norm_w.data_ptr(), (float)eps, pool.data_ptr(), slots.data_ptr<int>(),
                                               positions.data_ptr<int>(), inv_freq.data_ptr<float>(), (float)mscale, (int)q.size(0),
                                               cur_stream()));
}

Tensor mla_decode(const Tensor& q, const Tensor& pool, const Tensor& block_tables, const Tensor& context_lens, double scale,
                  int64_t max_ctx, int64_t nsplit_req, const c10::optional<Tensor>& trace) {
  check_bf16(q, "q"); check_bf16(pool, "pool");
  TORCH_CHECK(q.dim() == 3 && q.size(1) == 16 && q.size(2) == 576 && q.stride(2) == 1 && q.stride(1) == 576, "q must be [B,16,576] with packed heads");
  TORCH_CHECK(pool.is_contiguous() && pool.dim() == 4 && pool.size(1) == 1 && pool.size(2) == 64 && pool.size(3) == 576,
              "latent pool must be [pages, 1, 64, 576]");
  TORCH_CHECK(block_tables.scalar_type() == torch::kInt32 && block_tables.is_contiguous() && context_lens.scalar_type() == torch::kInt32);
  const c10::cuda::CUDAGuard guard(q.device());
  const int B = (int)q.size(0);
  Tensor out = torch::empty({B, 16, 512}, q.options());
  if (B == 0) return out;
  const int tiles = (int)((max_ctx + 63) / 64);
  int nsplit = (int)nsplit_req;
  if (nsplit <= 0) {
    // flash-decoding split: until one wave of CTAs exists, keeping >= 8 tiles (512 tokens) per split.  A split costs a second
    // kernel (the LSE combine) and a partial round trip: measured (bench/mla_bench.py sweep) 64 x 128 tokens 14.4 us un-split vs
    // 19.5 us in two splits, 64 x 1024 best at 2, 64 x 4096 at 2-4, 8 x 16 k at 16 — i.e. ~8+ tiles per split.  `max_ctx` is
    // the *bound* the caller's block tables allow (serving pads them to 8 pages), so short contexts must not split on it.
    nsplit = 1;
    while (B * nsplit < sm_count() && tiles / (nsplit * 2) >= 8 && nsplit < 64) nsplit *= 2;
  }
  if (nsplit > tiles) nsplit = tiles > 0 ? tiles : 1;
  float* ws = nullptr;
  if (nsplit > 1) ws = scratch().get_ws((int64_t)b200::mla_decode_workspace_floats(B, nsplit), q.device()).data_ptr<float>();
  LAUNCH_OK(b200::mla_decode_launch(q.data_ptr(), q.stride(0), B, pool.data_ptr(), pool.size(0), 64, block_tables.data_ptr<int>(),
                                    (int)block_tables.size(1), context_lens.data_ptr<int>(), (int)max_ctx, (float)scale, nsplit, ws,
                                    out.data_ptr(), (long long)16 * 512,
                                    trace.has_value() ? reinterpret_cast<long long*>(trace->data_ptr<int64_t>()) : nullptr, cur_stream()));
  if (nsplit > 1) ++g_launches;
  return out;
}

// ---- MoE --------------------------------------------------------------------------------------------------------
std::vector<Tensor> moe_route(const Tensor& x, const Tensor& gate_w, int64_t top_k, int64_t n_group, int64_t topk_group, double scaling,
                              bool norm_topk, int64_t extra, const c10::optional<Tensor>& sc_counts, int64_t sc_stride,
                              const c10::optional<Tensor>& sc_x, const c10::optional<Tensor>& norm_w, double norm_eps) {
  check_bf16(x, "x"); check_bf16(gate_w, "gate_w"); check_rows(x, "x");
  TORCH_CHECK(gate_w.is_contiguous());
  if (norm_w.has_value()) { check_bf16(*norm_w, "norm_w"); TORCH_CHECK(norm_w->is_contiguous() && norm_w->numel() == x.size(1), "bad norm weight"); }
  const c10::cuda::CUDAGuard guard(x.device());
  const int T = (int)x.size(0);
  Tensor idx = torch::empty({T, top_k + extra}, torch::dtype(torch::kInt32).device(x.device()));
  Tensor w = torch::empty({T, top_k + extra}, torch::dtype(torch::kFloat32).device(x.device()));
  const bool scatter = sc_counts.has_value();
  Tensor pair_row;
  if (scatter) {
    TORCH_CHECK(sc_x.has_value() && sc_counts->scalar_type() == torch::kInt32 && sc_x->scalar_type() == torch::kBFloat16 && sc_x->is_contiguous() &&
                sc_x->size(1) == x.size(1) && sc_stride >= T && sc_x->size(0) >= sc_counts->numel() * sc_stride &&
                sc_counts->numel() >= gate_w.size(0) + extra, "bad scatter buffers");
    pair_row = torch::empty({T, top_k + extra}, torch::dtype(torch::kInt32).device(x.device()));
  }
  LAUNCH_OK(b200::moe_route_launch(x.data_ptr(), x.stride(0), gate_w.data_ptr(), T, (int)x.size(1), (int)gate_w.size(0), (int)top_k,
                                 (int)n_group, (int)topk_group, (float)scaling, norm_topk, (int)extra, idx.data_ptr<int>(), w.data_ptr<float>(),
                                 scatter ? sc_counts->data_ptr<int>() : nullptr, (int)sc_stride, scatter ? pair_row.data_ptr<int>() : nullptr,
                                 scatter ? sc_x->data_ptr() : nullptr, norm_w.has_value() ? norm_w->data_ptr() : nullptr, (float)norm_eps,
                                 cur_stream()));
  if (scatter) return {idx, w, pair_row};
  return {idx, w};
}

std::vector<Tensor> moe_permute(const Tensor& idx, const Tensor& x, int64_t E) {
  check_bf16(x, "x"); check_rows(x, "x");
  TORCH_CHECK(idx.scalar_type() == torch::kInt32 && idx.is_contiguous());
  const c10::cuda::CUDAGuard guard(x.device());
  const int T = (int)idx.size(0), k = (int)idx.size(1), H = (int)x.size(1);
  auto io = torch::dtype(torch::kInt32).device(x.device());
  Tensor offs = torch::empty({E + 1}, io), pair_row = torch::empty({T * k}, io);
  Tensor xp = torch::empty({(int64_t)T * k, H}, x.options());
  LAUNCH_OK(b200::moe_permute_launch(idx.data_ptr<int>(), T, k, (int)E, offs.data_ptr<int>(), pair_row.data_ptr<int>(), nullptr,
                                   x.data_ptr(), x.stride(0), xp.data_ptr(), H, cur_stream()));
  ++g_launches;  // offsets + gather
  return {offs, pair_row, xp};
}

Tensor moe_combine(const Tensor& y_perm, const Tensor& pair_row, const Tensor& wts, const c10::optional<Tensor>& residual,
                   const c10::optional<Tensor>& out_, int64_t top_k, int64_t signal_flag_ptr, int64_t signal_value,
                   const c10::optional<Tensor>& zero_counts, const c10::optional<Tensor>& norm_w, double norm_eps,
                   const c10::optional<Tensor>& normed) {
  TORCH_CHECK(y_perm.is_cuda() && y_perm.scalar_type() == torch::kFloat32 && y_perm.is_contiguous());
  TORCH_CHECK(!zero_counts.has_value() || zero_counts->scalar_type() == torch::kInt32);
  TORCH_CHECK(wts.scalar_type() == torch::kFloat32 && wts.is_contiguous() && pair_row.scalar_type() == torch::kInt32);
  const c10::cuda::CUDAGuard guard(y_perm.device());
  const int H = (int)y_perm.size(1), T = (int)(pair_row.numel() / top_k);
  Tensor out = out_.has_value() ? *out_ : torch::empty({T, H}, y_perm.options().dtype(torch::kBFloat16));
  TORCH_CHECK(out.scalar_type() == torch::kBFloat16 && out.stride(1) == 1);
  const void* res = nullptr; long long ldr = 0;
  if (residual.has_value()) { check_bf16(*residual, "residual"); check_rows(*residual, "residual"); res = residual->data_ptr(); ldr = residual->stride(0); }
  if (norm_w.has_value()) {
    check_bf16(*norm_w, "norm_w");
    TORCH_CHECK(normed.has_value() && normed->scalar_type() == torch::kBFloat16 && normed->stride(1) == 1 && normed->size(0) >= T &&
                normed->size(1) == H && norm_w->is_contiguous() && norm_w->numel() == H, "bad fused-norm arguments");
  }
  unsigned int* done = nullptr;
  if (signal_flag_ptr != 0) done = reinterpret_cast<unsigned int*>(scratch().get_counters(y_perm.device()).data_ptr<int>()) + 65534;
  LAUNCH_OK(b200::moe_combine_launch(y_perm.data_ptr(), pair_row.data_ptr<int>(), wts.data_ptr<float>(), res, ldr, out.data_ptr(),
                                   out.stride(0), T, (int)top_k, H, reinterpret_cast<uint32_t*>(signal_flag_ptr), (uint32_t)signal_value,
                                   done, zero_counts.has_value() ? zero_counts->data_ptr<int>() : nullptr,
                                   zero_counts.has_value() ? (int)zero_counts->numel() : 0,
                                   norm_w.has_value() ? norm_w->data_ptr() : nullptr, (float)norm_eps,
                                   normed.has_value() ? normed->data_ptr() : nullptr, normed.has_value() ? normed->stride(0) : 0, cur_stream()));
  return out;
}

// ---- sampler ----------------------------------------------------------------------------------------------------
void apply_penalties_(Tensor logits, const Tensor& rep_ctx, const Tensor& penalty, const Tensor& bias_idx, const Tensor& bias_val) {
  TORCH_CHECK(logits.is_cuda() && logits.scalar_type() == torch::kFloat32 && logits.is_contiguous());
  TORCH_CHECK(rep_ctx.scalar_type() == torch::kInt32 && bias_idx.scalar_type() == torch::kInt32 && rep_ctx.is_contiguous() && bias_idx.is_contiguous());
  const c10::cuda::CUDAGuard guard(logits.device());
  LAUNCH_OK(b200::apply_penalties_launch(logits.data_ptr<float>(), (int)logits.size(0), (int)logits.size(1), rep_ctx.data_ptr<int>(),
                                       (int)rep_ctx.size(1), penalty.data_ptr<float>(), bias_idx.data_ptr<int>(), bias_val.data_ptr<float>(),
                                       (int)bias_idx.size(1), cur_stream()));
}

std::vector<Tensor> sample(const Tensor& logits, const Tensor& temperature, const Tensor& top_p, int64_t seed, int64_t step, int64_t top_k) {
  TORCH_CHECK(logits.is_cuda() && logits.scalar_type() == torch::kFloat32 && logits.is_contiguous());
  const c10::cuda::CUDAGuard guard(logits.device());
  const int B = (int)logits.size(0);
  auto dev = logits.device();
  Tensor tokens = torch::empty({B}, torch::dtype(torch::kInt64).device(dev));
  Tensor lp = torch::empty({B}, torch::dtype(torch::kFloat32).device(dev));
  Tensor top_ids = torch::empty({B, top_k}, torch::dtype(torch::kInt64).device(dev));
  Tensor top_lp = torch::empty({B, top_k}, torch::dtype(torch::kFloat32).device(dev));
  LAUNCH_OK(b200::sample_launch(logits.data_ptr<float>(), B, (int)logits.size(1), temperature.data_ptr<float>(), top_p.data_ptr<float>(),
                              (unsigned long long)seed, (unsigned long long)step, nullptr, reinterpret_cast<long long*>(tokens.data_ptr<int64_t>()),
                              lp.data_ptr<float>(), (int)top_k, reinterpret_cast<long long*>(top_ids.data_ptr<int64_t>()),
                              top_lp.data_ptr<float>(), nullptr, nullptr, cur_stream()));
  return {tokens, lp, top_ids, top_lp};
}

// Graph-replay-safe sampler: every per-step input (temperature, top-p, per-row RNG state, step tag) lives in device memory and the
// outputs go to caller-owned buffers (views into the result message that travels back to stage 0).
void sample_into(const Tensor& logits, const Tensor& temperature, const Tensor& top_p, const Tensor& row_rng, int64_t top_k,
                 Tensor tokens, Tensor lp, const c10::optional<Tensor>& top_ids, const c10::optional<Tensor>& top_lp,
                 const c10::optional<Tensor>& tag_src, const c10::optional<Tensor>& tag_dst) {
  TORCH_CHECK(logits.is_cuda() && logits.scalar_type() == torch::kFloat32 && logits.is_contiguous());
  TORCH_CHECK(row_rng.scalar_type() == torch::kInt64 && row_rng.is_contiguous() && row_rng.numel() >= 2 * logits.size(0));
  TORCH_CHECK(tokens.scalar_type() == torch::kInt64 && lp.scalar_type() == torch::kFloat32);
  TORCH_CHECK(top_k == 0 || (top_ids.has_value() && top_lp.has_value()), "top_k > 0 needs top_ids / top_lp buffers");
  TORCH_CHECK(tag_src.has_value() == tag_dst.has_value());
  if (tag_src.has_value())
    TORCH_CHECK(tag_src->numel() * tag_src->element_size() >= 16 && tag_dst->numel() * tag_dst->element_size() >= 16 &&
                reinterpret_cast<uintptr_t>(tag_src->data_ptr()) % 16 == 0 && reinterpret_cast<uintptr_t>(tag_dst->data_ptr()) % 16 == 0);
  const c10::cuda::CUDAGuard guard(logits.device());
  LAUNCH_OK(b200::sample_launch(logits.data_ptr<float>(), (int)logits.size(0), (int)logits.size(1), temperature.data_ptr<float>(),
                              top_p.data_ptr<float>(), 0ull, 0ull, reinterpret_cast<const unsigned long long*>(row_rng.data_ptr<int64_t>()),
                              reinterpret_cast<long long*>(tokens.data_ptr<int64_t>()), lp.data_ptr<float>(), (int)top_k,
                              top_k ? reinterpret_cast<long long*>(top_ids->data_ptr<int64_t>()) : nullptr,
                              top_k ? top_lp->data_ptr<float>() : nullptr, tag_src.has_value() ? tag_src->data_ptr() : nullptr,
                              tag_dst.has_value() ? tag_dst->data_ptr() : nullptr, cur_stream()));
}

// ---- P2P / IPC --------------------------------------------------------------------------------------------------
py::tuple ipc_alloc(int64_t nbytes) {
  void* p = nullptr;
  CUDA_OK(cudaMalloc(&p, (size_t)nbytes));
  CUDA_OK(cudaMemset(p, 0, (size_t)nbytes));
  cudaIpcMemHandle_t h;
  CUDA_OK(cudaIpcGetMemHandle(&h, p));
  return py::make_tuple((int64_t) reinterpret_cast<uintptr_t>(p), py::bytes(reinterpret_cast<const char*>(&h), sizeof(h)));
}
int64_t ipc_open(const std::string& handle) {
  TORCH_CHECK(handle.size() == sizeof(cudaIpcMemHandle_t), "bad IPC handle size");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle.data(), sizeof(h));
  void* p = nullptr;
  CUDA_OK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  return (int64_t) reinterpret_cast<uintptr_t>(p);
}
void enable_peer_access(int64_t peer) {
  int can = 0, dev = 0;
  CUDA_OK(cudaGetDevice(&dev));
  CUDA_OK(cudaDeviceCanAccessPeer(&can, dev, (int)peer));
  TORCH_CHECK(can, "device ", dev, " cannot access peer ", peer);
  cudaError_t e = cudaDeviceEnablePeerAccess((int)peer, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return; }
  CUDA_OK(e);
}
Tensor tensor_from_ptr(int64_t ptr, std::vector<int64_t> shape, const std::string& dtype, int64_t device) {
  auto dt = dtype == "bfloat16" ? torch::kBFloat16 : dtype == "float32" ? torch::kFloat32 : dtype == "int32" ? torch::kInt32
            : dtype == "int64" ? torch::kInt64 : torch::kUInt8;
  return torch::from_blob(reinterpret_cast<void*>(ptr), shape, torch::dtype(dt).device(torch::kCUDA, (int)device));
}
void wait_flag(int64_t flag_ptr, int64_t expected, int64_t error_ptr) {
  LAUNCH_OK(b200::wait_flag_launch(reinterpret_cast<const uint32_t*>(flag_ptr), (uint32_t)expected, reinterpret_cast<uint32_t*>(error_ptr), cur_stream()));
}
void wait_flag_counter(int64_t flag_ptr, int64_t counter_ptr, int64_t error_ptr, int64_t error_host_ptr) {
  LAUNCH_OK(b200::wait_flag_counter_launch(reinterpret_cast<const uint32_t*>(flag_ptr), reinterpret_cast<uint32_t*>(counter_ptr),
                                         reinterpret_cast<uint32_t*>(error_ptr), reinterpret_cast<uint32_t*>(error_host_ptr),
                                         cur_stream()));
}
void set_flag(int64_t flag_ptr, int64_t value) { LAUNCH_OK(b200::set_flag_launch(reinterpret_cast<uint32_t*>(flag_ptr), (uint32_t)value, cur_stream())); }
void copy_signal(const Tensor& src, int64_t dst_ptr, int64_t flag_ptr, int64_t value) {
  TORCH_CHECK(src.is_cuda() && src.is_contiguous());
  const c10::cuda::CUDAGuard guard(src.device());
  LAUNCH_OK(b200::copy_signal_launch(src.data_ptr(), reinterpret_cast<void*>(dst_ptr), (size_t)src.numel() * src.element_size(),
                                   reinterpret_cast<uint32_t*>(flag_ptr), (uint32_t)value,
                                   reinterpret_cast<unsigned int*>(scratch().get_counters(src.device()).data_ptr<int>()) + 65533,
                                   cur_stream()));
}
// allocate the persistent scratch eagerly (must happen before any CUDA-graph capture)
void init_scratch(int64_t device, int64_t ws_floats) {
  const c10::cuda::CUDAGuard guard(torch::Device(torch::kCUDA, (int)device));
  scratch().get_counters(torch::Device(torch::kCUDA, (int)device));
  scratch().get_ws(ws_floats, torch::Device(torch::kCUDA, (int)device));
}
void advance_meta(Tensor positions, Tensor context_lens, Tensor slots, const Tensor& block_tables, int64_t page) {
  TORCH_CHECK(positions.scalar_type() == torch::kInt32 && block_tables.scalar_type() == torch::kInt32 && block_tables.is_contiguous());
  const c10::cuda::CUDAGuard guard(positions.device());
  LAUNCH_OK(b200::advance_meta_launch(positions.data_ptr<int>(), context_lens.data_ptr<int>(), slots.data_ptr<int>(), block_tables.data_ptr<int>(),
                                    (int)block_tables.size(1), (int)page, (int)positions.numel(), cur_stream()));
}

// ---- expert parallel --------------------------------------------------------------------------------------------
std::vector<unsigned long long> to_u64(const std::vector<int64_t>& v) {
  std::vector<unsigned long long> o(v.size());
  for (size_t i = 0; i < v.size(); ++i) o[i] = (unsigned long long)v[i];
  return o;
}
void ep_dispatch_scatter(const Tensor& x, const Tensor& idx, int64_t experts_per_rank, int64_t my_rank, int64_t cap_e,
                         std::vector<int64_t> recv_x, std::vector<int64_t> recv_dst, std::vector<int64_t> recv_cnt,
                         std::vector<int64_t> recv_seq, std::vector<int64_t> my_ret, Tensor send_seq, Tensor done_counter,
                         const c10::optional<Tensor>& ret_expected) {
  check_bf16(x, "x"); check_rows(x, "x");
  TORCH_CHECK(idx.scalar_type() == torch::kInt32 && idx.is_contiguous() && idx.dim() == 2);
  const c10::cuda::CUDAGuard guard(x.device());
  const int world = (int)recv_x.size();
  auto a = to_u64(recv_x), b = to_u64(recv_dst), c = to_u64(recv_cnt), d = to_u64(recv_seq), e = to_u64(my_ret);
  LAUNCH_OK(b200::ep_dispatch_scatter_launch(x.data_ptr(), x.stride(0), idx.data_ptr<int>(), (int)idx.numel(), (int)idx.size(1), (int)x.size(1),
                                             (int)experts_per_rank, world, (int)my_rank, (int)cap_e, a.data(), b.data(), c.data(), d.data(),
                                             e.data(), reinterpret_cast<uint32_t*>(send_seq.data_ptr<int>()),
                                             reinterpret_cast<unsigned int*>(done_counter.data_ptr<int>()),
                                             ret_expected.has_value() ? reinterpret_cast<uint32_t*>(ret_expected->data_ptr<int>()) : nullptr,
                                             cur_stream()));
}

// Router + expert-parallel dispatch in one kernel: returns {idx, wts}; optionally normalises `x` first (norm_w) and
// stores the normalised rows (normed_out) for the shared-expert branch.
std::vector<Tensor> ep_route_dispatch(const Tensor& x, const Tensor& gate_w, int64_t top_k, int64_t n_group, int64_t topk_group, double scaling,
                                      bool norm_topk, int64_t experts_per_rank, int64_t my_rank, int64_t cap_e, std::vector<int64_t> recv_x,
                                      std::vector<int64_t> recv_dst, std::vector<int64_t> recv_cnt, std::vector<int64_t> recv_seq,
                                      std::vector<int64_t> my_ret, Tensor send_seq, Tensor done_counter, const c10::optional<Tensor>& ret_expected,
                                      const c10::optional<Tensor>& norm_w, double norm_eps, const c10::optional<Tensor>& normed_out) {
  check_bf16(x, "x"); check_bf16(gate_w, "gate_w"); check_rows(x, "x");
  TORCH_CHECK(gate_w.is_contiguous());
  const c10::cuda::CUDAGuard guard(x.device());
  const int T = (int)x.size(0), world = (int)recv_x.size();
  TORCH_CHECK(T >= 1 && T <= 1024 && world <= b200::kEpMaxWorld, "fused route + dispatch needs 1 <= T <= 1024");
  if (norm_w.has_value()) { check_bf16(*norm_w, "norm_w"); TORCH_CHECK(norm_w->is_contiguous() && norm_w->numel() == x.size(1)); }
  if (normed_out.has_value()) { check_bf16(*normed_out, "normed_out"); check_rows(*normed_out, "normed_out"); TORCH_CHECK(normed_out->size(0) >= T && normed_out->size(1) == x.size(1)); }
  Tensor idx = torch::empty({T, top_k}, torch::dtype(torch::kInt32).device(x.device()));
  Tensor w = torch::empty({T, top_k}, torch::dtype(torch::kFloat32).device(x.device()));
  b200::RouteEP ep;
  ep.enabled = 1; ep.experts_per_rank = (int)experts_per_rank; ep.world = world; ep.my_rank = (int)my_rank; ep.cap_e = (int)cap_e;
  auto fill = [&](b200::EpPeerTable& t, const std::vector<int64_t>& v) {
    for (int i = 0; i < b200::kEpMaxWorld; ++i) t.p[i] = i < world ? (unsigned long long)v[i] : 0ull;
  };
  TORCH_CHECK((int)recv_dst.size() == world && (int)recv_cnt.size() == world && (int)recv_seq.size() == world && (int)my_ret.size() == world);
  fill(ep.recv_x, recv_x); fill(ep.recv_dst, recv_dst); fill(ep.recv_cnt, recv_cnt); fill(ep.recv_seq, recv_seq); fill(ep.my_ret, my_ret);
  ep.send_seq = reinterpret_cast<uint32_t*>(send_seq.data_ptr<int>());
  ep.done_counter = reinterpret_cast<unsigned int*>(done_counter.data_ptr<int>());
  ep.ret_expected = ret_expected.has_value() ? reinterpret_cast<uint32_t*>(ret_expected->data_ptr<int>()) : nullptr;
  LAUNCH_OK(b200::moe_route_launch(x.data_ptr(), x.stride(0), gate_w.data_ptr(), T, (int)x.size(1), (int)gate_w.size(0), (int)top_k,
                                   (int)n_group, (int)topk_group, (float)scaling, norm_topk, 0, idx.data_ptr<int>(), w.data_ptr<float>(),
                                   nullptr, 0, nullptr, nullptr, norm_w.has_value() ? norm_w->data_ptr() : nullptr, (float)norm_eps,
                                   cur_stream(), &ep, normed_out.has_value() ? normed_out->data_ptr() : nullptr,
                                   normed_out.has_value() ? normed_out->stride(0) : 0));
  return {idx, w};
}

Tensor ep_combine(int64_t flag_ptr, const Tensor& expected, int64_t error_ptr, const Tensor& ret_y, const Tensor& wts,
                  const c10::optional<Tensor>& residual, const c10::optional<Tensor>& out_, const c10::optional<Tensor>& norm_w,
                  double norm_eps, const c10::optional<Tensor>& normed) {
  TORCH_CHECK(ret_y.scalar_type() == torch::kFloat32 && ret_y.is_contiguous() && wts.scalar_type() == torch::kFloat32 && wts.is_contiguous());
  const c10::cuda::CUDAGuard guard(ret_y.device());
  const int64_t T = wts.size(0), k = wts.size(1), H = ret_y.size(1);
  Tensor out = out_.has_value() ? *out_ : torch::empty({T, H}, ret_y.options().dtype(torch::kBFloat16));
  TORCH_CHECK(out.stride(1) == 1 && out.size(0) >= T && T * k <= ret_y.size(0));
  if (residual.has_value()) { check_bf16(*residual, "residual"); check_rows(*residual, "residual"); }
  if (norm_w.has_value()) {
    check_bf16(*norm_w, "norm_w");
    TORCH_CHECK(normed.has_value() && normed->scalar_type() == torch::kBFloat16 && normed->stride(1) == 1 && normed->size(0) >= T &&
                normed->size(1) == H && norm_w->is_contiguous() && norm_w->numel() == H, "bad fused-norm arguments");
  }
  LAUNCH_OK(b200::ep_combine_launch(reinterpret_cast<const uint32_t*>(flag_ptr), reinterpret_cast<const uint32_t*>(expected.data_ptr<int>()),
                                    reinterpret_cast<uint32_t*>(error_ptr), ret_y.data_ptr<float>(), wts.data_ptr<float>(),
                                    residual.has_value() ? residual->data_ptr() : nullptr, residual.has_value() ? residual->stride(0) : 0,
                                    out.data_ptr(), out.stride(0), (int)T, (int)k, (int)H, cur_stream(),
                                    norm_w.has_value() ? norm_w->data_ptr() : nullptr, (float)norm_eps,
                                    normed.has_value() ? normed->data_ptr() : nullptr, normed.has_value() ? normed->stride(0) : 0));
  return out;
}
}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "mlx_sharding_b200 sm_100a kernels";
  m.def("linear", &linear, py::arg("x"), py::arg("w"), py::arg("w2") = py::none(), py::arg("residual") = py::none(),
        py::arg("bias") = py::none(), py::arg("act") = 0, py::arg("softcap") = 0.0, py::arg("out_fp32") = false,
        py::arg("out") = py::none(), py::arg("splits") = 0, py::arg("signal_flag_ptr") = 0, py::arg("signal_value") = 0);
  m.def("grouped_linear", &grouped_linear, py::arg("x"), py::arg("w"), py::arg("w2") = py::none(), py::arg("expert_offsets"),
        py::arg("max_rows"), py::arg("act") = 0, py::arg("out_fp32") = false, py::arg("row_dst") = py::none(),
        py::arg("signal_peers") = py::none(), py::arg("done_counter") = py::none(), py::arg("expected_rows") = 0,
        py::arg("expert_stride") = 0, py::arg("ep_arrive_ptr") = 0, py::arg("ep_seq") = py::none(), py::arg("ep_error_ptr") = 0,
        py::arg("ep_world") = 0, py::arg("ep_zero_other") = false);
  m.def("linear_q", &linear_q);
  m.def("grouped_linear_q", &grouped_linear_q);
  m.def("gemm_q_supported", &gemm_q_supported);
  m.def("rmsnorm", &rmsnorm, py::arg("x"), py::arg("w"), py::arg("eps"), py::arg("gemma") = false, py::arg("residual") = py::none(),
        py::arg("out") = py::none(), py::arg("signal_flag_ptr") = 0, py::arg("signal_value") = 0);
  m.def("rope_", &rope_);
  m.def("embed", &embed, py::arg("ids"), py::arg("table"), py::arg("scales") = py::none(), py::arg("biases") = py::none(),
        py::arg("bits") = 0, py::arg("group") = 64, py::arg("scale") = 1.0);
  m.def("kv_write", &kv_write);
  m.def("kv_write_mla", &kv_write_mla);
  m.def("mla_rope_kv_write", &mla_rope_kv_write);
  m.def("paged_attention", &paged_attention);
  m.def("flash_prefill", &flash_prefill);
  m.def("flash_prefill_supported", &flash_prefill_supported);
  m.def("mla_absorbed_prologue", &mla_absorbed_prologue);
  m.def("mla_decode", &mla_decode, py::arg("q"), py::arg("pool"), py::arg("block_tables"), py::arg("context_lens"), py::arg("scale"),
        py::arg("max_ctx"), py::arg("nsplit") = 0, py::arg("trace") = py::none());
  m.def("quant_mxfp8", &quant_mxfp8);
  m.def("linear_fp8", &linear_fp8, py::arg("xq"), py::arg("xsf"), py::arg("wq"), py::arg("wsf"), py::arg("w2q") = py::none(),
        py::arg("w2sf") = py::none(), py::arg("expert_offsets") = py::none(), py::arg("max_rows") = 0, py::arg("residual") = py::none(),
        py::arg("act") = 0, py::arg("out_fp32") = false, py::arg("expected_rows") = 0, py::arg("expert_stride") = 0);
  m.def("moe_route", &moe_route, py::arg("x"), py::arg("gate_w"), py::arg("top_k"), py::arg("n_group"), py::arg("topk_group"),
        py::arg("scaling"), py::arg("norm_topk"), py::arg("extra") = 0, py::arg("sc_counts") = py::none(), py::arg("sc_stride") = 0,
        py::arg("sc_x") = py::none(), py::arg("norm_w") = py::none(), py::arg("norm_eps") = 1e-6);
  m.def("moe_permute", &moe_permute);
  m.def("moe_combine", &moe_combine, py::arg("y_perm"), py::arg("pair_row"), py::arg("wts"), py::arg("residual") = py::none(),
        py::arg("out") = py::none(), py::arg("top_k"), py::arg("signal_flag_ptr") = 0, py::arg("signal_value") = 0,
        py::arg("zero_counts") = py::none(), py::arg("norm_w") = py::none(), py::arg("norm_eps") = 1e-6, py::arg("normed") = py::none());
  m.def("apply_penalties_", &apply_penalties_);
  m.def("sample", &sample);
  m.def("sample_into", &sample_into, py::arg("logits"), py::arg("temperature"), py::arg("top_p"), py::arg("row_rng"), py::arg("top_k"),
        py::arg("tokens"), py::arg("logprobs"), py::arg("top_ids") = py::none(), py::arg("top_lp") = py::none(),
        py::arg("tag_src") = py::none(), py::arg("tag_dst") = py::none());
  m.def("ipc_alloc", &ipc_alloc);
  m.def("ipc_open", &ipc_open);
  m.def("enable_peer_access", &enable_peer_access);
  m.def("tensor_from_ptr", &tensor_from_ptr);
  m.def("wait_flag", &wait_flag);
  m.def("wait_flag_counter", &wait_flag_counter, py::arg("flag_ptr"), py::arg("counter_ptr"), py::arg("error_ptr"),
        py::arg("error_host_ptr") = 0);
  m.def("set_flag", &set_flag);
  m.def("copy_signal", &copy_signal);
  m.def("advance_meta", &advance_meta);
  m.def("ep_dispatch_scatter", &ep_dispatch_scatter, py::arg("x"), py::arg("idx"), py::arg("experts_per_rank"), py::arg("my_rank"),
        py::arg("cap_e"), py::arg("recv_x"), py::arg("recv_dst"), py::arg("recv_cnt"), py::arg("recv_seq"), py::arg("my_ret"),
        py::arg("send_seq"), py::arg("done_counter"), py::arg("ret_expected") = py::none());
  m.def("ep_combine", &ep_combine, py::arg("flag_ptr"), py::arg("expected"), py::arg("error_ptr"), py::arg("ret_y"), py::arg("wts"),
        py::arg("residual") = py::none(), py::arg("out") = py::none(), py::arg("norm_w") = py::none(), py::arg("norm_eps") = 1e-6,
        py::arg("normed") = py::none());
  m.def("ep_route_dispatch", &ep_route_dispatch, py::arg("x"), py::arg("gate_w"), py::arg("top_k"), py::arg("n_group"), py::arg("topk_group"),
        py::arg("scaling"), py::arg("norm_topk"), py::arg("experts_per_rank"), py::arg("my_rank"), py::arg("cap_e"), py::arg("recv_x"),
        py::arg("recv_dst"), py::arg("recv_cnt"), py::arg("recv_seq"), py::arg("my_ret"), py::arg("send_seq"), py::arg("done_counter"),
        py::arg("ret_expected") = py::none(), py::arg("norm_w") = py::none(), py::arg("norm_eps") = 1e-6, py::arg("normed_out") = py::none());
  m.def("init_scratch", &init_scratch);
  m.def("launch_count", []() { return g_launches; });
  m.def("pdl_skip_next", []() { b200::pdl_skip_next(); });
  m.def("sm_arch", []() { return std::string("sm_100a"); });
}
