// Expert-parallel MoE all-to-all over NVSwitch peer memory (SURVEY §2.4 "EP", §2.6 K11-EP, BASELINE config 5).
//
// The reference keeps all 64 routed experts of a layer on one stage (`mx.gather_qmm`); there is no
// collective anywhere in it.  Here the experts of every MoE layer can be sharded across the ranks of one
// NVSwitch domain and the token exchange is done by our own kernels in four launches — no NCCL call, no host hop:
//
//   dispatch  : slot reservation at the sender.  Every (token, k) pair claims a row in its owner's expert-major receive
//               buffer with one system-scope atomic on the owner's per-expert row counter, stores the token row there
//               (peer-mapped memory, 16 B stores) together with the address of the pair's slot in the sender's return
//               buffer; the last CTA publishes the step's sequence number to every destination (st.release.sys).
//               ep_dispatch_scatter_kernel below, or the router with the dispatch folded in (moe.cu, RouteEP).
//   gate/up   : the grouped swap-AB tcgen05 GEMM on the receive buffer; its CTAs first acquire every source's sequence
//               word (gemm_persistent.cu, GemmParams::ep_arrive), so the arrival wait needs no kernel of its own.
//   down      : the grouped down-projection's epilogue (GemmParams::row_dst / signal_peers) stores each fp32 output row
//               straight to its return address and the CTA completing the grid bumps every source's flag.
//   combine   : the source waits (in-kernel) for all W arrivals, then does the weighted combine (+ residual, optionally
//               + the next layer's input RMSNorm).
//
// Sequence numbers / counting flags + device-resident expectations make every step CUDA-graph replay safe; the per-expert
// row counters are double-buffered by step parity and the gate/up GEMM clears the other parity's.  Buffer reuse is race-free
// by construction: a source only dispatches layer l+1 after it has combined layer l, which requires every destination to have
// run its down-projection (consumed its receive buffer) for layer l and returned its rows.
#include "kernels.h"
#include "launch.h"
#include "ptx.cuh"

namespace b200 {

namespace {

constexpr int kMaxWorld = kEpMaxWorld;
using PeerTable = EpPeerTable;

// ---------------------------------------------------------------------------------------------- dispatch
// Sender-side slot reservation: each (token, k) pair claims a slot in the *destination's* expert-major receive buffer with one
// system-scope atomic on the destination's per-expert row counter (counters double-buffered by step parity), so rows land
// expert-contiguous where the grouped GEMM's TMA reads them and the receiver needs no counting sort or gather of its own.
// Next to the row the sender stores the address of the pair's slot in ITS return buffer *as mapped by the destination* (table
// exchanged at set-up), which is what the down-projection epilogue stores to.  Publication: the last CTA writes the step's sequence
// number to every destination (release.sys, after every CTA fenced its rows); the destination's grouped GEMM acquires all of them
// (gemm_persistent.cu, GemmParams::ep_arrive).
__global__ void ep_dispatch_scatter_kernel(const __nv_bfloat16* __restrict__ x, long long ld_x, const int* __restrict__ idx, int npairs,
                                           int top_k, int H, int experts_per_rank, int world, int my_rank, int cap_e,
                                           PeerTable recv_x,     // per dst: base of [E_local][cap_e][H] bf16
                                           PeerTable recv_dst,   // per dst: base of [E_local][cap_e] u64 (return address of each row)
                                           PeerTable recv_cnt,   // per dst: base of [2][E_local] int32 row counters
                                           PeerTable recv_seq,   // per dst: base of [world] u64 arrival words
                                           PeerTable my_ret,     // per dst: base of MY return buffer as mapped by that destination
                                           uint32_t* __restrict__ send_seq, unsigned int* __restrict__ done_counter,
                                           uint32_t* __restrict__ ret_expected) {
  pdl_sync();
  const int warps_per_cta = blockDim.x >> 5;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nvec = H / 8;
  const uint32_t seq = *reinterpret_cast<const volatile uint32_t*>(send_seq) + 1u;   // this step (bumped by the last CTA below)
  const int par = (int)(seq & 1u);
  for (int p = blockIdx.x * warps_per_cta + warp; p < npairs; p += gridDim.x * warps_per_cta) {
    const int e = idx[p];
    const int dst = e / experts_per_rank, le = e - dst * experts_per_rank;
    int slot = 0;
    if (lane == 0) slot = atomicAdd_system(reinterpret_cast<int*>(recv_cnt.p[dst]) + par * experts_per_rank + le, 1);
    slot = __shfl_sync(0xffffffffu, slot, 0);
    if (slot < cap_e) {
      const size_t row = (size_t)le * cap_e + slot;
      const uint4* src = reinterpret_cast<const uint4*>(x + (size_t)(p / top_k) * ld_x);
      uint4* drow = reinterpret_cast<uint4*>(recv_x.p[dst]) + row * nvec;
      for (int v = lane; v < nvec; v += 32) drow[v] = src[v];
      if (lane == 0)
        reinterpret_cast<unsigned long long*>(recv_dst.p[dst])[row] = my_ret.p[dst] + (unsigned long long)p * H * sizeof(float);
    }
  }
  __threadfence_system();
  __syncthreads();
  __shared__ bool last;
  if (threadIdx.x == 0) last = (atomicAdd(done_counter, 1u) + 1u == gridDim.x);
  __syncthreads();
  if (last) {
    __threadfence_system();
    for (int r = threadIdx.x; r < world; r += blockDim.x)
      st_release_sys_u64(reinterpret_cast<unsigned long long*>(recv_seq.p[r]) + my_rank, (unsigned long long)seq);
    __syncthreads();
    if (threadIdx.x == 0) {
      *send_seq = seq;
      *done_counter = 0u;
      if (ret_expected != nullptr) *ret_expected += (uint32_t)world;
    }
  }
}

// ---------------------------------------------------------------------------------------------- return + combine
// (the return all-to-all itself is the epilogue of the grouped down-projection: gemm_persistent.cu, GemmParams::row_dst)
// source side, fused: wait until every rank's down-projection has stored its share of my pairs into my return buffer,
// then the weighted combine (+ residual).  `expected` was advanced by this step's dispatch kernel (stream order).
__global__ void ep_combine_kernel(const uint32_t* flag, const uint32_t* __restrict__ expected_ptr, uint32_t* error_flag,
                                  unsigned long long timeout_ns, const float* __restrict__ ret_y, const float* __restrict__ wts,
                                  const __nv_bfloat16* __restrict__ residual, long long ld_res, __nv_bfloat16* __restrict__ out,
                                  long long ld_out, int T, int top_k, int H) {
  pdl_sync();
  if (threadIdx.x == 0) {
    const uint32_t expected = *reinterpret_cast<const volatile uint32_t*>(expected_ptr);
    unsigned long long t0;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
    while (true) {
      const uint32_t v = ld_acquire_sys(flag);
      if ((int32_t)(v - expected) >= 0) break;
      unsigned long long t1;
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
      if (t1 - t0 > timeout_ns) { if (error_flag) atomicExch(error_flag, 1u); break; }
      __nanosleep(32);
    }
    __threadfence_system();
  }
  __syncthreads();
  const int nvec = H / 8;
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)T * nvec) return;
  const int v = i % nvec;
  const int t = i / nvec;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  for (int k0 = 0; k0 < top_k; k0 += 4) {   // four pairs' loads in flight before any is used; accumulation order unchanged
    float4 a[4], b[4];
    float w[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int k = k0 + u < top_k ? k0 + u : top_k - 1;
      w[u] = k0 + u < top_k ? wts[(size_t)t * top_k + k] : 0.f;
      const float4* src = reinterpret_cast<const float4*>(ret_y + ((size_t)t * top_k + k) * H + v * 8);
      a[u] = __ldcv(src); b[u] = __ldcv(src + 1);   // rows were written by peers: never from a stale L1 line
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (k0 + u < top_k) {
        acc[0] += w[u] * a[u].x; acc[1] += w[u] * a[u].y; acc[2] += w[u] * a[u].z; acc[3] += w[u] * a[u].w;
        acc[4] += w[u] * b[u].x; acc[5] += w[u] * b[u].y; acc[6] += w[u] * b[u].z; acc[7] += w[u] * b[u].w;
      }
    }
  }
  if (residual != nullptr) {
    const uint4 r = reinterpret_cast<const uint4*>(residual + (size_t)t * ld_res)[v];
    const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      acc[2 * j] += __uint_as_float(rr[j] << 16);
      acc[2 * j + 1] += __uint_as_float(rr[j] & 0xffff0000u);
    }
  }
  uint4 o;
  __nv_bfloat162 h;
  h = __floats2bfloat162_rn(acc[0], acc[1]); o.x = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2bfloat162_rn(acc[2], acc[3]); o.y = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2bfloat162_rn(acc[4], acc[5]); o.z = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2bfloat162_rn(acc[6], acc[7]); o.w = *reinterpret_cast<uint32_t*>(&h);
  reinterpret_cast<uint4*>(out + (size_t)t * ld_out)[v] = o;
}

// Combine + the next layer's input RMSNorm (one CTA per token; same fusion as moe_combine_norm_kernel for the local MoE block)
constexpr int kEpCombThreads = 256;
constexpr int kEpCombMaxV = 4;   // H <= 8192
__global__ void __launch_bounds__(kEpCombThreads)
ep_combine_norm_kernel(const uint32_t* flag, const uint32_t* __restrict__ expected_ptr, uint32_t* error_flag, unsigned long long timeout_ns,
                       const float* __restrict__ ret_y, const float* __restrict__ wts, const __nv_bfloat16* __restrict__ residual,
                       long long ld_res, __nv_bfloat16* __restrict__ out, long long ld_out, int top_k, int H,
                       const __nv_bfloat16* __restrict__ norm_w, float norm_eps, __nv_bfloat16* __restrict__ normed, long long ld_normed) {
  pdl_sync();
  if (threadIdx.x == 0) {
    const uint32_t expected = *reinterpret_cast<const volatile uint32_t*>(expected_ptr);
    unsigned long long t0;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
    while (true) {
      const uint32_t v = ld_acquire_sys(flag);
      if ((int32_t)(v - expected) >= 0) break;
      unsigned long long t1;
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
      if (t1 - t0 > timeout_ns) { if (error_flag) atomicExch(error_flag, 1u); break; }
      __nanosleep(32);
    }
    __threadfence_system();
  }
  __shared__ float s_w[32];
  __shared__ float red[kEpCombThreads / 32];
  const int t = blockIdx.x;
  if (threadIdx.x < top_k) s_w[threadIdx.x] = wts[(size_t)t * top_k + threadIdx.x];
  __syncthreads();
  const int nvec = H / 8;
  uint4 keep[kEpCombMaxV];
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < kEpCombMaxV; ++i) {
    const int v = threadIdx.x + i * kEpCombThreads;
    if (v < nvec) {
      float acc[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = 0.f;
      for (int k0 = 0; k0 < top_k; k0 += 4) {
        float4 a[4], b[4];
        float w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int k = k0 + u < top_k ? k0 + u : top_k - 1;
          w[u] = k0 + u < top_k ? s_w[k] : 0.f;
          const float4* src = reinterpret_cast<const float4*>(ret_y + ((size_t)t * top_k + k) * H + v * 8);
          a[u] = __ldcv(src); b[u] = __ldcv(src + 1);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (k0 + u < top_k) {
            acc[0] += w[u] * a[u].x; acc[1] += w[u] * a[u].y; acc[2] += w[u] * a[u].z; acc[3] += w[u] * a[u].w;
            acc[4] += w[u] * b[u].x; acc[5] += w[u] * b[u].y; acc[6] += w[u] * b[u].z; acc[7] += w[u] * b[u].w;
          }
        }
      }
      if (residual != nullptr) {
        const uint4 r = reinterpret_cast<const uint4*>(residual + (size_t)t * ld_res)[v];
        const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) { acc[2 * j] += bf16_lo(rr[j]); acc[2 * j + 1] += bf16_hi(rr[j]); }
      }
      uint4 o;
      o.x = pack_bf16(acc[0], acc[1]); o.y = pack_bf16(acc[2], acc[3]);
      o.z = pack_bf16(acc[4], acc[5]); o.w = pack_bf16(acc[6], acc[7]);
      reinterpret_cast<uint4*>(out + (size_t)t * ld_out)[v] = o;
      keep[i] = o;
      const uint32_t oo[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) { const float a = bf16_lo(oo[j]), b = bf16_hi(oo[j]); ss += a * a + b * b; }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int i = 0; i < kEpCombThreads / 32; ++i) tot += red[i];
  const float inv = rsqrtf(tot / (float)H + norm_eps);
#pragma unroll
  for (int i = 0; i < kEpCombMaxV; ++i) {
    const int v = threadIdx.x + i * kEpCombThreads;
    if (v < nvec) {
      const uint4 g = __ldg(reinterpret_cast<const uint4*>(norm_w) + v);
      const uint32_t oo[4] = {keep[i].x, keep[i].y, keep[i].z, keep[i].w}, gg[4] = {g.x, g.y, g.z, g.w};
      uint32_t n[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) n[j] = pack_bf16(bf16_lo(oo[j]) * inv * bf16_lo(gg[j]), bf16_hi(oo[j]) * inv * bf16_hi(gg[j]));
      reinterpret_cast<uint4*>(normed + (size_t)t * ld_normed)[v] = make_uint4(n[0], n[1], n[2], n[3]);
    }
  }
}

constexpr unsigned long long kTimeoutNs = 20ull * 1000ull * 1000ull * 1000ull;

PeerTable make_table(const unsigned long long* v, int world) {
  PeerTable t;
  for (int i = 0; i < kMaxWorld; ++i) t.p[i] = i < world ? v[i] : 0ull;
  return t;
}

}  // namespace

cudaError_t ep_dispatch_scatter_launch(const void* x, long long ld_x, const int* idx, int npairs, int top_k, int H, int experts_per_rank,
                                       int world, int my_rank, int cap_e, const unsigned long long* recv_x,
                                       const unsigned long long* recv_dst, const unsigned long long* recv_cnt,
                                       const unsigned long long* recv_seq, const unsigned long long* my_ret, uint32_t* send_seq,
                                       unsigned int* done_counter, uint32_t* ret_expected, cudaStream_t s) {
  if (world > kMaxWorld || (H % 8)) return cudaErrorInvalidValue;
  int grid = (npairs + 7) / 8;
  if (grid < 1) grid = 1;
  if (grid > 592) grid = 592;
  (void)launch_pdl(ep_dispatch_scatter_kernel, dim3(grid), dim3(256), 0, s, static_cast<const __nv_bfloat16*>(x), ld_x, idx, npairs, top_k, H,
                   experts_per_rank, world, my_rank, cap_e, make_table(recv_x, world), make_table(recv_dst, world),
                   make_table(recv_cnt, world), make_table(recv_seq, world), make_table(my_ret, world), send_seq, done_counter,
                   ret_expected);
  return cudaGetLastError();
}

cudaError_t ep_combine_launch(const uint32_t* flag, const uint32_t* expected_ptr, uint32_t* error_flag, const float* ret_y,
                              const float* wts, const void* residual, long long ld_res, void* out, long long ld_out, int T, int top_k,
                              int H, cudaStream_t s, const void* norm_w, float norm_eps, void* normed, long long ld_normed) {
  if (T == 0) return cudaSuccess;
  if (H % 8) return cudaErrorInvalidValue;
  if (norm_w != nullptr) {
    if (normed == nullptr || top_k > 32 || H > kEpCombThreads * 8 * kEpCombMaxV) return cudaErrorInvalidValue;
    (void)launch_pdl(ep_combine_norm_kernel, dim3(T), dim3(kEpCombThreads), 0, s, flag, expected_ptr, error_flag, kTimeoutNs, ret_y, wts,
                     static_cast<const __nv_bfloat16*>(residual), ld_res, static_cast<__nv_bfloat16*>(out), ld_out, top_k, H,
                     static_cast<const __nv_bfloat16*>(norm_w), norm_eps, static_cast<__nv_bfloat16*>(normed), ld_normed);
    return cudaGetLastError();
  }
  const long long total = (long long)T * (H / 8);
  (void)launch_pdl(ep_combine_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, s, flag, expected_ptr, error_flag, kTimeoutNs,
                   ret_y, wts, static_cast<const __nv_bfloat16*>(residual), ld_res, static_cast<__nv_bfloat16*>(out), ld_out, T, top_k, H);
  return cudaGetLastError();
}

}  // namespace b200
