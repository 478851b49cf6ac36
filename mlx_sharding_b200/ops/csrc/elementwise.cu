// Memory-bound helper kernels of a decoder layer (SURVEY §2.6 K1, K2, K6, K7-append): embedding gather
// with in-kernel MLX-affine dequant, RMSNorm (+Gemma variant, + post-norm residual), rotary embedding
// (half-split and interleaved/YaRN), paged KV-cache append (plain and MLA-assembling).
// The reference gets all of these from MLX Metal kernels (mx.fast.rms_norm / mx.fast.rope / Embedding /
// KVCache.update_and_fetch via mlx_lm blocks); these are from-scratch sm_100a kernels: 128-bit
// vectorised accesses, one warp-shuffle reduction tree, no shared-memory round trips beyond one exchange.
#include <cuda_fp8.h>

#include "kernels.h"
#include "launch.h"
#include "ptx.cuh"

namespace b200 {

namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void unpack8(const uint4& r, float (&f)[8]) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) { f[2 * j] = bf16_lo(w[j]); f[2 * j + 1] = bf16_hi(w[j]); }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 o;
  o.x = pack_bf16(f[0], f[1]); o.y = pack_bf16(f[2], f[3]); o.z = pack_bf16(f[4], f[5]); o.w = pack_bf16(f[6], f[7]);
  return o;
}

}  // namespace

// ------------------------------------------------------------------------------------------------ MXFP8 activation quantisation
// x bf16 [R, K] -> e4m3 bytes [R, K] + one ue8m0 scale per 32 consecutive K values [R, K / 32] (OCP MX): scale = 2^ceil(log2(amax /
// 448)), the smallest power of two that brings the block into e4m3 range, elements rounded to nearest-even.  One thread per 8
// elements, 4 threads per block of 32.  (The weights get the same format once at load: utils/quant.py::to_mxfp8.)
__global__ void quant_mxfp8_kernel(const __nv_bfloat16* __restrict__ x, long long ld_x, uint8_t* __restrict__ q, uint8_t* __restrict__ sf,
                                   int K, long long total_vec) {
  pdl_sync();
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const int nvec = K / 8;
  const bool in = i < total_vec;
  const long long r = in ? i / nvec : 0;
  const int v = in ? (int)(i % nvec) : 0;
  float f[8];
  float amax = 0.f;
  if (in) {
    const uint4 raw = reinterpret_cast<const uint4*>(x + r * ld_x)[v];
    unpack8(raw, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) amax = fmaxf(amax, fabsf(f[j]));
  }
  amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 1));
  amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 2));
  if (!in) return;
  const uint32_t bits = __float_as_uint(amax * (1.0f / 448.0f));
  uint32_t e = ((bits >> 23) & 0xffu) + ((bits & 0x7fffffu) ? 1u : 0u);   // biased exponent of the next power of two >= amax / 448
  if (e > 254u) e = 254u;
  const float inv = __uint_as_float((254u - e) << 23);                     // 2^-(e - 127)
  uint32_t w[2];
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const __nv_fp8x2_storage_t lo = __nv_cvt_float2_to_fp8x2(make_float2(f[4 * j] * inv, f[4 * j + 1] * inv), __NV_SATFINITE, __NV_E4M3);
    const __nv_fp8x2_storage_t hi = __nv_cvt_float2_to_fp8x2(make_float2(f[4 * j + 2] * inv, f[4 * j + 3] * inv), __NV_SATFINITE, __NV_E4M3);
    w[j] = (uint32_t)lo | ((uint32_t)hi << 16);
  }
  reinterpret_cast<uint2*>(q + r * K)[v] = make_uint2(w[0], w[1]);
  if ((v & 3) == 0) sf[r * (K / 32) + (v >> 2)] = (uint8_t)e;
}

cudaError_t quant_mxfp8_launch(const void* x, long long ld_x, void* q, void* sf, long long rows, int K, cudaStream_t s) {
  if (rows == 0) return cudaSuccess;
  if ((K % 128) != 0 || (ld_x % 8) != 0) return cudaErrorInvalidValue;
  const long long total = rows * (K / 8);
  (void)launch_pdl(quant_mxfp8_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, s, static_cast<const __nv_bfloat16*>(x), ld_x,
                   static_cast<uint8_t*>(q), static_cast<uint8_t*>(sf), K, total);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ RMSNorm
// One CTA per row; each thread keeps up to MAXV 16-byte vectors of the row in registers (H <= 256*8*MAXV).
constexpr int kNormThreads = 256;
constexpr int kNormMaxV = 8;

__global__ void __launch_bounds__(kNormThreads)
rmsnorm_kernel(const __nv_bfloat16* __restrict__ x, long long ld_x, const __nv_bfloat16* __restrict__ w,
               const __nv_bfloat16* __restrict__ residual, long long ld_res, __nv_bfloat16* __restrict__ out,
               long long ld_out, int H, float eps, int gemma, uint32_t* signal_flag, uint32_t signal_value,
               unsigned int* done_counter) {
  pdl_sync();  // PDL: predecessor's writes visible; let the successor start its prologue
  const int row = blockIdx.x;
  const int nvec = H / 8;
  const uint4* xr = reinterpret_cast<const uint4*>(x + (size_t)row * ld_x);
  uint4 regs[kNormMaxV];
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < kNormMaxV; ++i) {
    const int v = threadIdx.x + i * kNormThreads;
    if (v < nvec) {
      regs[i] = xr[v];
      float f[8];
      unpack8(regs[i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) ss += f[j] * f[j];
    }
  }
  __shared__ float red[kNormThreads / 32];
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int i = 0; i < kNormThreads / 32; ++i) tot += red[i];
  const float inv = rsqrtf(tot / (float)H + eps);
  const uint4* wr = reinterpret_cast<const uint4*>(w);
  uint4* orow = reinterpret_cast<uint4*>(out + (size_t)row * ld_out);
#pragma unroll
  for (int i = 0; i < kNormMaxV; ++i) {
    const int v = threadIdx.x + i * kNormThreads;
    if (v < nvec) {
      float f[8], g[8];
      unpack8(regs[i], f);
      unpack8(wr[v], g);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float gg = gemma ? (1.0f + g[j]) : g[j];
        // match the unfused graph: the normalised value is rounded to bf16 before the optional residual add
        f[j] = f[j] * inv * gg;
      }
      if (residual != nullptr) {
        float r[8];
        unpack8(reinterpret_cast<const uint4*>(residual + (size_t)row * ld_res)[v], r);
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = __bfloat162float(__float2bfloat16_rn(f[j])) + r[j];
      }
      orow[v] = pack8(f);
    }
  }
  if (signal_flag != nullptr) {
    // fused stage boundary (Gemma-2: a stage's last kernel is the post-feed-forward norm + residual): `out` is the next stage's
    // inbox in peer memory; every CTA fences its row, the last one raises the consumer's flag with system scope
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned int done = atomicAdd(done_counter, 1u) + 1u;
      if (done == gridDim.x) {
        *done_counter = 0u;
        __threadfence_system();
        if (signal_value == 0u) atomicAdd_system(signal_flag, 1u);
        else st_release_sys(signal_flag, signal_value);
      }
    }
  }
}

cudaError_t rmsnorm_launch(const void* x, long long ld_x, const void* w, const void* residual, long long ld_res,
                           void* out, long long ld_out, int rows, int H, float eps, bool gemma, cudaStream_t s,
                           uint32_t* signal_flag, uint32_t signal_value, unsigned int* done_counter) {
  if (H % 8 != 0 || H > kNormThreads * 8 * kNormMaxV || (ld_x % 8) || (ld_out % 8)) return cudaErrorInvalidValue;
  if (rows == 0) return cudaSuccess;
  (void)launch_pdl(rmsnorm_kernel, dim3(rows), dim3(kNormThreads), 0, s, static_cast<const __nv_bfloat16*>(x), ld_x,
                                                 static_cast<const __nv_bfloat16*>(w),
                                                 static_cast<const __nv_bfloat16*>(residual), ld_res,
                                                 static_cast<__nv_bfloat16*>(out), ld_out, H, eps, gemma ? 1 : 0, signal_flag, signal_value,
                                                 done_counter);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ RoPE
// In place on x[T, heads, D] (token stride ld_t, head stride ld_h) over dims [rot_off, rot_off + rot_dim).
// One thread per rotated pair; angle = position * inv_freq[i], computed with full-range sincosf.
__global__ void rope_kernel(__nv_bfloat16* __restrict__ x, long long ld_t, long long ld_h, int heads,
                            const int* __restrict__ positions, const float* __restrict__ inv_freq, int rot_off,
                            int rot_dim, int interleaved, float mscale, int T) {
  pdl_sync();  // PDL: predecessor's writes visible; let the successor start its prologue
  const int half = rot_dim / 2;
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long total = (long long)T * heads * half;
  if (idx >= total) return;
  const int i = idx % half;
  const int h = (idx / half) % heads;
  const int t = idx / ((long long)half * heads);
  float sn, cs;
  sincosf((float)positions[t] * inv_freq[i], &sn, &cs);
  __nv_bfloat16* base = x + (size_t)t * ld_t + (size_t)h * ld_h + rot_off;
  const int i1 = interleaved ? 2 * i : i;
  const int i2 = interleaved ? 2 * i + 1 : i + half;
  const float a = __bfloat162float(base[i1]) * mscale, b = __bfloat162float(base[i2]) * mscale;
  base[i1] = __float2bfloat16_rn(a * cs - b * sn);
  base[i2] = __float2bfloat16_rn(interleaved ? (a * sn + b * cs) : (b * cs + a * sn));
}

cudaError_t rope_launch(void* x, long long ld_t, long long ld_h, int heads, const int* positions, const float* inv_freq,
                        int rot_off, int rot_dim, bool interleaved, float mscale, int T, cudaStream_t s) {
  const long long total = (long long)T * heads * (rot_dim / 2);
  if (total == 0) return cudaSuccess;
  (void)launch_pdl(rope_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, s, static_cast<__nv_bfloat16*>(x), ld_t, ld_h, heads, positions,
                                                              inv_freq, rot_off, rot_dim, interleaved ? 1 : 0, mscale, T);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ Embedding
// out[t, :] = table[ids[t], :] * scale; quantised tables are dequantised on the fly:
// w = scales * q + biases, group size g, codes packed LSB-first in uint32 words (MLX affine layout).
__global__ void embed_kernel(const long long* __restrict__ ids, const __nv_bfloat16* __restrict__ table,
                             __nv_bfloat16* __restrict__ out, int H, float scale, int T) {
  pdl_sync();  // PDL: predecessor's writes visible; let the successor start its prologue
  const int nvec = H / 8;
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= (long long)T * nvec) return;
  const int t = idx / nvec, v = idx % nvec;
  uint4 r = reinterpret_cast<const uint4*>(table + (size_t)ids[t] * H)[v];
  if (scale != 1.0f) {
    float f[8];
    unpack8(r, f);
    const float sc = __bfloat162float(__float2bfloat16_rn(scale));
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] *= sc;
    r = pack8(f);
  }
  reinterpret_cast<uint4*>(out + (size_t)t * H)[v] = r;
}

template <int BITS>
__global__ void embed_quant_kernel(const long long* __restrict__ ids, const uint32_t* __restrict__ wq,
                                   const __nv_bfloat16* __restrict__ scales, const __nv_bfloat16* __restrict__ biases,
                                   __nv_bfloat16* __restrict__ out, int H, int group, float scale, int T) {
  pdl_sync();  // PDL: predecessor's writes visible; let the successor start its prologue
  constexpr int PER = 32 / BITS;  // codes per word
  const int words = H / PER;
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= (long long)T * words) return;
  const int t = idx / words, wi = idx % words;
  const long long row = ids[t];
  const uint32_t word = wq[(size_t)row * words + wi];
  const int col0 = wi * PER;
  const int ng = H / group;
  const float s = __bfloat162float(scales[(size_t)row * ng + col0 / group]);
  const float b = __bfloat162float(biases[(size_t)row * ng + col0 / group]);
  const float sc = (scale != 1.0f) ? __bfloat162float(__float2bfloat16_rn(scale)) : 1.0f;
  __nv_bfloat16* o = out + (size_t)t * H + col0;
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const float q = (float)((word >> (j * BITS)) & ((1u << BITS) - 1u));
    float val = s * q + b;
    if (scale != 1.0f) val = __bfloat162float(__float2bfloat16_rn(val)) * sc;
    o[j] = __float2bfloat16_rn(val);
  }
}

cudaError_t embed_launch(const long long* ids, const void* table, const void* scales, const void* biases, int bits, int group,
                         void* out, int H, float scale, int T, cudaStream_t s) {
  if (T == 0) return cudaSuccess;
  if (bits == 0) {
    if (H % 8) return cudaErrorInvalidValue;
    const long long n = (long long)T * (H / 8);
    (void)launch_pdl(embed_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, s, ids, static_cast<const __nv_bfloat16*>(table),
                                                              static_cast<__nv_bfloat16*>(out), H, scale, T);
  } else {
    const int per = 32 / bits;
    const long long n = (long long)T * (H / per);
    auto sc = static_cast<const __nv_bfloat16*>(scales);
    auto bi = static_cast<const __nv_bfloat16*>(biases);
    auto wq = static_cast<const uint32_t*>(table);
    auto o = static_cast<__nv_bfloat16*>(out);
    const unsigned grid = (unsigned)((n + 255) / 256);
    if (bits == 4) (void)launch_pdl(embed_quant_kernel<4>, dim3(grid), dim3(256), 0, s, ids, wq, sc, bi, o, H, group, scale, T);
    else if (bits == 8) (void)launch_pdl(embed_quant_kernel<8>, dim3(grid), dim3(256), 0, s, ids, wq, sc, bi, o, H, group, scale, T);
    else if (bits == 2) (void)launch_pdl(embed_quant_kernel<2>, dim3(grid), dim3(256), 0, s, ids, wq, sc, bi, o, H, group, scale, T);
    else return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ KV append
// pools are [pages, kv_heads, page_size, D]; slot = page * page_size + offset.
__global__ void kv_write_kernel(const __nv_bfloat16* __restrict__ k, long long k_ld_t, long long k_ld_h,
                                const __nv_bfloat16* __restrict__ v, long long v_ld_t, long long v_ld_h,
                                __nv_bfloat16* __restrict__ kpool, __nv_bfloat16* __restrict__ vpool,
                                const int* __restrict__ slots, int heads, int dk, int dv, int page, int T) {
  pdl_sync();  // PDL: predecessor's writes visible; let the successor start its prologue
  const int vk = dk / 8, vv = dv / 8, per = vk + vv;
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= (long long)T * heads * per) return;
  const int c = idx % per;
  const int h = (idx / per) % heads;
  const int t = idx / ((long long)per * heads);
  const int slot = slots[t];
  const size_t pg = slot / page, off = slot % page;
  if (c < vk) {
    const uint4 r = reinterpret_cast<const uint4*>(k + (size_t)t * k_ld_t + (size_t)h * k_ld_h)[c];
    reinterpret_cast<uint4*>(kpool + ((pg * heads + h) * page + off) * dk)[c] = r;
  } else {
    const uint4 r = reinterpret_cast<const uint4*>(v + (size_t)t * v_ld_t + (size_t)h * v_ld_h)[c - vk];
    reinterpret_cast<uint4*>(vpool + ((pg * heads + h) * page + off) * dv)[c - vk] = r;
  }
}

cudaError_t kv_write_launch(const void* k, long long k_ld_t, long long k_ld_h, const void* v, long long v_ld_t,
                            long long v_ld_h, void* kpool, void* vpool, const int* slots, int heads, int dk, int dv,
                            int page, int T, cudaStream_t s) {
  if (T == 0) return cudaSuccess;
  if ((dk % 8) || (dv % 8) || (k_ld_t % 8) || (k_ld_h % 8) || (v_ld_t % 8) || (v_ld_h % 8)) return cudaErrorInvalidValue;
  const long long n = (long long)T * heads * (dk / 8 + dv / 8);
  (void)launch_pdl(kv_write_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, s, 
      static_cast<const __nv_bfloat16*>(k), k_ld_t, k_ld_h, static_cast<const __nv_bfloat16*>(v), v_ld_t, v_ld_h,
      static_cast<__nv_bfloat16*>(kpool), static_cast<__nv_bfloat16*>(vpool), slots, heads, dk, dv, page, T);
  return cudaGetLastError();
}

// MLA append (reference layout, deepseek_v2.py:120-125): kv[T, heads, nope + vd] from kv_b_proj, k_pe[T, rd]
// shared by all heads -> K row = [k_nope | k_pe], V row = v.
__global__ void kv_write_mla_kernel(const __nv_bfloat16* __restrict__ kv, long long kv_ld_t,
                                    const __nv_bfloat16* __restrict__ kpe, long long pe_ld_t,
                                    __nv_bfloat16* __restrict__ kpool, __nv_bfloat16* __restrict__ vpool,
                                    const int* __restrict__ slots, int heads, int nope, int rd, int vd, int page, int T) {
  pdl_sync();  // PDL: predecessor's writes visible; let the successor start its prologue
  const int vn = nope / 8, vr = rd / 8, vvv = vd / 8, per = vn + vr + vvv;
  const int dk = nope + rd;
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= (long long)T * heads * per) return;
  const int c = idx % per;
  const int h = (idx / per) % heads;
  const int t = idx / ((long long)per * heads);
  const int slot = slots[t];
  const size_t pg = slot / page, off = slot % page;
  const __nv_bfloat16* src = kv + (size_t)t * kv_ld_t + (size_t)h * (nope + vd);
  __nv_bfloat16* krow = kpool + ((pg * heads + h) * page + off) * dk;
  __nv_bfloat16* vrow = vpool + ((pg * heads + h) * page + off) * vd;
  if (c < vn) reinterpret_cast<uint4*>(krow)[c] = reinterpret_cast<const uint4*>(src)[c];
  else if (c < vn + vr) reinterpret_cast<uint4*>(krow + nope)[c - vn] = reinterpret_cast<const uint4*>(kpe + (size_t)t * pe_ld_t)[c - vn];
  else reinterpret_cast<uint4*>(vrow)[c - vn - vr] = reinterpret_cast<const uint4*>(src + nope)[c - vn - vr];
}

cudaError_t kv_write_mla_launch(const void* kv, long long kv_ld_t, const void* kpe, long long pe_ld_t, void* kpool,
                                void* vpool, const int* slots, int heads, int nope, int rd, int vd, int page, int T,
                                cudaStream_t s) {
  if (T == 0) return cudaSuccess;
  if ((nope % 8) || (rd % 8) || (vd % 8) || (kv_ld_t % 8) || (pe_ld_t % 8)) return cudaErrorInvalidValue;
  const long long n = (long long)T * heads * ((nope + rd + vd) / 8);
  (void)launch_pdl(kv_write_mla_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, s, 
      static_cast<const __nv_bfloat16*>(kv), kv_ld_t, static_cast<const __nv_bfloat16*>(kpe), pe_ld_t,
      static_cast<__nv_bfloat16*>(kpool), static_cast<__nv_bfloat16*>(vpool), slots, heads, nope, rd, vd, page, T);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ fused MLA prologue
// DeepSeek-V2 attention prologue in ONE launch (replaces rope(q) + rope(k_pe) + kv_write_mla):
//   * rotates the rope slice of every q head in place (interleaved pairs, YaRN inv_freq, mscale),
//   * assembles K = [k_nope | rope(k_pe)] and V straight into the paged cache.
// One thread per 32-bit word (= one interleaved pair) of the rope parts, one per 16 B vector of the copies.
__global__ void mla_rope_kv_kernel(__nv_bfloat16* __restrict__ q, long long q_ld_t, long long q_ld_h,
                                   const __nv_bfloat16* __restrict__ kpe, long long pe_ld_t,
                                   const __nv_bfloat16* __restrict__ kv, long long kv_ld_t,
                                   __nv_bfloat16* __restrict__ kpool, __nv_bfloat16* __restrict__ vpool,
                                   const int* __restrict__ slots, const int* __restrict__ positions,
                                   const float* __restrict__ inv_freq, float mscale, int heads, int nope, int rd, int vd,
                                   int page, int T) {
  pdl_sync();  // PDL: predecessor's writes visible; let the successor start its prologue
  const int half = rd / 2, vn = nope / 8, vv = vd / 8;
  const int per = half + vn + half + vv;  // work items per (token, head)
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= (long long)T * heads * per) return;
  const int c = idx % per;
  const int h = (idx / per) % heads;
  const int t = idx / ((long long)per * heads);
  const int dk = nope + rd;
  const int slot = slots[t];
  const size_t pg = slot / page, off = slot % page;
  __nv_bfloat16* krow = kpool + ((pg * heads + h) * page + off) * dk;
  const __nv_bfloat16* src = kv + (size_t)t * kv_ld_t + (size_t)h * (nope + vd);
  if (c < half) {  // q rope pair
    float sn, cs;
    sincosf((float)positions[t] * inv_freq[c], &sn, &cs);
    uint32_t* w = reinterpret_cast<uint32_t*>(q + (size_t)t * q_ld_t + (size_t)h * q_ld_h + nope) + c;
    const uint32_t u = *w;
    const float a = bf16_lo(u) * mscale, b = bf16_hi(u) * mscale;
    *w = pack_bf16(a * cs - b * sn, a * sn + b * cs);
  } else if (c < half + vn) {  // k_nope copy
    const int v = c - half;
    reinterpret_cast<uint4*>(krow)[v] = reinterpret_cast<const uint4*>(src)[v];
  } else if (c < half + vn + half) {  // k_pe rope pair -> cache (shared by all heads, rotated per head write)
    const int i = c - half - vn;
    float sn, cs;
    sincosf((float)positions[t] * inv_freq[i], &sn, &cs);
    const uint32_t u = reinterpret_cast<const uint32_t*>(kpe + (size_t)t * pe_ld_t)[i];
    const float a = bf16_lo(u) * mscale, b = bf16_hi(u) * mscale;
    reinterpret_cast<uint32_t*>(krow + nope)[i] = pack_bf16(a * cs - b * sn, a * sn + b * cs);
  } else {  // v copy
    const int v = c - half - vn - half;
    __nv_bfloat16* vrow = vpool + ((pg * heads + h) * page + off) * vd;
    reinterpret_cast<uint4*>(vrow)[v] = reinterpret_cast<const uint4*>(src + nope)[v];
  }
}

cudaError_t mla_rope_kv_launch(void* q, long long q_ld_t, long long q_ld_h, const void* kpe, long long pe_ld_t, const void* kv,
                               long long kv_ld_t, void* kpool, void* vpool, const int* slots, const int* positions,
                               const float* inv_freq, float mscale, int heads, int nope, int rd, int vd, int page, int T,
                               cudaStream_t s) {
  if (T == 0) return cudaSuccess;
  if ((nope % 8) || (rd % 8) || (vd % 8) || (kv_ld_t % 8) || (pe_ld_t % 2) || (q_ld_t % 2) || (q_ld_h % 2)) return cudaErrorInvalidValue;
  const long long n = (long long)T * heads * (rd + nope / 8 + vd / 8);
  (void)launch_pdl(mla_rope_kv_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, s, 
      static_cast<__nv_bfloat16*>(q), q_ld_t, q_ld_h, static_cast<const __nv_bfloat16*>(kpe), pe_ld_t,
      static_cast<const __nv_bfloat16*>(kv), kv_ld_t, static_cast<__nv_bfloat16*>(kpool), static_cast<__nv_bfloat16*>(vpool),
      slots, positions, inv_freq, mscale, heads, nope, rd, vd, page, T);
  return cudaGetLastError();
}

}  // namespace b200
