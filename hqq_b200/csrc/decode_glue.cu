// Decode-harness glue kernels (SURVEY.md 8 f-2: the caller of HQQLinear.forward, NOT the hot path): the few tiny ops
// between the fused linears of a Llama-style block at batch 1, written so a decode step is 8 launches per block
// instead of ~25 framework kernels.  fp16/bf16, one token.  All kernels are PDL-aware (griddepcontrol) so their
// launch latency overlaps the tail of the previous kernel inside a CUDA graph.
#ifndef HQQ_EMU
#include <cooperative_groups.h>
#endif

#include "device.cuh"

namespace hqq {

__device__ __forceinline__ float block_sum(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if ((threadIdx.x & 31) == 0) red[w] = v;
  __syncthreads();
  float s = 0.f;
  for (int i = 0; i < nw; ++i) s += red[i];
  __syncthreads();
  return s;
}

// h += delta (optional); y = rmsnorm(h) * w         (one CTA per row of [rows, H]; H <= 8 * blockDim)
template <typename T>
__global__ void __launch_bounds__(1024) add_rmsnorm_kernel(T* __restrict__ h, const T* __restrict__ delta, const T* __restrict__ w,
                                                           T* __restrict__ y, int H, float eps) {
  __shared__ float red[32];
  {
    const long long row = (long long)blockIdx.x * H;  // batched decode: one sequence per CTA
    h += row;
    y += row;
    if (delta) delta += row;
  }
  pdl_launch_dependents();
  pdl_wait();
  float v[8];
  int n = 0;
  float ss = 0.f;
  for (int i = threadIdx.x; i < H; i += blockDim.x, ++n) {
    float x = to_f32<T>(h[i]);
    if (delta) {
      x = to_f32<T>(from_f32<T>(x + to_f32<T>(delta[i])));  // residual stream stays in T, like h = h + o in the framework
      h[i] = from_f32<T>(x);
    }
    v[n] = x;
    ss += x * x;
  }
  const float tot = block_sum(ss, red);
  const float inv = rsqrtf(tot / (float)H + eps);
  n = 0;
  for (int i = threadIdx.x; i < H; i += blockDim.x, ++n) y[i] = from_f32<T>(to_f32<T>(from_f32<T>(v[n] * inv)) * to_f32<T>(w[i]));
}

// Same as add_rmsnorm_kernel, but the residual delta is the sum of `tp` tagged partial vectors that the peers' row-parallel
// kernels scattered into this rank's exchange buffer (see SKArgs in linear_small.cu).  As the last consumer of a token it
// bumps the step counter the exchange tags are derived from.
template <typename T>
__global__ void __launch_bounds__(1024) add_rmsnorm_tp_kernel(T* __restrict__ h, const uint32_t* red_data, int* step_ctr, int x_index, int x_per_step,
                                                              int tp, const T* __restrict__ w, T* __restrict__ y, int H, float eps) {
  __shared__ float red[32];
  pdl_launch_dependents();
  pdl_wait();
  const int step = *reinterpret_cast<volatile int*>(step_ctr);
  const uint32_t ex = (uint32_t)step * (uint32_t)x_per_step + (uint32_t)x_index;
  const uint32_t tag = ex & 0xFFFFu;
  const uint32_t* part = red_data + (size_t)(ex & 1u) * tp * H;
  float v[8];
  int n = 0;
  float ss = 0.f;
  for (int i = threadIdx.x; i < H; i += blockDim.x, ++n) {
    float d = 0.f;
    for (int r = 0; r < tp; ++r) {
      uint32_t wv;
      do { wv = ld_relaxed_sys_u32(part + (size_t)r * H + i); } while ((wv >> 16) != tag);
      const unsigned short hb = (unsigned short)(wv & 0xFFFFu);
      d += to_f32<T>(*reinterpret_cast<const T*>(&hb));
    }
    float x = to_f32<T>(from_f32<T>(to_f32<T>(h[i]) + to_f32<T>(from_f32<T>(d))));
    h[i] = from_f32<T>(x);
    v[n] = x;
    ss += x * x;
  }
  const float tot = block_sum(ss, red);
  const float inv = rsqrtf(tot / (float)H + eps);
  n = 0;
  for (int i = threadIdx.x; i < H; i += blockDim.x, ++n) y[i] = from_f32<T>(to_f32<T>(from_f32<T>(v[n] * inv)) * to_f32<T>(w[i]));
  if (threadIdx.x == 0) *step_ctr = step + 1;
}

// y = silu(g) * u
template <typename T>
__global__ void __launch_bounds__(256) silu_mul_kernel(const T* __restrict__ g, const T* __restrict__ u, T* __restrict__ y, int n) {
  pdl_launch_dependents();
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const float a = to_f32<T>(g[i]);
    const float s = to_f32<T>(from_f32<T>(a / (1.0f + __expf(-a))));
    y[i] = from_f32<T>(s * to_f32<T>(u[i]));
  }
}

// RoPE (rotate-half, cos/sin tables [L, hd]) + KV-cache append + single-token GQA attention over cache[0..pos].
// grid = n_q_heads, block = 256 threads (8 warps).  caches are [n_kv_heads, L, hd], hd = 128.
// The step streams ~5 GB of weights between two visits of a layer's cache, so the rows are cold in DRAM and the kernel is
// bound by load latency, not bandwidth: (1) rows 0..pos-1 were written by earlier steps, so they are prefetched into L2
// BEFORE griddepcontrol.wait, under the tail of the q/k/v kernel (pos itself is only written by the non-PDL kernel that ends
// a step, a full barrier); (2) both position loops keep 8-16 independent loads in flight per thread.
constexpr int kAttnThreads = 256;
template <typename T, bool BATCH>
__global__ void __launch_bounds__(kAttnThreads) rope_attn_decode_kernel(const T* __restrict__ q_in, const T* __restrict__ k_in, const T* __restrict__ v_in,
                                                                        const T* __restrict__ cos_t, const T* __restrict__ sin_t,
                                                                        T* __restrict__ k_cache, T* __restrict__ v_cache, const long long* __restrict__ pos_p,
                                                                        T* __restrict__ out, int n_q, int n_kv, int L, int hd, float scale) {
  extern __shared__ float sm[];  // q[hd] | knew[hd] | p[L]  (later reused as [8][hd] partial outputs) | red[32]
  constexpr int NW = kAttnThreads / 32;
  float* qs = sm;
  float* ks = sm + hd;
  float* ps = sm + 2 * hd;
  float* red = sm + max(2 * hd + L, NW * hd);
  const int h = blockIdx.x, kvh = h / (n_q / n_kv), d = threadIdx.x;
  if constexpr (BATCH) {  // sequence blockIdx.y of the lock-step batch (all at the same position); the one-sequence
    const long long b = blockIdx.y;  // instantiation is the kernel as it was (its position loops lost 1 us per layer at 200
    q_in += b * n_q * hd; out += b * n_q * hd;  // cached positions when the offsets were applied unconditionally)
    k_in += b * n_kv * hd; v_in += b * n_kv * hd;
    k_cache += b * n_kv * L * hd; v_cache += b * n_kv * L * hd;
  }
  const int pos = (int)pos_p[0];
  pdl_launch_dependents();
  {
    // one 128-byte line per prefetch; pos rows of hd * sizeof(T) bytes each in both caches
    const char* kb = reinterpret_cast<const char*>(k_cache + (long long)kvh * L * hd);
    const char* vb = reinterpret_cast<const char*>(v_cache + (long long)kvh * L * hd);
    const int lines = (int)(((long long)pos * hd * (int)sizeof(T)) >> 7);
    for (int i = d; i < lines; i += kAttnThreads) {
      prefetch_l2(kb + ((long long)i << 7));
      prefetch_l2(vb + ((long long)i << 7));
    }
  }
  pdl_wait();
  const int half = hd / 2;
  // rope: x*cos + rotate_half(x)*sin, computed in T like the framework ops
  if (d < hd) {
    const float c = to_f32<T>(cos_t[(long long)pos * hd + d]), s = to_f32<T>(sin_t[(long long)pos * hd + d]);
    const float qx = to_f32<T>(q_in[h * hd + d]);
    const float qr = (d < half) ? -to_f32<T>(q_in[h * hd + d + half]) : to_f32<T>(q_in[h * hd + d - half]);
    qs[d] = to_f32<T>(from_f32<T>(to_f32<T>(from_f32<T>(qx * c)) + to_f32<T>(from_f32<T>(qr * s))));
    const float kx = to_f32<T>(k_in[kvh * hd + d]);
    const float kr = (d < half) ? -to_f32<T>(k_in[kvh * hd + d + half]) : to_f32<T>(k_in[kvh * hd + d - half]);
    const T kn = from_f32<T>(to_f32<T>(from_f32<T>(kx * c)) + to_f32<T>(from_f32<T>(kr * s)));
    ks[d] = to_f32<T>(kn);
    if (h % (n_q / n_kv) == 0) {  // one head of the group owns the cache write
      k_cache[((long long)kvh * L + pos) * hd + d] = kn;
      v_cache[((long long)kvh * L + pos) * hd + d] = v_in[kvh * hd + d];
    }
  }
  __syncthreads();
  // scores: thread t handles positions t, t+blockDim, ... (a whole 256-byte row each, all 16 loads in flight at once);
  // the current position uses the freshly rotated k
  float mx = -INFINITY;
  for (int t = d; t <= pos; t += kAttnThreads) {
    float acc = 0.f;
    if (t == pos) {
      for (int i = 0; i < hd; ++i) acc += qs[i] * ks[i];
    } else {
      const T* kr = k_cache + ((long long)kvh * L + t) * hd;
      Vec<T, 8> kv[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) kv[i] = *reinterpret_cast<const Vec<T, 8>*>(kr + i * 8);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
#pragma unroll
        for (int j = 0; j < 8; ++j) acc += qs[i * 8 + j] * to_f32<T>(kv[i].v[j]);
      }
    }
    acc *= scale;
    ps[t] = acc;
    mx = fmaxf(mx, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((d & 31) == 0) red[d >> 5] = mx;
  __syncthreads();
  mx = red[0];
#pragma unroll
  for (int i = 1; i < NW; ++i) mx = fmaxf(mx, red[i]);
  __syncthreads();
  float sum = 0.f;
  for (int t = d; t <= pos; t += kAttnThreads) {
    const float e = __expf(ps[t] - mx);
    ps[t] = e;
    sum += e;
  }
  const float tot = block_sum(sum, red);
  const float ps_last = ps[pos];
  // output: warp w takes positions w, w+8, ... and each lane four consecutive dimensions (one 8-byte load per position);
  // eight positions per warp are loaded before any is consumed.  The eight partial outputs meet in shared memory.
  {
    const int w = d >> 5, l = d & 31;
    float o4[4] = {0.f, 0.f, 0.f, 0.f};
    const T* vbase = v_cache + (long long)kvh * L * hd + 4 * l;
    int t = w;
    for (; t + 7 * NW < pos; t += 8 * NW) {
      Vec<T, 4> vv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) vv[u] = *reinterpret_cast<const Vec<T, 4>*>(vbase + (long long)(t + u * NW) * hd);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float pt = ps[t + u * NW];
#pragma unroll
        for (int j = 0; j < 4; ++j) o4[j] += pt * to_f32<T>(vv[u].v[j]);
      }
    }
    for (; t < pos; t += NW) {
      const Vec<T, 4> vv = *reinterpret_cast<const Vec<T, 4>*>(vbase + (long long)t * hd);
      const float pt = ps[t];
#pragma unroll
      for (int j = 0; j < 4; ++j) o4[j] += pt * to_f32<T>(vv.v[j]);
    }
    __syncthreads();  // q, k and the probabilities are dead now: reuse the front of the buffer for the cross-warp reduction
    float* part = sm;  // [NW][hd] floats (the launcher sizes the buffer for max(2*hd + L, NW*hd) + 32)
#pragma unroll
    for (int j = 0; j < 4; ++j) part[w * hd + 4 * l + j] = o4[j];
    __syncthreads();
    if (d < hd) {
      float o = 0.f;
#pragma unroll
      for (int i = 0; i < NW; ++i) o += part[i * hd + d];
      o += ps_last * to_f32<T>(v_in[kvh * hd + d]);
      out[h * hd + d] = from_f32<T>(o / tot);
    }
  }
}

#ifndef HQQ_EMU
// argmax over n logits -> int64 index (first index on ties).  One thread-block cluster of 8 CTAs: each scans an
// interleaved eighth of the row, the eight candidates meet in CTA 0's shared memory over DSMEM (no workspace, one launch).
// key_offset >= 0 (vocabulary-sharded lm_head under tensor parallelism): out[0] = (ordered(max) >> 1) << 32 | (0xFFFFFFFF -
// (key_offset + index)) -- a signed 64-bit key whose MAX over the ranks is the global argmax with the first index on ties
// (ordered() is the usual monotone float -> uint32 map; fp16/bf16 values leave the low mantissa bits of the float zero, so the
// shift that keeps the sign bit clear loses nothing).
constexpr int kArgmaxCtas = 8;
//
// tp > 0 (hqq_b200_glue_argmax_tp): the key exchange happens in this launch.  Bits 32..43 of a key are the same for every fp16 /
// bf16 value of one sign (they are below the 16-bit value's precision), so they can carry a 12-bit tag of the token step without
// disturbing the order, as long as every rank uses the same tag in the same step.  CTA 0 stores its tagged key into slot
// [parity][rank] of every peer's key area (one aligned 8-byte store each: value, index and tag arrive together), polls its own
// slots [parity][0..tp) until all carry this step's tag, and writes the winner's index to out[0].  Two parities suffice: a rank
// cannot finish step s+1 before every peer has sent its step s+1 key, which a peer does only after it has read step s.
struct KeyPeers { unsigned long long* p[8]; };
template <typename T>
__global__ void __cluster_dims__(kArgmaxCtas, 1, 1) __launch_bounds__(1024) argmax_kernel(const T* __restrict__ x, int n, long long* __restrict__ out,
                                                                                            long long key_offset, KeyPeers peers, int tp, int tp_rank,
                                                                                            const int* __restrict__ step_ctr) {
  namespace cg = cooperative_groups;
  __shared__ float bv[32];
  __shared__ int bi[32];
  __shared__ float cv[kArgmaxCtas];
  __shared__ int ci[kArgmaxCtas];
  __shared__ unsigned long long xkey;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  pdl_launch_dependents();
  pdl_wait();
  float best = -INFINITY;
  int idx = 0;
  for (int i = (rank * 1024 + (int)threadIdx.x) * 8; i < n; i += kArgmaxCtas * 1024 * 8) {
    if (i + 8 <= n) {
      const Vec<T, 8> v = *reinterpret_cast<const Vec<T, 8>*>(x + i);
#pragma unroll
      for (int j = 0; j < 8; ++j) { const float f = to_f32<T>(v.v[j]); if (f > best) { best = f; idx = i + j; } }
    } else {
      for (int j = i; j < n; ++j) { const float f = to_f32<T>(x[j]); if (f > best) { best = f; idx = j; } }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (ob > best || (ob == best && oi < idx)) { best = ob; idx = oi; }
  }
  if ((threadIdx.x & 31) == 0) { bv[threadIdx.x >> 5] = best; bi[threadIdx.x >> 5] = idx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i)
      if (bv[i] > best || (bv[i] == best && bi[i] < idx)) { best = bv[i]; idx = bi[i]; }
    cluster.map_shared_rank(cv, 0)[rank] = best;
    cluster.map_shared_rank(ci, 0)[rank] = idx;
  }
  cluster.sync();
  if (rank == 0 && threadIdx.x == 0) {
    best = cv[0]; idx = ci[0];
    for (int i = 1; i < kArgmaxCtas; ++i)
      if (cv[i] > best || (cv[i] == best && ci[i] < idx)) { best = cv[i]; idx = ci[i]; }
    if (key_offset < 0) {
      out[0] = idx;
    } else {
      const uint32_t u = __float_as_uint(best);
      const uint32_t ord = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
      const unsigned long long key = ((unsigned long long)(ord >> 1) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)(key_offset + idx));
      if (tp <= 0) out[0] = (long long)key;
      else xkey = key;
    }
  }
  if (tp > 0 && rank == 0) {  // uniform per CTA
    __syncthreads();
    if ((int)threadIdx.x < 32) {
      const int seq = *reinterpret_cast<const volatile int*>(step_ctr);  // already bumped by this token's final norm: >= 1
      const unsigned long long tag = (unsigned long long)((unsigned)seq & 0xFFFu) << 32, tmask = 0xFFFull << 32;
      const int par = seq & 1, t = (int)threadIdx.x;
      long long got = 0;  // keys are non-negative
      if (t < tp) {
        const unsigned long long mine = (xkey & ~tmask) | tag;
        asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(peers.p[t] + par * tp + tp_rank), "l"(mine) : "memory");
        const unsigned long long* slot = peers.p[tp_rank] + par * tp + t;
        unsigned long long v;
        unsigned spins = 0;  // a peer that never arrives (it died) ends in a launch failure, not in a GPU that spins for ever
        do {
          asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(slot) : "memory");
          if (++spins == (1u << 27)) __trap();
        } while ((v & tmask) != tag);
        got = (long long)v;
      }
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) { const long long ov = __shfl_xor_sync(0xffffffffu, got, o); got = ov > got ? ov : got; }
      if (t == 0) out[0] = (long long)(0xFFFFFFFFu - (uint32_t)((unsigned long long)got & 0xFFFFFFFFull));
    }
  }
}

#endif  // !HQQ_EMU

}  // namespace hqq

using namespace hqq;

extern "C" int hqq_b200_glue_add_rmsnorm_rows(void* h, const void* delta, const void* weight, void* y, int rows, int H, float eps, int dtype,
                                              void* stream) {
  HQQ_REQUIRE(h && weight && y && H > 0 && H <= 8 * 1024 && rows > 0 && rows <= 65535, HQQ_E_INVALID,
              "hqq_b200_glue_add_rmsnorm: bad arguments (rows=%d H=%d)", rows, H);
  cudaStream_t st = (cudaStream_t)stream;
  const int threads = H > 2048 ? 1024 : 256;  // at most 8 elements per thread (the kernels keep them in registers)
  if (dtype == HQQ_F16) return launch_pdl("add_rmsnorm", add_rmsnorm_kernel<__half>, dim3(rows), dim3(threads), 0, st, true, (__half*)h, (const __half*)delta, (const __half*)weight, (__half*)y, H, eps);
  if (dtype == HQQ_BF16) return launch_pdl("add_rmsnorm", add_rmsnorm_kernel<__nv_bfloat16>, dim3(rows), dim3(threads), 0, st, true, (__nv_bfloat16*)h, (const __nv_bfloat16*)delta, (const __nv_bfloat16*)weight, (__nv_bfloat16*)y, H, eps);
  set_error("hqq_b200_glue_add_rmsnorm: dtype must be f16/bf16");
  return HQQ_E_INVALID;
}

extern "C" int hqq_b200_glue_add_rmsnorm(void* h, const void* delta, const void* weight, void* y, int H, float eps, int dtype, void* stream) {
  return hqq_b200_glue_add_rmsnorm_rows(h, delta, weight, y, 1, H, eps, dtype, stream);
}

extern "C" int hqq_b200_glue_add_rmsnorm_tp(void* h, const void* red_data, int* step_ctr, int x_index, int x_per_step, int tp, const void* weight,
                                            void* y, int H, float eps, int dtype, void* stream) {
  HQQ_REQUIRE(h && red_data && step_ctr && weight && y && H > 0 && H <= 8 * 1024 && tp >= 1 && tp <= 8 && x_per_step > 0, HQQ_E_INVALID,
              "hqq_b200_glue_add_rmsnorm_tp: bad arguments (H=%d tp=%d)", H, tp);
  cudaStream_t st = (cudaStream_t)stream;
  const int threads = H > 2048 ? 1024 : 256;  // at most 8 elements per thread (the kernels keep them in registers)
  if (dtype == HQQ_F16) return launch_pdl("add_rmsnorm_tp", add_rmsnorm_tp_kernel<__half>, dim3(1), dim3(threads), 0, st, true, (__half*)h, (const uint32_t*)red_data, step_ctr, x_index, x_per_step, tp, (const __half*)weight, (__half*)y, H, eps);
  if (dtype == HQQ_BF16) return launch_pdl("add_rmsnorm_tp", add_rmsnorm_tp_kernel<__nv_bfloat16>, dim3(1), dim3(threads), 0, st, true, (__nv_bfloat16*)h, (const uint32_t*)red_data, step_ctr, x_index, x_per_step, tp, (const __nv_bfloat16*)weight, (__nv_bfloat16*)y, H, eps);
  set_error("hqq_b200_glue_add_rmsnorm_tp: dtype must be f16/bf16");
  return HQQ_E_INVALID;
}

extern "C" int hqq_b200_glue_silu_mul(const void* gate, const void* up, void* y, int n, int dtype, void* stream) {
  HQQ_REQUIRE(gate && up && y && n > 0, HQQ_E_INVALID, "hqq_b200_glue_silu_mul: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid((unsigned)cdiv(n, 256));
  if (dtype == HQQ_F16) return launch_pdl("silu_mul", silu_mul_kernel<__half>, grid, dim3(256), 0, st, true, (const __half*)gate, (const __half*)up, (__half*)y, n);
  if (dtype == HQQ_BF16) return launch_pdl("silu_mul", silu_mul_kernel<__nv_bfloat16>, grid, dim3(256), 0, st, true, (const __nv_bfloat16*)gate, (const __nv_bfloat16*)up, (__nv_bfloat16*)y, n);
  set_error("hqq_b200_glue_silu_mul: dtype must be f16/bf16");
  return HQQ_E_INVALID;
}

extern "C" int hqq_b200_glue_rope_attn_decode_batch(const void* q, const void* k, const void* v, const void* cos_table, const void* sin_table,
                                              void* k_cache, void* v_cache, const int64_t* pos, void* out, int n_q_heads, int n_kv_heads,
                                              int cache_len, int head_dim, int batch, int dtype, void* stream) {
  HQQ_REQUIRE(q && k && v && cos_table && sin_table && k_cache && v_cache && pos && out, HQQ_E_INVALID, "hqq_b200_glue_rope_attn_decode: null pointer");
  HQQ_REQUIRE(batch > 0 && batch <= 65535, HQQ_E_INVALID, "hqq_b200_glue_rope_attn_decode: batch %d", batch);
  HQQ_REQUIRE(head_dim == 128 && n_kv_heads > 0 && n_q_heads % n_kv_heads == 0 && cache_len > 0 && cache_len <= 8192, HQQ_E_UNSUPPORTED,
              "hqq_b200_glue_rope_attn_decode: needs head_dim 128, cache_len <= 8192");
  cudaStream_t st = (cudaStream_t)stream;
  const int body = 2 * head_dim + cache_len > 8 * head_dim ? 2 * head_dim + cache_len : 8 * head_dim;
  const size_t smem = (size_t)(body + 32) * sizeof(float);
  const float scale = 1.0f / sqrtf((float)head_dim);
  auto go = [&](auto kernel, auto tag) {
    using T = decltype(tag);
    return launch_pdl("rope_attn_decode", kernel, dim3(n_q_heads, batch), dim3(kAttnThreads), smem, st, true, (const T*)q, (const T*)k, (const T*)v,
                      (const T*)cos_table, (const T*)sin_table, (T*)k_cache, (T*)v_cache, (const long long*)pos, (T*)out, n_q_heads, n_kv_heads,
                      cache_len, head_dim, scale);
  };
  if (dtype == HQQ_F16) return batch > 1 ? go(rope_attn_decode_kernel<__half, true>, __half()) : go(rope_attn_decode_kernel<__half, false>, __half());
  if (dtype == HQQ_BF16)
    return batch > 1 ? go(rope_attn_decode_kernel<__nv_bfloat16, true>, __nv_bfloat16())
                     : go(rope_attn_decode_kernel<__nv_bfloat16, false>, __nv_bfloat16());
  set_error("hqq_b200_glue_rope_attn_decode: dtype must be f16/bf16");
  return HQQ_E_INVALID;
}

extern "C" int hqq_b200_glue_rope_attn_decode(const void* q, const void* k, const void* v, const void* cos_table, const void* sin_table,
                                              void* k_cache, void* v_cache, const int64_t* pos, void* out, int n_q_heads, int n_kv_heads,
                                              int cache_len, int head_dim, int dtype, void* stream) {
  return hqq_b200_glue_rope_attn_decode_batch(q, k, v, cos_table, sin_table, k_cache, v_cache, pos, out, n_q_heads, n_kv_heads, cache_len, head_dim, 1,
                                              dtype, stream);
}

#ifndef HQQ_EMU
extern "C" int hqq_b200_glue_argmax(const void* logits, int n, int64_t* out, int dtype, void* stream) {
  HQQ_REQUIRE(logits && out && n > 0, HQQ_E_INVALID, "hqq_b200_glue_argmax: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == HQQ_F16) return launch_pdl("argmax", argmax_kernel<__half>, dim3(kArgmaxCtas), dim3(1024), 0, st, true, (const __half*)logits, n, (long long*)out, -1LL, KeyPeers{}, 0, 0, (const int*)nullptr);
  if (dtype == HQQ_BF16) return launch_pdl("argmax", argmax_kernel<__nv_bfloat16>, dim3(kArgmaxCtas), dim3(1024), 0, st, true, (const __nv_bfloat16*)logits, n, (long long*)out, -1LL, KeyPeers{}, 0, 0, (const int*)nullptr);
  set_error("hqq_b200_glue_argmax: dtype must be f16/bf16");
  return HQQ_E_INVALID;
}

extern "C" int hqq_b200_glue_argmax_key(const void* logits, int n, int64_t index_offset, int64_t* out_key, int dtype, void* stream) {
  HQQ_REQUIRE(logits && out_key && n > 0 && index_offset >= 0 && index_offset + n <= 0xFFFFFFFFll, HQQ_E_INVALID, "hqq_b200_glue_argmax_key: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == HQQ_F16) return launch_pdl("argmax_key", argmax_kernel<__half>, dim3(kArgmaxCtas), dim3(1024), 0, st, true, (const __half*)logits, n, (long long*)out_key, (long long)index_offset, KeyPeers{}, 0, 0, (const int*)nullptr);
  if (dtype == HQQ_BF16) return launch_pdl("argmax_key", argmax_kernel<__nv_bfloat16>, dim3(kArgmaxCtas), dim3(1024), 0, st, true, (const __nv_bfloat16*)logits, n, (long long*)out_key, (long long)index_offset, KeyPeers{}, 0, 0, (const int*)nullptr);
  set_error("hqq_b200_glue_argmax_key: dtype must be f16/bf16");
  return HQQ_E_INVALID;
}

extern "C" int hqq_b200_glue_argmax_tp(const void* logits, int n, int64_t index_offset, void* const* peer_keys, int tp, int rank, const int* step_ctr,
                                       int64_t* out, int dtype, void* stream) {
  HQQ_REQUIRE(logits && out && peer_keys && step_ctr && n > 0 && index_offset >= 0 && index_offset + n <= 0xFFFFFFFFll && tp >= 1 && tp <= 8 &&
                  rank >= 0 && rank < tp,
              HQQ_E_INVALID, "hqq_b200_glue_argmax_tp: bad arguments (n=%d tp=%d rank=%d)", n, tp, rank);
  KeyPeers kp = {};
  for (int i = 0; i < tp; ++i) {
    HQQ_REQUIRE(peer_keys[i] && ((uintptr_t)peer_keys[i] & 7) == 0, HQQ_E_INVALID, "hqq_b200_glue_argmax_tp: key area %d must be 8-byte aligned", i);
    kp.p[i] = (unsigned long long*)peer_keys[i];
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == HQQ_F16) return launch_pdl("argmax_tp", argmax_kernel<__half>, dim3(kArgmaxCtas), dim3(1024), 0, st, true, (const __half*)logits, n, (long long*)out, (long long)index_offset, kp, tp, rank, step_ctr);
  if (dtype == HQQ_BF16) return launch_pdl("argmax_tp", argmax_kernel<__nv_bfloat16>, dim3(kArgmaxCtas), dim3(1024), 0, st, true, (const __nv_bfloat16*)logits, n, (long long*)out, (long long)index_offset, kp, tp, rank, step_ctr);
  set_error("hqq_b200_glue_argmax_tp: dtype must be f16/bf16");
  return HQQ_E_INVALID;
}
#endif  // !HQQ_EMU
