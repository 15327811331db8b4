// HQQLinear.forward for small M (decode): fused unpack -> group-dequant -> MMA, weight-streaming (HBM-bound).
//
// y[M,N] = x[M,K] @ dequantize(W_q)^T (+bias)        reference: hqq/core/quantize.py:880-898
//
// The packed tensor keeps the reference's slab layout (bitpack.py): for axis=1 a byte at packed row p,
// column k holds the levels of output rows p + f*(N/F), f = 0..F-1 (F = 8/nbits).  A warp owns a 16-row
// MMA tile made of P = 16/F packed rows x F slabs and streams them along K with 16-byte loads straight
// into registers (each weight byte is read exactly once, L1::no_allocate).  The levels are NOT dequantised
// per element: with per-group scale s and zero z
//        sum_k x_k (q_k - z) s  =  s * (sum_k q_k x_k)  -  s z * (sum_k x_k)
// so the tensor core contracts the raw levels (bit-tricked into fp16/bf16 lanes, 6-9 ALU ops per 8 weights)
// against x, a second MMA with an all-ones A tile yields sum_k x_k in the same fragment layout, and the
// affine correction is applied once per group per accumulator (fp32).  mma.sync m16n8k16 with register A
// fragments is used on purpose: at M <= 32 the kernel is bound by HBM and instruction issue, and a
// register-operand MMA avoids the shared-memory round trip a tcgen05 operand would need.
//
// Scheduling: persistent CTAs walk the 16-row tiles of up to four weight matrices that share the activation (q/k/v,
// gate/up) round-robin; the 8 warps of a CTA split K of a tile and stream their chunks through private cp.async rings
// in shared memory (3 x 2 KB in flight per warp, prefetching across tile boundaries), then reduce through shared
// memory in a fixed order: deterministic, no atomics, no workspace.  Launched with programmatic dependent launch: the
// weight prefetch starts before the producer of x has finished.
#include <stdlib.h>
#include <type_traits>

#include "device.cuh"
#include "linear_internal.cuh"

namespace hqq {


constexpr int kMaxProb = 4;   // weight matrices sharing one activation in a single launch (q/k/v, gate/up)

struct SKProb {
  const uint8_t* Wq;
  const void* scale;
  const void* zero;
  const void* bias;
  void* y;
  uint32_t* ytag;  // optional tagged copy of the output [2 parities][N] (see the exchange notes in SKArgs)
  int N;
  int step;   // packed rows = N / F
  int tile0;  // first global 16-row tile of this matrix
};

struct SKArgs {
  SKProb p[kMaxProb];
  int nprob;
  const void* x;
  int M, K;
  int Gk;           // groups per output row = K / GS
  int KB;           // 256-k units per row tile = K / 256
  int total_tiles;
  // optional activation prologue (M == 1 decode kernel only; used by the decode harness to drop a launch):
  //   xop 0: x as is;  1: x = rmsnorm(x + x2) * xw, and h_out = x + x2 is written by CTA 0 (x2 may be null);
  //   xop 2: x = silu(x) * x2
  int xop;
  // optional epilogue (M == 1 decode kernel, nbits < 8, exactly two matrices of equal N -- the MLP's gate and up):
  //   yop 1: y[0][n] = silu(W0 x)[n] * (W1 x)[n]; every 16-row tile then holds P/2 packed rows of EACH matrix, so both
  //   operands of an output meet in one CTA and the activation is computed once instead of by every consumer CTA.
  int yop;
  const void* x2;
  const void* xw;
  void* h_out;
  float eps;
  // optional tensor-parallel exchange over NVLink peer memory (M == 1 decode kernel), "LL" style: every fp16/bf16 result
  // travels as one 32-bit word {tag16 : value16}, written with a single store into EVERY rank's exchange buffer
  // peer_data[dst][parity][rank][n]; a consumer polls the words until the tag matches -- no fences, no flags, no
  // collective launch.  tag = low 16 bits of the exchange number (*step_ctr * x_per_step + x_index), parity = its bit 0
  // (ranks can be at most one exchange apart).  *step_ctr lives in device memory and is bumped once per token by the
  // last consumer, so a captured graph can be replayed.
  //   producer (row-parallel o / down, single matrix): peer_data != null
  //   consumer (xop 1): red_data != null, the residual delta is sum_r red_data[parity][r][k]
  // The same tagged words chain kernels on ONE GPU: a producer may keep a tagged copy of its outputs (SKProb::ytag) and a
  // consumer may take x / x2 of the SiLU*mul prologue from tagged buffers (xtag / x2tag) or its residual delta from
  // red_data with tp == 1.
  int tp, rank;
  uint32_t* peer_data[8];
  const uint32_t* red_data;
  const uint32_t* xtag;
  const uint32_t* x2tag;
  const int* step_ctr;
  int x_index, x_per_step;
};

// the 16-bit activation / output type of an MMA tile
template <typename T> struct MT16 {
  static constexpr uint32_t ONE2 = std::is_same<T, __half>::value ? 0x3C003C00u : 0x3F803F80u;  // {1, 1}: the all-ones A tile
  __device__ __forceinline__ static T cvt(float v, const void* bias, int n) {
    T o = from_f32<T>(v);
    if (bias) o = __hadd(o, reinterpret_cast<const T*>(bias)[n]);  // out += bias, second rounding as in the reference
    return o;
  }
  __device__ __forceinline__ static void st(void* p, long long i, float v, const void* bias, int n) { reinterpret_cast<T*>(p)[i] = cvt(v, bias, n); }
};

// (a & b) | c
__device__ __forceinline__ uint32_t and_or(uint32_t a, uint32_t b, uint32_t c) { return lop3<0xEA>(a, b, c); }

// How the integer levels are planted into 16-bit float lanes (lane value = OFF + q * V):
//   fp16: bits | 0x6400 -> 1024 + q*2^sh          bf16: (bits >> sh) | 0x4300 -> 128 + q
template <typename T, int NBITS> struct Lanes;

// fp16, sub-byte fields: mask in place, no shift (1 PRMT + 1 SHF + 4 LOP3 per 8 weights)
template <int NBITS>
struct Lanes<__half, NBITS> {
  static constexpr uint32_t OR = 0x64006400u;
  uint32_t mask_a, mask_b;
  float invV_a, invV_b, offV_a, offV_b;
  __device__ __forceinline__ void init(int sh_a, int sh_b) {
    const uint32_t m = (1u << NBITS) - 1u;
    mask_a = (m << sh_a) * 0x00010001u;
    mask_b = (m << sh_b) * 0x00010001u;
    invV_a = exp2f(-(float)sh_a); invV_b = exp2f(-(float)sh_b);
    offV_a = 1024.0f * invV_a;    offV_b = 1024.0f * invV_b;
  }
  // w: 4 consecutive k-bytes of one packed row.  a0/a2: field A for k{0,1} / k{2,3}; a1/a3: field B.
  __device__ __forceinline__ void extract(uint32_t w, uint32_t& a0, uint32_t& a1, uint32_t& a2, uint32_t& a3) const {
    const uint32_t wp = prmt(w, 0u, 0x3120u);  // bytes [k0,k2,k1,k3]: 16-bit lanes {k0|k2<<8, k1|k3<<8}
    const uint32_t wh = wp >> 8;
    a0 = and_or(wp, mask_a, OR);
    a1 = and_or(wp, mask_b, OR);
    a2 = and_or(wh, mask_a, OR);
    a3 = and_or(wh, mask_b, OR);
  }
  // same without the byte shuffle: lanes pair {k0,k2} (a0/a1) and {k1,k3} (a2/a3); the caller permutes x instead
  __device__ __forceinline__ void extract_np(uint32_t w, uint32_t& a0, uint32_t& a1, uint32_t& a2, uint32_t& a3) const {
    const uint32_t wh = w >> 8;
    a0 = and_or(w, mask_a, OR);
    a1 = and_or(w, mask_b, OR);
    a2 = and_or(wh, mask_a, OR);
    a3 = and_or(wh, mask_b, OR);
  }
};

// bf16, sub-byte fields: only 7 mantissa bits -> shift the field down to bit 0 first
template <int NBITS>
struct Lanes<__nv_bfloat16, NBITS> {
  int sh_a, sh_b;
  float invV_a, invV_b, offV_a, offV_b;
  __device__ __forceinline__ void init(int sa, int sb) {
    sh_a = sa; sh_b = sb;
    invV_a = invV_b = 1.0f;
    offV_a = offV_b = 128.0f;
  }
  __device__ __forceinline__ void extract(uint32_t w, uint32_t& a0, uint32_t& a1, uint32_t& a2, uint32_t& a3) const {
    constexpr uint32_t M = ((1u << NBITS) - 1u) * 0x00010001u;
    const uint32_t wp = prmt(w, 0u, 0x3120u);
    a0 = and_or(wp >> sh_a, M, 0x43004300u);
    a1 = and_or(wp >> sh_b, M, 0x43004300u);
    a2 = and_or(wp >> (sh_a + 8), M, 0x43004300u);
    a3 = and_or(wp >> (sh_b + 8), M, 0x43004300u);
  }
  __device__ __forceinline__ void extract_np(uint32_t w, uint32_t& a0, uint32_t& a1, uint32_t& a2, uint32_t& a3) const {
    constexpr uint32_t M = ((1u << NBITS) - 1u) * 0x00010001u;
    a0 = and_or(w >> sh_a, M, 0x43004300u);
    a1 = and_or(w >> sh_b, M, 0x43004300u);
    a2 = and_or(w >> (sh_a + 8), M, 0x43004300u);
    a3 = and_or(w >> (sh_b + 8), M, 0x43004300u);
  }
};

// fp16, 8-bit: whole bytes, two packed rows per thread (rows r and r+8 of the tile)
template <>
struct Lanes<__half, 8> {
  static constexpr uint32_t HB = 0x64646464u;
  float invV_a, invV_b, offV_a, offV_b;
  __device__ __forceinline__ void init(int, int) { invV_a = invV_b = 1.0f; offV_a = offV_b = 1024.0f; }
  __device__ __forceinline__ void extract2(uint32_t wa, uint32_t wb, uint32_t& a0, uint32_t& a1, uint32_t& a2, uint32_t& a3) const {
    a0 = prmt(wa, HB, 0x4140u);  // lanes {k0, k1} of row r
    a2 = prmt(wa, HB, 0x4342u);  // lanes {k2, k3}
    a1 = prmt(wb, HB, 0x4140u);  // row r+8
    a3 = prmt(wb, HB, 0x4342u);
  }
  __device__ __forceinline__ void extract2_np(uint32_t wa, uint32_t wb, uint32_t& a0, uint32_t& a1, uint32_t& a2, uint32_t& a3) const {
    a0 = prmt(wa, HB, 0x4240u);  // lanes {k0, k2}
    a2 = prmt(wa, HB, 0x4341u);  // lanes {k1, k3}
    a1 = prmt(wb, HB, 0x4240u);
    a3 = prmt(wb, HB, 0x4341u);
  }
};

template <typename T, int NBITS, int GS, int MT>
struct SKCfg {
  static constexpr int F = 8 / NBITS;            // fields (slabs) per byte
  static constexpr int P = 16 / F;               // packed rows per 16-row MMA tile
  static constexpr int MPG = GS / 16;            // MMAs per quantisation group
  static constexpr int GPB = 256 / GS;           // quantisation groups per 256-k unit
  static constexpr int NWV = (F == 1) ? 8 : 4;   // 16-byte weight vectors per thread and unit
  static constexpr int ST = (F == 1) ? 2 : 4;    // ring stages
  static constexpr int W_BYTES = ST * NWV * 256 * 16;   // scale/zero travel through registers
  static constexpr int P_BYTES = 2 * 8 * MT * 128 * 4;  // double-buffered split-K partials, one 16x8 tile per warp
  static constexpr int SMEM = W_BYTES + P_BYTES;
  static constexpr int MIN_CTAS = (SMEM <= 110 * 1024 && MT <= 2) ? 2 : 1;
};

// Persistent CTAs; CTA b owns the 16-row tiles b, b+grid, b+2*grid, ... of the concatenated tile list of up to four
// matrices.  Its 8 warps split K of the current tile into 8 contiguous chunks of 256-k units and stream them through
// per-thread cp.async rings (the ring keeps prefetching across tile boundaries, so HBM requests never drain).  Partials
// meet in shared memory once per tile (one block barrier, double-buffered) and warp (tile % 8) adds them in warp order:
// deterministic, no atomics, no global workspace.
template <typename T, int NBITS, int GS, int MT>
__global__ void __launch_bounds__(256, SKCfg<T, NBITS, GS, MT>::MIN_CTAS) linear_small_kernel(const __grid_constant__ SKArgs a) {
  using C = SKCfg<T, NBITS, GS, MT>;
  constexpr int F = C::F, P = C::P, MPG = C::MPG, GPB = C::GPB, NWV = C::NWV, ST = C::ST;
  using MM = MT16<T>;
  extern __shared__ __align__(16) uint8_t smem[];
  uint4* wring = reinterpret_cast<uint4*>(smem);                  // [ST][NWV][256] one 16-byte slot per thread
  float* part_s = reinterpret_cast<float*>(smem + C::W_BYTES);  // [2][8][MT][128]

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int r = lane >> 2, c = lane & 3;
  const int p = (F == 1) ? r : (r % P);
  const int fa = (F == 1) ? 0 : (r / P), fb = (F == 1) ? 0 : (F / 2 + r / P);
  Lanes<T, NBITS> lanes;
  lanes.init(8 - NBITS * (fa + 1), 8 - NBITS * (fb + 1));

  // this warp's k-chunk of every tile (the same for all tiles: all matrices share K)
  const int kb0 = a.KB * warp / 8, kb1 = a.KB * (warp + 1) / 8;
  const int upt = kb1 - kb0;  // units per tile for this warp (may be 0 when K < 2048)
  const int n_tiles = (a.total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;  // tiles owned by this CTA
  if (n_tiles <= 0) return;

  struct Tile {
    const uint8_t* Wq; const T* scale; const T* zero; const T* bias; T* y;
    int N, step, tile0;
  };
  auto locate = [&](int gt, Tile& t) {
    int pi = 0;
#pragma unroll
    for (int i = 1; i < kMaxProb; ++i)
      if (i < a.nprob && gt >= a.p[i].tile0) pi = i;
    const uint8_t* Wq = a.p[0].Wq; const void* sc = a.p[0].scale; const void* ze = a.p[0].zero; const void* bi = a.p[0].bias;
    void* y = a.p[0].y; int N = a.p[0].N, step = a.p[0].step, tile0 = a.p[0].tile0;
#pragma unroll
    for (int i = 1; i < kMaxProb; ++i)
      if (pi == i) { Wq = a.p[i].Wq; sc = a.p[i].scale; ze = a.p[i].zero; bi = a.p[i].bias; y = a.p[i].y; N = a.p[i].N; step = a.p[i].step; tile0 = a.p[i].tile0; }
    t.Wq = Wq; t.scale = reinterpret_cast<const T*>(sc); t.zero = reinterpret_cast<const T*>(ze);
    t.bias = reinterpret_cast<const T*>(bi); t.y = reinterpret_cast<T*>(y); t.N = N; t.step = step; t.tile0 = tile0;
  };

  // ---- issue cursor -------------------------------------------------------------------------------------------
  int i_tile = 0, i_k = 0;  // index into this CTA's tile list / unit within the warp's chunk
  const uint8_t *iw_a, *iw_b;
  auto issue_setup = [&]() {
    Tile t; locate((int)blockIdx.x + i_tile * (int)gridDim.x, t);
    const int gt = (int)blockIdx.x + i_tile * (int)gridDim.x;
    const int prow_a = (gt - t.tile0) * P + p, prow_b = (F == 1) ? prow_a + 8 : prow_a;
    // rows past the ragged edge re-read row 0 (always mapped); their results are never stored
    const long long ra = prow_a < t.step ? prow_a : 0, rb = prow_b < t.step ? prow_b : 0;
    iw_a = t.Wq + ra * a.K + (long long)kb0 * 256 + 16 * c;
    iw_b = t.Wq + rb * a.K + (long long)kb0 * 256 + 16 * c;
  };
  int to_issue = n_tiles * upt;
  if (to_issue > 0) issue_setup();
  // ---- meta cursor: scale/zero of the NEXT unit travel through registers (plain cached loads, one unit ahead).  They
  // used to ride the cp.async ring, but 8-byte cp.async costs one shared-memory wavefront per lane (ncu: 60 % of all
  // shared wavefronts of the kernel).
  int m_tile = 0, m_k = 0, m_left = n_tiles * upt;
  const T *ms_a = nullptr, *mz_a = nullptr, *ms_b = nullptr, *mz_b = nullptr;
  auto meta_setup = [&]() {
    const int gt = (int)blockIdx.x + m_tile * (int)gridDim.x;
    Tile t; locate(gt, t);
    const int prow_a = (gt - t.tile0) * P + p, prow_b = (F == 1) ? prow_a + 8 : prow_a;
    const long long na = prow_a < t.step ? fa * t.step + prow_a : 0, nb = prow_b < t.step ? fb * t.step + prow_b : 0;
    ms_a = t.scale + na * a.Gk + kb0 * GPB; mz_a = t.zero + na * a.Gk + kb0 * GPB;
    ms_b = t.scale + nb * a.Gk + kb0 * GPB; mz_b = t.zero + nb * a.Gk + kb0 * GPB;
  };
  if (m_left > 0) meta_setup();
  Vec<T, GPB> mv[4];
  auto meta_fetch = [&]() {
    if (m_left > 0) {
      mv[0] = *reinterpret_cast<const Vec<T, GPB>*>(ms_a); mv[1] = *reinterpret_cast<const Vec<T, GPB>*>(mz_a);
      mv[2] = *reinterpret_cast<const Vec<T, GPB>*>(ms_b); mv[3] = *reinterpret_cast<const Vec<T, GPB>*>(mz_b);
      --m_left;
      if (++m_k == upt) {
        m_k = 0; ++m_tile;
        if (m_left > 0) meta_setup();
      } else {
        ms_a += GPB; mz_a += GPB; ms_b += GPB; mz_b += GPB;
      }
    }
  };
  meta_fetch();
  auto issue = [&](int stage) {
    if (to_issue > 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) cp_async16(&wring[(stage * NWV + i) * 256 + tid], iw_a + i * 64);
      if (F == 1) {
#pragma unroll
        for (int i = 0; i < 4; ++i) cp_async16(&wring[(stage * NWV + 4 + i) * 256 + tid], iw_b + i * 64);
      }
      --to_issue;
      if (++i_k == upt) {
        i_k = 0; ++i_tile;
        if (to_issue > 0) issue_setup();
      } else {
        iw_a += 256; iw_b += 256;
      }
    }
    cp_async_commit();  // always commit (possibly empty) so the group count per iteration is uniform
  };
  // Weights and meta never depend on the previous kernel: start streaming them before the programmatic-dependency wait,
  // so under PDL this prologue overlaps the tail of whatever produced x.
#pragma unroll
  for (int s = 0; s < ST - 1; ++s) issue(s);
  pdl_launch_dependents();
  pdl_wait();

  const T* xbase[MT];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) {
    // token columns >= M alias the last real token: MMA columns are independent and never stored
    const int m = min(mt * 8 + r, a.M - 1);
    xbase[mt] = reinterpret_cast<const T*>(a.x) + (long long)m * a.K + 16 * c;
  }
  // activations are software-pipelined one k64 step ahead (they come from L1/L2, 16 consecutive k per thread)
  uint4 xa[MT], xb[MT];
  auto load_x = [&](int kb, int us) {
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) {
      const uint4* q = reinterpret_cast<const uint4*>(xbase[mt] + kb * 256 + us * 64);
      xa[mt] = __ldg(q);
      xb[mt] = __ldg(q + 1);
    }
  };
  if (upt > 0) load_x(kb0, 0);

  int stage = 0;
  for (int ti = 0; ti < n_tiles; ++ti) {
    float tot[MT][4];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int i = 0; i < 4; ++i) tot[mt][i] = 0.0f;

    for (int ku = 0; ku < upt; ++ku) {
      {
        int is = stage + (ST - 1);
        if (is >= ST) is -= ST;
        issue(is);
      }
      cp_async_wait<ST - 1>();  // the group of this unit (and everything older) has landed in this thread's slots

      float sA[GPB], zA[GPB], sB[GPB], zB[GPB];
#pragma unroll
      for (int i = 0; i < GPB; ++i) { sA[i] = to_f32<T>(mv[0].v[i]); zA[i] = to_f32<T>(mv[1].v[i]); sB[i] = to_f32<T>(mv[2].v[i]); zB[i] = to_f32<T>(mv[3].v[i]); }
      meta_fetch();  // next unit's scale/zero: a full unit of work hides the (mostly L1/L2) latency
      const int kb = kb0 + ku;
      const int kb_next = (ku + 1 == upt) ? kb0 : kb + 1;  // x depends on k only: the next tile restarts at kb0
      float Sg[MT][4], Xg[MT][4];
#pragma unroll
      for (int us = 0; us < 4; ++us) {
        uint4 ya[MT], yb[MT];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) { ya[mt] = xa[mt]; yb[mt] = xb[mt]; }
        if (us < 3) load_x(kb, us + 1); else load_x(kb_next, 0);
        const uint4 va = wring[(stage * NWV + us) * 256 + tid];
        uint4 vb = va;
        if (F == 1) vb = wring[(stage * NWV + 4 + us) * 256 + tid];
        const uint32_t wa[4] = {va.x, va.y, va.z, va.w};
        const uint32_t wb[4] = {vb.x, vb.y, vb.z, vb.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t a0, a1, a2, a3;
          if constexpr (F == 1) lanes.extract2(wa[j], wb[j], a0, a1, a2, a3);
          else lanes.extract(wa[j], a0, a1, a2, a3);
          const bool first = ((us * 4 + j) % MPG) == 0;  // first MMA of a group starts from C = 0
#pragma unroll
          for (int mt = 0; mt < MT; ++mt) {
            const uint32_t b0 = (j == 0) ? ya[mt].x : (j == 1) ? ya[mt].z : (j == 2) ? yb[mt].x : yb[mt].z;
            const uint32_t b1 = (j == 0) ? ya[mt].y : (j == 1) ? ya[mt].w : (j == 2) ? yb[mt].y : yb[mt].w;
            mma_m16n8k16<T>(Sg[mt], a0, a1, a2, a3, b0, b1, first);
            mma_m16n8k16<T>(Xg[mt], MM::ONE2, MM::ONE2, MM::ONE2, MM::ONE2, b0, b1, first);
          }
          if (((us * 4 + j + 1) % MPG) == 0) {
            // a quantisation group is complete: tot += s*(Q - z*X), with lane value = OFF + q*V folded in
            const int gi = (us * 4 + j) / MPG;
            const float ka = sA[gi] * lanes.invV_a, la = -sA[gi] * (lanes.offV_a + zA[gi]);
            const float kb2 = sB[gi] * lanes.invV_b, lb = -sB[gi] * (lanes.offV_b + zB[gi]);
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
              tot[mt][0] = fmaf(ka, Sg[mt][0], fmaf(la, Xg[mt][0], tot[mt][0]));
              tot[mt][1] = fmaf(ka, Sg[mt][1], fmaf(la, Xg[mt][1], tot[mt][1]));
              tot[mt][2] = fmaf(kb2, Sg[mt][2], fmaf(lb, Xg[mt][0], tot[mt][2]));
              tot[mt][3] = fmaf(kb2, Sg[mt][3], fmaf(lb, Xg[mt][1], tot[mt][3]));
            }
          }
        }
      }
      if (++stage == ST) stage = 0;
    }

    // ---- tile done: partials meet in shared memory (double-buffered: one barrier per tile is enough) -----------
    float* buf = part_s + (ti & 1) * (8 * MT * 128);
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
      *reinterpret_cast<float4*>(buf + (warp * MT + mt) * 128 + lane * 4) = make_float4(tot[mt][0], tot[mt][1], tot[mt][2], tot[mt][3]);
    __syncthreads();
    if (warp == (ti & 7)) {
      const int gt = (int)blockIdx.x + ti * (int)gridDim.x;
      Tile t; locate(gt, t);
      const int prow_a = (gt - t.tile0) * P + p, prow_b = (F == 1) ? prow_a + 8 : prow_a;
      const bool ok_a = prow_a < t.step, ok_b = prow_b < t.step;
      const int n_a = fa * t.step + prow_a, n_b = fb * t.step + prow_b;
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int w = 0; w < 8; ++w) {
          const float4 v = *reinterpret_cast<const float4*>(buf + (w * MT + mt) * 128 + lane * 4);
          acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        const int m0 = mt * 8 + 2 * c;
        if (m0 < a.M) {
          if (ok_a) MM::st(t.y, (long long)m0 * t.N + n_a, acc.x, t.bias, n_a);
          if (ok_b) MM::st(t.y, (long long)m0 * t.N + n_b, acc.z, t.bias, n_b);
        }
        if (m0 + 1 < a.M) {
          if (ok_a) MM::st(t.y, (long long)(m0 + 1) * t.N + n_a, acc.y, t.bias, n_a);
          if (ok_b) MM::st(t.y, (long long)(m0 + 1) * t.N + n_b, acc.w, t.bias, n_b);
        }
      }
    }
  }
  cp_async_wait<0>();
}

// ---------------------------------------------------------------------------------------------------------
// M == 1 specialisation (the decode hot path).  Same scheduling and staging as linear_small_kernel, but everything that
// depends only on the activation is hoisted out of the per-tile loop: each warp stages ITS k-chunk of x once in shared
// memory, already permuted to the lane pairing the bit-tricks produce ({k0,k2},{k1,k3}: no PRMT on the weights), and
// sums it per quantisation group once (no all-ones MMA); the affine correction is applied to the single real column.
// MR = 1: scale/zero ride the cp.async ring at the same distance as the weights (16-byte copies of the aligned block that holds
// this unit's 8 bytes) instead of register loads one unit ahead -- ncu showed 18 % of all stall samples on the first use of
// those registers (DRAM latency under load exceeds one unit of work).
template <typename T, int NBITS, int GS, int ST, int MR = 0>
struct D1Cfg {
  static constexpr int F = 8 / NBITS, P = 16 / F, MPG = GS / 16, GPB = 256 / GS;
  static constexpr int NWV = (F == 1) ? 8 : 4;
  static constexpr int W_BYTES = ST * NWV * 256 * 16;
  static constexpr int M_BYTES = (MR & 1) ? ST * 8 * 4 * 8 * 16 : 0;  // MR: [stage][warp][vector][row] 16-byte blocks; else registers
  static constexpr int P_BYTES = 2 * 8 * 16 * 4;  // double-buffered: 8 warps x 16 rows
  static int smem(int K) { return W_BYTES + M_BYTES + P_BYTES + K * 2 + (K / GS) * 4; }
};

template <typename T, int NBITS, int GS, int ST, int MC, int MR = 0>
__global__ void __launch_bounds__(256, MC) linear_decode1_kernel(const __grid_constant__ SKArgs a) {
  using C = D1Cfg<T, NBITS, GS, ST, MR>;
  constexpr int F = C::F, P = C::P, MPG = C::MPG, GPB = C::GPB, NWV = C::NWV;
  using MM = MT16<T>;
  extern __shared__ __align__(16) uint8_t smem[];
  uint4* wring = reinterpret_cast<uint4*>(smem);
  uint4* mring = reinterpret_cast<uint4*>(smem + C::W_BYTES);  // MR only
  float* part_s = reinterpret_cast<float*>(smem + C::W_BYTES + C::M_BYTES);       // [2][8][16]
  T* xs = reinterpret_cast<T*>(smem + C::W_BYTES + C::M_BYTES + C::P_BYTES);      // [K] permuted activations
  float* xsum = reinterpret_cast<float*>(smem + C::W_BYTES + C::M_BYTES + C::P_BYTES + a.K * 2);  // [K/GS]

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int r = lane >> 2, c = lane & 3;
  const int p = (F == 1) ? r : (r % P);
  const int fa = (F == 1) ? 0 : (r / P), fb = (F == 1) ? 0 : (F / 2 + r / P);
  Lanes<T, NBITS> lanes;
  lanes.init(8 - NBITS * (fa + 1), 8 - NBITS * (fb + 1));

  const int kb0 = a.KB * warp / 8, kb1 = a.KB * (warp + 1) / 8;
  const int upt = kb1 - kb0;
  const int n_tiles = (a.total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  if (n_tiles <= 0) return;

  struct Tile { const uint8_t* Wq; const T* scale; const T* zero; const T* bias; T* y; uint32_t* ytag; int N, step, tile0; };
  auto pick = [&](int pi, Tile& t) {
    const uint8_t* Wq = a.p[0].Wq; const void* sc = a.p[0].scale; const void* ze = a.p[0].zero; const void* bi = a.p[0].bias;
    void* y = a.p[0].y; uint32_t* yt = a.p[0].ytag; int N = a.p[0].N, step = a.p[0].step, tile0 = a.p[0].tile0;
#pragma unroll
    for (int i = 1; i < kMaxProb; ++i)
      if (pi == i) { Wq = a.p[i].Wq; sc = a.p[i].scale; ze = a.p[i].zero; bi = a.p[i].bias; y = a.p[i].y; yt = a.p[i].ytag; N = a.p[i].N; step = a.p[i].step; tile0 = a.p[i].tile0; }
    t.Wq = Wq; t.scale = reinterpret_cast<const T*>(sc); t.zero = reinterpret_cast<const T*>(ze);
    t.bias = reinterpret_cast<const T*>(bi); t.y = reinterpret_cast<T*>(y); t.ytag = yt; t.N = N; t.step = step; t.tile0 = tile0;
  };
  auto locate = [&](int gt, Tile& t) {
    int pi = 0;
#pragma unroll
    for (int i = 1; i < kMaxProb; ++i)
      if (i < a.nprob && gt >= a.p[i].tile0) pi = i;
    pick(pi, t);
  };
  // paired epilogue (yop 1, F > 1): tile gt = packed rows [gt*PH, gt*PH + PH) of matrix 0 (fragment rows p < PH) and of matrix 1
  constexpr int PH = (P >= 2) ? P / 2 : 1;
  const bool paired = (F > 1) && a.yop == 1;
  auto my_rows = [&](int gt, Tile& t, int& prow_a, int& prow_b) {
    if (paired) {
      pick(p >= PH ? 1 : 0, t);
      prow_a = prow_b = gt * PH + (p % PH);
    } else {
      locate(gt, t);
      prow_a = (gt - t.tile0) * P + p;
      prow_b = (F == 1) ? prow_a + 8 : prow_a;
    }
  };

  int i_tile = 0, i_k = 0;
  const uint8_t *iw_a, *iw_b;
  const T* im = nullptr;  // MR: this lane's meta vector (c = 0: scale of row a, 1: zero of row a, 2: scale of row b, 3: zero of row b)
  auto issue_setup = [&]() {
    const int gt = (int)blockIdx.x + i_tile * (int)gridDim.x;
    Tile t; int prow_a, prow_b;
    my_rows(gt, t, prow_a, prow_b);
    const long long ra = prow_a < t.step ? prow_a : 0, rb = prow_b < t.step ? prow_b : 0;
    iw_a = t.Wq + ra * a.K + (long long)kb0 * 256 + 16 * c;
    iw_b = t.Wq + rb * a.K + (long long)kb0 * 256 + 16 * c;
    if constexpr ((MR & 1) != 0) {
      const long long na = prow_a < t.step ? fa * t.step + prow_a : 0, nb = prow_b < t.step ? fb * t.step + prow_b : 0;
      im = ((c & 1) ? t.zero : t.scale) + ((c & 2) ? nb : na) * a.Gk + kb0 * GPB;
    }
  };
  int to_issue = n_tiles * upt;
  if (to_issue > 0) issue_setup();
  // ---- meta cursor: scale/zero of the NEXT unit travel through registers (plain cached loads, one unit ahead).  They
  // used to ride the cp.async ring, but 8-byte cp.async costs one shared-memory wavefront per lane (ncu: 60 % of all
  // shared wavefronts of the kernel).
  int m_tile = 0, m_k = 0, m_left = (MR & 1) ? 0 : n_tiles * upt;
  const T *ms_a = nullptr, *mz_a = nullptr, *ms_b = nullptr, *mz_b = nullptr;
  auto meta_setup = [&]() {
    const int gt = (int)blockIdx.x + m_tile * (int)gridDim.x;
    Tile t; int prow_a, prow_b;
    my_rows(gt, t, prow_a, prow_b);
    const long long na = prow_a < t.step ? fa * t.step + prow_a : 0, nb = prow_b < t.step ? fb * t.step + prow_b : 0;
    ms_a = t.scale + na * a.Gk + kb0 * GPB; mz_a = t.zero + na * a.Gk + kb0 * GPB;
    ms_b = t.scale + nb * a.Gk + kb0 * GPB; mz_b = t.zero + nb * a.Gk + kb0 * GPB;
  };
  if (m_left > 0) meta_setup();
  Vec<T, GPB> mv[4];
  auto meta_fetch = [&]() {
    if (m_left > 0) {
      mv[0] = *reinterpret_cast<const Vec<T, GPB>*>(ms_a); mv[1] = *reinterpret_cast<const Vec<T, GPB>*>(mz_a);
      mv[2] = *reinterpret_cast<const Vec<T, GPB>*>(ms_b); mv[3] = *reinterpret_cast<const Vec<T, GPB>*>(mz_b);
      --m_left;
      if (++m_k == upt) {
        m_k = 0; ++m_tile;
        if (m_left > 0) meta_setup();
      } else {
        ms_a += GPB; mz_a += GPB; ms_b += GPB; mz_b += GPB;
      }
    }
  };
  meta_fetch();
  auto issue = [&](int stage) {
    if (to_issue > 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) cp_async16(&wring[(stage * NWV + i) * 256 + tid], iw_a + i * 64);
      if (F == 1) {
#pragma unroll
        for (int i = 0; i < 4; ++i) cp_async16(&wring[(stage * NWV + 4 + i) * 256 + tid], iw_b + i * 64);
      }
      if constexpr ((MR & 1) != 0)  // the aligned 16 bytes holding this unit's GPB values (rows are 16-byte aligned: host check)
        cp_async16(&mring[((stage * 8 + warp) * 4 + c) * 8 + r], reinterpret_cast<const void*>(reinterpret_cast<uintptr_t>(im) & ~uintptr_t(15)));
      --to_issue;
      if (++i_k == upt) {
        i_k = 0; ++i_tile;
        if (to_issue > 0) issue_setup();
      } else {
        iw_a += 256; iw_b += 256;
        if constexpr ((MR & 1) != 0) im += GPB;
      }
    }
    cp_async_commit();
  };
#pragma unroll
  for (int s = 0; s < ST - 1; ++s) issue(s);
  pdl_launch_dependents();  // our dependents' launch latency hides under our main loop
  pdl_wait();
  uint32_t send_tag = 0, send_par = 0;  // this launch's exchange number (shared by its producer and consumer sides)
  if (a.step_ctr) {
    const uint32_t ex = (uint32_t)(*reinterpret_cast<volatile const int*>(a.step_ctr)) * (uint32_t)a.x_per_step + (uint32_t)a.x_index;
    send_tag = ex & 0xFFFFu;
    send_par = ex & 1u;
  }

  // ---- stage this warp's k-chunk of x (permuted: k -> k with bits 0 and 1 swapped) and its per-group sums ----------
  {
    const T* x = reinterpret_cast<const T*>(a.x);
    const T* x2 = reinterpret_cast<const T*>(a.x2);
    const int k_lo = kb0 * 256, k_hi = kb1 * 256;
    float inv = 1.0f;
    const uint32_t* red = nullptr;  // this exchange's [tp][K] tagged partial results, written into our memory by the peers
    const uint32_t rtag = send_tag;
    if (a.xop == 1 && a.red_data) red = a.red_data + (size_t)send_par * a.tp * a.K;
    // poll eight consecutive tagged words until they all carry this exchange's tag (they may arrive in any order)
    auto poll8 = [&](const uint32_t* src, Vec<T, 8>& out) {
      uint4 w0, w1;
      bool ok;
      do {
        w0 = ld_relaxed_sys_v4(src);
        w1 = ld_relaxed_sys_v4(src + 4);
        ok = ((w0.x >> 16) == rtag) & ((w0.y >> 16) == rtag) & ((w0.z >> 16) == rtag) & ((w0.w >> 16) == rtag) &
             ((w1.x >> 16) == rtag) & ((w1.y >> 16) == rtag) & ((w1.z >> 16) == rtag) & ((w1.w >> 16) == rtag);
      } while (!ok);
      const uint32_t ws[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const unsigned short hb = (unsigned short)(ws[j] & 0xFFFFu);
        out.v[j] = *reinterpret_cast<const T*>(&hb);
      }
    };
    // delta of the residual stream: x2, or the sum of the tp partials (fp32 sum, rounded once like an all-reduce result)
    auto delta8 = [&](int k8, Vec<T, 8>& d) -> bool {
      if (red) {
        float acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = 0.0f;
        for (int rr = 0; rr < a.tp; ++rr) {
          Vec<T, 8> p8;
          poll8(red + (size_t)rr * a.K + k8, p8);
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] += to_f32<T>(p8.v[j]);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) d.v[j] = from_f32<T>(acc[j]);
        return true;
      }
      if (x2) { d = *reinterpret_cast<const Vec<T, 8>*>(x2 + k8); return true; }
      return false;
    };
    auto put_permuted = [&](int k8, const Vec<T, 8>& v) {
      Vec<T, 8> w;
      w.v[0] = v.v[0]; w.v[1] = v.v[2]; w.v[2] = v.v[1]; w.v[3] = v.v[3];
      w.v[4] = v.v[4]; w.v[5] = v.v[6]; w.v[6] = v.v[5]; w.v[7] = v.v[7];
      *reinterpret_cast<Vec<T, 8>*>(xs + k8) = w;
    };
    if (a.xop == 1) {
      // fused residual add + RMSNorm: every CTA needs the sum of squares of the whole vector (K elements, L2-resident).
      // One pass over global memory: t = x + delta is parked (unpermuted) in xs while its squares are summed, two vectors
      // per thread in flight; the norm weights of this lane's first two staging vectors are requested up front, so
      // after the reduction only shared memory is touched.
      const T* xw = reinterpret_cast<const T*>(a.xw);
      T* hout = reinterpret_cast<T*>(a.h_out);
      const int kg0 = k_lo + lane * 8;
      Vec<T, 8> g0, g1;
      if (kg0 < k_hi) g0 = *reinterpret_cast<const Vec<T, 8>*>(xw + kg0);
      if (kg0 + 256 < k_hi) g1 = *reinterpret_cast<const Vec<T, 8>*>(xw + kg0 + 256);
      float ss = 0.0f;
      for (int ka = tid * 8; ka < a.K; ka += 2 * 256 * 8) {
        const int kb = ka + 256 * 8;
        const bool has_b = kb < a.K;
        Vec<T, 8> va = *reinterpret_cast<const Vec<T, 8>*>(x + ka), vb, da, db;
        if (has_b) vb = *reinterpret_cast<const Vec<T, 8>*>(x + kb);
        const bool add_a = delta8(ka, da);
        const bool add_b = has_b && delta8(kb, db);
        if (add_a) {
#pragma unroll
          for (int j = 0; j < 8; ++j) va.v[j] = from_f32<T>(to_f32<T>(va.v[j]) + to_f32<T>(da.v[j]));
        }
        if (add_b) {
#pragma unroll
          for (int j = 0; j < 8; ++j) vb.v[j] = from_f32<T>(to_f32<T>(vb.v[j]) + to_f32<T>(db.v[j]));
        }
        *reinterpret_cast<Vec<T, 8>*>(xs + ka) = va;
        if (has_b) *reinterpret_cast<Vec<T, 8>*>(xs + kb) = vb;
        if (hout && blockIdx.x == 0) {  // the residual stream, written once
          *reinterpret_cast<Vec<T, 8>*>(hout + ka) = va;
          if (has_b) *reinterpret_cast<Vec<T, 8>*>(hout + kb) = vb;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) { const float f = to_f32<T>(va.v[j]); ss += f * f; }
        if (has_b) {
#pragma unroll
          for (int j = 0; j < 8; ++j) { const float f = to_f32<T>(vb.v[j]); ss += f * f; }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
      if (lane == 0) part_s[warp] = ss;
      __syncthreads();  // all 8 warps are still here (CTAs without tiles returned as a whole); also publishes xs
      float tot = 0.0f;
#pragma unroll
      for (int w = 0; w < 8; ++w) tot += part_s[w];
      inv = rsqrtf(tot / (float)a.K + a.eps);
      __syncthreads();  // part_s is reused by the tile reduction below
      int i = 0;
      for (int k8 = kg0; k8 < k_hi; k8 += 256, ++i) {
        Vec<T, 8> v = *reinterpret_cast<const Vec<T, 8>*>(xs + k8);
        const Vec<T, 8> g = (i == 0) ? g0 : (i == 1) ? g1 : *reinterpret_cast<const Vec<T, 8>*>(xw + k8);
#pragma unroll
        for (int j = 0; j < 8; ++j) v.v[j] = from_f32<T>(to_f32<T>(from_f32<T>(to_f32<T>(v.v[j]) * inv)) * to_f32<T>(g.v[j]));
        put_permuted(k8, v);  // in place: every lane rewrites exactly the eight elements it read
      }
    } else {
      for (int k8 = k_lo + lane * 8; k8 < k_hi; k8 += 256) {
        Vec<T, 8> v;
        if (a.xop == 2 && a.xtag) poll8(a.xtag + (size_t)send_par * a.K + k8, v);
        else v = *reinterpret_cast<const Vec<T, 8>*>(x + k8);
        if (a.xop == 2) {
          Vec<T, 8> u;
          if (a.x2tag) poll8(a.x2tag + (size_t)send_par * a.K + k8, u);
          else u = *reinterpret_cast<const Vec<T, 8>*>(x2 + k8);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float f = to_f32<T>(v.v[j]);
            v.v[j] = from_f32<T>(to_f32<T>(from_f32<T>(f / (1.0f + __expf(-f)))) * to_f32<T>(u.v[j]));
          }
        }
        put_permuted(k8, v);
      }
    }
    __syncwarp();
    for (int g = k_lo / GS + lane; g < k_hi / GS; g += 32) {
      float acc = 0.0f;
#pragma unroll 4
      for (int i = 0; i < GS; i += 8) {
        const Vec<T, 8> v = *reinterpret_cast<const Vec<T, 8>*>(xs + g * GS + i);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc += to_f32<T>(v.v[j]);
      }
      xsum[g] = acc;
    }
    __syncwarp();
  }

  int stage = 0;
  for (int ti = 0; ti < n_tiles; ++ti) {
    float tot_a = 0.0f, tot_b = 0.0f;
    for (int ku = 0; ku < upt; ++ku) {
      {
        int is = stage + (ST - 1);
        if (is >= ST) is -= ST;
        issue(is);
      }
      cp_async_wait<ST - 1>();
      const int kb = kb0 + ku;
      float sA[GPB], zA[GPB], sB[GPB], zB[GPB];
      if constexpr ((MR & 1) != 0) {
        // this unit's scale/zero arrived with its weights, copied by OTHER lanes of this warp: every lane has waited for its own
        // copies, the warp barrier makes them visible to the whole quad (and fences the slot against the next overwrite)
        __syncwarp();
        // lanes of a quad read the same 8 bytes (broadcast, conflict-free)
        const char* mr = reinterpret_cast<const char*>(mring + ((stage * 8 + warp) * 4) * 8) + r * 16 + ((kb * GPB * 2) & 15);
#pragma unroll
        for (int v = 0; v < 4; ++v) mv[v] = *reinterpret_cast<const Vec<T, GPB>*>(mr + v * 128);
      }
#pragma unroll
      for (int i = 0; i < GPB; ++i) { sA[i] = to_f32<T>(mv[0].v[i]); zA[i] = to_f32<T>(mv[1].v[i]); sB[i] = to_f32<T>(mv[2].v[i]); zB[i] = to_f32<T>(mv[3].v[i]); }
      if constexpr ((MR & 1) == 0) meta_fetch();  // next unit's scale/zero: a full unit of work hides the (mostly L1/L2) latency
      const T* xk = xs + kb * 256 + 16 * c;
      float Sg[4];
#pragma unroll
      for (int us = 0; us < 4; ++us) {
        const uint4 xa = *reinterpret_cast<const uint4*>(xk + us * 64);      // permuted: {k0,k2},{k1,k3},{k4,k6},{k5,k7}
        const uint4 xb = *reinterpret_cast<const uint4*>(xk + us * 64 + 8);
        const uint4 va = wring[(stage * NWV + us) * 256 + tid];
        uint4 vb = va;
        if (F == 1) vb = wring[(stage * NWV + 4 + us) * 256 + tid];
        const uint32_t wa[4] = {va.x, va.y, va.z, va.w};
        const uint32_t wb[4] = {vb.x, vb.y, vb.z, vb.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t a0, a1, a2, a3;
          if constexpr (F == 1) lanes.extract2_np(wa[j], wb[j], a0, a1, a2, a3);
          else lanes.extract_np(wa[j], a0, a1, a2, a3);
          const uint32_t b0 = (j == 0) ? xa.x : (j == 1) ? xa.z : (j == 2) ? xb.x : xb.z;
          const uint32_t b1 = (j == 0) ? xa.y : (j == 1) ? xa.w : (j == 2) ? xb.y : xb.w;
          mma_m16n8k16<T>(Sg, a0, a1, a2, a3, b0, b1, ((us * 4 + j) % MPG) == 0);
          if (((us * 4 + j + 1) % MPG) == 0) {
            const int gi = (us * 4 + j) / MPG;
            const float X = xsum[kb * GPB + gi];
            tot_a = fmaf(sA[gi] * lanes.invV_a, Sg[0], fmaf(-sA[gi] * (lanes.offV_a + zA[gi]), X, tot_a));
            tot_b = fmaf(sB[gi] * lanes.invV_b, Sg[2], fmaf(-sB[gi] * (lanes.offV_b + zB[gi]), X, tot_b));
          }
        }
      }
      if (++stage == ST) stage = 0;
    }
    // ---- tile done: every lane of a 4-lane group holds the same two row results; lane c == 0 publishes them ------
    float* buf = part_s + (ti & 1) * 128;
    if (c == 0) { buf[warp * 16 + r] = tot_a; buf[warp * 16 + 8 + r] = tot_b; }
    __syncthreads();
    if (warp == (ti & 7) && lane < 16) {
      const int gt = (int)blockIdx.x + ti * (int)gridDim.x;
      const int rr = lane & 7, hi = lane >> 3;  // fragment row lane = rr + 8*hi
      const int pp = (F == 1) ? rr : (rr % P);
      const int ff = (F == 1) ? 0 : (hi ? F / 2 + rr / P : rr / P);
      if (paired) {
        // lane (pp < PH) holds matrix 0's row, lane + PH the same row of matrix 1: activation computed once, here
        Tile tg, tu; pick(0, tg); pick(1, tu);
        const int prow = gt * PH + pp;
        if (pp < PH && prow < tg.step) {
          float ag = 0.0f, au = 0.0f;
#pragma unroll
          for (int w = 0; w < 8; ++w) { ag += buf[w * 16 + lane]; au += buf[w * 16 + lane + PH]; }
          const int n = ff * tg.step + prow;
          const float f = to_f32<T>(MM::cvt(ag, tg.bias, n));
          const float u = to_f32<T>(MM::cvt(au, tu.bias, n));
          tg.y[n] = from_f32<T>(to_f32<T>(from_f32<T>(f / (1.0f + __expf(-f)))) * u);
        }
        continue;
      }
      Tile t; locate(gt, t);
      const int prow = (gt - t.tile0) * P + pp + ((F == 1 && hi) ? 8 : 0);
      if (prow < t.step) {
        float acc = 0.0f;
#pragma unroll
        for (int w = 0; w < 8; ++w) acc += buf[w * 16 + lane];
        const int n = ff * t.step + prow;
        MM::st(t.y, n, acc, t.bias, n);
        if (a.peer_data[0] || t.ytag) {
          const T pv = from_f32<T>(acc);
          const uint32_t word = (send_tag << 16) | (uint32_t)(*reinterpret_cast<const unsigned short*>(&pv));
          if (a.peer_data[0]) {
            // scatter the (bias-free) partial over NVLink as one tagged word per value: slot [parity][rank][n] on every rank
            const size_t off = ((size_t)send_par * a.tp + a.rank) * t.N + n;
#pragma unroll
            for (int dst = 0; dst < 8; ++dst)
              if (dst < a.tp) st_relaxed_sys_u32(a.peer_data[dst] + off, word);
          }
          if (t.ytag) st_relaxed_sys_u32(t.ytag + (size_t)send_par * t.N + n, word);
        }
      }
    }
  }
  cp_async_wait<0>();
}

// ---------------------------------------------------------------------------------------------------------
// Persistent CTAs: every CTA slot of every SM (measured on the B200: the kernel is bound per SM, so filling every slot beats
// fewer, equally loaded CTAs), or one CTA per tile when there are fewer tiles.
template <typename T, int NBITS, int GS, int MT>
static int launch_sk(SKArgs& a, cudaStream_t st) {
  using C = SKCfg<T, NBITS, GS, MT>;
  constexpr auto k = linear_small_kernel<T, NBITS, GS, MT>;
  static int grids[kMaxDevices] = {};
  int& grid = grids[cur_device()];
  if (!grid) {
    const int rc = reserve_smem<k>(C::SMEM);
    if (rc) return rc;
    int occ = 0;
    const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, 256, C::SMEM);
    HQQ_REQUIRE(e == cudaSuccess && occ > 0, HQQ_E_CUDA, "hqq_b200_linear_fwd: occupancy query failed: %s", cudaGetErrorString(e));
    if (occ > 2) occ = 2;
    grid = sm_count() * occ;
  }
  return launch_pdl("hqq_b200_linear_fwd/small", k, dim3((unsigned)(a.total_tiles < grid ? a.total_tiles : grid)), dim3(256), C::SMEM, st,
                    pdl_enabled(), a);
}

template <typename T, int NBITS, int GS, int ST, int MC, int MR = 0>
static int launch_d1(SKArgs& a, cudaStream_t st) {
  using C = D1Cfg<T, NBITS, GS, ST, MR>;
  constexpr auto k = linear_decode1_kernel<T, NBITS, GS, ST, MC, MR>;
  const int smem = C::smem(a.K);
  const int rc = reserve_smem<k>(smem);
  if (rc) return rc;
  int per_sm = MC;
  while (per_sm > 1 && (smem + 1024) * per_sm > 227 * 1024) --per_sm;
  const int grid = sm_count() * per_sm;
  return launch_pdl("hqq_b200_linear_fwd/decode1", k, dim3((unsigned)(a.total_tiles < grid ? a.total_tiles : grid)), dim3(256), smem, st,
                    pdl_enabled(), a);
}

static bool d1_enabled() {
  HQQ_ENV_KNOB(on, ([] { const char* e = getenv("HQQ_B200_DECODE1"); return (e && e[0] == '0') ? 0 : 1; })());
  return on == 1;
}

template <typename T, int NBITS, int GS>
static int sk_mt(SKArgs& a, cudaStream_t st) {
  if (a.M == 1 && a.K <= 16384 && d1_enabled()) {
    if (NBITS == 8) return launch_d1<T, NBITS, GS, 2, 2>(a, st);
    // scale/zero ride the cp.async ring at the weights' distance (MR = 1) whenever the ring's aligned 16-byte copies are legal;
    // measured on the B200 (round 2, profiles/r2_variant_sweep.log): 1.70 ms per token against 1.91 ms with register loads one
    // unit ahead, bit-identical outputs.  evict-first hints, a third CTA per SM, L2 prefetch under the dependency wait and
    // cross-launch weight prefetch were measured in the same run, were not faster, and are gone.
    if constexpr (GS == 64 && NBITS != 8) {
      if (a.K % 512 == 0) {
        bool ok = true;  // the ring copies aligned 16-byte blocks: every group row must start on one
        for (int i = 0; i < a.nprob; ++i) ok = ok && aligned(a.p[i].scale, 16) && aligned(a.p[i].zero, 16);
        if (ok) return launch_d1<T, NBITS, GS, 4, 2, 1>(a, st);
      }
    }
    return launch_d1<T, NBITS, GS, 4, 2>(a, st);
  }
  if (a.M <= 8) return launch_sk<T, NBITS, GS, 1>(a, st);
  if (a.M <= 16) return launch_sk<T, NBITS, GS, 2>(a, st);
  return launch_sk<T, NBITS, GS, 4>(a, st);
}

template <typename T, int NBITS>
static int sk_gs(SKArgs& a, int gs, cudaStream_t st) {
  switch (gs) {
    case 64: return sk_mt<T, NBITS, 64>(a, st);
    case 128: return sk_mt<T, NBITS, 128>(a, st);
  }
  return HQQ_E_UNSUPPORTED;
}

template <typename T>
static int sk_bits(SKArgs& a, int gs, int nbits, cudaStream_t st) {
  switch (nbits) {
    case 8:
      if constexpr (std::is_same<T, __half>::value) return sk_gs<T, 8>(a, gs, st);
      else return HQQ_E_UNSUPPORTED;  // 8-bit levels need the fp16 lanes
    case 4: return sk_gs<T, 4>(a, gs, st);
    case 2: return sk_gs<T, 2>(a, gs, st);
    case 1: return sk_gs<T, 1>(a, gs, st);
  }
  return HQQ_E_UNSUPPORTED;
}

bool small_route_ok(int64_t M, int64_t N, int64_t K, int gs, int nbits, int axis, int dtype) {
  if (axis != 1) return false;
  if (dtype != HQQ_F16 && dtype != HQQ_BF16) return false;
  if (!(nbits == 8 || nbits == 4 || nbits == 2 || nbits == 1)) return false;
  if (nbits == 8 && dtype == HQQ_BF16) return false;  // 8-bit levels do not fit a bf16 mantissa trick
  if (!(gs == 64 || gs == 128)) return false;         // a 64-k MMA step must not straddle groups; meta is staged 4/8 bytes at a time
  if (M < 1 || M > 32) return false;
  if (K % 256 != 0 || K % gs != 0) return false;      // 256-k units; groups never straddle a row
  if (N % (8 / nbits) != 0) return false;
  if (N > (1 << 28) || K > (1 << 28)) return false;
  return true;
}

size_t small_workspace_bytes(int64_t) { return 0; }  // split-K partials meet in shared memory

bool small_xop_ok(int64_t M, int64_t K) { return M == 1 && K <= 16384 && d1_enabled(); }

int linear_small_multi(const void* x, int nprob, const void* const* Wq, const void* const* scale, const void* const* zero,
                       const void* const* bias, void* const* y, const int64_t* N, int64_t M, int64_t K, int gs, int nbits, int dtype,
                       void* ws, size_t ws_bytes, cudaStream_t st, int xop, const void* x2, const void* xw, void* h_out, float eps,
                       const TpExchange* tpx) {
  HQQ_REQUIRE(nprob >= 1 && nprob <= kMaxProb, HQQ_E_INVALID, "hqq_b200_linear_fwd_multi: 1..%d matrices per launch (got %d)", kMaxProb, nprob);
  HQQ_REQUIRE(aligned(x, 16), HQQ_E_INVALID, "hqq_b200_linear_fwd: x must be 16-byte aligned");
  (void)ws; (void)ws_bytes;
  const int F = 8 / nbits, P = 16 / F;
  SKArgs a;
  a.nprob = nprob; a.x = x; a.M = (int)M; a.K = (int)K; a.Gk = (int)(K / gs); a.KB = (int)(K / 256);
  const int yop = xop >> 4;  // HQQ_YOP_* travel in the high bits of x_op
  xop &= 15;
  a.xop = xop; a.yop = yop; a.x2 = x2; a.xw = xw; a.h_out = h_out; a.eps = eps;
  if (yop) {
    HQQ_REQUIRE(yop == 1, HQQ_E_INVALID, "hqq_b200_decode_linear_fwd: unknown epilogue %d", yop);
    HQQ_REQUIRE(nprob == 2 && N[0] == N[1], HQQ_E_INVALID, "hqq_b200_decode_linear_fwd: the silu*mul epilogue pairs exactly two matrices of equal N");
    if (!(small_xop_ok(M, K) && nbits < 8) || (tpx && (tpx->peer_data || tpx->y_tagged))) {
      set_error("hqq_b200_decode_linear_fwd: the silu*mul epilogue needs the M == 1 kernel, nbits < 8 and plain outputs");
      return HQQ_E_UNSUPPORTED;
    }
  }
  a.tp = 1; a.rank = 0; a.red_data = nullptr; a.xtag = nullptr; a.x2tag = nullptr; a.step_ctr = nullptr; a.x_index = 0; a.x_per_step = 1;
  for (int i = 0; i < 8; ++i) a.peer_data[i] = nullptr;
  if (tpx && !tpx->step_ctr) tpx = nullptr;
  if (tpx) {
    HQQ_REQUIRE(small_xop_ok(M, K) && nprob >= 1, HQQ_E_UNSUPPORTED, "hqq_b200_decode_linear_fwd_desc: needs the M == 1 kernel");
    HQQ_REQUIRE(tpx->tp >= 1 && tpx->tp <= 8 && tpx->rank >= 0 && tpx->rank < tpx->tp && tpx->step_ctr && tpx->x_per_step > 0, HQQ_E_INVALID,
                "hqq_b200_decode_linear_fwd_desc: bad tp/rank/step counter");
    a.tp = tpx->tp; a.rank = tpx->rank; a.step_ctr = tpx->step_ctr; a.x_index = tpx->x_index; a.x_per_step = tpx->x_per_step;
    if (tpx->peer_data) {
      HQQ_REQUIRE(nprob == 1, HQQ_E_INVALID, "hqq_b200_decode_linear_fwd_desc: the scatter side takes exactly one matrix");
      for (int i = 0; i < tpx->tp; ++i) a.peer_data[i] = reinterpret_cast<uint32_t*>(tpx->peer_data[i]);
    }
    if (tpx->red_data) {
      HQQ_REQUIRE(xop == 1, HQQ_E_INVALID, "hqq_b200_decode_linear_fwd_desc: a reduced delta needs x_op 1");
      a.red_data = reinterpret_cast<const uint32_t*>(tpx->red_data);
    }
    if (tpx->x_tagged || tpx->x2_tagged) {
      HQQ_REQUIRE(xop == 2 && tpx->x_tagged && tpx->x2_tagged, HQQ_E_INVALID, "hqq_b200_decode_linear_fwd_desc: tagged activations need x_op 2 and both operands");
      a.xtag = reinterpret_cast<const uint32_t*>(tpx->x_tagged); a.x2tag = reinterpret_cast<const uint32_t*>(tpx->x2_tagged);
    }
  }
  int tiles = 0;
  for (int i = 0; i < kMaxProb; ++i) {
    const int j = i < nprob ? i : 0;
    HQQ_REQUIRE(Wq[j] && scale[j] && zero[j] && y[j], HQQ_E_INVALID, "hqq_b200_linear_fwd: null pointer");
    HQQ_REQUIRE(aligned(Wq[j], 16) && aligned(scale[j], 8) && aligned(zero[j], 8), HQQ_E_INVALID,
                "hqq_b200_linear_fwd: W_q must be 16-byte and scale/zero 8-byte aligned");
    a.p[i].Wq = (const uint8_t*)Wq[j]; a.p[i].scale = scale[j]; a.p[i].zero = zero[j]; a.p[i].bias = bias ? bias[j] : nullptr;
    a.p[i].y = y[j]; a.p[i].ytag = (tpx && tpx->y_tagged) ? reinterpret_cast<uint32_t*>(tpx->y_tagged[j]) : nullptr; a.p[i].N = (int)N[j]; a.p[i].step = (int)(N[j] / F); a.p[i].tile0 = tiles;
    if (i < nprob) tiles += (int)cdiv(a.p[i].step, P);
  }
  a.total_tiles = yop ? (int)cdiv(a.p[0].step, P / 2) : tiles;
  if (dtype == HQQ_F16) return sk_bits<__half>(a, gs, nbits, st);
  return sk_bits<__nv_bfloat16>(a, gs, nbits, st);
}

}  // namespace hqq
