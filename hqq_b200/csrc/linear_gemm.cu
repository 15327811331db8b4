// HQQLinear.forward for M >= 33 (prefill / batched decode): fused unpack -> group-dequant -> tcgen05 GEMM.
//
//   y[M,N] = x[M,K] @ dequantize(W_q)^T (+bias)          reference: hqq/core/quantize.py:184-199, 880-898
//
// ONE persistent kernel, one CTA per SM, 14 warps with fixed roles; a CTA walks a static list of output tiles
// [128 weight rows] x [UN tokens] (UN = 256, or 128 for the ragged part of the schedule, see `Sched`):
//   warp 0       TMA producer: the activation tile [UN tokens x 64 k] of every k-block (cp.async.bulk.tensor.2d, 128B swizzle,
//                out-of-range tokens zero-filled by the hardware) into a 4-stage shared-memory ring = B operand (N = UN)
//   warps 2..9   dequant: stream the packed bytes of the weight tile from HBM/L2 (the reference's slab layout, bitpack.py: 128/F
//                packed rows x F slabs = 128 output rows), expand them in registers with the reference's two roundings
//                W_r = fl(fl(q - z) * s) (bit-identical to Quantizer.dequantize) and store K-major SWIZZLE_128B fp16/bf16 rows
//                into the ring = A operand (M = 128).  The dequantised matrix never exists in HBM.
//   warp 1       one elected thread issues tcgen05.mma (4 per 64-k stage) into one of TWO fp32 accumulators in TMEM
//                (2 x 256 columns = all 512); tcgen05.commit frees the stage / publishes the accumulator
//   warps 10..13 epilogue: tcgen05.ld (lane = weight row, column = token) -> bias -> y, for tile i while the other roles are
//                already in the main loop of tile i+1 (the rings never drain between tiles)
// Round 1 launched one CTA per tile: 512 tiles on 148 SMs = 3.46 -> 4 waves, prologue/epilogue exposed per tile, tensor pipe
// 61 % active.  tools/ummabench.cu (round 2) measured the same MMA stream alone at 1.35-1.40 PFLOP/s on this part, with A from
// TMEM (tcgen05.mma "ts" form) no faster than from shared memory -- so A stays in shared memory and the TMEM goes to the
// second accumulator.
// sm_100a only: tcgen05 / TMEM / TMA, no mma.sync fallback.
#include <stdlib.h>
#include <cuda.h>  // CUtensorMap types only; the encode entry point is resolved through the runtime (no -lcuda)

#include "device.cuh"

namespace hqq {

namespace gemm {

constexpr int kStages = 4;
constexpr int kBlockK = 64;          // k elements per stage = one 128-byte swizzle row
constexpr int kTileRows = 128;       // weight rows per CTA = UMMA M
constexpr int kDequantThreads = 256;
constexpr int kEpilogueThreads = 128;
constexpr int kThreads = 64 + kDequantThreads + kEpilogueThreads;  // warp 0: TMA + TMEM alloc, warp 1: MMA issue, 2..9: dequant, 10..13: epilogue
constexpr int kUN = 256;             // tokens per full tile = UMMA N; half tiles use 128
constexpr int kTmemCols = 512;       // two accumulators of kUN fp32 columns

// Static tile schedule.  Items 0 .. i_split-1 are full tiles: item j = (row tile j / n_tok, token tile j % n_tok), 256 tokens
// (128 when no more than 128 tokens remain).  The last r_split full tiles are cut into two 128-token halves each (items
// i_split ..): with T full tiles on P persistent CTAs the last round holds T % P tiles; as halves they spread over twice as
// many CTAs and the round costs half a tile (512 tiles on 148 SMs: 3.5 tile-times instead of 4).  CTA b owns items b, b + P, ...
struct Sched {
  int n_tok;     // token tiles of 256
  int i_split;   // first item that is a half tile
  int n_items;
  // Few tiles (M <= 512 on most matrices): `ksplit` CTAs share a tile, each accumulating a contiguous run of k-blocks and writing
  // its fp32 partial tile to the caller's workspace; splitk_reduce_kernel adds the partials in slice order (deterministic) and
  // rounds.  Without it a [128 x K] tile is ONE serial stream per CTA with four stages in flight: ~960 cycles per 64-k block
  // (first-touch DRAM latency), 32 CTAs busy out of 148 -- 32 us for 4096 x 4096 at any M <= 512 (profiles/r2_midm_options.log).
  int ksplit;    // 1 = off; items are then (tile, slice), slice fastest
  int n_row;     // row tiles
};

struct Args {
  const uint8_t* Wq;
  const void* scale;
  const void* zero;
  const void* bias;
  void* y;
  float* ws;     // ksplit > 1: [ksplit][n_row * n_tok][256 tokens][128 rows] fp32 partials
  int M, N, K;
  int step;  // packed rows = N / F
  int Gk;    // groups per row = K / GS
  Sched sched;
};

struct Item { int tile_n, m0, un, kb0, kb1, slice, tile; bool valid; };
__host__ __device__ __forceinline__ Item decode_item(const Args& a, int j) {
  Item it;
  const int num_kb = (a.K + kBlockK - 1) / kBlockK;
  it.kb0 = 0; it.kb1 = num_kb; it.slice = 0;
  int base = j, half = -1;
  if (a.sched.ksplit > 1) {
    it.slice = j % a.sched.ksplit;
    base = j / a.sched.ksplit;
    const int quads = num_kb >> 2, per = (quads + a.sched.ksplit - 1) / a.sched.ksplit;
    it.kb0 = it.slice * per * 4;
    it.kb1 = ((it.slice + 1) * per < quads ? (it.slice + 1) * per : quads) * 4;
  } else if (j >= a.sched.i_split) {
    base = a.sched.i_split + ((j - a.sched.i_split) >> 1); half = (j - a.sched.i_split) & 1;
  }
  it.tile = base;
  it.tile_n = base / a.sched.n_tok;
  it.m0 = (base % a.sched.n_tok) * kUN;
  it.un = (a.M - it.m0 > 128) ? 256 : 128;
  if (half >= 0) { it.m0 += half * 128; it.un = 128; }
  it.valid = it.m0 < a.M && it.kb0 < it.kb1;
  return it;
}

// ---- PTX wrappers -------------------------------------------------------------------------------------------------
#ifdef HQQ_EMU
// CPU emulation (tests/emu): the same entry points, backed by a functional model of mbarrier / TMA / tcgen05 / TMEM
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return ::emu::smem_offset(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) { ::emu::mbar_init(bar, count); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) { ::emu::mbar_arrive(bar); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) { ::emu::mbar_expect_tx(bar, bytes); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) { ::emu::mbar_wait(bar, parity); }
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) { ::emu::tma_load_2d(smem_dst, map, bar, c0, c1); }
__device__ __forceinline__ void fence_async_smem() {}
__device__ __forceinline__ void fence_barrier_init() {}
__device__ __forceinline__ void tc_fence_before() {}
__device__ __forceinline__ void tc_fence_after() {}
__device__ __forceinline__ void tc_commit(uint64_t* bar) { ::emu::tc_commit(bar); }  // arrives once the MMAs issued before it have executed
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  ::emu::umma_f16(tmem_d, adesc, bdesc, idesc, accumulate);
}
template <int NCOLS> __device__ __forceinline__ void tmem_alloc(uint32_t* dst_in_smem) { ::emu::tmem_alloc(dst_in_smem, NCOLS); }
template <int NCOLS> __device__ __forceinline__ void tmem_dealloc(uint32_t) {}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) { ::emu::tmem_ld32(taddr, v); }
#define HQQ_STS_V4(addr, a, b, c, d) ::emu::sts(addr, a, b, c, d)
#define HQQ_STS_V2(addr, a, b) ::emu::sts(addr, a, b)
#define HQQ_PREFETCH_TENSORMAP(p) ((void)(p))
#define HQQ_NAMED_BAR_SYNC(id, n) ::emu::named_barrier(id, n)
#else
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_in_smem) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_in_smem)), "n"(NCOLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
        "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
        "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
        "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

#define HQQ_STS_V4(addr, a, b, c, d) asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory")
#define HQQ_STS_V2(addr, a, b) asm volatile("st.shared.v2.b32 [%0], {%1,%2};" ::"r"(addr), "r"(a), "r"(b) : "memory")
#define HQQ_PREFETCH_TENSORMAP(p) asm volatile("prefetch.tensormap [%0];" ::"l"(p) : "memory")
#define HQQ_NAMED_BAR_SYNC(id, n) asm volatile("bar.sync %0, %1;" ::"n"(id), "n"(n) : "memory")
#endif  // HQQ_EMU

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 in bits [0,14),
// leading byte offset (unused for swizzled K-major, 1) in [16,30), stride byte offset = 1024 B between 8-row groups in
// [32,46), descriptor version 1 (Blackwell) in [46,48), layout type 2 = SWIZZLE_128B in [61,64).
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// Instruction descriptor for kind::f16 (cute::UMMA::InstrDescriptor): D = F32, A/B = F16 or BF16, both K-major, M = 128, N = UN.
template <typename T>
__device__ __forceinline__ uint32_t make_idesc(int UN) {
  const uint32_t fmt = std::is_same<T, __nv_bfloat16>::value ? 1u : 0u;
  uint32_t d = 0;
  d |= 1u << 4;                      // c_format = F32
  d |= fmt << 7;                     // a_format
  d |= fmt << 10;                    // b_format
  d |= (uint32_t)(UN >> 3) << 17;    // n_dim
  d |= (uint32_t)(128 >> 4) << 24;   // m_dim
  return d;
}

// ---- level -> T with the reference's roundings -------------------------------------------------------------------
// Four k-adjacent levels (one per byte of `t`, already masked to the field) -> two packed T2
//   {fl(fl(q0 - z) * s), fl(fl(q1 - z) * s)}, {.. q2, q3 ..}
template <typename T> struct Pair;
template <> struct Pair<__half> {
  using T2 = __half2;
  __device__ __forceinline__ static void deq4(uint32_t t, __half2 z2, __half2 s2, uint32_t& lo, uint32_t& hi) {
    // byte | 0x6400 == 1024 + q exactly (one PRMT per pair); subtracting 1024 is exact, so (q - z) and (.. * s) round
    // exactly like the reference's two steps
    const __half2 k1024 = __half2half2(__ushort_as_half((unsigned short)0x6400));
    uint32_t a = prmt(t, 0x64646464u, 0x4140u), b = prmt(t, 0x64646464u, 0x4342u);
    __half2 ha = __hmul2(__hsub2(__hsub2(*reinterpret_cast<__half2*>(&a), k1024), z2), s2);
    __half2 hb = __hmul2(__hsub2(__hsub2(*reinterpret_cast<__half2*>(&b), k1024), z2), s2);
    lo = *reinterpret_cast<uint32_t*>(&ha);
    hi = *reinterpret_cast<uint32_t*>(&hb);
  }
  __device__ __forceinline__ static __half2 bcast(__half v) { return __half2half2(v); }
};
template <> struct Pair<__nv_bfloat16> {
  using T2 = __nv_bfloat162;
  __device__ __forceinline__ static void deq4(uint32_t t, __nv_bfloat162 z2, __nv_bfloat162 s2, uint32_t& lo, uint32_t& hi) {
    // levels < 256 are exact in bf16 (8 significant bits); convert through the exact float 2^23 + q trick
    const float f0 = __uint_as_float(0x4B000000u | (t & 0xFFu)) - 8388608.0f, f1 = __uint_as_float(0x4B000000u | ((t >> 8) & 0xFFu)) - 8388608.0f;
    const float f2 = __uint_as_float(0x4B000000u | ((t >> 16) & 0xFFu)) - 8388608.0f, f3 = __uint_as_float(0x4B000000u | (t >> 24)) - 8388608.0f;
    __nv_bfloat162 ha = __hmul2(__hsub2(__floats2bfloat162_rn(f0, f1), z2), s2);
    __nv_bfloat162 hb = __hmul2(__hsub2(__floats2bfloat162_rn(f2, f3), z2), s2);
    lo = *reinterpret_cast<uint32_t*>(&ha);
    hi = *reinterpret_cast<uint32_t*>(&hb);
  }
  __device__ __forceinline__ static __nv_bfloat162 bcast(__nv_bfloat16 v) { return __bfloat162bfloat162(v); }
};


struct Smem {
  static constexpr int A_STAGE = kTileRows * 128;  // 128 rows x 128 B
  static constexpr int B_STAGE = kUN * 128;
  static constexpr int BYTES = kStages * (A_STAGE + B_STAGE) + 1024 /*align*/ + 256 /*barriers*/;
};

// NBITS = 16 ("dense"): the A operand is an ordinary [N, K] fp16/bf16 matrix fetched by TMA like B -- the dequant warps idle.  It is
// the second half of the routes no fused expansion exists for (3-bit's 10-field int32 slabs, axis = 0 groups, other group sizes,
// the backward pass): our dequantize kernel writes W_r once, this kernel multiplies (hqq_b200_linear_fwd route 4).
template <typename T, int NBITS, int GS>
__global__ void __launch_bounds__(kThreads, 1) linear_gemm_kernel(const __grid_constant__ CUtensorMap xmap256,
                                                                  const __grid_constant__ CUtensorMap xmap128,
                                                                  const __grid_constant__ CUtensorMap amap, const Args a) {
  constexpr bool DENSE = NBITS == 16;
  constexpr int F = DENSE ? 1 : 8 / NBITS;  // slabs per byte
  constexpr int PR = kTileRows / F;        // packed rows per tile
  constexpr int BPT = DENSE ? 32 : 64 * PR / kDequantThreads;  // packed bytes per dequant thread and k-block (32 / F)
  static_assert(BPT >= 4, "a dequant thread expands at least four packed bytes per k-block");
  constexpr int TPR = 64 / BPT;            // dequant threads per packed row
  constexpr uint32_t MASK = (1u << NBITS) - 1u;
  using S = Smem;
  using P2 = Pair<T>;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);  // SWIZZLE_128B atoms
  uint8_t* sA = smem;
  uint8_t* sB = smem + kStages * S::A_STAGE;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * (S::A_STAGE + S::B_STAGE));
  uint64_t* full_a = bars;                 // [kStages] dequant warps -> MMA (one arrival per warp)
  uint64_t* full_b = bars + kStages;       // [kStages] TMA -> MMA (1 arrival + tx bytes)
  uint64_t* empty = bars + 2 * kStages;    // [kStages] MMA (tcgen05.commit) -> both producers
  uint64_t* acc_full = bars + 3 * kStages;       // [2] MMA (tcgen05.commit) -> epilogue
  uint64_t* acc_empty = bars + 3 * kStages + 2;  // [2] epilogue (one arrival per warp) -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_kb = (a.K + kBlockK - 1) / kBlockK;  // quantised routes: K % 256 == 0; dense: the TMA zero-fills a ragged last block
  const int n_items = a.sched.n_items;

  if (warp == 0) {
    if (lane == 0) {
      for (int s = 0; s < kStages; ++s) { mbar_init(&full_a[s], kDequantThreads / 32); mbar_init(&full_b[s], 1); mbar_init(&empty[s], 1); }
      for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], kEpilogueThreads / 32); }
      fence_barrier_init();
      HQQ_PREFETCH_TENSORMAP(&xmap256);
      HQQ_PREFETCH_TENSORMAP(&xmap128);
      if constexpr (DENSE) HQQ_PREFETCH_TENSORMAP(&amap);
    }
    __syncwarp();
    tmem_alloc<kTmemCols>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Programmatic dependent launch, both sides.  Our dependents (the split-K second pass; the next forward of a chain of layers) may
  // become resident as our CTAs retire -- they block in griddepcontrol.wait until this grid has completed and flushed, so only
  // their launch latency and prologue move under our tail.  As a dependent ourselves, the one thing we read that a PDL-aware
  // predecessor may still be writing is the activation x (and, dense mode, W written by the dequantize kernel): the TMA producer
  // waits before its first load, and nothing is written (y, split-K partials) before an accumulator fed by those loads is full.
  // Packed weights, scale, zero and bias are never produced by a kernel that releases its dependents early.
  if (threadIdx.x == 0) pdl_launch_dependents();

  if (warp == 0) {
    // ================= TMA producer: activation tiles =================
    if (lane == 0) {
      uint32_t it = 0;  // k-blocks issued so far (ring position)
      pdl_wait();
      for (int j = blockIdx.x; j < n_items; j += gridDim.x) {
        const Item im = decode_item(a, j);
        if (!im.valid) continue;
        for (int kb = im.kb0; kb < im.kb1; ++kb, ++it) {
          const int s = it % kStages;
          mbar_wait(&empty[s], ((it / kStages) & 1) ^ 1);
          constexpr uint32_t A_TX = DENSE ? S::A_STAGE : 0;  // dense: the weight tile rides the same barrier
          if (im.un == kUN) {
            mbar_expect_tx(&full_b[s], S::B_STAGE + A_TX);
            tma_load_2d(sB + s * S::B_STAGE, &xmap256, &full_b[s], kb * kBlockK, im.m0);
          } else {
            mbar_expect_tx(&full_b[s], S::B_STAGE / 2 + A_TX);
            tma_load_2d(sB + s * S::B_STAGE, &xmap128, &full_b[s], kb * kBlockK, im.m0);
          }
          if constexpr (DENSE) tma_load_2d(sA + s * S::A_STAGE, &amap, &full_b[s], kb * kBlockK, im.tile_n * kTileRows);
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (one elected thread) =================
    uint32_t it = 0, q = 0;  // k-blocks consumed, tiles started
    for (int j = blockIdx.x; j < n_items; j += gridDim.x) {
      const Item im = decode_item(a, j);
      if (!im.valid) continue;
      const uint32_t buf = q & 1, use = q >> 1;
      mbar_wait(&acc_empty[buf], (use & 1) ^ 1);  // the epilogue has drained this accumulator (passes at once the first time)
      tc_fence_after();
      const uint32_t idesc = make_idesc<T>(im.un);
      const uint32_t tmem_d = tmem_base + buf * kUN;
      for (int kb = im.kb0; kb < im.kb1; ++kb, ++it) {
        const int s = it % kStages;
        const uint32_t ph = (it / kStages) & 1;
        if constexpr (!DENSE) mbar_wait(&full_a[s], ph);
        mbar_wait(&full_b[s], ph);
        tc_fence_after();
        if (lane == 0) {
          const uint64_t adesc = make_desc_sw128(smem_u32(sA + s * S::A_STAGE));
          const uint64_t bdesc = make_desc_sw128(smem_u32(sB + s * S::B_STAGE));
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k)  // UMMA_K = 16: advance 32 bytes inside the 128-byte swizzle row
            tc_mma_f16(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, ((kb - im.kb0) | k) != 0);
          tc_commit(&empty[s]);                              // frees the stage when these MMAs have read it
          if (kb == im.kb1 - 1) tc_commit(&acc_full[buf]);   // accumulator complete
        }
        __syncwarp();
      }
      ++q;
    }
  } else if (warp < 2 + kDequantThreads / 32) {
    if constexpr (!DENSE) {
    // ================= dequant warps: packed bytes -> swizzled fp16/bf16 A tile =================
    static_assert(kStages == 4, "the dequant loop is unrolled over the 4 ring stages");
    const int td = threadIdx.x - 64;
    const int pr = td / TPR, c = td % TPR;
    constexpr int GPQ = 256 / GS;  // quantisation groups per 4 k-blocks (4 or 2): one vector load per slab and array
    uint32_t soff[F];              // shared-memory offsets are tile invariant
#pragma unroll
    for (int f = 0; f < F; ++f) {
      const int row = f * PR + pr;
      // K-major SWIZZLE_128B: 16-byte chunk index XOR (row % 8) inside each 8-row x 128-byte atom
      if constexpr (BPT >= 8) soff[f] = (uint32_t)(row * 128) | ((uint32_t)(row & 7) << 16);  // chunk applied below
      else soff[f] = (uint32_t)(row * 128 + (((c >> 1) ^ (row & 7)) << 4) + (c & 1) * 8);
    }
    const uint32_t sA_u32 = smem_u32(sA);
    const uint8_t* wptr = nullptr;
    const T* sptr[F];
    const T* zptr[F];
    auto tile_ptrs = [&](const Item& im) {  // this thread's packed row / meta rows at the first k-block of an item
      const int prow0 = im.tile_n * PR;
      const bool row_ok = (prow0 + pr) < a.step;  // rows past the ragged edge re-read row 0 (always mapped); never stored
      wptr = a.Wq + (long long)(row_ok ? prow0 + pr : 0) * a.K + c * BPT + (long long)im.kb0 * kBlockK;
#pragma unroll
      for (int f = 0; f < F; ++f) {
        const long long mrow = (long long)(row_ok ? f * a.step + prow0 + pr : 0) * a.Gk + (im.kb0 >> 2) * GPQ;
        sptr[f] = reinterpret_cast<const T*>(a.scale) + mrow;
        zptr[f] = reinterpret_cast<const T*>(a.zero) + mrow;
      }
    };
    auto next_valid = [&](int j) {  // first valid item of this CTA at or after j (n_items if none)
      while (j < n_items && !decode_item(a, j).valid) j += gridDim.x;
      return j < n_items ? j : n_items;
    };
    // Packed bytes and scale/zero for the NEXT four k-blocks sit in registers while the current four are expanded -- across tile
    // boundaries too: their HBM/L2 latency stays off the critical path of the 64-k stages.
    uint32_t wbuf[4][BPT / 4];
    Vec<T, GPQ> sv[F], zv[F];
    auto load_w = [&](const uint8_t* p, uint32_t (&w)[BPT / 4]) {
      if constexpr (BPT == 32) { const uint4 v0 = ldg_stream_v4(p), v1 = ldg_stream_v4(p + 16); w[0] = v0.x; w[1] = v0.y; w[2] = v0.z; w[3] = v0.w; w[4] = v1.x; w[5] = v1.y; w[6] = v1.z; w[7] = v1.w; }
      else if constexpr (BPT == 16) { const uint4 v = ldg_stream_v4(p); w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w; }
      else if constexpr (BPT == 8) { const uint2 v = __ldg(reinterpret_cast<const uint2*>(p)); w[0] = v.x; w[1] = v.y; }
      else { w[0] = __ldg(reinterpret_cast<const uint32_t*>(p)); }
    };
    auto load_quad = [&]() {  // the four k-blocks starting at wptr, and their groups
#pragma unroll
      for (int d = 0; d < 4; ++d) load_w(wptr + d * kBlockK, wbuf[d]);
#pragma unroll
      for (int f = 0; f < F; ++f) { sv[f] = *reinterpret_cast<const Vec<T, GPQ>*>(sptr[f]); zv[f] = *reinterpret_cast<const Vec<T, GPQ>*>(zptr[f]); }
    };
    // K % 256 == 0 (checked by the router) and k-slices are whole quads: every item starts at ring stage 0
    int j = next_valid((int)blockIdx.x);
    if (j < n_items) { tile_ptrs(decode_item(a, j)); load_quad(); }
    uint32_t gq = 0;  // quads done so far (ring parity)
    while (j < n_items) {
      const int jn = next_valid(j + (int)gridDim.x);
      const Item cur = decode_item(a, j);
      const int num_quads = (cur.kb1 - cur.kb0) >> 2;
      for (int q = 0; q < num_quads; ++q, ++gq) {
        uint32_t wq[4][BPT / 4];
        typename P2::T2 s2[4][F], z2[4][F];
#pragma unroll
        for (int d = 0; d < 4; ++d) {
#pragma unroll
          for (int i = 0; i < BPT / 4; ++i) wq[d][i] = wbuf[d][i];
#pragma unroll
          for (int f = 0; f < F; ++f) { s2[d][f] = P2::bcast(sv[f].v[(d * kBlockK) / GS]); z2[d][f] = P2::bcast(zv[f].v[(d * kBlockK) / GS]); }
        }
        if (q + 1 < num_quads) {
          wptr += 4 * kBlockK;
#pragma unroll
          for (int f = 0; f < F; ++f) { sptr[f] += GPQ; zptr[f] += GPQ; }
          // the register prefetch reaches one quad ahead, about 1 us of main loop at small M -- less than a DRAM round trip under
          // load when a weight tile is read for the first time (M <= 512: every tile is); pull the line this thread will load
          // three quads from now into L2 (a packed row has 256 bytes = two lines per quad: even / odd threads of the row take one each)
          if (q + 4 < num_quads) prefetch_l2(wptr + 3 * 4 * kBlockK + (c & 1) * 128);
          load_quad();
        } else if (jn < n_items) {
          tile_ptrs(decode_item(a, jn));
          load_quad();
        }
        const uint32_t parity = (gq & 1u) ^ 1u;
#pragma unroll
        for (int d = 0; d < 4; ++d) {  // stage index == d because the ring has exactly four stages
          mbar_wait(&empty[d], parity);
          const uint32_t stage = sA_u32 + d * S::A_STAGE;
#pragma unroll
          for (int f = 0; f < F; ++f) {
            const int sh = 8 - NBITS * (f + 1);
            uint32_t out[BPT / 2];  // BPT levels -> BPT/2 packed pairs
#pragma unroll
            for (int i = 0; i < BPT / 4; ++i) {
              const uint32_t t = (wq[d][i] >> sh) & (MASK * 0x01010101u);
              P2::deq4(t, z2[d][f], s2[d][f], out[2 * i], out[2 * i + 1]);
            }
            if constexpr (BPT >= 8) {
              const uint32_t rowbase = stage + (soff[f] & 0xFFFFu), rx = soff[f] >> 16;
#pragma unroll
              for (int ch = 0; ch < BPT / 8; ++ch) {
                const uint32_t addr = rowbase + (((uint32_t)(c * (BPT / 8) + ch) ^ rx) << 4);
                HQQ_STS_V4(addr, out[4 * ch], out[4 * ch + 1], out[4 * ch + 2], out[4 * ch + 3]);
              }
            } else {  // BPT == 4: half a chunk
              HQQ_STS_V2(stage + soff[f], out[0], out[1]);
            }
          }
          fence_async_smem();  // make the generic-proxy stores visible to the tensor core (async proxy)
          __syncwarp();
          if (lane == 0) mbar_arrive(&full_a[d]);  // one arrival per warp: every lane has fenced its stores before the syncwarp
        }
      }
      j = jn;
    }
    }  // !DENSE
  } else {
    // ================= epilogue warps: TMEM -> registers -> y, one tile behind the main loop =================
    const int quarter = warp & 3;                 // TMEM lanes this warp may touch: 32*quarter .. +31
    const int t = quarter * 32 + lane;            // tile row = weight row inside the tile
    const int tf = t / PR, tp = t % PR;
    T* y = reinterpret_cast<T*>(a.y);
    const T* bias = reinterpret_cast<const T*>(a.bias);
    const bool has_bias = bias != nullptr;
    uint32_t q = 0;
    for (int j = blockIdx.x; j < n_items; j += gridDim.x) {
      const Item im = decode_item(a, j);
      if (!im.valid) continue;
      const uint32_t buf = q & 1, use = q >> 1;
      const int prow0 = im.tile_n * PR;
      const bool n_ok = (prow0 + tp) < a.step;
      const int n = tf * a.step + prow0 + tp;
      T bn = from_f32<T>(0.0f);
      if (has_bias && n_ok) bn = bias[n];
      mbar_wait(&acc_full[buf], use & 1);
      tc_fence_after();
#pragma unroll 1
      for (int col = 0; col < im.un; col += 32) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * kUN + (uint32_t)col, v);
        if (a.sched.ksplit > 1) {
          // fp32 partial of this k-slice: [slice][tile][token][tile row] -- 32 lanes write 32 consecutive rows (128 bytes)
          float* wsp = a.ws + (((size_t)im.slice * (size_t)(a.sched.n_row * a.sched.n_tok) + (size_t)im.tile) * kUN + (size_t)col) * kTileRows + t;
#pragma unroll
          for (int jj = 0; jj < 32; ++jj)
            if (im.m0 + col + jj < a.M) wsp[(size_t)jj * kTileRows] = __uint_as_float(v[jj]);
        } else {
#pragma unroll
          for (int jj = 0; jj < 32; ++jj) {
            const int m = im.m0 + col + jj;
            if (n_ok && m < a.M) {
              T o = from_f32<T>(__uint_as_float(v[jj]));
              if (has_bias) o = __hadd(o, bn);  // out += bias: second rounding, as in the reference
              y[(long long)m * a.N + n] = o;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);  // every lane's tcgen05.ld has completed (wait::ld) before the syncwarp
      ++q;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc<kTmemCols>(tmem_base);
  }
}

// Split-K second pass: y[m][n] = round(sum over slices, in slice order) (+ bias).  A thread owns V consecutive outputs (V = 4 when
// step, N and y allow 8-byte stores, else 1): they are consecutive rows of one tile column in the workspace, so both sides are
// coalesced vector accesses.  All slices are loaded before the first add -- the loads are independent, the adds keep the order.
template <typename T, int V>
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ ws, T* __restrict__ y, const T* __restrict__ bias, int M, int N,
                                                            int step, int PR, int S, int n_row, int n_tok) {
  const long long idx = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * V;
  pdl_wait();  // launched as a programmatic dependent of the GEMM: resident early, reads only after that grid has completed
  if (idx >= (long long)M * N) return;
  const int m = (int)(idx / N), n = (int)(idx % N);
  const int f = n / step, prg = n % step;
  const int tile_n = prg / PR, t = f * PR + prg % PR;
  const int tile = tile_n * n_tok + m / kUN, col = m % kUN;
  const size_t slice_stride = (size_t)n_row * n_tok * kUN * kTileRows;
  const float* p = ws + ((size_t)tile * kUN + col) * kTileRows + t;
  float part[8][V];
#pragma unroll
  for (int sidx = 0; sidx < 8; ++sidx) {
#pragma unroll
    for (int v = 0; v < V; ++v) part[sidx][v] = 0.0f;
    if (sidx < S) {
      if constexpr (V == 4) {
        const float4 q = *reinterpret_cast<const float4*>(p + (size_t)sidx * slice_stride);
        part[sidx][0] = q.x; part[sidx][1] = q.y; part[sidx][2] = q.z; part[sidx][3] = q.w;
      } else {
        part[sidx][0] = p[(size_t)sidx * slice_stride];
      }
    }
  }
  T o[V];
#pragma unroll
  for (int v = 0; v < V; ++v) {
    float acc = 0.0f;
#pragma unroll
    for (int sidx = 0; sidx < 8; ++sidx)
      if (sidx < S) acc += part[sidx][v];
    o[v] = from_f32<T>(acc);
    if (bias) o[v] = __hadd(o[v], bias[n + v]);
  }
  if constexpr (V == 4) {
    *reinterpret_cast<uint2*>(y + idx) = *reinterpret_cast<const uint2*>(o);
  } else {
    y[idx] = o[0];
  }
}

// ---- host side ------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
#ifdef HQQ_EMU
  return &::emu::encode_tiled;
#endif
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}


// [rows, K] row-major 16-bit matrix, boxes of 64 k x `box_rows` rows, 128B swizzle, out-of-range elements read as zero
static int encode_map(CUtensorMap* xmap, const void* x, int64_t rows, int64_t K, CUtensorMapDataType dt, size_t esize, int box_rows) {
  EncodeTiledFn enc = get_encode();
  HQQ_REQUIRE(enc != nullptr, HQQ_E_CUDA, "hqq_b200_linear_fwd: cuTensorMapEncodeTiled is not available from this driver");
  const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)K * esize};
  const cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(xmap, dt, 2, const_cast<void*>(x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  HQQ_REQUIRE(r == CUDA_SUCCESS, HQQ_E_CUDA, "hqq_b200_linear_fwd: cuTensorMapEncodeTiled failed (%d)", (int)r);
  return HQQ_OK;
}

// see `Sched`: full tiles first, the last partial round as half tiles when that shortens it
// HQQ_B200_GEMM_CTAS=<n> (test hook): the number of persistent CTAs the schedule is built for instead of the SM count, so that
// small problems exercise tile-after-tile execution, both accumulators, the half-tile round and split-K (the emulator tests and
// tests/test_linear_gpu.py set it; results never depend on it beyond the split-K summation order, which they pin)
static int persistent_ctas() {
  HQQ_ENV_KNOB(cta_cap, ([] { const char* e = getenv("HQQ_B200_GEMM_CTAS"); return e ? atoi(e) : 0; })());
  return cta_cap > 0 ? cta_cap : sm_count();
}

// HQQ_B200_GEMM_KSPLIT=<n> (test / measurement hook): the largest number of k-slices the schedule may use (1 = never split)
static int ksplit_cap() {
  HQQ_ENV_KNOB(cap, ([] { const char* e = getenv("HQQ_B200_GEMM_KSPLIT"); return e ? atoi(e) : 0; })());
  return cap > 0 ? (cap > 8 ? 8 : cap) : 8;
}

// see `Sched`: few tiles -> k-slices; else full tiles first, the last partial round as half tiles when that shortens it
Sched make_sched(int64_t M, int64_t K, int64_t row_tiles, int P, bool allow_splitk) {
  Sched s;
  s.n_tok = (int)cdiv(M, kUN);
  s.n_row = (int)row_tiles;
  s.ksplit = 1;
  const int64_t full = row_tiles * s.n_tok;
  const int64_t quads = K / 256;
  if (allow_splitk && full * 2 <= P && quads >= 2) {
    int64_t S = P / full;
    if (S > ksplit_cap()) S = ksplit_cap();
    if (S > quads) S = quads;
    S = cdiv(quads, cdiv(quads, S));  // every slice gets cdiv(quads, S) quads: drop the slices that would stay empty
    if (S >= 2) {
      s.ksplit = (int)S;
      s.i_split = s.n_items = (int)(full * S);
      return s;
    }
  }
  const int64_t r = full % P;
  const int64_t r_split = (r > 0 && 2 * r <= P) ? r : 0;
  s.i_split = (int)(full - r_split);
  s.n_items = (int)(full + r_split);
  return s;
}

static size_t splitk_ws_bytes(const Sched& s) {
  return s.ksplit > 1 ? (size_t)s.ksplit * (size_t)s.n_row * s.n_tok * kUN * kTileRows * sizeof(float) : 0;
}

template <typename T, int NBITS, int GS>
static int launch(const void* x, Args& a, cudaStream_t st, const void* dense_W = nullptr, void* ws = nullptr, size_t ws_bytes = 0) {
  CUtensorMap xmap256, xmap128, amap;
  const CUtensorMapDataType dt = std::is_same<T, __half>::value ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  int rc = encode_map(&xmap256, x, a.M, a.K, dt, sizeof(T), kUN);
  if (rc) return rc;
  rc = encode_map(&xmap128, x, a.M, a.K, dt, sizeof(T), kUN / 2);
  if (rc) return rc;
  if (NBITS == 16) {
    rc = encode_map(&amap, dense_W, a.N, a.K, dt, sizeof(T), kTileRows);
    if (rc) return rc;
  } else {
    amap = xmap128;  // unused
  }
  constexpr int PR = NBITS == 16 ? kTileRows : kTileRows / (NBITS == 16 ? 1 : 8 / NBITS);
  const int P = persistent_ctas();
  a.sched = make_sched(a.M, a.K, cdiv(a.step, PR), P, NBITS != 16);
  a.ws = nullptr;
  if (a.sched.ksplit > 1) {
    const size_t need = splitk_ws_bytes(a.sched);
    HQQ_REQUIRE(ws != nullptr && ws_bytes >= need && aligned(ws, 256), HQQ_E_WORKSPACE,
                "hqq_b200_linear_fwd: this shape runs split-K and needs a 256-byte aligned workspace of %zu bytes (got %zu)", need, ws_bytes);
    a.ws = reinterpret_cast<float*>(ws);
  }
  const int grid = a.sched.n_items < P ? a.sched.n_items : P;
  constexpr auto k = linear_gemm_kernel<T, NBITS, GS>;
  rc = reserve_smem<k>(Smem::BYTES);
  if (rc) return rc;
  rc = launch_pdl("hqq_b200_linear_fwd/tcgen05", k, dim3((unsigned)grid), dim3(kThreads), Smem::BYTES, st, pdl_enabled(), xmap256, xmap128, amap, a);
  if (rc) return rc;
  if (a.sched.ksplit > 1) {
    const long long total = (long long)a.M * a.N;
    const bool vec = a.step % 4 == 0 && PR % 4 == 0 && aligned(a.y, 8);
    const auto reduce = vec ? splitk_reduce_kernel<T, 4> : splitk_reduce_kernel<T, 1>;
    return launch_pdl("hqq_b200_linear_fwd/splitk-reduce", reduce, dim3((unsigned)cdiv(vec ? total / 4 : total, 256)), dim3(256), 0, st, pdl_enabled(),
                      (const float*)a.ws, reinterpret_cast<T*>(a.y), reinterpret_cast<const T*>(a.bias), a.M, a.N, a.step, (int)PR, a.sched.ksplit,
                      a.sched.n_row, a.sched.n_tok);
  }
  return HQQ_OK;
}

template <typename T, int NBITS>
static int by_gs(const void* x, Args& a, int gs, cudaStream_t st, void* ws, size_t ws_bytes) {
  if (gs == 64) return launch<T, NBITS, 64>(x, a, st, nullptr, ws, ws_bytes);
  return launch<T, NBITS, 128>(x, a, st, nullptr, ws, ws_bytes);
}

template <typename T>
static int by_bits(const void* x, Args& a, int gs, int nbits, cudaStream_t st, void* ws, size_t ws_bytes) {
  switch (nbits) {
    case 8: return by_gs<T, 8>(x, a, gs, st, ws, ws_bytes);
    case 4: return by_gs<T, 4>(x, a, gs, st, ws, ws_bytes);
    case 2: return by_gs<T, 2>(x, a, gs, st, ws, ws_bytes);
    case 1: return by_gs<T, 1>(x, a, gs, st, ws, ws_bytes);
  }
  return HQQ_E_UNSUPPORTED;
}

}  // namespace gemm

bool gemm_route_ok(int64_t M, int64_t N, int64_t K, int gs, int nbits, int axis, int dtype) {
  if (axis != 1) return false;
  if (dtype != HQQ_F16 && dtype != HQQ_BF16) return false;
  if (!(nbits == 8 || nbits == 4 || nbits == 2 || nbits == 1)) return false;
  if (!(gs == 64 || gs == 128)) return false;     // one 64-k stage never straddles a group
  if (M < 1 || K % 256 != 0 || K % gs != 0) return false;  // the dequant loop handles four 64-k stages per iteration
  if (N % (8 / nbits) != 0) return false;
  if (K % 8 != 0 || N > (1 << 28) || K > (1 << 28) || M > (1 << 28)) return false;
  return true;
}

size_t gemm_workspace_bytes(int64_t M, int64_t N, int64_t K, int, int nbits, int) {
  const int F = 8 / nbits, PR = gemm::kTileRows / F;
  return gemm::splitk_ws_bytes(gemm::make_sched(M, K, cdiv(N / F, PR), gemm::persistent_ctas(), true));
}

// y[M, N] = x[M, K] @ W[N, K]^T (+ bias), W an ordinary fp16/bf16 matrix: the same persistent tcgen05 kernel with both operands on TMA
bool dense_route_ok(int64_t M, int64_t N, int64_t K, int dtype) {
  if (dtype != HQQ_F16 && dtype != HQQ_BF16) return false;
  return M >= 1 && N >= 1 && K >= 8 && K % 8 == 0 && N <= (1 << 28) && K <= (1 << 28) && M <= (1 << 28);  // 16-byte row pitch for the TMA
}

int linear_dense(const void* x, const void* W, const void* bias, void* y, int64_t M, int64_t N, int64_t K, int dtype, cudaStream_t st) {
  HQQ_REQUIRE(x && W && y, HQQ_E_INVALID, "hqq_b200_dense_gemm: null pointer");
  HQQ_REQUIRE(dense_route_ok(M, N, K, dtype), HQQ_E_UNSUPPORTED, "hqq_b200_dense_gemm: needs fp16/bf16 and K a multiple of 8 (M=%lld N=%lld K=%lld)",
              (long long)M, (long long)N, (long long)K);
  HQQ_REQUIRE(aligned(x, 16) && aligned(W, 16), HQQ_E_INVALID, "hqq_b200_dense_gemm: x and W must be 16-byte aligned");
  gemm::Args a;
  a.Wq = nullptr; a.scale = nullptr; a.zero = nullptr; a.bias = bias; a.y = y;
  a.M = (int)M; a.N = (int)N; a.K = (int)K;
  a.step = (int)N;  // one "slab": tile row t is weight row tile_n * 128 + t
  a.Gk = 0;
  if (dtype == HQQ_F16) return gemm::launch<__half, 16, 64>(x, a, st, W);
  return gemm::launch<__nv_bfloat16, 16, 64>(x, a, st, W);
}

int linear_gemm(const void* x, const void* Wq, const void* scale, const void* zero, const void* bias, void* y, int64_t M, int64_t N,
                int64_t K, int gs, int nbits, int dtype, void* ws, size_t ws_bytes, cudaStream_t st) {
  HQQ_REQUIRE(aligned(x, 16) && aligned(Wq, 16), HQQ_E_INVALID, "hqq_b200_linear_fwd: x and W_q must be 16-byte aligned");
  gemm::Args a;
  a.Wq = (const uint8_t*)Wq; a.scale = scale; a.zero = zero; a.bias = bias; a.y = y;
  a.M = (int)M; a.N = (int)N; a.K = (int)K;
  a.step = (int)(N / (8 / nbits));
  a.Gk = (int)(K / gs);
  if (dtype == HQQ_F16) return gemm::by_bits<__half>(x, a, gs, nbits, st, ws, ws_bytes);
  return gemm::by_bits<__nv_bfloat16>(x, a, gs, nbits, st, ws, ws_bytes);
}

}  // namespace hqq
