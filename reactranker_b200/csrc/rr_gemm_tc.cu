// tcgen05 / TMEM / TMA GEMM for the nn.Linear call sites (forward and dgrad), sm_100a.
//
//   C[M, N] = epilogue( sum_src  A_src[M, K_src] * B_src[N, K_src]^T )        (both operands K-major)
//
// fp32 in, fp32 out, fp32-class accuracy through a 3xTF32 split done on chip:
//   a = a_hi + a_lo,  a_hi = a rounded to the nearest TF32 value (low 13 mantissa bits zero)
//   A*B ~= A_hi*B_hi + A_lo*B_hi + A_hi*B_lo          (the dropped A_lo*B_lo term is ~2^-22 relative)
// so the reference's fp32 results are reproduced to ~1e-6 while the contraction runs on the 5th-gen
// tensor cores (kind::tf32), accumulating in TMEM.
//
// Persistent warp-specialised CTAs (k_tc_gemm2): TMA producer, MMA issuer, four split warps that move the A operand through TENSOR
// MEMORY, sixteen epilogue warps; see the comment above the kernel.  The backward GEMMs (dgrad: k_tc_gemm2<.., true>, wgrad:
// k_tc_wgrad3) use a 3 x bf16 split instead.  Two-source K (concat-free [x1 || x2] W^T) walks both sources through one accumulator.
#include <cuda.h>

#include "rr_common.cuh"

namespace rr {

namespace tc {

constexpr int BM = 128;         // rows per CTA tile == UMMA_M
constexpr int BK = 32;          // fp32 per k-block == one 128-byte swizzle row
constexpr int UK = 8;           // UMMA_K for kind::tf32 (32 bytes)
constexpr int A_BYTES = BM * BK * 4;
constexpr int THREADS = 192;
constexpr int MAX_NT = 320;
constexpr int SMEM_LIMIT = 227 * 1024;

struct Src {
  CUtensorMap tmA;
  CUtensorMap tmB;
  CUtensorMap tmBlo;  // v2 kernel, pre-split weights: the lo image of B (tmB then maps the hi image)
  int K;
  int pad_[15];  // keep every CUtensorMap 64-byte aligned inside the kernel parameter block
};

struct Args {
  Src src[2];
  int nsrc;
  int M, N;
  float* C;
  int ldc;
  const float* bias;
  const float* resid;
  int ldr;
  int relu;
  int accumulate;
  float p, inv_keep;
  uint64_t seed, stream_id;
  int presplit;  // B arrives as two TF32-exact images (hi, lo) made once per step by the pack kernel: no B split in the main loop
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, 128-byte swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
// start address >> 4 | LBO(=1, unused for swizzled K-major) << 16 | SBO(1024 B between 8-row groups) << 32 |
// version 1 << 46 | layout SWIZZLE_128B (2) << 61
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// kind::tf32 instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, both K-major
__device__ __forceinline__ uint32_t umma_idesc(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
        "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// explicit shared-space accesses: pointers carved out of the dynamic shared buffer are generic to the compiler, which
// otherwise emits LD.E/ST.E (generic, long-scoreboard) instead of LDS/STS in the split loops
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_f4(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void split4(float4 v, float4& h, float4& l) {
  // round-to-nearest onto the TF32 grid (10 explicit mantissa bits): |lo| <= 2^-12 |x|, signs balanced
  h.x = __uint_as_float((__float_as_uint(v.x) + 0x1000u) & 0xFFFFE000u);
  h.y = __uint_as_float((__float_as_uint(v.y) + 0x1000u) & 0xFFFFE000u);
  h.z = __uint_as_float((__float_as_uint(v.z) + 0x1000u) & 0xFFFFE000u);
  h.w = __uint_as_float((__float_as_uint(v.w) + 0x1000u) & 0xFFFFE000u);
  l = f4_sub(v, h);
}

// split an fp32 tile in place into hi (TF32-exact) and lo = x - hi; 128 threads, 4 independent chunks in flight each
__device__ __forceinline__ void split_tile(uint8_t* hi_p, uint8_t* lo_p, int bytes, int wtid) {
  const uint32_t hi = smem_u32(hi_p), lo = smem_u32(lo_p);
  int off = wtid * 16;
  for (; off + 3 * 2048 < bytes; off += 4 * 2048) {
    float4 v[4], h[4], l[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = lds_f4(hi + off + u * 2048);
#pragma unroll
    for (int u = 0; u < 4; ++u) split4(v[u], h[u], l[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      sts_f4(hi + off + u * 2048, h[u]);
      sts_f4(lo + off + u * 2048, l[u]);
    }
  }
  for (; off < bytes; off += 2048) {
    float4 h, l;
    split4(lds_f4(hi + off), h, l);
    sts_f4(hi + off, h);
    sts_f4(lo + off, l);
  }
}

// ================================================================================================
// v2 forward / dgrad kernel: persistent, A operand through TENSOR MEMORY (tcgen05.mma "TS" form).
//
// v1 re-reads the A tile from shared memory for each of the three TF32 products and writes both halves of the
// split back to shared memory, so shared-memory bandwidth (128 B/clk) paces it.  Here the four A-split warps read
// their row of the landed fp32 tile once and store (hi, lo) straight into TMEM with tcgen05.st; the MMAs take A from
// TMEM and only B from shared memory.  The CTA is persistent (one per SM, static round-robin over tiles), a
// separate epilogue warpgroup drains the accumulator while the producer and the split warps already work on the
// next tile, and the epilogue moves 64-byte row segments (tcgen05.ld x16).
//   warp 0: TMA producer | warp 1: MMA issuer (+TMEM alloc) | warps 2-5: split (A -> TMEM, B -> smem hi/lo) |
//   warps 6-21: epilogue (EW = 16)
// TMEM columns: [0, 320) accumulator, [320 + 64 s, ...) A stage s = 32 columns hi + 32 columns lo.
// ================================================================================================
constexpr int THREADS2_BASE = 192;   // TMA warp + MMA warp + 4 split warps; the epilogue adds 16 warps

__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,"
      "%30,%31,%32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]),
      "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]),
      "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]),
               "r"(r[14]), "r"(r[15])
               : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]),
               "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
// Epilogue of one [32 rows x 16 columns] sub-block of the accumulator, held one row per lane.
// A lane owning a whole row would touch 32 different rows per global instruction (no coalescing, most of every 32-byte sector wasted), and that
// was half of the kernel's time.  The sub-block is therefore transposed through a warp-private 2 KB staging tile (rows of 64 B; chunk c of
// row r sits at c ^ ((r >> 1) & 3), conflict-free for both the row-per-lane writes and the 4-lanes-per-row reads): afterwards 4 consecutive
// lanes cover one row's 64 contiguous bytes, 8 rows per global instruction.
// The residual (or, for dgrad accumulation, the previous value of C) of a sub-block is loaded one sub-block AHEAD of its use (epi_issue_h),
// the first of a tile before the wait for its accumulator, so its latency hides behind the MMAs.
// Sub-blocks of 16 rather than 32 columns need half the registers, so 16 epilogue warps fit instead of 8: the epilogue is issue-bound, not
// bandwidth-bound, and the 16-warp epilogue took 14 % off the forward GEMM (DESIGN.md §6b).
__device__ __forceinline__ void epi_issue_h(const Args& g, float4 (&R)[4], int row0, int col0, int lane) {
  const float* src = g.resid ? g.resid : (g.accumulate ? g.C : nullptr);
  if (src == nullptr) return;
  const int ld = g.resid ? g.ldr : g.ldc;
  const int col = col0 + 4 * (lane & 3);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int row = row0 + i * 8 + (lane >> 2);
    if (row < g.M && col < g.N) R[i] = ld_f4_stream(src + static_cast<size_t>(row) * ld + col);
  }
}
__device__ __forceinline__ void epilogue_block_h(const Args& g, const float (&v)[16], const float4 (&R)[4], uint32_t stage, int row0, int col0, int lane) {
  const int j = lane & 3, rsub = lane >> 2;
  const int col = col0 + 4 * j;
  const bool col_ok = col < g.N;
  const float4 bs = (g.bias && col_ok) ? ld_f4(g.bias + col) : f4_zero();
#pragma unroll
  for (int c = 0; c < 4; ++c)
    sts_f4(stage + lane * 64 + ((c ^ ((lane >> 1) & 3)) << 4), make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]));
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = i * 8 + rsub, row = row0 + r;
    float4 o = lds_f4(stage + r * 64 + ((j ^ ((r >> 1) & 3)) << 4));
    if (row < g.M && col_ok) {
      float* cp = g.C + static_cast<size_t>(row) * g.ldc + col;
      if (g.bias) o = f4_add(o, bs);
      if (g.resid) o = f4_add(o, R[i]);
      if (g.relu) o = f4_relu(o);
      if (g.p > 0.f) o = dropout4(o, g.p, g.inv_keep, g.seed, g.stream_id, (static_cast<uint64_t>(row) * g.ldc + col) >> 2);
      if (g.accumulate) o = f4_add(o, g.resid ? *reinterpret_cast<const float4*>(cp) : R[i]);
      st_f4(cp, o);
    }
  }
  __syncwarp();
}

constexpr int NT2 = 160;                          // output columns per work item (<= 160, multiple of 16)
constexpr int S2 = 3;                             // pipeline stages (shared memory A/B tiles + TMEM A tiles)
constexpr int B2_BYTES = NT2 * BK * 4;            // one B box: 160 rows x 128 B
constexpr int STAGE2 = A_BYTES + 2 * B2_BYTES;    // A raw | B hi | B lo  = 57344 B
constexpr int TM_A2 = 2 * NT2;                    // TMEM: two accumulators [0,160) [160,320), then the A stages: 3 x (32 hi + 32 lo) columns of A

// BF = true: the BACKWARD flavour (dgrad).  Gradients flow linearly through the backward pass and never decide a ReLU mask, so 16
// significand bits per operand are plenty there (north star: 1e-3 on gradients): x = x1 + x2 with x1 = bf16(x), x2 = bf16(x - x1), and
//   A*B ~= A2*B1 + A1*B2 + A1*B1      (kind::f16 with bf16 operands, fp32 accumulation; ~5e-6 of a row's maximum)
// Every MMA covers K = 16 instead of 8, i.e. half the tensor-pipe time of the 3xTF32 split, the weights arrive pre-split as bf16
// images of half the size (64-byte-swizzled rows: 32 bf16 per k-block), and a stage shrinks from 56 to 36 KB: FIVE stages in flight.
constexpr int B2_BYTES_BF = NT2 * BK * 2;                  // one bf16 B box: 160 rows x 64 B
constexpr int STAGE2_BF = A_BYTES + 2 * B2_BYTES_BF;       // A raw fp32 | B hi | B lo = 36864 B
constexpr int S2_BF = 5;

// K-major, 64-byte swizzle (bf16 k-block of 32): 8-row groups are 512 B apart
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(512 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(4) << 61;                     // cute::UMMA::LayoutType::SWIZZLE_64B
  return d;
}
// kind::f16 instruction descriptor: D = F32, A = B = BF16, both K-major
__device__ __forceinline__ uint32_t umma_idesc_bf16(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// (x0, x1) -> packed bf16 pair (x0 in the low half: the lower k index) and the packed pair of the remainders
__device__ __forceinline__ void split_bf16_pair(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
  const float r0 = x0 - __uint_as_float(hi << 16), r1 = x1 - __uint_as_float(hi & 0xFFFF0000u);
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(r1), "f"(r0));
}

template <int EW, bool BF>
__global__ void __launch_bounds__(THREADS2_BASE + 32 * EW, 1) k_tc_gemm2(const __grid_constant__ Args g) {
  static_assert(EW == 16, "the epilogue is written for 16 warps, four per TMEM lane quadrant");
  constexpr int S2 = BF ? S2_BF : tc::S2;
  constexpr int STAGE2 = BF ? STAGE2_BF : tc::STAGE2;
  constexpr int B2_BYTES = BF ? B2_BYTES_BF : tc::B2_BYTES;
  constexpr int A_COLS = BF ? 32 : 64;                     // TMEM columns of one A stage (hi | lo)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + static_cast<size_t>(S2) * STAGE2);
  uint64_t* ready = full + S2;
  uint64_t* empty = ready + S2;
  uint64_t* acc_full = empty + S2;     // [2]
  uint64_t* acc_empty = acc_full + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tiles = (g.M + BM - 1) / BM, n_tiles = (g.N + NT2 - 1) / NT2;
  const int total_tiles = m_tiles * n_tiles;
  int nkb_total = 0;
  for (int s = 0; s < g.nsrc; ++s) nkb_total += (g.src[s].K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < S2; ++s) {
      mbar_init(full + s, 1);
      mbar_init(ready + s, 4);
      mbar_init(empty + s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(acc_full + b, 1);
      mbar_init(acc_empty + b, EW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int s = 0; s < g.nsrc; ++s) {
      prefetch_tmap(&g.src[s].tmA);
      prefetch_tmap(&g.src[s].tmB);
    }
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();             // nothing above touches global memory (tensor-map prefetches read kernel parameters)

  if (warp == 0) {
    // ---------------- TMA producer ----------------
    if (lane == 0) {
      int it = 0;
      const uint32_t tx = static_cast<uint32_t>(A_BYTES + ((g.presplit || BF) ? 2 : 1) * B2_BYTES);
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int m0 = (tile / n_tiles) * BM, n0 = (tile % n_tiles) * NT2;
        for (int s = 0; s < g.nsrc; ++s) {
          const int nkb = (g.src[s].K + BK - 1) / BK;
          for (int kb = 0; kb < nkb; ++kb, ++it) {
            const int st = it % S2;
            const uint32_t ph = (it / S2) & 1;
            mbar_wait(empty + st, ph ^ 1);
            uint8_t* base = smem + static_cast<size_t>(st) * STAGE2;
            mbar_expect_tx(full + st, tx);
            tma_load_2d(&g.src[s].tmA, full + st, base, kb * BK, m0);
            tma_load_2d(&g.src[s].tmB, full + st, base + A_BYTES, kb * BK, n0);   // rows past N are zero-filled
            if (g.presplit || BF) tma_load_2d(&g.src[s].tmBlo, full + st, base + A_BYTES + B2_BYTES, kb * BK, n0);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer ----------------
    if (lane == 0) {
      int it = 0, w = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++w) {
        const int n0 = (tile % n_tiles) * NT2;
        const int width = min(NT2, g.N - n0);
        const uint32_t idesc = BF ? umma_idesc_bf16(BM, width) : umma_idesc(BM, width);
        const int buf = w & 1;
        const uint32_t d = tmem_base + buf * NT2;
        mbar_wait(acc_empty + buf, ((w >> 1) & 1) ^ 1);     // the epilogue has drained this accumulator
        tc_fence_after();
        for (int kb = 0; kb < nkb_total; ++kb, ++it) {
          const int st = it % S2;
          const uint32_t ph = (it / S2) & 1;
          mbar_wait(ready + st, ph);
          tc_fence_after();
          const uint32_t base = smem_u32(smem + static_cast<size_t>(st) * STAGE2);
          const uint32_t b_hi = base + A_BYTES, b_lo = b_hi + B2_BYTES;
          const uint32_t a_hi = tmem_base + TM_A2 + st * A_COLS, a_lo = a_hi + A_COLS / 2;
          if constexpr (BF) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {           // UMMA_K = 16 bf16 = 32 bytes of the 64-byte row = 8 TMEM columns of packed pairs
              const uint32_t ko = k * 32;
              umma_bf16_ts(d, a_lo + k * 8, umma_desc_sw64(b_hi + ko), idesc, (kb > 0 || k > 0) ? 1u : 0u);
              umma_bf16_ts(d, a_hi + k * 8, umma_desc_sw64(b_lo + ko), idesc, 1u);
              umma_bf16_ts(d, a_hi + k * 8, umma_desc_sw64(b_hi + ko), idesc, 1u);
            }
          } else {
#pragma unroll
            for (int k = 0; k < BK / UK; ++k) {
              const uint32_t ko = k * UK * 4;
              umma_tf32_ts(d, a_lo + k * UK, umma_desc(b_hi + ko), idesc, (kb > 0 || k > 0) ? 1u : 0u);
              umma_tf32_ts(d, a_hi + k * UK, umma_desc(b_lo + ko), idesc, 1u);
              umma_tf32_ts(d, a_hi + k * UK, umma_desc(b_hi + ko), idesc, 1u);
            }
          }
          umma_commit(empty + st);
        }
        umma_commit(acc_full + buf);
      }
    }
  } else if (warp < 6) {
    // ---------------- split workers ----------------
    const int wtid = threadIdx.x - 64;       // 0..127
    const int quad = warp & 3;
    const int r = quad * 32 + lane;          // row of the A tile owned by this thread == its TMEM lane
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int n0 = (tile % n_tiles) * NT2;
      const int b_used = min(NT2, g.N - n0) * BK * 4;      // only the rows the MMA reads need splitting
      for (int kb = 0; kb < nkb_total; ++kb, ++it) {
        const int st = it % S2;
        const uint32_t ph = (it / S2) & 1;
        mbar_wait(full + st, ph);
        uint8_t* base = smem + static_cast<size_t>(st) * STAGE2;
        // A: this thread's row of 32 floats (128-byte swizzle: chunk c sits at c ^ (row & 7)) -> hi / lo -> TMEM
        // 704 threads cap the kernel at 88 registers: two halves of 16 floats each instead of the whole row at once
        const uint32_t rowp = smem_u32(base) + r * 128;
#pragma unroll
        for (int hlf = 0; hlf < 2; ++hlf) {
          float4 av[4];
#pragma unroll
          for (int c = 0; c < 4; ++c) av[c] = lds_f4(rowp + (((4 * hlf + c) ^ (r & 7)) << 4));
          if constexpr (BF) {
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              split_bf16_pair(av[c].x, av[c].y, hi[2 * c], lo[2 * c]);
              split_bf16_pair(av[c].z, av[c].w, hi[2 * c + 1], lo[2 * c + 1]);
            }
            tmem_st8(lane_addr + TM_A2 + st * A_COLS + 8 * hlf, hi);
            tmem_st8(lane_addr + TM_A2 + st * A_COLS + 16 + 8 * hlf, lo);
          } else {
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const float e[4] = {av[c].x, av[c].y, av[c].z, av[c].w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint32_t h = (__float_as_uint(e[j]) + 0x1000u) & 0xFFFFE000u;
                hi[4 * c + j] = h;
                lo[4 * c + j] = __float_as_uint(e[j] - __uint_as_float(h));
              }
            }
            tmem_st16(lane_addr + TM_A2 + st * A_COLS + 16 * hlf, hi);
            tmem_st16(lane_addr + TM_A2 + st * A_COLS + 32 + 16 * hlf, lo);
          }
        }
        // B: elementwise split in shared memory (unless the weights arrived pre-split)
        if (!BF && !g.presplit) split_tile(base + A_BYTES, base + A_BYTES + B2_BYTES, b_used, wtid);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        if (!BF && !g.presplit) fence_proxy_async();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(ready + st);
      }
    }
  } else {
    // ---------------- epilogue: EW / 4 warps per TMEM lane quadrant, taking the 16-column sub-blocks of a tile in turn ----------------
    constexpr int EPQ = EW / 4;
    const int quad = warp & 3;
    const int eidx = (warp - 6) >> 2;
    const uint32_t stage = smem_u32(reinterpret_cast<uint8_t*>(full) + 256) + (warp - 6) * 2048;   // warp-private 2 KB staging tile
    int w = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++w) {
      const int m0 = (tile / n_tiles) * BM, n0 = (tile % n_tiles) * NT2;
      const int nblk = (min(NT2, g.N - n0) + 15) >> 4;            // 16-column sub-blocks (tile widths are multiples of 16)
      const int row0 = m0 + quad * 32;
      const int buf = w & 1;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + buf * NT2;
      float4 R[4];
      int c = (eidx + w) & (EPQ - 1);                              // rotate the start so the 10 sub-blocks of a tile spread evenly over tiles
      if (c < nblk) epi_issue_h(g, R, row0, n0 + 16 * c, lane);
      mbar_wait(acc_full + buf, (w >> 1) & 1);
      tc_fence_after();
      if (c >= nblk) {                        // narrow tile: nothing for this warp, but the accumulator hand-back counts every epilogue warp
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty + buf);
      }
      for (; c < nblk; c += EPQ) {
        float v[16];
        tmem_ld16(taddr + 16 * c, v);
        const bool last = c + EPQ >= nblk;
        if (last) {                           // last read of this accumulator: hand it back before the global traffic
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(acc_empty + buf);
        }
        float4 Rn[4];
        if (!last) epi_issue_h(g, Rn, row0, n0 + 16 * (c + EPQ), lane);
        epilogue_block_h(g, v, R, stage, row0, n0 + 16 * c, lane);
        if (!last) {
#pragma unroll
          for (int i = 0; i < 4; ++i) R[i] = Rn[i];
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ================================================================================================
// wgrad:  dW[n, k] += sum_m dZ[m, n] * X[m, k]      (+ dbias[n] += sum_m dZ[m, n])
// The reduction runs over the ROWS of both operands, so both are MN-major for the tensor core:
// a TMA box [32 rows m x 32 floats] lands as 32 rows of 128 bytes (128B swizzle) = one MN-atom column,
// UMMA descriptors use LBO = bytes between 32-float column blocks, SBO = 512 (4 rows of the reduction, 32-byte-atom swizzle).
// One CTA = 128 rows of dW (n) x up to 320 columns (k) x a slab of the m range; partial results are
// added to dW with vector reductions (split over m like the SIMT kernel).
// ================================================================================================
constexpr int WG_BK = 32;                 // rows of the reduction per stage

struct WgArgs {
  CUtensorMap tmA;   // dZ [M, n]
  CUtensorMap tmB;   // X  [M, k]
  int M, n, k;
  int kt;            // k columns per CTA (multiple of 16, <= 320)
  int nb;            // TMA boxes of B per stage = ceil(kt / 32)
  int k_pad;         // k rounded up to 16: the last k-tile may be narrower than kt
  int tm_a;          // first TMEM column of the A stages (accumulator below it)
  int stages;        // pipeline stages (wgrad3: slots of the raw ring)
  int bf_stages;     // wgrad3: slots of the bf16 ring / TMEM A operand
  int m_chunk;       // rows of the reduction per blockIdx.z (multiple of WG_BK)
  float* dW;
  int lddw;
  float* dbias;
  long long slab_stride;   // SLAB kernels (deterministic mode): slab z stores to dW + z * slab_stride and dbias + z * n
};

// MN-major tf32 operands have exactly one legal shared-memory layout: 128-byte swizzle with 32-byte atomicity
// (cute::UMMA::LayoutType::SWIZZLE_128B_BASE32B = 1, TMA's CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B): atoms of 4 reduction rows x 128 B,
// so SBO = 512 B between 4-row groups and LBO = bytes between 32-float column blocks.
__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(lbo_bytes >> 4) << 16;
  d |= static_cast<uint64_t>(512 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(1) << 61;
  return d;
}
__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// ================================================================================================
// wgrad v2: the dZ operand goes through TENSOR MEMORY.
// v1 splits both operands in shared memory and reads both back for each of the three TF32 products: ~390 KB of shared-memory traffic per
// 32 rows of the reduction, twice what the MMAs themselves need.  Here the thread that owns TMEM lane n reads column n of the landed
// dZ tile (one LDS.32 per row: a warp reads 128 contiguous bytes, no swizzle needed), splits it in registers and tcgen05.st's (hi, lo)
// into TMEM as the [n x m] A operand; only X is split in shared memory (MN-major B, as in v1).  The bias gradient is the same thread's
// running sum.  BKR = rows of the reduction per pipeline stage (32: 2 stages at 320 columns; 16: 4 stages).
// TMEM: accumulator from column 0 | stage s: BKR columns hi + BKR columns lo from column tm_a + 2 BKR s.
// ================================================================================================

// SLAB = true (deterministic mode): the slab's tile is STORED to its own slice of scratch, never added (see tc_wgrad).
template <int BKR, bool SLAB>
__global__ void __launch_bounds__(THREADS, 1) k_tc_wgrad2(const __grid_constant__ WgArgs g) {
  constexpr int BOX = BKR * 128;          // bytes of one [BKR x 32 floats] TMA box
  constexpr int A_RAW = 4 * BOX;          // 128 n-columns
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  const int b_bytes = g.nb * BOX;
  const int stage_bytes = A_RAW + 2 * b_bytes;   // A raw | B hi | B lo
  const int S = g.stages;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + static_cast<size_t>(S) * stage_bytes);
  uint64_t* ready = full + S;
  uint64_t* empty = ready + S;
  uint64_t* acc_bar = empty + S;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * BM, k0 = blockIdx.y * g.kt;
  const int m_beg = blockIdx.z * g.m_chunk;
  const int m_end = min(g.M, m_beg + g.m_chunk);
  const int nst = (m_end - m_beg + BKR - 1) / BKR;   // >= 1 by construction of the grid

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(full + s, 1);
      mbar_init(ready + s, 4);
      mbar_init(empty + s, 1);
    }
    mbar_init(acc_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    prefetch_tmap(&g.tmA);
    prefetch_tmap(&g.tmB);
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();             // nothing above touches global memory (tensor-map prefetches read kernel parameters)

  if (warp == 0) {
    if (lane == 0) {
      const uint32_t tx = static_cast<uint32_t>(A_RAW + b_bytes);
      for (int it = 0; it < nst; ++it) {
        const int st = it % S;
        const uint32_t ph = (it / S) & 1;
        mbar_wait(empty + st, ph ^ 1);
        uint8_t* base = smem + static_cast<size_t>(st) * stage_bytes;
        const int m = m_beg + it * BKR;
        mbar_expect_tx(full + st, tx);
        for (int j = 0; j < 4; ++j) tma_load_2d(&g.tmA, full + st, base + j * BOX, n0 + 32 * j, m);
        for (int j = 0; j < g.nb; ++j) tma_load_2d(&g.tmB, full + st, base + A_RAW + j * BOX, k0 + 32 * j, m);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const int width = min(g.kt, g.k_pad - k0);
      const int n1 = (width <= 256) ? width : 160;    // 160 = five 32-float atoms: the second MMA starts on an atom boundary
      const int n2 = width - n1;
      const uint32_t mn = (1u << 16);                 // B is MN-major; A comes from TMEM
      const uint32_t idesc1 = umma_idesc(BM, n1) | mn;
      const uint32_t idesc2 = n2 ? (umma_idesc(BM, n2) | mn) : 0u;
      for (int it = 0; it < nst; ++it) {
        const int st = it % S;
        const uint32_t ph = (it / S) & 1;
        mbar_wait(ready + st, ph);
        tc_fence_after();
        const uint32_t base = smem_u32(smem + static_cast<size_t>(st) * stage_bytes);
        const uint32_t b_hi = base + A_RAW, b_lo = b_hi + b_bytes;
        const uint32_t a_hi = tmem_base + g.tm_a + st * 2 * BKR, a_lo = a_hi + BKR;
#pragma unroll
        for (int k = 0; k < BKR / UK; ++k) {
          const uint32_t ko = k * 1024;                  // next 8 rows of the reduction
          const uint32_t first = (it > 0 || k > 0) ? 1u : 0u;
          umma_tf32_ts(tmem_base, a_lo + k * UK, umma_desc_mn(b_hi + ko, BOX), idesc1, first);
          umma_tf32_ts(tmem_base, a_hi + k * UK, umma_desc_mn(b_lo + ko, BOX), idesc1, 1u);
          umma_tf32_ts(tmem_base, a_hi + k * UK, umma_desc_mn(b_hi + ko, BOX), idesc1, 1u);
          if (n2) {
            const uint32_t bo = static_cast<uint32_t>(n1 / 32) * BOX;
            umma_tf32_ts(tmem_base + n1, a_lo + k * UK, umma_desc_mn(b_hi + bo + ko, BOX), idesc2, first);
            umma_tf32_ts(tmem_base + n1, a_hi + k * UK, umma_desc_mn(b_lo + bo + ko, BOX), idesc2, 1u);
            umma_tf32_ts(tmem_base + n1, a_hi + k * UK, umma_desc_mn(b_hi + bo + ko, BOX), idesc2, 1u);
          }
        }
        umma_commit(empty + st);
      }
      umma_commit(acc_bar);
    }
  } else {
    const int wtid = threadIdx.x - 64;
    const int quad = warp & 3;
    const int r = quad * 32 + lane;                   // TMEM lane == column n0 + r of dZ
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    float bsum = 0.f;
    for (int it = 0; it < nst; ++it) {
      const int st = it % S;
      const uint32_t ph = (it / S) & 1;
      mbar_wait(full + st, ph);
      uint8_t* base = smem + static_cast<size_t>(st) * stage_bytes;
      const uint32_t colp = smem_u32(base) + quad * BOX + lane * 4;
      float a[BKR];
#pragma unroll
      for (int m = 0; m < BKR; ++m) asm volatile("ld.shared.f32 %0, [%1];" : "=f"(a[m]) : "r"(colp + m * 128));
      uint32_t hi[BKR], lo[BKR];
#pragma unroll
      for (int m = 0; m < BKR; ++m) {
        const uint32_t h = (__float_as_uint(a[m]) + 0x1000u) & 0xFFFFE000u;
        hi[m] = h;
        lo[m] = __float_as_uint(a[m] - __uint_as_float(h));
        bsum += a[m];
      }
      const uint32_t ta = lane_addr + g.tm_a + st * 2 * BKR;
      if constexpr (BKR == 32) {
        tmem_st32(ta, hi);
        tmem_st32(ta + BKR, lo);
      } else {
        tmem_st16(ta, hi);
        tmem_st16(ta + BKR, lo);
      }
      split_tile(base + A_RAW, base + A_RAW + b_bytes, b_bytes, wtid);
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(ready + st);
    }
    if constexpr (SLAB) {
      if (g.dbias != nullptr && blockIdx.y == 0 && n0 + r < g.n) g.dbias[static_cast<size_t>(blockIdx.z) * g.n + n0 + r] = bsum;
    } else {
      if (g.dbias != nullptr && blockIdx.y == 0 && n0 + r < g.n) atomicAdd(g.dbias + n0 + r, bsum);
    }
    mbar_wait(acc_bar, 0);
    tc_fence_after();
    const int row = n0 + r;
    const int width = min(g.kt, g.k_pad - k0);
    for (int c = 0; c < width; c += 16) {
      float v[16];
      tmem_ld16(lane_addr + c, v);
      if (row < g.n) {
        if constexpr (SLAB) {
          float* cp = g.dW + blockIdx.z * g.slab_stride + static_cast<size_t>(row) * g.lddw + k0 + c;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (k0 + c + 4 * q < g.k) st_f4(cp + 4 * q, make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]));
        } else {
          float* cp = g.dW + static_cast<size_t>(row) * g.lddw + k0 + c;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (k0 + c + 4 * q < g.k) red_add_v4(cp + 4 * q, v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ================================================================================================
// wgrad v3: 3 x bf16 split (backward flavour, see k_tc_gemm2<.., true>).
// dW is a sum over ~10^5 rows whose rounding errors are independent, and it feeds nothing but Adam: 16 significand bits per operand are
// ample, and they halve both the tensor-pipe time (UMMA_K = 16) and the shared-memory bytes the MMAs read, which is what bounds v2.
//   raw ring  : TMA lands fp32 tiles  dZ [32 x 128] (unswizzled: column reads)  |  X [32 x kt] in 32-float boxes (128-byte swizzle)
//   workers   : dZ column n -> registers -> bf16 pairs (hi, lo) -> TMEM (A operand, lane n);  bias gradient = running column sum
//               X -> bf16 (hi, lo) images in the canonical MN-major 128-byte-swizzle layout (64 columns per 128-byte row, 8-row atoms)
//   MMA       : kind::f16, A from TMEM, B MN-major from the bf16 ring; the raw slot is free again as soon as the conversion is done
// ================================================================================================
// The raw ring (R slots: what TMA has in flight) and the bf16 ring (SB slots: what the tensor core reads) are sized separately, and the rows
// of the reduction per stage (32 or 64) are a template parameter.
// Measured on [321 778 x 304]^T [321 778 x 304] (profiles/r02_wgrad_cfg.md): 32 rows, 2 + 2 slots 266-273 us; 32 rows, 3 + 1 slots 330 us;
// 16 rows with 4 + 2, 5 + 3, 6 + 2 or 5 + 2 slots 361 us each.  The timeline of one CTA's hand-offs (DESIGN.md §4.2) says why: a raw slot's
// turn-around is TMA issue ~1200 clk (14 boxes at the TMA unit's ~85 clk per 32-float box) + arrival ~1000 + conversion ~1650 (= the stage's
// 212 KB of shared-memory traffic at 128 B/clk) + hand-offs ~500, and two slots make that 2212 clk per stage; 16-row stages double the
// per-row box cost, and a third 57 KB raw slot does not fit beside two 40 KB bf16 slots.  Narrow X tiles do fit more raw slots (up to 6),
// worth 6-9 % there.

template <int BKR>
__device__ __forceinline__ uint64_t umma_desc_mn_bf16(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((BKR * 128) >> 4) << 16;   // LBO: next block of 64 columns
  d |= static_cast<uint64_t>(1024 >> 4) << 32;          // SBO: next 8 rows of the reduction
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;                  // SWIZZLE_128B
  return d;
}

constexpr int W3_WORKERS = 256;   // 8 conversion warps (12 measured no faster): with 4 the fp32 -> bf16 conversion (not the MMAs) paced the kernel
constexpr int W3_THREADS = 64 + W3_WORKERS;

template <int BKR, bool SLAB>
__global__ void __launch_bounds__(W3_THREADS, 1) k_tc_wgrad3(const __grid_constant__ WgArgs g) {
  static_assert(BKR == 32 || BKR == 64, "stages of 32 or 64 rows of the reduction");
  constexpr int BOX = BKR * 128;               // bytes of one raw TMA box [BKR x 32 floats] == one bf16 MN block [BKR x 64 bf16]
  constexpr int A_RAW = 4 * BOX;               // dZ: 128 columns
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  const int R = g.stages, SB = g.bf_stages;
  const int nblk = (g.kt + 63) / 64;                     // bf16 MN blocks per image
  const int raw_bytes = A_RAW + g.nb * BOX;              // dZ | X
  const int bf_bytes = 2 * nblk * BOX;                   // X hi | X lo
  uint8_t* raw0 = smem;
  uint8_t* bf0 = smem + static_cast<size_t>(R) * raw_bytes;
  uint64_t* raw_full = reinterpret_cast<uint64_t*>(bf0 + static_cast<size_t>(SB) * bf_bytes);
  uint64_t* raw_empty = raw_full + R;
  uint64_t* ready = raw_empty + R;
  uint64_t* mma_done = ready + SB;
  uint64_t* acc_bar = mma_done + SB;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * BM, k0 = blockIdx.y * g.kt;
  const int m_beg = blockIdx.z * g.m_chunk;
  const int m_end = min(g.M, m_beg + g.m_chunk);
  const int nst = (m_end - m_beg + BKR - 1) / BKR;
  const int width = min(g.kt, g.k_pad - k0);

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < R; ++s) {
      mbar_init(raw_full + s, 1);
      mbar_init(raw_empty + s, W3_WORKERS / 32);
    }
    for (int s = 0; s < SB; ++s) {
      mbar_init(ready + s, W3_WORKERS / 32);
      mbar_init(mma_done + s, 1);
    }
    mbar_init(acc_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    prefetch_tmap(&g.tmA);
    prefetch_tmap(&g.tmB);
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();             // nothing above touches global memory (tensor-map prefetches read kernel parameters)

  if (warp == 0) {
    if (lane == 0) {
      const uint32_t tx = static_cast<uint32_t>(raw_bytes);
      for (int it = 0; it < nst; ++it) {
        const int st = it % R;
        const uint32_t ph = (it / R) & 1;
        mbar_wait(raw_empty + st, ph ^ 1);
        uint8_t* base = raw0 + static_cast<size_t>(st) * raw_bytes;
        const int m = m_beg + it * BKR;
        mbar_expect_tx(raw_full + st, tx);
        // ~85 clk per box: the TMA unit's rate for 32-float x 32-row boxes (one box per lane from 14 lanes takes exactly as long)
        for (int j = 0; j < 4; ++j) tma_load_2d(&g.tmA, raw_full + st, base + j * BOX, n0 + 32 * j, m);
        for (int j = 0; j < g.nb; ++j) tma_load_2d(&g.tmB, raw_full + st, base + A_RAW + j * BOX, k0 + 32 * j, m);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const int n1 = (width <= 256) ? width : 192;     // 192 = three 64-column blocks: the second MMA starts on a block boundary
      const int n2 = width - n1;
      const uint32_t mn = (1u << 16);                  // B is MN-major; A comes from TMEM
      const uint32_t idesc1 = umma_idesc_bf16(BM, n1) | mn;
      const uint32_t idesc2 = n2 ? (umma_idesc_bf16(BM, n2) | mn) : 0u;
      for (int it = 0; it < nst; ++it) {
        const int st = it % SB;
        const uint32_t ph = (it / SB) & 1;
        mbar_wait(ready + st, ph);
        tc_fence_after();
        const uint32_t b_hi = smem_u32(bf0 + static_cast<size_t>(st) * bf_bytes), b_lo = b_hi + nblk * BOX;
        const uint32_t a_hi = tmem_base + g.tm_a + st * BKR, a_lo = a_hi + BKR / 2;
#pragma unroll
        for (int k = 0; k < BKR / 16; ++k) {
          const uint32_t ko = k * 2048;                // next 16 rows of the reduction = two 8-row atoms
          const uint32_t first = (it > 0 || k > 0) ? 1u : 0u;
          umma_bf16_ts(tmem_base, a_lo + k * 8, umma_desc_mn_bf16<BKR>(b_hi + ko), idesc1, first);
          umma_bf16_ts(tmem_base, a_hi + k * 8, umma_desc_mn_bf16<BKR>(b_lo + ko), idesc1, 1u);
          umma_bf16_ts(tmem_base, a_hi + k * 8, umma_desc_mn_bf16<BKR>(b_hi + ko), idesc1, 1u);
          if (n2) {
            const uint32_t bo = static_cast<uint32_t>(n1 / 64) * BOX;
            umma_bf16_ts(tmem_base + n1, a_lo + k * 8, umma_desc_mn_bf16<BKR>(b_hi + bo + ko), idesc2, first);
            umma_bf16_ts(tmem_base + n1, a_hi + k * 8, umma_desc_mn_bf16<BKR>(b_lo + bo + ko), idesc2, 1u);
            umma_bf16_ts(tmem_base + n1, a_hi + k * 8, umma_desc_mn_bf16<BKR>(b_hi + bo + ko), idesc2, 1u);
          }
        }
        umma_commit(mma_done + st);
      }
      umma_commit(acc_bar);
    }
  } else {
    const int wtid = threadIdx.x - 64;
    const int quad = warp & 3;
    const int r = quad * 32 + lane;                    // TMEM lane == column n0 + r of dZ
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    const int G = g.nb * 4;                            // 8-column groups per row of the X tile (whole boxes: the padding converts zeros)
    const int step_m = W3_WORKERS / G, step_c = W3_WORKERS % G;
    const bool a_warp = warp < 6;                     // warps 2..5 own the four TMEM lane quadrants: dZ conversion and the final read-out
    float bsum = 0.f;
    for (int it = 0; it < nst; ++it) {
      const int rs = it % R, bs = it % SB;
      mbar_wait(raw_full + rs, (it / R) & 1);
      mbar_wait(mma_done + bs, ((it / SB) & 1) ^ 1);  // the MMAs of the previous lap are done with this bf16 slot and TMEM slot
      tc_fence_after();
      const uint32_t raw = smem_u32(raw0 + static_cast<size_t>(rs) * raw_bytes);
      if (a_warp) {
        const uint32_t colp = raw + quad * BOX + lane * 4;
        float a[BKR];
#pragma unroll
        for (int m = 0; m < BKR; ++m) asm volatile("ld.shared.f32 %0, [%1];" : "=f"(a[m]) : "r"(colp + m * 128));
        uint32_t hi[BKR / 2], lo[BKR / 2];
#pragma unroll
        for (int m = 0; m < BKR / 2; ++m) {
          split_bf16_pair(a[2 * m], a[2 * m + 1], hi[m], lo[m]);
          bsum += a[2 * m] + a[2 * m + 1];
        }
        const uint32_t ta = lane_addr + g.tm_a + bs * BKR;
        if constexpr (BKR == 64) {
          tmem_st32(ta, hi);
          tmem_st32(ta + 32, lo);
        } else {
          tmem_st16(ta, hi);
          tmem_st16(ta + 16, lo);
        }
      }
      const uint32_t xraw = raw + A_RAW;
      const uint32_t xhi = smem_u32(bf0 + static_cast<size_t>(bs) * bf_bytes), xlo = xhi + nblk * BOX;
      int m = wtid / G, cg = wtid - m * G;
      for (; m < BKR;) {
        const int jb = cg >> 2, c2 = (cg & 3) << 1, sw = m & 7;
        const uint32_t rp = xraw + jb * BOX + m * 128;
        // two 16-byte chunks of 4 floats; boxes of odd index read theirs in the opposite order: 8 consecutive lanes hit 8 distinct bank groups
        const int first = c2 + (jb & 1), second = c2 + 1 - (jb & 1);
        const float4 f0 = lds_f4(rp + ((first ^ sw) << 4)), f1 = lds_f4(rp + ((second ^ sw) << 4));
        const float4 lo4 = (jb & 1) ? f1 : f0, hi4 = (jb & 1) ? f0 : f1;     // columns 8cg..8cg+3 | 8cg+4..8cg+7
        uint32_t h[4], l[4];
        split_bf16_pair(lo4.x, lo4.y, h[0], l[0]);
        split_bf16_pair(lo4.z, lo4.w, h[1], l[1]);
        split_bf16_pair(hi4.x, hi4.y, h[2], l[2]);
        split_bf16_pair(hi4.z, hi4.w, h[3], l[3]);
        const uint32_t off = (cg >> 3) * BOX + m * 128 + (((cg & 7) ^ sw) << 4);
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(xhi + off), "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3]) : "memory");
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(xlo + off), "r"(l[0]), "r"(l[1]), "r"(l[2]), "r"(l[3]) : "memory");
        m += step_m;
        cg += step_c;
        if (cg >= G) {
          cg -= G;
          ++m;
        }
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      fence_proxy_async();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(ready + bs);
        mbar_arrive(raw_empty + rs);
      }
    }
    if constexpr (SLAB) {
      if (a_warp && g.dbias != nullptr && blockIdx.y == 0 && n0 + r < g.n) g.dbias[static_cast<size_t>(blockIdx.z) * g.n + n0 + r] = bsum;
    } else {
      if (a_warp && g.dbias != nullptr && blockIdx.y == 0 && n0 + r < g.n) atomicAdd(g.dbias + n0 + r, bsum);
    }
    mbar_wait(acc_bar, 0);
    tc_fence_after();
    const int row = n0 + r;
    for (int c = 0; a_warp && c < width; c += 16) {
      float v[16];
      tmem_ld16(lane_addr + c, v);
      if (row < g.n) {
        if constexpr (SLAB) {
          float* cp = g.dW + blockIdx.z * g.slab_stride + static_cast<size_t>(row) * g.lddw + k0 + c;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (k0 + c + 4 * q < g.k) st_f4(cp + 4 * q, make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]));
        } else {
          float* cp = g.dW + static_cast<size_t>(row) * g.lddw + k0 + c;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (k0 + c + 4 * q < g.k) red_add_v4(cp + 4 * q, v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ---- host side -------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D fp32 row-major [rows, cols] with row stride ld floats; box = [box_rows x 32 floats], 128-byte swizzle
static int make_map(CUtensorMap* map, const float* ptr, int rows, int cols, int ld, int box_rows,
                    CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  if (box_rows < 1 || box_rows > 256) return fail(RR_ERR_INVALID, "TMA box of %d rows", box_rows);
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(RR_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 4};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_128B;   // 256 B measured no better (wgrad) or worse (forward)
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  swizzle, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(RR_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows %d cols %d ld %d box_rows %d", static_cast<int>(r), rows, cols, ld, box_rows);
  return RR_OK;
}

// 2-D bf16 row-major [rows, cols] with row stride ld elements; box = [box_rows x 32 bf16] (64-byte rows, 64-byte swizzle)
static int make_map_bf16(CUtensorMap* map, const uint16_t* ptr, int rows, int cols, int ld, int box_rows) {
  if (box_rows < 1 || box_rows > 256) return fail(RR_ERR_INVALID, "TMA box of %d rows", box_rows);
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(RR_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<uint16_t*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(RR_ERR_CUDA, "cuTensorMapEncodeTiled(bf16) failed (%d) rows %d cols %d ld %d box_rows %d", static_cast<int>(r), rows, cols, ld, box_rows);
  return RR_OK;
}

}  // namespace tc

// Can this problem run on k_tc_gemm2?  (everything the model produces can; odd C-ABI calls fall back to SIMT)
bool tc_supported(int M, int n, int k1, int k2, int ldx1, int ldx2) {
  return M > 0 && n >= 16 && !(n & 15) && k1 > 0 && !(k1 & 3) && !(k2 & 3) && !(ldx1 & 3) && !(ldx2 & 3);
}
// The same for one source with bf16 images of W (row stride ldw elements): 16-byte bf16 rows need ldw % 8 == 0.
bool tc_linear_bf16_supported(int M, int n, int k, int ldx, int ldw) {
  return M > 0 && n >= 16 && !(n & 15) && k > 0 && !(k & 3) && !(ldx & 3) && !(ldw & 7);
}

// TC_BF16_PAIR runs the backward flavour k_tc_gemm2<16, true> (3 x bf16 products, five pipeline stages), the others k_tc_gemm2<16, false>.
int tc_linear(TcSplit split, int M, int n, const TcSrc* src, int nsrc, const float* bias, const float* resid, int ldr, float* Y, int ldy, int relu,
              int accumulate, float p, uint64_t seed, uint64_t stream_id, int kclass, cudaStream_t s) {
  using namespace tc;
  ProfScope prof_scope(kclass, s);
  const bool bf = split == TC_BF16_PAIR;
  Args g{};
  g.nsrc = nsrc;
  g.presplit = split != TC_FP32;
  for (int i = 0; i < nsrc; ++i) {
    const TcSrc& q = src[i];
    RR_TRY(make_map(&g.src[i].tmA, q.X, M, q.K, q.ldx, BM));
    if (bf) {
      RR_TRY(make_map_bf16(&g.src[i].tmB, static_cast<const uint16_t*>(q.hi), n, q.K, q.ldw, NT2));
      RR_TRY(make_map_bf16(&g.src[i].tmBlo, static_cast<const uint16_t*>(q.lo), n, q.K, q.ldw, NT2));
    } else {
      RR_TRY(make_map(&g.src[i].tmB, static_cast<const float*>(q.hi), n, q.K, q.ldw, NT2));
      if (g.presplit) RR_TRY(make_map(&g.src[i].tmBlo, static_cast<const float*>(q.lo), n, q.K, q.ldw, NT2));
    }
    g.src[i].K = q.K;
  }
  g.M = M;
  g.N = n;
  g.C = Y;
  g.ldc = ldy;
  g.bias = bias;
  g.resid = resid;
  g.ldr = ldr;
  g.relu = relu;
  g.accumulate = accumulate;
  g.p = p;
  g.inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  g.seed = seed;
  g.stream_id = stream_id;
  static PerDeviceOnce attr_set;
  if (attr_set.need()) {
    RR_CUDA(cudaFuncSetAttribute(k_tc_gemm2<16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    RR_CUDA(cudaFuncSetAttribute(k_tc_gemm2<16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    attr_set.mark();
  }
  // ring | barriers | epilogue staging (16 warps x 2 KB)
  const size_t smem = static_cast<size_t>(bf ? S2_BF * STAGE2_BF : S2 * STAGE2) + 1024 + 256 + 16 * 2048;
  const int total_tiles = ((M + BM - 1) / BM) * ((n + NT2 - 1) / NT2);
  const int ctas = total_tiles < num_sms() ? total_tiles : num_sms();
  RR_CUDA(launch_pdl(bf ? k_tc_gemm2<16, true> : k_tc_gemm2<16, false>, dim3(ctas), dim3(THREADS2_BASE + 512), smem, s, g));
  RR_LAUNCH_CHECK(bf ? "k_tc_gemm2<bf16>" : "k_tc_gemm2");
  return RR_OK;
}

// ---- images for the stand-alone tensor-core dgrad (C ABI: rr_linear_dgrad_tc) ---------------------------------------------------------
// The model keeps the transposed, pre-split operand images of every weight in its packed workspace (k_pack).  A direct caller of the C ABI
// hands over W[n, k] only, so the images are made here, into caller-provided scratch: Wt[k, ldt] as TF32 (hi, lo) floats and bf16 (hi, lo).
__global__ void k_transpose_split(const float* __restrict__ W, int n, int k, int ldw, float* __restrict__ thi, float* __restrict__ tlo,
                                  uint16_t* __restrict__ bhi, uint16_t* __restrict__ blo, int ldt) {
  const long long total = static_cast<long long>(n) * k;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / k), c = static_cast<int>(i - static_cast<long long>(r) * k);
    const float v = W[static_cast<size_t>(r) * ldw + c];
    const size_t o = static_cast<size_t>(c) * ldt + r;
    const float hi = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);
    thi[o] = hi;
    tlo[o] = v - hi;
    uint16_t b1, b2;
    asm("cvt.rn.bf16.f32 %0, %1;" : "=h"(b1) : "f"(v));
    asm("cvt.rn.bf16.f32 %0, %1;" : "=h"(b2) : "f"(v - __uint_as_float(static_cast<uint32_t>(b1) << 16)));
    bhi[o] = b1;
    blo[o] = b2;
  }
}
// bytes of one TF32 image and of one bf16 image of Wt[k, ldt], each rounded up to 256
static void dgrad_image_bytes(int n, int k, int* ldt, size_t* fb, size_t* hb) {
  *ldt = (n + 7) / 8 * 8;
  const size_t e = static_cast<size_t>(k) * *ldt;
  *fb = (e * 4 + 255) / 256 * 256;
  *hb = (e * 2 + 255) / 256 * 256;
}
long long tc_dgrad_scratch_bytes(int n, int k) {
  int ldt;
  size_t fb, hb;
  dgrad_image_bytes(n, k, &ldt, &fb, &hb);
  return static_cast<long long>(2 * fb + 2 * hb);
}
WeightImages tc_dgrad_images(int n, int k, void* scratch, int* ldt) {
  size_t fb, hb;
  dgrad_image_bytes(n, k, ldt, &fb, &hb);
  char* base = static_cast<char*>(scratch);
  WeightImages img;
  img.tf32_hi = reinterpret_cast<float*>(base);
  img.tf32_lo = reinterpret_cast<float*>(base + fb);
  img.bf16_hi = reinterpret_cast<uint16_t*>(base + 2 * fb);
  img.bf16_lo = reinterpret_cast<uint16_t*>(base + 2 * fb + hb);
  img.base = img.tf32_hi;   // no fp32 copy of Wt is kept: the images are indexed like the hi image
  return img;
}
int tc_transpose_split(const float* W, int n, int k, int ldw, const WeightImages& img, int ldt, cudaStream_t s) {
  RR_CUDA(cudaMemsetAsync(img.tf32_hi, 0, tc_dgrad_scratch_bytes(n, k), s));   // the padding columns of every image are zero
  const long long total = static_cast<long long>(n) * k;
  int blocks = static_cast<int>((total + 255) / 256);
  if (blocks > num_sms() * 8) blocks = num_sms() * 8;
  k_transpose_split<<<blocks, 256, 0, s>>>(W, n, k, ldw, img.tf32_hi, img.tf32_lo, img.bf16_hi, img.bf16_lo, ldt);
  RR_LAUNCH_CHECK("k_transpose_split");
  return RR_OK;
}

// ---- weight gradient ----------------------------------------------------------------------------------------------------------------
bool tc_wgrad_supported(int M, int n, int k, int lddz, int ldx) {
  return M > 0 && n >= 4 && k >= 4 && !(n & 3) && !(k & 3) && !(lddz & 3) && !(ldx & 3);
}

// One CTA per SM (shared memory and TMEM are both taken whole): never more CTAs than SMs, or the stragglers run as a second wave.  Rounding
// the slab height up to whole stages only lowers the count, so the count before rounding bounds that of every stage height.
int tc_wgrad_splits(int M, int n, int k, int stage_rows, int* chunk) {
  using namespace tc;
  const int k_pad = (k + 15) / 16 * 16;
  const int tiles = ((n + BM - 1) / BM) * ((k_pad + MAX_NT - 1) / MAX_NT);
  int splits = num_sms() / tiles;
  const int max_splits = (M + 8 * WG_BK - 1) / (8 * WG_BK);
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  if (stage_rows <= 0) return splits;
  *chunk = ((M + splits - 1) / splits + stage_rows - 1) / stage_rows * stage_rows;   // a stage never reaches into the next slab's rows
  return (M + *chunk - 1) / *chunk;
}

int tc_wgrad(bool bf16, int M, int n, int k, const float* dZ, int lddz, const float* X, int ldx, float* dW, int lddw, float* dbias, cudaStream_t s,
             float* slab, int* n_splits) {
  using namespace tc;
  ProfScope prof_scope(KC_GEMM_WGRAD, s);
  WgArgs g{};
  const int k_pad = (k + 15) / 16 * 16;                  // columns past k are zero-filled by TMA and never written back
  const int ktiles = (k_pad + MAX_NT - 1) / MAX_NT;
  g.kt = ktiles == 1 ? k_pad : MAX_NT;
  g.nb = (g.kt + 31) / 32;
  g.tm_a = g.kt <= 160 ? 160 : 320;
  // the ring: rows of the reduction per stage (bkr), slots and shared memory, and the instantiation
  int bkr, stage_rows, threads;
  size_t smem;
  CUtensorMapSwizzle x_swizzle;
  void (*kernel)(WgArgs);
  if (bf16) {
    // 3 x bf16: raw ring (dZ + X boxes as TMA lands them, up to 6 slots) and bf16 ring (hi + lo images + the TMEM A slots, 2 slots),
    // sized separately.  Narrow X tiles (<= 96 columns: the feature-matrix gradients W_i, W_o[:, :64], MPNDiff W_h[:, h:]) take 64 rows per
    // stage: a stage's hand-offs and fixed conversion cost (~1400 clk, DESIGN.md §4.2) are then paid half as often, and two
    // 56 KB raw slots still fit.
    bkr = g.kt <= 96 ? 64 : 32;
    const int box = bkr * 128;
    const int nblk = (g.kt + 63) / 64;
    const int raw_bytes = 4 * box + g.nb * box, bf_bytes = 2 * nblk * box;
    int R = 6, SB = 2;
    if (SB > (512 - g.tm_a) / bkr) SB = (512 - g.tm_a) / bkr;       // TMEM: accumulator + bkr columns of A per bf16 slot
    while (SB > 1 && 2 * raw_bytes + SB * bf_bytes > SMEM_LIMIT - 2048) --SB;
    const int Rmax = (SMEM_LIMIT - 2048 - SB * bf_bytes) / raw_bytes;
    if (R > Rmax) R = Rmax;
    RR_REQUIRE(R >= 2, "tc_wgrad: %d columns do not fit two raw pipeline slots", g.kt);
    g.stages = R;
    g.bf_stages = SB;
    smem = static_cast<size_t>(R) * raw_bytes + static_cast<size_t>(SB) * bf_bytes + 1024 + 512;
    stage_rows = bkr;
    threads = W3_THREADS;
    x_swizzle = CU_TENSOR_MAP_SWIZZLE_128B;
    if (bkr == 32) kernel = slab ? k_tc_wgrad3<32, true> : k_tc_wgrad3<32, false>;
    else kernel = slab ? k_tc_wgrad3<64, true> : k_tc_wgrad3<64, false>;
  } else {
    // 3 x TF32 (rr_set_backward_bf16(0)): wide tiles take 16-row stages (4 x 48 KB in flight instead of 2 x 96 KB); narrow tiles fit 3+
    // stages of 32 rows
    bkr = g.kt > 160 ? 16 : 32;
    const int box = bkr * 128;
    const int stage_bytes = 4 * box + 2 * g.nb * box;
    int S = (SMEM_LIMIT - 2048) / stage_bytes;
    if (S > (512 - g.tm_a) / (2 * bkr)) S = (512 - g.tm_a) / (2 * bkr);   // TMEM: accumulator + 2 * bkr columns of A per stage
    if (S > 6) S = 6;
    RR_REQUIRE(S >= 2, "tc_wgrad: %d columns do not fit two pipeline stages", g.kt);
    g.stages = S;
    smem = static_cast<size_t>(S) * stage_bytes + 1024 + 256;
    stage_rows = WG_BK;
    threads = THREADS;
    x_swizzle = CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
    if (bkr == 32) kernel = slab ? k_tc_wgrad2<32, true> : k_tc_wgrad2<32, false>;
    else kernel = slab ? k_tc_wgrad2<16, true> : k_tc_wgrad2<16, false>;
  }
  RR_TRY(make_map(&g.tmA, dZ, M, n, lddz, bkr, CU_TENSOR_MAP_SWIZZLE_NONE));
  RR_TRY(make_map(&g.tmB, X, M, k, ldx, bkr, x_swizzle));
  g.M = M;
  g.n = n;
  g.k = k;
  g.k_pad = k_pad;
  g.dW = dW;
  g.lddw = lddw;
  g.dbias = dbias;
  g.slab_stride = static_cast<long long>(n) * k;
  int chunk = 0;
  const int splits = tc_wgrad_splits(M, n, k, stage_rows, &chunk);
  g.m_chunk = chunk;
  if (slab) {
    g.dW = slab;
    g.lddw = k;
    if (dbias) g.dbias = slab + splits * g.slab_stride;   // bias partials follow the slab tiles
    *n_splits = splits;
  }
  static PerDeviceOnce attr_set;
  if (attr_set.need()) {
    void (*const all[])(WgArgs) = {k_tc_wgrad2<16, false>, k_tc_wgrad2<32, false>, k_tc_wgrad2<16, true>, k_tc_wgrad2<32, true>,
                                   k_tc_wgrad3<32, false>, k_tc_wgrad3<64, false>, k_tc_wgrad3<32, true>, k_tc_wgrad3<64, true>};
    for (auto* f : all) RR_CUDA(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    attr_set.mark();
  }
  RR_CUDA(launch_pdl(kernel, dim3((n + BM - 1) / BM, ktiles, splits), dim3(threads), smem, s, g));
  RR_LAUNCH_CHECK(bf16 ? "k_tc_wgrad3" : "k_tc_wgrad2");
  return RR_OK;
}

}  // namespace rr
