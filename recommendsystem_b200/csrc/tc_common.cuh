// tc_common.cuh — inline-PTX wrappers for the Blackwell tensor-core path (tcgen05 / TMEM / TMA /
// mbarrier) shared by the GEMM and the fused InteractingLayer kernels.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace rs {

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
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
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns -> 32 registers per thread (thread = lane = row).
__device__ __forceinline__ void tc_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
//   [0,14) start address >> 4 | [16,30) LBO >> 4 (ignored for swizzled K-major) | [32,46) SBO >> 4
//   (8 rows x 128 B = 1024 B between 8-row groups) | [46,48) version = 1 | [61,64) layout = 2 (SW128)
__device__ __forceinline__ uint64_t make_sw128_kmajor_desc(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// General SWIZZLE_128B descriptor (K-major: LBO ignored, SBO = 1024; MN-major: LBO = byte stride
// between 64-element M|N atoms, SBO = byte stride between 8-row K groups).
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): c=f32 (1<<4), a=b=bf16 (1<<7, 1<<10),
// both K-major, N>>3 at bit 17, M>>4 at bit 24.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}


// Host: TMA map of a 2-D bf16 row-major [rows, cols] tensor (leading dim ld elements), box = 64 cols x box_rows rows,
// SWIZZLE_128B (gemm_tc.cu).
int make_map(CUtensorMap* map, const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows);

// Generic-proxy shared-memory writes -> visible to the async proxy (tcgen05.mma / TMA reads).
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// No-swizzle shared-memory matrix descriptor.  Core matrix = 8 rows x 16 bytes stored contiguously
// (128 B).  K-major operand: LBO = byte distance between the core matrices adjacent along K,
// SBO = between 8-row groups along M/N.  MN-major operand: SBO = between core matrices adjacent
// along M/N, LBO = between 8-deep groups along K (cute::UMMA::make_umma_desc, INTERLEAVE layout).
__device__ __forceinline__ uint64_t make_nosw_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
}

// kind::f16 / kind::tf32 instruction descriptor: fmt 1 = bf16, 2 = tf32; major 0 = K, 1 = MN.
__host__ __device__ constexpr uint32_t make_idesc(int fmt, int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)a_mn_major << 15) |
         ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// 32 lanes x 8 / 16 consecutive columns.
__device__ __forceinline__ void tc_ld_32x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tc_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

constexpr float ITC_LOG2E = 1.4426950408889634f;

// byte offset of (row, 16-byte chunk c) in a no-swizzle tile whose rows hold NCH 16-byte chunks:
// [row/8][chunk][row%8][16 B].  The SAME bytes are a K-major operand (rows = M/N, chunks along K:
// LBO = 128, SBO = NCH*128) and an MN-major operand (chunks along M/N, rows = K: SBO = 128,
// LBO = NCH*128) — a tile written once can feed an MMA and its transpose.
template <int NCH>
__device__ __forceinline__ uint32_t nosw_off(int row, int c) {
  return (uint32_t)((row >> 3) * (NCH * 128) + c * 128 + (row & 7) * 16);
}

__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c);
__device__ __forceinline__ float2 fadd2(float2 a, float2 b);
__device__ __forceinline__ float2 fmul2(float2 a, float2 b);

// LayerNorm of one register row (InteractingLayer.py:60).  ONE definition, explicit fma/mul, shared by
// the tcgen05 forward and backward so that the backward's recomputed iteration input is bit-identical
// to what the forward fed to its next iteration.
template <int U>
__device__ __forceinline__ void ln_row_stats(const float (&a)[U], float eps, float& mean, float& rstd) {
  static_assert(U == 16 || U == 8, "pairwise tree written for 8 / 16 columns");
  // fixed pairwise trees (depth 4) instead of 16-deep dependent chains: at 2-3 warps per scheduler the chain
  // latency was exposed; the order is still fixed, so forward and backward agree bit for bit
  float2 t[U / 2];
#pragma unroll
  for (int i = 0; i < U / 2; ++i) t[i] = make_float2(a[2 * i], a[2 * i + 1]);
#pragma unroll
  for (int w = U / 4; w >= 1; w >>= 1)
#pragma unroll
    for (int i = 0; i < w; ++i) t[i] = fadd2(t[i], t[i + w]);
  const float m = __fmul_rn(__fadd_rn(t[0].x, t[0].y), 1.f / U);
  const float2 nm = make_float2(-m, -m);
#pragma unroll
  for (int i = 0; i < U / 2; ++i) {
    const float2 d = fadd2(make_float2(a[2 * i], a[2 * i + 1]), nm);
    t[i] = fmul2(d, d);
  }
#pragma unroll
  for (int w = U / 4; w >= 1; w >>= 1)
#pragma unroll
    for (int i = 0; i < w; ++i) t[i] = fadd2(t[i], t[i + w]);
  mean = m;
  rstd = rsqrtf(__fmaf_rn(__fadd_rn(t[0].x, t[0].y), 1.f / U, eps));
}
__device__ __forceinline__ float ln_apply(float a, float mean, float rstd, float gamma, float beta) {
  return __fmaf_rn(__fmul_rn(__fsub_rn(a, mean), rstd), gamma, beta);
}

// 3xTF32 split: hi = the value with the 13 low mantissa bits cleared (exactly a tf32 number whatever
// rounding the tensor core applies), lo = v - hi (exact in fp32; the MMA keeps its top 11 bits).
// x.w ~ hi.Whi + lo.Whi + hi.Wlo to ~2^-21 relative: fp32-grade pre-activations, so the ReLU masks of
// the projections agree with an fp32/fp64 evaluation of the layer.
__device__ __forceinline__ float tf32_hi(float v) { return __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }

// The projection Z[128, 64] = X[128, 16] W[16, 64] as six kind::tf32 MMAs (K = 8 each) over
// A = [x_hi | x_lo] (no-swizzle, 8 chunks/row) and B = W_hi, W_lo ([64 n][16 k], 4 chunks/row each,
// W_lo 4096 bytes after W_hi).
__device__ __forceinline__ void issue_proj_3xtf32(uint32_t tmem_z, uint32_t x_addr, uint32_t w_addr, uint32_t idesc) {
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    const int ka = j < 4 ? j : j - 4;            // A K-step: 0,1 = hi ; 2,3 = lo
    const int kb = j & 1;                        // B K-step
    const uint32_t wb = w_addr + (j >= 4 ? 4096u : 0u);
    tc_mma_tf32(tmem_z, make_nosw_desc(x_addr + ka * 256, 128, 1024), make_nosw_desc(wb + kb * 256, 128, 512), idesc,
                j ? 1u : 0u);
  }
}
// W[16][64] (row-major [in, out]) -> W_hi | W_lo operand tiles
__device__ __forceinline__ void stage_w_3xtf32(uint8_t* w_smem, const float* __restrict__ W, int tid, int nthreads) {
  for (int i = tid; i < 64 * 4; i += nthreads) {
    const int n = i >> 2, c = i & 3;
    float w[4], hi[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) { w[e] = W[(c * 4 + e) * 64 + n]; hi[e] = tf32_hi(w[e]); }
    *reinterpret_cast<float4*>(w_smem + nosw_off<4>(n, c)) = make_float4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<float4*>(w_smem + 4096 + nosw_off<4>(n, c)) =
        make_float4(w[0] - hi[0], w[1] - hi[1], w[2] - hi[2], w[3] - hi[3]);
  }
}
// 4 consecutive x values of tile row `row` starting at column 4*c -> chunk c (hi) and chunk 4 + c (lo)
__device__ __forceinline__ void stage_x4_3xtf32(uint8_t* x_smem, int row, int c, float a, float b, float cc, float d) {
  const float ha = tf32_hi(a), hb = tf32_hi(b), hc = tf32_hi(cc), hd = tf32_hi(d);
  *reinterpret_cast<float4*>(x_smem + nosw_off<8>(row, c)) = make_float4(ha, hb, hc, hd);
  *reinterpret_cast<float4*>(x_smem + nosw_off<8>(row, 4 + c)) = make_float4(a - ha, b - hb, cc - hc, d - hd);
}

// No-swizzle descriptor from the tile base in 16-byte units (smem addresses are < 2^18, so the
// 14-bit start-address field needs no mask): one integer add per MMA operand.
__device__ __forceinline__ uint64_t mk_desc(uint32_t base16, uint32_t off_bytes, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  const uint32_t lo = (base16 + (off_bytes >> 4)) | ((lbo_bytes >> 4) << 16);
  const uint32_t hi = (sbo_bytes >> 4) | (1u << 14);
  return ((uint64_t)hi << 32) | lo;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Round two fp32 values to bf16 (RNE) and back.  ONE F2FP.PACK_AB (ALU pipe) + two integer unpacks; the
// scalar __float2bfloat16_rn compiles to F2F.BF16.F32, which shares the quarter-rate XU pipe with MUFU.EX2
// and made the softmax phases XU-bound (80 XU ops per 40 elements).
__device__ __forceinline__ void bf16_round2(float& a, float& b) {
  const uint32_t u = pack_bf16x2(a, b);
  a = __uint_as_float(u << 16);
  b = __uint_as_float(u & 0xFFFF0000u);
}


// ---- round-2 additions: TMEM-resident A operands (tcgen05.st + .mma [d], [a], bdesc), packed f32x2 math -------
__device__ __forceinline__ void tc_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tc_st_32x4(uint32_t taddr, const uint32_t (&r)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3])
               : "memory");
}
__device__ __forceinline__ void tc_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
      "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] . B[smem]: A rows = TMEM lanes, K along the columns (tf32: one value per column,
// bf16: two per column, even k in the low half); A cannot be transposed.
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc),
      "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc),
      "r"(accumulate)
      : "memory");
}
// Packed fp32 pairs (FFMA2 / FADD2 / FMUL2 on sm_100): two IEEE fp32 operations per instruction.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(reinterpret_cast<uint64_t&>(d))
      : "l"(reinterpret_cast<const uint64_t&>(a)), "l"(reinterpret_cast<const uint64_t&>(b)),
        "l"(reinterpret_cast<const uint64_t&>(c)));
  return d;
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  float2 d;
  asm("add.rn.f32x2 %0, %1, %2;"
      : "=l"(reinterpret_cast<uint64_t&>(d))
      : "l"(reinterpret_cast<const uint64_t&>(a)), "l"(reinterpret_cast<const uint64_t&>(b)));
  return d;
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  float2 d;
  asm("mul.rn.f32x2 %0, %1, %2;"
      : "=l"(reinterpret_cast<uint64_t&>(d))
      : "l"(reinterpret_cast<const uint64_t&>(a)), "l"(reinterpret_cast<const uint64_t&>(b)));
  return d;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
// warp index as a UNIFORM value (CREDUX -> uniform register): TMEM addresses, descriptors and warp-level loop
// bounds derived from it stay in the uniform datapath (tcgen05.ld/st/mma take uniform-register addresses; a
// threadIdx-derived base cost one R2UR per TMEM instruction)
__device__ __forceinline__ uint32_t uniform_u32(uint32_t v) { return __reduce_max_sync(0xffffffffu, v); }
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ float lg2_approx(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// Z[128, 64] = X[128, 16] W[16, 64] as 3xTF32 with A = [x_hi (16 columns) | x_lo (16 columns)] in TMEM.
__device__ __forceinline__ void issue_proj_3xtf32_ts(uint32_t tmem_z, uint32_t tmem_x, uint32_t w_addr, uint32_t idesc) {
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    const int ka = j < 4 ? j : j - 4;            // A K-step: 0,1 = hi ; 2,3 = lo
    const int kb = j & 1;                        // B K-step
    const uint32_t wb = w_addr + (j >= 4 ? 4096u : 0u);
    tc_mma_tf32_ts(tmem_z, tmem_x + ka * 8, make_nosw_desc(wb + kb * 256, 128, 512), idesc, j ? 1u : 0u);
  }
}

// samples per 128-row tile: whole samples of FP = 8 NCHF padded fields, at most 4 (the expanded Q operand has
// 8 SPT columns per head and the P.V product N = 8 SPT <= 32)
template <int NCHF> struct ItcGeom {
  static constexpr int FP = NCHF * 8;
  static constexpr int SPT = (128 / FP) < 4 ? (128 / FP) : 4;
  static constexpr int NCHK = SPT * 2;                 // 16-byte chunks per row of the expanded K operand (tf32)
  static constexpr int KP = (FP + 15) / 16 * 16;       // key dimension padded to the bf16 K step
  static constexpr int KX_BYTES = NCHF * NCHK * 128;   // [FP keys][8 SPT] tf32
  static constexpr int VX_BYTES = (KP / 8) * 512;      // [KP keys][32 = (sample, e)] bf16, MN-major
};

// bias through the MMA: B tile [64 n][8 k] tf32 with k = 0 -> b_hi[n], k = 1 -> b_lo[n]; the A operand carries
// the constant columns [1 1 0 0 0 0 0 0] next to [x_hi | x_lo]
__device__ __forceinline__ void stage_bias_tile(uint8_t* bt_smem, const float* __restrict__ bias, int tid, int nthreads) {
  for (int i = tid; i < 64 * 2; i += nthreads) {
    const int n = i >> 1, c = i & 1;
    const float bv = bias[n], bh = tf32_hi(bv);
    *reinterpret_cast<float4*>(bt_smem + nosw_off<2>(n, c)) =
        c ? make_float4(0.f, 0.f, 0.f, 0.f) : make_float4(bh, bv - bh, 0.f, 0.f);
  }
}

}  // namespace rs
