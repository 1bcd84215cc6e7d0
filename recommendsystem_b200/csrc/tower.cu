// tower.cu — the AutoInt tower's part of the bf16 train step in ONE launch (sm_100a), one CTA per 128-row block:
//   1. H0  = relu(X W0 + b0)                        -> H0, and a bf16 copy in TMEM (A operand of 2.)
//   2. H1  = relu(H0 W1 + b1)                       -> Z[:, :N1]
//   3. p   = sigmoid(Z w + b); dz = d BCE(clip(p)) / d logit   (as logit_head_kernel, head.cu)
//          -> p_out;  dZ = dz w, with dZ[:, :N1] multiplied by relu'(H1) (= dH1, also copied to TMEM)
//   4. dH0 = (dH1 W1^T) * relu'(H0)                 -> dH0, and a TMEM copy (A operand of 5.)
//   5. dX  = dH0 W0^T                               -> dX (plain store; the InteractingLayer backward adds its own part)
// The five products of the separate path (4 GEMM launches + the head pass) each paid a TMA pipeline fill, a TMEM
// epilogue and an HBM round trip of their output; here the activations stay in TMEM between the steps and only the
// tensors the rest of the step reads are written.  The head's own parameter gradients (Z^T dz, sum dz) and the loss
// are left to rs_logit_head_grad, a side branch: nothing on the critical chain needs them.
//
//   warp 0      TMA producer: one ring of 48 KB stages carries every operand the MMAs read from shared memory, in
//               the order they are consumed (X | W0^T slabs, the interacting half of Z, W1^T, W1, W0)
//   warp 1      TMEM allocator + MMA issuer (one thread)
//   warps 2..5  epilogues: a thread owns one row (TMEM lane); results go through SWIZZLE_128B staging slabs to TMA
//               stores (two buffers of 2 slabs, alternating)
//
// TMEM (512 columns):  [0, 256)   H0 accumulator, then dH0 accumulator, then dX chunk buffers 0 / 1
//                      [256, 384) head logit (2 columns), then H1 accumulator, then dH1 (bf16), then dH0 (bf16)
//                      [384, 512) H0 (bf16), then dX chunk buffer 2
// The Z·w dot of the interacting half runs on the tensor core: B = [w_hi; w_lo] (w = w_hi + w_lo to ~2^-17, both
// bf16), so it keeps the fp32 weight's precision.
#include "tc_common.cuh"

namespace rs {

constexpr int TW_THREADS = 192;
constexpr int TW_BM = 128;
constexpr int TW_N0 = 256;                     // hidden widths this kernel is laid out for
constexpr int TW_N1 = 128;
constexpr int TW_SLAB = TW_BM * 64 * 2;        // [128 rows][64 bf16] = one SWIZZLE_128B box, 16 KB
constexpr int TW_STAGES = 3;
constexpr int TW_STAGE = 3 * TW_SLAB;          // X slab + W0^T slab [256 rows][64]
constexpr int TW_OFF_STG = TW_STAGES * TW_STAGE;
constexpr int TW_STG_BYTES = 4 * TW_SLAB;
constexpr int TW_OFF_WS = TW_OFF_STG + TW_STG_BYTES;
constexpr uint32_t C_ACC0 = 0, C_ACC1 = 256, C_DH1 = 256, C_DH0 = 256, C_H0 = 384;

enum { B_ACC0, B_HEAD, B_ACC1, B_ACC4, B_WS, B_H0, B_DH1, B_DH0, B_XF, B_XE = B_XF + 3, B_COUNT = B_XE + 3 };
constexpr int TW_NBAR = 2 * TW_STAGES + B_COUNT;

struct TowerMaps {
  CUtensorMap x, w0t, w1t, w1, w0, z, dz, h0, dh0, dx;
};

__host__ __device__ inline int tower_kpad(int Ki) { return (Ki + 63) / 64 * 64; }
// ring | staging | [w_hi; w_lo] tile (8 rows x Kpad) | w (N1 + Kpad floats) | barriers
static size_t tower_smem_bytes(int Ki) {
  const int kp = tower_kpad(Ki);
  return (size_t)TW_OFF_WS + (size_t)kp * 16 + (size_t)(TW_N1 + kp) * 4 + TW_NBAR * 8 + 16 + 1024;
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// 16-byte chunk `c` (8 bf16 columns) of row `row` of a SWIZZLE_128B [128][64] bf16 slab
__device__ __forceinline__ void stg_put(uint8_t* slab, int row, int c, uint32_t a, uint32_t b, uint32_t d, uint32_t e) {
  *reinterpret_cast<uint4*>(slab + row * 128 + ((c ^ (row & 7)) << 4)) = make_uint4(a, b, d, e);
}
__device__ __forceinline__ float lo_bf(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float hi_bf(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }

__global__ void __launch_bounds__(TW_THREADS, 1)
tower_step_kernel(const __grid_constant__ TowerMaps tm, const float* __restrict__ b0, const float* __restrict__ b1,
                  const float* __restrict__ w, const float* __restrict__ ob, const float* __restrict__ y, float a,
                  __nv_bfloat16* __restrict__ p_out, int B, int K0, int Ki) {
  extern __shared__ uint8_t tw_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(tw_smem_raw) + 1023) & ~(uintptr_t)1023);
  const int kpad = tower_kpad(Ki);
  uint8_t* ring = smem;
  uint8_t* stg = smem + TW_OFF_STG;
  uint8_t* wsp = smem + TW_OFF_WS;                                   // [w_hi; w_lo; 0 x 6] no-swizzle K-major tile
  float* w_s = reinterpret_cast<float*>(wsp + kpad * 16);
  uint64_t* full = reinterpret_cast<uint64_t*>(w_s + TW_N1 + kpad);
  uint64_t* empty = full + TW_STAGES;
  uint64_t* bar = empty + TW_STAGES;                                 // B_*
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + B_COUNT);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * TW_BM;
  const int nk0 = (K0 + 63) / 64, nki = kpad / 64, nch = (K0 + 127) / 128;

  if (threadIdx.x == 0) {
    for (int s = 0; s < TW_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int i = 0; i < B_COUNT; ++i) {
      const bool from_epilogue = i == B_WS || i == B_H0 || i == B_DH1 || i == B_DH0 || i >= B_XE;
      mbar_init(&bar[i], from_epilogue ? 4 : 1);                      // epilogue: one arrival per warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    fence_async_smem();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int it = 0;
      auto slot = [&](uint32_t bytes) {
        const int s = it % TW_STAGES;
        mbar_wait(&empty[s], ((uint32_t)(it / TW_STAGES) & 1u) ^ 1u);
        mbar_expect_tx(&full[s], bytes);
        ++it;
        return s;
      };
      for (int kb = 0; kb < nk0; ++kb) {
        const int s = slot(3 * TW_SLAB);
        tma_load_2d(ring + s * TW_STAGE, &tm.x, &full[s], kb * 64, m0);
        tma_load_2d(ring + s * TW_STAGE + TW_SLAB, &tm.w0t, &full[s], kb * 64, 0);
      }
      for (int kb = 0; kb < nki; ++kb) {
        const int s = slot(TW_SLAB);
        tma_load_2d(ring + s * TW_STAGE, &tm.z, &full[s], TW_N1 + kb * 64, m0);
      }
      for (int kb = 0; kb < TW_N0 / 64; ++kb) {
        const int s = slot(TW_SLAB);
        tma_load_2d(ring + s * TW_STAGE, &tm.w1t, &full[s], kb * 64, 0);
      }
      for (int kb = 0; kb < TW_N1 / 64; ++kb) {
        const int s = slot(2 * TW_SLAB);
        tma_load_2d(ring + s * TW_STAGE, &tm.w1, &full[s], kb * 64, 0);
      }
      for (int ch = 0; ch < nch; ++ch)
        for (int kb = 0; kb < TW_N0 / 64; ++kb) {
          const int s = slot(TW_SLAB);
          tma_load_2d(ring + s * TW_STAGE, &tm.w0, &full[s], kb * 64, ch * 128);
        }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t ID256 = make_idesc_bf16(TW_BM, 256), ID128 = make_idesc_bf16(TW_BM, 128),
                         ID16 = make_idesc_bf16(TW_BM, 16);
      int it = 0;
      auto take = [&]() {
        const int s = it % TW_STAGES;
        mbar_wait(&full[s], (uint32_t)(it / TW_STAGES) & 1u);
        tc_fence_after();
        ++it;
        return s;
      };
      // 1. X W0 -> [0, 256)
      for (int kb = 0; kb < nk0; ++kb) {
        const int s = take();
        const uint32_t sa = smem_u32(ring + s * TW_STAGE);
        const uint64_t ad = make_sw128_kmajor_desc(sa), bd = make_sw128_kmajor_desc(sa + TW_SLAB);
#pragma unroll
        for (int k = 0; k < 4; ++k) tc_mma_bf16(tmem + C_ACC0, ad + 2 * k, bd + 2 * k, ID256, (kb | k) ? 1u : 0u);
        tc_commit(&empty[s]);
      }
      tc_commit(&bar[B_ACC0]);
      // 3a. Z[:, N1:] [w_hi w_lo] -> [256, 258); rows 8..15 of B alias rows 0..7 (SBO 0), their columns are unused
      mbar_wait(&bar[B_WS], 0);
      tc_fence_after();
      const uint32_t wsa = smem_u32(wsp);
      for (int kb = 0; kb < nki; ++kb) {
        const int s = take();
        const uint64_t ad = make_sw128_kmajor_desc(smem_u32(ring + s * TW_STAGE));
#pragma unroll
        for (int k = 0; k < 4; ++k)
          tc_mma_bf16(tmem + C_ACC1, ad + 2 * k, make_nosw_desc(wsa + (kb * 4 + k) * 256, 128, 0), ID16,
                      (kb | k) ? 1u : 0u);
        tc_commit(&empty[s]);
      }
      tc_commit(&bar[B_HEAD]);
      // 2. H0 W1 -> [256, 384), A = bf16 H0 in TMEM
      mbar_wait(&bar[B_H0], 0);
      tc_fence_after();
      for (int kb = 0; kb < TW_N0 / 64; ++kb) {
        const int s = take();
        const uint64_t bd = make_sw128_kmajor_desc(smem_u32(ring + s * TW_STAGE));
#pragma unroll
        for (int k = 0; k < 4; ++k)
          tc_mma_bf16_ts(tmem + C_ACC1, tmem + C_H0 + kb * 32 + k * 8, bd + 2 * k, ID128, (kb | k) ? 1u : 0u);
        tc_commit(&empty[s]);
      }
      tc_commit(&bar[B_ACC1]);
      // 4. dH1 W1^T -> [0, 256)
      mbar_wait(&bar[B_DH1], 0);
      tc_fence_after();
      for (int kb = 0; kb < TW_N1 / 64; ++kb) {
        const int s = take();
        const uint64_t bd = make_sw128_kmajor_desc(smem_u32(ring + s * TW_STAGE));
#pragma unroll
        for (int k = 0; k < 4; ++k)
          tc_mma_bf16_ts(tmem + C_ACC0, tmem + C_DH1 + kb * 32 + k * 8, bd + 2 * k, ID256, (kb | k) ? 1u : 0u);
        tc_commit(&empty[s]);
      }
      tc_commit(&bar[B_ACC4]);
      // 5. dH0 W0^T, 128 output columns per chunk, three TMEM buffers
      mbar_wait(&bar[B_DH0], 0);
      tc_fence_after();
      for (int ch = 0; ch < nch; ++ch) {
        const int buf = ch % 3, u = ch / 3;
        const uint32_t col = buf == 0 ? 0u : buf == 1 ? 128u : 384u;
        if (u > 0) {
          mbar_wait(&bar[B_XE + buf], (uint32_t)(u - 1) & 1u);
          tc_fence_after();
        }
        for (int kb = 0; kb < TW_N0 / 64; ++kb) {
          const int s = take();
          const uint64_t bd = make_sw128_kmajor_desc(smem_u32(ring + s * TW_STAGE));
#pragma unroll
          for (int k = 0; k < 4; ++k)
            tc_mma_bf16_ts(tmem + col, tmem + C_DH0 + kb * 32 + k * 8, bd + 2 * k, ID128, (kb | k) ? 1u : 0u);
          tc_commit(&empty[s]);
        }
        tc_commit(&bar[B_XF + buf]);
      }
    }
  } else {
    const int lg = warp & 3, row = lg * 32 + lane, et = threadIdx.x - 64;
    const int64_t grow = (int64_t)m0 + row;
    const uint32_t tl = tmem + ((uint32_t)(lg * 32) << 16);
    // head weights: the [w_hi; w_lo] B tile of 3a (core matrix = 8 rows x 8 k, 128 B; K chunks 128 B apart) and w
    for (int i = et; i < kpad; i += 128) {            // i = (16-byte K chunk, row) of the 8-row tile
      const int c = i >> 3, n = i & 7;
      uint32_t v[4] = {0u, 0u, 0u, 0u};
      if (n < 2) {
#pragma unroll
        for (int e = 0; e < 8; e += 2) {
          float q[2];
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            const int k = c * 8 + e + t;
            const float wv = k < Ki ? w[TW_N1 + k] : 0.f;
            const float hi = __bfloat162float(__float2bfloat16_rn(wv));
            q[t] = n == 0 ? hi : wv - hi;
          }
          v[e / 2] = pack_bf16x2(q[0], q[1]);
        }
      }
      *reinterpret_cast<uint4*>(wsp + c * 128 + n * 16) = make_uint4(v[0], v[1], v[2], v[3]);
    }
    for (int i = et; i < TW_N1 + kpad; i += 128) w_s[i] = i < TW_N1 + Ki ? w[i] : 0.f;
    fence_async_smem();
    named_bar_sync(1, 128);
    if (lane == 0) mbar_arrive(&bar[B_WS]);

    // store passes: pass n stages into buffer n & 1 (2 slabs); before it is rewritten, the TMA store issued from it
    // two passes ago must have read it
    int sp = 0;
    auto pass_begin = [&]() {
      if (et == 0) bulk_wait_read1();
      named_bar_sync(1, 128);
      return stg + (sp & 1) * 2 * TW_SLAB;
    };
    auto pass_end = [&]() {
      fence_async_smem();
      named_bar_sync(1, 128);
      ++sp;
    };

    // ---- 1. H0 = relu(acc + b0) -> global + TMEM (bf16)
    mbar_wait(&bar[B_ACC0], 0);
    tc_fence_after();
    for (int p = 0; p < 2; ++p) {
      uint8_t* sb = pass_begin();
#pragma unroll
      for (int c0 = 0; c0 < 128; c0 += 32) {
        const int c = p * 128 + c0;
        uint32_t r[32], h[16];
        tc_ld_32x32(tl + C_ACC0 + c, r);
#pragma unroll
        for (int j = 0; j < 16; ++j)
          h[j] = pack_bf16x2(fmaxf(__uint_as_float(r[2 * j]) + __ldg(b0 + c + 2 * j), 0.f),
                             fmaxf(__uint_as_float(r[2 * j + 1]) + __ldg(b0 + c + 2 * j + 1), 0.f));
        tc_st_32x16(tl + C_H0 + c / 2, h);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          stg_put(sb + (c0 >> 6) * TW_SLAB, row, ((c0 & 63) >> 3) + q, h[4 * q], h[4 * q + 1], h[4 * q + 2], h[4 * q + 3]);
      }
      pass_end();
      if (et == 0) {
        tma_store_2d(&tm.h0, sb, p * 128, m0);
        tma_store_2d(&tm.h0, sb + TW_SLAB, p * 128 + 64, m0);
        bulk_commit();
      }
    }
    tc_wait_st();
    // the interacting half's logit part leaves TMEM before the H1 accumulator takes its columns
    mbar_wait(&bar[B_HEAD], 0);
    tc_fence_after();
    float zi_dot;
    {
      uint32_t hr[8];
      tc_ld_32x8(tl + C_ACC1, hr);
      tc_wait_ld();
      zi_dot = __uint_as_float(hr[0]) + __uint_as_float(hr[1]);
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&bar[B_H0]);

    // ---- 2./3. H1 = relu(acc + b1) -> Z[:, :N1]; logit, p, dz
    mbar_wait(&bar[B_ACC1], 0);
    tc_fence_after();
    float dot = 0.f;
    uint32_t mask[TW_N1 / 32];
    {
      uint8_t* sb = pass_begin();
#pragma unroll
      for (int c0 = 0; c0 < TW_N1; c0 += 32) {
        uint32_t r[32], h[16], m = 0;
        tc_ld_32x32(tl + C_ACC1 + c0, r);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          h[j] = pack_bf16x2(fmaxf(__uint_as_float(r[2 * j]) + __ldg(b1 + c0 + 2 * j), 0.f),
                             fmaxf(__uint_as_float(r[2 * j + 1]) + __ldg(b1 + c0 + 2 * j + 1), 0.f));
          const float q0 = lo_bf(h[j]), q1 = hi_bf(h[j]);
          dot = fmaf(q0, w_s[c0 + 2 * j], dot);
          dot = fmaf(q1, w_s[c0 + 2 * j + 1], dot);
          m |= (q0 > 0.f ? 1u : 0u) << (2 * j);
          m |= (q1 > 0.f ? 1u : 0u) << (2 * j + 1);
        }
        mask[c0 / 32] = m;
#pragma unroll
        for (int q = 0; q < 4; ++q)
          stg_put(sb + (c0 >> 6) * TW_SLAB, row, ((c0 & 63) >> 3) + q, h[4 * q], h[4 * q + 1], h[4 * q + 2], h[4 * q + 3]);
      }
      pass_end();
      if (et == 0) {
        tma_store_2d(&tm.z, sb, 0, m0);
        tma_store_2d(&tm.z, sb + TW_SLAB, 64, m0);
        bulk_commit();
      }
    }
    const bool live = grow < B;
    const float pr = 1.f / (1.f + expf(-(dot + zi_dot + __ldg(ob))));
    const float prs = __bfloat162float(__float2bfloat16_rn(pr));   // the stored activation
    const float pc = fminf(fmaxf(prs, 1e-6f), 1.0f);
    const float yy = live ? y[grow] : 0.f;
    const float dp = (-yy / (pc + 1e-6f) + (a - yy) / (1.0f - pc + 1e-6f)) * (1.f / (float)B);
    const float dz = (live && prs >= 1e-6f && prs <= 1.0f) ? dp * prs * (1.f - prs) : 0.f;
    if (live) p_out[grow] = __float2bfloat16_rn(pr);
    // dH1 = dz w[:N1] relu'(H1) -> dZ[:, :N1] + TMEM
    {
      uint8_t* sb = pass_begin();
#pragma unroll
      for (int c0 = 0; c0 < TW_N1; c0 += 32) {
        uint32_t g[16];
#pragma unroll
        for (int j = 0; j < 16; ++j)
          g[j] = pack_bf16x2((mask[c0 / 32] >> (2 * j)) & 1u ? dz * w_s[c0 + 2 * j] : 0.f,
                             (mask[c0 / 32] >> (2 * j + 1)) & 1u ? dz * w_s[c0 + 2 * j + 1] : 0.f);
        tc_st_32x16(tl + C_DH1 + c0 / 2, g);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          stg_put(sb + (c0 >> 6) * TW_SLAB, row, ((c0 & 63) >> 3) + q, g[4 * q], g[4 * q + 1], g[4 * q + 2], g[4 * q + 3]);
      }
      pass_end();
      if (et == 0) {
        tma_store_2d(&tm.dz, sb, 0, m0);
        tma_store_2d(&tm.dz, sb + TW_SLAB, 64, m0);
        bulk_commit();
      }
    }
    tc_wait_st();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&bar[B_DH1]);
    // dZ[:, N1:] = dz w[N1:] (what the InteractingLayer backward reads), while the MMAs of 4. run
    for (int s0 = 0; s0 < nki; s0 += 2) {
      uint8_t* sb = pass_begin();
      const int ns = min(2, nki - s0);
      for (int sl = 0; sl < ns; ++sl) {
        const float* wc = w_s + TW_N1 + (s0 + sl) * 64;
#pragma unroll
        for (int q = 0; q < 8; ++q)
          stg_put(sb + sl * TW_SLAB, row, q, pack_bf16x2(dz * wc[q * 8 + 0], dz * wc[q * 8 + 1]),
                  pack_bf16x2(dz * wc[q * 8 + 2], dz * wc[q * 8 + 3]), pack_bf16x2(dz * wc[q * 8 + 4], dz * wc[q * 8 + 5]),
                  pack_bf16x2(dz * wc[q * 8 + 6], dz * wc[q * 8 + 7]));
      }
      pass_end();
      if (et == 0) {
        for (int sl = 0; sl < ns; ++sl) tma_store_2d(&tm.dz, sb + sl * TW_SLAB, TW_N1 + (s0 + sl) * 64, m0);
        bulk_commit();
      }
    }

    // ---- 4. dH0 = acc relu'(H0) -> global + TMEM (bf16)
    mbar_wait(&bar[B_ACC4], 0);
    tc_fence_after();
    for (int p = 0; p < 2; ++p) {
      uint8_t* sb = pass_begin();
#pragma unroll
      for (int c0 = 0; c0 < 128; c0 += 32) {
        const int c = p * 128 + c0;
        uint32_t r[32], hm[16], g[16];
        tc_ld_32x16(tl + C_H0 + c / 2, hm);
        tc_ld_32x32(tl + C_ACC0 + c, r);              // waits for both loads
#pragma unroll
        for (int j = 0; j < 16; ++j)
          g[j] = pack_bf16x2(lo_bf(hm[j]) > 0.f ? __uint_as_float(r[2 * j]) : 0.f,
                             hi_bf(hm[j]) > 0.f ? __uint_as_float(r[2 * j + 1]) : 0.f);
        tc_st_32x16(tl + C_DH0 + c / 2, g);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          stg_put(sb + (c0 >> 6) * TW_SLAB, row, ((c0 & 63) >> 3) + q, g[4 * q], g[4 * q + 1], g[4 * q + 2], g[4 * q + 3]);
      }
      pass_end();
      if (et == 0) {
        tma_store_2d(&tm.dh0, sb, p * 128, m0);
        tma_store_2d(&tm.dh0, sb + TW_SLAB, p * 128 + 64, m0);
        bulk_commit();
      }
    }
    tc_wait_st();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&bar[B_DH0]);

    // ---- 5. dX chunks -> global
    for (int ch = 0; ch < nch; ++ch) {
      const int buf = ch % 3;
      const uint32_t col = buf == 0 ? 0u : buf == 1 ? 128u : 384u;
      mbar_wait(&bar[B_XF + buf], (uint32_t)(ch / 3) & 1u);
      tc_fence_after();
      uint8_t* sb = pass_begin();
#pragma unroll
      for (int c0 = 0; c0 < 128; c0 += 32) {
        uint32_t r[32];
        tc_ld_32x32(tl + col + c0, r);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          stg_put(sb + (c0 >> 6) * TW_SLAB, row, ((c0 & 63) >> 3) + q,
                  pack_bf16x2(__uint_as_float(r[8 * q + 0]), __uint_as_float(r[8 * q + 1])),
                  pack_bf16x2(__uint_as_float(r[8 * q + 2]), __uint_as_float(r[8 * q + 3])),
                  pack_bf16x2(__uint_as_float(r[8 * q + 4]), __uint_as_float(r[8 * q + 5])),
                  pack_bf16x2(__uint_as_float(r[8 * q + 6]), __uint_as_float(r[8 * q + 7])));
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar[B_XE + buf]);
      pass_end();
      if (et == 0) {
        tma_store_2d(&tm.dx, sb, ch * 128, m0);
        if (ch * 128 + 64 < K0) tma_store_2d(&tm.dx, sb + TW_SLAB, ch * 128 + 64, m0);
        bulk_commit();
      }
    }
    if (et == 0) bulk_wait_all();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512));
  }
}

}  // namespace rs

using namespace rs;

extern "C" {

int rs_tower_supported(int K0, int N0, int N1, int Ki) {
  return N0 == TW_N0 && N1 == TW_N1 && K0 > 0 && K0 % 16 == 0 && Ki > 0 && Ki % 16 == 0 &&
         tower_smem_bytes(Ki) <= 232448;
}

int rs_tower_step(const void* X, const void* W0T, const void* W1T, const void* W0, const void* W1, const float* b0,
                  const float* b1, const float* w, const float* ob, const float* y, float a, void* Z, void* p_out,
                  void* dZ, void* H0, void* dH0, void* dX, int B, int K0, int N0, int N1, int Ki, void* stream) {
  RS_REQUIRE(B > 0 && rs_tower_supported(K0, N0, N1, Ki),
             "tower_step: B=%d K0=%d N0=%d N1=%d Ki=%d (N0 = %d, N1 = %d, K0 %% 16 == 0, Ki %% 16 == 0, Ki <= ~700)", B, K0,
             N0, N1, Ki, TW_N0, TW_N1);
  const void* ptrs[] = {X, W0T, W1T, W0, W1, Z, dZ, H0, dH0, dX};
  for (const void* p : ptrs) RS_REQUIRE(p != nullptr && (uintptr_t)p % 16 == 0, "tower_step: operands must be 16-byte aligned");
  const int zw = N1 + Ki;
  TowerMaps m;
  int e;
  if ((e = make_map(&m.x, X, B, K0, K0, TW_BM)) || (e = make_map(&m.w0t, W0T, N0, K0, K0, 256)) ||
      (e = make_map(&m.w1t, W1T, N1, N0, N0, TW_BM)) || (e = make_map(&m.w1, W1, N0, N1, N1, 256)) ||
      (e = make_map(&m.w0, W0, K0, N0, N0, TW_BM)) || (e = make_map(&m.z, Z, B, zw, zw, TW_BM)) ||
      (e = make_map(&m.dz, dZ, B, zw, zw, TW_BM)) || (e = make_map(&m.h0, H0, B, N0, N0, TW_BM)) ||
      (e = make_map(&m.dh0, dH0, B, N0, N0, TW_BM)) || (e = make_map(&m.dx, dX, B, K0, K0, TW_BM)))
    return e;
  const int smem = (int)tower_smem_bytes(Ki);
  RS_CUDA(cudaFuncSetAttribute(tower_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  tower_step_kernel<<<(unsigned)cdiv(B, TW_BM), TW_THREADS, smem, as_stream(stream)>>>(
      m, b0, b1, w, ob, y, a, (__nv_bfloat16*)p_out, B, K0, Ki);
  return check_launch("tower_step");
}

}  // extern "C"
