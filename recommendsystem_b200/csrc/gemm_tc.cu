// gemm_tc.cu — bf16 tensor-core GEMM for the MLP tower (K5) on sm_100a:
//   C[M,N] = epi( A[M,K] · B[N,K]^T )      A, B bf16 K-major; fp32 accumulation in TMEM.
//
// One CTA computes one 128 x BN output tile (optionally one K-split of it):
//   warp 0      TMA producer: cp.async.bulk.tensor 2-D tiles (64-element = 128-byte K slabs,
//               SWIZZLE_128B) of A and B into a 2-stage shared-memory ring (3 CTAs per SM), mbarrier expect_tx
//   warp 1      TMEM allocator + MMA issuer: one elected thread issues tcgen05.mma
//               (cta_group::1, kind::f16, M=128, N=BN, K=16) four times per stage and
//               tcgen05.commit's the stage back to the producer / the accumulator to the epilogue
//   warps 2..5  epilogue: tcgen05.ld (32 lanes x 32 columns per warp and step) -> registers ->
//               bias / activation / mask epilogue -> 16-byte global stores (a thread owns a row)
// Split-K (weight gradients: K = batch) writes fp32 partial tiles that a second kernel sums in
// split order (deterministic).  K tails and M/N tails rely on TMA zero fill + guarded stores.
#include "tc_common.cuh"

namespace rs {

constexpr int TC_BM = 128;
constexpr int TC_BK = 64;          // bf16 elements per stage along K = one 128-byte swizzle row
constexpr int TC_THREADS = 192;

#ifdef RS_GEMM_PROFILE
__device__ long long gemm_prof[16];
#define GPROF(i) if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) gemm_prof[i] = clock64();
#else
#define GPROF(i)
#endif


// ---- epilogue phase B: lane = column group of a staged [32 rows][BN] fp32 block; every warp instruction
// touches one contiguous row segment of C / aux.  Rows are unrolled by 4 so that the shared-memory and
// aux loads of four rows are in flight together; EPI is a compile-time constant here.
template <int BN, int EPI, typename CT>
__device__ __forceinline__ void epilogue_rows(const float* stg, int rows_here, int lane, int ncols, int N, CT* c_rows,
                                              int64_t ldc, const CT* a_rows, int64_t ldaux, const float* bias,
                                              int vec_ok) {
  constexpr int PITCH = BN + 4;
  constexpr int CPL = BN / 32;
  constexpr bool NEED_AUX = EPI == RS_EPI_MUL_RELU_MASK || EPI == RS_EPI_MUL_DSIGMOID;
  constexpr bool NEED_BIAS = EPI == RS_EPI_BIAS || EPI == RS_EPI_BIAS_RELU || EPI == RS_EPI_BIAS_SIGMOID;
  const int col = lane * CPL;
  if (col >= ncols) return;
  const bool lane_full = col + CPL <= ncols;
  const bool vec = vec_ok && lane_full && (CPL % 4) == 0;
  float bv[CPL];
#pragma unroll
  for (int e = 0; e < CPL; ++e) bv[e] = (NEED_BIAS && col + e < ncols) ? bias[col + e] : 0.f;
  constexpr int RU = 4;
  for (int r0 = 0; r0 < rows_here; r0 += RU) {
    float acc[RU][CPL], av[RU][CPL];
#pragma unroll
    for (int u = 0; u < RU; ++u) {
      const int rr = min(r0 + u, rows_here - 1);
#pragma unroll
      for (int e = 0; e < CPL; ++e) { acc[u][e] = stg[rr * PITCH + col + e]; av[u][e] = 0.f; }
      if (NEED_AUX || EPI == RS_EPI_ACCUM) {
        const CT* src = (NEED_AUX ? a_rows + (int64_t)rr * ldaux : c_rows + (int64_t)rr * ldc) + col;
        if (vec) {
          if constexpr (CPL % 4 == 0) {
#pragma unroll
            for (int q = 0; q < CPL; q += 4) {
              const float4 a4 = load4<CT>(src + q);
              av[u][q] = a4.x; av[u][q + 1] = a4.y; av[u][q + 2] = a4.z; av[u][q + 3] = a4.w;
            }
          }
        } else {
#pragma unroll
          for (int e = 0; e < CPL; ++e)
            if (col + e < ncols) av[u][e] = to_f<CT>(src[e]);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < RU; ++u) {
      if (r0 + u >= rows_here) break;
      float v[CPL];
#pragma unroll
      for (int e = 0; e < CPL; ++e) {
        const float a = acc[u][e];
        if (EPI == RS_EPI_BIAS) v[e] = a + bv[e];
        else if (EPI == RS_EPI_BIAS_RELU) v[e] = fmaxf(a + bv[e], 0.f);
        else if (EPI == RS_EPI_BIAS_SIGMOID) v[e] = 1.f / (1.f + __expf(-(a + bv[e])));
        else if (EPI == RS_EPI_MUL_RELU_MASK) v[e] = av[u][e] > 0.f ? a : 0.f;
        else if (EPI == RS_EPI_MUL_DSIGMOID) v[e] = a * av[u][e] * (1.f - av[u][e]);
        else if (EPI == RS_EPI_ACCUM) v[e] = a + av[u][e];
        else v[e] = a;
      }
      CT* crow = c_rows + (int64_t)(r0 + u) * ldc + col;
      if (vec) {
        if constexpr (CPL % 4 == 0) {
#pragma unroll
          for (int q = 0; q < CPL; q += 4) store4<CT>(crow + q, make_float4(v[q], v[q + 1], v[q + 2], v[q + 3]));
        }
      } else {
#pragma unroll
        for (int e = 0; e < CPL; ++e)
          if (col + e < ncols) crow[e] = from_f<CT>(v[e]);
      }
    }
  }
}

// RS_EPI_MUL_RELU_MASK on a full 32-row x 128-column bf16 block whose aux values (`pre`: this lane's four bf16 of each
// of the 32 rows) were loaded BEFORE the accumulator wait: the dgrad GEMMs of the tower are two K slabs deep, so eight
// dependent batches of aux loads after the MMAs (the generic path) cost more than the MMAs themselves.
template <int BN, typename CT>
__device__ __forceinline__ void epilogue_mask_pre(const float* stg, int lane, CT* c_rows, int64_t ldc,
                                                  const uint32_t (&pre)[64]) {
  static_assert(BN == 128 && sizeof(CT) == 2, "prefetched mask epilogue: 128-wide bf16 tiles");
  constexpr int PITCH = BN + 4;
  const int col = lane * 4;
#pragma unroll
  for (int rr = 0; rr < 32; ++rr) {
    const float4 a = *reinterpret_cast<const float4*>(stg + rr * PITCH + col);
    const uint32_t m01 = pre[2 * rr], m23 = pre[2 * rr + 1];
    float4 v;
    v.x = __uint_as_float(m01 << 16) > 0.f ? a.x : 0.f;
    v.y = __uint_as_float(m01 & 0xffff0000u) > 0.f ? a.y : 0.f;
    v.z = __uint_as_float(m23 << 16) > 0.f ? a.z : 0.f;
    v.w = __uint_as_float(m23 & 0xffff0000u) > 0.f ? a.w : 0.f;
    store4<CT>(c_rows + (int64_t)rr * ldc + col, v);
  }
}

// split-K partial tile rows (fp32, [splits][M][N])
template <int BN>
__device__ __forceinline__ void epilogue_partial(const float* stg, int rows_here, int lane, int ncols, int N, float* dst_rows) {
  constexpr int PITCH = BN + 4;
  constexpr int CPL = BN / 32;
  const int col = lane * CPL;
  if (col >= ncols) return;
  const bool vec = (col + CPL <= ncols) && (N % CPL) == 0;
#pragma unroll 4
  for (int rr = 0; rr < rows_here; ++rr) {
    float* dst = dst_rows + (int64_t)rr * N + col;
    const float* src = stg + rr * PITCH + col;
    if (vec) {
      if constexpr (CPL % 4 == 0) {
#pragma unroll
        for (int q = 0; q < CPL; q += 4)
          *reinterpret_cast<float4*>(dst + q) = *reinterpret_cast<const float4*>(src + q);
      } else if constexpr (CPL == 2) *reinterpret_cast<float2*>(dst) = make_float2(src[0], src[1]);
      else dst[0] = src[0];
    } else {
#pragma unroll
      for (int e = 0; e < CPL; ++e)
        if (col + e < ncols) dst[e] = src[e];
    }
  }
}

// STAGES: 6 (one CTA per SM, every K slab of a short-K GEMM in flight at once: the tile's time is ~2
// TMA round trips) when the grid is at most one wave; 2 (three CTAs per SM overlap each other's
// prologue / epilogue) when there are more tiles than SMs.
template <int BN, int STAGES>
struct TcSmem {
  static constexpr int A_BYTES = TC_BM * TC_BK * 2;   // 16 KB
  static constexpr int B_BYTES = BN * TC_BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STG_PITCH = BN + 4;                      // epilogue staging row pitch (floats)
  static constexpr int STG_BYTES = TC_BM * STG_PITCH * 4;       // [128 rows][BN + 4] fp32, reuses the stages
  static constexpr int MAIN_BYTES = STAGES * STAGE_BYTES > STG_BYTES ? STAGES * STAGE_BYTES : STG_BYTES;
  static constexpr int TOTAL = MAIN_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

template <int BN, int STAGES, bool MN, typename CT>
__global__ void __launch_bounds__(TC_THREADS, STAGES <= 2 ? 3 : 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               CT* __restrict__ C, int64_t ldc, const float* __restrict__ bias,
               const CT* __restrict__ aux, int64_t ldaux, int epi, int M, int N, int K,
               int kb_per_split, float* __restrict__ partial, int vec_ok) {
  using S = TcSmem<BN, STAGES>;
  constexpr int TC_STAGES = STAGES;
  extern __shared__ uint8_t tc_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + S::MAIN_BYTES);
  uint64_t* empty_bar = full_bar + TC_STAGES;
  uint64_t* acc_bar = empty_bar + TC_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) { GPROF(0) }
  const int m0 = blockIdx.y * TC_BM, n0 = blockIdx.x * BN;
  const int kb_total = (K + TC_BK - 1) / TC_BK;
  const int kb0 = blockIdx.z * kb_per_split;
  const int kb1 = min(kb_total, kb0 + kb_per_split);
  const int nkb = kb1 - kb0;       // >= 1 by construction of the grid

  if (threadIdx.x == 0) {
    for (int s = 0; s < TC_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(acc_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  auto issue_load = [&](int i) {
    const int s = i % TC_STAGES;
    mbar_expect_tx(&full_bar[s], S::STAGE_BYTES);
    uint8_t* a_dst = smem + s * S::STAGE_BYTES;
    if constexpr (!MN) {
      tma_load_2d(a_dst, &tmA, &full_bar[s], (kb0 + i) * TC_BK, m0);
      tma_load_2d(a_dst + S::A_BYTES, &tmB, &full_bar[s], (kb0 + i) * TC_BK, n0);
    } else {
      // MN-major operands (A stored [K, M], B stored [K, N]: weight gradients x^T dy with no
      // transposed copies): one box = 64 K rows x 64 M|N elements (128 B, SWIZZLE_128B) = one
      // canonical MN-major swizzle atom column of 8 KB
#pragma unroll
      for (int at = 0; at < TC_BM / 64; ++at)
        tma_load_2d(a_dst + at * 8192, &tmA, &full_bar[s], m0 + at * 64, (kb0 + i) * TC_BK);
#pragma unroll
      for (int at = 0; at < BN / 64; ++at)
        tma_load_2d(a_dst + S::A_BYTES + at * 8192, &tmB, &full_bar[s], n0 + at * 64, (kb0 + i) * TC_BK);
    }
  };
  // the first pass through the ring needs the barriers only: those loads are in flight while warp 1 allocates TMEM
  const int nfirst = nkb < TC_STAGES ? nkb : TC_STAGES;
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    for (int i = 0; i < nfirst; ++i) issue_load(i);
  }
  if (warp == 1) {   // TMEM: BN fp32 accumulator columns (power of two >= 32)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(BN));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) { GPROF(1) }

  if (warp == 0) {
    if (lane == 0) {
      for (int i = nfirst; i < nkb; ++i) {
        const int s = i % TC_STAGES;
        const uint32_t ph = (uint32_t)(i / TC_STAGES) & 1u;
        mbar_wait(&empty_bar[s], ph ^ 1u);
        issue_load(i);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = MN ? make_idesc(1, TC_BM, BN, 1, 1) : make_idesc_bf16(TC_BM, BN);
      for (int i = 0; i < nkb; ++i) {
        const int s = i % TC_STAGES;
        const uint32_t ph = (uint32_t)(i / TC_STAGES) & 1u;
        mbar_wait(&full_bar[s], ph);
        if (i == 0) { GPROF(2) }
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + s * S::STAGE_BYTES);
        if constexpr (!MN) {
          const uint64_t adesc = make_sw128_kmajor_desc(a_addr);
          const uint64_t bdesc = make_sw128_kmajor_desc(a_addr + S::A_BYTES);
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k)      // +32 B (>>4 = 2) per K=16 step inside the swizzle row
            tc_mma_bf16(tmem_base, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (i | k) ? 1u : 0u);
        } else {
          // MN-major SWIZZLE_128B: LBO = 8192 B between 64-element M|N atoms, SBO = 1024 B between
          // 8-row K groups; a K = 16 step is two K groups = +2048 B (>>4 = 128)
          const uint64_t adesc = make_sw128_desc(a_addr, 8192, 1024);
          const uint64_t bdesc = make_sw128_desc(a_addr + S::A_BYTES, 8192, 1024);
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k)
            tc_mma_bf16(tmem_base, adesc + (uint64_t)(128 * k), bdesc + (uint64_t)(128 * k), idesc, (i | k) ? 1u : 0u);
        }
        tc_commit(&empty_bar[s]);                  // stage free once these MMAs have read it
      }
      tc_commit(acc_bar);                          // accumulator complete
      GPROF(3)
    }
  } else {
    // ---- epilogue warps 2..5 (TMEM lane group = warp % 4).  A thread owns an accumulator ROW, but a
    // row-per-thread global access pattern costs one memory transaction per lane (measured: 22 k of the
    // tile's 28 k cycles).  So: accumulators -> shared memory (the pipeline stages are idle now; each warp
    // touches only its own 32 rows, __syncwarp suffices) -> lane = column group, and every warp
    // instruction reads aux / writes C as ONE contiguous row segment.
    const int lg = warp & 3;
    // relu-mask epilogue on a full bf16 block of a one-CTA-per-SM launch: fetch the mask while the MMAs run
    constexpr bool PRE_OK = STAGES > 2 && BN == 128 && sizeof(CT) == 2;
    uint32_t pre[PRE_OK ? 64 : 1];
    bool use_pre = false;
    if constexpr (PRE_OK) {
      use_pre = epi == RS_EPI_MUL_RELU_MASK && aux != nullptr && partial == nullptr && vec_ok &&
                m0 + lg * 32 + 32 <= M && n0 + BN <= N;
      if (use_pre) {
        const CT* src = aux + (int64_t)(m0 + lg * 32) * ldaux + n0 + lane * 4;
#pragma unroll
        for (int rr = 0; rr < 32; ++rr) {
          const uint2 v = __ldg(reinterpret_cast<const uint2*>(src + (int64_t)rr * ldaux));
          pre[2 * rr] = v.x; pre[2 * rr + 1] = v.y;
        }
      }
    }
    mbar_wait(acc_bar, 0);
    if (threadIdx.x == 64) { GPROF(4) }
    tc_fence_after();
    constexpr int PITCH = S::STG_PITCH;            // floats; (BN + 4) mod 32 = 4: conflict-free 16-byte row writes
    float* stg = reinterpret_cast<float*>(smem) + (size_t)lg * 32 * PITCH;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      if (n0 + c0 >= N) break;                     // warp-uniform
      uint32_t r[32];
      tc_ld_32x32(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)c0, r);
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<float4*>(stg + lane * PITCH + c0 + j) =
            make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
    }
    __syncwarp();
    const int rows_here = min(32, M - (m0 + lg * 32));      // warp-uniform
    if (rows_here > 0) {
      float* part_rows = partial ? partial + ((int64_t)blockIdx.z * M + m0 + lg * 32) * N + n0 : nullptr;
      CT* c_rows = C + (int64_t)(m0 + lg * 32) * ldc + n0;
      const CT* a_rows = aux ? aux + (int64_t)(m0 + lg * 32) * ldaux + n0 : nullptr;
      const int ncols = N - n0;
#define RS_EPI_GO(E) epilogue_rows<BN, E, CT>(stg, rows_here, lane, ncols, N, c_rows, ldc, a_rows, ldaux, bias ? bias + n0 : nullptr, vec_ok)
      if (part_rows) epilogue_partial<BN>(stg, rows_here, lane, ncols, N, part_rows);
      else if (use_pre) {
        if constexpr (PRE_OK) epilogue_mask_pre<BN, CT>(stg, lane, c_rows, ldc, pre);
      }
      else switch (epi) {
        case RS_EPI_BIAS: RS_EPI_GO(RS_EPI_BIAS); break;
        case RS_EPI_BIAS_RELU: RS_EPI_GO(RS_EPI_BIAS_RELU); break;
        case RS_EPI_BIAS_SIGMOID: RS_EPI_GO(RS_EPI_BIAS_SIGMOID); break;
        case RS_EPI_MUL_RELU_MASK: RS_EPI_GO(RS_EPI_MUL_RELU_MASK); break;
        case RS_EPI_MUL_DSIGMOID: RS_EPI_GO(RS_EPI_MUL_DSIGMOID); break;
        case RS_EPI_ACCUM: RS_EPI_GO(RS_EPI_ACCUM); break;
        default: RS_EPI_GO(RS_EPI_NONE);
      }
#undef RS_EPI_GO
    }
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) { GPROF(5) }
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(BN));
  }
}

// C = [C +] sum_z partial[z]  (split order fixed => deterministic)
template <typename CT>
__global__ void splitk_reduce_kernel(const float* __restrict__ partial, int splits, CT* __restrict__ C,
                                     int64_t ldc, int M, int N, int accumulate) {
  const int64_t total = (int64_t)M * N;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = t / N;
    const int n = (int)(t % N);
    float s = accumulate ? to_f<CT>(C[m * ldc + n]) : 0.f;
    for (int z = 0; z < splits; ++z) s += partial[(int64_t)z * total + t];
    C[m * ldc + n] = from_f<CT>(s);
  }
}

// Same sums, same order, four adjacent outputs per thread and eight splits' loads in flight per step (N % 4 == 0 and
// 16-byte aligned rows): the scalar kernel above is one dependent 4-byte load per split.
template <typename CT>
__global__ void splitk_reduce_vec_kernel(const float* __restrict__ partial, int splits, CT* __restrict__ C,
                                         int64_t ldc, int M, int N, int accumulate) {
  const int64_t total = (int64_t)M * N;
  const int n4 = N >> 2;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < (int64_t)M * n4; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = q / n4;
    const int n = (int)(q % n4) * 4;
    const float* p = partial + m * N + n;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (accumulate) s = load4<CT>(C + m * ldc + n);
    int z = 0;
    for (; z + 8 <= splits; z += 8) {
      float4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = *reinterpret_cast<const float4*>(p + (int64_t)(z + u) * total);
#pragma unroll
      for (int u = 0; u < 8; ++u) { s.x += v[u].x; s.y += v[u].y; s.z += v[u].z; s.w += v[u].w; }
    }
    for (; z < splits; ++z) {
      const float4 v = *reinterpret_cast<const float4*>(p + (int64_t)z * total);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    store4<CT>(C + m * ldc + n, s);
  }
}

int splitk_reduce(const float* partial, int splits, void* C, int64_t ldc, int M, int N, int accumulate,
                  int dtype_c, cudaStream_t st) {
  const int64_t total = (int64_t)M * N;
  const int esz = dtype_c == RS_F32 ? 4 : 2;
  if (N % 4 == 0 && ((uintptr_t)C % (4 * esz)) == 0 && ((ldc * esz) % (4 * esz)) == 0 && ((uintptr_t)partial % 16) == 0) {
    int64_t blocks = cdiv(total / 4, 128);
    if (blocks > (int64_t)sm_count() * 16) blocks = (int64_t)sm_count() * 16;
    if (dtype_c == RS_F32)
      splitk_reduce_vec_kernel<float><<<(unsigned)blocks, 128, 0, st>>>(partial, splits, (float*)C, ldc, M, N, accumulate);
    else
      splitk_reduce_vec_kernel<__nv_bfloat16><<<(unsigned)blocks, 128, 0, st>>>(partial, splits, (__nv_bfloat16*)C, ldc,
                                                                               M, N, accumulate);
    return check_launch("splitk_reduce");
  }
  int64_t blocks = cdiv(total, 256);
  if (blocks > (int64_t)sm_count() * 8) blocks = (int64_t)sm_count() * 8;
  if (dtype_c == RS_F32)
    splitk_reduce_kernel<float><<<(unsigned)blocks, 256, 0, st>>>(partial, splits, (float*)C, ldc, M, N, accumulate);
  else
    splitk_reduce_kernel<__nv_bfloat16><<<(unsigned)blocks, 256, 0, st>>>(partial, splits, (__nv_bfloat16*)C, ldc, M,
                                                                          N, accumulate);
  return check_launch("splitk_reduce");
}

// ---- host side --------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// 2-D bf16 row-major [rows, cols] with leading dim ld (elements); box = 64 cols x box_rows rows, SWIZZLE_128B.
int make_map(CUtensorMap* map, const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) { set_error("gemm_tc: cuTensorMapEncodeTiled unavailable"); return RS_ERR_UNSUPPORTED; }
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("gemm_tc: cuTensorMapEncodeTiled failed (%d)", (int)r); return RS_ERR_INVALID; }
  return 0;
}

template <int BN, int STAGES, bool MN, typename CT>
static int launch_tc(const CUtensorMap& tmA, const CUtensorMap& tmB, void* C, int64_t ldc, const float* bias,
                     const void* aux, int64_t ldaux, int epi, int M, int N, int K, int splits, int kbps,
                     float* partial, int vec_ok, cudaStream_t st) {
  auto kern = gemm_tc_kernel<BN, STAGES, MN, CT>;
  const int smem = TcSmem<BN, STAGES>::TOTAL;
  RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  dim3 grid((unsigned)cdiv(N, BN), (unsigned)cdiv(M, TC_BM), (unsigned)splits);
  kern<<<grid, TC_THREADS, smem, st>>>(tmA, tmB, (CT*)C, ldc, bias, (const CT*)aux, ldaux, epi, M, N, K, kbps,
                                       partial, vec_ok);
  return check_launch("gemm_tc");
}

// splits * M * N <= (sms / tiles) * tiles * 128 * 128 floats
// split-K partials: one 128 x 128 fp32 tile per SM for the bf16 kernel; the fp32 3xTF32 kernel caps an accumulation
// chain at K = 4096 and needs room for ceil(K / 4096) full [M, N] partials — 64 MiB covers the widest weight gradient
// of the composed models (staytime_output 1840 x 401 over a batch of 16 384 fell to the FFMA kernel for 1.8 ms without it)
size_t gemm_tc_workspace_bytes() {
  const size_t a = (size_t)sm_count() * TC_BM * 128 * sizeof(float), b = (size_t)64 << 20;
  return a > b ? a : b;
}

int gemm_bf16_tc(const void* A, int64_t lda, int transA, const void* B, int64_t ldb, int transB, void* C,
                 int64_t ldc, const float* bias, const void* aux, int64_t ldaux, int epilogue, int M, int N,
                 int K, int dtype_c, void* ws, size_t ws_bytes, cudaStream_t st) {
  RS_REQUIRE((!transA && transB) || (transA && !transB),
             "gemm(bf16): tensor-core path takes both operands K-major (A stored [M,K], transA=0; B stored [N,K], "
             "transB=1) or both MN-major (A stored [K,M], transA=1; B stored [K,N], transB=0)");
  const bool mn = transA != 0;
  RS_REQUIRE(lda % 8 == 0 && ldb % 8 == 0, "gemm(bf16): lda/ldb must be multiples of 8 elements (16-byte TMA strides)");
  RS_REQUIRE(((uintptr_t)A % 16 == 0) && ((uintptr_t)B % 16 == 0), "gemm(bf16): A/B must be 16-byte aligned");
  RS_REQUIRE(dtype_c == RS_F32 || dtype_c == RS_BF16, "gemm(bf16): bad C dtype");
  // tile width: the widest BN that still gives >= ~1 wave of CTAs
  const int sms = sm_count();
  int BN = 128;
  if (N <= 32) BN = 32;
  else if (N <= 64) BN = 64;
  else if (mn && N % 128 != 0 && N % 128 <= 64) BN = 64;   // MN-major boxes are 64 wide: no half-empty 128 tile
  else if ((int64_t)cdiv(M, TC_BM) * cdiv(N, 128) < sms && N % 128 != 0) BN = 64;
  else if ((int64_t)cdiv(M, TC_BM) * cdiv(N, 128) * 2 <= sms) BN = 64;
  const int tiles = (int)(cdiv(M, TC_BM) * cdiv(N, BN));
  const int kb_total = (int)cdiv(K, TC_BK);
  // split-K when the tile grid cannot fill the machine and K is deep (weight gradients)
  int splits = 1;
  if ((epilogue == RS_EPI_NONE || epilogue == RS_EPI_ACCUM) && tiles * 2 <= sms && kb_total >= 8) {
    splits = sms / tiles;
    if (splits > kb_total / 2) splits = kb_total / 2;
    if (splits < 1) splits = 1;
  }
  int kbps = (int)cdiv(kb_total, splits);
  splits = (int)cdiv(kb_total, kbps);
  float* partial = nullptr;
  if (splits > 1) {
    const size_t need = (size_t)splits * M * N * sizeof(float);
    if (ws == nullptr || ws_bytes < need) {
      set_error("gemm(bf16): split-K workspace %zu < %zu", ws_bytes, need);
      return RS_ERR_WORKSPACE;
    }
    partial = (float*)ws;
  }
  CUtensorMap tmA, tmB;
  if (!mn) {
    if (int e = make_map(&tmA, A, M, K, lda, TC_BM)) return e;
    if (int e = make_map(&tmB, B, N, K, ldb, BN)) return e;
  } else {
    RS_REQUIRE(BN >= 64, "gemm(bf16): MN-major operands need N > 32");
    if (int e = make_map(&tmA, A, K, M, lda, TC_BK)) return e;     // [K rows, M cols], box 64 x 64
    if (int e = make_map(&tmB, B, K, N, ldb, TC_BK)) return e;
  }
  const int esz = dtype_c == RS_F32 ? 4 : 2;
  int vec_ok = ((uintptr_t)C % 16 == 0) && ((ldc * esz) % 16 == 0);
  if (aux) vec_ok = vec_ok && ((uintptr_t)aux % 16 == 0) && ((ldaux * esz) % 16 == 0);
  int rc;
  const bool deep = (int64_t)tiles * splits <= sms;
#define RS_TC_GO3(BNV, ST, MNV)                                                                                  \
  rc = dtype_c == RS_F32                                                                                         \
           ? launch_tc<BNV, ST, MNV, float>(tmA, tmB, C, ldc, bias, aux, ldaux, epilogue, M, N, K, splits, kbps, \
                                            partial, vec_ok, st)                                                 \
           : launch_tc<BNV, ST, MNV, __nv_bfloat16>(tmA, tmB, C, ldc, bias, aux, ldaux, epilogue, M, N, K,      \
                                                    splits, kbps, partial, vec_ok, st)
#define RS_TC_GO2(BNV, ST) \
  if (mn) { RS_TC_GO3(BNV, ST, true); } else { RS_TC_GO3(BNV, ST, false); }
#define RS_TC_GO(BNV) \
  if (deep) { RS_TC_GO2(BNV, 6) } else { RS_TC_GO2(BNV, 2) }
  if (BN == 32) { RS_TC_GO3(32, 2, false); }
  else if (BN == 64) { RS_TC_GO(64) }
  else { RS_TC_GO(128) }
#undef RS_TC_GO3
#undef RS_TC_GO2
#undef RS_TC_GO
  if (rc) return rc;
  if (splits > 1)
    return splitk_reduce(partial, splits, C, ldc, M, N, epilogue == RS_EPI_ACCUM, dtype_c, st);
  return 0;
}

// =================================================================================================
// fp32 operands on the tensor cores: 3xTF32.  x = hi + lo with hi = x with the low 13 mantissa bits
// cleared (exactly a tf32 number) and lo = x - hi (exact in fp32, 13 significant bits of which the tensor
// core keeps 11): a.b ~= hi.hi + hi.lo + lo.hi, relative error ~2^-20 per product, i.e. fp32-grade
// results (the 1e-5 parity bar) at tensor-core rate instead of the FFMA kernel.
//
//   warp 0      TMA producer: raw fp32 tiles (32 floats = one 128-byte SWIZZLE_128B row per K slab)
//   warps 2..5  splitters: hi overwrites the raw tile in place, lo goes to a twin tile at the same
//               offsets (an elementwise pass is layout-agnostic, so the swizzle is untouched);
//               fence.proxy.async, then arrive on the stage's `split` barrier.  Afterwards: epilogue.
//   warp 1      MMA issuer: waits for `split`, issues 3 x 4 tcgen05.mma.kind::tf32 (K = 8) per stage.
// Operands may each be K-major (stored [rows, K]) or MN-major (stored [K, rows]): Dense forward
// x[M,K] . W[K,N] (Keras [in,out] weights as they lie), dgrad dy . W^T, wgrad x^T . dy - no transposes.
constexpr int T3_BK = 32;          // fp32 elements per stage along K

// MN-major tf32 operands exist in one shared-memory layout only: SWIZZLE_128B_BASE32B (descriptor layout
// type 1; TMA CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B): 32-byte chunks of a 128-byte row (32 floats along M|N)
// XOR-ed with the K row index mod 4; atom = 4 K rows x 128 B.  LBO = bytes between 32-float atoms along
// M|N, SBO = bytes between 4-row K groups.
__device__ __forceinline__ uint64_t make_sw128b32_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46) | ((uint64_t)1 << 61);
}

template <int BN, int STAGES>
struct T3Smem {
  static constexpr int A_BYTES = TC_BM * T3_BK * 4;            // 16 KB
  static constexpr int B_BYTES = BN * T3_BK * 4;
  static constexpr int RAW_BYTES = A_BYTES + B_BYTES;          // [A raw->hi | B raw->hi]
  static constexpr int STAGE_BYTES = 2 * RAW_BYTES;            // ... [A lo | B lo]
  static constexpr int STG_PITCH = BN + 4;
  static constexpr int STG_BYTES = TC_BM * STG_PITCH * 4;
  static constexpr int MAIN_BYTES = STAGES * STAGE_BYTES > STG_BYTES ? STAGES * STAGE_BYTES : STG_BYTES;
  static constexpr int TOTAL = MAIN_BYTES + 1024 + 256;
};

template <int BN, int STAGES, bool AMN, bool BMN, typename CT>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tf32x3_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   CT* __restrict__ C, int64_t ldc, const float* __restrict__ bias,
                   const CT* __restrict__ aux, int64_t ldaux, int epi, int M, int N, int K,
                   int kb_per_split, float* __restrict__ partial, int vec_ok) {
  using S = T3Smem<BN, STAGES>;
  extern __shared__ uint8_t tc_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + S::MAIN_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* split_bar = empty_bar + STAGES;
  uint64_t* acc_bar = split_bar + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * TC_BM, n0 = blockIdx.x * BN;
  const int kb_total = (K + T3_BK - 1) / T3_BK;
  const int kb0 = blockIdx.z * kb_per_split;
  const int kb1 = min(kb_total, kb0 + kb_per_split);
  const int nkb = kb1 - kb0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
      mbar_init(&split_bar[s], 128);
    }
    mbar_init(acc_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(2 * BN));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
      for (int i = 0; i < nkb; ++i) {
        const int s = i % STAGES;
        const uint32_t ph = (uint32_t)(i / STAGES) & 1u;
        mbar_wait(&empty_bar[s], ph ^ 1u);
        mbar_expect_tx(&full_bar[s], S::RAW_BYTES);
        uint8_t* a_dst = smem + s * S::STAGE_BYTES;
        const int k0 = (kb0 + i) * T3_BK;
        if constexpr (!AMN) {
          tma_load_2d(a_dst, &tmA, &full_bar[s], k0, m0);                 // box 32 K x 128 rows
        } else {
#pragma unroll
          for (int at = 0; at < TC_BM / 32; ++at)                          // box 32 M x 32 K rows = 4 KB atom column
            tma_load_2d(a_dst + at * 4096, &tmA, &full_bar[s], m0 + at * 32, k0);
        }
        if constexpr (!BMN) {
          tma_load_2d(a_dst + S::A_BYTES, &tmB, &full_bar[s], k0, n0);
        } else {
#pragma unroll
          for (int at = 0; at < BN / 32; ++at)
            tma_load_2d(a_dst + S::A_BYTES + at * 4096, &tmB, &full_bar[s], n0 + at * 32, k0);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(2, TC_BM, BN, AMN ? 1 : 0, BMN ? 1 : 0);
      for (int i = 0; i < nkb; ++i) {
        const int s = i % STAGES;
        const uint32_t ph = (uint32_t)(i / STAGES) & 1u;
        mbar_wait(&split_bar[s], ph);
        tc_fence_after();
        const uint32_t base = smem_u32(smem + s * S::STAGE_BYTES);
        // K-major: +32 B per K = 8 step inside the swizzle row; MN-major: LBO 4096 between 32-float
        // atoms (one TMA box each), SBO 512 between 4-row K groups, a K = 8 step is two groups = +1024 B
        const uint64_t a_hi = AMN ? make_sw128b32_desc(base, 4096, 512) : make_sw128_kmajor_desc(base);
        const uint64_t b_hi = BMN ? make_sw128b32_desc(base + S::A_BYTES, 4096, 512) : make_sw128_kmajor_desc(base + S::A_BYTES);
        const uint64_t a_lo = AMN ? make_sw128b32_desc(base + S::RAW_BYTES, 4096, 512) : make_sw128_kmajor_desc(base + S::RAW_BYTES);
        const uint64_t b_lo = BMN ? make_sw128b32_desc(base + S::RAW_BYTES + S::A_BYTES, 4096, 512)
                                  : make_sw128_kmajor_desc(base + S::RAW_BYTES + S::A_BYTES);
        constexpr uint64_t ka = AMN ? 64 : 2, kb = BMN ? 64 : 2;
        // The tensor core truncates when it adds a product into the fp32 accumulator: the error grows with
        // the number of accumulation steps times the accumulator's ulp.  The two correction products are
        // 2^-11 smaller, so they get their own accumulator (columns [BN, 2BN)): the main one then sees K/8
        // steps instead of 3K/8 (measured at K = 4096: 1.9e-5 -> 6e-6 of max|C|); the epilogue adds the two.
#pragma unroll
        for (int k = 0; k < T3_BK / 8; ++k)
          tc_mma_tf32(tmem_base + BN, a_lo + ka * k, b_hi + kb * k, idesc, (i | k) ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < T3_BK / 8; ++k) tc_mma_tf32(tmem_base + BN, a_hi + ka * k, b_lo + kb * k, idesc, 1u);
#pragma unroll
        for (int k = 0; k < T3_BK / 8; ++k)
          tc_mma_tf32(tmem_base, a_hi + ka * k, b_hi + kb * k, idesc, (i | k) ? 1u : 0u);
        tc_commit(&empty_bar[s]);
      }
      tc_commit(acc_bar);
    }
  } else {
    // ---- splitters, then epilogue (warps 2..5)
    const int t = threadIdx.x - 64;
    for (int i = 0; i < nkb; ++i) {
      const int s = i % STAGES;
      const uint32_t ph = (uint32_t)(i / STAGES) & 1u;
      mbar_wait(&full_bar[s], ph);
      uint8_t* raw = smem + s * S::STAGE_BYTES;
#pragma unroll 4
      for (int o = t * 16; o < S::RAW_BYTES; o += 128 * 16) {
        const uint4 x = *reinterpret_cast<const uint4*>(raw + o);
        uint4 h, l;
        h.x = x.x & 0xFFFFE000u; h.y = x.y & 0xFFFFE000u; h.z = x.z & 0xFFFFE000u; h.w = x.w & 0xFFFFE000u;
        l.x = __float_as_uint(__uint_as_float(x.x) - __uint_as_float(h.x));
        l.y = __float_as_uint(__uint_as_float(x.y) - __uint_as_float(h.y));
        l.z = __float_as_uint(__uint_as_float(x.z) - __uint_as_float(h.z));
        l.w = __float_as_uint(__uint_as_float(x.w) - __uint_as_float(h.w));
        *reinterpret_cast<uint4*>(raw + o) = h;
        *reinterpret_cast<uint4*>(raw + S::RAW_BYTES + o) = l;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&split_bar[s])) : "memory");
    }
    const int lg = warp & 3;
    mbar_wait(acc_bar, 0);
    tc_fence_after();
    constexpr int PITCH = S::STG_PITCH;
    float* stg = reinterpret_cast<float*>(smem) + (size_t)lg * 32 * PITCH;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      if (n0 + c0 >= N) break;
      uint32_t r[32], q[32];
      tc_ld_32x32(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)c0, r);
      tc_ld_32x32(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(BN + c0), q);
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<float4*>(stg + lane * PITCH + c0 + j) =
            make_float4(__uint_as_float(r[j]) + __uint_as_float(q[j]), __uint_as_float(r[j + 1]) + __uint_as_float(q[j + 1]),
                        __uint_as_float(r[j + 2]) + __uint_as_float(q[j + 2]), __uint_as_float(r[j + 3]) + __uint_as_float(q[j + 3]));
    }
    __syncwarp();
    const int rows_here = min(32, M - (m0 + lg * 32));
    if (rows_here > 0) {
      float* part_rows = partial ? partial + ((int64_t)blockIdx.z * M + m0 + lg * 32) * N + n0 : nullptr;
      CT* c_rows = C + (int64_t)(m0 + lg * 32) * ldc + n0;
      const CT* a_rows = aux ? aux + (int64_t)(m0 + lg * 32) * ldaux + n0 : nullptr;
      const int ncols = N - n0;
#define RS_EPI_GO(E) epilogue_rows<BN, E, CT>(stg, rows_here, lane, ncols, N, c_rows, ldc, a_rows, ldaux, bias ? bias + n0 : nullptr, vec_ok)
      if (part_rows) epilogue_partial<BN>(stg, rows_here, lane, ncols, N, part_rows);
      else switch (epi) {
        case RS_EPI_BIAS: RS_EPI_GO(RS_EPI_BIAS); break;
        case RS_EPI_BIAS_RELU: RS_EPI_GO(RS_EPI_BIAS_RELU); break;
        case RS_EPI_BIAS_SIGMOID: RS_EPI_GO(RS_EPI_BIAS_SIGMOID); break;
        case RS_EPI_MUL_RELU_MASK: RS_EPI_GO(RS_EPI_MUL_RELU_MASK); break;
        case RS_EPI_MUL_DSIGMOID: RS_EPI_GO(RS_EPI_MUL_DSIGMOID); break;
        case RS_EPI_ACCUM: RS_EPI_GO(RS_EPI_ACCUM); break;
        default: RS_EPI_GO(RS_EPI_NONE);
      }
#undef RS_EPI_GO
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(2 * BN));
  }
}

// 2-D fp32 row-major [rows, cols] with leading dim ld (elements); box = box_cols x box_rows.
static int make_map_f32(CUtensorMap* map, const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_cols,
                        int box_rows, bool mn_major) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) { set_error("gemm_tf32x3: cuTensorMapEncodeTiled unavailable"); return RS_ERR_UNSUPPORTED; }
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE,
                  mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("gemm_tf32x3: cuTensorMapEncodeTiled failed (%d)", (int)r); return RS_ERR_INVALID; }
  return 0;
}

template <int BN, int STAGES, bool AMN, bool BMN, typename CT>
static int launch_t3(const CUtensorMap& tmA, const CUtensorMap& tmB, void* C, int64_t ldc, const float* bias,
                     const void* aux, int64_t ldaux, int epi, int M, int N, int K, int splits, int kbps,
                     float* partial, int vec_ok, cudaStream_t st) {
  auto kern = gemm_tf32x3_kernel<BN, STAGES, AMN, BMN, CT>;
  const int smem = T3Smem<BN, STAGES>::TOTAL;
  RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  dim3 grid((unsigned)cdiv(N, BN), (unsigned)cdiv(M, TC_BM), (unsigned)splits);
  kern<<<grid, TC_THREADS, smem, st>>>(tmA, tmB, (CT*)C, ldc, bias, (const CT*)aux, ldaux, epi, M, N, K, kbps,
                                       partial, vec_ok);
  return check_launch("gemm_tf32x3");
}

// Can this fp32 problem run on the tensor cores?  (16-byte TMA strides and bases; big enough to matter.)
bool gemm_tf32x3_usable(const void* A, int64_t lda, const void* B, int64_t ldb, int M, int N, int K, int dtype_c,
                        int epilogue, size_t ws_bytes) {
  if (dtype_c != RS_F32) return false;
  // one accumulation chain stays <= 4096 deep (truncating accumulator, see the kernel): longer K needs
  // split-K, i.e. a plain / accumulate epilogue and room for the partial tiles
  if (K > 4096) {
    if (!(epilogue == RS_EPI_NONE || epilogue == RS_EPI_ACCUM)) return false;
    const size_t max_splits = ws_bytes / ((size_t)M * N * sizeof(float));
    if (max_splits < 1 || cdiv(K, (int64_t)max_splits) > 4096) return false;
  }
  if (lda % 4 || ldb % 4 || ((uintptr_t)A & 15) || ((uintptr_t)B & 15)) return false;
  if (N < 8 || K < 8 || M < 8) return false;
  return (int64_t)M * N * K >= ((int64_t)1 << 20);
}

int gemm_tf32x3(const void* A, int64_t lda, int transA, const void* B, int64_t ldb, int transB, void* C,
                int64_t ldc, const float* bias, const void* aux, int64_t ldaux, int epilogue, int M, int N,
                int K, void* ws, size_t ws_bytes, cudaStream_t st) {
  const bool amn = transA != 0;          // A stored [K, M]
  const bool bmn = transB == 0;          // B stored [K, N]
  const int sms = sm_count();
  int BN = 128;
  if (N <= 32) BN = 32;
  else if (N <= 64) BN = 64;
  else if ((int64_t)cdiv(M, TC_BM) * cdiv(N, 128) < sms && N % 128 != 0 && N % 128 <= 64) BN = 64;
  else if ((int64_t)cdiv(M, TC_BM) * cdiv(N, 128) * 2 <= sms) BN = 64;
  // wide tiles when 128-wide ones would need more than one round of CTAs: the A tile is split (and
  // streamed by the MMAs) once per 256 output columns instead of once per 128
  else if (N % 256 == 0 && (int64_t)cdiv(M, TC_BM) * (N / 128) > sms) BN = 256;
  const int tiles = (int)(cdiv(M, TC_BM) * cdiv(N, BN));
  const int kb_total = (int)cdiv(K, T3_BK);
  int splits = 1;
  const bool can_split = (epilogue == RS_EPI_NONE || epilogue == RS_EPI_ACCUM) && ws != nullptr;
  if (can_split && tiles * 2 <= sms && kb_total >= 16) {
    splits = sms / tiles;
    if (splits > kb_total / 4) splits = kb_total / 4;
  }
  if (can_split && cdiv(kb_total, splits) > 2048 / T3_BK) splits = (int)cdiv(kb_total, 2048 / T3_BK);   // chain <= 2048
  if (can_split && (size_t)splits * M * N * sizeof(float) > ws_bytes)
    splits = (int)(ws_bytes / ((size_t)M * N * sizeof(float)));
  if (splits < 1) splits = 1;
  if (cdiv(kb_total, splits) > 4096 / T3_BK) {
    set_error("gemm(fp32, 3xTF32): K=%d needs split-K workspace (%zu bytes given)", K, ws_bytes);
    return RS_ERR_WORKSPACE;
  }
  int kbps = (int)cdiv(kb_total, splits);
  splits = (int)cdiv(kb_total, kbps);
  float* partial = splits > 1 ? (float*)ws : nullptr;
  CUtensorMap tmA, tmB;
  if (!amn) { if (int e = make_map_f32(&tmA, A, M, K, lda, T3_BK, TC_BM, false)) return e; }
  else      { if (int e = make_map_f32(&tmA, A, K, M, lda, 32, T3_BK, true)) return e; }
  if (!bmn) { if (int e = make_map_f32(&tmB, B, N, K, ldb, T3_BK, BN, false)) return e; }
  else      { if (int e = make_map_f32(&tmB, B, K, N, ldb, 32, T3_BK, true)) return e; }
  int vec_ok = ((uintptr_t)C % 16 == 0) && ((ldc * 4) % 16 == 0);
  if (aux) vec_ok = vec_ok && ((uintptr_t)aux % 16 == 0) && ((ldaux * 4) % 16 == 0);
  int rc;
#define RS_T3_GO2(BNV, ST, AM, BM) \
  rc = launch_t3<BNV, ST, AM, BM, float>(tmA, tmB, C, ldc, bias, aux, ldaux, epilogue, M, N, K, splits, kbps, partial, vec_ok, st)
#define RS_T3_GO(BNV, ST)                                   \
  if (amn && bmn) { RS_T3_GO2(BNV, ST, true, true); }       \
  else if (amn) { RS_T3_GO2(BNV, ST, true, false); }        \
  else if (bmn) { RS_T3_GO2(BNV, ST, false, true); }        \
  else { RS_T3_GO2(BNV, ST, false, false); }
  if (BN == 32) { RS_T3_GO(32, 4) }
  else if (BN == 64) { RS_T3_GO(64, 4) }
  else if (BN == 256) { RS_T3_GO(256, 2) }
  else { RS_T3_GO(128, 3) }
#undef RS_T3_GO
#undef RS_T3_GO2
  if (rc) return rc;
  if (splits > 1) return splitk_reduce(partial, splits, C, ldc, M, N, epilogue == RS_EPI_ACCUM, RS_F32, st);
  return 0;
}

#ifdef RS_GEMM_PROFILE
extern "C" int rs_debug_gemm_profile(long long* out16) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out16, gemm_prof, sizeof(long long) * 16);
  return 0;
}
#endif

}  // namespace rs
