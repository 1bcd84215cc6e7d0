// interacting_tc.cu — K4 on the 5th-gen tensor cores (bf16 mode): fused InteractingLayer
// forward (InteractingLayer.py:37-61) with every contraction issued as tcgen05.mma and every A operand
// resident in TMEM.
//
// A CTA of 384 threads keeps THREE 128-row tiles in flight, one per warpgroup (own TMEM columns, own mbarrier,
// own named barrier); a tile holds SPT whole samples, sample s in tile rows [s*FP, s*FP + F) with FP = F rounded up
// to 8 (F = 39 -> 3 samples at rows 0 / 40 / 80).  Thread t of a warpgroup IS tile row t and TMEM lane t, so every
// accumulator row comes back to the thread that owns the (sample, field) row and the row-wise softmax / residual /
// ReLU / LayerNorm need no cross-thread traffic.  Per iteration of the layer_num loop (weights shared):
//
//   1. Z[128,4U]  = [X | 1] [Wqkvr ; b]         kind::tf32, 3xTF32 split (fp32-grade), A = [x_hi | x_lo | 1 1 0..]
//      written to TMEM by the row's thread (tcgen05.st); bias rides in the MMA
//   2. S_h[128,FP] = Qx_h Kx_h^T  per head      kind::tf32, A = the row's q placed in the K slot of its own sample
//      (zeros elsewhere), B row j = [k_(0,j) | k_(1,j) | ..]: every row finds ITS sample's FP keys in the same FP
//      accumulator columns — no 128-wide block-diagonal product, no per-lane window select
//      thread: softmax over its F keys (exp2, FFMA2 / FADD2 packed math), unnormalised bf16 P -> TMEM
//   3. O_h[128,32] = P_h V_h                    kind::f16, A = P from TMEM, B = [key][(sample, e)]: a row keeps the 8
//      columns of its own sample;  thread: O/l + r -> ReLU -> LayerNorm -> y (next iteration's X)
//
// Saved for the backward: the pre-LayerNorm activations of every iteration and the per-head softmax statistics
// lse = max + log2(sum) (so the backward recomputes P already normalised).  Optional fused lookup (K1 inside K4):
// the tile loader reads the embedding rows itself — from this GPU's table or, row-sharded, straight from the owners'
// HBM over NVLink — two tiles ahead for the ids and one for the rows, writes X (bf16, for the MLP tower and the
// backward) and the sort keys as by-products: the gather kernel disappears from the step.
#include "tc_common.cuh"
#include "interacting_args.cuh"
#include <type_traits>

namespace rs {


// tile-private TMEM columns (per warpgroup): Z [0,64) -> expanded Q_h over [0,32), [32,64) once the thread has its
// Z row in registers (a lane's columns are private to its thread) -> O_h at h*32 ; S_h at 64 + h*FP with P_h
// (packed bf16) over its first KP/2 columns and [x_hi | x_lo] over [64,96) before S is issued ; [1 1 0..] at 160
constexpr uint32_t ITC_TILE_COLS = 168;

// fused embedding lookup (K1 inside K4): ids [B, F] -> rows of the (row-sharded) tables.  tab[r] = rank r's shard
// (CUDA-IPC mapping; tab[0] = the local table when world == 1), row stride tld floats, owner = row mod world.
struct ItcGather {
  const float* tab[RS_MAX_PEERS];
  int64_t tld;
  int world;
  const int64_t* ids;
  const int64_t* lbase;      // [F] first local row of field f on every rank
  const int64_t* rows;       // [F] rows of field f (ids are taken mod rows)
  uint64_t* keys;            // [B*F] (local arena row << 32 | position) for the sorted-segment update, or NULL
};

// fused bag mean (rs_interacting_fwd_gather_bag, one GPU): ids [B, S], field f owns the slots [off[f], off[f+1]) of a
// sample; keys [B*S] per slot (all-ones for padding) and inv_cnt [B*F]
struct ItcBagGather : ItcGather {
  const int64_t* off;        // [F+1] exclusive cumsum of the per-field bag sizes, off[F] = S
  float* inv_cnt;            // [B*F] 1 / (valid ids of the bag), 0 for an empty bag
  int S;
};
// rows of one bag requested together (independent loads in flight per thread; the register budget of the 384-thread
// CTA bounds it: the chunk's rows live in registers until they are summed)
constexpr int ITC_BAG_CHUNK = 4;

__device__ __forceinline__ void ld_row64(const float* p, uint32_t (&v)[16]) {
  // one 64-byte embedding row as two 32-byte requests (LDG.256): a row-per-thread loader must not split a row into
  // four 16-byte requests (the NVLink path is request-rate bound); L2::64B: a miss fetches the 64-byte row, not 128 B
  asm volatile("ld.global.L1::no_allocate.L2::64B.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "l"(p) : "memory");
  asm volatile("ld.global.L1::no_allocate.L2::64B.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
               : "l"(p + 8) : "memory");
}

template <int NCHF, typename T, bool GATHER, typename GA = ItcGather>
__global__ void __launch_bounds__(384, 1)
interacting_tc_fwd_kernel(const GA ga, T* __restrict__ x, int64_t x_ld, int64_t x_bs, const float* __restrict__ W,
                          const float* __restrict__ bias, const float* __restrict__ gamma,
                          const float* __restrict__ beta, float eps, T* __restrict__ y, int64_t y_ld,
                          int64_t y_bs, float* __restrict__ saved, int B, int F, int L, int use_res) {
  constexpr int D = 16, U = 16, H = 2, DH = 8, N4 = 64;
  using G = ItcGeom<NCHF>;
  constexpr int FP = G::FP, SPT = G::SPT, NCHK = G::NCHK, KP = G::KP;
  constexpr int FMIN = NCHF == 2 ? 0 : FP - 8;           // F > FMIN is guaranteed (NCHF = 2 also serves F <= 8)
  constexpr bool BAG = !std::is_same<GA, ItcGather>::value;   // GATHER with a bag of slots per (sample, field)
  // ---- shared memory: only B operands live here (every A operand is TMEM-resident)
  constexpr int WG_BYTES = H * G::KX_BYTES + H * G::VX_BYTES;
  constexpr int OFF_KX = 0;                              // H x [FP keys][8 SPT] tf32, K-major: row j = [k_0j | k_1j | ..]
  constexpr int OFF_VX = H * G::KX_BYTES;                // H x [KP keys][32] bf16, MN-major: chunk s of row j = v_sj
  constexpr int OFF_W = 3 * WG_BYTES;                    // W_hi | W_lo, each [64 n][16 k] tf32
  constexpr int OFF_BT = OFF_W + 8192;                   // [64 n][8 k] tf32: k = 0 b_hi, k = 1 b_lo (bias through the MMA)
  constexpr int OFF_F = OFF_BT + 2048;                   // gamma[16] beta[16] fp32
  constexpr int OFF_BAR = OFF_F + 2 * U * 4;
  extern __shared__ __align__(128) uint8_t itc_smem[];
  uint8_t* smem = itc_smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);

  const uint32_t warp = uniform_u32(threadIdx.x >> 5);   // uniform register
  const uint32_t wg = warp >> 2, wq = warp & 3;          // warpgroup = tile slot, warp within it = TMEM subpartition
  const int row = threadIdx.x & 127;                     // tile row = TMEM lane
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < 3; ++i) mbar_init(bars + i, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  for (int i = threadIdx.x; i < OFF_W / 16; i += 384) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  if (threadIdx.x < 2 * U) reinterpret_cast<float*>(smem + OFF_F)[threadIdx.x] =
      threadIdx.x < U ? gamma[threadIdx.x] : beta[threadIdx.x - U];
  stage_w_3xtf32(smem + OFF_W, W, threadIdx.x, 384);
  stage_bias_tile(smem + OFF_BT, bias, threadIdx.x, 384);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform_u32(*tmem_slot) + wg * ITC_TILE_COLS;   // this tile's columns
  const uint32_t tl = tmem + ((wq * 32u) << 16);                        // this warp's lanes of them
  constexpr uint32_t C_Z = 0, C_S = 64, C_X = 64, C_ONE = 160;
  const int s_loc = row / FP, f_loc = row - s_loc * FP;
  const bool in_tile = s_loc < SPT;
  {
    uint32_t one8[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) one8[i] = i < 2 ? 0x3F800000u : 0u;
    tc_st_32x8(tl + C_ONE, one8);
    tc_wait_st();
  }
  uint8_t* wsm = smem + wg * WG_BYTES;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t wb16 = (sbase + wg * WG_BYTES) >> 4;
  uint64_t* bar = bars + wg;
  const float4* gb4 = reinterpret_cast<const float4*>(smem + OFF_F);
  constexpr uint32_t ID_Z = make_idesc(2, 128, N4, 0, 0);               // tf32, N = 64
  constexpr uint32_t ID_S = make_idesc(2, 128, FP, 0, 0);               // tf32, N = FP, K = 8 per sample
  constexpr uint32_t ID_O = make_idesc(1, 128, 32, 0, 1);               // bf16, B = V MN-major, N = 32

  const int ntiles = (B + SPT - 1) / SPT;
  const float scale_log2 = ITC_LOG2E / sqrtf((float)DH);
  uint32_t phase = 0;
  // samples whose rows intersect this warp's 32 lanes (uniform)
  const uint32_t ws_lo = min((wq * 32u) / FP, (uint32_t)(SPT - 1)), ws_hi = min((wq * 32u + 31u) / FP, (uint32_t)(SPT - 1));
  const int64_t total_rows = (int64_t)B * F;
  float* lse_base = saved ? saved + (int64_t)L * total_rows * U : nullptr;
  const int tstride = (int)gridDim.x * 3;

  auto load_x = [&](int tile_, float (&dst)[D]) {
    const int64_t smp_ = (int64_t)tile_ * SPT + s_loc;
    if (in_tile && f_loc < F && smp_ < B) {
#pragma unroll
      for (int c = 0; c < D; c += 4) {
        const float4 t4 = load4<T>(x + smp_ * x_bs + (int64_t)f_loc * x_ld + c);
        dst[c] = t4.x; dst[c + 1] = t4.y; dst[c + 2] = t4.z; dst[c + 3] = t4.w;
      }
    } else {
#pragma unroll
      for (int c = 0; c < D; ++c) dst[c] = 0.f;
    }
  };
  // ---- fused lookup: id of (tile, row) ; its table row (raw fp32 bits, zeros for padding / idle rows)
  uint64_t g_R = 1;
  int64_t g_lb = 0;
  if (GATHER && in_tile && f_loc < F) { g_R = (uint64_t)ga.rows[f_loc]; g_lb = ga.lbase[f_loc]; }
  auto load_id = [&](int tile_) -> int64_t {
    const int64_t smp_ = (int64_t)tile_ * SPT + s_loc;
    if (tile_ < ntiles && in_tile && f_loc < F && smp_ < B) return ga.ids[smp_ * F + f_loc];
    return -1;
  };
  auto load_row = [&](int64_t id, uint32_t (&raw)[D], int32_t& lrow) {
    lrow = -1;
#pragma unroll
    for (int c = 0; c < D; ++c) raw[c] = 0u;
    if (id >= 0) {
      uint64_t rr;
      if (((uint64_t)id | g_R) >> 32) rr = (uint64_t)id % g_R;
      else rr = (uint32_t)id % (uint32_t)g_R;
      const uint32_t owner = ga.world == 1 ? 0u : (uint32_t)(rr % (uint64_t)ga.world);
      const int64_t lr = g_lb + (int64_t)(ga.world == 1 ? rr : rr / (uint64_t)ga.world);
      lrow = (int32_t)lr;
      ld_row64(ga.tab[owner] + lr * ga.tld, raw);
    }
  };
  // row consumed: X = RNE bf16 of the fp32 row (what the separate gather kernel writes), stored for the MLP tower
  // and the backward; the layer's input is that bf16 value; sort key of the lookup
  auto consume_row = [&](int tile_, const uint32_t (&raw)[D], int32_t lrow, float (&dst)[D]) {
    const int64_t smp_ = (int64_t)tile_ * SPT + s_loc;
    const bool act_ = in_tile && f_loc < F && smp_ < B;
    uint32_t pk[D / 2];
#pragma unroll
    for (int c = 0; c < D; c += 2) {
      pk[c / 2] = pack_bf16x2(__uint_as_float(raw[c]), __uint_as_float(raw[c + 1]));
      dst[c] = __uint_as_float(pk[c / 2] << 16);
      dst[c + 1] = __uint_as_float(pk[c / 2] & 0xFFFF0000u);
    }
    if (act_) {
      T* xo = x + smp_ * x_bs + (int64_t)f_loc * x_ld;
#pragma unroll
      for (int c = 0; c < D / 2; c += 2) *reinterpret_cast<uint2*>(xo + 2 * c) = make_uint2(pk[c], pk[c + 1]);
      if (!BAG && ga.keys) ga.keys[smp_ * F + f_loc] = ((uint64_t)(uint32_t)lrow << 32) | (uint64_t)(uint32_t)(smp_ * F + f_loc);
    }
  };
  // BAG: the mean of the valid rows of (tile, row)'s bag as fp32 bits, with embed_bag_fwd_kernel's arithmetic (fp32 sum
  // in slot order, times 1 / count; an empty bag is zeros); the slots' sort keys and the bag's 1 / count are written
  // here.  Slots are read ITC_BAG_CHUNK at a time: the chunk's ids, then its rows, all requests independent.
  int64_t b_lo = 0, b_n = 0;
  if constexpr (BAG) {
    if (in_tile && f_loc < F) { b_lo = ga.off[f_loc]; b_n = ga.off[f_loc + 1] - b_lo; }
  }
  auto load_bag = [&](int tile_, uint32_t (&raw)[D]) {
    if constexpr (BAG) {
      const int64_t smp_ = (int64_t)tile_ * SPT + s_loc;
      const bool act_ = tile_ < ntiles && in_tile && f_loc < F && smp_ < B;
      float acc[D];
#pragma unroll
      for (int c = 0; c < D; ++c) acc[c] = 0.f;
      int cnt = 0;
      const int64_t p0 = smp_ * ga.S + b_lo;
      for (int64_t k0 = 0; act_ && k0 < b_n; k0 += ITC_BAG_CHUNK) {
        int64_t id[ITC_BAG_CHUNK];
#pragma unroll
        for (int j = 0; j < ITC_BAG_CHUNK; ++j) id[j] = k0 + j < b_n ? ga.ids[p0 + k0 + j] : -1;
        uint32_t rv[ITC_BAG_CHUNK][D];
        int32_t lr[ITC_BAG_CHUNK];
#pragma unroll
        for (int j = 0; j < ITC_BAG_CHUNK; ++j) load_row(id[j], rv[j], lr[j]);
#pragma unroll
        for (int j = 0; j < ITC_BAG_CHUNK; ++j) {
          if (k0 + j < b_n) {
            const uint64_t p = (uint64_t)(p0 + k0 + j);
            if (ga.keys) ga.keys[p] = id[j] >= 0 ? ((uint64_t)(uint32_t)lr[j] << 32) | (uint64_t)(uint32_t)p : ~0ULL;
            if (id[j] >= 0) {
#pragma unroll
              for (int c = 0; c < D; ++c) acc[c] += __uint_as_float(rv[j][c]);
              ++cnt;
            }
          }
        }
      }
      const float inv = cnt > 0 ? 1.f / (float)cnt : 0.f;
#pragma unroll
      for (int c = 0; c < D; ++c) raw[c] = __float_as_uint(acc[c] * inv);
      if (act_) ga.inv_cnt[smp_ * F + f_loc] = inv;
    }
  };
  auto wg_sync = [&]() { named_bar_sync(1 + wg, 128); };

  int tile = (int)blockIdx.x * 3 + (int)wg;
  float xr[D];
  uint32_t rawn[D];              // GATHER: the next tile's table row in flight
  int32_t lrown = -1;
  int64_t idn = -1;              // GATHER: the id of the tile after the next
  if (BAG) {
    if (tile < ntiles) {
      load_bag(tile, rawn);
      consume_row(tile, rawn, lrown, xr);
    }
  } else if (GATHER) {
    if (tile < ntiles) {
      load_row(load_id(tile), rawn, lrown);
      consume_row(tile, rawn, lrown, xr);
      idn = load_id(tile + tstride);
    }
  } else if (tile < ntiles) {
    load_x(tile, xr);
  }
  for (; tile < ntiles; tile += tstride) {
    const int64_t smp = (int64_t)tile * SPT + s_loc;
    const bool active = in_tile && f_loc < F && smp < B;
    float yv[U], xn[D];
    for (int it = 0; it < L; ++it) {
      // ---- 1. [x_hi | x_lo] -> TMEM ; Z = [X | 1] [W ; b] (3xTF32: fp32-grade pre-activations, bias included)
      {
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int c = 0; c < D; ++c) {
          const float h_ = tf32_hi(xr[c]);
          hi[c] = __float_as_uint(h_);
          lo[c] = __float_as_uint(xr[c] - h_);
        }
        tc_st_32x16(tl + C_X, hi);
        tc_st_32x16(tl + C_X + 16, lo);
        tc_wait_st();
      }
      tc_fence_before();
      wg_sync();
      if (wq == 0 && elect_one()) {
        tc_fence_after();
        issue_proj_3xtf32_ts(tmem + C_Z, tmem + C_X, sbase + OFF_W, ID_Z);
        tc_mma_tf32_ts(tmem + C_Z, tmem + C_ONE, make_nosw_desc(sbase + OFF_BT, 128, 256), ID_Z, 1u);
        tc_commit(bar);
      }
      if (BAG) {
        // the next tile's bag means, summed while this tile's projection runs on the tensor cores
        if (it == 0 && tile + tstride < ntiles) load_bag(tile + tstride, rawn);
      } else if (GATHER) {
        // the id fetched a tile ago turns into the next tile's row loads; the id of the tile after it is requested
        // (requested at the tile's FIRST iteration: a whole tile, ~10 us, of cover for the NVLink round trip)
        if (it == 0 && tile + tstride < ntiles) { load_row(idn, rawn, lrown); idn = load_id(tile + 2 * tstride); }
      } else if (it + 1 == L && tile + tstride < ntiles) {
        load_x(tile + tstride, xn);                                     // next tile's rows: a whole step of cover
      }
      mbar_wait(bar, phase); phase ^= 1u;
      tc_fence_after();
      float r[U];
      {
        uint32_t z[32], zvr[32];
        tc_ld_32x32(tl + C_Z, z);                                      // q | k
        tc_ld_32x32(tl + C_Z + 32, zvr);                               // v | r   (all of Z in registers: its columns are reused)
#pragma unroll
        for (int u = 0; u < 2 * U; ++u) z[u] = __float_as_uint(fmaxf(__uint_as_float(z[u]), 0.f));
#pragma unroll
        for (int h = 0; h < H; ++h) {
          // every sample slot is rewritten (zeros outside the row's own sample): the columns held Z a moment ago
#pragma unroll
          for (int s = 0; s < SPT; ++s) {
            uint32_t v8[8];
#pragma unroll
            for (int e = 0; e < DH; ++e) v8[e] = s == s_loc ? z[h * DH + e] : 0u;
            tc_st_32x8(tl + C_Z + h * 32 + s * 8, v8);
          }
          if (in_tile) {
#pragma unroll
            for (int c = 0; c < 2; ++c)
              *reinterpret_cast<uint4*>(wsm + OFF_KX + h * G::KX_BYTES + nosw_off<NCHK>(f_loc, s_loc * 2 + c)) =
                  make_uint4(z[U + h * DH + c * 4], z[U + h * DH + c * 4 + 1], z[U + h * DH + c * 4 + 2], z[U + h * DH + c * 4 + 3]);
          }
        }
        if (in_tile) {
#pragma unroll
          for (int h = 0; h < H; ++h) {
            float vv[DH];
#pragma unroll
            for (int e = 0; e < DH; ++e) vv[e] = fmaxf(__uint_as_float(zvr[h * DH + e]), 0.f);
            uint4 v;
            v.x = pack_bf16x2(vv[0], vv[1]); v.y = pack_bf16x2(vv[2], vv[3]);
            v.z = pack_bf16x2(vv[4], vv[5]); v.w = pack_bf16x2(vv[6], vv[7]);
            *reinterpret_cast<uint4*>(wsm + OFF_VX + h * G::VX_BYTES + nosw_off<4>(f_loc, s_loc)) = v;
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) r[u] = fmaxf(__uint_as_float(zvr[U + u]), 0.f);
      }
      // ---- 2. S_h[row, j] = q_row . k_(own sample, j): the Q operand is expanded along K by sample (zeros in the
      //         other samples' slots), so all 128 rows read THEIR keys from the same FP columns
      fence_async_smem();
      tc_wait_st();
      tc_fence_before();
      wg_sync();
      if (wq == 0 && elect_one()) {
        tc_fence_after();
#pragma unroll
        for (int h = 0; h < H; ++h)
#pragma unroll
          for (int ks = 0; ks < SPT; ++ks)
            tc_mma_tf32_ts(tmem + C_S + h * FP, tmem + C_Z + h * 32 + ks * 8,
                           mk_desc(wb16, OFF_KX + h * G::KX_BYTES + ks * 256, 128, NCHK * 128), ID_S, ks ? 1u : 0u);
        tc_commit(bar);
      }
      mbar_wait(bar, phase); phase ^= 1u;
      tc_fence_after();
      float linv[H], lse2[H];
#pragma unroll
      for (int h = 0; h < H; ++h) {
        float p[FP];
        {
          uint32_t t[FP];
#pragma unroll
          for (int c0 = 0; c0 < FP; c0 += 8) {
            uint32_t t8[8];
            tc_ld_32x8(tl + C_S + h * FP + c0, t8);
#pragma unroll
            for (int j = 0; j < 8; ++j) t[c0 + j] = t8[j];
          }
          tc_wait_ld();
#pragma unroll
          for (int j = 0; j < FP; ++j) p[j] = (j < FMIN || j < F) ? __uint_as_float(t[j]) : -INFINITY;
        }
        float m4[4] = {p[0], p[1], p[2], p[3]};
#pragma unroll
        for (int j = 4; j + 1 < FP; j += 2) m4[(j >> 1) & 3] = fmax3(m4[(j >> 1) & 3], p[j], p[j + 1]);
        const float m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
        const float mb = m * scale_log2;
        const float2 c2 = make_float2(scale_log2, scale_log2), nmb2 = make_float2(-mb, -mb);
        float2 l2[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) l2[i] = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < FP; j += 2) {
          float2 t0 = ffma2(make_float2(p[j], p[j + 1]), c2, nmb2);
          t0.x = ex2_approx(t0.x); t0.y = ex2_approx(t0.y);
          l2[(j >> 1) & 3] = fadd2(l2[(j >> 1) & 3], t0);
          p[j] = t0.x; p[j + 1] = t0.y;
        }
        const float2 lt = fadd2(fadd2(l2[0], l2[1]), fadd2(l2[2], l2[3]));
        const float l = lt.x + lt.y;
        linv[h] = 1.f / l;
        lse2[h] = mb + lg2_approx(l);
        // unnormalised bf16 P row -> TMEM (A operand of P.V), zero beyond the FP keys
#pragma unroll
        for (int c0 = 0; c0 < KP / 2; c0 += 8) {
          uint32_t v8[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int j = (c0 + e) * 2;
            v8[e] = j < FP ? pack_bf16x2(p[j < FP ? j : 0], p[j + 1 < FP ? j + 1 : 0]) : 0u;
          }
          tc_st_32x8(tl + C_S + h * FP + c0, v8);
        }
      }
      // ---- 3. O_h[row, (s, e)] = sum_j P[row, j] v_(s, j)[e]; a row keeps the 8 columns of its own sample
      tc_wait_st();
      tc_fence_before();
      wg_sync();
      if (wq == 0 && elect_one()) {
        tc_fence_after();
#pragma unroll
        for (int h = 0; h < H; ++h)
#pragma unroll
          for (int ks = 0; ks < KP / 16; ++ks)
            tc_mma_bf16_ts(tmem + C_Z + h * 32, tmem + C_S + h * FP + ks * 8,
                           mk_desc(wb16, OFF_VX + h * G::VX_BYTES + ks * 1024, 512, 128), ID_O, ks ? 1u : 0u);
        tc_commit(bar);
      }
      if (active && saved) {
        float* lp = lse_base + ((int64_t)it * total_rows + smp * F + f_loc) * H;
        *reinterpret_cast<float2*>(lp) = make_float2(lse2[0], lse2[1]);
      }
      mbar_wait(bar, phase); phase ^= 1u;
      tc_fence_after();
      {
        float o[U];
#pragma unroll
        for (int u = 0; u < U; ++u) o[u] = 0.f;
        for (uint32_t s = ws_lo; s <= ws_hi; ++s) {
          uint32_t t0[8], t1[8];
          tc_ld_32x8(tl + C_Z + s * 8, t0);
          tc_ld_32x8(tl + C_Z + 32 + s * 8, t1);
          tc_wait_ld();
          if ((int)s == s_loc) {
#pragma unroll
            for (int e = 0; e < DH; ++e) { o[e] = __uint_as_float(t0[e]); o[DH + e] = __uint_as_float(t1[e]); }
          }
        }
        // residual, ReLU, LayerNorm (InteractingLayer.py:57-60)
        float a[U], mean, rstd;
#pragma unroll
        for (int u = 0; u < U; ++u) a[u] = fmaxf(use_res ? fmaf(o[u], linv[u / DH], r[u]) : o[u] * linv[u / DH], 0.f);
        ln_row_stats<U>(a, eps, mean, rstd);
#pragma unroll
        for (int u4 = 0; u4 < U / 4; ++u4) {
          const float4 g4 = gb4[u4], b4 = gb4[U / 4 + u4];
          yv[u4 * 4 + 0] = ln_apply(a[u4 * 4 + 0], mean, rstd, g4.x, b4.x);
          yv[u4 * 4 + 1] = ln_apply(a[u4 * 4 + 1], mean, rstd, g4.y, b4.y);
          yv[u4 * 4 + 2] = ln_apply(a[u4 * 4 + 2], mean, rstd, g4.z, b4.z);
          yv[u4 * 4 + 3] = ln_apply(a[u4 * 4 + 3], mean, rstd, g4.w, b4.w);
        }
        // saved for the backward: the pre-LayerNorm activations of EVERY iteration (the backward
        // re-derives each iteration's input as LayerNorm(a) and differentiates ReLU/LayerNorm at a)
        if (active && saved) {
          float* sp = saved + ((int64_t)it * total_rows + smp * F + f_loc) * U;
#pragma unroll
          for (int u = 0; u < U; u += 4) *reinterpret_cast<float4*>(sp + u) = make_float4(a[u], a[u + 1], a[u + 2], a[u + 3]);
        }
      }
      if (it + 1 < L) {
#pragma unroll
        for (int u = 0; u < U; ++u) xr[u] = active ? yv[u] : 0.f;
      }
    }
    if (active) {
#pragma unroll
      for (int u = 0; u < U; u += 4)
        store4<T>(y + smp * y_bs + (int64_t)f_loc * y_ld + u, make_float4(yv[u], yv[u + 1], yv[u + 2], yv[u + 3]));
    }
    if (GATHER) {
      if (tile + tstride < ntiles) consume_row(tile + tstride, rawn, lrown, xr);
    } else {
#pragma unroll
      for (int c = 0; c < D; ++c) xr[c] = xn[c];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512));
  }
}

template <int NCHF, typename T>
static int launch_itc_fwd(const IFwdArgs& a) {
  using G = ItcGeom<NCHF>;
  constexpr int smem = 3 * (2 * G::KX_BYTES + 2 * G::VX_BYTES) + 8192 + 2048 + 128 + 64;
  const int ntiles = (a.B + G::SPT - 1) / G::SPT;
  int grid = sm_count();
  if (grid * 3 > ntiles) grid = (ntiles + 2) / 3;
  // (A grid trimmed to the number of rounds — 2731 tiles need 7 rounds of three tile streams on 148 CTAs and still 7 on
  // 131 — leaves 17 SMs to the step's other branches.  Measured on one and two GPUs: the key sort / NCCL kernels that
  // moved there ran 3x slower on so few SMs and slowed the step; every SM takes part.)
  ItcGather ga{};
  if (a.gather && a.gather->bag_off) {
    ItcBagGather gb{};
    gb.tab[0] = a.gather->tables[0];
    gb.tld = a.gather->table_ld; gb.world = 1; gb.ids = a.gather->ids; gb.lbase = a.gather->local_base;
    gb.rows = a.gather->rows; gb.keys = a.gather->sort_keys;
    gb.off = a.gather->bag_off; gb.inv_cnt = a.gather->inv_cnt; gb.S = a.gather->bag_slots;
    auto kern = interacting_tc_fwd_kernel<NCHF, T, true, ItcBagGather>;
    RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<grid, 384, smem, a.st>>>(gb, (T*)a.x, a.x_ld, a.x_bs, a.W, a.b, a.gm, a.bt, a.eps, (T*)a.y, a.y_ld, a.y_bs,
                                    (float*)a.saved, a.B, a.F, a.L, a.use_res);
  } else if (a.gather) {
    for (int r = 0; r < RS_MAX_PEERS; ++r) ga.tab[r] = r < a.gather->world ? a.gather->tables[r] : nullptr;
    ga.tld = a.gather->table_ld; ga.world = a.gather->world; ga.ids = a.gather->ids; ga.lbase = a.gather->local_base;
    ga.rows = a.gather->rows; ga.keys = a.gather->sort_keys;
    auto kern = interacting_tc_fwd_kernel<NCHF, T, true>;
    RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<grid, 384, smem, a.st>>>(ga, (T*)a.x, a.x_ld, a.x_bs, a.W, a.b, a.gm, a.bt, a.eps, (T*)a.y, a.y_ld, a.y_bs,
                                    (float*)a.saved, a.B, a.F, a.L, a.use_res);
  } else {
    auto kern = interacting_tc_fwd_kernel<NCHF, T, false>;
    RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<grid, 384, smem, a.st>>>(ga, (T*)a.x, a.x_ld, a.x_bs, a.W, a.b, a.gm, a.bt, a.eps, (T*)a.y, a.y_ld, a.y_bs,
                                    (float*)a.saved, a.B, a.F, a.L, a.use_res);
  }
  return check_launch("interacting_tc_fwd");
}

// Returns RS_ERR_UNSUPPORTED (without setting an error) when the shape is not built for the
// tensor-core path; the caller then uses the FFMA kernels.
// Built for D = U = 16, 2 heads, bf16 activations and up to 48 fields: a tile holds floor(128 / FP) whole samples
// with FP = F rounded up to 8 (F = 39 -> 3 samples, 26 -> 4, 16 -> 8, 48 -> 2).
bool interacting_tc_supported(int F, int D, int U, int H, int dtype) {
  return dtype == RS_BF16 && D == 16 && U == 16 && H == 2 && F >= 1 && F <= 48;
}

int interacting_tc_fwd(const IFwdArgs& a) {
  switch ((a.F + 7) / 8) {
    case 1:                                                            // N = 8 is not an M = 128 shape
    case 2: return launch_itc_fwd<2, __nv_bfloat16>(a);
    case 3: return launch_itc_fwd<3, __nv_bfloat16>(a);
    case 4: return launch_itc_fwd<4, __nv_bfloat16>(a);
    case 5: return launch_itc_fwd<5, __nv_bfloat16>(a);
    default: return launch_itc_fwd<6, __nv_bfloat16>(a);
  }
}

}  // namespace rs
