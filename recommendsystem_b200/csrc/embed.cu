// embed.cu — K1/K2 embedding gather, K3 sorted-segment gradient + fused sparse
// optimizers, K7 id routing.  All HBM-bound integer / copy work: the design
// goals are full-sector coalescing (a thread group covers one whole row with
// 16-B loads), many independent loads in flight per lane, and index math done
// once per lookup per warp (one lane per lookup, then shuffled to the group).
#include "common.cuh"
#include <cub/device/device_radix_sort.cuh>

namespace rs {

// ---------------------------------------------------------------- gather ---
// One warp handles 32*LPL lookups per iteration.
//   phase 1: lane l owns lookups base + l (+32, ...): loads the id (coalesced),
//            reduces it to an arena row with 32-bit math when it fits, emits
//            the sort key / row index.
//   phase 2: the warp is split in 32/G groups of G lanes; in step s group j
//            serves lookup s*(32/G)+j: the owning lane's row is shuffled in,
//            every lane of the group loads 16 B of the row.  All G*LPL loads
//            are issued before the first store.
template <int G, int LPL, typename OutT, bool FROM_IDS>
__global__ void __launch_bounds__(128)
embed_gather_kernel(const float* __restrict__ table, const int64_t* __restrict__ ids,
                    const int32_t* __restrict__ rowidx,
                    const int64_t* __restrict__ row_base, const int64_t* __restrict__ rows,
                    int64_t n, int F, int d, int64_t tld, OutT* __restrict__ out,
                    uint64_t* __restrict__ sort_keys, int32_t* __restrict__ rows_out,
                    uint8_t* __restrict__ mask_out) {
  constexpr int GROUPS = 32 / G;  // lookups served per step
  const int lane = threadIdx.x & 31;
  const int gl = lane % G;        // lane within group
  const int gj = lane / G;        // group within warp
  const int64_t warp_global = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const bool col_ok = gl * 4 < d;

  for (int64_t base = warp_global * (32 * LPL); base < n; base += nwarps * (32 * LPL)) {
    int32_t myrow[LPL];
#pragma unroll
    for (int k = 0; k < LPL; ++k) {
      const int64_t i = base + k * 32 + lane;
      int32_t r = -1;
      if (i < n) {
        if (FROM_IDS) {
          const int64_t id = ids[i];
          if (id >= 0) {
            int f;
            if (n < (int64_t)0x7fffffff) f = (int)((uint32_t)i % (uint32_t)F);
            else f = (int)(i % F);
            const uint64_t R = (uint64_t)__ldg(rows + f);
            uint64_t rr;
            if (((uint64_t)id | R) >> 32) rr = (uint64_t)id % R;
            else rr = (uint32_t)id % (uint32_t)R;
            r = (int32_t)(__ldg(row_base + f) + (int64_t)rr);
          }
        } else {
          r = rowidx[i];
        }
        if (sort_keys) sort_keys[i] = ((uint64_t)(uint32_t)r << 32) | (uint64_t)(uint32_t)i;
        if (rows_out) rows_out[i] = r;
        if (mask_out) mask_out[i] = r >= 0 ? 1 : 0;
      }
      myrow[k] = r;
    }

    float4 v[LPL][G];
#pragma unroll
    for (int k = 0; k < LPL; ++k) {
#pragma unroll
      for (int s = 0; s < G; ++s) {
        const int src = s * GROUPS + gj;
        const int32_t r = __shfl_sync(0xffffffffu, myrow[k], src);
        v[k][s] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r >= 0 && col_ok && out)
          v[k][s] = ldg_row_f4(reinterpret_cast<const float4*>(table + (int64_t)r * tld) + gl);
      }
    }
#pragma unroll
    for (int k = 0; k < LPL; ++k) {
#pragma unroll
      for (int s = 0; s < G; ++s) {
        const int64_t i = base + k * 32 + s * GROUPS + gj;
        if (i < n && col_ok && out) store4<OutT>(out + i * d + gl * 4, v[k][s]);
      }
    }
  }
}

template <int G, int LPL, bool FROM_IDS>
static int launch_gather(const float* table, int64_t tld, const int64_t* ids, const int32_t* rowidx,
                         const int64_t* row_base, const int64_t* rows, int64_t n, int F,
                         int d, void* out, int out_dtype, uint64_t* sort_keys,
                         int32_t* rows_out, uint8_t* mask_out, cudaStream_t st) {
  const int threads = 128;
  const int64_t per_block = (int64_t)(threads / 32) * 32 * LPL;
  int64_t blocks = cdiv(n, per_block);
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  if (out_dtype == RS_F32)
    embed_gather_kernel<G, LPL, float, FROM_IDS><<<(unsigned)blocks, threads, 0, st>>>(
        table, ids, rowidx, row_base, rows, n, F, d, tld, (float*)out, sort_keys, rows_out, mask_out);
  else
    embed_gather_kernel<G, LPL, __nv_bfloat16, FROM_IDS><<<(unsigned)blocks, threads, 0, st>>>(
        table, ids, rowidx, row_base, rows, n, F, d, tld, (__nv_bfloat16*)out, sort_keys, rows_out,
        mask_out);
  return check_launch("embed_gather");
}

template <bool FROM_IDS>
static int dispatch_gather(const float* table, int64_t tld, const int64_t* ids, const int32_t* rowidx,
                           const int64_t* row_base, const int64_t* rows, int64_t n, int F,
                           int d, void* out, int out_dtype, uint64_t* sort_keys,
                           int32_t* rows_out, uint8_t* mask_out, cudaStream_t st) {
  RS_REQUIRE(d > 0 && d % 4 == 0 && d <= 128, "embed_gather: d=%d must be a multiple of 4, <= 128", d);
  RS_REQUIRE(out_dtype == RS_F32 || out_dtype == RS_BF16, "embed_gather: bad out dtype %d", out_dtype);
  RS_REQUIRE(n >= 0 && n < ((int64_t)1 << 32), "embed_gather: n=%lld out of range", (long long)n);
  if (n == 0) return 0;
  if (tld == 0) tld = d;
  RS_REQUIRE(tld >= d && tld % 4 == 0, "embed_gather: table row stride %lld (d = %d)", (long long)tld, d);
  const int g = d / 4;
#define RS_GATHER_CASE(G, LPL)                                                                  \
  return launch_gather<G, LPL, FROM_IDS>(table, tld, ids, rowidx, row_base, rows, n, F, d, out, \
                                         out_dtype, sort_keys, rows_out, mask_out, st)
  if (g <= 1) RS_GATHER_CASE(1, 4);
  if (g <= 2) RS_GATHER_CASE(2, 4);
  if (g <= 4) RS_GATHER_CASE(4, 2);
  if (g <= 8) RS_GATHER_CASE(8, 1);
  if (g <= 16) RS_GATHER_CASE(16, 1);
  RS_GATHER_CASE(32, 1);
#undef RS_GATHER_CASE
}

// ------------------------------------------------ gather over peer memory ----
// Row-sharded tables, one process per GPU: owner(row) = row mod W, local row = local_base[f] + row div W
// (SURVEY §8e).  Instead of routing ids to the owners and shipping rows back with two all-to-alls,
// every rank reads the rows it needs straight out of the owners' HBM over NVLink / NVSwitch: the W
// shard base pointers are CUDA-IPC mappings (rs_ipc_export / rs_ipc_import) and a lookup is one
// 64-byte peer load.  Same warp shape as embed_gather_kernel (G lanes x 16 B per row, G*LPL loads in
// flight per lane).  Peer rows are written only by their owner's sparse update of the PREVIOUS step,
// which a cross-rank barrier orders before this kernel; plain (coherent) loads, no .nc.
struct PeerTables { const float* p[RS_MAX_PEERS]; };

__device__ __forceinline__ float4 ld_peer_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p) : "memory");
  return r;
}

template <int G, int LPL, typename OutT>
__global__ void __launch_bounds__(128)
embed_gather_peer_kernel(PeerTables tabs, const int64_t* __restrict__ ids, const int64_t* __restrict__ local_base,
                         const int64_t* __restrict__ rows, int64_t n, int F, int d, int64_t tld, int W,
                         OutT* __restrict__ out) {
  constexpr int GROUPS = 32 / G;
  const int lane = threadIdx.x & 31;
  const int gl = lane % G, gj = lane / G;
  const int64_t warp_global = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const bool col_ok = gl * 4 < d;
  for (int64_t base = warp_global * (32 * LPL); base < n; base += nwarps * (32 * LPL)) {
    const float* myptr[LPL];
#pragma unroll
    for (int k = 0; k < LPL; ++k) {
      const int64_t i = base + k * 32 + lane;
      const float* ptr = nullptr;
      if (i < n) {
        const int64_t id = ids[i];
        if (id >= 0) {
          const int f = (int)(i % F);
          const uint64_t R = (uint64_t)__ldg(rows + f);
          uint64_t rr;
          if (((uint64_t)id | R) >> 32) rr = (uint64_t)id % R;
          else rr = (uint32_t)id % (uint32_t)R;
          const uint32_t owner = (uint32_t)(rr % (uint64_t)W);
          const int64_t lrow = __ldg(local_base + f) + (int64_t)(rr / (uint64_t)W);
          ptr = tabs.p[owner] + lrow * tld;
        }
      }
      myptr[k] = ptr;
    }
    float4 v[LPL][G];
#pragma unroll
    for (int k = 0; k < LPL; ++k) {
#pragma unroll
      for (int s = 0; s < G; ++s) {
        const int src = s * GROUPS + gj;
        const float* r = reinterpret_cast<const float*>(
            __shfl_sync(0xffffffffu, (unsigned long long)(uintptr_t)myptr[k], src));
        v[k][s] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r != nullptr && col_ok) v[k][s] = ld_peer_f4(reinterpret_cast<const float4*>(r) + gl);
      }
    }
#pragma unroll
    for (int k = 0; k < LPL; ++k) {
#pragma unroll
      for (int s = 0; s < G; ++s) {
        const int64_t i = base + k * 32 + s * GROUPS + gj;
        if (i < n && col_ok) store4<OutT>(out + i * d + gl * 4, v[k][s]);
      }
    }
  }
}

template <int G, int LPL>
static int launch_gather_peer(const PeerTables& tabs, const int64_t* ids, const int64_t* local_base,
                              const int64_t* rows, int64_t n, int F, int d, int64_t tld, int W, void* out,
                              int out_dtype, cudaStream_t st) {
  const int threads = 128;
  const int64_t per_block = (int64_t)(threads / 32) * 32 * LPL;
  int64_t blocks = cdiv(n, per_block);
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  if (out_dtype == RS_F32)
    embed_gather_peer_kernel<G, LPL, float><<<(unsigned)blocks, threads, 0, st>>>(tabs, ids, local_base, rows, n, F, d,
                                                                                  tld, W, (float*)out);
  else
    embed_gather_peer_kernel<G, LPL, __nv_bfloat16><<<(unsigned)blocks, threads, 0, st>>>(
        tabs, ids, local_base, rows, n, F, d, tld, W, (__nv_bfloat16*)out);
  return check_launch("embed_gather_peer");
}

// ------------------------------------------------------------- bag mean ----
// One group of G lanes per bag; ids of a bag are walked in order (mean is the
// fp32 sum in id order divided by the count — the order tf's
// embedding_lookup_sparse(combiner='mean') segment-sum uses).
template <typename OutT>
__global__ void embed_bag_mean_kernel(const float* __restrict__ table,
                                      const int64_t* __restrict__ ids,
                                      const int64_t* __restrict__ offsets,
                                      const int64_t* __restrict__ row_base,
                                      const int64_t* __restrict__ rows, int64_t n_bags, int F,
                                      int d, int G, OutT* __restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t bag = t / G;
  const int gl = (int)(t % G);
  if (bag >= n_bags || gl * 4 >= d) return;
  const int f = (int)(bag % F);
  const int64_t lo = offsets[bag], hi = offsets[bag + 1];
  const uint64_t R = (uint64_t)rows[f];
  const int64_t rb = row_base[f];
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int cnt = 0;
  for (int64_t p = lo; p < hi; ++p) {
    const int64_t id = ids[p];
    if (id < 0) continue;
    const int64_t r = rb + (int64_t)((uint64_t)id % R);
    const float4 v = ldg_nc_f4(reinterpret_cast<const float4*>(table + r * d) + gl);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    ++cnt;
  }
  if (cnt > 0) {
    const float inv = (float)cnt;
    acc.x /= inv; acc.y /= inv; acc.z /= inv; acc.w /= inv;
  }
  store4<OutT>(out + bag * d + gl * 4, acc);
}


// CSR bags for TRAINING: mean over the valid ids of bag b (combiner='mean' on VarLenFeature ids, staytime/parse.py:22-23,
// staytime/VideoDnn.py:224-226) from a table with an explicit row stride ([w|m|v] records), plus what the backward needs:
// sort_keys[p] = (row << 32 | p) per occurrence p (padding / empty -> all-ones key, skipped by the segment sum) and
// inv_cnt[b] = 1 / (number of valid ids of bag b) (0 for an empty bag).
template <typename OutT>
__global__ void embed_bag_fwd_kernel(const float* __restrict__ table, int64_t table_ld, const int64_t* __restrict__ ids,
                                     const int64_t* __restrict__ offsets, const int64_t* __restrict__ row_base,
                                     const int64_t* __restrict__ rows, int64_t n_bags, int F, int d, int G,
                                     OutT* __restrict__ out, uint64_t* __restrict__ sort_keys, float* __restrict__ inv_cnt) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t bag = t / G;
  const int gl = (int)(t % G);
  if (bag >= n_bags || gl * 4 >= d) return;
  const int f = (int)(bag % F);
  const int64_t lo = offsets[bag], hi = offsets[bag + 1];
  const uint64_t R = (uint64_t)rows[f];
  const int64_t rb = row_base[f];
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int cnt = 0;
  for (int64_t p = lo; p < hi; ++p) {
    const int64_t id = ids[p];
    if (id < 0) {
      if (gl == 0 && sort_keys) sort_keys[p] = ~0ULL;
      continue;
    }
    const int64_t r = rb + (int64_t)((uint64_t)id % R);
    if (gl == 0 && sort_keys) sort_keys[p] = ((uint64_t)r << 32) | (uint64_t)(uint32_t)p;
    const float4 v = ldg_row_f4(reinterpret_cast<const float4*>(table + r * table_ld) + gl);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    ++cnt;
  }
  const float inv = cnt > 0 ? 1.f / (float)cnt : 0.f;
  acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv;
  store4<OutT>(out + bag * d + gl * 4, acc);
  if (gl == 0 && inv_cnt) inv_cnt[bag] = inv;
}

// backward of the mean combiner: occurrence p of bag b receives dout[b] / count(b)  (one row per occurrence, the
// layout the sorted-segment sum consumes)
template <typename T>
__global__ void embed_bag_grad_kernel(const T* __restrict__ dout, const int64_t* __restrict__ offsets,
                                      const float* __restrict__ inv_cnt, int64_t n_bags, int d, int G,
                                      float* __restrict__ g_occ) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t bag = t / G;
  const int gl = (int)(t % G);
  if (bag >= n_bags || gl * 4 >= d) return;
  const float4 g = load4<T>(dout + bag * d + gl * 4);
  const float s = inv_cnt[bag];
  const float4 v = make_float4(g.x * s, g.y * s, g.z * s, g.w * s);
  for (int64_t p = offsets[bag]; p < offsets[bag + 1]; ++p)
    *reinterpret_cast<float4*>(g_occ + p * d + gl * 4) = v;
}

// ----------------------------------------------- segment sum + optimizers ---
enum { OPT_NONE = 0, OPT_ADAM = 1, OPT_ADAGRAD_ROW = 2, OPT_ADAGRAD_ELEM = 3 };

struct OptArgs {
  float* w; float* s0; float* s1;   // adam: m, v ; adagrad: g2sum, -
  float lr, beta1, beta2, eps;
  int64_t ld;                       // row stride of w / s0 / s1 in floats (d, or 3d for interleaved [w|m|v] rows)
  const float* scalars;             // device {step, b1^t, b2^t, corr}
  float grad_scale;
  int32_t* seg_rows; float* seg_sum; // OPT_NONE outputs
};

template <typename GT>
__device__ __forceinline__ float4 load_grad(const GT* grad, uint32_t pos, int d, int gl, float sc) {
  float4 g = load4<GT>(grad + (int64_t)pos * d + gl * 4);
  g.x *= sc; g.y *= sc; g.z *= sc; g.w *= sc;
  return g;
}

// Same warp structure as the gather: lane l owns sorted position base+l
// (key, predecessor and successor rows are exchanged by shuffle), then group
// j serves position s*(32/G)+j in step s.  Only segment HEADS do work: the
// head's group walks its run left-to-right (fixed order => deterministic) and
// applies the optimizer once.  With uniform ids almost every position is a
// head of a length-1 run, so the G steps issue G independent grad loads and
// then 2-3 independent state-row loads each.
template <int G, int OPT, typename GT>
__global__ void __launch_bounds__(128)
embed_segsum_kernel(const uint64_t* __restrict__ keys, const GT* __restrict__ grad, int64_t n,
                    int d, OptArgs a) {
  constexpr int GROUPS = 32 / G;
  const int lane = threadIdx.x & 31;
  const int gl = lane % G;
  const int gj = lane / G;
  const int64_t warp_global = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const bool col_ok = gl * 4 < d;
  float lr_eff = a.lr;
  if (OPT == OPT_ADAM) lr_eff = a.lr * __ldg(a.scalars + 3);

  for (int64_t base = warp_global * 32; base < n; base += nwarps * 32) {
    const int64_t i = base + lane;
    uint64_t key = ~0ull;
    if (i < n) key = keys[i];
    uint32_t row = (uint32_t)(key >> 32);
    uint32_t prev = __shfl_up_sync(0xffffffffu, row, 1);
    uint32_t next = __shfl_down_sync(0xffffffffu, row, 1);
    if (lane == 0) prev = (base > 0) ? (uint32_t)(keys[base - 1] >> 32) : 0xffffffffu;
    if (lane == 31) next = (base + 32 < n) ? (uint32_t)(keys[base + 32] >> 32) : 0xffffffffu;
    // a head: first of its run, and a real (non-padding) row
    const bool head = (i < n) && (row != 0xffffffffu) && (i == 0 || row != prev);
    const bool more = head && (i + 1 < n) && (next == row);

    float4 acc[G];
    uint32_t srow[G];
    bool shead[G];
#pragma unroll
    for (int s = 0; s < G; ++s) {
      const int src = s * GROUPS + gj;
      srow[s] = __shfl_sync(0xffffffffu, row, src);
      shead[s] = __shfl_sync(0xffffffffu, (int)head, src) != 0;
      const uint32_t pos = __shfl_sync(0xffffffffu, (uint32_t)key, src);
      acc[s] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (shead[s] && col_ok) acc[s] = load_grad<GT>(grad, pos, d, gl, a.grad_scale);
    }
    // Adam: the state rows depend on the keys only — request them together with the gradient rows (two
    // dependent DRAM round trips per warp instead of three)
    float4 w[G], m[G], v[G];
    if (OPT == OPT_ADAM) {
#pragma unroll
      for (int s = 0; s < G; ++s) {
        if (shead[s] && col_ok) {
          const int64_t off = (int64_t)srow[s] * a.ld + gl * 4;
          w[s] = ld_row_f4(reinterpret_cast<const float4*>(a.w + off));
          m[s] = ld_row_f4(reinterpret_cast<const float4*>(a.s0 + off));
          v[s] = ld_row_f4(reinterpret_cast<const float4*>(a.s1 + off));
        }
      }
    }
    // runs longer than one: the head's group walks the rest of the run in order — inside this warp's 32-key
    // window only (at most 31 steps).
    const int64_t wend = base + 32 < n ? base + 32 : n;
#pragma unroll
    for (int s = 0; s < G; ++s) {
      const int src = s * GROUPS + gj;
      const bool smore = __shfl_sync(0xffffffffu, (int)more, src) != 0;
      if (smore && col_ok) {
        int64_t q = base + src + 1;
        while (q < wend) {
          const uint64_t kq = keys[q];
          if ((uint32_t)(kq >> 32) != srow[s]) break;
          const float4 g = load_grad<GT>(grad, (uint32_t)kq, d, gl, a.grad_scale);
          acc[s].x += g.x; acc[s].y += g.y; acc[s].z += g.z; acc[s].w += g.w;
          ++q;
        }
      }
    }
    // A run that leaves the window (skewed ids: a hot row can occur thousands of times in a batch) can only be
    // the window's LAST run.  If its head is in this window, the whole warp continues it: 32 keys per trip, their
    // gradient rows loaded by all lane groups at once, then added ONE ROW AT A TIME IN POSITION ORDER — the
    // same left-to-right fp32 sum as the sequential walk (bit-identical), without its dependent-load chain.
    {
      const uint32_t row_last = __shfl_sync(0xffffffffu, row, 31);
      const uint32_t next_last = __shfl_sync(0xffffffffu, next, 31);
      const uint32_t same = __ballot_sync(0xffffffffu, row == row_last);
      const int hi = __ffs(same) - 1;                                  // first key of the last run inside the window
      const bool hi_is_head = __shfl_sync(0xffffffffu, (int)head, hi) != 0;
      if (row_last != 0xffffffffu && base + 32 < n && next_last == row_last && hi_is_head) {   // warp-uniform
        const int s_h = hi / GROUPS, g_h = hi % GROUPS;
        float4 run = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int s = 0; s < G; ++s)
          if (s == s_h) run = acc[s];
        run.x = __shfl_sync(0xffffffffu, run.x, g_h * G + gl); run.y = __shfl_sync(0xffffffffu, run.y, g_h * G + gl);
        run.z = __shfl_sync(0xffffffffu, run.z, g_h * G + gl); run.w = __shfl_sync(0xffffffffu, run.w, g_h * G + gl);
        int64_t q = base + 32;
        bool done = false;
        while (!done) {
          const uint64_t kq = (q + lane < n) ? keys[q + lane] : ~0ull;
          const uint32_t mt = __ballot_sync(0xffffffffu, (uint32_t)(kq >> 32) == row_last);
          const int cnt = mt == 0xffffffffu ? 32 : __ffs(~mt) - 1;    // sorted keys: the matches are a prefix
          float4 v[G];
#pragma unroll
          for (int t = 0; t < G; ++t) {                                // group gj loads rows t*GROUPS + gj
            const int pidx = t * GROUPS + gj;
            const uint32_t pos = __shfl_sync(0xffffffffu, (uint32_t)kq, pidx);
            v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (pidx < cnt && col_ok) v[t] = load_grad<GT>(grad, pos, d, gl, a.grad_scale);
          }
#pragma unroll
          for (int t = 0; t < G; ++t) {
#pragma unroll
            for (int j = 0; j < GROUPS; ++j) {
              if (t * GROUPS + j < cnt) {                             // warp-uniform
                run.x += __shfl_sync(0xffffffffu, v[t].x, j * G + gl); run.y += __shfl_sync(0xffffffffu, v[t].y, j * G + gl);
                run.z += __shfl_sync(0xffffffffu, v[t].z, j * G + gl); run.w += __shfl_sync(0xffffffffu, v[t].w, j * G + gl);
              }
            }
          }
          q += 32;
          done = cnt < 32 || q >= n;
        }
        if (gj == g_h) {
#pragma unroll
          for (int s = 0; s < G; ++s)
            if (s == s_h) acc[s] = run;
        }
      }
    }

    if (OPT == OPT_NONE) {
#pragma unroll
      for (int s = 0; s < G; ++s) {
        const int64_t p = base + s * GROUPS + gj;
        if (p < n && col_ok) {
          store4<float>(a.seg_sum + p * d + gl * 4, acc[s]);
          if (gl == 0) a.seg_rows[p] = shead[s] ? (int32_t)srow[s] : -1;
        }
      }
    } else if (OPT == OPT_ADAM) {
      const float b1 = a.beta1, b2 = a.beta2, eps = a.eps;
#pragma unroll
      for (int s = 0; s < G; ++s) {
        if (shead[s] && col_ok) {
          const int64_t off = (int64_t)srow[s] * a.ld + gl * 4;
          const float4 g = acc[s];
#define RS_ADAM1(c)                                              \
  m[s].c = b1 * m[s].c + (1.f - b1) * g.c;                       \
  v[s].c = b2 * v[s].c + (1.f - b2) * g.c * g.c;                 \
  w[s].c = w[s].c - lr_eff * m[s].c / (sqrtf(v[s].c) + eps);
          RS_ADAM1(x) RS_ADAM1(y) RS_ADAM1(z) RS_ADAM1(w)
#undef RS_ADAM1
          *reinterpret_cast<float4*>(a.w + off) = w[s];
          *reinterpret_cast<float4*>(a.s0 + off) = m[s];
          *reinterpret_cast<float4*>(a.s1 + off) = v[s];
        }
      }
    } else {  // AdaGrad
      float4 w[G], e[G];
      float g2[G];
#pragma unroll
      for (int s = 0; s < G; ++s) {
        g2[s] = 0.f;
        if (shead[s] && col_ok) {
          const int64_t off = (int64_t)srow[s] * d + gl * 4;
          w[s] = *reinterpret_cast<const float4*>(a.w + off);
          if (OPT == OPT_ADAGRAD_ELEM) e[s] = *reinterpret_cast<const float4*>(a.s0 + off);
          else g2[s] = a.s0[srow[s]];
        }
      }
#pragma unroll
      for (int s = 0; s < G; ++s) {
        const float4 g = acc[s];
        if (OPT == OPT_ADAGRAD_ROW) {
          // mean over the row of g*g: reduce over the G lanes of the group in a
          // fixed butterfly order (all lanes of the group take part).
          float sq = (shead[s] && col_ok) ? (g.x * g.x + g.y * g.y + g.z * g.z + g.w * g.w) : 0.f;
#pragma unroll
          for (int o = G / 2; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
          if (shead[s] && col_ok) {
            const int64_t off = (int64_t)srow[s] * d + gl * 4;
            const float acc2 = g2[s] + sq / (float)d;
            const float den = sqrtf(acc2) + a.eps;
            w[s].x -= a.lr * g.x / den; w[s].y -= a.lr * g.y / den;
            w[s].z -= a.lr * g.z / den; w[s].w -= a.lr * g.w / den;
            *reinterpret_cast<float4*>(a.w + off) = w[s];
            if (gl == 0) a.s0[srow[s]] = acc2;
          }
        } else if (shead[s] && col_ok) {
          const int64_t off = (int64_t)srow[s] * d + gl * 4;
#define RS_ADAG1(c)                                   \
  e[s].c += g.c * g.c;                                \
  w[s].c -= a.lr * g.c / (sqrtf(e[s].c) + a.eps);
          RS_ADAG1(x) RS_ADAG1(y) RS_ADAG1(z) RS_ADAG1(w)
#undef RS_ADAG1
          *reinterpret_cast<float4*>(a.w + off) = w[s];
          *reinterpret_cast<float4*>(a.s0 + off) = e[s];
        }
      }
    }
  }
}

template <int OPT>
static int dispatch_segsum(const uint64_t* keys, const void* grad, int grad_dtype, int64_t n,
                           int d, const OptArgs& a, cudaStream_t st) {
  RS_REQUIRE(d > 0 && d % 4 == 0 && d <= 128, "embed_segsum: d=%d must be a multiple of 4, <= 128", d);
  RS_REQUIRE(grad_dtype == RS_F32 || grad_dtype == RS_BF16, "embed_segsum: bad grad dtype");
  if (n == 0) return 0;
  const int threads = 128;
  int64_t blocks = cdiv(n, (threads / 32) * 32);
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  const int g = d / 4;
#define RS_SEG_LAUNCH(G)                                                                          \
  do {                                                                                            \
    if (grad_dtype == RS_F32)                                                                     \
      embed_segsum_kernel<G, OPT, float><<<(unsigned)blocks, threads, 0, st>>>(                   \
          keys, (const float*)grad, n, d, a);                                                     \
    else                                                                                          \
      embed_segsum_kernel<G, OPT, __nv_bfloat16><<<(unsigned)blocks, threads, 0, st>>>(           \
          keys, (const __nv_bfloat16*)grad, n, d, a);                                             \
    return check_launch("embed_segsum");                                                          \
  } while (0)
  if (g <= 1) RS_SEG_LAUNCH(1);
  if (g <= 2) RS_SEG_LAUNCH(2);
  if (g <= 4) RS_SEG_LAUNCH(4);
  if (g <= 8) RS_SEG_LAUNCH(8);
  if (g <= 16) RS_SEG_LAUNCH(16);
  RS_SEG_LAUNCH(32);
#undef RS_SEG_LAUNCH
}

// -------------------------------------------------------- optimizer glue ---
__global__ void adam_advance_kernel(float* s, float b1, float b2) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    const float step = s[0] + 1.f;
    // powers are carried multiplicatively in fp32 like TF's beta_power vars
    const float p1 = (s[0] == 0.f ? 1.f : s[1]) * b1;
    const float p2 = (s[0] == 0.f ? 1.f : s[2]) * b2;
    s[0] = step; s[1] = p1; s[2] = p2;
    s[3] = sqrtf(1.f - p2) / (1.f - p1);
  }
}

__global__ void dense_adam_kernel(float* __restrict__ w, float* __restrict__ m,
                                  float* __restrict__ v, const float* __restrict__ g, int64_t n,
                                  float lr, float b1, float b2, float eps,
                                  const float* __restrict__ scalars,
                                  __nv_bfloat16* __restrict__ shadow) {
  const float lr_eff = lr * __ldg(scalars + 3);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float gi = g[i];
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    const float wi = w[i] - lr_eff * mi / (sqrtf(vi) + eps);
    m[i] = mi; v[i] = vi; w[i] = wi;
    if (shadow) shadow[i] = __float2bfloat16_rn(wi);
  }
}

// --------------------------------------------------------------- routing ---
// Stable bucket-by-owner in three launches: per-block owner histograms, a
// single-block exclusive scan in (owner-major, block-minor) order, and a
// scatter where each block ranks its lookups with warp ballots (stable).
constexpr int ROUTE_BLOCK = 256;
constexpr int ROUTE_MAX_WORLD = 64;

// pad_spread: padding ids (< 0) take a slot at owner hash(i) mod world (Fibonacci hash of the lookup index: padding
// sits at the tail of every sequence, a plain i mod world inherits that pattern) instead of owner 0, so that inputs that are mostly
// padding (sequence / bag columns) keep the buckets balanced (rs_route_ids_padded_spread)
__device__ __forceinline__ void route_of(const int64_t* ids, const int64_t* rows,
                                         const int64_t* local_base, int64_t i, int F, int world,
                                         int& owner, int32_t& lrow, int pad_spread = 0) {
  const int64_t id = ids[i];
  if (id < 0) {  // padding: row -1; owner 0 by convention, or round-robin over the owners
    owner = pad_spread ? (int)((((uint32_t)i * 0x9E3779B1u) >> 16) % (uint32_t)world) : 0; lrow = -1; return;
  }
  const int f = (int)(i % F);
  const uint64_t r = (uint64_t)id % (uint64_t)rows[f];
  owner = (int)(r % (uint64_t)world);
  lrow = (int32_t)(local_base[f] + (int64_t)(r / (uint64_t)world));
}

__global__ void route_hist_kernel(const int64_t* ids, int64_t n, int F, const int64_t* rows,
                                  const int64_t* local_base, int world, int32_t* hist /*[world][nblk]*/,
                                  int pad_spread = 0) {
  __shared__ int cnt[ROUTE_MAX_WORLD];
  if (threadIdx.x < ROUTE_MAX_WORLD) cnt[threadIdx.x] = 0;
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * ROUTE_BLOCK + threadIdx.x;
  if (i < n) {
    int owner; int32_t lrow;
    route_of(ids, rows, local_base, i, F, world, owner, lrow, pad_spread);
    atomicAdd(&cnt[owner], 1);
  }
  __syncthreads();
  if (threadIdx.x < world) hist[(int64_t)threadIdx.x * gridDim.x + blockIdx.x] = cnt[threadIdx.x];
}

__global__ void route_scan_kernel(int32_t* hist, int64_t total, int nblk, int world,
                                  int32_t* send_counts, int32_t* send_offsets) {
  // single block; sequential chunks of blockDim with a running carry.
  __shared__ int32_t buf[1024];
  __shared__ int32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t base = 0; base < total; base += blockDim.x) {
    const int64_t i = base + threadIdx.x;
    const int32_t v = i < total ? hist[i] : 0;
    buf[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < (int)blockDim.x; o <<= 1) {
      int32_t t = threadIdx.x >= (unsigned)o ? buf[threadIdx.x - o] : 0;
      __syncthreads();
      buf[threadIdx.x] += t;
      __syncthreads();
    }
    const int32_t incl = buf[threadIdx.x];
    const int32_t c = carry;
    if (i < total) {
      hist[i] = c + incl - v;  // exclusive
      if (i % nblk == 0) send_offsets[i / nblk] = c + incl - v;
    }
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry = c + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) send_offsets[world] = carry;
  __syncthreads();
  if (threadIdx.x < world) {
    // counts from consecutive offsets (offsets[world] just written by thread 0)
    send_counts[threadIdx.x] = send_offsets[threadIdx.x + 1] - send_offsets[threadIdx.x];
  }
}

__global__ void route_scatter_kernel(const int64_t* ids, int64_t n, int F, const int64_t* rows,
                                     const int64_t* local_base, int world,
                                     const int32_t* hist /*exclusive, [world][nblk]*/,
                                     int32_t* send_rows, int32_t* inverse) {
  __shared__ int warp_cnt[ROUTE_BLOCK / 32][ROUTE_MAX_WORLD];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t i = (int64_t)blockIdx.x * ROUTE_BLOCK + threadIdx.x;
  int owner = -1; int32_t lrow = -1;
  if (i < n) route_of(ids, rows, local_base, i, F, world, owner, lrow);
  // rank within warp among same-owner lanes with lower lane id
  int my_rank = 0;
  for (int o = 0; o < world; ++o) {
    const unsigned m = __ballot_sync(0xffffffffu, owner == o);
    if (owner == o) my_rank = __popc(m & ((1u << lane) - 1u));
    if (lane == 0) warp_cnt[wid][o] = __popc(m);
  }
  __syncthreads();
  if (i < n) {
    int before = 0;
    for (int w = 0; w < wid; ++w) before += warp_cnt[w][owner];
    const int32_t slot = hist[(int64_t)owner * gridDim.x + blockIdx.x] + before + my_rank;
    send_rows[slot] = lrow;
    inverse[i] = slot;
  }
}

// Fixed-capacity variant for CUDA-graph-capturable all-to-alls: bucket o owns slots
// [o*cap, (o+1)*cap); slot = o*cap + (stable rank of the lookup inside bucket o).  Lookups
// beyond the capacity are dropped and raise the overflow flag (the caller must then fail).
__global__ void route_scatter_padded_kernel(const int64_t* ids, int64_t n, int F, const int64_t* rows,
                                            const int64_t* local_base, int world, int cap,
                                            const int32_t* hist /*exclusive, [world][nblk]*/,
                                            const int32_t* send_offsets, int32_t* send_rows,
                                            int32_t* inverse, int32_t* overflow, int pad_spread) {
  __shared__ int warp_cnt[ROUTE_BLOCK / 32][ROUTE_MAX_WORLD];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t i = (int64_t)blockIdx.x * ROUTE_BLOCK + threadIdx.x;
  int owner = -1; int32_t lrow = -1;
  if (i < n) route_of(ids, rows, local_base, i, F, world, owner, lrow, pad_spread);
  int my_rank = 0;
  for (int o = 0; o < world; ++o) {
    const unsigned m = __ballot_sync(0xffffffffu, owner == o);
    if (owner == o) my_rank = __popc(m & ((1u << lane) - 1u));
    if (lane == 0) warp_cnt[wid][o] = __popc(m);
  }
  __syncthreads();
  if (i < n) {
    int before = 0;
    for (int w = 0; w < wid; ++w) before += warp_cnt[w][owner];
    const int k = hist[(int64_t)owner * gridDim.x + blockIdx.x] - send_offsets[owner] + before + my_rank;
    if (k < cap) {
      const int32_t slot = owner * cap + k;
      send_rows[slot] = lrow;
      inverse[i] = slot;
    } else {
      inverse[i] = -1;
      atomicExch(overflow, 1);
    }
  }
}

template <typename T>
__global__ void permute_rows_kernel(const T* __restrict__ src, T* __restrict__ out,
                                    const int32_t* __restrict__ index, int64_t n, int vec_per_row,
                                    int scatter) {
  // rows are moved in 8-byte units (vec_per_row of them)
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t i = t / vec_per_row;
  const int c = (int)(t % vec_per_row);
  if (i >= n) return;
  const int64_t j = index[i];
  const uint2* s = reinterpret_cast<const uint2*>(src);
  uint2* o = reinterpret_cast<uint2*>(out);
  if (scatter) {
    if (j >= 0) o[j * vec_per_row + c] = s[i * vec_per_row + c];
  } else {
    o[i * vec_per_row + c] = j >= 0 ? s[j * vec_per_row + c] : make_uint2(0u, 0u);
  }
}

// Gradient push of the row-sharded path as peer STORES over NVLink: lookup i of this rank sits in slot
// index[i] = owner * cap + k of its send order (rs_route_ids_padded); its gradient row goes straight into the
// owner's receive buffer at slot (my_rank * cap + k) — the permute and the all-to-all of the NCCL path in one
// kernel.  Slots that stay unwritten hold padding rows (row -1 in the owner's keys) and are never read.
struct PeerBufs { void* p[RS_MAX_PEERS]; };

__global__ void scatter_rows_peer_kernel(const uint2* __restrict__ src, PeerBufs dst, const int32_t* __restrict__ index,
                                         int64_t n, int vec_per_row, int cap, int my_rank) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t i = t / vec_per_row;
  const int c = (int)(t % vec_per_row);
  if (i >= n) return;
  const int32_t j = index[i];
  if (j < 0) return;
  const int owner = j / cap, k = j - owner * cap;
  uint2* o = reinterpret_cast<uint2*>(dst.p[owner]);
  o[((int64_t)my_rank * cap + k) * vec_per_row + c] = src[i * vec_per_row + c];
}

// sort keys of the owners' received row indices: (row << 32 | slot); row -1 (padding) sorts last
__global__ void __launch_bounds__(128) keys_from_rows_kernel(const int32_t* __restrict__ rowidx, int64_t n,
                                                             uint64_t* __restrict__ keys) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    keys[i] = ((uint64_t)(uint32_t)rowidx[i] << 32) | (uint64_t)(uint32_t)i;
}

// Cross-rank barrier over peer memory (one process per GPU, all ranks launch it in the same order): rank r
// publishes its next epoch into slot r of every rank's flag array (system-scope release store over NVLink)
// and spins until every slot of its own array has reached that epoch (acquire loads).  ~2 NVLink latencies
// instead of a NCCL all-reduce launch; no host state, so it is a CUDA-graph node.  The epoch lives in device
// memory next to the flags (slot `world`).
struct PeerFlags { unsigned int* p[RS_MAX_PEERS]; };

__global__ void peer_barrier_kernel(PeerFlags flags, int world, int rank) {
  unsigned int* mine = flags.p[rank];
  const unsigned int epoch = mine[RS_MAX_PEERS] + 1u;       // written only by this rank, read back next call
  const int t = threadIdx.x;
  if (t < world) {
    __threadfence_system();                                 // everything this rank wrote before is visible first
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flags.p[t] + rank), "r"(epoch) : "memory");
    unsigned int seen;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(mine + t) : "memory");
    } while ((int)(seen - epoch) < 0);
  }
  __syncthreads();
  if (t == 0) mine[RS_MAX_PEERS] = epoch;
}

}  // namespace rs

using namespace rs;

extern "C" {

int rs_peer_barrier(unsigned int* const* peer_flags, int world, int rank, void* stream) {
  RS_REQUIRE(world >= 1 && world <= RS_MAX_PEERS && rank >= 0 && rank < world, "peer_barrier: world=%d rank=%d", world, rank);
  PeerFlags f;
  for (int r = 0; r < RS_MAX_PEERS; ++r) f.p[r] = r < world ? peer_flags[r] : nullptr;
  peer_barrier_kernel<<<1, 32, 0, as_stream(stream)>>>(f, world, rank);
  return check_launch("peer_barrier");
}

int rs_embed_keys_from_rows(const int32_t* rowidx, int64_t n, uint64_t* sort_keys, void* stream) {
  RS_REQUIRE(n >= 0 && n < ((int64_t)1 << 32) && (n == 0 || (rowidx != nullptr && sort_keys != nullptr)),
             "embed_keys_from_rows: n=%lld", (long long)n);
  if (n == 0) return 0;
  int64_t blocks = cdiv(n, 128 * 4);
  if (blocks > (int64_t)sm_count() * 8) blocks = (int64_t)sm_count() * 8;
  keys_from_rows_kernel<<<(unsigned)blocks, 128, 0, as_stream(stream)>>>(rowidx, n, sort_keys);
  return check_launch("embed_keys_from_rows");
}

int rs_scatter_rows_peer(const void* src, void* const* peer_recv, int world, int my_rank, const int32_t* index,
                         int64_t n, int cap, int row_bytes, void* stream) {
  RS_REQUIRE(world >= 1 && world <= RS_MAX_PEERS && my_rank >= 0 && my_rank < world, "scatter_rows_peer: world=%d rank=%d",
             world, my_rank);
  RS_REQUIRE(row_bytes > 0 && row_bytes % 8 == 0 && cap > 0, "scatter_rows_peer: row_bytes=%d cap=%d", row_bytes, cap);
  if (n == 0) return 0;
  PeerBufs dst;
  for (int r = 0; r < RS_MAX_PEERS; ++r) dst.p[r] = r < world ? peer_recv[r] : nullptr;
  const int vec = row_bytes / 8;
  const int threads = 256;
  const int64_t blocks = cdiv(n * vec, threads);
  scatter_rows_peer_kernel<<<(unsigned)blocks, threads, 0, as_stream(stream)>>>((const uint2*)src, dst, index, n, vec, cap,
                                                                             my_rank);
  return check_launch("scatter_rows_peer");
}

int rs_embed_gather_fwd_ld(const float* table, int64_t table_ld, const int64_t* ids, const int64_t* row_base,
                           const int64_t* rows, int64_t n, int F, int d, void* out, int out_dtype,
                           uint64_t* sort_keys, int32_t* rows_out, void* stream) {
  RS_REQUIRE(F > 0, "embed_gather_fwd: F=%d", F);
  return dispatch_gather<true>(table, table_ld, ids, nullptr, row_base, rows, n, F, d, out, out_dtype,
                               sort_keys, rows_out, nullptr, as_stream(stream));
}
int rs_embed_gather_fwd(const float* table, const int64_t* ids, const int64_t* row_base,
                        const int64_t* rows, int64_t n, int F, int d, void* out, int out_dtype,
                        uint64_t* sort_keys, int32_t* rows_out, void* stream) {
  return rs_embed_gather_fwd_ld(table, d, ids, row_base, rows, n, F, d, out, out_dtype, sort_keys, rows_out, stream);
}

int rs_embed_gather_rows_ld(const float* table, int64_t table_ld, const int32_t* rowidx, int64_t n, int d, void* out,
                            int out_dtype, uint8_t* mask_out, uint64_t* sort_keys, void* stream) {
  return dispatch_gather<false>(table, table_ld, nullptr, rowidx, nullptr, nullptr, n, 1, d, out, out_dtype,
                                sort_keys, nullptr, mask_out, as_stream(stream));
}
int rs_embed_gather_rows(const float* table, const int32_t* rowidx, int64_t n, int d, void* out,
                         int out_dtype, uint8_t* mask_out, uint64_t* sort_keys, void* stream) {
  return rs_embed_gather_rows_ld(table, d, rowidx, n, d, out, out_dtype, mask_out, sort_keys, stream);
}

int rs_embed_gather_peer_fwd(const float* const* peer_tables, int64_t table_ld, int world, const int64_t* ids,
                             const int64_t* local_base, const int64_t* rows, int64_t n, int F, int d, void* out,
                             int out_dtype, void* stream) {
  if (table_ld == 0) table_ld = d;
  RS_REQUIRE(table_ld >= d && table_ld % 4 == 0, "embed_gather_peer: table row stride %lld", (long long)table_ld);
  RS_REQUIRE(world >= 1 && world <= RS_MAX_PEERS, "embed_gather_peer: world=%d (max %d)", world, RS_MAX_PEERS);
  RS_REQUIRE(F > 0 && d > 0 && d % 4 == 0 && d <= 128, "embed_gather_peer: F=%d d=%d", F, d);
  RS_REQUIRE(out_dtype == RS_F32 || out_dtype == RS_BF16, "embed_gather_peer: bad out dtype %d", out_dtype);
  if (n == 0) return 0;
  PeerTables tabs;
  for (int r = 0; r < RS_MAX_PEERS; ++r) tabs.p[r] = r < world ? peer_tables[r] : nullptr;
  const int g = d / 4;
  cudaStream_t st = as_stream(stream);
  if (g <= 1) return launch_gather_peer<1, 4>(tabs, ids, local_base, rows, n, F, d, table_ld, world, out, out_dtype, st);
  if (g <= 2) return launch_gather_peer<2, 4>(tabs, ids, local_base, rows, n, F, d, table_ld, world, out, out_dtype, st);
  // (measured at W = 2: 4 lookups per lane is slower than 2 — fewer, fatter CTAs; the NVLink request rate,
  //  not the loads in flight per lane, bounds the kernel)
  if (g <= 4) return launch_gather_peer<4, 2>(tabs, ids, local_base, rows, n, F, d, table_ld, world, out, out_dtype, st);
  if (g <= 8) return launch_gather_peer<8, 1>(tabs, ids, local_base, rows, n, F, d, table_ld, world, out, out_dtype, st);
  if (g <= 16) return launch_gather_peer<16, 1>(tabs, ids, local_base, rows, n, F, d, table_ld, world, out, out_dtype, st);
  return launch_gather_peer<32, 1>(tabs, ids, local_base, rows, n, F, d, table_ld, world, out, out_dtype, st);
}

int rs_embed_gather_bag_mean(const float* table, const int64_t* ids, const int64_t* offsets,
                             const int64_t* row_base, const int64_t* rows, int64_t n_bags, int F,
                             int d, void* out, int out_dtype, void* stream) {
  RS_REQUIRE(d > 0 && d % 4 == 0 && d <= 128, "embed_gather_bag_mean: d=%d", d);
  if (n_bags == 0) return 0;
  int G = 1;
  while (G * 4 < d) G <<= 1;
  const int threads = 128;
  const int64_t blocks = cdiv(n_bags * G, threads);
  if (out_dtype == RS_F32)
    embed_bag_mean_kernel<float><<<(unsigned)blocks, threads, 0, as_stream(stream)>>>(
        table, ids, offsets, row_base, rows, n_bags, F, d, G, (float*)out);
  else
    embed_bag_mean_kernel<__nv_bfloat16><<<(unsigned)blocks, threads, 0, as_stream(stream)>>>(
        table, ids, offsets, row_base, rows, n_bags, F, d, G, (__nv_bfloat16*)out);
  return check_launch("embed_bag_mean");
}

int rs_embed_bag_fwd_ld(const float* table, int64_t table_ld, const int64_t* ids, const int64_t* offsets,
                        const int64_t* row_base, const int64_t* rows, int64_t n_bags, int F, int d, void* out,
                        int out_dtype, uint64_t* sort_keys, float* inv_cnt, void* stream) {
  if (table_ld == 0) table_ld = d;
  RS_REQUIRE(d > 0 && d % 4 == 0 && d <= 128 && F > 0, "embed_bag_fwd: F=%d d=%d", F, d);
  RS_REQUIRE(table_ld >= d && table_ld % 4 == 0, "embed_bag_fwd: table row stride %lld", (long long)table_ld);
  RS_REQUIRE(out_dtype == RS_F32 || out_dtype == RS_BF16, "embed_bag_fwd: bad out dtype %d", out_dtype);
  if (n_bags == 0) return 0;
  int G = 1;
  while (G * 4 < d) G <<= 1;
  const int threads = 128;
  const int64_t blocks = cdiv(n_bags * G, threads);
  if (out_dtype == RS_F32)
    embed_bag_fwd_kernel<float><<<(unsigned)blocks, threads, 0, as_stream(stream)>>>(
        table, table_ld, ids, offsets, row_base, rows, n_bags, F, d, G, (float*)out, sort_keys, inv_cnt);
  else
    embed_bag_fwd_kernel<__nv_bfloat16><<<(unsigned)blocks, threads, 0, as_stream(stream)>>>(
        table, table_ld, ids, offsets, row_base, rows, n_bags, F, d, G, (__nv_bfloat16*)out, sort_keys, inv_cnt);
  return check_launch("embed_bag_fwd");
}

int rs_embed_bag_grad(const void* dout, int dtype, const int64_t* offsets, const float* inv_cnt, int64_t n_bags, int d,
                      float* g_occ, void* stream) {
  RS_REQUIRE(d > 0 && d % 4 == 0 && d <= 128, "embed_bag_grad: d=%d", d);
  RS_REQUIRE(dtype == RS_F32 || dtype == RS_BF16, "embed_bag_grad: bad dtype %d", dtype);
  if (n_bags == 0) return 0;
  int G = 1;
  while (G * 4 < d) G <<= 1;
  const int threads = 128;
  const int64_t blocks = cdiv(n_bags * G, threads);
  if (dtype == RS_F32)
    embed_bag_grad_kernel<float><<<(unsigned)blocks, threads, 0, as_stream(stream)>>>((const float*)dout, offsets, inv_cnt,
                                                                                      n_bags, d, G, g_occ);
  else
    embed_bag_grad_kernel<__nv_bfloat16><<<(unsigned)blocks, threads, 0, as_stream(stream)>>>(
        (const __nv_bfloat16*)dout, offsets, inv_cnt, n_bags, d, G, g_occ);
  return check_launch("embed_bag_grad");
}

size_t rs_embed_sort_workspace_bytes(int64_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortKeys((void*)nullptr, bytes, (const uint64_t*)nullptr,
                                 (uint64_t*)nullptr, (int)n, 32, 64, (cudaStream_t)0);
  return bytes + 256;
}

int rs_embed_sort_keys(const uint64_t* keys, uint64_t* keys_sorted, int64_t n, int row_bits,
                       void* ws, size_t ws_bytes, void* stream) {
  RS_REQUIRE(row_bits >= 1 && row_bits <= 32, "embed_sort_keys: row_bits=%d", row_bits);
  RS_REQUIRE(n < ((int64_t)1 << 31), "embed_sort_keys: n too large");
  if (n == 0) return 0;
  size_t need = 0;
  cub::DeviceRadixSort::SortKeys((void*)nullptr, need, keys, keys_sorted, (int)n, 32,
                                 32 + row_bits, as_stream(stream));
  if (need > ws_bytes) {
    set_error("embed_sort_keys: workspace %zu < %zu", ws_bytes, need);
    return RS_ERR_WORKSPACE;
  }
  RS_CUDA(cub::DeviceRadixSort::SortKeys(ws, need, keys, keys_sorted, (int)n, 32, 32 + row_bits,
                                         as_stream(stream)));
  g_launches.fetch_add(row_bits > 24 ? 6 : (row_bits > 16 ? 5 : 4), std::memory_order_relaxed);
  return 0;
}

int rs_embed_segsum_adam_ld(float* w, float* m, float* v, int64_t state_ld, const void* grad, int grad_dtype,
                            const uint64_t* keys_sorted, int64_t n, int d, float lr, float beta1,
                            float beta2, float eps, const float* opt_scalars, float grad_scale,
                            void* stream) {
  RS_REQUIRE(opt_scalars != nullptr, "embed_segsum_adam: opt_scalars is NULL");
  if (state_ld == 0) state_ld = d;
  RS_REQUIRE(state_ld >= d && state_ld % 4 == 0, "embed_segsum_adam: state row stride %lld", (long long)state_ld);
  OptArgs a{};
  a.w = w; a.s0 = m; a.s1 = v; a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps;
  a.ld = state_ld;
  a.scalars = opt_scalars; a.grad_scale = grad_scale;
  return dispatch_segsum<OPT_ADAM>(keys_sorted, grad, grad_dtype, n, d, a, as_stream(stream));
}
int rs_embed_segsum_adam(float* w, float* m, float* v, const void* grad, int grad_dtype,
                         const uint64_t* keys_sorted, int64_t n, int d, float lr, float beta1,
                         float beta2, float eps, const float* opt_scalars, float grad_scale,
                         void* stream) {
  return rs_embed_segsum_adam_ld(w, m, v, d, grad, grad_dtype, keys_sorted, n, d, lr, beta1, beta2, eps, opt_scalars,
                                 grad_scale, stream);
}

int rs_embed_segsum_adagrad(float* w, float* g2sum, const void* grad, int grad_dtype,
                            const uint64_t* keys_sorted, int64_t n, int d, float lr, float eps,
                            int per_element, float grad_scale, void* stream) {
  OptArgs a{};
  a.w = w; a.s0 = g2sum; a.lr = lr; a.eps = eps; a.grad_scale = grad_scale;
  if (per_element)
    return dispatch_segsum<OPT_ADAGRAD_ELEM>(keys_sorted, grad, grad_dtype, n, d, a, as_stream(stream));
  return dispatch_segsum<OPT_ADAGRAD_ROW>(keys_sorted, grad, grad_dtype, n, d, a, as_stream(stream));
}

int rs_embed_segsum(const void* grad, int grad_dtype, const uint64_t* keys_sorted, int64_t n,
                    int d, int32_t* seg_rows, float* seg_sum, void* stream) {
  OptArgs a{};
  a.grad_scale = 1.f; a.seg_rows = seg_rows; a.seg_sum = seg_sum;
  return dispatch_segsum<OPT_NONE>(keys_sorted, grad, grad_dtype, n, d, a, as_stream(stream));
}

int rs_adam_advance(float* opt_scalars, float beta1, float beta2, void* stream) {
  adam_advance_kernel<<<1, 32, 0, as_stream(stream)>>>(opt_scalars, beta1, beta2);
  return check_launch("adam_advance");
}

int rs_dense_adam(float* w, float* m, float* v, const float* g, int64_t n, float lr, float beta1,
                  float beta2, float eps, const float* opt_scalars, void* w_bf16_shadow,
                  void* stream) {
  RS_REQUIRE(opt_scalars != nullptr, "dense_adam: opt_scalars is NULL");
  if (n == 0) return 0;
  const int threads = 256;
  int64_t blocks = cdiv(n, threads);
  if (blocks > (int64_t)sm_count() * 8) blocks = (int64_t)sm_count() * 8;
  dense_adam_kernel<<<(unsigned)blocks, threads, 0, as_stream(stream)>>>(
      w, m, v, g, n, lr, beta1, beta2, eps, opt_scalars, (__nv_bfloat16*)w_bf16_shadow);
  return check_launch("dense_adam");
}

size_t rs_route_workspace_bytes(int64_t n, int world) {
  return (size_t)(cdiv(n, ROUTE_BLOCK) * world + 8) * sizeof(int32_t);
}

int rs_route_ids(const int64_t* ids, int64_t n, int F, const int64_t* rows,
                 const int64_t* local_base, int world, int32_t* send_rows, int32_t* inverse,
                 int32_t* send_counts, int32_t* send_offsets, void* ws, size_t ws_bytes,
                 void* stream) {
  RS_REQUIRE(world >= 1 && world <= ROUTE_MAX_WORLD, "route_ids: world=%d", world);
  RS_REQUIRE(F > 0 && n >= 0 && n < ((int64_t)1 << 31), "route_ids: n/F out of range");
  if (ws_bytes < rs_route_workspace_bytes(n, world)) {
    set_error("route_ids: workspace too small");
    return RS_ERR_WORKSPACE;
  }
  cudaStream_t st = as_stream(stream);
  int32_t* hist = (int32_t*)ws;
  const int nblk = (int)cdiv(n > 0 ? n : 1, ROUTE_BLOCK);
  route_hist_kernel<<<nblk, ROUTE_BLOCK, 0, st>>>(ids, n, F, rows, local_base, world, hist);
  if (int e = check_launch("route_hist")) return e;
  route_scan_kernel<<<1, 1024, 0, st>>>(hist, (int64_t)nblk * world, nblk, world, send_counts,
                                        send_offsets);
  if (int e = check_launch("route_scan")) return e;
  route_scatter_kernel<<<nblk, ROUTE_BLOCK, 0, st>>>(ids, n, F, rows, local_base, world, hist,
                                                     send_rows, inverse);
  return check_launch("route_scatter");
}

static int route_ids_padded_impl(const int64_t* ids, int64_t n, int F, const int64_t* rows,
                                 const int64_t* local_base, int world, int capacity, int32_t* send_rows,
                                 int32_t* inverse, int32_t* send_counts, int32_t* overflow, void* ws,
                                 size_t ws_bytes, void* stream, int pad_spread) {
  RS_REQUIRE(world >= 1 && world <= ROUTE_MAX_WORLD, "route_ids_padded: world=%d", world);
  RS_REQUIRE(F > 0 && n >= 0 && n < ((int64_t)1 << 31) && capacity > 0, "route_ids_padded: n/F/capacity out of range");
  RS_REQUIRE((int64_t)world * capacity < ((int64_t)1 << 31), "route_ids_padded: world*capacity too large");
  const size_t need = rs_route_workspace_bytes(n, world) + (size_t)(world + 1) * sizeof(int32_t);
  if (ws_bytes < need) { set_error("route_ids_padded: workspace %zu < %zu", ws_bytes, need); return RS_ERR_WORKSPACE; }
  cudaStream_t st = as_stream(stream);
  int32_t* hist = (int32_t*)ws;
  int32_t* offsets = (int32_t*)((char*)ws + rs_route_workspace_bytes(n, world));
  const int nblk = (int)cdiv(n > 0 ? n : 1, ROUTE_BLOCK);
  RS_CUDA(cudaMemsetAsync(send_rows, 0xFF, (size_t)world * capacity * sizeof(int32_t), st));   // row -1 = padding
  route_hist_kernel<<<nblk, ROUTE_BLOCK, 0, st>>>(ids, n, F, rows, local_base, world, hist, pad_spread);
  if (int e = check_launch("route_hist")) return e;
  route_scan_kernel<<<1, 1024, 0, st>>>(hist, (int64_t)nblk * world, nblk, world, send_counts, offsets);
  if (int e = check_launch("route_scan")) return e;
  route_scatter_padded_kernel<<<nblk, ROUTE_BLOCK, 0, st>>>(ids, n, F, rows, local_base, world, capacity, hist,
                                                            offsets, send_rows, inverse, overflow, pad_spread);
  return check_launch("route_scatter_padded");
}

int rs_route_ids_padded(const int64_t* ids, int64_t n, int F, const int64_t* rows,
                        const int64_t* local_base, int world, int capacity, int32_t* send_rows,
                        int32_t* inverse, int32_t* send_counts, int32_t* overflow, void* ws,
                        size_t ws_bytes, void* stream) {
  return route_ids_padded_impl(ids, n, F, rows, local_base, world, capacity, send_rows, inverse, send_counts, overflow, ws,
                               ws_bytes, stream, 0);
}
int rs_route_ids_padded_spread(const int64_t* ids, int64_t n, int F, const int64_t* rows,
                               const int64_t* local_base, int world, int capacity, int32_t* send_rows,
                               int32_t* inverse, int32_t* send_counts, int32_t* overflow, void* ws,
                               size_t ws_bytes, void* stream) {
  return route_ids_padded_impl(ids, n, F, rows, local_base, world, capacity, send_rows, inverse, send_counts, overflow, ws,
                               ws_bytes, stream, 1);
}

int rs_permute_rows(const void* src, void* out, const int32_t* index, int64_t n, int d, int dtype,
                    int scatter, void* stream) {
  const int64_t row_bytes = (int64_t)d * (dtype == RS_F32 ? 4 : 2);
  RS_REQUIRE(row_bytes % 8 == 0, "permute_rows: row bytes %lld not a multiple of 8", (long long)row_bytes);
  if (n == 0) return 0;
  const int vec = (int)(row_bytes / 8);
  const int threads = 256;
  const int64_t blocks = cdiv(n * vec, threads);
  permute_rows_kernel<float><<<(unsigned)blocks, threads, 0, as_stream(stream)>>>(
      (const float*)src, (float*)out, index, n, vec, scatter);
  return check_launch("permute_rows");
}

}  // extern "C"
