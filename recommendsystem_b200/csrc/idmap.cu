// idmap.cu — collision-free id -> arena-row map (the hash mode of EmbeddingFeatures / AutoIntTrainer).
//
// Each field f owns S_f = next_pow2(2 * R_f) open-addressing slots of 16 bytes {int64 key; int32 row; int32 pad}
// inside one slot array (key -1 = empty; row -1 = the key has no row: the field was full).  The slot of an id is
// mix64(id) & (S_f - 1), probed linearly.  Two passes per batch, separated by a kernel boundary:
//   insert  every lookup probes; the thread whose CAS puts a new key into an empty slot takes the field's next row
//           (atomicAdd on the row counter), records it in the slot and in key_of_row, and writes the row's whole
//           optimizer record (w from the counter-based init rule, moments / g2sum at their initial values);
//   lookup  every lookup probes again (read-only) and emits its arena row, or -1 (padding, unseen, overflowed).
// No thread waits for another: a probe loop ends after at most S_f slots, and a key found before its row is
// written is simply left alone (the lookup pass, after the kernel boundary, reads the row).
// Eviction (rs_idmap_evict) decays every live row's show count, drops the keys whose count falls below a threshold,
// compacts each field's live rows back to the front of its range and rebuilds the slots from key_of_row.
#include <cmath>

#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace rs {

struct __align__(16) IdSlot {
  long long key;
  int row;
  int pad;
};

// splitmix64 finaliser (as the attention-dropout hash in interacting_kernels.cuh)
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
constexpr uint64_t kGolden = 0x9E3779B97F4A7C15ULL;

// per-field geometry, int64[n_fields][4]
struct FieldGeom { long long row_base, cap, slot_base, slot_mask; };
__device__ __forceinline__ FieldGeom field_geom(const int64_t* geom, int f) {
  const longlong2* g = reinterpret_cast<const longlong2*>(geom + 4 * (int64_t)f);
  const longlong2 a = __ldg(g), b = __ldg(g + 1);
  return {a.x, a.y, b.x, b.y};
}

struct InitArgs {
  float* w; int64_t w_ld; int d; float scale; uint64_t seed;
  float* s[2]; int64_t s_ld[2]; int s_width[2]; float s_init[2];
};

// w[k] = scale * N(0,1), a pure function of (seed, field, id, k): pair p = k / 2 draws r = mix64(base + golden * (p+1))
// with base = mix64(mix64(seed + golden * (f+1)) ^ id); u1 = ((r >> 40) + 1) / 2^24 in (0, 1], u2 = ((r & 2^32-1) >> 8)
// / 2^24 in [0, 1); Box-Muller: w[2p] = scale * (sqrt(-2 ln u1) * cos(2 pi u2)), w[2p+1] the same with sin.
__device__ __forceinline__ void init_record(const InitArgs& a, int64_t row, int f, long long id) {
  float* w = a.w + row * a.w_ld;
  const uint64_t base = mix64(mix64(a.seed + kGolden * (uint64_t)(f + 1)) ^ (uint64_t)id);
  for (int p = 0; 2 * p < a.d; ++p) {
    const uint64_t r = mix64(base + kGolden * (uint64_t)(p + 1));
    const float u1 = (float)((uint32_t)(r >> 40) + 1u) * 5.9604644775390625e-8f;    // 2^-24
    const float u2 = (float)((uint32_t)r >> 8) * 5.9604644775390625e-8f;
    const float rad = sqrtf(-2.f * logf(u1));
    float sn, cs;
    sincospif(2.f * u2, &sn, &cs);
    w[2 * p] = a.scale * (rad * cs);
    if (2 * p + 1 < a.d) w[2 * p + 1] = a.scale * (rad * sn);
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    if (!a.s[j]) continue;
    float* s = a.s[j] + row * a.s_ld[j];
    for (int k = 0; k < a.s_width[j]; ++k) s[k] = a.s_init[j];
  }
}

__global__ void __launch_bounds__(256)
idmap_insert_kernel(IdSlot* __restrict__ slots, long long* __restrict__ key_of_row,
                    unsigned long long* __restrict__ count, const int64_t* __restrict__ geom,
                    const int64_t* __restrict__ ids, int64_t n, int F, const int32_t* __restrict__ field_of_col,
                    InitArgs ia) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const long long id = ids[i];
    if (id < 0) continue;
    const int f = __ldg(field_of_col + (int)(i % F));
    const FieldGeom g = field_geom(geom, f);
    const uint64_t h = mix64((uint64_t)id);
    for (long long t = 0; t <= g.slot_mask; ++t) {
      IdSlot* s = slots + g.slot_base + (long long)((h + (uint64_t)t) & (uint64_t)g.slot_mask);
      const long long key = __ldcg(&s->key);
      if (key == id) break;                                   // present (its row may still be being written)
      if (key != -1) continue;                                // another key: next slot
      if ((long long)__ldcg(count + f) >= g.cap) break;        // field full: claim no slot (lookup: overflow)
      const long long prev = (long long)atomicCAS(reinterpret_cast<unsigned long long*>(&s->key),
                                                  0xFFFFFFFFFFFFFFFFULL, (unsigned long long)id);
      if (prev == -1) {                                       // this thread inserted the key
        const unsigned long long r = atomicAdd(count + f, 1ULL);
        if ((long long)r < g.cap) {
          const int64_t row = g.row_base + (int64_t)r;
          key_of_row[row] = id;
          s->row = (int)row;
          init_record(ia, row, f, id);
        }                                                     // else: the slot keeps row -1 (overflowed key)
        break;
      }
      if (prev == id) break;                                  // inserted by another thread meanwhile
    }
  }
}

__global__ void __launch_bounds__(256)
idmap_lookup_kernel(const IdSlot* __restrict__ slots, long long* __restrict__ counters, const int64_t* __restrict__ geom,
                    int n_fields, const int64_t* __restrict__ ids, int64_t n, int F,
                    const int32_t* __restrict__ field_of_col, int64_t* __restrict__ rows_out, int after_insert) {
  if (after_insert && blockIdx.x == 0) {
    // the insert pass may have pushed a full field's counter past its capacity: clamp (no insert runs now)
    for (int f = threadIdx.x; f < n_fields; f += blockDim.x) {
      const long long cap = geom[4 * (int64_t)f + 1];
      if (counters[f] > cap) counters[f] = cap;
    }
  }
  unsigned long long* overflow = reinterpret_cast<unsigned long long*>(counters + n_fields);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const long long id = ids[i];
    int64_t row = -1;
    if (id >= 0) {
      const int f = __ldg(field_of_col + (int)(i % F));
      const FieldGeom g = field_geom(geom, f);
      const uint64_t h = mix64((uint64_t)id);
      bool found = false;
      for (long long t = 0; t <= g.slot_mask; ++t) {
        const longlong2 s = __ldg(reinterpret_cast<const longlong2*>(
            slots + g.slot_base + (long long)((h + (uint64_t)t) & (uint64_t)g.slot_mask)));
        if (s.x == id) { row = (int)(s.y & 0xFFFFFFFFLL); found = true; break; }
        if (s.x == -1) break;
      }
      if (after_insert && (!found || row < 0)) atomicAdd(overflow + f, 1ULL);
      if (!found) row = -1;
    }
    rows_out[i] = row;
  }
}

__global__ void __launch_bounds__(256)
idmap_rebuild_kernel(IdSlot* __restrict__ slots, long long* __restrict__ key_of_row,
                     const long long* __restrict__ counters, const int64_t* __restrict__ geom) {
  const int f = blockIdx.y;
  const FieldGeom g = field_geom(geom, f);
  const long long used = min(counters[f], g.cap);
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < g.cap; j += (long long)gridDim.x * blockDim.x) {
    const int64_t row = g.row_base + j;
    if (j >= used) { key_of_row[row] = -1; continue; }
    const long long id = key_of_row[row];
    if (id < 0) continue;
    const uint64_t h = mix64((uint64_t)id);
    for (long long t = 0; t <= g.slot_mask; ++t) {
      IdSlot* s = slots + g.slot_base + (long long)((h + (uint64_t)t) & (uint64_t)g.slot_mask);
      const long long prev = (long long)atomicCAS(reinterpret_cast<unsigned long long*>(&s->key),
                                                  0xFFFFFFFFFFFFFFFFULL, (unsigned long long)id);
      if (prev == -1) { s->row = (int)row; break; }
      if (prev == id) break;
    }
  }
}

// show[row] += 1 per training lookup that resolved to a row.  Every increment adds the same value, so the sum does not
// depend on the order of the atomics (it stops growing at 2^24, where x + 1 rounds back to x).
__global__ void __launch_bounds__(256)
idmap_count_kernel(float* __restrict__ show, const int64_t* __restrict__ rows, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = rows[i];
    if (r >= 0) atomicAdd(show + r, 1.f);
  }
}

// ---- eviction: decay + mark, exclusive scan of the keep flags (pos), hole list, moves, counters, rebuild.
// Field f (blockIdx.y) has used_f live rows [0, used_f) before and live_f = kept rows after; the k-th dropped row
// below live_f (a hole) receives the k-th kept row at or above live_f (a mover), both in ascending order.  Holes lie
// below live_f and movers at or above it, so no record is read after it is written.
__global__ void __launch_bounds__(256)
idmap_evict_mark_kernel(float* __restrict__ show, const long long* __restrict__ counters,
                        const int64_t* __restrict__ geom, float threshold, float decay, int* __restrict__ keep,
                        int64_t total_rows) {
  const int f = blockIdx.y;
  const FieldGeom g = field_geom(geom, f);
  const long long used = min(counters[f], g.cap);
  if (f == 0 && blockIdx.x == 0 && threadIdx.x == 0) keep[total_rows] = 0;    // pos[total_rows] = rows kept in all
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < g.cap; j += (long long)gridDim.x * blockDim.x) {
    const int64_t row = g.row_base + j;
    int k = 0;
    if (j < used) {
      const float s = __fmul_rn(show[row], decay);
      show[row] = s;
      k = !(s < threshold);
    }
    keep[row] = k;
  }
}

__global__ void __launch_bounds__(256)
idmap_evict_holes_kernel(const int* __restrict__ pos, const int64_t* __restrict__ geom, int* __restrict__ hole_row) {
  const int f = blockIdx.y;
  const FieldGeom g = field_geom(geom, f);
  const int k0 = pos[g.row_base];
  const long long live = pos[g.row_base + g.cap] - k0;
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < live; j += (long long)gridDim.x * blockDim.x) {
    const int64_t row = g.row_base + j;
    if (pos[row + 1] == pos[row])                                   // dropped: hole number j - (kept rows below j)
      hole_row[g.row_base + (j - (pos[row] - k0))] = (int)j;
  }
}

struct MoveArgs {
  float* w; int64_t w_ld; int d;
  float* s[2]; int64_t s_ld[2]; int s_width[2];
};

__global__ void __launch_bounds__(256)
idmap_evict_move_kernel(const int* __restrict__ pos, const int* __restrict__ hole_row,
                        const long long* __restrict__ counters, const int64_t* __restrict__ geom,
                        long long* __restrict__ key_of_row, float* __restrict__ show, MoveArgs a) {
  const int f = blockIdx.y;
  const FieldGeom g = field_geom(geom, f);
  const long long used = min(counters[f], g.cap);
  const int k0 = pos[g.row_base];
  const long long live = pos[g.row_base + g.cap] - k0;
  const long long kept_below = pos[g.row_base + live] - k0;       // kept rows that stay where they are
  for (long long j = live + (long long)blockIdx.x * blockDim.x + threadIdx.x; j < used;
       j += (long long)gridDim.x * blockDim.x) {
    const int64_t src = g.row_base + j;
    if (pos[src + 1] != pos[src]) {                                 // kept: mover number (kept rows in [live, j))
      const int64_t dst = g.row_base + hole_row[g.row_base + (pos[src] - k0 - kept_below)];
      const float* ws = a.w + src * a.w_ld;
      float* wd = a.w + dst * a.w_ld;
      for (int k = 0; k < a.d; ++k) wd[k] = ws[k];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        if (!a.s[q]) continue;
        const float* ss = a.s[q] + src * a.s_ld[q];
        float* sd = a.s[q] + dst * a.s_ld[q];
        for (int k = 0; k < a.s_width[q]; ++k) sd[k] = ss[k];
      }
      show[dst] = show[src];
      key_of_row[dst] = key_of_row[src];
    }
    show[src] = 0.f;                                                // vacated: owned by no key
    key_of_row[src] = -1;
  }
}

__global__ void idmap_evict_counters_kernel(const int* __restrict__ pos, long long* __restrict__ counters,
                                            const int64_t* __restrict__ geom, int n_fields,
                                            long long* __restrict__ evicted) {
  for (int f = threadIdx.x; f < n_fields; f += blockDim.x) {
    const FieldGeom g = field_geom(geom, f);
    const long long used = min(counters[f], g.cap);
    const long long live = pos[g.row_base + g.cap] - pos[g.row_base];
    evicted[f] += used - live;
    counters[f] = live;
  }
}

static unsigned grid_for(int64_t n, int threads) {
  int64_t blocks = cdiv(n, threads);
  const int64_t cap = (int64_t)sm_count() * 32;
  if (blocks > cap) blocks = cap;
  return (unsigned)(blocks < 1 ? 1 : blocks);
}

}  // namespace rs

using namespace rs;

extern "C" {

int rs_idmap_insert(void* slots, int64_t* key_of_row, int64_t* counters, const int64_t* geom, int n_fields,
                    const int64_t* ids, int64_t n, int F, const int32_t* field_of_col, uint64_t seed, float scale,
                    float* w, int64_t w_ld, int d, float* s0, int64_t s0_ld, int s0_width, float s0_init,
                    float* s1, int64_t s1_ld, int s1_width, float s1_init, void* stream) {
  RS_REQUIRE(n_fields > 0 && F > 0 && n >= 0, "idmap_insert: n_fields=%d F=%d n=%lld", n_fields, F, (long long)n);
  RS_REQUIRE(w && d > 0 && w_ld >= d, "idmap_insert: w / d=%d / w_ld=%lld", d, (long long)w_ld);
  RS_REQUIRE((!s0 || (s0_width > 0 && s0_ld >= s0_width)) && (!s1 || (s1_width > 0 && s1_ld >= s1_width)),
             "idmap_insert: optimizer state width / stride");
  RS_REQUIRE(((uintptr_t)slots & 15) == 0 && ((uintptr_t)geom & 15) == 0, "idmap_insert: slots / geom not 16-B aligned");
  if (n == 0) return 0;
  InitArgs ia{};
  ia.w = w; ia.w_ld = w_ld; ia.d = d; ia.scale = scale; ia.seed = seed;
  ia.s[0] = s0; ia.s_ld[0] = s0_ld; ia.s_width[0] = s0_width; ia.s_init[0] = s0_init;
  ia.s[1] = s1; ia.s_ld[1] = s1_ld; ia.s_width[1] = s1_width; ia.s_init[1] = s1_init;
  const int threads = 256;
  idmap_insert_kernel<<<grid_for(n, threads), threads, 0, as_stream(stream)>>>(
      (IdSlot*)slots, (long long*)key_of_row, (unsigned long long*)counters, geom, ids, n, F, field_of_col, ia);
  return check_launch("idmap_insert");
}

int rs_idmap_lookup(const void* slots, int64_t* counters, const int64_t* geom, int n_fields, const int64_t* ids,
                    int64_t n, int F, const int32_t* field_of_col, int64_t* rows_out, int after_insert, void* stream) {
  RS_REQUIRE(n_fields > 0 && F > 0 && n >= 0, "idmap_lookup: n_fields=%d F=%d n=%lld", n_fields, F, (long long)n);
  RS_REQUIRE(((uintptr_t)slots & 15) == 0 && ((uintptr_t)geom & 15) == 0, "idmap_lookup: slots / geom not 16-B aligned");
  if (n == 0) return 0;
  const int threads = 256;
  idmap_lookup_kernel<<<grid_for(n, threads), threads, 0, as_stream(stream)>>>(
      (const IdSlot*)slots, (long long*)counters, geom, n_fields, ids, n, F, field_of_col, rows_out, after_insert);
  return check_launch("idmap_lookup");
}

int rs_idmap_rebuild(void* slots, int64_t n_slots, int64_t* key_of_row, const int64_t* counters, const int64_t* geom,
                     int n_fields, int64_t max_rows, void* stream) {
  RS_REQUIRE(n_fields > 0 && n_fields <= 65535 && n_slots > 0 && max_rows > 0,
             "idmap_rebuild: n_fields=%d n_slots=%lld max_rows=%lld", n_fields, (long long)n_slots, (long long)max_rows);
  RS_REQUIRE(((uintptr_t)slots & 15) == 0 && ((uintptr_t)geom & 15) == 0, "idmap_rebuild: slots / geom not 16-B aligned");
  RS_CUDA(cudaMemsetAsync(slots, 0xFF, (size_t)n_slots * sizeof(IdSlot), as_stream(stream)));
  const int threads = 256;
  int64_t bx = cdiv(max_rows, threads);
  if (bx > 4096) bx = 4096;
  idmap_rebuild_kernel<<<dim3((unsigned)bx, (unsigned)n_fields), threads, 0, as_stream(stream)>>>(
      (IdSlot*)slots, (long long*)key_of_row, (const long long*)counters, geom);
  return check_launch("idmap_rebuild");
}

int rs_idmap_count(float* show, const int64_t* rows, int64_t n, void* stream) {
  RS_REQUIRE(n >= 0 && (show || n == 0), "idmap_count: n=%lld", (long long)n);
  if (n == 0) return 0;
  const int threads = 256;
  idmap_count_kernel<<<grid_for(n, threads), threads, 0, as_stream(stream)>>>(show, rows, n);
  return check_launch("idmap_count");
}

static size_t evict_flags_bytes(int64_t total_rows) { return (size_t)cdiv((total_rows + 1) * 4, 256) * 256; }

size_t rs_idmap_evict_workspace_bytes(int64_t total_rows) {
  if (total_rows <= 0 || total_rows >= INT32_MAX) return 0;
  size_t scan = 0;
  cub::DeviceScan::ExclusiveSum((void*)nullptr, scan, (const int*)nullptr, (int*)nullptr, (int)(total_rows + 1),
                                (cudaStream_t)0);
  return 2 * evict_flags_bytes(total_rows) + scan + 256;
}

int rs_idmap_evict(void* slots, int64_t n_slots, int64_t* key_of_row, int64_t* counters, const int64_t* geom,
                   int n_fields, int64_t total_rows, float* show, float threshold, float decay, float* w, int64_t w_ld,
                   int d, float* s0, int64_t s0_ld, int s0_width, float* s1, int64_t s1_ld, int s1_width,
                   int64_t* evicted, void* ws, size_t ws_bytes, void* stream) {
  RS_REQUIRE(n_fields > 0 && n_fields <= 65535 && n_slots > 0 && total_rows > 0 && total_rows < INT32_MAX,
             "idmap_evict: n_fields=%d n_slots=%lld total_rows=%lld", n_fields, (long long)n_slots,
             (long long)total_rows);
  RS_REQUIRE(decay > 0.f && decay <= 1.f && std::isfinite(threshold), "idmap_evict: decay=%g threshold=%g",
             (double)decay, (double)threshold);
  RS_REQUIRE(show && evicted && w && d > 0 && w_ld >= d, "idmap_evict: show / evicted / w / d=%d", d);
  RS_REQUIRE((!s0 || (s0_width > 0 && s0_ld >= s0_width)) && (!s1 || (s1_width > 0 && s1_ld >= s1_width)),
             "idmap_evict: optimizer state width / stride");
  RS_REQUIRE(((uintptr_t)slots & 15) == 0 && ((uintptr_t)geom & 15) == 0 && ((uintptr_t)ws & 255) == 0,
             "idmap_evict: slots / geom not 16-B aligned or workspace not 256-B aligned");
  const size_t need = rs_idmap_evict_workspace_bytes(total_rows);
  if (ws_bytes < need) {
    set_error("idmap_evict: workspace %zu < %zu", ws_bytes, need);
    return RS_ERR_WORKSPACE;
  }
  cudaStream_t st = as_stream(stream);
  int* keep = (int*)ws;                                            // keep flags, then the hole list
  int* pos = (int*)((char*)ws + evict_flags_bytes(total_rows));     // exclusive scan of the flags
  void* scan_ws = (char*)ws + 2 * evict_flags_bytes(total_rows);
  size_t scan_bytes = need - 2 * evict_flags_bytes(total_rows);
  const int threads = 256;
  int64_t bx = cdiv(total_rows, threads);
  if (bx > 4096) bx = 4096;
  const dim3 grid((unsigned)bx, (unsigned)n_fields);
  idmap_evict_mark_kernel<<<grid, threads, 0, st>>>(show, (const long long*)counters, geom, threshold, decay, keep,
                                                    total_rows);
  if (int rc = check_launch("idmap_evict_mark")) return rc;
  RS_CUDA(cub::DeviceScan::ExclusiveSum(scan_ws, scan_bytes, (const int*)keep, pos, (int)(total_rows + 1), st));
  g_launches.fetch_add(2, std::memory_order_relaxed);
  idmap_evict_holes_kernel<<<grid, threads, 0, st>>>(pos, geom, keep);
  if (int rc = check_launch("idmap_evict_holes")) return rc;
  MoveArgs ma{};
  ma.w = w; ma.w_ld = w_ld; ma.d = d;
  ma.s[0] = s0; ma.s_ld[0] = s0_ld; ma.s_width[0] = s0_width;
  ma.s[1] = s1; ma.s_ld[1] = s1_ld; ma.s_width[1] = s1_width;
  idmap_evict_move_kernel<<<grid, threads, 0, st>>>(pos, keep, (const long long*)counters, geom,
                                                    (long long*)key_of_row, show, ma);
  if (int rc = check_launch("idmap_evict_move")) return rc;
  idmap_evict_counters_kernel<<<1, 256, 0, st>>>(pos, (long long*)counters, geom, n_fields, (long long*)evicted);
  if (int rc = check_launch("idmap_evict_counters")) return rc;
  // (the rebuild kernel grid-strides over a field's rows, so total_rows serves as its max_rows)
  return rs_idmap_rebuild(slots, n_slots, key_of_row, counters, geom, n_fields, total_rows, stream);
}

}  // extern "C"
