// interacting_args.cuh — argument packs shared by the K4 dispatcher and the
// per-shape instantiations.
#pragma once
#include "common.cuh"
namespace rs {
// fused embedding lookup of the tensor-core forward (rs_interacting_fwd_gather)
struct IGatherArgs {
  const float* const* tables; int64_t table_ld; int world; const int64_t* ids; const int64_t* local_base;
  const int64_t* rows; uint64_t* sort_keys;
  // bags (rs_interacting_fwd_gather_bag): ids [B, bag_slots], field f owns slots [bag_off[f], bag_off[f+1])
  const int64_t* bag_off = nullptr; float* inv_cnt = nullptr; int bag_slots = 0;
};
// fused gradient push of the tensor-core backward (rs_interacting_bwd_scatter)
struct IScatterArgs {
  void* const* peer_recv; int world; int rank; const int32_t* inverse; int cap;
};
struct IFwdArgs {
  const void* x; int64_t x_ld, x_bs; const float* W; const float* b; const float* gm; const float* bt;
  float eps; void* y; int64_t y_ld, y_bs; void* saved; int B, F, L, use_res, dtype; cudaStream_t st;
  float drop_rate = 0.f; unsigned long long drop_seed = 0; const unsigned long long* drop_step = nullptr;
  const IGatherArgs* gather = nullptr;
};
struct IBwdArgs {
  const void* x; int64_t x_ld, x_bs; const void* saved; const float* W; const float* b; const float* gm;
  const float* bt; float eps; const void* dy; int64_t dy_ld, dy_bs; void* dx; int64_t dx_ld, dx_bs;
  float* dparams; int B, F, L, use_res, dtype; void* ws; size_t ws_bytes; cudaStream_t st;
  float drop_rate = 0.f; unsigned long long drop_seed = 0; const unsigned long long* drop_step = nullptr;
  const void* dx_add = nullptr;            // optional [B,F,D] rows added to dx (same strides as dx)
  const IScatterArgs* scatter = nullptr;   // dx rows go to the owners' receive buffers instead of dx
};
}  // namespace rs
