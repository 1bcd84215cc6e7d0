// interacting.cu — C-ABI entry points of K4 (InteractingLayer.py:37-61); the
// kernels live in interacting_kernels.cuh and are instantiated per (D, U, H)
// shape in interacting_inst.cu.
#include "interacting_args.cuh"

namespace rs {
// Shapes built (keep in sync with build.py INTERACT_SHAPES).
#define RS_INTERACT_SHAPES(X) X(16, 16, 1) X(16, 16, 2) X(16, 16, 4) X(8, 8, 1) X(8, 8, 2) X(16, 8, 2)
#define RS_DECL(DD, UU, HH)                                   \
  int interacting_fwd_##DD##_##UU##_##HH(const IFwdArgs& a); \
  int interacting_bwd_##DD##_##UU##_##HH(const IBwdArgs& a);
RS_INTERACT_SHAPES(RS_DECL)
#undef RS_DECL
// tensor-core (tcgen05) path, interacting_tc.cu
bool interacting_tc_supported(int F, int D, int U, int H, int dtype);
int interacting_tc_fwd(const IFwdArgs& a);
int interacting_tc_bwd(const IBwdArgs& a);
int interacting_tc_bwd_reduce(const void* ws, size_t ws_bytes, float* dparams, int B, int F, cudaStream_t st);
}  // namespace rs

using namespace rs;

extern "C" {

size_t rs_interacting_workspace_bytes(int B, int F, int D, int U) {
  (void)B; (void)F;
  return 16 + (size_t)(sm_count() * 2) * (size_t)(D * 4 * U + 6 * U) * sizeof(float);   // 16-byte header (tensor-core bwd)
}

size_t rs_interacting_saved_bytes(int B, int F, int U, int L) {
  // [L, B*F, U] activations, then [L, B*F, 4] per-head softmax statistics of the tensor-core kernels
  return (size_t)L * (size_t)B * (size_t)F * (size_t)(U + 4) * sizeof(float);
}

int rs_interacting_path(int F, int D, int U, int H, int dtype, int compute_bf16, float dropout_rate) {
  if (compute_bf16 && dropout_rate == 0.f && interacting_tc_supported(F, D, U, H, dtype)) return RS_PATH_TCGEN05;
#define RS_CASE(DD, UU, HH) \
  if (D == DD && U == UU && H == HH) return RS_PATH_FFMA;
  RS_INTERACT_SHAPES(RS_CASE)
#undef RS_CASE
  return RS_PATH_NONE;
}

int rs_interacting_fwd_dropout(const void* x, int64_t x_ld, int64_t x_bs, int dtype, const float* Wqkvr,
                               const float* bqkvr, const float* ln_gamma, const float* ln_beta,
                               float ln_eps, void* y, int64_t y_ld, int64_t y_bs, void* saved, int B, int F, int D, int U,
                               int H, int L, int use_res, int compute_bf16, float dropout_rate,
                               unsigned long long dropout_seed, const unsigned long long* dropout_step, void* stream) {
  RS_REQUIRE(dropout_rate >= 0.f && dropout_rate < 1.f, "interacting_fwd: dropout_rate %g not in [0, 1)", dropout_rate);
  RS_REQUIRE(B > 0 && F > 0 && L >= 1, "interacting_fwd: B=%d F=%d L=%d", B, F, L);
  RS_REQUIRE(H > 0 && U % H == 0, "interacting_fwd: head_num %d must divide unit_num %d", H, U);
  RS_REQUIRE(L == 1 || D == U, "interacting_fwd: layer_num>1 needs input dim %d == unit_num %d", D, U);
  RS_REQUIRE(F <= 256, "interacting_fwd: F=%d > 256 fields not supported", F);
  RS_REQUIRE(dtype == RS_F32 || dtype == RS_BF16, "interacting_fwd: bad dtype");
  RS_REQUIRE(x_ld % 4 == 0 && y_ld % 4 == 0, "interacting_fwd: leading dims must be multiples of 4");
  if (x_bs == 0) x_bs = (int64_t)F * x_ld;
  if (y_bs == 0) y_bs = (int64_t)F * y_ld;
  RS_REQUIRE(x_bs % 4 == 0 && y_bs % 4 == 0, "interacting_fwd: batch strides must be multiples of 4");
  IFwdArgs a{x, x_ld, x_bs, Wqkvr, bqkvr, ln_gamma, ln_beta, ln_eps, y, y_ld, y_bs, saved, B, F, L, use_res,
             dtype, as_stream(stream)};
  a.drop_rate = dropout_rate;
  a.drop_seed = dropout_seed;
  a.drop_step = dropout_step;
  // attention dropout is built into the FFMA kernels only: the tensor-core path is taken without it
  if (rs_interacting_path(F, D, U, H, dtype, compute_bf16, dropout_rate) == RS_PATH_TCGEN05) return interacting_tc_fwd(a);
#define RS_CASE(DD, UU, HH) \
  if (D == DD && U == UU && H == HH) return interacting_fwd_##DD##_##UU##_##HH(a);
  RS_INTERACT_SHAPES(RS_CASE)
#undef RS_CASE
  set_error("interacting_fwd: (D=%d, U=%d, H=%d) not built", D, U, H);
  return RS_ERR_UNSUPPORTED;
}

int rs_interacting_fwd_gather(const float* const* peer_tables, int64_t table_ld, int world, const int64_t* ids,
                              const int64_t* local_base, const int64_t* rows, void* x_out, int64_t x_ld, int64_t x_bs,
                              unsigned long long* sort_keys, int dtype, const float* Wqkvr, const float* bqkvr,
                              const float* ln_gamma, const float* ln_beta, float ln_eps, void* y, int64_t y_ld,
                              int64_t y_bs, void* saved, int B, int F, int D, int U, int H, int L, int use_res,
                              void* stream) {
  RS_REQUIRE(rs_interacting_path(F, D, U, H, dtype, 1, 0.f) == RS_PATH_TCGEN05,
             "interacting_fwd_gather: only the tensor-core path fuses the lookup (F=%d D=%d U=%d H=%d dtype=%d)", F, D, U, H,
             dtype);
  RS_REQUIRE(B > 0 && L >= 1 && world >= 1 && world <= RS_MAX_PEERS, "interacting_fwd_gather: B=%d L=%d world=%d", B, L, world);
  RS_REQUIRE(table_ld >= D && table_ld % 16 == 0, "interacting_fwd_gather: table row stride %lld (64-byte aligned rows)",
             (long long)table_ld);
  RS_REQUIRE(x_ld % 4 == 0 && y_ld % 4 == 0, "interacting_fwd_gather: leading dims must be multiples of 4");
  if (x_bs == 0) x_bs = (int64_t)F * x_ld;
  if (y_bs == 0) y_bs = (int64_t)F * y_ld;
  RS_REQUIRE(x_bs % 4 == 0 && y_bs % 4 == 0, "interacting_fwd_gather: batch strides must be multiples of 4");
  IFwdArgs a{x_out, x_ld, x_bs, Wqkvr, bqkvr, ln_gamma, ln_beta, ln_eps, y, y_ld, y_bs, saved, B, F, L, use_res,
             dtype, as_stream(stream)};
  IGatherArgs g{peer_tables, table_ld, world, ids, local_base, rows, (uint64_t*)sort_keys};
  a.gather = &g;
  return interacting_tc_fwd(a);
}

int rs_interacting_fwd_gather_bag(const float* table, int64_t table_ld, const int64_t* ids, const int64_t* slot_off,
                                  const int64_t* row_base, const int64_t* rows, void* x_out, int64_t x_ld, int64_t x_bs,
                                  unsigned long long* sort_keys, float* inv_cnt, int dtype, const float* Wqkvr,
                                  const float* bqkvr, const float* ln_gamma, const float* ln_beta, float ln_eps, void* y,
                                  int64_t y_ld, int64_t y_bs, void* saved, int B, int F, int S, int D, int U, int H, int L,
                                  int use_res, void* stream) {
  RS_REQUIRE(rs_interacting_path(F, D, U, H, dtype, 1, 0.f) == RS_PATH_TCGEN05,
             "interacting_fwd_gather_bag: only the tensor-core path fuses the lookup (F=%d D=%d U=%d H=%d dtype=%d)", F, D,
             U, H, dtype);
  RS_REQUIRE(B > 0 && L >= 1 && S >= F, "interacting_fwd_gather_bag: B=%d L=%d S=%d F=%d", B, L, S, F);
  RS_REQUIRE((int64_t)B * S < ((int64_t)1 << 31), "interacting_fwd_gather_bag: B*S = %lld slots (32-bit key positions)",
             (long long)B * S);
  RS_REQUIRE(table != nullptr && slot_off != nullptr && inv_cnt != nullptr,
             "interacting_fwd_gather_bag: table, slot offsets and inv_cnt are required");
  RS_REQUIRE(table_ld >= D && table_ld % 16 == 0, "interacting_fwd_gather_bag: table row stride %lld (64-byte aligned rows)",
             (long long)table_ld);
  RS_REQUIRE(x_ld % 4 == 0 && y_ld % 4 == 0, "interacting_fwd_gather_bag: leading dims must be multiples of 4");
  if (x_bs == 0) x_bs = (int64_t)F * x_ld;
  if (y_bs == 0) y_bs = (int64_t)F * y_ld;
  RS_REQUIRE(x_bs % 4 == 0 && y_bs % 4 == 0, "interacting_fwd_gather_bag: batch strides must be multiples of 4");
  IFwdArgs a{x_out, x_ld, x_bs, Wqkvr, bqkvr, ln_gamma, ln_beta, ln_eps, y, y_ld, y_bs, saved, B, F, L, use_res,
             dtype, as_stream(stream)};
  IGatherArgs g{&table, table_ld, 1, ids, row_base, rows, (uint64_t*)sort_keys, slot_off, inv_cnt, S};
  a.gather = &g;
  return interacting_tc_fwd(a);
}

int rs_interacting_bwd_scatter(const void* x, int64_t x_ld, int64_t x_bs, const void* saved, int dtype,
                               const float* Wqkvr, const float* bqkvr, const float* ln_gamma, const float* ln_beta,
                               float ln_eps, const void* dy, int64_t dy_ld, int64_t dy_bs, void* dx, int64_t dx_ld,
                               int64_t dx_bs, const void* dx_add, void* const* peer_recv, int world, int rank,
                               const int* inverse, int cap, float* dparams, int B, int F, int D, int U, int H, int L,
                               int use_res, void* ws, size_t ws_bytes, void* stream) {
  RS_REQUIRE(rs_interacting_path(F, D, U, H, dtype, 1, 0.f) == RS_PATH_TCGEN05,
             "interacting_bwd_scatter: only the tensor-core path fuses the gradient push (F=%d D=%d U=%d H=%d)", F, D, U, H);
  RS_REQUIRE(B > 0 && L >= 1 && saved != nullptr, "interacting_bwd_scatter: B=%d L=%d saved=%p", B, L, saved);
  RS_REQUIRE(x_ld % 4 == 0 && dy_ld % 4 == 0 && dx_ld % 4 == 0, "interacting_bwd_scatter: leading dims must be multiples of 4");
  if (x_bs == 0) x_bs = (int64_t)F * x_ld;
  if (dy_bs == 0) dy_bs = (int64_t)F * dy_ld;
  if (dx_bs == 0) dx_bs = (int64_t)F * dx_ld;
  IBwdArgs a{x, x_ld, x_bs, saved, Wqkvr, bqkvr, ln_gamma, ln_beta, ln_eps, dy, dy_ld, dy_bs, dx, dx_ld, dx_bs, dparams,
             B, F, L, use_res, dtype, ws, ws_bytes, as_stream(stream)};
  a.dx_add = dx_add;
  IScatterArgs s{peer_recv, world, rank, (const int32_t*)inverse, cap};
  if (inverse != nullptr) {
    RS_REQUIRE(world >= 1 && world <= RS_MAX_PEERS && rank >= 0 && rank < world && cap > 0 && peer_recv != nullptr,
               "interacting_bwd_scatter: world=%d rank=%d cap=%d", world, rank, cap);
    a.scatter = &s;
  }
  return interacting_tc_bwd(a);
}

int rs_interacting_bwd_reduce(const void* ws, size_t ws_bytes, float* dparams, int B, int F, int D, int U, int H,
                              void* stream) {
  RS_REQUIRE(rs_interacting_path(F, D, U, H, RS_BF16, 1, 0.f) == RS_PATH_TCGEN05,
             "interacting_bwd_reduce: only the tensor-core backward defers its reduction (F=%d D=%d U=%d H=%d)", F, D, U, H);
  RS_REQUIRE(B > 0 && ws != nullptr && dparams != nullptr, "interacting_bwd_reduce: B=%d ws=%p dparams=%p", B, ws, (void*)dparams);
  return interacting_tc_bwd_reduce(ws, ws_bytes, dparams, B, F, as_stream(stream));
}

int rs_interacting_fwd(const void* x, int64_t x_ld, int64_t x_bs, int dtype, const float* Wqkvr,
                       const float* bqkvr, const float* ln_gamma, const float* ln_beta,
                       float ln_eps, void* y, int64_t y_ld, int64_t y_bs, void* saved, int B, int F, int D, int U,
                       int H, int L, int use_res, int compute_bf16, void* stream) {
  return rs_interacting_fwd_dropout(x, x_ld, x_bs, dtype, Wqkvr, bqkvr, ln_gamma, ln_beta, ln_eps, y, y_ld, y_bs, saved,
                                    B, F, D, U, H, L, use_res, compute_bf16, 0.f, 0ULL, nullptr, stream);
}

int rs_interacting_bwd_dropout(const void* x, int64_t x_ld, int64_t x_bs, const void* saved, int dtype,
                               const float* Wqkvr, const float* bqkvr, const float* ln_gamma,
                               const float* ln_beta, float ln_eps, const void* dy, int64_t dy_ld,
                               int64_t dy_bs, void* dx, int64_t dx_ld, int64_t dx_bs, float* dparams, int B, int F, int D,
                               int U, int H, int L, int use_res, int compute_bf16, float dropout_rate,
                               unsigned long long dropout_seed, const unsigned long long* dropout_step, void* ws,
                               size_t ws_bytes, void* stream) {
  RS_REQUIRE(dropout_rate >= 0.f && dropout_rate < 1.f, "interacting_bwd: dropout_rate %g not in [0, 1)", dropout_rate);
  RS_REQUIRE(B > 0 && F > 0 && L >= 1, "interacting_bwd: B=%d F=%d L=%d", B, F, L);
  RS_REQUIRE(H > 0 && U % H == 0, "interacting_bwd: head_num %d must divide unit_num %d", H, U);
  RS_REQUIRE(L == 1 || D == U, "interacting_bwd: layer_num>1 needs input dim == unit_num");
  RS_REQUIRE(L == 1 || saved != nullptr, "interacting_bwd: saved activations required for L>1");
  RS_REQUIRE(F <= 256, "interacting_bwd: F=%d > 256 fields not supported", F);
  RS_REQUIRE(dtype == RS_F32 || dtype == RS_BF16, "interacting_bwd: bad dtype");
  RS_REQUIRE(x_ld % 4 == 0 && dy_ld % 4 == 0 && dx_ld % 4 == 0,
             "interacting_bwd: leading dims must be multiples of 4");
  if (x_bs == 0) x_bs = (int64_t)F * x_ld;
  if (dy_bs == 0) dy_bs = (int64_t)F * dy_ld;
  if (dx_bs == 0) dx_bs = (int64_t)F * dx_ld;
  RS_REQUIRE(x_bs % 4 == 0 && dy_bs % 4 == 0 && dx_bs % 4 == 0, "interacting_bwd: batch strides must be multiples of 4");
  IBwdArgs a{x, x_ld, x_bs, saved, Wqkvr, bqkvr, ln_gamma, ln_beta, ln_eps, dy, dy_ld, dy_bs, dx, dx_ld, dx_bs, dparams,
             B, F, L, use_res, dtype, ws, ws_bytes, as_stream(stream)};
  a.drop_rate = dropout_rate;
  a.drop_seed = dropout_seed;
  a.drop_step = dropout_step;
  if (rs_interacting_path(F, D, U, H, dtype, compute_bf16, dropout_rate) == RS_PATH_TCGEN05) return interacting_tc_bwd(a);
#define RS_CASE(DD, UU, HH) \
  if (D == DD && U == UU && H == HH) return interacting_bwd_##DD##_##UU##_##HH(a);
  RS_INTERACT_SHAPES(RS_CASE)
#undef RS_CASE
  set_error("interacting_bwd: (D=%d, U=%d, H=%d) not built", D, U, H);
  return RS_ERR_UNSUPPORTED;
}

int rs_interacting_bwd(const void* x, int64_t x_ld, int64_t x_bs, const void* saved, int dtype,
                       const float* Wqkvr, const float* bqkvr, const float* ln_gamma,
                       const float* ln_beta, float ln_eps, const void* dy, int64_t dy_ld,
                       int64_t dy_bs, void* dx, int64_t dx_ld, int64_t dx_bs, float* dparams, int B, int F, int D, int U, int H, int L,
                       int use_res, int compute_bf16, void* ws, size_t ws_bytes, void* stream) {
  return rs_interacting_bwd_dropout(x, x_ld, x_bs, saved, dtype, Wqkvr, bqkvr, ln_gamma, ln_beta, ln_eps, dy, dy_ld, dy_bs,
                                    dx, dx_ld, dx_bs, dparams, B, F, D, U, H, L, use_res, compute_bf16, 0.f, 0ULL, nullptr, ws,
                                    ws_bytes, stream);
}

}  // extern "C"
