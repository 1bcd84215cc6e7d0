// head.cu — fused logits head of the AutoInt tower (k = 1):
//   p_raw = sigmoid(Z w + b)                      final MultiLayerDense(1, sigmoid)   autoint:49-50
//   p     = clip(p_raw, 1e-6, 1)                  autoint:52
//   loss  = mean_b( -y log(p+1e-6) - (a-y) log(1-p+1e-6) )   rank/ctr/base_model.py:7-12
//   dZ = dz w^T, dw = Z^T dz, db = sum dz   with dz = dloss/d(pre-activation)
// One pass over Z (read) and dZ (write): a warp owns a row, a lane owns the same
// columns of every row, so w and the dw accumulators live in registers and the only
// cross-lane traffic is the 5-step shuffle of the row dot product.  Partials are
// reduced over warps and CTAs in a fixed order (deterministic, no atomics).
#include "common.cuh"

namespace rs {

constexpr int HEAD_WARPS = 8;

// FROM_P: the forward and dZ were computed elsewhere (tower.cu): p is read from p_out (the stored bf16 activation,
// the value every derivative below starts from) and only the partials of dw / db / loss are produced.
template <int NV, typename T, bool FROM_P = false>
__global__ void __launch_bounds__(HEAD_WARPS * 32)
logit_head_kernel(const T* __restrict__ Z, int64_t ldz, const float* __restrict__ w,
                  const float* __restrict__ bias, const float* __restrict__ y, float a,
                  T* __restrict__ p_out, T* __restrict__ dZ, int64_t lddz, float* __restrict__ part,
                  int B, int zw, int relu_cols) {
  extern __shared__ float head_smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float wv[NV][4], dw[NV][4];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      wv[i][u] = (!FROM_P && c + u < zw) ? w[c + u] : 0.f;
      dw[i][u] = 0.f;
    }
  }
  const float b0 = FROM_P ? 0.f : bias[0];
  const float invB = 1.f / (float)B;
  float db = 0.f, loss = 0.f;
  // rows are software-pipelined: the next row's loads are in flight while the current row is reduced
  const int64_t rstep = (int64_t)gridDim.x * HEAD_WARPS;
  int64_t r = (int64_t)blockIdx.x * HEAD_WARPS + wid;
  float zn[NV][4];
  auto load_row = [&](int64_t rr, float (&zz)[NV][4]) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (i * 32 + lane) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c < zw && rr < B) v = load4<T>(Z + rr * ldz + c);
      zz[i][0] = v.x; zz[i][1] = v.y; zz[i][2] = v.z; zz[i][3] = v.w;
    }
  };
  load_row(r, zn);
  for (; r < B; r += rstep) {
    float z[NV][4];
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        z[i][u] = zn[i][u];
        if (!FROM_P) dot = fmaf(z[i][u], wv[i][u], dot);
      }
    }
    load_row(r + rstep, zn);
    float pr, prs;
    if constexpr (FROM_P) {
      pr = prs = to_f<T>(p_out[r]);
    } else {
      dot = warp_sum(dot);
      pr = 1.f / (1.f + expf(-(dot + b0)));
      prs = to_f<T>(from_f<T>(pr));                  // the stored activation (bf16-rounded in bf16 mode)
    }
    const float p = fminf(fmaxf(prs, 1e-6f), 1.0f);
    const float yy = y[r];
    loss += -yy * logf(p + 1e-6f) - (a - yy) * logf(1.0f - p + 1e-6f);
    const float dp = (-yy / (p + 1e-6f) + (a - yy) / (1.0f - p + 1e-6f)) * invB;
    const float dz = (prs >= 1e-6f && prs <= 1.0f) ? dp * prs * (1.f - prs) : 0.f;
    db += dz;
    if (!FROM_P && lane == 0) p_out[r] = from_f<T>(pr);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (i * 32 + lane) * 4;
#pragma unroll
      for (int u = 0; u < 4; ++u) dw[i][u] = fmaf(dz, z[i][u], dw[i][u]);
      if (!FROM_P && c < zw) {
        float o[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          o[u] = dz * wv[i][u];
          // columns [0, relu_cols) of Z are the output of a Dense(relu): their gradient is handed on already
          // masked by relu' (saves the separate activation-backward pass over dZ[:, :relu_cols])
          if (c + u < relu_cols && !(z[i][u] > 0.f)) o[u] = 0.f;
        }
        store4<T>(dZ + r * lddz + c, make_float4(o[0], o[1], o[2], o[3]));
      }
    }
  }
  // warp partials -> smem [HEAD_WARPS][zw + 2] -> CTA partial (fixed warp order)
  const int np = zw + 2;
  float* mine = head_smem + wid * np;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (c + u < zw) mine[c + u] = dw[i][u];
  }
  if (lane == 0) { mine[zw] = db; mine[zw + 1] = loss; }
  __syncthreads();
  float* dst = part + (int64_t)blockIdx.x * np;
  for (int i = threadIdx.x; i < np; i += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < HEAD_WARPS; ++k) s += head_smem[k * np + i];
    dst[i] = s;
  }
}

__global__ void logit_head_reduce_kernel(const float* __restrict__ part, int nparts, int zw,
                                         float* __restrict__ dw, float* __restrict__ db,
                                         float* __restrict__ loss, float invB) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // one warp per output
  const int np = zw + 2;
  if (i >= np) return;
  const float s = warp_ordered_sum(part + i, nparts, np);
  if ((threadIdx.x & 31) != 0) return;
  if (i < zw) dw[i] = s;
  else if (i == zw) db[0] = s;
  else loss[0] = s * invB;
}

static int head_grid(int B) {
  int64_t g = cdiv(B, HEAD_WARPS * 4);
  const int64_t cap = (int64_t)sm_count() * 2;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace rs

using namespace rs;

extern "C" {

int rs_logit_head_reduce(const void* ws, size_t ws_bytes, float* dw, float* db, float* loss_out, int B, int zw,
                         void* stream);

size_t rs_logit_head_workspace_bytes(int B, int zw) {
  return (size_t)head_grid(B > 0 ? B : 1) * (size_t)(zw + 2) * sizeof(float);
}

int rs_logit_head_fwd_bwd_relu(const void* Z, int64_t ldz, int dtype, const float* w, const float* bias,
                               const float* y, float a, void* p_out, float* loss_out, void* dZ,
                               int64_t lddz, float* dw, float* db, int B, int zw, int relu_cols, void* ws,
                               size_t ws_bytes, void* stream) {
  RS_REQUIRE(relu_cols >= 0 && relu_cols <= zw, "logit_head: relu_cols=%d", relu_cols);
  RS_REQUIRE(B > 0 && zw > 0 && zw % 4 == 0 && zw <= 2048, "logit_head: B=%d zw=%d (zw %% 4 == 0, <= 2048)", B, zw);
  RS_REQUIRE(ldz % 4 == 0 && lddz % 4 == 0, "logit_head: leading dims must be multiples of 4");
  RS_REQUIRE(dtype == RS_F32 || dtype == RS_BF16, "logit_head: bad dtype");
  if (ws_bytes < rs_logit_head_workspace_bytes(B, zw)) { set_error("logit_head: workspace too small"); return RS_ERR_WORKSPACE; }
  cudaStream_t st = as_stream(stream);
  const int grid = head_grid(B);
  const size_t smem = (size_t)HEAD_WARPS * (zw + 2) * sizeof(float);
  const int nv = (int)cdiv(zw, 128);
#define RS_HEAD_GO(NV, TT)                                                                          \
  do {                                                                                              \
    auto kern = logit_head_kernel<NV, TT>;                                                          \
    RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));    \
    kern<<<grid, HEAD_WARPS * 32, smem, st>>>((const TT*)Z, ldz, w, bias, y, a, (TT*)p_out, (TT*)dZ, \
                                              lddz, (float*)ws, B, zw, relu_cols);                  \
  } while (0)
  if (dtype == RS_F32) {
    if (nv <= 4) RS_HEAD_GO(4, float); else if (nv <= 6) RS_HEAD_GO(6, float); else if (nv <= 8) RS_HEAD_GO(8, float);
    else RS_HEAD_GO(16, float);
  } else {
    if (nv <= 4) RS_HEAD_GO(4, __nv_bfloat16); else if (nv <= 6) RS_HEAD_GO(6, __nv_bfloat16);
    else if (nv <= 8) RS_HEAD_GO(8, __nv_bfloat16); else RS_HEAD_GO(16, __nv_bfloat16);
  }
#undef RS_HEAD_GO
  if (int e = check_launch("logit_head")) return e;
  // dw == NULL: the per-CTA partials stay in `ws` and the caller sums them with rs_logit_head_reduce — on another
  // stream if it wishes (only the dense optimizer reads dw / db / loss; dZ, which the tower's backward waits for, is
  // complete here)
  if (dw == nullptr) return 0;
  return rs_logit_head_reduce(ws, ws_bytes, dw, db, loss_out, B, zw, stream);
}

int rs_logit_head_grad(const void* Z, int64_t ldz, int dtype, const void* p, const float* y, float a, int B, int zw,
                       void* ws, size_t ws_bytes, void* stream) {
  RS_REQUIRE(B > 0 && zw > 0 && zw % 4 == 0 && zw <= 2048, "logit_head_grad: B=%d zw=%d (zw %% 4 == 0, <= 2048)", B, zw);
  RS_REQUIRE(ldz % 4 == 0, "logit_head_grad: leading dim must be a multiple of 4");
  RS_REQUIRE(dtype == RS_F32 || dtype == RS_BF16, "logit_head_grad: bad dtype");
  if (ws_bytes < rs_logit_head_workspace_bytes(B, zw)) { set_error("logit_head_grad: workspace too small"); return RS_ERR_WORKSPACE; }
  cudaStream_t st = as_stream(stream);
  const int grid = head_grid(B);
  const size_t smem = (size_t)HEAD_WARPS * (zw + 2) * sizeof(float);
  const int nv = (int)cdiv(zw, 128);
#define RS_HEADG_GO(NV, TT)                                                                                \
  do {                                                                                                     \
    auto kern = logit_head_kernel<NV, TT, true>;                                                           \
    RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));           \
    kern<<<grid, HEAD_WARPS * 32, smem, st>>>((const TT*)Z, ldz, nullptr, nullptr, y, a, (TT*)p, nullptr, 0, \
                                              (float*)ws, B, zw, 0);                                       \
  } while (0)
  if (dtype == RS_F32) {
    if (nv <= 4) RS_HEADG_GO(4, float); else if (nv <= 6) RS_HEADG_GO(6, float); else if (nv <= 8) RS_HEADG_GO(8, float);
    else RS_HEADG_GO(16, float);
  } else {
    if (nv <= 4) RS_HEADG_GO(4, __nv_bfloat16); else if (nv <= 6) RS_HEADG_GO(6, __nv_bfloat16);
    else if (nv <= 8) RS_HEADG_GO(8, __nv_bfloat16); else RS_HEADG_GO(16, __nv_bfloat16);
  }
#undef RS_HEADG_GO
  return check_launch("logit_head_grad");
}

int rs_logit_head_reduce(const void* ws, size_t ws_bytes, float* dw, float* db, float* loss_out, int B, int zw,
                         void* stream) {
  RS_REQUIRE(B > 0 && zw > 0 && dw != nullptr && db != nullptr && loss_out != nullptr, "logit_head_reduce: B=%d zw=%d", B, zw);
  if (ws_bytes < rs_logit_head_workspace_bytes(B, zw)) { set_error("logit_head_reduce: workspace too small"); return RS_ERR_WORKSPACE; }
  logit_head_reduce_kernel<<<(unsigned)cdiv((zw + 2) * 32, 256), 256, 0, as_stream(stream)>>>(
      (const float*)ws, head_grid(B), zw, dw, db, loss_out, 1.f / (float)B);
  return check_launch("logit_head_reduce");
}

int rs_logit_head_fwd_bwd(const void* Z, int64_t ldz, int dtype, const float* w, const float* bias,
                          const float* y, float a, void* p_out, float* loss_out, void* dZ,
                          int64_t lddz, float* dw, float* db, int B, int zw, void* ws,
                          size_t ws_bytes, void* stream) {
  return rs_logit_head_fwd_bwd_relu(Z, ldz, dtype, w, bias, y, a, p_out, loss_out, dZ, lddz, dw, db, B, zw, 0, ws, ws_bytes,
                                    stream);
}

}  // extern "C"
