// sm100_ew.h -- launchers for the HBM-bound kernels of the backend (elementwise, normalisation, pooling, softmax,
// loss, optimizer, layout / datatype transforms).  Device pointers, element counts; every function only enqueues.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace sm100 {

// ---- fill / n-ary sum / axpby / relu --------------------------------------------------------------------------
int ew_set_f32(cudaStream_t s, float* p, size_t n, float v);
int ew_set_u16(cudaStream_t s, uint16_t* p, size_t n, uint16_t v);
int ew_set_u64(cudaStream_t s, uint64_t* p, size_t n, uint64_t v);
int ew_sum_i32(cudaStream_t s, const int* const* inputs, int k, int* out, size_t n); // k <= 64
int ew_sum_f32(cudaStream_t s, const float* const* inputs, int k, float* out, size_t n); // out = sum_k inputs[k] (out may alias any input)
// c = p * a + q * b (b may be NULL: c = p * a); all contiguous and same shape
int ew_axpby_f32(cudaStream_t s, float p, const float* a, float q, const float* b, float* c, size_t n);
// c[i] = p * a[ia(i)] + q * b[ib(i)] over a <= 4-d index space with per-operand strides (0 = broadcast); b may be NULL
int ew_axpby_bcast_f32(cudaStream_t s, float p, const float* a, const int* astride, float q, const float* b, const int* bstride, float* c, const int* cstride, const int* dim);
// c = p * a * b, same broadcasting form
int ew_mul_bcast_f32(cudaStream_t s, float p, const float* a, const int* astride, const float* b, const int* bstride, float* c, const int* cstride, const int* dim);
int ew_relu_fwd_f32(cudaStream_t s, const float* a, float* b, size_t n);
int ew_relu_bwd_f32(cudaStream_t s, const float* g, const float* b, float* h, size_t n); // h = b > 0 ? g : 0
// the same on bf16 (kind 1) / fp16 (kind 2) tensors
int ew_relu_fwd_16(cudaStream_t s, int kind, const void* a, void* b, size_t n);
int ew_relu_bwd_16(cudaStream_t s, int kind, const void* g, const void* b, void* h, size_t n);
int ew_sum_16(cudaStream_t s, int kind, const void* const* inputs, int k, void* out, size_t n); // k <= 8
// out[c] (+)= sum over rows of g[row * ld + c]  (bias gradients of GEMM / convolution)
// workspace (colsum_workspace_bytes(cols), may be NULL): per-block partial rows, combined in a fixed order instead of by atomics
size_t colsum_workspace_bytes(int cols);
int colsum_f32(cudaStream_t s, const float* g, size_t rows, int cols, long long ld, float* out, int accumulate, void* workspace);
// g of element kind g_kind (0 = fp32, 1 = bf16, 2 = fp16), out of kind out_kind; fp32 accumulation
int colsum_any(cudaStream_t s, int g_kind, const void* g, size_t rows, int cols, long long ld, void* out, int out_kind, int accumulate, void* workspace);
// reduce a <= 4-d tensor over the axes where rdim == 1 (sum); out has rdim shape, contiguous
int reduce_sum_bcast_f32(cudaStream_t s, const float* a, const int* adim, const int* astride, float* out, const int* rdim, float scale, int accumulate);

// ---- pooling (NHWC, window clipped at the border exactly like CPU_REF) ---------------------------------------
struct PoolGeom {
	int N, H, W, C, P, Q;
	int R, S, stride_h, stride_w, pad_h, pad_w;
	long long an, ah, aw; // input strides (elements), channel stride 1
	long long bn, bh, bw; // output strides
};
int pool_max_fwd_f32(cudaStream_t s, const PoolGeom& g, const float* a, float* b);
int pool_max_bwd_f32(cudaStream_t s, const PoolGeom& g, const float* grad_b, const float* a, const float* b, float* grad_a);
int pool_avg_fwd_f32(cudaStream_t s, const PoolGeom& g, const float* a, float* b);
int pool_avg_bwd_f32(cudaStream_t s, const PoolGeom& g, const float* grad_b, float* grad_a);
int pool_max_fwd_16(cudaStream_t s, int kind, const PoolGeom& g, const void* a, void* b);
int pool_max_bwd_16(cudaStream_t s, int kind, const PoolGeom& g, const void* grad_b, const void* a, const void* b, void* grad_a);
int pool_avg_fwd_16(cudaStream_t s, int kind, const PoolGeom& g, const void* a, void* b);
int pool_avg_bwd_16(cudaStream_t s, int kind, const PoolGeom& g, const void* grad_b, void* grad_a);

// ---- batch norm over [outer, C, inner] (NHWC: inner = 1; NCHW: outer = N, inner = H * W) ----------------------
// training forward: writes y, saved_mean, saved_inv_std and updates the running mean / var in place
// fuse_relu: y = relu(bn(x)) in the same pass (BATCH_NORM_FORWARD followed by an in-place RELU_FORWARD)
// ext_part / ext_rows: per-channel statistics slots (four planes [ext_rows][C]: count, shift, shifted sum, shifted sum of squares) produced by the convolution that wrote x
// (conv_stats_request); the statistics pass over x is then skipped
// coef_out: statistics only -- y is not written; the per-channel a, b of y = x * a + b go to coef_out[0, C) and [C, 2C)
int bn_fwd_train_f32(cudaStream_t s, const float* x, float* y, const float* scale, const float* bias, float* running_mean, float* running_var, float* saved_mean, float* saved_inv_std, size_t outer, int C, size_t inner, float epsilon, float momentum, void* workspace, int fuse_relu, const float* ext_part = 0, int ext_rows = 0, float* coef_out = 0);
size_t bn_workspace_bytes(int C);
int bn_fwd_test_f32(cudaStream_t s, const float* x, float* y, const float* scale, const float* bias, const float* mean, const float* var, size_t outer, int C, size_t inner, float epsilon, void* workspace);
// backward: dx, dscale, dbias from g, x, scale, saved_mean, saved_inv_std.  bias != NULL = fused with the RELU_BACKWARD
// in front of it: g is masked by bn(x) > 0 on the fly (the mask is recomputed from x, bit-identical to the forward)
// dx_colsum != NULL: also writes sum over rows of dx per channel (NHWC only; = the bias gradient of the convolution in front)
// ext_part / ext_rows: the partial rows of the reduction over (g, x), already made by bn_add_relu_bwd_reduce_* (NHWC vector path only)
int bn_bwd_f32(cudaStream_t s, const float* g, const float* x, const float* scale, const float* bias, const float* saved_mean, const float* saved_inv_std, float* dx, float* dscale, float* dbias, size_t outer, int C, size_t inner, void* workspace, float* dx_colsum = 0, const float* ext_part = 0, int ext_rows = 0);
// the same on 16-bit activations (kind 1 = bf16, 2 = fp16): scale / bias / running and saved statistics / dscale / dbias stay fp32
// (lib/nnc/ccv_cnnp_model_addons.c:954-956); dx_colsum is written in element kind colsum_kind (0 = fp32)
int bn_fwd_train_16(cudaStream_t s, int kind, const void* x, void* y, const float* scale, const float* bias, float* running_mean, float* running_var, float* saved_mean, float* saved_inv_std, size_t outer, int C, size_t inner, float epsilon, float momentum, void* workspace, int fuse_relu, const float* ext_part = 0, int ext_rows = 0, float* coef_out = 0);
int bn_fwd_test_16(cudaStream_t s, int kind, const void* x, void* y, const float* scale, const float* bias, const float* mean, const float* var, size_t outer, int C, size_t inner, float epsilon, void* workspace);
int bn_bwd_16(cudaStream_t s, int kind, const void* g, const void* x, const float* scale, const float* bias, const float* saved_mean, const float* saved_inv_std, void* dx, float* dscale, float* dbias, size_t outer, int C, size_t inner, void* workspace, void* dx_colsum = 0, int colsum_kind = 0, const float* ext_part = 0, int ext_rows = 0);
int ew_add_relu_fwd_16(cudaStream_t s, int kind, const void* a, const void* b, void* out, size_t n);
int ew_add_relu_bwd_16(cudaStream_t s, int kind, const void* a, const void* b, const void* y, void* out, size_t n);
// out = relu(a + b); out = y > 0 ? a + b : 0  (residual block end, forward / backward)
int ew_add_relu_fwd_f32(cudaStream_t s, const float* a, const float* b, float* out, size_t n);
int ew_add_relu_bwd_f32(cudaStream_t s, const float* a, const float* b, const float* y, float* out, size_t n);
// residual block end with the batch norm of the main branch folded in (NHWC, C = innermost dimension):
// forward  out = relu(roundT(x * coef[c] + coef[C + c]) + r), coef from bn_fwd_train_*(..., coef_out);
// backward g = y > 0 ? a + b : 0 (b may be NULL) plus the partial rows of the batch-norm backward reduction over (g, x) in part
//          (*part_rows of them, 0 when the layout takes the plain path), for bn_bwd_*(..., ext_part, ext_rows)
int bn_add_relu_fwd_f32(cudaStream_t s, const float* x, const float* r, float* out, const float* coef, size_t outer, int C);
int bn_add_relu_fwd_16(cudaStream_t s, int kind, const void* x, const void* r, void* out, const float* coef, size_t outer, int C);
int bn_add_relu_bwd_reduce_f32(cudaStream_t s, const float* a, const float* b, const float* y, const float* x, const float* mean, float* g, size_t outer, int C, float* part, int part_cap, int* part_rows);
int bn_add_relu_bwd_reduce_16(cudaStream_t s, int kind, const void* a, const void* b, const void* y, const void* x, const float* mean, void* g, size_t outer, int C, float* part, int part_cap, int* part_rows);

// ---- softmax / losses over [batch, count] --------------------------------------------------------------------
int softmax_fwd_f32(cudaStream_t s, const float* a, float* b, int batch, int count);
int softmax_bwd_f32(cudaStream_t s, const float* g, const float* b, float* h, int batch, int count);
// label_kind: 0 = fp32 class index, 1 = int32 class index, 2 = fp32 one-hot / distribution [batch, count]
int cce_fwd_f32(cudaStream_t s, const float* a, const void* label, int label_kind, float* c, int batch, int count, float trim0, float trim1);
int cce_bwd_f32(cudaStream_t s, const float* g, const float* a, const void* label, int label_kind, float* h, int batch, int count, float trim0, float trim1);
// fused softmax + cross entropy: c = loss (may be NULL), d = softmax probabilities
int softmax_cce_fwd_f32(cudaStream_t s, const float* a, const void* label, int label_kind, float* c, float* d, int batch, int count, float trim0, float trim1);
int softmax_cce_bwd_f32(cudaStream_t s, const float* g, const void* label, int label_kind, const float* d, float* h, int batch, int count, float trim0, float trim1);

// ---- SGD ------------------------------------------------------------------------------------------------------
int sgd_f32(cudaStream_t s, const float* g, const float* a, const float* m, float* b, float* n, size_t count, int nesterov, float rate, float scale, float decay, float momentum, float dampening);

// g of element kind g_kind (0 = fp32, 1 = bf16, 2 = fp16) with fp32 parameters / momenta: the reference's mixed-precision form
// (sgd/gpu/ccv_nnc_sgd_gpu_ref.cu:71-74)
int sgd_any(cudaStream_t s, int g_kind, const void* g, const float* a, const float* m, float* b, float* n, size_t count, int nesterov, float rate, float scale, float decay, float momentum, float dampening);
int sgd_multi_any(cudaStream_t s, int tensors, int g_kind, const void* const* g, const float* const* a, const float* const* m, float* const* b, float* const* n, const size_t* counts, int nesterov, float rate, float scale, float decay, float momentum, float dampening);
// `tensors` independent SGD updates with the same hyper-parameters in ceil(tensors / 32) launches
int sgd_multi_f32(cudaStream_t s, int tensors, const float* const* g, const float* const* a, const float* const* m, float* const* b, float* const* n, const size_t* counts, int nesterov, float rate, float scale, float decay, float momentum, float dampening);

// strided matrix of element kind `kind` (0 fp32, 1 bf16, 2 fp16) <-> dense fp32 (16-bit GEMM operands with strides TMA cannot take)
int widen_matrix(cudaStream_t s, const void* src, int kind, long long rs, long long cs, float* dst, int rows, int cols);
int narrow_matrix(cudaStream_t s, const float* src, void* dst, int kind, long long rs, long long cs, int rows, int cols, int accumulate);

// ---- datatype / layout ----------------------------------------------------------------------------------------
// dtype codes: 0 = f32, 1 = f16 (CPU_REF semantics: f32 -> f16 truncates, lib/ccv_util.c:1434-1440), 2 = f64, 3 = bf16 (RNE)
int convert_dtype(cudaStream_t s, const void* a, int a_dtype, void* b, int b_dtype, size_t n);
// generic <= 4-d strided copy b[i] = a[i] (views, NCHW <-> NHWC via permuted strides, transpose); elem_size 2, 4 or 8
int copy_strided(cudaStream_t s, const void* a, const int* astride, void* b, const int* bstride, const int* dim, int elem_size);

// ---- layer norm / rms norm over the last `inner` elements of each of `rows` rows -----------------------------
int layer_norm_fwd_f32(cudaStream_t s, const float* x, const float* scale, const float* bias, float* y, float* saved_mean, float* saved_inv_std, int rows, int inner, float epsilon);
int layer_norm_bwd_f32(cudaStream_t s, const float* g, const float* x, const float* scale, const float* saved_mean, const float* saved_inv_std, float* dx, float* dscale, float* dbias, int rows, int inner, void* workspace);
int rmsnorm_fwd_f32(cudaStream_t s, const float* x, const float* scale, float* y, float* saved_inv_std, int rows, int inner, float epsilon);
int rmsnorm_bwd_f32(cudaStream_t s, const float* g, const float* x, const float* scale, const float* saved_inv_std, float* dx, float* dscale, int rows, int inner, void* workspace);

// ---- group norm: <= 4-d index space, statistics / scale / bias tensors with dims dividing it (slot = i * rdim / dim) ----
struct GroupNormGeom {
	int dim[4];            // x / y / g / h dims (leading dims padded with 1)
	int rdim[4];           // saved_mean / saved_inv_std dims (packed)
	int sdim[4];           // scale / bias / dscale / dbias dims (packed)
	long long xstride[4], ystride[4], hstride[4]; // element strides of x, of y (forward) or g (backward), of h
};
int group_norm_fwd_f32(cudaStream_t s, const GroupNormGeom& g, const float* x, const float* scale, const float* bias, float* y, float* saved_mean, float* saved_inv_std, float epsilon);
size_t group_norm_bwd_workspace_bytes(const GroupNormGeom& g);
int group_norm_bwd_f32(cudaStream_t s, const GroupNormGeom& g, const float* grad, const float* x, const float* scale, const float* saved_mean, const float* saved_inv_std, float* h, float* dscale, float* dbias, void* workspace);

// ---- upsample (NHWC) ------------------------------------------------------------------------------------------
int upsample_fwd_f32(cudaStream_t s, const float* a, float* b, int N, int H, int W, int C, int OH, int OW, int type, int align_corners, int nchw);
int upsample_bwd_f32(cudaStream_t s, const float* g, float* h, int N, int H, int W, int C, int OH, int OW, int type, int align_corners, int nchw);

} // namespace sm100
