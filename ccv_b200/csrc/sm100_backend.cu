// sm100_backend.cu -- group (A) of include/ccv_nnc_sm100.h: the command layer of CCV_NNC_BACKEND_GPU_SM100.
//
// One exec function per command, with the reference's signature (lib/nnc/ccv_nnc.h:315) and positional tensor
// conventions (lib/nnc/ccv_nnc.h:308-314), and one registration function per command spelled exactly as
// REGISTER_COMMAND_BACKEND(cmd, CCV_NNC_BACKEND_GPU_SM100) would (lib/nnc/ccv_nnc_internal.h:196-202).  An exec only
// validates shapes, pulls the CUDA stream / workspace from the stream context and enqueues kernels; it never
// synchronises and there is no CPU path: anything it cannot run returns CCV_NNC_EXEC_INVALID.
#include "../../include/ccv_nnc_sm100.h"
#include "sm100_contract.h"
#include "sm100_ew.h"
#include <cuda_runtime.h>
#include <string.h>
#include <algorithm>
#include <vector>

using namespace sm100;

namespace {

struct TV {
	unsigned char* p;
	int nd;
	int dim[CCV_NNC_MAX_DIM_ALLOC];
	int stride[CCV_NNC_MAX_DIM_ALLOC];
	int contiguous;
	int datatype;
	int format;
	size_t count;
};

int tensor_nd(const int* const dim)
{
	int i;
	for (i = 0; i < CCV_NNC_MAX_DIM_ALLOC; i++)
		if (dim[i] == 0)
			return i;
	return CCV_NNC_MAX_DIM_ALLOC;
}

// ccv_nnc_tensor_view_get_stride (lib/nnc/ccv_nnc_easy.h): a view carries its strides, a plain tensor is packed
TV view_of(const ccv_nnc_tensor_t* const t)
{
	TV v;
	memset(&v, 0, sizeof(v));
	v.p = t->data.u8;
	v.nd = tensor_nd(t->info.dim);
	v.datatype = CCV_GET_DATA_TYPE(t->info.datatype);
	v.format = t->info.format;
	v.count = 1;
	int i;
	for (i = 0; i < v.nd; i++)
		v.dim[i] = t->info.dim[i], v.count *= (size_t)t->info.dim[i];
	if (CCV_IS_TENSOR_VIEW(t))
	{
		const ccv_nnc_tensor_view_t* const tv = (const ccv_nnc_tensor_view_t*)t;
		int packed = 1;
		v.contiguous = 1;
		for (i = v.nd - 1; i >= 0; i--)
		{
			v.stride[i] = tv->stride[i];
			if (v.dim[i] != 1 && tv->stride[i] != packed)
				v.contiguous = 0;
			packed *= v.dim[i];
		}
	} else {
		int packed = 1;
		for (i = v.nd - 1; i >= 0; i--)
			v.stride[i] = packed, packed *= v.dim[i];
		v.contiguous = 1;
	}
	return v;
}

// ccv_nnc_tensor_view_get_dim: right-align into 4 dims with leading 1s
void dims4(const TV& v, int dim[4], int stride[4])
{
	const int off = 4 - v.nd;
	int i;
	for (i = 0; i < 4; i++)
	{
		if (i < off)
			dim[i] = 1, stride[i] = 0;
		else
			dim[i] = v.dim[i - off], stride[i] = v.stride[i - off];
	}
}

inline cudaStream_t stream_of(ccv_nnc_stream_context_t* const stream_context)
{
	return (cudaStream_t)ccv_nnc_stream_context_get_stream(stream_context);
}

// split-K scratch of one command: the stream workspace (grow-only, one buffer per stream: lib/nnc/gpu/ccv_nnc_compat.cu:438-471).
// A command that also stages tensors in the workspace asks for both at once and passes the tail (scratch_at).
inline Scratch scratch_of(ccv_nnc_stream_context_t* const stream_context)
{
	void* const p = ccv_nnc_stream_context_get_workspace(stream_context, CONTRACT_SCRATCH_BYTES, CCV_TENSOR_GPU_MEMORY);
	const Scratch s = { p, p ? CONTRACT_SCRATCH_BYTES : 0 };
	return s;
}
inline Scratch scratch_at(void* const p, const size_t bytes)
{
	const Scratch s = { p, p ? bytes : 0 };
	return s;
}

inline bool is_f32(const ccv_nnc_tensor_t* const t) { return CCV_GET_DATA_TYPE(t->info.datatype) == CCV_32F; }
// element kind of the kernels that exist for three floating-point types: 0 = fp32, 1 = bf16, 2 = fp16; -1 otherwise
inline int kind_of(const ccv_nnc_tensor_t* const t)
{
	switch (CCV_GET_DATA_TYPE(t->info.datatype))
	{
		case CCV_32F: return 0;
		case CCV_16BF: return 1;
		case CCV_16F: return 2;
	}
	return -1;
}
inline size_t kind_size(const int kind) { return kind == 0 ? 4 : 2; }
inline uint16_t f32_to_16(const float v, const int kind); // host-side rounding of a fill value (defined with exec_via_f32)

bool same_shape(const TV& a, const TV& b)
{
	if (a.nd != b.nd)
		return false;
	for (int i = 0; i < a.nd; i++)
		if (a.dim[i] != b.dim[i])
			return false;
	return true;
}

int dtype_code(const int datatype)
{
	switch (CCV_GET_DATA_TYPE(datatype))
	{
		case CCV_32F: return 0;
		case CCV_16F: return 1;
		case CCV_64F: return 2;
		case CCV_16BF: return 3;
	}
	return -1;
}

size_t dtype_size(const int datatype)
{
	switch (CCV_GET_DATA_TYPE(datatype))
	{
		case CCV_8U: return 1;
		case CCV_16F: case CCV_16BF: return 2;
		case CCV_32F: case CCV_32S: return 4;
		case CCV_64F: case CCV_64S: return 8;
	}
	return 0;
}

#define RC(x) do { const int rc_ = (x); if (rc_ < 0) return CCV_NNC_EXEC_INVALID; if (rc_ > 0) return CCV_NNC_EXEC_INVALID; } while (0)

// ================================================================================================ GEMM
struct Mat {
	float* p;
	int batch, rows, cols;
	long long batch_inc, rs, cs;
};

// ccv_nnc_tensor_get_matrix_params (lib/nnc/ccv_nnc_easy.h:421-444) for nd <= 3
bool mat_of(const TV& v, const int transpose[2], Mat& m)
{
	if (v.nd < 1 || v.nd > 3)
		return false;
	m.p = (float*)v.p;
	m.batch = v.nd < 3 ? 1 : v.dim[v.nd - 3];
	m.batch_inc = v.nd < 3 ? 0 : v.stride[v.nd - 3];
	m.rows = v.nd == 1 ? 1 : v.dim[v.nd - 2];
	m.rs = v.nd >= 2 ? v.stride[v.nd - 2] : (long long)v.stride[0] * v.dim[0];
	m.cols = v.dim[v.nd - 1];
	m.cs = v.stride[v.nd - 1];
	if (transpose[0] != transpose[1])
	{
		const int t = m.rows;
		m.rows = m.cols, m.cols = t;
		const long long u = m.rs;
		m.rs = m.cs, m.cs = u;
	}
	return true;
}

// Algorithm of a GEMM command.  An explicit cmd.algorithm (what ccv_nnc_cmd_autotune stores) wins; otherwise fp32 data means
// fp32-grade products -- the reference's cuBLAS path computes fp32 GEMMs in CUBLAS_COMPUTE_32F
// (lib/nnc/gpu/ccv_nnc_compat.cu:786-803) -- i.e. the error-compensated 3xTF32 kernel, unless the caller opted into TF32 with
// CCV_NNC_GEMM_32TF (lib/nnc/ccv_nnc.h:103-105).
int gemm_algorithm(const ccv_nnc_cmd_t& cmd)
{
	if (cmd.algorithm >= 0 && cmd.algorithm < CCV_NNC_SM100_ALGO_COUNT)
		return cmd.algorithm;
	return (cmd.info.blas.flags & CCV_NNC_GEMM_32TF) ? CCV_NNC_SM100_ALGO_TF32 : CCV_NNC_SM100_ALGO_3XTF32;
}
// Algorithm of a CONVOLUTION command: explicit, else one-pass TF32 -- the reference's own GPU convolution sets
// CUDNN_TENSOR_OP_MATH on every convolution descriptor (lib/nnc/gpu/ccv_nnc_compat.cu:1393), which is TF32 tensor-core math
// for fp32 data; CCV_NNC_SM100_ALGO_3XTF32 / _FFMA are there for callers that need fp32-grade convolutions.
int conv_algorithm(const ccv_nnc_cmd_t& cmd)
{
	if (cmd.algorithm >= 0 && cmd.algorithm < CCV_NNC_SM100_ALGO_COUNT)
		return cmd.algorithm;
	return CCV_NNC_SM100_ALGO_TF32;
}

// C[M, N] (+)= A[M, K] * B[K, N] + bias over arbitrary (row, col) element strides
int gemm_dispatch(cudaStream_t s, const Scratch& scratch, const int algorithm, const int M, const int N, const int K, const float* a, long long a_rs, long long a_cs, const float* b, long long b_rs, long long b_cs, float* c, long long c_rs, long long c_cs, const float* bias, const int accumulate)
{
	if (M <= 0 || N <= 0)
		return 0;
	if (K <= 0)
		return 1;
	if (c_cs != 1 && N > 1)
	{
		if (c_rs != 1 && M > 1)
			return 1;
		if (bias)
			return 1;
		// C^T = B^T A^T
		return gemm_dispatch(s, scratch, algorithm, N, M, K, b, b_cs, b_rs, a, a_cs, a_rs, c, c_cs, 1, 0, accumulate);
	}
	if (algorithm != CCV_NNC_SM100_ALGO_FFMA)
	{
		int ta = -1, tb = -1;
		long long lda = 0, ldb = 0;
		if (a_cs == 1 || K == 1)
			ta = 0, lda = a_rs;
		else if (a_rs == 1 || M == 1)
			ta = 1, lda = a_cs;
		if (b_cs == 1 || N == 1)
			tb = 0, ldb = b_rs;
		else if (b_rs == 1 || K == 1)
			tb = 1, ldb = b_cs;
		if (ta >= 0 && tb >= 0)
		{
			const int rc = gemm_tf32(s, M, N, K, a, lda, ta, b, ldb, tb, c, c_rs, bias, accumulate, scratch, algorithm == CCV_NNC_SM100_ALGO_3XTF32);
			if (rc <= 0)
				return rc;
		}
	}
	return gemm_ffma(s, M, N, K, a, a_rs, a_cs, b, b_rs, b_cs, c, c_rs, bias, accumulate);
}

// the same for 16-bit tensors (kind 1 = bf16, 2 = fp16): tensor-core path only (unit stride along one axis of every operand)
int gemm_dispatch16(cudaStream_t s, const Scratch& scratch, const int kind, const int M, const int N, const int K, const void* a, long long a_rs, long long a_cs, const void* b, long long b_rs, long long b_cs, void* c, long long c_rs, long long c_cs, const float* bias32, const void* bias16, const int accumulate)
{
	if (M <= 0 || N <= 0)
		return 0;
	if (K <= 0)
		return 1;
	if (c_cs != 1 && N > 1)
	{
		if ((c_rs != 1 && M > 1) || bias32 || bias16)
			return 1;
		return gemm_dispatch16(s, scratch, kind, N, M, K, b, b_cs, b_rs, a, a_cs, a_rs, c, c_cs, 1, 0, 0, accumulate); // C^T = B^T A^T
	}
	int ta = -1, tb = -1;
	long long lda = 0, ldb = 0;
	if (a_cs == 1 || K == 1)
		ta = 0, lda = a_rs;
	else if (a_rs == 1 || M == 1)
		ta = 1, lda = a_cs;
	if (b_cs == 1 || N == 1)
		tb = 0, ldb = b_rs;
	else if (b_rs == 1 || K == 1)
		tb = 1, ldb = b_cs;
	if (ta >= 0 && tb >= 0)
	{
		const int rc = gemm_16(s, kind, M, N, K, a, lda, ta, b, ldb, tb, c, c_rs, bias32, bias16, accumulate, scratch);
		if (rc <= 0)
			return rc;
	}
	// Shapes the tensor-core path cannot take (a leading dimension that is not a multiple of 16 bytes, e.g. a 10-class head):
	// widen the operands into the command's scratch, multiply in fp32 on the CUDA cores, narrow the result (one rounding).  Small
	// by construction: anything large has TMA-friendly strides.
	const size_t need = ((size_t)M * K + (size_t)K * N + (size_t)M * N + (size_t)N) * sizeof(float) + 1024;
	if (!scratch.ptr || scratch.bytes < need)
		return 1;
	float* const a32 = (float*)scratch.ptr;
	float* const b32 = a32 + (((size_t)M * K + 63) & ~(size_t)63);
	float* const c32 = b32 + (((size_t)K * N + 63) & ~(size_t)63);
	float* const bias_w = c32 + (((size_t)M * N + 63) & ~(size_t)63);
	if (widen_matrix(s, a, kind, a_rs, a_cs, a32, M, K) || widen_matrix(s, b, kind, b_rs, b_cs, b32, K, N))
		return -1;
	const float* bias_f = bias32;
	if (!bias_f && bias16)
	{
		if (widen_matrix(s, bias16, kind, 0, 1, bias_w, 1, N))
			return -1;
		bias_f = bias_w;
	}
	const int rc = gemm_ffma(s, M, N, K, a32, K, 1, b32, N, 1, c32, N, bias_f, 0);
	if (rc)
		return rc;
	return narrow_matrix(s, c32, c, kind, c_rs, c_cs, M, N, accumulate) ? -1 : 0;
}

// blas/ccv_nnc_gemm_cpu_ref.c:110-184
int exec_gemm_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 2 || output_size < 1 || !inputs[0] || !inputs[1] || !outputs[0])
		return CCV_NNC_EXEC_INVALID;
	const ccv_nnc_tensor_t* const bias_t = input_size > 2 ? inputs[2] : 0;
	const int kind = kind_of(inputs[0]);
	if (kind < 0 || kind_of(inputs[1]) != kind || kind_of(outputs[0]) != kind || (bias_t && kind_of(bias_t) != kind && !is_f32(bias_t)))
		return CCV_NNC_EXEC_INVALID;
	const int no_transpose[2] = { 0, 0 };
	Mat a, w, b, bias;
	if (!mat_of(view_of(inputs[0]), cmd.info.blas.transpose_a, a) || !mat_of(view_of(inputs[1]), cmd.info.blas.transpose_b, w) || !mat_of(view_of(outputs[0]), no_transpose, b))
		return CCV_NNC_EXEC_INVALID;
	if (a.rows != b.rows || a.cols != w.rows || w.cols != b.cols)
		return CCV_NNC_EXEC_INVALID;
	if ((a.batch != b.batch && a.batch != 1) || (w.batch != b.batch && w.batch != 1))
		return CCV_NNC_EXEC_INVALID;
	if (a.batch == 1)
		a.batch_inc = 0;
	if (w.batch == 1)
		w.batch_inc = 0;
	bool matrix_bias = false;
	if (bias_t)
	{
		if (!mat_of(view_of(bias_t), no_transpose, bias) || bias.cols != b.cols || bias.cs != 1)
			return CCV_NNC_EXEC_INVALID;
		// the third operand is a row vector added to every row, or (blas/gpu/ccv_nnc_gemm_gpu_cublas.cu; test/int/nnc/cublas.tests.c:164-211)
		// a full [M, N] matrix: then c = a w + d, applied as a second pass
		matrix_bias = bias.rows == b.rows && bias.rows != 1;
		if ((bias.rows != 1 && !matrix_bias) || (matrix_bias && (kind != 0 || b.cs != 1)))
			return CCV_NNC_EXEC_INVALID;
		if (bias.batch == 1)
			bias.batch_inc = 0;
	}
	cudaStream_t s = stream_of(stream_context);
	const Scratch scratch = scratch_of(stream_context);
	if (matrix_bias)
	{
		for (int i = 0; i < b.batch; i++)
		{
			RC(gemm_dispatch(s, scratch, gemm_algorithm(cmd), b.rows, b.cols, a.cols, a.p + i * a.batch_inc, a.rs, a.cs, w.p + i * w.batch_inc, w.rs, w.cs, b.p + i * b.batch_inc, b.rs, b.cs, 0, 0));
			const int d4[4] = { 1, 1, b.rows, b.cols }, cs4[4] = { 0, 0, (int)b.rs, 1 }, ds4[4] = { 0, 0, (int)bias.rs, 1 };
			RC(ew_axpby_bcast_f32(s, 1.f, b.p + i * b.batch_inc, cs4, 1.f, bias.p + i * bias.batch_inc, ds4, b.p + i * b.batch_inc, cs4, d4));
		}
		return CCV_NNC_EXEC_SUCCESS;
	}
	if (kind != 0)
	{
		// 16-bit operands: tcgen05 kind::f16, fp32 accumulate; the bias may be fp32 or in the operands' type
		const char* const bias_p = bias_t ? (const char*)bias.p : 0;
		const bool bias32 = bias_t && is_f32(bias_t);
		for (int i = 0; i < b.batch; i++)
			RC(gemm_dispatch16(s, scratch, kind, b.rows, b.cols, a.cols, (const char*)a.p + (size_t)i * a.batch_inc * 2, a.rs, a.cs, (const char*)w.p + (size_t)i * w.batch_inc * 2, w.rs, w.cs, (char*)b.p + (size_t)i * b.batch_inc * 2, b.rs, b.cs,
				bias32 ? (const float*)(bias_p + (size_t)i * bias.batch_inc * 4) : 0, bias_t && !bias32 ? bias_p + (size_t)i * bias.batch_inc * 2 : 0, 0));
		return CCV_NNC_EXEC_SUCCESS;
	}
	for (int i = 0; i < b.batch; i++)
		RC(gemm_dispatch(s, scratch, gemm_algorithm(cmd), b.rows, b.cols, a.cols, a.p + i * a.batch_inc, a.rs, a.cs, w.p + i * w.batch_inc, w.rs, w.cs, b.p + i * b.batch_inc, b.rs, b.cs, bias_t ? bias.p + i * bias.batch_inc : 0, 0));
	return CCV_NNC_EXEC_SUCCESS;
}

// blas/ccv_nnc_gemm_cpu_ref.c:318-448: inputs (g, a, w), outputs (h, dw, dbias), each optional
int exec_gemm_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 2 || output_size < 1 || !inputs[0])
		return CCV_NNC_EXEC_INVALID;
	const int no_transpose[2] = { 0, 0 };
	const int accumulate = (flags & CCV_NNC_ACCUMULATE_OUTPUT) ? 1 : 0;
	Mat g;
	const int kind = kind_of(inputs[0]);
	if (kind < 0 || !mat_of(view_of(inputs[0]), no_transpose, g))
		return CCV_NNC_EXEC_INVALID;
	const size_t esz = kind_size(kind);
	cudaStream_t s = stream_of(stream_context);
	ccv_nnc_tensor_t* const dbias_t = output_size > 2 ? outputs[2] : 0;
	ccv_nnc_tensor_t* const dw_t = output_size > 1 ? outputs[1] : 0;
	ccv_nnc_tensor_t* const h_t = outputs[0];
	if (dbias_t)
	{
		Mat db;
		if (!mat_of(view_of(dbias_t), no_transpose, db) || db.cols != g.cols || db.cs != 1 || g.cs != 1 || db.rows != 1)
			return CCV_NNC_EXEC_INVALID;
		if (db.batch != 1 && db.batch != g.batch)
			return CCV_NNC_EXEC_INVALID;
		const int db_kind = kind_of(dbias_t);
		if (db_kind < 0)
			return CCV_NNC_EXEC_INVALID;
		for (int i = 0; i < g.batch; i++)
			RC(colsum_any(s, kind, (const char*)g.p + (size_t)i * g.batch_inc * esz, g.rows, g.cols, g.rs, (char*)db.p + (db.batch == 1 ? 0 : (size_t)i * db.batch_inc * kind_size(db_kind)), db_kind, accumulate || (db.batch == 1 && i > 0), ccv_nnc_stream_context_get_workspace(stream_context, colsum_workspace_bytes(g.cols), CCV_TENSOR_GPU_MEMORY)));
	}
	if (dw_t)
	{
		if (!inputs[1] || kind_of(inputs[1]) != kind || kind_of(dw_t) != kind)
			return CCV_NNC_EXEC_INVALID;
		Mat a, dw;
		if (!mat_of(view_of(inputs[1]), cmd.info.blas.transpose_a, a) || !mat_of(view_of(dw_t), cmd.info.blas.transpose_b, dw))
			return CCV_NNC_EXEC_INVALID;
		if (a.rows != g.rows || a.cols != dw.rows || dw.cols != g.cols)
			return CCV_NNC_EXEC_INVALID;
		if (a.batch == 1)
			a.batch_inc = 0;
		// dw[K, N] = a^T[K, M] * g[M, N]; a shared dw sums over the batch
		if (kind != 0)
		{
			for (int i = 0; i < g.batch; i++)
				RC(gemm_dispatch16(s, scratch_of(stream_context), kind, dw.rows, dw.cols, g.rows, (const char*)a.p + (size_t)i * a.batch_inc * 2, a.cs, a.rs, (const char*)g.p + (size_t)i * g.batch_inc * 2, g.rs, g.cs, (char*)dw.p + (dw.batch == 1 ? 0 : (size_t)i * dw.batch_inc * 2), dw.rs, dw.cs, 0, 0, accumulate || (dw.batch == 1 && i > 0)));
		} else
		for (int i = 0; i < g.batch; i++)
			RC(gemm_dispatch(s, scratch_of(stream_context), gemm_algorithm(cmd), dw.rows, dw.cols, g.rows, a.p + i * a.batch_inc, a.cs, a.rs, g.p + i * g.batch_inc, g.rs, g.cs, dw.p + (dw.batch == 1 ? 0 : i * dw.batch_inc), dw.rs, dw.cs, 0, accumulate || (dw.batch == 1 && i > 0)));
	}
	if (h_t)
	{
		if (input_size < 3 || !inputs[2] || kind_of(inputs[2]) != kind || kind_of(h_t) != kind)
			return CCV_NNC_EXEC_INVALID;
		Mat h, w;
		if (!mat_of(view_of(h_t), cmd.info.blas.transpose_a, h) || !mat_of(view_of(inputs[2]), cmd.info.blas.transpose_b, w))
			return CCV_NNC_EXEC_INVALID;
		if (h.cols != w.rows || w.cols != g.cols || h.rows != g.rows)
			return CCV_NNC_EXEC_INVALID;
		if (w.batch == 1)
			w.batch_inc = 0;
		// h[M, K] = g[M, N] * w^T[N, K]
		if (kind != 0)
		{
			for (int i = 0; i < g.batch; i++)
				RC(gemm_dispatch16(s, scratch_of(stream_context), kind, h.rows, h.cols, g.cols, (const char*)g.p + (size_t)i * g.batch_inc * 2, g.rs, g.cs, (const char*)w.p + (size_t)i * w.batch_inc * 2, w.cs, w.rs, (char*)h.p + (h.batch == 1 ? 0 : (size_t)i * h.batch_inc * 2), h.rs, h.cs, 0, 0, accumulate || (h.batch == 1 && i > 0)));
		} else
		for (int i = 0; i < g.batch; i++)
			RC(gemm_dispatch(s, scratch_of(stream_context), gemm_algorithm(cmd), h.rows, h.cols, g.cols, g.p + i * g.batch_inc, g.rs, g.cs, w.p + i * w.batch_inc, w.cs, w.rs, h.p + (h.batch == 1 ? 0 : i * h.batch_inc), h.rs, h.cs, 0, accumulate || (h.batch == 1 && i > 0)));
	}
	return CCV_NNC_EXEC_SUCCESS;
}

// ------------------------------------------------------------------------------------------------ GEMM with two batch axes
// ccv_nnc_tensor_get_matrix_params (lib/nnc/ccv_nnc_easy.h:421-444) and the reference GEMMs take up to 4-d operands
// [b0, b1, rows, cols] (attention-style "batch (2, 4)" products, test/int/nnc/cublas.tests.c:1801-2100), any of them possibly a
// view, an operand with fewer axes being shared by every outer batch.  The 3-d commands above are run once per outer index on
// sub-views; an output that is shared across the outer axis accumulates from the second index on (in a call of its own, so
// that per-index outputs are still overwritten).
struct Slice4 {
	ccv_nnc_tensor_view_t v;
	int is4;
};
inline void slice4_make(ccv_nnc_tensor_t* const t, Slice4& sl)
{
	sl.is4 = t && tensor_nd(t->info.dim) == 4;
	if (!sl.is4)
		return;
	const TV tv = view_of(t);
	memset(&sl.v, 0, sizeof(sl.v));
	memcpy(&sl.v, t, sizeof(ccv_nnc_tensor_t));
	sl.v.type |= CCV_TENSOR_VIEW;
	memset(sl.v.info.dim, 0, sizeof(sl.v.info.dim));
	int packed = 1, contiguous = 1;
	for (int i = 2; i >= 0; i--)
	{
		sl.v.info.dim[i] = tv.dim[i + 1], sl.v.stride[i] = tv.stride[i + 1];
		if (tv.dim[i + 1] != 1 && tv.stride[i + 1] != packed)
			contiguous = 0;
		packed *= tv.dim[i + 1];
	}
	sl.v.contiguous = contiguous;
}
template <ccv_nnc_cmd_exec_f F>
int exec_gemm_nd4(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	enum { MAXT = 4 };
	int outer = 0;
	for (int i = 0; i < input_size; i++)
		if (inputs[i] && tensor_nd(inputs[i]->info.dim) == 4)
			outer = std::max(outer, inputs[i]->info.dim[0]);
	for (int i = 0; i < output_size; i++)
		if (outputs[i] && tensor_nd(outputs[i]->info.dim) == 4)
			outer = std::max(outer, outputs[i]->info.dim[0]);
	if (outer == 0)
		return F(cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
	if (input_size > MAXT || output_size > MAXT)
		return CCV_NNC_EXEC_INVALID;
	Slice4 si[MAXT], so[MAXT];
	ccv_nnc_tensor_t* in[MAXT];
	ccv_nnc_tensor_t* out[MAXT];
	ccv_nnc_tensor_t* out_shared[MAXT];
	int any_shared = 0, any_sliced = 0;
	for (int i = 0; i < input_size; i++)
	{
		slice4_make(inputs[i], si[i]);
		if (si[i].is4 && inputs[i]->info.dim[0] != outer && inputs[i]->info.dim[0] != 1)
			return CCV_NNC_EXEC_INVALID;
	}
	for (int i = 0; i < output_size; i++)
	{
		slice4_make(outputs[i], so[i]);
		if (so[i].is4 && outputs[i]->info.dim[0] != outer && outputs[i]->info.dim[0] != 1)
			return CCV_NNC_EXEC_INVALID;
		if (outputs[i])
		{
			const int shared = !so[i].is4 || outputs[i]->info.dim[0] == 1;
			any_shared |= shared, any_sliced |= !shared;
		}
	}
	for (int o = 0; o < outer; o++)
	{
		for (int i = 0; i < input_size; i++)
		{
			in[i] = inputs[i];
			if (si[i].is4)
			{
				const size_t step = inputs[i]->info.dim[0] == 1 ? 0 : (size_t)o * view_of(inputs[i]).stride[0];
				si[i].v.data.u8 = inputs[i]->data.u8 + step * dtype_size(inputs[i]->info.datatype);
				in[i] = (ccv_nnc_tensor_t*)&si[i].v;
			}
		}
		for (int i = 0; i < output_size; i++)
		{
			out[i] = outputs[i], out_shared[i] = 0;
			if (!outputs[i])
				continue;
			const int shared = !so[i].is4 || outputs[i]->info.dim[0] == 1;
			if (so[i].is4)
			{
				const size_t step = outputs[i]->info.dim[0] == 1 ? 0 : (size_t)o * view_of(outputs[i]).stride[0];
				so[i].v.data.u8 = outputs[i]->data.u8 + step * dtype_size(outputs[i]->info.datatype);
				out[i] = (ccv_nnc_tensor_t*)&so[i].v;
			}
			if (shared && o > 0 && any_sliced)
				out_shared[i] = out[i], out[i] = 0; // second call, accumulating
		}
		if (o == 0 || any_sliced)
		{
			const int rc = F(cmd, hint, (o > 0 && !any_sliced) ? (flags | CCV_NNC_ACCUMULATE_OUTPUT) : flags, in, input_size, out, output_size, stream_context);
			if (rc != CCV_NNC_EXEC_SUCCESS)
				return rc;
		}
		if (o > 0 && any_shared)
		{
			const int rc = F(cmd, hint, flags | CCV_NNC_ACCUMULATE_OUTPUT, in, input_size, any_sliced ? out_shared : out, output_size, stream_context);
			if (rc != CCV_NNC_EXEC_SUCCESS)
				return rc;
		}
	}
	return CCV_NNC_EXEC_SUCCESS;
}

// ================================================================================================ CONVOLUTION
// NHWC activations ([N,] H, W, C), filters [K, R, S, C / groups] (convolution/ccv_nnc_conv_cpu_ref.c:47-65)
bool conv_geom(const ccv_nnc_cmd_t& cmd, const ccv_nnc_hint_t& hint, const TV& a, const TV& w, const TV& b, ConvGeom& g)
{
	if (a.format != CCV_TENSOR_FORMAT_NHWC || b.format != CCV_TENSOR_FORMAT_NHWC)
		return false;
	if ((a.nd != 3 && a.nd != 4) || (b.nd != 3 && b.nd != 4) || w.nd != 4 || !w.contiguous)
		return false;
	const int ao = a.nd - 3, bo = b.nd - 3;
	memset(&g, 0, sizeof(g));
	g.N = a.nd == 4 ? a.dim[0] : 1;
	if ((b.nd == 4 ? b.dim[0] : 1) != g.N)
		return false;
	g.H = a.dim[ao], g.W = a.dim[ao + 1], g.C = a.dim[ao + 2];
	g.P = b.dim[bo], g.Q = b.dim[bo + 1], g.K = b.dim[bo + 2];
	g.R = w.dim[1], g.S = w.dim[2];
	if (a.stride[ao + 2] != 1 || b.stride[bo + 2] != 1)
		return false;
	g.an = a.nd == 4 ? a.stride[0] : (long long)g.H * a.stride[ao];
	g.ah = a.stride[ao], g.aw = a.stride[ao + 1];
	g.bn = b.nd == 4 ? b.stride[0] : (long long)g.P * b.stride[bo];
	g.bh = b.stride[bo], g.bw = b.stride[bo + 1];
	g.stride_h = hint.stride.dim[0] > 0 ? hint.stride.dim[0] : 1;
	g.stride_w = hint.stride.dim[1] > 0 ? hint.stride.dim[1] : 1;
	g.dil_h = cmd.info.convolution.dilation[0] > 1 ? cmd.info.convolution.dilation[0] : 1;
	g.dil_w = cmd.info.convolution.dilation[1] > 1 ? cmd.info.convolution.dilation[1] : 1;
	g.pad_h0 = hint.border.begin[0], g.pad_w0 = hint.border.begin[1];
	// CPU_REF clips the window at the far edge (SET_BORDER_OFFSET_SIZE_FOR), i.e. the effective end padding is whatever
	// the output extent implies, not hint.border.end
	g.pad_h1 = (g.P - 1) * g.stride_h + (g.R - 1) * g.dil_h + 1 - g.H - g.pad_h0;
	g.pad_w1 = (g.Q - 1) * g.stride_w + (g.S - 1) * g.dil_w + 1 - g.W - g.pad_w0;
	const int groups = cmd.info.convolution.groups > 0 ? cmd.info.convolution.groups : 1;
	if (w.dim[0] != g.K || g.K != cmd.info.convolution.count || w.dim[3] * groups != g.C || g.K % groups != 0)
		return false;
	if (cmd.info.size.dim[0] != g.R || cmd.info.size.dim[1] != g.S)
		return false;
	return true;
}

// ------------------------------------------------------------------------------------------------ grouped convolution on tensor cores
// groups > 1 (convolution/ccv_nnc_conv_cpu_ref.c:47-65; the reference's GPU path hands groups to cuDNN,
// convolution/gpu/ccv_nnc_conv_gpu_cudnn.cu:204-357): group i contracts channels [i C/g, (i+1) C/g) against filters
// [i K/g, (i+1) K/g) -- `groups` independent dense convolutions whose operands are channel SLICES of the NHWC tensors (pixel stride
// C, not C/g) except for the filters, whose rows are contiguous per group.  When a group is wide enough to fill tensor-core tiles
// (C/g and K/g multiples of the 16-byte vector and >= 16) each group's slices are made dense in the stream workspace (one strided
// copy in, one out), and the dense tcgen05 kernels above do the arithmetic; narrower groups (depthwise and the like) stay on the
// FFMA kernels, where the contraction is too short for a 64-deep MMA anyway.  PASS 0 = fprop, 1 = wgrad, 2 = dgrad.
// returns 0 done, 1 not applicable (caller falls back), < 0 error
template <int PASS>
int conv_grouped_tc(ccv_nnc_stream_context_t* const stream_context, const int kind, const ConvGeom& g, const int groups, const int x3, const int accumulate,
	const void* const act, const void* const filt, const float* const bias32, const void* const bias16, const void* const res, void* const out)
{
	const int align = kind == 0 ? 4 : 8;
	const size_t es = kind_size(kind);
	if (groups <= 1 || g.C % groups || g.K % groups)
		return 1;
	const int Cg = g.C / groups, Kg = g.K / groups;
	if (Cg % align || Kg % align || Cg < 16 || Kg < 16)
		return 1;
	const long long lim = 0x7fffffffll;
	if ((long long)g.N * g.an > lim || (long long)g.N * g.bn > lim)
		return 1; // copy_strided walks int strides
	ConvGeom gg = g;
	gg.C = Cg, gg.K = Kg;
	gg.aw = Cg, gg.ah = (long long)g.W * Cg, gg.an = (long long)g.H * g.W * Cg;
	gg.bw = Kg, gg.bh = (long long)g.Q * Kg, gg.bn = (long long)g.P * g.Q * Kg;
	const size_t nx = (size_t)g.N * g.H * g.W * Cg, ny = (size_t)g.N * g.P * g.Q * Kg;
	const size_t xb = (nx * es + 255) & ~(size_t)255, yb = (ny * es + 255) & ~(size_t)255;
	unsigned char* const ws = (unsigned char*)ccv_nnc_stream_context_get_workspace(stream_context, CONTRACT_SCRATCH_BYTES + xb + yb, CCV_TENSOR_GPU_MEMORY);
	if (!ws)
		return 1;
	const Scratch scratch = scratch_at(ws, CONTRACT_SCRATCH_BYTES);
	unsigned char* const xg = ws + CONTRACT_SCRATCH_BYTES;
	unsigned char* const yg = xg + xb;
	cudaStream_t s = stream_of(stream_context);
	const int xd[4] = { g.N, g.H, g.W, Cg }, xs_t[4] = { (int)g.an, (int)g.ah, (int)g.aw, 1 }, xs_d[4] = { g.H * g.W * Cg, g.W * Cg, Cg, 1 };
	const int yd[4] = { g.N, g.P, g.Q, Kg }, ys_t[4] = { (int)g.bn, (int)g.bh, (int)g.bw, 1 }, ys_d[4] = { g.P * g.Q * Kg, g.Q * Kg, Kg, 1 };
	const size_t wstep = (size_t)Kg * g.R * g.S * Cg * es;
	for (int i = 0; i < groups; i++)
	{
		// (an operand a pass does not use is NULL: no arithmetic on it)
		const unsigned char* const act_i = act ? (const unsigned char*)act + (size_t)i * Cg * es : 0;
		const unsigned char* const res_i = res ? (const unsigned char*)res + (size_t)i * Kg * es : 0;
		const unsigned char* const w_i = filt ? (const unsigned char*)filt + (size_t)i * wstep : 0;
		int rc;
		if (PASS == 0)
		{
			// y_i = conv(x_i, w_i) + bias_i
			if (copy_strided(s, act_i, xs_t, xg, xs_d, xd, (int)es))
				return -1;
			if (kind == 0)
				rc = conv_fprop_tf32(s, gg, (const float*)xg, (const float*)w_i, bias32 ? bias32 + (size_t)i * Kg : 0, (float*)yg, scratch, x3);
			else
				rc = conv_fprop_16(s, kind, gg, xg, w_i, bias32 ? bias32 + (size_t)i * Kg : 0, bias16 ? (const unsigned char*)bias16 + (size_t)i * Kg * 2 : 0, yg, scratch);
			if (rc)
				return i == 0 ? rc : -1;
			if (copy_strided(s, yg, ys_d, (unsigned char*)out + (size_t)i * Kg * es, ys_t, yd, (int)es))
				return -1;
		} else if (PASS == 1) {
			// dw_i (+)= wgrad(g_i, x_i): the filter gradient's rows of a group are contiguous
			if (copy_strided(s, act_i, xs_t, xg, xs_d, xd, (int)es) || copy_strided(s, res_i, ys_t, yg, ys_d, yd, (int)es))
				return -1;
			unsigned char* const dw_i = (unsigned char*)out + (size_t)i * wstep;
			if (kind == 0)
				rc = conv_wgrad_tf32(s, gg, (const float*)yg, (const float*)xg, (float*)dw_i, accumulate, scratch, x3);
			else
				rc = conv_wgrad_16(s, kind, gg, yg, xg, dw_i, accumulate, scratch);
			if (rc)
				return i == 0 ? rc : -1;
		} else {
			// h_i = dgrad(g_i, w_i)
			if (copy_strided(s, res_i, ys_t, yg, ys_d, yd, (int)es))
				return -1;
			if (kind == 0)
				rc = conv_dgrad_tf32(s, gg, (const float*)yg, (const float*)w_i, (float*)xg, scratch, x3);
			else
				rc = conv_dgrad_16(s, kind, gg, yg, w_i, xg, scratch);
			if (rc)
				return i == 0 ? rc : -1;
			if (copy_strided(s, xg, xs_d, (unsigned char*)out + (size_t)i * Cg * es, xs_t, xd, (int)es))
				return -1;
		}
	}
	return 0;
}

int conv_forw_nhwc(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 2 || output_size < 1 || !inputs[0] || !inputs[1] || !outputs[0])
		return CCV_NNC_EXEC_INVALID;
	const ccv_nnc_tensor_t* const bias_t = input_size > 2 ? inputs[2] : 0;
	const int kind = kind_of(inputs[0]);
	if (kind > 0)
	{
		// bf16 / fp16 tensors: NHWC, one group, tcgen05 kind::f16 with fp32 accumulation; the bias is fp32 or of the tensors' type
		if (kind_of(inputs[1]) != kind || kind_of(outputs[0]) != kind || (bias_t && ((kind_of(bias_t) != kind && !is_f32(bias_t)) || CCV_IS_TENSOR_VIEW(bias_t))))
			return CCV_NNC_EXEC_INVALID;
		ConvGeom g16;
		if (!conv_geom(cmd, hint, view_of(inputs[0]), view_of(inputs[1]), view_of(outputs[0]), g16) || (bias_t && bias_t->info.dim[0] != g16.K))
			return CCV_NNC_EXEC_INVALID;
		cudaStream_t s16 = stream_of(stream_context);
		const float* const bias32 = bias_t && is_f32(bias_t) ? bias_t->data.f32 : 0;
		const void* const bias16 = bias_t && !is_f32(bias_t) ? (const void*)bias_t->data.u8 : 0;
		if (cmd.info.convolution.groups > 1) // wide groups only: there is no 16-bit FFMA kernel to fall back to
			return conv_grouped_tc<0>(stream_context, kind, g16, cmd.info.convolution.groups, 0, 0, inputs[0]->data.u8, inputs[1]->data.u8, bias32, bias16, 0, outputs[0]->data.u8) == 0 ? CCV_NNC_EXEC_SUCCESS : CCV_NNC_EXEC_INVALID;
		int rc = conv_fprop_16(s16, kind, g16, inputs[0]->data.u8, inputs[1]->data.u8, bias32, bias16, outputs[0]->data.u8, scratch_of(stream_context));
		if (rc > 0 && g16.C % 8 != 0)
		{
			// pixels that TMA cannot address (the 3-channel stem): explicit im2col + tensor-core GEMM
			void* const ws = ccv_nnc_stream_context_get_workspace(stream_context, conv_im2col_workspace_bytes(g16, kind), CCV_TENSOR_GPU_MEMORY);
			if (ws)
				rc = conv_fprop_im2col_16(s16, kind, g16, inputs[0]->data.u8, inputs[1]->data.u8, bias32, bias16, outputs[0]->data.u8, ws);
		}
		return rc == 0 ? CCV_NNC_EXEC_SUCCESS : CCV_NNC_EXEC_INVALID;
	}
	if (!is_f32(inputs[0]) || !is_f32(inputs[1]) || !is_f32(outputs[0]) || (bias_t && (!is_f32(bias_t) || CCV_IS_TENSOR_VIEW(bias_t))))
		return CCV_NNC_EXEC_INVALID;
	ConvGeom g;
	const int groups = cmd.info.convolution.groups > 0 ? cmd.info.convolution.groups : 1;
	const int algo = conv_algorithm(cmd), x3 = algo == CCV_NNC_SM100_ALGO_3XTF32;
	cudaStream_t s = stream_of(stream_context);
	const float* a = inputs[0]->data.f32;
	const float* w = inputs[1]->data.f32;
	const float* bias = bias_t ? bias_t->data.f32 : 0;
	float* b = outputs[0]->data.f32;
	const TV ta = view_of(inputs[0]), tw = view_of(inputs[1]), tb = view_of(outputs[0]);
	if (!conv_geom(cmd, hint, ta, tw, tb, g))
		return CCV_NNC_EXEC_INVALID;
	if (bias_t && bias_t->info.dim[0] != g.K)
		return CCV_NNC_EXEC_INVALID;
	if (groups == 1 && algo != CCV_NNC_SM100_ALGO_FFMA)
	{
		int rc = conv_fprop_tf32(s, g, a, w, bias, b, scratch_of(stream_context), x3);
		if (rc > 0 && g.C % 4 != 0)
		{
			// TMA cannot address 12-byte pixels (the 3-channel stem): explicit im2col + tensor-core GEMM
			void* const ws = ccv_nnc_stream_context_get_workspace(stream_context, conv_im2col_workspace_bytes(g), CCV_TENSOR_GPU_MEMORY);
			if (ws)
				rc = conv_fprop_im2col_tf32(s, g, a, w, bias, b, ws, x3);
		}
		if (rc == 0)
			return CCV_NNC_EXEC_SUCCESS;
		if (rc < 0)
			return CCV_NNC_EXEC_INVALID;
	}
	if (groups > 1 && algo != CCV_NNC_SM100_ALGO_FFMA)
	{
		const int rc = conv_grouped_tc<0>(stream_context, 0, g, groups, x3, 0, a, w, bias, 0, 0, b);
		if (rc == 0)
			return CCV_NNC_EXEC_SUCCESS;
		if (rc < 0)
			return CCV_NNC_EXEC_INVALID;
	}
	RC(conv_fprop_ffma(s, g, groups, a, w, bias, b));
	return CCV_NNC_EXEC_SUCCESS;
}

// convolution/ccv_nnc_conv_cpu_ref.c:174-345: inputs (g, a, w), outputs (h, dw, dbias); dw / dbias honour
// CCV_NNC_ACCUMULATE_OUTPUT, h is always overwritten (:286)
int conv_back_nhwc(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 2 || output_size < 1 || !inputs[0] || !inputs[1])
		return CCV_NNC_EXEC_INVALID;
	ccv_nnc_tensor_t* const h_t = outputs[0];
	ccv_nnc_tensor_t* const dw_t = output_size > 1 ? outputs[1] : 0;
	ccv_nnc_tensor_t* const dbias_t = output_size > 2 ? outputs[2] : 0;
	const ccv_nnc_tensor_t* const w_t = input_size > 2 ? inputs[2] : 0;
	const ccv_nnc_tensor_t* const filt = dw_t ? dw_t : w_t;
	const int kind = kind_of(inputs[0]);
	if (kind > 0 && filt)
	{
		// bf16 / fp16: the same three products on the kind::f16 kernels; dbias in fp32 or the tensors' type
		if (kind_of(inputs[1]) != kind || kind_of(filt) != kind || (h_t && kind_of(h_t) != kind) || (w_t && kind_of(w_t) != kind))
			return CCV_NNC_EXEC_INVALID;
		const int groups16 = cmd.info.convolution.groups > 1 ? cmd.info.convolution.groups : 1;
		ConvGeom g16;
		if (!conv_geom(cmd, hint, view_of(inputs[1]), view_of(filt), view_of(inputs[0]), g16))
			return CCV_NNC_EXEC_INVALID;
		const int acc16 = (flags & CCV_NNC_ACCUMULATE_OUTPUT) ? 1 : 0;
		cudaStream_t s16 = stream_of(stream_context);
		if (dbias_t)
		{
			const int db_kind = kind_of(dbias_t);
			if (db_kind < 0 || dbias_t->info.dim[0] != g16.K || g16.bh != (long long)g16.Q * g16.bw || g16.bn != (long long)g16.P * g16.bh)
				return CCV_NNC_EXEC_INVALID;
			RC(colsum_any(s16, kind, inputs[0]->data.u8, (size_t)g16.N * g16.P * g16.Q, g16.K, g16.bw, dbias_t->data.u8, db_kind, acc16, ccv_nnc_stream_context_get_workspace(stream_context, colsum_workspace_bytes(g16.K), CCV_TENSOR_GPU_MEMORY)));
		}
		if (dw_t && groups16 > 1)
		{
			if (conv_grouped_tc<1>(stream_context, kind, g16, groups16, 0, acc16, inputs[1]->data.u8, 0, 0, 0, inputs[0]->data.u8, dw_t->data.u8))
				return CCV_NNC_EXEC_INVALID;
		} else if (dw_t) {
			int rc = conv_wgrad_16(s16, kind, g16, inputs[0]->data.u8, inputs[1]->data.u8, dw_t->data.u8, acc16, scratch_of(stream_context));
			if (rc > 0 && g16.C % 8 != 0)
			{
				void* const ws = ccv_nnc_stream_context_get_workspace(stream_context, conv_im2col_workspace_bytes(g16, kind), CCV_TENSOR_GPU_MEMORY);
				if (ws)
					rc = conv_wgrad_im2col_16(s16, kind, g16, inputs[0]->data.u8, inputs[1]->data.u8, dw_t->data.u8, acc16, ws);
			}
			if (rc)
				return CCV_NNC_EXEC_INVALID;
		}
		if (h_t)
		{
			ConvGeom gh16;
			if (!w_t || !conv_geom(cmd, hint, view_of(h_t), view_of(w_t), view_of(inputs[0]), gh16))
				return CCV_NNC_EXEC_INVALID;
			if (groups16 > 1)
			{
				if (conv_grouped_tc<2>(stream_context, kind, gh16, groups16, 0, 0, 0, w_t->data.u8, 0, 0, inputs[0]->data.u8, h_t->data.u8))
					return CCV_NNC_EXEC_INVALID;
			} else {
				const int rc = conv_dgrad_16(s16, kind, gh16, inputs[0]->data.u8, w_t->data.u8, h_t->data.u8, scratch_of(stream_context));
				if (rc < 0)
					return CCV_NNC_EXEC_INVALID;
				if (rc > 0)
				{
					// shapes the tensor-core path cannot take (3-channel pixels: the image gradient of a stem, test/int/nnc/cudnn.tests.c:499-577):
					// functional form -- widen g and w, fp32 FFMA data gradient, one rounding on the way back.  Dense tensors only.
					const size_t ng = (size_t)gh16.N * gh16.P * gh16.Q * gh16.K, nw = (size_t)gh16.K * gh16.R * gh16.S * gh16.C, nh = (size_t)gh16.N * gh16.H * gh16.W * gh16.C;
					if (gh16.bw != gh16.K || gh16.bh != (long long)gh16.Q * gh16.K || gh16.bn != (long long)gh16.P * gh16.Q * gh16.K || gh16.aw != gh16.C || gh16.ah != (long long)gh16.W * gh16.C || gh16.an != (long long)gh16.H * gh16.W * gh16.C || ng > 0x7fffffffull || nh > 0x7fffffffull)
						return CCV_NNC_EXEC_INVALID;
					float* const g32 = (float*)ccv_nnc_stream_context_get_workspace(stream_context, (ng + nw + nh) * sizeof(float) + 1024, CCV_TENSOR_GPU_MEMORY);
					if (!g32)
						return CCV_NNC_EXEC_OOM;
					float* const w32 = (float*)(((uintptr_t)(g32 + ng) + 255) & ~(uintptr_t)255);
					float* const h32 = (float*)(((uintptr_t)(w32 + nw) + 255) & ~(uintptr_t)255);
					RC(widen_matrix(s16, inputs[0]->data.u8, kind, (long long)ng, 1, g32, 1, (int)ng));
					RC(widen_matrix(s16, w_t->data.u8, kind, (long long)nw, 1, w32, 1, (int)nw));
					RC(conv_dgrad_ffma(s16, gh16, 1, g32, w32, h32));
					RC(narrow_matrix(s16, h32, h_t->data.u8, kind, (long long)nh, 1, 1, (int)nh, 0));
				}
			}
		}
		return CCV_NNC_EXEC_SUCCESS;
	}
	if (!filt || !is_f32(inputs[0]) || !is_f32(inputs[1]))
		return CCV_NNC_EXEC_INVALID;
	ConvGeom g;
	if (!conv_geom(cmd, hint, view_of(inputs[1]), view_of(filt), view_of(inputs[0]), g))
		return CCV_NNC_EXEC_INVALID;
	const int groups = cmd.info.convolution.groups > 0 ? cmd.info.convolution.groups : 1;
	const int accumulate = (flags & CCV_NNC_ACCUMULATE_OUTPUT) ? 1 : 0;
	const int algo = conv_algorithm(cmd), x3 = algo == CCV_NNC_SM100_ALGO_3XTF32;
	cudaStream_t s = stream_of(stream_context);
	const float* gb = inputs[0]->data.f32;
	const float* a = inputs[1]->data.f32;
	if (dbias_t)
	{
		if (dbias_t->info.dim[0] != g.K || g.bh != (long long)g.Q * g.bw || g.bn != (long long)g.P * g.bh)
			return CCV_NNC_EXEC_INVALID;
		RC(colsum_f32(s, gb, (size_t)g.N * g.P * g.Q, g.K, g.bw, dbias_t->data.f32, accumulate, ccv_nnc_stream_context_get_workspace(stream_context, colsum_workspace_bytes(g.K), CCV_TENSOR_GPU_MEMORY)));
	}
	if (dw_t)
	{
		int rc = 1;
		if (groups == 1 && algo != CCV_NNC_SM100_ALGO_FFMA)
		{
			rc = conv_wgrad_tf32(s, g, gb, a, dw_t->data.f32, accumulate, scratch_of(stream_context), x3);
			if (rc > 0 && g.C % 4 != 0)
			{
				void* const ws = ccv_nnc_stream_context_get_workspace(stream_context, conv_im2col_workspace_bytes(g), CCV_TENSOR_GPU_MEMORY);
				if (ws)
					rc = conv_wgrad_im2col_tf32(s, g, gb, a, dw_t->data.f32, accumulate, ws, x3);
			}
		}
		if (groups > 1 && algo != CCV_NNC_SM100_ALGO_FFMA)
			rc = conv_grouped_tc<1>(stream_context, 0, g, groups, x3, accumulate, a, 0, 0, 0, gb, dw_t->data.f32);
		if (rc < 0)
			return CCV_NNC_EXEC_INVALID;
		if (rc > 0)
			RC(conv_wgrad_ffma(s, g, groups, gb, a, dw_t->data.f32, accumulate));
	}
	if (h_t)
	{
		if (!w_t || !is_f32(h_t))
			return CCV_NNC_EXEC_INVALID;
		ConvGeom gh;
		if (!conv_geom(cmd, hint, view_of(h_t), view_of(w_t), view_of(inputs[0]), gh))
			return CCV_NNC_EXEC_INVALID;
		int rc = 1;
		if (groups == 1 && algo != CCV_NNC_SM100_ALGO_FFMA)
			rc = conv_dgrad_tf32(s, gh, gb, w_t->data.f32, h_t->data.f32, scratch_of(stream_context), x3);
		if (groups > 1 && algo != CCV_NNC_SM100_ALGO_FFMA)
			rc = conv_grouped_tc<2>(stream_context, 0, gh, groups, x3, 0, 0, w_t->data.f32, 0, 0, gb, h_t->data.f32);
		if (rc < 0)
			return CCV_NNC_EXEC_INVALID;
		if (rc > 0)
			RC(conv_dgrad_ffma(s, gh, groups, gb, w_t->data.f32, h_t->data.f32));
	}
	return CCV_NNC_EXEC_SUCCESS;
}

// ------------------------------------------------------------------------------------------------ NCHW / mixed formats
// The kernels are NHWC.  The reference's GPU convolution takes any mix of formats -- its tests run NHWC activations against NCHW
// filters and all-NCHW forward and backward (convolution/gpu/ccv_nnc_conv_gpu_cudnn.cu:204-357; test/int/nnc/cudnn.tests.c:24-85,
// 87-140, 417-497) -- so every NCHW operand is re-laid out into the stream workspace (one strided copy each way), the NHWC
// command runs on shadow tensors, and NCHW results are copied back.  The workspace is one grow-only buffer per stream: this
// layer asks for [inner | staging] in ONE request, `inner` being the most the NHWC command will ask for, so that the nested
// requests (smaller) return the same base and never move the staged tensors.
struct Staged {
	ccv_nnc_tensor_t shadow;
	ccv_nnc_tensor_t* orig;
	int d[4], src[4], dst[4]; // index space N, H, W, C with the NCHW and the NHWC strides
	size_t bytes;
	int elem;
};

inline bool is_nchw(const ccv_nnc_tensor_t* const t) { return t && t->info.format == CCV_TENSOR_FORMAT_NCHW && tensor_nd(t->info.dim) >= 3; }

bool stage_plan(ccv_nnc_tensor_t* const t, Staged& st)
{
	const TV v = view_of(t);
	const size_t elem = dtype_size(t->info.datatype);
	if (!v.contiguous || (v.nd != 3 && v.nd != 4) || elem == 0)
		return false;
	const int N = v.nd == 4 ? v.dim[0] : 1, C = v.dim[v.nd - 3], H = v.dim[v.nd - 2], W = v.dim[v.nd - 1];
	const int d[4] = { N, H, W, C }, src[4] = { C * H * W, W, 1, H * W }, dst[4] = { H * W * C, W * C, C, 1 };
	memcpy(st.d, d, sizeof(d)), memcpy(st.src, src, sizeof(src)), memcpy(st.dst, dst, sizeof(dst));
	st.orig = t;
	st.elem = (int)elem;
	st.bytes = (v.count * elem + 255) & ~(size_t)255;
	memcpy(&st.shadow, t, sizeof(ccv_nnc_tensor_t));
	st.shadow.type &= ~CCV_TENSOR_VIEW;
	st.shadow.info.format = CCV_TENSOR_FORMAT_NHWC;
	memset(st.shadow.info.dim, 0, sizeof(st.shadow.info.dim));
	if (v.nd == 4)
		st.shadow.info.dim[0] = N, st.shadow.info.dim[1] = H, st.shadow.info.dim[2] = W, st.shadow.info.dim[3] = C;
	else
		st.shadow.info.dim[0] = H, st.shadow.info.dim[1] = W, st.shadow.info.dim[2] = C;
	return true;
}

// upper bound of what the NHWC command requests from the workspace for this geometry
size_t conv_inner_workspace(const ConvGeom& g, const int kind, const int groups)
{
	size_t need = CONTRACT_SCRATCH_BYTES;
	if (groups > 1 && g.C % groups == 0 && g.K % groups == 0)
	{
		// conv_grouped_tc: split-K scratch + one group's dense activations and results
		const size_t es = kind_size(kind), nx = (size_t)g.N * g.H * g.W * (g.C / groups), ny = (size_t)g.N * g.P * g.Q * (g.K / groups);
		need += ((nx * es + 255) & ~(size_t)255) + ((ny * es + 255) & ~(size_t)255);
	}
	if (g.C % (kind == 0 ? 4 : 8) != 0)
		need = std::max(need, kind == 0 ? conv_im2col_workspace_bytes(g) : conv_im2col_workspace_bytes(g, kind));
	need = std::max(need, colsum_workspace_bytes(g.K));
	return (need + 255) & ~(size_t)255;
}

// `exec` = the NHWC command, `inner_of` = the most it requests from the workspace given the shadow tensor lists; `accumulating`
// = outputs[1..] may be read before they are written (CCV_NNC_ACCUMULATE_OUTPUT), so they are staged in as well
typedef size_t (*staged_inner_f)(const ccv_nnc_cmd_t& cmd, const ccv_nnc_hint_t& hint, ccv_nnc_tensor_t* const* in, int input_size, ccv_nnc_tensor_t* const* out, int output_size);
int nchw_staged(const ccv_nnc_cmd_exec_f exec, const staged_inner_f inner_of, const int accumulating, const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	enum { MAXT = 6 };
	if (input_size > 3 || output_size > 3)
		return CCV_NNC_EXEC_INVALID;
	Staged st[MAXT];
	ccv_nnc_tensor_t* in[3] = { 0, 0, 0 };
	ccv_nnc_tensor_t* out[3] = { 0, 0, 0 };
	int n = 0, slot_in[3] = { -1, -1, -1 }, slot_out[3] = { -1, -1, -1 };
	size_t staging = 0;
	for (int i = 0; i < input_size; i++)
	{
		in[i] = inputs[i];
		if (is_nchw(inputs[i]))
		{
			if (!stage_plan(inputs[i], st[n]))
				return CCV_NNC_EXEC_INVALID;
			staging += st[n].bytes, slot_in[i] = n++;
		}
	}
	for (int i = 0; i < output_size; i++)
	{
		out[i] = outputs[i];
		if (is_nchw(outputs[i]))
		{
			if (!stage_plan(outputs[i], st[n]))
				return CCV_NNC_EXEC_INVALID;
			staging += st[n].bytes, slot_out[i] = n++;
		}
	}
	for (int i = 0; i < 3; i++)
	{
		if (slot_in[i] >= 0)
			in[i] = &st[slot_in[i]].shadow;
		if (slot_out[i] >= 0)
			out[i] = &st[slot_out[i]].shadow;
	}
	const size_t inner = inner_of(cmd, hint, in, input_size, out, output_size);
	if (inner == (size_t)-1)
		return CCV_NNC_EXEC_INVALID;
	unsigned char* const ws = (unsigned char*)ccv_nnc_stream_context_get_workspace(stream_context, inner + staging, CCV_TENSOR_GPU_MEMORY);
	if (!ws)
		return CCV_NNC_EXEC_OOM;
	cudaStream_t s = stream_of(stream_context);
	unsigned char* p = ws + inner;
	for (int i = 0; i < n; i++)
		st[i].shadow.data.u8 = p, p += st[i].bytes;
	// operands in; outputs that accumulate come in too
	for (int i = 0; i < 3; i++)
		if (slot_in[i] >= 0)
		{
			const Staged& t = st[slot_in[i]];
			RC(copy_strided(s, t.orig->data.u8, t.src, t.shadow.data.u8, t.dst, t.d, t.elem));
		}
	if (accumulating && (flags & CCV_NNC_ACCUMULATE_OUTPUT))
		for (int i = 1; i < 3; i++)
			if (slot_out[i] >= 0)
			{
				const Staged& t = st[slot_out[i]];
				RC(copy_strided(s, t.orig->data.u8, t.src, t.shadow.data.u8, t.dst, t.d, t.elem));
			}
	const int rc = exec(cmd, hint, flags, in, input_size, out, output_size, stream_context);
	if (rc != CCV_NNC_EXEC_SUCCESS)
		return rc;
	if (ccv_nnc_stream_context_get_workspace(stream_context, 1, CCV_TENSOR_GPU_MEMORY) != (void*)ws)
	{
		// the NHWC command asked for more than `inner`: the workspace moved and the staged tensors with it (a bound above is wrong)
		set_last_error("staged convolution / pooling: workspace moved under the staged tensors", cudaErrorInvalidValue);
		return CCV_NNC_EXEC_INVALID;
	}
	for (int i = 0; i < 3; i++)
		if (slot_out[i] >= 0)
		{
			const Staged& t = st[slot_out[i]];
			RC(copy_strided(s, t.shadow.data.u8, t.dst, t.orig->data.u8, t.src, t.d, t.elem));
		}
	return CCV_NNC_EXEC_SUCCESS;
}

template <int BACKWARD>
size_t conv_staged_inner(const ccv_nnc_cmd_t& cmd, const ccv_nnc_hint_t& hint, ccv_nnc_tensor_t* const* const in, const int input_size, ccv_nnc_tensor_t* const* const out, const int output_size)
{
	// geometry on the shadows: activations, filter, output of the forward convolution
	ccv_nnc_tensor_t* const act = BACKWARD ? in[1] : in[0];
	ccv_nnc_tensor_t* const filt = BACKWARD ? (output_size > 1 && out[1] ? out[1] : (input_size > 2 ? in[2] : 0)) : in[1];
	ccv_nnc_tensor_t* const res = BACKWARD ? in[0] : out[0];
	ConvGeom g;
	if (!act || !filt || !res || kind_of(act) < 0 || !conv_geom(cmd, hint, view_of(act), view_of(filt), view_of(res), g))
		return (size_t)-1;
	return conv_inner_workspace(g, kind_of(act), cmd.info.convolution.groups > 1 ? cmd.info.convolution.groups : 1);
}
template <int BACKWARD>
int conv_staged(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	return nchw_staged(BACKWARD ? conv_back_nhwc : conv_forw_nhwc, conv_staged_inner<BACKWARD>, BACKWARD, cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

inline bool any_nchw(ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size)
{
	for (int i = 0; i < input_size; i++)
		if (is_nchw(inputs[i]))
			return true;
	for (int i = 0; i < output_size; i++)
		if (is_nchw(outputs[i]))
			return true;
	return false;
}

int exec_conv_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (any_nchw(inputs, input_size, outputs, output_size))
		return conv_staged<0>(cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
	return conv_forw_nhwc(cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

int exec_conv_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (any_nchw(inputs, input_size, outputs, output_size))
		return conv_staged<1>(cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
	return conv_back_nhwc(cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}


// ================================================================================================ BATCH NORM
// norm/ccv_nnc_batch_norm_cpu_ref.c:16-250.  Supported reduction shapes: per-channel statistics of an NHWC
// ([.., C], scale dims [1,1,1,C]) or NCHW ([N, C, H, W], scale dims [1,C,1,1]) tensor.
bool bn_layout(const TV& a, const TV& scale, size_t& outer, int& C, size_t& inner)
{
	int ad[4], as[4], rd[4], rs[4];
	if (a.nd > 4 || scale.nd > 4 || !a.contiguous || !scale.contiguous)
		return false;
	dims4(a, ad, as);
	dims4(scale, rd, rs);
	int axis = -1;
	for (int i = 0; i < 4; i++)
		if (rd[i] != 1)
		{
			if (axis >= 0 || rd[i] != ad[i])
				return false;
			axis = i;
		}
	if (axis < 0)
		axis = 3; // a single statistic over everything: C = 1
	if (rd[axis] == 1 && ad[axis] != 1)
	{
		// scale has one element but the tensor does not: treat the whole tensor as one channel
		outer = 1, C = 1, inner = a.count;
		return true;
	}
	outer = 1, inner = 1;
	for (int i = 0; i < axis; i++)
		outer *= ad[i];
	for (int i = axis + 1; i < 4; i++)
		inner *= ad[i];
	C = ad[axis];
	return true;
}

int bnorm_forw(const int fuse_relu, const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	// a 6th input is the statistics tensor of a fused convolution -> batch norm pair (ccv_nnc_sm100_graph_fuse): its `sig`
	// field carries the number of valid partial rows the convolution produced for this issue (0 = none: reduce here)
	const ccv_nnc_tensor_t* const stats_t = input_size == 6 ? inputs[5] : 0;
	if ((input_size != 5 && input_size != 6) || output_size < 1)
		return CCV_NNC_EXEC_INVALID;
	// x / y may be fp32, bf16 or fp16; scale, bias and the statistics are fp32 (lib/nnc/ccv_cnnp_model_addons.c:954-956)
	for (int i = 1; i < 5; i++)
		if (!inputs[i] || !is_f32(inputs[i]))
			return CCV_NNC_EXEC_INVALID;
	const int kind = inputs[0] ? kind_of(inputs[0]) : -1;
	if (kind < 0 || !outputs[0] || kind_of(outputs[0]) != kind)
		return CCV_NNC_EXEC_INVALID;
	const TV a = view_of(inputs[0]), scale = view_of(inputs[1]), b = view_of(outputs[0]);
	size_t outer, inner;
	int C;
	if (!same_shape(a, b) || !b.contiguous || !bn_layout(a, scale, outer, C, inner))
		return CCV_NNC_EXEC_INVALID;
	for (int i = 2; i < 5; i++)
		if (view_of(inputs[i]).count != (size_t)C)
			return CCV_NNC_EXEC_INVALID;
	cudaStream_t s = stream_of(stream_context);
	if (cmd.info.bnorm.is_test)
	{
		if (fuse_relu)
			return CCV_NNC_EXEC_INVALID;
		void* const tws = ccv_nnc_stream_context_get_workspace(stream_context, bn_workspace_bytes(C), CCV_TENSOR_GPU_MEMORY);
		if (!tws)
			return CCV_NNC_EXEC_OOM;
		if (kind == 0)
			RC(bn_fwd_test_f32(s, inputs[0]->data.f32, outputs[0]->data.f32, inputs[1]->data.f32, inputs[2]->data.f32, inputs[3]->data.f32, inputs[4]->data.f32, outer, C, inner, cmd.info.bnorm.epsilon, tws));
		else
			RC(bn_fwd_test_16(s, kind, inputs[0]->data.u8, outputs[0]->data.u8, inputs[1]->data.f32, inputs[2]->data.f32, inputs[3]->data.f32, inputs[4]->data.f32, outer, C, inner, cmd.info.bnorm.epsilon, tws));
		return CCV_NNC_EXEC_SUCCESS;
	}
	// a 6th output is the [2, C] fp32 coefficient tensor of a statistics-only batch norm (rewrite (h) of ccv_nnc_sm100_graph_fuse):
	// it receives the a, b of y = x * a + b and y itself is not written -- the residual add behind it applies them
	ccv_nnc_tensor_t* const coef_t = output_size == 6 ? outputs[5] : 0;
	if ((output_size != 5 && !coef_t) || !outputs[1] || !outputs[2] || !outputs[3] || !outputs[4])
		return CCV_NNC_EXEC_INVALID;
	if (coef_t && (fuse_relu || !is_f32(coef_t) || !view_of(coef_t).contiguous || view_of(coef_t).count != 2 * (size_t)C))
		return CCV_NNC_EXEC_INVALID;
	// running mean / var are updated in place (:45-46)
	if (inputs[3]->data.f32 != outputs[1]->data.f32 || inputs[4]->data.f32 != outputs[2]->data.f32)
		return CCV_NNC_EXEC_INVALID;
	if (view_of(outputs[3]).count != (size_t)C || view_of(outputs[4]).count != (size_t)C)
		return CCV_NNC_EXEC_INVALID;
	void* const ws = ccv_nnc_stream_context_get_workspace(stream_context, bn_workspace_bytes(C), CCV_TENSOR_GPU_MEMORY);
	if (!ws)
		return CCV_NNC_EXEC_OOM;
	for (int i = 1; i < 5; i++)
		if (!is_f32(outputs[i]))
			return CCV_NNC_EXEC_INVALID;
	if (kind == 0)
		RC(bn_fwd_train_f32(s, inputs[0]->data.f32, outputs[0]->data.f32, inputs[1]->data.f32, inputs[2]->data.f32, outputs[1]->data.f32, outputs[2]->data.f32, outputs[3]->data.f32, outputs[4]->data.f32, outer, C, inner, cmd.info.bnorm.epsilon, cmd.info.bnorm.momentum, ws, fuse_relu,
			stats_t && inner == 1 ? stats_t->data.f32 : 0, stats_t ? (int)stats_t->sig : 0, coef_t ? coef_t->data.f32 : 0));
	else
		RC(bn_fwd_train_16(s, kind, inputs[0]->data.u8, outputs[0]->data.u8, inputs[1]->data.f32, inputs[2]->data.f32, outputs[1]->data.f32, outputs[2]->data.f32, outputs[3]->data.f32, outputs[4]->data.f32, outer, C, inner, cmd.info.bnorm.epsilon, cmd.info.bnorm.momentum, ws, fuse_relu,
			stats_t && inner == 1 ? stats_t->data.f32 : 0, stats_t ? (int)stats_t->sig : 0, coef_t ? coef_t->data.f32 : 0));
	return CCV_NNC_EXEC_SUCCESS;
}

int exec_bnorm_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	return bnorm_forw(0, cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

static inline bool h_t_ok(const ccv_nnc_tensor_t* const h) { return h != 0; }

// norm/ccv_nnc_batch_norm_cpu_ref.c:312-470: inputs[0] = g, [5] = a, [6] = scale, [13] = saved_mean, [14] = saved_inv_std;
// outputs (h, dscale, dbias)
int bnorm_back(const int fused_relu, const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if ((input_size != 15 && input_size != 16) || output_size < 1)
		return CCV_NNC_EXEC_INVALID;
	// a 16th input is the partial-row tensor the add + ReLU backward in front filled (rewrite (i) of ccv_nnc_sm100_graph_fuse): its
	// `sig` field carries the number of rows written for this issue (0 = none: reduce here)
	const ccv_nnc_tensor_t* const part_t = input_size == 16 ? inputs[15] : 0;
	// the fused form carries the forward bias in slot 7 (unused by BATCH_NORM_BACKWARD, norm/ccv_nnc_norm.c:28-37)
	const ccv_nnc_tensor_t* const bias_t = fused_relu ? inputs[7] : 0;
	if (fused_relu && !bias_t)
		return CCV_NNC_EXEC_INVALID;
	const ccv_nnc_tensor_t* const g_t = inputs[0];
	const ccv_nnc_tensor_t* const a_t = inputs[5];
	const ccv_nnc_tensor_t* const scale_t = inputs[6];
	const ccv_nnc_tensor_t* const mean_t = inputs[13];
	const ccv_nnc_tensor_t* const istd_t = inputs[14];
	if (!g_t || !a_t || !scale_t || !mean_t || !istd_t)
		return CCV_NNC_EXEC_INVALID;
	ccv_nnc_tensor_t* const h_t = outputs[0];
	ccv_nnc_tensor_t* const dscale_t = output_size > 1 ? outputs[1] : 0;
	ccv_nnc_tensor_t* const dbias_t = output_size > 2 ? outputs[2] : 0;
	// a 4th output is the bias gradient of the convolution that produced this batch norm's input (graph rewrite (g) of
	// ccv_nnc_sm100_graph_fuse): sum over pixels of the dx written here
	ccv_nnc_tensor_t* const conv_dbias_t = output_size > 3 ? outputs[3] : 0;
	const TV a = view_of(a_t), g = view_of(g_t), scale = view_of(scale_t);
	size_t outer, inner;
	int C;
	if (!same_shape(a, g) || !g.contiguous || !bn_layout(a, scale, outer, C, inner))
		return CCV_NNC_EXEC_INVALID;
	const int kind = kind_of(g_t);
	if (kind < 0 || kind_of(a_t) != kind || (h_t && kind_of(h_t) != kind) || !is_f32(scale_t) || !is_f32(mean_t) || !is_f32(istd_t) || (bias_t && !is_f32(bias_t)) || (dscale_t && !is_f32(dscale_t)) || (dbias_t && !is_f32(dbias_t)))
		return CCV_NNC_EXEC_INVALID;
	if (conv_dbias_t && (!h_t_ok(outputs[0]) || kind_of(conv_dbias_t) < 0 || view_of(conv_dbias_t).count != (size_t)C || !view_of(conv_dbias_t).contiguous))
		return CCV_NNC_EXEC_INVALID;
	if (h_t && (!same_shape(view_of(h_t), a) || !view_of(h_t).contiguous))
		return CCV_NNC_EXEC_INVALID;
	const bool ext = part_t && !fused_relu && inner == 1 && part_t->sig > 0 && is_f32(part_t) && part_t->info.dim[1] == 2 * C && (int)part_t->sig <= part_t->info.dim[0];
	const float* const ext_part = ext ? part_t->data.f32 : 0;
	const int ext_rows = ext ? (int)part_t->sig : 0;
	cudaStream_t s = stream_of(stream_context);
	void* const ws = ccv_nnc_stream_context_get_workspace(stream_context, bn_workspace_bytes(C), CCV_TENSOR_GPU_MEMORY);
	if (!ws)
		return CCV_NNC_EXEC_OOM;
	if (kind == 0 && (!conv_dbias_t || is_f32(conv_dbias_t)))
		RC(bn_bwd_f32(s, g_t->data.f32, a_t->data.f32, scale_t->data.f32, bias_t ? bias_t->data.f32 : 0, mean_t->data.f32, istd_t->data.f32, h_t ? h_t->data.f32 : 0, dscale_t ? dscale_t->data.f32 : 0, dbias_t ? dbias_t->data.f32 : 0, outer, C, inner, ws, conv_dbias_t ? conv_dbias_t->data.f32 : 0, ext_part, ext_rows));
	else if (kind != 0)
		RC(bn_bwd_16(s, kind, g_t->data.u8, a_t->data.u8, scale_t->data.f32, bias_t ? bias_t->data.f32 : 0, mean_t->data.f32, istd_t->data.f32, h_t ? (void*)h_t->data.u8 : 0, dscale_t ? dscale_t->data.f32 : 0, dbias_t ? dbias_t->data.f32 : 0, outer, C, inner, ws,
			conv_dbias_t ? (void*)conv_dbias_t->data.u8 : 0, conv_dbias_t ? kind_of(conv_dbias_t) : 0, ext_part, ext_rows));
	else
		return CCV_NNC_EXEC_INVALID;
	return CCV_NNC_EXEC_SUCCESS;
}

int exec_bnorm_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	return bnorm_back(0, cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

// ================================================================================================ RELU / EW
int exec_relu_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 1 || output_size < 1 || !inputs[0] || !outputs[0] || kind_of(inputs[0]) < 0 || kind_of(outputs[0]) != kind_of(inputs[0]))
		return CCV_NNC_EXEC_INVALID;
	const TV a = view_of(inputs[0]), b = view_of(outputs[0]);
	if (!a.contiguous || !b.contiguous || a.count != b.count)
		return CCV_NNC_EXEC_INVALID;
	if (kind_of(inputs[0]) == 0)
		RC(ew_relu_fwd_f32(stream_of(stream_context), inputs[0]->data.f32, outputs[0]->data.f32, a.count));
	else
		RC(ew_relu_fwd_16(stream_of(stream_context), kind_of(inputs[0]), inputs[0]->data.u8, outputs[0]->data.u8, a.count));
	return CCV_NNC_EXEC_SUCCESS;
}

int exec_relu_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size != 3 || output_size < 1 || !inputs[0] || !inputs[2] || !outputs[0])
		return CCV_NNC_EXEC_INVALID;
	const TV g = view_of(inputs[0]), b = view_of(inputs[2]), h = view_of(outputs[0]);
	if (!g.contiguous || !b.contiguous || !h.contiguous || g.count != b.count || g.count != h.count)
		return CCV_NNC_EXEC_INVALID;
	const int kind = kind_of(inputs[0]);
	if (kind < 0 || kind_of(inputs[2]) != kind || kind_of(outputs[0]) != kind)
		return CCV_NNC_EXEC_INVALID;
	if (kind == 0)
		RC(ew_relu_bwd_f32(stream_of(stream_context), inputs[0]->data.f32, inputs[2]->data.f32, outputs[0]->data.f32, g.count));
	else
		RC(ew_relu_bwd_16(stream_of(stream_context), kind, inputs[0]->data.u8, inputs[2]->data.u8, outputs[0]->data.u8, g.count));
	return CCV_NNC_EXEC_SUCCESS;
}

// ew/ccv_nnc_ew_cpu_ref.c:15-110,207-214
int exec_ewsum_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size >= 1 && output_size >= 1 && outputs[0] && CCV_GET_DATA_TYPE(outputs[0]->info.datatype) == CCV_32S)
	{
		// int32 tensors (ew/gpu/ccv_nnc_ew_gpu_cudnn.cu registers CCV_32S; test/int/nnc/cudnn.tests.c:4817-4850)
		const TV ci = view_of(outputs[0]);
		const int* iptrs[64];
		if (!ci.contiguous || input_size > 64)
			return CCV_NNC_EXEC_INVALID;
		for (int i = 0; i < input_size; i++)
		{
			if (!inputs[i] || CCV_GET_DATA_TYPE(inputs[i]->info.datatype) != CCV_32S || !view_of(inputs[i]).contiguous || view_of(inputs[i]).count != ci.count)
				return CCV_NNC_EXEC_INVALID;
			iptrs[i] = inputs[i]->data.i32;
		}
		RC(ew_sum_i32(stream_of(stream_context), iptrs, input_size, outputs[0]->data.i32, ci.count));
		return CCV_NNC_EXEC_SUCCESS;
	}
	if (input_size < 1 || output_size < 1 || !outputs[0] || kind_of(outputs[0]) < 0)
		return CCV_NNC_EXEC_INVALID;
	const TV c = view_of(outputs[0]);
	if (!c.contiguous || input_size > 64)
		return CCV_NNC_EXEC_INVALID;
	if (kind_of(outputs[0]) > 0)
	{
		// bf16 / fp16: up to 8 operands, summed in fp32 and rounded once
		const int kind = kind_of(outputs[0]);
		const void* p16[8];
		if (input_size > 8)
			return CCV_NNC_EXEC_INVALID;
		for (int i = 0; i < input_size; i++)
		{
			if (!inputs[i] || kind_of(inputs[i]) != kind || !view_of(inputs[i]).contiguous || view_of(inputs[i]).count != c.count)
				return CCV_NNC_EXEC_INVALID;
			p16[i] = inputs[i]->data.u8;
		}
		if (input_size == 1)
		{
			if (p16[0] != outputs[0]->data.u8 && cudaMemcpyAsync(outputs[0]->data.u8, p16[0], c.count * 2, cudaMemcpyDeviceToDevice, stream_of(stream_context)) != cudaSuccess)
				return CCV_NNC_EXEC_INVALID;
			return CCV_NNC_EXEC_SUCCESS;
		}
		RC(ew_sum_16(stream_of(stream_context), kind, p16, input_size, outputs[0]->data.u8, c.count));
		return CCV_NNC_EXEC_SUCCESS;
	}
	const float* ptrs[64];
	for (int i = 0; i < input_size; i++)
	{
		if (!inputs[i] || !is_f32(inputs[i]))
			return CCV_NNC_EXEC_INVALID;
		const TV a = view_of(inputs[i]);
		if (!a.contiguous || a.count != c.count)
			return CCV_NNC_EXEC_INVALID;
		ptrs[i] = inputs[i]->data.f32;
	}
	cudaStream_t s = stream_of(stream_context);
	if (input_size == 1)
	{
		if (ptrs[0] != outputs[0]->data.f32 && cudaMemcpyAsync(outputs[0]->data.f32, ptrs[0], c.count * 4, cudaMemcpyDeviceToDevice, s) != cudaSuccess)
			return CCV_NNC_EXEC_INVALID;
		return CCV_NNC_EXEC_SUCCESS;
	}
	RC(ew_sum_f32(s, ptrs, input_size, outputs[0]->data.f32, c.count));
	return CCV_NNC_EXEC_SUCCESS;
}

// ew/ccv_nnc_ew_cpu_ref.c:216-233: every output receives the incoming gradient (or ones if it is absent)
int exec_ewsum_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	cudaStream_t s = stream_of(stream_context);
	for (int i = 0; i < output_size; i++)
	{
		if (!outputs[i])
			continue;
		const TV h = view_of(outputs[i]);
		const int kind = kind_of(outputs[i]);
		if (!h.contiguous || kind < 0)
			return CCV_NNC_EXEC_INVALID;
		if (input_size < 1 || !inputs[0])
		{
			if (kind == 0)
				RC(ew_set_f32(s, outputs[i]->data.f32, h.count, 1.f));
			else
				RC(ew_set_u16(s, (uint16_t*)outputs[i]->data.u8, h.count, kind == 1 ? (uint16_t)0x3f80 : (uint16_t)0x3c00));
		} else if (inputs[0]->data.u8 != outputs[i]->data.u8) {
			const TV g = view_of(inputs[0]);
			if (!g.contiguous || g.count != h.count || kind_of(inputs[0]) != kind)
				return CCV_NNC_EXEC_INVALID;
			if (cudaMemcpyAsync(outputs[i]->data.u8, inputs[0]->data.u8, h.count * kind_size(kind), cudaMemcpyDeviceToDevice, s) != cudaSuccess)
				return CCV_NNC_EXEC_INVALID;
		}
	}
	return CCV_NNC_EXEC_SUCCESS;
}

// broadcasting helper: c's 4-d shape drives the loop; an operand dimension of 1 broadcasts (stride 0)
bool bcast_strides(const TV& c, const TV& x, int xs[4])
{
	int cd[4], cs[4], xd[4], xs0[4];
	if (c.nd > 4 || x.nd > 4)
		return false;
	dims4(c, cd, cs);
	dims4(x, xd, xs0);
	for (int i = 0; i < 4; i++)
	{
		if (xd[i] == cd[i])
			xs[i] = xd[i] == 1 ? 0 : xs0[i];
		else if (xd[i] == 1)
			xs[i] = 0;
		else
			return false;
	}
	return true;
}

// blas/ccv_nnc_add_cpu_ref.c:13-198: c = p * a + q * b, b optional, numpy-style broadcast of a and b into c
int exec_add_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 1 || output_size < 1 || !inputs[0] || !outputs[0] || !is_f32(inputs[0]) || !is_f32(outputs[0]))
		return CCV_NNC_EXEC_INVALID;
	const ccv_nnc_tensor_t* const b_t = input_size > 1 ? inputs[1] : 0;
	const float p = cmd.info.blas.a[0], q = cmd.info.blas.a[1];
	const TV a = view_of(inputs[0]), c = view_of(outputs[0]);
	cudaStream_t s = stream_of(stream_context);
	if (a.contiguous && c.contiguous && same_shape(a, c) && (!b_t || (view_of(b_t).contiguous && same_shape(view_of(b_t), c))))
	{
		RC(ew_axpby_f32(s, p, inputs[0]->data.f32, q, b_t ? b_t->data.f32 : 0, outputs[0]->data.f32, c.count));
		return CCV_NNC_EXEC_SUCCESS;
	}
	int cd[4], cs[4], as[4], bs[4];
	if (c.nd > 4)
		return CCV_NNC_EXEC_INVALID;
	dims4(c, cd, cs);
	if (!bcast_strides(c, a, as) || (b_t && !bcast_strides(c, view_of(b_t), bs)))
		return CCV_NNC_EXEC_INVALID;
	RC(ew_axpby_bcast_f32(s, p, inputs[0]->data.f32, as, q, b_t ? b_t->data.f32 : 0, b_t ? bs : 0, outputs[0]->data.f32, cs, cd));
	return CCV_NNC_EXEC_SUCCESS;
}

// gradient of a broadcast operand: scale * g summed over the broadcast axes
int reduce_to(cudaStream_t s, const float scale, const ccv_nnc_tensor_t* const g_t, ccv_nnc_tensor_t* const out_t)
{
	const TV g = view_of(g_t), o = view_of(out_t);
	if (!o.contiguous || g.nd > 4 || o.nd > 4)
		return 1;
	if (g.contiguous && same_shape(g, o))
		return ew_axpby_f32(s, scale, g_t->data.f32, 0.f, 0, out_t->data.f32, o.count);
	int gd[4], gs[4], od[4], os[4];
	dims4(g, gd, gs);
	dims4(o, od, os);
	for (int i = 0; i < 4; i++)
		if (od[i] != gd[i] && od[i] != 1)
			return 1;
	return reduce_sum_bcast_f32(s, g_t->data.f32, gd, gs, out_t->data.f32, od, scale, 0);
}

// blas/ccv_nnc_add_cpu_ref.c:200-330
int exec_add_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	cudaStream_t s = stream_of(stream_context);
	const float pq[2] = { cmd.info.blas.a[0], cmd.info.blas.a[1] };
	for (int i = 0; i < 2 && i < output_size; i++)
	{
		if (!outputs[i])
			continue;
		if (!is_f32(outputs[i]))
			return CCV_NNC_EXEC_INVALID;
		if (input_size < 1 || !inputs[0])
		{
			const TV o = view_of(outputs[i]);
			if (!o.contiguous)
				return CCV_NNC_EXEC_INVALID;
			RC(ew_set_f32(s, outputs[i]->data.f32, o.count, pq[i]));
		} else
			RC(reduce_to(s, pq[i], inputs[0], outputs[i]));
	}
	return CCV_NNC_EXEC_SUCCESS;
}

// blas/ccv_nnc_mul_cpu_ref.c: MUL c = p * a * b (broadcast); SCALAR_MUL c = p * a
int exec_mul_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 2 || output_size < 1 || !inputs[0] || !inputs[1] || !outputs[0])
		return CCV_NNC_EXEC_INVALID;
	if (!is_f32(inputs[0]) || !is_f32(inputs[1]) || !is_f32(outputs[0]))
		return CCV_NNC_EXEC_INVALID;
	const TV a = view_of(inputs[0]), b = view_of(inputs[1]), c = view_of(outputs[0]);
	int cd[4], cs[4], as[4], bs[4];
	if (c.nd > 4)
		return CCV_NNC_EXEC_INVALID;
	dims4(c, cd, cs);
	if (!bcast_strides(c, a, as) || !bcast_strides(c, b, bs))
		return CCV_NNC_EXEC_INVALID;
	RC(ew_mul_bcast_f32(stream_of(stream_context), cmd.info.blas.a[0], inputs[0]->data.f32, as, inputs[1]->data.f32, bs, outputs[0]->data.f32, cs, cd));
	return CCV_NNC_EXEC_SUCCESS;
}

// blas/ccv_nnc_mul_cpu_ref.c:192-330: d(p a b)/da = p g b, d/db = p g a, each summed over the axes along which that operand was
// broadcast (g == NULL reads as ones).  Same shapes: one fused pass; otherwise the product is formed over the full index space in
// the stream workspace and reduced onto the operand's shape in a fixed order.
int exec_mul_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 3)
		return CCV_NNC_EXEC_INVALID;
	cudaStream_t s = stream_of(stream_context);
	const float p = cmd.info.blas.a[0];
	for (int i = 0; i < 2 && i < output_size; i++)
	{
		if (!outputs[i])
			continue;
		const ccv_nnc_tensor_t* const other = inputs[2 - i]; // ha needs b (inputs[2]), hb needs a (inputs[1])
		if (!other || !is_f32(other) || !is_f32(outputs[i]) || (inputs[0] && !is_f32(inputs[0])))
			return CCV_NNC_EXEC_INVALID;
		const TV o = view_of(outputs[i]), x = view_of(other);
		if (!o.contiguous || o.nd > 4 || x.nd > 4)
			return CCV_NNC_EXEC_INVALID;
		if (x.contiguous && same_shape(o, x) && (!inputs[0] || (view_of(inputs[0]).contiguous && same_shape(view_of(inputs[0]), o))))
		{
			if (!inputs[0])
				RC(ew_axpby_f32(s, p, other->data.f32, 0.f, 0, outputs[i]->data.f32, o.count));
			else {
				int d[4], st[4];
				dims4(o, d, st);
				RC(ew_mul_bcast_f32(s, p, inputs[0]->data.f32, st, other->data.f32, st, outputs[i]->data.f32, st, d));
			}
			continue;
		}
		// the full index space: the gradient's shape, or (no gradient) the broadcast of the two operands
		int fd[4], od[4], os[4], xd[4], xs[4], gd[4] = { 1, 1, 1, 1 }, gs[4] = { 0, 0, 0, 0 };
		dims4(o, od, os);
		dims4(x, xd, xs);
		if (inputs[0])
		{
			const TV g = view_of(inputs[0]);
			if (g.nd > 4)
				return CCV_NNC_EXEC_INVALID;
			dims4(g, gd, gs);
		}
		size_t fcount = 1;
		for (int k = 0; k < 4; k++)
		{
			fd[k] = std::max(std::max(od[k], xd[k]), gd[k]);
			if ((od[k] != fd[k] && od[k] != 1) || (xd[k] != fd[k] && xd[k] != 1) || (gd[k] != fd[k] && gd[k] != 1))
				return CCV_NNC_EXEC_INVALID;
			if (xd[k] == 1)
				xs[k] = 0;
			if (gd[k] == 1)
				gs[k] = 0;
			fcount *= (size_t)fd[k];
		}
		float* const t = (float*)ccv_nnc_stream_context_get_workspace(stream_context, fcount * sizeof(float), CCV_TENSOR_GPU_MEMORY);
		if (!t)
			return CCV_NNC_EXEC_OOM;
		int fs[4];
		for (int k = 3, packed = 1; k >= 0; k--)
			fs[k] = packed, packed *= fd[k];
		if (inputs[0])
			RC(ew_mul_bcast_f32(s, p, inputs[0]->data.f32, gs, other->data.f32, xs, t, fs, fd));
		else
			RC(ew_axpby_bcast_f32(s, p, other->data.f32, xs, 0.f, 0, 0, t, fs, fd));
		RC(reduce_sum_bcast_f32(s, t, fd, fs, outputs[i]->data.f32, od, 1.f, 0));
	}
	return CCV_NNC_EXEC_SUCCESS;
}

int exec_scalar_mul_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 1 || output_size < 1 || !inputs[0] || !outputs[0] || !is_f32(inputs[0]) || !is_f32(outputs[0]))
		return CCV_NNC_EXEC_INVALID;
	const TV a = view_of(inputs[0]), c = view_of(outputs[0]);
	if (!a.contiguous || !c.contiguous || a.count != c.count)
		return CCV_NNC_EXEC_INVALID;
	RC(ew_axpby_f32(stream_of(stream_context), cmd.info.blas.a[0], inputs[0]->data.f32, 0.f, 0, outputs[0]->data.f32, c.count));
	return CCV_NNC_EXEC_SUCCESS;
}

int exec_scalar_mul_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (output_size < 1 || !outputs[0] || !is_f32(outputs[0]))
		return CCV_NNC_EXEC_INVALID;
	const TV h = view_of(outputs[0]);
	if (!h.contiguous)
		return CCV_NNC_EXEC_INVALID;
	cudaStream_t s = stream_of(stream_context);
	if (input_size < 1 || !inputs[0])
		RC(ew_set_f32(s, outputs[0]->data.f32, h.count, cmd.info.blas.a[0]));
	else {
		if (!view_of(inputs[0]).contiguous || view_of(inputs[0]).count != h.count)
			return CCV_NNC_EXEC_INVALID;
		RC(ew_axpby_f32(s, cmd.info.blas.a[0], inputs[0]->data.f32, 0.f, 0, outputs[0]->data.f32, h.count));
	}
	return CCV_NNC_EXEC_SUCCESS;
}

// ================================================================================================ POOLING
bool pool_geom(const ccv_nnc_cmd_t& cmd, const ccv_nnc_hint_t& hint, const TV& a, const TV& b, PoolGeom& g)
{
	if (a.format != CCV_TENSOR_FORMAT_NHWC || b.format != CCV_TENSOR_FORMAT_NHWC)
		return false;
	if ((a.nd != 3 && a.nd != 4) || a.nd != b.nd)
		return false;
	const int ao = a.nd - 3, bo = b.nd - 3;
	memset(&g, 0, sizeof(g));
	g.N = a.nd == 4 ? a.dim[0] : 1;
	if (b.nd == 4 && b.dim[0] != g.N)
		return false;
	g.H = a.dim[ao], g.W = a.dim[ao + 1], g.C = a.dim[ao + 2];
	g.P = b.dim[bo], g.Q = b.dim[bo + 1];
	if (b.dim[bo + 2] != g.C || a.stride[ao + 2] != 1 || b.stride[bo + 2] != 1)
		return false;
	g.an = a.nd == 4 ? a.stride[0] : 0, g.ah = a.stride[ao], g.aw = a.stride[ao + 1];
	g.bn = b.nd == 4 ? b.stride[0] : 0, g.bh = b.stride[bo], g.bw = b.stride[bo + 1];
	g.R = cmd.info.size.dim[0], g.S = cmd.info.size.dim[1];
	g.stride_h = hint.stride.dim[0] > 0 ? hint.stride.dim[0] : 1;
	g.stride_w = hint.stride.dim[1] > 0 ? hint.stride.dim[1] : 1;
	g.pad_h = hint.border.begin[0], g.pad_w = hint.border.begin[1];
	return g.R > 0 && g.S > 0;
}

// pool/ccv_nnc_max_pool_cpu_ref.c:13-59 / pool/ccv_nnc_avg_pool_cpu_ref.c:13-58 (all N images, unlike CPU_REF which
// only walks image 0 -- SURVEY.md 0.6)
template <int IS_MAX>
int exec_pool_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 1 || output_size < 1 || !inputs[0] || !outputs[0] || kind_of(inputs[0]) < 0 || kind_of(outputs[0]) != kind_of(inputs[0]))
		return CCV_NNC_EXEC_INVALID;
	const int kind = kind_of(inputs[0]);
	PoolGeom g;
	if (!pool_geom(cmd, hint, view_of(inputs[0]), view_of(outputs[0]), g))
		return CCV_NNC_EXEC_INVALID;
	if (kind != 0)
		RC(IS_MAX ? pool_max_fwd_16(stream_of(stream_context), kind, g, inputs[0]->data.u8, outputs[0]->data.u8) : pool_avg_fwd_16(stream_of(stream_context), kind, g, inputs[0]->data.u8, outputs[0]->data.u8));
	else if (IS_MAX)
		RC(pool_max_fwd_f32(stream_of(stream_context), g, inputs[0]->data.f32, outputs[0]->data.f32));
	else
		RC(pool_avg_fwd_f32(stream_of(stream_context), g, inputs[0]->data.f32, outputs[0]->data.f32));
	return CCV_NNC_EXEC_SUCCESS;
}

// max: inputs (g, a, b) -> h; avg: inputs (g, ...) -> h
template <int IS_MAX>
int exec_pool_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 1 || output_size < 1 || !inputs[0] || !outputs[0] || kind_of(inputs[0]) < 0 || kind_of(outputs[0]) != kind_of(inputs[0]))
		return CCV_NNC_EXEC_INVALID;
	const int kind = kind_of(inputs[0]);
	PoolGeom g;
	if (!pool_geom(cmd, hint, view_of(outputs[0]), view_of(inputs[0]), g))
		return CCV_NNC_EXEC_INVALID;
	if (IS_MAX)
	{
		if (input_size < 3 || !inputs[1] || !inputs[2])
			return CCV_NNC_EXEC_INVALID;
		const TV a = view_of(inputs[1]), b = view_of(inputs[2]), gv = view_of(inputs[0]), h = view_of(outputs[0]);
		// the kernel addresses a with h's strides and b with g's strides
		if (!same_shape(a, h) || !same_shape(b, gv))
			return CCV_NNC_EXEC_INVALID;
		for (int i = 0; i < a.nd; i++)
			if (a.stride[i] != h.stride[i])
				return CCV_NNC_EXEC_INVALID;
		for (int i = 0; i < b.nd; i++)
			if (b.stride[i] != gv.stride[i])
				return CCV_NNC_EXEC_INVALID;
		if (kind_of(inputs[1]) != kind || kind_of(inputs[2]) != kind)
			return CCV_NNC_EXEC_INVALID;
		if (kind != 0)
			RC(pool_max_bwd_16(stream_of(stream_context), kind, g, inputs[0]->data.u8, inputs[1]->data.u8, inputs[2]->data.u8, outputs[0]->data.u8));
		else
			RC(pool_max_bwd_f32(stream_of(stream_context), g, inputs[0]->data.f32, inputs[1]->data.f32, inputs[2]->data.f32, outputs[0]->data.f32));
	} else if (kind != 0)
		RC(pool_avg_bwd_16(stream_of(stream_context), kind, g, inputs[0]->data.u8, outputs[0]->data.u8));
	else
		RC(pool_avg_bwd_f32(stream_of(stream_context), g, inputs[0]->data.f32, outputs[0]->data.f32));
	return CCV_NNC_EXEC_SUCCESS;
}

// ================================================================================================ SOFTMAX / LOSSES
bool rows_of(const TV& a, int& batch, int& count)
{
	if (!a.contiguous || a.nd < 1)
		return false;
	batch = a.nd < 2 ? 1 : a.dim[0];
	count = (int)(a.count / (size_t)batch);
	return true;
}

int exec_softmax_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 1 || output_size < 1 || !inputs[0] || !outputs[0] || !is_f32(inputs[0]) || !is_f32(outputs[0]))
		return CCV_NNC_EXEC_INVALID;
	int batch, count;
	const TV a = view_of(inputs[0]), b = view_of(outputs[0]);
	if (!rows_of(a, batch, count) || !b.contiguous || !same_shape(a, b))
		return CCV_NNC_EXEC_INVALID;
	RC(softmax_fwd_f32(stream_of(stream_context), inputs[0]->data.f32, outputs[0]->data.f32, batch, count));
	return CCV_NNC_EXEC_SUCCESS;
}

int exec_softmax_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size != 3 || output_size < 1 || !inputs[0] || !inputs[2] || !outputs[0])
		return CCV_NNC_EXEC_INVALID;
	int batch, count;
	const TV g = view_of(inputs[0]), b = view_of(inputs[2]), h = view_of(outputs[0]);
	if (!rows_of(g, batch, count) || !b.contiguous || !h.contiguous || !same_shape(g, b) || !same_shape(g, h))
		return CCV_NNC_EXEC_INVALID;
	RC(softmax_bwd_f32(stream_of(stream_context), inputs[0]->data.f32, inputs[2]->data.f32, outputs[0]->data.f32, batch, count));
	return CCV_NNC_EXEC_SUCCESS;
}

// label tensor -> kind (0 fp32 index, 1 int32 index, 2 fp32 distribution), following the reference's "range" rule
// (loss/ccv_nnc_categorical_crossentropy_cpu_ref.c:27-30)
bool label_kind_of(const ccv_nnc_tensor_t* const b_t, const int batch, int& kind)
{
	const TV b = view_of(b_t);
	if (!b.contiguous)
		return false;
	if (CCV_GET_DATA_TYPE(b_t->info.datatype) == CCV_32S)
	{
		kind = 1;
		return true;
	}
	if (CCV_GET_DATA_TYPE(b_t->info.datatype) != CCV_32F)
		return false;
	int range;
	if (b.nd > 1)
		range = b.dim[b.nd - 1]; // ccv_nnc_tensor_get_c for the 2-d [batch, count] case
	else
		range = batch == 1 ? b.dim[0] : 1;
	kind = range == 1 ? 0 : 2;
	return true;
}

int exec_cce_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size != 2 || output_size < 1 || !inputs[0] || !inputs[1] || !outputs[0])
		return CCV_NNC_EXEC_INVALID;
	int batch, count, kind;
	if (!is_f32(inputs[0]) || !rows_of(view_of(inputs[0]), batch, count) || !label_kind_of(inputs[1], batch, kind) || !view_of(outputs[0]).contiguous)
		return CCV_NNC_EXEC_INVALID;
	RC(cce_fwd_f32(stream_of(stream_context), inputs[0]->data.f32, inputs[1]->data.ptr, kind, outputs[0]->data.f32, batch, count, cmd.info.label_smoothing.trim0, cmd.info.label_smoothing.trim1));
	return CCV_NNC_EXEC_SUCCESS;
}

// inputs (g, a, b) -> h
int exec_cce_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 3 || output_size < 1 || !inputs[1] || !inputs[2] || !outputs[0])
		return CCV_NNC_EXEC_INVALID;
	int batch, count, kind;
	if (!is_f32(inputs[1]) || !rows_of(view_of(inputs[1]), batch, count) || !label_kind_of(inputs[2], batch, kind) || !view_of(outputs[0]).contiguous || !same_shape(view_of(inputs[1]), view_of(outputs[0])))
		return CCV_NNC_EXEC_INVALID;
	RC(cce_bwd_f32(stream_of(stream_context), inputs[0] ? inputs[0]->data.f32 : 0, inputs[1]->data.f32, inputs[2]->data.ptr, kind, outputs[0]->data.f32, batch, count, cmd.info.label_smoothing.trim0, cmd.info.label_smoothing.trim1));
	return CCV_NNC_EXEC_SUCCESS;
}

// softmax_loss/ccv_nnc_softmax_crossentropy_cpu_ref.c:13-170: inputs (a, label) -> outputs (c, d)
int exec_softmax_cce_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size != 2 || output_size != 2 || !inputs[0] || !inputs[1] || !outputs[1])
		return CCV_NNC_EXEC_INVALID;
	int batch, count, kind;
	if (!is_f32(inputs[0]) || !rows_of(view_of(inputs[0]), batch, count) || !label_kind_of(inputs[1], batch, kind) || !view_of(outputs[1]).contiguous || !same_shape(view_of(inputs[0]), view_of(outputs[1])))
		return CCV_NNC_EXEC_INVALID;
	RC(softmax_cce_fwd_f32(stream_of(stream_context), inputs[0]->data.f32, inputs[1]->data.ptr, kind, outputs[0] ? outputs[0]->data.f32 : 0, outputs[1]->data.f32, batch, count, cmd.info.label_smoothing.trim0, cmd.info.label_smoothing.trim1));
	return CCV_NNC_EXEC_SUCCESS;
}

// inputs: [0] = g (may be NULL), [3] = label, [5] = d; outputs[0] = h (:172-181)
int exec_softmax_cce_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size < 6 || output_size < 1 || !inputs[3] || !inputs[5] || !outputs[0])
		return CCV_NNC_EXEC_INVALID;
	int batch, count, kind;
	if (!is_f32(inputs[5]) || !rows_of(view_of(inputs[5]), batch, count) || !label_kind_of(inputs[3], batch, kind) || !view_of(outputs[0]).contiguous || !same_shape(view_of(inputs[5]), view_of(outputs[0])))
		return CCV_NNC_EXEC_INVALID;
	RC(softmax_cce_bwd_f32(stream_of(stream_context), inputs[0] ? inputs[0]->data.f32 : 0, inputs[3]->data.ptr, kind, inputs[5]->data.f32, outputs[0]->data.f32, batch, count, cmd.info.label_smoothing.trim0, cmd.info.label_smoothing.trim1));
	return CCV_NNC_EXEC_SUCCESS;
}

// ================================================================================================ SGD
// sgd/ccv_nnc_sgd_cpu_ref.c:16-126: inputs (g, a, m) -> outputs (b, n)
int exec_sgd_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size != 3 || output_size != 2)
		return CCV_NNC_EXEC_INVALID;
	size_t count = 0;
	// the gradient may be fp32, bf16 or fp16; parameters and momenta are fp32 (the reference's GPU kernel takes the mixed form
	// g 16-bit / a, m fp32 too: sgd/gpu/ccv_nnc_sgd_gpu_ref.cu:71-74)
	for (int i = 0; i < 3; i++)
	{
		if (!inputs[i] || (i == 0 ? kind_of(inputs[i]) < 0 : !is_f32(inputs[i])) || !view_of(inputs[i]).contiguous)
			return CCV_NNC_EXEC_INVALID;
		if (i == 0)
			count = view_of(inputs[0]).count;
		else if (view_of(inputs[i]).count != count)
			return CCV_NNC_EXEC_INVALID;
	}
	for (int i = 0; i < 2; i++)
		if (!outputs[i] || !is_f32(outputs[i]) || !view_of(outputs[i]).contiguous || view_of(outputs[i]).count != count)
			return CCV_NNC_EXEC_INVALID;
	if (cmd.info.sgd.nesterov && cmd.info.sgd.dampening != 0)
		return CCV_NNC_EXEC_INVALID;
	RC(sgd_any(stream_of(stream_context), kind_of(inputs[0]), inputs[0]->data.u8, inputs[1]->data.f32, inputs[2]->data.f32, outputs[0]->data.f32, outputs[1]->data.f32, count, cmd.info.sgd.nesterov, cmd.info.sgd.rate, cmd.info.sgd.scale, cmd.info.sgd.decay, cmd.info.sgd.momentum, cmd.info.sgd.dampening));
	return CCV_NNC_EXEC_SUCCESS;
}

// A run of SGD_FORWARD commands with identical parameters, merged by ccv_nnc_sm100_graph_fuse: inputs = (g, a, m) x T,
// outputs = (b, n) x T.  Every triple is validated exactly as exec_sgd_forw validates one command.
int exec_sgd_multi(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size % 3 != 0 || output_size * 3 != input_size * 2 || input_size == 0)
		return CCV_NNC_EXEC_INVALID;
	if (cmd.info.sgd.nesterov && cmd.info.sgd.dampening != 0)
		return CCV_NNC_EXEC_INVALID;
	const int T = input_size / 3;
	std::vector<const void*> g(T);
	std::vector<const float*> a(T), m(T);
	std::vector<float*> b(T), n(T);
	const int g_kind = inputs[0] ? kind_of(inputs[0]) : -1;
	if (g_kind < 0)
		return CCV_NNC_EXEC_INVALID;
	std::vector<size_t> counts(T);
	for (int t = 0; t < T; t++)
	{
		for (int i = 0; i < 3; i++)
			if (!inputs[3 * t + i] || (i == 0 ? kind_of(inputs[3 * t]) != g_kind : !is_f32(inputs[3 * t + i])) || !view_of(inputs[3 * t + i]).contiguous)
				return CCV_NNC_EXEC_INVALID;
		counts[t] = view_of(inputs[3 * t]).count;
		if (view_of(inputs[3 * t + 1]).count != counts[t] || view_of(inputs[3 * t + 2]).count != counts[t])
			return CCV_NNC_EXEC_INVALID;
		for (int i = 0; i < 2; i++)
			if (!outputs[2 * t + i] || !is_f32(outputs[2 * t + i]) || !view_of(outputs[2 * t + i]).contiguous || view_of(outputs[2 * t + i]).count != counts[t])
				return CCV_NNC_EXEC_INVALID;
		g[t] = inputs[3 * t]->data.u8, a[t] = inputs[3 * t + 1]->data.f32, m[t] = inputs[3 * t + 2]->data.f32;
		b[t] = outputs[2 * t]->data.f32, n[t] = outputs[2 * t + 1]->data.f32;
	}
	RC(sgd_multi_any(stream_of(stream_context), T, g_kind, g.data(), a.data(), m.data(), b.data(), n.data(), counts.data(), cmd.info.sgd.nesterov, cmd.info.sgd.rate, cmd.info.sgd.scale, cmd.info.sgd.decay, cmd.info.sgd.momentum, cmd.info.sgd.dampening));
	return CCV_NNC_EXEC_SUCCESS;
}

int exec_invalid(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	return CCV_NNC_EXEC_INVALID; // e.g. SGD backward (sgd/ccv_nnc_sgd_cpu_ref.c:128-131)
}

// ================================================================================================ SET / MOVES
// util/ccv_nnc_util_cpu_ref.c:637-664
int exec_set_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	cudaStream_t s = stream_of(stream_context);
	const float v = cmd.cmd == CCV_NNC_SET_BACKWARD ? 0.f : cmd.info.blas.a[0];
	for (int i = 0; i < output_size; i++)
	{
		if (!outputs[i])
			continue;
		const TV o = view_of(outputs[i]);
		if (!o.contiguous)
			return CCV_NNC_EXEC_INVALID;
		const int dt = CCV_GET_DATA_TYPE(outputs[i]->info.datatype);
		if (v == 0.f)
		{
			if (cudaMemsetAsync(outputs[i]->data.u8, 0, o.count * dtype_size(dt), s) != cudaSuccess)
				return CCV_NNC_EXEC_INVALID;
		} else if (dt == CCV_32F)
			RC(ew_set_f32(s, outputs[i]->data.f32, o.count, v));
		else if (dt == CCV_32S) {
			const int iv = (int)v;
			float fv;
			memcpy(&fv, &iv, 4);
			RC(ew_set_f32(s, outputs[i]->data.f32, o.count, fv));
		} else if (dt == CCV_64F) {
			// a double is two 32-bit words: fill the word pairs (o.count * 2 words, even / odd word pattern)
			const double dv = (double)v;
			RC(ew_set_u64(s, (uint64_t*)outputs[i]->data.u8, o.count, *(const uint64_t*)&dv));
		} else if (dt == CCV_16F || dt == CCV_16BF)
			RC(ew_set_u16(s, (uint16_t*)outputs[i]->data.u8, o.count, f32_to_16(v, dt == CCV_16BF ? 1 : 2)));
		else
			return CCV_NNC_EXEC_INVALID;
	}
	return CCV_NNC_EXEC_SUCCESS;
}

// copy between two tensors of equal shape and datatype: memcpy when both are packed, strided kernel otherwise
int copy_tensor(cudaStream_t s, const ccv_nnc_tensor_t* const a_t, ccv_nnc_tensor_t* const b_t)
{
	const TV a = view_of(a_t), b = view_of(b_t);
	if (a.datatype != b.datatype || a.count != b.count)
		return 1;
	const size_t es = dtype_size(a.datatype);
	const int a_gpu = CCV_TENSOR_GET_MEMORY(a_t->info.type) == CCV_TENSOR_GPU_MEMORY, b_gpu = CCV_TENSOR_GET_MEMORY(b_t->info.type) == CCV_TENSOR_GPU_MEMORY;
	if (a.contiguous && b.contiguous)
	{
		const cudaMemcpyKind kind = a_gpu ? (b_gpu ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost) : (b_gpu ? cudaMemcpyHostToDevice : cudaMemcpyHostToHost);
		const cudaError_t e = cudaMemcpyAsync(b.p, a.p, a.count * es, kind, s);
		if (e != cudaSuccess)
		{
			set_last_error("cudaMemcpyAsync(data transfer)", e);
			return -1;
		}
		count_launch(0);
		return 0;
	}
	if (!a_gpu || !b_gpu || a.nd > 4 || !same_shape(a, b))
		return 1;
	int ad[4], as[4], bd[4], bs[4];
	dims4(a, ad, as);
	dims4(b, bd, bs);
	return copy_strided(s, a.p, as, b.p, bs, ad, (int)es);
}

// util/ccv_nnc_util_cpu_ref.c:596-617
int exec_data_transfer(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	cudaStream_t s = stream_of(stream_context);
	const int n = input_size < output_size ? input_size : output_size;
	for (int i = 0; i < n; i++)
		if (inputs[i] && outputs[i] && inputs[i] != outputs[i])
			RC(copy_tensor(s, inputs[i], outputs[i]));
	// Without a stream context the reference's transfer is the BLOCKING cudaMemcpy (util/gpu/ccv_nnc_util_gpu_ref.cu:44-60): the
	// caller reads a pinned host tensor right after the call (test/int/nnc/schedule.tests.c:56-59).  The copies above were enqueued
	// on the default stream; wait for them.
	if (!stream_context && cudaStreamSynchronize(s) != cudaSuccess)
		return CCV_NNC_EXEC_INVALID;
	return CCV_NNC_EXEC_SUCCESS;
}

// util/ccv_nnc_util_cpu_ref.c:996-1082: same format = copy; NHWC <-> NCHW = copy over permuted strides
int exec_format_transform(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	cudaStream_t s = stream_of(stream_context);
	for (int i = 0; i < output_size && i < input_size; i++)
	{
		if (!inputs[i] || !outputs[i])
			continue;
		const TV a = view_of(inputs[i]), b = view_of(outputs[i]);
		if (a.dim[0] == 0 || b.dim[0] == 0)
			continue;
		if (a.format == b.format)
		{
			RC(copy_tensor(s, inputs[i], outputs[i]));
			continue;
		}
		if (a.nd == b.nd && a.nd < 3)
		{
			// a vector / matrix tagged with another format (the bias gradient of an NCHW convolution, test/int/nnc/cudnn.tests.c:455-471): plain copy
			RC(copy_tensor(s, inputs[i], outputs[i]));
			continue;
		}
		if (a.datatype != b.datatype || a.nd != b.nd || (a.nd != 3 && a.nd != 4))
			return CCV_NNC_EXEC_INVALID;
		// express both in (n, c, h, w) index order
		int d[4], as[4], bs[4];
		const int o = a.nd - 3;
		auto nchw_of = [&](const TV& t, int dim[4], int st[4]) -> bool {
			dim[0] = t.nd == 4 ? t.dim[0] : 1, st[0] = t.nd == 4 ? t.stride[0] : 0;
			if (t.format == CCV_TENSOR_FORMAT_NHWC)
				dim[1] = t.dim[o + 2], st[1] = t.stride[o + 2], dim[2] = t.dim[o], st[2] = t.stride[o], dim[3] = t.dim[o + 1], st[3] = t.stride[o + 1];
			else if (t.format == CCV_TENSOR_FORMAT_NCHW)
				dim[1] = t.dim[o], st[1] = t.stride[o], dim[2] = t.dim[o + 1], st[2] = t.stride[o + 1], dim[3] = t.dim[o + 2], st[3] = t.stride[o + 2];
			else
				return false;
			return true;
		};
		int bd[4];
		if (!nchw_of(a, d, as) || !nchw_of(b, bd, bs))
			return CCV_NNC_EXEC_INVALID;
		for (int k = 0; k < 4; k++)
			if (d[k] != bd[k])
				return CCV_NNC_EXEC_INVALID;
		RC(copy_strided(s, a.p, as, b.p, bs, d, (int)dtype_size(a.datatype)));
	}
	return CCV_NNC_EXEC_SUCCESS;
}

// util/ccv_nnc_util_cpu_ref.c:1102-1180: swap two axes
int exec_transpose(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	cudaStream_t s = stream_of(stream_context);
	for (int i = 0; i < output_size && i < input_size; i++)
	{
		if (!inputs[i] || !outputs[i])
			continue;
		const TV a = view_of(inputs[i]), b = view_of(outputs[i]);
		if (a.nd != b.nd || a.nd > 4 || a.datatype != b.datatype)
			return CCV_NNC_EXEC_INVALID;
		const int ax0 = cmd.info.transpose.axis[0], ax1 = cmd.info.transpose.axis[1];
		if (ax0 < 0 || ax1 < 0 || ax0 >= a.nd || ax1 >= a.nd)
			return CCV_NNC_EXEC_INVALID;
		int d[4], as[4], bs[4];
		const int off = 4 - a.nd;
		for (int k = 0; k < 4; k++)
		{
			if (k < off)
			{
				d[k] = 1, as[k] = bs[k] = 0;
				continue;
			}
			const int bk = k - off; // index in b
			const int ak = bk == ax0 ? ax1 : (bk == ax1 ? ax0 : bk);
			if (b.dim[bk] != a.dim[ak])
				return CCV_NNC_EXEC_INVALID;
			d[k] = b.dim[bk], bs[k] = b.stride[bk], as[k] = a.stride[ak];
		}
		RC(copy_strided(s, a.p, as, b.p, bs, d, (int)dtype_size(a.datatype)));
	}
	return CCV_NNC_EXEC_SUCCESS;
}

// util/ccv_nnc_util_cpu_ref.c:1200-1260
int exec_datatype_conversion(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	cudaStream_t s = stream_of(stream_context);
	for (int i = 0; i < output_size && i < input_size; i++)
	{
		if (!inputs[i] || !outputs[i])
			continue;
		const TV a = view_of(inputs[i]), b = view_of(outputs[i]);
		if (a.count != b.count)
			return CCV_NNC_EXEC_INVALID;
		if (a.datatype == b.datatype)
		{
			RC(copy_tensor(s, inputs[i], outputs[i]));
			continue;
		}
		if (!a.contiguous || !b.contiguous || dtype_code(a.datatype) < 0 || dtype_code(b.datatype) < 0)
			return CCV_NNC_EXEC_INVALID;
		RC(convert_dtype(s, a.p, dtype_code(a.datatype), b.p, dtype_code(b.datatype), a.count));
	}
	return CCV_NNC_EXEC_SUCCESS;
}

// ================================================================================================ 16-bit tensors on fp32-only commands
// The commands below have fp32 kernels only; the reference's GPU backends register them for CCV_16F as well (e.g.
// softmax/gpu/ccv_nnc_softmax_gpu_cudnn.cu, blas/gpu/ccv_nnc_add_gpu_cudnn.cu) and its half-precision tests run them
// (test/int/nnc/cudnn.tests.c:3504-3678, 4151-4323, 4363-4735).  For bf16 / fp16 tensors the command runs in its functional form:
// every 16-bit operand is widened into the stream workspace, the fp32 command runs on shadow tensors, every 16-bit result is
// rounded once (to nearest even) on the way back.  One workspace request [inner | staging], as in conv_staged.
inline uint16_t f32_to_16(const float v, const int kind)
{
	uint32_t u;
	memcpy(&u, &v, 4);
	if (kind == 1)
		return (uint16_t)((u + 0x7fffu + ((u >> 16) & 1u)) >> 16); // bf16, round to nearest even
	// fp16, round to nearest even (finite range; the fill values this is used for are small)
	const uint32_t sign = (u >> 16) & 0x8000u;
	const int32_t e = (int32_t)((u >> 23) & 0xff) - 127 + 15;
	uint32_t m = u & 0x7fffffu;
	if (e >= 31)
		return (uint16_t)(sign | 0x7c00u);
	if (e <= 0)
	{
		if (e < -10)
			return (uint16_t)sign;
		m |= 0x800000u;
		const int shift = 14 - e;
		const uint32_t r = m >> shift, rem = m & ((1u << shift) - 1), half = 1u << (shift - 1);
		return (uint16_t)(sign | (r + (rem > half || (rem == half && (r & 1)))));
	}
	const uint32_t r = (uint32_t)(e << 10) | (m >> 13), rem = m & 0x1fffu;
	return (uint16_t)(sign | (r + (rem > 0x1000u || (rem == 0x1000u && (r & 1)))));
}

int via_f32(const ccv_nnc_cmd_exec_f F32, const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	enum { MAXT = 16 };
	bool any16 = false;
	for (int i = 0; i < input_size; i++)
		any16 = any16 || (inputs[i] && kind_of(inputs[i]) > 0);
	for (int i = 0; i < output_size; i++)
		any16 = any16 || (outputs[i] && kind_of(outputs[i]) > 0);
	if (!any16)
		return F32(cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
	if (input_size > MAXT || output_size > MAXT)
		return CCV_NNC_EXEC_INVALID;
	struct Shadow { ccv_nnc_tensor_t t; ccv_nnc_tensor_t* orig; size_t n; int kind; int is_out; } sh[2 * MAXT];
	ccv_nnc_tensor_t* in[MAXT];
	ccv_nnc_tensor_t* out[MAXT];
	int n = 0;
	size_t staging = 0;
	const auto shadow_of = [&](ccv_nnc_tensor_t* const t, const int is_out) -> ccv_nnc_tensor_t* {
		if (!t || kind_of(t) <= 0)
			return t;
		for (int j = 0; j < n; j++)
			if (sh[j].orig == t || sh[j].orig->data.u8 == t->data.u8)
			{
				sh[j].is_out |= is_out;
				return &sh[j].t;
			}
		const TV v = view_of(t);
		if (!v.contiguous || v.count > 0x7fffffffull)
			return 0;
		Shadow& x = sh[n++];
		memcpy(&x.t, t, sizeof(ccv_nnc_tensor_t));
		x.t.type &= ~CCV_TENSOR_VIEW;
		x.t.info.datatype = CCV_32F;
		x.orig = t, x.n = v.count, x.kind = kind_of(t), x.is_out = is_out;
		staging += (v.count * sizeof(float) + 255) & ~(size_t)255;
		return &x.t;
	};
	for (int i = 0; i < input_size; i++)
		if (!(in[i] = shadow_of(inputs[i], 0)) && inputs[i])
			return CCV_NNC_EXEC_INVALID;
	for (int i = 0; i < output_size; i++)
		if (!(out[i] = shadow_of(outputs[i], 1)) && outputs[i])
			return CCV_NNC_EXEC_INVALID;
	// what the fp32 command itself may ask the workspace for: partial rows, or (MUL backward with broadcasting) one temporary of
	// the full index space, which is the size of its largest operand
	size_t largest = 0;
	for (int j = 0; j < n; j++)
		largest = std::max(largest, (sh[j].n * sizeof(float) + 255) & ~(size_t)255);
	const size_t inner = ((size_t)4 << 20) + largest;
	unsigned char* const ws = (unsigned char*)ccv_nnc_stream_context_get_workspace(stream_context, inner + staging, CCV_TENSOR_GPU_MEMORY);
	if (!ws)
		return CCV_NNC_EXEC_OOM;
	cudaStream_t s = stream_of(stream_context);
	unsigned char* p = ws + inner;
	for (int j = 0; j < n; j++)
	{
		sh[j].t.data.u8 = p, p += (sh[j].n * sizeof(float) + 255) & ~(size_t)255;
		// every shadow is filled: inputs carry data, and an output may be read by the command (in-place forms)
		RC(widen_matrix(s, sh[j].orig->data.u8, sh[j].kind, (long long)sh[j].n, 1, sh[j].t.data.f32, 1, (int)sh[j].n));
	}
	const int rc = F32(cmd, hint, flags, in, input_size, out, output_size, stream_context);
	if (rc != CCV_NNC_EXEC_SUCCESS)
		return rc;
	if (ccv_nnc_stream_context_get_workspace(stream_context, 1, CCV_TENSOR_GPU_MEMORY) != (void*)ws)
	{
		set_last_error("functional 16-bit form: the fp32 command moved the workspace under the widened tensors", cudaErrorInvalidValue);
		return CCV_NNC_EXEC_INVALID;
	}
	for (int j = 0; j < n; j++)
		if (sh[j].is_out)
			RC(narrow_matrix(s, sh[j].t.data.f32, sh[j].orig->data.u8, sh[j].kind, (long long)sh[j].n, 1, 1, (int)sh[j].n, 0));
	return CCV_NNC_EXEC_SUCCESS;
}
template <ccv_nnc_cmd_exec_f F32>
int exec_via_f32(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	return via_f32(F32, cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

// SGD: fp32 parameters / momenta with gradients of any type run natively (the mixed-precision form); 16-bit PARAMETERS
// (sgd/gpu/ccv_nnc_sgd_gpu_ref.cu:75-77, test/int/nnc/sgd.tests.c:73-137) go through the functional form
int exec_sgd_any(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size >= 2 && inputs[1] && kind_of(inputs[1]) > 0)
		return exec_via_f32<exec_sgd_forw>(cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
	return exec_sgd_forw(cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

// pooling on NCHW tensors ([N,] C, H, W: pool/gpu/ccv_nnc_max_pool_gpu_cudnn.cu takes both formats; test/int/nnc/cudnn.tests.c:2772-2870):
// the kernels are NHWC (channel-contiguous 16-byte accesses), NCHW operands are staged like the convolution's
size_t pool_staged_inner(const ccv_nnc_cmd_t&, const ccv_nnc_hint_t&, ccv_nnc_tensor_t* const*, int, ccv_nnc_tensor_t* const*, int) { return 256; }
template <ccv_nnc_cmd_exec_f F>
int exec_pool_any(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (any_nchw(inputs, input_size, outputs, output_size))
		return nchw_staged(F, pool_staged_inner, 0, cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
	return F(cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

void fill(ccv_nnc_cmd_backend_registry_t* const registry, const int formats, const int datatypes, const int algorithms, const ccv_nnc_cmd_exec_f exec)
{
	registry->tensor_formats = formats;
	registry->tensor_datatypes = datatypes;
	registry->tensor_memory = CCV_TENSOR_GPU_MEMORY;
	registry->algorithms = algorithms;
	registry->exec = exec;
	registry->autotune = 0;
	registry->aux = 0;
}

const int ALL_FORMATS = CCV_TENSOR_FORMAT_NCHW | CCV_TENSOR_FORMAT_NHWC | CCV_TENSOR_FORMAT_CHWN;

// registry->autotune of the contraction commands (lib/nnc/ccv_nnc.h:323; called by ccv_nnc_cmd_autotune, ccv_nnc_cmd.c:519-531, on
// scratch copies of the operands): every algorithm of this backend that accepts the shapes is timed on the device (CUDA
// events on the caller's stream, best of 3 after a warm-up) and the index of the fastest one is returned.  The generic
// fallback of the reference times the asynchronous *enqueue* with a host clock (ccv_nnc_cmd.c:549-555), which says nothing
// about a GPU kernel -- hence a real autotune function.
template <ccv_nnc_cmd_exec_f EXEC>
int autotune_contraction(const ccv_nnc_cmd_t cmd, const size_t max_workspace_size, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	cudaStream_t s = stream_of(stream_context);
	cudaEvent_t e0, e1;
	if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess)
		return 0;
	int best = 0;
	float best_ms = -1.f;
	const int candidates[3] = { CCV_NNC_SM100_ALGO_TF32, CCV_NNC_SM100_ALGO_3XTF32, CCV_NNC_SM100_ALGO_FFMA };
	for (int k = 0; k < 3; k++)
	{
		ccv_nnc_cmd_t c = cmd;
		c.algorithm = candidates[k];
		if (EXEC(c, hint, flags, inputs, input_size, outputs, output_size, stream_context) != CCV_NNC_EXEC_SUCCESS) // warm-up + applicability
			continue;
		float ms = -1.f;
		for (int rep = 0; rep < 3; rep++)
		{
			cudaEventRecord(e0, s);
			EXEC(c, hint, flags, inputs, input_size, outputs, output_size, stream_context);
			cudaEventRecord(e1, s);
			float t = 0.f;
			if (cudaEventSynchronize(e1) != cudaSuccess || cudaEventElapsedTime(&t, e0, e1) != cudaSuccess)
				continue;
			if (ms < 0.f || t < ms)
				ms = t;
		}
		if (ms >= 0.f && (best_ms < 0.f || ms < best_ms))
			best_ms = ms, best = candidates[k];
	}
	cudaEventDestroy(e0);
	cudaEventDestroy(e1);
	return best;
}

} // namespace

namespace sm100 {
int backend_gemm_nt_bias(void* stream_context, int kind, int M, int N, int K, const void* a, const void* w, void* c, const void* bias, int bias_is_f32)
{
	ccv_nnc_stream_context_t* const ctx = (ccv_nnc_stream_context_t*)stream_context;
	const Scratch scratch = scratch_of(ctx);
	cudaStream_t s = stream_of(ctx);
	if (kind == 0)
		return gemm_dispatch(s, scratch, CCV_NNC_SM100_ALGO_3XTF32, M, N, K, (const float*)a, K, 1, (const float*)w, 1, K, (float*)c, N, 1, (const float*)bias, 0);
	return gemm_dispatch16(s, scratch, kind, M, N, K, a, K, 1, w, 1, K, c, N, 1, bias && bias_is_f32 ? (const float*)bias : 0, bias && !bias_is_f32 ? bias : 0, 0);
}
} // namespace sm100

// implemented in sm100_backend_ext.cu (attention, layer / rms norm, upsample, allreduce)
extern "C" {
int ccv_nnc_sm100_exec_sdpa_forw(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_exec_sdpa_back(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_exec_lnorm_forw(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_exec_lnorm_back(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_exec_rmsnorm_forw(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_exec_rmsnorm_back(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_exec_upsample_forw(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_exec_upsample_back(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_exec_gnorm_forw(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_exec_gnorm_back(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_exec_allreduce(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
}

// ================================================================================================ fused pairs
// Used by the flat graph runner's peephole pass (ccv_nnc_sm100_graph_fuse): each stands for two adjacent reference
// commands and produces what the pair would have produced.
extern "C" int ccv_nnc_sm100_fused_bn_relu_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	return bnorm_forw(1, cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

// BATCH_NORM_FORWARD with the statistics tensor of its producing convolution as a 6th input (no ReLU)
extern "C" int ccv_nnc_sm100_fused_bn_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	return bnorm_forw(0, cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

// BATCH_NORM_BACKWARD with the bias gradient of the producing convolution as a 4th output (no ReLU in front)
extern "C" int ccv_nnc_sm100_fused_bn_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	return bnorm_back(0, cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

extern "C" int ccv_nnc_sm100_fused_relu_bn_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	return bnorm_back(1, cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

// inputs (a, b) -> y = relu(a + b)
extern "C" int ccv_nnc_sm100_fused_add_relu_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size != 2 || output_size != 1 || !inputs[0] || !inputs[1] || !outputs[0])
		return CCV_NNC_EXEC_INVALID;
	const TV a = view_of(inputs[0]), b = view_of(inputs[1]), y = view_of(outputs[0]);
	const int kind = kind_of(outputs[0]);
	if (!a.contiguous || !b.contiguous || !y.contiguous || a.count != y.count || b.count != y.count || kind < 0 || kind_of(inputs[0]) != kind || kind_of(inputs[1]) != kind)
		return CCV_NNC_EXEC_INVALID;
	if (kind != 0)
		RC(ew_add_relu_fwd_16(stream_of(stream_context), kind, inputs[0]->data.u8, inputs[1]->data.u8, outputs[0]->data.u8, y.count));
	else
		RC(ew_add_relu_fwd_f32(stream_of(stream_context), inputs[0]->data.f32, inputs[1]->data.f32, outputs[0]->data.f32, y.count));
	return CCV_NNC_EXEC_SUCCESS;
}

// inputs (a, b, y) -> out = y > 0 ? a + b : 0   (EWSUM of two branch gradients followed by RELU_BACKWARD)
extern "C" int ccv_nnc_sm100_fused_add_relu_back(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size != 3 || output_size != 1 || !inputs[0] || !inputs[1] || !inputs[2] || !outputs[0])
		return CCV_NNC_EXEC_INVALID;
	const TV a = view_of(inputs[0]), b = view_of(inputs[1]), y = view_of(inputs[2]), o = view_of(outputs[0]);
	const int kind = kind_of(outputs[0]);
	if (!a.contiguous || !b.contiguous || !y.contiguous || !o.contiguous || a.count != o.count || b.count != o.count || y.count != o.count || kind < 0 || kind_of(inputs[0]) != kind || kind_of(inputs[1]) != kind || kind_of(inputs[2]) != kind)
		return CCV_NNC_EXEC_INVALID;
	if (kind != 0)
		RC(ew_add_relu_bwd_16(stream_of(stream_context), kind, inputs[0]->data.u8, inputs[1]->data.u8, inputs[2]->data.u8, outputs[0]->data.u8, o.count));
	else
		RC(ew_add_relu_bwd_f32(stream_of(stream_context), inputs[0]->data.f32, inputs[1]->data.f32, inputs[2]->data.f32, outputs[0]->data.f32, o.count));
	return CCV_NNC_EXEC_SUCCESS;
}

// The end of a residual block with the batch norm of the main branch folded in (rewrite (h)): inputs (x, shortcut, coef) ->
// out = relu(x * a + b + shortcut), where coef ([2, C] fp32) holds the a, b a statistics-only BATCH_NORM_FORWARD just wrote.
// NHWC: the channel is the innermost dimension.  Bit-identical to BATCH_NORM_FORWARD, EWSUM, RELU_FORWARD.
extern "C" int ccv_nnc_sm100_fused_bn_add_relu_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size != 3 || output_size != 1 || !inputs[0] || !inputs[1] || !inputs[2] || !outputs[0])
		return CCV_NNC_EXEC_INVALID;
	const TV x = view_of(inputs[0]), r = view_of(inputs[1]), c = view_of(inputs[2]), y = view_of(outputs[0]);
	const int kind = kind_of(outputs[0]);
	if (!x.contiguous || !r.contiguous || !y.contiguous || !c.contiguous || !is_f32(inputs[2]) || x.count != y.count || r.count != y.count || kind < 0 || kind_of(inputs[0]) != kind || kind_of(inputs[1]) != kind || x.nd < 1)
		return CCV_NNC_EXEC_INVALID;
	const int C = x.dim[x.nd - 1];
	if (C <= 0 || c.count != 2 * (size_t)C)
		return CCV_NNC_EXEC_INVALID;
	if (kind != 0)
		RC(bn_add_relu_fwd_16(stream_of(stream_context), kind, inputs[0]->data.u8, inputs[1]->data.u8, outputs[0]->data.u8, inputs[2]->data.f32, x.count / C, C));
	else
		RC(bn_add_relu_fwd_f32(stream_of(stream_context), inputs[0]->data.f32, inputs[1]->data.f32, outputs[0]->data.f32, inputs[2]->data.f32, x.count / C, C));
	return CCV_NNC_EXEC_SUCCESS;
}

// The add + ReLU backward of a residual block end (b = NULL: a plain RELU_BACKWARD) carrying the reduction of the batch-norm
// backward behind it (rewrite (i)): inputs (a, b, y, x, saved_mean) -> outputs (g, part); g = y > 0 ? a + b : 0 and part
// ([rows, 2C] fp32) receives the per-block partial sums of g and g * (x - mean), their number in its `sig` field (0 when the layout
// takes the plain path; the batch norm then reduces g itself).  x / mean are that batch norm's input and saved mean, NHWC.
extern "C" int ccv_nnc_sm100_fused_add_relu_back_stats(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (input_size != 5 || output_size != 2 || !inputs[0] || !inputs[2] || !inputs[3] || !inputs[4] || !outputs[0] || !outputs[1])
		return CCV_NNC_EXEC_INVALID;
	ccv_nnc_tensor_t* const part_t = outputs[1];
	part_t->sig = 0;
	const TV a = view_of(inputs[0]), y = view_of(inputs[2]), x = view_of(inputs[3]), m = view_of(inputs[4]), o = view_of(outputs[0]);
	const int kind = kind_of(outputs[0]);
	if (!a.contiguous || !y.contiguous || !x.contiguous || !o.contiguous || a.count != o.count || y.count != o.count || x.count != o.count || kind < 0 || kind_of(inputs[0]) != kind || kind_of(inputs[2]) != kind || kind_of(inputs[3]) != kind)
		return CCV_NNC_EXEC_INVALID;
	if (inputs[1] && (!view_of(inputs[1]).contiguous || view_of(inputs[1]).count != o.count || kind_of(inputs[1]) != kind))
		return CCV_NNC_EXEC_INVALID;
	if (!is_f32(inputs[4]) || !is_f32(part_t) || x.nd < 1)
		return CCV_NNC_EXEC_INVALID;
	// the reduction is only done for the batch norm's NHWC layout: one statistic per innermost element, a [rows, 2C] partial tensor
	const int C = x.dim[x.nd - 1];
	const int cap = C > 0 && m.count == (size_t)C && part_t->info.dim[1] == 2 * C ? part_t->info.dim[0] : 0;
	int rows = 0;
	if (kind != 0)
		RC(bn_add_relu_bwd_reduce_16(stream_of(stream_context), kind, inputs[0]->data.u8, inputs[1] ? inputs[1]->data.u8 : 0, inputs[2]->data.u8, inputs[3]->data.u8, inputs[4]->data.f32, outputs[0]->data.u8, o.count / (cap ? C : 1), cap ? C : 1, cap ? part_t->data.f32 : 0, cap, &rows));
	else
		RC(bn_add_relu_bwd_reduce_f32(stream_of(stream_context), inputs[0]->data.f32, inputs[1] ? inputs[1]->data.f32 : 0, inputs[2]->data.f32, inputs[3]->data.f32, inputs[4]->data.f32, outputs[0]->data.f32, o.count / (cap ? C : 1), cap ? C : 1, cap ? part_t->data.f32 : 0, cap, &rows));
	part_t->sig = (uint64_t)rows;
	return CCV_NNC_EXEC_SUCCESS;
}

// CONVOLUTION_FORWARD whose output feeds a training BATCH_NORM_FORWARD: outputs[1] is the statistics tensor
// ([4 planes x rows, K] fp32: count, shift, shifted sum, shifted sum of squares per (CTA, warp quarter) row) shared with the
// batch-norm node; the tensor-core epilogue folds its output into it and the number of rows in use lands in the `sig` field
// (0 when the launch took a path without that epilogue).
extern "C" int ccv_nnc_sm100_fused_conv_stats_forw(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (output_size != 2 || !outputs[1])
		return CCV_NNC_EXEC_INVALID;
	ccv_nnc_tensor_t* const stats_t = outputs[1];
	int rows = 0;
	const int max_rows = stats_t->info.dim[0] / 4;
	if (outputs[0] && stats_t->info.dim[1] == cmd.info.convolution.count)
		conv_stats_request(stats_t->data.f32, max_rows, &rows);
	const int rc = exec_conv_forw(cmd, hint, flags, inputs, input_size, outputs, 1, stream_context);
	conv_stats_request(0, 0, 0); // never leave a request pending for an unrelated launch
	stats_t->sig = rc == CCV_NNC_EXEC_SUCCESS ? (uint64_t)rows : 0;
	return rc;
}

// T SGD_FORWARD commands with identical parameters as one command: inputs (g, a, m) x T -> outputs (b, n) x T
extern "C" int ccv_nnc_sm100_fused_sgd_multi(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	return exec_sgd_multi(cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

// ================================================================================================ registration
namespace sm100 {
int exec_via_f32_rt(ccv_nnc_cmd_exec_f f32, const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	return via_f32(f32, cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
}
}

#define REGISTER_SM100(cmd) extern "C" void _register_command_ ## cmd ## _backend_CCV_NNC_BACKEND_GPU_SM100(ccv_nnc_cmd_backend_registry_t* const registry)

REGISTER_SM100(CCV_NNC_GEMM_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, CCV_NNC_SM100_ALGO_COUNT, exec_gemm_nd4<exec_gemm_forw>); registry->autotune = autotune_contraction<exec_gemm_nd4<exec_gemm_forw> >; }
REGISTER_SM100(CCV_NNC_GEMM_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, CCV_NNC_SM100_ALGO_COUNT, exec_gemm_nd4<exec_gemm_back>); registry->autotune = autotune_contraction<exec_gemm_nd4<exec_gemm_back> >; }
REGISTER_SM100(CCV_NNC_CONVOLUTION_FORWARD) { fill(registry, CCV_TENSOR_FORMAT_NHWC | CCV_TENSOR_FORMAT_NCHW, CCV_32F | CCV_16F | CCV_16BF, CCV_NNC_SM100_ALGO_COUNT, exec_conv_forw); registry->autotune = autotune_contraction<exec_conv_forw>; }
REGISTER_SM100(CCV_NNC_CONVOLUTION_BACKWARD) { fill(registry, CCV_TENSOR_FORMAT_NHWC | CCV_TENSOR_FORMAT_NCHW, CCV_32F | CCV_16F | CCV_16BF, CCV_NNC_SM100_ALGO_COUNT, exec_conv_back); registry->autotune = autotune_contraction<exec_conv_back>; }
REGISTER_SM100(CCV_NNC_SCALED_DOT_PRODUCT_ATTENTION_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, ccv_nnc_sm100_exec_sdpa_forw); }
REGISTER_SM100(CCV_NNC_SCALED_DOT_PRODUCT_ATTENTION_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, ccv_nnc_sm100_exec_sdpa_back); }
REGISTER_SM100(CCV_NNC_SOFTMAX_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_via_f32<exec_softmax_forw>); }
REGISTER_SM100(CCV_NNC_SOFTMAX_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_via_f32<exec_softmax_back>); }
REGISTER_SM100(CCV_NNC_BATCH_NORM_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_bnorm_forw); }
REGISTER_SM100(CCV_NNC_BATCH_NORM_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_bnorm_back); }
REGISTER_SM100(CCV_NNC_LAYER_NORM_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F, 1, ccv_nnc_sm100_exec_lnorm_forw); }
REGISTER_SM100(CCV_NNC_LAYER_NORM_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F, 1, ccv_nnc_sm100_exec_lnorm_back); }
REGISTER_SM100(CCV_NNC_GROUP_NORM_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F, 1, ccv_nnc_sm100_exec_gnorm_forw); }
REGISTER_SM100(CCV_NNC_GROUP_NORM_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F, 1, ccv_nnc_sm100_exec_gnorm_back); }
REGISTER_SM100(CCV_NNC_RMSNORM_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F, 1, ccv_nnc_sm100_exec_rmsnorm_forw); }
REGISTER_SM100(CCV_NNC_RMSNORM_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F, 1, ccv_nnc_sm100_exec_rmsnorm_back); }
REGISTER_SM100(CCV_NNC_EWSUM_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF | CCV_32S, 1, exec_ewsum_forw); }
REGISTER_SM100(CCV_NNC_EWSUM_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_ewsum_back); }
REGISTER_SM100(CCV_NNC_ADD_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_via_f32<exec_add_forw>); }
REGISTER_SM100(CCV_NNC_ADD_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_via_f32<exec_add_back>); }
REGISTER_SM100(CCV_NNC_MUL_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_via_f32<exec_mul_forw>); }
REGISTER_SM100(CCV_NNC_MUL_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_via_f32<exec_mul_back>); }
REGISTER_SM100(CCV_NNC_SCALAR_MUL_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_via_f32<exec_scalar_mul_forw>); }
REGISTER_SM100(CCV_NNC_SCALAR_MUL_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_via_f32<exec_scalar_mul_back>); }
REGISTER_SM100(CCV_NNC_RELU_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_relu_forw); }
REGISTER_SM100(CCV_NNC_RELU_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_relu_back); }
REGISTER_SM100(CCV_NNC_MAX_POOL_FORWARD) { fill(registry, CCV_TENSOR_FORMAT_NHWC | CCV_TENSOR_FORMAT_NCHW, CCV_32F | CCV_16F | CCV_16BF, 1, exec_pool_any<exec_pool_forw<1> >); }
REGISTER_SM100(CCV_NNC_MAX_POOL_BACKWARD) { fill(registry, CCV_TENSOR_FORMAT_NHWC | CCV_TENSOR_FORMAT_NCHW, CCV_32F | CCV_16F | CCV_16BF, 1, exec_pool_any<exec_pool_back<1> >); }
REGISTER_SM100(CCV_NNC_AVERAGE_POOL_FORWARD) { fill(registry, CCV_TENSOR_FORMAT_NHWC | CCV_TENSOR_FORMAT_NCHW, CCV_32F | CCV_16F | CCV_16BF, 1, exec_pool_any<exec_pool_forw<0> >); }
REGISTER_SM100(CCV_NNC_AVERAGE_POOL_BACKWARD) { fill(registry, CCV_TENSOR_FORMAT_NHWC | CCV_TENSOR_FORMAT_NCHW, CCV_32F | CCV_16F | CCV_16BF, 1, exec_pool_any<exec_pool_back<0> >); }
REGISTER_SM100(CCV_NNC_UPSAMPLE_FORWARD) { fill(registry, CCV_TENSOR_FORMAT_NHWC | CCV_TENSOR_FORMAT_NCHW, CCV_32F | CCV_16F | CCV_16BF, 1, exec_via_f32<ccv_nnc_sm100_exec_upsample_forw>); }
REGISTER_SM100(CCV_NNC_UPSAMPLE_BACKWARD) { fill(registry, CCV_TENSOR_FORMAT_NHWC | CCV_TENSOR_FORMAT_NCHW, CCV_32F | CCV_16F | CCV_16BF, 1, exec_via_f32<ccv_nnc_sm100_exec_upsample_back>); }
REGISTER_SM100(CCV_NNC_SET_FORWARD) { fill(registry, ALL_FORMATS, CCV_64F | CCV_32F | CCV_16F | CCV_16BF | CCV_32S, 1, exec_set_forw); }
REGISTER_SM100(CCV_NNC_SET_BACKWARD) { fill(registry, ALL_FORMATS, CCV_64F | CCV_32F | CCV_16F | CCV_16BF | CCV_32S, 1, exec_set_forw); }
REGISTER_SM100(CCV_NNC_DATA_TRANSFER_FORWARD) { fill(registry, ALL_FORMATS, CCV_64F | CCV_32F | CCV_16F | CCV_16BF | CCV_32S | CCV_8U, 1, exec_data_transfer); registry->tensor_memory = CCV_TENSOR_CPU_MEMORY | CCV_TENSOR_GPU_MEMORY; }
REGISTER_SM100(CCV_NNC_DATA_TRANSFER_BACKWARD) { fill(registry, ALL_FORMATS, CCV_64F | CCV_32F | CCV_16F | CCV_16BF | CCV_32S | CCV_8U, 1, exec_data_transfer); registry->tensor_memory = CCV_TENSOR_CPU_MEMORY | CCV_TENSOR_GPU_MEMORY; }
REGISTER_SM100(CCV_NNC_FORMAT_TRANSFORM_FORWARD) { fill(registry, ALL_FORMATS, CCV_64F | CCV_32F | CCV_32S | CCV_16F | CCV_16BF | CCV_8U, 1, exec_format_transform); }
REGISTER_SM100(CCV_NNC_FORMAT_TRANSFORM_BACKWARD) { fill(registry, ALL_FORMATS, CCV_64F | CCV_32F | CCV_32S | CCV_16F | CCV_16BF | CCV_8U, 1, exec_format_transform); }
REGISTER_SM100(CCV_NNC_TRANSPOSE_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_transpose); }
REGISTER_SM100(CCV_NNC_TRANSPOSE_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_transpose); }
REGISTER_SM100(CCV_NNC_DATATYPE_CONVERSION_FORWARD) { fill(registry, ALL_FORMATS, CCV_64F | CCV_32F | CCV_16F | CCV_16BF, 1, exec_datatype_conversion); }
REGISTER_SM100(CCV_NNC_DATATYPE_CONVERSION_BACKWARD) { fill(registry, ALL_FORMATS, CCV_64F | CCV_32F | CCV_16F | CCV_16BF, 1, exec_datatype_conversion); }
REGISTER_SM100(CCV_NNC_SGD_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, exec_sgd_any); }
REGISTER_SM100(CCV_NNC_SGD_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F, 1, exec_invalid); }
REGISTER_SM100(CCV_NNC_CATEGORICAL_CROSSENTROPY_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF | CCV_32S, 1, exec_via_f32<exec_cce_forw>); }
REGISTER_SM100(CCV_NNC_CATEGORICAL_CROSSENTROPY_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF | CCV_32S, 1, exec_via_f32<exec_cce_back>); }
REGISTER_SM100(CCV_NNC_SOFTMAX_CROSSENTROPY_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF | CCV_32S, 1, exec_via_f32<exec_softmax_cce_forw>); }
REGISTER_SM100(CCV_NNC_SOFTMAX_CROSSENTROPY_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF | CCV_32S, 1, exec_via_f32<exec_softmax_cce_back>); }
REGISTER_SM100(CCV_NNC_COMM_ALLREDUCE_FORWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, ccv_nnc_sm100_exec_allreduce); }
REGISTER_SM100(CCV_NNC_COMM_ALLREDUCE_BACKWARD) { fill(registry, ALL_FORMATS, CCV_32F | CCV_16F | CCV_16BF, 1, ccv_nnc_sm100_exec_allreduce); }
