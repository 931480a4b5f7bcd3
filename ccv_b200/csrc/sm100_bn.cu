// sm100_bn.cu -- batch normalisation (training / inference forward, backward), optionally fused with the ReLU that
// follows it in a ResNet block, and the two fused residual-add kernels.  All HBM-bound: every pass streams each tensor
// once with 128-bit accesses and several independent loads in flight per thread.
//
// Semantics: norm/ccv_nnc_batch_norm_cpu_ref.c:16-250 (forward), :312-470 (backward); relu/ccv_nnc_relu_cpu_ref.c:13-55;
// ew/ccv_nnc_ew_cpu_ref.c:15-110 (paths relative to /root/reference/lib/nnc/cmd).  Statistics are biased; running =
// momentum * running + (1 - momentum) * batch.  Layout [outer, C, inner] (NHWC: inner = 1).
//
// Workspace (bn_workspace_bytes): double s[2C] (cross-block sums) followed by float coef[4C] (per-channel a, b, p, q).
#include "sm100_ew.h"
#include "sm100_contract.h"
#include "sm100_elem.cuh"

namespace sm100 {

static int g_sms_bn = 0;
static int sms()
{
	if (!g_sms_bn)
	{
		int dev = 0;
		cudaGetDevice(&dev);
		cudaDeviceGetAttribute(&g_sms_bn, cudaDevAttrMultiProcessorCount, dev);
		if (g_sms_bn <= 0)
			g_sms_bn = 148;
	}
	return g_sms_bn;
}
static int check(const char* what)
{
	count_launch();
	const cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess)
	{
		set_last_error(what, e);
		return -1;
	}
	return 0;
}
static int grid_for(size_t work_items, int threads, int max_waves = 8)
{
	size_t blocks = (work_items + threads - 1) / threads;
	const size_t cap = (size_t)sms() * max_waves;
	if (blocks > cap)
		blocks = cap;
	return blocks < 1 ? 1 : (int)blocks;
}

// workspace: double s[2C] (reduced sums), float coef[4C] (per-channel a, b, p, q), float part[gy_max][2C] (per-block partial sums)
static inline size_t bn_part_rows() { return (size_t)sms() * 4 + 8; }
size_t bn_workspace_bytes(int C) { return (size_t)C * (2 * sizeof(double) + 4 * sizeof(float)) + bn_part_rows() * 2 * (size_t)C * sizeof(float) + 256; }
static inline double* ws_sums(void* ws) { return (double*)ws; }
static inline float* ws_coef(void* ws, int C) { return (float*)((double*)ws + 2 * (size_t)C); }
static inline float* ws_part(void* ws, int C) { return (float*)(((uintptr_t)(ws_coef(ws, C) + 4 * (size_t)C) + 255) & ~(uintptr_t)255); }


// ------------------------------------------------------------------------------------------------ reductions
// NHWC: thread = (column-vector tx, row-lane ty); each thread walks rows with 4 independent 128-bit loads in flight.
// MODE 0: s1 = sum(x - k), s2 = sum((x - k)^2), k = x[0, c] (shift keeps the one-pass variance well conditioned).
// MODE 1: s1 = sum(g'), s2 = sum(g' * (x - mean)); g' = g, or g masked by relu(x * a + b) > 0 when MASK.
// MODE 2: MODE 1 on g' = ym > 0 ? ga + gb : 0 (gb may be NULL: ym > 0 ? ga : 0), which is also stored to gout -- the residual
//         block end's add + ReLU backward feeding the batch-norm reduction behind it.  The row walk and the in-block combine are
//         those of MODE 1, so the partial rows are bit-identical to storing g' first and reducing it with MODE 1.
template <typename T, int MODE, int MASK>
__global__ void __launch_bounds__(256) bn_reduce_kernel(const T* __restrict__ x, const T* __restrict__ g, const float* __restrict__ mean, const float* __restrict__ coef, const size_t rows, const int C, float* __restrict__ part, const int cpb,
	const T* __restrict__ ga = 0, const T* __restrict__ gb = 0, const T* __restrict__ ym = 0, T* __restrict__ gout = 0)
{
	// one 16-byte access = W channels (4 fp32 / 8 bf16 or fp16); thread = (channel group tx, row lane ty)
	constexpr int W = Vec16<T>::W;
	__shared__ float sh[2][256][W + 1];
	const int CW = C / W;
	const int tx = threadIdx.x % cpb, ty = threadIdx.x / cpb, rpi = 256 / cpb;
	const int cw = blockIdx.x * cpb + tx;
	float s1[W], s2[W];
#pragma unroll
	for (int k = 0; k < W; k++)
		s1[k] = s2[k] = 0.f;
	if (ty < rpi && cw < CW)
	{
		float kk[W], a[W], b[W];
		if (MODE == 0)
			ldv(x + cw * W, kk);
		else {
#pragma unroll
			for (int k = 0; k < W; k++)
				kk[k] = mean[cw * W + k];
		}
#pragma unroll
		for (int k = 0; k < W; k++)
			a[k] = MASK ? coef[cw * W + k] : 0.f, b[k] = MASK ? coef[C + cw * W + k] : 0.f;
		const size_t step = (size_t)gridDim.y * rpi;
		size_t r = (size_t)blockIdx.y * rpi + ty;
		auto acc = [&](const float (&xv)[W], const float (&gv)[W]) {
#pragma unroll
			for (int k = 0; k < W; k++)
			{
				if (MODE == 0)
				{
					const float d = xv[k] - kk[k];
					s1[k] += d, s2[k] += d * d;
				} else {
					float m = gv[k];
					if (MASK)
						m = fmaf(xv[k], a[k], b[k]) > 0.f ? m : 0.f;
					s1[k] += m, s2[k] += m * (xv[k] - kk[k]);
				}
			}
		};
		// MODE 2: g' of one row from the two branch gradients and the block output, rounded to T as a store would round it
		auto grad = [&](const size_t off, float (&gv)[W]) {
			float u[W], v[W], m[W];
			ldv(ga + off, u), ldv(ym + off, m);
			if (gb)
				ldv(gb + off, v);
#pragma unroll
			for (int k = 0; k < W; k++)
				gv[k] = rnd<T>(m[k] > 0.f ? (gb ? u[k] + v[k] : u[k]) : 0.f);
			stv(gout + off, gv);
		};
		for (; r + 3 * step < rows; r += 4 * step)
		{
			float xv[4][W], gv[4][W];
#pragma unroll
			for (int u = 0; u < 4; u++)
			{
				ldv(x + (r + u * step) * C + cw * W, xv[u]);
				if (MODE == 1)
					ldv(g + (r + u * step) * C + cw * W, gv[u]);
				else if (MODE == 2)
					grad((r + u * step) * C + cw * W, gv[u]);
			}
#pragma unroll
			for (int u = 0; u < 4; u++)
				acc(xv[u], MODE >= 1 ? gv[u] : xv[u]);
		}
		for (; r < rows; r += step)
		{
			float xv[W], gv[W];
			ldv(x + r * C + cw * W, xv);
			if (MODE == 1)
				ldv(g + r * C + cw * W, gv);
			else if (MODE == 2)
				grad(r * C + cw * W, gv);
			acc(xv, MODE >= 1 ? gv : xv);
		}
	}
#pragma unroll
	for (int k = 0; k < W; k++)
		sh[0][threadIdx.x][k] = s1[k], sh[1][threadIdx.x][k] = s2[k];
	__syncthreads();
	if (ty == 0 && cw < CW)
	{
		for (int t = 1; t < rpi; t++)
#pragma unroll
			for (int k = 0; k < W; k++)
				s1[k] += sh[0][t * cpb + tx][k], s2[k] += sh[1][t * cpb + tx][k];
		// per-block partial sums; bn_finalize_partials_kernel adds the gridDim.y rows in a fixed order (no atomics: 600 same-address
		// fp64 atomics per channel cost ~15 us per launch, profiles/r01_ncu_bn_reduce_apply.txt, and made the result run-dependent)
		float* const row = part + (size_t)blockIdx.y * 2 * C;
#pragma unroll
		for (int k = 0; k < W; k++)
			row[cw * W + k] = s1[k], row[C + cw * W + k] = s2[k];
	}
}

// any layout [outer, C, inner], scalar: one block per channel (NCHW, or C not a multiple of 4)
template <typename T, int MODE, int MASK>
__global__ void bn_reduce_generic_kernel(const T* __restrict__ x, const T* __restrict__ g, const float* __restrict__ mean, const float* __restrict__ coef, const size_t outer, const int C, const size_t inner, double* __restrict__ ws)
{
	__shared__ float sh[2][32];
	const int c = blockIdx.x;
	const float k = MODE == 0 ? ldf(x + (size_t)c * inner) : mean[c];
	const float a = MASK ? coef[c] : 0.f, b = MASK ? coef[C + c] : 0.f;
	float s1 = 0.f, s2 = 0.f;
	const size_t total = outer * inner;
	for (size_t i = threadIdx.x; i < total; i += blockDim.x)
	{
		const size_t o = i / inner, in = i - o * inner;
		const size_t idx = (o * C + c) * inner + in;
		const float xv = ldf(x + idx);
		if (MODE == 0)
		{
			const float d = xv - k;
			s1 += d, s2 += d * d;
		} else {
			float gv = ldf(g + idx);
			if (MASK)
				gv = fmaf(xv, a, b) > 0.f ? gv : 0.f;
			s1 += gv, s2 += gv * (xv - k);
		}
	}
	for (int o = 16; o > 0; o >>= 1)
		s1 += __shfl_xor_sync(0xffffffff, s1, o), s2 += __shfl_xor_sync(0xffffffff, s2, o);
	if ((threadIdx.x & 31) == 0)
		sh[0][threadIdx.x >> 5] = s1, sh[1][threadIdx.x >> 5] = s2;
	__syncthreads();
	if (threadIdx.x < 32)
	{
		const int nw = blockDim.x >> 5;
		s1 = threadIdx.x < nw ? sh[0][threadIdx.x] : 0.f, s2 = threadIdx.x < nw ? sh[1][threadIdx.x] : 0.f;
		for (int o = 16; o > 0; o >>= 1)
			s1 += __shfl_xor_sync(0xffffffff, s1, o), s2 += __shfl_xor_sync(0xffffffff, s2, o);
		if (threadIdx.x == 0)
			ws[c] = (double)s1, ws[C + c] = (double)s2;
	}
}

// per-channel forward affine, shared by forward and (for the ReLU mask) backward so that both see identical bits
__device__ __forceinline__ void bn_affine(const float scale, const float bias, const float mean, const float inv_std, float& a, float& b)
{
	a = scale * inv_std;
	b = bias - mean * a;
}

template <typename T>
__global__ void bn_fwd_finalize_kernel(const T* __restrict__ x, const size_t shift_stride, const double* __restrict__ ws, const int C, const double count, const float epsilon, const float momentum, const float* __restrict__ scale, const float* __restrict__ bias, float* __restrict__ running_mean, float* __restrict__ running_var, float* __restrict__ saved_mean, float* __restrict__ saved_inv_std, float* __restrict__ coef)
{
	const int c = blockIdx.x * blockDim.x + threadIdx.x;
	if (c >= C)
		return;
	const double k = (double)ldf(x + (size_t)c * shift_stride);
	const double s1 = ws[c], s2 = ws[C + c];
	const double mean = k + s1 / count;
	double var = (s2 - s1 * s1 / count) / count;
	if (var < 0)
		var = 0;
	const float meanf = (float)mean, varf = (float)var;
	const float inv_std = 1.f / sqrtf(varf + epsilon);
	saved_mean[c] = meanf;
	saved_inv_std[c] = inv_std;
	running_mean[c] = momentum * running_mean[c] + (1.f - momentum) * meanf;
	running_var[c] = momentum * running_var[c] + (1.f - momentum) * varf;
	float a, b;
	bn_affine(scale[c], bias[c], meanf, inv_std, a, b);
	coef[c] = a, coef[C + c] = b;
}
// inference: inv_std = 1 / (sqrt(var) + eps)  (batch_norm_cpu_ref.c:262-279)
__global__ void bn_test_coef_kernel(const int C, const float epsilon, const float* __restrict__ scale, const float* __restrict__ bias, const float* __restrict__ mean, const float* __restrict__ var, float* __restrict__ coef)
{
	const int c = blockIdx.x * blockDim.x + threadIdx.x;
	if (c >= C)
		return;
	const float a = scale[c] / (sqrtf(var[c]) + epsilon);
	coef[c] = a, coef[C + c] = bias[c] - mean[c] * a;
}
// backward coefficients: with a = scale * inv_std, dx = a * g' + p * x + q,
//   p = -a * inv_std * dscale / count,  q = -a * dbias / count - p * mean      (same algebra as batch_norm_cpu_ref.c:430-466)
__global__ void bn_bwd_finalize_kernel(const double* __restrict__ ws, const int C, const float count, const float* __restrict__ scale, const float* __restrict__ mean, const float* __restrict__ inv_std, float* __restrict__ dscale, float* __restrict__ dbias, float* __restrict__ coef)
{
	const int c = blockIdx.x * blockDim.x + threadIdx.x;
	if (c >= C)
		return;
	const float db = (float)ws[c];
	const float ds = (float)ws[C + c] * inv_std[c];
	if (dbias)
		dbias[c] = db;
	if (dscale)
		dscale[c] = ds;
	const float a = scale[c] * inv_std[c];
	const float p = -a * inv_std[c] * ds / count;
	coef[2 * C + c] = p;
	coef[3 * C + c] = -a * db / count - p * mean[c];
}
__global__ void bn_mask_coef_kernel(const int C, const float* __restrict__ scale, const float* __restrict__ bias, const float* __restrict__ mean, const float* __restrict__ inv_std, float* __restrict__ coef)
{
	const int c = blockIdx.x * blockDim.x + threadIdx.x;
	if (c >= C)
		return;
	float a, b;
	bn_affine(scale[c], bias[c], mean[c], inv_std[c], a, b);
	coef[c] = a, coef[C + c] = b;
}

// The same finalisation fed directly from the per-block partial rows of bn_reduce_kernel (one launch instead of partials-reduce +
// finalize): 32 channels x 32 row-lanes per block; row-lane 0 of each channel finishes the statistics.
// MODE 0 forward, MODE 1 backward; WITH_A (backward without a fused ReLU): also writes a = scale * inv_std for the apply pass.
template <typename T, int MODE, int WITH_A>
__global__ void __launch_bounds__(1024) bn_finalize_partials_kernel(const float* __restrict__ part, const int gy, const T* __restrict__ x, const int C, const double count, const float epsilon, const float momentum,
	const float* __restrict__ scale, const float* __restrict__ bias, float* __restrict__ running_mean, float* __restrict__ running_var, float* __restrict__ saved_mean, float* __restrict__ saved_inv_std,
	float* __restrict__ dscale, float* __restrict__ dbias, float* __restrict__ coef)
{
	__shared__ double sh[2][32][33];
	const int cx = threadIdx.x & 31, yl = threadIdx.x >> 5;
	const int c = blockIdx.x * 32 + cx;
	double a1 = 0, a2 = 0;
	if (c < C)
		for (int y = yl; y < gy; y += 32)
		{
			const float* const row = part + (size_t)y * 2 * C;
			a1 += (double)row[c], a2 += (double)row[C + c];
		}
	sh[0][yl][cx] = a1, sh[1][yl][cx] = a2;
	__syncthreads();
	if (yl != 0 || c >= C)
		return;
	double s1 = 0, s2 = 0;
#pragma unroll
	for (int j = 0; j < 32; j++)
		s1 += sh[0][j][cx], s2 += sh[1][j][cx];
	if (MODE == 0)
	{
		const double k = (double)ldf(x + c);
		const double mean = k + s1 / count;
		double var = (s2 - s1 * s1 / count) / count;
		if (var < 0)
			var = 0;
		const float meanf = (float)mean, varf = (float)var;
		const float inv_std = 1.f / sqrtf(varf + epsilon);
		saved_mean[c] = meanf;
		saved_inv_std[c] = inv_std;
		running_mean[c] = momentum * running_mean[c] + (1.f - momentum) * meanf;
		running_var[c] = momentum * running_var[c] + (1.f - momentum) * varf;
		float a, b;
		bn_affine(scale[c], bias[c], meanf, inv_std, a, b);
		coef[c] = a, coef[C + c] = b;
	} else {
		const float cnt = (float)count;
		const float inv_std = saved_inv_std[c];
		const float db = (float)s1;
		const float ds = (float)s2 * inv_std;
		if (dbias)
			dbias[c] = db;
		if (dscale)
			dscale[c] = ds;
		const float a = scale[c] * inv_std;
		const float pp = -a * inv_std * ds / cnt;
		if (WITH_A)
			coef[c] = a;
		coef[2 * C + c] = pp;
		coef[3 * C + c] = -a * db / cnt - pp * saved_mean[c];
	}
}

// Forward finalisation from the statistics a convolution epilogue produced (sm100_umma_persistent.cuh): four planes [rows][C] --
// count n_i, shift k_i, s1_i = sum(v - k_i), s2_i = sum((v - k_i)^2) -- one row per (CTA, epilogue warp quarter); rows with
// count 0 were never touched.  Each slot is its own shifted one-pass estimate.  They are combined in double precision, in a
// fixed order (32 row-lanes per channel, then lane by lane), in two sweeps over the (L2-resident) slots:
//   mean = sum_i (n_i k_i + s1_i) / N
//   M2   = sum_i [ s2_i - 2 d_i s1_i + n_i d_i^2 ],  d_i = mean - k_i        (= sum over the slot of (v - mean)^2, exactly)
// Both are plain sums (no serial dependency, several loads in flight), deterministic, and free of the E[v^2] - E[v]^2
// cancellation however far the channel mean is from zero, because every d_i is of the order of one standard deviation
// (norm/ccv_nnc_batch_norm_cpu_ref.c:66-110 is the two-pass form this has to agree with).
__global__ void __launch_bounds__(1024) bn_finalize_ext_kernel(const float* __restrict__ part, const int rows, const int C, const float epsilon, const float momentum,
	const float* __restrict__ scale, const float* __restrict__ bias, float* __restrict__ running_mean, float* __restrict__ running_var, float* __restrict__ saved_mean, float* __restrict__ saved_inv_std, float* __restrict__ coef)
{
	__shared__ double sh[2][32][33];
	__shared__ double sh_mean[32];
	const int cx = threadIdx.x & 31, yl = threadIdx.x >> 5;
	const int c = blockIdx.x * 32 + cx;
	const size_t plane = (size_t)rows * C;
	const float* const p0 = part + c;
	double a0 = 0, a1 = 0, n0 = 0, n1 = 0;
	if (c < C)
	{
		int y = yl;
		for (; y + 32 < rows; y += 64)
		{
			const size_t u = (size_t)y * C, v = (size_t)(y + 32) * C;
			const float nu = p0[u], nv = p0[v], ku = p0[plane + u], kv = p0[plane + v], su = p0[2 * plane + u], sv = p0[2 * plane + v];
			n0 += (double)nu, n1 += (double)nv;
			// untouched slots (count 0) hold whatever the buffer held: never let them into the sums
			a0 += nu > 0.f ? (double)nu * (double)ku + (double)su : 0.0, a1 += nv > 0.f ? (double)nv * (double)kv + (double)sv : 0.0;
		}
		for (; y < rows; y += 32)
		{
			const size_t u = (size_t)y * C;
			const float nu = p0[u];
			n0 += (double)nu;
			a0 += nu > 0.f ? (double)nu * (double)p0[plane + u] + (double)p0[2 * plane + u] : 0.0;
		}
	}
	sh[0][yl][cx] = n0 + n1, sh[1][yl][cx] = a0 + a1;
	__syncthreads();
	if (yl == 0)
	{
		double n = 0, a = 0;
#pragma unroll
		for (int j = 0; j < 32; j++)
			n += sh[0][j][cx], a += sh[1][j][cx];
		sh_mean[cx] = n > 0 ? a / n : 0.0;
		sh[0][0][cx] = n; // total count, read back after the second sweep
	}
	__syncthreads();
	const double mean = sh_mean[cx];
	const double total = sh[0][0][cx];
	__syncthreads();
	double m0 = 0, m1 = 0;
	if (c < C)
	{
		int y = yl;
		for (; y + 32 < rows; y += 64)
		{
			const size_t u = (size_t)y * C, v = (size_t)(y + 32) * C;
			const float nu = p0[u], nv = p0[v];
			if (nu > 0.f)
			{
				const double d = mean - (double)p0[plane + u];
				m0 += (double)p0[3 * plane + u] - 2.0 * d * (double)p0[2 * plane + u] + (double)nu * d * d;
			}
			if (nv > 0.f)
			{
				const double d = mean - (double)p0[plane + v];
				m1 += (double)p0[3 * plane + v] - 2.0 * d * (double)p0[2 * plane + v] + (double)nv * d * d;
			}
		}
		for (; y < rows; y += 32)
		{
			const size_t u = (size_t)y * C;
			const float nu = p0[u];
			if (nu > 0.f)
			{
				const double d = mean - (double)p0[plane + u];
				m0 += (double)p0[3 * plane + u] - 2.0 * d * (double)p0[2 * plane + u] + (double)nu * d * d;
			}
		}
	}
	sh[1][yl][cx] = m0 + m1;
	__syncthreads();
	if (yl != 0 || c >= C)
		return;
	double m2 = 0;
#pragma unroll
	for (int j = 0; j < 32; j++)
		m2 += sh[1][j][cx];
	if (m2 < 0)
		m2 = 0;
	const float meanf = (float)mean, varf = total > 0 ? (float)(m2 / total) : 0.f;
	const float inv_std = 1.f / sqrtf(varf + epsilon);
	saved_mean[c] = meanf;
	saved_inv_std[c] = inv_std;
	running_mean[c] = momentum * running_mean[c] + (1.f - momentum) * meanf;
	running_var[c] = momentum * running_var[c] + (1.f - momentum) * varf;
	float a, b;
	bn_affine(scale[c], bias[c], meanf, inv_std, a, b);
	coef[c] = a, coef[C + c] = b;
}

// ------------------------------------------------------------------------------------------------ elementwise passes
// forward: y = x * a + b (optionally relu'd).  backward: dx = a * g' + p * x + q with the optional relu mask on g.
// COLSUM (backward only): also leaves per-channel sums of the values written in `part` (rows of C floats; the caller guarantees
// stride % CV == 0, so a thread stays on one channel group, and 256 % CV == 0 or CV % 256 == 0) -- the bias gradient of the
// convolution that consumes dx, without another pass over dx.
template <typename T, int BWD, int RELU, int COLSUM>
__global__ void __launch_bounds__(256) bn_apply_vec_kernel(const T* __restrict__ x, const T* __restrict__ g, T* __restrict__ out, const float* __restrict__ coef, const size_t total4, const int C, float* __restrict__ part)
{
	const int CV = C >> 2;
	const size_t stride = (size_t)gridDim.x * blockDim.x;
	float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
	for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total4; i += 2 * stride)
	{
		const size_t j = i + stride;
		const bool two = j < total4;
		const float4 x0 = ld4(x + i * 4), x1 = two ? ld4(x + j * 4) : x0;
		float4 g0 = x0, g1 = x0;
		if (BWD)
			g0 = ld4(g + i * 4), g1 = two ? ld4(g + j * 4) : g0;
#pragma unroll
		for (int u = 0; u < 2; u++)
		{
			if (u == 1 && !two)
				break;
			const size_t e = u ? j : i;
			const float4 xv = u ? x1 : x0, gv = u ? g1 : g0;
			const int c0 = (int)(e % CV) * 4;
			const float4 a = ld4(coef + c0), b = ld4(coef + C + c0);
			float4 o;
			if (!BWD)
			{
				o.x = fmaf(xv.x, a.x, b.x), o.y = fmaf(xv.y, a.y, b.y), o.z = fmaf(xv.z, a.z, b.z), o.w = fmaf(xv.w, a.w, b.w);
				if (RELU)
					o.x = fmaxf(o.x, 0.f), o.y = fmaxf(o.y, 0.f), o.z = fmaxf(o.z, 0.f), o.w = fmaxf(o.w, 0.f);
			} else {
				const float4 p = ld4(coef + 2 * C + c0), q = ld4(coef + 3 * C + c0);
				float h0 = gv.x, h1 = gv.y, h2 = gv.z, h3 = gv.w;
				if (RELU)
				{
					h0 = fmaf(xv.x, a.x, b.x) > 0.f ? h0 : 0.f, h1 = fmaf(xv.y, a.y, b.y) > 0.f ? h1 : 0.f;
					h2 = fmaf(xv.z, a.z, b.z) > 0.f ? h2 : 0.f, h3 = fmaf(xv.w, a.w, b.w) > 0.f ? h3 : 0.f;
				}
				o.x = fmaf(a.x, h0, fmaf(p.x, xv.x, q.x)), o.y = fmaf(a.y, h1, fmaf(p.y, xv.y, q.y));
				o.z = fmaf(a.z, h2, fmaf(p.z, xv.z, q.z)), o.w = fmaf(a.w, h3, fmaf(p.w, xv.w, q.w));
			}
			st4(out + e * 4, o);
			if (COLSUM)
				cs.x += o.x, cs.y += o.y, cs.z += o.z, cs.w += o.w;
		}
	}
	if (COLSUM)
	{
		if (CV < 256)
		{
			// 256 / CV threads of this block share a channel group (256 % CV == 0): one partial row per block
			__shared__ float4 sh[256];
			sh[threadIdx.x] = cs;
			__syncthreads();
			if ((int)threadIdx.x < CV)
			{
				for (int k = threadIdx.x + CV; k < 256; k += CV)
				{
					const float4 v = sh[k];
					cs.x += v.x, cs.y += v.y, cs.z += v.z, cs.w += v.w;
				}
				st4(part + ((size_t)blockIdx.x * CV + threadIdx.x) * 4, cs);
			}
		} else // CV % 256 == 0: every thread of the grid owns (row, channel group) = divmod(global thread id, CV)
			st4(part + (blockIdx.x * (size_t)blockDim.x + threadIdx.x) * 4, cs);
	}
}
// The same pass for the common case in which the grid stride is a multiple of the channel groups per pixel (every power-of-two
// channel count): a thread then stays on ONE channel group for the whole tensor, so its a / b / p / q coefficients are loaded once
// into registers instead of on every iteration (they were 4 of the 6 loads per element group: the pass was L1 / issue bound at
// 0.5 of the HBM rate, worse for 16-bit data), every access is 16 bytes (4 fp32 or 8 bf16 / fp16 elements) and four row loads
// are in flight per thread.  COLSUM as above.
// RES (forward, no RELU): g is a residual operand and out = relu(roundT(x * a + b) + g) -- the batch norm at the end of a residual
// block, the shortcut add and the ReLU in one pass, rounded as the batch norm's own store would round before the add.
template <typename T, int BWD, int RELU, int COLSUM, int RES = 0>
__global__ void __launch_bounds__(256) bn_apply_fixed_kernel(const T* __restrict__ x, const T* __restrict__ g, T* __restrict__ out, const float* __restrict__ coef, const size_t totalw, const int C, float* __restrict__ part)
{
	constexpr int W = Vec16<T>::W;
	const int CW = C / W;
	const size_t stride = (size_t)gridDim.x * blockDim.x; // a multiple of CW (launcher)
	const size_t i0 = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	const int c0 = (int)(i0 % CW) * W;
	float a[W], b[W], p[W], q[W], cs[W];
#pragma unroll
	for (int k = 0; k < W; k++)
	{
		a[k] = coef[c0 + k], b[k] = coef[C + c0 + k];
		p[k] = BWD ? coef[2 * C + c0 + k] : 0.f, q[k] = BWD ? coef[3 * C + c0 + k] : 0.f;
		cs[k] = 0.f;
	}
	for (size_t i = i0; i < totalw; i += 4 * stride)
	{
		float xv[4][W], gv[4][W];
#pragma unroll
		for (int u = 0; u < 4; u++)
			if (i + u * stride < totalw)
			{
				ldv(x + (i + u * stride) * W, xv[u]);
				if (BWD || RES)
					ldv(g + (i + u * stride) * W, gv[u]);
			}
#pragma unroll
		for (int u = 0; u < 4; u++)
			if (i + u * stride < totalw)
			{
				float o[W];
#pragma unroll
				for (int k = 0; k < W; k++)
				{
					if (RES)
						o[k] = fmaxf(rnd<T>(fmaf(xv[u][k], a[k], b[k])) + gv[u][k], 0.f);
					else if (!BWD)
					{
						o[k] = fmaf(xv[u][k], a[k], b[k]);
						if (RELU)
							o[k] = fmaxf(o[k], 0.f);
					} else {
						float h = gv[u][k];
						if (RELU)
							h = fmaf(xv[u][k], a[k], b[k]) > 0.f ? h : 0.f;
						o[k] = fmaf(a[k], h, fmaf(p[k], xv[u][k], q[k]));
					}
					if (COLSUM)
						cs[k] += o[k];
				}
				stv(out + (i + u * stride) * W, o);
			}
	}
	if (COLSUM)
	{
		if (CW < 256)
		{
			// 256 / CW threads of this block share a channel group (256 % CW == 0): one partial row per block
			__shared__ float sh[256][W + 1];
#pragma unroll
			for (int k = 0; k < W; k++)
				sh[threadIdx.x][k] = cs[k];
			__syncthreads();
			if ((int)threadIdx.x < CW)
			{
				for (int t = threadIdx.x + CW; t < 256; t += CW)
#pragma unroll
					for (int k = 0; k < W; k++)
						cs[k] += sh[t][k];
#pragma unroll
				for (int k = 0; k < W; k++)
					part[((size_t)blockIdx.x * CW + threadIdx.x) * W + k] = cs[k];
			}
		} else { // CW % 256 == 0: every thread of the grid owns (row, channel group) = divmod(global thread id, CW)
#pragma unroll
			for (int k = 0; k < W; k++)
				part[i0 * W + k] = cs[k];
		}
	}
}
// out[c] = sum over rows of part[row][c] in a fixed order: 32 columns x 32 row-lanes per block
__global__ void __launch_bounds__(1024) bn_colsum_rows_kernel(const float* __restrict__ part, const int rows, const int C, void* __restrict__ out, const int out_kind)
{
	__shared__ float sh[32][33];
	const int cx = threadIdx.x & 31, yl = threadIdx.x >> 5;
	const int c = blockIdx.x * 32 + cx;
	float acc = 0.f;
	if (c < C)
	{
		int y = yl;
		for (; y + 96 < rows; y += 128)
			acc += (part[(size_t)y * C + c] + part[(size_t)(y + 32) * C + c]) + (part[(size_t)(y + 64) * C + c] + part[(size_t)(y + 96) * C + c]);
		for (; y < rows; y += 32)
			acc += part[(size_t)y * C + c];
	}
	sh[yl][cx] = acc;
	__syncthreads();
	if (yl == 0 && c < C)
	{
		float t = 0.f;
#pragma unroll
		for (int j = 0; j < 32; j++)
			t += sh[j][cx];
		st_kind(out, c, t, out_kind);
	}
}
template <typename T, int BWD, int RELU, int RES = 0>
__global__ void bn_apply_generic_kernel(const T* __restrict__ x, const T* __restrict__ g, T* __restrict__ out, const float* __restrict__ coef, const size_t total, const int C, const size_t inner)
{
	for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
	{
		const int c = (int)((i / inner) % C);
		const float a = coef[c], b = coef[C + c], xv = ldf(x + i);
		if (RES)
			stf(out + i, fmaxf(rnd<T>(fmaf(xv, a, b)) + ldf(g + i), 0.f));
		else if (!BWD)
		{
			const float o = fmaf(xv, a, b);
			stf(out + i, RELU ? fmaxf(o, 0.f) : o);
		} else {
			float h = ldf(g + i);
			if (RELU)
				h = fmaf(xv, a, b) > 0.f ? h : 0.f;
			stf(out + i, fmaf(a, h, fmaf(coef[2 * C + c], xv, coef[3 * C + c])));
		}
	}
}

static void reduce_config(size_t rows, int CV, int& cpb, dim3& grid)
{
	cpb = CV >= 256 ? 256 : CV;
	const int rpi = 256 / cpb;
	const int gx = (CV + cpb - 1) / cpb;
	size_t gy = (rows + (size_t)rpi * 32 - 1) / ((size_t)rpi * 32);
	const size_t cap = (size_t)(sms() * 4 + gx - 1) / gx;
	if (gy > cap)
		gy = cap;
	if (gy < 1)
		gy = 1;
	grid = dim3(gx, (unsigned)gy);
}

template <typename T, int MODE, int MASK>
static int run_reduce(cudaStream_t s, const T* x, const T* g, const float* mean, const float* coef, size_t outer, int C, size_t inner, double* ws, float* part, int* part_rows)
{
	// NHWC vector path: leaves *part_rows > 0 rows of per-block partial sums in `part` (finished by bn_finalize_partials_kernel);
	// generic path: one block per channel writes the sums to ws directly (*part_rows = 0)
	constexpr int W = Vec16<T>::W;
	if (inner == 1 && C % W == 0 && aligned_v16(x) && (MODE == 0 || aligned_v16(g)))
	{
		int cpb;
		dim3 grid;
		reduce_config(outer, C / W, cpb, grid);
		bn_reduce_kernel<T, MODE, MASK><<<grid, 256, 0, s>>>(x, g, mean, coef, outer, C, part, cpb);
		*part_rows = (int)grid.y;
		return check("bn_reduce");
	}
	*part_rows = 0;
	bn_reduce_generic_kernel<T, MODE, MASK><<<C, 512, 0, s>>>(x, g, mean, coef, outer, C, inner, ws);
	return check("bn_reduce");
}

// colsum_out / colsum_kind: per-channel sums of the values written (backward only), stored in element kind colsum_kind
template <typename T, int BWD, int RELU>
static int run_apply(cudaStream_t s, const T* x, const T* g, T* out, const float* coef, size_t outer, int C, size_t inner, float* part = 0, void* colsum_out = 0, int colsum_kind = 0, int* colsum_done = 0)
{
	const size_t total = outer * C * inner;
	constexpr int W = Vec16<T>::W;
	const int CW = C / W;
	if (inner == 1 && C % W == 0 && (256 % CW == 0 || CW % 256 == 0) && aligned_v16(x) && aligned_v16(out) && (!BWD || aligned_v16(g)))
	{
		// channel-stationary threads: the grid stride is a multiple of the channel groups per pixel
		int grid = grid_for(total / W / 4, 256);
		if (CW > 256)
			grid = (grid + CW / 256 - 1) / (CW / 256) * (CW / 256);
		if (BWD && part && colsum_out)
		{
			bn_apply_fixed_kernel<T, BWD, RELU, 1><<<grid, 256, 0, s>>>(x, g, out, coef, total / W, C, part);
			if (check("bn_apply"))
				return -1;
			const int rows = CW < 256 ? grid : (int)((size_t)grid * 256 / CW);
			bn_colsum_rows_kernel<<<(C + 31) / 32, 1024, 0, s>>>(part, rows, C, colsum_out, colsum_kind);
			*colsum_done = 1;
			return check("bn_colsum_rows");
		}
		bn_apply_fixed_kernel<T, BWD, RELU, 0><<<grid, 256, 0, s>>>(x, g, out, coef, total / W, C, 0);
		return check("bn_apply");
	}
	if (inner == 1 && C % 4 == 0 && aligned_v4(x) && aligned_v4(out) && (!BWD || aligned_v4(g)))
	{
		int grid = grid_for(total / 8, 256);
		const int CV = C / 4;
		if (BWD && part && colsum_out && (256 % CV == 0 || CV % 256 == 0))
		{
			if (CV > 256) // the grid stride must be a multiple of CV
				grid = (grid + CV / 256 - 1) / (CV / 256) * (CV / 256);
			bn_apply_vec_kernel<T, BWD, RELU, 1><<<grid, 256, 0, s>>>(x, g, out, coef, total / 4, C, part);
			if (check("bn_apply"))
				return -1;
			const int rows = CV < 256 ? grid : (int)((size_t)grid * 256 / CV);
			bn_colsum_rows_kernel<<<(C + 31) / 32, 1024, 0, s>>>(part, rows, C, colsum_out, colsum_kind);
			*colsum_done = 1;
			return check("bn_colsum_rows");
		}
		bn_apply_vec_kernel<T, BWD, RELU, 0><<<grid, 256, 0, s>>>(x, g, out, coef, total / 4, C, 0);
	} else
		bn_apply_generic_kernel<T, BWD, RELU><<<grid_for(total, 256), 256, 0, s>>>(x, g, out, coef, total, C, inner);
	return check("bn_apply");
}

template <typename T>
static int bn_fwd_train_t(cudaStream_t s, const T* x, T* y, const float* scale, const float* bias, float* running_mean, float* running_var, float* saved_mean, float* saved_inv_std, size_t outer, int C, size_t inner, float epsilon, float momentum, void* workspace, int fuse_relu, const float* ext_part, int ext_rows, float* coef_out)
{
	if (outer * C * inner == 0)
		return 0;
	double* ws = ws_sums(workspace);
	// coef_out: statistics only -- the per-channel a, b go to the caller's [2, C] buffer and y is not written
	float* coef = coef_out ? coef_out : ws_coef(workspace, C);
	int part_rows = 0;
	if (ext_part && ext_rows > 0)
	{
		// the producing convolution already folded its output into per-(CTA, warp quarter) shifted sums (four planes of ext_rows x C)
		bn_finalize_ext_kernel<<<(C + 31) / 32, 1024, 0, s>>>(ext_part, ext_rows, C, epsilon, momentum, scale, bias, running_mean, running_var, saved_mean, saved_inv_std, coef);
		if (check("bn_fwd_finalize(ext)"))
			return -1;
		if (coef_out)
			return 0;
		return fuse_relu ? run_apply<T, 0, 1>(s, x, (const T*)0, y, coef, outer, C, inner) : run_apply<T, 0, 0>(s, x, (const T*)0, y, coef, outer, C, inner);
	}
	if (run_reduce<T, 0, 0>(s, x, (const T*)0, 0, 0, outer, C, inner, ws, ws_part(workspace, C), &part_rows))
		return -1;
	if (part_rows > 0)
		bn_finalize_partials_kernel<T, 0, 0><<<(C + 31) / 32, 1024, 0, s>>>(ws_part(workspace, C), part_rows, x, C, (double)outer * (double)inner, epsilon, momentum, scale, bias, running_mean, running_var, saved_mean, saved_inv_std, 0, 0, coef);
	else
		bn_fwd_finalize_kernel<T><<<(C + 127) / 128, 128, 0, s>>>(x, inner, ws, C, (double)outer * (double)inner, epsilon, momentum, scale, bias, running_mean, running_var, saved_mean, saved_inv_std, coef);
	if (check("bn_fwd_finalize"))
		return -1;
	if (coef_out)
		return 0;
	return fuse_relu ? run_apply<T, 0, 1>(s, x, (const T*)0, y, coef, outer, C, inner) : run_apply<T, 0, 0>(s, x, (const T*)0, y, coef, outer, C, inner);
}

template <typename T>
static int bn_fwd_test_t(cudaStream_t s, const T* x, T* y, const float* scale, const float* bias, const float* mean, const float* var, size_t outer, int C, size_t inner, float epsilon, void* workspace)
{
	if (outer * C * inner == 0)
		return 0;
	float* coef = ws_coef(workspace, C);
	bn_test_coef_kernel<<<(C + 127) / 128, 128, 0, s>>>(C, epsilon, scale, bias, mean, var, coef);
	if (check("bn_test_coef"))
		return -1;
	return run_apply<T, 0, 0>(s, x, (const T*)0, y, coef, outer, C, inner);
}

// bias != NULL selects the fused form: g is the gradient w.r.t. relu(bn(x)) and is masked by bn(x) > 0 on the fly
// ext_part / ext_rows: the partial rows of the reduction over (g, x), already produced by bn_add_relu_bwd_reduce_t
template <typename T>
static int bn_bwd_t(cudaStream_t s, const T* g, const T* x, const float* scale, const float* bias, const float* saved_mean, const float* saved_inv_std, T* dx, float* dscale, float* dbias, size_t outer, int C, size_t inner, void* workspace, void* dx_colsum, int colsum_kind, const float* ext_part, int ext_rows)
{
	if (outer * C * inner == 0)
		return 0;
	double* ws = ws_sums(workspace);
	float* coef = ws_coef(workspace, C);
	const int mask = bias != 0;
	const bool vec = inner == 1 && C % Vec16<T>::W == 0 && aligned_v16(x) && aligned_v16(g); // = the condition under which run_reduce leaves partial rows
	if (mask)
	{
		bn_mask_coef_kernel<<<(C + 127) / 128, 128, 0, s>>>(C, scale, bias, saved_mean, saved_inv_std, coef);
		if (check("bn_mask_coef"))
			return -1;
	} else if (!vec) {
		// a is still needed by the apply pass (the vector path gets it from bn_finalize_partials_kernel<1, 1>)
		bn_mask_coef_kernel<<<(C + 127) / 128, 128, 0, s>>>(C, scale, scale, saved_mean, saved_inv_std, coef);
		if (check("bn_coef"))
			return -1;
	}
	int part_rows = 0;
	const float* part_in = ws_part(workspace, C);
	if (ext_part && ext_rows > 0 && vec && !mask)
		part_in = ext_part, part_rows = ext_rows;
	else if (mask ? run_reduce<T, 1, 1>(s, x, g, saved_mean, coef, outer, C, inner, ws, ws_part(workspace, C), &part_rows) : run_reduce<T, 1, 0>(s, x, g, saved_mean, coef, outer, C, inner, ws, ws_part(workspace, C), &part_rows))
		return -1;
	const double count = (double)outer * (double)inner;
	if (part_rows > 0 && mask)
		bn_finalize_partials_kernel<T, 1, 0><<<(C + 31) / 32, 1024, 0, s>>>(part_in, part_rows, (const T*)0, C, count, 0.f, 0.f, scale, 0, 0, 0, const_cast<float*>(saved_mean), const_cast<float*>(saved_inv_std), dscale, dbias, coef);
	else if (part_rows > 0)
		bn_finalize_partials_kernel<T, 1, 1><<<(C + 31) / 32, 1024, 0, s>>>(part_in, part_rows, (const T*)0, C, count, 0.f, 0.f, scale, 0, 0, 0, const_cast<float*>(saved_mean), const_cast<float*>(saved_inv_std), dscale, dbias, coef);
	else
		bn_bwd_finalize_kernel<<<(C + 127) / 128, 128, 0, s>>>(ws, C, (float)count, scale, saved_mean, saved_inv_std, dscale, dbias, coef);
	if (check("bn_bwd_finalize"))
		return -1;
	if (!dx)
		return 0;
	// dx_colsum: per-channel sum of dx (the bias gradient of the convolution that produced x), gathered by the apply pass itself;
	// the partial rows reuse the reduce pass's partial area (its contents were consumed by the finalize kernel above)
	int done = 0;
	float* const part = dx_colsum ? ws_part(workspace, C) : 0;
	if (mask ? run_apply<T, 1, 1>(s, x, g, dx, coef, outer, C, inner, part, dx_colsum, colsum_kind, &done) : run_apply<T, 1, 0>(s, x, g, dx, coef, outer, C, inner, part, dx_colsum, colsum_kind, &done))
		return -1;
	if (dx_colsum && !done) // layouts the vector path does not take: a separate column sum over dx
		return colsum_any(s, ElemKind<T>::value, dx, outer * inner, C, C, dx_colsum, colsum_kind, 0, 0);
	return 0;
}

int bn_fwd_train_f32(cudaStream_t s, const float* x, float* y, const float* scale, const float* bias, float* running_mean, float* running_var, float* saved_mean, float* saved_inv_std, size_t outer, int C, size_t inner, float epsilon, float momentum, void* workspace, int fuse_relu, const float* ext_part, int ext_rows, float* coef_out)
{
	return bn_fwd_train_t<float>(s, x, y, scale, bias, running_mean, running_var, saved_mean, saved_inv_std, outer, C, inner, epsilon, momentum, workspace, fuse_relu, ext_part, ext_rows, coef_out);
}
int bn_fwd_test_f32(cudaStream_t s, const float* x, float* y, const float* scale, const float* bias, const float* mean, const float* var, size_t outer, int C, size_t inner, float epsilon, void* workspace)
{
	return bn_fwd_test_t<float>(s, x, y, scale, bias, mean, var, outer, C, inner, epsilon, workspace);
}
int bn_bwd_f32(cudaStream_t s, const float* g, const float* x, const float* scale, const float* bias, const float* saved_mean, const float* saved_inv_std, float* dx, float* dscale, float* dbias, size_t outer, int C, size_t inner, void* workspace, float* dx_colsum, const float* ext_part, int ext_rows)
{
	return bn_bwd_t<float>(s, g, x, scale, bias, saved_mean, saved_inv_std, dx, dscale, dbias, outer, C, inner, workspace, dx_colsum, 0, ext_part, ext_rows);
}
// 16-bit activations (kind 1 = bf16, 2 = fp16); scale / bias / statistics / parameter gradients stay fp32
// (lib/nnc/ccv_cnnp_model_addons.c:954-956)
int bn_fwd_train_16(cudaStream_t s, int kind, const void* x, void* y, const float* scale, const float* bias, float* running_mean, float* running_var, float* saved_mean, float* saved_inv_std, size_t outer, int C, size_t inner, float epsilon, float momentum, void* workspace, int fuse_relu, const float* ext_part, int ext_rows, float* coef_out)
{
	if (kind == 1)
		return bn_fwd_train_t<__nv_bfloat16>(s, (const __nv_bfloat16*)x, (__nv_bfloat16*)y, scale, bias, running_mean, running_var, saved_mean, saved_inv_std, outer, C, inner, epsilon, momentum, workspace, fuse_relu, ext_part, ext_rows, coef_out);
	return bn_fwd_train_t<__half>(s, (const __half*)x, (__half*)y, scale, bias, running_mean, running_var, saved_mean, saved_inv_std, outer, C, inner, epsilon, momentum, workspace, fuse_relu, ext_part, ext_rows, coef_out);
}
int bn_fwd_test_16(cudaStream_t s, int kind, const void* x, void* y, const float* scale, const float* bias, const float* mean, const float* var, size_t outer, int C, size_t inner, float epsilon, void* workspace)
{
	if (kind == 1)
		return bn_fwd_test_t<__nv_bfloat16>(s, (const __nv_bfloat16*)x, (__nv_bfloat16*)y, scale, bias, mean, var, outer, C, inner, epsilon, workspace);
	return bn_fwd_test_t<__half>(s, (const __half*)x, (__half*)y, scale, bias, mean, var, outer, C, inner, epsilon, workspace);
}
int bn_bwd_16(cudaStream_t s, int kind, const void* g, const void* x, const float* scale, const float* bias, const float* saved_mean, const float* saved_inv_std, void* dx, float* dscale, float* dbias, size_t outer, int C, size_t inner, void* workspace, void* dx_colsum, int colsum_kind, const float* ext_part, int ext_rows)
{
	if (kind == 1)
		return bn_bwd_t<__nv_bfloat16>(s, (const __nv_bfloat16*)g, (const __nv_bfloat16*)x, scale, bias, saved_mean, saved_inv_std, (__nv_bfloat16*)dx, dscale, dbias, outer, C, inner, workspace, dx_colsum, colsum_kind, ext_part, ext_rows);
	return bn_bwd_t<__half>(s, (const __half*)g, (const __half*)x, scale, bias, saved_mean, saved_inv_std, (__half*)dx, dscale, dbias, outer, C, inner, workspace, dx_colsum, colsum_kind, ext_part, ext_rows);
}

// ------------------------------------------------------------------------------------------------ fused residual adds
// MODE 0: out = relu(a + b)                      (EWSUM then RELU_FORWARD at the end of a residual block)
// MODE 1: out = y > 0 ? a + b : 0                (EWSUM of the two branch gradients then RELU_BACKWARD)
template <typename T, int MODE>
__global__ void __launch_bounds__(256) add_relu_kernel(const T* __restrict__ a, const T* __restrict__ b, const T* __restrict__ y, T* __restrict__ out, const size_t n, const int vec)
{
	constexpr int W = Vec16<T>::W; // one 16-byte access per operand and iteration
	const size_t nw = vec ? n / W : 0;
	for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nw; i += (size_t)gridDim.x * blockDim.x)
	{
		float u[W], v[W], m[W], o[W];
		ldv(a + i * W, u), ldv(b + i * W, v);
		if (MODE == 1)
			ldv(y + i * W, m);
#pragma unroll
		for (int k = 0; k < W; k++)
		{
			o[k] = u[k] + v[k];
			o[k] = MODE == 0 ? fmaxf(o[k], 0.f) : (m[k] > 0.f ? o[k] : 0.f);
		}
		stv(out + i * W, o);
	}
	for (size_t i = nw * W + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
	{
		const float o = ldf(a + i) + ldf(b + i);
		stf(out + i, MODE == 0 ? fmaxf(o, 0.f) : (ldf(y + i) > 0.f ? o : 0.f));
	}
}
template <typename T>
static int add_relu_fwd_t(cudaStream_t s, const T* a, const T* b, T* out, size_t n)
{
	if (n == 0)
		return 0;
	const int vec = aligned_v16(a) && aligned_v16(b) && aligned_v16(out);
	add_relu_kernel<T, 0><<<grid_for(vec ? n / Vec16<T>::W + 1 : n, 256), 256, 0, s>>>(a, b, (const T*)0, out, n, vec);
	return check("add_relu_fwd");
}
template <typename T>
static int add_relu_bwd_t(cudaStream_t s, const T* a, const T* b, const T* y, T* out, size_t n)
{
	if (n == 0)
		return 0;
	const int vec = aligned_v16(a) && aligned_v16(b) && aligned_v16(out) && aligned_v16(y);
	add_relu_kernel<T, 1><<<grid_for(vec ? n / Vec16<T>::W + 1 : n, 256), 256, 0, s>>>(a, b, y, out, n, vec);
	return check("add_relu_bwd");
}
int ew_add_relu_fwd_f32(cudaStream_t s, const float* a, const float* b, float* out, size_t n) { return add_relu_fwd_t<float>(s, a, b, out, n); }
int ew_add_relu_bwd_f32(cudaStream_t s, const float* a, const float* b, const float* y, float* out, size_t n) { return add_relu_bwd_t<float>(s, a, b, y, out, n); }
int ew_add_relu_fwd_16(cudaStream_t s, int kind, const void* a, const void* b, void* out, size_t n)
{
	return kind == 1 ? add_relu_fwd_t<__nv_bfloat16>(s, (const __nv_bfloat16*)a, (const __nv_bfloat16*)b, (__nv_bfloat16*)out, n) : add_relu_fwd_t<__half>(s, (const __half*)a, (const __half*)b, (__half*)out, n);
}
int ew_add_relu_bwd_16(cudaStream_t s, int kind, const void* a, const void* b, const void* y, void* out, size_t n)
{
	return kind == 1 ? add_relu_bwd_t<__nv_bfloat16>(s, (const __nv_bfloat16*)a, (const __nv_bfloat16*)b, (const __nv_bfloat16*)y, (__nv_bfloat16*)out, n) : add_relu_bwd_t<__half>(s, (const __half*)a, (const __half*)b, (const __half*)y, (__half*)out, n);
}

// ------------------------------------------------------------------------------------------------ residual block end
// Forward: out = relu(roundT(x * a + b) + r) with the [2, C] coefficients a statistics-only batch norm left in coef (NHWC, C =
// the innermost dimension); the same bits as the batch-norm apply pass followed by add_relu_kernel, without writing / reading
// the normalised tensor in between.
template <typename T>
static int bn_add_relu_fwd_t(cudaStream_t s, const T* x, const T* r, T* out, const float* coef, size_t outer, int C)
{
	const size_t total = outer * C;
	if (total == 0)
		return 0;
	constexpr int W = Vec16<T>::W;
	const int CW = C / W;
	if (C % W == 0 && (256 % CW == 0 || CW % 256 == 0) && aligned_v16(x) && aligned_v16(r) && aligned_v16(out))
	{
		// the launch rules of run_apply's channel-stationary path
		int grid = grid_for(total / W / 4, 256);
		if (CW > 256)
			grid = (grid + CW / 256 - 1) / (CW / 256) * (CW / 256);
		bn_apply_fixed_kernel<T, 0, 0, 0, 1><<<grid, 256, 0, s>>>(x, r, out, coef, total / W, C, 0);
	} else
		bn_apply_generic_kernel<T, 0, 0, 1><<<grid_for(total, 256), 256, 0, s>>>(x, r, out, coef, total, C, 1);
	return check("bn_add_relu_fwd");
}
int bn_add_relu_fwd_f32(cudaStream_t s, const float* x, const float* r, float* out, const float* coef, size_t outer, int C) { return bn_add_relu_fwd_t<float>(s, x, r, out, coef, outer, C); }
int bn_add_relu_fwd_16(cudaStream_t s, int kind, const void* x, const void* r, void* out, const float* coef, size_t outer, int C)
{
	return kind == 1 ? bn_add_relu_fwd_t<__nv_bfloat16>(s, (const __nv_bfloat16*)x, (const __nv_bfloat16*)r, (__nv_bfloat16*)out, coef, outer, C) : bn_add_relu_fwd_t<__half>(s, (const __half*)x, (const __half*)r, (__half*)out, coef, outer, C);
}

// Backward: g = y > 0 ? a + b : 0 (b may be NULL: y > 0 ? a : 0) stored to g, and in the same pass the partial rows of the
// reduction the batch-norm backward behind it needs over (g, x), into part (room for part_cap rows of 2C floats).  The grid and
// row walk are run_reduce's, so the rows are bit-identical to what bn_bwd_t would reduce from g itself.  *part_rows = the number
// of rows written; 0 when the layout does not take the vector path (then only g is written, by the plain kernels).
template <typename T>
static int bn_add_relu_bwd_reduce_t(cudaStream_t s, const T* a, const T* b, const T* y, const T* x, const float* mean, T* g, size_t outer, int C, float* part, int part_cap, int* part_rows)
{
	*part_rows = 0;
	const size_t n = outer * C;
	if (n == 0)
		return 0;
	constexpr int W = Vec16<T>::W;
	if (part && C % W == 0 && aligned_v16(x) && aligned_v16(g) && aligned_v16(a) && aligned_v16(y) && (!b || aligned_v16(b)))
	{
		int cpb;
		dim3 grid;
		reduce_config(outer, C / W, cpb, grid);
		if ((int)grid.y <= part_cap)
		{
			bn_reduce_kernel<T, 2, 0><<<grid, 256, 0, s>>>(x, (const T*)0, mean, (const float*)0, outer, C, part, cpb, a, b, y, g);
			*part_rows = (int)grid.y;
			return check("bn_add_relu_bwd_reduce");
		}
	}
	if (b)
		return add_relu_bwd_t<T>(s, a, b, y, g, n);
	if (ElemKind<T>::value == 0)
		return ew_relu_bwd_f32(s, (const float*)a, (const float*)y, (float*)g, n);
	return ew_relu_bwd_16(s, ElemKind<T>::value, a, y, g, n);
}
int bn_add_relu_bwd_reduce_f32(cudaStream_t s, const float* a, const float* b, const float* y, const float* x, const float* mean, float* g, size_t outer, int C, float* part, int part_cap, int* part_rows)
{
	return bn_add_relu_bwd_reduce_t<float>(s, a, b, y, x, mean, g, outer, C, part, part_cap, part_rows);
}
int bn_add_relu_bwd_reduce_16(cudaStream_t s, int kind, const void* a, const void* b, const void* y, const void* x, const float* mean, void* g, size_t outer, int C, float* part, int part_cap, int* part_rows)
{
	if (kind == 1)
		return bn_add_relu_bwd_reduce_t<__nv_bfloat16>(s, (const __nv_bfloat16*)a, (const __nv_bfloat16*)b, (const __nv_bfloat16*)y, (const __nv_bfloat16*)x, mean, (__nv_bfloat16*)g, outer, C, part, part_cap, part_rows);
	return bn_add_relu_bwd_reduce_t<__half>(s, (const __half*)a, (const __half*)b, (const __half*)y, (const __half*)x, mean, (__half*)g, outer, C, part, part_cap, part_rows);
}

} // namespace sm100
