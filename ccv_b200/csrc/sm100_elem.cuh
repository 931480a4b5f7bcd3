// sm100_elem.cuh -- element access for the HBM-bound kernels that exist for fp32, bf16 and fp16 tensors: 4 consecutive elements
// at a time as a float4 (16-byte accesses for fp32, 8-byte for the 16-bit types), single elements, and a runtime "kind" for the
// few places where the element type of an output is only known at run time.  Arithmetic is always fp32; 16-bit stores round to
// nearest even.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sm100 {

// element kinds used across the backend: 0 = fp32, 1 = bf16, 2 = fp16
template <typename T> struct ElemKind;
template <> struct ElemKind<float> { static constexpr int value = 0; };
template <> struct ElemKind<__nv_bfloat16> { static constexpr int value = 1; };
template <> struct ElemKind<__half> { static constexpr int value = 2; };

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, const float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float4 ld4(const __nv_bfloat16* p)
{
	const uint2 u = *reinterpret_cast<const uint2*>(p);
	return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16), __uint_as_float(u.y & 0xffff0000u));
}
__device__ __forceinline__ void st4(__nv_bfloat16* p, const float4 v)
{
	const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
	*reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
}
__device__ __forceinline__ float4 ld4(const __half* p)
{
	const uint2 u = *reinterpret_cast<const uint2*>(p);
	const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
	return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void st4(__half* p, const float4 v)
{
	const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
	*reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
}
__device__ __forceinline__ float ldf(const float* p) { return *p; }
__device__ __forceinline__ float ldf(const __nv_bfloat16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ float ldf(const __half* p) { return __half2float(*p); }
__device__ __forceinline__ void stf(float* p, const float v) { *p = v; }
__device__ __forceinline__ void stf(__nv_bfloat16* p, const float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void stf(__half* p, const float v) { *p = __float2half_rn(v); }

// v rounded to the storage type T and back: what a store followed by a load of T gives (a no-op for fp32)
template <typename T> __device__ __forceinline__ float rnd(const float v);
template <> __device__ __forceinline__ float rnd<float>(const float v) { return v; }
template <> __device__ __forceinline__ float rnd<__nv_bfloat16>(const float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
template <> __device__ __forceinline__ float rnd<__half>(const float v) { return __half2float(__float2half_rn(v)); }

// element i of a buffer whose kind is only known at run time
__device__ __forceinline__ float ld_kind(const void* p, const size_t i, const int kind)
{
	return kind == 0 ? reinterpret_cast<const float*>(p)[i] : kind == 1 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]) : __half2float(reinterpret_cast<const __half*>(p)[i]);
}
__device__ __forceinline__ void st_kind(void* p, const size_t i, const float v, const int kind)
{
	if (kind == 0)
		reinterpret_cast<float*>(p)[i] = v;
	else if (kind == 1)
		reinterpret_cast<__nv_bfloat16*>(p)[i] = __float2bfloat16_rn(v);
	else
		reinterpret_cast<__half*>(p)[i] = __float2half_rn(v);
}

// One 16-byte access = W elements (4 fp32, 8 bf16 / fp16): the widest single load / store, what the streaming kernels use when
// the channel count allows it
template <typename T> struct Vec16 { static constexpr int W = 16 / sizeof(T); };
__device__ __forceinline__ void ldv(const float* p, float (&v)[4])
{
	const float4 t = *reinterpret_cast<const float4*>(p);
	v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
}
__device__ __forceinline__ void stv(float* p, const float (&v)[4]) { *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]); }
__device__ __forceinline__ void ldv(const __nv_bfloat16* p, float (&v)[8])
{
	const uint4 u = *reinterpret_cast<const uint4*>(p);
	const uint32_t w[4] = { u.x, u.y, u.z, u.w };
#pragma unroll
	for (int i = 0; i < 4; i++)
		v[2 * i] = __uint_as_float(w[i] << 16), v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
}
__device__ __forceinline__ void stv(__nv_bfloat16* p, const float (&v)[8])
{
	uint32_t w[4];
#pragma unroll
	for (int i = 0; i < 4; i++)
	{
		const __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
		w[i] = *reinterpret_cast<const uint32_t*>(&t);
	}
	*reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ void ldv(const __half* p, float (&v)[8])
{
	const uint4 u = *reinterpret_cast<const uint4*>(p);
	const uint32_t w[4] = { u.x, u.y, u.z, u.w };
#pragma unroll
	for (int i = 0; i < 4; i++)
	{
		const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
		v[2 * i] = t.x, v[2 * i + 1] = t.y;
	}
}
__device__ __forceinline__ void stv(__half* p, const float (&v)[8])
{
	uint32_t w[4];
#pragma unroll
	for (int i = 0; i < 4; i++)
	{
		const __half2 t = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
		w[i] = *reinterpret_cast<const uint32_t*>(&t);
	}
	*reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}
template <typename T>
static inline bool aligned_v16(const T* p) { return (((uintptr_t)p) & 15) == 0; }

// a pointer is usable by ld4 / st4 when it is aligned to 4 elements
template <typename T>
static inline bool aligned_v4(const T* p) { return (((uintptr_t)p) & (4 * sizeof(T) - 1)) == 0; }

} // namespace sm100
