// nnc_host.cu -- group (B) of include/ccv_nnc_sm100.h: a minimal stand-alone host for the backend, with the
// reference's names and semantics (ccv_nnc_init / ccv_nnc_cmd / ccv_nnc_cmd_exec / tensors / stream contexts),
// so that the backend can be driven without libccv.  When the backend is linked under lib/nnc these symbols are
// ccv's own and this file is left out (see INTEGRATION.md).
//
// Reference being mirrored: lib/nnc/ccv_nnc_cmd.c:27-30,117-131,307-328,651-693 (init, ok, find_backend, exec),
// lib/nnc/ccv_nnc_tensor.c:13-110 (tensor new/free/view), lib/nnc/ccv_nnc_stream.c:27-161,289-294 and
// lib/nnc/gpu/ccv_nnc_compat.cu:255-511 (stream contexts, grow-only workspace), lib/nnc/ccv_nnc_graph_run.c:911-979.
#include "../../include/ccv_nnc_sm100.h"
#include "sm100_contract.h"
#include <cuda_runtime.h>
#include <mutex>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unordered_map>
#include <vector>

struct ccv_nnc_stream_context_s {
	int type;
	int device;
	cudaStream_t stream;
	void* gpu_workspace;
	size_t gpu_workspace_size;
	void* cpu_workspace;
	size_t cpu_workspace_size;
	ccv_nnc_stream_context_neighbor_discovery_f neighbor_discovery;
	void* neighbor_discovery_context;
	uint64_t rng_state; // the per-context generator of ccv_nnc_stream.c:247-281 (there an sfmt_t): 0 = not seeded yet
};

namespace {

// The registry of lib/nnc/ccv_nnc_cmd.c:27-66: init_map[command slot].backends[backend slot], both slots found by the generated
// perfect hashes (lib/nnc/cmd/ccv_nnc_cmd.inc:152-190; here nnc_registry_generated.inc, written by tools/gen_backend_ph.py:
// the reference's own command hash and the 8-slot backend hash that includes CCV_NNC_BACKEND_GPU_SM100).  Only the SM100 column
// is ever filled in this stand-alone host -- the other seven backends are the reference's -- but lookup, capability matching and
// the backend preference order are the reference's code paths, slot for slot.
#include "nnc_registry_generated.inc"
struct sm100_cmd_init_t {
	const char* name;
	uint32_t cmd;
	ccv_nnc_cmd_backend_registry_t backends[CCV_NNC_SM100_BACKEND_SLOTS];
};
sm100_cmd_init_t init_map[CCV_NNC_SM100_CMD_SLOTS];
std::once_flag g_init_once;

// registry record of (cmd, backend), or NULL when either id is not one the tables know
const ccv_nnc_cmd_backend_registry_t* registry_of(const uint32_t cmd, const uint32_t backend)
{
	const int cmd_idx = _ccv_nnc_cmd_ph(cmd), backend_idx = _ccv_nnc_cmd_backend_ph(backend);
	if (cmd_idx < 0 || cmd_idx >= CCV_NNC_SM100_CMD_SLOTS || init_map[cmd_idx].cmd != cmd)
		return 0;
	if (backend_idx < 0 || backend_idx >= CCV_NNC_SM100_BACKEND_SLOTS || sm100_backend_init_map[backend_idx].backend != backend)
		return 0;
	return &init_map[cmd_idx].backends[backend_idx];
}

enum { MATRIX_DENSE = 0x00100000, UNMANAGED = 0x20000000, NO_DATA_ALLOC = 0x10000000 };

size_t datatype_size(const int datatype)
{
	switch (CCV_GET_DATA_TYPE(datatype))
	{
		case CCV_8U: return 1;
		case CCV_32S: case CCV_32F: return 4;
		case CCV_64S: case CCV_64F: return 8;
		case CCV_16F: case CCV_16BF: return 2;
		case CCV_QX: return 1;
	}
	return 0;
}

int tensor_nd(const int* const dim)
{
	int i;
	for (i = 0; i < CCV_NNC_MAX_DIM_ALLOC; i++)
		if (dim[i] == 0)
			return i;
	return CCV_NNC_MAX_DIM_ALLOC;
}

// per-thread default stream contexts, one per device (lib/nnc/gpu/ccv_nnc_compat.cu:342-350).  As in the reference, whose
// per-thread context is zero-initialised, their CUDA stream is the legacy default stream (0): work issued with
// stream_context == NULL is ordered with every later synchronous CUDA call of the caller, so ccv_nnc_cmd_exec only has to
// drain (not wait) on that path (lib/nnc/ccv_nnc_cmd.c:690-691).
thread_local ccv_nnc_stream_context_t* t_default_streams[64] = { 0 };

ccv_nnc_stream_context_t* default_stream(const int device)
{
	const int d = device < 0 ? 0 : device & 63;
	if (!t_default_streams[d])
	{
		ccv_nnc_stream_context_t* const s = (ccv_nnc_stream_context_t*)calloc(1, sizeof(ccv_nnc_stream_context_t));
		s->type = CCV_STREAM_CONTEXT_GPU;
		CCV_STREAM_SET_DEVICE_ID(s->type, d);
		s->device = d;
		s->stream = 0;
		t_default_streams[d] = s;
	}
	return t_default_streams[d];
}

int device_of(ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size)
{
	int i;
	for (i = 0; i < output_size; i++)
		if (outputs[i] && CCV_TENSOR_GET_MEMORY(outputs[i]->info.type) == CCV_TENSOR_GPU_MEMORY)
			return CCV_TENSOR_GET_DEVICE_ID(outputs[i]->info.type);
	for (i = 0; i < input_size; i++)
		if (inputs[i] && CCV_TENSOR_GET_MEMORY(inputs[i]->info.type) == CCV_TENSOR_GPU_MEMORY)
			return CCV_TENSOR_GET_DEVICE_ID(inputs[i]->info.type);
	return -1;
}

} // namespace

extern "C" {

void ccv_nnc_init(void)
{
	std::call_once(g_init_once, []() {
		memset(init_map, 0, sizeof(init_map));
		for (int i = 0; i < CCV_NNC_SM100_CMD_SLOTS; i++)
			init_map[i].name = sm100_cmd_init_map[i].name, init_map[i].cmd = sm100_cmd_init_map[i].cmd;
		// what the generated _ccv_nnc_cmd_init() does for every (command, backend) pair (integration/ccv_nnc_cmd_sm100_init.inc)
#define CCV_SM100_CALL_REGISTER(cmd) _register_command_ ## cmd ## _backend_CCV_NNC_BACKEND_GPU_SM100(&init_map[_ccv_nnc_cmd_ph((uint32_t)cmd)].backends[_ccv_nnc_cmd_backend_ph(CCV_NNC_BACKEND_GPU_SM100)]);
		CCV_NNC_SM100_COMMANDS(CCV_SM100_CALL_REGISTER)
#undef CCV_SM100_CALL_REGISTER
	});
}

ccv_nnc_cmd_t ccv_nnc_cmd(const uint32_t cmd, ccv_nnc_cmd_vtab_t* const isa, const ccv_nnc_cmd_param_t params, const int flags)
{
	ccv_nnc_cmd_t c;
	memset(&c, 0, sizeof(c));
	c.cmd = cmd;
	c.backend = CCV_NNC_NO_BACKEND;
	c.algorithm = -1;
	c.info = params;
	c.isa = isa;
	return c;
}

int ccv_nnc_cmd_ok(const uint32_t cmd, const uint32_t backend)
{
	if (cmd == CCV_NNC_NOOP)
		return 1;
	ccv_nnc_init();
	// lib/nnc/ccv_nnc_cmd.c:117-131
	const ccv_nnc_cmd_backend_registry_t* const r = registry_of(cmd, backend == CCV_NNC_NO_BACKEND ? (uint32_t)CCV_NNC_BACKEND_GPU_SM100 : backend);
	return r && r->exec != 0;
}

uint32_t ccv_nnc_cmd_find_backend(const ccv_nnc_cmd_t cmd, const int tensor_memory, const int tensor_formats, const int tensor_datatypes)
{
	if (cmd.cmd == CCV_NNC_NOOP || cmd.cmd == CCV_NNC_CUSTOM_FORWARD || cmd.cmd == CCV_NNC_CUSTOM_BACKWARD)
		return cmd.backend;
	ccv_nnc_init();
	// lib/nnc/ccv_nnc_cmd.c:307-328: the first backend slot, in table order, whose record has a kernel and covers every memory
	// kind, format and datatype of the operands
	const int cmd_idx = _ccv_nnc_cmd_ph(cmd.cmd);
	if (cmd_idx < 0 || cmd_idx >= CCV_NNC_SM100_CMD_SLOTS || init_map[cmd_idx].cmd != cmd.cmd)
		return cmd.backend;
	for (int i = 0; i < CCV_NNC_SM100_BACKEND_SLOTS; i++)
	{
		const ccv_nnc_cmd_backend_registry_t& r = init_map[cmd_idx].backends[i];
		if (r.exec && (r.tensor_memory & tensor_memory) == tensor_memory && (r.tensor_formats & tensor_formats) == tensor_formats && (r.tensor_datatypes & tensor_datatypes) == tensor_datatypes)
			return sm100_backend_init_map[i].backend;
	}
	return cmd.backend;
}

uint64_t ccv_nnc_cmd_mono_time(void)
{
	struct timespec ts;
	clock_gettime(CLOCK_MONOTONIC, &ts);
	return ts.tv_sec * 1000000000ULL + ts.tv_nsec;
}

int ccv_nnc_cmd_exec(const ccv_nnc_cmd_t cmd, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	if (cmd.cmd == CCV_NNC_NOOP)
		return CCV_NNC_EXEC_SUCCESS;
	ccv_nnc_init();
	if (!stream_context)
	{
		const int device = device_of(inputs, input_size, outputs, output_size);
		if (device >= 0)
			cudaSetDevice(device);
	} else if (CCV_STREAM_GET_CONTEXT(stream_context->type) == CCV_STREAM_CONTEXT_GPU)
		cudaSetDevice(stream_context->device); // the reference's stream getter does this (gpu/ccv_nnc_compat.cu:319-340); kernels, workspace and function attributes follow the stream's device
	if (cmd.cmd == CCV_NNC_CUSTOM_FORWARD || cmd.cmd == CCV_NNC_CUSTOM_BACKWARD)
		return CCV_NNC_EXEC_NO_KERNEL; // custom vtabs live above this slice of the API
	uint32_t backend = cmd.backend;
	if (backend == CCV_NNC_NO_BACKEND)
	{
		int tensor_memory = 0, tensor_formats = 0, tensor_datatypes = 0, i;
		for (i = 0; i < input_size; i++)
			if (inputs[i])
				tensor_memory |= CCV_TENSOR_GET_MEMORY(inputs[i]->info.type), tensor_formats |= inputs[i]->info.format, tensor_datatypes |= CCV_GET_DATA_TYPE(inputs[i]->info.datatype);
		for (i = 0; i < output_size; i++)
			if (outputs[i])
				tensor_memory |= CCV_TENSOR_GET_MEMORY(outputs[i]->info.type), tensor_formats |= outputs[i]->info.format, tensor_datatypes |= CCV_GET_DATA_TYPE(outputs[i]->info.datatype);
		backend = ccv_nnc_cmd_find_backend(cmd, tensor_memory, tensor_formats, tensor_datatypes);
	}
	// init_map[cmd].backends[backend].exec (lib/nnc/ccv_nnc_cmd.c:682-686); every column but GPU_SM100 is empty here: there is
	// deliberately no CPU fallback in this library
	const ccv_nnc_cmd_backend_registry_t* const reg = registry_of(cmd.cmd, backend);
	if (!reg || !reg->exec)
		return CCV_NNC_EXEC_NO_KERNEL;
	// a backend named explicitly is still held to its registered tensor memory (ccv_nnc_cmd_find_backend does the same test,
	// ccv_nnc_cmd.c:307-328): host tensors never reach a device kernel, except through the transfer commands that register both
	int memory = 0;
	for (int i = 0; i < input_size; i++)
		if (inputs[i])
			memory |= CCV_TENSOR_GET_MEMORY(inputs[i]->info.type);
	for (int i = 0; i < output_size; i++)
		if (outputs[i])
			memory |= CCV_TENSOR_GET_MEMORY(outputs[i]->info.type);
	if ((reg->tensor_memory & memory) != memory)
		return CCV_NNC_EXEC_NO_KERNEL;
	const int ret = reg->exec(cmd, hint, flags, inputs, input_size, outputs, output_size, stream_context);
	if (!stream_context)
	{
		// lib/nnc/ccv_nnc_cmd.c:690-691: without a stream the per-thread context is drained (its workspace released); the work
		// itself sits on the legacy default stream, ordered before whatever the caller does next
		const int device = device_of(inputs, input_size, outputs, output_size);
		if (device >= 0)
			ccv_nnc_stream_context_drain(default_stream(device));
	}
	return ret;
}

ccv_nnc_hint_t ccv_nnc_hint_auto(const ccv_nnc_cmd_param_t cmd, const ccv_nnc_tensor_param_t a, const ccv_nnc_tensor_param_t b)
{
	// lib/nnc/ccv_nnc_cmd.c:181-217.  Per spatial axis: the stride that roughly maps a's extent onto b's, then whatever total
	// border makes (b - 1) * stride + size cover a, the larger half in front.  Nothing is clamped: a window smaller than the
	// stride yields a negative border, exactly as the reference reports it (ccv_nnc_hint_verify is what rejects bad hints).
	ccv_nnc_hint_t hint;
	memset(&hint, 0, sizeof(hint));
	if (a.format != b.format)
		return hint;
	const int a_nd = tensor_nd(a.dim), b_nd = tensor_nd(b.dim);
	if (a_nd != b_nd || (a_nd != CCV_NNC_MAX_DIM + 1 && a_nd != CCV_NNC_MAX_DIM + 2))
		return hint;
	int hw;
	if (a.format == CCV_TENSOR_FORMAT_CHWN || (a.format == CCV_TENSOR_FORMAT_NHWC && a_nd == CCV_NNC_MAX_DIM + 1))
		hw = 0;
	else if ((a.format == CCV_TENSOR_FORMAT_NHWC && a_nd == CCV_NNC_MAX_DIM + 2) || (a.format == CCV_TENSOR_FORMAT_NCHW && a_nd == CCV_NNC_MAX_DIM + 1))
		hw = 1;
	else if (a.format == CCV_TENSOR_FORMAT_NCHW && a_nd == CCV_NNC_MAX_DIM + 2)
		hw = 2;
	else
		return hint;
	for (int i = 0; i < CCV_NNC_MAX_DIM; i++)
	{
		const int ad = a.dim[i + hw], bd = b.dim[i + hw];
		if (ad <= 0 || bd <= 0)
		{
			memset(&hint, 0, sizeof(hint));
			return hint;
		}
		const int stride = (ad + bd / 2) / bd;
		const int border = (bd - 1) * stride - ad + cmd.size.dim[i];
		hint.stride.dim[i] = stride;
		hint.border.begin[i] = (border + 1) / 2;
		hint.border.end[i] = border - hint.border.begin[i];
	}
	return hint;
}

size_t ccv_nnc_tensor_data_size(const ccv_nnc_tensor_param_t params)
{
	size_t count = 1;
	int i;
	for (i = 0; i < CCV_NNC_MAX_DIM_ALLOC && params.dim[i] > 0; i++)
		count *= (size_t)params.dim[i];
	const size_t size = count * datatype_size(params.datatype);
	return (size + 63) & ~(size_t)63;
}

ccv_nnc_tensor_t* ccv_nnc_tensor_new(const void* const ptr, const ccv_nnc_tensor_param_t params, const int flags)
{
	ccv_nnc_tensor_t* tensor = (ccv_nnc_tensor_t*)calloc(1, sizeof(ccv_nnc_tensor_t));
	tensor->refcount = 1;
	tensor->info = params;
	if (ptr)
	{
		tensor->type = NO_DATA_ALLOC | MATRIX_DENSE | CCV_GET_DATA_TYPE(params.datatype);
		tensor->data.u8 = (unsigned char*)ptr;
		return tensor;
	}
	const size_t size = ccv_nnc_tensor_data_size(params);
	tensor->data_size = size;
	tensor->type = UNMANAGED | MATRIX_DENSE | CCV_GET_DATA_TYPE(params.datatype);
	if (size == 0)
		return tensor;
	if (CCV_TENSOR_GET_MEMORY(params.type) == CCV_TENSOR_GPU_MEMORY)
	{
		cudaSetDevice(CCV_TENSOR_GET_DEVICE_ID(params.type));
		void* p = 0;
		const cudaError_t e = cudaMalloc(&p, size);
		if (e != cudaSuccess)
		{
			sm100::set_last_error("cudaMalloc(tensor)", e);
			free(tensor);
			return 0;
		}
		tensor->data.u8 = (unsigned char*)p;
	} else {
		void* p = 0;
		if (posix_memalign(&p, 64, size))
		{
			free(tensor);
			return 0;
		}
		tensor->data.u8 = (unsigned char*)p;
	}
	return tensor;
}

int ccv_nnc_tensor_pin_memory(ccv_nnc_tensor_t* const tensor)
{
	if (CCV_TENSOR_GET_MEMORY(tensor->info.type) != CCV_TENSOR_CPU_MEMORY || (tensor->type & CCV_TENSOR_PINNED_MEM) || !tensor->data.u8)
		return 0;
	const size_t size = tensor->data_size ? tensor->data_size : ccv_nnc_tensor_data_size(tensor->info);
	if (cudaHostRegister(tensor->data.u8, size, cudaHostRegisterPortable) != cudaSuccess)
	{
		cudaGetLastError();
		return -1;
	}
	tensor->type |= CCV_TENSOR_PINNED_MEM;
	return 0;
}

void ccv_nnc_tensor_free(ccv_nnc_tensor_t* const tensor)
{
	if (!tensor)
		return;
	if (!(tensor->type & NO_DATA_ALLOC) && !CCV_IS_TENSOR_VIEW(tensor) && tensor->data.u8)
	{
		if (CCV_TENSOR_GET_MEMORY(tensor->info.type) == CCV_TENSOR_GPU_MEMORY)
			cudaFree(tensor->data.u8);
		else {
			if (tensor->type & CCV_TENSOR_PINNED_MEM)
				cudaHostUnregister(tensor->data.u8);
			free(tensor->data.u8);
		}
	}
	free(tensor);
}

ccv_nnc_tensor_view_t* ccv_nnc_tensor_view_new(const ccv_nnc_tensor_t* const tensor, const ccv_nnc_tensor_param_t params, const int ofs[CCV_NNC_MAX_DIM_ALLOC], const int stride[CCV_NNC_MAX_DIM_ALLOC])
{
	// lib/nnc/ccv_nnc_tensor.c:247-310: data already includes the view offset; contiguous iff strides are the packed ones
	ccv_nnc_tensor_view_t* tv = (ccv_nnc_tensor_view_t*)calloc(1, sizeof(ccv_nnc_tensor_view_t));
	tv->type = (tensor->type & ~0xfff) | CCV_TENSOR_VIEW | NO_DATA_ALLOC;
	tv->refcount = 1;
	tv->info = params;
	tv->alias_ref = (uintptr_t)tensor;
	const int nd = tensor_nd(params.dim);
	size_t off = 0;
	int i;
	for (i = 0; i < nd; i++)
		off += (size_t)ofs[i] * stride[i];
	off *= datatype_size(params.datatype);
	tv->off = (off_t)off;
	tv->data.u8 = tensor->data.u8 + off;
	tv->dataof = tensor->dataof;
	memcpy(tv->stride, stride, sizeof(int) * CCV_NNC_MAX_DIM_ALLOC);
	int packed = 1, contiguous = 1;
	for (i = nd - 1; i >= 0; i--)
	{
		if (stride[i] != packed)
			contiguous = 0;
		packed *= params.dim[i];
	}
	tv->contiguous = contiguous;
	return tv;
}

void ccv_nnc_tensor_view_free(ccv_nnc_tensor_view_t* const tensor_view)
{
	free(tensor_view);
}

// ---------------------------------------------------------------------------------------------------- streams
ccv_nnc_stream_context_t* ccv_nnc_stream_context_new(const int type)
{
	ccv_nnc_stream_context_t* s = (ccv_nnc_stream_context_t*)calloc(1, sizeof(ccv_nnc_stream_context_t));
	s->type = type;
	s->device = CCV_STREAM_GET_DEVICE_ID(type);
	if (CCV_STREAM_GET_CONTEXT(type) == CCV_STREAM_CONTEXT_GPU)
	{
		cudaSetDevice(s->device);
		const cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
		if (e != cudaSuccess)
		{
			sm100::set_last_error("cudaStreamCreate", e);
			free(s);
			return 0;
		}
	}
	return s;
}

// ccv_nnc_stream.c:247-281: a generator per stream context, seeded lazily from the calling thread's generator; the random-fill
// commands draw ONE 32-bit seed per launch from it.  (The reference keeps an SFMT state; any well-mixed 64-bit generator serves
// the contract -- the drop-in build uses the reference's own function, this is the stand-alone host's.)
static inline uint32_t splitmix_next(uint64_t* const state)
{
	uint64_t z = (*state += 0x9E3779B97F4A7C15ull);
	z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
	z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
	return (uint32_t)((z ^ (z >> 31)) >> 16);
}
static thread_local uint64_t t_rng_state = 0;
void ccv_nnc_stream_context_set_seed(ccv_nnc_stream_context_t* const stream_context, uint32_t seed)
{
	uint64_t* const st = stream_context ? &stream_context->rng_state : &t_rng_state;
	*st = ((uint64_t)seed << 1) | 1; // never 0 (0 = unseeded)
}
uint32_t ccv_nnc_stream_context_genrand_uint32(ccv_nnc_stream_context_t* const stream_context)
{
	if (!stream_context)
	{
		if (!t_rng_state)
			t_rng_state = ((uint64_t)(uintptr_t)&t_rng_state << 1) | 1;
		return splitmix_next(&t_rng_state);
	}
	if (!stream_context->rng_state)
		stream_context->rng_state = ((uint64_t)ccv_nnc_stream_context_genrand_uint32(0) << 1) | 1;
	return splitmix_next(&stream_context->rng_state);
}

int ccv_nnc_stream_context_type(const ccv_nnc_stream_context_t* const stream_context)
{
	return stream_context->type;
}

void* ccv_nnc_stream_context_get_stream(const ccv_nnc_stream_context_t* const stream_context)
{
	if (!stream_context)
	{
		int device = 0;
		cudaGetDevice(&device);
		return (void*)default_stream(device)->stream;
	}
	return (void*)stream_context->stream;
}

int ccv_nnc_stream_context_get_device(const ccv_nnc_stream_context_t* const stream_context)
{
	if (!stream_context)
	{
		int device = 0;
		cudaGetDevice(&device);
		return device;
	}
	return stream_context->device;
}

void* ccv_nnc_stream_context_get_workspace(ccv_nnc_stream_context_t* const stream_context, const size_t workspace_size, const int mem)
{
	// a single grow-only buffer per (stream, device): one op's scratch is invalidated by the next request on the same
	// stream, which is safe because work on a stream is ordered (lib/nnc/gpu/ccv_nnc_compat.cu:438-471)
	ccv_nnc_stream_context_t* s = stream_context;
	if (!s)
	{
		int device = 0;
		cudaGetDevice(&device);
		s = default_stream(device);
	}
	if (mem == CCV_TENSOR_CPU_MEMORY)
	{
		if (s->cpu_workspace_size < workspace_size)
		{
			free(s->cpu_workspace);
			s->cpu_workspace = 0;
			s->cpu_workspace_size = 0;
			if (posix_memalign(&s->cpu_workspace, 64, workspace_size))
				return 0;
			s->cpu_workspace_size = workspace_size;
		}
		return s->cpu_workspace;
	}
	if (s->gpu_workspace_size < workspace_size)
	{
		cudaSetDevice(s->device); // the buffer belongs to the stream's device, whichever device happens to be current
		if (s->gpu_workspace)
		{
			// kernels already enqueued may still be using the old buffer
			cudaStreamSynchronize(s->stream);
			cudaFree(s->gpu_workspace);
		}
		s->gpu_workspace = 0;
		s->gpu_workspace_size = 0;
		const size_t rounded = (workspace_size + (1 << 20) - 1) & ~(size_t)((1 << 20) - 1);
		const cudaError_t e = cudaMalloc(&s->gpu_workspace, rounded);
		if (e != cudaSuccess)
		{
			sm100::set_last_error("cudaMalloc(workspace)", e);
			return 0;
		}
		s->gpu_workspace_size = rounded;
	}
	return s->gpu_workspace;
}

void ccv_nnc_stream_context_drain(ccv_nnc_stream_context_t* const stream_context)
{
	if (!stream_context)
		return;
	if (stream_context->gpu_workspace)
	{
		cudaStreamSynchronize(stream_context->stream);
		cudaFree(stream_context->gpu_workspace);
		stream_context->gpu_workspace = 0;
		stream_context->gpu_workspace_size = 0;
	}
	free(stream_context->cpu_workspace);
	stream_context->cpu_workspace = 0;
	stream_context->cpu_workspace_size = 0;
}

void ccv_nnc_stream_context_wait(const ccv_nnc_stream_context_t* const stream_context)
{
	if (!stream_context)
	{
		int device = 0;
		cudaGetDevice(&device);
		cudaStreamSynchronize(default_stream(device)->stream);
		return;
	}
	if (CCV_STREAM_GET_CONTEXT(stream_context->type) == CCV_STREAM_CONTEXT_GPU)
	{
		const cudaError_t e = cudaStreamSynchronize(stream_context->stream);
		if (e != cudaSuccess)
			sm100::set_last_error("cudaStreamSynchronize", e);
	}
}

void ccv_nnc_stream_context_free(ccv_nnc_stream_context_t* const stream_context)
{
	if (!stream_context)
		return;
	ccv_nnc_stream_context_drain(stream_context);
	if (stream_context->stream)
		cudaStreamDestroy(stream_context->stream);
	free(stream_context);
}

int ccv_nnc_device_count(const int type)
{
	if (CCV_STREAM_GET_CONTEXT(type) != CCV_STREAM_CONTEXT_GPU)
		return 1;
	int count = 0;
	if (cudaGetDeviceCount(&count) != cudaSuccess)
	{
		cudaGetLastError();
		return 0;
	}
	return count;
}

// lib/nnc/ccv_nnc.h:1022-1064 / lib/nnc/ccv_nnc_stream.c: stream signals = CUDA events (no timing) that one stream emits and
// another waits for, without blocking the host -- how the reference's graph runner orders work across streams.
struct ccv_nnc_stream_signal_s {
	int type;
	cudaEvent_t event;
	ccv_nnc_stream_context_t* emitter;
};

ccv_nnc_stream_signal_t* ccv_nnc_stream_signal_new(const int type)
{
	ccv_nnc_stream_signal_t* const signal = (ccv_nnc_stream_signal_t*)calloc(1, sizeof(ccv_nnc_stream_signal_t));
	signal->type = type;
	if (CCV_STREAM_GET_CONTEXT(type) == CCV_STREAM_CONTEXT_GPU)
	{
		cudaSetDevice(CCV_STREAM_GET_DEVICE_ID(type));
		if (cudaEventCreateWithFlags(&signal->event, cudaEventDisableTiming) != cudaSuccess)
		{
			free(signal);
			return 0;
		}
	}
	return signal;
}

int ccv_nnc_stream_signal_type(const ccv_nnc_stream_signal_t* const signal) { return signal->type; }

void ccv_nnc_stream_context_emit_signal(ccv_nnc_stream_context_t* const stream, ccv_nnc_stream_signal_t* const signal)
{
	signal->emitter = stream;
	if (signal->event)
		cudaEventRecord(signal->event, (cudaStream_t)ccv_nnc_stream_context_get_stream(stream));
}

void ccv_nnc_stream_context_wait_signal(const ccv_nnc_stream_context_t* const stream, const ccv_nnc_stream_signal_t* const signal)
{
	if (signal->event)
		cudaStreamWaitEvent((cudaStream_t)ccv_nnc_stream_context_get_stream(stream), signal->event, 0);
}

ccv_nnc_stream_context_t* ccv_nnc_stream_signal_get_emitter(const ccv_nnc_stream_signal_t* const signal) { return signal->emitter; }

void ccv_nnc_stream_signal_free(ccv_nnc_stream_signal_t* const signal)
{
	if (!signal)
		return;
	if (signal->event)
		cudaEventDestroy(signal->event);
	free(signal);
}

void ccv_nnc_stream_context_set_neighbor_discovery(ccv_nnc_stream_context_t* const stream_context, ccv_nnc_stream_context_neighbor_discovery_f discovery, void* const context)
{
	stream_context->neighbor_discovery = discovery;
	stream_context->neighbor_discovery_context = context;
}

ccv_nnc_stream_context_t* ccv_nnc_stream_context_find_neighbor(ccv_nnc_stream_context_t* const stream_context, const int device_id)
{
	if (stream_context->device == device_id)
		return stream_context;
	if (stream_context->neighbor_discovery)
		return stream_context->neighbor_discovery(device_id, stream_context->neighbor_discovery_context);
	return 0;
}

// ---------------------------------------------------------------------------------------------------- FFI helpers
// lib/nnc/ccv_nnc_cmd.c:399-600 reduced to the one backend this host carries: ask the backend's autotune function (if the command has
// one and more than one algorithm) which algorithm to use for these operands; inputs / outputs are used as scratch exactly as
// the reference uses its copies.  Returns the command with .backend and .algorithm filled in.
ccv_nnc_cmd_t ccv_nnc_cmd_autotune(const ccv_nnc_cmd_t cmd, const size_t max_workspace_size, const ccv_nnc_hint_t hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	ccv_nnc_init();
	ccv_nnc_cmd_t tuned = cmd;
	const ccv_nnc_cmd_backend_registry_t* const reg = registry_of(cmd.cmd, CCV_NNC_BACKEND_GPU_SM100);
	if (!reg || !reg->exec)
		return tuned;
	tuned.backend = CCV_NNC_BACKEND_GPU_SM100;
	if (reg->algorithms <= 1)
	{
		tuned.algorithm = 0;
		return tuned;
	}
	if (reg->autotune)
		tuned.algorithm = reg->autotune(tuned, max_workspace_size, hint, flags, inputs, input_size, outputs, output_size, stream_context);
	return tuned;
}

void ccv_nnc_sm100_cmd_autotune(const uint32_t cmd, const ccv_nnc_cmd_param_t* const info, const ccv_nnc_hint_t* const hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context, int* const algorithm)
{
	ccv_nnc_cmd_t c = ccv_nnc_cmd(cmd, 0, *info, 0);
	c.backend = CCV_NNC_BACKEND_GPU_SM100;
	c.algorithm = -1;
	*algorithm = ccv_nnc_cmd_autotune(c, 0, *hint, flags, inputs, input_size, outputs, output_size, stream_context).algorithm;
}

int ccv_nnc_sm100_cmd_exec(const uint32_t cmd, const uint32_t backend, const int algorithm, const ccv_nnc_cmd_param_t* const info, const ccv_nnc_hint_t* const hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size, ccv_nnc_stream_context_t* const stream_context)
{
	ccv_nnc_cmd_t c = ccv_nnc_cmd(cmd, 0, *info, 0);
	c.backend = backend;
	c.algorithm = algorithm;
	return ccv_nnc_cmd_exec(c, *hint, flags, inputs, input_size, outputs, output_size, stream_context);
}

ccv_nnc_tensor_t* ccv_nnc_sm100_tensor_new(const void* const ptr, const ccv_nnc_tensor_param_t* const params)
{
	return ccv_nnc_tensor_new(ptr, *params, 0);
}

ccv_nnc_tensor_view_t* ccv_nnc_sm100_tensor_view_new(const ccv_nnc_tensor_t* const tensor, const ccv_nnc_tensor_param_t* const params, const int* const ofs, const int* const stride)
{
	return ccv_nnc_tensor_view_new(tensor, *params, ofs, stride);
}

void ccv_nnc_sm100_hint_auto(const ccv_nnc_cmd_param_t* const info, const ccv_nnc_tensor_param_t* const a, const ccv_nnc_tensor_param_t* const b, ccv_nnc_hint_t* const hint)
{
	*hint = ccv_nnc_hint_auto(*info, *a, *b);
}

int ccv_nnc_sm100_memcpy_h2d(void* const dst_device, const void* const src_host, const size_t bytes, ccv_nnc_stream_context_t* const stream_context)
{
	cudaStream_t stream = (cudaStream_t)ccv_nnc_stream_context_get_stream(stream_context);
	cudaError_t e = cudaMemcpyAsync(dst_device, src_host, bytes, cudaMemcpyHostToDevice, stream);
	if (e == cudaSuccess)
		e = cudaStreamSynchronize(stream);
	if (e != cudaSuccess)
	{
		sm100::set_last_error("memcpy_h2d", e);
		return -1;
	}
	return 0;
}

int ccv_nnc_sm100_memcpy_d2h(void* const dst_host, const void* const src_device, const size_t bytes, ccv_nnc_stream_context_t* const stream_context)
{
	cudaStream_t stream = (cudaStream_t)ccv_nnc_stream_context_get_stream(stream_context);
	cudaError_t e = cudaMemcpyAsync(dst_host, src_device, bytes, cudaMemcpyDeviceToHost, stream);
	if (e == cudaSuccess)
		e = cudaStreamSynchronize(stream);
	if (e != cudaSuccess)
	{
		sm100::set_last_error("memcpy_d2h", e);
		return -1;
	}
	return 0;
}

// CUDA-event timing on a stream context's stream (device time, the way every number in bench.py is taken)
void* ccv_nnc_sm100_event_new(void)
{
	cudaEvent_t e = 0;
	if (cudaEventCreate(&e) != cudaSuccess)
		return 0;
	return (void*)e;
}

int ccv_nnc_sm100_event_record(void* const event, ccv_nnc_stream_context_t* const stream_context)
{
	return cudaEventRecord((cudaEvent_t)event, (cudaStream_t)ccv_nnc_stream_context_get_stream(stream_context)) == cudaSuccess ? 0 : -1;
}

float ccv_nnc_sm100_event_elapsed_ms(void* const begin, void* const end)
{
	float ms = -1.f;
	if (cudaEventSynchronize((cudaEvent_t)end) != cudaSuccess)
		return -1.f;
	if (cudaEventElapsedTime(&ms, (cudaEvent_t)begin, (cudaEvent_t)end) != cudaSuccess)
		return -1.f;
	return ms;
}

void ccv_nnc_sm100_event_free(void* const event)
{
	if (event)
		cudaEventDestroy((cudaEvent_t)event);
}

uint64_t ccv_nnc_sm100_launch_count(void)
{
	return (uint64_t)sm100::launch_count();
}

const char* ccv_nnc_sm100_last_error(void)
{
	return sm100::last_error();
}

// ---------------------------------------------------------------------------------------------------- flat graph
} // extern "C"

struct ccv_nnc_sm100_graph_node_t {
	ccv_nnc_cmd_t cmd;
	ccv_nnc_hint_t hint;
	int flags;
	std::vector<ccv_nnc_tensor_t*> inputs, outputs;
	ccv_nnc_cmd_exec_f fused; // non-NULL: a fused pair installed by ccv_nnc_sm100_graph_fuse, called instead of ccv_nnc_cmd_exec
	int side;                 // 1: issued on the graph's side stream context (ccv_nnc_sm100_graph_exec_set_side_stream)
};

extern "C" {
int ccv_nnc_sm100_fused_bn_relu_forw(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_fused_relu_bn_back(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_fused_add_relu_forw(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_fused_add_relu_back(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_fused_sgd_multi(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_fused_conv_stats_forw(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_fused_bn_forw(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_fused_bn_back(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_fused_bn_add_relu_forw(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
int ccv_nnc_sm100_fused_add_relu_back_stats(const ccv_nnc_cmd_t, const ccv_nnc_hint_t, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_tensor_t* const*, const int, ccv_nnc_stream_context_t*);
}

struct ccv_nnc_sm100_graph_s {
	std::vector<ccv_nnc_sm100_graph_node_t> nodes;
	std::vector<cudaGraphExec_t> captures;
	std::vector<ccv_nnc_tensor_t*> owned; // small tensors the fusion rewrites pass between the two nodes of a pair (statistics, coefficients)
	// second stream context for nodes marked `side` (gradient-exchange commands that overlap the rest of the backward pass), on the
	// device of the stream the graph runs on; two reusable signals order it with the main stream (what the reference's graph
	// runner does with per-node wait / emit signals across its streams, lib/nnc/ccv_nnc_graph_run.c:451-543)
	ccv_nnc_stream_context_t* side_stream;
	ccv_nnc_stream_signal_t* fork_signal;
	ccv_nnc_stream_signal_t* join_signal;
	ccv_nnc_sm100_graph_s() : side_stream(0), fork_signal(0), join_signal(0) {}
};

extern "C" {

ccv_nnc_sm100_graph_t* ccv_nnc_sm100_graph_new(void)
{
	return new ccv_nnc_sm100_graph_s();
}

int ccv_nnc_sm100_graph_exec_new(ccv_nnc_sm100_graph_t* const graph, const uint32_t cmd, const uint32_t backend, const int algorithm, const ccv_nnc_cmd_param_t* const info, const ccv_nnc_hint_t* const hint, const int flags, ccv_nnc_tensor_t* const* const inputs, const int input_size, ccv_nnc_tensor_t* const* const outputs, const int output_size)
{
	ccv_nnc_sm100_graph_node_t node;
	node.cmd = ccv_nnc_cmd(cmd, 0, *info, 0);
	node.cmd.backend = backend;
	node.cmd.algorithm = algorithm;
	node.hint = *hint;
	node.flags = flags;
	node.inputs.assign(inputs, inputs + input_size);
	node.outputs.assign(outputs, outputs + output_size);
	node.fused = 0;
	node.side = 0;
	graph->nodes.push_back(node);
	return (int)graph->nodes.size() - 1;
}

// Marks node `i` as asynchronous to the main stream: when the runner reaches it, the side stream waits for everything issued
// on the main stream so far, the node is issued on the side stream, and the main stream carries on; the main stream waits for the
// side stream in front of the first later node that reads or writes memory the side node writes, and at the end of the run (or
// of the captured CUDA graph) at the latest.  For commands whose results are only needed after the run -- the
// COMM_ALLREDUCE of a gradient bucket that is complete while the rest of the backward pass still computes
// (lib/nnc/ccv_nnc_symbolic_graph_parallel.c:546-575 places its allreduce nodes the same way, one stream per device).
int ccv_nnc_sm100_graph_exec_set_side_stream(ccv_nnc_sm100_graph_t* const graph, const int i, const int side)
{
	if (i < 0 || i >= (int)graph->nodes.size() || !graph->captures.empty())
		return -1;
	graph->nodes[i].side = side ? 1 : 0;
	return 0;
}

int ccv_nnc_sm100_graph_size(const ccv_nnc_sm100_graph_t* const graph)
{
	return (int)graph->nodes.size();
}

int ccv_nnc_sm100_graph_run(ccv_nnc_sm100_graph_t* const graph, const int begin, const int end, ccv_nnc_stream_context_t* const stream_context)
{
	// lib/nnc/ccv_nnc_graph_run.c:911-979: for each exec in topological order: ccv_nnc_cmd_exec(...); non-zero is reported, not fatal
	int status = 0, i;
	const int last = end < 0 || end > (int)graph->nodes.size() ? (int)graph->nodes.size() : end;
	bool side_pending = false;
	// byte ranges written by side-stream nodes that have not been joined yet: a main-stream node that touches one of them is a
	// consumer (or an overwriter) of that result, so the join is issued in front of it instead of at the end of the run
	std::vector<std::pair<const unsigned char*, const unsigned char*> > side_writes;
	auto range_of = [](const ccv_nnc_tensor_t* const t) {
		size_t elems = 1;
		if (CCV_IS_TENSOR_VIEW(t))
		{
			const ccv_nnc_tensor_view_t* const tv = (const ccv_nnc_tensor_view_t*)t;
			for (int d = 0; d < CCV_NNC_MAX_DIM_ALLOC && t->info.dim[d] > 0; d++)
				elems += (size_t)(t->info.dim[d] - 1) * (size_t)tv->stride[d];
		} else
			for (int d = 0; d < CCV_NNC_MAX_DIM_ALLOC && t->info.dim[d] > 0; d++)
				elems *= (size_t)t->info.dim[d];
		return std::make_pair((const unsigned char*)t->data.u8, (const unsigned char*)t->data.u8 + elems * datatype_size(t->info.datatype));
	};
	auto join = [&]() {
		ccv_nnc_stream_context_emit_signal(graph->side_stream, graph->join_signal);
		ccv_nnc_stream_context_wait_signal(stream_context, graph->join_signal);
		side_pending = false;
		side_writes.clear();
	};
	for (i = begin < 0 ? 0 : begin; i < last; i++)
	{
		ccv_nnc_sm100_graph_node_t& n = graph->nodes[i];
		ccv_nnc_stream_context_t* sc = stream_context;
		if (side_pending && !n.side)
		{
			bool touches = false;
			for (int pass = 0; pass < 2 && !touches; pass++)
				for (ccv_nnc_tensor_t* t : (pass ? n.outputs : n.inputs))
					if (t && t->data.u8)
					{
						const auto r = range_of(t);
						for (const auto& w : side_writes)
							if (r.first < w.second && w.first < r.second)
								touches = true;
					}
			if (touches)
				join();
		}
		if (n.side && stream_context && CCV_STREAM_GET_CONTEXT(stream_context->type) == CCV_STREAM_CONTEXT_GPU)
		{
			if (!graph->side_stream || graph->side_stream->device != stream_context->device)
			{
				if (graph->side_stream)
					ccv_nnc_stream_context_free(graph->side_stream);
				if (graph->fork_signal)
					ccv_nnc_stream_signal_free(graph->fork_signal), ccv_nnc_stream_signal_free(graph->join_signal);
				graph->side_stream = ccv_nnc_stream_context_new(stream_context->type);
				graph->fork_signal = ccv_nnc_stream_signal_new(stream_context->type);
				graph->join_signal = ccv_nnc_stream_signal_new(stream_context->type);
			}
			if (graph->side_stream && graph->fork_signal && graph->join_signal)
			{
				// fork: the side stream sees everything the main stream has been given so far
				ccv_nnc_stream_context_emit_signal(stream_context, graph->fork_signal);
				ccv_nnc_stream_context_wait_signal(graph->side_stream, graph->fork_signal);
				sc = graph->side_stream;
				side_pending = true;
				for (ccv_nnc_tensor_t* t : n.outputs)
					if (t && t->data.u8)
						side_writes.push_back(range_of(t));
			}
		}
		const int ret = n.fused ? n.fused(n.cmd, n.hint, n.flags, n.inputs.data(), (int)n.inputs.size(), n.outputs.data(), (int)n.outputs.size(), sc) :
			ccv_nnc_cmd_exec(n.cmd, n.hint, n.flags, n.inputs.data(), (int)n.inputs.size(), n.outputs.data(), (int)n.outputs.size(), sc);
		if (ret != 0 && status == 0)
		{
			fprintf(stderr, "[ccv_nnc_sm100] graph node %d (cmd 0x%08x) returned %d\n", i, n.cmd.cmd, ret);
			status = ret;
		}
	}
	if (side_pending)
		join(); // whatever runs after this graph on the main stream is ordered behind the side stream's commands
	return status;
}

// Peephole fusion over adjacent nodes (the "fusion of adjacent nodes" item of the graph-runner launch path, SURVEY.md 8f-2).
// Every rewrite keeps the tensors the pair would have written, except the in-place intermediate of (b) and (d):
//  (a) BATCH_NORM_FORWARD(train) ; RELU_FORWARD in place on its output      -> one pass writes relu(bn(x))
//  (b) RELU_BACKWARD in place on g (mask y) ; BATCH_NORM_BACKWARD(g, x = bn input of y) -> mask recomputed from x; g is left
//      unmasked, so the rewrite is only applied when no later node reads g
//  (c) EWSUM(a, b -> y) ; RELU_FORWARD in place on y                          -> y = relu(a + b)
//  (d) EWSUM(a, b -> a) ; RELU_BACKWARD in place on a (mask y)                -> a = y > 0 ? a + b : 0
//  (e) a run of SGD_FORWARD nodes with identical parameters (the per-parameter updates of a model; none of them reads
//      what another one writes) -> one multi-tensor command; counts as (run length - 1) fused nodes
// (f) - (i) below pair nodes without removing either.
int ccv_nnc_sm100_graph_fuse(ccv_nnc_sm100_graph_t* const graph)
{
	std::vector<ccv_nnc_sm100_graph_node_t>& nodes = graph->nodes;
	if (!graph->captures.empty())
		return -1;
	std::vector<ccv_nnc_sm100_graph_node_t> out;
	int fused = 0;
	const size_t n = nodes.size();
	auto is_gpu_sm100 = [](const ccv_nnc_sm100_graph_node_t& x) { return x.fused == 0 && !x.side && (x.cmd.backend == CCV_NNC_BACKEND_GPU_SM100 || x.cmd.backend == CCV_NNC_NO_BACKEND); };
	for (size_t i = 0; i < n; i++)
	{
		ccv_nnc_sm100_graph_node_t& a = nodes[i];
		// (e)
		if (is_gpu_sm100(a) && a.cmd.cmd == CCV_NNC_SGD_FORWARD && a.inputs.size() == 3 && a.outputs.size() == 2)
		{
			size_t j = i + 1;
			auto independent = [&](const ccv_nnc_sm100_graph_node_t& x, size_t from, size_t to) {
				// x must not read anything the nodes [from, to) write (in-place a -> b, m -> n of the SAME node is fine)
				for (size_t k = from; k < to; k++)
					for (ccv_nnc_tensor_t* o : nodes[k].outputs)
						for (ccv_nnc_tensor_t* in : x.inputs)
							if (o == in || (o && in && o->data.u8 == in->data.u8))
								return false;
				return true;
			};
			// the maximal run of mutually independent SGD nodes: inside it the order is free, so nodes are grouped by their
			// hyper-parameters (weights with decay, biases / norm parameters without) even when the groups interleave
			while (j < n && is_gpu_sm100(nodes[j]) && nodes[j].cmd.cmd == CCV_NNC_SGD_FORWARD && nodes[j].inputs.size() == 3 && nodes[j].outputs.size() == 2 && independent(nodes[j], i, j))
				j++;
			std::vector<char> done(j - i, 0);
			for (size_t k = i; k < j; k++)
			{
				if (done[k - i])
					continue;
				ccv_nnc_sm100_graph_node_t f = nodes[k];
				int members = 1;
				for (size_t q = k + 1; q < j; q++)
					if (!done[q - i] && memcmp(&nodes[q].cmd.info.sgd, &f.cmd.info.sgd, sizeof(f.cmd.info.sgd)) == 0 && nodes[q].flags == f.flags && nodes[q].cmd.algorithm == f.cmd.algorithm &&
					nodes[q].inputs[0] && f.inputs[0] && nodes[q].inputs[0]->info.datatype == f.inputs[0]->info.datatype) // one gradient type per launch (16-bit and fp32 gradients of a mixed-precision model go separately)
					{
						f.inputs.insert(f.inputs.end(), nodes[q].inputs.begin(), nodes[q].inputs.end());
						f.outputs.insert(f.outputs.end(), nodes[q].outputs.begin(), nodes[q].outputs.end());
						done[q - i] = 1;
						members++;
					}
				if (members > 1)
				{
					f.fused = ccv_nnc_sm100_fused_sgd_multi;
					fused += members - 1;
				}
				out.push_back(f);
			}
			i = j - 1;
			continue;
		}
		if (i + 1 < n && is_gpu_sm100(a) && is_gpu_sm100(nodes[i + 1]))
		{
			ccv_nnc_sm100_graph_node_t& b = nodes[i + 1];
			// (a)
			if (a.cmd.cmd == CCV_NNC_BATCH_NORM_FORWARD && !a.cmd.info.bnorm.is_test && a.outputs.size() == 5 && b.cmd.cmd == CCV_NNC_RELU_FORWARD && b.inputs.size() == 1 && b.outputs.size() == 1 &&
				b.inputs[0] == a.outputs[0] && b.outputs[0] == a.outputs[0])
			{
				ccv_nnc_sm100_graph_node_t f = a;
				f.fused = ccv_nnc_sm100_fused_bn_relu_forw;
				out.push_back(f);
				fused++, i++;
				continue;
			}
			// (c)
			if (a.cmd.cmd == CCV_NNC_EWSUM_FORWARD && a.inputs.size() == 2 && a.outputs.size() == 1 && b.cmd.cmd == CCV_NNC_RELU_FORWARD && b.inputs.size() == 1 && b.inputs[0] == a.outputs[0] && b.outputs[0] == a.outputs[0])
			{
				ccv_nnc_sm100_graph_node_t f = a;
				f.fused = ccv_nnc_sm100_fused_add_relu_forw;
				out.push_back(f);
				fused++, i++;
				continue;
			}
			// (d)
			if (a.cmd.cmd == CCV_NNC_EWSUM_FORWARD && a.inputs.size() == 2 && a.outputs.size() == 1 && a.outputs[0] == a.inputs[0] && b.cmd.cmd == CCV_NNC_RELU_BACKWARD && b.inputs.size() == 3 && b.inputs[0] == a.outputs[0] &&
				b.outputs.size() == 1 && b.outputs[0] == a.outputs[0] && b.inputs[2])
			{
				ccv_nnc_sm100_graph_node_t f = a;
				f.inputs.push_back(b.inputs[2]);
				f.fused = ccv_nnc_sm100_fused_add_relu_back;
				out.push_back(f);
				fused++, i++;
				continue;
			}
			// (b)
			if (a.cmd.cmd == CCV_NNC_RELU_BACKWARD && a.inputs.size() == 3 && a.outputs.size() == 1 && a.outputs[0] == a.inputs[0] && a.inputs[2] && b.cmd.cmd == CCV_NNC_BATCH_NORM_BACKWARD && b.inputs.size() == 15 &&
				b.inputs[0] == a.outputs[0] && b.inputs[5] && !b.inputs[7])
			{
				// the forward batch norm that produced the mask tensor from this x supplies the bias
				ccv_nnc_tensor_t* bias = 0;
				for (size_t j = 0; j < n && !bias; j++)
					if (nodes[j].cmd.cmd == CCV_NNC_BATCH_NORM_FORWARD && nodes[j].inputs.size() == 5 && nodes[j].outputs.size() >= 1 && nodes[j].outputs[0] == a.inputs[2] && nodes[j].inputs[0] == b.inputs[5] && nodes[j].inputs[1] == b.inputs[6])
						bias = nodes[j].inputs[2];
				bool g_read_later = false;
				for (size_t j = i + 2; j < n && !g_read_later; j++)
					for (ccv_nnc_tensor_t* t : nodes[j].inputs)
						if (t == a.outputs[0] || (t && a.outputs[0] && t->data.u8 && t->data.u8 == a.outputs[0]->data.u8)) // the same memory through another tensor / view counts
						{
							// a later node that overwrites g before reading it would be fine, but keep the rule simple
							g_read_later = true;
							break;
						}
				if (bias && !g_read_later)
				{
					ccv_nnc_sm100_graph_node_t f = b;
					f.inputs[7] = bias;
					f.fused = ccv_nnc_sm100_fused_relu_bn_back;
					out.push_back(f);
					fused++, i++;
					continue;
				}
			}
		}
		out.push_back(a);
	}
	// (f) CONVOLUTION_FORWARD ; BATCH_NORM_FORWARD(train) (plain or already fused with its ReLU) reading the convolution's output:
	//     the convolution's tensor-core epilogue also produces the per-channel sums the batch norm needs, through a small
	//     statistics tensor owned by the graph (one fewer pass over the activation).  CCV_NNC_SM100_FUSE_CONV_BN=0 turns it off.
	const char* const env = getenv("CCV_NNC_SM100_FUSE_CONV_BN");
	if (!env || atoi(env) != 0)
		for (size_t i = 0; i + 1 < out.size(); i++)
		{
			ccv_nnc_sm100_graph_node_t& c = out[i];
			ccv_nnc_sm100_graph_node_t& b = out[i + 1];
			if (c.fused || c.cmd.cmd != CCV_NNC_CONVOLUTION_FORWARD || c.outputs.size() != 1 || !c.outputs[0] || c.cmd.algorithm == CCV_NNC_SM100_ALGO_FFMA || c.cmd.info.convolution.groups != 1)
				continue;
			if (b.cmd.cmd != CCV_NNC_BATCH_NORM_FORWARD || b.cmd.info.bnorm.is_test || b.inputs.size() != 5 || b.inputs[0] != c.outputs[0] || (b.fused && b.fused != ccv_nnc_sm100_fused_bn_relu_forw))
				continue;
			if (CCV_IS_TENSOR_VIEW(c.outputs[0]) || CCV_TENSOR_GET_MEMORY(c.outputs[0]->info.type) != CCV_TENSOR_GPU_MEMORY)
				continue;
			const int K = c.cmd.info.convolution.count;
			ccv_nnc_tensor_param_t params = c.outputs[0]->info;
			memset(params.dim, 0, sizeof(params.dim));
			params.dim[0] = 4 * 4 * 160, params.dim[1] = K; // four planes (count, shift, sum, sum of squares) of >= 4 rows per SM
			params.datatype = CCV_32F;
			ccv_nnc_tensor_t* const stats = ccv_nnc_tensor_new(0, params, 0);
			if (!stats || !stats->data.u8)
				continue;
			stats->sig = 0;
			graph->owned.push_back(stats);
			c.outputs.push_back(stats);
			c.fused = ccv_nnc_sm100_fused_conv_stats_forw;
			b.inputs.push_back(stats);
			if (!b.fused)
				b.fused = ccv_nnc_sm100_fused_bn_forw;
			// no node is removed by this rewrite: the return value keeps counting removed nodes only
		}
	// (g) BATCH_NORM_BACKWARD (plain or fused with the ReLU backward in front) ; CONVOLUTION_BACKWARD whose incoming gradient is the
	//     dx of that batch norm and which wants a bias gradient: the batch norm's apply pass sums the dx it writes per channel and
	//     stores the convolution's dbias directly; the convolution skips its column-sum pass over dx.
	if (!env || atoi(env) != 0)
		for (size_t i = 0; i + 1 < out.size(); i++)
		{
			ccv_nnc_sm100_graph_node_t& b = out[i];
			ccv_nnc_sm100_graph_node_t& c = out[i + 1];
			if (b.cmd.cmd != CCV_NNC_BATCH_NORM_BACKWARD || (b.fused && b.fused != ccv_nnc_sm100_fused_relu_bn_back) || b.outputs.size() != 3 || !b.outputs[0])
				continue;
			if (c.fused || c.cmd.cmd != CCV_NNC_CONVOLUTION_BACKWARD || (c.flags & CCV_NNC_ACCUMULATE_OUTPUT) || c.inputs.empty() || c.inputs[0] != b.outputs[0] || c.outputs.size() < 3 || !c.outputs[2])
				continue;
			if (CCV_IS_TENSOR_VIEW(c.outputs[2]) || CCV_IS_TENSOR_VIEW(b.outputs[0]))
				continue;
			b.outputs.push_back(c.outputs[2]);
			c.outputs[2] = 0;
			if (!b.fused)
				b.fused = ccv_nnc_sm100_fused_bn_back;
		}
	// The end of a residual block: the last batch norm of the main branch (no ReLU), the shortcut add and the ReLU.
	// CCV_NNC_SM100_FUSE_BLOCK_END=0 turns (h) and (i) off.  Neither removes a node.
	const char* const env_end = getenv("CCV_NNC_SM100_FUSE_BLOCK_END");
	const bool block_end = !env_end || atoi(env_end) != 0;
	auto same_mem = [](const ccv_nnc_tensor_t* const x, const ccv_nnc_tensor_t* const y) { return x == y || (x && y && x->data.u8 && x->data.u8 == y->data.u8); };
	auto plain_node = [](const ccv_nnc_sm100_graph_node_t& x) { return !x.side && (x.cmd.backend == CCV_NNC_BACKEND_GPU_SM100 || x.cmd.backend == CCV_NNC_NO_BACKEND); };
	// the batch norm normalises the innermost dimension of a packed GPU tensor (NHWC): C of it, or 0
	auto nhwc_channels = [](const ccv_nnc_tensor_t* const x, const ccv_nnc_tensor_t* const scale) {
		if (!x || !scale || CCV_IS_TENSOR_VIEW(x) || CCV_IS_TENSOR_VIEW(scale) || CCV_TENSOR_GET_MEMORY(x->info.type) != CCV_TENSOR_GPU_MEMORY)
			return 0;
		int nd = 0;
		size_t count = 1;
		while (nd < CCV_NNC_MAX_DIM_ALLOC && scale->info.dim[nd] > 0)
			count *= (size_t)scale->info.dim[nd++];
		if (nd == 0 || (size_t)scale->info.dim[nd - 1] != count)
			return 0;
		int xnd = 0;
		while (xnd < CCV_NNC_MAX_DIM_ALLOC && x->info.dim[xnd] > 0)
			xnd++;
		return xnd > 0 && x->info.dim[xnd - 1] == (int)count ? (int)count : 0;
	};
	auto owned_f32 = [&](const ccv_nnc_tensor_t* const like, const int rows, const int cols) -> ccv_nnc_tensor_t* {
		ccv_nnc_tensor_param_t params = like->info;
		memset(params.dim, 0, sizeof(params.dim));
		params.dim[0] = rows, params.dim[1] = cols;
		params.datatype = CCV_32F;
		ccv_nnc_tensor_t* const t = ccv_nnc_tensor_new(0, params, 0);
		if (!t || !t->data.u8)
		{
			if (t)
				ccv_nnc_tensor_free(t);
			return 0;
		}
		t->sig = 0;
		graph->owned.push_back(t);
		return t;
	};
	// (h) BATCH_NORM_FORWARD(train, no ReLU; plain or reading convolution statistics) ; the fused add + ReLU (c) whose first operand
	//     is the batch norm's output y, which no later node reads: the batch norm only computes the statistics and leaves its
	//     per-channel a, b in a [2, C] tensor owned by the graph; the add node computes relu(x * a + b + shortcut) from the batch
	//     norm's input x.  y is never written (one write and one read of the activation fewer).
	if (block_end)
		for (size_t i = 0; i + 1 < out.size(); i++)
		{
			ccv_nnc_sm100_graph_node_t& b = out[i];
			ccv_nnc_sm100_graph_node_t& e = out[i + 1];
			if (!plain_node(b) || b.cmd.cmd != CCV_NNC_BATCH_NORM_FORWARD || b.cmd.info.bnorm.is_test || (b.fused && b.fused != ccv_nnc_sm100_fused_bn_forw) || (b.inputs.size() != 5 && b.inputs.size() != 6) || b.outputs.size() != 5 || !b.outputs[0])
				continue;
			if (!plain_node(e) || e.fused != ccv_nnc_sm100_fused_add_relu_forw || e.inputs.size() != 2 || e.inputs[0] != b.outputs[0] || same_mem(e.inputs[1], b.outputs[0]) || same_mem(e.outputs[0], b.outputs[0]))
				continue;
			const int C = nhwc_channels(b.inputs[0], b.inputs[1]);
			if (!C)
				continue;
			bool y_read_later = false;
			for (size_t j = i + 2; j < out.size() && !y_read_later; j++)
				for (ccv_nnc_tensor_t* t : out[j].inputs)
					if (same_mem(t, b.outputs[0]))
					{
						y_read_later = true;
						break;
					}
			if (y_read_later)
				continue;
			ccv_nnc_tensor_t* const coef = owned_f32(b.inputs[1], 2, C);
			if (!coef)
				continue;
			b.outputs.push_back(coef);
			if (!b.fused)
				b.fused = ccv_nnc_sm100_fused_bn_forw;
			e.inputs[0] = b.inputs[0];
			e.inputs.push_back(coef);
			e.fused = ccv_nnc_sm100_fused_bn_add_relu_forw;
		}
	// (i) the fused add + ReLU backward (d), or a RELU_BACKWARD left plain by (b) ; BATCH_NORM_BACKWARD (no ReLU; plain or with the
	//     convolution's bias gradient of (g)) of its output: the first node also produces the batch norm's reduction over (g, x)
	//     as per-block partial rows in a tensor owned by the graph; the batch norm only finalises and applies (one read of g fewer).
	if (block_end)
		for (size_t i = 0; i + 1 < out.size(); i++)
		{
			ccv_nnc_sm100_graph_node_t& r = out[i];
			ccv_nnc_sm100_graph_node_t& b = out[i + 1];
			if (!plain_node(r) || r.inputs.size() != 3 || r.outputs.size() != 1 || !r.inputs[0] || !r.inputs[2] || !r.outputs[0])
				continue;
			if (!(r.fused == ccv_nnc_sm100_fused_add_relu_back || (!r.fused && r.cmd.cmd == CCV_NNC_RELU_BACKWARD)))
				continue;
			if (!plain_node(b) || b.cmd.cmd != CCV_NNC_BATCH_NORM_BACKWARD || (b.fused && b.fused != ccv_nnc_sm100_fused_bn_back) || b.inputs.size() != 15 || b.inputs[0] != r.outputs[0] || b.inputs[7] || !b.inputs[5] || !b.inputs[13])
				continue;
			const int C = nhwc_channels(b.inputs[5], b.inputs[6]);
			if (!C)
				continue;
			// room for bn_reduce_kernel's grid rows: at most 4 per SM (reduce_config), for up to 160 SMs
			ccv_nnc_tensor_t* const part = owned_f32(b.inputs[13], 4 * 160 + 8, 2 * C);
			if (!part)
				continue;
			if (!r.fused) // RELU_BACKWARD (g, -, y): the add's second operand stays empty
				r.inputs[1] = 0;
			r.inputs.push_back(b.inputs[5]);
			r.inputs.push_back(b.inputs[13]);
			r.outputs.push_back(part);
			r.fused = ccv_nnc_sm100_fused_add_relu_back_stats;
			b.inputs.push_back(part);
			if (!b.fused)
				b.fused = ccv_nnc_sm100_fused_bn_back;
		}
	nodes.swap(out);
	return fused;
}

// introspection + per-node device timing (CUDA events around each node, best of `reps`), for bench.py's per-command table
int ccv_nnc_sm100_graph_node(const ccv_nnc_sm100_graph_t* const graph, const int i, uint32_t* const cmd, int* const fused_kind, int* const input_size, int* const output_size)
{
	if (i < 0 || i >= (int)graph->nodes.size())
		return -1;
	const ccv_nnc_sm100_graph_node_t& n = graph->nodes[i];
	*cmd = n.cmd.cmd;
	*fused_kind = n.fused == ccv_nnc_sm100_fused_bn_relu_forw ? 1 : n.fused == ccv_nnc_sm100_fused_relu_bn_back ? 2 : n.fused == ccv_nnc_sm100_fused_add_relu_forw || n.fused == ccv_nnc_sm100_fused_bn_add_relu_forw ? 3 : n.fused == ccv_nnc_sm100_fused_add_relu_back || n.fused == ccv_nnc_sm100_fused_add_relu_back_stats ? 4 : n.fused == ccv_nnc_sm100_fused_sgd_multi ? 5 : n.fused == ccv_nnc_sm100_fused_conv_stats_forw ? 6 : n.fused == ccv_nnc_sm100_fused_bn_forw ? 7 : n.fused == ccv_nnc_sm100_fused_bn_back ? 8 : 0;
	*input_size = (int)n.inputs.size();
	*output_size = (int)n.outputs.size();
	return 0;
}

void* ccv_nnc_sm100_graph_node_tensor(const ccv_nnc_sm100_graph_t* const graph, const int i, const int is_output, const int k)
{
	if (i < 0 || i >= (int)graph->nodes.size())
		return 0;
	const std::vector<ccv_nnc_tensor_t*>& v = is_output ? graph->nodes[i].outputs : graph->nodes[i].inputs;
	return k >= 0 && k < (int)v.size() ? (void*)v[k] : 0;
}

int ccv_nnc_sm100_graph_profile(ccv_nnc_sm100_graph_t* const graph, ccv_nnc_stream_context_t* const stream_context, const int reps, float* const ms)
{
	if (!stream_context)
		return -1;
	cudaEvent_t e0, e1;
	if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess)
		return -1;
	cudaStream_t stream = stream_context->stream;
	int status = 0;
	for (int i = 0; i < (int)graph->nodes.size(); i++)
	{
		if (graph->nodes[i].side || graph->nodes[i].cmd.cmd == CCV_NNC_COMM_ALLREDUCE_FORWARD || graph->nodes[i].cmd.cmd == CCV_NNC_COMM_ALLREDUCE_BACKWARD)
		{
			ms[i] = 0.f; // a collective cannot be timed by one rank on its own: every rank would have to issue it
			continue;
		}
		float best = 1e30f;
		for (int r = 0; r < (reps < 1 ? 1 : reps); r++)
		{
			cudaEventRecord(e0, stream);
			const int ret = ccv_nnc_sm100_graph_run(graph, i, i + 1, stream_context);
			cudaEventRecord(e1, stream);
			cudaEventSynchronize(e1);
			float t = 0;
			cudaEventElapsedTime(&t, e0, e1);
			if (t < best)
				best = t;
			if (ret != 0)
				status = ret;
		}
		ms[i] = best;
	}
	cudaEventDestroy(e0);
	cudaEventDestroy(e1);
	return status;
}

int ccv_nnc_sm100_graph_capture(ccv_nnc_sm100_graph_t* const graph, const int begin, const int end, ccv_nnc_stream_context_t* const stream_context)
{
	if (!stream_context)
		return -1;
	cudaStream_t stream = stream_context->stream;
	// one eager pass first: sizes the workspace (allocation is illegal during capture) and loads kernels
	int status = ccv_nnc_sm100_graph_run(graph, begin, end, stream_context);
	if (status != 0)
		return -1;
	if (cudaStreamSynchronize(stream) != cudaSuccess)
		return -1;
	cudaError_t e = cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal);
	if (e != cudaSuccess)
	{
		sm100::set_last_error("cudaStreamBeginCapture", e);
		return -1;
	}
	status = ccv_nnc_sm100_graph_run(graph, begin, end, stream_context);
	cudaGraph_t g = 0;
	e = cudaStreamEndCapture(stream, &g);
	if (e != cudaSuccess || status != 0 || !g)
	{
		sm100::set_last_error("cudaStreamEndCapture", e);
		if (g)
			cudaGraphDestroy(g);
		return -1;
	}
	cudaGraphExec_t ge = 0;
	e = cudaGraphInstantiate(&ge, g, 0);
	cudaGraphDestroy(g);
	if (e != cudaSuccess)
	{
		sm100::set_last_error("cudaGraphInstantiate", e);
		return -1;
	}
	graph->captures.push_back(ge);
	return (int)graph->captures.size() - 1;
}

int ccv_nnc_sm100_graph_replay(ccv_nnc_sm100_graph_t* const graph, const int capture_id, ccv_nnc_stream_context_t* const stream_context)
{
	if (capture_id < 0 || capture_id >= (int)graph->captures.size() || !stream_context)
		return -1;
	const cudaError_t e = cudaGraphLaunch(graph->captures[capture_id], stream_context->stream);
	if (e != cudaSuccess)
	{
		sm100::set_last_error("cudaGraphLaunch", e);
		return -1;
	}
	return 0;
}

void ccv_nnc_sm100_graph_free(ccv_nnc_sm100_graph_t* const graph)
{
	if (!graph)
		return;
	for (cudaGraphExec_t ge : graph->captures)
		cudaGraphExecDestroy(ge);
	for (ccv_nnc_tensor_t* t : graph->owned)
		ccv_nnc_tensor_free(t);
	if (graph->side_stream)
		ccv_nnc_stream_context_free(graph->side_stream);
	if (graph->fork_signal)
		ccv_nnc_stream_signal_free(graph->fork_signal);
	if (graph->join_signal)
		ccv_nnc_stream_signal_free(graph->join_signal);
	delete graph;
}

} // extern "C"
