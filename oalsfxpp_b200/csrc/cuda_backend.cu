// cuda_backend.cu -- the one Backend the product links: CUDA runtime + the sm_100a kernels.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false (no FMA contraction: parity
// with the CPU reference needs separate FMUL/FADD, SURVEY.md section 0 fact 5), IEEE div/sqrt and
// no flush-to-zero (nvcc defaults; -use_fast_math must never be passed).
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "backend.h"
#include "kernel_table.h"
#include "launch.h"

namespace oalsfx {
namespace {

__global__ void zero_lanes_kernel(uint32_t* base, long long tile_stride, int words, const TileRef* tiles)
{
	const TileRef t = tiles[blockIdx.y];
	const int lane = threadIdx.x % kLanes;
	if (!((t.mask >> lane) & 1U)) {
		return;
	}
	const int warps_per_block = blockDim.x / kLanes;
	uint32_t* p = base + static_cast<long long>(t.tile) * tile_stride + lane;
	for (int w = blockIdx.x * warps_per_block + threadIdx.x / kLanes; w < words; w += gridDim.x * warps_per_block) {
		p[static_cast<long long>(w) * kLanes] = 0U;
	}
}

// One block per (frame, channel) pair; threads stride over the streams in a fixed pattern and the
// partial sums are combined by a fixed shared-memory tree, so the result is deterministic.
__global__ void reduce_bus_kernel(const float* data, long long ts, long long ls, long long fs, long long cs,
	int num_streams, int channels, float* bus)
{
	__shared__ float partial[256];
	const int frame = blockIdx.x / channels;
	const int chan = blockIdx.x % channels;
	float sum = 0.0F;
	for (int s = threadIdx.x; s < num_streams; s += blockDim.x) {
		sum += data[(s / kLanes) * ts + (s % kLanes) * ls + frame * fs + chan * cs];
	}
	partial[threadIdx.x] = sum;
	__syncthreads();
	for (int stride = blockDim.x / 2; stride > 0; stride /= 2) {
		if (threadIdx.x < stride) {
			partial[threadIdx.x] += partial[threadIdx.x + stride];
		}
		__syncthreads();
	}
	if (threadIdx.x == 0) {
		bus[blockIdx.x] = partial[0];
	}
}

// ---- PCM formats either side of the path (SURVEY.md 8f rank 2) ---------------------------------------
// HBM-bound element-wise kernels: 16-byte accesses, grid-stride over a multiple of the SM count.
// FxDistortion::shape (fx.cuh) on plain arrays, four samples per call as in FxDistortion::step (test hook)
__global__ void __launch_bounds__(256) debug_waveshaper_kernel(const float* __restrict__ samples, float edge_coeff, float* __restrict__ out, long long count)
{
	const long long stride = static_cast<long long>(gridDim.x) * blockDim.x * 4;
	for (long long i = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4; i < count; i += stride) {
		float smp[4];
		for (int k = 0; k < 4; ++k) {
			smp[k] = samples[i + k < count ? i + k : count - 1];
		}
		FxDistortion::shape(smp, edge_coeff);
		for (int k = 0; k < 4; ++k) {
			if (i + k < count) {
				out[i + k] = smp[k];
			}
		}
	}
}

__global__ void __launch_bounds__(256) pcm16_to_float_kernel(const int16_t* __restrict__ src, float* __restrict__ dst, long long count, bool vector_ok)
{
	// reference: oalsfxpp_test.cpp:728-733  dst[i] = little(src[i]) / 32768.0F
	const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
	const long long vec = vector_ok ? count / 8 : 0;   // 16-byte accesses need 16-byte aligned buffers
	for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < vec; i += stride) {
		const int4 raw = __ldcs(reinterpret_cast<const int4*>(src) + i);
		const int w[4] = {raw.x, raw.y, raw.z, raw.w};
		float o[8];
#pragma unroll
		for (int k = 0; k < 4; ++k) {
			o[2 * k] = static_cast<float>(static_cast<int16_t>(w[k] & 0xFFFF)) / 32768.0F;
			o[2 * k + 1] = static_cast<float>(static_cast<int16_t>(static_cast<unsigned>(w[k]) >> 16)) / 32768.0F;
		}
		float4* out = reinterpret_cast<float4*>(dst) + 2 * i;
		__stcs(out, make_float4(o[0], o[1], o[2], o[3]));
		__stcs(out + 1, make_float4(o[4], o[5], o[6], o[7]));
	}
	for (long long i = vec * 8 + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += stride) {
		dst[i] = static_cast<float>(src[i]) / 32768.0F;
	}
}

__global__ void __launch_bounds__(256) pcm8_to_float_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst, long long count, bool vector_ok)
{
	// reference: oalsfxpp_test.cpp:714-719  dst[i] = (int(src[i]) - 128) / 128.0F
	const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
	const long long vec = vector_ok ? count / 4 : 0;
	for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < vec; i += stride) {
		const unsigned raw = __ldcs(reinterpret_cast<const unsigned*>(src) + i);
		float4 o;
		o.x = static_cast<float>(static_cast<int>(raw & 0xFFU) - 128) / 128.0F;
		o.y = static_cast<float>(static_cast<int>((raw >> 8) & 0xFFU) - 128) / 128.0F;
		o.z = static_cast<float>(static_cast<int>((raw >> 16) & 0xFFU) - 128) / 128.0F;
		o.w = static_cast<float>(static_cast<int>(raw >> 24) - 128) / 128.0F;
		__stcs(reinterpret_cast<float4*>(dst) + i, o);
	}
	for (long long i = vec * 4 + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += stride) {
		dst[i] = static_cast<float>(static_cast<int>(src[i]) - 128) / 128.0F;
	}
}

// One CTA per row (= one stream's buffer).  Pass 1: min / max of the row (the reference's scan,
// oalsfxpp_test.cpp:605-620: min starts at -1, max at +1; min and max are order-independent).  Pass 2:
// dst = int16(scale * x * 32767.0F), scale = 1 / max(max, -min) (oalsfxpp_test.cpp:622-640).  The second
// pass re-reads the row from L2 when it fits.
__global__ void __launch_bounds__(256) float_to_s16_kernel(const float* __restrict__ src, int16_t* __restrict__ dst, long long row_len,
	float* __restrict__ row_scale)
{
	__shared__ float lo_s[8], hi_s[8];
	const float* row = src + static_cast<long long>(blockIdx.x) * row_len;
	int16_t* out = dst + static_cast<long long>(blockIdx.x) * row_len;
	float lo = -1.0F, hi = 1.0F;
	for (long long i = threadIdx.x; i < row_len; i += blockDim.x) {
		const float v = row[i];
		lo = fminf(lo, v);
		hi = fmaxf(hi, v);
	}
#pragma unroll
	for (int d = 16; d > 0; d >>= 1) {
		lo = fminf(lo, __shfl_xor_sync(0xFFFFFFFFU, lo, d));
		hi = fmaxf(hi, __shfl_xor_sync(0xFFFFFFFFU, hi, d));
	}
	if ((threadIdx.x & 31) == 0) {
		lo_s[threadIdx.x >> 5] = lo;
		hi_s[threadIdx.x >> 5] = hi;
	}
	__syncthreads();
	lo = lo_s[0];
	hi = hi_s[0];
#pragma unroll
	for (int w = 1; w < 8; ++w) {
		lo = fminf(lo, lo_s[w]);
		hi = fmaxf(hi, hi_s[w]);
	}
	const float scale = 1.0F / fmaxf(hi, -lo);
	if (threadIdx.x == 0 && row_scale) {
		row_scale[blockIdx.x] = scale;
	}
	for (long long i = threadIdx.x; i < row_len; i += blockDim.x) {
		out[i] = static_cast<int16_t>(scale * row[i] * 32767.0F);
	}
}

// Stream-major buffers are a row-major matrix [stream][frame * C + c]: column sums in two coalesced,
// deterministic passes.  Pass 1: a CTA sums kBusRows consecutive rows of a 1024-column slab (each thread
// one float4 column group, rows in ascending order) into partial[row group][column]; pass 2 sums the row
// groups in ascending order.  Reads the matrix once at full HBM rate (the generic kernel above strides
// by a whole row between threads and moves 8x the bytes).
constexpr int kBusRows = 128;   // rows per group for tall matrices; fewer when there are few rows (see reduce_bus)

__global__ void __launch_bounds__(256) bus_partial_kernel(const float* __restrict__ data, long long row_stride, int rows, int cols4,
	int group_rows, float4* __restrict__ partial)
{
	const int col4 = blockIdx.x * blockDim.x + threadIdx.x; // float4 column index
	if (col4 >= cols4) {
		return;
	}
	const int r0 = blockIdx.y * group_rows;
	const int r1 = min(r0 + group_rows, rows);
	float4 acc = make_float4(0.0F, 0.0F, 0.0F, 0.0F);
	for (int r = r0; r < r1; ++r) {
		const float4 v = __ldcs(reinterpret_cast<const float4*>(data + r * row_stride) + col4);
		acc.x += v.x;
		acc.y += v.y;
		acc.z += v.z;
		acc.w += v.w;
	}
	partial[static_cast<long long>(blockIdx.y) * cols4 + col4] = acc;
}

// 32 float4 columns per CTA, 8 slices of the row groups per column; slice sums are combined in slice order
// (fixed summation order, independent of scheduling).
__global__ void __launch_bounds__(256) bus_final_kernel(const float4* __restrict__ partial, int groups, int cols4, float4* __restrict__ bus)
{
	__shared__ float4 part[8][32];
	const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
	const int col4 = blockIdx.x * 32 + lane;
	float4 acc = make_float4(0.0F, 0.0F, 0.0F, 0.0F);
	if (col4 < cols4) {
		const int g0 = static_cast<int>(static_cast<long long>(groups) * slice / 8);
		const int g1 = static_cast<int>(static_cast<long long>(groups) * (slice + 1) / 8);
		for (int g = g0; g < g1; ++g) {
			const float4 v = partial[static_cast<long long>(g) * cols4 + col4];
			acc.x += v.x;
			acc.y += v.y;
			acc.z += v.z;
			acc.w += v.w;
		}
	}
	part[slice][lane] = acc;
	__syncthreads();
	if (slice == 0 && col4 < cols4) {
#pragma unroll
		for (int k = 1; k < 8; ++k) {
			const float4 v = part[k][lane];
			acc.x += v.x;
			acc.y += v.y;
			acc.z += v.z;
			acc.w += v.w;
		}
		bus[col4] = acc;
	}
}

class CudaBackend final : public Backend {
public:
	explicit CudaBackend(int device) : device_(device) {}

	const char* name() const override { return "cuda"; }

	bool check(cudaError_t err, const char* what)
	{
		if (err == cudaSuccess) {
			return true;
		}
		error_ = std::string(what) + ": " + cudaGetErrorString(err);
		return false;
	}

	bool bind() { return check(cudaSetDevice(device_), "cudaSetDevice"); }
	// Every entry point runs on the engine's device and leaves the calling thread's current device as it found it
	// (a host process with several GPUs keeps its own notion of "current").
	struct DeviceScope {
		int previous = -1;
		bool ok;
		explicit DeviceScope(CudaBackend* be)
		{
			cudaGetDevice(&previous);
			ok = previous == be->device_ || be->bind();
			if (previous == be->device_) {
				previous = -1;
			}
		}
		~DeviceScope()
		{
			if (previous >= 0) {
				cudaSetDevice(previous);
			}
		}
	};

	void* alloc(size_t bytes) override
	{
		DeviceScope scope(this);
		if (!scope.ok) {
			return nullptr;
		}
		void* p = nullptr;
		if (!check(cudaMalloc(&p, bytes ? bytes : 1), "cudaMalloc")) {
			return nullptr;
		}
		if (!check(cudaMemset(p, 0, bytes), "cudaMemset")) {
			cudaFree(p);
			return nullptr;
		}
		return p;
	}

	void release(void* p) override
	{
		if (p) {
			cudaFree(p);
		}
	}

	bool zero(void* p, size_t bytes, void* stream) override
	{
		DeviceScope scope(this);
		return scope.ok && check(cudaMemsetAsync(p, 0, bytes, static_cast<cudaStream_t>(stream)), "cudaMemsetAsync");
	}

	bool upload(void* dst, const void* src, size_t bytes, void* stream) override
	{
		DeviceScope scope(this);
		return scope.ok && check(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream)),
			"cudaMemcpyAsync(H2D)");
	}

	bool download(void* dst, const void* src, size_t bytes, void* stream) override
	{
		DeviceScope scope(this);
		return scope.ok && check(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)),
			"cudaMemcpyAsync(D2H)");
	}

	// Page-lock a caller's host buffer in place so that copies to / from it run at the pinned rate and overlap with kernels.
	// Already page-locked memory (cudaHostAlloc, torch pin_memory) is fine and reported as success.
	bool host_register(void* p, size_t bytes) override
	{
		DeviceScope scope(this);
		if (!scope.ok) {
			return false;
		}
		const cudaError_t err = cudaHostRegister(p, bytes, cudaHostRegisterDefault);
		if (err == cudaErrorHostMemoryAlreadyRegistered) {
			cudaGetLastError();
			return true;
		}
		return check(err, "cudaHostRegister");
	}
	void host_unregister(void* p) override
	{
		if (cudaHostUnregister(p) != cudaSuccess) {
			cudaGetLastError();
		}
	}
	void* host_alloc(size_t bytes) override
	{
		DeviceScope scope(this);
		void* p = nullptr;
		if (!scope.ok || !check(cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault), "cudaHostAlloc")) {
			return nullptr;
		}
		std::memset(p, 0, bytes);
		return p;
	}
	void host_free(void* p) override
	{
		if (p) {
			cudaFreeHost(p);
		}
	}

	bool copy_2d(void* dst, size_t dst_pitch, const void* src, size_t src_pitch, size_t width, size_t rows,
		void* stream) override
	{
		DeviceScope scope(this);
		return scope.ok && check(cudaMemcpy2DAsync(dst, dst_pitch, src, src_pitch, width, rows, cudaMemcpyDeviceToDevice,
			static_cast<cudaStream_t>(stream)), "cudaMemcpy2DAsync");
	}

	bool zero_lanes(uint32_t* base, long long tile_stride, int words, const TileRef* tiles, int n_tiles,
		void* stream) override
	{
		DeviceScope scope(this);
		if (!scope.ok) {
			return false;
		}
		if (n_tiles <= 0 || words <= 0) {
			return true;
		}
		cudaStream_t st = static_cast<cudaStream_t>(stream);
		// Whole consecutive tiles: plain memset.
		bool dense = true;
		for (int i = 0; i < n_tiles && dense; ++i) {
			dense = tiles[i].mask == 0xFFFFFFFFU && tiles[i].tile == tiles[0].tile + static_cast<uint32_t>(i);
		}
		if (dense && tile_stride == static_cast<long long>(words) * kLanes) {
			return check(cudaMemsetAsync(base + static_cast<long long>(tiles[0].tile) * tile_stride, 0,
				static_cast<size_t>(n_tiles) * static_cast<size_t>(tile_stride) * sizeof(uint32_t), st), "cudaMemsetAsync");
		}
		// the tile list lives in a buffer that is kept and grown on demand (no allocation per call)
		const size_t need = static_cast<size_t>(n_tiles) * sizeof(TileRef);
		if (need > zero_tiles_bytes_) {
			cudaFree(zero_tiles_);
			zero_tiles_ = nullptr;
			zero_tiles_bytes_ = 0;
			if (!check(cudaMalloc(&zero_tiles_, need), "cudaMalloc(zero_lanes tile list)")) {
				return false;
			}
			zero_tiles_bytes_ = need;
		}
		TileRef* dev_tiles = static_cast<TileRef*>(zero_tiles_);
		bool ok = check(cudaMemcpyAsync(dev_tiles, tiles, need, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync");
		if (ok) {
			for (int first = 0; first < n_tiles && ok; first += 65535) {
				const int n = (n_tiles - first < 65535 ? n_tiles - first : 65535);
				const int gx = (words + 7) / 8 < 64 ? (words + 7) / 8 : 64;
				zero_lanes_kernel<<<dim3(static_cast<unsigned>(gx), static_cast<unsigned>(n)), 256, 0, st>>>(
					base, tile_stride, words, dev_tiles + first);
				ok = check(cudaGetLastError(), "zero_lanes_kernel");
			}
		}
		// the host array may go away and the list buffer be rewritten by the next call
		return check(cudaStreamSynchronize(st), "cudaStreamSynchronize") && ok;
	}

	bool copy_lanes(uint32_t* dst, long long dst_ts, int dst_w0, const uint32_t* src, long long src_ts, int src_w0, int words,
		const int32_t* from, const int32_t* to, int n, void* stream) override
	{
		DeviceScope scope(this);
		return scope.ok && launch_copy_lanes(dst, dst_ts, dst_w0, src, src_ts, src_w0, words, from, to, n, static_cast<cudaStream_t>(stream)) &&
			check(cudaGetLastError(), "copy_lanes_kernel");
	}

	bool gather_io(const float* src, long long ts, long long ls, long long fs, long long cs, const int32_t* stream_of_lane,
		int lane_tiles, int frames, int channels, float* dst, void* stream) override
	{
		DeviceScope scope(this);
		return scope.ok && launch_gather_io(src, ts, ls, fs, cs, stream_of_lane, lane_tiles, frames, channels, dst,
			static_cast<cudaStream_t>(stream)) && check(cudaGetLastError(), "gather_io_kernel");
	}

	bool scatter_io(const float* src, const int32_t* stream_of_lane, int lane_tiles, int frames, int channels, float* dst,
		long long ts, long long ls, long long fs, long long cs, void* stream) override
	{
		DeviceScope scope(this);
		return scope.ok && launch_scatter_io(src, stream_of_lane, lane_tiles, frames, channels, dst, ts, ls, fs, cs,
			static_cast<cudaStream_t>(stream)) && check(cudaGetLastError(), "scatter_io_kernel");
	}

	bool zero_rows(float* dst, long long ts, long long ls, long long fs, long long cs, const int32_t* rows, int n, int frames,
		int channels, void* stream) override
	{
		DeviceScope scope(this);
		return scope.ok && launch_zero_rows(dst, ts, ls, fs, cs, rows, n, frames, channels, static_cast<cudaStream_t>(stream)) &&
			check(cudaGetLastError(), "zero_rows_kernel");
	}

	bool launch_mix(int kernel_id, const MixArgs& args, void* stream) override
	{
		DeviceScope scope(this);
		if (!scope.ok) {
			return false;
		}
		cudaStream_t st = static_cast<cudaStream_t>(stream);
		if (!(launch_duo_family(kernel_id, args, st) || launch_span_family(kernel_id, args, st) || launch_quartet_family(kernel_id, args, st) ||
				launch_relay_family(kernel_id, args, st) || launch_scan_family(kernel_id, args, st) || launch_mix_family(kernel_id, args, st))) {
			error_ = "unknown kernel id";
			return false;
		}
		return check(cudaGetLastError(), kernel_name(kernel_id));
	}

	bool has_relay() const override { return true; }

	bool reduce_bus(const float* data, long long ts, long long ls, long long fs, long long cs,
		int num_streams, int frames, int channels, float* bus, void* stream) override
	{
		DeviceScope scope(this);
		if (!scope.ok) {
			return false;
		}
		cudaStream_t st = static_cast<cudaStream_t>(stream);
		const long long cols = static_cast<long long>(frames) * channels;
		const bool rows_contiguous = cs == 1 && fs == channels && ls == cols && ts == ls * kLanes && cols % 4 == 0 &&
			((reinterpret_cast<unsigned long long>(data) | reinterpret_cast<unsigned long long>(bus)) & 15ULL) == 0;
		if (rows_contiguous) {
			const int cols4 = static_cast<int>(cols / 4);
			const unsigned gx = static_cast<unsigned>((cols4 + 255) / 256);
			// Rows per group: 128 for tall matrices; with few rows (the per-tile bus rows of mix_bus: one row per 32 streams)
			// fewer, so that pass 1 still fills the GPU (~4 CTAs per SM).  A function of the shape only: deterministic.
			int group_rows = kBusRows;
			while (group_rows > 4 && static_cast<long long>((num_streams + group_rows - 1) / group_rows) * gx < 592) {
				group_rows /= 2;
			}
			const int groups = (num_streams + group_rows - 1) / group_rows;
			const size_t need = static_cast<size_t>(groups) * static_cast<size_t>(cols) * sizeof(float);
			if (need > bus_partial_bytes_) {
				cudaFree(bus_partial_);
				bus_partial_ = nullptr;
				bus_partial_bytes_ = 0;
				if (!check(cudaMalloc(&bus_partial_, need), "cudaMalloc(bus partials)")) {
					return false;
				}
				bus_partial_bytes_ = need;
			}
			bus_partial_kernel<<<dim3(gx, static_cast<unsigned>(groups)), 256, 0, st>>>(data, ls, num_streams, cols4, group_rows,
				static_cast<float4*>(bus_partial_));
			bus_final_kernel<<<static_cast<unsigned>((cols4 + 31) / 32), 256, 0, st>>>(static_cast<const float4*>(bus_partial_), groups, cols4,
				reinterpret_cast<float4*>(bus));
			return check(cudaGetLastError(), "bus_partial_kernel / bus_final_kernel");
		}
		reduce_bus_kernel<<<static_cast<unsigned>(frames * channels), 256, 0, st>>>(
			data, ts, ls, fs, cs, num_streams, channels, bus);
		return check(cudaGetLastError(), "reduce_bus_kernel");
	}

	bool reduce_buses(const bus::Chunk& chunk, void* stream) override
	{
		DeviceScope scope(this);
		return scope.ok && launch_reduce_buses(chunk, static_cast<cudaStream_t>(stream)) &&
			check(cudaGetLastError(), "bus_rows_kernel / bus_tiled_kernel");
	}

	bool pcm_to_float(const void* src, int bits, float* dst, long long count, void* stream) override
	{
		DeviceScope scope(this);
		if (!scope.ok) {
			return false;
		}
		if (count <= 0) {
			return true;
		}
		int sms = 148;
		cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device_);
		const long long want = (count / 8 + 255) / 256;
		const unsigned blocks = static_cast<unsigned>(want < 1 ? 1 : want > 8LL * sms ? 8LL * sms : want);
		cudaStream_t st = static_cast<cudaStream_t>(stream);
		// a payload behind a 44-byte WAV header, a tensor slice ...: misaligned buffers take the scalar loop
		const bool aligned = ((reinterpret_cast<unsigned long long>(src) | reinterpret_cast<unsigned long long>(dst)) & 15ULL) == 0;
		if (bits == 16) {
			pcm16_to_float_kernel<<<blocks, 256, 0, st>>>(static_cast<const int16_t*>(src), dst, count, aligned);
		} else if (bits == 8) {
			pcm8_to_float_kernel<<<blocks, 256, 0, st>>>(static_cast<const uint8_t*>(src), dst, count, aligned);
		} else {
			error_ = "Invalid bit depth."; // the reference's message (oalsfxpp_test.cpp:738)
			return false;
		}
		return check(cudaGetLastError(), "pcm_to_float");
	}

	bool debug_waveshaper(const float* samples, float edge_coeff, float* out, long long count, void* stream) override
	{
		DeviceScope scope(this);
		if (!scope.ok) {
			return false;
		}
		if (count <= 0) {
			return true;
		}
		debug_waveshaper_kernel<<<1184, 256, 0, static_cast<cudaStream_t>(stream)>>>(samples, edge_coeff, out, count);
		return check(cudaGetLastError(), "debug_waveshaper_kernel");
	}

	bool float_to_s16(const float* src, int16_t* dst, int rows, long long row_len, float* row_scale, void* stream) override
	{
		DeviceScope scope(this);
		if (!scope.ok) {
			return false;
		}
		if (rows <= 0 || row_len <= 0) {
			return true;
		}
		float_to_s16_kernel<<<static_cast<unsigned>(rows), 256, 0, static_cast<cudaStream_t>(stream)>>>(src, dst, row_len, row_scale);
		return check(cudaGetLastError(), "float_to_s16");
	}

	bool sync(void* stream) override
	{
		DeviceScope scope(this);
		return scope.ok && check(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)), "cudaStreamSynchronize");
	}

	void* stream_create() override
	{
		cudaStream_t s = nullptr;
		if (!bind() || !check(cudaStreamCreate(&s), "cudaStreamCreate")) {
			return nullptr;
		}
		return s;
	}

	void stream_destroy(void* stream) override
	{
		if (stream) {
			cudaStreamDestroy(static_cast<cudaStream_t>(stream));
		}
	}

	bool stream_wait(void* waiter, void* signal) override
	{
		DeviceScope scope(this);
		if (!scope.ok) {
			return false;
		}
		if (events_.empty()) {
			events_.resize(64, nullptr);
		}
		cudaEvent_t& ev = events_[next_event_++ % events_.size()];
		if (!ev && !check(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming), "cudaEventCreate")) {
			return false;
		}
		return check(cudaEventRecord(ev, static_cast<cudaStream_t>(signal)), "cudaEventRecord") &&
			check(cudaStreamWaitEvent(static_cast<cudaStream_t>(waiter), ev, 0), "cudaStreamWaitEvent");
	}

	~CudaBackend() override
	{
		cudaFree(bus_partial_);
		cudaFree(zero_tiles_);
		for (cudaEvent_t ev : events_) {
			if (ev) {
				cudaEventDestroy(ev);
			}
		}
	}

	const std::string& error() const override { return error_; }

private:
	int device_;
	std::string error_;
	std::vector<cudaEvent_t> events_;
	size_t next_event_ = 0;
	void* zero_tiles_ = nullptr;       // device copy of zero_lanes' tile list
	size_t zero_tiles_bytes_ = 0;
	void* bus_partial_ = nullptr;      // row-group partial sums of the bus reduction
	size_t bus_partial_bytes_ = 0;
};

} // namespace

Backend* make_backend(int device, std::string& error)
{
	int count = 0;
	const cudaError_t err = cudaGetDeviceCount(&count);
	if (err != cudaSuccess || count <= 0) {
		error = std::string("No usable CUDA device (there is no CPU fallback): ") +
			(err != cudaSuccess ? cudaGetErrorString(err) : "device count is 0");
		return nullptr;
	}
	if (device < 0 || device >= count) {
		error = "CUDA device ordinal out of range.";
		return nullptr;
	}
	CudaBackend* be = new CudaBackend(device);
	if (!be->bind()) {
		error = be->error();
		delete be;
		return nullptr;
	}
	return be;
}

const char* backend_build_info() { return "oalsfx_b200 sm_100a cuda (fmad=false)"; }

} // namespace oalsfx
