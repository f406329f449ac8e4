// backend.h -- the thin device-services interface the engine's host logic (engine.cpp) talks to.
//
// The product links exactly one implementation: cuda_backend.cu (CUDA runtime + the sm_100a
// kernels).  tests/emu/host_backend.cpp is a second one that exists ONLY so the host logic and the
// __host__ __device__ kernel bodies can be exercised by `pytest -m "not gpu"` in a container
// without a GPU; it is compiled into tests/_build/, never into the package, and nothing under
// oalsfxpp_b200/ can load it.
#ifndef OALSFX_BACKEND_H
#define OALSFX_BACKEND_H

#include <cstddef>
#include <cstdint>
#include <cstdlib>
#include <string>

#include "bus.cuh"
#include "mix.cuh"
#include "place.cuh"

namespace oalsfx {

// Kernel instantiations (see OALSFX_KERNEL_TABLE in kernel_table.h).
enum KernelId : int;

class Backend {
public:
	virtual ~Backend() {}
	virtual const char* name() const = 0;
	// Device memory.  alloc() returns zero-filled memory or null.
	virtual void* alloc(size_t bytes) = 0;
	virtual void release(void* p) = 0;
	virtual bool zero(void* p, size_t bytes, void* stream) = 0;
	virtual bool upload(void* dst, const void* src, size_t bytes, void* stream) = 0;
	virtual bool download(void* dst, const void* src, size_t bytes, void* stream) = 0;
	// Page-lock / release a caller's host buffer (no-ops in the CPU test backend).
	virtual bool host_register(void*, size_t) { return true; }
	virtual void host_unregister(void*) {}
	// Page-locked host memory of the engine's own (zero-filled, or null); plain heap memory in the CPU test backend.
	virtual void* host_alloc(size_t bytes) { return std::calloc(bytes ? bytes : 1, 1); }
	virtual void host_free(void* p) { std::free(p); }
	// dst/src are device pointers; rows of `width` bytes.
	virtual bool copy_2d(void* dst, size_t dst_pitch, const void* src, size_t src_pitch, size_t width, size_t rows,
		void* stream) = 0;
	// Zero `words` words of the selected lanes: base[tile * tile_stride + w * 32 + lane].
	// `tiles` is a HOST array.
	virtual bool zero_lanes(uint32_t* base, long long tile_stride, int words, const TileRef* tiles, int n_tiles,
		void* stream) = 0;
	// Stream placement (place.cuh).  Arenas are tile-major, base[tile * tile_stride + word * 32 + lane]; lane lists are
	// DEVICE arrays.  copy_lanes: for every entry i, dst lane to[i] words [dst_w0, +words) = src lane from[i] words
	// [src_w0, +words); from[i] < 0 writes zeros, to[i] < 0 skips the entry, a null list is the identity (lane i).
	// gather_io: dst (TILED, `frames` frames, lane_tiles tiles) lane l = caller stream stream_of_lane[l] of src
	// (src[(s/32)*ts + (s%32)*ls + f*fs + c*cs]), zeros where stream_of_lane[l] < 0.  scatter_io: the reverse, caller
	// rows only, and zeros in the caller row -2 - stream_of_lane[l] of a parked lane (a paused stream).  zero_rows: zeros in
	// frames [0, frames) of the caller rows rows[0..n) (DEVICE array, ascending).  These defaults are place.cuh's host
	// loops over the kernels' element bodies and need device memory the host can address: the CPU test backend's.
	// cuda_backend.cu overrides all four with the sm_100a kernels.
	virtual bool copy_lanes(uint32_t* dst, long long dst_ts, int dst_w0, const uint32_t* src, long long src_ts, int src_w0,
		int words, const int32_t* from, const int32_t* to, int n, void*)
	{
		place::copy_lanes_host(dst, dst_ts, dst_w0, src, src_ts, src_w0, words, from, to, n);
		return true;
	}
	virtual bool gather_io(const float* src, long long ts, long long ls, long long fs, long long cs, const int32_t* stream_of_lane,
		int lane_tiles, int frames, int channels, float* dst, void*)
	{
		place::gather_io_host(src, ts, ls, fs, cs, stream_of_lane, lane_tiles, frames, channels, dst);
		return true;
	}
	virtual bool scatter_io(const float* src, const int32_t* stream_of_lane, int lane_tiles, int frames, int channels, float* dst,
		long long ts, long long ls, long long fs, long long cs, void*)
	{
		place::scatter_io_host(src, stream_of_lane, lane_tiles, frames, channels, dst, ts, ls, fs, cs);
		return true;
	}
	virtual bool zero_rows(float* dst, long long ts, long long ls, long long fs, long long cs, const int32_t* rows, int n, int frames,
		int channels, void*)
	{
		place::zero_rows_host(dst, ts, ls, fs, cs, rows, n, frames, channels);
		return true;
	}
	virtual bool launch_mix(int kernel_id, const MixArgs& args, void* stream) = 0;
	// The relay kernels (relay.cuh) are device-only code: the CPU test backend answers false and the engine
	// keeps such groups on the single-effect passes.
	virtual bool has_relay() const { return false; }
	// bus[frame*C + c] = sum over streams (fixed order: lane-major tree per tile, then tiles).
	virtual bool reduce_bus(const float* data, long long ts, long long ls, long long fs, long long cs,
		int num_streams, int frames, int channels, float* bus, void* stream) = 0;
	// Submix buses (bus.cuh): every level of one chunk of frames, in level order; plan and scratch are device memory.  The
	// default is bus.cuh's host loop over the kernels' element body, for the CPU test backend; cuda_backend.cu overrides it
	// with the sm_100a kernels of k_bus.cu.
	virtual bool reduce_buses(const bus::Chunk& chunk, void*)
	{
		bus::reduce_buses_host(chunk);
		return true;
	}
	// PCM formats either side of the path (SURVEY.md 8f rank 2; the reference's only producer/consumer of
	// sample buffers, its WAV demo: oalsfxpp_test.cpp:703-740 ingest, :602-651 egress).  Device pointers.
	//   pcm_to_float : bits = 8  -> (int(u8) - 128) / 128.0f ;  bits = 16 -> s16 / 32768.0f
	//   float_to_s16 : per row (= one stream's buffer, `row_len` samples): scale = 1 / max(max(1, max x), -min(-1, min x)),
	//                  out = int16(scale * x * 32767.0f) (truncation); row_scale[row] receives the scale if non-null
	virtual bool pcm_to_float(const void* src, int bits, float* dst, long long count, void* stream) = 0;
	virtual bool float_to_s16(const float* src, int16_t* dst, int rows, long long row_len, float* row_scale, void* stream) = 0;
	// Test hook: the distortion stage's three waveshapers (fx.cuh, FxDistortion::shape) on device buffers, four samples at a
	// time as in the stage.
	virtual bool debug_waveshaper(const float* samples, float edge_coeff, float* out, long long count, void* stream) = 0;
	virtual bool sync(void* stream) = 0;
	// Engine-owned streams for overlapping host copies with kernels (host-buffer mix): create /
	// destroy, and "everything enqueued on `signal` so far happens before what `waiter` gets next".
	virtual void* stream_create() = 0;
	virtual void stream_destroy(void* stream) = 0;
	virtual bool stream_wait(void* waiter, void* signal) = 0;
	virtual const std::string& error() const = 0;
};

// Provided by the one backend linked into the library.
Backend* make_backend(int device, std::string& error);
const char* backend_build_info();

} // namespace oalsfx

#endif
