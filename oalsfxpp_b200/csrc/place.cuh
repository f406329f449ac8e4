// place.cuh -- data movement behind the engine's stream placement (OALSFX_PLACEMENT_AUTO, engine.cpp): the element
// bodies and host loops here, the kernels in k_place.cu.
//
//   copy_lanes_kernel : lane-to-lane copies between tile-major arenas base[tile * tile_stride + word * 32 + lane].  The
//                       engine builds every move on it: an in-place lane permutation is a gather of the moving lanes
//                       into a bounded scratch arena followed by a scatter to their new lanes; padding lanes get a
//                       tile-mate's state; a snapshot gathers the caller streams into canonical order.
//   gather_io_kernel  : the caller's sample buffer (either layout, four strides) -> an engine-internal TILED block in
//                       lane order, zeros for padding lanes.
//   scatter_io_kernel : the reverse, writing the caller rows only.  A parked lane (a paused stream s, encoded in the lane
//                       map as -2 - s: the gather treats it as absent) receives zeros in its caller row instead.
//   zero_rows_kernel  : zeros in the caller rows of a list of streams: the paused streams of an unplaced engine.
// The mix kernels then run unchanged on the TILED block.  copy_lane_word is the element body the kernel and the host loop
// share; the host loops (the Backend defaults, backend.h) serve the CPU test backend, the kernels the device.
#ifndef OALSFX_PLACE_CUH
#define OALSFX_PLACE_CUH

#include <cstdint>

#include "mix.cuh"

namespace oalsfx {
namespace place {

constexpr int kIoFrames = 32;   // frames per CTA of the I/O passes (32 lanes x 32 frames x up to 8 channels in shared memory)

// One entry i, word w of Backend::copy_lanes: the element body of copy_lanes_kernel and of the host loop below.
OALSFX_HD void copy_lane_word(uint32_t* dst, long long dst_ts, int dst_w0, const uint32_t* src, long long src_ts, int src_w0,
	const int32_t* from, const int32_t* to, int i, long long w)
{
	const int d = to ? to[i] : i;
	if (d < 0) {
		return;
	}
	const int s = from ? from[i] : i;
	const uint32_t v = s < 0 ? 0U : src[(s / kLanes) * src_ts + (src_w0 + w) * kLanes + s % kLanes];
	dst[(d / kLanes) * dst_ts + (dst_w0 + w) * kLanes + d % kLanes] = v;
}

// Index of (lane l, frame f, channel c) in a TILED block of `frames` frames.
OALSFX_HD long long tiled_index(long long l, int f, int c, int frames, int channels)
{
	return (l / kLanes) * frames * channels * kLanes + (static_cast<long long>(f) * channels + c) * kLanes + l % kLanes;
}

// Host loops with the kernels' semantics, for a backend whose device memory the host addresses (the Backend defaults).
inline void copy_lanes_host(uint32_t* dst, long long dst_ts, int dst_w0, const uint32_t* src, long long src_ts, int src_w0, int words,
	const int32_t* from, const int32_t* to, int n)
{
	for (long long w = 0; w < words; ++w) {
		for (int i = 0; i < n; ++i) {
			copy_lane_word(dst, dst_ts, dst_w0, src, src_ts, src_w0, from, to, i, w);
		}
	}
}

inline void gather_io_host(const float* src, long long ts, long long ls, long long fs, long long cs, const int32_t* stream_of_lane,
	int lane_tiles, int frames, int channels, float* dst)
{
	for (long long l = 0; l < static_cast<long long>(lane_tiles) * kLanes; ++l) {
		const int s = stream_of_lane[l];
		for (int f = 0; f < frames; ++f) {
			for (int c = 0; c < channels; ++c) {
				dst[tiled_index(l, f, c, frames, channels)] = s < 0 ? 0.0F : src[(s / kLanes) * ts + (s % kLanes) * ls + f * fs + c * cs];
			}
		}
	}
}

inline void scatter_io_host(const float* src, const int32_t* stream_of_lane, int lane_tiles, int frames, int channels, float* dst,
	long long ts, long long ls, long long fs, long long cs)
{
	for (long long l = 0; l < static_cast<long long>(lane_tiles) * kLanes; ++l) {
		const int m = stream_of_lane[l];
		const int s = m >= 0 ? m : -2 - m;   // (m == -1: padding lane, s < 0)
		for (int f = 0; s >= 0 && f < frames; ++f) {
			for (int c = 0; c < channels; ++c) {
				dst[(s / kLanes) * ts + (s % kLanes) * ls + f * fs + c * cs] = m >= 0 ? src[tiled_index(l, f, c, frames, channels)] : 0.0F;
			}
		}
	}
}

inline void zero_rows_host(float* dst, long long ts, long long ls, long long fs, long long cs, const int32_t* rows, int n, int frames,
	int channels)
{
	for (int i = 0; i < n; ++i) {
		const int s = rows[i];
		for (int f = 0; f < frames; ++f) {
			for (int c = 0; c < channels; ++c) {
				dst[(s / kLanes) * ts + (s % kLanes) * ls + f * fs + c * cs] = 0.0F;
			}
		}
	}
}

} // namespace place
} // namespace oalsfx

#endif
