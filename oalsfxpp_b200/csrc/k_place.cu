// k_place.cu -- the kernels of stream placement (place.cuh): lane copies between arenas, the I/O permutation, and the
// zeros in the rows of paused streams.
#include "launch.h"
#include "place.cuh"

namespace oalsfx {
namespace place {

// Thread k: entry i = k % n (fastest), word w = k / n.  The engine sorts the entries by destination lane, so the
// lanes a warp writes sit in one 128-byte line (one word of one tile) and every line is written by one store; the
// gather into scratch lists its sources in lane order, so lanes read from one source tile are fetched together.
// from[i] < 0: the destination receives zero; to[i] < 0: the entry is skipped.  A null list is the identity.
__global__ void __launch_bounds__(256) copy_lanes_kernel(uint32_t* dst, long long dst_ts, int dst_w0, const uint32_t* src,
	long long src_ts, int src_w0, int words, const int32_t* __restrict__ from, const int32_t* __restrict__ to, int n)
{
	const long long total = static_cast<long long>(n) * words;
	for (long long k = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; k < total;
		 k += static_cast<long long>(gridDim.x) * blockDim.x) {
		copy_lane_word(dst, dst_ts, dst_w0, src, src_ts, src_w0, from, to, static_cast<int>(k % n), k / n);
	}
}

// One CTA per (lane tile, 32-frame chunk).  The caller rows of the tile's 32 lanes go through shared memory
// ([lane][frame * C + channel]) so that both sides are coalesced: a stream-major row is read with 16-byte loads where
// the strides allow (`vec`), the TILED block is written one 128-byte line per (frame, channel).
__global__ void __launch_bounds__(256) gather_io_kernel(const float* __restrict__ src, long long ts, long long ls, long long fs,
	long long cs, bool vec, const int32_t* __restrict__ stream_of_lane, int frames, int channels, float* __restrict__ dst)
{
	__shared__ float buf[kLanes][kIoFrames * kMaxChannels + 1];
	const int tile = blockIdx.x;
	const int f0 = blockIdx.y * kIoFrames;
	const int nf = min(kIoFrames, frames - f0);
	const int row_len = nf * channels;
	// a tile without live caller streams (only padding or parked lanes) is not launched by the mix: nothing to gather
	if (!__syncthreads_or(threadIdx.x < kLanes && stream_of_lane[tile * kLanes + threadIdx.x] >= 0)) {
		return;
	}
	const int warp = threadIdx.x / kLanes, t = threadIdx.x % kLanes;
	for (int r = warp; r < kLanes; r += blockDim.x / kLanes) {
		const int s = stream_of_lane[tile * kLanes + r];
		if (s < 0) {   // padding or parked lane
			for (int j = t; j < row_len; j += kLanes) {
				buf[r][j] = 0.0F;
			}
			continue;
		}
		const float* row = src + (s / kLanes) * ts + (s % kLanes) * ls + f0 * fs;
		if (vec) {
			for (int j = t * 4; j < row_len; j += kLanes * 4) {
				if (j + 4 <= row_len) {
					const float4 v = *reinterpret_cast<const float4*>(row + j);
					buf[r][j] = v.x;
					buf[r][j + 1] = v.y;
					buf[r][j + 2] = v.z;
					buf[r][j + 3] = v.w;
				} else {
					for (int q = j; q < row_len; ++q) {
						buf[r][q] = row[q];
					}
				}
			}
		} else {
			for (int j = t; j < row_len; j += kLanes) {
				buf[r][j] = row[(j / channels) * fs + (j % channels) * cs];
			}
		}
	}
	__syncthreads();
	float* out = dst + static_cast<long long>(tile) * frames * channels * kLanes + static_cast<long long>(f0) * channels * kLanes;
	for (int k = threadIdx.x; k < row_len * kLanes; k += blockDim.x) {
		out[k] = buf[k % kLanes][k / kLanes];
	}
}

__global__ void __launch_bounds__(256) scatter_io_kernel(const float* __restrict__ src, const int32_t* __restrict__ stream_of_lane,
	int frames, int channels, float* __restrict__ dst, long long ts, long long ls, long long fs, long long cs, bool vec)
{
	__shared__ float buf[kLanes][kIoFrames * kMaxChannels + 1];
	const int tile = blockIdx.x;
	const int f0 = blockIdx.y * kIoFrames;
	const int nf = min(kIoFrames, frames - f0);
	const int row_len = nf * channels;
	// live lanes (>= 0) copy the mixed block; parked lanes (<= -2, a paused stream) receive zeros and were not mixed
	const int m = threadIdx.x < kLanes ? stream_of_lane[tile * kLanes + threadIdx.x] : -1;
	const bool live = __syncthreads_or(m >= 0);
	if (!live && !__syncthreads_or(m <= -2)) {
		return;
	}
	if (live) {
		const float* in = src + static_cast<long long>(tile) * frames * channels * kLanes + static_cast<long long>(f0) * channels * kLanes;
		for (int k = threadIdx.x; k < row_len * kLanes; k += blockDim.x) {
			buf[k % kLanes][k / kLanes] = in[k];
		}
		__syncthreads();
	}
	const int warp = threadIdx.x / kLanes, t = threadIdx.x % kLanes;
	for (int r = warp; r < kLanes; r += blockDim.x / kLanes) {
		const int ms = stream_of_lane[tile * kLanes + r];
		if (ms == -1) {
			continue;
		}
		const bool zero = ms < 0;
		const int s = zero ? -2 - ms : ms;
		float* row = dst + (s / kLanes) * ts + (s % kLanes) * ls + f0 * fs;
		if (vec) {
			for (int j = t * 4; j < row_len; j += kLanes * 4) {
				if (j + 4 <= row_len) {
					*reinterpret_cast<float4*>(row + j) = zero ? make_float4(0.0F, 0.0F, 0.0F, 0.0F) :
						make_float4(buf[r][j], buf[r][j + 1], buf[r][j + 2], buf[r][j + 3]);
				} else {
					for (int q = j; q < row_len; ++q) {
						row[q] = zero ? 0.0F : buf[r][q];
					}
				}
			}
		} else {
			for (int j = t; j < row_len; j += kLanes) {
				row[(j / channels) * fs + (j % channels) * cs] = zero ? 0.0F : buf[r][j];
			}
		}
	}
}

// One CTA per (32 entries of the row list, 32-frame chunk).  Stream-major rows take 16-byte stores where the strides allow
// (`vec`), a warp per row; otherwise thread k writes entry k % 32, element k / 32, so that for TILED rows (the list is
// ascending: the paused lanes of one tile are consecutive entries) a warp's stores fall into one 128-byte line per
// (frame, channel).
__global__ void __launch_bounds__(256) zero_rows_kernel(float* __restrict__ dst, long long ts, long long ls, long long fs, long long cs,
	bool vec, const int32_t* __restrict__ rows, int n, int frames, int channels)
{
	const int i0 = blockIdx.x * kLanes;
	const int f0 = blockIdx.y * kIoFrames;
	const int nf = min(kIoFrames, frames - f0);
	const int row_len = nf * channels;
	const int count = min(kLanes, n - i0);
	if (vec) {
		const int warp = threadIdx.x / kLanes, t = threadIdx.x % kLanes;
		for (int r = warp; r < count; r += blockDim.x / kLanes) {
			const int s = rows[i0 + r];
			float* row = dst + (s / kLanes) * ts + (s % kLanes) * ls + f0 * fs;
			for (int j = t * 4; j < row_len; j += kLanes * 4) {
				if (j + 4 <= row_len) {
					*reinterpret_cast<float4*>(row + j) = make_float4(0.0F, 0.0F, 0.0F, 0.0F);
				} else {
					for (int q = j; q < row_len; ++q) {
						row[q] = 0.0F;
					}
				}
			}
		}
		return;
	}
	for (int k = threadIdx.x; k < row_len * kLanes; k += blockDim.x) {
		const int r = k % kLanes, j = k / kLanes;
		if (r < count) {
			const int s = rows[i0 + r];
			dst[(s / kLanes) * ts + (s % kLanes) * ls + (f0 + j / channels) * fs + (j % channels) * cs] = 0.0F;
		}
	}
}

} // namespace place

bool launch_copy_lanes(uint32_t* dst, long long dst_ts, int dst_w0, const uint32_t* src, long long src_ts, int src_w0, int words,
	const int32_t* from, const int32_t* to, int n, cudaStream_t st)
{
	const long long total = static_cast<long long>(n) * words;
	if (total <= 0) {
		return true;
	}
	const long long want = (total + 255) / 256;
	const unsigned blocks = static_cast<unsigned>(want < 148LL * 16 ? want : 148LL * 16);
	place::copy_lanes_kernel<<<blocks, 256, 0, st>>>(dst, dst_ts, dst_w0, src, src_ts, src_w0, words, from, to, n);
	return true;
}

namespace {
bool rows_vectorizable(const void* p, long long ts, long long ls, long long fs, long long cs, int channels)
{
	return cs == 1 && fs == channels && ts % 4 == 0 && ls % 4 == 0 && (reinterpret_cast<unsigned long long>(p) & 15ULL) == 0;
}
} // namespace

bool launch_gather_io(const float* src, long long ts, long long ls, long long fs, long long cs, const int32_t* stream_of_lane,
	int lane_tiles, int frames, int channels, float* dst, cudaStream_t st)
{
	if (lane_tiles <= 0 || frames <= 0) {
		return true;
	}
	const dim3 grid(static_cast<unsigned>(lane_tiles), static_cast<unsigned>((frames + place::kIoFrames - 1) / place::kIoFrames));
	place::gather_io_kernel<<<grid, 256, 0, st>>>(src, ts, ls, fs, cs, rows_vectorizable(src, ts, ls, fs, cs, channels),
		stream_of_lane, frames, channels, dst);
	return true;
}

bool launch_scatter_io(const float* src, const int32_t* stream_of_lane, int lane_tiles, int frames, int channels, float* dst,
	long long ts, long long ls, long long fs, long long cs, cudaStream_t st)
{
	if (lane_tiles <= 0 || frames <= 0) {
		return true;
	}
	const dim3 grid(static_cast<unsigned>(lane_tiles), static_cast<unsigned>((frames + place::kIoFrames - 1) / place::kIoFrames));
	place::scatter_io_kernel<<<grid, 256, 0, st>>>(src, stream_of_lane, frames, channels, dst, ts, ls, fs, cs,
		rows_vectorizable(dst, ts, ls, fs, cs, channels));
	return true;
}

bool launch_zero_rows(float* dst, long long ts, long long ls, long long fs, long long cs, const int32_t* rows, int n, int frames,
	int channels, cudaStream_t st)
{
	if (n <= 0 || frames <= 0) {
		return true;
	}
	const dim3 grid(static_cast<unsigned>((n + kLanes - 1) / kLanes), static_cast<unsigned>((frames + place::kIoFrames - 1) / place::kIoFrames));
	place::zero_rows_kernel<<<grid, 256, 0, st>>>(dst, ts, ls, fs, cs, rows_vectorizable(dst, ts, ls, fs, cs, channels), rows, n, frames,
		channels);
	return true;
}

} // namespace oalsfx
