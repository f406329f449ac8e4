// k_bus.cu -- the kernels of the submix buses (bus.cuh): one launch per level of a chunk, one CTA per (run, column slab).
// Level 0 comes in two instantiations: the plain sum (unity plans) and the weighted one (route gains, steady or ramping).
// Memory-bound: every level reads its entries once from HBM (level 0: the caller's block) or L2 (partial rows) and writes
// one row per run.  A column of a chunk is one (frame, channel) pair, j = f * C + c.
#include "bus.cuh"
#include "launch.h"

namespace oalsfx {
namespace bus {

constexpr int kRowsThreads = 256;
constexpr int kRowsVecPerThread = 4;                                        // float4 column groups per thread
constexpr long long kRowsSlab = 4LL * kRowsThreads * kRowsVecPerThread;     // columns per CTA
constexpr int kTiledCols = 256;                                             // columns per CTA of the TILED level 0

namespace {

// Entry i of a run at column j (loaders for run_sum)
struct RowLoad4 {
	const float* src;
	const long long* off;
	long long j;
	__device__ __forceinline__ Vec4 operator()(int i) const
	{
		const float4 v = *reinterpret_cast<const float4*>(src + off[i] + j);
		return Vec4{v.x, v.y, v.z, v.w};
	}
};
struct RowLoad {
	const float* src;
	const long long* off;
	long long j;
	__device__ __forceinline__ float operator()(int i) const { return src[off[i] + j]; }
};
struct SharedLoad {
	const float* column;   // [member], stride 1
	__device__ __forceinline__ float operator()(int i) const { return column[i]; }
};
// Weighted level 0 (routes with gains): entry i's value is gain * x, one rounding.  kSteady: every entry's gain over the
// chunk is its g1 (staged in g1[]).  kRamp: route_gain at the column's clock value t[e]; columns of one frame (equal t)
// share one evaluation.
enum Weight { kUnity = 0, kSteady = 1, kRamp = 2 };
struct SteadyRowLoad4 {
	const float* src;
	const long long* off;
	const float* g1;
	long long j;
	__device__ __forceinline__ Vec4 operator()(int i) const
	{
		const float4 v = *reinterpret_cast<const float4*>(src + off[i] + j);
		const float g = g1[i];
		return Vec4{g * v.x, g * v.y, g * v.z, g * v.w};
	}
};
struct RampRowLoad4 {
	const float* src;
	const long long* off;
	const RouteGain* gain;
	long long j;
	long long t[4];
	__device__ __forceinline__ Vec4 operator()(int i) const
	{
		const float4 v = *reinterpret_cast<const float4*>(src + off[i] + j);
		float g[4];
		g[0] = route_gain(gain[i], t[0]);
#pragma unroll
		for (int e = 1; e < 4; ++e) {
			g[e] = t[e] == t[e - 1] ? g[e - 1] : route_gain(gain[i], t[e]);
		}
		return Vec4{g[0] * v.x, g[1] * v.y, g[2] * v.z, g[3] * v.w};
	}
};
struct SteadyRowLoad {
	const float* src;
	const long long* off;
	const float* g1;
	long long j;
	__device__ __forceinline__ float operator()(int i) const { return g1[i] * src[off[i] + j]; }
};
struct RampRowLoad {
	const float* src;
	const long long* off;
	const RouteGain* gain;
	long long j, t;
	__device__ __forceinline__ float operator()(int i) const { return route_gain(gain[i], t) * src[off[i] + j]; }
};

// Runs over contiguous rows: level 0 of a STREAM_MAJOR block (member rows through the strides, columns contiguous) and
// every level above 0 (partial rows).  Thread t takes four adjacent columns, kRowsVecPerThread times, a warp 512
// consecutive bytes of each entry row; with `vec` (16-byte aligned rows and a column count divisible by 4) as float4.
// kWeight != kUnity (level 0 of a chunk with route gains): the run's gains sit in shared memory next to its row offsets,
// and column j of the chunk (j < 2048 * C) is at clock value t_col0 + j / channels.  kUnity is the plain sum.
template <int kWeight>
__global__ void __launch_bounds__(kRowsThreads) bus_rows_kernel(const float* __restrict__ src, const int32_t* __restrict__ members,
	long long ts, long long ls, long long col_off, long long row_stride, const Run* __restrict__ runs, long long cols, bool vec,
	float* __restrict__ partial, float* __restrict__ buses, long long bus_stride, long long bus_col0,
	const RouteGain* __restrict__ gains, long long t_col0, int channels)
{
	__shared__ long long off[kBusRun];
	__shared__ float g1[kWeight == kSteady ? kBusRun : 1];
	__shared__ RouteGain gain[kWeight == kRamp ? kBusRun : 1];
	const Run run = runs[blockIdx.x];
	if (static_cast<int>(threadIdx.x) < run.count) {
		if (members) {
			const int s = members[run.src + threadIdx.x];
			off[threadIdx.x] = (s / kLanes) * ts + (s % kLanes) * ls + col_off;
		} else {
			off[threadIdx.x] = static_cast<long long>(run.src + threadIdx.x) * row_stride;
		}
		if (kWeight == kSteady) {
			g1[threadIdx.x] = gains[run.src + threadIdx.x].g1;
		}
		if (kWeight == kRamp) {
			gain[threadIdx.x] = gains[run.src + threadIdx.x];
		}
	}
	__syncthreads();
	float* out = run.dst >= 0 ? partial + run.dst * cols : buses + static_cast<long long>(-1 - run.dst) * bus_stride + bus_col0;
	const long long slab = static_cast<long long>(blockIdx.y) * kRowsSlab;
	for (int k = 0; k < kRowsVecPerThread; ++k) {
		const long long j = slab + (static_cast<long long>(k) * kRowsThreads + threadIdx.x) * 4;
		if (j >= cols) {
			break;
		}
		if (vec) {
			Vec4 v;
			if (kWeight == kRamp) {
				RampRowLoad4 load{src, off, gain, j, {}};
#pragma unroll
				for (int e = 0; e < 4; ++e) {
					load.t[e] = t_col0 + (static_cast<int>(j) + e) / channels;
				}
				v = run_sum<Vec4>(run.count, load);
			} else if (kWeight == kSteady) {
				v = run_sum<Vec4>(run.count, SteadyRowLoad4{src, off, g1, j});
			} else {
				v = run_sum<Vec4>(run.count, RowLoad4{src, off, j});
			}
			*reinterpret_cast<float4*>(out + j) = make_float4(v.x, v.y, v.z, v.w);
			continue;
		}
		for (int e = 0; e < 4 && j + e < cols; ++e) {
			out[j + e] = kWeight == kRamp ? run_sum<float>(run.count, RampRowLoad{src, off, gain, j + e, t_col0 + (static_cast<int>(j) + e) / channels}) :
				kWeight == kSteady ? run_sum<float>(run.count, SteadyRowLoad{src, off, g1, j + e}) :
				run_sum<float>(run.count, RowLoad{src, off, j + e});
		}
	}
}

// Level 0 of a TILED block: a member's value is 4 bytes of a 128-byte line (one (frame, channel) of its tile) that its
// tile-mates share.  Lane i of each warp loads member i, so a warp reads the lines of one column together -- one line for
// a run of whole tiles -- into shared memory ([column][member]); then thread t sums column t in member order.  The grid
// runs every run of one column slab before the next slab, so lines that runs of other buses read again are still in L2.
// kWeight != kUnity: lane i stores gain * x of member i (gains as in bus_rows_kernel), so the sums read finished values.
template <int kWeight>
__global__ void __launch_bounds__(256) bus_tiled_kernel(const float* __restrict__ src, const int32_t* __restrict__ members,
	long long ts, long long ls, long long cs, long long col_off, const Run* __restrict__ runs, long long cols,
	float* __restrict__ partial, float* __restrict__ buses, long long bus_stride, long long bus_col0,
	const RouteGain* __restrict__ gains, long long t_col0, int channels)
{
	__shared__ float vals[kTiledCols][kBusRun + 1];
	__shared__ long long off[kBusRun];
	__shared__ RouteGain gain[kWeight != kUnity ? kBusRun : 1];
	const Run run = runs[blockIdx.x];
	const int lane = threadIdx.x % kLanes, warp = threadIdx.x / kLanes;
	if (static_cast<int>(threadIdx.x) < run.count) {
		const int s = members[run.src + threadIdx.x];
		off[threadIdx.x] = (s / kLanes) * ts + (s % kLanes) * ls + col_off;
		if (kWeight != kUnity) {
			gain[threadIdx.x] = gains[run.src + threadIdx.x];
		}
	}
	__syncthreads();
	const long long j0 = static_cast<long long>(blockIdx.y) * kTiledCols;
	const int n = static_cast<int>(min(static_cast<long long>(kTiledCols), cols - j0));
	if (lane < run.count) {
		const float* p = src + off[lane] + j0 * cs;
		if (kWeight == kRamp) {
			const RouteGain g = gain[lane];
#pragma unroll 8
			for (int j = warp; j < n; j += 256 / kLanes) {
				vals[j][lane] = route_gain(g, t_col0 + (static_cast<int>(j0) + j) / channels) * p[j * cs];
			}
		} else if (kWeight == kSteady) {
			const float g1 = gain[lane].g1;
#pragma unroll 8
			for (int j = warp; j < n; j += 256 / kLanes) {
				vals[j][lane] = g1 * p[j * cs];
			}
		} else {
#pragma unroll 8
			for (int j = warp; j < n; j += 256 / kLanes) {
				vals[j][lane] = p[j * cs];
			}
		}
	}
	__syncthreads();
	if (static_cast<int>(threadIdx.x) < n) {
		float* out = run.dst >= 0 ? partial + run.dst * cols : buses + static_cast<long long>(-1 - run.dst) * bus_stride + bus_col0;
		out[j0 + threadIdx.x] = run_sum<float>(run.count, SharedLoad{vals[threadIdx.x]});
	}
}

bool aligned16(const void* p) { return (reinterpret_cast<unsigned long long>(p) & 15ULL) == 0; }

} // namespace
} // namespace bus

bool launch_reduce_buses(const bus::Chunk& k, cudaStream_t st)
{
	const long long cols = static_cast<long long>(k.nf) * k.channels;
	const long long bus_stride = static_cast<long long>(k.frames) * k.channels;
	const long long bus_col0 = static_cast<long long>(k.f0) * k.channels;
	const bool rows_layout = k.cs == 1 && k.fs == k.channels;   // STREAM_MAJOR; otherwise TILED (fs == channels * cs)
	// one flag for every level: the caller's rows, the partial rows and the bus rows all start on 16-byte boundaries
	const bool vec = cols % 4 == 0 && bus_stride % 4 == 0 && bus_col0 % 4 == 0 && bus::aligned16(k.buses) &&
		(!rows_layout || (k.ts % 4 == 0 && k.ls % 4 == 0 && (k.f0 * k.fs) % 4 == 0 && bus::aligned16(k.dst)));
	for (int level = 0; level < k.levels; ++level) {
		const unsigned n_runs = static_cast<unsigned>(k.n_runs[level]);
		if (n_runs == 0) {
			continue;
		}
		float* partial = k.partial[level];
		// level 0 reads the caller's block, weighted by the route gains unless the chunk is unity (k.gains null)
		const long long t_col0 = k.clock + k.f0;
		const int weight = !k.gains ? bus::kUnity : k.ramping ? bus::kRamp : bus::kSteady;
		if (level == 0 && !rows_layout) {
			const dim3 grid(n_runs, static_cast<unsigned>((cols + bus::kTiledCols - 1) / bus::kTiledCols));
			auto kernel = weight == bus::kRamp ? bus::bus_tiled_kernel<bus::kRamp> : weight == bus::kSteady ?
				bus::bus_tiled_kernel<bus::kSteady> : bus::bus_tiled_kernel<bus::kUnity>;
			kernel<<<grid, 256, 0, st>>>(k.dst, k.members, k.ts, k.ls, k.cs, k.f0 * k.fs, k.runs[0], cols, partial, k.buses, bus_stride,
				bus_col0, k.gains, t_col0, k.channels);
			continue;
		}
		const bool vec_level = vec && (!partial || bus::aligned16(partial)) && (level == 0 || bus::aligned16(k.partial[level - 1]));
		const dim3 grid(n_runs, static_cast<unsigned>((cols + bus::kRowsSlab - 1) / bus::kRowsSlab));
		if (level == 0) {
			auto kernel = weight == bus::kRamp ? bus::bus_rows_kernel<bus::kRamp> : weight == bus::kSteady ?
				bus::bus_rows_kernel<bus::kSteady> : bus::bus_rows_kernel<bus::kUnity>;
			kernel<<<grid, bus::kRowsThreads, 0, st>>>(k.dst, k.members, k.ts, k.ls, k.f0 * k.fs, 0, k.runs[0], cols, vec_level,
				partial, k.buses, bus_stride, bus_col0, k.gains, t_col0, k.channels);
		} else {
			bus::bus_rows_kernel<bus::kUnity><<<grid, bus::kRowsThreads, 0, st>>>(k.partial[level - 1], nullptr, 0, 0, 0, cols,
				k.runs[level], cols, vec_level, partial, k.buses, bus_stride, bus_col0, nullptr, 0, k.channels);
		}
	}
	return true;
}

} // namespace oalsfx
