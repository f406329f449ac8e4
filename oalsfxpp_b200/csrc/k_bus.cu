// k_bus.cu -- the kernels of the submix buses (bus.cuh): one launch per level of a chunk, one CTA per (run, column slab).
// Level 0 comes in three kinds: the plain sum (unity plans), the weighted one (route gains, steady or ramping) and the pan
// kernels (a plan with pan routes or buses of another channel count: a member's value mixes the frame's channels).
// Memory-bound: every level reads its entries once from HBM (level 0: the caller's block) or L2 (partial rows) and writes
// one row per run.  A column of a chunk is one (frame, bus channel) pair, j = f * Cb + c.
#include "bus.cuh"
#include "launch.h"

namespace oalsfx {
namespace bus {

constexpr int kRowsThreads = 256;
constexpr int kRowsVecPerThread = 4;                                        // float4 column groups per thread
constexpr long long kRowsSlab = 4LL * kRowsThreads * kRowsVecPerThread;     // columns per CTA
constexpr int kTiledCols = 256;                                             // columns per CTA of the TILED level 0
constexpr int kPanFrames = 512;                                             // frames per CTA of the STREAM_MAJOR pan level 0
// (frame, channel) lines per CTA of the TILED one: 256 steady, 128 ramping (whose g0 matrices take the rest of the 48 KB)
__host__ __device__ constexpr int pan_lines(int weight) { return weight == 2 ? 128 : 256; }
constexpr int kPanMaxCoef = 64;                                             // Cb * C <= 8 * 8
constexpr int kPanTiledThreads = 256;

// Frames per thread of the STREAM_MAJOR pan kernel: the fewest whose C samples are whole float4s (mono: 4 per float4).
__host__ __device__ constexpr int pan_group(int C) { return C % 4 == 0 ? 1 : C % 2 == 0 ? 2 : 4; }
// Members whose samples a thread of that kernel loads before it adds them (ramping: 2 for C <= 2, else 1), and how far the
// loop over such batches is unrolled (steady: 4 members).  Ramping batches keep the division's slow path from spilling;
// steady kernels run fastest with one member per batch and the loop unrolled, which keeps registers below the batched
// version's (a batch of up to 8 members took 17-37 % longer).
__host__ __device__ constexpr int pan_batch(int weight, int C) { return weight == 2 && C <= 2 ? 2 : 1; }
__host__ __device__ constexpr int pan_unroll(int weight) { return weight == 2 ? 1 : 4; }

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

__host__ __device__ bool aligned16(const void* p) { return (reinterpret_cast<unsigned long long>(p) & 15ULL) == 0; }

// The run's member records and, for its pan routes, their coefficients (kRamp: g0 and g1 matrices, else g1 only) into
// shared memory; scalar members leave their coefficient rows unread.
template <int kWeight>
__device__ __forceinline__ void stage_pan_run(const Run& run, const RouteGain* __restrict__ gains, const float* __restrict__ pan,
	int cm, RouteGain* gain, float (*coef)[kBusRun * kPanMaxCoef])
{
	if (static_cast<int>(threadIdx.x) < run.count) {
		gain[threadIdx.x] = gains[run.src + threadIdx.x];
	}
	__syncthreads();
	for (int q = threadIdx.x; q < run.count * cm; q += blockDim.x) {
		const int i = q / cm;
		if (gain[i].pan) {
			const float* m = pan + static_cast<long long>(run.src + i) * (2 * cm) + (q - i * cm);
			if (kWeight == kRamp) {
				coef[0][q] = m[0];
			}
			coef[kWeight == kRamp ? 1 : 0][q] = m[cm];
		}
	}
}

// Frames [fr0, fr0 + n) of the chunk of a STREAM_MAJOR pan run's output row, from `stage` ([frame][bus channel]).
__device__ __forceinline__ void write_pan_row(const Run& run, float* __restrict__ partial, float* __restrict__ buses, long long cols,
	long long bus_stride, long long bus_col0, int fr0, int Cb, int n, const float* stage)
{
	float* out = (run.dst >= 0 ? partial + run.dst * cols : buses + static_cast<long long>(-1 - run.dst) * bus_stride + bus_col0) +
		static_cast<long long>(fr0) * Cb;
	const int count = n * Cb;
	if (aligned16(out) && count % 4 == 0) {
		for (int q = threadIdx.x; q < count / 4; q += blockDim.x) {
			reinterpret_cast<float4*>(out)[q] = reinterpret_cast<const float4*>(stage)[q];
		}
	} else {
		for (int q = threadIdx.x; q < count; q += blockDim.x) {
			out[q] = stage[q];
		}
	}
}

// Pan level 0 of a STREAM_MAJOR block (kWeight kSteady or kRamp, C = kC channels, Cb <= 8 bus channels).  A CTA takes
// kPanFrames frames of one run, thread t the G = pan_group(kC) frames from t * G: per member, in run order, it reads their
// G * kC contiguous samples (with `vec` as float4) and adds the member's Cb values per frame to Cb register accumulators
// (pan_member: one ramp_pos per member and frame); the row goes out through shared memory as whole float4s.
template <int kWeight, int kC>
__global__ void __launch_bounds__(kPanFrames / pan_group(kC)) bus_pan_rows_kernel(const float* __restrict__ src,
	const int32_t* __restrict__ members, long long ts, long long ls, long long col_off, const Run* __restrict__ runs, int nf, int Cb,
	bool vec, float* __restrict__ partial, float* __restrict__ buses, long long bus_stride, long long bus_col0,
	const RouteGain* __restrict__ gains, const float* __restrict__ pan, long long t_f0)
{
	constexpr int G = pan_group(kC);
	__shared__ long long off[kBusRun];
	__shared__ RouteGain gain[kBusRun];
	__shared__ __align__(16) float coef[kWeight == kRamp ? 2 : 1][kBusRun * kPanMaxCoef];
	__shared__ __align__(16) float stage[kPanFrames * 8];
	const Run run = runs[blockIdx.x];
	const int cm = Cb * kC;
	if (static_cast<int>(threadIdx.x) < run.count) {
		const int s = members[run.src + threadIdx.x];
		off[threadIdx.x] = (s / kLanes) * ts + (s % kLanes) * ls + col_off;
	}
	stage_pan_run<kWeight>(run, gains, pan, cm, gain, coef);
	__syncthreads();
	const int fr0 = static_cast<int>(blockIdx.y) * kPanFrames;
	const int n = min(kPanFrames, nf - fr0);
	const int fl = static_cast<int>(threadIdx.x) * G;
	if (fl < n) {
		float acc[G][8];
#pragma unroll
		for (int g = 0; g < G; ++g) {
#pragma unroll
			for (int j = 0; j < 8; ++j) {
				acc[g][j] = 0.0F;
			}
		}
		const bool whole = vec && fl + G <= n;
		// members in batches of U: the batch's loads are issued together, then its values are added in member order
		constexpr int U = pan_batch(kWeight, kC);
#pragma unroll(pan_unroll(kWeight))
		for (int i0 = 0; i0 < run.count; i0 += U) {
			float x[U][G][kC];
#pragma unroll
			for (int u = 0; u < U; ++u) {
				const float* p = src + off[min(i0 + u, run.count - 1)] + static_cast<long long>(fr0 + fl) * kC;
				if (whole) {
#pragma unroll
					for (int q = 0; q < G * kC / 4; ++q) {
						const float4 v = reinterpret_cast<const float4*>(p)[q];
						x[u][(4 * q) / kC][(4 * q) % kC] = v.x;
						x[u][(4 * q + 1) / kC][(4 * q + 1) % kC] = v.y;
						x[u][(4 * q + 2) / kC][(4 * q + 2) % kC] = v.z;
						x[u][(4 * q + 3) / kC][(4 * q + 3) % kC] = v.w;
					}
				} else {
#pragma unroll
					for (int g = 0; g < G; ++g) {
#pragma unroll
						for (int c = 0; c < kC; ++c) {
							x[u][g][c] = fl + g < n ? p[g * kC + c] : 0.0F;
						}
					}
				}
			}
#pragma unroll
			for (int u = 0; u < U; ++u) {
				const int i = i0 + u;
				if (i >= run.count) {
					break;
				}
				const RouteGain gi = gain[i];
				const float* c0 = coef[0] + i * cm;
				const float* c1 = coef[kWeight == kRamp ? 1 : 0] + i * cm;
#pragma unroll
				for (int g = 0; g < G; ++g) {
					const float pos = kWeight == kRamp ? ramp_pos(gi.rf, gi.t0, t_f0 + fr0 + fl + g) : kRampAfter;
#pragma unroll
					for (int j = 0; j < 8; ++j) {
						if (j < Cb) {
							acc[g][j] = acc[g][j] + pan_member(gi, c0, c1, pos, kWeight == kSteady, j, kC, [&](int c) { return x[u][g][c]; });
						}
					}
				}
			}
		}
#pragma unroll
		for (int g = 0; g < G; ++g) {
#pragma unroll
			for (int j = 0; j < 8; ++j) {
				if (j < Cb && fl + g < n) {
					stage[(fl + g) * Cb + j] = acc[g][j];
				}
			}
		}
	}
	__syncthreads();
	write_pan_row(run, partial, buses, static_cast<long long>(nf) * Cb, bus_stride, bus_col0, fr0, Cb, n, stage);
}

// Pan level 0 of a TILED block: as bus_tiled_kernel, lane i of each warp stages member i's kC lines of each of the CTA's
// pan_lines / kC frames ([line][member]); then a thread computes one (frame, bus channel) column over the members in run
// order, reading its frame's kC staged values, and writes it (consecutive threads, consecutive columns).
template <int kWeight, int kC>
__global__ void __launch_bounds__(kPanTiledThreads) bus_pan_tiled_kernel(const float* __restrict__ src, const int32_t* __restrict__ members,
	long long ts, long long ls, long long cs, long long fs, long long col_off, const Run* __restrict__ runs, int nf, int Cb,
	float* __restrict__ partial, float* __restrict__ buses, long long bus_stride, long long bus_col0,
	const RouteGain* __restrict__ gains, const float* __restrict__ pan, long long t_f0)
{
	constexpr int kLines = pan_lines(kWeight);
	__shared__ float vals[kLines][kBusRun + 1];
	__shared__ long long off[kBusRun];
	__shared__ RouteGain gain[kBusRun];
	__shared__ __align__(16) float coef[kWeight == kRamp ? 2 : 1][kBusRun * kPanMaxCoef];
	const Run run = runs[blockIdx.x];
	const int lane = threadIdx.x % kLanes, warp = threadIdx.x / kLanes;
	const int cm = Cb * kC;
	if (static_cast<int>(threadIdx.x) < run.count) {
		const int s = members[run.src + threadIdx.x];
		off[threadIdx.x] = (s / kLanes) * ts + (s % kLanes) * ls + col_off;
	}
	stage_pan_run<kWeight>(run, gains, pan, cm, gain, coef);
	__syncthreads();
	constexpr int per_cta = kLines / kC;
	const int fr0 = static_cast<int>(blockIdx.y) * per_cta;
	const int n = min(per_cta, nf - fr0);
	if (lane < run.count) {
		const float* p = src + off[lane] + static_cast<long long>(fr0) * fs;
#pragma unroll 8
		for (int l = warp; l < n * kC; l += kPanTiledThreads / kLanes) {
			vals[l][lane] = p[l * cs];   // (fs == C * cs: line l is frame l / C, channel l % C)
		}
	}
	__syncthreads();
	float* out = (run.dst >= 0 ? partial + run.dst * static_cast<long long>(nf) * Cb :
		buses + static_cast<long long>(-1 - run.dst) * bus_stride + bus_col0) + static_cast<long long>(fr0) * Cb;
	for (int col = threadIdx.x; col < n * Cb; col += kPanTiledThreads) {
		const int f = col / Cb, j = col - f * Cb;
		const long long t = t_f0 + fr0 + f;
		float acc = 0.0F;
		for (int i = 0; i < run.count; ++i) {
			const RouteGain& gi = gain[i];
			const float pos = kWeight == kRamp ? ramp_pos(gi.rf, gi.t0, t) : kRampAfter;
			acc = acc + pan_member(gi, coef[0] + i * cm, coef[kWeight == kRamp ? 1 : 0] + i * cm, pos, kWeight == kSteady, j, kC,
				[&](int c) { return vals[f * kC + c][i]; });
		}
		out[col] = acc;
	}
}

template <int kWeight, int kC>
void launch_pan(const Chunk& k, unsigned n_runs, bool rows_layout, float* partial, long long bus_stride, long long bus_col0, cudaStream_t st)
{
	if (!rows_layout) {
		constexpr int per_cta = pan_lines(kWeight) / kC;
		const dim3 grid(n_runs, static_cast<unsigned>((k.nf + per_cta - 1) / per_cta));
		bus_pan_tiled_kernel<kWeight, kC><<<grid, kPanTiledThreads, 0, st>>>(k.dst, k.members, k.ts, k.ls, k.cs, k.fs, k.f0 * k.fs,
			k.runs[0], k.nf, k.bus_channels, partial, k.buses, bus_stride, bus_col0, k.gains, k.pan, k.clock + k.f0);
		return;
	}
	const bool vec = k.ts % 4 == 0 && k.ls % 4 == 0 && (k.f0 * k.fs) % 4 == 0 && aligned16(k.dst);
	const dim3 grid(n_runs, static_cast<unsigned>((k.nf + kPanFrames - 1) / kPanFrames));
	bus_pan_rows_kernel<kWeight, kC><<<grid, kPanFrames / pan_group(kC), 0, st>>>(k.dst, k.members, k.ts, k.ls, k.f0 * k.fs,
		k.runs[0], k.nf, k.bus_channels, vec, partial, k.buses, bus_stride, bus_col0, k.gains, k.pan, k.clock + k.f0);
}

// Level 0 of a pan plan: the STREAM_MAJOR or TILED kernel instantiated per engine channel count (1, 2, 4, 6, 7 or 8).
template <int kWeight>
bool launch_pan_level0(const Chunk& k, unsigned n_runs, bool rows_layout, float* partial, long long bus_stride, long long bus_col0,
	cudaStream_t st)
{
	switch (k.channels) {
	case 1: launch_pan<kWeight, 1>(k, n_runs, rows_layout, partial, bus_stride, bus_col0, st); return true;
	case 2: launch_pan<kWeight, 2>(k, n_runs, rows_layout, partial, bus_stride, bus_col0, st); return true;
	case 4: launch_pan<kWeight, 4>(k, n_runs, rows_layout, partial, bus_stride, bus_col0, st); return true;
	case 6: launch_pan<kWeight, 6>(k, n_runs, rows_layout, partial, bus_stride, bus_col0, st); return true;
	case 7: launch_pan<kWeight, 7>(k, n_runs, rows_layout, partial, bus_stride, bus_col0, st); return true;
	case 8: launch_pan<kWeight, 8>(k, n_runs, rows_layout, partial, bus_stride, bus_col0, st); return true;
	default: return false;
	}
}

} // namespace
} // namespace bus

bool launch_reduce_buses(const bus::Chunk& k, cudaStream_t st)
{
	const long long cols = static_cast<long long>(k.nf) * k.bus_channels;
	const long long bus_stride = static_cast<long long>(k.frames) * k.bus_channels;
	const long long bus_col0 = static_cast<long long>(k.f0) * k.bus_channels;
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
		if (level == 0 && k.pan_plan) {
			if (!(weight == bus::kRamp ? bus::launch_pan_level0<bus::kRamp> : bus::launch_pan_level0<bus::kSteady>)(k, n_runs, rows_layout,
					partial, bus_stride, bus_col0, st)) {
				return false;
			}
			continue;
		}
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
