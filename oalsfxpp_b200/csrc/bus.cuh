// bus.cuh -- submix buses (oalsfx_engine_route_streams / oalsfx_engine_reduce_buses): the summation order, the element
// body and the host loop here, the kernels in k_bus.cu.
//
// Order (the ABI's contract, include/oalsfx_engine.h): bus b's members -- the active streams routed to b -- in ascending
// caller stream index are the level-0 list of every (frame, channel).  While a list has more than one entry it is cut
// into consecutive runs of kBusRun (the last one shorter), each run is summed left to right in fp32 from +0.0f, and the
// run sums are the next level's list.  A bus without members is one empty run: +0.0f.  The engine (engine.cpp) turns the
// routing into a plan -- the member list, CSR by bus, and per level the runs -- that depends on caller stream indices and
// activity only, so neither the layout, the placement nor the cut of a call into chunks of frames changes a bit.
//
//   level 0 : a run reads up to 32 member rows of the caller's block through its strides and writes one row;
//   level >0: a run reads up to 32 consecutive partial rows of the level below;
//   a bus's last run writes its row of `buses` directly, every other run a partial row in the scratch arena.
// run_sum is the element body of every level, on the device (k_bus.cu) and in the host loop below (the Backend default,
// which the CPU test backend runs).
//
// Routes (oalsfx_engine_set_routes): a stream may feed up to four buses, each through its own gain.  A member is then one
// (stream, bus) route, its level-0 value gain(T) * x with T the frame's clock value; route_gain is the one definition of
// gain(T), for the kernels, the host loop and the engine's start gains.  A chunk without gains (a unity plan) reads x.
#ifndef OALSFX_BUS_CUH
#define OALSFX_BUS_CUH

#include <cstdint>

#include "fx.cuh"

#if defined(__CUDACC__)
#define OALSFX_BUS_UNROLL _Pragma("unroll 8")
#else
#define OALSFX_BUS_UNROLL
#endif

namespace oalsfx {
namespace bus {

constexpr int kBusRun = 32;          // entries per run
constexpr int kBusMaxLevels = 8;     // 32^7 > 2^31 streams
constexpr int kBusChunkFrames = 2048; // frames per pass: bounds the partial rows whatever the call's frame count

// One run of one level.  src: level 0 -- first entry in the member list; level > 0 -- first partial row of the level
// below.  dst >= 0: partial row of this level; dst < 0: the run is its bus's last, bus -1 - dst.
struct Run {
	int32_t src, count, dst;
};

// A route's gain parameters: start gain g0, target g1, ramp length rf (frames) and ramp start t0 (frame clock).
struct RouteGain {
	float g0, g1;
	int32_t rf, pad;
	long long t0;
};

// The gain at clock value t (the header's contract): g0 before t0, g1 from t0 + rf on (or at once when rf == 0), the
// linear ramp in between, every operation rounded on its own (no contraction: -fmad=false / -ffp-contract=off).
OALSFX_HD float route_gain(const RouteGain& p, long long t)
{
	if (t < p.t0) {
		return p.g0;
	}
	const long long d = t - p.t0;
	if (p.rf == 0 || d >= p.rf) {
		return p.g1;
	}
	const float diff = p.g1 - p.g0;
	const float frac = static_cast<float>(static_cast<int32_t>(d) + 1) / static_cast<float>(p.rf);   // (d < rf <= 2^24)
	const float step = diff * frac;
	return p.g0 + step;
}

// One pass over frames [f0, f0 + nf) of a call of `frames` frames.  Level L's partial rows hold nf * channels floats each
// ([frame][channel]), row r at partial[L] + r * nf * channels.
struct Chunk {
	const float* dst;                 // the caller's block: stream s, frame f, channel c at (s/32)*ts + (s%32)*ls + f*fs + c*cs
	long long ts, ls, fs, cs;
	int f0, nf, frames, channels;
	const int32_t* members;           // device: caller stream indices, by bus, ascending
	int levels;
	const Run* runs[kBusMaxLevels];   // device
	int n_runs[kBusMaxLevels];
	float* partial[kBusMaxLevels];
	float* buses;                     // bus b, frame f, channel c at buses[(b * frames + f) * channels + c]
	const RouteGain* gains;           // device, per member entry; null: every member's gain is 1 over the chunk (unity)
	long long clock;                  // frame clock value of frame 0 of the call (M): frame f is at clock + f
	bool ramping;                     // with gains: some member's gain changes inside the chunk; else each is its g1
};

struct Vec4 {
	float x, y, z, w;
};

OALSFX_HD float bus_add(float a, float b) { return a + b; }
OALSFX_HD Vec4 bus_add(const Vec4& a, const Vec4& b) { return Vec4{a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w}; }

// The element body: `count` (<= kBusRun) entries of one column (or four adjacent columns), left to right from +0.0f.
template <class V, class Load>
OALSFX_HD V run_sum(int count, Load load)
{
	V acc{};
	OALSFX_BUS_UNROLL
	for (int i = 0; i < count; ++i) {
		acc = bus_add(acc, load(i));
	}
	return acc;
}

// Entry i of a run at column j of a chunk: level 0 reads member rows of the caller's block, higher levels partial rows.
struct HostLoad {
	const Chunk* k;
	int level;
	Run run;
	long long j;
	OALSFX_HD float operator()(int i) const
	{
		const long long cols = static_cast<long long>(k->nf) * k->channels;
		if (level > 0) {
			return k->partial[level - 1][(run.src + i) * cols + j];
		}
		const int s = k->members[run.src + i];
		const long long f = k->f0 + j / k->channels, c = j % k->channels;
		const float x = k->dst[(s / kLanes) * k->ts + (s % kLanes) * k->ls + f * k->fs + c * k->cs];
		return k->gains ? route_gain(k->gains[run.src + i], k->clock + f) * x : x;
	}
};

// Host loop with the kernels' semantics, for a backend whose device memory the host addresses (the Backend default).
inline void reduce_buses_host(const Chunk& k)
{
	const long long cols = static_cast<long long>(k.nf) * k.channels;
	for (int level = 0; level < k.levels; ++level) {
		for (int r = 0; r < k.n_runs[level]; ++r) {
			const Run run = k.runs[level][r];
			float* out = run.dst >= 0 ? k.partial[level] + run.dst * cols :
				k.buses + (static_cast<long long>(-1 - run.dst) * k.frames + k.f0) * k.channels;
			for (long long j = 0; j < cols; ++j) {
				out[j] = run_sum<float>(run.count, HostLoad{&k, level, run, j});
			}
		}
	}
}

} // namespace bus
} // namespace oalsfx

#endif
