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
//
// Pans (oalsfx_engine_set_bus_format / set_route_pans): the buses have Cb channels of their own.  A pan route carries a
// Cb x C matrix whose coefficients ramp like gains (ramp_pos once per route and frame, ramp_apply per coefficient); its
// level-0 value in bus channel j is pan_dot of row j with the frame's C samples.  A scalar route in such a plan feeds bus
// channel j < C with gain(T) * x_j and adds +0.0f to the others (a run sum never holds -0.0f, so +0.0f changes no bit).
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

// A route's gain parameters: start gain g0, target g1, ramp length rf (frames) and ramp start t0 (frame clock).  pan != 0:
// a pan route, whose coefficients (per member entry of the plan, Chunk::pan) take g0 / g1's place with the same rf and t0.
struct RouteGain {
	float g0, g1;
	int32_t rf, pan;
	long long t0;
};

// A ramp's arithmetic, in two parts so that one evaluation of the fraction serves every coefficient of a route at a clock
// value: the fraction (d + 1) / rf at d = t - t0 frames into the ramp (0 <= d < rf <= 2^24), and its application to g0, g1,
// every operation rounded on its own (no contraction: -fmad=false / -ffp-contract=off).
OALSFX_HD float ramp_frac(long long d, int32_t rf) { return static_cast<float>(static_cast<int32_t>(d) + 1) / static_cast<float>(rf); }
OALSFX_HD float ramp_lerp(float g0, float g1, float frac)
{
	const float diff = g1 - g0;
	const float step = diff * frac;
	return g0 + step;
}

// The gain at clock value t (the header's contract): g0 before t0, g1 from t0 + rf on (or at once when rf == 0), the
// linear ramp in between.
OALSFX_HD float route_gain(const RouteGain& p, long long t)
{
	if (t < p.t0) {
		return p.g0;
	}
	const long long d = t - p.t0;
	if (p.rf == 0 || d >= p.rf) {
		return p.g1;
	}
	return ramp_lerp(p.g0, p.g1, ramp_frac(d, p.rf));
}

// The same rule for every coefficient of a pan route: ramp_pos is where clock value t stands, as one float -- the fraction
// on the ramp (in (0, 1]), kRampBefore before it (g0 holds) or kRampAfter from its end on (g1 holds) -- and ramp_apply the
// coefficient there.  ramp_apply(g0, g1, ramp_pos(rf, t0, t)) == route_gain({g0, g1, rf, t0}, t).
constexpr float kRampBefore = -1.0F;
constexpr float kRampAfter = 2.0F;
OALSFX_HD float ramp_pos(int32_t rf, long long t0, long long t)
{
	if (t < t0) {
		return kRampBefore;
	}
	const long long d = t - t0;
	return rf == 0 || d >= rf ? kRampAfter : ramp_frac(d, rf);
}
OALSFX_HD float ramp_apply(float g0, float g1, float pos) { return pos < 0.0F ? g0 : pos > 1.0F ? g1 : ramp_lerp(g0, g1, pos); }

// Row j of a pan matrix applied to one frame: c(0) * x(0), then + c(k) * x(k) for k = 1..C-1, each operation rounded.
template <class Coef, class X>
OALSFX_HD float pan_dot(int C, Coef c, X x)
{
	float p = c(0) * x(0);
	for (int k = 1; k < C; ++k) {
		p = p + c(k) * x(k);
	}
	return p;
}

// One pass over frames [f0, f0 + nf) of a call of `frames` frames.  Level L's partial rows hold nf * bus_channels floats
// each ([frame][bus channel]), row r at partial[L] + r * nf * bus_channels.
struct Chunk {
	const float* dst;                 // the caller's block: stream s, frame f, channel c at (s/32)*ts + (s%32)*ls + f*fs + c*cs
	long long ts, ls, fs, cs;
	int f0, nf, frames, channels, bus_channels;
	const int32_t* members;           // device: caller stream indices, by bus, ascending
	int levels;
	const Run* runs[kBusMaxLevels];   // device
	int n_runs[kBusMaxLevels];
	float* partial[kBusMaxLevels];
	float* buses;                     // bus b, frame f, bus channel j at buses[(b * frames + f) * bus_channels + j]
	const RouteGain* gains;           // device, per member entry; null: every member's gain is 1 over the chunk (unity)
	long long clock;                  // frame clock value of frame 0 of the call (M): frame f is at clock + f
	bool ramping;                     // with gains: some member's gain changes inside the chunk; else each is its g1
	bool pan_plan;                    // some member is a pan route or bus_channels != channels: level 0 runs the pan kernels
	const float* pan;                 // device, per member entry 2 * bus_channels * channels floats: g0 then g1 matrix
};

// Size of a member entry's pan coefficients (g0 and g1 matrices, [bus channel][channel] each).
OALSFX_HD int pan_stride(int bus_channels, int channels) { return 2 * bus_channels * channels; }

// The level-0 value of a member of a pan plan in bus channel j at clock position `pos` of its route: a pan route's row j of
// its matrix (g0 / g1: its coefficients) applied to the frame x(0..C-1); a scalar route's gain times x(j) for j < C, else
// +0.0f.  `steady`: every coefficient and gain is its g1 (no ramp inside the chunk).
template <class X>
OALSFX_HD float pan_member(const RouteGain& g, const float* g0, const float* g1, float pos, bool steady, int j, int C, X x)
{
	if (!g.pan) {
		return j < C ? (steady ? g.g1 : ramp_apply(g.g0, g.g1, pos)) * x(j) : 0.0F;
	}
	const float* r0 = g0 + j * C;
	const float* r1 = g1 + j * C;
	return steady ? pan_dot(C, [&](int k) { return r1[k]; }, x) : pan_dot(C, [&](int k) { return ramp_apply(r0[k], r1[k], pos); }, x);
}

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
		const long long cols = static_cast<long long>(k->nf) * k->bus_channels;
		if (level > 0) {
			return k->partial[level - 1][(run.src + i) * cols + j];
		}
		const int e = run.src + i, s = k->members[e];
		const long long f = k->f0 + j / k->bus_channels, c = j % k->bus_channels;
		const float* row = k->dst + (s / kLanes) * k->ts + (s % kLanes) * k->ls + f * k->fs;
		if (k->pan_plan) {
			const RouteGain& g = k->gains[e];
			const float* m = g.pan ? k->pan + static_cast<long long>(e) * pan_stride(k->bus_channels, k->channels) : nullptr;
			const int cm = k->bus_channels * k->channels;
			return pan_member(g, m, m ? m + cm : nullptr, ramp_pos(g.rf, g.t0, k->clock + f), !k->ramping, static_cast<int>(c),
				k->channels, [&](int q) { return row[q * k->cs]; });
		}
		const float x = row[c * k->cs];
		return k->gains ? route_gain(k->gains[e], k->clock + f) * x : x;
	}
};

// Host loop with the kernels' semantics, for a backend whose device memory the host addresses (the Backend default).
inline void reduce_buses_host(const Chunk& k)
{
	const long long cols = static_cast<long long>(k.nf) * k.bus_channels;
	for (int level = 0; level < k.levels; ++level) {
		for (int r = 0; r < k.n_runs[level]; ++r) {
			const Run run = k.runs[level][r];
			float* out = run.dst >= 0 ? k.partial[level] + run.dst * cols :
				k.buses + (static_cast<long long>(-1 - run.dst) * k.frames + k.f0) * k.bus_channels;
			for (long long j = 0; j < cols; ++j) {
				out[j] = run_sum<float>(run.count, HostLoad{&k, level, run, j});
			}
		}
	}
}

} // namespace bus
} // namespace oalsfx

#endif
