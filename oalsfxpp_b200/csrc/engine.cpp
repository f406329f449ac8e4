// engine.cpp -- host logic of the batched engine behind include/oalsfx_engine.h.
//
// What it does (replacing the per-instance bookkeeping of the reference's Api::Impl,
// oalsfxpp.cpp:2820-3432, for thousands of streams at once):
//   * keeps per stream and slot an effect "class" (effect type + normalized properties) and per
//     stream a send class; classes are de-duplicated, their coefficient blocks derived once on the
//     host (derive.cpp);
//   * owns the HBM arenas: per slot a lane-interleaved ring region sized by the largest effect type
//     in that slot, per slot a state region, one send-filter state region;
//   * at mix time groups streams by (slot classes, send class, pending-update bits) and launches one
//     fused kernel per group and <= 2048-frame block, with the group's coefficient blocks as kernel
//     arguments; signatures without a fused kernel run as a chain of single-effect passes that
//     accumulate onto the bus in slot order (same summation order as the reference).
//
// No CUDA types here: device services come through backend.h.
#include "oalsfx_engine.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "backend.h"
#include "derive.h"
#include "kernel_table.h"
#include "span.cuh"

using namespace oalsfx;

namespace {

std::string g_create_error;

struct FxClass {
	int type = kFxNull;
	oalsfxpp::EffectProps props;
	SlotCoef coef;          // device table pointers already patched in
	bool used = false;      // scratch for compaction
};

struct SendClass {
	SendSettings direct;
	SendSettings aux[kMaxSlots];
	SendCoef direct_coef;
	SendCoef aux_coef[kMaxSlots];
};

struct GroupKey {
	int fx[kMaxSlots];
	int send;
	uint32_t pending;
	uint32_t paused;   // 1: the streams are not mixed (oalsfx_engine_set_active).  Last, so that keys of active streams keep their order.
	bool operator<(const GroupKey& o) const
	{
		return std::memcmp(this, &o, sizeof(GroupKey)) < 0;
	}
	bool operator==(const GroupKey& o) const { return std::memcmp(this, &o, sizeof(GroupKey)) == 0; }
};

struct Group {
	GroupKey key;
	bool identity = false;     // covers tiles 0..T-1 with all lanes
	bool full_tiles = false;   // every listed tile takes part with all of its (existing) lanes
	bool table = false;        // table mode: key.fx[] holds effect KINDS, streams differ in parameters
	bool multi = false;        // class-per-tile launch: every tile has ONE parameter class, coefficient blocks per tile from HBM
	size_t tile_begin = 0;     // into the concatenated tile list
	int tile_count = 0;
	int multi_kernel = -1;     // class-per-tile launch: its kernel and slot kinds
	int multi_kinds[kMaxSlots] = {};
};

} // namespace

struct oalsfx_engine {
	oalsfx_engine_desc desc{};
	DeviceLayout dev;
	Backend* be = nullptr;
	int streams = 0, tiles = 0, channels = 0, slots = 0;

	// per-lane configuration (host): lane = caller stream unless the engine places its streams (placed)
	std::vector<int> fx_class[kMaxSlots];
	std::vector<int> send_class;
	std::vector<uint8_t> pending;       // bit s: slot s has an un-consumed `update`
	std::vector<uint8_t> active;        // 0: paused, the mix neither runs nor reads the stream and writes zeros to its rows
	// Frames mixed since a launch last carried an update (or the engine was created / restored): a hint for the
	// kernels that only run streams in the steady state (span.cuh) -- a reverb's tap cross-fade takes 128 frames
	// from its update on.  The device checks the real per-stream state; this only avoids launches that would fall back.
	long long frames_since_update = 0;

	std::vector<FxClass> classes;
	std::unordered_map<std::string, int> class_index;
	std::vector<SendClass> send_classes;
	struct Table { void* p; size_t bytes; };
	std::map<std::string, Table> tables; // device lookup tables by content key (released when no class refers to them)
	size_t table_bytes = 0;
	// The stream the caller last handed to a mix / bus / PCM call: work may still be running there (a non-blocking
	// stream does not order against the legacy NULL stream), so everything that mutates, reallocates, uploads or
	// reads back engine state waits for it first (quiesce).
	void* last_stream = nullptr;
	bool stream_busy = false;
	void note_stream(void* stream)
	{
		last_stream = stream;
		stream_busy = true;
	}
	bool quiesce()
	{
		bool ok = true;
		if (stream_busy) {
			ok = be->sync(last_stream);
			stream_busy = false;
		}
		return be->sync(nullptr) && ok;
	}

	// device arenas
	float* ring[kMaxSlots] = {};
	int ring_cap[kMaxSlots] = {};        // words per lane
	uint32_t* slot_state[kMaxSlots] = {};
	uint32_t* send_state = nullptr;
	TileRef* tile_list = nullptr;
	size_t tile_list_cap = 0;
	float* stage_in = nullptr;
	float* stage_out = nullptr;
	size_t stage_cap = 0;                // floats
	long long device_bytes = 0;

	// Table mode (many parameter sets per engine): coefficient blocks of every class and every stream's
	// class indices in HBM, read by the kTab* kernels.  Rebuilt with the groups.
	SlotCoef* slot_table_dev = nullptr;
	size_t slot_table_cap = 0;
	SendCoef* send_table_dev = nullptr;
	size_t send_table_cap = 0;
	int32_t* lane_class_dev[kMaxSlots] = {};
	int32_t* lane_send_dev = nullptr;

	// Stream placement (oalsfx_engine_set_placement).  `tiles` stays the caller's ceil(streams / 32); the arenas hold
	// arena_tiles >= tiles (only AUTO placement grows them).  While `placed`, the configuration vectors above are indexed
	// by lane (arena_tiles * 32 entries) and lane_of_stream / stream_of_lane (-1: padding lane) map caller streams.
	int placement = OALSFX_PLACEMENT_CALLER;
	bool placed = false;
	bool place_oom = false;             // the last placement could not grow the arenas (nothing was changed)
	int arena_tiles = 0;
	std::vector<int32_t> lane_of_stream, stream_of_lane;
	std::vector<GroupKey> tile_key;     // per arena tile: the key its caller streams share
	std::vector<uint8_t> tile_active;   // per arena tile: holds a caller stream
	bool refill_padding = true;         // every padding lane gets its tile-mate's state at the next placement
	// Device lane map of the I/O passes: stream_of_lane, except that a lane of a paused stream s holds -2 - s (parked:
	// neither gathered nor mixed; the scatter writes zeros to its caller row).
	int32_t* stream_of_lane_dev = nullptr;
	size_t stream_of_lane_cap = 0;
	// Unplaced engine with paused streams: their caller rows, zeroed after every block's mix launches (zero_rows).
	int32_t* paused_rows_dev = nullptr;
	size_t paused_rows_cap = 0;
	int paused_rows = 0;
	int32_t* lane_list_dev = nullptr;   // lane lists of copy_lanes
	size_t lane_list_cap = 0;
	uint32_t* move_scratch = nullptr;   // bounded staging arena of the lane moves and of snapshot / restore
	size_t move_scratch_cap = 0;        // words
	float* io_in = nullptr;             // one block of the mix in lane order (TILED)
	float* io_out = nullptr;
	size_t io_cap = 0;                  // floats each
	int lane_count() const { return placed ? arena_tiles * kLanes : streams; }
	int lane_of(int s) const { return placed ? lane_of_stream[static_cast<size_t>(s)] : s; }

	// Submix buses (oalsfx_engine_set_routes / route_streams / reduce_buses, bus.cuh).  The routes are kept in caller
	// order; the plan -- the members of every bus (the routes to it of active streams, ascending stream index) and the runs
	// of every level of the summation tree -- depends on caller streams, the (stream, bus) pairs and activity only, is
	// rebuilt on the host at the first reduce after such a change and uploaded once.  Lane moves do not touch it.  A change
	// of gains or ramps alone rewrites the routes' entries of the gain image, uploaded at the next reduce.  Pan routes
	// (oalsfx_engine_set_route_pans) keep their matrices beside the gains, and the plan's entries of them in the pan image.
	std::vector<int32_t> route_bus;          // stream s's routes at [s * OALSFX_MAX_ROUTES, +OALSFX_MAX_ROUTES): used ones first, then OALSFX_BUS_NONE
	std::vector<bus::RouteGain> route_gain;  // their gain parameters (pan != 0: a pan route; rf and t0 are its ramp's)
	std::vector<std::vector<float>> route_pan; // a pan route's g0 and g1 matrices ([bus channel][channel] each); empty: scalar
	long long pan_routes = 0;                // routes with a matrix (0: set_routes calls leave route_pan untouched)
	int bus_channels = 0;                    // channel count Cb of the submix buses (oalsfx_engine_set_bus_format)
	std::vector<int32_t> route_entry;        // their entries in the member list (-1: none: a free slot or a paused stream)
	int max_bus = 0;                     // largest bus index any route names (-1: none)
	bool bus_plan_dirty = true;
	std::vector<int32_t> bus_plan;       // host image of bus_plan_dev: the member list, then every level's runs
	int bus_entries = 0;                 // length of the member list
	bus::RouteGain* gain_host = nullptr; // page-locked image of gain_dev: per member entry its route's gains
	size_t gain_host_cap = 0;            // entries
	bus::RouteGain* gain_dev = nullptr;
	size_t gain_dev_cap = 0;             // entries
	bool gains_dirty = false;            // gain_host changed since the last upload
	bool gains_unity = true;             // every member's g1 is 1.0f ...
	long long gains_ramp_end = 0;        // ... and from this clock value on every member's gain is its g1
	bool gains_pan = false;              // some member is a pan route: level 0 runs the pan kernels (as with bus_channels != channels)
	float* pan_host = nullptr;           // page-locked image of pan_dev: per member entry bus::pan_stride floats (used by pan routes)
	size_t pan_host_cap = 0;             // floats; >= bus_entries * pan_stride whenever a member entry is a pan route
	float* pan_dev = nullptr;
	size_t pan_dev_cap = 0;              // floats
	int bus_levels = 0;
	size_t bus_run_word[bus::kBusMaxLevels] = {};       // word offset of the level's runs in the plan
	int bus_runs[bus::kBusMaxLevels] = {};
	long long bus_partial_row[bus::kBusMaxLevels] = {}; // first scratch row of the level's partial rows
	long long bus_partial_rows = 0;
	int32_t* bus_plan_dev = nullptr;
	size_t bus_plan_cap = 0;            // words
	float* bus_scratch = nullptr;       // partial rows of one chunk (<= kBusChunkFrames frames)
	size_t bus_scratch_cap = 0;         // floats

	std::vector<Group> groups;
	// Class-per-tile launch (duo_multi_kernel): the class table and every tile's class index in HBM; `groups` is
	// then the single multi group and `fallback_groups` holds the per-class / table-mode groups for the blocks the
	// fused kernel cannot take (frames < 2).
	std::vector<Group> fallback_groups;
	MixClassEntry* class_table_dev = nullptr;
	size_t class_table_cap = 0;
	int32_t* tile_class_dev = nullptr;
	bool groups_dirty = true;
	long long launches = 0;
	int last_kernel = -1;               // id of the most recent mix kernel launched (oalsfx_engine_last_kernel)
	// The frame clock (include/oalsfx_engine.h): frames mixed by successful mix / mix_bus / mix_buses calls, and its value
	// at the start of the most recent one (frame f of a reduce_buses block is at clock_mix + f).
	long long clock_total = 0;
	long long clock_mix = 0;
	// Host buffers the engine has page-locked in place (oalsfx_engine_pin_host, or on first sight with OALSFX_PIN_HOST=1)
	struct PinnedHost { void* p; size_t bytes; bool automatic; };
	std::vector<PinnedHost> pinned_host;
	bool auto_pin_host = false;
	bool pin_host(void* p, size_t bytes, bool automatic)
	{
		for (PinnedHost& h : pinned_host) {
			if (h.p == p && h.bytes >= bytes) {
				return true;
			}
		}
		// a new size or place: automatic registrations that overlap it are stale (the caller's buffer moved)
		for (size_t i = 0; i < pinned_host.size();) {
			const char* a0 = static_cast<const char*>(pinned_host[i].p);
			const char* b0 = static_cast<const char*>(p);
			if (pinned_host[i].automatic && a0 < b0 + bytes && b0 < a0 + pinned_host[i].bytes) {
				be->host_unregister(pinned_host[i].p);
				pinned_host.erase(pinned_host.begin() + static_cast<long>(i));
			} else {
				++i;
			}
		}
		if (automatic && pinned_host.size() >= 16) { // keep the table small: forget the oldest automatic entry
			for (size_t i = 0; i < pinned_host.size(); ++i) {
				if (pinned_host[i].automatic) {
					be->host_unregister(pinned_host[i].p);
					pinned_host.erase(pinned_host.begin() + static_cast<long>(i));
					break;
				}
			}
		}
		if (!be->host_register(p, bytes)) {
			return false;
		}
		pinned_host.push_back(PinnedHost{p, bytes, automatic});
		return true;
	}

	bool mix_launch(int id, const MixArgs& a, void* stream)
	{
		last_kernel = id;
		return be->launch_mix(id, a, stream);
	}
	// Which fused kernel family serves whole-tile groups: 2 = automatic (default): the two-stage duo kernel,
	// or the four-stage quartet pipeline when the group has too few tiles to fill the GPU (and for
	// signatures that only have a quartet entry); 3 = quartet wherever it exists; 4 = duo wherever it exists;
	// 0 = the plain thread-per-stream twin, 5 = the relay pipeline wherever eligible.
	// 6 = as automatic (names the span kernel's tests).  OALSFX_KERNEL=auto|quartet|duo|single|relay|span overrides
	// (A/B measurements and the parity tests of every family).
	int family = 2;
	bool scan_enabled = false;          // OALSFX_SCAN=1
	int family_span_bulk = 1;           // OALSFX_SPAN_BULK=0: whole-tile spans stay on the load / store kernel; 2: whole tiles (and the bulk kernel) however few (A/B, tests)
	// Host-buffer mix: tile slice the next launches are restricted to (0 = all tiles), and the
	// engine-owned streams that overlap H2D, kernels and D2H of consecutive slices.
	int slice_first = 0, slice_count = 0;
	void* pipe_in = nullptr;
	void* pipe_run = nullptr;
	void* pipe_out = nullptr;
	std::string error;

	~oalsfx_engine()
	{
		if (!be) {
			return;
		}
		be->sync(nullptr);
		for (int s = 0; s < kMaxSlots; ++s) {
			be->release(ring[s]);
			be->release(slot_state[s]);
		}
		be->release(send_state);
		be->release(tile_list);
		be->release(class_table_dev);
		be->release(tile_class_dev);
		be->release(slot_table_dev);
		be->release(send_table_dev);
		be->release(lane_send_dev);
		for (int s = 0; s < kMaxSlots; ++s) {
			be->release(lane_class_dev[s]);
		}
		for (const PinnedHost& h : pinned_host) {
			be->host_unregister(h.p);
		}
		be->release(stage_in);
		be->release(stage_out);
		be->release(stream_of_lane_dev);
		be->release(paused_rows_dev);
		be->release(lane_list_dev);
		be->release(move_scratch);
		be->release(io_in);
		be->release(io_out);
		be->release(bus_plan_dev);
		be->release(bus_scratch);
		be->release(gain_dev);
		be->host_free(gain_host);
		be->release(pan_dev);
		be->host_free(pan_host);
		be->stream_destroy(pipe_in);
		be->stream_destroy(pipe_run);
		be->stream_destroy(pipe_out);
		for (auto& kv : tables) {
			be->release(kv.second.p);
		}
		delete be;
	}

	int fail(int code, const std::string& msg)
	{
		error = msg;
		return code;
	}

	void* dev_alloc(size_t bytes)
	{
		void* p = be->alloc(bytes);
		if (p) {
			device_bytes += static_cast<long long>(bytes);
		}
		return p;
	}

	// ---- classes --------------------------------------------------------------------------------
	void* table_for(const std::string& key, const void* data, size_t bytes)
	{
		auto it = tables.find(key);
		if (it != tables.end()) {
			return it->second.p;
		}
		void* p = dev_alloc(bytes);
		if (!p || !be->upload(p, data, bytes, nullptr) || !be->sync(nullptr)) {
			return nullptr;
		}
		tables.emplace(key, Table{p, bytes});
		table_bytes += bytes;
		return p;
	}

	int class_for(int type, const oalsfxpp::EffectProps& props_in)
	{
		oalsfxpp::Effect fx;
		std::memset(&fx, 0, sizeof(fx));
		fx.type_ = static_cast<oalsfxpp::EffectType>(type);
		if (type != kFxNull) {
			fx.props_ = props_in;
		}
		fx.normalize();
		// Key = type + the bytes of the property block that type uses.
		size_t used = 0;
		switch (type) {
		case kFxChorus: used = sizeof(fx.props_.chorus_); break;
		case kFxCompressor: used = sizeof(fx.props_.compressor_); break;
		case kFxDedicatedDialog: case kFxDedicatedLfe: used = sizeof(fx.props_.dedicated_); break;
		case kFxDistortion: used = sizeof(fx.props_.distortion_); break;
		case kFxEcho: used = sizeof(fx.props_.echo_); break;
		case kFxEqualizer: used = sizeof(fx.props_.equalizer_); break;
		case kFxFlanger: used = sizeof(fx.props_.flanger_); break;
		case kFxRingModulator: used = sizeof(fx.props_.ring_modulator_); break;
		case kFxReverb: case kFxEaxReverb: used = offsetof(oalsfxpp::EffectProps::Reverb, decay_hf_limit_) + 1; break;
		default: break;
		}
		std::string key(reinterpret_cast<const char*>(&type), sizeof(type));
		key.append(reinterpret_cast<const char*>(&fx.props_), used);
		auto it = class_index.find(key);
		if (it != class_index.end()) {
			return it->second;
		}
		FxClass c;
		c.type = type;
		c.props = fx.props_;
		SlotTables t;
		derive_slot(dev, desc.sampling_rate, type, fx.props_, c.coef, t);
		if (!t.sin_delays.empty()) {
			const ModDelayCoef& m = c.coef.u.mod_delay;
			std::string tk = "sd";
			tk.append(reinterpret_cast<const char*>(&m.lfo_range), 4);
			tk.append(reinterpret_cast<const char*>(&m.lfo_scale), 4);
			tk.append(reinterpret_cast<const char*>(&m.depth), 4);
			tk.append(reinterpret_cast<const char*>(&m.delay), 4);
			void* p = table_for(tk, t.sin_delays.data(), t.sin_delays.size() * sizeof(int32_t));
			if (!p) {
				return -1;
			}
			c.coef.u.mod_delay.sin_delays = static_cast<const int32_t*>(p);
		}
		if (!t.mod_sinus.empty()) {
			std::string tk = "ms";
			tk.append(reinterpret_cast<const char*>(&c.coef.u.reverb.mod_range), 4);
			void* p = table_for(tk, t.mod_sinus.data(), t.mod_sinus.size() * sizeof(float));
			if (!p) {
				return -1;
			}
			c.coef.u.reverb.mod_sinus = static_cast<const float*>(p);
		}
		classes.push_back(c);
		const int id = static_cast<int>(classes.size()) - 1;
		class_index.emplace(key, id);
		return id;
	}

	// Drop classes no stream refers to any more (cfg2-style per-block parameter changes would
	// otherwise grow the table without bound).  Class 0 (null) always stays.
	void compact_classes()
	{
		for (auto& c : classes) {
			c.used = false;
		}
		classes[0].used = true;
		for (int s = 0; s < kMaxSlots; ++s) {
			for (int id : fx_class[s]) {
				classes[static_cast<size_t>(id)].used = true;
			}
		}
		std::vector<int> remap(classes.size(), -1);
		std::vector<FxClass> kept;
		for (size_t i = 0; i < classes.size(); ++i) {
			if (classes[i].used) {
				remap[i] = static_cast<int>(kept.size());
				kept.push_back(classes[i]);
			}
		}
		for (int s = 0; s < kMaxSlots; ++s) {
			for (int& id : fx_class[s]) {
				id = remap[static_cast<size_t>(id)];
			}
		}
		for (auto it = class_index.begin(); it != class_index.end();) {
			const int to = remap[static_cast<size_t>(it->second)];
			if (to < 0) {
				it = class_index.erase(it);
			} else {
				it->second = to;
				++it;
			}
		}
		classes.swap(kept);
		// lookup tables no surviving class points at: nothing may still be reading them
		std::vector<const void*> live;
		for (const FxClass& c : classes) {
			const int kind = kind_of_type(c.type);
			if (kind == kKindModDelay && c.coef.u.mod_delay.sin_delays) {
				live.push_back(c.coef.u.mod_delay.sin_delays);
			} else if (kind == kKindReverb && c.coef.u.reverb.mod_sinus) {
				live.push_back(c.coef.u.reverb.mod_sinus);
			}
		}
		bool quiet = false;
		for (auto it = tables.begin(); it != tables.end();) {
			if (std::find(live.begin(), live.end(), it->second.p) == live.end()) {
				if (!quiet) {
					quiesce();
					quiet = true;
				}
				be->release(it->second.p);
				device_bytes -= static_cast<long long>(it->second.bytes);
				table_bytes -= it->second.bytes;
				it = tables.erase(it);
			} else {
				++it;
			}
		}
		// send classes no stream uses any more
		std::vector<int> send_remap(send_classes.size(), -1);
		std::vector<SendClass> send_kept;
		for (int id : send_class) {
			if (send_remap[static_cast<size_t>(id)] < 0) {
				send_remap[static_cast<size_t>(id)] = static_cast<int>(send_kept.size());
				send_kept.push_back(send_classes[static_cast<size_t>(id)]);
			}
		}
		for (int& id : send_class) {
			id = send_remap[static_cast<size_t>(id)];
		}
		send_classes.swap(send_kept);
		compacted_at_bytes = table_bytes;
	}
	size_t compacted_at_bytes = 0;

	int send_class_for(const SendSettings& direct, const SendSettings* aux)
	{
		for (size_t i = 0; i < send_classes.size(); ++i) {
			const SendClass& sc = send_classes[i];
			if (std::memcmp(&sc.direct, &direct, sizeof(direct)) == 0 &&
				std::memcmp(sc.aux, aux, sizeof(SendSettings) * static_cast<size_t>(slots)) == 0) {
				return static_cast<int>(i);
			}
		}
		SendClass sc;
		std::memset(&sc, 0, sizeof(sc));
		sc.direct = direct;
		for (int i = 0; i < slots; ++i) {
			sc.aux[i] = aux[i];
		}
		derive_sends(dev, desc.sampling_rate, slots, sc.direct, sc.aux, sc.direct_coef, sc.aux_coef);
		send_classes.push_back(sc);
		return static_cast<int>(send_classes.size()) - 1;
	}

	// ---- arenas -------------------------------------------------------------------------------------
	bool ensure_ring(int slot, int words)
	{
		if (words <= ring_cap[slot]) {
			return true;
		}
		const size_t new_tile_bytes = static_cast<size_t>(words) * kLanes * sizeof(float);
		float* fresh = static_cast<float*>(dev_alloc(new_tile_bytes * static_cast<size_t>(arena_tiles)));
		if (!fresh) {
			return false;
		}
		if (ring[slot]) {
			const size_t old_tile_bytes = static_cast<size_t>(ring_cap[slot]) * kLanes * sizeof(float);
			if (!be->copy_2d(fresh, new_tile_bytes, ring[slot], old_tile_bytes, old_tile_bytes,
					static_cast<size_t>(arena_tiles), nullptr) || !be->sync(nullptr)) {
				return false;
			}
			device_bytes -= static_cast<long long>(old_tile_bytes) * arena_tiles;
			be->release(ring[slot]);
		}
		ring[slot] = fresh;
		ring_cap[slot] = words;
		return true;
	}

	// (tile, mask) list of a stream range
	static void tiles_of_range(int first, int n, std::vector<TileRef>& out)
	{
		out.clear();
		const int last = first + n - 1;
		for (int t = first / kLanes; t <= last / kLanes; ++t) {
			const int lo = std::max(first, t * kLanes) - t * kLanes;
			const int hi = std::min(last, t * kLanes + kLanes - 1) - t * kLanes;
			const uint32_t mask = (hi - lo == 31 ? 0xFFFFFFFFU : ((1U << (hi - lo + 1)) - 1U) << lo);
			out.push_back(TileRef{static_cast<uint32_t>(t), mask});
		}
	}

	// ---- grouping -----------------------------------------------------------------------------------
	GroupKey key_of(int s) const
	{
		GroupKey k;
		std::memset(&k, 0, sizeof(k));
		for (int i = 0; i < kMaxSlots; ++i) {
			k.fx[i] = fx_class[i][static_cast<size_t>(s)];
		}
		k.send = send_class[static_cast<size_t>(s)];
		k.pending = pending[static_cast<size_t>(s)];
		k.paused = active[static_cast<size_t>(s)] ? 0U : 1U;
		return k;
	}

	// ---- submix buses ------------------------------------------------------------------------------
	// The reason a reduce_buses / mix_buses call is refused, checked before anything runs, or null.
	const char* bad_bus_args(int frames, const float* dst, int layout, int n_buses, const float* buses) const
	{
		if (!dst || !buses) {
			return "No block or bus buffer.";
		}
		if (frames <= 0) {
			return "Frame count must be positive.";
		}
		if (layout != OALSFX_LAYOUT_STREAM_MAJOR && layout != OALSFX_LAYOUT_TILED) {
			return "Unknown layout.";
		}
		if (n_buses < 1 || n_buses <= max_bus) {
			return "n_buses must be at least 1 and above every bus index a stream is routed to.";
		}
		return nullptr;
	}

	// Members of every bus 0..max_bus in CSR order (one entry per route of an active stream: its stream index; its gains at
	// the same index of gain_host), then level by level: a bus whose list has one run left ends in that run (it writes the
	// bus row), every other bus cuts its list into runs of 32 that write partial rows, which are the bus's list at the
	// next level.
	bool rebuild_bus_plan(void* stream)
	{
		const int nb = max_bus + 1;
		const size_t routes = route_bus.size();
		std::vector<int32_t> start(static_cast<size_t>(nb) + 1, 0);
		for (size_t r = 0; r < routes; ++r) {
			const int b = route_bus[r];
			if (b >= 0 && active[static_cast<size_t>(lane_of(static_cast<int>(r / OALSFX_MAX_ROUTES)))]) {
				++start[static_cast<size_t>(b) + 1];
			}
		}
		for (int b = 0; b < nb; ++b) {
			start[static_cast<size_t>(b) + 1] += start[static_cast<size_t>(b)];
		}
		bus_entries = start[static_cast<size_t>(nb)];
		if (static_cast<size_t>(bus_entries) > gain_host_cap) {
			// (nothing reads the old image: the route and activity calls that dirty the plan wait for the caller's stream)
			be->host_free(gain_host);
			gain_host_cap = 0;
			gain_host = static_cast<bus::RouteGain*>(be->host_alloc(static_cast<size_t>(bus_entries) * sizeof(bus::RouteGain)));
			if (!gain_host) {
				return false;
			}
			gain_host_cap = static_cast<size_t>(bus_entries);
		}
		const size_t stride = static_cast<size_t>(bus::pan_stride(bus_channels, channels));
		bool any_pan = false;
		for (size_t r = 0; r < routes && !any_pan; ++r) {
			any_pan = route_bus[r] >= 0 && !route_pan[r].empty();
		}
		if (any_pan && static_cast<size_t>(bus_entries) * stride > pan_host_cap) {
			be->host_free(pan_host);
			pan_host_cap = 0;
			pan_host = static_cast<float*>(be->host_alloc(static_cast<size_t>(bus_entries) * stride * sizeof(float)));
			if (!pan_host) {
				return false;
			}
			pan_host_cap = static_cast<size_t>(bus_entries) * stride;
		}
		bus_plan.assign(static_cast<size_t>(bus_entries), 0);
		std::vector<int32_t> fill(start.begin(), start.end() - 1);
		for (size_t r = 0; r < routes; ++r) {
			const int b = route_bus[r];
			const int s = static_cast<int>(r / OALSFX_MAX_ROUTES);
			route_entry[r] = -1;
			if (b >= 0 && active[static_cast<size_t>(lane_of(s))]) {
				const int32_t entry = fill[static_cast<size_t>(b)]++;
				bus_plan[static_cast<size_t>(entry)] = s;
				gain_host[entry] = route_gain[r];
				if (!route_pan[r].empty()) {
					std::memcpy(pan_host + static_cast<size_t>(entry) * stride, route_pan[r].data(), stride * sizeof(float));
				}
				route_entry[r] = entry;
			}
		}
		gains_dirty = true;
		struct List {
			int bus;
			int32_t src, len;
		};
		std::vector<List> open, next;
		for (int b = 0; b < nb; ++b) {
			open.push_back(List{b, start[static_cast<size_t>(b)], start[static_cast<size_t>(b) + 1] - start[static_cast<size_t>(b)]});
		}
		bus_levels = 0;
		bus_partial_rows = 0;
		while (!open.empty()) {
			const int level = bus_levels++;
			bus_run_word[level] = bus_plan.size();
			bus_partial_row[level] = bus_partial_rows;
			int32_t partials = 0;
			next.clear();
			for (const List& l : open) {
				const int32_t n_runs = std::max<int32_t>(1, (l.len + bus::kBusRun - 1) / bus::kBusRun);
				if (n_runs == 1) {
					bus_plan.insert(bus_plan.end(), {l.src, l.len, -1 - l.bus});
					continue;
				}
				next.push_back(List{l.bus, partials, n_runs});
				for (int32_t r = 0; r < n_runs; ++r) {
					bus_plan.insert(bus_plan.end(), {l.src + r * bus::kBusRun, std::min<int32_t>(bus::kBusRun, l.len - r * bus::kBusRun), partials++});
				}
			}
			bus_runs[level] = static_cast<int>((bus_plan.size() - bus_run_word[level]) / 3);
			bus_partial_rows += partials;
			open.swap(next);
		}
		if (bus_plan.size() > bus_plan_cap) {
			quiesce();   // a reduce may still read the old plan
			be->release(bus_plan_dev);
			device_bytes -= static_cast<long long>(bus_plan_cap * sizeof(int32_t));
			bus_plan_cap = 0;
			bus_plan_dev = static_cast<int32_t*>(dev_alloc(bus_plan.size() * sizeof(int32_t)));
			if (!bus_plan_dev) {
				return false;
			}
			bus_plan_cap = bus_plan.size();
		}
		if (!bus_plan.empty() && !be->upload(bus_plan_dev, bus_plan.data(), bus_plan.size() * sizeof(int32_t), stream)) {
			return false;
		}
		bus_plan_dirty = false;
		return true;
	}

	// Whether level 0 runs the pan kernels: some member is a pan route, or the buses have a channel count of their own.
	bool pan_plan() const { return gains_pan || bus_channels != channels; }

	// After a change of gain_host (or of the bus format): whether every member's gain is 1 (gains_unity) from which clock
	// value on (gains_ramp_end; a pan route's coefficients count as its gains), whether some member is a pan route
	// (gains_pan), and the upload of the images unless no chunk from now on needs them (a steady unity plan of scalar routes
	// into buses of the engine's format: the clock only grows, and the next change of gains marks the image dirty again).
	bool upload_gains(void* stream)
	{
		gains_unity = true;
		gains_ramp_end = 0;
		gains_pan = false;
		const int stride = bus::pan_stride(bus_channels, channels);
		for (int i = 0; i < bus_entries; ++i) {
			const bus::RouteGain& g = gain_host[i];
			bool ramps = g.g0 != g.g1;   // (g0 == g1: route_gain is g1 at every t, up to the sign of a zero, which no bus sum shows)
			if (g.pan) {
				const float* m = pan_host + static_cast<size_t>(i) * static_cast<size_t>(stride);
				ramps = !std::equal(m, m + stride / 2, m + stride / 2);
				gains_pan = true;
			}
			gains_unity = gains_unity && g.g1 == 1.0F && !g.pan;
			if (ramps) {
				gains_ramp_end = std::max(gains_ramp_end, g.t0 + g.rf);
			}
		}
		if (gains_pan) {
			const size_t need = static_cast<size_t>(bus_entries) * static_cast<size_t>(stride);
			if (need > pan_dev_cap) {
				quiesce();   // a reduce may still read the old array
				be->release(pan_dev);
				device_bytes -= static_cast<long long>(pan_dev_cap * sizeof(float));
				pan_dev_cap = 0;
				pan_dev = static_cast<float*>(dev_alloc(need * sizeof(float)));
				if (!pan_dev) {
					return false;
				}
				pan_dev_cap = need;
			}
			if (!be->upload(pan_dev, pan_host, need * sizeof(float), stream)) {
				return false;
			}
		}
		if ((!(gains_unity && gains_ramp_end <= clock_mix) || pan_plan()) && bus_entries > 0) {
			if (static_cast<size_t>(bus_entries) > gain_dev_cap) {
				quiesce();   // a reduce may still read the old array
				be->release(gain_dev);
				device_bytes -= static_cast<long long>(gain_dev_cap * sizeof(bus::RouteGain));
				gain_dev_cap = 0;
				gain_dev = static_cast<bus::RouteGain*>(dev_alloc(gain_host_cap * sizeof(bus::RouteGain)));
				if (!gain_dev) {
					return false;
				}
				gain_dev_cap = gain_host_cap;
			}
			if (!be->upload(gain_dev, gain_host, static_cast<size_t>(bus_entries) * sizeof(bus::RouteGain), stream)) {
				return false;
			}
		}
		gains_dirty = false;
		return true;
	}

	// oalsfx_engine_reduce_buses with checked arguments: chunks of <= kBusChunkFrames frames, one launch per level each;
	// buses above every routed index have no members and are zeroed.  A chunk whose members all have gain 1 over its frames
	// runs the plain sum; any other reads the gains, steady (each member at its g1) or ramping.
	int reduce_buses(int frames, const float* dst, int layout, int n_buses, float* buses, void* stream)
	{
		note_stream(stream);
		if (bus_plan_dirty && !rebuild_bus_plan(stream)) {
			return fail(OALSFX_ERR_DEVICE, "Bus plan upload failed: " + be->error());
		}
		if (gains_dirty && !upload_gains(stream)) {
			return fail(OALSFX_ERR_DEVICE, "Route gain upload failed: " + be->error());
		}
		const int chunk = std::min(frames, bus::kBusChunkFrames);
		const size_t need = static_cast<size_t>(bus_partial_rows) * static_cast<size_t>(chunk) * static_cast<size_t>(bus_channels);
		if (need > bus_scratch_cap) {
			quiesce();
			be->release(bus_scratch);
			device_bytes -= static_cast<long long>(bus_scratch_cap * sizeof(float));
			bus_scratch_cap = 0;
			bus_scratch = static_cast<float*>(dev_alloc(need * sizeof(float)));
			if (!bus_scratch) {
				return fail(OALSFX_ERR_MEMORY, "Bus scratch allocation failed: " + be->error());
			}
			bus_scratch_cap = need;
		}
		bus::Chunk k;
		std::memset(&k, 0, sizeof(k));
		k.dst = dst;
		k.ts = static_cast<long long>(frames) * channels * kLanes;
		k.ls = layout == OALSFX_LAYOUT_TILED ? 1 : static_cast<long long>(frames) * channels;
		k.fs = layout == OALSFX_LAYOUT_TILED ? static_cast<long long>(channels) * kLanes : channels;
		k.cs = layout == OALSFX_LAYOUT_TILED ? kLanes : 1;
		k.frames = frames;
		k.channels = channels;
		k.bus_channels = bus_channels;
		k.pan_plan = pan_plan();
		k.pan = pan_dev;
		k.members = bus_plan_dev;
		k.levels = bus_levels;
		k.buses = buses;
		k.clock = clock_mix;
		for (int level = 0; level < bus_levels; ++level) {
			k.runs[level] = reinterpret_cast<const bus::Run*>(bus_plan_dev + bus_run_word[level]);
			k.n_runs[level] = bus_runs[level];
		}
		for (int f0 = 0; f0 < frames; f0 += bus::kBusChunkFrames) {
			k.f0 = f0;
			k.nf = std::min(frames - f0, bus::kBusChunkFrames);
			k.ramping = clock_mix + f0 < gains_ramp_end;
			k.gains = gains_unity && !k.ramping && !k.pan_plan ? nullptr : gain_dev;
			for (int level = 0; level < bus_levels; ++level) {
				k.partial[level] = bus_scratch ? bus_scratch + bus_partial_row[level] * k.nf * bus_channels : nullptr;
			}
			launches += bus_levels;
			if (!be->reduce_buses(k, stream)) {
				return fail(OALSFX_ERR_DEVICE, be->error());
			}
		}
		const long long per_bus = static_cast<long long>(frames) * bus_channels;
		if (n_buses > max_bus + 1 && !be->zero(buses + (max_bus + 1) * per_bus,
				static_cast<size_t>(n_buses - max_bus - 1) * static_cast<size_t>(per_bus) * sizeof(float), stream)) {
			return fail(OALSFX_ERR_DEVICE, be->error());
		}
		return OALSFX_OK;
	}

	// After a block that consumed updates: the lanes that were mixed have none left; paused lanes keep theirs for the
	// block that mixes them again (the reference applies changes at an Api's next mix).
	void clear_mixed_pending()
	{
		for (size_t l = 0; l < pending.size(); ++l) {
			if (active[l]) {
				pending[l] = 0;
			}
		}
	}

	template <class T>
	bool grow(T*& p, size_t& cap, size_t need)
	{
		if (need <= cap) {
			return true;
		}
		be->sync(nullptr);
		if (p) {
			device_bytes -= static_cast<long long>(cap * sizeof(T));
			be->release(p);
		}
		cap = need * 2;
		p = static_cast<T*>(dev_alloc(cap * sizeof(T)));
		return p != nullptr;
	}

	// Table mode: every class's coefficient block, every send class's five send blocks and every stream's
	// class indices go to HBM (~0.7 KB per class, 20 bytes per stream).
	bool upload_tables()
	{
		std::vector<SlotCoef> coefs(classes.size());
		for (size_t i = 0; i < classes.size(); ++i) {
			coefs[i] = classes[i].coef;
		}
		std::vector<SendCoef> sends(send_classes.size() * kSendCount);
		for (size_t i = 0; i < send_classes.size(); ++i) {
			sends[i * kSendCount] = send_classes[i].direct_coef;
			for (int k = 0; k < kMaxSlots; ++k) {
				sends[i * kSendCount + 1 + static_cast<size_t>(k)] = send_classes[i].aux_coef[k];
			}
		}
		const size_t padded = static_cast<size_t>(arena_tiles) * kLanes;
		if (!grow(slot_table_dev, slot_table_cap, coefs.size()) || !grow(send_table_dev, send_table_cap, sends.size())) {
			return false;
		}
		if (!lane_send_dev && !(lane_send_dev = static_cast<int32_t*>(dev_alloc(padded * sizeof(int32_t))))) {
			return false;
		}
		for (int s = 0; s < kMaxSlots; ++s) {
			if (!lane_class_dev[s] && !(lane_class_dev[s] = static_cast<int32_t*>(dev_alloc(padded * sizeof(int32_t))))) {
				return false;
			}
		}
		bool ok = be->upload(slot_table_dev, coefs.data(), coefs.size() * sizeof(SlotCoef), nullptr) &&
			be->upload(send_table_dev, sends.data(), sends.size() * sizeof(SendCoef), nullptr);
		std::vector<int32_t> idx(padded, 0);
		for (int s = 0; s < lane_count(); ++s) {
			idx[static_cast<size_t>(s)] = send_class[static_cast<size_t>(s)];
		}
		ok = ok && be->upload(lane_send_dev, idx.data(), padded * sizeof(int32_t), nullptr) && be->sync(nullptr);
		for (int k = 0; k < kMaxSlots && ok; ++k) {
			std::fill(idx.begin(), idx.end(), 0);
			for (int s = 0; s < lane_count(); ++s) {
				idx[static_cast<size_t>(s)] = fx_class[k][static_cast<size_t>(s)];
			}
			ok = be->upload(lane_class_dev[k], idx.data(), padded * sizeof(int32_t), nullptr) && be->sync(nullptr);
		}
		return ok;
	}

	bool rebuild_groups()
	{
		// parameter automation leaves unused classes, send classes and lookup tables behind: compact by count and by bytes
		if (classes.size() > 256 || send_classes.size() > 64 || table_bytes > compacted_at_bytes + (size_t(32) << 20)) {
			compact_classes();
		}
		quiesce();  // the group tables below are uploaded in place
		if (placed) {
			return place_streams() && build_placed_groups();
		}
		groups.clear();
		// paused streams: in no tile list, their rows zeroed by one pass per block
		std::vector<int32_t> paused_list;
		for (int s = 0; s < streams; ++s) {
			if (!active[static_cast<size_t>(s)]) {
				paused_list.push_back(s);
			}
		}
		paused_rows = static_cast<int>(paused_list.size());
		if (paused_rows > 0 && (!grow(paused_rows_dev, paused_rows_cap, paused_list.size()) ||
				!be->upload(paused_rows_dev, paused_list.data(), paused_list.size() * sizeof(int32_t), nullptr) || !be->sync(nullptr))) {
			return false;
		}
		const GroupKey k0 = key_of(0);
		bool uniform = true;
		for (int s = 1; s < streams && uniform; ++s) {
			uniform = key_of(s) == k0;
		}
		if (uniform) {
			if (!k0.paused) {
				Group g;
				g.key = k0;
				g.identity = true;
				g.tile_count = tiles;
				groups.push_back(g);
			}
			fallback_groups.clear();
			groups_dirty = false;
			return true;
		}
		std::map<GroupKey, std::vector<TileRef>> by_key;
		for (int s = 0; s < streams; ++s) {
			if (!active[static_cast<size_t>(s)]) {
				continue;
			}
			std::vector<TileRef>& v = by_key[key_of(s)];
			const uint32_t tile = static_cast<uint32_t>(s / kLanes);
			if (v.empty() || v.back().tile != tile) {
				v.push_back(TileRef{tile, 0});
			}
			v.back().mask |= 1U << (s % kLanes);
		}
		const std::map<GroupKey, std::vector<TileRef>> full_keys = by_key;
		// One launch per parameter class is fine for a handful of classes (each runs the fused kernels with
		// constant-bank coefficients).  Beyond that the launches multiply -- every class touches most tiles --
		// so the streams are grouped by effect KINDS only and the kTab* kernels fetch each stream's own
		// coefficient block from HBM.
		constexpr size_t kTableModeMinGroups = 8;
		const bool table_mode = by_key.size() > kTableModeMinGroups;
		if (table_mode) {
			by_key.clear();
			for (int s = 0; s < streams; ++s) {
				if (!active[static_cast<size_t>(s)]) {
					continue;
				}
				GroupKey k = key_of(s);
				for (int i = 0; i < kMaxSlots; ++i) {
					k.fx[i] = kind_of_type(classes[static_cast<size_t>(k.fx[i])].type);
				}
				k.send = 0;
				std::vector<TileRef>& v = by_key[k];
				const uint32_t tile = static_cast<uint32_t>(s / kLanes);
				if (v.empty() || v.back().tile != tile) {
					v.push_back(TileRef{tile, 0});
				}
				v.back().mask |= 1U << (s % kLanes);
			}
			if (!upload_tables()) {
				return false;
			}
		}
		std::vector<TileRef> all;
		for (auto& kv : by_key) {
			Group g;
			g.key = kv.first;
			g.table = table_mode;
			g.tile_begin = all.size();
			g.tile_count = static_cast<int>(kv.second.size());
			g.full_tiles = true;
			for (const TileRef& t : kv.second) {
				const int lanes_here = std::min(kLanes, streams - static_cast<int>(t.tile) * kLanes);
				const uint32_t want = (lanes_here == kLanes ? 0xFFFFFFFFU : ((1U << lanes_here) - 1U));
				g.full_tiles = g.full_tiles && t.mask == want;
			}
			all.insert(all.end(), kv.second.begin(), kv.second.end());
			groups.push_back(g);
		}
		if (all.size() > tile_list_cap) {
			be->sync(nullptr);
			be->release(tile_list);
			tile_list_cap = all.size() * 2;
			tile_list = static_cast<TileRef*>(dev_alloc(tile_list_cap * sizeof(TileRef)));
			if (!tile_list) {
				return false;
			}
		}
		if ((!all.empty() && !be->upload(tile_list, all.data(), all.size() * sizeof(TileRef), nullptr)) || !be->sync(nullptr)) {
			return false;
		}
		if (!build_multi(full_keys)) {
			return false;
		}
		groups_dirty = false;
		return true;
	}

	// Class-per-tile launch: possible when every tile holds ONE parameter class (presets assigned in runs of 32
	// streams), all classes share one slot signature that has a *_multi kernel (the fused stereo chain, or the relay
	// pipeline for anything else with one or two channels) and nothing needs the exact kernels.  One launch then
	// covers all classes at the fused kernel's speed.
	int multi_kernel = -1;
	int multi_kinds[kMaxSlots] = {};   // per slot
	bool build_multi(const std::map<GroupKey, std::vector<TileRef>>& by_key)
	{
		fallback_groups.clear();
		multi_kernel = -1;
		constexpr size_t kMultiMinGroups = 3; // one or two big classes: a constant-bank launch each is faster
		if (by_key.size() < kMultiMinGroups || !be->has_relay() || (channels != 1 && channels != 2) || (family != 2 && family != 4)) {
			return true;
		}
		std::vector<int32_t> tile_class(static_cast<size_t>(tiles), -1);
		std::vector<MixClassEntry> table;
		table.reserve(by_key.size());
		uint32_t pending_any = 0;
		const KernelInfo* infos = kernel_infos();
		bool first = true, heavy = false, chain = false;
		int active = 0;
		for (const auto& kv : by_key) {
			const GroupKey& key = kv.first;
			int kinds[kMaxSlots];
			bool ok = multi_kinds_of(key, kinds);
			if (first) {
				std::memcpy(multi_kinds, kinds, sizeof(kinds));
				chain = channels == 2 && std::memcmp(infos[kChainStereo].kind, kinds, sizeof(kinds)) == 0;
				for (int s = 0; s < kMaxSlots; ++s) {
					active += kinds[s] != kKindNull ? 1 : 0;
					heavy = heavy || kinds[s] == kKindReverb;
				}
				first = false;
			}
			ok = ok && std::memcmp(multi_kinds, kinds, sizeof(kinds)) == 0 && active >= 1;
			for (const TileRef& t : kv.second) {
				const int lanes_here = std::min(kLanes, streams - static_cast<int>(t.tile) * kLanes);
				const uint32_t want = (lanes_here == kLanes ? 0xFFFFFFFFU : ((1U << lanes_here) - 1U));
				ok = ok && t.mask == want;
				tile_class[t.tile] = static_cast<int32_t>(table.size());
			}
			if (!ok) {
				return true;
			}
			table.push_back(multi_entry(key, kinds, chain));
			pending_any |= key.pending;
		}
		if (!grow(class_table_dev, class_table_cap, table.size())) {
			return false;
		}
		if (!tile_class_dev) {
			tile_class_dev = static_cast<int32_t*>(dev_alloc(static_cast<size_t>(arena_tiles) * sizeof(int32_t)));
			if (!tile_class_dev) {
				return false;
			}
		}
		if (!be->upload(class_table_dev, table.data(), table.size() * sizeof(MixClassEntry), nullptr) ||
			!be->upload(tile_class_dev, tile_class.data(), tile_class.size() * sizeof(int32_t), nullptr) || !be->sync(nullptr)) {
			return false;
		}
		multi_kernel = chain ? kMultiChainStereo :
			channels == 1 ? (heavy ? kRelayMultiMonoHeavy : kRelayMultiMono) : (heavy ? kRelayMultiStereoHeavy : kRelayMultiStereo);
		fallback_groups.swap(groups);
		Group g;
		g.key = by_key.begin()->first;
		g.key.pending = pending_any;
		g.identity = true;
		g.multi = true;
		g.tile_count = tiles;
		if (paused_rows > 0) {
			// tiles of paused streams are not launched: the tile list of the per-key groups names every other tile once
			g.identity = false;
			g.tile_begin = 0;
			g.tile_count = 0;
			for (const Group& f : fallback_groups) {
				g.tile_count += f.tile_count;
			}
		}
		g.multi_kernel = multi_kernel;
		std::memcpy(g.multi_kinds, multi_kinds, sizeof(multi_kinds));
		groups.assign(1, g);
		return true;
	}

	// ---- stream placement (OALSFX_PLACEMENT_AUTO) ----------------------------------------------------------
	// Every arena is tile-major, base[tile * words * 32 + word * 32 + lane]: the rings of each slot, its state, the send state.
	struct Arena { uint32_t* base; int words; };
	std::vector<Arena> arenas(bool with_rings) const
	{
		std::vector<Arena> out;
		for (int s = 0; s < slots; ++s) {
			if (with_rings && ring_cap[s] > 0) {
				out.push_back(Arena{reinterpret_cast<uint32_t*>(ring[s]), ring_cap[s]});
			}
			out.push_back(Arena{slot_state[s], kSlotStateWords});
		}
		out.push_back(Arena{send_state, kSendStateWords});
		return out;
	}

	static constexpr size_t kMoveScratchWords = size_t(64) << 20; // 256 MB: the lane moves and snapshots go through it in chunks

	bool ensure_scratch(size_t words)
	{
		if (words <= move_scratch_cap) {
			return true;
		}
		be->sync(nullptr);
		if (move_scratch) {
			device_bytes -= static_cast<long long>(move_scratch_cap * sizeof(uint32_t));
			be->release(move_scratch);
		}
		move_scratch_cap = words;
		move_scratch = static_cast<uint32_t*>(dev_alloc(words * sizeof(uint32_t)));
		if (!move_scratch) {
			move_scratch_cap = 0;
		}
		return move_scratch != nullptr;
	}

	bool upload_lane_list(const std::vector<int32_t>& v)
	{
		return grow(lane_list_dev, lane_list_cap, v.size()) &&
			be->upload(lane_list_dev, v.data(), v.size() * sizeof(int32_t), nullptr) && be->sync(nullptr);
	}

	// Moves the contents of lane `first` to lane `second` in every arena, in place (the moving lanes may swap): per chunk
	// of words, a gather of the sources (in source-lane order) into the scratch arena, then a scatter sorted by destination.
	bool move_lanes(const std::vector<std::pair<int32_t, int32_t>>& moves)
	{
		if (moves.empty()) {
			return true;
		}
		const size_t n = moves.size();
		std::vector<std::pair<int32_t, int32_t>> by_src(moves);
		std::sort(by_src.begin(), by_src.end());
		std::vector<std::pair<int32_t, int32_t>> by_dst(n);   // (destination lane, scratch position)
		for (size_t p = 0; p < n; ++p) {
			by_dst[p] = std::make_pair(by_src[p].second, static_cast<int32_t>(p));
		}
		std::sort(by_dst.begin(), by_dst.end());
		std::vector<int32_t> lists(3 * n);
		for (size_t i = 0; i < n; ++i) {
			lists[i] = by_src[i].first;
			lists[n + i] = by_dst[i].first;
			lists[2 * n + i] = by_dst[i].second;
		}
		if (!upload_lane_list(lists)) {
			return false;
		}
		const int32_t* src_lanes = lane_list_dev;
		const int32_t* dst_lanes = lane_list_dev + n;
		const int32_t* scratch_pos = lane_list_dev + 2 * n;
		const size_t rows = (n + kLanes - 1) / kLanes * kLanes;
		bool ok = true;
		for (const Arena& a : arenas(true)) {
			const int cw = static_cast<int>(std::max<size_t>(1, std::min<size_t>(static_cast<size_t>(a.words), kMoveScratchWords / rows)));
			ok = ok && ensure_scratch(rows * static_cast<size_t>(cw));
			const long long ts = static_cast<long long>(a.words) * kLanes;
			for (int w0 = 0; w0 < a.words && ok; w0 += cw) {
				const int nw = std::min(cw, a.words - w0);
				const long long sts = static_cast<long long>(nw) * kLanes;
				ok = be->copy_lanes(move_scratch, sts, 0, a.base, ts, w0, nw, src_lanes, nullptr, static_cast<int>(n), nullptr) &&
					be->copy_lanes(a.base, ts, w0, move_scratch, sts, 0, nw, scratch_pos, dst_lanes, static_cast<int>(n), nullptr);
			}
		}
		return ok && be->sync(nullptr);
	}

	// More tiles in every arena: the new buffers are allocated first, so a failure leaves the engine as it was.  Rings
	// are tile-major: the old contents are one prefix of the new buffer.
	bool grow_arena(int new_tiles)
	{
		struct Resize { void** p; size_t tile_bytes; void* fresh; };
		std::vector<Resize> list;
		for (int s = 0; s < slots; ++s) {
			if (ring[s]) {
				list.push_back(Resize{reinterpret_cast<void**>(&ring[s]), static_cast<size_t>(ring_cap[s]) * kLanes * sizeof(float), nullptr});
			}
			list.push_back(Resize{reinterpret_cast<void**>(&slot_state[s]), static_cast<size_t>(kSlotStateWords) * kLanes * sizeof(uint32_t), nullptr});
		}
		list.push_back(Resize{reinterpret_cast<void**>(&send_state), static_cast<size_t>(kSendStateWords) * kLanes * sizeof(uint32_t), nullptr});
		if (tile_class_dev) {
			list.push_back(Resize{reinterpret_cast<void**>(&tile_class_dev), sizeof(int32_t), nullptr});
		}
		for (Resize& r : list) {
			r.fresh = dev_alloc(r.tile_bytes * static_cast<size_t>(new_tiles));
			if (!r.fresh) {
				for (Resize& q : list) {
					if (q.fresh) {
						be->release(q.fresh);
						device_bytes -= static_cast<long long>(q.tile_bytes) * new_tiles;
					}
				}
				return false;
			}
		}
		bool ok = true;
		for (Resize& r : list) {
			ok = ok && be->copy_2d(r.fresh, r.tile_bytes, *r.p, r.tile_bytes, r.tile_bytes, static_cast<size_t>(arena_tiles), nullptr);
		}
		ok = ok && be->sync(nullptr);
		for (Resize& r : list) {
			be->release(*r.p);
			device_bytes -= static_cast<long long>(r.tile_bytes) * arena_tiles;
			*r.p = r.fresh;
		}
		// the table-mode lane arrays are re-created at their next upload
		const long long lane_array_bytes = static_cast<long long>(arena_tiles) * kLanes * static_cast<long long>(sizeof(int32_t));
		if (lane_send_dev) {
			be->release(lane_send_dev);
			lane_send_dev = nullptr;
			device_bytes -= lane_array_bytes;
		}
		for (int s = 0; s < kMaxSlots; ++s) {
			if (lane_class_dev[s]) {
				be->release(lane_class_dev[s]);
				lane_class_dev[s] = nullptr;
				device_bytes -= lane_array_bytes;
			}
		}
		arena_tiles = new_tiles;
		const size_t lanes = static_cast<size_t>(new_tiles) * kLanes;
		for (int s = 0; s < kMaxSlots; ++s) {
			fx_class[s].resize(lanes, 0);
		}
		send_class.resize(lanes, send_class[0]);
		pending.resize(lanes, 0);
		active.resize(lanes, 1);
		stream_of_lane.resize(lanes, -1);
		tile_key.resize(static_cast<size_t>(new_tiles));
		tile_active.resize(static_cast<size_t>(new_tiles), 0);
		return ok;
	}

	// The configuration vectors become lane-indexed over the arena; the streams stay where they are until the next mix.
	void enter_placed()
	{
		const size_t lanes = static_cast<size_t>(arena_tiles) * kLanes;
		lane_of_stream.resize(static_cast<size_t>(streams));
		stream_of_lane.assign(lanes, -1);
		for (int s = 0; s < streams; ++s) {
			lane_of_stream[static_cast<size_t>(s)] = s;
			stream_of_lane[static_cast<size_t>(s)] = s;
		}
		for (int s = 0; s < kMaxSlots; ++s) {
			fx_class[s].resize(lanes, 0);
		}
		send_class.resize(lanes, send_class[0]);
		pending.resize(lanes, 0);
		active.resize(lanes, 1);
		paused_rows = 0;
		tile_key.assign(static_cast<size_t>(arena_tiles), GroupKey());
		tile_active.assign(static_cast<size_t>(arena_tiles), 0);
		refill_padding = true;
		placed = true;
	}

	// Every stream back to lane = stream, the configuration vectors back to caller order.
	bool leave_placed()
	{
		std::vector<std::pair<int32_t, int32_t>> moves;
		for (int s = 0; s < streams; ++s) {
			if (lane_of_stream[static_cast<size_t>(s)] != s) {
				moves.push_back(std::make_pair(lane_of_stream[static_cast<size_t>(s)], s));
			}
		}
		if (!move_lanes(moves)) {
			return false;
		}
		auto to_caller = [&](auto& v) {
			auto out = v;
			out.resize(static_cast<size_t>(streams));
			for (int s = 0; s < streams; ++s) {
				out[static_cast<size_t>(s)] = v[static_cast<size_t>(lane_of_stream[static_cast<size_t>(s)])];
			}
			v.swap(out);
		};
		for (int s = 0; s < kMaxSlots; ++s) {
			to_caller(fx_class[s]);
		}
		to_caller(send_class);
		to_caller(pending);
		to_caller(active);
		placed = false;
		lane_of_stream.clear();
		stream_of_lane.clear();
		tile_key.clear();
		tile_active.clear();
		return true;
	}

	// The placement itself (run before the groups are built, engine quiesced).  Keyed on the full GroupKey -- pending bits
	// included, so that the block that consumes an update is class-pure as well.  Afterwards:
	//   1. every tile that holds a caller stream holds one key; its padding lanes carry that key;
	//   2. a stream already in a pure tile of its key is not moved (except by 3), so changing k streams moves about k;
	//   3. a key of n streams spans at most ceil(n / 32) + 1 tiles, else it is re-packed into ceil(n / 32);
	//   4. freed tiles are reused before the arenas grow; they never shrink.
	bool place_streams()
	{
		place_oom = false;
		const int T = arena_tiles;
		std::map<GroupKey, int> ids;
		std::vector<GroupKey> keys;
		std::vector<int> kid(static_cast<size_t>(streams));
		for (int s = 0; s < streams; ++s) {
			const GroupKey k = key_of(lane_of_stream[static_cast<size_t>(s)]);
			auto it = ids.emplace(k, static_cast<int>(keys.size()));
			if (it.second) {
				keys.push_back(k);
			}
			kid[static_cast<size_t>(s)] = it.first->second;
		}
		const int K = static_cast<int>(keys.size());
		// each tile stays with the key most of its streams have (ties: the key seen first); the others move
		std::vector<int> owner(static_cast<size_t>(T), -1), kept(static_cast<size_t>(T), 0);
		for (int t = 0; t < T; ++t) {
			int ids_here[kLanes], counts[kLanes], distinct = 0;
			for (int l = t * kLanes; l < (t + 1) * kLanes; ++l) {
				const int s = stream_of_lane[static_cast<size_t>(l)];
				if (s < 0) {
					continue;
				}
				const int k = kid[static_cast<size_t>(s)];
				int j = 0;
				while (j < distinct && ids_here[j] != k) {
					++j;
				}
				if (j == distinct) {
					ids_here[distinct] = k;
					counts[distinct++] = 0;
				}
				++counts[j];
			}
			for (int j = 0; j < distinct; ++j) {
				if (counts[j] > kept[static_cast<size_t>(t)] || (counts[j] == kept[static_cast<size_t>(t)] && ids_here[j] < owner[static_cast<size_t>(t)])) {
					owner[static_cast<size_t>(t)] = ids_here[j];
					kept[static_cast<size_t>(t)] = counts[j];
				}
			}
		}
		std::vector<std::vector<int>> owned(static_cast<size_t>(K)), movers(static_cast<size_t>(K));
		std::vector<int> members(static_cast<size_t>(K), 0);
		for (int t = 0; t < T; ++t) {
			if (owner[static_cast<size_t>(t)] >= 0) {
				owned[static_cast<size_t>(owner[static_cast<size_t>(t)])].push_back(t);
			}
		}
		for (int s = 0; s < streams; ++s) {
			const int k = kid[static_cast<size_t>(s)];
			++members[static_cast<size_t>(k)];
			if (owner[static_cast<size_t>(lane_of_stream[static_cast<size_t>(s)] / kLanes)] != k) {
				movers[static_cast<size_t>(k)].push_back(s);
			}
		}
		auto new_tiles_for = [&](int k) {
			long long kept_k = 0;
			for (int t : owned[static_cast<size_t>(k)]) {
				kept_k += kept[static_cast<size_t>(t)];
			}
			const long long spare = static_cast<long long>(owned[static_cast<size_t>(k)].size()) * kLanes - kept_k;
			const long long extra = static_cast<long long>(movers[static_cast<size_t>(k)].size()) - spare;
			return static_cast<int>(extra > 0 ? (extra + kLanes - 1) / kLanes : 0);
		};
		for (int k = 0; k < K; ++k) {
			std::vector<int>& mine = owned[static_cast<size_t>(k)];
			const int bound = (members[static_cast<size_t>(k)] + kLanes - 1) / kLanes;
			if (static_cast<int>(mine.size()) + new_tiles_for(k) <= bound + 1) {
				continue;
			}
			// re-pack: keep the fullest `bound` tiles, the streams of the others move into their free lanes
			std::stable_sort(mine.begin(), mine.end(), [&](int a, int b) { return kept[static_cast<size_t>(a)] > kept[static_cast<size_t>(b)]; });
			for (size_t i = static_cast<size_t>(bound); i < mine.size(); ++i) {
				const int t = mine[i];
				owner[static_cast<size_t>(t)] = -1;
				for (int l = t * kLanes; l < (t + 1) * kLanes; ++l) {
					const int s = stream_of_lane[static_cast<size_t>(l)];
					if (s >= 0 && kid[static_cast<size_t>(s)] == k) {
						movers[static_cast<size_t>(k)].push_back(s);
					}
				}
			}
			mine.resize(std::min(mine.size(), static_cast<size_t>(bound)));
			std::sort(movers[static_cast<size_t>(k)].begin(), movers[static_cast<size_t>(k)].end());
		}
		// new tiles: freed ones first (lowest index), then growth
		std::vector<int> free_tiles;
		for (int t = 0; t < T; ++t) {
			if (owner[static_cast<size_t>(t)] < 0) {
				free_tiles.push_back(t);
			}
		}
		size_t next_free = 0;
		int new_T = T;
		for (int k = 0; k < K; ++k) {
			for (int n = new_tiles_for(k); n > 0; --n) {
				owned[static_cast<size_t>(k)].push_back(next_free < free_tiles.size() ? free_tiles[next_free++] : new_T++);
			}
		}
		// Growing copies every arena: grow by an eighth or by one spare tile per key, whichever is more, so that the new
		// (class, pending) tiles of later updates and the partial tiles they leave behind find free tiles instead of
		// another copy of the whole arena.
		if (new_T > T) {
			new_T = std::max(new_T + K, T + (T + 7) / 8);
		}
		if (new_T > T && !grow_arena(new_T)) {
			place_oom = true;
			return false;
		}
		owner.resize(static_cast<size_t>(new_T), -1);
		for (int k = 0; k < K; ++k) {
			for (int t : owned[static_cast<size_t>(k)]) {
				owner[static_cast<size_t>(t)] = k;
			}
		}
		// movers into the free lanes of their key's tiles, in stream order
		std::vector<int32_t> next_sol(stream_of_lane);
		std::vector<uint8_t> touched(static_cast<size_t>(new_T), 0);
		for (int k = 0; k < K; ++k) {
			for (int s : movers[static_cast<size_t>(k)]) {
				const int l = lane_of_stream[static_cast<size_t>(s)];
				next_sol[static_cast<size_t>(l)] = -1;
				touched[static_cast<size_t>(l / kLanes)] = 1;
			}
		}
		std::vector<std::pair<int32_t, int32_t>> moves;
		for (int k = 0; k < K; ++k) {
			size_t m = 0;
			for (int t : owned[static_cast<size_t>(k)]) {
				for (int l = t * kLanes; l < (t + 1) * kLanes && m < movers[static_cast<size_t>(k)].size(); ++l) {
					if (next_sol[static_cast<size_t>(l)] < 0) {
						const int s = movers[static_cast<size_t>(k)][m++];
						next_sol[static_cast<size_t>(l)] = s;
						touched[static_cast<size_t>(t)] = 1;
						if (lane_of_stream[static_cast<size_t>(s)] != l) {
							moves.push_back(std::make_pair(lane_of_stream[static_cast<size_t>(s)], l));
						}
					}
				}
			}
		}
		if (!move_lanes(moves)) {
			return false;
		}
		for (int s = 0; s < kMaxSlots; ++s) {
			const std::vector<int> before(fx_class[s]);
			for (const auto& mv : moves) {
				fx_class[s][static_cast<size_t>(mv.second)] = before[static_cast<size_t>(mv.first)];
			}
		}
		const std::vector<int> send_before(send_class);
		const std::vector<uint8_t> pending_before(pending);
		const std::vector<uint8_t> active_before(active);
		for (const auto& mv : moves) {
			send_class[static_cast<size_t>(mv.second)] = send_before[static_cast<size_t>(mv.first)];
			pending[static_cast<size_t>(mv.second)] = pending_before[static_cast<size_t>(mv.first)];
			active[static_cast<size_t>(mv.second)] = active_before[static_cast<size_t>(mv.first)];
		}
		stream_of_lane.swap(next_sol);
		for (const auto& mv : moves) {
			lane_of_stream[static_cast<size_t>(stream_of_lane[static_cast<size_t>(mv.second)])] = mv.second;
		}
		// padding lanes: their tile's key, and (where the tile changed) a tile-mate's slot and send state -- the kernels'
		// warp-uniform checks (ring offsets) then see the padding lanes agree with the tile
		std::vector<int32_t> pad_to, pad_from;
		for (int t = 0; t < new_T; ++t) {
			const int k = owner[static_cast<size_t>(t)];
			int mate = -1;
			for (int l = t * kLanes; l < (t + 1) * kLanes && mate < 0; ++l) {
				mate = stream_of_lane[static_cast<size_t>(l)] >= 0 ? l : -1;
			}
			const bool occupied = mate >= 0;
			const bool changed = refill_padding || touched[static_cast<size_t>(t)] || !tile_active[static_cast<size_t>(t)] ||
				!(tile_key[static_cast<size_t>(t)] == keys[static_cast<size_t>(std::max(k, 0))]);
			tile_active[static_cast<size_t>(t)] = occupied ? 1 : 0;
			if (!occupied) {
				continue;
			}
			const GroupKey& key = keys[static_cast<size_t>(k)];
			tile_key[static_cast<size_t>(t)] = key;
			for (int l = t * kLanes; l < (t + 1) * kLanes; ++l) {
				if (stream_of_lane[static_cast<size_t>(l)] >= 0) {
					continue;
				}
				for (int s = 0; s < kMaxSlots; ++s) {
					fx_class[s][static_cast<size_t>(l)] = key.fx[s];
				}
				send_class[static_cast<size_t>(l)] = key.send;
				pending[static_cast<size_t>(l)] = static_cast<uint8_t>(key.pending);
				active[static_cast<size_t>(l)] = key.paused ? 0 : 1;
				if (changed) {
					pad_to.push_back(l);
					pad_from.push_back(mate);
				}
			}
		}
		refill_padding = false;
		if (!pad_to.empty()) {
			std::vector<int32_t> lists(pad_from);
			lists.insert(lists.end(), pad_to.begin(), pad_to.end());
			if (!upload_lane_list(lists)) {
				return false;
			}
			const int n = static_cast<int>(pad_to.size());
			for (const Arena& a : arenas(false)) {
				const long long ts = static_cast<long long>(a.words) * kLanes;
				if (!be->copy_lanes(a.base, ts, 0, a.base, ts, 0, a.words, lane_list_dev, lane_list_dev + n, n, nullptr)) {
					return false;
				}
			}
		}
		std::vector<int32_t> lane_map(stream_of_lane);
		for (size_t l = 0; l < lane_map.size(); ++l) {
			if (lane_map[l] >= 0 && !active[l]) {
				lane_map[l] = -2 - lane_map[l];
			}
		}
		return grow(stream_of_lane_dev, stream_of_lane_cap, lane_map.size()) &&
			be->upload(stream_of_lane_dev, lane_map.data(), lane_map.size() * sizeof(int32_t), nullptr) && be->sync(nullptr);
	}

	// Groups of a placed engine: the active tiles only, every one of them whole and of one key.  Each slot signature with
	// enough keys gets ONE class-per-tile launch; the remaining keys run per key (a handful) or in table mode.  For blocks
	// the class-per-tile kernels cannot take (frames < 2), fallback_groups covers every key without them.
	bool build_placed_groups()
	{
		constexpr size_t kTableModeMinGroups = 8; // as in rebuild_groups
		constexpr size_t kMultiMinGroups = 3;     // as in build_multi
		groups.clear();
		fallback_groups.clear();
		multi_kernel = -1;
		std::map<GroupKey, std::vector<TileRef>> by_key;
		for (int t = 0; t < arena_tiles; ++t) {
			if (tile_active[static_cast<size_t>(t)] && !tile_key[static_cast<size_t>(t)].paused) {
				by_key[tile_key[static_cast<size_t>(t)]].push_back(TileRef{static_cast<uint32_t>(t), 0xFFFFFFFFU});
			}
		}
		std::vector<TileRef> all;
		std::vector<MixClassEntry> table;
		std::vector<int32_t> tile_class(static_cast<size_t>(arena_tiles), -1);
		std::map<std::vector<int>, std::vector<const GroupKey*>> by_signature;
		std::map<GroupKey, std::vector<TileRef>> rest;
		const bool multi_ok = be->has_relay() && (channels == 1 || channels == 2) && (family == 2 || family == 4);
		for (const auto& kv : by_key) {
			int kinds[kMaxSlots];
			bool ok = multi_ok && multi_kinds_of(kv.first, kinds);
			int active = 0;
			for (int s = 0; s < kMaxSlots; ++s) {
				active += kinds[s] != kKindNull ? 1 : 0;
			}
			if (ok && active >= 1) {
				by_signature[std::vector<int>(kinds, kinds + kMaxSlots)].push_back(&kv.first);
			} else {
				rest.insert(kv);
			}
		}
		const KernelInfo* infos = kernel_infos();
		for (const auto& sig : by_signature) {
			if (sig.second.size() < kMultiMinGroups) { // one or two big classes: a constant-bank launch each is faster
				for (const GroupKey* k : sig.second) {
					rest.emplace(*k, by_key[*k]);
				}
				continue;
			}
			const int* kinds = sig.first.data();
			const bool chain = channels == 2 && std::memcmp(infos[kChainStereo].kind, kinds, sizeof(int) * kMaxSlots) == 0;
			bool heavy = false;
			for (int s = 0; s < kMaxSlots; ++s) {
				heavy = heavy || kinds[s] == kKindReverb;
			}
			Group g;
			g.key = *sig.second.front();
			g.key.pending = 0;
			g.multi = true;
			g.tile_begin = all.size();
			for (const GroupKey* k : sig.second) {
				for (const TileRef& t : by_key[*k]) {
					tile_class[t.tile] = static_cast<int32_t>(table.size());
					all.push_back(t);
				}
				table.push_back(multi_entry(*k, kinds, chain));
				g.key.pending |= k->pending;
			}
			g.tile_count = static_cast<int>(all.size() - g.tile_begin);
			g.multi_kernel = chain ? kMultiChainStereo :
				channels == 1 ? (heavy ? kRelayMultiMonoHeavy : kRelayMultiMono) : (heavy ? kRelayMultiStereoHeavy : kRelayMultiStereo);
			std::memcpy(g.multi_kinds, kinds, sizeof(g.multi_kinds));
			groups.push_back(g);
		}
		bool tables_needed = false;
		auto add_groups = [&](const std::map<GroupKey, std::vector<TileRef>>& keyed, std::vector<Group>& out) {
			const bool table_mode = keyed.size() > kTableModeMinGroups;
			std::map<GroupKey, std::vector<TileRef>> by_kinds;
			const std::map<GroupKey, std::vector<TileRef>>* src = &keyed;
			if (table_mode) {
				tables_needed = true;
				for (const auto& kv : keyed) {
					GroupKey k = kv.first;
					for (int i = 0; i < kMaxSlots; ++i) {
						k.fx[i] = kind_of_type(classes[static_cast<size_t>(k.fx[i])].type);
					}
					k.send = 0;
					std::vector<TileRef>& v = by_kinds[k];
					v.insert(v.end(), kv.second.begin(), kv.second.end());
				}
				src = &by_kinds;
			}
			for (const auto& kv : *src) {
				Group g;
				g.key = kv.first;
				g.table = table_mode;
				g.full_tiles = true;
				g.tile_begin = all.size();
				g.tile_count = static_cast<int>(kv.second.size());
				all.insert(all.end(), kv.second.begin(), kv.second.end());
				out.push_back(g);
			}
		};
		add_groups(rest, groups);
		if (!table.empty()) {
			add_groups(by_key, fallback_groups);
		}
		if (tables_needed && !upload_tables()) {
			return false;
		}
		if (all.size() > tile_list_cap) {
			be->sync(nullptr);
			be->release(tile_list);
			device_bytes -= static_cast<long long>(tile_list_cap * sizeof(TileRef));
			tile_list_cap = all.size() * 2;
			tile_list = static_cast<TileRef*>(dev_alloc(tile_list_cap * sizeof(TileRef)));
			if (!tile_list) {
				tile_list_cap = 0;
				return false;
			}
		}
		if (!all.empty() && !be->upload(tile_list, all.data(), all.size() * sizeof(TileRef), nullptr)) {
			return false;
		}
		if (!table.empty()) {
			if (!grow(class_table_dev, class_table_cap, table.size())) {
				return false;
			}
			if (!tile_class_dev && !(tile_class_dev = static_cast<int32_t*>(dev_alloc(static_cast<size_t>(arena_tiles) * sizeof(int32_t))))) {
				return false;
			}
			if (!be->upload(class_table_dev, table.data(), table.size() * sizeof(MixClassEntry), nullptr) ||
				!be->upload(tile_class_dev, tile_class.data(), tile_class.size() * sizeof(int32_t), nullptr)) {
				return false;
			}
		}
		if (!be->sync(nullptr)) {
			return false;
		}
		groups_dirty = false;
		return true;
	}

	// Snapshot / restore of a placed engine: every arena in caller stream order (stream s at tile s / 32, lane s % 32;
	// zeros past the last stream), `tiles` tiles per arena, gathered through the scratch arena in chunks of whole tiles.
	// (snapshot: `out` receives the arenas; restore: `in` holds them)
	bool canonical_state(char* out, const char* in)
	{
		std::vector<int32_t> canon(static_cast<size_t>(tiles) * kLanes, -1);
		for (int s = 0; s < streams; ++s) {
			canon[static_cast<size_t>(s)] = lane_of_stream[static_cast<size_t>(s)];
		}
		if (!upload_lane_list(canon)) {
			return false;
		}
		bool ok = true;
		for (const Arena& a : arenas(true)) {
			const size_t tile_words = static_cast<size_t>(a.words) * kLanes;
			const int per = static_cast<int>(std::max<size_t>(1, std::min<size_t>(static_cast<size_t>(tiles), kMoveScratchWords / tile_words)));
			ok = ok && ensure_scratch(tile_words * static_cast<size_t>(per));
			const long long ts = static_cast<long long>(tile_words);
			for (int t0 = 0; t0 < tiles && ok; t0 += per) {
				const int nt = std::min(per, tiles - t0);
				const size_t bytes = tile_words * static_cast<size_t>(nt) * sizeof(uint32_t);
				const int32_t* lanes = lane_list_dev + static_cast<size_t>(t0) * kLanes;
				if (in) {
					ok = be->upload(move_scratch, in, bytes, nullptr) &&
						be->copy_lanes(a.base, ts, 0, move_scratch, ts, 0, a.words, nullptr, lanes, nt * kLanes, nullptr) && be->sync(nullptr);
				} else {
					ok = be->copy_lanes(move_scratch, ts, 0, a.base, ts, 0, a.words, lanes, nullptr, nt * kLanes, nullptr) &&
						be->download(out, move_scratch, bytes, nullptr) && be->sync(nullptr);
				}
				if (in) {
					in += bytes;
				} else {
					out += bytes;
				}
			}
		}
		return ok;
	}

	// Class-per-tile eligibility of one key: its slot kinds, and false when it needs the exact kernels (an active send
	// filter, an unstable filter design).
	bool multi_kinds_of(const GroupKey& key, int kinds[kMaxSlots]) const
	{
		const SendClass& sc = send_classes[static_cast<size_t>(key.send)];
		bool ok = sc.direct_coef.filter_type == 0;
		for (int s = 0; s < kMaxSlots; ++s) {
			const FxClass& fc = classes[static_cast<size_t>(key.fx[s])];
			kinds[s] = kind_of_type(fc.type);
			ok = ok && (kinds[s] == kKindNull || sc.aux_coef[s].filter_type == 0) && !(fc.coef.flags & kCoefUnstable);
		}
		return ok;
	}

	// The class-table entry of one key: its coefficient blocks as the kernel arguments would hold them.
	MixClassEntry multi_entry(const GroupKey& key, const int kinds[kMaxSlots], bool chain) const
	{
		Group g;
		g.key = key;
		MixArgs a;
		fill_common(a, g, 2, nullptr, nullptr, OALSFX_LAYOUT_STREAM_MAJOR, 2, 0);
		MixClassEntry e;
		std::memset(&e, 0, sizeof(e));
		int pos = 0;
		for (int s = 0; s < kMaxSlots; ++s) { // the chain kernel addresses slots by index, the relay by compacted position
			if (chain || kinds[s] != kKindNull) {
				fill_slot(a, g, pos, s, false);
				e.pending |= ((key.pending >> s) & 1U) << pos;
				++pos;
			}
		}
		sanitize_gains(a);
		std::memcpy(e.coefs, reinterpret_cast<const char*>(&a) + kMixCoefOffset, kMixCoefBytes);
		return e;
	}

	// ---- launching ----------------------------------------------------------------------------------
	void fill_common(MixArgs& a, const Group& g, int frames, const float* src, float* dst, int layout,
		long long frames_total, long long frame0) const
	{
		std::memset(&a, 0, sizeof(a));
		a.frames = frames;
		a.channels = channels;
		a.num_streams = lane_count();
		if (layout == OALSFX_LAYOUT_TILED) {
			a.io_ts = frames_total * channels * kLanes;
			a.io_ls = 1;
			a.io_fs = static_cast<long long>(channels) * kLanes;
			a.io_cs = kLanes;
		} else {
			a.io_ts = frames_total * channels * kLanes;
			a.io_ls = frames_total * channels;
			a.io_fs = channels;
			a.io_cs = 1;
		}
		a.src = src + frame0 * a.io_fs;
		a.dst = dst + frame0 * a.io_fs;
		a.tiles = g.identity ? nullptr : tile_list + g.tile_begin;
		a.tile_count = g.tile_count;
		if (g.identity && slice_count > 0) { // host-buffer pipelining: only tiles [slice_first, +slice_count)
			a.tile_first = slice_first;
			a.tile_count = slice_count;
		}
		a.send_state = send_state;
		if (g.table) {
			a.slot_table = slot_table_dev;
			a.send_table = send_table_dev;
			a.lane_send = lane_send_dev;
			return;
		}
		const SendClass& sc = send_classes[static_cast<size_t>(g.key.send)];
		a.direct = sc.direct_coef;
	}

	void fill_slot(MixArgs& a, const Group& g, int pos, int slot, bool first_block) const
	{
		if (g.table) {
			a.lane_class[pos] = lane_class_dev[slot];
		} else {
			const FxClass& fc = classes[static_cast<size_t>(g.key.fx[slot])];
			const SendClass& sc = send_classes[static_cast<size_t>(g.key.send)];
			a.slot[pos] = fc.coef;
			a.aux[pos] = sc.aux_coef[slot];
		}
		a.aux_index[pos] = slot;
		a.ring[pos] = ring[slot];
		a.ring_tile_stride[pos] = static_cast<long long>(ring_cap[slot]) * kLanes;
		a.slot_state[pos] = slot_state[slot];
		if (first_block && ((g.key.pending >> slot) & 1U)) {
			a.update_mask |= 1U << pos;
		}
	}

	// Fast kernels add `sample * gain` unconditionally: make every static gain the reference would
	// skip (|g| <= 1e-5, oalsfxpp.cpp:56) an exact zero so the sum is unchanged.
	static void sanitize(float* gains, int n)
	{
		for (int i = 0; i < n; ++i) {
			if (!(std::fabs(gains[i]) > kSilenceGain)) {
				gains[i] = 0.0F;
			}
		}
	}

	static void sanitize_gains(MixArgs& a)
	{
		sanitize(&a.direct.gains[0][0], kMaxChannels * kMaxChannels);
		for (int p = 0; p < kMaxSlots; ++p) {
			sanitize(&a.aux[p].gains[0][0], kMaxChannels * kMaxChannels);
			SlotCoef& sc = a.slot[p];
			switch (kind_of_type(sc.type)) {
			case kKindModDelay: sanitize(&sc.u.mod_delay.gains[0][0], 2 * kMaxChannels); break;
			case kKindCompressor: sanitize(&sc.u.compressor.gains[0][0], kWetChannels * kMaxChannels); break;
			case kKindDedicated: sanitize(sc.u.dedicated.gains, kMaxChannels); break;
			case kKindDistortion: sanitize(sc.u.distortion.gains, kMaxChannels); break;
			case kKindEcho: sanitize(&sc.u.echo.gains[0][0], 2 * kMaxChannels); break;
			case kKindEqualizer: sanitize(&sc.u.equalizer.gains[0][0], kWetChannels * kMaxChannels); break;
			case kKindRingMod: sanitize(&sc.u.ring_mod.gains[0][0], kWetChannels * kMaxChannels); break;
			default: break; // reverb: its pan gains are running state, tested per sub-chunk on the device
			}
		}
	}

	bool launch_group(const Group& g, int frames, const float* src, float* dst, int layout,
		long long frames_total, long long frame0, bool first_block, void* stream)
	{
		if (g.multi) {
			MixArgs a;
			fill_common(a, g, frames, src, dst, layout, frames_total, frame0);
			a.with_dry = 1;
			const bool chain = g.multi_kernel == kMultiChainStereo;
			int pos = 0, floats = 0;
			for (int s = 0; s < kMaxSlots; ++s) {
				if (chain || g.multi_kinds[s] != kKindNull) {
					fill_slot(a, g, pos, s, false); // pointers and strides; the coefficient blocks come from the class table
					a.relay_kind[pos] = g.multi_kinds[s];
					a.relay_win[pos] = floats;
					floats += g.multi_kinds[s] == kKindReverb ? kPfWarpFloats :
						(g.multi_kinds[s] == kKindModDelay || g.multi_kinds[s] == kKindEcho) ? kFwWarpFloats : 0;
					++pos;
				}
			}
			a.relay_count = pos;
			a.relay_smem_floats = floats;
			a.update_mask = first_block ? 0xFFFFFFFFU : 0U;
			a.class_table = class_table_dev;
			a.tile_class = tile_class_dev;
			++launches;
			return mix_launch(g.multi_kernel, a, stream);
		}
		if (g.table) {
			// key.fx[] holds the kinds; one exact single-effect pass per slot, coefficients from the tables
			bool first = true;
			for (int s = 0; s < kMaxSlots; ++s) {
				if (g.key.fx[s] == kKindNull) {
					continue;
				}
				MixArgs a;
				fill_common(a, g, frames, src, dst, layout, frames_total, frame0);
				a.with_dry = first ? 1 : 0;
				a.accumulate = first ? 0 : 1;
				fill_slot(a, g, 0, s, first_block);
				++launches;
				if (!mix_launch(tab_kernel_for_kind(g.key.fx[s]), a, stream)) {
					return false;
				}
				first = false;
			}
			if (first) {
				MixArgs a;
				fill_common(a, g, frames, src, dst, layout, frames_total, frame0);
				a.with_dry = 1;
				fill_slot(a, g, 0, 0, first_block);
				++launches;
				return mix_launch(kTabDry, a, stream);
			}
			return true;
		}
		const SendClass& sc = send_classes[static_cast<size_t>(g.key.send)];
		int kinds[kMaxSlots];
		bool send_filter = sc.direct_coef.filter_type != 0;   // a send's shelf filter is active (apply_filters, oalsfxpp.cpp:3101-3143)
		bool unstable = false;
		for (int s = 0; s < kMaxSlots; ++s) {
			const int type = classes[static_cast<size_t>(g.key.fx[s])].type;
			kinds[s] = kind_of_type(type);
			if (kinds[s] != kKindNull && sc.aux_coef[s].filter_type != 0) {
				send_filter = true;
			}
			if (classes[static_cast<size_t>(g.key.fx[s])].coef.flags & kCoefUnstable) {
				unstable = true; // keeps the group on the exact (generic) kernels, see coefs.h
			}
		}
		const bool any_filter = send_filter || unstable;
		// The relay pipeline (relay.cuh): any signature of two or more effects in one launch, one warp per effect.
		const bool whole_tiles_group = g.identity || g.full_tiles;
		int active = 0;
		for (int s = 0; s < kMaxSlots; ++s) {
			active += kinds[s] != kKindNull ? 1 : 0;
		}
		// (with an active send filter the relay's filter-carrying variant is the only one-launch kernel: also for one slot)
		const bool relay_ok = be->has_relay() && !unstable && frames >= 2 && whole_tiles_group &&
			active >= (send_filter ? 1 : 2) && family != 0;
		auto launch_relay = [&]() {
			MixArgs a;
			fill_common(a, g, frames, src, dst, layout, frames_total, frame0);
			a.with_dry = 1;
			int pos = 0, floats = 0;
			bool heavy = false;
			for (int s = 0; s < kMaxSlots; ++s) {
				if (kinds[s] == kKindNull) {
					continue;
				}
				fill_slot(a, g, pos, s, first_block);
				a.relay_kind[pos] = kinds[s];
				a.relay_win[pos] = floats;
				floats += kinds[s] == kKindReverb ? kPfWarpFloats : (kinds[s] == kKindModDelay || kinds[s] == kKindEcho) ? kFwWarpFloats : 0;
				heavy = heavy || kinds[s] == kKindReverb;
				++pos;
			}
			a.relay_count = pos;
			a.relay_smem_floats = floats;
			sanitize_gains(a);
			++launches;
			// quad / 5.1 / 6.1 / 7.1: the kernels with a run-time channel count
			if (send_filter) {
				return mix_launch(channels == 1 ? (heavy ? kRelaySfMonoHeavy : kRelaySfMono) : channels == 2 ? (heavy ? kRelaySfStereoHeavy : kRelaySfStereo) :
					(heavy ? kRelaySfWideHeavy : kRelaySfWide), a, stream);
			}
			return mix_launch(channels == 1 ? (heavy ? kRelayMonoHeavy : kRelayMono) : channels == 2 ? (heavy ? kRelayStereoHeavy : kRelayStereo) :
				(heavy ? kRelayWideHeavy : kRelayWide), a, stream);
		};
		if (relay_ok && family == 5) { // OALSFX_KERNEL=relay: wherever eligible (A/B measurements, parity tests)
			return launch_relay();
		}
		// Opt-in (OALSFX_SCAN=1): a lone equalizer slot on few streams as a linear-recurrence scan over time (scan.cuh).
		// Re-associates the filter sums: within 1e-5 of the reference, not bit-exact -- hence never chosen by default.
		if (scan_enabled && be->has_relay() && active == 1 && !any_filter && g.identity && slice_count == 0 &&
			(channels == 1 || channels == 2) && frames >= 64 && streams <= 4096) {
			for (int s = 0; s < kMaxSlots; ++s) {
				if (kinds[s] == kKindEqualizer) {
					MixArgs a;
					fill_common(a, g, frames, src, dst, layout, frames_total, frame0);
					a.with_dry = 1;
					fill_slot(a, g, 0, s, first_block);
					sanitize_gains(a);
					++launches;
					return mix_launch(channels == 1 ? kScanEqualizerMono : kScanEqualizerStereo, a, stream);
				}
			}
		}
		// A fused single-pass kernel for this signature?
		const KernelInfo* infos = kernel_infos();
		for (int k = 0; k < kKernelCount; ++k) {
			const KernelInfo& ki = infos[k];
			if (ki.ct != channels || ki.sf || any_filter || frames < 2) {
				continue;
			}
			if (std::memcmp(ki.kind, kinds, sizeof(kinds)) != 0) {
				continue;
			}
			// A signature whose only fused kernel is the thread-per-stream one (cfg3's flanger + ring modulator +
			// distortion + compressor): below ~1000 tiles a stream's serial per-sample work bounds the block, and
			// the relay pipeline (a warp per effect) halves it -- B200, ms per 1024-frame block, mono 96 kHz:
			// 32 tiles 0.58 vs 1.08, 512 tiles 0.76 vs 1.40; 2048 tiles 2.34 vs 1.83 (throughput-bound: fewer
			// instructions win).
			constexpr int kRelayMaxTiles = 1024;
			if (relay_ok && family == 2 && duo_for_twin(ki.id) < 0 && quartet_for_twin(ki.id) < 0 &&
				(slice_count > 0 ? slice_count : g.tile_count) <= kRelayMaxTiles) {
				return launch_relay();
			}
			MixArgs a;
			fill_common(a, g, frames, src, dst, layout, frames_total, frame0);
			a.with_dry = 1;
			for (int s = 0; s < kMaxSlots; ++s) {
				if (kinds[s] != kKindNull) {
					fill_slot(a, g, s, s, first_block);
				}
			}
			++launches;
			sanitize_gains(a);
			const bool whole_tiles = g.identity || g.full_tiles;
			int id = ki.id;
			// Few tiles: block-parallel in time (span.cuh) for the single reverb slot and for the 4-slot chain, whenever no
			// update is pending and the delays allow a span (the device verifies the stream state and falls back).
			// A CTA fills an SM, so beyond one wave of the 148 SMs the kernel pays whole extra waves; few enough tiles are
			// shared among 2 or 4 CTAs each (16 / 8 streams per CTA).
			constexpr int kSpanMaxTiles = 296;
			const bool span_chain = ki.id == kChainStereo;
			if ((ki.id == kReverbMono || ki.id == kReverbStereo || span_chain) && whole_tiles && be->has_relay() && (family == 2 || family == 6) &&
				a.update_mask == 0 && a.tile_count <= kSpanMaxTiles && slice_count == 0 && frames_since_update >= 128) {
				const int share = family_span_bulk == 2 ? 0 : a.tile_count * 4 <= 148 ? 2 : a.tile_count * 2 <= 148 ? 1 : 0;
				// whole tiles per CTA: the ring traffic as bulk copies (span_bulk_kernel) if its timing is legal for this preset
				if (share == 0 && family_span_bulk) {
					const int tb = span::plan_bulk_frames(a, span_chain);
					if (tb > 0) {
						a.span_frames = tb;
						return mix_launch(span_chain ? kSpanBulkChainStereo : ki.id == kReverbMono ? kSpanBulkReverbMono : kSpanBulkReverbStereo, a, stream);
					}
				}
				const int t = span::plan_frames(a, span_chain, kLanes >> share);
				if (t > 0) {
					a.span_frames = t;
					return mix_launch((span_chain ? kSpanChainStereo : ki.id == kReverbMono ? kSpanReverbMono : kSpanReverbStereo) + share, a, stream);
				}
			}
			// Few tiles cannot fill the GPU with two warps each: below ~one tile per SM the four-stage pipeline
			// (twice the warps per tile) wins -- measured on B200, 4-slot stereo chain, ms per 1024-frame block:
			// 128 tiles 0.47 (quartet) vs 0.63 (duo); 256 tiles 0.64 vs 0.64; 2048 tiles 3.6 vs 3.07.
			constexpr int kPipelineMaxTiles = 160;
			// (Not for the tile slices of the host-buffer path: there the copies bound the step, and the duo
			// kernel measured 12.4 ms per step against 13.4 ms with quartet slices.)
			const bool few_tiles = a.tile_count <= kPipelineMaxTiles && slice_count == 0;
			if (whole_tiles && (family == 3 || (family == 2 && few_tiles)) && quartet_for_twin(ki.id) >= 0) {
				id = quartet_for_twin(ki.id);
			} else if (whole_tiles && family >= 2 && duo_for_twin(ki.id) >= 0) {
				id = duo_for_twin(ki.id);

			} else if (whole_tiles && family >= 2 && quartet_for_twin(ki.id) >= 0) {
				id = quartet_for_twin(ki.id); // no duo entry for this signature (single reverb slot)
			}
			return mix_launch(id, a, stream);
		}
		if (relay_ok) {
			return launch_relay();
		}
		// Chain of single-effect passes: the dry pass carries the first non-null slot.
		static const int gen_for_kind[] = {kGenDry, kGenModDelay, kGenCompressor, kGenDedicated, kGenDistortion,
			kGenEcho, kGenEqualizer, kGenRingMod, kGenReverb};
		bool first = true;
		for (int s = 0; s < kMaxSlots; ++s) {
			if (kinds[s] == kKindNull) {
				continue;
			}
			MixArgs a;
			fill_common(a, g, frames, src, dst, layout, frames_total, frame0);
			a.with_dry = first ? 1 : 0;
			a.accumulate = first ? 0 : 1;
			fill_slot(a, g, 0, s, first_block);
			++launches;
			if (!mix_launch(gen_for_kind[kinds[s]], a, stream)) {
				return false;
			}
			first = false;
		}
		if (first) { // no effect at all: dry only
			MixArgs a;
			fill_common(a, g, frames, src, dst, layout, frames_total, frame0);
			a.with_dry = 1;
			++launches;
			return mix_launch(kGenDry, a, stream);
		}
		return true;
	}
};

// =================================================================================================
extern "C" {

int oalsfx_engine_create(const oalsfx_engine_desc* desc, oalsfx_engine** out)
{
	if (!desc || !out) {
		g_create_error = "Null argument.";
		return OALSFX_ERR_ARGUMENT;
	}
	*out = nullptr;
	DeviceLayout dev;
	// Same checks, same order and same messages as Api::Impl::initialize (oalsfxpp.cpp:2853-2875).
	if (!make_device_layout(desc->channel_format, dev)) {
		g_create_error = "Invalid channel format.";
		return OALSFX_ERR_FORMAT;
	}
	if (desc->sampling_rate < 8000) {
		g_create_error = "Sampling rate is out of range.";
		return OALSFX_ERR_RATE;
	}
	if (desc->effect_count <= 0 || desc->effect_count > kMaxSlots) {
		g_create_error = "Effect count is out of range.";
		return OALSFX_ERR_EFFECTS;
	}
	if (desc->num_streams < 1) {
		g_create_error = "Stream count is out of range.";
		return OALSFX_ERR_ARGUMENT;
	}
	oalsfx_engine* e = new (std::nothrow) oalsfx_engine;
	if (!e) {
		g_create_error = "Failed to allocate the engine.";
		return OALSFX_ERR_MEMORY;
	}
	e->desc = *desc;
	e->dev = dev;
	e->streams = desc->num_streams;
	e->tiles = (desc->num_streams + kLanes - 1) / kLanes;
	e->arena_tiles = e->tiles;
	e->channels = dev.channels;
	e->slots = desc->effect_count;
	if (const char* fam = std::getenv("OALSFX_KERNEL")) {
		e->family = (std::strcmp(fam, "single") == 0 ? 0 : std::strcmp(fam, "quartet") == 0 ? 3 : std::strcmp(fam, "duo") == 0 ? 4 : std::strcmp(fam, "relay") == 0 ? 5 : std::strcmp(fam, "span") == 0 ? 6 : 2);
	}
	if (const char* sc = std::getenv("OALSFX_SCAN")) {
		e->scan_enabled = std::atoi(sc) != 0;
	}
	if (const char* ph = std::getenv("OALSFX_PIN_HOST")) {
		e->auto_pin_host = std::atoi(ph) != 0;
	}
	if (const char* sb = std::getenv("OALSFX_SPAN_BULK")) {
		e->family_span_bulk = std::atoi(sb);
	}
	e->be = make_backend(desc->device, g_create_error);
	if (!e->be) {
		delete e;
		return OALSFX_ERR_DEVICE;
	}
	const size_t slot_bytes = static_cast<size_t>(e->tiles) * kSlotStateWords * kLanes * sizeof(uint32_t);
	for (int s = 0; s < e->slots; ++s) {
		e->slot_state[s] = static_cast<uint32_t*>(e->dev_alloc(slot_bytes));
		if (!e->slot_state[s]) {
			g_create_error = "Device allocation failed: " + e->be->error();
			delete e;
			return OALSFX_ERR_MEMORY;
		}
	}
	e->send_state = static_cast<uint32_t*>(
		e->dev_alloc(static_cast<size_t>(e->tiles) * kSendStateWords * kLanes * sizeof(uint32_t)));
	if (!e->send_state) {
		g_create_error = "Device allocation failed: " + e->be->error();
		delete e;
		return OALSFX_ERR_MEMORY;
	}
	// Every slot starts as the null effect, every send at its defaults (oalsfxpp.cpp:2877-2902).
	oalsfxpp::EffectProps none;
	std::memset(&none, 0, sizeof(none));
	e->class_for(kFxNull, none);
	for (int s = 0; s < kMaxSlots; ++s) {
		e->fx_class[s].assign(static_cast<size_t>(e->streams), 0);
	}
	SendSettings unit = {1.0F, 1.0F, 1.0F};
	SendSettings aux[kMaxSlots] = {unit, unit, unit, unit};
	e->send_class.assign(static_cast<size_t>(e->streams), e->send_class_for(unit, aux));
	e->pending.assign(static_cast<size_t>(e->streams), 0);
	e->active.assign(static_cast<size_t>(e->streams), 1);
	// every stream routed to bus 0 at gain 1, buses in the engine's format
	e->route_bus.assign(static_cast<size_t>(e->streams) * OALSFX_MAX_ROUTES, OALSFX_BUS_NONE);
	e->route_gain.assign(e->route_bus.size(), bus::RouteGain{1.0F, 1.0F, 0, 0, 0});
	e->route_pan.assign(e->route_bus.size(), std::vector<float>());
	e->bus_channels = e->channels;
	e->route_entry.assign(e->route_bus.size(), -1);
	for (int s = 0; s < e->streams; ++s) {
		e->route_bus[static_cast<size_t>(s) * OALSFX_MAX_ROUTES] = 0;
	}
	*out = e;
	return OALSFX_OK;
}

void oalsfx_engine_destroy(oalsfx_engine* e) { delete e; }

int oalsfx_engine_set_effect(oalsfx_engine* e, int first_stream, int n_streams, int slot,
	int effect_type, const void* props, size_t props_bytes)
{
	if (!e) {
		return OALSFX_ERR_ARGUMENT;
	}
	if (first_stream < 0 || n_streams < 1 || first_stream + n_streams > e->streams) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Stream range is out of range.");
	}
	if (slot < 0 || slot >= e->slots) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Effect index is out of range.");
	}
	if (effect_type < 0 || effect_type >= kFxTypeCount) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Unknown effect type.");
	}
	oalsfxpp::EffectProps p;
	std::memset(&p, 0, sizeof(p));
	if (effect_type != kFxNull) {
		if (!props || props_bytes != sizeof(oalsfxpp::EffectProps)) {
			return e->fail(OALSFX_ERR_ARGUMENT, "props must be the bytes of an oalsfxpp::EffectProps.");
		}
		std::memcpy(&p, props, sizeof(p));
	}
	const int id = e->class_for(effect_type, p);
	if (id < 0) {
		return e->fail(OALSFX_ERR_MEMORY, "Lookup table upload failed: " + e->be->error());
	}
	if (ring_words_for(effect_type, e->desc.sampling_rate) > e->ring_cap[slot]) {
		e->quiesce();  // the arena is about to be copied and freed: no mix may still be running on the caller's stream
	}
	if (!e->ensure_ring(slot, ring_words_for(effect_type, e->desc.sampling_rate))) {
		return e->fail(OALSFX_ERR_MEMORY, "Delay-line arena allocation failed: " + e->be->error());
	}
	// A type change constructs a fresh effect state (oalsfxpp.cpp:2692-2698): zero the slot state and
	// the rings of exactly those streams.
	// (the streams' lanes: placed streams sit in any order, so the tiles are collected by index)
	std::map<uint32_t, uint32_t> reset_masks;
	for (int s = first_stream; s < first_stream + n_streams; ++s) {
		const int lane = e->lane_of(s);
		int& cur = e->fx_class[slot][static_cast<size_t>(lane)];
		if (e->classes[static_cast<size_t>(cur)].type != effect_type) {
			reset_masks[static_cast<uint32_t>(lane / kLanes)] |= 1U << (lane % kLanes);
		}
		cur = id;
		e->pending[static_cast<size_t>(lane)] |= static_cast<uint8_t>(1U << slot); // is_props_changed_ (oalsfxpp.cpp:2707)
	}
	std::vector<TileRef> reset;
	for (const auto& tm : reset_masks) {
		reset.push_back(TileRef{tm.first, tm.second});
	}
	if (!reset.empty()) {
		const int n = static_cast<int>(reset.size());
		e->quiesce();  // zeroing state a running mix may still be using
		if (!e->be->zero_lanes(e->slot_state[slot], static_cast<long long>(kSlotStateWords) * kLanes, kSlotStateWords,
				reset.data(), n, nullptr)) {
			return e->fail(OALSFX_ERR_DEVICE, e->be->error());
		}
		if (e->ring_cap[slot] > 0 && !e->be->zero_lanes(reinterpret_cast<uint32_t*>(e->ring[slot]),
				static_cast<long long>(e->ring_cap[slot]) * kLanes, e->ring_cap[slot], reset.data(), n, nullptr)) {
			return e->fail(OALSFX_ERR_DEVICE, e->be->error());
		}
	}
	e->groups_dirty = true;
	return OALSFX_OK;
}

int oalsfx_engine_set_sends(oalsfx_engine* e, int first_stream, int n_streams, const float* direct, const float* aux)
{
	if (!e) {
		return OALSFX_ERR_ARGUMENT;
	}
	if (first_stream < 0 || n_streams < 1 || first_stream + n_streams > e->streams || !direct || !aux) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Bad stream range or null send properties.");
	}
	SendSettings d = {direct[0], direct[1], direct[2]};
	SendSettings a[kMaxSlots];
	std::memset(a, 0, sizeof(a));
	for (int i = 0; i < e->slots; ++i) {
		a[i] = SendSettings{aux[3 * i], aux[3 * i + 1], aux[3 * i + 2]};
	}
	const int id = e->send_class_for(d, a);
	for (int s = first_stream; s < first_stream + n_streams; ++s) {
		e->send_class[static_cast<size_t>(e->lane_of(s))] = id;
	}
	e->groups_dirty = true;
	return OALSFX_OK;
}

int oalsfx_engine_set_active(oalsfx_engine* e, int first_stream, int n_streams, int active)
{
	if (!e) {
		return OALSFX_ERR_ARGUMENT;
	}
	if (first_stream < 0 || n_streams < 1 || first_stream + n_streams > e->streams) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Stream range is out of range.");
	}
	e->quiesce();
	const uint8_t flag = active ? 1 : 0;
	for (int s = first_stream; s < first_stream + n_streams; ++s) {
		uint8_t& cur = e->active[static_cast<size_t>(e->lane_of(s))];
		if (cur != flag) {
			cur = flag;
			e->groups_dirty = true;   // (an engine whose flags do not change keeps its groups)
			e->bus_plan_dirty = true;
		}
	}
	return OALSFX_OK;
}

int oalsfx_engine_reset_streams(oalsfx_engine* e, int first_stream, int n_streams)
{
	if (!e) {
		return OALSFX_ERR_ARGUMENT;
	}
	if (first_stream < 0 || n_streams < 1 || first_stream + n_streams > e->streams) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Stream range is out of range.");
	}
	if (!e->quiesce()) {  // zeroing state a running mix may still be using
		return e->fail(OALSFX_ERR_DEVICE, e->be->error());
	}
	// The streams' lanes, by tile (placed streams sit in any order).  Every slot of them is marked pending as the
	// set_effect call that configured it did, so the next block that mixes them runs `update` on fresh state: a slot
	// holding an effect, that is -- the null effect has no update and no state.
	std::map<uint32_t, uint32_t> masks;
	for (int s = first_stream; s < first_stream + n_streams; ++s) {
		const int lane = e->lane_of(s);
		masks[static_cast<uint32_t>(lane / kLanes)] |= 1U << (lane % kLanes);
		for (int slot = 0; slot < e->slots; ++slot) {
			if (e->classes[static_cast<size_t>(e->fx_class[slot][static_cast<size_t>(lane)])].type != kFxNull) {
				e->pending[static_cast<size_t>(lane)] |= static_cast<uint8_t>(1U << slot);
			}
		}
	}
	std::vector<TileRef> reset;
	for (const auto& tm : masks) {
		reset.push_back(TileRef{tm.first, tm.second});
	}
	const int n = static_cast<int>(reset.size());
	bool ok = true;
	for (int slot = 0; slot < e->slots && ok; ++slot) {
		ok = e->be->zero_lanes(e->slot_state[slot], static_cast<long long>(kSlotStateWords) * kLanes, kSlotStateWords, reset.data(), n, nullptr);
		if (ok && e->ring_cap[slot] > 0) {
			ok = e->be->zero_lanes(reinterpret_cast<uint32_t*>(e->ring[slot]), static_cast<long long>(e->ring_cap[slot]) * kLanes,
				e->ring_cap[slot], reset.data(), n, nullptr);
		}
	}
	ok = ok && e->be->zero_lanes(e->send_state, static_cast<long long>(kSendStateWords) * kLanes, kSendStateWords, reset.data(), n, nullptr);
	if (!ok) {
		return e->fail(OALSFX_ERR_DEVICE, e->be->error());
	}
	e->groups_dirty = true;
	return OALSFX_OK;
}

// A pan route's matrices (set_routes_impl): target m1 = `target` (a Cb x C matrix), or gain g1 on the index diagonal when
// `target` is null; start m0 = m1 without a ramp, else the old route's coefficients at t0 - 1 (`old_pan`, or a scalar route's
// gain on the diagonal, `old`), or 0 for a new route.
static void pan_route_start(std::vector<float>& out, const float* target, float g1, int C, int Cb, int ramp_frames,
	const std::vector<float>* old_pan, const bus::RouteGain* old, long long t0)
{
	const int cm = Cb * C;
	out.assign(static_cast<size_t>(2 * cm), 0.0F);
	float* m0 = out.data();
	float* m1 = m0 + cm;
	if (target) {
		std::copy_n(target, cm, m1);
	} else {
		for (int j = 0; j < std::min(C, Cb); ++j) {
			m1[j * C + j] = g1;
		}
	}
	if (ramp_frames == 0) {
		std::copy_n(m1, cm, m0);
	} else if (old_pan) {
		const float pos = bus::ramp_pos(old->rf, old->t0, t0 - 1);
		for (int q = 0; q < cm; ++q) {
			m0[q] = bus::ramp_apply((*old_pan)[static_cast<size_t>(q)], (*old_pan)[static_cast<size_t>(cm + q)], pos);
		}
	} else if (old) {
		const float g = bus::route_gain(*old, t0 - 1);
		for (int j = 0; j < std::min(C, Cb); ++j) {
			m0[j * C + j] = g;
		}
	}
}

extern "C++" {
template <bool kPans>
static int replace_routes(oalsfx_engine* e, int first_stream, int n_streams, int R, const int32_t* bus, const float* gain,
	const float* pan, int ramp_frames);
}

// oalsfx_engine_set_routes (gain: per route, or NULL: 1.0f) and oalsfx_engine_set_route_pans (pan: per route a Cb x C
// matrix): one body, so that both check, replace and ramp routes alike.  A route becomes a pan route through set_route_pans,
// and stays one under set_routes with a ramp, which then ramps it to its gain on the index diagonal.
static int set_routes_impl(oalsfx_engine* e, int first_stream, int n_streams, int routes_per_stream, const int32_t* bus,
	const float* gain, const float* pan, int ramp_frames)
{
	const int R = routes_per_stream;
	const int C = e->channels, Cb = e->bus_channels, cm = Cb * C;
	if (first_stream < 0 || n_streams < 1 || first_stream + n_streams > e->streams || !bus) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Bad stream range or null bus list.");
	}
	if (R < 1 || R > OALSFX_MAX_ROUTES) {
		return e->fail(OALSFX_ERR_ARGUMENT, "routes_per_stream must be 1..OALSFX_MAX_ROUTES.");
	}
	if (ramp_frames < 0 || ramp_frames > (1 << 24)) {
		return e->fail(OALSFX_ERR_ARGUMENT, "ramp_frames must be 0..2^24.");
	}
	for (int i = 0; i < n_streams; ++i) {
		for (int r = 0; r < R; ++r) {
			const int32_t b = bus[i * R + r];
			if (b < OALSFX_BUS_NONE) {
				return e->fail(OALSFX_ERR_ARGUMENT, "Bus index below OALSFX_BUS_NONE.");
			}
			for (int q = 0; q < r && b != OALSFX_BUS_NONE; ++q) {
				if (bus[i * R + q] == b) {
					return e->fail(OALSFX_ERR_ARGUMENT, "A stream names the same bus twice.");
				}
			}
			if (gain && b != OALSFX_BUS_NONE && !std::isfinite(gain[i * R + r])) {
				return e->fail(OALSFX_ERR_ARGUMENT, "Route gains must be finite.");
			}
			const float* m = pan ? pan + static_cast<size_t>(i * R + r) * static_cast<size_t>(cm) : nullptr;
			if (m && b != OALSFX_BUS_NONE && !std::all_of(m, m + cm, [](float v) { return std::isfinite(v); })) {
				return e->fail(OALSFX_ERR_ARGUMENT, "Pan coefficients must be finite.");
			}
		}
	}
	e->quiesce();
	// without a pan route before or after the call, the loop leaves the matrices alone: set_routes keeps its cost
	return pan || e->pan_routes > 0 ? replace_routes<true>(e, first_stream, n_streams, R, bus, gain, pan, ramp_frames) :
		replace_routes<false>(e, first_stream, n_streams, R, bus, gain, nullptr, ramp_frames);
}

extern "C++" {
// The routes of streams [first_stream, first_stream + n_streams) after set_routes_impl's checks.  kPans: some route has a
// matrix, before or after the call.
template <bool kPans>
static int replace_routes(oalsfx_engine* e, int first_stream, int n_streams, int R, const int32_t* bus, const float* gain,
	const float* pan, int ramp_frames)
{
	const int C = e->channels, Cb = e->bus_channels, cm = Cb * C;
	const long long t0 = e->clock_total;
	const size_t stride = static_cast<size_t>(2 * cm);
	constexpr bool pans = kPans;
	auto put_pan = [e](size_t slot, std::vector<float>& m) {   // slot's matrices become m's (m gets the old ones)
		e->pan_routes += static_cast<long long>(!m.empty()) - static_cast<long long>(!e->route_pan[slot].empty());
		e->route_pan[slot].swap(m);
	};
	bool pairs_changed = false;
	std::vector<float> new_pan[OALSFX_MAX_ROUTES];   // (reused from stream to stream: swapped with the routes' matrices)
	for (int i = 0; i < n_streams; ++i) {
		const size_t base = static_cast<size_t>(first_stream + i) * OALSFX_MAX_ROUTES;
		int32_t* cur = e->route_bus.data() + base;
		bus::RouteGain* cur_gain = e->route_gain.data() + base;
		int32_t new_bus[OALSFX_MAX_ROUTES];
		bus::RouteGain new_gain[OALSFX_MAX_ROUTES];
		int old_slot[OALSFX_MAX_ROUTES];
		int n = 0;
		bool same = true;   // the same (stream, bus) pairs: every route keeps its slot and member entry, only its gains change
		for (int r = 0; r < R; ++r) {
			const int32_t b = bus[i * R + r];
			if (b == OALSFX_BUS_NONE) {
				continue;
			}
			int k = 0;
			while (k < OALSFX_MAX_ROUTES && cur[k] != b) {
				++k;
			}
			const bool had = k < OALSFX_MAX_ROUTES;
			const std::vector<float>* old_pan = pans && had && !e->route_pan[base + static_cast<size_t>(k)].empty() ?
				&e->route_pan[base + static_cast<size_t>(k)] : nullptr;
			// the start gain: the route's gain at the last mixed frame, or 0 for a new route; without a ramp the new gain holds
			// at once, also for a block mixed before the call
			const float g1 = gain ? gain[i * R + r] : 1.0F;
			if (!pans || (!pan && !(old_pan && ramp_frames > 0))) {
				if (pans) {
					new_pan[n].clear();
				}
				const float g0 = ramp_frames == 0 ? g1 : had ? bus::route_gain(cur_gain[k], t0 - 1) : 0.0F;
				new_gain[n] = bus::RouteGain{g0, g1, ramp_frames, 0, t0};
			} else {
				pan_route_start(new_pan[n], pan ? pan + static_cast<size_t>(i * R + r) * static_cast<size_t>(cm) : nullptr, g1, C, Cb,
					ramp_frames, old_pan, had ? &cur_gain[k] : nullptr, t0);
				new_gain[n] = bus::RouteGain{0.0F, 0.0F, ramp_frames, 1, t0};
			}
			same = same && had;
			old_slot[n] = k;
			new_bus[n] = b;
			++n;
		}
		same = same && (n == OALSFX_MAX_ROUTES || cur[n] == OALSFX_BUS_NONE);   // (used slots come first)
		for (int r = 0; r < n && same; ++r) {
			const size_t k = base + static_cast<size_t>(old_slot[r]);
			e->route_gain[k] = new_gain[r];
			if (pans) {
				put_pan(k, new_pan[r]);
			}
			const int entry = e->route_entry[k];
			if (entry < 0) {
				continue;
			}
			e->gain_host[entry] = new_gain[r];
			e->gains_dirty = true;
			if (pans && !e->route_pan[k].empty()) {
				if (static_cast<size_t>(e->bus_entries) * stride > e->pan_host_cap) {
					e->bus_plan_dirty = true;   // the plan's first pan route: the rebuild sizes the pan image for every entry
				} else {
					std::copy(e->route_pan[k].begin(), e->route_pan[k].end(), e->pan_host + static_cast<size_t>(entry) * stride);
				}
			}
		}
		if (!same) {
			for (int k = 0; k < OALSFX_MAX_ROUTES; ++k) {
				cur[k] = k < n ? new_bus[k] : OALSFX_BUS_NONE;
				cur_gain[k] = k < n ? new_gain[k] : bus::RouteGain{};
				if (pans) {
					if (k >= n) {
						new_pan[k].clear();   // (the slot has no route)
					}
					put_pan(base + static_cast<size_t>(k), new_pan[k]);
				}
			}
			pairs_changed = true;
		}
	}
	if (pairs_changed) {
		e->max_bus = *std::max_element(e->route_bus.begin(), e->route_bus.end());
		e->bus_plan_dirty = true;
	}
	return OALSFX_OK;
}
}

int oalsfx_engine_set_routes(oalsfx_engine* e, int first_stream, int n_streams, int routes_per_stream, const int32_t* bus,
	const float* gain, int ramp_frames)
{
	if (!e) {
		return OALSFX_ERR_ARGUMENT;
	}
	return set_routes_impl(e, first_stream, n_streams, routes_per_stream, bus, gain, nullptr, ramp_frames);
}

int oalsfx_engine_set_route_pans(oalsfx_engine* e, int first_stream, int n_streams, int routes_per_stream, const int32_t* bus,
	const float* pan, int ramp_frames)
{
	if (!e) {
		return OALSFX_ERR_ARGUMENT;
	}
	if (!pan) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Null pan matrices.");
	}
	return set_routes_impl(e, first_stream, n_streams, routes_per_stream, bus, nullptr, pan, ramp_frames);
}

int oalsfx_engine_set_bus_format(oalsfx_engine* e, int channel_format)
{
	if (!e) {
		return OALSFX_ERR_ARGUMENT;
	}
	DeviceLayout d;
	if (!make_device_layout(channel_format, d)) {
		return e->fail(OALSFX_ERR_FORMAT, "Invalid channel format.");
	}
	if (d.channels != e->bus_channels && e->pan_routes > 0) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Pan routes are sized for the current bus channel count.");
	}
	e->quiesce();
	if (d.channels != e->bus_channels) {
		e->bus_channels = d.channels;
		e->gains_dirty = true;   // the plan may change kernels: the gain image decides again whether it is needed
	}
	return OALSFX_OK;
}

int oalsfx_engine_route_streams(oalsfx_engine* e, int first_stream, int n_streams, const int32_t* bus)
{
	return oalsfx_engine_set_routes(e, first_stream, n_streams, 1, bus, nullptr, 0);
}

static int mix_blocks(oalsfx_engine* e, int frames, const float* src, float* dst, int layout, int space, void* cuda_stream)
{
	if (!e) {
		return OALSFX_ERR_ARGUMENT;
	}
	if (frames == 0) {
		return OALSFX_OK; // reference: oalsfxpp.cpp:3796-3799
	}
	if (frames < 0) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Negative frame count.");
	}
	if (!src) {
		return e->fail(OALSFX_ERR_ARGUMENT, "No source samples.");
	}
	if (!dst) {
		return e->fail(OALSFX_ERR_ARGUMENT, "No destination samples.");
	}
	if (layout != OALSFX_LAYOUT_STREAM_MAJOR && layout != OALSFX_LAYOUT_TILED) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Unknown layout.");
	}
	const long long padded = (layout == OALSFX_LAYOUT_TILED ? static_cast<long long>(e->tiles) * kLanes : e->streams);
	const size_t count = static_cast<size_t>(padded) * static_cast<size_t>(frames) * static_cast<size_t>(e->channels);
	const float* dsrc = src;
	float* ddst = dst;
	e->note_stream(cuda_stream);
	if (space == OALSFX_SPACE_HOST && e->auto_pin_host) {
		// pageable buffers copy at a fraction of the pinned rate and do not overlap with the kernels: lock them in place
		// (a failure only means the copies stay slow)
		e->pin_host(const_cast<float*>(src), count * sizeof(float), true);
		e->pin_host(dst, count * sizeof(float), true);
	}
	if (space == OALSFX_SPACE_HOST) {
		if (count > e->stage_cap) {
			e->be->sync(cuda_stream);
			e->be->release(e->stage_in);
			e->be->release(e->stage_out);
			e->device_bytes -= static_cast<long long>(e->stage_cap) * 2 * sizeof(float);
			e->stage_in = static_cast<float*>(e->dev_alloc(count * sizeof(float)));
			e->stage_out = static_cast<float*>(e->dev_alloc(count * sizeof(float)));
			e->stage_cap = count;
			if (!e->stage_in || !e->stage_out) {
				e->stage_cap = 0;
				return e->fail(OALSFX_ERR_MEMORY, "Staging allocation failed: " + e->be->error());
			}
		}
		dsrc = e->stage_in;
		ddst = e->stage_out;
		// One block, one group covering every tile (the common case): slice the tiles and overlap the
		// upload of slice j+1, the kernel of slice j and the download of slice j-1 (PCIe is full duplex
		// and the copies, not the kernel, bound this path).
		if (e->groups_dirty && !e->rebuild_groups()) {
			return e->fail(OALSFX_ERR_DEVICE, "Group table upload failed: " + e->be->error());
		}
		int max_slices = 16;
		if (const char* tune = std::getenv("OALSFX_TUNE_SLICES")) { // experiments only
			max_slices = std::max(2, std::atoi(tune));
		}
		const int slices = std::min(e->tiles / 64, max_slices);
		if (frames <= kMaxBlockFrames && e->groups.size() == 1 && e->groups[0].identity && (!e->groups[0].multi || frames >= 2) && slices >= 2 &&
			layout == OALSFX_LAYOUT_STREAM_MAJOR) {
			if (!e->pipe_in) {
				e->pipe_in = e->be->stream_create();
				e->pipe_run = e->be->stream_create();
				e->pipe_out = e->be->stream_create();
			}
			if (e->pipe_in && e->pipe_run && e->pipe_out) {
				if (!e->be->sync(cuda_stream)) {
					return e->fail(OALSFX_ERR_DEVICE, e->be->error());
				}
				const Group g = e->groups[0];
				const size_t per_tile = static_cast<size_t>(kLanes) * static_cast<size_t>(frames) * static_cast<size_t>(e->channels);
				bool ok = true;
				for (int j = 0; j < slices && ok; ++j) {
					const int t0 = static_cast<int>(static_cast<long long>(e->tiles) * j / slices);
					const int t1 = static_cast<int>(static_cast<long long>(e->tiles) * (j + 1) / slices);
					const size_t first = per_tile * static_cast<size_t>(t0);
					const size_t last = std::min(per_tile * static_cast<size_t>(t1), count);
					ok = e->be->upload(e->stage_in + first, src + first, (last - first) * sizeof(float), e->pipe_in) &&
						e->be->stream_wait(e->pipe_run, e->pipe_in);
					e->slice_first = t0;
					e->slice_count = t1 - t0;
					ok = ok && e->launch_group(g, frames, dsrc, ddst, layout, frames, 0, true, e->pipe_run);
					e->slice_first = e->slice_count = 0;
					ok = ok && e->be->stream_wait(e->pipe_out, e->pipe_run) &&
						e->be->download(dst + first, e->stage_out + first, (last - first) * sizeof(float), e->pipe_out);
				}
				ok = ok && e->be->sync(e->pipe_out) && e->be->sync(e->pipe_run);
				if (!ok) {
					return e->fail(OALSFX_ERR_DEVICE, e->be->error());
				}
				if (g.key.pending != 0) {
					e->clear_mixed_pending();
					e->groups_dirty = true;
					e->frames_since_update = 0;
				}
				e->frames_since_update += frames;
				return OALSFX_OK;
			}
		}
		if (!e->be->upload(e->stage_in, src, count * sizeof(float), cuda_stream)) {
			return e->fail(OALSFX_ERR_DEVICE, e->be->error());
		}
	} else if (space != OALSFX_SPACE_DEVICE) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Unknown pointer space.");
	}

	// caller strides of the buffers (a placed engine permutes each block into lane order and back)
	const long long io_ts = static_cast<long long>(frames) * e->channels * kLanes;
	const long long io_ls = layout == OALSFX_LAYOUT_TILED ? 1 : static_cast<long long>(frames) * e->channels;
	const long long io_fs = layout == OALSFX_LAYOUT_TILED ? static_cast<long long>(e->channels) * kLanes : e->channels;
	const long long io_cs = layout == OALSFX_LAYOUT_TILED ? kLanes : 1;
	bool first_block = true;
	for (int done = 0; done < frames;) {
		const int todo = std::min(frames - done, kMaxBlockFrames); // oalsfxpp.cpp:3818-3826
		if (e->groups_dirty && !e->rebuild_groups()) {
			if (e->place_oom) {
				return e->fail(OALSFX_ERR_MEMORY, "Placement could not grow the arenas: " + e->be->error());
			}
			return e->fail(OALSFX_ERR_DEVICE, "Group table upload failed: " + e->be->error());
		}
		const float* bsrc = dsrc;
		float* bdst = ddst;
		int blayout = layout;
		long long btotal = frames, bframe0 = done;
		if (e->placed) {
			const size_t need = static_cast<size_t>(e->arena_tiles) * kLanes * static_cast<size_t>(std::min(frames, kMaxBlockFrames)) *
				static_cast<size_t>(e->channels);
			if (need > e->io_cap) {
				e->be->sync(cuda_stream);
				e->be->release(e->io_in);
				e->be->release(e->io_out);
				e->device_bytes -= static_cast<long long>(e->io_cap) * 2 * sizeof(float);
				e->io_in = static_cast<float*>(e->dev_alloc(need * sizeof(float)));
				e->io_out = static_cast<float*>(e->dev_alloc(need * sizeof(float)));
				e->io_cap = need;
				if (!e->io_in || !e->io_out) {
					e->io_cap = 0;
					return e->fail(OALSFX_ERR_MEMORY, "Placement block allocation failed: " + e->be->error());
				}
			}
			if (!e->be->gather_io(dsrc + done * io_fs, io_ts, io_ls, io_fs, io_cs, e->stream_of_lane_dev, e->arena_tiles, todo,
					e->channels, e->io_in, cuda_stream)) {
				return e->fail(OALSFX_ERR_DEVICE, e->be->error());
			}
			bsrc = e->io_in;
			bdst = e->io_out;
			blayout = OALSFX_LAYOUT_TILED;
			btotal = todo;
			bframe0 = 0;
		}
		bool had_pending = false;
		const bool use_fallback = !e->fallback_groups.empty() && todo < 2; // (only class-per-tile launches have fallback groups)
		had_pending = use_fallback && e->groups[0].key.pending != 0;
		for (const Group& g : (use_fallback ? e->fallback_groups : e->groups)) {
			had_pending = had_pending || g.key.pending != 0;
			if (!e->launch_group(g, todo, bsrc, bdst, blayout, btotal, bframe0, first_block, cuda_stream)) {
				return e->fail(OALSFX_ERR_DEVICE, e->be->error());
			}
		}
		if (e->placed && !e->be->scatter_io(e->io_out, e->stream_of_lane_dev, e->arena_tiles, todo, e->channels, ddst + done * io_fs,
				io_ts, io_ls, io_fs, io_cs, cuda_stream)) {
			return e->fail(OALSFX_ERR_DEVICE, e->be->error());
		}
		if (!e->placed && e->paused_rows > 0 && !e->be->zero_rows(ddst + done * io_fs, io_ts, io_ls, io_fs, io_cs, e->paused_rows_dev,
				e->paused_rows, todo, e->channels, cuda_stream)) {
			return e->fail(OALSFX_ERR_DEVICE, e->be->error());
		}
		if (had_pending) {
			e->clear_mixed_pending();
			e->groups_dirty = true;
			e->frames_since_update = 0;
		}
		e->frames_since_update += todo;
		first_block = false;
		done += todo;
	}

	if (space == OALSFX_SPACE_HOST) {
		if (!e->be->download(dst, e->stage_out, count * sizeof(float), cuda_stream) || !e->be->sync(cuda_stream)) {
			return e->fail(OALSFX_ERR_DEVICE, e->be->error());
		}
	}
	return OALSFX_OK;
}

// Every mix entry point (mix, mix_bus, mix_buses) comes through here: a successful call of `frames` frames advances the
// frame clock; a refused or failed one leaves it.
int oalsfx_engine_mix(oalsfx_engine* e, int frames, const float* src, float* dst, int layout, int space, void* cuda_stream)
{
	const int rc = mix_blocks(e, frames, src, dst, layout, space, cuda_stream);
	if (rc == OALSFX_OK && frames > 0) {
		e->clock_mix = e->clock_total;
		e->clock_total += frames;
	}
	return rc;
}

int oalsfx_engine_pin_host(oalsfx_engine* e, void* buffer, size_t bytes)
{
	if (!e || !buffer || bytes == 0) {
		return e ? e->fail(OALSFX_ERR_ARGUMENT, "Bad pin_host arguments.") : OALSFX_ERR_ARGUMENT;
	}
	return e->pin_host(buffer, bytes, false) ? OALSFX_OK : e->fail(OALSFX_ERR_DEVICE, "Page-locking the buffer failed: " + e->be->error());
}

int oalsfx_engine_unpin_host(oalsfx_engine* e, void* buffer)
{
	if (!e || !buffer) {
		return e ? e->fail(OALSFX_ERR_ARGUMENT, "Bad unpin_host arguments.") : OALSFX_ERR_ARGUMENT;
	}
	e->quiesce();
	for (size_t i = 0; i < e->pinned_host.size(); ++i) {
		if (e->pinned_host[i].p == buffer) {
			e->be->host_unregister(buffer);
			e->pinned_host.erase(e->pinned_host.begin() + static_cast<long>(i));
			return OALSFX_OK;
		}
	}
	return e->fail(OALSFX_ERR_ARGUMENT, "The buffer is not pinned by this engine.");
}

int oalsfx_engine_mix_bus(oalsfx_engine* e, int frames, const float* src, float* dst, int layout, float* bus, void* cuda_stream)
{
	if (!e || !src || !dst || !bus || frames <= 0) {
		return e ? e->fail(OALSFX_ERR_ARGUMENT, "Bad mix_bus arguments.") : OALSFX_ERR_ARGUMENT;
	}
	// One pass over the block's output right behind the mix, on the same stream.  (Summing inside the fused kernel's
	// epilogue -- per-tile shuffle trees in its back warp, in one go, spread over the next hand-off, or in a third warp --
	// was measured at +0.21 / +0.35 / +0.57 ms per 65 536-stream block against 0.10 ms for this pass: that warp is the
	// kernel's critical path.  profiles/r02_history.md.)
	const int rc = oalsfx_engine_mix(e, frames, src, dst, layout, OALSFX_SPACE_DEVICE, cuda_stream);
	return rc != OALSFX_OK ? rc : oalsfx_engine_reduce_bus(e, frames, dst, layout, bus, cuda_stream);
}

int oalsfx_engine_reduce_bus(oalsfx_engine* e, int frames, const float* dst, int layout, float* bus, void* cuda_stream)
{
	if (!e || !dst || !bus || frames <= 0) {
		return e ? e->fail(OALSFX_ERR_ARGUMENT, "Bad reduce_bus arguments.") : OALSFX_ERR_ARGUMENT;
	}
	long long ts, ls, fs, cs;
	if (layout == OALSFX_LAYOUT_TILED) {
		ts = static_cast<long long>(frames) * e->channels * kLanes;
		ls = 1;
		fs = static_cast<long long>(e->channels) * kLanes;
		cs = kLanes;
	} else {
		ts = static_cast<long long>(frames) * e->channels * kLanes;
		ls = static_cast<long long>(frames) * e->channels;
		fs = e->channels;
		cs = 1;
	}
	e->note_stream(cuda_stream);
	++e->launches;
	if (!e->be->reduce_bus(dst, ts, ls, fs, cs, e->streams, frames, e->channels, bus, cuda_stream)) {
		return e->fail(OALSFX_ERR_DEVICE, e->be->error());
	}
	return OALSFX_OK;
}

int oalsfx_engine_reduce_buses(oalsfx_engine* e, int frames, const float* dst, int layout, int n_buses, float* buses, void* cuda_stream)
{
	if (!e) {
		return OALSFX_ERR_ARGUMENT;
	}
	if (const char* bad = e->bad_bus_args(frames, dst, layout, n_buses, buses)) {
		return e->fail(OALSFX_ERR_ARGUMENT, bad);
	}
	return e->reduce_buses(frames, dst, layout, n_buses, buses, cuda_stream);
}

int oalsfx_engine_mix_buses(oalsfx_engine* e, int frames, const float* src, float* dst, int layout, int n_buses, float* buses,
	void* cuda_stream)
{
	if (!e) {
		return OALSFX_ERR_ARGUMENT;
	}
	// everything is checked before the mix: a refused call advances no stream
	if (!src) {
		return e->fail(OALSFX_ERR_ARGUMENT, "No source samples.");
	}
	if (const char* bad = e->bad_bus_args(frames, dst, layout, n_buses, buses)) {
		return e->fail(OALSFX_ERR_ARGUMENT, bad);
	}
	const int rc = oalsfx_engine_mix(e, frames, src, dst, layout, OALSFX_SPACE_DEVICE, cuda_stream);
	return rc != OALSFX_OK ? rc : e->reduce_buses(frames, dst, layout, n_buses, buses, cuda_stream);
}

int oalsfx_pcm_to_float(oalsfx_engine* e, const void* src, int bit_depth, float* dst, long long count, void* cuda_stream)
{
	if (!e || !src || !dst || count < 0) {
		return e ? e->fail(OALSFX_ERR_ARGUMENT, "Bad pcm_to_float arguments.") : OALSFX_ERR_ARGUMENT;
	}
	if (bit_depth != 8 && bit_depth != 16) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Invalid bit depth."); // reference: oalsfxpp_test.cpp:738
	}
	e->note_stream(cuda_stream);
	++e->launches;
	if (!e->be->pcm_to_float(src, bit_depth, dst, count, cuda_stream)) {
		return e->fail(OALSFX_ERR_DEVICE, e->be->error());
	}
	return OALSFX_OK;
}

int oalsfx_debug_waveshaper(oalsfx_engine* e, const float* samples, float edge_coeff, float* out, long long count, void* cuda_stream)
{
	if (!e || !samples || !out || count < 0) {
		return e ? e->fail(OALSFX_ERR_ARGUMENT, "Bad debug_waveshaper arguments.") : OALSFX_ERR_ARGUMENT;
	}
	e->note_stream(cuda_stream);
	if (!e->be->debug_waveshaper(samples, edge_coeff, out, count, cuda_stream)) {
		return e->fail(OALSFX_ERR_DEVICE, e->be->error());
	}
	return OALSFX_OK;
}

int oalsfx_float_to_s16(oalsfx_engine* e, const float* src, int16_t* dst, int rows, long long row_len, float* row_scale,
	void* cuda_stream)
{
	if (!e || !src || !dst || rows < 0 || row_len < 0) {
		return e ? e->fail(OALSFX_ERR_ARGUMENT, "Bad float_to_s16 arguments.") : OALSFX_ERR_ARGUMENT;
	}
	e->note_stream(cuda_stream);
	++e->launches;
	if (!e->be->float_to_s16(src, dst, rows, row_len, row_scale, cuda_stream)) {
		return e->fail(OALSFX_ERR_DEVICE, e->be->error());
	}
	return OALSFX_OK;
}

// ---- state snapshot / restore (SURVEY.md 8f rank 3) --------------------------------------------------
// Everything a stream carries from one block to the next lives in three kinds of device arenas (delay-line
// rings and slot state per slot, send filter history) plus one host byte per stream (pending `update`
// bits).  A snapshot is those bytes behind a header that pins the geometry.
namespace {
struct SnapshotHeader {
	uint32_t magic, version;
	int32_t streams, tiles, channels, slots, rate, format;
	int32_t ring_cap[kMaxSlots];
	uint64_t total_bytes;
};
constexpr uint32_t kSnapshotMagic = 0x58464C4FU; // "OLFX"

void snapshot_header(const oalsfx_engine* e, SnapshotHeader& h)
{
	std::memset(&h, 0, sizeof(h));
	h.magic = kSnapshotMagic;
	h.version = 1;
	h.streams = e->streams;
	h.tiles = e->tiles;
	h.channels = e->channels;
	h.slots = e->slots;
	h.rate = e->desc.sampling_rate;
	h.format = e->desc.channel_format;
	uint64_t bytes = sizeof(SnapshotHeader) + static_cast<uint64_t>(e->streams);
	for (int s = 0; s < kMaxSlots; ++s) {
		h.ring_cap[s] = (s < e->slots ? e->ring_cap[s] : 0);
		if (s < e->slots) {
			bytes += static_cast<uint64_t>(e->tiles) * static_cast<uint64_t>(h.ring_cap[s]) * kLanes * sizeof(float);
			bytes += static_cast<uint64_t>(e->tiles) * kSlotStateWords * kLanes * sizeof(uint32_t);
		}
	}
	bytes += static_cast<uint64_t>(e->tiles) * kSendStateWords * kLanes * sizeof(uint32_t);
	h.total_bytes = bytes;
}
} // namespace

long long oalsfx_engine_snapshot_size(const oalsfx_engine* e)
{
	if (!e) {
		return 0;
	}
	SnapshotHeader h;
	snapshot_header(e, h);
	return static_cast<long long>(h.total_bytes);
}

int oalsfx_engine_snapshot(oalsfx_engine* e, void* dst, size_t bytes)
{
	if (!e || !dst) {
		return e ? e->fail(OALSFX_ERR_ARGUMENT, "Bad snapshot arguments.") : OALSFX_ERR_ARGUMENT;
	}
	SnapshotHeader h;
	snapshot_header(e, h);
	if (bytes < h.total_bytes) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Snapshot buffer too small.");
	}
	if (!e->quiesce()) {
		return e->fail(OALSFX_ERR_DEVICE, e->be->error());
	}
	char* out = static_cast<char*>(dst);
	std::memcpy(out, &h, sizeof(h));
	out += sizeof(h);
	if (e->placed) {
		for (int s = 0; s < e->streams; ++s) {
			out[s] = static_cast<char>(e->pending[static_cast<size_t>(e->lane_of(s))]);
		}
		out += e->streams;
		return e->canonical_state(out, nullptr) ? OALSFX_OK : e->fail(OALSFX_ERR_DEVICE, e->be->error());
	}
	std::memcpy(out, e->pending.data(), static_cast<size_t>(e->streams));
	out += e->streams;
	bool ok = true;
	for (int s = 0; s < e->slots && ok; ++s) {
		const size_t ring_bytes = static_cast<size_t>(e->tiles) * static_cast<size_t>(e->ring_cap[s]) * kLanes * sizeof(float);
		const size_t state_bytes = static_cast<size_t>(e->tiles) * kSlotStateWords * kLanes * sizeof(uint32_t);
		if (ring_bytes) {
			ok = e->be->download(out, e->ring[s], ring_bytes, nullptr);
			out += ring_bytes;
		}
		ok = ok && e->be->download(out, e->slot_state[s], state_bytes, nullptr);
		out += state_bytes;
	}
	ok = ok && e->be->download(out, e->send_state, static_cast<size_t>(e->tiles) * kSendStateWords * kLanes * sizeof(uint32_t), nullptr);
	ok = ok && e->be->sync(nullptr);
	return ok ? OALSFX_OK : e->fail(OALSFX_ERR_DEVICE, e->be->error());
}

int oalsfx_engine_restore(oalsfx_engine* e, const void* src, size_t bytes)
{
	if (!e || !src || bytes < sizeof(SnapshotHeader)) {
		return e ? e->fail(OALSFX_ERR_ARGUMENT, "Bad restore arguments.") : OALSFX_ERR_ARGUMENT;
	}
	SnapshotHeader want, got;
	snapshot_header(e, want);
	std::memcpy(&got, src, sizeof(got));
	if (got.magic != kSnapshotMagic || got.version != want.version) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Not an engine snapshot.");
	}
	if (std::memcmp(&got, &want, sizeof(got)) != 0 || bytes < got.total_bytes) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Snapshot does not match this engine (streams, format, rate, slots or effect types differ).");
	}
	if (!e->quiesce()) {
		return e->fail(OALSFX_ERR_DEVICE, e->be->error());
	}
	const char* in = static_cast<const char*>(src) + sizeof(SnapshotHeader);
	e->groups_dirty = true;
	e->frames_since_update = 128; // unknown history: let the steady-state kernels try (they check the stream state)
	if (e->placed) {
		for (int s = 0; s < e->streams; ++s) {
			e->pending[static_cast<size_t>(e->lane_of(s))] = static_cast<uint8_t>(in[s]);
		}
		in += e->streams;
		e->refill_padding = true;
		return e->canonical_state(nullptr, in) ? OALSFX_OK : e->fail(OALSFX_ERR_DEVICE, e->be->error());
	}
	std::memcpy(e->pending.data(), in, static_cast<size_t>(e->streams));
	in += e->streams;
	bool ok = true;
	for (int s = 0; s < e->slots && ok; ++s) {
		const size_t ring_bytes = static_cast<size_t>(e->tiles) * static_cast<size_t>(e->ring_cap[s]) * kLanes * sizeof(float);
		const size_t state_bytes = static_cast<size_t>(e->tiles) * kSlotStateWords * kLanes * sizeof(uint32_t);
		if (ring_bytes) {
			ok = e->be->upload(e->ring[s], in, ring_bytes, nullptr);
			in += ring_bytes;
		}
		ok = ok && e->be->upload(e->slot_state[s], in, state_bytes, nullptr);
		in += state_bytes;
	}
	ok = ok && e->be->upload(e->send_state, in, static_cast<size_t>(e->tiles) * kSendStateWords * kLanes * sizeof(uint32_t), nullptr);
	ok = ok && e->be->sync(nullptr);
	return ok ? OALSFX_OK : e->fail(OALSFX_ERR_DEVICE, e->be->error());
}

int oalsfx_engine_debug_state(oalsfx_engine* e, int stream, int slot, int32_t out[4])
{
	if (!e || !out || stream < 0 || stream >= e->streams || slot < 0 || slot >= e->slots) {
		return e ? e->fail(OALSFX_ERR_ARGUMENT, "Bad debug_state arguments.") : OALSFX_ERR_ARGUMENT;
	}
	const int lane = e->lane_of(stream);
	std::vector<uint32_t> words(static_cast<size_t>(kSlotStateWords) * kLanes);
	const uint32_t* p = e->slot_state[slot] + static_cast<size_t>(lane / kLanes) * kSlotStateWords * kLanes;
	if (!e->quiesce() || !e->be->download(words.data(), p, words.size() * sizeof(uint32_t), nullptr) ||
		!e->be->sync(nullptr)) {
		return e->fail(OALSFX_ERR_DEVICE, e->be->error());
	}
	auto word = [&](size_t i) { return static_cast<int32_t>(words[i * kLanes + static_cast<size_t>(lane % kLanes)]); };
	out[0] = out[1] = out[2] = out[3] = 0;
	const int type = e->classes[static_cast<size_t>(e->fx_class[slot][static_cast<size_t>(lane)])].type;
	switch (kind_of_type(type)) {
	case kKindModDelay: out[0] = word(offsetof(FxModDelay::State, offset) / 4); break;
	case kKindEcho: out[0] = word(offsetof(FxEcho::State, offset) / 4); break;
	case kKindRingMod: out[3] = word(offsetof(FxRingMod::State, index) / 4); break;
	case kKindReverb:
		out[0] = word(offsetof(FxReverb::State, offset) / 4);
		out[1] = word(offsetof(FxReverb::State, fade_count) / 4);
		out[2] = word(offsetof(FxReverb::State, mod_index) / 4);
		break;
	default: break;
	}
	return OALSFX_OK;
}

int oalsfx_engine_set_placement(oalsfx_engine* e, int mode)
{
	if (!e) {
		return OALSFX_ERR_ARGUMENT;
	}
	if (mode != OALSFX_PLACEMENT_CALLER && mode != OALSFX_PLACEMENT_AUTO) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Unknown placement mode.");
	}
	if (!e->quiesce()) {
		return e->fail(OALSFX_ERR_DEVICE, e->be->error());
	}
	e->placement = mode;
	if (mode == OALSFX_PLACEMENT_AUTO && !e->placed) {
		e->enter_placed();
	} else if (mode == OALSFX_PLACEMENT_CALLER && e->placed && !e->leave_placed()) {
		return e->fail(OALSFX_ERR_DEVICE, "Moving the streams back failed: " + e->be->error());
	}
	e->groups_dirty = true;
	return OALSFX_OK;
}

long long oalsfx_engine_lanes(oalsfx_engine* e, int32_t* lane_of_stream, int n)
{
	if (!e) {
		return OALSFX_ERR_ARGUMENT;
	}
	if (n < 0 || n > e->streams || (n > 0 && !lane_of_stream)) {
		return e->fail(OALSFX_ERR_ARGUMENT, "Bad lanes arguments.");
	}
	for (int s = 0; s < n; ++s) {
		lane_of_stream[s] = e->lane_of(s);
	}
	return static_cast<long long>(e->placed ? e->arena_tiles : e->tiles) * kLanes;
}

long long oalsfx_engine_launch_count(const oalsfx_engine* e) { return e ? e->launches : 0; }

const char* oalsfx_engine_last_kernel(const oalsfx_engine* e) { return (e && e->last_kernel >= 0) ? kernel_name(e->last_kernel) : ""; }

long long oalsfx_engine_device_bytes(const oalsfx_engine* e) { return e ? e->device_bytes : 0; }

const char* oalsfx_last_error(const oalsfx_engine* e) { return e ? e->error.c_str() : g_create_error.c_str(); }

const char* oalsfx_build_info(void) { return backend_build_info(); }

int oalsfx_effect_defaults(int effect_type, void* props, size_t props_bytes)
{
	if (!props || props_bytes != sizeof(oalsfxpp::EffectProps) || effect_type < 0 || effect_type >= kFxTypeCount) {
		return OALSFX_ERR_ARGUMENT;
	}
	oalsfxpp::Effect fx;
	std::memset(&fx, 0, sizeof(fx));
	fx.set_type_and_defaults(static_cast<oalsfxpp::EffectType>(effect_type));
	std::memcpy(props, &fx.props_, sizeof(fx.props_));
	return OALSFX_OK;
}

int oalsfx_effect_normalize(int effect_type, void* props, size_t props_bytes)
{
	if (!props || props_bytes != sizeof(oalsfxpp::EffectProps) || effect_type < 0 || effect_type >= kFxTypeCount) {
		return OALSFX_ERR_ARGUMENT;
	}
	oalsfxpp::Effect fx;
	fx.type_ = static_cast<oalsfxpp::EffectType>(effect_type);
	std::memcpy(&fx.props_, props, sizeof(fx.props_));
	fx.normalize();
	std::memcpy(props, &fx.props_, sizeof(fx.props_));
	return OALSFX_OK;
}

namespace {
struct PresetRow { const char* full; const oalsfxpp::EffectProps::Reverb* value; };
const PresetRow kPresets[] = {
#define OALSFX_PRESET_GROUP_BEGIN(G)
#define OALSFX_PRESET(G, N, ...) {#G "::" #N, &oalsfxpp::ReverbPresets::G::N},
#define OALSFX_PRESET_GROUP_END(G)
#include "oalsfxpp_presets.inc"
#undef OALSFX_PRESET_GROUP_BEGIN
#undef OALSFX_PRESET
#undef OALSFX_PRESET_GROUP_END
};
constexpr int kPresetCount = static_cast<int>(sizeof(kPresets) / sizeof(kPresets[0]));
} // namespace

int oalsfx_reverb_preset(const char* group, const char* name, void* props, size_t props_bytes)
{
	if (!group || !name || !props || props_bytes != sizeof(oalsfxpp::EffectProps)) {
		return OALSFX_ERR_ARGUMENT;
	}
	const std::string full = std::string(group) + "::" + name;
	for (int i = 0; i < kPresetCount; ++i) {
		if (full == kPresets[i].full) {
			oalsfxpp::EffectProps p;
			std::memset(&p, 0, sizeof(p));
			p.reverb_ = *kPresets[i].value;
			std::memcpy(props, &p, sizeof(p));
			return OALSFX_OK;
		}
	}
	return OALSFX_ERR_ARGUMENT;
}

long long oalsfx_plan_placement(const int32_t* class_of_stream, int n_streams, int32_t* engine_index_of_stream,
	int32_t* class_triples, int class_capacity, int* class_count)
{
	if (!class_of_stream || !engine_index_of_stream || n_streams < 1 || class_capacity < 0 || (class_capacity > 0 && !class_triples)) {
		return OALSFX_ERR_ARGUMENT;
	}
	// classes in order of first appearance, with their stream counts
	std::map<int32_t, int> slot_of_label;
	std::vector<int32_t> labels;
	std::vector<long long> count;
	for (int s = 0; s < n_streams; ++s) {
		auto it = slot_of_label.find(class_of_stream[s]);
		if (it == slot_of_label.end()) {
			it = slot_of_label.emplace(class_of_stream[s], static_cast<int>(labels.size())).first;
			labels.push_back(class_of_stream[s]);
			count.push_back(0);
		}
		++count[static_cast<size_t>(it->second)];
	}
	// every class starts on a tile boundary
	std::vector<long long> next(labels.size());
	long long at = 0;
	for (size_t c = 0; c < labels.size(); ++c) {
		next[c] = at;
		if (static_cast<int>(c) < class_capacity) {
			class_triples[3 * c + 0] = labels[c];
			class_triples[3 * c + 1] = static_cast<int32_t>(at);
			class_triples[3 * c + 2] = static_cast<int32_t>((count[c] + kLanes - 1) / kLanes * kLanes);
		}
		at += (count[c] + kLanes - 1) / kLanes * kLanes;
		if (at > 0x7FFFFFFFLL) {
			return OALSFX_ERR_ARGUMENT;
		}
	}
	for (int s = 0; s < n_streams; ++s) {
		engine_index_of_stream[s] = static_cast<int32_t>(next[static_cast<size_t>(slot_of_label[class_of_stream[s]])]++);
	}
	if (class_count) {
		*class_count = static_cast<int>(labels.size());
	}
	return at;
}

const char* oalsfx_reverb_preset_name(int index)
{
	return (index >= 0 && index < kPresetCount) ? kPresets[index].full : nullptr;
}

} // extern "C"
