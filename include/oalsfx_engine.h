/* oalsfx_engine.h -- C ABI of the batched B200 effects engine (the drop-in boundary).
 *
 * The reference has no FFI of its own; its only boundary is the C++ class oalsfxpp::Api
 * (reference: src/oalsfxpp.h:760-922).  This ABI is what a binding for that class's hot path
 * would call: one engine owns `num_streams` independent streams, each of which behaves exactly
 * like one reference `Api` instance (same channel format, sampling rate and slot count for the
 * whole engine).  include/oalsfxpp.h re-exports the reference's C++ class on top of it with
 * num_streams = 1.
 *
 * Plain pointers and sizes only; no exceptions cross this boundary.  Every call returns
 * OALSFX_OK (0) or a negative error code; oalsfx_last_error() gives the message.
 * There is no CPU implementation behind this ABI: creation fails without a CUDA device.
 */
#ifndef OALSFX_ENGINE_H
#define OALSFX_ENGINE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct oalsfx_engine oalsfx_engine;

enum {
	OALSFX_OK = 0,
	OALSFX_ERR_ARGUMENT = -1,   /* bad index / pointer / size */
	OALSFX_ERR_FORMAT = -2,     /* invalid channel format        (reference: oalsfxpp.cpp:2855-2861) */
	OALSFX_ERR_RATE = -3,       /* sampling rate out of range    (reference: oalsfxpp.cpp:2863-2868) */
	OALSFX_ERR_EFFECTS = -4,    /* effect count out of range     (reference: oalsfxpp.cpp:2870-2875) */
	OALSFX_ERR_DEVICE = -5,     /* CUDA failure / no device */
	OALSFX_ERR_MEMORY = -6
};

/* Sample buffer layouts for oalsfx_engine_mix.  F = frames of the call, C = channels. */
enum {
	OALSFX_LAYOUT_STREAM_MAJOR = 0, /* [stream][frame][channel]: every stream's buffer is exactly the
	                                   interleaved buffer Api::mix takes (reference: oalsfxpp.h:872-875) */
	OALSFX_LAYOUT_TILED = 1         /* [tile = stream/32][frame][channel][lane = stream%32]: engine-native,
	                                   fully coalesced; the stream count is padded to a multiple of 32 */
};

enum { OALSFX_SPACE_HOST = 0, OALSFX_SPACE_DEVICE = 1 };

typedef struct oalsfx_engine_desc {
	int32_t device;         /* CUDA device ordinal */
	int32_t num_streams;    /* >= 1 */
	int32_t channel_format; /* oalsfxpp::ChannelFormat value (1 mono .. 7 seven_point_one) */
	int32_t sampling_rate;  /* >= 8000 */
	int32_t effect_count;   /* 1..4 slots per stream */
} oalsfx_engine_desc;

/* Replaces Api::initialize (reference: oalsfxpp.cpp:3480-3504, 2846-2905). */
int oalsfx_engine_create(const oalsfx_engine_desc* desc, oalsfx_engine** out);

/* Replaces Api::uninitialize / ~Api (reference: oalsfxpp.cpp:3831-3834). */
void oalsfx_engine_destroy(oalsfx_engine* e);

/* Replaces EffectSlot::set_effect as reached from Api::apply_changes (reference:
 * oalsfxpp.cpp:2688-2709, 3748-3756) for streams [first_stream, first_stream + n_streams).
 * `props` points at the bytes of an oalsfxpp::EffectProps (108 bytes; ignored for the null
 * effect); they are normalized (clamped) like Effect::normalize does.  A change of effect TYPE
 * resets that slot's state (delay lines, filter history), a change of properties keeps it.  The
 * new coefficients take effect at the top of the next mixed block (reference: oalsfxpp.cpp:3000). */
int oalsfx_engine_set_effect(oalsfx_engine* e, int first_stream, int n_streams, int slot,
	int effect_type, const void* props, size_t props_bytes);

/* Replaces the send half of Api::apply_changes (reference: oalsfxpp.cpp:3760-3780, 3348-3395).
 * direct = {gain, gain_hf, gain_lf}; aux = effect_count such triples (slot order). */
int oalsfx_engine_set_sends(oalsfx_engine* e, int first_stream, int n_streams,
	const float* direct, const float* aux);

/* Voice lifecycle.  In the reference each voice is one Api, and a host mixes only the voices that play; a voice it does
 * not mix keeps its delay lines and filter histories as they are.
 * oalsfx_engine_set_active: streams [first_stream, first_stream + n_streams) are mixed (active != 0, the default for
 * every stream) or paused.  From the next mix on the engine does not process a paused stream -- it is an Api whose mix is
 * not called: its rings, slot state, send filter histories, ring offsets, LFO / modulator phases, tap cross-fade counter
 * and pending updates stay exactly as they are, and it costs no mix work.  Its src rows are not read and its dst rows
 * receive +0.0f in every frame and channel (both layouts, both spaces, mix and mix_bus; so the bus of a block is the sum
 * over the streams that were mixed).  A resumed stream continues bit for bit like that Api on its next mix.  set_effect /
 * set_sends on a paused stream behave as always: a type change resets the slot at once, property changes are consumed by
 * the first block that mixes the stream again.  Activity is configuration, like effect types: snapshots do not hold it
 * and restore leaves it alone.  Pausing whole 32-stream tiles keeps the fused kernels of the rest; scattered pauses leave
 * partly paused tiles, which an unplaced engine runs on the slower per-stream path -- OALSFX_PLACEMENT_AUTO packs paused
 * streams into tiles of their own instead (a pause or resume then costs a lane move, like a preset change).
 * oalsfx_engine_reset_streams: the streams restart from silence -- every slot's delay lines and state and the send
 * filter histories are zeroed and every slot holding an effect gets its update again, as from the set_effect that
 * configured it -- so that each continues like a freshly created engine given the same set_effect / set_sends calls
 * (a fresh Api with the same effects and sends after apply_changes).  The configuration and the activity flag are kept.
 * Both wait for the stream the caller last passed in, as set_effect does, and return OALSFX_ERR_ARGUMENT for a bad
 * range. */
int oalsfx_engine_set_active(oalsfx_engine* e, int first_stream, int n_streams, int active);
int oalsfx_engine_reset_streams(oalsfx_engine* e, int first_stream, int n_streams);

/* Ordering: with device buffers oalsfx_engine_mix / mix_bus / reduce_bus / the PCM conversions are ENQUEUED on
 * `cuda_stream` and return at once; consecutive calls on the same stream run in order.  Every other call that touches
 * engine state on the device -- set_effect / set_sends / set_active / reset_streams (state reset, arena growth, table
 * uploads at the next mix), snapshot, restore, debug_state, destroy -- first waits for the stream the caller last passed in, so it is safe to
 * call them at any time, also with cudaStreamNonBlocking streams.  Using several streams on one engine concurrently
 * is the caller's to order.  Precondition of the fused kernels: finite input samples (an Inf / NaN sample times a
 * gain the reference skips as inaudible would reach output channels the reference leaves untouched). */
/* Replaces Api::mix for all streams at once (reference: oalsfxpp.cpp:3785-3829, 2984-3037).
 * `frames` per stream; internally cut into blocks of <= 2048 frames exactly like the reference.
 * src/dst hold num_streams*frames*C floats (TILED: stream count rounded up to 32) in `space`;
 * dst is overwritten, not clipped.  Device buffers must not overlap.  With host buffers the call
 * stages through device memory and returns after the results are back; with device buffers the
 * work is enqueued on `cuda_stream` (a cudaStream_t, may be NULL) and the call returns at once. */
int oalsfx_engine_mix(oalsfx_engine* e, int frames, const float* src, float* dst,
	int layout, int space, void* cuda_stream);

/* Optional all-streams output bus: bus[frame][channel] (device, frames*C floats) = sum over this
 * engine's streams of a STREAM_MAJOR/TILED device buffer `dst` produced by oalsfx_engine_mix.
 * No reference counterpart (SURVEY.md 8e); the cross-GPU sum is one all-reduce of `bus`. */
int oalsfx_engine_reduce_bus(oalsfx_engine* e, int frames, const float* dst, int layout,
	float* bus, void* cuda_stream);

/* Host buffers: oalsfx_engine_mix with OALSFX_SPACE_HOST copies at the pinned rate (and overlaps copies with kernels)
 * only from page-locked memory; pageable memory (malloc, new, std::vector) goes through the driver's bounce buffers at a
 * fraction of it.  oalsfx_engine_pin_host page-locks a caller's buffer IN PLACE (cudaHostRegister) until
 * oalsfx_engine_unpin_host or oalsfx_engine_destroy; the buffer must stay allocated for that long.  With the environment
 * variable OALSFX_PIN_HOST=1 the engine does this by itself for every host buffer it is handed (same lifetime rule:
 * do not free or unmap such a buffer while the engine lives; moving or resizing is detected by address overlap). */
int oalsfx_engine_pin_host(oalsfx_engine* e, void* buffer, size_t bytes);
int oalsfx_engine_unpin_host(oalsfx_engine* e, void* buffer);

/* oalsfx_engine_mix (device buffers) followed by oalsfx_engine_reduce_bus on the same stream: the block's output and
 * bus[frame * C + c] = its sum over the engine's streams (device array of frames * C floats) from one call. */
int oalsfx_engine_mix_bus(oalsfx_engine* e, int frames, const float* src, float* dst, int layout,
	float* bus, void* cuda_stream);

/* Submix buses.  A host sums its voices into a few buses -- per listener, player, room or category -- rather than
 * consuming one output row per stream.  Every stream is routed to one bus (>= 0) or to none (OALSFX_BUS_NONE); a new
 * engine routes every stream to bus 0.  Routing is configuration, like effect types and activity: reset_streams and
 * set_placement keep it, snapshots do not hold it and restore leaves it alone.
 * oalsfx_engine_route_streams: bus[i] becomes the bus of stream first_stream + i.  Waits for the stream the caller last
 * passed in, as set_active does; OALSFX_ERR_ARGUMENT for a bad range, a null `bus` or an entry below OALSFX_BUS_NONE.
 * oalsfx_engine_reduce_buses: buses[(b * frames + f) * C + c] (DEVICE array of n_buses * frames * C floats) = the sum over
 * the members of bus b of a device buffer `dst` produced by oalsfx_engine_mix (either layout).  The members of bus b are
 * the streams routed to b that are active at the time of the call (paused streams are not members and their rows are
 * not read; padding lanes of TILED buffers never are).  Every one of the n_buses buses is written; a bus without
 * members receives +0.0f.  Summation order, the same for every (frame, channel):
 *   - the members of the bus in ascending caller stream index are the level-0 list;
 *   - while the list has more than one entry, it is cut into consecutive runs of 32 (the last one shorter); each run is
 *     summed left to right in fp32 starting from +0.0f; the run sums, in order, are the next level's list;
 *   - a single member gives +0.0f + v.
 * The order depends neither on the layout nor on the placement mode nor on how the frames of a call are processed, so
 * STREAM_MAJOR and TILED give bit-identical buses, so do CALLER and AUTO placement, and one call of many frames equals
 * one call per block.  (The all-streams bus of oalsfx_engine_reduce_bus keeps its own order.)  OALSFX_ERR_ARGUMENT for a
 * null pointer, frames <= 0, an unknown layout, n_buses < 1 or n_buses not above every routed bus index.  Enqueued on
 * `cuda_stream`, returns at once; after a routing or activity change the first call rebuilds and uploads the bus plan,
 * the others neither synchronize, allocate nor upload.  With several GPUs each rank's buses sum with one all-reduce.
 * oalsfx_engine_mix_buses: oalsfx_engine_mix (device buffers) and oalsfx_engine_reduce_buses on the same stream; every
 * argument is checked before the mix, so a refused call advances no stream. */
enum { OALSFX_BUS_NONE = -1 };
int oalsfx_engine_route_streams(oalsfx_engine* e, int first_stream, int n_streams, const int32_t* bus);

/* Routes with gains.  A stream may feed up to OALSFX_MAX_ROUTES buses -- its category bus and a room's reverb send, one bus
 * per listener in split screen, two rooms while a voice moves between them -- each route with its own gain, and a gain
 * change ramps over a given number of frames instead of jumping (the reference ramps every gain it changes: MixHelpers
 * gain steps, oalsfxpp.cpp:2762-2797).
 * oalsfx_engine_set_routes: with R = routes_per_stream (1..OALSFX_MAX_ROUTES), the routes of stream first_stream + i
 * become the entries r < R with bus[i * R + r] != OALSFX_BUS_NONE, each with gain gain[i * R + r] (gain NULL: 1.0f);
 * every other route of the stream is removed.  OALSFX_ERR_ARGUMENT, with nothing changed, for a bad range, R outside
 * 1..OALSFX_MAX_ROUTES, a null `bus`, a bus index below OALSFX_BUS_NONE, a stream naming the same bus twice, a gain that is
 * not finite, or ramp_frames outside [0, 2^24].  Waits for the stream the caller last passed in, as route_streams does.
 * oalsfx_engine_route_streams(e, first, n, bus) is set_routes(e, first, n, 1, bus, NULL, 0): it also removes a stream's
 * other routes.  Routes and ramps in progress are configuration like the routing: reset_streams, set_placement and
 * restore keep them, snapshots do not hold them.  In reduce_buses / mix_buses n_buses must be above every bus any route
 * names.
 *   - The frame clock: the engine counts the frames it has mixed; every successful mix / mix_bus / mix_buses call adds its
 *     `frames`, whichever streams are paused and whichever space its buffers are in (a refused call adds nothing).  M is
 *     the clock at the start of the most recent such call (0 before the first), and reduce_buses gives frame f of its
 *     block the clock value T = M + f.  So reduce_buses right after mix equals mix_buses, reducing a block twice or in
 *     both layouts gives the same bits, and one long call equals one call per block.
 *   - A route holds a start gain g0, a target gain g1, a ramp length Rf and a ramp start T0.  Its gain at clock T, in fp32
 *     with one rounding per operation, in this order, no contraction:  T < T0: g0;  Rf == 0 or T - T0 >= Rf: g1;
 *     otherwise g0 + (g1 - g0) * ((float)(T - T0 + 1) / (float)Rf).
 *   - set_routes(..., ramp_frames) sets, for every route it lists: T0 = the clock now (the first frame of the next mix),
 *     Rf = ramp_frames, g1 = the new gain, and g0 = the route's gain at T0 - 1 when the stream already had a route to that
 *     bus (the gain its last mixed frame received, or its old g0 if nothing was mixed since the last change), else 0.0f.
 *     With ramp_frames == 0, g0 = g1: the new gain holds at every T, so a block mixed before the call is reduced with it,
 *     as route_streams has always done.
 *     A crossfade between rooms is therefore one call, {old: 0, new: 1} with a ramp, and once the ramp has ended
 *     {new: 1}.  A removed route stops at once: ramp it to 0 first.
 *   - Bus b's members are the routes to b of the streams active at the call, in ascending caller stream index (a stream
 *     has at most one route per bus); a member's value is the fp32 product gain(T) * x, one rounding, and the members are
 *     summed in the order above.  Routes of gain 0 are members (0 * Inf is NaN on the bus).  A chunk of frames in which
 *     every member's gain is 1.0f runs the unweighted sum, which gives the same bits at the speed of plain routing.
 *   - A call that changes gains or ramps only, keeping every (stream, bus) pair, costs one upload of the gains at the next
 *     reduce; a change of the pairs rebuilds the bus plan as route_streams does. */
enum { OALSFX_MAX_ROUTES = 4 };
int oalsfx_engine_set_routes(oalsfx_engine* e, int first_stream, int n_streams, int routes_per_stream,
	const int32_t* bus, const float* gain, int ramp_frames);
/* Bus format and pans.  A host with mono voices and a stereo or 5.1 output, or one listener bus per player in split screen,
 * pans each voice into each bus with gains of its own, in the buses' deterministic order.
 * oalsfx_engine_set_bus_format: every submix bus gets the channel format `channel_format` (an oalsfxpp::ChannelFormat value,
 * as in oalsfx_engine_desc) and Cb = its channel count (1..8); the default is the engine's own format (Cb = C).  From then
 * on reduce_buses / mix_buses write buses[(b * frames + f) * Cb + j], n_buses * frames * Cb floats, in both layouts; the
 * all-streams bus of reduce_bus / mix_bus keeps the engine's format.  OALSFX_ERR_FORMAT for an invalid format;
 * OALSFX_ERR_ARGUMENT, with nothing changed, for a change of Cb while any route is a pan route (its matrix is sized for the
 * old Cb); setting the current format again always succeeds.  Waits for the stream the caller last passed in, as
 * set_routes does.  The bus format is configuration: reset_streams, set_placement and restore keep it, snapshots do not
 * hold it.
 * oalsfx_engine_set_route_pans: as set_routes -- the same `bus` array, the same checks, nothing changed by a refused call,
 * every route of a listed stream that the call does not name removed -- but each named route r of stream first_stream + i
 * gets a Cb x C matrix instead of a gain: pan[((i * R + r) * Cb + j) * C + k] is the weight of stream channel k in bus
 * channel j.  OALSFX_ERR_ARGUMENT also for a null `pan` or a coefficient of a named route that is not finite.
 *   - Scalar routes (route_streams, set_routes, the default routing) feed bus channel j < min(C, Cb) with g(T) * x_j and
 *     bus channels j >= C with nothing.  With Cb == C this is the plain routing above, with the same kernels and bits.
 *     With Cb != C the mapping is by index: a mono engine routed by default feeds only the left channel of a stereo bus,
 *     and a stereo voice routed to a mono bus feeds it its left channel.  Pan the voice to mix its channels.
 *   - A pan route's value in bus channel j is, in fp32 with one rounding per operation and no contraction,
 *     p = c_j0(T) * x_0, then p = p + c_jk(T) * x_k for k = 1..C-1.  Every coefficient takes part (0 * Inf is NaN, as for a
 *     route of gain 0).  Each coefficient ramps as a gain does: c_jk(T) is the gain expression above with g0_jk, g1_jk and
 *     the route's Rf and T0.  set_route_pans sets T0 = the clock now, Rf = ramp_frames, g1 = the new matrix, and g0 = each
 *     coefficient's value at T0 - 1 when the stream already had a route to that bus, else 0.0f (a scalar route's matrix is
 *     its gain g(T0 - 1) where j == k and 0.0f elsewhere); with ramp_frames == 0, g0 = g1 and the matrix applies at once,
 *     also to a block mixed before the call.
 *   - set_routes / route_streams on a pan route: with ramp_frames == 0 it becomes a scalar route at once; with a ramp it
 *     stays a pan route whose target is the gain on the index diagonal (j == k) and 0.0f elsewhere, so that the other
 *     coefficients ramp out, and a later call without a ramp makes it scalar (the crossfade idiom above).
 *   - The members and their order are those above; a member's value is now per (frame, bus channel).  So the buses stay
 *     bit-identical across layouts, placements, repeated reduces and the cut of a call into blocks.  With Cb == C an
 *     identity matrix times g gives the bits of set_routes(g) for a finite block (the extra terms are +-0.0f, and a run sum
 *     starting from +0.0f never becomes -0.0f); with C == Cb == 1 a pan route is bit-identical to a scalar route.
 *   - A set_route_pans that keeps every (stream, bus) pair costs one upload of the coefficients at the next reduce, as a
 *     gain change does; a change of the pairs rebuilds the plan.  Pan coefficients on the device count in device_bytes. */
int oalsfx_engine_set_bus_format(oalsfx_engine* e, int channel_format);
int oalsfx_engine_set_route_pans(oalsfx_engine* e, int first_stream, int n_streams, int routes_per_stream,
	const int32_t* bus, const float* pan, int ramp_frames);
int oalsfx_engine_reduce_buses(oalsfx_engine* e, int frames, const float* dst, int layout,
	int n_buses, float* buses, void* cuda_stream);
int oalsfx_engine_mix_buses(oalsfx_engine* e, int frames, const float* src, float* dst, int layout,
	int n_buses, float* buses, void* cuda_stream);

/* PCM formats either side of the path (device buffers; SURVEY.md 8f rank 2).  The reference's only
 * producer and consumer of Api::mix buffers is its WAV demo, and these are its conversions:
 *   oalsfx_pcm_to_float : bit_depth 8: (u8 - 128) / 128.0f, 16: s16 / 32768.0f  (oalsfxpp_test.cpp:703-740)
 *   oalsfx_float_to_s16 : each of `rows` buffers of `row_len` samples (one per stream) is peak-normalised the
 *                         way WavFile::save does it -- scale = 1 / max(max(1, max x), -min(-1, min x)),
 *                         s16 = (int16)(scale * x * 32767.0f), truncating (oalsfxpp_test.cpp:602-651);
 *                         row_scale (device, `rows` floats, may be NULL) receives the scales.
 * They let a caller keep 2-byte samples on the host side of PCIe and in HBM between calls. */
int oalsfx_pcm_to_float(oalsfx_engine* e, const void* src, int bit_depth, float* dst, long long count,
	void* cuda_stream);
int oalsfx_float_to_s16(oalsfx_engine* e, const float* src, int16_t* dst, int rows, long long row_len,
	float* row_scale, void* cuda_stream);

/* State snapshot / restore (SURVEY.md 8f rank 3; the reference has no counterpart: an Api's delay lines
 * and filter histories are private).  A snapshot holds every byte the streams carry from one block to the
 * next (delay-line rings, slot state, send filter histories, pending-update flags) into a HOST buffer of
 * oalsfx_engine_snapshot_size() bytes; restore puts it back into an engine of identical geometry whose
 * slots hold the same effect types and properties (the caller's configuration is not part of it).  After
 * a restore the engine continues bit for bit as the snapshotted one would have.  Both synchronize. */
long long oalsfx_engine_snapshot_size(const oalsfx_engine* e);
int oalsfx_engine_snapshot(oalsfx_engine* e, void* dst, size_t bytes);
int oalsfx_engine_restore(oalsfx_engine* e, const void* src, size_t bytes);

/* Integer state of one stream's slot, for bit-exact checks: out[0]=ring write offset,
 * out[1]=reverb fade_count, out[2]=reverb mod index, out[3]=ring-mod phase index.
 * Unused entries are 0.  Synchronizes the device. */
int oalsfx_engine_debug_state(oalsfx_engine* e, int stream, int slot, int32_t out[4]);

/* Test hook: the three waveshapers of the distortion effect (oalsfxpp.cpp:4720-4722) applied to `count` samples in a
 * DEVICE buffer with the given edge coefficient, through the very function the distortion stage runs (fx.cuh,
 * FxDistortion::shape: the divisions as one batched correctly-rounded sequence instead of the `/` operator), so that a
 * test can hold it bit for bit against IEEE division over the whole operand range.  Asynchronous on cuda_stream. */
int oalsfx_debug_waveshaper(oalsfx_engine* e, const float* samples, float edge_coeff, float* out, long long count, void* cuda_stream);

/* How many of the engine's kernels have been launched so far (bench.py's gpu_launches). */
long long oalsfx_engine_launch_count(const oalsfx_engine* e);

/* Name of the mix kernel the engine launched most recently ("" before the first mix), e.g. "kDuoChainStereo":
 * which of the kernel families served the last block (measurement records, tests of the selection logic). */
const char* oalsfx_engine_last_kernel(const oalsfx_engine* e);

/* Bytes of device memory the engine currently holds. */
long long oalsfx_engine_device_bytes(const oalsfx_engine* e);

/* Message for the last failed call on this engine (or on creation when e == NULL). */
const char* oalsfx_last_error(const oalsfx_engine* e);

/* Property helpers for bindings (reference: Effect::set_type_and_defaults / Effect::normalize,
 * oalsfxpp.cpp:1782-1833; ReverbPresets, oalsfxpp.cpp:1938-2191).  `props` = 108-byte EffectProps. */
int oalsfx_effect_defaults(int effect_type, void* props, size_t props_bytes);
int oalsfx_effect_normalize(int effect_type, void* props, size_t props_bytes);
/* group/name as in the header, e.g. ("Default", "forest"); index-based enumeration via
 * oalsfx_reverb_preset_name(i) which returns "Group::name" or NULL past the end. */
int oalsfx_reverb_preset(const char* group, const char* name, void* props, size_t props_bytes);
const char* oalsfx_reverb_preset_name(int index);

/* Stream placement for many parameter sets (SURVEY.md 8 f1).  The engine runs a 32-stream tile at the fused kernels' speed
 * when all of its streams share one parameter set ("class"); a tile of mixed classes takes table mode, ~15x slower per
 * stream.  A host that owns many voices with arbitrary presets decides the ORDER of its streams in the engine -- each
 * stream is an independent row of the mix buffers, as each Api instance of the reference has its own buffer
 * (oalsfxpp.cpp:2820-2827) -- and this helper computes an order that keeps every tile class-pure: given one label per
 * caller stream (equal labels = the same settings in every slot and send), classes are laid out one after the other in
 * order of first appearance, each padded to a multiple of 32; streams of a class keep their relative order.
 * engine_index_of_stream[s] receives the engine stream index of caller stream s.  Returns the number of engine streams to
 * create (>= n_streams; indices nobody was assigned are silent streams: feed zeros, ignore their output), or a negative
 * OALSFX_ERR_* code.  class_triples / class_count are optional: with class_capacity > 0, up to class_capacity triples
 * (label, first engine index, length of the class's range INCLUDING its padding streams: a multiple of 32) are written,
 * so that one oalsfx_engine_set_effect call per class configures its whole range -- the padding streams must carry their
 * tile's settings, or the tile is a mixed one again. */
long long oalsfx_plan_placement(const int32_t* class_of_stream, int n_streams, int32_t* engine_index_of_stream,
	int32_t* class_triples, int class_capacity, int* class_count);

/* Stream placement inside the engine.  In OALSFX_PLACEMENT_AUTO mode the engine keeps every 32-stream tile class-pure
 * by itself: before a block whose configuration changed (set_effect, set_sends, a consumed update) it moves streams
 * between its internal lanes -- a stream already in a pure tile of its own settings stays where it is, so changing k
 * streams moves about k streams -- growing its arenas by whole tiles when needed (they never shrink).  Caller stream
 * indices and every buffer keep their meaning and layout: set_effect, set_sends, mix, mix_bus, reduce_bus,
 * debug_state, snapshot and restore take and return caller streams; the mix permutes the block into lane order and
 * back on the device (two extra passes over the block).  A snapshot is written in caller stream order, so it restores
 * into an engine in either mode.  Only speed, launch_count, last_kernel and device_bytes show the placement; host
 * buffers take the unsliced staging path.  Switching back to OALSFX_PLACEMENT_CALLER (the default: lane = stream)
 * moves every stream back to its own lane, after which the engine runs as one that was never placed.  Returns
 * OALSFX_OK or OALSFX_ERR_ARGUMENT for an unknown mode; a failed move reports OALSFX_ERR_DEVICE.  Synchronizes. */
enum {
	OALSFX_PLACEMENT_CALLER = 0, /* default: engine lane of stream s is s */
	OALSFX_PLACEMENT_AUTO = 1    /* the engine moves streams between lanes so that every tile holds one class */
};
int oalsfx_engine_set_placement(oalsfx_engine* e, int mode);
/* lane_of_stream[s] for s < n (n <= num_streams, lane_of_stream may be NULL when n == 0): the engine lane that holds
 * caller stream s now.  Returns the engine's lane count (a multiple of 32) or a negative OALSFX_ERR_* code. */
long long oalsfx_engine_lanes(oalsfx_engine* e, int32_t* lane_of_stream, int n);

/* Library build identification, e.g. "oalsfx_b200 sm_100a cuda". */
const char* oalsfx_build_info(void);

#ifdef __cplusplus
}
#endif

#endif /* OALSFX_ENGINE_H */
