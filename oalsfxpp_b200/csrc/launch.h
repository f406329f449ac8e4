// launch.h -- the kernel families, one translation unit each (k_*.cu), so that nvcc compiles them in parallel.
//
// Every launcher answers whether `kernel_id` belongs to its family; if it does, the kernel has been launched on
// `stream` and the caller checks cudaGetLastError().
#ifndef OALSFX_LAUNCH_H
#define OALSFX_LAUNCH_H

#include <cuda_runtime.h>

#include <cstdlib>

#include "bus.cuh"
#include "kernel_table.h"

namespace oalsfx {

bool launch_mix_family(int kernel_id, const MixArgs& args, cudaStream_t stream);      // k_mix.cu: thread per stream (Gen*, fused, Tab*)
bool launch_duo_family(int kernel_id, const MixArgs& args, cudaStream_t stream);      // k_duo.cu: duo_kernel, duo_multi_kernel
bool launch_quartet_family(int kernel_id, const MixArgs& args, cudaStream_t stream);  // k_quartet.cu
bool launch_relay_family(int kernel_id, const MixArgs& args, cudaStream_t stream);    // k_relay.cu: relay_kernel, relay_multi_kernel
bool launch_span_family(int kernel_id, const MixArgs& args, cudaStream_t stream);     // k_span.cu: block-parallel in time
bool launch_scan_family(int kernel_id, const MixArgs& args, cudaStream_t stream);     // k_scan.cu: linear-recurrence scan over time

// k_place.cu: stream placement and paused streams (see Backend::copy_lanes / gather_io / scatter_io / zero_rows)
bool launch_copy_lanes(uint32_t* dst, long long dst_ts, int dst_w0, const uint32_t* src, long long src_ts, int src_w0, int words,
	const int32_t* from, const int32_t* to, int n, cudaStream_t stream);
bool launch_gather_io(const float* src, long long ts, long long ls, long long fs, long long cs, const int32_t* stream_of_lane,
	int lane_tiles, int frames, int channels, float* dst, cudaStream_t stream);
bool launch_scatter_io(const float* src, const int32_t* stream_of_lane, int lane_tiles, int frames, int channels, float* dst,
	long long ts, long long ls, long long fs, long long cs, cudaStream_t stream);
bool launch_zero_rows(float* dst, long long ts, long long ls, long long fs, long long cs, const int32_t* rows, int n, int frames,
	int channels, cudaStream_t stream);
// k_bus.cu: every level of one chunk of the submix buses (see Backend::reduce_buses)
bool launch_reduce_buses(const bus::Chunk& chunk, cudaStream_t stream);

// Shared-memory carve-out of a kernel, set once.  Tuning knobs (experiments only): OALSFX_TUNE_CARVEOUT = percent or
// -1 (driver default), OALSFX_TUNE_DYN_SMEM = bytes of unused dynamic shared memory per CTA (caps residency).
template <class K>
inline size_t prefer_shared(bool& done, K kernel, int default_carveout)
{
	static size_t tune_dyn_smem = 0;
	if (!done) {
		int carveout = default_carveout;
		if (const char* e = getenv("OALSFX_TUNE_CARVEOUT")) {
			carveout = atoi(e);
		}
		if (const char* e = getenv("OALSFX_TUNE_DYN_SMEM")) {
			tune_dyn_smem = static_cast<size_t>(atoi(e));
			cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(tune_dyn_smem));
		}
		if (carveout >= 0) {
			cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carveout);
		}
		done = true;
	}
	return tune_dyn_smem;
}

} // namespace oalsfx

#endif
