// rsx_cta.cuh -- the shared-memory counting-sort pass of the one-CTA kernels: the single-CTA sort
// (rsx_small.cu) and the segmented sort's group kernel (rsx_segments.cu).
#pragma once

#include <type_traits>

#include "rsx_scatter.cuh"

namespace rsx {

constexpr int kCtaThreads = 1024;
constexpr int kCtaWarps = kCtaThreads / 32;
constexpr int kCtaItems = 16;              // records per thread per pass, at most
constexpr size_t kCtaBufBytes = 64 * 1024; // per ping-pong buffer (records + lane)

template <typename T> __device__ __forceinline__ void store_index(void *ib, uint32_t idx_bytes, size_t at, T v) {
	switch (idx_bytes) {
	case 1: static_cast<uint8_t *>(ib)[at] = (uint8_t)v; break;
	case 2: static_cast<uint16_t *>(ib)[at] = (uint16_t)v; break;
	case 4: static_cast<uint32_t *>(ib)[at] = (uint32_t)v; break;
	default: static_cast<unsigned long long *>(ib)[at] = (unsigned long long)v; break;
	}
}

// One stable counting-sort pass (radix_sort.hpp:83-88) of the n records in[0, n) into out by the
// 8-bit digit(r, at) of record r = in[at].  A lane of type Lane (the rank sort's index, the segmented sort's
// segment id; void = none) travels with the records.  Each warp owns one contiguous chunk of the
// array (item i of lane l = chunk start + i*32 + l) and ranks it privately, with the ticket or the
// ballot ranking like K3; only as many warps as the input needs take part in the per-warp prefix
// loops.  s_wh: [32 warps][256] counters, s_scan: 8 words.  Ends with a __syncthreads.
template <int ES, int RANK, typename Lane, typename DigitFn>
__device__ __forceinline__ void cta_pass(const typename Rec<ES>::type *in, typename Rec<ES>::type *out, const Lane *lane_in,
                                         Lane *lane_out, uint32_t n, uint32_t *s_wh, uint32_t *s_scan, DigitFn digit) {
	constexpr uint32_t FULL = 0xFFFFFFFFu;
	constexpr uint32_t chunk = kCtaItems * 32;
	const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
	const uint32_t lt = lanemask_lt();
	const uint32_t nwarps = (n + chunk - 1) / chunk;
	const uint32_t w0 = warp * chunk;
	const uint32_t wend = min(n, w0 + chunk);
	uint32_t *wh = s_wh + warp * kBins;
	if (warp < nwarps)
		for (uint32_t b = lane; b < kBins; b += 32)
			wh[b] = 0;
	__syncwarp();
	// rank inside the warp, stable (items ascending, lanes ascending)
	uint32_t rank[kCtaItems];
#pragma unroll
	for (int i = 0; i < kCtaItems; ++i) {
		const uint32_t at = w0 + i * 32 + lane;
		const bool valid = at < wend;
		uint32_t d = 0;
		if (valid)
			d = digit(in[at], at);
		if constexpr (RANK == RANK_TICKET) {
			rank[i] = valid ? atomicAdd(&wh[d], 1u) : 0u;
		} else {
			uint32_t peers = __ballot_sync(FULL, valid);
#pragma unroll
			for (int b = 0; b < 8; ++b) {
				const bool bit = (d >> b) & 1u;
				const uint32_t v = __ballot_sync(FULL, bit);
				peers &= bit ? v : ~v;
			}
			uint32_t old = 0;
			const uint32_t leader = __ffs(peers) - 1;
			if (valid && lane == leader)
				old = atomicAdd(&wh[d], (uint32_t)__popc(peers));
			old = __shfl_sync(FULL, old, valid ? leader : lane);
			rank[i] = old + __popc(peers & lt);
		}
	}
	__syncthreads();
	// digit threads: prefix over the warps, exclusive scan over the digits
	if (tid < kBins) {
		uint32_t total = 0;
		for (uint32_t w = 0; w < nwarps; ++w)
			total += s_wh[w * kBins + tid];
		uint32_t x = total;
#pragma unroll
		for (int o = 1; o < 32; o <<= 1) {
			const uint32_t y = __shfl_up_sync(FULL, x, o);
			if (lane >= o)
				x += y;
		}
		if (lane == 31)
			s_scan[warp] = x;
		asm volatile("bar.sync 1, 256;" ::: "memory");
		uint32_t run = x - total;
		for (uint32_t w = 0; w < warp; ++w)
			run += s_scan[w];
		for (uint32_t w = 0; w < nwarps; ++w) {
			const uint32_t cnt = s_wh[w * kBins + tid];
			s_wh[w * kBins + tid] = run;
			run += cnt;
		}
	}
	__syncthreads();
	// place (radix_sort.hpp:83-88)
#pragma unroll
	for (int i = 0; i < kCtaItems; ++i) {
		const uint32_t at = w0 + i * 32 + lane;
		if (at < wend) {
			const typename Rec<ES>::type r = in[at];
			const uint32_t pos = wh[digit(r, at)] + rank[i];
			out[pos] = r;
			if constexpr (!std::is_void<Lane>::value)
				lane_out[pos] = lane_in[at];
		}
	}
	__syncthreads();
}

} // namespace rsx
