// rsx_segments.cu -- the segmented sort: many independent arrays sorted in one call.
//
// A batch of segments costs two launches however many segments it has (DESIGN.md "Segmented sort"):
//   pre-pass     one read of the keys: OR / NAND of the derived keys (the batch's live columns) and
//                the descents inside segments; the last CTA writes the batch pass table (Ctl)
//   group kernel one CTA per group of consecutive short segments: one stable sort of the composite
//                key (segment in group, derived key) in shared memory -- the key columns that vary
//                inside the group, then one pass on the segment id -- written into the buffer the
//                batch's parity designates
// Segments longer than one CTA holds are sorted by the host layer with the ordinary path.
#include "rsx_cta.cuh"

namespace rsx {

namespace {

constexpr int kPreThreads = 512;

template <int ES>
__global__ void __launch_bounds__(kPreThreads) segment_prepass_kernel(const typename Rec<ES>::type *__restrict__ data, size_t n,
                                                                    KeyDesc kd, const unsigned long long *__restrict__ offsets,
                                                                    size_t nseg, WsHead *ws, Ctl *host_ctl) {
	const unsigned long long m = width_mask(kd.key_bytes);
	auto key = [&](size_t i) { return derive_key(key_word<ES>(data[i], kd.word_sel), kd); };
	unsigned long long kor = 0, knand = 0, desc = 0;
	const size_t first = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
	for (size_t i = first; i < n; i += stride) {
		const unsigned long long k = key(i);
		kor |= k;
		knand |= ~k & m;
		if (i + 1 < n)
			desc += k > key(i + 1);
	}
	// a descent across the boundary between two non-empty segments is not a descent inside a segment;
	// every distinct interior boundary b is counted once (empty segments repeat it)
	for (size_t s = first + 1; s < nseg; s += stride) {
		const unsigned long long b = offsets[s];
		if (offsets[s - 1] < b && b < n)
			desc -= key(b - 1) > key(b);
	}
	for (int o = 16; o; o >>= 1) {
		kor |= __shfl_xor_sync(0xFFFFFFFFu, kor, o);
		knand |= __shfl_xor_sync(0xFFFFFFFFu, knand, o);
		desc += __shfl_xor_sync(0xFFFFFFFFu, desc, o);
	}
	if ((threadIdx.x & 31u) == 0) {
		atomicOr(&ws->key_or, kor);
		atomicOr(&ws->key_nand, knand);
		atomicAdd(&ws->descents, desc); // modulo 2^64: the total is the count of descents inside segments
		__threadfence();
	}
	__shared__ bool s_last;
	__syncthreads();
	if (threadIdx.x == 0)
		s_last = atomicAdd(&ws->tickets[0], 1u) == gridDim.x - 1;
	__syncthreads();
	if (!s_last || threadIdx.x != 0)
		return;
	// last CTA: the batch pass table (radix_sort.hpp:60-70 over the whole batch)
	__threadfence();
	const unsigned long long k_or = atomicOr(&ws->key_or, 0ULL), k_nand = atomicOr(&ws->key_nand, 0ULL);
	const unsigned long long varying = k_or & k_nand & m;
	Ctl ctl = {};
	ctl.early_exit = atomicAdd(&ws->descents, 0ULL) == 0;
	for (uint32_t c = 0; c < kd.key_bytes; ++c)
		if ((varying >> (8 * c)) & 0xFFu) { // the digit of column c is not the same in every record
			ctl.ordinal[c] = ctl.ncols++;
			ctl.live_mask |= 1u << c;
		}
	ctl.n = n;
	ctl.key_or = k_or;
	ctl.key_nand = k_nand;
	ws->ctl = ctl;
	if (host_ctl != nullptr)
		*host_ctl = ctl; // mapped pinned memory: the host reads it after the stream has drained
}

template <int ES, bool RANKSORT> __host__ __device__ constexpr uint32_t group_capacity() {
	// records + the lane that travels with them: the group-local index (rank sort) or a 1-byte segment id
	constexpr uint32_t by_bytes = (uint32_t)((kCtaBufBytes - 16) / (ES + (RANKSORT ? 4 : 1)));
	constexpr uint32_t by_items = (uint32_t)kCtaThreads * kCtaItems;
	return by_bytes < by_items ? by_bytes : by_items;
}

struct GroupParams {
	const void *src;
	void *out_even, *out_odd; // value sort: src, aux
	void *index_buffer;       // rank sort: 2n entries of idx_bytes
	uint32_t idx_bytes;       // 0 = value sort
	size_t n;
	KeyDesc kd;
	const SegGroup *groups;
	const uint32_t *segtab;
	const Ctl *ctl;
};

// index of the segment holding group-local record i: s_seg[0 .. nseg] are the ascending segment starts
// (all segments non-empty) and the group length
__device__ __forceinline__ uint32_t segment_of(const uint32_t *s_seg, uint32_t nseg, uint32_t i) {
	uint32_t lo = 0, hi = nseg;
	while (hi - lo > 1) {
		const uint32_t mid = (lo + hi) >> 1;
		if (s_seg[mid] <= i)
			lo = mid;
		else
			hi = mid;
	}
	return lo;
}

template <int ES, bool RANKSORT, int RANK>
__global__ void __launch_bounds__(kCtaThreads, 1) segment_group_kernel(const GroupParams p) {
	using R = typename Rec<ES>::type;
	using Lane = typename std::conditional<RANKSORT, uint32_t, uint8_t>::type;
	constexpr uint32_t kCap = group_capacity<ES, RANKSORT>();
	constexpr size_t kLaneOff = ((size_t)kCap * ES + 15) & ~(size_t)15;
	extern __shared__ __align__(16) unsigned char smem[];
	R *const rec0 = reinterpret_cast<R *>(smem), *const rec1 = reinterpret_cast<R *>(smem + kCtaBufBytes);
	Lane *const lane0 = reinterpret_cast<Lane *>(smem + kLaneOff), *const lane1 = reinterpret_cast<Lane *>(smem + kCtaBufBytes + kLaneOff);
	uint32_t *const s_wh = reinterpret_cast<uint32_t *>(smem + 2 * kCtaBufBytes); // [32 warps][256]
	uint32_t *const s_scan = s_wh + kCtaWarps * kBins;                            // 16 words
	unsigned long long *const s_var = reinterpret_cast<unsigned long long *>(s_scan + 16); // OR, NAND of the group
	uint32_t *const s_seg = reinterpret_cast<uint32_t *>(s_var + 2);             // kMaxGroupSegments + 1

	const Ctl *ctl = p.ctl;
	const uint32_t early = ctl->early_exit;
	if (!RANKSORT && early)
		return; // every segment is ordered: nothing moves (radix_sort.hpp:60-62)
	const SegGroup g = p.groups[blockIdx.x];
	const uint32_t tid = threadIdx.x, n = g.len, nseg = g.nseg;
	for (uint32_t i = tid; i <= nseg; i += kCtaThreads)
		s_seg[i] = p.segtab[g.tab + i];
	if (tid < 2)
		s_var[tid] = 0;
	__syncthreads();
	if (RANKSORT && early) { // segment-relative identity in the first half (radix_sort_rank.hpp:52-57)
		for (uint32_t i = tid; i < n; i += kCtaThreads)
			store_index(p.index_buffer, p.idx_bytes, g.begin + i, i - s_seg[segment_of(s_seg, nseg, i)]);
		return;
	}

	// ---- load; which key bits vary inside the group ----
	const KeyDesc kd = p.kd;
	const R *in = static_cast<const R *>(p.src) + g.begin;
	const unsigned long long m = width_mask(kd.key_bytes);
	unsigned long long kor = 0, knand = 0;
	for (uint32_t i = tid; i < n; i += kCtaThreads) {
		const R r = in[i];
		rec0[i] = r;
		lane0[i] = RANKSORT ? i : segment_of(s_seg, nseg, i);
		const unsigned long long k = derive_key(key_word<ES>(r, kd.word_sel), kd);
		kor |= k;
		knand |= ~k & m;
	}
	for (int o = 16; o; o >>= 1) {
		kor |= __shfl_xor_sync(0xFFFFFFFFu, kor, o);
		knand |= __shfl_xor_sync(0xFFFFFFFFu, knand, o);
	}
	if ((tid & 31u) == 0) {
		atomicOr(&s_var[0], kor);
		atomicOr(&s_var[1], knand);
	}
	__syncthreads();
	const unsigned long long varying = s_var[0] & s_var[1];

	// ---- one pass per column that varies inside the group, then the segment id ----
	// A column that is constant inside the group leaves the group's order as it is, so skipping it
	// gives the same content as the batch's pass on it would.
	bool flip = false; // records in rec1 / lane1
	for (uint32_t c = 0; c < kd.key_bytes; ++c) {
		if (!((varying >> (8 * c)) & 0xFFu))
			continue;
		const R *rin = flip ? rec1 : rec0;
		const auto digit = [&](const R &r, uint32_t) {
			return (uint32_t)(derive_key(key_word<ES>(r, kd.word_sel), kd) >> (8 * c)) & 0xFFu;
		};
		cta_pass<ES, RANK>(rin, flip ? rec0 : rec1, flip ? lane1 : lane0, flip ? lane0 : lane1, n, s_wh, s_scan, digit);
		flip = !flip;
	}
	if (nseg > 1) { // the most significant digit: every segment lands back in its own range
		const Lane *lin = flip ? lane1 : lane0;
		const auto digit = [&](const R &, uint32_t at) -> uint32_t {
			if constexpr (RANKSORT)
				return segment_of(s_seg, nseg, lin[at]);
			else
				return lin[at];
		};
		cta_pass<ES, RANK>(flip ? rec1 : rec0, flip ? rec0 : rec1, lin, flip ? lane0 : lane1, n, s_wh, s_scan, digit);
		flip = !flip;
	}

	// ---- into the buffer the batch's parity designates (radix_sort.hpp:89-92) ----
	const uint32_t odd = ctl->ncols & 1u;
	if constexpr (RANKSORT) {
		const Lane *res = flip ? lane1 : lane0;
		const size_t off = (odd ? p.n : 0) + g.begin; // radix_sort_rank.hpp:77-91
		for (uint32_t i = tid; i < n; i += kCtaThreads)
			store_index(p.index_buffer, p.idx_bytes, off + i, res[i] - s_seg[segment_of(s_seg, nseg, i)]);
	} else {
		const R *res = flip ? rec1 : rec0;
		R *out = static_cast<R *>(odd ? p.out_odd : p.out_even) + g.begin;
		for (uint32_t i = tid; i < n; i += kCtaThreads)
			out[i] = res[i];
	}
}

constexpr size_t kGroupSmem = 2 * kCtaBufBytes + (size_t)kCtaWarps * kBins * 4 + 16 * 4 + 2 * 8 + (kMaxGroupSegments + 1) * 4;

template <int ES, bool RANKSORT>
cudaError_t launch_groups_t(const GroupParams &gp, size_t ngroups, cudaStream_t st) {
	const bool ticket = rank_mode() == RANK_TICKET;
	auto k0 = segment_group_kernel<ES, RANKSORT, RANK_TICKET>;
	auto k1 = segment_group_kernel<ES, RANKSORT, RANK_BALLOT>;
	auto kern = ticket ? k0 : k1;
	cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGroupSmem);
	if (e != cudaSuccess)
		return e;
	kern<<<(unsigned)ngroups, kCtaThreads, kGroupSmem, st>>>(gp);
	count_launch();
	return cudaGetLastError();
}

} // namespace

size_t segment_group_capacity(uint32_t record_bytes, bool ranksort) {
	switch (record_bytes) {
	case 1: return ranksort ? group_capacity<1, true>() : group_capacity<1, false>();
	case 2: return ranksort ? group_capacity<2, true>() : group_capacity<2, false>();
	case 4: return ranksort ? group_capacity<4, true>() : group_capacity<4, false>();
	case 8: return ranksort ? group_capacity<8, true>() : group_capacity<8, false>();
	case 16: return ranksort ? group_capacity<16, true>() : group_capacity<16, false>();
	}
	return 0;
}

cudaError_t launch_segment_prepass(const void *src, size_t n, uint32_t record_bytes, const KeyDesc &kd,
                                   const unsigned long long *offsets, size_t nseg, WsHead *ws, Ctl *host_ctl,
                                   int num_sms, cudaStream_t st) {
	const size_t want = (n + kPreThreads - 1) / kPreThreads;
	const unsigned grid = (unsigned)(want < (size_t)num_sms * 4 ? (want ? want : 1) : (size_t)num_sms * 4);
	switch (record_bytes) {
#define PRE(ES)                                                                                                     \
	case ES:                                                                                                        \
		segment_prepass_kernel<ES><<<grid, kPreThreads, 0, st>>>(static_cast<const typename Rec<ES>::type *>(src), n, kd, \
		                                                         offsets, nseg, ws, host_ctl);                        \
		break;
		PRE(1) PRE(2) PRE(4) PRE(8) PRE(16)
#undef PRE
	default: return cudaErrorInvalidValue;
	}
	count_launch();
	return cudaGetLastError();
}

cudaError_t launch_segment_groups(const void *src, void *out_even, void *out_odd, void *index_buffer, int idx_bytes, size_t n,
                                  uint32_t record_bytes, const KeyDesc &kd, const SegGroup *groups, size_t ngroups,
                                  const uint32_t *segtab, const Ctl *ctl, cudaStream_t st) {
	GroupParams gp;
	gp.src = src;
	gp.out_even = out_even;
	gp.out_odd = out_odd;
	gp.index_buffer = index_buffer;
	gp.idx_bytes = (uint32_t)idx_bytes;
	gp.n = n;
	gp.kd = kd;
	gp.groups = groups;
	gp.segtab = segtab;
	gp.ctl = ctl;
	const bool rs = idx_bytes != 0;
	switch (record_bytes) {
	case 1: return rs ? launch_groups_t<1, true>(gp, ngroups, st) : launch_groups_t<1, false>(gp, ngroups, st);
	case 2: return rs ? launch_groups_t<2, true>(gp, ngroups, st) : launch_groups_t<2, false>(gp, ngroups, st);
	case 4: return rs ? launch_groups_t<4, true>(gp, ngroups, st) : launch_groups_t<4, false>(gp, ngroups, st);
	case 8: return rs ? launch_groups_t<8, true>(gp, ngroups, st) : launch_groups_t<8, false>(gp, ngroups, st);
	case 16: return rs ? launch_groups_t<16, true>(gp, ngroups, st) : launch_groups_t<16, false>(gp, ngroups, st);
	}
	return cudaErrorInvalidValue;
}

} // namespace rsx
