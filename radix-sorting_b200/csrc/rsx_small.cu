// rsx_small.cu -- the whole sort in ONE launch for inputs that fit one CTA's shared memory.
//
// The multi-kernel path (memset, K1, K2, one K3 per column, read-back) has a floor of ~100 us
// whatever n is; the reference at n = 1000 takes ~2 us on a CPU core (README.md:640-650 makes the
// same point about fixed overheads and hybrids).  Below kSmallBytes of records this kernel does
// everything rs_sort_main / rs_sort_rank do (radix_sort.hpp:31-93, radix_sort_rank.hpp:22-92) inside
// one 1024-thread CTA: load, all-column histograms + pre-sorted detection, column probe, one
// stable counting-sort pass per live column between two shared-memory buffers (warp-private
// ticket / ballot ranking exactly like K3), and a final store into the buffer the reference's
// parity rule designates.  Same device pass table (Ctl) as the big path, so the host side is
// unchanged: one launch, one 40-byte read-back.
#include "rsx_cta.cuh"

namespace rsx {

namespace {

constexpr int kSmallThreads = kCtaThreads;
constexpr int kSmallWarps = kCtaWarps;
constexpr size_t kSmallBytes = kCtaBufBytes; // per ping-pong buffer (records + index lane)

struct SmallParams {
	const void *src;      // input records
	void *out_even;       // value sort: where the result goes if #live columns is even (src itself)
	void *out_odd;        // value sort: ... odd (aux)
	void *index_buffer;   // rank sort: 2n entries of idx_bytes
	uint32_t idx_bytes;   // 0 = value sort
	uint32_t n;
	KeyDesc kd;
	Ctl *ctl;
};

template <int ES, bool RANKSORT, int RANK>
__global__ void __launch_bounds__(kSmallThreads, 1) small_sort_kernel(const SmallParams p) {
	using R = typename Rec<ES>::type;
	constexpr uint32_t kCap = (uint32_t)((kSmallBytes - 16) / (ES + (RANKSORT ? 4 : 0)));
	constexpr size_t kIdxOff = ((size_t)kCap * ES + 15) & ~(size_t)15; // index lane behind the records
	extern __shared__ __align__(16) unsigned char smem[];
	R *buf[2] = {reinterpret_cast<R *>(smem), reinterpret_cast<R *>(smem + kSmallBytes)};
	uint32_t *idx[2] = {reinterpret_cast<uint32_t *>(smem + kIdxOff),
	                    reinterpret_cast<uint32_t *>(smem + kSmallBytes + kIdxOff)};
	uint32_t *s_wh = reinterpret_cast<uint32_t *>(smem + 2 * kSmallBytes);          // [32 warps][256]
	uint32_t *s_hist = s_wh + kSmallWarps * kBins;                                  // [8 columns][256]
	uint32_t *s_misc = s_hist + kMaxCols * kBins;                                   // scan scratch, live flags

	const uint32_t tid = threadIdx.x;
	const uint32_t n = p.n;
	const KeyDesc kd = p.kd;
	const R *in = static_cast<const R *>(p.src);

	// ---- load + zero the column histograms ----
	for (uint32_t i = tid; i < n; i += kSmallThreads) {
		buf[0][i] = in[i];
		if constexpr (RANKSORT)
			idx[0][i] = i; // radix_sort_rank.hpp:52
	}
	for (uint32_t i = tid; i < kMaxCols * kBins; i += kSmallThreads)
		s_hist[i] = 0;
	__syncthreads();

	// ---- all histograms in one read + pre-sorted detection (radix_sort.hpp:48-58) ----
	uint32_t descents = 0;
	for (uint32_t i = tid; i < n; i += kSmallThreads) {
		const unsigned long long k = derive_key(key_word<ES>(buf[0][i], kd.word_sel), kd);
		for (uint32_t c = 0; c < kd.key_bytes; ++c)
			atomicAdd(&s_hist[c * kBins + ((uint32_t)(k >> (8 * c)) & 0xFFu)], 1u);
		if (i + 1 < n)
			descents += k > derive_key(key_word<ES>(buf[0][i + 1], kd.word_sel), kd);
	}
	const int unsorted = __syncthreads_or((int)descents);
	if (!unsorted) { // radix_sort.hpp:60-62 / radix_sort_rank.hpp:55-57: nothing moves
		if constexpr (RANKSORT)
			for (uint32_t i = tid; i < n; i += kSmallThreads)
				store_index(p.index_buffer, p.idx_bytes, i, i);
		if (tid == 0) {
			Ctl ctl = {};
			ctl.early_exit = 1;
			ctl.n = n;
			*p.ctl = ctl;
		}
		return;
	}

	// ---- column probe with the first key (radix_sort.hpp:65-70) ----
	if (tid < kMaxCols) {
		const unsigned long long key0 = derive_key(key_word<ES>(buf[0][0], kd.word_sel), kd);
		s_misc[16 + tid] = tid < kd.key_bytes && s_hist[tid * kBins + ((uint32_t)(key0 >> (8 * tid)) & 0xFFu)] != n;
	}
	__syncthreads();

	uint32_t cur = 0, ncols = 0, live_mask = 0;

	for (uint32_t c = 0; c < kd.key_bytes; ++c) {
		if (!s_misc[16 + c])
			continue; // trivial column (uniform)
		const auto digit = [&](const R &r, uint32_t) {
			return (uint32_t)(derive_key(key_word<ES>(r, kd.word_sel), kd) >> (8 * c)) & 0xFFu;
		};
		R *const r0 = cur ? buf[1] : buf[0], *const r1 = cur ? buf[0] : buf[1];
		if constexpr (RANKSORT)
			cta_pass<ES, RANK>(r0, r1, cur ? idx[1] : idx[0], cur ? idx[0] : idx[1], n, s_wh, s_misc, digit);
		else
			cta_pass<ES, RANK, void>(r0, r1, nullptr, nullptr, n, s_wh, s_misc, digit);
		cur ^= 1; // swap(src, aux), radix_sort.hpp:89
		++ncols;
		live_mask |= 1u << c;
	}

	// ---- result into the buffer the parity rule designates (radix_sort.hpp:89-92) ----
	if constexpr (RANKSORT) {
		const size_t off = (ncols & 1u) ? n : 0; // radix_sort_rank.hpp:77-91
		for (uint32_t i = tid; i < n; i += kSmallThreads)
			store_index(p.index_buffer, p.idx_bytes, off + i, idx[cur][i]);
	} else {
		R *out = static_cast<R *>((ncols & 1u) ? p.out_odd : p.out_even);
		for (uint32_t i = tid; i < n; i += kSmallThreads)
			out[i] = buf[cur][i];
	}
	if (tid == 0) {
		Ctl ctl = {};
		ctl.ncols = ncols;
		ctl.live_mask = live_mask;
		ctl.n = n;
		*p.ctl = ctl;
	}
}

constexpr size_t kSmallSmem = 2 * kSmallBytes + (size_t)kSmallWarps * kBins * 4 + (size_t)kMaxCols * kBins * 4 + 256;

template <int ES, bool RANKSORT>
cudaError_t launch_small_t(const SmallParams &sp, cudaStream_t st) {
	const bool ticket = rank_mode() == RANK_TICKET;
	auto k0 = small_sort_kernel<ES, RANKSORT, RANK_TICKET>;
	auto k1 = small_sort_kernel<ES, RANKSORT, RANK_BALLOT>;
	auto kern = ticket ? k0 : k1;
	cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmallSmem);
	if (e != cudaSuccess)
		return e;
	kern<<<1, kSmallThreads, kSmallSmem, st>>>(sp);
	count_launch();
	return cudaGetLastError();
}

} // namespace

size_t small_sort_capacity(uint32_t record_bytes, bool ranksort) {
	size_t cap = (kSmallBytes - 16) / (record_bytes + (ranksort ? 4 : 0));
	const size_t by_items = (size_t)kSmallWarps * 32 * kCtaItems; // 16 records per thread
	return cap < by_items ? cap : by_items;
}

cudaError_t launch_small_sort(const void *src, void *out_even, void *out_odd, void *index_buffer, int idx_bytes,
                              size_t n, uint32_t record_bytes, const KeyDesc &kd, Ctl *ctl, cudaStream_t st) {
	SmallParams sp;
	sp.src = src;
	sp.out_even = out_even;
	sp.out_odd = out_odd;
	sp.index_buffer = index_buffer;
	sp.idx_bytes = (uint32_t)idx_bytes;
	sp.n = (uint32_t)n;
	sp.kd = kd;
	sp.ctl = ctl;
	const bool rs = idx_bytes != 0;
	switch (record_bytes) {
	case 1: return rs ? launch_small_t<1, true>(sp, st) : launch_small_t<1, false>(sp, st);
	case 2: return rs ? launch_small_t<2, true>(sp, st) : launch_small_t<2, false>(sp, st);
	case 4: return rs ? launch_small_t<4, true>(sp, st) : launch_small_t<4, false>(sp, st);
	case 8: return rs ? launch_small_t<8, true>(sp, st) : launch_small_t<8, false>(sp, st);
	case 16: return rs ? launch_small_t<16, true>(sp, st) : launch_small_t<16, false>(sp, st);
	}
	return cudaErrorInvalidValue;
}

} // namespace rsx
