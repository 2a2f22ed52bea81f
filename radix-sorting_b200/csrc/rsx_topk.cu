// rsx_topk.cu -- top-k selection: the first k records (or indices) of the stable sort without
// sorting the whole array (rsx_topk / rsx_topk_rank, include/rsx.h; DESIGN.md "Top-k").
//
//   1. threshold search: MSD radix select on the derived key.  One read-only histogram launch per
//      column, top column first, counts the digits of the records whose higher columns equal the
//      prefix chosen so far.  The last CTA of the launch picks the bucket holding the k-th record and
//      extends the prefix (TopkState).  A launch that finds the search done returns at once, so the
//      host enqueues all key_bytes launches without waiting.
//   2. stable select: one read-only pass writes the records below the prefix, in input order, then
//      the first k - less records equal to it, in input order.  Each CTA owns one contiguous chunk of
//      the input; the search passes left per-chunk counts, so a CTA knows where its records go.
//   3. the k selected records are sorted by the ordinary paths (rsx_api.cu).
#include "rsx_device.cuh"

namespace rsx {

namespace {

constexpr int kTopkThreads = 1024; // the block scan below assumes 32 warps
constexpr int kTopkUnroll = 4;     // 16-byte vectors in flight per thread

// Records of chunk j, in input order: the unaligned head (j == 0), vectors [j * per, (j + 1) * per),
// the tail (j == last).
struct ChunkRange {
	size_t v0, v1;
};
__device__ __forceinline__ ChunkRange chunk_range(const TopkChunks &g) {
	const size_t v0 = (size_t)blockIdx.x * g.per;
	return {v0 < g.n_vec ? v0 : g.n_vec, v0 + g.per < g.n_vec ? v0 + g.per : g.n_vec};
}

// Digit histogram of column `col` over the records whose derived-key bits above it equal s->prefix.
// Lane-private shared counters (copy l of a bin lives in bank l, as in K1), so a constant or heavily
// tied column does not serialise on one counter.
template <int ES>
__global__ void __launch_bounds__(kTopkThreads, 1)
topk_hist_kernel(const typename Rec<ES>::type *__restrict__ src, size_t n, KeyDesc kd, uint32_t col, TopkChunks g, size_t k,
                 TopkState *s, uint32_t *__restrict__ chunk_hist, unsigned long long *__restrict__ chunk_lt,
                 unsigned long long *__restrict__ chunk_eq) {
	using R = typename Rec<ES>::type;
	constexpr int VEC = 16 / ES;
	__shared__ uint32_t sh[kBins * 32];
	__shared__ unsigned long long s_scan[8];
	__shared__ uint32_t s_last, s_bucket;
	__shared__ unsigned long long s_below, s_count;
	if (__ldcg(&s->done))
		return;
	const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
	const unsigned long long prefix = __ldcg(&s->prefix);
	const bool top = col + 1 == kd.key_bytes;
	const uint32_t hs = top ? 0u : 8u * (col + 1), ds = 8u * col;
	for (uint32_t i = tid; i < kBins * 32; i += kTopkThreads)
		sh[i] = 0;
	__syncthreads();
	auto count = [&](const R &r) {
		const unsigned long long key = derive_key(key_word<ES>(r, kd.word_sel), kd);
		if (top || (key >> hs) == prefix)
			atomicAdd(&sh[(((uint32_t)(key >> ds)) & 0xFFu) * 32u + lane], 1u);
	};
	const ChunkRange cr = chunk_range(g);
	const uint4 *vsrc = reinterpret_cast<const uint4 *>(src + g.head);
	for (size_t b = cr.v0; b < cr.v1; b += (size_t)kTopkThreads * kTopkUnroll) {
		uint4 q[kTopkUnroll];
#pragma unroll
		for (int u = 0; u < kTopkUnroll; ++u) {
			const size_t v = b + (size_t)u * kTopkThreads + tid;
			q[u] = v < cr.v1 ? __ldg(vsrc + v) : make_uint4(0, 0, 0, 0);
		}
#pragma unroll
		for (int u = 0; u < kTopkUnroll; ++u) {
			if (b + (size_t)u * kTopkThreads + tid < cr.v1) {
				const R *e = reinterpret_cast<const R *>(&q[u]);
#pragma unroll
				for (int j = 0; j < VEC; ++j)
					count(e[j]);
			}
		}
	}
	if (blockIdx.x == 0)
		for (size_t i = tid; i < g.head; i += kTopkThreads)
			count(src[i]);
	if (blockIdx.x == gridDim.x - 1)
		for (size_t i = g.head + g.n_vec * VEC + tid; i < n; i += kTopkThreads)
			count(src[i]);
	__syncthreads();
	// a chunk holds fewer than 2^32 records, so its counts fit 32 bits
	for (uint32_t bin = warp; bin < kBins; bin += kTopkThreads / 32) {
		const uint32_t v = __reduce_add_sync(0xFFFFFFFFu, sh[bin * 32u + lane]);
		if (lane == 0) {
			chunk_hist[(size_t)blockIdx.x * kBins + bin] = v;
			if (v)
				atomicAdd(&s->hist[bin], (unsigned long long)v);
		}
	}
	__threadfence();
	__syncthreads();
	if (tid == 0)
		s_last = atomicAdd(&s->ticket, 1u) == gridDim.x - 1;
	__syncthreads();
	if (!s_last)
		return;
	__threadfence();

	// ---- the last CTA: pick the bucket that holds record k - 1 (0-based) of the sort ----
	const unsigned long long less = __ldcg(&s->less), need = k - less; // records still to take, >= 1
	unsigned long long h = 0, x = 0;
	if (tid < kBins) {
		h = __ldcg(&s->hist[tid]);
		x = h;
#pragma unroll
		for (int o = 1; o < 32; o <<= 1) {
			const unsigned long long y = __shfl_up_sync(0xFFFFFFFFu, x, o);
			if (lane >= (uint32_t)o)
				x += y;
		}
		if (lane == 31)
			s_scan[warp] = x;
	}
	__syncthreads();
	if (tid < kBins) {
		for (uint32_t w = 0; w < warp; ++w)
			x += s_scan[w];
		const unsigned long long below = x - h; // records of the prefix bucket in lower digits
		if (below < need && need <= x) {
			s_bucket = tid;
			s_below = below;
			s_count = h;
		}
	}
	__syncthreads();
	const uint32_t bkt = s_bucket;
	// per chunk: records below the new prefix (accumulated over the columns) and records equal to it
	for (uint32_t c = warp; c < gridDim.x; c += kTopkThreads / 32) {
		uint32_t lt = 0, eq = 0;
#pragma unroll
		for (uint32_t i = 0; i < 8; ++i) {
			const uint32_t d = lane * 8u + i;
			const uint32_t v = __ldcg(&chunk_hist[(size_t)c * kBins + d]);
			lt += d < bkt ? v : 0u;
			eq += d == bkt ? v : 0u;
		}
		lt = __reduce_add_sync(0xFFFFFFFFu, lt);
		eq = __reduce_add_sync(0xFFFFFFFFu, eq);
		if (lane == 0) {
			chunk_lt[c] += lt;
			chunk_eq[c] = eq;
		}
	}
	if (tid < kBins)
		s->hist[tid] = 0;
	if (tid == 0) {
		s->less = less + s_below;
		s->prefix = (top ? 0ull : prefix << 8) | bkt;
		s->ncols += 1;
		s->col = col;
		s->done = s_count == need - s_below || col == 0;
		s->ticket = 0;
	}
}

// Exclusive scan of two counters over the 1024 threads of the block; ta / tb get the block totals.
// Callers separate two calls by a barrier (sw is reused).
__device__ __forceinline__ void block_scan2(unsigned long long &a, unsigned long long &b, unsigned long long &ta,
                                            unsigned long long &tb, unsigned long long (*sw)[2]) {
	const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
	unsigned long long xa = a, xb = b;
#pragma unroll
	for (int o = 1; o < 32; o <<= 1) {
		const unsigned long long ya = __shfl_up_sync(0xFFFFFFFFu, xa, o), yb = __shfl_up_sync(0xFFFFFFFFu, xb, o);
		if (lane >= (uint32_t)o) {
			xa += ya;
			xb += yb;
		}
	}
	if (lane == 31) {
		sw[warp][0] = xa;
		sw[warp][1] = xb;
	}
	__syncthreads();
	if (warp == 0) {
		unsigned long long wa = sw[lane][0], wb = sw[lane][1];
#pragma unroll
		for (int o = 1; o < 32; o <<= 1) {
			const unsigned long long ya = __shfl_up_sync(0xFFFFFFFFu, wa, o), yb = __shfl_up_sync(0xFFFFFFFFu, wb, o);
			if (lane >= (uint32_t)o) {
				wa += ya;
				wb += yb;
			}
		}
		sw[lane][0] = wa;
		sw[lane][1] = wb;
	}
	__syncthreads();
	a = (warp ? sw[warp - 1][0] : 0ull) + xa - a;
	b = (warp ? sw[warp - 1][1] : 0ull) + xb - b;
	ta = sw[31][0];
	tb = sw[31][1];
}

template <int ES, typename I> struct SelectCtx {
	using R = typename Rec<ES>::type;
	R *out;
	I *idx;          // nullptr: value form
	KeyDesc kd;
	uint32_t ds;     // bit offset of the last searched column
	unsigned long long prefix, less, q;
	unsigned long long lt_base, eq_base; // records of this kind written (seen) before the current step
};

// One step of the select: thread t holds NU groups of NV consecutive records; group u of every thread
// precedes group u + 1 in input order, and inside a group the threads are in order.  Per-group counts
// are packed 16 bits apiece (a group has at most 1024 x 16 records), so one block scan serves all.
// rec(u, j) returns record j of group u (the records stay packed in the loaded vectors: 64 one-byte
// records in separate registers would spill).
template <int ES, typename I, int NU, int NV, typename At>
__device__ __forceinline__ void select_step(SelectCtx<ES, I> &c, const At &rec, const bool (&valid)[NU], const size_t (&pos)[NU],
                                            unsigned long long (*sw)[2]) {
	auto cls = [&](const typename Rec<ES>::type &x) -> uint32_t { // 1: below the prefix, 2: equal to it
		const unsigned long long p = derive_key(key_word<ES>(x, c.kd.word_sel), c.kd) >> c.ds;
		return p < c.prefix ? 1u : p == c.prefix ? 2u : 0u;
	};
	unsigned long long lt = 0, eq = 0;
#pragma unroll
	for (int u = 0; u < NU; ++u) {
		if (!valid[u])
			continue;
#pragma unroll
		for (int j = 0; j < NV; ++j) {
			const uint32_t k = cls(rec(u, j));
			lt += (unsigned long long)(k == 1u) << (16 * u);
			eq += (unsigned long long)(k == 2u) << (16 * u);
		}
	}
	if (!__syncthreads_or((lt | eq) != 0))
		return;
	unsigned long long tl, te;
	block_scan2(lt, eq, tl, te, sw);
	unsigned long long gl = c.lt_base, ge = c.eq_base;
#pragma unroll
	for (int u = 0; u < NU; ++u) {
		unsigned long long pl = gl + ((lt >> (16 * u)) & 0xFFFFu), pe = ge + ((eq >> (16 * u)) & 0xFFFFu);
		if (valid[u]) {
#pragma unroll
			for (int j = 0; j < NV; ++j) {
				const uint32_t k = cls(rec(u, j));
				if (k == 1u) {
					c.out[pl] = rec(u, j);
					if (c.idx)
						c.idx[pl] = (I)(pos[u] + j);
					++pl;
				} else if (k == 2u) {
					if (pe < c.q) {
						c.out[c.less + pe] = rec(u, j);
						if (c.idx)
							c.idx[c.less + pe] = (I)(pos[u] + j);
					}
					++pe;
				}
			}
		}
		gl += (tl >> (16 * u)) & 0xFFFFu;
		ge += (te >> (16 * u)) & 0xFFFFu;
	}
	c.lt_base = gl;
	c.eq_base = ge;
}

template <int ES, typename I>
__global__ void __launch_bounds__(kTopkThreads, 1)
topk_select_kernel(const typename Rec<ES>::type *__restrict__ src, size_t n, size_t k, KeyDesc kd, TopkChunks g,
                   const TopkState *s, const unsigned long long *__restrict__ chunk_lt, const unsigned long long *__restrict__ chunk_eq,
                   typename Rec<ES>::type *__restrict__ out, I *__restrict__ idx) {
	using R = typename Rec<ES>::type;
	constexpr int VEC = 16 / ES;
	__shared__ unsigned long long sw[32][2];
	__shared__ unsigned long long s_base[2];
	const uint32_t tid = threadIdx.x, lane = tid & 31u;
	SelectCtx<ES, I> c;
	c.out = out;
	c.idx = idx;
	c.kd = kd;
	c.ds = 8u * __ldcg(&s->col);
	c.prefix = __ldcg(&s->prefix);
	c.less = __ldcg(&s->less);
	c.q = k - c.less;
	if (tid < 32) { // this chunk's offsets: the counts of the chunks before it
		unsigned long long a = 0, b = 0;
		for (uint32_t j = lane; j < blockIdx.x; j += 32) {
			a += chunk_lt[j];
			b += chunk_eq[j];
		}
		for (int o = 16; o; o >>= 1) {
			a += __shfl_xor_sync(0xFFFFFFFFu, a, o);
			b += __shfl_xor_sync(0xFFFFFFFFu, b, o);
		}
		if (lane == 0) {
			s_base[0] = a;
			s_base[1] = b;
		}
	}
	__syncthreads();
	c.lt_base = s_base[0];
	c.eq_base = s_base[1];
	const unsigned long long lt_end = c.lt_base + chunk_lt[blockIdx.x], eq_end = c.eq_base + chunk_eq[blockIdx.x];
	auto finished = [&]() { return c.lt_base == lt_end && (c.eq_base == eq_end || c.eq_base >= c.q); };
	auto scalar = [&](size_t from, size_t to) {
		for (size_t i0 = from; i0 < to && !finished(); i0 += kTopkThreads) {
			const size_t i = i0 + tid;
			bool valid[1] = {i < to};
			size_t pos[1] = {i};
			const R r = valid[0] ? src[i] : R{};
			select_step<ES, I, 1, 1>(c, [&](int, int) { return r; }, valid, pos, sw);
		}
	};
	if (blockIdx.x == 0)
		scalar(0, g.head);
	const ChunkRange cr = chunk_range(g);
	const uint4 *vsrc = reinterpret_cast<const uint4 *>(src + g.head);
	for (size_t b = cr.v0; b < cr.v1 && !finished(); b += (size_t)kTopkThreads * kTopkUnroll) {
		uint4 q[kTopkUnroll];
		bool valid[kTopkUnroll];
		size_t pos[kTopkUnroll];
#pragma unroll
		for (int u = 0; u < kTopkUnroll; ++u) {
			const size_t v = b + (size_t)u * kTopkThreads + tid;
			valid[u] = v < cr.v1;
			pos[u] = g.head + v * VEC;
			q[u] = valid[u] ? __ldg(vsrc + v) : make_uint4(0, 0, 0, 0);
		}
		select_step<ES, I, kTopkUnroll, VEC>(c, [&](int u, int j) { return reinterpret_cast<const R *>(&q[u])[j]; }, valid, pos, sw);
	}
	if (blockIdx.x == gridDim.x - 1)
		scalar(g.head + g.n_vec * VEC, n);
}

template <typename IR, typename IS, typename IO>
__global__ void topk_gather_kernel(const IR *__restrict__ rank, const IS *__restrict__ sel, IO *__restrict__ out, size_t k) {
	for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < k; i += (size_t)gridDim.x * blockDim.x)
		out[i] = (IO)sel[rank ? (size_t)rank[i] : i];
}

template <typename IR, typename IS>
cudaError_t gather_to(const void *rank, const void *sel, void *out, int idx_bytes, size_t k, int grid, cudaStream_t st) {
	const IR *r = static_cast<const IR *>(rank);
	const IS *s = static_cast<const IS *>(sel);
	switch (idx_bytes) {
	case 1: topk_gather_kernel<<<grid, 256, 0, st>>>(r, s, static_cast<uint8_t *>(out), k); break;
	case 2: topk_gather_kernel<<<grid, 256, 0, st>>>(r, s, static_cast<uint16_t *>(out), k); break;
	case 4: topk_gather_kernel<<<grid, 256, 0, st>>>(r, s, static_cast<uint32_t *>(out), k); break;
	case 8: topk_gather_kernel<<<grid, 256, 0, st>>>(r, s, static_cast<unsigned long long *>(out), k); break;
	default: return cudaErrorInvalidValue;
	}
	return cudaSuccess;
}

template <int ES>
cudaError_t launch_select_es(const void *src, size_t n, size_t k, const KeyDesc &kd, const TopkChunks &g, const TopkState *s,
                             const unsigned long long *clt, const unsigned long long *ceq, void *out, void *sel_idx,
                             int sel_idx_bytes, cudaStream_t st) {
	using R = typename Rec<ES>::type;
	const R *sr = static_cast<const R *>(src);
	R *o = static_cast<R *>(out);
	if (sel_idx_bytes == 0)
		topk_select_kernel<ES, uint32_t><<<g.nchunks, kTopkThreads, 0, st>>>(sr, n, k, kd, g, s, clt, ceq, o, nullptr);
	else if (sel_idx_bytes == 4)
		topk_select_kernel<ES, uint32_t><<<g.nchunks, kTopkThreads, 0, st>>>(sr, n, k, kd, g, s, clt, ceq, o, static_cast<uint32_t *>(sel_idx));
	else if (sel_idx_bytes == 8)
		topk_select_kernel<ES, unsigned long long><<<g.nchunks, kTopkThreads, 0, st>>>(sr, n, k, kd, g, s, clt, ceq, o,
		                                                                               static_cast<unsigned long long *>(sel_idx));
	else
		return cudaErrorInvalidValue;
	return cudaSuccess;
}

} // namespace

TopkChunks topk_chunks(const void *src, size_t n, uint32_t record_bytes, int num_sms) {
	TopkChunks g;
	const uintptr_t addr = reinterpret_cast<uintptr_t>(src);
	g.head = ((16 - (addr & 15)) & 15) / record_bytes; // as K1: records are aligned to their size
	if (g.head > n)
		g.head = n;
	g.n_vec = (n - g.head) / (16 / record_bytes);
	// one 1024-thread CTA per SM; fewer when the input is small
	const size_t step = (size_t)kTopkThreads * kTopkUnroll;
	size_t want = (g.n_vec + step - 1) / step;
	want = want < 1 ? 1 : want > (size_t)num_sms ? (size_t)num_sms : want;
	g.nchunks = (uint32_t)want;
	g.per = (g.n_vec + want - 1) / want;
	return g;
}

cudaError_t launch_topk_hist(const void *src, size_t n, size_t k, uint32_t record_bytes, const KeyDesc &kd, int col,
                             const TopkChunks &g, TopkState *s, uint32_t *chunk_hist, unsigned long long *chunk_lt,
                             unsigned long long *chunk_eq, cudaStream_t st) {
	const uint32_t c = (uint32_t)col;
	switch (record_bytes) {
	case 1: topk_hist_kernel<1><<<g.nchunks, kTopkThreads, 0, st>>>(static_cast<const uint8_t *>(src), n, kd, c, g, k, s, chunk_hist, chunk_lt, chunk_eq); break;
	case 2: topk_hist_kernel<2><<<g.nchunks, kTopkThreads, 0, st>>>(static_cast<const uint16_t *>(src), n, kd, c, g, k, s, chunk_hist, chunk_lt, chunk_eq); break;
	case 4: topk_hist_kernel<4><<<g.nchunks, kTopkThreads, 0, st>>>(static_cast<const uint32_t *>(src), n, kd, c, g, k, s, chunk_hist, chunk_lt, chunk_eq); break;
	case 8: topk_hist_kernel<8><<<g.nchunks, kTopkThreads, 0, st>>>(static_cast<const unsigned long long *>(src), n, kd, c, g, k, s, chunk_hist, chunk_lt, chunk_eq); break;
	case 16: topk_hist_kernel<16><<<g.nchunks, kTopkThreads, 0, st>>>(static_cast<const ulonglong2 *>(src), n, kd, c, g, k, s, chunk_hist, chunk_lt, chunk_eq); break;
	default: return cudaErrorInvalidValue;
	}
	count_launch();
	return cudaGetLastError();
}

cudaError_t launch_topk_select(const void *src, size_t n, size_t k, uint32_t record_bytes, const KeyDesc &kd, const TopkChunks &g,
                               const TopkState *s, const unsigned long long *chunk_lt, const unsigned long long *chunk_eq,
                               void *out, void *sel_idx, int sel_idx_bytes, cudaStream_t st) {
	cudaError_t e;
	switch (record_bytes) {
	case 1: e = launch_select_es<1>(src, n, k, kd, g, s, chunk_lt, chunk_eq, out, sel_idx, sel_idx_bytes, st); break;
	case 2: e = launch_select_es<2>(src, n, k, kd, g, s, chunk_lt, chunk_eq, out, sel_idx, sel_idx_bytes, st); break;
	case 4: e = launch_select_es<4>(src, n, k, kd, g, s, chunk_lt, chunk_eq, out, sel_idx, sel_idx_bytes, st); break;
	case 8: e = launch_select_es<8>(src, n, k, kd, g, s, chunk_lt, chunk_eq, out, sel_idx, sel_idx_bytes, st); break;
	case 16: e = launch_select_es<16>(src, n, k, kd, g, s, chunk_lt, chunk_eq, out, sel_idx, sel_idx_bytes, st); break;
	default: return cudaErrorInvalidValue;
	}
	if (e != cudaSuccess)
		return e;
	count_launch();
	return cudaGetLastError();
}

cudaError_t launch_topk_gather(const void *rank, int rank_bytes, const void *sel_idx, int sel_idx_bytes, void *index_out,
                               int idx_bytes, size_t k, int num_sms, cudaStream_t st) {
	size_t g = (k + 255) / 256;
	const int grid = (int)(g < 1 ? 1 : g > (size_t)num_sms * 8 ? (size_t)num_sms * 8 : g);
	cudaError_t e;
	if (rank_bytes == 8)
		e = sel_idx_bytes == 8 ? gather_to<unsigned long long, unsigned long long>(rank, sel_idx, index_out, idx_bytes, k, grid, st)
		                       : gather_to<unsigned long long, uint32_t>(rank, sel_idx, index_out, idx_bytes, k, grid, st);
	else
		e = sel_idx_bytes == 8 ? gather_to<uint32_t, unsigned long long>(rank, sel_idx, index_out, idx_bytes, k, grid, st)
		                       : gather_to<uint32_t, uint32_t>(rank, sel_idx, index_out, idx_bytes, k, grid, st);
	if (e != cudaSuccess)
		return e;
	count_launch();
	return cudaGetLastError();
}

} // namespace rsx
