// rsx_scatter2.cuh -- K3, register-resident form of the stable 8-bit-digit scatter pass.
//
// Same algorithm and the same output as scatter_kernel (rsx_scatter.cuh; radix_sort.hpp:83-88),
// different data movement inside the SM.  scatter_kernel parks every tile in a shared-memory
// staging buffer (TMA bulk copy) and reads each record from it twice; at B200's HBM-to-SM ratio
// that kernel is bound by the shared-memory / LSU data pipe (ncu: 81 % of peak with DRAM at
// 36 %), and the staging buffer doubles the shared memory per CTA, which caps the SM at two CTAs
// (u32) or one (u64).  Here
//   * the tile is loaded straight into REGISTERS with coalesced streaming loads (warp-striped:
//     item i of lane l is record warp*ITEMS*32 + i*32 + l), and the loads of the NEXT tile are
//     issued right before the current tile's write-out, so they are in flight while the sorted
//     tile drains to global memory -- the register file is the prefetch buffer;
//   * a record is touched in shared memory exactly twice: the scatter into its tile-sorted slot
//     and the linear read of the write-out;
//   * ranking only counts; once the digit scan has turned the warp counters into slot bases, the
//     placement sweep takes each record's slot with the ticket atomic itself (same sweep order,
//     hence the same stable order): 2 ATOMS per record and no rank registers, which leaves the
//     register file to the tile;
//   * shared memory per CTA is one sorted tile + the warp counters, so more CTAs (or larger
//     tiles) fit per SM and the barrier / look-back bubbles of one CTA are filled by another.
// Ranking is the one-instruction ticket (rank = atomicAdd(&warp_counter[digit], 1), see
// rsx_scatter.cuh) with the previous tile's hot digit ranked by a vote; when the per-device probe
// rejects ticket ranking the library runs scatter_kernel's ballot path instead.
#pragma once

#include "rsx_scatter.cuh"

namespace rsx {

// Predicated shared-memory ticket: lanes with skip == true keep `r` (their vote-derived rank).
// One predicated ATOMS instead of a divergent branch per item.
__device__ __forceinline__ uint32_t ticket_unless(uint32_t *addr, bool skip, uint32_t r) {
	asm volatile("{\n"
	             ".reg .pred q;\n"
	             "setp.eq.u32 q, %2, 0;\n"
	             "@q atom.shared.add.u32 %0, [%1], 1;\n"
	             "}\n"
	             : "+r"(r)
	             : "r"((uint32_t)__cvta_generic_to_shared(addr)), "r"((uint32_t)skip)
	             : "memory");
	return r;
}
__device__ __forceinline__ void count_unless(uint32_t *addr, bool skip) {
	asm volatile("{\n"
	             ".reg .pred q;\n"
	             "setp.eq.u32 q, %1, 0;\n"
	             "@q red.shared.add.u32 [%0], 1;\n"
	             "}\n" ::"r"((uint32_t)__cvta_generic_to_shared(addr)), "r"((uint32_t)skip)
	             : "memory");
}

template <int ES, int PL, class Cfg> struct Scatter2Smem {
	static constexpr int kTile = Cfg::kThreads * Cfg::kItems;
	static constexpr int kWarps = Cfg::kThreads / 32;
	static constexpr size_t kRecBytes = (size_t)kTile * ES;
	static constexpr size_t kPlBytes = (size_t)kTile * PL;
	// layout: [sorted rec | sorted pl | warp counters | gadj | look-back partner partials | misc]
	static constexpr size_t kOffPl = (kRecBytes + 15) / 16 * 16;
	static constexpr size_t kOffWh = (kOffPl + kPlBytes + 15) / 16 * 16;
	static constexpr size_t kOffAdj = kOffWh + (size_t)kWarps * kBins * 4;
	static constexpr size_t kOffLb = kOffAdj + (size_t)kBins * 8;
	static constexpr size_t kOffMisc = kOffLb + (size_t)kBins * 12;
	static constexpr size_t kBytes = kOffMisc + 96;
};

// ---- footprints (record + payload bytes) that run the register-resident kernel ---------------
// A single-GPU, ticket-ranked pass of footprint (ES, PL) runs this kernel with the tile Cfg2<ES, PL>
// where PreferV2<ES, PL> holds, and scatter_kernel otherwise: flipped per footprint by measurement
// (profiles/r2_variants.md).  Every other footprint measured slower than the staging kernel
// (tools/footprints.py).
template <int ES, int PL> struct PreferV2 { static constexpr bool value = false; };
// 8-byte records without a payload lane (u64 / i64 / f64 keys, {u32 key, u32 payload} records):
// 256 threads x 36 records, two CTAs per SM -- 3.95 ms per pass of 1 B u64 keys (4.01 ms at 32
// records per thread) against 4.22 ms for the staging kernel, which has room for only one CTA per SM.
template <> struct PreferV2<8, 0> {
	static constexpr bool value = true;
	using Cfg = CfgT<256, 36, 2, 8>;
};
// u32 keys + u32 index lane (radix_sort_rank on 32-bit keys), 256 threads x 32 records: 18.6 vs
// 19.8 ms per 1 B-key rank sort.
template <> struct PreferV2<4, 4> {
	static constexpr bool value = true;
	using Cfg = CfgT<256, 32, 2, 8>;
};
template <int ES, int PL> using Cfg2 = typename PreferV2<ES, PL>::Cfg;

// Streaming load: every record is read exactly once per pass.
template <typename R> __device__ __forceinline__ R ld_stream(const R *p) { return __ldcs(p); }

template <int ES, int PL, int DM, typename OffT, class Cfg>
__global__ void __launch_bounds__(Cfg::kThreads, Cfg::kMinBlocks) scatter2_kernel(const ScatterParams p) {
	using R = typename Rec<ES>::type;
	using P = typename Payload<PL>::type;
	using SM = Scatter2Smem<ES, PL, Cfg>;
	using SB = StatusBits<OffT>;
	constexpr int THREADS = Cfg::kThreads, ITEMS = Cfg::kItems;
	constexpr int TILE = SM::kTile;
	constexpr int WARPS = SM::kWarps;
	constexpr int LB = Cfg::kLookback;
	constexpr int kWriteBatch = 2; // records per write-out batch (see scatter_kernel)
	constexpr uint32_t FULL = 0xFFFFFFFFu;
	static_assert(THREADS >= kBins && THREADS % 32 == 0, "one digit thread per bin: the digit scan synchronises 256 threads");

	extern __shared__ __align__(128) unsigned char smem[];
	R *s_rec = reinterpret_cast<R *>(smem);
	P *s_pl = reinterpret_cast<P *>(smem + SM::kOffPl);
	uint32_t *s_wh = reinterpret_cast<uint32_t *>(smem + SM::kOffWh);
	OffT *s_gadj = reinterpret_cast<OffT *>(smem + SM::kOffAdj);
	OffT *s_lbsum = reinterpret_cast<OffT *>(smem + SM::kOffLb);
	uint32_t *s_lbst = reinterpret_cast<uint32_t *>(smem + SM::kOffLb + (size_t)kBins * 8);
	uint32_t *s_misc = reinterpret_cast<uint32_t *>(smem + SM::kOffMisc);
	// s_misc[0] = next tile ticket, [1..8] = warp totals of the digit scan, [9] = hot digit,
	// [10..17] = per-warp maxima of (count << 8 | digit)

	// ---- pass table (device-side column skipping, radix_sort.hpp:60-70) ----
	uint32_t ord = 0;
	bool last = true;
	if (p.ctl != nullptr) {
		const uint32_t early = p.ctl->early_exit, live = p.ctl->live_mask;
		if (early || !((live >> p.col) & 1u))
			return;
		ord = p.ctl->ordinal[p.col];
		last = ord + 1 == p.ctl->ncols;
	}
	const R *__restrict__ in = static_cast<const R *>(ord == 0 ? p.pb.rec_first : p.pb.rec_buf[(ord - 1) & 1]);
	R *__restrict__ out = static_cast<R *>(p.pb.rec_buf[ord & 1]);
	const P *__restrict__ pin = static_cast<const P *>(ord == 0 ? p.pb.pl_first : p.pb.pl_buf[(ord - 1) & 1]);
	P *__restrict__ pout = static_cast<P *>(p.pb.pl_buf[ord & 1]);
	const bool synth = PL != 0 && ord == 0 && p.pb.synth_index;
	const bool write_rec = !(last && p.pb.skip_last_rec);
	const bool load_pl = PL != 0 && !synth;

	const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
	const uint32_t lt = lanemask_lt();
	const DigitDesc dd = p.dd;
	uint32_t *wh = s_wh + warp * kBins;
	OffT *status = static_cast<OffT *>(p.status);
	const R pad = make_pad<ES>(p.pad_rec);
	const uint32_t full_tiles = (uint32_t)(p.n / TILE); // tiles [0, full_tiles) are complete
	const uint32_t t0 = warp * (ITEMS * 32) + lane;     // this thread's first record inside a tile

	R key[ITEMS];
	P pay[PL != 0 ? ITEMS : 1];
	auto load_tile = [&](uint32_t t) {
		if (t >= p.num_tiles)
			return;
		const size_t base = (size_t)t * TILE;
		if (t < full_tiles) {
#pragma unroll
			for (int i = 0; i < ITEMS; ++i)
				key[i] = ld_stream(in + base + t0 + i * 32);
			if constexpr (PL != 0) {
				if (load_pl) {
#pragma unroll
					for (int i = 0; i < ITEMS; ++i)
						pay[i] = ld_stream(pin + base + t0 + i * 32);
				}
			}
		} else { // the partial last tile: padding sorts last
			const uint32_t valid = (uint32_t)(p.n - base);
#pragma unroll
			for (int i = 0; i < ITEMS; ++i) {
				const uint32_t t_ = t0 + i * 32;
				key[i] = t_ < valid ? ld_stream(in + base + t_) : pad;
				if constexpr (PL != 0)
					pay[i] = (load_pl && t_ < valid) ? ld_stream(pin + base + t_) : (P)0;
			}
		}
	};

	// Tile tickets: claimed as late as possible (right before the previous tile's write-out), see
	// rsx_scatter.cuh -- every later tile's look-back waits for this tile's aggregate.
	if (tid == 0) {
		s_misc[0] = atomicAdd(p.ticket, 1u);
		s_misc[9] = 0; // first tile: digit 0 as the hot-digit guess
	}
	__syncthreads();
	uint32_t tile = s_misc[0];
	load_tile(tile);

	while (tile < p.num_tiles) {
		const size_t base = (size_t)tile * TILE;
		const bool full = tile < full_tiles;
		const uint32_t valid = full ? (uint32_t)TILE : (uint32_t)(p.n - base);

		{
			uint4 *z = reinterpret_cast<uint4 *>(wh);
			z[lane] = make_uint4(0, 0, 0, 0);
			z[lane + 32] = make_uint4(0, 0, 0, 0);
		}
		__syncwarp();

		// ---- 1. count per warp and digit; the previous tile's hot digit is counted by a vote ----
		uint32_t hotcnt = 0;
		const uint32_t hot = s_misc[9];
		{
#pragma unroll
			for (int i = 0; i < ITEMS; ++i) {
				const uint32_t d = tile_digit<ES, DM>(p, key[i], dd);
				const bool is_hot = d == hot;
				const uint32_t m = __ballot_sync(FULL, is_hot);
				count_unless(&wh[d], is_hot);
				hotcnt += __popc(m);
			}
			if (lane == 0)
				wh[hot] = hotcnt; // no atomic touched this counter
		}
		__syncthreads(); // (A) all warp counters final

		// ---- 2. digit threads: warp prefixes, tile scan, publish the aggregate ----
		uint32_t tcount = 0, tstart = 0;
		if (tid < kBins) {
#pragma unroll
			for (int w = 0; w < WARPS; ++w)
				tcount += s_wh[w * kBins + tid];
			// tail padding sorts last (after every real record of the last digit): not part of the aggregate
			const uint32_t agg = (!full && tid == (uint32_t)kBins - 1) ? tcount - ((uint32_t)TILE - valid) : tcount;
			st_status(&status[(size_t)tile * kBins + tid], (OffT)((tile == 0 ? SB::kPfx : SB::kAgg) | (OffT)agg));
			uint32_t x = tcount;
#pragma unroll
			for (int o = 1; o < 32; o <<= 1) {
				const uint32_t y = __shfl_up_sync(FULL, x, o);
				if (lane >= o)
					x += y;
			}
			const uint32_t wmax = __reduce_max_sync(FULL, (tcount << 8) | tid); // hot digit for the next tile
			if (lane == 31) {
				s_misc[1 + warp] = x;
				s_misc[10 + warp] = wmax;
			}
			asm volatile("bar.sync 1, 256;" ::: "memory");
			uint32_t wbase = 0, hmax = 0;
#pragma unroll
			for (int w = 0; w < 8; ++w) {
				wbase += (w < (int)warp) ? s_misc[1 + w] : 0u;
				hmax = max(hmax, s_misc[10 + w]);
			}
			if (tid == 0)
				s_misc[9] = hmax & 0xFFu;
			tstart = wbase + x - tcount;
			uint32_t run = tstart; // second sweep: counts -> slot bases (no register array: the keys live there)
#pragma unroll
			for (int w = 0; w < WARPS; ++w) {
				const uint32_t c = s_wh[w * kBins + tid];
				s_wh[w * kBins + tid] = run;
				run += c;
			}
			tcount = agg;
		}
		__syncthreads(); // (C)

		// ---- 3. records / payloads to their tile-sorted slot: stable rank inside the warp (items
		//      ascending, lanes ascending) in the same sweep order as the count, so the ticket
		//      returns the slot itself ----
		uint32_t hotpos = wh[hot];
		__syncwarp();
#pragma unroll
		for (int i = 0; i < ITEMS; ++i) {
			const uint32_t d = tile_digit<ES, DM>(p, key[i], dd);
			const bool is_hot = d == hot;
			const uint32_t m = __ballot_sync(FULL, is_hot);
			const uint32_t pos = ticket_unless(&wh[d], is_hot, hotpos + __popc(m & lt));
			hotpos += __popc(m);
			s_rec[pos] = key[i];
			if constexpr (PL != 0)
				s_pl[pos] = synth ? (P)(base + t0 + i * 32) : pay[i];
		}

		// ---- 4. decoupled look-back, one chain per digit; the first round is split over two
		//      threads per digit so that 2*LB predecessors cost one L2 round trip ----
		{
			constexpr bool kPair = THREADS >= 2 * kBins;
			const uint32_t dgt = tid & (kBins - 1), half = tid / kBins;
			OffT part = 0;
			uint32_t st = 0, used = 0; // st: 0 = only aggregates so far, 1 = reached a prefix, 2 = hit an unpublished word
			if (half < (kPair ? 2u : 1u)) {
				const int q = (int)tile - 1 - (int)half * LB;
				OffT w[LB];
#pragma unroll
				for (int j = 0; j < LB; ++j)
					w[j] = (q - j >= 0) ? ld_status(&status[(size_t)(q - j) * kBins + dgt]) : (OffT)SB::kPfx;
#pragma unroll
				for (int j = 0; j < LB; ++j) {
					if (st == 0) {
						if ((w[j] & ~SB::kMask) == 0) {
							st = 2;
						} else {
							part += w[j] & SB::kMask;
							++used;
							if (w[j] & SB::kPfx)
								st = 1;
						}
					}
				}
			}
			if constexpr (kPair) {
				if (half == 1) {
					s_lbsum[dgt] = part;
					s_lbst[dgt] = st;
					asm volatile("bar.arrive %0, 64;" ::"r"(2 + (warp & 7)) : "memory");
				}
			}
			if (half == 0) {
				OffT excl = part;
				bool done = st == 1;
				int q = (int)tile - 1 - (int)used;
				if constexpr (kPair) {
					asm volatile("bar.sync %0, 64;" ::"r"(2 + warp) : "memory");
					if (st == 0) { // own window was all aggregates: splice the partner's window
						const uint32_t pst = s_lbst[dgt];
						if (pst != 2) {
							excl += s_lbsum[dgt];
							q -= LB;
							done = pst == 1;
						}
					}
				}
				while (!done) { // rare: long chains and unpublished predecessors
					OffT w[LB];
#pragma unroll
					for (int j = 0; j < LB; ++j)
						w[j] = (q - j >= 0) ? ld_status(&status[(size_t)(q - j) * kBins + dgt]) : (OffT)SB::kPfx;
#pragma unroll
					for (int j = 0; j < LB; ++j) {
						if (!done) {
							OffT v = w[j];
							while ((v & ~SB::kMask) == 0) { // not published yet: poll this one word, politely
								__nanosleep(40);
								v = ld_status(&status[(size_t)(q - j) * kBins + dgt]);
							}
							excl += v & SB::kMask;
							done = (v & SB::kPfx) != 0;
						}
					}
					q -= LB;
				}
				if (tile != 0)
					st_status(&status[(size_t)tile * kBins + dgt], (OffT)(SB::kPfx | (excl + (OffT)tcount)));
				s_gadj[dgt] = (OffT)p.offs[dgt] + excl - (OffT)tstart;
			}
		}
		if (tid == 0) // next ticket: claimed as late as possible
			s_misc[0] = atomicAdd(p.ticket, 1u);
		__syncthreads(); // (D) sorted tile + gadj complete
		const uint32_t next_tile = s_misc[0];

		// ---- 5. the next tile's loads go out now and land while this tile is being stored ----
		load_tile(next_tile);

		// ---- 6. coalesced per-bucket stores ----
		if (full) {
			// batches: loads, then bucket-offset lookups, then stores (see scatter_kernel)
			auto write_full = [&](auto wr_tag) {
				constexpr bool WR = decltype(wr_tag)::value;
				constexpr int U = kWriteBatch;
#pragma unroll 1
				for (int i0 = 0; i0 < ITEMS; i0 += U) {
					R r[U];
					OffT g[U];
#pragma unroll
					for (int u = 0; u < U; ++u)
						if (i0 + u < ITEMS)
							r[u] = s_rec[tid + (i0 + u) * THREADS];
#pragma unroll
					for (int u = 0; u < U; ++u)
						if (i0 + u < ITEMS)
							g[u] = s_gadj[tile_digit<ES, DM>(p, r[u], dd)] + (OffT)(tid + (i0 + u) * THREADS);
#pragma unroll
					for (int u = 0; u < U; ++u)
						if (i0 + u < ITEMS) {
							if constexpr (ES + PL <= 4) {
								if constexpr (WR)
									__stcs(out + g[u], r[u]);
							} else {
								if constexpr (WR)
									out[g[u]] = r[u];
								if constexpr (PL != 0)
									pout[g[u]] = s_pl[tid + (i0 + u) * THREADS];
							}
						}
				}
			};
			if (write_rec)
				write_full(std::true_type{});
			else if (PL != 0)
				write_full(std::false_type{});
		} else {
			for (uint32_t s = tid; s < valid; s += THREADS) {
				const R r = s_rec[s];
				const OffT g = s_gadj[tile_digit<ES, DM>(p, r, dd)] + (OffT)s;
				if (write_rec)
					out[g] = r;
				if constexpr (PL != 0)
					pout[g] = s_pl[s];
			}
		}
		tile = next_tile;
	}
}

template <int ES, int PL, int DM, typename OffT, class Cfg>
cudaError_t launch_scatter2_c(const ScatterParams &sp, int num_sms, cudaStream_t st) {
	using SM = Scatter2Smem<ES, PL, Cfg>;
	auto kern = scatter2_kernel<ES, PL, DM, OffT, Cfg>;
	static int occ_cache[64] = {}; // per device
	int dev = 0;
	cudaGetDevice(&dev);
	int &ctas_per_sm = occ_cache[dev & 63];
	if (ctas_per_sm == 0) {
		cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM::kBytes);
		if (e != cudaSuccess)
			return e;
		int occ = 0;
		e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, Cfg::kThreads, SM::kBytes);
		if (e != cudaSuccess)
			return e;
		ctas_per_sm = occ > 0 ? occ : 1;
	}
	ScatterParams q = sp;
	q.num_tiles = (uint32_t)((sp.n + SM::kTile - 1) / SM::kTile);
	uint32_t grid = (uint32_t)num_sms * (uint32_t)ctas_per_sm;
	if (grid > q.num_tiles)
		grid = q.num_tiles;
	kern<<<grid, Cfg::kThreads, SM::kBytes, st>>>(q);
	count_launch();
	return cudaGetLastError();
}

} // namespace rsx
