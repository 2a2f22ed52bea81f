// rsx_scatter.cuh -- K3: one stable 8-bit-digit scatter pass ("onesweep" style).
//
// Replaces the reference's sort loop for one live column (radix_sort.hpp:83-88):
//     for j in 0..n: k = src[j]; dst = offsets[digit(kf(k))]++; aux[dst] = k
// The serial `offsets[..]++` is what makes the reference stable; here the same destination
// index is computed in parallel as
//     dst = column_offset[d]                 (exclusive scan of the global histogram, K2)
//         + #records with digit d in earlier tiles      (decoupled look-back, one chain per digit)
//         + #records with digit d earlier in this tile  (stable rank in the warp + cross-warp prefix)
// which is exactly the value the reference's counter would have had, so the output is
// bit-identical, including the order of equal keys (stability) and of payloads.
//
// Per pass the algorithmic HBM traffic is n * (record + payload) read + the same written;
// the look-back state adds 256 words written + ~256 read per tile (L2 resident).
//
// Tile pipeline (persistent CTAs, tiles handed out by an atomic ticket so that a tile's
// predecessors are always owned by running CTAs -> the look-back cannot deadlock):
//   1. the tile sits in a shared staging buffer, put there by a TMA bulk copy issued while the
//      previous tile was being stored (plain loads for unaligned input and the partial last tile);
//      warp-striped ownership; the KDF is folded into digit_of()
//   2. per warp, per item: stable rank of the record among the warp's records with the same
//      digit.  Two implementations (template RANK):
//        RANK_TICKET  rank = atomicAdd(&warp_counter[digit], 1): ONE shared-memory instruction
//                     per key.  Stable because this hardware hands out same-address tickets of
//                     one warp instruction in ascending lane order and applies a warp's
//                     back-to-back atomics in program order -- verified per device at first use
//                     by ticket_probe_kernel (and offline by tools/probe_atoms.cu); if the probe
//                     ever disagreed the library would use RANK_BALLOT.
//        RANK_BALLOT  8 votes -> peer mask; the group leader bumps the warp counter and
//                     broadcasts the old value.  Provably stable, ~2.5x cheaper on B200 than
//                     __match_any_sync on 8 random bits (tools/yardstick.cu: 24 vs 60 clk/SM per
//                     32 keys), but still above the ~13 clk/SM budget of a 70 %-of-peak pass.
//   3. threads 0..255 (one per digit): sum / prefix the warp counters, scan the 256 tile
//      counts, publish the tile aggregate, later walk back over predecessor tiles
//   4. records (and payloads) are written to shared memory at their tile-sorted position
//   5. thread t stores shared slot t, t+T, ...: consecutive threads hit consecutive addresses
//      inside each digit bucket, so global writes coalesce per bucket
#pragma once

#include "rsx_device.cuh"
#include <type_traits>

namespace rsx {

constexpr int kMaxSplit = 15; // up to 16 destinations for key-range routing

struct ScatterParams {
	PassBuffers pb;
	size_t n;
	uint32_t num_tiles;
	uint32_t col;
	DigitDesc dd;
	const unsigned long long *offs; // this column's exclusive scan (256 entries)
	const Ctl *ctl;                 // nullptr: forced pass
	void *status;                   // OffT[num_tiles][256], zeroed by the host (one buffer per column)
	unsigned int *ticket;
	ulonglong2 pad_rec;             // record whose derived key is all ones (tail padding)
	unsigned long long *dbg;        // RSX_PHASE_TIMING builds only: per-phase cycle accumulators
	// Fused partition + exchange (multi-GPU): when dest_base is non-null, bucket d belongs to
	// destination owner[d] (contiguous bucket ranges) and every tile appends ONE contiguous run
	// per destination at dest_base[D] -- typically a peer GPU's receive buffer mapped over NVLink.
	// Inside a destination the order is (tile, bucket, position): stable, not grouped by bucket
	// across tiles (the receiver's LSD sort does not need that).  Records only (no payload).
	const unsigned long long *dest_base; // device memory, one byte address per destination
	const unsigned char *owner;          // device memory, 256 entries
	uint32_t ndest;
	// Keys-only records (the whole record is the key): equal records are indistinguishable, so the
	// order INSIDE one (tile, destination) run is free -- its 16-byte-aligned body can then leave as
	// ONE TMA bulk store (shared -> peer memory) instead of LSU stores.
	uint32_t unordered_runs;
	// Append mode (keys-only multi-GPU exchange without a routing histogram): every destination has
	// an append cursor in ITS memory; a tile reserves room for its run with one system-scope atomic
	// and needs neither the exact per-source offsets nor a look-back.  dest_cursor[k] = address of
	// destination k's cursor (records), dest_capacity[k] = records it can take; a run that would not
	// fit is dropped and *overflow set (the caller retries with more room; src is only read).
	const unsigned long long *dest_cursor;
	const unsigned long long *dest_capacity;
	unsigned int *overflow;
	// Key-range routing (DIGIT_SPLIT): the "digit" of a record is the number of splitters that are
	// <= its derived key, i.e. its destination among nsplit + 1 key ranges.
	KeyDesc kd;
	uint32_t nsplit;
	unsigned long long split[kMaxSplit];
};

enum { DIGIT_PLAIN = 0, DIGIT_FLOAT = 1, DIGIT_SPLIT = 2 };

template <int ES, int DM>
__device__ __forceinline__ uint32_t tile_digit(const ScatterParams &p, const typename Rec<ES>::type &r, const DigitDesc &dd) {
	if constexpr (DM == DIGIT_SPLIT) {
		const unsigned long long k = derive_key(key_word<ES>(r, p.kd.word_sel), p.kd);
		uint32_t d = 0;
		for (uint32_t j = 0; j < p.nsplit; ++j)
			d += k >= p.split[j];
		return d;
	} else {
		return digit_of<ES, DM == DIGIT_FLOAT>(r, dd);
	}
}

#ifdef RSX_PHASE_TIMING
#define RSX_T(k)                                                    \
	do {                                                            \
		if (tid == 0) {                                             \
			const long long now_ = clock64();                       \
			dbg_acc[k] += (unsigned long long)(now_ - dbg_last);    \
			dbg_last = now_;                                        \
		}                                                           \
	} while (0)
#else
#define RSX_T(k) do { } while (0)
#endif

// RANK_TICKET or RANK_BALLOT for the current device (probe result or rsx_set_option override).
int rank_mode();

template <typename OffT> struct StatusBits;
template <> struct StatusBits<uint32_t> {
	static constexpr uint32_t kAgg = 1u << 30, kPfx = 2u << 30, kMask = (1u << 30) - 1u;
};
template <> struct StatusBits<unsigned long long> {
	static constexpr unsigned long long kAgg = 1ULL << 62, kPfx = 2ULL << 62, kMask = (1ULL << 62) - 1ULL;
};

// Look-back status words are self-contained messages (flag + value in one word): relaxed
// device-scope accesses suffice, no fences.
__device__ __forceinline__ uint32_t ld_status(const uint32_t *p) {
	uint32_t v;
	asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
	return v;
}
__device__ __forceinline__ unsigned long long ld_status(const unsigned long long *p) {
	unsigned long long v;
	asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
	return v;
}
__device__ __forceinline__ void st_status(uint32_t *p, uint32_t v) {
	asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_status(unsigned long long *p, unsigned long long v) {
	asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// ---- TMA 1-D bulk copy (global -> shared) completing on an mbarrier -------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
	asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, unsigned long long *bar) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
	             ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// TMA 1-D bulk store (shared -> global, possibly peer memory over NVLink), bulk-group completion
__device__ __forceinline__ void bulk_s2g(unsigned long long dst, const void *src, uint32_t bytes) {
	asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
	asm volatile("{\n"
	             ".reg .pred P1;\n"
	             "LAB_WAIT:\n"
	             "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
	             "@P1 bra DONE;\n"
	             "bra LAB_WAIT;\n"
	             "DONE:\n"
	             "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

template <int ES> __device__ __forceinline__ typename Rec<ES>::type make_pad(const ulonglong2 &p) {
	if constexpr (ES == 16)
		return p;
	else
		return (typename Rec<ES>::type)p.x;
}

// Tile geometry per (record, payload) footprint: threads, records per thread, minimum CTAs per SM
// (launch bounds) and look-back window (status words per digit thread and round).
template <int T, int I, int MB, int LBK> struct CfgT {
	static constexpr int kThreads = T, kItems = I, kMinBlocks = MB, kLookback = LBK;
};

// Defaults from the B200 sweeps recorded in profiles/r1_variants.md.  The pass is bound by the
// shared-memory/LSU data pipe and by per-tile fixed costs (barriers, look-back), so the tile is as
// large as shared memory allows: 4-byte footprints run 512 threads x 22 records with two CTAs per
// SM (2 x 111.7 KB); wider footprints run ONE 512-thread CTA per SM with 192 / footprint records
// per thread (8 bytes: 512 x 24, 96 KB staging + 96 KB sorted tile) -- fewer, fatter threads beat
// 1024 x 11 by 9 % on u64 keys (16 instead of 32 warp histograms to zero, sum and rewrite per tile).
// Look-back window: every tile reads 2 x LB x 256 status words in its first round (32 KB at LB 16
// against a 45 KB tile of 4-byte keys); 8 words per thread cost a few more serial rounds but 7 % less
// time per u32 pass (LB 4 / 6 / 8 / 12 / 16: 2.59 / 2.58 / 2.59 / 2.67 / 2.79 ms).
template <int ES, int PL> struct ScatterCfg
	: CfgT<512, ((ES + PL <= 4) ? 22 : 192 / (ES + PL)), ((ES + PL <= 4) ? 2 : 1), 8> {};
// The fused partition + exchange passes (multi-GPU) carry a 4 KB destination table in shared
// memory and keep the geometry they were tuned and measured with.  It is the smallest tile of any
// default kernel, so it also sizes the look-back state (scatter_geometry()).
template <int ES, int PL> struct FusedCfg
	: CfgT<((ES + PL > 4 && ES + PL <= 8) ? 1024 : 512),
	       ((ES + PL <= 4) ? 20 : (ES + PL <= 8) ? 10 : (ES + PL <= 16) ? 8 : 4), ((ES + PL <= 4) ? 2 : 1),
	       ((ES + PL <= 4) ? 8 : 16)> {};

template <int ES, int PL, class Cfg, bool FUSED = true> struct ScatterSmem {
	static constexpr int kTile = Cfg::kThreads * Cfg::kItems;
	static constexpr int kWarps = Cfg::kThreads / 32;
	static constexpr size_t kRecBytes = (size_t)kTile * ES;
	static constexpr size_t kPlBytes = (size_t)kTile * PL;
	static constexpr size_t kWhBytes = (size_t)kWarps * kBins * 4;
	static constexpr size_t kAdjBytes = (size_t)kBins * 8;
	// layout: [stage rec | stage pl | sorted rec | sorted pl | warp counters | gadj | misc]
	static constexpr size_t kOffSorted = kRecBytes + kPlBytes; // after the staging buffer
	static constexpr size_t kSortedSlack = 0; // fused mode may read one 16-byte vector past the sorted buffer: that is the counter area, harmless
	static constexpr size_t kOffWh = kOffSorted + kRecBytes + kSortedSlack + kPlBytes;
	static constexpr size_t kOffAdj = kOffWh + kWhBytes;
	static constexpr size_t kOffLb = kOffAdj + kAdjBytes; // look-back partner partials: 256 x (8 + 4) bytes
	static constexpr size_t kOffDst = kOffLb + (size_t)kBins * 12; // fused mode: per-destination offsets
	static constexpr size_t kOffMisc = kOffDst + (FUSED ? (size_t)kBins * 16 : 0); // single-GPU passes have no destination table
	static constexpr size_t kBytes = kOffMisc + 96;
};

enum { RANK_TICKET = 0, RANK_BALLOT = 1 };

template <int ES, int PL, int DM, bool FUSED, typename OffT, int RANK, class Cfg>
__global__ void __launch_bounds__(Cfg::kThreads, Cfg::kMinBlocks) scatter_kernel(const ScatterParams p) {
	using R = typename Rec<ES>::type;
	using P = typename Payload<PL>::type;
	using SM = ScatterSmem<ES, PL, Cfg, FUSED>;
	using SB = StatusBits<OffT>;
	constexpr int THREADS = Cfg::kThreads, ITEMS = Cfg::kItems;
	constexpr int TILE = SM::kTile;
	constexpr int WARPS = SM::kWarps;
	constexpr int LB = Cfg::kLookback;
	constexpr int kWriteBatch = 2; // records per write-out batch (see step 5)
	constexpr uint32_t FULL = 0xFFFFFFFFu;
	static_assert(THREADS >= kBins && THREADS % 32 == 0, "one digit thread per bin: the digit scan synchronises 256 threads");

	extern __shared__ __align__(128) unsigned char smem[];
	R *s_stage = reinterpret_cast<R *>(smem);
	P *s_stage_pl = reinterpret_cast<P *>(smem + SM::kRecBytes);
	R *s_rec = reinterpret_cast<R *>(smem + SM::kOffSorted);
	P *s_pl = reinterpret_cast<P *>(smem + SM::kOffSorted + SM::kRecBytes + SM::kSortedSlack);
	uint32_t *s_wh = reinterpret_cast<uint32_t *>(smem + SM::kOffWh);
	OffT *s_gadj = reinterpret_cast<OffT *>(smem + SM::kOffAdj);
	unsigned long long *s_gptr = reinterpret_cast<unsigned long long *>(smem + SM::kOffAdj); // fused mode view
	unsigned long long *s_dexcl = reinterpret_cast<unsigned long long *>(smem + SM::kOffDst); // fused mode
	uint32_t *s_dstart = reinterpret_cast<uint32_t *>(smem + SM::kOffDst + (size_t)kBins * 8);
	uint32_t *s_dcount = reinterpret_cast<uint32_t *>(smem + SM::kOffDst + (size_t)kBins * 12);
	OffT *s_lbsum = reinterpret_cast<OffT *>(smem + SM::kOffLb);
	uint32_t *s_lbst = reinterpret_cast<uint32_t *>(smem + SM::kOffLb + (size_t)kBins * 8);
	uint32_t *s_misc = reinterpret_cast<uint32_t *>(smem + SM::kOffMisc);
	unsigned long long *s_bar = reinterpret_cast<unsigned long long *>(smem + SM::kOffMisc + 80);
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
	const bool stage_pl = PL != 0 && !synth;
	// TMA needs 16-byte aligned global addresses; tiles are multiples of 16 bytes
	const bool can_stage = (reinterpret_cast<uintptr_t>(in) & 15) == 0 &&
	                       (!stage_pl || (reinterpret_cast<uintptr_t>(pin) & 15) == 0);

	const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
	const uint32_t lt = lanemask_lt();
	const DigitDesc dd = p.dd;
	uint32_t *wh = s_wh + warp * kBins;
	OffT *status = static_cast<OffT *>(p.status);
	const R pad = make_pad<ES>(p.pad_rec);
	const uint32_t full_tiles = (uint32_t)(p.n / TILE); // tiles [0, full_tiles) are complete
	const uint32_t my_owner = (FUSED && tid < kBins) ? p.owner[tid] : 0u;

	auto prefetch = [&](uint32_t t) { // one thread
		const size_t base = (size_t)t * TILE;
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
		mbar_expect_tx(s_bar, (uint32_t)(SM::kRecBytes + (stage_pl ? SM::kPlBytes : 0)));
		bulk_g2s(s_stage, in + base, (uint32_t)SM::kRecBytes, s_bar);
		if constexpr (PL != 0) {
			if (stage_pl)
				bulk_g2s(s_stage_pl, pin + base, (uint32_t)SM::kPlBytes, s_bar);
		}
	};

	// Tile tickets.  A ticket is claimed as late as possible -- right before the previous tile's
	// write-out -- because every later tile's look-back has to wait for this tile's aggregate:
	// claiming earlier (e.g. to prefetch sooner) makes successors queue up behind an idle claim.
	if (tid == 0) {
		mbar_init(s_bar, 1);
		const uint32_t t = atomicAdd(p.ticket, 1u);
		s_misc[0] = t;
		s_misc[9] = 0; // first tile: digit 0 as the hot-digit guess
		if (can_stage && t < full_tiles)
			prefetch(t);
	}
	__syncthreads();
	uint32_t tile = s_misc[0];
	uint32_t phase = 0;
#ifdef RSX_PHASE_TIMING
	unsigned long long dbg_acc[12] = {};
	long long dbg_last = clock64();
#endif

	while (tile < p.num_tiles) {
		RSX_T(9);
		const size_t base = (size_t)tile * TILE;
		const bool full = tile < full_tiles;
		const uint32_t valid = full ? (uint32_t)TILE : (uint32_t)(p.n - base);
		const bool staged = can_stage && full;

		// ---- 1. tile -> staging buffer (warp-striped ownership: item i of lane l is record
		//         warp*ITEMS*32 + i*32 + l).  Normally the TMA prefetch already put it there. ----
		const uint32_t t0 = warp * (ITEMS * 32) + lane;
		{
			uint4 *z = reinterpret_cast<uint4 *>(wh);
			z[lane] = make_uint4(0, 0, 0, 0);
			z[lane + 32] = make_uint4(0, 0, 0, 0);

		}
		if (staged) {
			mbar_wait(s_bar, phase);
			phase ^= 1u;
		} else {
			// unaligned input or the partial last tile: plain loads, parked in the same buffer
#pragma unroll
			for (int i = 0; i < ITEMS; ++i) {
				const uint32_t t = t0 + i * 32;
				s_stage[t] = (t < valid) ? __ldg(in + base + t) : pad;
				if constexpr (PL != 0) {
					if (!synth)
						s_stage_pl[t] = (t < valid) ? __ldg(pin + base + t) : (P)0;
				}
			}
		}
		__syncwarp();
		RSX_T(0);

		// ---- 2. rank inside the warp (stable: items ascending, lanes ascending) ----
		uint32_t rank[ITEMS];
		if constexpr (RANK == RANK_TICKET) {
			// The tile's most frequent digit of the previous tile ("hot") is ranked in registers:
			// one vote per item instead of up to 32 same-address atomics when a digit dominates
			// (low-entropy columns); for uniform digits it only removes a few lanes from the atomic.
			const uint32_t hot = s_misc[9];
			uint32_t hotcnt = 0;
#pragma unroll
			for (int i = 0; i < ITEMS; ++i) { // fully unrolled on purpose (partial: +8 %)
				const uint32_t d = tile_digit<ES, DM>(p, s_stage[t0 + i * 32], dd);
				const bool is_hot = d == hot;
				const uint32_t m = __ballot_sync(FULL, is_hot);
				// a branch, not a predicated atomic: 1-2 % faster on uniform digits (profiles/r2_variants.md)
				if (is_hot)
					rank[i] = hotcnt + __popc(m & lt);
				else
					rank[i] = atomicAdd(&wh[d], 1u);
				hotcnt += __popc(m);
			}
			if (lane == 0)
				wh[hot] = hotcnt; // no atomic touched this counter
		} else {
#pragma unroll
			for (int i = 0; i < ITEMS; ++i) {
				const uint32_t d = tile_digit<ES, DM>(p, s_stage[t0 + i * 32], dd);
				uint32_t peers = FULL;
#pragma unroll
				for (int b = 0; b < 8; ++b) {
					const bool bit = (d >> b) & 1u;
					const uint32_t v = __ballot_sync(FULL, bit);
					peers &= bit ? v : ~v;
				}
				const uint32_t leader = __ffs(peers) - 1;
				uint32_t old = 0;
				if (lane == leader)
					old = atomicAdd(&wh[d], (uint32_t)__popc(peers));
				old = __shfl_sync(FULL, old, leader);
				rank[i] = old + __popc(peers & lt);
			}
		}
		RSX_T(1);
		if constexpr (FUSED) {
			if (tid == 0 && p.unordered_runs)
				bulk_wait_read(); // the previous tile's bulk stores have read the sorted buffer
		}
		__syncthreads(); // (A) all warp counters final
		RSX_T(2);

		// ---- 3a. digit threads: warp prefixes, tile scan, publish aggregate ----
		constexpr bool fusedm = FUSED;
		uint32_t tcount = 0, tstart = 0;
		[[maybe_unused]] unsigned long long append_off = 0;
		if (tid < kBins) {
			uint32_t c[WARPS];
			if constexpr (FUSED) {
				// reset the per-destination accumulators: every reader of the previous tile's values
				// is past barrier (A), every adder of this tile is behind the scan's bar.sync below
				s_dexcl[tid] = 0;
				s_dcount[tid] = 0;
			}
#pragma unroll
			for (int w = 0; w < WARPS; ++w)
				c[w] = s_wh[w * kBins + tid];
#pragma unroll
			for (int w = 0; w < WARPS; ++w)
				tcount += c[w];
			// tail padding sorts last (after every real record of the last used digit): not part of the aggregate
			const uint32_t pad_digit = DM == DIGIT_SPLIT ? p.nsplit : (uint32_t)kBins - 1;
			const uint32_t agg = (!full && tid == pad_digit) ? tcount - ((uint32_t)TILE - valid) : tcount;
			bool append = false;
			if constexpr (FUSED)
				append = p.dest_cursor != nullptr;
			if (!append)
				st_status(&status[(size_t)tile * kBins + tid], (OffT)((tile == 0 ? SB::kPfx : SB::kAgg) | (OffT)agg));
			// exclusive scan of tcount over the 256 digit threads (8 warps)
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
			uint32_t run = tstart;
#pragma unroll
			for (int w = 0; w < WARPS; ++w) {
				s_wh[w * kBins + tid] = run;
				run += c[w];
			}
			tcount = agg;
			if constexpr (FUSED) {
				if (append) {
					// records per destination (a contiguous digit range, hence contiguous lanes), then
					// one system-scope atomic per destination reserves the run's place in the owner's
					// buffer; the reply travels while the tile is being placed
					const uint32_t D = my_owner;
					const uint32_t grp = __match_any_sync(FULL, D);
					uint32_t cnt = tcount;
#pragma unroll
					for (int o = 1; o < 32; o <<= 1) {
						const uint32_t cnt2 = __shfl_down_sync(FULL, cnt, o);
						if (lane + o < 32 && ((grp >> (lane + o)) & 1u))
							cnt += cnt2;
					}
					if (lane == (uint32_t)__ffs(grp) - 1)
						atomicAdd(&s_dcount[D], cnt);
					if (tid == 0 || p.owner[tid - 1] != D)
						s_dstart[D] = tstart;
					asm volatile("bar.sync 1, 256;" ::: "memory");
					if (tid < p.ndest) {
						const uint32_t mine = s_dcount[tid];
						unsigned long long off = 0;
						if (mine)
							off = atomicAdd_system(reinterpret_cast<unsigned long long *>(p.dest_cursor[tid]), (unsigned long long)mine);
						append_off = off;
					}
				}
			}
		}
		RSX_T(3);

		__syncthreads(); // (C)
		RSX_T(4);

		// ---- 4. records / payloads to their tile-sorted slot.  (A lambda called once: written
		//      inline, the compiler hoists the warp-counter address differently and allocates
		//      registers differently for the whole kernel.) ----
		auto place = [&]() {
#pragma unroll
			for (int i = 0; i < ITEMS; ++i) { // fully unrolled on purpose: partial unrolling costs 10 %
				const R r = s_stage[t0 + i * 32];
				const uint32_t pos = wh[tile_digit<ES, DM>(p, r, dd)] + rank[i];
				s_rec[pos] = r;
				if constexpr (PL != 0)
					s_pl[pos] = synth ? (P)(base + t0 + i * 32) : s_stage_pl[t0 + i * 32];
			}
		};
		place();
		RSX_T(5);

		// ---- 3b. decoupled look-back, one chain per digit.  The first round is split over two
		//      threads per digit (warp w and warp w+8), so 2*LB predecessors cost one L2 round trip;
		//      whatever is still unresolved afterwards is walked serially by the digit thread. ----
		constexpr bool kPair = THREADS >= 2 * kBins;
		const uint32_t dgt = tid & (kBins - 1), half = tid / kBins;
		bool append_mode = false;
		if constexpr (FUSED)
			append_mode = p.dest_cursor != nullptr;
		if (append_mode) {
			// append mode: no look-back at all -- the reservation made after the digit scan is the
			// run's offset in the destination
			if (tid < p.ndest) {
				const uint32_t mine = s_dcount[tid];
				if (mine && append_off + mine > p.dest_capacity[tid]) {
					*p.overflow = 1u; // does not fit: drop the run, the caller retries with more room
					s_dcount[tid] = 0;
				}
				s_dexcl[tid] = append_off;
			}
		} else {
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
#ifdef RSX_PHASE_TIMING
					if (tid == 0) dbg_acc[10] += 1;
#endif
					OffT w[LB];
#pragma unroll
					for (int j = 0; j < LB; ++j)
						w[j] = (q - j >= 0) ? ld_status(&status[(size_t)(q - j) * kBins + dgt]) : (OffT)SB::kPfx;
#pragma unroll
					for (int j = 0; j < LB; ++j) {
						if (!done) {
							OffT v = w[j];
							while ((v & ~SB::kMask) == 0) { // not published yet: poll this one word, politely
#ifdef RSX_PHASE_TIMING
								if (tid == 0) dbg_acc[11] += 1;
#endif
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
				if (fusedm) {
					// Per destination D (a contiguous range of digits, hence one contiguous run of the
					// sorted buffer): remote element offset = sum of its digits' exclusive prefixes,
					// records = sum of its digits' counts, run start = its first digit's tstart.
					// Lanes of one destination are contiguous in a warp: segmented warp reduction,
					// then one shared atomic per (warp, destination) -- 64-bit shared atomics are CAS
					// loops and 128 digit threads hammering one address cost more than the whole pass.
					const uint32_t D = my_owner;
					const uint32_t grp = __match_any_sync(FULL, D);
					unsigned long long ex = (unsigned long long)excl;
					uint32_t cnt = tcount;
#pragma unroll
					for (int o = 1; o < 32; o <<= 1) {
						const unsigned long long ex2 = __shfl_down_sync(FULL, ex, o);
						const uint32_t cnt2 = __shfl_down_sync(FULL, cnt, o);
						if (lane + o < 32 && ((grp >> (lane + o)) & 1u)) {
							ex += ex2;
							cnt += cnt2;
						}
					}
					if (lane == (uint32_t)__ffs(grp) - 1) {
						atomicAdd(&s_dexcl[D], ex);
						atomicAdd(&s_dcount[D], cnt);
					}
					if (dgt == 0 || p.owner[dgt - 1] != D)
						s_dstart[D] = tstart;
				} else {
					s_gadj[dgt] = (OffT)p.offs[dgt] + excl - (OffT)tstart;
				}
			}
		}
		RSX_T(6);
		if (tid == 0) // next ticket: claimed as late as possible (see above)
			s_misc[0] = atomicAdd(p.ticket, 1u);
		if constexpr (FUSED) {
			if (p.unordered_runs)
				fence_async_smem(); // the sorted tile (generic-proxy stores) becomes visible to the TMA
		}
		__syncthreads(); // (D) sorted tile + gadj complete; nobody reads the staging buffer any more
		const uint32_t next_tile = s_misc[0];
		if (tid == 0 && can_stage && next_tile < full_tiles)
			prefetch(next_tile); // TMA: lands while this tile is being stored
		RSX_T(7);

		// ---- 5. coalesced per-bucket stores ----
		if (fusedm) {
			// Straight into the owners' buffers (peer memory over NVLink).  Per destination one
			// contiguous run; its body goes out as 16-byte vector stores aligned to the REMOTE address
			// (708 vs 480 GB/s for 4-byte stores, tools/peer_bw.py).  The shared-memory side is then
			// misaligned by a per-run constant: two aligned 16-byte loads + a funnel shift.
			constexpr uint32_t G = ES >= 16 ? 1u : 16u / ES; // records per 16-byte chunk
			if (p.unordered_runs && ES < 16) {
				// Keys-only: per destination ONE bulk store of the largest body that is 16-byte aligned
				// on both sides; the < 3 G records around it go out as scalar stores, the j-th left-over
				// slot to the j-th left-over remote position (order inside the run is free).
				for (uint32_t k = 0; k < p.ndest; ++k) {
					const uint32_t beg = s_dstart[k], cnt = s_dcount[k];
					const unsigned long long r0 = p.dest_base[k] + s_dexcl[k] * ES;
					const uint32_t hs = (G - (beg & (G - 1))) & (G - 1);                    // slots to shared alignment
					const uint32_t hr = (uint32_t)((G - ((r0 / ES) & (G - 1))) & (G - 1));  // records to remote alignment
					const uint32_t hmax = hs > hr ? hs : hr;
					const uint32_t L = cnt > hmax ? (cnt - hmax) / G * G : 0u;
					if (tid == 0 && L)
						bulk_s2g(r0 + (unsigned long long)hr * ES, s_rec + beg + hs, L * ES);
					const uint32_t left = cnt - L;
					if (tid < left) {
						const uint32_t sl = tid < hs ? beg + tid : beg + hs + L + (tid - hs);
						const uint32_t rl = tid < hr ? tid : hr + L + (tid - hr);
						*reinterpret_cast<R *>(r0 + (unsigned long long)rl * ES) = s_rec[sl];
					}
				}
				if (tid == 0)
					bulk_commit();
			} else
			for (uint32_t k = 0; k < p.ndest; ++k) {
				const uint32_t beg = s_dstart[k], end = beg + s_dcount[k];
				const unsigned long long r0 = p.dest_base[k] + s_dexcl[k] * ES; // remote byte address of slot `beg`
				uint32_t a0 = beg + (uint32_t)((G - ((r0 / ES) & (G - 1))) & (G - 1));
				if (a0 > end)
					a0 = end;
				const uint32_t a1 = a0 + (end - a0) / G * G;
				const uint32_t nhead = a0 - beg, ntail = end - a1;
				if (tid < nhead + ntail) {
					const uint32_t sl = tid < nhead ? beg + tid : a1 + (tid - nhead);
					*reinterpret_cast<R *>(r0 + (unsigned long long)(sl - beg) * ES) = s_rec[sl];
				}
				if constexpr (ES == 16) {
					// a 16-byte record is already one full vector and dest_base is record-aligned
					R *rv = reinterpret_cast<R *>(r0);
					for (uint32_t q = tid; q < end - beg; q += THREADS)
						rv[q] = s_rec[beg + q];
				} else {
					const uint32_t shb = (a0 & (G - 1)) * ES;          // byte misalignment of the shared side
					const uint32_t dw = shb >> 2, db = (shb & 3u) * 8u; // whole words + bits inside a word
					const uint4 *sv = reinterpret_cast<const uint4 *>(s_rec + (a0 - (a0 & (G - 1))));
					uint4 *rv = reinterpret_cast<uint4 *>(r0 + (unsigned long long)(a0 - beg) * ES);
					for (uint32_t q = tid; q < (a1 - a0) / G; q += THREADS) {
						const uint4 v0 = sv[q], v1 = sv[q + 1];
						const uint32_t w[9] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w, 0u};
						uint4 o;
						switch (dw) {
						case 0: o = make_uint4(__funnelshift_r(w[0], w[1], db), __funnelshift_r(w[1], w[2], db), __funnelshift_r(w[2], w[3], db), __funnelshift_r(w[3], w[4], db)); break;
						case 1: o = make_uint4(__funnelshift_r(w[1], w[2], db), __funnelshift_r(w[2], w[3], db), __funnelshift_r(w[3], w[4], db), __funnelshift_r(w[4], w[5], db)); break;
						case 2: o = make_uint4(__funnelshift_r(w[2], w[3], db), __funnelshift_r(w[3], w[4], db), __funnelshift_r(w[4], w[5], db), __funnelshift_r(w[5], w[6], db)); break;
						default: o = make_uint4(__funnelshift_r(w[3], w[4], db), __funnelshift_r(w[4], w[5], db), __funnelshift_r(w[5], w[6], db), __funnelshift_r(w[6], w[7], db)); break;
						}
						rv[q] = o;
					}
				}
			}
		} else if (full) {
			// Batches of kWriteBatch records: a batch's tile loads, then its bucket-offset lookups, then
			// its stores.  (A test of `write_rec` inside the loop makes the compiler branch around every
			// store and serialises load -> lookup -> store per record, hence the two instantiations.)
			// The pass is bound by shared-memory throughput, not by this latency chain: 1 B keys, ms per
			// pass u32 / u64, serial 2.596 / 3.95, batches of 2: 2.580 / 3.87, 4: 2.637 / 3.93,
			// 6: 2.66 / 3.96, 8: 2.66 / 4.62, 11: 2.61 / 5.29 (profiles/r2_write_batch.log).
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
							if constexpr (ES + PL <= 4) { // streaming (evict-first) stores: 1.4 % on 4-byte keys, neutral or worse on wider records
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
		RSX_T(8);
		tile = next_tile;
		// the next iteration rewrites wh (read in step 4, fenced by D) and s_rec (fenced by A', C')
	}
	if constexpr (FUSED) {
		if (tid == 0 && p.unordered_runs)
			bulk_wait_all(); // every bulk store of this CTA has been written
	}
#ifdef RSX_PHASE_TIMING
	if (tid == 0 && p.dbg) {
		for (int k = 0; k < 12; ++k)
			atomicAdd(&p.dbg[k], dbg_acc[k]);
		atomicAdd(&p.dbg[12], 1ULL);
	}
#endif
}

template <int ES, int PL, int DM, bool FUSED, typename OffT, int RANK, class Cfg>
cudaError_t launch_scatter_c(const ScatterParams &sp, int num_sms, cudaStream_t st) {
	using SM = ScatterSmem<ES, PL, Cfg, FUSED>;
	auto kern = scatter_kernel<ES, PL, DM, FUSED, OffT, RANK, Cfg>;
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
	q.num_tiles = (uint32_t)((sp.n + SM::kTile - 1) / SM::kTile); // status rows are sized for the smallest tile (scatter_geometry)
	uint32_t grid = (uint32_t)num_sms * (uint32_t)ctas_per_sm;
	if (grid > q.num_tiles)
		grid = q.num_tiles;
	kern<<<grid, Cfg::kThreads, SM::kBytes, st>>>(q);
	count_launch();
	return cudaGetLastError();
}

// one translation unit per record size (parallel builds)
cudaError_t launch_scatter_1(const ScatterParams &, int, bool, bool, int, cudaStream_t);
cudaError_t launch_scatter_2(const ScatterParams &, int, bool, bool, int, cudaStream_t);
cudaError_t launch_scatter_4(const ScatterParams &, int, bool, bool, int, cudaStream_t);
cudaError_t launch_scatter_8(const ScatterParams &, int, bool, bool, int, cudaStream_t);
cudaError_t launch_scatter_16(const ScatterParams &, int, bool, bool, int, cudaStream_t);

} // namespace rsx
