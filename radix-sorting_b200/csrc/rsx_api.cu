// rsx_api.cu -- the C ABI (include/rsx.h): argument checking, workspace, pass orchestration.
//
// Host-side control flow mirrors rs_sort_main (radix_sort.hpp:31-93) with the data-dependent
// decisions moved to the device:
//     memset(workspace head + look-back state)
//     K1 histogram_kernel      radix_sort.hpp:48-58
//     K2 setup_kernel          radix_sort.hpp:60-80   (writes the device pass table)
//     K3 scatter_kernel x wc   radix_sort.hpp:83-90   (trivial columns return at once)
//     8-byte read-back of {early_exit, ncols} -> which buffer to return (radix_sort.hpp:89-92)
// There is no CPU implementation anywhere in this file: without a device every entry point
// fails.
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <vector>

#include "rsx_scatter_dispatch.cuh"

namespace rsx {

static std::atomic<unsigned long long> g_launches{0};
static std::atomic<int> g_force_wide{0};
static std::atomic<int> g_small_path{1};
static std::atomic<int> g_fused_bulk{1}; // rsx_set_option("fused_bulk", 0/1): TMA bulk stores in the fused partition pass
static std::atomic<long> g_compact_min_n{1L << 26}; // rsx_set_option("compact_min_n", n); <= 0 disables
void count_launch(unsigned n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

namespace {

thread_local char t_err[512] = "";

// ---- optional per-kernel profiling (rsx_set_option("profile", 1)) ------------------------------
std::atomic<int> g_profile{0};
constexpr int kMaxProf = 2 + kMaxCols;
struct Prof {
	cudaEvent_t ev[kMaxProf + 1] = {};
	bool created = false;
	int count = 0; // events recorded - 1 = intervals
	float ms[kMaxProf] = {};
	int n_ms = 0;
};
thread_local Prof t_prof;

void prof_mark(cudaStream_t st, bool first = false) {
	if (!g_profile.load(std::memory_order_relaxed))
		return;
	Prof &P = t_prof;
	if (!P.created) {
		for (auto &e : P.ev)
			cudaEventCreate(&e);
		P.created = true;
	}
	if (first)
		P.count = 0;
	if (P.count <= kMaxProf)
		cudaEventRecord(P.ev[P.count++], st);
}
void prof_collect() {
	if (!g_profile.load(std::memory_order_relaxed))
		return;
	Prof &P = t_prof;
	P.n_ms = 0;
	for (int i = 0; i + 1 < P.count; ++i) {
		float ms = 0;
		if (cudaEventElapsedTime(&ms, P.ev[i], P.ev[i + 1]) != cudaSuccess)
			ms = -1.f;
		P.ms[P.n_ms++] = ms;
	}
}

int fail_cuda(cudaError_t e, const char *what) {
	snprintf(t_err, sizeof(t_err), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
	(void)cudaGetLastError(); // clear the sticky-free error state
	return e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? RSX_ERR_NO_DEVICE : RSX_ERR_CUDA;
}
#define CU(call)                                  \
	do {                                          \
		cudaError_t e_ = (call);                  \
		if (e_ != cudaSuccess)                    \
			return fail_cuda(e_, #call);          \
	} while (0)

// ---- per-device state: SM count, grow-only workspace and staging buffers ----------------------
// A cached grow-only device buffer, used by one call at a time (guarded by `busy`).
struct Slot {
	void *ptr = nullptr;
	size_t bytes = 0;
	bool busy = false;
	Ctl *pinned = nullptr; // workspace slot only: the mapped pinned pass table + read-back area
};
enum SlotId { WORKSPACE, STAGE };
struct DeviceState {
	std::mutex mu;
	int num_sms = 0;
	int rank_mode = -1; // -1 = not probed yet
	// WORKSPACE: look-back state, head and rank-sort buffers.  STAGE: device copies of host buffers
	// (cached so that a caller sorting host arrays repeatedly does not pay cudaMalloc/cudaFree of
	// gigabytes on every call) and the scratch of segmented sorts and top-k around their inner sorts.
	Slot slot[2];
};
constexpr int kMaxDevices = 64;
DeviceState g_dev[kMaxDevices];

int current_device(int *dev) {
	CU(cudaGetDevice(dev));
	if (*dev < 0 || *dev >= kMaxDevices)
		return RSX_ERR_INVALID;
	DeviceState &D = g_dev[*dev];
	std::lock_guard<std::mutex> lk(D.mu);
	if (D.num_sms == 0)
		CU(cudaDeviceGetAttribute(&D.num_sms, cudaDevAttrMultiProcessorCount, *dev));
	return RSX_OK;
}

std::atomic<int> g_rank_override{-1};

// Decide once per device whether the one-instruction ticket ranking is usable (see
// rsx_scatter.cuh).  Any failure to run the probe selects the provably stable ballot ranking.
int probe_rank_mode(int dev) {
	DeviceState &D = g_dev[dev];
	std::lock_guard<std::mutex> lk(D.mu);
	if (D.rank_mode >= 0)
		return D.rank_mode;
	int mode = RANK_BALLOT;
	unsigned long long *d = nullptr, h = ~0ULL;
	if (cudaMalloc((void **)&d, sizeof(*d)) == cudaSuccess) {
		if (cudaMemset(d, 0, sizeof(*d)) == cudaSuccess && launch_ticket_probe(d, D.num_sms ? D.num_sms : 148, 0) == cudaSuccess &&
		    cudaMemcpy(&h, d, sizeof(h), cudaMemcpyDeviceToHost) == cudaSuccess && h == 0)
			mode = RANK_TICKET;
		cudaFree(d);
	}
	(void)cudaGetLastError();
	D.rank_mode = mode;
	return mode;
}

// The pinned slot of a lease: the mirrored pass table, then a read-back area for histograms (D2H
// copies into pageable memory are staged by the driver and cost tens of microseconds more).
constexpr size_t kPinnedReadback = 256, kPinnedBytes = kPinnedReadback + sizeof(unsigned long long) * kMaxCols * kBins;

// One call's use of a slot: the cached buffer, or a private one when another host thread holds it.
struct Lease {
	int dev = -1;
	Slot *cached = nullptr; // null: ptr (and pinned, for a workspace) are this call's own
	void *ptr = nullptr;
	Ctl *pinned = nullptr;
	unsigned long long *readback() const { return reinterpret_cast<unsigned long long *>(reinterpret_cast<unsigned char *>(pinned) + kPinnedReadback); }
	// Set once copies or kernels that use the leased memory have been enqueued; cleared once the
	// stream has been synchronised.  If a call fails in between, the destructor drains the stream
	// before another host thread can be handed the same buffer.
	cudaStream_t inflight = nullptr;
	bool has_inflight = false;
	void enqueued(cudaStream_t st) { inflight = st; has_inflight = true; }
	void drained() { has_inflight = false; }
	~Lease() {
		if (dev < 0)
			return;
		if (has_inflight) {
			cudaStreamSynchronize(inflight);
			(void)cudaGetLastError();
		}
		if (cached) {
			std::lock_guard<std::mutex> lk(g_dev[dev].mu);
			cached->busy = false;
		} else {
			if (ptr)
				cudaFree(ptr);
			if (pinned)
				cudaFreeHost(pinned);
		}
	}
};

int acquire(Lease &L, int dev, SlotId id, size_t bytes) {
	DeviceState &D = g_dev[dev];
	Slot &S = D.slot[id];
	L.dev = dev;
	std::unique_lock<std::mutex> lk(D.mu);
	if (!S.busy) {
		if (S.bytes < bytes) {
			if (S.ptr) {
				cudaFree(S.ptr);
				S.ptr = nullptr;
				S.bytes = 0;
			}
			CU(cudaMalloc(&S.ptr, bytes));
			S.bytes = bytes;
		}
		if (id == WORKSPACE && !S.pinned)
			CU(cudaHostAlloc((void **)&S.pinned, kPinnedBytes, cudaHostAllocMapped));
		S.busy = true;
		L.ptr = S.ptr;
		L.pinned = S.pinned;
		L.cached = &S;
		return RSX_OK;
	}
	lk.unlock(); // another host thread is sorting on this device: private scratch for this call
	CU(cudaMalloc(&L.ptr, bytes));
	if (id == WORKSPACE)
		CU(cudaHostAlloc((void **)&L.pinned, kPinnedBytes, cudaHostAllocMapped));
	return RSX_OK;
}

// rsx_release: the buffer of a slot no call is using goes back to the driver.
void free_if_idle(Slot &S) {
	if (!S.busy && S.ptr) {
		cudaFree(S.ptr);
		S.ptr = nullptr;
		S.bytes = 0;
	}
}

// ---- layout ---------------------------------------------------------------------------------
int check_layout(const rsx_layout *L, KeyDesc *kd) {
	if (!L)
		return RSX_ERR_INVALID;
	const uint32_t rb = L->record_bytes, kb = L->key_bytes, ko = L->key_offset;
	if (!(rb == 1 || rb == 2 || rb == 4 || rb == 8 || rb == 16))
		return RSX_ERR_INVALID;
	if (!(kb == 1 || kb == 2 || kb == 4 || kb == 8))
		return RSX_ERR_INVALID;
	if (ko + kb > rb || (ko / 8) != ((ko + kb - 1) / 8)) // key inside one aligned 8-byte word
		return RSX_ERR_INVALID;
	if (L->kdf_kind > RSX_KDF_FLOAT || (L->flags & ~RSX_FLAG_INVERT))
		return RSX_ERR_INVALID;
	if (L->kdf_kind == RSX_KDF_FLOAT && !((kb == 4 || kb == 8) && ko % kb == 0))
		return RSX_ERR_INVALID;
	kd->word_sel = ko / 8;
	kd->key_shift = 8u * (ko % 8);
	kd->key_bytes = kb;
	kd->kdf_kind = L->kdf_kind;
	kd->invert = (L->flags & RSX_FLAG_INVERT) ? 1u : 0u;
	return RSX_OK;
}

// rsx_sort / rsx_sort_rank also take records the tile kernels cannot move directly: any
// record_bytes up to kMaxGenericRecord and a key anywhere inside the record.  *generic is set for
// those; kd then describes the EXTRACTED key (a key_bytes-sized scalar).
constexpr uint32_t kMaxGenericRecord = 4096;
int check_layout_any(const rsx_layout *L, KeyDesc *kd, bool *generic) {
	*generic = false;
	if (check_layout(L, kd) == RSX_OK)
		return RSX_OK;
	if (!L)
		return RSX_ERR_INVALID;
	const uint32_t rb = L->record_bytes, kb = L->key_bytes, ko = L->key_offset;
	if (rb < 1 || rb > kMaxGenericRecord || !(kb == 1 || kb == 2 || kb == 4 || kb == 8) || (uint64_t)ko + kb > rb)
		return RSX_ERR_INVALID;
	if (L->kdf_kind > RSX_KDF_FLOAT || (L->flags & ~RSX_FLAG_INVERT) || (L->kdf_kind == RSX_KDF_FLOAT && kb < 4))
		return RSX_ERR_INVALID;
	const rsx_layout key_layout = {kb, 0, kb, L->kdf_kind, L->flags};
	*generic = true;
	return check_layout(&key_layout, kd);
}

// Record whose derived key is all ones: pads the last tile so that padding sorts last.
ulonglong2 pad_record(const KeyDesc &kd) {
	const unsigned long long m = kd.key_bytes >= 8 ? ~0ULL : ((1ULL << (8 * kd.key_bytes)) - 1ULL);
	const unsigned long long top = 1ULL << (8 * kd.key_bytes - 1);
	unsigned long long k = kd.invert ? 0ULL : m; // undo the complement
	if (kd.kdf_kind == RSX_KDF_SIGNED)
		k ^= top;
	else if (kd.kdf_kind == RSX_KDF_FLOAT)
		k ^= (k & top) ? top : m; // inverse of: sign set -> ^m, sign clear -> ^top
	ulonglong2 r = make_ulonglong2(0, 0);
	(kd.word_sel ? r.y : r.x) = k << kd.key_shift;
	return r;
}

enum PtrKind { PK_HOST, PK_DEVICE };
int ptr_kind(const void *p, PtrKind *k) {
	cudaPointerAttributes a;
	cudaError_t e = cudaPointerGetAttributes(&a, p);
	if (e != cudaSuccess)
		return fail_cuda(e, "cudaPointerGetAttributes");
	*k = (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) ? PK_DEVICE : PK_HOST;
	if (a.type == cudaMemoryTypeDevice) { // kernels are launched on the CURRENT device
		int dev = -1;
		if (cudaGetDevice(&dev) == cudaSuccess && a.device != dev) {
			snprintf(t_err, sizeof(t_err), "pointer %p belongs to device %d, the current device is %d", p, a.device, dev);
			return RSX_ERR_INVALID;
		}
	}
	return RSX_OK;
}

// The buffers a and b (b may be null) must all be device memory; with `common`, they may instead
// all be host memory, and *common receives their kind.
int check_residency(PtrKind *common, const void *a, const void *b = nullptr) {
	PtrKind ka, kb = PK_DEVICE;
	int r;
	if ((r = ptr_kind(a, &ka)) || (b && (r = ptr_kind(b, &kb))))
		return r;
	if (common ? ka != kb : (ka != PK_DEVICE || kb != PK_DEVICE))
		return RSX_ERR_MIXED_MEMORY;
	if (common)
		*common = ka;
	return RSX_OK;
}

bool overlaps(const void *a, size_t abytes, const void *b, size_t bbytes) {
	const unsigned char *pa = static_cast<const unsigned char *>(a), *pb = static_cast<const unsigned char *>(b);
	return pa < pb + bbytes && pb < pa + abytes;
}

bool valid_idx_bytes(int b) { return b == 1 || b == 2 || b == 4 || b == 8; }

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct Plan {
	KeyDesc kd;
	uint32_t rb;
	int pl_bytes;       // payload lane carried by the passes (0, 4, 8)
	size_t n;
	PassGeometry geo;
	uint32_t tiles;
	bool wide;
	size_t status_bytes; // look-back state of one column: tiles x 256 status words
	size_t off_head, off_rec[2], off_idx[2], total;
	int n_rec_bufs;
};

Plan make_plan(size_t n, uint32_t record_bytes, const KeyDesc &kd, int rank_idx_bytes, int forced_pl = -1) {
	Plan P;
	P.kd = kd;
	P.rb = record_bytes;
	P.n = n;
	P.pl_bytes = forced_pl >= 0 ? forced_pl : rank_idx_bytes == 0 ? 0 : (rank_idx_bytes == 8 ? 8 : 4);
	P.geo = scatter_geometry(P.rb, P.pl_bytes);
	P.tiles = (uint32_t)((n + P.geo.tile - 1) / P.geo.tile);
	P.wide = n >= (1ULL << 30) || g_force_wide.load(std::memory_order_relaxed);
	P.status_bytes = align_up((size_t)P.tiles * kBins * (P.wide ? 8 : 4), 256);
	// [status of column 0 .. key_bytes-1 | WsHead | rank-sort buffers]: the look-back state and the
	// head's counters are adjacent, so ONE memset prepares a sort.  (Two buffers re-zeroed by the
	// passes themselves were measured: the extra 1 KB of stores per tile costs 1.6 % of a pass, the
	// memset of all columns 0.7 % of a sort.)
	P.off_head = P.status_bytes * kd.key_bytes;
	size_t off = P.off_head + align_up(sizeof(WsHead), 256);
	P.n_rec_bufs = 0;
	P.off_rec[0] = P.off_rec[1] = P.off_idx[0] = P.off_idx[1] = 0;
	if (rank_idx_bytes) {
		// records travel beside the indices; the last live pass writes no records, so at most
		// min(2, columns - 1) record buffers are ever needed.
		P.n_rec_bufs = kd.key_bytes >= 3 ? 2 : (int)kd.key_bytes - 1;
		for (int i = 0; i < P.n_rec_bufs; ++i) {
			P.off_rec[i] = off;
			off += align_up(n * P.rb, 256);
		}
		if (rank_idx_bytes < 4) {
			for (int i = 0; i < 2; ++i) {
				P.off_idx[i] = off;
				off += align_up(n * 4, 256);
			}
		}
	}
	P.total = off;
	return P;
}

// The workspace of a call that runs no pass: the head, behind one tile's look-back rows per column.
Plan head_plan(uint32_t record_bytes, const KeyDesc &kd) { return make_plan(2, record_bytes, kd, 0); }

int run_scatter(const PassBuffers &pb, const Plan &P, int col, unsigned char *wsp, bool forced, int num_sms,
                cudaStream_t st, const Exchange &ex = {}) {
	WsHead *ws = reinterpret_cast<WsHead *>(wsp + P.off_head);
	CU(launch_scatter(pb, P.n, P.rb, P.pl_bytes, P.kd, col, ws, forced, wsp + (size_t)col * P.status_bytes,
	                  &ws->tickets[col], P.wide, num_sms, st, ex));
	return RSX_OK;
}

// zero the look-back state of every column + the head's counters: one memset
cudaError_t zero_workspace(const Plan &P, unsigned char *wsp, cudaStream_t st) {
	return cudaMemsetAsync(wsp, 0, P.off_head + kWsZeroBytes, st);
}

// Enqueue memset + K1 + K2 (+ passes).  Everything is asynchronous on `st`.
int enqueue_front(const void *src, const Plan &P, unsigned char *wsp, Ctl *host_ctl, int num_sms, cudaStream_t st) {
	WsHead *ws = reinterpret_cast<WsHead *>(wsp + P.off_head);
	CU(zero_workspace(P, wsp, st));
	prof_mark(st, true);
	CU(launch_histogram(src, P.n, P.rb, P.kd, ws, num_sms, st));
	prof_mark(st);
	CU(launch_setup(src, P.n, P.rb, P.kd, ws, host_ctl, st));
	prof_mark(st);
	return RSX_OK;
}

int enqueue_passes(const PassBuffers &pb, const Plan &P, unsigned char *wsp, int num_sms, cudaStream_t st) {
	for (uint32_t c = 0; c < P.kd.key_bytes; ++c) {
		int r = run_scatter(pb, P, (int)c, wsp, false, num_sms, st);
		if (r)
			return r;
		prof_mark(st);
	}
	return RSX_OK;
}

// The pass table (which buffer holds the result, radix_sort.hpp:89-92) reaches the host without a
// copy: the setup kernel (or the single-CTA kernel) also stores it into the lease's mapped pinned
// slot, so the host only has to wait for the stream.
void fill_report(rsx_report *rep, const Ctl &c, unsigned long long launches0, bool staged) {
	if (rep) {
		rep->early_exit = c.early_exit;
		rep->ncols = c.early_exit ? 0 : c.ncols;
		rep->live_mask = c.early_exit ? 0 : c.live_mask;
		rep->result_in_aux = c.early_exit ? 0 : (c.ncols & 1u); // radix_sort.hpp:89-92
		rep->kernel_launches = (uint32_t)(g_launches.load() - launches0);
		rep->staged = staged;
		rep->compacted_passes = 0;
	}
}

int read_ctl(Lease &L, cudaStream_t st, unsigned long long launches0, rsx_report *rep, bool staged) {
	CU(cudaStreamSynchronize(st));
	L.drained();
	prof_collect();
	fill_report(rep, *L.pinned, launches0, staged);
	return RSX_OK;
}

void trivial_report(rsx_report *rep) {
	if (rep) {
		memset(rep, 0, sizeof(*rep));
		rep->early_exit = 1;
	}
}

// Paths that read their own report back (which buffer holds the result) take a NULL `report` into
// this one.
rsx_report *report_or_scratch(rsx_report *rep) {
	thread_local rsx_report scratch;
	return rep ? rep : &scratch;
}

// The prologue of an entry point that runs on the current device: open() looks the device up,
// lease() takes the workspace for plan P and counts its kernels as in flight from then on.
struct DeviceCall {
	int dev = -1, sms = 0;
	cudaStream_t st = nullptr;
	Plan P;
	Lease L;
	unsigned char *wsp = nullptr;
	WsHead *ws = nullptr;

	int open(void *stream) {
		int r = current_device(&dev);
		if (r)
			return r;
		sms = g_dev[dev].num_sms;
		st = static_cast<cudaStream_t>(stream);
		return RSX_OK;
	}
	int lease(const Plan &plan) {
		P = plan;
		int r = acquire(L, dev, WORKSPACE, P.total);
		if (r)
			return r;
		L.enqueued(st);
		wsp = static_cast<unsigned char *>(L.ptr);
		ws = reinterpret_cast<WsHead *>(wsp + P.off_head);
		return RSX_OK;
	}
	// Waits for the call's work; the workspace is free for the next call.
	int finish() {
		CU(cudaStreamSynchronize(st));
		L.drained();
		return RSX_OK;
	}
	// Device bytes -> host_out, through the lease's pinned read-back area, after the call's work.
	int read_back(const void *from, size_t bytes, void *host_out) {
		L.enqueued(st);
		CU(cudaMemcpyAsync(L.readback(), from, bytes, cudaMemcpyDeviceToHost, st));
		int r = finish();
		if (r)
			return r;
		memcpy(host_out, L.readback(), bytes);
		return RSX_OK;
	}
};

} // namespace

int rank_mode() {
	const int o = g_rank_override.load(std::memory_order_relaxed);
	if (o == RANK_TICKET || o == RANK_BALLOT)
		return o;
	int dev = 0;
	if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices)
		return RANK_BALLOT;
	return probe_rank_mode(dev);
}

// ---- launch glue declared in rsx_internal.cuh --------------------------------------------------
template <class Cfg> void take_smaller_tile(PassGeometry &g, size_t smem) {
	if (g.tile == 0 || Cfg::kThreads * Cfg::kItems < g.tile)
		g = PassGeometry{Cfg::kThreads, Cfg::kItems, Cfg::kThreads * Cfg::kItems, smem, 0};
}
// Tile geometry that sizes the look-back state: the smallest tile any kernel of this footprint may
// run with (the fused geometry, or the register-resident one), so every kernel uses at most this
// many status rows.  Rank sorts of 1- and 2-byte keys through 32-bit index lanes reserve the rows of
// a u32 rank sort, so their rsx_workspace_bytes stays what callers have been reserving.
template <int ES, int PL> PassGeometry footprint_geometry() {
	static_assert(FusedCfg<ES, PL>::kThreads * FusedCfg<ES, PL>::kItems <=
	              ScatterCfg<ES, PL>::kThreads * ScatterCfg<ES, PL>::kItems, "fused tile must be the smallest");
	PassGeometry g{};
	take_smaller_tile<FusedCfg<ES, PL>>(g, ScatterSmem<ES, PL, FusedCfg<ES, PL>, true>::kBytes);
	if constexpr (PreferV2<ES, PL>::value)
		take_smaller_tile<Cfg2<ES, PL>>(g, Scatter2Smem<ES, PL, Cfg2<ES, PL>>::kBytes);
	else if constexpr (ES < 4 && PL == 4)
		take_smaller_tile<Cfg2<4, 4>>(g, Scatter2Smem<ES, PL, Cfg2<4, 4>>::kBytes);
	return g;
}
template <int ES> PassGeometry footprint_geometry(int payload_bytes) {
	switch (payload_bytes) {
	case 0: return footprint_geometry<ES, 0>();
	case 4: return footprint_geometry<ES, 4>();
	case 8: return footprint_geometry<ES, 8>();
	}
	return PassGeometry{};
}

PassGeometry scatter_geometry(uint32_t record_bytes, int payload_bytes) {
	switch (record_bytes) {
	case 1: return footprint_geometry<1>(payload_bytes);
	case 2: return footprint_geometry<2>(payload_bytes);
	case 4: return footprint_geometry<4>(payload_bytes);
	case 8: return footprint_geometry<8>(payload_bytes);
	case 16: return footprint_geometry<16>(payload_bytes);
	}
	return PassGeometry{};
}

cudaError_t launch_scatter(const PassBuffers &pb, size_t n, uint32_t record_bytes, int payload_bytes,
                           const KeyDesc &kd, int col, const WsHead *ws, bool forced, void *status,
                           unsigned int *ticket, bool wide, int num_sms, cudaStream_t st, const Exchange &ex) {
	ScatterParams sp;
	sp.pb = pb;
	sp.n = n;
	const PassGeometry g = scatter_geometry(record_bytes, payload_bytes);
	if (g.tile == 0)
		return cudaErrorInvalidValue;
	sp.num_tiles = (uint32_t)((n + g.tile - 1) / g.tile);
	sp.col = (uint32_t)col;
	sp.dd = make_digit_desc(kd, col);
	sp.offs = ws->offs + (size_t)col * kBins;
	sp.ctl = forced ? nullptr : &ws->ctl;
	sp.status = status;
	sp.ticket = ticket;
	sp.pad_rec = pad_record(kd);
	sp.dbg = nullptr;
	sp.dest_base = ex.dest_base;
	sp.owner = ex.owner;
	sp.ndest = (uint32_t)ex.ndest;
	sp.dest_cursor = ex.dest_cursor;
	sp.dest_capacity = ex.dest_capacity;
	sp.overflow = ex.overflow;
	// keys-only records: the order inside a (tile, destination) run is free -> TMA bulk stores
	sp.unordered_runs = (ex.dest_base != nullptr && record_bytes == kd.key_bytes && record_bytes < 16 && g_fused_bulk.load(std::memory_order_relaxed)) ? 1u : 0u;
	sp.kd = kd;
	sp.nsplit = (uint32_t)ex.nsplit;
	for (int j = 0; j < kMaxSplit; ++j)
		sp.split[j] = (ex.splitters && j < ex.nsplit) ? ex.splitters[j] : ~0ULL;
#ifdef RSX_PHASE_TIMING
	{
		static unsigned long long *d_dbg = nullptr;
		if (!d_dbg) {
			cudaMalloc((void **)&d_dbg, 16 * sizeof(unsigned long long));
			cudaMemset(d_dbg, 0, 16 * sizeof(unsigned long long));
		}
		sp.dbg = d_dbg;
		extern unsigned long long *g_dbg_ptr;
		g_dbg_ptr = d_dbg;
	}
#endif
	const bool is_float = kd.kdf_kind == RSX_KDF_FLOAT;
	switch (record_bytes) {
	case 1: return launch_scatter_1(sp, payload_bytes, is_float, wide, num_sms, st);
	case 2: return launch_scatter_2(sp, payload_bytes, is_float, wide, num_sms, st);
	case 4: return launch_scatter_4(sp, payload_bytes, is_float, wide, num_sms, st);
	case 8: return launch_scatter_8(sp, payload_bytes, is_float, wide, num_sms, st);
	case 16: return launch_scatter_16(sp, payload_bytes, is_float, wide, num_sms, st);
	}
	return cudaErrorInvalidValue;
}

} // namespace rsx

#ifdef RSX_PHASE_TIMING
namespace rsx { unsigned long long *g_dbg_ptr = nullptr; }
extern "C" int rsx_dbg_phase(unsigned long long *out16, int reset) {
	if (!rsx::g_dbg_ptr)
		return -1;
	cudaDeviceSynchronize();
	cudaMemcpy(out16, rsx::g_dbg_ptr, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
	if (reset)
		cudaMemset(rsx::g_dbg_ptr, 0, 16 * sizeof(unsigned long long));
	return 0;
}
#endif

using namespace rsx;

// ================================================================================================
extern "C" {

int rsx_version(void) { return RSX_VERSION; }

const char *rsx_strerror(int s) {
	switch (s) {
	case RSX_OK: return "ok";
	case RSX_ERR_INVALID: return "invalid argument or unsupported record layout";
	case RSX_ERR_CUDA: return "CUDA error (see rsx_last_cuda_error)";
	case RSX_ERR_NO_DEVICE: return "no CUDA device (librsx has no CPU path)";
	case RSX_ERR_WORKSPACE: return "workspace too small";
	case RSX_ERR_IDX_RANGE: return "n - 1 does not fit the index type";
	case RSX_ERR_MIXED_MEMORY: return "buffers must be all host or all device memory";
	}
	return "unknown status";
}

const char *rsx_last_cuda_error(void) { return t_err; }

uint64_t rsx_total_kernel_launches(void) { return g_launches.load(); }

int rsx_set_option(const char *name, long value) {
	if (name && strcmp(name, "profile") == 0) {
		g_profile.store(value ? 1 : 0);
		return RSX_OK;
	}
	if (name && strcmp(name, "rank_mode") == 0) { // -1 auto (probe), 0 ticket, 1 ballot
		if (value < -1 || value > 1)
			return RSX_ERR_INVALID;
		g_rank_override.store((int)value);
		return RSX_OK;
	}
	if (name && strcmp(name, "scatter_variant") == 0) // only the default kernel choice exists
		return value == 0 ? RSX_OK : RSX_ERR_INVALID;
	if (name && strcmp(name, "small_path") == 0) { // 0: always use the multi-kernel path (tests)
		g_small_path.store(value ? 1 : 0);
		return RSX_OK;
	}
	if (name && strcmp(name, "compact_min_n") == 0) { // key compaction for keys-only sorts of >= value keys; <= 0: never
		g_compact_min_n.store(value > 0 ? value : (1L << 62));
		return RSX_OK;
	}
	if (name && strcmp(name, "fused_bulk") == 0) { // A/B: keys-only fused passes store their runs with TMA bulk copies
		g_fused_bulk.store(value ? 1 : 0);
		return RSX_OK;
	}
	if (name && strcmp(name, "force_wide") == 0) { // tests: run the n >= 2^30 (64-bit offset) kernels at small n
		g_force_wide.store(value ? 1 : 0);
		return RSX_OK;
	}
	if (name && strcmp(name, "query_rank_mode") == 0)
		return rank_mode(); // 0 ticket, 1 ballot
	return RSX_ERR_INVALID;
}

int rsx_get_profile(float *ms_out, int cap) {
	if (!ms_out || cap < 0)
		return RSX_ERR_INVALID;
	const int k = t_prof.n_ms < cap ? t_prof.n_ms : cap;
	for (int i = 0; i < k; ++i)
		ms_out[i] = t_prof.ms[i];
	return k;
}

size_t rsx_workspace_bytes(size_t n, const rsx_layout *layout, int rank_idx_bytes) {
	KeyDesc kd;
	bool generic = false;
	if (check_layout_any(layout, &kd, &generic) != RSX_OK)
		return 0;
	if (generic) // the keys are ranked, the records gathered: the passes see key_bytes-sized records
		return make_plan(n < 2 ? 2 : n, layout->key_bytes, kd, rank_idx_bytes ? rank_idx_bytes : (n <= 0xFFFFFFFFull ? 4 : 8)).total;
	return make_plan(n < 2 ? 2 : n, layout->record_bytes, kd, rank_idx_bytes).total;
}

int rsx_reserve(size_t bytes) {
	int dev;
	int r = current_device(&dev);
	if (r)
		return r;
	Lease L;
	return acquire(L, dev, WORKSPACE, bytes);
}

void rsx_release(void) {
	int dev;
	if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices)
		return;
	DeviceState &D = g_dev[dev];
	std::lock_guard<std::mutex> lk(D.mu);
	for (Slot &S : D.slot)
		free_if_idle(S);
}

// ---- key compaction (N4) ---------------------------------------------------------------------------

// Runs of contiguous varying bits -> Compaction.  More than kMaxRuns runs are merged across the
// smallest gaps (a constant bit inside a run is harmless: it is the same in every key).  Returns
// false when compaction would not save at least two passes.
static bool plan_compaction(const Ctl &c, const KeyDesc &kd, Compaction *out) {
	const unsigned long long m = kd.key_bytes >= 8 ? ~0ULL : ((1ULL << (8 * kd.key_bytes)) - 1ULL);
	const unsigned long long varying = c.key_or & c.key_nand & m;
	if (varying == 0 || c.ncols < 3)
		return false;
	struct Run { uint32_t lo, hi; }; // bits [lo, hi)
	Run runs[64];
	int nr = 0;
	for (uint32_t b = 0; b < 8 * kd.key_bytes;) {
		if (!((varying >> b) & 1ULL)) {
			++b;
			continue;
		}
		uint32_t e = b;
		while (e < 8 * kd.key_bytes && ((varying >> e) & 1ULL))
			++e;
		runs[nr++] = {b, e};
		b = e;
	}
	while (nr > kMaxRuns) { // merge the two neighbours with the smallest gap
		int best = 0;
		for (int i = 1; i + 1 < nr; ++i)
			if (runs[i + 1].lo - runs[i].hi < runs[best + 1].lo - runs[best].hi)
				best = i;
		runs[best].hi = runs[best + 1].hi;
		for (int i = best + 1; i + 1 < nr; ++i)
			runs[i] = runs[i + 1];
		--nr;
	}
	Compaction k{};
	unsigned long long covered = 0;
	uint32_t at = 0;
	for (int i = 0; i < nr; ++i) {
		k.src_shift[i] = runs[i].lo;
		k.width[i] = runs[i].hi - runs[i].lo;
		k.dst_shift[i] = at;
		k.wmask[i] = k.width[i] >= 64 ? ~0ULL : ((1ULL << k.width[i]) - 1ULL);
		at += k.width[i];
		covered |= (k.width[i] >= 64 ? ~0ULL : ((1ULL << k.width[i]) - 1ULL)) << runs[i].lo;
	}
	k.nruns = (uint32_t)nr;
	k.bits = at;
	k.const_bits = c.key_or & ~covered & m; // constant bits: set in every key or in none
	// The compacting histogram + the expansion cost about as much as 1.5 (4-byte keys) to 1.8
	// (8-byte keys) passes: compact only when clearly more passes are saved (profiles/r2_variants.md).
	const uint32_t passes = (at + 7) / 8;
	if (passes + (kd.key_bytes == 4 ? 3u : 2u) > c.ncols)
		return false;
	*out = k;
	return true;
}

// src holds the original keys (K1/K2 have run).  K1c writes the compacted keys to aux and their
// digit histograms to the workspace, the ordinary passes sort them (only ceil(bits/8) columns are
// live), and the expansion puts the original keys into the buffer the reference returns.
static int sort_compacted(void *src, void *aux, const Plan &P, unsigned char *wsp, Lease &L, const Compaction &cmp,
                          const Ctl &first, int sms, cudaStream_t st) {
	WsHead *ws = reinterpret_cast<WsHead *>(wsp + P.off_head);
	KeyDesc plain = P.kd; // compacted keys are plain unsigned values
	plain.kdf_kind = RSX_KDF_UNSIGNED;
	plain.invert = 0;
	Plan Pc = P;
	Pc.kd = plain;
	CU(zero_workspace(P, wsp, st));
	prof_mark(st, true);
	CU(launch_histogram(src, P.n, P.rb, P.kd, ws, sms, st, &cmp, aux));
	prof_mark(st);
	CU(launch_setup(aux, P.n, P.rb, plain, ws, L.pinned, st));
	prof_mark(st);
	PassBuffers pb{};
	pb.rec_first = aux;
	pb.rec_buf[0] = src;
	pb.rec_buf[1] = aux;
	int r = enqueue_passes(pb, Pc, wsp, sms, st);
	if (r)
		return r;
	const uint32_t passes = (cmp.bits + 7) / 8; // every compacted column is live by construction
	void *sorted = (passes & 1u) ? src : aux;
	void *target = (first.ncols & 1u) ? aux : src; // radix_sort.hpp:89-92 with the reference's column count
	CU(launch_expand_keys(sorted, target, P.n, P.kd, cmp, sms, st));
	CU(cudaStreamSynchronize(st));
	L.drained();
	prof_collect();
	if (L.pinned->ncols != passes || L.pinned->early_exit) {
		snprintf(t_err, sizeof(t_err), "key compaction: expected %u live columns, the device found %u", passes, L.pinned->ncols);
		return RSX_ERR_CUDA;
	}
	return RSX_OK;
}

// ---- value sort --------------------------------------------------------------------------------
// Value or rank sort of an input that fits one CTA: one launch (rsx_small.cu), the pass table read
// back like the multi-kernel path's.
static bool fits_one_cta(size_t n, uint32_t record_bytes, bool ranksort) {
	return g_small_path.load(std::memory_order_relaxed) && n <= small_sort_capacity(record_bytes, ranksort);
}
static int sort_one_cta(const void *src, void *out_even, void *out_odd, void *ib, int idx_bytes, size_t n, uint32_t record_bytes,
                        const KeyDesc &kd, rsx_report *rep, cudaStream_t st, int dev, bool staged, unsigned long long launches0) {
	Lease L;
	int r = acquire(L, dev, WORKSPACE, sizeof(WsHead) + 256);
	if (r)
		return r;
	L.enqueued(st);
	prof_mark(st, true);
	CU(launch_small_sort(src, out_even, out_odd, ib, idx_bytes, n, record_bytes, kd, L.pinned, st));
	prof_mark(st);
	return read_ctl(L, st, launches0, rep, staged);
}

// rep must not be NULL (report_or_scratch).
static int sort_device(void *src, void *aux, size_t n, const rsx_layout *layout, const KeyDesc &kd,
                       void **result, rsx_report *rep, cudaStream_t st, int dev, bool staged) {
	const unsigned long long l0 = g_launches.load();
	int r;
	if (fits_one_cta(n, layout->record_bytes, false)) {
		if ((r = sort_one_cta(src, src, aux, nullptr, 0, n, layout->record_bytes, kd, rep, st, dev, staged, l0)))
			return r;
		*result = rep->result_in_aux ? aux : src;
		return RSX_OK;
	}
	const Plan P = make_plan(n, layout->record_bytes, kd, 0);
	Lease L;
	if ((r = acquire(L, dev, WORKSPACE, P.total)))
		return r;
	L.enqueued(st);
	unsigned char *wsp = static_cast<unsigned char *>(L.ptr);
	const int sms = g_dev[dev].num_sms;
	if ((r = enqueue_front(src, P, wsp, L.pinned, sms, st)))
		return r;
	// Key compaction (README.md:716-758) for large keys-only sorts: one early look at what K1 found.
	// If the bits that vary over the input fit in at least two fewer 8-bit columns than the live
	// byte columns, the keys are compacted and sorted in that many fewer passes.
	if (layout->record_bytes == kd.key_bytes && kd.key_bytes >= 4 && n >= (size_t)g_compact_min_n.load(std::memory_order_relaxed)) {
		CU(cudaStreamSynchronize(st));
		const Ctl first = *L.pinned;
		Compaction cmp;
		if (!first.early_exit && plan_compaction(first, kd, &cmp)) {
			if ((r = sort_compacted(src, aux, P, wsp, L, cmp, first, sms, st)))
				return r;
			fill_report(rep, first, l0, staged); // the reference's pass table, on ITS column count
			rep->compacted_passes = (cmp.bits + 7) / 8;
			*result = rep->result_in_aux ? aux : src;
			return RSX_OK;
		}
	}
	PassBuffers pb{};
	pb.rec_first = src;
	pb.rec_buf[0] = aux; // pass 0: src -> aux, pass 1: aux -> src, ... (radix_sort.hpp:89)
	pb.rec_buf[1] = src;
	if ((r = enqueue_passes(pb, P, wsp, sms, st)))
		return r;
	if ((r = read_ctl(L, st, l0, rep, staged)))
		return r;
	*result = rep->result_in_aux ? aux : src;
	return RSX_OK;
}

static int rank_device(const void *src, void *ib, size_t n, const rsx_layout *layout, const KeyDesc &kd,
                       int idx_bytes, void **result, rsx_report *rep, cudaStream_t st, int dev, bool staged);

// Records of any size (see check_layout_any): keys are extracted, rank-sorted, and one gather puts
// every record in its final place -- in the buffer the reference's parity rule designates.
static int sort_device_generic(void *src, void *aux, size_t n, const rsx_layout *layout, const KeyDesc &kdk,
                               void **result, rsx_report *rep, cudaStream_t st, int dev, bool staged) {
	const uint32_t rb = layout->record_bytes, kb = layout->key_bytes;
	const int idxb = n <= 0xFFFFFFFFull ? 4 : 8;
	const rsx_layout key_layout = {kb, 0, kb, layout->kdf_kind, layout->flags};
	const size_t kbytes = align_up(n * kb, 256);
	Lease SL;
	int r = acquire(SL, dev, STAGE, kbytes + 2 * n * (size_t)idxb);
	if (r)
		return r;
	SL.enqueued(st);
	unsigned char *keys = static_cast<unsigned char *>(SL.ptr), *ib = keys + kbytes;
	const int sms = g_dev[dev].num_sms;
	CU(launch_extract_keys(src, n, rb, layout->key_offset, kb, keys, sms, st));
	void *ranks = nullptr;
	if ((r = rank_device(keys, ib, n, &key_layout, kdk, idxb, &ranks, rep, st, dev, staged)))
		return r;
	rep->kernel_launches += 1;
	if (rep->early_exit) { // radix_sort.hpp:60-62: nothing moves
		SL.drained();
		*result = src;
		return RSX_OK;
	}
	CU(launch_gather_records(src, ranks, idxb, aux, n, rb, sms, st));
	rep->kernel_launches += 1;
	if (!rep->result_in_aux) // even number of live columns: the reference's result is in src
		CU(cudaMemcpyAsync(src, aux, n * (size_t)rb, cudaMemcpyDeviceToDevice, st));
	CU(cudaStreamSynchronize(st));
	SL.drained();
	*result = rep->result_in_aux ? aux : src;
	return RSX_OK;
}

// Host buffers: stage through device memory.  The first src_bytes of the stage lease receive src,
// the next other_bytes are the second buffer; sort_dev(dsrc, dother, &dres) sorts there.  out_bytes
// of the result come back to out_even, or to out_odd when the result is in the second buffer (the
// reference's parity rule); an early exit copies nothing back unless always_copy.
static int sort_staged(const void *src, size_t src_bytes, size_t other_bytes, void *out_even, void *out_odd, size_t out_bytes,
                       bool always_copy, int dev, cudaStream_t st, rsx_report *rep, void **result,
                       const std::function<int(void *, void *, void **)> &sort_dev) {
	Lease SL;
	int r = acquire(SL, dev, STAGE, align_up(src_bytes, 256) + other_bytes);
	if (r)
		return r;
	SL.enqueued(st); // drained below on success, by ~Lease on any failure
	unsigned char *dsrc = static_cast<unsigned char *>(SL.ptr), *dother = dsrc + align_up(src_bytes, 256);
	cudaError_t e = cudaMemcpyAsync(dsrc, src, src_bytes, cudaMemcpyHostToDevice, st);
	if (e != cudaSuccess)
		return fail_cuda(e, "H2D");
	void *dres = nullptr;
	if ((r = sort_dev(dsrc, dother, &dres)))
		return r;
	void *hres = rep->result_in_aux ? out_odd : out_even;
	if (always_copy || !rep->early_exit) {
		e = cudaMemcpyAsync(hres, dres, out_bytes, cudaMemcpyDeviceToHost, st);
		if (e == cudaSuccess)
			e = cudaStreamSynchronize(st);
		if (e != cudaSuccess)
			return fail_cuda(e, "D2H");
	}
	SL.drained(); // sort_dev / the D2H copy synchronised the stream
	*result = hres;
	return RSX_OK;
}

int rsx_sort(void *src, void *aux, size_t n, const rsx_layout *layout, void **result, rsx_report *rep,
             void *stream) {
	KeyDesc kd;
	bool generic = false;
	int r = check_layout_any(layout, &kd, &generic);
	if (r)
		return r;
	if (!result || (n && (!src || !aux)))
		return RSX_ERR_INVALID;
	const size_t bytes = n * layout->record_bytes;
	// src and aux are __restrict__ in the reference (radix_sort.hpp:32): overlapping buffers are a bug
	if (n >= 2 && overlaps(src, bytes, aux, bytes))
		return RSX_ERR_INVALID;
	if (n < 2) { // radix_sort.hpp:100-101
		*result = src;
		trivial_report(rep);
		return RSX_OK;
	}
	int dev;
	if ((r = current_device(&dev)))
		return r;
	PtrKind kind;
	if ((r = check_residency(&kind, src, aux)))
		return r;
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	rep = report_or_scratch(rep);
	auto sort_dev = [&](void *s_, void *a_, void **res_, bool staged_) {
		return generic ? sort_device_generic(s_, a_, n, layout, kd, res_, rep, st, dev, staged_)
		               : sort_device(s_, a_, n, layout, kd, res_, rep, st, dev, staged_);
	};
	if (kind == PK_DEVICE)
		return sort_dev(src, aux, result, false);
	// The reference sorts host memory in place: the bytes land in the buffer it would have returned,
	// the other buffer is left as is (the reference leaves the penultimate pass there, which callers
	// must treat as garbage).
	return sort_staged(src, bytes, align_up(bytes, 256), src, aux, bytes, false, dev, st, rep, result,
	                   [&](void *ds, void *da, void **dres) { return sort_dev(ds, da, dres, true); });
}

// ---- rank sort ---------------------------------------------------------------------------------
static int rank_device(const void *src, void *ib, size_t n, const rsx_layout *layout, const KeyDesc &kd,
                       int idx_bytes, void **result, rsx_report *rep, cudaStream_t st, int dev, bool staged) {
	const unsigned long long l0 = g_launches.load();
	int r;
	if (fits_one_cta(n, layout->record_bytes, true)) {
		if ((r = sort_one_cta(src, nullptr, nullptr, ib, idx_bytes, n, layout->record_bytes, kd, rep, st, dev, staged, l0)))
			return r;
		*result = static_cast<unsigned char *>(ib) + (rep->result_in_aux ? n * (size_t)idx_bytes : 0);
		return RSX_OK;
	}
	const Plan P = make_plan(n, layout->record_bytes, kd, idx_bytes);
	Lease L;
	if ((r = acquire(L, dev, WORKSPACE, P.total)))
		return r;
	L.enqueued(st);
	unsigned char *wsp = static_cast<unsigned char *>(L.ptr);
	WsHead *ws = reinterpret_cast<WsHead *>(wsp + P.off_head);
	const int sms = g_dev[dev].num_sms;
	if ((r = enqueue_front(src, P, wsp, L.pinned, sms, st)))
		return r;
	CU(launch_iota_if_early(ib, idx_bytes, n, &ws->ctl, st)); // radix_sort_rank.hpp:52-57
	unsigned char *ibb = static_cast<unsigned char *>(ib);
	PassBuffers pb{};
	pb.rec_first = src;
	pb.rec_buf[0] = P.n_rec_bufs > 0 ? wsp + P.off_rec[0] : nullptr;
	pb.rec_buf[1] = P.n_rec_bufs > 1 ? wsp + P.off_rec[1] : pb.rec_buf[0];
	pb.pl_first = nullptr;
	pb.synth_index = 1;   // radix_sort_rank.hpp:52: index_buffer[i] = i, never materialised
	pb.skip_last_rec = 1;
	if (idx_bytes >= 4) {
		pb.pl_buf[0] = ibb + n * (size_t)idx_bytes; // radix_sort_rank.hpp:77-78: first pass writes the 2nd half
		pb.pl_buf[1] = ibb;
	} else {
		pb.pl_buf[0] = wsp + P.off_idx[0];
		pb.pl_buf[1] = wsp + P.off_idx[1];
	}
	if ((r = enqueue_passes(pb, P, wsp, sms, st)))
		return r;
	if (idx_bytes < 4)
		CU(launch_narrow_index(reinterpret_cast<uint32_t *>(wsp + P.off_idx[0]),
		                       reinterpret_cast<uint32_t *>(wsp + P.off_idx[1]), ib, idx_bytes, n, &ws->ctl, st));
	if ((r = read_ctl(L, st, l0, rep, staged)))
		return r;
	*result = rep->result_in_aux ? ibb + n * (size_t)idx_bytes : ibb; // radix_sort_rank.hpp:91
	return RSX_OK;
}

int rsx_sort_rank(const void *src, void *index_buffer, size_t n, const rsx_layout *layout, int idx_bytes,
                  void **result, rsx_report *rep, void *stream) {
	KeyDesc kd;
	bool generic = false;
	int r = check_layout_any(layout, &kd, &generic);
	if (r)
		return r;
	if (!valid_idx_bytes(idx_bytes))
		return RSX_ERR_INVALID;
	if (!result || (n && (!src || !index_buffer)))
		return RSX_ERR_INVALID;
	if (idx_bytes < 8 && n && (n - 1) >> (8 * idx_bytes))
		return RSX_ERR_IDX_RANGE;
	int dev;
	if (n < 2) { // radix_sort_rank.hpp:28-32
		if (n == 1) {
			PtrKind k;
			if ((r = current_device(&dev)) || (r = ptr_kind(index_buffer, &k)))
				return r;
			if (k == PK_DEVICE)
				CU(cudaMemset(index_buffer, 0, idx_bytes));
			else
				memset(index_buffer, 0, idx_bytes);
		}
		*result = index_buffer;
		trivial_report(rep);
		return RSX_OK;
	}
	if ((r = current_device(&dev)))
		return r;
	PtrKind kind;
	if ((r = check_residency(&kind, src, index_buffer)))
		return r;
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	rep = report_or_scratch(rep);
	// records of any size: rank the extracted keys (src itself is never written either way)
	const rsx_layout key_layout = {layout->key_bytes, 0, layout->key_bytes, layout->kdf_kind, layout->flags};
	auto rank_dev = [&](const void *s_, void *ib_, void **res_, bool staged_) -> int {
		if (!generic)
			return rank_device(s_, ib_, n, layout, kd, idx_bytes, res_, rep, st, dev, staged_);
		void *keys = nullptr;
		cudaError_t e = cudaMallocAsync(&keys, n * (size_t)layout->key_bytes, st);
		if (e != cudaSuccess)
			return fail_cuda(e, "cudaMallocAsync(keys)");
		e = launch_extract_keys(s_, n, layout->record_bytes, layout->key_offset, layout->key_bytes, keys, g_dev[dev].num_sms, st);
		int rr = e == cudaSuccess ? rank_device(keys, ib_, n, &key_layout, kd, idx_bytes, res_, rep, st, dev, staged_)
		                          : fail_cuda(e, "extract_keys");
		cudaFreeAsync(keys, st);
		return rr;
	};
	if (kind == PK_DEVICE)
		return rank_dev(src, index_buffer, result, false);
	// the indices of an early exit are the identity, written by the device: always copied back
	const size_t ibytes = n * (size_t)idx_bytes;
	return sort_staged(src, n * layout->record_bytes, 2 * ibytes, index_buffer, static_cast<unsigned char *>(index_buffer) + ibytes,
	                   ibytes, true, dev, st, rep, result,
	                   [&](void *ds, void *dib, void **dres) { return rank_dev(ds, dib, dres, true); });
}

// ---- segmented sort ------------------------------------------------------------------------------
// Host plan: consecutive short segments are packed into groups that one CTA sorts (rsx_segments.cu);
// longer segments go through sort_device / rank_device one by one.  The batch's pass table comes
// from one pre-pass over all n records, so every group writes into the buffer the reference's
// parity rule designates for the batch.

// offsets[0] == 0, non-decreasing, offsets[nseg] == n.  *max_len: the longest segment.
static int check_offsets(const uint64_t *off, size_t nseg, size_t n, size_t *max_len) {
	if (off[0] != 0 || off[nseg] != n)
		return RSX_ERR_INVALID;
	size_t m = 0;
	for (size_t s = 0; s < nseg; ++s) {
		if (off[s + 1] < off[s])
			return RSX_ERR_INVALID;
		m = off[s + 1] - off[s] > m ? off[s + 1] - off[s] : m;
	}
	*max_len = m;
	return RSX_OK;
}

static bool idx_fits(int idx_bytes, size_t max_len) {
	return idx_bytes == 0 || idx_bytes == 8 || max_len == 0 || ((max_len - 1) >> (8 * idx_bytes)) == 0;
}

// A pointer the runtime cannot classify (no driver, no device) cannot be device memory.
static bool is_device_memory(const void *p) {
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
		(void)cudaGetLastError();
		return false;
	}
	return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Grow-only pinned host memory of the calling thread: segmented sorts read the device offsets back
// into it and build and upload their group plan in it, top-k reads back its column count.  The calls
// using it are synchronous.
static int thread_pinned_buffer(size_t bytes, unsigned char **out) {
	thread_local void *buf = nullptr;
	thread_local size_t cap = 0;
	if (cap < bytes) {
		if (buf)
			cudaFreeHost(buf);
		buf = nullptr;
		cap = 0;
		CU(cudaHostAlloc(&buf, bytes, cudaHostAllocPortable));
		cap = bytes;
	}
	*out = static_cast<unsigned char *>(buf);
	return RSX_OK;
}

// One walk over the offsets.  A group closes when the next segment would overflow one CTA (`cap`
// records) or when it holds kMaxGroupSegments segments; empty segments take no part.  tab receives
// every group's segment starts and length (see SegGroup).
static void plan_groups(const uint64_t *off, size_t nseg, size_t cap, uint32_t *tab, size_t *ntab,
                        std::vector<SegGroup> &groups, std::vector<size_t> &large) {
	SegGroup g{};
	size_t t = 0;
	auto close = [&]() {
		if (g.nseg) {
			tab[t++] = g.len;
			groups.push_back(g);
		}
		g = SegGroup{};
	};
	for (size_t s = 0; s < nseg; ++s) {
		const size_t len = off[s + 1] - off[s];
		if (len == 0)
			continue;
		if (len > cap) {
			close();
			large.push_back(s);
			continue;
		}
		if (g.len + len > cap || g.nseg == kMaxGroupSegments)
			close();
		if (g.nseg == 0) {
			g.begin = off[s];
			g.tab = (uint32_t)t;
		}
		tab[t++] = g.len;
		g.len += (uint32_t)len;
		++g.nseg;
	}
	close();
	*ntab = t;
}

static int sort_segments_common(const void *src, void *aux, void *ib, int idx_bytes, size_t n, const uint64_t *offsets,
                                size_t nseg, const rsx_layout *layout, void **result, rsx_report *rep, void *stream) {
	const bool ranksort = idx_bytes != 0;
	KeyDesc kd;
	int r = check_layout(layout, &kd); // records the tile kernels move directly: 1, 2, 4, 8 or 16 bytes
	if (r)
		return r;
	if (ranksort && !valid_idx_bytes(idx_bytes))
		return RSX_ERR_INVALID;
	if (!result || !offsets || (n && (!src || !(ranksort ? ib : aux))) || (nseg == 0 && n > 0))
		return RSX_ERR_INVALID;
	const uint32_t rb = layout->record_bytes;
	if (!ranksort && n >= 2 && overlaps(src, n * rb, aux, n * rb))
		return RSX_ERR_INVALID;
	// host offsets: everything is checked before any device work
	const bool dev_offsets = is_device_memory(offsets);
	size_t max_len = 0;
	if (!dev_offsets) {
		if ((r = check_offsets(offsets, nseg, n, &max_len)))
			return r;
		if (!idx_fits(idx_bytes, max_len))
			return RSX_ERR_IDX_RANGE;
	}
	if (n < 2) { // one segment of at most one record: what rsx_sort / rsx_sort_rank do
		if (ranksort)
			return rsx_sort_rank(src, ib, n, layout, idx_bytes, result, rep, stream);
		*result = const_cast<void *>(src);
		trivial_report(rep);
		return RSX_OK;
	}
	int dev;
	if ((r = current_device(&dev)))
		return r;
	if ((r = check_residency(nullptr, src, ranksort ? ib : aux)))
		return r;
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	const unsigned long long l0 = g_launches.load();
	const size_t off_bytes = (nseg + 1) * sizeof(uint64_t);

	// ---- plan on the host ----
	unsigned char *hbuf = nullptr;
	const size_t rd_bytes = dev_offsets ? align_up(off_bytes, 256) : 0;
	const size_t tab_cap = align_up(2 * nseg * sizeof(uint32_t), 256); // <= one start per segment + one end per group
	if ((r = thread_pinned_buffer(rd_bytes + tab_cap + nseg * sizeof(SegGroup), &hbuf)))
		return r;
	const uint64_t *hoff = offsets;
	if (dev_offsets) { // read back once
		CU(cudaMemcpyAsync(hbuf, offsets, off_bytes, cudaMemcpyDeviceToHost, st));
		CU(cudaStreamSynchronize(st));
		hoff = reinterpret_cast<const uint64_t *>(hbuf);
		if ((r = check_offsets(hoff, nseg, n, &max_len)))
			return r;
		if (!idx_fits(idx_bytes, max_len))
			return RSX_ERR_IDX_RANGE;
	}
	uint32_t *tab = reinterpret_cast<uint32_t *>(hbuf + rd_bytes);
	size_t ntab = 0;
	std::vector<SegGroup> groups;
	std::vector<size_t> large;
	plan_groups(hoff, nseg, segment_group_capacity(rb, ranksort), tab, &ntab, groups, large);
	// the plan travels as [segment starts | groups]
	const size_t tab_bytes = align_up(ntab * sizeof(uint32_t), 16), grp_bytes = groups.size() * sizeof(SegGroup);
	memcpy(hbuf + rd_bytes + tab_bytes, groups.data(), grp_bytes);

	// ---- pre-pass + group kernel: two launches for any number of short segments ----
	Ctl c;
	{
		const size_t off_head = 0, off_offs = align_up(sizeof(WsHead), 256);
		const size_t off_plan = off_offs + (dev_offsets ? 0 : align_up(off_bytes, 256));
		Lease L;
		if ((r = acquire(L, dev, WORKSPACE, off_plan + tab_bytes + grp_bytes)))
			return r;
		L.enqueued(st);
		unsigned char *wsp = static_cast<unsigned char *>(L.ptr);
		WsHead *ws = reinterpret_cast<WsHead *>(wsp + off_head);
		const unsigned long long *d_off = reinterpret_cast<const unsigned long long *>(offsets);
		CU(cudaMemsetAsync(ws, 0, kWsZeroBytes, st));
		if (!dev_offsets) {
			CU(cudaMemcpyAsync(wsp + off_offs, offsets, off_bytes, cudaMemcpyHostToDevice, st));
			d_off = reinterpret_cast<const unsigned long long *>(wsp + off_offs);
		}
		if (!groups.empty())
			CU(cudaMemcpyAsync(wsp + off_plan, tab, tab_bytes + grp_bytes, cudaMemcpyHostToDevice, st));
		CU(launch_segment_prepass(src, n, rb, kd, d_off, nseg, ws, L.pinned, g_dev[dev].num_sms, st));
		if (!groups.empty())
			CU(launch_segment_groups(src, const_cast<void *>(src), aux, ib, idx_bytes, n, rb, kd,
			                         reinterpret_cast<const SegGroup *>(wsp + off_plan + tab_bytes), groups.size(),
			                         reinterpret_cast<const uint32_t *>(wsp + off_plan), &ws->ctl, st));
		CU(cudaStreamSynchronize(st));
		L.drained();
		c = *L.pinned;
	} // the workspace is free again for the long segments' own sorts

	const bool early = c.early_exit != 0, odd = !early && (c.ncols & 1u);
	// ---- long segments: the ordinary path on the sub-range, result moved where the batch's lies ----
	if (!large.empty() && !(early && !ranksort)) {
		Lease SL;
		size_t max_large = 0;
		for (size_t s : large)
			max_large = hoff[s + 1] - hoff[s] > max_large ? hoff[s + 1] - hoff[s] : max_large;
		if (ranksort) {
			if ((r = acquire(SL, dev, STAGE, 2 * max_large * (size_t)idx_bytes)))
				return r;
			SL.enqueued(st);
		}
		for (size_t s : large) {
			const size_t o = hoff[s], len = hoff[s + 1] - o;
			void *res = nullptr;
			rsx_report srep;
			if (ranksort) {
				if ((r = rank_device(static_cast<const unsigned char *>(src) + o * rb, SL.ptr, len, layout, kd, idx_bytes, &res, &srep,
				                     st, dev, false)))
					return r;
				unsigned char *to = static_cast<unsigned char *>(ib) + ((odd ? n : 0) + o) * (size_t)idx_bytes;
				CU(cudaMemcpyAsync(to, res, len * (size_t)idx_bytes, cudaMemcpyDeviceToDevice, st));
				CU(cudaStreamSynchronize(st)); // the staging buffer is reused by the next segment
			} else {
				unsigned char *s0 = static_cast<unsigned char *>(const_cast<void *>(src)) + o * rb;
				unsigned char *a0 = static_cast<unsigned char *>(aux) + o * rb;
				if ((r = sort_device(s0, a0, len, layout, kd, &res, &srep, st, dev, false)))
					return r;
				void *want = odd ? a0 : s0;
				if (res != want)
					CU(cudaMemcpyAsync(want, res, len * (size_t)rb, cudaMemcpyDeviceToDevice, st));
			}
		}
		CU(cudaStreamSynchronize(st));
		SL.drained();
	}
	fill_report(rep, c, l0, false);
	if (ranksort)
		*result = static_cast<unsigned char *>(ib) + (odd ? n * (size_t)idx_bytes : 0);
	else
		*result = odd ? aux : const_cast<void *>(src);
	return RSX_OK;
}

int rsx_sort_segments(void *src, void *aux, size_t n, const uint64_t *offsets, size_t nseg, const rsx_layout *layout,
                      void **result, rsx_report *report, void *stream) {
	return sort_segments_common(src, aux, nullptr, 0, n, offsets, nseg, layout, result, report, stream);
}

int rsx_sort_rank_segments(const void *src, void *index_buffer, size_t n, const uint64_t *offsets, size_t nseg,
                           const rsx_layout *layout, int idx_bytes, void **result, rsx_report *report, void *stream) {
	if (idx_bytes == 0)
		return RSX_ERR_INVALID;
	return sort_segments_common(src, nullptr, index_buffer, idx_bytes, n, offsets, nseg, layout, result, report, stream);
}

// ---- top-k --------------------------------------------------------------------------------------
// Threshold search (key_bytes histogram launches, most of them returning at once for random keys),
// one stable select of the k records in front of the threshold, then the ordinary sort of those k
// records (rsx_topk.cu).  The search state, the per-chunk counts and the buffers around the sort of k
// records live in the stage lease; the sort itself uses the workspace lease.
static int topk_common(const void *src, size_t n, size_t k, const rsx_layout *layout, int idx_bytes, void *out,
                       rsx_report *rep, void *stream) {
	const bool ranksort = idx_bytes != 0;
	KeyDesc kd;
	int r = check_layout(layout, &kd); // records the tile kernels move directly: 1, 2, 4, 8 or 16 bytes
	if (r)
		return r;
	if (ranksort && !valid_idx_bytes(idx_bytes))
		return RSX_ERR_INVALID;
	if (k > n || (k > 0 && (!src || !out)))
		return RSX_ERR_INVALID;
	const uint32_t rb = layout->record_bytes;
	if (k > 0 && overlaps(src, n * rb, out, k * (ranksort ? (size_t)idx_bytes : rb))) // src is never written
		return RSX_ERR_INVALID;
	if (ranksort && !idx_fits(idx_bytes, n))
		return RSX_ERR_IDX_RANGE;
	if (rep)
		memset(rep, 0, sizeof(*rep));
	if (k == 0)
		return RSX_OK;
	int dev;
	if ((r = current_device(&dev)))
		return r;
	if ((r = check_residency(nullptr, src, out)))
		return r;
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	const unsigned long long l0 = g_launches.load();
	const int sms = g_dev[dev].num_sms;
	const TopkChunks g = topk_chunks(src, n, rb, sms);
	// positions of the selected records (rank form) and the ranks of their sort
	const int sel_ib = n - 1 <= 0xFFFFFFFFull ? 4 : 8, rank_ib = k - 1 <= 0xFFFFFFFFull ? 4 : 8;
	// stage: [state | chunk histograms | chunk lt | chunk eq | records | positions | 2k ranks]
	const size_t off_hist = align_up(sizeof(TopkState), 256);
	const size_t off_lt = off_hist + align_up((size_t)g.nchunks * kBins * sizeof(uint32_t), 256);
	const size_t off_eq = off_lt + align_up((size_t)g.nchunks * sizeof(unsigned long long), 256);
	const size_t off_rec = off_eq + align_up((size_t)g.nchunks * sizeof(unsigned long long), 256);
	const size_t off_pos = off_rec + align_up(k * rb, 256);
	const size_t off_ib = off_pos + (ranksort ? align_up(k * (size_t)sel_ib, 256) : 0);
	const size_t total = off_ib + (ranksort ? 2 * k * (size_t)rank_ib : 0);
	unsigned char *hbuf = nullptr;
	if ((r = thread_pinned_buffer(sizeof(uint32_t), &hbuf)))
		return r;
	Lease SL;
	if ((r = acquire(SL, dev, STAGE, total)))
		return r;
	SL.enqueued(st); // drained below on success, by ~Lease on any failure
	unsigned char *sp = static_cast<unsigned char *>(SL.ptr);
	TopkState *s = reinterpret_cast<TopkState *>(sp);
	auto *clt = reinterpret_cast<unsigned long long *>(sp + off_lt), *ceq = reinterpret_cast<unsigned long long *>(sp + off_eq);
	CU(cudaMemsetAsync(sp, 0, off_rec, st));
	for (int c = (int)kd.key_bytes - 1; c >= 0; --c)
		CU(launch_topk_hist(src, n, k, rb, kd, c, g, s, reinterpret_cast<uint32_t *>(sp + off_hist), clt, ceq, st));
	// value form: the selection goes straight to `out` and is sorted there, the stage buffer is aux
	void *sel = ranksort ? static_cast<void *>(sp + off_rec) : out;
	CU(launch_topk_select(src, n, k, rb, kd, g, s, clt, ceq, sel, ranksort ? sp + off_pos : nullptr, ranksort ? sel_ib : 0, st));
	CU(cudaMemcpyAsync(hbuf, &s->ncols, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
	void *res = nullptr;
	rsx_report srep;
	if (!ranksort) {
		if (k >= 2) {
			if ((r = sort_device(out, sp + off_rec, k, layout, kd, &res, &srep, st, dev, false)))
				return r;
			if (res != out)
				CU(cudaMemcpyAsync(out, res, k * rb, cudaMemcpyDeviceToDevice, st));
		}
	} else {
		if (k >= 2 && (r = rank_device(sel, sp + off_ib, k, layout, kd, rank_ib, &res, &srep, st, dev, false)))
			return r;
		CU(launch_topk_gather(res, rank_ib, sp + off_pos, sel_ib, out, idx_bytes, k, sms, st));
	}
	CU(cudaStreamSynchronize(st));
	SL.drained();
	Ctl c{};
	c.ncols = *reinterpret_cast<const uint32_t *>(hbuf); // the columns the threshold search histogrammed
	fill_report(rep, c, l0, false);
	if (rep)
		rep->result_in_aux = 0; // the k records are always in `out`
	return RSX_OK;
}

int rsx_topk(const void *src, size_t n, size_t k, const rsx_layout *layout, void *out, rsx_report *report, void *stream) {
	return topk_common(src, n, k, layout, 0, out, report, stream);
}

int rsx_topk_rank(const void *src, size_t n, size_t k, const rsx_layout *layout, int idx_bytes, void *index_out,
                  rsx_report *report, void *stream) {
	if (idx_bytes == 0)
		return RSX_ERR_INVALID;
	return topk_common(src, n, k, layout, idx_bytes, index_out, report, stream);
}

// ---- halves of the path, for parity tests and profiling ------------------------------------------
int rsx_histogram(const void *src, size_t n, const rsx_layout *layout, uint64_t *hist_out,
                  uint64_t *descents_out, rsx_report *rep, void *stream) {
	KeyDesc kd;
	int r = check_layout(layout, &kd);
	if (r)
		return r;
	if (!src || n < 2)
		return RSX_ERR_INVALID;
	DeviceCall C;
	if ((r = C.open(stream)) || (r = check_residency(nullptr, src)))
		return r;
	const unsigned long long l0 = g_launches.load();
	if ((r = C.lease(make_plan(n, layout->record_bytes, kd, 0))))
		return r;
	if ((r = enqueue_front(src, C.P, C.wsp, C.L.pinned, C.sms, C.st)))
		return r;
	rep = report_or_scratch(rep);
	if ((r = read_ctl(C.L, C.st, l0, rep, false)))
		return r;
	rep->live_mask = C.L.pinned->live_mask; // report the probe even when the input is presorted
	rep->ncols = C.L.pinned->ncols;
	if (hist_out && (r = C.read_back(C.ws->hist, sizeof(uint64_t) * kBins * kd.key_bytes, hist_out)))
		return r;
	if (descents_out && (r = C.read_back(&C.ws->descents, sizeof(uint64_t), descents_out)))
		return r;
	return RSX_OK;
}

int rsx_histogram_column(const void *src, size_t n, const rsx_layout *layout, int col, uint64_t *hist_out, void *stream) {
	KeyDesc kd;
	int r = check_layout(layout, &kd);
	if (r)
		return r;
	if (!src || !hist_out || n < 1 || col < 0 || col >= (int)kd.key_bytes)
		return RSX_ERR_INVALID;
	DeviceCall C;
	if ((r = C.open(stream)) || (r = check_residency(nullptr, src)))
		return r;
	// The digit of column `col` of the derived key is the derived key of a ONE-byte key at that
	// byte position: the top column keeps the sign / float flip (the sign bit lives in it), lower
	// columns are plain bytes; a complemented key complements every byte.
	KeyDesc k1 = kd;
	k1.key_shift = kd.key_shift + 8u * (uint32_t)col;
	k1.key_bytes = 1;
	if ((uint32_t)col + 1u != kd.key_bytes) {
		if (kd.kdf_kind == RSX_KDF_FLOAT)
			return RSX_ERR_INVALID; // a lower column of a float key depends on the sign in the top byte
		k1.kdf_kind = RSX_KDF_UNSIGNED;
	}
	if ((r = C.lease(head_plan(layout->record_bytes, k1))))
		return r;
	CU(zero_workspace(C.P, C.wsp, C.st));
	CU(launch_histogram(src, n, layout->record_bytes, k1, C.ws, C.sms, C.st));
	return C.read_back(C.ws->hist, sizeof(uint64_t) * kBins, hist_out);
}

int rsx_scatter_pass(const void *src, void *dst, const void *payload_src, void *payload_dst,
                     int payload_bytes, size_t n, const rsx_layout *layout, int col, void *stream) {
	KeyDesc kd;
	int r = check_layout(layout, &kd);
	if (r)
		return r;
	if (!src || !dst || n < 1 || col < 0 || col >= (int)kd.key_bytes)
		return RSX_ERR_INVALID;
	if (!(payload_bytes == 0 || payload_bytes == 4 || payload_bytes == 8))
		return RSX_ERR_INVALID;
	if (payload_bytes && (!payload_src || !payload_dst))
		return RSX_ERR_INVALID;
	DeviceCall C;
	if ((r = C.open(stream)) || (r = C.lease(make_plan(n, layout->record_bytes, kd, 0, payload_bytes))))
		return r;
	if ((r = enqueue_front(src, C.P, C.wsp, C.L.pinned, C.sms, C.st))) // histogram + scan give this column's offsets
		return r;
	PassBuffers pb{};
	pb.rec_first = src;
	pb.rec_buf[0] = dst;
	pb.rec_buf[1] = dst;
	pb.pl_first = payload_src;
	pb.pl_buf[0] = payload_dst;
	pb.pl_buf[1] = payload_dst;
	if ((r = run_scatter(pb, C.P, col, C.wsp, true, C.sms, C.st)))
		return r;
	return C.finish();
}

// ---- fused partition + exchange ------------------------------------------------------------------
// owner: contiguous bucket ranges, non-decreasing and < ndest.
static bool valid_owner(const uint8_t *owner, int ndest) {
	for (int b = 0; b < kBins; ++b)
		if (owner[b] >= ndest || (b && owner[b] < owner[b - 1]))
			return false;
	return true;
}

// Key-range routing (sample-sort style splitters) for skewed multi-GPU inputs.
static int check_splitters(const uint64_t *splitters, int nsplit) {
	if (!splitters || nsplit < 1 || nsplit > kMaxSplit)
		return RSX_ERR_INVALID;
	for (int j = 1; j < nsplit; ++j)
		if (splitters[j] < splitters[j - 1])
			return RSX_ERR_INVALID;
	return RSX_OK;
}

// With splitters, the "digit" of a record is its key range: range j goes to destination j.
static void splitter_owner(int nsplit, unsigned char owner[kBins]) {
	for (int b = 0; b < kBins; ++b)
		owner[b] = (unsigned char)(b <= nsplit ? b : nsplit);
}

// One exchange pass over column col (key ranges when splitters != nullptr), on a workspace the caller
// has prepared.  The HOST arrays dest_base and owner -- in append mode (dest_cursor != nullptr) also
// dest_cursor and dest_capacity -- are uploaded into the workspace head first; append mode reads back
// whether a run did not fit.
static int exchange_pass(DeviceCall &C, const void *src, int col, const uint8_t *owner, const uint64_t *dest_base, int ndest,
                         const uint64_t *splitters, int nsplit, const uint64_t *dest_cursor = nullptr,
                         const uint64_t *dest_capacity = nullptr, uint32_t *overflow_out = nullptr) {
	WsHead *ws = C.ws;
	const size_t dbytes = sizeof(uint64_t) * ndest;
	CU(cudaMemcpyAsync(ws->dest_base, dest_base, dbytes, cudaMemcpyHostToDevice, C.st));
	if (dest_cursor) {
		CU(cudaMemcpyAsync(ws->dest_cursor, dest_cursor, dbytes, cudaMemcpyHostToDevice, C.st));
		CU(cudaMemcpyAsync(ws->dest_capacity, dest_capacity, dbytes, cudaMemcpyHostToDevice, C.st));
	}
	CU(cudaMemcpyAsync(ws->owner, owner, kBins, cudaMemcpyHostToDevice, C.st));
	Exchange ex;
	ex.dest_base = ws->dest_base;
	ex.owner = ws->owner;
	ex.splitters = reinterpret_cast<const unsigned long long *>(splitters);
	ex.nsplit = nsplit;
	ex.ndest = ndest;
	if (dest_cursor) {
		ex.dest_cursor = ws->dest_cursor;
		ex.dest_capacity = ws->dest_capacity;
		ex.overflow = &ws->overflow;
	}
	PassBuffers pb{};
	pb.rec_first = src;
	int r = run_scatter(pb, C.P, col, C.wsp, true, C.sms, C.st, ex);
	if (r)
		return r;
	return overflow_out ? C.read_back(&ws->overflow, sizeof(uint32_t), overflow_out) : C.finish();
}

int rsx_scatter_pass_to(const void *src, size_t n, const rsx_layout *layout, int col,
                        const uint8_t *owner, const uint64_t *dest_base, int ndest, void *stream) {
	KeyDesc kd;
	int r = check_layout(layout, &kd);
	if (r)
		return r;
	if (!src || !owner || !dest_base || n < 1 || col < 0 || col >= (int)kd.key_bytes || ndest < 1 || ndest > kBins)
		return RSX_ERR_INVALID;
	if (!valid_owner(owner, ndest))
		return RSX_ERR_INVALID;
	DeviceCall C;
	if ((r = C.open(stream)) || (r = C.lease(make_plan(n, layout->record_bytes, kd, 0, 0))))
		return r;
	// no histogram needed: destinations get explicit base addresses; only the look-back state and
	// the tile ticket have to be zero (the caller already histogrammed this shard to route it)
	CU(zero_workspace(C.P, C.wsp, C.st));
	return exchange_pass(C, src, col, owner, dest_base, ndest, nullptr, 0);
}

int rsx_split_counts(const void *src, size_t n, const rsx_layout *layout, const uint64_t *splitters, int nsplit,
                     uint64_t *counts_out, void *stream) {
	KeyDesc kd;
	int r = check_layout(layout, &kd);
	if (r || (r = check_splitters(splitters, nsplit)))
		return r;
	if (!counts_out || (n && !src))
		return RSX_ERR_INVALID;
	DeviceCall C;
	if ((r = C.open(stream)))
		return r;
	for (int j = 0; j <= nsplit; ++j)
		counts_out[j] = 0;
	if (n == 0)
		return RSX_OK;
	// the counters live in the (zeroed) head of the cached workspace: no allocation per call
	if ((r = C.lease(head_plan(layout->record_bytes, kd))))
		return r;
	CU(zero_workspace(C.P, C.wsp, C.st));
	CU(launch_split_counts(src, n, layout->record_bytes, kd, reinterpret_cast<const unsigned long long *>(splitters),
	                       (uint32_t)nsplit, C.ws->hist, C.sms, C.st));
	return C.read_back(C.ws->hist, sizeof(uint64_t) * (nsplit + 1), counts_out);
}

int rsx_split_pass_to(const void *src, size_t n, const rsx_layout *layout, const uint64_t *splitters, int nsplit,
                      const uint64_t *dest_base, void *stream) {
	KeyDesc kd;
	int r = check_layout(layout, &kd);
	if (r || (r = check_splitters(splitters, nsplit)))
		return r;
	if (!src || !dest_base || n < 1)
		return RSX_ERR_INVALID;
	DeviceCall C;
	if ((r = C.open(stream)) || (r = C.lease(make_plan(n, layout->record_bytes, kd, 0, 0))))
		return r;
	// no histogram needed: destinations get explicit base addresses; only the look-back state and
	// the tile ticket have to be zero
	CU(zero_workspace(C.P, C.wsp, C.st));
	unsigned char owner[kBins];
	splitter_owner(nsplit, owner);
	return exchange_pass(C, src, 0, owner, dest_base, nsplit + 1, splitters, nsplit);
}

// Append-mode partition + exchange (keys-only records): like rsx_scatter_pass_to / rsx_split_pass_to,
// but a tile's run is placed where the destination's append cursor says instead of at an offset
// derived from exact per-source counts -- no routing histogram has to precede the pass.
int rsx_scatter_pass_append(const void *src, size_t n, const rsx_layout *layout, int col, const uint8_t *owner,
                            const uint64_t *splitters, int nsplit, const uint64_t *dest_base,
                            const uint64_t *dest_cursor, const uint64_t *dest_capacity, int ndest,
                            uint32_t *overflow_out, void *stream) {
	KeyDesc kd;
	int r = check_layout(layout, &kd);
	if (r)
		return r;
	if (!src || !dest_base || !dest_cursor || !dest_capacity || !overflow_out || n < 1 || ndest < 1 || ndest > kMaxSplit + 1)
		return RSX_ERR_INVALID;
	if (layout->record_bytes != kd.key_bytes)
		return RSX_ERR_INVALID; // append order is arbitrary: only where equal records are indistinguishable
	unsigned char split_owner[kBins];
	if (col >= 0) {
		if (!owner || col >= (int)kd.key_bytes || !valid_owner(owner, ndest))
			return RSX_ERR_INVALID;
		splitters = nullptr;
		nsplit = 0;
	} else {
		if ((r = check_splitters(splitters, nsplit)) || ndest != nsplit + 1)
			return r ? r : RSX_ERR_INVALID;
		splitter_owner(nsplit, split_owner);
		owner = split_owner;
		col = 0;
	}
	DeviceCall C;
	if ((r = C.open(stream)) || (r = C.lease(make_plan(n, layout->record_bytes, kd, 0, 0))))
		return r;
	CU(cudaMemsetAsync(C.ws, 0, kWsZeroBytes, C.st)); // ticket + overflow flag; no look-back state in this mode
	return exchange_pass(C, src, col, owner, dest_base, ndest, splitters, nsplit, dest_cursor, dest_capacity, overflow_out);
}

// `count` evenly spaced records' DERIVED keys (record i * (n / count)), HOST output: the sample the
// key-range splitters are quantiles of.  count <= 8192.
int rsx_sample_keys(const void *src, size_t n, const rsx_layout *layout, size_t count, uint64_t *derived_out, void *stream) {
	KeyDesc kd;
	int r = check_layout(layout, &kd);
	if (r)
		return r;
	if (!src || !derived_out || count < 1 || count > n || count > kMaxCols * kBins)
		return RSX_ERR_INVALID;
	DeviceCall C;
	if ((r = C.open(stream)) || (r = C.lease(head_plan(layout->record_bytes, kd))))
		return r;
	CU(launch_sample_keys(src, count, n / count, layout->record_bytes, kd, C.ws->offs, C.st)); // offs: 16 KB of scratch in the head
	return C.read_back(C.ws->offs, sizeof(uint64_t) * count, derived_out);
}

// The 256-bin histogram of one column over a SAMPLE of the records (every stride-th one): what
// the append-mode exchange balances its bucket ranges with.
int rsx_histogram_column_sampled(const void *src, size_t n, const rsx_layout *layout, int col, size_t stride,
                                 uint64_t *hist_out, void *stream) {
	KeyDesc kd;
	int r = check_layout(layout, &kd);
	if (r)
		return r;
	if (!src || !hist_out || n < 1 || stride < 1 || col < 0 || col >= (int)kd.key_bytes)
		return RSX_ERR_INVALID;
	DeviceCall C;
	if ((r = C.open(stream)) || (r = C.lease(head_plan(layout->record_bytes, kd))))
		return r;
	CU(zero_workspace(C.P, C.wsp, C.st));
	CU(launch_sample_column_hist(src, n, layout->record_bytes, kd, col, stride, C.ws->hist, C.sms, C.st));
	return C.read_back(C.ws->hist, sizeof(uint64_t) * kBins, hist_out);
}

// The key-compaction plan for given OR / NAND masks (pure host arithmetic; tests/test_abi.py checks
// it against a bit-level model without a device).  runs_out: up to 8 x {src_shift, width, dst_shift}.
// Returns the number of compacted passes (0: compaction would not pay) or a negative rsx_status.
int rsx_plan_compaction(uint64_t key_or, uint64_t key_nand, int key_bytes, int live_columns, uint32_t *runs_out,
                        uint64_t *const_bits_out) {
	if (!(key_bytes == 4 || key_bytes == 8) || live_columns < 0 || live_columns > key_bytes)
		return RSX_ERR_INVALID;
	Ctl c{};
	c.key_or = key_or;
	c.key_nand = key_nand;
	c.ncols = (uint32_t)live_columns;
	KeyDesc kd{};
	kd.key_bytes = (uint32_t)key_bytes;
	Compaction cmp{};
	if (!plan_compaction(c, kd, &cmp))
		return 0;
	if (runs_out)
		for (uint32_t i = 0; i < (uint32_t)kMaxRuns; ++i) {
			runs_out[3 * i] = i < cmp.nruns ? cmp.src_shift[i] : 0;
			runs_out[3 * i + 1] = i < cmp.nruns ? cmp.width[i] : 0;
			runs_out[3 * i + 2] = i < cmp.nruns ? cmp.dst_shift[i] : 0;
		}
	if (const_bits_out)
		*const_bits_out = cmp.const_bits;
	return (int)((cmp.bits + 7) / 8);
}

// ---- bench helpers ---------------------------------------------------------------------------------
int rsx_fill_keys(void *dst, size_t count, int key_bytes, uint64_t seed, uint64_t start, int dist,
                  uint64_t mask, uint64_t orv, void *stream) {
	if (!dst && count)
		return RSX_ERR_INVALID;
	if (count == 0)
		return RSX_OK;
	CU(launch_fill(dst, count, key_bytes, seed, start, dist, mask, orv, static_cast<cudaStream_t>(stream)));
	return RSX_OK;
}

int rsx_verify(const void *data, size_t n, const rsx_layout *layout, uint64_t *descents_out,
               uint64_t *sum_out, uint64_t *xor_out, void *stream) {
	KeyDesc kd;
	int r = check_layout(layout, &kd);
	if (r)
		return r;
	DeviceCall C;
	if ((r = C.open(stream)))
		return r;
	unsigned long long h3[3] = {0, 0, 0};
	if (n) { // the three accumulators live in the (zeroed) head of the cached workspace
		if ((r = C.lease(head_plan(layout->record_bytes, kd))))
			return r;
		CU(zero_workspace(C.P, C.wsp, C.st));
		CU(launch_verify(data, n, layout->record_bytes, kd, C.ws->hist, C.sms, C.st));
		if ((r = C.read_back(C.ws->hist, sizeof(h3), h3)))
			return r;
	}
	if (descents_out) *descents_out = h3[0];
	if (sum_out) *sum_out = h3[1];
	if (xor_out) *xor_out = h3[2];
	return RSX_OK;
}

} // extern "C"
