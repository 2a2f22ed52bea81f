/*
 * rsx.h -- C ABI of librsx.so: the B200 (sm_100a) LSD radix-sort hot path.
 *
 * This is the drop-in boundary.  The reference (eloj/radix-sorting) has no FFI: its surface
 * is two header-only C++ templates.  Each entry point below names the reference interface it
 * replaces; include/radix_sort.hpp, include/radix_sort_rank.hpp and
 * include/radix_sort_basic_kdf.hpp re-create the reference's template signatures on top of
 * these calls (see INTEGRATION.md for the binding a reference maintainer would add).
 *
 * Plain pointers and sizes only; no C++/torch types.  All functions return 0 (RSX_OK) or a
 * negative rsx_status; none of them has a CPU fallback -- without a CUDA device they fail
 * with RSX_ERR_NO_DEVICE / RSX_ERR_CUDA.
 */
#ifndef RSX_H
#define RSX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSX_VERSION 100 /* 0.1.0 */

typedef enum rsx_status {
	RSX_OK = 0,
	RSX_ERR_INVALID = -1,     /* bad layout / null pointer / unsupported combination        */
	RSX_ERR_CUDA = -2,        /* a CUDA runtime call failed (see rsx_last_cuda_error)        */
	RSX_ERR_NO_DEVICE = -3,   /* no CUDA device: there is no CPU path                         */
	RSX_ERR_WORKSPACE = -4,   /* caller workspace too small                                   */
	RSX_ERR_IDX_RANGE = -5,   /* n - 1 does not fit idx_bytes (reference would silently wrap) */
	RSX_ERR_MIXED_MEMORY = -6 /* src / aux / index_buffer not all host or all device          */
} rsx_status;

/* How the reference's KeyFunc (radix_sort.hpp:31-35) is expressed across a C ABI.
 * A device kernel cannot call a host lambda, so the key derivation is described, not passed:
 *   key      = key_bytes little-endian bytes at key_offset inside a record_bytes-sized record
 *   derived  = kdf(key), optionally complemented
 * which covers every KDF the reference ships or documents (radix_sort_basic_kdf.hpp:19-46,
 * README.md:562-627) and the record lambdas of its tests (radix_tests.cpp:41-43,111-113,175-177). */
typedef enum rsx_kdf {
	RSX_KDF_UNSIGNED = 0, /* identity                  radix_sort_basic_kdf.hpp:19-23 */
	RSX_KDF_SIGNED = 1,   /* key ^ highbit             radix_sort_basic_kdf.hpp:26-30 */
	RSX_KDF_FLOAT = 2     /* IEEE-754 total-order flip radix_sort_basic_kdf.hpp:32-46 (key_bytes 4 or 8) */
} rsx_kdf;

#define RSX_FLAG_INVERT 1u /* derived = ~derived: descending order, README.md:564-574 */

typedef struct rsx_layout {
	uint32_t record_bytes; /* sizeof(T): 1, 2, 4, 8 or 16                                 */
	uint32_t key_offset;   /* key must lie inside one aligned 8-byte word of the record   */
	uint32_t key_bytes;    /* sizeof(KeyType) = number of 8-bit columns: 1, 2, 4 or 8      */
	uint32_t kdf_kind;     /* rsx_kdf                                                      */
	uint32_t flags;        /* RSX_FLAG_*                                                   */
} rsx_layout;

/* What the sort found out on the device (read back once, 1 small D2H at the end). */
typedef struct rsx_report {
	uint32_t early_exit;   /* n < 2 or input already ordered: nothing was moved (radix_sort.hpp:60-62) */
	uint32_t ncols;        /* live (non-trivial) 8-bit columns actually sorted (radix_sort.hpp:65-70) */
	uint32_t live_mask;    /* bit c set <=> column c was live                               */
	uint32_t result_in_aux;/* 1 <=> result pointer is aux / index_buffer + n (radix_sort.hpp:89-92) */
	uint32_t kernel_launches; /* kernels launched by this call                             */
	uint32_t staged;       /* 1 <=> host buffers were staged through device memory         */
	uint32_t compacted_passes; /* != 0: key compaction ran -- the varying key bits were gathered and
	                              sorted in this many passes instead of ncols (README.md:716-758) */
} rsx_report;

/* ---- value sort --------------------------------------------------------------------------
 * Replaces  T* radix_sort(T* src, T* aux, size_t n, KeyFunc&& kf)      radix_sort.hpp:98-115
 *      and  rs_sort_main                                               radix_sort.hpp:31-93
 * src and aux hold n records each, both are clobbered, *result aliases one of them by the
 * reference's rule: src if the number of live columns is even or on early exit, else aux.
 * Device (or managed) pointers are sorted in place on the GPU; plain host pointers are
 * staged H2D -> sort -> D2H into the buffer the reference would have returned.
 * `stream` is a cudaStream_t (NULL = default stream).  The call is synchronous like the
 * reference: it returns after the result is complete.  `report` may be NULL. */
int rsx_sort(void *src, void *aux, size_t n, const rsx_layout *layout, void **result,
             rsx_report *report, void *stream);

/* ---- rank sort (argsort) -----------------------------------------------------------------
 * Replaces  IdxType* radix_sort_rank(const T* src, IdxType* index_buffer, size_t n, KeyFunc&&)
 *                                                                 radix_sort_rank.hpp:97-112
 *      and  rs_sort_rank                                          radix_sort_rank.hpp:22-92
 * src is never written.  index_buffer holds 2n entries of idx_bytes (1, 2, 4 or 8) each;
 * *result = index_buffer or index_buffer + n (same parity rule).  The output is the stable
 * argsort by derived key -- the semantics the reference documents (README.md:485-490) and
 * its C listing implements (radix_sort_u32_ranks.c:91-107); the shipped header deviates from
 * it for >= 2 live columns (radix_sort_rank.hpp:82, see DESIGN.md).  Keys travel beside the
 * indices in library workspace, so no pass gathers through the index. */
int rsx_sort_rank(const void *src, void *index_buffer, size_t n, const rsx_layout *layout,
                  int idx_bytes, void **result, rsx_report *report, void *stream);

/* ---- segmented sort: many independent arrays in one call ----------------------------------
 * No reference equivalent (the reference sorts one array per call); what CUB's segmented sort and
 * torch.sort(dim=-1) offer.  `offsets` holds nseg + 1 non-decreasing record offsets, offsets[0] == 0,
 * offsets[nseg] == n; segment s is records [offsets[s], offsets[s+1]).  It may be a HOST or a
 * DEVICE pointer (a device array is read back once); host offsets are checked before any device work.
 *   content  every segment ends up exactly as radix_sort / radix_sort_rank of that segment alone
 *            would leave it: stable by derived key, any KDF and RSX_FLAG_INVERT.  Rank indices are
 *            relative to the segment's start (what torch.sort(dim=-1) returns).
 *   result   ONE pointer for the batch, by the reference's parity rule applied to the batch: a column
 *            is live if its digit is not the same in all n records; *result is src (index_buffer) if
 *            the number of live columns is even, else aux (index_buffer + n).  A segment that is
 *            trivial in a column live for the batch still goes through that pass, which for a stable
 *            sort changes nothing.
 *   early    only if every segment is already ordered (descents across a segment boundary do not
 *            count): nothing moves and *result = src; a rank sort writes the segment-relative
 *            identity into the first half and *result = index_buffer.
 *   report   describes the batch (early_exit, ncols, live_mask, result_in_aux, kernel_launches).
 * src / aux / index_buffer must be device (or managed) memory (RSX_ERR_MIXED_MEMORY otherwise), record
 * sizes 1, 2, 4, 8 or 16 bytes (RSX_ERR_INVALID otherwise); idx_bytes must hold the longest segment's
 * length - 1 (RSX_ERR_IDX_RANGE).  n < 2 returns src without touching the device, as rsx_sort does
 * (a rank sort does what rsx_sort_rank does).  Synchronous like rsx_sort.  Short segments cost two
 * kernel launches per batch however many there are; a segment longer than one CTA holds is sorted
 * by the rsx_sort / rsx_sort_rank path on its own (DESIGN.md "Segmented sort"). */
int rsx_sort_segments(void *src, void *aux, size_t n, const uint64_t *offsets, size_t nseg,
                      const rsx_layout *layout, void **result, rsx_report *report, void *stream);
int rsx_sort_rank_segments(const void *src, void *index_buffer, size_t n, const uint64_t *offsets, size_t nseg,
                           const rsx_layout *layout, int idx_bytes, void **result, rsx_report *report, void *stream);

/* ---- the two halves of the path, exposed for parity tests and profiling --------------------
 * rsx_histogram = phase 1-3 of rs_sort_main (radix_sort.hpp:46-80): one read of the keys
 * producing all key_bytes x 256 digit counts (column-major, BEFORE the exclusive scan, bins
 * indexed by the DERIVED key's digit), the number of descents (i with kdf(a[i]) > kdf(a[i+1]);
 * the reference's n_unsorted equals 1 + descents for n >= 1) and the live-column mask.
 * `src` must be a device pointer; hist_out / descents_out / report are HOST pointers. */
int rsx_histogram(const void *src, size_t n, const rsx_layout *layout,
                  uint64_t *hist_out /* key_bytes*256 */, uint64_t *descents_out,
                  rsx_report *report, void *stream);

/* The 256-bin histogram of ONE column of the derived key (one shared-memory atomic per record
 * instead of key_bytes: the kernel then runs at HBM speed).  The multi-GPU sort routes on the top
 * column and does not need the others.  `src` device, `hist_out` host (256 entries).  Float keys:
 * top column only (a lower column's digit depends on the sign bit in the top byte). */
int rsx_histogram_column(const void *src, size_t n, const rsx_layout *layout, int col,
                         uint64_t *hist_out /* 256 */, void *stream);

/* One stable 8-bit-digit scatter pass (radix_sort.hpp:83-88) on column `col`, device
 * pointers only, unconditionally (no column skipping).  payload_* may be NULL; otherwise a
 * payload_bytes (4 or 8) lane is carried with the records. */
int rsx_scatter_pass(const void *src, void *dst, const void *payload_src, void *payload_dst,
                     int payload_bytes, size_t n, const rsx_layout *layout, int col, void *stream);

/* Fused partition + exchange for the multi-GPU sort (no reference equivalent; SURVEY.md §8e):
 * the same stable pass on column `col`, but the output goes to `ndest` destinations instead of
 * one dst: bucket d belongs to destination owner[d] (owner[] non-decreasing: contiguous bucket
 * ranges) and every tile appends ONE contiguous run per destination at byte address
 * dest_base[D] -- e.g. a peer GPU's receive buffer mapped over NVLink, so the all-to-all
 * costs no extra HBM pass and every remote store run is KiBs long.  Inside a destination the
 * records are in (tile, bucket, position) order: stable for equal keys, not grouped by bucket
 * across tiles (the receiver's LSD sort does not need that).  owner / dest_base are HOST
 * arrays (256 / ndest entries).  Returns after the pass has completed on this device;
 * cross-device visibility additionally needs a barrier between the ranks. */
int rsx_scatter_pass_to(const void *src, size_t n, const rsx_layout *layout, int col,
                        const uint8_t *owner, const uint64_t *dest_base, int ndest, void *stream);

/* Append-mode form of the two fused passes, for keys-only records (record_bytes == key_bytes): a
 * tile's run for destination D is placed where D's append cursor says -- one system-scope atomicAdd
 * on *dest_cursor[D] (a uint64 record count in D's memory, zeroed by its owner) -- instead of at an
 * offset derived from exact per-source counts, so no histogram pass has to precede it and the pass
 * needs no look-back.  The order in which runs land is arbitrary, which is invisible for keys-only
 * records.  col >= 0: destination = owner[digit]; col < 0: key ranges (splitters).  A run that would
 * exceed dest_capacity[D] records is dropped and *overflow_out set (src is only read: retry with
 * more room).  rsx_histogram_column_sampled counts one column over every stride-th record: the
 * estimate the bucket ranges are balanced with. */
int rsx_scatter_pass_append(const void *src, size_t n, const rsx_layout *layout, int col, const uint8_t *owner,
                            const uint64_t *splitters, int nsplit, const uint64_t *dest_base,
                            const uint64_t *dest_cursor, const uint64_t *dest_capacity, int ndest,
                            uint32_t *overflow_out, void *stream);
int rsx_histogram_column_sampled(const void *src, size_t n, const rsx_layout *layout, int col, size_t stride,
                                 uint64_t *hist_out /* 256 */, void *stream);
/* DERIVED keys of `count` (<= 2048) evenly spaced records, record i * (n / count): the sample the
 * key-range splitters are quantiles of.  `derived_out` is a HOST array. */
int rsx_sample_keys(const void *src, size_t n, const rsx_layout *layout, size_t count, uint64_t *derived_out, void *stream);

/* Key-range routing for skewed multi-GPU inputs (sample-sort style): `splitters` are nsplit
 * (<= 15) ascending DERIVED keys; a record's destination is the number of splitters <= its
 * derived key (0 .. nsplit).  rsx_split_counts counts the records per destination (HOST array of
 * nsplit + 1 entries); rsx_split_pass_to is the stable fused partition pass with that routing:
 * every tile appends one contiguous run per destination at byte address dest_base[D] (HOST array
 * of nsplit + 1 addresses: local or peer memory), records in input order inside a destination. */
int rsx_split_counts(const void *src, size_t n, const rsx_layout *layout, const uint64_t *splitters, int nsplit,
                     uint64_t *counts_out, void *stream);
int rsx_split_pass_to(const void *src, size_t n, const rsx_layout *layout, const uint64_t *splitters, int nsplit,
                      const uint64_t *dest_base, void *stream);

/* ---- multi-GPU partitioned sort (BASELINE config 5; SURVEY.md section 8e) ----------------------
 * No reference equivalent: eloj/radix-sorting is single-threaded host code.  This is the
 * MSD-then-LSD composition of the entry points above over the GPUs of one box: per-shard
 * histogram -> all-gather of the (columns x 256) counts -> routing of the top live digit's buckets
 * (or of key ranges, for skewed keys) to ranks -> ONE fused partition + exchange pass that stores
 * every record straight into its owner's receive buffer over NVLink -> local LSD sort.  The
 * concatenation of the shards' outputs in rank order is bit-identical to radix_sort() of the
 * concatenated input (stable across source ranks).
 *
 * The host orchestration is C++ inside librsx.so (csrc/rsx_multi.cu); the two collectives it needs
 * are callbacks, so it runs as one process with a thread per GPU (rsx_sort_multi) or as one process
 * per GPU under torchrun / MPI (rsx_sort_shard with the launcher's all-gather and barrier). */
#define RSX_MAX_RANKS 16

typedef struct rsx_comm {
	int rank, world;
	/* recv = world blocks of `bytes`, block g = rank g's `send`; HOST buffers */
	int (*allgather)(void *ctx, const void *send, void *recv, size_t bytes);
	/* every rank's device work issued so far is complete and visible to its peers */
	int (*barrier)(void *ctx);
	/* optional (non-fused exchange): DEVICE buffers, byte counts per peer, chunks in rank order */
	int (*alltoallv)(void *ctx, const void *send, const uint64_t *send_bytes, void *recv, const uint64_t *recv_bytes);
	void *ctx;
} rsx_comm;

/* Local primitives used by the orchestration.  NULL selects the CUDA kernels of this library; the
 * table exists so that the CPU test-suite can run the same host logic over gloo with oracle-backed
 * primitives (tests/test_dist.py) -- the product never substitutes them. */
typedef struct rsx_shard_ops {
	int (*hist)(void *ctx, const void *src, size_t n, const rsx_layout *L, uint64_t *hist /* key_bytes*256 */, void *stream);
	int (*sample)(void *ctx, const void *src, size_t n, const rsx_layout *L, size_t count, uint64_t *derived, void *stream);
	int (*split_counts)(void *ctx, const void *src, size_t n, const rsx_layout *L, const uint64_t *splitters, int nsplit,
	                    uint64_t *counts, void *stream);
	/* stable partition; destination D's records are appended at byte address dest_base[D].
	 * col >= 0: destination = owner[digit of column col]; col < 0: key ranges (splitters) */
	int (*partition_to)(void *ctx, const void *src, size_t n, const rsx_layout *L, int col, const uint8_t *owner,
	                    const uint64_t *splitters, int nsplit, const uint64_t *dest_base, int ndest, void *stream);
	int (*sort)(void *ctx, void *src, void *aux, size_t n, const rsx_layout *L, void **result, void *stream);
	void *ctx;
	/* optional: histogram of one column only (NULL: the orchestration always uses `hist`) */
	int (*hist_column)(void *ctx, const void *src, size_t n, const rsx_layout *L, int col, uint64_t *hist256, void *stream);
} rsx_shard_ops;

/* Routing decision, a pure function of the all-gathered histograms (identical on every rank). */
typedef struct rsx_route {
	int32_t routing_column;              /* highest globally-live column, -1: nothing to route   */
	uint32_t live_mask;                  /* columns that are not constant over all ranks          */
	uint32_t key_range;                  /* 1: bucket ranges cannot balance, use key-range splitters */
	uint32_t pad;
	uint8_t owner[256];                  /* bucket -> rank, non-decreasing                         */
	uint64_t n_in[RSX_MAX_RANKS];        /* shard sizes                                            */
	uint64_t send_counts[RSX_MAX_RANKS]; /* this rank -> rank d                                    */
	uint64_t recv_counts[RSX_MAX_RANKS]; /* rank g -> this rank                                    */
	uint64_t dest_offset[RSX_MAX_RANKS]; /* record offset of this rank's chunk inside rank d's receive buffer */
	uint64_t n_out, max_n_out, n_total;
	double imbalance;                    /* max_n_out / (n_total / world)                          */
} rsx_route;

typedef struct rsx_multi_report {
	int32_t routing_column;   /* -1: key-range routing or nothing routed */
	uint32_t key_range;       /* 1: routed by sample-based key ranges    */
	uint32_t live_mask;
	uint32_t fused;           /* 1: records went straight into peer memory */
	uint32_t append;          /* 1: keys-only append-mode exchange (sampled routing, no histogram pass) */
	uint32_t pad;
	uint64_t n_total;
	uint64_t needed_capacity; /* records each buffer must hold (valid also on RSX_ERR_WORKSPACE) */
	double imbalance;
	double seconds_histogram, seconds_routing, seconds_exchange, seconds_local_sort; /* host clock per phase */
} rsx_multi_report;

#define RSX_MULTI_NO_FUSED 1u     /* exchange through comm->alltoallv instead of peer stores */
#define RSX_MULTI_NO_KEY_RANGE 2u /* always route by bucket ranges (tests)                  */
#define RSX_MULTI_FULL_HISTOGRAM 4u /* count every column for routing, not just the top one (tests) */
#define RSX_MULTI_EXACT 8u        /* keys-only records too take the exact (histogram + offsets) exchange */
#define RSX_MULTI_APPEND 16u      /* keys-only records append even where the cursor contention heuristic says no */

int rsx_multi_route(const uint64_t *hist_all /* [world][cols][256] */, int world, int cols, int rank,
                    double skew_threshold, rsx_route *out);
int rsx_multi_splitters(const uint64_t *samples, size_t count, int world, uint64_t *splitters /* world-1 */);

/* One rank's view.  `src` holds this rank's n records, `recv` is this rank's receive buffer; both
 * hold `capacity` records and both are clobbered.  recv_peers[d] is rank d's receive buffer as
 * THIS rank can address it (peer mapping; recv_peers[rank] == recv), or NULL for the non-fused
 * exchange.  *result aliases src or recv and holds *n_out records.  If `capacity` is too small
 * for the routed sizes every rank returns RSX_ERR_WORKSPACE before anything is moved and
 * report->needed_capacity says what to allocate.  Collective: every rank must call it. */
int rsx_sort_shard(const rsx_comm *comm, const rsx_shard_ops *ops /* NULL = CUDA */, void *src, size_t n, void *recv,
                   void *const *recv_peers, size_t capacity, const rsx_layout *layout, uint32_t flags, void **result,
                   size_t *n_out, rsx_multi_report *report, void *stream);

/* One process, one host thread per GPU, peer access over NVLink.  src[g] / aux[g] live on
 * devices[g] and hold `capacity` records each; shard g has n[g] records in src[g].  On return
 * result[g] (src[g] or aux[g]) holds n_out[g] records.  reports: ngpus entries or NULL. */
int rsx_sort_multi(int ngpus, const int *devices, void *const *src, void *const *aux, const size_t *n,
                   size_t capacity, const rsx_layout *layout, uint32_t flags, void **result, size_t *n_out,
                   rsx_multi_report *reports);

/* ---- workspace ---------------------------------------------------------------------------
 * The reference allocates nothing (stack histograms).  The device path needs scratch for the
 * digit histograms, the pass table and the decoupled look-back state, and -- for rank sorts --
 * key/index ping-pong buffers.  By default it is a grow-only per-device cache owned by the
 * library; rsx_workspace_bytes lets a caller reserve it up front (rsx_reserve) so that no
 * cudaMalloc happens inside a timed region. */
size_t rsx_workspace_bytes(size_t n, const rsx_layout *layout, int rank_idx_bytes /* 0 = value sort */);
int rsx_reserve(size_t bytes);
void rsx_release(void);

/* ---- synthetic inputs for the benchmark (not on the sort path) ----------------------------
 * Device-side twin of keygen.py: dst[i] = ((dist(seed, start + i) & mask) | orv) truncated to
 * key_bytes, for i in [0, count). */
int rsx_fill_keys(void *dst, size_t count, int key_bytes, uint64_t seed, uint64_t start,
                  int dist, uint64_t mask, uint64_t orv, void *stream);

/* Device-side verification for inputs too large for a CPU oracle: number of descents of the
 * derived key over the array, plus order-independent multiset checksums (sum and xor of
 * mix64(record's first 8 bytes... of the derived key)).  Outputs are HOST pointers. */
int rsx_verify(const void *data, size_t n, const rsx_layout *layout, uint64_t *descents_out,
               uint64_t *sum_out, uint64_t *xor_out, void *stream);

/* The key-compaction plan (README.md:716-758) for the OR of all derived keys and the OR of their
 * complements: up to 8 runs {src_shift, width, dst_shift} of varying bits gathered into a narrower
 * key, and the constant bits.  Pure host arithmetic.  Returns the number of 8-bit passes the
 * compacted key needs, 0 if compaction would not pay, or a negative rsx_status. */
int rsx_plan_compaction(uint64_t key_or, uint64_t key_nand, int key_bytes, int live_columns,
                        uint32_t *runs_out /* 24 */, uint64_t *const_bits_out);

/* ---- misc -------------------------------------------------------------------------------- */
const char *rsx_strerror(int status);
const char *rsx_last_cuda_error(void); /* thread-local text of the last failing CUDA call */
int rsx_version(void);
uint64_t rsx_total_kernel_launches(void); /* process-wide count, for bench.py's gpu_launches */
/* Options: "rank_mode" (-1 auto [default]: per-device hardware probe picks the one-instruction
 * ticket ranking or the ballot ranking, 0 force ticket, 1 force ballot; DESIGN.md "K3");
 * "query_rank_mode" returns the mode in effect (0 / 1).  "scatter_variant" (0..5) selects a tile
 * geometry used in tuning sweeps, "force_wide" (0/1) runs the n >= 2^30 (64-bit offset) kernels
 * at any n (tests).  "compact_min_n": key compaction is considered for keys-only sorts of at least
 * this many 4/8-byte keys (default 2^26: below that the extra stream wait costs more than compaction can save; <= 0 disables it).  "profile" (0/1): bracket every kernel of rsx_sort / rsx_sort_rank with CUDA events on
 * the launch stream so that per-kernel device times can be read back with rsx_get_profile
 * (bench.py's roofline leg; off by default because the extra events perturb nothing but are
 * not free). */
int rsx_set_option(const char *name, long value);
/* Device time in ms of each kernel of the LAST profiled sort on this thread, in launch order:
 * [0] histogram (K1), [1] setup (K2), [2 + c] scatter pass of column c (0 if trivial/skipped).
 * Returns the number of entries written (<= cap), or a negative rsx_status. */
int rsx_get_profile(float *ms_out, int cap);

#ifdef __cplusplus
}
#endif
#endif /* RSX_H */
