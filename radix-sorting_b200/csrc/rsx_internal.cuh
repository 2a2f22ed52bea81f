// rsx_internal.cuh -- shared declarations between the kernels and the C-ABI host layer.
//
// Vocabulary follows the reference (eloj/radix-sorting): records with a key, 8-bit digit
// "columns" (radix_sort.hpp:40-44), a per-column 256-bin histogram, live vs trivial columns
// (radix_sort.hpp:65-70), src/aux ping-pong buffers (radix_sort.hpp:83-92).
#pragma once

#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

#include "rsx.h"

namespace rsx {

constexpr int kMaxCols = 8;     // sizeof(KeyType) <= 8, radix_sort.hpp:34
constexpr int kBins = 256;      // hist_len, radix_sort.hpp:42

// Where the key sits in a record, resolved once on the host (uniform kernel argument).
struct KeyDesc {
	uint32_t word_sel;   // which aligned 8-byte word of the record holds the key (16 B records)
	uint32_t key_shift;  // bit offset of the key inside that word (or inside the 1/2/4 B record)
	uint32_t key_bytes;  // number of columns
	uint32_t kdf_kind;   // rsx_kdf
	uint32_t invert;     // RSX_FLAG_INVERT
};

// Device-resident control block, written by the setup kernel, read by every scatter pass.
// This is the device-side form of `cols[] / ncols` + the early-exit test of
// radix_sort.hpp:60-70: the host never learns them before the passes are enqueued.
struct Ctl {
	uint32_t early_exit;            // descents == 0  <=>  n_unsorted < 2
	uint32_t ncols;                 // number of live columns
	uint32_t live_mask;             // bit c <=> column c live
	uint32_t ordinal[kMaxCols];     // index of column c among the live columns (if live)
	uint32_t pad;
	uint64_t n;
	// OR of all derived keys and OR of their complements (K1): bit b varies over the input iff it
	// is set in both.  The host reads them to decide on key compaction (README.md:716-758).
	unsigned long long key_or, key_nand;
};

// Key compaction (the reference README's "future work", README.md:716-758): bits of the derived key
// that are the same in every input key cannot influence the order, so the bits that DO vary are
// gathered (a software PEXT over <= kMaxRuns runs of contiguous bits) into a narrower key that
// needs fewer 8-bit passes; the last step scatters them back (PDEP) and restores the constant bits.
constexpr int kMaxRuns = 8;
struct Compaction {
	uint32_t nruns;                       // 0: no compaction
	uint32_t src_shift[kMaxRuns], width[kMaxRuns], dst_shift[kMaxRuns];
	unsigned long long wmask[kMaxRuns];   // (1 << width) - 1; 0 for unused runs (they then contribute nothing)
	unsigned long long const_bits;        // derived-key bits outside the runs (all constant)
	uint32_t bits;                        // total width of the compacted key
};

// Fixed-size head of the workspace.  Everything that must be zero before a sort comes first.
struct WsHead {
	unsigned long long hist[kMaxCols * kBins]; // raw digit counts per column (zeroed)
	unsigned long long descents;               // #i: kdf(a[i]) > kdf(a[i+1])       (zeroed)
	unsigned int tickets[kMaxCols];            // tile tickets, one per column      (zeroed)
	unsigned long long key_or, key_nand;       // see Ctl                            (zeroed)
	unsigned int overflow;                     // append-mode exchange: a run did not fit (zeroed)
	unsigned int pad0[1];
	// -- not zeroed below --
	unsigned long long offs[kMaxCols * kBins]; // exclusive scan per column (radix_sort.hpp:72-80)
	Ctl ctl;
	unsigned long long dest_base[kBins];       // fused partition + exchange: per-destination base address
	unsigned char owner[kBins];                // ... and the destination of every bucket
	unsigned long long dest_cursor[kBins];     // append mode: address of every destination's cursor ...
	unsigned long long dest_capacity[kBins];   // ... and the records it can take
};
constexpr size_t kWsZeroBytes = offsetof(WsHead, offs);

// Buffers of one scatter pass, selected on the device by the column's live ordinal j:
//   j == 0 : records from rec_first, payload from pl_first (or synthesised index)
//   j >= 1 : records from rec_buf[(j-1)&1], payload from pl_buf[(j-1)&1]
//   output : rec_buf[j&1], pl_buf[j&1]
// Value sort: rec_first = src, rec_buf = {aux, src}  -> the reference's swap(src, aux).
// Rank sort : rec_first = src (const), rec_buf = workspace pair, pl_buf = {ib + n, ib}.
struct PassBuffers {
	const void *rec_first;
	void *rec_buf[2];
	const void *pl_first;
	void *pl_buf[2];
	uint32_t synth_index;      // ordinal-0 payload = global element index
	uint32_t skip_last_rec;    // last live pass does not write records (rank sort)
};

struct PassGeometry {
	uint32_t threads, items, tile;   // tile = threads * items records
	size_t smem_bytes;
	int ctas_per_sm;
};

// ---- launchers (each returns the cudaError_t of the launch) ---------------------------------

// compact_out != nullptr (keys-only records): histogram the COMPACTED derived keys and write them
// to compact_out (record-sized unsigned values), see Compaction.
cudaError_t launch_histogram(const void *src, size_t n, uint32_t record_bytes, const KeyDesc &kd,
                             WsHead *ws, int num_sms, cudaStream_t st, const Compaction *cmp = nullptr,
                             void *compact_out = nullptr);
// compacted keys -> original keys (PDEP + constant bits + inverse key derivation); in == out allowed
cudaError_t launch_expand_keys(const void *in, void *out, size_t n, const KeyDesc &kd, const Compaction &cmp,
                               int num_sms, cudaStream_t st);

// host_ctl: mapped pinned mirror of ws->ctl (may be null)
cudaError_t launch_setup(const void *src, size_t n, uint32_t record_bytes, const KeyDesc &kd,
                         WsHead *ws, Ctl *host_ctl, cudaStream_t st);

// Fused partition + exchange (rsx_scatter_pass_to / rsx_split_pass_to / rsx_scatter_pass_append):
// device copies of the routing tables.  dest_base == nullptr: an ordinary pass.
struct Exchange {
	const unsigned long long *dest_base = nullptr; // one byte address per destination
	const unsigned char *owner = nullptr;          // the destination of every bucket
	const unsigned long long *splitters = nullptr; // HOST array: key-range routing instead of digits
	int nsplit = 0, ndest = 0;
	const unsigned long long *dest_cursor = nullptr, *dest_capacity = nullptr; // append mode
	unsigned int *overflow = nullptr;                                           // append mode
};

// status: look-back words for this column, tiles * 256 entries of 4 (n < 2^30) or 8 bytes, zeroed.
// ctl == nullptr: forced pass (ordinal 0, never skipped) for rsx_scatter_pass.
cudaError_t launch_scatter(const PassBuffers &pb, size_t n, uint32_t record_bytes, int payload_bytes,
                           const KeyDesc &kd, int col, const WsHead *ws_offsets /*offs + ctl*/,
                           bool forced, void *status, unsigned int *ticket, bool wide_offsets,
                           int num_sms, cudaStream_t st, const Exchange &ex);

PassGeometry scatter_geometry(uint32_t record_bytes, int payload_bytes);

// single-CTA path for inputs that fit one CTA's shared memory (rsx_small.cu)
size_t small_sort_capacity(uint32_t record_bytes, bool ranksort);
cudaError_t launch_small_sort(const void *src, void *out_even, void *out_odd, void *index_buffer, int idx_bytes,
                              size_t n, uint32_t record_bytes, const KeyDesc &kd, Ctl *ctl, cudaStream_t st);

// segmented sort (rsx_segments.cu).  A group is a run of consecutive non-empty segments that one CTA
// sorts: records [begin, begin + len) of the batch, nseg segments whose group-local starts are
// segtab[tab .. tab + nseg) followed by len.
constexpr uint32_t kMaxGroupSegments = 256; // the segment id is one 8-bit digit
struct SegGroup {
	unsigned long long begin;
	uint32_t len, nseg, tab, pad;
};
size_t segment_group_capacity(uint32_t record_bytes, bool ranksort);
// OR / NAND of the derived keys and the descents inside segments -> the batch pass table in ws->ctl
// (and host_ctl); ws's zeroed head must be clear.  offsets: nseg + 1 DEVICE entries.
cudaError_t launch_segment_prepass(const void *src, size_t n, uint32_t record_bytes, const KeyDesc &kd,
                                   const unsigned long long *offsets, size_t nseg, WsHead *ws, Ctl *host_ctl,
                                   int num_sms, cudaStream_t st);
cudaError_t launch_segment_groups(const void *src, void *out_even, void *out_odd, void *index_buffer, int idx_bytes, size_t n,
                                  uint32_t record_bytes, const KeyDesc &kd, const SegGroup *groups, size_t ngroups,
                                  const uint32_t *segtab, const Ctl *ctl, cudaStream_t st);

// top-k (rsx_topk.cu).  The threshold search is MSD radix select on the derived key: one histogram
// launch per column, from the top column down, over the records whose derived-key bits above the
// column equal `prefix`.  The last CTA of each launch picks the bucket that holds the k-th record and
// updates this block, so every launch is enqueued without the host waiting.  Zeroed before the search.
struct TopkState {
	unsigned long long hist[kBins]; // the current column's counts (reset by the deciding CTA)
	unsigned long long prefix;      // derived-key bits of columns col .. key_bytes-1 of the k-th record
	unsigned long long less;        // records whose derived key sorts below that prefix
	uint32_t ticket;                // CTAs done with the current column (reset by the deciding CTA)
	uint32_t done;                  // the prefix bucket holds exactly k - less records, or col == 0
	uint32_t ncols;                 // columns histogrammed
	uint32_t col;                   // the last column histogrammed
};
// Every top-k kernel of one call splits the records the same way: chunk j is a contiguous range, so
// per-chunk counts of the search passes give each CTA of the select its output offsets.  Records
// [0, head) go to chunk 0 and the tail that does not fill a 16-byte vector to the last chunk.
struct TopkChunks {
	size_t head, n_vec, per; // unaligned head records, 16-byte vectors after them, vectors per chunk
	uint32_t nchunks;
};
TopkChunks topk_chunks(const void *src, size_t n, uint32_t record_bytes, int num_sms);
// chunk_hist: nchunks x 256 counts of this column; chunk_lt / chunk_eq: per chunk, records below the
// prefix and records equal to it (zeroed before the search)
cudaError_t launch_topk_hist(const void *src, size_t n, size_t k, uint32_t record_bytes, const KeyDesc &kd, int col,
                             const TopkChunks &g, TopkState *s, uint32_t *chunk_hist, unsigned long long *chunk_lt,
                             unsigned long long *chunk_eq, cudaStream_t st);
// out[0, less): records below the prefix in input order; out[less, k): the first k - less records
// equal to it.  sel_idx_bytes 4 or 8: each record's input position goes to sel_idx; 0: none.
cudaError_t launch_topk_select(const void *src, size_t n, size_t k, uint32_t record_bytes, const KeyDesc &kd, const TopkChunks &g,
                               const TopkState *s, const unsigned long long *chunk_lt, const unsigned long long *chunk_eq,
                               void *out, void *sel_idx, int sel_idx_bytes, cudaStream_t st);
// index_out[i] = sel_idx[rank[i]] (rank == nullptr: sel_idx[i]), narrowed to idx_bytes
cudaError_t launch_topk_gather(const void *rank, int rank_bytes, const void *sel_idx, int sel_idx_bytes, void *index_out,
                               int idx_bytes, size_t k, int num_sms, cudaStream_t st);

// rank-sort helpers
cudaError_t launch_iota_if_early(void *index_buffer, int idx_bytes, size_t n, const Ctl *ctl,
                                 cudaStream_t st);
cudaError_t launch_narrow_index(const uint32_t *wide0, const uint32_t *wide1, void *index_buffer,
                                int idx_bytes, size_t n, const Ctl *ctl, cudaStream_t st);

cudaError_t launch_sample_keys(const void *data, size_t count, size_t stride, uint32_t record_bytes, const KeyDesc &kd,
                               unsigned long long *d_out, cudaStream_t st);
cudaError_t launch_sample_column_hist(const void *data, size_t n, uint32_t record_bytes, const KeyDesc &kd, int col, size_t stride,
                                      unsigned long long *d_hist, int num_sms, cudaStream_t st);

// records of any size: key extraction + final gather around a rank sort of the keys
cudaError_t launch_extract_keys(const void *recs, size_t n, uint32_t record_bytes, uint32_t key_offset, uint32_t key_bytes,
                                void *keys_out, int num_sms, cudaStream_t st);
cudaError_t launch_gather_records(const void *src, const void *rank, int idx_bytes, void *dst, size_t n, uint32_t record_bytes,
                                  int num_sms, cudaStream_t st);

// key-range routing counts (h_split: HOST array of nsplit splitters; d_counts: 16 zeroed device entries)
cudaError_t launch_split_counts(const void *data, size_t n, uint32_t record_bytes, const KeyDesc &kd,
                                const unsigned long long *h_split, uint32_t nsplit, unsigned long long *d_counts,
                                int num_sms, cudaStream_t st);

// hardware probe for the ticket ranking (see rsx_scatter.cuh); *d_mismatch must be zeroed
cudaError_t launch_ticket_probe(unsigned long long *d_mismatch, int num_sms, cudaStream_t st);

// bench / verification helpers
cudaError_t launch_fill(void *dst, size_t count, int key_bytes, uint64_t seed, uint64_t start,
                        int dist, uint64_t mask, uint64_t orv, cudaStream_t st);
cudaError_t launch_verify(const void *data, size_t n, uint32_t record_bytes, const KeyDesc &kd,
                          unsigned long long *out3 /*descents,sum,xor (zeroed)*/, int num_sms,
                          cudaStream_t st);

void count_launch(unsigned n = 1);

} // namespace rsx
