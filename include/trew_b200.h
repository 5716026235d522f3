/*
 * trew_b200.h -- C ABI of the B200-native TREW hot path (libtrew_b200.so).
 *
 * The reference (Chemical118/TREW) has no plugin/FFI layer.  The seam this library replaces is the
 * worker side of its single-producer / multi-consumer queue:
 *
 *   in : QueueData{char* buffer; LocationVector* loc_vector}  (src/kmer.h:93-96) and PairQueueData
 *        (src/kmer.h:98-103), produced by read_fastq_thread / read_pair_fastq_thread /
 *        read_fastq_long_thread (src/kmer.cpp:987-1213) and consumed by
 *   op : buffer_task / buffer_task_pair / buffer_task_long (src/kmer.h:206-212, src/kmer.cpp:80-985)
 *   out: ResultMapData = six maps (int k, uint128 seq) -> uint32 (src/kmer.h:65-81), summed over
 *        workers in process_output (src/kmer.cpp:1486-1515).
 *
 * Everything is plain C: pointers, sizes, integer status codes.  No C++ or torch types cross the line.
 * All device work is hand-written CUDA for sm_100a; there is NO CPU fallback: every entry point that
 * needs the GPU fails with TREW_ERR_CUDA when no device is usable.
 */
#ifndef TREW_B200_H
#define TREW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TREW_ABI_VERSION 2

/* status codes (the reference prints a message and exit(1)s instead; src/kmer.cpp:85-86, 1007-1008) */
#define TREW_OK 0
#define TREW_ERR_ARG 1        /* bad argument / configuration                                   */
#define TREW_ERR_CUDA 2       /* CUDA runtime failure or no usable device                        */
#define TREW_ERR_TABLE_FULL 3 /* device count table overflowed within one batch (raise table_log2_slots) */
#define TREW_ERR_TOO_LONG 4   /* short mode: read longer than MAX_SEQ=1000 (src/kmer.cpp:1006);  */
                              /* paired mode: mate longer than 1023 (one warp's window)          */
#define TREW_ERR_IO 5         /* file open / read failure (src/kmer.cpp:1021, 1288)              */
#define TREW_ERR_PAIRING 6    /* paired files disagree (src/kmer.cpp:1111-1123)                  */
#define TREW_ERR_NOMEM 7

/* which buffer_task* the context stands in for */
#define TREW_MODE_SHORT 0 /* buffer_task       src/kmer.cpp:80  */
#define TREW_MODE_PAIR 1  /* buffer_task_pair  src/kmer.cpp:268 */
#define TREW_MODE_LONG 2  /* buffer_task_long  src/kmer.cpp:747 */

/* table ids of the six result maps, FinalData<ResultMapPair> order (src/kmer.h:65-81) */
#define TREW_TABLE_FORWARD_HIGH 0
#define TREW_TABLE_FORWARD_LOW 1
#define TREW_TABLE_BACKWARD_HIGH 2
#define TREW_TABLE_BACKWARD_LOW 3
#define TREW_TABLE_BOTH_HIGH 4
#define TREW_TABLE_BOTH_LOW 5

/* Replaces the reference's mutable globals (src/trew.cpp:10-20, src/kmer.h:55-63). */
typedef struct trew_config {
    int32_t mode;             /* TREW_MODE_*                                                       */
    int32_t min_mer;          /* MIN_MER  >= 3                                                     */
    int32_t max_mer;          /* MAX_MER  <= 64; > 32 switches to 128-bit repeat units             */
    int32_t slice_length;     /* SLICE_LENGTH (long mode, default 150, >= 2*MAX_MER, <= 512 here)  */
    double low_baseline;      /* LOW_BASELINE  (-L, default 0.5)                                   */
    double high_baseline;     /* HIGH_BASELINE (-H, default 0.8)                                   */
    int32_t device;           /* CUDA device ordinal                                               */
    int32_t table_log2_slots; /* initial device count-table capacity, 0 = default (2^22 slots); the
                                 streaming path grows it when it passes a quarter full          */
    int32_t n_staging;        /* pinned staging buffers (double buffering = 2), 0 = default (3)    */
    int32_t host_threads;     /* host packing threads, 0 = all cores (capped at 32)                 */
    uint64_t staging_bytes;   /* bytes per staging buffer, 0 = default (64 MiB)                    */
} trew_config;

/*
 * A packed batch: reads as length-delimited planar 2-bit codes.
 *   bit_off[n_reads + 1]  start of every read in BASES inside the plane streams; read r occupies
 *                          bases [bit_off[r], bit_off[r+1]) (tightly packed, no per-read padding)
 *   hi / lo               the two bit-planes of the reference's 2-bit code T=0 G=1 C=2 A=3
 *                          (codes[], src/kmer.cpp:14-31): base j is bit (j & 31) of word (j >> 5)
 *   val                   validity plane: 1 for ACGTacgt, 0 for every other byte (N, '\r', ...);
 *                          invalid bases still count toward the read length, as in the reference
 * In TREW_MODE_PAIR reads 2u and 2u+1 are the two mates of pair u.  Plane arrays must be padded with
 * at least TREW_PLANE_PAD_WORDS zero words past word (bit_off[n_reads] >> 5).
 * Algorithmic bytes per read of length L: 4 + 3 * L / 8  (60.25 B at L = 150).
 */
#define TREW_PLANE_PAD_WORDS 40
typedef struct trew_batch {
    uint32_t n_reads;
    uint32_t max_read_len; /* at least the longest read in the batch: it sizes the exact kernel's
                            * workspace, the long-read scratch and the filter variant.  Larger is
                            * allowed (a larger workspace); smaller is TREW_ERR_ARG.                */
    const uint32_t* bit_off;
    const uint32_t* hi;
    const uint32_t* lo;
    const uint32_t* val;
} trew_batch;

/* One (table, k, seq) -> count entry of the merged result maps.  seq is the reference's KmerSeq.second
 * (first base in the most significant of 2k bits), split into two 64-bit halves. */
typedef struct trew_entry {
    uint64_t seq_lo;
    uint64_t seq_hi;
    uint64_t count;
    int32_t table; /* TREW_TABLE_* */
    int32_t k;
} trew_entry;

typedef struct trew_stats {
    uint64_t reads;        /* reads submitted                                                     */
    uint64_t bases;        /* bases submitted (all bytes of every sequence line)                  */
    uint64_t units;        /* reads (short/long) or pairs                                         */
    uint64_t survivors;    /* units the filter kernel sent to the exact kernel                     */
    uint64_t kernel_launches;
    uint64_t h2d_bytes;
    uint64_t d2h_bytes;
    double device_ms;      /* CUDA-event time of all scan kernels so far                          */
    uint64_t host_pack_bytes; /* ASCII bases the host packer turned into planes (streaming path)   */
    double host_pack_ms;   /* wall time the submitting thread spent in the packer (all pool threads busy) */
} trew_stats;

typedef struct trew_ctx trew_ctx;

/* ---- life cycle ------------------------------------------------------------------------------ */
int trew_abi_version(void);
const char* trew_status_string(int status);

/* Creates the device context: count table, staging buffers, streams.  Stands in for thread start +
 * ThreadData::init_check (src/kmer.h:139-153, src/kmer.cpp:1278-1282). */
int trew_dev_create(const trew_config* cfg, trew_ctx** out);
void trew_dev_destroy(trew_ctx* ctx);
/* Message of the last failed call on ctx; with ctx == NULL, of the calling thread's last failed trew_dev_create
 * (e.g. the SLICE_LENGTH <= 512 limit of the GPU path). */
const char* trew_dev_last_error(const trew_ctx* ctx);

/* ---- input: the QueueData side (src/kmer.h:93-103) --------------------------------------------- */

/* Push one raw chunk exactly as the reference's reader threads produce it: `buffer` holds text and
 * `locs` the inclusive (st, nd) byte offsets of n sequence lines (LocationVector, src/kmer.h:73).
 * The library packs it (host threads), stages it in pinned memory and launches the scan
 * asynchronously; the caller's memory may be reused as soon as the call returns.
 * For TREW_MODE_PAIR pass both mates' chunks; pairs are matched index-wise up to min(n1, n2)
 * (src/kmer.cpp:321-322).  buffer2/locs2 must be NULL/0 otherwise. */
int trew_dev_submit_chunk(trew_ctx* ctx, const char* buffer1, const int32_t* locs1, uint32_t n1,
                          const char* buffer2, const int32_t* locs2, uint32_t n2);

/* Check a packed batch for the context's mode before anything is copied or launched (trew_dev_submit_packed and
 * trew_dev_upload call it first).  TREW_ERR_ARG when bit_off[0] != 0, when bit_off decreases, when a paired batch has
 * an odd n_reads, or when max_read_len is smaller than the longest read.  TREW_ERR_TOO_LONG, as trew_dev_submit_chunk
 * gives it, for a short read above 1000 bases or a paired mate above 1023.  Long mode has no length limit.
 * The message of a failure goes to the context's trew_dev_last_error; called alone, only the status is returned. */
int trew_check_batch(int mode, const trew_batch* batch);

/* Push an already packed batch held in host memory (copied into pinned staging, then H2D).  The batch is checked
 * with trew_check_batch first. */
int trew_dev_submit_packed(trew_ctx* ctx, const trew_batch* batch);

/* ---- input: device-resident batches (benchmarking the scan alone) ------------------------------ */
typedef struct trew_resident trew_resident;
/* Copies a packed batch to device memory for trew_dev_scan_resident; checked with trew_check_batch first. */
int trew_dev_upload(trew_ctx* ctx, const trew_batch* batch, trew_resident** out);
int trew_dev_scan_resident(trew_ctx* ctx, const trew_resident* batch); /* async on the ctx stream */
void trew_dev_free_resident(trew_ctx* ctx, trew_resident* batch);
/* CUDA-event time (ms) of the last trew_dev_scan_resident; waits for it to complete. */
int trew_dev_last_resident_ms(trew_ctx* ctx, float* ms);

/* Benchmark tooling: fill a device-resident batch with synthetic fixed-length reads of BASELINE.json's
 * configs[1] shape (uniform ACGT; tel_ppm of the reads (TTAGGG)^n at random phase, half of them
 * reverse-complemented, sub_ppm per-base substitutions; half_ppm reads telomeric in one half only; n_ppm of
 * all bases invalid).  Counter-based generator, mirrored bit-for-bit by trew_b200/synth.py:device_mirror so
 * parity can be checked on small n.  Not part of the scan path. */
int trew_synth_resident(trew_ctx* ctx, uint64_t seed, uint32_t n_reads, uint32_t read_len, uint32_t tel_ppm,
                        uint32_t half_ppm, uint32_t n_ppm, uint32_t sub_ppm, trew_resident** out);

/* The same generator for the other BASELINE.json shapes: flavor 0 = single reads (as above); 1 = pairs (reads 2u and
 * 2u+1 are the two ends of one fragment: both telomeric or neither, mate 2 on the opposite strand; configs[2]);
 * 2 = long reads whose first or last 500-5000 bases are telomeric (tel_ppm of the reads; configs[3]). */
int trew_synth_resident_ex(trew_ctx* ctx, uint64_t seed, uint32_t n_reads, uint32_t read_len, uint32_t tel_ppm,
                           uint32_t half_ppm, uint32_t n_ppm, uint32_t sub_ppm, uint32_t flavor, trew_resident** out);

/* CUDA-event stopwatch on the context's scan stream (for device-resident scans). */
int trew_dev_timer_start(trew_ctx* ctx);
int trew_dev_timer_stop(trew_ctx* ctx, float* ms); /* waits for the stream */
/* Per-kernel CUDA-event times (ms) accumulated over resident scans since the last call -- screen kernel, decide
 * kernel, exact kernel -- and the number of scans they cover. */
int trew_dev_kernel_times(trew_ctx* ctx, double* screen_ms, double* decide_ms, double* exact_ms, uint64_t* n_scans);

/* ---- output: the ResultMapData side (src/kmer.h:79-81, src/kmer.cpp:1486-1515) ------------------ */

/* Wait for all submitted work (end-of-stream; replaces the {nullptr,nullptr} sentinels,
 * src/kmer.cpp:1304-1310). */
int trew_dev_sync(trew_ctx* ctx);

/* Drain, compact the device table and return the six maps as one array sorted by (table, k, seq).
 * The array (pinned host memory) is owned by the context and valid until the next call that touches the tables. */
int trew_dev_finish(trew_ctx* ctx, const trew_entry** entries, uint64_t* n_entries);

/* Device-side view of the same entries (compacted and sorted on the device): n entries in device memory, owned by
 * the context and valid until the next call that touches the tables. */
int trew_dev_export_device(trew_ctx* ctx, const trew_entry** d_entries, uint64_t* n_entries);

/* Cross-rank merge (one process per GPU): copy the compacted table (trew_entry rows, 32 bytes each) into
 * caller-owned DEVICE memory -- e.g. the buffer of an NCCL gather -- and add rows received from another rank to this
 * context's table.  Integer sums, hence exact; this is the multi-GPU form of the per-worker map sum in
 * process_output (src/kmer.cpp:1486-1515).  trew_dev_export_rows with d_rows == NULL only reports the row count; its
 * rows are in no particular order.  trew_dev_merge_rows is asynchronous: the rows must stay valid until the next
 * trew_dev_sync / trew_dev_finish / export on this context, which also reports a table overflow. */
int trew_dev_export_rows(trew_ctx* ctx, trew_entry* d_rows, uint64_t capacity_rows, uint64_t* n_rows);
int trew_dev_merge_rows(trew_ctx* ctx, const trew_entry* d_rows, uint64_t n_rows);
/* End of file on the merging rank: the union of this context's table and the other ranks' rows (device pointers, as
 * written by trew_dev_export_rows on those ranks and moved here by an NCCL gather) -- concatenated, sorted by
 * (table, k, seq) and equal keys summed on the device, then copied to the host like trew_dev_finish.  The context's own
 * table is left as it is. */
int trew_dev_finish_merged(trew_ctx* ctx, const trew_entry* const* d_lists, const uint64_t* n_rows, uint32_t n_lists,
                           const trew_entry** entries, uint64_t* n_entries);
/* Report filter.  With min_total > 0, trew_dev_finish / trew_dev_finish_merged copy to the host only the rows that can
 * reach the report of a ONE-FILE run: a row's group is (k, min(seq, canonical rotation of its reverse complement)) --
 * every forward / backward / both count of one report entry comes from one group (src/kmer.cpp:1518-1549) -- and the
 * group is kept when its high-class or its low-class total reaches min_total.  With min_total = 10 (ABS_MIN_PRINT_COUNT,
 * the print and scoring threshold, src/kmer.cpp:1615-1620, 2693-2761) trew_report_add_file + trew_report_finish print
 * exactly what they print from the full tables, while the one- and two-window repeats that N-bearing reads leave behind
 * (most rows of a large file, exactly as in the reference) stay on the device.  Runs over several files must keep 0:
 * entries below the threshold still add up across files (src/trew.cpp:454-467).  0 (default) = no filter. */
int trew_dev_set_report_filter(trew_ctx* ctx, uint32_t min_total);
/* Make room for about expected_new_keys more distinct keys (grows and re-hashes the table when it would pass a
 * quarter full).  Call before merging other ranks' rows. */
int trew_dev_reserve(trew_ctx* ctx, uint64_t expected_new_keys);

/* ---- per-unit hit records: which unit put each count into the six tables ----------------------------------------------
 *
 * A unit is what the routing handles: one read (short and long mode) or one pair (paired mode).  A unit's records are the
 * adds the reference's routing (buffer_task*) makes into the six final maps for that unit (the temp maps resolved), with
 * adds to the same (table, k, seq) within the unit merged.  Summed over all units, the records give back the tables of
 * trew_dev_finish (without the report filter, which records do not follow).
 *
 * The ordinal of a unit is its 0-based position among all units submitted to the context since create or reset, in call
 * order, whatever the entry point: trew_dev_submit_chunk, trew_dev_submit_packed and trew_dev_scan_resident all count.
 * trew_dev_process_file numbers the FASTQ records (pairs of records) of the file: after create or reset, the ordinal is the
 * 0-based index of the record in the file (sequence line 4i + 2 for ordinal i).  Records the reader drops count too: in long
 * mode the reads shorter than SLICE_LENGTH are kept and passed to the scan when records are on (they emit nothing, and
 * trew_dev_get_stats counts them as reads).  Not supported on the one-process-per-GPU merge path (trew_dev_export_rows /
 * trew_dev_merge_rows / trew_dev_finish_merged): merged rows have no unit. */
typedef struct trew_unit_record { /* 32 bytes */
    uint64_t unit;                  /* ordinal, see above                                                   */
    uint64_t seq_lo, seq_hi;        /* the key exactly as added to the table (folded where the table is)    */
    uint32_t count;
    uint8_t table;                  /* TREW_TABLE_*                                                         */
    uint8_t k;
    uint16_t reserved;              /* 0                                                                    */
} trew_unit_record;

/* Record up to capacity_records records (32 bytes each, device memory) from now on; 0 switches recording off.  Only
 * valid while the table is empty -- after create or reset -- TREW_ERR_ARG otherwise.  The appends keep counting past the
 * capacity: nothing is lost silently (see trew_dev_unit_records), and the tables are not affected. */
int trew_dev_enable_unit_records(trew_ctx* ctx, uint64_t capacity_records);
/* Wait for all submitted work and return the records sorted by (unit, table, k, seq_hi, seq_lo), one row per key and
 * unit.  The array (pinned host memory) belongs to the context and stays valid until the next call that touches the
 * tables.  TREW_ERR_TABLE_FULL when more records were made than the capacity holds; trew_dev_last_error then names the
 * capacity that would have been enough. */
int trew_dev_unit_records(trew_ctx* ctx, const trew_unit_record** recs, uint64_t* n);

/* Zero the count table (start of a new file; the reference allocates fresh maps per file,
 * src/kmer.cpp:89).  Also clears the unit records and restarts the unit ordinals at 0. */
int trew_dev_reset(trew_ctx* ctx);
int trew_dev_get_stats(trew_ctx* ctx, trew_stats* out);

/* ---- several GPUs in one process: the consumer fan-out of process_kmer* (src/kmer.cpp:1271-1325) --------------------
 *
 * The reference starts NUM_THREAD consumers on one queue and sums their maps at the end (src/kmer.cpp:1486-1515).  A
 * trew_multi is the same thing with GPUs as the consumers: one trew_ctx per device, one host packing pool shared by all
 * of them, chunks dealt round-robin (the two mates of a pair always travel together, reads are independent --
 * src/kmer.cpp:111, 322, 785), and at end of file the devices' compacted tables are copied to the first device over
 * NVLink (cudaMemcpyPeerAsync) and united there exactly (sort by key, integer sums) before one D2H copy.
 * devices == NULL or n_devices == 0: every visible device (a device listed k times gets k contexts).  cfg->device is ignored; cfg->host_threads sizes the shared
 * pool (0 = all cores).  All calls on one group must come from one thread at a time. */
typedef struct trew_multi trew_multi;
int trew_multi_create(const trew_config* cfg, const int32_t* devices, int32_t n_devices, trew_multi** out);
void trew_multi_destroy(trew_multi* m);
int trew_multi_device_count(const trew_multi* m);
const char* trew_multi_last_error(const trew_multi* m);
int trew_multi_submit_chunk(trew_multi* m, const char* buffer1, const int32_t* locs1, uint32_t n1, const char* buffer2,
                            const int32_t* locs2, uint32_t n2);
int trew_multi_process_file(trew_multi* m, const char* file1, int is_gz1, const char* file2, int is_gz2);
int trew_multi_reset(trew_multi* m);
/* Drain every device, merge, return the six maps sorted by (table, k, seq) like trew_dev_finish (the array belongs to
 * the group and is valid until the next call that touches the tables). */
int trew_multi_finish(trew_multi* m, const trew_entry** entries, uint64_t* n_entries);
/* trew_dev_enable_unit_records / trew_dev_unit_records for the group.  The group assigns the ordinals in its own
 * submission order (trew_multi_submit_chunk calls, across the round-robin dealing; trew_multi_process_file numbers
 * the file's records as trew_dev_process_file does), and the devices' records are united on the first device.  trew_multi_reset
 * clears them and restarts the ordinals at 0. */
int trew_multi_enable_unit_records(trew_multi* m, uint64_t capacity_records);
int trew_multi_unit_records(trew_multi* m, const trew_unit_record** recs, uint64_t* n);
/* trew_dev_set_report_filter for the group's merged result. */
int trew_multi_set_report_filter(trew_multi* m, uint32_t min_total);
/* Sums over the group's contexts (device_ms: the largest). */
int trew_multi_get_stats(trew_multi* m, trew_stats* out);
/* The context of the i-th device of the group (e.g. for device-resident batches); owned by the group. */
trew_ctx* trew_multi_ctx(trew_multi* m, int32_t i);

/* ---- host packer: ASCII -> planar 2-bit (codes[], src/kmer.cpp:14-31) ---------------------------- */

/* Bytes a packed batch of n_reads reads with total_bases bases needs (offsets + three planes + pad). */
size_t trew_pack_bound(uint32_t n_reads, uint64_t total_bases);

/* Pack n reads given as (st, nd) inclusive offsets into `buffer` into caller memory `dst` (8-byte aligned) of at
 * least trew_pack_bound bytes; fills *out with pointers into dst.  Single-threaded building block. */
int trew_pack_reads(const char* buffer, const int32_t* locs, uint32_t n, void* dst, size_t dst_bytes,
                    trew_batch* out);

/* The same batch, packed the way trew_dev_submit_chunk fills a staging slot: the reads are cut into n_ranges
 * consecutive ranges that n_threads host threads pack concurrently (a range may start in the middle of a plane
 * word; the shared words are stitched afterwards).  With inv != NULL the bit positions of the bases that are not
 * A/C/G/T (the zero bits of the val plane below bit_off[n]) are also listed, in no particular order: *n_inv is
 * their number, and at most inv_cap of them are stored.  The streaming path sends this list instead of the val
 * plane when it is short, and then does not write the plane either: TREW_PACK_NO_VAL in `flags` (needs inv) asks
 * for the same -- the contents of out->val are then unspecified. */
#define TREW_PACK_NO_VAL 1u
int trew_pack_reads_ranges(const char* buffer, const int32_t* locs, const char* buffer2, const int32_t* locs2, uint32_t n,
                           uint32_t n_ranges, uint32_t n_threads, uint32_t flags, void* dst, size_t dst_bytes, trew_batch* out,
                           uint32_t* inv, size_t inv_cap, size_t* n_inv);

/* ---- whole-file convenience: process_kmer / _pair / _long (src/kmer.cpp:1266-1476) -------------- */

/* Reads FASTQ / FASTQ.gz with the reference's record semantics (every 4k+2-th line is a sequence, short mode
 * rejects reads > 1000, long mode drops reads < SLICE_LENGTH; the reference's 4 MiB - 1 chunking has no observable
 * effect and is not reproduced) and feeds the context.  file2 must be NULL unless mode is TREW_MODE_PAIR.
 * is_gz*: 1 = gzip (BGZF members are inflated in parallel), 0 = plain (regular files are mapped). */
int trew_dev_process_file(trew_ctx* ctx, const char* file1, int is_gz1, const char* file2, int is_gz2);

/* The reader alone (no device): calls `sink` once per chunk with the text buffer(s) and the inclusive
 * (st, nd) offsets of the sequence lines it found -- what the reference's reader threads push as
 * QueueData / PairQueueData.  The buffers are read-only and valid only during the call.  chunk_bytes: bytes per
 * block, 0 = chosen by input kind.  A non-zero return from sink aborts.  message (may be NULL) receives the
 * reference's error text on failure. */
typedef int (*trew_chunk_sink)(void* user, const char* buffer1, const int32_t* locs1, uint32_t n1,
                               const char* buffer2, const int32_t* locs2, uint32_t n2);
int trew_ingest_file(int mode, int slice_length, const char* file1, int is_gz1, const char* file2, int is_gz2,
                     uint64_t chunk_bytes, trew_chunk_sink sink, void* user, char* message, size_t message_cap);

/* ---- report: process_output / final_process_output (src/kmer.cpp:1478-1634, 2571-2761) ---------- */
typedef struct trew_report trew_report;
int trew_report_create(int min_mer, trew_report** out);
void trew_report_destroy(trew_report* r);
/* Fold + filter + sort one file's six maps and append ">H:" / ">L:" sections to the report text;
 * accumulates the per-file vectors for the cross-file scoring (src/trew.cpp:454-467). */
int trew_report_add_file(trew_report* r, const char* file_name, const trew_entry* entries, uint64_t n);
/* The text so far (owned by r, valid until the next call on r): lets a caller print each file's sections as soon as
 * that file is done, as process_output does (src/kmer.cpp:1615-1631). */
int trew_report_text(trew_report* r, const char** text, size_t* len);
/* Append ">Putative_TRM" (src/kmer.cpp:2571-2691) and return the whole text (owned by r). */
int trew_report_finish(trew_report* r, const char** text, size_t* len);

#ifdef __cplusplus
}
#endif
#endif /* TREW_B200_H */
