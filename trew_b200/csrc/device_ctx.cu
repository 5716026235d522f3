// C ABI implementation: device context, pinned staging ring, asynchronous submit, table export.
//
// Stands in for the consumer side of the reference's queue (buffer_task* workers started by
// process_kmer*, src/kmer.cpp:1278-1325) and for the per-worker result maps that process_output sums
// (src/kmer.cpp:1486-1515).  One context = one GPU.  Per staging slot: pinned host buffer, device
// buffer, stream and completion event, so packing of batch i+1 on the host overlaps the H2D copy and
// the kernels of batch i (double/triple buffering with cudaMemcpyAsync).
#include <algorithm>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "host_internal.h"
#include "scan_kernels.cuh"

using namespace trew;

namespace {

struct SlotRes {
    void* h_buf = nullptr;      // pinned
    void* d_buf = nullptr;
    unsigned char* h_inv = nullptr;  // pinned: the batch's invalid-base records (sparse validity, see submit_ranges)
    unsigned char* d_inv = nullptr;
    size_t inv_cap = 0;              // records
    unsigned int* h_keys = nullptr;  // pinned: the table's distinct-key count as of this slot's last batch
    unsigned int* d_survivors = nullptr;
    unsigned int* d_counters = nullptr;  // [0] n_survivors [1] work counter [2] n_deferred
    unsigned char* d_scratch = nullptr;
    size_t scratch_bytes = 0;
    size_t survivors_cap = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_start = nullptr, ev_done = nullptr;
    bool in_flight = false;
};

// reads [r0, r1) of a chunk with their base total and longest read
struct RangeInfo { uint32_t r0, r1; uint64_t bases; uint32_t max_len; };

}  // namespace

struct trew_resident {
    void* d_buf = nullptr;
    DevBatch batch{};
    uint32_t n_reads = 0, n_units = 0, max_read_len = 0;
    uint64_t bases = 0;
    unsigned int* d_survivors = nullptr;
    unsigned int* d_counters = nullptr;
    unsigned char* d_scratch = nullptr;
    size_t scratch_bytes = 0;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};  // before screen, after screen, after decide, after exact
    bool ev_pending = false;
};

struct trew_ctx {
    trew_config cfg{};
    int sm_count = 0;
    LaunchPlan plan{};
    cudaStream_t aux_stream = nullptr;   // second stream for device-resident scans (consecutive batches overlap)
    cudaEvent_t ev_join = nullptr;
    int resident_streams = 1;
    uint64_t resident_seq = 0;
    DevCfg dcfg{};
    size_t n_slots = 0;
    unsigned int* d_error = nullptr;
    unsigned short* d_thr = nullptr;
    unsigned long long* d_total_surv = nullptr;
    std::vector<SlotRes> slots;
    size_t next_slot = 0;
    size_t staging_bytes = 0;
    cudaStream_t main_stream = nullptr;
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;
    // export buffers
    trew_entry* d_entries = nullptr; size_t d_entries_cap = 0;   // compacted table (device, unsorted)
    trew_entry* d_sorted = nullptr; size_t d_sorted_cap = 0;     // the same rows sorted by (table, k, seq)
    trew_entry* d_concat = nullptr; size_t d_concat_cap = 0;     // finish_merged: this table's rows + the other ranks'
    bool sorted_valid = false;
    void* d_sort_tmp = nullptr; size_t sort_tmp_bytes = 0;
    unsigned int* d_n = nullptr;
    uint64_t n_export = 0;
    bool export_valid = false;   // d_entries reflects the current table (no scan / merge / reset since the last export)
    trew_stats stats{};
    Pool* pool = nullptr;
    bool own_pool = true;                        // false: the pool belongs to a trew_multi group
    std::string err;
    std::vector<RangeInfo> ranges_tmp;
    unsigned int keys_seen = 0;                  // distinct keys reported by the batches retired so far (lags the device)
    bool sparse_val = true;                      // TREW_DENSE_VAL=1: always copy the validity plane
    unsigned int exact_flags = 0;                // TREW_EXACT_FLAGS: switches parts of the exact kernel off (A/B measurements)
    std::vector<InvList> inv_tmp;                // per packing range: records of its blocks with invalid bases
    IngestScratch ingest;   // file block buffers, kept across files
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
    double screen_ms = 0, decide_ms = 0, exact_ms = 0; uint64_t n_prof_scans = 0;
    std::vector<trew_resident*> pending_prof;
    void* h_export = nullptr; size_t h_export_bytes = 0;
    unsigned int report_min = 0;                                 // > 0: finish copies only the rows a one-file report can show
    trew_entry* d_filtered = nullptr; size_t d_filtered_cap = 0;
    // unit records (trew_dev_enable_unit_records): dcfg.recs points at d_recs when they are on
    UnitRecs* d_recs = nullptr; trew_unit_record* d_rec_buf = nullptr; uint64_t rec_cap = 0;
    uint64_t unit_next = 0;                      // ordinal of the next unit submitted
    bool table_used = false;                     // something was scanned or merged since create / reset
    trew_unit_record* d_rec_out = nullptr; size_t d_rec_out_cap = 0;   // sorted, combined records
    trew_unit_record* d_rec_cat = nullptr; size_t d_rec_cat_cap = 0;   // trew_multi: every device's records on the first one
    void* h_rec = nullptr; size_t h_rec_bytes = 0;
};

namespace {

int fail(trew_ctx* c, int status, const char* fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
    if (c) c->err = buf;
    return status;
}

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) return fail(ctx, TREW_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

// smallest M with (double)M / (double)T >= B, exactly as the reference forms the ratio (src/kmer.cpp:2223-2224)
void build_thr(double B, std::vector<unsigned short>& thr) {
    thr.assign(kThrTableSize, 0xFFFF);
    for (int T = 1; T < kThrTableSize; T++) {
        int lo = 0, hi = T;  // ratio is monotone in M; M = T gives 1.0 >= B
        while (lo < hi) {
            int mid = (lo + hi) / 2;
            if ((double)mid / (double)T >= B) hi = mid; else lo = mid + 1;
        }
        thr[T] = (unsigned short)lo;
    }
}

int run_cap_for(const trew_config& cfg, uint32_t max_read_len) {
    uint32_t w = max_read_len;
    if (cfg.mode == TREW_MODE_LONG) w = std::min<uint32_t>(max_read_len, 2u * (uint32_t)cfg.slice_length);
    w = std::min<uint32_t>(w, (uint32_t)kMaxWindow);
    return (int)std::max<uint32_t>((w + 2 + 7) & ~7u, 32u);   // >= 32: eval_k's serial path keeps 96 words in htab + grp_*
}

constexpr unsigned int kLongThreadCap = 32768;   // survivors per batch the long-read thread path takes (the rest: warp kernel)

// warp kernel: per-warp (th, tl) per slice; long-read thread path (behind it, at *long_off): statistics + emissions per
// (survivor, slice)
size_t scratch_need(const trew_ctx* ctx, uint32_t max_read_len, uint32_t n_units, unsigned int* stride, size_t* long_off,
                    unsigned int* s_cap, unsigned int* max_slices) {
    unsigned int st = 16;
    if (ctx->cfg.mode == TREW_MODE_LONG) st = 2u * (max_read_len / (uint32_t)ctx->cfg.slice_length + 2u);
    st = (st + 15u) & ~15u;
    *stride = st;
    size_t bytes = ((size_t)st * (size_t)exact_warps_total(ctx->sm_count) + 255) & ~(size_t)255;
    *long_off = bytes;
    *s_cap = 0; *max_slices = 0;
    // off unless TREW_EXACT_FLAGS has bit 16: measured slower than the warp kernel's serial walk on configs[3] (2.0 against
    // 1.03 ms per 200 k x 15 kb batch; 6.3 against 3.7 ms with 10 % telomeric reads) -- scanning every slice of a survivor
    // is 5x the slices the walks look at when the repeat sits at one end (DESIGN.md section 3)
    if (long_thread_path_applies(ctx->dcfg) && (ctx->exact_flags & 16u)) {
        *s_cap = std::min<unsigned int>(std::max<unsigned int>(n_units, 1u), kLongThreadCap);
        *max_slices = max_read_len / (uint32_t)ctx->cfg.slice_length + 1u;
        bytes += long_thread_scratch_bytes(*s_cap, *max_slices);
    }
    return bytes;
}

constexpr int kScanCounters = 8;

static int env_blocks_thread() {   // TREW_GRID_THREAD: thread-kernel blocks per SM (experiments)
    static const int v = [] { const char* e = getenv("TREW_GRID_THREAD"); int x = e && *e ? atoi(e) : 0; return x > 0 ? x : 0; }();
    return v;
}

// d_survivors holds 2 * n_units entries: survivors in the first half, the screen kernel's deferred list in the second
int launch_scan(trew_ctx* ctx, const DevBatch& b, uint32_t n_units, uint32_t max_read_len, unsigned int* d_survivors,
                unsigned int* d_counters, unsigned char** d_scratch, size_t* scratch_bytes, cudaStream_t st,
                cudaEvent_t* ev = nullptr) {
    unsigned int stride, s_cap, max_slices;
    size_t long_off;
    size_t need = scratch_need(ctx, max_read_len, n_units, &stride, &long_off, &s_cap, &max_slices);
    if (need > *scratch_bytes) {
        if (*d_scratch) { CK(cudaStreamSynchronize(st)); CK(cudaFree(*d_scratch)); *d_scratch = nullptr; }
        CK(cudaMalloc((void**)d_scratch, need));
        *scratch_bytes = need;
    }
    ctx->export_valid = false;
    ctx->table_used = true;
    DevCfg cfg = ctx->dcfg;
    cfg.unit_base = ctx->unit_next;
    ctx->unit_next += n_units;
    // d_counters: [0] survivors (list A) [1] work counter [2] deferred [3] thread-kernel bails [4] survivors, list B [5] work counter [6] work counter of the thread kernel [7] work counter of the decide kernel
    CK(cudaMemsetAsync(d_counters, 0, kScanCounters * sizeof(unsigned int), st));
    if (ev) CK(cudaEventRecord(ev[0], st));
    const bool thread_path = thread_path_applies(cfg, max_read_len) && !(ctx->exact_flags & 4u) && n_units < (1u << 28);
    launch_filter(cfg, b, n_units, max_read_len, d_survivors + n_units, d_counters + 2, d_survivors, d_counters, ctx->plan, st,
                  ev ? ev[1] : nullptr, thread_path ? d_survivors + n_units - 1 : nullptr, thread_path ? d_counters + 4 : nullptr,
                  d_counters + 7);
    if (ev) CK(cudaEventRecord(ev[2], st));
    ExactArgs a{};
    a.survivors = d_survivors; a.n_survivors = d_counters; a.work_counter = d_counters + 1;
    a.slice_scratch = *d_scratch; a.slice_scratch_stride = stride; a.run_cap = run_cap_for(ctx->cfg, max_read_len);
    a.total_survivors = ctx->d_total_surv;
    a.packed_probes = n_units < (1u << 28) ? 1 : 0;
    a.exp_flags = ctx->exact_flags;
    if (thread_path) {
        // list A: thread per survivor; what it cannot take after all (its length limits) lands in the dead deferred list
        unsigned int* hard = d_survivors + n_units;
        launch_exact_thread(cfg, b, d_survivors, d_counters, a.packed_probes, hard, d_counters + 3, ctx->d_total_surv,
                            ctx->sm_count, env_blocks_thread(), d_counters + 6, st);
        // list B (downwards from the top of the survivor array): warp per survivor
        ExactArgs ab = a;
        ab.survivors = d_survivors + n_units - 1; ab.reverse = 1; ab.n_survivors = d_counters + 4;
        launch_exact(cfg, b, ab, ctx->plan, st);
        // ... and the thread kernel's leftovers (normally none)
        a.survivors = hard; a.n_survivors = d_counters + 3; a.work_counter = d_counters + 5; a.total_survivors = nullptr;
        ctx->stats.kernel_launches += 2;
    } else if (s_cap > 0 && n_units < (1u << 28)) {
        // long reads: statistics of every slice of a survivor, the walks over them, the emissions (three kernels); reads
        // whose walk reaches the long middle slice -- or beyond the scratch's capacity -- go to the warp kernel
        unsigned int* hard = d_survivors + n_units;
        launch_long_thread(cfg, b, d_survivors, d_counters, a.packed_probes, s_cap, max_slices, *d_scratch + long_off, hard,
                           d_counters + 3, ctx->d_total_surv, ctx->sm_count, st);
        a.survivors = hard; a.n_survivors = d_counters + 3; a.total_survivors = nullptr;
        ctx->stats.kernel_launches += 3;
    }
    launch_exact(cfg, b, a, ctx->plan, st);
    if (ev) CK(cudaEventRecord(ev[3], st));
    CK(cudaGetLastError());
    ctx->stats.kernel_launches += 3;
    return TREW_OK;
}

int retire_slot(trew_ctx* ctx, SlotRes& s) {
    if (!s.in_flight) return TREW_OK;
    CK(cudaEventSynchronize(s.ev_done));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, s.ev_start, s.ev_done));
    ctx->stats.device_ms += ms;
    s.in_flight = false;
    ctx->keys_seen = std::max(ctx->keys_seen, *s.h_keys);
    return TREW_OK;
}

// Pack ranges [g0, g1) of a chunk (host threads) into the next free staging slot and launch copy + kernels on its stream.
int export_sorted(trew_ctx* ctx, uint64_t* n_out);
int check_device_error(trew_ctx* ctx);

// The streaming path keeps the count table at most a quarter full between batches: when the number of distinct keys
// passes that, all in-flight batches are drained and the entries are re-inserted into a larger table (load <= 1/8).
// The check runs once per batch, so a single batch that inserts more new keys than three quarters of the table can
// still overflow it (TREW_ERR_TABLE_FULL: start with a larger table_log2_slots).
// re-insert the table's entries into a table of at least min_slots slots (rounded up to a power of two, at most 2^28)
int grow_table_to(trew_ctx* ctx, size_t min_slots) {
    size_t new_slots = ctx->n_slots;
    while (new_slots < ((size_t)1 << 28) && new_slots < min_slots) new_slots <<= 1;
    if (new_slots == ctx->n_slots) return TREW_OK;
    uint64_t n = 0;
    int rc = export_sorted(ctx, &n);   // drains every stream, compacts into ctx->d_entries
    if (rc) return rc;
    Slot* d_new = nullptr;
    CK(cudaMalloc((void**)&d_new, new_slots * sizeof(Slot)));
    CK(cudaMemsetAsync(d_new, 0, new_slots * sizeof(Slot), ctx->main_stream));
    CK(cudaMemsetAsync(ctx->d_error + 1, 0, sizeof(unsigned int), ctx->main_stream));
    Slot* d_old = ctx->dcfg.slots;
    ctx->dcfg.slots = d_new; ctx->dcfg.slot_mask = (unsigned int)(new_slots - 1); ctx->n_slots = new_slots;
    launch_merge_entries(ctx->dcfg, ctx->d_entries, (unsigned int)n, ctx->main_stream);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->main_stream));
    CK(cudaFree(d_old));
    ctx->stats.kernel_launches += 1;
    ctx->keys_seen = (unsigned int)n;
    for (auto& sl : ctx->slots) *sl.h_keys = (unsigned int)n;
    return check_device_error(ctx);
}

int maybe_grow_table(trew_ctx* ctx) {
    // Every batch copies the key counter back behind its kernels (no host wait); that value lags by the batches in
    // flight, so it only serves to skip the exact, blocking read while the table is far (4x) from the threshold.
    if ((size_t)ctx->keys_seen * 16 <= ctx->n_slots) return TREW_OK;
    unsigned int keys = 0;
    CK(cudaMemcpy(&keys, ctx->d_error + 1, sizeof(keys), cudaMemcpyDeviceToHost));
    ctx->keys_seen = std::max(ctx->keys_seen, keys);
    if ((size_t)keys * 4 <= ctx->n_slots) return TREW_OK;
    return grow_table_to(ctx, (size_t)keys * 8);
}

int submit_ranges(trew_ctx* ctx, const ChunkView& cv, const RangeInfo* rg, int n_ranges) {
    uint64_t total_bases = 0; uint32_t max_len = 0;
    for (int i = 0; i < n_ranges; i++) { total_bases += rg[i].bases; max_len = std::max(max_len, rg[i].max_len); }
    const uint32_t n = n_ranges ? rg[n_ranges - 1].r1 - rg[0].r0 : 0u;
    if (n == 0) return TREW_OK;
    SlotRes& s = ctx->slots[ctx->next_slot];
    ctx->next_slot = (ctx->next_slot + 1) % ctx->slots.size();
    static const bool trace = getenv("TREW_SUBMIT_TRACE") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t0 = trace ? now() : 0;
    int rc = retire_slot(ctx, s);
    if (rc) return rc;
    const double t1 = trace ? now() : 0;
    if ((rc = maybe_grow_table(ctx)) != TREW_OK) return rc;
    const double t2 = now();
    BatchView v;
    batch_layout(s.h_buf, n, total_bases, &v);
    std::vector<uint64_t> bit0((size_t)n_ranges);
    uint64_t acc = 0;
    for (int i = 0; i < n_ranges; i++) { bit0[i] = acc; acc += rg[i].bases; }
    v.bit_off[n] = (uint32_t)total_bases;
    const uint32_t first = rg[0].r0;
    std::vector<uint64_t> side_flat((size_t)3 * n_ranges);
    uint64_t (*side)[3] = (uint64_t (*)[3])side_flat.data();
    // Validity travels as a list when it is sparse (it nearly always is: a few N per thousand bases at most): the
    // packers record the 64-base blocks whose validity mask is not all ones (position + mask, 12 bytes) instead of
    // writing the val plane, only [bit_off | hi | lo] and the records cross PCIe, and the device plane is a memset
    // plus a scatter.  A batch with more such blocks than the record buffer holds is packed again with its val
    // plane and copied whole.
    if (ctx->inv_tmp.size() < (size_t)n_ranges) ctx->inv_tmp.resize((size_t)n_ranges);
    auto pack = [&](bool list) {
        pack_prepare(bit0.data(), n_ranges, total_bases, v);
        ctx->pool->run(n_ranges, [&](int i) {
            pack_chunk_range(cv, rg[i].r0, rg[i].r1, rg[i].r0 - first, bit0[i], v, side[i], list ? &ctx->inv_tmp[(size_t)i] : nullptr, list,
                             rg[i].bases);
        });
        pack_fixup(bit0.data(), side, n_ranges, v);
    };
    size_t n_inv = 0;
    bool sparse = ctx->sparse_val;
    pack(sparse);
    const bool tail_pad = (total_bases & 31) != 0;   // the padding bits of the last plane word are "invalid" too
    if (sparse) {
        n_inv = tail_pad ? 1 : 0;
        for (int i = 0; i < n_ranges; i++) n_inv += ctx->inv_tmp[(size_t)i].size();
        if (n_inv > s.inv_cap) { sparse = false; pack(false); }
    }

    const double t3 = now();
    ctx->stats.host_pack_bytes += total_bases; ctx->stats.host_pack_ms += t3 - t2;
    CK(cudaEventRecord(s.ev_start, s.stream));
    const size_t head_bytes = (size_t)((char*)v.val - (char*)s.h_buf);
    unsigned int* d_val = (unsigned int*)((char*)s.d_buf + head_bytes);
    size_t sent = v.bytes;
    if (sparse) {
        // the ranges' record lists, back to back in the pinned buffer (on the pool: ~2 MB per batch at 0.1 % N)
        std::vector<size_t> at((size_t)n_ranges + 1, 0);
        for (int i = 0; i < n_ranges; i++) at[(size_t)i + 1] = at[(size_t)i] + ctx->inv_tmp[(size_t)i].bytes();
        ctx->pool->run(n_ranges, [&](int i) {
            const InvList& l = ctx->inv_tmp[(size_t)i];
            if (l.bytes()) memcpy(s.h_inv + at[(size_t)i], l.buf.get(), l.bytes());
        });
        if (tail_pad) inv_record(s.h_inv + at[(size_t)n_ranges], (uint32_t)total_bases, (1ULL << (32 - (total_bases & 31))) - 1ULL);
        const size_t ones_words = (size_t)((total_bases + 31) / 32);
        CK(cudaMemsetAsync(d_val, 0xFF, ones_words * 4, s.stream));
        CK(cudaMemsetAsync(d_val + ones_words, 0, (v.plane_words - ones_words) * 4, s.stream));
        CK(cudaMemcpyAsync(s.d_buf, s.h_buf, head_bytes, cudaMemcpyHostToDevice, s.stream));
        if (n_inv) {
            CK(cudaMemcpyAsync(s.d_inv, s.h_inv, n_inv * kInvRecBytes, cudaMemcpyHostToDevice, s.stream));
            launch_clear_invalid(d_val, (const unsigned int*)s.d_inv, (unsigned int)n_inv, s.stream);
            ctx->stats.kernel_launches += 1;
        }
        sent = head_bytes + n_inv * kInvRecBytes;
    } else {
        CK(cudaMemcpyAsync(s.d_buf, s.h_buf, v.bytes, cudaMemcpyHostToDevice, s.stream));
    }
    DevBatch b{};
    b.n_reads = n;
    b.bit_off = (const unsigned int*)s.d_buf;
    b.hi = (const unsigned int*)((char*)s.d_buf + ((char*)v.hi - (char*)s.h_buf));
    b.lo = b.hi + v.plane_words; b.val = d_val;
    uint32_t n_units = ctx->cfg.mode == TREW_MODE_PAIR ? n / 2 : n;
    rc = launch_scan(ctx, b, n_units, max_len, s.d_survivors, s.d_counters, &s.d_scratch, &s.scratch_bytes, s.stream);
    if (rc) return rc;
    CK(cudaMemcpyAsync(s.h_keys, ctx->d_error + 1, sizeof(unsigned int), cudaMemcpyDeviceToHost, s.stream));
    CK(cudaEventRecord(s.ev_done, s.stream));
    s.in_flight = true;
    ctx->stats.reads += n; ctx->stats.bases += total_bases; ctx->stats.units += n_units; ctx->stats.h2d_bytes += sent;
    if (trace)
        fprintf(stderr, "[submit] %u reads: wait slot %.3f ms, table check %.3f ms, pack %.3f ms, enqueue %.3f ms\n", n, t1 - t0, t2 - t1,
                t3 - t2, now() - t3);
    return TREW_OK;
}

// Split a chunk of n reads into ranges (statistics gathered on the pool), group consecutive ranges into batches
// that fit one staging slot and submit them.
int submit_chunk_view(trew_ctx* ctx, const ChunkView& cv, uint32_t n) {
    if (n == 0) return TREW_OK;
    const uint32_t unit = cv.unit;
    const uint32_t n_units = n / unit;
    // ranges small enough that any single one is far below a staging slot, and enough of them to feed the pool
    uint64_t span = 0;
    for (int sd = 0; sd < (int)unit; sd++) {
        const int32_t* l = cv.locs[sd];
        span += (uint64_t)std::max<int64_t>(0, (int64_t)l[2 * (size_t)(n_units - 1) + 1] - l[0] + 1);
    }
    uint64_t by_size = span / std::max<uint64_t>(1, ctx->staging_bytes / 16) + 1;
    uint32_t n_ranges = (uint32_t)std::min<uint64_t>(n_units, std::max<uint64_t>(by_size, (uint64_t)ctx->pool->size() * 4));
    auto& rg = ctx->ranges_tmp;
    rg.resize(n_ranges);
    for (uint32_t i = 0; i < n_ranges; i++) {
        rg[i].r0 = (uint32_t)((uint64_t)n_units * i / n_ranges) * unit;
        rg[i].r1 = (uint32_t)((uint64_t)n_units * (i + 1) / n_ranges) * unit;
    }
    ctx->pool->run((int)n_ranges, [&](int i) { chunk_stats(cv, rg[i].r0, rg[i].r1, &rg[i].bases, &rg[i].max_len); });
    uint32_t mx = 0;
    for (auto& r : rg) mx = std::max(mx, r.max_len);
    if (ctx->cfg.mode == TREW_MODE_SHORT && mx > 1000)  // MAX_SEQ, src/kmer.cpp:1006-1008
        return fail(ctx, TREW_ERR_TOO_LONG, "%s", trew_status_string(TREW_ERR_TOO_LONG));
    if (ctx->cfg.mode == TREW_MODE_PAIR && mx > (uint32_t)kMaxWindow) return fail(ctx, TREW_ERR_TOO_LONG, "paired read longer than %d", kMaxWindow);
    const size_t cap = ctx->slots[0].survivors_cap;
    uint32_t g = 0;
    while (g < n_ranges) {
        uint32_t h = g; uint64_t bases = 0; uint64_t reads = 0;
        while (h < n_ranges) {
            uint64_t nb = bases + rg[h].bases, nr = reads + (rg[h].r1 - rg[h].r0);
            if (batch_bytes((uint32_t)nr, nb) > ctx->staging_bytes || nr > cap || nb >= 0xfffff000ULL) break;
            bases = nb; reads = nr; h++;
        }
        if (h == g) {
            // a single range does not fit: fall back to unit-sized ranges for it
            if (rg[g].r1 - rg[g].r0 <= unit)
                return fail(ctx, TREW_ERR_ARG, "a single read/pair (%llu bases) does not fit a staging buffer of %zu bytes",
                            (unsigned long long)rg[g].bases, ctx->staging_bytes);
            std::vector<RangeInfo> fine;
            for (uint32_t r = rg[g].r0; r < rg[g].r1; r += unit) {
                RangeInfo f{r, r + unit, 0, 0};
                chunk_stats(cv, f.r0, f.r1, &f.bases, &f.max_len);
                fine.push_back(f);
            }
            size_t a = 0;
            while (a < fine.size()) {
                size_t e = a; uint64_t fb = 0, fr = 0;
                while (e < fine.size()) {
                    uint64_t nb = fb + fine[e].bases, nr = fr + unit;
                    if (batch_bytes((uint32_t)nr, nb) > ctx->staging_bytes || nr > cap || nb >= 0xfffff000ULL) break;
                    fb = nb; fr = nr; e++;
                }
                if (e == a)
                    return fail(ctx, TREW_ERR_ARG, "a single read/pair (%llu bases) does not fit a staging buffer of %zu bytes",
                                (unsigned long long)fine[a].bases, ctx->staging_bytes);
                // merge the unit ranges of this batch into at most pool-size ranges
                std::vector<RangeInfo> merged;
                size_t per = std::max<size_t>(1, (e - a) / (size_t)ctx->pool->size());
                for (size_t i = a; i < e; i += per) {
                    RangeInfo m{fine[i].r0, 0, 0, 0};
                    for (size_t j = i; j < std::min(e, i + per); j++) { m.r1 = fine[j].r1; m.bases += fine[j].bases; m.max_len = std::max(m.max_len, fine[j].max_len); }
                    merged.push_back(m);
                }
                int rc = submit_ranges(ctx, cv, merged.data(), (int)merged.size());
                if (rc) return rc;
                a = e;
            }
            g++;
            continue;
        }
        int rc = submit_ranges(ctx, cv, rg.data() + g, (int)(h - g));
        if (rc) return rc;
        g = h;
    }
    return TREW_OK;
}

int collect_prof(trew_ctx* ctx) {
    for (trew_resident* r : ctx->pending_prof) {
        if (!r->ev_pending) continue;
        CK(cudaEventSynchronize(r->ev[3]));
        float a = 0, b = 0, c = 0;
        CK(cudaEventElapsedTime(&a, r->ev[0], r->ev[1]));
        CK(cudaEventElapsedTime(&b, r->ev[1], r->ev[2]));
        CK(cudaEventElapsedTime(&c, r->ev[2], r->ev[3]));
        ctx->screen_ms += a; ctx->decide_ms += b; ctx->exact_ms += c; ctx->n_prof_scans++;
        ctx->stats.device_ms += a + b + c;
        r->ev_pending = false;
    }
    ctx->pending_prof.clear();
    return TREW_OK;
}

// main_stream waits for everything queued on aux_stream so far
int join_aux(trew_ctx* ctx) {
    if (ctx->resident_streams != 2) return TREW_OK;
    CK(cudaEventRecord(ctx->ev_join, ctx->aux_stream));
    CK(cudaStreamWaitEvent(ctx->main_stream, ctx->ev_join, 0));
    return TREW_OK;
}

// aux_stream waits for everything queued on main_stream so far
int fork_aux(trew_ctx* ctx) {
    if (ctx->resident_streams != 2) return TREW_OK;
    CK(cudaEventRecord(ctx->ev_join, ctx->main_stream));
    CK(cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_join, 0));
    return TREW_OK;
}

// Long mode: the reader drops reads shorter than SLICE_LENGTH (src/kmer.cpp:1184).  With unit records on it keeps them, so
// that unit ordinals are the file's record indices; the scan emits nothing for them (unit_probes, route_long), so the tables
// are the same.
int reader_slice_length(const trew_ctx* ctx) { return ctx->d_recs ? 0 : ctx->cfg.slice_length; }

int check_device_error(trew_ctx* ctx) {
    unsigned int e = 0;
    CK(cudaMemcpy(&e, ctx->d_error, sizeof(e), cudaMemcpyDeviceToHost));
    if (e == 3u) return fail(ctx, TREW_ERR_TABLE_FULL, "device count table full (%zu slots): raise table_log2_slots", ctx->n_slots);
    if (e) return fail(ctx, TREW_ERR_CUDA, "device error flag %u", e);
    return TREW_OK;
}

}  // namespace

extern "C" {

int trew_abi_version(void) { return TREW_ABI_VERSION; }

const char* trew_status_string(int status) {
    switch (status) {
        case TREW_OK: return "ok";
        case TREW_ERR_ARG: return "bad argument";
        case TREW_ERR_CUDA: return "CUDA failure";
        case TREW_ERR_TABLE_FULL: return "device count table full";
        case TREW_ERR_TOO_LONG: return "This mode is designed for short-read sequencing. Please use 'trew long'.";
        case TREW_ERR_IO: return "file I/O error";
        case TREW_ERR_PAIRING: return "paired-end record mismatch";
        case TREW_ERR_NOMEM: return "memory allocation failure";
        default: return "unknown status";
    }
}

// trew_dev_create has no context to hang its message on: it is kept here and read with trew_dev_last_error(NULL)
static thread_local std::string g_create_error;
// set by trew_multi_create around its trew_dev_create calls: the group's contexts share one packing pool

static int default_host_threads(int asked) {
    return asked > 0 ? asked : (int)std::min(64u, std::max(1u, std::thread::hardware_concurrency()));
}

const char* trew_dev_last_error(const trew_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

// err: the message of a failed creation (trew_dev_create keeps it for trew_dev_last_error(NULL); trew_multi_create runs
// one of these per device on threads of its own)
static int create_ctx(const trew_config* cfg, trew_ctx** out, std::string& g_create_error, Pool* shared_pool) {
    if (!cfg || !out) return TREW_ERR_ARG;
    *out = nullptr;
    g_create_error.clear();
    auto bad_arg = [&](const char* msg) { g_create_error = msg; return TREW_ERR_ARG; };
    // same range checks as the reference CLI (src/trew.cpp:174-228, 255-304)
    if (cfg->mode < 0 || cfg->mode > 2) return bad_arg("mode must be TREW_MODE_SHORT, _PAIR or _LONG");
    if (cfg->min_mer < 3 || cfg->max_mer > 64 || cfg->min_mer > cfg->max_mer) return bad_arg("need 3 <= MIN_MER <= MAX_MER <= 64");
    if (!(0 < cfg->low_baseline && cfg->low_baseline <= 1) || !(0 < cfg->high_baseline && cfg->high_baseline <= 1) ||
        cfg->low_baseline > cfg->high_baseline) return bad_arg("need 0 < LOW_BASELINE <= HIGH_BASELINE <= 1");
    if (cfg->mode == TREW_MODE_LONG && cfg->slice_length > 0 && cfg->slice_length < 2 * cfg->max_mer)
        return bad_arg("SLICE_LENGTH must be greater than or equal to twice of MAX_MER.");
    // The middle slice of a long read is up to 2 * SLICE_LENGTH - 1 bases (src/kmer.cpp:790-798) and a window lives in
    // one warp's 32 x 32-bit registers (1023 bases), so SLICE_LENGTH stops at 512 here; the reference has no limit.
    if (cfg->mode == TREW_MODE_LONG && cfg->slice_length > 512)
        return bad_arg("SLICE_LENGTH above 512 is not supported by the GPU path (a slice of up to 2*SLICE_LENGTH-1 bases must fit "
                       "a 1023-base window); use -s 512 or less.");
    trew_ctx* ctx = new trew_ctx();
    ctx->cfg = *cfg;
    if (ctx->cfg.slice_length <= 0) ctx->cfg.slice_length = 150;
    auto bail = [&](int rc) { g_create_error = ctx->err; trew_dev_destroy(ctx); return rc; };
#define CKC(call)                                                                                   \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess) { fail(ctx, TREW_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); return bail(TREW_ERR_CUDA); } \
    } while (0)
    // TREW_CLI_TIMING=1: where the start-up time goes (stderr)
    const bool timing = getenv("TREW_CLI_TIMING") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t_prev = now();
    auto lap = [&](const char* what) {
        if (!timing) return;
        const double t = now();
        fprintf(stderr, "[trew] create, device %d: %s %.1f ms\n", cfg->device, what, t - t_prev);
        t_prev = t;
    };
    int ndev = 0;
    CKC(cudaGetDeviceCount(&ndev));
    lap("driver init");
    if (cfg->device < 0 || cfg->device >= ndev) { fail(ctx, TREW_ERR_CUDA, "no CUDA device %d (found %d)", cfg->device, ndev); return bail(TREW_ERR_CUDA); }
    CKC(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CKC(cudaGetDeviceProperties(&prop, cfg->device));
    ctx->sm_count = prop.multiProcessorCount;
    ctx->plan = default_launch_plan(ctx->sm_count);
    {
        // tuning knobs (experiments): blocks per SM of each scan kernel, and 2 streams for resident scans
        auto env_int = [](const char* name, int dflt) { const char* e = getenv(name); return e && *e ? atoi(e) : dflt; };
        int v;
        if ((v = env_int("TREW_GRID_SCREEN", 0)) > 0) ctx->plan.screen_blocks = ctx->sm_count * v;
        if ((v = env_int("TREW_GRID_DECIDE", 0)) > 0) ctx->plan.decide_blocks = ctx->sm_count * v;
        if ((v = env_int("TREW_GRID_EXACT", 0)) > 0) ctx->plan.exact_blocks = std::min(ctx->plan.exact_blocks, ctx->sm_count * v);
        ctx->resident_streams = env_int("TREW_RESIDENT_STREAMS", 1) >= 2 ? 2 : 1;
        ctx->sparse_val = env_int("TREW_DENSE_VAL", 0) == 0;
        ctx->exact_flags = (unsigned int)env_int("TREW_EXACT_FLAGS", 0);
    }
    int lg = cfg->table_log2_slots > 0 ? cfg->table_log2_slots : 22;
    if (lg < 10 || lg > 28) { fail(ctx, TREW_ERR_ARG, "table_log2_slots out of range"); return bail(TREW_ERR_ARG); }
    ctx->n_slots = (size_t)1 << lg;
    Slot* d_slots = nullptr;
    CKC(cudaMalloc((void**)&d_slots, ctx->n_slots * sizeof(Slot)));
    CKC(cudaMemset(d_slots, 0, ctx->n_slots * sizeof(Slot)));
    lap("primary context + count table");
    CKC(cudaMalloc((void**)&ctx->d_error, 2 * sizeof(unsigned int)));
    CKC(cudaMemset(ctx->d_error, 0, 2 * sizeof(unsigned int)));
    CKC(cudaMalloc((void**)&ctx->d_total_surv, sizeof(unsigned long long)));
    CKC(cudaMemset(ctx->d_total_surv, 0, sizeof(unsigned long long)));
    std::vector<unsigned short> thr;
    build_thr(cfg->low_baseline, thr);
    std::vector<unsigned short> thr_hi;
    build_thr(cfg->high_baseline, thr_hi);
    CKC(cudaMalloc((void**)&ctx->d_thr, 2 * thr.size() * sizeof(unsigned short)));
    CKC(cudaMemcpy(ctx->d_thr, thr.data(), thr.size() * sizeof(unsigned short), cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(ctx->d_thr + thr.size(), thr_hi.data(), thr_hi.size() * sizeof(unsigned short), cudaMemcpyHostToDevice));
    ctx->dcfg.mode = cfg->mode; ctx->dcfg.min_mer = cfg->min_mer; ctx->dcfg.max_mer = cfg->max_mer;
    ctx->dcfg.slice_len = ctx->cfg.slice_length; ctx->dcfg.low = cfg->low_baseline; ctx->dcfg.high = cfg->high_baseline;
    ctx->dcfg.slots = d_slots; ctx->dcfg.slot_mask = (unsigned int)(ctx->n_slots - 1);
    ctx->dcfg.error_flag = ctx->d_error; ctx->dcfg.thr_low = ctx->d_thr; ctx->dcfg.thr_high = ctx->d_thr + kThrTableSize;
    CKC(prepare_exact(kMaxWindow + 9));
    lap("kernel attributes (module load)");
    CKC(cudaStreamCreateWithFlags(&ctx->main_stream, cudaStreamNonBlocking));
    CKC(cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
    CKC(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    CKC(cudaEventCreate(&ctx->ev_a));
    CKC(cudaEventCreate(&ctx->ev_b));
    CKC(cudaEventCreate(&ctx->ev_t0));
    CKC(cudaEventCreate(&ctx->ev_t1));
    ctx->staging_bytes = cfg->staging_bytes ? (size_t)cfg->staging_bytes : ((size_t)64 << 20);
    int ns = cfg->n_staging > 0 ? cfg->n_staging : 3;
    ctx->slots.resize((size_t)ns);
    for (auto& s : ctx->slots) {
        CKC(cudaHostAlloc(&s.h_buf, ctx->staging_bytes, cudaHostAllocDefault));
        CKC(cudaMalloc(&s.d_buf, ctx->staging_bytes));
        s.inv_cap = ctx->staging_bytes / 8 / kInvRecBytes;   // 1/8 of the slot: past that the dense plane is no larger
        CKC(cudaHostAlloc((void**)&s.h_inv, (s.inv_cap + 1) * kInvRecBytes, cudaHostAllocDefault));
        CKC(cudaMalloc((void**)&s.d_inv, (s.inv_cap + 1) * kInvRecBytes));
        CKC(cudaHostAlloc((void**)&s.h_keys, sizeof(unsigned int), cudaHostAllocDefault));
        *s.h_keys = 0;
        s.survivors_cap = ctx->staging_bytes / 8;  // >= reads of >= 11 bases; submit_split enforces it
        CKC(cudaMalloc((void**)&s.d_survivors, 2 * s.survivors_cap * sizeof(unsigned int)));
        CKC(cudaMalloc((void**)&s.d_counters, kScanCounters * sizeof(unsigned int)));
        CKC(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        CKC(cudaEventCreate(&s.ev_start));
        CKC(cudaEventCreate(&s.ev_done));
    }
    CKC(cudaMalloc((void**)&ctx->d_n, sizeof(unsigned int)));
    lap("staging ring (pinned + device buffers)");
    if (shared_pool) { ctx->pool = shared_pool; ctx->own_pool = false; }
    else ctx->pool = new Pool(default_host_threads(cfg->host_threads));
#undef CKC
    *out = ctx;
    return TREW_OK;
}

int trew_dev_create(const trew_config* cfg, trew_ctx** out) { return create_ctx(cfg, out, g_create_error, nullptr); }

void trew_dev_destroy(trew_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->cfg.device);
    cudaDeviceSynchronize();
    for (auto& s : ctx->slots) {
        if (s.h_buf) cudaFreeHost(s.h_buf);
        if (s.d_buf) cudaFree(s.d_buf);
        if (s.h_inv) cudaFreeHost(s.h_inv);
        if (s.d_inv) cudaFree(s.d_inv);
        if (s.h_keys) cudaFreeHost(s.h_keys);
        if (s.d_survivors) cudaFree(s.d_survivors);
        if (s.d_counters) cudaFree(s.d_counters);
        if (s.d_scratch) cudaFree(s.d_scratch);
        if (s.stream) cudaStreamDestroy(s.stream);
        if (s.ev_start) cudaEventDestroy(s.ev_start);
        if (s.ev_done) cudaEventDestroy(s.ev_done);
    }
    if (ctx->dcfg.slots) cudaFree(ctx->dcfg.slots);
    if (ctx->d_error) cudaFree(ctx->d_error);
    if (ctx->d_thr) cudaFree(ctx->d_thr);
    if (ctx->d_total_surv) cudaFree(ctx->d_total_surv);
    if (ctx->d_entries) cudaFree(ctx->d_entries);
    if (ctx->d_sorted) cudaFree(ctx->d_sorted);
    if (ctx->d_concat) cudaFree(ctx->d_concat);
    if (ctx->d_filtered) cudaFree(ctx->d_filtered);
    if (ctx->d_sort_tmp) cudaFree(ctx->d_sort_tmp);
    if (ctx->d_n) cudaFree(ctx->d_n);
    if (ctx->h_export) cudaFreeHost(ctx->h_export);
    if (ctx->d_recs) cudaFree(ctx->d_recs);
    if (ctx->d_rec_buf) cudaFree(ctx->d_rec_buf);
    if (ctx->d_rec_out) cudaFree(ctx->d_rec_out);
    if (ctx->d_rec_cat) cudaFree(ctx->d_rec_cat);
    if (ctx->h_rec) cudaFreeHost(ctx->h_rec);
    if (ctx->main_stream) cudaStreamDestroy(ctx->main_stream);
    if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->ev_a) cudaEventDestroy(ctx->ev_a);
    if (ctx->ev_b) cudaEventDestroy(ctx->ev_b);
    if (ctx->ev_t0) cudaEventDestroy(ctx->ev_t0);
    if (ctx->ev_t1) cudaEventDestroy(ctx->ev_t1);
    if (ctx->own_pool) delete ctx->pool;
    delete ctx;
}

int trew_dev_submit_chunk(trew_ctx* ctx, const char* buffer1, const int32_t* locs1, uint32_t n1,
                          const char* buffer2, const int32_t* locs2, uint32_t n2) {
    if (!ctx) return TREW_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    const bool pair = ctx->cfg.mode == TREW_MODE_PAIR;
    if (pair ? (!buffer2 && n2) : (buffer2 != nullptr || n2 != 0)) return fail(ctx, TREW_ERR_ARG, "second chunk only in pair mode");
    if ((n1 && (!buffer1 || !locs1)) || (n2 && !locs2)) return fail(ctx, TREW_ERR_ARG, "null chunk");
    ChunkView cv{{buffer1, buffer2}, {locs1, locs2}, {nullptr, nullptr}, pair ? 2u : 1u};
    const uint32_t n = pair ? 2u * std::min(n1, n2) : n1;  // index-wise pairing, src/kmer.cpp:321-322
    if (n == 0) return TREW_OK;
    // one past the last byte the caller vouches for: lets the packer load whole 32-byte blocks at read tails
    // (sequence lines are produced in ascending order, so the last one bounds the buffer from below)
    for (int sd = 0; sd < (pair ? 2 : 1); sd++) {
        const int32_t* l = cv.locs[sd];
        uint32_t cnt = pair ? n / 2 : n;
        int32_t last = l[2 * (size_t)(cnt - 1) + 1];
        if (last >= l[2 * (size_t)(cnt - 1)]) cv.end[sd] = cv.buf[sd] + last + 1;
    }
    return submit_chunk_view(ctx, cv, n);
}

int trew_dev_submit_packed(trew_ctx* ctx, const trew_batch* batch) {
    if (!ctx || !batch) return TREW_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    uint32_t n = batch->n_reads;
    if (n == 0) return TREW_OK;
    uint64_t bases = batch->bit_off[n];
    size_t bytes = batch_bytes(n, bases);
    if (bytes > ctx->staging_bytes || n > ctx->slots[0].survivors_cap)
        return fail(ctx, TREW_ERR_ARG, "packed batch (%zu bytes) larger than a staging buffer (%zu)", bytes, ctx->staging_bytes);
    if (batch->bit_off[0] != 0) return fail(ctx, TREW_ERR_ARG, "bit_off[0] must be 0");
    SlotRes& s = ctx->slots[ctx->next_slot];
    ctx->next_slot = (ctx->next_slot + 1) % ctx->slots.size();
    int rc = retire_slot(ctx, s);
    if (rc) return rc;
    BatchView v;
    batch_layout(s.h_buf, n, bases, &v);
    size_t words = (size_t)((bases + 31) / 32);
    memcpy(v.bit_off, batch->bit_off, (size_t)(n + 1) * 4);
    const uint32_t* src[3] = {batch->hi, batch->lo, batch->val};
    uint32_t* dst[3] = {v.hi, v.lo, v.val};
    ctx->pool->run(3, [&](int i) {
        memcpy(dst[i], src[i], words * 4);
        memset(dst[i] + words, 0, (v.plane_words - words) * 4);
    });
    CK(cudaEventRecord(s.ev_start, s.stream));
    CK(cudaMemcpyAsync(s.d_buf, s.h_buf, v.bytes, cudaMemcpyHostToDevice, s.stream));
    DevBatch b{};
    b.n_reads = n;
    b.bit_off = (const unsigned int*)s.d_buf;
    b.hi = (const unsigned int*)((char*)s.d_buf + ((char*)v.hi - (char*)s.h_buf));
    b.lo = b.hi + v.plane_words; b.val = b.lo + v.plane_words;
    uint32_t n_units = ctx->cfg.mode == TREW_MODE_PAIR ? n / 2 : n;
    rc = launch_scan(ctx, b, n_units, batch->max_read_len, s.d_survivors, s.d_counters, &s.d_scratch, &s.scratch_bytes, s.stream);
    if (rc) return rc;
    CK(cudaMemcpyAsync(s.h_keys, ctx->d_error + 1, sizeof(unsigned int), cudaMemcpyDeviceToHost, s.stream));
    CK(cudaEventRecord(s.ev_done, s.stream));
    s.in_flight = true;
    ctx->stats.reads += n; ctx->stats.bases += bases; ctx->stats.units += n_units; ctx->stats.h2d_bytes += v.bytes;
    return TREW_OK;
}

int trew_dev_upload(trew_ctx* ctx, const trew_batch* batch, trew_resident** out) {
    if (!ctx || !batch || !out) return TREW_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    uint32_t n = batch->n_reads;
    uint64_t bases = n ? batch->bit_off[n] : 0;
    trew_resident* r = new trew_resident();
    size_t bytes = batch_bytes(n, bases);
    std::vector<char> tmp(bytes, 0);
    BatchView v;
    batch_layout(tmp.data(), n, bases, &v);
    size_t words = (size_t)((bases + 31) / 32);
    if (n) {
        memcpy(v.bit_off, batch->bit_off, (size_t)(n + 1) * 4);
        memcpy(v.hi, batch->hi, words * 4); memcpy(v.lo, batch->lo, words * 4); memcpy(v.val, batch->val, words * 4);
    }
    CK(cudaMalloc(&r->d_buf, bytes));
    CK(cudaMemcpy(r->d_buf, tmp.data(), bytes, cudaMemcpyHostToDevice));
    r->batch.n_reads = n;
    r->batch.bit_off = (const unsigned int*)r->d_buf;
    r->batch.hi = (const unsigned int*)((char*)r->d_buf + ((char*)v.hi - tmp.data()));
    r->batch.lo = r->batch.hi + v.plane_words; r->batch.val = r->batch.lo + v.plane_words;
    r->n_reads = n; r->n_units = ctx->cfg.mode == TREW_MODE_PAIR ? n / 2 : n; r->max_read_len = batch->max_read_len; r->bases = bases;
    CK(cudaMalloc((void**)&r->d_survivors, 2 * (size_t)std::max<uint32_t>(r->n_units, 1) * sizeof(unsigned int)));
    CK(cudaMalloc((void**)&r->d_counters, kScanCounters * sizeof(unsigned int)));
    *out = r;
    return TREW_OK;
}

int trew_dev_scan_resident(trew_ctx* ctx, const trew_resident* rb) {
    if (!ctx || !rb) return TREW_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    trew_resident* r = const_cast<trew_resident*>(rb);
    ctx->keys_seen = std::max<unsigned int>(ctx->keys_seen, (unsigned int)(ctx->n_slots / 16 + 1));   // keys arrive outside the staging ring: streaming batches ask the device again
    if (r->ev_pending) { int rc0 = collect_prof(ctx); if (rc0) return rc0; }
    if (!r->ev[0]) for (int i = 0; i < 4; i++) CK(cudaEventCreate(&r->ev[i]));
    cudaStream_t st = (ctx->resident_streams == 2 && (ctx->resident_seq++ & 1)) ? ctx->aux_stream : ctx->main_stream;
    CK(cudaEventRecord(ctx->ev_a, st));
    int rc = launch_scan(ctx, r->batch, r->n_units, r->max_read_len, r->d_survivors, r->d_counters, &r->d_scratch,
                         &r->scratch_bytes, st, r->ev);
    r->ev_pending = true; ctx->pending_prof.push_back(r);
    if (rc) return rc;
    CK(cudaEventRecord(ctx->ev_b, st));
    ctx->stats.reads += r->n_reads; ctx->stats.bases += r->bases; ctx->stats.units += r->n_units;
    return TREW_OK;
}

void trew_dev_free_resident(trew_ctx* ctx, trew_resident* r) {
    if (!r) return;
    if (ctx) { cudaSetDevice(ctx->cfg.device); cudaStreamSynchronize(ctx->main_stream); cudaStreamSynchronize(ctx->aux_stream); collect_prof(ctx); }
    for (int i = 0; i < 4; i++) if (r->ev[i]) cudaEventDestroy(r->ev[i]);
    if (r->d_buf) cudaFree(r->d_buf);
    if (r->d_survivors) cudaFree(r->d_survivors);
    if (r->d_counters) cudaFree(r->d_counters);
    if (r->d_scratch) cudaFree(r->d_scratch);
    delete r;
}

int trew_dev_sync(trew_ctx* ctx) {
    if (!ctx) return TREW_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    for (auto& s : ctx->slots) { int rc = retire_slot(ctx, s); if (rc) return rc; }
    { int rc = join_aux(ctx); if (rc) return rc; }
    CK(cudaStreamSynchronize(ctx->main_stream));
    { int rc = collect_prof(ctx); if (rc) return rc; }
    return check_device_error(ctx);
}

}  // extern "C"

namespace {

// Compact the table into ctx->d_entries (cached until the table changes) and, on request, sort the rows by
// (table, k, seq) into ctx->d_sorted with three radix passes.
int export_entries(trew_ctx* ctx, bool need_sorted, const trew_entry** out, uint64_t* n_out) {
    int rc = trew_dev_sync(ctx);
    if (rc) return rc;
    if (!ctx->export_valid) {
        // count first (the table is sparse: sizing the entry array by the slot count would waste 128 MB)
        unsigned int n = 0;
        for (int pass = 0; pass < 2; pass++) {
            CK(cudaMemsetAsync(ctx->d_n, 0, sizeof(unsigned int), ctx->main_stream));
            if (pass == 0 && ctx->d_entries_cap == 0) {
                ctx->d_entries_cap = (size_t)1 << 20;
                CK(cudaMalloc((void**)&ctx->d_entries, ctx->d_entries_cap * sizeof(trew_entry)));
            }
            launch_compact(ctx->dcfg.slots, (unsigned int)ctx->n_slots, ctx->d_entries, ctx->d_n, ctx->main_stream,
                           (unsigned int)ctx->d_entries_cap);
            CK(cudaGetLastError());
            ctx->stats.kernel_launches += 1;
            CK(cudaMemcpyAsync(&n, ctx->d_n, sizeof(n), cudaMemcpyDeviceToHost, ctx->main_stream));
            CK(cudaStreamSynchronize(ctx->main_stream));
            if (n <= ctx->d_entries_cap) break;
            // the array was too small (the kernel only counted past its end): grow and compact again
            CK(cudaFree(ctx->d_entries));
            ctx->d_entries = nullptr;
            ctx->d_entries_cap = (size_t)n + n / 4 + 1024;
            CK(cudaMalloc((void**)&ctx->d_entries, ctx->d_entries_cap * sizeof(trew_entry)));
        }
        ctx->n_export = n;
        ctx->export_valid = true;
        ctx->sorted_valid = false;
    }
    const unsigned int n = (unsigned int)ctx->n_export;
    if (need_sorted && !ctx->sorted_valid) {
        if (n > ctx->d_sorted_cap) {
            if (ctx->d_sorted) CK(cudaFree(ctx->d_sorted));
            ctx->d_sorted = nullptr;
            ctx->d_sorted_cap = std::max<size_t>((size_t)n + n / 4 + 1024, (size_t)1 << 20);
            CK(cudaMalloc((void**)&ctx->d_sorted, ctx->d_sorted_cap * sizeof(trew_entry)));
        }
        if (n == 1) CK(cudaMemcpyAsync(ctx->d_sorted, ctx->d_entries, sizeof(trew_entry), cudaMemcpyDeviceToDevice, ctx->main_stream));
        if (n > 1) {
            const bool wide = ctx->cfg.max_mer > 32;
            size_t need = 0;
            CK(sort_entries_radix(ctx->d_entries, ctx->d_sorted, n, wide, nullptr, &need, ctx->main_stream));
            if (need > ctx->sort_tmp_bytes) {
                if (ctx->d_sort_tmp) CK(cudaFree(ctx->d_sort_tmp));
                ctx->d_sort_tmp = nullptr;
                ctx->sort_tmp_bytes = need + need / 4;
                CK(cudaMalloc(&ctx->d_sort_tmp, ctx->sort_tmp_bytes));
            }
            size_t bytes = ctx->sort_tmp_bytes;
            CK(sort_entries_radix(ctx->d_entries, ctx->d_sorted, n, wide, ctx->d_sort_tmp, &bytes, ctx->main_stream));
            ctx->stats.kernel_launches += wide ? 11 : 8;
        }
        CK(cudaStreamSynchronize(ctx->main_stream));
        ctx->sorted_valid = true;
    }
    if (out) *out = need_sorted ? ctx->d_sorted : ctx->d_entries;
    if (n_out) *n_out = n;
    return TREW_OK;
}

int export_sorted(trew_ctx* ctx, uint64_t* n_out) { return export_entries(ctx, false, nullptr, n_out); }

// n rows in device memory -> the pinned host array handed to the caller
int rows_to_host(trew_ctx* ctx, const trew_entry* d_rows, uint64_t n, const trew_entry** entries, uint64_t* n_entries) {
    // one D2H of the rows into a pinned array (grown on demand) that is handed to the caller as is
    size_t need_host = (size_t)n * sizeof(trew_entry) + 64;
    if (need_host > ctx->h_export_bytes) {
        if (ctx->h_export) CK(cudaFreeHost(ctx->h_export));
        ctx->h_export = nullptr;
        size_t cap = std::max(need_host * 2, (size_t)1 << 20);
        CK(cudaHostAlloc(&ctx->h_export, cap, cudaHostAllocDefault));
        ctx->h_export_bytes = cap;
    }
    if (n) {
        CK(cudaMemcpyAsync(ctx->h_export, d_rows, n * sizeof(trew_entry), cudaMemcpyDeviceToHost, ctx->main_stream));
        CK(cudaStreamSynchronize(ctx->main_stream));
    }
    ctx->stats.d2h_bytes += n * sizeof(trew_entry) + 4;
    if (entries) *entries = (const trew_entry*)ctx->h_export;
    if (n_entries) *n_entries = n;
    return TREW_OK;
}

// Unsorted rows in device memory (with repeated keys when they come from several tables: combine) -> [report filter] ->
// sort by (table, k, seq) -> [sum equal keys] -> host.  The filter runs first: it needs neither order nor unique keys
// (group totals add up either way), and what it keeps is a few thousand rows where the tables of a large file hold
// hundreds of thousands.
int finish_rows(trew_ctx* ctx, const trew_entry* d_in, uint64_t n_in, bool combine, const trew_entry** entries, uint64_t* n_entries) {
    auto ensure = [&](trew_entry** buf, size_t* cap, size_t want) -> int {
        if (want <= *cap) return TREW_OK;
        if (*buf) CK(cudaFree(*buf));
        *buf = nullptr;
        *cap = std::max<size_t>(want + want / 4 + 1024, (size_t)1 << 20);
        CK(cudaMalloc((void**)buf, *cap * sizeof(trew_entry)));
        return TREW_OK;
    };
    auto ensure_tmp = [&](size_t need) -> int {
        if (need <= ctx->sort_tmp_bytes) return TREW_OK;
        CK(cudaStreamSynchronize(ctx->main_stream));
        if (ctx->d_sort_tmp) CK(cudaFree(ctx->d_sort_tmp));
        ctx->d_sort_tmp = nullptr;
        ctx->sort_tmp_bytes = need + need / 4;
        CK(cudaMalloc(&ctx->d_sort_tmp, ctx->sort_tmp_bytes));
        return TREW_OK;
    };
    int rc;
    if ((rc = ensure(&ctx->d_sorted, &ctx->d_sorted_cap, (size_t)n_in)) != TREW_OK) return rc;
    if ((rc = ensure(&ctx->d_filtered, &ctx->d_filtered_cap, (size_t)n_in)) != TREW_OK) return rc;
    ctx->sorted_valid = false;   // d_sorted is reused below
    const bool wide = ctx->cfg.max_mer > 32;
    const trew_entry* src = d_in;
    unsigned int n = (unsigned int)n_in;
    if (ctx->report_min > 0 && n > 0) {
        size_t need = 0;
        CK(filter_report_rows(src, n, ctx->report_min, ctx->d_filtered, ctx->d_n, nullptr, &need, ctx->main_stream));
        if ((rc = ensure_tmp(need)) != TREW_OK) return rc;
        size_t bytes = ctx->sort_tmp_bytes;
        CK(filter_report_rows(src, n, ctx->report_min, ctx->d_filtered, ctx->d_n, ctx->d_sort_tmp, &bytes, ctx->main_stream));
        CK(cudaMemcpyAsync(&n, ctx->d_n, sizeof(n), cudaMemcpyDeviceToHost, ctx->main_stream));
        CK(cudaStreamSynchronize(ctx->main_stream));
        ctx->stats.kernel_launches += 5;
        src = ctx->d_filtered;
    }
    if (n == 1) CK(cudaMemcpyAsync(ctx->d_sorted, src, sizeof(trew_entry), cudaMemcpyDeviceToDevice, ctx->main_stream));
    if (n > 1) {
        size_t need = 0;
        CK(sort_entries_radix(src, ctx->d_sorted, n, wide, nullptr, &need, ctx->main_stream));
        if ((rc = ensure_tmp(need)) != TREW_OK) return rc;
        size_t bytes = ctx->sort_tmp_bytes;
        CK(sort_entries_radix(src, ctx->d_sorted, n, wide, ctx->d_sort_tmp, &bytes, ctx->main_stream));
        ctx->stats.kernel_launches += wide ? 11 : 8;
    }
    const trew_entry* rows = ctx->d_sorted;
    if (combine && n > 0) {   // the sort's input is no longer needed: d_filtered takes the combined rows
        size_t need = 0;
        CK(combine_sorted_rows(ctx->d_sorted, n, ctx->d_filtered, ctx->d_n, nullptr, &need, ctx->main_stream));
        if ((rc = ensure_tmp(need)) != TREW_OK) return rc;
        size_t bytes = ctx->sort_tmp_bytes;
        CK(combine_sorted_rows(ctx->d_sorted, n, ctx->d_filtered, ctx->d_n, ctx->d_sort_tmp, &bytes, ctx->main_stream));
        CK(cudaMemcpyAsync(&n, ctx->d_n, sizeof(n), cudaMemcpyDeviceToHost, ctx->main_stream));
        CK(cudaStreamSynchronize(ctx->main_stream));
        ctx->stats.kernel_launches += 3;
        rows = ctx->d_filtered;
    }
    return rows_to_host(ctx, rows, n, entries, n_entries);
}

// records made so far on ctx (synchronised); TREW_ERR_TABLE_FULL when they did not fit its capacity
int unit_record_count(trew_ctx* ctx, uint64_t* made) {
    unsigned long long m = 0;
    CK(cudaMemcpy(&m, &ctx->d_recs->n, sizeof(m), cudaMemcpyDeviceToHost));
    *made = m;
    if (m > ctx->rec_cap)
        return fail(ctx, TREW_ERR_TABLE_FULL, "unit records overflowed: %llu records made, capacity %llu (a capacity of %llu is enough)", m,
                    (unsigned long long)ctx->rec_cap, m);
    return TREW_OK;
}

// n unit records in ctx's device memory -> sorted by (unit, table, k, seq), equal keys summed -> the pinned host array
int records_to_host(trew_ctx* ctx, const trew_unit_record* d_in, uint64_t n_in, const trew_unit_record** recs, uint64_t* n_out) {
    if (n_in > 0x7fffffffULL) return fail(ctx, TREW_ERR_ARG, "too many unit records (%llu)", (unsigned long long)n_in);
    if (n_in > ctx->d_rec_out_cap) {
        if (ctx->d_rec_out) CK(cudaFree(ctx->d_rec_out));
        ctx->d_rec_out = nullptr;
        ctx->d_rec_out_cap = (size_t)n_in + n_in / 4 + 1024;
        CK(cudaMalloc((void**)&ctx->d_rec_out, ctx->d_rec_out_cap * sizeof(trew_unit_record)));
    }
    const unsigned int n = (unsigned int)n_in;
    const bool wide = ctx->cfg.max_mer > 32;
    size_t need = 0;
    CK(sort_combine_records(d_in, n, wide, ctx->d_rec_out, ctx->d_n, nullptr, &need, ctx->main_stream));
    if (need > ctx->sort_tmp_bytes) {
        CK(cudaStreamSynchronize(ctx->main_stream));
        if (ctx->d_sort_tmp) CK(cudaFree(ctx->d_sort_tmp));
        ctx->d_sort_tmp = nullptr;
        ctx->sort_tmp_bytes = need + need / 4;
        CK(cudaMalloc(&ctx->d_sort_tmp, ctx->sort_tmp_bytes));
    }
    size_t bytes = ctx->sort_tmp_bytes;
    CK(sort_combine_records(d_in, n, wide, ctx->d_rec_out, ctx->d_n, ctx->d_sort_tmp, &bytes, ctx->main_stream));
    unsigned int m = 0;
    CK(cudaMemcpyAsync(&m, ctx->d_n, sizeof(m), cudaMemcpyDeviceToHost, ctx->main_stream));
    CK(cudaStreamSynchronize(ctx->main_stream));
    const size_t need_host = (size_t)m * sizeof(trew_unit_record) + 64;
    if (need_host > ctx->h_rec_bytes) {
        if (ctx->h_rec) CK(cudaFreeHost(ctx->h_rec));
        ctx->h_rec = nullptr;
        const size_t cap = std::max(need_host + need_host / 2, (size_t)1 << 20);
        CK(cudaHostAlloc(&ctx->h_rec, cap, cudaHostAllocDefault));
        ctx->h_rec_bytes = cap;
    }
    if (m) CK(cudaMemcpy(ctx->h_rec, ctx->d_rec_out, (size_t)m * sizeof(trew_unit_record), cudaMemcpyDeviceToHost));
    ctx->stats.d2h_bytes += (uint64_t)m * sizeof(trew_unit_record) + 4;
    *recs = (const trew_unit_record*)ctx->h_rec;
    *n_out = m;
    return TREW_OK;
}

}  // namespace

extern "C" {

int trew_dev_export_device(trew_ctx* ctx, const trew_entry** d_entries, uint64_t* n_entries) {
    if (!ctx) return TREW_ERR_ARG;
    return export_entries(ctx, true, d_entries, n_entries);
}

int trew_dev_finish(trew_ctx* ctx, const trew_entry** entries, uint64_t* n_entries) {
    if (!ctx) return TREW_ERR_ARG;
    uint64_t n = 0;
    const trew_entry* d_rows = nullptr;
    if (ctx->report_min > 0) {   // filter first, then sort the few rows that are left
        int rc = export_entries(ctx, false, &d_rows, &n);
        if (rc) return rc;
        return finish_rows(ctx, d_rows, n, false, entries, n_entries);
    }
    int rc = export_entries(ctx, true, &d_rows, &n);
    if (rc) return rc;
    return rows_to_host(ctx, d_rows, n, entries, n_entries);
}

int trew_dev_finish_merged(trew_ctx* ctx, const trew_entry* const* d_lists, const uint64_t* n_rows, uint32_t n_lists,
                           const trew_entry** entries, uint64_t* n_entries) {
    if (!ctx || (n_lists && (!d_lists || !n_rows))) return TREW_ERR_ARG;
    uint64_t n0 = 0;
    const trew_entry* d_own = nullptr;
    int rc = export_entries(ctx, false, &d_own, &n0);
    if (rc) return rc;
    uint64_t total = n0;
    for (uint32_t i = 0; i < n_lists; i++) total += n_rows[i];
    if (total > 0xfffffff0ULL) return fail(ctx, TREW_ERR_ARG, "too many rows to merge (%llu)", (unsigned long long)total);
    // concatenate, sort, sum the counts of equal keys: the union of the tables without touching this context's table
    auto ensure = [&](trew_entry** buf, size_t* cap) -> int {
        if (total <= *cap) return TREW_OK;
        if (*buf) CK(cudaFree(*buf));
        *buf = nullptr;
        *cap = std::max<size_t>((size_t)total + total / 4 + 1024, (size_t)1 << 20);
        CK(cudaMalloc((void**)buf, *cap * sizeof(trew_entry)));
        return TREW_OK;
    };
    if ((rc = ensure(&ctx->d_concat, &ctx->d_concat_cap)) != TREW_OK) return rc;
    uint64_t at = 0;
    if (n0) CK(cudaMemcpyAsync(ctx->d_concat, d_own, n0 * sizeof(trew_entry), cudaMemcpyDeviceToDevice, ctx->main_stream));
    at += n0;
    for (uint32_t i = 0; i < n_lists; i++) {
        if (n_rows[i]) CK(cudaMemcpyAsync(ctx->d_concat + at, d_lists[i], n_rows[i] * sizeof(trew_entry), cudaMemcpyDeviceToDevice, ctx->main_stream));
        at += n_rows[i];
    }
    return finish_rows(ctx, ctx->d_concat, total, true, entries, n_entries);
}

int trew_dev_export_rows(trew_ctx* ctx, trew_entry* d_rows, uint64_t capacity_rows, uint64_t* n_rows) {
    if (!ctx || !n_rows) return TREW_ERR_ARG;
    uint64_t n = 0;
    const trew_entry* d_src = nullptr;
    int rc = export_entries(ctx, false, &d_src, &n);   // the merge does not care about row order
    if (rc) return rc;
    *n_rows = n;
    if (!d_rows) return TREW_OK;  // size query
    if (n > capacity_rows) return fail(ctx, TREW_ERR_ARG, "row buffer too small: %llu rows, capacity %llu", (unsigned long long)n,
                                       (unsigned long long)capacity_rows);
    if (n) CK(cudaMemcpyAsync(d_rows, d_src, n * sizeof(trew_entry), cudaMemcpyDeviceToDevice, ctx->main_stream));
    CK(cudaStreamSynchronize(ctx->main_stream));
    return TREW_OK;
}

int trew_dev_merge_rows(trew_ctx* ctx, const trew_entry* d_rows, uint64_t n_rows) {
    if (!ctx || (n_rows && !d_rows) || n_rows > 0xffffffffULL) return TREW_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    ctx->export_valid = false;
    ctx->table_used = true;
    ctx->keys_seen = std::max<unsigned int>(ctx->keys_seen, (unsigned int)(ctx->n_slots / 16 + 1));
    launch_merge_entries(ctx->dcfg, d_rows, (unsigned int)n_rows, ctx->main_stream);   // asynchronous: the next sync / export
    CK(cudaGetLastError());                                                             // waits and checks the error flag
    ctx->stats.kernel_launches += n_rows ? 1 : 0;
    return TREW_OK;
}

int trew_dev_set_report_filter(trew_ctx* ctx, uint32_t min_total) {
    if (!ctx) return TREW_ERR_ARG;
    ctx->report_min = min_total;
    return TREW_OK;
}

int trew_dev_reserve(trew_ctx* ctx, uint64_t expected_new_keys) {
    if (!ctx) return TREW_ERR_ARG;
    int rc = trew_dev_sync(ctx);
    if (rc) return rc;
    unsigned int keys = 0;
    CK(cudaMemcpy(&keys, ctx->d_error + 1, sizeof(keys), cudaMemcpyDeviceToHost));
    const uint64_t want = ((uint64_t)keys + expected_new_keys) * 4;   // load factor <= 1/4 once they are all in
    if (want <= ctx->n_slots) return TREW_OK;
    return grow_table_to(ctx, (size_t)std::min<uint64_t>(want, (uint64_t)1 << 28));
}

int trew_dev_reset(trew_ctx* ctx) {
    if (!ctx) return TREW_ERR_ARG;
    int rc = trew_dev_sync(ctx);
    if (rc && rc != TREW_ERR_TABLE_FULL) return rc;
    ctx->export_valid = false;
    // on the scan stream (the context's streams do not synchronise with the legacy default stream)
    CK(cudaMemsetAsync(ctx->dcfg.slots, 0, ctx->n_slots * sizeof(Slot), ctx->main_stream));
    CK(cudaMemsetAsync(ctx->d_error, 0, 2 * sizeof(unsigned int), ctx->main_stream));
    if (ctx->d_recs) CK(cudaMemsetAsync(&ctx->d_recs->n, 0, sizeof(unsigned long long), ctx->main_stream));
    CK(cudaStreamSynchronize(ctx->main_stream));
    ctx->unit_next = 0;
    ctx->table_used = false;
    ctx->keys_seen = 0;
    for (auto& sl : ctx->slots) *sl.h_keys = 0;
    return TREW_OK;
}

int trew_dev_enable_unit_records(trew_ctx* ctx, uint64_t capacity_records) {
    if (!ctx) return TREW_ERR_ARG;
    if (ctx->table_used) return fail(ctx, TREW_ERR_ARG, "unit records can only be switched on or off while the table is empty (after create or reset)");
    if (capacity_records > 0x7fffffffULL) return fail(ctx, TREW_ERR_ARG, "unit record capacity above 2^31 - 1");
    CK(cudaSetDevice(ctx->cfg.device));
    CK(cudaStreamSynchronize(ctx->main_stream));
    if (ctx->d_rec_buf) CK(cudaFree(ctx->d_rec_buf));
    if (ctx->d_recs) CK(cudaFree(ctx->d_recs));
    ctx->d_rec_buf = nullptr; ctx->d_recs = nullptr; ctx->dcfg.recs = nullptr; ctx->rec_cap = 0;
    if (capacity_records == 0) return TREW_OK;
    CK(cudaMalloc((void**)&ctx->d_rec_buf, capacity_records * sizeof(trew_unit_record)));
    CK(cudaMalloc((void**)&ctx->d_recs, sizeof(UnitRecs)));
    const UnitRecs r{ctx->d_rec_buf, (unsigned long long)capacity_records, 0ULL};
    CK(cudaMemcpy(ctx->d_recs, &r, sizeof(r), cudaMemcpyHostToDevice));
    ctx->rec_cap = capacity_records;
    ctx->dcfg.recs = ctx->d_recs;
    return TREW_OK;
}

int trew_dev_unit_records(trew_ctx* ctx, const trew_unit_record** recs, uint64_t* n) {
    if (!ctx || !recs || !n) return TREW_ERR_ARG;
    if (!ctx->d_recs) return fail(ctx, TREW_ERR_ARG, "unit records are off (trew_dev_enable_unit_records)");
    int rc = trew_dev_sync(ctx);
    if (rc) return rc;
    uint64_t made = 0;
    if ((rc = unit_record_count(ctx, &made)) != TREW_OK) return rc;
    return records_to_host(ctx, ctx->d_rec_buf, made, recs, n);
}

int trew_dev_get_stats(trew_ctx* ctx, trew_stats* out) {
    if (!ctx || !out) return TREW_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    unsigned long long s = 0;
    CK(cudaMemcpy(&s, ctx->d_total_surv, sizeof(s), cudaMemcpyDeviceToHost));
    ctx->stats.survivors = s;
    *out = ctx->stats;
    return TREW_OK;
}

// elapsed device time of the last trew_dev_scan_resident (ms); the caller must have synchronised
int trew_dev_last_resident_ms(trew_ctx* ctx, float* ms) {
    if (!ctx || !ms) return TREW_ERR_ARG;
    CK(cudaEventSynchronize(ctx->ev_b));
    CK(cudaEventElapsedTime(ms, ctx->ev_a, ctx->ev_b));
    return TREW_OK;
}

int trew_dev_timer_start(trew_ctx* ctx) {
    if (!ctx) return TREW_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    CK(cudaEventRecord(ctx->ev_t0, ctx->main_stream));
    return fork_aux(ctx);
}

int trew_dev_timer_stop(trew_ctx* ctx, float* ms) {
    if (!ctx || !ms) return TREW_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    { int rc = join_aux(ctx); if (rc) return rc; }
    CK(cudaEventRecord(ctx->ev_t1, ctx->main_stream));
    CK(cudaEventSynchronize(ctx->ev_t1));
    CK(cudaEventElapsedTime(ms, ctx->ev_t0, ctx->ev_t1));
    return TREW_OK;
}

int trew_dev_kernel_times(trew_ctx* ctx, double* screen_ms, double* decide_ms, double* exact_ms, uint64_t* n_scans) {
    if (!ctx) return TREW_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    { int rc0 = join_aux(ctx); if (rc0) return rc0; }
    CK(cudaStreamSynchronize(ctx->main_stream));
    int rc = collect_prof(ctx);
    if (rc) return rc;
    if (screen_ms) *screen_ms = ctx->screen_ms;
    if (decide_ms) *decide_ms = ctx->decide_ms;
    if (exact_ms) *exact_ms = ctx->exact_ms;
    if (n_scans) *n_scans = ctx->n_prof_scans;
    ctx->screen_ms = ctx->decide_ms = ctx->exact_ms = 0; ctx->n_prof_scans = 0;
    return TREW_OK;
}

int trew_synth_resident(trew_ctx* ctx, uint64_t seed, uint32_t n_reads, uint32_t read_len, uint32_t tel_ppm,
                        uint32_t half_ppm, uint32_t n_ppm, uint32_t sub_ppm, trew_resident** out) {
    return trew_synth_resident_ex(ctx, seed, n_reads, read_len, tel_ppm, half_ppm, n_ppm, sub_ppm, 0, out);
}

int trew_synth_resident_ex(trew_ctx* ctx, uint64_t seed, uint32_t n_reads, uint32_t read_len, uint32_t tel_ppm,
                           uint32_t half_ppm, uint32_t n_ppm, uint32_t sub_ppm, uint32_t flavor, trew_resident** out) {
    if (!ctx || !out || read_len == 0 || flavor > 2 || (uint64_t)n_reads * read_len >= 0xfffff000ULL) return TREW_ERR_ARG;
    CK(cudaSetDevice(ctx->cfg.device));
    auto thr = [](uint32_t ppm) { return (unsigned int)(((unsigned long long)ppm << 32) / 1000000ULL); };
    uint64_t bases = (uint64_t)n_reads * read_len;
    size_t bytes = batch_bytes(n_reads, bases);
    trew_resident* r = new trew_resident();
    CK(cudaMalloc(&r->d_buf, bytes));
    BatchView v;
    batch_layout(r->d_buf, n_reads, bases, &v);
    launch_synth(seed, n_reads, read_len, thr(tel_ppm), thr(half_ppm), thr(n_ppm), thr(sub_ppm), flavor, v.bit_off, v.hi, v.lo, v.val,
                 v.plane_words, ctx->main_stream);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->main_stream));
    r->batch.n_reads = n_reads; r->batch.bit_off = v.bit_off; r->batch.hi = v.hi; r->batch.lo = v.lo; r->batch.val = v.val;
    r->n_reads = n_reads; r->n_units = ctx->cfg.mode == TREW_MODE_PAIR ? n_reads / 2 : n_reads;
    r->max_read_len = read_len; r->bases = bases;
    CK(cudaMalloc((void**)&r->d_survivors, 2 * (size_t)std::max<uint32_t>(r->n_units, 1) * sizeof(unsigned int)));
    CK(cudaMalloc((void**)&r->d_counters, kScanCounters * sizeof(unsigned int)));
    *out = r;
    return TREW_OK;
}

int trew_dev_process_file(trew_ctx* ctx, const char* file1, int is_gz1, const char* file2, int is_gz2) {
    if (!ctx || !file1) return TREW_ERR_ARG;
    if ((ctx->cfg.mode == TREW_MODE_PAIR) != (file2 != nullptr)) return fail(ctx, TREW_ERR_ARG, "second file only in pair mode");
    // plain files: large blocks read and indexed by the pool; .gz: the inflate stream is sequential, keep blocks small
    const size_t chunk = 0;   // the reader picks the block size by input kind
    IngestResult r = ingest_file(ctx->cfg.mode, reader_slice_length(ctx), file1, is_gz1 != 0, file2, is_gz2 != 0, chunk,
                                 [&](const char* b1, const std::vector<int32_t>& l1, const char* b2, const std::vector<int32_t>& l2) {
                                     return trew_dev_submit_chunk(ctx, b1, l1.data(), (uint32_t)(l1.size() / 2), b2,
                                                                  b2 ? l2.data() : nullptr, b2 ? (uint32_t)(l2.size() / 2) : 0u);
                                 },
                                 ctx->pool, &ctx->ingest);
    if (r.status != TREW_OK && r.status != TREW_ERR_CUDA && !r.message.empty()) ctx->err = r.message;
    return r.status;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// several GPUs in one process (see include/trew_b200.h, "several GPUs in one process")
// ------------------------------------------------------------------------------------------------

struct trew_multi {
    std::vector<trew_ctx*> ctx;
    Pool* pool = nullptr;
    size_t next = 0;                  // device the next chunk goes to
    uint64_t unit_next = 0;           // unit ordinal of the group's next submitted unit
    std::string err;
    // per peer device: its rows as copied to the first device (device-0 memory)
    std::vector<trew_entry*> d_peer; std::vector<size_t> d_peer_cap;
};

namespace {
int mfail(trew_multi* m, int status, const std::string& msg) { if (m) m->err = msg; return status; }
// units of one submitted chunk (index-wise pairing in paired mode, src/kmer.cpp:321-322)
uint64_t chunk_units(const trew_ctx* x, uint32_t n1, uint32_t n2) { return x->cfg.mode == TREW_MODE_PAIR ? std::min(n1, n2) : n1; }
}  // namespace

extern "C" {

int trew_multi_create(const trew_config* cfg, const int32_t* devices, int32_t n_devices, trew_multi** out) {
    if (!cfg || !out || n_devices < 0 || (n_devices > 0 && !devices)) return TREW_ERR_ARG;
    *out = nullptr;
    std::vector<int32_t> dev;
    if (n_devices == 0) {
        int nd = 0;
        if (cudaGetDeviceCount(&nd) != cudaSuccess || nd <= 0) { g_create_error = "no CUDA device"; return TREW_ERR_CUDA; }
        for (int i = 0; i < nd; i++) dev.push_back(i);
    } else {
        dev.assign(devices, devices + n_devices);   // a device listed k times gets k contexts (used by the tests)
    }
    trew_multi* m = new trew_multi();
    m->pool = new Pool(default_host_threads(cfg->host_threads));
    // one thread per device: a primary context takes ~0.5 s to come up, and the devices do not wait for each other
    int rc = TREW_OK;
    {
        std::vector<trew_ctx*> made(dev.size(), nullptr);
        std::vector<int> rcs(dev.size(), TREW_OK);
        std::vector<std::string> errs(dev.size());
        std::vector<std::thread> th;
        auto make = [&](size_t i) {
            trew_config c = *cfg;
            c.device = dev[i];
            rcs[i] = create_ctx(&c, &made[i], errs[i], m->pool);
        };
        for (size_t i = 1; i < dev.size(); i++) th.emplace_back(make, i);
        make(0);
        for (auto& t : th) t.join();
        for (size_t i = 0; i < dev.size(); i++) {
            if (rcs[i] != TREW_OK && rc == TREW_OK) { rc = rcs[i]; g_create_error = errs[i]; }
            if (made[i]) m->ctx.push_back(made[i]);
        }
    }
    if (rc != TREW_OK) { trew_multi_destroy(m); return rc; }   // g_create_error holds the message
    // rows travel to the first device at end of file: direct NVLink copies where the devices are peers (the copy also
    // works without, staged through the host)
    for (size_t i = 1; i < m->ctx.size(); i++) {
        int can = 0;
        if (dev[i] != dev[0] && cudaDeviceCanAccessPeer(&can, dev[0], dev[i]) == cudaSuccess && can) {
            cudaSetDevice(dev[0]);
            cudaError_t e = cudaDeviceEnablePeerAccess(dev[i], 0);
            if (e != cudaSuccess) cudaGetLastError();   // already enabled is fine
        }
    }
    m->d_peer.assign(m->ctx.size(), nullptr);
    m->d_peer_cap.assign(m->ctx.size(), 0);
    *out = m;
    return TREW_OK;
}

void trew_multi_destroy(trew_multi* m) {
    if (!m) return;
    if (!m->ctx.empty()) {
        cudaSetDevice(m->ctx[0]->cfg.device);
        for (trew_entry* p : m->d_peer) if (p) cudaFree(p);
    }
    for (trew_ctx* x : m->ctx) trew_dev_destroy(x);
    delete m->pool;
    delete m;
}

int trew_multi_device_count(const trew_multi* m) { return m ? (int)m->ctx.size() : 0; }

const char* trew_multi_last_error(const trew_multi* m) { return m ? m->err.c_str() : g_create_error.c_str(); }

trew_ctx* trew_multi_ctx(trew_multi* m, int32_t i) { return m && i >= 0 && (size_t)i < m->ctx.size() ? m->ctx[(size_t)i] : nullptr; }

int trew_multi_submit_chunk(trew_multi* m, const char* buffer1, const int32_t* locs1, uint32_t n1, const char* buffer2,
                            const int32_t* locs2, uint32_t n2) {
    if (!m) return TREW_ERR_ARG;
    trew_ctx* x = m->ctx[m->next];
    m->next = (m->next + 1) % m->ctx.size();
    x->unit_next = m->unit_next;   // the group's submission order
    int rc = trew_dev_submit_chunk(x, buffer1, locs1, n1, buffer2, locs2, n2);
    if (rc != TREW_OK) return mfail(m, rc, x->err);
    m->unit_next += chunk_units(x, n1, n2);
    return TREW_OK;
}

int trew_multi_process_file(trew_multi* m, const char* file1, int is_gz1, const char* file2, int is_gz2) {
    if (!m || !file1) return TREW_ERR_ARG;
    trew_ctx* x0 = m->ctx[0];
    if ((x0->cfg.mode == TREW_MODE_PAIR) != (file2 != nullptr)) return mfail(m, TREW_ERR_ARG, "second file only in pair mode");
    // one reader, N consumers: every block of the file goes to the next device
    IngestResult r = ingest_file(x0->cfg.mode, reader_slice_length(x0), file1, is_gz1 != 0, file2, is_gz2 != 0, 0,
                                 [&](const char* b1, const std::vector<int32_t>& l1, const char* b2, const std::vector<int32_t>& l2) {
                                     return trew_multi_submit_chunk(m, b1, l1.data(), (uint32_t)(l1.size() / 2), b2, b2 ? l2.data() : nullptr,
                                                                    b2 ? (uint32_t)(l2.size() / 2) : 0u);
                                 },
                                 m->pool, &x0->ingest);
    if (r.status != TREW_OK && !r.message.empty()) m->err = r.message;
    return r.status;
}

int trew_multi_reset(trew_multi* m) {
    if (!m) return TREW_ERR_ARG;
    for (trew_ctx* x : m->ctx) { int rc = trew_dev_reset(x); if (rc != TREW_OK) return mfail(m, rc, x->err); }
    m->next = 0;
    m->unit_next = 0;
    return TREW_OK;
}

int trew_multi_finish(trew_multi* m, const trew_entry** entries, uint64_t* n_entries) {
    if (!m) return TREW_ERR_ARG;
    trew_ctx* x0 = m->ctx[0];
    const size_t nd = m->ctx.size();
    if (nd == 1) {
        int rc = trew_dev_finish(x0, entries, n_entries);
        return rc == TREW_OK ? rc : mfail(m, rc, x0->err);
    }
    // every peer compacts its table on its own device (they do so concurrently: the kernels are queued on all devices
    // before the first wait) ...
    std::vector<const trew_entry*> d_src(nd, nullptr);
    std::vector<uint64_t> n_rows(nd, 0);
    for (size_t i = 1; i < nd; i++) {
        int rc = export_entries(m->ctx[i], false, &d_src[i], &n_rows[i]);
        if (rc != TREW_OK) return mfail(m, rc, m->ctx[i]->err);
    }
    // ... and its rows are copied to the first device over NVLink
    trew_ctx* ctx = x0;   // for CK
    CK(cudaSetDevice(x0->cfg.device));
    std::vector<const trew_entry*> lists;
    std::vector<uint64_t> sizes;
    for (size_t i = 1; i < nd; i++) {
        if (n_rows[i] == 0) continue;
        if (n_rows[i] > m->d_peer_cap[i]) {
            if (m->d_peer[i]) CK(cudaFree(m->d_peer[i]));
            m->d_peer[i] = nullptr;
            m->d_peer_cap[i] = (size_t)n_rows[i] + n_rows[i] / 4 + 1024;
            CK(cudaMalloc((void**)&m->d_peer[i], m->d_peer_cap[i] * sizeof(trew_entry)));
        }
        CK(cudaMemcpyPeerAsync(m->d_peer[i], x0->cfg.device, d_src[i], m->ctx[i]->cfg.device, n_rows[i] * sizeof(trew_entry), x0->main_stream));
        lists.push_back(m->d_peer[i]);
        sizes.push_back(n_rows[i]);
    }
    int rc = trew_dev_finish_merged(x0, lists.data(), sizes.data(), (uint32_t)lists.size(), entries, n_entries);
    return rc == TREW_OK ? rc : mfail(m, rc, x0->err);
}

int trew_multi_enable_unit_records(trew_multi* m, uint64_t capacity_records) {
    if (!m) return TREW_ERR_ARG;
    for (trew_ctx* x : m->ctx) {
        int rc = trew_dev_enable_unit_records(x, capacity_records);
        if (rc != TREW_OK) return mfail(m, rc, x->err);
    }
    return TREW_OK;
}

int trew_multi_unit_records(trew_multi* m, const trew_unit_record** recs, uint64_t* n) {
    if (!m || !recs || !n) return TREW_ERR_ARG;
    trew_ctx* x0 = m->ctx[0];
    if (!x0->d_recs) return mfail(m, TREW_ERR_ARG, "unit records are off (trew_multi_enable_unit_records)");
    const size_t nd = m->ctx.size();
    std::vector<uint64_t> made(nd, 0);
    uint64_t total = 0, most = 0;
    int full = TREW_OK;
    for (size_t i = 0; i < nd; i++) {
        int rc = trew_dev_sync(m->ctx[i]);   // a count-table overflow is reported as such
        if (rc != TREW_OK) return mfail(m, rc, m->ctx[i]->err);
        rc = unit_record_count(m->ctx[i], &made[i]);
        if (rc == TREW_ERR_TABLE_FULL) full = rc;
        else if (rc != TREW_OK) return mfail(m, rc, m->ctx[i]->err);
        total += made[i]; most = std::max(most, made[i]);
    }
    if (full != TREW_OK)
        return mfail(m, full, "unit records overflowed on a device: " + std::to_string(most) + " records made, capacity " +
                                  std::to_string(x0->rec_cap) + " (a capacity of " + std::to_string(most) + " is enough)");
    if (nd == 1) {
        int rc = records_to_host(x0, x0->d_rec_buf, made[0], recs, n);
        return rc == TREW_OK ? rc : mfail(m, rc, x0->err);
    }
    // every device's records to the first device (units are disjoint across devices), then one sort
    trew_ctx* ctx = x0;   // for CK
    CK(cudaSetDevice(x0->cfg.device));
    if (total > x0->d_rec_cat_cap) {
        if (x0->d_rec_cat) CK(cudaFree(x0->d_rec_cat));
        x0->d_rec_cat = nullptr;
        x0->d_rec_cat_cap = (size_t)total + total / 4 + 1024;
        CK(cudaMalloc((void**)&x0->d_rec_cat, x0->d_rec_cat_cap * sizeof(trew_unit_record)));
    }
    uint64_t at = 0;
    for (size_t i = 0; i < nd; i++) {
        if (made[i])
            CK(cudaMemcpyPeerAsync(x0->d_rec_cat + at, x0->cfg.device, m->ctx[i]->d_rec_buf, m->ctx[i]->cfg.device,
                                   made[i] * sizeof(trew_unit_record), x0->main_stream));
        at += made[i];
    }
    int rc = records_to_host(x0, x0->d_rec_cat, total, recs, n);
    return rc == TREW_OK ? rc : mfail(m, rc, x0->err);
}

int trew_multi_set_report_filter(trew_multi* m, uint32_t min_total) {
    if (!m) return TREW_ERR_ARG;
    return trew_dev_set_report_filter(m->ctx[0], min_total);   // the first device copies the merged rows to the host
}

int trew_multi_get_stats(trew_multi* m, trew_stats* out) {
    if (!m || !out) return TREW_ERR_ARG;
    trew_stats t;
    memset(&t, 0, sizeof(t));
    for (trew_ctx* x : m->ctx) {
        trew_stats s;
        int rc = trew_dev_get_stats(x, &s);
        if (rc != TREW_OK) return mfail(m, rc, x->err);
        t.reads += s.reads; t.bases += s.bases; t.units += s.units; t.survivors += s.survivors;
        t.kernel_launches += s.kernel_launches; t.h2d_bytes += s.h2d_bytes; t.d2h_bytes += s.d2h_bytes;
        t.host_pack_bytes += s.host_pack_bytes; t.host_pack_ms += s.host_pack_ms;
        t.device_ms = std::max(t.device_ms, s.device_ms);
    }
    *out = t;
    return TREW_OK;
}

}  // extern "C"
