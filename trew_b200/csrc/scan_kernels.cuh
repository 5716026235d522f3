// Device-side declarations shared by scan_kernels.cu (kernels) and device_ctx.cu (host driver).
//
// Two kernels implement the reference's per-read scan-and-count (buffer_task*, src/kmer.cpp:80-985,
// with k_mer_check/k_mer_target, src/kmer.cpp:1894-2547):
//
//   (short single-end mode adds trew_exact_thread_kernel, one THREAD per survivor, in front of the warp kernel: see
//   exact_thread.cuh; the decide kernel then writes two survivor lists, one per exact kernel)
//   trew_filter_kernel  one THREAD per read/pair.  Bit-parallel, sound rejection test: for every probe
//                       window the routing would scan first and every period k, an upper bound U_k on
//                       the largest rotation-class count M_k is compared with the smallest count that
//                       would pass LOW_BASELINE.  Units where no (window, k) can pass emit nothing in
//                       the reference, so they are done; the rest go to a survivor list.
//   trew_exact_kernel   one WARP per survivor.  Re-does the reference's routing exactly: per-period
//                       class counts via match-bit runs + canonical rotations, the ascending-k
//                       selection with IEEE double ratios, and emission into the device count table.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/trew_b200.h"

namespace trew {

constexpr int kThrTableSize = 1025;  // thr[T] for T = 0..1024 valid windows
constexpr int kMaxWindow = 1023;     // longest window the exact kernel handles (32 lanes x 32 bits)

// 32-byte open-addressing slot of the device count table
struct __align__(32) Slot {
    unsigned long long seq_lo;
    unsigned long long seq_hi;
    unsigned long long count;
    unsigned int meta;   // table << 8 | k
    unsigned int state;  // 0 empty, 1 being written, 2 ready
};

// per-unit hit records (device memory): rows are appended at n, which keeps counting past cap
struct UnitRecs {
    trew_unit_record* buf;
    unsigned long long cap;
    unsigned long long n;
};

struct DevCfg {
    int mode, min_mer, max_mer, slice_len;
    double low, high;
    Slot* slots;
    unsigned int slot_mask;
    unsigned int* error_flag;        // [0] set to TREW_ERR_TABLE_FULL on overflow, [1] number of distinct keys inserted
    const unsigned short* thr_low;   // kThrTableSize entries: min M with (double)M/(double)T >= low; 0xFFFF for T = 0
    const unsigned short* thr_high;  // the same for the high baseline
    UnitRecs* recs;                  // nullptr: no records
    unsigned long long unit_base;    // ordinal of the batch's unit 0
};

struct DevBatch {
    unsigned int n_reads;
    const unsigned int* bit_off;
    const unsigned int* hi;
    const unsigned int* lo;
    const unsigned int* val;
};

struct ExactArgs {
    const unsigned int* survivors;
    const unsigned int* n_survivors;
    unsigned int* work_counter;      // zeroed before launch
    unsigned char* slice_scratch;    // long mode: per-warp (th, tl) per slice
    unsigned int slice_scratch_stride;  // bytes per warp
    int run_cap;                     // run-list capacity per warp (>= longest window + 1)
    unsigned long long* total_survivors;  // running total over all launches (statistics)
    int packed_probes;               // survivor entries carry the undecided-probe mask in bits 28..31
    int reverse;                     // the list grows downwards: entry idx is survivors[-idx]
    unsigned int exp_flags;          // experiments (TREW_EXACT_FLAGS): 1 = serial path for few runs in eval_k, 2 = no composition bound,
                                     // 4 = no thread-per-survivor kernel, 16 = long reads through the three-step thread path
};

// grid sizes (total blocks) of the three scan kernels; all three are grid-stride / work-counter kernels
struct LaunchPlan { int screen_blocks, decide_blocks, exact_blocks; };
LaunchPlan default_launch_plan(int sm_count);

// host-side launchers (scan_kernels.cu)
// deferred / n_deferred: scratch list of n_units entries + its counter (zeroed) for the screen kernel
void launch_filter(const DevCfg& cfg, const DevBatch& b, unsigned int n_units, unsigned int max_read_len,
                   unsigned int* deferred, unsigned int* n_deferred, unsigned int* survivors, unsigned int* n_survivors,
                   const LaunchPlan& plan, cudaStream_t stream, cudaEvent_t after_screen,
                   unsigned int* surv_b_top, unsigned int* n_surv_b, unsigned int* work_counter);
size_t exact_smem_bytes(int run_cap, bool wide);
cudaError_t prepare_exact(int run_cap_max);
void launch_exact(const DevCfg& cfg, const DevBatch& b, const ExactArgs& a, const LaunchPlan& plan, cudaStream_t stream);
int exact_warps_total(int sm_count);
// long reads through the thread path (exact_thread.cuh: statistics of every slice, the walks, the emissions -- three
// kernels); scratch: long_thread_scratch_bytes(s_cap, max_slices); what it cannot take lands in hard / n_hard
bool long_thread_path_applies(const DevCfg& cfg);
size_t long_thread_scratch_bytes(unsigned int s_cap, unsigned int max_slices);
void launch_long_thread(const DevCfg& cfg, const DevBatch& b, const unsigned int* survivors, const unsigned int* n_survivors,
                        int packed_probes, unsigned int s_cap, unsigned int max_slices, unsigned char* scratch, unsigned int* hard,
                        unsigned int* n_hard, unsigned long long* total_survivors, int sm_count, cudaStream_t stream);
// thread-per-survivor exact kernel (exact_thread.cuh): takes the survivors of a short-mode batch, appends the ones
// outside its limits to `hard` (counter n_hard, zeroed) for launch_exact
bool thread_path_applies(const DevCfg& cfg, unsigned int max_read_len);
void launch_exact_thread(const DevCfg& cfg, const DevBatch& b, const unsigned int* survivors, const unsigned int* n_survivors,
                         int packed_probes, unsigned int* hard, unsigned int* n_hard, unsigned long long* total_survivors, int sm_count,
                         int blocks_per_sm, unsigned int* work_counter, cudaStream_t stream);
// table_kernels.cu
void launch_compact(const Slot* slots, unsigned int n_slots, trew_entry* out, unsigned int* d_n, cudaStream_t stream, unsigned int cap);
// sort by (table, k, seq): sorted rows into d_out (d_entries untouched); wide = some key uses seq_hi (MAX_MER > 32);
// call with d_temp == nullptr to query *temp_bytes
cudaError_t sort_entries_radix(const trew_entry* d_entries, trew_entry* d_out, unsigned int n, bool wide, void* d_temp,
                               size_t* temp_bytes, cudaStream_t stream);
// sorted rows with repeated keys -> one row per key, counts summed (the union of several tables' rows)
cudaError_t combine_sorted_rows(const trew_entry* d_sorted, unsigned int n, trew_entry* d_out, unsigned int* d_n_out, void* d_temp,
                                size_t* temp_bytes, cudaStream_t stream);
// the rows of groups (k, folded key) whose high- or low-class total reaches min_total (what the report of a one-file run
// can show), order kept; d_temp == nullptr queries *temp_bytes
cudaError_t filter_report_rows(const trew_entry* d_rows, unsigned int n, unsigned int min_total, trew_entry* d_out, unsigned int* d_n_out,
                               void* d_temp, size_t* temp_bytes, cudaStream_t stream);
// validity plane from n 12-byte records (u32 block position, u64 mask of invalid bases): clears those bits of val
void launch_clear_invalid(unsigned int* val, const unsigned int* rec, unsigned int n, cudaStream_t stream);
void launch_merge_entries(const DevCfg& cfg, const trew_entry* entries, unsigned int n, cudaStream_t stream);

// unit records -> sorted by (unit, table, k, seq_hi, seq_lo) into d_out, equal keys summed, *d_n_out rows; wide = some key
// uses seq_hi; d_temp == nullptr queries *temp_bytes
cudaError_t sort_combine_records(const trew_unit_record* d_in, unsigned int n, bool wide, trew_unit_record* d_out, unsigned int* d_n_out,
                                 void* d_temp, size_t* temp_bytes, cudaStream_t stream);

// flavor 0: single reads (configs[1]); 1: pairs -- reads 2u, 2u+1 are the two ends of one fragment, both telomeric or
// neither, mate 2 on the opposite strand (configs[2]); 2: long reads whose first or last 0.5-5 kb are telomeric (configs[3])
void launch_synth(unsigned long long seed, unsigned int n_reads, unsigned int read_len, unsigned int tel_thr,
                  unsigned int half_thr, unsigned int n_thr, unsigned int sub_thr, unsigned int flavor, unsigned int* bit_off,
                  unsigned int* hi, unsigned int* lo, unsigned int* val, size_t plane_words, cudaStream_t stream);

}  // namespace trew
