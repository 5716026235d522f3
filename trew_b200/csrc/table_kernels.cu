// Count-table export: compaction of the open-addressing table into an array of trew_entry, device-side radix sort by
// (table, k, seq) and the cross-rank merge kernel.  Stands in for the end of buffer_task* (the six ResultMaps
// handed to process_output, src/kmer.cpp:1486-1515).
#include "scan_kernels.cuh"

#include <algorithm>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

namespace trew {

typedef unsigned int u32;
typedef unsigned long long u64;

// slot -> entry; unused slots are skipped, the survivors are appended in arbitrary order.  A warp looks at 128 slots per
// round -- four independent 16-byte loads of the halves that hold count / meta / state per lane, so that the (mostly empty)
// table streams at memory speed instead of one dependent 32-byte load per ballot -- and fetches the key halves of used
// slots only.
__global__ void compact_kernel(const Slot* __restrict__ slots, u32 n_slots, trew_entry* __restrict__ out, u32* __restrict__ d_n, u32 cap) {
    const u32 lane = threadIdx.x & 31;
    const u32 warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (u32 i0 = warp * 128u; i0 < n_slots; i0 += n_warps * 128u) {   // n_slots is a multiple of 128
        uint4 h[4];
#pragma unroll
        for (int r = 0; r < 4; r++) h[r] = __ldg(reinterpret_cast<const uint4*>(slots + i0 + 32u * r + lane) + 1);   // count lo, count hi, meta, state
        u32 m[4], total = 0;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            m[r] = __ballot_sync(0xffffffffu, h[r].w == 2u && (h[r].x | h[r].y) != 0u);
            total += (u32)__popc(m[r]);
        }
        if (total == 0u) continue;
        // one atomic per 128 slots: every add goes to the same address, and same-address atomics retire one at a time
        u32 base = 0;
        if (lane == 0) base = atomicAdd(d_n, total);
        base = __shfl_sync(0xffffffffu, base, 0);
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const u32 o = base + __popc(m[r] & ((1u << lane) - 1u));
            if (((m[r] >> lane) & 1u) && o < cap) {  // past the end of the array: count only, the host grows it and runs again
                const uint4 key = __ldg(reinterpret_cast<const uint4*>(slots + i0 + 32u * r + lane));
                trew_entry e;
                e.seq_lo = (u64)key.x | ((u64)key.y << 32); e.seq_hi = (u64)key.z | ((u64)key.w << 32);
                e.count = (u64)h[r].x | ((u64)h[r].y << 32);
                e.table = (int)(h[r].z >> 8); e.k = (int)(h[r].z & 0xffu);
                out[o] = e;
            }
            base += (u32)__popc(m[r]);
        }
    }
}

void launch_compact(const Slot* slots, unsigned int n_slots, trew_entry* out, unsigned int* d_n, cudaStream_t stream, unsigned int cap) {
    // n_slots is a power of two >= 1024
    compact_kernel<<<592, 256, 0, stream>>>(slots, n_slots, out, d_n, cap);
}

// ---- validity plane from a list: the streaming path sends one record per 64-base block that holds a base other than
// A/C/G/T (u32 bit position of the block, u64 mask of its invalid bases; 12 bytes) instead of the whole plane; the
// plane is set to ones by a memset and the recorded bits are cleared here.
__global__ void clear_invalid_kernel(u32* __restrict__ val, const u32* __restrict__ rec, u32 n) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const u32 pos = rec[3 * (size_t)i];
        const u64 z = (u64)rec[3 * (size_t)i + 1] | ((u64)rec[3 * (size_t)i + 2] << 32);
        const u32 sh = pos & 31u;
        const u64 lo = z << sh;
        const u32 m0 = (u32)lo, m1 = (u32)(lo >> 32), m2 = sh ? (u32)(z >> (64u - sh)) : 0u;
        u32* w = val + (pos >> 5);
        if (m0) atomicAnd(w, ~m0);
        if (m1) atomicAnd(w + 1, ~m1);
        if (m2) atomicAnd(w + 2, ~m2);
    }
}

void launch_clear_invalid(unsigned int* val, const unsigned int* rec, unsigned int n, cudaStream_t stream) {
    if (n == 0) return;
    const unsigned int blocks = (n + 255u) / 256u;
    clear_invalid_kernel<<<blocks < 592u ? blocks : 592u, 256, 0, stream>>>(val, rec, n);
}

// ---- sort by (table, k, seq): three stable LSD passes over (seq_lo, seq_hi, table << 8 | k) with a row index as payload, then one
// gather of the 32-byte rows.  Moves 12 bytes per row and pass instead of merge-sorting 32-byte rows by a comparator.

__global__ void key_from_entries_kernel(const trew_entry* __restrict__ e, const u32* __restrict__ idx, u32 n, int which,
                                        u64* __restrict__ key64, unsigned short* __restrict__ key16, u32* __restrict__ idx_out) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const u32 j = idx ? idx[i] : i;
        if (which == 0) { key64[i] = e[j].seq_lo; idx_out[i] = i; }
        else if (which == 1) key64[i] = e[j].seq_hi;
        else key16[i] = (unsigned short)(((u32)e[j].table << 8) | (u32)e[j].k);
    }
}

__global__ void gather_entries_kernel(const trew_entry* __restrict__ e, const u32* __restrict__ idx, u32 n, trew_entry* __restrict__ out) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = e[idx[i]];
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// d_out receives the sorted rows (d_entries is left untouched).  Call with d_temp == nullptr to query *temp_bytes.
cudaError_t sort_entries_radix(const trew_entry* d_entries, trew_entry* d_out, unsigned int n, bool wide, void* d_temp,
                               size_t* temp_bytes, cudaStream_t stream) {
    size_t cub64 = 0, cub16 = 0;
    cub::DoubleBuffer<u64> k64(nullptr, nullptr);
    cub::DoubleBuffer<unsigned short> k16(nullptr, nullptr);
    cub::DoubleBuffer<u32> ix(nullptr, nullptr);
    cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, cub64, k64, ix, (int)n, 0, 64, stream);
    if (e != cudaSuccess) return e;
    e = cub::DeviceRadixSort::SortPairs(nullptr, cub16, k16, ix, (int)n, 0, 11, stream);
    if (e != cudaSuccess) return e;
    const size_t cub_bytes = align256(std::max(cub64, cub16));
    const size_t need = 2 * align256((size_t)n * 8) + 2 * align256((size_t)n * 4) + 2 * align256((size_t)n * 2) + cub_bytes;
    if (!d_temp) { *temp_bytes = need; return cudaSuccess; }
    if (*temp_bytes < need) return cudaErrorInvalidValue;
    char* p = (char*)d_temp;
    u64* ka = (u64*)p; p += align256((size_t)n * 8);
    u64* kb = (u64*)p; p += align256((size_t)n * 8);
    u32* ia = (u32*)p; p += align256((size_t)n * 4);
    u32* ib = (u32*)p; p += align256((size_t)n * 4);
    unsigned short* sa = (unsigned short*)p; p += align256((size_t)n * 2);
    unsigned short* sb = (unsigned short*)p; p += align256((size_t)n * 2);
    void* cub_tmp = p;
    const int blocks = (int)std::min<unsigned int>((n + 255) / 256, 4736u);
    k64 = cub::DoubleBuffer<u64>(ka, kb);
    ix = cub::DoubleBuffer<u32>(ia, ib);
    key_from_entries_kernel<<<blocks, 256, 0, stream>>>(d_entries, nullptr, n, 0, k64.Current(), nullptr, ix.Current());
    size_t tb = cub_bytes;
    e = cub::DeviceRadixSort::SortPairs(cub_tmp, tb, k64, ix, (int)n, 0, 64, stream);
    if (e != cudaSuccess) return e;
    if (wide) {
        key_from_entries_kernel<<<blocks, 256, 0, stream>>>(d_entries, ix.Current(), n, 1, k64.Current(), nullptr, nullptr);
        tb = cub_bytes;
        e = cub::DeviceRadixSort::SortPairs(cub_tmp, tb, k64, ix, (int)n, 0, 64, stream);
        if (e != cudaSuccess) return e;
    }
    k16 = cub::DoubleBuffer<unsigned short>(sa, sb);
    key_from_entries_kernel<<<blocks, 256, 0, stream>>>(d_entries, ix.Current(), n, 2, nullptr, k16.Current(), nullptr);
    tb = cub_bytes;
    e = cub::DeviceRadixSort::SortPairs(cub_tmp, tb, k16, ix, (int)n, 0, 11, stream);
    if (e != cudaSuccess) return e;
    gather_entries_kernel<<<blocks, 256, 0, stream>>>(d_entries, ix.Current(), n, d_out);
    return cudaGetLastError();
}

// ---- union of several tables' rows: after the sort equal keys are adjacent; the first row of every key sums its run ----

__device__ __forceinline__ bool same_key(const trew_entry& a, const trew_entry& b) {
    return a.seq_lo == b.seq_lo && a.seq_hi == b.seq_hi && a.table == b.table && a.k == b.k;
}

__global__ void head_flags_kernel(const trew_entry* __restrict__ e, u32 n, u32* __restrict__ flags) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        flags[i] = (i == 0 || !same_key(e[i], e[i - 1])) ? 1u : 0u;
}

__global__ void combine_runs_kernel(const trew_entry* __restrict__ e, u32 n, const u32* __restrict__ flags, const u32* __restrict__ pos,
                                    trew_entry* __restrict__ out, u32* __restrict__ n_out) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (!flags[i]) continue;
        trew_entry r = e[i];
        for (u32 j = i + 1; j < n && !flags[j]; j++) r.count += e[j].count;
        out[pos[i]] = r;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *n_out = n ? pos[n - 1] + flags[n - 1] : 0u;
}

// sorted rows with repeated keys -> one row per key with the counts summed.  d_temp == nullptr queries *temp_bytes.
cudaError_t combine_sorted_rows(const trew_entry* d_sorted, unsigned int n, trew_entry* d_out, unsigned int* d_n_out, void* d_temp,
                                size_t* temp_bytes, cudaStream_t stream) {
    size_t scan_bytes = 0;
    cudaError_t e = cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (u32*)nullptr, (u32*)nullptr, (int)n, stream);
    if (e != cudaSuccess) return e;
    const size_t need = 2 * align256((size_t)n * 4) + align256(scan_bytes);
    if (!d_temp) { *temp_bytes = need; return cudaSuccess; }
    if (*temp_bytes < need) return cudaErrorInvalidValue;
    char* p = (char*)d_temp;
    u32* flags = (u32*)p; p += align256((size_t)n * 4);
    u32* pos = (u32*)p; p += align256((size_t)n * 4);
    const int blocks = (int)std::min<unsigned int>((n + 255) / 256, 4736u);
    if (n) head_flags_kernel<<<blocks, 256, 0, stream>>>(d_sorted, n, flags);
    size_t sb = align256(scan_bytes);
    e = cub::DeviceScan::ExclusiveSum(p, sb, flags, pos, (int)n, stream);
    if (e != cudaSuccess) return e;
    combine_runs_kernel<<<n ? blocks : 1, 256, 0, stream>>>(d_sorted, n, flags, pos, d_out, d_n_out);
    return cudaGetLastError();
}

// ---- unit records: sort by (unit, table, k, seq_hi, seq_lo) the way sort_entries_radix sorts rows -- stable LSD passes over
// the key fields with a row index as payload, one gather -- then sum the rows of equal keys as combine_sorted_rows does.

__global__ void key_from_records_kernel(const trew_unit_record* __restrict__ r, const u32* __restrict__ idx, u32 n, int which,
                                        u64* __restrict__ key64, unsigned short* __restrict__ key16, u32* __restrict__ idx_out) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const u32 j = idx ? idx[i] : i;
        if (which == 0) { key64[i] = r[j].seq_lo; idx_out[i] = i; }
        else if (which == 1) key64[i] = r[j].seq_hi;
        else if (which == 2) key16[i] = (unsigned short)(((u32)r[j].table << 8) | (u32)r[j].k);
        else key64[i] = r[j].unit;
    }
}

__device__ __forceinline__ bool same_record_key(const trew_unit_record& a, const trew_unit_record& b) {
    return a.unit == b.unit && a.seq_lo == b.seq_lo && a.seq_hi == b.seq_hi && a.table == b.table && a.k == b.k;
}

// gathers the sorted order and flags the first row of every key
__global__ void gather_records_kernel(const trew_unit_record* __restrict__ r, const u32* __restrict__ idx, u32 n,
                                      trew_unit_record* __restrict__ out, u32* __restrict__ flags) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        out[i] = r[idx[i]];
        flags[i] = (i == 0 || !same_record_key(r[idx[i]], r[idx[i - 1]])) ? 1u : 0u;
    }
}

__global__ void combine_records_kernel(const trew_unit_record* __restrict__ r, u32 n, const u32* __restrict__ flags,
                                       const u32* __restrict__ pos, trew_unit_record* __restrict__ out, u32* __restrict__ n_out) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (!flags[i]) continue;
        trew_unit_record x = r[i];
        for (u32 j = i + 1; j < n && !flags[j]; j++) x.count += r[j].count;
        out[pos[i]] = x;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *n_out = n ? pos[n - 1] + flags[n - 1] : 0u;
}

cudaError_t sort_combine_records(const trew_unit_record* d_in, unsigned int n, bool wide, trew_unit_record* d_out, unsigned int* d_n_out,
                                 void* d_temp, size_t* temp_bytes, cudaStream_t stream) {
    size_t cub64 = 0, cub16 = 0, scan_bytes = 0;
    cub::DoubleBuffer<u64> k64(nullptr, nullptr);
    cub::DoubleBuffer<unsigned short> k16(nullptr, nullptr);
    cub::DoubleBuffer<u32> ix(nullptr, nullptr);
    cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, cub64, k64, ix, (int)n, 0, 64, stream);
    if (e != cudaSuccess) return e;
    e = cub::DeviceRadixSort::SortPairs(nullptr, cub16, k16, ix, (int)n, 0, 11, stream);
    if (e != cudaSuccess) return e;
    e = cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (u32*)nullptr, (u32*)nullptr, (int)n, stream);
    if (e != cudaSuccess) return e;
    const size_t cub_bytes = align256(std::max(std::max(cub64, cub16), scan_bytes));
    const size_t rows = align256((size_t)n * sizeof(trew_unit_record));
    const size_t need = 2 * align256((size_t)n * 8) + 4 * align256((size_t)n * 4) + 2 * align256((size_t)n * 2) + rows + cub_bytes;
    if (!d_temp) { *temp_bytes = need; return cudaSuccess; }
    if (*temp_bytes < need) return cudaErrorInvalidValue;
    char* p = (char*)d_temp;
    u64* ka = (u64*)p; p += align256((size_t)n * 8);
    u64* kb = (u64*)p; p += align256((size_t)n * 8);
    u32* ia = (u32*)p; p += align256((size_t)n * 4);
    u32* ib = (u32*)p; p += align256((size_t)n * 4);
    u32* flags = (u32*)p; p += align256((size_t)n * 4);
    u32* pos = (u32*)p; p += align256((size_t)n * 4);
    unsigned short* sa = (unsigned short*)p; p += align256((size_t)n * 2);
    unsigned short* sb = (unsigned short*)p; p += align256((size_t)n * 2);
    trew_unit_record* sorted = (trew_unit_record*)p; p += rows;
    void* cub_tmp = p;
    const int blocks = (int)std::min<unsigned int>((n + 255) / 256, 4736u);
    if (n) {
        k64 = cub::DoubleBuffer<u64>(ka, kb);
        ix = cub::DoubleBuffer<u32>(ia, ib);
        k16 = cub::DoubleBuffer<unsigned short>(sa, sb);
        size_t tb;
        key_from_records_kernel<<<blocks, 256, 0, stream>>>(d_in, nullptr, n, 0, k64.Current(), nullptr, ix.Current());
        e = cub::DeviceRadixSort::SortPairs(cub_tmp, tb = cub_bytes, k64, ix, (int)n, 0, 64, stream);
        if (e != cudaSuccess) return e;
        if (wide) {
            key_from_records_kernel<<<blocks, 256, 0, stream>>>(d_in, ix.Current(), n, 1, k64.Current(), nullptr, nullptr);
            e = cub::DeviceRadixSort::SortPairs(cub_tmp, tb = cub_bytes, k64, ix, (int)n, 0, 64, stream);
            if (e != cudaSuccess) return e;
        }
        key_from_records_kernel<<<blocks, 256, 0, stream>>>(d_in, ix.Current(), n, 2, nullptr, k16.Current(), nullptr);
        e = cub::DeviceRadixSort::SortPairs(cub_tmp, tb = cub_bytes, k16, ix, (int)n, 0, 11, stream);
        if (e != cudaSuccess) return e;
        key_from_records_kernel<<<blocks, 256, 0, stream>>>(d_in, ix.Current(), n, 3, k64.Current(), nullptr, nullptr);
        e = cub::DeviceRadixSort::SortPairs(cub_tmp, tb = cub_bytes, k64, ix, (int)n, 0, 64, stream);
        if (e != cudaSuccess) return e;
        gather_records_kernel<<<blocks, 256, 0, stream>>>(d_in, ix.Current(), n, sorted, flags);
    }
    size_t sb2 = cub_bytes;
    e = cub::DeviceScan::ExclusiveSum(cub_tmp, sb2, flags, pos, (int)n, stream);
    if (e != cudaSuccess) return e;
    combine_records_kernel<<<n ? blocks : 1, 256, 0, stream>>>(sorted, n, flags, pos, d_out, d_n_out);
    return cudaGetLastError();
}

// ---- report filter: only the rows that can reach the report of a one-file run ------------------------------------------
//
// process_output prints an entry when forward + backward + both >= 10 (ABS_MIN_PRINT_COUNT, src/kmer.cpp:1615-1620) and
// final_process_output scores entries with a sum >= 10, then looks the scored keys up in BOTH classes
// (src/kmer.cpp:2604-2650, 2693-2761).  Every count of such an entry comes from rows whose key folds to the entry's
// (k, min(seq, crc(seq))) -- forward / backward / both rows of either strand (src/kmer.cpp:1518-1549).  So a row
// matters iff its GROUP (k, folded key), classes high and low taken together, has a per-class total >= min_total in at
// least one class.  Groups are accumulated under a 64-bit fingerprint of (k, folded key): two groups that collide are
// merged, which can only keep more rows (the host recomputes everything exactly from the rows it gets).
// Most rows of a large file are one- and two-window repeats an N made (exactly as in the reference); none of them
// prints, and without the filter they are most of the device-to-host copy.

typedef unsigned __int128 u128;

__device__ __forceinline__ u128 filt_canon(u128 w, int k) {
    u128 best = w, cur = w;
    const int sh = 2 * (k - 1);
    for (int r = 1; r < k; r++) { cur = ((cur & 3) << sh) | (cur >> 2); best = cur < best ? cur : best; }
    return best;
}
__device__ __forceinline__ u128 filt_fold(u128 w, int k) {   // min(w, canonical rotation of the reverse complement)
    u128 r = 0, x = w;
    for (int i = 0; i < k; i++) { r = (r << 2) | (3 - (x & 3)); x >>= 2; }
    const u128 t = filt_canon(r, k);
    // rows of the forward / backward tables hold canonical rotations; 'both' rows from the large-k path may not, and fold
    // with their own canonical rotation's group
    const u128 c = filt_canon(w, k);
    return t < c ? t : c;
}
__device__ __forceinline__ u64 filt_tag(const trew_entry& e) {
    const u128 f = filt_fold(((u128)e.seq_hi << 64) | e.seq_lo, e.k);
    u64 x = (u64)f ^ ((u64)(f >> 64) * 0x9e3779b97f4a7c15ULL) ^ ((u64)e.k << 56);
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x | 1ULL;   // 0 = empty slot
}

struct FiltGroup { u64 tag; u32 tot[2]; };

__global__ void filter_accumulate_kernel(const trew_entry* __restrict__ e, u32 n, FiltGroup* __restrict__ g, u32 gmask, u32 cap_add,
                                         u64* __restrict__ tags) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const u64 tag = filt_tag(e[i]);
        tags[i] = tag;
        const u32 add = (u32)(e[i].count < (u64)cap_add ? e[i].count : (u64)cap_add);   // saturating: only ">= min_total" matters
        u32 s = (u32)(tag >> 20) & gmask;
        for (;;) {
            const u64 old = atomicCAS((unsigned long long*)&g[s].tag, 0ULL, (unsigned long long)tag);
            if (old == 0ULL || old == tag) { atomicAdd(&g[s].tot[e[i].table & 1], add); break; }
            s = (s + 1) & gmask;
        }
    }
}

__global__ void filter_flags_kernel(const trew_entry* __restrict__ e, u32 n, const FiltGroup* __restrict__ g, u32 gmask, u32 min_total,
                                    const u64* __restrict__ tags, u32* __restrict__ flags) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const u64 tag = tags[i];
        u32 s = (u32)(tag >> 20) & gmask;
        while (g[s].tag != tag) s = (s + 1) & gmask;
        flags[i] = (g[s].tot[0] >= min_total || g[s].tot[1] >= min_total) ? 1u : 0u;
    }
}

__global__ void filter_scatter_kernel(const trew_entry* __restrict__ e, u32 n, const u32* __restrict__ flags, const u32* __restrict__ pos,
                                      trew_entry* __restrict__ out, u32* __restrict__ n_out) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        if (flags[i]) out[pos[i]] = e[i];
    if (blockIdx.x == 0 && threadIdx.x == 0) *n_out = n ? pos[n - 1] + flags[n - 1] : 0u;
}

// d_rows (n rows, any order) -> d_out: the rows of groups with a per-class total >= min_total, order kept.
// d_temp == nullptr queries *temp_bytes.
cudaError_t filter_report_rows(const trew_entry* d_rows, unsigned int n, unsigned int min_total, trew_entry* d_out, unsigned int* d_n_out,
                               void* d_temp, size_t* temp_bytes, cudaStream_t stream) {
    size_t scan_bytes = 0;
    cudaError_t err = cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (u32*)nullptr, (u32*)nullptr, (int)n, stream);
    if (err != cudaSuccess) return err;
    size_t gslots = 1024;
    while (gslots < (size_t)n * 2) gslots <<= 1;
    const size_t need = align256(gslots * sizeof(FiltGroup)) + align256((size_t)n * 8) + 2 * align256((size_t)n * 4) + align256(scan_bytes);
    if (!d_temp) { *temp_bytes = need; return cudaSuccess; }
    if (*temp_bytes < need) return cudaErrorInvalidValue;
    char* p = (char*)d_temp;
    FiltGroup* g = (FiltGroup*)p; p += align256(gslots * sizeof(FiltGroup));
    u64* tags = (u64*)p; p += align256((size_t)n * 8);
    u32* flags = (u32*)p; p += align256((size_t)n * 4);
    u32* pos = (u32*)p; p += align256((size_t)n * 4);
    const int blocks = (int)std::min<unsigned int>((n + 255) / 256, 4736u);
    err = cudaMemsetAsync(g, 0, gslots * sizeof(FiltGroup), stream);
    if (err != cudaSuccess) return err;
    if (n) {
        filter_accumulate_kernel<<<blocks, 256, 0, stream>>>(d_rows, n, g, (u32)(gslots - 1), min_total, tags);
        filter_flags_kernel<<<blocks, 256, 0, stream>>>(d_rows, n, g, (u32)(gslots - 1), min_total, tags, flags);
    }
    size_t sb = align256(scan_bytes);
    err = cub::DeviceScan::ExclusiveSum(p, sb, flags, pos, (int)n, stream);
    if (err != cudaSuccess) return err;
    filter_scatter_kernel<<<n ? blocks : 1, 256, 0, stream>>>(d_rows, n, flags, pos, d_out, d_n_out);
    return cudaGetLastError();
}

}  // namespace trew
