// Host build of the thread-per-read exact routing with a RECORDING emission: every emission is attributed to the unit
// (read, pair) being routed, as the device kernels' REC instantiations do, so tests/test_unit_records.py can diff the
// per-unit records against the CPU oracle's without a GPU.  Reuses the loader of exact_thread_check.cpp.  Test
// infrastructure.
#include "exact_thread_check.cpp"

namespace {
typedef std::map<std::tuple<uint64_t, int, int, uint64_t, uint64_t>, uint64_t> Records;   // (unit, table, k, hi, lo) -> count
struct RecordEmit {
    Records* r; uint64_t unit;
    void operator()(int table, int k, u64 key, uint64_t count) { (*r)[std::make_tuple(unit, table, k, (uint64_t)0, key)] += count; }
    void operator()(int table, int k, u128 key, uint64_t count) {
        (*r)[std::make_tuple(unit, table, k, (uint64_t)(key >> 64), (uint64_t)key)] += count;
    }
};
inline int read_len(const int32_t* locs, int r) { return locs[2 * r + 1] >= locs[2 * r] ? locs[2 * r + 1] - locs[2 * r] + 1 : 0; }

template <class K>
bool route_unit(int mode, const char* buf1, const int32_t* locs1, const char* buf2, const int32_t* locs2, int r, int min_mer, int max_mer,
                int slice_len, const unsigned short* thr_low, const unsigned short* thr_high, RecordEmit& emit) {
    u32 work[Lay<K>::WORDS];
    memset(work, 0xA5, sizeof(work));   // the workspace is not cleared between units on the device either
    Mem m{work, 1};
    const int n = read_len(locs1, r);
    if (mode == 0) {
        if (n > kMaxRead) return n < 2 * min_mer;
        StringLoad load{m, {buf1 + locs1[2 * r], nullptr}};
        return route_short_thread<K>(m, n, 7u, min_mer, max_mer, thr_low, thr_high, load, emit);
    }
    if (mode == 1) {
        StringLoad load{m, {buf1 + locs1[2 * r], buf2 + locs2[2 * r]}};
        return route_pair_thread<K>(m, n, read_len(locs2, r), min_mer, max_mer, thr_low, thr_high, load, emit);
    }
    if (n < slice_len) return true;   // the reader drops these (src/kmer.cpp:1184)
    if (sizeof(K) != 8 || max_mer > 32 || slice_len > kMaxRead) return false;
    StringLoad load{m, {buf1 + locs1[2 * r], nullptr}};
    ClsSpill<u64> x;
    LongGeom g(n, slice_len);
    std::vector<u32> stats((size_t)g.snum + 1, 0u);
    for (int t = 1; t <= g.snum; t++)
        if (g.len(t) <= kMaxRead) stats[(size_t)t] = long_slice_stats(m, g, t, min_mer, max_mer, thr_low, thr_high, load, x);
    std::vector<LongTask> tasks;
    auto stat = [&](int t) { return stats[(size_t)t]; };
    auto task = [&](const LongTask& tk) { tasks.push_back(tk); };
    if (!long_walk(g, stat, task)) return false;
    for (const LongTask& tk : tasks) long_emit(m, g, tk, load, x, emit);
    return true;
}
}  // namespace

extern "C" {

// mode 0 short / 1 paired / 2 long; wide: the 128-bit-key instantiation.  Records sorted by (unit, table, k, hi, lo);
// returns their number (-1 when cap is too small).  *n_bailed / bailed_index: units outside the thread path's limits
// (nothing recorded for them).
long urc_scan(int mode, int wide, const char* buf1, const int32_t* locs1, const char* buf2, const int32_t* locs2, int n_units, int min_mer,
              int max_mer, int slice_len, const unsigned short* thr_low, const unsigned short* thr_high, uint64_t* out_unit, int32_t* out_table,
              int32_t* out_k, uint64_t* out_lo, uint64_t* out_hi, uint64_t* out_count, long cap, long* n_bailed, int32_t* bailed_index) {
    Records recs;
    long bailed = 0;
    for (int r = 0; r < n_units; r++) {
        RecordEmit emit{&recs, (uint64_t)r};
        const bool ok = wide ? route_unit<u128>(mode, buf1, locs1, buf2, locs2, r, min_mer, max_mer, slice_len, thr_low, thr_high, emit)
                             : route_unit<u64>(mode, buf1, locs1, buf2, locs2, r, min_mer, max_mer, slice_len, thr_low, thr_high, emit);
        if (!ok) { bailed_index[bailed++] = r; }
    }
    *n_bailed = bailed;
    if ((long)recs.size() > cap) return -1;
    long i = 0;
    for (auto& kv : recs) {
        out_unit[i] = std::get<0>(kv.first); out_table[i] = std::get<1>(kv.first); out_k[i] = std::get<2>(kv.first);
        out_hi[i] = std::get<3>(kv.first); out_lo[i] = std::get<4>(kv.first); out_count[i] = kv.second;
        i++;
    }
    return i;
}

}  // extern "C"
