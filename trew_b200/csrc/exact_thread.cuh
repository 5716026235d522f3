// Thread-per-read exact routing for short single-end reads: the whole of buffer_task (src/kmer.cpp:80-266) with
// k_mer_check (src/kmer.cpp:2144-2344) and k_mer_target (src/kmer.cpp:1894-2017) as plain scalar code.
//
// Why it exists: the warp-per-survivor kernel (scan_kernels.cu, trew_exact_kernel) spends its time on latency -- one
// survivor per warp, most instructions warp-uniform, stack traffic around its calls, an instruction footprint that
// does not fit the instruction cache.  Here every THREAD owns a survivor, so an SM works on several hundred survivors
// at once instead of 32 and the per-survivor instruction stream is issued for 32 survivors at a time.
//
// Layout: a thread's working set (the window being scanned, masks, the first classes of an evaluation: 47 words with
// 64-bit keys, 59 with 128-bit ones) lives in a per-thread slice of SHARED memory, word i of thread t at
// base[i * stride + t]: consecutive threads hit consecutive banks, array indices may be run-time values (register arrays
// would need compile-time indices, i.e. fully unrolled code -- tried for the whole workspace: 256 KB of SASS and spilled
// planes), and the functions below stay small, out-of-line and loop-based, which keeps the instruction footprint at a
// few KB.  The one exception is scan_window's loop over the periods, the hottest loop: its prefix planes and valid mask
// are small register arrays indexed by unrolled loops (scan_periods), and only a period that passes the bound stores
// its mask to the workspace for the class statistics.  With the staging table that is 27.5 KB per 128-thread block
// (64-bit keys); blocks per SM: scan_kernels.cu, thread_kernel_bps.
//
// The code is scalar (no warp intrinsics), so it also compiles for the host: tests/native/exact_thread_check.cpp runs
// this very file against the oracle without a GPU (stride 1, base = a plain array).
//
// Limits (anything else is handed to the warp kernel through the `false` return, before anything was emitted):
// reads of at most 160 bases and MAX_MER <= 32 (64-bit units); pairs additionally min(n1, n2) >= 4 * MAX_MER.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define ET_HD __host__ __device__ __forceinline__
#define ET_FN __host__ __device__ __noinline__
#else
#define ET_HD inline
#define ET_FN inline
#endif
#if defined(__CUDA_ARCH__)
#define ET_UNROLL _Pragma("unroll")
#define ET_NO_UNROLL _Pragma("unroll 1")
#else
#define ET_UNROLL
#define ET_NO_UNROLL
#endif

namespace trew {
namespace et {

typedef uint32_t u32;
typedef uint64_t u64;
typedef unsigned __int128 u128;   // repeat units above 32 bases (MAX_MER <= 64): the reference's uint128_t path

constexpr int kReadWords = 5;      // read planes: up to 160 bases
constexpr int kMaxRead = 32 * kReadWords;
constexpr int kClsCap = 6;         // distinct rotation classes of an evaluated (window, period) kept in the workspace ...
constexpr int kClsSpill = kMaxRead - kClsCap;   // ... the rest (noisy windows, rare) in thread-local memory
constexpr int kApproxMaxWindows = 48;           // scan_window: composition pre-pass only for periods with at most this many windows

// workspace words of one thread.  The read itself stays in global memory: a window is brought in by the caller's
// load(mate, off, len), which fills W_H / W_L (kReadWords + 2 words each, zero beyond the window) and W_V (kReadWords).
enum {
    W_H = 0, W_L = W_H + kReadWords + 2, W_V = W_L + kReadWords + 2,          // the current window: hi / lo / valid planes
    W_WV = W_V + kReadWords, W_LINK = W_WV + kReadWords,                     // valid k-windows, links between neighbours
    W_CKEY = W_LINK + kReadWords                                             // class keys, least significant word first
};
template <class K>
struct Lay {   // ... then per class: the key (2 or 4 words) and total << 16 | last window
    static constexpr int KW = (int)(sizeof(K) / 4);
    static constexpr int CT = W_CKEY + KW * kClsCap, WORDS = CT + kClsCap;
};
constexpr int kWorkWords = Lay<u64>::WORDS;

struct Mem {
    u32* base; int stride;
    ET_HD u32& operator[](int i) const { return base[i * stride]; }
};

ET_HD int popc(u32 x) {
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}
ET_HD int ffs1(u32 x) {   // index of the lowest set bit, x != 0
#if defined(__CUDA_ARCH__)
    return __ffs(x) - 1;
#else
    return __builtin_ctz(x);
#endif
}
ET_HD u32 fshr(u32 lo, u32 hi, int sh) {   // low word of (hi:lo) >> (sh & 31)
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, sh);
#else
    sh &= 31;
    return sh ? (lo >> sh) | (hi << (32 - sh)) : lo;
#endif
}
ET_HD u32 brev32(u32 x) {
#if defined(__CUDA_ARCH__)
    return __brev(x);
#else
    x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
    x = ((x >> 2) & 0x33333333u) | ((x & 0x33333333u) << 2);
    x = ((x >> 4) & 0x0f0f0f0fu) | ((x & 0x0f0f0f0fu) << 4);
    x = ((x >> 8) & 0x00ff00ffu) | ((x & 0x00ff00ffu) << 8);
    return (x >> 16) | (x << 16);
#endif
}
ET_HD u32 lowmask(int bits) { return bits >= 32 ? 0xffffffffu : (bits <= 0 ? 0u : ((1u << bits) - 1u)); }
ET_HD u32 pxor32(u32 x) { x ^= x << 1; x ^= x << 2; x ^= x << 4; x ^= x << 8; x ^= x << 16; return x; }
ET_HD u64 spread(u32 x) {   // bit m -> bit 2m
    u64 v = x;
    v = (v | (v << 16)) & 0x0000FFFF0000FFFFULL;
    v = (v | (v << 8)) & 0x00FF00FF00FF00FFULL;
    v = (v | (v << 4)) & 0x0F0F0F0F0F0F0F0FULL;
    v = (v | (v << 2)) & 0x3333333333333333ULL;
    v = (v | (v << 1)) & 0x5555555555555555ULL;
    return v;
}

// minimal rotation of a k-mer (get_rot_seq / get_rot_seq_128, src/kmer.cpp:1815-1833)
ET_FN u64 canon64(u64 w, int k) {
    const int sh = 2 * (k - 1);
    if (k <= 16) {
        u32 b = (u32)w, c = (u32)w;
        for (int r = 1; r < k; r++) { c = ((c & 3u) << sh) | (c >> 2); b = c < b ? c : b; }
        return b;
    }
    u64 best = w, cur = w;
    for (int r = 1; r < k; r++) { cur = ((cur & 3ULL) << sh) | (cur >> 2); best = cur < best ? cur : best; }
    return best;
}
ET_FN u128 canon128(u128 w, int k) {
    const int sh = 2 * (k - 1);
    u128 best = w, cur = w;
    for (int r = 1; r < k; r++) { cur = ((cur & 3) << sh) | (cur >> 2); best = cur < best ? cur : best; }
    return best;
}
ET_HD u64 canon(u64 w, int k) { return canon64(w, k); }
ET_HD u128 canon(u128 w, int k) { return k <= 32 ? (u128)canon64((u64)w, k) : canon128(w, k); }
// canonical rotation of the reverse complement (rot_reverse_complement, src/kmer.cpp:72-74)
ET_HD u64 crc(u64 w, int k) {
    const u32 lo = brev32((u32)w), hi = brev32((u32)(w >> 32));
    u64 x = ((u64)lo << 32) | hi;                                                 // all 64 bits reversed
    x = ((x >> 1) & 0x5555555555555555ULL) | ((x & 0x5555555555555555ULL) << 1);   // 2-bit symbols reversed
    return canon64(~x >> (64 - 2 * k), k);
}
ET_HD u128 crc(u128 w, int k) {
    if (k <= 32) return (u128)crc((u64)w, k);
    u128 r = 0;
    for (int i = 0; i < k; i++) { r = (r << 2) | (3 - (w & 3)); w >>= 2; }
    return canon128(r, k);
}
ET_HD bool homo(u64 w, int k) {   // get_repeat_check: at most one distinct base
    return k <= 1 || ((w ^ (w >> 2)) & ((1ULL << (2 * (k - 1))) - 1ULL)) == 0;
}
ET_HD bool homo(u128 w, int k) {
    return k <= 1 || ((w ^ (w >> 2)) & ((((u128)1) << (2 * (k - 1))) - 1)) == 0;
}

// the spill part of a class list (classes beyond the first kClsCap of an evaluation)
template <class K>
struct ClsSpill {
    K key[kClsSpill];
    unsigned short tot[kClsSpill], last[kClsSpill];
};

template <class K>
ET_HD K cls_key(Mem m, int q) {
    K v = 0;
    for (int i = Lay<K>::KW - 1; i >= 0; i--) v = (v << 16 << 16) | (K)m[W_CKEY + Lay<K>::KW * q + i];
    return v;
}
template <class K>
ET_HD void cls_put(Mem m, int q, K key) {
    for (int i = 0; i < Lay<K>::KW; i++) { m[W_CKEY + Lay<K>::KW * q + i] = (u32)key; key = key >> 16 >> 16; }
}

// word j of (plane >> k), 0 < k <= 64; the planes have two zero words behind the window
ET_HD u32 shr_plane(Mem m, int base, int j, int k) {
    if (k < 32) return fshr(m[base + j], m[base + j + 1], k);
    if (k == 32) return m[base + j + 1];
    if (k < 64) return fshr(m[base + j + 1], m[base + j + 2], k - 32);
    return m[base + j + 2];
}

// the k-mer starting at bit b of word j of the current window, first base most significant (the reference's shift-in
// order, src/kmer.cpp:2186-2189); hk / lk receive its hi and lo plane bits (for the composition key)
ET_HD u64 raw_kmer(Mem m, int j, int b, int k, u64& hk, u64& lk, u64) {
    const u32 km = lowmask(k);
    const u32 h = fshr(m[W_H + j], m[W_H + j + 1], b) & km, l = fshr(m[W_L + j], m[W_L + j + 1], b) & km;
    hk = h; lk = l;
    return (spread(brev32(h) >> (32 - k)) << 1) | spread(brev32(l) >> (32 - k));
}
ET_HD u128 raw_kmer(Mem m, int j, int b, int k, u64& hk, u64& lk, u128) {
    if (k <= 32) return (u128)raw_kmer(m, j, b, k, hk, lk, (u64)0);
    const u64 km = k >= 64 ? ~0ULL : ((1ULL << k) - 1ULL);
    hk = ((u64)fshr(m[W_H + j], m[W_H + j + 1], b) | ((u64)fshr(m[W_H + j + 1], m[W_H + j + 2], b) << 32)) & km;
    lk = ((u64)fshr(m[W_L + j], m[W_L + j + 1], b) | ((u64)fshr(m[W_L + j + 1], m[W_L + j + 2], b) << 32)) & km;
    // reverse the k bits of each plane, then interleave: bit (k - 1 - i) of hr / lr is base i
    const u64 hr = (((u64)brev32((u32)hk) << 32) | brev32((u32)(hk >> 32))) >> (64 - k);
    const u64 lr = (((u64)brev32((u32)lk) << 32) | brev32((u32)(lk >> 32))) >> (64 - k);
    const u64 lo = (spread((u32)hr) << 1) | spread((u32)lr), hi = (spread((u32)(hr >> 32)) << 1) | spread((u32)(lr >> 32));
    return ((u128)hi << 64) | lo;
}

// Match-bit runs of the current window for one period (Lemma L1: windows i and i+1 are in the same rotation class iff
// both are valid and base[i] == base[i+k], so classes are unions of maximal runs).  W_WV = valid k-windows (input);
// fills W_LINK and returns the number of runs.
ET_HD u32 run_starts(Mem m, int j) {   // valid windows of word j without a link from their predecessor
    return m[W_WV + j] & ~((m[W_LINK + j] << 1) | (j ? m[W_LINK + j - 1] >> 31 : 0u));
}
ET_FN int prepare_runs(Mem m, int nw, int k) {
    for (int j = 0; j < nw; j++) {
        const u32 hs = shr_plane(m, W_H, j, k), ls = shr_plane(m, W_L, j, k);
        const u32 eq = ~((hs ^ m[W_H + j]) | (ls ^ m[W_L + j]));
        const u32 wvj = m[W_WV + j];
        const u32 nxt = (wvj >> 1) | (j + 1 < nw ? m[W_WV + j + 1] << 31 : 0u);
        m[W_LINK + j] = eq & wvj & nxt;
    }
    int runs = 0;
    for (int j = 0; j < nw; j++) runs += popc(run_starts(m, j));
    return runs;
}

// Class statistics from the runs: the inner loops of k_mer_check (src/kmer.cpp:2183-2216), one minimal rotation per
// run.  Returns the number of classes: the first kClsCap in the workspace, the others in `x`.
// approx: classes by base composition (#C|A, #G|A, #A of the run's first window) instead of by minimal rotation.
// Rotation keeps the composition, so these classes are unions of the true ones and their largest total bounds the true
// largest class from above -- at a fraction of the cost (no k-step rotation loop); used to turn away noisy windows.
// T, need_min: the windows of the evaluation and the smallest largest-class total anybody is interested in; the pass
// stops (returns -1) as soon as the largest class so far plus every window not yet seen cannot reach it -- a noisy window
// (one run per k-window, ever more classes to search) is turned away about half way through.  need_min = 0: full statistics.
// Exact mode: in a tandem repeat whose period does not divide k the runs recur every period with the same raw k-mer
// (TTAGGG at k = 5: ~35 runs per 75-base half, three distinct raw k-mers), so the first kMemo distinct raw k-mers of the
// evaluation are remembered with the class they went to; a run that starts with one of them skips the rotation and the
// search.  A hit only ever finds an existing class, so classes are created in the same order as without the memo.
constexpr int kMemo = 4;
#if defined(ET_MEMO_STATS) && !defined(__CUDA_ARCH__)
inline long memo_runs = 0, memo_hits = 0;   // host builds only (tools/memo_hits.py): exact-mode runs, memo hits
#define ET_MEMO_COUNT(hit) (memo_runs++, memo_hits += (hit) >= 0)
#else
#define ET_MEMO_COUNT(hit) ((void)0)
#endif
template <class K>
ET_FN int classify_runs(Mem m, int runs, int k, ClsSpill<K>& x, bool approx, int T = 0, int need_min = 0) {
    int n = 0, ord = 0, j = 0, best = 0;
    const int slack = T - need_min;   // windows seen outside the largest class may not exceed this
    K mraw[kMemo];
    u32 mcls = 0;   // class of entry e in byte e
    int nm = 0;
    u32 wvj = m[W_WV], rr = run_starts(m, 0);
    // one loop over the runs, not one per plane word: the lanes of a warp then meet in the body for their r-th run
    // wherever it lies (a per-word loop serialises lanes whose runs start in different words)
    for (int r = 0; r < runs; r++) {
        while (!rr) { ord += popc(wvj); j++; rr = run_starts(m, j); wvj = m[W_WV + j]; }
        {
            const int b = ffs1(rr);
            rr &= rr - 1;
            const u32 c0 = (u32)(ord + popc(wvj & ((1u << b) - 1u)));
            // the run ends at the first window without a link to its successor (the last valid window has none)
            int jj = j;
            u32 z = ~m[W_LINK + j] & (0xffffffffu << b);
            while (!z) { jj++; z = ~m[W_LINK + jj]; }
            const u32 cnt = (u32)(32 * (jj - j) + ffs1(z) - b + 1);
            u64 hk, lk;
            const K raw = raw_kmer(m, j, b, k, hk, lk, (K)0);
            const u32 last = c0 + cnt - 1u;
            int hit = -1;
            if (!approx) {
ET_UNROLL
                for (int e = 0; e < kMemo; e++) hit = e < nm && mraw[e] == raw ? (int)((mcls >> (8 * e)) & 0xffu) : hit;
            }
            if (!approx) ET_MEMO_COUNT(hit);
            u32 tot = cnt;
            if (hit >= kClsCap) {
                const int s = hit - kClsCap;
                tot = x.tot[s] + cnt; x.tot[s] = (unsigned short)tot; x.last[s] = (unsigned short)last;
            } else if (hit >= 0) {
                const u32 ct = (m[Lay<K>::CT + hit] & 0xffff0000u) + (cnt << 16);
                m[Lay<K>::CT + hit] = ct | last;
                tot = ct >> 16;
            } else {
                K key;
                if (approx) key = (K)((u32)(popc((u32)hk) + popc((u32)(hk >> 32))) | ((u32)(popc((u32)lk) + popc((u32)(lk >> 32))) << 8) |
                                      ((u32)(popc((u32)(hk & lk)) + popc((u32)((hk & lk) >> 32))) << 16));
                else key = canon(raw, k);
                int q = 0;
                const int nq = n < kClsCap ? n : kClsCap;
                while (q < nq && cls_key<K>(m, q) != key) q++;
                if (q < nq) {
                    const u32 ct = (m[Lay<K>::CT + q] & 0xffff0000u) + (cnt << 16);
                    m[Lay<K>::CT + q] = ct | last;
                    tot = ct >> 16;
                } else if (n < kClsCap) {
                    cls_put<K>(m, n, key); m[Lay<K>::CT + n] = (cnt << 16) | last;
                    n++;
                } else {
                    int s = 0;
                    while (s < n - kClsCap && x.key[s] != key) s++;
                    if (s < n - kClsCap) { tot = x.tot[s] + cnt; x.tot[s] = (unsigned short)tot; x.last[s] = (unsigned short)last; }
                    else { x.key[s] = key; x.tot[s] = (unsigned short)cnt; x.last[s] = (unsigned short)last; n++; }
                    q = kClsCap + s;
                }
                if (!approx && nm < kMemo) {
ET_UNROLL
                    for (int e = 0; e < kMemo; e++) if (e == nm) mraw[e] = raw;
                    mcls |= (u32)q << (8 * nm);
                    nm++;
                }
            }
            if (need_min > 0) {
                // seen = last + 1 windows so far, `best` of them in the largest class: best + (T - seen) >= need_min must stay possible
                best = (int)tot > best ? (int)tot : best;
                if ((int)last + 1 - best > slack) return -1;
            }
        }
    }
    return n;
}

// M and K_MER_DATA_MAX_SEQ of the last evaluation: the class whose running count first reaches the final maximum (strict
// '<' at src/kmer.cpp:2202) = largest total, ties broken by the EARLIEST last window
template <class K>
ET_FN int cls_max(Mem m, int n, const ClsSpill<K>& x, K& S) {
    u32 best = 0;
    S = 0;
    for (int q = 0; q < n && q < kClsCap; q++) {
        const u32 ct = m[Lay<K>::CT + q];
        const u32 score = ((ct >> 16) << 10) | (1023u - (ct & 0xffffu));
        if (score > best) { best = score; S = cls_key<K>(m, q); }
    }
    for (int q = 0; q < n - kClsCap; q++) {
        const u32 score = ((u32)x.tot[q] << 10) | (1023u - x.last[q]);
        if (score > best) { best = score; S = x.key[q]; }
    }
    return (int)(best >> 10);
}

// max(baseline, last accepted frequency) without floating point: see scan_kernels.cu, need_pass
ET_HD bool need_pass(const unsigned short* thr, u32 need, int M, int T) {
    const u32 mm = need & 0xffffu, t = need >> 16;
    return M >= (int)thr[T] && (t == 0u || (u32)M * t >= mm * (u32)T);
}

// the smallest M need_pass lets through (M only grows the left sides)
ET_HD int min_accept(const unsigned short* thr, u32 need, int T) {
    const u32 mm = need & 0xffffu, t = need >> 16;
    const int a = (int)thr[T], b = t ? (int)((mm * (u32)T + t - 1u) / t) : 0;
    return a > b ? a : b;
}

ET_HD void shrink_valid(Mem m, int nw) {   // valid k-windows -> valid (k+1)-windows
    for (int j = 0; j < nw; j++) m[W_WV + j] &= (m[W_WV + j] >> 1) | (j + 1 < nw ? m[W_WV + j + 1] << 31 : 0u);
}

// scan_periods' register copies of the prefix planes (NW + 2 words: shifts up to 64) and of the valid k-windows (NW words,
// zero beyond the window)
template <int NW>
ET_HD void shrink_valid(u32 (&wv)[NW]) {
ET_UNROLL
    for (int j = 0; j < NW; j++) wv[j] &= (wv[j] >> 1) | (j + 1 < NW ? wv[j + 1] << 31 : 0u);
}
// the (hi parity, lo parity) signature counts of period k = 32 * S + (k & 31): windows whose hi / lo / both parities differ
template <int S, int NW>
ET_HD void sig_counts(const u32 (&ph)[NW + 2], const u32 (&pl)[NW + 2], const u32 (&wv)[NW], int k, int& cH, int& cL, int& c11) {
ET_UNROLL
    for (int j = 0; j < NW; j++) {
        const u32 dh = (fshr(ph[S + j], S + j + 1 < NW + 2 ? ph[S + j + 1] : 0u, k) ^ ph[j]) & wv[j];
        const u32 dl = (fshr(pl[S + j], S + j + 1 < NW + 2 ? pl[S + j + 1] : 0u, k) ^ pl[j]) & wv[j];
        cH += popc(dh); cL += popc(dl); c11 += popc(dh & dl);
    }
}

// bit k - 1 of a set of periods k <= 4 * sizeof(K): 32 bits hold every period with 64-bit units, 64 with 128-bit ones
template <class K> struct PeriodSet { typedef u64 T; };
template <> struct PeriodSet<u64> { typedef u32 T; };

// k_mer_check without emission (src/kmer.cpp:2144-2258) on the current window of at most 32 * NW bases: returns
// target_k_high | target_k_low << 8; S[0] / S[1]: the K_MER_DATA_MAX_SEQ of the two (the paired routing compares them
// between segments)
template <class K, int NW>
ET_HD u32 scan_periods(Mem m, int len, int kmin, int kmax, const unsigned short* thr_low, const unsigned short* thr_high, ClsSpill<K>& x,
                       K (&S)[2]) {
    const int nw = (len + 31) >> 5;
    // exclusive prefix-XOR planes: entry i = parity of the hi (lo) bits of bases [0, i).  Beyond the window the planes
    // hold the total parity; only windows that are not valid read those entries.
    u32 ph[NW + 2], pl[NW + 2], wv[NW];
    {
        u32 ch = 0, cl = 0, tph = 0, tpl = 0;
ET_UNROLL
        for (int j = 0; j <= NW; j++) {
            const u32 ih = pxor32(m[W_H + j]) ^ ch, il = pxor32(m[W_L + j]) ^ cl;
            ph[j] = (ih << 1) | tph; pl[j] = (il << 1) | tpl;
            tph = ih >> 31; tpl = il >> 31;
            ch = 0u - tph; cl = 0u - tpl;
        }
        ph[NW + 1] = 0u; pl[NW + 1] = 0u;
    }
ET_UNROLL
    for (int j = 0; j < NW; j++) wv[j] = j < nw ? m[W_V + j] : 0u;
    for (int t = 1; t < kmin; t++) shrink_valid<NW>(wv);
    typedef typename PeriodSet<K>::T Set;
    Set blockedL = 0, blockedH = 0;   // periods with an accepted divisor (src/kmer.cpp:2225-2230); bit k - 1, k <= kmax
    u32 needL = 0, needH = 0;         // last accepted ratio, m | t << 16
    u32 res = 0;
ET_NO_UNROLL
    for (int k = kmin; k <= kmax; k++, shrink_valid<NW>(wv)) {
        const bool blkL = (bool)((blockedL >> (k - 1)) & 1u), blkH = (bool)((blockedH >> (k - 1)) & 1u);
        // upper bound on the largest class: largest bucket of the (hi parity, lo parity) signature (Lemma L2)
        int T = 0, cH = 0, cL = 0, c11 = 0;
ET_UNROLL
        for (int j = 0; j < NW; j++) T += popc(wv[j]);
        if (T == 0) break;   // the valid-window mask only shrinks with k
        if (blkL && blkH) continue;
        if (k < 32) sig_counts<0, NW>(ph, pl, wv, k, cH, cL, c11);
        else if constexpr (sizeof(K) == 8) sig_counts<1, NW>(ph, pl, wv, k, cH, cL, c11);   // k == 32, the largest with 64-bit units
        else if (k < 64) sig_counts<1, NW>(ph, pl, wv, k, cH, cL, c11);
        else sig_counts<2, NW>(ph, pl, wv, k, cH, cL, c11);
        const int c10 = cH - c11, c01 = cL - c11, c00 = T - cH - cL + c11;
        int U = c00 > c01 ? c00 : c01;
        U = U > c10 ? U : c10;
        U = U > c11 ? U : c11;
        if (!((!blkL && need_pass(thr_low, needL, U, T)) || (!blkH && need_pass(thr_high, needH, U, T)))) continue;
        K Sk;
ET_UNROLL
        for (int j = 0; j < NW; j++) m[W_WV + j] = wv[j];
        const int runs = prepare_runs(m, nw, k);
        int need_min = 1 << 20;
        if (!blkL) need_min = min_accept(thr_low, needL, T);
        if (!blkH) { const int a = min_accept(thr_high, needH, T); need_min = a < need_min ? a : need_min; }
        // several runs over few windows (what an N leaves of a window): first the cheap bound from the runs' base
        // compositions.  With many windows it is not worth its price: TTAGGG at k = 5 has ~35 runs per half, half of them in
        // one class AND one composition, so the bound never rejects there (measured: 5 % of the kernel).
        if (runs > 3 && T <= kApproxMaxWindows) {
            const int na = classify_runs(m, runs, k, x, true, T, need_min);
            if (na < 0) continue;
            const int Mu = cls_max(m, na, x, Sk);
            if (!((!blkL && need_pass(thr_low, needL, Mu, T)) || (!blkH && need_pass(thr_high, needH, Mu, T)))) continue;
        }
        const int n = classify_runs(m, runs, k, x, false, T, need_min);
        if (n < 0) continue;
        const int M = cls_max(m, n, x, Sk);
        if (homo(Sk, k)) continue;
        const bool accL = !blkL && need_pass(thr_low, needL, M, T), accH = !blkH && need_pass(thr_high, needH, M, T);
        if (accL || accH) {
            Set mm = 0;
            for (int j = k; j <= kmax; j += k) mm |= ((Set)1) << (j - 1);
            const u32 need = (u32)M | ((u32)T << 16);
            if (accL) { res = (res & 0xffu) | ((u32)k << 8); needL = need; blockedL |= mm; S[1] = Sk; }
            if (accH) { res = (res & 0xff00u) | (u32)k; needH = need; blockedH |= mm; S[0] = Sk; }
        }
    }
    return res;
}
// windows of up to 96 bases (every half and pair segment the thread path takes) in three words, longer ones (the
// whole-read scan) in kReadWords
template <class K>
ET_FN u32 scan_window(Mem m, int len, int kmin, int kmax, const unsigned short* thr_low, const unsigned short* thr_high, ClsSpill<K>& x,
                      K (&S)[2]) {
    S[0] = S[1] = 0;
    if (kmax > len) kmax = len;
    if (kmax < kmin) return 0u;
    if (len <= 96) return scan_periods<K, 3>(m, len, kmin, kmax, thr_low, thr_high, x, S);
    return scan_periods<K, kReadWords>(m, len, kmin, kmax, thr_low, thr_high, x, S);
}

enum { T_F = 0, T_B = 2, T_O = 4 };

template <class K, class Emit>
ET_HD void emit_window_classes(Mem m, int len, int k, int table, bool folded, ClsSpill<K>& x, Emit& emit);

// buffer_task for one read (src/kmer.cpp:111-171).  load(0, off, len) brings bases [off, off + len) of the read in.
// pm: probes (unit_probes order: left half, right half, whole read -- or the whole read alone when n < 4 * MIN_MER)
// the filter kernels could not rule out; the scan of any other window finds nothing.  emit(table, k, key, count) receives the emissions.  Returns false when the read is outside this
// path's limits: then nothing was emitted and the warp kernel has to take it.
template <class K, class Load, class Emit>
ET_HD bool route_short_thread(Mem m, int n, u32 pm, int min_mer, int max_mer, const unsigned short* thr_low,
                              const unsigned short* thr_high, Load& load, Emit& emit) {
    if (n < 2 * min_mer) return true;                                   // src/kmer.cpp:113
    if (max_mer > (int)(4 * sizeof(K)) || n > kMaxRead) return false;    // outside the limits (K = u64: 32, u128: 64)
    const int kmax = n / 4 < max_mer ? n / 4 : max_mer;
    const int llen = n / 2, rlen = (n + 1) / 2, roff = n - rlen;
    ClsSpill<K> x;
    u32 L = 0, R = 0;   // target_k_high | target_k_low << 8 of the two halves
    K S[2];
    const bool halves = n >= 4 * min_mer;
    // both halves are "always evaluated"; every lane starts with ITS first vouched-for half (half-repeats and chance
    // survivors have one), so the lanes of a warp scan together instead of taking turns by half
    for (u32 todo = halves ? pm & 3u : 0u; todo != 0u; todo &= todo - 1u) {
        const bool right = (todo & 1u) == 0u;
        const int len = right ? rlen : llen;
        load(0, right ? roff : 0, len);
        const u32 r = scan_window(m, len, min_mer, kmax, thr_low, thr_high, x, S);
        if (right) R = r; else L = r;
    }
    if (4 * max_mer > n) {
        // short reads: periods above n / 4 are looked for in the whole read, for the selections that found nothing in
        // either half; their classes go into 'both' UN-folded (src/kmer.cpp:165-171).  The probe of this scan is bit 2
        // when the halves were probed (bits 0, 1), bit 0 when the read is too short for halves.
        const bool hc0 = ((L | R) & 0xffu) == 0u, hc1 = ((L | R) >> 8) == 0u;
        const u32 wbit = halves ? 4u : 1u;
        if ((hc0 || hc1) && (pm & wbit)) {
            const int lo = n / 4 + 1 > min_mer ? n / 4 + 1 : min_mer, hi = n / 2 < max_mer ? n / 2 : max_mer;
            load(0, 0, n);
            const u32 W = scan_window(m, n, lo, hi, thr_low, thr_high, x, S);
            for (int c = 0; c < 2; c++) {
                const int k = (int)((W >> (8 * c)) & 0xffu);
                if ((c == 0 ? hc0 : hc1) && k) emit_window_classes(m, n, k, T_O + c, false, x, emit);
            }
        }
    }
    if ((L | R) == 0u) return true;
    // right-half emissions survive only for classes where the left half found nothing (src/kmer.cpp:123-159)
    int cur_win = -1, cur_k = 0, ncls = 0, T = 0;   // the evaluation in the workspace
    for (int c = 0; c < 2; c++) {
        const int Lc = (int)((L >> (8 * c)) & 0xffu), Rc = (int)((R >> (8 * c)) & 0xffu);
        int win, k, table;
        if (Lc > 0 && Lc == Rc) { win = 2; k = Lc; table = T_O + c; }          // k_mer_target on the whole read -> both
        else if (Lc > 0) { win = 0; k = Lc; table = T_F + c; }
        else if (Rc > 0) { win = 1; k = Rc; table = T_B + c; }
        else continue;
        if (win != cur_win || k != cur_k) {   // the two selections usually ask for the same evaluation
            const int off = win == 1 ? roff : 0, len = win == 2 ? n : (win == 0 ? llen : rlen), nw = (len + 31) >> 5;
            load(0, off, len);
            for (int j = 0; j < nw; j++) m[W_WV + j] = m[W_V + j];
            for (int t = 1; t < k; t++) shrink_valid(m, nw);
            T = 0;
            for (int j = 0; j < nw; j++) T += popc(m[W_WV + j]);
            ncls = 0;
            if (T) ncls = classify_runs(m, prepare_runs(m, nw, k), k, x, false);
            cur_win = win; cur_k = k;
        }
        if (T == 0) continue;
        const bool target = win == 2;
        if (target) {   // k_mer_target (src/kmer.cpp:1894-2017): largest class no homopolymer and at the baseline, classes RC-folded
            K S;
            const int M = cls_max(m, ncls, x, S);
            if (homo(S, k) || M < (int)(c == 0 ? thr_high : thr_low)[T]) continue;
        }
        for (int q = 0; q < ncls; q++) {
            K key = q < kClsCap ? cls_key<K>(m, q) : x.key[q - kClsCap];
            const u64 cnt = q < kClsCap ? (u64)(m[Lay<K>::CT + q] >> 16) : (u64)x.tot[q - kClsCap];
            if (target) { const K t = crc(key, k); key = t < key ? t : key; }
            emit(table, k, key, cnt);
        }
    }
    return true;
}

// every class of (current window, k) into `table`, RC-folded on request: the emission half of k_mer_check
// (src/kmer.cpp:2264-2328)
template <class K, class Emit>
ET_HD void emit_window_classes(Mem m, int len, int k, int table, bool folded, ClsSpill<K>& x, Emit& emit) {
    const int nw = (len + 31) >> 5;
    for (int j = 0; j < nw; j++) m[W_WV + j] = m[W_V + j];
    for (int t = 1; t < k; t++) shrink_valid(m, nw);
    int T = 0;
    for (int j = 0; j < nw; j++) T += popc(m[W_WV + j]);
    if (T == 0) return;
    const int ncls = classify_runs(m, prepare_runs(m, nw, k), k, x, false);
    for (int q = 0; q < ncls; q++) {
        K key = q < kClsCap ? cls_key<K>(m, q) : x.key[q - kClsCap];
        const u64 cnt = q < kClsCap ? (u64)(m[Lay<K>::CT + q] >> 16) : (u64)x.tot[q - kClsCap];
        if (folded) { const K t = crc(key, k); key = t < key ? t : key; }
        emit(table, k, key, cnt);
    }
}

// buffer_task_pair for one pair (src/kmer.cpp:268-745; the 128-bit path's semantics where the two differ, like the warp
// kernel's route_pair, which this mirrors statement by statement).  load(mate, off, len) brings bases [off, off + len) of
// that mate in.  Limits: both mates <= 160 bases, MAX_MER <= 32, min(n1, n2) >= 4 * MAX_MER (so the large-k block of
// src/kmer.cpp:467-505 never runs); false = outside them, nothing emitted.
template <class K, class Load, class Emit>
ET_HD bool route_pair_thread(Mem m, int n1, int n2, int min_mer, int max_mer, const unsigned short* thr_low,
                             const unsigned short* thr_high, Load& load, Emit& emit) {
    const int n = n1 < n2 ? n1 : n2;
    if (n < 2 * min_mer) return true;
    if (max_mer > (int)(4 * sizeof(K)) || n1 > kMaxRead || n2 > kMaxRead || 4 * max_mer > n) return false;
    const int kmax = n / 4 < max_mer ? n / 4 : max_mer;
    // segments in fragment order: R1 left, R1 right, R2 right, R2 left (src/kmer.cpp:338-340)
    const int soff[5] = {0, 0, n1 - (n1 + 1) / 2, n2 - (n2 + 1) / 2, 0};
    const int slen[5] = {0, n1 / 2, (n1 + 1) / 2, (n2 + 1) / 2, n2 / 2};
    ClsSpill<K> x;
    u32 res[5] = {0, 0, 0, 0, 0};
    K S[5][2];
    bool have[5] = {false, false, false, false, false};
    auto window = [&](int t) { load(t <= 2 ? 0 : 1, soff[t], slen[t]); };
    auto scan = [&](int t) {
        if (have[t]) return;
        window(t);
        res[t] = scan_window(m, slen[t], min_mer, kmax, thr_low, thr_high, x, S[t]);
        have[t] = true;
    };
    // pending emissions per class: segment + temp map id (0 = left, 1 = right)
    int pseg[2][8], ptmp[2][8], np[2] = {0, 0};
    int si[2] = {1, 1}, km[2] = {0, 0};
    bool ended[2] = {false, false};
    K ks[2] = {0, 0};
    for (int ti = 1; ti <= 4 && !(ended[0] && ended[1]); ti++) {   // forward walk
        scan(ti);
        for (int c = 0; c < 2; c++) {
            const int k = (int)((res[ti] >> (8 * c)) & 0xffu);
            if (!ended[c] && k) { pseg[c][np[c]] = ti; ptmp[c][np[c]] = ti <= 2 ? 0 : 1; np[c]++; }   // emission before the test
            bool ok = !ended[c] && k > 0;
            if (ok && ti != 1) {
                const K ds = ti > 2 ? crc(S[ti][c], k) : S[ti][c];   // get_dir_seq, src/kmer.cpp:307-313
                ok = km[c] == k && ks[c] == ds;
            }
            if (ok) { si[c]++; km[c] = k; if (ti == 1) ks[c] = S[ti][c]; }
            else ended[c] = true;
        }
    }
    for (int c = 0; c < 2; c++) {
        if (si[c] == 5) {   // every segment agreed: everything into 'both', RC-folded (src/kmer.cpp:378-399)
            for (int e = 0; e < np[c]; e++) {
                const int sg = pseg[c][e];
                window(sg);
                emit_window_classes(m, slen[sg], (int)((res[sg] >> (8 * c)) & 0xffu), T_O + c, true, x, emit);
            }
        }
    }
    if (si[0] <= 4 || si[1] <= 4) {   // backward walk (src/kmer.cpp:401-436), temps swapped
        int sj[2] = {4, 4};
        km[0] = km[1] = 0; ended[0] = ended[1] = false;
        for (int tj = 4; tj >= 1 && !(ended[0] && ended[1]); tj--) {
            scan(tj);
            for (int c = 0; c < 2; c++) {
                const int k = (int)((res[tj] >> (8 * c)) & 0xffu);
                if (!ended[c] && k) { pseg[c][np[c]] = tj; ptmp[c][np[c]] = tj <= 2 ? 1 : 0; np[c]++; }
                bool ok = sj[c] >= si[c] && !ended[c] && k > 0;
                if (ok && tj != 4) {
                    const K ds = tj <= 2 ? crc(S[tj][c], k) : S[tj][c];
                    ok = km[c] == k && ks[c] == ds;
                }
                if (ok) { sj[c]--; km[c] = k; if (tj == 4) ks[c] = S[tj][c]; }
                else ended[c] = true;
            }
        }
    }
    for (int c = 0; c < 2; c++) {
        if (si[c] <= 4) {   // forward += left temp, backward += right temp (src/kmer.cpp:438-455)
            for (int e = 0; e < np[c]; e++) {
                const int sg = pseg[c][e];
                window(sg);
                emit_window_classes(m, slen[sg], (int)((res[sg] >> (8 * c)) & 0xffu), (ptmp[c][e] == 0 ? T_F : T_B) + c, false, x, emit);
            }
        }
    }
    return true;
}

// ---- long reads (buffer_task_long, src/kmer.cpp:747-985) in three data-parallel steps ---------------------------------
//
// The reference walks a read's slices inwards from both ends and stops a walk at the first slice that breaks it, so a
// telomere-rich read is a long serial chain (one warp, up to ~100 slice scans, in the warp kernel).  The statistics of a
// slice do not depend on the walk, only which of them are LOOKED at does.  So for a surviving read:
//   1. long_slice_stats   target_k_high / target_k_low of EVERY slice but the middle one (threads: one per slice);
//   2. long_walk          the two walks over those numbers (cheap, one thread per read) -> a list of emissions;
//   3. long_emit          one emission = the classes of one (slice, k) into one table (threads: one per emission).
// The middle slice carries the read's remainder and can be up to 2 * SLICE_LENGTH - 1 bases: a walk that reaches it makes
// the read a case for the warp kernel (long_walk returns false before anything is emitted), as does SLICE_LENGTH > 160.

struct LongGeom {   // src/kmer.cpp:790-798
    int n, SL, snum, mid, bonus;
    ET_HD LongGeom(int n_, int SL_) : n(n_), SL(SL_), snum(n_ / SL_), mid((n_ / SL_ + 1) / 2), bonus(n_ % SL_) {}
    ET_HD int start(int t) const { return (t - 1) * SL + (t > mid ? bonus : 0); }   // slices are 1-based
    ET_HD int len(int t) const { return SL + (t == mid ? bonus : 0); }
};

// step 1 for one slice: load(0, off, len) brings bases [off, off + len) of the read in
template <class Load>
ET_HD u32 long_slice_stats(Mem m, const LongGeom& g, int t, int min_mer, int max_mer, const unsigned short* thr_low,
                           const unsigned short* thr_high, Load& load, ClsSpill<u64>& x) {
    const int len = g.len(t);
    load(0, g.start(t), len);
    u64 S[2];
    return scan_window(m, len, min_mer, max_mer, thr_low, thr_high, x, S);
}

// one emission of a long read: slice t, period k, destination table, RC-folded or not
struct LongTask { unsigned short slice; unsigned char k, table_folded; };   // table | folded << 3

// step 2.  stat(t) = target_k_high | target_k_low << 8 of slice t (never asked for the middle slice: the walk bails out
// first when the slice is longer than the thread path takes); task(LongTask) receives the emissions in the reference's
// order.  Returns false when the read has to go to the warp kernel; then no task was produced.
// The walks are run twice: first only to see whether the middle slice is needed, then to produce the tasks.
template <class Stat, class Task>
ET_HD bool long_walk(const LongGeom& g, Stat& stat, Task& task) {
    const int snum = g.snum;
    const bool mid_ok = g.len(g.mid) <= kMaxRead;
    for (int pass = mid_ok ? 1 : 0; pass < 2; pass++) {
        int si[2] = {1, 1}, km[2] = {0, 0};
        bool ended[2] = {false, false};
        int nf = 0;
        for (int ti = 1; ti <= snum && !(ended[0] && ended[1]); ti++) {   // forward walk
            if (pass == 0 && ti == g.mid) return false;
            const u32 r = stat(ti);
            for (int c = 0; c < 2; c++) {
                const int k = (int)((r >> (8 * c)) & 0xffu);
                if (!ended[c] && k > 0 && (ti == 1 || km[c] == k)) { si[c]++; km[c] = k; }
                else ended[c] = true;
            }
            nf = ti;
        }
        if (pass == 1) {
            // replay: emit into 'both' (folded) when every slice survived, else into 'forward' (src/kmer.cpp:819-830, 858-867)
            bool en[2] = {false, false};
            int kk[2] = {0, 0};
            const bool full[2] = {si[0] == snum + 1, si[1] == snum + 1};
            for (int ti = 1; ti <= nf; ti++) {
                const u32 r = stat(ti);
                for (int c = 0; c < 2; c++) {
                    const int k = (int)((r >> (8 * c)) & 0xffu);
                    if (!en[c] && k) task(LongTask{(unsigned short)ti, (unsigned char)k, (unsigned char)(((full[c] ? T_O : T_F) + c) | (full[c] ? 8 : 0))});
                    if (!en[c] && k > 0 && (ti == 1 || kk[c] == k)) kk[c] = k;
                    else en[c] = true;
                }
            }
        }
        if (si[0] <= snum || si[1] <= snum) {   // backward walk: straight into 'backward' (src/kmer.cpp:836-856)
            int sj[2] = {snum, snum};
            km[0] = km[1] = 0; ended[0] = ended[1] = false;
            for (int tj = snum; tj >= 1 && !(ended[0] && ended[1]); tj--) {
                if (pass == 0 && tj == g.mid) return false;
                const u32 r = stat(tj);
                for (int c = 0; c < 2; c++) {
                    const int k = (int)((r >> (8 * c)) & 0xffu);
                    if (pass == 1 && !ended[c] && k) task(LongTask{(unsigned short)tj, (unsigned char)k, (unsigned char)(T_B + c)});
                    if (sj[c] >= si[c] && !ended[c] && k > 0 && (tj == snum || km[c] == k)) { sj[c]--; km[c] = k; }
                    else ended[c] = true;
                }
            }
        }
    }
    return true;
}

// step 3 for one emission
template <class Load, class Emit>
ET_HD void long_emit(Mem m, const LongGeom& g, const LongTask& tk, Load& load, ClsSpill<u64>& x, Emit& emit) {
    const int len = g.len(tk.slice);
    load(0, g.start(tk.slice), len);
    emit_window_classes(m, len, tk.k, tk.table_folded & 7, (tk.table_folded & 8) != 0, x, emit);
}

}  // namespace et
}  // namespace trew
