// Hand-written CUDA (sm_100a) for TREW's per-read tandem-repeat scan-and-count.
// See scan_kernels.cuh for the two-kernel structure and DESIGN.md for the derivation.
//
// Reference semantics restated here (paths into /root/reference):
//   codes / canonical rotation / reverse complement   src/kmer.cpp:7-78, 1815-1867
//   k_mer_check(_128)  (SCAN)                          src/kmer.cpp:2144-2547
//   k_mer_target(_128) (TARGET)                        src/kmer.cpp:1894-2142
//   buffer_task / _pair / _long (routing)              src/kmer.cpp:80-985
//
// Key facts used (proved in DESIGN.md):
//   L1  two adjacent valid k-windows i, i+1 are in the same rotation class iff base[i] == base[i+k];
//       so classes are unions of maximal match-bit runs and one canonicalisation per run suffices.
//   L2  any rotation-invariant signature partitions windows more coarsely than rotation classes, so the
//       largest signature bucket bounds the largest class from above.  The signature used is the parity
//       of the hi-bit count, lo-bit count (and, second level, A count) of the window, computed for all
//       window positions at once from prefix-XOR bit-planes: sig_k = (P >> k) ^ P.
#include "scan_kernels.cuh"
#include "exact_thread.cuh"

#include <cstdio>

namespace trew {

typedef unsigned int u32;
typedef unsigned long long u64;
typedef unsigned __int128 u128;

// ------------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------------

__device__ __forceinline__ u32 lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ u32 low_mask(int bits) {  // bits in [0, 32]
    return bits >= 32 ? 0xffffffffu : ((1u << bits) - 1u);
}

__device__ __forceinline__ u32 prefix_xor32(u32 x) {  // bit j = xor of bits 0..j
    x ^= x << 1; x ^= x << 2; x ^= x << 4; x ^= x << 8; x ^= x << 16;
    return x;
}

__device__ __forceinline__ u64 mix64(u64 x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x;
}

// ------------------------------------------------------------------------------------------------
// device count table: (table, k, seq128) -> count, open addressing, linear probing
// (stands in for the per-worker ResultMap objects, src/kmer.h:79-81)
// ------------------------------------------------------------------------------------------------

__device__ __noinline__ void table_add_impl(Slot* slots, u32 slot_mask, u32* error_flag, u32 meta, u64 lo, u64 hi, u64 cnt) {
#ifdef TREW_EXP_NOADD
    return;
#endif
    u64 h = mix64(lo ^ mix64(hi + 0x9e3779b97f4a7c15ULL * (u64)(meta + 1)));
    u32 i = (u32)h & slot_mask;
    for (u32 probe = 0; probe <= slot_mask; probe++, i = (i + 1) & slot_mask) {
        Slot* s = slots + i;
        // fast path (almost every add hits an existing key): one 32-byte read of the slot, then a fire-and-forget add
        const uint4 a = __ldcg(reinterpret_cast<const uint4*>(s)), c = __ldcg(reinterpret_cast<const uint4*>(s) + 1);
        u32 st = c.w;
        if (st == 2u) {
            if (c.z == meta && a.x == (u32)lo && a.y == (u32)(lo >> 32) && a.z == (u32)hi && a.w == (u32)(hi >> 32)) {
                atomicAdd(&s->count, cnt);  // keys never change once written, so a match cannot be a torn read
                return;
            }
            // mismatch: the two 16-byte reads are not ordered against a concurrent writer, so look again now that the
            // slot is known to be ready before concluding that another key lives here
            __threadfence();
            if (__ldcg(&s->meta) == meta && __ldcg(&s->seq_lo) == lo && __ldcg(&s->seq_hi) == hi) {
                atomicAdd(&s->count, cnt);
                return;
            }
            continue;
        }
        // The slot is empty or being written.  Lanes of ONE warp may be here with the same key (the thread-per-survivor
        // kernel: 32 reads of the same repeat), so nobody spins on the writer: every round all of them try the CAS, the
        // winner publishes inside the same round, and the others meet a ready slot in the next one.  (A plain spin on
        // `state == 1` leaves it to the scheduler when the winner's branch runs -- measured: tens of ms.)
        int outcome = 0;   // 0 look again, 1 added, 2 the slot holds another key
        do {
            st = atomicCAS(&s->state, 0u, 1u);
            if (st == 0u) {
                s->seq_lo = lo; s->seq_hi = hi; s->meta = meta;
                __threadfence();
                atomicExch(&s->state, 2u);
                atomicAdd(&s->count, cnt);
                atomicAdd(error_flag + 1, 1u);  // distinct keys so far: the host grows the table before it fills up
                outcome = 1;
            } else if (st == 2u) {
                __threadfence();
                if (__ldcg(&s->meta) == meta && __ldcg(&s->seq_lo) == lo && __ldcg(&s->seq_hi) == hi) {
                    atomicAdd(&s->count, cnt);
                    outcome = 1;
                } else outcome = 2;
            }
        } while (outcome == 0);
        if (outcome == 1) return;
    }
    atomicExch(error_flag, 3u);  // TREW_ERR_TABLE_FULL
}

// one unit record per calling thread.  Space is reserved once for the threads of the warp that arrive together (the
// routing emits the same few keys from every survivor, and same-address atomics retire one at a time in L2); the counter
// keeps counting past the capacity so that the host can tell how much would have been enough.
__device__ __forceinline__ void rec_append(UnitRecs* R, u64 unit, int table, int k, u64 lo, u64 hi, u64 count) {
    const u32 act = __activemask(), lane = threadIdx.x & 31;
    const int leader = __ffs(act) - 1;
    u64 base = 0;
    if ((int)lane == leader) base = atomicAdd(&R->n, (u64)__popc(act));
    base = __shfl_sync(act, base, leader);
    const u64 i = base + (u64)__popc(act & ((1u << lane) - 1u));
    if (i < R->cap) {
        uint4* p = reinterpret_cast<uint4*>(R->buf + i);
        p[0] = make_uint4((u32)unit, (u32)(unit >> 32), (u32)lo, (u32)(lo >> 32));
        p[1] = make_uint4((u32)hi, (u32)(hi >> 32), (u32)count, (u32)table | ((u32)k << 8));
    }
}

// adds another table's entries to this one: the device-side analogue of the per-thread map sum, src/kmer.cpp:1486-1515
__global__ void merge_entries_kernel(Slot* slots, u32 slot_mask, u32* error_flag, const trew_entry* __restrict__ e, u32 n) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        table_add_impl(slots, slot_mask, error_flag, ((u32)e[i].table << 8) | (u32)e[i].k, e[i].seq_lo, e[i].seq_hi, e[i].count);
}

void launch_merge_entries(const DevCfg& cfg, const trew_entry* entries, unsigned int n, cudaStream_t stream) {
    if (n) merge_entries_kernel<<<(n + 255) / 256, 256, 0, stream>>>(cfg.slots, cfg.slot_mask, cfg.error_flag, entries, n);
}

// ------------------------------------------------------------------------------------------------
// synthetic batch generator (benchmark tooling; mirrored by trew_b200/synth.py:device_mirror)
// ------------------------------------------------------------------------------------------------

__host__ __device__ inline u32 synth_hash(u64 seed, u64 a, u64 b) {
    u64 x = seed + 0x9e3779b97f4a7c15ULL * (a + 1) + 0xbf58476d1ce4e5b9ULL * (b + 1);
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ULL; x ^= x >> 27; x *= 0x94d049bb133111ebULL; x ^= x >> 31;
    return (u32)(x >> 32);
}

__global__ void synth_kernel(u64 seed, u32 n_reads, u32 L, u32 tel_thr, u32 half_thr, u32 n_thr, u32 sub_thr, u32 flavor,
                             u32* __restrict__ bit_off, u32* __restrict__ hi, u32* __restrict__ lo, u32* __restrict__ val,
                             size_t plane_words) {
    const u64 total = (u64)n_reads * L;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i <= n_reads; i += stride) bit_off[i] = (u32)(i * L);
    // codes T=0 G=1 C=2 A=3; TTAGGG and its reverse complement CCCTAA as code strings
    const int unit_f[6] = {0, 0, 3, 1, 1, 1};
    const int unit_r[6] = {2, 2, 2, 0, 3, 3};
    for (size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x; w < plane_words; w += stride) {
        u32 h = 0, l = 0, v = 0;
        for (int b = 0; b < 32; b++) {
            u64 pos = (u64)w * 32 + b;
            if (pos >= total) break;
            u64 r = pos / L; u32 j = (u32)(pos % L);
            const u64 frag = flavor == 1 ? r >> 1 : r;   // pairs: both mates share the fragment's draw
            u32 kind = synth_hash(seed, frag, 0xffffffffULL);
            u32 aux = synth_hash(seed, frag, 0xfffffffeULL);
            u32 code = synth_hash(seed, r, j) & 3u;
            bool tel = kind < tel_thr;
            bool halfk = !tel && kind < tel_thr + half_thr;
            if (halfk) tel = ((aux >> 8) & 1u) ? (j < L / 2) : (j >= L / 2);
            if (flavor == 2 && tel) {   // long reads: telomeric for the first or the last 500..5000 bases only
                u32 tl = 500u + synth_hash(seed, frag, 0xfffffffdULL) % 4501u;
                if (tl > L) tl = L;
                tel = ((aux >> 9) & 1u) ? (j < tl) : (j >= L - tl);
            }
            if (tel) {
                u32 phase = aux % 6u;
                bool rc = (((aux >> 4) & 1u) ^ (flavor == 1 ? (u32)(r & 1u) : 0u)) != 0u;
                u32 idx = (j + phase) % 6u;
                u32 c = rc ? unit_r[idx] : unit_f[idx];
                u32 sh = synth_hash(seed ^ 0x5555555555555555ULL, r, j);
                code = sh < sub_thr ? (sh >> 3) & 3u : c;   // note: sh < sub_thr keeps (sh >> 3) & 3 uniform enough
            }
            bool inval = synth_hash(seed ^ 0xaaaaaaaaaaaaaaaaULL, r, j) < n_thr;
            if (!inval) { v |= 1u << b; h |= (code >> 1) << b; l |= (code & 1u) << b; }
        }
        hi[w] = h; lo[w] = l; val[w] = v;
    }
}

void launch_synth(unsigned long long seed, unsigned int n_reads, unsigned int read_len, unsigned int tel_thr,
                  unsigned int half_thr, unsigned int n_thr, unsigned int sub_thr, unsigned int flavor, unsigned int* bit_off,
                  unsigned int* hi, unsigned int* lo, unsigned int* val, size_t plane_words, cudaStream_t stream) {
    synth_kernel<<<1184, 256, 0, stream>>>(seed, n_reads, read_len, tel_thr, half_thr, n_thr, sub_thr, flavor, bit_off, hi, lo, val,
                                            plane_words);
}

// ------------------------------------------------------------------------------------------------
// probe windows: the first windows the reference's routing scans for a unit.  If none of them can
// produce a target k, the unit emits nothing (see DESIGN.md, "Why the filter is sound").
// ------------------------------------------------------------------------------------------------

struct Probe { u32 pos; int wl, k0, k1; };

__device__ __forceinline__ int unit_probes(const DevCfg& c, const DevBatch& b, u32 u, Probe* p) {
    const int MINM = c.min_mer, MAXM = c.max_mer;
    int np = 0;
    if (c.mode == 0) {  // buffer_task, src/kmer.cpp:111-171
        u32 b0 = __ldg(b.bit_off + u);
        int n = (int)(__ldg(b.bit_off + u + 1) - b0);
        if (n < 2 * MINM) return 0;
        if (n >= 4 * MINM) {
            int kmax = min(n / 4, MAXM);
            p[np++] = Probe{b0, n / 2, MINM, kmax};
            p[np++] = Probe{b0 + (u32)(n - (n + 1) / 2), (n + 1) / 2, MINM, kmax};
        }
        if (4 * MAXM > n) p[np++] = Probe{b0, n, max(n / 4 + 1, MINM), min(n / 2, MAXM)};
    } else if (c.mode == 1) {  // buffer_task_pair, src/kmer.cpp:322-505
        u32 a0 = __ldg(b.bit_off + 2 * u), a1 = __ldg(b.bit_off + 2 * u + 1), a2 = __ldg(b.bit_off + 2 * u + 2);
        int n1 = (int)(a1 - a0), n2 = (int)(a2 - a1);
        int n = min(n1, n2);
        if (n < 2 * MINM) return 0;
        if (n >= 4 * MINM) {
            int kmax = min(n / 4, MAXM);
            p[np++] = Probe{a0, n1 / 2, MINM, kmax};  // segment 1: forward walk starts here
            p[np++] = Probe{a1, n2 / 2, MINM, kmax};  // segment 4: backward walk starts here
        }
        if (4 * MAXM > n) {
            int lo = max(n / 4 + 1, MINM), hi = min(n / 2, MAXM);
            p[np++] = Probe{a0, n1, lo, hi};
            p[np++] = Probe{a1, n2, lo, hi};
        }
    } else {  // buffer_task_long, src/kmer.cpp:785-856
        u32 b0 = __ldg(b.bit_off + u);
        int n = (int)(__ldg(b.bit_off + u + 1) - b0);
        const int SL = c.slice_len;
        if (n < SL) return 0;
        int snum = n / SL, mid = (snum + 1) / 2, bonus = n % SL;
        int l1 = SL + (1 == mid ? bonus : 0);
        p[np++] = Probe{b0, l1, MINM, MAXM};
        if (snum > 1) {
            int l2 = SL + (snum == mid ? bonus : 0);
            p[np++] = Probe{b0 + (u32)(n - l2), l2, MINM, MAXM};
        }
    }
    return np;
}

// ------------------------------------------------------------------------------------------------
// filter kernel: thread per unit, multiword bit-planes in registers
// ------------------------------------------------------------------------------------------------

template <int NW>
__device__ __forceinline__ void load_bits(const u32* __restrict__ plane, u32 pos, u32 (&out)[NW]) {
    const u32* p = plane + (pos >> 5);
    u32 sh = pos & 31;
    u32 prev = __ldg(p);
#pragma unroll
    for (int j = 0; j < NW; j++) {
        u32 nxt = __ldg(p + j + 1);
        out[j] = __funnelshift_r(prev, nxt, sh);
        prev = nxt;
    }
}

template <int NW>
__device__ __forceinline__ void mask_bits(u32 (&x)[NW], int wl) {
#pragma unroll
    for (int j = 0; j < NW; j++) {
        int v = wl - 32 * j;
        x[j] &= v <= 0 ? 0u : low_mask(v);
    }
}

// exclusive prefix XOR over the multiword bit vector: out bit i = xor of in bits [0, i)
template <int NW>
__device__ __forceinline__ void prefix_xor_excl(const u32 (&in)[NW], u32 (&out)[NW]) {
    u32 carry = 0, prev_top = 0;
#pragma unroll
    for (int j = 0; j < NW; j++) {
        u32 inc = prefix_xor32(in[j]) ^ carry;
        out[j] = (inc << 1) | prev_top;
        prev_top = inc >> 31;
        carry = 0u - prev_top;
    }
}

template <int NW>
__device__ __forceinline__ void shr1(u32 (&x)[NW]) {
#pragma unroll
    for (int j = 0; j < NW; j++) x[j] = __funnelshift_r(x[j], j + 1 < NW ? x[j + 1] : 0u, 1);
}

template <int NW>
__device__ __forceinline__ void shr_var(const u32 (&in)[NW], int k, u32 (&out)[NW]) {
#pragma unroll
    for (int j = 0; j < NW; j++) out[j] = in[j];
    for (int s = k >> 5; s > 0; s--) {
#pragma unroll
        for (int j = 0; j < NW; j++) out[j] = j + 1 < NW ? out[j + 1] : 0u;
    }
    u32 r = k & 31;
#pragma unroll
    for (int j = 0; j < NW; j++) out[j] = __funnelshift_r(out[j], j + 1 < NW ? out[j + 1] : 0u, r);
}

// window-valid mask for period k: bit i set iff bases i..i+k-1 are all valid (doubling)
template <int NW>
__device__ __forceinline__ void sliding_and(u32 (&a)[NW], int k) {
    u32 t[NW];
    int w = 1;
    while (2 * w <= k) {
        shr_var<NW>(a, w, t);
#pragma unroll
        for (int j = 0; j < NW; j++) a[j] &= t[j];
        w *= 2;
    }
    if (k > w) {
        shr_var<NW>(a, k - w, t);
#pragma unroll
        for (int j = 0; j < NW; j++) a[j] &= t[j];
    }
}

__device__ __forceinline__ void csa(u32 a, u32 b, u32 c, u32& s, u32& cy) {
    s = a ^ b ^ c;
    cy = (a & b) | (c & (a ^ b));
}

// popcount of a multiword vector with carry-save compression (POPC is quarter-rate; LOP3 is not)
template <int NW>
__device__ __forceinline__ int popc_multi(const u32 (&x)[NW]) {
    if constexpr (NW == 1) return __popc(x[0]);
    else if constexpr (NW == 2) return __popc(x[0]) + __popc(x[1]);
    else if constexpr (NW == 3) {
        u32 s, c; csa(x[0], x[1], x[2], s, c);
        return __popc(s) + 2 * __popc(c);
    } else if constexpr (NW == 5) {
        u32 s1, c1, s2, c2; csa(x[0], x[1], x[2], s1, c1); csa(s1, x[3], x[4], s2, c2);
        return __popc(s2) + 2 * (__popc(c1) + __popc(c2));
    } else if constexpr (NW == 8) {
        u32 s1, c1, s2, c2, s3, c3, s4, c4;
        csa(x[0], x[1], x[2], s1, c1); csa(x[3], x[4], x[5], s2, c2); csa(s1, s2, x[6], s3, c3);
        csa(c1, c2, c3, s4, c4);
        return __popc(s3) + __popc(x[7]) + 2 * __popc(s4) + 4 * __popc(c4);
    } else {
        int t = 0;
#pragma unroll
        for (int j = 0; j < NW; j++) t += __popc(x[j]);
        return t;
    }
}

// Returns true iff some k in [k0, k1] MAY reach the LOW threshold in window [pos, pos + wl).
template <int NW>
__device__ __noinline__ bool probe_filter(const DevBatch& b, u32 pos, int wl, int k0, int k1,
                                          const unsigned short* __restrict__ thr) {
    u32 PH[NW], PL[NW], QH[NW], QL[NW], WV[NW];
    {
        u32 t[NW];
        load_bits<NW>(b.hi, pos, t); prefix_xor_excl<NW>(t, PH);
        load_bits<NW>(b.lo, pos, t); prefix_xor_excl<NW>(t, PL);
        load_bits<NW>(b.val, pos, WV); mask_bits<NW>(WV, wl);
    }
    shr_var<NW>(PH, k0, QH);
    shr_var<NW>(PL, k0, QL);
    sliding_and<NW>(WV, k0);
    u32 PA[NW];
    bool have_pa = false;
    for (int k = k0; k <= k1; k++) {
        u32 a[NW], bb[NW], c[NW];
#pragma unroll
        for (int j = 0; j < NW; j++) {
            u32 dh = QH[j] ^ PH[j], dl = QL[j] ^ PL[j];
            a[j] = dh & WV[j]; bb[j] = dl & WV[j]; c[j] = a[j] & dl;
        }
        int T = popc_multi<NW>(WV);
        if (T == 0) break;  // the valid-window mask only shrinks with k
        int cH = popc_multi<NW>(a), cL = popc_multi<NW>(bb), c11 = popc_multi<NW>(c);
        int c10 = cH - c11, c01 = cL - c11, c00 = T - cH - cL + c11;
        int U = max(max(c00, c01), max(c10, c11));
        int need = thr[T];
        if (U >= need) {
            // second level: add the parity of the A count (rare: ~2.5e-4 per (window, k) on random reads)
            u32 QA[NW];
            if (!have_pa) {
                u32 A[NW], t[NW];
                load_bits<NW>(b.hi, pos, A); load_bits<NW>(b.lo, pos, t);
#pragma unroll
                for (int j = 0; j < NW; j++) A[j] &= t[j];
                prefix_xor_excl<NW>(A, PA);
                have_pa = true;
            }
            shr_var<NW>(PA, k, QA);
            u32 x11[NW], x10[NW], x01[NW], x00[NW];
#pragma unroll
            for (int j = 0; j < NW; j++) {
                u32 da = QA[j] ^ PA[j];
                u32 dh = QH[j] ^ PH[j], dl = QL[j] ^ PL[j];
                x11[j] = c[j] & da; x10[j] = a[j] & ~dl & da; x01[j] = bb[j] & ~dh & da; x00[j] = WV[j] & ~dh & ~dl & da;
            }
            int n11 = popc_multi<NW>(x11), n10 = popc_multi<NW>(x10), n01 = popc_multi<NW>(x01), n00 = popc_multi<NW>(x00);
            int U2 = max(max(max(n11, c11 - n11), max(n10, c10 - n10)), max(max(n01, c01 - n01), max(n00, c00 - n00)));
            if (U2 >= need) return true;
        }
        shr1<NW>(QH); shr1<NW>(QL);
        u32 t[NW];
#pragma unroll
        for (int j = 0; j < NW; j++) t[j] = WV[j];
        shr1<NW>(t);
#pragma unroll
        for (int j = 0; j < NW; j++) WV[j] &= t[j];
    }
    return false;
}

template <int MAXNW>
__device__ __forceinline__ bool probe_dispatch(const DevBatch& b, const Probe& p, const unsigned short* thr) {
    if (p.k1 < p.k0) return false;
    int need_bits = p.wl + 1;  // prefix planes hold wl + 1 entries
    if (need_bits <= 96) return probe_filter<3>(b, p.pos, p.wl, p.k0, p.k1, thr);
    if constexpr (MAXNW >= 5) { if (need_bits <= 160) return probe_filter<5>(b, p.pos, p.wl, p.k0, p.k1, thr); }
    if constexpr (MAXNW >= 8) { if (need_bits <= 256) return probe_filter<8>(b, p.pos, p.wl, p.k0, p.k1, thr); }
    return true;  // window too long for the bit-parallel filter: let the exact kernel decide
}

// ---- screen kernel: fast first level ---------------------------------------------------------------
//
// For probe windows of at most 95 bases without invalid bases the first-level test runs on the first 64
// window positions only (two words per plane): with T = wl - k + 1 windows, T01 = min(T, 64) of them start
// in [0, 64) and E = T - T01 beyond, and
//     M <= U01 + E,   U01 = largest of the four parity-signature buckets among the first 64 positions,
// so "U01 >= need(T) - E" is necessary for period k to reach LOW.  The four bucket counts are formed as the
// four bytes of one word on the FMA pipe (byte0 = c11, byte1 = cH - c11, byte2 = cL - c11,
// byte3 = T01 - cH - cL + c11) on top of a per-T base that adds 128 - (need - E) to every byte: a bucket
// reaches the threshold iff the top bit of its byte is set.  A unit whose probes all fail the test emits
// nothing.  Everything else -- a first-level hit, an invalid base, a longer window -- is put on the
// deferred list and decided by the exact-bound kernel below, so this level only has to be sound, not tight.

constexpr u32 kPackC11 = 1u - (1u << 8) - (1u << 16) + (1u << 24);
constexpr u32 kPackH = (1u << 8) - (1u << 24);
constexpr u32 kPackL = (1u << 16) - (1u << 24);
#ifndef TREW_SCREEN_UNROLL
#define TREW_SCREEN_UNROLL 2
#endif
constexpr int kScreenUnroll = TREW_SCREEN_UNROLL;
constexpr int kFastMaxWl = 95;
constexpr int kFastTabSize = kFastMaxWl + 2;
constexpr int kProbeShift = 28;  // deferred-list entry: unit index | probe mask << 28
constexpr int kMod4BelowWindows = 48;    // decide kernel: the third (mod-4) level is asked for periods with fewer valid windows than this (measured: 24 / 36 / 48 / always -> 2.07 / 2.05 / 2.03 / 2.14 ms decide + exact per 25 M reads, none: 2.18)
constexpr int kThreadMinWindows = 36;   // decide kernel: survivors whose first passing period has fewer valid windows go to the warp kernel

// per-T entry: x = packed base word, y / z = masks of the window positions in words 0 / 1
__device__ __forceinline__ uint4 fast_entry(int T, int need) {
    uint4 e = make_uint4(0u, 0u, 0u, 0u);
    if (T <= 0) return e;                       // no window: every byte stays 0
    int T01 = min(T, 64);
    e.y = T >= 32 ? 0xffffffffu : ((1u << T) - 1u);
    e.z = T <= 32 ? 0u : (T >= 64 ? 0xffffffffu : ((1u << (T - 32)) - 1u));
    int np = need - (T - T01);
    if (np <= 0) e.x = 0x80808080u;             // the bound cannot reject: always a hit
    else if (np > 64) e.x = (u32)T01 << 24;     // no bucket of <= 64 positions can reach it
    else e.x = ((u32)T01 << 24) + (u32)(128 - np) * 0x01010101u;
    return e;
}

// periods ka..kb (all with k >> 5 == S) of one all-valid window; true iff some period passes the first level
template <int S>
__device__ __forceinline__ bool fast_span(const u32 (&ph)[5], const u32 (&pl)[5], int wl, int ka, int kb,
                                          const uint4* __restrict__ tab) {
    const uint4* tp = tab + (wl - ka + 1);
#pragma unroll (kScreenUnroll)
    for (int k = ka; k <= kb; k++, tp--) {
        const uint4 e = *tp;
        u32 qh0 = __funnelshift_r(ph[S], ph[S + 1], k), qh1 = __funnelshift_r(ph[S + 1], ph[S + 2], k);
        u32 ql0 = __funnelshift_r(pl[S], pl[S + 1], k), ql1 = __funnelshift_r(pl[S + 1], pl[S + 2], k);
        u32 a0 = (qh0 ^ ph[0]) & e.y, a1 = (qh1 ^ ph[1]) & e.z;
        u32 b0 = (ql0 ^ pl[0]) & e.y, b1 = (ql1 ^ pl[1]) & e.z;
        u32 x = e.x + (u32)(__popc(a0) + __popc(a1)) * kPackH + (u32)(__popc(b0) + __popc(b1)) * kPackL +
                (u32)(__popc(a0 & b0) + __popc(a1 & b1)) * kPackC11;
        if (x & 0x80808080u) return true;
    }
    return false;
}

__device__ __forceinline__ bool probe_is_fast(const Probe& p) { return p.wl <= kFastMaxWl && p.k1 <= 63 && p.k1 <= p.wl; }

// true iff the probe must be decided by the exact-bound kernel
__device__ __forceinline__ bool screen_probe(const DevBatch& b, const Probe& p, const uint4* __restrict__ tab) {
    if (p.k1 < p.k0) return false;
    if (!probe_is_fast(p)) return true;
    u32 t[3], full[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu};
    mask_bits<3>(full, p.wl);
    load_bits<3>(b.val, p.pos, t);
    if ((((t[0] & full[0]) ^ full[0]) | ((t[1] & full[1]) ^ full[1]) | ((t[2] & full[2]) ^ full[2])) != 0u) return true;
    u32 ph[5], pl[5], q[3];
    load_bits<3>(b.hi, p.pos, t); mask_bits<3>(t, p.wl); prefix_xor_excl<3>(t, q);
    ph[0] = q[0]; ph[1] = q[1]; ph[2] = q[2]; ph[3] = 0u; ph[4] = 0u;
    load_bits<3>(b.lo, p.pos, t); mask_bits<3>(t, p.wl); prefix_xor_excl<3>(t, q);
    pl[0] = q[0]; pl[1] = q[1]; pl[2] = q[2]; pl[3] = 0u; pl[4] = 0u;
    int k0 = p.k0;
    if (k0 < 32) {
        if (fast_span<0>(ph, pl, p.wl, k0, min(p.k1, 31), tab)) return true;
        k0 = 32;
    }
    return p.k1 >= 32 && fast_span<1>(ph, pl, p.wl, k0, p.k1, tab);
}

// ---- the same first level for windows of 96..159 bases (long-read slices, 300-base short reads, the whole-read probe
// of 150-base reads when MAX_MER > 37): four words per plane, i.e. the first 128 window positions, E = T - 128 beyond.
constexpr int kFastMaxWlLong = 159;
constexpr int kFastTabSizeLong = kFastMaxWlLong + 2;
struct __align__(16) FastEntryLong { u32 base, m0, m1, m2, m3, pad0, pad1, pad2; };

__device__ __forceinline__ FastEntryLong fast_entry_long(int T, int need) {
    FastEntryLong e = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
    if (T <= 0) return e;
    const int T01 = min(T, 128);
    u32 m[4];
#pragma unroll
    for (int j = 0; j < 4; j++) { int vb = T - 32 * j; m[j] = vb <= 0 ? 0u : low_mask(min(32, vb)); }
    e.m0 = m[0]; e.m1 = m[1]; e.m2 = m[2]; e.m3 = m[3];
    const int np = need - (T - T01);
    if (np <= 0) e.base = 0x80808080u;
    else if (np > 128) e.base = 0u;   // no bucket of <= 128 positions can reach it: never a hit (T01 dropped on purpose:
                                      // without the offset the byte arithmetic is not needed at all)
    else e.base = ((u32)T01 << 24) + (u32)(128 - np) * 0x01010101u;
    return e;
}

template <int S>
__device__ __forceinline__ bool fast_span_long(const u32 (&ph)[8], const u32 (&pl)[8], int wl, int ka, int kb,
                                               const FastEntryLong* __restrict__ tab) {
    const FastEntryLong* tp = tab + (wl - ka + 1);
    for (int k = ka; k <= kb; k++, tp--) {
        const uint4 e0 = *reinterpret_cast<const uint4*>(tp);       // base, m0, m1, m2
        const u32 m3 = tp->m3;
        if (e0.x == 0u) continue;                                    // unreachable threshold (or no window)
        const u32 mk[4] = {e0.y, e0.z, e0.w, m3};
        int cH = 0, cL = 0, c11 = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            u32 a = (__funnelshift_r(ph[S + j], ph[S + j + 1], k) ^ ph[j]) & mk[j];
            u32 bb = (__funnelshift_r(pl[S + j], pl[S + j + 1], k) ^ pl[j]) & mk[j];
            cH += __popc(a); cL += __popc(bb); c11 += __popc(a & bb);
        }
        u32 x = e0.x + (u32)cH * kPackH + (u32)cL * kPackL + (u32)c11 * kPackC11;
        if (x & 0x80808080u) return true;
    }
    return false;
}

__device__ __forceinline__ bool probe_is_fast_long(const Probe& p) { return p.wl <= kFastMaxWlLong && p.k1 <= 64 && p.k1 <= p.wl; }

__device__ __noinline__ bool screen_probe_long(const DevBatch& b, const Probe& p, const FastEntryLong* __restrict__ tab) {
    u32 t[5], full[5] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
    mask_bits<5>(full, p.wl);
    load_bits<5>(b.val, p.pos, t);
    u32 bad = 0;
#pragma unroll
    for (int j = 0; j < 5; j++) bad |= (t[j] & full[j]) ^ full[j];
    if (bad) return true;
    u32 ph[8], pl[8], q[5];
    load_bits<5>(b.hi, p.pos, t); mask_bits<5>(t, p.wl); prefix_xor_excl<5>(t, q);
#pragma unroll
    for (int j = 0; j < 8; j++) ph[j] = j < 5 ? q[j] : 0u;
    load_bits<5>(b.lo, p.pos, t); mask_bits<5>(t, p.wl); prefix_xor_excl<5>(t, q);
#pragma unroll
    for (int j = 0; j < 8; j++) pl[j] = j < 5 ? q[j] : 0u;
    int k0 = p.k0;
    if (k0 < 32) {
        if (fast_span_long<0>(ph, pl, p.wl, k0, min(p.k1, 31), tab)) return true;
        k0 = 32;
    }
    if (k0 < 64 && p.k1 >= 32) {
        if (fast_span_long<1>(ph, pl, p.wl, k0, min(p.k1, 63), tab)) return true;
        k0 = 64;
    }
    return p.k1 >= 64 && fast_span_long<2>(ph, pl, p.wl, k0, p.k1, tab);
}

// warp-aggregated append of the flagged lanes' values to a global list
__device__ __forceinline__ void list_append(bool flag, u32 value, u32* __restrict__ list, u32* __restrict__ count) {
    u32 m = __ballot_sync(0xffffffffu, flag);
    if (m) {
        u32 base = 0;
        if (lane_id() == 0) base = atomicAdd(count, (u32)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (flag) list[base + __popc(m & ((1u << lane_id()) - 1u))] = value;
    }
}

// the same, for a list that grows downwards from *top
__device__ __forceinline__ void list_append_rev(bool flag, u32 value, u32* __restrict__ top, u32* __restrict__ count) {
    u32 m = __ballot_sync(0xffffffffu, flag);
    if (m) {
        u32 base = 0;
        if (lane_id() == 0) base = atomicAdd(count, (u32)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (flag) *(top - (base + __popc(m & ((1u << lane_id()) - 1u)))) = value;
    }
}

#ifndef TREW_SCREEN_BPS
#define TREW_SCREEN_BPS 8
#endif
template <bool LONG>
__global__ void __launch_bounds__(256, LONG ? 4 : TREW_SCREEN_BPS) trew_screen_kernel(DevCfg cfg, DevBatch b, u32 n_units,
                                                                                     u32* __restrict__ deferred, u32* __restrict__ n_deferred) {
    __shared__ uint4 tab[kFastTabSize];
    __shared__ FastEntryLong tab_long[LONG ? kFastTabSizeLong : 1];
    for (int T = threadIdx.x; T < kFastTabSize; T += blockDim.x) tab[T] = fast_entry(T, (int)cfg.thr_low[T]);
    if (LONG) for (int T = threadIdx.x; T < kFastTabSizeLong; T += blockDim.x) tab_long[T] = fast_entry_long(T, (int)cfg.thr_low[T]);
    __syncthreads();
    u32 stride = gridDim.x * blockDim.x;
    u32 n_round = (n_units + 31u) & ~31u;
    for (u32 u = blockIdx.x * blockDim.x + threadIdx.x; u < n_round; u += stride) {
        u32 pm = 0;  // probes the decide kernel has to look at
        if (u < n_units) {
            Probe p[4];
            int np = unit_probes(cfg, b, u, p);
            for (int i = 0; i < np; i++) {
                bool d;
                if (LONG && p[i].k1 >= p[i].k0 && !probe_is_fast(p[i]) && probe_is_fast_long(p[i])) d = screen_probe_long(b, p[i], tab_long);
                else d = screen_probe(b, p[i], tab);
                pm |= d ? 1u << i : 0u;
            }
        }
        list_append(pm != 0, u | (pm << kProbeShift), deferred, n_deferred);
    }
}

// Deciding test for one probe window of at most 95 bases, invalid bases allowed: per period, the 4-bucket bound on the
// first 64 window positions plus the E windows beyond them (necessary condition, as in the screen), then the exact
// 3-word bound, then the #A-parity second level.  Same decisions as probe_filter<3>, fewer instructions.
__device__ __forceinline__ int max4(int a, int b, int c, int d) { return max(max(a, b), max(c, d)); }

// Third level of the decide test: the counts of hi bits, lo bits and A's of a k-window MOD 4 are rotation invariants too
// (the first two levels use them mod 2), so a class lies inside one of 64 buckets.  The second bits of the three counts
// come from second-order prefix planes -- P1 = exclusive prefix XOR of (x & P0), the carries of a running 2-bit count;
// bit 1 of a window's count is P1[i + k] ^ P1[i] ^ (~P0[i + k] & P0[i]) (the borrow of the low bits).  What an N leaves
// of a window -- a dozen k-windows, half of which fall into one of 8 buckets by chance at some period -- stops here
// instead of becoming a survivor.  Reached by a few percent of the decided probes, so it is a function of its own: nothing
// of it lives in the registers of the loop over the periods; the probe's first call builds the six prefix planes from the
// batch and parks them in shared memory (cache: word i of the thread at cache[i * 256]), later calls reload them.
// pass8: the buckets of the second level that hold `need` windows (bit = hi | lo << 1 | A << 2 parity differences).
// true = some bucket of the 64 may still hold `need` of the valid windows wv (the k-windows of this period).
__device__ __forceinline__ u32 shr3(const u32 (&p)[3], int j, int k) {   // word j of (p >> k), k < 64, zero beyond word 2
    const int s = k >> 5;
    const u32 lo = j + s < 3 ? (s ? (j == 0 ? p[1] : p[2]) : p[j]) : 0u;
    const u32 hi = j + s + 1 < 3 ? (s ? p[2] : (j == 0 ? p[1] : p[2])) : 0u;
    return __funnelshift_r(lo, hi, k);
}
constexpr int kDecideThreads = 256;
__device__ __noinline__ bool mod4_level(const DevBatch& b, u32 pos, int wl, int k, int need, u32 pass8, u32 wv0, u32 wv1, u32 wv2, u32* cache,
                                        bool& cached) {
    const u32 wv[3] = {wv0, wv1, wv2};
    u32 p0[3][3], p1[3][3];   // planes: hi, lo, A
    if (!cached) {
        u32 x[3][3];
        load_bits<3>(b.hi, pos, x[0]); mask_bits<3>(x[0], wl);
        load_bits<3>(b.lo, pos, x[1]); mask_bits<3>(x[1], wl);
#pragma unroll
        for (int j = 0; j < 3; j++) x[2][j] = x[0][j] & x[1][j];
#pragma unroll
        for (int p = 0; p < 3; p++) {
            prefix_xor_excl<3>(x[p], p0[p]);
            u32 c[3];
#pragma unroll
            for (int j = 0; j < 3; j++) c[j] = x[p][j] & p0[p][j];
            prefix_xor_excl<3>(c, p1[p]);
#pragma unroll
            for (int j = 0; j < 3; j++) { cache[(6 * p + j) * kDecideThreads] = p0[p][j]; cache[(6 * p + 3 + j) * kDecideThreads] = p1[p][j]; }
        }
        cached = true;
    } else {
#pragma unroll
        for (int p = 0; p < 3; p++)
#pragma unroll
            for (int j = 0; j < 3; j++) { p0[p][j] = cache[(6 * p + j) * kDecideThreads]; p1[p][j] = cache[(6 * p + 3 + j) * kDecideThreads]; }
    }
    u32 d0[3][3], d1[3][3];   // first and second bit of the three counts of the window starting at each position
#pragma unroll
    for (int p = 0; p < 3; p++) {
#pragma unroll
        for (int j = 0; j < 3; j++) {
            const u32 q0 = shr3(p0[p], j, k);
            d0[p][j] = q0 ^ p0[p][j];
            d1[p][j] = shr3(p1[p], j, k) ^ p1[p][j] ^ (~q0 & p0[p][j]);
        }
    }
#pragma unroll 1
    for (int c2 = 0; c2 < 8; c2++) {   // buckets of the second level
        if (!((pass8 >> c2) & 1u)) continue;
        u32 mw[3];
        int cnt = 0;
#pragma unroll
        for (int j = 0; j < 3; j++) {
            mw[j] = wv[j] & (d0[0][j] ^ ((c2 & 1) ? 0u : ~0u)) & (d0[1][j] ^ ((c2 & 2) ? 0u : ~0u)) & (d0[2][j] ^ ((c2 & 4) ? 0u : ~0u));
            cnt += __popc(mw[j]);
        }
        if (cnt < need) continue;
        // split by the three second bits in turn, following the larger side; a smaller side that could still reach `need`
        // too (a tie at exactly half) is not followed but counted as "may"
        bool may = true;
#pragma unroll
        for (int p = 0; p < 3 && may; p++) {
            const int one = __popc(mw[0] & d1[p][0]) + __popc(mw[1] & d1[p][1]) + __popc(mw[2] & d1[p][2]);
            const int zero = cnt - one;
            if (min(one, zero) >= need) return true;
            const u32 flip = one >= zero ? 0u : ~0u;
#pragma unroll
            for (int j = 0; j < 3; j++) mw[j] &= d1[p][j] ^ flip;
            cnt = max(one, zero);
            may = cnt >= need;
        }
        if (may) return true;
    }
    return false;
}

template <int S>
__device__ __forceinline__ bool decide_span(const u32 (&ph)[5], const u32 (&pl)[5], const u32 (&pa)[5], u32 (&wv)[3], int ka, int kb,
                                            const unsigned short* __restrict__ thr, bool& done, int& t_hit, const DevBatch& bt, u32 pos, int wl,
                                            u32* cache, bool& cached, int m4_below) {
    for (int k = ka; k <= kb; k++) {
        const int T01 = __popc(wv[0]) + __popc(wv[1]), E = __popc(wv[2]), T = T01 + E;
        if (T == 0) { done = true; return false; }  // the valid-window mask only shrinks with k
        const int need = thr[T];
        u32 a0 = (__funnelshift_r(ph[S], ph[S + 1], k) ^ ph[0]) & wv[0], a1 = (__funnelshift_r(ph[S + 1], ph[S + 2], k) ^ ph[1]) & wv[1];
        u32 b0 = (__funnelshift_r(pl[S], pl[S + 1], k) ^ pl[0]) & wv[0], b1 = (__funnelshift_r(pl[S + 1], pl[S + 2], k) ^ pl[1]) & wv[1];
        int cH = __popc(a0) + __popc(a1), cL = __popc(b0) + __popc(b1), c11 = __popc(a0 & b0) + __popc(a1 & b1);
        if (max4(c11, cH - c11, cL - c11, T01 - cH - cL + c11) + E >= need) {
            u32 a2 = (__funnelshift_r(ph[S + 2], ph[S + 3], k) ^ ph[2]) & wv[2], b2 = (__funnelshift_r(pl[S + 2], pl[S + 3], k) ^ pl[2]) & wv[2];
            cH += __popc(a2); cL += __popc(b2); c11 += __popc(a2 & b2);
            const int c10 = cH - c11, c01 = cL - c11, c00 = T - cH - cL + c11;
            if (max4(c11, c10, c01, c00) >= need) {
                u32 x0 = __funnelshift_r(pa[S], pa[S + 1], k) ^ pa[0], x1 = __funnelshift_r(pa[S + 1], pa[S + 2], k) ^ pa[1];
                u32 x2 = __funnelshift_r(pa[S + 2], pa[S + 3], k) ^ pa[2];
                int n11 = __popc(a0 & b0 & x0) + __popc(a1 & b1 & x1) + __popc(a2 & b2 & x2);
                int n10 = __popc(a0 & ~b0 & x0) + __popc(a1 & ~b1 & x1) + __popc(a2 & ~b2 & x2);
                int n01 = __popc(b0 & ~a0 & x0) + __popc(b1 & ~a1 & x1) + __popc(b2 & ~a2 & x2);
                int n00 = __popc(wv[0] & ~a0 & ~b0 & x0) + __popc(wv[1] & ~a1 & ~b1 & x1) + __popc(wv[2] & ~a2 & ~b2 & x2);
                int U2 = max(max4(n11, c11 - n11, n10, c10 - n10), max4(n01, c01 - n01, n00, c00 - n00));
                if (U2 >= need) {
                    const u32 pass8 = (u32)(c00 - n00 >= need) | (u32)(c10 - n10 >= need) << 1 | (u32)(c01 - n01 >= need) << 2 |
                                      (u32)(c11 - n11 >= need) << 3 | (u32)(n00 >= need) << 4 | (u32)(n10 >= need) << 5 |
                                      (u32)(n01 >= need) << 6 | (u32)(n11 >= need) << 7;
                    // with most of the window's k-windows still valid this is nearly always a repeat: no need to ask
                    if (T >= m4_below || mod4_level(bt, pos, wl, k, need, pass8, wv[0], wv[1], wv[2], cache, cached)) { t_hit = T; return true; }
                }
            }
        }
        u32 t0 = __funnelshift_r(wv[0], wv[1], 1), t1 = __funnelshift_r(wv[1], wv[2], 1), t2 = wv[2] >> 1;
        wv[0] &= t0; wv[1] &= t1; wv[2] &= t2;
    }
    return false;
}

// t_hit: the number of valid windows at the first period that passes (tells a repeat -- most of the window -- from a
// window an N left a dozen k-windows of)
__device__ __noinline__ bool decide_short(const DevBatch& b, u32 pos, int wl, int k0, int k1, const unsigned short* __restrict__ thr, int& t_hit,
                                          u32* cache, int m4_below) {
    bool cached = false;
    u32 wv[3], ph[5], pl[5], pa[5];
    load_bits<3>(b.val, pos, wv); mask_bits<3>(wv, wl);
    {
        u32 h[3], l[3], q[3];
        load_bits<3>(b.hi, pos, h); mask_bits<3>(h, wl); prefix_xor_excl<3>(h, q);
        ph[0] = q[0]; ph[1] = q[1]; ph[2] = q[2]; ph[3] = 0u; ph[4] = 0u;
        load_bits<3>(b.lo, pos, l); mask_bits<3>(l, wl); prefix_xor_excl<3>(l, q);
        pl[0] = q[0]; pl[1] = q[1]; pl[2] = q[2]; pl[3] = 0u; pl[4] = 0u;
#pragma unroll
        for (int j = 0; j < 3; j++) h[j] &= l[j];
        prefix_xor_excl<3>(h, q);
        pa[0] = q[0]; pa[1] = q[1]; pa[2] = q[2]; pa[3] = 0u; pa[4] = 0u;
    }
    sliding_and<3>(wv, k0);
    bool done = false;
    if (k0 < 32) {
        if (decide_span<0>(ph, pl, pa, wv, k0, min(k1, 31), thr, done, t_hit, b, pos, wl, cache, cached, m4_below)) return true;
        if (done) return false;
        k0 = 32;
    }
    return k1 >= 32 && decide_span<1>(ph, pl, pa, wv, k0, k1, thr, done, t_hit, b, pos, wl, cache, cached, m4_below);
}

// ---- decide kernel: exact 4-bucket bound + A-parity second level for every (probe, k) of the deferred units ----
template <int MAXNW>
__global__ void __launch_bounds__(kDecideThreads, (MAXNW <= 5 ? 4 : 2)) trew_filter_kernel(DevCfg cfg, DevBatch b, const u32* __restrict__ units,
                                                          const u32* __restrict__ n_units_ptr, u32 n_units_all,
                                                          u32* __restrict__ survivors, u32* __restrict__ n_survivors,
                                                          u32* __restrict__ surv_b_top, u32* __restrict__ n_surv_b, int thread_min_windows, int third_level,   // third_level: asked for periods with fewer valid windows than this
                                                          u32* __restrict__ work_counter) {
    __shared__ unsigned short thr[kThrTableSize];
    __shared__ u32 s_m4[18 * kDecideThreads];   // mod4_level: the probe's prefix planes, per thread
    for (int i = threadIdx.x; i < kThrTableSize; i += blockDim.x) thr[i] = cfg.thr_low[i];
    __syncthreads();
    const u32 n_units = units ? *n_units_ptr : n_units_all;   // no list: every unit of the batch
    const bool pack_probes = n_units_all < (1u << kProbeShift);
    // Lane-level work queue.  A probe is ~2 400 instructions; most units have one flagged probe (the half an N fell into),
    // some two or three, repeats leave their first after two periods.  With a unit per lane and round the few lanes with a
    // second probe cost the warp a whole pass (ncu: 18 of 32 lanes in the period loop).  Instead every round each lane
    // decides ONE probe; a lane whose unit is done hands it in and takes the next unit from the shared counter, so the
    // warp keeps 32 probes in flight until the list is empty.
    const u32 lane = lane_id();
    bool have = false, maybe = false, exhausted = false;
    u32 u = 0, live = 0, todo = 0;
    int t_hit = 1 << 20;
    Probe p[4];
    for (;;) {
        const u32 idle = __ballot_sync(0xffffffffu, !have);
        if (idle != 0u && !exhausted) {
            u32 base = 0;
            if (lane == 0) base = atomicAdd(work_counter, (u32)__popc(idle));
            base = __shfl_sync(0xffffffffu, base, 0);
            exhausted = base + (u32)__popc(idle) >= n_units;
            const u32 i = base + (u32)__popc(idle & ((1u << lane) - 1u));
            if (!have && i < n_units) {
                u32 pm = 0xfu;
                u = i;
                if (units) { const u32 e = units[i]; u = e & ((1u << kProbeShift) - 1u); pm = e >> kProbeShift; }
                const int np = unit_probes(cfg, b, u, p);
                live = todo = pm & ((1u << np) - 1u);   // live: probes that may still find a target period
                maybe = false; t_hit = 1 << 20; have = true;
            }
        }
        if (__ballot_sync(0xffffffffu, have) == 0u) break;
        if (have && todo != 0u) {
            const int j = __ffs(todo) - 1;
            todo &= todo - 1u;
            if (p[j].k1 >= p[j].k0)
                maybe = probe_is_fast(p[j]) ? decide_short(b, p[j].pos, p[j].wl, p[j].k0, p[j].k1, thr, t_hit, s_m4 + threadIdx.x, third_level)
                                            : probe_dispatch<MAXNW>(b, p[j], thr);
            if (!maybe) live &= ~(1u << j);
        }
        const bool fin = have && (todo == 0u || maybe);
        const bool keep = fin && maybe;
        // the exact kernel skips the scan of a window no probe vouches for (its result is "no target period")
        const u32 entry = pack_probes ? u | (live << kProbeShift) : u;
        if (surv_b_top == nullptr) {
            list_append(keep, entry, survivors, n_survivors);
        } else {
            // Two lists for the two exact kernels (short and paired mode).  Up from the bottom of the survivor array: reads
            // the thread-per-survivor kernel takes -- at most 160 bases, and the period that made them survivors still
            // has most of its windows (a repeat).  Down from the top: the others, above all reads an N made survivors of
            // (a period the N leaves a dozen windows of passes the bound easily; turning those away means comparing
            // many one-window runs -- long, lane-divergent loops in the thread kernel, a few warp-wide instructions in the
            // warp kernel's comp_bound).  Both kernels are exact for every read; the split only places the work.
            bool to_b = false;
            if (keep) {
                int len;
                if (cfg.mode == 1) {
                    const u32 a0 = __ldg(b.bit_off + 2 * u), a1 = __ldg(b.bit_off + 2 * u + 1), a2 = __ldg(b.bit_off + 2 * u + 2);
                    len = (int)max(a1 - a0, a2 - a1);
                } else {
                    len = (int)(__ldg(b.bit_off + u + 1) - __ldg(b.bit_off + u));
                }
                to_b = len > et::kMaxRead || t_hit < thread_min_windows;
            }
            list_append(keep && !to_b, entry, survivors, n_survivors);
            list_append_rev(keep && to_b, entry, surv_b_top, n_surv_b);
        }
        if (fin) have = false;
    }
}

void launch_filter(const DevCfg& cfg, const DevBatch& b, unsigned int n_units, unsigned int max_read_len,
                   unsigned int* deferred, unsigned int* n_deferred, unsigned int* survivors, unsigned int* n_survivors,
                   const LaunchPlan& plan, cudaStream_t stream, cudaEvent_t after_screen, unsigned int* surv_b_top,
                   unsigned int* n_surv_b, unsigned int* work_counter) {
    if (n_units == 0) return;
    // longest probe window: a half read, a whole read (n < 4*MAX) or a slice (long mode)
    unsigned int longest;
    if (cfg.mode == 2) longest = 2u * (unsigned)cfg.slice_len;
    else longest = (max_read_len < 4u * (unsigned)cfg.max_mer) ? max_read_len : (max_read_len + 1) / 2;
    unsigned int need = (n_units + 255) / 256;
    // the screen handles windows of at most 159 bases; long-mode slices longer than that all go to the decide kernel
    const bool screen = deferred != nullptr && !(cfg.mode == 2 && cfg.slice_len > kFastMaxWlLong) && n_units < (1u << kProbeShift);
    if (screen) {
        int blocks = plan.screen_blocks;
        if ((unsigned)blocks > need) blocks = (int)need;
        if (longest <= (unsigned)kFastMaxWl) trew_screen_kernel<false><<<blocks, 256, 0, stream>>>(cfg, b, n_units, deferred, n_deferred);
        else trew_screen_kernel<true><<<blocks, 256, 0, stream>>>(cfg, b, n_units, deferred, n_deferred);
    }
    if (after_screen) cudaEventRecord(after_screen, stream);
    static const int tmw = [] { const char* e = getenv("TREW_THREAD_MIN_WINDOWS"); return e && *e ? atoi(e) : kThreadMinWindows; }();   // experiments
    static const int m4_on = [] { const char* e = getenv("TREW_MOD4_BELOW"); return e && *e ? atoi(e) : kMod4BelowWindows; }();   // experiments (0: no third level)
    const unsigned int* list = screen ? deferred : nullptr;
    int blocks = plan.decide_blocks;
    if ((unsigned)blocks > need) blocks = (int)need;
    if (longest + 1 <= 96) trew_filter_kernel<3><<<blocks, 256, 0, stream>>>(cfg, b, list, n_deferred, n_units, survivors, n_survivors, surv_b_top, n_surv_b, tmw, m4_on, work_counter);
    else if (longest + 1 <= 160) trew_filter_kernel<5><<<blocks, 256, 0, stream>>>(cfg, b, list, n_deferred, n_units, survivors, n_survivors, surv_b_top, n_surv_b, tmw, m4_on, work_counter);
    else trew_filter_kernel<8><<<blocks, 256, 0, stream>>>(cfg, b, list, n_deferred, n_units, survivors, n_survivors, surv_b_top, n_surv_b, tmw, m4_on, work_counter);
}

// ------------------------------------------------------------------------------------------------
// exact kernel: warp per survivor unit
// ------------------------------------------------------------------------------------------------
//
// Per-warp shared-memory region (all state a warp needs between its building blocks lives here, addressed from
// the kernel's dynamic shared-memory base so every access is a shared-space LDS/STS):
//   header (16 words)  | planes H L V PH PL (36 words each, word j owned by lane j) | rev2 (36 x u64)
//   run_lo / run_hi (u64[cap])  | htab (u32[hs])  | grp_tot / grp_last (u32[cap])
//   run_start (u16[cap]) | run_cw (u16[cap + 4]) | run_total (u16[cap])

extern __shared__ __align__(16) unsigned char g_smem[];

constexpr int kPlaneWords = 36;  // 32 window words + zero padding for shifted reads
#ifndef TREW_EXACT_BPS
#define TREW_EXACT_BPS 8   // resident exact-kernel blocks per SM the register budget allows
#endif
#ifndef TREW_EXACT_WARPS
#define TREW_EXACT_WARPS 4
#endif
constexpr int kExactWarps = TREW_EXACT_WARPS;
constexpr u32 kEmptySlot = 0xffffffffu;
constexpr int kSerialMaxRuns = 12;   // eval_k: windows with at most this many match-bit runs take the collective-free path

// header words.  12..27: the state of one scan_stats() call -- warp-uniform, so it lives here once instead of in
// every lane's registers (which the calls into eval_k would spill to local memory)
enum { HD_CUR_POS = 0, HD_CUR_LEN, HD_ALLVALID, HD_EV_POS, HD_EV_LEN, HD_EV_K, HD_EV_PACK, HD_UNIT = 7 /* the survivor's unit index in the batch */,
       HD_S = 8 /* 4 words: s_lo, s_hi */,
       HD_BLK_L = 12 /* 2 words */, HD_BLK_H = 14 /* 2 words */, HD_NEED_L = 16, HD_NEED_H = 17, HD_BLK64 = 18, HD_RES = 19,
       HD_SH = 20 /* 4 words */, HD_SL = 24 /* 4 words */, HD_UNIT_BASE = 28 /* 2 words: ordinal of the batch's unit 0 */,
       HD_RECS = 30 /* 2 words: UnitRecs*, 0 = no records */ };
constexpr int kHeaderBytes = 128;

__host__ __device__ inline int exact_hash_slots(int cap) {
    int hs = 64;
    while (hs < cap + cap / 4) hs <<= 1;
    return hs;
}

__host__ __device__ inline size_t exact_warp_bytes(int cap) {
    size_t b = kHeaderBytes + 5 * kPlaneWords * sizeof(u32) + kPlaneWords * sizeof(u64);
    b += (size_t)2 * cap * sizeof(u64) + (size_t)exact_hash_slots(cap) * sizeof(u32) + (size_t)2 * cap * sizeof(u32);
    b += (size_t)(3 * cap + 4) * sizeof(unsigned short);
    return (b + 15) & ~(size_t)15;
}

size_t exact_smem_bytes(int run_cap, bool) { return exact_warp_bytes(run_cap) * kExactWarps; }

struct WS {  // this warp's region
    u32 off; int cap; int hs; u32 lane; u32 flags;
    __device__ __forceinline__ u32* hdr() const { return (u32*)(g_smem + off); }
    __device__ __forceinline__ u32* H() const { return (u32*)(g_smem + off + kHeaderBytes); }
    __device__ __forceinline__ u32* L() const { return H() + kPlaneWords; }
    __device__ __forceinline__ u32* V() const { return H() + 2 * kPlaneWords; }
    __device__ __forceinline__ u32* PH() const { return H() + 3 * kPlaneWords; }
    __device__ __forceinline__ u32* PL() const { return H() + 4 * kPlaneWords; }
    __device__ __forceinline__ u64* rev2() const { return (u64*)(H() + 5 * kPlaneWords); }
    __device__ __forceinline__ u64* run_lo() const { return rev2() + kPlaneWords; }
    __device__ __forceinline__ u64* run_hi() const { return run_lo() + cap; }
    __device__ __forceinline__ u32* htab() const { return (u32*)(run_hi() + cap); }
    __device__ __forceinline__ u32* grp_tot() const { return htab() + hs; }
    __device__ __forceinline__ u32* grp_last() const { return grp_tot() + cap; }
    __device__ __forceinline__ unsigned short* run_start() const { return (unsigned short*)(grp_last() + cap); }
    __device__ __forceinline__ unsigned short* run_cw() const { return run_start() + cap; }
    __device__ __forceinline__ unsigned short* run_total() const { return run_cw() + cap + 4; }
};

struct TableRef { Slot* slots; u32 mask; u32* err; };

struct ScanRes { int th, tl; u64 sh_lo, sh_hi, sl_lo, sl_hi; };

// packed result of eval_k: T (bits 0-9), M (10-19), number of runs (20-29), homopolymer flag (30)
__device__ __forceinline__ int pk_T(u32 p) { return (int)(p & 1023u); }
__device__ __forceinline__ int pk_M(u32 p) { return (int)((p >> 10) & 1023u); }
__device__ __forceinline__ int pk_runs(u32 p) { return (int)((p >> 20) & 1023u); }
__device__ __forceinline__ bool pk_homo(u32 p) { return ((p >> 30) & 1u) != 0; }

// ---- k-mer arithmetic (src/kmer.cpp:39-74, 1815-1867) ------------------------------------------

__device__ __noinline__ u64 canon64(u64 w, int k) {
    int sh = 2 * (k - 1);
    if (k <= 16) {  // the k-mer fits 32 bits: a third of the instructions per rotation step
        u32 b32 = (u32)w, c32 = (u32)w;
        for (int r = 1; r < k; r++) {
            c32 = ((c32 & 3u) << sh) | (c32 >> 2);
            b32 = min(b32, c32);
        }
        return b32;
    }
    u64 best = w, cur = w;
    for (int r = 1; r < k; r++) {
        cur = ((cur & 3ULL) << sh) | (cur >> 2);
        best = cur < best ? cur : best;
    }
    return best;
}

__device__ __noinline__ u128 canon128(u128 w, int k) {
    u128 best = w, cur = w;
    int sh = 2 * (k - 1);
    for (int r = 1; r < k; r++) {
        cur = ((cur & 3) << sh) | (cur >> 2);
        best = cur < best ? cur : best;
    }
    return best;
}

__device__ __forceinline__ u64 rev_pairs64(u64 x) {  // reverse the order of the 32 two-bit symbols
    x = __brevll(x);
    return ((x >> 1) & 0x5555555555555555ULL) | ((x & 0x5555555555555555ULL) << 1);
}

__device__ __forceinline__ void canon_pair(u64& lo, u64& hi, int k) {
    if (k <= 32) { lo = canon64(lo, k); hi = 0; }
    else { u128 c = canon128(((u128)hi << 64) | lo, k); lo = (u64)c; hi = (u64)(c >> 64); }
}

// canonical rotation of the reverse complement (rot_reverse_complement, src/kmer.cpp:72-74)
__device__ __forceinline__ void crc_pair(u64& lo, u64& hi, int k) {
    if (k <= 32) {
        u64 r = ~rev_pairs64(lo) >> (64 - 2 * k);
        lo = canon64(r, k); hi = 0;
    } else {
        u128 r = ((u128)(~rev_pairs64(lo)) << 64) | (u128)(~rev_pairs64(hi));
        r >>= (128 - 2 * k);
        u128 c = canon128(r, k); lo = (u64)c; hi = (u64)(c >> 64);
    }
}

__device__ __forceinline__ bool homo_pair(u64 lo, u64 hi, int k) {  // get_repeat_check: <= 1 distinct base
    if (k <= 1) return true;
    if (k <= 32) return ((lo ^ (lo >> 2)) & ((1ULL << (2 * (k - 1))) - 1ULL)) == 0;
    u128 w = ((u128)hi << 64) | lo;
    u128 m = (((u128)1 << (2 * (k - 1))) - 1);
    return ((w ^ (w >> 2)) & m) == 0;
}

__device__ __forceinline__ bool less_pair(u64 alo, u64 ahi, u64 blo, u64 bhi) {
    return ahi < bhi || (ahi == bhi && alo < blo);
}

__device__ __forceinline__ u32 shfl_next_bit0(u32 x, u32 lane) {  // bit 0 of the next lane's word (0 for lane 31)
    u32 nx = __shfl_down_sync(0xffffffffu, x, 1);
    return lane == 31 ? 0u : (nx & 1u);
}

// ---- window loading --------------------------------------------------------------------------------

// load window [pos, pos+len) of the batch planes; builds prefix-XOR planes and the reversed 2-bit stream
__device__ __noinline__ void load_window(WS ws, const u32* __restrict__ bhi, const u32* __restrict__ blo,
                                         const u32* __restrict__ bval, u32 pos, int len) {
    u32* hd = ws.hdr();
    if ((int)hd[HD_CUR_LEN] == len && hd[HD_CUR_POS] == pos) return;
    __syncwarp();
    const u32 lane = ws.lane;
    int vbits = len - 32 * (int)lane;
    u32 msk = vbits <= 0 ? 0u : low_mask(vbits);
    u32 h = 0, l = 0, v = 0;
    if (vbits > 0) {
        u32 wi = (pos >> 5) + lane, sh = pos & 31;
        h = __funnelshift_r(__ldg(bhi + wi), __ldg(bhi + wi + 1), sh) & msk;
        l = __funnelshift_r(__ldg(blo + wi), __ldg(blo + wi + 1), sh) & msk;
        v = __funnelshift_r(__ldg(bval + wi), __ldg(bval + wi + 1), sh) & msk;
    }
    const bool all_valid = __all_sync(0xffffffffu, v == msk);
    // exclusive prefix-XOR planes, word j in lane j (len + 1 <= 1024 entries)
    u32 ih = prefix_xor32(h), il = prefix_xor32(l);
    u32 bh = __ballot_sync(0xffffffffu, ih >> 31), bl = __ballot_sync(0xffffffffu, il >> 31);
    u32 lt = (1u << lane) - 1u;
    if (__popc(bh & lt) & 1) ih = ~ih;
    if (__popc(bl & lt) & 1) il = ~il;
    u32 ph_prev = __shfl_up_sync(0xffffffffu, ih, 1), pl_prev = __shfl_up_sync(0xffffffffu, il, 1);
    u32 ph = (ih << 1) | (lane ? ph_prev >> 31 : 0u);
    u32 pl = (il << 1) | (lane ? pl_prev >> 31 : 0u);
    u32 *H = ws.H(), *L = ws.L(), *V = ws.V(), *PH = ws.PH(), *PL = ws.PL();
    u64* rev2 = ws.rev2();
    H[lane] = h; L[lane] = l; V[lane] = v; PH[lane] = ph; PL[lane] = pl;
    if (lane < kPlaneWords - 32) {
        H[32 + lane] = 0; L[32 + lane] = 0; V[32 + lane] = 0; PH[32 + lane] = 0; PL[32 + lane] = 0;
        rev2[32 + lane] = 0;
    }
    __syncwarp();
    // reversed interleaved stream: 64-bit word j covers reversed positions [32j, 32j+32), i.e. original
    // bases cs .. cs+31 with cs = len - 32j - 32, highest base first (so a k-mer read from it has its
    // first base in the most significant bits, like the reference's shift-in order, src/kmer.cpp:2186-2189)
    {
        int cs = len - 32 * (int)lane - 32;
        u32 hb = 0, lb = 0;
        if (cs > -32) {
            if (cs >= 0) {
                int wi = cs >> 5, sh = cs & 31;
                hb = __funnelshift_r(H[wi], H[wi + 1], sh);
                lb = __funnelshift_r(L[wi], L[wi + 1], sh);
            } else {
                hb = H[0] << (-cs);
                lb = L[0] << (-cs);
            }
        }
        hb = __brev(hb); lb = __brev(lb);
        u64 x = hb, y = lb;
        x = (x | (x << 16)) & 0x0000FFFF0000FFFFULL; y = (y | (y << 16)) & 0x0000FFFF0000FFFFULL;
        x = (x | (x << 8)) & 0x00FF00FF00FF00FFULL;  y = (y | (y << 8)) & 0x00FF00FF00FF00FFULL;
        x = (x | (x << 4)) & 0x0F0F0F0F0F0F0F0FULL;  y = (y | (y << 4)) & 0x0F0F0F0F0F0F0F0FULL;
        x = (x | (x << 2)) & 0x3333333333333333ULL;  y = (y | (y << 2)) & 0x3333333333333333ULL;
        x = (x | (x << 1)) & 0x5555555555555555ULL;  y = (y | (y << 1)) & 0x5555555555555555ULL;
        rev2[lane] = (x << 1) | y;
    }
    if (lane == 0) { hd[HD_CUR_POS] = pos; hd[HD_CUR_LEN] = (u32)len; hd[HD_ALLVALID] = all_valid ? 1u : 0u; }
    __syncwarp();
}

// k-mer starting at base i of the loaded window (first base most significant)
__device__ __forceinline__ void kmer_at(const u64* __restrict__ rev2, int len, int i, int k, u64& lo, u64& hi) {
    int o = 2 * (len - i - k);
    int wi = o >> 6, sh = o & 63;
    u64 a = rev2[wi], b = rev2[wi + 1];
    lo = sh ? (a >> sh) | (b << (64 - sh)) : a;
    if (k <= 32) {
        if (k < 32) lo &= (1ULL << (2 * k)) - 1ULL;
        hi = 0;
    } else {
        u64 c = rev2[wi + 2];
        hi = sh ? (b >> sh) | (c << (64 - sh)) : b;
        if (k < 64) hi &= (1ULL << (2 * k - 64)) - 1ULL;
    }
}

// this lane's window-valid word for period k: bit i of word j set iff bases 32j+i .. 32j+i+k-1 are all valid
__device__ __forceinline__ u32 wv_for_k(WS ws, int len, int k) {
    const u32 lane = ws.lane;
    if (ws.hdr()[HD_ALLVALID]) {
        int vb = len - k + 1 - 32 * (int)lane;
        return vb <= 0 ? 0u : low_mask(min(32, vb));
    }
    u32 wv = ws.V()[lane];
    for (int t = 1; t < k; t++) {
        u32 nb = shfl_next_bit0(wv, lane);
        wv &= (wv >> 1) | (nb << 31);
    }
    return wv;
}

__device__ __forceinline__ u32 wv_step(u32 wv, u32 lane) {
    u32 nb = shfl_next_bit0(wv, lane);
    return wv & ((wv >> 1) | (nb << 31));
}

// upper bound on the largest class count for period k from the 4-bucket parity signature (warp-cooperative)
__device__ __forceinline__ int bound_k(WS ws, int k, u32 wv, int T) {
    const u32 lane = ws.lane;
    const u32 *PH = ws.PH(), *PL = ws.PL();
    int s = k >> 5, r = k & 31;
    u32 qh = __funnelshift_r(PH[lane + s], PH[lane + s + 1], r);
    u32 ql = __funnelshift_r(PL[lane + s], PL[lane + s + 1], r);
    u32 dh = (qh ^ PH[lane]) & wv, dl = (ql ^ PL[lane]) & wv;
    u32 packed = (u32)__popc(dh) | ((u32)__popc(dl) << 10) | ((u32)__popc(dh & dl) << 20);
    packed = __reduce_add_sync(0xffffffffu, packed);
    int cH = packed & 1023, cL = (packed >> 10) & 1023, c11 = packed >> 20;
    int c10 = cH - c11, c01 = cL - c11, c00 = T - cH - cL + c11;
    return max(max(c00, c01), max(c10, c11));
}

// Second upper bound on the largest class count, for periods with at most 32 valid windows (what an N leaves of a
// window at large k): rotation keeps the multiset of bases, so windows of one class have the same (#C|A, #G|A, #A)
// composition.  One window per lane, equal compositions counted with MATCH.  Exact compositions reject nearly every
// such period of a non-repeat read, where the parity signature (8 buckets for a dozen windows) cannot.
// Uses run_start as scratch (emit_classes does not read it).
__device__ __noinline__ int comp_bound(WS ws, int k, u32 wv, int T) {
    const u32 lane = ws.lane;
    const u32 cnt = (u32)__popc(wv);
    u32 inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, inc, d);
        if ((int)lane >= d) inc += t;
    }
    unsigned short* pos = ws.run_start();
    {
        u32 rb = inc - cnt, x = wv;
        while (x) {
            int bit = __ffs(x) - 1;
            x &= x - 1;
            pos[rb++] = (unsigned short)(32 * lane + bit);
        }
    }
    __syncwarp();
    const bool act = (int)lane < T;
    u32 key = 0;
    if (act) {
        const u32 *H = ws.H(), *L = ws.L();
        const int p = pos[lane], w0 = p >> 5, o = p & 31;
        const u32 m0 = low_mask(min(k, 32)), m1 = k <= 32 ? 0u : low_mask(k - 32);
        const u32 h0 = __funnelshift_r(H[w0], H[w0 + 1], o) & m0, h1 = __funnelshift_r(H[w0 + 1], H[w0 + 2], o) & m1;
        const u32 l0 = __funnelshift_r(L[w0], L[w0 + 1], o) & m0, l1 = __funnelshift_r(L[w0 + 1], L[w0 + 2], o) & m1;
        key = (u32)(__popc(h0) + __popc(h1)) | ((u32)(__popc(l0) + __popc(l1)) << 8) | ((u32)(__popc(h0 & l0) + __popc(h1 & l1)) << 16);
    }
    const u32 actm = __ballot_sync(0xffffffffu, act);
    const u32 same = __match_any_sync(0xffffffffu, key) & actm;
    const u32 best = __reduce_max_sync(0xffffffffu, act ? (u32)__popc(same) : 0u);
    __syncwarp();
    return (int)best;
}

// Exact class statistics of the loaded window for one period (the inner loops of k_mer_check,
// src/kmer.cpp:2183-2216, without the early break): T valid windows, M largest class, S the class that
// first reaches M (stored in the header).  Leaves the run list in shared memory (run_lo/hi canonical class
// per run, run_total = class total on one run of each class, 0 on the others) for emit_classes().
__device__ __noinline__ u32 eval_k(WS ws, int len, int k, u32 wv) {
    const u32 lane = ws.lane;
    u32* hd = ws.hdr();
    const u32 *H = ws.H(), *L = ws.L();
    // link bits: windows i and i+1 are both valid and base[i] == base[i+k]   (Lemma L1)
    int s = k >> 5, r = k & 31;
    u32 hs = __funnelshift_r(H[lane + s], H[lane + s + 1], r);
    u32 ls = __funnelshift_r(L[lane + s], L[lane + s + 1], r);
    u32 eq = ~((hs ^ H[lane]) | (ls ^ L[lane]));
    u32 nb = shfl_next_bit0(wv, lane);
    u32 link = eq & wv & ((wv >> 1) | (nb << 31));
    u32 link_prev = __shfl_up_sync(0xffffffffu, link, 1);
    u32 rs = wv & ~((link << 1) | (lane ? link_prev >> 31 : 0u));  // run starts
    u32 pk = (u32)__popc(wv) | ((u32)__popc(rs) << 16);
    const u32 tot_pk = __reduce_add_sync(0xffffffffu, pk);
    const int T = (int)(tot_pk & 0xffffu), R = (int)(tot_pk >> 16);
    if (T == 0) return 0u;
    unsigned short *run_start = ws.run_start(), *run_cw = ws.run_cw(), *run_total = ws.run_total();
    u64 *run_lo = ws.run_lo(), *run_hi = ws.run_hi();
    u32 *htab = ws.htab(), *grp_tot = ws.grp_tot(), *grp_last = ws.grp_last();
    const u64* rev2 = ws.rev2();
    const bool wide = k > 32;
    if (!wide && R <= kSerialMaxRuns && (ws.flags & 1u)) {   // off by default: measured slower than the general path below (DESIGN.md)
        // Few runs (every repeat read: a perfect repeat is one run, each substitution adds at most two).  The warp
        // collectives of the general path below (prefix scans, shared-memory atomics, reductions) cost more latency
        // than the work they spread, so here every lane walks the runs redundantly in plain ALU / shared-memory
        // instructions: the three mask words per lane go to shared memory once, then run by run -- end of the run,
        // minimal rotation of its first k-mer, linear search in the class list.  Classes land in run_lo / run_total
        // (entries 0 .. classes-1), which is what emit_classes() reads.
        u32* scr = htab;                       // [wv | link | run starts], 32 words each (htab + grp_tot + grp_last: >= 96 words)
        scr[lane] = wv; scr[32 + lane] = link; scr[64 + lane] = rs;
        __syncwarp();
        unsigned short* cls_last = run_cw;     // ordinal of the class's last window
        int ncls = 0, ord = 0;
        const int nw = (len + 31) >> 5;
        for (int j = 0; j < nw; j++) {
            const u32 wvj = scr[j];
            u32 rr = scr[64 + j];
            while (rr) {
                const int b = __ffs(rr) - 1;
                rr &= rr - 1;
                const int c0 = ord + __popc(wvj & ((1u << b) - 1u));
                // the run ends at the first window without a link to its successor
                int jj = j;
                u32 x = ~scr[32 + j] & (0xffffffffu << b);
                while (!x) { jj++; x = ~scr[32 + jj]; }     // lanes past the window hold wv = 0, hence link = 0: terminates
                const int cnt = 32 * (jj - j) + (__ffs(x) - 1) - b + 1;
                u64 lo, hi;
                kmer_at(rev2, len, 32 * j + b, k, lo, hi);
                lo = canon64(lo, k);
                int q = 0;
                while (q < ncls && run_lo[q] != lo) q++;
                u32 tot = (u32)cnt;
                if (q == ncls) { ncls++; run_lo[q] = lo; }
                else tot += run_total[q];
                run_total[q] = (unsigned short)tot;
                cls_last[q] = (unsigned short)(c0 + cnt - 1);
            }
            ord += __popc(wvj);
        }
        // K_MER_DATA_MAX_SEQ: the class whose running count first reaches the final maximum
        // (strict '<' at src/kmer.cpp:2202) = max total, ties broken by the EARLIEST last window
        u32 best = 0; int bq = 0;
        for (int q = 0; q < ncls; q++) {
            const u32 score = ((u32)run_total[q] << 10) | (1023u - cls_last[q]);
            if (score > best) { best = score; bq = q; }
        }
        const u64 s_lo = run_lo[bq];
        const bool homo = homo_pair(s_lo, 0ULL, k);
        __syncwarp();
        if (lane == 0) { hd[HD_S] = (u32)s_lo; hd[HD_S + 1] = (u32)(s_lo >> 32); hd[HD_S + 2] = 0u; hd[HD_S + 3] = 0u; }
        __syncwarp();
        return (u32)T | ((best >> 10) << 10) | ((u32)ncls << 20) | (homo ? 1u << 30 : 0u);
    }
    // exclusive scans over lanes of (valid windows, run starts), packed 16:16
    u32 inc = pk;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, inc, d);
        if ((int)lane >= d) inc += t;
    }
    u32 exc = inc - pk;
    {
        u32 cwb = exc & 0xffffu, rb = exc >> 16;
        u32 x = rs;
        while (x) {
            int bit = __ffs(x) - 1;
            x &= x - 1;
            run_start[rb] = (unsigned short)(32 * lane + bit);
            run_cw[rb] = (unsigned short)(cwb + __popc(wv & ((1u << bit) - 1u)));
            rb++;
        }
        if (lane == 0) run_cw[R] = (unsigned short)T;
    }
    // hash table sized to the run count (power of two >= 1.5 R, so hsz > R; at most hs >= 1.25 cap)
    int hsz = 32;
    while (hsz < R + (R >> 1) && hsz < ws.hs) hsz <<= 1;
    const u32 hmask = (u32)hsz - 1u;
    for (int i = lane; i < hsz; i += 32) {
        htab[i] = kEmptySlot;
        if (i < R) { grp_tot[i] = 0u; grp_last[i] = 0u; }
    }
    __syncwarp();
    // one canonicalisation per run
    for (int q = lane; q < R; q += 32) {
        u64 lo, hi;
        kmer_at(rev2, len, run_start[q], k, lo, hi);
        canon_pair(lo, hi, k);
        run_lo[q] = lo; if (wide) run_hi[q] = hi;
    }
    __syncwarp();
    // group runs of the same class through the hash table: the first run to claim a slot leads its class and
    // collects the class's window total and the ordinal of its last window
    for (int q = lane; q < R; q += 32) {
        u64 lo = run_lo[q], hi = wide ? run_hi[q] : 0ULL;
        u32 hsh = (u32)lo ^ (u32)(lo >> 32) ^ (u32)hi ^ (u32)(hi >> 32);
        u32 slot = (hsh * 0x9e3779b1u) >> 7 & hmask;
        int leader;
        for (;;) {
            u32 old = atomicCAS(&htab[slot], kEmptySlot, (u32)q);
            if (old == kEmptySlot) { leader = q; break; }
            if (run_lo[old] == lo && (!wide || run_hi[old] == hi)) { leader = (int)old; break; }
            slot = (slot + 1) & hmask;
        }
        u32 c0 = run_cw[q], c1 = run_cw[q + 1];
        atomicAdd(&grp_tot[leader], c1 - c0);
        atomicMax(&grp_last[leader], c1 - 1u);
    }
    __syncwarp();
    u32 best = 0; int best_q = -1;
    for (int q = lane; q < R; q += 32) {
        u32 total = grp_tot[q];
        run_total[q] = (unsigned short)total;
        if (total) {
            // K_MER_DATA_MAX_SEQ: the class whose running count first reaches the final maximum
            // (strict '<' at src/kmer.cpp:2202) = max total, ties broken by the EARLIEST last window
            u32 score = (total << 10) | (1023u - grp_last[q]);
            if (score > best) { best = score; best_q = q; }
        }
    }
    u32 wbest = __reduce_max_sync(0xffffffffu, best);
    u32 who = __ballot_sync(0xffffffffu, best == wbest && best_q >= 0);
    int bq = __shfl_sync(0xffffffffu, best_q, __ffs(who) - 1);
    u64 s_lo = run_lo[bq], s_hi = wide ? run_hi[bq] : 0ULL;
    bool homo = homo_pair(s_lo, s_hi, k);
    u32 packed = (u32)T | ((wbest >> 10) << 10) | ((u32)R << 20) | (homo ? 1u << 30 : 0u);
    if (lane == 0) {
        hd[HD_S] = (u32)s_lo; hd[HD_S + 1] = (u32)(s_lo >> 32); hd[HD_S + 2] = (u32)s_hi; hd[HD_S + 3] = (u32)(s_hi >> 32);
    }
    __syncwarp();
    return packed;
}

__device__ __forceinline__ void eval_S(WS ws, u64& lo, u64& hi) {
    const u32* hd = ws.hdr();
    lo = (u64)hd[HD_S] | ((u64)hd[HD_S + 1] << 32);
    hi = (u64)hd[HD_S + 2] | ((u64)hd[HD_S + 3] << 32);
}

// add every distinct class of the last eval_k() to a result table (optionally RC-folded); REC: and record them for the
// survivor's unit (the kernel's instantiation with records)
template <bool REC>
__device__ __noinline__ void emit_classes(TableRef tr, WS ws, int k, int nruns, int table, bool folded) {
    u32 meta = ((u32)table << 8) | (u32)k;
    const unsigned short* run_total = ws.run_total();
    const u64 *run_lo = ws.run_lo(), *run_hi = ws.run_hi();
    for (int q = ws.lane; q < nruns; q += 32) {
        u32 total = run_total[q];
        if (total == 0) continue;
        u64 lo = run_lo[q], hi = k > 32 ? run_hi[q] : 0ULL;
        if (folded) {
            u64 rlo = lo, rhi = hi;
            crc_pair(rlo, rhi, k);
            if (less_pair(rlo, rhi, lo, hi)) { lo = rlo; hi = rhi; }
        }
        table_add_impl(tr.slots, tr.mask, tr.err, meta, lo, hi, (u64)total);
        if constexpr (REC) {
            const u32* hd = ws.hdr();
            UnitRecs* R = reinterpret_cast<UnitRecs*>((u64)hd[HD_RECS] | ((u64)hd[HD_RECS + 1] << 32));
            rec_append(R, ((u64)hd[HD_UNIT_BASE] | ((u64)hd[HD_UNIT_BASE + 1] << 32)) + hd[HD_UNIT], table, k, lo, hi, (u64)total);
        }
    }
    __syncwarp();
}

// multiples of k below 64 as a bit mask (bit j set iff k | j, 0 < j < 64); k = 64 is tracked separately
struct MultTab { u64 m[65]; };
constexpr MultTab make_mult_tab() {
    MultTab t{};
    for (int k = 1; k <= 64; k++) {
        u64 m = 0;
        for (int j = k; j < 64; j += k) m |= 1ULL << j;
        t.m[k] = m;
    }
    return t;
}
__constant__ MultTab c_mult = make_mult_tab();

// k_mer_check / k_mer_check_128 (src/kmer.cpp:2144-2547) without emission: target_k_high / target_k_low and
// the K_MER_DATA_MAX_SEQ of each.  Periods that cannot be accepted by either selection (divisor rule,
// or the signature bound below the running threshold) are skipped without an exact count.
//
// The reference accepts k iff fl(M/T) >= max(B, f_prev) in doubles
// (src/kmer.cpp:2223-2224, 2243-2244).  "fl(M/T) >= B" is "M >= thr_B[T]", thr_B built on the host with the same IEEE
// division (device_ctx.cu:build_thr); "fl(M/T) >= fl(M'/T')" between two ratios with denominators <= 1023 is
// "M * T' >= M' * T" exactly (distinct such ratios differ by > 1e-6, far more than an ulp, and rounding is monotone).
// The pre-test replaces M by its upper bound U in the same two comparisons, so it never rejects a period the
// reference would accept.
// max(baseline, last accepted frequency) of one selection: need = m | t << 16 of the last accepted ratio (0: none yet)
__device__ __forceinline__ int thr_at(const WS& ws, const unsigned short* thr_low, bool high, int T) {
    return (int)__ldg(thr_low + (high ? kThrTableSize : 0) + T);
}
// the exact acceptance test (a table read: only behind an exact evaluation, a few times per survivor)
__device__ __forceinline__ bool need_pass(const WS& ws, const unsigned short* thr_low, bool high, u32 need, int M, int T) {
    const u32 m = need & 0xffffu, t = need >> 16;
    return M >= thr_at(ws, thr_low, high, T) && (t == 0u || (u32)M * t >= m * (u32)T);
}
// the pre-test on an upper bound U of M, without a memory access (it runs for every lane and period): the baseline half
// in doubles with a slack -- fl(M/T) >= B implies M >= B*T*(1 - 2^-53) and U >= M, so "U >= B*T*(1 - 1e-12)" never
// rejects a period the reference accepts -- the ratio half exactly
__device__ __forceinline__ bool need_pre(double B, u32 need, int U, int T) {
    const u32 m = need & 0xffffu, t = need >> 16;
    return (double)U >= B * (double)T * (1.0 - 1e-12) && (t == 0u || (u32)U * t >= m * (u32)T);
}

__device__ __forceinline__ bool blocked_k(const u32* hd, int which /* HD_BLK_L or HD_BLK_H */, int k) {
    if (k >= 64) return (hd[HD_BLK64] >> (which == HD_BLK_H ? 1 : 0)) & 1u;
    return (hd[which + (k >> 5)] >> (k & 31)) & 1u;
}

// one exact evaluation + the two acceptance tests of src/kmer.cpp:2221-2258 for period kk; the selection state is in the
// header.  Returns true when the period was accepted (the thresholds / divisor masks changed).
__device__ __forceinline__ bool try_k(WS ws, const unsigned short* thr_low, double low, double high, u32 pos, int len, int kk, int Uk, int Tk, u32 wv) {
    u32* hd = ws.hdr();
    const bool blkL = blocked_k(hd, HD_BLK_L, kk), blkH = blocked_k(hd, HD_BLK_H, kk);
    if (blkL && blkH) return false;
    const u32 needL = hd[HD_NEED_L], needH = hd[HD_NEED_H];
    bool candL = !blkL && need_pre(low, needL, Uk, Tk), candH = !blkH && need_pre(high, needH, Uk, Tk);
    if (!candL && !candH) return false;
#ifndef TREW_NO_COMP_BOUND
    if (Tk <= 32 && !(ws.flags & 2u)) {   // few windows: the exact-composition bound is cheap and far tighter than the parity signature
        const int Mc = comp_bound(ws, kk, wv, Tk);
        if (Mc < Uk) {
            candL = !blkL && need_pre(low, needL, Mc, Tk); candH = !blkH && need_pre(high, needH, Mc, Tk);
            if (!candL && !candH) return false;
        }
    }
#endif
    const u32 ev = eval_k(ws, len, kk, wv);
    if (ws.lane == 0) { hd[HD_EV_POS] = pos; hd[HD_EV_LEN] = (u32)len; hd[HD_EV_K] = (u32)kk; hd[HD_EV_PACK] = ev; }
    __syncwarp();
    if (pk_homo(ev) || pk_T(ev) == 0) return false;
    const int M = pk_M(ev), T = pk_T(ev);
    const bool accL = !blkL && need_pass(ws, thr_low, false, needL, M, T), accH = !blkH && need_pass(ws, thr_low, true, needH, M, T);
    if (!(accL || accH)) return false;
    if (ws.lane == 0) {
        const u64 mm = c_mult.m[kk];   // multiples of kk below 64
        const u32 m64 = (64 % kk) == 0 ? 1u : 0u;
        const u32 need = (u32)M | ((u32)T << 16);
        u32 res = hd[HD_RES];
        if (accL) {
            hd[HD_NEED_L] = need; hd[HD_BLK_L] |= (u32)mm; hd[HD_BLK_L + 1] |= (u32)(mm >> 32); hd[HD_BLK64] |= m64;
            res = (res & 0xffu) | ((u32)kk << 8);
            hd[HD_SL] = hd[HD_S]; hd[HD_SL + 1] = hd[HD_S + 1]; hd[HD_SL + 2] = hd[HD_S + 2]; hd[HD_SL + 3] = hd[HD_S + 3];
        }
        if (accH) {
            hd[HD_NEED_H] = need; hd[HD_BLK_H] |= (u32)mm; hd[HD_BLK_H + 1] |= (u32)(mm >> 32); hd[HD_BLK64] |= m64 << 1;
            res = (res & 0xff00u) | (u32)kk;
            hd[HD_SH] = hd[HD_S]; hd[HD_SH + 1] = hd[HD_S + 1]; hd[HD_SH + 2] = hd[HD_S + 2]; hd[HD_SH + 3] = hd[HD_S + 3];
        }
        hd[HD_RES] = res;
    }
    __syncwarp();
    return true;
}

// k_mer_check without emission for window [pos, pos + len), periods kmin..kmax: returns target_k_high | target_k_low << 8;
// the K_MER_DATA_MAX_SEQ of the two are left in the header (HD_SH, HD_SL).
__device__ __noinline__ u32 scan_core(WS ws, DevBatch b, u32 pos, int len, int kmin, int kmax, const unsigned short* thr_low, double low,
                                      double high) {
    if (kmax < kmin) return 0u;
    load_window(ws, b.hi, b.lo, b.val, pos, len);
    const u32 lane = ws.lane;
    u32* hd = ws.hdr();
    if (lane >= HD_BLK_L && lane <= HD_SL + 3) hd[lane] = 0u;   // fresh selection state
    __syncwarp();
    const bool all_valid = hd[HD_ALLVALID] != 0;

    if (len <= 127 || all_valid) {
        // Every lane bounds its own period (lane <-> k); the qualifying periods are then visited in ascending order.
        const u32 *PH = ws.PH(), *PL = ws.PL(), *V = ws.V();
        const int nw = (len + 31) >> 5;
        for (int kb = kmin; kb <= kmax; kb += 32) {
            const int k = kb + (int)lane;
            int U = 0, T = 0;
            u32 wvv[4] = {0u, 0u, 0u, 0u};   // this lane's window-valid words (short windows with invalid bases only)
            if (k <= kmax && k <= len) {
                const int s = k >> 5, r = k & 31;
                int cH = 0, cL = 0, c11 = 0;
                if (all_valid) {
                    T = len - k + 1;
                    for (int j = 0; j * 32 < T; j++) {
                        u32 wvj = low_mask(min(32, T - 32 * j));
                        u32 dh = (__funnelshift_r(PH[j + s], PH[j + s + 1], r) ^ PH[j]) & wvj;
                        u32 dl = (__funnelshift_r(PL[j + s], PL[j + s + 1], r) ^ PL[j]) & wvj;
                        cH += __popc(dh); cL += __popc(dl); c11 += __popc(dh & dl);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; j++) wvv[j] = V[j];
                    sliding_and<4>(wvv, k);
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        if (j < nw) {
                            u32 dh = (__funnelshift_r(PH[j + s], PH[j + s + 1], r) ^ PH[j]) & wvv[j];
                            u32 dl = (__funnelshift_r(PL[j + s], PL[j + s + 1], r) ^ PL[j]) & wvv[j];
                            T += __popc(wvv[j]); cH += __popc(dh); cL += __popc(dl); c11 += __popc(dh & dl);
                        }
                    }
                }
                int c10 = cH - c11, c01 = cL - c11, c00 = T - cH - cL + c11;
                U = max(max(c00, c01), max(c10, c11));
            }
            bool cand = T > 0 && need_pre(low, 0u, U, T);
            u32 cm = __ballot_sync(0xffffffffu, cand);
            while (cm) {
                int bit = __ffs(cm) - 1;
                cm &= cm - 1;
                int Uk = __shfl_sync(0xffffffffu, U, bit), Tk = __shfl_sync(0xffffffffu, T, bit);
                u32 wv;
                if (all_valid) {
                    int vb = Tk - 32 * (int)lane;
                    wv = vb <= 0 ? 0u : low_mask(min(32, vb));
                } else {
                    u32 a0 = __shfl_sync(0xffffffffu, wvv[0], bit), a1 = __shfl_sync(0xffffffffu, wvv[1], bit);
                    u32 a2 = __shfl_sync(0xffffffffu, wvv[2], bit), a3 = __shfl_sync(0xffffffffu, wvv[3], bit);
                    wv = lane == 0 ? a0 : lane == 1 ? a1 : lane == 2 ? a2 : lane == 3 ? a3 : 0u;
                }
                if (try_k(ws, thr_low, low, high, pos, len, kb + bit, Uk, Tk, wv) && cm) {
                    // an acceptance raised the thresholds / blocked multiples: drop the remaining periods of
                    // this block that can no longer be accepted by either selection (lane <-> period again)
                    bool still = false;
                    if (T > 0 && k <= 64)
                        still = (!blocked_k(hd, HD_BLK_L, k) && need_pre(low, hd[HD_NEED_L], U, T)) ||
                                (!blocked_k(hd, HD_BLK_H, k) && need_pre(high, hd[HD_NEED_H], U, T));
                    cm &= __ballot_sync(0xffffffffu, still);
                }
            }
        }
        return hd[HD_RES];
    }

    // long windows with invalid bases: walk the periods in order, keeping the window-valid mask incrementally
    u32 wv = wv_for_k(ws, len, kmin);
    for (int k = kmin; k <= kmax; k++, wv = wv_step(wv, lane)) {
        int T = (int)__reduce_add_sync(0xffffffffu, (u32)__popc(wv));
        if (T == 0) break;
        int U = bound_k(ws, k, wv, T);
        try_k(ws, thr_low, low, high, pos, len, k, U, T, wv);
    }
    return hd[HD_RES];
}

// the result of scan_core with the two K_MER_DATA_MAX_SEQ read back from the header (callers that do not look at them --
// short and long routing -- never load them)
__device__ __forceinline__ ScanRes scan_stats(WS ws, const DevBatch& b, u32 pos, int len, int kmin, int kmax, const DevCfg& cfg) {
    const u32 r = scan_core(ws, b, pos, len, kmin, kmax, cfg.thr_low, cfg.low, cfg.high);
    const u32* hd = ws.hdr();
    ScanRes res;
    res.th = (int)(r & 0xffu); res.tl = (int)(r >> 8);
    res.sh_lo = (u64)hd[HD_SH] | ((u64)hd[HD_SH + 1] << 32); res.sh_hi = (u64)hd[HD_SH + 2] | ((u64)hd[HD_SH + 3] << 32);
    res.sl_lo = (u64)hd[HD_SL] | ((u64)hd[HD_SL + 1] << 32); res.sl_hi = (u64)hd[HD_SL + 2] | ((u64)hd[HD_SL + 3] << 32);
    return res;
}

// class statistics + run list of (window, k), re-using the last evaluation when it is the same one
__device__ __noinline__ u32 eval_cached(WS ws, DevBatch b, u32 pos, int len, int k) {
    u32* hd = ws.hdr();
    if ((int)hd[HD_EV_K] == k && hd[HD_EV_POS] == pos && (int)hd[HD_EV_LEN] == len) return hd[HD_EV_PACK];
    load_window(ws, b.hi, b.lo, b.val, pos, len);
    u32 wv = wv_for_k(ws, len, k);
    u32 ev = eval_k(ws, len, k, wv);
    if (ws.lane == 0) { hd[HD_EV_POS] = pos; hd[HD_EV_LEN] = (u32)len; hd[HD_EV_K] = (u32)k; hd[HD_EV_PACK] = ev; }
    __syncwarp();
    return ev;
}

// the emission half of k_mer_check for one target k (src/kmer.cpp:2264-2328): every class, un-folded unless asked
template <bool REC>
__device__ void emit_window(TableRef tr, WS ws, const DevBatch& b, u32 pos, int len, int k, int table, bool folded) {
    u32 ev = eval_cached(ws, b, pos, len, k);
    emit_classes<REC>(tr, ws, k, pk_runs(ev), table, folded);
}

// k_mer_target / k_mer_target_128 (src/kmer.cpp:1894-2142)
template <bool REC>
__device__ void target_window(TableRef tr, WS ws, const DevBatch& b, u32 pos, int len, int k, const unsigned short* thr_low, bool high, int table) {
    u32 ev = eval_cached(ws, b, pos, len, k);
    if (pk_T(ev) > 0 && !pk_homo(ev) && pk_M(ev) >= thr_at(ws, thr_low, high, pk_T(ev))) emit_classes<REC>(tr, ws, k, pk_runs(ev), table, true);
}

// ---- routing -----------------------------------------------------------------------------------

enum { T_F = 0, T_B = 2, T_O = 4 };

// buffer_task (src/kmer.cpp:80-266)
// pm: probes (unit_probes order) the filter kernels could not rule out; the scan of any other window finds nothing
template <bool REC>
__device__ void route_short(const DevCfg& cfg, TableRef tr, WS ws, const DevBatch& b, u32 u, u32 pm) {
    const int MINM = cfg.min_mer, MAXM = cfg.max_mer;
    u32 b0 = __ldg(b.bit_off + u);
    int n = (int)(__ldg(b.bit_off + u + 1) - b0);
    if (n < 2 * MINM || n > kMaxWindow) return;
    int L[2] = {0, 0}, R[2] = {0, 0};
    if (n >= 4 * MINM) {
        int kmax = min(n / 4, MAXM);
        u32 lpos = b0, rpos = b0 + (u32)(n - (n + 1) / 2);
        int llen = n / 2, rlen = (n + 1) / 2;
        if (pm & 1u) { ScanRes l = scan_stats(ws, b, lpos, llen, MINM, kmax, cfg); L[0] = l.th; L[1] = l.tl; }
        if (pm & 2u) { ScanRes r = scan_stats(ws, b, rpos, rlen, MINM, kmax, cfg); R[0] = r.th; R[1] = r.tl; }  // "always evaluated"
        pm >>= 2;
        // right-half emissions survive only for classes where the left half found nothing
        // (nullptr maps at src/kmer.cpp:125, result.backward at :158)
#pragma unroll
        for (int c = 0; c < 2; c++) {
            if (L[c] > 0 && L[c] == R[c]) target_window<REC>(tr, ws, b, b0, n, L[c], cfg.thr_low, c == 0, T_O + c);
            else if (L[c] > 0) emit_window<REC>(tr, ws, b, lpos, llen, L[c], T_F + c, false);
            else if (R[c] > 0) emit_window<REC>(tr, ws, b, rpos, rlen, R[c], T_B + c, false);
        }
    }
    bool hc[2] = {L[0] == 0 && R[0] == 0, L[1] == 0 && R[1] == 0};
    if (4 * MAXM > n && (hc[0] || hc[1]) && (pm & 1u)) {
        ScanRes s = scan_stats(ws, b, b0, n, max(n / 4 + 1, MINM), min(n / 2, MAXM), cfg);
        if (hc[0] && s.th) emit_window<REC>(tr, ws, b, b0, n, s.th, T_O + 0, false);  // un-folded into 'both'
        if (hc[1] && s.tl) emit_window<REC>(tr, ws, b, b0, n, s.tl, T_O + 1, false);
    }
}

// buffer_task_pair (src/kmer.cpp:268-745); follows the 128-bit path where the two differ (temp map cleared
// after the large-k block, src/kmer.cpp:722-723)
template <bool REC>
__device__ void route_pair(const DevCfg& cfg, TableRef tr, WS ws, const DevBatch& b, u32 u) {
    const int MINM = cfg.min_mer, MAXM = cfg.max_mer;
    u32 a0 = __ldg(b.bit_off + 2 * u), a1 = __ldg(b.bit_off + 2 * u + 1), a2 = __ldg(b.bit_off + 2 * u + 2);
    int n1 = (int)(a1 - a0), n2 = (int)(a2 - a1);
    int n = min(n1, n2);
    if (n < 2 * MINM || n1 > kMaxWindow || n2 > kMaxWindow) return;
    int lef[2] = {0, 0}, km[2] = {0, 0};
    if (n >= 4 * MINM) {
        u32 spos[5] = {0, a0, a0 + (u32)(n1 - (n1 + 1) / 2), a1 + (u32)(n2 - (n2 + 1) / 2), a1};
        int slen[5] = {0, n1 / 2, (n1 + 1) / 2, (n2 + 1) / 2, n2 / 2};
        int kmax = min(n / 4, MAXM);
        ScanRes sr[5]; bool have[5] = {false, false, false, false, false};
        // pending emissions per class: segment + temp map id (0 = left, 1 = right)
        int pseg[2][8], ptmp[2][8], np[2] = {0, 0};
        int si[2] = {1, 1}; bool ended[2] = {false, false};
        u64 ks_lo[2] = {0, 0}, ks_hi[2] = {0, 0};
        for (int ti = 1; ti <= 4 && !(ended[0] && ended[1]); ti++) {
            if (!have[ti]) { sr[ti] = scan_stats(ws, b, spos[ti], slen[ti], MINM, kmax, cfg); have[ti] = true; }
            int k[2] = {sr[ti].th, sr[ti].tl};
            u64 slo[2] = {sr[ti].sh_lo, sr[ti].sl_lo}, shi[2] = {sr[ti].sh_hi, sr[ti].sl_hi};
#pragma unroll
            for (int c = 0; c < 2; c++) {
                if (!ended[c] && k[c]) { pseg[c][np[c]] = ti; ptmp[c][np[c]] = ti <= 2 ? 0 : 1; np[c]++; }  // emission before the test
                bool ok = !ended[c] && k[c] > 0;
                if (ok && ti != 1) {
                    u64 dlo = slo[c], dhi = shi[c];
                    if (ti > 2) crc_pair(dlo, dhi, k[c]);  // get_dir_seq, src/kmer.cpp:307-313
                    ok = km[c] == k[c] && ks_lo[c] == dlo && ks_hi[c] == dhi;
                }
                if (ok) { si[c]++; km[c] = k[c]; if (ti == 1) { ks_lo[c] = slo[c]; ks_hi[c] = shi[c]; } }
                else ended[c] = true;
            }
        }
        lef[0] = km[0]; lef[1] = km[1];
#pragma unroll
        for (int c = 0; c < 2; c++) {
            if (si[c] == 5) {
                for (int e = 0; e < np[c]; e++) {
                    int sg = pseg[c][e];
                    emit_window<REC>(tr, ws, b, spos[sg], slen[sg], c == 0 ? sr[sg].th : sr[sg].tl, T_O + c, true);
                }
            }
        }
        if (si[0] <= 4 || si[1] <= 4) {
            int sj[2] = {4, 4}; km[0] = km[1] = 0; ended[0] = ended[1] = false;
            for (int tj = 4; tj >= 1 && !(ended[0] && ended[1]); tj--) {
                if (!have[tj]) { sr[tj] = scan_stats(ws, b, spos[tj], slen[tj], MINM, kmax, cfg); have[tj] = true; }
                int k[2] = {sr[tj].th, sr[tj].tl};
                u64 slo[2] = {sr[tj].sh_lo, sr[tj].sl_lo}, shi[2] = {sr[tj].sh_hi, sr[tj].sl_hi};
#pragma unroll
                for (int c = 0; c < 2; c++) {
                    if (!ended[c] && k[c]) { pseg[c][np[c]] = tj; ptmp[c][np[c]] = tj <= 2 ? 1 : 0; np[c]++; }  // temps swapped
                    bool ok = sj[c] >= si[c] && !ended[c] && k[c] > 0;
                    if (ok && tj != 4) {
                        u64 dlo = slo[c], dhi = shi[c];
                        if (tj <= 2) crc_pair(dlo, dhi, k[c]);
                        ok = km[c] == k[c] && ks_lo[c] == dlo && ks_hi[c] == dhi;
                    }
                    if (ok) { sj[c]--; km[c] = k[c]; if (tj == 4) { ks_lo[c] = slo[c]; ks_hi[c] = shi[c]; } }
                    else ended[c] = true;
                }
            }
        }
#pragma unroll
        for (int c = 0; c < 2; c++) {
            if (si[c] <= 4) {
                for (int e = 0; e < np[c]; e++) {
                    int sg = pseg[c][e];
                    emit_window<REC>(tr, ws, b, spos[sg], slen[sg], c == 0 ? sr[sg].th : sr[sg].tl,
                                (ptmp[c][e] == 0 ? T_F : T_B) + c, false);
                }
            }
        }
    }
    if (4 * MAXM > n && (lef[0] == 0 || lef[1] == 0 || km[0] == 0 || km[1] == 0)) {
        int lo = max(n / 4 + 1, MINM), hi = min(n / 2, MAXM);
        ScanRes l, r; l.th = l.tl = r.th = r.tl = 0; l.sh_lo = l.sh_hi = l.sl_lo = l.sl_hi = 0; r = l;
        if (lef[0] == 0 || lef[1] == 0) l = scan_stats(ws, b, a0, n1, lo, hi, cfg);
        if (km[0] == 0 || km[1] == 0) r = scan_stats(ws, b, a1, n2, lo, hi, cfg);
        int ltk[2] = {l.th, l.tl}, rtk[2] = {r.th, r.tl};
        u64 llo[2] = {l.sh_lo, l.sl_lo}, lhi[2] = {l.sh_hi, l.sl_hi}, rlo[2] = {r.sh_lo, r.sl_lo}, rhi[2] = {r.sh_hi, r.sl_hi};
#pragma unroll
        for (int c = 0; c < 2; c++) {
            bool el = lef[c] == 0 && ltk[c] > 0, er = km[c] == 0 && rtk[c] > 0;  // both land in the 'left' temp map
            bool both = lef[c] == 0 && km[c] == 0 && ltk[c] == rtk[c] && ltk[c] > 0;
            if (both) {
                u64 dlo = rlo[c], dhi = rhi[c];
                crc_pair(dlo, dhi, rtk[c]);
                both = llo[c] == dlo && lhi[c] == dhi;
            }
            if (both) {
                if (el) emit_window<REC>(tr, ws, b, a0, n1, ltk[c], T_O + c, true);
                if (er) emit_window<REC>(tr, ws, b, a1, n2, rtk[c], T_O + c, true);
            }
            if (el) emit_window<REC>(tr, ws, b, a0, n1, ltk[c], T_F + c, false);
            if (er) emit_window<REC>(tr, ws, b, a1, n2, rtk[c], T_F + c, false);
        }
    }
}

// buffer_task_long (src/kmer.cpp:747-985)
template <bool REC>
__device__ void route_long(const DevCfg& cfg, TableRef tr, WS ws, const DevBatch& b, u32 u, unsigned char* scratch) {
    const int MINM = cfg.min_mer, MAXM = cfg.max_mer, SL = cfg.slice_len;
    u32 b0 = __ldg(b.bit_off + u);
    int n = (int)(__ldg(b.bit_off + u + 1) - b0);
    if (n < SL) return;  // the reader drops these (src/kmer.cpp:1184)
    int snum = n / SL, mid = (snum + 1) / 2, bonus = n % SL;
    auto s_start = [&](int t) { return (u32)((t - 1) * SL + (t > mid ? bonus : 0)); };
    auto s_len = [&](int t) { return SL + (t == mid ? bonus : 0); };
    // forward walk, pass 1: statistics only; the destination of its emissions is known at its end
    int si[2] = {1, 1}, km[2] = {0, 0}; bool ended[2] = {false, false};
    int nf = 0;
    for (int ti = 1; ti <= snum && !(ended[0] && ended[1]); ti++) {
        ScanRes sr = scan_stats(ws, b, b0 + s_start(ti), s_len(ti), MINM, MAXM, cfg);
        if (ws.lane == 0) { scratch[2 * (ti - 1)] = (unsigned char)sr.th; scratch[2 * (ti - 1) + 1] = (unsigned char)sr.tl; }
        int k[2] = {sr.th, sr.tl};
#pragma unroll
        for (int c = 0; c < 2; c++) {
            if (!ended[c] && k[c] > 0 && (ti == 1 || km[c] == k[c])) { si[c]++; km[c] = k[c]; }
            else ended[c] = true;
        }
        nf = ti;
    }
    __syncwarp();
    // pass 2: replay the walk and emit into 'both' (folded) when every slice survived, else 'forward'
    {
        bool en[2] = {false, false}; int kk[2] = {0, 0};
        bool full[2] = {si[0] == snum + 1, si[1] == snum + 1};
        for (int ti = 1; ti <= nf; ti++) {
            int k[2] = {scratch[2 * (ti - 1)], scratch[2 * (ti - 1) + 1]};
#pragma unroll
            for (int c = 0; c < 2; c++) {
                if (!en[c] && k[c]) emit_window<REC>(tr, ws, b, b0 + s_start(ti), s_len(ti), k[c], (full[c] ? T_O : T_F) + c, full[c]);
                if (!en[c] && k[c] > 0 && (ti == 1 || kk[c] == k[c])) kk[c] = k[c];
                else en[c] = true;
            }
        }
    }
    if (si[0] <= snum || si[1] <= snum) {
        int sj[2] = {snum, snum}; km[0] = km[1] = 0; ended[0] = ended[1] = false;
        for (int tj = snum; tj >= 1 && !(ended[0] && ended[1]); tj--) {
            ScanRes sr = scan_stats(ws, b, b0 + s_start(tj), s_len(tj), MINM, MAXM, cfg);
            int k[2] = {sr.th, sr.tl};
#pragma unroll
            for (int c = 0; c < 2; c++) {
                if (!ended[c] && k[c]) emit_window<REC>(tr, ws, b, b0 + s_start(tj), s_len(tj), k[c], T_B + c, false);  // straight into 'backward'
                if (sj[c] >= si[c] && !ended[c] && k[c] > 0 && (tj == snum || km[c] == k[c])) { sj[c]--; km[c] = k[c]; }
                else ended[c] = true;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// thread-per-survivor exact kernel (short single-end reads within the limits of exact_thread.cuh)
// ------------------------------------------------------------------------------------------------
//
// One THREAD per survivor: the read's planes in registers, buffer_task as scalar code (exact_thread.cuh, also built
// for the host and diffed against the oracle in tests/test_exact_thread.py).  A survivor outside the limits of that
// path is appended to `hard`; the warp-per-survivor kernel below then takes exactly those.

// Emissions are staged in a per-block shared-memory count table and flushed to the global table once, when the block
// is done: nearly every emission of a batch hits the same handful of keys (TTAGGG and its one-error variants), and
// global atomics to one address retire one at a time in L2 (measured: 2 M all-telomeric survivors cost the same
// 4.7 ms whatever the kernel in front of the atomics does).  Staged, a block adds to shared memory -- 148 SMs in
// parallel -- and sends one global add per distinct key.  A key that finds no free slot within a few probes goes
// straight to the global table (noisy batches: many distinct keys of count 1).
constexpr int kStageSlots = 256;            // per block; 16 bytes each
constexpr int kStageProbes = 6;
constexpr u32 kStageLock = 0xffffffffu;     // s_meta: 0 empty, kStageLock being written, else (meta | 1 << 31) ready

struct StageEmit {
    u32* s_meta; u32* s_cnt; u64* s_key;    // shared
    Slot* slots; u32 mask; u32* err;        // global table
    // 128-bit keys (units above 32 bases): staged when they fit 64 bits (the period is part of the tag), else -- a unit of 33+
    // bases whose first bases are not all T, rarely the same one twice in a block -- straight to the global table
    __device__ __forceinline__ void operator()(int table, int k, et::u128 key, u64 count) const {
        const u64 hi = (u64)(key >> 64);
        if (hi) table_add_impl(slots, mask, err, ((u32)table << 8) | (u32)k, (u64)key, hi, count);
        else (*this)(table, k, (et::u64)key, count);
    }
    __device__ __forceinline__ void operator()(int table, int k, et::u64 key_, u64 count) const {
        const u64 key = (u64)key_;
        const u32 meta = ((u32)table << 8) | (u32)k, tag = meta | 0x80000000u;
        u32 i = (u32)(mix64(key ^ ((u64)meta << 53)) >> 40) & (kStageSlots - 1);
        bool done = false;
        for (int p = 0; p < kStageProbes && !done; p++, i = (i + 1) & (kStageSlots - 1)) {
            int outcome = 0;   // 0 look again (a neighbour is publishing this slot), 1 added, 2 another key lives here
            do {               // same protocol as table_add_impl: no lane waits inside a divergent branch
                const u32 st = atomicCAS(&s_meta[i], 0u, kStageLock);
                if (st == 0u) {
                    s_key[i] = key;
                    __threadfence_block();
                    atomicExch(&s_meta[i], tag);
                    atomicAdd(&s_cnt[i], (u32)count);
                    outcome = 1;
                } else if (st != kStageLock) {
                    __threadfence_block();
                    if (st == tag && *(volatile u64*)&s_key[i] == key) { atomicAdd(&s_cnt[i], (u32)count); outcome = 1; }
                    else outcome = 2;
                }
            } while (outcome == 0);
            done = outcome == 1;
        }
        if (!done) table_add_impl(slots, mask, err, meta, key, 0ULL, count);
    }
};

// StageEmit plus one unit record per emission (the kernels' REC instantiations)
struct RecStageEmit {
    StageEmit add; UnitRecs* recs; u64 unit;
    __device__ __forceinline__ void operator()(int table, int k, et::u128 key, u64 count) const {
        add(table, k, key, count);
        rec_append(recs, unit, table, k, (u64)key, (u64)(key >> 64), count);
    }
    __device__ __forceinline__ void operator()(int table, int k, et::u64 key, u64 count) const {
        add(table, k, key, count);
        rec_append(recs, unit, table, k, (u64)key, 0ULL, count);
    }
};

#ifndef TREW_THREAD_BLOCK
#define TREW_THREAD_BLOCK 128
#endif
template <class K>
constexpr size_t thread_kernel_smem() { return (size_t)et::Lay<K>::WORDS * TREW_THREAD_BLOCK * sizeof(u32) + (size_t)kStageSlots * 16; }
constexpr size_t kThreadKernelSmem = thread_kernel_smem<et::u64>();
// blocks per SM the kernels are built for.  Shared memory would allow 8 (64-bit units: 47 words per thread + the staging
// table = 27.5 KB, + 1 KB the driver reserves per block) or 6 (128-bit units, 59 words); the registers decide.  Short
// reads, 64-bit units: 6 (80 registers); at 7 or 8 (72 / 64 registers) scan_window spills and the kernel is slower
// (B200, 25 M-read batch: 0.589 / 0.613 / 0.641 ms at 6 / 7 / 8).  5 with 128-bit units, one less for the paired routing.
template <int MODE, class K>
constexpr int thread_kernel_bps() { return (sizeof(K) == 8 ? 6 : 5) - (MODE == 1 ? 1 : 0); }

// brings bases [off, off + len) of a read (mate 0 / 1 of a pair) into the thread's workspace as the current window
struct PlaneLoad {
    et::Mem m; const u32 *hi, *lo, *val; u32 b0[2];
    __device__ __forceinline__ void operator()(int mate, int off, int len) const {
        const u32 pos = b0[mate] + (u32)off, w0 = pos >> 5, sh = pos & 31u;
        for (int j = 0; j < et::kReadWords + 2; j++) {
            const u32 msk = low_mask(min(32, max(0, len - 32 * j)));
            u32 h = 0u, l = 0u;
            if (msk) {
                h = __funnelshift_r(__ldg(hi + w0 + j), __ldg(hi + w0 + j + 1), sh) & msk;
                l = __funnelshift_r(__ldg(lo + w0 + j), __ldg(lo + w0 + j + 1), sh) & msk;
            }
            m[et::W_H + j] = h; m[et::W_L + j] = l;
            if (j < et::kReadWords) m[et::W_V + j] = msk ? __funnelshift_r(__ldg(val + w0 + j), __ldg(val + w0 + j + 1), sh) & msk : 0u;
        }
    }
};

// MODE 0 short single-end, 1 paired; K: u64 (MAX_MER <= 32) or u128 (<= 64); REC: one unit record per emission
template <int MODE, class K, bool REC>
__global__ void __launch_bounds__(TREW_THREAD_BLOCK, (thread_kernel_bps<MODE, K>())) trew_exact_thread_kernel(DevCfg cfg, DevBatch b, const u32* __restrict__ survivors,
                                                                              const u32* __restrict__ n_survivors, int packed_probes,
                                                                              u32* __restrict__ hard, u32* __restrict__ n_hard,
                                                                              unsigned long long* total_survivors, u32* work_counter) {
    // word i of thread t's workspace at work[i * blockDim + t]: no bank conflicts
    u32* work = reinterpret_cast<u32*>(g_smem);
    u64* s_key = reinterpret_cast<u64*>(work + et::Lay<K>::WORDS * TREW_THREAD_BLOCK);
    u32* s_meta = reinterpret_cast<u32*>(s_key + kStageSlots);
    u32* s_cnt = s_meta + kStageSlots;
    for (int i = threadIdx.x; i < kStageSlots; i += blockDim.x) { s_meta[i] = 0u; s_cnt[i] = 0u; }
    __syncthreads();
    const et::Mem m{work + threadIdx.x, TREW_THREAD_BLOCK};
    const u32 n = *n_survivors;
    if (blockIdx.x == 0 && threadIdx.x == 0 && total_survivors) atomicAdd(total_survivors, (unsigned long long)n);
    StageEmit emit{s_meta, s_cnt, s_key, cfg.slots, cfg.slot_mask, cfg.error_flag};
    // a warp takes 32 survivors at a time from a shared counter: the cost of a survivor varies by an order of magnitude
    // (a clean repeat against a noisy window), and with one or two rounds per warp a fixed assignment leaves most warps
    // waiting at the final barrier for the unlucky ones
    for (;;) {
        u32 base = 0;
        if (lane_id() == 0) base = atomicAdd(work_counter, 32u);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= n) break;
        const u32 i = base + lane_id();
        bool bail = false;
        u32 entry = 0;
        if (i < n) {
            entry = survivors[i];
            u32 u = entry, pm = 3u;
            if (packed_probes) { pm = entry >> kProbeShift; u &= (1u << kProbeShift) - 1u; }
            auto route = [&](auto& em) {
                if (MODE == 0) {
                    const u32 b0 = __ldg(b.bit_off + u);
                    const int len = (int)(__ldg(b.bit_off + u + 1) - b0);
                    if (len > et::kMaxRead) return false;
                    PlaneLoad load{m, b.hi, b.lo, b.val, {b0, 0u}};
                    return et::route_short_thread<K>(m, len, pm & 7u, cfg.min_mer, cfg.max_mer, cfg.thr_low, cfg.thr_high, load, em);
                }
                const u32 a0 = __ldg(b.bit_off + 2 * u), a1 = __ldg(b.bit_off + 2 * u + 1), a2 = __ldg(b.bit_off + 2 * u + 2);
                const int n1 = (int)(a1 - a0), n2 = (int)(a2 - a1);
                PlaneLoad load{m, b.hi, b.lo, b.val, {a0, a1}};
                return et::route_pair_thread<K>(m, n1, n2, cfg.min_mer, cfg.max_mer, cfg.thr_low, cfg.thr_high, load, em);
            };
            if constexpr (REC) {
                RecStageEmit rem{emit, cfg.recs, cfg.unit_base + u};
                bail = !route(rem);
            } else {
                bail = !route(emit);
            }
        }
        list_append(bail, entry, hard, n_hard);
    }
    // flush the staged counts
    __syncthreads();
    for (int i = threadIdx.x; i < kStageSlots; i += blockDim.x) {
        const u32 st = s_meta[i], c = s_cnt[i];
        if (st != 0u && st != kStageLock && c != 0u) table_add_impl(cfg.slots, cfg.slot_mask, cfg.error_flag, st & 0x7fffffffu, s_key[i], 0ULL, (u64)c);
    }
}

// ---- long reads: the three steps of exact_thread.cuh (long_slice_stats / long_walk / long_emit) as kernels -------------
//
// Survivor idx (at most s_cap of them; the rest goes to the warp kernel) owns row idx of two arrays of max_slices + 1
// entries: stats (u16: target_k_high | target_k_low << 8 per slice) and emis (u32 per slice: one byte per emission --
// forward walk high / low: k | 0x80 when it goes to 'both' folded; backward walk high / low: k).

struct LongArgs {
    const u32* survivors; const u32* n_survivors; int packed_probes;
    u32 s_cap, max_slices;
    unsigned short* stats; u32* emis;
    u32* hard; u32* n_hard;
    unsigned long long* total_survivors;
};

// step 1: warp per survivor, lane per slice
__global__ void __launch_bounds__(TREW_THREAD_BLOCK, 4) trew_long_stats_kernel(DevCfg cfg, DevBatch b, LongArgs a) {
    u32* work = reinterpret_cast<u32*>(g_smem);
    const et::Mem m{work + threadIdx.x, TREW_THREAD_BLOCK};
    const u32 n = min(*a.n_survivors, a.s_cap);
    const u32 warps = gridDim.x * (blockDim.x >> 5), lane = lane_id();
    et::ClsSpill<et::u64> x;
    for (u32 idx = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); idx < n; idx += warps) {
        u32 u = a.survivors[idx];
        if (a.packed_probes) u &= (1u << kProbeShift) - 1u;
        const u32 b0 = __ldg(b.bit_off + u);
        const int len = (int)(__ldg(b.bit_off + u + 1) - b0);
        if (len < cfg.slice_len) continue;
        const et::LongGeom g(len, cfg.slice_len);
        PlaneLoad load{m, b.hi, b.lo, b.val, {b0, 0u}};
        unsigned short* row = a.stats + (size_t)idx * (a.max_slices + 1);
        for (int t = 1 + (int)lane; t <= g.snum; t += 32) {
            u32 r = 0;
            if (g.len(t) <= et::kMaxRead) r = et::long_slice_stats(m, g, t, cfg.min_mer, cfg.max_mer, cfg.thr_low, cfg.thr_high, load, x);
            row[t] = (unsigned short)r;
        }
    }
}

// step 2: thread per survivor
__global__ void __launch_bounds__(256) trew_long_walk_kernel(DevCfg cfg, DevBatch b, LongArgs a) {
    const u32 n_all = *a.n_survivors;
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.total_survivors) atomicAdd(a.total_survivors, (unsigned long long)n_all);
    const u32 stride = gridDim.x * blockDim.x, n_round = (n_all + 31u) & ~31u;
    for (u32 idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n_round; idx += stride) {
        bool bail = false;
        u32 entry = 0;
        if (idx < n_all) {
            entry = a.survivors[idx];
            u32 u = entry;
            if (a.packed_probes) u &= (1u << kProbeShift) - 1u;
            const int len = (int)(__ldg(b.bit_off + u + 1) - __ldg(b.bit_off + u));
            if (idx >= a.s_cap) bail = len >= cfg.slice_len;
            else if (len >= cfg.slice_len) {
                const et::LongGeom g(len, cfg.slice_len);
                const unsigned short* row = a.stats + (size_t)idx * (a.max_slices + 1);
                u32* em = a.emis + (size_t)idx * (a.max_slices + 1);
                for (int t = 1; t <= g.snum; t++) em[t] = 0u;
                auto stat = [&](int t) { return (u32)row[t]; };
                auto task = [&](const et::LongTask& tk) {
                    const int tb = tk.table_folded & 7, c = tb & 1;
                    const bool backward = (tb & 6) == et::T_B;
                    const u32 byte = (u32)tk.k | ((tk.table_folded & 8) ? 0x80u : 0u);
                    em[tk.slice] |= byte << (8 * ((backward ? 2 : 0) + c));
                };
                bail = !et::long_walk(g, stat, task);
                if (bail) for (int t = 1; t <= g.snum; t++) em[t] = 0u;
            }
        }
        list_append(bail, entry, a.hard, a.n_hard);
    }
}

// step 3: warp per survivor, lane per slice with emissions; REC: one unit record per emission
template <bool REC>
__global__ void __launch_bounds__(TREW_THREAD_BLOCK, 4) trew_long_emit_kernel(DevCfg cfg, DevBatch b, LongArgs a) {
    u32* work = reinterpret_cast<u32*>(g_smem);
    u64* s_key = reinterpret_cast<u64*>(work + et::Lay<et::u64>::WORDS * TREW_THREAD_BLOCK);
    u32* s_meta = reinterpret_cast<u32*>(s_key + kStageSlots);
    u32* s_cnt = s_meta + kStageSlots;
    for (int i = threadIdx.x; i < kStageSlots; i += blockDim.x) { s_meta[i] = 0u; s_cnt[i] = 0u; }
    __syncthreads();
    const et::Mem m{work + threadIdx.x, TREW_THREAD_BLOCK};
    StageEmit emit{s_meta, s_cnt, s_key, cfg.slots, cfg.slot_mask, cfg.error_flag};
    const u32 n = min(*a.n_survivors, a.s_cap);
    const u32 warps = gridDim.x * (blockDim.x >> 5), lane = lane_id();
    et::ClsSpill<et::u64> x;
    for (u32 idx = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); idx < n; idx += warps) {
        u32 u = a.survivors[idx];
        if (a.packed_probes) u &= (1u << kProbeShift) - 1u;
        const u32 b0 = __ldg(b.bit_off + u);
        const int len = (int)(__ldg(b.bit_off + u + 1) - b0);
        if (len < cfg.slice_len) continue;
        const et::LongGeom g(len, cfg.slice_len);
        PlaneLoad load{m, b.hi, b.lo, b.val, {b0, 0u}};
        const u32* em = a.emis + (size_t)idx * (a.max_slices + 1);
        for (int t = 1 + (int)lane; t <= g.snum; t += 32) {
            const u32 e = em[t];
            if (e == 0u) continue;
            for (int f = 0; f < 4; f++) {   // forward high, forward low, backward high, backward low
                const u32 byte = (e >> (8 * f)) & 0xffu;
                if (byte == 0u) continue;
                const int c = f & 1;
                const bool folded = (byte & 0x80u) != 0u;
                const int table = (f >= 2 ? et::T_B : (folded ? et::T_O : et::T_F)) + c;
                et::LongTask tk{(unsigned short)t, (unsigned char)(byte & 0x7fu), (unsigned char)(table | (folded ? 8 : 0))};
                if constexpr (REC) {
                    RecStageEmit rem{emit, cfg.recs, cfg.unit_base + u};
                    et::long_emit(m, g, tk, load, x, rem);
                } else {
                    et::long_emit(m, g, tk, load, x, emit);
                }
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kStageSlots; i += blockDim.x) {
        const u32 st = s_meta[i], c = s_cnt[i];
        if (st != 0u && st != kStageLock && c != 0u) table_add_impl(cfg.slots, cfg.slot_mask, cfg.error_flag, st & 0x7fffffffu, s_key[i], 0ULL, (u64)c);
    }
}

bool long_thread_path_applies(const DevCfg& cfg) { return cfg.mode == 2 && cfg.max_mer <= 32 && cfg.slice_len <= et::kMaxRead; }

size_t long_thread_scratch_bytes(unsigned int s_cap, unsigned int max_slices) {
    return (size_t)s_cap * (max_slices + 1) * (sizeof(unsigned short) + sizeof(u32)) + 64;
}

// survivors (list, counter) -> statistics, walks, emissions; reads the path cannot take are appended to hard / n_hard
void launch_long_thread(const DevCfg& cfg, const DevBatch& b, const unsigned int* survivors, const unsigned int* n_survivors,
                        int packed_probes, unsigned int s_cap, unsigned int max_slices, unsigned char* scratch, unsigned int* hard,
                        unsigned int* n_hard, unsigned long long* total_survivors, int sm_count, cudaStream_t stream) {
    LongArgs a{};
    a.survivors = survivors; a.n_survivors = n_survivors; a.packed_probes = packed_probes;
    a.s_cap = s_cap; a.max_slices = max_slices;
    a.emis = reinterpret_cast<u32*>(scratch);
    a.stats = reinterpret_cast<unsigned short*>(scratch + (size_t)s_cap * (max_slices + 1) * sizeof(u32));
    a.hard = hard; a.n_hard = n_hard; a.total_survivors = total_survivors;
    const size_t smem_stats = (size_t)et::Lay<et::u64>::WORDS * TREW_THREAD_BLOCK * sizeof(u32);
    trew_long_stats_kernel<<<sm_count * 4, TREW_THREAD_BLOCK, smem_stats, stream>>>(cfg, b, a);
    trew_long_walk_kernel<<<sm_count * 2, 256, 0, stream>>>(cfg, b, a);
    if (cfg.recs) trew_long_emit_kernel<true><<<sm_count * 4, TREW_THREAD_BLOCK, kThreadKernelSmem, stream>>>(cfg, b, a);
    else trew_long_emit_kernel<false><<<sm_count * 4, TREW_THREAD_BLOCK, kThreadKernelSmem, stream>>>(cfg, b, a);
}

// true when the thread kernel can take (most of) a batch: short single-end or paired mode, 64-bit units
bool thread_path_applies(const DevCfg& cfg, unsigned int max_read_len) {
    if (cfg.max_mer > 64) return false;
    if (cfg.mode == 0) return true;
    return cfg.mode == 1 && max_read_len >= 4u * (unsigned)cfg.max_mer;   // pairs below 4 * MAX_MER all take the large-k block
}

void launch_exact_thread(const DevCfg& cfg, const DevBatch& b, const unsigned int* survivors, const unsigned int* n_survivors,
                         int packed_probes, unsigned int* hard, unsigned int* n_hard, unsigned long long* total_survivors, int sm_count,
                         int blocks_per_sm, unsigned int* work_counter, cudaStream_t stream) {
    const bool wide = cfg.max_mer > 32;
    // blocks_per_sm 0: as many as the kernel was built to have resident (one wave)
#define TREW_LAUNCH_THREAD(MODE, K, REC)                                                                                          \
    trew_exact_thread_kernel<MODE, K, REC><<<sm_count * (blocks_per_sm > 0 ? blocks_per_sm : thread_kernel_bps<MODE, K>()),       \
                                             TREW_THREAD_BLOCK, thread_kernel_smem<K>(), stream>>>(                               \
        cfg, b, survivors, n_survivors, packed_probes, hard, n_hard, total_survivors, work_counter)
#define TREW_LAUNCH_THREAD_MODE(MODE)                                                                                             \
    if (cfg.recs) { if (wide) TREW_LAUNCH_THREAD(MODE, et::u128, true); else TREW_LAUNCH_THREAD(MODE, et::u64, true); }            \
    else          { if (wide) TREW_LAUNCH_THREAD(MODE, et::u128, false); else TREW_LAUNCH_THREAD(MODE, et::u64, false); }
    if (cfg.mode == 0) { TREW_LAUNCH_THREAD_MODE(0) }
    else               { TREW_LAUNCH_THREAD_MODE(1) }
#undef TREW_LAUNCH_THREAD_MODE
#undef TREW_LAUNCH_THREAD
}

template <int MODE, bool REC>   // REC: one unit record per class added
__global__ void __launch_bounds__(kExactWarps * 32, TREW_EXACT_BPS) trew_exact_kernel(DevCfg cfg, DevBatch b, ExactArgs a) {
    const int wid = threadIdx.x >> 5;
    const u32 lane = lane_id();
    WS ws;
    ws.cap = a.run_cap; ws.hs = exact_hash_slots(a.run_cap);
    ws.off = (u32)((size_t)wid * exact_warp_bytes(a.run_cap)); ws.lane = lane; ws.flags = a.exp_flags;
    TableRef tr{cfg.slots, cfg.slot_mask, cfg.error_flag};
    ws.hdr()[lane] = lane == HD_CUR_LEN || lane == HD_EV_LEN || lane == HD_EV_K ? 0xffffffffu : 0u;
    if constexpr (REC) {
        if (lane == HD_UNIT_BASE) { ws.hdr()[lane] = (u32)cfg.unit_base; ws.hdr()[lane + 1] = (u32)(cfg.unit_base >> 32); }
        if (lane == HD_RECS) { ws.hdr()[lane] = (u32)(u64)cfg.recs; ws.hdr()[lane + 1] = (u32)((u64)cfg.recs >> 32); }
    }
    __syncwarp();
    const u32 n = *a.n_survivors;
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.total_survivors) atomicAdd(a.total_survivors, (u64)n);
    unsigned char* scratch = a.slice_scratch + (size_t)(blockIdx.x * kExactWarps + wid) * a.slice_scratch_stride;
    for (;;) {
        u32 idx = 0;
        if (lane == 0) idx = atomicAdd(a.work_counter, 1u);
        idx = __shfl_sync(0xffffffffu, idx, 0);
        if (idx >= n) break;
        u32 u = a.reverse ? *(a.survivors - idx) : a.survivors[idx], pm = 0xfu;
        if (a.packed_probes) { pm = u >> kProbeShift; u &= (1u << kProbeShift) - 1u; }
        if constexpr (REC) ws.hdr()[HD_UNIT] = u;   // for emit_classes (every lane stores the same value)
        if constexpr (MODE == 0) route_short<REC>(cfg, tr, ws, b, u, pm);
        else if constexpr (MODE == 1) route_pair<REC>(cfg, tr, ws, b, u);
        else route_long<REC>(cfg, tr, ws, b, u, scratch);
    }
}

constexpr int kExactBlocksPerSM = TREW_EXACT_BPS;
int exact_warps_total(int sm_count) { return sm_count * kExactBlocksPerSM * kExactWarps; }

cudaError_t prepare_exact(int run_cap_max) {
    int bytes = (int)exact_smem_bytes(run_cap_max, true);
    cudaError_t e = cudaSuccess;
#define TREW_SMEM_ATTR(F, BYTES) if (e == cudaSuccess) e = cudaFuncSetAttribute(F, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(BYTES))
    TREW_SMEM_ATTR((trew_exact_kernel<0, false>), bytes);
    TREW_SMEM_ATTR((trew_exact_kernel<1, false>), bytes);
    TREW_SMEM_ATTR((trew_exact_kernel<2, false>), bytes);
    TREW_SMEM_ATTR((trew_exact_kernel<0, true>), bytes);
    TREW_SMEM_ATTR((trew_exact_kernel<1, true>), bytes);
    TREW_SMEM_ATTR((trew_exact_kernel<2, true>), bytes);
    TREW_SMEM_ATTR((trew_exact_thread_kernel<0, et::u64, false>), thread_kernel_smem<et::u64>());
    TREW_SMEM_ATTR((trew_exact_thread_kernel<1, et::u64, false>), thread_kernel_smem<et::u64>());
    TREW_SMEM_ATTR((trew_exact_thread_kernel<0, et::u128, false>), thread_kernel_smem<et::u128>());
    TREW_SMEM_ATTR((trew_exact_thread_kernel<1, et::u128, false>), thread_kernel_smem<et::u128>());
    TREW_SMEM_ATTR((trew_exact_thread_kernel<0, et::u64, true>), thread_kernel_smem<et::u64>());
    TREW_SMEM_ATTR((trew_exact_thread_kernel<1, et::u64, true>), thread_kernel_smem<et::u64>());
    TREW_SMEM_ATTR((trew_exact_thread_kernel<0, et::u128, true>), thread_kernel_smem<et::u128>());
    TREW_SMEM_ATTR((trew_exact_thread_kernel<1, et::u128, true>), thread_kernel_smem<et::u128>());
    TREW_SMEM_ATTR(trew_long_stats_kernel, kThreadKernelSmem);
    TREW_SMEM_ATTR(trew_long_emit_kernel<false>, kThreadKernelSmem);
    TREW_SMEM_ATTR(trew_long_emit_kernel<true>, kThreadKernelSmem);
#undef TREW_SMEM_ATTR
    return e;
}

// screen: many more blocks than are resident (8 per SM).  Its threads all do the same amount of work, but the warps of an
// SM drift apart, and in a single wave a third of the warp slots stood empty on average (ncu: 42 of 64 warps active)
// while the last warps finished; with 16 waves the block scheduler refills the slots.  Measured on 25 M reads: 2.24 ->
// 2.05 ms (8 -> 128 blocks per SM; 64: 2.06, 256: 2.05).  decide: resident blocks that share a work counter.
LaunchPlan default_launch_plan(int sm_count) { return LaunchPlan{sm_count * 128, sm_count * 4, sm_count * kExactBlocksPerSM}; }

void launch_exact(const DevCfg& cfg, const DevBatch& b, const ExactArgs& a, const LaunchPlan& plan, cudaStream_t stream) {
    size_t smem = exact_smem_bytes(a.run_cap, true);
    dim3 grid(plan.exact_blocks), block(kExactWarps * 32);
    if (cfg.recs) {
        if (cfg.mode == 0) trew_exact_kernel<0, true><<<grid, block, smem, stream>>>(cfg, b, a);
        else if (cfg.mode == 1) trew_exact_kernel<1, true><<<grid, block, smem, stream>>>(cfg, b, a);
        else trew_exact_kernel<2, true><<<grid, block, smem, stream>>>(cfg, b, a);
    } else {
        if (cfg.mode == 0) trew_exact_kernel<0, false><<<grid, block, smem, stream>>>(cfg, b, a);
        else if (cfg.mode == 1) trew_exact_kernel<1, false><<<grid, block, smem, stream>>>(cfg, b, a);
        else trew_exact_kernel<2, false><<<grid, block, smem, stream>>>(cfg, b, a);
    }
}

}  // namespace trew
