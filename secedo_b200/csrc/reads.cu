// K2 — read linking, paired-end mate rule and tail cutoff.
//
// The reference walks the filtered loci sequentially and rebuilds reads in a hash map keyed by
// read id (similarity_matrix.cpp:342-403). What the counting kernels need from that walk is: which
// entries share a read with another entry (same id twice at one locus = overlapping mates, or at
// several loci within one fragment length), what the mate rule (:387-395) makes of those reads, and
// the per-chromosome cutoff K implied by the batching at :354-373 + the clear() at :407-408
// (SURVEY.md Appendix A.4). In real pileups the overwhelming majority of the entries are the only
// entry of their read; everything about them is implicit (cell = own group, read created at the own
// locus). So the work is split into ONE dense pass that only finds the exceptions and a chain of
// small kernels over those exceptions ("special" entries):
//
//   link_window_kernel   dense, one CTA per owner locus: the owner's read ids go into a shared-memory
//                        table (plain stores for the first round, CAS only for the ~10 % displaced
//                        ids), the loci of the following L bp are streamed against it. Output: a
//                        compact list of links (entry x, entry y) carrying the same read id.
//   mark / rank / list   bitmap of special entries, popcount prefix = dense numbering ("sid")
//   link_min             first entry of every special entry's read (two atomicMin sweeps)
//   group / mate_rule    entry lists per read, sequential replay of the insertion rules (:383-402)
//   cutoff               K per chromosome from the per-locus number of reads created
//   sp_finish            code (cell, base, tail, multi | dropped) per special entry
// The bitmap is all the dense counting kernels read (1 bit per entry).
#include "common.cuh"

#include <algorithm>
#include <cstdlib>
#include <vector>

namespace {

constexpr int TB = 256;
constexpr uint64_t KEY_EMPTY = ~0ull;

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdull;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ull;
    x ^= x >> 33;
    return x;
}

__device__ __forceinline__ uint32_t chr_of_locus(const uint64_t *__restrict__ chr_ptr, uint32_t n_chr, uint64_t l) {
    uint32_t lo = 0, hi = n_chr; // largest c with chr_ptr[c] <= l
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (chr_ptr[mid] <= l) {
            lo = mid;
        } else {
            hi = mid;
        }
    }
    return lo;
}

// locus of entry e: largest l with row_ptr[l] <= e
__device__ __forceinline__ uint32_t locus_of_entry(const uint64_t *__restrict__ row_ptr, uint64_t n_loci, uint64_t e) {
    uint64_t lo = 0, hi = n_loci;
    while (hi - lo > 1) {
        const uint64_t mid = (lo + hi) >> 1;
        if (row_ptr[mid] <= e) {
            lo = mid;
        } else {
            hi = mid;
        }
    }
    return static_cast<uint32_t>(lo);
}

// lchr[l] = chromosome of locus l; checks strictly increasing positions; largest locus
__global__ void __launch_bounds__(TB) locus_meta_kernel(const uint64_t *__restrict__ row_ptr,
                                                        const uint32_t *__restrict__ position,
                                                        const uint64_t *__restrict__ chr_ptr, uint32_t n_chr,
                                                        uint64_t n_loci, uint8_t *__restrict__ lchr,
                                                        unsigned int *__restrict__ max_row, int *__restrict__ err) {
    const uint64_t l = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    unsigned int n = 0;
    if (l < n_loci) {
        const uint32_t c = chr_of_locus(chr_ptr, n_chr, l);
        lchr[l] = static_cast<uint8_t>(c);
        if (l > chr_ptr[c] && position[l] <= position[l - 1]) {
            atomicExch(err, SGPU_E_POSITIONS);
        }
        n = static_cast<unsigned int>(min(row_ptr[l + 1] - row_ptr[l], static_cast<uint64_t>(0xFFFFFFFFu)));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n = max(n, __shfl_xor_sync(0xffffffffu, n, o));
    }
    if ((threadIdx.x & 31) == 0 && n) {
        atomicMax(max_row, n);
    }
}

// ---- windowed linking ----------------------------------------------------------------------------
// A fragment spans less than L bp, so all entries of a read lie in the loci within L bp after the
// locus of its first entry. One CTA per "owner" locus puts the owner's read ids into a shared-memory
// open-addressing table of 16-bit entry indices and streams the entries of the following loci inside
// the window against it. Shared-memory atomics cost ~2 cycles per lane on this machine, plain
// loads/stores 1/8 of that, so the table is built optimistically: every entry stores its index at its
// home slot (last writer wins), reads it back, and only the losers (another id won the slot) insert
// themselves with CAS. An id that occurs several times at the owner keeps ONE representative in the
// table; the others are linked to it. Links go to a CTA-local buffer that is flushed with one global
// atomic per flush.
constexpr int WIN_THREADS = 512;
constexpr uint32_t SLOT_EMPTY = 0xFFFFu;
constexpr uint32_t REC_BUF = 1024;      // links staged per CTA between flushes
constexpr uint32_t WIN_MAX_ENTRIES = 0xFFFEu;
constexpr size_t WIN_SMEM_LIMIT = 220 * 1024;

struct WinCounters {
    unsigned long long n_links; // links produced (may exceed the capacity of the list: the host then retries)
};

__device__ __forceinline__ uint32_t slot_hash(uint32_t id, uint32_t shift) { return (id * 0x9E3779B1u) >> shift; }

__device__ __forceinline__ void emit_link(uint2 *rbuf, uint32_t *s_cnt, uint2 *__restrict__ links, uint64_t cap,
                                          WinCounters *__restrict__ ctr, uint32_t x, uint32_t y) {
    const uint32_t k = atomicAdd(s_cnt, 1u);
    if (k < REC_BUF) {
        rbuf[k] = make_uint2(x, y);
    } else { // staging buffer full: straight to the global list
        const unsigned long long g = atomicAdd(&ctr->n_links, 1ull);
        if (g < cap) {
            links[g] = make_uint2(x, y);
        }
    }
}

// cp.async helpers: global -> shared without staging registers
__device__ __forceinline__ void cp_async4(void *dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(dst))), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(void *dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(dst))), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

constexpr uint32_t WIN_RING = 3;   // at most: loci whose read ids are resident in shared memory (the owner and the two after it)
constexpr uint32_t WIN_META = 64;  // owners per block of locus metadata kept in shared memory
constexpr uint32_t WIN_META_N = WIN_META + WIN_RING + 1;

// Every CTA owns a CONTIGUOUS range of owner loci, so the loci of an owner's window are the next owners: the read ids of
// a locus are fetched from global memory once per CTA (cp.async into a ring of WIN_RING slots, two loci ahead of the
// owner being processed) and serve first as window entries of the preceding owners, then as the owner's own table.
// Neither the window probes nor the table build wait for global memory any more (the version that took the owners in
// a grid-stride loop read every entry 1 + (loci per window) times and exposed four dependent global round trips per
// owner: 14 % of HBM, barrier stalls). Window loci beyond the ring (dense loci: more than two within L bp) are still
// streamed from global memory.
__global__ void __launch_bounds__(WIN_THREADS, 2) link_window_kernel(
        const uint64_t *__restrict__ row_ptr, const uint32_t *__restrict__ position, const uint32_t *__restrict__ read_id,
        const uint64_t *__restrict__ src_off /* null, or: the ids of locus l start at read_id[src_off[l]] (sgpu_pileup::view_off) */,
        const uint8_t *__restrict__ lchr, uint64_t n_loci, uint32_t L, uint32_t loci_per_cta,
        uint32_t slots /* power of two */, uint32_t id_cap /* multiple of 4, >= largest locus + 4 */,
        uint32_t n_ring /* 1 .. WIN_RING slots of id_cap ids: as many as shared memory holds (huge loci: 1) */,
        uint2 *__restrict__ links, uint64_t cap, WinCounters *__restrict__ ctr) {
    extern __shared__ __align__(16) uint32_t s_mem[];
    uint32_t *ring = s_mem;                                                          // [n_ring][id_cap]
    uint2 *rbuf = reinterpret_cast<uint2 *>(s_mem + n_ring * id_cap);                // [REC_BUF]
    unsigned short *tab = reinterpret_cast<unsigned short *>(rbuf + REC_BUF);       // [slots]
    __shared__ uint64_t s_row[WIN_META_N + 1];
    __shared__ uint64_t s_src[WIN_META_N]; // first element of the locus in read_id (= s_row unless the ids are a view)
    __shared__ uint32_t s_pos[WIN_META_N];
    __shared__ uint8_t s_chr[WIN_META_N];
    __shared__ uint32_t s_cnt;
    __shared__ unsigned long long s_base;
    const uint32_t mask = slots - 1, shift = 32 - (31 - __clz(slots));
    const uint64_t la = static_cast<uint64_t>(blockIdx.x) * loci_per_cta;
    const uint64_t lb = min(n_loci, la + loci_per_cta);
    if (threadIdx.x == 0) {
        s_cnt = 0;
    }
    if (la >= lb) {
        return;
    }
    const bool aligned16 = (reinterpret_cast<uintptr_t>(read_id) & 15u) == 0; // else everything goes in 4-byte copies
    uint64_t meta0 = la; // first locus of the metadata block in shared memory
    auto load_meta = [&](uint64_t base) {
        for (uint32_t i = threadIdx.x; i <= WIN_META_N; i += WIN_THREADS) {
            const uint64_t l = base + i;
            s_row[i] = row_ptr[min(l, n_loci)];
            if (i < WIN_META_N) {
                s_pos[i] = l < n_loci ? position[l] : 0;
                s_chr[i] = l < n_loci ? lchr[l] : 0xFF;
                s_src[i] = l < n_loci ? (src_off ? src_off[l] : row_ptr[l]) : 0;
            }
        }
    };
    // the ids of locus l start at ring slot (l % WIN_RING) at element (first entry & 3): source and destination are
    // congruent modulo 16 bytes, so the body goes in 16-byte copies
    auto prefetch = [&](uint64_t l) {
        if (l < n_loci && l - meta0 < WIN_META_N) {
            const uint64_t e0 = s_src[l - meta0];
            uint32_t *dst = ring + (l % n_ring) * id_cap + (e0 & 3u);
            const uint32_t *src = read_id + e0;
            const uint32_t n = static_cast<uint32_t>(s_row[l - meta0 + 1] - s_row[l - meta0]);
            const uint32_t head = aligned16 ? min(n, static_cast<uint32_t>((4 - (e0 & 3u)) & 3u)) : n;
            const uint32_t body = (n - head) >> 2;
            for (uint32_t i = threadIdx.x; i < head; i += WIN_THREADS) {
                cp_async4(dst + i, src + i);
            }
            for (uint32_t i = threadIdx.x; i < body; i += WIN_THREADS) {
                cp_async16(dst + head + 4 * i, src + head + 4 * i);
            }
            const uint32_t done = head + 4 * body;
            if (threadIdx.x < n - done) {
                cp_async4(dst + done + threadIdx.x, src + done + threadIdx.x);
            }
        }
        cp_async_commit(); // one group per call, also when nothing was copied: the group arithmetic below stays uniform
    };
    load_meta(meta0);
    __syncthreads();
    for (uint32_t k = 0; k + 1 < n_ring; ++k) { // the ring runs n_ring - 1 loci ahead of the owner
        prefetch(la + k);
    }
    for (uint64_t lo = la; lo < lb; ++lo) {
        if (lo - meta0 >= WIN_META) { // next block of metadata (nothing is in flight that reads the old one: see the barrier below)
            cp_async_wait<0>();
            __syncthreads();
            meta0 = lo;
            load_meta(meta0);
            __syncthreads();
        }
        const uint32_t mi = static_cast<uint32_t>(lo - meta0);
        const uint64_t e0 = s_row[mi];
        const uint32_t n = static_cast<uint32_t>(s_row[mi + 1] - e0);
        const uint32_t p0 = s_pos[mi];
        const uint32_t chr = s_chr[mi];
        const uint32_t *ids = ring + (lo % n_ring) * id_cap + (s_src[mi] & 3u);
        // flush the staged links while nobody emits (uniform: s_cnt is read after the barrier that ended the last owner)
        if (s_cnt > REC_BUF / 2) {
            const uint32_t m = min(s_cnt, REC_BUF);
            if (threadIdx.x == 0) {
                s_base = atomicAdd(&ctr->n_links, static_cast<unsigned long long>(m));
            }
            __syncthreads();
            for (uint32_t i = threadIdx.x; i < m; i += WIN_THREADS) {
                if (s_base + i < cap) {
                    links[s_base + i] = rbuf[i];
                }
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                s_cnt = 0;
            }
        }
        prefetch(lo + n_ring - 1); // into the slot of owner lo - 1, which the barrier at the end of its turn released
        for (uint32_t i = threadIdx.x; i < slots / 2; i += WIN_THREADS) {
            reinterpret_cast<uint32_t *>(tab)[i] = 0xFFFFFFFFu;
        }
        if (n_ring == 1) {
            cp_async_wait<0>(); // the owner's ids were requested just now
        } else {
            cp_async_wait<1>(); // everything but the locus requested just now has arrived (issued at least one owner ago)
        }
        __syncthreads();
        // round 1: optimistic placement at the home slot
        for (uint32_t i = threadIdx.x; i < n; i += WIN_THREADS) {
            tab[slot_hash(ids[i], shift)] = static_cast<unsigned short>(i);
        }
        __syncthreads();
        // round 2: losers either carry the winner's id (overlapping mates: link) or insert with CAS
        for (uint32_t i = threadIdx.x; i < n; i += WIN_THREADS) {
            const uint32_t id = ids[i];
            uint32_t s = slot_hash(id, shift);
            uint32_t cur = tab[s];
            if (cur == i) {
                continue;
            }
            for (;;) {
                if (cur == SLOT_EMPTY) {
                    cur = atomicCAS(&tab[s], static_cast<unsigned short>(SLOT_EMPTY), static_cast<unsigned short>(i));
                    if (cur == SLOT_EMPTY) {
                        break; // placed
                    }
                }
                if (ids[cur] == id) {
                    emit_link(rbuf, &s_cnt, links, cap, ctr, static_cast<uint32_t>(e0) + cur, static_cast<uint32_t>(e0) + i);
                    break;
                }
                s = (s + 1) & mask;
                cur = tab[s];
            }
        }
        __syncthreads();
        // the loci of the window: same chromosome, less than L bp after the owner
        for (uint64_t l = lo + 1; l < n_loci; ++l) {
            const bool meta_here = l - meta0 < WIN_META_N;
            const uint32_t pl = meta_here ? s_pos[l - meta0] : position[l];
            const uint32_t cl = meta_here ? s_chr[l - meta0] : lchr[l];
            if (cl != chr || pl - p0 >= L) {
                break;
            }
            const uint64_t a0 = meta_here ? s_row[l - meta0] : row_ptr[l];
            const uint64_t a1 = meta_here ? s_row[l - meta0 + 1] : row_ptr[l + 1];
            const uint32_t nl = static_cast<uint32_t>(a1 - a0);
            if (l + 1 <= lo + n_ring && meta_here) {
                if (l + 1 == lo + n_ring) { // the locus prefetched in this turn
                    cp_async_wait<0>();
                    __syncthreads();
                }
                const uint32_t *wid = ring + (l % n_ring) * id_cap + (s_src[l - meta0] & 3u);
                for (uint32_t ib = threadIdx.x; ib < nl; ib += 4 * WIN_THREADS) {
                    uint32_t id4[4], cur4[4], s4[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) { // four independent table look-ups in flight
                        const uint32_t i = ib + u * WIN_THREADS;
                        id4[u] = i < nl ? wid[i] : 0;
                        s4[u] = slot_hash(id4[u], shift);
                        cur4[u] = i < nl ? tab[s4[u]] : SLOT_EMPTY;
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        uint32_t cur = cur4[u], sl = s4[u];
                        while (cur != SLOT_EMPTY) {
                            if (ids[cur] == id4[u]) {
                                emit_link(rbuf, &s_cnt, links, cap, ctr, static_cast<uint32_t>(e0) + cur,
                                          static_cast<uint32_t>(a0) + ib + u * WIN_THREADS);
                                break;
                            }
                            sl = (sl + 1) & mask;
                            cur = tab[sl];
                        }
                    }
                }
            } else {
                // where the ids of this locus start in read_id, relative to its entry numbers
                const uint64_t shift_src = (meta_here ? s_src[l - meta0] : (src_off ? src_off[l] : a0)) - a0;
                for (uint64_t eb = a0 + threadIdx.x; eb < a1; eb += 4 * WIN_THREADS) {
                    uint32_t id4[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) { // four loads in flight
                        const uint64_t e = eb + u * WIN_THREADS;
                        id4[u] = e < a1 ? read_id[e + shift_src] : 0;
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const uint64_t e = eb + u * WIN_THREADS;
                        if (e >= a1) {
                            break;
                        }
                        const uint32_t id = id4[u];
                        uint32_t sl = slot_hash(id, shift);
                        for (;;) {
                            const uint32_t cur = tab[sl];
                            if (cur == SLOT_EMPTY) {
                                break;
                            }
                            if (ids[cur] == id) {
                                emit_link(rbuf, &s_cnt, links, cap, ctr, static_cast<uint32_t>(e0) + cur, static_cast<uint32_t>(e));
                                break;
                            }
                            sl = (sl + 1) & mask;
                        }
                    }
                }
            }
        }
        __syncthreads(); // the probes of this owner are done: its table and its ring slot may be reused
    }
    cp_async_wait<0>();
    const uint32_t m = min(s_cnt, REC_BUF);
    if (m) {
        if (threadIdx.x == 0) {
            s_base = atomicAdd(&ctr->n_links, static_cast<unsigned long long>(m));
        }
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < m; i += WIN_THREADS) {
            if (s_base + i < cap) {
                links[s_base + i] = rbuf[i];
            }
        }
    }
}

// ---- fallback for loci too large for the shared-memory table: global (chromosome, id) hash ---------
__global__ void __launch_bounds__(TB) ghash_insert_kernel(const uint64_t *__restrict__ row_ptr,
                                                          const uint32_t *__restrict__ read_id,
                                                          const uint8_t *__restrict__ lchr, uint64_t n_loci,
                                                          uint64_t *__restrict__ keys, uint32_t *__restrict__ vals,
                                                          uint64_t mask) {
    for (uint64_t l = blockIdx.x; l < n_loci; l += gridDim.x) {
        const uint64_t e0 = row_ptr[l], e1 = row_ptr[l + 1];
        const uint64_t chr = lchr[l];
        for (uint64_t e = e0 + threadIdx.x; e < e1; e += TB) {
            const uint64_t key = (chr << 32) | read_id[e];
            uint64_t slot = mix64(key) & mask;
            for (;;) {
                uint64_t cur = keys[slot];
                if (cur == KEY_EMPTY) {
                    cur = atomicCAS(reinterpret_cast<unsigned long long *>(&keys[slot]), KEY_EMPTY, key);
                    if (cur == KEY_EMPTY) {
                        break;
                    }
                }
                if (cur == key) {
                    break;
                }
                slot = (slot + 1) & mask;
            }
            atomicMin(&vals[slot], static_cast<uint32_t>(e));
        }
    }
}

__global__ void __launch_bounds__(TB) ghash_emit_kernel(const uint64_t *__restrict__ row_ptr,
                                                        const uint32_t *__restrict__ read_id,
                                                        const uint8_t *__restrict__ lchr, uint64_t n_loci,
                                                        const uint64_t *__restrict__ keys, const uint32_t *__restrict__ vals,
                                                        uint64_t mask, uint2 *__restrict__ links, uint64_t cap,
                                                        WinCounters *__restrict__ ctr) {
    for (uint64_t l = blockIdx.x; l < n_loci; l += gridDim.x) {
        const uint64_t e0 = row_ptr[l], e1 = row_ptr[l + 1];
        const uint64_t chr = lchr[l];
        for (uint64_t base = e0; base < e1; base += TB) {
            const uint64_t e = base + threadIdx.x;
            uint32_t first = 0xFFFFFFFFu;
            if (e < e1) {
                const uint64_t key = (chr << 32) | read_id[e];
                uint64_t slot = mix64(key) & mask;
                while (keys[slot] != key) {
                    slot = (slot + 1) & mask;
                }
                first = vals[slot];
            }
            const bool hit = e < e1 && first != static_cast<uint32_t>(e);
            const uint32_t ballot = __ballot_sync(0xffffffffu, hit);
            if (ballot) {
                const int lane = threadIdx.x & 31, leader = __ffs(ballot) - 1;
                unsigned long long g = 0;
                if (lane == leader) {
                    g = atomicAdd(&ctr->n_links, static_cast<unsigned long long>(__popc(ballot)));
                }
                g = __shfl_sync(0xffffffffu, g, leader);
                if (hit) {
                    g += __popc(ballot & ((1u << lane) - 1u));
                    if (g < cap) {
                        links[g] = make_uint2(first, static_cast<uint32_t>(e));
                    }
                }
            }
        }
    }
}

// ---- special entries ------------------------------------------------------------------------------
__global__ void __launch_bounds__(TB) mark_kernel(const uint2 *__restrict__ links, uint64_t n_links,
                                                  uint32_t *__restrict__ bits) {
    const uint64_t i = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (i < n_links) {
        const uint2 r = links[i];
        atomicOr(&bits[r.x >> 5], 1u << (r.x & 31));
        atomicOr(&bits[r.y >> 5], 1u << (r.y & 31));
    }
}

__global__ void __launch_bounds__(TB) popc_kernel(const uint32_t *__restrict__ bits, uint64_t n_words,
                                                  uint32_t *__restrict__ pc) {
    const uint64_t w = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (w < n_words) {
        pc[w] = __popc(bits[w]);
    }
}

__device__ __forceinline__ uint32_t sid_of(const uint32_t *__restrict__ bits, const uint64_t *__restrict__ rank, uint32_t e) {
    return static_cast<uint32_t>(rank[e >> 5]) + __popc(bits[e >> 5] & ((1u << (e & 31)) - 1u));
}

// word_locus[w] = locus of entry 32 w (the first entry of bitmap word w)
__global__ void __launch_bounds__(TB) word_locus_kernel(const uint64_t *__restrict__ row_ptr, uint64_t n_loci,
                                                        uint64_t n_words, uint32_t *__restrict__ word_locus) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps_total = static_cast<uint64_t>(gridDim.x) * (TB / 32);
    for (uint64_t l = static_cast<uint64_t>(blockIdx.x) * (TB / 32) + (threadIdx.x >> 5); l < n_loci; l += warps_total) {
        const uint64_t e0 = row_ptr[l], e1 = l + 1 < n_loci ? row_ptr[l + 1] : n_words * 32;
        // words whose first entry lies in [e0, e1)
        for (uint64_t w = (e0 + 31) / 32 + lane; w * 32 < e1 && w < n_words; w += 32) {
            word_locus[w] = static_cast<uint32_t>(l);
        }
    }
}

__global__ void __launch_bounds__(TB) sp_list_kernel(const uint32_t *__restrict__ bits, const uint64_t *__restrict__ rank,
                                                     uint64_t n_words, const uint64_t *__restrict__ row_ptr,
                                                     const uint32_t *__restrict__ word_locus, uint32_t *__restrict__ sp_entry,
                                                     uint32_t *__restrict__ sp_first, uint32_t *__restrict__ sp_locus) {
    const uint64_t w = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (w >= n_words) {
        return;
    }
    uint32_t b = bits[w];
    if (b == 0) {
        return;
    }
    uint64_t k = rank[w];
    uint32_t l = word_locus[w];
    uint64_t l_end = row_ptr[l + 1];
    while (b) {
        const uint32_t bit = __ffs(b) - 1;
        b &= b - 1;
        const uint32_t e = static_cast<uint32_t>(w * 32 + bit);
        while (e >= l_end) { // entries are ascending: walk on to the locus that holds e
            ++l;
            l_end = row_ptr[l + 1];
        }
        sp_entry[k] = e;
        sp_first[k] = e;
        sp_locus[k] = l;
        ++k;
    }
}

// one sweep of "first entry of my read = smallest entry linked to me"; two sweeps settle every read
// whose entries all lie in the window of its first locus, a third one only verifies
__global__ void __launch_bounds__(TB) link_min_kernel(const uint2 *__restrict__ links, uint64_t n_links,
                                                      const uint32_t *__restrict__ bits, const uint64_t *__restrict__ rank,
                                                      uint32_t *__restrict__ sp_first, int *__restrict__ changed) {
    const uint64_t i = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (i >= n_links) {
        return;
    }
    const uint2 r = links[i];
    const uint32_t sx = sid_of(bits, rank, r.x), sy = sid_of(bits, rank, r.y);
    const uint32_t fx = sp_first[sx], fy = sp_first[sy];
    const uint32_t m = min(fx, fy);
    if (fx != m) {
        atomicMin(&sp_first[sx], m);
        *changed = 1;
    }
    if (fy != m) {
        atomicMin(&sp_first[sy], m);
        *changed = 1;
    }
}

__global__ void __launch_bounds__(TB) group_count_kernel(const uint32_t *__restrict__ bits, const uint64_t *__restrict__ rank,
                                                         const uint32_t *__restrict__ sp_first, uint64_t n_special,
                                                         uint32_t *__restrict__ sp_head, uint32_t *__restrict__ g_cnt) {
    const uint64_t s = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (s < n_special) {
        const uint32_t h = sid_of(bits, rank, sp_first[s]);
        sp_head[s] = h;
        atomicAdd(&g_cnt[h], 1u);
    }
}

__global__ void __launch_bounds__(TB) group_fill_kernel(const uint32_t *__restrict__ sp_head,
                                                        const uint32_t *__restrict__ sp_locus,
                                                        const uint64_t *__restrict__ g_off, uint64_t n_special,
                                                        uint32_t *__restrict__ cursor, uint32_t *__restrict__ g_list) {
    const uint64_t s = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (s < n_special) {
        const uint32_t h = sp_head[s];
        const uint32_t k = atomicAdd(&cursor[h], 1u);
        g_list[g_off[h] + k] = static_cast<uint32_t>(s);
    }
    (void)sp_locus;
}

// nf_locus[l] = entries of locus l that do not create a read (special entries that are not the first of
// their read); the special entries of a locus are contiguous: one warp per locus, no atomics
__global__ void __launch_bounds__(TB) nonfirst_kernel(const uint32_t *__restrict__ sp_head, const uint32_t *__restrict__ sp_start,
                                                      uint64_t n_loci, uint32_t *__restrict__ nf_locus) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps_total = static_cast<uint64_t>(gridDim.x) * (TB / 32);
    for (uint64_t l = static_cast<uint64_t>(blockIdx.x) * (TB / 32) + (threadIdx.x >> 5); l < n_loci; l += warps_total) {
        const uint32_t s0 = sp_start[l], s1 = sp_start[l + 1];
        uint32_t n = 0;
        for (uint32_t s = s0 + lane; s < s1; s += 32) {
            n += sp_head[s] != s;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            n += __shfl_xor_sync(0xffffffffu, n, o);
        }
        if (lane == 0) {
            nf_locus[l] = n;
        }
    }
}

// A read id chained over >= L bp (e.g. a long-insert pair whose mates, and a locus in between, all fall on kept loci):
// the reference retires a read once start + L <= position and makes a NEW read of the next entry with that id
// (similarity_matrix.cpp:348-372, 379-382; exactly so whenever the batch fires at every locus, i.e. on any pileup with
// >= 4 * num_threads new reads per locus; on sparser ones its outcome depends on batch timing). One thread per read:
// sort the entries, walk them, and re-root every entry that lies >= L bp behind the start of its segment to the entry
// that opens the next segment. sp_first holds ENTRY indices.
__global__ void __launch_bounds__(TB) split_span_kernel(const uint32_t *__restrict__ sp_head, const uint32_t *__restrict__ sp_entry,
                                                        const uint32_t *__restrict__ sp_locus, const uint64_t *__restrict__ g_off,
                                                        uint64_t n_special, uint32_t *__restrict__ g_list /* sids of the read */,
                                                        const uint32_t *__restrict__ position, uint32_t L,
                                                        uint32_t *__restrict__ sp_first, unsigned long long *__restrict__ n_splits) {
    const uint64_t h = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (h >= n_special || sp_head[h] != h) {
        return;
    }
    const uint64_t o = g_off[h];
    const uint32_t n = static_cast<uint32_t>(g_off[h + 1] - o);
    uint32_t *lst = g_list + o;
    for (uint32_t i = 1; i < n; ++i) { // insertion sort, n is tiny
        const uint32_t v = lst[i];
        uint32_t j = i;
        while (j > 0 && lst[j - 1] > v) {
            lst[j] = lst[j - 1];
            --j;
        }
        lst[j] = v;
    }
    uint32_t seg = lst[0], splits = 0;
    uint32_t seg_pos = position[sp_locus[seg]];
    for (uint32_t i = 1; i < n; ++i) {
        const uint32_t s = lst[i];
        const uint32_t pos = position[sp_locus[s]];
        if (pos - seg_pos >= L) {
            seg = s;
            seg_pos = pos;
            ++splits;
        }
        sp_first[s] = sp_entry[seg];
    }
    if (splits) {
        atomicAdd(n_splits, static_cast<unsigned long long>(splits));
    }
}

// One thread per read with >= 2 entries: sort its entries (entry order = the order in which the
// reference meets them), replay the insertion rules (similarity_matrix.cpp:383-402) and leave the
// stored (locus, base) list in place. g_nst[head] = number of loci the read keeps.
template <typename GB>
__global__ void __launch_bounds__(TB) mate_rule_kernel(const uint32_t *__restrict__ sp_head,
                                                       const uint32_t *__restrict__ sp_entry,
                                                       const uint32_t *__restrict__ sp_locus,
                                                       const uint64_t *__restrict__ g_off, uint64_t n_special,
                                                       uint32_t *__restrict__ g_list /* in: sids, out: stored loci */,
                                                       uint8_t *__restrict__ g_base, const GB *__restrict__ gid_base,
                                                       const uint32_t *__restrict__ position, uint32_t L,
                                                       uint8_t *__restrict__ sp_drop, uint32_t *__restrict__ g_nst,
                                                       int *__restrict__ err) {
    const uint64_t h = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (h >= n_special || sp_head[h] != h) {
        return;
    }
    const uint64_t o = g_off[h];
    const uint32_t n = static_cast<uint32_t>(g_off[h + 1] - o);
    uint32_t *lst = g_list + o;
    for (uint32_t i = 1; i < n; ++i) { // insertion sort, n is tiny
        const uint32_t v = lst[i];
        uint32_t j = i;
        while (j > 0 && lst[j - 1] > v) {
            lst[j] = lst[j - 1];
            --j;
        }
        lst[j] = v;
    }
    if (lst[0] != h) {
        atomicExch(err, SGPU_E_FRAGMENT_SPAN); // the linking did not converge: a chain of windows
        g_nst[h] = 0;
        return;
    }
    const uint32_t start_pos = position[sp_locus[h]];
    uint32_t n_st = 0;
    uint32_t last_sid = 0; // special entry that produced the last stored element
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t s = lst[i];
        const uint32_t loc = sp_locus[s];
        const uint8_t base = gid_base[sp_entry[s]] & 3;
        if (position[loc] - start_pos >= L) {
            atomicExch(err, SGPU_E_FRAGMENT_SPAN);
        }
        if (n_st > 0 && lst[n_st - 1] == loc) { // read.pos.back() == pd.position (:387)
            if (g_base[o + n_st - 1] != base) { // mates disagree: remove the stored base too (:390-393)
                sp_drop[last_sid] = 1;
                --n_st;
                // the element below (if any) was produced by an entry we no longer track; it can only
                // be popped by a further entry at ITS locus, which cannot come (loci are increasing)
            }
            sp_drop[s] = 1;
            continue;
        }
        // lst[0..n_st) is overwritten with stored loci; i >= n_st always holds
        lst[n_st] = loc;
        g_base[o + n_st] = base;
        last_sid = s;
        ++n_st;
    }
    g_nst[h] = n_st;
}

// readbase[l] = number of reads created before locus l (l = 0..n_loci)
__global__ void __launch_bounds__(TB) readbase_kernel(const uint64_t *__restrict__ row_ptr,
                                                      const uint64_t *__restrict__ nf_scan /* may be null */,
                                                      uint64_t n_loci, uint64_t *__restrict__ readbase) {
    const uint64_t l = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (l <= n_loci) {
        readbase[l] = row_ptr[l] - (nf_scan ? nf_scan[l] : 0);
    }
}

// SURVEY Appendix A.4. One CTA per chromosome. u(l) = number of reads whose start + L <= position[l]
// (a binary search over the positions, reads are created locus by locus); the reference's batching
// rule "if u - front >= need: front = u" is sequential, but a locus with u(l) - u(l-1) >= need fires
// whatever happened before it (front <= u(l-1)), so the replay only has to start at the LAST such locus:
// found by all threads scanning chunks backwards from the chromosome's end, then one thread replays
// the few loci behind it.
constexpr int CUT_THREADS = 256;
constexpr int CUT_CHUNK = 1024;

// number of completed reads at locus l and the first locus whose reads are not complete yet
__device__ __forceinline__ uint64_t completed_at(const uint32_t *__restrict__ position, const uint64_t *__restrict__ readbase,
                                                 uint64_t l0, uint64_t l, uint32_t L, uint64_t rb0, uint32_t *j_out) {
    const uint64_t p = position[l];
    uint64_t lo = l0, hi = l; // first locus in [l0, l] with position + L > p
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (static_cast<uint64_t>(position[mid]) + L > p) {
            hi = mid;
        } else {
            lo = mid + 1;
        }
    }
    *j_out = static_cast<uint32_t>(lo - l0);
    return readbase[lo] - rb0; // reads with start + L <= p, all created before locus l
}

// exact_from (may be null): per chromosome the first locus from which the numbers of reads created per locus are exact
// (a SUFFIX of a chromosome: the loci within L bp of its first locus may continue reads that started before it). Only
// a sure trigger whose inputs are all exact may then anchor the replay; if there is none, resolved[c] = 0 and the
// caller has to come back with a longer suffix.
__global__ void __launch_bounds__(CUT_THREADS) cutoff_kernel(const uint64_t *__restrict__ chr_ptr, uint32_t n_chr,
                                                             const uint32_t *__restrict__ position,
                                                             const uint64_t *__restrict__ readbase, uint32_t L,
                                                             uint32_t num_threads, uint64_t *__restrict__ n_tail_reads,
                                                             uint64_t *__restrict__ tail_locus,
                                                             const uint64_t *__restrict__ exact_from = nullptr,
                                                             uint8_t *__restrict__ resolved = nullptr) {
    __shared__ uint64_t s_u[CUT_CHUNK + 1];
    __shared__ uint32_t s_j[CUT_CHUNK + 1];
    __shared__ unsigned long long s_sure; // 1 + last locus that fires for sure, 0 = none found yet
    const uint32_t c = blockIdx.x;
    if (c >= n_chr) {
        return;
    }
    const uint64_t l0 = chr_ptr[c], l1 = chr_ptr[c + 1];
    const uint64_t rb0 = readbase[l0];
    const uint64_t need = 4ull * num_threads; // BATCH_SIZE * num_threads (similarity_matrix.cpp:354-356)
    const uint64_t ex0 = exact_from ? exact_from[c] : l0;
    if (threadIdx.x == 0) {
        s_sure = 0;
    }
    __syncthreads();
    // ---- backwards: the last locus whose trigger fires whatever the history
    for (uint64_t end = l1; end > l0; end = end > l0 + CUT_CHUNK ? end - CUT_CHUNK : l0) {
        const uint64_t base = end > l0 + CUT_CHUNK ? end - CUT_CHUNK : l0;
        const uint32_t n = static_cast<uint32_t>(end - base);
        // s_u[0] belongs to locus base - 1 (0 completed reads before the first locus), s_u[1 + i] to base + i
        for (uint32_t i = threadIdx.x; i <= n; i += CUT_THREADS) {
            uint32_t j = 0;
            s_u[i] = (i == 0 && base == l0) ? 0 : completed_at(position, readbase, l0, base + i - 1, L, rb0, &j);
            s_j[i] = j;
        }
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < n; i += CUT_THREADS) {
            // s_u[i + 1] - s_u[i] = reads created at the loci [l0 + s_j[i], l0 + s_j[i + 1])
            if (s_u[i + 1] - s_u[i] >= need && l0 + s_j[i] >= ex0) {
                atomicMax(&s_sure, static_cast<unsigned long long>(base + i + 1));
            }
        }
        __syncthreads();
        if (s_sure) {
            break;
        }
    }
    if (resolved && threadIdx.x == 0) {
        resolved[c] = (s_sure != 0 || ex0 <= l0) ? 1 : 0;
    }
    // ---- forwards from there: one thread replays the batching rule chunk by chunk
    uint64_t front = 0, jk = l0, start = l0; // used by thread 0 only
    if (s_sure) {
        start = s_sure; // the locus after the sure one
        if (threadIdx.x == 0) {
            uint32_t j = 0;
            front = completed_at(position, readbase, l0, s_sure - 1, L, rb0, &j);
            jk = l0 + j;
        }
    }
    for (uint64_t base = start; base < l1; base += CUT_CHUNK) {
        const uint32_t n = static_cast<uint32_t>(min(static_cast<uint64_t>(CUT_CHUNK), l1 - base));
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < n; i += CUT_THREADS) {
            s_u[i] = completed_at(position, readbase, l0, base + i, L, rb0, &s_j[i]);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (uint32_t i = 0; i < n; ++i) {
                const uint64_t u = s_u[i];
                if (u > front && u - front >= need) {
                    front = u;
                    jk = l0 + s_j[i];
                }
            }
        }
    }
    if (threadIdx.x == 0) {
        // reads with index >= K = rb0 + front are exactly those created at loci >= jk
        n_tail_reads[c] = readbase[l1] - (rb0 + front);
        tail_locus[c] = jk;
    }
}

// ranged accumulation: per chromosome the loci that hold tail reads and the owned loci, from positions
__global__ void range_bounds_kernel(const uint64_t *__restrict__ chr_ptr, uint32_t n_chr, const uint32_t *__restrict__ position,
                                    const uint32_t *__restrict__ own_pos_begin, const uint32_t *__restrict__ own_pos_end,
                                    const uint32_t *__restrict__ tail_position, uint64_t *__restrict__ tail_locus,
                                    uint64_t *__restrict__ own_lo, uint64_t *__restrict__ own_hi) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chr) {
        return;
    }
    const uint64_t l0 = chr_ptr[c], l1 = chr_ptr[c + 1];
    auto lower = [&](uint32_t pos) { // first locus of the chromosome with position >= pos
        uint64_t lo = l0, hi = l1;
        while (lo < hi) {
            const uint64_t mid = (lo + hi) >> 1;
            if (position[mid] < pos) {
                lo = mid + 1;
            } else {
                hi = mid;
            }
        }
        return lo;
    };
    if (tail_position[c] != SGPU_TAIL_AUTO) { // else: decided by cutoff_kernel from this piece, which holds the chromosome's end
        tail_locus[c] = lower(tail_position[c]);
    }
    own_lo[c] = lower(own_pos_begin[c]);
    own_hi[c] = max(own_lo[c], lower(own_pos_end[c]));
}

// suffix mode of the cutoff: first locus of every chromosome whose number of created reads is exact
__global__ void exact_from_kernel(const uint64_t *__restrict__ chr_ptr, uint32_t n_chr, const uint32_t *__restrict__ position,
                                  uint32_t L, const uint8_t *__restrict__ whole, uint64_t *__restrict__ exact_from) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chr) {
        return;
    }
    const uint64_t l0 = chr_ptr[c], l1 = chr_ptr[c + 1];
    uint64_t lo = l0, hi = l1;
    if (!whole[c] && l1 > l0) {
        const uint64_t want = static_cast<uint64_t>(position[l0]) + L;
        while (lo < hi) {
            const uint64_t mid = (lo + hi) >> 1;
            if (position[mid] < want) {
                lo = mid + 1;
            } else {
                hi = mid;
            }
        }
    }
    exact_from[c] = lo;
}

__global__ void tail_position_kernel(const uint64_t *__restrict__ chr_ptr, uint32_t n_chr, const uint32_t *__restrict__ position,
                                     const uint64_t *__restrict__ tail_locus, uint32_t *__restrict__ tail_position) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n_chr) {
        const uint64_t t = tail_locus[c];
        tail_position[c] = t < chr_ptr[c + 1] ? position[t] : 0xFFFFFFFFu; // no tail reads at all
    }
}

__global__ void __launch_bounds__(TB) owned_fill_kernel(const uint8_t *__restrict__ lchr, const uint64_t *__restrict__ own_lo,
                                                        const uint64_t *__restrict__ own_hi, uint64_t n_loci,
                                                        uint8_t *__restrict__ owned) {
    const uint64_t l = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (l < n_loci) {
        const uint32_t c = lchr[l];
        owned[l] = (l >= own_lo[c] && l < own_hi[c]) ? 1 : 0;
    }
}

template <typename GB>
__global__ void __launch_bounds__(TB) sp_finish_kernel(
        const uint32_t *__restrict__ sp_head, const uint32_t *__restrict__ sp_entry, const uint32_t *__restrict__ sp_locus,
        const uint8_t *__restrict__ sp_drop, const uint32_t *__restrict__ g_nst, const GB *__restrict__ gid_base,
        const uint8_t *__restrict__ lchr, const uint64_t *__restrict__ tail_locus, const uint32_t *__restrict__ gmap,
        uint32_t n_groups, uint32_t num_cells, uint64_t n_special, uint32_t *__restrict__ sp_code,
        uint32_t *__restrict__ sp_rcode,
        unsigned long long *__restrict__ stats /* [0]=dropped [1]=multi reads */, int *__restrict__ err) {
    // grid-stride: the two counters are summed per thread, per block, and reach global memory once per block (one
    // same-address atomic per WARP, 200 000 of them on the bench workload, had made this kernel 0.32 ms)
    __shared__ unsigned int s_dropped, s_multi;
    if (threadIdx.x == 0) {
        s_dropped = 0;
        s_multi = 0;
    }
    __syncthreads();
    uint32_t dropped = 0, multi_head = 0;
    for (uint64_t s = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x; s < n_special; s += static_cast<uint64_t>(gridDim.x) * TB) {
        const uint32_t h = sp_head[s];
        const uint32_t multi = g_nst[h] >= 2 ? 1u : 0u;
        multi_head += (h == s) & multi;
        const bool drop = sp_drop[s] != 0;
        if (drop) {
            sp_code[s] = CODE_DROPPED;
            ++dropped;
        }
        if (!drop || h == s) {
            // the read's cell is fixed by its first entry (similarity_matrix.cpp:379, :208-209)
            const uint32_t gid = gid_base[sp_entry[h]] >> 2;
            uint32_t cell = 0;
            if (gid >= n_groups || (cell = gmap[gid]) >= num_cells) {
                atomicExch(err, SGPU_E_CELL_RANGE);
                cell = 0;
            }
            const uint32_t base = gid_base[sp_entry[s]] & 3u;
            const uint32_t hl = sp_locus[h];
            const uint32_t tail = hl >= tail_locus[lchr[hl]] ? 1u : 0u; // read created behind the cutoff
            if (!drop) {
                sp_code[s] = (cell << 4) | (base << 2) | (tail << 1) | multi;
            }
            if (h == s) { // the read as a whole (its first entry may itself have been removed by the mate rule)
                sp_rcode[s] = (cell << 4) | (tail << 1) | multi;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        dropped += __shfl_xor_sync(0xffffffffu, dropped, o);
        multi_head += __shfl_xor_sync(0xffffffffu, multi_head, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (dropped) {
            atomicAdd(&s_dropped, dropped);
        }
        if (multi_head) {
            atomicAdd(&s_multi, multi_head);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_dropped) {
            atomicAdd(&stats[0], static_cast<unsigned long long>(s_dropped));
        }
        if (s_multi) {
            atomicAdd(&stats[1], static_cast<unsigned long long>(s_multi));
        }
    }
}

// sp_start[l] = first special entry with locus >= l, l = 0 .. n_loci
__global__ void __launch_bounds__(TB) sp_start_kernel(const uint32_t *__restrict__ sp_locus, uint64_t n_special,
                                                      uint64_t n_loci, uint32_t *__restrict__ sp_start) {
    const uint64_t l = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (l > n_loci) {
        return;
    }
    uint64_t lo = 0, hi = n_special;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (sp_locus[mid] < l) {
            lo = mid + 1;
        } else {
            hi = mid;
        }
    }
    sp_start[l] = static_cast<uint32_t>(lo);
}

// ---- candidates of the multi-locus correction ---------------------------------------------------------
__global__ void __launch_bounds__(TB) me_flag_kernel(const uint32_t *__restrict__ sp_code, const uint32_t *__restrict__ sp_head,
                                                     const uint32_t *__restrict__ sp_locus, const uint64_t *__restrict__ g_off,
                                                     const uint32_t *__restrict__ g_list, const uint32_t *__restrict__ g_nst,
                                                     uint64_t n_special, uint32_t min_nst, uint32_t *__restrict__ flag,
                                                     uint32_t *__restrict__ pos) {
    const uint64_t s = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (s >= n_special) {
        return;
    }
    const uint32_t c = sp_code[s];
    uint32_t f = 0;
    if (c != CODE_DROPPED && (c & 1u) && g_nst[sp_head[s]] >= min_nst) {
        const uint32_t h = sp_head[s], loc = sp_locus[s], n = g_nst[h];
        const uint64_t o = g_off[h];
        uint32_t i = 0;
        while (i < n && g_list[o + i] != loc) { // a surviving entry's locus is stored exactly once
            ++i;
        }
        f = i + 1 < n ? 1u : 0u;
        pos[s] = static_cast<uint32_t>(o + i);
    }
    flag[s] = f;
}

__global__ void __launch_bounds__(TB) me_compact_kernel(const uint32_t *__restrict__ flag, const uint32_t *__restrict__ pos,
                                                        const uint64_t *__restrict__ me_idx, const uint32_t *__restrict__ sp_code,
                                                        const uint32_t *__restrict__ sp_head, const uint32_t *__restrict__ sp_locus,
                                                        const uint64_t *__restrict__ g_off, const uint32_t *__restrict__ g_nst,
                                                        uint64_t n_special, uint32_t *__restrict__ me_code,
                                                        uint32_t *__restrict__ me_locus, uint32_t *__restrict__ me_pos,
                                                        uint32_t *__restrict__ me_beg, uint32_t *__restrict__ me_end) {
    const uint64_t s = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (s >= n_special || !flag[s]) {
        return;
    }
    const uint64_t k = me_idx[s];
    const uint32_t h = sp_head[s];
    me_code[k] = sp_code[s];
    me_locus[k] = sp_locus[s];
    me_pos[k] = pos[s];
    me_beg[k] = static_cast<uint32_t>(g_off[h]);
    me_end[k] = static_cast<uint32_t>(g_off[h]) + g_nst[h];
}

// ---- dense codes (scatter path only) ----------------------------------------------------------------
template <typename GB>
__global__ void __launch_bounds__(TB) dense_codes_kernel(const uint64_t *__restrict__ row_ptr,
                                                         const GB *__restrict__ gid_base,
                                                         const uint8_t *__restrict__ lchr,
                                                         const uint64_t *__restrict__ tail_locus,
                                                         const uint32_t *__restrict__ gmap, uint32_t n_groups,
                                                         uint32_t num_cells, uint64_t n_loci, uint32_t *__restrict__ code,
                                                         int *__restrict__ err) {
    for (uint64_t l = blockIdx.x; l < n_loci; l += gridDim.x) {
        const uint64_t e0 = row_ptr[l], e1 = row_ptr[l + 1];
        const uint32_t tail = l >= tail_locus[lchr[l]] ? 2u : 0u;
        for (uint64_t e = e0 + threadIdx.x; e < e1; e += TB) {
            const uint32_t gb = gid_base[e];
            const uint32_t gid = gb >> 2;
            uint32_t cell = 0;
            if (gid >= n_groups || (cell = gmap[gid]) >= num_cells) {
                atomicExch(err, SGPU_E_CELL_RANGE);
                cell = 0;
            }
            code[e] = (cell << 4) | ((gb & 3u) << 2) | tail; // special entries are overwritten afterwards
        }
    }
}

__global__ void __launch_bounds__(TB) sp_codes_kernel(const uint32_t *__restrict__ sp_entry,
                                                      const uint32_t *__restrict__ sp_code, uint64_t n_special,
                                                      uint32_t *__restrict__ code) {
    const uint64_t s = static_cast<uint64_t>(blockIdx.x) * TB + threadIdx.x;
    if (s < n_special) {
        code[sp_entry[s]] = sp_code[s];
    }
}

unsigned blocks_for(uint64_t n) { return static_cast<unsigned>(ceil_div_u64(n ? n : 1, TB)); }

bool env_is_1(const char *name) {
    const char *v = getenv(name);
    return v && v[0] == '1';
}

struct WinGeometry {
    uint32_t n_ring, slots, id_cap;
    size_t smem;
    bool use_window; // false: the global hash
};

// link_window's shared memory for loci of up to max_n entries: table slots >= 3 x the largest locus if shared memory
// allows, never below 1.25 x (else the global hash); the ring holds the read ids of n_ring loci (each slot: the largest
// locus + up to 3 elements of alignment offset)
WinGeometry window_geometry(uint32_t max_n, bool force_global) {
    WinGeometry g{ WIN_RING, 1024, (max_n + 3 + 3) & ~3u, 0, false };
    auto pow2_slots = [](unsigned long long want) {
        uint32_t sl = 1024;
        while (sl < want && sl < 65536) {
            sl <<= 1;
        }
        return sl;
    };
    auto win_smem = [&]() {
        return static_cast<size_t>(g.n_ring) * g.id_cap * 4 + REC_BUF * sizeof(uint2) + static_cast<size_t>(g.slots) * 2;
    };
    // preference: a ring of at least two loci (no exposed global latency per owner) before a sparse table (fewer second
    // probes); huge loci (cfg5: 20 000 reads) end at one resident locus and the largest table that fits. A CTA takes a
    // whole SM's shared memory: a geometry that fits beside the previous batch's tensor kernel (60 KB: one CTA per SM, a
    // denser table) was slower than letting link_window wait for it (profiles/r2_overlap_probes.txt).
    const uint32_t s_full = pow2_slots(3ull * max_n), s_half = std::min(s_full, pow2_slots(2ull * max_n));
    const uint32_t cand[4][2] = { { WIN_RING, s_full }, { 2, s_full }, { WIN_RING, s_half }, { 2, s_half } };
    for (const auto &cd : cand) {
        g.n_ring = cd[0];
        g.slots = cd[1];
        if (win_smem() <= WIN_SMEM_LIMIT) {
            break;
        }
    }
    if (win_smem() > WIN_SMEM_LIMIT) {
        g.n_ring = 1;
        g.slots = s_full;
        while (g.slots > 1024 && win_smem() > WIN_SMEM_LIMIT) {
            g.slots >>= 1;
        }
    }
    g.smem = win_smem();
    g.use_window = max_n <= WIN_MAX_ENTRIES && g.smem <= WIN_SMEM_LIMIT && 4ull * g.slots >= 5ull * max_n && !force_global;
    return g;
}

// device -> host scalars, over the context's pinned scratch
struct LinkScalars {
    uint64_t count, unused;      // count: one at a time (largest locus, links, special entries, unsettled sweep, span splits)
    int err, unsettled;          // d_err
    uint64_t n_dropped, n_multi; // d_stats
    uint64_t n_reads;            // readbase[n_loci]
};

constexpr int LINK_CAREFUL = 1; // status of a fast pass that met a read id chained over >= L bp: run the careful pass
const char *const MSG_CELL_RANGE = "a group id is >= n_groups or maps to a cell >= num_cells (filter the pileup first)";

// The stages of sgpu_link_reads and sgpu_cutoff_from_suffix, in the order they run, and what they share. A pass (from
// build_reads on) runs a second time, careful, only when the fast one ends with LINK_CAREFUL.
struct ReadLinker {
    sgpu_ctx *ctx;
    cudaStream_t st;
    const sgpu_pileup *p;
    LinkResult *out;
    uint32_t L;
    uint64_t E, P, W;    // entries, loci, words of the bitmap of special entries
    unsigned locus_grid; // kernels that stride over the loci
    bool strict_span;    // SECEDO_B200_STRICT_SPAN=1: a read id chained over >= L bp is an error instead of being split (tests)
    LinkScalars *hs;
    DevBuf<int> d_err;   // [0] error code, [1] "third sweep still changed something"
    DevBuf<WinCounters> d_ctr;
    DevBuf<unsigned long long> d_stats; // [0] dropped entries, [1] multi-locus reads
    DevBuf<uint64_t> readbase, n_tail_reads, nf_scan;
    DevBuf<uint2> links;
    uint64_t NL = 0, NS = 0; // links, special entries
    DevBuf<uint32_t> sp_first, g_cnt, cursor, nf_locus;

    ReadLinker(sgpu_ctx *c, const sgpu_pileup *pl, LinkResult *o, uint32_t L_)
        : ctx(c), st(c->stream), p(pl), out(o), L(L_), E(pl->n_entries), P(pl->n_loci), W(pl->n_entries / 32 + 1),
          locus_grid(static_cast<unsigned>(std::min<uint64_t>(pl->n_loci, static_cast<uint64_t>(c->sm_count) * 16))),
          strict_span(env_is_1("SECEDO_B200_STRICT_SPAN")), hs(reinterpret_cast<LinkScalars *>(c->h_scratch)) {}

    // the status of a pass from the error word in hs: a read id chained over >= L bp ends the fast pass with
    // LINK_CAREFUL and fails the careful one (or any with strict_span; name_strict: the message says so)
    int status(bool careful, bool name_strict) {
        if (hs->err == SGPU_E_CELL_RANGE) {
            return sgpu_fail(ctx, hs->err, "%s", MSG_CELL_RANGE);
        }
        if (hs->err == SGPU_E_POSITIONS) {
            return sgpu_fail(ctx, hs->err, "positions are not strictly increasing inside a chromosome");
        }
        if (hs->err == SGPU_E_FRAGMENT_SPAN || hs->unsettled) {
            if (careful || strict_span) {
                return sgpu_fail(ctx, SGPU_E_FRAGMENT_SPAN, "a read id spans >= max_fragment_length (%u)%s", L,
                                 strict_span && name_strict ? " (SECEDO_B200_STRICT_SPAN=1: not split)" : "");
            }
            return LINK_CAREFUL;
        }
        return SGPU_OK;
    }

    // argument checks, the result's arrays per group and locus, the error and statistics words, the largest locus
    int prepare(uint32_t num_cells, const uint32_t *h_group_id_to_pos, uint32_t n_groups, uint32_t num_threads, bool ranged) {
        if (E >= 0x7FFFFFF0ull || P >= 0x7FFFFFF0ull) {
            return sgpu_fail(ctx, SGPU_E_ARG, "more than 2^31 entries in one call: pass the pileup in batches of chromosomes");
        }
        if (p->n_chr > 255) {
            return sgpu_fail(ctx, SGPU_E_ARG, "more than 255 chromosomes in one call");
        }
        if (num_threads == 0) {
            return sgpu_fail(ctx, SGPU_E_ARG, "num_threads must be >= 1");
        }
        if (num_cells >= (1u << 27)) {
            return sgpu_fail(ctx, SGPU_E_ARG, "num_cells too large");
        }
        out->n_reads = out->n_multi = out->n_dropped = out->n_tail = out->n_special = out->n_tail_loci = out->n_own = 0;
        out->n_span_splits = 0;
        out->ranged = ranged;
        out->n_groups = n_groups;
        out->num_cells = num_cells;
        SGPU_CUDA(ctx, out->gmap.alloc(n_groups ? n_groups : 1, ctx));
        SGPU_CUDA(ctx, cudaMemcpyAsync(out->gmap.p, h_group_id_to_pos, n_groups * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        out->gmap_identity = n_groups <= num_cells;
        for (uint32_t g = 0; g < n_groups && out->gmap_identity; ++g) {
            out->gmap_identity = h_group_id_to_pos[g] == g;
        }
        SGPU_CUDA(ctx, out->sp_bits.alloc(W, ctx));
        SGPU_CUDA(ctx, cudaMemsetAsync(out->sp_bits.p, 0, W * sizeof(uint32_t), st));
        SGPU_CUDA(ctx, out->lchr.alloc(P ? P : 1, ctx));
        SGPU_CUDA(ctx, out->tail_locus.alloc(p->n_chr ? p->n_chr : 1, ctx));
        if (E == 0 || P == 0) {
            // nothing to link; tail_locus = end of every chromosome
            if (p->n_chr) {
                SGPU_CUDA(ctx, cudaMemcpyAsync(out->tail_locus.p, p->d_chr_ptr + 1, p->n_chr * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
            }
            SGPU_CUDA(ctx, out->tail_loci.alloc(1, ctx));
            return SGPU_OK;
        }

        SGPU_TRACE(ctx, "link: enter");
        DevBuf<unsigned int> d_maxn;
        SGPU_CUDA(ctx, d_err.alloc(2, ctx));
        SGPU_CUDA(ctx, d_maxn.alloc(1, ctx));
        SGPU_CUDA(ctx, d_ctr.alloc(1, ctx));
        SGPU_CUDA(ctx, d_stats.alloc(2, ctx));
        SGPU_CUDA(ctx, readbase.alloc(P + 1, ctx));
        SGPU_CUDA(ctx, n_tail_reads.alloc(p->n_chr, ctx));
        SGPU_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, 2 * sizeof(int), st));
        SGPU_CUDA(ctx, cudaMemsetAsync(d_maxn.p, 0, sizeof(unsigned int), st));
        SGPU_CUDA(ctx, cudaMemsetAsync(d_ctr.p, 0, sizeof(WinCounters), st));
        SGPU_CUDA(ctx, cudaMemsetAsync(d_stats.p, 0, 2 * sizeof(unsigned long long), st));

        SGPU_LAUNCH(ctx, (locus_meta_kernel<<<blocks_for(P), TB, 0, st>>>(p->d_row_ptr, p->d_position, p->d_chr_ptr, p->n_chr, P,
                                                                           out->lchr.p, d_maxn.p, d_err.p)));
        if (p->max_row == 0) {
            SGPU_CUDA(ctx, cudaMemcpyAsync(&hs->count, d_maxn.p, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
            SGPU_CUDA(ctx, cudaStreamSynchronize(st));
            p->max_row = static_cast<uint32_t>(hs->count); // cached: the pileup is immutable
        }
        SGPU_TRACE(ctx, "link: allocs+meta");
        return SGPU_OK;
    }

    // links between entries of one read
    int link_entries() {
        // SECEDO_B200_FORCE_GLOBAL_HASH=1 forces the large-locus path (tests)
        const WinGeometry g = window_geometry(p->max_row, env_is_1("SECEDO_B200_FORCE_GLOBAL_HASH"));
        uint64_t cap = std::max<uint64_t>(E / 8, 4096);
        for (int attempt = 0; attempt < 2; ++attempt) {
            SGPU_CUDA(ctx, links.alloc(cap, ctx));
            SGPU_CUDA(ctx, cudaMemsetAsync(d_ctr.p, 0, sizeof(WinCounters), st));
            if (g.use_window) {
                SGPU_CUDA(ctx, cudaFuncSetAttribute(link_window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(g.smem)));
                const unsigned per_sm = static_cast<unsigned>(std::max<size_t>(1, std::min<size_t>(4, (224 * 1024) / (g.smem + 2560))));
                // contiguous ranges of owner loci, one per CTA, all CTAs resident at once
                const uint64_t want = std::min<uint64_t>(P, static_cast<uint64_t>(ctx->sm_count) * per_sm);
                const uint32_t loci_per_cta = static_cast<uint32_t>(ceil_div_u64(P, want));
                const unsigned wgrid = static_cast<unsigned>(ceil_div_u64(P, loci_per_cta));
                // this kernel never fits beside the tensor kernel of the previous batch, so it and everything behind it on the
                // stream run alone: back to the default shared-memory / L1 split
                SGPU_TRY(sgpu_cache_preference(ctx, false));
                SGPU_LAUNCH(ctx, (link_window_kernel<<<wgrid, WIN_THREADS, g.smem, st>>>(p->d_row_ptr, p->d_position,
                                                                                        p->d_read_id ? p->d_read_id : p->view_read_id,
                                                                                        p->d_read_id ? nullptr : p->view_off, out->lchr.p, P, L,
                                                                                        loci_per_cta, g.slots, g.id_cap, g.n_ring, links.p, cap, d_ctr.p)));
            } else {
                SGPU_TRY(sgpu_pileup_materialize(ctx, p)); // the global hash reads the ids by entry number
                DevBuf<uint64_t> keys;
                DevBuf<uint32_t> vals;
                uint64_t hcap = 1024;
                while (hcap < 2 * E) {
                    hcap <<= 1;
                }
                SGPU_CUDA(ctx, keys.alloc(hcap, ctx));
                SGPU_CUDA(ctx, vals.alloc(hcap, ctx));
                SGPU_CUDA(ctx, cudaMemsetAsync(keys.p, 0xFF, hcap * sizeof(uint64_t), st));
                SGPU_CUDA(ctx, cudaMemsetAsync(vals.p, 0xFF, hcap * sizeof(uint32_t), st));
                SGPU_LAUNCH(ctx, (ghash_insert_kernel<<<locus_grid, TB, 0, st>>>(p->d_row_ptr, p->d_read_id, out->lchr.p, P, keys.p, vals.p, hcap - 1)));
                SGPU_LAUNCH(ctx, (ghash_emit_kernel<<<locus_grid, TB, 0, st>>>(p->d_row_ptr, p->d_read_id, out->lchr.p, P, keys.p, vals.p, hcap - 1,
                                                                                links.p, cap, d_ctr.p)));
            }
            SGPU_CUDA(ctx, cudaGetLastError());
            // the previous batch's tensor kernel, if its launch has been held back: behind the dense linking pass, beside
            // everything that follows (sgpu_tensor_flush)
            SGPU_TRY(sgpu_tensor_flush(ctx, true));
            SGPU_CUDA(ctx, cudaMemcpyAsync(&hs->count, d_ctr.p, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
            SGPU_CUDA(ctx, cudaStreamSynchronize(st));
            NL = hs->count;
            if (NL <= cap) {
                break;
            }
            if (attempt == 1) {
                return sgpu_fail(ctx, SGPU_E_CUDA, "link list overflow on retry (%llu > %llu)", (unsigned long long)NL, (unsigned long long)cap);
            }
            cap = NL; // the list was too small: the count is exact, run once more
        }
        SGPU_TRACE(ctx, "link: window kernel");
        return SGPU_OK;
    }

    // special entries: numbering, first entry of the read, groups, mate rule
    int number_special() {
        if (NL) {
            DevBuf<uint32_t> pc;
            SGPU_CUDA(ctx, pc.alloc(W, ctx));
            SGPU_CUDA(ctx, out->sp_rank.alloc(W + 1, ctx));
            SGPU_LAUNCH(ctx, (mark_kernel<<<blocks_for(NL), TB, 0, st>>>(links.p, NL, out->sp_bits.p)));
            SGPU_LAUNCH(ctx, (popc_kernel<<<blocks_for(W), TB, 0, st>>>(out->sp_bits.p, W, pc.p)));
            SGPU_TRY(sgpu_scan_u32_u64(ctx, pc.p, out->sp_rank.p, W));
            SGPU_CUDA(ctx, cudaMemcpyAsync(&hs->count, out->sp_rank.p + W, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
            SGPU_CUDA(ctx, cudaStreamSynchronize(st));
            NS = hs->count;
        }
        SGPU_TRACE(ctx, "link: mark+rank");
        out->n_special = NS;
        SGPU_CUDA(ctx, out->sp_start.alloc(P + 1, ctx));
        if (NS == 0) {
            SGPU_CUDA(ctx, cudaMemsetAsync(out->sp_start.p, 0, (P + 1) * sizeof(uint32_t), st));
            return SGPU_OK;
        }
        SGPU_CUDA(ctx, out->sp_entry.alloc(NS, ctx));
        SGPU_CUDA(ctx, out->sp_locus.alloc(NS, ctx));
        SGPU_CUDA(ctx, out->sp_head.alloc(NS, ctx));
        SGPU_CUDA(ctx, out->sp_code.alloc(NS, ctx));
        SGPU_CUDA(ctx, out->sp_drop.alloc(NS, ctx));
        SGPU_CUDA(ctx, out->sp_rcode.alloc(NS, ctx));
        SGPU_CUDA(ctx, out->g_off.alloc(NS + 1, ctx));
        SGPU_CUDA(ctx, out->g_list.alloc(NS, ctx));
        SGPU_CUDA(ctx, out->g_base.alloc(NS, ctx));
        SGPU_CUDA(ctx, out->g_nst.alloc(NS, ctx));
        SGPU_CUDA(ctx, sp_first.alloc(NS, ctx));
        SGPU_CUDA(ctx, g_cnt.alloc(NS, ctx));
        SGPU_CUDA(ctx, cursor.alloc(NS, ctx));
        SGPU_CUDA(ctx, nf_locus.alloc(P, ctx));
        SGPU_CUDA(ctx, nf_scan.alloc(P + 1, ctx));
        {
            DevBuf<uint32_t> word_locus;
            SGPU_CUDA(ctx, word_locus.alloc(W, ctx));
            SGPU_LAUNCH(ctx, (word_locus_kernel<<<locus_grid, TB, 0, st>>>(p->d_row_ptr, P, W, word_locus.p)));
            SGPU_LAUNCH(ctx, (sp_list_kernel<<<blocks_for(W), TB, 0, st>>>(out->sp_bits.p, out->sp_rank.p, W, p->d_row_ptr, word_locus.p,
                                                                            out->sp_entry.p, sp_first.p, out->sp_locus.p)));
        }
        SGPU_LAUNCH(ctx, (sp_start_kernel<<<blocks_for(P + 1), TB, 0, st>>>(out->sp_locus.p, NS, P, out->sp_start.p)));
        return SGPU_OK;
    }

    // reads from the links: first entry of every read, entry lists, mate rule. careful = false: two sweeps settle every
    // read whose entries all lie within L bp of its first one (a third one verifies); careful = true (only after the fast
    // pass reported a read id chained over >= L bp): from cleared error and statistics words, sweep until nothing moves,
    // then split such chains into reads
    int build_reads(bool careful) {
        if (careful) {
            SGPU_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, 2 * sizeof(int), st));
            SGPU_CUDA(ctx, cudaMemsetAsync(d_stats.p, 0, 2 * sizeof(unsigned long long), st));
            out->n_tail = 0;
        }
        if (NS == 0) {
            return SGPU_OK;
        }
        SGPU_CUDA(ctx, cudaMemsetAsync(g_cnt.p, 0, NS * sizeof(uint32_t), st));
        SGPU_CUDA(ctx, cudaMemsetAsync(cursor.p, 0, NS * sizeof(uint32_t), st));
        SGPU_CUDA(ctx, cudaMemsetAsync(out->g_nst.p, 0, NS * sizeof(uint32_t), st));
        SGPU_CUDA(ctx, cudaMemsetAsync(out->sp_drop.p, 0, NS, st));
        if (!careful) {
            for (int sweep = 0; sweep < 3; ++sweep) {
                SGPU_LAUNCH(ctx, (link_min_kernel<<<blocks_for(NL), TB, 0, st>>>(links.p, NL, out->sp_bits.p, out->sp_rank.p, sp_first.p,
                                                                                 d_err.p + 1)));
                if (sweep == 1) {
                    SGPU_CUDA(ctx, cudaMemsetAsync(d_err.p + 1, 0, sizeof(int), st)); // only the verifying sweep counts
                }
            }
        } else {
            SGPU_CUDA(ctx, cudaMemcpyAsync(sp_first.p, out->sp_entry.p, NS * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
            for (int sweep = 0;; ++sweep) {
                SGPU_CUDA(ctx, cudaMemsetAsync(d_err.p + 1, 0, sizeof(int), st));
                SGPU_LAUNCH(ctx, (link_min_kernel<<<blocks_for(NL), TB, 0, st>>>(links.p, NL, out->sp_bits.p, out->sp_rank.p, sp_first.p,
                                                                                 d_err.p + 1)));
                SGPU_CUDA(ctx, cudaMemcpyAsync(&hs->count, d_err.p + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
                SGPU_CUDA(ctx, cudaStreamSynchronize(st));
                if (static_cast<uint32_t>(hs->count) == 0) {
                    break;
                }
                if (sweep > 100000) {
                    return sgpu_fail(ctx, SGPU_E_FRAGMENT_SPAN, "read linking did not settle");
                }
            }
        }
        auto group = [&]() -> int {
            SGPU_LAUNCH(ctx, (group_count_kernel<<<blocks_for(NS), TB, 0, st>>>(out->sp_bits.p, out->sp_rank.p, sp_first.p, NS, out->sp_head.p, g_cnt.p)));
            SGPU_TRY(sgpu_scan_u32_u64(ctx, g_cnt.p, out->g_off.p, NS));
            SGPU_LAUNCH(ctx, (group_fill_kernel<<<blocks_for(NS), TB, 0, st>>>(out->sp_head.p, out->sp_locus.p, out->g_off.p, NS, cursor.p,
                                                                               out->g_list.p)));
            return SGPU_OK;
        };
        SGPU_TRY(group());
        if (careful) {
            DevBuf<unsigned long long> d_splits;
            SGPU_CUDA(ctx, d_splits.alloc(1, ctx));
            SGPU_CUDA(ctx, cudaMemsetAsync(d_splits.p, 0, sizeof(unsigned long long), st));
            SGPU_LAUNCH(ctx, (split_span_kernel<<<blocks_for(NS), TB, 0, st>>>(out->sp_head.p, out->sp_entry.p, out->sp_locus.p, out->g_off.p, NS,
                                                                               out->g_list.p, p->d_position, L, sp_first.p, d_splits.p)));
            SGPU_CUDA(ctx, cudaMemcpyAsync(&hs->count, d_splits.p, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
            SGPU_CUDA(ctx, cudaStreamSynchronize(st));
            out->n_span_splits = hs->count;
            SGPU_CUDA(ctx, cudaMemsetAsync(g_cnt.p, 0, NS * sizeof(uint32_t), st));
            SGPU_CUDA(ctx, cudaMemsetAsync(cursor.p, 0, NS * sizeof(uint32_t), st));
            SGPU_TRY(group());
        }
        SGPU_LAUNCH(ctx, (nonfirst_kernel<<<locus_grid, TB, 0, st>>>(out->sp_head.p, out->sp_start.p, P, nf_locus.p)));
        SGPU_GB(p, SGPU_LAUNCH(ctx, (mate_rule_kernel<GB><<<blocks_for(NS), TB, 0, st>>>(out->sp_head.p, out->sp_entry.p, out->sp_locus.p, out->g_off.p, NS,
                                                                          out->g_list.p, out->g_base.p, gid_base_, p->d_position, L,
                                                                          out->sp_drop.p, out->g_nst.p, d_err.p))));
        SGPU_TRY(sgpu_scan_u32_u64(ctx, nf_locus.p, nf_scan.p, P));
        return SGPU_OK;
    }

    int read_bases() {
        SGPU_TRACE(ctx, "link: groups+mate rule");
        SGPU_LAUNCH(ctx, (readbase_kernel<<<blocks_for(P + 1), TB, 0, st>>>(p->d_row_ptr, NS ? nf_scan.p : nullptr, P, readbase.p)));
        return SGPU_OK;
    }

    // the cutoff K per chromosome. h_whole (null: all) flags the chromosomes the pileup holds whole; of the others it holds
    // the END, and resolved[c] = 0 if that is too short to decide the cutoff (cutoff_kernel)
    int launch_cutoff(uint32_t num_threads, const uint8_t *h_whole = nullptr, DevBuf<uint8_t> *resolved = nullptr) {
        DevBuf<uint8_t> d_whole;
        DevBuf<uint64_t> exact_from;
        if (h_whole) {
            SGPU_CUDA(ctx, d_whole.alloc(p->n_chr, ctx));
            SGPU_CUDA(ctx, resolved->alloc(p->n_chr, ctx));
            SGPU_CUDA(ctx, exact_from.alloc(p->n_chr, ctx));
            SGPU_CUDA(ctx, cudaMemcpyAsync(d_whole.p, h_whole, p->n_chr, cudaMemcpyHostToDevice, st));
            SGPU_LAUNCH(ctx, (exact_from_kernel<<<(p->n_chr + 63) / 64, 64, 0, st>>>(p->d_chr_ptr, p->n_chr, p->d_position, L, d_whole.p, exact_from.p)));
        }
        SGPU_LAUNCH(ctx, (cutoff_kernel<<<p->n_chr, CUT_THREADS, 0, st>>>(p->d_chr_ptr, p->n_chr, p->d_position, readbase.p, L, num_threads,
                                                                          n_tail_reads.p, out->tail_locus.p, exact_from.p,
                                                                          h_whole ? resolved->p : nullptr)));
        return SGPU_OK;
    }

    // the cutoff of a whole call; a piece of the chromosomes (range) gets it from outside (sgpu_chromosome_cutoff) or, for
    // SGPU_TAIL_AUTO, from the piece itself, and its owned loci [own_lo[c], own_hi[c]) from positions
    int cutoff(uint32_t num_threads, const RangeSpec *range, DevBuf<uint64_t> &own_lo, DevBuf<uint64_t> &own_hi) {
        if (!range) {
            return launch_cutoff(num_threads);
        }
        DevBuf<uint32_t> spec;
        SGPU_CUDA(ctx, spec.alloc(3 * static_cast<size_t>(p->n_chr), ctx));
        SGPU_CUDA(ctx, own_lo.alloc(p->n_chr, ctx));
        SGPU_CUDA(ctx, own_hi.alloc(p->n_chr, ctx));
        SGPU_CUDA(ctx, out->owned.alloc(P, ctx));
        SGPU_CUDA(ctx, cudaMemcpyAsync(spec.p, range->own_pos_begin, p->n_chr * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        SGPU_CUDA(ctx, cudaMemcpyAsync(spec.p + p->n_chr, range->own_pos_end, p->n_chr * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        SGPU_CUDA(ctx, cudaMemcpyAsync(spec.p + 2 * p->n_chr, range->tail_position, p->n_chr * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        SGPU_CUDA(ctx, cudaMemsetAsync(n_tail_reads.p, 0, p->n_chr * sizeof(uint64_t), st));
        // SGPU_TAIL_AUTO: the piece holds the END of the chromosome (all of it if the piece starts the chromosome)
        bool any_auto = false;
        std::vector<uint8_t> h_whole(p->n_chr, 0);
        for (uint32_t c = 0; c < p->n_chr; ++c) {
            any_auto = any_auto || range->tail_position[c] == SGPU_TAIL_AUTO;
            h_whole[c] = range->own_pos_begin[c] == 0;
        }
        DevBuf<uint8_t> d_resolved;
        if (any_auto) {
            SGPU_TRY(launch_cutoff(num_threads, h_whole.data(), &d_resolved));
        }
        SGPU_LAUNCH(ctx, (range_bounds_kernel<<<(p->n_chr + 63) / 64, 64, 0, st>>>(p->d_chr_ptr, p->n_chr, p->d_position, spec.p, spec.p + p->n_chr,
                                                                                  spec.p + 2 * p->n_chr, out->tail_locus.p, own_lo.p, own_hi.p)));
        SGPU_LAUNCH(ctx, (owned_fill_kernel<<<blocks_for(P), TB, 0, st>>>(out->lchr.p, own_lo.p, own_hi.p, P, out->owned.p)));
        std::vector<uint8_t> h_resolved(p->n_chr, 1);
        if (any_auto) {
            SGPU_CUDA(ctx, cudaMemcpyAsync(h_resolved.data(), d_resolved.p, p->n_chr, cudaMemcpyDeviceToHost, st));
        }
        SGPU_CUDA(ctx, cudaStreamSynchronize(st)); // the caller's arrays are pageable
        for (uint32_t c = 0; c < p->n_chr; ++c) {
            if (range->tail_position[c] == SGPU_TAIL_AUTO && !h_resolved[c]) {
                return sgpu_fail(ctx, SGPU_E_ARG, "chromosome %u of the piece: too short to decide the tail cutoff from it (SGPU_TAIL_AUTO); "
                                 "use sgpu_chromosome_cutoff with a longer suffix", c);
            }
        }
        return SGPU_OK;
    }

    int finish() {
        if (NS) {
            const unsigned fin_grid = std::min<unsigned>(blocks_for(NS), static_cast<unsigned>(ctx->sm_count) * 16u);
            SGPU_GB(p, SGPU_LAUNCH(ctx, (sp_finish_kernel<GB><<<fin_grid, TB, 0, st>>>(out->sp_head.p, out->sp_entry.p, out->sp_locus.p, out->sp_drop.p,
                                                                              out->g_nst.p, gid_base_, out->lchr.p, out->tail_locus.p,
                                                                              out->gmap.p, out->n_groups, out->num_cells, NS, out->sp_code.p,
                                                                              out->sp_rcode.p, d_stats.p, d_err.p))));
            SGPU_TRY(sgpu_link_candidates(ctx, out, 2));
        }
        SGPU_CUDA(ctx, cudaGetLastError());
        SGPU_TRACE(ctx, "link: cutoff+finish");
        return SGPU_OK;
    }

    // scalars to the host: errors, stats, reads created, tail loci per chromosome; then the lists of tail loci and, for a
    // piece, of owned loci
    int collect(bool careful, const RangeSpec *range, const DevBuf<uint64_t> &own_lo, const DevBuf<uint64_t> &own_hi) {
        std::vector<uint64_t> h_nt(p->n_chr), h_tl(p->n_chr);
        SGPU_CUDA(ctx, cudaMemcpyAsync(h_tl.data(), out->tail_locus.p, p->n_chr * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaMemcpyAsync(h_nt.data(), n_tail_reads.p, p->n_chr * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaMemcpyAsync(&hs->err, d_err.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaMemcpyAsync(&hs->n_dropped, d_stats.p, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaMemcpyAsync(&hs->n_reads, readbase.p + P, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        SGPU_TRY(status(careful, true));
        out->n_dropped = hs->n_dropped;
        out->n_multi = hs->n_multi;
        out->n_reads = hs->n_reads;
        std::vector<uint32_t> h_tail_loci, h_own_loci;
        std::vector<uint64_t> h_lo(p->n_chr), h_hi(p->n_chr);
        out->h_tail_locus = h_tl;
        if (range) {
            SGPU_CUDA(ctx, cudaMemcpyAsync(h_lo.data(), own_lo.p, p->n_chr * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
            SGPU_CUDA(ctx, cudaMemcpyAsync(h_hi.data(), own_hi.p, p->n_chr * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
            SGPU_CUDA(ctx, cudaStreamSynchronize(st));
        }
        for (uint32_t c = 0; c < p->n_chr; ++c) {
            out->n_tail += h_nt[c];
            const uint64_t lo = range ? h_lo[c] : p->h_chr_ptr[c], hi = range ? h_hi[c] : p->h_chr_ptr[c + 1];
            for (uint64_t l = std::max(h_tl[c], lo); l < hi; ++l) { // tail x tail pairs are taken out at the OWNED loci only
                h_tail_loci.push_back(static_cast<uint32_t>(l));
            }
            if (range) {
                for (uint64_t l = lo; l < hi; ++l) {
                    h_own_loci.push_back(static_cast<uint32_t>(l));
                }
            }
        }
        if (range) {
            out->n_own = h_own_loci.size();
            SGPU_CUDA(ctx, out->own_loci.alloc(h_own_loci.size() ? h_own_loci.size() : 1, ctx));
            if (!h_own_loci.empty()) {
                SGPU_CUDA(ctx, cudaMemcpyAsync(out->own_loci.p, h_own_loci.data(), h_own_loci.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
                SGPU_CUDA(ctx, cudaStreamSynchronize(st));
            }
        }
        SGPU_TRACE(ctx, "link: scalars");
        out->n_tail_loci = h_tail_loci.size();
        SGPU_CUDA(ctx, out->tail_loci.alloc(h_tail_loci.size() ? h_tail_loci.size() : 1, ctx));
        if (!h_tail_loci.empty()) {
            SGPU_CUDA(ctx, cudaMemcpyAsync(out->tail_loci.p, h_tail_loci.data(), h_tail_loci.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
            SGPU_CUDA(ctx, cudaStreamSynchronize(st)); // h_tail_loci is pageable
        }
        return SGPU_OK;
    }
};

} // namespace

int sgpu_link_reads(sgpu_ctx *ctx, const sgpu_pileup *p, uint32_t num_cells, uint32_t L,
                    const uint32_t *h_group_id_to_pos, uint32_t n_groups, uint32_t num_threads,
                    LinkResult *out, const RangeSpec *range) {
    ReadLinker k(ctx, p, out, L);
    SGPU_TRY(k.prepare(num_cells, h_group_id_to_pos, n_groups, num_threads, range != nullptr));
    if (k.E == 0 || k.P == 0) {
        return SGPU_OK;
    }
    SGPU_TRY(k.link_entries());
    SGPU_TRY(k.number_special());
    auto pass = [&](bool careful) -> int {
        DevBuf<uint64_t> own_lo, own_hi;
        SGPU_TRY(k.build_reads(careful));
        SGPU_TRY(k.read_bases());
        SGPU_TRY(k.cutoff(num_threads, range, own_lo, own_hi));
        SGPU_TRY(k.finish());
        return k.collect(careful, range, own_lo, own_hi);
    };
    const int rc = pass(false);
    return rc == LINK_CAREFUL ? pass(true) : rc;
}

int sgpu_link_candidates(sgpu_ctx *ctx, LinkResult *out, uint32_t min_nst) {
    cudaStream_t st = ctx->stream;
    const uint64_t NS = out->n_special;
    if (NS == 0) {
        return SGPU_OK;
    }
    DevBuf<uint32_t> me_flag, me_tmp;
    SGPU_CUDA(ctx, me_flag.alloc(NS, ctx));
    SGPU_CUDA(ctx, me_tmp.alloc(NS, ctx));
    if (out->me_idx.p == nullptr) {
        SGPU_CUDA(ctx, out->me_idx.alloc(NS + 1, ctx));
        SGPU_CUDA(ctx, out->me_code.alloc(NS, ctx));
        SGPU_CUDA(ctx, out->me_locus.alloc(NS, ctx));
        SGPU_CUDA(ctx, out->me_pos.alloc(NS, ctx));
        SGPU_CUDA(ctx, out->me_beg.alloc(NS, ctx));
        SGPU_CUDA(ctx, out->me_end.alloc(NS, ctx));
    }
    SGPU_LAUNCH(ctx, (me_flag_kernel<<<blocks_for(NS), TB, 0, st>>>(out->sp_code.p, out->sp_head.p, out->sp_locus.p, out->g_off.p, out->g_list.p,
                                                                    out->g_nst.p, NS, min_nst, me_flag.p, me_tmp.p)));
    SGPU_TRY(sgpu_scan_u32_u64(ctx, me_flag.p, out->me_idx.p, NS));
    SGPU_LAUNCH(ctx, (me_compact_kernel<<<blocks_for(NS), TB, 0, st>>>(me_flag.p, me_tmp.p, out->me_idx.p, out->sp_code.p, out->sp_head.p,
                                                                       out->sp_locus.p, out->g_off.p, out->g_nst.p, NS, out->me_code.p,
                                                                       out->me_locus.p, out->me_pos.p, out->me_beg.p, out->me_end.p)));
    SGPU_CUDA(ctx, cudaGetLastError());
    return SGPU_OK;
}

// dense per-entry codes for the pair-scatter kernel
int sgpu_link_dense_codes(sgpu_ctx *ctx, const sgpu_pileup *p, LinkResult *lr) {
    cudaStream_t st = ctx->stream;
    const uint64_t E = p->n_entries, P = p->n_loci;
    SGPU_CUDA(ctx, lr->code.alloc(E ? E : 1, ctx));
    if (E == 0 || P == 0) {
        return SGPU_OK;
    }
    DevBuf<int> d_err;
    SGPU_CUDA(ctx, d_err.alloc(1, ctx));
    SGPU_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(int), st));
    const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(P, static_cast<uint64_t>(ctx->sm_count) * 16));
    SGPU_GB(p, SGPU_LAUNCH(ctx, (dense_codes_kernel<GB><<<grid, TB, 0, st>>>(p->d_row_ptr, gid_base_, lr->lchr.p, lr->tail_locus.p, lr->gmap.p,
                                                              lr->n_groups, lr->num_cells, P, lr->code.p, d_err.p))));
    if (lr->n_special) {
        SGPU_LAUNCH(ctx, (sp_codes_kernel<<<blocks_for(lr->n_special), TB, 0, st>>>(lr->sp_entry.p, lr->sp_code.p, lr->n_special, lr->code.p)));
    }
    SGPU_CUDA(ctx, cudaGetLastError());
    SGPU_CUDA(ctx, cudaMemcpyAsync(&ctx->h_scratch[0], d_err.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    SGPU_CUDA(ctx, cudaStreamSynchronize(st));
    if (static_cast<int>(ctx->h_scratch[0] & 0xFFFFFFFFu) != 0) {
        return sgpu_fail(ctx, SGPU_E_CELL_RANGE, "%s", MSG_CELL_RANGE);
    }
    return SGPU_OK;
}
int sgpu_cutoff_from_suffix(sgpu_ctx *ctx, const sgpu_pileup *p, uint32_t L, uint32_t num_threads, const uint8_t *h_whole,
                            uint32_t *h_tail_position, uint8_t *h_resolved) {
    for (uint32_t c = 0; c < p->n_chr; ++c) { // chromosomes without loci: nothing is tail, trivially decided
        h_tail_position[c] = 0xFFFFFFFFu;
        h_resolved[c] = 1;
    }
    if (p->n_entries == 0 || p->n_loci == 0) {
        return SGPU_OK;
    }
    LinkResult lr;
    ReadLinker k(ctx, p, &lr, L);
    const uint32_t none = 0;
    SGPU_TRY(k.prepare(1, &none, 0, num_threads, false));
    SGPU_TRY(k.link_entries());
    SGPU_TRY(k.number_special());
    auto pass = [&](bool careful) -> int {
        SGPU_TRY(k.build_reads(careful));
        SGPU_TRY(k.read_bases());
        DevBuf<uint8_t> d_resolved;
        SGPU_TRY(k.launch_cutoff(num_threads, h_whole, &d_resolved));
        DevBuf<uint32_t> d_tailpos;
        SGPU_CUDA(ctx, d_tailpos.alloc(p->n_chr, ctx));
        SGPU_LAUNCH(ctx, (tail_position_kernel<<<(p->n_chr + 63) / 64, 64, 0, k.st>>>(p->d_chr_ptr, p->n_chr, p->d_position, lr.tail_locus.p,
                                                                                      d_tailpos.p)));
        SGPU_CUDA(ctx, cudaGetLastError());
        SGPU_CUDA(ctx, cudaMemcpyAsync(h_tail_position, d_tailpos.p, p->n_chr * sizeof(uint32_t), cudaMemcpyDeviceToHost, k.st));
        SGPU_CUDA(ctx, cudaMemcpyAsync(h_resolved, d_resolved.p, p->n_chr, cudaMemcpyDeviceToHost, k.st));
        SGPU_CUDA(ctx, cudaMemcpyAsync(&k.hs->err, k.d_err.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, k.st));
        SGPU_CUDA(ctx, cudaStreamSynchronize(k.st));
        return k.status(careful, false);
    };
    const int rc = pass(false);
    return rc == LINK_CAREFUL ? pass(true) : rc;
}
