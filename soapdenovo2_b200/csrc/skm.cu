// skm.cu -- aggregated pass 1 (the default insert path, and the ONLY one across GPUs): super-k-mer partition per chunk, run records
// scattered straight into the memory of the GPU that owns their bucket, one shared-memory aggregation per bucket, ONE global table
// update per distinct k-mer.  Logic shared with the host tests lives in skm.cuh.
//
//   feed_text(chunk):  k_skm_count    minimizers of every read -> runs, run count per bucket, runs kept in a side buffer
//                      device_scan    bucket counts -> offsets of the chunk's bucket-major record blob
//                      k_skm_publish  reserves room for the blob in every owner's arena (sender-private region: no coordination),
//                                     writes the segment descriptor and the owner's slice of the offsets INTO THE OWNER'S MEMORY
//                      k_skm_scatter  builds the self-contained records and stores each one at its final position in its owner's
//                                     arena: plain stores for the local GPU, NVLink peer stores (CUDA IPC / peer access mappings)
//                                     for the others.  Partition and "all-to-all" are the same kernel; no library collective, no
//                                     staging buffer, no second pass over the records.
//   flush (end of pass 1 / arena full):  k_skm_apply over the owned buckets; buckets whose worst case does not fit the global table
//                                     are deferred, the table grows, the deferred buckets run again.  When the launch is the whole
//                                     pass (the normal case) the end-of-pass sweeps -- delow, linear flag, coverage histogram
//                                     (thread_delow / thread_mark / freqStat, prlHashReads.c:953-1132) -- are applied to every
//                                     entry as it is stored: no separate pass over the table.
// Replaces, for the same result, chopKmer4read + the owner filter + put_kmerset (prlHashReads.c:163-259, 79-90; newhash.c:473-528).
#include "engine_impl.cuh"
#include "skm.cuh"
#include "scan.cuh"

namespace pgb {

constexpr int SKM_PART_THREADS = 128;
constexpr int SKM_APPLY_THREADS = 256;
// Shared-memory table of a bucket: 1024 slots (32 KB at K <= 63) and at most 42 registers per thread put 6 CTAs = 48 warps on an SM;
// measured at configs[1] (gpurun_out/i_bench_*.json): 2048 slots / 3 CTAs 50.4 ms, 1024 / 6 CTAs 47.8 ms, 512 / 8 CTAs (32 registers,
// spills) 51.7 ms per 1.76e9 instances.  256-bit keys (48 B slots, 78 live registers) stay at 3 CTAs.
#ifndef SKM_LOG2_SLOTS
#define SKM_LOG2_SLOTS 10
#endif
#ifndef SKM_APPLY_MIN_BLOCKS
#define SKM_APPLY_MIN_BLOCKS(NW) ((NW) == 2 ? 6 : 3)
#endif
constexpr int SKM_SLOTS = 1 << SKM_LOG2_SLOTS;                       // shared-memory table slots per CTA
constexpr int SKM_SOFT_LIMIT = SKM_SLOTS - SKM_APPLY_THREADS - 64;   // claims stop here: the table can never fill up completely
constexpr int SKM_SIDE_RUNS = 16;
constexpr int SKM_MAXW = 16;                                         // GPUs of one box

// ------------------------------------------------------------------------------------------------ partition: count
struct CountEmit {
    u32* cnt;
    u32* side;
    int nrun;
    __device__ __forceinline__ void operator()(u32 b, int, int n, bool last) {
        atomicAdd(&cnt[b], 1u);
        if (nrun < SKM_SIDE_RUNS) side[nrun] = skm_side_pack(b, n, last);
        nrun++;
    }
};

__global__ void __launch_bounds__(SKM_PART_THREADS) k_skm_count(SkmGeom g, const u64* __restrict__ words, const u32* __restrict__ lens, u64 n_rec, int W64,
                                                               u32* cnt, u32* side, u8* nruns) {
    extern __shared__ u32 s_ring[];   // [g.w][blockDim.x]: one column per thread, bank = thread -> conflict-free
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < n_rec; r += (u64)gridDim.x * blockDim.x) {
        CountEmit e{cnt, side + r * SKM_SIDE_RUNS, 0};
        skm_scan_read(g, words + r * (u64)W64, (int)lens[r], s_ring + threadIdx.x, (int)blockDim.x, e);
        nruns[r] = e.nrun <= SKM_SIDE_RUNS ? (u8)e.nrun : (u8)255;
    }
}

struct BucketCntIn {
    const u32* a;
    __device__ u64 operator()(u64 i) const { return a[i]; }
};
struct BucketOffOut {
    u32* a;
    __device__ void operator()(u64 i, u64 prefix, u64) const { a[i] = (u32)prefix; }
};

// ------------------------------------------------------------------------------------------------ partition: publish + scatter
struct SkmSendArgs {
    u32 n_buckets;
    int world, rank;
    int own_shift;            // >= 0: owner(b) = b >> own_shift (power-of-two split), else the generic range search
    u32 seg_idx, max_seg, bo_stride;
    u64 cap_pair, epoch;
    const u32* segoff;        // [B] exclusive offsets of this chunk's blob (bucket-major), *total = record count
    const u64* total;
    u64* cursor;              // [world] records this GPU has already placed in owner o's region this epoch
    u64* dst_delta;           // [world] out: position of record i of bucket b = dst_delta[o] + segoff[b] + i   (mod 2^64)
    u32* dst_ok;              // [world] out: 0 = the blob does not fit owner o's region (error raised, records dropped)
    // this epoch's half of every owner's arena, as mapped into this process
    u32* peer_nseg[SKM_MAXW];
    SkmSegDesc* peer_ring[SKM_MAXW];
    u32* peer_segoff[SKM_MAXW];
    u64* peer_recs[SKM_MAXW];   // start of THIS sender's region in owner o's arena
    u64* counters;
};
__device__ __forceinline__ int skm_owner(const SkmSendArgs& a, u32 b) {
    return a.own_shift >= 0 ? (int)(b >> a.own_shift) : skm_owner_of(a.n_buckets, a.world, b);
}
__device__ __forceinline__ u32 skm_segoff_at(const SkmSendArgs& a, u32 b) { return b < a.n_buckets ? a.segoff[b] : (u32)*a.total; }

__global__ void __launch_bounds__(256) k_skm_publish(SkmSendArgs a) {
    if (blockIdx.x == 0 && (int)threadIdx.x < a.world) {
        const int o = threadIdx.x;
        const u32 lo = skm_owner_lo(a.n_buckets, a.world, o), hi = o + 1 < a.world ? skm_owner_lo(a.n_buckets, a.world, o + 1) : a.n_buckets;
        const u32 first = skm_segoff_at(a, lo), n = skm_segoff_at(a, hi) - first;
        const u64 base = a.cursor[o];
        const bool fits = base + n <= a.cap_pair;
        if (!fits) atomicAdd(&a.counters[C_XERR], 1ull);
        a.dst_ok[o] = fits ? 1u : 0u;
        a.dst_delta[o] = base - (u64)first;
        if (fits) a.cursor[o] = base + n;
        SkmSegDesc d;
        d.rec_off = base;
        d.n_recs = fits ? n : 0u;
        d.pad = 0;
        a.peer_ring[o][(u64)a.rank * a.max_seg + a.seg_idx] = d;
        a.peer_nseg[o][a.rank] = a.seg_idx + 1;
        atomicMax((unsigned long long*)&a.counters[C_XUSED], (unsigned long long)(fits ? base + n : base));   // fullest region (host-side room checks)
        if (o == 0) {
            __threadfence();
            a.counters[C_XEPOCH] = a.epoch;
            atomicAdd((unsigned long long*)&a.counters[C_XSEGS], 1ull);
        }
    }
    // the owner's slice of the offsets, relative to the blob: entry (b - lo) for its buckets, plus the end entry
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < (u64)a.n_buckets + a.world; i += (u64)gridDim.x * blockDim.x) {
        int o;
        u32 b;
        if (i < a.n_buckets) { b = (u32)i; o = skm_owner(a, b); }
        else { o = (int)(i - a.n_buckets); b = o + 1 < a.world ? skm_owner_lo(a.n_buckets, a.world, o + 1) : a.n_buckets; }   // end entry of owner o
        const u32 lo = skm_owner_lo(a.n_buckets, a.world, o);
        const u32 first = skm_segoff_at(a, lo);
        a.peer_segoff[o][((u64)a.rank * a.max_seg + a.seg_idx) * a.bo_stride + (b - lo)] = skm_segoff_at(a, b) - first;
    }
}

// A record goes out with as few stores as possible: ONE 256-bit store per 32 bytes (STG.E.256 on sm_100a) -- over NVLink every store
// is a packet, and 32-byte packets measured at only ~200 GB/s when a record was two 16-byte stores.
__device__ __forceinline__ void st256(u64* dst, u64 a, u64 b, u64 c, u64 d) {
    asm volatile("st.global.v4.u64 [%0], {%1,%2,%3,%4};" ::"l"(dst), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}
template <int NW>
__device__ __forceinline__ void skm_store_rec(u64* dst, const SkmRec<NW>& r) {
    if (NW == 2) {
        st256(dst, r.w[0], r.w[1], r.w[2], r.w[3]);                       // 32-byte records are 32-byte aligned
    } else {
        // 48-byte records: 16-byte aligned only
#pragma unroll
        for (int p = 0; p < (NW + 2) / 2; p++) {
            uint4 v;
            v.x = (unsigned)r.w[2 * p]; v.y = (unsigned)(r.w[2 * p] >> 32);
            v.z = (unsigned)r.w[2 * p + 1]; v.w = (unsigned)(r.w[2 * p + 1] >> 32);
            reinterpret_cast<uint4*>(dst)[p] = v;
        }
    }
}
template <int NW>
__device__ __forceinline__ void skm_emit_rec(const SkmSendArgs& a, u32* cursor_b, int K, const u64* wp, int W64, u64 ordinal, u32 b, int start, int n, bool last) {
    const u32 i = atomicAdd(&cursor_b[b], 1u);
    const int o = skm_owner(a, b);
    if (!a.dst_ok[o]) return;
    const u64 idx = a.dst_delta[o] + (u64)a.segoff[b] + i;
    const SkmRec<NW> r = skm_make_rec<NW>(K, wp, W64, ordinal, start, n, last);
    skm_store_rec<NW>(a.peer_recs[o] + idx * (NW + 2), r);
}

// one thread per read: the runs come from the side buffer (no minimizer work), the records go to their owners
template <int NW>
__global__ void __launch_bounds__(256) k_skm_scatter(SkmSendArgs a, int K, const u64* __restrict__ words, u64 n_rec, int W64, u64 ord_base, u64 ord_stride,
                                                     const u32* __restrict__ side, const u8* __restrict__ nruns, u32* cursor_b) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < n_rec; r += (u64)gridDim.x * blockDim.x) {
        const int nr = nruns[r];
        if (nr == 255 || nr == 0) continue;
        const u64* wp = words + r * (u64)W64;
        const u64 ordinal = ord_base + r * ord_stride;
        const uint4* row = reinterpret_cast<const uint4*>(side + r * SKM_SIDE_RUNS);
        int start = 0;
        for (int q = 0; q < nr; q += 4) {
            const uint4 v = __ldg(row + (q >> 2));
            const u32 e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int x = 0; x < 4; x++) {
                if (q + x >= nr) break;
                const int n = skm_side_n(e[x]);
                skm_emit_rec<NW>(a, cursor_b, K, wp, W64, ordinal, skm_side_bucket(e[x]), start, n, skm_side_last(e[x]));
                start += n;
            }
        }
    }
}

// reads with more than SKM_SIDE_RUNS runs (rare): full re-scan of just those reads
template <int NW>
struct RescanEmit {
    const SkmSendArgs& a;
    u32* cursor_b;
    int K;
    const u64* wp;
    int W64;
    u64 ordinal;
    __device__ __forceinline__ void operator()(u32 b, int s, int n, bool last) { skm_emit_rec<NW>(a, cursor_b, K, wp, W64, ordinal, b, s, n, last); }
};
template <int NW>
__global__ void __launch_bounds__(SKM_PART_THREADS) k_skm_rescan(SkmSendArgs a, SkmGeom g, const u64* __restrict__ words, const u32* __restrict__ lens, u64 n_rec,
                                                                int W64, u64 ord_base, u64 ord_stride, const u8* __restrict__ nruns, u32* cursor_b) {
    extern __shared__ u32 s_ring[];
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < n_rec; r += (u64)gridDim.x * blockDim.x) {
        if (nruns[r] != 255) continue;
        const u64* wp = words + r * (u64)W64;
        RescanEmit<NW> e{a, cursor_b, g.K, wp, W64, ord_base + r * ord_stride};
        skm_scan_read(g, wp, (int)lens[r], s_ring + threadIdx.x, (int)blockDim.x, e);
    }
}

// ------------------------------------------------------------------------------------------------ aggregation
// Shared-memory table of one bucket, structure of arrays: key words [NW][S], payload [S], rank [S], claim list [S] (u16).
// Claim protocol: CAS(key0, EMPTY -> w0|BUSY), write the other key words, fence, store w0.  Empty slots hold {PAYLOAD_FRESH, ~0} in
// their payload / rank words, so the claimer records its own instance together with the lanes that found the key (one update path).
// A thread that meets a BUSY key0 whose other bits match waits for the publication (independent thread scheduling: the claimer makes
// progress even inside the same warp).  The claimer also appends the slot to the claim list (the flush walks the list, not the
// table).  (Prefetching the k-mer's home slot of the GLOBAL table into L2 at claim time measured no difference and was dropped.)
// S slots (any size: the slot index is a multiply-shift range reduction of a 32-bit hash), claims stop at LIMIT so that the
// table can never fill up completely whatever the number of concurrent claimers; LT = type of the claim-list entries.
template <int NW, int S, int LIMIT, class LT>
struct SmemTable {
    u64* key;   // [NW * S]
    u64* pay;
    u64* rnk;
    LT* list;
    u32* count;
    // Two phases with a warp barrier between them (the caller's __syncwarp over the lanes that have an instance): first every lane
    // finds or claims its slot (lanes differ only in the number of probes), then the lanes that found an existing key apply their
    // instance TOGETHER (without the barrier the lanes that match on their first probe run the long update on their own while the
    // others keep probing: the update code then executes several times per step with a few active lanes each).
    // find(): 1 = key present at idx (found, or claimed by this lane just now), 3 = no room (caller spills)
    __device__ __forceinline__ int find(const Table<NW>& tab, const Kmer<NW>& k, u32& idx) const {
        idx = (u32)(((u64)skm_slot_hash(k, 32) * (u64)S) >> 32);
        volatile u64* vkey = key;
        for (int probe = 0; probe < S; probe++) {
            u64 k0 = vkey[idx];
            if (k0 == EMPTY64) {
                if (*(volatile u32*)count >= (u32)LIMIT) return 3;
                u64 old = atomicCAS(&key[idx], EMPTY64, k.w[0] | BUSY_BIT);
                if (old == EMPTY64) {
#pragma unroll
                    for (int w = 1; w < NW; w++) vkey[w * S + idx] = k.w[w];
                    __threadfence_block();
                    vkey[idx] = k.w[0];
                    const u32 n = atomicAdd(count, 1u);
                    list[n] = (LT)idx;
                    return 1;   // an empty slot holds {PAYLOAD_FRESH, ~0}: the claimer records its instance with everybody else in apply()
                }
                k0 = old;
            }
            if ((k0 & ~BUSY_BIT) == k.w[0]) {
                while (k0 & BUSY_BIT) k0 = vkey[idx];
                bool same = true;
#pragma unroll
                for (int w = 1; w < NW; w++) same = same && vkey[w * S + idx] == k.w[w];
                if (same) return 1;
            }
            idx = idx + 1 == (u32)S ? 0u : idx + 1;
        }
        return 3;
    }
    __device__ __forceinline__ void apply(u32 idx, unsigned left, unsigned right, u64 rank) const {
        volatile u64* vpay = pay;
        volatile u64* vrnk = rnk;
        u64 cur = vpay[idx];
        for (;;) {
            u64 nxt = payload_apply(cur, left, right);
            if (nxt == cur) break;
            u64 old = atomicCAS(&pay[idx], cur, nxt);
            if (old == cur) break;
            cur = old;
        }
        if (rank < vrnk[idx]) atomicMin(&rnk[idx], rank);
    }
};

// One aggregated k-mer -> the global table.  A k-mer lives in exactly one bucket and a bucket is aggregated by one CTA at a time, so
// when this call CLAIMS the slot nobody else can be touching its {payload, aux} words: they are written with one plain 16-byte store
// (probe load -> claim CAS -> store: two dependent memory round trips per new key).  A key that already exists (earlier epoch: the
// arena was flushed mid-stream; or instances of this bucket that were spilled) is merged with the same 64-bit CAS + atomicMin protocol
// every other writer uses.  `on_claim` maps the aggregate to what a claimed slot stores; a merged aggregate is stored as it is.
template <int NW, class OnClaim>
__device__ __forceinline__ bool table_merge(const Table<NW>& t, const Kmer<NW>& k, u64 agg, u64 rank, OnClaim on_claim) {
    bool claimed;
    u64 idx = table_find_or_claim(t, k, &claimed);
    Slot<NW>* s = t.slots + idx;
    if (claimed) {
        stcg128(&s->payload, U128{on_claim(agg), rank});
        return true;
    }
    u64 cur = ldcg64(&s->payload);
    for (;;) {
        u64 nxt = payload_merge(cur, agg);
        if (nxt == cur) break;
        u64 old = atomicCAS(&s->payload, cur, nxt);
        if (old == cur) break;
        cur = old;
    }
    atomicMin(&s->aux, rank);
    return false;
}

// the segments one aggregation launch reads, in device memory (built by k_skm_segs from what the senders published)
struct SkmSegList {
    const u64* recs[SKM_MAX_SEGS];
    const u32* segoff[SKM_MAX_SEGS];
    u32 n;
    u32 pad;
};
struct SkmFlushArgs {
    int world;
    u32 max_seg, bo_stride;
    u64 cap_pair;
    int rec_words;
    const u32* nseg;
    const SkmSegDesc* ring;
    const u32* segoff;
    const u64* recs;
    SkmSegList* segs;
    u64* counters;
};
__global__ void __launch_bounds__(256) k_skm_segs(SkmFlushArgs a) {
    __shared__ u32 s_base[SKM_MAXW + 1];
    if (threadIdx.x == 0) {
        u32 acc = 0;
        for (int s = 0; s < a.world; s++) { s_base[s] = acc; acc += a.nseg[s] < a.max_seg ? a.nseg[s] : a.max_seg; }
        s_base[a.world] = acc;
        if (acc > (u32)SKM_MAX_SEGS) { atomicAdd(&a.counters[C_XERR], 1ull); acc = SKM_MAX_SEGS; }
        a.segs->n = acc;
        a.counters[C_RESERVED] = a.counters[C_DISTINCT];   // keys the table already holds; the launch that follows adds its reservations
        a.counters[C_DEFER] = 0;
        a.counters[C_MAXU] = 0;
    }
    __syncthreads();
    for (int s = 0; s < a.world; s++) {
        const u32 n = s_base[s + 1] - s_base[s];
        for (u32 i = threadIdx.x; i < n; i += blockDim.x) {
            const u32 j = s_base[s] + i;
            if (j >= (u32)SKM_MAX_SEGS) continue;
            const SkmSegDesc d = a.ring[(u64)s * a.max_seg + i];
            a.segs->recs[j] = a.recs + ((u64)s * a.cap_pair + d.rec_off) * a.rec_words;
            a.segs->segoff[j] = a.segoff + ((u64)s * a.max_seg + i) * a.bo_stride;
        }
    }
}

struct SkmApplyArgs {
    const SkmSegList* segs;
    const u32* bucket_list;   // nullptr: buckets 0 .. n_list-1; else the deferred buckets of the previous launch
    u32 n_list;
    u64* counters;            // C_RESERVED: keys the table is committed to hold; C_DEFER / C_MAXU: deferred buckets, their largest bound
    u64 limit;
    u32* deferred;
    int sweep;                // 1: the flush applies the end-of-pass sweeps to every entry it stores (the launch is the whole pass)
    int D;
    u64* hist;                // [256] coverage histogram of the swept entries
    u64* spill_list;          // slots of the keys stored unswept (spilled instances): the host sweeps them afterwards
    u64 spill_cap;
};
constexpr u64 SKM_CREDIT = 1ull << 16;   // table room a CTA reserves at a time (keys)

__device__ __forceinline__ u64 shfl64(u64 v, int src) { return (u64)__shfl_sync(0xffffffffu, (unsigned long long)v, src); }

// One CTA per bucket (static round-robin over the list: buckets are hash-uniform), one shared-memory table per CTA.  Inside a bucket
// the WARPS run on their own: a warp loads 32 consecutive records of the bucket (one 32 / 48 B record per lane, coalesced), an
// inclusive scan of their k-mer counts maps instance q of the batch to (record, position), and every warp step takes 32 CONSECUTIVE
// instances -- all lanes busy whatever the run lengths -- fetching its record from the lane that holds it with shuffles.  No CTA-wide
// barrier and no staging buffer inside a bucket; the next batch's records and the next bucket's segment ranges are loaded while the
// current ones are processed.
template <int NW>
__global__ void __launch_bounds__(SKM_APPLY_THREADS, SKM_APPLY_MIN_BLOCKS(NW)) k_skm_apply(Table<NW> tab, KParams<NW> kp, SkmApplyArgs a) {
    constexpr int RW = NW + 2, WARPS = SKM_APPLY_THREADS / 32;
    extern __shared__ __align__(16) u64 s_dyn[];   // key[NW][S], pay[S], rnk[S], list[S] (u16)
    __shared__ const u64* s_ptr[SKM_MAX_SEGS];
    __shared__ u32 s_cum[SKM_MAX_SEGS + 1];
    __shared__ u32 s_warp[WARPS];
    __shared__ u32 s_count, s_defer, s_batch;
    __shared__ unsigned s_new, s_tot_new, s_tot_spill;
    __shared__ unsigned s_hist[256], s_lin, s_rem;   // the fused sweeps (a.sweep)
    SmemTable<NW, SKM_SLOTS, SKM_SOFT_LIMIT, unsigned short> st{s_dyn, s_dyn + NW * SKM_SLOTS, s_dyn + (NW + 1) * SKM_SLOTS, reinterpret_cast<unsigned short*>(s_dyn + (NW + 2) * SKM_SLOTS), &s_count};
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned lane_le = 0xffffffffu >> (31 - lane);
    for (int i = tid; i < SKM_SLOTS; i += SKM_APPLY_THREADS) {   // the flush re-empties what it merges
        st.key[i] = EMPTY64;
        st.pay[i] = PAYLOAD_FRESH;
        st.rnk[i] = ~0ull;
    }
    if (tid == 0) { s_tot_new = 0; s_tot_spill = 0; s_lin = 0; s_rem = 0; }
    static_assert(SKM_APPLY_THREADS == 256, "one histogram bin per thread");
    s_hist[tid] = 0;
    unsigned sw_lin = 0, sw_rem = 0;
    const int n_segs = (int)a.segs->n;
    const u32* my_so = tid < n_segs ? a.segs->segoff[tid] : nullptr;
    const u64* my_recs = tid < n_segs ? a.segs->recs[tid] : nullptr;
    unsigned tot_new = 0, tot_spill = 0;
    u64 credit = 0;                      // thread 0: table room this CTA holds
    u32 pos = blockIdx.x;
    u32 nlo = 0, ncnt = 0;               // this thread's segment range of the NEXT bucket
    if (pos < a.n_list && my_so) {
        const u32 b = a.bucket_list ? a.bucket_list[pos] : pos;
        nlo = my_so[b];
        ncnt = my_so[b + 1] - nlo;
    }
    for (; pos < a.n_list; pos += gridDim.x) {
        __syncthreads();   // previous bucket fully flushed (and the empty table visible on the first trip)
        const u32 cnt = ncnt;
        if (my_so) s_ptr[tid] = my_recs + (u64)nlo * RW;
        if (tid == 0) { s_count = 0; s_new = 0; s_batch = WARPS; }
        if (pos + gridDim.x < a.n_list && my_so) {
            const u32 nb = a.bucket_list ? a.bucket_list[pos + gridDim.x] : pos + gridDim.x;
            nlo = my_so[nb];
            ncnt = my_so[nb + 1] - nlo;
        }
        {
            u32 inc = cnt;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const u32 v = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane >= d) inc += v;
            }
            if (lane == 31) s_warp[wid] = inc;
            __syncthreads();
            u32 off = 0;
            for (int w = 0; w < wid; w++) off += s_warp[w];
            if (tid < n_segs) s_cum[tid] = off + inc - cnt;
            if (tid == (n_segs > 0 ? n_segs - 1 : 0)) s_cum[n_segs] = n_segs > 0 ? off + inc : 0u;
        }
        __syncthreads();
        const u32 R = s_cum[n_segs];
        // ---- room in the global table: every k-mer instance could be a new key.  Credits are taken SKM_CREDIT keys at a time.
        if (tid == 0) {
            bool defer = false;
            const u64 bound = (u64)R * SKM_MAX_RUN;
            if (credit < bound) {
                unsigned long long* res = (unsigned long long*)&a.counters[C_RESERVED];
                const u64 want = bound - credit, ask = want > SKM_CREDIT ? want : SKM_CREDIT;
                u64 old = atomicAdd(res, (unsigned long long)ask);
                if (old + ask <= a.limit) credit += ask;
                else {
                    atomicAdd(res, (unsigned long long)(0ull - ask));
                    bool got = false;
                    if (ask != want) {
                        old = atomicAdd(res, (unsigned long long)want);
                        if (old + want <= a.limit) { credit += want; got = true; }
                        else atomicAdd(res, (unsigned long long)(0ull - want));
                    }
                    if (!got) {
                        defer = true;
                        const u32 b = a.bucket_list ? a.bucket_list[pos] : pos;
                        a.deferred[atomicAdd((unsigned long long*)&a.counters[C_DEFER], 1ull)] = b;
                        atomicMax((unsigned long long*)&a.counters[C_MAXU], (unsigned long long)bound);
                    }
                }
            }
            if (!defer) credit -= bound;
            s_defer = defer ? 1u : 0u;
        }
        __syncthreads();
        if (s_defer || R == 0) {
            if (tid == 0 && !s_defer) credit += (u64)R * SKM_MAX_RUN;
            continue;
        }
        unsigned my_new = 0;
        // ---- the warps: batches of 32 records, 32 consecutive instances per step
        u64 nh = 0, nx[NW + 1];
#pragma unroll
        for (int i = 0; i < NW + 1; i++) nx[i] = 0;
        // batch size: the bucket's records are split evenly over a multiple of WARPS batches (R = 210 records on 8 warps: 8 batches of
        // 27, not 6 of 32 + 1 of 18 + an idle warp), so the warps reach the barrier before the flush together
        const u32 n_batches = (u32)WARPS * ((R + 32u * WARPS - 1) / (32u * WARPS));
        const u32 bsz = (R + n_batches - 1) / n_batches;   // <= 32
        auto load_rec = [&](u32 q) {
            nh = 0;
            if (q < R && lane < (int)bsz) {
                int lo = 0, hi = n_segs;
                while (hi - lo > 1) {
                    const int mid = (lo + hi) >> 1;
                    if (s_cum[mid] <= q) lo = mid; else hi = mid;
                }
                const uint4* p = reinterpret_cast<const uint4*>(s_ptr[lo] + (u64)(q - s_cum[lo]) * RW);
                u64 w[RW];
#pragma unroll
                for (int i = 0; i < RW / 2; i++) {
                    const uint4 v = __ldg(p + i);
                    w[2 * i] = (u64)v.x | ((u64)v.y << 32);
                    w[2 * i + 1] = (u64)v.z | ((u64)v.w << 32);
                }
                nh = w[0];
#pragma unroll
                for (int i = 0; i < NW + 1; i++) nx[i] = w[1 + i];
            }
        };
        // batches are handed out dynamically (the first WARPS ones are pre-assigned): a warp that draws short runs takes more of them,
        // so the warps reach the barrier before the flush together
        load_rec((u32)wid * bsz + lane);
        u32 nb = 0x7FFFFFFu;                                  // (a warp without a first batch must not draw one; x 32 still fits)
        if ((u32)wid * bsz < R) {
            if (lane == 0) nb = atomicAdd(&s_batch, 1u);
            nb = __shfl_sync(0xffffffffu, nb, 0);
        }
        for (u32 rb = (u32)wid * bsz; rb < R;) {
            const u64 hdr = nh;
            u64 x[NW + 1];
#pragma unroll
            for (int i = 0; i < NW + 1; i++) x[i] = nx[i];
            const u32 rb_next = nb * bsz;
            load_rec(rb_next + lane);                         // the next batch is in flight while this one is processed
            if (rb_next < R) {
                if (lane == 0) nb = atomicAdd(&s_batch, 1u);
                nb = __shfl_sync(0xffffffffu, nb, 0);
            }
            const bool valid = rb + lane < R && lane < (int)bsz;
            const u32 n = valid ? (u32)skm_rec_n(hdr) : 0u;
            u32 inc = n;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const u32 v = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane >= d) inc += v;
            }
            const u32 I = __shfl_sync(0xffffffffu, inc, 31);
            const u32 pe = inc - n;                            // first instance of this lane's record inside the batch
            for (u32 q0 = 0; q0 < I; q0 += 32) {
                const u32 q = q0 + lane;
                const bool has = q < I;
                // record of instance q: the record that holds q0, plus the records that start at window positions 1 .. lane
                const unsigned starts = __reduce_or_sync(0xffffffffu, (valid && pe > q0 && pe - q0 < 32u) ? 1u << (pe - q0) : 0u);
                const int first = __popc(__ballot_sync(0xffffffffu, valid && pe <= q0)) - 1;
                const int src = (first + __popc(starts & lane_le)) & 31;
                const int t = (int)(q - __shfl_sync(0xffffffffu, pe, src));
                const u64 h = shfl64(hdr, src);
                u64 y[NW + 1];
#pragma unroll
                for (int i = 0; i < NW + 1; i++) y[i] = shfl64(x[i], src);
                const unsigned has_mask = __ballot_sync(0xffffffffu, has);
                if (has) {
                    const SkmInst<NW> in = skm_instance_rec<NW>(kp, h, y, t);
                    const u64 rank = skm_rec_rank(h, t);
                    u32 slot;
                    const int state = st.find(tab, in.canon, slot);
                    __syncwarp(has_mask);   // the lanes re-join before the counter update (see SmemTable)
                    if (state == 1) st.apply(slot, in.left, in.right, rank);
                    else if (state == 3) {
                        // bucket holds more distinct k-mers than the shared-memory table: this instance goes to HBM directly (same result)
                        u64 at;
                        const bool fresh = table_insert(tab, in.canon, in.left, in.right, rank, &at);
                        my_new += fresh;
                        tot_spill++;
                        if (fresh && a.sweep) {   // its other instances follow the same way: swept after the launch, from this list
                            const u64 n = atomicAdd((unsigned long long*)&a.counters[C_SPILLKEYS], 1ull);
                            if (n < a.spill_cap) a.spill_list[n] = at;
                        }
                    }
                }
                __syncwarp();
            }
            rb = rb_next;
        }
        __syncthreads();
        // ---- flush: one global update per distinct k-mer of the bucket, walking the claim list (every thread busy).
        // With a.sweep (this launch is the whole pass, into an empty table) an aggregate is swept only when this flush CLAIMS the key's
        // global slot: every instance of the bucket has been applied (barrier above) and none of them reached the table, so the
        // aggregate is the whole entry.  A key that is already there got there in this launch from instances of this bucket that
        // were spilled (a warp saw its slot still empty and the claim count at the limit while another warp claimed it): that
        // aggregate is partial, so it is merged unswept.  The first spilled instance put the slot on the spill list, which
        // k_sweep_list sweeps after the launch, or found the list full, which makes the host sweep the whole table.
        const u32 n_claimed = s_count;
        for (u32 i = tid; i < n_claimed; i += SKM_APPLY_THREADS) {
            const u32 idx = st.list[i];
            Kmer<NW> k;
#pragma unroll
            for (int w = 0; w < NW; w++) k.w[w] = st.key[w * SKM_SLOTS + idx];
            const bool fresh = table_merge(tab, k, st.pay[idx], st.rnk[idx],
                                           [&](u64 agg) { return a.sweep ? sweep_payload(agg, a.D, sw_rem, sw_lin, s_hist) : agg; });
            my_new += fresh;
            st.key[idx] = EMPTY64;
            st.pay[idx] = PAYLOAD_FRESH;
            st.rnk[idx] = ~0ull;
        }
        if (my_new) atomicAdd(&s_new, my_new);
        tot_new += my_new;
        __syncthreads();
        if (tid == 0) credit += (u64)R * SKM_MAX_RUN - (u64)s_new;   // what the bound over-reserved stays with the CTA
    }
    __syncthreads();
    if (tid == 0 && credit) atomicAdd((unsigned long long*)&a.counters[C_RESERVED], (unsigned long long)(0ull - credit));
    if (tot_new) atomicAdd(&s_tot_new, tot_new);
    if (tot_spill) atomicAdd(&s_tot_spill, tot_spill);
    if (sw_lin) atomicAdd(&s_lin, sw_lin);
    if (sw_rem) atomicAdd(&s_rem, sw_rem);
    __syncthreads();
    if (tid == 0) {
        if (s_tot_new) atomicAdd(&a.counters[C_DISTINCT], (u64)s_tot_new);
        if (s_tot_spill) atomicAdd(&a.counters[C_MISC2], (u64)s_tot_spill);
        if (s_lin) atomicAdd(&a.counters[C_LINEAR], (u64)s_lin);
        if (s_rem) atomicAdd(&a.counters[C_REMOVED], (u64)s_rem);
    }
    if (a.sweep && s_hist[tid]) atomicAdd(&a.hist[tid], (u64)s_hist[tid]);
}

// ------------------------------------------------------------------------------------------------ host side
template <int NW>
static constexpr size_t skm_apply_smem() {
    return (size_t)(NW + 2) * SKM_SLOTS * sizeof(u64) + (size_t)SKM_SLOTS * sizeof(unsigned short);
}
static u64 next_pow2_u64(u64 x) { u64 p = 1; while (p < x) p <<= 1; return p; }

template <int NW>
void EngineT<NW>::skm_init() {
    if (skm_geom_.n_buckets) return;
    const int world = prm_.world > 1 ? prm_.world : 1;
    if (world > SKM_MAXW) throw std::runtime_error("pgb200: at most 16 GPUs");
    u64 est = 0;   // expected number of distinct k-mers on THIS GPU
    if (prm_.table_slots) est = prm_.table_slots / 2;
    else if (prm_.initG) est = (u64)((double)prm_.P * (double)ref_static_set_size(prm_.initG, prm_.P, prm_.flavour127 != 0) * 0.77) / world;
    u64 Bo = est ? next_pow2_u64((est + SKM_SLOTS / 2 - 1) / (SKM_SLOTS / 2)) : (1ull << 16);   // half a shared-memory table per bucket on average
    if (Bo < 1024) Bo = 1024;
    u64 B = Bo * world;
    if (const char* e = getenv("PGB200_SKM_BUCKETS")) B = strtoull(e, nullptr, 0);
    if (B < (u64)world) B = world;
    if (B > (1ull << SKM_MAX_BUCKET_BITS)) B = 1ull << SKM_MAX_BUCKET_BITS;   // the side buffer packs the bucket in 26 bits
    skm_geom_ = make_skm_geom(prm_.K, (u32)B);
    skm_own_lo_ = skm_owner_lo((u32)B, world, prm_.rank);
    skm_own_hi_ = prm_.rank + 1 < world ? skm_owner_lo((u32)B, world, prm_.rank + 1) : (u32)B;
    skm_own_shift_ = -1;
    if ((B & (B - 1)) == 0 && (world & (world - 1)) == 0 && B >= (u64)world) {
        int s = 0;
        while (((u64)world << s) < B) s++;
        skm_own_shift_ = s;
    }
    skm_cnt_.alloc((B + 1) * sizeof(u32));
    skm_segoff_.alloc((B + 1) * sizeof(u32));
    skm_cursor_.alloc((B + 1) * sizeof(u32));
    skm_scan_.alloc(scan_scratch_elems(B) * sizeof(u64) + 256);
    // device-side scratch: sender cursors [world], dst_delta [world], dst_ok [world], next-bucket counter, segment list, deferred lists
    skm_misc_.alloc(4096 + sizeof(SkmSegList) + 2 * (size_t)(skm_own_hi_ - skm_own_lo_ + 1) * sizeof(u32));
    PG_CUDA(cudaMemsetAsync(skm_misc_.p, 0, skm_misc_.bytes, st_));
    for (auto& e : ev_skm_) PG_CUDA(cudaEventCreate(&e));
    skm_part_threads_ = SKM_PART_THREADS;
    while ((size_t)skm_part_threads_ * skm_geom_.w * sizeof(u32) > 160 * 1024 && skm_part_threads_ > 32) skm_part_threads_ /= 2;
    const size_t ring = (size_t)skm_part_threads_ * skm_geom_.w * sizeof(u32);
    if (ring > 48 * 1024) {
        PG_CUDA(cudaFuncSetAttribute(k_skm_count, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ring));
        PG_CUDA(cudaFuncSetAttribute(k_skm_rescan<NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ring));
    }
    PG_CUDA(cudaFuncSetAttribute(k_skm_apply<NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)skm_apply_smem<NW>()));
    if (prm_.verbose) fprintf(stderr, "[pgb200] aggregated pass 1: %u buckets (%u owned by GPU %d of %d), minimizer length %d, window %d\n", skm_geom_.n_buckets,
                              skm_own_hi_ - skm_own_lo_, prm_.rank, world, skm_geom_.m, skm_geom_.w);
}

// ---- the exchange arena
template <int NW>
void EngineT<NW>::xchg_setup(uint64_t cap_records) {
    skm_init();
    const int world = prm_.world > 1 ? prm_.world : 1;
    if (xa_buf_.p) throw std::runtime_error("pgb200: exchange arena already set up");
    if (!cap_records) {   // default: a fifth of the free HBM, at most 32 GB, split into the two epoch halves
        create_table_if_needed();
        size_t free_b = 0, total_b = 0;
        PG_CUDA(cudaMemGetInfo(&free_b, &total_b));
        u64 bytes = std::min<u64>((u64)free_b / 5, 32ull << 30);
        if (const char* e = getenv("PGB200_SKM_ARENA_MB")) bytes = strtoull(e, nullptr, 0) << 20;
        cap_records = bytes / ((NW + 2) * sizeof(u64)) / 2;
    }
    u64 cap_pair = cap_records / world;
    if (cap_pair < 4096) cap_pair = 4096;
    u32 max_seg = (u32)(SKM_MAX_SEGS / world);   // an aggregation launch reads at most SKM_MAX_SEGS segments over all senders
    if (const char* e = getenv("PGB200_SKM_MAX_SEG")) max_seg = (u32)atoi(e);
    if (max_seg < 1) max_seg = 1;
    if (max_seg > (u32)SKM_MAX_SEGS) max_seg = SKM_MAX_SEGS;
    xa_geom_ = make_skm_arena_geom(world, skm_geom_.n_buckets, max_seg, cap_pair, NW + 2);
    xa_halves_ = 2;   // epoch parity: an epoch is aggregated (asynchronously) while the next one is being delivered
    xa_buf_.alloc(xa_geom_.half_bytes * xa_halves_);
    for (int h = 0; h < xa_halves_; h++)
        PG_CUDA(cudaMemsetAsync(static_cast<char*>(xa_buf_.p) + h * xa_geom_.half_bytes, 0, xa_geom_.off_recs, st_));   // nseg, ring, offsets
    sync();
    xa_peer_.assign(world, nullptr);
    xa_peer_[prm_.rank] = xa_buf_.p;
    xa_send_epoch_ = 0;
    xa_seg_idx_ = 0;
    xa_flushed_epoch_ = 0;
    xa_reads_cum_.assign(1, 0);
    if (prm_.verbose) fprintf(stderr, "[pgb200] exchange arena: %d x %.2f GB (%llu records per sender, %u segments per sender and epoch)\n", xa_halves_,
                              xa_geom_.half_bytes / 1e9, (unsigned long long)cap_pair, max_seg);
}
template <int NW>
void EngineT<NW>::xchg_export(void* handle64) {
    if (!xa_buf_.p) throw std::runtime_error("pgb200: xchg_export before xchg_setup");
    cudaIpcMemHandle_t h;
    PG_CUDA(cudaIpcGetMemHandle(&h, xa_buf_.p));
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(handle64, &h, 64);
}
template <int NW>
void EngineT<NW>::xchg_import(int peer, const void* handle64) {
    if (peer < 0 || peer >= (int)xa_peer_.size() || peer == prm_.rank) throw std::runtime_error("pgb200: xchg_import: bad peer");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    void* p = nullptr;
    PG_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    xa_peer_[peer] = p;
    xa_ipc_opened_.push_back(p);
}
template <int NW>
void EngineT<NW>::xchg_import_ptr(int peer, int peer_device, void* base) {
    if (peer < 0 || peer >= (int)xa_peer_.size() || peer == prm_.rank) throw std::runtime_error("pgb200: xchg_import_ptr: bad peer");
    PG_CUDA(cudaSetDevice(prm_.device));
    int can = 0;
    PG_CUDA(cudaDeviceCanAccessPeer(&can, prm_.device, peer_device));
    if (!can) throw std::runtime_error("pgb200: GPUs cannot access each other's memory (no peer access)");
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) PG_CUDA(e);
    cudaGetLastError();
    xa_peer_[peer] = base;
}
template <int NW>
void* EngineT<NW>::xchg_base() { return xa_buf_.p; }

template <int NW>
void EngineT<NW>::xchg_default_setup() {
    if (xa_buf_.p) return;
    if (prm_.world > 1) throw std::runtime_error("pgb200: multi-GPU engines need pgb200_xchg_setup + xchg_import before the first chunk");
    xchg_setup(0);
}

template <int NW>
void EngineT<NW>::skm_send_args(void* out_args, int half) {
    SkmSendArgs& a = *reinterpret_cast<SkmSendArgs*>(out_args);
    const int world = xa_geom_.world;
    a.n_buckets = skm_geom_.n_buckets;
    a.world = world;
    a.rank = prm_.rank;
    a.own_shift = skm_own_shift_;
    a.seg_idx = xa_seg_idx_;
    a.epoch = xa_send_epoch_ + 1;   // 0 = nothing published yet
    a.max_seg = xa_geom_.max_seg;
    a.bo_stride = xa_geom_.bo_max + 1;
    a.cap_pair = xa_geom_.cap_pair;
    a.segoff = skm_segoff_.template as<u32>();
    u64* misc = skm_misc_.template as<u64>();
    a.total = misc + 60;
    a.cursor = misc;                 // [16]
    a.dst_delta = misc + 16;         // [16]
    a.dst_ok = reinterpret_cast<u32*>(misc + 32);   // [16]
    for (int o = 0; o < world; o++) {
        if (!xa_peer_[o]) throw std::runtime_error("pgb200: exchange peer not imported");
        char* h = static_cast<char*>(xa_peer_[o]) + (u64)half * xa_geom_.half_bytes;
        a.peer_nseg[o] = reinterpret_cast<u32*>(h + xa_geom_.off_nseg);
        a.peer_ring[o] = reinterpret_cast<SkmSegDesc*>(h + xa_geom_.off_ring);
        a.peer_segoff[o] = reinterpret_cast<u32*>(h + xa_geom_.off_segoff);
        a.peer_recs[o] = reinterpret_cast<u64*>(h + xa_geom_.off_recs) + (u64)prm_.rank * xa_geom_.cap_pair * (NW + 2);
    }
    a.counters = d_cnt_;
}

// Upper estimate of the fullest arena region's fill once a chunk of n_rec more reads has been partitioned.  What the host knows
// (C_XUSED after C_XSEGS segments of epoch C_XEPOCH) lags behind the stream; the chunks it does not know yet are assumed to make
// twice the records per read seen so far in this epoch -- before anything has been seen: four times a run every w/4 k-mers, runs being
// about w/3 long on random sequence -- and never more than one record per k-mer.  An estimate that turns out too low is caught on the
// device: k_skm_publish refuses the blob and raises C_XERR (an error, not a wrong result).
template <int NW>
u64 EngineT<NW>::skm_room_estimate(u64 n_rec) {
    const u64 per_read_worst = (u64)std::max(1, prm_.max_rd_len - prm_.K + 1);
    const bool current = h_cnt_[C_XEPOCH] == xa_send_epoch_ + 1;
    u64 segs_done = current ? h_cnt_[C_XSEGS] : 0, used = current ? h_cnt_[C_XUSED] : 0;
    if (xa_reads_cum_.empty()) xa_reads_cum_.push_back(0);
    if (segs_done >= xa_reads_cum_.size()) segs_done = xa_reads_cum_.size() - 1;
    const u64 reads_done = xa_reads_cum_[segs_done], reads_fed = xa_reads_cum_.back();
    u64 per_read = 4 * (per_read_worst / (u64)std::max(1, skm_geom_.w / 4) + 1);
    if (reads_done) per_read = std::max<u64>(1, (2 * used * (u64)xa_geom_.world + reads_done - 1) / reads_done);   // `used` is ONE region's fill
    per_read = std::min(per_read, per_read_worst);
    return used + ((reads_fed - reads_done + n_rec) * per_read + xa_geom_.world - 1) / xa_geom_.world;
}

// Room for the next chunk's records and segment (called OUTSIDE the caller's per-chunk event bracket: an aggregation times itself).
// Single GPU: decided here; the aggregation launch is asynchronous (it is ordered behind the scatter kernels by the stream, and
// the next chunks go to the other arena half).  Several GPUs: the caller fences + flushes all GPUs collectively (pgb200_xchg_room).
template <int NW>
void EngineT<NW>::skm_make_room(u64 n_rec, bool host_text) {
    skm_init();
    xchg_default_setup();
    if (xa_geom_.world == 1) {
        // Host text arrives at PCIe speed and leaves the GPU idle most of the time: whenever the insert stream has drained and at least
        // two chunks are waiting, they are aggregated right away, so that only the last couple of chunks remain for pgb200_finish_pass1.
        // Device-resident text is fed faster than it is partitioned: the stream never drains and everything is aggregated once.
        // PGB200_SKM_FLUSH_EVERY=n forces a fixed cadence (0: only when the arena is full).
        bool early = false;
        if (skm_flush_every_ > 0) early = xa_seg_idx_ >= (u32)skm_flush_every_;
        else if (skm_flush_every_ < 0 && host_text && xa_seg_idx_ >= 2) {
            early = cudaStreamQuery(st_) == cudaSuccess;
            if (!early) cudaGetLastError();   // cudaErrorNotReady is not an error; do not leave it for the next launch check
        }
        const bool full = xa_seg_idx_ >= xa_geom_.max_seg || skm_room_estimate(n_rec) > xa_geom_.cap_pair;
        if ((full || early) && xa_seg_idx_ > 0) {
            skm_close_epoch(false);
            skm_flush();
        }
    } else if (xa_seg_idx_ >= xa_geom_.max_seg) {
        throw std::runtime_error("pgb200: too many chunks in one exchange epoch: call pgb200_xchg_fence + pgb200_flush (on all GPUs) more often");
    }
}

// several GPUs: the coordinator asks before it feeds the next chunk
template <int NW>
bool EngineT<NW>::xchg_room(uint64_t n_rec) {
    if (!xa_buf_.p) return true;
    return xa_seg_idx_ < xa_geom_.max_seg && skm_room_estimate(n_rec) <= xa_geom_.cap_pair;
}

// partition the chunk just decoded and deliver its records (inside the caller's "insert" event bracket)
template <int NW>
void EngineT<NW>::skm_feed_chunk(size_t ci) {
    const ReadChunk& ch = chunks_[ci];
    const u32 B = skm_geom_.n_buckets;
    const int world = xa_geom_.world;
    PG_CUDA(cudaMemsetAsync(skm_cnt_.p, 0, (B + 1) * sizeof(u32), st_));
    PG_CUDA(cudaMemsetAsync(skm_cursor_.p, 0, (B + 1) * sizeof(u32), st_));
    const size_t ring = (size_t)skm_part_threads_ * skm_geom_.w * sizeof(u32);
    const unsigned blocks = (unsigned)std::min<u64>((ch.n_rec + skm_part_threads_ - 1) / skm_part_threads_, 148ull * 16);
    skm_side_.ensure(ch.n_rec * (SKM_SIDE_RUNS * sizeof(u32) + 1) + 256);
    u32* side = skm_side_.template as<u32>();
    u8* nruns = reinterpret_cast<u8*>(side + ch.n_rec * SKM_SIDE_RUNS);
    k_skm_count<<<blocks, skm_part_threads_, ring, st_>>>(skm_geom_, ch.words, ch.len, ch.n_rec, W64_, skm_cnt_.template as<u32>(), side, nruns);
    PG_CUDA(cudaGetLastError());
    u64* misc = skm_misc_.template as<u64>();
    device_scan(BucketCntIn{skm_cnt_.template as<u32>()}, BucketOffOut{skm_segoff_.template as<u32>()}, (u64)B, skm_scan_.template as<u64>(), misc + 60, st_);
    SkmSendArgs a;
    skm_send_args(&a, (int)(xa_send_epoch_ % xa_halves_));
    k_skm_publish<<<(unsigned)std::min<u64>(((u64)B + world + 255) / 256, 148ull * 8), 256, 0, st_>>>(a);
    PG_CUDA(cudaGetLastError());
    u32* cursor_b = skm_cursor_.template as<u32>();
    k_skm_scatter<NW><<<(unsigned)std::min<u64>((ch.n_rec + 255) / 256, 148ull * 16), 256, 0, st_>>>(a, prm_.K, ch.words, ch.n_rec, W64_, ch.ord_base, ch.ord_stride, side, nruns, cursor_b);
    PG_CUDA(cudaGetLastError());
    k_skm_rescan<NW><<<blocks, skm_part_threads_, ring, st_>>>(a, skm_geom_, ch.words, ch.len, ch.n_rec, W64_, ch.ord_base, ch.ord_stride, nruns, cursor_b);
    PG_CUDA(cudaGetLastError());
    if (xa_reads_cum_.empty()) xa_reads_cum_.push_back(0);
    xa_reads_cum_.push_back(xa_reads_cum_.back() + ch.n_rec);
    xa_seg_idx_++;
    xa_dirty_ = true;
    p1_.launches += 7;
}

// Close the current exchange epoch: the chunks fed from now on go to the other arena half.
//   hard (pgb200_xchg_fence; several GPUs: before the caller's barrier): waits until every record this GPU produced has reached its
//        owner, books the chunk timings, raises decode / arena errors;
//   soft (single GPU, mid-stream): nothing to wait for -- the aggregation launch is stream-ordered behind the scatter kernels.
// Either way the previous aggregation (it read the half that is about to be written again) is completed first.
template <int NW>
void EngineT<NW>::skm_close_epoch(bool hard) {
    if (hard) {
        settle_timing();
        read_counters();
        check_format_counter();
        if (h_cnt_[C_XERR])
            throw std::runtime_error("pgb200: exchange arena overflow (records of a chunk did not fit their owner's region, or too many segments): "
                                     "raise the arena capacity (pgb200_xchg_setup / PGB200_SKM_ARENA_MB) or flush more often");
    }
    if (!xa_buf_.p) return;
    skm_flush_complete();
    if (xa_dirty_ || prm_.world > 1) {
        xa_send_epoch_++;
        xa_seg_idx_ = 0;
        xa_reads_cum_.assign(1, 0);
        xa_dirty_ = false;
        PG_CUDA(cudaMemsetAsync(skm_misc_.p, 0, 16 * sizeof(u64), st_));          // sender cursors
        PG_CUDA(cudaMemsetAsync(d_cnt_ + C_XUSED, 0, sizeof(u64), st_));
        PG_CUDA(cudaMemsetAsync(d_cnt_ + C_XSEGS, 0, sizeof(u64), st_));
    }
}
template <int NW>
void EngineT<NW>::skm_fence() { skm_close_epoch(true); }

template <int NW>
void EngineT<NW>::skm_launch_apply(const u32* list, u32 n_list, u32* deferred_out) {
    u64* misc = skm_misc_.template as<u64>();
    SkmSegList* segs = reinterpret_cast<SkmSegList*>(reinterpret_cast<char*>(misc) + 4096);
    char* hb = static_cast<char*>(xa_buf_.p) + (u64)xa_flush_half_ * xa_geom_.half_bytes;
    SkmFlushArgs fa;
    fa.world = xa_geom_.world; fa.max_seg = xa_geom_.max_seg; fa.bo_stride = xa_geom_.bo_max + 1; fa.cap_pair = xa_geom_.cap_pair; fa.rec_words = NW + 2;
    fa.nseg = reinterpret_cast<const u32*>(hb + xa_geom_.off_nseg);
    fa.ring = reinterpret_cast<const SkmSegDesc*>(hb + xa_geom_.off_ring);
    fa.segoff = reinterpret_cast<const u32*>(hb + xa_geom_.off_segoff);
    fa.recs = reinterpret_cast<const u64*>(hb + xa_geom_.off_recs);
    fa.segs = segs;
    fa.counters = d_cnt_;
    k_skm_segs<<<1, 256, 0, st_>>>(fa);   // segment list + C_RESERVED = keys in the table, C_DEFER = C_MAXU = 0
    PG_CUDA(cudaGetLastError());
    SkmApplyArgs aa;
    aa.segs = segs; aa.bucket_list = list; aa.n_list = n_list; aa.counters = d_cnt_;
    aa.limit = (u64)(0.85 * (double)cap_);
    aa.deferred = deferred_out;
    aa.sweep = flush_sweeps_ ? 1 : 0;
    aa.D = (int)(signed char)prm_.D;   // deLowKmer is a `char` (inc/global.h:67)
    aa.hist = hist_buf_.template as<u64>();
    aa.spill_list = spill_list_.template as<u64>();
    aa.spill_cap = SPILL_CAP;
    int per_sm = 0, n_sm = 148;
    PG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_skm_apply<NW>, SKM_APPLY_THREADS, skm_apply_smem<NW>()));
    PG_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, prm_.device));
    if (per_sm < 1) per_sm = 1;
    const unsigned blocks = (unsigned)std::min<u64>((u64)n_list, (u64)n_sm * per_sm);   // persistent CTAs: as many as are resident
    if (blocks) k_skm_apply<NW><<<blocks, SKM_APPLY_THREADS, skm_apply_smem<NW>(), st_>>>(tab_, kp_, aa);
    PG_CUDA(cudaGetLastError());
    PG_CUDA(cudaMemcpyAsync(h_flush_, d_cnt_ + C_XERR, 5 * sizeof(u64), cudaMemcpyDeviceToHost, st_));   // XERR, XUSED, RESERVED, DEFER, MAXU
    p1_.launches += 2;
}

// Aggregate the closed epoch into the global table (several GPUs: only after every GPU has fenced -- the caller's barrier).
// Returns as soon as the work is queued; skm_flush_complete (next epoch close, pgb200_finish_pass1) reads the outcome.
template <int NW>
void EngineT<NW>::skm_flush(bool final_of_pass) {
    if (!xa_buf_.p || xa_flushed_epoch_ >= xa_send_epoch_) return;
    skm_flush_complete();
    if (xa_flushed_epoch_ + 1 != xa_send_epoch_) throw std::runtime_error("pgb200: internal: more than one unflushed exchange epoch");
    create_table_if_needed();
    // The end-of-pass sweeps (K4) ride on this launch when it is the pass so far -- empty table, no launch and no per-instance insert
    // before it: every entry it stores is then complete, and one pass over the table (5 ms per 2^29 slots) is saved.  Without -d the
    // sweeps only SET flags that k_sweep recomputes anyway, so it is safe to do this speculatively: whatever touches the table later
    // in the pass marks the result stale (inline_sweep_ = 2) and sweeps() runs k_sweep as before.  With -d the link counters are
    // zeroed for good, so the launch must be known to be the last of the pass (finish_pass1 on one GPU).
    flush_sweeps_ = pass_flushes_ == 0 && !pass_direct_ && inline_sweep_ == 0 && ((signed char)prm_.D <= 0 || final_of_pass);
    if (flush_sweeps_) {
        hist_buf_.ensure(256 * sizeof(u64));
        spill_list_.ensure(SPILL_CAP * sizeof(u64));
        PG_CUDA(cudaMemsetAsync(d_cnt_ + C_SPILLKEYS, 0, sizeof(u64), st_));
        PG_CUDA(cudaMemsetAsync(hist_buf_.p, 0, 256 * sizeof(u64), st_));
        PG_CUDA(cudaMemsetAsync(d_cnt_ + C_LINEAR, 0, 2 * sizeof(u64), st_));
        inline_sweep_ = 1;
    } else if (inline_sweep_ == 1) inline_sweep_ = 2;
    pass_flushes_++;
    xa_flush_half_ = (int)(xa_flushed_epoch_ % xa_halves_);
    PG_CUDA(cudaEventRecord(ev_skm_[0], st_));
    const u32 n_owned = skm_own_hi_ - skm_own_lo_;
    u32* deferred0 = reinterpret_cast<u32*>(skm_misc_.template as<char>() + 4096 + sizeof(SkmSegList));
    skm_launch_apply(nullptr, n_owned, deferred0);
    PG_CUDA(cudaEventRecord(ev_flush_, st_));
    xa_flush_inflight_ = true;
}

template <int NW>
void EngineT<NW>::skm_flush_complete() {
    if (!xa_flush_inflight_) return;
    xa_flush_inflight_ = false;
    PG_CUDA(cudaEventSynchronize(ev_flush_));
    float ms;
    PG_CUDA(cudaEventElapsedTime(&ms, ev_skm_[0], ev_flush_));
    const u32 n_owned = skm_own_hi_ - skm_own_lo_;
    u32* deferred[2];
    deferred[0] = reinterpret_cast<u32*>(skm_misc_.template as<char>() + 4096 + sizeof(SkmSegList));
    deferred[1] = deferred[0] + n_owned + 1;
    int launches = 1, which = 0;
    u64 n_def = h_flush_[3], maxu = h_flush_[4];
    if (h_flush_[0])
        throw std::runtime_error("pgb200: exchange arena overflow (the records of one chunk do not fit an arena half, or too many segments): "
                                 "raise the arena capacity (pgb200_xchg_setup / PGB200_SKM_ARENA_MB) or feed smaller chunks");
    while (n_def) {
        // buckets whose worst case did not fit the table: grow so that (at least) the largest one fits, run them again
        read_counters();
        u64 cap = cap_ * 2;
        while (0.85 * (double)cap < (double)(h_cnt_[C_DISTINCT] + maxu)) cap <<= 1;
        size_t free_b = 0, total_b = 0;
        PG_CUDA(cudaMemGetInfo(&free_b, &total_b));
        if (cap * sizeof(Slot<NW>) + (1ull << 28) > free_b)
            throw std::runtime_error("pgb200: k-mer table cannot grow further (out of HBM); use more GPUs");
        grow_table(cap);
        if (inline_sweep_ == 1) inline_sweep_ = 2;   // the list of unswept keys holds slots of the table that was just replaced
        PG_CUDA(cudaEventRecord(ev_skm_[0], st_));
        skm_launch_apply(deferred[which], (u32)n_def, deferred[which ^ 1]);
        PG_CUDA(cudaEventRecord(ev_flush_, st_));
        PG_CUDA(cudaEventSynchronize(ev_flush_));
        float ms2;
        PG_CUDA(cudaEventElapsedTime(&ms2, ev_skm_[0], ev_flush_));
        ms += ms2;
        which ^= 1;
        launches++;
        n_def = h_flush_[3];
        maxu = h_flush_[4];
    }
    // the epoch's half is free again: senders may use it from the epoch after next
    char* hb = static_cast<char*>(xa_buf_.p) + (u64)xa_flush_half_ * xa_geom_.half_bytes;
    PG_CUDA(cudaMemsetAsync(hb + xa_geom_.off_nseg, 0, (size_t)xa_geom_.world * sizeof(u32), st_));
    p1_.ms_insert += ms;
    p1_.ms_apply += ms;
    xa_flushed_epoch_++;
    if (prm_.verbose >= 2 || getenv("PGB200_SKM_STATS"))
        fprintf(stderr, "[pgb200] aggregated epoch %llu: %u owned bucket(s), %d launch(es), %.2f ms, table %llu slots\n", (unsigned long long)xa_flushed_epoch_, n_owned,
                launches, ms, (unsigned long long)cap_);
}

template <int NW>
void EngineT<NW>::skm_reset() {
    // single GPU: nothing of the arena survives a reset; several GPUs: the epochs keep alternating (peers may already deliver)
    if (!xa_buf_.p) return;
    sync();
    skm_flush_complete();
    if (prm_.world <= 1 && (xa_dirty_ || xa_flushed_epoch_ != xa_send_epoch_)) {
        skm_close_epoch(false);
        for (int h = 0; h < xa_halves_; h++)
            PG_CUDA(cudaMemsetAsync(static_cast<char*>(xa_buf_.p) + (u64)h * xa_geom_.half_bytes + xa_geom_.off_nseg, 0, sizeof(u32), st_));
        xa_flushed_epoch_ = xa_send_epoch_;
    }
}

template <int NW>
void EngineT<NW>::skm_release() {
    for (void* p : xa_ipc_opened_) cudaIpcCloseMemHandle(p);
    xa_ipc_opened_.clear();
    for (auto& e : ev_skm_) if (e) cudaEventDestroy(e);
}

#define PGB_INST(NW)                                                         \
    template void EngineT<NW>::skm_init();                                   \
    template void EngineT<NW>::xchg_setup(uint64_t);                         \
    template void EngineT<NW>::xchg_export(void*);                           \
    template void EngineT<NW>::xchg_import(int, const void*);                \
    template void EngineT<NW>::xchg_import_ptr(int, int, void*);             \
    template void* EngineT<NW>::xchg_base();                                 \
    template void EngineT<NW>::xchg_default_setup();                         \
    template void EngineT<NW>::skm_send_args(void*, int);                    \
    template void EngineT<NW>::skm_feed_chunk(size_t);                       \
    template void EngineT<NW>::skm_make_room(u64, bool);                     \
    template bool EngineT<NW>::xchg_room(uint64_t);                          \
    template void EngineT<NW>::skm_fence();                                  \
    template void EngineT<NW>::skm_close_epoch(bool);                        \
    template void EngineT<NW>::skm_flush_complete();                         \
    template void EngineT<NW>::skm_launch_apply(const u32*, u32, u32*);      \
    template u64 EngineT<NW>::skm_room_estimate(u64);                        \
    template void EngineT<NW>::skm_flush(bool);                              \
    template void EngineT<NW>::skm_reset();                                  \
    template void EngineT<NW>::skm_release();
PGB_INST(2)
PGB_INST(4)

}   // namespace pgb
