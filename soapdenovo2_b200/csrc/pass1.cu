// pass1.cu -- pass 1 of pregraph on the GPU: the per-instance insert (the second exact insert path; the default is the aggregated
// one in skm.cu), the table management, and the per-entry sweeps (delow, mark-linear, kmerFreq histogram).
//
// Replaces (reference file:line, standardPregraph/):
//   K2  chopKmer4read (prlHashReads.c:163-259)                                              -> k_chop_insert (rolling part)
//   K3  threadRoutine sig 1 + put_kmerset (prlHashReads.c:79-90, newhash.c:473-528)         -> k_chop_insert (insert part)
//   K4  thread_delow, thread_mark, freqStat (prlHashReads.c:953-996, 1020-1077, 1104-1132)  -> k_sweep
// Design differences that matter: no owner filter (the reference makes every thread scan the whole batch and keep
// hash % P == id); the CRC set hash is not computed per instance at all -- it only defines the reference's iteration
// order and is evaluated once per DISTINCT k-mer in layout.cu.  (K1, the text decoder, and feed_text live in decode.cu.)
#include "engine_impl.cuh"
#include "scan.cuh"
#include "chop.cuh"
#include <ctime>

namespace pgb {

static double host_now() { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return t.tv_sec * 1e3 + t.tv_nsec * 1e-6; }

// ------------------------------------------------------------------------------------------------ K2+K3: chop + insert
// One thread per read: roll the forward k-mer (nextKmer) and its reverse complement (prevKmer on the complement strand)
// one base at a time, pick the canonical one, derive the left/right neighbour codes in the canonical orientation
// (SURVEY.md A.2) and apply the instance to the table.  rank = (read ordinal << 16) | position.
// This kernel sits on the measured rate of random DRAM slot updates (profiles/r01_rmw_ubench.md, r01_insert_ncu.md): one slot
// read + write-back per k-mer INSTANCE.  It is kept as the independent second implementation that every parity test also runs
// (PGB200_SKM=0); the product default touches HBM once per DISTINCT k-mer (skm.cu).
constexpr int INS_THREADS = 256;
#ifndef INS_MIN_BLOCKS
#define INS_MIN_BLOCKS 5
#endif

template <int NW>
struct InsertSink {
    const Table<NW>& tab;
    u64 rank_base;
    unsigned& my_new;
    __device__ __forceinline__ void operator()(const Kmer<NW>& canon, unsigned left, unsigned right, int j) {
        my_new += table_insert(tab, canon, left, right, rank_base | (u64)j);
    }
};

template <int NW>
__global__ void __launch_bounds__(INS_THREADS, INS_MIN_BLOCKS) k_chop_insert(Table<NW> tab, KParams<NW> kp, const u64* __restrict__ words,
                                                             const u32* __restrict__ lens, u64 n_rec, int W64, u64 ord_base, u64 ord_stride,
                                                             u64* counters, int use_tma) {
    extern __shared__ __align__(128) u64 s_words[];   // [INS_THREADS][W64] when use_tma
    __shared__ __align__(8) u64 s_bar;
    __shared__ unsigned s_new;
    if (threadIdx.x == 0) { s_new = 0; if (use_tma) mbar_init(&s_bar, 1); }
    __syncthreads();
    unsigned my_new = 0;
    const u64 n_tiles = (n_rec + INS_THREADS - 1) / INS_THREADS;
    unsigned parity = 0;
    for (u64 tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const u64 r0 = tile * INS_THREADS;
        const u64 r = r0 + threadIdx.x;
        const u64* wp = words + r * (u64)W64;
        if (use_tma) {
            u64 cnt = n_rec - r0 < (u64)INS_THREADS ? n_rec - r0 : (u64)INS_THREADS;
            unsigned bytes = (unsigned)((cnt * (u64)W64 * 8 + 15) & ~15ull);   // the arena pads every allocation to 256 B
            if (threadIdx.x == 0) {
                mbar_expect_tx(&s_bar, bytes);
                tma_bulk_g2s(s_words, words + r0 * (u64)W64, bytes, &s_bar);
            }
            mbar_wait(&s_bar, parity);
            parity ^= 1;
            wp = s_words + (u64)threadIdx.x * W64;
        }
        if (r < n_rec) {
            const int L = (int)lens[r];
            if (L >= kp.K + 1) {
                InsertSink<NW> sink{tab, (ord_base + r * ord_stride) << 16, my_new};
                chop_read(kp, wp, L, sink);
            }
        }
        if (use_tma) __syncthreads();   // the tile buffer is reused by the next bulk copy
    }
    if (my_new) atomicAdd(&s_new, my_new);
    __syncthreads();
    if (threadIdx.x == 0 && s_new) atomicAdd(&counters[C_DISTINCT], (u64)s_new);
}

template <int NW>
void EngineT<NW>::chop_insert_chunk(const ReadChunk& ch) {
    const unsigned blocks = (unsigned)std::min<u64>((ch.n_rec + INS_THREADS - 1) / INS_THREADS, 148ull * 64);
    const size_t smem = (size_t)INS_THREADS * W64_ * sizeof(u64);
    const int use_tma = smem <= 96 * 1024;
    // opt in whatever the size: the kernel's static shared memory (barrier, counter) comes on top of the tile, so a 48 KB tile
    // (max_rd_len 737..768) already exceeds the default limit
    if (use_tma) PG_CUDA(cudaFuncSetAttribute(k_chop_insert<NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_chop_insert<NW><<<blocks, INS_THREADS, use_tma ? smem : 0, st_>>>(tab_, kp_, ch.words, ch.len, ch.n_rec, W64_, ch.ord_base, ch.ord_stride, d_cnt_, use_tma);
    pass_direct_ = true;
    if (inline_sweep_ == 1) inline_sweep_ = 2;   // entries swept by an aggregation launch have changed since
    PG_CUDA(cudaGetLastError());
    p1_.launches += 1;
}

// ------------------------------------------------------------------------------------------------ table management
template <int NW>
__global__ void k_rehash(Table<NW> oldt, Table<NW> newt) {
    u64 n = oldt.mask + 1;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const Slot<NW>* s = oldt.slots + i;
        if (!slot_occupied(s)) continue;
        Kmer<NW> k = slot_key(s);
        bool claimed;
        u64 idx = table_find_or_claim(newt, k, &claimed);
        newt.slots[idx].payload = s->payload;
        newt.slots[idx].aux = s->aux;
    }
}

static u64 next_pow2(u64 x) { u64 p = 1; while (p < x) p <<= 1; return p; }

template <int NW>
void EngineT<NW>::alloc_table(u64 cap) {
    tab_buf_.alloc(cap * sizeof(Slot<NW>));
    PG_CUDA(cudaMemsetAsync(tab_buf_.p, 0xFF, cap * sizeof(Slot<NW>), st_));
    tab_.slots = tab_buf_.template as<Slot<NW>>();
    tab_.mask = cap - 1;
    cap_ = cap;
}

template <int NW>
void EngineT<NW>::grow_table(u64 new_cap) {
    if (prm_.verbose) fprintf(stderr, "[pgb200] growing k-mer table %llu -> %llu slots\n", cap_, new_cap);
    DevBuf nb;
    nb.alloc(new_cap * sizeof(Slot<NW>));
    PG_CUDA(cudaMemsetAsync(nb.p, 0xFF, new_cap * sizeof(Slot<NW>), st_));
    Table<NW> nt{nb.template as<Slot<NW>>(), new_cap - 1};
    k_rehash<NW><<<148 * 8, 256, 0, st_>>>(tab_, nt);
    PG_CUDA(cudaGetLastError());
    sync();
    std::swap(tab_buf_.p, nb.p);
    std::swap(tab_buf_.bytes, nb.bytes);
    tab_ = nt;
    cap_ = new_cap;
}

template <int NW>
void EngineT<NW>::create_table_if_needed() {
    join_table_clear();
    if (tab_.slots) return;
    u64 want = prm_.table_slots;
    if (!want) {
        if (prm_.initG) {
            // the reference's own budget: P sets of the static prime size (prlHashReads.c:369-390)
            want = (u64)prm_.P * ref_static_set_size(prm_.initG, prm_.P, prm_.flavour127 != 0);
            want = (want + want / 4) / (u64)(prm_.world > 1 ? prm_.world : 1);
        } else {
            want = 1ull << 24;
        }
    }
    alloc_table(next_pow2(want < 1024 ? 1024 : want));
}

// have = distinct keys already in the table (exact as of the last sync), incoming = upper bound of new keys about to arrive
template <int NW>
void EngineT<NW>::ensure_table_bound(u64 have, u64 incoming) {
    create_table_if_needed();
    u64 need = have + incoming;   // every incoming instance could be a new key
    if ((double)need <= 0.80 * (double)cap_) return;
    u64 cap = cap_;
    while ((double)need > 0.80 * (double)cap) cap <<= 1;
    size_t free_b = 0, total_b = 0;
    PG_CUDA(cudaMemGetInfo(&free_b, &total_b));
    while (cap > cap_ && cap * sizeof(Slot<NW>) + (1ull << 30) > free_b) cap >>= 1;
    if (cap > cap_) { grow_table(cap); return; }
    if ((double)need > 0.97 * (double)cap_)
        throw std::runtime_error("pgb200: k-mer table cannot grow further (out of HBM); use more GPUs or a smaller batch");
}

template <int NW>
void EngineT<NW>::ensure_table(u64 incoming) {
    create_table_if_needed();
    read_counters();
    ensure_table_bound(h_cnt_[C_DISTINCT], incoming);
}

// read-store arena: chunks are carved out of large blocks (no cudaMalloc / cudaFree per chunk)
template <int NW>
void* EngineT<NW>::arena_alloc(size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    if (arena_.empty() || arena_used_ + bytes > arena_.back().second) {
        size_t blk = std::max<size_t>(bytes, (size_t)1 << 30);
        void* p = nullptr;
        PG_CUDA(cudaMalloc(&p, blk));
        arena_.push_back({p, blk});
        arena_used_ = 0;
    }
    void* r = static_cast<char*>(arena_.back().first) + arena_used_;
    arena_used_ += bytes;
    return r;
}

template <int NW>
void EngineT<NW>::finish_pass1(Pass1Stats* st) {
    if (prm_.world > 1) {
        sync();
        skm_flush_complete();
        if (xa_dirty_ || xa_flushed_epoch_ != xa_send_epoch_)
            throw std::runtime_error("pgb200: multi-GPU pass 1: call pgb200_xchg_fence, a barrier over all GPUs, then pgb200_flush before pgb200_finish_pass1");
    } else if (xa_buf_.p) {
        skm_close_epoch(false);
        skm_flush(true);   // nothing of this pass comes after it
    }
    settle_timing();
    sync();
    skm_flush_complete();
    read_counters();
    if (inline_sweep_ == 1 && h_cnt_[C_SPILLKEYS] > SPILL_CAP) inline_sweep_ = 2;   // more unswept keys than the list holds
    check_format_counter();
    p1_.records = total_records_;
    p1_.reads_kept = h_cnt_[C_KEPT];
    p1_.instances = h_cnt_[C_INSTANCES];
    p1_.distinct = h_cnt_[C_DISTINCT];
    p1_.table_slots = cap_;
    n_nodes_ = p1_.distinct;
    if (st) *st = p1_;
}

// Fold another engine of the same job into this one: its table shard (disjoint keys: a k-mer lives on the GPU that owns its bucket)
// is read over NVLink and re-inserted here with its payload and rank words, its packed reads are copied into this engine's store.
template <int NW>
void EngineT<NW>::absorb(IEngine* other_i) {
    EngineT<NW>* o = dynamic_cast<EngineT<NW>*>(other_i);
    if (!o || o == this) throw std::runtime_error("pgb200: absorb: engines of different key width");
    PG_CUDA(cudaSetDevice(o->prm_.device));
    o->settle_timing();
    o->read_counters();
    o->sync();   // (also a table clear nobody joined)
    PG_CUDA(cudaSetDevice(prm_.device));
    int can = 0;
    PG_CUDA(cudaDeviceCanAccessPeer(&can, prm_.device, o->prm_.device));
    if (!can) throw std::runtime_error("pgb200: GPUs cannot access each other's memory (no peer access)");
    cudaError_t pe = cudaDeviceEnablePeerAccess(o->prm_.device, 0);
    if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) PG_CUDA(pe);
    cudaGetLastError();
    settle_timing();
    read_counters();
    const u64 have = h_cnt_[C_DISTINCT], inc = o->h_cnt_[C_DISTINCT];
    ensure_table_bound(have, inc);
    if (o->tab_.slots && inc) {
        k_rehash<NW><<<148 * 8, 256, 0, st_>>>(o->tab_, tab_);
        PG_CUDA(cudaGetLastError());
    }
    const u64 sums[3] = {have + inc, h_cnt_[C_INSTANCES] + o->h_cnt_[C_INSTANCES], h_cnt_[C_KEPT] + o->h_cnt_[C_KEPT]};   // C_DISTINCT, C_INSTANCES, C_KEPT
    PG_CUDA(cudaMemcpyAsync(d_cnt_ + C_DISTINCT, sums, sizeof sums, cudaMemcpyHostToDevice, st_));
    for (const ReadChunk& c : o->chunks_) {
        ReadChunk n = c;
        const size_t wb = c.n_rec * (u64)W64_ * sizeof(u64), lb = c.n_rec * sizeof(u32);
        n.words = reinterpret_cast<u64*>(arena_alloc(wb));
        n.len = reinterpret_cast<u32*>(arena_alloc(lb));
        PG_CUDA(cudaMemcpyPeerAsync(n.words, prm_.device, c.words, o->prm_.device, wb, st_));
        PG_CUDA(cudaMemcpyPeerAsync(n.len, prm_.device, c.len, o->prm_.device, lb, st_));
        chunks_.push_back(n);
    }
    sync();
    total_records_ += o->total_records_;
    p1_.ms_decode += o->p1_.ms_decode;
    p1_.ms_insert += o->p1_.ms_insert;
    p1_.ms_apply += o->p1_.ms_apply;
    p1_.launches += o->p1_.launches;
    n_nodes_ = have + inc;
    h_cnt_[C_DISTINCT] = sums[0]; h_cnt_[C_INSTANCES] = sums[1]; h_cnt_[C_KEPT] = sums[2];
}

template <int NW>
void EngineT<NW>::reset_pass1() {
    double t0 = host_now();
    settle_timing();
    sync();
    chunks_.clear();
    skm_reset();
    inline_sweep_ = 0;
    pass_flushes_ = 0;
    pass_direct_ = false;
    // keep the first arena block for the next pass, release the rest
    while (arena_.size() > 1) { cudaFree(arena_.back().first); arena_.pop_back(); }
    arena_used_ = 0;
    total_records_ = 0;
    p1_ = Pass1Stats();
    PG_CUDA(cudaMemsetAsync(d_cnt_, 0, C_COUNT * sizeof(u64), st_));
    order_buf_.release();
    n_nodes_ = 0;
    sync();
    // the table is cleared on its own stream WITHOUT waiting: the next pass starts with decoding and partitioning, which do not touch
    // the table; whatever touches it next joins the clear first (create_table_if_needed -> join_table_clear)
    if (tab_.slots) {
        PG_CUDA(cudaMemsetAsync(tab_buf_.p, 0xFF, cap_ * sizeof(Slot<NW>), st_clear_));
        PG_CUDA(cudaEventRecord(ev_clear_, st_clear_));
        clear_pending_ = true;
    }
    for (int i = 0; i < C_COUNT; i++) h_cnt_[i] = 0;
    if (prm_.verbose >= 2) fprintf(stderr, "[pgb200] reset_pass1: %.2f ms host\n", host_now() - t0);
}

// ------------------------------------------------------------------------------------------------ K4: sweeps
// delow (thread_delow): zero every link counter <= D, deleted=1 if nothing is left.  mark (thread_mark): linear=1 iff exactly
// one non-zero left and one non-zero right link (NO deleted check there); histogram of cov.  All per-entry => one pass.
// The table is streamed once: K <= 63 slots arrive with one 256-bit load each (key + payload in one 32 B sector), two slots per
// thread in flight; the payload is written back only when a flag or a counter changed.
template <int NW>
__global__ void __launch_bounds__(256) k_sweep(Table<NW> tab, int D, u64* hist, u64* counters) {
    __shared__ unsigned s_hist[256];
    __shared__ unsigned s_lin, s_rem;
    s_hist[threadIdx.x] = 0;
    if (threadIdx.x == 0) { s_lin = 0; s_rem = 0; }
    __syncthreads();
    const u64 n = tab.mask + 1, stride = (u64)gridDim.x * blockDim.x;
    unsigned rem = 0, lin = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += 2 * stride) {
        Slot<NW>* s0 = tab.slots + i;
        Slot<NW>* s1 = tab.slots + (i + stride < n ? i + stride : i);
        const bool two = i + stride < n;
        u64 k0a, k0b, p0, k1a, k1b, p1;
        if constexpr (NW == 2) {
            const U256 v0 = ld256(s0), v1 = ld256(s1);
            k0a = v0.a; k0b = v0.b; p0 = v0.c;
            k1a = v1.a; k1b = v1.b; p1 = v1.c;
        } else {
            const U128 a0 = ldcg128(s0->key), a1 = ldcg128(s1->key);
            k0a = a0.a; k0b = a0.b; k1a = a1.a; k1b = a1.b;
            p0 = ldcg64(&s0->payload); p1 = ldcg64(&s1->payload);
        }
        if (!(k0a == EMPTY64 && k0b == EMPTY64)) {
            const u64 q = sweep_payload(p0, D, rem, lin, s_hist);
            if (q != p0) s0->payload = q;
        }
        if (two && !(k1a == EMPTY64 && k1b == EMPTY64)) {
            const u64 q = sweep_payload(p1, D, rem, lin, s_hist);
            if (q != p1) s1->payload = q;
        }
    }
    if (lin) atomicAdd(&s_lin, lin);
    if (rem) atomicAdd(&s_rem, rem);
    __syncthreads();
    if (s_hist[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (u64)s_hist[threadIdx.x]);
    if (threadIdx.x == 0) {
        if (s_lin) atomicAdd(&counters[C_LINEAR], (u64)s_lin);
        if (s_rem) atomicAdd(&counters[C_REMOVED], (u64)s_rem);
    }
}

// the same for a list of slots (the keys an aggregation launch with fused sweeps stored unswept)
template <int NW>
__global__ void __launch_bounds__(256) k_sweep_list(Table<NW> tab, int D, const u64* __restrict__ list, u64 n, u64* hist, u64* counters) {
    __shared__ unsigned s_hist[256];
    __shared__ unsigned s_lin, s_rem;
    s_hist[threadIdx.x] = 0;
    if (threadIdx.x == 0) { s_lin = 0; s_rem = 0; }
    __syncthreads();
    unsigned rem = 0, lin = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        Slot<NW>* s = tab.slots + list[i];
        const u64 p = ldcg64(&s->payload);
        const u64 q = sweep_payload(p, D, rem, lin, s_hist);
        if (q != p) s->payload = q;
    }
    if (lin) atomicAdd(&s_lin, lin);
    if (rem) atomicAdd(&s_rem, rem);
    __syncthreads();
    if (s_hist[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (u64)s_hist[threadIdx.x]);
    if (threadIdx.x == 0) {
        if (s_lin) atomicAdd(&counters[C_LINEAR], (u64)s_lin);
        if (s_rem) atomicAdd(&counters[C_REMOVED], (u64)s_rem);
    }
}

template <int NW>
void EngineT<NW>::sweeps(SweepStats* st) {
    double t0 = host_now();
    create_table_if_needed();
    DevBuf& hist = hist_buf_;   // persistent: a cudaMalloc / cudaFree pair per call costs more than the sweep of a small table
    hist.ensure(256 * sizeof(u64));
    // inline_sweep_ == 1: the pass was ONE aggregation launch into an empty table and nothing touched the table since -- its flush
    // already applied the sweeps to every entry it stored (skm.cu), the histogram and the counters are complete
    const int D = (int)(signed char)prm_.D;   // deLowKmer is a `char` (inc/global.h:67)
    if (inline_sweep_ != 1) {
        PG_CUDA(cudaMemsetAsync(hist.p, 0, 256 * sizeof(u64), st_));
        PG_CUDA(cudaMemsetAsync(d_cnt_ + C_LINEAR, 0, 2 * sizeof(u64), st_));
        k_sweep<NW><<<148 * 8, 256, 0, st_>>>(tab_, D, hist.template as<u64>(), d_cnt_);
        PG_CUDA(cudaGetLastError());
    } else if (h_cnt_[C_SPILLKEYS]) {
        // the few keys whose instances went straight to the table (their bucket had more distinct k-mers than its shared-memory table)
        const u64 n = h_cnt_[C_SPILLKEYS];
        k_sweep_list<NW><<<(unsigned)std::min<u64>((n + 255) / 256, 148ull * 8), 256, 0, st_>>>(tab_, D, spill_list_.template as<u64>(), n, hist.template as<u64>(), d_cnt_);
        PG_CUDA(cudaGetLastError());
        PG_CUDA(cudaMemsetAsync(d_cnt_ + C_SPILLKEYS, 0, sizeof(u64), st_));   // a second call must not sweep (and count) them again
        h_cnt_[C_SPILLKEYS] = 0;
    }
    u64 h[256];
    PG_CUDA(cudaMemcpyAsync(h, hist.p, sizeof h, cudaMemcpyDeviceToHost, st_));
    read_counters();
    for (int i = 0; i < 256; i++) st->hist[i] = (long long)h[i];
    st->linear = h_cnt_[C_LINEAR];
    st->removed = h_cnt_[C_REMOVED];
    if (prm_.verbose >= 2) fprintf(stderr, "[pgb200] sweeps: %.2f ms host\n", host_now() - t0);
}

// ------------------------------------------------------------------------------------------------ ctor / dtor
template <int NW>
EngineT<NW>::EngineT(const PgParams& p) : prm_(p) {
    PG_CUDA(cudaSetDevice(p.device));
    if (const char* g = getenv("PGB200_SKM")) skm_mode_ = atoi(g) ? 1 : 0;
    if (const char* g = getenv("PGB200_SKM_FLUSH_EVERY")) skm_flush_every_ = atoi(g);
    if (p.world > 1) skm_mode_ = 1;   // records are the only exchange format
    kp_ = make_kparams<NW>(p.K);
    PG_CUDA(cudaStreamCreateWithFlags(&st_, cudaStreamNonBlocking));
    PG_CUDA(cudaStreamCreateWithFlags(&st_copy_, cudaStreamNonBlocking));
    PG_CUDA(cudaStreamCreateWithFlags(&st_clear_, cudaStreamNonBlocking));
    PG_CUDA(cudaEventCreateWithFlags(&ev_clear_, cudaEventDisableTiming));
    PG_CUDA(cudaStreamCreateWithFlags(&st_dec_, cudaStreamNonBlocking));
    PG_CUDA(cudaEventCreateWithFlags(&ev_dec_done_, cudaEventDisableTiming));
    PG_CUDA(cudaEventCreate(&ev_flush_));
    PG_CUDA(cudaHostAlloc(&h_flush_, 8 * sizeof(u64), cudaHostAllocDefault));
    for (auto& q : ev_ring_) for (auto& e : q) PG_CUDA(cudaEventCreate(&e));
    PG_CUDA(cudaEventCreateWithFlags(&ev_copy_, cudaEventDisableTiming));
    PG_CUDA(cudaMalloc(&d_cnt_, C_COUNT * sizeof(u64)));
    PG_CUDA(cudaMemsetAsync(d_cnt_, 0, C_COUNT * sizeof(u64), st_));
    PG_CUDA(cudaHostAlloc(&h_cnt_, (C_COUNT + 2) * sizeof(u64), cudaHostAllocDefault));
    for (int i = 0; i < C_COUNT; i++) h_cnt_[i] = 0;
    W64_ = (p.max_rd_len + 31) / 32;
    if (W64_ < 1) W64_ = 1;
    sync();
}

template <int NW>
EngineT<NW>::~EngineT() {
    cudaStreamSynchronize(st_);
    for (auto& a : arena_) cudaFree(a.first);
    skm_release();
    if (d_cnt_) cudaFree(d_cnt_);
    if (h_cnt_) cudaFreeHost(h_cnt_);
    for (auto& q : ev_ring_) for (auto& e : q) if (e) cudaEventDestroy(e);
    if (ev_dec_done_) cudaEventDestroy(ev_dec_done_);
    if (ev_flush_) cudaEventDestroy(ev_flush_);
    if (h_flush_) cudaFreeHost(h_flush_);
    if (st_dec_) { cudaStreamSynchronize(st_dec_); cudaStreamDestroy(st_dec_); }
    if (ev_copy_) cudaEventDestroy(ev_copy_);
    if (st_copy_) cudaStreamDestroy(st_copy_);
    if (st_clear_) { cudaStreamSynchronize(st_clear_); cudaStreamDestroy(st_clear_); }
    if (ev_clear_) cudaEventDestroy(ev_clear_);
    if (st_) cudaStreamDestroy(st_);
}

template class EngineT<2>;
template class EngineT<4>;

IEngine* make_engine(const PgParams& p) {
    if (p.K <= 63) return new EngineT<2>(p);
    return new EngineT<4>(p);
}

}   // namespace pgb
