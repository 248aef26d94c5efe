// pass2.cu -- K7/K8: re-scan the (HBM-resident, 2-bit packed) reads against the frozen k-mer table, turn every read
// into its edge path, count pre-arcs, and (with -R) record read paths + markers.
//
// Reference (standardPregraph/prlRead2path.c): chopKmer4read :271-345, searchKmer :348-368, parse1read :598-745,
// search1kmerPlus :558-596, thread_add1preArc :388-403, output_arcs :426-476, recordPathBin :478-543.
// The reference does this in five barrier-separated sweeps over a 1e8-k-mer batch (each thread scanning the whole batch
// and keeping hash % P == id); here one thread owns one read end to end: roll the k-mer, look it up (one 32 B sector),
// run parse1read's state machine, resolve (K+1)-mers in the patch table on the spot, and push arcs into a GPU hash
// table keyed by (from,to) with {multiplicity, first-seen rank}.  The reference's adjacency lists are head-inserted in
// read-stream order, so a `from` line lists its arcs by DESCENDING first-seen rank -- regenerated at output time.
// Quirks kept: IsPrevKmer/prevKmer survive a restart (:617-630 vs :690-714); paths restart only while fewer than 2
// segments were kept; a missing (K+1)-mer becomes 0 and cuts the arc / path loops.
#include "engine_impl.cuh"
#include "scan.cuh"
#include "patch.cuh"
#include "chop.cuh"
#include <algorithm>

namespace pgb {

struct alignas(32) ArcSlot {
    u64 key;     // from << 32 | to ; EMPTY64 = free
    u64 rank;    // first creation: (read ordinal << 16) | index in path
    u64 count;
    u64 pad;
};

__device__ __forceinline__ bool arc_add(ArcSlot* t, u64 mask, u32 from, u32 to, u64 rank) {
    u64 key = ((u64)from << 32) | to;
    u64 idx = mix64(key) & mask;
    for (u64 probes = 0; probes <= mask; probes++) {
        u64 cur = t[idx].key;
        if (cur == EMPTY64) {
            u64 old = atomicCAS(&t[idx].key, EMPTY64, key);
            cur = old == EMPTY64 ? key : old;
        }
        if (cur == key) {
            atomicAdd(&t[idx].count, 1ull);
            atomicMin(&t[idx].rank, rank);
            return true;
        }
        idx = (idx + 1) & mask;
    }
    return false;   // table full
}

template <int NW>
__global__ void __launch_bounds__(128) k_pass2(Table<NW> tab, KParams<NW> kp, const u64* __restrict__ words, const u32* __restrict__ lens, u64 n_rec,
                                               int W64, u64 ord_base, u64 ord_stride, int stride, u32* pathbuf, u32* reclen, int repsTie,
                                               const PatchSlot<NW>* patch, u64 pmask, bool quirk128, ArcSlot* arcs, u64 amask, u32* marker,
                                               u64* counters, u64* err, int use_tma) {
    extern __shared__ __align__(128) u64 s_words[];   // TMA-staged tile of packed reads (see chop.cuh)
    __shared__ __align__(8) u64 s_bar;
    if (threadIdx.x == 0 && use_tma) mbar_init(&s_bar, 1);
    __syncthreads();
    const int K = kp.K;
    unsigned deleted_reads = 0;
    unsigned parity = 0;
    const u64 n_tiles = (n_rec + blockDim.x - 1) / blockDim.x;
    for (u64 tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const u64 r0 = tile * blockDim.x;
        const u64 r = r0 + threadIdx.x;
        if (use_tma) {
            if (tile != blockIdx.x) __syncthreads();   // previous tile fully consumed
            u64 cnt = n_rec - r0 < (u64)blockDim.x ? n_rec - r0 : (u64)blockDim.x;
            unsigned bytes = (unsigned)((cnt * (u64)W64 * 8 + 15) & ~15ull);
            if (threadIdx.x == 0) { mbar_expect_tx(&s_bar, bytes); tma_bulk_g2s(s_words, words + r0 * (u64)W64, bytes, &s_bar); }
            mbar_wait(&s_bar, parity);
            parity ^= 1;
        }
        if (r >= n_rec) continue;
        const int L = (int)lens[r];
        if (L < K + 1) continue;                       // skipped exactly like pass 1 (prlRead2path.c:1012 etc.)
        const u64 ord = ord_base + r * ord_stride;
        const u64* wp = use_tma ? s_words + (u64)threadIdx.x * W64 : words + r * (u64)W64;
        u32* mix = pathbuf + r * (u64)stride;
        const int n = L - K + 1;
        Kmer<NW> fwd = kzero<NW>(), rc = kzero<NW>(), prevK = kzero<NW>();
        int retain = 0, pos = 0;
        bool IsPrev = false, stop = false;
        u64 cur = wp[0];
        for (int i = 0; i < L && !stop; i++) {
            if (i && (i & 31) == 0) cur = wp[i >> 5];
            unsigned c = (unsigned)((cur >> (2 * (i & 31))) & 3);
            fwd = knext(fwd, c, kp);
            rc = kprev(rc, c ^ 2u, kp);
            if (i < K - 1) continue;
            bool sm = kless(fwd, rc);
            Kmer<NW> canon = sm ? fwd : rc;
            u64 slot = table_find(tab, canon);
            if (slot == ~0ull) { atomicAdd(err, 1ull); stop = true; break; }
            const Slot<NW>* nd = tab.slots + slot;
            u64 p = nd->payload;
            if ((p & PL_DELETED) || ((p & PL_LINEAR) && !pl_inedge(p))) {      // deleted or in a floating loop
                if (retain < 2) { retain = 0; pos = 0; continue; }              // NB IsPrev / prevK are NOT reset
                stop = true;
                break;
            }
            if (p & PL_LINEAR) {
                u32 eid = (u32)nd->aux;
                u32 ei = sm ? eid : eid + pl_twin(p) - 1;
                if (retain == 0 || IsPrev) { retain++; mix[pos++] = ei; IsPrev = false; }
                else if (ei != mix[pos - 1]) { retain++; mix[pos++] = ei; }
            } else {
                // currentKmer = the node's k-mer in read orientation = fwd
                if (IsPrev) {
                    retain++;
                    Kmer<NW> w = kshl2(prevK);
                    w.w[NW - 1] |= klast(fwd);
                    Kmer<NW> bw = krc_ref(w, K + 1, quirk128);
                    bool wsm = kless(w, bw);
                    u64 v = patch_find(patch, pmask, wsm ? w : bw);
                    u32 id = 0;
                    if (v) { u32 e = (u32)v; u32 tw = (u32)((v >> 32) & 3); id = wsm ? e : e + tw - 1; }
                    mix[pos++] = id;
                }
                IsPrev = true;
                prevK = fwd;
            }
        }
        if (retain < 1) deleted_reads++;
        int np = retain < 2 ? 0 : pos;
        for (int j = 0; j + 1 < np; j++) {                                     // thread_add1preArc
            if (mix[j] == 0 || mix[j + 1] == 0) break;
            if (!arc_add(arcs, amask, mix[j], mix[j + 1], (ord << 16) | (u64)j)) { atomicAdd(err + 1, 1ull); break; }
        }
        if (repsTie) {                                                         // recordPathBin
            u32 cnt = 0;
            if (n >= 3 && np >= 3 && mix[0] && mix[1] && mix[2]) {
                while ((int)cnt < np && mix[cnt]) { atomicAdd(&marker[mix[cnt]], 1u); cnt++; }
            }
            reclen[ord] = cnt ? 1 + 4 * (cnt & 255u) : 0;   // the count is an unsigned char in the reference
            mix[stride - 1] = cnt;                          // remembered for the writer (pos <= n <= stride - 1)
        }
    }
    if (deleted_reads) atomicAdd(&counters[C_MISC0], (u64)deleted_reads);
}

__global__ void __launch_bounds__(128) k_write_paths(const u32* __restrict__ lens, u64 n_rec, int K, u64 ord_base, u64 ord_stride, int stride,
                                                     const u32* pathbuf, const u32* reclen, const u64* recoff, unsigned char* out) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < n_rec; r += (u64)gridDim.x * blockDim.x) {
        if ((int)lens[r] < K + 1) continue;
        u64 ord = ord_base + r * ord_stride;
        if (!reclen[ord]) continue;
        const u32* mix = pathbuf + r * (u64)stride;
        u32 cnt = mix[stride - 1] & 255u;
        unsigned char* o = out + recoff[ord];
        *o++ = (unsigned char)cnt;
        for (u32 j = 0; j < cnt; j++) { u32 v = mix[j]; o[0] = v; o[1] = v >> 8; o[2] = v >> 16; o[3] = v >> 24; o += 4; }
    }
}

struct RecIn {
    const u32* reclen;
    __device__ u64 operator()(u64 i) const { return reclen[i]; }
};
struct RecOut {
    u64* off;
    __device__ void operator()(u64 i, u64 prefix, u64) const { off[i] = prefix; }
};
struct CountOnly {
    __device__ void operator()(u64, u64, u64) const {}
};
struct ArcOccIn {
    const ArcSlot* t;
    __device__ u64 operator()(u64 i) const { return t[i].key != EMPTY64; }
};
struct ArcCompactOut {
    const ArcSlot* t;
    ArcSlot* out;
    __device__ void operator()(u64 i, u64 prefix, u64 v) const { if (v) out[prefix] = t[i]; }
};

template <int NW>
void EngineT<NW>::pass2(Pass2Stats* st, std::string* prearc_text, std::string* path_bin, std::string* mark_text) {
    if (!patch_buf_.p) throw std::runtime_error("pgb200: pass2 before build_edges");
    const int K = prm_.K;
    const int stride = prm_.max_rd_len - K + 1 + 1;   // path entries + one bookkeeping word
    const bool quirk128 = prm_.flavour127 && K + 1 == 128;
    u64 total_ord = 0, max_rec = 0;
    for (auto& c : chunks_) {
        if (c.n_rec) total_ord = std::max(total_ord, c.ord_base + (c.n_rec - 1) * c.ord_stride + 1);
        max_rec = std::max(max_rec, c.n_rec);
    }
    // arc table: a proper de Bruijn graph has <= 4 arcs per edge; leave generous head room and fail loudly if exceeded
    u64 acap = 1024;
    while (acap < 16 * num_ed_ + 1024) acap <<= 1;
    DevBuf arcb, markb, reclenb, recoffb, errb, scratch;
    arcb.alloc(acap * sizeof(ArcSlot));
    PG_CUDA(cudaMemsetAsync(arcb.p, 0xFF, acap * sizeof(ArcSlot), st_));
    markb.alloc((num_ed_ + 2) * sizeof(u32));
    PG_CUDA(cudaMemsetAsync(markb.p, 0, (num_ed_ + 2) * sizeof(u32), st_));
    errb.alloc(2 * sizeof(u64));
    PG_CUDA(cudaMemsetAsync(errb.p, 0, 2 * sizeof(u64), st_));
    PG_CUDA(cudaMemsetAsync(d_cnt_ + C_MISC0, 0, sizeof(u64), st_));
    if (prm_.repsTie) {
        reclenb.alloc((total_ord + 1) * sizeof(u32));
        PG_CUDA(cudaMemsetAsync(reclenb.p, 0, (total_ord + 1) * sizeof(u32), st_));
    }
    ArcSlot* arcs = arcb.template as<ArcSlot>();
    // zero the count words (memset 0xFF made them ~0): one strided memset
    PG_CUDA(cudaMemset2DAsync(&arcs[0].count, sizeof(ArcSlot), 0, sizeof(u64), acap, st_));
    std::vector<DevBuf> pathbufs(chunks_.size());
    DevBuf shared_path;
    if (!prm_.repsTie) shared_path.alloc(std::max<u64>(1, max_rec) * (u64)stride * sizeof(u32));
    const size_t smem = (size_t)128 * W64_ * sizeof(u64);
    const int use_tma = smem <= 48 * 1024 && !getenv("PGB200_NO_TMA");
    // (the kernel's static shared memory comes on top of the tile: a 48 KB tile, max_rd_len 1505..1536, needs the opt-in)
    if (use_tma) PG_CUDA(cudaFuncSetAttribute(k_pass2<NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (size_t ci = 0; ci < chunks_.size(); ci++) {
        ReadChunk& c = chunks_[ci];
        if (!c.n_rec) continue;
        u32* pb;
        if (prm_.repsTie) { pathbufs[ci].alloc(c.n_rec * (u64)stride * sizeof(u32)); pb = pathbufs[ci].template as<u32>(); }
        else pb = shared_path.template as<u32>();
        unsigned blocks = (unsigned)std::min<u64>((c.n_rec + 127) / 128, 148ull * 32);
        k_pass2<NW><<<blocks, 128, use_tma ? smem : 0, st_>>>(tab_, kp_, c.words, c.len, c.n_rec, W64_, c.ord_base, c.ord_stride, stride, pb,
                                             reclenb.template as<u32>(), prm_.repsTie, patch_buf_.template as<PatchSlot<NW>>(), patch_mask_,
                                             quirk128, arcs, acap - 1, markb.template as<u32>(), d_cnt_, errb.template as<u64>(), use_tma);
        PG_CUDA(cudaGetLastError());
    }
    u64 herr[2];
    PG_CUDA(cudaMemcpyAsync(herr, errb.p, sizeof herr, cudaMemcpyDeviceToHost, st_));
    read_counters();
    if (herr[0]) throw std::runtime_error("pgb200: pass-2 k-mer lookup missed (the reference only prints a message here)");
    if (herr[1]) throw std::runtime_error("pgb200: pre-arc table overflow");
    st->deleted_reads = h_cnt_[C_MISC0];

    // ---- arcs: compact, copy, order by (from asc, first-seen rank desc), print (output_arcs)
    scratch.alloc(scan_scratch_elems(std::max<u64>(acap, total_ord + 1)) * sizeof(u64));
    DevBuf compb;
    device_scan(ArcOccIn{arcs}, CountOnly{}, acap, scratch.template as<u64>(), d_cnt_ + C_MISC1, st_);
    read_counters();
    u64 n_arcs = h_cnt_[C_MISC1];
    compb.alloc((n_arcs + 1) * sizeof(ArcSlot));
    device_scan(ArcOccIn{arcs}, ArcCompactOut{arcs, compb.template as<ArcSlot>()}, acap, scratch.template as<u64>(), d_cnt_ + C_MISC1, st_);
    std::vector<ArcSlot> h(n_arcs);
    if (n_arcs) PG_CUDA(cudaMemcpyAsync(h.data(), compb.p, n_arcs * sizeof(ArcSlot), cudaMemcpyDeviceToHost, st_));
    sync();
    std::sort(h.begin(), h.end(), [](const ArcSlot& a, const ArcSlot& b) {
        u32 fa = (u32)(a.key >> 32), fb = (u32)(b.key >> 32);
        if (fa != fb) return fa < fb;
        return a.rank > b.rank;   // head insertion: the most recently created arc comes first
    });
    std::string& s = *prearc_text;
    s.clear();
    s.reserve(n_arcs * 16 + 16);
    char b[64];
    for (u64 i = 0; i < n_arcs;) {
        u32 from = (u32)(h[i].key >> 32);
        s.append(b, snprintf(b, sizeof b, "%u", from));
        for (; i < n_arcs && (u32)(h[i].key >> 32) == from; i++) s.append(b, snprintf(b, sizeof b, " %u %u", (u32)h[i].key, (u32)h[i].count));
        s.push_back('\n');
    }
    st->arcs = n_arcs;

    // ---- -R: .path (binary, read-stream order) and .markOnEdge
    path_bin->clear();
    mark_text->clear();
    if (prm_.repsTie) {
        recoffb.alloc((total_ord + 1) * sizeof(u64));
        device_scan(RecIn{reclenb.template as<u32>()}, RecOut{recoffb.template as<u64>()}, total_ord, scratch.template as<u64>(), d_cnt_ + C_MISC2, st_);
        read_counters();
        u64 pbytes = h_cnt_[C_MISC2];
        DevBuf outb;
        outb.alloc(pbytes + 16);
        for (size_t ci = 0; ci < chunks_.size(); ci++) {
            ReadChunk& c = chunks_[ci];
            if (!c.n_rec) continue;
            unsigned blocks = (unsigned)std::min<u64>((c.n_rec + 127) / 128, 148ull * 32);
            k_write_paths<<<blocks, 128, 0, st_>>>(c.len, c.n_rec, K, c.ord_base, c.ord_stride, stride, pathbufs[ci].template as<u32>(),
                                                   reclenb.template as<u32>(), recoffb.template as<u64>(), outb.template as<unsigned char>());
            PG_CUDA(cudaGetLastError());
        }
        path_bin->resize(pbytes);
        if (pbytes) PG_CUDA(cudaMemcpyAsync(&(*path_bin)[0], outb.p, pbytes, cudaMemcpyDeviceToHost, st_));
        std::vector<u32> hm(num_ed_ + 2);
        PG_CUDA(cudaMemcpyAsync(hm.data(), markb.p, (num_ed_ + 2) * sizeof(u32), cudaMemcpyDeviceToHost, st_));
        sync();
        u64 markers = 0;
        mark_text->reserve(num_ed_ * 3 + 16);
        for (u64 i = 1; i <= num_ed_; i++) {
            markers += hm[i];
            mark_text->append(b, snprintf(b, sizeof b, "%d\n", (int)std::min<u32>(hm[i], 255u)));
        }
        st->markers = markers;
    }
}

template void EngineT<2>::pass2(Pass2Stats*, std::string*, std::string*, std::string*);
template void EngineT<4>::pass2(Pass2Stats*, std::string*, std::string*, std::string*);

}   // namespace pgb
