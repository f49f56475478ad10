// engine.cu — the C ABI of libflowagg.so (include/flowagg.h) and the host-side engine:
// device memory, streams, staging of host batches, the ACCOUNTER "full" logic, stats.
// There is NO CPU fallback: without a CUDA device fa_create fails with FA_E_NODEV.
#include <cuda_runtime.h>

#include <array>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/flowagg.h"
#include "flowgen.h"
#include "kernels.cuh"
#include "kmap_body.cuh"

static_assert(sizeof(fa_flow_id) == 40, "flow_id ABI");
static_assert(sizeof(fa_flow_metrics) == 104, "flow_metrics ABI");
static_assert(sizeof(fa_flow_record) == 144, "flow_record ABI");
static_assert(sizeof(fa_dns_metrics) == 64, "dns_metrics ABI");
static_assert(sizeof(fa_additional_metrics) == 32, "additional_metrics ABI");
static_assert(sizeof(fa_dns_record) == 104 && sizeof(fa_additional_record) == 72, "feature record ABI");
static_assert(offsetof(fa_flow_metrics, if_index_first_seen) == 44 && offsetof(fa_flow_metrics, observed_intf) == 68 &&
              offsetof(fa_flow_metrics, ssl_version) == 92 && offsetof(fa_flow_metrics, misc_flags) == 99, "flow_metrics offsets");
static_assert(offsetof(fa_dns_metrics, name) == 31 && offsetof(fa_additional_metrics, ipsec_encrypted) == 30, "feature offsets");

namespace {

thread_local std::string g_err;
int fail(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    g_err = buf;
    return code;
}
#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) return fail(FA_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

enum PtrKind { PTR_PAGEABLE, PTR_PINNED, PTR_DEVICE };
PtrKind classify(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return PTR_PAGEABLE; }
    if (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) return PTR_DEVICE;
    if (a.type == cudaMemoryTypeHost) return PTR_PINNED;
    return PTR_PAGEABLE;
}

// ---------------------------------------------------------------- Zipf threshold tables
struct ZipfTable {
    std::vector<uint64_t> thresholds;
    std::vector<uint32_t> first, size;
    uint64_t* d_thresholds = nullptr; uint32_t* d_first = nullptr; uint32_t* d_size = nullptr;   // per device, lazily
    int device = -1;
};
std::mutex g_zipf_mu;
std::map<std::pair<uint64_t, uint32_t>, ZipfTable*> g_zipf;

// Ranks 1..N split into octaves [2^o, 2^(o+1)), each octave into <= 256 equal sub-ranges.
ZipfTable* zipf_table(uint64_t n_keys, uint32_t s_milli) {
    std::lock_guard<std::mutex> lk(g_zipf_mu);
    auto key = std::make_pair(n_keys, s_milli);
    auto it = g_zipf.find(key);
    if (it != g_zipf.end()) return it->second;
    ZipfTable* z = new ZipfTable();
    const double s = s_milli / 1000.0;
    std::vector<long double> mass;
    for (uint64_t lo = 1; lo <= n_keys; lo <<= 1) {
        const uint64_t hi = std::min<uint64_t>(n_keys + 1, lo << 1);      // ranks [lo, hi)
        const uint64_t span = hi - lo;
        const uint64_t parts = std::min<uint64_t>(span, 256);
        for (uint64_t pi = 0; pi < parts; pi++) {
            const uint64_t a = lo + span * pi / parts, b = lo + span * (pi + 1) / parts;
            long double m = 0;
            for (uint64_t k = a; k < b; k++) m += std::pow((double)k, -s);
            z->first.push_back((uint32_t)(a - 1));
            z->size.push_back((uint32_t)(b - a));
            mass.push_back(m);
        }
    }
    long double total = 0; for (auto m : mass) total += m;
    long double run = 0;
    z->thresholds.resize(mass.size());
    for (size_t i = 0; i < mass.size(); i++) {
        run += mass[i];
        long double f = run / total * 18446744073709551616.0L;
        z->thresholds[i] = f >= 18446744073709551615.0L ? ~0ull : (uint64_t)f;
    }
    z->thresholds.back() = ~0ull;
    g_zipf[key] = z;
    return z;
}

}  // namespace

// ------------------------------------------------------------------------ engine
// Owner of one device (cudaMalloc) or pinned host (cudaHostAlloc) allocation; it converts to the raw pointer.
// reserve(need, want) grows it: when it holds fewer than `need` bytes it frees the buffer and allocates max(need, want)
// bytes, without copying the contents.
template <class T, bool kPinned>
class Buf {
  public:
    Buf() = default;
    Buf(Buf&& o) noexcept { swap(o); }
    Buf& operator=(Buf&& o) noexcept { swap(o); return *this; }
    ~Buf() { reset(); }
    cudaError_t reserve(size_t need, size_t want = 0) {
        if (need <= bytes_) return cudaSuccess;
        reset();
        void* p = nullptr;
        want = std::max(need, want);
        const cudaError_t r = kPinned ? cudaHostAlloc(&p, want, cudaHostAllocDefault) : cudaMalloc(&p, want);
        if (r == cudaSuccess) { p_ = static_cast<T*>(p); bytes_ = want; }
        return r;
    }
    void swap(Buf& o) noexcept { std::swap(p_, o.p_); std::swap(bytes_, o.bytes_); }
    T* get() const { return p_; }
    operator T*() const { return p_; }
    T* operator->() const { return p_; }

  private:
    void reset() {
        if (p_) { if (kPinned) cudaFreeHost(p_); else cudaFree(p_); }
        p_ = nullptr; bytes_ = 0;
    }
    T* p_ = nullptr;
    size_t bytes_ = 0;
};
template <class T> using DevBuf = Buf<T, false>;
template <class T> using PinnedBuf = Buf<T, true>;

// The flow table's arrays.  Kernels take the plain fa::Table view by value.
struct FlowTable {
    DevBuf<uint4> ident, hot, feat_add, feat_dns, feat_drop;
    DevBuf<uint32_t> occ;
    uint64_t mask = 0;
    fa::Table view() const { return {ident, hot, feat_add, feat_dns, feat_drop, occ, mask}; }
    bool has_features() const { return feat_add || feat_dns || feat_drop; }
};

static uint64_t pow2_at_least(uint64_t p, uint64_t want) { while (p < want) p <<= 1; return p; }   // p: a power of two

struct fa_engine {
    fa_config cfg{};
    int device = 0, sm_count = 148;
    cudaStream_t stream = nullptr; bool own_stream = false;
    cudaStream_t copy_stream = nullptr;
    std::mutex mu;

    FlowTable table;
    uint64_t slots = 0, epoch = 0;
    // FA_F_NONBLOCKING_EVICT: a second, empty table.  fa_evict swaps the two under `mu` (the Accounter hands its map
    // over and goes on with a fresh one, pkg/flow/account.go:67-68,86-87) and scans the retired one on its own stream.
    FlowTable table_spare;
    bool double_buffered = false;
    std::mutex evict_mu;                      // one eviction at a time (the reference's evictor is single-flight)
    cudaStream_t evict_stream = nullptr;
    cudaEvent_t ev_swap = nullptr;
    DevBuf<fa::Counters> d_ctr_ev;            // evict_out cursor of the scan of the retired table
    PinnedBuf<unsigned long long> h_ev_out;
    DevBuf<fa::Counters> d_ctr;
    PinnedBuf<fa::Counters> h_ctr;            // mirror of d_ctr
    uint64_t max_batch = 0;

    // staging for host input (double buffered)
    DevBuf<uint8_t> d_stage[2];
    PinnedBuf<uint8_t> h_stage[2];
    cudaEvent_t ev_stage_free[2] = {nullptr, nullptr};   // kernel that consumed the stage finished
    cudaEvent_t ev_copied[2] = {nullptr, nullptr};       // H2D copy into the stage finished
    int stage_cur = 0;

    DevBuf<fa::FixupScratch> d_scratch; uint32_t scratch_slots = 0;
    DevBuf<uint32_t> d_spill_idx;
    DevBuf<uint32_t> d_cut_set; uint32_t cut_set_slots = 0;
    DevBuf<uint32_t> d_cut_bitmap, d_cut_out; PinnedBuf<uint32_t> h_cut_out;

    DevBuf<uint8_t> d_expanded;               // 144-byte expansion of events, and records parsed out of snapshots
    DevBuf<uint32_t> d_snap_src;              // fa_ingest_snaps: snapshot index of every record parsed out of a chunk
    DevBuf<uint32_t> d_snap_cnt;              // ... records per CTA of the parse kernels, then the total + 3 filter counters (u64)
    DevBuf<uint8_t> d_snap_verdict;           // ... with a flow filter: keep / skip per snapshot of the chunk
    fa::FilterSet filter{};                   // fa_set_flow_filter (n_rules == 0: no filter)
    DevBuf<uint8_t> d_evict;                  // eviction records for host memory, grown on demand
    DevBuf<uint8_t> d_evict_dns, d_evict_add, d_evict_drop, d_evict_rttmin, d_evict_present;   // ... and its feature outputs
    DevBuf<uint32_t> d_slot_of_out;
    DevBuf<uint32_t> d_slot_of;               // per-sample slot scratch of the feature folds
    uint64_t feat_seq[3] = {0, 0, 0};         // running sample numbers (additional, dns, packet drops)
    DevBuf<uint32_t> d_route_tmp; DevBuf<unsigned long long> d_route_counts;

    fa::SketchParams sk{};                    // cms / hll point into sk_cms / sk_hll
    DevBuf<unsigned long long> sk_cms; DevBuf<uint32_t> sk_hll;
    DevBuf<unsigned long long> d_prof;        // FA_PHASE_PROFILE=1: per-phase warp-cycle counters of K1
#ifndef FA_K1_DEFAULT_OPT
#define FA_K1_DEFAULT_OPT 0u                  // K1 switches an engine starts with (kernels.cuh, AggLaunch::opt); FA_K1_OPT overrides (diagnostics)
#endif
    uint32_t k1_opt = FA_K1_DEFAULT_OPT;

    // live-flow bookkeeping for the "full" rule: live_known is exact as of the last retired
    // launch; unsynced_records bounds the flows that launches still in flight can add.
    uint64_t live_known = 0;
    uint64_t unsynced_records = 0;
    static constexpr int kLiveRing = 8;
    PinnedBuf<unsigned long long> h_live_ring;   // kLiveRing entries
    cudaEvent_t ev_live[kLiveRing] = {};
    uint32_t ring_n[kLiveRing] = {};
    uint32_t ring_head = 0, ring_tail = 0;       // monotonically increasing; slot = idx % kLiveRing

    // KERNEL_MAP mode (kmap.cu): metrics lines, per-batch scratch, fallback ring
    DevBuf<uint8_t> km_met;
    DevBuf<uint32_t> km_slot_of;
    DevBuf<fa::KmBEntry> km_bset; uint32_t km_bset_slots = 0;
    DevBuf<uint32_t> km_blist;
    DevBuf<uint32_t> km_touched, km_deferred, km_brec;   // v2 work lists
    int km_impl = 2;                          // FA_KMAP_IMPL: 1 = seven per-record passes, 2 = per-flow finalisation
    DevBuf<uint8_t> km_spill; uint64_t km_spill_cap = 0;
    DevBuf<fa::KmCounters> d_km_ctr;
    PinnedBuf<fa::KmCounters> h_km_ctr;       // mirror of d_km_ctr
    uint64_t km_spilled_total = 0;            // records read back by fa_read_spilled so far

    // K8 scratch (fa_pb_encode), grown on demand
    DevBuf<uint32_t> d_pb_sizes; DevBuf<unsigned long long> d_pb_offsets, d_pb_sums;
    DevBuf<fa::PbIface> d_pb_ifaces;

    // K7 (dnscorr.cu): the dns_flows map + per-chunk scratch, allocated by the first fa_ingest_dns_packets
    fa::DnsCorr dnsc{};                       // tab == nullptr until then; tab / ctr point into dnsc_tab / dnsc_ctr
    DevBuf<fa::DnsEntry> dnsc_tab, dnsc_spare;   // the map, and the other table of a rebuild
    DevBuf<unsigned long long> dnsc_ctr;
    PinnedBuf<unsigned long long> h_dnsc_ctr; // mirror of dnsc_ctr
    DevBuf<uint32_t> d_dnsc_state, d_dnsc_warps; DevBuf<uint8_t> d_dnsc_samples, d_dnsc_out;
    uint64_t dnsc_chunk = 0;                  // packets per launch_dns_correlate
    uint64_t dnsc_used = 0;                   // upper bound of the table entries in use (present + answered keys)
    uint64_t dnsc_slots = 0;                  // 4 x max_entries: answered keys keep their entry until the next rebuild

    fa_stats st{};
};

namespace fa {
int launch_kmap_batch(KmParams P, uint32_t cut, int sm_count, cudaStream_t st);
int launch_kmap_batch_v2(KmParams P, uint32_t cut, int sm_count, cudaStream_t st);
int launch_kmap_evict(const Table& t, uint8_t* met, uint8_t* out, unsigned long long cap, unsigned long long* cursor,
                      uint32_t* slot_of_out, int sm_count, cudaStream_t st);
}

namespace {

int sync_counters(fa_engine* e) {
    CU(cudaMemcpyAsync(e->h_ctr, e->d_ctr, sizeof(fa::Counters), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    e->live_known = e->h_ctr->live;
    e->unsynced_records = 0;
    e->ring_head = e->ring_tail;
    return FA_OK;
}

// Retire launches whose live-count read-back has landed (never blocks).
void retire_completed(fa_engine* e) {
    while (e->ring_head != e->ring_tail) {
        const uint32_t s = e->ring_head % fa_engine::kLiveRing;
        if (cudaEventQuery(e->ev_live[s]) != cudaSuccess) { cudaGetLastError(); break; }
        e->live_known = e->h_live_ring[s];
        e->unsynced_records -= e->ring_n[s];
        e->ring_head++;
    }
}

// Book-keeping after the launches of one chunk: asynchronous read-back of the live-flow count.
int note_launch(fa_engine* e, uint32_t n) {
    e->unsynced_records += n;
    e->st.records_ingested += n;
    if (e->ring_tail - e->ring_head == fa_engine::kLiveRing) {
        CU(cudaEventSynchronize(e->ev_live[e->ring_head % fa_engine::kLiveRing]));
        retire_completed(e);
    }
    const uint32_t s = e->ring_tail % fa_engine::kLiveRing;
    CU(cudaMemcpyAsync(&e->h_live_ring[s], &e->d_ctr->live, 8, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaEventRecord(e->ev_live[s], e->stream));
    e->ring_n[s] = n;
    e->ring_tail++;
    return FA_OK;
}

// Launch K1 on a device-resident chunk (n <= max_batch).
int launch_chunk(fa_engine* e, const uint8_t* d_recs, uint32_t n) {
    fa::AggLaunch a{};
    a.recs = reinterpret_cast<const uint4*>(d_recs);
    a.n = n;
    a.table = e->table.view();
    a.epoch = ++e->epoch;
    a.ctr = e->d_ctr;
    a.spill_idx = e->d_spill_idx;
    a.sk = (e->cfg.flags & FA_F_ENABLE_SKETCH) ? e->sk : fa::SketchParams{};
    a.scratch = e->d_scratch;
    a.scratch_slots = e->scratch_slots;
    a.sm_count = e->sm_count;
    a.prof = e->d_prof;
    a.opt = e->k1_opt;
    e->st.kernel_launches += fa::launch_aggregate(a, e->stream);
    CU(cudaGetLastError());
    return note_launch(e, n);
}

// How many of the next n records to hand to a cache that may fill.  ACCOUNTER mode cuts a chunk after roughly `room`
// new keys, so it gets a window proportional to the room left: the work stays linear in the records consumed however
// small the cache is, and a "full" return does not leave most of a staged chunk unused (the caller hands the rest in
// again after its eviction).  Other modes take all n.
uint64_t room_window(fa_engine* e, uint64_t n) {
    if (e->cfg.mode != FA_MODE_ACCOUNTER || (e->cfg.flags & FA_F_NO_FULL_CUT)) return n;
    retire_completed(e);
    const uint64_t used = e->live_known + e->unsynced_records;
    const uint64_t room = e->cfg.max_entries > used ? e->cfg.max_entries - used : 0;
    return std::min<uint64_t>(n, std::max<uint64_t>(4096, 4 * room));
}

// *cut = index of the first of the n records whose key is new while the cache holds max_entries flows (n: none).
// e->live_known must be exact.
int full_cut(fa_engine* e, const uint8_t* d_recs, uint32_t n, uint32_t* cut) {
    e->st.kernel_launches += fa::launch_full_cut(reinterpret_cast<const uint4*>(d_recs), n, e->table.view(), e->live_known,
                                                 e->cfg.max_entries, e->d_cut_set, e->cut_set_slots, e->d_cut_bitmap,
                                                 e->d_cut_out, e->sm_count, e->stream);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(e->h_cut_out, e->d_cut_out, 4, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    *cut = *e->h_cut_out;
    return FA_OK;
}

// ACCOUNTER mode: fold a device-resident chunk honouring max_entries.
// Returns FA_OK (all folded) or FA_FULL with *consumed < n.
int ingest_chunk_accounter(fa_engine* e, const uint8_t* d_recs, uint32_t n, uint32_t* consumed) {
    *consumed = 0;
    const uint64_t M = e->cfg.max_entries;
    retire_completed(e);
    if (e->cfg.flags & FA_F_NO_FULL_CUT) {              // max_entries only sizes the table
        int rc = launch_chunk(e, d_recs, n);
        if (rc) return rc;
        *consumed = n;
        return FA_OK;
    }
    // Launches still in flight may add up to unsynced_records flows.  When that bound does not leave room for this
    // chunk, wait for the OLDEST launch's live-count read-back only (the stream keeps working on the younger ones),
    // and drain the stream only when nothing is left in flight.
    while (e->live_known + e->unsynced_records + n > M && e->ring_head != e->ring_tail) {
        CU(cudaEventSynchronize(e->ev_live[e->ring_head % fa_engine::kLiveRing]));
        retire_completed(e);
    }
    if (e->live_known + e->unsynced_records + n > M && e->unsynced_records) {
        int rc = sync_counters(e);                     // exact live count (feature folds do not use the ring)
        if (rc) return rc;
    }
    if (e->live_known + e->unsynced_records + n <= M) { // cannot overflow: fast path
        int rc = launch_chunk(e, d_recs, n);
        if (rc) return rc;
        *consumed = n;
        return FA_OK;
    }
    // slow path: find the first record whose key is new while the cache is full.  The counters were just read, so the
    // room of the window is exact.  A window without a cut is folded and the caller goes on with the rest of its chunk.
    const uint32_t win = (uint32_t)room_window(e, n);
    uint32_t cut = 0;
    if (int rc = full_cut(e, d_recs, win, &cut)) return rc;
    if (cut > 0) {
        int rc = launch_chunk(e, d_recs, cut);
        if (rc) return rc;
        rc = sync_counters(e);
        if (rc) return rc;
    }
    *consumed = cut;
    if (cut < win) { e->st.full_cuts++; return FA_FULL; }
    return FA_OK;
}

// KERNEL_MAP mode: the map update of flow_monitor (bpf/flows.c:222-288) for a device-resident chunk.  The map
// never "fills and flushes": once max_entries flows are live, packets of unknown flows go to the fallback ring
// (or only count), so the whole chunk is always consumed.
int ingest_chunk_kmap(fa_engine* e, const uint8_t* d_recs, uint32_t n, uint32_t* consumed) {
    *consumed = 0;
    const uint64_t M = e->cfg.max_entries;
    retire_completed(e);
    if (e->live_known + e->unsynced_records + n > M) {
        int rc = sync_counters(e);                     // exact live count
        if (rc) return rc;
    }
    uint32_t cut = n;                                  // records [cut, n) find the map full
    if (e->live_known + e->unsynced_records + n > M) {
        if (int rc = full_cut(e, d_recs, n, &cut)) return rc;
        if (cut < n) e->st.full_cuts++;
    }
    fa::KmParams P{};
    P.recs = d_recs; P.n = n;
    P.ringbuf = (e->cfg.flags & FA_F_RINGBUF_FALLBACK) ? 1 : 0;
    P.t = e->table.view(); P.met = e->km_met;
    P.epoch = ++e->epoch;
    P.slot_of = e->km_slot_of;
    P.live = &e->d_ctr->live;
    P.c = e->d_km_ctr;
    P.spill = e->km_spill; P.spill_cap = e->km_spill_cap;
    P.bset = e->km_bset; P.bset_mask = e->km_bset_slots - 1; P.blist = e->km_blist;
    P.touched = e->km_touched; P.deferred = e->km_deferred; P.brec = e->km_brec;
    e->st.kernel_launches += e->km_impl == 1 ? fa::launch_kmap_batch(P, cut, e->sm_count, e->stream)
                                             : fa::launch_kmap_batch_v2(P, cut, e->sm_count, e->stream);
    CU(cudaGetLastError());
    *consumed = n;
    return note_launch(e, n);
}

int ingest_chunk(fa_engine* e, const uint8_t* d_recs, uint32_t n, uint32_t* consumed) {
    return e->cfg.mode == FA_MODE_KERNEL_MAP ? ingest_chunk_kmap(e, d_recs, n, consumed)
                                             : ingest_chunk_accounter(e, d_recs, n, consumed);
}

int ingest_device(fa_engine* e, const uint8_t* d_recs, size_t n, size_t* consumed) {
    size_t done = 0;
    while (done < n) {
        const uint32_t c = (uint32_t)std::min<size_t>(n - done, e->max_batch);
        uint32_t took = 0;
        int rc = ingest_chunk(e, d_recs + done * fa::kRecBytes, c, &took);
        done += took;
        if (rc != FA_OK) { if (consumed) *consumed = done; return rc; }
    }
    if (consumed) *consumed = done;
    return FA_OK;
}

// Host data reaches the device through two staging buffers of stage_records() records: the copy of chunk k+1 (copy
// stream) overlaps the kernels of chunk k (engine stream).  The staging grain is independent of max_batch, the K1
// launch size for device-resident input: a large launch amortises K1's start-up, a small stage keeps the pipeline fine.
static uint64_t stage_records(const fa_engine* e) { return std::min<uint64_t>(e->max_batch, 1ull << 20); }   // 151 MB of records per copy

static int stage_alloc(fa_engine* e, bool pageable) {
    const size_t bytes = stage_records(e) * fa::kRecBytes;
    for (int i = 0; i < 2; i++) {
        CU(e->d_stage[i].reserve(bytes));
        if (pageable) CU(e->h_stage[i].reserve(bytes));
    }
    return FA_OK;
}

// Copy `bytes` of host data into the next staging buffer; the engine stream waits for the copy.  -> *sidx for stage_release.
static int stage_copy(fa_engine* e, const uint8_t* src, size_t bytes, bool pinned, int* sidx_out) {
    const int sidx = e->stage_cur; e->stage_cur ^= 1;
    CU(cudaEventSynchronize(e->ev_stage_free[sidx]));                // previous consumer of this stage is done
    if (!pinned) { memcpy(e->h_stage[sidx], src, bytes); src = e->h_stage[sidx]; }
    CU(cudaMemcpyAsync(e->d_stage[sidx], src, bytes, cudaMemcpyHostToDevice, e->copy_stream));
    CU(cudaEventRecord(e->ev_copied[sidx], e->copy_stream));
    CU(cudaStreamWaitEvent(e->stream, e->ev_copied[sidx], 0));
    e->st.h2d_bytes += bytes;
    *sidx_out = sidx;
    return FA_OK;
}

static int stage_release(fa_engine* e, int sidx) {                   // the kernels enqueued so far were the stage's last readers
    CU(cudaEventRecord(e->ev_stage_free[sidx], e->stream));
    return FA_OK;
}

// One chunk of caller memory as the device reads it: the caller's device memory in place, or a staging buffer.
struct Chunk {
    fa_engine* e;
    const uint8_t* d;
    int sidx;                                  // staging buffer, -1: none (or already released)
    int release() {                            // the work enqueued so far was the chunk's last reader
        const int s = sidx;
        sidx = -1;
        return s >= 0 ? stage_release(e, s) : FA_OK;
    }
};

// Walks n items of `width` bytes of caller memory chunk by chunk.  Device memory (`align`-byte aligned) is read in
// place; host memory goes through the staging buffers.  For each chunk, rule(left, staged, &c) sets its size c and may
// enqueue work that has to come first; body(chunk, c, &took) enqueues the chunk's work, calls chunk.release() as soon
// as the rest of that work no longer reads the chunk, and sets how many items it consumed.  The walk stops at the first
// rule or body that does not return FA_OK.  The caller's buffer is not referenced after return.
template <class Rule, class Body>
int ingest_caller_memory(fa_engine* e, const char* who, const char* what, unsigned align, const void* src, size_t n,
                         size_t width, size_t* consumed, Rule rule, Body body) {
    const PtrKind k = classify(src);
    if (k == PTR_DEVICE && (reinterpret_cast<uintptr_t>(src) & (align - 1)))
        return fail(FA_E_INVAL, "%s: device %s must be %u-byte aligned", who, what, align);
    const bool staged = k != PTR_DEVICE;
    if (staged) { if (int rc = stage_alloc(e, k == PTR_PAGEABLE)) return rc; }
    size_t done = 0;
    int rc = FA_OK;
    while (rc == FA_OK && done < n) {
        size_t c = 0, took = 0;
        if ((rc = rule(n - done, staged, &c))) break;
        Chunk ch{e, static_cast<const uint8_t*>(src) + done * width, -1};
        if (staged) {
            if ((rc = stage_copy(e, ch.d, c * width, k == PTR_PINNED, &ch.sidx))) break;
            ch.d = e->d_stage[ch.sidx];
        }
        rc = body(ch, c, &took);
        if (int rel_rc = ch.release()) rc = rel_rc;
        done += took;
    }
    if (consumed) *consumed = done;
    if (staged) CU(cudaStreamSynchronize(e->copy_stream));
    return rc;
}

// Feature samples may create flows: never let the table pass 7/8 of its slots.
int check_headroom(fa_engine* e, size_t n, const char* who, const char* what) {
    if (int rc = sync_counters(e)) return rc;
    if (e->live_known + n > e->slots - e->slots / 8)
        return fail(FA_E_2BIG, "%s: %zu %s could overfill the flow table (%llu live of %llu slots): evict first", who, n, what,
                    (unsigned long long)e->live_known, (unsigned long long)e->slots);
    return FA_OK;
}

// Allocates `bytes` for b and zeroes them on the engine's stream.
template <class T>
int alloc_zeroed(fa_engine* e, DevBuf<T>& b, size_t bytes) {
    CU(b.reserve(bytes));
    CU(cudaMemsetAsync(b, 0, bytes, e->stream));
    return FA_OK;
}

// fa_evict_out's optional per-flow outputs in the order they are copied back: the caller's pointer, the bytes per flow,
// and the device buffer that stages the output when the caller's pointer is host memory.
struct EvictOut { void* dst; size_t width; DevBuf<uint8_t>* stage; };
using EvictOuts = std::array<EvictOut, 5>;
EvictOuts evict_outputs(fa_engine* e, const fa_evict_out* o) {
    return {{{o->dns, 64, &e->d_evict_dns}, {o->additional, 32, &e->d_evict_add}, {o->pkt_drops, 32, &e->d_evict_drop},
             {o->rtt_min, 8, &e->d_evict_rttmin}, {o->present, 1, &e->d_evict_present}}};
}

// Grows an eviction buffer to `live` entries of `width` bytes, with room for twice as many (at most max_entries).
template <class T>
int reserve_evict(fa_engine* e, DevBuf<T>& b, uint64_t live, size_t width) {
    CU(b.reserve(live * width, std::max<uint64_t>(live, std::min<uint64_t>(e->cfg.max_entries, live * 2)) * width));
    return FA_OK;
}

// Where an eviction writes its records: the caller's device memory in place, else the engine's staging buffer.
int evict_records_dst(fa_engine* e, void* records, uint64_t live, uint8_t** d_out) {
    if (classify(records) == PTR_DEVICE) { *d_out = static_cast<uint8_t*>(records); return FA_OK; }
    if (int rc = reserve_evict(e, e->d_evict, live, fa::kRecBytes)) return rc;
    *d_out = e->d_evict;
    return FA_OK;
}

// Without feature tables, the feature outputs in host memory come back zeroed.
void zero_host_outputs(const EvictOuts& outs, uint64_t live) {
    for (const EvictOut& x : outs)
        if (x.dst && classify(x.dst) != PTR_DEVICE) memset(x.dst, 0, live * x.width);
}

}  // namespace

extern "C" {

uint32_t fa_abi_version(void) { return FA_ABI_VERSION; }
const char* fa_last_error(void) { return g_err.c_str(); }

int fa_create(const fa_config* cfg, fa_engine** out) {
    if (!cfg || !out) return fail(FA_E_INVAL, "fa_create: null argument");
    if (cfg->abi_version != FA_ABI_VERSION) return fail(FA_E_INVAL, "fa_create: abi_version %u != %u", cfg->abi_version, FA_ABI_VERSION);
    if (cfg->max_entries == 0) return fail(FA_E_INVAL, "fa_create: max_entries must be >= 1");
    if (cfg->mode != FA_MODE_ACCOUNTER && cfg->mode != FA_MODE_KERNEL_MAP) return fail(FA_E_INVAL, "fa_create: unknown mode %u", cfg->mode);
    const bool kmap = cfg->mode == FA_MODE_KERNEL_MAP;
    if (kmap) {
        if (cfg->flags & (FA_F_ENABLE_SKETCH | FA_F_NO_FULL_CUT))
            return fail(FA_E_INVAL, "fa_create: mode KERNEL_MAP does not take FA_F_ENABLE_SKETCH / FA_F_NO_FULL_CUT (flags 0x%x)", cfg->flags);
    } else if (cfg->flags & FA_F_RINGBUF_FALLBACK) {
        return fail(FA_E_INVAL, "fa_create: FA_F_RINGBUF_FALLBACK needs mode KERNEL_MAP");
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(FA_E_NODEV, "fa_create: no CUDA device; this engine has no CPU fallback");
    }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(FA_E_INVAL, "fa_create: device %d out of range (%d devices)", cfg->device, ndev);
    CU(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major < 10) return fail(FA_E_NODEV, "fa_create: device sm_%d%d is not Blackwell (sm_100a kernels only)", prop.major, prop.minor);

    fa_engine* e = new (std::nothrow) fa_engine();
    if (!e) return fail(FA_E_NOMEM, "fa_create: out of memory");
    struct Guard { fa_engine* e; ~Guard() { if (e) fa_destroy(e); } } guard{e};   // releases everything on any early return
    e->cfg = *cfg;
    e->device = cfg->device;
    e->sm_count = prop.multiProcessorCount;
    e->max_batch = std::min<uint64_t>(cfg->max_batch ? cfg->max_batch : (1ull << 22), 1ull << 28);
    if (cfg->cuda_stream) { e->stream = (cudaStream_t)cfg->cuda_stream; }
    else { CU(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking)); e->own_stream = true; }
    CU(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));

    // table: load factor <= 0.75 at max_entries
    const uint64_t slots = pow2_at_least(1024, (4 * cfg->max_entries + 2) / 3);   // 0.75 x 2^k entries get exactly 2^k slots
    e->slots = slots;
    e->table.mask = slots - 1;
    if (int rc = alloc_zeroed(e, e->table.ident, slots * fa::kIdentBytes)) return rc;
    if (!kmap) {
        if (int rc = alloc_zeroed(e, e->table.hot, slots * fa::kHotBytes)) return rc;
    } else {
        if (slots > (1ull << 30)) return fail(FA_E_INVAL, "fa_create: KERNEL_MAP mode supports at most 2^30 slots");
        if (int rc = alloc_zeroed(e, e->km_met, slots * fa::kMetLineBytes)) return rc;
        CU(e->km_slot_of.reserve(e->max_batch * 4));
        e->km_bset_slots = (uint32_t)pow2_at_least(1024, 2 * e->max_batch);
        if (int rc = alloc_zeroed(e, e->km_bset, (size_t)e->km_bset_slots * sizeof(fa::KmBEntry))) return rc;
        CU(e->km_blist.reserve(e->max_batch * 4));
        CU(e->km_touched.reserve(e->max_batch * 4));
        CU(e->km_deferred.reserve(e->max_batch * 4));
        CU(e->km_brec.reserve(e->max_batch * 4));
        if (const char* ki = getenv("FA_KMAP_IMPL")) e->km_impl = ki[0] == '1' ? 1 : 2;
        if (cfg->flags & FA_F_RINGBUF_FALLBACK) {
            e->km_spill_cap = 131072;                   // >= the 16 MiB direct_flows ring (bpf/maps_definition.h:7-11)
            CU(e->km_spill.reserve(e->km_spill_cap * fa::kRecBytes));
        }
        if (int rc = alloc_zeroed(e, e->d_km_ctr, sizeof(fa::KmCounters))) return rc;
        CU(e->h_km_ctr.reserve(sizeof(fa::KmCounters)));
        memset(e->h_km_ctr, 0, sizeof(fa::KmCounters));
    }
    if (int rc = alloc_zeroed(e, e->table.occ, slots / 8)) return rc;
    if (cfg->flags & FA_F_NONBLOCKING_EVICT) {
        if (kmap || (cfg->flags & (FA_F_ENABLE_RTT | FA_F_ENABLE_DNS | FA_F_ENABLE_PKT_DROP)))
            return fail(FA_E_INVAL, "fa_create: FA_F_NONBLOCKING_EVICT is available in ACCOUNTER mode without feature folds");
        e->table_spare.mask = slots - 1;
        if (int rc = alloc_zeroed(e, e->table_spare.ident, slots * fa::kIdentBytes)) return rc;
        if (int rc = alloc_zeroed(e, e->table_spare.hot, slots * fa::kHotBytes)) return rc;
        if (int rc = alloc_zeroed(e, e->table_spare.occ, slots / 8)) return rc;
        CU(cudaStreamCreateWithFlags(&e->evict_stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&e->ev_swap, cudaEventDisableTiming));
        if (int rc = alloc_zeroed(e, e->d_ctr_ev, sizeof(fa::Counters))) return rc;
        CU(e->h_ev_out.reserve(8));
        e->double_buffered = true;
    }
    if (cfg->flags & FA_F_ENABLE_RTT) { if (int rc = alloc_zeroed(e, e->table.feat_add, slots * 80)) return rc; }
    if (cfg->flags & FA_F_ENABLE_DNS) { if (int rc = alloc_zeroed(e, e->table.feat_dns, slots * 128)) return rc; }
    if (cfg->flags & FA_F_ENABLE_PKT_DROP) { if (int rc = alloc_zeroed(e, e->table.feat_drop, slots * 96)) return rc; }
    if (cfg->flags & (FA_F_ENABLE_RTT | FA_F_ENABLE_DNS | FA_F_ENABLE_PKT_DROP)) CU(e->d_slot_of.reserve(e->max_batch * 4));
    if (int rc = alloc_zeroed(e, e->d_ctr, sizeof(fa::Counters))) return rc;
    CU(e->h_ctr.reserve(sizeof(fa::Counters)));
    memset(e->h_ctr, 0, sizeof(fa::Counters));
    CU(e->h_live_ring.reserve(fa_engine::kLiveRing * 8));
    for (int i = 0; i < fa_engine::kLiveRing; i++) CU(cudaEventCreateWithFlags(&e->ev_live[i], cudaEventDisableTiming));

    for (int i = 0; i < 2; i++) {
        CU(cudaEventCreateWithFlags(&e->ev_stage_free[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&e->ev_copied[i], cudaEventDisableTiming));
    }
    // one entry per flow that needs the ordered re-fold in a launch: at most one per record, and never more than the
    // table has slots (entries are keyed by table slot)
    e->scratch_slots = (uint32_t)pow2_at_least(1024, 2 * std::min<uint64_t>(e->max_batch, e->slots));
    if (int rc = alloc_zeroed(e, e->d_scratch, (size_t)e->scratch_slots * sizeof(fa::FixupScratch))) return rc;
    CU(cudaStreamSynchronize(e->stream));
    CU(e->d_spill_idx.reserve(e->max_batch * sizeof(uint32_t)));
    e->cut_set_slots = (uint32_t)pow2_at_least(1024, 2 * e->max_batch);
    CU(e->d_cut_set.reserve((size_t)e->cut_set_slots * 4));
    CU(e->d_cut_bitmap.reserve((e->max_batch + 31) / 32 * 4 + 4));
    CU(e->d_cut_out.reserve(4));
    CU(e->h_cut_out.reserve(4));

    // sketches
    e->sk.log2w = cfg->cms_log2_width ? cfg->cms_log2_width : 20;
    e->sk.depth = cfg->cms_depth ? cfg->cms_depth : 4;
    e->sk.p = cfg->hll_precision ? cfg->hll_precision : 14;
    e->sk.seed = cfg->sketch_seed;
    if (e->sk.depth > 8 || e->sk.log2w < 4 || e->sk.log2w > 30 || e->sk.p < 4 || e->sk.p > 18)
        return fail(FA_E_INVAL, "fa_create: sketch parameters out of range");
    if (cfg->flags & FA_F_ENABLE_SKETCH) {
        if (int rc = alloc_zeroed(e, e->sk_cms, ((size_t)e->sk.depth << e->sk.log2w) * 8)) return rc;
        if (int rc = alloc_zeroed(e, e->sk_hll, ((size_t)1 << e->sk.p) * 4)) return rc;
        e->sk.cms = e->sk_cms; e->sk.hll = e->sk_hll;
    }
    if (const char* ko = getenv("FA_K1_OPT")) e->k1_opt = (uint32_t)strtoul(ko, nullptr, 0);
    if (const char* pp = getenv("FA_PHASE_PROFILE")) {
        if (pp[0] == '1') { if (int rc = alloc_zeroed(e, e->d_prof, 16 * 8)) return rc; }
    }
    CU(cudaStreamSynchronize(e->stream));
    guard.e = nullptr;
    *out = e;
    return FA_OK;
}

void fa_destroy(fa_engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    for (cudaStream_t s : {e->stream, e->copy_stream, e->evict_stream}) if (s) cudaStreamSynchronize(s);
    if (e->d_prof) {
        unsigned long long p[16];
        if (cudaMemcpy(p, e->d_prof, 128, cudaMemcpyDeviceToHost) == cudaSuccess) {
            static const char* names[8] = {"tile wait", "hash+elect+fold", "S1 barrier", "pipelined probe", "general probe",
                                           "totals", "S2 barrier", "reductions"};
            double tot = 0; for (int i = 0; i < 8; i++) tot += (double)p[i];
            fprintf(stderr, "[flowagg] K1 phase profile (warp-cycles):");
            for (int i = 0; i < 8; i++) fprintf(stderr, " %s %.1f%%;", names[i], tot > 0 ? 100.0 * p[i] / tot : 0.0);
            fprintf(stderr, " total %.3g\n", tot);
            fprintf(stderr, "[flowagg] K1 records %llu: cache hits %.1f%%, representatives %.1f%% (general-loop %.2f%%), cache installs %llu\n",
                    (unsigned long long)e->st.records_ingested, 100.0 * p[8] / (double)std::max<uint64_t>(1, e->st.records_ingested),
                    100.0 * p[9] / (double)std::max<uint64_t>(1, e->st.records_ingested),
                    100.0 * p[10] / (double)std::max<uint64_t>(1, e->st.records_ingested), p[11]);
            fprintf(stderr, "[flowagg] K1 probes: home-slot collisions %llu, resolved one slot on %llu, unsettled at first probe %llu\n", p[12], p[13], p[14]);
        }
    }
    for (cudaStream_t s : {e->copy_stream, e->evict_stream, e->own_stream ? e->stream : nullptr}) if (s) cudaStreamDestroy(s);
    for (cudaEvent_t ev : e->ev_live) if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : {e->ev_swap, e->ev_stage_free[0], e->ev_stage_free[1], e->ev_copied[0], e->ev_copied[1]}) if (ev) cudaEventDestroy(ev);
    delete e;                                         // the buffers free themselves
}

int fa_ingest(fa_engine* e, const void* recs, size_t n, size_t* consumed) {
    if (consumed) *consumed = 0;
    if (!e) return fail(FA_E_INVAL, "fa_ingest: null engine");
    if (n == 0) return FA_OK;
    if (!recs) return fail(FA_E_INVAL, "fa_ingest: null records");
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    // device records are folded in place, host records as their chunks are staged
    return ingest_caller_memory(
        e, "fa_ingest", "records", 16, recs, n, fa::kRecBytes, consumed,
        [&](size_t left, bool staged, size_t* c) {
            *c = staged ? room_window(e, std::min<uint64_t>(left, stage_records(e))) : left;
            return FA_OK;
        },
        [&](Chunk& ch, size_t c, size_t* took) { return ingest_device(e, ch.d, c, took); });
}

int fa_ingest_events(fa_engine* e, const void* events, size_t n, size_t* consumed) {
    if (consumed) *consumed = 0;
    if (!e) return fail(FA_E_INVAL, "fa_ingest_events: null engine");
    if (n == 0) return FA_OK;
    if (!events) return fail(FA_E_INVAL, "fa_ingest_events: null events");
    static_assert(sizeof(fa_packet_event) == 64, "fa_packet_event ABI");
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    CU(e->d_expanded.reserve(e->max_batch * fa::kRecBytes));
    // the expansion and K1 of successive chunks are ordered on the engine's stream, so one d_expanded is enough
    return ingest_caller_memory(
        e, "fa_ingest_events", "events", 16, events, n, 64, consumed,
        [&](size_t left, bool staged, size_t* c) {
            *c = room_window(e, std::min<uint64_t>(left, staged ? stage_records(e) : e->max_batch));
            return FA_OK;
        },
        [&](Chunk& ch, size_t c, size_t* took) {
            e->st.kernel_launches += fa::launch_expand_events(reinterpret_cast<const uint4*>(ch.d), (uint32_t)c,
                                                              reinterpret_cast<uint4*>(e->d_expanded.get()), e->stream);
            CU(cudaGetLastError());
            if (int rc = ch.release()) return rc;
            return ingest_device(e, e->d_expanded, c, took);   // a chunk may be folded in several windows ("full" cuts)
        });
}

int fa_ingest_snaps(fa_engine* e, const void* snaps, size_t n, uint32_t stride, size_t* consumed) {
    if (consumed) *consumed = 0;
    if (!e) return fail(FA_E_INVAL, "fa_ingest_snaps: null engine");
    if (stride < 40 || stride > 152 || (stride & 7)) return fail(FA_E_INVAL, "fa_ingest_snaps: stride %u must be a multiple of 8 in 40..152", stride);
    if (n == 0) return FA_OK;
    if (!snaps) return fail(FA_E_INVAL, "fa_ingest_snaps: null snapshots");
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    CU(e->d_expanded.reserve(e->max_batch * fa::kRecBytes));
    CU(e->d_snap_src.reserve(e->max_batch * sizeof(uint32_t)));
    CU(e->d_snap_cnt.reserve((fa::kSnapMaxCtas + 8) * sizeof(uint32_t)));
    if (e->filter.n_rules) CU(e->d_snap_verdict.reserve(e->max_batch));
    unsigned long long* d_total = reinterpret_cast<unsigned long long*>(e->d_snap_cnt.get() + fa::kSnapMaxCtas);
    return ingest_caller_memory(
        e, "fa_ingest_snaps", "snapshots", 8, snaps, n, stride, consumed,
        [&](size_t left, bool staged, size_t* c) {
            // host chunks are bounded by the staging buffers (stage_records() x 144 bytes), device chunks by max_batch records
            *c = std::min<uint64_t>(left, staged ? std::min<uint64_t>(e->max_batch, stage_records(e) * fa::kRecBytes / stride) : e->max_batch);
            return FA_OK;
        },
        [&](Chunk& ch, size_t c, size_t* took) {
            CU(cudaMemsetAsync(d_total + 1, 0, 24, e->stream));             // the filter's three counters of this chunk
            e->st.kernel_launches += fa::launch_parse_snaps(ch.d, (uint32_t)c, stride, &e->filter, e->d_snap_cnt, e->d_snap_verdict,
                                                            reinterpret_cast<uint4*>(e->d_expanded.get()), e->d_snap_src, d_total,
                                                            d_total + 1, e->sm_count, e->stream);
            CU(cudaGetLastError());
            if (int rc = ch.release()) return rc;
            // how many packets were submitted decides the launch sizes of the fold: one 8-byte read-back per chunk
            unsigned long long back[4] = {0, 0, 0, 0};                      // submitted + kept | filter accept / reject / no match
            CU(cudaMemcpyAsync(back, d_total, 32, cudaMemcpyDeviceToHost, e->stream));
            CU(cudaStreamSynchronize(e->stream));
            const uint32_t m = (uint32_t)back[0];
            e->st.filter_accept += back[1]; e->st.filter_reject += back[2]; e->st.filter_nomatch += back[3];
            // every submitted packet bumps exactly one of the three counters: what the filter skipped = submitted - kept
            const uint64_t filtered_out = e->filter.n_rules ? back[1] + back[2] + back[3] - (uint64_t)m : 0;
            size_t off = 0;
            const int rc = ingest_device(e, e->d_expanded, m, &off);       // a chunk may be folded in several windows ("full" cuts)
            if (rc == FA_FULL && off < m) {
                // the cut is reported in snapshots: everything before the first record that was not folded, discarded ones included
                uint32_t first_left = 0;
                CU(cudaMemcpyAsync(&first_left, e->d_snap_src.get() + off, 4, cudaMemcpyDeviceToHost, e->stream));
                CU(cudaStreamSynchronize(e->stream));
                // discarded snapshots before the cut: first_left - off
                // (with a filter the discarded / filtered split of a partially consumed chunk is not known: both count as discarded)
                e->st.snaps_ingested += first_left;
                e->st.snaps_discarded += first_left - off;
                *took = first_left;
                return rc;
            }
            if (rc != FA_OK) return rc;
            e->st.snaps_ingested += c;
            e->st.snaps_discarded += c - m - filtered_out;                  // fill_ethhdr's DISCARDs; the filter's skips are in its counters
            *took = c;
            return FA_OK;
        });
}

int fa_set_flow_filter(fa_engine* e, const fa_filter_rule* rules, size_t n_rules, const fa_filter_cidr* peers, size_t n_peers) {
    if (!e) return fail(FA_E_INVAL, "fa_set_flow_filter: null engine");
    static_assert(sizeof(fa_filter_rule) == 64 && sizeof(fa_filter_cidr) == 20, "filter ABI");
    if (n_rules > (size_t)fa::kMaxFilterEntries || n_peers > (size_t)fa::kMaxFilterEntries)
        return fail(FA_E_INVAL, "fa_set_flow_filter: at most %d rules and %d peer CIDRs (MAX_FILTER_ENTRIES)", fa::kMaxFilterEntries, fa::kMaxFilterEntries);
    if ((n_rules && !rules) || (n_peers && !peers)) return fail(FA_E_INVAL, "fa_set_flow_filter: null table");
    std::lock_guard<std::mutex> lk(e->mu);
    fa::FilterSet F{};
    auto words = [](const uint8_t ip[16], uint32_t w[4]) {
        for (int i = 0; i < 4; i++) w[i] = ((uint32_t)ip[4 * i] << 24) | ((uint32_t)ip[4 * i + 1] << 16) | ((uint32_t)ip[4 * i + 2] << 8) | ip[4 * i + 3];
    };
    for (size_t i = 0; i < n_rules; i++) {
        const fa_filter_rule& r = rules[i];
        if (r.prefix_len > 128 || r.direction > 2 || r.action > 2) return fail(FA_E_INVAL, "fa_set_flow_filter: rule %zu out of range", i);
        fa::FilterRuleDev& d = F.rules[i];
        words(r.ip, d.ipw); d.prefix = r.prefix_len; d.sample = r.sample;
        d.dps = r.dst_port_start; d.dpe = r.dst_port_end; d.dp1 = r.dst_port1; d.dp2 = r.dst_port2;
        d.sps = r.src_port_start; d.spe = r.src_port_end; d.sp1 = r.src_port1; d.sp2 = r.src_port2;
        d.ps = r.port_start; d.pe = r.port_end; d.p1 = r.port1; d.p2 = r.port2; d.tcp_flags = r.tcp_flags;
        d.proto = r.protocol; d.icmp_type = r.icmp_type; d.icmp_code = r.icmp_code; d.direction = r.direction; d.action = r.action;
        d.filter_drops = r.filter_drops; d.peer = r.do_peer_cidr_lookup;
    }
    for (size_t i = 0; i < n_peers; i++) {
        if (peers[i].prefix_len > 128) return fail(FA_E_INVAL, "fa_set_flow_filter: peer CIDR %zu out of range", i);
        words(peers[i].ip, F.peers[i].ipw); F.peers[i].prefix = peers[i].prefix_len;
    }
    F.n_rules = (uint32_t)n_rules; F.n_peers = (uint32_t)n_peers;
    e->filter = F;
    return FA_OK;
}

static int ingest_feature(fa_engine* e, int kind, const void* recs, size_t n, const char* who) {
    const uint32_t flag = kind == 0 ? FA_F_ENABLE_RTT : kind == 1 ? FA_F_ENABLE_DNS : FA_F_ENABLE_PKT_DROP;
    if (!e) return fail(FA_E_INVAL, "%s: null engine", who);
    if (!(e->cfg.flags & flag)) return fail(FA_E_INVAL, "%s: engine was created without %s", who, kind == 0 ? "FA_F_ENABLE_RTT" : kind == 1 ? "FA_F_ENABLE_DNS" : "FA_F_ENABLE_PKT_DROP");
    if (n == 0) return FA_OK;
    if (!recs) return fail(FA_E_INVAL, "%s: null records", who);
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    if (int rc = check_headroom(e, n, who, "samples")) return rc;
    const size_t rec_bytes = kind == 1 ? fa::kDnsRecBytes : fa::kAddRecBytes;      // additional and packet-drop samples: 72 B
    return ingest_caller_memory(
        e, who, "records", 8, recs, n, rec_bytes, nullptr,
        [&](size_t left, bool staged, size_t* c) {
            *c = std::min<uint64_t>(left, staged ? stage_records(e) : e->max_batch);
            return FA_OK;
        },
        [&](Chunk& ch, size_t c, size_t* took) {
            e->st.kernel_launches += fa::launch_feature_fold(kind, ch.d, (uint32_t)c, e->table.view(), ++e->epoch, e->feat_seq[kind],
                                                             e->d_slot_of, e->d_ctr, e->sm_count, e->stream);
            CU(cudaGetLastError());
            e->feat_seq[kind] += c;
            e->unsynced_records += c;
            if (kind == 0) e->st.additional_ingested += c; else if (kind == 1) e->st.dns_ingested += c; else e->st.pkt_drops_ingested += c;
            *took = c;
            return FA_OK;
        });
}

int fa_ingest_additional(fa_engine* e, const void* recs, size_t n) { return ingest_feature(e, 0, recs, n, "fa_ingest_additional"); }
int fa_ingest_dns(fa_engine* e, const void* recs, size_t n) { return ingest_feature(e, 1, recs, n, "fa_ingest_dns"); }
int fa_ingest_pkt_drops(fa_engine* e, const void* recs, size_t n) { return ingest_feature(e, 2, recs, n, "fa_ingest_pkt_drops"); }

int fa_live_flows(fa_engine* e, size_t* n) {
    if (!e || !n) return fail(FA_E_INVAL, "fa_live_flows: null argument");
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    int rc = sync_counters(e);
    if (rc) return rc;
    *n = (size_t)e->live_known;
    return FA_OK;
}

// FA_F_NONBLOCKING_EVICT: swap the tables under `mu` (fa_ingest goes on at once, into the empty one), then lookup-and-
// delete the retired table on the eviction stream.  Only the K1 launches already queued are waited for.
static int evict_swapped(fa_engine* e, const fa_evict_out* o, size_t cap, size_t* n_out) {
    std::lock_guard<std::mutex> elk(e->evict_mu);
    CU(cudaSetDevice(e->device));
    fa::Table retired{};
    uint64_t live = 0;
    {
        std::lock_guard<std::mutex> lk(e->mu);
        int rc = sync_counters(e);                     // the queued folds finish; exact live count
        if (rc) return rc;
        live = e->live_known;
        e->st.evictions++;
        if (live == 0) return FA_OK;
        if (!o->records) return fail(FA_E_INVAL, "fa_evict: null out_records");
        if (cap < live) return fail(FA_E_2BIG, "fa_evict: capacity %zu < %llu live flows", cap, (unsigned long long)live);
        retired = e->table.view();
        std::swap(e->table, e->table_spare);           // the spare is empty: the previous eviction deleted every flow in place
        CU(cudaMemsetAsync(&e->d_ctr->live, 0, sizeof(unsigned long long), e->stream));
        CU(cudaEventRecord(e->ev_swap, e->stream));
        e->live_known = 0; e->unsynced_records = 0; e->ring_head = e->ring_tail;
        e->st.flows_evicted += live;
    }
    // from here on fa_ingest runs concurrently
    uint8_t* d_out = nullptr;
    if (int rc = evict_records_dst(e, o->records, live, &d_out)) return rc;
    const bool staged = d_out != o->records;
    CU(cudaStreamWaitEvent(e->evict_stream, e->ev_swap, 0));
    CU(cudaMemsetAsync(&e->d_ctr_ev->evict_out, 0, sizeof(unsigned long long), e->evict_stream));
    const int launched = fa::launch_evict(retired, reinterpret_cast<uint4*>(d_out), nullptr, live, e->d_ctr_ev, e->sm_count, e->evict_stream);
    CU(cudaGetLastError());
    if (staged) CU(cudaMemcpyAsync(o->records, d_out, live * fa::kRecBytes, cudaMemcpyDeviceToHost, e->evict_stream));
    CU(cudaMemcpyAsync(e->h_ev_out, &e->d_ctr_ev->evict_out, 8, cudaMemcpyDeviceToHost, e->evict_stream));
    CU(cudaStreamSynchronize(e->evict_stream));
    if (*e->h_ev_out != live)
        return fail(FA_E_CUDA, "fa_evict: table scan found %llu flows, counter says %llu", *e->h_ev_out, (unsigned long long)live);
    if (staged) zero_host_outputs(evict_outputs(e, o), live);   // double buffering is only available without feature tables
    {
        std::lock_guard<std::mutex> lk(e->mu);
        e->st.kernel_launches += launched;
        if (staged) e->st.d2h_bytes += live * fa::kRecBytes;
    }
    *n_out = (size_t)live;
    return FA_OK;
}

int fa_evict_ex(fa_engine* e, const fa_evict_out* o, size_t cap, size_t* n_out) {
    if (n_out) *n_out = 0;
    if (!e || !n_out || !o) return fail(FA_E_INVAL, "fa_evict: null argument");
    if (e->double_buffered) return evict_swapped(e, o, cap, n_out);
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    int rc = sync_counters(e);
    if (rc) return rc;
    const uint64_t live = e->live_known;
    e->st.evictions++;
    if (live == 0) return FA_OK;
    if (!o->records) return fail(FA_E_INVAL, "fa_evict: null out_records");
    if (cap < live) return fail(FA_E_2BIG, "fa_evict: capacity %zu < %llu live flows", cap, (unsigned long long)live);
    const bool feats = e->table.has_features();
    uint8_t* d_out = nullptr;
    if ((rc = evict_records_dst(e, o->records, live, &d_out))) return rc;
    const EvictOuts outs = evict_outputs(e, o);
    std::array<uint8_t*, 5> d_feat{};                  // feature outputs are staged unless the caller handed device pointers
    if (feats) {
        for (const EvictOut& x : outs) { if ((rc = reserve_evict(e, *x.stage, live, x.width))) return rc; }
        if ((rc = reserve_evict(e, e->d_slot_of_out, live, 4))) return rc;
        for (size_t i = 0; i < outs.size(); i++)
            if (outs[i].dst) d_feat[i] = classify(outs[i].dst) == PTR_DEVICE ? static_cast<uint8_t*>(outs[i].dst) : outs[i].stage->get();
    }
    const fa::Table t = e->table.view();
    uint32_t* slot_of_out = feats ? e->d_slot_of_out.get() : nullptr;
    CU(cudaMemsetAsync(&e->d_ctr->evict_out, 0, sizeof(unsigned long long), e->stream));
    if (e->cfg.mode == FA_MODE_KERNEL_MAP)
        e->st.kernel_launches += fa::launch_kmap_evict(t, e->km_met, d_out, live, &e->d_ctr->evict_out, slot_of_out, e->sm_count, e->stream);
    else
        e->st.kernel_launches += fa::launch_evict(t, reinterpret_cast<uint4*>(d_out), slot_of_out, live, e->d_ctr, e->sm_count, e->stream);
    if (feats)
        e->st.kernel_launches += fa::launch_evict_features(t, slot_of_out, live, d_out, d_feat[0], d_feat[1], d_feat[2],
                                                           reinterpret_cast<unsigned long long*>(d_feat[3]), d_feat[4],
                                                           e->sm_count, e->stream);
    CU(cudaGetLastError());
    CU(cudaMemsetAsync(&e->d_ctr->live, 0, sizeof(unsigned long long), e->stream));
    if (d_out != o->records) {
        CU(cudaMemcpyAsync(o->records, d_out, live * fa::kRecBytes, cudaMemcpyDeviceToHost, e->stream));
        e->st.d2h_bytes += live * fa::kRecBytes;
    }
    for (size_t i = 0; i < outs.size(); i++) {
        if (!d_feat[i] || d_feat[i] == outs[i].dst) continue;
        CU(cudaMemcpyAsync(outs[i].dst, d_feat[i], live * outs[i].width, cudaMemcpyDeviceToHost, e->stream));
        e->st.d2h_bytes += live * outs[i].width;
    }
    CU(cudaMemcpyAsync(e->h_ctr, e->d_ctr, sizeof(fa::Counters), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    if (e->h_ctr->evict_out != live)
        return fail(FA_E_CUDA, "fa_evict: table scan found %llu flows, counter says %llu", (unsigned long long)e->h_ctr->evict_out, (unsigned long long)live);
    if (!feats) zero_host_outputs(outs, live);
    e->live_known = 0; e->unsynced_records = 0; e->ring_head = e->ring_tail;
    e->st.flows_evicted += live;
    *n_out = (size_t)live;
    return FA_OK;
}

int fa_evict(fa_engine* e, void* out_records, void* out_dns, void* out_additional, uint8_t* out_present,
             size_t cap, size_t* n_out) {
    fa_evict_out o{};
    o.records = out_records; o.dns = out_dns; o.additional = out_additional; o.present = out_present;
    return fa_evict_ex(e, &o, cap, n_out);
}

int fa_drain_active(fa_engine* e, void* out_records_dev, size_t cap, size_t* n_out) {
    if (n_out) *n_out = 0;
    if (!e || !n_out || !out_records_dev) return fail(FA_E_INVAL, "fa_drain_active: null argument");
    if (classify(out_records_dev) != PTR_DEVICE) return fail(FA_E_INVAL, "fa_drain_active: out_records must be device memory");
    if (e->table.has_features()) return fail(FA_E_INVAL, "fa_drain_active: not available with feature folds enabled");
    if (e->cfg.mode != FA_MODE_ACCOUNTER) return fail(FA_E_INVAL, "fa_drain_active: ACCOUNTER mode only");
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    CU(cudaMemsetAsync(&e->d_ctr->evict_out, 0, sizeof(unsigned long long), e->stream));
    e->st.kernel_launches += fa::launch_evict(e->table.view(), static_cast<uint4*>(out_records_dev), nullptr, cap, e->d_ctr,
                                              e->sm_count, e->stream, /*drain=*/true);
    CU(cudaGetLastError());
    int rc = sync_counters(e);
    if (rc) return rc;
    if (e->h_ctr->evict_out > cap)
        return fail(FA_E_2BIG, "fa_drain_active: %llu active flows > capacity %zu (flows beyond it were reset but not written)",
                    (unsigned long long)e->h_ctr->evict_out, cap);
    *n_out = (size_t)e->h_ctr->evict_out;
    return FA_OK;
}

int fa_drain_active_counted(fa_engine* e, void* out_records_dev, size_t cap, uint64_t* n_dev_out) {
    if (!e || !out_records_dev || !n_dev_out) return fail(FA_E_INVAL, "fa_drain_active_counted: null argument");
    if (e->table.has_features()) return fail(FA_E_INVAL, "fa_drain_active_counted: not available with feature folds enabled");
    if (e->cfg.mode != FA_MODE_ACCOUNTER) return fail(FA_E_INVAL, "fa_drain_active_counted: ACCOUNTER mode only");
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    CU(cudaMemsetAsync(&e->d_ctr->evict_out, 0, sizeof(unsigned long long), e->stream));
    e->st.kernel_launches += fa::launch_evict(e->table.view(), static_cast<uint4*>(out_records_dev), nullptr, cap, e->d_ctr,
                                              e->sm_count, e->stream, /*drain=*/true);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(n_dev_out, &e->d_ctr->evict_out, 8, cudaMemcpyDeviceToDevice, e->stream));
    return FA_OK;
}

int fa_route_peer(fa_engine* e, const void* recs, const uint64_t* n_dev, size_t max_n, uint32_t n_shards, uint32_t self_shard,
                  void* const* peer_bufs, uint64_t* const* peer_counts, size_t cap, uint64_t* overflow_dev) {
    if (!e || !recs || !peer_bufs || !peer_counts || !overflow_dev) return fail(FA_E_INVAL, "fa_route_peer: null argument");
    if (n_shards == 0 || n_shards > 16) return fail(FA_E_INVAL, "fa_route_peer: n_shards must be 1..16");
    if (max_n > 0xFFFFFFFFull) return fail(FA_E_INVAL, "fa_route_peer: max_n too large");
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    fa::PeerTargets pt{};
    for (uint32_t i = 0; i < n_shards; i++) {
        pt.buf[i] = static_cast<uint4*>(peer_bufs[i]);
        pt.count[i] = reinterpret_cast<unsigned long long*>(peer_counts[i]);
    }
    e->st.kernel_launches += fa::launch_route_peer(static_cast<const uint4*>(recs), reinterpret_cast<const unsigned long long*>(n_dev),
                                                   (uint32_t)max_n, n_shards, self_shard, pt, cap, reinterpret_cast<unsigned long long*>(overflow_dev), e->sm_count, e->stream);
    CU(cudaGetLastError());
    return FA_OK;
}

int fa_ingest_counted(fa_engine* e, const void* recs, uint64_t* n_dev, size_t max_n, int reset_count) {
    if (!e || !recs || !n_dev) return fail(FA_E_INVAL, "fa_ingest_counted: null argument");
    if (!(e->cfg.flags & FA_F_NO_FULL_CUT)) return fail(FA_E_INVAL, "fa_ingest_counted: engine needs FA_F_NO_FULL_CUT");
    if (e->cfg.mode != FA_MODE_ACCOUNTER) return fail(FA_E_INVAL, "fa_ingest_counted: ACCOUNTER mode only");
    if (max_n == 0 || max_n > e->max_batch) return fail(FA_E_INVAL, "fa_ingest_counted: max_n must be 1..max_batch");
    if (reinterpret_cast<uintptr_t>(recs) & 15) return fail(FA_E_INVAL, "fa_ingest_counted: records must be 16-byte aligned");
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    CU(cudaMemcpyAsync(&e->d_ctr->launch_n, n_dev, 8, cudaMemcpyDeviceToDevice, e->stream));
    const uint32_t saved = e->k1_opt;
    e->k1_opt |= 16u;
    int rc = launch_chunk(e, static_cast<const uint8_t*>(recs), (uint32_t)max_n);
    e->k1_opt = saved;
    if (rc) return rc;
    if (reset_count) CU(cudaMemsetAsync(n_dev, 0, 8, e->stream));
    return FA_OK;
}

int fa_ipc_export(fa_engine* e, void* dev_ptr, uint8_t handle_out[FA_IPC_HANDLE_BYTES]) {
    if (!e || !dev_ptr || !handle_out) return fail(FA_E_INVAL, "fa_ipc_export: null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == FA_IPC_HANDLE_BYTES, "IPC handle size");
    CU(cudaSetDevice(e->device));
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, dev_ptr));
    memcpy(handle_out, &h, sizeof h);
    return FA_OK;
}
int fa_ipc_open(fa_engine* e, const uint8_t handle[FA_IPC_HANDLE_BYTES], void** out) {
    if (!e || !handle || !out) return fail(FA_E_INVAL, "fa_ipc_open: null argument");
    CU(cudaSetDevice(e->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof h);
    CU(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
    return FA_OK;
}
int fa_ipc_close(fa_engine* e, void* mapped) {
    if (!e) return fail(FA_E_INVAL, "fa_ipc_close: null engine");
    CU(cudaSetDevice(e->device));
    CU(cudaIpcCloseMemHandle(mapped));
    return FA_OK;
}

// ---------------------------------------------------------------- K7: DNS query -> response correlation (dnscorr.cu)
static constexpr uint64_t kDnsMaxEntries = 1ull << 20;        // dns_flows max_entries (bpf/maps_definition.h:84); FA_DNS_MAX_ENTRIES overrides (tests)

static int dnsc_sync(fa_engine* e) {                          // device counters -> pinned mirror
    CU(cudaMemcpyAsync(e->h_dnsc_ctr, e->dnsc.ctr, fa::DNSC_N * 8, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    e->st.dns_queries_pending = e->h_dnsc_ctr[fa::DNSC_PRESENT];
    e->st.dns_map_full = e->h_dnsc_ctr[fa::DNSC_FULL];
    e->st.dns_queries_purged = e->h_dnsc_ctr[fa::DNSC_PURGED];
    return FA_OK;
}

static int dnsc_init(fa_engine* e) {
    if (e->dnsc.tab) return FA_OK;
    e->dnsc_chunk = std::min<uint64_t>(e->max_batch, 1ull << 20);
    uint64_t max_entries = kDnsMaxEntries;
    if (const char* me = getenv("FA_DNS_MAX_ENTRIES")) max_entries = std::max<uint64_t>(1, strtoull(me, nullptr, 0));
    e->dnsc_slots = pow2_at_least(64, 4 * max_entries);
    if (int rc = alloc_zeroed(e, e->dnsc_tab, e->dnsc_slots * sizeof(fa::DnsEntry))) return rc;
    if (int rc = alloc_zeroed(e, e->dnsc_ctr, fa::DNSC_N * 8)) return rc;
    CU(e->h_dnsc_ctr.reserve(fa::DNSC_N * 8));
    CU(e->d_dnsc_state.reserve(e->dnsc_chunk * 4));
    CU(e->d_dnsc_samples.reserve(e->dnsc_chunk * fa::kDnsRecBytes));
    CU(e->d_dnsc_out.reserve(e->dnsc_chunk * fa::kDnsRecBytes));
    CU(e->d_dnsc_warps.reserve((e->dnsc_chunk + 31) / 32 * 4));
    e->dnsc.mask = e->dnsc_slots - 1; e->dnsc.max_entries = max_entries;
    e->dnsc.ctr = e->dnsc_ctr;
    e->dnsc.tab = e->dnsc_tab;
    return FA_OK;
}

// move the pending queries into an empty table: the entries of answered queries are dropped
static int dnsc_rebuild(fa_engine* e) {
    if (int rc = alloc_zeroed(e, e->dnsc_spare, e->dnsc_slots * sizeof(fa::DnsEntry))) return rc;
    CU(cudaMemsetAsync(&e->dnsc.ctr[fa::DNSC_CREATED], 0, 8, e->stream));
    fa::DnsCorr to = e->dnsc;
    to.tab = e->dnsc_spare;
    e->st.kernel_launches += fa::launch_dns_rebuild(e->dnsc, to, e->sm_count, e->stream);
    CU(cudaGetLastError());
    e->dnsc_tab.swap(e->dnsc_spare);
    e->dnsc.tab = e->dnsc_tab;
    if (int rc = dnsc_sync(e)) return rc;
    e->dnsc_used = e->h_dnsc_ctr[fa::DNSC_CREATED];
    return FA_OK;
}

int fa_ingest_dns_packets(fa_engine* e, const void* pkts, size_t n) {
    const char* who = "fa_ingest_dns_packets";
    if (!e) return fail(FA_E_INVAL, "%s: null engine", who);
    if (!(e->cfg.flags & FA_F_ENABLE_DNS)) return fail(FA_E_INVAL, "%s: engine was created without FA_F_ENABLE_DNS", who);
    if (n == 0) return FA_OK;
    if (!pkts) return fail(FA_E_INVAL, "%s: null packets", who);
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    if (int rc = dnsc_init(e)) return rc;
    if (int rc = check_headroom(e, n, who, "packets")) return rc;     // every packet may add a sample for a new flow
    return ingest_caller_memory(
        e, who, "packets", 8, pkts, n, fa::kDnsRecBytes, nullptr,
        [&](size_t left, bool staged, size_t* c) {
            // a chunk never takes more than a quarter of the table: with at most max_entries = slots / 4 present keys after
            // a rebuild the table stays at most half full, so a probe sequence cannot run out
            const uint64_t cmax = std::min<uint64_t>(e->dnsc_chunk, e->dnsc_slots / 4);
            *c = std::min<uint64_t>(left, staged ? std::min<uint64_t>(cmax, stage_records(e)) : cmax);
            return e->dnsc_used + *c > e->dnsc_slots / 2 ? dnsc_rebuild(e) : FA_OK;
        },
        [&](Chunk& ch, size_t c, size_t* took) {
            e->st.kernel_launches += fa::launch_dns_correlate(ch.d, (uint32_t)c, e->dnsc, e->d_dnsc_state, e->d_dnsc_samples,
                                                              e->d_dnsc_warps, e->d_dnsc_out, e->sm_count, e->stream);
            CU(cudaGetLastError());
            if (int rc = ch.release()) return rc;
            if (int rc = dnsc_sync(e)) return rc;                     // how many samples the chunk produced (sizes the fold)
            e->dnsc_used += c;
            const uint32_t m = (uint32_t)e->h_dnsc_ctr[fa::DNSC_EMITTED];
            if (m) {
                e->st.kernel_launches += fa::launch_feature_fold(1, e->d_dnsc_out, m, e->table.view(), ++e->epoch, e->feat_seq[1],
                                                                 e->d_slot_of, e->d_ctr, e->sm_count, e->stream);
                CU(cudaGetLastError());
                e->feat_seq[1] += m;
                e->unsynced_records += m;
                e->st.dns_ingested += m;
            }
            e->st.dns_packets_ingested += c;
            *took = c;
            return FA_OK;
        });
}

int fa_purge_stale_dns(fa_engine* e, uint64_t mono_now_ns, uint64_t timeout_ns) {
    if (!e) return fail(FA_E_INVAL, "fa_purge_stale_dns: null engine");
    std::lock_guard<std::mutex> lk(e->mu);
    if (!e->dnsc.tab) return FA_OK;   // no packet stream was correlated (pre-computed-latency contract, SURVEY.md §8 a12'): nothing to purge
    CU(cudaSetDevice(e->device));
    e->st.kernel_launches += fa::launch_dns_purge(e->dnsc, mono_now_ns, timeout_ns, e->sm_count, e->stream);
    CU(cudaGetLastError());
    return dnsc_sync(e);
}

int fa_cms_query(fa_engine* e, const void* keys, size_t n, uint64_t* est) {
    if (!e || (!keys && n) || (!est && n)) return fail(FA_E_INVAL, "fa_cms_query: null argument");
    if (!(e->cfg.flags & FA_F_ENABLE_SKETCH)) return fail(FA_E_INVAL, "fa_cms_query: engine was created without FA_F_ENABLE_SKETCH");
    if (n == 0) return FA_OK;
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    DevBuf<uint8_t> d_keys;
    DevBuf<unsigned long long> d_est;
    CU(d_keys.reserve(n * 40 + 16));
    CU(d_est.reserve(n * 8));
    CU(cudaMemcpyAsync(d_keys, keys, n * 40, cudaMemcpyDefault, e->stream));
    e->st.kernel_launches += fa::launch_cms_query(e->sk, reinterpret_cast<const uint4*>(d_keys.get()), (uint32_t)n, d_est, e->stream);
    CU(cudaMemcpyAsync(est, d_est, n * 8, cudaMemcpyDefault, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return FA_OK;
}

int fa_sketch_export(fa_engine* e, uint64_t* cms_out, size_t cms_words, uint8_t* hll_out, size_t hll_regs) {
    if (!e) return fail(FA_E_INVAL, "fa_sketch_export: null engine");
    if (!(e->cfg.flags & FA_F_ENABLE_SKETCH)) return fail(FA_E_INVAL, "fa_sketch_export: engine was created without FA_F_ENABLE_SKETCH");
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    const size_t words = (size_t)e->sk.depth << e->sk.log2w, regs = (size_t)1 << e->sk.p;
    if (cms_out) {
        if (cms_words < words) return fail(FA_E_2BIG, "fa_sketch_export: cms buffer too small");
        CU(cudaMemcpyAsync(cms_out, e->sk.cms, words * 8, cudaMemcpyDeviceToHost, e->stream));
    }
    if (hll_out) {
        if (hll_regs < regs) return fail(FA_E_2BIG, "fa_sketch_export: hll buffer too small");
        DevBuf<uint8_t> d_regs;
        CU(d_regs.reserve(regs));
        e->st.kernel_launches += fa::launch_hll_pack(e->sk, d_regs, e->stream);
        CU(cudaMemcpyAsync(hll_out, d_regs, regs, cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
    }
    CU(cudaStreamSynchronize(e->stream));
    return FA_OK;
}

int fa_sketch_reset(fa_engine* e) {
    if (!e) return fail(FA_E_INVAL, "fa_sketch_reset: null engine");
    if (!(e->cfg.flags & FA_F_ENABLE_SKETCH)) return FA_OK;
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    CU(cudaMemsetAsync(e->sk.cms, 0, ((size_t)e->sk.depth << e->sk.log2w) * 8, e->stream));
    CU(cudaMemsetAsync(e->sk.hll, 0, ((size_t)1 << e->sk.p) * 4, e->stream));
    return FA_OK;
}

int fa_hll_estimate(fa_engine* e, double* estimate) {
    if (!e || !estimate) return fail(FA_E_INVAL, "fa_hll_estimate: null argument");
    const size_t m = (size_t)1 << e->sk.p;
    std::vector<uint8_t> regs(m);
    int rc = fa_sketch_export(e, nullptr, 0, regs.data(), m);
    if (rc) return rc;
    double sum = 0.0; size_t zeros = 0;
    for (size_t i = 0; i < m; i++) { sum += std::ldexp(1.0, -(int)regs[i]); if (!regs[i]) zeros++; }
    const double alpha = m >= 128 ? 0.7213 / (1.0 + 1.079 / (double)m) : (m == 64 ? 0.709 : (m == 32 ? 0.697 : 0.673));
    double est = alpha * (double)m * (double)m / sum;
    if (est <= 2.5 * (double)m && zeros) est = (double)m * std::log((double)m / (double)zeros);
    *estimate = est;
    return FA_OK;
}

int fa_get_stats(fa_engine* e, fa_stats* out) {
    if (!e || !out) return fail(FA_E_INVAL, "fa_get_stats: null argument");
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    int rc = sync_counters(e);
    if (rc) return rc;
    e->st.live_flows = e->h_ctr->live;
    e->st.spills = e->h_ctr->spills;
    e->st.order_fixups = e->h_ctr->fixups_total;
    if (e->d_km_ctr) {
        CU(cudaMemcpyAsync(e->h_km_ctr, e->d_km_ctr, sizeof(fa::KmCounters), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
        e->st.observed_intf_missed = e->h_km_ctr->intf_missed;
        e->st.hashmap_fail_create = e->h_km_ctr->fail_create;
        e->st.ringbuf_dropped = e->h_km_ctr->spill_dropped;
        e->st.ringbuf_spilled = e->km_spilled_total + std::min<uint64_t>(e->h_km_ctr->spill_cursor, e->km_spill_cap);
        e->st.spills = e->h_km_ctr->table_full;
    }
    *out = e->st;
    return FA_OK;
}

int fa_read_spilled(fa_engine* e, void* out_records, size_t cap, size_t* n_out) {
    if (n_out) *n_out = 0;
    if (!e || !n_out) return fail(FA_E_INVAL, "fa_read_spilled: null argument");
    if (e->cfg.mode != FA_MODE_KERNEL_MAP || !(e->cfg.flags & FA_F_RINGBUF_FALLBACK))
        return fail(FA_E_INVAL, "fa_read_spilled: needs mode KERNEL_MAP with FA_F_RINGBUF_FALLBACK");
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    CU(cudaMemcpyAsync(e->h_km_ctr, e->d_km_ctr, sizeof(fa::KmCounters), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    const uint64_t n = std::min<uint64_t>(e->h_km_ctr->spill_cursor, e->km_spill_cap);
    if (n == 0) return FA_OK;
    if (!out_records) return fail(FA_E_INVAL, "fa_read_spilled: null out_records");
    if (cap < n) return fail(FA_E_2BIG, "fa_read_spilled: capacity %zu < %llu spilled records", cap, (unsigned long long)n);
    CU(cudaMemcpyAsync(out_records, e->km_spill, n * fa::kRecBytes, cudaMemcpyDefault, e->stream));
    CU(cudaMemsetAsync(&e->d_km_ctr->spill_cursor, 0, sizeof(unsigned long long), e->stream));
    CU(cudaStreamSynchronize(e->stream));
    if (classify(out_records) != PTR_DEVICE) e->st.d2h_bytes += n * fa::kRecBytes;
    e->km_spilled_total += n;
    *n_out = (size_t)n;
    return FA_OK;
}

// ------------------------------------------------------------------ K8: protobuf batch encode
static_assert(sizeof(fa_iface_name) == sizeof(fa::PbIface) && offsetof(fa_iface_name, name) == offsetof(fa::PbIface, name) &&
              offsetof(fa_iface_name, udn) == offsetof(fa::PbIface, udn), "fa_iface_name layout");

int fa_pb_encode(fa_engine* e, const void* records, const void* dns, const void* additional, const void* pkt_drops,
                 const uint8_t* present, size_t n, const fa_pb_params* p, void* out_bytes, size_t out_cap, uint64_t* offsets,
                 void* keys_out, size_t* out_len) {
    if (out_len) *out_len = 0;
    if (!e || !p || !out_len) return fail(FA_E_INVAL, "fa_pb_encode: null argument");
    if (n == 0) return FA_OK;
    if (!records) return fail(FA_E_INVAL, "fa_pb_encode: null records");
    if (n > 0xFFFFFFFFull) return fail(FA_E_INVAL, "fa_pb_encode: n too large");
    if (p->n_ifaces && !p->ifaces) return fail(FA_E_INVAL, "fa_pb_encode: n_ifaces without ifaces");
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    // inputs: device pointers are used in place, host buffers are staged
    DevBuf<uint8_t> in_bufs[5], out_buf, keys_buf;
    const void* src[5] = {records, dns, additional, present, pkt_drops};
    const size_t width[5] = {fa::kRecBytes, 64, 32, 1, 32};
    const uint8_t* d_in[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    for (int i = 0; i < 5; i++) {
        if (!src[i]) continue;
        if (classify(src[i]) == PTR_DEVICE) { d_in[i] = static_cast<const uint8_t*>(src[i]); continue; }
        CU(in_bufs[i].reserve(n * width[i]));
        CU(cudaMemcpyAsync(in_bufs[i], src[i], n * width[i], cudaMemcpyHostToDevice, e->stream));
        e->st.h2d_bytes += n * width[i];
        d_in[i] = in_bufs[i];
    }
    CU(e->d_pb_sizes.reserve(n * 4));
    CU(e->d_pb_offsets.reserve((n + 1) * 8));
    CU(e->d_pb_sums.reserve(((n + 1023) / 1024 + 1) * 8));
    CU(e->d_pb_ifaces.reserve((size_t)p->n_ifaces * sizeof(fa::PbIface)));
    if (p->n_ifaces) CU(cudaMemcpyAsync(e->d_pb_ifaces, p->ifaces, (size_t)p->n_ifaces * sizeof(fa::PbIface), cudaMemcpyHostToDevice, e->stream));
    fa::PbParams P{};
    P.now_unix_ns = p->now_unix_ns; P.mono_now_ns = p->mono_now_ns;
    memcpy(P.agent_ip, p->agent_ip, 16);
    P.agent_is_v4 = p->agent_ip_is_v4 ? 1u : 0u;
    P.wrap = (p->flags & FA_PB_WRAP_ENTRIES) ? 1u : 0u;
    P.ifaces = e->d_pb_ifaces; P.n_ifaces = p->n_ifaces;
    fa::PbInputs in{d_in[0], d_in[1], d_in[2], d_in[4], d_in[3]};
    e->st.kernel_launches += fa::launch_pb_sizes(in, (uint32_t)n, P, e->d_pb_sizes, e->d_pb_offsets, e->d_pb_sums, e->sm_count, e->stream);
    CU(cudaGetLastError());
    unsigned long long total = 0;
    CU(cudaMemcpyAsync(&total, e->d_pb_offsets + n, 8, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    *out_len = (size_t)total;
    if (total > out_cap) return fail(FA_E_2BIG, "fa_pb_encode: %llu bytes needed, capacity %zu", total, out_cap);
    if (!out_bytes) return fail(FA_E_INVAL, "fa_pb_encode: null out_bytes");
    uint8_t* d_out = static_cast<uint8_t*>(out_bytes);
    const bool out_dev = classify(out_bytes) == PTR_DEVICE;
    if (!out_dev) { CU(out_buf.reserve(total ? total : 16)); d_out = out_buf; }
    uint8_t* d_keys = static_cast<uint8_t*>(keys_out);
    const bool keys_dev = keys_out && classify(keys_out) == PTR_DEVICE;
    if (keys_out && !keys_dev) { CU(keys_buf.reserve(n * 32)); d_keys = keys_buf; }
    e->st.kernel_launches += fa::launch_pb_write(in, (uint32_t)n, P, e->d_pb_offsets, e->d_pb_sizes, d_out, d_keys, e->stream);
    CU(cudaGetLastError());
    if (!out_dev) { CU(cudaMemcpyAsync(out_bytes, d_out, total, cudaMemcpyDeviceToHost, e->stream)); e->st.d2h_bytes += total; }
    if (keys_out && !keys_dev) { CU(cudaMemcpyAsync(keys_out, d_keys, n * 32, cudaMemcpyDeviceToHost, e->stream)); e->st.d2h_bytes += n * 32; }
    if (offsets) CU(cudaMemcpyAsync(offsets, e->d_pb_offsets, (n + 1) * 8, cudaMemcpyDefault, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return FA_OK;
}

int fa_sync(fa_engine* e) {
    if (!e) return fail(FA_E_INVAL, "fa_sync: null engine");
    CU(cudaSetDevice(e->device));
    CU(cudaStreamSynchronize(e->copy_stream));
    CU(cudaStreamSynchronize(e->stream));
    return FA_OK;
}

// ------------------------------------------------------------------ routing
uint64_t fa_owner_hash(const fa_flow_id* key) {
    uint64_t w[5];
    memcpy(w, key, 40);
    return fa::owner_hash(fa::key_premix(w[0], w[1], w[2], w[3], w[4]));
}

int fa_route(fa_engine* e, const void* recs, size_t n, uint32_t n_shards, void* out, uint64_t* counts_host) {
    if (!e || !counts_host || (n && (!recs || !out))) return fail(FA_E_INVAL, "fa_route: null argument");
    if (n_shards == 0 || n_shards > 16) return fail(FA_E_INVAL, "fa_route: n_shards must be 1..16");
    if (n > e->max_batch) return fail(FA_E_INVAL, "fa_route: n %zu > max_batch %llu", n, (unsigned long long)e->max_batch);
    std::lock_guard<std::mutex> lk(e->mu);
    CU(cudaSetDevice(e->device));
    CU(e->d_route_tmp.reserve((e->max_batch + 16 * ((e->max_batch + 2047) / 2048) + 16) * 4));
    CU(e->d_route_counts.reserve(16 * 8));
    e->st.kernel_launches += fa::launch_route(reinterpret_cast<const uint4*>(recs), (uint32_t)n, n_shards,
                                              reinterpret_cast<uint4*>(out), e->d_route_counts, e->d_route_tmp, e->sm_count, e->stream);
    CU(cudaGetLastError());
    unsigned long long h[16];
    CU(cudaMemcpyAsync(h, e->d_route_counts, n_shards * 8, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    for (uint32_t i = 0; i < n_shards; i++) counts_host[i] = h[i];
    return FA_OK;
}

// ------------------------------------------------------------------ memory + generator
int fa_device_alloc(fa_engine* e, size_t bytes, void** out) {
    if (!e || !out) return fail(FA_E_INVAL, "fa_device_alloc: null argument");
    CU(cudaSetDevice(e->device));
    CU(cudaMalloc(out, bytes ? bytes : 16));
    CU(cudaMemset(*out, 0, bytes ? bytes : 16));       // zero-initialised (counters, receive buffers)
    return FA_OK;
}
int fa_device_free(fa_engine* e, void* p) {
    if (!e) return fail(FA_E_INVAL, "fa_device_free: null engine");
    CU(cudaSetDevice(e->device));
    CU(cudaFree(p));
    return FA_OK;
}
int fa_host_alloc(size_t bytes, void** out) {
    if (!out) return fail(FA_E_INVAL, "fa_host_alloc: null argument");
    CU(cudaHostAlloc(out, bytes ? bytes : 16, cudaHostAllocDefault));
    return FA_OK;
}
int fa_host_free(void* p) { CU(cudaFreeHost(p)); return FA_OK; }

static int gen_params(const fa_gen_params* p, int device, fa::GenDeviceParams* g) {
    if (!p || p->n_keys == 0 || p->n_keys > (1ull << 32)) return fail(FA_E_INVAL, "fa_gen: n_keys must be 1..2^32");
    g->seed = p->seed; g->n_keys = p->n_keys; g->t0_ns = p->t0_ns; g->dist = p->dist; g->varying_desc = p->varying_desc;
    g->thresholds = nullptr; g->bucket_first = nullptr; g->bucket_size = nullptr; g->n_buckets = 0; g->reserved = 0;
    if (p->dist == FA_GEN_ZIPF) {
        ZipfTable* z = zipf_table(p->n_keys, p->zipf_s_milli ? p->zipf_s_milli : 1100);
        g->n_buckets = (uint32_t)z->thresholds.size();
        if (device < 0) {
            g->thresholds = z->thresholds.data(); g->bucket_first = z->first.data(); g->bucket_size = z->size.data();
        } else {
            std::lock_guard<std::mutex> lk(g_zipf_mu);
            if (z->device != device) {
                if (z->d_thresholds) { cudaFree(z->d_thresholds); cudaFree(z->d_first); cudaFree(z->d_size); }
                CU(cudaMalloc(&z->d_thresholds, z->thresholds.size() * 8));
                CU(cudaMalloc(&z->d_first, z->first.size() * 4));
                CU(cudaMalloc(&z->d_size, z->size.size() * 4));
                CU(cudaMemcpy(z->d_thresholds, z->thresholds.data(), z->thresholds.size() * 8, cudaMemcpyHostToDevice));
                CU(cudaMemcpy(z->d_first, z->first.data(), z->first.size() * 4, cudaMemcpyHostToDevice));
                CU(cudaMemcpy(z->d_size, z->size.data(), z->size.size() * 4, cudaMemcpyHostToDevice));
                z->device = device;
            }
            g->thresholds = z->d_thresholds; g->bucket_first = z->d_first; g->bucket_size = z->d_size;
        }
    }
    return FA_OK;
}

int fa_gen_records(fa_engine* e, const fa_gen_params* p, uint64_t first_index, size_t n, void* dst) {
    if (!dst && n) return fail(FA_E_INVAL, "fa_gen_records: null dst");
    const PtrKind k = e ? classify(dst) : PTR_PAGEABLE;
    fa::GenDeviceParams g;
    if (k == PTR_DEVICE) {
        CU(cudaSetDevice(e->device));
        int rc = gen_params(p, e->device, &g);
        if (rc) return rc;
        std::lock_guard<std::mutex> lk(e->mu);
        size_t done = 0;
        while (done < n) {
            const uint32_t c = (uint32_t)std::min<size_t>(n - done, 1u << 24);
            e->st.kernel_launches += fa::launch_generate(g, first_index + done, c, reinterpret_cast<uint4*>(static_cast<uint8_t*>(dst) + done * fa::kRecBytes), e->stream);
            done += c;
        }
        CU(cudaGetLastError());
        return FA_OK;
    }
    int rc = gen_params(p, -1, &g);
    if (rc) return rc;
    uint8_t* o = static_cast<uint8_t*>(dst);
    for (size_t i = 0; i < n; i++) {
        uint32_t w[36];
        fa::gen_record_words(g, first_index + i, w);
        memcpy(o + i * fa::kRecBytes, w, fa::kRecBytes);
    }
    return FA_OK;
}

int fa_gen_key(const fa_gen_params* p, uint64_t rank, fa_flow_id* out) {
    if (!p || !out) return fail(FA_E_INVAL, "fa_gen_key: null argument");
    uint32_t w[10];
    fa::gen_key_words(p->seed, rank, w);
    memcpy(out, w, 40);
    return FA_OK;
}

}  // extern "C"
