// C ABI of the B200 pair-HMM engine (include/phmm_b200.h): host-side orchestration only. All arithmetic of the
// hot path runs in the kernels of phmm_kernels.cuh; there is no CPU fallback — without a usable GPU every
// computing entry point returns PHMM_ERR_CUDA.
#include "../../include/phmm_b200.h"
#include "phmm_kernels.cuh"

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <condition_variable>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace phmm;

namespace {

struct DBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { e = cudaMalloc(&p, bytes); want = bytes; }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <typename T> T* as() const { return static_cast<T*>(p); }
};

int round_band(int requested)
{
    // simd_pair_hmm_wrapper.hpp:218-241: smallest supported band >= request, from {8,16,32,64,128,256}
    for (int b = 8; b <= 256; b <<= 1) if (requested <= b) return b;
    return -1;
}

} // namespace

struct phmm_engine {
    int device = 0;
    int sm_count = 148;
    int reserved_sms = 0;       // phmm_reserve_sms
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    int64_t launches_last = 0, launches_total = 0;
    double last_dp_ms = 0.0;
    int64_t last_dp_cells = 0;
    // device copies of caller arrays (host-space calls)
    DBuf h_off, h_seq, h_mf, h_pf, h_mr, h_pr, h_go, h_ge, h_begin;
    DBuf r_off, r_bases, r_quals, r_mapq, r_rev, r_begin;
    DBuf c_off, c_pos;
    // derived / scratch
    DBuf tab_f, tab_r, rowhalf, info, flags, best, status, out, slow, counters, pairs, generic_reads, wide_reads, bp, regs, rregion, rpbase, rpstride;
    DBuf tasks_lane, tasks_generic, works, scores;
    DBuf rhash, kbins, kitems, kpos, kcnt, ftasks, fcnt, gtasks, atasks, gcnt, sched, sorted, fb_scratch, fb_pairs, npre_f, npre_r;
    DBuf toff, tregion;                 // template offsets (host-space calls) and the region of every template
    std::vector<cudaEvent_t> tile_events;
    std::vector<int2> info_host;
    // per-kernel launch configuration already applied / queried (the runtime calls are not free and need not be repeated)
    std::map<std::pair<const void*, size_t>, int> occupancy;
    // host-space calls on large batches are pipelined over two sub-engines (own stream + buffers each), driven by two host
    // threads, so that the H2D / D2H copies of one read chunk overlap the kernels of the other
    phmm_engine* sub[2] = {nullptr, nullptr};
    bool is_sub = false;
    // Chunk c's DP kernels wait (on the device) for chunk c-1's, so that the DP kernels run back to back in chunk order —
    // each with the whole GPU — while the other chunk's copies, preparation and classify pass fill in around them.
    // order_ev marks "this sub-engine's DP kernels of its current chunk are done"; the parent's order state tells the other
    // worker thread that the event has been recorded (a wait enqueued before the record would see the previous one).
    phmm_engine* parent = nullptr;
    phmm_engine* peer = nullptr;
    cudaEvent_t order_ev = nullptr;
    long long chunk_index = -1;
    struct OrderState { std::mutex m; std::condition_variable cv; long long recorded = -1; } order;
};

// Sub-engine side of the chunk ordering; no-ops on a plain engine.
struct ChunkOrder {
    phmm_engine* e;
    bool waited = false, recorded = false;
    explicit ChunkOrder(phmm_engine* eng) : e(eng) {}
    cudaError_t wait_for_previous()   // before this chunk's first DP launch
    {
        if (!e->is_sub || !e->parent || waited) return cudaSuccess;
        waited = true;
        if (e->chunk_index <= 0) return cudaSuccess;
        phmm_engine::OrderState& st = e->parent->order;
        {
            std::unique_lock<std::mutex> lk(st.m);
            st.cv.wait(lk, [&] { return st.recorded >= e->chunk_index - 1; });
        }
        return cudaStreamWaitEvent(e->stream, e->peer->order_ev, 0);
    }
    void publish(bool record)         // after this chunk's last DP launch (or on any exit)
    {
        if (!e->is_sub || !e->parent || recorded) return;
        recorded = true;
        if (record) cudaEventRecord(e->order_ev, e->stream);
        phmm_engine::OrderState& st = e->parent->order;
        { std::lock_guard<std::mutex> lk(st.m); st.recorded = std::max(st.recorded, e->chunk_index); }
        st.cv.notify_all();
    }
    ~ChunkOrder() { publish(false); }
};

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            e->err = std::string(#call) + ": " + cudaGetErrorString(_e);                           \
            return _e == cudaErrorMemoryAllocation ? PHMM_ERR_NOMEM : PHMM_ERR_CUDA;               \
        }                                                                                          \
    } while (0)

#define LAUNCHED() do { ++e->launches_last; ++e->launches_total; } while (0)

namespace {

// Bring one caller array into device memory (copy for host space, alias for device space).
template <typename T>
int stage(phmm_engine* e, DBuf& buf, const T* src, size_t count, int space, const T** dev)
{
    if (src == nullptr) { *dev = nullptr; return PHMM_OK; }
    if (space == PHMM_SPACE_DEVICE) { *dev = src; return PHMM_OK; }
    CU(buf.ensure(std::max<size_t>(count, 1) * sizeof(T)));
    if (count) CU(cudaMemcpyAsync(buf.p, src, count * sizeof(T), cudaMemcpyHostToDevice, e->stream));
    *dev = buf.as<T>();
    return PHMM_OK;
}

struct Staged {
    DevHaps hp {};
    DevReads rd {};
    long long hap_bases = 0, read_bases = 0;
    std::vector<long long> hap_off_host;                  // haplotype offsets on the host (sizes, window checks); H + 1 entries
    long long read_len_min = 0, read_len_max = 0;         // all the host needs to know about the (possibly millions of) reads
};

int fetch_offsets(phmm_engine* e, const int64_t* off, int n, int space, std::vector<long long>& out)
{
    out.resize((size_t)n + 1);
    if (space == PHMM_SPACE_HOST) {
        for (int i = 0; i <= n; ++i) out[i] = off[i];
    } else {
        static_assert(sizeof(long long) == sizeof(int64_t), "");
        CU(cudaMemcpyAsync(out.data(), off, ((size_t)n + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
    }
    return PHMM_OK;
}

// Upload (or alias) the batch and run the preparation kernels: column tables, row half-words, read info.
int stage_batch(phmm_engine* e, const phmm_haplotypes* haps, const phmm_reads* reads, int space, Staged& s, bool need_info_host = true,
                bool defer_flag_check = false)
{
    if (!haps || !reads || haps->n <= 0 || reads->n <= 0 || !haps->off || !reads->off) {
        e->err = "empty or null haplotype / read block";
        return PHMM_ERR_INVALID;
    }
    if (!haps->seq || !haps->snv_mask_fwd || !haps->snv_prior_fwd || !haps->snv_mask_rev || !haps->snv_prior_rev ||
        !haps->gap_open || !haps->gap_extend || !reads->bases || !reads->quals) {
        e->err = "null per-base array";
        return PHMM_ERR_INVALID;
    }
    int rc;
    if ((rc = fetch_offsets(e, haps->off, haps->n, space, s.hap_off_host)) != PHMM_OK) return rc;
    OffsetSummary rs {};
    if (space == PHMM_SPACE_HOST) {
        const int64_t* off = reads->off;
        long long lo = 1LL << 62, hi = 0;
        for (int r = 0; r < reads->n; ++r) { const long long len = off[r + 1] - off[r]; lo = std::min(lo, len); hi = std::max(hi, len); }
        rs.first = off[0]; rs.last = off[reads->n]; rs.len_max = hi; rs.inv_len_min = kOffsetBig - lo;
    } else {
        // device-resident offsets: reduce them where they are instead of copying the array back
        CU(e->scores.ensure(sizeof(OffsetSummary)));
        CU(cudaMemsetAsync(e->scores.p, 0, sizeof(OffsetSummary), e->stream));
        k_offsets_summary<<<(unsigned)std::min<long long>(((long long)reads->n + 255) / 256, 1024), 256, 0, e->stream>>>((const long long*)reads->off, reads->n,
                                                                                                                          e->scores.as<OffsetSummary>());
        LAUNCHED();
        CU(cudaMemcpyAsync(&rs, e->scores.p, sizeof(OffsetSummary), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
    }
    s.hap_bases = s.hap_off_host[haps->n];
    s.read_bases = rs.last;
    s.read_len_min = kOffsetBig - rs.inv_len_min;
    s.read_len_max = rs.len_max;
    if (s.hap_off_host[0] != 0 || rs.first != 0 || s.hap_bases <= 0 || s.read_bases <= 0) {
        e->err = "offset arrays must start at 0 and be increasing";
        return PHMM_ERR_INVALID;
    }
    if (s.read_len_min < 1) { e->err = "empty read (offsets must be strictly increasing)"; return PHMM_ERR_INVALID; }
    if (s.read_len_max > (1LL << 30)) { e->err = "read too long"; return PHMM_ERR_INVALID; }
    DevHaps& hp = s.hp;
    DevReads& rd = s.rd;
    hp.n = haps->n; rd.n = reads->n;
    const long long* tmp_ll;
    if ((rc = stage(e, e->h_off, (const long long*)haps->off, (size_t)haps->n + 1, space, &tmp_ll))) return rc; hp.off = tmp_ll;
    if ((rc = stage(e, e->h_seq, haps->seq, s.hap_bases, space, &hp.seq))) return rc;
    if ((rc = stage(e, e->h_mf, haps->snv_mask_fwd, s.hap_bases, space, &hp.mask_f))) return rc;
    if ((rc = stage(e, e->h_pf, haps->snv_prior_fwd, s.hap_bases, space, &hp.prior_f))) return rc;
    if ((rc = stage(e, e->h_mr, haps->snv_mask_rev, s.hap_bases, space, &hp.mask_r))) return rc;
    if ((rc = stage(e, e->h_pr, haps->snv_prior_rev, s.hap_bases, space, &hp.prior_r))) return rc;
    if ((rc = stage(e, e->h_go, haps->gap_open, s.hap_bases, space, &hp.gap_open))) return rc;
    if ((rc = stage(e, e->h_ge, haps->gap_extend, s.hap_bases, space, &hp.gap_extend))) return rc;
    if ((rc = stage(e, e->h_begin, (const long long*)haps->begin, haps->n, space, &tmp_ll))) return rc; hp.begin = tmp_ll;
    if ((rc = stage(e, e->r_off, (const long long*)reads->off, (size_t)reads->n + 1, space, &tmp_ll))) return rc; rd.off = tmp_ll;
    if ((rc = stage(e, e->r_bases, reads->bases, s.read_bases, space, &rd.bases))) return rc;
    if ((rc = stage(e, e->r_quals, reads->quals, s.read_bases, space, &rd.quals))) return rc;
    if ((rc = stage(e, e->r_mapq, reads->mapq, reads->n, space, &rd.mapq))) return rc;
    if ((rc = stage(e, e->r_rev, reads->reverse, reads->n, space, &rd.reverse))) return rc;
    if ((rc = stage(e, e->r_begin, (const long long*)reads->begin, reads->n, space, &tmp_ll))) return rc; rd.begin = tmp_ll;

    CU(e->tab_f.ensure((size_t)s.hap_bases * sizeof(ColEntry)));
    CU(e->tab_r.ensure((size_t)s.hap_bases * sizeof(ColEntry)));
    CU(e->rowhalf.ensure((size_t)s.read_bases * sizeof(uint16_t)));
    CU(e->info.ensure((size_t)rd.n * sizeof(int2)));
    CU(e->flags.ensure(64));
    CU(cudaMemsetAsync(e->flags.p, 0, 64, e->stream));
    k_build_tables<<<(unsigned)((s.hap_bases + 255) / 256), 256, 0, e->stream>>>(s.hap_bases, hp.seq, hp.mask_f, hp.prior_f, hp.mask_r, hp.prior_r,
                                                                                 hp.gap_open, hp.gap_extend, e->tab_f.as<ColEntry>(),
                                                                                 e->tab_r.as<ColEntry>(), e->flags.as<int>());
    LAUNCHED();
    k_read_info<<<(unsigned)(((long long)rd.n * 32 + 255) / 256), 256, 0, e->stream>>>(rd.n, rd.off, rd.bases, rd.quals, e->rowhalf.as<uint16_t>(),
                                                                                       e->info.as<int2>());
    LAUNCHED();
    CU(cudaGetLastError());
    hp.tab_f = e->tab_f.as<ColEntry>(); hp.tab_r = e->tab_r.as<ColEntry>();
    rd.rowhalf = e->rowhalf.as<uint16_t>(); rd.info = e->info.as<int2>();
    // read info is needed on the host where the host schedules (8 bytes per read); phmm_populate schedules on the device
    if (need_info_host) {
        e->info_host.resize(rd.n);
        CU(cudaMemcpyAsync(e->info_host.data(), e->info.p, (size_t)rd.n * sizeof(int2), cudaMemcpyDeviceToHost, e->stream));
    }
    if (defer_flag_check) return PHMM_OK;   // the caller reads flags bit 0 at its own final synchronisation
    int flags_host[1] = {0};
    CU(cudaMemcpyAsync(flags_host, e->flags.p, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    if (flags_host[0] & 1) {
        e->err = "snv prior / gap penalty outside [0,127]";
        return PHMM_ERR_INVALID;
    }
    return PHMM_OK;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the (device, kernel) pair, not to an engine: several engines of one process
// (the two pipeline sub-engines, an application's own) share it, and setting it to a smaller value LOWERS the limit another engine's
// next launch relies on. So the high-water mark is kept per process and the attribute is only ever raised.
template <typename F>
int fast_smem_attr(phmm_engine* e, F kernel, size_t bytes)
{
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, size_t> high_water;
    std::lock_guard<std::mutex> lock(mu);
    size_t& have = high_water[std::make_pair(e->device, (const void*)kernel)];
    if (bytes <= have) return PHMM_OK;
    CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    have = bytes;
    return PHMM_OK;
}

template <typename F>
int blocks_per_sm_of(phmm_engine* e, F kernel, int threads, size_t smem, int* out)
{
    const auto key = std::make_pair((const void*)kernel, smem);
    const auto it = e->occupancy.find(key);
    if (it != e->occupancy.end()) { *out = it->second; return PHMM_OK; }
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(out, kernel, threads, smem));
    e->occupancy[key] = *out;
    return PHMM_OK;
}

} // namespace

extern "C" {

const char* phmm_version(void) { return "octopus_b200 phmm 0.1 (sm_100a)"; }

void phmm_default_config(phmm_config* c)
{
    if (!c) return;
    c->max_indel_error = 8;                 // HaplotypeLikelihoodModel::Config defaults, haplotype_likelihood_model.hpp:36-44
    c->use_int_scores = 0;
    c->use_mapping_quality = 1;
    c->mapping_quality_cap = 120;
    c->mapping_quality_cap_trigger = -1;
    c->use_flank_state = 1;
    c->nuc_prior = 2;
    c->disable_naive_shortcut = 0;
    c->map_positions = 1;
}

static std::string g_create_error;

int phmm_create(phmm_engine** out, int device)
{
    if (!out) return PHMM_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    cudaError_t ce = cudaGetDeviceCount(&count);
    if (ce != cudaSuccess || count == 0) {
        g_create_error = std::string("no CUDA device: ") + (ce != cudaSuccess ? cudaGetErrorString(ce) : "device count 0");
        return PHMM_ERR_CUDA;
    }
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
    if (device >= count) { g_create_error = "device ordinal out of range"; return PHMM_ERR_INVALID; }
    if (cudaSetDevice(device) != cudaSuccess) { g_create_error = "cudaSetDevice failed"; return PHMM_ERR_CUDA; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { g_create_error = "cudaGetDeviceProperties failed"; return PHMM_ERR_CUDA; }
    if (prop.major < 10) {
        g_create_error = "this library is built for sm_100a (B200) only; found compute capability " + std::to_string(prop.major) + "." + std::to_string(prop.minor);
        return PHMM_ERR_CUDA;
    }
    phmm_engine* e = new phmm_engine();
    e->device = device;
    e->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&e->ev0) != cudaSuccess || cudaEventCreate(&e->ev1) != cudaSuccess) {
        g_create_error = "stream / event creation failed";
        delete e;
        return PHMM_ERR_CUDA;
    }
    *out = e;
    return PHMM_OK;
}

void phmm_destroy(phmm_engine* e)
{
    if (!e) return;
    for (phmm_engine*& sub : e->sub) { if (sub) phmm_destroy(sub); sub = nullptr; }
    cudaSetDevice(e->device);
    DBuf* all[] = {&e->h_off, &e->h_seq, &e->h_mf, &e->h_pf, &e->h_mr, &e->h_pr, &e->h_go, &e->h_ge, &e->h_begin,
                   &e->r_off, &e->r_bases, &e->r_quals, &e->r_mapq, &e->r_rev, &e->r_begin, &e->c_off, &e->c_pos,
                   &e->tab_f, &e->tab_r, &e->rowhalf, &e->info, &e->flags, &e->best, &e->status, &e->out, &e->slow,
                   &e->counters, &e->pairs, &e->generic_reads, &e->wide_reads, &e->bp, &e->regs, &e->rregion, &e->rpbase, &e->rpstride, &e->tasks_lane, &e->tasks_generic, &e->works, &e->scores,
                   &e->rhash, &e->kbins, &e->kitems, &e->kpos, &e->kcnt, &e->ftasks, &e->fcnt, &e->gtasks, &e->atasks, &e->gcnt, &e->sched, &e->sorted, &e->fb_scratch, &e->fb_pairs, &e->npre_f, &e->npre_r,
                   &e->toff, &e->tregion};
    for (DBuf* b : all) b->release();
    for (cudaEvent_t ev : e->tile_events) cudaEventDestroy(ev);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    if (e->order_ev) cudaEventDestroy(e->order_ev);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

const char* phmm_last_error(const phmm_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

// Ordering against the caller's streams. Every call runs on the engine's own stream and is complete on return; what a caller
// cannot express that way is "the buffer this call will WRITE is still being read by work I enqueued earlier on another stream"
// (a gather of the previous result). phmm_wait_event makes the engine's stream(s) wait, on the device, for that work.
int phmm_wait_event(phmm_engine* e, void* cuda_event)
{
    if (!e || !cuda_event) return PHMM_ERR_INVALID;
    if (cudaSetDevice(e->device) != cudaSuccess) { e->err = "cudaSetDevice failed"; return PHMM_ERR_CUDA; }
    CU(cudaStreamWaitEvent(e->stream, (cudaEvent_t)cuda_event, 0));
    for (phmm_engine* sub : e->sub) if (sub) CU(cudaStreamWaitEvent(sub->stream, (cudaEvent_t)cuda_event, 0));
    return PHMM_OK;
}
void* phmm_engine_stream(phmm_engine* e) { return e ? (void*)e->stream : nullptr; }

int phmm_reserve_sms(phmm_engine* e, int n_sms)
{
    if (!e || n_sms < 0) return PHMM_ERR_INVALID;
    e->reserved_sms = std::min(n_sms, std::max(0, e->sm_count - 1));
    for (phmm_engine* sub : e->sub) if (sub) sub->reserved_sms = e->reserved_sms;
    return PHMM_OK;
}

// Page-locked host memory for callers without the CUDA headers (the C++ adapter's blocks): a PHMM_SPACE_HOST call copies from /
// to pinned buffers at full PCIe / C2C rate and overlaps with compute; pageable memory is staged by the driver.
void* phmm_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (bytes == 0) bytes = 1;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void phmm_host_free(void* p) { if (p) cudaFreeHost(p); }

int64_t phmm_launch_count(const phmm_engine* e, int total) { return e ? (total ? e->launches_total : e->launches_last) : 0; }
double phmm_last_dp_kernel_ms(const phmm_engine* e) { return e ? e->last_dp_ms : 0.0; }
int64_t phmm_last_dp_cells(const phmm_engine* e) { return e ? e->last_dp_cells : 0; }

// -------------------------------------------------------------------------------------------------------------
// phmm_align_scores
// -------------------------------------------------------------------------------------------------------------
int phmm_align_scores(phmm_engine* e, int band, int precision_bits, int nuc_prior,
                      const phmm_haplotypes* haps, const phmm_reads* reads,
                      const phmm_task* tasks, int64_t n_tasks, int32_t* scores, int space)
{
    if (!e) return PHMM_ERR_INVALID;
    e->err.clear(); e->launches_last = 0; e->last_dp_ms = 0.0; e->last_dp_cells = 0;
    if (cudaSetDevice(e->device) != cudaSuccess) { e->err = "cudaSetDevice failed"; return PHMM_ERR_CUDA; }
    if (band > 256) { e->err = "band > 256"; return PHMM_ERR_BAND; }
    if (band < 8 || (band & (band - 1))) { e->err = "band must be one of 8,16,...,256"; return PHMM_ERR_INVALID; }
    if (precision_bits != 16 && precision_bits != 32) { e->err = "precision_bits must be 16 or 32"; return PHMM_ERR_INVALID; }
    if (nuc_prior < 0 || nuc_prior > 127) { e->err = "nuc_prior outside [0,127]"; return PHMM_ERR_INVALID; }
    if (n_tasks < 0 || n_tasks > 0x7fffffff) { e->err = "task count out of range"; return PHMM_ERR_INVALID; }
    if (n_tasks == 0) return PHMM_OK;
    if (!tasks || !scores) { e->err = "null tasks / scores"; return PHMM_ERR_INVALID; }
    Staged s;
    int rc = stage_batch(e, haps, reads, space, s);
    if (rc != PHMM_OK) return rc;
    // tasks on the host for scheduling
    std::vector<phmm_task> th;
    const phmm_task* tk = tasks;
    if (space == PHMM_SPACE_DEVICE) {
        th.resize(n_tasks);
        CU(cudaMemcpyAsync(th.data(), tasks, (size_t)n_tasks * sizeof(phmm_task), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
        tk = th.data();
    }
    const int n = (int)n_tasks, H = s.hp.n, R = s.rd.n;
    std::vector<int> fast_idx, wide_idx;
    std::vector<GenericTask> gen;
    // packed s16x2 lanes where they are exact (precision 16, ACGT reads whose quality sum fits); 32-bit multi-lane kernel for the
    // rest of the ACGTN reads; thread-per-task generic kernel for foreign bytes / qualities above 127 / reads beyond shared memory
    const int NL = lanes_per_alignment(band), TPR = 32 / NL;
    int64_t cells = 0;
    int Lmax = 1, Lmax_wide = 1;
    for (int j = 0; j < n; ++j) {
        const phmm_task& t = tk[j];
        if (t.read < 0 || t.read >= R || t.hap < 0 || t.hap >= H) { e->err = "task index out of range"; return PHMM_ERR_INVALID; }
        const int L = e->info_host[t.read].x, fl = e->info_host[t.read].y;
        const long long hl = s.hap_off_host[t.hap + 1] - s.hap_off_host[t.hap];
        if (L < 1 || t.win_off < 0 || (long long)t.win_off + L + 2 * band - 1 > hl) { e->err = "task window outside the haplotype"; return PHMM_ERR_INVALID; }
        cells += 2LL * (L + band) * band;
        if (precision_bits == 16 && (fl & (kReadNonACGT | kReadBadQual | kReadUnsafe16 | kReadTooLong | kReadHasN)) == 0) { fast_idx.push_back(j); Lmax = std::max(Lmax, L); }
        else if ((fl & (kReadNonACGT | kReadBadQual)) == 0 && L <= kWideMaxReadLen) { wide_idx.push_back(j); Lmax_wide = std::max(Lmax_wide, L); }
        else gen.push_back(GenericTask {t.read, t.hap, t.win_off, t.reverse ? 1 : 0, j});
    }
    e->last_dp_cells = cells;
    CU(e->scores.ensure((size_t)n * sizeof(int)));
    int* d_scores = space == PHMM_SPACE_DEVICE ? scores : e->scores.as<int>();
    auto by_length_and_read = [&](int a, int b) {
        const int la = e->info_host[tk[a].read].x, lb = e->info_host[tk[b].read].x;
        if (la != lb) return la < lb;
        if (tk[a].read != tk[b].read) return tk[a].read < tk[b].read;
        return a < b;
    };
    struct Chunk { int read, first, n, L; };
    bool have_ev0 = false;

    if (!fast_idx.empty()) {
        // group by (length, read); chunks of 32 / NL tasks of one read; chunks of equal length are paired into one warp
        std::sort(fast_idx.begin(), fast_idx.end(), by_length_and_read);
        std::vector<LaneTask> lane(fast_idx.size());
        std::vector<Chunk> chunks;
        for (size_t i = 0; i < fast_idx.size(); ++i) {
            const phmm_task& t = tk[fast_idx[i]];
            lane[i] = LaneTask {s.hap_off_host[t.hap] + t.win_off, t.reverse ? 1 : 0, fast_idx[i]};
            if (chunks.empty() || chunks.back().read != t.read || chunks.back().n == TPR)
                chunks.push_back(Chunk {t.read, (int)i, 0, e->info_host[t.read].x});
            ++chunks.back().n;
        }
        std::vector<WarpWork> works;
        for (size_t c = 0; c < chunks.size();) {
            WarpWork w {};
            w.read0 = chunks[c].read; w.first0 = chunks[c].first; w.n0 = chunks[c].n; w.L = chunks[c].L;
            w.read1 = -1; w.first1 = chunks[c].first; w.n1 = 0;
            if (c + 1 < chunks.size() && chunks[c + 1].L == w.L) {
                w.read1 = chunks[c + 1].read; w.first1 = chunks[c + 1].first; w.n1 = chunks[c + 1].n;
                c += 2;
            } else c += 1;
            works.push_back(w);
        }
        CU(e->tasks_lane.ensure(lane.size() * sizeof(LaneTask)));
        CU(e->works.ensure(works.size() * sizeof(WarpWork)));
        CU(cudaMemcpyAsync(e->tasks_lane.p, lane.data(), lane.size() * sizeof(LaneTask), cudaMemcpyHostToDevice, e->stream));
        CU(cudaMemcpyAsync(e->works.p, works.data(), works.size() * sizeof(WarpWork), cudaMemcpyHostToDevice, e->stream));
        const int row_stride = (Lmax + 2) & ~1;
        const size_t smem = (size_t)kFastWarpsPerBlock * row_stride * sizeof(RowEntry);
        const int nw = (int)works.size();
        const unsigned grid = (unsigned)((nw + kFastWarpsPerBlock - 1) / kFastWarpsPerBlock);
        const uint32_t nucp = (uint32_t)nuc_prior | ((uint32_t)nuc_prior << 16);
        CU(cudaEventRecord(e->ev0, e->stream)); have_ev0 = true;
#define PHMM_PACKED_TASKS(B) \
        { if ((rc = fast_smem_attr(e, k_packed_tasks<B>, smem))) return rc; \
          k_packed_tasks<B><<<grid, kFastWarpsPerBlock * 32, smem, e->stream>>>(e->works.as<WarpWork>(), nw, e->tasks_lane.as<LaneTask>(), s.hp, s.rd, row_stride, nucp, d_scores, e->flags.as<int>(), 1u); }
        switch (band) {
            case 8: PHMM_PACKED_TASKS(8) break;     case 16: PHMM_PACKED_TASKS(16) break;   case 32: PHMM_PACKED_TASKS(32) break;
            case 64: PHMM_PACKED_TASKS(64) break;   case 128: PHMM_PACKED_TASKS(128) break; default: PHMM_PACKED_TASKS(256) break;
        }
#undef PHMM_PACKED_TASKS
        LAUNCHED();
        CU(cudaEventRecord(e->ev1, e->stream));
        CU(cudaGetLastError());
    }
    if (!wide_idx.empty()) {
        std::sort(wide_idx.begin(), wide_idx.end(), by_length_and_read);
        std::vector<LaneTask> lane(wide_idx.size());
        std::vector<WarpWork> works;
        for (size_t i = 0; i < wide_idx.size(); ++i) {
            const phmm_task& t = tk[wide_idx[i]];
            lane[i] = LaneTask {s.hap_off_host[t.hap] + t.win_off, t.reverse ? 1 : 0, wide_idx[i]};
            if (works.empty() || works.back().read0 != t.read || works.back().n0 == TPR) {
                WarpWork w {};
                w.read0 = t.read; w.read1 = -1; w.first0 = (int)i; w.n0 = 0; w.first1 = (int)i; w.n1 = 0; w.L = e->info_host[t.read].x;
                works.push_back(w);
            }
            ++works.back().n0;
        }
        CU(e->ftasks.ensure(lane.size() * sizeof(LaneTask)));
        CU(e->gtasks.ensure(works.size() * sizeof(WarpWork)));
        CU(cudaMemcpyAsync(e->ftasks.p, lane.data(), lane.size() * sizeof(LaneTask), cudaMemcpyHostToDevice, e->stream));
        CU(cudaMemcpyAsync(e->gtasks.p, works.data(), works.size() * sizeof(WarpWork), cudaMemcpyHostToDevice, e->stream));
        const int row_stride = (Lmax_wide + 2) & ~1;
        const int warps = (int)std::max<long long>(1, std::min<long long>(kFastWarpsPerBlock, (220LL << 10) / ((long long)row_stride * (long long)sizeof(RowEntry))));
        const size_t smem = (size_t)warps * row_stride * sizeof(RowEntry);
        const int nw = (int)works.size();
        const unsigned grid = (unsigned)((nw + warps - 1) / warps);
        if (!have_ev0) { CU(cudaEventRecord(e->ev0, e->stream)); have_ev0 = true; }
#define PHMM_WIDE_TASKS(CC, NN) \
        { if ((rc = fast_smem_attr(e, k_wide_tasks<CC, NN>, smem))) return rc; \
          k_wide_tasks<CC, NN><<<grid, warps * 32, smem, e->stream>>>(e->gtasks.as<WarpWork>(), nw, e->ftasks.as<LaneTask>(), s.hp, s.rd, row_stride, nuc_prior, d_scores, e->flags.as<int>()); }
        switch (band) {
            case 8: PHMM_WIDE_TASKS(16, 1) break;  case 16: PHMM_WIDE_TASKS(32, 1) break;  case 32: PHMM_WIDE_TASKS(32, 2) break;
            case 64: PHMM_WIDE_TASKS(32, 4) break; case 128: PHMM_WIDE_TASKS(32, 8) break; default: PHMM_WIDE_TASKS(32, 16) break;
        }
#undef PHMM_WIDE_TASKS
        LAUNCHED();
        CU(cudaEventRecord(e->ev1, e->stream));
        CU(cudaGetLastError());
    }
    if (!gen.empty()) {
        CU(e->tasks_generic.ensure(gen.size() * sizeof(GenericTask)));
        CU(cudaMemcpyAsync(e->tasks_generic.p, gen.data(), gen.size() * sizeof(GenericTask), cudaMemcpyHostToDevice, e->stream));
        const int ng = (int)gen.size();
        if (!have_ev0) CU(cudaEventRecord(e->ev0, e->stream));
        if (band <= 32) k_generic_tasks<64><<<(ng + 63) / 64, 64, 0, e->stream>>>(e->tasks_generic.as<GenericTask>(), ng, s.hp, s.rd, band, nuc_prior, d_scores);
        else k_generic_tasks<kGenericMaxDiag><<<(ng + 63) / 64, 64, 0, e->stream>>>(e->tasks_generic.as<GenericTask>(), ng, s.hp, s.rd, band, nuc_prior, d_scores);
        LAUNCHED();
        if (!have_ev0) CU(cudaEventRecord(e->ev1, e->stream));
        CU(cudaGetLastError());
    }
    if (space == PHMM_SPACE_HOST) CU(cudaMemcpyAsync(scores, d_scores, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, e->ev0, e->ev1) == cudaSuccess) e->last_dp_ms = ms;
    return PHMM_OK;
}

// -------------------------------------------------------------------------------------------------------------
// phmm_align_traceback
// -------------------------------------------------------------------------------------------------------------
int phmm_align_traceback(phmm_engine* e, int band,
                         const char* truth, const char* target, const int8_t* quals, int truth_len, int target_len,
                         const char* snv_mask, const int8_t* snv_prior, const int8_t* gap_open,
                         const int8_t* gap_extend, int gap_extend_scalar, int nuc_prior,
                         int* score, int* first_pos, char* align1, char* align2)
{
    if (!e) return PHMM_ERR_INVALID;
    e->err.clear(); e->launches_last = 0;
    if (cudaSetDevice(e->device) != cudaSuccess) { e->err = "cudaSetDevice failed"; return PHMM_ERR_CUDA; }
    if (band > 256) { e->err = "band > 256"; return PHMM_ERR_BAND; }
    if (band < 1 || !truth || !target || !quals || !gap_open || !score || !first_pos || !align1 || !align2 ||
        target_len < 1 || truth_len != target_len + 2 * band - 1) {
        e->err = "bad argument (truth_len must be target_len + 2*band - 1)";
        return PHMM_ERR_INVALID;
    }
    if (snv_mask && !snv_prior) { e->err = "snv_mask given without snv_prior"; return PHMM_ERR_INVALID; }
    const int W = truth_len, L = target_len;
    std::vector<char> host((size_t)5 * W + 2 * L);
    std::memcpy(host.data(), truth, W);
    if (snv_mask) { std::memcpy(host.data() + W, snv_mask, W); std::memcpy(host.data() + 2 * W, snv_prior, W); }
    else { std::memset(host.data() + W, 0, W); std::memset(host.data() + 2 * W, 127, W); }   // a mask byte no base equals
    std::memcpy(host.data() + 3 * W, gap_open, W);
    if (gap_extend) std::memcpy(host.data() + 4 * W, gap_extend, W); else std::memset(host.data() + 4 * W, gap_extend_scalar, W);
    std::memcpy(host.data() + 5 * W, target, L);
    std::memcpy(host.data() + 5 * W + L, quals, L);
    const size_t nal = (size_t)2 * (L + band) + 1, nbp = (size_t)(L + 1) * 2 * band;
    CU(e->tasks_generic.ensure(host.size()));
    CU(e->bp.ensure(nbp + 2 * nal + 64));
    CU(e->scores.ensure(2 * sizeof(int)));
    CU(cudaMemcpyAsync(e->tasks_generic.p, host.data(), host.size(), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemsetAsync(e->bp.p, 0, nbp + 2 * nal, e->stream));
    unsigned char* bp = e->bp.as<unsigned char>();
    k_align_one<<<1, 32, 0, e->stream>>>(band, L, e->tasks_generic.as<char>(), nuc_prior, bp, e->scores.as<int>(), (char*)bp + nbp, (char*)bp + nbp + nal);
    LAUNCHED();
    CU(cudaGetLastError());
    int out[2];
    CU(cudaMemcpyAsync(out, e->scores.p, sizeof(out), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(align1, bp + nbp, nal, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(align2, bp + nbp + nal, nal, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    *score = out[0]; *first_pos = out[1];
    return PHMM_OK;
}

// -------------------------------------------------------------------------------------------------------------
// phmm_genotype_likelihoods
// -------------------------------------------------------------------------------------------------------------
int phmm_genotype_likelihoods(phmm_engine* e, const double* lnl, int32_t H, int32_t R,
                              const int32_t* genotypes, int32_t G, int32_t ploidy, double* out, int space)
{
    if (!e) return PHMM_ERR_INVALID;
    e->err.clear(); e->launches_last = 0;
    if (cudaSetDevice(e->device) != cudaSuccess) { e->err = "cudaSetDevice failed"; return PHMM_ERR_CUDA; }
    if (!lnl || !genotypes || !out || H <= 0 || R <= 0 || G < 0 || ploidy < 0 || ploidy > 64) { e->err = "bad argument"; return PHMM_ERR_INVALID; }
    if (G == 0) return PHMM_OK;
    const double* d_lnl; const int32_t* d_gt;
    int rc;
    if ((rc = stage(e, e->out, lnl, (size_t)H * R, space, &d_lnl))) return rc;
    if ((rc = stage(e, e->pairs, genotypes, (size_t)G * std::max(ploidy, 1), space, &d_gt))) return rc;
    if (space == PHMM_SPACE_HOST) {   // haplotype indices are checked where they are cheap to read
        for (long long i = 0; i < (long long)G * ploidy; ++i) if (genotypes[i] < 0 || genotypes[i] >= H) { e->err = "haplotype index out of range"; return PHMM_ERR_INVALID; }
    }
    CU(e->scores.ensure((size_t)G * sizeof(double)));
    double* d_out = space == PHMM_SPACE_DEVICE ? out : e->scores.as<double>();
    k_genotype_likelihoods<<<G, 256, 0, e->stream>>>(d_lnl, R, d_gt, ploidy, d_out);
    LAUNCHED();
    CU(cudaGetLastError());
    if (space == PHMM_SPACE_HOST) CU(cudaMemcpyAsync(out, d_out, (size_t)G * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return PHMM_OK;
}

// -------------------------------------------------------------------------------------------------------------
// phmm_align_reads
// -------------------------------------------------------------------------------------------------------------
// Shared by phmm_align_reads (HaplotypeLikelihoodModel::align: candidate positions, in-range rule, fallback) and phmm_align_pairs
// (hmm::align: one explicit offset per pair).
static int align_impl(phmm_engine* e, const phmm_config* cfg, const phmm_haplotypes* haps, const phmm_reads* reads,
                      const phmm_pair* pairs, int64_t n_pairs, const phmm_positions* positions, const int32_t* raw_offsets,
                      const phmm_flank_state* flank,
                      int64_t* mapping_position, double* likelihood, char* cigar, int32_t cigar_stride, int32_t* status, int space)
{
    if (!e) return PHMM_ERR_INVALID;
    e->err.clear(); e->launches_last = 0; e->last_dp_ms = 0.0; e->last_dp_cells = 0;
    if (cudaSetDevice(e->device) != cudaSuccess) { e->err = "cudaSetDevice failed"; return PHMM_ERR_CUDA; }
    if (!cfg || !pairs || !mapping_position || !likelihood || !cigar || !status || cigar_stride < 8) { e->err = "null argument / cigar_stride < 8"; return PHMM_ERR_INVALID; }
    if (cfg->max_indel_error > 256) { e->err = "max_indel_error > 256"; return PHMM_ERR_BAND; }
    if (cfg->nuc_prior < 0 || cfg->nuc_prior > 127) { e->err = "nuc_prior outside [0,127]"; return PHMM_ERR_INVALID; }
    if (n_pairs < 0 || n_pairs > 0x7fffffff) { e->err = "pair count out of range"; return PHMM_ERR_INVALID; }
    if (n_pairs == 0) return PHMM_OK;
    if (!reads || !reads->reverse || (!reads->mapq && cfg->use_mapping_quality)) { e->err = "reads->mapq / reads->reverse required"; return PHMM_ERR_INVALID; }
    const int band = round_band(std::max(1, cfg->max_indel_error));
    Staged s;
    int rc = stage_batch(e, haps, reads, space, s);
    if (rc != PHMM_OK) return rc;
    const int n = (int)n_pairs;
    if (space == PHMM_SPACE_HOST) {      // indices are checked where they are cheap to read
        for (int i = 0; i < n; ++i) if (pairs[i].read < 0 || pairs[i].read >= s.rd.n || pairs[i].hap < 0 || pairs[i].hap >= s.hp.n) { e->err = "pair index out of range"; return PHMM_ERR_INVALID; }
    }
    AlignParams p {};
    p.hp = s.hp; p.rd = s.rd; p.n_pairs = n;
    p.band = band; p.nuc_prior = cfg->nuc_prior;
    p.use_flanks = (flank && flank->has_flank && cfg->use_flank_state) ? 1 : 0;
    p.lhs_flank = p.use_flanks ? (int)flank->lhs_flank : 0;
    p.rhs_flank = p.use_flanks ? (int)flank->rhs_flank : 0;
    p.use_mapq = cfg->use_mapping_quality; p.mapq_cap = cfg->mapping_quality_cap; p.mapq_trigger = cfg->mapping_quality_cap_trigger;
    const int2* d_pairs;
    if ((rc = stage(e, e->pairs, (const int2*)pairs, (size_t)n, space, &d_pairs))) return rc;
    p.pairs = d_pairs;
    if (raw_offsets) {
        const int32_t* pv;
        if ((rc = stage(e, e->c_pos, raw_offsets, (size_t)n, space, &pv))) return rc;
        p.pos = pv; p.raw_offsets = 1;
    } else if (positions && positions->off && positions->pos) {
        std::vector<long long> ends(1);
        if (space == PHMM_SPACE_HOST) ends[0] = positions->off[n];
        else { CU(cudaMemcpyAsync(ends.data(), positions->off + n, sizeof(int64_t), cudaMemcpyDeviceToHost, e->stream)); CU(cudaStreamSynchronize(e->stream)); }
        const long long* po; const int32_t* pv;
        if ((rc = stage(e, e->c_off, (const long long*)positions->off, (size_t)n + 1, space, &po))) return rc;
        if ((rc = stage(e, e->c_pos, positions->pos, (size_t)std::max<long long>(ends[0], 1), space, &pv))) return rc;
        p.pos_off = po; p.pos = pv;
    }
    int Lmax = 1;
    for (int r = 0; r < s.rd.n; ++r) Lmax = std::max(Lmax, e->info_host[r].x);
    // Register traceback for bands up to 32 (one thread per pair, its read in shared memory, one back-pointer word per cell);
    // the generic kernel for wider bands and the reads the register kernel cannot take.
    const int K = 2 * band;
    static const bool no_fast_align = std::getenv("PHMM_NO_FAST_ALIGN") != nullptr;      // measurement hook: the generic traceback kernel for everything
    p.fast_band = (band <= 32 && !no_fast_align) ? band : 0;
    const int fast_cap = (int)((200 << 10) / (kAlignFastThreads * (int)sizeof(uint16_t))) - 4;      // one block's rows in shared memory
    p.fast_max_len = std::min(Lmax, fast_cap);
    p.fast_row_stride = 2 * (((p.fast_max_len + 2) / 2) | 1);                                      // in half-words; 2 * odd (bank spread)
    const size_t fsmem = (size_t)kAlignFastThreads * p.fast_row_stride * sizeof(uint16_t);
    int fast_blocks_per_sm = 1;
    if (p.fast_band) {
        switch (band) {
            case 8:  if ((rc = fast_smem_attr(e, k_align_reads_fast<8>, fsmem)) || (rc = blocks_per_sm_of(e, k_align_reads_fast<8>, kAlignFastThreads, fsmem, &fast_blocks_per_sm))) return rc; break;
            case 16: if ((rc = fast_smem_attr(e, k_align_reads_fast<16>, fsmem)) || (rc = blocks_per_sm_of(e, k_align_reads_fast<16>, kAlignFastThreads, fsmem, &fast_blocks_per_sm))) return rc; break;
            default: if ((rc = fast_smem_attr(e, k_align_reads_fast<32>, fsmem)) || (rc = blocks_per_sm_of(e, k_align_reads_fast<32>, kAlignFastThreads, fsmem, &fast_blocks_per_sm))) return rc; break;
        }
        if (fast_blocks_per_sm < 1) p.fast_band = 0;
    }
    // threads: bounded by the pairs and by the scratch budgets (byte back-pointers of the generic kernel; words of the register kernel)
    const long long words_per_thread = (long long)(p.fast_max_len + K) * K;
    int fast_threads = p.fast_band ? std::min(e->sm_count * fast_blocks_per_sm * kAlignFastThreads, ((n + kAlignFastThreads - 1) / kAlignFastThreads) * kAlignFastThreads) : 0;
    if (p.fast_band) fast_threads = (int)std::max<long long>(kAlignFastThreads, std::min<long long>(fast_threads, ((6LL << 30) / (4 * words_per_thread)) / kAlignFastThreads * kAlignFastThreads));
    const long long bp_per_thread = (long long)(Lmax + 1) * K;
    int slow_threads = std::min(e->sm_count * 256, ((n + 63) / 64) * 64);
    slow_threads = (int)std::max<long long>(64, std::min<long long>(slow_threads, ((4LL << 30) / bp_per_thread) / 64 * 64));
    const int threads_total = std::max(fast_threads, slow_threads);
    p.str_cap = 2 * (Lmax + band) + 2;
    CU(e->bp.ensure((size_t)slow_threads * (size_t)bp_per_thread));
    if (p.fast_band) CU(e->ftasks.ensure((size_t)fast_threads * (size_t)words_per_thread * sizeof(uint32_t)));
    CU(e->slow.ensure((size_t)threads_total * 4 * p.str_cap));
    p.bp = e->bp.as<unsigned char>();
    p.bp32 = e->ftasks.as<uint32_t>();
    p.strings = e->slow.as<char>();
    // outputs
    const bool dev = space == PHMM_SPACE_DEVICE;
    CU(e->best.ensure((size_t)n * sizeof(long long)));
    CU(e->out.ensure((size_t)n * sizeof(double)));
    CU(e->status.ensure((size_t)n * sizeof(int)));
    CU(e->kpos.ensure((size_t)n * cigar_stride));
    p.mapping_position = dev ? (long long*)mapping_position : e->best.as<long long>();
    p.likelihood = dev ? likelihood : e->out.as<double>();
    p.status = dev ? status : e->status.as<int>();
    p.cigar = dev ? cigar : e->kpos.as<char>();
    p.cigar_stride = cigar_stride;
    CU(cudaEventRecord(e->ev0, e->stream));
    if (p.fast_band) {
        const unsigned fgrid = (unsigned)(fast_threads / kAlignFastThreads);
        switch (band) {
            case 8:  k_align_reads_fast<8><<<fgrid, kAlignFastThreads, fsmem, e->stream>>>(p); break;
            case 16: k_align_reads_fast<16><<<fgrid, kAlignFastThreads, fsmem, e->stream>>>(p); break;
            default: k_align_reads_fast<32><<<fgrid, kAlignFastThreads, fsmem, e->stream>>>(p); break;
        }
        LAUNCHED();
    }
    {
        const unsigned grid = (unsigned)(slow_threads / 64);
        if (band <= 32) k_align_reads<64><<<grid, 64, 0, e->stream>>>(p);
        else k_align_reads<kGenericMaxDiag><<<grid, 64, 0, e->stream>>>(p);
        LAUNCHED();
    }
    CU(cudaEventRecord(e->ev1, e->stream));
    CU(cudaGetLastError());
    if (!dev) {
        CU(cudaMemcpyAsync(mapping_position, p.mapping_position, (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaMemcpyAsync(likelihood, p.likelihood, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaMemcpyAsync(status, p.status, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaMemcpyAsync(cigar, p.cigar, (size_t)n * cigar_stride, cudaMemcpyDeviceToHost, e->stream));
    }
    CU(cudaStreamSynchronize(e->stream));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, e->ev0, e->ev1) == cudaSuccess) e->last_dp_ms = ms;
    return PHMM_OK;
}

int phmm_align_reads(phmm_engine* e, const phmm_config* cfg,
                     const phmm_haplotypes* haps, const phmm_reads* reads,
                     const phmm_pair* pairs, int64_t n_pairs,
                     const phmm_positions* positions, const phmm_flank_state* flank,
                     int64_t* mapping_position, double* likelihood, char* cigar, int32_t cigar_stride, int32_t* status, int space)
{
    return align_impl(e, cfg, haps, reads, pairs, n_pairs, positions, nullptr, flank, mapping_position, likelihood, cigar, cigar_stride, status, space);
}

int phmm_align_pairs(phmm_engine* e, const phmm_config* cfg,
                     const phmm_haplotypes* truths, const phmm_reads* targets,
                     const phmm_pair* pairs, const int32_t* target_offsets, int64_t n_pairs, const phmm_flank_state* flank,
                     int64_t* target_offset_out, double* likelihood, char* cigar, int32_t cigar_stride, int32_t* status, int space)
{
    if (!e) return PHMM_ERR_INVALID;
    if (!target_offsets) { e->err = "null target offsets"; return PHMM_ERR_INVALID; }
    return align_impl(e, cfg, truths, targets, pairs, n_pairs, nullptr, target_offsets, flank, target_offset_out, likelihood, cigar, cigar_stride, status, space);
}

// -------------------------------------------------------------------------------------------------------------
// phmm_populate
// -------------------------------------------------------------------------------------------------------------
// One synchronous pass over (all haplotypes) x (the given reads). out / status are written with a row pitch of out_pitch
// elements (0: dense [H][R]) so that a read chunk can land in its column block of the caller's [H][R_total] matrix.
// One region list for every call: phmm_populate is the one-region case. Host copies of the region arrays (a few KB).
// With templates, every region owns at least one template and the template values of the call number total_tout.
struct RegionSetup {
    std::vector<RegionInfo> regs;
    long long total_out = 0, total_tout = 0;
    int Hmax = 0, n_templates = 0;
    bool any_flank = false;
};

// template_off (CSR over the reads, n_templates + 1 entries, in `space`): one value per (haplotype, template) instead of per read. Host
// offsets have been validated by the caller; device ones are checked here, on the device.
static int populate_impl(phmm_engine* e, const phmm_config* cfg,
                         const phmm_haplotypes* haps, const phmm_reads* reads,
                         const phmm_positions* positions, const phmm_flank_state* flank,
                         double* out, int32_t* status, int space, long long out_pitch,
                         const int64_t* template_off = nullptr, int n_templates = 0, const RegionSetup* multi = nullptr)
{
    if (!e) return PHMM_ERR_INVALID;
    static const bool trace = std::getenv("PHMM_TRACE") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (trace) std::fprintf(stderr, "[phmm %p] %-18s %8.3f ms  (abs %.3f)\n", (void*)e, what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(),
                                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count());
    };
    e->err.clear(); e->launches_last = 0; e->last_dp_ms = 0.0; e->last_dp_cells = 0;
    if (cudaSetDevice(e->device) != cudaSuccess) { e->err = "cudaSetDevice failed"; return PHMM_ERR_CUDA; }
    if (!cfg || !out) { e->err = "null config / output"; return PHMM_ERR_INVALID; }
    if (cfg->max_indel_error > 256) { e->err = "max_indel_error > 256"; return PHMM_ERR_BAND; }
    const int band = round_band(std::max(1, cfg->max_indel_error));
    if (cfg->nuc_prior < 0 || cfg->nuc_prior > 127) { e->err = "nuc_prior outside [0,127]"; return PHMM_ERR_INVALID; }
    if (!reads || !reads->mapq || !reads->reverse) { e->err = "reads->mapq / reads->reverse required"; return PHMM_ERR_INVALID; }
    Staged s;
    int rc = stage_batch(e, haps, reads, space, s, false, true);
    if (rc != PHMM_OK) return rc;
    const int H_total = s.hp.n, R = s.rd.n;
    RegionSetup single;
    if (!multi) {
        const bool fl = flank && flank->has_flank && cfg->use_flank_state;
        RegionInfo g {};
        g.h0 = 0; g.nH = H_total; g.r0 = 0; g.nR = R; g.out_off = 0;
        g.use_flanks = fl ? 1 : 0; g.lhs = fl ? (int)flank->lhs_flank : 0; g.rhs = fl ? (int)flank->rhs_flank : 0;
        g.t0 = 0; g.nT = template_off ? n_templates : 0; g.tout_off = 0;
        single.regs.push_back(g); single.total_out = (long long)H_total * R; single.Hmax = H_total; single.any_flank = fl;
        single.n_templates = g.nT; single.total_tout = (long long)H_total * g.nT;
        multi = &single;
    }
    const int T = template_off ? multi->n_templates : 0;
    const int G = (int)multi->regs.size();
    // H: haplotype slots per read (the widest region); HR: result slots of the whole call
    const int H = multi->Hmax;
    const long long HR = multi->total_out;
    {   // regions to the device; per-read region / result slot
        CU(e->regs.ensure((size_t)G * sizeof(RegionInfo)));
        CU(cudaMemcpyAsync(e->regs.p, multi->regs.data(), (size_t)G * sizeof(RegionInfo), cudaMemcpyHostToDevice, e->stream));
        CU(e->rregion.ensure((size_t)R * sizeof(int)));
        CU(e->rpbase.ensure((size_t)R * sizeof(long long)));
        CU(e->rpstride.ensure((size_t)R * sizeof(int)));
        k_read_regions<<<(R + 255) / 256, 256, 0, e->stream>>>(R, G, e->regs.as<RegionInfo>(), e->rregion.as<int>(), e->rpbase.as<long long>(), e->rpstride.as<int>());
        LAUNCHED();
        s.rd.region = e->rregion.as<int>(); s.rd.pbase = e->rpbase.as<long long>(); s.rd.pstride = e->rpstride.as<int>();
    }
    // Everything from here to the final copy-out is enqueued without waiting for the device: sizes come from upper bounds
    // the host can derive from the offsets, the kernels clip them against the scheduler's device-resident totals.
    const long long len_min = s.read_len_min;
    const int Lmax_all = (int)s.read_len_max;
    const int Lmax_fast = std::min(Lmax_all, kFastMaxReadLen);
    // distinct read lengths the fast path can see: bounds the padding of the length-bucketed pair list
    const long long len_bins = std::max<long long>(1, std::min<long long>({(long long)R, (long long)Lmax_fast - std::min<long long>(len_min, Lmax_fast) + 1, (long long)kLenBins}));
    lap("staged");

    PopParams p {};
    p.hp = s.hp; p.rd = s.rd;
    p.band = band; p.nuc_prior = cfg->nuc_prior; p.one = 1;
    p.shortcut = cfg->disable_naive_shortcut ? 0 : 1;
    p.regs = e->regs.as<RegionInfo>();
    p.Hmax = H;
    p.use_flanks = multi->any_flank ? 1 : 0;
    if (p.use_flanks && band <= kFlankFbMaxBand) {
        // prefix counts of the 'N'-like table columns per haplotype and strand: the flank kernels' replay test in four loads
        CU(e->npre_f.ensure((size_t)s.hap_bases * sizeof(uint32_t)));
        CU(e->npre_r.ensure((size_t)s.hap_bases * sizeof(uint32_t)));
        k_ncol_prefix<<<(unsigned)((2LL * s.hp.n * 32 + 127) / 128), 128, 0, e->stream>>>(s.hp.n, s.hp.off, s.hp.tab_f, s.hp.tab_r, e->npre_f.as<uint32_t>(), e->npre_r.as<uint32_t>());
        LAUNCHED();
        p.hp.npre_f = e->npre_f.as<uint32_t>(); p.hp.npre_r = e->npre_r.as<uint32_t>();
    }
    // candidates a pair can have: listed / mapped positions + the original position + the shifted fallback
    // (haplotype_likelihood_model.cpp:211-259); at most (listed + 1) of them reach a DP
    int max_cand = 2, max_dp_per_pair = 1;
    if (positions && positions->off && positions->pos) {
        // Candidate lists: CSR arrays on the device; the host needs the total (to size the copy) and the longest list (to size the
        // per-read task lists: the reference accepts lists of any length) — reduced on the device, 32 bytes back.
        std::vector<long long> ends(1);
        if (space == PHMM_SPACE_HOST) ends[0] = positions->off[HR];
        else { CU(cudaMemcpyAsync(ends.data(), positions->off + HR, sizeof(int64_t), cudaMemcpyDeviceToHost, e->stream)); CU(cudaStreamSynchronize(e->stream)); }
        if (ends[0] < 0) { e->err = "candidate position offsets must be non-decreasing and start at 0"; return PHMM_ERR_INVALID; }
        const long long* po; const int32_t* pv;
        if ((rc = stage(e, e->c_off, (const long long*)positions->off, (size_t)HR + 1, space, &po))) return rc;
        if ((rc = stage(e, e->c_pos, positions->pos, (size_t)std::max<long long>(ends[0], 1), space, &pv))) return rc;
        p.pos_off = po; p.pos = pv;
        OffsetSummary ps {};
        CU(e->scores.ensure(sizeof(OffsetSummary)));
        CU(cudaMemsetAsync(e->scores.p, 0, sizeof(OffsetSummary), e->stream));
        k_offsets_summary<<<(unsigned)std::min<long long>((HR + 255) / 256, 2048), 256, 0, e->stream>>>(po, HR > 0x7fffffffLL ? 0x7fffffff : (int)HR, e->scores.as<OffsetSummary>());
        LAUNCHED();
        CU(cudaMemcpyAsync(&ps, e->scores.p, sizeof(OffsetSummary), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
        if (ps.first != 0 || kOffsetBig - ps.inv_len_min < 0 || ps.last != ends[0]) { e->err = "candidate position offsets must be non-decreasing and start at 0"; return PHMM_ERR_INVALID; }
        if (ps.len_max > 4096) { e->err = "more than 4096 candidate positions for one (haplotype, read) pair"; return PHMM_ERR_INVALID; }
        max_cand = (int)ps.len_max + 2;
        max_dp_per_pair = (int)ps.len_max + 1;
    } else if (cfg->map_positions) {
        max_cand = kMaxMapped + 2;   // the mapper emits <= 10 (haplotype_likelihood_array.hpp:103-104)
        max_dp_per_pair = kMaxMapped + 1;
    }
    const bool use_mapper = !(positions && positions->off && positions->pos) && cfg->map_positions;
    p.single_candidate = max_dp_per_pair == 1 ? 1 : 0;
    p.reserved_sms = e->reserved_sms;
    int mapper_maxt = 0;
    if (use_mapper) {
        long long max_hap = 0;
        for (int h = 0; h < H_total; ++h) max_hap = std::max(max_hap, s.hap_off_host[h + 1] - s.hap_off_host[h]);
        mapper_maxt = max_hap - 5 <= 512 ? 512 : 2048;       // vote-array capacity per thread (longer haplotypes: tiles of 2048 diagonals)
        if (max_hap > 65535) { e->err = "haplotype longer than 65535 bp: the device k-mer mapper indexes k-mer positions with 16 bits (pass explicit positions)"; return PHMM_ERR_INVALID; }
        if (s.hap_bases > 65535LL * 65535LL) { e->err = "haplotype block too large"; return PHMM_ERR_INVALID; }
        CU(e->rhash.ensure((size_t)s.read_bases * sizeof(uint16_t)));
        CU(e->kbins.ensure((size_t)H_total * (kKmerBins + 1) * sizeof(int)));
        CU(e->kitems.ensure((size_t)s.hap_bases * sizeof(uint16_t)));
        k_read_kmers<<<(unsigned)(((long long)R * 32 + 255) / 256), 256, 0, e->stream>>>(s.read_bases, R, s.rd.off, s.rd.bases, e->rhash.as<uint16_t>());
        LAUNCHED();
        k_build_kmer_table<<<H_total, 256, 0, e->stream>>>(H_total, s.hp.off, s.hp.seq, e->kbins.as<uint32_t>(), e->kitems.as<uint16_t>());
        LAUNCHED();
        CU(cudaGetLastError());
    }

    // scheduling: equal-length read pairs for the packed kernels, 32-bit multi-lane kernels for what they cannot take, and the
    // thread-per-pair generic kernel for the rest (foreign alphabet, qualities above 127, reads beyond the shared-memory budget)
    long long max_hap_len = 0;
    for (int h = 0; h < H_total; ++h) max_hap_len = std::max(max_hap_len, s.hap_off_host[h + 1] - s.hap_off_host[h]);
    // the DP task word packs (haplotype, window offset) into 16 + 16 bits
    const bool task_word_ok = H_total <= 65535 && max_hap_len <= 65535;
    const int NL = lanes_per_alignment(band);
    // wide (32-bit) path: row entries of one read per warp in shared memory; long reads get fewer warps per block
    const int wide_row_stride = (int)((std::min<long long>(Lmax_all, kWideMaxReadLen) + 2) & ~1LL);
    const int wide_warps = (int)std::max<long long>(0, std::min<long long>(kFastWarpsPerBlock, (220LL << 10) / ((long long)wide_row_stride * (long long)sizeof(RowEntry))));
    SchedMode mode {};
    mode.packed_ok = task_word_ok ? 1 : 0;
    mode.wide_ok = (task_word_ok && wide_warps >= 1) ? 1 : 0;
    mode.force_wide = cfg->use_int_scores ? 1 : 0;
    mode.n_to_wide = band > 32 ? 1 : 0;
    mode.wide_max_len = kWideMaxReadLen;
    const bool fast_ok = mode.packed_ok && !mode.force_wide;
    // lane groups per warp of the packed kernel: with few haplotypes a read has few DP tasks, so several read pairs share a warp
    const int groups = std::max(1, std::min(32 / NL, H >= 17 ? 1 : (H >= 9 ? 2 : 4)));
    // device-side scheduling: length buckets → equal-length read pairs (padded to multiples of `groups` per bucket) + wide + generic lists
    const size_t pairs_cap = (size_t)R / 2 + (size_t)kLenBins * groups + 8;
    SchedTotals tot {};
    {
        CU(e->sched.ensure((size_t)(4 * (kLenBins + 1) + 16) * sizeof(int) + sizeof(SchedTotals) + 16));
        CU(e->sorted.ensure((size_t)R * sizeof(int)));
        CU(e->pairs.ensure(2 * pairs_cap * sizeof(int)));
        CU(e->generic_reads.ensure((size_t)R * sizeof(int)));
        CU(e->wide_reads.ensure((size_t)R * sizeof(int)));
        int* base = e->sched.as<int>();
        int* hist = base, *read_start = base + (kLenBins + 1), *pair_start = base + 2 * (kLenBins + 1), *cursors = base + 3 * (kLenBins + 1);
        int* misc = base + 4 * (kLenBins + 1);          // [0] n_generic, [1] lmax_all, [2] bad, [3] packed reads with 'N', [4] n_wide
        SchedTotals* d_tot = (SchedTotals*)(misc + 16);
        unsigned long long* d_cells = (unsigned long long*)((char*)d_tot + ((sizeof(SchedTotals) + 7) & ~size_t(7)));
        CU(cudaMemsetAsync(base, 0, (size_t)(4 * (kLenBins + 1) + 16) * sizeof(int) + sizeof(SchedTotals) + 16, e->stream));
        k_sched_hist<<<(R + 255) / 256, 256, 0, e->stream>>>(R, s.rd.info, mode, hist, e->generic_reads.as<int>(), e->wide_reads.as<int>(), misc,
                                                              s.rd.region, e->regs.as<RegionInfo>(), band, d_cells);
        LAUNCHED();
        k_sched_scan<<<1, kLenBins, 0, e->stream>>>(hist, groups, read_start, pair_start, cursors, misc, d_cells, d_tot);
        LAUNCHED();
        k_sched_scatter<<<(R + 255) / 256, 256, 0, e->stream>>>(R, s.rd.info, mode, read_start, cursors, e->sorted.as<int>());
        LAUNCHED();
        k_sched_pairs<<<(unsigned)((pairs_cap + 255) / 256), 256, 0, e->stream>>>(d_tot, read_start, pair_start, e->sorted.as<int>(), e->pairs.as<int>());
        LAUNCHED();
        CU(cudaGetLastError());
        p.tot = d_tot;
    }
    const SchedTotals* d_tot = p.tot;
    // upper bounds of the work lists (exact counts stay on the device)
    // (a bucket of c reads holds ceil(c / 2) pairs rounded up to a multiple of `groups`)
    long long n_pairs = fast_ok ? std::min<long long>((long long)pairs_cap, R / 2 + len_bins * groups + 1) : 0;
    // reads the packed path cannot take exist only if the host can see a reason (int scores, a long read) or the device finds one
    // (quality sums, foreign bytes): the wide and generic tiles are always enqueued, their kernels clip against the device totals
    long long n_wide = mode.wide_ok ? R : 0, n_generic = R;
    lap("sched enqueued");

    CU(e->best.ensure((size_t)HR * sizeof(int)));
    CU(e->status.ensure((size_t)HR * sizeof(int)));
    CU(e->counters.ensure(256));
    CU(cudaMemsetAsync(e->counters.p, 0, 256, e->stream));
    CU(cudaMemsetAsync(e->status.p, 0, (size_t)HR * sizeof(int), e->stream));
    k_fill_int<<<(unsigned)((HR + 255) / 256), 256, 0, e->stream>>>(e->best.as<int>(), HR, kBestInf);
    LAUNCHED();
    p.best = e->best.as<int>();
    p.status = e->status.as<int>();
    p.flags = e->flags.as<int>();
    int* counters = e->counters.as<int>();
    p.pair_cursor = counters + 0;
    p.flank_cursor = counters + 1;
    p.any_flank_tasks = counters + 2;
    p.slow_count = counters + 3;
    p.acc_cursor = counters + 4;
    p.any_acc_tasks = counters + 5;
    p.fb_cursor = counters + 6;
    p.fb_rounds = counters + 7;

    // Tile size: the per-tile scratch (mapped candidate lists, DP task lists, traceback queue) must fit fixed budgets.
    const long long slow_budget = 8LL << 20;   // traceback-queue entries (16 bytes each)
    // DP tasks a pair can queue: listed / mapped positions (any number when the caller lists them) + the original position
    p.fcap = (int)std::min<long long>(0x7fffffff, (long long)H * max_dp_per_pair);   // a read's task list: one DP task per (haplotype, candidate position)
    long long reads_per_tile = std::max<long long>(R, 2 * n_pairs);   // one tile unless a budget says otherwise
    if (use_mapper) reads_per_tile = std::max<long long>(2, std::min<long long>(reads_per_tile, (1LL << 30) / (41LL * H)));   // (10 x int32 + 1 byte) per pair
    reads_per_tile = std::max<long long>(2, std::min<long long>(reads_per_tile, (160LL << 20) / p.fcap));   // two lists of 4-byte entries: <= 1.25 GiB
    if (p.use_flanks) reads_per_tile = std::max<long long>(2, std::min<long long>(reads_per_tile, slow_budget / ((long long)H * max_cand)));
    const long long pairs_per_tile = std::max<long long>((long long)groups, ((reads_per_tile + 1) / 2 + groups - 1) / (long long)groups * (long long)groups);
    // With several tiles per list the exact list sizes are worth one early synchronisation: empty wide / generic tiles cost a
    // handful of launches each.
    if (reads_per_tile < R) {
        CU(cudaMemcpyAsync(&tot, d_tot, sizeof(SchedTotals), cudaMemcpyDeviceToHost, e->stream));
        CU(cudaStreamSynchronize(e->stream));
        n_pairs = std::min<long long>(n_pairs, tot.n_pairs);
        n_wide = std::min<long long>(n_wide, tot.n_wide);
        n_generic = std::min<long long>(n_generic, tot.n_generic);
    }
    // work-list entries one tile can hold (pair tiles: two per pair, padding entries included)
    const size_t tile_list_cap = (size_t)std::max<long long>(std::min<long long>(2 * pairs_per_tile, 2 * std::max<long long>(n_pairs, groups)), std::min<long long>(reads_per_tile, R)) + 2;
    if (use_mapper) {
        CU(e->kpos.ensure(tile_list_cap * H * kMaxMapped * sizeof(int32_t)));
        CU(e->kcnt.ensure(tile_list_cap * H));
    }
    {
        CU(e->ftasks.ensure(tile_list_cap * p.fcap * sizeof(uint32_t)));
        CU(e->fcnt.ensure(4 * tile_list_cap * sizeof(int)));
        p.ftasks = e->ftasks.as<uint32_t>();
        p.fcnt = e->fcnt.as<int>();
        // the 32-bit flank kernel's lists (near-flank candidates, reads holding 'N'): whether any exist is only known on the device
        CU(e->gtasks.ensure(tile_list_cap * p.fcap * sizeof(uint32_t)));
        p.gtasks = e->gtasks.as<uint32_t>();
        p.gcnt = p.fcnt + tile_list_cap;
        p.acnt = p.fcnt + 2 * tile_list_cap;
        p.fb_round_base = p.fcnt + 3 * tile_list_cap;
        if (p.use_flanks && band <= 32) {            // the lean flank kernel's lists
            CU(e->atasks.ensure(tile_list_cap * p.fcap * sizeof(uint32_t)));
            p.atasks = e->atasks.as<uint32_t>();
        }
    }
    // traceback scratch: 1 byte per band cell per resident thread; very long reads get fewer threads instead of more memory
    const long long bp_per_thread = (long long)(Lmax_all + 1) * (2 * band);
    const int slow_blocks = (int)std::max<long long>(1, std::min<long long>(e->sm_count, (4LL << 30) / (bp_per_thread * 256)));
    const int slow_threads = slow_blocks * 256;
    if (p.use_flanks) {
        p.slow_cap = (int)std::min<long long>(slow_budget, (long long)H * max_cand * (long long)tile_list_cap);
        CU(e->slow.ensure((size_t)p.slow_cap * sizeof(int4)));
        p.slow = e->slow.as<int4>();
        CU(e->bp.ensure((size_t)slow_threads * (size_t)(Lmax_all + 1) * (size_t)(2 * band)));
    } else {
        p.slow_cap = 0;
        CU(e->slow.ensure(sizeof(int4)));
        p.slow = e->slow.as<int4>();
    }

    lap("buffers");
    const int fast_row_stride = (Lmax_fast + 2) & ~1;
    const size_t smem = (size_t)kFastWarpsPerBlock * groups * fast_row_stride * sizeof(RowEntry);
    int blocks_per_sm = 1;
    if (n_pairs) {
#define PHMM_FAST_SETUP(B, GG) \
        { if ((rc = fast_smem_attr(e, k_populate_fast<B, GG>, smem))) return rc; \
          if ((rc = blocks_per_sm_of(e, k_populate_fast<B, GG>, kFastWarpsPerBlock * 32, smem, &blocks_per_sm))) return rc; }
#define PHMM_FAST_DISPATCH(MACRO) \
        switch (band * 10 + (int)groups) { \
            case 81: MACRO(8, 1) break;   case 82: MACRO(8, 2) break;   case 84: MACRO(8, 4) break; \
            case 161: MACRO(16, 1) break; case 162: MACRO(16, 2) break; case 164: MACRO(16, 4) break; \
            case 321: MACRO(32, 1) break; case 322: MACRO(32, 2) break; case 324: MACRO(32, 4) break; \
            case 641: MACRO(64, 1) break; case 642: MACRO(64, 2) break; case 644: MACRO(64, 4) break; \
            case 1281: MACRO(128, 1) break; case 1282: MACRO(128, 2) break; case 1284: MACRO(128, 4) break; \
            case 2561: MACRO(256, 1) break; default: MACRO(256, 2) break; }
        PHMM_FAST_DISPATCH(PHMM_FAST_SETUP)
        if (blocks_per_sm < 1) { e->err = "fast kernel does not fit on an SM (read too long?)"; return PHMM_ERR_INVALID; }
    }
    // bands 32 / 64 with enough tasks per read to fill a warp: one WARP per chunk of the band (k_populate_roles) instead of one lane
    static const bool no_role_warps = std::getenv("PHMM_NO_ROLE_WARPS") != nullptr;       // measurement hook: the lane-per-chunk kernel for every band
    bool role_warps = n_pairs && (band == 32 || band == 64) && groups == 1 && !no_role_warps;
    const int role_groups = kFastWarpsPerBlock / std::max(1, NL);
    const size_t role_smem = role_warps ? (size_t)role_groups * fast_row_stride * sizeof(RowEntry) + (size_t)role_groups * kRoleWordsPerGroup(NL) * sizeof(uint32_t) : 0;
    int role_blocks_per_sm = 0;
    if (role_warps) {
        if (band == 32) { if ((rc = fast_smem_attr(e, k_populate_roles<32>, role_smem)) || (rc = blocks_per_sm_of(e, k_populate_roles<32>, kFastWarpsPerBlock * 32, role_smem, &role_blocks_per_sm))) return rc; }
        else            { if ((rc = fast_smem_attr(e, k_populate_roles<64>, role_smem)) || (rc = blocks_per_sm_of(e, k_populate_roles<64>, kFastWarpsPerBlock * 32, role_smem, &role_blocks_per_sm))) return rc; }
        if (role_blocks_per_sm < 1) role_warps = false;
    }
    // wide kernel: chunk / lanes by band
    const size_t wsmem = (size_t)std::max(1, wide_warps) * wide_row_stride * sizeof(RowEntry);
    int wide_blocks_per_sm = 1;
#define PHMM_WIDE_DISPATCH(MACRO) \
    switch (band) { case 8: MACRO(16, 1) break; case 16: MACRO(32, 1) break; case 32: MACRO(32, 2) break; case 64: MACRO(32, 4) break; \
                    case 128: MACRO(32, 8) break; default: MACRO(32, 16) break; }
#define PHMM_WIDE_SETUP(CC, NN) \
    { if ((rc = fast_smem_attr(e, k_populate_wide<CC, NN>, wsmem))) return rc; \
      if ((rc = blocks_per_sm_of(e, k_populate_wide<CC, NN>, wide_warps * 32, wsmem, &wide_blocks_per_sm))) return rc; }
    if (n_wide) {
        PHMM_WIDE_DISPATCH(PHMM_WIDE_SETUP)
        if (wide_blocks_per_sm < 1) { e->err = "wide kernel does not fit on an SM"; return PHMM_ERR_INVALID; }
    }

    lap("kernel attrs");
    // k-mer mapper variant: vote-array capacity by the longest haplotype, byte counters when no read can cast > 255 votes
    const bool mapper_bytes = Lmax_all - kKmer + 1 <= 255;
    auto launch_mapper = [&](const int* list, int n_list, int base, int kind) {
        const long long threads = (long long)n_list * H;
        const unsigned grid = (unsigned)std::max<long long>(1, std::min<long long>((threads + 127) / 128, (long long)e->sm_count * 64));
#define PHMM_MAP_ARGS list, n_list, d_tot, base, kind, s.hp, s.rd, e->rhash.as<uint16_t>(), e->kbins.as<uint32_t>(), e->kitems.as<uint16_t>(), e->kpos.as<int32_t>(), e->kcnt.as<uint8_t>(), e->regs.as<RegionInfo>(), H
        if (mapper_maxt == 512) {
            if (mapper_bytes) k_kmer_map<512, uint8_t><<<grid, 128, 0, e->stream>>>(PHMM_MAP_ARGS);
            else k_kmer_map<512, uint16_t><<<grid, 128, 0, e->stream>>>(PHMM_MAP_ARGS);
        } else {
            if (mapper_bytes) k_kmer_map<2048, uint8_t><<<grid, 128, 0, e->stream>>>(PHMM_MAP_ARGS);
            else k_kmer_map<2048, uint16_t><<<grid, 128, 0, e->stream>>>(PHMM_MAP_ARGS);
        }
#undef PHMM_MAP_ARGS
    };
    // the 32-bit flank kernel over the current list (near-flank candidates, and every candidate of pair-list reads holding 'N')
    static const bool no_flank_fb = std::getenv("PHMM_NO_FLANK_FB") != nullptr;           // measurement hook: the labelled one-alignment-per-thread flank kernels only
    const bool flank_fb_ok = !no_flank_fb && band <= kFlankFbMaxBand;
    auto launch_flank = [&](int n_entries, int row_stride) -> int {
        if (band > 32) return PHMM_OK;              // wide bands: near-flank candidates take the traceback queue
        if (p.atasks && p.fb_route) {
            // the packed forward / backward flank kernels over the atasks lists; they run BEFORE k_populate_flank, which also resolves the
            // candidates they report as tied or could not place in the forward scratch (appended to the gtasks lists)
            // lane groups: a read's candidates (about one per haplotype) should fill its group's 2 * LG half-lanes; rows must fit 4 blocks / SM
            const int fb_stride = (row_stride + 2 * band + 1) & ~1;                  // + the backward pass's pad rows
            int lg = 5;
            while (lg > 2 && (1 << lg) >= H && (size_t)kFastWarpsPerBlock * (32 >> (lg - 1)) * fb_stride * sizeof(RowEntry) <= (48u << 10)) --lg;
            const int fbG = 32 >> lg;
            const size_t fbsmem = (size_t)kFastWarpsPerBlock * fbG * fb_stride * sizeof(RowEntry);
            // forward scratch: one warp-round (64 candidates) per fb_round_words; worst case = every claim's longest task list, capped at 4 GiB
            const long long rounds_worst = ((long long)n_entries / fbG + 1) * ((p.fcap + (2 << lg) - 1) >> (lg + 1));
            int fb_blocks = 1, frc2;
#define PHMM_FB_LAUNCH(B) \
            { if ((frc2 = fast_smem_attr(e, k_flank_fwd<B>, fbsmem)) || (frc2 = fast_smem_attr(e, k_flank_bwd<B>, fbsmem)) || \
                  (frc2 = blocks_per_sm_of(e, k_flank_bwd<B>, kFastWarpsPerBlock * 32, fbsmem, &fb_blocks))) return frc2; \
              if (fb_blocks < 1) { e->err = "flank kernel does not fit on an SM (read too long?)"; return PHMM_ERR_INVALID; } \
              const unsigned bgrid = (unsigned)std::max(1, std::min((n_entries / fbG + kFastWarpsPerBlock) / kFastWarpsPerBlock, e->sm_count * fb_blocks)); \
              const size_t round_bytes = fb_round_words(B) * sizeof(uint32_t); \
              const long long cap = std::max<long long>(1, std::min<long long>(rounds_worst, (long long)((4ull << 30) / round_bytes))); \
              cudaError_t ce = e->fb_pairs.ensure((size_t)cap * round_bytes); \
              if (ce == cudaSuccess) ce = e->fb_scratch.ensure((size_t)bgrid * kFastWarpsPerBlock * 32 * fb_scratch_words(B) * sizeof(uint32_t)); \
              if (ce != cudaSuccess) { e->err = cudaGetErrorString(ce); return PHMM_ERR_NOMEM; } \
              p.fb_round_cap = (int)std::min<long long>(0x7fffffff, (long long)(e->fb_pairs.cap / round_bytes)); \
              k_flank_fwd<B><<<bgrid, kFastWarpsPerBlock * 32, fbsmem, e->stream>>>(p, e->fb_pairs.as<uint32_t>(), fb_stride, lg); \
              LAUNCHED(); \
              k_flank_bwd<B><<<bgrid, kFastWarpsPerBlock * 32, fbsmem, e->stream>>>(p, e->fb_pairs.as<uint32_t>(), e->fb_scratch.as<uint32_t>(), fb_stride, lg); }
            if (band == 8) PHMM_FB_LAUNCH(8) else PHMM_FB_LAUNCH(16)
#undef PHMM_FB_LAUNCH
            LAUNCHED();
        }
        // the labelled kernel: whole warps per read when its lists are dense, groups of 4 lanes when they only hold what the packed kernels
        // passed on (ties: one or two candidates per read; the rare reads with 'N' or shorter than 2 * band then take more rounds)
        int flg = 5;
        if (p.atasks && p.fb_route) { flg = 2; while (flg < 5 && (size_t)kFastWarpsPerBlock * (32 >> flg) * row_stride * sizeof(RowEntry) > (48u << 10)) ++flg; }
        const int fG = 32 >> flg;
        const unsigned fgrid = (unsigned)std::max(1, std::min((n_entries / fG + kFastWarpsPerBlock) / kFastWarpsPerBlock, e->sm_count * 3));
        const size_t fsmem = (size_t)kFastWarpsPerBlock * fG * row_stride * sizeof(RowEntry);
        int frc;
        switch (band) {
            case 8:  if ((frc = fast_smem_attr(e, k_populate_flank<8>, fsmem))) return frc;
                     k_populate_flank<8><<<fgrid, kFastWarpsPerBlock * 32, fsmem, e->stream>>>(p, row_stride, flg); break;
            case 16: if ((frc = fast_smem_attr(e, k_populate_flank<16>, fsmem))) return frc;
                     k_populate_flank<16><<<fgrid, kFastWarpsPerBlock * 32, fsmem, e->stream>>>(p, row_stride, flg); break;
            default: if ((frc = fast_smem_attr(e, k_populate_flank<32>, fsmem))) return frc;
                     k_populate_flank<32><<<fgrid, kFastWarpsPerBlock * 32, fsmem, e->stream>>>(p, row_stride, flg); break;
        }
        LAUNCHED();
        if (p.atasks && !p.fb_route) {
            const unsigned agrid = (unsigned)std::max(1, std::min((n_entries + kFastWarpsPerBlock - 1) / kFastWarpsPerBlock, e->sm_count * 4));
            switch (band) {
                case 8:  if ((frc = fast_smem_attr(e, k_populate_flank_acc<8>, fsmem))) return frc;
                         k_populate_flank_acc<8><<<agrid, kFastWarpsPerBlock * 32, fsmem, e->stream>>>(p); break;
                case 16: if ((frc = fast_smem_attr(e, k_populate_flank_acc<16>, fsmem))) return frc;
                         k_populate_flank_acc<16><<<agrid, kFastWarpsPerBlock * 32, fsmem, e->stream>>>(p); break;
                default: if ((frc = fast_smem_attr(e, k_populate_flank_acc<32>, fsmem))) return frc;
                         k_populate_flank_acc<32><<<agrid, kFastWarpsPerBlock * 32, fsmem, e->stream>>>(p); break;
            }
            LAUNCHED();
        }
        return PHMM_OK;
    };
    ChunkOrder chunk_order(e);
    bool timed = false;
    size_t n_timed = 0;
    for (long long p0 = 0, w0 = 0, g0 = 0; p0 < n_pairs || w0 < n_wide || g0 < n_generic;) {
        if (p0 < n_pairs) {
            const int np = (int)std::min<long long>(pairs_per_tile, n_pairs - p0);
            p.pair_reads = e->pairs.as<int>() + 2 * p0;
            p.n_pairs = np;
            p.pair_base = (int)p0;
            p.list = p.pair_reads; p.list_kind = 0; p.n_list = 2 * np; p.list_base = (int)(2 * p0);
            p.row_stride = fast_row_stride;
            p.fb_route = (p.atasks && flank_fb_ok) ? 1 : 0;
            if (use_mapper) {
                launch_mapper(p.list, p.n_list, p.list_base, 0);
                LAUNCHED();
                p.kpos = e->kpos.as<int32_t>(); p.kcnt = e->kcnt.as<uint8_t>();
            }
            CU(cudaMemsetAsync(counters, 0, 8 * sizeof(int), e->stream));                       // cursors, any-tasks flags (the traceback queue is empty between tiles)
            CU(cudaMemsetAsync(p.fcnt, 0, (size_t)2 * np * sizeof(int), e->stream));
            CU(cudaMemsetAsync(p.gcnt, 0, (size_t)2 * np * sizeof(int), e->stream));
            CU(cudaMemsetAsync(p.acnt, 0, (size_t)2 * np * sizeof(int), e->stream));
            {   // classify pass: shortcut values → best[], near-flank candidates → slow queue, DP candidates → task lists
                const long long threads = 2LL * np * H;
                k_populate_generic<64, true><<<(unsigned)((threads + 127) / 128), 128, 0, e->stream>>>(p);
                LAUNCHED();
            }
            lap(" classify queued");
            const int tasks_per_round = role_warps ? 32 : (32 / groups) / NL;
            p.units_per_pair = std::max(1, (p.fcap + tasks_per_round * kRoundsPerUnit - 1) / (tasks_per_round * kRoundsPerUnit));
            const int claimers_per_block = role_warps ? role_groups : kFastWarpsPerBlock;      // groups of warps / warps that claim work units
            const int want_blocks = (int)std::min<long long>(1LL << 30, ((long long)(np / groups) * p.units_per_pair + claimers_per_block - 1) / claimers_per_block);
            const unsigned grid = (unsigned)std::max(1, std::min(want_blocks, e->sm_count * (role_warps ? role_blocks_per_sm : blocks_per_sm)));
            while (e->tile_events.size() < 2 * (n_timed + 1)) { cudaEvent_t ev; CU(cudaEventCreate(&ev)); e->tile_events.push_back(ev); }
            CU(chunk_order.wait_for_previous());
            CU(cudaEventRecord(e->tile_events[2 * n_timed], e->stream));
#define PHMM_FAST_LAUNCH(B, GG) k_populate_fast<B, GG><<<grid, kFastWarpsPerBlock * 32, smem, e->stream>>>(p);
            if (role_warps && band == 32) k_populate_roles<32><<<grid, kFastWarpsPerBlock * 32, role_smem, e->stream>>>(p);
            else if (role_warps) k_populate_roles<64><<<grid, kFastWarpsPerBlock * 32, role_smem, e->stream>>>(p);
            else { PHMM_FAST_DISPATCH(PHMM_FAST_LAUNCH) }
            LAUNCHED();
            // with a flank state the tile's DP work is split between the score-only kernel and the flank-aware kernels: time them together
            if (!p.use_flanks) CU(cudaEventRecord(e->tile_events[2 * n_timed + 1], e->stream));
            lap(" dp queued");
            if ((rc = launch_flank(2 * np, fast_row_stride))) return rc;
            if (p.use_flanks) CU(cudaEventRecord(e->tile_events[2 * n_timed + 1], e->stream));
            ++n_timed; timed = true;
            p0 += np;
        } else if (w0 < n_wide) {
            const int nw = (int)std::min<long long>(reads_per_tile, n_wide - w0);
            p.list = e->wide_reads.as<int>() + w0; p.list_kind = 1; p.n_list = nw; p.list_base = (int)w0;
            p.row_stride = wide_row_stride;
            p.fb_route = 0;
            const long long threads = (long long)nw * H;
            const unsigned cgrid = (unsigned)std::max<long long>(1, std::min<long long>((threads + 127) / 128, (long long)e->sm_count * 64));
            if (use_mapper) {
                launch_mapper(p.list, nw, (int)w0, 1);
                LAUNCHED();
                p.kpos = e->kpos.as<int32_t>(); p.kcnt = e->kcnt.as<uint8_t>();
            }
            CU(cudaMemsetAsync(counters, 0, 8 * sizeof(int), e->stream));
            CU(cudaMemsetAsync(p.fcnt, 0, (size_t)nw * sizeof(int), e->stream));
            CU(cudaMemsetAsync(p.gcnt, 0, (size_t)nw * sizeof(int), e->stream));
            CU(cudaMemsetAsync(p.acnt, 0, (size_t)nw * sizeof(int), e->stream));
            k_populate_generic<64, true><<<cgrid, 128, 0, e->stream>>>(p);          // classify pass over the wide list
            LAUNCHED();
            const unsigned wgrid = (unsigned)std::max(1, std::min((nw + wide_warps - 1) / wide_warps, e->sm_count * wide_blocks_per_sm));
            const bool time_wide = n_pairs == 0;
            if (time_wide) { while (e->tile_events.size() < 2 * (n_timed + 1)) { cudaEvent_t ev; CU(cudaEventCreate(&ev)); e->tile_events.push_back(ev); } }
            CU(chunk_order.wait_for_previous());
            if (time_wide) CU(cudaEventRecord(e->tile_events[2 * n_timed], e->stream));
#define PHMM_WIDE_LAUNCH(CC, NN) k_populate_wide<CC, NN><<<wgrid, wide_warps * 32, wsmem, e->stream>>>(p);
            PHMM_WIDE_DISPATCH(PHMM_WIDE_LAUNCH)
            LAUNCHED();
            if (time_wide) { CU(cudaEventRecord(e->tile_events[2 * n_timed + 1], e->stream)); ++n_timed; timed = true; }
            if (wide_row_stride <= fast_row_stride + 8 || (size_t)kFastWarpsPerBlock * wide_row_stride * sizeof(RowEntry) <= (200u << 10)) {
                if ((rc = launch_flank(nw, wide_row_stride))) return rc;
            }
            w0 += nw;
        } else {
            const int ng = (int)std::min<long long>(reads_per_tile, n_generic - g0);
            p.list = e->generic_reads.as<int>() + g0; p.list_kind = 2; p.n_list = ng; p.list_base = (int)g0;
            p.fb_route = 0;
            // ng is an upper bound (normally there are no generic reads at all): grid-stride kernels on a bounded grid
            const long long threads = (long long)ng * H;
            const unsigned ggrid = (unsigned)std::max<long long>(1, std::min<long long>((threads + 63) / 64, (long long)e->sm_count * 32));
            if (use_mapper) {
                launch_mapper(p.list, ng, (int)g0, 2);
                LAUNCHED();
                p.kpos = e->kpos.as<int32_t>(); p.kcnt = e->kcnt.as<uint8_t>();
            }
            const bool time_generic = n_pairs == 0 && n_wide == 0 && n_timed == 0;
            CU(chunk_order.wait_for_previous());
            if (time_generic) CU(cudaEventRecord(e->ev0, e->stream));
            if (band <= 32) k_populate_generic<64, false><<<ggrid, 64, 0, e->stream>>>(p);
            else k_populate_generic<kGenericMaxDiag, false><<<ggrid, 64, 0, e->stream>>>(p);
            LAUNCHED();
            if (time_generic) { CU(cudaEventRecord(e->ev1, e->stream)); timed = true; }
            g0 += ng;
        }
        if (p.use_flanks) {
            if (band <= 32) k_slow_flank<64><<<slow_blocks, 256, 0, e->stream>>>(p, e->bp.as<unsigned char>());
            else k_slow_flank<kGenericMaxDiag><<<slow_blocks, 256, 0, e->stream>>>(p, e->bp.as<unsigned char>());
            LAUNCHED();
            CU(cudaMemsetAsync(p.slow_count, 0, sizeof(int), e->stream));
        }
        CU(cudaGetLastError());
    }

    chunk_order.publish(true);
    lap("tiles enqueued");
    if (template_off) {
        // paired / linked reads: one value per (haplotype, template), summed straight from the integer penalties
        const long long* d_toff;
        if ((rc = stage(e, e->toff, (const long long*)template_off, (size_t)T + 1, space, &d_toff))) return rc;
        CU(e->tregion.ensure((size_t)T * sizeof(int)));
        k_template_regions<<<(T + 255) / 256, 256, 0, e->stream>>>(T, G, e->regs.as<RegionInfo>(), e->tregion.as<int>());
        LAUNCHED();
        if (space == PHMM_SPACE_DEVICE) {
            k_check_templates<<<(T + 255) / 256, 256, 0, e->stream>>>(T, d_toff, e->tregion.as<int>(), e->regs.as<RegionInfo>(), e->flags.as<int>());
            LAUNCHED();
        }
        const long long HT = multi->total_tout;
        CU(e->out.ensure((size_t)std::max<long long>(HT, 1) * sizeof(double)));
        double* d_tout = space == PHMM_SPACE_DEVICE ? out : e->out.as<double>();
        const long long threads = (long long)H * T;
        k_template_epilogue<<<(unsigned)((threads + 255) / 256), 256, 0, e->stream>>>(p.best, p.status, s.rd, e->regs.as<RegionInfo>(), H, T, d_toff,
                                                                                      e->tregion.as<int>(), cfg->use_mapping_quality, cfg->mapping_quality_cap,
                                                                                      cfg->mapping_quality_cap_trigger, e->flags.as<int>(), d_tout);
        LAUNCHED();
        CU(cudaGetLastError());
        if (space == PHMM_SPACE_HOST) {
            CU(cudaMemcpyAsync(out, d_tout, (size_t)HT * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
            if (status) CU(cudaMemcpyAsync(status, p.status, (size_t)HR * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
        } else if (status) {
            CU(cudaMemcpyAsync(status, p.status, (size_t)HR * sizeof(int), cudaMemcpyDeviceToDevice, e->stream));
        }
    } else {
        CU(e->out.ensure((size_t)HR * sizeof(double)));
        double* d_out = space == PHMM_SPACE_DEVICE ? out : e->out.as<double>();
        const long long threads = (long long)H * R;
        k_epilogue<<<(unsigned)((threads + 255) / 256), 256, 0, e->stream>>>(p.best, p.status, s.rd, e->regs.as<RegionInfo>(), H, cfg->use_mapping_quality,
                                                                             cfg->mapping_quality_cap, cfg->mapping_quality_cap_trigger, d_out,
                                                                             d_out == out && space == PHMM_SPACE_DEVICE && out_pitch > R ? out_pitch - R : 0LL);
        LAUNCHED();
        CU(cudaGetLastError());
        if (space == PHMM_SPACE_HOST) {
            if (out_pitch == 0 || out_pitch == R) {
                CU(cudaMemcpyAsync(out, d_out, (size_t)HR * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
                if (status) CU(cudaMemcpyAsync(status, p.status, (size_t)HR * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
            } else {
                CU(cudaMemcpy2DAsync(out, (size_t)out_pitch * sizeof(double), d_out, (size_t)R * sizeof(double), (size_t)R * sizeof(double), H, cudaMemcpyDeviceToHost, e->stream));
                if (status) CU(cudaMemcpy2DAsync(status, (size_t)out_pitch * sizeof(int), p.status, (size_t)R * sizeof(int), (size_t)R * sizeof(int), H, cudaMemcpyDeviceToHost, e->stream));
            }
        } else if (status) {
            CU(cudaMemcpyAsync(status, p.status, (size_t)HR * sizeof(int), cudaMemcpyDeviceToDevice, e->stream));
        }
    }
    int flags_host[1] = {0};
    lap("enqueued");
    CU(cudaMemcpyAsync(flags_host, e->flags.p, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaMemcpyAsync(&tot, d_tot, sizeof(SchedTotals), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    lap("done");
    if (flags_host[0] & 1) { e->err = "snv prior / gap penalty outside [0,127]"; return PHMM_ERR_INVALID; }
    if (flags_host[0] & kFlagBadTemplates) { e->err = "template offsets must be non-decreasing and cover each region's reads exactly"; return PHMM_ERR_INVALID; }
    if (trace && n_timed) { float ms = 0.f; cudaEventElapsedTime(&ms, e->tile_events[0], e->tile_events[2 * n_timed - 1]); std::fprintf(stderr, "[phmm %p] dp span %.3f ms\n", (void*)e, ms); }
    if (n_timed) {
        double total = 0.0;
        for (size_t t = 0; t < n_timed; ++t) { float ms = 0.f; if (cudaEventElapsedTime(&ms, e->tile_events[2 * t], e->tile_events[2 * t + 1]) == cudaSuccess) total += ms; }
        e->last_dp_ms = total;
    } else if (timed) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, e->ev0, e->ev1) == cudaSuccess) e->last_dp_ms = ms;
    }
    // GCUPS numerator when every pair runs exactly one DP (benchmark mode); otherwise an upper bound on DP work
    e->last_dp_cells = tot.cells;
    if (flags_host[0] & (4 | 8)) { e->err = "internal task queue overflow"; return PHMM_ERR_NOMEM; }
    if (flags_host[0] & 2) { e->err = "Haplotype is too short for alignment"; return PHMM_ERR_SHORT_HAPLOTYPE; }
    return PHMM_OK;
}

int phmm_populate_regions(phmm_engine* e, const phmm_config* cfg,
                          const phmm_haplotypes* haps, const phmm_reads* reads, const phmm_regions* regions,
                          double* out, int32_t* status, int space)
{
    return phmm_populate_regions_ex(e, cfg, haps, reads, regions, nullptr, nullptr, out, status, space);
}

int phmm_populate_regions_ex(phmm_engine* e, const phmm_config* cfg,
                             const phmm_haplotypes* haps, const phmm_reads* reads, const phmm_regions* regions,
                             const phmm_region_templates* templates, const phmm_positions* positions,
                             double* out, int32_t* status, int space)
{
    if (!e) return PHMM_ERR_INVALID;
    if (!regions || regions->n <= 0 || !regions->hap_first || !regions->read_first || !haps || !reads) { e->err = "null / empty region list"; return PHMM_ERR_INVALID; }
    if (templates && (!templates->template_first || !templates->template_off)) { e->err = "null template arrays"; return PHMM_ERR_INVALID; }
    RegionSetup setup;
    setup.regs.resize((size_t)regions->n);
    if (regions->hap_first[0] != 0 || regions->read_first[0] != 0 || regions->hap_first[regions->n] != haps->n || regions->read_first[regions->n] != reads->n) {
        e->err = "region ranges must cover the haplotype and read blocks exactly"; return PHMM_ERR_INVALID;
    }
    for (int g = 0; g < regions->n; ++g) {
        RegionInfo& r = setup.regs[(size_t)g];
        r.h0 = regions->hap_first[g]; r.nH = regions->hap_first[g + 1] - r.h0;
        r.r0 = regions->read_first[g]; r.nR = regions->read_first[g + 1] - r.r0;
        if (r.nH <= 0 || r.nR <= 0) { e->err = "every region needs at least one haplotype and one read"; return PHMM_ERR_INVALID; }
        r.out_off = setup.total_out;
        setup.total_out += (long long)r.nH * r.nR;
        setup.Hmax = std::max(setup.Hmax, r.nH);
        const bool fl = regions->flank && regions->flank[g].has_flank && cfg && cfg->use_flank_state;
        r.use_flanks = fl ? 1 : 0; r.lhs = fl ? (int)regions->flank[g].lhs_flank : 0; r.rhs = fl ? (int)regions->flank[g].rhs_flank : 0; r.pad = 0;
        setup.any_flank = setup.any_flank || fl;
    }
    if (templates) {
        const int32_t* tf = templates->template_first;
        if (tf[0] != 0) { e->err = "template_first must start at 0"; return PHMM_ERR_INVALID; }
        for (int g = 0; g < regions->n; ++g) {
            RegionInfo& r = setup.regs[(size_t)g];
            r.t0 = tf[g]; r.nT = tf[g + 1] - tf[g];
            // a region has reads, so at least one template covers them
            if (r.nT <= 0) { e->err = "template_first must be increasing: every region needs at least one template"; return PHMM_ERR_INVALID; }
            r.tout_off = setup.total_tout;
            setup.total_tout += (long long)r.nH * r.nT;
        }
        setup.n_templates = tf[regions->n];
        if (space == PHMM_SPACE_HOST) {
            const int64_t* to = templates->template_off;
            for (int t = 0; t < setup.n_templates; ++t) if (to[t + 1] < to[t]) { e->err = "template offsets must be non-decreasing"; return PHMM_ERR_INVALID; }
            for (const RegionInfo& r : setup.regs) {
                if (to[r.t0] != r.r0 || to[r.t0 + r.nT] != (int64_t)r.r0 + r.nR) { e->err = "each region's templates must cover exactly its reads"; return PHMM_ERR_INVALID; }
            }
        }
    }
    return populate_impl(e, cfg, haps, reads, positions, nullptr, out, status, space, 0, templates ? templates->template_off : nullptr,
                         setup.n_templates, &setup);
}

int phmm_populate_ld(phmm_engine* e, const phmm_config* cfg,
                     const phmm_haplotypes* haps, const phmm_reads* reads,
                     const phmm_positions* positions, const phmm_flank_state* flank,
                     double* out, int64_t out_ld, int32_t* status)
{
    if (!e) return PHMM_ERR_INVALID;
    if (!reads || out_ld < reads->n) { e->err = "out_ld must be at least the number of reads"; return PHMM_ERR_INVALID; }
    return populate_impl(e, cfg, haps, reads, positions, flank, out, status, PHMM_SPACE_DEVICE, (long long)out_ld);
}

// -------------------------------------------------------------------------------------------------------------
// Peer output: one rank's matrix mapped into the other ranks' address spaces (CUDA IPC over NVLink / NVSwitch)
// -------------------------------------------------------------------------------------------------------------
int phmm_device_alloc(int device, size_t bytes, void** dev_ptr)
{
    if (!dev_ptr || bytes == 0) return PHMM_ERR_INVALID;
    *dev_ptr = nullptr;
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return PHMM_ERR_CUDA; }
    if (cudaMalloc(dev_ptr, bytes) != cudaSuccess) { cudaGetLastError(); *dev_ptr = nullptr; return PHMM_ERR_NOMEM; }
    return PHMM_OK;
}

int phmm_device_free(void* dev_ptr)
{
    if (dev_ptr && cudaFree(dev_ptr) != cudaSuccess) { cudaGetLastError(); return PHMM_ERR_CUDA; }
    return PHMM_OK;
}

int phmm_ipc_export(const void* dev_ptr, unsigned char handle[PHMM_IPC_HANDLE_BYTES])
{
    static_assert(sizeof(cudaIpcMemHandle_t) == PHMM_IPC_HANDLE_BYTES, "handle size");
    if (!dev_ptr || !handle) return PHMM_ERR_INVALID;
    cudaIpcMemHandle_t h;
    if (cudaIpcGetMemHandle(&h, const_cast<void*>(dev_ptr)) != cudaSuccess) { cudaGetLastError(); return PHMM_ERR_CUDA; }
    std::memcpy(handle, &h, sizeof(h));
    return PHMM_OK;
}

int phmm_ipc_open(int device, const unsigned char handle[PHMM_IPC_HANDLE_BYTES], void** dev_ptr)
{
    if (!handle || !dev_ptr) return PHMM_ERR_INVALID;
    *dev_ptr = nullptr;
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return PHMM_ERR_CUDA; }
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    if (cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); *dev_ptr = nullptr; return PHMM_ERR_CUDA; }
    return PHMM_OK;
}

int phmm_ipc_close(void* dev_ptr)
{
    if (dev_ptr && cudaIpcCloseMemHandle(dev_ptr) != cudaSuccess) { cudaGetLastError(); return PHMM_ERR_CUDA; }
    return PHMM_OK;
}

int phmm_populate_templates(phmm_engine* e, const phmm_config* cfg,
                            const phmm_haplotypes* haps, const phmm_reads* reads,
                            const int64_t* template_off, int32_t n_templates,
                            const phmm_positions* positions, const phmm_flank_state* flank,
                            double* out, int32_t* status, int space)
{
    if (!e) return PHMM_ERR_INVALID;
    if (!template_off || n_templates <= 0 || !reads) { e->err = "null / empty template offsets"; return PHMM_ERR_INVALID; }
    if (space == PHMM_SPACE_HOST) {
        if (template_off[0] != 0 || template_off[n_templates] != reads->n) { e->err = "template offsets must cover the reads exactly"; return PHMM_ERR_INVALID; }
        for (int t = 0; t < n_templates; ++t) if (template_off[t + 1] < template_off[t]) { e->err = "template offsets must be non-decreasing"; return PHMM_ERR_INVALID; }
    }
    return populate_impl(e, cfg, haps, reads, positions, flank, out, status, space, 0, template_off, n_templates);
}

int phmm_populate(phmm_engine* e, const phmm_config* cfg,
                  const phmm_haplotypes* haps, const phmm_reads* reads,
                  const phmm_positions* positions, const phmm_flank_state* flank,
                  double* out, int32_t* status, int space)
{
    if (!e) return PHMM_ERR_INVALID;
    // Pipelined path: host-resident batch, no caller-supplied position lists (a [H][R] CSR cannot be sliced by columns
    // without a pass over it), enough pairs to amortise the per-chunk overheads.
    static const long long kForcedChunkPairs = [] {
        const char* v = std::getenv("PHMM_CHUNK_PAIRS");          // test hook: force the pipelined path on small batches
        const long long n = v ? std::atoll(v) : 0;
        return n > 0 ? n : 0LL;
    }();
    // chunk size: an eighth of the batch, between 2M pairs (below that the per-chunk launch chain shows) and 8M pairs
    const long long all_pairs = (haps && reads) ? (long long)haps->n * reads->n : 0;
    const long long kChunkPairs = kForcedChunkPairs ? kForcedChunkPairs : std::max<long long>(2LL << 20, std::min<long long>(8LL << 20, all_pairs / 8));
    const bool can_chunk = !e->is_sub && space == PHMM_SPACE_HOST && haps && reads && cfg && out && haps->n > 0 && reads->n > 1 &&
                           reads->off && reads->mapq && reads->reverse && !(positions && positions->off && positions->pos) &&
                           all_pairs >= 2 * kChunkPairs;
    if (!can_chunk) return populate_impl(e, cfg, haps, reads, positions, flank, out, status, space, 0);
    e->err.clear(); e->launches_last = 0; e->last_dp_ms = 0.0; e->last_dp_cells = 0;
    for (phmm_engine*& sub : e->sub) {
        if (!sub) {
            const int rc = phmm_create(&sub, e->device);
            if (rc != PHMM_OK) { e->err = std::string("sub-engine: ") + phmm_last_error(nullptr); return rc; }
            sub->is_sub = true;
            sub->parent = e;
            sub->reserved_sms = e->reserved_sms;
            if (cudaEventCreateWithFlags(&sub->order_ev, cudaEventDisableTiming) != cudaSuccess) {
                phmm_destroy(sub);          // a sub-engine without its ordering event must not survive into the next call
                sub = nullptr;
                e->err = "sub-engine: event creation failed";
                return PHMM_ERR_CUDA;
            }
        }
    }
    e->sub[0]->peer = e->sub[1]; e->sub[1]->peer = e->sub[0];
    e->order.recorded = -1;
    const int R = reads->n, H = haps->n;
    const long long reads_per_chunk = std::max<long long>(64, kChunkPairs / H);
    const int n_chunks = (int)((R + reads_per_chunk - 1) / reads_per_chunk);
    int rcs[2] = {PHMM_OK, PHMM_OK};
    std::string errs[2];
    int64_t cells[2] = {0, 0}, launches[2] = {0, 0};
    auto worker = [&](int k) {
        phmm_engine* se = e->sub[k];
        std::vector<int64_t> off;
        for (int c = k; c < n_chunks; c += 2) {
            const long long lo = (long long)c * reads_per_chunk, hi = std::min<long long>(R, lo + reads_per_chunk);
            const int n = (int)(hi - lo);
            off.resize((size_t)n + 1);
            const int64_t base = reads->off[lo];
            for (int i = 0; i <= n; ++i) off[i] = reads->off[lo + i] - base;
            phmm_reads sub_reads {n, off.data(), reads->bases + base, reads->quals + base, reads->mapq + lo, reads->reverse + lo,
                                  reads->begin ? reads->begin + lo : nullptr};
            se->chunk_index = c;
            const int rc = populate_impl(se, cfg, haps, &sub_reads, nullptr, flank, out + lo, status ? status + lo : nullptr, PHMM_SPACE_HOST, R);
            {   // a chunk that failed before reaching its DP phase must not leave the other worker waiting for it
                std::lock_guard<std::mutex> lk(e->order.m);
                e->order.recorded = std::max<long long>(e->order.recorded, rc != PHMM_OK && rc != PHMM_ERR_SHORT_HAPLOTYPE ? (long long)n_chunks : (long long)c);
            }
            e->order.cv.notify_all();
            cells[k] += se->last_dp_cells; launches[k] += se->launches_last;
            if (rc != PHMM_OK && rc != PHMM_ERR_SHORT_HAPLOTYPE) { rcs[k] = rc; errs[k] = se->err; return; }
            if (rc == PHMM_ERR_SHORT_HAPLOTYPE) { rcs[k] = rc; errs[k] = se->err; }   // keep going: every pair's status is still written
        }
    };
    std::thread t1(worker, 1);
    worker(0);
    t1.join();
    e->last_dp_cells = cells[0] + cells[1];
    e->launches_last = launches[0] + launches[1];
    e->launches_total += e->launches_last;
    for (int k = 0; k < 2; ++k) if (rcs[k] != PHMM_OK && rcs[k] != PHMM_ERR_SHORT_HAPLOTYPE) { e->err = errs[k]; return rcs[k]; }
    for (int k = 0; k < 2; ++k) if (rcs[k] == PHMM_ERR_SHORT_HAPLOTYPE) { e->err = errs[k]; return rcs[k]; }
    return PHMM_OK;
}

} // extern "C"
