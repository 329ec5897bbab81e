// pob_b200.cu -- host side of the C-ABI (include/pob_b200.h) of the batched witness generator; the CUDA kernels
// (sm_100a) live in kernels.cuh.  There is no host execution path for any witness value: without a device pob_create fails.
//
// Scheduling model.  A batch is cut into eval CHUNKS (instances per k_eval launch; the compact stores of two chunks are
// resident) and expand GROUPS (witnesses materialised per k_expand_round / k_expand_codes launch pair, each into its own
// HBM slot).  A small pump (advance()) queues work as far as resources allow: eval(c) once the store ring half it
// overwrites has been expanded, group g once every slot it writes is free.  Three streams: inputs H2D one chunk ahead,
// k_eval on the highest-priority stream (its 32-CTA grid must get SMs while the expand grid of hundreds of thousands of
// CTAs drains), expand on the lowest.  Slots are freed by the consumer (pob_release; stream-ordered, so the stall happens
// on the GPU), by the built-in digest consumer, or -- only when the caller says POB_RUN_DISCARD -- at once.
#include <cuda.h>             // driver API types only: the entry points are looked up at run time (witness slots below)
#include <cuda_runtime.h>
#include <fcntl.h>
#include <unistd.h>
#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>
#include "../../include/pob_b200.h"
#include "compiler.h"
#include "kernels.cuh"

using namespace pob;

static thread_local std::string g_err;
static int fail(int code, const std::string &msg) { g_err = msg; return code; }
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) throw std::runtime_error(std::string(#call) + ": " + cudaGetErrorString(e_)); } while (0)

// Tuning / profiling knobs (POB_* environment variables) exist only in the -DPOB_TUNING build (`make tuning`, used by
// tools/gpu_sweep3.sh); the shipped library reads no environment variable.
static const char *tune_env(const char *name) {
#ifdef POB_TUNING
    return getenv(name);
#else
    (void)name; return nullptr;
#endif
}

// =============================================================================================================
// exporter: resident witness -> host (.wtns image), several copy streams into a pinned staging ring, file I/O on a
// writer thread so that D2H DMA and disk writes overlap (SURVEY.md 8(f) rank 1)
// =============================================================================================================
namespace {

struct Exporter {
    static const int NB = 8, NS = 2;
    const size_t bb = 32u << 20;                       // 32 MiB per hop
    int device; void *buf[NB] = {}; cudaEvent_t ev[NB] = {}; cudaStream_t cs[NS] = {}; cudaEvent_t ev_join = nullptr;
    struct Job { int b; int fd; uint64_t off; size_t bytes; bool close_fd; };
    std::deque<Job> q; bool busy[NB] = {}; bool stop = false, io_err = false;
    std::mutex m; std::condition_variable cv; std::thread th;
    int next_b = 0; unsigned rr = 0; uint64_t bytes_moved = 0;

    explicit Exporter(int dev) : device(dev) {
        CU(cudaSetDevice(device));
        for (int i = 0; i < NB; i++) { CU(cudaMallocHost(&buf[i], bb)); CU(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming)); }
        for (int i = 0; i < NS; i++) CU(cudaStreamCreateWithFlags(&cs[i], cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
        th = std::thread([this] { run(); });
    }
    ~Exporter() {
        { std::lock_guard<std::mutex> l(m); stop = true; }
        cv.notify_all();
        if (th.joinable()) th.join();
        cudaSetDevice(device);
        for (int i = 0; i < NS; i++) if (cs[i]) { cudaStreamSynchronize(cs[i]); cudaStreamDestroy(cs[i]); }
        for (int i = 0; i < NB; i++) { if (buf[i]) cudaFreeHost(buf[i]); if (ev[i]) cudaEventDestroy(ev[i]); }
        if (ev_join) cudaEventDestroy(ev_join);
    }
    void run() {                                       // writer thread
        cudaSetDevice(device);
        for (;;) {
            Job j;
            { std::unique_lock<std::mutex> l(m); cv.wait(l, [this] { return stop || !q.empty(); }); if (q.empty()) return; j = q.front(); q.pop_front(); }
            bool ok = cudaEventSynchronize(ev[j.b]) == cudaSuccess;
            if (ok && j.fd >= 0) {
                const char *p = (const char *)buf[j.b]; size_t left = j.bytes; uint64_t off = j.off;
                while (left) { ssize_t w = pwrite(j.fd, p, left, (off_t)off); if (w <= 0) { ok = false; break; } p += w; left -= (size_t)w; off += (uint64_t)w; }
            }
            if (j.close_fd && j.fd >= 0 && close(j.fd) != 0) ok = false;
            { std::lock_guard<std::mutex> l(m); busy[j.b] = false; if (!ok) io_err = true; }
            cv.notify_all();
        }
    }
    int grab() {                                       // staging buffers are used strictly round-robin
        std::unique_lock<std::mutex> l(m);
        const int b = next_b; cv.wait(l, [&] { return !busy[b]; });
        busy[b] = true; next_b = (b + 1) % NB; return b;
    }
    void drain() { std::unique_lock<std::mutex> l(m); cv.wait(l, [this] { if (!q.empty()) return false; for (int i = 0; i < NB; i++) if (busy[i]) return false; return true; }); }
    // iden3 binary witness format, version 2 (what the circom runtime's writeBinWitness emits; SURVEY.md Appendix B)
    static size_t header(uint8_t *o, uint64_t n) {
        uint32_t u32; uint64_t u64; Fr p = fr_p(); size_t k = 0;
        auto put = [&](const void *s, size_t b) { memcpy(o + k, s, b); k += b; };
        put("wtns", 4); u32 = 2; put(&u32, 4); u32 = 2; put(&u32, 4);
        u32 = 1; put(&u32, 4); u64 = 40; put(&u64, 8); u32 = 32; put(&u32, 4); put(p.l, 32); u32 = (uint32_t)n; put(&u32, 4);
        u32 = 2; put(&u32, 4); u64 = 32ull * n; put(&u64, 8);
        return k;                                      // 76
    }
    // queue the transfer of one resident witness; fd < 0: host memory only.  On return every D2H copy has been issued;
    // stream cs[0] is ordered after all of them (the caller releases the slot on cs[0]).
    void send(const uint64_t *dwit, uint64_t n_signals, int fd) {
        CU(cudaSetDevice(device));
        if (fd >= 0) { uint8_t hd[80]; size_t hb = header(hd, n_signals); if (pwrite(fd, hd, hb, 0) != (ssize_t)hb) { std::lock_guard<std::mutex> l(m); io_err = true; } }
        const uint64_t total = 32ull * n_signals; const uint64_t nch = (total + bb - 1) / bb;
        for (uint64_t c = 0; c < nch; c++) {
            const uint64_t off = c * bb; const size_t bytes = (size_t)std::min<uint64_t>(bb, total - off);
            const int b = grab(); cudaStream_t s = cs[rr++ % NS];
            CU(cudaMemcpyAsync(buf[b], (const char *)dwit + off, bytes, cudaMemcpyDeviceToHost, s));
            CU(cudaEventRecord(ev[b], s));
            { std::lock_guard<std::mutex> l(m); q.push_back(Job{b, fd, 76 + off, bytes, c + 1 == nch}); }
            cv.notify_all();
            bytes_moved += bytes;
        }
        if (nch == 0 && fd >= 0) close(fd);
        for (int i = 1; i < NS; i++) { CU(cudaEventRecord(ev_join, cs[i])); CU(cudaStreamWaitEvent(cs[0], ev_join, 0)); }
    }
};

}  // namespace

// =============================================================================================================
// handle
// =============================================================================================================
struct pob_handle {
    Program P; int device = 0;
    // device program
    Op *d_ops = nullptr; PsumOp *d_psums = nullptr; PoseidonOp *d_pos = nullptr; Fr *d_pos_konst = nullptr; AbsorbOp *d_abs = nullptr; Level *d_levels = nullptr; Code *d_aux = nullptr; Fr *d_konst = nullptr;
    Code *d_codes = nullptr; Tile *d_tiles = nullptr; Fr *d_invtab = nullptr; uint64_t *d_round_desc = nullptr;
    // stores (ring of RING chunks)
    static const uint32_t RING = 2;
    uint32_t chunk = 0; uint64_t store_stride = 0; uint64_t *d_stores = nullptr; uint64_t *d_inputs = nullptr;
    // witness slots (slot_alloc): mapped address, and the physical allocation and mapped size behind it
    struct SlotMem { CUmemGenericAllocationHandle handle; size_t bytes; };
    std::vector<uint64_t *> slots; std::vector<SlotMem> slot_mem;
    std::vector<int64_t> slot_owner;              // instance (of the current / last batch) whose witness the slot holds, -1 = none
    std::vector<cudaEvent_t> slot_rel_ev; std::vector<uint8_t> slot_rel_pending;   // stream-ordered release by the consumer
    std::vector<uint32_t> last_status; uint32_t last_n = 0;
    // per-batch buffers
    uint32_t cap_n = 0; uint32_t *d_status = nullptr; uint64_t *d_outputs = nullptr; unsigned long long *d_digests = nullptr;
    uint64_t **d_witptr = nullptr; uint32_t *d_planinst = nullptr;
    uint32_t *h_status = nullptr; uint64_t *h_outputs = nullptr; uint64_t *h_digests = nullptr; uint64_t **h_witptr = nullptr; uint32_t *h_planinst = nullptr;
    uint64_t *d_staged = nullptr; uint32_t n_staged = 0;
    long long *d_prof = nullptr; std::string prof_path;   // POB_TUNING: per-level clock stamps
    uint32_t xgroup = 0;                       // instances per expand launch (distinct witness slots)
    uint32_t n_round_tiles = 0;                // tiles [0, n_round_tiles) are KeccakfRound tiles, the rest code tiles
    uint64_t *d_block_base = nullptr; uint32_t n_blocks = 0;   // witness index of every KeccakfRound block (self-check)
    // Into PLAIN slots k_expand_round is launched with 85 KiB of (unused) dynamic shared memory so that only TWO of its CTAs are
    // resident per SM: fewer concurrent write streams give the DRAM controllers longer same-row bursts -- measured 7.35 TB/s with
    // 2 CTAs/SM vs 7.26 / 7.19 / 7.09 / 6.97 TB/s with 3 / 4 / 5 / 8, and 5.96 TB/s with 1 (profiles/r01_expand_sweep.md).
    // Into compressible slots the trade-off turns: 8 CTAs/SM (no cap) 1164 witnesses/s against 1108 with the 85 KiB cap
    // (profiles/r03b_compressed_expand_sweep.log).  Set in pob_create.
    uint32_t round_dyn_smem = 0;
    uint32_t round_threads = 256, codes_dyn_smem = 0, codes_ug = 4, codes_overlap = 0; bool serialize = false;   // changed by POB_TUNING knobs only
    int eval_threads = 512; uint32_t eval_cluster = 0, eval_prefetch = 0;   // operand prefetch measured no gain (profiles/r02c_eval_sweep.log)   // k_eval: threads per CTA; CTAs per instance (0 = chosen per launch)
    uint32_t pos_konst_bytes = 0, levels_bytes = 0, eval_smem = 0;
    bool skip_eval = false;                     // tuning: evaluate only the first two chunks, then re-expand their stores (isolates the cost of concurrency)
    uint32_t expand_cs = 0, eval_l2_mb = 0;     // tuning: streaming witness stores; persisting-L2 window (MB) for the eval stream's store accesses
    cudaStream_t s_eval = nullptr, s_exp = nullptr, s_exp2 = nullptr, s_h2d = nullptr;
    cudaEvent_t ev_eval_done[RING] = {nullptr, nullptr}, ev_exp_done[RING] = {nullptr, nullptr}, ev_h2d[RING] = {nullptr, nullptr},
                ev_start = nullptr, ev_end = nullptr, ev_tmp = nullptr, ev_fork = nullptr, ev_join = nullptr;
    std::vector<cudaEvent_t> ev_pool; size_t ev_used = 0;
    // the batch in flight
    struct Group { uint32_t begin, end, chunk; cudaEvent_t t0, t1; };
    struct Batch {
        bool active = false, async = false, staged = false, expand = false, digest = false;
        const uint64_t *inputs = nullptr; uint32_t n = 0, nchunks = 0, next_eval = 0, next_group = 0, acq_pos = 0;
        std::vector<uint32_t> plan, slot;         // instances to materialise (ascending) and their slots
        std::vector<uint8_t> st;                  // per plan entry: 0 = not handed out yet, 1 = held by the consumer, 2 = released / dropped
        std::vector<uint32_t> group_of;           // per plan entry
        std::vector<Group> groups; std::vector<uint32_t> chunk_gend;   // groups sorted by chunk; chunk_gend[c] = one past the last group of chunks <= c
        std::vector<cudaEvent_t> e0, e1, est;     // per chunk: eval begin / end, status+outputs on the host
        pob_timing T{};
    } B;
    Exporter *exporter = nullptr;
    pob_timing timing{};
    // constraint system for pob_selfcheck, built on first use
    struct DevCons {
        bool ready = false; ConsView flat{}, round{}; Fr *konst = nullptr; uint64_t *bases = nullptr; uint32_t n_blocks = 0;
        unsigned long long *rep = nullptr; std::vector<void *> allocs; pob_check_report info{};
    } cons;
};

static void cons_info(const Program &P, pob_check_report *r) {
    memset(r, 0, sizeof *r);
    const uint64_t nb = P.round_block_sig.size();
    auto count = [&](const ConsSet &S, uint64_t mult) {
        r->n_constraints += mult * (S.eq.size() / 2 + S.kc.size());
        for (const ConsR1 &q : S.r1) { if (r1_hint(q)) r->n_hints += mult; else { r->n_constraints += mult; if (q.na) r->n_nonlinear += mult; } }
    };
    count(P.cons_flat, 1); count(P.cons_round, nb);
    std::vector<uint8_t> seen(P.n_signals, 0);
    auto mark = [&](const ConsSet &S, uint64_t base) {
        for (uint32_t i : S.eq) seen[base + i] = 1;
        for (const ConsTerm &t : S.kc) seen[base + t.idx] = 1;
        for (const ConsTerm &t : S.terms) if (t.idx != CONS_ONE) seen[base + t.idx] = 1;
    };
    mark(P.cons_flat, 0);
    for (uint64_t b : P.round_block_sig) mark(P.cons_round, b);
    for (uint8_t v : seen) r->signals_read += v;
    r->first_failed = ~0ull;
}
static ConsView upload_cons(pob_handle *h, const ConsSet &S) {
    ConsView v{};
    auto up = [&](const void *src, size_t bytes) { void *d = nullptr; CU(cudaMalloc(&d, std::max<size_t>(16, bytes))); if (bytes) CU(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice)); h->cons.allocs.push_back(d); return d; };
    v.eq = (const uint32_t *)up(S.eq.data(), S.eq.size() * 4); v.n_eq = S.eq.size() / 2;
    v.kc = (const ConsTerm *)up(S.kc.data(), S.kc.size() * sizeof(ConsTerm)); v.n_kc = S.kc.size();
    v.r1 = (const ConsR1 *)up(S.r1.data(), S.r1.size() * sizeof(ConsR1)); v.n_r1 = S.r1.size();
    v.terms = (const ConsTerm *)up(S.terms.data(), S.terms.size() * sizeof(ConsTerm));
    return v;
}

static void fill_desc(const Program &P, pob_desc *d) {
    memset(d, 0, sizeof *d);
    d->n_signals = P.n_signals; d->n_outputs = P.n_outputs; d->n_inputs = P.n_inputs;
    d->witness_bytes = 32ull * P.n_signals; d->wtns_file_bytes = 76ull + 32ull * P.n_signals;
    d->store_bytes = 8ull * P.store_u64(); d->n_ops = P.ops.size(); d->n_absorbs = (uint32_t)P.absorbs.size();
    d->n_levels = (uint32_t)P.levels.size(); d->n_tiles = (uint32_t)P.tiles.size();
    d->opt_level = (uint32_t)P.opt_level; d->n_signals_o0 = P.n_signals_o0;
}
static bool flag_hcreate(int f) { return (f & POB_CREATE_HCREATE) != 0; }
static int flag_opt(int f) { return (f & POB_CREATE_O1) ? 1 : 0; }
static std::vector<Fr> params_vec(const uint64_t *params, int nparams) {
    std::vector<Fr> ps((size_t)(nparams > 0 ? nparams : 0));
    for (int i = 0; i < nparams; i++) memcpy(ps[(size_t)i].l, params + 4 * i, 32);
    return ps;
}
template <class T> static T *upload(const std::vector<T> &v) {
    T *d = nullptr; size_t bytes = std::max<size_t>(1, v.size()) * sizeof(T);
    CU(cudaMalloc(&d, bytes));
    if (!v.empty()) CU(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return d;
}
static cudaEvent_t pool_event(pob_handle *h) {
    if (h->ev_used == h->ev_pool.size()) { cudaEvent_t e; CU(cudaEventCreate(&e)); h->ev_pool.push_back(e); }
    return h->ev_pool[h->ev_used++];
}

// ---- witness slots ------------------------------------------------------------------------------------------------
// Every slot is its own cuMemCreate allocation, asked for with generic compression: the memory system then compresses each
// line on its way from L2 to DRAM, and 97.5 % of the entries are a single bit in a 32-byte field element.  Every reader
// (kernels, cudaMemcpy, the copy engines) still sees the plain bytes.  The driver entry points are looked up through the
// runtime, not linked, so that the library still loads on a machine without a driver.
namespace {
struct DriverVmm {
    decltype(&cuDeviceGet) device_get; decltype(&cuDeviceGetAttribute) device_attr; decltype(&cuMemGetAllocationGranularity) granularity;
    decltype(&cuMemCreate) create; decltype(&cuMemRelease) release;
    decltype(&cuMemAddressReserve) reserve; decltype(&cuMemAddressFree) address_free; decltype(&cuMemMap) map; decltype(&cuMemUnmap) unmap;
    decltype(&cuMemSetAccess) set_access;
    template <class F> static void sym(const char *name, F &fn) {
        void *p = nullptr; cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPointByVersion(name, &p, 12000, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !p)
            throw std::runtime_error(std::string("the CUDA driver has no entry point ") + name);
        fn = reinterpret_cast<F>(p);
    }
    DriverVmm() {
        sym("cuDeviceGet", device_get); sym("cuDeviceGetAttribute", device_attr); sym("cuMemGetAllocationGranularity", granularity);
        sym("cuMemCreate", create); sym("cuMemRelease", release);
        sym("cuMemAddressReserve", reserve); sym("cuMemAddressFree", address_free); sym("cuMemMap", map); sym("cuMemUnmap", unmap);
        sym("cuMemSetAccess", set_access);
    }
};
const DriverVmm &drv() { static const DriverVmm d; return d; }
}  // namespace
#define CUD(call) do { CUresult r_ = (call); if (r_ != CUDA_SUCCESS) throw std::runtime_error(std::string(#call) + ": CUresult " + std::to_string((int)r_)); } while (0)

static CUmemAllocationProp slot_prop(int device, bool compressible) {
    CUmemAllocationProp p{};
    p.type = CU_MEM_ALLOCATION_TYPE_PINNED; p.location.type = CU_MEM_LOCATION_TYPE_DEVICE; p.location.id = device;
    p.allocFlags.compressionType = compressible ? CU_MEM_ALLOCATION_COMP_GENERIC : CU_MEM_ALLOCATION_COMP_NONE;
    return p;
}
// bytes of one slot: the witness rounded up to the allocation granularity (of both props, in case a compressible create fails)
static size_t slot_bytes(int device, uint64_t wbytes) {
    size_t g = 1;
    for (bool c : {true, false}) { const CUmemAllocationProp p = slot_prop(device, c); size_t gc = 0; CUD(drv().granularity(&gc, &p, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED)); g = std::max(g, gc); }
    return (size_t)((wbytes + g - 1) / g * g);
}
// append one slot.  The compression type is a request: granted uncompressed, the slot is plain; a compressible create that
// fails is retried as a plain one.
static void slot_alloc(pob_handle *h, size_t bytes, bool compressible) {
    const DriverVmm &D = drv();
    pob_handle::SlotMem m{0, bytes};
    CUmemAllocationProp p = slot_prop(h->device, compressible);
    CUresult r = D.create(&m.handle, bytes, &p, 0);
    if (r != CUDA_SUCCESS && compressible) { p = slot_prop(h->device, false); r = D.create(&m.handle, bytes, &p, 0); }
    if (r != CUDA_SUCCESS) throw std::runtime_error("cuMemCreate of a witness slot failed: CUresult " + std::to_string((int)r));
    CUdeviceptr va = 0;
    r = D.reserve(&va, bytes, 0, 0, 0);
    if (r == CUDA_SUCCESS) {
        r = D.map(va, bytes, 0, m.handle, 0);
        if (r == CUDA_SUCCESS) {
            CUmemAccessDesc ad{}; ad.location = p.location; ad.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
            r = D.set_access(va, bytes, &ad, 1);
            if (r != CUDA_SUCCESS) D.unmap(va, bytes);
        }
        if (r != CUDA_SUCCESS) D.address_free(va, bytes);
    }
    if (r != CUDA_SUCCESS) { D.release(m.handle); throw std::runtime_error("mapping a witness slot failed: CUresult " + std::to_string((int)r)); }
    h->slots.push_back(reinterpret_cast<uint64_t *>(va)); h->slot_mem.push_back(m);
}
static void slots_free(pob_handle *h) {
    if (h->slots.empty()) return;
    cudaDeviceSynchronize();                   // as cudaFree would: no copy or kernel of any stream may still touch a slot
    const DriverVmm &D = drv();
    for (size_t s = 0; s < h->slots.size(); s++) {
        const CUdeviceptr va = reinterpret_cast<CUdeviceptr>(h->slots[s]); const size_t bytes = h->slot_mem[s].bytes;
        D.unmap(va, bytes); D.address_free(va, bytes); D.release(h->slot_mem[s].handle);
    }
    h->slots.clear(); h->slot_mem.clear();
}

// ---- batch machinery ------------------------------------------------------------------------------------------
static void ensure_batch_buffers(pob_handle *h, uint32_t n) {
    if (n <= h->cap_n) return;
    const Program &P = h->P;
    for (void *p : {(void *)h->d_status, (void *)h->d_outputs, (void *)h->d_digests, (void *)h->d_witptr, (void *)h->d_planinst}) if (p) cudaFree(p);
    for (void *p : {(void *)h->h_status, (void *)h->h_outputs, (void *)h->h_digests, (void *)h->h_witptr, (void *)h->h_planinst}) if (p) cudaFreeHost(p);
    h->d_status = nullptr; h->d_outputs = nullptr; h->d_digests = nullptr; h->d_witptr = nullptr; h->d_planinst = nullptr;
    h->h_status = nullptr; h->h_outputs = nullptr; h->h_digests = nullptr; h->h_witptr = nullptr; h->h_planinst = nullptr; h->cap_n = 0;
    const size_t no = std::max<uint32_t>(1, P.n_outputs);
    CU(cudaMalloc(&h->d_status, (size_t)n * 4)); CU(cudaMalloc(&h->d_outputs, (size_t)n * no * 32));
    CU(cudaMalloc(&h->d_digests, (size_t)n * 8)); CU(cudaMalloc(&h->d_witptr, (size_t)n * sizeof(uint64_t *))); CU(cudaMalloc(&h->d_planinst, (size_t)n * 4));
    CU(cudaMallocHost(&h->h_status, (size_t)n * 4)); CU(cudaMallocHost(&h->h_outputs, (size_t)n * no * 32));
    CU(cudaMallocHost(&h->h_digests, (size_t)n * 8)); CU(cudaMallocHost(&h->h_witptr, (size_t)n * sizeof(uint64_t *))); CU(cudaMallocHost(&h->h_planinst, (size_t)n * 4));
    h->cap_n = n;
}

static void enqueue_eval(pob_handle *h, uint32_t c) {
    pob_handle::Batch &B = h->B; const Program &P = h->P;
    const uint32_t E = h->chunk, R = pob_handle::RING, r = c % R, first = c * E, cnt = std::min(E, B.n - first);
    const size_t in_stride = (size_t)P.n_inputs * 4, no = std::max<uint32_t>(1, P.n_outputs);
    const uint64_t *d_in;
    if (B.staged) d_in = h->d_staged + (size_t)first * in_stride;
    else {
        // inputs travel on their own stream, one chunk ahead of the eval kernel that consumes them
        uint64_t *dst = h->d_inputs + (size_t)r * E * in_stride;
        if (c >= R) CU(cudaStreamWaitEvent(h->s_h2d, h->ev_eval_done[r], 0));
        if (in_stride) { CU(cudaMemcpyAsync(dst, B.inputs + (size_t)first * in_stride, (size_t)cnt * in_stride * 8, cudaMemcpyHostToDevice, h->s_h2d)); B.T.h2d_bytes += (uint64_t)cnt * in_stride * 8; }
        CU(cudaEventRecord(h->ev_h2d[r], h->s_h2d));
        CU(cudaStreamWaitEvent(h->s_eval, h->ev_h2d[r], 0));
        d_in = dst;
    }
    if (c >= R) CU(cudaStreamWaitEvent(h->s_eval, h->ev_exp_done[r], 0));      // store ring half r is free again
    uint64_t *stores = h->d_stores + (size_t)r * E * h->store_stride;
    EvalArgs ea{h->d_ops, h->d_abs, h->d_pos, h->d_pos_konst, h->d_psums, h->d_levels, (uint32_t)P.levels.size(), P.inv_begin, P.ginv_begin, P.inv_end, h->d_aux, h->d_konst, h->d_invtab,
                h->d_codes + P.out_code_off, P.n_outputs, P.n_inputs, P.val_base, stores, h->store_stride, d_in,
                h->d_status + first, h->d_outputs + (size_t)first * no * 4, (c == 0) ? h->d_prof : nullptr, h->pos_konst_bytes, h->levels_bytes, h->eval_prefetch, P.ginv_level};
    CU(cudaEventRecord(B.e0[c], h->s_eval));
    {   // one thread-block cluster per instance.  Cluster size: the largest power of two (<= 8) that still lets every instance of
        // the launch have its own SMs -- 8 CTAs for a single witness (latency), 4 for the 32-instance chunks of the main shape,
        // 1 when a chunk fills the GPU anyway (reduced witness, Spend); profiles/r02b_eval_sweep.log
        uint32_t C = h->eval_cluster;
        if (C == 0) { C = 8; while (C > 1 && cnt * C > 148) C >>= 1; }
        cudaLaunchConfig_t cfg{}; cudaLaunchAttribute at[1];
        cfg.gridDim = dim3(cnt * C); cfg.blockDim = dim3((unsigned)h->eval_threads); cfg.dynamicSmemBytes = h->eval_smem; cfg.stream = h->s_eval;
        at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        if (h->skip_eval && c >= R) CU(cudaMemsetAsync(h->d_status + first, 0, (size_t)cnt * 4, h->s_eval));   // TUNING: expand-only timing (stale stores)
        else switch (h->eval_threads) {
        case 256: CU(cudaLaunchKernelEx(&cfg, k_eval<256>, ea)); break;
        case 512: CU(cudaLaunchKernelEx(&cfg, k_eval<512>, ea)); break;
        default: CU(cudaLaunchKernelEx(&cfg, k_eval<1024>, ea)); break;
        }
    }
    CU(cudaEventRecord(B.e1[c], h->s_eval));
    CU(cudaEventRecord(h->ev_eval_done[r], h->s_eval));
    B.T.eval_launches++;
    // accept/reject and the output signals of this chunk go to the host right away (the consumer needs the status)
    CU(cudaMemcpyAsync(h->h_status + first, h->d_status + first, (size_t)cnt * 4, cudaMemcpyDeviceToHost, h->s_eval));
    B.T.d2h_bytes += (uint64_t)cnt * 4;
    if (P.n_outputs) { CU(cudaMemcpyAsync(h->h_outputs + (size_t)first * no * 4, h->d_outputs + (size_t)first * no * 4, (size_t)cnt * no * 32, cudaMemcpyDeviceToHost, h->s_eval)); B.T.d2h_bytes += (uint64_t)cnt * no * 32; }
    CU(cudaEventRecord(B.est[c], h->s_eval));
    const uint32_t g0 = c ? B.chunk_gend[c - 1] : 0;
    if (B.chunk_gend[c] == g0) CU(cudaEventRecord(h->ev_exp_done[r], h->s_eval));   // nothing of this chunk is materialised
}

static void enqueue_group(pob_handle *h, uint32_t g) {
    pob_handle::Batch &B = h->B; const Program &P = h->P;
    const pob_handle::Group &G = B.groups[g];
    const uint32_t E = h->chunk, R = pob_handle::RING, r = G.chunk % R, gc = G.end - G.begin;
    CU(cudaStreamWaitEvent(h->s_exp, h->ev_eval_done[r], 0));
    for (uint32_t k = G.begin; k < G.end; k++) {
        const uint32_t s = B.slot[k];
        if (h->slot_rel_pending[s]) { CU(cudaStreamWaitEvent(h->s_exp, h->slot_rel_ev[s], 0)); h->slot_rel_pending[s] = 0; }
        h->slot_owner[s] = (int64_t)B.plan[k];
    }
    ExpandArgs xa{h->d_tiles, h->d_codes, h->d_konst, reinterpret_cast<const uint2 *>(h->d_round_desc), h->d_stores + (size_t)r * E * h->store_stride, h->store_stride, P.val_base,
                  h->d_witptr + G.begin, h->d_planinst + G.begin, h->d_status, G.chunk * E, 0, h->expand_cs};
    CU(cudaEventRecord(G.t0, h->s_exp));
    // launch 1: KeccakfRound tiles, tile-major (each CTA's tables are staged in shared memory);
    // launch 2: code tiles, INSTANCE-major, so that a tile's code stream is fetched from DRAM once and
    // served from L2 to the other witnesses of the group
    // codes_overlap: the code-tile kernel (latency-bound gathers) runs on a second stream NEXT TO the round kernel (bandwidth-bound)
    // instead of after it; 1 = round kernel launched first, 2 = code kernel launched first
    const uint32_t n_round = h->n_round_tiles, n_code = (uint32_t)P.tiles.size() - n_round;
    const bool fork = h->codes_overlap && n_round && n_code;
    cudaStream_t s_codes = fork ? h->s_exp2 : h->s_exp;
    auto launch_codes = [&]() {
        xa.tile0 = n_round;
        if (h->codes_ug == 8) k_expand_codes<8><<<dim3(gc, n_code), 256, h->codes_dyn_smem, s_codes>>>(xa);
        else k_expand_codes<4><<<dim3(gc, n_code), 256, h->codes_dyn_smem, s_codes>>>(xa);
        B.T.other_launches++;
    };
    if (fork) { CU(cudaEventRecord(h->ev_fork, h->s_exp)); CU(cudaStreamWaitEvent(h->s_exp2, h->ev_fork, 0)); if (h->codes_overlap == 2) launch_codes(); }
    if (n_round) {
        xa.tile0 = 0;
        if (h->round_threads == 128) k_expand_round<128><<<dim3(n_round, gc), 128, h->round_dyn_smem, h->s_exp>>>(xa);
        else if (h->round_threads == 512) k_expand_round<512><<<dim3(n_round, gc), 512, h->round_dyn_smem, h->s_exp>>>(xa);
        else if (h->round_threads == 1024) k_expand_round<1024><<<dim3(n_round, gc), 1024, h->round_dyn_smem, h->s_exp>>>(xa);
        else k_expand_round<256><<<dim3(n_round, gc), 256, h->round_dyn_smem, h->s_exp>>>(xa);
    }
    if (n_code && !(fork && h->codes_overlap == 2)) launch_codes();
    if (fork) { CU(cudaEventRecord(h->ev_join, h->s_exp2)); CU(cudaStreamWaitEvent(h->s_exp, h->ev_join, 0)); }
    CU(cudaEventRecord(G.t1, h->s_exp));
    B.T.expand_launches++;
    if (B.digest) for (uint32_t k = G.begin; k < G.end; k++) {     // built-in on-GPU consumer: reads every entry of the witness once
        k_digest<<<1184, 256, 0, h->s_exp>>>(h->slots[B.slot[k]], P.n_signals, h->d_digests + B.plan[k], h->d_status + B.plan[k]);
        B.T.other_launches++;
    }
    if (!B.async) for (uint32_t k = G.begin; k < G.end; k++) B.st[k] = 2;   // synchronous batch: consumed by the digest (same stream) or dropped on request
    if (g + 1 == B.chunk_gend[G.chunk]) {
        CU(cudaEventRecord(h->ev_exp_done[r], h->s_exp));
        if (h->serialize) CU(cudaStreamWaitEvent(h->s_eval, h->ev_exp_done[r], 0));
    }
}

static bool group_slots_free(const pob_handle *h, uint32_t g) {
    const pob_handle::Batch &B = h->B; const uint32_t ns = (uint32_t)h->slots.size();
    for (uint32_t k = B.groups[g].begin; k < B.groups[g].end; k++) if (k >= ns && B.st[k - ns] != 2) return false;
    return true;
}
// queue as much work as the store ring and the witness slots allow
static void advance(pob_handle *h) {
    pob_handle::Batch &B = h->B; const uint32_t R = pob_handle::RING, ng = (uint32_t)B.groups.size();
    for (;;) {
        bool progressed = false;
        if (B.next_eval < B.nchunks && (B.next_eval < R || B.next_group >= B.chunk_gend[B.next_eval - R])) { enqueue_eval(h, B.next_eval++); progressed = true; }
        if (B.next_group < ng && B.groups[B.next_group].chunk < B.next_eval && group_slots_free(h, B.next_group)) { enqueue_group(h, B.next_group++); progressed = true; }
        if (!progressed) break;
    }
    CU(cudaGetLastError());
}

static int begin_batch(pob_handle *h, const uint64_t *inputs, uint32_t n, uint32_t flags, const uint32_t *retain, uint32_t n_retain, bool async, const char *who) {
    const bool staged = (flags & POB_RUN_INPUTS_STAGED) != 0, digest = (flags & POB_RUN_DIGEST) != 0;
    const bool expand = async || (flags & (POB_RUN_EXPAND | POB_RUN_DIGEST)) != 0 || retain != nullptr;
    if (h->B.active) return fail(POB_E_BUSY, std::string(who) + ": a batch is in flight on this handle (pob_finish it first)");
    if (staged ? (h->n_staged < n) : (inputs == nullptr && h->P.n_inputs)) return fail(POB_E_BAD_ARG, std::string(who) + ": no inputs");
    const uint32_t ns = (uint32_t)h->slots.size();
    if (retain) {
        if (n_retain > ns) return fail(POB_E_RANGE, std::string(who) + ": more retained instances than witness slots");
        for (uint32_t k = 0; k < n_retain; k++) if (retain[k] >= n || (k && retain[k] <= retain[k - 1])) return fail(POB_E_BAD_ARG, std::string(who) + ": retain[] must be strictly ascending instance indices");
    } else if (expand && !async && n > ns && !(flags & (POB_RUN_DIGEST | POB_RUN_DISCARD)))
        return fail(POB_E_RANGE, std::string(who) + ": n exceeds the resident witness slots; earlier witnesses would be overwritten unread -- use pob_submit/pob_acquire/pob_release, a retain list, POB_RUN_DIGEST or POB_RUN_DISCARD");
    CU(cudaSetDevice(h->device));
    ensure_batch_buffers(h, n);
    pob_handle::Batch &B = h->B;
    B = pob_handle::Batch();
    B.async = async; B.staged = staged; B.expand = expand; B.digest = digest; B.inputs = inputs; B.n = n;
    const uint32_t E = h->chunk;
    B.nchunks = (n + E - 1) / E;
    // with a consumer in the loop two groups must fit the slot ring, else generation and consumption cannot overlap
    const uint32_t X = async ? std::max<uint32_t>(1, std::min(h->xgroup, ns / 2 ? ns / 2 : 1)) : h->xgroup;
    if (expand) {
        if (retain) B.plan.assign(retain, retain + n_retain);
        else { B.plan.resize(n); for (uint32_t i = 0; i < n; i++) B.plan[i] = i; }
    }
    const uint32_t np = (uint32_t)B.plan.size();
    B.slot.resize(np); B.st.assign(np, 0); B.group_of.resize(np);
    for (uint32_t k = 0; k < np; k++) { B.slot[k] = k % ns; h->h_witptr[k] = h->slots[B.slot[k]]; h->h_planinst[k] = B.plan[k]; }
    h->ev_used = 0;
    B.chunk_gend.assign(B.nchunks, 0);
    for (uint32_t k = 0; k < np;) {
        const uint32_t c = B.plan[k] / E; uint32_t e = k;
        while (e < np && e - k < X && B.plan[e] / E == c) e++;
        for (uint32_t j = k; j < e; j++) B.group_of[j] = (uint32_t)B.groups.size();
        B.groups.push_back(pob_handle::Group{k, e, c, pool_event(h), pool_event(h)});
        B.chunk_gend[c] = (uint32_t)B.groups.size();
        k = e;
    }
    for (uint32_t c = 1; c < B.nchunks; c++) B.chunk_gend[c] = std::max(B.chunk_gend[c], B.chunk_gend[c - 1]);
    B.e0.resize(B.nchunks); B.e1.resize(B.nchunks); B.est.resize(B.nchunks);
    for (uint32_t c = 0; c < B.nchunks; c++) { B.e0[c] = pool_event(h); B.e1[c] = pool_event(h); B.est[c] = pool_event(h); }
    // the previous batch's residency ends here: its slots are about to be reused
    std::fill(h->slot_owner.begin(), h->slot_owner.end(), (int64_t)-1);
    std::fill(h->slot_rel_pending.begin(), h->slot_rel_pending.end(), (uint8_t)0);
    h->last_n = 0; h->last_status.clear();
    CU(cudaEventRecord(h->ev_start, h->s_eval));
    if (np) {
        CU(cudaMemcpyAsync(h->d_witptr, h->h_witptr, (size_t)np * sizeof(uint64_t *), cudaMemcpyHostToDevice, h->s_eval));
        CU(cudaMemcpyAsync(h->d_planinst, h->h_planinst, (size_t)np * 4, cudaMemcpyHostToDevice, h->s_eval));
    }
    if (digest) CU(cudaMemsetAsync(h->d_digests, 0, (size_t)n * 8, h->s_eval));
    CU(cudaEventRecord(h->ev_tmp, h->s_eval));
    CU(cudaStreamWaitEvent(h->s_h2d, h->ev_tmp, 0));
    B.active = true;
    advance(h);
    return POB_OK;
}

static int finish_batch(pob_handle *h, uint32_t *status, uint64_t *outputs, uint64_t *digests) {
    pob_handle::Batch &B = h->B; const Program &P = h->P;
    const uint32_t n = B.n; const size_t no = std::max<uint32_t>(1, P.n_outputs);
    for (auto &s : B.st) s = 2;                            // whatever the consumer did not take is generated and dropped
    advance(h);
    if (B.next_eval != B.nchunks || B.next_group != B.groups.size()) throw std::runtime_error("internal: batch did not drain");
    CU(cudaEventRecord(h->ev_tmp, h->s_eval));
    CU(cudaStreamWaitEvent(h->s_exp, h->ev_tmp, 0));
    if (B.digest) { CU(cudaMemcpyAsync(h->h_digests, h->d_digests, (size_t)n * 8, cudaMemcpyDeviceToHost, h->s_exp)); B.T.d2h_bytes += (uint64_t)n * 8; }
    CU(cudaEventRecord(h->ev_end, h->s_exp));
    CU(cudaStreamSynchronize(h->s_exp)); CU(cudaStreamSynchronize(h->s_eval)); CU(cudaStreamSynchronize(h->s_h2d));
    CU(cudaGetLastError());
    if (status) memcpy(status, h->h_status, (size_t)n * 4);
    if (outputs && P.n_outputs) memcpy(outputs, h->h_outputs, (size_t)n * no * 32);
    if (B.digest && digests) memcpy(digests, h->h_digests, (size_t)n * 8);
    pob_timing &T = B.T;
    CU(cudaEventElapsedTime(&T.total_ms, h->ev_start, h->ev_end));
    for (uint32_t c = 0; c < B.nchunks; c++) { float ms = 0; CU(cudaEventElapsedTime(&ms, B.e0[c], B.e1[c])); T.eval_ms += ms; }
    for (auto &G : B.groups) { float ms = 0; CU(cudaEventElapsedTime(&ms, G.t0, G.t1)); T.expand_ms += ms; }
    if (h->d_prof) {
        std::vector<long long> st(P.levels.size() + 3);
        CU(cudaMemcpy(st.data(), h->d_prof, st.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        if (FILE *f = fopen(h->prof_path.c_str(), "w")) {
            for (size_t l = 0; l + 1 < st.size(); l++) {
                if (l < P.levels.size()) fprintf(f, "level %zu ops %u absorbs %u poseidons %u cycles %lld\n", l, P.levels[l].t_end - P.levels[l].t_begin, P.levels[l].w_end - P.levels[l].w_begin, P.levels[l].p_end - P.levels[l].p_begin, st[l + 1] - st[l]);
                else if (l == P.levels.size()) fprintf(f, "inverse-batch(table) ops %u cycles %lld\n", P.ginv_begin - P.inv_begin, st[l + 1] - st[l]);
                else fprintf(f, "inverse-batch(generic) ops %u cycles %lld\n", P.inv_end - P.ginv_begin, st[l + 1] - st[l]);
            }
            fclose(f);
        }
    }
    h->timing = T; h->last_n = n; h->last_status.assign(h->h_status, h->h_status + n);
    B.active = false;
    return POB_OK;
}
// a failure inside a batch leaves streams in an unknown state: drop the batch, keep the handle usable
static void abort_batch(pob_handle *h) {
    cudaDeviceSynchronize(); cudaGetLastError();
    h->B.active = false; h->last_n = 0; h->last_status.clear();
    std::fill(h->slot_owner.begin(), h->slot_owner.end(), (int64_t)-1);
}

extern "C" {

const char *pob_last_error(void) { return g_err.c_str(); }
const char *pob_version(void) {
#ifdef POB_TUNING
    return "pob_b200 0.2 (sm_100a, TUNING build)";
#else
    return "pob_b200 0.2 (sm_100a)";
#endif
}

const char *pob_input_schema(const char *main_name, int *nparams) {
    if (!main_name) return nullptr;
    return main_input_schema(main_name, nparams);
}

int pob_layout_info(const char *main_name, const uint64_t *params, int nparams, int hcreate, pob_desc *out) {
    if (!main_name || !out || (nparams > 0 && !params)) return fail(POB_E_BAD_ARG, "pob_layout_info: null argument");
    try { Program P = compile_circuit(main_name, params_vec(params, nparams), flag_hcreate(hcreate), false, flag_opt(hcreate)); fill_desc(P, out); }
    catch (const std::exception &e) { return fail(POB_E_COMPILE, e.what()); }
    return POB_OK;
}

int pob_write_components(const char *main_name, const uint64_t *params, int nparams, int hcreate, const char *path, uint64_t *n_components) {
    if (!main_name || !path || (nparams > 0 && !params)) return fail(POB_E_BAD_ARG, "pob_write_components: null argument");
    try { uint64_t n = write_components(main_name, params_vec(params, nparams), flag_hcreate(hcreate), path); if (n_components) *n_components = n; }
    catch (const std::exception &e) { return fail(POB_E_COMPILE, e.what()); }
    return POB_OK;
}

void pob_destroy(pob_handle *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    delete h->exporter; h->exporter = nullptr;
    for (void *p : h->cons.allocs) cudaFree(p);
    if (h->s_eval) cudaStreamSynchronize(h->s_eval);
    if (h->s_exp2) cudaStreamSynchronize(h->s_exp2);
    if (h->s_exp) cudaStreamSynchronize(h->s_exp);
    if (h->s_h2d) cudaStreamSynchronize(h->s_h2d);
    for (void *p : {(void *)h->d_ops, (void *)h->d_psums, (void *)h->d_pos, (void *)h->d_pos_konst, (void *)h->d_abs, (void *)h->d_levels, (void *)h->d_aux, (void *)h->d_konst, (void *)h->d_codes,
                    (void *)h->d_tiles, (void *)h->d_invtab, (void *)h->d_round_desc, (void *)h->d_stores, (void *)h->d_inputs, (void *)h->d_status,
                    (void *)h->d_outputs, (void *)h->d_digests, (void *)h->d_witptr, (void *)h->d_planinst, (void *)h->d_staged, (void *)h->d_prof, (void *)h->d_block_base})
        if (p) cudaFree(p);
    slots_free(h);
    for (void *p : {(void *)h->h_status, (void *)h->h_outputs, (void *)h->h_digests, (void *)h->h_witptr, (void *)h->h_planinst}) if (p) cudaFreeHost(p);
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    for (cudaEvent_t e : h->slot_rel_ev) cudaEventDestroy(e);
    for (uint32_t r = 0; r < pob_handle::RING; r++) {
        if (h->ev_eval_done[r]) cudaEventDestroy(h->ev_eval_done[r]);
        if (h->ev_exp_done[r]) cudaEventDestroy(h->ev_exp_done[r]);
        if (h->ev_h2d[r]) cudaEventDestroy(h->ev_h2d[r]);
    }
    for (cudaEvent_t e : {h->ev_start, h->ev_end, h->ev_tmp, h->ev_fork, h->ev_join}) if (e) cudaEventDestroy(e);
    for (cudaStream_t s : {h->s_h2d, h->s_eval, h->s_exp, h->s_exp2}) if (s) cudaStreamDestroy(s);
    delete h;
}

int pob_create(const char *main_name, const uint64_t *params, int nparams, int hcreate, int device, uint32_t max_slots, pob_handle **out) {
    if (!main_name || !out || (nparams > 0 && !params)) return fail(POB_E_BAD_ARG, "pob_create: null argument");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(POB_E_NO_DEVICE, "pob_create: no CUDA device (this library has no CPU path)");
    if (device < 0 || device >= ndev) return fail(POB_E_NO_DEVICE, "pob_create: device index out of range");
    pob_handle *h = new pob_handle(); h->device = device;
    try { h->P = compile_circuit(main_name, params_vec(params, nparams), flag_hcreate(hcreate), false, flag_opt(hcreate)); }
    catch (const std::exception &e) { delete h; return fail(POB_E_COMPILE, e.what()); }
    try {
        const Program &P = h->P;
        CU(cudaSetDevice(device));
        h->d_ops = upload(P.ops); h->d_psums = upload(P.psums); h->d_pos = upload(P.poseidons); h->d_pos_konst = upload(P.pos_konst); h->d_abs = upload(P.absorbs); h->d_levels = upload(P.levels); h->d_aux = upload(P.aux);
        h->pos_konst_bytes = (uint32_t)(P.pos_konst.size() * sizeof(Fr)); h->levels_bytes = (uint32_t)(std::max<size_t>(1, P.levels.size()) * sizeof(Level));   // both multiples of 32
        h->d_konst = upload(P.konst);
        { std::vector<Code> cd = P.codes; cd.resize(cd.size() + 8, 0); h->d_codes = upload(cd); }   // + 32 bytes: TMA copies whole 16-byte units
        if (const char *v = tune_env("POB_TILE_FILTER")) {      // TUNING build only: 1 = KeccakfRound tiles only, 2 = the others only (witness incomplete!)
            std::vector<Tile> sub; for (const Tile &t : P.tiles) if ((atoi(v) == 1) == (t.pad != 0)) sub.push_back(t);
            h->P.tiles = sub;
        }
        h->d_tiles = upload(h->P.tiles);
        for (const Tile &t : h->P.tiles) if (t.pad) h->n_round_tiles++;
        { std::vector<uint64_t> bases; for (const Tile &t : P.tiles) if (t.pad && t.code_off == 0) bases.push_back(t.dst);
          std::sort(bases.begin(), bases.end()); h->n_blocks = (uint32_t)bases.size(); h->d_block_base = upload(bases); }
        h->d_invtab = upload(build_inverse_table());
        { std::vector<uint64_t> rd = P.round_desc; rd.resize(rd.size() + 2, 0); h->d_round_desc = upload(rd); }   // + 16 bytes: TMA copies whole 16-byte units
        // the small eval grid must get SMs while the expand grid (hundreds of thousands of CTAs) is draining:
        // eval runs on the highest-priority stream, expand on the lowest
        int pr_least = 0, pr_greatest = 0; CU(cudaDeviceGetStreamPriorityRange(&pr_least, &pr_greatest));
        CU(cudaStreamCreateWithPriority(&h->s_eval, cudaStreamNonBlocking, pr_greatest));
        CU(cudaStreamCreateWithPriority(&h->s_h2d, cudaStreamNonBlocking, pr_greatest));
        CU(cudaStreamCreateWithPriority(&h->s_exp, cudaStreamNonBlocking, pr_least));
        CU(cudaStreamCreateWithPriority(&h->s_exp2, cudaStreamNonBlocking, pr_least));
        for (uint32_t r = 0; r < pob_handle::RING; r++) {
            CU(cudaEventCreateWithFlags(&h->ev_eval_done[r], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&h->ev_exp_done[r], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&h->ev_h2d[r], cudaEventDisableTiming));
        }
        CU(cudaEventCreate(&h->ev_start)); CU(cudaEventCreate(&h->ev_end)); CU(cudaEventCreateWithFlags(&h->ev_tmp, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming)); CU(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
        // (an L2 persisting access-policy window for the code stream was tried and REDUCED the expand kernel to 4.9 TB/s: the
        // carve-out takes L2 away from write combining -- profiles/r01_expand_sweep.md)
        if (const char *v = tune_env("POB_EVAL_PROFILE")) { h->prof_path = v; CU(cudaMalloc(&h->d_prof, (P.levels.size() + 3) * sizeof(long long))); }
        // witness slots: as many as fit in 80 % of free HBM after the store ring
        size_t free_b = 0, total_b = 0; CU(cudaMemGetInfo(&free_b, &total_b));
        CUdevice cu_dev = 0; int compressible = 0;
        CUD(drv().device_get(&cu_dev, device));
        CUD(drv().device_attr(&compressible, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, cu_dev));
        // the reduced witness measured slower into compressible slots (expand 5.41 against 6.30 TB/s, profiles/r03b_slots_ab.log)
        if (P.opt_level) compressible = 0;
        if (const char *v = tune_env("POB_PLAIN_SLOTS")) if (atoi(v) != 0) compressible = 0;
        h->round_dyn_smem = compressible ? 0 : 85 * 1024;
        const uint64_t wbytes = slot_bytes(device, 32ull * P.n_signals);
        h->store_stride = std::max<uint64_t>(32, (P.store_u64() + 31) & ~31ull);     // never 0 (constant-only gadgets such as EIP7503())
        // eval chunk: enough instances per launch to keep the SMs busy on small circuits, bounded by a ~0.5 GB store ring
        // half (main_proof_of_burn: 32; Spend: 1024)
        uint32_t chunk = (uint32_t)std::min<uint64_t>(1024, std::max<uint64_t>(32, (512ull << 20) / (h->store_stride * 8)));
        // the reduced witness is ~10x smaller, so the eval kernel must cover all SMs to keep up with the expand kernels:
        // one wave of one-CTA-per-SM instances (store ring 2 x 128 x 22.7 MB for the main shape)
        if (P.opt_level) chunk = std::max<uint32_t>(chunk, 128);
        chunk -= chunk % 32;
        if (const char *v = tune_env("POB_EVAL_CHUNK")) chunk = (uint32_t)std::max(1, atoi(v));
        const uint64_t ring_bytes_per_inst = pob_handle::RING * (h->store_stride * 8 + (uint64_t)P.n_inputs * 32);
        uint64_t budget = (uint64_t)(free_b * 0.8);
        uint64_t nslots = budget > chunk * ring_bytes_per_inst ? (budget - chunk * ring_bytes_per_inst) / wbytes : 0;
        if (max_slots && nslots > max_slots) nslots = max_slots;
        if (nslots > 4096) nslots = 4096;
        if (nslots == 0) throw std::runtime_error("not even one witness slot fits in free HBM");
        // expand group: ~100 GB of witness per launch pair (main_proof_of_burn: 16 witnesses; Spend: up to the whole chunk)
        h->xgroup = (uint32_t)std::min<uint64_t>(std::min<uint64_t>(nslots, chunk), std::max<uint64_t>(16, (100ull << 30) / wbytes));
        if (const char *v = tune_env("POB_EVAL_THREADS")) h->eval_threads = atoi(v);
        if (const char *v = tune_env("POB_EVAL_CLUSTER")) h->eval_cluster = (uint32_t)std::max(0, std::min(8, atoi(v)));
        if (const char *v = tune_env("POB_EVAL_PREFETCH")) h->eval_prefetch = (uint32_t)(atoi(v) != 0);
        if (const char *v = tune_env("POB_SKIP_EVAL")) h->skip_eval = atoi(v) != 0;
        if (const char *v = tune_env("POB_EXPAND_CS")) h->expand_cs = (uint32_t)(atoi(v) != 0);
        if (const char *v = tune_env("POB_EVAL_L2_MB")) h->eval_l2_mb = (uint32_t)std::max(0, atoi(v));
        if (h->eval_threads != 256 && h->eval_threads != 512) h->eval_threads = 1024;
        h->eval_smem = h->pos_konst_bytes + h->levels_bytes + INV_WORKERS * INV_PARK_WORDS * 4u;   // + the parked inversion state of 256 workers (33 KB)
        if (h->eval_smem > 200 * 1024) throw std::runtime_error("the Poseidon constant table, the level table and the parked inversions do not fit in shared memory");
        CU(cudaFuncSetAttribute(k_eval<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->eval_smem));
        CU(cudaFuncSetAttribute(k_eval<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->eval_smem));
        CU(cudaFuncSetAttribute(k_eval<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->eval_smem));
        if (const char *v = tune_env("POB_SERIALIZE")) h->serialize = atoi(v) != 0;
        if (const char *v = tune_env("POB_EXPAND_SMEM_KB")) h->round_dyn_smem = (uint32_t)atoi(v) * 1024u;
        if (const char *v = tune_env("POB_EXPAND_THREADS")) h->round_threads = (uint32_t)atoi(v);
        if (const char *v = tune_env("POB_CODES_UG")) h->codes_ug = (uint32_t)atoi(v);
        if (const char *v = tune_env("POB_CODES_OVERLAP")) h->codes_overlap = (uint32_t)atoi(v);
        if (const char *v = tune_env("POB_CODES_SMEM_KB")) { h->codes_dyn_smem = (uint32_t)atoi(v) * 1024u; if (h->codes_dyn_smem > 48 * 1024) { CU(cudaFuncSetAttribute(k_expand_codes<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->codes_dyn_smem)); CU(cudaFuncSetAttribute(k_expand_codes<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->codes_dyn_smem)); } }
        if (h->round_dyn_smem > 48 * 1024) {
            CU(cudaFuncSetAttribute(k_expand_round<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->round_dyn_smem));
            CU(cudaFuncSetAttribute(k_expand_round<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->round_dyn_smem));
            CU(cudaFuncSetAttribute(k_expand_round<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->round_dyn_smem));
            CU(cudaFuncSetAttribute(k_expand_round<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->round_dyn_smem));
        }
        if (const char *v = tune_env("POB_EXPAND_GROUP")) h->xgroup = (uint32_t)std::max(1, std::min<int>(atoi(v), (int)std::min<uint64_t>(nslots, chunk)));
        h->chunk = chunk;
        CU(cudaMalloc(&h->d_stores, (size_t)pob_handle::RING * chunk * h->store_stride * 8));
        CU(cudaMalloc(&h->d_inputs, std::max<size_t>(32, (size_t)pob_handle::RING * chunk * P.n_inputs * 32)));
        for (uint64_t s = 0; s < nslots; s++) slot_alloc(h, wbytes, compressible != 0);
        if (h->eval_l2_mb) {       // tuning: keep (part of) the store ring persisting in L2 for the kernels of the eval stream
            const size_t ring = (size_t)pob_handle::RING * chunk * h->store_stride * 8, carve = (size_t)h->eval_l2_mb << 20;
            CU(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve));
            cudaDeviceProp prop; CU(cudaGetDeviceProperties(&prop, device));
            cudaStreamAttrValue av{};
            av.accessPolicyWindow.base_ptr = h->d_stores;
            av.accessPolicyWindow.num_bytes = std::min<size_t>(ring, (size_t)prop.accessPolicyMaxWindowSize);
            av.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)carve / (double)av.accessPolicyWindow.num_bytes);
            av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting; av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
            CU(cudaStreamSetAttribute(h->s_eval, cudaStreamAttributeAccessPolicyWindow, &av));
        }
        h->slot_owner.assign(nslots, -1); h->slot_rel_pending.assign(nslots, 0);
        for (uint64_t s = 0; s < nslots; s++) { cudaEvent_t e; CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); h->slot_rel_ev.push_back(e); }
    } catch (const std::exception &e) {
        std::string m = e.what(); pob_destroy(h);
        return fail(m.find("slot") != std::string::npos ? POB_E_NO_MEMORY : POB_E_CUDA, "pob_create: " + m);
    }
    *out = h; return POB_OK;
}

int pob_witness_map(const pob_handle *h, uint32_t *map) {
    if (!h || !map) return fail(POB_E_BAD_ARG, "pob_witness_map: null argument");
    if (!h->P.opt_level) return fail(POB_E_BAD_ARG, "pob_witness_map: the handle produces the full --O0 witness (identity map)");
    memcpy(map, h->P.witness_map.data(), h->P.witness_map.size() * 4);
    return POB_OK;
}

int pob_describe(const pob_handle *h, pob_desc *out) {
    if (!h || !out) return fail(POB_E_BAD_ARG, "pob_describe: null argument");
    fill_desc(h->P, out); out->n_slots = (uint32_t)h->slots.size(); out->chunk = h->chunk; out->expand_group = h->xgroup; return POB_OK;
}

void *pob_alloc_pinned(uint64_t bytes) { void *p = nullptr; if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { g_err = "cudaMallocHost failed"; return nullptr; } return p; }
void pob_free_pinned(void *p) { if (p) cudaFreeHost(p); }

int pob_stage_inputs(pob_handle *h, const uint64_t *inputs, uint32_t n) {
    if (!h || !inputs || n == 0) return fail(POB_E_BAD_ARG, "pob_stage_inputs: bad argument");
    if (h->B.active) return fail(POB_E_BUSY, "pob_stage_inputs: a batch is in flight");
    try {
        CU(cudaSetDevice(h->device));
        if (h->d_staged) { cudaFree(h->d_staged); h->d_staged = nullptr; h->n_staged = 0; }
        size_t bytes = std::max<size_t>(32, (size_t)n * h->P.n_inputs * 32);
        CU(cudaMalloc(&h->d_staged, bytes));
        if (h->P.n_inputs) CU(cudaMemcpy(h->d_staged, inputs, (size_t)n * h->P.n_inputs * 32, cudaMemcpyHostToDevice));
        h->n_staged = n;
    } catch (const std::exception &e) { return fail(POB_E_CUDA, e.what()); }
    return POB_OK;
}

static int run_batch_impl(pob_handle *h, const uint64_t *inputs, uint32_t n, uint32_t flags, const uint32_t *retain, uint32_t n_retain,
                          uint32_t *status, uint64_t *outputs, uint64_t *digests, const char *who) {
    if (!h || n == 0 || !status) return fail(POB_E_BAD_ARG, std::string(who) + ": bad argument");
    if ((flags & POB_RUN_DIGEST) && !digests) return fail(POB_E_BAD_ARG, std::string(who) + ": POB_RUN_DIGEST needs a digests array");
    try {
        int rc = begin_batch(h, inputs, n, flags, retain, n_retain, false, who);
        if (rc) return rc;
        return finish_batch(h, status, outputs, digests);
    } catch (const std::exception &e) { abort_batch(h); return fail(POB_E_CUDA, std::string(who) + ": " + e.what()); }
}
int pob_run_batch(pob_handle *h, const uint64_t *inputs, uint32_t n, uint32_t flags, uint32_t *status, uint64_t *outputs, uint64_t *digests) {
    return run_batch_impl(h, inputs, n, flags, nullptr, 0, status, outputs, digests, "pob_run_batch");
}
int pob_run_batch_retain(pob_handle *h, const uint64_t *inputs, uint32_t n, uint32_t flags, const uint32_t *retain, uint32_t n_retain,
                         uint32_t *status, uint64_t *outputs, uint64_t *digests) {
    static const uint32_t none = 0;
    if (!retain && n_retain) return fail(POB_E_BAD_ARG, "pob_run_batch_retain: null retain list");
    return run_batch_impl(h, inputs, n, flags, retain ? retain : &none, n_retain, status, outputs, digests, "pob_run_batch_retain");
}

// ---- consumer-paced hand-off ------------------------------------------------------------------------------------
int pob_submit(pob_handle *h, const uint64_t *inputs, uint32_t n, uint32_t flags) {
    if (!h || n == 0) return fail(POB_E_BAD_ARG, "pob_submit: bad argument");
    try { return begin_batch(h, inputs, n, flags | POB_RUN_EXPAND, nullptr, 0, true, "pob_submit"); }
    catch (const std::exception &e) { abort_batch(h); return fail(POB_E_CUDA, std::string("pob_submit: ") + e.what()); }
}
int pob_acquire(pob_handle *h, uint32_t *index, void **dptr, void *consumer_stream) {
    if (!h || !index || !dptr) return fail(POB_E_BAD_ARG, "pob_acquire: null argument");
    pob_handle::Batch &B = h->B;
    if (!B.active || !B.async) return fail(POB_E_BAD_ARG, "pob_acquire: no submitted batch");
    try {
        CU(cudaSetDevice(h->device));
        if (B.acq_pos >= B.plan.size()) return POB_DONE;
        const uint32_t k = B.acq_pos, g = B.group_of[k], i = B.plan[k];
        advance(h);
        if (B.next_group <= g) return fail(POB_E_BUSY, "pob_acquire: every witness slot is held by the consumer; pob_release one first");
        CU(cudaEventSynchronize(B.est[i / h->chunk]));          // accept/reject of this instance (known long before its witness is complete)
        *index = i;
        if (h->h_status[i] != 0) { *dptr = nullptr; B.st[k] = 2; B.acq_pos++; advance(h); return fail(POB_E_REJECTED, "pob_acquire: the instance failed a constraint and has no witness"); }
        if (consumer_stream) CU(cudaStreamWaitEvent((cudaStream_t)consumer_stream, B.groups[g].t1, 0));
        else CU(cudaEventSynchronize(B.groups[g].t1));
        *dptr = h->slots[B.slot[k]]; B.st[k] = 1; B.acq_pos++;
        return POB_OK;
    } catch (const std::exception &e) { abort_batch(h); return fail(POB_E_CUDA, std::string("pob_acquire: ") + e.what()); }
}
int pob_release(pob_handle *h, uint32_t index, void *consumer_stream) {
    if (!h) return fail(POB_E_BAD_ARG, "pob_release: null argument");
    pob_handle::Batch &B = h->B;
    if (!B.active || !B.async) return fail(POB_E_BAD_ARG, "pob_release: no submitted batch");
    auto it = std::lower_bound(B.plan.begin(), B.plan.end(), index);
    if (it == B.plan.end() || *it != index) return fail(POB_E_RANGE, "pob_release: no such instance");
    const uint32_t k = (uint32_t)(it - B.plan.begin());
    if (B.st[k] != 1) return fail(POB_E_RANGE, "pob_release: the instance is not held by the consumer");
    try {
        CU(cudaSetDevice(h->device));
        const uint32_t s = B.slot[k];
        if (consumer_stream) { CU(cudaEventRecord(h->slot_rel_ev[s], (cudaStream_t)consumer_stream)); h->slot_rel_pending[s] = 1; }
        B.st[k] = 2; h->slot_owner[s] = -1;
        advance(h);
    } catch (const std::exception &e) { abort_batch(h); return fail(POB_E_CUDA, std::string("pob_release: ") + e.what()); }
    return POB_OK;
}
int pob_finish(pob_handle *h, uint32_t *status, uint64_t *outputs, uint64_t *digests) {
    if (!h) return fail(POB_E_BAD_ARG, "pob_finish: null argument");
    if (!h->B.active) return fail(POB_E_BAD_ARG, "pob_finish: no batch in flight");
    try { CU(cudaSetDevice(h->device)); return finish_batch(h, status, outputs, digests); }
    catch (const std::exception &e) { abort_batch(h); return fail(POB_E_CUDA, std::string("pob_finish: ") + e.what()); }
}

int pob_export_batch(pob_handle *h, const uint64_t *inputs, uint32_t n, uint32_t flags, const char *const *paths,
                     uint32_t *status, uint64_t *outputs, pob_export_stats *stats) {
    if (!h || n == 0 || !status) return fail(POB_E_BAD_ARG, "pob_export_batch: bad argument");
    const auto t0 = std::chrono::steady_clock::now();
    bool open_err = false; std::string bad_path;
    try {
        CU(cudaSetDevice(h->device));
        if (!h->exporter) h->exporter = new Exporter(h->device);
        Exporter &X = *h->exporter; X.io_err = false; const uint64_t bytes0 = X.bytes_moved;
        int rc = begin_batch(h, inputs, n, (flags & POB_RUN_INPUTS_STAGED) | POB_RUN_EXPAND, nullptr, 0, true, "pob_export_batch");
        if (rc) return rc;
        uint64_t nw = 0;
        for (;;) {
            uint32_t idx = 0; void *dptr = nullptr;
            rc = pob_acquire(h, &idx, &dptr, nullptr);
            if (rc == POB_DONE) break;
            if (rc == POB_E_REJECTED) continue;
            if (rc) { if (h->B.active) abort_batch(h); return rc; }
            int fd = -1;
            if (paths && paths[idx]) { fd = open(paths[idx], O_WRONLY | O_CREAT | O_TRUNC, 0644); if (fd < 0) { open_err = true; bad_path = paths[idx]; } }
            if (fd >= 0 || !(paths && paths[idx])) { X.send((const uint64_t *)dptr, h->P.n_signals, fd); nw++; }
            rc = pob_release(h, idx, X.cs[0]);                 // the slot is reusable once its last D2H copy has run
            if (rc) return rc;
        }
        rc = finish_batch(h, status, outputs, nullptr);
        X.drain();
        if (stats) {
            stats->witnesses = nw; stats->bytes = X.bytes_moved - bytes0 + 76 * nw;
            stats->total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
            stats->d2h_gbs = stats->total_ms > 0 ? (float)(stats->bytes / 1e6 / stats->total_ms) : 0.f;
        }
        if (open_err) return fail(POB_E_IO, "pob_export_batch: cannot open " + bad_path);
        if (X.io_err) return fail(POB_E_IO, "pob_export_batch: short write");
        return rc;
    } catch (const std::exception &e) { abort_batch(h); return fail(POB_E_CUDA, std::string("pob_export_batch: ") + e.what()); }
}

int pob_pow_grind(int device, const uint64_t start_key[4], const uint64_t reveal_amount[4], const uint64_t burn_extra_commitment[4],
                  uint32_t zero_bytes, uint64_t max_tries, uint64_t found_key[4], uint64_t *tries) {
    if (!start_key || !reveal_amount || !burn_extra_commitment || !found_key || zero_bytes > 8 || max_tries == 0)
        return fail(POB_E_BAD_ARG, "pob_pow_grind: bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return fail(POB_E_NO_DEVICE, "pob_pow_grind: no such CUDA device");
    unsigned long long *d_hit = nullptr;
    try {
        CU(cudaSetDevice(device));
        GrindArgs ga; memcpy(ga.start, start_key, 32); ga.zero_bytes = zero_bytes;
        uint8_t msg[72];                                     // bytes 32..103 of the message
        for (int i = 0; i < 32; i++) { msg[i] = (uint8_t)(reveal_amount[3 - i / 8] >> (8 * (7 - i % 8))); msg[32 + i] = (uint8_t)(burn_extra_commitment[3 - i / 8] >> (8 * (7 - i % 8))); }
        memcpy(msg + 64, "EIP-7503", 8);
        memcpy(ga.lanes_tail, msg, 72);                      // little-endian lanes of a little-endian host
        CU(cudaMalloc(&d_hit, 8));
        ga.hit = d_hit;
        const uint64_t WINDOW = 1ull << 22;
        for (uint64_t first = 0; first < max_tries; first += WINDOW) {
            unsigned long long none = ~0ull, hit = ~0ull;
            CU(cudaMemcpy(d_hit, &none, 8, cudaMemcpyHostToDevice));
            ga.first = first; ga.count = std::min<uint64_t>(WINDOW, max_tries - first);
            k_pow_grind<<<(unsigned)((ga.count + 255) / 256), 256>>>(ga);
            CU(cudaGetLastError());
            CU(cudaMemcpy(&hit, d_hit, 8, cudaMemcpyDeviceToHost));
            if (hit != ~0ull) {
                uint64_t add = first + hit, k[4] = {start_key[0], start_key[1], start_key[2], start_key[3]};
                k[0] += add; if (k[0] < add) { if (++k[1] == 0) { if (++k[2] == 0) ++k[3]; } }
                memcpy(found_key, k, 32); if (tries) *tries = add + 1;
                cudaFree(d_hit); return POB_OK;
            }
        }
        cudaFree(d_hit);
    } catch (const std::exception &e) { if (d_hit) cudaFree(d_hit); return fail(POB_E_CUDA, std::string("pob_pow_grind: ") + e.what()); }
    if (tries) *tries = max_tries;
    return fail(POB_E_RANGE, "pob_pow_grind: no key in the search window satisfies the proof-of-work check");
}

int pob_last_timing(const pob_handle *h, pob_timing *out) {
    if (!h || !out) return fail(POB_E_BAD_ARG, "pob_last_timing: null argument");
    *out = h->timing; return POB_OK;
}

// slot of a resident, ACCEPTED instance of the last finished batch (or of one the consumer currently holds)
static int resident_slot(pob_handle *h, uint32_t index, uint64_t **slot) {
    const uint32_t *st = nullptr; uint32_t n = 0;
    if (h->B.active) { st = h->h_status; n = h->B.n; } else { st = h->last_status.data(); n = h->last_n; }
    if (index >= n) return fail(POB_E_RANGE, "witness index not in the last batch");
    if (h->B.active) {
        auto it = std::lower_bound(h->B.plan.begin(), h->B.plan.end(), index);
        if (it == h->B.plan.end() || *it != index || h->B.st[(size_t)(it - h->B.plan.begin())] != 1) return fail(POB_E_RANGE, "a batch is in flight and the consumer does not hold this witness");
    }
    if (st[index] != 0) return fail(POB_E_REJECTED, "the instance failed a circuit constraint: it has no witness");
    for (size_t s = 0; s < h->slots.size(); s++) if (h->slot_owner[s] == (int64_t)index) { *slot = h->slots[s]; return POB_OK; }
    return fail(POB_E_RANGE, "witness not resident: not materialised, released, or its slot was reused by a later instance");
}

int pob_selfcheck_keccak(pob_handle *h, uint32_t index, uint64_t *n_blocks, uint64_t *n_bad) {
    if (!h || !n_blocks || !n_bad) return fail(POB_E_BAD_ARG, "pob_selfcheck_keccak: null argument");
    if (h->P.opt_level) return fail(POB_E_BAD_ARG, "pob_selfcheck_keccak: needs the --O0 witness layout");
    uint64_t *s = nullptr; int rc = resident_slot(h, index, &s); if (rc) return rc;
    unsigned long long *d_bad = nullptr, bad = 0;
    try {
        CU(cudaSetDevice(h->device));
        CU(cudaMalloc(&d_bad, 8)); CU(cudaMemset(d_bad, 0, 8));
        if (h->n_blocks) k_check_rounds<<<(h->n_blocks * 32 + 255) / 256, 256>>>(s, h->d_block_base, h->n_blocks, d_bad);
        CU(cudaGetLastError());
        CU(cudaMemcpy(&bad, d_bad, 8, cudaMemcpyDeviceToHost));
        cudaFree(d_bad);
    } catch (const std::exception &e) { if (d_bad) cudaFree(d_bad); return fail(POB_E_CUDA, std::string("pob_selfcheck_keccak: ") + e.what()); }
    *n_blocks = h->n_blocks; *n_bad = bad;
    return POB_OK;
}

int pob_constraint_info(const char *main_name, const uint64_t *params, int nparams, int hcreate, pob_check_report *out) {
    if (!main_name || !out || (nparams > 0 && !params)) return fail(POB_E_BAD_ARG, "pob_constraint_info: null argument");
    try { Program P = compile_circuit(main_name, params_vec(params, nparams), flag_hcreate(hcreate), true); cons_info(P, out); }
    catch (const std::exception &e) { return fail(POB_E_COMPILE, e.what()); }
    return POB_OK;
}

int pob_selfcheck(pob_handle *h, uint32_t index, pob_check_report *out) {
    if (!h || !out) return fail(POB_E_BAD_ARG, "pob_selfcheck: null argument");
    if (h->P.opt_level) return fail(POB_E_BAD_ARG, "pob_selfcheck: the constraint system is stated over the --O0 witness; create the handle without POB_CREATE_O1");
    uint64_t *s = nullptr; int rc = resident_slot(h, index, &s); if (rc) return rc;
    try {
        CU(cudaSetDevice(h->device));
        pob_handle::DevCons &C = h->cons;
        if (!C.ready) {
            Program Q = compile_circuit(h->P.main_name, h->P.params, h->P.hcreate, true);
            if (Q.n_signals != h->P.n_signals) throw std::runtime_error("internal: constraint compile disagrees on the witness size");
            cons_info(Q, &C.info);
            C.flat = upload_cons(h, Q.cons_flat); C.round = upload_cons(h, Q.cons_round);
            C.konst = upload(Q.cons_konst); C.allocs.push_back(C.konst);
            C.bases = upload(Q.round_block_sig); C.allocs.push_back(C.bases); C.n_blocks = (uint32_t)Q.round_block_sig.size();
            CU(cudaMalloc(&C.rep, 24)); C.allocs.push_back(C.rep);
            C.ready = true;
        }
        const unsigned long long init[3] = {0, 0, ~0ull};
        CU(cudaMemcpy(C.rep, init, 24, cudaMemcpyHostToDevice));
        cudaEvent_t e0, e1; CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
        CU(cudaEventRecord(e0, 0));
        auto grid = [](uint64_t n) { return (unsigned)std::min<uint64_t>((n + 255) / 256, 148ull * 64); };
        CheckArgs fa{C.flat, C.konst, s, nullptr, 0, 0, C.rep};
        if (C.flat.n_eq) k_check_eq<<<grid(C.flat.n_eq), 256>>>(fa);
        if (C.flat.n_kc) k_check_kc<<<grid(C.flat.n_kc), 256>>>(fa);
        if (C.flat.n_r1) k_check_r1<<<grid(C.flat.n_r1), 256>>>(fa);
        if (C.n_blocks) {
            CheckArgs ra{C.round, C.konst, s, C.bases, C.n_blocks, C.flat.n_records(), C.rep};
            k_check_eq<<<grid(C.round.n_eq * C.n_blocks), 256>>>(ra);
            k_check_kc<<<grid(C.round.n_kc * C.n_blocks), 256>>>(ra);
            k_check_r1<<<grid(C.round.n_r1 * C.n_blocks), 256>>>(ra);
        }
        CU(cudaEventRecord(e1, 0));
        CU(cudaGetLastError());
        unsigned long long rep[3];
        CU(cudaMemcpy(rep, C.rep, 24, cudaMemcpyDeviceToHost));
        *out = C.info;
        CU(cudaEventElapsedTime(&out->ms, e0, e1));
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        out->n_failed = rep[0]; out->n_hint_failed = rep[1]; out->first_failed = rep[2];
    } catch (const std::exception &e) { return fail(POB_E_CUDA, std::string("pob_selfcheck: ") + e.what()); }
    return POB_OK;
}

int pob_witness_device_ptr(pob_handle *h, uint32_t index, void **dptr) {
    if (!h || !dptr) return fail(POB_E_BAD_ARG, "pob_witness_device_ptr: null argument");
    uint64_t *s = nullptr; int rc = resident_slot(h, index, &s); if (rc) return rc;
    *dptr = s; return POB_OK;
}

int pob_copy_witness(pob_handle *h, uint32_t index, uint64_t first_signal, uint64_t n_signals, uint64_t *dst_host) {
    if (!h || !dst_host) return fail(POB_E_BAD_ARG, "pob_copy_witness: null argument");
    uint64_t *s = nullptr; int rc = resident_slot(h, index, &s); if (rc) return rc;
    const uint64_t n = h->P.n_signals;
    if (first_signal > n || n_signals > n - first_signal) return fail(POB_E_RANGE, "pob_copy_witness: range exceeds the witness");
    if (cudaSetDevice(h->device) != cudaSuccess || cudaMemcpy(dst_host, s + 4 * first_signal, (size_t)n_signals * 32, cudaMemcpyDeviceToHost) != cudaSuccess)
        return fail(POB_E_CUDA, "pob_copy_witness: cudaMemcpy failed");
    return POB_OK;
}

int pob_write_wtns(pob_handle *h, uint32_t index, const char *path) {
    if (!h || !path) return fail(POB_E_BAD_ARG, "pob_write_wtns: null argument");
    uint64_t *s = nullptr; int rc = resident_slot(h, index, &s); if (rc) return rc;
    int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) return fail(POB_E_IO, std::string("cannot open ") + path);
    try {
        CU(cudaSetDevice(h->device));
        if (!h->exporter) h->exporter = new Exporter(h->device);
        h->exporter->io_err = false;
        h->exporter->send(s, h->P.n_signals, fd);
        h->exporter->drain();
        if (h->exporter->io_err) return fail(POB_E_IO, std::string("short write to ") + path);
    } catch (const std::exception &e) { return fail(POB_E_CUDA, std::string("pob_write_wtns: ") + e.what()); }
    return POB_OK;
}

}  // extern "C"
