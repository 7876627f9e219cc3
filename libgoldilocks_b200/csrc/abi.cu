// abi.cu -- CUDA launch wrappers and the C ABI of include/goldilocks_b200.h.
//
// Host arrays -> device arena (one grow-only allocation per device) -> kernel sequence -> host.
// Everything between the first and the last kernel of a call stays in HBM.  There is NO CPU
// implementation behind these symbols: without a usable sm_100 GPU every call fails loudly.
#include <cuda_runtime.h>
#include <sys/random.h>
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <typeinfo>
#include <vector>

#include "../../include/goldilocks_b200.h"
#include "launch.cuh"
#include "staged.cuh"
#include "shard.h"
#include "coalesce.h"

// kernels live in k_*.cu
LANES_PLAIN(DECLARE_PLAIN)
STAGED_GF(DECLARE_STAGED_GF)
STAGED_PT(DECLARE_STAGED_PT)
LANES_SM(DECLARE_SM)
LANES_SMP(DECLARE_SMP)

// ------------------------------------------------------------------------------------------------
// Per-device context
// ------------------------------------------------------------------------------------------------
namespace {

thread_local std::string g_err;
std::atomic<uint64_t> g_launches{0};

struct Block { void *p; size_t cap; };
struct Ctx {
    std::mutex mu;
    bool ready = false, failed = false;
    int dev = -1, lane = 0, sms = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;   // signatures and messages of a verification cross PCIe here while the main stream groups the keys
    cudaEvent_t copy_done[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaStream_t side_stream = nullptr;   // the latency-bound doubling chain of the key class (rlc.cuh) runs here beside the R-class buckets
    cudaEvent_t side_evt[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    /* the same fork / join for the device-pointer verification (caller's stream, context lock NOT held while kernels run): its own side
     * stream and events, and a lock that covers only the enqueue, so that two threads cannot interleave record / wait pairs */
    cudaStream_t dev_side = nullptr;
    cudaEvent_t dev_evt[2] = {nullptr, nullptr};
    std::mutex dev_side_mu;
    fixed_tables *ft = nullptr;
    niels *wide = nullptr;       // WIDE_TABLES x WIDE_ENTRIES verification tables: odd multiples of 2^(18m) B (25 x 131072 x 192 B = 629 MB, algos.cuh)
    std::vector<Block> blocks;   // arena blocks; blocks.back() is the active one
    size_t used = 0;             // bytes used in the active block
    void *slot_scratch = nullptr;
    unsigned *work_counter = nullptr;   // dynamic hand-out counter of the persistent kernels (launch_smp)
    unsigned rlc_skip = 0;              // calls of the RLC entry point that go straight to the per-signature path (rlc_core)
    size_t slot_cap = 0;
};
constexpr int MAX_DEV = 64;
Ctx g_ctx[MAX_DEV][shard::LANES];   /* lane 0 serves the caller's own thread; lanes 1.. belong to the shard workers (shard.h) */

bool fail(const char *what, cudaError_t e) {
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    fprintf(stderr, "[goldilocks_b200] %s\n", g_err.c_str());
    return false;
}
#define CU(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return fail(#x, e_); } while (0)

// Optional per-launch CUDA-event timing (bench.py's roofline leg): when enabled every launch is
// bracketed by two events on its own stream; goldilocks_b200_profile_read() resolves them later.
struct ProfRec { const char *name; cudaEvent_t a, b; };
std::mutex g_prof_mu;
std::vector<ProfRec> g_prof;
std::atomic<int> g_prof_on{0};
cudaEvent_t prof_begin(const char *name, cudaStream_t s, cudaEvent_t *end) {
    cudaEvent_t a = nullptr;
    *end = nullptr;
    if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(end) != cudaSuccess) return nullptr;
    cudaEventRecord(a, s);
    (void)name;
    return a;
}
void prof_end(const char *name, cudaStream_t s, cudaEvent_t a, cudaEvent_t b) {
    if (!a || !b) return;
    cudaEventRecord(b, s);
    std::lock_guard<std::mutex> g(g_prof_mu);
    g_prof.push_back({name, a, b});
}

template <class F>
bool launch(Ctx &c, const F &f, size_t n, cudaStream_t s) {
    if (n == 0) return true;
    g_launches++;
    cudaEvent_t a = nullptr, b = nullptr;
    const bool prof = g_prof_on.load() != 0;
    if (prof) a = prof_begin(typeid(F).name(), s, &b);
    CU(launch_lanes<F>(f, n, s));
    if (prof) prof_end(typeid(F).name(), s, a, b);
    return true;
}
// The HBM-bound field / point entry points run in their shared-memory staged shape (staged.cuh); these
// overloads are more specialised than launch<F>, so every caller of launch() picks them up.
template <int OP>
bool launch(Ctx &c, const LaneGf<OP> &f, size_t n, cudaStream_t s) {
    if (n == 0) return true;
    g_launches++;
    cudaEvent_t a = nullptr, b = nullptr;
    const bool prof = g_prof_on.load() != 0;
    if (prof) a = prof_begin(typeid(StagedGf<OP>).name(), s, &b);
    const StagedGf<OP> sf = {f.out, f.status, f.a, f.b, f.w};
    CU(launch_gf_staged<OP>(sf, n, s));
    if (prof) prof_end(typeid(StagedGf<OP>).name(), s, a, b);
    return true;
}
template <int OP>
bool launch(Ctx &c, const LanePt<OP> &f, size_t n, cudaStream_t s) {
    if (n == 0) return true;
    g_launches++;
    cudaEvent_t a = nullptr, b = nullptr;
    const bool prof = g_prof_on.load() != 0;
    if constexpr (OP == PTOP_ADD || OP == PTOP_SUB || OP == PTOP_DBL) {
        if (prof) a = prof_begin(typeid(StagedPt<OP>).name(), s, &b);
        const StagedPt<OP> sf = {f.out, f.a, f.b};
        CU(launch_pt_staged<OP>(sf, n, s));
        if (prof) prof_end(typeid(StagedPt<OP>).name(), s, a, b);
    } else {
        if (prof) a = prof_begin(typeid(LanePt<OP>).name(), s, &b);
        CU(launch_lanes<LanePt<OP>>(f, n, s));
        if (prof) prof_end(typeid(LanePt<OP>).name(), s, a, b);
    }
    return true;
}
template <class F>
bool launch_slots(Ctx &c, const F &f, size_t n, cudaStream_t s) { /* shared-memory slot machine (slots.cuh) */
    if (n == 0) return true;
    g_launches++;
    cudaEvent_t a = nullptr, b = nullptr;
    const bool prof = g_prof_on.load() != 0;
    if (prof) a = prof_begin(typeid(F).name(), s, &b);
    CU(launch_sm<F>(f, n, s));
    if (prof) prof_end(typeid(F).name(), s, a, b);
    return true;
}
// persistent slot-machine kernels: grid = SMs x resident blocks, so every thread owns one scratch area
template <class F>
bool smp_grid(Ctx &c, int *grid) {
    int occ = 0;
    CU(sm_configure<F>(&occ)); /* also sets the dynamic shared-memory attributes on this device */
    if (occ < 1) { g_err = "slot-machine kernel does not fit on an SM"; return false; }
    *grid = c.sms * occ;
    return true;
}
// `counter`: a zeroed device word for the kernel's dynamic hand-out.  Null = the context's own word, zeroed here on `s`
// (host-pointer calls hold the context lock until their stream has drained, so one launch uses it at a time);
// GRID_STRIDE = no counter, fixed assignment (device-pointer calls on caller streams that bring no word of their own).
unsigned *const GRID_STRIDE = reinterpret_cast<unsigned *>(1);
template <class F>
bool launch_smp(Ctx &c, const F &f, size_t n, int grid, cudaStream_t s, unsigned *counter = nullptr) {
    if (n == 0) return true;
    if (counter == GRID_STRIDE) counter = nullptr;
    else if (!counter) {
        counter = c.work_counter;
        CU(cudaMemsetAsync(counter, 0, sizeof(unsigned), s));
    }
    size_t need_blocks = (n + SLOT_BLOCK - 1) / SLOT_BLOCK;
    if ((size_t)grid > need_blocks) grid = (int)need_blocks;
    g_launches++;
    cudaEvent_t a = nullptr, b = nullptr;
    const bool prof = g_prof_on.load() != 0;
    if (prof) a = prof_begin(typeid(F).name(), s, &b);
    CU(launch_sm_persist<F>(f, n, grid, s, counter));
    if (prof) prof_end(typeid(F).name(), s, a, b);
    return true;
}
bool ctx_init(Ctx &c, int dev, int lane = 0) {
    if (c.ready) return true;
    if (c.failed) { g_err = "device initialisation failed earlier"; return false; }
    if (lane > 0) { /* the read-only tables are built once per device, by lane 0 */
        Ctx &c0 = g_ctx[dev][0];
        std::lock_guard<std::mutex> g0(c0.mu);
        if (!ctx_init(c0, dev, 0)) return false;
    }
    c.failed = true;
    cudaDeviceProp p;
    CU(cudaGetDeviceProperties(&p, dev));
    if (p.major < 10) {
        g_err = "goldilocks_b200 needs an sm_100-class GPU (found sm_" + std::to_string(p.major) + std::to_string(p.minor) + ")";
        fprintf(stderr, "[goldilocks_b200] %s\n", g_err.c_str());
        return false;
    }
    c.dev = dev;
    c.lane = lane;
    c.sms = p.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
    for (auto &e : c.copy_done) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    {   /* the side stream carries short latency-bound chains next to kernels that fill the machine: its blocks go first */
        int prio_lo = 0, prio_hi = 0;
        CU(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CU(cudaStreamCreateWithPriority(&c.side_stream, cudaStreamNonBlocking, prio_hi));
    }
    for (auto &e : c.side_evt) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CU(cudaStreamCreateWithFlags(&c.dev_side, cudaStreamNonBlocking));
    for (auto &e : c.dev_evt) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CU(cudaMalloc(&c.work_counter, 256));
    if (lane > 0) {
        c.ft = g_ctx[dev][0].ft;
        c.wide = g_ctx[dev][0].wide;
        c.failed = false;
        c.ready = true;
        return true;
    }
    CU(cudaMalloc(&c.ft, sizeof(fixed_tables)));
    LaneBuildTables f = {c.ft};
    if (!launch(c, f, TABLE_LANES, c.stream)) return false;
    CU(cudaMalloc(&c.wide, sizeof(niels) * WIDE_ENTRIES * WIDE_TABLES));
    {
        pniels *tmp = nullptr; gf *pre = nullptr;
        CU(cudaMalloc(&tmp, sizeof(pniels) * WIDE_ENTRIES * WIDE_TABLES));
        CU(cudaMalloc(&pre, sizeof(gf) * WIDE_ENTRIES * WIDE_TABLES));
        LaneBuildWide fw = {c.wide, tmp, pre, c.ft};
        if (!launch(c, fw, WIDE_LANES * WIDE_TABLES, c.stream)) return false;
        CU(cudaStreamSynchronize(c.stream));
        cudaFree(tmp); cudaFree(pre);
    }
    CU(cudaStreamSynchronize(c.stream));
    c.failed = false;
    c.ready = true;
    return true;
}

// Context lane of the calling thread: workers are bound to theirs; caller threads are dealt the lanes round-robin on their first
// call, so up to shard::LANES host threads run host-pointer calls on one GPU side by side instead of queueing on one lock.
std::atomic<unsigned> g_next_lane{0};
int my_lane() {
    if (shard::t_lane < 0) shard::t_lane = (int)(g_next_lane.fetch_add(1) % shard::LANES);
    return shard::t_lane;
}
// One API call: locks the device context, carves device buffers from the arena, copies, launches.
struct Call {
    Ctx *c = nullptr;
    std::unique_lock<std::mutex> lk;
    bool ok = false;
    Call() {
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) { fail("cudaGetDevice (is there a GPU?)", e); return; }
        if (dev >= MAX_DEV) { g_err = "device index too large"; return; }
        c = &g_ctx[dev][my_lane()];
        lk = std::unique_lock<std::mutex>(c->mu);
        ok = ctx_init(*c, dev, my_lane());
        if (ok && !c->blocks.empty()) c->used = 0;
    }
    /* device copies of secrets (private keys, scalars, nonces, window tables of the secret paths): zeroed by finish() on
     * every path out of the call, like the reference's goldilocks_bzero of its stack copies (eddsa.c:120-126,220-229) */
    std::vector<std::pair<void *, size_t>> wipes;
    template <class T> T *secret(T *dev_ptr, size_t count) {
        if (dev_ptr && count) wipes.push_back({(void *)dev_ptr, count * sizeof(T)});
        return dev_ptr;
    }
    void *alloc(size_t bytes) {
        if (!ok) return nullptr;
        bytes = (bytes + 255) & ~(size_t)255;
        if (bytes == 0) bytes = 256;
        if (c->blocks.empty() || c->used + bytes > c->blocks.back().cap) {
            size_t cap = c->blocks.empty() ? 0 : c->blocks.back().cap;
            size_t want = bytes > 2 * cap ? bytes : 2 * cap;
            if (want < (1u << 20)) want = 1u << 20;
            void *p = nullptr;
            cudaError_t e = cudaMalloc(&p, want);
            if (e != cudaSuccess) { ok = fail("cudaMalloc(arena)", e); return nullptr; }
            c->blocks.push_back({p, want});
            c->used = 0;
        }
        void *r = (char *)c->blocks.back().p + c->used;
        c->used += bytes;
        return r;
    }
    template <class T> T *in(const T *host, size_t count) {
        T *d = (T *)alloc(count * sizeof(T));
        if (!d || count == 0) return d;
        cudaError_t e = cudaMemcpyAsync(d, host, count * sizeof(T), cudaMemcpyHostToDevice, c->stream);
        if (e != cudaSuccess) { ok = fail("cudaMemcpyAsync(H2D)", e); return nullptr; }
        return d;
    }
    template <class T> T *out(size_t count) { return (T *)alloc(count * sizeof(T)); }
    // host -> device on the copy stream; `dev` was carved with out<>()
    template <class T> void push(T *dev, const T *host, size_t count) {
        if (!ok || count == 0) return;
        cudaError_t e = cudaMemcpyAsync(dev, host, count * sizeof(T), cudaMemcpyHostToDevice, c->copy_stream);
        if (e != cudaSuccess) ok = fail("cudaMemcpyAsync(H2D, copy stream)", e);
    }
    template <class T> void fetch(T *host, const T *dev, size_t count) {
        if (!ok || count == 0) return;
        cudaError_t e = cudaMemcpyAsync(host, dev, count * sizeof(T), cudaMemcpyDeviceToHost, c->stream);
        if (e != cudaSuccess) ok = fail("cudaMemcpyAsync(D2H)", e);
    }
    uint4 *slots(size_t nthreads, size_t tables_per_thread) { /* per-thread window tables (wtab, slot_algos.cuh) */
        if (!ok) return nullptr;
        size_t bytes = nthreads * tables_per_thread * WTAB_QUADS_PER_LANE * sizeof(uint4);
        if (bytes > c->slot_cap) {
            if (c->slot_scratch) cudaFree(c->slot_scratch);
            c->slot_scratch = nullptr; c->slot_cap = 0;
            cudaError_t e = cudaMalloc(&c->slot_scratch, bytes);
            if (e != cudaSuccess) { ok = fail("cudaMalloc(slot scratch)", e); return nullptr; }
            c->slot_cap = bytes;
        }
        return (uint4 *)c->slot_scratch;
    }
    template <class F> void run(const F &f, size_t n) { if (ok) ok = launch(*c, f, n, c->stream); }
    template <class F> void run_sm(const F &f, size_t n) { if (ok) ok = launch_slots(*c, f, n, c->stream); }
    template <class F> int smp_grid_for() { int g = 1; if (ok) ok = smp_grid<F>(*c, &g); return g; }
    template <class F> void run_smp(const F &f, size_t n, int grid) { if (ok) ok = launch_smp(*c, f, n, grid, c->stream); }
    goldilocks_error_t finish() {
        if (c && c->ready && lk.owns_lock()) {
            for (auto &w : wipes)
                if (cudaMemsetAsync(w.first, 0, w.second, c->stream) != cudaSuccess) ok = false;
            wipes.clear();
            cudaError_t e = cudaStreamSynchronize(c->stream);
            if (e != cudaSuccess && ok) ok = fail("cudaStreamSynchronize", e);
        }
        if (c && lk.owns_lock() && c->blocks.size() > 1) { /* coalesce into one block for the next call */
            size_t total = 0;
            for (auto &b : c->blocks) { total += b.cap; cudaFree(b.p); }
            c->blocks.clear();
            void *p = nullptr;
            if (cudaMalloc(&p, total) == cudaSuccess) c->blocks.push_back({p, total});
            c->used = 0;
        }
        return ok ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
    }
};

typedef goldilocks_448_point_s hpt;
typedef goldilocks_448_scalar_s hsc;
inline const abi_pt *P(const hpt *p) { return (const abi_pt *)p; }
inline abi_pt *P(hpt *p) { return (abi_pt *)p; }
inline const abi_sc *S(const hsc *p) { return (const abi_sc *)p; }
inline abi_sc *S(hsc *p) { return (abi_sc *)p; }
static_assert(sizeof(hpt) == sizeof(abi_pt) && sizeof(hsc) == sizeof(abi_sc), "ABI layout");
static_assert(sizeof(niels) == 192 && sizeof(pniels) == 256, "table layout");
static_assert(15 * WINDOW_NTABLE * 16 * 4 <= KTAB_QUADS * 9 && 30 * WINDOW_NTABLE * 16 * 4 <= KTAB_QUADS * 32 && 90 * WINDOW_NTABLE * 16 * 4 <= KTAB_QUADS * 256,
              "every column shape of vsh_pick (taken from 9 / 32 / 256 signatures per table on) must fit the buffer sized for n/4 + 1 tables of KTAB_QUADS");
/* work items of the column kernel: ten per table of the narrow shape (at most n/4 + 1 tables), 15 per table for at most n/9 tables, ... */
static size_t verify_column_items(size_t n) { return std::max((n / 4 + 1) * VSH_CHUNKS, n * VSH_MAX_CHUNKS_PER_SIG_NUM / VSH_MAX_CHUNKS_PER_SIG_DEN + 90); }
static_assert(sizeof(verify_aux) == sizeof(abi_pt), "the aux record of a signature lives in the R half of its point pair");

cudaStream_t as_stream(void *s) { return (cudaStream_t)s; }

// ---- device sets: one batch over several GPUs (shard.h) ---------------------------------------------------------
std::mutex g_pool_mu;
std::shared_ptr<shard::Pool> g_pool;                      /* null = the caller's current device only */
std::vector<shard::Worker *> g_workers[MAX_DEV];          /* created on first use, kept for the life of the process */
bool g_env_read = false;
bool pool_install(const int *devs, int n) { /* g_pool_mu held */
    if (n <= 0) { g_pool.reset(); return true; }
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count < 1) { g_err = "goldilocks_b200_set_devices: no CUDA device"; return false; }
    auto pool = std::make_shared<shard::Pool>();
    for (int i = 0; i < n; i++) {
        if (devs[i] < 0 || devs[i] >= count || devs[i] >= MAX_DEV) { g_err = "goldilocks_b200_set_devices: device index out of range"; return false; }
        pool->devs.push_back(devs[i]);
    }
    for (int d : pool->devs) {
        if (g_workers[d].empty())
            for (int l = 0; l < shard::LANES; l++) g_workers[d].push_back(new shard::Worker(d, l));
        for (auto *w : g_workers[d]) pool->workers.push_back(w);
    }
    g_pool = pool;
    return true;
}
void pool_from_env() { /* GOLDILOCKS_B200_DEVICES = "all" | "0,1,2,..." ; read once, an explicit set_devices() wins */
    if (g_env_read) return;
    g_env_read = true;
    const char *e = getenv("GOLDILOCKS_B200_DEVICES");
    if (!e || !*e) return;
    std::vector<int> devs;
    if (!strcmp(e, "all")) {
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess) return;
        for (int i = 0; i < count && i < MAX_DEV; i++) devs.push_back(i);
    } else {
        for (const char *q = e; *q;) {
            char *end = nullptr;
            long v = strtol(q, &end, 10);
            if (end == q) break;
            devs.push_back((int)v);
            q = (*end == ',') ? end + 1 : end;
            if (*end && *end != ',') break;
        }
    }
    if (!devs.empty() && !pool_install(devs.data(), (int)devs.size()))
        fprintf(stderr, "[goldilocks_b200] GOLDILOCKS_B200_DEVICES ignored: %s\n", g_err.c_str());
}
// The plan of a call, or null when it runs on the caller's device as one piece: worker threads never re-shard, a set of
// one device only pipelines the light operations.
constexpr size_t HEAVY_MIN = 2048;   /* elements per device below which a heavy batch is not cut */
std::shared_ptr<shard::Pool> shard_pool(size_t n, bool pipelined, size_t bytes_per_elem) {
    if (shard::t_worker || n < 2 * shard::MIN_CHUNK) return nullptr;
    std::shared_ptr<shard::Pool> p;
    {
        std::lock_guard<std::mutex> g(g_pool_mu);
        pool_from_env();
        p = g_pool;
    }
    if (!p) return nullptr;
    if (!pipelined && (p->devs.size() < 2 || n < 2 * HEAVY_MIN)) return nullptr;
    if (pipelined && p->devs.size() < 2 && n * bytes_per_elem < 2 * shard::CHUNK_BYTES) return nullptr;
    return p;
}
template <class Fn>
goldilocks_error_t shard_go(const std::shared_ptr<shard::Pool> &p, size_t n, bool pipelined, size_t bytes_per_elem, Fn fn) {
    std::string err;
    const int r = shard::run(p, n, HEAVY_MIN, bytes_per_elem, pipelined, &err, fn);
    if (r != -1) g_err = err;
    return r == -1 ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
// SHARD_HEAVY / SHARD_LIGHT(bytes per element) open a batch entry point: with a device set configured the call re-enters
// itself once per range on the workers (`lo` = first element, `m` = count of the range) and returns their verdict.
#define SHARD_HEAVY(n, call) \
    if (auto pool_ = shard_pool((n), false, 0)) return shard_go(pool_, (n), false, 0, [=](size_t lo, size_t m) { return (call); });
#define SHARD_LIGHT(n, bytes, call) \
    if (auto pool_ = shard_pool((n), true, (bytes))) return shard_go(pool_, (n), true, (bytes), [=](size_t lo, size_t m) { return (call); });
// offsets of messages [lo, lo + m] rebased to the first one of the range
struct SubOffsets {
    std::vector<size_t> v;
    SubOffsets(const size_t *off, size_t lo, size_t m) : v(m + 1) { for (size_t i = 0; i <= m; i++) v[i] = off[lo + i] - off[lo]; }
};
// Device-pointer entry points only need the tables; they never touch the arena or the lock while
// kernels run (the caller owns the stream ordering).
Ctx *dev_ctx() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev >= MAX_DEV) { g_err = "no CUDA device"; return nullptr; }
    Ctx &c = g_ctx[dev][my_lane()];
    std::lock_guard<std::mutex> g(c.mu);
    return ctx_init(c, dev, my_lane()) ? &c : nullptr;
}

}  // namespace

namespace shard {
thread_local bool t_worker = false;
thread_local int t_lane = -1;     /* caller threads pick a context lane on their first call (my_lane) */
const std::string &worker_error() { return g_err; }
std::shared_ptr<Pool> current() { std::lock_guard<std::mutex> g(g_pool_mu); return g_pool; }
}  // namespace shard

extern "C" {

// ---- data symbols ----------------------------------------------------------------------------------
static const int precomputed_base_tag = 448;
const goldilocks_448_precomputed_s *goldilocks_448_precomputed_base = (const goldilocks_448_precomputed_s *)&precomputed_base_tag;
const goldilocks_448_point_p goldilocks_448_point_base = {{{GOLD_CONST_BASE_X56}, {GOLD_CONST_BASE_Y56}, {{1, 0, 0, 0, 0, 0, 0, 0}}, {GOLD_CONST_BASE_T56}}};
const goldilocks_448_point_p goldilocks_448_point_identity = {{{{0}}, {{1}}, {{1}}, {{0}}}};
const goldilocks_448_scalar_p goldilocks_448_scalar_one = {{{1}}}, goldilocks_448_scalar_zero = {{{0}}};
const uint8_t goldilocks_x448_base_point[GOLDILOCKS_X448_PUBLIC_BYTES] = {5};
const size_t goldilocks_448_sizeof_precomputed_s = 15360, goldilocks_448_alignof_precomputed_s = 32; /* goldilocks.c:65-66 */

// ---- control -------------------------------------------------------------------------------------------
goldilocks_error_t goldilocks_b200_init(void) { Call k; return k.finish(); }
const char *goldilocks_b200_last_error(void) { return g_err.c_str(); }
uint64_t goldilocks_b200_launch_count(void) { return g_launches.load(); }
goldilocks_error_t goldilocks_b200_set_devices(const int *devices, int count) {
    std::shared_ptr<shard::Pool> p;
    {
        std::lock_guard<std::mutex> g(g_pool_mu);
        g_env_read = true; /* an explicit set wins over GOLDILOCKS_B200_DEVICES */
        if (!pool_install(devices, count)) return GOLDILOCKS_FAILURE;
        p = g_pool;
    }
    if (!p) return GOLDILOCKS_SUCCESS;
    /* build every device's tables now (in parallel, on the workers), not inside the first timed call */
    std::string err;
    const int r = shard::run_everywhere(p, &err, [](size_t, size_t) { return (int)goldilocks_b200_init(); });
    if (r != -1) { g_err = err; return GOLDILOCKS_FAILURE; }
    return GOLDILOCKS_SUCCESS;
}
int goldilocks_b200_get_devices(int *devices, int max) {
    std::lock_guard<std::mutex> g(g_pool_mu);
    pool_from_env();
    if (!g_pool) return 0;
    const int n = (int)g_pool->devs.size();
    for (int i = 0; i < n && i < max; i++) devices[i] = g_pool->devs[i];
    return n;
}
size_t goldilocks_b200_shard_plan(size_t *lo, size_t *hi, int *device_slot, int *lane, size_t max, size_t n, int ndev, size_t bytes_per_elem, int pipelined) {
    const std::vector<shard::Piece> pl = shard::plan(n, ndev, HEAVY_MIN, bytes_per_elem, pipelined != 0);
    for (size_t i = 0; i < pl.size() && i < max; i++) {
        lo[i] = pl[i].lo; hi[i] = pl[i].hi;
        device_slot[i] = pl[i].slot / shard::LANES; lane[i] = pl[i].slot % shard::LANES;
    }
    return pl.size();
}
void goldilocks_b200_profile(int enable) {
    std::lock_guard<std::mutex> g(g_prof_mu);
    if (enable) {
        for (auto &r : g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
        g_prof.clear();
    }
    g_prof_on.store(enable ? 1 : 0);
}
size_t goldilocks_b200_profile_read(char *names, float *ms, size_t max) {
    std::lock_guard<std::mutex> g(g_prof_mu);
    size_t k = 0;
    for (auto &r : g_prof) {
        if (k >= max) break;
        float t = 0.f;
        if (cudaEventSynchronize(r.b) != cudaSuccess || cudaEventElapsedTime(&t, r.a, r.b) != cudaSuccess) t = -1.f;
        const char *nm = r.name;
        while (*nm >= '0' && *nm <= '9') nm++; /* strip the Itanium length prefix of typeid().name() */
        snprintf(names + 64 * k, 64, "%s", nm);
        ms[k] = t;
        k++;
    }
    return k;
}

size_t goldilocks_b200_profile_timeline(char *names, float *start_ms, float *end_ms, size_t max) {
    /* the same log as profile_read(), as a timeline: begin / end of every launch relative to the begin of the first one
     * (events of different streams compare), for paths that run kernels on more than one stream */
    std::lock_guard<std::mutex> g(g_prof_mu);
    size_t k = 0;
    for (auto &r : g_prof) {
        if (k >= max) break;
        float t0 = -1.f, t1 = -1.f;
        if (cudaEventSynchronize(r.b) == cudaSuccess) {
            if (cudaEventElapsedTime(&t0, g_prof[0].a, r.a) != cudaSuccess) t0 = -1.f;
            if (cudaEventElapsedTime(&t1, g_prof[0].a, r.b) != cudaSuccess) t1 = -1.f;
        }
        const char *nm = r.name;
        while (*nm >= '0' && *nm <= '9') nm++;
        snprintf(names + 64 * k, 64, "%s", nm);
        start_ms[k] = t0; end_ms[k] = t1;
        k++;
    }
    return k;
}

goldilocks_error_t goldilocks_b200_export_comb_table(uint8_t out[15360]) {
    Call k;
    if (!k.ok) return k.finish();
    std::vector<niels> h(COMB_ENTRIES);
    k.fetch(h.data(), k.c->ft->comb, COMB_ENTRIES);
    goldilocks_error_t r = k.finish();
    if (r != GOLDILOCKS_SUCCESS) return r;
    uint64_t *o = (uint64_t *)out;
    for (int e = 0; e < COMB_ENTRIES; e++) {
        const gf *g[3] = {&h[e].a, &h[e].b, &h[e].c};
        for (int j = 0; j < 3; j++)
            for (int l = 0; l < 8; l++) o[(e * 3 + j) * 8 + l] = (uint64_t)g[j]->v[2 * l] | ((uint64_t)g[j]->v[2 * l + 1] << 28);
    }
    return r;
}
goldilocks_error_t goldilocks_b200_export_wnaf_table(uint8_t out[6144]) {
    Call k;
    if (!k.ok) return k.finish();
    std::vector<niels> h(WNAF_FIXED_ENTRIES);
    k.fetch(h.data(), k.c->wide, WNAF_FIXED_ENTRIES); /* first 32 entries = 1B..63B, the reference's wNAF table */
    goldilocks_error_t r = k.finish();
    if (r != GOLDILOCKS_SUCCESS) return r;
    uint64_t *o = (uint64_t *)out;
    for (int e = 0; e < WNAF_FIXED_ENTRIES; e++) {
        const gf *g[3] = {&h[e].a, &h[e].b, &h[e].c};
        for (int j = 0; j < 3; j++)
            for (int l = 0; l < 8; l++) o[(e * 3 + j) * 8 + l] = (uint64_t)g[j]->v[2 * l] | ((uint64_t)g[j]->v[2 * l + 1] << 28);
    }
    return r;
}

// ---- field level ---------------------------------------------------------------------------------------
#define GF_BINOP(NAME, OP)                                                                                   \
    goldilocks_error_t NAME(uint8_t *out, const uint8_t *a, const uint8_t *b, size_t n) {                    \
        SHARD_LIGHT(n, 168, NAME(out + 56 * lo, a + 56 * lo, b + 56 * lo, m))                                \
        Call k;                                                                                              \
        LaneGf<OP> f = {k.out<uint8_t>(56 * n), nullptr, k.in(a, 56 * n), k.in(b, 56 * n), 0};               \
        k.run(f, n);                                                                                         \
        k.fetch(out, f.out, 56 * n);                                                                         \
        return k.finish();                                                                                   \
    }
GF_BINOP(goldilocks_448_gf_mul_batch, GFOP_MUL)
GF_BINOP(goldilocks_448_gf_add_batch, GFOP_ADD)
GF_BINOP(goldilocks_448_gf_sub_batch, GFOP_SUB)
goldilocks_error_t goldilocks_448_gf_sqr_batch(uint8_t *out, const uint8_t *a, size_t n) {
    SHARD_LIGHT(n, 112, goldilocks_448_gf_sqr_batch(out + 56 * lo, a + 56 * lo, m))
    Call k;
    LaneGf<GFOP_SQR> f = {k.out<uint8_t>(56 * n), nullptr, k.in(a, 56 * n), nullptr, 0};
    k.run(f, n);
    k.fetch(out, f.out, 56 * n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_gf_mulw_batch(uint8_t *out, const uint8_t *a, uint32_t w, size_t n) {
    SHARD_LIGHT(n, 112, goldilocks_448_gf_mulw_batch(out + 56 * lo, a + 56 * lo, w, m))
    Call k;
    if (w >= (1u << 28)) { g_err = "gf_mulw: w must be < 2^28"; return GOLDILOCKS_FAILURE; }
    LaneGf<GFOP_MULW> f = {k.out<uint8_t>(56 * n), nullptr, k.in(a, 56 * n), nullptr, w};
    k.run(f, n);
    k.fetch(out, f.out, 56 * n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_gf_isr_batch(uint8_t *out, goldilocks_error_t *status, const uint8_t *x, size_t n) {
    SHARD_LIGHT(n, 116, goldilocks_448_gf_isr_batch(out + 56 * lo, status + lo, x + 56 * lo, m))
    Call k;
    LaneGf<GFOP_ISR> f = {k.out<uint8_t>(56 * n), k.out<int32_t>(n), k.in(x, 56 * n), nullptr, 0};
    k.run(f, n);
    k.fetch(out, f.out, 56 * n);
    k.fetch((int32_t *)status, f.status, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_gf_invert_batch(uint8_t *out, const uint8_t *x, size_t n) {
    SHARD_LIGHT(n, 112, goldilocks_448_gf_invert_batch(out + 56 * lo, x + 56 * lo, m))
    Call k;
    LaneGf<GFOP_INVERT> f = {k.out<uint8_t>(56 * n), nullptr, k.in(x, 56 * n), nullptr, 0};
    k.run(f, n);
    k.fetch(out, f.out, 56 * n);
    return k.finish();
}

// ---- group level ---------------------------------------------------------------------------------------
#define PT_BINOP(NAME, OP)                                                                                   \
    goldilocks_error_t NAME(hpt *out, const hpt *a, const hpt *b, size_t n) {                                \
        SHARD_LIGHT(n, 768, NAME(out + lo, a + lo, b + lo, m))                                               \
        Call k;                                                                                              \
        LanePt<OP> f = {k.out<abi_pt>(n), k.in(P(a), n), k.in(P(b), n)};                                     \
        k.run(f, n);                                                                                         \
        k.fetch(P(out), f.out, n);                                                                           \
        return k.finish();                                                                                   \
    }
PT_BINOP(goldilocks_448_point_add_batch, PTOP_ADD)
PT_BINOP(goldilocks_448_point_sub_batch, PTOP_SUB)
#define PT_UNOP(NAME, OP)                                                                                    \
    goldilocks_error_t NAME(hpt *out, const hpt *a, size_t n) {                                              \
        SHARD_LIGHT(n, 512, NAME(out + lo, a + lo, m))                                                       \
        Call k;                                                                                              \
        LanePt<OP> f = {k.out<abi_pt>(n), k.in(P(a), n), nullptr};                                           \
        k.run(f, n);                                                                                         \
        k.fetch(P(out), f.out, n);                                                                           \
        return k.finish();                                                                                   \
    }
PT_UNOP(goldilocks_448_point_double_batch, PTOP_DBL)
PT_UNOP(goldilocks_448_point_negate_batch, PTOP_NEG)
PT_UNOP(goldilocks_448_point_debugging_torque_batch, PTOP_TORQUE)
goldilocks_error_t goldilocks_448_point_debugging_pscale_batch(hpt *out, const hpt *a, const uint8_t *factor, size_t n) {
    SHARD_LIGHT(n, 568, goldilocks_448_point_debugging_pscale_batch(out + lo, a + lo, factor + 56 * lo, m))
    Call k;
    LanePtPscale f = {k.out<abi_pt>(n), k.in(P(a), n), k.in(factor, 56 * n)};
    k.run(f, n);
    k.fetch(P(out), f.out, n);
    return k.finish();
}

goldilocks_error_t goldilocks_448_point_eq_batch(goldilocks_bool_t *out, const hpt *a, const hpt *b, size_t n) {
    SHARD_LIGHT(n, 520, goldilocks_448_point_eq_batch(out + lo, a + lo, b + lo, m))
    Call k;
    LanePtEq f = {k.out<uint64_t>(n), k.in(P(a), n), k.in(P(b), n)};
    k.run(f, n);
    k.fetch((uint64_t *)out, f.out, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_point_valid_batch(goldilocks_bool_t *out, const hpt *a, size_t n) {
    SHARD_LIGHT(n, 264, goldilocks_448_point_valid_batch(out + lo, a + lo, m))
    Call k;
    LanePtValid f = {k.out<uint64_t>(n), k.in(P(a), n)};
    k.run(f, n);
    k.fetch((uint64_t *)out, f.out, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_point_encode_batch(uint8_t *ser, const hpt *pts, size_t n) {
    SHARD_LIGHT(n, 312, goldilocks_448_point_encode_batch(ser + 56 * lo, pts + lo, m))
    Call k;
    LanePtEncode f = {k.out<uint8_t>(56 * n), k.in(P(pts), n)};
    k.run(f, n);
    k.fetch(ser, f.out, 56 * n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_point_decode_batch(hpt *pts, goldilocks_error_t *status, const uint8_t *ser, goldilocks_bool_t allow_identity, size_t n) {
    SHARD_LIGHT(n, 316, goldilocks_448_point_decode_batch(pts + lo, status + lo, ser + 56 * lo, allow_identity, m))
    Call k;
    LanePtDecode f = {k.out<abi_pt>(n), k.out<int32_t>(n), k.in(ser, 56 * n), allow_identity ? 1u : 0u};
    k.run(f, n);
    k.fetch(P(pts), f.out, n);
    k.fetch((int32_t *)status, f.status, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_point_from_hash_nonuniform_batch(hpt *pts, const uint8_t *hashed, size_t n) {
    SHARD_LIGHT(n, 312, goldilocks_448_point_from_hash_nonuniform_batch(pts + lo, hashed + 56 * lo, m))
    Call k;
    LaneFromHash<false> f = {k.out<abi_pt>(n), k.in(hashed, 56 * n)};
    k.run(f, n);
    k.fetch(P(pts), f.out, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_point_from_hash_uniform_batch(hpt *pts, const uint8_t *hashed, size_t n) {
    SHARD_LIGHT(n, 368, goldilocks_448_point_from_hash_uniform_batch(pts + lo, hashed + 112 * lo, m))
    Call k;
    LaneFromHash<true> f = {k.out<abi_pt>(n), k.in(hashed, 112 * n)};
    k.run(f, n);
    k.fetch(P(pts), f.out, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_invert_elligator_nonuniform_batch(uint8_t *recovered, goldilocks_error_t *status, const hpt *pts, const uint32_t *which, size_t n) {
    SHARD_LIGHT(n, 320, goldilocks_448_invert_elligator_nonuniform_batch(recovered + 56 * lo, status + lo, pts + lo, which + lo, m))
    Call k;
    LaneInvertElligator<false> f = {k.out<uint8_t>(56 * n), k.out<int32_t>(n), k.in(P(pts), n), k.in(which, n)};
    k.run(f, n);
    k.fetch(recovered, f.hashed, 56 * n);
    k.fetch((int32_t *)status, f.status, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_invert_elligator_uniform_batch(uint8_t *partial, goldilocks_error_t *status, const hpt *pts, const uint32_t *which, size_t n) {
    SHARD_LIGHT(n, 488, goldilocks_448_invert_elligator_uniform_batch(partial + 112 * lo, status + lo, pts + lo, which + lo, m))
    Call k;
    LaneInvertElligator<true> f = {k.in(partial, 112 * n), k.out<int32_t>(n), k.in(P(pts), n), k.in(which, n)};
    k.run(f, n);
    k.fetch(partial, f.hashed, 112 * n);
    k.fetch((int32_t *)status, f.status, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_point_mul_by_ratio_and_encode_like_eddsa_batch(uint8_t *enc, const hpt *pts, size_t n) {
    SHARD_LIGHT(n, 313, goldilocks_448_point_mul_by_ratio_and_encode_like_eddsa_batch(enc + 57 * lo, pts + lo, m))
    Call k;
    LaneEncodeEddsa f = {k.out<uint8_t>(57 * n), k.in(P(pts), n)};
    k.run(f, n);
    k.fetch(enc, f.out, 57 * n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_point_decode_like_eddsa_and_mul_by_ratio_batch(hpt *pts, goldilocks_error_t *status, const uint8_t *enc, size_t n) {
    SHARD_LIGHT(n, 317, goldilocks_448_point_decode_like_eddsa_and_mul_by_ratio_batch(pts + lo, status + lo, enc + 57 * lo, m))
    Call k;
    LaneDecodeEddsa f = {k.out<abi_pt>(n), k.out<int32_t>(n), k.in(enc, 57 * n)};
    k.run(f, n);
    k.fetch(P(pts), f.out, n);
    k.fetch((int32_t *)status, f.status, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_point_mul_by_ratio_and_encode_like_x448_batch(uint8_t *out, const hpt *pts, size_t n) {
    SHARD_LIGHT(n, 312, goldilocks_448_point_mul_by_ratio_and_encode_like_x448_batch(out + 56 * lo, pts + lo, m))
    Call k;
    LaneEncodeX448 f = {k.out<uint8_t>(56 * n), k.in(P(pts), n)};
    k.run(f, n);
    k.fetch(out, f.out, 56 * n);
    return k.finish();
}

/* test entry point: one mixed addition / conversion of goldilocks.c:271-380 per element (slot_lanes.cuh LanePtNiels, SlotNielsDebug) */
goldilocks_error_t goldilocks_b200_debug_niels_batch(hpt *out, const hpt *p, const hpt *q, const uint32_t *which, uint32_t op, size_t n) {
    if (op > 9) { g_err = "goldilocks_b200_debug_niels_batch: op must be 0..9"; return GOLDILOCKS_FAILURE; }
    Call k;
    abi_pt *dout = k.out<abi_pt>(n);
    const abi_pt *dp = k.in(P(p), n), *dq = k.in(P(q), n);
    const uint32_t *dw = k.in(which, n);
    pt *recs = k.out<pt>(n);
    const niels *comb = k.ok ? k.c->ft->comb : nullptr;
    if (op < 6) {
        LanePtNiels f = {dout, recs, dp, dq, comb, dw, op};
        k.run(f, n);
    } else {
        LanePtNiels f0 = {dout, recs, dp, dq, comb, dw, 10};
        k.run(f0, n);
        SlotNielsDebug f = {dout, dp, recs, comb, dw, op};
        k.run_sm(f, n);
    }
    k.fetch(P(out), dout, n);
    return k.finish();
}

// ---- scalar multiplications ------------------------------------------------------------------------------
goldilocks_error_t goldilocks_448_precomputed_scalarmul_batch(hpt *out, const goldilocks_448_precomputed_s *base, const hsc *scalar, size_t n) {
    SHARD_LIGHT(n, 312, goldilocks_448_precomputed_scalarmul_batch(out + lo, base, scalar + lo, m))
    Call k;
    if (base == goldilocks_448_precomputed_base) { /* the library's own base-point table: doubling-free comb */
        SlotComb f = {k.out<abi_pt>(n), k.secret(k.in(S(scalar), n), n), k.ok ? k.c->ft : nullptr};
        k.run_sm(f, n);
        k.fetch(P(out), f.out, n);
        return k.finish();
    }
    /* a table made by goldilocks_448_precompute(): upload it, convert to device limbs, reference-shaped comb */
    const abi_niels *up = k.in((const abi_niels *)base, COMB_ENTRIES);
    niels *tab = k.out<niels>(COMB_ENTRIES);
    LaneNielsFromAbi cv = {tab, up};
    k.run(cv, COMB_ENTRIES);
    SlotCombTable f = {k.out<abi_pt>(n), k.secret(k.in(S(scalar), n), n), tab};
    k.run_sm(f, n);
    k.fetch(P(out), f.out, n);
    return k.finish();
}
/* tables[k] = precompute(points[k]): 15 360 bytes each, byte-identical to the reference's (goldilocks.c:757-818) */
goldilocks_error_t goldilocks_448_precompute_batch(goldilocks_448_precomputed_s *tables, const hpt *points, size_t n) {
    SHARD_LIGHT(n, 15616, goldilocks_448_precompute_batch((goldilocks_448_precomputed_s *)((uint8_t *)tables + 15360 * lo), points + lo, m))
    Call k;
    LanePrecompute f = {k.out<abi_niels>(COMB_ENTRIES * n), k.in(P(points), n), k.out<niels>(16 * COMB_N * n)};
    k.run(f, COMB_N * n);
    k.fetch((abi_niels *)tables, f.tables, COMB_ENTRIES * n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_point_dual_scalarmul_batch(hpt *out1, hpt *out2, const hpt *base, const hsc *scalar1, const hsc *scalar2, size_t n) {
    SHARD_HEAVY(n, goldilocks_448_point_dual_scalarmul_batch(out1 + lo, out2 + lo, base + lo, scalar1 + lo, scalar2 + lo, m))
    Call k;
    int grid = k.smp_grid_for<SlotDualScalarmul>();
    SlotDualScalarmul f = {k.secret(k.out<abi_pt>(n), n), k.secret(k.out<abi_pt>(n), n), k.in(P(base), n), k.secret(k.in(S(scalar1), n), n), k.secret(k.in(S(scalar2), n), n), k.slots((size_t)grid * SLOT_BLOCK, 1)};
    k.run_smp(f, n, grid);
    k.fetch(P(out1), f.out1, n);
    k.fetch(P(out2), f.out2, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_direct_scalarmul_batch(uint8_t *scaled, goldilocks_error_t *status, const uint8_t *base, const hsc *scalar,
                                                         goldilocks_bool_t allow_identity, goldilocks_bool_t short_circuit, size_t n) {
    SHARD_HEAVY(n, goldilocks_448_direct_scalarmul_batch(scaled + 56 * lo, status + lo, base + 56 * lo, scalar + lo, allow_identity, short_circuit, m))
    Call k;
    int grid = k.smp_grid_for<SlotDirectScalarmul>();
    uint8_t *dout = k.in(scaled, 56 * n); /* short-circuited elements keep the caller's bytes */
    k.secret(dout, 56 * n);
    SlotDirectScalarmul f = {dout, k.out<int32_t>(n), k.in(base, 56 * n), k.secret(k.in(S(scalar), n), n), allow_identity ? 1u : 0u, short_circuit ? 1u : 0u,
                             k.ok ? k.c->ft : nullptr, k.slots((size_t)grid * SLOT_BLOCK, 1)};
    k.run_smp(f, n, grid);
    k.fetch(scaled, dout, 56 * n);
    k.fetch((int32_t *)status, f.status, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_point_scalarmul_batch(hpt *out, const hpt *base, const hsc *scalar, size_t n) {
    SHARD_HEAVY(n, goldilocks_448_point_scalarmul_batch(out + lo, base + lo, scalar + lo, m))
    Call k;
    int grid = k.smp_grid_for<SlotScalarmul>();
    SlotScalarmul f = {k.secret(k.out<abi_pt>(n), n), k.in(P(base), n), k.secret(k.in(S(scalar), n), n), k.slots((size_t)grid * SLOT_BLOCK, 1)};
    k.run_smp(f, n, grid);
    k.fetch(P(out), f.out, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_point_double_scalarmul_batch(hpt *out, const hpt *base1, const hsc *scalar1, const hpt *base2, const hsc *scalar2, size_t n) {
    SHARD_HEAVY(n, goldilocks_448_point_double_scalarmul_batch(out + lo, base1 + lo, scalar1 + lo, base2 + lo, scalar2 + lo, m))
    Call k;
    int grid = k.smp_grid_for<SlotDoubleScalarmul>();
    SlotDoubleScalarmul f = {k.secret(k.out<abi_pt>(n), n), k.in(P(base1), n), k.secret(k.in(S(scalar1), n), n), k.in(P(base2), n), k.secret(k.in(S(scalar2), n), n),
                             k.slots((size_t)grid * SLOT_BLOCK, 2), (size_t)grid * SLOT_BLOCK};
    k.run_smp(f, n, grid);
    k.fetch(P(out), f.out, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_base_double_scalarmul_non_secret_batch(hpt *out, const hsc *scalar1, const hpt *base2, const hsc *scalar2, size_t n) {
    SHARD_HEAVY(n, goldilocks_448_base_double_scalarmul_non_secret_batch(out + lo, scalar1 + lo, base2 + lo, scalar2 + lo, m))
    Call k;
    int grid = k.smp_grid_for<SlotBaseDoubleScalarmul>();
    SlotBaseDoubleScalarmul f = {k.out<abi_pt>(n), k.in(S(scalar1), n), k.in(P(base2), n), k.in(S(scalar2), n), k.ok ? k.c->wide : nullptr,
                                 k.slots((size_t)grid * SLOT_BLOCK, 1)};
    k.run_smp(f, n, grid);
    k.fetch(P(out), f.out, n);
    return k.finish();
}

// ---- scalars -----------------------------------------------------------------------------------------------
#define SC_BINOP(NAME, OP)                                                                                   \
    goldilocks_error_t NAME(hsc *out, const hsc *a, const hsc *b, size_t n) {                                \
        SHARD_LIGHT(n, 168, NAME(out + lo, a + lo, b + lo, m))                                               \
        Call k;                                                                                              \
        LaneSc<OP> f = {k.out<abi_sc>(n), k.in(S(a), n), k.in(S(b), n)};                                     \
        k.run(f, n);                                                                                         \
        k.fetch(S(out), f.out, n);                                                                           \
        return k.finish();                                                                                   \
    }
SC_BINOP(goldilocks_448_scalar_add_batch, SCOP_ADD)
SC_BINOP(goldilocks_448_scalar_sub_batch, SCOP_SUB)
SC_BINOP(goldilocks_448_scalar_mul_batch, SCOP_MUL)
goldilocks_error_t goldilocks_448_scalar_invert_batch(hsc *out, goldilocks_error_t *status, const hsc *a, size_t n) {
    SHARD_LIGHT(n, 116, goldilocks_448_scalar_invert_batch(out + lo, status + lo, a + lo, m))
    Call k;
    LaneScInvert f = {k.out<abi_sc>(n), k.out<int32_t>(n), k.in(S(a), n)};
    k.run(f, n);
    k.fetch(S(out), f.out, n);
    k.fetch((int32_t *)status, f.status, n);
    return k.finish();
}
goldilocks_error_t goldilocks_ed448_convert_public_key_to_x448_batch(uint8_t *x, const uint8_t *ed, size_t n) {
    SHARD_LIGHT(n, 113, goldilocks_ed448_convert_public_key_to_x448_batch(x + 56 * lo, ed + 57 * lo, m))
    Call k;
    LaneEdPkToX448 f = {k.out<uint8_t>(56 * n), k.in(ed, 57 * n)};
    k.run(f, n);
    k.fetch(x, f.x, 56 * n);
    return k.finish();
}
goldilocks_error_t goldilocks_ed448_convert_private_key_to_x448_batch(uint8_t *x, const uint8_t *ed, size_t n) {
    SHARD_LIGHT(n, 113, goldilocks_ed448_convert_private_key_to_x448_batch(x + 56 * lo, ed + 57 * lo, m))
    Call k;
    LaneEdSkToX448 f = {k.secret(k.out<uint8_t>(56 * n), 56 * n), k.secret(k.in(ed, 57 * n), 57 * n)};
    k.run(f, n);
    k.fetch(x, f.x, 56 * n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_scalar_halve_batch(hsc *out, const hsc *a, size_t n) {
    SHARD_LIGHT(n, 112, goldilocks_448_scalar_halve_batch(out + lo, a + lo, m))
    Call k;
    LaneSc<SCOP_HALVE> f = {k.out<abi_sc>(n), k.in(S(a), n), nullptr};
    k.run(f, n);
    k.fetch(S(out), f.out, n);
    return k.finish();
}
goldilocks_error_t goldilocks_448_scalar_decode_long_batch(hsc *out, const uint8_t *ser, size_t ser_len, size_t n) {
    SHARD_LIGHT(n, ser_len + 56, goldilocks_448_scalar_decode_long_batch(out + lo, ser + ser_len * lo, ser_len, m))
    Call k;
    LaneScDecodeLong f = {k.out<abi_sc>(n), k.in(ser, ser_len * n), ser_len};
    k.run(f, n);
    k.fetch(S(out), f.out, n);
    return k.finish();
}

// ---- CFRG ----------------------------------------------------------------------------------------------------
goldilocks_error_t goldilocks_x448_batch(uint8_t *out, goldilocks_error_t *status, const uint8_t *base, const uint8_t *scalar, size_t n) {
    SHARD_HEAVY(n, goldilocks_x448_batch(out + 56 * lo, status + lo, base + 56 * lo, scalar + 56 * lo, m))
    Call k;
    SlotX448 f = {k.secret(k.out<uint8_t>(56 * n), 56 * n), k.out<int32_t>(n), k.in(base, 56 * n), k.secret(k.in(scalar, 56 * n), 56 * n)};
    k.run_sm(f, n);
    k.fetch(out, f.out, 56 * n);
    k.fetch((int32_t *)status, f.status, n);
    return k.finish();
}
goldilocks_error_t goldilocks_x448_derive_public_key_batch(uint8_t *out, const uint8_t *scalar, size_t n) {
    SHARD_HEAVY(n, goldilocks_x448_derive_public_key_batch(out + 56 * lo, scalar + 56 * lo, m))
    Call k;
    SlotX448DerivePk f = {k.out<uint8_t>(56 * n), k.secret(k.in(scalar, 56 * n), 56 * n), k.ok ? k.c->ft : nullptr};
    k.run_sm(f, n);
    k.fetch(out, f.out, 56 * n);
    return k.finish();
}
goldilocks_error_t goldilocks_shake256_hash_batch(uint8_t *out, size_t outlen, const uint8_t *in, const size_t *in_off, size_t n) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    SHARD_LIGHT(n, outlen + in_off[n] / n, goldilocks_shake256_hash_batch(out + outlen * lo, outlen, in + in_off[lo], SubOffsets(in_off, lo, m).v.data(), m))
    Call k;
    size_t total = n ? in_off[n] : 0;
    LaneShake256 f = {k.out<uint8_t>(outlen * n), outlen, k.in(in, total), k.in(in_off, n + 1)};
    k.run(f, n);
    k.fetch(out, f.out, outlen * n);
    return k.finish();
}
goldilocks_error_t goldilocks_ed448_derive_public_key_batch(uint8_t *pubkey, const uint8_t *privkey, size_t n) {
    SHARD_HEAVY(n, goldilocks_ed448_derive_public_key_batch(pubkey + 57 * lo, privkey + 57 * lo, m))
    Call k;
    SlotEdDerivePk f = {k.out<uint8_t>(57 * n), k.secret(k.in(privkey, 57 * n), 57 * n), k.ok ? k.c->ft : nullptr};
    k.run_sm(f, n);
    k.fetch(pubkey, f.pk, 57 * n);
    return k.finish();
}
goldilocks_error_t goldilocks_ed448_sign_batch(uint8_t *signature, const uint8_t *privkey, const uint8_t *pubkey, const uint8_t *msg, const size_t *msg_off,
                                               uint8_t prehashed, const uint8_t *context, uint8_t context_len, size_t n) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    SHARD_HEAVY(n, goldilocks_ed448_sign_batch(signature + 114 * lo, privkey + 57 * lo, pubkey + 57 * lo, msg + msg_off[lo], SubOffsets(msg_off, lo, m).v.data(), prehashed, context, context_len, m))
    Call k;
    size_t total = n ? msg_off[n] : 0;
    const uint8_t *dmsg = k.in(msg, total);
    const size_t *doff = k.in(msg_off, n + 1);
    const uint8_t *dctx = k.in(context, context_len);
    const uint8_t *dsk = k.secret(k.in(privkey, 57 * n), 57 * n), *dpk = k.in(pubkey, 57 * n);
    abi_sc *secret = k.secret(k.out<abi_sc>(n), n), *nonce = k.secret(k.out<abi_sc>(n), n), *nonce4 = k.secret(k.out<abi_sc>(n), n);
    uint8_t *dsig = k.out<uint8_t>(114 * n);
    uint8_t *seed = k.secret(k.out<uint8_t>(57 * n), 57 * n);
    LaneEdSignExpand f0 = {secret, seed, dsk};
    k.run(f0, n);
    LaneEdSignNonce f1 = {nonce, nonce4, seed, dmsg, doff, prehashed, dctx, context_len};
    k.run(f1, n);
    SlotEdSignR f2 = {dsig, nonce4, k.ok ? k.c->ft : nullptr};
    k.run_sm(f2, n);
    LaneEdSignFinish f3 = {dsig, secret, nonce, dpk, dmsg, doff, prehashed, dctx, context_len};
    k.run(f3, n);
    k.fetch(signature, dsig, 114 * n);
    return k.finish(); /* zeroes the device copies of the private keys, secret scalars, nonces and seeds on every path */
}

// Batches of at least VERIFY_GROUP_MIN signatures are grouped by public key on the device (k_group.cu); keys that
// occur more than once get one shared table (at most n/4 + 1 tables per call -- every key of a batch with four or more signatures per key; the rest verify stand-alone).
constexpr size_t VERIFY_GROUP_MIN = 64;
static size_t verify_tab_cap(size_t n) { return n / 4 + 1; }
static bool verify_groups(size_t n) { return n >= VERIFY_GROUP_MIN && n < ((size_t)1 << 31); } /* the work lists are 32-bit */
static size_t verify_core_scratch_bytes(size_t n) {
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    size_t base = al(2 * n * sizeof(abi_pt)) + al(2 * n * sizeof(int32_t)) + 2 * al(n * sizeof(abi_sc));
    if (verify_groups(n)) base += al(group_scratch_bytes(n, verify_tab_cap(n))) + al(verify_tab_cap(n) * KTAB_QUADS * sizeof(uint4));
    return base;
}
struct VerifyGrids { int unique = 1, shared = 1, chain = 1, columns = 1; };
static bool verify_grids(Ctx &c, VerifyGrids *g) {
    return smp_grid<SlotEdVerifyFinish>(c, &g->unique) && smp_grid<SlotEdVerifyFinishShared>(c, &g->shared) && smp_grid<SlotKeyChain>(c, &g->chain) &&
           smp_grid<SlotKeyColumns>(c, &g->columns);
}
// per-thread window tables of the stand-alone signatures (wtab, slot_algos.cuh): one per resident lane of the finish kernel
static size_t verify_slot_bytes(const VerifyGrids &g, size_t n) {
    const int grid = std::max(std::max(g.unique, g.shared), g.columns);
    size_t lanes = (size_t)grid * SLOT_BLOCK;
    const size_t items = std::max(n, verify_groups(n) ? verify_column_items(n) : (size_t)0);
    const size_t need = (items + SLOT_BLOCK - 1) / SLOT_BLOCK * SLOT_BLOCK;
    if (lanes > need) lanes = need;
    return (lanes * 2 * WTAB_QUADS_PER_LANE * sizeof(uint4) + 255) & ~(size_t)255;   /* two tables per lane: the key's and R's (s_verify_half_item) */
}
size_t goldilocks_b200_verify_scratch_bytes(size_t n) {
    /* the device-pointer call carves EVERYTHING it writes from the caller's scratch (two verifications in flight on two
     * streams share nothing), so the figure includes the window tables and depends on the current device's SM count */
    Ctx *c = dev_ctx();
    VerifyGrids grids;
    if (!c || !verify_grids(*c, &grids)) return 0;
    return verify_core_scratch_bytes(n) + verify_slot_bytes(grids, n);
}
// Host-pointer calls feed the signatures and messages in two halves on the copy stream: [0, split) is on the device
// when ready[0] fires, the rest at ready[1]; the public keys (all the grouping pass needs) go first on the main stream.
struct VerifyFeed { size_t split; cudaEvent_t ready[2]; };
static bool verify_dev(Ctx &c, int32_t *status, const uint8_t *sig, const uint8_t *pk, const uint8_t *msg, const size_t *off, uint8_t prehashed,
                       const uint8_t *ctx, uint8_t ctx_len, size_t n, void *scratch, uint4 *slots, const VerifyGrids &grids, cudaStream_t s,
                       const VerifyFeed *feed = nullptr, cudaStream_t side = nullptr, cudaEvent_t *side_evt = nullptr) {
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    char *p = (char *)scratch;
    abi_pt *pts = (abi_pt *)p; p += al(2 * n * sizeof(abi_pt));
    int32_t *ok = (int32_t *)p; p += al(2 * n * sizeof(int32_t));
    abi_sc *chal = (abi_sc *)p; p += al(n * sizeof(abi_sc));
    abi_sc *resp = (abi_sc *)p; p += al(n * sizeof(abi_sc));
    verify_plan plan = {nullptr, nullptr, nullptr, nullptr, nullptr};
    uint4 *ktabs = nullptr;
    const size_t cap = verify_tab_cap(n);
    if (verify_groups(n)) {
        void *gs = p; p += al(group_scratch_bytes(n, cap));
        ktabs = (uint4 *)p;
        uint64_t launched = 0;
        cudaError_t e = group_keys(pk, n, (uint32_t)cap, gs, &plan, s, &launched);
        if (e != cudaSuccess) return fail("group_keys", e);
        g_launches += launched;
    }
    /* without a plan: R and public key of signatures [lo, hi) (interleaved lanes).  With a plan nothing decodes R: the
     * finish kernel works from its bytes (s_verify_accept_prep, slot_lanes.cuh). */
    auto decode_range = [&](size_t lo, size_t hi) {
        if (plan.unique_sig) return true;
        LaneEdVerifyDecode f = {pts, ok, sig, pk, n, plan, 2 * lo};
        return launch(c, f, 2 * (hi - lo), s);
    };
    auto scalars_range = [&](size_t lo, size_t hi) {
        LaneEdVerifyScalars f = {chal, resp, sig, pk, msg, off, prehashed, ctx, ctx_len, lo};
        return launch(c, f, hi - lo, s);
    };
    const size_t split = feed ? feed->split : n;
    if (plan.unique_sig && side) {
        CU(cudaEventRecord(side_evt[0], s));            /* fork here: the hashes also run beside the per-key decodes (one inverse square root chain per key) */
    }
    if (plan.unique_sig) { /* one decode per distinct key: needs the keys only, so it runs while the signatures still cross PCIe */
        LaneEdVerifyDecode fa = {pts, ok, sig, pk, n, plan, n};
        if (!launch(c, fa, n, s)) return false;
    }
    if (plan.unique_sig && side) {
        /* The key tables need the decoded keys only; the challenge hashes need the signatures and messages only.  The table kernel is
         * a multiplier-bound chain on less than one wave of lanes (one lane per distinct key), the hashes are ALU work: the hashes go
         * to the side stream and fill the issue slots the table kernel leaves (verify_dev's caller owns `side` for the call). */
        CU(cudaStreamWaitEvent(side, side_evt[0], 0));
        if (feed) CU(cudaStreamWaitEvent(side, feed->ready[0], 0));
        {
            LaneEdVerifyScalars f = {chal, resp, sig, pk, msg, off, prehashed, ctx, ctx_len, 0};
            if (!launch(c, f, split, side)) return false;
        }
        if (feed) CU(cudaStreamWaitEvent(side, feed->ready[1], 0));
        if (split < n) {
            LaneEdVerifyScalars f = {chal, resp, sig, pk, msg, off, prehashed, ctx, ctx_len, split};
            if (!launch(c, f, n - split, side)) return false;
        }
        {   /* the stand-alone signatures: the half-size multipliers and their R (the lanes past counts[1] retire at once) */
            LaneVerifyHalf fh = {chal, resp, plan};
            if (!launch(c, fh, n, side)) return false;
            LaneEdVerifyDecode fr = {pts, ok, sig, pk, n, plan, 2 * n};
            if (!launch(c, fr, n, side)) return false;
        }
        CU(cudaEventRecord(side_evt[1], side));
        SlotKeyChain fc = {pts, ktabs, plan};           /* the doubling chain: one lane per key table ... */
        if (!launch_smp(c, fc, cap, grids.chain, s, const_cast<uint32_t *>(plan.counts) + 4)) return false; /* counts[3..5] = 0, left by the grouping pass */
        SlotKeyColumns ft = {ktabs, slots, plan};       /* ... then a lane per key and column fills the column tables (10 or 15 per key, vsh_pick) */
        if (!launch_smp(c, ft, verify_column_items(n), grids.columns, s, const_cast<uint32_t *>(plan.counts) + 5)) return false;
        CU(cudaStreamWaitEvent(s, side_evt[1], 0));
        if (feed) { CU(cudaStreamWaitEvent(s, feed->ready[0], 0)); CU(cudaStreamWaitEvent(s, feed->ready[1], 0)); } /* the finish kernel reads the signature bytes too */
        SlotEdVerifyFinishShared fs = {pts, ok, chal, resp, c.wide, ktabs, slots, plan, sig};
        if (!launch_smp(c, fs, n, grids.shared, s, const_cast<uint32_t *>(plan.counts) + 3)) return false;
        LaneVerifySign fv = {status, (verify_aux *)(pts + 1), 2, n};    /* aux record of signature i = the R half of pts[2i..2i+1] */
        return launch(c, fv, (n + VSIGN_BATCH - 1) / VSIGN_BATCH, s);
    }
    if (feed) CU(cudaStreamWaitEvent(s, feed->ready[0], 0));
    if (!decode_range(0, split) || !scalars_range(0, split)) return false;
    if (feed) CU(cudaStreamWaitEvent(s, feed->ready[1], 0));
    if (split < n && (!decode_range(split, n) || !scalars_range(split, n))) return false;
    {
        LaneVerifyHalf fh = {chal, resp, plan};
        if (!launch(c, fh, n, s)) return false;
        if (plan.unique_sig) {
            LaneEdVerifyDecode fr = {pts, ok, sig, pk, n, plan, 2 * n};
            if (!launch(c, fr, n, s)) return false;
        }
    }
    if (plan.unique_sig) {
        SlotKeyChain fc = {pts, ktabs, plan};           /* the doubling chain: one lane per key table ... */
        if (!launch_smp(c, fc, cap, grids.chain, s, const_cast<uint32_t *>(plan.counts) + 4)) return false; /* counts[3..5] = 0, left by the grouping pass */
        SlotKeyColumns ft = {ktabs, slots, plan};       /* ... then a lane per key and column fills the column tables (10 or 15 per key, vsh_pick) */
        if (!launch_smp(c, ft, verify_column_items(n), grids.columns, s, const_cast<uint32_t *>(plan.counts) + 5)) return false;
        SlotEdVerifyFinishShared fs = {pts, ok, chal, resp, c.wide, ktabs, slots, plan, sig};
        if (!launch_smp(c, fs, n, grids.shared, s, const_cast<uint32_t *>(plan.counts) + 3)) return false;
        LaneVerifySign fv = {status, (verify_aux *)(pts + 1), 2, n};    /* aux record of signature i = the R half of pts[2i..2i+1] */
        return launch(c, fv, (n + VSIGN_BATCH - 1) / VSIGN_BATCH, s);
    }
    SlotEdVerifyFinish f3 = {status, pts, ok, chal, resp, c.wide, slots};
    return launch_smp(c, f3, n, grids.unique, s, GRID_STRIDE); /* no plan: fewer than 64 signatures (one partial round), or more than 2^31 */
}
goldilocks_error_t goldilocks_ed448_verify_batch(goldilocks_error_t *status, const uint8_t *signature, const uint8_t *pubkey, const uint8_t *msg, const size_t *msg_off,
                                                 uint8_t prehashed, const uint8_t *context, uint8_t context_len, size_t n) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    SHARD_HEAVY(n, goldilocks_ed448_verify_batch(status + lo, signature + 114 * lo, pubkey + 57 * lo, msg + msg_off[lo], SubOffsets(msg_off, lo, m).v.data(), prehashed, context, context_len, m))
    /* One pass over the whole batch (splitting the BATCH costs more than it hides: every chunk pays its own key-grouping
     * pass and key-table wave, 67.9 ms split vs 66.3 ms whole at 2^20).  Only the COPIES are split: keys first, then the
     * signatures and messages in two halves on the copy stream, so the grouping pass, the per-key decodes and the first
     * half's challenge hashes run while the rest is still crossing PCIe. */
    Call k;
    size_t total = n ? msg_off[n] : 0;
    const size_t *doff = k.in(msg_off, n + 1);
    const uint8_t *dctx = k.in(context, context_len);
    const uint8_t *dpk = k.in(pubkey, 57 * n);
    uint8_t *dsig = k.out<uint8_t>(114 * n), *dmsg = k.out<uint8_t>(total);
    int32_t *dst = k.out<int32_t>(n);
    VerifyGrids grids;
    if (k.ok) k.ok = verify_grids(*k.c, &grids);
    const int grid = std::max(std::max(grids.unique, grids.shared), grids.columns);
    uint4 *slots = k.slots((size_t)grid * SLOT_BLOCK, 2);
    void *scratch = k.alloc(verify_core_scratch_bytes(n));
    VerifyFeed feed = {n >= 2 * VERIFY_GROUP_MIN ? n / 2 : n, {nullptr, nullptr}};
    if (k.ok) {
        feed.ready[0] = k.c->copy_done[0]; feed.ready[1] = k.c->copy_done[1];
        const size_t lo[2] = {0, feed.split}, hi[2] = {feed.split, n};
        for (int h = 0; h < 2 && k.ok; h++) {
            k.push(dsig + 114 * lo[h], signature + 114 * lo[h], 114 * (hi[h] - lo[h]));
            if (hi[h] > lo[h]) k.push(dmsg + msg_off[lo[h]], msg + msg_off[lo[h]], msg_off[hi[h]] - msg_off[lo[h]]);
            if (cudaEventRecord(feed.ready[h], k.c->copy_stream) != cudaSuccess) k.ok = false;
        }
    }
    if (k.ok) k.ok = verify_dev(*k.c, dst, dsig, dpk, dmsg, doff, prehashed, dctx, context_len, n, scratch, slots, grids, k.c->stream, &feed, k.c->side_stream, k.c->side_evt);
    k.fetch((int32_t *)status, dst, n);
    if (!k.ok && k.c) cudaStreamSynchronize(k.c->copy_stream); /* never leave copies in flight behind an error */
    return k.finish();
}

// ---- random-linear-combination batch verification (rlc.cuh; SURVEY 8(f)3): optional fast path, per-element fallback --
// One multi-scalar multiplication decides the whole batch; if its equation fails (or anything looks odd) the ordinary
// per-signature path above runs over the same device buffers, so the statuses are per element either way.
constexpr size_t RLC_MIN = 64;
static bool rlc_seed(uint8_t seed[32]) { /* fresh secret weights per call: the signer must not be able to predict them */
    size_t got = 0;
    while (got < 32) {
        ssize_t r = getrandom(seed + got, 32 - got, 0);
        if (r <= 0) { g_err = "getrandom failed: no entropy for the batch-verification weights"; return false; }
        got += (size_t)r;
    }
    return true;
}
static bool rlc_usable(size_t n) { return n >= RLC_MIN && n < ((size_t)1 << 26); } /* pair lists are 32-bit, CUB counts are int */
// One class of points through the bucket method: digits -> radix sort -> buckets -> segments -> tree nodes.  The window
// sums (the c*w doublings) are a separate launch so that the key class can run its long chain on the side stream.
struct RlcClass { rlc_shape sh; size_t count, npairs, nb; uint32_t *keys, *vals, *keys_s, *vals_s; void *sort_tmp; size_t sort_bytes; pt *buckets, *segsum, *nodesum, *winsum, *total;
                  uint32_t *bstart, *blen, *bid, *blen_s, *perm; void *bsort_tmp; size_t bsort_bytes; };
static bool rlc_class_alloc(Call &k, RlcClass &q, const rlc_shape &sh, size_t count) {
    const size_t nw = (size_t)sh.nch * sh.wn; /* window ids run over chunks x windows */
    q.sh = sh; q.count = count; q.npairs = count * sh.wn; q.nb = nw << sh.c;
    q.keys = k.out<uint32_t>(q.npairs); q.vals = k.out<uint32_t>(q.npairs); q.keys_s = k.out<uint32_t>(q.npairs); q.vals_s = k.out<uint32_t>(q.npairs);
    q.sort_bytes = pair_sort_scratch_bytes(q.npairs);
    q.sort_tmp = k.alloc(q.sort_bytes);
    q.bstart = k.out<uint32_t>(q.nb); q.blen = k.out<uint32_t>(q.nb); q.bid = k.out<uint32_t>(q.nb); q.blen_s = k.out<uint32_t>(q.nb); q.perm = k.out<uint32_t>(q.nb);
    q.bsort_bytes = pair_sort_scratch_bytes(q.nb);
    q.bsort_tmp = k.alloc(q.bsort_bytes);
    q.buckets = k.out<pt>(q.nb); q.segsum = k.out<pt>(nw * sh.segs); q.nodesum = k.out<pt>(nw * sh.nodes); q.winsum = k.out<pt>(nw); q.total = k.out<pt>(sh.nch);
    return k.ok;
}
static bool rlc_class_pairs(Ctx &c, const RlcClass &q, const uint32_t *scal, uint32_t nwords, size_t p0, cudaStream_t s, const uint32_t *chunk_of) { /* digits -> sorted pair list */
    LaneRlcDigits f6 = {q.keys, q.vals, scal, nwords, p0, q.sh, chunk_of};
    if (!launch(c, f6, q.count, s)) return false;
    int key_bits = 1;
    while (((q.sh.nch * q.sh.wn) << q.sh.c) >> key_bits) key_bits++;
    cudaError_t e = pair_sort(q.sort_tmp, q.sort_bytes, q.keys, q.keys_s, q.vals, q.vals_s, q.npairs, key_bits, s);
    if (e != cudaSuccess) return fail("pair_sort", e);
    /* the runs of the buckets and the order the bucket kernel takes them in (longest first: equal lengths share a warp) */
    LaneRlcBucketRuns fr = {q.bstart, q.blen, q.bid, q.keys_s, q.npairs, q.sh};
    if (!launch(c, fr, q.nb, s)) return false;
    e = pair_sort(q.bsort_tmp, q.bsort_bytes, q.blen, q.blen_s, q.bid, q.perm, q.nb, 8, s);
    if (e != cudaSuccess) return fail("pair_sort (bucket lengths)", e);
    return true;
}
static bool rlc_class_sum(Ctx &c, const RlcClass &q, const pt *recs, cudaStream_t s, bool subtract, const int32_t *valid) { /* buckets -> window sums */
    /* plain grid, not the persistent shape: blocks retire all the time, so the high-priority blocks of the side stream get onto
     * the SMs between them (persistent blocks held the SMs and starved the side stream: 22.6 vs 20.9 ms per 2^20) */
    SlotRlcBucket f7 = {q.buckets, q.keys_s, q.vals_s, q.npairs, recs, q.sh, subtract ? ~0u : 0u, valid, q.perm, q.bstart};
    if (!launch_slots(c, f7, q.nb, s)) return false;
    const size_t nw = (size_t)q.sh.nch * q.sh.wn;
    LaneRlcSegments f8 = {q.segsum, q.buckets, q.sh};
    if (!launch(c, f8, nw * q.sh.segs, s)) return false;
    LaneRlcNodes f9 = {q.nodesum, q.segsum, q.sh};
    if (!launch(c, f9, nw * q.sh.nodes, s)) return false;
    LaneRlcWindows f10 = {q.winsum, q.nodesum, q.sh};
    if (!launch(c, f10, nw, s)) return false;
    LaneRlcTotal f11 = {q.total, q.winsum, q.sh.wn, q.sh.nch > 1 ? q.sh.c : 0u};
    return launch(c, f11, q.sh.nch, s);
}
// Host-pointer calls feed the copy stream in the order the work can start in: the first half of the signatures (the R decodes,
// 55 % of the call, need nothing else), then keys / offsets / context (the grouping pass), then the rest.
struct RlcFeed { size_t split[2]; cudaEvent_t sig0, keys, sig1, rest; }; /* signatures [0, split[0]) | keys | [split[0], split[1]) | the rest */
// goldilocks_ed448_verify_rlc_batch, on device buffers.  *fast: 1 = the whole-batch equation decided the call; 2 = it failed, the
// equations were run again per chunk of consecutive signatures (same R decodes, challenges and weights) and only the chunks that
// failed were re-verified one signature at a time; 0 = the ordinary per-signature path ran over everything.
//
// Why two passes instead of chunks from the start: chunks cost digit width (a chunk of 4 096 signatures fills its buckets with
// c = 9, i.e. 15 additions per signature instead of 9, and every chunk pays its own bucket folding and key class), so the
// all-valid call -- the one this entry point exists for -- stays one equation; what a failure adds is the second pass
// (no decodes, no hashes) plus the per-signature path over the failed chunks only, packed into one batch.
// Traffic that keeps failing most chunks gains nothing from either pass, so the context remembers the last outcome: after
// a call in which more than RLC_GIVE_UP of the chunks failed, the next reprobe - 1 calls on this context (goldilocks_b200_rlc_policy, default 16) go straight to the
// per-signature path (cost: the ordinary call's) and the one after that tries the equation again.
constexpr size_t RLC_CHUNK_TARGET = 4096;   /* signatures per chunk of the localisation pass (GOLDILOCKS_B200_RLC_CHUNK overrides) */
constexpr uint32_t RLC_MAX_CHUNKS = 1024;
std::atomic<unsigned> g_rlc_reprobe{16};     /* goldilocks_b200_rlc_policy */
static bool rlc_core(Call &k, int32_t *dst, const uint8_t *dsig, const uint8_t *dpk, const uint8_t *dmsg, const size_t *doff, uint8_t prehashed,
                     const uint8_t *dctx, uint8_t ctx_len, size_t n, cudaStream_t s, int *fast, const RlcFeed *feed = nullptr) {
    Ctx &c = *k.c;
    *fast = 0;
    auto ordinary_on = [&](int32_t *st, const uint8_t *sig, const uint8_t *pk, const uint8_t *msg, const size_t *off, size_t cnt) {
        VerifyGrids grids;
        if (!verify_grids(c, &grids)) return false;
        const int grid = std::max(std::max(grids.unique, grids.shared), grids.columns);
        uint4 *slots = k.slots((size_t)grid * SLOT_BLOCK, 2);
        void *scratch = k.alloc(verify_core_scratch_bytes(cnt));
        if (!k.ok) return false;
        return verify_dev(c, st, sig, pk, msg, off, prehashed, dctx, ctx_len, cnt, scratch, slots, grids, s);
    };
    auto ordinary = [&]() { return ordinary_on(dst, dsig, dpk, dmsg, doff, n); }; /* every copy has been waited for on `s` by the time this runs */
    const bool skip = c.rlc_skip > 0;       /* recent calls failed most of their chunks: do not even try (see above) */
    if (skip) c.rlc_skip--;
    if (!rlc_usable(n) || skip) {
        if (feed) CU(cudaStreamWaitEvent(s, feed->rest, 0));
        return ordinary();
    }
    uint8_t seed[32];
    if (!rlc_seed(seed)) return false;
    cudaStream_t side = c.side_stream;
    /* shared by both passes: everything sized by n alone -- the R decodes start before the number of distinct keys is known */
    void *gs = k.alloc(group_all_scratch_bytes(n));
    uint8_t *dseed = k.out<uint8_t>(32);
    const uint32_t max_ch = RLC_MAX_CHUNKS;
    pt *pts = k.out<pt>(2 * n + max_ch);                               /* n R records, then at most n key groups, then one B per chunk */
    int32_t *ok = k.out<int32_t>(2 * n + max_ch), *valid = k.out<int32_t>(n);
    uint32_t *flags = k.out<uint32_t>(2 + (size_t)max_ch);             /* [0] force fallback, [1 + ch] verdict of chunk ch, [1 + chunks] redo the key class */
    abi_sc *chal = k.out<abi_sc>(n), *resp = k.out<abi_sc>(n);
    uint32_t *z = k.out<uint32_t>(RLC_ZWORDS * n);
    k.secret(z, RLC_ZWORDS * n);                                      /* the weights are secret until the verdict is out: wiped when the call ends */
    if (!k.ok) return false;
    CU(cudaMemcpyAsync(dseed, seed, 32, cudaMemcpyHostToDevice, s));
    std::vector<uint32_t> hflags;
    uint32_t zbits = 0;
    /* one pass of equations over chunks of `csize` consecutive signatures (csize = n: the one whole-batch equation).  Everything that
     * depends on the chunking is built here: the key groups (a key that occurs in two chunks is two groups) and their decodes, the
     * per-group scalar sums, both sorted pair lists, the bucket sums, one verdict per chunk. */
    auto equations = [&](size_t csize, bool first) -> bool {
        const uint32_t nch = (uint32_t)((n + csize - 1) / csize);
        auto log2_floor = [](size_t v) { int l = 0; while (((size_t)2 << l) <= v) l++; return l; };
        /* digit widths of a chunked pass: with many chunks the lanes are plentiful, so the widths minimise additions (bucket
         * accumulation + folding = count + 2 * 2^c per window) instead of filling one wave: ~16 points per R bucket, ~8 per key bucket */
        rlc_shape sh_r = rlc_shape_for(csize, nch > 1 ? std::max(2, std::min((int)RLC_MAX_C, log2_floor(csize) - 4)) : 0, 0);
        sh_r.nch = nch; sh_r.csize = (uint32_t)csize;
        if (first) zbits = sh_r.zbits;
        else sh_r.wn = (zbits + sh_r.c - 1) / sh_r.c;        /* the weights were drawn for the first pass: the digits must cover all of their bits */
        const uint32_t cells = rlc_scells(sh_r);
        unsigned long long *s_acc = k.out<unsigned long long>((size_t)RLC_ACC_WORDS * cells * nch);
        RlcClass cr, ck;
        if (!rlc_class_alloc(k, cr, sh_r, n)) return false;
        CU(cudaMemsetAsync(flags, 0, (2 + (size_t)nch) * sizeof(uint32_t), s));
        CU(cudaMemsetAsync(s_acc, 0, sizeof(unsigned long long) * RLC_ACC_WORDS * cells * nch, s));
        /* Two streams.  Main: the multiplier-bound work -- the R decodes as the signatures land, later the bucket sums of the R class.
         * Side (high priority): what needs no decoded R -- the weights and the sorted pair list of the R class (they depend on the
         * seed alone; excluded signatures are skipped by the bucket kernel), the key grouping and the key decodes, the challenge
         * hashes (ALU work, it shares the SMs with the decodes) -- and later the whole key class, whose kernels are short chains of
         * dependent additions and doublings (latency-bound: up to 446 - c doublings in a row). */
        CU(cudaEventRecord(c.side_evt[0], s));
        CU(cudaStreamWaitEvent(side, c.side_evt[0], 0)); /* whatever produced the inputs on `s`, and the seed */
        if (first) {
            LaneRlcZ f3 = {z, dseed, n, sh_r.zbits};         /* zbits = 9 x 15 = 135 for the whole-batch shape: enough for any later digit width */
            if (!launch(c, f3, (n + RLC_Z_PER_LANE - 1) / RLC_Z_PER_LANE, side)) return false;
        }
        if (!rlc_class_pairs(c, cr, z, RLC_ZWORDS, 0, side, nullptr)) return false;
        if (first) {
            const size_t s0 = feed ? feed->split[0] : n, s1 = feed ? feed->split[1] : n;
            const size_t lo[3] = {0, s0, s1}, hi[3] = {s0, s1, n};
            const rlc_groups no_groups = {nullptr, nullptr, nullptr, 0};
            for (int h = 0; h < 3; h++) {
                if (feed) CU(cudaStreamWaitEvent(s, h == 0 ? feed->sig0 : h == 1 ? feed->sig1 : feed->rest, 0));
                if (hi[h] == lo[h]) continue;
                LaneRlcDecode f1 = {pts, ok, flags, dsig, dpk, n, no_groups, lo[h]}; /* lanes below n never look at the groups */
                if (!launch(c, f1, hi[h] - lo[h], s)) return false;
            }
            if (feed) CU(cudaStreamWaitEvent(side, feed->keys, 0));
        }
        key_groups kg;
        uint64_t launched = 0;
        cudaError_t e = group_keys_all(dpk, n, gs, &kg, side, &launched, nch > 1 ? (uint32_t)csize : 0u);
        if (e != cudaSuccess) return fail("group_keys_all", e);
        g_launches += launched;
        uint32_t m = 0;
        CU(cudaMemcpyAsync(&m, kg.ngroups, sizeof m, cudaMemcpyDeviceToHost, side));
        CU(cudaStreamSynchronize(side)); /* the number of key groups sizes the key class; the R decodes are already queued */
        if (m == 0 || m > n) { g_err = "rlc: key grouping returned an impossible group count"; return false; }
        const rlc_groups g = {kg.order, kg.gid, kg.gstart, m};
        const size_t nkey = (size_t)m + nch;                                 /* key groups, then the B of every chunk */
        rlc_shape sh_k = rlc_shape_for((nkey + nch - 1) / nch, nch > 1 ? std::max(2, std::min((int)RLC_MAX_C, log2_floor((nkey + nch - 1) / nch) - 3)) : 0, 1);
        sh_k.nch = nch; sh_k.csize = (uint32_t)csize;
        unsigned long long *key_acc = k.out<unsigned long long>((size_t)RLC_ACC_WORDS * m);
        uint32_t *kscal = k.out<uint32_t>(SC_WORDS * nkey), *kchunk = k.out<uint32_t>(nkey);
        if (!rlc_class_alloc(k, ck, sh_k, nkey)) return false;
        CU(cudaMemsetAsync(key_acc, 0, sizeof(unsigned long long) * RLC_ACC_WORDS * m, side));
        e = key_chunks(kchunk, &kg, m, nch, nch > 1 ? (uint32_t)csize : 0u, side);
        if (e != cudaSuccess) return fail("key_chunks", e);
        g_launches++;
        LaneRlcDecode fk = {pts, ok, flags, dsig, dpk, n, g, n};
        if (!launch(c, fk, nkey, side)) return false;
        /* the key class from its scalars to its totals, on `side` */
        auto key_class = [&]() -> bool {
            LaneRlcKeyScalars f5 = {kscal, key_acc, s_acc, m, cells};
            if (!launch(c, f5, nkey, side)) return false;
            if (!rlc_class_pairs(c, ck, kscal, SC_WORDS, n, side, kchunk)) return false;
            CU(cudaEventRecord(c.side_evt[4], side));
            if (!rlc_class_sum(c, ck, pts, side, false, nullptr)) return false;
            CU(cudaEventRecord(c.side_evt[3], side));
            return true;
        };
        if (first) {
            /* whole-batch pass: the key class does not wait for the R decodes.  The scalar sums are taken as soon as the key decodes and
             * the challenge hashes are in (a signature counts if its KEY decodes), the key class runs on them beside the decodes, and
             * LaneRlcLate settles the rest: it writes `valid` and takes a signature whose R does not decode out of the sums again, raising
             * the redo flag -- then the key class (only) is run once more on the corrected sums, below.  Never on honest traffic. */
            if (feed) CU(cudaStreamWaitEvent(side, feed->rest, 0));
            LaneEdVerifyScalars f2 = {chal, resp, dsig, dpk, dmsg, doff, prehashed, dctx, ctx_len, 0};
            if (!launch(c, f2, n, side)) return false;
            LaneRlcWeights f4 = {z, valid, key_acc, s_acc, chal, resp, ok, n, g, sh_r, 1u};
            if (!launch(c, f4, n, side)) return false;
            CU(cudaEventRecord(c.side_evt[1], side));
            if (!key_class()) return false;
            CU(cudaStreamWaitEvent(s, c.side_evt[1], 0));          /* behind the R decodes on `s` */
            LaneRlcLate fl = {z, valid, key_acc, s_acc, chal, resp, ok, n, g, sh_r, flags + 1 + nch};
            if (!launch(c, fl, n, s)) return false;
        } else {
            CU(cudaEventRecord(c.side_evt[1], side));
            CU(cudaStreamWaitEvent(s, c.side_evt[1], 0));
            LaneRlcWeights f4 = {z, valid, key_acc, s_acc, chal, resp, ok, n, g, sh_r, 0u};
            if (!launch(c, f4, n, s)) return false;
            CU(cudaEventRecord(c.side_evt[2], s));
            CU(cudaStreamWaitEvent(side, c.side_evt[2], 0));
            if (!key_class()) return false;
        }
        CU(cudaStreamWaitEvent(s, c.side_evt[4], 0)); /* the radix sort of the key class wants the whole machine for its 0.3 ms: the R buckets wait for it */
        if (!rlc_class_sum(c, cr, pts, s, true, valid)) return false;
        CU(cudaStreamWaitEvent(s, c.side_evt[3], 0));
        LaneRlcVerdict f11 = {flags + 1, cr.total, ck.total, flags};
        if (!launch(c, f11, nch, s)) return false;
        hflags.assign(2 + (size_t)nch, 0);
        CU(cudaMemcpyAsync(hflags.data(), flags, hflags.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        if (first && hflags[1 + nch]) { /* an R that does not decode under a key that does: the key class again, on the corrected sums */
            CU(cudaEventRecord(c.side_evt[2], s));
            CU(cudaStreamWaitEvent(side, c.side_evt[2], 0));
            if (!key_class()) return false;
            CU(cudaStreamWaitEvent(s, c.side_evt[3], 0));
            if (!launch(c, f11, nch, s)) return false;
            CU(cudaMemcpyAsync(hflags.data(), flags, hflags.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
            CU(cudaStreamSynchronize(s));
        }
        return true;
    };
    if (!equations(n, true)) return false;
    if (hflags[1]) {
        *fast = 1;
        CU(cudaMemcpyAsync(dst, valid, sizeof(int32_t) * n, cudaMemcpyDeviceToDevice, s));
        return true;
    }
    /* the whole-batch equation failed: localise.  Chunk size from the batch (about RLC_CHUNK_TARGET signatures, at most RLC_MAX_CHUNKS chunks). */
    size_t csize = RLC_CHUNK_TARGET;
    if (const char *e = getenv("GOLDILOCKS_B200_RLC_CHUNK")) { const long v = atol(e); if (v >= (long)RLC_MIN) csize = (size_t)v; }
    if ((n + csize - 1) / csize > RLC_MAX_CHUNKS) csize = (n + RLC_MAX_CHUNKS - 1) / RLC_MAX_CHUNKS;
    const uint32_t nch = (uint32_t)((n + csize - 1) / csize);
    if (hflags[0] || nch < 4 || csize < RLC_MIN) return ordinary();      /* a decoded Z = 0 (never for a curve point), or nothing to localise */
    if (!equations(csize, false)) return false;
    std::vector<uint32_t> failed;
    for (uint32_t ch = 0; ch < nch; ch++) if (!hflags[1 + ch]) failed.push_back(ch);
    /* Both passes are spent by now; what is left to decide is how to finish THIS call and whether to try again on the NEXT ones.  The
     * packed per-signature pass over a fraction f of the batch costs about f of the ordinary call, so it wins up to f ~ 0.9.  But a call
     * that had to run both passes plus a fallback over more than a fifth of the batch was slower than the ordinary path would have been
     * (two passes ~ 2/3 of an ordinary call): traffic like that should skip the equation for a while. */
    if (failed.size() * 5 > nch) { const unsigned rp = g_rlc_reprobe.load(); c.rlc_skip = rp ? rp - 1 : 0; }
    if (hflags[0] || failed.size() * 10 > (size_t)nch * 9) return ordinary();
    *fast = 2;
    CU(cudaMemcpyAsync(dst, valid, sizeof(int32_t) * n, cudaMemcpyDeviceToDevice, s));  /* chunks whose equation held: decided */
    if (failed.empty()) return true;                                   /* (cannot happen unless the first equation failed on its own) */
    size_t np = 0;
    for (uint32_t ch : failed) np += ((size_t)ch * csize + csize <= n) ? csize : n - (size_t)ch * csize;
    size_t total = 0;
    CU(cudaMemcpyAsync(&total, doff + n, sizeof(size_t), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    uint32_t *fc = k.out<uint32_t>(failed.size());
    size_t *mbase = k.out<size_t>(failed.size() + 1), *poff = k.out<size_t>(np + 1);
    uint8_t *psig = k.out<uint8_t>(114 * np), *ppk = k.out<uint8_t>(57 * np), *pmsg = k.out<uint8_t>(total);
    uint32_t *src = k.out<uint32_t>(np);
    int32_t *pst = k.out<int32_t>(np);
    if (!k.ok) return false;
    CU(cudaMemcpyAsync(fc, failed.data(), failed.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    LaneRlcPackPlan fp = {mbase, fc, (uint32_t)failed.size(), doff, n, (uint32_t)csize};
    if (!launch(c, fp, 1, s)) return false;
    LaneRlcPack fq = {psig, ppk, pmsg, poff, src, dsig, dpk, dmsg, doff, mbase, fc, (uint32_t)failed.size(), np, (uint32_t)csize};
    if (!launch(c, fq, np + 1, s)) return false;
    CU(cudaStreamSynchronize(s));                                      /* `failed` (host vector) must outlive its copy */
    if (!ordinary_on(pst, psig, ppk, pmsg, poff, np)) return false;
    LaneRlcUnpack fu = {dst, pst, src};
    return launch(c, fu, np, s);
}
void goldilocks_b200_rlc_policy(unsigned reprobe) {
    g_rlc_reprobe.store(reprobe);
    for (int d = 0; d < MAX_DEV; d++)
        for (int l = 0; l < shard::LANES; l++) { std::lock_guard<std::mutex> g(g_ctx[d][l].mu); g_ctx[d][l].rlc_skip = 0; }
}
goldilocks_error_t goldilocks_ed448_verify_rlc_batch(goldilocks_error_t *status, const uint8_t *signature, const uint8_t *pubkey, const uint8_t *msg, const size_t *msg_off,
                                                     uint8_t prehashed, const uint8_t *context, uint8_t context_len, size_t n, int *fast_path) {
    if (n == 0) { if (fast_path) *fast_path = 0; return GOLDILOCKS_SUCCESS; }
    if (auto pool_ = shard_pool(n, false, 0)) { /* every range decides its own equation; fast_path = 1 iff all of them did */
        std::atomic<int> slow{0};
        std::atomic<int> *slowp = &slow;
        goldilocks_error_t r = shard_go(pool_, n, false, 0, [=](size_t lo, size_t m) {
            int f = 0;
            goldilocks_error_t e = goldilocks_ed448_verify_rlc_batch(status + lo, signature + 114 * lo, pubkey + 57 * lo, msg + msg_off[lo], SubOffsets(msg_off, lo, m).v.data(),
                                                                     prehashed, context, context_len, m, &f);
            if (!f) slowp->fetch_add(1);
            return e;
        });
        if (fast_path) *fast_path = slow.load() == 0 ? 1 : 0;
        return r;
    }
    {   /* recent calls on this context failed most of their chunks: this one goes straight to the ordinary entry point (rlc_core explains) */
        int dev = 0;
        if (cudaGetDevice(&dev) == cudaSuccess && dev < MAX_DEV) {
            Ctx &cx = g_ctx[dev][my_lane()];
            bool skip = false;
            { std::lock_guard<std::mutex> g(cx.mu); if (cx.rlc_skip > 0) { cx.rlc_skip--; skip = true; } }
            if (skip) {
                if (fast_path) *fast_path = 0;
                return goldilocks_ed448_verify_batch(status, signature, pubkey, msg, msg_off, prehashed, context, context_len, n);
            }
        }
    }
    Call k;
    int fast = 0;
    size_t total = n ? msg_off[n] : 0;
    size_t *doff = k.out<size_t>(n + 1);
    uint8_t *dctx = k.out<uint8_t>(context_len), *dpk = k.out<uint8_t>(57 * n), *dsig = k.out<uint8_t>(114 * n), *dmsg = k.out<uint8_t>(total);
    int32_t *dst = k.out<int32_t>(n);
    /* a quarter of the signatures first (the R decodes start half a millisecond into the call), the keys, the second quarter, the rest */
    const bool chunked = n >= 4 * RLC_MIN;
    RlcFeed feed = {{chunked ? n / 4 : n, chunked ? n / 2 : n}, nullptr, nullptr, nullptr, nullptr};
    if (k.ok) {
        feed.sig0 = k.c->copy_done[0]; feed.keys = k.c->copy_done[1]; feed.sig1 = k.c->copy_done[2]; feed.rest = k.c->copy_done[3];
        k.push(dsig, signature, 114 * feed.split[0]);
        if (k.ok && cudaEventRecord(feed.sig0, k.c->copy_stream) != cudaSuccess) k.ok = false;
        k.push(dpk, pubkey, 57 * n);
        k.push(doff, msg_off, n + 1);
        k.push(dctx, context, context_len);
        if (k.ok && cudaEventRecord(feed.keys, k.c->copy_stream) != cudaSuccess) k.ok = false;
        k.push(dsig + 114 * feed.split[0], signature + 114 * feed.split[0], 114 * (feed.split[1] - feed.split[0]));
        if (k.ok && cudaEventRecord(feed.sig1, k.c->copy_stream) != cudaSuccess) k.ok = false;
        k.push(dsig + 114 * feed.split[1], signature + 114 * feed.split[1], 114 * (n - feed.split[1]));
        k.push(dmsg, msg, total);
        if (k.ok && cudaEventRecord(feed.rest, k.c->copy_stream) != cudaSuccess) k.ok = false;
    }
    if (k.ok && n) k.ok = rlc_core(k, dst, dsig, dpk, dmsg, doff, prehashed, dctx, context_len, n, k.c->stream, &fast, &feed);
    k.fetch((int32_t *)status, dst, n);
    if (!k.ok && k.c) { cudaStreamSynchronize(k.c->copy_stream); cudaStreamSynchronize(k.c->side_stream); }
    if (fast_path) *fast_path = fast;
    return k.finish();
}
goldilocks_error_t goldilocks_ed448_verify_rlc_batch_dev(goldilocks_error_t *status, const uint8_t *signature, const uint8_t *pubkey, const uint8_t *msg, const size_t *msg_off,
                                                         uint8_t prehashed, const uint8_t *context, uint8_t context_len, size_t n, void *stream, int *fast_path) {
    /* device pointers; scratch comes from the library's arena (the call holds the device lock) and the call synchronises
     * `stream` twice (the number of distinct keys, the verdict): it returns with the statuses written */
    Call k;
    int fast = 0;
    cudaStream_t s = as_stream(stream);
    if (k.ok && n) {
        if (cudaStreamSynchronize(k.c->stream) != cudaSuccess) k.ok = false; /* arena reuse: nothing of an earlier call may still run */
        if (k.ok) k.ok = rlc_core(k, (int32_t *)status, signature, pubkey, msg, msg_off, prehashed, context, context_len, n, s, &fast);
        if (cudaStreamSynchronize(s) != cudaSuccess || cudaStreamSynchronize(k.c->side_stream) != cudaSuccess) k.ok = false;
    }
    if (fast_path) *fast_path = fast;
    return k.finish();
}

// ---- device-resident sets: tables built once on one device and used by many calls (key, X448 peer, decaf peer and point sets) --
extern "C++" {   /* the helpers shared by the sets are templates */
/* What every set struct inherits: the device it belongs to, its size m and the device buffers it owns.  The handles are opaque in
 * the header, so each *_destroy is `delete`; the destructor frees the buffers on the set's own device, whichever is current. */
struct DeviceSet {
    static constexpr int MAX_BUFFERS = 4;   /* a key set's pk, key_ok, ktabs and sorted */
    int dev; size_t m;
    void *owned[MAX_BUFFERS] = {};
    int n_owned = 0;
    DeviceSet(int dev, size_t m) : dev(dev), m(m) {}
    DeviceSet(const DeviceSet &) = delete;
    DeviceSet &operator=(const DeviceSet &) = delete;
    ~DeviceSet() {
        int cur = 0;
        const bool sw = cudaGetDevice(&cur) == cudaSuccess && cur != dev && cudaSetDevice(dev) == cudaSuccess;
        for (int i = 0; i < n_owned; i++) cudaFree(owned[i]);
        if (sw) cudaSetDevice(cur);
    }
    template <class T> bool alloc(T **p, size_t count) {
        if (n_owned == MAX_BUFFERS || cudaMalloc(p, sizeof(T) * count) != cudaSuccess) return false;
        owned[n_owned++] = *p;
        return true;
    }
};
/* the end of every *_create: on failure `err` (unless the call set its own) and the set freed, else the set in *out */
template <class S>
static goldilocks_error_t finish_create(Call &k, bool ok, S *s, S **out, const char *err) {
    const goldilocks_error_t r = k.finish();
    if (!ok || r != GOLDILOCKS_SUCCESS) {
        if (!ok) g_err = err;
        delete s;
        return GOLDILOCKS_FAILURE;
    }
    *out = s;
    return GOLDILOCKS_SUCCESS;
}
/* The checks of a call on a set, each overload adding one: the set belongs to the calling device; the batch has fewer than 2^31
 * elements; the caller passed scratch. */
template <class S> static bool set_call(const S *s, int dev, const char *fn) {
    if (s && s->dev == dev) return true;
    g_err = std::string(fn) + ": the " + S::noun + " lives on another device";
    return false;
}
template <class S> static bool set_call(const S *s, int dev, const char *fn, size_t n) {
    if (!set_call(s, dev, fn)) return false;
    if (n > (size_t)INT32_MAX) { g_err = std::string(fn) + ": n >= 2^31"; return false; }
    return true;
}
template <class S> static bool set_call(const S *s, int dev, const char *fn, size_t n, const void *scratch) {
    if (!set_call(s, dev, fn, n)) return false;
    if (!scratch) { g_err = std::string(fn) + ": no scratch"; return false; }
    return true;
}
/* the persistent kernel of a set's layout over n elements: make(std::true_type{}) / make(std::false_type{}) returns the functor of
 * the flat / the compact kernel */
template <class Make>
static bool launch_layout(Ctx &c, bool flat, size_t n, cudaStream_t st, unsigned *counter, const Make &make) {
    auto go = [&](auto f) {
        int grid = 1;
        return smp_grid<decltype(f)>(c, &grid) && launch_smp(c, f, n, grid, st, counter);
    };
    return flat ? go(make(std::true_type{})) : go(make(std::false_type{}));
}
/* the reference's (5,5,18) comb tables of `count` points (X448 and decaf peer sets), as affine niels */
static void comb_tables(Call &k, const abi_pt *pts, niels *out, size_t count) {
    LanePrecompute fp = {k.out<abi_niels>(COMB_ENTRIES * count), pts, k.out<niels>(16 * COMB_N * count)};
    k.run(fp, COMB_N * count);
    LaneNielsFromAbi fc = {out, fp.tables};
    k.run(fc, COMB_ENTRIES * count);
}
/* the scratch of one call's ordering, carved from `base` (null: sizes only): sort keys and values in and out, CUB's temporary storage */
struct OrderScratch { uint32_t *keys, *vals, *keys_s, *order; void *sort_tmp; size_t sort_bytes; };
static size_t order_scratch(OrderScratch *s, void *base, size_t n) {
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t words = al(sizeof(uint32_t) * n), sort_bytes = pair_sort_scratch_bytes(n);
    if (s) {
        char *p = (char *)base;
        s->keys = (uint32_t *)p; s->vals = (uint32_t *)(p + words); s->keys_s = (uint32_t *)(p + 2 * words); s->order = (uint32_t *)(p + 3 * words);
        s->sort_tmp = p + 4 * words; s->sort_bytes = sort_bytes;
    }
    return 4 * words + al(sort_bytes);
}
/* s.order = the elements sorted by set entry: keys (min(index[j], m), j) -> stable radix sort.  Decaf peer sets, point sets and
 * key-set lookup order every call this way.  The sort is bracketed like a launch when profiling is on, so
 * goldilocks_b200_profile_timeline shows its share of the call. */
static bool set_order(Ctx &c, const uint32_t *index, uint32_t m, size_t n, const OrderScratch &s, cudaStream_t st, const char *what) {
    LaneDecafPeerKeys fk = {s.keys, s.vals, index, m};
    if (!launch(c, fk, n, st)) return false;
    int key_bits = 1;
    while (key_bits < 32 && (m >> key_bits)) key_bits++;   /* the bit length of m, the largest key */
    cudaEvent_t a = nullptr, b = nullptr;
    const bool prof = g_prof_on.load() != 0;
    if (prof) a = prof_begin("pair_sort", st, &b);
    const cudaError_t e = pair_sort(s.sort_tmp, s.sort_bytes, s.keys, s.keys_s, s.vals, s.order, n, key_bits, st);
    if (prof) prof_end("pair_sort", st, a, b);
    if (e != cudaSuccess) return fail(what, e);
    return true;
}
static size_t order_scratch_bytes(size_t n) { return dev_ctx() ? order_scratch(nullptr, nullptr, n) : 0; }
}  // extern "C++"

// ---- key sets: per-key verification tables that outlive a call (SURVEY 8(f)4) ---------------------------------------
struct goldilocks_b200_keyset_s : DeviceSet {
    static constexpr const char *noun = "key set";
    uint8_t *pk;      /* m x 57 key bytes (the challenge hashes them) */
    int32_t *key_ok;  /* decode status per key */
    uint4 *ktabs;     /* m tables of KTAB_QUADS quads (10 columns x 9 rows), or of KSET_QUADS (flat: a column per digit position) */
    bool flat;
    uint32_t *sorted; /* the m indices ordered by key bytes (memcmp), ties by index: the lookup calls' binary search (LaneKeysetLookup) */
};
/* A set whose flat tables (369 KB per key) fit this many bytes gets them; larger sets keep the 41 KB layout (goldilocks_b200_keyset_policy) */
std::atomic<unsigned long long> g_keyset_flat_bytes{32ull << 30};
void goldilocks_b200_keyset_policy(unsigned long long max_table_bytes) { g_keyset_flat_bytes.store(max_table_bytes); }
static bool keyset_flat(size_t tables) { return (unsigned long long)tables * KSET_QUADS * sizeof(uint4) <= g_keyset_flat_bytes.load(); }
/* the per-key tables of `count` points into ktabs (key sets and point sets): the flat layout's doubling chain and 90 column tables, or
 * the ten-column layout; then affine entries -- the set pays one inversion per column once, every call saves a multiplication per addition */
static void keyset_tables(Call &k, const abi_pt *pts, uint4 *ktabs, size_t count, bool flat) {
    if (flat) {
        int grid = k.smp_grid_for<SlotKeysetChain>();
        SlotKeysetChain fc = {pts, ktabs};
        k.run_smp(fc, count, grid);
        grid = k.smp_grid_for<SlotKeysetColumns>();
        SlotKeysetColumns fcol = {ktabs, k.slots((size_t)grid * SLOT_BLOCK, 1)};
        k.run_smp(fcol, count * KSET_COLS, grid);
    } else {
        int grid = k.smp_grid_for<SlotKeysetTables>();
        SlotKeysetTables ft = {pts, ktabs};
        k.run_smp(ft, count, grid);
    }
    LaneKeysetNormalize fn = {ktabs, flat ? (uint32_t)KSET_COLS : (uint32_t)VSH_CHUNKS, flat ? (uint32_t)KSET_QUADS : (uint32_t)KTAB_QUADS};
    k.run(fn, count * (flat ? KSET_COLS : VSH_CHUNKS));
}
goldilocks_error_t goldilocks_b200_keyset_create(goldilocks_b200_keyset **out, const uint8_t *pubkeys, size_t m) {
    if (!out) return GOLDILOCKS_FAILURE;
    *out = nullptr;
    Call k;
    if (!k.ok) return k.finish();
    const size_t mm = m ? m : 1;
    const bool flat = keyset_flat(mm);
    goldilocks_b200_keyset_s *ks = new goldilocks_b200_keyset_s{{k.c->dev, m}, nullptr, nullptr, nullptr, flat, nullptr};
    bool ok = ks->alloc(&ks->pk, 57 * mm) && ks->alloc(&ks->key_ok, mm) && ks->alloc(&ks->ktabs, mm * (flat ? KSET_QUADS : KTAB_QUADS)) &&
              ks->alloc(&ks->sorted, mm);
    /* the bytes are on the host already: sort there (a byte order, not a hash order -- nobody can make the search longer) */
    std::vector<uint32_t> sorted(m);
    for (size_t i = 0; i < m; i++) sorted[i] = (uint32_t)i;
    std::stable_sort(sorted.begin(), sorted.end(), [pubkeys](uint32_t a, uint32_t b) { return memcmp(pubkeys + 57 * (size_t)a, pubkeys + 57 * (size_t)b, 57) < 0; });
    if (ok && m) {
        ok = cudaMemcpyAsync(ks->pk, pubkeys, 57 * m, cudaMemcpyHostToDevice, k.c->stream) == cudaSuccess &&
             cudaMemcpyAsync(ks->sorted, sorted.data(), sizeof(uint32_t) * m, cudaMemcpyHostToDevice, k.c->stream) == cudaSuccess;
        abi_pt *pts = k.out<abi_pt>(m);
        LaneDecodeEddsa fd = {pts, ks->key_ok, ks->pk};
        k.run(fd, m);
        keyset_tables(k, pts, ks->ktabs, m, flat);
    }
    return finish_create(k, ok, ks, out, "goldilocks_b200_keyset_create: device allocation or copy failed");
}
void goldilocks_b200_keyset_destroy(goldilocks_b200_keyset *ks) { delete ks; }
size_t goldilocks_b200_keyset_size(const goldilocks_b200_keyset *ks) { return ks ? ks->m : 0; }
/* the index form on device buffers: challenges under the set's key bytes, the finish kernel of the set's layout, the sign check */
static bool keyset_enqueue(Ctx &c, int32_t *status, const goldilocks_b200_keyset_s *ks, const uint32_t *key_index, const uint8_t *sig, const uint8_t *msg,
                           const size_t *off, uint8_t prehashed, const uint8_t *ctx, uint8_t ctx_len, size_t n, abi_sc *chal, abi_sc *resp, verify_aux *aux,
                           cudaStream_t st, unsigned *counter) {
    LaneEdVerifyScalars f2 = {chal, resp, sig, ks->pk, msg, off, prehashed, ctx, ctx_len, 0, key_index, (uint32_t)ks->m};
    if (!launch(c, f2, n, st)) return false;
    if (!launch_layout(c, ks->flat, n, st, counter, [&](auto flat) {
            return SlotEdVerifyFinishKeysetLayout<decltype(flat)::value>{aux, ks->key_ok, chal, resp, c.wide, ks->ktabs, key_index, (uint32_t)ks->m, sig};
        }))
        return false;
    LaneVerifySign fv = {status, aux, 1, n};
    return launch(c, fv, (n + VSIGN_BATCH - 1) / VSIGN_BATCH, st);
}
goldilocks_error_t goldilocks_ed448_verify_keyset_batch(goldilocks_error_t *status, const goldilocks_b200_keyset *ks, const uint32_t *key_index,
                                                        const uint8_t *signature, const uint8_t *msg, const size_t *msg_off, uint8_t prehashed,
                                                        const uint8_t *context, uint8_t context_len, size_t n) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Call k;
    if (!k.ok) return k.finish();
    if (!set_call(ks, k.c->dev, "goldilocks_ed448_verify_keyset_batch")) return GOLDILOCKS_FAILURE;
    const size_t total = n ? msg_off[n] : 0;
    const size_t *doff = k.in(msg_off, n + 1);
    const uint8_t *dctx = k.in(context, context_len);
    const uint32_t *dki = k.in(key_index, n);
    const uint8_t *dsig = k.in(signature, 114 * n), *dmsg = k.in(msg, total);
    int32_t *dst = k.out<int32_t>(n);
    abi_sc *chal = k.out<abi_sc>(n), *resp = k.out<abi_sc>(n);
    verify_aux *aux = k.out<verify_aux>(n);
    if (k.ok) k.ok = keyset_enqueue(*k.c, dst, ks, dki, dsig, dmsg, doff, prehashed, dctx, context_len, n, chal, resp, aux, k.c->stream, nullptr);
    k.fetch((int32_t *)status, dst, n);
    return k.finish();
}

// ---- X448 peer sets: per-peer comb tables for key agreement with recurring public keys (slot_lanes.cuh SlotX448Peer) -------
struct goldilocks_b200_x448_peerset_s : DeviceSet {
    static constexpr const char *noun = "peer set";
    uint8_t *peers;     /* m x 56 u bytes: what the ladder reads for the peers that keep it */
    int32_t *table_ok;  /* per peer: SUCCESS = the comb table is valid (public) */
    niels *tables;      /* m tables of COMB_ENTRIES affine niels, 15 360 bytes each */
    uint32_t *sorted;   /* the m indices ordered by peer bytes (memcmp), ties by index: the lookup calls' binary search (LaneX448PeerLookup) */
};
goldilocks_error_t goldilocks_b200_x448_peerset_create(goldilocks_b200_x448_peerset **out, const uint8_t *peers, size_t m) {
    if (!out) return GOLDILOCKS_FAILURE;
    *out = nullptr;
    Call k;
    if (!k.ok) return k.finish();
    const size_t mm = m ? m : 1;
    goldilocks_b200_x448_peerset_s *ps = new goldilocks_b200_x448_peerset_s{{k.c->dev, m}, nullptr, nullptr, nullptr, nullptr};
    bool ok = m <= UINT32_MAX && ps->alloc(&ps->peers, 56 * mm) && ps->alloc(&ps->table_ok, mm) && ps->alloc(&ps->tables, mm * COMB_ENTRIES) &&
              ps->alloc(&ps->sorted, mm);
    std::vector<uint32_t> sorted;   /* lives until finish_create has synchronised the copy from it */
    if (ok && m) {
        ok = cudaMemcpyAsync(ps->peers, peers, 56 * m, cudaMemcpyHostToDevice, k.c->stream) == cudaSuccess;
        abi_pt *pts = k.out<abi_pt>(m);
        LaneX448PeerLift fl = {pts, ps->table_ok, ps->peers};
        k.run(fl, m);
        comb_tables(k, pts, ps->tables, m);
        /* the byte order for the lookup calls, sorted on the host while the lift and the tables run (as goldilocks_b200_keyset_create) */
        sorted.resize(m);
        for (size_t i = 0; i < m; i++) sorted[i] = (uint32_t)i;
        std::stable_sort(sorted.begin(), sorted.end(), [peers](uint32_t a, uint32_t b) { return memcmp(peers + 56 * (size_t)a, peers + 56 * (size_t)b, 56) < 0; });
        ok = ok && cudaMemcpyAsync(ps->sorted, sorted.data(), sizeof(uint32_t) * m, cudaMemcpyHostToDevice, k.c->stream) == cudaSuccess;
    }
    return finish_create(k, ok, ps, out, "goldilocks_b200_x448_peerset_create: device allocation or copy failed");
}
void goldilocks_b200_x448_peerset_destroy(goldilocks_b200_x448_peerset *ps) { delete ps; }
size_t goldilocks_b200_x448_peerset_size(const goldilocks_b200_x448_peerset *ps) { return ps ? ps->m : 0; }
goldilocks_error_t goldilocks_x448_peerset_batch(uint8_t *out, goldilocks_error_t *status, const goldilocks_b200_x448_peerset *ps, const uint32_t *peer_index,
                                                 const uint8_t *scalar, size_t n) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Call k;
    if (!k.ok) return k.finish();
    if (!set_call(ps, k.c->dev, "goldilocks_x448_peerset_batch")) return GOLDILOCKS_FAILURE;
    SlotX448Peer f = {k.secret(k.out<uint8_t>(56 * n), 56 * n), k.out<int32_t>(n), ps->tables, ps->table_ok, ps->peers, k.in(peer_index, n),
                      k.secret(k.in(scalar, 56 * n), 56 * n), (uint32_t)ps->m};
    k.run_sm(f, n);
    k.fetch(out, f.out, 56 * n);
    k.fetch((int32_t *)status, f.status, n);
    return k.finish();
}

/* X448 against the set by the peers' bytes: looked-up indices into idx (LaneX448PeerLookup), the batch ordered by them (hits grouped
 * by peer, the misses as one tail), then one kernel in which the hits with a table run its comb and everything else the ladder.
 * No read-back: the misses need no packing, so the call stays asynchronous. */
static size_t x448_peer_lookup_scratch(OrderScratch *s, uint32_t **idx, void *base, size_t n) {
    const size_t order_bytes = order_scratch(s, base, n);
    if (idx) *idx = (uint32_t *)((char *)base + order_bytes);
    return order_bytes + ((sizeof(uint32_t) * n + 255) & ~(size_t)255);
}
static bool x448_peer_lookup_enqueue(Ctx &c, uint8_t *out, int32_t *status, uint32_t *idx, const goldilocks_b200_x448_peerset_s *ps, const uint8_t *base,
                                     const uint8_t *scalar, size_t n, const OrderScratch &s, cudaStream_t st) {
    const uint32_t m = (uint32_t)ps->m;
    LaneX448PeerLookup fl = {idx, base, ps->peers, ps->sorted, m};
    if (!launch(c, fl, n, st) || !set_order(c, idx, m, n, s, st, "pair_sort (X448 peer set lookup)")) return false;
    SlotX448PeerLookup f = {out, status, ps->tables, ps->table_ok, idx, s.order, base, scalar, m};
    return launch_slots(c, f, n, st);
}
goldilocks_error_t goldilocks_x448_peerset_lookup_batch(uint8_t *out, goldilocks_error_t *status, uint32_t *peer_index, const goldilocks_b200_x448_peerset *ps,
                                                        const uint8_t *base, const uint8_t *scalar, size_t n) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Call k;
    if (!k.ok) return k.finish();
    if (!set_call(ps, k.c->dev, "goldilocks_x448_peerset_lookup_batch", n)) return GOLDILOCKS_FAILURE;
    uint8_t *dout = k.secret(k.out<uint8_t>(56 * n), 56 * n);
    int32_t *dst = k.out<int32_t>(n);
    const uint8_t *dbase = k.in(base, 56 * n);
    const uint8_t *dsc = k.secret(k.in(scalar, 56 * n), 56 * n);
    OrderScratch s = {};
    uint32_t *idx = nullptr;
    void *scratch = k.alloc(x448_peer_lookup_scratch(nullptr, nullptr, nullptr, n));
    if (k.ok) x448_peer_lookup_scratch(&s, &idx, scratch, n);
    if (k.ok) k.ok = x448_peer_lookup_enqueue(*k.c, dout, dst, idx, ps, dbase, dsc, n, s, k.c->stream);
    k.fetch(out, dout, 56 * n);
    k.fetch((int32_t *)status, dst, n);
    if (peer_index) k.fetch(peer_index, idx, n);
    return k.finish();
}

// ---- decaf peer sets: per-peer comb tables for goldilocks_448_direct_scalarmul against recurring points (slot_lanes.cuh SlotDecafPeer)
struct goldilocks_b200_decaf_peerset_s : DeviceSet {
    static constexpr const char *noun = "peer set";
    int32_t *peer_ok;   /* m + 1 decode statuses (public); entry m, the base point with FAILURE, stands for every index >= m */
    niels *tables;      /* m + 1 tables of COMB_ENTRIES affine niels, 15 360 bytes each */
};
/* the sort by peer, then the comb kernel over the elements in that order */
static bool decaf_peer_enqueue(Ctx &c, uint8_t *scaled, int32_t *status, const goldilocks_b200_decaf_peerset_s *ps, const uint32_t *peer_index,
                               const abi_sc *scalar, bool short_circuit, size_t n, const OrderScratch &s, cudaStream_t st) {
    const uint32_t m = (uint32_t)ps->m;
    if (!set_order(c, peer_index, m, n, s, st, "pair_sort (decaf peer set)")) return false;
    SlotDecafPeer f = {scaled, status, ps->tables, ps->peer_ok, peer_index, s.order, scalar, m, short_circuit ? ~0u : 0u};
    return launch_slots(c, f, n, st);
}
goldilocks_error_t goldilocks_b200_decaf_peerset_create(goldilocks_b200_decaf_peerset **out, const uint8_t *peers, goldilocks_bool_t allow_identity, size_t m) {
    if (!out) return GOLDILOCKS_FAILURE;
    *out = nullptr;
    Call k;
    if (!k.ok) return k.finish();
    if (m >= UINT32_MAX) { g_err = "goldilocks_b200_decaf_peerset_create: at most 2^32 - 2 peers"; return GOLDILOCKS_FAILURE; }
    const size_t mm = m + 1;
    goldilocks_b200_decaf_peerset_s *ps = new goldilocks_b200_decaf_peerset_s{{k.c->dev, m}, nullptr, nullptr};
    bool ok = ps->alloc(&ps->peer_ok, mm) && ps->alloc(&ps->tables, mm * COMB_ENTRIES);
    if (ok) {
        abi_pt *pts = k.out<abi_pt>(mm);
        LaneDecafPeerDecode fd = {pts, ps->peer_ok, k.in(peers, 56 * m), k.c->ft, (uint32_t)m, allow_identity ? 1u : 0u};
        k.run(fd, mm);
        comb_tables(k, pts, ps->tables, mm);
    }
    return finish_create(k, ok, ps, out, "goldilocks_b200_decaf_peerset_create: device allocation failed");
}
void goldilocks_b200_decaf_peerset_destroy(goldilocks_b200_decaf_peerset *ps) { delete ps; }
size_t goldilocks_b200_decaf_peerset_size(const goldilocks_b200_decaf_peerset *ps) { return ps ? ps->m : 0; }
goldilocks_error_t goldilocks_448_direct_scalarmul_peerset_batch(uint8_t *scaled, goldilocks_error_t *status, const goldilocks_b200_decaf_peerset *ps,
                                                                 const uint32_t *peer_index, const hsc *scalar, goldilocks_bool_t short_circuit, size_t n) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Call k;
    if (!k.ok) return k.finish();
    if (!set_call(ps, k.c->dev, "goldilocks_448_direct_scalarmul_peerset_batch", n)) return GOLDILOCKS_FAILURE;
    uint8_t *dout = k.secret(k.in(scaled, 56 * n), 56 * n); /* short-circuited elements keep the caller's bytes */
    int32_t *dst = k.out<int32_t>(n);
    const uint32_t *didx = k.in(peer_index, n);
    const abi_sc *dsc = k.secret(k.in(S(scalar), n), n);
    OrderScratch s;
    order_scratch(&s, k.alloc(order_scratch(nullptr, nullptr, n)), n);
    if (k.ok) k.ok = decaf_peer_enqueue(*k.c, dout, dst, ps, didx, dsc, short_circuit != 0, n, s, k.c->stream);
    k.fetch(scaled, dout, 56 * n);
    k.fetch((int32_t *)status, dst, n);
    return k.finish();
}

// ---- point sets: key-set tables for goldilocks_448_base_double_scalarmul_non_secret against recurring points (slot_lanes.cuh SlotPointset)
struct goldilocks_b200_pointset_s : DeviceSet {
    static constexpr const char *noun = "point set";
    uint4 *ktabs;   /* m + 1 key-set tables (KSET_QUADS each when flat, else KTAB_QUADS); table m, the identity's, stands for every index >= m */
    bool flat;
};
/* the sort by point (as decaf peer sets), then the point-set kernel of the set's layout over the elements in that order */
static bool pointset_enqueue(Ctx &c, abi_pt *out, const goldilocks_b200_pointset_s *ps, const uint32_t *point_index, const abi_sc *scalar1,
                             const abi_sc *scalar2, size_t n, const OrderScratch &s, cudaStream_t st, unsigned *counter) {
    const uint32_t m = (uint32_t)ps->m;
    if (!set_order(c, point_index, m, n, s, st, "pair_sort (point set)")) return false;
    return launch_layout(c, ps->flat, n, st, counter, [&](auto flat) {
        return SlotPointset<decltype(flat)::value>{out, scalar1, scalar2, c.wide, ps->ktabs, point_index, s.order, m};
    });
}
goldilocks_error_t goldilocks_b200_pointset_create(goldilocks_b200_pointset **out, const hpt *points, size_t m) {
    if (!out) return GOLDILOCKS_FAILURE;
    *out = nullptr;
    Call k;
    if (!k.ok) return k.finish();
    if (m >= UINT32_MAX) { g_err = "goldilocks_b200_pointset_create: at most 2^32 - 2 points"; return GOLDILOCKS_FAILURE; }
    const size_t mm = m + 1;
    const bool flat = keyset_flat(mm);
    goldilocks_b200_pointset_s *ps = new goldilocks_b200_pointset_s{{k.c->dev, m}, nullptr, flat};
    bool ok = ps->alloc(&ps->ktabs, mm * (flat ? KSET_QUADS : KTAB_QUADS));
    if (ok) {
        static const abi_pt identity = {{{0}}, {{1}}, {{1}}, {{0}}};
        abi_pt *pts = k.out<abi_pt>(mm);
        ok = k.ok && (m == 0 || cudaMemcpyAsync(pts, points, sizeof(abi_pt) * m, cudaMemcpyHostToDevice, k.c->stream) == cudaSuccess) &&
             cudaMemcpyAsync(pts + m, &identity, sizeof(abi_pt), cudaMemcpyHostToDevice, k.c->stream) == cudaSuccess;
        if (ok) keyset_tables(k, pts, ps->ktabs, mm, flat);
    }
    return finish_create(k, ok, ps, out, "goldilocks_b200_pointset_create: device allocation or copy failed");
}
void goldilocks_b200_pointset_destroy(goldilocks_b200_pointset *ps) { delete ps; }
size_t goldilocks_b200_pointset_size(const goldilocks_b200_pointset *ps) { return ps ? ps->m : 0; }
goldilocks_error_t goldilocks_448_base_double_scalarmul_non_secret_pointset_batch(hpt *out, const goldilocks_b200_pointset *ps, const uint32_t *point_index,
                                                                              const hsc *scalar1, const hsc *scalar2, size_t n) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Call k;
    if (!k.ok) return k.finish();
    if (!set_call(ps, k.c->dev, "goldilocks_448_base_double_scalarmul_non_secret_pointset_batch", n)) return GOLDILOCKS_FAILURE;
    abi_pt *dout = k.out<abi_pt>(n);
    const uint32_t *didx = k.in(point_index, n);
    const abi_sc *ds1 = k.in(S(scalar1), n), *ds2 = k.in(S(scalar2), n);
    OrderScratch s;
    order_scratch(&s, k.alloc(order_scratch(nullptr, nullptr, n)), n);
    if (k.ok) k.ok = pointset_enqueue(*k.c, dout, ps, didx, ds1, ds2, n, s, k.c->stream, nullptr);
    k.fetch(P(out), dout, n);
    return k.finish();
}

// ---- key-set lookup: verification by public-key bytes against a key set, the keys outside it through the ordinary path --------
// Looked-up index per element (LaneKeysetLookup) -> the sets' order (hits grouped by key, the misses as one tail)
// -> the miss count, read back once -> the hits through the ordered key-set finish kernel, the misses packed and through verify_dev
// unchanged -> every status scattered back to its element.
struct KeysetLookupScratch {
    OrderScratch sort;
    uint32_t *idx, *hits;
    abi_sc *chal, *resp;
    verify_aux *aux;
    int32_t *st;                 /* statuses in sorted order: the hits', then the misses' */
    uint8_t *sig2, *pk2;         /* the misses, packed */
    size_t *len, *off2;
    void *scan_tmp; size_t scan_bytes;
    void *verify; uint4 *slots;  /* verify_dev's scratch and window tables, sized for n misses */
    uint8_t *msg2;               /* last: msg_bytes of it */
};
static size_t keyset_lookup_scratch(KeysetLookupScratch *s, void *base, size_t n, size_t msg_bytes, const VerifyGrids &g) {
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    char *p = (char *)base;
    size_t used = 0;
    auto take = [&](size_t bytes) { void *r = p ? p + used : nullptr; used += al(bytes); return r; };
    OrderScratch sort;
    void *pb = take(order_scratch(nullptr, nullptr, n));
    if (s) order_scratch(&sort, pb, n);
    uint32_t *idx = (uint32_t *)take(sizeof(uint32_t) * n), *hits = (uint32_t *)take(sizeof(uint32_t));
    abi_sc *chal = (abi_sc *)take(sizeof(abi_sc) * n), *resp = (abi_sc *)take(sizeof(abi_sc) * n);
    verify_aux *aux = (verify_aux *)take(sizeof(verify_aux) * n);
    int32_t *st = (int32_t *)take(sizeof(int32_t) * n);
    uint8_t *sig2 = (uint8_t *)take(114 * n), *pk2 = (uint8_t *)take(57 * n);
    size_t *len = (size_t *)take(sizeof(size_t) * (n + 1)), *off2 = (size_t *)take(sizeof(size_t) * (n + 1));
    const size_t scan_bytes = length_scan_scratch_bytes(n + 1);
    void *scan_tmp = take(scan_bytes);
    void *verify = take(verify_core_scratch_bytes(n));
    uint4 *slots = (uint4 *)take(verify_slot_bytes(g, n));
    uint8_t *msg2 = (uint8_t *)take(msg_bytes);
    if (s) *s = {sort, idx, hits, chal, resp, aux, st, sig2, pk2, len, off2, scan_tmp, scan_bytes, verify, slots, msg2};
    return used;
}
/* the first half: looked-up indices into idx, the order, the number of hits on the host (synchronises st) */
static bool keyset_lookup_order(Ctx &c, uint32_t *idx, const goldilocks_b200_keyset_s *ks, const uint8_t *pk, size_t n, const KeysetLookupScratch &s,
                                cudaStream_t st, size_t *hits) {
    const uint32_t m = (uint32_t)ks->m;
    LaneKeysetLookup fl = {idx, pk, ks->pk, ks->sorted, m};
    if (!launch(c, fl, n, st) || !set_order(c, idx, m, n, s.sort, st, "pair_sort (key set lookup)")) return false;
    LaneKeysetHits fh = {s.hits, s.sort.keys_s, m, n};
    if (!launch(c, fh, n, st)) return false;
    uint32_t h = 0;
    CU(cudaMemcpyAsync(&h, s.hits, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *hits = h;
    return true;
}
/* the second half: hits through the key set, misses through verify_dev (on `side` beside it where verify_dev forks), statuses back */
static bool keyset_lookup_verify(Ctx &c, int32_t *status, const goldilocks_b200_keyset_s *ks, const uint32_t *idx, const uint8_t *sig, const uint8_t *pk,
                                 const uint8_t *msg, const size_t *off, uint8_t prehashed, const uint8_t *ctx, uint8_t ctx_len, size_t n, size_t hits,
                                 const KeysetLookupScratch &s, const VerifyGrids &grids, cudaStream_t st, unsigned *counter, cudaStream_t side, cudaEvent_t *side_evt) {
    if (hits) {
        LaneEdVerifyScalars f2 = {s.chal, s.resp, sig, pk, msg, off, prehashed, ctx, ctx_len, 0};   /* a hit's key bytes are its set key's */
        if (!launch(c, f2, n, st)) return false;
        if (!launch_layout(c, ks->flat, hits, st, counter, [&](auto flat) {
                return SlotEdVerifyFinishKeysetOrdered<decltype(flat)::value>{s.aux, ks->key_ok, s.chal, s.resp, c.wide, ks->ktabs, idx, s.sort.order, sig};
            }))
            return false;
        LaneVerifySign fv = {s.st, s.aux, 1, hits};
        if (!launch(c, fv, (hits + VSIGN_BATCH - 1) / VSIGN_BATCH, st)) return false;
    }
    const size_t misses = n - hits;
    if (misses) {
        LaneKeysetMissLengths fl = {s.len, off, s.sort.order, hits, misses};
        if (!launch(c, fl, misses + 1, st)) return false;
        CU(length_scan(s.scan_tmp, s.scan_bytes, s.len, s.off2, misses + 1, st));
        LaneKeysetMissGather fg = {s.sig2, s.pk2, s.msg2, s.off2, sig, pk, msg, off, s.sort.order, hits};
        if (!launch(c, fg, misses, st)) return false;
        if (!verify_dev(c, s.st + hits, s.sig2, s.pk2, s.msg2, s.off2, prehashed, ctx, ctx_len, misses, s.verify, s.slots, grids, st, nullptr, side, side_evt))
            return false;
    }
    LaneKeysetScatter fs = {status, s.st, s.sort.order};
    return launch(c, fs, n, st);
}
goldilocks_error_t goldilocks_ed448_verify_keyset_lookup_batch(goldilocks_error_t *status, uint32_t *key_index, const goldilocks_b200_keyset *ks, const uint8_t *signature,
                                                               const uint8_t *pubkey, const uint8_t *msg, const size_t *msg_off, uint8_t prehashed,
                                                               const uint8_t *context, uint8_t context_len, size_t n) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Call k;
    if (!k.ok) return k.finish();
    if (!set_call(ks, k.c->dev, "goldilocks_ed448_verify_keyset_lookup_batch", n)) return GOLDILOCKS_FAILURE;
    /* the keys first, as goldilocks_ed448_verify_batch: the lookup, the sort and the read-back of the miss count run while the
     * signatures and messages still cross PCIe on the copy stream */
    const size_t total = msg_off[n];
    const size_t *doff = k.in(msg_off, n + 1);
    const uint8_t *dctx = k.in(context, context_len);
    const uint8_t *dpk = k.in(pubkey, 57 * n);
    uint8_t *dsig = k.out<uint8_t>(114 * n), *dmsg = k.out<uint8_t>(total);
    int32_t *dst = k.out<int32_t>(n);
    k.push(dsig, signature, 114 * n);
    k.push(dmsg, msg, total);
    if (k.ok && cudaEventRecord(k.c->copy_done[0], k.c->copy_stream) != cudaSuccess) k.ok = false;
    VerifyGrids grids;
    if (k.ok) k.ok = verify_grids(*k.c, &grids);
    KeysetLookupScratch s = {};
    void *base = k.alloc(keyset_lookup_scratch(nullptr, nullptr, n, total, grids));
    if (k.ok) keyset_lookup_scratch(&s, base, n, total, grids);
    size_t hits = 0;
    if (k.ok) k.ok = keyset_lookup_order(*k.c, s.idx, ks, dpk, n, s, k.c->stream, &hits);
    if (k.ok) k.ok = cudaStreamWaitEvent(k.c->stream, k.c->copy_done[0], 0) == cudaSuccess;
    if (k.ok) k.ok = keyset_lookup_verify(*k.c, dst, ks, s.idx, dsig, dpk, dmsg, doff, prehashed, dctx, context_len, n, hits, s, grids, k.c->stream, nullptr,
                                          k.c->side_stream, k.c->side_evt);
    k.fetch((int32_t *)status, dst, n);
    if (key_index) k.fetch(key_index, s.idx, n);
    if (!k.ok && k.c) cudaStreamSynchronize(k.c->copy_stream); /* never leave copies in flight behind an error */
    return k.finish();
}

// ---- device-resident variants -------------------------------------------------------------------------------
goldilocks_error_t goldilocks_ed448_verify_batch_dev(goldilocks_error_t *status, const uint8_t *signature, const uint8_t *pubkey, const uint8_t *msg, const size_t *msg_off,
                                                     uint8_t prehashed, const uint8_t *context, uint8_t context_len, size_t n, void *scratch, void *stream) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    VerifyGrids grids;
    if (!verify_grids(*c, &grids)) return GOLDILOCKS_FAILURE;
    /* nothing of the context is written while the kernels run: window tables, work lists and hand-out counters all live in
     * the caller's scratch, so calls on different streams (and host-pointer calls of other threads) do not interfere */
    uint4 *slots = (uint4 *)((char *)scratch + verify_core_scratch_bytes(n));
    std::lock_guard<std::mutex> g(c->dev_side_mu); /* held while the launches are queued, not while they run */
    return verify_dev(*c, (int32_t *)status, signature, pubkey, msg, msg_off, prehashed, context, context_len, n, scratch, slots, grids, as_stream(stream), nullptr,
                      c->dev_side, c->dev_evt) ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
goldilocks_error_t goldilocks_x448_batch_dev(uint8_t *out, goldilocks_error_t *status, const uint8_t *base, const uint8_t *scalar, size_t n, void *stream) {
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    SlotX448 f = {out, (int32_t *)status, base, scalar};
    return launch_slots(*c, f, n, as_stream(stream)) ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
goldilocks_error_t goldilocks_x448_peerset_batch_dev(uint8_t *out, goldilocks_error_t *status, const goldilocks_b200_x448_peerset *ps, const uint32_t *peer_index,
                                                     const uint8_t *scalar, size_t n, void *stream) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    if (!set_call(ps, c->dev, "goldilocks_x448_peerset_batch_dev")) return GOLDILOCKS_FAILURE;
    SlotX448Peer f = {out, (int32_t *)status, ps->tables, ps->table_ok, ps->peers, peer_index, scalar, (uint32_t)ps->m};
    return launch_slots(*c, f, n, as_stream(stream)) ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
size_t goldilocks_b200_x448_peerset_scratch_bytes(size_t n) { return dev_ctx() ? x448_peer_lookup_scratch(nullptr, nullptr, nullptr, n) : 0; }
goldilocks_error_t goldilocks_x448_peerset_lookup_batch_dev(uint8_t *out, goldilocks_error_t *status, uint32_t *peer_index, const goldilocks_b200_x448_peerset *ps,
                                                            const uint8_t *base, const uint8_t *scalar, size_t n, void *scratch, void *stream) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    if (!set_call(ps, c->dev, "goldilocks_x448_peerset_lookup_batch_dev", n, scratch)) return GOLDILOCKS_FAILURE;
    /* everything the call writes besides out / status / peer_index lives in the caller's scratch: calls on different streams do not
     * interfere, and nothing waits for the stream */
    OrderScratch s;
    uint32_t *idx = nullptr;
    x448_peer_lookup_scratch(&s, &idx, scratch, n);
    return x448_peer_lookup_enqueue(*c, out, (int32_t *)status, peer_index ? peer_index : idx, ps, base, scalar, n, s, as_stream(stream)) ? GOLDILOCKS_SUCCESS
                                                                                                                                        : GOLDILOCKS_FAILURE;
}
size_t goldilocks_b200_decaf_peerset_scratch_bytes(size_t n) { return order_scratch_bytes(n); }
goldilocks_error_t goldilocks_448_direct_scalarmul_peerset_batch_dev(uint8_t *scaled, goldilocks_error_t *status, const goldilocks_b200_decaf_peerset *ps,
                                                                     const uint32_t *peer_index, const hsc *scalar, goldilocks_bool_t short_circuit, size_t n,
                                                                     void *scratch, void *stream) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    if (!set_call(ps, c->dev, "goldilocks_448_direct_scalarmul_peerset_batch_dev", n, scratch)) return GOLDILOCKS_FAILURE;
    /* everything the call writes besides scaled / status lives in the caller's scratch: calls on different streams do not interfere */
    OrderScratch s;
    order_scratch(&s, scratch, n);
    return decaf_peer_enqueue(*c, scaled, (int32_t *)status, ps, peer_index, S(scalar), short_circuit != 0, n, s, as_stream(stream)) ? GOLDILOCKS_SUCCESS
                                                                                                                                      : GOLDILOCKS_FAILURE;
}
size_t goldilocks_b200_pointset_scratch_bytes(size_t n) { return order_scratch_bytes(n); }
goldilocks_error_t goldilocks_448_base_double_scalarmul_non_secret_pointset_batch_dev(hpt *out, const goldilocks_b200_pointset *ps, const uint32_t *point_index,
                                                                                  const hsc *scalar1, const hsc *scalar2, size_t n, void *scratch, void *stream) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    if (!set_call(ps, c->dev, "goldilocks_448_base_double_scalarmul_non_secret_pointset_batch_dev", n, scratch)) return GOLDILOCKS_FAILURE;
    /* the sort lives in the caller's scratch and the kernel takes a fixed grid-stride assignment (no hand-out counter of the
     * context): calls on different streams do not interfere */
    OrderScratch s;
    order_scratch(&s, scratch, n);
    return pointset_enqueue(*c, P(out), ps, point_index, S(scalar1), S(scalar2), n, s, as_stream(stream), GRID_STRIDE) ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
size_t goldilocks_b200_keyset_scratch_bytes(size_t n, size_t msg_bytes) {
    Ctx *c = dev_ctx();
    VerifyGrids grids;
    if (!c || !verify_grids(*c, &grids)) return 0;
    return keyset_lookup_scratch(nullptr, nullptr, n, msg_bytes, grids);
}
goldilocks_error_t goldilocks_ed448_verify_keyset_batch_dev(goldilocks_error_t *status, const goldilocks_b200_keyset *ks, const uint32_t *key_index,
                                                            const uint8_t *signature, const uint8_t *msg, const size_t *msg_off, uint8_t prehashed,
                                                            const uint8_t *context, uint8_t context_len, size_t n, void *scratch, void *stream) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    if (!set_call(ks, c->dev, "goldilocks_ed448_verify_keyset_batch_dev", n, scratch)) return GOLDILOCKS_FAILURE;
    VerifyGrids grids;
    if (!verify_grids(*c, &grids)) return GOLDILOCKS_FAILURE;
    KeysetLookupScratch s = {};
    keyset_lookup_scratch(&s, scratch, n, 0, grids);
    /* fixed grid-stride assignment (no hand-out counter of the context): calls on different streams do not interfere */
    return keyset_enqueue(*c, (int32_t *)status, ks, key_index, signature, msg, msg_off, prehashed, context, context_len, n, s.chal, s.resp, s.aux,
                          as_stream(stream), GRID_STRIDE) ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
goldilocks_error_t goldilocks_ed448_verify_keyset_lookup_batch_dev(goldilocks_error_t *status, uint32_t *key_index, const goldilocks_b200_keyset *ks,
                                                                   const uint8_t *signature, const uint8_t *pubkey, const uint8_t *msg, const size_t *msg_off,
                                                                   uint8_t prehashed, const uint8_t *context, uint8_t context_len, size_t n, void *scratch, void *stream) {
    if (n == 0) return GOLDILOCKS_SUCCESS;
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    if (!set_call(ks, c->dev, "goldilocks_ed448_verify_keyset_lookup_batch_dev", n, scratch)) return GOLDILOCKS_FAILURE;
    VerifyGrids grids;
    if (!verify_grids(*c, &grids)) return GOLDILOCKS_FAILURE;
    KeysetLookupScratch s = {};
    keyset_lookup_scratch(&s, scratch, n, 0, grids);   /* the packed messages sit last, so the layout does not depend on msg_bytes */
    cudaStream_t st = as_stream(stream);
    uint32_t *idx = key_index ? key_index : s.idx;
    size_t hits = 0;
    if (!keyset_lookup_order(*c, idx, ks, pubkey, n, s, st, &hits)) return GOLDILOCKS_FAILURE;
    /* everything from here on lives in the caller's scratch, as in goldilocks_ed448_verify_batch_dev */
    std::lock_guard<std::mutex> g(c->dev_side_mu); /* held while the launches are queued, not while they run */
    return keyset_lookup_verify(*c, (int32_t *)status, ks, idx, signature, pubkey, msg, msg_off, prehashed, context, context_len, n, hits, s, grids, st, GRID_STRIDE,
                                c->dev_side, c->dev_evt) ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
goldilocks_error_t goldilocks_448_precomputed_scalarmul_batch_dev(hpt *out, const hsc *scalar, size_t n, void *stream) {
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    SlotComb f = {P(out), S(scalar), c->ft};
    return launch_slots(*c, f, n, as_stream(stream)) ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
goldilocks_error_t goldilocks_448_gf_mul_batch_dev(uint8_t *out, const uint8_t *a, const uint8_t *b, size_t n, void *stream) {
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    LaneGf<GFOP_MUL> f = {out, nullptr, a, b, 0};
    return launch(*c, f, n, as_stream(stream)) ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
goldilocks_error_t goldilocks_448_point_add_batch_dev(hpt *out, const hpt *a, const hpt *b, size_t n, void *stream) {
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    LanePt<PTOP_ADD> f = {P(out), P(a), P(b)};
    return launch(*c, f, n, as_stream(stream)) ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
goldilocks_error_t goldilocks_448_point_double_batch_dev(hpt *out, const hpt *a, size_t n, void *stream) {
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    LanePt<PTOP_DBL> f = {P(out), P(a), nullptr};
    return launch(*c, f, n, as_stream(stream)) ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
goldilocks_error_t goldilocks_448_point_decode_batch_dev(hpt *pts, goldilocks_error_t *status, const uint8_t *ser, goldilocks_bool_t allow_identity, size_t n, void *stream) {
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    LanePtDecode f = {P(pts), (int32_t *)status, ser, allow_identity ? 1u : 0u};
    return launch(*c, f, n, as_stream(stream)) ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
goldilocks_error_t goldilocks_448_point_encode_batch_dev(uint8_t *ser, const hpt *pts, size_t n, void *stream) {
    Ctx *c = dev_ctx();
    if (!c) return GOLDILOCKS_FAILURE;
    LanePtEncode f = {ser, P(pts)};
    return launch(*c, f, n, as_stream(stream)) ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}

// ---- concurrent single-element calls gathered into one batch (coalesce.h; goldilocks_b200_coalesce) ----------
extern "C++" {
namespace {
coalesce::Settings g_coalesce;
coalesce::Stats g_coalesce_stats;
std::once_flag g_coalesce_env;
bool coalescing() {
    std::call_once(g_coalesce_env, [] {
        if (const char *w = getenv("GOLDILOCKS_B200_COALESCE_US")) g_coalesce.window_us.store((unsigned)strtoul(w, nullptr, 10));
        if (const char *m = getenv("GOLDILOCKS_B200_COALESCE_MAX")) { const unsigned v = (unsigned)strtoul(m, nullptr, 10); if (v) g_coalesce.max_batch.store(v); }
    });
    return g_coalesce.window_us.load(std::memory_order_relaxed) != 0 && !shard::t_worker;
}
struct MsgArgs { uint8_t prehashed; const uint8_t *context; uint8_t context_len; const uint8_t *message; size_t message_len; };
struct VerifyReq { bool done; MsgArgs m; const uint8_t *sig, *pk; goldilocks_error_t st; };
struct SignReq { bool done; MsgArgs m; uint8_t *sig; const uint8_t *sk, *pk; };
struct X448Req { bool done; uint8_t *out; const uint8_t *base, *scalar; goldilocks_error_t st; };
coalesce::Gate<VerifyReq> g_gate_verify;
coalesce::Gate<SignReq> g_gate_sign;
coalesce::Gate<X448Req> g_gate_x448;
bool same_domain(const MsgArgs &a, const MsgArgs &b) { /* the batch entry points take one (prehashed, context) for the whole batch */
    return a.prehashed == b.prehashed && a.context_len == b.context_len && (a.context_len == 0 || memcmp(a.context, b.context, a.context_len) == 0);
}
// Requests of one gathering, split into runs that share (prehashed, context); fn(first request, indices of the run, messages, offsets).
template <class Req, class Fn>
void for_each_domain(Req **q, size_t n, Fn fn) {
    std::vector<char> taken(n, 0);
    std::vector<size_t> idx, off;
    std::vector<uint8_t> msg;
    for (size_t i = 0; i < n; i++) {
        if (taken[i]) continue;
        idx.clear(); off.assign(1, 0); msg.clear();
        for (size_t j = i; j < n; j++) {
            if (taken[j] || !same_domain(q[i]->m, q[j]->m)) continue;
            taken[j] = 1;
            idx.push_back(j);
            if (q[j]->m.message_len) msg.insert(msg.end(), q[j]->m.message, q[j]->m.message + q[j]->m.message_len);
            off.push_back(msg.size());
        }
        if (msg.empty()) msg.push_back(0);
        fn(q[i]->m, idx, msg, off);
    }
}
void run_verify_requests(VerifyReq **q, size_t n) {
    for_each_domain(q, n, [&](const MsgArgs &d, const std::vector<size_t> &idx, const std::vector<uint8_t> &msg, const std::vector<size_t> &off) {
        const size_t m = idx.size();
        std::vector<uint8_t> sig(114 * m), pk(57 * m);
        std::vector<goldilocks_error_t> st(m, GOLDILOCKS_FAILURE);
        for (size_t k = 0; k < m; k++) { memcpy(&sig[114 * k], q[idx[k]]->sig, 114); memcpy(&pk[57 * k], q[idx[k]]->pk, 57); }
        const bool ok = goldilocks_ed448_verify_batch(st.data(), sig.data(), pk.data(), msg.data(), off.data(), d.prehashed, d.context, d.context_len, m) == GOLDILOCKS_SUCCESS;
        for (size_t k = 0; k < m; k++) q[idx[k]]->st = ok ? st[k] : GOLDILOCKS_FAILURE;
    });
}
void run_sign_requests(SignReq **q, size_t n) {
    for_each_domain(q, n, [&](const MsgArgs &d, const std::vector<size_t> &idx, const std::vector<uint8_t> &msg, const std::vector<size_t> &off) {
        const size_t m = idx.size();
        std::vector<uint8_t> sig(114 * m), sk(57 * m), pk(57 * m);
        for (size_t k = 0; k < m; k++) { memcpy(&sk[57 * k], q[idx[k]]->sk, 57); memcpy(&pk[57 * k], q[idx[k]]->pk, 57); }
        const bool ok = goldilocks_ed448_sign_batch(sig.data(), sk.data(), pk.data(), msg.data(), off.data(), d.prehashed, d.context, d.context_len, m) == GOLDILOCKS_SUCCESS;
        for (size_t k = 0; k < m; k++) {
            if (ok) memcpy(q[idx[k]]->sig, &sig[114 * k], 114);
            else memset(q[idx[k]]->sig, 0, 114);
        }
        goldilocks_bzero(sk.data(), sk.size());             /* the gathered private keys */
    });
}
void run_x448_requests(X448Req **q, size_t n) {
    std::vector<uint8_t> out(56 * n), base(56 * n), scalar(56 * n);
    std::vector<goldilocks_error_t> st(n, GOLDILOCKS_FAILURE);
    for (size_t k = 0; k < n; k++) { memcpy(&base[56 * k], q[k]->base, 56); memcpy(&scalar[56 * k], q[k]->scalar, 56); }
    const bool ok = goldilocks_x448_batch(out.data(), st.data(), base.data(), scalar.data(), n) == GOLDILOCKS_SUCCESS;
    for (size_t k = 0; k < n; k++) {
        if (ok) memcpy(q[k]->out, &out[56 * k], 56);
        else memset(q[k]->out, 0, 56);
        q[k]->st = ok ? st[k] : GOLDILOCKS_FAILURE;
    }
    goldilocks_bzero(scalar.data(), scalar.size());         /* the gathered secret scalars ... */
    goldilocks_bzero(out.data(), out.size());               /* ... and shared secrets */
}
}  // namespace
}  // extern "C++"
void goldilocks_b200_coalesce(unsigned window_us, unsigned max_batch) {
    coalescing();                                           /* read the environment first, so that this call wins over it */
    g_coalesce.max_batch.store(max_batch ? max_batch : 4096);
    g_coalesce.window_us.store(window_us);
}
void goldilocks_b200_coalesce_stats(unsigned long long *calls, unsigned long long *batches, unsigned long long *largest) {
    if (calls) *calls = g_coalesce_stats.calls.load();
    if (batches) *batches = g_coalesce_stats.batches.load();
    if (largest) *largest = g_coalesce_stats.largest.load();
}

// ---- legacy single-element entry points: a batch of one on the GPU ------------------------------------------
void goldilocks_448_point_add(goldilocks_448_point_p o, const goldilocks_448_point_p a, const goldilocks_448_point_p b) { goldilocks_448_point_add_batch(o, a, b, 1); }
void goldilocks_448_point_sub(goldilocks_448_point_p o, const goldilocks_448_point_p a, const goldilocks_448_point_p b) { goldilocks_448_point_sub_batch(o, a, b, 1); }
void goldilocks_448_point_double(goldilocks_448_point_p o, const goldilocks_448_point_p a) { goldilocks_448_point_double_batch(o, a, 1); }
void goldilocks_448_point_negate(goldilocks_448_point_p o, const goldilocks_448_point_p a) { goldilocks_448_point_negate_batch(o, a, 1); }
void goldilocks_448_point_encode(uint8_t ser[56], const goldilocks_448_point_p pt) { goldilocks_448_point_encode_batch(ser, pt, 1); }
goldilocks_error_t goldilocks_448_point_decode(goldilocks_448_point_p pt, const uint8_t ser[56], goldilocks_bool_t allow_identity) {
    goldilocks_error_t st = GOLDILOCKS_FAILURE;
    if (goldilocks_448_point_decode_batch(pt, &st, ser, allow_identity, 1) != GOLDILOCKS_SUCCESS) return GOLDILOCKS_FAILURE;
    return st;
}
goldilocks_bool_t goldilocks_448_point_eq(const goldilocks_448_point_p a, const goldilocks_448_point_p b) {
    goldilocks_bool_t r = 0;
    goldilocks_448_point_eq_batch(&r, a, b, 1);
    return r;
}
goldilocks_bool_t goldilocks_448_point_valid(const goldilocks_448_point_p a) {
    goldilocks_bool_t r = 0;
    goldilocks_448_point_valid_batch(&r, a, 1);
    return r;
}
void goldilocks_448_point_scalarmul(goldilocks_448_point_p o, const goldilocks_448_point_p b, const goldilocks_448_scalar_p s) { goldilocks_448_point_scalarmul_batch(o, b, s, 1); }
void goldilocks_448_precomputed_scalarmul(goldilocks_448_point_p o, const goldilocks_448_precomputed_s *b, const goldilocks_448_scalar_p s) { goldilocks_448_precomputed_scalarmul_batch(o, b, s, 1); }
void goldilocks_448_point_double_scalarmul(goldilocks_448_point_p o, const goldilocks_448_point_p b1, const goldilocks_448_scalar_p s1, const goldilocks_448_point_p b2, const goldilocks_448_scalar_p s2) {
    goldilocks_448_point_double_scalarmul_batch(o, b1, s1, b2, s2, 1);
}
void goldilocks_448_base_double_scalarmul_non_secret(goldilocks_448_point_p o, const goldilocks_448_scalar_p s1, const goldilocks_448_point_p b2, const goldilocks_448_scalar_p s2) {
    goldilocks_448_base_double_scalarmul_non_secret_batch(o, s1, b2, s2, 1);
}
void goldilocks_448_point_from_hash_nonuniform(goldilocks_448_point_p pt, const uint8_t h[56]) { goldilocks_448_point_from_hash_nonuniform_batch(pt, h, 1); }
void goldilocks_448_point_from_hash_uniform(goldilocks_448_point_p pt, const uint8_t h[112]) { goldilocks_448_point_from_hash_uniform_batch(pt, h, 1); }
goldilocks_error_t goldilocks_448_invert_elligator_nonuniform(uint8_t recovered_hash[56], const goldilocks_448_point_p pt, uint32_t which) {
    goldilocks_error_t st = GOLDILOCKS_FAILURE;
    return goldilocks_448_invert_elligator_nonuniform_batch(recovered_hash, &st, pt, &which, 1) == GOLDILOCKS_SUCCESS ? st : GOLDILOCKS_FAILURE;
}
goldilocks_error_t goldilocks_448_invert_elligator_uniform(uint8_t partial_hash[112], const goldilocks_448_point_p pt, uint32_t which) {
    goldilocks_error_t st = GOLDILOCKS_FAILURE;
    return goldilocks_448_invert_elligator_uniform_batch(partial_hash, &st, pt, &which, 1) == GOLDILOCKS_SUCCESS ? st : GOLDILOCKS_FAILURE;
}
void goldilocks_448_point_mul_by_ratio_and_encode_like_eddsa(uint8_t enc[57], const goldilocks_448_point_p p) { goldilocks_448_point_mul_by_ratio_and_encode_like_eddsa_batch(enc, p, 1); }
goldilocks_error_t goldilocks_448_point_decode_like_eddsa_and_mul_by_ratio(goldilocks_448_point_p p, const uint8_t enc[57]) {
    goldilocks_error_t st = GOLDILOCKS_FAILURE;
    if (goldilocks_448_point_decode_like_eddsa_and_mul_by_ratio_batch(p, &st, enc, 1) != GOLDILOCKS_SUCCESS) return GOLDILOCKS_FAILURE;
    return st;
}
void goldilocks_448_point_mul_by_ratio_and_encode_like_x448(uint8_t out[56], const goldilocks_448_point_p p) { goldilocks_448_point_mul_by_ratio_and_encode_like_x448_batch(out, p, 1); }
goldilocks_error_t goldilocks_x448(uint8_t out[56], const uint8_t base[56], const uint8_t scalar[56]) {
    if (coalescing()) {
        X448Req r = {false, out, base, scalar, GOLDILOCKS_FAILURE};
        g_gate_x448.submit(&r, g_coalesce, g_coalesce_stats, run_x448_requests);
        return r.st;
    }
    goldilocks_error_t st = GOLDILOCKS_FAILURE;
    if (goldilocks_x448_batch(out, &st, base, scalar, 1) != GOLDILOCKS_SUCCESS) return GOLDILOCKS_FAILURE;
    return st;
}
void goldilocks_x448_derive_public_key(uint8_t out[56], const uint8_t scalar[56]) { goldilocks_x448_derive_public_key_batch(out, scalar, 1); }
void goldilocks_ed448_derive_secret_scalar(goldilocks_448_scalar_p secret, const uint8_t privkey[57]) {
    Call k;
    LaneEdSecretScalar f = {k.secret(k.out<abi_sc>(1), 1), k.secret(k.in(privkey, 57), 57)};
    k.run(f, 1);
    k.fetch(S(secret), f.out, 1);
    k.finish();
}
void goldilocks_ed448_derive_public_key(uint8_t pubkey[57], const uint8_t privkey[57]) { goldilocks_ed448_derive_public_key_batch(pubkey, privkey, 1); }
void goldilocks_ed448_sign(uint8_t signature[114], const uint8_t privkey[57], const uint8_t pubkey[57], const uint8_t *message, size_t message_len,
                           uint8_t prehashed, const uint8_t *context, uint8_t context_len) {
    if (coalescing()) {
        SignReq r = {false, {prehashed, context, context_len, message, message_len}, signature, privkey, pubkey};
        g_gate_sign.submit(&r, g_coalesce, g_coalesce_stats, run_sign_requests);
        return;
    }
    const size_t off[2] = {0, message_len};
    goldilocks_ed448_sign_batch(signature, privkey, pubkey, message, off, prehashed, context, context_len, 1);
}
goldilocks_error_t goldilocks_ed448_verify(const uint8_t signature[114], const uint8_t pubkey[57], const uint8_t *message, size_t message_len,
                                           uint8_t prehashed, const uint8_t *context, uint8_t context_len) {
    if (coalescing()) {
        VerifyReq r = {false, {prehashed, context, context_len, message, message_len}, signature, pubkey, GOLDILOCKS_FAILURE};
        g_gate_verify.submit(&r, g_coalesce, g_coalesce_stats, run_verify_requests);
        return r.st;
    }
    const size_t off[2] = {0, message_len};
    goldilocks_error_t st = GOLDILOCKS_FAILURE;
    if (goldilocks_ed448_verify_batch(&st, signature, pubkey, message, off, prehashed, context, context_len, 1) != GOLDILOCKS_SUCCESS) return GOLDILOCKS_FAILURE;
    return st;
}
void goldilocks_448_point_dual_scalarmul(goldilocks_448_point_p a1, goldilocks_448_point_p a2, const goldilocks_448_point_p b, const goldilocks_448_scalar_p s1, const goldilocks_448_scalar_p s2) {
    goldilocks_448_point_dual_scalarmul_batch(a1, a2, b, s1, s2, 1);
}
goldilocks_error_t goldilocks_448_direct_scalarmul(uint8_t scaled[56], const uint8_t base[56], const goldilocks_448_scalar_p scalar, goldilocks_bool_t allow_identity, goldilocks_bool_t short_circuit) {
    goldilocks_error_t st = GOLDILOCKS_FAILURE;
    if (goldilocks_448_direct_scalarmul_batch(scaled, &st, base, scalar, allow_identity, short_circuit, 1) != GOLDILOCKS_SUCCESS) return GOLDILOCKS_FAILURE;
    return st;
}
void goldilocks_448_precompute(goldilocks_448_precomputed_s *table, const goldilocks_448_point_p base) { goldilocks_448_precompute_batch(table, base, 1); }
void goldilocks_448_point_debugging_torque(goldilocks_448_point_p q, const goldilocks_448_point_p p) { goldilocks_448_point_debugging_torque_batch(q, p, 1); }
void goldilocks_448_point_debugging_pscale(goldilocks_448_point_p q, const goldilocks_448_point_p p, const uint8_t factor[56]) { goldilocks_448_point_debugging_pscale_batch(q, p, factor, 1); }
void goldilocks_ed448_convert_public_key_to_x448(uint8_t x[56], const uint8_t ed[57]) { goldilocks_ed448_convert_public_key_to_x448_batch(x, ed, 1); }
void goldilocks_ed448_convert_private_key_to_x448(uint8_t x[56], const uint8_t ed[57]) { goldilocks_ed448_convert_private_key_to_x448_batch(x, ed, 1); }
goldilocks_error_t goldilocks_448_scalar_invert(goldilocks_448_scalar_p out, const goldilocks_448_scalar_p a) {
    goldilocks_error_t st = GOLDILOCKS_FAILURE;
    if (goldilocks_448_scalar_invert_batch(out, &st, a, 1) != GOLDILOCKS_SUCCESS) return GOLDILOCKS_FAILURE;
    return st;
}
/* Pure data movement / comparison on host structs: no arithmetic, nothing to run on the device.
 * (reference scalar.c:190-232,305-312; goldilocks.c:879-886; utils.c) */
static void ct_select(void *out, const void *a, const void *b, size_t bytes, goldilocks_bool_t pick_b) {
    const uint8_t m = (uint8_t)(pick_b ? 0xff : 0x00);
    for (size_t i = 0; i < bytes; i++) ((uint8_t *)out)[i] = (uint8_t)((((const uint8_t *)a)[i] & (uint8_t)~m) | (((const uint8_t *)b)[i] & m));
}
void goldilocks_bzero(void *data, size_t size) { volatile uint8_t *p = (volatile uint8_t *)data; for (size_t i = 0; i < size; i++) p[i] = 0; }
goldilocks_bool_t goldilocks_memeq(const void *data1, const void *data2, size_t size) {
    uint8_t d = 0;
    for (size_t i = 0; i < size; i++) d |= (uint8_t)(((const uint8_t *)data1)[i] ^ ((const uint8_t *)data2)[i]);
    return d ? 0 : ~(goldilocks_bool_t)0;
}
goldilocks_bool_t goldilocks_448_scalar_eq(const goldilocks_448_scalar_p a, const goldilocks_448_scalar_p b) { return goldilocks_memeq(a, b, sizeof(goldilocks_448_scalar_s)); }
void goldilocks_448_scalar_cond_sel(goldilocks_448_scalar_p out, const goldilocks_448_scalar_p a, const goldilocks_448_scalar_p b, goldilocks_bool_t pick_b) { ct_select(out, a, b, sizeof(goldilocks_448_scalar_s), pick_b); }
void goldilocks_448_point_cond_sel(goldilocks_448_point_p out, const goldilocks_448_point_p a, const goldilocks_448_point_p b, goldilocks_bool_t pick_b) { ct_select(out, a, b, sizeof(goldilocks_448_point_s), pick_b); }
void goldilocks_448_scalar_set_unsigned(goldilocks_448_scalar_p out, uint64_t w) { memset(out, 0, sizeof(goldilocks_448_scalar_s)); out->limb[0] = w; }
void goldilocks_448_scalar_destroy(goldilocks_448_scalar_p s) { goldilocks_bzero(s, sizeof(goldilocks_448_scalar_s)); }
void goldilocks_448_point_destroy(goldilocks_448_point_p p) { goldilocks_bzero(p, sizeof(goldilocks_448_point_s)); }
void goldilocks_448_precomputed_destroy(goldilocks_448_precomputed_s *t) { goldilocks_bzero(t, 15360); }
// ---- streaming SHA-3 / SHAKE objects and Ed448ph (reference shake.c:89-250, eddsa.c:76-80,232-251,309-329) ----
#define KP(n, rate, pad, maxo) const struct goldilocks_kparams_s n = {0, 'A', rate, 0, pad, 0x80, maxo, maxo};
KP(GOLDILOCKS_SHAKE128_params_s, 200 - 128 / 4, 0x1f, 0xFF)
KP(GOLDILOCKS_SHAKE256_params_s, 200 - 256 / 4, 0x1f, 0xFF)
KP(GOLDILOCKS_SHA3_224_params_s, 200 - 224 / 4, 0x06, 224 / 8)
KP(GOLDILOCKS_SHA3_256_params_s, 200 - 256 / 4, 0x06, 256 / 8)
KP(GOLDILOCKS_SHA3_384_params_s, 200 - 384 / 4, 0x06, 384 / 8)
KP(GOLDILOCKS_SHA3_512_params_s, 200 - 512 / 4, 0x06, 512 / 8)
#undef KP
static_assert(sizeof(goldilocks_keccak_sponge_s) == sizeof(sponge_abi) && sizeof(sponge_abi) == 208, "sponge layout (keccak_internal.h)");
static sponge_abi *SP(goldilocks_keccak_sponge_s *s) { return (sponge_abi *)s; }
void goldilocks_sha3_init(goldilocks_keccak_sponge_p sponge, const struct goldilocks_kparams_s *params) {
    struct goldilocks_kparams_s p = *params; /* params may alias the sponge's own copy (reset) */
    memset(sponge, 0, sizeof(goldilocks_keccak_sponge_s));
    memcpy(&SP(sponge)->position, &p, sizeof p);
    SP(sponge)->position = 0;
}
void goldilocks_sha3_reset(goldilocks_keccak_sponge_p sponge) {
    goldilocks_sha3_init(sponge, (const struct goldilocks_kparams_s *)&SP(sponge)->position);
    SP(sponge)->flags = 'A';
    SP(sponge)->remaining = SP(sponge)->max_out;
}
void goldilocks_sha3_destroy(goldilocks_keccak_sponge_p sponge) { goldilocks_bzero(sponge, sizeof(goldilocks_keccak_sponge_s)); }
goldilocks_error_t goldilocks_sha3_update(struct goldilocks_keccak_sponge_s *sponge, const uint8_t *in, size_t len) {
    sponge_abi *h = SP(sponge);
    if (h->start_round != 0 || h->rate == 0 || h->rate >= 200 || h->position >= h->rate) return GOLDILOCKS_FAILURE;
    if (len) {
        Call k;
        LaneSpongeUpdate f = {k.in(h, 1), k.in(in, len), len};
        k.run(f, 1);
        k.fetch(h, f.sp, 1);
        if (k.finish() != GOLDILOCKS_SUCCESS) return GOLDILOCKS_FAILURE;
    }
    return h->flags == 'A' ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
goldilocks_error_t goldilocks_sha3_output(goldilocks_keccak_sponge_p sponge, uint8_t *out, size_t len) {
    sponge_abi *h = SP(sponge);
    if (h->start_round != 0 || h->rate == 0 || h->rate >= 200 || h->position >= h->rate) return GOLDILOCKS_FAILURE;
    Call k;
    LaneSpongeOutput f = {k.in(h, 1), k.out<uint8_t>(len), len, k.out<int32_t>(1)};
    k.run(f, 1);
    int32_t st = 0;
    k.fetch(h, f.sp, 1);
    k.fetch(out, f.out, len);
    k.fetch(&st, f.status, 1);
    if (k.finish() != GOLDILOCKS_SUCCESS) return GOLDILOCKS_FAILURE;
    return st == -1 ? GOLDILOCKS_SUCCESS : GOLDILOCKS_FAILURE;
}
goldilocks_error_t goldilocks_sha3_final(goldilocks_keccak_sponge_p sponge, uint8_t *out, size_t len) {
    goldilocks_error_t ret = goldilocks_sha3_output(sponge, out, len);
    goldilocks_sha3_reset(sponge);
    return ret;
}
goldilocks_error_t goldilocks_sha3_hash(uint8_t *out, size_t outlen, const uint8_t *in, size_t inlen, const struct goldilocks_kparams_s *params) {
    goldilocks_keccak_sponge_p sponge;
    goldilocks_sha3_init(sponge, params);
    goldilocks_sha3_update(sponge, in, inlen);
    goldilocks_error_t ret = goldilocks_sha3_output(sponge, out, outlen);
    goldilocks_sha3_destroy(sponge);
    return ret;
}
size_t goldilocks_sha3_default_output_bytes(const goldilocks_keccak_sponge_p s) {
    const sponge_abi *h = (const sponge_abi *)s;
    return h->max_out == 0xFF ? (size_t)(200 - h->rate) : (size_t)((200 - h->rate) / 2);
}
size_t goldilocks_sha3_max_output_bytes(const goldilocks_keccak_sponge_p s) {
    const sponge_abi *h = (const sponge_abi *)s;
    return h->max_out == 0xFF ? SIZE_MAX : (size_t)((200 - h->rate) / 2);
}
// ---- sponge CSPRNG (reference spongerng.c:92-205): host composition of the streaming calls above ----
static void os_entropy(uint8_t *buf, size_t len) { /* stands in for the reference's RDRAND/RDTSC read (spongerng.c:28-90) */
    size_t got = 0;
    while (got < len) {
        ssize_t r = getrandom(buf + got, len - got, 0);
        if (r <= 0) break;
        got += (size_t)r;
    }
    if (got < len) { /* a non-deterministic generator without entropy must not keep going on zeros: fail closed */
        fprintf(stderr, "[goldilocks_b200] spongerng: getrandom() failed, no entropy available\n");
        abort();
    }
}
void goldilocks_spongerng_stir(goldilocks_keccak_prng_p prng, const uint8_t *in, size_t len) {
    uint8_t seed[32];
    (void)goldilocks_sha3_output(prng->sponge, seed, sizeof seed);
    const uint8_t nondet = SP(prng->sponge)->remaining;
    goldilocks_sha3_reset(prng->sponge);
    (void)goldilocks_sha3_update(prng->sponge, seed, sizeof seed);
    (void)goldilocks_sha3_update(prng->sponge, in, len);
    SP(prng->sponge)->remaining = nondet;
    goldilocks_bzero(seed, sizeof seed);
}
void goldilocks_spongerng_next(goldilocks_keccak_prng_p prng, uint8_t *out, size_t len) {
    uint8_t lenx[8];
    if (SP(prng->sponge)->remaining) { /* non-deterministic generator */
        uint8_t fresh[32] = {0};
        os_entropy(fresh, sizeof fresh);
        goldilocks_spongerng_stir(prng, fresh, sizeof fresh);
        goldilocks_bzero(fresh, sizeof fresh);
    }
    for (unsigned i = 0; i < sizeof lenx; i++) lenx[i] = (uint8_t)((uint64_t)len >> (8 * i));
    (void)goldilocks_sha3_update(prng->sponge, lenx, sizeof lenx);
    (void)goldilocks_sha3_output(prng->sponge, out, len);
    goldilocks_spongerng_stir(prng, lenx, 0);
}
void goldilocks_spongerng_init_from_buffer(goldilocks_keccak_prng_p prng, const uint8_t *in, size_t len, int deterministic) {
    goldilocks_sha3_init(prng->sponge, &GOLDILOCKS_SHAKE256_params_s);
    SP(prng->sponge)->remaining = !deterministic; /* the reference parks the flag in a field SHAKE ignores */
    goldilocks_spongerng_stir(prng, in, len);
}
goldilocks_error_t goldilocks_spongerng_init_from_file(goldilocks_keccak_prng_p prng, const char *file, size_t len, int deterministic) {
    uint8_t buffer[128];
    goldilocks_sha3_init(prng->sponge, &GOLDILOCKS_SHAKE256_params_s);
    SP(prng->sponge)->remaining = !deterministic;
    if (!len) return GOLDILOCKS_FAILURE;
    FILE *f = fopen(file, "rb");
    if (!f) return GOLDILOCKS_FAILURE;
    setvbuf(f, nullptr, _IONBF, 0); /* read exactly `len` bytes, like the reference's read(2) loop */
    while (len) {
        size_t got = fread(buffer, 1, len > sizeof buffer ? sizeof buffer : len, f);
        if (got == 0) { fclose(f); return GOLDILOCKS_FAILURE; }
        (void)goldilocks_sha3_update(prng->sponge, buffer, got);
        len -= got;
    }
    fclose(f);
    goldilocks_spongerng_stir(prng, buffer, 0);
    goldilocks_bzero(buffer, sizeof buffer);
    return GOLDILOCKS_SUCCESS;
}
goldilocks_error_t goldilocks_spongerng_init_from_dev_urandom(goldilocks_keccak_prng_p prng) {
    return goldilocks_spongerng_init_from_file(prng, "/dev/urandom", 64, 0);
}
void goldilocks_ed448_prehash_init(goldilocks_keccak_sponge_p hash) { goldilocks_sha3_init(hash, &GOLDILOCKS_SHAKE256_params_s); }
static void prehash_output(uint8_t ph[64], const goldilocks_keccak_sponge_p hash) {
    goldilocks_keccak_sponge_p too;
    memcpy(too, hash, sizeof(too));
    goldilocks_sha3_final(too, ph, 64);
    goldilocks_sha3_destroy(too);
}
void goldilocks_ed448_sign_prehash(uint8_t signature[114], const uint8_t privkey[57], const uint8_t pubkey[57], const goldilocks_keccak_sponge_p hash,
                                   const uint8_t *context, uint8_t context_len) {
    uint8_t ph[64];
    prehash_output(ph, hash);
    goldilocks_ed448_sign(signature, privkey, pubkey, ph, sizeof ph, 1, context, context_len);
    goldilocks_bzero(ph, sizeof ph);
}
goldilocks_error_t goldilocks_ed448_verify_prehash(const uint8_t signature[114], const uint8_t pubkey[57], const goldilocks_keccak_sponge_p hash,
                                                   const uint8_t *context, uint8_t context_len) {
    uint8_t ph[64];
    prehash_output(ph, hash);
    return goldilocks_ed448_verify(signature, pubkey, ph, sizeof ph, 1, context, context_len);
}
void goldilocks_448_scalar_add(goldilocks_448_scalar_p o, const goldilocks_448_scalar_p a, const goldilocks_448_scalar_p b) { goldilocks_448_scalar_add_batch(o, a, b, 1); }
void goldilocks_448_scalar_sub(goldilocks_448_scalar_p o, const goldilocks_448_scalar_p a, const goldilocks_448_scalar_p b) { goldilocks_448_scalar_sub_batch(o, a, b, 1); }
void goldilocks_448_scalar_mul(goldilocks_448_scalar_p o, const goldilocks_448_scalar_p a, const goldilocks_448_scalar_p b) { goldilocks_448_scalar_mul_batch(o, a, b, 1); }
void goldilocks_448_scalar_halve(goldilocks_448_scalar_p o, const goldilocks_448_scalar_p a) { goldilocks_448_scalar_halve_batch(o, a, 1); }
void goldilocks_448_scalar_decode_long(goldilocks_448_scalar_p o, const uint8_t *ser, size_t ser_len) { goldilocks_448_scalar_decode_long_batch(o, ser, ser_len, 1); }
goldilocks_error_t goldilocks_448_scalar_decode(goldilocks_448_scalar_p o, const uint8_t ser[56]) { /* scalar.c:234-249 */
    /* success iff the 448-bit value is < q: compare on the host (56 bytes), reduce on the device */
    static const uint8_t q_le[56] = {0xf3, 0x44, 0x58, 0xab, 0x92, 0xc2, 0x78, 0x23, 0x55, 0x8f, 0xc5, 0x8d, 0x72, 0xc2, 0x6c, 0x21, 0x90, 0x36, 0xd6, 0xae,
                                     0x49, 0xdb, 0x4e, 0xc4, 0xe9, 0x23, 0xca, 0x7c, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff,
                                     0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0xff, 0x3f};
    int borrow = 0; /* ser - q over all 56 bytes, no early exit: the value is often a secret scalar (the reference's loop, scalar.c:240-245) */
    for (int i = 0; i < 56; i++) borrow = ((int)ser[i] - (int)q_le[i] - borrow) >> 8 & 1;
    goldilocks_448_scalar_decode_long_batch(o, ser, 56, 1);
    return (goldilocks_error_t)(-borrow); /* borrow = 1 iff ser < q: SUCCESS = -1, FAILURE = 0 */
}
void goldilocks_448_scalar_encode(uint8_t ser[56], const goldilocks_448_scalar_p s) { memcpy(ser, s->limb, 56); }

}  // extern "C"
