// Host side of the data plane: engine, jobs and the C ABI (include/tsnap_b200.h).
//
// Save pipeline (one job = the raw-tensor WriteReqs of one Snapshot.take on this rank):
//
//   live tensors --pack kernels--> HBM staging arena --cudaMemcpyAsync(s_copy)--> pinned slot ring
//        (s_kernel, ~TB/s)              |  async_take returns here                  | completion thread
//                                        v                                           v
//                                  sources reusable                     I/O workers: pwrite(fd, slot, off)
//
// Load pipeline is the mirror: I/O workers pread into pinned slots, enqueue the H2D copy into the
// arena themselves, and the worker that uploads the last chunk of a wave launches the scatter
// kernels that write straight into the live (possibly strided / resharded) tensors.
//
// This replaces, for the requests it is handed, the asyncio state machine + ThreadPoolExecutor(4)
// of T:scheduler.py:222-339/386-446, the pageable `tensor.to("cpu")` of T:io_preparers/tensor.py:353,
// the per-member D2D copies + blocking `.cpu()` of T:batcher.py:144-159 and the aiofiles hop of
// T:storage_plugins/fs.py:28-51.
#include "engine.h"

#include <ctype.h>
#include <errno.h>
#include <sched.h>
#include <fcntl.h>
#include <string.h>
#include <dirent.h>
#include <sys/ipc.h>
#include <sys/mman.h>
#include <sys/resource.h>
#include <sys/sem.h>
#include <sys/syscall.h>
#include <sys/stat.h>
#include <sys/types.h>
#include <unistd.h>

#include <algorithm>
#include <cstdlib>

#include <nvtx3/nvToolsExt.h>

#include "kernels.h"

namespace tsnap {

// NVTX ranges make the pack / drain / write overlap visible in a timeline profiler (no-ops when none is attached)
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

static thread_local std::string g_err;
int set_err(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
const char* last_err() { return g_err.c_str(); }

#define CUDA_TRY(expr)                                                                        \
    do {                                                                                      \
        cudaError_t e__ = (expr);                                                             \
        if (e__ != cudaSuccess)                                                               \
            return set_err(TSNAP_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
    } while (0)

using clk = std::chrono::steady_clock;
static double ms_since(clk::time_point t0) { return std::chrono::duration<double, std::milli>(clk::now() - t0).count(); }

// ---- NUMA placement ---------------------------------------------------------------------------------------
// The pinned ring is first-touched by the drain thread and read by the I/O workers; keeping those threads on
// the socket the GPU's PCIe root complex belongs to keeps the DMA target and the page-cache copies local.
static void bind_current_thread(const std::vector<int>& cpus) {
    if (cpus.empty()) return;
    cpu_set_t set;
    CPU_ZERO(&set);
    for (int c : cpus)
        if (c >= 0 && c < CPU_SETSIZE) CPU_SET(c, &set);
    sched_setaffinity(0, sizeof(set), &set);
}

static std::vector<int> parse_cpulist(const std::string& s) {
    std::vector<int> out;
    size_t i = 0;
    while (i < s.size()) {
        while (i < s.size() && !isdigit(s[i])) ++i;
        if (i >= s.size()) break;
        int a = 0;
        while (i < s.size() && isdigit(s[i])) a = a * 10 + (s[i++] - '0');
        int b = a;
        if (i < s.size() && s[i] == '-') {
            ++i;
            b = 0;
            while (i < s.size() && isdigit(s[i])) b = b * 10 + (s[i++] - '0');
        }
        for (int c = a; c <= b; ++c) out.push_back(c);
    }
    return out;
}

static std::string read_small_file(const std::string& path) {
    FILE* f = fopen(path.c_str(), "r");
    if (!f) return "";
    char buf[4096];
    size_t n = fread(buf, 1, sizeof(buf) - 1, f);
    fclose(f);
    buf[n] = 0;
    return buf;
}

static std::vector<int> gpu_numa_cpus(int device) {
    // opt-in: on the measured 2-socket hosts confining the 16 writers to the GPU's socket LOWERED end-to-end
    // throughput (34 vs 39 GB/s, profiles/r01_ncu_summary.md) — the page-cache copy is memory-bound and
    // benefits from both sockets' channels — so the default leaves placement to the scheduler
    const char* env = getenv("TSNAP_B200_NUMA");
    if (!env || env[0] != '1') return {};
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) return {};
    std::string id(bus);
    for (char& c : id) c = char(tolower(c));
    std::string node = read_small_file("/sys/bus/pci/devices/" + id + "/numa_node");
    if (node.empty()) return {};
    int n = atoi(node.c_str());
    if (n < 0) return {};
    std::vector<int> cpus = parse_cpulist(read_small_file("/sys/devices/system/node/node" + std::to_string(n) + "/cpulist"));
    // respect the affinity the process was started with (taskset / cgroup cpusets)
    cpu_set_t cur;
    if (sched_getaffinity(0, sizeof(cur), &cur) == 0) {
        std::vector<int> allowed;
        for (int c : cpus)
            if (c < CPU_SETSIZE && CPU_ISSET(c, &cur)) allowed.push_back(c);
        cpus.swap(allowed);
    }
    return cpus;
}

// ---- host-wide I/O tokens -----------------------------------------------------------------------------------
// The kernel's buffered-write path peaks at ~16 concurrent writers per HOST and degrades beyond
// (profiles/r01_host_write_probe.json), so the engines of all ranks on a host draw every chunk I/O from one pool of
// tokens (a SysV semaphore: SEM_UNDO gives a killed process's tokens back).  A rank that drains alone — the last one
// of a take, a restore on fewer ranks than the save — gets the whole pool instead of a static 1/N share.
// TSNAP_B200_HOST_IO_TOKENS: pool size, 0 = off (default: off for one rank per host, 16 otherwise; see engine_create).
struct HostTokens {
    int semid = -1;
    void init(int tokens) {
        if (tokens <= 0) return;
        // one semaphore per (uid, pool size): engines configured with different pool sizes do not share a counter
        const key_t key = key_t(0x74530000 | ((tokens & 0xff) << 8) | (getuid() & 0xff));
        int id = semget(key, 1, IPC_CREAT | IPC_EXCL | 0600);
        if (id >= 0) {
            union semun_ {
                int val;
                struct semid_ds* buf;
                unsigned short* array;
            } arg;
            arg.val = tokens;
            if (semctl(id, 0, SETVAL, arg) != 0) return;
        } else {
            id = semget(key, 1, 0600);
            if (id < 0) return;
            // the creator may not have initialised it yet: sem_otime stays 0 until the first semop
            for (int i = 0; i < 100; ++i) {
                struct semid_ds ds;
                union semun_ {
                    int val;
                    struct semid_ds* buf;
                    unsigned short* array;
                } arg;
                arg.buf = &ds;
                if (semctl(id, 0, IPC_STAT, arg) == 0 && (ds.sem_otime != 0 || semctl(id, 0, GETVAL) > 0)) break;
                usleep(1000);
            }
        }
        semid = id;
    }
    void acquire() {
        if (semid < 0) return;
        struct sembuf op = {0, -1, SEM_UNDO};
        while (semop(semid, &op, 1) != 0 && errno == EINTR) {
        }
    }
    void release() {
        if (semid < 0) return;
        struct sembuf op = {0, 1, SEM_UNDO};
        while (semop(semid, &op, 1) != 0 && errno == EINTR) {
        }
    }
};
static HostTokens g_tokens;
struct TokenGuard {
    TokenGuard() { g_tokens.acquire(); }
    ~TokenGuard() { g_tokens.release(); }
};

// ---- host topology -------------------------------------------------------------------------------------------
struct NumaNode {
    int id;
    std::vector<int> cpus;   // allowed hardware threads
    std::vector<int> cores;  // first hardware thread of every allowed physical core
};
static std::vector<NumaNode> numa_nodes() {
    cpu_set_t cur;
    const bool have_aff = sched_getaffinity(0, sizeof(cur), &cur) == 0;
    std::vector<NumaNode> out;
    for (int node = 0; node < 64; ++node) {
        std::string cl = read_small_file("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist");
        if (cl.empty()) {
            if (node > 8) break;
            continue;
        }
        NumaNode n;
        n.id = node;
        for (int c : parse_cpulist(cl)) {
            if (have_aff && (c >= CPU_SETSIZE || !CPU_ISSET(c, &cur))) continue;
            n.cpus.push_back(c);
            std::vector<int> sib = parse_cpulist(read_small_file("/sys/devices/system/cpu/cpu" + std::to_string(c) + "/topology/thread_siblings_list"));
            if (sib.empty() || sib[0] == c) n.cores.push_back(c);
        }
        if (!n.cpus.empty()) out.push_back(n);
    }
    return out;
}

// Placement of the I/O workers (TSNAP_B200_IO_PIN):
//   none   leave it to the scheduler
//   local  all workers on the CPUs of the GPU's NUMA node
//   node   (default) workers split evenly over the NUMA nodes, each bound to its node's CPUs and serving that node's queue:
//          with TSNAP_B200_RING_NUMA=interleave every page-cache copy reads a pinned slot of the worker's own node
//   spread one physical core per worker, alternating between the NUMA nodes, offset by LOCAL_RANK so that ranks
//          sharing a host do not pile onto the same cores
static std::vector<WorkerSpec> io_worker_specs(int n, const std::vector<int>& gpu_node_cpus, const std::vector<int>& ring_nodes,
                                               int* n_queues) {
    const char* env = getenv("TSNAP_B200_IO_PIN");
    std::string mode = env ? env : "node";
    std::vector<WorkerSpec> out(size_t(n), WorkerSpec{});
    *n_queues = 1;
    if (mode == "local") {
        for (WorkerSpec& w : out) w.cpus = gpu_node_cpus;
        return out;
    }
    if (mode != "spread" && mode != "node") return out;
    const std::vector<NumaNode> nodes = numa_nodes();
    if (nodes.size() < 2 && mode == "node") return out;  // one node: nothing to be affine to
    if (nodes.empty()) return out;
    // queue q serves ring_nodes[q] when the ring is placed, else node q
    std::vector<const NumaNode*> qnode;
    if (!ring_nodes.empty()) {
        for (int id : ring_nodes)
            for (const NumaNode& nd : nodes)
                if (nd.id == id) qnode.push_back(&nd);
    }
    if (qnode.empty())
        for (const NumaNode& nd : nodes) qnode.push_back(&nd);
    *n_queues = int(qnode.size());
    const char* lr = getenv("LOCAL_RANK");
    const int rank = lr ? atoi(lr) : 0;
    for (int i = 0; i < n; ++i) {
        const int g = rank * n + i;  // global worker ordinal on this host
        const int q = i % int(qnode.size());
        out[size_t(i)].queue = q;
        const NumaNode& nd = *qnode[size_t(q)];
        if (mode == "node" || nd.cores.empty()) out[size_t(i)].cpus = nd.cpus;
        else out[size_t(i)].cpus = {nd.cores[(size_t(g) / qnode.size()) % nd.cores.size()]};
    }
    return out;
}

// ---- WorkerPool ---------------------------------------------------------------------------------------
static thread_local int g_lane = 0;  // ordinal of the current I/O worker (trace lanes)
WorkerPool::WorkerPool(const std::vector<WorkerSpec>& workers, int n_queues) {
    q_.resize(size_t(std::max(1, n_queues)));
    for (size_t i = 0; i < workers.size(); ++i) {
        const WorkerSpec w = workers[i];
        threads_.emplace_back([this, w, i] {
            g_lane = int(i);
            bind_current_thread(w.cpus);
            run(w.queue);
        });
    }
}
WorkerPool::~WorkerPool() {
    {
        std::lock_guard<std::mutex> g(mu_);
        stop_ = true;
    }
    cv_.notify_all();
    for (auto& t : threads_) t.join();
}
void WorkerPool::post(std::function<void()> fn, int queue) {
    {
        std::lock_guard<std::mutex> g(mu_);
        const size_t q = queue >= 0 ? size_t(queue) % q_.size() : (rr_++ % q_.size());
        q_[q].push_back(std::move(fn));
    }
    cv_.notify_all();
}
void WorkerPool::run(int home) {
    const size_t nq = q_.size();
    for (;;) {
        std::function<void()> fn;
        {
            std::unique_lock<std::mutex> g(mu_);
            size_t found = nq;
            for (;;) {
                // own node's queue first, then help the others out (a remote copy beats an idle worker)
                for (size_t k = 0; k < nq; ++k) {
                    const size_t q = (size_t(home) + k) % nq;
                    if (!q_[q].empty()) {
                        found = q;
                        break;
                    }
                }
                if (found < nq || stop_) break;
                cv_.wait(g);
            }
            if (found == nq) return;
            fn = std::move(q_[found].front());
            q_[found].pop_front();
        }
        fn();
    }
}

// ---- SlotRing -------------------------------------------------------------------------------------------
// anonymous memory bound to one NUMA node, faulted in, then pinned for DMA
static char* alloc_on_node(size_t len, int node, bool pin) {
    void* p = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (p == MAP_FAILED) return nullptr;
    unsigned long mask[4] = {0, 0, 0, 0};
    mask[size_t(node) / (8 * sizeof(unsigned long))] |= 1UL << (size_t(node) % (8 * sizeof(unsigned long)));
    const long rc = syscall(SYS_mbind, p, len, 2 /* MPOL_BIND */, mask, sizeof(mask) * 8 + 1, 0);
    if (rc != 0) {
        munmap(p, len);
        return nullptr;
    }
    madvise(p, len, MADV_HUGEPAGE);
    memset(p, 0, len);
    if (pin && cudaHostRegister(p, len, cudaHostRegisterDefault) != cudaSuccess) {
        cudaGetLastError();
        munmap(p, len);
        return nullptr;
    }
    return static_cast<char*>(p);
}

int SlotRing::init(size_t slot_bytes, int n, bool pinned, size_t slack, const std::vector<int>& nodes) {
    slot_bytes_ = slot_bytes;
    slack_ = slack;
    pinned_ = pinned;
    for (int i = 0; i < n; ++i) {
        void* p = nullptr;
        size_t maplen = 0;
        int queue = -1;
        if (!nodes.empty()) {
            const size_t len = (slot_bytes + slack + (2u << 20) - 1) / (2u << 20) * (2u << 20);
            p = alloc_on_node(len, nodes[size_t(i) % nodes.size()], pinned);
            if (p) {
                maplen = len;
                queue = int(size_t(i) % nodes.size());
            }
        }
        if (!p && pinned) {
            // cudaHostAlloc returns page-aligned memory: fit for O_DIRECT as it is
            cudaError_t e = cudaHostAlloc(&p, slot_bytes + slack, cudaHostAllocDefault);
            if (e != cudaSuccess) return set_err(TSNAP_ECUDA, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
        } else if (!p) {
            if (posix_memalign(&p, 4096, slot_bytes + slack) != 0) return set_err(TSNAP_ENOMEM, "posix_memalign failed");
        }
        placed_.push_back(Placed{static_cast<char*>(p), maplen, queue});
        all_.push_back(static_cast<char*>(p));
        free_.push_back(static_cast<char*>(p));
    }
    return TSNAP_OK;
}
void SlotRing::destroy() {
    for (const Placed& s : placed_) {
        if (s.len) {
            if (pinned_) cudaHostUnregister(s.p);
            munmap(s.p, s.len);
        } else if (pinned_) {
            cudaFreeHost(s.p);
        } else {
            free(s.p);
        }
    }
    placed_.clear();
    all_.clear();
    free_.clear();
}
int SlotRing::queue_of(const char* p) const {
    for (const Placed& s : placed_)
        if (s.p == p) return s.queue;
    return -1;
}
char* SlotRing::acquire() {
    std::unique_lock<std::mutex> g(mu_);
    cv_.wait(g, [this] { return !free_.empty(); });
    char* p = free_.back();
    free_.pop_back();
    return p;
}
void SlotRing::release(char* p) {
    {
        std::lock_guard<std::mutex> g(mu_);
        free_.push_back(p);
    }
    cv_.notify_one();
}

// ---- small file helpers -----------------------------------------------------------------------------------
static int make_parent_dirs(const std::string& path) {
    size_t pos = path.rfind('/');
    if (pos == std::string::npos || pos == 0) return 0;
    std::string dir = path.substr(0, pos);
    struct stat st;
    if (stat(dir.c_str(), &st) == 0) return 0;
    for (size_t i = 1; i <= dir.size(); ++i) {
        if (i == dir.size() || dir[i] == '/') {
            std::string sub = dir.substr(0, i);
            if (mkdir(sub.c_str(), 0777) != 0 && errno != EEXIST) return -1;
        }
    }
    return 0;
}
static int pwrite_all(int fd, const char* p, size_t n, uint64_t off) {
    while (n > 0) {
        ssize_t w = pwrite(fd, p, n, off_t(off));
        if (w < 0) {
            if (errno == EINTR) continue;
            return -1;
        }
        p += w;
        n -= size_t(w);
        off += uint64_t(w);
    }
    return 0;
}
static int pread_all(int fd, char* p, size_t n, uint64_t off) {
    while (n > 0) {
        ssize_t r = pread(fd, p, n, off_t(off));
        if (r < 0) {
            if (errno == EINTR) continue;
            return -1;
        }
        if (r == 0) {
            errno = ENODATA;  // short file
            return -1;
        }
        p += r;
        n -= size_t(r);
        off += uint64_t(r);
    }
    return 0;
}

static inline uint64_t align_up(uint64_t x, uint64_t a) { return (x + a - 1) / a * a; }

}  // namespace tsnap

using namespace tsnap;

// ---- job plumbing -----------------------------------------------------------------------------------------
void tsnap_job::fail(int code, const std::string& msg) {
    std::lock_guard<std::mutex> g(mu);
    if (err_code == 0) {
        err_code = code;
        err_msg = msg;
    }
}
void tsnap_job::add_trace(int kind, int lane, int file, double t0, double t1, uint64_t bytes) {
    std::lock_guard<std::mutex> g(trace_mu);
    trace.push_back(tsnap_trace_rec{kind, lane, file, 0, t0, t1, bytes});
}
char* tsnap_job::take_slot() {
    {
        std::unique_lock<std::mutex> g(slot_mu);
        slot_cv.wait(g, [this] { return max_slots <= 0 || slots_held < max_slots; });
        ++slots_held;
        slots_peak = std::max(slots_peak, slots_held);
    }
    return eng->ring.acquire();
}
void tsnap_job::give_slot(char* p) {
    eng->ring.release(p);
    {
        std::lock_guard<std::mutex> g(slot_mu);
        --slots_held;
    }
    slot_cv.notify_one();
}
bool tsnap_job::failed() {
    std::lock_guard<std::mutex> g(mu);
    return err_code != 0;
}
void tsnap_job::part_done() {
    if (parts_left.fetch_sub(1, std::memory_order_acq_rel) == 1) {
        if (holds_arena) {
            {
                std::lock_guard<std::mutex> ga(eng->arena_mu);
                eng->arena_in_use = false;
            }
            eng->arena_cv.notify_all();
        }
        eng->active_jobs.fetch_sub(1, std::memory_order_acq_rel);
        std::lock_guard<std::mutex> g(mu);
        stats.total_ms = ms_since(t_submit);
        if (!device_done) {
            device_done = true;
            stats.device_done_ms = stats.total_ms;
        }
        done = true;
        cv.notify_all();
    }
}

cudaEvent_t tsnap_engine::get_event() {
    {
        std::lock_guard<std::mutex> g(ev_mu);
        if (!ev_free.empty()) {
            cudaEvent_t e = ev_free.back();
            ev_free.pop_back();
            return e;
        }
    }
    cudaEvent_t e = nullptr;
    cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    return e;
}
void tsnap_engine::put_event(cudaEvent_t e) {
    std::lock_guard<std::mutex> g(ev_mu);
    ev_free.push_back(e);
}

void* tsnap_engine::get_table(size_t bytes, size_t* cap) {
    {
        std::lock_guard<std::mutex> g(tbl_mu);
        size_t best = SIZE_MAX;
        for (size_t i = 0; i < tbl_free.size(); ++i)
            if (tbl_free[i].first >= bytes && (best == SIZE_MAX || tbl_free[i].first < tbl_free[best].first)) best = i;
        if (best != SIZE_MAX) {
            auto kv = tbl_free[best];
            tbl_free.erase(tbl_free.begin() + best);
            *cap = kv.first;
            return kv.second;
        }
    }
    const size_t c = std::max<size_t>((bytes + (1u << 20) - 1) >> 20 << 20, 1u << 20);
    void* p = nullptr;
    if (cudaMalloc(&p, c) != cudaSuccess) return nullptr;
    *cap = c;
    return p;
}
void tsnap_engine::put_table(void* p, size_t cap) {
    std::lock_guard<std::mutex> g(tbl_mu);
    tbl_free.emplace_back(cap, p);
}

static void push_pending(tsnap_engine* eng, cudaEvent_t ev, std::function<void(bool)> fn) {
    {
        std::lock_guard<std::mutex> g(eng->c_mu);
        eng->pending.push_back({ev, std::move(fn)});
    }
    eng->c_cv.notify_one();
}

static void completion_main(tsnap_engine* eng) {
    bind_current_thread(eng->numa_cpus);
    cudaSetDevice(eng->device);
    for (;;) {
        tsnap_engine::Pending p;
        {
            std::unique_lock<std::mutex> g(eng->c_mu);
            eng->c_cv.wait(g, [eng] { return eng->stopping || !eng->pending.empty(); });
            if (eng->pending.empty()) return;
            p = std::move(eng->pending.front());
            eng->pending.pop_front();
        }
        cudaError_t e = cudaEventSynchronize(p.ev);
        p.done(e == cudaSuccess);
    }
}

// ---- planning of one wave ----------------------------------------------------------------------------------
static int plan_wave(tsnap_job* job, Wave& w) {
    if (w.direct) return TSNAP_OK;
    tsnap_engine* eng = job->eng;
    std::string err;
    for (int fi : w.files) {
        FileSpec& f = job->files[fi];
        const uint64_t wire_base = uint64_t(uintptr_t(job->arena)) + w.region_off + f.arena_off;
        for (const tsnap_copy_desc& d : f.members) {
            NormalizedCopy nc;
            int rc = normalize_copy(d, wire_base, eng->allow_bulk, &nc, &err);
            if (rc != TSNAP_OK) return set_err(rc, "member of " + f.path + ": " + err);
            for (int k = 0; k < nc.n; ++k) {
                Member& m = nc.m[k];
                if (eng->allow_bulk && m.mode == kModeTranspose && m.bytes) {
                    // addresses are final here: transposes the TMA unit can address get their tensor maps and move to its kernel
                    TmaPair tp;
                    uint32_t variant = 0;
                    if (make_tma_pair(m, &tp, &variant)) {
                        m.mode = kModeTransposeTma;
                        m.shift = (m.shift & 0xffffu) | (variant << kTmaVariantShift);
                        m.q_zero_point = int64_t(w.tmaps.size());
                        w.tmaps.push_back(tp);
                    }
                }
                if (m.mode == kModeRows && m.bytes) {
                    TmaPair tp;
                    if (make_rows_tma_pair(m, &tp)) {  // short runs: a box of many runs per TMA request
                        m.mode = kModeRowsTma;
                        m.q_zero_point = int64_t(w.tmaps.size());
                        w.tmaps.push_back(tp);
                    }
                }
                const uint64_t nt = tile_count(m);
                if (nt == 0) continue;
                const uint32_t mi = uint32_t(w.members.size());
                w.members.push_back(m);
                std::vector<Tile>& tv = m.mode == kModeRowsTma ? w.tiles_rows_tma : m.mode == kModeBulk ? w.tiles_bulk : m.mode == kModeRows ? w.tiles_rows : m.mode == kModeStrided ? w.tiles_strided : m.mode == kModeTranspose ? w.tiles_transpose : m.mode == kModeTransposeTma ? w.tiles_tma : w.tiles_lsu;
                (m.mode == kModeBulk ? job->stats.bytes_bulk : (m.mode == kModeRows || m.mode == kModeRowsTma) ? job->stats.bytes_rows : job->stats.bytes_lsu) += m.bytes;
                for (uint64_t t = 0; t < nt; ++t) tv.push_back(Tile{mi, uint32_t(t)});
            }
        }
    }
    job->stats.n_tiles_bulk += w.tiles_bulk.size();
    job->stats.n_tiles_rows += w.tiles_rows.size() + w.tiles_rows_tma.size();
    job->stats.n_tiles_lsu += w.tiles_lsu.size() + w.tiles_strided.size() + w.tiles_transpose.size() + w.tiles_tma.size();
    return TSNAP_OK;
}

// copies the tables to the device and launches both kernels on s_kernel; records timing events
static int launch_wave(tsnap_job* job, Wave& w) {
    tsnap_engine* eng = job->eng;
    const size_t mb = w.members.size() * sizeof(Member);
    const size_t bb = w.tiles_bulk.size() * sizeof(Tile);
    const size_t rb = w.tiles_rows.size() * sizeof(Tile);
    const size_t lb = w.tiles_lsu.size() * sizeof(Tile);
    const size_t sb2 = w.tiles_strided.size() * sizeof(Tile);
    const size_t tb2 = w.tiles_transpose.size() * sizeof(Tile);
    const size_t tmb = w.tiles_tma.size() * sizeof(Tile), mpb = w.tmaps.size() * sizeof(TmaPair), rtb = w.tiles_rows_tma.size() * sizeof(Tile);
    w.table_bytes = align_up(mb, 256) + align_up(bb, 256) + align_up(rb, 256) + align_up(lb, 256) + align_up(sb2, 256) + align_up(tb2, 256) + align_up(tmb, 256) + align_up(mpb, 256) + align_up(rtb, 256);
    CUDA_TRY(cudaEventCreate(&w.ev_k0));
    CUDA_TRY(cudaEventCreate(&w.ev_k1));
    CUDA_TRY(cudaEventCreate(&w.ev_kr));
    CUDA_TRY(cudaEventCreate(&w.ev_k2));
    CUDA_TRY(cudaEventCreateWithFlags(&w.ev_done, cudaEventDisableTiming));
    if (w.members.empty()) {
        CUDA_TRY(cudaEventRecord(w.ev_k0, eng->s_kernel));
        CUDA_TRY(cudaEventRecord(w.ev_k1, eng->s_kernel));
        CUDA_TRY(cudaEventRecord(w.ev_kr, eng->s_kernel));
        CUDA_TRY(cudaEventRecord(w.ev_k2, eng->s_kernel));
        CUDA_TRY(cudaEventRecord(w.ev_done, eng->s_kernel));
        return TSNAP_OK;
    }
    w.d_tables = eng->get_table(w.table_bytes, &w.table_cap);  // returned to the pool when the job is destroyed
    if (!w.d_tables) return set_err(TSNAP_ECUDA, "out of device memory for the launch tables");
    char* d = static_cast<char*>(w.d_tables);
    Member* d_members = reinterpret_cast<Member*>(d);
    Tile* d_bulk = reinterpret_cast<Tile*>(d + align_up(mb, 256));
    Tile* d_rows = reinterpret_cast<Tile*>(d + align_up(mb, 256) + align_up(bb, 256));
    Tile* d_lsu = reinterpret_cast<Tile*>(d + align_up(mb, 256) + align_up(bb, 256) + align_up(rb, 256));
    Tile* d_strided = reinterpret_cast<Tile*>(d + align_up(mb, 256) + align_up(bb, 256) + align_up(rb, 256) + align_up(lb, 256));
    Tile* d_transpose = reinterpret_cast<Tile*>(d + align_up(mb, 256) + align_up(bb, 256) + align_up(rb, 256) + align_up(lb, 256) + align_up(sb2, 256));
    Tile* d_tma = reinterpret_cast<Tile*>(reinterpret_cast<char*>(d_transpose) + align_up(tb2, 256));
    TmaPair* d_maps = reinterpret_cast<TmaPair*>(reinterpret_cast<char*>(d_tma) + align_up(tmb, 256));
    Tile* d_rows_tma = reinterpret_cast<Tile*>(reinterpret_cast<char*>(d_maps) + align_up(mpb, 256));
    // pageable sources: the runtime stages them before returning, so the vectors may be freed later
    CUDA_TRY(cudaMemcpyAsync(d_members, w.members.data(), mb, cudaMemcpyHostToDevice, eng->s_kernel));
    if (bb) CUDA_TRY(cudaMemcpyAsync(d_bulk, w.tiles_bulk.data(), bb, cudaMemcpyHostToDevice, eng->s_kernel));
    if (rb) CUDA_TRY(cudaMemcpyAsync(d_rows, w.tiles_rows.data(), rb, cudaMemcpyHostToDevice, eng->s_kernel));
    if (lb) CUDA_TRY(cudaMemcpyAsync(d_lsu, w.tiles_lsu.data(), lb, cudaMemcpyHostToDevice, eng->s_kernel));
    if (sb2) CUDA_TRY(cudaMemcpyAsync(d_strided, w.tiles_strided.data(), sb2, cudaMemcpyHostToDevice, eng->s_kernel));
    if (tb2) CUDA_TRY(cudaMemcpyAsync(d_transpose, w.tiles_transpose.data(), tb2, cudaMemcpyHostToDevice, eng->s_kernel));
    if (tmb) CUDA_TRY(cudaMemcpyAsync(d_tma, w.tiles_tma.data(), tmb, cudaMemcpyHostToDevice, eng->s_kernel));
    if (mpb) CUDA_TRY(cudaMemcpyAsync(d_maps, w.tmaps.data(), mpb, cudaMemcpyHostToDevice, eng->s_kernel));
    if (rtb) CUDA_TRY(cudaMemcpyAsync(d_rows_tma, w.tiles_rows_tma.data(), rtb, cudaMemcpyHostToDevice, eng->s_kernel));
    job->stats.table_h2d_bytes += mb + bb + rb + lb + sb2 + tb2 + tmb + mpb + rtb;
    CUDA_TRY(cudaEventRecord(w.ev_k0, eng->s_kernel));
    CUDA_TRY(launch_bulk(d_members, d_bulk, uint32_t(w.tiles_bulk.size()), eng->sm_count, eng->s_kernel));
    CUDA_TRY(cudaEventRecord(w.ev_k1, eng->s_kernel));
    CUDA_TRY(launch_rows(d_members, d_rows, uint32_t(w.tiles_rows.size()), eng->sm_count, eng->s_kernel));
    CUDA_TRY(launch_rows_tma(d_members, d_rows_tma, d_maps, uint32_t(w.tiles_rows_tma.size()), eng->sm_count, eng->s_kernel));
    CUDA_TRY(cudaEventRecord(w.ev_kr, eng->s_kernel));
    CUDA_TRY(launch_lsu(d_members, d_lsu, uint32_t(w.tiles_lsu.size()), eng->sm_count, eng->s_kernel, kLsuDefault));
    CUDA_TRY(launch_lsu(d_members, d_strided, uint32_t(w.tiles_strided.size()), eng->sm_count, eng->s_kernel, kLsuStrided));
    CUDA_TRY(launch_lsu(d_members, d_transpose, uint32_t(w.tiles_transpose.size()), eng->sm_count, eng->s_kernel, kLsuTranspose));
    CUDA_TRY(launch_transpose_tma(d_members, d_tma, d_maps, uint32_t(w.tiles_tma.size()), eng->sm_count, eng->s_kernel));
    CUDA_TRY(cudaEventRecord(w.ev_k2, eng->s_kernel));
    CUDA_TRY(cudaEventRecord(w.ev_done, eng->s_kernel));
    const int nl = (w.tiles_bulk.empty() ? 0 : 1) + (w.tiles_rows.empty() ? 0 : 1) + (w.tiles_lsu.empty() ? 0 : 1) + (w.tiles_strided.empty() ? 0 : 1) + (w.tiles_transpose.empty() ? 0 : 1) + (w.tiles_tma.empty() ? 0 : 1) + (w.tiles_rows_tma.empty() ? 0 : 1);
    job->stats.n_kernel_launches += nl;
    eng->kernels_launched += nl;
    return TSNAP_OK;
}

static void collect_wave_timing(tsnap_job* job, Wave& w) {
    float a = 0, r = 0, b = 0;
    if (w.timed || !w.ev_k0) return;
    if (cudaEventElapsedTime(&a, w.ev_k0, w.ev_k1) == cudaSuccess && cudaEventElapsedTime(&r, w.ev_k1, w.ev_kr) == cudaSuccess &&
        cudaEventElapsedTime(&b, w.ev_kr, w.ev_k2) == cudaSuccess) {
        std::lock_guard<std::mutex> g(job->mu);
        w.timed = true;
        job->stats.kernel_bulk_ms += a;
        job->stats.kernel_rows_ms += r;
        job->stats.kernel_lsu_ms += b;
        job->stats.kernel_ms += a + r + b;
        w.kernel_ms = a + r + b;
    }
}

// What a job asks of the HBM staging arena.
struct ArenaNeed {
    uint64_t total = 0, largest = 0;          // all device files
    uint64_t nd_total = 0, nd_largest = 0;    // files that cannot be drained without staging (strided / cast members)
};
static ArenaNeed arena_need(const tsnap_job* job) {
    ArenaNeed n;
    for (const FileSpec& f : job->files) {
        if (f.host_only || f.nbytes == 0) continue;
        const uint64_t fb = align_up(f.nbytes, 256);
        n.total += fb;
        n.largest = std::max(n.largest, fb);
        if (!f.dense) {
            n.nd_total += fb;
            n.nd_largest = std::max(n.nd_largest, fb);
        }
    }
    return n;
}

// Engine-owned arena (callers that lend none): grow towards the best operating point that fits — the whole
// payload, else two half-arenas of the largest file, else just the strided files — and never fail: with no arena
// at all the job drains dense members straight from the live tensors (the reference's fallback when its GPU slab
// allocation OOMs is a CPU slab, T:batcher.py:144-152).
static void ensure_arena(tsnap_engine* eng, const ArenaNeed& need) {
    if (need.total <= eng->arena_bytes) return;
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return;
    const uint64_t reserve = std::max<uint64_t>(total_b / 8, 4ull << 30);
    uint64_t allowed = eng->arena_bytes + (free_b > reserve ? free_b - reserve : 0);
    if (eng->cfg.hbm_staging_bytes) allowed = std::min<uint64_t>(allowed, eng->cfg.hbm_staging_bytes);
    // candidate sizes, best first: the whole payload; as much as the reserve policy allows when that still holds two
    // largest files (multi-wave); else only what the strided files need — that much is taken even below the reserve
    // line, because those members cannot be drained without staging
    uint64_t cands[4] = {0, 0, 0, 0};
    if (need.total <= allowed) cands[0] = need.total;
    else if (allowed >= 2 * need.largest) cands[1] = allowed;
    if (need.nd_total && need.nd_total <= allowed) cands[2] = need.nd_total;
    cands[3] = std::min(need.nd_total, 2 * need.nd_largest);
    for (int i = 0; i < 4; ++i) {
        if (cands[i] == 0) continue;
        const uint64_t target = align_up(cands[i], 2ull << 20);
        if (target <= eng->arena_bytes) return;  // what we hold is already as good as this candidate
        if (target > eng->arena_bytes + free_b) continue;
        if (eng->arena) {
            cudaStreamSynchronize(eng->s_kernel);
            cudaStreamSynchronize(eng->s_copy);
            cudaFree(eng->arena);
            eng->arena = nullptr;
            eng->arena_bytes = 0;
        }
        void* p = nullptr;
        if (cudaMalloc(&p, target) == cudaSuccess) {
            eng->arena = static_cast<char*>(p);
            eng->arena_bytes = target;
            return;
        }
        cudaGetLastError();  // clear the OOM and look again at what is free
        cudaMemGetInfo(&free_b, &total_b);
    }
}

static int ensure_ring(tsnap_engine* eng) {
    if (eng->ring.count() > 0) return TSNAP_OK;
    size_t sb = eng->cfg.pinned_slot_bytes ? eng->cfg.pinned_slot_bytes : (32ull << 20);
    sb = align_up(sb, 4096);
    const int n = eng->cfg.pinned_slots ? eng->cfg.pinned_slots : 32;
    return eng->ring.init(sb, n, eng->has_device, 8192, eng->ring_nodes);
}

// Decides, per device file, between staging in the arena (pack/scatter kernels) and the direct link path, and
// groups the staged files into waves that fit the arena.  job->waves = staged waves, then at most one direct wave.
static int build_waves(tsnap_job* job) {
    tsnap_engine* eng = job->eng;
    const ArenaNeed all = arena_need(job);
    if (all.total == 0) return TSNAP_OK;
    if (!eng->has_device) return set_err(TSNAP_ECUDA, "job has device members but the engine is host-only");
    // TSNAP_ENGINE_NO_ARENA: dense members never go through HBM staging; strided/converting ones still have to
    ArenaNeed need = all;
    if (eng->no_arena) {
        need.total = all.nd_total;
        need.largest = all.nd_largest;
    }
    if (!job->arena_set) {
        if (need.total) ensure_arena(eng, need);
        job->arena = eng->arena;
        job->arena_bytes = eng->arena_bytes;
    }
    const uint64_t A = job->arena_bytes;
    bool stage_dense;
    uint64_t staged_total, staged_largest;
    if (!eng->no_arena && (A >= all.total || (A >= 2 * all.largest && all.largest > 0))) {
        stage_dense = true;
        staged_total = all.total;
        staged_largest = all.largest;
    } else {
        stage_dense = false;
        staged_total = all.nd_total;
        staged_largest = all.nd_largest;
        if (staged_total > A && 2 * staged_largest > A)
            return set_err(TSNAP_ECUDA, "not enough HBM staging for the strided/converting members: have " + std::to_string(A) +
                                            " bytes, need " + std::to_string(std::min(staged_total, 2 * staged_largest)));
    }
    const bool single = staged_total <= A;
    const uint64_t cap = single ? A : (A / 2) / 256 * 256;
    std::vector<int> direct_files, staged_files;
    for (size_t i = 0; i < job->files.size(); ++i) {
        FileSpec& f = job->files[i];
        if (f.host_only || f.nbytes == 0) continue;
        if (f.dense && !stage_dense) {
            f.direct = true;
            std::sort(f.segs.begin(), f.segs.end(), [](const FileSpec::Seg& x, const FileSpec::Seg& y) { return x.off < y.off; });
            direct_files.push_back(int(i));
            job->stats.direct_bytes += f.nbytes;
            continue;
        }
        staged_files.push_back(int(i));
    }
    // A job that fits the arena is still cut in two launches so that the link never waits for a full-size kernel:
    // on save a small head wave (its D2H starts ~0.1 ms after submit while the big pack launch runs behind it), on
    // restore a small tail wave (the only scatter that nothing overlaps is ~0.1 ms instead of the whole payload's 5 ms).
    size_t split = SIZE_MAX;  // first file of the second wave
    if (single && staged_total > (1ull << 30) && staged_files.size() >= 2) {
        const uint64_t small = 128ull << 20;
        uint64_t acc = 0;
        if (job->kind == kSave) {
            for (size_t k = 0; k + 1 < staged_files.size(); ++k) {
                acc += align_up(job->files[staged_files[k]].nbytes, 256);
                if (acc >= small) {
                    split = k + 1;
                    break;
                }
            }
        } else if (job->kind == kLoad) {
            for (size_t k = staged_files.size() - 1; k >= 1; --k) {
                acc += align_up(job->files[staged_files[k]].nbytes, 256);
                if (acc >= small) {
                    split = k;
                    break;
                }
            }
        }
    }
    for (size_t k = 0; k < staged_files.size(); ++k) {
        FileSpec& f = job->files[staged_files[k]];
        const uint64_t fb = align_up(f.nbytes, 256);
        if (job->waves.empty() || job->waves.back().bytes + fb > cap || k == split) job->waves.emplace_back();
        Wave& w = job->waves.back();
        f.arena_off = w.bytes;
        f.wave = int(job->waves.size()) - 1;
        w.bytes += fb;
        w.files.push_back(staged_files[k]);
    }
    if (single) {
        uint64_t off = 0;  // waves of a job that fits sit side by side
        for (Wave& w : job->waves) {
            w.region_off = off;
            off += w.bytes;
        }
    } else {
        for (size_t i = 0; i < job->waves.size(); ++i) job->waves[i].region_off = (i % 2) * cap;
    }
    job->n_staged_waves = job->waves.size();
    job->stats.n_waves = job->waves.size();
    job->stats.arena_bytes = job->waves.empty() ? 0 : A;
    if (!direct_files.empty()) {
        job->waves.emplace_back();
        Wave& w = job->waves.back();
        w.direct = true;
        w.files = direct_files;
        for (int fi : direct_files) job->files[fi].wave = int(job->waves.size()) - 1;
    }
    return TSNAP_OK;
}

// ---- host-only files -----------------------------------------------------------------------------------
// true when the file is exactly one dense, cast-free member that covers it: I/O goes straight
// from/to the tensor's own memory (the reference's zero-copy tensor_as_memoryview, T:serialization.py:177-204)
static bool direct_host_member(const FileSpec& f, bool save, Member* out) {
    if (f.members.size() != 1) return false;
    NormalizedCopy nc;
    std::string err;
    if (normalize_copy(f.members[0], 0, false, &nc, &err) != TSNAP_OK || nc.n != 1) return false;
    const Member& m = nc.m[0];
    if (m.mode != kModeContig || m.bytes != f.nbytes) return false;
    if ((save ? m.dst : m.src) != 0) return false;
    *out = m;
    return true;
}

static void finish_file_part(tsnap_job* job, FileSpec& f, uint64_t bytes_io, bool save) {
    if (save) job->eng->bytes_written += bytes_io;
    else job->eng->bytes_read += bytes_io;
    if (f.parts_left.fetch_sub(1, std::memory_order_acq_rel) == 1) {
        std::lock_guard<std::mutex> g(f.open_mu);
        if (f.fd >= 0) {
            // O_DIRECT tails were written padded to a whole block: cut the file back to its size
            if (save && f.direct_io && (f.nbytes & 4095) && ftruncate(f.fd, off_t(f.nbytes)) != 0)
                job->fail(TSNAP_EIO, "ftruncate " + f.path + ": " + strerror(errno));
            if (save && (job->eng->cfg.flags & TSNAP_ENGINE_FSYNC)) fsync(f.fd);
            close(f.fd);
            f.fd = -1;
        }
    }
    job->part_done();
}

// Files are opened by the worker that performs their first I/O and closed by the one that performs the last:
// at most (workers + ring slots) descriptors are open at a time however many files the job has (the reference
// keeps <= 16 I/Os in flight, T:knobs.py:38), and the creates overlap the drain instead of preceding it.
static bool ensure_open(tsnap_job* job, FileSpec& f, bool save) {
    std::lock_guard<std::mutex> g(f.open_mu);
    if (f.opened) return !f.open_failed;
    f.opened = true;
    const double t0 = job->eng->trace ? job->now_ms() : 0;
    if (save && make_parent_dirs(f.path) != 0) {
        f.open_failed = true;
        job->fail(TSNAP_EIO, "mkdir for " + f.path + ": " + strerror(errno));
        return false;
    }
    const int base = save ? (O_WRONLY | O_CREAT | O_TRUNC) : O_RDONLY;
    // host-only files do their I/O from/to tensor memory of arbitrary alignment: always buffered
    const bool want_direct = job->eng->odirect && !f.host_only;
    if (want_direct) {
        f.fd = open(f.path.c_str(), base | O_DIRECT, 0644);
        f.direct_io = f.fd >= 0;
    }
    if (f.fd < 0) f.fd = open(f.path.c_str(), base, 0644);
    if (f.fd < 0) {
        f.open_failed = true;
        job->fail(TSNAP_EIO, "open " + f.path + ": " + strerror(errno));
        return false;
    }
    if (job->eng->trace) job->add_trace(TSNAP_TR_OPEN, g_lane, int(&f - &job->files[0]), t0, job->now_ms(), 0);
    return true;
}

// one chunk of a file from a ring slot (capacity >= slot_bytes + slack, 4 KiB aligned)
static int write_chunk(FileSpec& f, const char* slot, uint64_t n, uint64_t lo) {
    if (!f.direct_io) return pwrite_all(f.fd, slot, n, lo);
    // lo is a multiple of the slot size (a multiple of 4 KiB); only the last chunk of a file is ragged
    return pwrite_all(f.fd, slot, align_up(n, 4096), lo);
}
// reads file bytes [off, off+n) into the slot; *skip = where they start inside it
static int read_chunk(FileSpec& f, char* slot, uint64_t n, uint64_t off, uint64_t* skip) {
    *skip = 0;
    if (!f.direct_io) return pread_all(f.fd, slot, n, off);
    const uint64_t a = off & ~uint64_t(4095);
    const uint64_t want = align_up(off + n, 4096) - a;  // <= n + 8190 <= slot capacity
    *skip = off - a;
    uint64_t got = 0;
    while (got < *skip + n) {
        ssize_t r = pread(f.fd, slot + got, want - got, off_t(a + got));
        if (r < 0) {
            if (errno == EINTR) continue;
            return -1;
        }
        if (r == 0) {
            errno = ENODATA;
            return -1;
        }
        got += uint64_t(r);
        if (got & 4095) break;  // short read at the end of the file
    }
    if (got < *skip + n) {
        errno = ENODATA;
        return -1;
    }
    return 0;
}

// number of I/O parts a file contributes
static int64_t count_parts(tsnap_engine* eng, const FileSpec& f, bool save) {
    if (f.nbytes == 0) return save ? 1 : 0;  // an empty file still has to be created on save
    const uint64_t sb = eng->ring.slot_bytes();
    if (f.host_only) {
        Member m;
        // direct reads run in parallel parts (shared inode lock); direct writes of one file are one sequential
        // part: buffered writes serialise on the inode lock anyway, parallel parts only add contention
        if (!save && direct_host_member(f, save, &m)) return int64_t((f.nbytes + sb - 1) / sb);
        return 1;
    }
    return int64_t((f.nbytes + sb - 1) / sb);
}

static void post_host_file(tsnap_job* job, int fi, bool save) {
    tsnap_engine* eng = job->eng;
    FileSpec& f = job->files[fi];
    const uint64_t sb = eng->ring.slot_bytes();
    if (f.nbytes == 0) {
        if (save)
            eng->io->post([job, &f] {
                ensure_open(job, f, true);
                finish_file_part(job, f, 0, true);
            });
        return;
    }
    Member dm;
    if (save && direct_host_member(f, save, &dm)) {
        eng->io->post([job, &f, dm, sb] {
            if (!job->failed() && ensure_open(job, f, true)) {
                for (uint64_t lo = 0; lo < f.nbytes && !job->failed(); lo += sb) {
                    const uint64_t n = std::min<uint64_t>(sb, f.nbytes - lo);
                    if (pwrite_all(f.fd, reinterpret_cast<const char*>(uintptr_t(dm.src)) + lo, n, lo) != 0)
                        job->fail(TSNAP_EIO, "pwrite " + f.path + ": " + strerror(errno));
                }
            }
            finish_file_part(job, f, f.nbytes, true);
        });
        return;
    }
    if (direct_host_member(f, save, &dm)) {
        for (uint64_t lo = 0; lo < f.nbytes; lo += sb) {
            const uint64_t n = std::min(sb, f.nbytes - lo);
            eng->io->post([job, &f, dm, lo, n] {
                if (!job->failed() && ensure_open(job, f, false)) {
                    if (pread_all(f.fd, reinterpret_cast<char*>(uintptr_t(dm.dst)) + lo, n, f.offset + lo) != 0)
                        job->fail(TSNAP_EIO, "pread " + f.path + ": " + strerror(errno));
                }
                finish_file_part(job, f, n, false);
            });
        }
        return;
    }
    eng->io->post([job, &f, save] {
        if (!job->failed() && ensure_open(job, f, save)) {
            char* tmp = static_cast<char*>(malloc(f.nbytes));
            if (!tmp) {
                job->fail(TSNAP_ENOMEM, "malloc of a host slab failed");
            } else {
                std::string err;
                bool ok = true;
                if (!save && pread_all(f.fd, tmp, f.nbytes, f.offset) != 0) {
                    job->fail(TSNAP_EIO, "pread " + f.path + ": " + strerror(errno));
                    ok = false;
                }
                for (size_t i = 0; ok && i < f.members.size(); ++i) {
                    NormalizedCopy nc;
                    int rc = normalize_copy(f.members[i], uint64_t(uintptr_t(tmp)), false, &nc, &err);
                    if (rc != TSNAP_OK) {
                        job->fail(rc, "member of " + f.path + ": " + err);
                        ok = false;
                        break;
                    }
                    for (int k = 0; k < nc.n; ++k) host_copy_range(nc.m[k], 0, nc.m[k].bytes);
                }
                if (ok && save && pwrite_all(f.fd, tmp, f.nbytes, 0) != 0)
                    job->fail(TSNAP_EIO, "pwrite " + f.path + ": " + strerror(errno));
                free(tmp);
            }
        }
        finish_file_part(job, f, f.nbytes, save);
    });
}

// ---- save ------------------------------------------------------------------------------------------------
static void mark_device_done(tsnap_job* job) {
    std::lock_guard<std::mutex> g(job->mu);
    if (!job->device_done) {
        job->device_done = true;
        job->stats.device_done_ms = ms_since(job->t_submit);
        job->cv.notify_all();
    }
}

// parts_left = asynchronous parts + 1: the extra token belongs to the drain thread, which drops it when
// it no longer touches the job (run_job).  Waiters may destroy the job the moment the count hits zero.
static void account_parts(tsnap_job* job, int64_t async_parts) {
    job->parts_left.store(async_parts + 1);
    job->accounted = true;
}

// chunk I/O goes to the queue of the NUMA node the pinned slot lives on (node-affine workers, see io_worker_specs)
static void post_slot(tsnap_engine* eng, char* slot, std::function<void()> fn) {
    eng->io->post(std::move(fn), eng->ring.queue_of(slot));
}

// payload memcpys of chunk [lo, lo+n) of a direct file: one per dense run that intersects it
static bool direct_chunk_copies(tsnap_job* job, const FileSpec& f, char* slot, uint64_t lo, uint64_t n, bool to_host) {
    tsnap_engine* eng = job->eng;
    size_t i = size_t(std::upper_bound(f.segs.begin(), f.segs.end(), lo, [](uint64_t v, const FileSpec::Seg& s) { return v < s.off + s.bytes; }) - f.segs.begin());
    bool ok = true;
    for (; ok && i < f.segs.size() && f.segs[i].off < lo + n; ++i) {
        const FileSpec::Seg& sg = f.segs[i];
        const uint64_t a = std::max(lo, sg.off), b = std::min(lo + n, sg.off + sg.bytes);
        if (a >= b) continue;
        char* dev = reinterpret_cast<char*>(uintptr_t(sg.addr)) + (a - sg.off);
        ok = to_host ? cudaMemcpyAsync(slot + (a - lo), dev, b - a, cudaMemcpyDeviceToHost, eng->s_copy) == cudaSuccess
                     : cudaMemcpyAsync(dev, slot + (a - lo), b - a, cudaMemcpyHostToDevice, eng->s_copy) == cudaSuccess;
        job->n_memcpy.fetch_add(1, std::memory_order_relaxed);
    }
    return ok;
}

static int run_save_inner(tsnap_job* job) {
    NvtxRange nvtx_job("tsnap:save_job issue (plan, pack launch, D2H issue)");
    tsnap_engine* eng = job->eng;
    int rc = ensure_ring(eng);
    if (rc != TSNAP_OK) return rc;
    auto t0 = clk::now();
    const double tr0 = job->now_ms();
    rc = build_waves(job);
    if (rc != TSNAP_OK) return rc;
    for (Wave& w : job->waves) {
        rc = plan_wave(job, w);
        if (rc != TSNAP_OK) return rc;
    }
    job->stats.plan_ms = ms_since(t0);
    if (eng->trace) job->add_trace(TSNAP_TR_PLAN, 0, -1, tr0, job->now_ms(), 0);
    // The first waves' pack kernels go out before anything else: they run while the rest of the job is set up,
    // which keeps the async_take blocking window at plan + pack.  Nothing asynchronous references the job yet,
    // so a failure below only has to drain the stream before returning.
    const size_t nw = job->waves.size();
    const size_t ns = job->n_staged_waves;
    const bool has_direct = nw > ns;
    size_t launched = 0;
    if (job->ev_producer && ns > 0) CUDA_TRY(cudaStreamWaitEvent(eng->s_kernel, job->ev_producer, 0));
    for (; launched < std::min<size_t>(2, ns); ++launched) {
        rc = launch_wave(job, job->waves[launched]);
        if (rc != TSNAP_OK) {
            cudaStreamSynchronize(eng->s_kernel);
            return rc;
        }
    }
    auto bail = [&](int code) {
        std::string msg = last_err();
        cudaStreamSynchronize(eng->s_kernel);
        return set_err(code, msg);
    };
    // part count of every file before anything can complete (files are opened by the workers, see ensure_open)
    int64_t parts = 0;
    for (FileSpec& f : job->files) {
        const int64_t p = count_parts(eng, f, true);
        f.parts_left.store(p);
        parts += p;
    }
    for (Wave& w : job->waves)
        if (cudaEventCreateWithFlags(&w.ev_copied, cudaEventDisableTiming) != cudaSuccess) return bail(set_err(TSNAP_ECUDA, "event create failed"));
    if (nw > 0) {
        if (cudaEventCreate(&job->ev_copy_begin) != cudaSuccess || cudaEventCreate(&job->ev_copy_end) != cudaSuccess)
            return bail(set_err(TSNAP_ECUDA, "event create failed"));
    }
    // the "direct copies finished" notification is retired by the completion thread AFTER the wave's chunk entries, i.e.
    // possibly after the last write: it keeps the job alive with a part of its own
    if (has_direct) parts += 1;
    account_parts(job, parts);
    if (nw == 0) mark_device_done(job);
    if (parts == 0) return TSNAP_OK;

    // Sources are reusable (the async_take gate) once the last pack kernel has finished and, when files are drained
    // straight from the live tensors, once the last of those copies has finished.
    auto arm_kernel_done = [&](Wave& w, size_t wi, bool gate) {
        Wave* wp = &w;
        push_pending(eng, w.ev_done, [job, wp, wi, gate, eng](bool ok) {
            if (!ok) job->fail(TSNAP_ECUDA, "pack kernel failed");
            if (eng->trace) {
                collect_wave_timing(job, *wp);
                const double t1 = job->now_ms();
                job->add_trace(TSNAP_TR_KERNEL, int(wi), -1, t1 - wp->kernel_ms, t1, wp->bytes);
            }
            if (gate) mark_device_done(job);
        });
    };
    for (size_t wi = 0; wi < launched; ++wi) {
        const bool gate = !has_direct && wi + 1 == ns;
        if (gate || eng->trace) arm_kernel_done(job->waves[wi], wi, gate);
    }
    auto launch_next = [&]() -> int {
        Wave& w = job->waves[launched];
        if (launched >= 2) CUDA_TRY(cudaStreamWaitEvent(eng->s_kernel, job->waves[launched - 2].ev_copied, 0));
        int r = launch_wave(job, w);
        if (r != TSNAP_OK) return r;
        const bool gate = !has_direct && launched + 1 == ns;
        if (gate || eng->trace) arm_kernel_done(w, launched, gate);
        ++launched;
        return TSNAP_OK;
    };
    // host-only files go straight to the I/O workers
    for (size_t i = 0; i < job->files.size(); ++i) {
        FileSpec& f = job->files[i];
        if (f.host_only || f.nbytes == 0) post_host_file(job, int(i), true);
    }
    const uint64_t sb = eng->ring.slot_bytes();
    static const bool dbg_skip_d2h = getenv("TSNAP_B200_DEBUG_SKIP_D2H") != nullptr;      // experiments only
    static const bool dbg_skip_write = getenv("TSNAP_B200_DEBUG_SKIP_WRITE") != nullptr;  // experiments only
    for (size_t wi = 0; wi < nw; ++wi) {
        Wave& w = job->waves[wi];
        bool ok;
        if (w.direct) ok = !job->ev_producer || cudaStreamWaitEvent(eng->s_copy, job->ev_producer, 0) == cudaSuccess;
        else ok = cudaStreamWaitEvent(eng->s_copy, w.ev_done, 0) == cudaSuccess;
        if (wi == 0) cudaEventRecord(job->ev_copy_begin, eng->s_copy);
        // Buffered writes take the inode lock exclusively, so two chunks of one file never make progress at
        // the same time.  Treat every file as a sequential job and spread its chunks evenly over the whole
        // schedule of the wave: chunk k of a file with c chunks is due at (k + 1/2) / c.  Consecutive chunks of
        // a 512 MiB piece (16 chunks) then sit ~T/16 positions apart instead of back to back, and the
        // workers always find chunks of distinct files at the head of the queue.
        struct ChunkRef {
            int fi;
            uint64_t lo;
            double due;
        };
        std::vector<ChunkRef> order;
        for (int fi : w.files) {
            const uint64_t nb = job->files[fi].nbytes;
            const uint64_t c = (nb + sb - 1) / sb;
            for (uint64_t k = 0; k < c; ++k) order.push_back({fi, k * sb, (double(k) + 0.5) / double(c)});
        }
        std::stable_sort(order.begin(), order.end(), [](const ChunkRef& x, const ChunkRef& y) { return x.due < y.due; });
        for (const ChunkRef& cr : order) {
            FileSpec& f = job->files[cr.fi];
            const uint64_t lo = cr.lo;
            const uint64_t n = std::min(sb, f.nbytes - lo);
            auto tw = clk::now();
            const double tw_ms = eng->trace ? job->now_ms() : 0;
            const bool link_idle = job->copies_in_flight.load(std::memory_order_acquire) == 0;
            char* slot = job->take_slot();
            const double waited = ms_since(tw);
            job->slot_wait_us += int64_t(waited * 1000.0);
            if (link_idle) job->link_starved_us += int64_t(waited * 1000.0);
            job->copies_in_flight.fetch_add(1, std::memory_order_acq_rel);
            if (eng->trace && waited > 0.05) job->add_trace(TSNAP_TR_SLOT_WAIT, 0, cr.fi, tw_ms, job->now_ms(), 0);
            cudaEvent_t ev = eng->get_event();
            const double t_issue = eng->trace ? job->now_ms() : 0;
            if (ok && !job->failed() && !dbg_skip_d2h) {
                if (w.direct) {
                    ok = direct_chunk_copies(job, f, slot, lo, n, true);
                } else {
                    ok = cudaMemcpyAsync(slot, job->arena + w.region_off + f.arena_off + lo, n, cudaMemcpyDeviceToHost, eng->s_copy) == cudaSuccess;
                    job->n_memcpy.fetch_add(1, std::memory_order_relaxed);
                }
            }
            ok = ok && cudaEventRecord(ev, eng->s_copy) == cudaSuccess;
            if (!ok) job->fail(TSNAP_ECUDA, std::string("D2H copy: ") + cudaGetErrorString(cudaGetLastError()));
            eng->bytes_d2h += n;
            FileSpec* fp = &f;
            const int fidx = cr.fi;
            push_pending(eng, ev, [eng, job, fp, fidx, slot, lo, n, ev, t_issue](bool evok) {
                eng->put_event(ev);
                job->copies_in_flight.fetch_sub(1, std::memory_order_acq_rel);
                if (!evok) job->fail(TSNAP_ECUDA, "D2H copy failed");
                if (eng->trace) {
                    // the copy engine runs the chunks of s_copy back to back: busy since the later of "issued" and
                    // "previous chunk done"
                    const double t1 = job->now_ms();
                    job->add_trace(TSNAP_TR_D2H, 0, fidx, std::max(t_issue, job->last_copy_done_ms), t1, n);
                    job->last_copy_done_ms = t1;
                }
                auto tq = clk::now();
                post_slot(eng, slot, [eng, job, fp, fidx, slot, lo, n, tq] {
                    job->io_queue_us += int64_t(ms_since(tq) * 1000.0);
                    NvtxRange nvtx_w("tsnap:pwrite chunk");
                    if (!dbg_skip_write && !job->failed() && ensure_open(job, *fp, true)) {
                        auto tb = clk::now();
                        const double t0w = eng->trace ? job->now_ms() : 0;
                        {
                            TokenGuard tok;
                            if (write_chunk(*fp, slot, n, lo) != 0) job->fail(TSNAP_EIO, "pwrite " + fp->path + ": " + strerror(errno));
                        }
                        job->io_busy_us += int64_t(ms_since(tb) * 1000.0);
                        if (eng->trace) job->add_trace(TSNAP_TR_PWRITE, g_lane, fidx, t0w, job->now_ms(), n);
                    }
                    job->give_slot(slot);
                    finish_file_part(job, *fp, n, true);
                });
            });
        }
        if (wi + 1 == nw) cudaEventRecord(job->ev_copy_end, eng->s_copy);
        if (cudaEventRecord(w.ev_copied, eng->s_copy) != cudaSuccess) job->fail(TSNAP_ECUDA, "event record failed");
        if (w.direct)  // (this entry is queued behind the wave's chunk entries: it holds a part of its own, see below)
            push_pending(eng, w.ev_copied, [job](bool evok) {
                if (!evok) job->fail(TSNAP_ECUDA, "D2H copy failed");
                mark_device_done(job);
                job->part_done();
            });
        if (launched < ns) {
            rc = launch_next();
            if (rc != TSNAP_OK) {
                job->fail(rc, last_err());
                mark_device_done(job);
                // remaining waves are never issued
                int64_t remaining = 0;
                for (size_t wj = wi + 1; wj < nw; ++wj)
                    for (int fj : job->waves[wj].files) remaining += job->files[fj].parts_left.load();
                if (has_direct) remaining += 1;  // the direct wave's completion entry is never queued either
                for (int64_t i = 0; i < remaining; ++i) job->part_done();
                return TSNAP_OK;
            }
        }
    }
    return TSNAP_OK;
}

// ---- load ------------------------------------------------------------------------------------------------
struct LoadShared {
    std::mutex mu;
    std::condition_variable cv;
    std::vector<char> launched;  // per wave: scatter kernels enqueued
};

static int run_load_inner(tsnap_job* job) {
    NvtxRange nvtx_job("tsnap:load_job issue (plan, reads)");
    tsnap_engine* eng = job->eng;
    int rc = ensure_ring(eng);
    if (rc != TSNAP_OK) return rc;
    auto t0 = clk::now();
    const double tr0 = job->now_ms();
    rc = build_waves(job);
    if (rc != TSNAP_OK) return rc;
    for (Wave& w : job->waves) {
        rc = plan_wave(job, w);
        if (rc != TSNAP_OK) return rc;
    }
    job->stats.plan_ms = ms_since(t0);
    if (eng->trace) job->add_trace(TSNAP_TR_PLAN, 0, -1, tr0, job->now_ms(), 0);
    const uint64_t sb = eng->ring.slot_bytes();
    int64_t parts = 0;
    for (FileSpec& f : job->files) {
        if (f.nbytes == 0) continue;
        const int64_t p = count_parts(eng, f, false);
        f.parts_left.store(p);
        parts += p;
    }
    parts += int64_t(job->waves.size());  // one part per wave for its scatter kernels
    account_parts(job, parts);
    if (parts == 0) {
        mark_device_done(job);
        return TSNAP_OK;
    }
    for (Wave& w : job->waves) {
        int64_t c = 0;
        for (int fi : w.files) c += int64_t((job->files[fi].nbytes + sb - 1) / sb);
        w.chunks_to_upload.store(c);
    }
    for (size_t i = 0; i < job->files.size(); ++i)
        if (job->files[i].host_only && job->files[i].nbytes) post_host_file(job, int(i), false);

    // Everything that writes destination tensors is ordered after the work already queued on the caller's stream:
    // the scatter kernels (s_kernel) and, for files uploaded straight into the live tensors, the copies (s_copy).
    bool any_direct = false;
    for (Wave& w : job->waves) any_direct = any_direct || w.direct;
    // A lent arena comes from the caller's stream-ordered allocator: the block may still be in use by kernels queued
    // on that stream (its previous owner was freed "in stream order"), so uploads into it wait as well.
    if (job->ev_consumer) {
        if (job->n_staged_waves) cudaStreamWaitEvent(eng->s_kernel, job->ev_consumer, 0);
        if (any_direct || (job->arena_set && job->n_staged_waves)) cudaStreamWaitEvent(eng->s_copy, job->ev_consumer, 0);
    }

    auto shared = std::make_shared<LoadShared>();
    shared->launched.assign(job->waves.size(), 0);
    const size_t nw = job->waves.size();
    for (size_t wi = 0; wi < nw; ++wi) {
        Wave* w = &job->waves[wi];
        if (!w->direct && wi >= 2) {
            // the region is reused: wait until the scatter of wave wi-2 has been enqueued, then order
            // this wave's uploads after it on the device
            std::unique_lock<std::mutex> g(shared->mu);
            shared->cv.wait(g, [&] { return shared->launched[wi - 2] != 0; });
            g.unlock();
            if (job->waves[wi - 2].ev_done)
                cudaStreamWaitEvent(eng->s_copy, job->waves[wi - 2].ev_done, 0);
        }
        const bool last_wave = (wi + 1 == nw);
        for (int fi : w->files) {
            FileSpec* f = &job->files[fi];
            char* base = w->direct ? nullptr : job->arena + w->region_off + f->arena_off;
            for (uint64_t lo = 0; lo < f->nbytes; lo += sb) {
                const uint64_t n = std::min(sb, f->nbytes - lo);
                char* slot = job->take_slot();
                post_slot(eng, slot, [eng, job, w, wi, f, fi, base, slot, lo, n, shared, last_wave] {
                    NvtxRange nvtx_r("tsnap:pread chunk + H2D enqueue");
                    cudaSetDevice(eng->device);
                    bool ok = !job->failed();
                    uint64_t skip = 0;
                    const double t0r = eng->trace ? job->now_ms() : 0;
                    if (ok && f->mem_src) {
                        memcpy(slot, f->mem_src + lo, n);
                    } else if (ok) {
                        auto tb = clk::now();
                        if (!ensure_open(job, *f, false)) {
                            ok = false;
                        } else {
                            TokenGuard tok;
                            if (read_chunk(*f, slot, n, f->offset + lo, &skip) != 0) {
                                job->fail(TSNAP_EIO, "pread " + f->path + ": " + strerror(errno));
                                ok = false;
                            }
                        }
                        job->io_busy_us += int64_t(ms_since(tb) * 1000.0);
                    }
                    const double t_issue = eng->trace ? job->now_ms() : 0;
                    if (eng->trace) job->add_trace(TSNAP_TR_PREAD, g_lane, fi, t0r, t_issue, n);
                    cudaEvent_t ev = eng->get_event();
                    if (ok) {
                        bool cok;
                        if (w->direct) {
                            cok = direct_chunk_copies(job, *f, slot + skip, lo, n, false);
                        } else {
                            cok = cudaMemcpyAsync(base + lo, slot + skip, n, cudaMemcpyHostToDevice, eng->s_copy) == cudaSuccess;
                            job->n_memcpy.fetch_add(1, std::memory_order_relaxed);
                        }
                        if (!cok) {
                            job->fail(TSNAP_ECUDA, "H2D copy failed to enqueue");
                            ok = false;
                        }
                    }
                    cudaEventRecord(ev, eng->s_copy);
                    eng->bytes_h2d += n;
                    push_pending(eng, ev, [eng, job, f, fi, slot, n, ev, t_issue](bool evok) {
                        eng->put_event(ev);
                        if (!evok) job->fail(TSNAP_ECUDA, "H2D copy failed");
                        if (eng->trace) {
                            const double t1 = job->now_ms();
                            job->add_trace(TSNAP_TR_H2D, 0, fi, std::max(t_issue, job->last_copy_done_ms), t1, n);
                            job->last_copy_done_ms = t1;
                        }
                        job->give_slot(slot);
                        finish_file_part(job, *f, n, false);
                    });
                    // the worker that enqueues the last upload of the wave launches its scatter kernels
                    if (w->chunks_to_upload.fetch_sub(1, std::memory_order_acq_rel) == 1) {
                        int r = TSNAP_OK;
                        if (!job->failed()) {
                            cudaEventCreateWithFlags(&w->ev_copied, cudaEventDisableTiming);
                            cudaEventRecord(w->ev_copied, eng->s_copy);
                            if (w->direct) {
                                // no scatter: the uploads were the restore
                                cudaEventCreateWithFlags(&w->ev_done, cudaEventDisableTiming);
                                cudaEventRecord(w->ev_done, eng->s_copy);
                            } else {
                                cudaStreamWaitEvent(eng->s_kernel, w->ev_copied, 0);
                                r = launch_wave(job, *w);
                                if (r != TSNAP_OK) job->fail(r, last_err());
                            }
                        }
                        {
                            std::lock_guard<std::mutex> g(shared->mu);
                            shared->launched[wi] = 1;
                        }
                        shared->cv.notify_all();
                        if (r == TSNAP_OK && w->ev_done && !job->failed()) {
                            push_pending(eng, w->ev_done, [eng, job, w, wi, last_wave](bool evok) {
                                if (!evok) job->fail(TSNAP_ECUDA, "scatter kernel failed");
                                collect_wave_timing(job, *w);
                                if (eng->trace && !w->direct) {
                                    const double t1 = job->now_ms();
                                    job->add_trace(TSNAP_TR_KERNEL, int(wi), -1, t1 - w->kernel_ms, t1, w->bytes);
                                }
                                if (last_wave) mark_device_done(job);
                                job->part_done();
                            });
                        } else {
                            if (last_wave) mark_device_done(job);
                            job->part_done();
                        }
                    }
                });
            }
        }
    }
    if (nw == 0) mark_device_done(job);
    return TSNAP_OK;
}

// ---- stage (whole-buffer pinned sink) ---------------------------------------------------------------------
static int run_stage_inner(tsnap_job* job) {
    tsnap_engine* eng = job->eng;
    FileSpec& f = job->files[0];
    auto t0 = clk::now();
    // host members are copied right here; device members go through the pack kernels
    std::vector<tsnap_copy_desc> dev;
    std::string err;
    for (const tsnap_copy_desc& d : f.members) {
        if (d.src_space == TSNAP_SPACE_HOST) {
            NormalizedCopy nc;
            int rc = normalize_copy(d, uint64_t(uintptr_t(job->stage_buf)), false, &nc, &err);
            if (rc != TSNAP_OK) return set_err(rc, err);
            for (int k = 0; k < nc.n; ++k) host_copy_range(nc.m[k], 0, nc.m[k].bytes);
        } else {
            dev.push_back(d);
        }
    }
    if (dev.empty() || f.nbytes == 0) {
        account_parts(job, 0);
        mark_device_done(job);
        return TSNAP_OK;
    }
    if (!eng->has_device) return set_err(TSNAP_ECUDA, "device members on a host-only engine");
    // device members may be interleaved with host members; pack into the arena image of the whole
    // buffer and copy back only the spans that device members cover (here: the whole buffer when no
    // host member exists, else per-member spans)
    const bool mixed = dev.size() != f.members.size();
    f.members = dev;
    int rc = build_waves(job);
    if (rc != TSNAP_OK) return rc;
    Wave& w = job->waves[0];
    rc = plan_wave(job, w);
    if (rc != TSNAP_OK) return rc;
    job->stats.plan_ms = ms_since(t0);
    CUDA_TRY(cudaEventCreate(&job->ev_copy_begin));
    CUDA_TRY(cudaEventCreate(&job->ev_copy_end));
    char* out = static_cast<char*>(job->stage_buf);
    Wave* wp = &w;
    if (w.direct) {
        // no HBM staging available: dense members go straight from the live tensors into the pinned buffer
        if (job->ev_producer) CUDA_TRY(cudaStreamWaitEvent(eng->s_copy, job->ev_producer, 0));
        CUDA_TRY(cudaEventRecord(job->ev_copy_begin, eng->s_copy));
        for (const FileSpec::Seg& sg : f.segs) {
            CUDA_TRY(cudaMemcpyAsync(out + sg.off, reinterpret_cast<const void*>(uintptr_t(sg.addr)), sg.bytes, cudaMemcpyDeviceToHost, eng->s_copy));
            eng->bytes_d2h += sg.bytes;
            job->n_memcpy.fetch_add(1, std::memory_order_relaxed);
        }
    } else {
        if (job->ev_producer) CUDA_TRY(cudaStreamWaitEvent(eng->s_kernel, job->ev_producer, 0));
        rc = launch_wave(job, w);
        if (rc != TSNAP_OK) return rc;
        CUDA_TRY(cudaStreamWaitEvent(eng->s_copy, w.ev_done, 0));
        CUDA_TRY(cudaEventRecord(job->ev_copy_begin, eng->s_copy));
        const char* base = job->arena + w.region_off + f.arena_off;
        if (!mixed) {
            CUDA_TRY(cudaMemcpyAsync(out, base, f.nbytes, cudaMemcpyDeviceToHost, eng->s_copy));
            eng->bytes_d2h += f.nbytes;
            job->n_memcpy.fetch_add(1, std::memory_order_relaxed);
        } else {
            for (const tsnap_copy_desc& d : dev) {
                uint64_t numel = 1;
                for (int i = 0; i < d.ndim; ++i) numel *= uint64_t(d.sizes[i]);
                const uint64_t nb = numel * dtype_size(d.dst_dtype);
                if (nb == 0) continue;
                CUDA_TRY(cudaMemcpyAsync(out + d.dst_addr, base + d.dst_addr, nb, cudaMemcpyDeviceToHost, eng->s_copy));
                eng->bytes_d2h += nb;
                job->n_memcpy.fetch_add(1, std::memory_order_relaxed);
            }
        }
    }
    CUDA_TRY(cudaEventRecord(job->ev_copy_end, eng->s_copy));
    cudaEvent_t ev = eng->get_event();
    CUDA_TRY(cudaEventRecord(ev, eng->s_copy));
    account_parts(job, 1);
    if (!w.direct)
        push_pending(eng, w.ev_done, [job](bool ok) {
            if (!ok) job->fail(TSNAP_ECUDA, "pack kernel failed");
            mark_device_done(job);
        });
    push_pending(eng, ev, [eng, job, ev, wp](bool ok) {
        eng->put_event(ev);
        if (!ok) job->fail(TSNAP_ECUDA, "D2H copy failed");
        collect_wave_timing(job, *wp);
        mark_device_done(job);
        job->part_done();
    });
    return TSNAP_OK;
}

static void run_job(tsnap_job* job) {
    tsnap_engine* eng = job->eng;
    if (eng->has_device) cudaSetDevice(eng->device);
    // Jobs are issued back to back, but the staging arena (and its two wave regions) belongs to one device job
    // at a time: a job that touches the GPU waits here until its predecessor has completely drained.
    bool device_job = job->kind == kStage;
    for (const FileSpec& f : job->files) device_job = device_job || (!f.host_only && f.nbytes > 0);
    if (device_job && eng->has_device && !job->arena_set && !eng->no_arena) {
        std::unique_lock<std::mutex> ga(eng->arena_mu);
        eng->arena_cv.wait(ga, [eng] { return !eng->arena_in_use; });
        eng->arena_in_use = true;
        job->holds_arena = true;
    }
    int rc;
    if (job->kind == kSave) rc = run_save_inner(job);
    else if (job->kind == kLoad) rc = run_load_inner(job);
    else rc = run_stage_inner(job);
    if (rc != TSNAP_OK) {
        job->fail(rc, last_err());
        mark_device_done(job);
        if (!job->accounted) {
            // failed before any asynchronous part was handed out
            account_parts(job, 0);
        }
    }
    job->part_done();  // the drain thread's token: `job` may be destroyed by a waiter from here on
}

// Frees the staging arena.  Only the drain thread calls this, between jobs; the arena may still be the source
// of in-flight D2H copies of the previous job, so both streams are drained first.
static void free_arena(tsnap_engine* eng) {
    if (!eng->arena) return;
    // load jobs keep enqueueing uploads/scatters from the I/O workers after the drain thread moved on
    while (eng->active_jobs.load(std::memory_order_acquire) > 0) std::this_thread::sleep_for(std::chrono::milliseconds(1));
    cudaSetDevice(eng->device);
    cudaStreamSynchronize(eng->s_kernel);
    cudaStreamSynchronize(eng->s_copy);
    cudaFree(eng->arena);
    eng->arena = nullptr;
    eng->arena_bytes = 0;
}

static void drain_main(tsnap_engine* eng) {
    bind_current_thread(eng->numa_cpus);
    for (;;) {
        tsnap_job* job = nullptr;
        {
            std::unique_lock<std::mutex> g(eng->q_mu);
            eng->busy = false;
            eng->q_cv.notify_all();
            // An engine-owned arena is given back once the engine has been idle for a moment (it is invisible to the
            // host runtime's allocator, so holding it across training steps can OOM them); TSNAP_B200_KEEP_ARENA=1 keeps
            // it for back-to-back snapshots.
            while (!(eng->stopping || !eng->job_q.empty() || eng->trim_arena)) {
                if (eng->arena && !eng->keep_arena && eng->active_jobs.load(std::memory_order_acquire) == 0) {
                    if (eng->q_cv.wait_for(g, std::chrono::milliseconds(50)) == std::cv_status::timeout && eng->job_q.empty() &&
                        !eng->stopping && eng->active_jobs.load(std::memory_order_acquire) == 0)
                        eng->trim_arena = true;
                } else if (eng->arena && !eng->keep_arena) {
                    eng->q_cv.wait_for(g, std::chrono::milliseconds(5));
                } else {
                    eng->q_cv.wait(g);
                }
            }
            if (eng->trim_arena && eng->job_q.empty()) {
                g.unlock();
                free_arena(eng);
                g.lock();
                eng->trim_arena = false;
                eng->q_cv.notify_all();
                continue;
            }
            if (eng->job_q.empty()) return;
            job = eng->job_q.front();
            eng->job_q.pop_front();
            eng->busy = true;
        }
        run_job(job);
    }
}

// ==========================================================================================================
// C ABI
// ==========================================================================================================
extern "C" {

int tsnap_abi_version(void) { return TSNAP_ABI_VERSION; }
const char* tsnap_last_error(void) { return last_err(); }
size_t tsnap_dtype_size(int dtype) { return dtype_size(dtype); }

int tsnap_engine_create(const tsnap_engine_config* cfg, tsnap_engine** out) {
    if (!cfg || !out) return set_err(TSNAP_EINVAL, "null argument");
    tsnap_engine* eng = new tsnap_engine();
    eng->cfg = *cfg;
    eng->device = cfg->device;
    eng->allow_bulk = !(cfg->flags & TSNAP_ENGINE_NO_BULK);
    eng->trace = (cfg->flags & TSNAP_ENGINE_TRACE) != 0;
    eng->odirect = (cfg->flags & TSNAP_ENGINE_ODIRECT) != 0;
    eng->no_arena = (cfg->flags & TSNAP_ENGINE_NO_ARENA) != 0;
    {
        // one descriptor per in-flight chunk at most, but leave room for the host process: lift the soft limit
        struct rlimit rl;
        if (getrlimit(RLIMIT_NOFILE, &rl) == 0 && rl.rlim_cur < rl.rlim_max) {
            rl.rlim_cur = rl.rlim_max == RLIM_INFINITY ? std::max<rlim_t>(rl.rlim_cur, 65536) : rl.rlim_max;
            setrlimit(RLIMIT_NOFILE, &rl);
        }
    }
    if (cfg->device >= 0) {
        cudaError_t e = cudaSetDevice(cfg->device);
        cudaDeviceProp prop;
        if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, cfg->device);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&eng->s_kernel, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&eng->s_copy, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = init_kernels();
        if (e == cudaSuccess) e = init_transpose_tma();
        if (e != cudaSuccess) {
            std::string msg = std::string("CUDA device ") + std::to_string(cfg->device) +
                              " is not usable: " + cudaGetErrorString(e);
            delete eng;
            return set_err(TSNAP_ECUDA, msg);
        }
        if (prop.major < 10) {
            delete eng;
            return set_err(TSNAP_ECUDA, "tsnap_b200 kernels are built for sm_100a only");
        }
        eng->sm_count = prop.multiProcessorCount;
        eng->has_device = true;
        eng->numa_cpus = gpu_numa_cpus(cfg->device);
        const char* keep = getenv("TSNAP_B200_KEEP_ARENA");
        eng->keep_arena = keep && keep[0] == '1';
        eng->completion_thread = std::thread(completion_main, eng);
    }
    {
        static std::once_flag once;
        std::call_once(once, [] {
            const char* t = getenv("TSNAP_B200_HOST_IO_TOKENS");
            const char* lw = getenv("LOCAL_WORLD_SIZE");
            const int local_world = lw ? atoi(lw) : 1;
            g_tokens.init(t ? atoi(t) : (local_world > 1 ? 16 : 0));
        });
    }
    {
        // TSNAP_B200_RING_NUMA: interleave (default: slot i on node i % nodes) | gpu (all slots on the GPU's node) | none.
        // With interleave + TSNAP_B200_IO_PIN=node (default) every page-cache copy reads a slot of the worker's own node
        // and both sockets' memory channels and LRU locks share the load (profiles/r02_sink_sweep.md).
        const char* rn = getenv("TSNAP_B200_RING_NUMA");
        const std::string ring_mode = rn ? rn : "interleave";
        if (ring_mode == "interleave") {
            const std::vector<NumaNode> nodes = numa_nodes();
            if (nodes.size() >= 2)
                for (const NumaNode& nd : nodes) eng->ring_nodes.push_back(nd.id);
        } else if (ring_mode == "gpu" && cfg->device >= 0) {
            char bus[32] = {0};
            if (cudaDeviceGetPCIBusId(bus, sizeof(bus), cfg->device) == cudaSuccess) {
                std::string id(bus);
                for (char& c : id) c = char(tolower(c));
                const std::string node = read_small_file("/sys/bus/pci/devices/" + id + "/numa_node");
                if (!node.empty() && atoi(node.c_str()) >= 0) eng->ring_nodes.push_back(atoi(node.c_str()));
            }
        }
        const int nio = cfg->io_threads > 0 ? cfg->io_threads : 16;
        int nq = 1;
        std::vector<WorkerSpec> specs = io_worker_specs(nio, eng->numa_cpus.empty() ? std::vector<int>() : eng->numa_cpus, eng->ring_nodes, &nq);
        if (!eng->numa_cpus.empty())
            for (WorkerSpec& w : specs)
                if (w.cpus.empty()) w.cpus = eng->numa_cpus;  // TSNAP_B200_NUMA=1
        eng->io = new WorkerPool(specs, nq);
    }
    eng->drain_thread = std::thread(drain_main, eng);
    *out = eng;
    return TSNAP_OK;
}

int tsnap_engine_trim(tsnap_engine* eng) {
    if (!eng) return set_err(TSNAP_EINVAL, "null engine");
    if (eng->has_device) {
        // the arena belongs to the drain thread: ask it to free it once it is idle, and wait for that
        std::unique_lock<std::mutex> g(eng->q_mu);
        eng->trim_arena = true;
        eng->q_cv.notify_all();
        eng->q_cv.wait(g, [eng] { return !eng->trim_arena || eng->stopping; });
    }
    std::lock_guard<std::mutex> g(eng->pin_mu);
    for (auto& kv : eng->pin_cache) {
        if (eng->has_device) cudaFreeHost(kv.second);
        else free(kv.second);
    }
    eng->pin_cache.clear();
    return TSNAP_OK;
}

int tsnap_engine_destroy(tsnap_engine* eng) {
    if (!eng) return TSNAP_OK;
    {
        std::lock_guard<std::mutex> g(eng->q_mu);
        eng->stopping = true;
    }
    eng->q_cv.notify_all();
    if (eng->drain_thread.joinable()) eng->drain_thread.join();
    delete eng->io;  // drains queued I/O
    eng->io = nullptr;
    {
        std::lock_guard<std::mutex> g(eng->c_mu);
        eng->stopping = true;
    }
    eng->c_cv.notify_all();
    if (eng->completion_thread.joinable()) eng->completion_thread.join();
    tsnap_engine_trim(eng);
    if (eng->has_device) {
        cudaSetDevice(eng->device);
        cudaStreamSynchronize(eng->s_kernel);
        cudaStreamSynchronize(eng->s_copy);
        if (eng->arena) cudaFree(eng->arena);
        for (auto& kv : eng->tbl_free) cudaFree(kv.second);
        for (cudaEvent_t e : eng->ev_free) cudaEventDestroy(e);
        cudaStreamDestroy(eng->s_kernel);
        cudaStreamDestroy(eng->s_copy);
    }
    eng->ring.destroy();
    delete eng;
    return TSNAP_OK;
}

int tsnap_engine_get_stats(tsnap_engine* eng, tsnap_engine_stats* out) {
    if (!eng || !out) return set_err(TSNAP_EINVAL, "null argument");
    uint64_t pinned = eng->has_device ? eng->ring.total_bytes() : 0;
    {
        std::lock_guard<std::mutex> g(eng->pin_mu);
        for (auto& kv : eng->pin_cache) pinned += kv.first;
    }
    out->pinned_bytes = pinned;
    out->hbm_arena_bytes = eng->arena_bytes;
    out->kernels_launched = eng->kernels_launched.load();
    out->bytes_d2h = eng->bytes_d2h.load();
    out->bytes_h2d = eng->bytes_h2d.load();
    out->bytes_written = eng->bytes_written.load();
    out->bytes_read = eng->bytes_read.load();
    out->sm_count = eng->sm_count;
    out->device = eng->device;
    return TSNAP_OK;
}

static int job_create(tsnap_engine* eng, int kind, tsnap_job** out) {
    if (!eng || !out) return set_err(TSNAP_EINVAL, "null argument");
    tsnap_job* j = new tsnap_job();
    j->eng = eng;
    j->kind = kind;
    *out = j;
    return TSNAP_OK;
}
int tsnap_save_job_create(tsnap_engine* eng, tsnap_job** out) { return job_create(eng, kSave, out); }
int tsnap_load_job_create(tsnap_engine* eng, tsnap_job** out) { return job_create(eng, kLoad, out); }

static int add_file(tsnap_job* job, const char* path, uint64_t offset, uint64_t nbytes, int32_t* idx) {
    if (!job || !path || !idx) return set_err(TSNAP_EINVAL, "null argument");
    if (job->submitted) return set_err(TSNAP_ESTATE, "job already submitted");
    job->files.emplace_back();
    FileSpec& f = job->files.back();
    f.path = path;
    f.offset = offset;
    f.nbytes = nbytes;
    f.dense = true;
    *idx = int32_t(job->files.size()) - 1;
    return TSNAP_OK;
}
int tsnap_save_job_add_file(tsnap_job* job, const char* path, uint64_t nbytes, int32_t* file_index) {
    if (job && job->kind != kSave) return set_err(TSNAP_ESTATE, "not a save job");
    return add_file(job, path, 0, nbytes, file_index);
}
int tsnap_load_job_add_file(tsnap_job* job, const char* path, uint64_t offset, uint64_t nbytes, int32_t* file_index) {
    if (job && job->kind != kLoad) return set_err(TSNAP_ESTATE, "not a load job");
    return add_file(job, path, offset, nbytes, file_index);
}

static int add_member(tsnap_job* job, int32_t fi, const tsnap_copy_desc* d, bool save) {
    if (!job || !d) return set_err(TSNAP_EINVAL, "null argument");
    if (job->submitted) return set_err(TSNAP_ESTATE, "job already submitted");
    if (fi < 0 || size_t(fi) >= job->files.size()) return set_err(TSNAP_EINVAL, "bad file index");
    if (save ? d->dst_space != TSNAP_SPACE_WIRE : d->src_space != TSNAP_SPACE_WIRE)
        return set_err(TSNAP_EINVAL, save ? "save members must have a WIRE destination"
                                          : "load members must have a WIRE source");
    // validate now so that errors surface at the call site, like the reference's prepare_* would
    NormalizedCopy nc;
    std::string err;
    int rc = normalize_copy(*d, 0, false, &nc, &err);
    if (rc != TSNAP_OK) return set_err(rc, err);
    FileSpec& f = job->files[size_t(fi)];
    uint64_t numel = 1;
    for (int i = 0; i < d->ndim; ++i) numel *= uint64_t(d->sizes[i]);
    if (save) {
        const bool quant = d->dst_dtype == TSNAP_QINT8 || d->dst_dtype == TSNAP_QUINT8;
        const uint64_t end = d->dst_addr + numel * dtype_size(d->dst_dtype) + (quant && numel ? 16 : 0);
        if (end > f.nbytes) return set_err(TSNAP_EINVAL, "member exceeds the file's wire image");
    } else if (numel) {
        // furthest byte touched on the wire side
        uint64_t last = d->src_addr;
        for (int i = 0; i < d->ndim; ++i)
            last += uint64_t(d->sizes[i] - 1) * uint64_t(d->src_strides[i]) * dtype_size(d->src_dtype);
        if (last + dtype_size(d->src_dtype) > f.nbytes) return set_err(TSNAP_EINVAL, "member reads past the byte range");
    }
    // dense, cast-free device members can be drained / uploaded without staging: remember their runs
    const int tensor_space = save ? d->src_space : d->dst_space;
    if (numel && tensor_space == TSNAP_SPACE_DEVICE) {
        if (nc.n == 1 && nc.m[0].mode == kModeContig)
            f.segs.push_back(FileSpec::Seg{save ? nc.m[0].dst : nc.m[0].src, save ? nc.m[0].src : nc.m[0].dst, nc.m[0].bytes});
        else
            f.dense = false;
    }
    f.members.push_back(*d);
    job->stats.n_members++;
    return TSNAP_OK;
}
int tsnap_save_job_add_member(tsnap_job* job, int32_t file_index, const tsnap_copy_desc* desc) {
    return add_member(job, file_index, desc, true);
}
int tsnap_load_job_add_member(tsnap_job* job, int32_t file_index, const tsnap_copy_desc* desc) {
    return add_member(job, file_index, desc, false);
}

static int submit(tsnap_job* job, void* stream, bool is_consumer) {
    if (!job) return set_err(TSNAP_EINVAL, "null job");
    if (job->submitted) return set_err(TSNAP_ESTATE, "job already submitted");
    tsnap_engine* eng = job->eng;
    job->stats.n_files = job->files.size();
    bool any_device = false;
    for (FileSpec& f : job->files) {
        job->stats.payload_bytes += f.nbytes;
        bool host = true;
        for (const tsnap_copy_desc& d : f.members) {
            const int sp = job->kind == kLoad ? d.dst_space : d.src_space;
            if (sp != TSNAP_SPACE_HOST) host = false;
        }
        if (job->kind == kStage) {
            f.host_only = false;
            any_device = any_device || !host;
            continue;
        }
        if (!host) {
            for (const tsnap_copy_desc& d : f.members) {
                const int sp = job->kind == kLoad ? d.dst_space : d.src_space;
                if (sp == TSNAP_SPACE_HOST)
                    return set_err(TSNAP_EUNSUP, "a file mixes HOST and DEVICE members: " + f.path +
                                                     " (the batcher keeps CPU and GPU slabs apart, T:batcher.py:300-303)");
            }
        }
        f.host_only = host;
        any_device = any_device || !host;
    }
    if (any_device && !eng->has_device) return set_err(TSNAP_ECUDA, "device members on a host-only engine");
    if (any_device && !is_consumer) {
        cudaSetDevice(eng->device);
        CUDA_TRY(cudaEventCreateWithFlags(&job->ev_producer, cudaEventDisableTiming));
        CUDA_TRY(cudaEventRecord(job->ev_producer, static_cast<cudaStream_t>(stream)));
    }
    if (is_consumer) {
        job->consumer_stream = stream;
        if (any_device) {
            // restored bytes must not be overtaken by work already queued on the caller's stream
            cudaSetDevice(eng->device);
            CUDA_TRY(cudaEventCreateWithFlags(&job->ev_consumer, cudaEventDisableTiming));
            CUDA_TRY(cudaEventRecord(job->ev_consumer, static_cast<cudaStream_t>(stream)));
        }
    }
    job->submitted = true;
    job->t_submit = clk::now();
    eng->active_jobs.fetch_add(1, std::memory_order_acq_rel);
    {
        std::lock_guard<std::mutex> g(eng->q_mu);
        eng->job_q.push_back(job);
    }
    eng->q_cv.notify_one();
    return TSNAP_OK;
}
int tsnap_save_job_submit(tsnap_job* job, void* producer_stream) {
    if (job && job->kind != kSave) return set_err(TSNAP_ESTATE, "not a save job");
    return submit(job, producer_stream, false);
}
int tsnap_load_job_submit(tsnap_job* job, void* consumer_stream) {
    if (job && job->kind != kLoad) return set_err(TSNAP_ESTATE, "not a load job");
    return submit(job, consumer_stream, true);
}

int tsnap_job_wait_device(tsnap_job* job) {
    if (!job) return set_err(TSNAP_EINVAL, "null job");
    if (!job->submitted) return set_err(TSNAP_ESTATE, "job not submitted");
    std::unique_lock<std::mutex> g(job->mu);
    job->cv.wait(g, [job] { return job->device_done || job->done; });
    if (job->err_code) return set_err(job->err_code, job->err_msg);
    return TSNAP_OK;
}
int tsnap_job_wait(tsnap_job* job) {
    if (!job) return set_err(TSNAP_EINVAL, "null job");
    if (!job->submitted) return set_err(TSNAP_ESTATE, "job not submitted");
    std::unique_lock<std::mutex> g(job->mu);
    job->cv.wait(g, [job] { return job->done; });
    if (job->err_code) return set_err(job->err_code, job->err_msg);
    return TSNAP_OK;
}
int tsnap_job_done(tsnap_job* job) {
    if (!job) return 1;
    std::lock_guard<std::mutex> g(job->mu);
    return job->done ? 1 : 0;
}
int tsnap_job_get_stats(tsnap_job* job, tsnap_job_stats* out) {
    if (!job || !out) return set_err(TSNAP_EINVAL, "null argument");
    bool collect = false, copy_collect = false;
    {
        std::lock_guard<std::mutex> g(job->mu);
        if (job->done && !job->timing_collected) {
            job->timing_collected = true;
            collect = job->kind == kSave;
            copy_collect = true;
        }
    }
    if (job->eng->has_device && (collect || copy_collect)) cudaSetDevice(job->eng->device);
    if (collect)
        for (Wave& w : job->waves) collect_wave_timing(job, w);
    if (copy_collect && job->ev_copy_begin && job->ev_copy_end) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, job->ev_copy_begin, job->ev_copy_end) == cudaSuccess) {
            std::lock_guard<std::mutex> g(job->mu);
            job->stats.copy_ms = ms;
        }
    }
    std::lock_guard<std::mutex> g(job->mu);
    job->stats.slot_wait_ms = job->slot_wait_us.load() / 1000.0;
    job->stats.io_busy_ms = job->io_busy_us.load() / 1000.0;
    job->stats.io_queue_ms = job->io_queue_us.load() / 1000.0;
    job->stats.n_memcpy = uint64_t(job->n_memcpy.load());
    job->stats.link_starved_ms = job->link_starved_us.load() / 1000.0;
    {
        std::lock_guard<std::mutex> gs(job->slot_mu);
        job->stats.max_slots_in_flight = uint64_t(job->slots_peak);
    }
    *out = job->stats;
    return TSNAP_OK;
}
int tsnap_job_destroy(tsnap_job* job) {
    if (!job) return TSNAP_OK;
    if (job->submitted) {
        std::unique_lock<std::mutex> g(job->mu);
        job->cv.wait(g, [job] { return job->done; });
    }
    if (job->eng->has_device) cudaSetDevice(job->eng->device);
    for (Wave& w : job->waves) {
        if (w.d_tables) job->eng->put_table(w.d_tables, w.table_cap);  // the job is done: its kernels have finished
        if (w.ev_k0) cudaEventDestroy(w.ev_k0);
        if (w.ev_k1) cudaEventDestroy(w.ev_k1);
        if (w.ev_kr) cudaEventDestroy(w.ev_kr);
        if (w.ev_k2) cudaEventDestroy(w.ev_k2);
        if (w.ev_done) cudaEventDestroy(w.ev_done);
        if (w.ev_copied) cudaEventDestroy(w.ev_copied);
    }
    if (job->ev_producer) cudaEventDestroy(job->ev_producer);
    if (job->ev_consumer) cudaEventDestroy(job->ev_consumer);
    if (job->ev_copy_begin) cudaEventDestroy(job->ev_copy_begin);
    if (job->ev_copy_end) cudaEventDestroy(job->ev_copy_end);
    for (FileSpec& f : job->files)
        if (f.fd >= 0) close(f.fd);
    delete job;
    return TSNAP_OK;
}

// ---- caller-supplied arena, timeline, probes ------------------------------------------------------------------
int tsnap_job_arena_hint(tsnap_job* job, tsnap_arena_hint* out) {
    if (!job || !out) return set_err(TSNAP_EINVAL, "null argument");
    // host_only is only known at submit: recompute from the members
    ArenaNeed n;
    for (const FileSpec& f : job->files) {
        if (f.nbytes == 0) continue;
        bool device = false;
        for (const tsnap_copy_desc& d : f.members)
            device = device || (job->kind == kLoad ? d.dst_space : d.src_space) == TSNAP_SPACE_DEVICE;
        if (!device) continue;
        const uint64_t fb = align_up(f.nbytes, 256);
        n.total += fb;
        n.largest = std::max(n.largest, fb);
        if (!f.dense) {
            n.nd_total += fb;
            n.nd_largest = std::max(n.nd_largest, fb);
        }
    }
    out->total_bytes = n.total;
    out->largest_file_bytes = n.largest;
    out->strided_total_bytes = n.nd_total;
    out->strided_largest_bytes = n.nd_largest;
    return TSNAP_OK;
}
int tsnap_job_set_arena(tsnap_job* job, void* device_ptr, uint64_t nbytes) {
    if (!job) return set_err(TSNAP_EINVAL, "null job");
    if (job->submitted) return set_err(TSNAP_ESTATE, "job already submitted");
    if (nbytes && !device_ptr) return set_err(TSNAP_EINVAL, "null arena");
    if (uintptr_t(device_ptr) & 255) return set_err(TSNAP_EINVAL, "the arena must be 256 B aligned");
    job->arena = static_cast<char*>(device_ptr);
    job->arena_bytes = nbytes / 512 * 512;  // two equal 256 B-aligned halves
    job->arena_set = true;
    return TSNAP_OK;
}

int tsnap_job_set_host_budget(tsnap_job* job, uint64_t bytes) {
    if (!job) return set_err(TSNAP_EINVAL, "null job");
    if (job->submitted) return set_err(TSNAP_ESTATE, "job already submitted");
    const uint64_t sb = job->eng->cfg.pinned_slot_bytes ? job->eng->cfg.pinned_slot_bytes : (32ull << 20);
    job->max_slots = bytes ? int(std::max<uint64_t>(2, std::min<uint64_t>(bytes / sb, 1u << 20))) : 0;
    return TSNAP_OK;
}

int tsnap_job_get_trace(tsnap_job* job, tsnap_trace_rec* out, uint64_t cap, uint64_t* n) {
    if (!job || !n) return set_err(TSNAP_EINVAL, "null argument");
    std::lock_guard<std::mutex> g(job->trace_mu);
    *n = job->trace.size();
    if (out)
        for (uint64_t i = 0; i < cap && i < job->trace.size(); ++i) out[i] = job->trace[i];
    return TSNAP_OK;
}

int tsnap_engine_probe(tsnap_engine* eng, int kind, const char* dir, uint64_t bytes, double* out_gbs) {
    if (!eng || !out_gbs) return set_err(TSNAP_EINVAL, "null argument");
    int rc = ensure_ring(eng);
    if (rc != TSNAP_OK) return rc;
    const uint64_t sb = eng->ring.slot_bytes();
    const uint64_t chunks = std::max<uint64_t>(1, bytes / sb);
    if (kind == TSNAP_PROBE_D2H || kind == TSNAP_PROBE_H2D) {
        if (!eng->has_device) return set_err(TSNAP_ECUDA, "link probe on a host-only engine");
        cudaSetDevice(eng->device);
        const int depth = std::min<int>(eng->ring.count(), 8);
        char* dev = nullptr;
        CUDA_TRY(cudaMalloc(&dev, sb * depth));
        std::vector<char*> slots;
        for (int i = 0; i < depth; ++i) slots.push_back(eng->ring.acquire());
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0);
        cudaEventCreate(&e1);
        for (int pass = 0; pass < 2; ++pass) {  // pass 0 warms the path
            const uint64_t c = pass == 0 ? std::min<uint64_t>(chunks, 8) : chunks;
            cudaEventRecord(e0, eng->s_copy);
            for (uint64_t i = 0; i < c; ++i) {
                char* h = slots[i % depth];
                char* d = dev + (i % depth) * sb;
                if (kind == TSNAP_PROBE_D2H) cudaMemcpyAsync(h, d, sb, cudaMemcpyDeviceToHost, eng->s_copy);
                else cudaMemcpyAsync(d, h, sb, cudaMemcpyHostToDevice, eng->s_copy);
            }
            cudaEventRecord(e1, eng->s_copy);
            cudaEventSynchronize(e1);
        }
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        for (char* p : slots) eng->ring.release(p);
        cudaFree(dev);
        *out_gbs = ms > 0 ? double(chunks * sb) / 1e9 / (ms / 1e3) : 0;
        return TSNAP_OK;
    }
    if (kind != TSNAP_PROBE_WRITE && kind != TSNAP_PROBE_READ) return set_err(TSNAP_EINVAL, "unknown probe kind");
    if (!dir) return set_err(TSNAP_EINVAL, "null dir");
    // Same shape as a save job: files of 8 chunks, chunks of different files interleaved, I/O by the engine's workers.
    // Every call uses fresh file names (writes never truncate an older probe's dirty pages) and removes its files; the
    // READ probe first writes its files (untimed), then times reading them back.  Only the I/O itself is timed.
    static std::atomic<uint64_t> serial{0};
    const uint64_t per_file = 8;
    const uint64_t nfiles = (chunks + per_file - 1) / per_file;
    std::vector<int> fds(nfiles, -1);
    std::vector<std::string> paths(nfiles);
    std::string base = std::string(dir) + "/tsnap_probe_" + std::to_string(getpid()) + "_" + std::to_string(serial.fetch_add(1)) + "_";
    if (make_parent_dirs(base) != 0) return set_err(TSNAP_EIO, std::string("mkdir ") + dir + ": " + strerror(errno));
    auto cleanup = [&] {
        for (size_t i = 0; i < fds.size(); ++i) {
            if (fds[i] >= 0) close(fds[i]);
            if (!paths[i].empty()) unlink(paths[i].c_str());
        }
    };
    for (uint64_t i = 0; i < nfiles; ++i) {
        paths[i] = base + std::to_string(i);
        const int flags = O_RDWR | O_CREAT | O_TRUNC;
        if (eng->odirect) fds[i] = open(paths[i].c_str(), flags | O_DIRECT, 0644);
        if (fds[i] < 0) fds[i] = open(paths[i].c_str(), flags, 0644);
        if (fds[i] < 0) {
            const std::string msg = "open " + paths[i] + ": " + strerror(errno);
            cleanup();
            return set_err(TSNAP_EIO, msg);
        }
    }
    std::atomic<int> err{0};
    auto pass = [&](bool write) -> double {
        std::atomic<uint64_t> left{chunks};
        std::mutex mu;
        std::condition_variable cv;
        auto t0 = clk::now();
        for (uint64_t c = 0; c < chunks; ++c) {
            const uint64_t fi = c % nfiles, k = c / nfiles;
            char* slot = eng->ring.acquire();
            eng->io->post([&, fi, k, slot, write] {
                int r;
                {
                    TokenGuard tok;
                    r = write ? pwrite_all(fds[fi], slot, sb, k * sb) : pread_all(fds[fi], slot, sb, k * sb);
                }
                if (r != 0) err.store(errno ? errno : EIO);
                eng->ring.release(slot);
                if (left.fetch_sub(1) == 1) {
                    std::lock_guard<std::mutex> g(mu);
                    cv.notify_all();
                }
            });
        }
        std::unique_lock<std::mutex> g(mu);
        cv.wait(g, [&] { return left.load() == 0; });
        return ms_since(t0);
    };
    double ms = pass(true);
    if (kind == TSNAP_PROBE_READ && !err.load()) ms = pass(false);
    cleanup();
    if (err.load()) return set_err(TSNAP_EIO, std::string("probe I/O failed: ") + strerror(err.load()));
    *out_gbs = double(chunks * sb) / 1e9 / (ms / 1e3);
    return TSNAP_OK;
}

// ---- stager / consumer seam ---------------------------------------------------------------------------------
static void* pin_get(tsnap_engine* eng, size_t nbytes, size_t* cap) {
    {
        std::lock_guard<std::mutex> g(eng->pin_mu);
        size_t best = SIZE_MAX;
        for (size_t i = 0; i < eng->pin_cache.size(); ++i)
            if (eng->pin_cache[i].first >= nbytes && (best == SIZE_MAX || eng->pin_cache[i].first < eng->pin_cache[best].first))
                best = i;
        if (best != SIZE_MAX && eng->pin_cache[best].first <= 2 * std::max<size_t>(nbytes, 4096)) {
            auto kv = eng->pin_cache[best];
            eng->pin_cache.erase(eng->pin_cache.begin() + best);
            *cap = kv.first;
            return kv.second;
        }
    }
    size_t c = align_up(std::max<size_t>(nbytes, 4096), 4096);
    void* p = nullptr;
    if (eng->has_device) {
        cudaSetDevice(eng->device);
        if (cudaHostAlloc(&p, c, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    } else if (posix_memalign(&p, 4096, c) != 0) {
        return nullptr;
    }
    *cap = c;
    return p;
}

int tsnap_stage_submit(tsnap_engine* eng, const tsnap_copy_desc* members, int32_t n, uint64_t nbytes,
                       void* producer_stream, tsnap_buffer** out) {
    if (!eng || !out || (n > 0 && !members)) return set_err(TSNAP_EINVAL, "null argument");
    tsnap_job* job = nullptr;
    int rc = job_create(eng, kStage, &job);
    if (rc != TSNAP_OK) return rc;
    int32_t fi;
    add_file(job, "<stage>", 0, nbytes, &fi);
    for (int32_t i = 0; i < n; ++i) {
        if (members[i].dst_space != TSNAP_SPACE_WIRE) {
            delete job;
            return set_err(TSNAP_EINVAL, "stage members must have a WIRE destination");
        }
        rc = add_member(job, fi, &members[i], true);
        if (rc != TSNAP_OK) {
            delete job;
            return rc;
        }
    }
    job->stage_buf = pin_get(eng, nbytes, &job->stage_cap);
    if (!job->stage_buf) {
        delete job;
        return set_err(TSNAP_ENOMEM, "pinned allocation failed");
    }
    rc = submit(job, producer_stream, false);
    if (rc != TSNAP_OK) {
        std::lock_guard<std::mutex> g(eng->pin_mu);
        eng->pin_cache.emplace_back(job->stage_cap, job->stage_buf);
        delete job;
        return rc;
    }
    tsnap_buffer* b = new tsnap_buffer{job};
    *out = b;
    return TSNAP_OK;
}
int tsnap_buffer_wait_device(tsnap_buffer* buf) {
    if (!buf) return set_err(TSNAP_EINVAL, "null buffer");
    return tsnap_job_wait_device(buf->job);
}
int tsnap_buffer_wait(tsnap_buffer* buf, void** host_ptr, uint64_t* nbytes) {
    if (!buf) return set_err(TSNAP_EINVAL, "null buffer");
    int rc = tsnap_job_wait(buf->job);
    if (host_ptr) *host_ptr = buf->job->stage_buf;
    if (nbytes) *nbytes = buf->job->files[0].nbytes;
    return rc;
}
int tsnap_buffer_get_stats(tsnap_buffer* buf, tsnap_job_stats* out) {
    if (!buf) return set_err(TSNAP_EINVAL, "null buffer");
    return tsnap_job_get_stats(buf->job, out);
}
int tsnap_buffer_release(tsnap_buffer* buf) {
    if (!buf) return TSNAP_OK;
    tsnap_job* job = buf->job;
    tsnap_engine* eng = job->eng;
    {
        std::unique_lock<std::mutex> g(job->mu);
        job->cv.wait(g, [job] { return job->done; });
    }
    {
        std::lock_guard<std::mutex> g(eng->pin_mu);
        eng->pin_cache.emplace_back(job->stage_cap, job->stage_buf);
        // keep the cache bounded: drop the largest buffers beyond 8 entries
        while (eng->pin_cache.size() > 8) {
            size_t big = 0;
            for (size_t i = 1; i < eng->pin_cache.size(); ++i)
                if (eng->pin_cache[i].first > eng->pin_cache[big].first) big = i;
            if (eng->has_device) cudaFreeHost(eng->pin_cache[big].second);
            else free(eng->pin_cache[big].second);
            eng->pin_cache.erase(eng->pin_cache.begin() + big);
        }
    }
    tsnap_job_destroy(job);
    delete buf;
    return TSNAP_OK;
}

int tsnap_consume(tsnap_engine* eng, const void* host_buf, uint64_t nbytes, const tsnap_copy_desc* members,
                  int32_t n, void* consumer_stream) {
    if (!eng || (nbytes && !host_buf) || (n > 0 && !members)) return set_err(TSNAP_EINVAL, "null argument");
    std::string err;
    // host destinations: plain host execution against the caller's buffer
    std::vector<tsnap_copy_desc> dev;
    for (int32_t i = 0; i < n; ++i) {
        if (members[i].src_space != TSNAP_SPACE_WIRE) return set_err(TSNAP_EINVAL, "consume members must have a WIRE source");
        if (members[i].dst_space == TSNAP_SPACE_HOST) {
            NormalizedCopy nc;
            int rc = normalize_copy(members[i], uint64_t(uintptr_t(host_buf)), false, &nc, &err);
            if (rc != TSNAP_OK) return set_err(rc, err);
            for (int k = 0; k < nc.n; ++k) host_copy_range(nc.m[k], 0, nc.m[k].bytes);
        } else {
            dev.push_back(members[i]);
        }
    }
    if (dev.empty() || nbytes == 0) return TSNAP_OK;
    if (!eng->has_device) return set_err(TSNAP_ECUDA, "device members on a host-only engine");
    // device destinations: a load job whose "file" is the caller's memory
    tsnap_job* job = nullptr;
    int rc = job_create(eng, kLoad, &job);
    if (rc != TSNAP_OK) return rc;
    int32_t fi;
    add_file(job, "<memory>", 0, nbytes, &fi);
    for (const tsnap_copy_desc& d : dev) {
        rc = add_member(job, fi, &d, false);
        if (rc != TSNAP_OK) {
            delete job;
            return rc;
        }
    }
    job->files[0].mem_src = static_cast<const char*>(host_buf);
    rc = submit(job, consumer_stream, true);
    if (rc != TSNAP_OK) {
        delete job;
        return rc;
    }
    rc = tsnap_job_wait(job);
    std::string msg = rc != TSNAP_OK ? std::string(last_err()) : std::string();
    tsnap_job_destroy(job);
    if (rc != TSNAP_OK) return set_err(rc, msg);
    return TSNAP_OK;
}

int tsnap_scatter_device(tsnap_engine* eng, const void* device_wire, uint64_t nbytes, const tsnap_copy_desc* members,
                         int32_t n, void* consumer_stream) {
    if (!eng || (nbytes && !device_wire) || (n > 0 && !members)) return set_err(TSNAP_EINVAL, "null argument");
    if (n == 0 || nbytes == 0) return TSNAP_OK;
    if (!eng->has_device) return set_err(TSNAP_ECUDA, "device members on a host-only engine");
    cudaSetDevice(eng->device);
    // a job that is never queued: it only carries the planner state of one wave whose "arena" is the caller's buffer
    tsnap_job job;
    job.eng = eng;
    job.kind = kLoad;
    job.arena = static_cast<char*>(const_cast<void*>(device_wire));
    job.arena_bytes = nbytes;
    job.files.emplace_back();
    FileSpec& f = job.files.back();
    f.path = "<device wire>";
    f.nbytes = nbytes;
    for (int32_t i = 0; i < n; ++i) {
        if (members[i].src_space != TSNAP_SPACE_WIRE || members[i].dst_space != TSNAP_SPACE_DEVICE)
            return set_err(TSNAP_EINVAL, "scatter_device members go from WIRE to DEVICE");
        int rc = add_member(&job, 0, &members[i], false);
        if (rc != TSNAP_OK) return rc;
    }
    Wave w;
    w.files.push_back(0);
    int rc = plan_wave(&job, w);
    if (rc != TSNAP_OK) return rc;
    cudaEvent_t ev = eng->get_event();
    cudaError_t e = cudaEventRecord(ev, static_cast<cudaStream_t>(consumer_stream));
    if (e == cudaSuccess) e = cudaStreamWaitEvent(eng->s_kernel, ev, 0);
    eng->put_event(ev);
    if (e != cudaSuccess) return set_err(TSNAP_ECUDA, std::string("scatter_device: ") + cudaGetErrorString(e));
    rc = launch_wave(&job, w);
    if (rc == TSNAP_OK && cudaEventSynchronize(w.ev_done) != cudaSuccess) rc = set_err(TSNAP_ECUDA, "scatter kernel failed");
    if (w.d_tables) {
        if (rc != TSNAP_OK) cudaStreamSynchronize(eng->s_kernel);
        eng->put_table(w.d_tables, w.table_cap);
    }
    for (cudaEvent_t x : {w.ev_k0, w.ev_k1, w.ev_kr, w.ev_k2, w.ev_done})
        if (x) cudaEventDestroy(x);
    return rc;
}

// ---- planning introspection + host execution -----------------------------------------------------------------
int tsnap_plan_describe(const tsnap_copy_desc* members, int32_t n, uint64_t wire_base_align, tsnap_plan_info* out) {
    if (!out || (n > 0 && !members)) return set_err(TSNAP_EINVAL, "null argument");
    memset(out, 0, sizeof(*out));
    std::string err;
    // a synthetic wire base with the requested alignment residue
    const uint64_t base = (1ull << 40) + (wire_base_align & 255);
    for (int32_t i = 0; i < n; ++i) {
        NormalizedCopy nc;
        int rc = normalize_copy(members[i], base, true, &nc, &err);
        if (rc != TSNAP_OK) return set_err(rc, err);
        const bool host = members[i].src_space == TSNAP_SPACE_HOST || members[i].dst_space == TSNAP_SPACE_HOST;
        for (int k = 0; k < nc.n; ++k) {
            const Member& m = nc.m[k];
            const uint64_t nt = tile_count(m);
            // every tile range must tile [0, bytes) exactly (transpose tiles are 2-D blocks, not byte ranges)
            uint64_t expect = 0;
            for (uint64_t t = 0; t < nt && m.mode != kModeTranspose; ++t) {
                uint64_t lo, hi;
                tile_range(m, uint32_t(t), &lo, &hi);
                if (lo != expect || hi <= lo) return set_err(TSNAP_EINVAL, "internal: tile cover broken");
                expect = hi;
            }
            if (m.mode != kModeTranspose && expect != m.bytes) return set_err(TSNAP_EINVAL, "internal: tile cover incomplete");
            if (host) {
                out->n_members_host++;
                out->bytes_host += m.bytes;
            } else if (m.mode == kModeRows) {
                out->n_members_rows++;
                out->n_tiles_rows += nt;
                out->bytes_rows += m.bytes;
            } else if (m.mode == kModeBulk) {
                out->n_members_bulk++;
                out->n_tiles_bulk += nt;
                out->bytes_bulk += m.bytes;
            } else {
                out->n_members_lsu++;
                out->n_tiles_lsu += nt;
                out->bytes_lsu += m.bytes;
            }
        }
    }
    return TSNAP_OK;
}

int tsnap_host_execute(const tsnap_copy_desc* members, int32_t n, void* wire_buf, uint64_t wire_nbytes,
                       int32_t threads) {
    if ((n > 0 && !members) || (!wire_buf && wire_nbytes)) return set_err(TSNAP_EINVAL, "null argument");
    std::string err;
    struct Work {
        Member m;
        uint64_t lo, hi;
    };
    std::vector<Work> work;
    const uint64_t grain = 8ull << 20;
    for (int32_t i = 0; i < n; ++i) {
        const tsnap_copy_desc& d = members[i];
        if (d.src_space == TSNAP_SPACE_DEVICE || d.dst_space == TSNAP_SPACE_DEVICE)
            return set_err(TSNAP_EINVAL, "tsnap_host_execute only handles HOST <-> WIRE copies");
        NormalizedCopy nc;
        int rc = normalize_copy(d, uint64_t(uintptr_t(wire_buf)), false, &nc, &err);
        if (rc != TSNAP_OK) return set_err(rc, err);
        for (int k = 0; k < nc.n; ++k) {
            const Member& m = nc.m[k];
            const uint64_t wire_off = (d.dst_space == TSNAP_SPACE_WIRE ? m.dst : m.src) - uint64_t(uintptr_t(wire_buf));
            const uint64_t trailer = (m.mode == kModeCast && (m.shift & 1)) ? 16 : 0;  // quantised: [scale][zero_point]
            if (d.dst_space == TSNAP_SPACE_WIRE && wire_off + m.bytes + trailer > wire_nbytes)
                return set_err(TSNAP_EINVAL, "member exceeds the wire buffer");
            // grains must not split a destination element of a cast
            const uint64_t g = grain / 16 * 16;
            for (uint64_t lo = 0; lo < m.bytes; lo += g) work.push_back({m, lo, std::min(m.bytes, lo + g)});
        }
    }
    if (threads <= 1 || work.size() <= 1) {
        for (const Work& w : work) host_copy_range(w.m, w.lo, w.hi);
        return TSNAP_OK;
    }
    std::atomic<size_t> next{0};
    std::vector<std::thread> ts;
    const int nt = int(std::min<size_t>(size_t(threads), work.size()));
    for (int t = 0; t < nt; ++t)
        ts.emplace_back([&] {
            for (;;) {
                size_t i = next.fetch_add(1);
                if (i >= work.size()) return;
                host_copy_range(work[i].m, work[i].lo, work[i].hi);
            }
        });
    for (auto& t : ts) t.join();
    return TSNAP_OK;
}

}  // extern "C"
