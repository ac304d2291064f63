// vmig_engine.cu -- process-wide GPU context, pinned/HBM slot pools and the per-GPU streaming
// pipeline (see vmig_engine.h for the data flow).  Replaces the byte-moving loop of the
// reference's `tar c | tar x` pipe (utils/copy.go:17-27) and of `mv` in the helper container
// (utils/copy.go:116); everything here is new design, there is no reference counterpart.
#include "vmig_engine.h"
#include "vmig_kernels.cuh"
#include "vmig_cufile.h"
#include "vmig_sched.h"

#include <sched.h>
#include <unistd.h>
#include <sys/resource.h>
#include <sys/mman.h>
#include <sys/syscall.h>
#include <condition_variable>
#include <deque>
#include <thread>
#include <fstream>
#include <sstream>
#include <algorithm>
#include <unordered_map>
#include <cstdlib>

namespace vmig {

// ---------------------------------------------------------------------------------------------
// errors
static thread_local std::string g_last_error;
void set_last_error_str(const std::string& s) { g_last_error = s; }
void set_last_error(const char* fmt, ...) {
    char buf[1024]; va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap); g_last_error = buf;
}
const char* last_error_cstr() { return g_last_error.c_str(); }
long env_long(const char* name, long dflt) {
    const char* v = getenv(name);
    if (!v || !*v) return dflt;
    char* end = nullptr; long r = strtol(v, &end, 10);
    return end && *end == 0 ? r : dflt;
}

// ---------------------------------------------------------------------------------------------
// tunables (env, read once per process)
static constexpr uint32_t kMaxBatchBlocks = 4096;
static uint32_t g_slot_bytes = 0, g_slots = 0, g_pipes_per_gpu = 0;
static void load_tunables() {
    if (g_slot_bytes) return;
    long mb = env_long("VMIG_SLOT_MB", 32);
    if (mb < 4) mb = 4; if (mb > 1024) mb = 1024;
    long ns = env_long("VMIG_SLOTS", 16);
    if (ns < 2) ns = 2; if (ns > 64) ns = 64;
    long pp = env_long("VMIG_PIPES_PER_GPU", 2);
    if (pp < 1) pp = 1; if (pp > 8) pp = 8;
    g_slots = (uint32_t)ns; g_pipes_per_gpu = (uint32_t)pp;
    g_slot_bytes = (uint32_t)(mb << 20);
}
uint32_t pipe_slot_bytes() { load_tunables(); return g_slot_bytes; }

// ---------------------------------------------------------------------------------------------
// slot / pipe
struct Slot {
    uint8_t* h_out = nullptr;   // pinned, slot_bytes + pad
    uint8_t* d_buf = nullptr;   // HBM,    slot_bytes + pad
    uint8_t* h_desc = nullptr;  // pinned: packed [offs u64][prior u64][lens u32][valid u8] for n blocks
    uint8_t* d_desc = nullptr;
    uint8_t* h_res = nullptr;   // pinned: packed [hashes u64][changed u8]
    uint8_t* d_res = nullptr;
    uint32_t* d_counter = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr, ev_hash = nullptr, ev_d2h = nullptr;
    size_t out_mapped = 0;                  // > 0: ring is an mmap'ed huge-page region registered with CUDA
    bool cf_registered = false;             // d_buf is registered with cuFile (GPUDirect Storage backends)
};

// Staging rings: 2 MiB-aligned anonymous memory with MADV_HUGEPAGE, faulted in, then page-locked
// with cudaHostRegister -- the kernel's copy_to/from_user and the DMA engines then walk 16 huge
// pages per 32 MiB slot instead of 8 192 small ones.  The OUT ring has one per slot, the readers' pieces one per pipe.
// Falls back to cudaHostAlloc (VMIG_HUGE=0, or if the mapping / registration fails).
static int ring_alloc(uint8_t** out, size_t bytes, size_t* mapped)
{
    *mapped = 0;
    if (env_long("VMIG_HUGE", 1) != 0) {
        const size_t len = align_up(bytes, 2u << 20);
        void* p = mmap(nullptr, len + (2u << 20), PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
        if (p != MAP_FAILED) {
            uint8_t* a = (uint8_t*)align_up((uint64_t)(uintptr_t)p, 2u << 20);
            if (a != p) munmap(p, (size_t)(a - (uint8_t*)p));
            const size_t tail = (size_t)(((uint8_t*)p + len + (2u << 20)) - (a + len));
            if (tail) munmap(a + len, tail);
            madvise(a, len, MADV_HUGEPAGE);
            madvise(a, len, MADV_DONTFORK);        // a forked child (the control plane exec's tools) must not share DMA targets
            if (env_long("VMIG_RING_MBIND", 0) != 0) {
                // experiment knob (off by default, untested on the bench box in round 1): give the ring an explicit
                // memory policy (preferred = the creating thread's node, which is the GPU's) -- VMAs with their own
                // policy are skipped by the kernel's automatic NUMA-balancing scanner, whose PROT_NONE sweeps and
                // TLB shootdowns hit every thread of a many-lane process
                unsigned cpu = 0, node = 0;
                if (syscall(SYS_getcpu, &cpu, &node, nullptr) == 0 && node < 64) {
                    unsigned long mask = 1ul << node;
                    syscall(SYS_mbind, a, len, 1 /* MPOL_PREFERRED */, &mask, 65ul, 0u);
                }
            }
            memset(a, 0, len);
            if (cudaHostRegister(a, len, cudaHostRegisterPortable) == cudaSuccess) { *out = a; *mapped = len; return VMIG_OK; }
            cudaGetLastError();
            munmap(a, len);
        }
    }
    CU_API(cudaHostAlloc((void**)out, bytes, cudaHostAllocPortable));
    memset(*out, 0, bytes);
    return VMIG_OK;
}
static void ring_free(uint8_t* p, size_t mapped)
{
    if (!p) return;
    if (mapped) { cudaHostUnregister(p); munmap(p, mapped); } else cudaFreeHost(p);
}
static constexpr size_t kDescBytes = (size_t)kMaxBatchBlocks * (8 + 8 + 4 + 1) + 64;
static constexpr size_t kResBytes  = (size_t)kMaxBatchBlocks * (8 + 1) + 64;

// Reader staging: each reader owns kPieces pinned pieces of kPieceBytes and copies each one into the HBM slot as soon as
// it is filled, so a staged byte is still in the CPU's cache when the DMA reads it (a 32 MiB slot staged whole is written
// back to DRAM and read from there again).  The probe loop measured 22.2-22.9 GiB/s with 4 x 1 MiB private pieces against
// 12.3-13.9 with pieces rotating through a 512 MiB ring (profiles/r01_piece_probe.txt); 16 pieces per reader gained
// nothing over 4 (profiles/r03_piece_variants.txt).  Pieces are whole sectors, so the rounded-up O_DIRECT read of a
// file's short last block ends inside its piece.
static constexpr uint32_t kPieces = 4, kPieceBytes = 1u << 20;
static_assert(kPieceBytes % 4096 == 0, "an O_DIRECT piece is whole sectors");
struct PieceReader {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[kPieces] = {};     // the last copy out of each piece
};

class Pipe {
public:
    DeviceInfo dev;
    uint32_t slot_bytes = 0;
    std::vector<Slot> slots;
    uint8_t* pieces = nullptr;        // readers.size() x kPieces x kPieceBytes, pinned
    size_t pieces_mapped = 0;
    std::vector<PieceReader> readers;
    int create(const DeviceInfo& d);
    int create_here(const DeviceInfo& d);
    int reserve_readers(uint32_t n);
    void destroy();
};

static void bind_thread(const DeviceInfo& d);
static void bind_thread_complement(const DeviceInfo& d);

// A pipe is created by a thread bound to the GPU's NUMA-local CPUs, so that what it first-touches stays on the GPU's
// socket; only the OUT ring is placed on purpose (create_here).
int Pipe::create(const DeviceInfo& d)
{
    int rc = VMIG_OK; std::string msg;
    std::thread t([&] { bind_thread(d); rc = create_here(d); if (rc) msg = last_error_cstr(); });
    t.join();
    if (rc) set_last_error_str(msg);
    return rc;
}

int Pipe::create_here(const DeviceInfo& d)
{
    load_tunables();
    dev = d; slot_bytes = g_slot_bytes;
    CU_API(cudaSetDevice(d.dev));
    slots.resize(g_slots);
    const size_t cap = (size_t)slot_bytes + kTailPad;
    // Which socket's DRAM holds the OUT ring (first touch decides).  0 = the GPU's socket, 1 = the other socket(s),
    // 2 = alternate slot by slot.  It defaults to the writers' side (VMIG_BIND_WRITERS=2 puts them on the other socket):
    // the D2H DMA crosses UPI once, the writers then read it locally.
    const long out_node = env_long("VMIG_RING_OUT_NODE", env_long("VMIG_BIND_WRITERS", 2) == 2 ? 1 : 0);      // +5..8 % end to end (profiles/r02_sweep_ring_placement.txt)
    auto place = [&](long mode, size_t idx) {
        const bool far = mode == 1 || (mode == 2 && (idx & 1));
        if (far) bind_thread_complement(d); else bind_thread(d);
    };
    size_t slot_idx = 0;
    for (auto& s : slots) {
        place(out_node, slot_idx);
        { int rc = ring_alloc(&s.h_out, cap, &s.out_mapped); if (rc) return rc; }
        bind_thread(d);
        slot_idx++;
        CU_API(cudaMalloc((void**)&s.d_buf, cap));
        CU_API(cudaMemset(s.d_buf, 0, cap));
        CU_API(cudaHostAlloc((void**)&s.h_desc, kDescBytes, cudaHostAllocPortable));
        CU_API(cudaMalloc((void**)&s.d_desc, kDescBytes));
        CU_API(cudaHostAlloc((void**)&s.h_res, kResBytes, cudaHostAllocPortable));
        CU_API(cudaMalloc((void**)&s.d_res, kResBytes));
        CU_API(cudaMalloc((void**)&s.d_counter, 256));
        CU_API(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        CU_API(cudaEventCreate(&s.ev_k0)); CU_API(cudaEventCreate(&s.ev_k1));
        CU_API(cudaEventCreateWithFlags(&s.ev_hash, cudaEventDisableTiming));
        CU_API(cudaEventCreateWithFlags(&s.ev_d2h, cudaEventDisableTiming));
    }
    CU_API(cudaDeviceSynchronize());
    return VMIG_OK;
}
// Pieces for n readers.  The pool grows (up to the 64 readers a call may ask for) and is never shrunk; it is only replaced
// between calls, when no copy reads it.  Allocated and first-touched on the GPU's socket, where the readers run.
int Pipe::reserve_readers(uint32_t n)
{
    if (n <= readers.size() && pieces) return VMIG_OK;
    int rc = VMIG_OK; std::string msg;
    std::thread t([&] {
        bind_thread(dev);
        rc = [&]() -> int {
            CU_API(cudaSetDevice(dev.dev));
            ring_free(pieces, pieces_mapped); pieces = nullptr; pieces_mapped = 0;
            { int r = ring_alloc(&pieces, (size_t)n * kPieces * kPieceBytes, &pieces_mapped); if (r) return r; }
            while (readers.size() < n) {
                readers.emplace_back();
                PieceReader& pr = readers.back();
                CU_API(cudaStreamCreateWithFlags(&pr.stream, cudaStreamNonBlocking));
                for (auto& e : pr.ev) CU_API(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            }
            return VMIG_OK;
        }();
        if (rc) msg = last_error_cstr();
    });
    t.join();
    if (rc) set_last_error_str(msg);
    return rc;
}
void Pipe::destroy()
{
    cudaSetDevice(dev.dev);
    for (auto& r : readers) {
        if (r.stream) { cudaStreamSynchronize(r.stream); cudaStreamDestroy(r.stream); }
        for (auto e : r.ev) if (e) cudaEventDestroy(e);
    }
    readers.clear();
    ring_free(pieces, pieces_mapped); pieces = nullptr; pieces_mapped = 0;
    for (auto& s : slots) {
        if (s.stream) cudaStreamSynchronize(s.stream);
        if (s.cf_registered) { cufile_buf_deregister(s.d_buf); s.cf_registered = false; }
        ring_free(s.h_out, s.out_mapped); cudaFree(s.d_buf); cudaFreeHost(s.h_desc); cudaFree(s.d_desc);
        cudaFreeHost(s.h_res); cudaFree(s.d_res); cudaFree(s.d_counter);
        if (s.stream) cudaStreamDestroy(s.stream);
        if (s.ev_k0) cudaEventDestroy(s.ev_k0); if (s.ev_k1) cudaEventDestroy(s.ev_k1);
        if (s.ev_hash) cudaEventDestroy(s.ev_hash); if (s.ev_d2h) cudaEventDestroy(s.ev_d2h);
    }
    slots.clear();
}

// ---------------------------------------------------------------------------------------------
// context
struct DevPool {
    DeviceInfo info;
    std::vector<Pipe*> free_pipes;
    uint32_t n_pipes = 0;
};
static cpu_set_t g_proc_cpus; static bool g_have_proc_cpus = false;     // affinity of the first thread that initialised the library
static std::mutex g_mu;
static std::condition_variable g_cv;
static bool g_inited = false;
static std::vector<DevPool> g_devs;

static std::vector<int> parse_cpulist(const std::string& s) {
    std::vector<int> out; std::stringstream ss(s); std::string tok;
    while (std::getline(ss, tok, ',')) {
        int a, b;
        if (sscanf(tok.c_str(), "%d-%d", &a, &b) == 2) { for (int i = a; i <= b; i++) out.push_back(i); }
        else if (sscanf(tok.c_str(), "%d", &a) == 1) out.push_back(a);
    }
    return out;
}
static std::vector<int> gpu_local_cpus(int dev) {
    if (env_long("VMIG_NUMA", 1) == 0) return {};
    char bus[64] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, dev) != cudaSuccess) { cudaGetLastError(); return {}; }
    for (char* p = bus; *p; p++) *p = (char)tolower(*p);
    std::ifstream f(std::string("/sys/bus/pci/devices/") + bus + "/local_cpulist");
    std::string line;
    if (!f || !std::getline(f, line)) return {};
    std::vector<int> cpus = parse_cpulist(line);
    // intersect with what this process may run on
    cpu_set_t cur; CPU_ZERO(&cur);
    if (sched_getaffinity(0, sizeof cur, &cur) == 0) {
        std::vector<int> keep; for (int c : cpus) if (c < CPU_SETSIZE && CPU_ISSET(c, &cur)) keep.push_back(c);
        cpus.swap(keep);
    }
    return cpus;
}

int ctx_device_count()
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) { cudaGetLastError(); return fail(VMIG_ENOGPU, "no CUDA device (%s); libvmig has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "count 0"); }
    int ok = 0;
    for (int i = 0; i < n; i++) { cudaDeviceProp p; if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ok++; }
    if (!ok) return fail(VMIG_ENOGPU, "no sm_100 (Blackwell B200) device among %d CUDA devices; libvmig ships sm_100a code only", n);
    return ok;
}

int ctx_init(uint32_t gpu_mask)
{
    std::lock_guard<std::mutex> lk(g_mu);
    load_tunables();
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) { cudaGetLastError(); return fail(VMIG_ENOGPU, "no CUDA device (%s); libvmig has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "count 0"); }
    if (!g_inited) {
        CPU_ZERO(&g_proc_cpus);
        g_have_proc_cpus = sched_getaffinity(0, sizeof g_proc_cpus, &g_proc_cpus) == 0;
        struct rlimit rl;
        if (getrlimit(RLIMIT_NOFILE, &rl) == 0 && rl.rlim_cur < rl.rlim_max) { rl.rlim_cur = rl.rlim_max; setrlimit(RLIMIT_NOFILE, &rl); }
    }
    int added = 0;
    for (int i = 0; i < n && i < 32; i++) {
        if (gpu_mask && !(gpu_mask & (1u << i))) continue;
        bool have = false;
        for (auto& d : g_devs) if (d.info.dev == i) have = true;
        if (have) { added++; continue; }
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, i) != cudaSuccess) { cudaGetLastError(); continue; }
        if (p.major != 10) continue;          // sm_100a SASS only
        DevPool dp; dp.info.dev = i; dp.info.sm_count = p.multiProcessorCount; dp.info.cpus = gpu_local_cpus(i);
        g_devs.push_back(dp);
        added++;
    }
    if (!added && g_devs.empty()) return fail(VMIG_ENOGPU, "no sm_100 device selected by mask 0x%x (%d CUDA devices)", gpu_mask, n);
    std::sort(g_devs.begin(), g_devs.end(), [](const DevPool& a, const DevPool& b) { return a.info.dev < b.info.dev; });
    g_inited = true;
    return VMIG_OK;
}

void ctx_shutdown()
{
    std::lock_guard<std::mutex> lk(g_mu);
    for (auto& d : g_devs) {
        for (Pipe* p : d.free_pipes) { p->destroy(); delete p; }
        d.free_pipes.clear(); d.n_pipes = 0;
    }
    g_devs.clear();
    g_inited = false;
}

int ctx_select(uint32_t mask, std::vector<DeviceInfo>* out)
{
    {
        std::unique_lock<std::mutex> lk(g_mu);
        bool need = !g_inited;
        if (!need && mask) for (int i = 0; i < 32; i++) if (mask & (1u << i)) { bool have = false; for (auto& d : g_devs) if (d.info.dev == i) have = true; if (!have) need = true; }
        if (need) { lk.unlock(); int rc = ctx_init(mask); if (rc) return rc; }
    }
    std::lock_guard<std::mutex> lk(g_mu);
    out->clear();
    for (auto& d : g_devs) if (!mask || (mask & (1u << d.info.dev))) out->push_back(d.info);
    if (out->empty()) return fail(VMIG_ENOGPU, "gpu_mask 0x%x selects no initialised sm_100 device", mask);
    return VMIG_OK;
}

static std::atomic<long> g_active_lanes{0};     // pipes checked out by calls in flight in this process

// Check out one Pipe per entry of lane_devs (a device may appear several times: lanes_per_gpu).  The
// whole set is reserved in ONE step under the lock -- a call that needs k pipes of one GPU never holds
// some of them while waiting for the rest, so two such calls cannot deadlock each other.  The per-GPU
// cap (VMIG_PIPES_PER_GPU) grows to what a single call asks for.
int ctx_acquire_pipes(const std::vector<DeviceInfo>& lane_devs, std::vector<Pipe*>* out)
{
    out->assign(lane_devs.size(), nullptr);
    std::vector<int> need_dev; std::vector<uint32_t> need_cnt;
    for (auto& d : lane_devs) {
        size_t k = 0; while (k < need_dev.size() && need_dev[k] != d.dev) k++;
        if (k == need_dev.size()) { need_dev.push_back(d.dev); need_cnt.push_back(0); }
        need_cnt[k]++;
    }
    std::vector<uint32_t> to_create(need_dev.size(), 0);
    {
        std::unique_lock<std::mutex> lk(g_mu);
        for (;;) {
            bool ok = true;
            for (size_t k = 0; k < need_dev.size() && ok; k++) {
                DevPool* dp = nullptr;
                for (auto& x : g_devs) if (x.info.dev == need_dev[k]) dp = &x;
                if (!dp) return fail(VMIG_ENOGPU, "device %d not initialised", need_dev[k]);
                const uint32_t cap = std::max(g_pipes_per_gpu, need_cnt[k]);
                const uint32_t room = dp->n_pipes < cap ? cap - dp->n_pipes : 0;
                if (dp->free_pipes.size() + room < need_cnt[k]) ok = false;
            }
            if (ok) break;
            g_cv.wait(lk);
        }
        for (size_t k = 0; k < need_dev.size(); k++) {
            DevPool* dp = nullptr;
            for (auto& x : g_devs) if (x.info.dev == need_dev[k]) dp = &x;
            uint32_t left = need_cnt[k];
            for (size_t i = 0; i < lane_devs.size() && left; i++) {
                if (lane_devs[i].dev != need_dev[k] || (*out)[i]) continue;
                if (dp->free_pipes.empty()) break;
                (*out)[i] = dp->free_pipes.back(); dp->free_pipes.pop_back(); left--;
            }
            to_create[k] = left; dp->n_pipes += left;        // reserved; created outside the lock
        }
    }
    // new pipes of different lanes are created in parallel (each page-locks a 512 MiB OUT ring)
    int rc = VMIG_OK; std::string msg; std::mutex rmu;
    std::vector<std::thread> th;
    for (size_t i = 0; i < lane_devs.size(); i++) {
        if ((*out)[i]) continue;
        th.emplace_back([&, i] {
            Pipe* p = new Pipe();
            int r = p->create(lane_devs[i]);
            if (r) {
                std::lock_guard<std::mutex> lk(rmu);
                if (!rc) { rc = r; msg = last_error_cstr(); }
                p->destroy(); delete p; return;
            }
            (*out)[i] = p;
        });
    }
    for (auto& t : th) t.join();
    if (rc) {
        std::lock_guard<std::mutex> lk(g_mu);
        for (size_t i = 0; i < lane_devs.size(); i++) {
            DevPool* dp = nullptr;
            for (auto& x : g_devs) if (x.info.dev == lane_devs[i].dev) dp = &x;
            if (!dp) continue;
            if ((*out)[i]) { dp->free_pipes.push_back((*out)[i]); (*out)[i] = nullptr; }
            else dp->n_pipes--;
        }
        g_cv.notify_all(); set_last_error_str(msg);
        return rc;
    }
    g_active_lanes += (long)lane_devs.size();
    return VMIG_OK;
}
int ctx_acquire_pipe(const DeviceInfo& d, Pipe** out)
{
    std::vector<Pipe*> v; std::vector<DeviceInfo> one{d};
    int rc = ctx_acquire_pipes(one, &v);
    if (!rc) *out = v[0];
    return rc;
}
void ctx_release_pipe(Pipe* p)
{
    g_active_lanes--;
    std::lock_guard<std::mutex> lk(g_mu);
    for (auto& x : g_devs) if (x.info.dev == p->dev.dev) { x.free_pipes.push_back(p); g_cv.notify_all(); return; }
    p->destroy(); delete p;    // context was shut down underneath us
}

int io_threads_default(uint32_t* readers, uint32_t* writers, uint32_t requested, size_t lanes, size_t n_gpus, bool many_files,
                       bool has_prior, bool hash_only)
{
    long r = env_long("VMIG_READERS", 0), w = env_long("VMIG_WRITERS", 0);
    if (requested) { r = (requested + 1) * 2 / 5; w = requested - r; }
    if (r <= 0 || w <= 0) {
        cpu_set_t cur; CPU_ZERO(&cur);
        long ncpu = sched_getaffinity(0, sizeof cur, &cur) == 0 ? CPU_COUNT(&cur) : sysconf(_SC_NPROCESSORS_ONLN);
        ncpu = env_long("VMIG_PLAN_CPUS", ncpu);                  // test hook: plan as if the box had this many CPUs
        // The host's page-cache copy capacity is a property of the BOX, not of a lane: measured on the 2-socket bench box,
        // ONE GPU is served best by ~20 copy threads in total however many lanes share it (8 readers + 12 writers; 40
        // threads: 12.4 GiB/s instead of 19.3, 96 threads: 8.8 -- profiles/r02_sweep_lanes_1gpu.txt), and eight GPUs by
        // ~13 per GPU (104 in total: 41.8 GiB/s; 64: 39.7, 160: 39.2 -- profiles/r01_e2e_rank_scaling.txt).  So the
        // budget is per GPU in use and is DIVIDED among the lanes that share the box: this call's lanes, the lanes of other
        // calls in flight in this process, and -- one process per GPU, as bench.py under torchrun runs -- whatever
        // VMIG_IO_SHARE says (migrations expected at once).
        const long other = std::max<long>(0, g_active_lanes.load() - (long)lanes);           // lanes of other calls in this process
        const long share = std::max<long>((long)lanes + other, env_long("VMIG_IO_SHARE", 1));
        const long gpus = std::max<long>(1, std::max<long>((long)n_gpus + (other > 0 ? other : 0), env_long("VMIG_IO_SHARE", 1)));
        const long box = std::min<long>(std::max<long>(20, 13 * gpus), std::max<long>(4, ncpu * 7 / 8));
        const long budget = std::max<long>(4, box / share);
        // few large files: the destination serialises per file, extra readers only steal memory
        // bandwidth from the writers; many files: reads are the longer pole
        if (hash_only) {
            // nothing is written: all of the budget reads (pread scales to ~16 threads on the bench box:
            // 28 GiB/s with 8 readers, 43.7 with 16, 34 with 24 -- profiles/r01_e2e_threads.txt)
            if (r <= 0) r = std::max<long>(2, budget * 4 / 5);
            if (w <= 0) w = 1;
        } else if (has_prior) {
            // diff path: every block is read, only the changed ones are written
            if (r <= 0) r = std::max<long>(2, budget * 3 / 5);
            if (w <= 0) w = std::max<long>(2, budget * 3 / 5);
        } else {
            if (r <= 0) r = std::max<long>(2, many_files ? budget / 2 : budget * 2 / 5);
            if (w <= 0) w = std::max<long>(2, budget - r);
        }
    }
    *readers = (uint32_t)std::min<long>(r, 64); *writers = (uint32_t)std::min<long>(w, 64);
    return VMIG_OK;
}

static void bind_thread_complement(const DeviceInfo& d) {
    if (d.cpus.empty()) return;
    cpu_set_t cur, set; CPU_ZERO(&cur); CPU_ZERO(&set);
    // complement within what the PROCESS may use (captured at init), not within this thread's present mask: the thread
    // may already be bound to the GPU's CPUs
    if (g_have_proc_cpus) cur = g_proc_cpus;
    else if (sched_getaffinity(0, sizeof cur, &cur) != 0) return;
    for (int c = 0; c < CPU_SETSIZE; c++) if (CPU_ISSET(c, &cur)) CPU_SET(c, &set);
    for (int c : d.cpus) if (c < CPU_SETSIZE) CPU_CLR(c, &set);
    if (CPU_COUNT(&set) > 0) sched_setaffinity(0, sizeof set, &set);
}

// ---------------------------------------------------------------------------------------------
// blocking queue
template <class T>
class BQ {
    std::mutex mu; std::condition_variable cv; std::deque<T> q; bool closed = false;
public:
    void push(T v) { { std::lock_guard<std::mutex> lk(mu); q.push_back(std::move(v)); } cv.notify_one(); }
    bool pop(T* out) {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return closed || !q.empty(); });
        if (q.empty()) return false;
        *out = std::move(q.front()); q.pop_front(); return true;
    }
    bool try_pop(T* out) {
        std::lock_guard<std::mutex> lk(mu);
        if (q.empty()) return false;
        *out = std::move(q.front()); q.pop_front(); return true;
    }
    void close() { { std::lock_guard<std::mutex> lk(mu); closed = true; } cv.notify_all(); }
};

struct Batch {
    size_t b0 = 0, b1 = 0;          // block range in the lane's list
    size_t bytes_used = 0;          // staged bytes (aligned layout) in the slot
    int slot = -1;
    std::atomic<int> reads_left{0}, writes_left{0};
    bool failed = false;
    std::vector<uint8_t> survive;   // per block, filled after hashing
    uint64_t t_disp = 0, t_read = 0, t_sub = 0, t_hash = 0, t_d2h = 0, t_done = 0;   // VMIG_TRACE
};
struct IoTask { Batch* batch; size_t i0, i1; };

static void bind_thread(const DeviceInfo& d) {
    if (d.cpus.empty()) return;
    cpu_set_t set; CPU_ZERO(&set);
    for (int c : d.cpus) if (c < CPU_SETSIZE) CPU_SET(c, &set);
    sched_setaffinity(0, sizeof set, &set);
}

int run_lane(Pipe* pipe, const std::vector<BlockRef>& blocks, BlockIO* io, bool has_prior, bool hash_only,
             uint32_t n_readers, uint32_t n_writers, uint32_t max_slots, uint64_t* hashes_out, LaneStats* stats,
             std::atomic<int>* err, std::string* err_msg, std::mutex* err_mu)
{
    if (blocks.empty()) return VMIG_OK;
    const uint32_t slot_bytes = pipe->slot_bytes;
    const long fail_block = env_long("VMIG_FAIL_BLOCK", -1);
    const bool bind_io = env_long("VMIG_BIND_IO", 1) != 0;      // reader/writer threads on the GPU's socket
    // writers default to the CPUs of the OTHER socket(s): destination pages then land in that socket's
    // DRAM and the GPU-local socket (the readers' pieces, both DMA directions, the readers) is relieved of a
    // third of the traffic (+15% end to end on the bench box); 1 = GPU-local CPUs, 0 = unbound
    const long bind_wr = env_long("VMIG_BIND_WRITERS", 2);

    auto set_err = [&](int code) {
        int expect = 0;
        if (err->compare_exchange_strong(expect, code)) { std::lock_guard<std::mutex> lk(*err_mu); *err_msg = last_error_cstr(); }
    };

    // ---- plan: pack consecutive blocks into slot-sized batches, 512-B aligned (4 KiB for O_DIRECT backends)
    const uint32_t blk_align = std::max<uint32_t>(kBlockAlign, io->slot_align());
    std::vector<uint32_t> slot_off(blocks.size());
    std::vector<std::unique_ptr<Batch>> batches;
    {
        size_t i = 0;
        while (i < blocks.size()) {
            auto b = std::make_unique<Batch>();
            b->b0 = i; size_t used = 0;
            while (i < blocks.size() && (i - b->b0) < kMaxBatchBlocks) {
                const size_t need = align_up(std::max<uint32_t>(blocks[i].len, 1), blk_align);
                if (need > slot_bytes) { set_last_error("block of %u bytes exceeds the %u-byte staging slot (VMIG_SLOT_MB)", blocks[i].len, slot_bytes); set_err(VMIG_EINVAL); return VMIG_EINVAL; }
                if (used + need > slot_bytes) break;
                slot_off[i] = (uint32_t)used; used += need; i++;
            }
            b->b1 = i; b->bytes_used = used;
            batches.push_back(std::move(b));
        }
    }
    const size_t n_batches = batches.size();

    BQ<int> free_slots;
    const int use_slots = max_slots ? (int)std::min<size_t>(max_slots, pipe->slots.size()) : (int)pipe->slots.size();
    for (int s = 0; s < use_slots; s++) free_slots.push(s);     // one side stream per slot in use
    BQ<IoTask> read_q;
    // Writers.  A destination file takes writes from one thread at a time anyway (inode lock), so two writers on one file
    // only queue up behind each other: writes are queued PER FILE and any idle writer takes the next file that has work and
    // is not being written right now.  (Round 1 pinned file -> writer by `file % n_writers`: the whole-file split hands
    // lane l of L the files l, l+L, ... and they all landed on 1-3 writers -- the in-process multi-GPU collapse, 17.6 GiB/s
    // on 8 GPUs, profiles/r02_lanes_vs_procs_1gpu.txt.  Pinning by rank fixed that but left 10 files on 7 writers with
    // three writers carrying two files while four idled half the time: profiles/r02_lanes_vs_procs_8gpu.txt.)
    std::unordered_map<uint32_t, uint32_t> key_rank;         // write key -> dense rank of first appearance in this lane
    if (!hash_only) {
        key_rank.reserve(256);
        for (const auto& b : blocks) { const uint32_t k = io->write_key(b); key_rank.emplace(k, (uint32_t)(key_rank.size() & 0xFFFFu)); }
    }
    KeyedQueue<IoTask> wsched;      // vmig_sched.h
    wsched.init(std::min<size_t>(std::max<size_t>(key_rank.size(), 1), 0x10000));
    BQ<Batch*> submit_q, hashwait_q, d2hwait_q;
    std::mutex done_mu; std::condition_variable done_cv; size_t batches_done = 0;
    std::mutex stat_mu;

    std::atomic<uint64_t> rd_busy{0}, wr_busy{0}, slot_wait{0}, piece_wait{0};
    const uint64_t lane_t0 = now_ns();
    auto finish_batch = [&](Batch* b) {
        b->t_done = now_ns();
        free_slots.push(b->slot);
        std::lock_guard<std::mutex> lk(done_mu);
        if (++batches_done == n_batches) done_cv.notify_all();
    };
    const bool direct_src = io->pinned_src(blocks[0]) != nullptr;
    const bool direct_dst = !hash_only && io->pinned_dst(blocks[0]) != nullptr;
    // GPUDirect Storage backends: file <-> HBM slot without the pinned rings
    const bool dev_src = !direct_src && io->device_reads();
    const bool dev_dst = !hash_only && !direct_dst && io->device_writes();
    const bool staged_src = !direct_src && !dev_src;       // read into the readers' pinned pieces
    if (staged_src) { int rc = pipe->reserve_readers(n_readers); if (rc) { set_err(rc); return rc; } }
    if (dev_src || dev_dst) {
        cudaSetDevice(pipe->dev.dev);
        for (int s = 0; s < use_slots; s++) {
            Slot& sl = pipe->slots[s];
            if (!sl.cf_registered) { cufile_buf_register(sl.d_buf, (size_t)slot_bytes + kTailPad); sl.cf_registered = true; }
        }
    }

    // ---- stage 1: dispatcher -> read tasks
    std::thread dispatcher([&] {
        bind_thread(pipe->dev);
        for (auto& bp : batches) {
            Batch* b = bp.get();
            int s;
            const uint64_t w0 = now_ns();
            if (!free_slots.pop(&s)) return;
            b->slot = s; b->t_disp = now_ns(); slot_wait += b->t_disp - w0;
            if (direct_src || err->load()) { b->failed = err->load() != 0; submit_q.push(b); continue; }
            // group small blocks so a task carries >= 1 MiB or 64 blocks
            std::vector<IoTask> tasks;
            size_t i = b->b0;
            while (i < b->b1) {
                size_t j = i, bytes = 0;
                while (j < b->b1 && (j - i) < 64 && bytes < (1u << 20)) { bytes += blocks[j].len; j++; }
                tasks.push_back({b, i, j}); i = j;
            }
            b->reads_left.store((int)tasks.size());
            for (auto& t : tasks) read_q.push(t);
        }
    });

    // ---- stage 2: readers.  Reader t stages the slot window by window (vmig_common.h block_piece): it reads the parts of
    // a task's blocks that fall in one window into one of its kPieces pieces, copies the filled range into the HBM slot on
    // its own stream and records the piece's event.  A piece is refilled, and a task counts as read (so that its batch may
    // be hashed, or its slot handed out again after an error), only once the copies out of it have completed.  The stream
    // runs its copies in order, so one completed event vouches for every copy issued before it.  Two tasks never copy the
    // same slot bytes: a copy spans the blocks' bytes only, never past the last one.
    std::vector<std::thread> readers;
    for (uint32_t t = 0; t < n_readers; t++)
        readers.emplace_back([&, t] {
            if (bind_io) bind_thread(pipe->dev);
            if (dev_src || staged_src) cudaSetDevice(pipe->dev.dev);
            auto task_read = [&](Batch* b) { if (b->reads_left.fetch_sub(1) == 1) { b->t_read = now_ns(); submit_q.push(b); } };
            PieceReader* pr = staged_src ? &pipe->readers[t] : nullptr;
            uint8_t* const pbase = staged_src ? pipe->pieces + (size_t)t * kPieces * kPieceBytes : nullptr;
            uint64_t piece_seq[kPieces] = {};       // sequence number of the last copy out of each piece
            uint64_t issued = 0, done = 0;          // copies issued / known complete
            std::deque<std::pair<Batch*, uint64_t>> pending;     // tasks read, and the copy that completes each
            // the window being filled: slot window `win` of d_win, held in piece issued % kPieces, bytes [lo, hi) filled
            uint8_t* d_win = nullptr; size_t win = 0, lo = 0, hi = 0;
            auto reap = [&] {
                while (!pending.empty() && pending.front().second <= done) { task_read(pending.front().first); pending.pop_front(); }
            };
            // wait until copy number `seq` has completed.  Polled: a blocking wait's wake-up left readers waiting for
            // pieces 25-66 % of their time, polling 7-14 % (profiles/r03_piece_variants.txt)
            auto wait_copy = [&](uint64_t seq) -> int {
                if (seq <= done) return VMIG_OK;
                const uint64_t w0 = now_ns();
                cudaError_t e;
                while ((e = cudaEventQuery(pr->ev[(seq - 1) % kPieces])) == cudaErrorNotReady) {}
                piece_wait += now_ns() - w0;
                if (e != cudaSuccess) { cudaGetLastError(); return fail(VMIG_ECUDA, "cudaEventQuery(piece): %s", cudaGetErrorString(e)); }
                done = seq;
                return VMIG_OK;
            };
            // every copy of this reader has completed: after an error, before idling and before exiting
            auto drain = [&] {
                if (!staged_src) return;
                d_win = nullptr;
                if (int rc = wait_copy(issued)) {
                    set_err(rc);
                    cudaStreamSynchronize(pr->stream); cudaGetLastError(); done = issued;
                }
                reap();
            };
            auto flush = [&]() -> int {
                if (!d_win) return VMIG_OK;
                const uint32_t p = (uint32_t)(issued % kPieces);
                uint8_t* const d = d_win; d_win = nullptr;
                CU_API(cudaMemcpyAsync(d + win * kPieceBytes + lo, pbase + (size_t)p * kPieceBytes + lo, hi - lo, cudaMemcpyHostToDevice, pr->stream));
                CU_API(cudaEventRecord(pr->ev[p], pr->stream));
                piece_seq[p] = ++issued;
                return VMIG_OK;
            };
            auto read_part = [&](size_t i, const Piece& pc, uint8_t* d_buf) -> int {
                if (!pc.len) return io->read_block(blocks[i], pc.off, pc.len, pbase);
                if (d_win && (d_win != d_buf || win != pc.window)) { if (int rc = flush()) return rc; }
                if (!d_win) {
                    // the newest copy is usually done already: one query reaps every task it completes
                    if (issued > done && cudaEventQuery(pr->ev[(issued - 1) % kPieces]) == cudaSuccess) { done = issued; reap(); }
                    if (int rc = wait_copy(piece_seq[issued % kPieces])) return rc;
                    reap();
                    d_win = d_buf; win = pc.window; lo = kPieceBytes; hi = 0;
                }
                const size_t at = slot_off[i] + pc.off - win * kPieceBytes;
                if (int rc = io->read_block(blocks[i], pc.off, pc.len, pbase + (size_t)(issued % kPieces) * kPieceBytes + at)) return rc;
                lo = std::min(lo, at); hi = std::max(hi, at + pc.len);
                return VMIG_OK;
            };
            IoTask k;
            for (;;) {
                if (!read_q.try_pop(&k)) { drain(); if (!read_q.pop(&k)) break; }
                if (err->load()) drain();
                const uint64_t r0 = now_ns();
                if (!err->load()) {
                    uint8_t* const d_buf = pipe->slots[k.batch->slot].d_buf;
                    int rc = VMIG_OK;
                    for (size_t i = k.i0; i < k.i1 && !rc; i++) {
                        if (dev_src) { rc = io->read_block_dev(blocks[i], d_buf, slot_off[i]); continue; }
                        for (size_t j = 0, np = piece_count(slot_off[i], blocks[i].len, kPieceBytes); j < np && !rc; j++)
                            rc = read_part(i, block_piece(slot_off[i], blocks[i].len, kPieceBytes, 0, j), d_buf);
                    }
                    if (!rc && staged_src) rc = flush();
                    if (rc) set_err(rc);
                }
                rd_busy += now_ns() - r0;
                if (!staged_src) { task_read(k.batch); continue; }
                pending.emplace_back(k.batch, issued);
                if (err->load()) drain(); else reap();
            }
            drain();
        });

    // ---- stage 3: submit H2D + kernel (+ D2H) on the slot's side stream
    auto submit_one = [&](Batch* b) -> int {
        Slot& sl = pipe->slots[b->slot];
        const uint32_t n = (uint32_t)(b->b1 - b->b0);
        uint64_t* h_offs = (uint64_t*)sl.h_desc; uint64_t* h_prior = h_offs + n;
        uint32_t* h_lens = (uint32_t*)(h_prior + n); uint8_t* h_valid = (uint8_t*)(h_lens + n);
        for (uint32_t i = 0; i < n; i++) {
            const BlockRef& r = blocks[b->b0 + i];
            h_offs[i] = slot_off[b->b0 + i]; h_prior[i] = r.prior_hash; h_lens[i] = r.len; h_valid[i] = r.prior_valid;
        }
        const size_t desc_bytes = (size_t)n * 21;
        CU_API(cudaMemcpyAsync(sl.d_desc, sl.h_desc, desc_bytes, cudaMemcpyHostToDevice, sl.stream));
        uint64_t h2d = 0;
        if (direct_src) {
            for (uint32_t i = 0; i < n; i++) {
                const BlockRef& r = blocks[b->b0 + i];
                if (!r.len) continue;
                CU_API(cudaMemcpyAsync(sl.d_buf + slot_off[b->b0 + i], io->pinned_src(r), r.len, cudaMemcpyHostToDevice, sl.stream));
                h2d += r.len;
            }
        } else {
            // the reader threads already put the bytes into the HBM slot
            for (uint32_t i = 0; i < n; i++) h2d += blocks[b->b0 + i].len;
        }
        HashLaunch a;
        a.base = sl.d_buf; a.offs = (const uint64_t*)sl.d_desc; a.prior = a.offs + n;
        a.lens = (const uint32_t*)(a.prior + n); a.prior_valid = (const uint8_t*)(a.lens + n);
        a.n = n; a.hashes = (uint64_t*)sl.d_res; a.changed = (uint8_t*)(a.hashes + n);
        a.work_counter = sl.d_counter;
        if (!has_prior) { a.prior = nullptr; a.prior_valid = nullptr; }
        CU_API(cudaEventRecord(sl.ev_k0, sl.stream));
        CU_API(launch_xxh64_blocks(a, pipe->dev.sm_count, sl.stream));
        CU_API(cudaEventRecord(sl.ev_k1, sl.stream));
        CU_API(cudaMemcpyAsync(sl.h_res, sl.d_res, (size_t)n * 9, cudaMemcpyDeviceToHost, sl.stream));
        CU_API(cudaEventRecord(sl.ev_hash, sl.stream));
        uint64_t d2h = 0;
        if (!has_prior && !hash_only && !dev_dst) {       // every block survives: stream it back right away
            if (direct_dst) {
                for (uint32_t i = 0; i < n; i++) {
                    const BlockRef& r = blocks[b->b0 + i];
                    if (!r.len) continue;
                    CU_API(cudaMemcpyAsync(io->pinned_dst(r), sl.d_buf + slot_off[b->b0 + i], r.len, cudaMemcpyDeviceToHost, sl.stream));
                    d2h += r.len;
                }
            } else {
                CU_API(cudaMemcpyAsync(sl.h_out, sl.d_buf, b->bytes_used, cudaMemcpyDeviceToHost, sl.stream));
                d2h = h2d;
            }
            CU_API(cudaEventRecord(sl.ev_d2h, sl.stream));
        }
        std::lock_guard<std::mutex> lk(stat_mu);
        stats->bytes_h2d += h2d; stats->bytes_d2h += d2h; stats->kernel_launches += 1;
        return VMIG_OK;
    };
    std::thread submitter([&] {
        bind_thread(pipe->dev);
        cudaSetDevice(pipe->dev.dev);
        Batch* b;
        while (submit_q.pop(&b)) {
            if (err->load()) b->failed = true;
            if (!b->failed) { int rc = submit_one(b); if (rc) { set_err(rc); b->failed = true; } }
            b->t_sub = now_ns();
            hashwait_q.push(b);
        }
    });

    // ---- stage 4: wait for hashes, pick survivors, issue their D2H
    auto after_hash = [&](Batch* b) -> int {
        Slot& sl = pipe->slots[b->slot];
        const uint32_t n = (uint32_t)(b->b1 - b->b0);
        CU_API(cudaEventSynchronize(sl.ev_hash));
        float ms = 0; CU_API(cudaEventElapsedTime(&ms, sl.ev_k0, sl.ev_k1));
        const uint64_t* h_hash = (const uint64_t*)sl.h_res; const uint8_t* h_changed = (const uint8_t*)(h_hash + n);
        b->survive.assign(n, 1);
        uint64_t skipped = 0, d2h = 0;
        for (uint32_t i = 0; i < n; i++) {
            const BlockRef& r = blocks[b->b0 + i];
            hashes_out[r.table_idx] = h_hash[i];
            if (fail_block >= 0 && (uint64_t)fail_block == r.table_idx) return fail(VMIG_EFAULT, "injected fault at block %ld (VMIG_FAIL_BLOCK)", fail_block);
            if (has_prior && !h_changed[i]) { b->survive[i] = 0; skipped++; }
        }
        if (dev_dst) {
            for (uint32_t i = 0; i < n; i++) if (b->survive[i]) d2h += blocks[b->b0 + i].len;      // drained by the writers straight from HBM
        } else if (has_prior && !hash_only) {
            uint32_t i = 0;
            while (i < n) {      // coalesce runs of adjacent survivors into one DMA
                if (!b->survive[i] || !blocks[b->b0 + i].len) { i++; continue; }
                if (direct_dst) {
                    const BlockRef& r = blocks[b->b0 + i];
                    CU_API(cudaMemcpyAsync(io->pinned_dst(r), sl.d_buf + slot_off[b->b0 + i], r.len, cudaMemcpyDeviceToHost, sl.stream));
                    d2h += r.len; i++; continue;
                }
                uint32_t j = i; size_t start = slot_off[b->b0 + i], end = start;
                while (j < n && b->survive[j]) { end = slot_off[b->b0 + j] + blocks[b->b0 + j].len; d2h += blocks[b->b0 + j].len; j++; }
                CU_API(cudaMemcpyAsync(sl.h_out + start, sl.d_buf + start, end - start, cudaMemcpyDeviceToHost, sl.stream));
                i = j;
            }
            CU_API(cudaEventRecord(sl.ev_d2h, sl.stream));
        }
        std::lock_guard<std::mutex> lk(stat_mu);
        stats->ms_kernel += ms; stats->blocks_skipped += skipped; stats->bytes_d2h += d2h;
        return VMIG_OK;
    };
    std::thread hashwaiter([&] {
        bind_thread(pipe->dev);
        cudaSetDevice(pipe->dev.dev);
        Batch* b;
        while (hashwait_q.pop(&b)) {
            if (err->load()) b->failed = true;
            if (!b->failed) { int rc = after_hash(b); if (rc) { set_err(rc); b->failed = true; } }
            if (b->failed) b->survive.assign(b->b1 - b->b0, 0);
            b->t_hash = now_ns();
            d2hwait_q.push(b);
        }
    });

    // ---- stage 5: wait for the survivors' D2H, hand them to the writers
    std::thread d2hwaiter([&] {
        bind_thread(pipe->dev);
        cudaSetDevice(pipe->dev.dev);
        Batch* b;
        while (d2hwait_q.pop(&b)) {
            Slot& sl = pipe->slots[b->slot];
            if (!b->failed && !hash_only && !dev_dst) {
                cudaError_t e = cudaEventSynchronize(sl.ev_d2h);
                if (e != cudaSuccess) { fail(VMIG_ECUDA, "cudaEventSynchronize(d2h): %s", cudaGetErrorString(e)); set_err(VMIG_ECUDA); b->failed = true; }
            }
            const size_t n = b->b1 - b->b0;
            b->t_d2h = now_ns();
            std::vector<IoTask> tasks;
            if (!b->failed && !hash_only && !direct_dst) {
                size_t i = 0;
                while (i < n) {
                    if (!b->survive[i]) { i++; continue; }
                    size_t j = i, bytes = 0;
                    while (j < n && b->survive[j] && (j - i) < 64 && bytes < (1u << 20)) { bytes += blocks[b->b0 + j].len; j++; }
                    tasks.push_back({b, b->b0 + i, b->b0 + j}); i = j;
                }
            }
            // blocks that need no write are complete now
            for (size_t i = 0; i < n; i++) {
                const bool written_later = !tasks.empty() && b->survive[i];
                if (!written_later) {
                    const bool was_written = !b->failed && !hash_only && direct_dst && b->survive[i];
                    if (b->failed) continue;            // do not finalize files of a failed call
                    int rc = io->block_done(blocks[b->b0 + i], was_written);
                    if (rc) set_err(rc);
                    if (was_written) { std::lock_guard<std::mutex> lk(stat_mu); stats->bytes_written += blocks[b->b0 + i].len; }
                }
            }
            if (tasks.empty()) { finish_batch(b); continue; }
            b->writes_left.store((int)tasks.size());
            for (auto& t : tasks) wsched.push(key_rank[io->write_key(blocks[t.i0])], t);
        }
    });

    // ---- stage 6: writers
    std::vector<std::thread> writers;
    for (uint32_t t = 0; t < n_writers; t++)
        writers.emplace_back([&] {
            if (bind_io && bind_wr == 1) bind_thread(pipe->dev);
            else if (bind_io && bind_wr == 2) bind_thread_complement(pipe->dev);
            if (dev_dst) cudaSetDevice(pipe->dev.dev);
            IoTask k; uint32_t krank = 0;
            while (wsched.pop(&krank, &k)) {
                Slot& sl = pipe->slots[k.batch->slot];
                uint64_t wrote = 0;
                const uint64_t w0 = now_ns();
                for (size_t i = k.i0; i < k.i1; i++) {
                    if (err->load()) break;
                    int rc = dev_dst ? io->write_block_dev(blocks[i], sl.d_buf, slot_off[i]) : io->write_block(blocks[i], sl.h_out + slot_off[i]);
                    if (!rc) { wrote += blocks[i].len; rc = io->block_done(blocks[i], true); }
                    if (rc) { set_err(rc); break; }
                }
                wr_busy += now_ns() - w0;
                wsched.done(krank);
                { std::lock_guard<std::mutex> lk(stat_mu); stats->bytes_written += wrote; }
                if (k.batch->writes_left.fetch_sub(1) == 1) finish_batch(k.batch);
            }
        });

    {
        std::unique_lock<std::mutex> lk(done_mu);
        done_cv.wait(lk, [&] { return batches_done == n_batches; });
    }
    read_q.close(); submit_q.close(); hashwait_q.close(); d2hwait_q.close(); free_slots.close();
    wsched.close();
    dispatcher.join();
    for (auto& t : readers) t.join();
    submitter.join(); hashwaiter.join(); d2hwaiter.join();
    for (auto& t : writers) t.join();
    if (env_long("VMIG_TRACE", 0)) {
        const double wall = (now_ns() - lane_t0) / 1e6;
        double a[5] = {0, 0, 0, 0, 0}; size_t nb = 0;
        for (auto& bp : batches) {
            const Batch& b = *bp;
            if (!b.t_done || !b.t_disp) continue;
            a[0] += (b.t_read ? b.t_read - b.t_disp : 0) / 1e6; a[1] += (b.t_sub - std::max(b.t_read, b.t_disp)) / 1e6;
            a[2] += (b.t_hash - b.t_sub) / 1e6; a[3] += (b.t_d2h - b.t_hash) / 1e6; a[4] += (b.t_done - b.t_d2h) / 1e6; nb++;
        }
        fprintf(stderr, "[vmig trace] gpu %d: %zu batches in %.1f ms; mean ms/batch: read %.2f submit-wait %.2f h2d+hash %.2f d2h %.2f write %.2f; "
                        "reader busy %.0f%% of %u, writer busy %.0f%% of %u; dispatcher waited %.1f ms for slots; kernel sum %.1f ms; "
                        "readers waited %.1f ms for pieces\n",
                pipe->dev.dev, nb, wall, a[0] / nb, a[1] / nb, a[2] / nb, a[3] / nb, a[4] / nb,
                100.0 * rd_busy.load() / 1e6 / (wall * n_readers), n_readers, 100.0 * wr_busy.load() / 1e6 / (wall * n_writers), n_writers,
                slot_wait.load() / 1e6, stats->ms_kernel, piece_wait.load() / 1e6);
    }
    // the slots go back to the pool idle
    cudaSetDevice(pipe->dev.dev);
    for (auto& s : pipe->slots) cudaStreamSynchronize(s.stream);
    for (auto& r : pipe->readers) cudaStreamSynchronize(r.stream);
    return err->load();
}

}  // namespace vmig
