// vmig_api.cu -- the C ABI of libvmig (include/vmig.h): tree migration, buffer migration, direct
// block hashing, the HBM-resident batch, and the host-side helpers.
//
// Reference seam (SURVEY.md §8b): utils.CopyDir (utils/copy.go:21-27), moveVolumeData
// (utils/copy.go:74-128), utils.DirSize / utils.ToBytes (utils/file.go:13-48).
#include "vmig_engine.h"
#include "vmig_kernels.cuh"
#include "vmig_tree.h"
#include "vmig_table.h"
#include "vmig_cufile.h"

#include <fcntl.h>
#include <unistd.h>
#include <sys/stat.h>
#include <algorithm>
#include <unordered_map>
#include <thread>
#include <cmath>

using namespace vmig;

namespace {

inline std::string pjoin(const std::string& a, const std::string& b) { return b == "." ? a : a + "/" + b; }

inline int64_t ctime_ns(const struct stat& st) { return (int64_t)st.st_ctim.tv_sec * 1000000000ll + st.st_ctim.tv_nsec; }

// Opens destination file p for writing, O_DIRECT if *direct; *direct then says whether O_DIRECT took.  create: a new
// file, replacing what is there like tar does (a directory in the way is an error); else the existing file.  A
// filesystem that refuses O_DIRECT (EINVAL) gets the same open without it, and without O_EXCL: the refused attempt may
// already have created the file.
int open_for_write(const std::string& p, bool create, bool* direct, int* out)
{
    if (create) {
        bool was_dir = false;
        int rc = unlink_if_exists(p, &was_dir);
        if (rc) return rc;
        if (was_dir) return fail(VMIG_EIO, "%s: a directory is in the way of a regular file", p.c_str());
    }
    const int flags = O_WRONLY | O_CLOEXEC | O_NOFOLLOW | (create ? O_CREAT | O_EXCL : 0);
    const bool want = *direct;
    *out = open(p.c_str(), flags | (want ? O_DIRECT : 0), 0600);
    *direct = want && *out >= 0;
    if (*out < 0 && want && errno == EINVAL) *out = open(p.c_str(), flags & ~O_EXCL, 0600);
    if (*out < 0) return fail(VMIG_EIO, "open %s for writing: %s", p.c_str(), errno_str(errno).c_str());
    return VMIG_OK;
}

// ---------------------------------------------------------------------------------------------
// file-backed BlockIO
class FileIO : public BlockIO {
public:
    struct FS {
        std::atomic<int> sfd{-1}, dfd{-1};
        std::atomic<uint32_t> reads_left{0}, blocks_left{0};
        bool inplace = false;            // diff path: destination file is the prior version, patched in place
        uint64_t dst_old_size = 0;
        uint64_t id_ino = 0; int64_t id_ctime_ns = 0;   // identity of the file the table will speak for (vmig_table.h)
        bool s_direct = false, d_direct = false;         // this file's descriptor was opened with O_DIRECT
        std::atomic<void*> s_cfh{nullptr}, d_cfh{nullptr};   // cuFile handles of sfd / dfd (VMIG_F_CUFILE)
        std::atomic<bool> wrote{false};                  // at least one block of the file was written in this call
        void set_identity(const struct stat& st) { id_ino = (uint64_t)st.st_ino; id_ctime_ns = ctime_ns(st); }
    };
    std::string src_root, dst_root;
    int src_root_fd = -1;                // source files are opened beneath this descriptor, never by absolute path
    const Manifest* m = nullptr;
    MetaPolicy pol;
    bool hash_only = false;
    bool direct = false;                 // VMIG_F_DIRECT_IO: O_DIRECT into / out of the pinned rings
    bool cufile = false;                 // VMIG_F_CUFILE: file <-> HBM slot through libcufile (GPUDirect Storage)
    std::atomic<uint64_t> n_direct{0};   // descriptors that really were opened O_DIRECT
    static constexpr uint32_t kSector = 4096;
    uint32_t slot_align() override { return direct || cufile ? kSector : 512; }
    bool device_reads() override { return cufile; }
    bool device_writes() override { return cufile && !hash_only; }
    long corrupt_block = -1;             // VMIG_CORRUPT_BLOCK test hook: flip one bit of this block on its way to disk
    std::unique_ptr<FS[]> fs;
    std::mutex stripes[64];

    // One pass over man's files, reading them beneath `root`: every file with blocks of its own is opened at its first
    // block and closed after its last.
    int setup(const std::string& root, const Manifest& man) {
        src_root = root; m = &man;
        fs.reset(new FS[man.files.size() ? man.files.size() : 1]);
        for (size_t f = 0; f < man.files.size(); f++) {
            const Entry& e = man.files[f];
            if (e.hardlink_of >= 0 || e.n_blocks == 0) continue;
            fs[f].reads_left.store((uint32_t)e.n_blocks); fs[f].blocks_left.store((uint32_t)e.n_blocks);
        }
        if (cufile) { int rc = cufile_open(); if (rc) return rc; }
        src_root_fd = open(src_root.c_str(), O_RDONLY | O_DIRECTORY | O_CLOEXEC);
        if (src_root_fd < 0) return fail(VMIG_EIO, "open %s: %s", src_root.c_str(), errno_str(errno).c_str());
        return VMIG_OK;
    }
    ~FileIO() { close_all(); if (src_root_fd >= 0) close(src_root_fd); }

    // Swaps *fd for a descriptor registered with libcufile, whose handle goes to h; *fd is closed on failure.
    // libcufile refuses descriptors whose open flags include O_NOFOLLOW / O_NONBLOCK ("unsupported file open flags"),
    // which is exactly how the safe opens below are made, and F_SETFL cannot clear O_NOFOLLOW.  The descriptor already
    // refers to the checked regular file, so it is re-opened through /proc/self/fd with plain flags.
    static int cufile_attach(int* fd, int flags, const std::string& name, std::atomic<void*>& h) {
        char path[64]; snprintf(path, sizeof path, "/proc/self/fd/%d", *fd);
        const int nfd = open(path, flags | O_CLOEXEC);
        if (nfd < 0) { const int e = errno; close(*fd); return fail(VMIG_EIO, "reopen %s for cuFile: %s", name.c_str(), errno_str(e).c_str()); }
        close(*fd); *fd = nfd;
        void* handle = nullptr;
        const int rc = cufile_handle_open(nfd, &handle);
        if (rc) { close(nfd); return rc; }
        h.store(handle, std::memory_order_release);
        return VMIG_OK;
    }
    int open_src(uint32_t f, int* out) {
        FS& s = fs[f];
        int fd = s.sfd.load(std::memory_order_acquire);
        if (fd < 0) {
            std::lock_guard<std::mutex> lk(stripes[f & 63]);
            fd = s.sfd.load(std::memory_order_acquire);
            if (fd < 0) {
                // the tenant may still be running on this layer: no symlink is followed and the root is never
                // left (vmig_tree.h open_beneath); O_NONBLOCK so a FIFO swapped in cannot park a reader thread
                int rc = VMIG_EIO;
                if (direct) { rc = open_beneath(src_root_fd, m->files[f].rel, O_RDONLY | O_NONBLOCK | O_DIRECT, &fd); s.s_direct = rc == VMIG_OK; }
                if (rc) rc = open_beneath(src_root_fd, m->files[f].rel, O_RDONLY | O_NONBLOCK, &fd);     // the filesystem may refuse O_DIRECT
                if (rc) return rc;
                struct stat st;
                if (fstat(fd, &st) != 0 || !S_ISREG(st.st_mode)) {
                    close(fd);
                    return fail(VMIG_ESRCCHANGED, "%s is not a regular file any more", m->files[f].rel.c_str());
                }
                if (hash_only && st.st_nlink == 1) s.set_identity(st);
                if (s.s_direct) n_direct++;
                if (cufile) { rc = cufile_attach(&fd, O_RDONLY | (s.s_direct ? O_DIRECT : 0), m->files[f].rel, s.s_cfh); if (rc) return rc; }
                s.sfd.store(fd, std::memory_order_release);
            }
        }
        *out = fd; return VMIG_OK;
    }
    int open_dst(uint32_t f, int* out) {
        FS& s = fs[f];
        int fd = s.dfd.load(std::memory_order_acquire);
        if (fd < 0) {
            std::lock_guard<std::mutex> lk(stripes[f & 63]);
            fd = s.dfd.load(std::memory_order_acquire);
            if (fd < 0) {
                const std::string p = pjoin(dst_root, m->files[f].rel);
                bool dio = direct && corrupt_block < 0;       // the fault hook's one-byte pwrite cannot be O_DIRECT
                int rc = open_for_write(p, !s.inplace, &dio, &fd);
                if (rc) return rc;
                s.d_direct = dio;
                if (dio) n_direct++;
                if (cufile && !hash_only) { rc = cufile_attach(&fd, O_WRONLY | (dio ? O_DIRECT : 0), p, s.d_cfh); if (rc) return rc; }
                s.dfd.store(fd, std::memory_order_release);
            }
        }
        *out = fd; return VMIG_OK;
    }
    // O_DIRECT: buffer, offset and length in whole sectors (pieces are whole sectors; the device DMAs straight into the
    // reader's pinned piece).  The source is closed after the last piece of its last block.
    int read_block(const BlockRef& b, size_t off, size_t len, uint8_t* dst) override {
        int fd; int rc = open_src(b.file, &fd);
        if (rc) return rc;
        FS& s = fs[b.file];
        const char* name = m->files[b.file].rel.c_str();
        const uint64_t at = b.file_off + off;
        rc = transfer_block(name, at, len, s.s_direct ? kSector : 0, VMIG_ESRCCHANGED, [&](size_t pos, size_t n) -> ssize_t {
            ssize_t r;
            while ((r = pread(fd, dst + pos, n, (off_t)(at + pos))) < 0 && errno == EINTR) {}
            return r < 0 ? fail(VMIG_EIO, "pread %s: %s", name, errno_str(errno).c_str()) : r;
        });
        if (!rc && off + len == b.len && s.reads_left.fetch_sub(1) == 1) close_src(s, fd);
        return rc;
    }
    void close_src(FS& s, int fd) {
        void* h = s.s_cfh.exchange(nullptr);
        if (h) cufile_handle_close(h);
        close(fd); s.sfd.store(-1);
    }
    // GPUDirect Storage: file -> HBM slot
    int read_block_dev(const BlockRef& b, uint8_t* d_base, size_t d_off) override {
        int fd; int rc = open_src(b.file, &fd);
        if (rc) return rc;
        FS& s = fs[b.file];
        void* h = s.s_cfh.load(std::memory_order_acquire);
        rc = transfer_block(m->files[b.file].rel.c_str(), b.file_off, b.len, s.s_direct ? kSector : 0, VMIG_ESRCCHANGED, [&](size_t pos, size_t n) {
            return cufile_read(h, d_base, n, (off_t)(b.file_off + pos), (off_t)(d_off + pos));
        });
        if (!rc && s.reads_left.fetch_sub(1) == 1) close_src(s, fd);
        return rc;
    }
    // GPUDirect Storage: HBM slot -> file (surviving blocks only)
    int write_block_dev(const BlockRef& b, const uint8_t* d_base, size_t d_off) override {
        int fd; int rc = open_dst(b.file, &fd);
        if (rc) return rc;
        FS& s = fs[b.file];
        s.wrote.store(true, std::memory_order_relaxed);
        void* h = s.d_cfh.load(std::memory_order_acquire);
        return transfer_block(m->files[b.file].rel.c_str(), b.file_off, b.len, s.d_direct ? kSector : 0, VMIG_EIO, [&](size_t pos, size_t n) {
            return cufile_write(h, d_base, n, (off_t)(b.file_off + pos), (off_t)(d_off + pos));
        });
    }
    // O_DIRECT: whole sectors out of the pinned ring; a short last block is written padded (whatever follows it in the
    // slot) and block_done() cuts the file back to its size
    int write_block(const BlockRef& b, const uint8_t* src) override {
        int fd; int rc = open_dst(b.file, &fd);
        if (rc) return rc;
        FS& s = fs[b.file];
        s.wrote.store(true, std::memory_order_relaxed);
        const char* name = m->files[b.file].rel.c_str();
        rc = transfer_block(name, b.file_off, b.len, s.d_direct ? kSector : 0, VMIG_EIO, [&](size_t pos, size_t n) -> ssize_t {
            ssize_t w;
            while ((w = pwrite(fd, src + pos, n, (off_t)(b.file_off + pos))) < 0 && errno == EINTR) {}
            return w < 0 ? fail(VMIG_EIO, "pwrite %s: %s", name, errno_str(errno).c_str()) : w;
        });
        if (rc || corrupt_block < 0 || (uint64_t)corrupt_block != b.table_idx || !b.len) return rc;
        const uint8_t bad = src[0] ^ 1u;           // what VMIG_F_VERIFY exists to catch
        return pwrite(fd, &bad, 1, (off_t)b.file_off) == 1 ? VMIG_OK : fail(VMIG_EIO, "pwrite (fault hook)");
    }
    int block_done(const BlockRef& b, bool) override {
        FS& s = fs[b.file];
        if (s.blocks_left.fetch_sub(1) != 1) return VMIG_OK;
        if (hash_only) return VMIG_OK;
        const Entry& e = m->files[b.file];
        int fd; int rc = open_dst(b.file, &fd);      // also covers "every block was skipped"
        if (rc) return rc;
        const std::string p = pjoin(dst_root, e.rel);
        if (((s.inplace && s.dst_old_size != e.size) || (s.d_direct && (e.size & (kSector - 1)))) && ftruncate(fd, (off_t)e.size) != 0) {
            close(fd); return fail(VMIG_EIO, "ftruncate %s: %s", p.c_str(), errno_str(errno).c_str());
        }
        // a patched-in-place file none of whose blocks changed and whose metadata is already right is not touched at all:
        // its ctime -- by which the block table knows it -- stays what the table recorded
        const bool untouched = s.inplace && !s.wrote.load() && s.dst_old_size == e.size && file_meta_matches(fd, e, pol);
        rc = untouched ? VMIG_OK : apply_file_meta(fd, p, e, pol);
        struct stat ids;                             // nothing touches the file after this point: its ctime is final
        if (!rc && fstat(fd, &ids) == 0) s.set_identity(ids);
        { void* h = s.d_cfh.exchange(nullptr); if (h) cufile_handle_close(h); }
        if (close(fd) != 0 && !rc) rc = fail(VMIG_EIO, "close %s: %s", p.c_str(), errno_str(errno).c_str());
        s.dfd.store(-1);
        return rc;
    }
    void close_all() {
        for (size_t i = 0; fs && i < m->files.size(); i++) {
            void* h = fs[i].s_cfh.exchange(nullptr); if (h) cufile_handle_close(h);
            h = fs[i].d_cfh.exchange(nullptr); if (h) cufile_handle_close(h);
            int a = fs[i].sfd.exchange(-1); if (a >= 0) close(a);
            int b = fs[i].dfd.exchange(-1); if (b >= 0) close(b);
        }
    }
};

// ---------------------------------------------------------------------------------------------
// memory-backed BlockIO (vmig_migrate_buffer, vmig_hash_blocks)
class MemIO : public BlockIO {
public:
    const uint8_t* src = nullptr; uint8_t* dst = nullptr;
    bool src_pinned = false, dst_pinned = false;
    int read_block(const BlockRef& b, size_t off, size_t len, uint8_t* d) override { if (len) memcpy(d, src + b.file_off + off, len); return VMIG_OK; }
    int write_block(const BlockRef& b, const uint8_t* s) override { if (b.len) memcpy(dst + b.file_off, s, b.len); return VMIG_OK; }
    uint32_t write_key(const BlockRef& b) override { return (uint32_t)b.table_idx; }
    const uint8_t* pinned_src(const BlockRef& b) override { return src_pinned ? src + b.file_off : nullptr; }
    uint8_t* pinned_dst(const BlockRef& b) override { return dst_pinned ? dst + b.file_off : nullptr; }
};

bool is_pinned(const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// ---------------------------------------------------------------------------------------------
// run a block list over the selected GPUs: n_gpus x lanes_per_gpu lanes, whole files per lane (LPT by bytes);
// contiguous byte-balanced ranges only when there are fewer than two files per lane
int run_blocks(const std::vector<BlockRef>& blocks, BlockIO* io, bool has_prior, bool hash_only, const vmig_opts& o,
               uint64_t* hashes, vmig_stats* st)
{
    std::vector<DeviceInfo> devs;
    int rc = ctx_select(o.gpu_mask, &devs);
    if (rc) return rc;
    if (blocks.empty()) { st->gpus_used = 0; return VMIG_OK; }
    // lanes: one per GPU of the mask, times lanes_per_gpu (lane i runs on GPU i % n_gpus); the split below
    // does not care whether two lanes share a device
    uint32_t lpg = o.lanes_per_gpu ? o.lanes_per_gpu : (uint32_t)std::max<long>(1, env_long("VMIG_LANES_PER_GPU", 1));
    if (lpg > 16) lpg = 16;
    const size_t n_gpus = devs.size();
    size_t lanes = std::min(n_gpus * lpg, blocks.size());
    std::vector<DeviceInfo> lane_devs(lanes);
    for (size_t i = 0; i < lanes; i++) lane_devs[i] = devs[i % n_gpus];
    uint64_t total = 0;
    for (auto& b : blocks) total += std::max<uint32_t>(b.len, 4096);
    std::vector<std::vector<BlockRef>> share(lanes);
    if (lanes == 1) {
        share[0] = blocks;
    } else {
        // Prefer giving each GPU whole files (write keys): two lanes writing one destination file
        // would queue on its inode lock.  Longest-processing-time packing of the keys by bytes; the
        // interleaved block order is kept inside every lane.  With fewer keys than GPUs (one huge
        // file) the list is cut into contiguous byte-balanced ranges instead.
        std::unordered_map<uint32_t, uint64_t> key_bytes;
        for (auto& b : blocks) key_bytes[io->write_key(b)] += std::max<uint32_t>(b.len, 4096);
        if (key_bytes.size() >= 2 * lanes) {
            std::vector<std::pair<uint64_t, uint32_t>> keys;
            for (auto& kv : key_bytes) keys.push_back({kv.second, kv.first});
            std::sort(keys.begin(), keys.end(), [](auto& a, auto& b) { return a.first != b.first ? a.first > b.first : a.second < b.second; });
            std::vector<uint64_t> load(lanes, 0);
            std::unordered_map<uint32_t, uint32_t> key_lane;
            for (auto& k : keys) {
                size_t best = 0;
                for (size_t l = 1; l < lanes; l++) if (load[l] < load[best]) best = l;
                load[best] += k.first; key_lane[k.second] = (uint32_t)best;
            }
            for (auto& b : blocks) share[key_lane[io->write_key(b)]].push_back(b);
        } else {
            uint64_t acc = 0; size_t lane = 0;
            for (auto& b : blocks) {
                share[lane].push_back(b);
                acc += std::max<uint32_t>(b.len, 4096);
                if (lane + 1 < lanes && acc >= total * (lane + 1) / lanes) lane++;
            }
        }
    }
    std::vector<Pipe*> pipes;
    rc = ctx_acquire_pipes(lane_devs, &pipes);
    if (rc) return rc;
    uint32_t readers, writers;       // sized AFTER the pipes are checked out: the count of lanes in flight includes this call's
    {
        std::unordered_map<uint32_t, int> seen;                  // blocks are interleaved across <= 64 files
        for (size_t i = 0; i < blocks.size() && i < 256; i++) seen[io->write_key(blocks[i])] = 1;
        // "many files" is a property of what ONE lane sees: 100 x 1 GiB over 8 lanes is 12 large files per lane
        io_threads_default(&readers, &writers, o.io_threads, lanes, std::min(n_gpus, lanes), seen.size() / lanes >= 32, has_prior, hash_only);
    }
    std::atomic<int> err{0}; std::string err_msg; std::mutex err_mu;
    std::vector<LaneStats> ls(lanes);
    std::vector<std::thread> th;
    for (size_t i = 0; i < lanes; i++)
        th.emplace_back([&, i] {
            run_lane(pipes[i], share[i], io, has_prior, hash_only, readers, writers, o.streams_per_gpu, hashes, &ls[i], &err, &err_msg, &err_mu);
        });
    for (auto& t : th) t.join();
    for (size_t i = 0; i < lanes; i++) ctx_release_pipe(pipes[i]);
    for (auto& l : ls) {
        st->bytes_h2d += l.bytes_h2d; st->bytes_d2h += l.bytes_d2h; st->bytes_written += l.bytes_written;
        st->blocks_skipped += l.blocks_skipped; st->kernel_launches += l.kernel_launches; st->ms_kernel += l.ms_kernel;
    }
    st->gpus_used = (uint32_t)std::min(n_gpus, lanes);
    st->lanes_used = (uint32_t)lanes;          // lanes the block list was sharded over
    if (err.load()) { set_last_error_str(err_msg); return err.load(); }
    return VMIG_OK;
}

int norm_opts(const vmig_opts* in, vmig_opts* o) {
    memset(o, 0, sizeof *o);
    if (in) *o = *in;
    if (!o->block_bytes) o->block_bytes = 4u << 20;
    if (env_long("VMIG_DIRECT_IO", 0) == 1) o->flags |= VMIG_F_DIRECT_IO;
    if (env_long("VMIG_CUFILE", 0) == 1) o->flags |= VMIG_F_CUFILE;
    if (o->block_bytes & 4095u) return fail(VMIG_EINVAL, "block_bytes %u is not a multiple of 4096", o->block_bytes);
    if (o->block_bytes > pipe_slot_bytes()) return fail(VMIG_EINVAL, "block_bytes %u exceeds the staging slot (%u)", o->block_bytes, pipe_slot_bytes());
    return VMIG_OK;
}

// The arguments, before anything is touched: both directories are there, and so is a GPU (no CPU fallback).
int check_args(const char* src_dir, const char* dst_dir, const vmig_opts* opts_in, vmig_opts* o)
{
    if (!src_dir || !*src_dir) return fail(VMIG_EINVAL, "src_dir is NULL/empty");
    int rc = norm_opts(opts_in, o);
    if (rc) return rc;
    const bool hash_only = (o->flags & VMIG_F_HASH_ONLY) != 0;
    if (!hash_only && (!dst_dir || !*dst_dir)) return fail(VMIG_EINVAL, "dst_dir is NULL/empty");
    struct stat sst;
    if (stat(src_dir, &sst) != 0) return fail(VMIG_EIO, "stat %s: %s", src_dir, errno_str(errno).c_str());
    if (!S_ISDIR(sst.st_mode)) return fail(VMIG_ENOTDIR, "%s is not a directory", src_dir);
    if (!hash_only) {
        if (stat(dst_dir, &sst) != 0) return fail(VMIG_EIO, "stat %s: %s", dst_dir, errno_str(errno).c_str());
        if (!S_ISDIR(sst.st_mode)) return fail(VMIG_ENOTDIR, "%s is not a directory", dst_dir);
    }
    std::vector<DeviceInfo> devs;
    return ctx_select(o->gpu_mask, &devs);
}

// Per-file state and the block list.  A destination file that still IS the one the prior table was written for (same
// inode, same ctime -- any write, truncate, chmod or replacement since then moved it --, same size) is patched in place;
// one the table names but that changed since is counted in *untrusted and rewritten.  Files are taken in groups of 64
// (bounds open fds) and blocks round-robin across the group's files so many destination files are written at once (a
// single tmpfs/xfs file takes writes one thread at a time: profiles/r01_hostio_probe.txt).
void plan_blocks(const Manifest& man, const BlockTable* prior, uint32_t block_bytes, FileIO& io,
                 std::vector<BlockRef>* blocks, uint64_t* untrusted)
{
    blocks->reserve(man.n_blocks);
    std::vector<uint32_t> group;
    auto flush_group = [&]() {
        uint64_t maxb = 0;
        for (uint32_t f : group) maxb = std::max(maxb, man.files[f].n_blocks);
        for (uint64_t r = 0; r < maxb; r++)
            for (uint32_t f : group) {
                const Entry& e = man.files[f];
                if (r >= e.n_blocks) continue;
                BlockRef b; b.file = f; b.file_off = r * (uint64_t)block_bytes;
                b.len = (uint32_t)std::min<uint64_t>(block_bytes, e.size - b.file_off);
                b.table_idx = e.first_block + r; b.prior_hash = 0; b.prior_valid = 0;
                if (io.fs[f].inplace) {
                    const TableFile& pf = prior->files[prior->index.at(e.rel)];
                    const uint64_t plen = r < prior->blocks_of(pf) ? std::min<uint64_t>(block_bytes, pf.size - b.file_off) : 0;
                    if (plen == b.len) { b.prior_hash = prior->hashes[pf.first_block + r]; b.prior_valid = 1; }
                }
                blocks->push_back(b);
            }
        group.clear();
    };
    for (uint32_t f = 0; f < man.files.size(); f++) {
        const Entry& e = man.files[f];
        if (e.hardlink_of >= 0 || e.n_blocks == 0) continue;
        if (prior) {
            auto it = prior->index.find(e.rel);
            struct stat ds;
            if (it != prior->index.end() && lstat(pjoin(io.dst_root, e.rel).c_str(), &ds) == 0 && S_ISREG(ds.st_mode) && ds.st_nlink == 1) {
                const TableFile& pf = prior->files[it->second];
                if (pf.ino != 0 && (uint64_t)ds.st_ino == pf.ino && ctime_ns(ds) == pf.ctime_ns && (uint64_t)ds.st_size == pf.size) {
                    io.fs[f].inplace = true; io.fs[f].dst_old_size = (uint64_t)ds.st_size;
                } else if (pf.ino != 0) {
                    (*untrusted)++;
                }
            }
        }
        group.push_back(f);
        if (group.size() == 64) flush_group();
    }
    flush_group();
}

// empty regular files carry no blocks: created here, after the data pass
int create_empty_files(const Manifest& man, FileIO& io)
{
    for (size_t f = 0; f < man.files.size(); f++) {
        const Entry& e = man.files[f];
        if (e.hardlink_of >= 0 || e.n_blocks) continue;
        const std::string p = pjoin(io.dst_root, e.rel);
        bool dio = false; int fd;
        int rc = open_for_write(p, true, &dio, &fd);
        if (rc) return rc;
        rc = apply_file_meta(fd, p, e, io.pol);
        struct stat ids;
        if (!rc && fstat(fd, &ids) == 0) io.fs[f].set_identity(ids);
        close(fd);
        if (rc) return rc;
    }
    return VMIG_OK;
}

// read the destination back through the same GPU path (hash only) and compare with the source's hashes
int verify_destination(const Manifest& man, const FileIO& io, const std::vector<BlockRef>& blocks,
                       const std::vector<uint64_t>& hashes, const vmig_opts& o, vmig_stats* st)
{
    FileIO vio;
    vio.hash_only = true;
    vio.direct = io.direct;          // O_DIRECT re-read: what is verified is what the device holds, not the page cache
    vio.cufile = io.cufile;
    int rc = vio.setup(io.dst_root, man);
    if (rc) return rc;
    std::vector<BlockRef> vblocks = blocks;
    for (auto& b : vblocks) { b.prior_hash = 0; b.prior_valid = 0; }
    std::vector<uint64_t> vh(man.n_blocks, 0);
    vmig_stats vst; memset(&vst, 0, sizeof vst);
    rc = run_blocks(vblocks, &vio, false, true, o, vh.data(), &vst);
    if (rc) return rc;
    st->kernel_launches += vst.kernel_launches; st->ms_kernel += vst.ms_kernel; st->bytes_h2d += vst.bytes_h2d;
    for (auto& b : vblocks)
        if (vh[b.table_idx] != hashes[b.table_idx])
            return fail(VMIG_EVERIFY, "verify: %s block %llu hashes %016llx in the destination, %016llx in the source",
                        man.files[b.file].rel.c_str(), (unsigned long long)(b.file_off / o.block_bytes),
                        (unsigned long long)vh[b.table_idx], (unsigned long long)hashes[b.table_idx]);
    if (o.flags & VMIG_F_PRUNE) {               // the destination's entry set must now equal the source's
        uint64_t extras = 0;
        rc = prune_extras(io.dst_root, man, true, &extras); if (rc) return rc;
        if (extras) return fail(VMIG_EVERIFY, "verify: %llu destination entries are not in the source after pruning", (unsigned long long)extras);
    }
    return VMIG_OK;
}

int store_table(const char* out_path, const Manifest& man, const FileIO& io, const std::vector<uint64_t>& hashes, uint32_t block_bytes)
{
    BlockTable t; t.block_bytes = block_bytes; t.algo = 1;
    t.files.reserve(man.files.size());
    for (uint32_t f = 0; f < man.files.size(); f++) {
        const Entry& e = man.files[f];
        const bool own = e.hardlink_of < 0 && (e.n_blocks || !io.hash_only);         // hard-linked paths are never patched in place
        t.files.push_back({e.rel, e.size, e.first_block, own ? io.fs[f].id_ino : 0, own ? io.fs[f].id_ctime_ns : 0});
    }
    t.hashes = hashes;
    return table_store(out_path, t);
}

// the old volume's data is about to be unlinked: deferred write-back errors (ENOSPC / EIO on delayed allocation, network
// filesystems) must surface first.  A no-op on tmpfs; one flush on a disk.
int flush_and_remove_source(const std::string& src, const std::string& dst, const Manifest& man)
{
    int dfd = open(dst.c_str(), O_RDONLY | O_DIRECTORY | O_CLOEXEC);
    if (dfd < 0) return fail(VMIG_EIO, "open %s: %s", dst.c_str(), errno_str(errno).c_str());
    const int sr = syncfs(dfd); const int se = errno;
    close(dfd);
    if (sr != 0) return fail(VMIG_EIO, "syncfs %s: %s (source left in place)", dst.c_str(), errno_str(se).c_str());
    return remove_source(src, man);
}

int migrate_tree_impl(const char* src_dir, const char* dst_dir, const char* prior_path, const char* out_path,
                      const vmig_opts* opts_in, vmig_stats* stats_out)
{
    vmig_stats st; memset(&st, 0, sizeof st);
    const uint64_t t_begin = now_ns();
    vmig_opts o;
    int rc = check_args(src_dir, dst_dir, opts_in, &o);
    if (rc) return rc;
    const bool hash_only = (o.flags & VMIG_F_HASH_ONLY) != 0;
    const std::string src(src_dir), dst(dst_dir ? dst_dir : "");

    Manifest man;
    uint64_t t0 = now_ns();
    rc = walk_tree(src, o.block_bytes, (o.flags & VMIG_F_SKIP_HIDDEN_TOPDIRS) != 0, &man);
    if (rc) return rc;
    st.ns_walk = now_ns() - t0;

    t0 = now_ns();
    BlockTable prior; const bool has_prior = prior_path && *prior_path && !hash_only;
    if (has_prior) {
        rc = table_load(prior_path, &prior);
        if (rc) return rc;
        if (prior.block_bytes != o.block_bytes) return fail(VMIG_ETABLE, "prior table block size %u != %u", prior.block_bytes, o.block_bytes);
    }
    FileIO io;
    io.dst_root = dst; io.pol = default_meta_policy(o.flags); io.hash_only = hash_only;
    io.corrupt_block = env_long("VMIG_CORRUPT_BLOCK", -1);
    io.direct = (o.flags & VMIG_F_DIRECT_IO) != 0;
    io.cufile = (o.flags & VMIG_F_CUFILE) != 0;
    rc = io.setup(src, man);
    if (rc) return rc;
    std::vector<uint64_t> hashes(man.n_blocks, 0);
    std::vector<BlockRef> blocks;
    plan_blocks(man, has_prior ? &prior : nullptr, o.block_bytes, io, &blocks, &st.files_untrusted);
    st.ns_plan = now_ns() - t0;

    // VMIG_F_PRUNE runs first: what it removes is by definition not in the source, a directory sitting where the source
    // now has a file (or the reverse) is out of the way before anything is created, and the directory mtimes restored
    // at the end are not disturbed by unlinks
    if ((o.flags & VMIG_F_PRUNE) && !hash_only) { rc = prune_extras(dst, man, false, &st.pruned); if (rc) return rc; }
    if (!hash_only) { rc = make_dirs(dst, man); if (rc) return rc; }

    t0 = now_ns();
    rc = run_blocks(blocks, &io, has_prior, hash_only, o, hashes.data(), &st);
    st.ns_data = now_ns() - t0;
    if (rc) return rc;

    t0 = now_ns();
    for (auto& e : man.files)                      // hard-linked paths share their primary's hashes
        if (e.hardlink_of >= 0) {
            const Entry& p = man.files[(size_t)e.hardlink_of];
            for (uint64_t r = 0; r < e.n_blocks; r++) hashes[e.first_block + r] = hashes[p.first_block + r];
        }
    if (!hash_only) {
        rc = create_empty_files(man, io);
        if (!rc) rc = replay_metadata(dst, man, io.pol, &st.symlinks, &st.hardlinks, &st.specials);
        if (rc) return rc;
    }
    st.ns_meta = now_ns() - t0;

    if ((o.flags & VMIG_F_VERIFY) && !hash_only) { rc = verify_destination(man, io, blocks, hashes, o, &st); if (rc) return rc; }

    t0 = now_ns();
    if (out_path && *out_path) { rc = store_table(out_path, man, io, hashes, o.block_bytes); if (rc) return rc; }
    st.ns_table = now_ns() - t0;

    if ((o.flags & VMIG_F_MOVE_SRC) && !hash_only) { rc = flush_and_remove_source(src, dst, man); if (rc) return rc; }

    st.files_direct = io.n_direct.load();
    st.bytes_total = man.bytes_total; st.blocks_total = man.n_blocks;
    st.files = man.files.size(); st.dirs = man.dirs.size();
    st.ns_total = now_ns() - t_begin;
    if (stats_out) *stats_out = st;
    return VMIG_OK;
}

}  // namespace

// =============================================================================================
extern "C" {

int vmig_init(uint32_t gpu_mask) { return ctx_init(gpu_mask); }
void vmig_shutdown(void) { ctx_shutdown(); cufile_shutdown(); }
int vmig_device_count(void) { return ctx_device_count(); }
const char* vmig_last_error(void) { return last_error_cstr(); }
const char* vmig_version(void) { return "libvmig 0.2 (abi 2, sm_100a)"; }
const char* vmig_strerror(int code)
{
    switch (code) {
    case VMIG_OK: return "ok";
    case VMIG_EINVAL: return "invalid argument";
    case VMIG_ENOGPU: return "no usable sm_100 GPU (no CPU fallback)";
    case VMIG_ECUDA: return "CUDA error";
    case VMIG_EIO: return "I/O error";
    case VMIG_ENOMEM: return "out of memory";
    case VMIG_ETABLE: return "bad block table";
    case VMIG_EFAULT: return "injected fault";
    case VMIG_ENOTDIR: return "not a directory";
    case VMIG_ESRCCHANGED: return "source changed during migration";
    case VMIG_EVERIFY: return "destination does not verify against the source";
    default: return "unknown vmig error";
    }
}

int vmig_migrate_tree(const char* src_dir, const char* dst_dir, const char* prior_table, const char* out_table,
                      const vmig_opts* opts, vmig_stats* stats)
{
    return migrate_tree_impl(src_dir, dst_dir, prior_table, out_table, opts, stats);
}
int vmig_copy_dir(const char* src_dir, const char* dst_dir) { return migrate_tree_impl(src_dir, dst_dir, nullptr, nullptr, nullptr, nullptr); }
int vmig_move_dir(const char* src_dir, const char* dst_dir)
{
    // a move destroys the only other copy: the destination is re-read through the GPU and must hash like the
    // source (VMIG_F_VERIFY) and is flushed (syncfs) before anything is unlinked
    vmig_opts o; memset(&o, 0, sizeof o); o.flags = VMIG_F_MOVE_SRC | VMIG_F_VERIFY;
    return migrate_tree_impl(src_dir, dst_dir, nullptr, nullptr, &o, nullptr);
}

int vmig_thread_plan(uint32_t lanes, uint32_t n_gpus, uint32_t flags, int has_prior, uint32_t* readers, uint32_t* writers)
{
    if (!readers || !writers || !lanes || !n_gpus) return fail(VMIG_EINVAL, "bad thread-plan arguments");
    return io_threads_default(readers, writers, 0, lanes, std::min<size_t>(n_gpus, lanes), false, has_prior != 0, (flags & VMIG_F_HASH_ONLY) != 0);
}

int vmig_host_alloc(void** p, uint64_t nbytes)
{
    if (!p) return fail(VMIG_EINVAL, "null out pointer");
    std::vector<DeviceInfo> devs; int rc = ctx_select(0, &devs); if (rc) return rc;
    cudaError_t e = cudaHostAlloc(p, nbytes ? nbytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(VMIG_ENOMEM, "cudaHostAlloc(%llu): %s", (unsigned long long)nbytes, cudaGetErrorString(e)); }
    return VMIG_OK;
}
void vmig_host_free(void* p) { if (p) cudaFreeHost(p); }

int vmig_migrate_buffer(const void* src, void* dst, uint64_t nbytes, const uint64_t* prior_hashes, const uint8_t* prior_valid,
                        uint64_t* out_hashes, const vmig_opts* opts, vmig_stats* stats)
{
    vmig_stats st; memset(&st, 0, sizeof st);
    const uint64_t t0 = now_ns();
    vmig_opts o;
    int rc = norm_opts(opts, &o);
    if (rc) return rc;
    const bool hash_only = (o.flags & VMIG_F_HASH_ONLY) != 0;
    if (!src || (!dst && !hash_only)) return fail(VMIG_EINVAL, "null buffer");
    std::vector<DeviceInfo> devs; rc = ctx_select(o.gpu_mask, &devs); if (rc) return rc;
    const uint64_t nb = (nbytes + o.block_bytes - 1) / o.block_bytes;
    std::vector<BlockRef> blocks(nb);
    const bool has_prior = prior_hashes != nullptr && prior_valid != nullptr;
    for (uint64_t i = 0; i < nb; i++) {
        BlockRef& b = blocks[i];
        b.file = 0; b.file_off = i * o.block_bytes; b.len = (uint32_t)std::min<uint64_t>(o.block_bytes, nbytes - b.file_off);
        b.table_idx = i; b.prior_hash = has_prior ? prior_hashes[i] : 0; b.prior_valid = has_prior ? prior_valid[i] : 0;
    }
    MemIO io; io.src = (const uint8_t*)src; io.dst = (uint8_t*)dst;
    io.src_pinned = is_pinned(src); io.dst_pinned = !hash_only && is_pinned(dst);
    std::vector<uint64_t> hashes(nb);
    rc = run_blocks(blocks, &io, has_prior, hash_only, o, hashes.data(), &st);
    if (rc) return rc;
    if (out_hashes && nb) memcpy(out_hashes, hashes.data(), nb * 8);
    st.bytes_total = nbytes; st.blocks_total = nb; st.ns_total = st.ns_data = now_ns() - t0;
    if (stats) *stats = st;
    return VMIG_OK;
}

int vmig_hash_blocks(int gpu, const void* host_buf, const uint64_t* offs, const uint32_t* lens, uint64_t n,
                     uint64_t* out_hashes, double* kernel_ms)
{
    if (n && (!offs || !lens || !out_hashes)) return fail(VMIG_EINVAL, "null array");
    if (gpu < 0 || gpu > 31) return fail(VMIG_EINVAL, "bad gpu index %d", gpu);
    vmig_opts o; memset(&o, 0, sizeof o); o.gpu_mask = 1u << gpu; o.block_bytes = 4u << 20; o.flags = VMIG_F_HASH_ONLY;
    std::vector<DeviceInfo> devs; int rc = ctx_select(o.gpu_mask, &devs); if (rc) return rc;
    std::vector<BlockRef> blocks(n);
    for (uint64_t i = 0; i < n; i++) {
        if (lens[i] && !host_buf) return fail(VMIG_EINVAL, "null host_buf");
        blocks[i].file = 0; blocks[i].file_off = offs[i]; blocks[i].len = lens[i]; blocks[i].table_idx = i;
        blocks[i].prior_hash = 0; blocks[i].prior_valid = 0;
    }
    MemIO io; io.src = (const uint8_t*)host_buf; io.dst = nullptr;   // staged: arbitrary offsets become 512-B aligned in HBM
    vmig_stats st; memset(&st, 0, sizeof st);
    rc = run_blocks(blocks, &io, false, true, o, out_hashes, &st);
    if (kernel_ms) *kernel_ms = st.ms_kernel;
    return rc;
}

// ---------------------------------------------------------------------------------------------
// host<->HBM link probe

static int link_probe_here(int gpu, uint64_t bytes, double* gbs)
{
    const size_t piece = 32u << 20, ring = 8;           // 8 x 32 MiB per direction: larger than any host cache
    CU_API(cudaSetDevice(gpu));
    uint8_t *h_a = nullptr, *h_b = nullptr, *d_a = nullptr, *d_b = nullptr;
    cudaStream_t s0 = nullptr, s1 = nullptr; cudaEvent_t e[4] = {nullptr, nullptr, nullptr, nullptr};
    auto cleanup = [&] {
        if (h_a) cudaFreeHost(h_a); if (h_b) cudaFreeHost(h_b); if (d_a) cudaFree(d_a); if (d_b) cudaFree(d_b);
        if (s0) cudaStreamDestroy(s0); if (s1) cudaStreamDestroy(s1);
        for (auto& x : e) if (x) cudaEventDestroy(x);
    };
    auto run = [&]() -> int {
        CU_API(cudaHostAlloc((void**)&h_a, piece * ring, cudaHostAllocPortable)); memset(h_a, 1, piece * ring);
        CU_API(cudaHostAlloc((void**)&h_b, piece * ring, cudaHostAllocPortable)); memset(h_b, 2, piece * ring);
        CU_API(cudaMalloc((void**)&d_a, piece * ring)); CU_API(cudaMalloc((void**)&d_b, piece * ring));
        CU_API(cudaMemset(d_b, 3, piece * ring));
        CU_API(cudaStreamCreateWithFlags(&s0, cudaStreamNonBlocking)); CU_API(cudaStreamCreateWithFlags(&s1, cudaStreamNonBlocking));
        for (auto& x : e) CU_API(cudaEventCreate(&x));
        const uint64_t n = std::max<uint64_t>(1, bytes / piece);
        auto pass = [&](bool up, bool down, double* up_gbs, double* down_gbs) -> int {
            for (int rep = 0; rep < 2; rep++) {          // rep 0 warms up
                if (up) CU_API(cudaEventRecord(e[0], s0));
                if (down) CU_API(cudaEventRecord(e[2], s1));
                for (uint64_t i = 0; i < n; i++) {
                    const size_t o = (size_t)(i % ring) * piece;
                    if (up) CU_API(cudaMemcpyAsync(d_a + o, h_a + o, piece, cudaMemcpyHostToDevice, s0));
                    if (down) CU_API(cudaMemcpyAsync(h_b + o, d_b + o, piece, cudaMemcpyDeviceToHost, s1));
                }
                if (up) CU_API(cudaEventRecord(e[1], s0));
                if (down) CU_API(cudaEventRecord(e[3], s1));
                CU_API(cudaStreamSynchronize(s0)); CU_API(cudaStreamSynchronize(s1));
            }
            float ms = 0;
            if (up) { CU_API(cudaEventElapsedTime(&ms, e[0], e[1])); *up_gbs = (double)(n * piece) / (ms * 1e-3) / 1e9; }
            if (down) { CU_API(cudaEventElapsedTime(&ms, e[2], e[3])); *down_gbs = (double)(n * piece) / (ms * 1e-3) / 1e9; }
            return VMIG_OK;
        };
        double dummy = 0;
        int rc = pass(true, false, &gbs[0], &dummy); if (rc) return rc;
        rc = pass(false, true, &dummy, &gbs[1]); if (rc) return rc;
        return pass(true, true, &gbs[2], &gbs[3]);
    };
    const int rc = run();
    const std::string keep = rc ? last_error_cstr() : "";
    cleanup();
    if (rc) set_last_error_str(keep);
    return rc;
}

int vmig_link_probe(int gpu, uint64_t bytes, double gbs[4])
{
    if (!gbs || gpu < 0 || gpu > 31) return fail(VMIG_EINVAL, "bad link-probe arguments");
    std::vector<DeviceInfo> devs; int rc = ctx_select(1u << gpu, &devs); if (rc) return rc;
    gbs[0] = gbs[1] = gbs[2] = gbs[3] = 0;
    // allocate and first-touch the pinned buffers on the GPU's NUMA node, like the staging rings
    std::string msg;
    std::thread t([&] {
        if (!devs[0].cpus.empty()) {
            cpu_set_t set; CPU_ZERO(&set);
            for (int c : devs[0].cpus) if (c < CPU_SETSIZE) CPU_SET(c, &set);
            sched_setaffinity(0, sizeof set, &set);
        }
        rc = link_probe_here(gpu, bytes ? bytes : (4ull << 30), gbs);
        if (rc) msg = last_error_cstr();
    });
    t.join();
    if (rc) set_last_error_str(msg);
    return rc;
}

// ---------------------------------------------------------------------------------------------
// HBM-resident batch
struct vmig_resident {
    int dev; int sm_count; uint64_t n; uint32_t block_bytes;
    uint8_t* d_data; uint64_t* d_offs; uint32_t* d_lens; uint64_t* d_hashes; uint64_t* d_prior; uint8_t* d_valid;
    uint8_t* d_changed; uint32_t* d_survivors; uint32_t* d_nsurv; uint32_t* d_counter; uint64_t* d_scratch;
    bool has_prior; cudaStream_t stream; cudaEvent_t e0, e1, e2, e3;
};


void vmig_resident_close(vmig_resident* r);

static int resident_alloc(vmig_resident* r, uint64_t n_blocks, uint32_t block_bytes)
{
    CU_API(cudaSetDevice(r->dev));
    CU_API(cudaMalloc((void**)&r->d_data, n_blocks * (uint64_t)block_bytes + kTailPad));
    CU_API(cudaMalloc((void**)&r->d_offs, n_blocks * 8)); CU_API(cudaMalloc((void**)&r->d_lens, n_blocks * 4));
    CU_API(cudaMalloc((void**)&r->d_hashes, n_blocks * 8)); CU_API(cudaMalloc((void**)&r->d_prior, n_blocks * 8));
    CU_API(cudaMalloc((void**)&r->d_valid, n_blocks)); CU_API(cudaMalloc((void**)&r->d_changed, n_blocks));
    CU_API(cudaMalloc((void**)&r->d_survivors, n_blocks * 4)); CU_API(cudaMalloc((void**)&r->d_nsurv, 256));
    CU_API(cudaMalloc((void**)&r->d_counter, 256)); CU_API(cudaMalloc((void**)&r->d_scratch, n_blocks * 8));
    CU_API(cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking));
    CU_API(cudaEventCreate(&r->e0)); CU_API(cudaEventCreate(&r->e1)); CU_API(cudaEventCreate(&r->e2)); CU_API(cudaEventCreate(&r->e3));
    std::vector<uint64_t> offs(n_blocks); std::vector<uint32_t> lens(n_blocks, block_bytes);
    for (uint64_t i = 0; i < n_blocks; i++) offs[i] = i * (uint64_t)block_bytes;
    CU_API(cudaMemcpy(r->d_offs, offs.data(), n_blocks * 8, cudaMemcpyHostToDevice));
    CU_API(cudaMemcpy(r->d_lens, lens.data(), n_blocks * 4, cudaMemcpyHostToDevice));
    CU_API(cudaMemset(r->d_valid, 0, n_blocks)); CU_API(cudaMemset(r->d_prior, 0, n_blocks * 8));
    CU_API(cudaMemset(r->d_data + n_blocks * (uint64_t)block_bytes, 0, kTailPad));
    return VMIG_OK;
}

int vmig_resident_open(int gpu, uint64_t n_blocks, uint32_t block_bytes, vmig_resident** out)
{
    if (!out || !n_blocks || !block_bytes || (block_bytes & 511u) || n_blocks > 0x7FFFFFFFull) return fail(VMIG_EINVAL, "bad resident geometry");
    if (gpu < 0 || gpu > 31) return fail(VMIG_EINVAL, "bad gpu index %d", gpu);
    std::vector<DeviceInfo> devs; int rc = ctx_select(1u << gpu, &devs); if (rc) return rc;
    vmig_resident* r = new vmig_resident(); memset(r, 0, sizeof *r);
    r->dev = gpu; r->sm_count = devs[0].sm_count; r->n = n_blocks; r->block_bytes = block_bytes;
    rc = resident_alloc(r, n_blocks, block_bytes);
    if (rc) {                                   // e.g. the batch does not fit in HBM: give back what was taken
        const std::string keep = last_error_cstr();
        vmig_resident_close(r);
        set_last_error_str(keep);
        return rc;
    }
    *out = r;
    return VMIG_OK;
}
void vmig_resident_close(vmig_resident* r)
{
    if (!r) return;
    cudaSetDevice(r->dev);
    if (r->stream) cudaStreamSynchronize(r->stream);
    cudaFree(r->d_data); cudaFree(r->d_offs); cudaFree(r->d_lens); cudaFree(r->d_hashes); cudaFree(r->d_prior); cudaFree(r->d_valid);
    cudaFree(r->d_changed); cudaFree(r->d_survivors); cudaFree(r->d_nsurv); cudaFree(r->d_counter); cudaFree(r->d_scratch);
    if (r->stream) cudaStreamDestroy(r->stream);
    if (r->e0) cudaEventDestroy(r->e0); if (r->e1) cudaEventDestroy(r->e1); if (r->e2) cudaEventDestroy(r->e2); if (r->e3) cudaEventDestroy(r->e3);
    delete r;
}
int vmig_resident_fill(vmig_resident* r, uint64_t seed)
{
    if (!r) return fail(VMIG_EINVAL, "null handle");
    CU_API(cudaSetDevice(r->dev));
    CU_API(launch_splitmix_fill(r->d_data, r->n * (uint64_t)r->block_bytes, seed, r->stream));
    std::vector<uint32_t> lens(r->n, r->block_bytes);
    CU_API(cudaMemcpyAsync(r->d_lens, lens.data(), r->n * 4, cudaMemcpyHostToDevice, r->stream));
    CU_API(cudaStreamSynchronize(r->stream));
    return VMIG_OK;
}
int vmig_resident_set_len(vmig_resident* r, uint64_t block, uint32_t len)
{
    if (!r || block >= r->n || len > r->block_bytes) return fail(VMIG_EINVAL, "bad block/len");
    CU_API(cudaSetDevice(r->dev));
    CU_API(cudaMemcpy(r->d_lens + block, &len, 4, cudaMemcpyHostToDevice));
    return VMIG_OK;
}
int vmig_resident_upload(vmig_resident* r, uint64_t block, const void* host, uint32_t len)
{
    if (!r || block >= r->n || len > r->block_bytes || (len && !host)) return fail(VMIG_EINVAL, "bad block/len");
    CU_API(cudaSetDevice(r->dev));
    if (len) CU_API(cudaMemcpy(r->d_data + block * (uint64_t)r->block_bytes, host, len, cudaMemcpyHostToDevice));
    CU_API(cudaMemcpy(r->d_lens + block, &len, 4, cudaMemcpyHostToDevice));
    return VMIG_OK;
}
int vmig_resident_download(vmig_resident* r, uint64_t block, void* host, uint32_t len)
{
    if (!r || block >= r->n || len > r->block_bytes || !host) return fail(VMIG_EINVAL, "bad block/len");
    CU_API(cudaSetDevice(r->dev));
    CU_API(cudaMemcpy(host, r->d_data + block * (uint64_t)r->block_bytes, len, cudaMemcpyDeviceToHost));
    return VMIG_OK;
}
int vmig_resident_flip(vmig_resident* r, const uint64_t* blocks, uint64_t n)
{
    if (!r || (n && !blocks) || n > r->n) return fail(VMIG_EINVAL, "bad flip list");
    for (uint64_t i = 0; i < n; i++) if (blocks[i] >= r->n) return fail(VMIG_EINVAL, "flip index out of range");
    CU_API(cudaSetDevice(r->dev));
    if (n) {
        CU_API(cudaMemcpyAsync(r->d_scratch, blocks, n * 8, cudaMemcpyHostToDevice, r->stream));
        CU_API(launch_flip_first8(r->d_data, r->d_offs, r->d_scratch, n, r->stream));
        CU_API(cudaStreamSynchronize(r->stream));
    }
    return VMIG_OK;
}
int vmig_resident_set_prior(vmig_resident* r, const uint64_t* hashes, const uint8_t* valid)
{
    if (!r) return fail(VMIG_EINVAL, "null handle");
    CU_API(cudaSetDevice(r->dev));
    r->has_prior = hashes != nullptr && valid != nullptr;
    if (r->has_prior) {
        CU_API(cudaMemcpy(r->d_prior, hashes, r->n * 8, cudaMemcpyHostToDevice));
        CU_API(cudaMemcpy(r->d_valid, valid, r->n, cudaMemcpyHostToDevice));
    } else {
        CU_API(cudaMemset(r->d_valid, 0, r->n));
    }
    return VMIG_OK;
}
int vmig_resident_pass(vmig_resident* r, uint32_t iters, double* ms_hash_last, double* ms_total)
{
    if (!r || !iters) return fail(VMIG_EINVAL, "bad arguments");
    CU_API(cudaSetDevice(r->dev));
    HashLaunch a;
    a.base = r->d_data; a.offs = r->d_offs; a.lens = r->d_lens; a.n = (uint32_t)r->n; a.hashes = r->d_hashes;
    a.prior = r->d_prior; a.prior_valid = r->d_valid; a.changed = r->d_changed; a.work_counter = r->d_counter;
    CU_API(cudaEventRecord(r->e0, r->stream));
    for (uint32_t it = 0; it < iters; it++) {
        if (it + 1 == iters) CU_API(cudaEventRecord(r->e1, r->stream));
        CU_API(launch_xxh64_blocks(a, r->sm_count, r->stream));
        if (it + 1 == iters) CU_API(cudaEventRecord(r->e2, r->stream));
        CU_API(launch_diff_select(r->d_changed, (uint32_t)r->n, r->d_survivors, r->d_nsurv, r->stream));
    }
    CU_API(cudaEventRecord(r->e3, r->stream));
    CU_API(cudaStreamSynchronize(r->stream));
    float a_ms = 0, b_ms = 0;
    CU_API(cudaEventElapsedTime(&a_ms, r->e1, r->e2));
    CU_API(cudaEventElapsedTime(&b_ms, r->e0, r->e3));
    if (ms_hash_last) *ms_hash_last = a_ms;
    if (ms_total) *ms_total = b_ms;
    return VMIG_OK;
}
int vmig_resident_results(vmig_resident* r, uint64_t* hashes, uint32_t* survivors, uint64_t* n_survivors)
{
    if (!r) return fail(VMIG_EINVAL, "null handle");
    CU_API(cudaSetDevice(r->dev));
    if (hashes) CU_API(cudaMemcpy(hashes, r->d_hashes, r->n * 8, cudaMemcpyDeviceToHost));
    uint32_t ns = 0;
    CU_API(cudaMemcpy(&ns, r->d_nsurv, 4, cudaMemcpyDeviceToHost));
    if (n_survivors) *n_survivors = ns;
    if (survivors && ns) CU_API(cudaMemcpy(survivors, r->d_survivors, (size_t)ns * 4, cudaMemcpyDeviceToHost));
    return VMIG_OK;
}

}  // extern "C"
