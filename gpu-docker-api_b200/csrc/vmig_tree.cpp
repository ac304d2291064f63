// vmig_tree.cpp -- source-tree walk and destination metadata replay (see vmig_tree.h).
#include "vmig_tree.h"
#include <unordered_set>
#include <dirent.h>
#include "vmig_common.h"

#include <dirent.h>
#include <fcntl.h>
#include <unistd.h>
#include <linux/openat2.h>
#include <sys/syscall.h>
#include <sys/sysmacros.h>
#include <algorithm>
#include <atomic>
#include <map>
#include <utility>
#include <thread>
#include <mutex>
#include <iterator>

namespace vmig {

static inline std::string join(const std::string& a, const std::string& b) {
    if (b == ".") return a;
    return a + "/" + b;
}

// The source may belong to a container that is still running (the first pass of a two-pass hand-off), so
// nothing on the source side trusts a path twice: directories are entered with openat(O_NOFOLLOW) relative to
// their parent's descriptor, and files are opened later with open_beneath() below.  A directory that a tenant
// swaps for a symlink between the lstat and the open makes the call fail; it is never followed out of the tree
// (GNU tar walks the same way, which is what the reference's `tar c .` relies on).
int open_beneath(int root_fd, const std::string& rel, int flags, int* out_fd)
{
    static std::atomic<int> have_openat2{1};
    if (rel.empty() || rel[0] == '/') return fail(VMIG_EINVAL, "open_beneath: bad relative path '%s'", rel.c_str());
    if (have_openat2.load(std::memory_order_relaxed)) {
        struct open_how how; memset(&how, 0, sizeof how);
        how.flags = (uint64_t)(flags | O_CLOEXEC | O_NOFOLLOW);
        how.resolve = RESOLVE_BENEATH | RESOLVE_NO_SYMLINKS | RESOLVE_NO_MAGICLINKS;
        long fd = syscall(SYS_openat2, root_fd, rel.c_str(), &how, sizeof how);
        if (fd >= 0) { *out_fd = (int)fd; return VMIG_OK; }
        if (errno != ENOSYS) {
            const int e = errno;
            if (e == ELOOP || e == EXDEV || e == ENOTDIR)
                return fail(VMIG_ESRCCHANGED, "%s is no longer a plain path beneath the source root (%s): a symlink or rename raced the walk", rel.c_str(), errno_str(e).c_str());
            return fail(e == ENOENT ? VMIG_ESRCCHANGED : VMIG_EIO, "open %s: %s", rel.c_str(), errno_str(e).c_str());
        }
        have_openat2.store(0, std::memory_order_relaxed);      // pre-5.6 kernel: walk the components by hand
    }
    return open_beneath_walk(root_fd, rel, flags, out_fd);
}

int open_beneath_walk(int root_fd, const std::string& rel, int flags, int* out_fd)
{
    if (rel.empty() || rel[0] == '/') return fail(VMIG_EINVAL, "open_beneath: bad relative path '%s'", rel.c_str());
    int cur = root_fd; bool own = false;
    size_t pos = 0;
    for (;;) {
        const size_t slash = rel.find('/', pos);
        const std::string comp = rel.substr(pos, slash == std::string::npos ? std::string::npos : slash - pos);
        const bool last = slash == std::string::npos;
        if (comp.empty() || comp == "." || comp == "..") { if (own) close(cur); return fail(VMIG_EINVAL, "open_beneath: bad component in '%s'", rel.c_str()); }
        const int fl = last ? (flags | O_CLOEXEC | O_NOFOLLOW) : (O_RDONLY | O_DIRECTORY | O_CLOEXEC | O_NOFOLLOW);
        const int fd = openat(cur, comp.c_str(), fl);
        const int e = errno;
        if (own) close(cur);
        if (fd < 0) {
            if (e == ELOOP || e == ENOTDIR || e == ENOENT)
                return fail(VMIG_ESRCCHANGED, "%s is no longer a plain path beneath the source root (%s)", rel.c_str(), errno_str(e).c_str());
            return fail(VMIG_EIO, "open %s: %s", rel.c_str(), errno_str(e).c_str());
        }
        if (last) { *out_fd = fd; return VMIG_OK; }
        cur = fd; own = true; pos = slash + 1;
    }
}

// dfd: open descriptor of the directory `rel`; consumed (closed) by this call.
// defer_subdirs != nullptr: do not descend; list the sub-directories (name, rel) for the caller to walk (in parallel).
static int walk_dir(int dfd, const std::string& rel, uint32_t block_bytes, bool skip_hidden_topdirs,
                    Manifest* m, int depth, std::vector<std::pair<std::string, std::string>>* defer_subdirs = nullptr)
{
    const int dfd_dup = dup(dfd);
    DIR* d = dfd_dup >= 0 ? fdopendir(dfd) : nullptr;
    if (!d) { const int e = errno; close(dfd); if (dfd_dup >= 0) close(dfd_dup); return fail(VMIG_EIO, "opendir %s: %s", rel.c_str(), errno_str(e).c_str()); }
    std::vector<std::string> names;
    errno = 0;
    while (struct dirent* de = readdir(d)) {
        const char* n = de->d_name;
        if (n[0] == '.' && (n[1] == 0 || (n[1] == '.' && n[2] == 0))) continue;
        names.emplace_back(n);
    }
    const int rd_errno = errno;
    closedir(d);                                   // closes dfd; dfd_dup stays for the *at() calls
    if (rd_errno) { close(dfd_dup); return fail(VMIG_EIO, "readdir %s: %s", rel.c_str(), errno_str(rd_errno).c_str()); }
    std::sort(names.begin(), names.end());

    std::vector<std::pair<std::string, std::string>> subdirs;     // (name, rel)
    for (const auto& n : names) {
        struct stat st;
        if (fstatat(dfd_dup, n.c_str(), &st, AT_SYMLINK_NOFOLLOW) != 0) {
            const int e = errno; close(dfd_dup);
            return fail(VMIG_EIO, "lstat %s/%s: %s", rel.c_str(), n.c_str(), errno_str(e).c_str());
        }
        Entry e;
        e.rel = rel == "." ? n : rel + "/" + n;
        e.mode = st.st_mode; e.uid = st.st_uid; e.gid = st.st_gid; e.mtime = st.st_mtim; e.atime = st.st_atim;
        switch (st.st_mode & S_IFMT) {
        case S_IFDIR:
            if (skip_hidden_topdirs && depth == 0 && n[0] == '.') continue;   // `mv /root/src/*` misses these
            e.type = kDir; m->dirs.push_back(e); subdirs.push_back({n, e.rel});
            break;
        case S_IFREG: {
            e.type = kFile; e.size = (uint64_t)st.st_size;
            e.n_blocks = (e.size + block_bytes - 1) / block_bytes;
            if (st.st_nlink > 1) {                   // group key (device:inode); resolved to an index after sorting
                char key[48]; snprintf(key, sizeof key, "%llx:%llx", (unsigned long long)st.st_dev, (unsigned long long)st.st_ino);
                e.target = key;
            }
            m->files.push_back(e);
            break;
        }
        case S_IFLNK: {
            e.type = kSymlink;
            std::string buf((size_t)st.st_size + 256, '\0');
            ssize_t k = readlinkat(dfd_dup, n.c_str(), &buf[0], buf.size());
            if (k < 0) { const int er = errno; close(dfd_dup); return fail(VMIG_EIO, "readlink %s: %s", e.rel.c_str(), errno_str(er).c_str()); }
            buf.resize((size_t)k); e.target = buf;
            m->symlinks.push_back(e);
            break;
        }
        case S_IFCHR: case S_IFBLK: case S_IFIFO:
            e.type = kSpecial; e.rdev = st.st_rdev; m->specials.push_back(e);
            break;
        case S_IFSOCK:
            m->sockets_skipped++;        // GNU tar: "socket ignored"
            break;
        default: break;
        }
    }
    if (defer_subdirs) { *defer_subdirs = subdirs; close(dfd_dup); return VMIG_OK; }
    for (const auto& sd : subdirs) {
        const int cfd = openat(dfd_dup, sd.first.c_str(), O_RDONLY | O_DIRECTORY | O_NOFOLLOW | O_CLOEXEC);
        if (cfd < 0) {
            const int e = errno; close(dfd_dup);
            return fail(e == ELOOP || e == ENOTDIR || e == ENOENT ? VMIG_ESRCCHANGED : VMIG_EIO,
                        "open directory %s: %s%s", sd.second.c_str(), errno_str(e).c_str(),
                        e == ELOOP || e == ENOTDIR ? " (it was a directory a moment ago: not following)" : "");
        }
        int rc = walk_dir(cfd, sd.second, block_bytes, skip_hidden_topdirs, m, depth + 1);
        if (rc) { close(dfd_dup); return rc; }
    }
    close(dfd_dup);
    return VMIG_OK;
}

int walk_tree(const std::string& src_root, uint32_t block_bytes, bool skip_hidden_topdirs, Manifest* m)
{
    *m = Manifest();
    struct stat st;
    if (stat(src_root.c_str(), &st) != 0) return fail(VMIG_EIO, "stat %s: %s", src_root.c_str(), errno_str(errno).c_str());
    if (!S_ISDIR(st.st_mode)) return fail(VMIG_ENOTDIR, "%s is not a directory", src_root.c_str());
    Entry root;
    root.rel = "."; root.type = kDir; root.mode = st.st_mode; root.uid = st.st_uid; root.gid = st.st_gid;
    root.mtime = st.st_mtim; root.atime = st.st_atim;
    m->dirs.push_back(root);
    const int rfd = open(src_root.c_str(), O_RDONLY | O_DIRECTORY | O_CLOEXEC);
    if (rfd < 0) return fail(VMIG_EIO, "open %s: %s", src_root.c_str(), errno_str(errno).c_str());
    const int rfd2 = dup(rfd);                         // walk_dir consumes rfd; the sub-walks open beneath rfd2
    // The root level is read here; its sub-directories are walked by up to 8 threads, each into a private manifest
    // (a 40 960-file layer: 71 ms -> ~15 ms; the lstat()s are the cost).  Merged in name order, which is the order
    // the single-threaded descent produced: parents before children, files sorted afterwards anyway.
    std::vector<std::pair<std::string, std::string>> top;
    int rc = walk_dir(rfd, ".", block_bytes, skip_hidden_topdirs, m, 0, &top);
    if (rc) { if (rfd2 >= 0) close(rfd2); return rc; }
    if (!top.empty()) {
        if (rfd2 < 0) return fail(VMIG_EIO, "dup: %s", errno_str(errno).c_str());
        std::vector<Manifest> sub(top.size());
        std::atomic<size_t> next{0}; std::atomic<int> bad{0};
        std::string bad_msg; std::mutex bad_mu;
        auto work = [&] {
            for (;;) {
                const size_t i = next.fetch_add(1);
                if (i >= top.size() || bad.load()) return;
                int r;
                const int cfd = openat(rfd2, top[i].first.c_str(), O_RDONLY | O_DIRECTORY | O_NOFOLLOW | O_CLOEXEC);
                if (cfd < 0) {
                    const int e = errno;
                    r = fail(e == ELOOP || e == ENOTDIR || e == ENOENT ? VMIG_ESRCCHANGED : VMIG_EIO, "open directory %s: %s%s", top[i].second.c_str(),
                             errno_str(e).c_str(), e == ELOOP || e == ENOTDIR ? " (it was a directory a moment ago: not following)" : "");
                } else {
                    r = walk_dir(cfd, top[i].second, block_bytes, skip_hidden_topdirs, &sub[i], 1);
                }
                if (r) { std::lock_guard<std::mutex> lk(bad_mu); if (!bad.load()) { bad_msg = last_error_cstr(); bad.store(r); } return; }
            }
        };
        const size_t nth = std::min<size_t>((size_t)std::max<long>(1, env_long("VMIG_WALK_THREADS", 8)), top.size());
        if (nth <= 1) work();
        else { std::vector<std::thread> th; for (size_t t = 0; t < nth; t++) th.emplace_back(work); for (auto& t : th) t.join(); }
        close(rfd2);
        if (bad.load()) { set_last_error_str(bad_msg); return bad.load(); }
        for (auto& sm : sub) {
            m->dirs.insert(m->dirs.end(), std::make_move_iterator(sm.dirs.begin()), std::make_move_iterator(sm.dirs.end()));
            m->files.insert(m->files.end(), std::make_move_iterator(sm.files.begin()), std::make_move_iterator(sm.files.end()));
            m->symlinks.insert(m->symlinks.end(), std::make_move_iterator(sm.symlinks.begin()), std::make_move_iterator(sm.symlinks.end()));
            m->specials.insert(m->specials.end(), std::make_move_iterator(sm.specials.begin()), std::make_move_iterator(sm.specials.end()));
            m->sockets_skipped += sm.sockets_skipped;
        }
    } else if (rfd2 >= 0) close(rfd2);

    std::sort(m->files.begin(), m->files.end(), [](const Entry& a, const Entry& b) { return a.rel < b.rel; });
    // resolve hard links to indices; the primary of a group is its bytewise-smallest path
    // (a group with a single member inside the tree is just a regular file)
    std::map<std::string, int64_t> group_min;
    for (size_t i = 0; i < m->files.size(); i++) {
        const Entry& e = m->files[i];
        if (e.target.empty()) continue;
        auto it = group_min.find(e.target);
        if (it == group_min.end()) group_min[e.target] = (int64_t)i;     // files are sorted: first seen = smallest
    }
    for (size_t i = 0; i < m->files.size(); i++) {
        Entry& e = m->files[i];
        if (e.target.empty()) continue;
        const int64_t p = group_min[e.target];
        if (p != (int64_t)i) e.hardlink_of = p;
        e.target.clear();
    }
    uint64_t fb = 0;
    for (auto& e : m->files) { e.first_block = fb; fb += e.n_blocks; m->bytes_total += e.size; }
    m->n_blocks = fb;
    return VMIG_OK;
}

MetaPolicy default_meta_policy(uint32_t flags)
{
    MetaPolicy p;
    p.is_root = geteuid() == 0;
    mode_t um = umask(0); umask(um);
    p.umask_bits = um;
    p.mtime_ns = (flags & VMIG_F_MTIME_NS) != 0 || (flags & VMIG_F_MOVE_SRC) != 0;
    p.no_metadata = (flags & VMIG_F_NO_METADATA) != 0;
    p.keep_atime = (flags & VMIG_F_MOVE_SRC) != 0;
    return p;
}

static inline mode_t eff_mode(const Entry& e, const MetaPolicy& pol) {
    mode_t m = e.mode & 07777;
    if (!pol.is_root) m &= ~pol.umask_bits & 0777;   // tar without -p: umask applied, setuid/setgid/sticky dropped
    return m;
}
static inline void fill_times(const Entry& e, const MetaPolicy& pol, struct timespec ts[2]) {
    if (pol.keep_atime) ts[0] = e.atime; else { ts[0].tv_sec = 0; ts[0].tv_nsec = UTIME_OMIT; }
    ts[1] = e.mtime;
    if (!pol.mtime_ns) ts[1].tv_nsec = 0;   // tar's gnu format stores whole seconds
}

int unlink_if_exists(const std::string& path, bool* was_dir)
{
    struct stat st;
    if (was_dir) *was_dir = false;
    if (lstat(path.c_str(), &st) != 0) {
        if (errno == ENOENT) return VMIG_OK;
        return fail(VMIG_EIO, "lstat %s: %s", path.c_str(), errno_str(errno).c_str());
    }
    if (S_ISDIR(st.st_mode)) { if (was_dir) *was_dir = true; return VMIG_OK; }
    if (unlink(path.c_str()) != 0 && errno != ENOENT)
        return fail(VMIG_EIO, "unlink %s: %s", path.c_str(), errno_str(errno).c_str());
    return VMIG_OK;
}

int make_dirs(const std::string& dst_root, const Manifest& m)
{
    for (size_t i = 1; i < m.dirs.size(); i++) {
        const std::string p = join(dst_root, m.dirs[i].rel);
        if (mkdir(p.c_str(), 0700) == 0) continue;
        if (errno != EEXIST) return fail(VMIG_EIO, "mkdir %s: %s", p.c_str(), errno_str(errno).c_str());
        struct stat st;
        if (lstat(p.c_str(), &st) == 0 && S_ISDIR(st.st_mode)) continue;
        // a non-directory is in the way: tar replaces it
        if (unlink(p.c_str()) != 0 || mkdir(p.c_str(), 0700) != 0)
            return fail(VMIG_EIO, "replace %s by directory: %s", p.c_str(), errno_str(errno).c_str());
    }
    return VMIG_OK;
}

bool file_meta_matches(int fd, const Entry& e, const MetaPolicy& pol)
{
    if (pol.no_metadata) return true;
    struct stat st;
    if (fd < 0 || fstat(fd, &st) != 0) return false;
    struct timespec ts[2];
    fill_times(e, pol, ts);
    if (pol.keep_atime) return false;                       // move semantics restore atime too: always apply
    if (pol.is_root && (st.st_uid != e.uid || st.st_gid != e.gid)) return false;
    if ((st.st_mode & 07777) != eff_mode(e, pol)) return false;
    return st.st_mtim.tv_sec == ts[1].tv_sec && st.st_mtim.tv_nsec == ts[1].tv_nsec;
}

int apply_file_meta(int fd, const std::string& path, const Entry& e, const MetaPolicy& pol)
{
    if (pol.no_metadata) return VMIG_OK;
    struct timespec ts[2];
    fill_times(e, pol, ts);
    if (fd >= 0) {
        if (pol.is_root && fchown(fd, e.uid, e.gid) != 0) return fail(VMIG_EIO, "fchown %s: %s", path.c_str(), errno_str(errno).c_str());
        if (fchmod(fd, eff_mode(e, pol)) != 0) return fail(VMIG_EIO, "fchmod %s: %s", path.c_str(), errno_str(errno).c_str());
        if (futimens(fd, ts) != 0) return fail(VMIG_EIO, "futimens %s: %s", path.c_str(), errno_str(errno).c_str());
    } else {
        if (pol.is_root && lchown(path.c_str(), e.uid, e.gid) != 0) return fail(VMIG_EIO, "lchown %s: %s", path.c_str(), errno_str(errno).c_str());
        if (chmod(path.c_str(), eff_mode(e, pol)) != 0) return fail(VMIG_EIO, "chmod %s: %s", path.c_str(), errno_str(errno).c_str());
        if (utimensat(AT_FDCWD, path.c_str(), ts, 0) != 0) return fail(VMIG_EIO, "utimensat %s: %s", path.c_str(), errno_str(errno).c_str());
    }
    return VMIG_OK;
}

int replay_metadata(const std::string& dst_root, const Manifest& m, const MetaPolicy& pol,
                    uint64_t* n_symlinks, uint64_t* n_hardlinks, uint64_t* n_specials)
{
    struct timespec ts[2];
    for (const auto& e : m.symlinks) {
        const std::string p = join(dst_root, e.rel);
        bool was_dir = false;
        int rc = unlink_if_exists(p, &was_dir);
        if (rc) return rc;
        if (was_dir && rmdir(p.c_str()) != 0) return fail(VMIG_EIO, "rmdir %s (symlink over directory): %s", p.c_str(), errno_str(errno).c_str());
        if (symlink(e.target.c_str(), p.c_str()) != 0) return fail(VMIG_EIO, "symlink %s: %s", p.c_str(), errno_str(errno).c_str());
        if (!pol.no_metadata) {
            if (pol.is_root && lchown(p.c_str(), e.uid, e.gid) != 0) return fail(VMIG_EIO, "lchown %s: %s", p.c_str(), errno_str(errno).c_str());
            fill_times(e, pol, ts);
            if (utimensat(AT_FDCWD, p.c_str(), ts, AT_SYMLINK_NOFOLLOW) != 0) return fail(VMIG_EIO, "utimensat %s: %s", p.c_str(), errno_str(errno).c_str());
        }
        if (n_symlinks) (*n_symlinks)++;
    }
    for (const auto& e : m.specials) {
        const std::string p = join(dst_root, e.rel);
        bool was_dir = false;
        int rc = unlink_if_exists(p, &was_dir);
        if (rc) return rc;
        if (was_dir && rmdir(p.c_str()) != 0) return fail(VMIG_EIO, "rmdir %s: %s", p.c_str(), errno_str(errno).c_str());
        if (mknod(p.c_str(), (e.mode & S_IFMT) | 0600, e.rdev) != 0) return fail(VMIG_EIO, "mknod %s: %s", p.c_str(), errno_str(errno).c_str());
        rc = apply_file_meta(-1, p, e, pol);
        if (rc) return rc;
        if (n_specials) (*n_specials)++;
    }
    for (const auto& e : m.files) {
        if (e.hardlink_of < 0) continue;
        const std::string p = join(dst_root, e.rel);
        const std::string prim = join(dst_root, m.files[(size_t)e.hardlink_of].rel);
        bool was_dir = false;
        int rc = unlink_if_exists(p, &was_dir);
        if (rc) return rc;
        if (was_dir) return fail(VMIG_EIO, "%s: directory in the way of a hard link", p.c_str());
        if (link(prim.c_str(), p.c_str()) != 0) return fail(VMIG_EIO, "link %s -> %s: %s", p.c_str(), prim.c_str(), errno_str(errno).c_str());
        if (n_hardlinks) (*n_hardlinks)++;
    }
    if (!pol.no_metadata) {
        for (size_t i = m.dirs.size(); i-- > 0;) {     // children before parents
            const Entry& e = m.dirs[i];
            const std::string p = join(dst_root, e.rel);
            if (pol.is_root && chown(p.c_str(), e.uid, e.gid) != 0) return fail(VMIG_EIO, "chown %s: %s", p.c_str(), errno_str(errno).c_str());
            if (chmod(p.c_str(), eff_mode(e, pol)) != 0) return fail(VMIG_EIO, "chmod %s: %s", p.c_str(), errno_str(errno).c_str());
            fill_times(e, pol, ts);
            if (utimensat(AT_FDCWD, p.c_str(), ts, 0) != 0) return fail(VMIG_EIO, "utimensat %s: %s", p.c_str(), errno_str(errno).c_str());
        }
    }
    return VMIG_OK;
}

int remove_source(const std::string& src_root, const Manifest& m)
{
    // unlinkat() relative to the entry's parent directory, itself re-opened beneath the root without following
    // symlinks: a path swapped under us can make the call fail, not delete something outside the tree
    const int rfd = open(src_root.c_str(), O_RDONLY | O_DIRECTORY | O_CLOEXEC);
    if (rfd < 0) return fail(VMIG_EIO, "open %s: %s", src_root.c_str(), errno_str(errno).c_str());
    std::string cur_parent = "\x01"; int pfd = -1;
    auto parent_of = [&](const std::string& rel, std::string* base) -> int {
        const size_t slash = rel.rfind('/');
        const std::string parent = slash == std::string::npos ? "." : rel.substr(0, slash);
        *base = slash == std::string::npos ? rel : rel.substr(slash + 1);
        if (parent == cur_parent) return VMIG_OK;
        if (pfd >= 0 && pfd != rfd) close(pfd);
        pfd = -1; cur_parent = "\x01";
        if (parent == ".") pfd = rfd;
        else { int rc = open_beneath(rfd, parent, O_RDONLY | O_DIRECTORY, &pfd); if (rc) return rc; }
        cur_parent = parent;
        return VMIG_OK;
    };
    auto finish = [&](int rc) { if (pfd >= 0 && pfd != rfd) close(pfd); close(rfd); return rc; };
    auto rm = [&](const std::vector<Entry>& v) -> int {
        for (const auto& e : v) {
            std::string base;
            int rc = parent_of(e.rel, &base);
            if (rc) return rc;
            if (unlinkat(pfd, base.c_str(), 0) != 0 && errno != ENOENT) return fail(VMIG_EIO, "unlink %s: %s", e.rel.c_str(), errno_str(errno).c_str());
        }
        return VMIG_OK;
    };
    int rc;
    if ((rc = rm(m.files)) || (rc = rm(m.symlinks)) || (rc = rm(m.specials))) return finish(rc);
    for (size_t i = m.dirs.size(); i-- > 1;) {
        std::string base;
        rc = parent_of(m.dirs[i].rel, &base);
        if (rc) return finish(rc);
        if (unlinkat(pfd, base.c_str(), AT_REMOVEDIR) != 0 && errno != ENOENT && errno != ENOTEMPTY)
            return finish(fail(VMIG_EIO, "rmdir %s: %s", m.dirs[i].rel.c_str(), errno_str(errno).c_str()));
    }
    return finish(VMIG_OK);
}

// ---------------------------------------------------------------------------------------------
// VMIG_F_PRUNE: make the destination hold nothing the source does not (the final pass of a hand-off: a file the
// tenant deleted or renamed between the live pass and the paused pass must not reappear in the new container).
static int rm_tree_at(int dfd, const char* name, uint64_t* n)
{
    int fd = openat(dfd, name, O_RDONLY | O_DIRECTORY | O_NOFOLLOW | O_CLOEXEC);
    if (fd < 0) return fail(VMIG_EIO, "prune: open %s: %s", name, errno_str(errno).c_str());
    DIR* d = fdopendir(fd);
    if (!d) { close(fd); return fail(VMIG_EIO, "prune: fdopendir %s: %s", name, errno_str(errno).c_str()); }
    int rc = VMIG_OK;
    while (struct dirent* de = readdir(d)) {
        if (!strcmp(de->d_name, ".") || !strcmp(de->d_name, "..")) continue;
        struct stat st;
        if (fstatat(fd, de->d_name, &st, AT_SYMLINK_NOFOLLOW) != 0) continue;
        if (S_ISDIR(st.st_mode)) { rc = rm_tree_at(fd, de->d_name, n); if (rc) break; }
        else if (unlinkat(fd, de->d_name, 0) != 0 && errno != ENOENT) { rc = fail(VMIG_EIO, "prune: unlink %s: %s", de->d_name, errno_str(errno).c_str()); break; }
        else (*n)++;
    }
    closedir(d);
    if (rc) return rc;
    if (unlinkat(dfd, name, AT_REMOVEDIR) != 0 && errno != ENOENT) return fail(VMIG_EIO, "prune: rmdir %s: %s", name, errno_str(errno).c_str());
    (*n)++;
    return VMIG_OK;
}

static int prune_dir(int dfd, const std::string& prefix, const std::unordered_set<std::string>& keep_dirs,
                     const std::unordered_set<std::string>& keep_other, bool dry, uint64_t* n)
{
    DIR* d = fdopendir(dfd);                       // takes ownership of dfd
    if (!d) { close(dfd); return fail(VMIG_EIO, "prune: fdopendir: %s", errno_str(errno).c_str()); }
    int rc = VMIG_OK;
    std::vector<std::string> names;
    while (struct dirent* de = readdir(d)) if (strcmp(de->d_name, ".") && strcmp(de->d_name, "..")) names.push_back(de->d_name);
    for (const auto& name : names) {
        const std::string rel = prefix.empty() ? name : prefix + "/" + name;
        struct stat st;
        if (fstatat(dfd, name.c_str(), &st, AT_SYMLINK_NOFOLLOW) != 0) continue;
        if (S_ISDIR(st.st_mode) && keep_dirs.count(rel)) {
            int sub = openat(dfd, name.c_str(), O_RDONLY | O_DIRECTORY | O_NOFOLLOW | O_CLOEXEC);
            if (sub < 0) { rc = fail(VMIG_EIO, "prune: open %s: %s", rel.c_str(), errno_str(errno).c_str()); break; }
            rc = prune_dir(sub, rel, keep_dirs, keep_other, dry, n);
            if (rc) break;
            continue;
        }
        if (!S_ISDIR(st.st_mode) && keep_other.count(rel)) continue;
        if (dry) { (*n)++; continue; }
        if (S_ISDIR(st.st_mode)) { rc = rm_tree_at(dfd, name.c_str(), n); if (rc) break; }
        else if (unlinkat(dfd, name.c_str(), 0) != 0 && errno != ENOENT) { rc = fail(VMIG_EIO, "prune: unlink %s: %s", rel.c_str(), errno_str(errno).c_str()); break; }
        else (*n)++;
    }
    closedir(d);
    return rc;
}

int prune_extras(const std::string& dst_root, const Manifest& m, bool dry_run, uint64_t* n_extras)
{
    std::unordered_set<std::string> keep_dirs, keep_other;
    keep_dirs.reserve(m.dirs.size() * 2); keep_other.reserve((m.files.size() + m.symlinks.size() + m.specials.size()) * 2);
    for (auto& e : m.dirs) keep_dirs.insert(e.rel);
    for (auto& e : m.files) keep_other.insert(e.rel);
    for (auto& e : m.symlinks) keep_other.insert(e.rel);
    for (auto& e : m.specials) keep_other.insert(e.rel);
    *n_extras = 0;
    int fd = open(dst_root.c_str(), O_RDONLY | O_DIRECTORY | O_CLOEXEC);
    if (fd < 0) return fail(VMIG_EIO, "prune: open %s: %s", dst_root.c_str(), errno_str(errno).c_str());
    return prune_dir(fd, "", keep_dirs, keep_other, dry_run, n_extras);
}

}  // namespace vmig
