// tree_unit.cpp -- CPU unit test of the source-side path safety in csrc/vmig_tree.cpp (compiled and run by
// tests/test_host.py).  The source layer may belong to a running tenant: open_beneath() must refuse symlinks and
// escapes, the walk must not descend through a symlinked directory, remove_source() must not leave the tree.
//   g++ -std=c++17 -I gpu-docker-api_b200/csrc tests/tree_unit.cpp gpu-docker-api_b200/csrc/vmig_tree.cpp -o tree_unit
#include "vmig_tree.h"
#include "vmig_common.h"
#include <fcntl.h>
#include <unistd.h>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <sys/stat.h>

namespace vmig {   // the three error-channel functions normally provided by vmig_engine.cu
static thread_local std::string g_err;
void set_last_error(const char* fmt, ...) { char b[1024]; va_list ap; va_start(ap, fmt); vsnprintf(b, sizeof b, fmt, ap); va_end(ap); g_err = b; }
void set_last_error_str(const std::string& s) { g_err = s; }
const char* last_error_cstr() { return g_err.c_str(); }
long env_long(const char* name, long d) { const char* v = getenv(name); return v && *v ? atol(v) : d; }
}
using namespace vmig;

#define CHECK(c) do { if (!(c)) { printf("FAIL line %d: %s   [last error: %s]\n", __LINE__, #c, last_error_cstr()); return 1; } } while (0)
static void put(const std::string& p, const char* s) { FILE* f = fopen(p.c_str(), "w"); fputs(s, f); fclose(f); }
static std::string get(int fd) { char b[64] = {0}; ssize_t n = read(fd, b, 63); close(fd); return std::string(b, n > 0 ? (size_t)n : 0); }

int main(int argc, char** argv) {
    if (argc < 2) return 2;
    const std::string base = argv[1], root = base + "/root", outside = base + "/outside";
    CHECK(system(("mkdir -p " + root + "/a/b " + root + "/victim " + outside).c_str()) == 0);
    put(root + "/a/b/file", "inside"); put(root + "/victim/f", "inside2"); put(outside + "/f", "SECRET"); put(outside + "/secret", "SECRET");
    CHECK(symlink(outside.c_str(), (root + "/a/link").c_str()) == 0);
    CHECK(symlink("b/file", (root + "/a/sl").c_str()) == 0);
    const int rfd = open(root.c_str(), O_RDONLY | O_DIRECTORY);
    CHECK(rfd >= 0);
    int fd = -1;
    CHECK(open_beneath(rfd, "a/b/file", O_RDONLY, &fd) == VMIG_OK && get(fd) == "inside");
    CHECK(open_beneath(rfd, "a/link/secret", O_RDONLY, &fd) == VMIG_ESRCCHANGED);        // symlinked directory on the way
    CHECK(open_beneath(rfd, "a/sl", O_RDONLY, &fd) == VMIG_ESRCCHANGED);                 // symlink as the last component
    CHECK(open_beneath(rfd, "../outside/secret", O_RDONLY, &fd) != VMIG_OK);             // lexical escape
    CHECK(open_beneath(rfd, "/etc/passwd", O_RDONLY, &fd) == VMIG_EINVAL);               // absolute
    CHECK(open_beneath(rfd, "a/missing", O_RDONLY, &fd) == VMIG_ESRCCHANGED);            // vanished since the walk

    // the same through the component-wise fallback used on kernels without openat2
    CHECK(open_beneath_walk(rfd, "a/b/file", O_RDONLY, &fd) == VMIG_OK && get(fd) == "inside");
    CHECK(open_beneath_walk(rfd, "a/link/secret", O_RDONLY, &fd) == VMIG_ESRCCHANGED);
    CHECK(open_beneath_walk(rfd, "a/sl", O_RDONLY, &fd) == VMIG_ESRCCHANGED);
    CHECK(open_beneath_walk(rfd, "../outside/secret", O_RDONLY, &fd) == VMIG_EINVAL);
    CHECK(open_beneath_walk(rfd, "a/missing", O_RDONLY, &fd) == VMIG_ESRCCHANGED);

    Manifest m;
    CHECK(walk_tree(root, 4096, false, &m) == VMIG_OK);
    CHECK(m.files.size() == 2 && m.symlinks.size() == 2 && m.dirs.size() == 4);          // ".", a, a/b, victim; nothing from outside/
    for (auto& e : m.files) CHECK(e.rel == "a/b/file" || e.rel == "victim/f");

    // the tenant swaps victim/ for a symlink to outside/ after the walk: the file must not be reachable any more,
    // and a move's clean-up must not delete outside/f
    CHECK(rename((root + "/victim").c_str(), (root + "/victim.bak").c_str()) == 0);
    CHECK(symlink(outside.c_str(), (root + "/victim").c_str()) == 0);
    CHECK(open_beneath(rfd, "victim/f", O_RDONLY, &fd) == VMIG_ESRCCHANGED);
    CHECK(remove_source(root, m) != VMIG_OK);
    CHECK(access((outside + "/f").c_str(), F_OK) == 0);
    close(rfd);

    // ---- VMIG_F_PRUNE: prune_extras() removes exactly what the manifest does not list, by descriptor, never through a symlink
    {
        const std::string psrc = base + "/psrc", pdst = base + "/pdst";
        CHECK(system(("mkdir -p " + psrc + "/keep/sub " + pdst + "/keep/sub " + pdst + "/gone/deep " + pdst + "/keep/extra_dir").c_str()) == 0);
        put(psrc + "/keep/f", "1"); put(psrc + "/keep/sub/g", "2"); put(psrc + "/top", "3");
        CHECK(symlink("keep/f", (psrc + "/ln").c_str()) == 0);
        put(pdst + "/keep/f", "old"); put(pdst + "/keep/sub/g", "old"); put(pdst + "/top", "old"); CHECK(symlink("keep/f", (pdst + "/ln").c_str()) == 0);
        put(pdst + "/gone/deep/x", "x"); put(pdst + "/keep/stale", "s"); put(pdst + "/keep/extra_dir/y", "y");
        CHECK(symlink(outside.c_str(), (pdst + "/escape").c_str()) == 0);                 // an extra that points out of the tree
        CHECK(symlink(outside.c_str(), (pdst + "/gone/deep/esc2").c_str()) == 0);
        Manifest pm;
        CHECK(walk_tree(psrc, 4096, false, &pm) == VMIG_OK);
        uint64_t n = 0;
        CHECK(prune_extras(pdst, pm, true, &n) == VMIG_OK && n == 4);                     // dry run: gone/, keep/stale, keep/extra_dir/, escape
        CHECK(access((pdst + "/gone/deep/x").c_str(), F_OK) == 0);                        // ... and nothing was touched
        CHECK(prune_extras(pdst, pm, false, &n) == VMIG_OK);
        CHECK(n == 8);                          // gone/deep/{x,esc2}, gone/deep, gone, keep/stale, keep/extra_dir/y, keep/extra_dir, escape
        CHECK(access((pdst + "/gone").c_str(), F_OK) != 0 && access((pdst + "/keep/stale").c_str(), F_OK) != 0 && access((pdst + "/keep/extra_dir").c_str(), F_OK) != 0);
        struct stat lst; CHECK(lstat((pdst + "/escape").c_str(), &lst) != 0);
        CHECK(access((outside + "/f").c_str(), F_OK) == 0 && access((outside + "/secret").c_str(), F_OK) == 0);   // the symlinks were unlinked, not followed
        CHECK(access((pdst + "/keep/sub/g").c_str(), F_OK) == 0 && access((pdst + "/top").c_str(), F_OK) == 0 && lstat((pdst + "/ln").c_str(), &lst) == 0);
        CHECK(prune_extras(pdst, pm, true, &n) == VMIG_OK && n == 0);
        // an entry that changed TYPE since the destination was written is in the way and goes too: a file where the source
        // now has a directory, a directory (with content) where the source now has a file, a directory where it has a symlink
        CHECK(system(("mkdir -p " + psrc + "/flip_dir " + pdst + "/flip_file/inner " + pdst + "/ln2").c_str()) == 0);
        put(psrc + "/flip_file", "now a file"); put(pdst + "/flip_dir", "was a file"); put(pdst + "/flip_file/inner/z", "z");
        CHECK(symlink("top", (psrc + "/ln2").c_str()) == 0);
        CHECK(walk_tree(psrc, 4096, false, &pm) == VMIG_OK);
        CHECK(prune_extras(pdst, pm, false, &n) == VMIG_OK && n == 5);            // flip_dir (file), flip_file/{inner/z, inner}, flip_file, ln2 (dir)
        struct stat fst;
        CHECK(lstat((pdst + "/flip_dir").c_str(), &fst) != 0 && lstat((pdst + "/flip_file").c_str(), &fst) != 0 && lstat((pdst + "/ln2").c_str(), &fst) != 0);
        CHECK(make_dirs(pdst, pm) == VMIG_OK && lstat((pdst + "/flip_dir").c_str(), &fst) == 0 && S_ISDIR(fst.st_mode));
    }

    // ---- the walk is the same whether the root's sub-directories are taken by one thread or by eight
    {
        const std::string w = base + "/wide";
        CHECK(system(("mkdir -p " + w).c_str()) == 0);
        for (int d = 0; d < 11; d++) {
            const std::string dd = w + "/d" + std::to_string(d);
            CHECK(system(("mkdir -p " + dd + "/x/y").c_str()) == 0);
            for (int f = 0; f < 7; f++) put(dd + (f % 2 ? "/x/y/f" : "/f") + std::to_string(f), "data");
            CHECK(symlink("f0", (dd + "/sl").c_str()) == 0);
        }
        CHECK(link((w + "/d3/f0").c_str(), (w + "/d9/hard").c_str()) == 0);               // a hard-link pair across two sub-walks
        Manifest a, b;
        setenv("VMIG_WALK_THREADS", "1", 1); CHECK(walk_tree(w, 4096, false, &a) == VMIG_OK);
        setenv("VMIG_WALK_THREADS", "8", 1); CHECK(walk_tree(w, 4096, false, &b) == VMIG_OK);
        CHECK(a.dirs.size() == b.dirs.size() && a.files.size() == b.files.size() && a.symlinks.size() == b.symlinks.size() && a.files.size() == 78);
        for (size_t i = 0; i < a.dirs.size(); i++) CHECK(a.dirs[i].rel == b.dirs[i].rel);
        for (size_t i = 0; i < a.files.size(); i++) CHECK(a.files[i].rel == b.files[i].rel && a.files[i].hardlink_of == b.files[i].hardlink_of && a.files[i].first_block == b.files[i].first_block);
        for (size_t i = 0; i < a.symlinks.size(); i++) CHECK(a.symlinks[i].rel == b.symlinks[i].rel);
        int links = 0; for (auto& e : b.files) if (e.hardlink_of >= 0) { links++; CHECK(b.files[(size_t)e.hardlink_of].rel == "d3/f0" && e.rel == "d9/hard"); }
        CHECK(links == 1);
    }

    // ---- metadata as an ordinary user, like tar without -p: the umask applies, setuid/setgid/sticky bits are dropped
    {
        const std::string d = base + "/modes", f = d + "/suid";
        CHECK(mkdir(d.c_str(), 0700) == 0);
        put(f, "x");
        const MetaPolicy pol{false, 022, false, false, false};
        Entry e;
        e.mtime = {1577934245, 0}; e.atime = {0, 0};
        struct stat st;
        e.rel = "modes/suid"; e.type = kFile; e.mode = S_IFREG | 04770;
        CHECK(apply_file_meta(-1, f, e, pol) == VMIG_OK && stat(f.c_str(), &st) == 0 && (st.st_mode & 07777) == 0750);
        e.rel = "modes"; e.type = kDir; e.mode = S_IFDIR | 03777;
        CHECK(apply_file_meta(-1, d, e, pol) == VMIG_OK && stat(d.c_str(), &st) == 0 && (st.st_mode & 07777) == 0755);
    }
    printf("tree unit ok\n");
    return 0;
}
