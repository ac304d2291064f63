// tests/xfer_unit.cpp -- CPU unit test of transfer_block() in csrc/vmig_common.h, the loop every file read and write of
// libvmig goes through (pread / pwrite, cuFileRead / cuFileWrite): compiled and run by
// tests/test_host.py::test_block_transfer_loop.  A scripted fake transfer stands in for the system call, so the
// branches a real filesystem rarely takes -- a short transfer in the middle of an O_DIRECT block -- run here.
#include "vmig_common.h"
#include <algorithm>
#include <cstdlib>
#include <vector>

namespace vmig {   // the error-channel functions normally provided by vmig_engine.cu
static thread_local std::string g_err;
void set_last_error(const char* fmt, ...) { char b[1024]; va_list ap; va_start(ap, fmt); vsnprintf(b, sizeof b, fmt, ap); va_end(ap); g_err = b; }
void set_last_error_str(const std::string& s) { g_err = s; }
const char* last_error_cstr() { return g_err.c_str(); }
long env_long(const char* name, long d) { const char* v = getenv(name); return v && *v ? atol(v) : d; }
}
using namespace vmig;

#define CHECK(c) do { if (!(c)) { printf("FAIL line %d: %s   [last error: %s]\n", __LINE__, #c, last_error_cstr()); return 1; } } while (0)

// A file of `size` bytes read into a block buffer; each call moves at most the next scripted count (or returns it when
// it is <= 0), never past EOF, and records the buffer offset, file offset and length it was asked for.
struct FakeRead {
    std::vector<uint8_t> file, buf;
    std::vector<ssize_t> script;
    struct Call { size_t buf_off; uint64_t file_off; size_t n; };
    std::vector<Call> calls;
    FakeRead(size_t size, size_t buf_size) : file(size), buf(buf_size, 0xEE) { for (size_t i = 0; i < size; i++) file[i] = (uint8_t)(i * 131 + 7); }
    int run(uint64_t file_off, size_t len, size_t align, int stuck) {
        return transfer_block("f.bin", file_off, len, align, stuck, [&](size_t pos, size_t n) -> ssize_t {
            calls.push_back({pos, file_off + pos, n});
            const ssize_t cap = calls.size() <= script.size() ? script[calls.size() - 1] : (ssize_t)n;
            if (cap <= 0) return cap;
            const uint64_t at = file_off + pos;
            const size_t m = std::min({(size_t)cap, n, at < file.size() ? (size_t)(file.size() - at) : (size_t)0});
            memcpy(buf.data() + pos, file.data() + at, m);
            return (ssize_t)m;
        });
    }
    bool holds(uint64_t file_off, size_t len) const { return memcmp(buf.data(), file.data() + file_off, len) == 0; }
};

int main()
{
    {   // buffered: a short transfer resumes at the exact byte
        FakeRead f(1 << 20, 10000); f.script = {3001, 4000};
        CHECK(f.run(8192, 10000, 0, VMIG_ESRCCHANGED) == VMIG_OK);
        CHECK(f.calls.size() == 3);
        CHECK(f.calls[0].buf_off == 0 && f.calls[0].file_off == 8192 && f.calls[0].n == 10000);
        CHECK(f.calls[1].buf_off == 3001 && f.calls[1].file_off == 8192 + 3001 && f.calls[1].n == 6999);
        CHECK(f.calls[2].buf_off == 7001 && f.calls[2].file_off == 8192 + 7001 && f.calls[2].n == 2999);
        CHECK(f.holds(8192, 10000));
    }
    {   // O_DIRECT: whole sectors; a short transfer resumes from the last sector boundary it reached
        FakeRead f(1 << 20, 3 * 4096); f.script = {5000};
        CHECK(f.run(4096, 10000, 4096, VMIG_ESRCCHANGED) == VMIG_OK);
        CHECK(f.calls.size() == 2);
        CHECK(f.calls[0].buf_off == 0 && f.calls[0].file_off == 4096 && f.calls[0].n == 3 * 4096);
        CHECK(f.calls[1].buf_off == 4096 && f.calls[1].file_off == 2 * 4096 && f.calls[1].n == 2 * 4096);
        CHECK(f.holds(4096, 3 * 4096));
    }
    {   // O_DIRECT, resume exactly on a boundary: 8192 moved, the next call starts there
        FakeRead f(1 << 20, 3 * 4096); f.script = {8192};
        CHECK(f.run(0, 3 * 4096, 4096, VMIG_ESRCCHANGED) == VMIG_OK);
        CHECK(f.calls.size() == 2 && f.calls[1].buf_off == 8192 && f.calls[1].file_off == 8192 && f.calls[1].n == 4096);
    }
    {   // O_DIRECT, the file's short last block: asks for the whole sector, EOF returns fewer bytes, no error
        FakeRead f(4096 + 1234, 2 * 4096);
        CHECK(f.run(4096, 1234, 4096, VMIG_ESRCCHANGED) == VMIG_OK);
        CHECK(f.calls.size() == 1 && f.calls[0].buf_off == 0 && f.calls[0].file_off == 4096 && f.calls[0].n == 4096);
        CHECK(f.holds(4096, 1234));
    }
    {   // a zero-length block moves nothing
        FakeRead f(4096, 4096);
        CHECK(f.run(0, 0, 4096, VMIG_ESRCCHANGED) == VMIG_OK && f.calls.empty());
    }
    {   // a transfer that returns 0 fails with the code passed in and says where
        set_last_error_str("");
        FakeRead f(1 << 20, 4096); f.script = {100, 0};
        CHECK(f.run(0, 4096, 0, VMIG_ESRCCHANGED) == VMIG_ESRCCHANGED);
        CHECK(f.calls.size() == 2);
        CHECK(strstr(last_error_cstr(), "f.bin") && strstr(last_error_cstr(), "100 of 4096"));
        set_last_error_str("");
        FakeRead g(1 << 20, 4096); g.script = {0};
        CHECK(g.run(0, 4096, 0, VMIG_EIO) == VMIG_EIO && *last_error_cstr());
    }
    {   // O_DIRECT: a retry from the sector boundary that ends at or before what was already there is no progress
        set_last_error_str("");
        FakeRead f(1 << 20, 2 * 4096); f.script = {5000, 904};
        CHECK(f.run(0, 2 * 4096, 4096, VMIG_EIO) == VMIG_EIO);
        CHECK(f.calls.size() == 2 && f.calls[1].buf_off == 4096 && *last_error_cstr());
    }
    {   // a negative result is the transfer's own VMIG_E* code, passed through with its message
        set_last_error_str("");
        FakeRead f(1 << 20, 4096); f.script = {2000, fail(VMIG_EIO, "pread f.bin: Input/output error")};
        CHECK(f.run(0, 4096, 0, VMIG_ESRCCHANGED) == VMIG_EIO);
        CHECK(std::string(last_error_cstr()) == "pread f.bin: Input/output error");
        FakeRead g(1 << 20, 4096); g.script = {VMIG_EINVAL};
        CHECK(g.run(0, 4096, 4096, VMIG_ESRCCHANGED) == VMIG_EINVAL);
    }
    printf("xfer unit ok\n");
    return 0;
}
