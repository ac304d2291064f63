// vmig_common.h -- shared host-side helpers of libvmig (errors, timing, small utilities).
#pragma once
#include <stdint.h>
#include <sys/types.h>
#include <string>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cerrno>
#include <cstring>
#include "../../include/vmig.h"

namespace vmig {

// Thread-local detail of the last failure on this thread (vmig_last_error()).
void set_last_error(const char* fmt, ...) __attribute__((format(printf, 1, 2)));
void set_last_error_str(const std::string& s);
const char* last_error_cstr();

inline uint64_t now_ns() {
    return (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(
               std::chrono::steady_clock::now().time_since_epoch()).count();
}

inline int fail(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
inline int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    set_last_error_str(buf);
    return code;
}

inline std::string errno_str(int e) { char b[128]; return std::string(strerror_r(e, b, sizeof b)); }

inline uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

// Moves the `len` bytes of a block at file offset `file_off` through op(pos, n) -> bytes moved, or a negative VMIG_E*
// code, for the n bytes at offset pos inside the block.  `name` and `file_off` only label the error.
//   align == 0: buffered I/O; a short transfer resumes at the exact byte.
//   align != 0 (an O_DIRECT descriptor: buffer, offset and length in whole sectors): every transfer runs to the
//     rounded-up end of the block, so the file's short last block reads or writes past EOF and simply moves fewer
//     bytes; a short transfer inside the block resumes from the last sector boundary it reached.
// A transfer that moves nothing new fails with `stuck` (VMIG_ESRCCHANGED for a source that shrank under a reader).
template <class Op>
inline int transfer_block(const char* name, uint64_t file_off, size_t len, size_t align, int stuck, Op&& op) {
    const size_t want = align ? (size_t)align_up(len, align) : len;
    size_t done = 0;
    while (done < len) {
        const size_t pos = align ? (done & ~(align - 1)) : done;
        const ssize_t r = op(pos, want - pos);
        if (r < 0) return (int)r;
        if (r == 0 || pos + (size_t)r <= done)
            return fail(stuck, "%s: no progress after %zu of %zu bytes at offset %llu", name, done, len, (unsigned long long)file_off);
        done = pos + (size_t)r;
    }
    return VMIG_OK;
}

// Readers stage a slot in windows of `piece` bytes: window w is slot bytes [w * piece, (w + 1) * piece), filled in one
// pinned piece and copied to the GPU in one go, so that consecutive small blocks share a copy.  A block at slot offset
// `at` is read in the parts that fall in successive windows; an empty block is one empty part, so that every block is
// read exactly once whatever its length.
struct Piece {
    size_t window;   // index of the window
    size_t off;      // offset of the part inside the block
    size_t len;      // bytes of the block in this part
    size_t io_len;   // what the read asks for: len rounded up to whole sectors when align != 0 (O_DIRECT), which the
                     // file's short last block reads past EOF.  With `at` and `piece` whole sectors, the read ends
                     // inside its window
};
inline size_t piece_count(size_t at, size_t len, size_t piece) { return len ? (at + len - 1) / piece - at / piece + 1 : 1; }
inline Piece block_piece(size_t at, size_t len, size_t piece, size_t align, size_t k) {
    const size_t w = at / piece + k, w0 = w * piece, w1 = w0 + piece;
    const size_t start = at > w0 ? at : w0, end = at + len < w1 ? at + len : w1;
    const size_t n = end > start ? end - start : 0;
    return {w, start - at, n, align ? (size_t)align_up(n, align) : n};
}

long env_long(const char* name, long dflt);

}  // namespace vmig
