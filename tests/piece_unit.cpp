// tests/piece_unit.cpp -- CPU unit test of the piece split in csrc/vmig_common.h (piece_count / block_piece): how a
// reader cuts the blocks of a slot into the windows it stages through its pinned pieces.  Compiled and run by
// tests/test_piece_staging.py::test_piece_split.
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

#define CHECK(c) do { if (!(c)) { printf("FAIL line %d: %s   [at %zu len %zu]\n", __LINE__, #c, at, len); return 1; } } while (0)

static constexpr size_t S = 1u << 20, kSector = 4096;

// Every part of a block of `len` bytes at slot offset `at`: the parts tile [0, len) in order, each lies in one window,
// windows are consecutive, and the O_DIRECT read length is whole sectors and ends inside the window when `at` is.
static int check_split(size_t at, size_t len, size_t piece) {
    const size_t np = piece_count(at, len, piece);
    CHECK(np >= 1 && (len == 0 || np == (at + len - 1) / piece - at / piece + 1));
    size_t got = 0;
    for (size_t k = 0; k < np; k++) {
        const Piece b = block_piece(at, len, piece, 0, k), d = block_piece(at, len, piece, kSector, k);
        CHECK(b.off == got && d.off == got && b.len == d.len && b.window == d.window);
        CHECK(b.window == at / piece + k);
        CHECK(b.io_len == b.len);
        CHECK(len == 0 || b.len > 0);
        const size_t in_win = at + b.off - b.window * piece;
        CHECK(in_win + b.len <= piece);
        CHECK(k == 0 || in_win == 0);                           // every part after the first starts its window
        CHECK(k + 1 == np || in_win + b.len == piece);          // every part before the last fills its window to the end
        CHECK(d.io_len % kSector == 0 && d.io_len >= d.len && d.io_len - d.len < kSector);
        if (at % kSector == 0 && piece % kSector == 0) CHECK(in_win + d.io_len <= piece);
        got += b.len;
    }
    CHECK(got == len);
    return 0;
}

// A slot laid out as the engine lays it out (blocks at `align`-multiple offsets), filled from a source the way a reader
// fills it: each window in a piece buffer through transfer_block with a pread-like fake that stops at the file's end,
// then the filled range [lo, hi) copied into the slot.  Every block's bytes arrive where the slot layout puts them.
static int stage_slot(const std::vector<size_t>& lens, size_t align, bool eof_after_each) {
    size_t at = 0, len = 0;
    std::vector<size_t> offs;
    for (size_t l : lens) { offs.push_back(at); at += align_up(l ? l : 1, align); }
    const size_t slot_bytes = align_up(at, S);
    std::vector<uint8_t> slot(slot_bytes, 0xEE), piece(S);
    for (size_t i = 0; i < lens.size(); i++) {
        at = offs[i]; len = lens[i];
        // the block's source: its own file when eof_after_each (every block is a file's short last block)
        std::vector<uint8_t> src(len);
        for (size_t j = 0; j < len; j++) src[j] = (uint8_t)(i * 7 + j * 131 + 3);
        for (size_t k = 0; k < piece_count(at, len, S); k++) {
            const Piece pc = block_piece(at, len, S, align == kSector ? kSector : 0, k);
            const size_t in_win = at + pc.off - pc.window * S;
            size_t first_ask = 0; bool inside = true;
            int rc = transfer_block("f.bin", pc.off, pc.len, align == kSector ? kSector : 0, VMIG_ESRCCHANGED, [&](size_t pos, size_t n) -> ssize_t {
                if (!first_ask) first_ask = n;
                const size_t from = pc.off + pos, have = eof_after_each ? len : len + (1u << 30);
                const size_t m = from < have ? std::min(n, have - from) : 0;
                inside = inside && in_win + pos + n <= S;      // the read never runs past the piece
                for (size_t j = 0; j < m && from + j < len; j++) piece[in_win + pos + j] = src[from + j];
                return (ssize_t)m;
            });
            CHECK(rc == VMIG_OK && inside && (pc.len == 0 || first_ask == pc.io_len));
            memcpy(slot.data() + pc.window * S + in_win, piece.data() + in_win, pc.len);
        }
        CHECK(memcmp(slot.data() + at, src.data(), len) == 0);
    }
    return 0;
}

int main() {
    const size_t lens[] = {0, 1, 4095, 4096, 4097, S - 1, S, S + 1, 3 * S + 17, (4u << 20) - 1, 4u << 20};
    const size_t ats[] = {0, 512, 4096, S - 4096, S, 3 * S + 8192, (32u << 20) - (4u << 20)};
    for (size_t len : lens)
        for (size_t at : ats)
            for (size_t piece : {S, (size_t)64 << 10})
                if (check_split(at, len, piece)) return 1;
    {   // a short last block in the middle of a window: one part, rounded up to one sector under O_DIRECT
        const size_t at = S + 8192, len = 100;
        const Piece p = block_piece(at, len, S, kSector, 0);
        CHECK(piece_count(at, len, S) == 1 && p.window == 1 && p.off == 0 && p.len == 100 && p.io_len == kSector);
        // 2.5 MiB starting half-way into window 2: windows 2, 3 and 4, the middle one whole
        const Piece a = block_piece(2 * S + S / 2, 5 * S / 2, S, kSector, 0), b = block_piece(2 * S + S / 2, 5 * S / 2, S, kSector, 1),
                    c = block_piece(2 * S + S / 2, 5 * S / 2, S, kSector, 2);
        CHECK(piece_count(2 * S + S / 2, 5 * S / 2, S) == 3 && a.len == S / 2 && b.len == S && c.len == S && c.window == 4);
    }
    // many small blocks share windows; large ones span several; both with the buffered and the O_DIRECT layout
    std::vector<size_t> mix;
    for (size_t i = 0; i < 200; i++) mix.push_back(1 + (i * 7919) % (300u << 10));
    for (size_t l : {(size_t)0, (size_t)1, S - 1, S + 1, 3 * S + 17, (size_t)(4u << 20) - 1, (size_t)(4u << 20)}) mix.push_back(l);
    for (size_t align : {(size_t)512, kSector})
        for (bool eof : {false, true})
            if (stage_slot(mix, align, eof)) { printf("  align %zu eof %d\n", align, (int)eof); return 1; }
    printf("piece unit ok\n");
    return 0;
}
