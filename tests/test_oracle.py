"""CPU: the oracle is pinned before it is trusted (spec ③).

The reference has no tests, fixtures or hashing (SURVEY.md §4, F3): the byte oracle is the
reference's literal shell pipeline (utils/copy.go:18,116), the hash oracle is the public XXH64
spec pinned by the known-answer vectors in tests/golden/xxh64_kat.json (SURVEY.md Appendix A)."""
import json
import os
import stat
from pathlib import Path

import numpy as np
import pytest

from conftest import make_rich_tree

KAT = json.loads((Path(__file__).parent / "golden" / "xxh64_kat.json").read_text())


def test_xxh64_restatement_matches_known_answers(orc):
    buf = orc.sanity_buffer(4 << 20)
    for n, want in KAT["sanity"].items():
        assert orc.xxh64(buf[: int(n)]) == int(want, 16), n
    for s, want in KAT["ascii"].items():
        assert orc.xxh64(s.encode()) == int(want, 16)
    assert orc.xxh64(bytes(4 << 20)) == int(KAT["zeros_4MiB"], 16)


def test_pure_python_restatement_agrees(orc):
    buf = orc.sanity_buffer(5000)
    for n in list(range(0, 100)) + [222, 1023, 1024, 4095, 4096, 4097]:
        assert orc.xxh64_py(buf[:n]) == orc.xxh64(buf[:n]), n


def test_libxxhash_agrees_when_present(orc):
    xxhash = pytest.importorskip("xxhash")
    rng = np.random.default_rng(3)
    for n in [0, 5, 31, 32, 100, 4096, 1 << 20, (4 << 20) + 5]:
        b = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert orc.xxh64(b) == xxhash.xxh64_intdigest(b, 0)
        assert orc.xxh64(b, seed=7) == xxhash.xxh64_intdigest(b, 7)


def test_hash_blocks_and_hash_file(orc, shm_tmp):
    rng = np.random.default_rng(4)
    buf = rng.integers(0, 256, 3_000_000, dtype=np.uint8)
    offs = np.array([0, 7, 1000, 2_000_001], dtype=np.uint64)
    lens = np.array([7, 993, 1_000_000, 999_999], dtype=np.uint32)
    got = orc.hash_blocks(buf, offs, lens)
    for o, l, h in zip(offs, lens, got):
        assert h == orc.xxh64(buf[int(o): int(o) + int(l)])
    p = shm_tmp / "f.bin"
    data = rng.integers(0, 256, (9 << 20) + 11, dtype=np.uint8)
    p.write_bytes(data.tobytes())
    hs = orc.hash_file(p)
    assert len(hs) == 3
    assert hs[0] == orc.xxh64(data[: 4 << 20]) and hs[2] == orc.xxh64(data[8 << 20:])
    (shm_tmp / "e").write_bytes(b"")
    assert len(orc.hash_file(shm_tmp / "e")) == 0


def test_splitmix_numpy_matches_c(orc):
    import ctypes
    out = np.empty(1003, dtype=np.uint8)
    orc.lib().oracle_splitmix_fill(99, 5, 1003, out.ctypes.data)
    assert (orc.splitmix_bytes(99, 1003, first_word=5) == out).all()
    # SplitMix64 reference value: first output for seed 0 is 0xE220A8397B1DCDAF
    assert int(orc.splitmix_bytes(0, 8).view("<u8")[0]) == 0xE220A8397B1DCDAF


def test_reference_pipeline_semantics(orc, shm_tmp):
    """What `tar c | tar x` (utils/copy.go:18) actually does, pinned: these are the behaviours
    the engine must reproduce (SURVEY.md Appendix C)."""
    src, dst = shm_tmp / "src", shm_tmp / "dst"
    src.mkdir(), dst.mkdir()
    make_rich_tree(src, orc)
    (dst / "big.bin").write_bytes(b"old content")
    os.link(dst / "big.bin", dst / "extra_link")
    r = orc.ref_copy(src, dst)
    assert r.returncode == 0
    # (1) whole-second mtimes (tar's default gnu format)
    assert os.lstat(dst / "big.bin").st_mtime_ns == 1_577_934_245_000_000_000
    assert os.lstat(dst / "lnk").st_mtime_ns == 1_577_934_246_000_000_000
    # (2) the root's own mode/mtime are restored from "./"
    assert os.lstat(dst).st_mtime_ns % 10**9 == 0
    # (3) an existing file is replaced, not overwritten in place; extras are kept
    assert (dst / "extra_link").read_bytes() == b"old content"
    assert os.lstat(dst / "big.bin").st_nlink == 2      # re-linked to sub/hard1 inside the tree
    # (4) hard links, symlinks (dangling too), fifo, setuid bit, sticky dir
    assert os.lstat(dst / "big.bin").st_ino == os.lstat(dst / "sub" / "hard1").st_ino
    assert os.readlink(dst / "sub" / "dangling") == "/nonexistent/target"
    assert stat.S_ISFIFO(os.lstat(dst / "fifo").st_mode)
    # root's tar restores modes exactly (-p is its default); an ordinary user's applies the umask and drops
    # setuid/setgid/sticky bits
    umask = os.umask(0)
    os.umask(umask)
    mode = (lambda m: m) if os.geteuid() == 0 else (lambda m: m & 0o777 & ~umask)
    assert stat.S_IMODE(os.lstat(dst / "big.bin").st_mode) == mode(0o4750)
    assert stat.S_IMODE(os.lstat(dst / "emptydir").st_mode) == mode(0o1777)
    assert stat.S_IMODE(os.lstat(dst / "sub" / "deep").st_mode) == mode(0o711)
    # (5) hidden directories ARE copied by tar (only `mv *` misses them)
    assert (dst / ".hidden_dir" / "inner").exists()
    if os.geteuid() == 0:
        assert os.lstat(dst / "sub").st_uid == 1234 and os.lstat(dst / "sub").st_gid == 4321
        assert stat.S_ISCHR(os.lstat(dst / "whiteout").st_mode)
    # the comparator sees the trees as equal at whole-second granularity, apart from the kept extra and the modes tar
    # changed, and flags a mutation
    set_modes = {"big.bin": 0o4750, "sub/hard1": 0o4750, "emptydir": 0o1777, "sub/deep": 0o711}
    want = ["only in B: extra_link"] + [f"{rel}: mode {m!r} != {mode(m)!r}" for rel, m in set_modes.items() if mode(m) != m]
    assert sorted(orc.compare_trees(src, dst, ignore_root_mtime=True)) == sorted(want)
    (dst / "sub" / "deep" / "tiny").write_bytes(b"abd")
    assert any("tiny" in d for d in orc.compare_trees(src, dst))


def test_reference_move_semantics(orc, shm_tmp, tmp_path):
    """`find -maxdepth 1 -type f | xargs mv -t; mv src/*` (utils/copy.go:116) across two
    mounts: top-level hidden DIRECTORIES stay behind, everything else moves."""
    src, dst = shm_tmp / "src", tmp_path / "dst"       # /dev/shm vs /tmp: different mounts -> EXDEV copy
    src.mkdir(), dst.mkdir()
    (src / ".hid").mkdir(); (src / ".hid" / "x").write_bytes(b"1")
    (src / "d").mkdir(); (src / "d" / ".inner_hidden").mkdir(); (src / "d" / "y").write_bytes(b"2")
    (src / ".dotfile").write_bytes(b"3"); (src / "plain").write_bytes(b"4")
    orc.ref_move(src, dst)
    assert sorted(os.listdir(src)) == [".hid"]
    assert sorted(os.listdir(dst)) == [".dotfile", "d", "plain"]
    assert (dst / "d" / ".inner_hidden").is_dir()
