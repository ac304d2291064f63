"""CPU tests of bench.py's own machinery (no GPU): the config-4 block selection and mutation, the memory guard, the
synthetic-tree generator both arms share, the oracle-side parity gate, and the one-JSON-line-on-stdout rule."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402

MiB = 1 << 20


def test_config4_selection_is_deterministic_and_exact():
    """BASELINE.md §3 config 4: 30 % of 12 800 blocks = exactly 3 840 distinct indices from a SplitMix64(seed 44) shuffle."""
    a = bench.splitmix_shuffle_pick(12800, 12800 * 3 // 10, 44)
    assert len(a) == 3840 == len(set(a)) and a == sorted(a) and 0 <= a[0] and a[-1] < 12800
    assert a == bench.splitmix_shuffle_pick(12800, 3840, 44)                      # same seed, same set
    assert a != bench.splitmix_shuffle_pick(12800, 3840, 45)
    assert bench.splitmix_shuffle_pick(10, 10, 1) == list(range(10))              # k == n: a permutation


def test_flip_blocks_is_an_involution_on_the_first_8_bytes(tmp_path):
    bpf = 3                                                                        # blocks per file (4 MiB each)
    for i in range(2):
        (tmp_path / f"f{i:05d}.bin").write_bytes(os.urandom(bpf * bench.BLOCK))
    before = [(tmp_path / f"f{i:05d}.bin").read_bytes() for i in range(2)]
    bench.flip_blocks(tmp_path, [1, 5], bpf)                                       # block 1 of file 0, block 2 of file 1
    after = [(tmp_path / f"f{i:05d}.bin").read_bytes() for i in range(2)]
    for f, blk in ((0, 1), (1, 2)):
        o = blk * bench.BLOCK
        assert after[f][o:o + 8] == bytes(x ^ 0xFF for x in before[f][o:o + 8])
        assert after[f][:o] == before[f][:o] and after[f][o + 8:] == before[f][o + 8:]
    bench.flip_blocks(tmp_path, [1, 5], bpf)
    assert [(tmp_path / f"f{i:05d}.bin").read_bytes() for i in range(2)] == before


def test_memory_guard_refuses_what_does_not_fit():
    have = bench.mem_budget_bytes()
    assert 0 < have < 1 << 62
    bench.require_memory(1, "a byte")                                              # fits
    with pytest.raises(SystemExit) as ei:
        bench.require_memory(have * 2, "config X")
    assert "config X" in str(ei.value) and "refusing" in str(ei.value)


def test_datagen_tool_matches_the_oracle_generator_and_builds_the_layer(tmp_path):
    """tools/vmig_datagen (stand-alone; the reference arm's only input source): `files` writes the SplitMix64 stream the oracle
    restates, `layer` the config-2B shape (file count, exact symlink / empty-file shares, one hard-link pair, depth 4)."""
    from oracle import oracle as orc
    n = bench.datagen("files", tmp_path / "f", 7, 2, 5 * MiB + 3, threads=4)
    assert n == 2 * (5 * MiB + 3)
    got = np.fromfile(tmp_path / "f" / "f00001.bin", dtype=np.uint8)
    assert (got == orc.splitmix_bytes(orc.file_seed(7, "f00001.bin"), 5 * MiB + 3)).all()
    total = bench.datagen("layer", tmp_path / "l", 2, 8 * MiB, 400, threads=4)
    files = [p for p in (tmp_path / "l").rglob("*") if p.is_file() and not p.is_symlink()]
    links = [p for p in (tmp_path / "l").rglob("*") if p.is_symlink()]
    assert len(files) == 401 and len(links) == 4                                   # 400 + the second path of the hard-link pair; 1 % symlinks
    assert sum(1 for p in files if p.stat().st_size == 0) == 2                     # 0.5 % empty
    assert sum(p.stat().st_size for p in files if p.name != "hard") == total and abs(total - 8 * MiB) < 8 * MiB // 50
    assert (tmp_path / "l" / "a1" / "hard").stat().st_nlink == 2
    assert max(len(p.relative_to(tmp_path / "l").parts) for p in files) == 5       # a*/b*/c*/d*/file


def test_oracle_side_of_the_parity_gate(tmp_path):
    """parity_gate() with a stand-in for the engine's table reader: equal trees and a correct table pass, one flipped bit in the
    destination or one wrong hash in the table raises."""
    from oracle import oracle as orc
    orc.build()
    src, dst = tmp_path / "s", tmp_path / "d"
    (src / "x").mkdir(parents=True), (dst / "x").mkdir(parents=True)
    for name, n in (("a.bin", 5 * MiB + 1), ("x/b.bin", 123)):
        data = orc.splitmix_bytes(3, n).tobytes()
        (src / name).write_bytes(data), (dst / name).write_bytes(data)
    want = bench.oracle_table(orc, src, threads=2)

    class FakeVm:
        table = want

        def table_hashes(self, _path):
            return self.table
    r = bench.parity_gate(FakeVm(), orc, src, dst, tmp_path / "t", None, "unit")
    assert r["blocks_checked_vs_oracle"] == 3 and r["dst_equals_src"]
    bad = FakeVm(); bad.table = want.copy(); bad.table[1] ^= np.uint64(1)
    with pytest.raises(AssertionError, match="engine block table"):
        bench.parity_gate(bad, orc, src, dst, tmp_path / "t", None, "unit")
    with open(dst / "a.bin", "r+b") as f:
        f.seek(4 * MiB + 0); f.write(b"\\x00" if (dst / "a.bin").read_bytes()[4 * MiB] else b"\\x01")
    with pytest.raises(AssertionError, match="destination bytes differ"):
        bench.parity_gate(FakeVm(), orc, src, dst, tmp_path / "t", None, "unit")


def test_dump_outputs_writes_exact_float_arrays(tmp_path):
    """--dump-outputs with a stand-in for the engine's table reader: the hashes come back exactly from their 32-bit halves,
    file sizes and the seeded byte sample match the trees, and a second dump of the same trees is identical."""
    src = tmp_path / "s"
    (src / "x").mkdir(parents=True)
    data = {"b.bin": os.urandom(3 * MiB + 5), "a.bin": b"", "x/c.bin": os.urandom(1000)}
    for name, b in data.items():
        (src / name).write_bytes(b)
    os.symlink("b.bin", src / "lnk")
    other = tmp_path / "o"
    other.mkdir()
    (other / "d.bin").write_bytes(os.urandom(MiB))

    class FakeVm:
        def table_hashes(self, path):
            return {"t1": np.array([0, 1 << 63, (1 << 64) - 1], np.uint64), "t2": np.array([0x123456789ABCDEF0], np.uint64)}[path]
    stats = {k: i for i, k in enumerate(bench.DUMP_STATS)}
    stats["ns_total"] = 123
    for d in ("d1", "d2"):
        bench.dump_outputs(tmp_path / d, FakeVm(), [src, other], ["t1", "t2"], stats)
    got = {p.stem: np.load(p) for p in (tmp_path / "d1").glob("*.npy")}
    assert set(got) == {"block_hash_hi32", "block_hash_lo32", "stats", "dst_file_bytes", "dst_byte_sample"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    h = (got["block_hash_hi32"].astype(np.uint64) << np.uint64(32)) | got["block_hash_lo32"].astype(np.uint64)
    assert h.tolist() == [0, 1 << 63, (1 << 64) - 1, 0x123456789ABCDEF0]
    assert got["stats"].tolist() == list(range(len(bench.DUMP_STATS)))
    order = [data["a.bin"], data["b.bin"], data["x/c.bin"], (other / "d.bin").read_bytes()]
    assert got["dst_file_bytes"].tolist() == [len(b) for b in order]
    stream = np.frombuffer(b"".join(order), np.uint8)
    pos = np.sort(np.random.default_rng(20).integers(0, stream.size, bench.DUMP_SAMPLE_BYTES))
    assert (got["dst_byte_sample"] == stream[pos]).all()
    for p in (tmp_path / "d2").glob("*.npy"):
        assert (np.load(p) == got[p.stem]).all()


def test_reference_arm_prints_exactly_one_json_line_on_stdout():
    """The contract is one JSON line on stdout; helpers and libraries may only write to stderr (config 1: the 1 GiB move)."""
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--config", "1", "--steps", "1", "--warmup", "3"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-800:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == "GiB/s" and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "reference" and d["e2e"]["h2d_bytes_per_step"] == 0 and d["higher_is_better"] is True
