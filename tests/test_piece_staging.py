"""Reads staged through each reader's small pinned pieces (csrc/vmig_engine.cu, stage 2).

CPU: the piece split (csrc/vmig_common.h piece_count / block_piece) in a compiled unit.
GPU: trees whose file sizes straddle piece and block edges, copied, hashed and verified through the pieces, against
the literal tar pipe and the oracle's block table -- with one reader turning its four pieces over hundreds of times and
with the default thread budget, buffered and O_DIRECT, and an injected fault followed by a clean call on the same pipe."""
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
MiB = 1 << 20
S = MiB     # kPieceBytes


def test_piece_split(tmp_path):
    """Block lengths 0, 1, S-1, S, S+1, 3S+17, 4 MiB-1 and 4 MiB at offsets inside and across windows: the parts tile the
    block exactly, one window each, O_DIRECT read lengths are whole 4 KiB sectors that end inside the piece, and a slot
    of small and large blocks staged window by window through transfer_block comes out byte for byte, short last blocks
    included."""
    exe = tmp_path / "piece_unit"
    csrc = ROOT / "gpu-docker-api_b200" / "csrc"
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Werror", "-I", str(csrc), str(ROOT / "tests" / "piece_unit.cpp"),
                    "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and "piece unit ok" in r.stdout, r.stdout + r.stderr


# ------------------------------------------------------------------------------------------------ GPU

EDGE_SIZES = [0, 1, S - 1, S, S + 1, 3 * S + 17, 4 * MiB - 1, 4 * MiB, 4 * MiB + 1, 64 * MiB + 5]


def _edge_tree(root: Path, orc, seed: int = 40):
    (root / "small").mkdir(parents=True)
    for i, n in enumerate(EDGE_SIZES):
        (root / f"edge{i:02d}.bin").write_bytes(orc.splitmix_bytes(seed + i, n).tobytes())
    rng_sizes = orc.splitmix_bytes(seed + 99, 2 * 300).view("<u2")      # deterministic 1-300 KiB sizes
    for i, v in enumerate(rng_sizes[:300]):
        n = 1024 + int(v) * (299 * 1024) // 65535
        (root / "small" / f"s{i:03d}").write_bytes(orc.splitmix_bytes(seed + 1000 + i, n).tobytes())


def _check_copy(vm, orc, src, dst, ref, table, flags=0):
    st = vm.migrate_tree(src, dst, None, table, flags=flags | vm.F_VERIFY)
    orc.ref_copy(src, ref)
    assert orc.compare_trees(ref, dst, mtime_ns=True) == []
    _, want = orc.block_table_of_tree(src)
    assert (vm.table_hashes(table) == want).all()
    total = sum(p.stat().st_size for p in src.rglob("*") if p.is_file())
    assert st["bytes_total"] == total and st["bytes_written"] == total
    assert st["bytes_h2d"] == 2 * total and st["bytes_d2h"] == total        # the verify pass reads every byte again
    return want


@pytest.fixture()
def gpu(vm):
    vm.init(0)          # raises VMIG_ENOGPU loudly if the box has no B200: no fallback to test
    yield
    vm.shutdown()


@pytest.mark.gpu
@pytest.mark.parametrize("readers", ["1", "default"])
def test_edge_sizes_through_the_pieces(vm, orc, shm_tmp, monkeypatch, gpu, readers):
    if readers != "default":
        monkeypatch.setenv("VMIG_READERS", readers)
    src, dst, ref = shm_tmp / "src", shm_tmp / "dst", shm_tmp / "ref"
    dst.mkdir(), ref.mkdir()
    _edge_tree(src, orc)
    want = _check_copy(vm, orc, src, dst, ref, shm_tmp / "t.vmig")
    st = vm.hash_tree(src, shm_tmp / "h.vmig")
    assert (vm.table_hashes(shm_tmp / "h.vmig") == want).all() and st["bytes_written"] == 0


@pytest.mark.gpu
def test_edge_sizes_through_the_pieces_o_direct(vm, orc, tmp_path, monkeypatch, gpu):
    """The same tree on pytest's disk-backed tmp_path, read with O_DIRECT into the pieces (whole sectors; the short last
    piece of a file asks for the rounded-up length)."""
    monkeypatch.setenv("VMIG_READERS", "1")
    src, dst, ref = tmp_path / "src", tmp_path / "dst", tmp_path / "ref"
    dst.mkdir(), ref.mkdir()
    _edge_tree(src, orc, seed=70)
    want = _check_copy(vm, orc, src, dst, ref, tmp_path / "t.vmig", flags=vm.F_DIRECT_IO)
    vm.hash_tree(src, tmp_path / "h.vmig")
    assert (vm.table_hashes(tmp_path / "h.vmig") == want).all()


@pytest.mark.gpu
def test_fault_mid_run_then_clean_call_on_the_same_pipe(vm, orc, shm_tmp, monkeypatch, gpu):
    """A fault in the middle of a one-reader run fails the call with that fault; every piece's copy has drained before
    the slots go back, so the next call through the same pooled pipe is bit-exact."""
    monkeypatch.setenv("VMIG_READERS", "1")
    src, dst, ref = shm_tmp / "src", shm_tmp / "dst", shm_tmp / "ref"
    dst.mkdir(), ref.mkdir()
    _edge_tree(src, orc, seed=90)
    _, want = orc.block_table_of_tree(src)
    monkeypatch.setenv("VMIG_FAIL_BLOCK", str(len(want) // 2))
    with pytest.raises(vm.VmigError) as ei:
        vm.migrate_tree(src, dst, None, shm_tmp / "bad.vmig")
    assert ei.value.code == vm.VMIG_EFAULT and "VMIG_FAIL_BLOCK" in str(ei.value)
    assert not (shm_tmp / "bad.vmig").exists()
    monkeypatch.delenv("VMIG_FAIL_BLOCK")
    (shm_tmp / "dst2").mkdir()
    _check_copy(vm, orc, src, shm_tmp / "dst2", ref, shm_tmp / "t.vmig")
