"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against the oracle.

Bar (spec ③): bit-exact.  Copied bytes and metadata vs the reference's literal tar / mv pipeline
(oracle.ref_copy / ref_move = utils/copy.go:18,116), block hashes vs the pinned XXH64 oracle."""
import json
import os
import shutil
import stat
import threading
import time
from pathlib import Path

import numpy as np
import pytest

from conftest import make_rich_tree

pytestmark = pytest.mark.gpu
KAT = json.loads((Path(__file__).parent / "golden" / "xxh64_kat.json").read_text())
MiB = 1 << 20


@pytest.fixture(scope="module", autouse=True)
def _gpu(vm):
    vm.init(0)          # raises VMIG_ENOGPU loudly if the box has no B200: no fallback to test
    yield
    vm.shutdown()


# ------------------------------------------------------------------------------------------ K1
def test_k1_known_answer_vectors(vm, orc):
    buf = np.frombuffer(orc.sanity_buffer(4 * MiB), dtype=np.uint8)
    lens = np.array(sorted(int(n) for n in KAT["sanity"]), dtype=np.uint32)
    offs = np.zeros(len(lens), dtype=np.uint64)          # every vector is a prefix of the buffer
    got, _ = vm.hash_blocks(buf, offs, lens)
    for n, h in zip(lens, got):
        assert int(h) == int(KAT["sanity"][str(int(n))], 16), int(n)
    z, _ = vm.hash_blocks(np.zeros(4 * MiB, np.uint8), [0], [4 * MiB])
    assert int(z[0]) == int(KAT["zeros_4MiB"], 16)
    for s, want in KAT["ascii"].items():
        b = np.frombuffer(s.encode(), dtype=np.uint8)
        g, _ = vm.hash_blocks(b, [0], [len(b)])
        assert int(g[0]) == int(want, 16), s


def test_k1_every_short_length_and_tail(vm, orc):
    """lengths 0..300 (all tail shapes: 8-, 4-, 1-byte steps, no-stripe path) at odd offsets."""
    rng = np.random.default_rng(1)
    lens = np.arange(0, 301, dtype=np.uint32)
    offs = np.cumsum(np.concatenate([[1], lens[:-1].astype(np.uint64) + 1])).astype(np.uint64)
    buf = rng.integers(0, 256, int(offs[-1] + lens[-1] + 8), dtype=np.uint8)
    got, _ = vm.hash_blocks(buf, offs, lens)
    assert (got == orc.hash_blocks(buf, offs, lens)).all()


def test_k1_ragged_blocks_vs_oracle(vm, orc):
    """random lengths up to 4 MiB+; chunk (2 KiB) and stripe (32 B) boundaries +-1; > one batch."""
    rng = np.random.default_rng(2)
    special = [2047, 2048, 2049, 2079, 2080, 4095, 4096, 4097, 6143, 6144, 6176, 65535, 65536, 65537,
               4 * MiB - 33, 4 * MiB - 32, 4 * MiB - 1, 4 * MiB, 4 * MiB + 1, 4 * MiB + 33, 5 * MiB + 7]
    lens = np.array(special + list(rng.integers(0, 3 * MiB, 40)), dtype=np.uint32)
    rng.shuffle(lens)
    offs = np.cumsum(np.concatenate([[5], lens[:-1].astype(np.uint64) + rng.integers(0, 9, len(lens) - 1).astype(np.uint64)])).astype(np.uint64)
    buf = rng.integers(0, 256, int(offs[-1] + lens[-1]), dtype=np.uint8)
    got, ms = vm.hash_blocks(buf, offs, lens)
    want = orc.hash_blocks(buf, offs, lens)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, [(int(i), int(lens[i])) for i in bad[:10]]
    assert ms > 0


def test_k1_chunk_and_ring_boundaries_vs_oracle(vm, orc):
    """The kernel stages 1 KiB chunks through a 6-stage shared-memory ring: every length k*1024 + {-33..33 around the
    stripe and chunk edges} for k = 1..14 (two wraps of the ring), plus the 6 KiB / 12 KiB wrap points +-1 and lengths that
    end exactly where a stage is refilled.  One launch holds all of them next to full 4 MiB blocks (long and short
    quads share a ring)."""
    rng = np.random.default_rng(22)
    deltas = (-33, -32, -31, -1, 0, 1, 31, 32, 33)
    lens = sorted({k * 1024 + d for k in range(1, 15) for d in deltas} | {6 * 1024 * m + d for m in (1, 2, 3, 4) for d in (-1, 0, 1)}
                  | {1025, 1055, 1056, 1057, 4 * MiB - 1024 - 1, 4 * MiB - 1024, 4 * MiB - 1024 + 1})
    lens = np.array(lens + [4 * MiB] * 3, dtype=np.uint32)
    rng.shuffle(lens)
    offs = np.cumsum(np.concatenate([[3], lens[:-1].astype(np.uint64) + rng.integers(0, 17, len(lens) - 1).astype(np.uint64)])).astype(np.uint64)
    buf = rng.integers(0, 256, int(offs[-1] + lens[-1]), dtype=np.uint8)
    got, _ = vm.hash_blocks(buf, offs, lens)
    want = orc.hash_blocks(buf, offs, lens)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, [(int(i), int(lens[i])) for i in bad[:10]]


def test_k1_repeated_under_load_from_another_stream(vm, orc):
    """The stage hand-offs of K1 are shared-memory counters, not mbarriers, and the pre-multiplied bytes are refilled by
    TMA without a proxy fence (csrc/vmig_kernels.cu): 20 launches back to back, while a second stream keeps every SM busy
    with the 2.5 GiB resident pass (so the CTAs of the launch under test are descheduled and co-scheduled at random),
    must all equal the oracle bit for bit."""
    rng = np.random.default_rng(23)
    lens = np.array([4 * MiB] * 24 + [4 * MiB - 1, 3 * MiB + 1025, 2 * MiB + 31, 1055, 6143, 6145, 12 * 1024 + 33, 0, 7],
                    dtype=np.uint32)
    offs = np.cumsum(np.concatenate([[0], lens[:-1].astype(np.uint64) + 1])).astype(np.uint64)
    buf = rng.integers(0, 256, int(offs[-1] + lens[-1]), dtype=np.uint8)
    want = orc.hash_blocks(buf, offs, lens)
    r = vm.Resident(640, 4 * MiB)
    stop, errs = threading.Event(), []

    def load():
        try:
            r.fill(5); r.set_prior(None)
            while not stop.is_set():
                r.run(4)
        except Exception as e:      # noqa: BLE001
            errs.append(e)
    t = threading.Thread(target=load)
    t.start()
    try:
        for rep in range(20):
            got, _ = vm.hash_blocks(buf, offs, lens)
            bad = np.nonzero(got != want)[0]
            assert bad.size == 0, (rep, [(int(i), int(lens[i])) for i in bad[:10]])
    finally:
        stop.set(); t.join(); r.close()
    assert not errs, errs


def test_k1_many_small_blocks_dynamic_scheduling(vm, orc):
    """20 000 small blocks: several batches of 4096, work-stealing counter, zero-length blocks."""
    rng = np.random.default_rng(3)
    lens = rng.integers(0, 700, 20000).astype(np.uint32)
    lens[::97] = 0
    offs = np.concatenate([[0], np.cumsum(lens[:-1].astype(np.uint64))]).astype(np.uint64)
    buf = rng.integers(0, 256, int(lens.astype(np.uint64).sum()) + 1, dtype=np.uint8)
    got, _ = vm.hash_blocks(buf, offs, lens)
    assert (got == orc.hash_blocks(buf, offs, lens)).all()


def test_k1_rejects_block_larger_than_slot(vm):
    with pytest.raises(vm.VmigError) as ei:
        vm.hash_blocks(np.zeros(40 * MiB, np.uint8), [0], [40 * MiB])
    assert ei.value.code == vm.VMIG_EINVAL


# ------------------------------------------------------------------------------------ resident
def test_resident_open_that_does_not_fit_fails_cleanly(vm):
    """A batch larger than HBM is refused with VMIG_ENOMEM and leaves nothing behind: a normal batch
    opens right after it (the partial allocation was given back)."""
    with pytest.raises(vm.VmigError) as ei:
        vm.Resident(100_000, 4 * MiB)                 # 400 GB > 180 GB of HBM
    assert ei.value.code == vm.VMIG_ENOMEM
    with pytest.raises(vm.VmigError) as ei:
        vm.Resident(4, 4 * MiB, gpu=77)
    assert ei.value.code in (vm.VMIG_EINVAL, vm.VMIG_ENOGPU)
    r = vm.Resident(64, 4 * MiB)
    try:
        r.fill(1); r.set_prior(None); r.run(1)
        h, surv = r.results()
        assert len(surv) == 64 and len(set(h.tolist())) == 64
    finally:
        r.close()


def test_resident_fill_hash_diff_select(vm, orc):
    """HBM-resident pass: device generator == oracle generator, hashes == oracle on sampled
    blocks, and diff_select returns exactly the flipped / invalid-prior blocks, ascending."""
    n, bb = 300, 4 * MiB
    r = vm.Resident(n, bb)
    try:
        r.fill(1234)
        words = bb // 8
        sample = [0, 1, 147, 148, 149, 299]
        for b in sample:
            dev = r.download(b, bb)
            assert (dev == orc.splitmix_bytes(1234, bb, first_word=b * words)).all(), b
        r.set_prior(None)
        r.run(1)
        h1, surv = r.results()
        assert len(surv) == n and (surv == np.arange(n)).all()      # no prior: everything survives
        for b in sample:
            assert int(h1[b]) == orc.xxh64(orc.splitmix_bytes(1234, bb, first_word=b * words)), b
        assert len(set(h1.tolist())) == n
        # prior = these hashes; flip 30% of the blocks; two blocks have no valid prior
        flip = np.sort(np.random.default_rng(44).permutation(n)[: n * 3 // 10]).astype(np.uint64)
        valid = np.ones(n, np.uint8)
        valid[[5, 250]] = 0
        r.set_prior(h1, valid)
        r.flip(flip)
        ms_hash, ms_total = r.run(2)
        h2, surv = r.results()
        want = sorted(set(flip.tolist()) | {5, 250})
        assert surv.tolist() == want
        same = np.setdiff1d(np.arange(n), flip)
        assert (h2[same] == h1[same]).all() and (h2[flip.astype(int)] != h1[flip.astype(int)]).all()
        b = int(flip[0])
        blk = orc.splitmix_bytes(1234, bb, first_word=b * words).copy()
        blk[:8] ^= 0xFF
        assert int(h2[b]) == orc.xxh64(blk)
        assert 0 < ms_hash <= ms_total
        # ragged lengths inside resident slots
        for b, ln in [(0, 0), (1, 31), (2, 4 * MiB - 1), (3, 2049)]:
            r.set_len(b, ln)
        r.run(1)
        h3, _ = r.results()
        for b, ln in [(0, 0), (1, 31), (2, 4 * MiB - 1), (3, 2049)]:
            blk = r.download(b, bb)[:ln]
            assert int(h3[b]) == orc.xxh64(blk), (b, ln)
    finally:
        r.close()


# ------------------------------------------------------------------------------------- the tree
def test_copydir_matches_reference_tar_pipeline(vm, orc, shm_tmp):
    """utils.CopyDir parity: same tree as `(cd src; tar c .) | (cd dst; tar x)` incl. ns-exact
    (i.e. whole-second) mtimes, hard links, specials, replaced pre-existing entries."""
    src, dst, ref = shm_tmp / "src", shm_tmp / "dst", shm_tmp / "ref"
    for d in (src, dst, ref):
        d.mkdir()
    make_rich_tree(src, orc)
    for d in (dst, ref):        # pre-existing destination entries
        (d / "big.bin").write_bytes(b"old")
        os.link(d / "big.bin", d / "keepme")
        (d / "lnk").write_bytes(b"was a file")
        (d / "sub").mkdir()
        (d / "sub" / "stale").write_bytes(b"stale")
        for p in (d / "keepme", d / "sub" / "stale"):          # entries outside src keep their own times
            os.utime(p, ns=(10**18, 10**18 + 7))
    vm.CopyDir(str(src), str(dst))
    assert orc.ref_copy(src, ref).returncode == 0
    assert orc.compare_trees(ref, dst, mtime_ns=True) == []
    assert (dst / "keepme").read_bytes() == b"old" and (dst / "sub" / "stale").exists()
    assert orc.compare_trees(src, dst, ignore_root_mtime=True)[:0] == []      # src untouched:
    assert (src / "big.bin").exists()


def test_copydir_awkward_names_and_shapes(vm, orc, shm_tmp):
    """Names tar has to escape or extend (spaces, newline, non-UTF-8 bytes, >100 and >255 byte paths),
    read-only and setgid directories, a sparse file (tar densifies it), hard-linked empty files,
    a symlink to a directory, an empty source subtree."""
    src, dst, ref = shm_tmp / "src", shm_tmp / "dst", shm_tmp / "ref"
    for d in (src, dst, ref):
        d.mkdir()
    bsrc = os.fsencode(src)
    names = [b"sp ace", b"new\nline", b"tab\there", b"quote'\"", b"\xff\xfe-not-utf8", "uni-\u00e7o\u2202\u00e9".encode(), b"-dash", b"x" * 200]
    for i, n in enumerate(names):
        with open(os.path.join(bsrc, n), "wb") as f:
            f.write(orc.splitmix_bytes(90 + i, 1000 * i + 1).tobytes())
    deep = src
    for i in range(12):                                   # 12 x 30 = 360-byte relative path
        deep = deep / ("d%02d_" % i + "y" * 25)
    deep.mkdir(parents=True)
    (deep / "leaf.bin").write_bytes(orc.splitmix_bytes(70, 4 * MiB + 17).tobytes())
    (src / "ro_dir").mkdir(); (src / "ro_dir" / "inside").write_bytes(b"in a read-only dir")
    os.chmod(src / "ro_dir", 0o555)
    (src / "sgid").mkdir(); os.chmod(src / "sgid", 0o2775)
    with open(src / "sparse.bin", "wb") as f:             # 6 MiB hole, then data
        f.seek(6 * MiB); f.write(b"tail-after-hole")
    (src / "e1").write_bytes(b""); os.link(src / "e1", src / "e2")
    os.symlink("ro_dir", src / "dirlink")
    (src / "empty_tree" / "a" / "b").mkdir(parents=True)
    vm.CopyDir(str(src), str(dst))
    assert orc.ref_copy(src, ref).returncode == 0
    assert orc.compare_trees(ref, dst, mtime_ns=True) == []
    assert os.lstat(dst / "e1").st_ino == os.lstat(dst / "e2").st_ino
    assert (dst / "sparse.bin").stat().st_size == 6 * MiB + 15
    os.chmod(src / "ro_dir", 0o755)                       # let the fixture clean up
    os.chmod(dst / "ro_dir", 0o755), os.chmod(ref / "ro_dir", 0o755)


def test_copydir_of_empty_directory(vm, orc, shm_tmp):
    src, dst = shm_tmp / "src", shm_tmp / "dst"
    src.mkdir(), dst.mkdir()
    os.chmod(src, 0o750)
    st = vm.migrate_tree(src, dst, None, shm_tmp / "t.vmig")
    assert st["blocks_total"] == 0 and st["kernel_launches"] == 0 and os.listdir(dst) == []
    assert os.stat(dst).st_mode & 0o7777 == 0o750
    assert orc.read_table(shm_tmp / "t.vmig")["entries"] == []


def test_block_table_matches_oracle(vm, orc, shm_tmp):
    src, dst = shm_tmp / "src", shm_tmp / "dst"
    src.mkdir(), dst.mkdir()
    make_rich_tree(src, orc)
    st = vm.migrate_tree(src, dst, None, shm_tmp / "t.vmig")
    entries, want = orc.block_table_of_tree(src)
    tab = orc.read_table(shm_tmp / "t.vmig")
    assert tab["entries"] == entries
    assert (tab["hashes"] == want).all()
    assert st["blocks_total"] == len(want) and st["bytes_total"] == sum(e[1] for e in entries)
    assert st["blocks_skipped"] == 0 and st["kernel_launches"] >= 1 and st["ms_kernel"] > 0
    # hard-linked paths are hashed once: fewer bytes cross PCIe than the table describes
    assert st["bytes_h2d"] < st["bytes_total"] and st["bytes_d2h"] == st["bytes_h2d"] == st["bytes_written"]
    # hash-only mode: same table, destination untouched
    vm.hash_tree(src, shm_tmp / "t2.vmig")
    tab2 = orc.read_table(shm_tmp / "t2.vmig")
    assert tab2["entries"] == tab["entries"] and (tab2["hashes"] == tab["hashes"]).all()
    # ... and each table names the files it speaks for: the destination's for a migration, the source's for hash-only
    for (rel, _size, _first), (ino, ct), (ino2, ct2) in zip(entries, tab["identity"], tab2["identity"]):
        d, s_ = os.lstat(dst / os.fsdecode(rel)), os.lstat(src / os.fsdecode(rel))
        if d.st_nlink == 1 and d.st_size:
            assert (ino, ct) == (d.st_ino, d.st_ctime_ns) and (ino2, ct2) == (s_.st_ino, s_.st_ctime_ns), rel


def _mutate(path: Path, block: int, bb=4 * MiB):
    with open(path, "r+b") as f:
        f.seek(block * bb)
        w = bytearray(f.read(8))
        for i in range(len(w)):
            w[i] ^= 0xFF
        f.seek(block * bb)
        f.write(w)


def test_diff_skip_copies_exactly_the_changed_blocks(vm, orc, shm_tmp):
    """BASELINE config 4 in miniature: dst holds the prior version + its block table; only the
    changed blocks travel back over PCIe and get written; dst == src afterwards."""
    src, dst = shm_tmp / "src", shm_tmp / "dst"
    src.mkdir(), dst.mkdir()
    sizes = {"a.bin": 24 * MiB, "b.bin": 12 * MiB + 100, "c.bin": 5 * MiB, "d/e.bin": 9 * MiB, "same.bin": 8 * MiB}
    for name, sz in sizes.items():
        (src / name).parent.mkdir(exist_ok=True)
        (src / name).write_bytes(orc.splitmix_bytes(orc.file_seed(9, name), sz).tobytes())
    vm.CopyDir(str(src), str(dst))                               # v1 in dst
    vm.hash_tree(dst, shm_tmp / "v1.vmig")                       # the prior table
    assert (orc.read_table(shm_tmp / "v1.vmig")["hashes"] == orc.block_table_of_tree(dst)[1]).all()
    # v2 = src with: 3 blocks changed in a, last (short) block changed in b, c grown, e shrunk,
    # a brand-new file, and one file deleted from dst behind the table's back
    for blk in (0, 3, 5):
        _mutate(src / "a.bin", blk)
    _mutate(src / "b.bin", 3)
    with open(src / "c.bin", "ab") as f:
        f.write(orc.splitmix_bytes(77, 3 * MiB + 5).tobytes())
    os.truncate(src / "d" / "e.bin", 6 * MiB + 9)
    (src / "new.bin").write_bytes(orc.splitmix_bytes(78, 4 * MiB + 1).tobytes())
    mtime_same = os.lstat(dst / "same.bin").st_mtime_ns
    st = vm.migrate_tree(src, dst, shm_tmp / "v1.vmig", shm_tmp / "v2.vmig")
    # expected survivors: a:3, b:1 (short tail block), c: block 1 (was 1 MiB, now full) + block 2 (new),
    # e: block 1 (was full, now 2 MiB+9), new.bin: 2  -> 9; everything else skipped
    n_blocks = sum((os.path.getsize(src / n) + 4 * MiB - 1) // (4 * MiB) for n in list(sizes) + ["new.bin"])
    assert st["blocks_total"] == n_blocks
    assert st["blocks_total"] - st["blocks_skipped"] == 9, st
    changed_bytes = 3 * 4 * MiB + 100 + 4 * MiB + 5 + (2 * MiB + 9) + 4 * MiB + 1
    assert st["bytes_d2h"] == changed_bytes == st["bytes_written"]
    assert st["bytes_h2d"] == st["bytes_total"]
    ref = shm_tmp / "ref"
    ref.mkdir()
    orc.ref_copy(src, ref)
    assert orc.compare_trees(ref, dst, mtime_ns=True) == []
    assert (orc.read_table(shm_tmp / "v2.vmig")["hashes"] == orc.block_table_of_tree(src)[1]).all()
    assert os.lstat(dst / "same.bin").st_mtime_ns == mtime_same
    # re-running against the new table moves nothing at all ("resume for free")
    st2 = vm.migrate_tree(src, dst, shm_tmp / "v2.vmig", None)
    assert st2["blocks_skipped"] == st2["blocks_total"] and st2["bytes_d2h"] == 0 and st2["bytes_written"] == 0
    # a stale table entry for a file that vanished from dst is not trusted
    os.unlink(dst / "a.bin")
    st3 = vm.migrate_tree(src, dst, shm_tmp / "v2.vmig", None)
    assert st3["blocks_total"] - st3["blocks_skipped"] == 6
    assert orc.compare_trees(ref, dst, mtime_ns=True) == []


def test_move_matches_reference_mv(vm, orc, shm_tmp, tmp_path):
    """CopyOldMountPointToContainerMountPoint parity with the helper container's command
    (utils/copy.go:116) run across two mounts; plus the documented divergence (hidden top dirs)."""
    def build(root):
        root.mkdir()
        (root / "d").mkdir(); (root / "d" / ".inner").mkdir()
        (root / "d" / "y.bin").write_bytes(orc.splitmix_bytes(5, 5 * MiB + 3).tobytes())
        (root / ".dotfile").write_bytes(b"3"); (root / "plain").write_bytes(b"4" * 5000)
        os.symlink("plain", root / "l")
        (root / ".hid").mkdir(); (root / ".hid" / "x").write_bytes(b"1")
        t = 1_577_934_245_123_456_789
        for dp, dn, fn in os.walk(root, topdown=False):      # identical times in every copy of the tree
            for n in fn + dn:
                os.utime(os.path.join(dp, n), ns=(t, t + len(n)), follow_symlinks=False)
    s1, s2 = shm_tmp / "s1", shm_tmp / "s2"
    d1, d2 = tmp_path / "d1", tmp_path / "d2"
    build(s1), build(s2), d1.mkdir(), d2.mkdir()
    orc.ref_move(s1, d1)
    st = vm.migrate_tree(s2, d2, flags=vm.F_MOVE_SRC | vm.F_SKIP_HIDDEN_TOPDIRS)
    assert st["files"] == 3
    diffs = [d for d in orc.compare_trees(d1, d2, mtime_ns=True) if not d.startswith(".:")]
    assert diffs == [], diffs
    assert sorted(os.listdir(s1)) == sorted(os.listdir(s2)) == [".hid"]
    # default move (the resolver-backed reference call): hidden top-level dirs migrate too
    s3, d3 = shm_tmp / "s3", tmp_path / "d3"
    build(s3), d3.mkdir()
    vm.set_resolver(None, {"vol-1": str(s3), "vol-2": str(d3)}.get)
    vm.CopyOldMountPointToContainerMountPoint("vol-1", "vol-2")
    vm.set_resolver(None, None)
    assert os.listdir(s3) == [] and (d3 / ".hid" / "x").read_bytes() == b"1"
    assert os.lstat(d3 / "plain").st_mtime_ns == 1_577_934_245_123_456_789 + 5     # mv keeps ns


def test_container_layer_copy_through_reference_names(vm, orc, shm_tmp):
    """CopyOldMergedToNewContainerMerged(old, new): the call PatchContainer makes
    (services/replicaset.go:333) with the Docker inspect injected."""
    up = {"rs-3": shm_tmp / "overlay2" / "aaa" / "diff", "rs-4": shm_tmp / "overlay2" / "bbb" / "diff"}
    for p in up.values():
        p.mkdir(parents=True)
    make_rich_tree(up["rs-3"], orc, seed=21, big=5 * MiB + 1)
    vm.set_resolver(lambda n: str(up.get(n, "")), None)
    vm.CopyOldMergedToNewContainerMerged("rs-3", "rs-4")
    with pytest.raises(vm.VmigError):
        vm.CopyOldMergedToNewContainerMerged("rs-3", "rs-unknown")
    vm.set_resolver(None, None)
    ref = shm_tmp / "ref"
    ref.mkdir()
    orc.ref_copy(up["rs-3"], ref)
    assert orc.compare_trees(ref, up["rs-4"], mtime_ns=True) == []


def test_many_small_files_tree(vm, orc, shm_tmp):
    """diff-layer shaped input: 3 000 files of 0..200 KiB in a depth-3 tree (groups of 64 files,
    several batches of packed short blocks)."""
    rng = np.random.default_rng(8)
    src, dst, ref = shm_tmp / "src", shm_tmp / "dst", shm_tmp / "ref"
    for d in (src, dst, ref):
        d.mkdir()
    for i in range(3000):
        d = src / f"p{i % 7}" / f"q{i % 13}"
        d.mkdir(parents=True, exist_ok=True)
        n = int(rng.integers(0, 200 * 1024)) if i % 50 else 0
        (d / f"f{i}.dat").write_bytes(rng.integers(0, 256, n, dtype=np.uint8).tobytes())
    st = vm.migrate_tree(src, dst, None, shm_tmp / "t.vmig")
    orc.ref_copy(src, ref)
    assert orc.compare_trees(ref, dst, mtime_ns=True) == []
    assert (orc.read_table(shm_tmp / "t.vmig")["hashes"] == orc.block_table_of_tree(src)[1]).all()
    assert st["files"] == 3000


def test_concurrent_calls_are_reentrant(vm, orc, shm_tmp):
    """SURVEY.md F9: N gin goroutines call the copy at once with no lock (BASELINE config 5)."""
    n = 4
    errs = []
    for i in range(n):
        (shm_tmp / f"s{i}").mkdir(), (shm_tmp / f"d{i}").mkdir()
        (shm_tmp / f"s{i}" / "x.bin").write_bytes(orc.splitmix_bytes(100 + i, 13 * MiB + i).tobytes())
        (shm_tmp / f"s{i}" / "y.txt").write_bytes(b"y" * (i + 1))

    def work(i):
        try:
            vm.migrate_tree(shm_tmp / f"s{i}", shm_tmp / f"d{i}", None, shm_tmp / f"t{i}.vmig")
        except Exception as e:      # noqa: BLE001
            errs.append(e)
    th = [threading.Thread(target=work, args=(i,)) for i in range(n)]
    [t.start() for t in th], [t.join() for t in th]
    assert not errs, errs
    for i in range(n):
        assert orc.compare_trees(shm_tmp / f"s{i}", shm_tmp / f"d{i}", ignore_root_mtime=True) == []
        assert (orc.read_table(shm_tmp / f"t{i}.vmig")["hashes"] == orc.block_table_of_tree(shm_tmp / f"s{i}")[1]).all()


def test_injected_fault_is_reported_not_swallowed(vm, orc, shm_tmp, monkeypatch):
    """The reference ignores a failed copy (SURVEY.md F10); the engine must not."""
    src, dst = shm_tmp / "src", shm_tmp / "dst"
    src.mkdir(), dst.mkdir()
    (src / "x.bin").write_bytes(orc.splitmix_bytes(1, 20 * MiB).tobytes())
    monkeypatch.setenv("VMIG_FAIL_BLOCK", "3")
    with pytest.raises(vm.VmigError) as ei:
        vm.migrate_tree(src, dst, None, shm_tmp / "t.vmig")
    assert ei.value.code == vm.VMIG_EFAULT
    assert not (shm_tmp / "t.vmig").exists()          # no table for a failed migration
    monkeypatch.delenv("VMIG_FAIL_BLOCK")
    vm.CopyDir(str(src), str(dst))                    # and the engine is still usable afterwards
    assert (dst / "x.bin").read_bytes() == (src / "x.bin").read_bytes()


_OUT_OF_SPACE = r"""
import os, subprocess, sys
from pathlib import Path
root, base = sys.argv[1], Path(sys.argv[2])
sys.path.insert(0, root)
import __graft_entry__ as g
from oracle import oracle as orc
vm = g.load_pkg()
small, src = base / "small", base / "src"
subprocess.run(["mount", "-t", "tmpfs", "-o", "size=48m", "tmpfs", str(small)], check=True)
vm.init(0)
try:
    vm.migrate_tree(src, small, None, base / "t.vmig", flags=vm.F_MOVE_SRC)
    raise AssertionError("a 120 MiB tree fitted on a 48 MiB tmpfs")
except vm.VmigError as e:
    assert e.code == vm.VMIG_EIO and "No space left" in str(e), e
assert not (base / "t.vmig").exists() and len(os.listdir(src)) == 6        # a failed move keeps its source
r = subprocess.run(["umount", str(small)], capture_output=True, text=True)
assert r.returncode == 0, "destination descriptors were left open: " + r.stderr
dst = base / "dst"
dst.mkdir()
vm.migrate_tree(src, dst, None, None)
assert orc.compare_trees(src, dst) == []
vm.shutdown()
print("out of space ok")
"""


def test_destination_out_of_space_fails_the_call(vm, orc, shm_tmp):
    """A real write error (ENOSPC on a 48 MiB tmpfs taking a 120 MiB tree) surfaces as VMIG_EIO with the errno
    text, leaves no descriptor open on the mount (it unmounts), and the engine keeps working.  The tmpfs is mounted in
    a private mount namespace of a child process (a user namespace too where the test does not run as root), so it
    needs no privilege and cannot outlive the test."""
    import subprocess
    import sys
    (shm_tmp / "small").mkdir()
    src = shm_tmp / "src"
    src.mkdir()
    for i in range(6):
        (src / f"f{i}.bin").write_bytes(orc.splitmix_bytes(70 + i, 20 * MiB).tobytes())
    ns = ["unshare", "--mount"] + (["--user", "--map-root-user"] if os.geteuid() != 0 else [])
    r = subprocess.run(ns + [sys.executable, "-c", _OUT_OF_SPACE, str(Path(__file__).resolve().parent.parent), str(shm_tmp)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "out of space ok" in r.stdout, r.stdout + r.stderr


def test_verify_flag_catches_a_corrupted_destination(vm, orc, shm_tmp, monkeypatch):
    """VMIG_F_VERIFY re-reads the destination through the GPU; a block that reached the disk wrong
    (test hook flips one bit while writing) fails the call, and a move then keeps its source."""
    src, dst = shm_tmp / "src", shm_tmp / "dst"
    src.mkdir(), dst.mkdir()
    (src / "a.bin").write_bytes(orc.splitmix_bytes(3, 13 * MiB + 5).tobytes())
    (src / "b.bin").write_bytes(orc.splitmix_bytes(4, 6 * MiB).tobytes())
    st = vm.migrate_tree(src, dst, None, shm_tmp / "t.vmig", flags=vm.F_VERIFY)          # clean run verifies
    assert st["bytes_h2d"] == 2 * st["bytes_total"] and st["bytes_d2h"] == st["bytes_total"]
    monkeypatch.setenv("VMIG_CORRUPT_BLOCK", "2")
    shutil.rmtree(dst); dst.mkdir()
    with pytest.raises(vm.VmigError) as ei:
        vm.migrate_tree(src, dst, None, None, flags=vm.F_VERIFY | vm.F_MOVE_SRC)
    assert ei.value.code == vm.VMIG_EVERIFY and "a.bin block 2" in str(ei.value)
    assert (src / "a.bin").exists() and (src / "b.bin").exists()          # nothing was unlinked
    vm.migrate_tree(src, dst, None, None)                                 # without VERIFY the bad bit goes unnoticed ...
    assert (dst / "a.bin").read_bytes() != (src / "a.bin").read_bytes()   # ... which is what the flag is for
    monkeypatch.delenv("VMIG_CORRUPT_BLOCK")
    vm.migrate_tree(src, dst, None, None, flags=vm.F_VERIFY | vm.F_MOVE_SRC)
    assert os.listdir(src) == [] and sorted(os.listdir(dst)) == ["a.bin", "b.bin"]


def test_source_swapped_for_symlink_mid_copy_never_leaks(vm, shm_tmp):
    """The source layer can belong to a tenant that is still running (first pass of a two-pass hand-off).  While
    migrations run, a thread keeps swapping src/victim/ for a symlink to a directory OUTSIDE the tree that holds
    same-named files.  Whatever the interleaving, no byte from outside may reach the destination: a call either
    copies the real files or fails with VMIG_ESRCCHANGED/VMIG_EIO (the reference's `tar c .` walks by directory
    descriptor in the same way)."""
    import threading
    src, outside = shm_tmp / "src", shm_tmp / "outside"
    (src / "victim").mkdir(parents=True), (src / "calm").mkdir(), outside.mkdir()
    real, secret = b"R" * (1 << 20), b"SECRET-OUTSIDE!!" * (1 << 16)
    for i in range(48):
        (src / "victim" / f"f{i:02d}").write_bytes(real)
        (outside / f"f{i:02d}").write_bytes(secret)
        (src / "calm" / f"g{i:02d}").write_bytes(real)
    stop = threading.Event()

    def swapper():
        v, bak = src / "victim", src / "victim.bak"
        while not stop.is_set():
            os.rename(v, bak); os.symlink(outside, v)
            time.sleep(0.0005)
            os.unlink(v); os.rename(bak, v)
            time.sleep(0.0005)

    t = threading.Thread(target=swapper); t.start()
    outcomes = {"ok": 0, "refused": 0}
    try:
        for rep in range(12):
            dst = shm_tmp / f"dst{rep}"
            dst.mkdir()
            try:
                vm.migrate_tree(src, dst, None, None)
                outcomes["ok"] += 1
            except vm.VmigError as e:
                assert e.code in (vm.VMIG_ESRCCHANGED, vm.VMIG_EIO), e
                outcomes["refused"] += 1
            for root, _dirs, files in os.walk(dst, followlinks=False):
                for f in files:
                    p = Path(root) / f
                    if not p.is_symlink():
                        assert b"SECRET" not in p.read_bytes()[:64], f"{p} holds bytes from outside the source tree"
            shutil.rmtree(dst)
    finally:
        stop.set(); t.join()
    assert outcomes["ok"] + outcomes["refused"] == 12


def test_side_stream_limit_option(vm, orc, shm_tmp):
    """vmig_opts.streams_per_gpu bounds the staging slots (= side streams) in flight; results are identical."""
    src, d1, d2 = shm_tmp / "src", shm_tmp / "d1", shm_tmp / "d2"
    src.mkdir(), d1.mkdir(), d2.mkdir()
    for i in range(3):
        (src / f"f{i}").write_bytes(orc.splitmix_bytes(40 + i, 40 * MiB + i).tobytes())
    vm.migrate_tree(src, d1, None, shm_tmp / "t1", streams_per_gpu=1)
    vm.migrate_tree(src, d2, None, shm_tmp / "t2")
    assert (vm.table_hashes(shm_tmp / "t1") == vm.table_hashes(shm_tmp / "t2")).all()      # (the tables differ in the file identities they carry)
    assert orc.read_table(shm_tmp / "t1")["entries"] == orc.read_table(shm_tmp / "t2")["entries"]
    assert orc.compare_trees(d1, d2, mtime_ns=True) == []


def test_missing_prior_table_is_an_error(vm, shm_tmp):
    (shm_tmp / "s").mkdir(), (shm_tmp / "d").mkdir()
    (shm_tmp / "s" / "f").write_bytes(b"1" * 100)
    with pytest.raises(vm.VmigError) as ei:
        vm.migrate_tree(shm_tmp / "s", shm_tmp / "d", shm_tmp / "nope.vmig")
    assert ei.value.code == vm.VMIG_ETABLE
    assert os.listdir(shm_tmp / "d") == []


# ----------------------------------------------------------------------------------- buffers
@pytest.mark.parametrize("pinned", [False, True])
def test_migrate_buffer_roundtrip_and_diff(vm, orc, pinned):
    n = 37 * MiB + 4321
    data = orc.splitmix_bytes(31, n)
    if pinned:
        a, b = vm.PinnedBuffer(n), vm.PinnedBuffer(n)
        src, dst = a.array, b.array
    else:
        src, dst = np.empty(n, np.uint8), np.empty(n, np.uint8)
    src[:] = data
    dst[:] = 0
    h, st = vm.migrate_buffer(src, dst)
    assert (dst == data).all()
    nb = (n + 4 * MiB - 1) // (4 * MiB)
    want = orc.hash_blocks(data, np.arange(nb, dtype=np.uint64) * (4 * MiB),
                           [min(4 * MiB, n - i * 4 * MiB) for i in range(nb)])
    assert (h == want).all()
    assert st["bytes_h2d"] == n == st["bytes_d2h"]
    # diff: change two blocks of src, poison dst's other blocks, migrate against the prior hashes
    src[5 * 4 * MiB + 17] ^= 1
    src[-1] ^= 0x80
    dst2 = dst.copy() if not pinned else dst
    h2, st2 = vm.migrate_buffer(src, dst2, h, np.ones(nb, np.uint8))
    assert st2["blocks_skipped"] == nb - 2 and st2["bytes_d2h"] == 4 * MiB + (n - (nb - 1) * 4 * MiB)
    assert (dst2 == src).all()
    assert (np.nonzero(h2 != h)[0] == [5, nb - 1]).all()
    if pinned:
        a.free(), b.free()


@pytest.mark.parametrize("lanes", [2, 3, 8])
def test_sharded_block_list_matches_oracle(vm, orc, shm_tmp, lanes):
    """North-star split (SURVEY.md §8e): ONE call whose block list is sharded over several lanes.  On a 1-GPU box
    the lanes share the device (vmig_opts.lanes_per_gpu), on an N-GPU box they spread over the GPUs first -- the
    split, the shared hash array and the cross-lane per-file counters are the same code either way.  Tree and
    table are compared with the ORACLE (the literal tar pipe, the C XXH64), not with a 1-lane run."""
    ndev = vm.device_count()
    gpus = min(ndev, lanes)
    src, dst, ref = shm_tmp / "src", shm_tmp / "dst", shm_tmp / "ref"
    (src / "d").mkdir(parents=True), dst.mkdir(), ref.mkdir()
    sizes = [11 * MiB + 1, 4 * MiB, 4 * MiB - 1, 1, 37 * MiB + 5, 0, 9 * MiB, 123457, 8 * MiB, 5 * MiB + 4095,
             2 * MiB, 6 * MiB + 31, 3 * MiB + 33, 17, 4 * MiB + 1, 12 * MiB, 70001, 21 * MiB + 7]
    for i, n in enumerate(sizes):
        (src / ("d" if i % 3 == 0 else ".") / f"f{i:02d}.bin").write_bytes(orc.splitmix_bytes(600 + i, n).tobytes())
    os.link(src / "f04.bin", src / "d" / "hard04")
    os.symlink("f01.bin", src / "lnk")
    st = vm.migrate_tree(src, dst, None, shm_tmp / "t.vmig", gpu_mask=(1 << gpus) - 1, lanes_per_gpu=-(-lanes // gpus))
    assert st["gpus_used"] == gpus and st["lanes_used"] >= lanes
    orc.ref_copy(src, ref)
    assert orc.compare_trees(ref, dst) == []
    _, want = orc.block_table_of_tree(src)
    assert (vm.table_hashes(shm_tmp / "t.vmig") == want).all()
    # one huge file and fewer files than lanes: the contiguous byte-range split (lanes share a destination file)
    one, d2 = shm_tmp / "one", shm_tmp / "d2"
    one.mkdir(), d2.mkdir()
    (one / "big.bin").write_bytes(orc.splitmix_bytes(77, 61 * MiB + 13).tobytes())
    st = vm.migrate_tree(one, d2, None, shm_tmp / "t2.vmig", gpu_mask=(1 << gpus) - 1, lanes_per_gpu=-(-lanes // gpus))
    assert st["lanes_used"] >= lanes
    assert (d2 / "big.bin").read_bytes() == (one / "big.bin").read_bytes()
    assert (vm.table_hashes(shm_tmp / "t2.vmig") == orc.hash_file(one / "big.bin")).all()
    # diff pass against the table just written: only the two mutated blocks move, on whichever lanes own them
    _mutate(one / "big.bin", 3), _mutate(one / "big.bin", 14)
    st = vm.migrate_tree(one, d2, shm_tmp / "t2.vmig", shm_tmp / "t3.vmig", gpu_mask=(1 << gpus) - 1,
                         lanes_per_gpu=-(-lanes // gpus))
    assert st["blocks_total"] - st["blocks_skipped"] == 2
    assert (d2 / "big.bin").read_bytes() == (one / "big.bin").read_bytes()


def test_full_size_resident_pass_properties(vm, orc):
    """BASELINE config 2 size (10 GiB = 2 560 blocks resident in HBM): ALL 2 560 block hashes == oracle, the
    30 % mutation of config 4 is found exactly, and hashing is deterministic across passes."""
    n, bb = 2560, 4 * MiB
    r = vm.Resident(n, bb)
    try:
        r.fill(0xB200)
        r.set_prior(None)
        r.run(1)
        h1, surv = r.results()
        assert len(surv) == n
        words = bb // 8
        for b in [0, 1, 147, 148, 1279, 2047, 2559]:          # the device generator == the oracle's generator
            assert int(h1[b]) == orc.xxh64(orc.splitmix_bytes(0xB200, bb, first_word=b * words)), b
        # EVERY one of the 2 560 hashes against the oracle: the resident bytes are downloaded 64 blocks at a time and
        # hashed by oracle/xxh64_ref.c (10 GiB at ~7 GB/s on one core)
        batch = np.empty(64 * bb, dtype=np.uint8)
        boffs, blens = np.arange(64, dtype=np.uint64) * bb, [bb] * 64
        for b0 in range(0, n, 64):
            for j in range(64):
                batch[j * bb:(j + 1) * bb] = r.download(b0 + j, bb)
            want = orc.hash_blocks(batch, boffs, blens)
            bad = np.nonzero(want != h1[b0:b0 + 64])[0]
            assert bad.size == 0, (b0, bad[:8].tolist())
        r.run(2)
        h1b, _ = r.results()
        assert (h1 == h1b).all()
        flip = np.sort(np.random.default_rng(44).permutation(n)[: n * 3 // 10]).astype(np.uint64)
        r.set_prior(h1, np.ones(n, np.uint8))
        r.flip(flip)
        r.run(1)
        h2, surv = r.results()
        assert surv.tolist() == flip.tolist() and len(surv) == 768
        r.flip(flip)                       # flipping back restores every hash (involution)
        r.run(1)
        h3, surv = r.results()
        assert (h3 == h1).all() and len(surv) == 0
    finally:
        r.close()


def test_full_size_rollback_diff_properties(vm, orc, shm_tmp):
    """BASELINE config 4 at 10 GiB: 30 % of the blocks differ from the prior version; exactly those
    travel back over PCIe and are written, and the destination ends up identical to the source
    (block table of dst == block table of src; two whole files re-hashed by the oracle)."""
    src, dst = shm_tmp / "src", shm_tmp / "dst"
    dst.mkdir()
    nf, fb, bb = 10, 1 << 30, 4 * MiB
    vm.datagen_files(src, 4, nf, fb, threads=32)
    st0 = vm.migrate_tree(src, dst, None, shm_tmp / "v1.vmig")              # dst := v1, with its table
    assert st0["blocks_total"] == 2560 and st0["blocks_skipped"] == 0
    nblk = nf * fb // bb
    changed = np.sort(np.random.default_rng(44).permutation(nblk)[: nblk * 3 // 10])
    for g in changed:                                                         # block g of the table = file g//256, block g%256
        with open(src / f"f{g // 256:05d}.bin", "r+b") as f:
            f.seek((g % 256) * bb)
            w = bytes(x ^ 0xFF for x in f.read(8))
            f.seek((g % 256) * bb)
            f.write(w)
    st = vm.migrate_tree(src, dst, shm_tmp / "v1.vmig", shm_tmp / "v2.vmig")
    assert st["blocks_total"] - st["blocks_skipped"] == len(changed) == 768
    assert st["bytes_d2h"] == st["bytes_written"] == 768 * bb and st["bytes_h2d"] == nf * fb
    t1, t2 = vm.table_hashes(shm_tmp / "v1.vmig"), vm.table_hashes(shm_tmp / "v2.vmig")
    assert np.nonzero(t1 != t2)[0].tolist() == changed.tolist()
    vm.hash_tree(dst, shm_tmp / "dst.vmig")
    assert (vm.table_hashes(shm_tmp / "dst.vmig") == t2).all()              # dst == src, block for block
    for name in ("f00000.bin", "f00007.bin"):
        want = orc.hash_file(src / name)
        k = int(name[1:6]) * 256
        assert (t2[k:k + 256] == want).all() and (orc.hash_file(dst / name) == want).all()


def test_c_abi_data_path_from_plain_c(vm, orc, shm_tmp):
    """The C program of tests/c_abi_smoke.c (what cgo does: vmig_opts / vmig_stats by value, nullable tables, thread-local
    errors, vmig_move_dir) against the GPU: copy + verify on 2 lanes, a no-op diff pass, then the move; the moved tree is
    compared with the literal tar pipe's output."""
    import subprocess
    from test_host import build_c_abi_smoke, check_c_layout_line
    import tempfile
    exe_dir = Path(tempfile.mkdtemp(prefix="vmig_cabi_"))          # not /dev/shm: it is mounted noexec on the GPU box
    exe = build_c_abi_smoke(vm, exe_dir)
    src, dst, moved, ref = shm_tmp / "s", shm_tmp / "d", shm_tmp / "m", shm_tmp / "ref"
    src.mkdir(), dst.mkdir(), moved.mkdir(), ref.mkdir()
    make_rich_tree(src, orc)
    orc.ref_copy(src, ref)
    r = subprocess.run([str(exe), str(src), str(dst), str(moved), str(shm_tmp / "t.vmig")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    check_c_layout_line(vm, r.stdout)
    assert "copy ok" in r.stdout and "lanes=2" in r.stdout and "diff ok" in r.stdout and "move ok" in r.stdout, r.stdout
    shutil.rmtree(exe_dir, ignore_errors=True)
    assert orc.compare_trees(ref, moved, ignore_root_mtime=True) == []
    _, want = orc.block_table_of_tree(src)
    assert (vm.table_hashes(shm_tmp / "t.vmig") == want).all()


def test_prune_removes_what_the_source_no_longer_has(vm, orc, shm_tmp):
    """VMIG_F_PRUNE (final pass of a hand-off): entries the tenant deleted or renamed between two passes must not
    survive in the destination; without the flag they do (tar never prunes)."""
    src, dst, ref = shm_tmp / "src", shm_tmp / "dst", shm_tmp / "ref"
    src.mkdir(), dst.mkdir(), ref.mkdir()
    make_rich_tree(src, orc)
    (src / "gone_dir" / "deep").mkdir(parents=True)
    (src / "gone_dir" / "deep" / "x.bin").write_bytes(orc.splitmix_bytes(9, 5 * MiB).tobytes())
    (src / "old_name.bin").write_bytes(orc.splitmix_bytes(10, 4 * MiB + 5).tobytes())
    os.symlink("old_name.bin", src / "gone_link")
    vm.migrate_tree(src, dst, None, shm_tmp / "t1.vmig")
    shutil.rmtree(src / "gone_dir")
    os.rename(src / "old_name.bin", src / "new_name.bin")
    os.unlink(src / "gone_link")
    os.unlink(src / "sub" / "small.txt")              # one path of a hard-link pair
    st = vm.migrate_tree(src, dst, shm_tmp / "t1.vmig", shm_tmp / "t2.vmig")           # tar semantics: extras stay
    assert st["pruned"] == 0 and (dst / "gone_dir" / "deep" / "x.bin").exists() and (dst / "old_name.bin").exists()
    st = vm.migrate_tree(src, dst, shm_tmp / "t2.vmig", shm_tmp / "t3.vmig", flags=vm.F_PRUNE | vm.F_VERIFY)
    assert st["pruned"] == 6, st["pruned"]            # x.bin, deep, gone_dir, old_name.bin, gone_link, sub/small.txt
    orc.ref_copy(src, ref)
    assert orc.compare_trees(ref, dst) == []
    # an entry planted in the destination alone is removed as well, whatever it is
    (dst / "planted").mkdir(); (dst / "planted" / "f").write_bytes(b"x"); os.symlink("/etc", dst / "planted" / "esc")
    st = vm.migrate_tree(src, dst, shm_tmp / "t3.vmig", None, flags=vm.F_PRUNE)
    assert st["pruned"] == 3 and orc.compare_trees(ref, dst) == [] and os.path.isdir("/etc")


def test_stale_prior_table_is_not_trusted(vm, orc, shm_tmp):
    """The in-place diff path skips blocks whose source hash equals the prior table's entry, so the table must still
    describe the destination FILE.  Tables record (inode, ctime) of the file they were written for: after an
    out-of-band change of a destination file -- same size, mtime put back -- or with a table that belongs to another
    directory, that file is copied in full and the destination still ends up equal to the source."""
    src, dst = shm_tmp / "src", shm_tmp / "dst"
    src.mkdir(), dst.mkdir()
    for i in range(4):
        (src / f"f{i}.bin").write_bytes(orc.splitmix_bytes(80 + i, 9 * MiB + i).tobytes())
    vm.migrate_tree(src, dst, None, shm_tmp / "t1.vmig")
    ident = orc.read_table(shm_tmp / "t1.vmig")["identity"]
    for (ino, ct), name in zip(ident, sorted(os.listdir(dst))):
        stt = os.stat(dst / name)
        assert (ino, ct) == (stt.st_ino, stt.st_ctime_ns), name
    # tamper with dst/f1.bin behind the engine's back: block 1 now differs from the source, size and mtime unchanged
    before = os.stat(dst / "f1.bin")
    _mutate(dst / "f1.bin", 1)
    os.utime(dst / "f1.bin", ns=(before.st_atime_ns, before.st_mtime_ns))
    st = vm.migrate_tree(src, dst, shm_tmp / "t1.vmig", shm_tmp / "t2.vmig")
    assert st["files_untrusted"] == 1
    assert st["blocks_total"] - st["blocks_skipped"] == 3          # f1.bin's three blocks travel, nothing else
    for i in range(4):
        assert (dst / f"f{i}.bin").read_bytes() == (src / f"f{i}.bin").read_bytes(), i
    # a table written for ANOTHER directory is no licence to skip anything here
    other = shm_tmp / "other"
    other.mkdir()
    vm.migrate_tree(src, other, None, shm_tmp / "t_other.vmig")
    _mutate(dst / "f2.bin", 0)
    st = vm.migrate_tree(src, dst, shm_tmp / "t_other.vmig", None)
    assert st["files_untrusted"] == 4 and st["blocks_skipped"] == 0
    assert (dst / "f2.bin").read_bytes() == (src / "f2.bin").read_bytes()
    # format-01 tables (no identity) are read but never patched in place
    t = orc.read_table(shm_tmp / "t2.vmig")
    import struct
    raw = b"VMIGBT01" + struct.pack("<IIQQ", t["block_bytes"], 1, len(t["entries"]), len(t["hashes"]))
    for rel, size, first in t["entries"]:
        raw += struct.pack("<I", len(rel)) + rel + struct.pack("<QQ", size, first)
    (shm_tmp / "t_v1.vmig").write_bytes(raw + t["hashes"].astype("<u8").tobytes())
    _mutate(dst / "f3.bin", 2)
    st = vm.migrate_tree(src, dst, shm_tmp / "t_v1.vmig", None)
    assert st["blocks_skipped"] == 0 and (dst / "f3.bin").read_bytes() == (src / "f3.bin").read_bytes()


def _fs_type(path) -> str:
    import subprocess
    return subprocess.run(["stat", "-f", "-c", "%T", str(path)], capture_output=True, text=True).stdout.strip()


@pytest.mark.parametrize("mode", ["direct", "cufile", "direct+cufile"])
def test_disk_backed_tree_direct_io_and_gpudirect_storage(vm, orc, tmp_path, mode):
    """SURVEY.md §8f N4: a tree that is NOT on tmpfs (pytest's tmp_path lives on the box's root filesystem; the documented
    deployment keeps the Docker root on xfs/LVM, reference docs/volume/volume-size-scale-en.md:5-21).  O_DIRECT in and out
    of the pinned rings, cuFile in and out of the HBM slot, and both together must give what the literal tar pipe gives:
    every length that is awkward for whole-sector I/O is in the tree, and the in-place diff pass runs on the same path."""
    flags = {"direct": vm.F_DIRECT_IO, "cufile": vm.F_CUFILE, "direct+cufile": vm.F_DIRECT_IO | vm.F_CUFILE}[mode]
    src, dst, ref = tmp_path / "src", tmp_path / "dst", tmp_path / "ref"
    src.mkdir(), dst.mkdir(), ref.mkdir()
    if flags & vm.F_CUFILE:
        if not os.path.exists("/proc/driver/nvidia-fs"):
            # without the driver there is no GPUDirect Storage to test, only libcufile's POSIX compatibility mode, which on
            # B200 machines whose /tmp sits on a block device made no progress at all
            pytest.skip("the nvidia-fs driver is not loaded: no GPUDirect Storage on this machine")
        # libcufile decides per box whether it will take a descriptor at all (nvidia-fs module, filesystem, container):
        # where it refuses even a plain file, the path cannot be exercised here -- say so instead of failing on the box
        (tmp_path / "p").mkdir(), (tmp_path / "q").mkdir()
        (tmp_path / "p" / "x").write_bytes(b"probe" * 1000)
        try:
            vm.migrate_tree(tmp_path / "p", tmp_path / "q", flags=flags)
        except vm.VmigError as e:
            if "cuFileHandleRegister" in str(e) or "GPUDirect Storage unavailable" in str(e):
                pytest.skip(f"libcufile on this box accepts no descriptor on {_fs_type(tmp_path)}: {e}")
            raise
    make_rich_tree(src, orc)
    for i, n in enumerate([1, 511, 512, 4095, 4096, 4097, 8191, 4 * MiB - 1, 4 * MiB + 1, 8 * MiB, 13 * MiB + 4099]):
        (src / f"len{i:02d}.bin").write_bytes(orc.splitmix_bytes(300 + i, n).tobytes())
    st = vm.migrate_tree(src, dst, None, tmp_path / "t1.vmig", flags=flags | vm.F_VERIFY)
    orc.ref_copy(src, ref)
    assert orc.compare_trees(ref, dst) == []
    _, want = orc.block_table_of_tree(src)
    assert (vm.table_hashes(tmp_path / "t1.vmig") == want).all()
    assert st["bytes_written"] == st["bytes_total"] - (9 * MiB + 777) - 4097      # hard-linked paths are written once
    print(f"[{mode}] filesystem {_fs_type(tmp_path)}: {st['files_direct']} descriptors opened O_DIRECT, "
          f"{st['bytes_total'] / max(1, st['ns_total']):.2f} GB/s")
    if flags & vm.F_DIRECT_IO and _fs_type(tmp_path) not in ("tmpfs", "ramfs"):
        assert st["files_direct"] > 0, "the filesystem refused O_DIRECT for every file"
    # the diff pass patches in place through the same I/O path (whole-sector writes inside a file, truncation kept)
    _mutate(src / "len10.bin", 2)
    with open(src / "len09.bin", "r+b") as f:
        f.truncate(8 * MiB - 5)
    with open(src / "len07.bin", "ab") as f:
        f.write(b"tail" * 1000)
    st = vm.migrate_tree(src, dst, tmp_path / "t1.vmig", tmp_path / "t2.vmig", flags=flags | vm.F_VERIFY)
    assert st["blocks_skipped"] > 0 and st["files_untrusted"] == 0
    for name in ("len10.bin", "len09.bin", "len07.bin", "len00.bin", "big.bin"):
        assert (dst / name).read_bytes() == (src / name).read_bytes(), name
    _, want = orc.block_table_of_tree(src)
    assert (vm.table_hashes(tmp_path / "t2.vmig") == want).all()


def _handoff(vm):
    import importlib
    return importlib.import_module(vm.__name__ + ".handoff")


def test_handoff_two_pass_with_a_live_writer(vm, orc, shm_tmp):
    """SURVEY.md §8f N2, the sequence of integration/go/services/vmig_handoff.go::HandoffCopy: pass 1 while a writer
    keeps overwriting and appending to files of the source layer, pause (the writer stops), delete / rename in the
    paused layer, pass 2 with prior = pass 1's table + VERIFY + PRUNE.  The destination must equal the literal tar
    pipe's copy of the quiesced source, pass 2 must move only blocks of files the tenant touched, and the artefacts
    must sit where setToMergeMap puts them (merges/<rs>/<rs>-<v>/, internal/services/replicaset.go:681-704)."""
    ho = _handoff(vm)
    old, new, ref = shm_tmp / "upper_old", shm_tmp / "upper_new", shm_tmp / "ref"
    old.mkdir(), new.mkdir(), ref.mkdir()
    sizes = {f"f{i:02d}.bin": (6 + i) * MiB + 17 * i for i in range(12)}
    for name, n in sizes.items():
        (old / name).write_bytes(orc.splitmix_bytes(700 + len(name) + n, n).tobytes())
    hot = ["f00.bin", "f01.bin", "f02.bin"]                   # the tenant only touches these (and creates new ones)
    stop, paused = threading.Event(), threading.Event()

    def tenant():
        rng = np.random.default_rng(1)
        k = 0
        while not stop.is_set():
            name = hot[k % 3]
            with open(old / name, "r+b") as f:
                if k % 3 == 1:
                    f.seek(0, 2); f.write(rng.integers(0, 256, 7000, dtype=np.uint8).tobytes())       # append
                else:
                    f.seek(int(rng.integers(0, sizes[name] - 4096))); f.write(rng.integers(0, 256, 4096, dtype=np.uint8).tobytes())
            if k % 40 == 7:
                (old / f"new{k}.log").write_bytes(b"log line\n" * (k + 1))
            k += 1
            time.sleep(0.0005)
    th = threading.Thread(target=tenant)

    def pause(name):
        assert name == "rs-1"
        stop.set(); th.join(); paused.set()
        os.unlink(old / "f05.bin")                            # what the tenant did between the passes, seen only by pass 2
        os.rename(old / "f06.bin", old / "renamed06.bin")

    vm.set_resolver(container_upperdir=lambda n: str({"rs-1": old, "rs-2": new}[n]))
    ho.set_merges_root(shm_tmp)
    th.start()
    try:
        out = ho.HandoffCopy("rs-1", "rs-2", pause, lambda n: pytest.fail("resume called: the final pass failed"))
    finally:
        stop.set()
        if th.is_alive():
            th.join()
        vm.set_resolver(None, None); ho.set_merges_root(None)
    assert paused.is_set() and out["pass1"] is not None, out            # overwrite/append never shrinks a file: pass 1 succeeds
    p2 = out["pass2"]
    orc.ref_copy(old, ref)                                               # the reference's copy of the quiesced layer
    assert orc.compare_trees(ref, new) == []
    assert not (new / "f05.bin").exists() and not (new / "f06.bin").exists() and p2["pruned"] >= 2
    nblk = lambda n: -(-n // (4 * MiB))                                  # noqa: E731
    untouched = sum(nblk(sizes[f]) for f in sizes if f not in hot + ["f05.bin", "f06.bin"])
    assert p2["blocks_skipped"] >= untouched, (p2["blocks_skipped"], untouched)      # cold files did not travel again
    moved = p2["blocks_total"] - p2["blocks_skipped"]
    budget = sum(nblk((old / f).stat().st_size) for f in hot) + nblk(sizes["f06.bin"]) + sum(1 for p in old.glob("new*.log"))
    assert 0 < moved <= budget, (moved, budget)
    assert p2["bytes_d2h"] < p2["bytes_total"] // 2
    vdir = shm_tmp / "merges" / "rs" / "rs-2"
    assert (vdir / "blocks.vmig").exists() and not (vdir / "blocks.vmig.pass1").exists()
    _, want = orc.block_table_of_tree(old)
    assert (vm.table_hashes(vdir / "blocks.vmig") == want).all()


def test_handoff_live_pass_failure_falls_back_to_one_paused_pass(vm, orc, shm_tmp):
    """A tenant that truncates a file under the reader makes the live pass fail with VMIG_ESRCCHANGED (or not, if the
    race is lost); either way HandoffCopy ends with a verified paused pass and dst == src.  Then SnapshotVersion /
    RollbackFromSnapshot (N1): the snapshot sits in merges/<rs>/<rs>-<v>/diff with its table, and a rollback onto a
    layer seeded with another version moves only the differing blocks."""
    ho = _handoff(vm)
    old, new, ref = shm_tmp / "upper_old", shm_tmp / "upper_new", shm_tmp / "ref"
    old.mkdir(), new.mkdir(), ref.mkdir()
    for i in range(6):
        (old / f"g{i}.bin").write_bytes(orc.splitmix_bytes(900 + i, 24 * MiB + i).tobytes())
    stop = threading.Event()

    def tenant():
        k = 0
        while not stop.is_set():
            with open(old / "g0.bin", "r+b") as f:
                f.truncate(1 * MiB if k % 2 == 0 else 24 * MiB)
            k += 1
    th = threading.Thread(target=tenant)

    def pause(name):
        stop.set(); th.join()
        with open(old / "g0.bin", "r+b") as f:
            f.truncate(24 * MiB)

    vm.set_resolver(container_upperdir=lambda n: str({"rs-1": old, "rs-2": new, "rs-3": shm_tmp / "upper_3"}[n]))
    ho.set_merges_root(shm_tmp)
    th.start()
    try:
        out = ho.HandoffCopy("rs-1", "rs-2", pause, lambda n: pytest.fail("resume called"))
        assert out["pass1"] is not None or out["pass1_error"] == vm.VMIG_ESRCCHANGED
        orc.ref_copy(old, ref)
        assert orc.compare_trees(ref, new) == []
        # N1: snapshot version 2, create version 3 = version 2 with two blocks changed, roll a seeded layer back to 2
        st = ho.SnapshotVersion("rs-2")
        data, table = ho.snapshotPaths("rs-2")
        assert data == shm_tmp / "merges" / "rs" / "rs-2" / "diff" and table.exists() and st["blocks_skipped"] == 0
        assert orc.compare_trees(new, data) == []
        up3 = shm_tmp / "upper_3"
        up3.mkdir()
        seed = shm_tmp / "seed3.vmig"
        vm.migrate_tree(new, up3, None, seed)                  # the layer currently holds (a copy of) version 2 ...
        _mutate(up3 / "g3.bin", 2)                             # ... then drifts behind the engine's back: g3 is untrusted,
        st = ho.RollbackFromSnapshot("rs-2", "rs-3", seed)     # copied in full; the other five files do not travel
        assert st["files_untrusted"] == 1 and st["blocks_total"] - st["blocks_skipped"] == 7
        assert orc.compare_trees(data, up3) == []
    finally:
        stop.set()
        if th.is_alive():
            th.join()
        vm.set_resolver(None, None); ho.set_merges_root(None)


def test_smoke_entry_point():
    import __graft_entry__ as g
    g.smoke()
