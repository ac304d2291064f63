"""CPU: the C-ABI library loads, exports every symbol include/vmig.h declares, its host-side
helpers agree with the oracle / the reference's Go helpers, and the data path FAILS LOUDLY
without a GPU (no CPU fallback).  No compute is done here."""
import ctypes
import json
import os
import re
import struct
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def _no_gpu(vm):
    try:
        vm.device_count()
        return False
    except vm.VmigError:
        return True


def test_library_exports_every_declared_symbol(vm):
    header = (ROOT / "include" / "vmig.h").read_text()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = sorted(set(re.findall(r"\b(vmig_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 25
    lib = ctypes.CDLL(str(vm.LIB_PATH))
    missing = [n for n in declared if not hasattr(lib, n)]
    assert not missing, missing
    assert sorted(vm.EXPORTS) == declared
    assert "sm_100a" in vm.version()


def build_c_abi_smoke(vm, out_dir):
    import subprocess
    exe = Path(out_dir) / "c_abi_smoke"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", str(ROOT / "include"), str(ROOT / "tests" / "c_abi_smoke.c"),
                    "-o", str(exe), str(vm.LIB_PATH), "-lpthread", "-Wl,-rpath," + str(vm.LIB_PATH.parent)], check=True)
    return exe


def check_c_layout_line(vm, stdout: str):
    """The `layout` line of c_abi_smoke (sizeof/offsetof as the C compiler sees include/vmig.h) == the ctypes mirror."""
    line = next(l for l in stdout.splitlines() if l.startswith("layout "))
    f = dict(kv.split("=") for kv in line.split()[1:])
    O, S, T = vm.Opts, vm.Stats, vm.TableInfo
    assert f["opts"] == f"{ctypes.sizeof(O)}:" + ",".join(str(getattr(O, n).offset) for n in
                                                        ("gpu_mask", "block_bytes", "streams_per_gpu", "flags", "io_threads", "lanes_per_gpu"))
    assert f["stats"] == f"{ctypes.sizeof(S)}:" + ",".join(str(getattr(S, n).offset) for n in (
        "bytes_total", "bytes_d2h", "blocks_skipped", "kernel_launches", "ns_total", "ns_table", "ms_kernel", "gpus_used", "lanes_used", "pruned"))
    assert f["tinfo"] == f"{ctypes.sizeof(T)}:" + ",".join(str(getattr(T, n).offset) for n in ("algo", "n_files", "bytes_total"))
    assert int(f["abi"]) == 2


def test_c_abi_from_plain_c(vm, shm_tmp):
    """include/vmig.h is plain C and the library links from C the way cgo would link it; the struct layout the C
    compiler sees equals the ctypes mirror's; without a GPU the data-path call is refused before it touches dst."""
    import subprocess
    import tempfile
    exe_dir = Path(tempfile.mkdtemp(prefix="vmig_cabi_"))          # /dev/shm may be mounted noexec
    exe = build_c_abi_smoke(vm, exe_dir)
    src, dst, moved = shm_tmp / "s", shm_tmp / "d", shm_tmp / "m"
    (src / "sub").mkdir(parents=True), dst.mkdir(), moved.mkdir()
    (src / "a").write_bytes(b"x" * 5000), (src / "sub" / "b").write_bytes(b"y" * 70)
    r = subprocess.run([str(exe), str(src), str(dst), str(moved), str(shm_tmp / "t.vmig")], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    check_c_layout_line(vm, r.stdout)
    assert "files=2 bytes=5070 dir_size=5070" in r.stdout
    if "copy ok" in r.stdout:
        assert "diff ok skipped=2 of 2" in r.stdout and "move ok" in r.stdout
        assert (moved / "sub" / "b").read_bytes() == b"y" * 70
    else:
        assert "no CPU fallback" in r.stdout and os.listdir(dst) == []


def test_source_side_path_safety_unit(shm_tmp, tmp_path):
    """csrc/vmig_tree.cpp alone (no GPU, no CUDA): open_beneath refuses symlinks and escapes, the walk does not
    descend through symlinked directories, remove_source cannot be steered out of the tree; prune_extras (VMIG_F_PRUNE)
    removes exactly the entries the manifest lacks and never follows a symlink; the walk gives the same manifest with
    one thread and with eight (hard-link pair across two sub-walks included); without root, modes follow tar without -p."""
    import subprocess
    exe = tmp_path / "tree_unit"          # not /dev/shm: it may be mounted noexec
    csrc = ROOT / "gpu-docker-api_b200" / "csrc"
    subprocess.run(["g++", "-std=c++17", "-Wall", "-Werror", "-pthread", "-I", str(csrc), str(ROOT / "tests" / "tree_unit.cpp"),
                    str(csrc / "vmig_tree.cpp"), "-o", str(exe)], check=True)
    work = shm_tmp / "tu"
    work.mkdir()
    r = subprocess.run([str(exe), str(work)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and "tree unit ok" in r.stdout, r.stdout + r.stderr


def test_copy_thread_budget_is_per_box_and_divided_among_lanes(vm, monkeypatch):
    """The host's page-cache copy capacity belongs to the box: 20 copy threads for one GPU however many lanes share it,
    13 per GPU beyond (DESIGN.md §3, profiles/r02_sweep_lanes_1gpu.txt, r01_e2e_rank_scaling.txt)."""
    for k in ("VMIG_READERS", "VMIG_WRITERS", "VMIG_IO_SHARE"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("VMIG_PLAN_CPUS", "128")
    assert vm.thread_plan(1, 1) == (8, 12)                       # one lane, one GPU
    assert vm.thread_plan(2, 1) == (4, 6) and vm.thread_plan(4, 1) == (2, 3)      # lanes share the GPU's 20
    assert vm.thread_plan(8, 8) == (5, 8)                        # 104 for eight GPUs, 13 per lane
    assert vm.thread_plan(1, 1, flags=vm.F_HASH_ONLY) == (16, 1)
    assert vm.thread_plan(1, 1, has_prior=True) == (12, 12)
    monkeypatch.setenv("VMIG_IO_SHARE", "8")                     # one process per GPU (bench.py under torchrun)
    assert vm.thread_plan(1, 1) == (5, 8)
    monkeypatch.delenv("VMIG_IO_SHARE")
    monkeypatch.setenv("VMIG_PLAN_CPUS", "8")                    # a small host caps the budget at 7/8 of its CPUs
    r, w = vm.thread_plan(1, 1)
    assert r + w <= 7 and r >= 2 and w >= 2
    monkeypatch.setenv("VMIG_READERS", "3"), monkeypatch.setenv("VMIG_WRITERS", "9")
    assert vm.thread_plan(4, 2) == (3, 9)                        # explicit per-lane counts win


def test_writer_queue_invariants(tmp_path):
    """csrc/vmig_sched.h alone (no GPU): one worker per key at a time, per-key FIFO, every task exactly once."""
    import subprocess
    exe = tmp_path / "sched_unit"
    csrc = ROOT / "gpu-docker-api_b200" / "csrc"
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Werror", "-pthread", "-I", str(csrc), str(ROOT / "tests" / "sched_unit.cpp"),
                    "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "sched unit ok" in r.stdout, r.stdout + r.stderr


def test_block_transfer_loop(tmp_path):
    """csrc/vmig_common.h transfer_block alone (no GPU): buffered resume at the exact byte, O_DIRECT resume from the
    sector boundary, a short last block, no progress and a failing transfer -- with a scripted fake in place of the I/O."""
    import subprocess
    exe = tmp_path / "xfer_unit"
    csrc = ROOT / "gpu-docker-api_b200" / "csrc"
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Werror", "-I", str(csrc), str(ROOT / "tests" / "xfer_unit.cpp"),
                    "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and "xfer unit ok" in r.stdout, r.stdout + r.stderr


def test_struct_layouts_match_header(vm):
    assert ctypes.sizeof(vm.Opts) == 32
    assert ctypes.sizeof(vm.Stats) == 18 * 8 + 8 + 8 + 24
    assert ctypes.sizeof(vm.TableInfo) == 32


def test_strerror_table(vm):
    assert vm.strerror(0) == "ok"
    assert "no CPU fallback" in vm.strerror(vm.VMIG_ENOGPU)
    assert vm.strerror(-12345).startswith("unknown")


def test_to_bytes_matches_reference_rules(vm):
    # reference utils/file.go:24-48: 1024-based, unit = last two chars, ParseFloat on the rest
    assert vm.ToBytes("20GB") == 20 << 30
    assert vm.ToBytes("1.5MB") == int(1.5 * (1 << 20))
    assert vm.ToBytes("100KB") == 100 << 10 and vm.ToBytes("2TB") == 2 << 40
    for bad in ["20gb", "GB", "12", "1PB", "x1GB", " 1GB", "\t2MB", "1 GB", "1.5.5KB"]:
        with pytest.raises(vm.VmigError):
            vm.ToBytes(bad)


def test_dir_size_matches_walk(vm, shm_tmp):
    (shm_tmp / "a" / "b").mkdir(parents=True)
    (shm_tmp / "a" / "f1").write_bytes(b"x" * 1000)
    (shm_tmp / "a" / "b" / "f2").write_bytes(b"y" * 4097)
    os.symlink("f1", shm_tmp / "a" / "l")
    want = sum(os.lstat(os.path.join(d, f)).st_size for d, _, fs in os.walk(shm_tmp) for f in fs)
    assert vm.DirSize(str(shm_tmp)) == want
    with pytest.raises(vm.VmigError):
        vm.DirSize(str(shm_tmp / "nope"))


def test_datagen_matches_oracle_generator(vm, orc, shm_tmp):
    vm.datagen_files(shm_tmp / "g", 7, 3, (4 << 20) + 12345, threads=4)
    for i in range(3):
        name = f"f{i:05d}.bin"
        got = np.fromfile(shm_tmp / "g" / name, dtype=np.uint8)
        want = orc.splitmix_bytes(orc.file_seed(7, name), (4 << 20) + 12345)
        assert got.size == want.size and (got == want).all(), name


def _write_table(path, entries, hashes, block_bytes=4 << 20, identity=None):
    """identity None -> format 01 (no file identity); else a list of (ino, ctime_ns) -> format 02."""
    raw = (b"VMIGBT01" if identity is None else b"VMIGBT02") + struct.pack("<IIQQ", block_bytes, 1, len(entries), len(hashes))
    for i, (rel, size, first) in enumerate(entries):
        raw += struct.pack("<I", len(rel)) + rel + struct.pack("<QQ", size, first)
        if identity is not None:
            raw += struct.pack("<Qq", *identity[i])
    raw += np.asarray(hashes, dtype="<u8").tobytes()
    Path(path).write_bytes(raw)
    return raw


def test_block_table_reader_accepts_good_and_rejects_bad(vm, orc, shm_tmp):
    entries = [(b"a/x.bin", (8 << 20) + 1, 0), (b"b.bin", 100, 3), (b"empty", 0, 4)]
    hashes = [11, 22, 33, 44]
    p = shm_tmp / "t.vmig"
    raw = _write_table(p, entries, hashes)
    info = vm.table_info(p)
    assert info == {"block_bytes": 4 << 20, "algo": 1, "n_files": 3, "n_blocks": 4, "bytes_total": (8 << 20) + 101}
    assert list(vm.table_hashes(p)) == hashes
    assert orc.read_table(p)["entries"] == entries              # the oracle's parser agrees on the format
    ident = [(12345, 1_700_000_000_123_456_789), (7, -5), (0, 0)]     # format 02: + (inode, ctime_ns) per file
    raw2 = _write_table(shm_tmp / "t2.vmig", entries, hashes, identity=ident)
    assert vm.table_info(shm_tmp / "t2.vmig") == info and list(vm.table_hashes(shm_tmp / "t2.vmig")) == hashes
    t2 = orc.read_table(shm_tmp / "t2.vmig")
    assert t2["entries"] == entries and t2["identity"] == ident
    for bad in [raw2[:-1], raw2[:60], b"VMIGBT01" + raw2[8:], b"VMIGBT03" + raw2[8:]]:
        (shm_tmp / "bad").write_bytes(bad)
        with pytest.raises(vm.VmigError) as ei:
            vm.table_info(shm_tmp / "bad")
        assert ei.value.code == vm.VMIG_ETABLE
    for bad in [raw[:-1], b"XMIGBT01" + raw[8:], raw[:40], raw + b"\0" * 8]:
        (shm_tmp / "bad").write_bytes(bad)
        with pytest.raises(vm.VmigError) as ei:
            vm.table_info(shm_tmp / "bad")
        assert ei.value.code == vm.VMIG_ETABLE
    _write_table(shm_tmp / "unsorted", [(b"b", 1, 0), (b"a", 1, 1)], [1, 2])
    with pytest.raises(vm.VmigError):
        vm.table_info(shm_tmp / "unsorted")
    _write_table(shm_tmp / "gap", [(b"a", 1, 0), (b"b", 1, 2)], [1, 2, 3])
    with pytest.raises(vm.VmigError):
        vm.table_info(shm_tmp / "gap")


def test_block_table_golden_fixture(vm, orc):
    """tests/golden/table_v2.vmig (committed bytes, written by make_table_golden.py): libvmig's reader and the oracle's parser
    both return what the fixture's JSON says -- the on-disk format VMIGBT02 is pinned."""
    g = ROOT / "tests" / "golden"
    want = json.loads((g / "table_v2.json").read_text())
    info = vm.table_info(g / "table_v2.vmig")
    assert info == {k: want[k] for k in ("block_bytes", "algo", "n_files", "n_blocks", "bytes_total")}
    assert [f"{int(h):016x}" for h in vm.table_hashes(g / "table_v2.vmig")] == want["hashes"]
    t = orc.read_table(g / "table_v2.vmig")
    assert [[rel.decode("utf-8"), size] for rel, size, _ in t["entries"]] == want["entries"]
    assert [list(i) for i in t["identity"]] == want["identity"]
    assert [f"{int(h):016x}" for h in t["hashes"]] == want["hashes"]


def test_block_table_reader_survives_corruption(vm, shm_tmp):
    """A prior table is an input file: 400 random truncations / byte flips / count edits of a valid table are
    either rejected with VMIG_ETABLE or load as a self-consistent table -- the reader never crashes or over-reads
    (each mutant is parsed in this process, so a wild read would take the test run down)."""
    rng = np.random.default_rng(7)
    entries = [(f"d{i % 7}/f{i:03d}.bin".encode(), int(rng.integers(0, 20 << 20)), 0) for i in range(40)]
    entries.sort()
    fixed, fb = [], 0
    for rel, size, _ in entries:
        fixed.append((rel, size, fb))
        fb += (size + (4 << 20) - 1) // (4 << 20)
    raw = bytearray(_write_table(shm_tmp / "good.vmig", fixed, [int(x) for x in rng.integers(0, 1 << 63, fb)]))
    assert vm.table_info(shm_tmp / "good.vmig")["n_blocks"] == fb
    p = shm_tmp / "mut.vmig"
    rejected = 0
    for k in range(400):
        m = bytearray(raw)
        kind = k % 4
        if kind == 0:
            m = m[: int(rng.integers(0, len(m)))]
        elif kind == 1:
            for _ in range(int(rng.integers(1, 6))):
                m[int(rng.integers(0, len(m)))] ^= 1 << int(rng.integers(0, 8))
        elif kind == 2:                                   # header counts / a path length blown up
            off = int(rng.choice([8, 16, 24, 32]))
            m[off:off + 4] = int(rng.integers(0, 1 << 32)).to_bytes(4, "little")
        else:
            m += bytes(int(rng.integers(1, 64)))
        p.write_bytes(bytes(m))
        try:
            info = vm.table_info(p)
            h = vm.table_hashes(p)
            assert len(h) == info["n_blocks"] and info["n_files"] <= 40 + 1
        except vm.VmigError as e:
            assert e.code == vm.VMIG_ETABLE, e
            rejected += 1
    assert rejected > 200          # most mutants are structurally broken; flips inside hashes/sizes may load


def test_manifest_pass_matches_oracle_walk(vm, orc, shm_tmp):
    """The engine's tree walk (ordering, block layout, hard links, specials, the `mv *` quirk) against the
    oracle's independent walk -- no GPU involved (vmig_manifest)."""
    from conftest import make_rich_tree
    src = shm_tmp / "src"
    src.mkdir()
    make_rich_tree(src, orc)
    st = vm.manifest(src, shm_tmp / "m.vmig")
    entries, hashes = orc.block_table_of_tree(src)
    tab = orc.read_table(shm_tmp / "m.vmig")
    assert tab["entries"] == entries                              # same files, sizes, first_block, bytewise order
    assert len(tab["hashes"]) == len(hashes) and not tab["hashes"].any()
    assert st["bytes_total"] == sum(e[1] for e in entries) and st["blocks_total"] == len(hashes)
    assert st["files"] == len(entries) and st["symlinks"] == 2 and st["hardlinks"] == 2
    assert st["specials"] == (2 if os.geteuid() == 0 else 1)      # fifo (+ whiteout char device as root)
    n_dirs = 1 + sum(len(d) for _, d, _ in os.walk(src))
    assert st["dirs"] == n_dirs
    # DirSize (utils/file.go:13-22) counts every non-directory's st_size; the manifest counts regular files
    assert vm.DirSize(str(src)) >= st["bytes_total"]
    # the reference's `mv /root/src/*` leaves top-level hidden directories behind
    st2 = vm.manifest(src, shm_tmp / "m2.vmig", flags=vm.F_SKIP_HIDDEN_TOPDIRS)
    assert st2["files"] == st["files"] - 1 and st2["dirs"] == st["dirs"] - 1
    assert all(not e[0].startswith(b".hidden_dir/") for e in orc.read_table(shm_tmp / "m2.vmig")["entries"])
    with pytest.raises(vm.VmigError):
        vm.manifest(shm_tmp / "nope")


def test_manifest_matches_oracle_walk_on_random_trees(vm, orc, shm_tmp):
    """Property test (hypothesis): for random directory trees -- awkward names, empty files and directories, sizes around the
    block size (a tiny block size keeps the trees small), hard links across directories, symlinks -- the engine's manifest
    (parallel walk) lists the same files, sizes and block layout as the oracle's independent walk, and DirSize / the used-bytes
    figure agree with a plain os.walk."""
    from hypothesis import given, settings, strategies as st, HealthCheck
    names = st.text(alphabet=st.sampled_from(list("abcXYZ019 ._-é#")), min_size=1, max_size=6).filter(lambda n: n not in (".", "..") and "/" not in n)
    counter = [0]

    @settings(max_examples=25, deadline=None, suppress_health_check=[HealthCheck.function_scoped_fixture])
    @given(st.lists(st.tuples(st.lists(names, min_size=0, max_size=3), names, st.integers(0, 3 * 4096 + 7), st.sampled_from(["file", "file", "file", "dir", "symlink", "hardlink"])),
                    min_size=0, max_size=14))
    def run(items):
        counter[0] += 1
        root = shm_tmp / f"t{counter[0]}"
        root.mkdir()
        made_files = []
        for dirs, name, size, kind in items:
            d = root.joinpath(*dirs) if dirs else root
            try:
                d.mkdir(parents=True, exist_ok=True)
            except (FileExistsError, NotADirectoryError):
                continue
            p = d / name
            if p.exists() or p.is_symlink():
                continue
            if kind == "file":
                p.write_bytes(bytes(size)); made_files.append(p)
            elif kind == "dir":
                p.mkdir()
            elif kind == "symlink":
                os.symlink("some/where", p)
            elif made_files:
                os.link(made_files[0], p)
        bb = 4096
        stt = vm.manifest(root, shm_tmp / f"m{counter[0]}.vmig", block_bytes=bb)
        entries, hashes = orc.block_table_of_tree(root, bb)
        tab = orc.read_table(shm_tmp / f"m{counter[0]}.vmig")
        assert tab["block_bytes"] == bb and tab["entries"] == entries and len(tab["hashes"]) == len(hashes)
        want_bytes = sum(os.lstat(os.path.join(dp, f)).st_size for dp, _, fs in os.walk(root) for f in fs if not os.path.islink(os.path.join(dp, f)))
        assert stt["bytes_total"] == want_bytes == sum(e[1] for e in entries)
        assert stt["dirs"] == 1 + sum(len(ds) for _, ds, _ in os.walk(root))
        assert vm.DirSize(str(root)) == sum(os.lstat(os.path.join(dp, f)).st_size for dp, _, fs in os.walk(root) for f in fs)
    run()


def test_to_bytes_property(vm):
    """Property test: vmig_to_bytes == the reference's rule (utils/file.go:24-48: last two characters are the unit, the rest is
    strconv.ParseFloat, 1024-based, truncated to int64) for random magnitudes and units; anything else is VMIG_EINVAL."""
    from hypothesis import given, settings, strategies as st
    mult = {"KB": 1 << 10, "MB": 1 << 20, "GB": 1 << 30, "TB": 1 << 40}

    @settings(max_examples=200, deadline=None)
    @given(st.floats(min_value=0, max_value=4096, allow_nan=False, allow_infinity=False), st.sampled_from(sorted(mult)), st.integers(0, 3))
    def ok(x, unit, digits):
        text = f"{x:.{digits}f}{unit}"
        assert vm.ToBytes(text) == int(float(f"{x:.{digits}f}") * mult[unit])
    ok()

    @settings(max_examples=100, deadline=None)
    @given(st.text(alphabet=st.sampled_from(list("0123456789.kKmMgGtTbBxX -")), min_size=0, max_size=8))
    def bad(text):
        good = len(text) >= 3 and text[-2:] in mult
        try:
            float(text[:-2]) if good else None
            if good and (text[:-2].strip() != text[:-2] or text[:-2].lower() in ("inf", "nan") or "x" in text[:-2].lower()):
                good = False
        except ValueError:
            good = False
        if not good:
            with pytest.raises(vm.VmigError):
                vm.ToBytes(text)
    bad()


def test_reference_interface_resolvers(vm):
    vm.set_resolver(None, None)
    with pytest.raises(vm.VmigError):
        vm.GetContainerMergedLayer("rs-1")
    vm.set_resolver(lambda n: "" if n == "missing" else f"/var/lib/docker/overlay2/{n}/diff", lambda n: f"/vol/{n}/_data")
    assert vm.GetContainerMergedLayer("rs-2") == "/var/lib/docker/overlay2/rs-2/diff"
    assert vm.GetVolumeMountPoint("v-1") == "/vol/v-1/_data"
    with pytest.raises(vm.VmigError):           # empty UpperDir is an error (utils/copy.go:50-52)
        vm.GetContainerMergedLayer("missing")
    vm.set_resolver(None, None)


def test_argument_validation_needs_no_gpu(vm, shm_tmp):
    with pytest.raises(vm.VmigError) as ei:
        vm.migrate_tree(None, shm_tmp)
    assert ei.value.code == vm.VMIG_EINVAL
    with pytest.raises(vm.VmigError) as ei:
        vm.migrate_tree(shm_tmp / "nope", shm_tmp)
    assert ei.value.code == vm.VMIG_EIO
    (shm_tmp / "file").write_bytes(b"1")
    with pytest.raises(vm.VmigError) as ei:
        vm.migrate_tree(shm_tmp / "file", shm_tmp)
    assert ei.value.code == vm.VMIG_ENOTDIR
    with pytest.raises(vm.VmigError) as ei:
        vm.migrate_tree(shm_tmp, shm_tmp, block_bytes=1000)
    assert ei.value.code == vm.VMIG_EINVAL


def test_no_cpu_fallback_without_gpu(vm, shm_tmp):
    """On a GPU-less box every data-path call must fail with VMIG_ENOGPU and leave dst alone."""
    if not _no_gpu(vm):
        pytest.skip("a GPU is present; the -m gpu tests cover the data path")
    src, dst = shm_tmp / "s", shm_tmp / "d"
    src.mkdir(), dst.mkdir()
    (src / "f").write_bytes(b"payload")
    for call in (lambda: vm.CopyDir(str(src), str(dst)),
                 lambda: vm.migrate_tree(src, dst),
                 lambda: vm.hash_blocks(np.zeros(64, np.uint8), [0], [64]),
                 lambda: vm.migrate_buffer(np.zeros(4096, np.uint8), np.zeros(4096, np.uint8)),
                 lambda: vm.Resident(4),
                 lambda: vm.init(0)):
        with pytest.raises(vm.VmigError) as ei:
            call()
        assert ei.value.code == vm.VMIG_ENOGPU, ei.value
    assert os.listdir(dst) == []
    assert (src / "f").exists()
