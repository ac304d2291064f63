#!/usr/bin/env python
"""bench.py -- headline benchmark of the volume-migration hot path (BASELINE.json).

  python bench.py --gpus N --steps K --warmup W [--config 2A]      # our arm (libvmig on B200)
  python bench.py --impl reference --gpus N --steps K ...          # the reference's CPU path (tar | tar, mv)
  (N>1: python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...)

The metric of BOTH arms is "GiB/s data-disk migration on Patch": logical source bytes / wall time of the
call the control plane makes (ours: vmig_migrate_tree through the C ABI on host files, host<->HBM copies
inside the timed region; reference: the literal shell pipeline of utils/copy.go).  `value` and `e2e.value`
are that number; the HBM-resident hash pass ("block-hash GB/s") lives under `roofline`.

Configs (BASELINE.md §3; --config, default 2A which is what BASELINE.json's metric is quoted on for one GPU):
  1   1 GiB single file, Volume resize move across two mounts (reference: the `mv` command of copy.go:116)
  2A  ReplicaSet Patch, 10 GiB diff layer as 10 x 1 GiB files                       (the driver's workload)
  2B  the same 10 GiB as 40 960 files, log-uniform sizes, depth-4 tree, symlinks, empty files, a hard-link pair
  3   Volume resize 100 GiB: 100 x 1 GiB, ONE call whose block list is sharded over all N GPUs of the process
  4   Rollback, 50 GiB with 30 % changed blocks: prior table, exactly 3 840 written / 8 960 skipped
  5   N concurrent Patches (8 by default), 10 GiB each, N threads of ONE process, thread i on gpu_mask 1<<(i % gpus)
Weak scaling at N>1 (config 2A under torchrun): every rank migrates its own 10 GiB tree on its own GPU (blocks
are independent: no collective on the data path); rank 0 then also runs ONE call over an N x 10 GiB tree sharded
across all N GPUs in-process (`e2e_sharded`, the config-3 shape at N x 10 GiB).  Configs 3 and 5 are driven by
rank 0 alone.  Every config passes a parity gate (oracle block tables of src and dst, metadata vs the literal
tar pipe, exact skip counts) BEFORE its number is printed.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from (it may be read-only)
GiB, MiB = 1 << 30, 1 << 20
BLOCK = 4 << 20
METRIC = "GiB/s data-disk migration on Patch"
DATAGEN = ROOT / "tools" / "vmig_datagen"

CONFIGS = {
    "1": "cfg1 Volume resize move: 1 file x 1 GiB across two mounts (tmpfs)",
    "2A": "cfg2A ReplicaSet Patch 10 GiB data-disk: 10 x 1 GiB files, 4 MiB blocks, no prior table (tmpfs)",
    "2B": "cfg2B ReplicaSet Patch 10 GiB diff layer: 40 960 files log-uniform 1 KiB-64 MiB scaled to 10 GiB, depth-4 tree, 1 % symlinks, empty files, one hard-link pair (tmpfs)",
    "3": "cfg3 Volume resize 100 GiB: 100 x 1 GiB files, one call sharded across the GPUs (tmpfs)",
    "4": "cfg4 Rollback 50 GiB: 50 x 1 GiB files, 30 % of the blocks differ from the prior version, diff-skip (tmpfs)",
    "5": "cfg5 concurrent Patches: one 10 GiB tree (10 x 1 GiB) per caller thread, all in one process (tmpfs)",
}


_JSON_OUT = [None]


def claim_stdout() -> None:
    """The contract is ONE JSON line on stdout.  Native libraries (NCCL prints its version banner) and helpers write there
    too, so the real stdout is kept aside for the result line and fd 1 is pointed at stderr for everything else."""
    if _JSON_OUT[0] is None:
        sys.stdout.flush()
        _JSON_OUT[0] = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        sys.stdout = sys.stderr


def emit(line: dict) -> None:
    out = _JSON_OUT[0] or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def shm_base() -> Path:
    return Path(os.environ.get("VMIG_BENCH_DIR", "/dev/shm"))


class ClockSampler:
    """nvidia-smi clocks + throttle reasons while the timed region runs (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu: int):
        self.gpu, self.proc, self.lines = gpu, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
        except OSError:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "note": "sampled while the end-to-end steps ran; the path is host/PCIe-bound, so SM clocks idle low between the per-slot hash launches"}


_CPU_WAIT = [lambda: None]       # set by dist_setup: a barrier that parks ranks on the CPU (gloo), not inside an NCCL kernel
_BCAST = [lambda v: v]           # set by dist_setup: rank 0's value for everybody (gloo)


def bcast_from_rank0(v):
    return _BCAST[0](v)


def cpu_barrier() -> None:
    """Long waits (other ranks idle while rank 0 drives every GPU from one process) must not sit in an NCCL barrier:
    its kernel spins on the waiting rank's GPU and would time-slice against rank 0's hash kernels there."""
    _CPU_WAIT[0]()


def dist_setup():
    """(rank, world, local_rank, barrier, allmax).  torch.distributed (NCCL) is plumbing only."""
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world == 1:
        return rank, world, local, (lambda: None), (lambda x: x)
    import torch
    import torch.distributed as dist
    use_cuda = torch.cuda.is_available()
    if use_cuda:
        torch.cuda.set_device(local)
    dist.init_process_group("nccl" if use_cuda else "gloo")
    dev = torch.device("cuda", local) if use_cuda else torch.device("cpu")
    import datetime
    cpu_group = dist.new_group(backend="gloo", timeout=datetime.timedelta(minutes=30))
    _CPU_WAIT[0] = lambda: dist.barrier(group=cpu_group)

    def bcast(v):
        box = [v]
        dist.broadcast_object_list(box, src=0, group=cpu_group)
        return box[0]
    _BCAST[0] = bcast

    def barrier():
        dist.barrier()
        if use_cuda:
            torch.cuda.synchronize()

    def allmax(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return rank, world, local, barrier, allmax


def mem_budget_bytes() -> int:
    """Bytes this process may still put into tmpfs + page-locked memory: the tightest of the cgroup limit (v2 or v1),
    MemAvailable and the free space of the bench directory.  A GPU box that runs out of memory is lost, not slowed."""
    cands = []
    for lim, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                     ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            l = Path(lim).read_text().strip()
            if l != "max" and int(l) < (1 << 60):
                cands.append(int(l) - int(Path(cur).read_text().strip()))
        except (OSError, ValueError):
            pass
    try:
        for line in Path("/proc/meminfo").read_text().splitlines():
            if line.startswith("MemAvailable:"):
                cands.append(int(line.split()[1]) * 1024)
    except OSError:
        pass
    try:
        st = os.statvfs(shm_base())
        cands.append(st.f_bavail * st.f_frsize)
    except OSError:
        pass
    return min(cands) if cands else 1 << 62


def require_memory(need: int, what: str) -> None:
    have = mem_budget_bytes()
    if need > have * 0.85:
        raise SystemExit(f"bench.py: {what} needs {need / GiB:.0f} GiB of tmpfs + pinned memory but only {have / GiB:.0f} GiB "
                         f"are available to this container (cgroup limit / MemAvailable / {shm_base()}); refusing to run it "
                         "rather than drive the box out of memory")


def fresh_dir(p: Path) -> Path:
    shutil.rmtree(p, ignore_errors=True)
    p.mkdir(parents=True)
    return p


def datagen(mode: str, d: Path, seed: int, a: int, b: int, threads: int = 32) -> int:
    """tools/vmig_datagen (stand-alone: neither libvmig nor oracle/).  Returns the logical bytes generated."""
    if not DATAGEN.exists():
        subprocess.run(["make", "-C", str(ROOT / "tools"), "-s"], check=True)
    out = subprocess.run([str(DATAGEN), mode, str(d), str(seed), str(a), str(b), str(threads)], check=True,
                         capture_output=True, text=True).stdout
    return int(out.split("bytes=")[1].split()[0])


def ref_copy_cmd(src: Path, dst: Path) -> float:
    """Wall seconds of the reference's own copy engine (utils/copy.go:17-27) -- oracle/ref_copy.sh, verbatim."""
    t0 = time.perf_counter()
    r = subprocess.run([str(ROOT / "oracle" / "ref_copy.sh"), str(src), str(dst)], capture_output=True, text=True)
    dt = time.perf_counter() - t0
    if r.returncode != 0:
        raise RuntimeError(f"reference tar pipeline failed: {r.stderr}")
    return dt


def ref_move_cmd(src: Path, dst: Path) -> float:
    """Wall seconds of moveVolumeData's command (utils/copy.go:116) on host paths -- oracle/ref_move.sh, verbatim."""
    t0 = time.perf_counter()
    subprocess.run([str(ROOT / "oracle" / "ref_move.sh"), str(src), str(dst)], capture_output=True, text=True)
    return time.perf_counter() - t0


class TwoMounts:
    """Two separate tmpfs mounts (the reference's `mv` crosses bind mounts -> EXDEV copy + unlink, BASELINE.md §2).
    Falls back to /dev/shm vs /tmp when mounting is not permitted."""

    def __init__(self, tag: str, gib: int):
        self.base = shm_base() / f"vmig_mnt_{tag}"
        self.a, self.b, self.mounted = self.base / "a", self.base / "b", []
        fresh_dir(self.a), fresh_dir(self.b)
        for m in (self.a, self.b):
            if subprocess.run(["mount", "-t", "tmpfs", "-o", f"size={gib}g", "tmpfs", str(m)], capture_output=True).returncode == 0:
                self.mounted.append(m)
        if len(self.mounted) != 2:
            self.close()
            self.base = None
            self.a = fresh_dir(shm_base() / f"vmig_mnt_{tag}_a")
            self.b = fresh_dir(Path("/tmp") / f"vmig_mnt_{tag}_b")
        self.kind = "two tmpfs mounts" if len(self.mounted) == 2 else "/dev/shm (tmpfs) -> /tmp (different mount)"

    def close(self):
        for m in self.mounted:
            subprocess.run(["umount", "-l", str(m)], capture_output=True)
        self.mounted = []
        for p in (self.a, self.b, self.base):
            if p is not None:
                shutil.rmtree(p, ignore_errors=True)


def splitmix_shuffle_pick(n: int, k: int, seed: int) -> list:
    """First k entries of the Fisher-Yates shuffle of range(n) driven by the SplitMix64 stream `seed` (BASELINE.md §3 cfg4)."""
    M = (1 << 64) - 1

    def sm(j):
        z = (seed + (j + 1) * 0x9E3779B97F4A7C15) & M
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
        return z ^ (z >> 31)
    idx = list(range(n))
    for i in range(k):
        j = i + sm(i) % (n - i)
        idx[i], idx[j] = idx[j], idx[i]
    return sorted(idx[:k])


def flip_blocks(tree: Path, blocks: list, blocks_per_file: int) -> None:
    """XOR the first 8 bytes of each listed block (table order over f%05d.bin files) with 0xFF.. (cfg4's mutation)."""
    for g in blocks:
        with open(tree / f"f{g // blocks_per_file:05d}.bin", "r+b") as f:
            f.seek((g % blocks_per_file) * BLOCK)
            w = bytes(x ^ 0xFF for x in f.read(8))
            f.seek((g % blocks_per_file) * BLOCK)
            f.write(w)


# ------------------------------------------------------------------------------------------------ parity gates
def oracle_table(orc, tree: Path, threads: int = 16):
    """Oracle block table of a tree (oracle/xxh64_ref.c), files hashed by a thread pool (ctypes drops the GIL)."""
    import numpy as np
    files = []
    for dp, _dn, fn in os.walk(tree):
        for n in fn:
            p = os.path.join(dp, n)
            if os.path.isfile(p) and not os.path.islink(p):
                files.append((os.fsencode(os.path.relpath(p, tree)), p))
    files.sort()
    with ThreadPoolExecutor(threads) as ex:
        hs = list(ex.map(lambda t: orc.hash_file(t[1]), files))
    return np.concatenate(hs) if hs else np.empty(0, np.uint64)


def parity_gate(vm, orc, src: Path, dst: Path, table: Path | None, ref_tree: Path | None, what: str) -> dict:
    """BASELINE.md §5: every block hash == the oracle's; destination bytes == source bytes (oracle tables of both
    trees agree); metadata == what the literal tar pipe produced.  Raises before any number is printed."""
    t0 = time.perf_counter()
    want = oracle_table(orc, src)
    if table is not None:
        got = vm.table_hashes(table)
        assert got.shape == want.shape and (got == want).all(), f"{what}: engine block table != oracle"
    have = oracle_table(orc, dst)
    assert have.shape == want.shape and (have == want).all(), f"{what}: destination bytes differ from the source"
    meta = None
    if ref_tree is not None:
        diffs = orc.compare_trees(ref_tree, dst, content=False)
        assert not diffs, f"{what}: metadata differs from the tar pipe's output: {diffs[:5]}"
        meta = "mode/uid/gid/mtime/symlink/hardlink/special == literal tar pipe"
    return {"blocks_checked_vs_oracle": int(want.size), "dst_equals_src": True, "metadata": meta,
            "gate_s": round(time.perf_counter() - t0, 1)}


# ------------------------------------------------------------------------------------------------ --dump-outputs
DUMP_STATS = ("bytes_total", "bytes_h2d", "bytes_d2h", "bytes_written", "blocks_total", "blocks_skipped", "files", "dirs",
              "symlinks", "hardlinks", "specials", "pruned", "files_untrusted")
DUMP_SAMPLE_BYTES = 1 << 20


def dump_outputs(out_dir: Path, vm, dsts: list, tables: list, stats: dict) -> None:
    """What the last timed step handed its caller, as .npy arrays, so that two builds can be compared output for output on
    the same seeded workload: the block tables' XXH64 hashes (split into their 32-bit halves, which float64 holds exactly),
    the statistics counters that do not depend on timing (in DUMP_STATS order), the size of every destination file and a
    fixed, seeded sample of DUMP_SAMPLE_BYTES destination bytes.  Regular files are taken tree by tree, in bytewise path
    order.  A few MB in all: 16 B per block, 8 B per file, 4 MB of sample."""
    import numpy as np
    out_dir.mkdir(parents=True, exist_ok=True)
    if tables:
        h = np.concatenate([vm.table_hashes(t) for t in tables])
        np.save(out_dir / "block_hash_hi32.npy", (h >> np.uint64(32)).astype(np.float64))
        np.save(out_dir / "block_hash_lo32.npy", (h & np.uint64(0xFFFFFFFF)).astype(np.float64))
    np.save(out_dir / "stats.npy", np.array([stats[k] for k in DUMP_STATS], dtype=np.float64))
    files = []
    for d in dsts:
        tree = []
        for dp, _dn, fn in os.walk(d):
            for n in fn:
                p = os.path.join(dp, n)
                if os.path.isfile(p) and not os.path.islink(p):
                    tree.append((os.fsencode(os.path.relpath(p, d)), p))
        files += sorted(tree)
    sizes = np.array([os.path.getsize(p) for _rel, p in files], dtype=np.int64)
    np.save(out_dir / "dst_file_bytes.npy", sizes.astype(np.float64))
    ends = np.cumsum(sizes)
    total = int(ends[-1]) if len(ends) else 0
    pos = np.sort(np.random.default_rng(20).integers(0, total, min(total, DUMP_SAMPLE_BYTES))) if total else np.empty(0, np.int64)
    sample, lo = np.empty(len(pos), np.float32), 0
    for (_rel, p), size, end in zip(files, sizes, ends):
        hi = int(np.searchsorted(pos, end))
        if hi > lo:
            sample[lo:hi] = np.memmap(p, dtype=np.uint8, mode="r")[pos[lo:hi] - (end - size)]
        lo = hi
    np.save(out_dir / "dst_byte_sample.npy", sample)


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args) -> None:
    """--impl reference: the reference's CPU implementation of the path on this box's host cores.  Its engine is
    `sh -c "(cd S; tar c .) | (cd D; tar x)"` (two single-threaded processes per call: <= 2 cores per migration
    however many the box has) and, for Volume resize, the `mv` command.  Rank 0 alone runs; no GPU, no libvmig."""
    if int(os.environ.get("RANK", 0)) != 0:
        return
    cfg = args.config
    n_par, per_tree_files, seed0, mode = max(1, args.gpus), 10, 2, "tar"
    sample_note = "the full workload"
    if cfg == "1":
        n_par, per_tree_files, seed0, mode = 1, 1, 1, "mv"
    elif cfg == "2B":
        n_par = 1
    elif cfg == "3":
        n_par, per_tree_files, seed0 = 1, args.ref_sample_gib, 3
        sample_note = f"bounded sample: {per_tree_files} of the 100 x 1 GiB files per step"
    elif cfg == "4":
        n_par, per_tree_files, seed0 = 1, args.ref_sample_gib, 4
        sample_note = f"bounded sample: {per_tree_files} of the 50 x 1 GiB files per step (the reference has no diff path: it copies everything)"
    elif cfg == "5":
        n_par, seed0 = args.callers, 50
    base = fresh_dir(shm_base() / "vmig_bench_ref")
    mnt = None
    require_memory(int(2.1 * n_par * per_tree_files * GiB) if cfg != "2B" else 22 * GiB, f"reference arm, config {cfg}")
    try:
        srcs, nbytes = [], 0
        if mode == "mv":
            mnt = TwoMounts("ref", 3)
        for i in range(n_par):
            src = (mnt.a / "src") if mnt else base / f"src{i}"
            if cfg == "2B":
                nbytes += datagen("layer", src, 2, 10 * GiB, 40960)
            else:
                nbytes += datagen("files", src, seed0 + (i if cfg == "5" else 1000 * i), per_tree_files, GiB)
            srcs.append(src)
        times = []
        for i in range(args.warmup + args.steps):
            dsts = [fresh_dir((mnt.b / "dst") if mnt else base / f"dst{j}") for j in range(n_par)]
            if mode == "mv" and i > 0:
                datagen("files", srcs[0], seed0, per_tree_files, GiB)      # the move emptied it
            errs = []

            def one(j):
                try:
                    (ref_move_cmd if mode == "mv" else ref_copy_cmd)(srcs[j], dsts[j])
                except Exception as e:      # noqa: BLE001
                    errs.append(e)
            th = [threading.Thread(target=one, args=(j,)) for j in range(n_par)]
            t0 = time.perf_counter()
            [t.start() for t in th], [t.join() for t in th]
            dt = time.perf_counter() - t0
            if errs:
                raise errs[0]
            if mode == "mv":
                assert (dsts[0] / "f00000.bin").stat().st_size == GiB and not (srcs[0] / "f00000.bin").exists()
            if i >= args.warmup:
                times.append(dt)
        total = sum(times)
        v = nbytes * len(times) / total / GiB
        cmd = ("find SRC/ -maxdepth 1 -type f | xargs mv --target-directory=DST; mv SRC/* DST" if mode == "mv"
               else "(cd SRC; tar c .) | (cd DST; tar x)")
        sample = (f"{n_par} concurrent reference pipeline(s), {nbytes / GiB:.2f} GiB per step ({sample_note}), "
                  f"{args.steps} steps after {args.warmup} warm-up")
        cores = n_par * (1 if mode == "mv" else 2)
        line = {"impl": "reference", "metric": METRIC, "value": round(v, 3), "unit": "GiB/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * total / len(times), 1),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": CONFIGS[cfg], "reference_cmd": cmd, "mounts": mnt.kind if mnt else "tmpfs /dev/shm",
                           "parallelism": f"{n_par} independent trees, one reference pipeline each"},
                "cpu_baseline": {"value": round(v, 3), "unit": "GiB/s", "cores": cores, "kind": "reference",
                                 "sample": sample, "host_cpus": os.cpu_count()},
                "e2e": {"value": round(v, 3), "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit(line)
    finally:
        if mnt:
            mnt.close()
        shutil.rmtree(base, ignore_errors=True)


# ------------------------------------------------------------------------------------------------ our arm
def rank_plan(cfg: str, rank: int, world: int, gpus: int) -> dict:
    """Who does what at N>1 (spec: shard independent units across ranks, no data-path collective).  Config 2A is the
    weak-scaling workload: every rank migrates its OWN tree on its OWN GPU.  The other configs are single calls
    (or caller threads) of ONE process over all N GPUs -- the way the one-process control plane would run them --
    so rank 0 drives them alone and the other ranks only keep the barriers."""
    solo = cfg != "2A"
    n_box = max(1, world if world > 1 else gpus)
    return {"solo": solo, "active": rank == 0 or not solo, "n_gpus_box": n_box, "all_mask": (1 << n_box) - 1,
            "gpu": (rank if world > 1 else 0), "own_mask": 1 << (rank if world > 1 else 0),
            "tree": f"vmig_bench_r{rank}", "seed": 2 + 1000 * rank}


def hbm_resident_roofline(vm, gpu: int, passes: int) -> dict:
    """The dominant kernel (xxh64_blocks) over the config-2 batch ALREADY RESIDENT IN HBM (10 GiB = 2 560 blocks),
    CUDA events on the launching stream; inputs are far larger than the 126 MB L2, so no flush is needed."""
    n_blocks, nbytes = 10 * GiB // BLOCK, 10 * GiB
    res = vm.Resident(n_blocks, BLOCK, gpu)
    try:
        res.fill(0xB200)
        res.set_prior(None)
        for _ in range(3):
            res.run(1)
        k1_ms = [res.run(1)[0] for _ in range(max(3, passes))]
    finally:
        res.close()
    peaks_p = ROOT / "MEASURED_PEAKS.json"
    if peaks_p.exists():
        peak, peak_src = float(json.loads(peaks_p.read_text())["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"
    k1 = statistics.mean(k1_ms)
    algo = nbytes + 8 * n_blocks                      # N read + 8 B/block written (SURVEY.md §8d)
    achieved = algo / (k1 / 1e3) / 1e9
    traffic = None
    tp = ROOT / "profiles" / "k1_traffic.json"
    if tp.exists():
        traffic = json.loads(tp.read_text()).get("dram_bytes_per_launch")
    return {"bound": "hbm", "kernel": "xxh64_blocks", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
            "frac": round(achieved / peak, 4), "traffic": traffic, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": algo, "kernel_ms": round(k1, 4), "launches_timed": len(k1_ms),
            "block_hash_GBps": round(nbytes / (k1 / 1e3) / 1e9, 1),
            "what": "xxh64_blocks over 10 GiB (2 560 x 4 MiB blocks) resident in HBM, timed alone with CUDA events"}


def link_roofline(link: dict, nbytes: int, d2h_bytes: int, wall_s: float, n_gpu: int, hbm_peak: float) -> dict:
    """BASELINE.md §4: achieved fraction of the host<->HBM link (measured by vmig_link_probe in this run) and of HBM."""
    up, down = nbytes / wall_s / 1e9, d2h_bytes / wall_s / 1e9
    s = d2h_bytes / nbytes if nbytes else 0.0
    return {"h2d_GBps": round(up, 2), "d2h_GBps": round(down, 2),
            "h2d_peak_GBps": round(link["h2d_GBps"], 1), "d2h_peak_GBps": round(link["d2h_GBps"], 1),
            "duplex_h2d_peak_GBps": round(link["duplex_h2d_GBps"], 1), "duplex_d2h_peak_GBps": round(link["duplex_d2h_GBps"], 1),
            "h2d_frac": round(up / (n_gpu * link["h2d_GBps"]), 4), "d2h_frac": round(down / (n_gpu * link["d2h_GBps"]), 4),
            "h2d_frac_of_duplex": round(up / (n_gpu * link["duplex_h2d_GBps"]), 4),
            "d2h_frac_of_duplex": round(down / (n_gpu * link["duplex_d2h_GBps"]), 4) if d2h_bytes else 0.0,
            "hbm_e2e_frac": round((2 + s) * nbytes / wall_s / 1e9 / (n_gpu * hbm_peak), 5),
            "peak_source": "vmig_link_probe: pinned cudaMemcpyAsync sweep on GPU 0 in this run (4 GiB per direction, CUDA events), x n_gpus"}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="vmig", choices=["vmig", "reference"])
    ap.add_argument("--config", default="2A", choices=sorted(CONFIGS))
    ap.add_argument("--callers", type=int, default=8, help="config 5: concurrent caller threads")
    ap.add_argument("--lanes-per-gpu", type=int, default=0, help="vmig_opts.lanes_per_gpu (0 = library default)")
    ap.add_argument("--ref-sample-gib", type=int, default=20, help="reference arm, configs 3/4: GiB copied per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="N>1, config 2A: skip rank 0's one-call-over-all-GPUs leg")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the engine's outputs; it does not apply to --impl reference")
    if args.warmup < 3:
        args.warmup = 3
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
        return

    rank, world, local, barrier, allmax = dist_setup()
    import numpy as np           # noqa: F401  (oracle / package need it)
    import __graft_entry__ as g
    vm = g.load_pkg()
    cfg = args.config
    plan = rank_plan(cfg, local if world > 1 else 0, world, args.gpus)
    solo, n_gpus_box, gpu, all_mask = plan["solo"], plan["n_gpus_box"], plan["gpu"], plan["all_mask"]
    if world > 1 and not solo:
        # one process per GPU: tell each rank's engine how many migrations share the host's copy threads
        os.environ.setdefault("VMIG_IO_SHARE", str(world))
    active = plan["active"]
    if world > 1 and cfg == "2A" and not args.no_sharded:
        # rank 0's extra leg (one call over an N x 10 GiB tree) needs 22 GiB per GPU on top of the per-rank trees: drop it,
        # on every rank alike, where the container's memory does not allow it rather than fail the whole run
        fits = (32 + 22) * world * GiB <= 0.85 * mem_budget_bytes() if rank == 0 else None
        if not bcast_from_rank0(fits):
            args.no_sharded = True
    line = None
    base = fresh_dir(shm_base() / plan["tree"])
    mnt = None
    try:
        if active:
            vm.init(all_mask if (solo or (rank == 0 and world > 1 and not args.no_sharded)) else 1 << gpu)   # fails loudly without a B200
        orc = None
        if rank == 0:
            from oracle import oracle as orc        # parity gate + cpu_baseline leg only: the checker, never the measured path
            orc.build()
        lanes = args.lanes_per_gpu
        launches = 0
        gate = None
        extra = {}
        stats = None
        times: list = []
        nbytes = 0
        d2h_bytes = 0
        n_gpu_used = 1 if not solo else n_gpus_box
        ref_tree = None
        out_dsts, out_tables = [], []           # where the step leaves what it computed (--dump-outputs)
        clocks = ClockSampler(gpu)

        # ---------------- build the workload and the step
        need_gib = {"1": 4, "2A": 32 * (world if world > 1 else max(1, args.gpus)) + (22 * world if world > 1 and not args.no_sharded else 0), "2B": 32,
                    "3": 204, "4": 104, "5": 21 * args.callers + 4}[cfg]
        if rank == 0:
            require_memory(need_gib * GiB, f"config {cfg}")
        if cfg in ("2A", "2B"):
            if active:
                src = base / "src"
                # `--gpus N` WITHOUT torchrun: one process drives N GPUs, so the weak-scaled workload (N x 10 GiB) is ONE
                # call sharded across them in-process; under torchrun every rank has its own 10 GiB tree and GPU
                inproc_n = args.gpus if (world == 1 and cfg == "2A" and args.gpus > 1) else 1
                nbytes = datagen("files", src, plan["seed"], 10 * inproc_n, GiB) if cfg == "2A" else datagen("layer", src, 2, 10 * GiB, 40960)
                mask = (all_mask if inproc_n > 1 else 1 << gpu) if cfg == "2A" else 1
                n_gpu_used = inproc_n
                out_dsts, out_tables = [base / "dst"], [base / "table.vmig"]

                def step(i):
                    dst = fresh_dir(base / "dst")
                    barrier() if not solo else None
                    t0 = time.perf_counter()
                    st = vm.migrate_tree(src, dst, None, base / "table.vmig", gpu_mask=mask, lanes_per_gpu=lanes)
                    return time.perf_counter() - t0, st

                def gate_fn():
                    return parity_gate(vm, orc, src, base / "dst", base / "table.vmig", ref_tree, cfg)
        elif cfg == "3":
            if active:
                src = base / "src"
                nbytes = datagen("files", src, 3, 100, GiB)
                out_dsts, out_tables = [base / "dst"], [base / "table.vmig"]

                def step(i):
                    dst = fresh_dir(base / "dst")
                    t0 = time.perf_counter()
                    st = vm.migrate_tree(src, dst, None, base / "table.vmig", gpu_mask=all_mask, lanes_per_gpu=lanes)
                    return time.perf_counter() - t0, st

                def gate_fn():
                    return parity_gate(vm, orc, src, base / "dst", base / "table.vmig", None, cfg)
        elif cfg == "4":
            if active:
                src, dst = base / "src", fresh_dir(base / "dst")
                nfiles = 50
                nbytes = datagen("files", src, 4, nfiles, GiB)
                nblk = nbytes // BLOCK
                changed = splitmix_shuffle_pick(nblk, nblk * 3 // 10, 44)
                vm.migrate_tree(src, dst, None, None, gpu_mask=all_mask)            # dst := copy of src ...
                flip_blocks(dst, changed, GiB // BLOCK)                             # ... in which 30 % of the blocks differ = v1
                vm.hash_tree(dst, base / "v1.vmig", gpu_mask=all_mask)               # prior table = table of the pre-seeded dst
                v1_want = oracle_table(orc, dst)
                assert (vm.table_hashes(base / "v1.vmig") == v1_want).all(), "cfg4: prior table != oracle table of v1"
                out_dsts, out_tables = [dst], [base / "v2.vmig"]

                def step(i):
                    if i > 0:                       # outside the timed region: put dst back to v1 and re-take v1's table
                        flip_blocks(dst, changed, GiB // BLOCK)                     # (a table names the files it speaks for by inode +
                        vm.hash_tree(dst, base / "v1.vmig", gpu_mask=all_mask)       # ctime; the flips moved the ctimes)
                    t0 = time.perf_counter()
                    st = vm.migrate_tree(src, dst, base / "v1.vmig", base / "v2.vmig", gpu_mask=all_mask, lanes_per_gpu=lanes)
                    dt = time.perf_counter() - t0
                    assert st["blocks_total"] - st["blocks_skipped"] == len(changed) == 3840 and st["blocks_skipped"] == 8960, st
                    assert st["bytes_d2h"] == st["bytes_written"] == len(changed) * BLOCK, st
                    return dt, st

                def gate_fn():
                    r = parity_gate(vm, orc, src, dst, base / "v2.vmig", None, cfg)
                    t1, t2 = vm.table_hashes(base / "v1.vmig"), vm.table_hashes(base / "v2.vmig")
                    assert np.nonzero(t1 != t2)[0].tolist() == changed, "cfg4: the changed set differs from the mutated set"
                    r.update({"blocks_written": 3840, "blocks_skipped": 8960})
                    return r
        elif cfg == "5":
            if active:
                callers = args.callers
                srcs = []
                for i in range(callers):
                    nbytes += datagen("files", base / f"src{i}", 50 + i, 10, GiB)
                    srcs.append(base / f"src{i}")
                per_call = [[] for _ in range(callers)]
                out_dsts, out_tables = [base / f"dst{j}" for j in range(callers)], [base / f"t{j}.vmig" for j in range(callers)]

                def step(i):
                    dsts = [fresh_dir(base / f"dst{j}") for j in range(callers)]
                    out, errs = [None] * callers, []
                    go = threading.Barrier(callers + 1)

                    def one(j):
                        try:
                            go.wait()
                            t0 = time.perf_counter()
                            out[j] = vm.migrate_tree(srcs[j], dsts[j], None, base / f"t{j}.vmig", gpu_mask=1 << (j % n_gpus_box),
                                                     lanes_per_gpu=lanes)
                            per_call[j].append(time.perf_counter() - t0)
                        except Exception as e:      # noqa: BLE001
                            errs.append(e)
                    th = [threading.Thread(target=one, args=(j,)) for j in range(callers)]
                    [t.start() for t in th]
                    go.wait()
                    t0 = time.perf_counter()
                    [t.join() for t in th]
                    dt = time.perf_counter() - t0
                    if errs:
                        raise errs[0]
                    agg = dict(out[0])
                    for k in ("bytes_h2d", "bytes_d2h", "kernel_launches", "bytes_total"):
                        agg[k] = sum(o[k] for o in out)
                    return dt, agg

                def gate_fn():
                    r = None
                    for j in (0, callers - 1):
                        r = parity_gate(vm, orc, srcs[j], base / f"dst{j}", base / f"t{j}.vmig", None, f"cfg5 call {j}")
                    return r
        else:   # cfg 1
            if active:
                mnt = TwoMounts("vmig", 3)
                src = mnt.a / "src"
                nbytes = GiB
                want1 = None
                out_dsts = [mnt.b / "dst"]

                def step(i):
                    datagen("files", src, 1, 1, GiB)                 # the previous move emptied it
                    dst = fresh_dir(mnt.b / "dst")
                    t0 = time.perf_counter()
                    # exactly what vmig_move_dir / CopyOldMountPointToContainerMountPoint does, with the statistics returned
                    st = vm.migrate_tree(src, dst, None, None, gpu_mask=1, flags=vm.MOVE_DIR_FLAGS, lanes_per_gpu=lanes)
                    return time.perf_counter() - t0, st

                def gate_fn():
                    got = orc.hash_file(mnt.b / "dst" / "f00000.bin")
                    buf = orc.splitmix_bytes(orc.file_seed(1, "f00000.bin"), GiB)
                    assert (got == orc.hash_blocks(buf, np.arange(256, dtype=np.uint64) * BLOCK, [BLOCK] * 256)).all()
                    assert not (src / "f00000.bin").exists(), "cfg1: the move left the source file behind"
                    return {"blocks_checked_vs_oracle": 256, "dst_equals_src": True, "source_emptied": True}

        # ---------------- the reference tree for the metadata gate + the cpu_baseline leg (rank 0, outside the timed region)
        cpu = None
        if rank == 0 and not args.no_cpu_baseline and cfg in ("2A", "2B"):
            ref_tree = fresh_dir(base / "ref_dst")
            dt = ref_copy_cmd(src, ref_tree)
            buf = np.fromfile(src / "f00000.bin", dtype=np.uint8, count=256 * MiB) if cfg == "2A" else orc.splitmix_bytes(9, 256 * MiB)
            t0 = time.perf_counter(); orc.hash_blocks(buf, np.arange(64, dtype=np.uint64) * BLOCK, [BLOCK] * 64)
            hash_gbs = buf.size / (time.perf_counter() - t0) / 1e9
            cpu = {"value": round(nbytes / dt / GiB, 3), "unit": "GiB/s", "cores": 2, "kind": "reference",
                   "sample": f"the full {nbytes / GiB:.0f} GiB tree once through `(cd src; tar c .) | (cd dst; tar x)` (2 processes)",
                   "host_cpus": os.cpu_count(), "oracle_xxh64_1core_GBps": round(hash_gbs, 2)}

        # ---------------- timed steps: W warm-up (the first one is parity-gated), then K timed
        if active:
            for i in range(args.warmup + args.steps):
                if i == args.warmup:
                    clocks.start()
                dt, stats = step(i)
                if not solo:
                    barrier()
                    dt = allmax(dt)
                if i == 0 and rank == 0:
                    gate = gate_fn()                 # raises on any mismatch: no number without parity
                if i >= args.warmup:
                    times.append(dt)
                    launches += stats["kernel_launches"]
            d2h_bytes = stats["bytes_d2h"]
        elif not solo:
            pass
        clk = clocks.stop() if active else None
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, vm, out_dsts, out_tables, stats)
        if ref_tree is not None:
            shutil.rmtree(ref_tree, ignore_errors=True)

        # ---------------- N>1, config 2A: rank 0 alone drives all N GPUs with ONE call (north-star split)
        sharded = None
        if world > 1 and cfg == "2A" and not args.no_sharded:
            cpu_barrier()
            if rank == 0:
                shutil.rmtree(base / "dst", ignore_errors=True)
                big = base / "src_all"
                nb_all = datagen("files", big, 3, 10 * world, GiB)
                ts = []
                for i in range(2 + 3):
                    dst = fresh_dir(base / "dst_all")
                    t0 = time.perf_counter()
                    st = vm.migrate_tree(big, dst, None, base / "t_all.vmig", gpu_mask=all_mask, lanes_per_gpu=lanes)
                    dt = time.perf_counter() - t0
                    if i == 0:
                        parity_gate(vm, orc, big, dst, base / "t_all.vmig", None, "e2e_sharded")
                    if i >= 2:
                        ts.append(dt)
                sharded = {"value": round(nb_all * len(ts) / sum(ts) / GiB, 3), "unit": "GiB/s", "gpus_used": st["gpus_used"],
                           "lanes_used": st["lanes_used"], "bytes": nb_all, "ms_per_step": round(1e3 * statistics.mean(ts), 1),
                           "api": f"ONE vmig_migrate_tree call in rank 0's process, gpu_mask=0x{all_mask:x}: {10 * world} x 1 GiB sharded "
                                  "across the GPUs (whole files per lane); the other ranks idle", "steps": len(ts), "warmup": 2}
                shutil.rmtree(big, ignore_errors=True), shutil.rmtree(base / "dst_all", ignore_errors=True)
            cpu_barrier()

        if rank == 0:
            n_trees = world if not solo else 1
            total_bytes = nbytes * n_trees
            wall = sum(times) / len(times)
            value = total_bytes / wall / GiB
            roof = hbm_resident_roofline(vm, 0, args.steps)
            link = vm.link_probe(0, 4 * GiB)
            n_gpu_line = (world if world > 1 else n_gpu_used) if not solo else n_gpu_used
            roof["link"] = link_roofline(link, total_bytes, d2h_bytes * n_trees, wall, n_gpu_line, roof["peak"])
            roof["in_pipeline"] = {"launches_per_step": int(stats["kernel_launches"]), "mean_launch_ms": round(stats["ms_kernel"] / max(1, stats["kernel_launches"]), 3)
                                   if "ms_kernel" in stats else None,
                                   "note": "the e2e path hashes one staging slot per launch; launches of all slots overlap on side streams"}
            par = (f"one process, ONE call over {n_gpu_used} GPUs, block list sharded in-process (whole files per lane)" if (not solo and world == 1 and n_gpu_used > 1) else
                   f"{world} independent trees, one per GPU/rank, no collective" if not solo else
                   f"one process, {n_gpu_used} GPU(s)" + (f", {args.callers} caller threads" if cfg == "5" else ", block list sharded in-process"))
            line = {
                "metric": METRIC, "value": round(value, 3), "unit": "GiB/s", "n_gpus": world if world > 1 else args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * wall, 1), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None,
                "dtype": "u8 bytes moved; u64 XXH64 (integer mul/add/rotl) per 4 MiB block", "data": "synthetic",
                "config": {"workload": CONFIGS[cfg], "bytes_per_step": total_bytes, "blocks_per_step": total_bytes // BLOCK,
                           "l2": "every step streams >= 1 GiB (10 GiB by default) through HBM, far larger than the 126 MB L2; no flush needed",
                           "parallelism": par, "timing": "wall clock around the C-ABI call, barrier on both sides, max over ranks",
                           "lanes_per_gpu": lanes or int(os.environ.get("VMIG_LANES_PER_GPU", "1"))},
                "e2e": {"value": round(value, 3), "unit": "GiB/s", "h2d_bytes_per_step": int(stats["bytes_h2d"] * n_trees),
                        "d2h_bytes_per_step": int(d2h_bytes * n_trees), "ms_per_step": round(1e3 * wall, 1),
                        "api": "vmig_migrate_tree (utils.CopyDir drop-in) through the C ABI, tmpfs -> tmpfs, host files in and out",
                        "phases_ms": {k[3:]: round(stats[k] / 1e6, 1) for k in ("ns_walk", "ns_plan", "ns_data", "ns_meta", "ns_table")}},
                "gpu_launches": int(launches * n_trees), "parity_gate": gate,
                "roofline": roof, "cpu_baseline": cpu, "clocks": clk,
            }
            if sharded:
                line["e2e_sharded"] = sharded
            if cfg == "5":
                line["per_call_GiBps"] = [round(10 * GiB / statistics.mean(t[args.warmup:]) / GiB, 2) for t in per_call]
            if mnt:
                line["config"]["mounts"] = mnt.kind
            emit(line)
    finally:
        if mnt:
            mnt.close()
        shutil.rmtree(base, ignore_errors=True)
        try:
            vm.shutdown()
        except Exception:       # noqa: BLE001
            pass
    if world > 1:
        import torch.distributed as dist
        cpu_barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
