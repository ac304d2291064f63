/*
 * vmig.h -- C ABI of libvmig, the B200-native volume-migration engine.
 *
 * Drop-in boundary for the ONE data-parallel path of XShengTech/gpu-docker-api: the bulk copy
 * of a container's system-disk diff layer (ReplicaSet Patch / Rollback / Restart) and of a
 * Docker-volume data disk (Volume resize).  The reference has no plugin/FFI interface; the
 * seam is three package-level Go functions in package utils (SURVEY.md §8b):
 *
 *   utils.CopyDir(src, dest string) error                         reference utils/copy.go:21-27
 *   utils.CopyOldMergedToNewContainerMerged(old, new string) error reference utils/copy.go:31-46
 *   utils.CopyOldMountPointToContainerMountPoint(old, new) error   reference utils/copy.go:58-63
 *     (-> moveVolumeData, reference utils/copy.go:74-128)
 *
 * called from internal/services/replicaset.go:333,421,831 and internal/services/volume.go:150.
 * A cgo shim (INTEGRATION.md) re-implements those three functions on top of the entry points
 * below; nothing else in the reference changes.
 *
 * Conventions (what a cgo binding needs):
 *   - every function returns 0 (VMIG_OK) or a negative VMIG_E* code; vmig_last_error() gives a
 *     thread-local human-readable message for the calling thread's last failure;
 *   - all pointers are borrowed for the duration of the call only (no Go memory is retained);
 *   - no callbacks into the caller; every entry point is re-entrant and thread-safe (the
 *     reference calls the copy from concurrent gin goroutines with no locking, SURVEY.md F9);
 *   - there is NO CPU fallback: without a usable sm_100 device the data-path calls fail with
 *     VMIG_ENOGPU.
 *
 * Data path of one migration (DESIGN.md):  source file blocks (4 MiB, file-aligned) -> pinned
 * host slot -> cudaMemcpyAsync H2D on a side stream -> xxh64_blocks kernel (canonical XXH64,
 * seed 0, one hash per block) -> compare with the prior version's block table -> surviving
 * blocks cudaMemcpyAsync D2H into the destination pinned slot -> destination file.
 */
#ifndef VMIG_H
#define VMIG_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VMIG_ABI_VERSION 2     /* 2: vmig_opts.lanes_per_gpu, vmig_stats.lanes_used/.pruned, VMIG_F_PRUNE, table format 02 */

/* ---- error codes ------------------------------------------------------------------------ */
#define VMIG_OK          0
#define VMIG_EINVAL     (-1)   /* bad argument (NULL path, unaligned device offset, ...)        */
#define VMIG_ENOGPU     (-2)   /* no CUDA driver / no sm_100 device in the mask: no CPU fallback */
#define VMIG_ECUDA      (-3)   /* a CUDA runtime call or kernel failed                          */
#define VMIG_EIO        (-4)   /* open/read/write/metadata syscall failed, or short read/write   */
#define VMIG_ENOMEM     (-5)   /* host or device allocation failed                              */
#define VMIG_ETABLE     (-6)   /* malformed / incompatible block-table file                     */
#define VMIG_EFAULT     (-7)   /* injected fault (VMIG_FAIL_BLOCK test hook)                    */
#define VMIG_ENOTDIR    (-8)   /* src or dst is not a directory (reference utils/file.go:50-59)  */
#define VMIG_ESRCCHANGED (-9)  /* a source file shrank while it was being read                  */
#define VMIG_EVERIFY    (-10)  /* VMIG_F_VERIFY: a destination block does not hash like its source */

/* ---- lifecycle --------------------------------------------------------------------------- */
/* Idempotent, thread-safe.  gpu_mask bit i selects CUDA device i; 0 = all visible devices.
 * Creates the per-GPU contexts lazily (streams, pinned staging rings, HBM slots).  Hook:
 * reference cmd/gpu-docker-api/main.go:53-97 (Init); optional -- every call inits on demand. */
int  vmig_init(uint32_t gpu_mask);
/* Frees every pooled resource.  Hook: reference cmd/gpu-docker-api/main.go:139-154 (Stop). */
void vmig_shutdown(void);
int  vmig_device_count(void);                 /* usable sm_100 devices, or VMIG_ENOGPU          */
const char* vmig_strerror(int code);
const char* vmig_last_error(void);            /* thread-local detail of the last failure         */
const char* vmig_version(void);

/* ---- options / statistics ------------------------------------------------------------------ */
#define VMIG_F_MOVE_SRC          0x01u  /* unlink source entries after the copy succeeded and the destination
                                           was flushed (syncfs): the `mv` of moveVolumeData (reference
                                           utils/copy.go:116).  Combine with VMIG_F_VERIFY (vmig_move_dir
                                           does) to also re-hash the destination before unlinking           */
#define VMIG_F_SKIP_HIDDEN_TOPDIRS 0x02u /* reproduce `mv /root/src/ *`: top-level hidden DIRECTORIES
                                           are left behind (reference utils/copy.go:116)           */
#define VMIG_F_MTIME_NS          0x04u  /* keep nanosecond mtimes (mv does; GNU tar's default archive
                                           format keeps whole seconds only -> default off)         */
#define VMIG_F_NO_METADATA       0x08u  /* data only: no chown/chmod/utimens                       */
#define VMIG_F_HASH_ONLY         0x10u  /* build the block table of src; dst is not touched        */
#define VMIG_F_VERIFY            0x20u  /* after the copy, re-read the DESTINATION through the GPU and
                                           require its block hashes to equal the source's; with
                                           VMIG_F_MOVE_SRC the source is only unlinked if they do    */

#define VMIG_F_PRUNE             0x40u  /* after the copy, remove every destination entry the source does not
                                           have (files, symlinks, specials, whole directories).  tar never does
                                           (default off); the final, paused pass of a hand-off needs it: a file
                                           the tenant deleted or renamed since the live pass must not reappear
                                           in the new container.  With VMIG_F_VERIFY the destination's entry set
                                           is then re-walked and must equal the source's                       */

#define VMIG_F_DIRECT_IO         0x80u  /* disk-backed trees (the documented deployment keeps the Docker root on
                                           xfs/LVM: reference docs/volume/volume-size-scale-en.md:5-21): source
                                           files are read with O_DIRECT straight INTO the readers' pinned pieces
                                           and destination files written with O_DIRECT straight OUT of the pinned
                                           OUT ring -- the NVMe DMAs to/from the same page-locked memory the
                                           GPU's copy engines use, and
                                           the page cache (two CPU copies per byte) is bypassed.  Falls back to
                                           buffered I/O per file where the filesystem refuses O_DIRECT.  Env
                                           VMIG_DIRECT_IO=1 sets it for every call.                              */
#define VMIG_F_CUFILE            0x100u /* GPUDirect Storage: source blocks are read with cuFileRead straight into the
                                           HBM slot (no pinned pieces, no H2D copy) and surviving blocks written with
                                           cuFileWrite straight out of it (no D2H copy, no OUT ring).  libcufile is
                                           dlopen()ed: VMIG_EINVAL if it cannot be loaded or its driver cannot be
                                           opened, VMIG_EIO with libcufile's own reason if it refuses a descriptor
                                           (inside containers it needs a udev-visible block device: DESIGN.md §10).
                                           Without the nvidia-fs kernel module libcufile runs in its compatibility
                                           mode (POSIX I/O + bounce buffers).  Env VMIG_CUFILE=1.                 */

typedef struct vmig_opts {
    uint32_t gpu_mask;         /* 0 = every initialised GPU; blocks are sharded across the set   */
    uint32_t block_bytes;      /* 0 -> 4 MiB (4194304); must be a multiple of 4096               */
    uint32_t streams_per_gpu;  /* side streams = staging slots in flight per GPU; 0 -> all (16)   */
    uint32_t flags;            /* VMIG_F_*                                                       */
    uint32_t io_threads;       /* 0 -> default: host reader+writer threads per GPU               */
    uint32_t lanes_per_gpu;    /* 0/1 -> one lane (staging-ring set + thread pipeline) per GPU of the
                                  mask; k -> k lanes per GPU, the block list is sharded over
                                  n_gpus*k lanes exactly as it is over n_gpus*k GPUs (more host
                                  copy parallelism per link; also how the multi-GPU split is
                                  exercised on a 1-GPU box).  Env VMIG_LANES_PER_GPU overrides 0. */
    uint32_t reserved[2];
} vmig_opts;

typedef struct vmig_stats {
    uint64_t bytes_total;      /* N: sum of regular-file sizes migrated                          */
    uint64_t bytes_h2d;        /* bytes DMA'd host->HBM                                          */
    uint64_t bytes_d2h;        /* bytes DMA'd HBM->host (surviving blocks)                       */
    uint64_t bytes_written;    /* bytes written to destination files                             */
    uint64_t blocks_total;
    uint64_t blocks_skipped;   /* unchanged vs prior table: no D2H, no write                     */
    uint64_t files, dirs, symlinks, hardlinks, specials;
    uint64_t kernel_launches;  /* xxh64_blocks + diff_select launches                            */
    uint64_t ns_total, ns_walk, ns_plan, ns_data, ns_meta, ns_table;
    double   ms_kernel;        /* sum of CUDA-event time of the hash kernels                     */
    uint32_t gpus_used;
    uint32_t lanes_used;       /* lanes the block list was sharded over (gpus_used * lanes_per_gpu) */
    uint64_t pruned;           /* VMIG_F_PRUNE: destination entries removed                      */
    uint64_t files_untrusted;  /* prior table given, but the destination file is no longer the one it was
                                  written for (inode/ctime/size): copied in full, not patched    */
    uint64_t files_direct;     /* VMIG_F_DIRECT_IO / VMIG_F_CUFILE: descriptors (source + destination) the
                                  filesystem really let us open with O_DIRECT                    */
} vmig_stats;

/* ---- the hot path -------------------------------------------------------------------------- */
/* Migrate directory tree src_dir/. into the existing directory dst_dir (semantics of
 * `(cd src; tar c .) | (cd dst; tar x)` run as root: reference utils/copy.go:17-27 -- file
 * bytes, mode, uid, gid, mtime, symlinks, hard links, device nodes and FIFOs are reproduced;
 * xattrs are not; existing destination entries are overwritten, extras are never pruned).
 *   prior_table : nullable path of the block table describing what dst ALREADY holds (the prior
 *                 version).  Blocks whose XXH64 equals the prior entry are neither copied back
 *                 from HBM nor written (diff-skip) -- per file, and only while the destination file
 *                 still is the one the table was written for (see "Block-table file").
 *   out_table   : nullable path; receives the block table of src (tmp + rename, after all data
 *                 writes completed).
 * Blocking; re-entrant; returns 0 or -VMIG_E*.  On error the destination may be partially
 * written (the reference does no cleanup either: SURVEY.md §8b) but the call never reports
 * success after a short read/write or a CUDA error. */
int vmig_migrate_tree(const char* src_dir, const char* dst_dir,
                      const char* prior_table, const char* out_table,
                      const vmig_opts* opts /*nullable*/, vmig_stats* stats /*nullable*/);

/* utils.CopyDir(src, dest) (reference utils/copy.go:21-27) == vmig_migrate_tree with defaults. */
int vmig_copy_dir(const char* src_dir, const char* dst_dir);

/* moveVolumeData(src, dest) on resolved host paths (reference utils/copy.go:74-128): copy, re-read the
 * destination through the GPU and require it to hash like the source (VMIG_F_VERIFY), syncfs the destination,
 * and only then unlink the source entries; nanosecond mtimes; synchronous, exit status checked.
 * Divergence from `mv`: sockets are skipped and stay in the source (tar skips them too; a listening socket's
 * inode means nothing in another volume). */
int vmig_move_dir(const char* src_dir, const char* dst_dir);

/* Host buffer -> host buffer through the same pipeline (H2D, hash, diff, D2H of survivors).
 * n_blocks = ceil(nbytes / block_bytes).  prior_hashes/prior_valid nullable (all blocks survive);
 * out_hashes nullable.  dst regions of skipped blocks are left untouched.  Buffers allocated by
 * vmig_host_alloc (or cudaHostRegister'ed by the caller) are DMA'd directly. */
int vmig_migrate_buffer(const void* src, void* dst, uint64_t nbytes,
                        const uint64_t* prior_hashes, const uint8_t* prior_valid,
                        uint64_t* out_hashes, const vmig_opts* opts, vmig_stats* stats);
int  vmig_host_alloc(void** p, uint64_t nbytes);   /* pinned host memory                        */
void vmig_host_free(void* p);

/* K1 direct: canonical XXH64(seed 0) of n blocks (host_buf + offs[i], lens[i]); the blocks are
 * staged to HBM at 16-byte-aligned offsets and hashed by the xxh64_blocks kernel.  kernel_ms
 * (nullable) receives the CUDA-event time of the kernel alone. */
int vmig_hash_blocks(int gpu, const void* host_buf, const uint64_t* offs, const uint32_t* lens,
                     uint64_t n, uint64_t* out_hashes, double* kernel_ms);

/* ---- HBM-resident batch (the "block-hash GB/s" metric: inputs already in HBM) --------------- */
typedef struct vmig_resident vmig_resident;
/* n_blocks slots of block_bytes each in one device allocation (+ hash/prior/survivor arrays). */
int  vmig_resident_open(int gpu, uint64_t n_blocks, uint32_t block_bytes, vmig_resident** out);
void vmig_resident_close(vmig_resident* r);
/* Device-side generator: 8-byte word w of block b = SplitMix64 stream `seed` at word index
 * b*(block_bytes/8)+w (the generator of BASELINE.md §3; restated in oracle/).  All lens reset
 * to block_bytes. */
int  vmig_resident_fill(vmig_resident* r, uint64_t seed);
int  vmig_resident_set_len(vmig_resident* r, uint64_t block, uint32_t len);
int  vmig_resident_upload(vmig_resident* r, uint64_t block, const void* host, uint32_t len);
int  vmig_resident_download(vmig_resident* r, uint64_t block, void* host, uint32_t len);
/* XOR the first 8 bytes of each listed block with ~0 (BASELINE.md §3 config 4's mutation). */
int  vmig_resident_flip(vmig_resident* r, const uint64_t* blocks, uint64_t n);
/* prior table for diff_select: hashes (nullable = none valid) + per-block validity bytes. */
int  vmig_resident_set_prior(vmig_resident* r, const uint64_t* hashes, const uint8_t* valid);
/* One pass = xxh64_blocks over all blocks + diff_select (ordered compaction of changed block
 * indices).  Repeats `iters` times back to back; ms_hash / ms_total are CUDA-event times of the
 * LAST iteration's hash kernel / of all iterations together (on the launching stream). */
int  vmig_resident_pass(vmig_resident* r, uint32_t iters, double* ms_hash_last, double* ms_total);
int  vmig_resident_results(vmig_resident* r, uint64_t* hashes /*n_blocks, nullable*/,
                           uint32_t* survivors /*n_blocks cap, nullable*/, uint64_t* n_survivors);

/* ---- host<->HBM link probe (the e2e roofline denominator; BASELINE.md §4) ----------------------------------
 * Pinned-memory cudaMemcpyAsync sweep on GPU `gpu`: `bytes` per direction in 32 MiB pieces out of a NUMA-local
 * page-locked buffer, timed with CUDA events.  gbs[0] = H2D alone, gbs[1] = D2H alone, gbs[2] / gbs[3] = H2D / D2H
 * while both directions run at once (two streams) -- the state the copy-back path of a migration is in.
 * GB/s = 1e9 bytes per second. */
int vmig_link_probe(int gpu, uint64_t bytes, double gbs[4]);

/* What the engine would use on THIS box right now: host reader / writer threads PER LANE for a call of `lanes` lanes on
 * `n_gpus` GPUs (plain copy; has_prior = 1: diff path; flags & VMIG_F_HASH_ONLY: hash-only), given the per-box budget
 * (20 copy threads for one GPU, 13 per GPU beyond, capped by the CPUs), the lanes other calls of this process have in
 * flight, and VMIG_READERS / VMIG_WRITERS / VMIG_IO_SHARE.  No GPU needed; for operators and tests. */
int vmig_thread_plan(uint32_t lanes, uint32_t n_gpus, uint32_t flags, int has_prior, uint32_t* readers, uint32_t* writers);

/* ---- block table + host-side helpers (no GPU needed) ---------------------------------------- */
/* Block-table file, little-endian:
 *   char[8] "VMIGBT02"; u32 block_bytes; u32 algo (1 = XXH64 seed 0); u64 n_files; u64 n_blocks;
 *   n_files x { u32 path_len; char path[path_len] (relative, no leading ./); u64 size;
 *               u64 first_block; u64 ino; i64 ctime_ns } sorted bytewise by path;
 *   u64 hashes[n_blocks].
 * A file of `size` bytes owns ceil(size/block_bytes) consecutive hashes (0 for an empty file).
 * ino/ctime_ns identify the on-disk file the table speaks FOR: the destination file as the migration that wrote
 * the table left it (the source file for a VMIG_F_HASH_ONLY table); 0/0 = unknown.  A later call that is handed
 * the table as prior_table patches a destination file in place -- skipping blocks whose hash matches -- only
 * while the file's inode, ctime and size still equal the record; otherwise (failed or partial earlier pass,
 * out-of-band write, a table that belongs to another directory) that file is copied in full.  Format "VMIGBT01"
 * (no ino/ctime_ns fields) is still read; its files are never patched in place.
 * Home in the reference: merges/<rs>/<rs>-<version>/ (internal/services/replicaset.go:681-704,
 * internal/version/merge.go:16). */
typedef struct vmig_table_info {
    uint32_t block_bytes, algo;
    uint64_t n_files, n_blocks, bytes_total;
} vmig_table_info;
int vmig_table_info_read(const char* path, vmig_table_info* out);
/* Copies up to cap hashes of the table into out; returns VMIG_OK. */
int vmig_table_hashes(const char* path, uint64_t* out, uint64_t cap);
/* Walk src_dir exactly as vmig_migrate_tree would (same ordering, block layout, hard-link grouping,
 * VMIG_F_SKIP_HIDDEN_TOPDIRS) and return the totals in *stats (bytes_total, blocks_total, files, dirs,
 * symlinks, hardlinks, specials); if out_table is non-NULL also write the manifest as a block table
 * whose hashes are all zero.  No GPU involved: this is the single metadata pass that can replace the
 * separate DirSize walk of PatchVolumeSize's shrink check (reference internal/services/volume.go:126-140,
 * SURVEY.md §8f N3). */
int vmig_manifest(const char* src_dir, uint32_t flags, uint32_t block_bytes,
                  const char* out_table /*nullable*/, vmig_stats* stats /*nullable*/);
/* utils.DirSize (reference utils/file.go:13-22): sum of non-directory sizes under dir. */
int vmig_dir_size(const char* dir, int64_t* bytes, uint64_t* n_files);
/* utils.ToBytes (reference utils/file.go:24-48): "20GB" -> 21474836480; 1024-based; KB/MB/GB/TB. */
int vmig_to_bytes(const char* s, int64_t* out);
/* Deterministic synthetic tree (BASELINE.md §3): n_files files of file_bytes each named
 * f%05d.bin under dir, bytes = SplitMix64 stream seeded seed ^ fnv1a64(relative path). */
int vmig_datagen_files(const char* dir, uint64_t seed, uint32_t n_files, uint64_t file_bytes,
                       uint32_t threads);

#ifdef __cplusplus
}
#endif
#endif /* VMIG_H */
