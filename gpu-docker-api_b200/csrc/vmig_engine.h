// vmig_engine.h -- per-GPU streaming pipeline of libvmig (internal interface).
//
//   source blocks --(reader threads: pread / memcpy, 1 MiB at a time)--> the reader's own pinned pieces
//       --cudaMemcpyAsync H2D per piece (the reader's stream)--> HBM slot
//       --xxh64_blocks kernel (+ compare with prior table)--> hashes, changed flags
//       --cudaMemcpyAsync D2H of the surviving blocks--> pinned OUT slot
//       --(writer threads: pwrite / memcpy)--> destination
//
// One Pipe owns VMIG_SLOTS slots (HBM buffer + pinned OUT buffer) and the readers' pieces on one GPU; a lane (one GPU's
// share of one call) checks a Pipe out of the process-wide pool, runs its block list through it and returns it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include <memory>
#include <mutex>
#include <string>
#include <vector>
#include "vmig_common.h"

namespace vmig {

// Return VMIG_ENOMEM / VMIG_ECUDA from the enclosing function when a CUDA runtime call fails.  The runtime's last error
// is cleared, so a later launch check on this thread (cudaGetLastError) does not report it a second time.
#define CU_API(call)                                                                                  \
    do {                                                                                              \
        cudaError_t e__ = (call);                                                                     \
        if (e__ != cudaSuccess) {                                                                     \
            cudaGetLastError();                                                                       \
            return fail(e__ == cudaErrorMemoryAllocation ? VMIG_ENOMEM : VMIG_ECUDA, "%s: %s", #call, \
                        cudaGetErrorString(e__));                                                     \
        }                                                                                             \
    } while (0)

struct BlockRef {
    uint32_t file;         // backend-defined (index of the file in the manifest; 0 for buffers)
    uint32_t len;          // bytes in this block (<= block_bytes; 0 allowed)
    uint64_t file_off;     // byte offset inside the file / buffer
    uint64_t table_idx;    // where this block's hash goes in the call-wide hash array
    uint64_t prior_hash;   // prior version's hash of the same block ...
    uint8_t  prior_valid;  // ... if 1
};

// Where block bytes come from and go to.  Implementations must be thread-safe.
class BlockIO {
public:
    virtual ~BlockIO() {}
    // bytes [off, off + len) of block b into dst; off and len come from block_piece() (vmig_common.h), and dst has room
    // for the piece's io_len
    virtual int  read_block(const BlockRef& b, size_t off, size_t len, uint8_t* dst) = 0;
    virtual int  write_block(const BlockRef& b, const uint8_t* src) = 0;
    // called exactly once per block when it needs nothing more (written == false: skipped)
    virtual int  block_done(const BlockRef&, bool /*written*/) { return VMIG_OK; }
    // writes with the same key are issued by one writer thread, in order (a file takes writes from one
    // thread at a time anyway); backends without such a constraint spread the keys
    virtual uint32_t write_key(const BlockRef& b) { return b.file; }
    // staging layout: every block starts at a multiple of this inside a slot (>= 512, a power of two).  O_DIRECT
    // file I/O needs logical-sector alignment of buffer, offset and length: 4096.
    virtual uint32_t slot_align() { return 512; }
    // GPUDirect-Storage style backends move bytes between the file and the HBM slot themselves (no pinned ring, no
    // cudaMemcpyAsync): read_block_dev fills d_base + d_off, write_block_dev drains it.  Called on reader / writer threads.
    virtual bool device_reads()  { return false; }
    virtual bool device_writes() { return false; }
    virtual int  read_block_dev(const BlockRef&, uint8_t* /*d_base*/, size_t /*d_off*/) { return VMIG_EINVAL; }
    virtual int  write_block_dev(const BlockRef&, const uint8_t* /*d_base*/, size_t /*d_off*/) { return VMIG_EINVAL; }
    // non-null: page-locked memory the DMA engines can use directly (no staging copy)
    virtual const uint8_t* pinned_src(const BlockRef&) { return nullptr; }
    virtual uint8_t*       pinned_dst(const BlockRef&) { return nullptr; }
};

struct LaneStats {
    uint64_t bytes_h2d = 0, bytes_d2h = 0, bytes_written = 0, blocks_skipped = 0, kernel_launches = 0;
    double   ms_kernel = 0;
};

struct DeviceInfo {
    int dev = -1;
    int sm_count = 0;
    std::vector<int> cpus;     // NUMA-local CPUs of the GPU (empty: no affinity)
};

class Pipe;   // defined in vmig_engine.cu

// ---- process-wide context -------------------------------------------------------------------
int  ctx_init(uint32_t gpu_mask);
void ctx_shutdown();
int  ctx_device_count();
// devices selected by `mask` (0 = all initialised); error if none
int  ctx_select(uint32_t mask, std::vector<DeviceInfo>* out);
int  ctx_acquire_pipe(const DeviceInfo& d, Pipe** out);
// one Pipe per lane, all reserved atomically (a device may repeat: lanes_per_gpu)
int  ctx_acquire_pipes(const std::vector<DeviceInfo>& lane_devs, std::vector<Pipe*>* out);
void ctx_release_pipe(Pipe* p);
uint32_t pipe_slot_bytes();
int  io_threads_default(uint32_t* readers, uint32_t* writers, uint32_t requested, size_t lanes, size_t n_gpus, bool many_files,
                        bool has_prior, bool hash_only);

// Run blocks[] through one GPU.  hashes_out[b.table_idx] receives every block's hash.
//   hash_only : no D2H of data, no writes (block_done(b,false) is still called).
//   err       : call-wide first-error latch shared by all lanes (0 = fine).
int run_lane(Pipe* pipe, const std::vector<BlockRef>& blocks, BlockIO* io, bool has_prior, bool hash_only,
             uint32_t readers, uint32_t writers, uint32_t max_slots, uint64_t* hashes_out, LaneStats* stats,
             std::atomic<int>* err, std::string* err_msg, std::mutex* err_mu);

}  // namespace vmig
