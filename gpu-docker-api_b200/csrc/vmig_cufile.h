// vmig_cufile.h -- GPUDirect Storage (cuFile) ingest, SURVEY.md §8f row N4: source blocks go from the file straight into
// the HBM staging slot (no pinned pieces, no separate H2D copy).  libcufile is dlopen()ed at first use, so libvmig has
// no link-time dependency on it; with the nvidia-fs kernel module the read is a DMA from the NVMe into HBM, without it
// libcufile's compatibility mode (POSIX read + its own bounce buffers) gives the same bytes.
// Deployment the row targets: Docker root on local xfs/LVM (reference docs/volume/volume-size-scale-en.md:5-21).
#pragma once
#include <stdint.h>
#include <stddef.h>
#include <sys/types.h>

namespace vmig {

// 0 on success; VMIG_EINVAL (with a message) when libcufile.so cannot be loaded or its driver cannot be opened.
int  cufile_open();
bool cufile_loaded();
// Register / deregister an open descriptor (O_DIRECT where the filesystem allows it).  *handle is opaque.
int  cufile_handle_open(int fd, void** handle);
void cufile_handle_close(void* handle);
// Optional: pin a device range for direct DMA (a no-op in compatibility mode).  Failure is not an error.
void cufile_buf_register(void* dev_ptr, size_t bytes);
void cufile_buf_deregister(void* dev_ptr);
// Read `bytes` at file offset `off` into dev_base + dev_off.  Returns bytes read (>= 0) or a negative VMIG_E* code.
ssize_t cufile_read(void* handle, void* dev_base, size_t bytes, off_t off, off_t dev_off);
ssize_t cufile_write(void* handle, const void* dev_base, size_t bytes, off_t off, off_t dev_off);
void cufile_shutdown();

}  // namespace vmig
