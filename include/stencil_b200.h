/* stencil_b200.h -- C ABI of the B200-native halo-exchange / jacobi hot path.
 *
 * This is the drop-in boundary below the C++ API (include/stencil/*.hpp): plain pointers and
 * sizes, no C++ or torch types.  Each entry point names the interface of cwpearson/stencil it
 * replaces (paths relative to the reference checkout).  Device pointers are raw CUDA device
 * addresses (cudaMalloc, cudaIpcOpenMemHandle or peer-mapped); `stream` is a cudaStream_t passed
 * as void*.  All functions return 0 on success or a negative sb_status; sb_last_error() gives the
 * message.  Nothing here falls back to the CPU: without a CUDA device every launch fails loudly.
 *
 * Memory layout (reference src/local_domain.cu:187-203): quantity allocation = x fastest,
 * element (x,y,z) at byte offset (z*ysize + y)*pitch + x*elem_size, where (pitch, ysize) are the
 * cudaPitchedPtr fields the reference carries (pitch == xsize == row bytes, unpitched).
 */
#ifndef STENCIL_B200_H
#define STENCIL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB_VERSION 1

typedef enum sb_status {
  SB_OK = 0,
  SB_ERR_INVALID = -1, /* bad argument */
  SB_ERR_CUDA = -2,    /* a CUDA runtime call failed */
  SB_ERR_NOGPU = -3,   /* no usable CUDA device */
  SB_ERR_ALLOC = -4
} sb_status;

/* Thread-local message for the last failing call on this thread. */
const char *sb_last_error(void);
int sb_version(void);
/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
uint64_t sb_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Geometry.  radius27 is the reference's DirectionMap<size_t> storage order:
 * radius27[(dz+1)*9 + (dy+1)*3 + (dx+1)]  (include/stencil/direction_map.hpp:15,44-50).
 * ------------------------------------------------------------------------------------------- */

/* LocalDomain::halo_pos, src/local_domain.cu:86-125 */
int sb_halo_pos(const int64_t dir[3], const int64_t size[3], const int64_t radius27[27], int halo, int64_t out[3]);
/* LocalDomain::halo_extent, include/stencil/local_domain.cuh:212-222 */
int sb_halo_extent(const int64_t dir[3], const int64_t size[3], const int64_t radius27[27], int64_t out[3]);
/* LocalDomain::raw_size, local_domain.cuh:236-239 */
int sb_raw_size(const int64_t size[3], const int64_t radius27[27], int64_t out[3]);
/* prime_factors (descending), src/numeric.cpp:6-26.  Returns the count (<= cap) or <0. */
int sb_prime_factors(int64_t n, int64_t *out, int cap);
/* RankPartition, include/stencil/partition.hpp:20-116: dim, base subdomain size, remainder */
int sb_rank_partition(const int64_t size[3], int64_t n, int64_t dim[3], int64_t base[3], int64_t rem[3]);
/* NodePartition, partition.hpp:120-256 */
int sb_node_partition(const int64_t size[3], const int64_t radius27[27], int64_t nodes, int64_t gpus, int64_t sys_dim[3],
                      int64_t node_dim[3], int64_t base[3], int64_t rem[3]);
/* subdomain_size / subdomain_origin of either partition, partition.hpp:55-86 */
int sb_subdomain_size(const int64_t base[3], const int64_t rem[3], const int64_t idx[3], int64_t out[3]);
int sb_subdomain_origin(const int64_t base[3], const int64_t rem[3], const int64_t idx[3], int64_t out[3]);
/* DistributedDomain::get_interior / get_exterior for one subdomain, src/stencil.cu:878-977.
 * lo/hi = compute region of the subdomain (global coords).  Exterior: up to 6 boxes in the order
 * +x,+y,+z,-x,-y,-z; returns the number written to ext_lo/ext_hi (each 6*3 int64). */
int sb_interior(const int64_t lo[3], const int64_t hi[3], const int64_t radius27[27], int64_t int_lo[3], int64_t int_hi[3]);
int sb_exterior(const int64_t lo[3], const int64_t hi[3], const int64_t radius27[27], int64_t *ext_lo, int64_t *ext_hi);

/* ---------------------------------------------------------------------------------------------
 * Box copies: the one engine behind pack, unpack, translate and the fused direct halo write.
 * ------------------------------------------------------------------------------------------- */

/* A 3-D strided allocation, the cudaPitchedPtr the reference passes around. */
typedef struct sb_pitched {
  void *ptr;
  int64_t pitch; /* bytes between rows */
  int64_t ysize; /* rows per z-plane */
} sb_pitched;

/* One strided->strided copy of `extent` elements (x,y,z) from src@src_pos to dst@dst_pos.
 * Replaces translate() (src/copy.cu:34-77); with a dense dst it is pack_kernel
 * (src/pack_kernel.cu:3-59), with a dense src unpack_kernel (:61-108). */
typedef struct sb_box_copy {
  sb_pitched dst;
  int64_t dst_pos[3];
  sb_pitched src;
  int64_t src_pos[3];
  int64_t extent[3];
  int64_t elem_size;
} sb_box_copy;

/* pack_kernel / unpack_kernel / translate one-shots (tests launch these directly in the reference:
 * test/test_cuda_pack.cu:76, test/test_cuda_translate_kernel.cu). */
int sb_pack(void *dst, sb_pitched src, const int64_t pos[3], const int64_t extent[3], int64_t elem_size, void *stream);
int sb_unpack(sb_pitched dst, const void *src, const int64_t pos[3], const int64_t extent[3], int64_t elem_size,
              void *stream);
int sb_translate(sb_pitched dst, const int64_t dst_pos[3], sb_pitched src, const int64_t src_pos[3],
                 const int64_t extent[3], int64_t elem_size, void *stream);

/* A persistent plan: any number of box copies executed by ONE kernel launch on `device`.
 * This is what replaces, per source GPU, the reference's per-message launches of
 * dev_packer_pack_domain (src/packer.cu:10-26, 109-148), multi_translate (src/copy.cu:79-85,
 * tx_cuda.cuh:74-104), cudaMemcpyPeerAsync (tx_cuda.cuh:162) and dev_unpacker_unpack_domain
 * (src/packer.cu:28-44): destination pointers may be local, or a peer GPU's ghost cells
 * (peer-access or CUDA-IPC mapped), in which case the halo is written straight over NVLink. */
typedef struct sb_copy_plan sb_copy_plan;
int sb_copy_plan_create(sb_copy_plan **out, int device, const sb_box_copy *copies, int64_t n);
int sb_copy_plan_launch(sb_copy_plan *plan, void *stream);
int64_t sb_copy_plan_bytes(const sb_copy_plan *plan);     /* payload bytes per launch */
int64_t sb_copy_plan_num_tiles(const sb_copy_plan *plan); /* work items per launch */
/* how many of the plan's copies are carried by the TMA (cp.async.bulk.tensor) path: wide rows whose source
 * and destination are 16-byte aligned in base and strides; the rest use the LDG/STG path.  SB_TMA=0 disables. */
int64_t sb_copy_plan_num_tma_segments(const sb_copy_plan *plan);
int sb_copy_plan_destroy(sb_copy_plan *plan);

/* Cross-GPU completion flags for the fused exchange when source and destination GPUs are driven
 * by different processes (the reference's IPC event + 0-byte MPI notify, tx_cuda.cuh:225-315,
 * src/tx_ipc.cpp).  flags are uint32 slots in device memory that peers map via CUDA IPC.
 *  - sb_signal: after all prior work on `stream`, store `value` (release, system scope) to each
 *    of the n remote slots.
 *  - sb_wait:   make `stream` wait until each of n local slots is >= value (acquire). */
int sb_signal(uint32_t *const *remote_slots, int n, uint32_t value, int device, void *stream);
int sb_wait(const uint32_t *local_slots, int n, uint32_t value, int device, void *stream);

/* ---------------------------------------------------------------------------------------------
 * 7-point jacobi step (the reference's user kernel, bin/jacobi3d.cu:40-85) over a region.
 * dtype_size 4 = float, 8 = double.  acc_origin = global coordinate of allocation element (0,0,0)
 * (Accessor origin, include/stencil/local_domain.cuh:153-173).  [lo,hi) = region to update,
 * [clo,chi) = the whole distributed compute region (hot/cold sphere placement).
 * dst[p] = 1 in the hot sphere, 0 in the cold sphere, else ((((((0+px)+mx)+py)+my)+pz)+mz)/6 with
 * IEEE round-to-nearest division (bit-identical to the CPU oracle).
 * ------------------------------------------------------------------------------------------- */
int sb_jacobi3d(sb_pitched dst, sb_pitched src, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3],
                const int64_t hi[3], const int64_t clo[3], const int64_t chi[3], void *stream);
/* The same update over n <= 8 regions in ONE launch: the exterior slabs of a subdomain
 * (bin/jacobi3d.cu:324-342 launches stencil_kernel once per slab).  lo/hi are n*3 int64. */
int sb_jacobi3d_regions(sb_pitched dst, sb_pitched src, int dtype_size, const int64_t acc_origin[3], int n,
                        const int64_t *lo, const int64_t *hi, const int64_t clo[3], const int64_t chi[3], void *stream);
/* ---------------------------------------------------------------------------------------------
 * Astaroth MHD substep: replaces `integrate_substep` + `solve<step>` of the reference's astaroth extract
 * (astaroth/kernels.cu:62-87, astaroth/user_kernels.h:437-469, astaroth/integration.cuh:14-52).
 * in / out: the VertexBufferArray (astaroth/kernels.h:22-27): 8 device arrays each, order lnrho, uux, uuy, uuz,
 * ax, ay, az, entropy (astaroth/user_defines.h:112-120), all of raw size raw[3] = (mx, my, mz) elements, x fastest,
 * including the radius-3 ghost cells.  [lo, hi): box to update in the reference's memory-offset coordinates
 * (what the driver passes as Rect3 cr, astaroth/astaroth.cu:563-566); every cell needs 3 allocated cells around it.
 * step 0..2 = Williamson RK3 substep; step 0 ignores the previous contents of `out`.
 * params: the uniforms solve<> reads through DCONST (acDeviceLoadMeshInfo / acDeviceLoadScalarUniform,
 * astaroth/kernels.cu:89-163).  variant: 0 auto, 1 cell kernel, 2 tile kernel (one thread per cell), 3 team kernel (two specialised
 * threads per cell on the same shared-memory ring; FP64: ring fed by TMA when the buffers allow it), 4 / 5 the TMA-fed
 * two- / three-team kernel or an error.
 * dtype_size 8 = double (the reference's AcReal), 4 = float.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  double inv_dsx, inv_dsy, inv_dsz;
  double dt;
  double cs2_sound, gamma, cp_sound, lnrho0, lnT0;
  double mu0, nu_visc, zeta, eta;
} sb_astaroth_params;
int sb_astaroth_substep(int step, const void *const in[8], void *const out[8], int dtype_size, const int64_t raw[3],
                        const int64_t lo[3], const int64_t hi[3], const sb_astaroth_params *params, int variant, void *stream);
/* The jacobi step over the WHOLE compute region of a subdomain with the halo exchange of the NEXT iteration fused
 * into it: every cell on a face of [lo, hi) is also stored into the ghost cell of the face neighbour that reads it
 * next iteration.  Replaces, per iteration, the interior stencil_kernel launch + DistributedDomain::exchange()
 * (src/stencil.cu:1002-1186: pack -> copy -> unpack of 6 face messages) + the <= 6 exterior launches of
 * bin/jacobi3d.cu:296-368 by one kernel; results are bit-identical.  Face radius 1 only (bin/jacobi3d.cu:237-246).
 * nbr[d], d = -x,+x,-y,+y,-z,+z: the neighbour's OUTPUT allocation of this iteration (its `next` buffer; may be this
 * subdomain's own dst for a periodic self-neighbour, or a peer GPU's memory mapped by peer access / CUDA IPC);
 * nbr_zsize[d]: planes of that allocation.  ptr == NULL: nothing is pushed in that direction.  The neighbour must
 * have the same extent as this subdomain on the two axes orthogonal to d (always true for a grid partition).
 * The caller orders iterations: this launch may start once every neighbour has finished the previous iteration. */
typedef struct {
  sb_pitched nbr[6];
  int64_t nbr_zsize[6];
  /* Dense x faces (x neighbour owned by another rank): if x_dense[s] != 0 (s = 0: -x side, 1: +x side), nbr[s].ptr is
   * not a field allocation but a dense array in the NEIGHBOUR's memory, (rows x planes) elements indexed [y][z] (z
   * fastest, like the march) in THIS subdomain's allocation coordinates; nbr[s].ysize = rows, nbr_zsize[s] = planes.
   * The kernel stages the column in shared memory and writes 256-byte lines instead of one 8-byte store per row and
   * plane.  x_recv[s], if not NULL, is such an array (this subdomain's rows x planes) received FROM the neighbour on
   * side s: the out-of-subdomain x neighbour of the first / last column is read from it instead of from the ghost
   * column of src.  Needs a 16-byte aligned first compute cell and whole warp strips along x. */
  int64_t x_dense[2];
  const void *x_recv[2];
} sb_halo_push;
int sb_jacobi3d_fused(sb_pitched dst, sb_pitched src, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3],
                      const int64_t hi[3], const int64_t clo[3], const int64_t chi[3], const sb_halo_push *push, void *stream);
/* The same launch with the ordering BETWEEN RANKS inside the kernel, replacing the reference's per-iteration host
 * synchronisation (DistributedDomain::exchange() returns after MPI_Waitall / stream syncs, src/stencil.cu:1120-1186;
 * bin/jacobi3d.cu:337-365) and this library's own sb_wait / sb_signal launches.
 * Every boundary tile of the kernel (256 threads: one 32-lane strip x 8 rows x one z chunk of 32 planes) parks its face
 * cells in shared memory while it marches and stores them into the neighbour when it is done; there is no fence and no
 * flag per tile.  Instead the FIRST CTA of the launch writes signal_value (release, system scope) into signal_rows[f][0]
 * for every face f with a row -- a uint32 word in the NEIGHBOUR's memory (peer / IPC mapped): its mailbox for the face it
 * shares with this subdomain.  The kernel boundary has completed every store of the previous launch on this stream, so
 * the word says "my previous iteration is complete, pushes and reads".  Before marching, a CTA on face f polls
 * wait_rows[f][0] (this GPU's own mailbox for face f, written by the neighbour across f; ld.acquire.sys) until
 * (int32)(word - wait_value) >= 0.  Protocol: the launch of iteration e carries wait_value = signal_value = e -- a
 * neighbour that has STARTED iteration e has (a) filled the ghost cells iteration e reads here and (b) stopped reading
 * the ghost cells iteration e overwrites there.  Tiles that touch no face never wait.  (Round-2 measurements, 8 ranks:
 * one release per boundary tile cost 19 us per iteration -- the releasing warp lingers for an NVLink round trip and
 * keeps its CTA slot -- against a skew of a few microseconds between the ranks' kernel starts.)
 * Faces: -x,+x,-y,+y,-z,+z.  NULL rows: no wait / no signal on that face (neighbour in the same process: order the
 * launches with stream events).  sync == NULL: no handshake at all.  The rows keep SB_FUSED_MAX_GROUPS words (the
 * per-tile protocol's size); only word 0 is used. */
#define SB_FUSED_MAX_GROUPS 4096
typedef struct {
  const uint32_t *wait_rows[6];
  uint32_t *signal_rows[6];
  uint32_t wait_value, signal_value;
} sb_step_sync;
int sb_jacobi3d_fused_sync(sb_pitched dst, sb_pitched src, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3],
                           const int64_t hi[3], const int64_t clo[3], const int64_t chi[3], const sb_halo_push *push,
                           const sb_step_sync *sync, void *stream);
/* init_kernel, bin/jacobi3d.cu:18-29: fill region with a constant */
int sb_fill(sb_pitched dst, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3], const int64_t hi[3],
            double value, void *stream);
/* sum over [lo,hi) of (a-b)^2 accumulated in double into *out_dev (device double, zeroed by the
 * call): the FP64 residual BASELINE.json asks for (not in the reference). */
int sb_sqdiff(sb_pitched a, sb_pitched b, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3],
              const int64_t hi[3], double *out_dev, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Field reductions: the filters of the reference's astaroth extract (astaroth/reductions.cuh:18-52) over a box of
 * 1-4 operand allocations with the same pitch and ysize.  Per cell a value f and a square g are evaluated in FP64
 * (FP32 inputs are widened; VALUE, DIFF and VECTOR round every operation, so f is bit-identical to float64 numpy):
 *   VALUE  (a)          f = a                            g = a*a
 *   DIFF   (a, b)       f = a - b                        g = (a - b)^2
 *   VECTOR (a, b, c)    f = sqrt(s), s = (a*a + b*b) + c*c   g = s
 *   EXP    (a)          f = exp(a)                       g = exp(a)*exp(a)
 *   ALFVEN (a, b, c, d) f = sqrt(s) / sqrt(4 pi exp(d))  g = s / (4 pi exp(d))
 * and the launch returns min f, max f, sum f, sum g (FP64 sums).  NaN propagates to all four; an empty box gives
 * +inf, -inf, 0, 0.  RTYPE_MAX / MIN / SUM are max / min / sum; RTYPE_RMS, RMS_EXP and ALFVEN_RMS are sqrt(sum2 / cells).
 * Deterministic: no floating-point atomics; the same box on the same GPU gives the same bits on every call.
 * ------------------------------------------------------------------------------------------- */
typedef enum sb_reduce_kind {
  SB_REDUCE_VALUE = 0,
  SB_REDUCE_DIFF = 1,
  SB_REDUCE_VECTOR = 2,
  SB_REDUCE_EXP = 3,
  SB_REDUCE_ALFVEN = 4
} sb_reduce_kind;
typedef struct {
  double min, max, sum, sum2;
} sb_reduce_result;
/* Bytes of device memory one sb_reduce launch on `device` needs as workspace.  The caller zeroes a workspace once;
 * every launch leaves it ready for the next.  One workspace serves one launch at a time: concurrent reductions (other
 * streams) need their own. */
int64_t sb_reduce_workspace_bytes(int device);
/* One launch on `stream`: reduces [lo, hi) (global coordinates; acc_origin = global coordinate of allocation element
 * (0,0,0), as in sb_sqdiff) of operands[0 .. n) (n = 1, 2, 3, 1, 4 by kind), and stores an sb_reduce_result at the start
 * of `workspace` (device memory) when the launch completes. */
int sb_reduce(int kind, const sb_pitched *operands, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3],
              const int64_t hi[3], void *workspace, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Device memory + peer plumbing used by the host layers (C++ and Python).
 * ------------------------------------------------------------------------------------------- */
int sb_device_count(int *count);
int sb_malloc(void **ptr, size_t bytes, int device);
int sb_free(void *ptr, int device);
int sb_memset(void *ptr, int value, size_t bytes, int device, void *stream);
/* cudaMemcpyAsync(cudaMemcpyDefault) on `stream` of `device`: host<->device and device<->device (UVA).
 * Host buffers should be pinned for the copy to be asynchronous. */
int sb_memcpy(void *dst, const void *src, size_t bytes, int device, void *stream);
int sb_stream_sync(int device, void *stream);
int sb_device_sync(int device);
/* cudaDeviceEnablePeerAccess both ways if possible (gpu_topo::enable_peer, src/gpu_topology.cpp:97-129);
 * *ok = 1 when src can address dst's memory. */
int sb_enable_peer(int src_device, int dst_device, int *ok);
/* CUDA IPC handle export / import (cudaIpcGetMemHandle / OpenMemHandle, tx_cuda.cuh:225-243). handle = 64 bytes. */
int sb_ipc_export(void *ptr, void *handle64);
int sb_ipc_import(const void *handle64, int device, void **ptr);
int sb_ipc_close(void *ptr, int device);

#ifdef __cplusplus
}
#endif
#endif /* STENCIL_B200_H */
