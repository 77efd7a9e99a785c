/*
 * ddc.h -- C ABI of the B200 domain-decomposition library (libddc_cuda.so).
 *
 * This is the drop-in boundary for the reference's hot path
 *     land-sea mask -> rectilinear RCB -> part boxes / pid labels / neighbours / halos
 * i.e. what ZoltanPartitioner::partition() + Partitioner::discover_neighbours() compute
 * (reference: ZoltanPartitioner.cpp:93-224, Partitioner.cpp:329-435).  Plain C: pointers and
 * sizes only, no STL, no exceptions, no torch types.  The C++ host API in
 * include/domain_decomp/ (Grid, Partitioner, CudaRcbPartitioner) and the Python test/bench
 * harness both sit on top of exactly these entry points.
 *
 * Conventions
 *   - every function returns 0 on success, a negative ddc_status otherwise;
 *     ddc_last_error(h) returns the message (h may be NULL for create-time errors).
 *   - mask layout: mask[y][x], x fastest, int32, ocean <=> value > 0
 *     (Grid.cpp:176-186, Grid.hpp:131-137).
 *   - a part is what the reference calls an MPI rank: part p owns box
 *     {x0,y0,ext_x,ext_y} = {_global_new[0], _global_new[1], _local_ext_new[0], _local_ext_new[1]}
 *     (Partitioner.hpp:166-170).  The number of parts is a parameter here, not the world size.
 *   - edges are numbered as DomainUtils.hpp:15: LEFT=0, RIGHT=1, BOTTOM=2, TOP=3.
 *   - one handle drives one GPU.  With nranks > 1 every rank owns a contiguous block of mask
 *     rows; the per-column and per-strip-row histograms are exchanged through peer memory over
 *     NVLink (ddc_peer_export / ddc_peer_import) or, without that, with NCCL.  All ranks
 *     hold identical boxes / neighbour tables afterwards; pid stays row-sharded.
 *   - a handle is not thread-safe; distinct handles are independent.
 */
#ifndef DDC_H
#define DDC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define DDC_API __attribute__((visibility("default")))
#else
#define DDC_API
#endif

typedef struct ddc_handle_s* ddc_handle_t;

typedef enum {
    DDC_OK = 0,
    DDC_ERR_ARG = -1, /* bad argument / call order */
    DDC_ERR_CUDA = -2, /* CUDA runtime error (message has the detail) */
    DDC_ERR_NCCL = -3, /* NCCL error */
    DDC_ERR_NOMEM = -4,
    DDC_ERR_STATE = -5, /* result requested before ddc_partition() */
    DDC_ERR_PEER = -6 /* a rank did not reach an exchange step in time (peer-memory exchange) */
} ddc_status;

enum { DDC_LEFT = 0, DDC_RIGHT = 1, DDC_BOTTOM = 2, DDC_TOP = 3, DDC_N_EDGE = 4 };
/* corners of a part's ghost frame (ddc_get_corner_neighbours, ddc_halo_exchange_full_f64) */
enum { DDC_BOTTOM_LEFT = 0, DDC_BOTTOM_RIGHT = 1, DDC_TOP_LEFT = 2, DDC_TOP_RIGHT = 3, DDC_N_CORNER = 4 };

/* flags of ddc_partition() */
enum {
    DDC_WANT_PID = 1, /* write the pid map (owner labelling, ZoltanPartitioner.cpp:201-219) */
    DDC_WANT_NEIGHBOURS = 2, /* neighbour / halo tables (Partitioner.cpp:329-435) */
    DDC_PROFILE = 4, /* record per-stage CUDA-event timings into ddc_stats */
    DDC_ASYNC = 8 /* only enqueue the step on the stream; the first result getter (or
                     ddc_synchronize) waits for it.  Without it ddc_partition() returns when the
                     step is complete.  With nranks > 1 all ranks must then call the same first getter. */
};

#define DDC_NCCL_ID_BYTES 128
#define DDC_IPC_HANDLE_BYTES 64
#define DDC_N_STAGES 8

typedef struct {
    int32_t nx, ny, nparts;
    int32_t nlev, n_xlev, n_ylev; /* RCB recursion levels and how many cut x / y */
    int32_t nstrips; /* vertical strips after the x levels */
    int32_t changes; /* Zoltan's `changes`: 0 => naive blocks were reported */
    int64_t n_ocean; /* global number of ocean cells (dots) */
    int64_t load_min, load_max; /* ocean cells of the lightest / heaviest part */
    int64_t edge_cut; /* sum of all interior halo lengths (0 unless neighbours were built) */
    int32_t median_iters; /* total Zoltan_RB_find_median iterations over all cuts */
    int32_t gpu_launches; /* kernels launched by the last ddc_partition() on this rank */
    /* DDC_PROFILE: milliseconds per stage on this rank (0 when not profiled)
       0 mask scan, 1 x cuts, 2 strip rows, 3 y cuts, 4 label, 5 finalize, 6 neighbours, 7 total */
    float stage_ms[DDC_N_STAGES];
    int32_t exchange; /* how the ranks exchanged their histograms: 0 single GPU, 1 NCCL collectives,
                         2 peer memory (loads from the other ranks' buffers inside the kernels) */
} ddc_stats;

/* ---- life cycle ---------------------------------------------------------------------------- */

/* rank 0 obtains a NCCL unique id; the host distributes it (MPI_Bcast / torch.distributed). */
DDC_API int ddc_get_nccl_unique_id(void* out /* DDC_NCCL_ID_BYTES */);

/* replaces Zoltan_Initialize + new Zoltan(comm) (ZoltanPartitioner.cpp:69-86).
   nranks == 1: nccl_id may be NULL and NCCL is never touched. */
DDC_API int ddc_create(ddc_handle_t* h, int device, int rank, int nranks, const void* nccl_id);
DDC_API int ddc_destroy(ddc_handle_t h);
DDC_API const char* ddc_last_error(ddc_handle_t h);

/* Peer-memory exchange (nranks > 1, all GPUs of one NVLink / NVSwitch box, one process per GPU).
   The reference exchanges through MPI inside Zoltan and with four MPI_Allgather calls in
   discover_neighbours (Partitioner.cpp:378-388).  Here the kernels that produce a histogram store it
   straight into the other ranks' exchange buffers, and the kernels that consume it wait for a flag
   and read their own memory: ddc_peer_export() allocates this rank's exchange buffer for masks up
   to nx * ny into nparts parts (one slot per rank and histogram) and returns its CUDA IPC
   handle; the host gathers the handles of all ranks (MPI_Allgather / torch.distributed) and hands
   them, in rank order, to ddc_peer_import().  Without these two calls -- or for a decomposition
   that does not fit the exported capacity -- the exchange steps are NCCL collectives.
   The flags and data words of the exchange carry the number of the decomposition: every rank must have made the
   same number of ddc_partition() calls when the buffers are imported (normally none), and make them together
   afterwards.  (ddc_peer_connect, all handles in one process, aligns the counters itself.) */
DDC_API int ddc_peer_export(ddc_handle_t h, int nx, int ny, int nparts, void* ipc_handle_out /* DDC_IPC_HANDLE_BYTES */);
DDC_API int ddc_peer_import(ddc_handle_t h, const void* all_handles /* nranks * DDC_IPC_HANDLE_BYTES */);
/* unmap the other ranks' buffers (back to NCCL).  Shutdown order: every rank calls ddc_peer_close(),
   the host synchronises the ranks (a barrier), then every rank calls ddc_destroy(), which frees its
   own buffer -- so that no buffer is freed while another rank still has it mapped. */
DDC_API int ddc_peer_close(ddc_handle_t h);
/* The same exchange for handles that live in ONE process (one host thread per GPU instead of one process per
   GPU; this is what `decomp --gpus G` / CudaRcbPartitioner use): handles[q] must be rank q of n, created on
   different devices with nccl_id == NULL.  Allocates every handle's exchange buffer for masks up to nx * ny into
   nparts parts and enables peer access between the devices; no CUDA IPC.  Each handle is then driven by its own
   thread (ddc_partition blocks in the exchange steps until all ranks have enqueued theirs). */
DDC_API int ddc_peer_connect(ddc_handle_t* handles, int n, int nx, int ny, int nparts);

/* Page-locked host memory (cudaHostAlloc / cudaFreeHost) for masks and pid maps: ddc_set_mask_host and
   ddc_get_pid_host move such memory at link speed in asynchronous chunks; pageable memory goes through the
   driver's staging copies.  No counterpart in the reference (its mask never leaves the host). */
DDC_API int ddc_host_alloc(void** ptr, size_t bytes);
DDC_API int ddc_host_free(void* ptr);

/* launch everything on this CUDA stream (a cudaStream_t; NULL = the handle's own stream) */
DDC_API int ddc_set_stream(ddc_handle_t h, void* cuda_stream);

/* ---- input: replaces the Grid -> Zoltan callbacks (ZoltanPartitioner.cpp:19-67) ------------- */

/* rows [y_begin, y_begin + y_count) of the global nx * ny mask; `rows` points at row y_begin.
   host variant: copied to the device (pinned memory makes the copy asynchronous);
   device variant: the pointer is borrowed until the next set_mask / destroy.
   With nranks == 1 pass y_begin = 0, y_count = ny.  With nranks > 1 the shards must be
   ddc_shard_rows() of (ny, nranks, rank). */
DDC_API int ddc_set_mask_host(ddc_handle_t h, const int32_t* rows, int nx, int ny, int y_begin,
    int y_count);
DDC_API int ddc_set_mask_device(ddc_handle_t h, const int32_t* rows, int nx, int ny, int y_begin,
    int y_count);

/* The same with one byte per cell (a bool / uint8 tensor, a netCDF byte or ubyte variable): the same arguments,
   shard rule, ownership and status codes.  A cell is ocean <=> its byte is non-zero, read as unsigned, so 0xFF is
   ocean (the int32 rule makes -1 land): a signed byte mask that stores land as a negative value must be converted
   first.  The scan reads a quarter of the int32 bytes and computes the same decomposition bit for bit.  The handle
   keeps the type of the mask it was last given; switching between decompositions is allowed, and with nranks > 1
   every rank may use either type.  Fastest with nx % 4 == 0 and a 4-byte aligned pointer; other masks are read
   byte by byte, never past a row's nx bytes. */
DDC_API int ddc_set_mask_u8_host(ddc_handle_t h, const uint8_t* rows, int nx, int ny, int y_begin,
    int y_count);
DDC_API int ddc_set_mask_u8_device(ddc_handle_t h, const uint8_t* rows, int nx, int ny, int y_begin,
    int y_count);

/* the row block of `rank`: rows_per_rank = ceil(ny / nranks), last ranks may be short / empty */
DDC_API void ddc_shard_rows(int ny, int nranks, int rank, int* y_begin, int* y_count);

/* ---- the hot path: replaces Zoltan::LB_Partition + RCB_Box + discover_neighbours ------------ */
DDC_API int ddc_partition(ddc_handle_t h, int nparts, int periodic_x, int periodic_y, int flags);

/* wait for the stream (results below synchronise on their own) */
DDC_API int ddc_synchronize(ddc_handle_t h);

/* ---- results -------------------------------------------------------------------------------- */

/* replaces Partitioner::get_bounding_box for every part: four int32[nparts] host arrays */
DDC_API int ddc_get_boxes(ddc_handle_t h, int32_t* x0, int32_t* y0, int32_t* ext_x, int32_t* ext_y);

/* pid of this rank's rows, [y_count][nx] int32, -1 on land (save_mask payload) */
DDC_API int ddc_get_pid_host(ddc_handle_t h, int32_t* out);
DDC_API int ddc_get_pid_device(ddc_handle_t h, const int32_t** dev_ptr);

/* replaces get_neighbour_info[_periodic] for every part, in save_metadata's flat layout
   (Partitioner.cpp:190-206,277-316): counts[nparts]; ids/halos/starts = concatenation over parts
   0..nparts-1 of each part's id-ascending list.  total = sum(counts). */
DDC_API int ddc_get_neighbour_counts(ddc_handle_t h, int edge, int periodic, int32_t* counts);
DDC_API int ddc_get_neighbour_total(ddc_handle_t h, int edge, int periodic, int64_t* total);
DDC_API int ddc_get_neighbours(ddc_handle_t h, int edge, int periodic, int32_t* ids, int32_t* halos,
    int32_t* halo_starts);

/* ocean cells per part: int64[nparts] */
DDC_API int ddc_get_part_loads(ddc_handle_t h, int64_t* loads);

DDC_API int ddc_get_stats(ddc_handle_t h, ddc_stats* out);

/* ---- DomainUtils on the device boundary (DomainUtils.cpp:15-35, Partitioner.cpp:20-80) ------ */
/* neighbour tables for caller-supplied boxes (no mask needed): what discover_neighbours()
   computes for every rank.  Results are fetched with the ddc_get_neighbour_* calls above. */
DDC_API int ddc_neighbours_from_boxes(ddc_handle_t h, int nparts, int nx, int ny, const int32_t* x0,
    const int32_t* y0, const int32_t* ext_x, const int32_t* ext_y, int periodic_x, int periodic_y);

/* Halo exchange driven by the neighbour tables of the last decomposition -- the consumer side, what
   examples/zoltan_comm.cpp:84-246 of the reference does with MPI subarray types and MPI_Neighbor_alltoallw.  All
   parts live in ONE device buffer: tile p is a row-major (ext_y[p] + 2) x (ext_x[p] + 2) array with a ghost frame of
   one cell around the part's box, starting at element offsets[p] (ddc_halo_tile_offsets: offsets[nparts] = total
   elements).  ddc_halo_exchange_f64 fills every ghost cell that faces a neighbour with that neighbour's adjacent
   interior cell (interior lists; periodic != 0: the periodic lists too).  It leaves the four corner cells of every
   frame as they are; ddc_halo_exchange_full_f64 below fills them too. */
DDC_API int ddc_halo_tile_offsets(ddc_handle_t h, int64_t* offsets /* nparts + 1 */);
DDC_API int ddc_halo_exchange_f64(ddc_handle_t h, double* tiles_dev, int periodic);

/* The same exchange with the parts SHARDED over the ranks (nranks >= 1, one GPU each; several ranks of one process may
   share a device).  Rank r owns parts [p_begin, p_begin + p_count) of ddc_shard_parts and holds their tiles in ONE
   library-owned device buffer, in the ddc_halo_tile_offsets layout restricted to those parts and rebased to 0
   (ddc_halo_shard_offsets: offsets[p_count] = this rank's total), so the ranks' buffers concatenated in rank order ARE
   the single-buffer layout.  ddc_halo_exchange_shards_f64 then does what ddc_halo_exchange_f64 does on that
   concatenation, bit for bit: each rank's kernels store the ghost cells its parts are the source of straight into the
   receiving part's tile, on whichever GPU it lives (posted stores over NVLink), between two flag barriers.
   Set-up: one process per GPU -- ddc_halo_export allocates this rank's buffer for up to `elems` doubles (every rank
   passes the same elems) and returns its CUDA IPC handle; the host gathers the handles (MPI_Allgather /
   torch.distributed) and hands them, in rank order, to ddc_halo_import.  One process -- ddc_halo_connect(handles, n,
   elems, tiles_dev): handles[q] is rank q of n; ranks that share a device must run on different streams.  These
   buffers are independent of the ddc_peer_* exchange buffers: decompositions may use NCCL or peer memory alike.
   The flags of the exchange carry the number of the exchange: after the buffers are joined every rank makes the same
   number of ddc_halo_exchange_shards_f64 calls, as every rank makes the same ddc_partition calls for the peer
   buffers above.  The call only enqueues (on the handle's stream) and returns, so one host thread can drive several
   handles in turn; ddc_synchronize reports a rank that did not reach an exchange within the timeout as DDC_ERR_PEER.
   Errors are the same on every rank and come before anything is enqueued: DDC_ERR_STATE without buffers or without
   ddc_halo_shard_offsets for the current decomposition, DDC_ERR_ARG when some rank's tiles exceed `elems`.  Without
   neighbour tables (one part, or no DDC_WANT_NEIGHBOURS) the exchange does nothing on every rank. */
DDC_API void ddc_shard_parts(int nparts, int nranks, int rank, int* p_begin, int* p_count); /* p_begin = rank * nparts / nranks */
DDC_API int ddc_halo_shard_offsets(ddc_handle_t h, int64_t* offsets /* p_count + 1 */);
DDC_API int ddc_halo_export(ddc_handle_t h, int64_t elems, double** tiles_dev, void* ipc_handle_out /* DDC_IPC_HANDLE_BYTES */);
DDC_API int ddc_halo_import(ddc_handle_t h, const void* all_handles /* nranks * DDC_IPC_HANDLE_BYTES, rank order */);
DDC_API int ddc_halo_connect(ddc_handle_t* handles, int n, int64_t elems, double** tiles_dev /* n */);
DDC_API int ddc_halo_exchange_shards_f64(ddc_handle_t h, int periodic);
/* unmap the other ranks' halo buffers.  Shutdown order as for ddc_peer_close: every rank calls ddc_halo_close(), the
   host synchronises the ranks, then every rank calls ddc_destroy(), which frees its own halo buffer. */
DDC_API int ddc_halo_close(ddc_handle_t h);

/* Halo scatter and gather: a field between its rows and the parts' tiles.  A field is double [ny][nx], x fastest, the
   layout of the mask and the pid map; rank r of a sharded run holds rows [y_begin, y_begin + y_count) of
   ddc_shard_rows(ny, nranks, r).  Scatter writes the INTERIOR of every tile from the field: row j + 1, column i + 1 of
   part p's tile gets field[y0[p] + j][x0[p] + i].  Gather is the inverse: it reads interiors only and writes every
   cell of the field (or of this rank's rows) exactly once -- the boxes tile the whole domain, land included.  Neither
   reads nor writes a ghost frame.  Values are copied bit for bit (NaN payloads, -0.0, subnormals): no arithmetic.
   Single buffer (the ddc_halo_exchange_f64 layout, all parts): field_dev is the whole field.  Needs
   ddc_halo_tile_offsets for the current decomposition (else DDC_ERR_STATE) and non-null pointers (else DDC_ERR_ARG);
   it does NOT need neighbour tables: with one part, or without DDC_WANT_NEIGHBOURS, the whole field still moves.
   Sharded (the ddc_halo_exchange_shards_f64 buffers): rows_dev is this rank's row block; scatter stores every cell of
   it into its part's tile on whichever rank owns the part (posted stores), gather loads every cell of it from there.
   The buffers, shard offsets and capacity are checked as for the exchange, with the same status codes, from
   replicated data and before anything is enqueued, so they come out the same on every rank.  One check is this
   rank's alone: rows_dev == NULL on a rank whose block has rows is DDC_ERR_ARG on that rank (NULL is fine for an empty
   block: ddc_shard_rows' ceil rule leaves the last ranks empty when ny is small).  Its peers then wait for it in vain
   and ddc_synchronize reports DDC_ERR_PEER on them, as for a rank that never makes the call.
   Scatter and gather are sharded halo calls like the exchange: each takes the next halo step number, behind the same
   two flag barriers, so every rank must make the same sequence of sharded halo calls; exchanges, scatters and gathers
   may be mixed freely as long as the order is the same on every rank.  After a sharded gather returns on the stream,
   no rank still reads this rank's tiles.  The calls only enqueue (on the handle's stream), so one host thread can
   drive several handles. */
DDC_API int ddc_halo_scatter_f64(ddc_handle_t h, const double* field_dev, double* tiles_dev);
DDC_API int ddc_halo_gather_f64(ddc_handle_t h, const double* tiles_dev, double* field_dev);
DDC_API int ddc_halo_scatter_shards_f64(ddc_handle_t h, const double* rows_dev);
DDC_API int ddc_halo_gather_shards_f64(ddc_handle_t h, double* rows_dev);

/* Corner ghosts: the whole frame, for stencils that read the diagonal neighbour (9-point stencils, bilinear
   interpolation at cell corners, B/C-grid averaging).  Corner c of part p with box {x0, y0, ex, ey} is the cell
       DDC_BOTTOM_LEFT  (x0 - 1,  y0 - 1)   tile row 0,      column 0
       DDC_BOTTOM_RIGHT (x0 + ex, y0 - 1)   tile row 0,      column ex + 1
       DDC_TOP_LEFT     (x0 - 1,  y0 + ey)  tile row ey + 1, column 0
       DDC_TOP_RIGHT    (x0 + ex, y0 + ey)  tile row ey + 1, column ex + 1
   Its SOURCE is the box that contains that cell; when several do (caller-supplied boxes may overlap), the lowest-id box
   of positive area.  The owner of a corner is often a box that touches p at that corner only, which is no neighbour in
   the edge lists.  A corner is INTERIOR when its cell lies in [0, nx) x [0, ny); it is PERIODIC when the cell lies
   outside in x and / or y, the decomposition is periodic in every direction in which it lies outside, and the wrapped
   cell has a source.  Every other corner has no source.  The source may be p itself (a periodic corner of a part that
   spans the domain), and zero-area parts have corners by the same rule.
   ddc_get_corner_neighbours: for every part p, ids[p] = the source of corner `corner` in the interior (periodic = 0) or
   periodic (periodic = 1) set, -1 when it has none there, and starts[p] = the cell's index in the source's flattened
   box, (y - y0[q]) * ex[q] + (x - x0[q]) with x and y wrapped for a periodic corner (the halo_starts convention of
   ddc_get_neighbours).  int32[nparts] host arrays, either may be NULL.  Valid after ddc_partition or
   ddc_neighbours_from_boxes.
   ddc_halo_exchange_full_f64 fills exactly what ddc_halo_exchange_f64 fills, bit for bit, plus every corner ghost
   that has a source (interior set; periodic != 0: the periodic set too), copied as 64-bit words.  Preconditions and
   status codes are those of ddc_halo_exchange_f64, and like it the call does nothing without neighbour tables (one
   part, or no DDC_WANT_NEIGHBOURS).  ddc_halo_exchange_full_shards_f64 is the same on the sharded buffers, with the
   checks and status codes of ddc_halo_exchange_shards_f64: it takes the next halo step number and mixes with sharded
   exchanges, scatters and gathers in any order that is the same on every rank.  A corner ghost is stored by the rank
   that owns its source part.
   Parts of zero area, in every halo exchange above: a part of zero area is never a source; its entries in the edge
   lists are skipped.  When the boxes tile the domain, which ddc_partition's always do, every ghost cell that faces a
   neighbour therefore holds its (wrapped) cell, whatever the part sizes.  A zero-area receiver gets its ghosts by the
   same rule: a zero-width part has a left and a right ghost column, a zero-height part a bottom and a top ghost row.
   Boxes given to ddc_neighbours_from_boxes that overlap or leave cells uncovered are outside this rule: an edge ghost
   may then have several sources, and which one it ends up holding is not defined. */
DDC_API int ddc_get_corner_neighbours(ddc_handle_t h, int corner, int periodic, int32_t* ids /* nparts */,
    int32_t* starts /* nparts */);
DDC_API int ddc_halo_exchange_full_f64(ddc_handle_t h, double* tiles_dev, int periodic);
DDC_API int ddc_halo_exchange_full_shards_f64(ddc_handle_t h, int periodic);

/* Wide halos: ghost frames of width w for stencils that reach further than one cell (biharmonic operators, high-order
   advection, or k sweeps of a 5- or 9-point stencil per exchange with w = k).  ddc_halo_set_width sets the w that every
   halo call of the handle uses; the default is 1, which is exactly the layout and behaviour described above.  It may be
   called before ddc_partition.  A w that differs from the current one drops the tile and shard offsets, as a new
   decomposition does: every halo call returns DDC_ERR_STATE until ddc_halo_tile_offsets / ddc_halo_shard_offsets are
   called again.  w < 1 or w > DDC_MAX_HALO_WIDTH is DDC_ERR_ARG.  The bound keeps a corner block (w * w cells) and
   x0 - w, x0 + ext + w of every box whose extents stay below INT_MAX - 2 DDC_MAX_HALO_WIDTH within the 32-bit ints of
   the kernels' index arithmetic.
   With width w:
     - Layout: tile p is a row-major (ext_y + 2 w) x (ext_x + 2 w) array; interior cell (i, j) is at row j + w, column
       i + w.  ddc_halo_tile_offsets and ddc_halo_shard_offsets return these sizes; the sharded buffers remain the
       single-buffer layout restricted to the rank's parts.  Scatter and gather read and write the interiors only, at
       that position, bit for bit.
     - Source rule: a frame cell of p lies outside p's box at (x, y), x0 - w <= x < x0 + ext_x + w and the same in y.
       Its source is the positive-area box that contains the cell -- the cell itself when it lies in [0, nx) x [0, ny)
       (interior), else the wrapped cell (x mod nx, y mod ny) when the decomposition is periodic in every direction in
       which the cell lies outside (periodic).  A frame wider than the domain wraps as often as it needs.  This is the
       corner rule above applied to every frame cell; on a tiling at w = 1 it selects exactly the ghosts the edge lists
       fill.
     - ddc_halo_exchange_f64 / ddc_halo_exchange_shards_f64 fill every cell of the four w-deep edge strips that has a
       source (interior; periodic != 0: periodic too); the _full_ calls also fill the four w x w corner blocks.  Cells
       with no source keep what they held.  When the boxes tile the domain, which ddc_partition's always do, every
       filled cell holds its wrapped cell, zero-width and zero-height parts included; overlapping caller boxes stay
       outside the rule as above.  Without neighbour tables the exchanges still do nothing; the status codes and the
       shared step counter of the sharded calls are unchanged; ddc_get_corner_neighbours still describes the diagonal
       cell, whatever w.
     - Sharded: every rank must set the same w.  A mismatch cannot make a kernel write past a buffer -- each rank
       checks every rank's tile total at its own w against the common elems, and its items address only tiles of
       that size -- but its ghosts are wrong. */
#define DDC_MAX_HALO_WIDTH 1024
DDC_API int ddc_halo_set_width(ddc_handle_t h, int width);

/* ---- synthetic masks (SURVEY 8d): deterministic value-noise land-sea mask, generated directly
   into device memory so that no 4 GiB file is needed for the large configurations.
   land_frac in [0,1] is the target land fraction; rows as in ddc_set_mask_device. */
DDC_API int ddc_generate_mask_device(ddc_handle_t h, int32_t* dev_rows, int nx, int ny, int y_begin,
    int y_count, uint64_t seed, double land_frac);

/* the same generator on the host (input staging for end-to-end runs and for the CPU baseline) */
DDC_API int ddc_generate_mask_host(int32_t* rows, int nx, int ny, int y_begin, int y_count,
    uint64_t seed, double land_frac);

DDC_API const char* ddc_version(void);

#ifdef __cplusplus
}
#endif
#endif /* DDC_H */
