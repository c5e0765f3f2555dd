/*
 * mkb200.h -- C-ABI of libmkb200.so: the B200-native voxel-occupancy and trajectory-distance engine.
 *
 * This is the drop-in boundary for ONE hot path of Acellera/moleculekit (SURVEY.md section 8):
 *   moleculekit/occupancy_utils/occupancy_utils.pyx   (calculate_occupancy)
 *   moleculekit/distance_utils/distance_utils.pyx     (dist_trajectory, contacts_trajectory,
 *                                                      dist_trajectory_reduction[_pairs], cdist, pdist,
 *                                                      squareform, get_collisions)
 * The reference exposes these as Cython `def` functions over numpy memoryviews (no C header); each entry
 * point below cites the reference function it replaces.  Conventions:
 *   - plain C types only: pointers, sizes, scalars.  No torch / numpy types.
 *   - bulk arrays are DEVICE pointers (the Python host obtains them from torch.Tensor.data_ptr());
 *     small per-grid descriptors are HOST arrays (they size the launch); `stream` is a cudaStream_t
 *     passed as void* (0 = legacy default stream).  All work is stream-ordered; nothing blocks the host
 *     except where stated (mkb_contacts_count returns a host total).
 *   - every function returns MKB_OK (0) or a negative mkb_status; mkb_last_error(h) gives the message.
 *   - the caller owns every input/output array; the handle owns only scratch (cell lists, scan temp),
 *     grown on demand and freed by mkb_destroy.  One handle per device; not thread-safe per handle.
 *   - there is NO CPU fallback: without a CUDA device mkb_create fails with MKB_ERR_CUDA.
 */
#ifndef MKB200_H
#define MKB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MKB_VERSION 100 /* 0.1.0 */

typedef enum {
    MKB_OK = 0,
    MKB_ERR_BAD_ARG = -1,
    MKB_ERR_CUDA = -2,
    MKB_ERR_NOMEM = -3,
    MKB_ERR_CAPACITY = -4,
    MKB_ERR_UNSUPPORTED = -5 /* a valid request this entry point cannot serve (e.g. compact output outside its domain) */
} mkb_status;

typedef struct mkb_ctx *mkb_handle_t;

/* flags for the occupancy entry points */
#define MKB_OCC_ACCUMULATE 1u /* out = max(out, value): the reference accumulates into the caller's buffer
                                 (occupancy_utils.pyx:61); without it `out` is overwritten (caller passes zeros,
                                 voxeldescriptors.py:531, so both agree) */
#define MKB_OCC_LAYOUT_CXYZ 2u /* SURVEY 8f row 1: grid b is written channel-major, out[b] = float32 [C][nx][ny][nz]
                                 (the layout a Conv3d consumer wants, instead of the reference's [nx][ny][nz][C]
                                 reshaped view, voxeldescriptors.py:298-299); grid b still starts at out + out_offset*C.
                                 Same values bit for bit.  mkb_occupancy_grid_batch only. */

/* output modes of the distance entry points (host post-ops of projections/util.py:74-84 fused in) */
#define MKB_DIST_DISTANCES 0 /* float32 distances, optionally truncated */
#define MKB_DIST_CONTACTS 1  /* uint8 (bool) = distance <= threshold, after optional truncate */
#define MKB_DIST_DISTANCES_FAST 4 /* float32 distances within 4 ulp of the reference's float32 sequence (the reference's
                                     minimum-image roundings, fused sum of squares, approximate square root); same NaN
                                     pattern; BASELINE north star asks for 1e-5 relative.  mkb_dist_trajectory only. */

int mkb_version(void);
int mkb_create(int device, mkb_handle_t *out);
int mkb_destroy(mkb_handle_t h);
const char *mkb_last_error(mkb_handle_t h);
/* number of kernels this handle has launched so far (bench.py's gpu_launches) */
int64_t mkb_launch_count(mkb_handle_t h);
/* Per-kernel device timing for the roofline report: when on, the occupancy and distance entry points record CUDA
 * events on the launch stream before their preparation kernels, before the main kernel and after it.
 * mkb_get_timing synchronises on the last event and returns the two intervals of the most recent call (ms). */
int mkb_set_timing(mkb_handle_t h, int on);
int mkb_get_timing(mkb_handle_t h, float *prep_ms, float *main_ms);
/* name of the main kernel the most recent occupancy / distance entry point launched (static string; "" before any call) */
const char *mkb_last_kernel(mkb_handle_t h);

/* One regular voxel grid: centre of voxel (ix,iy,iz) = fl(fl(i*voxelsize) + origin[d]) in float64, exactly
 * as moleculekit/tools/voxeldescriptors.py:125-132,245 builds `centers`; flat voxel index
 * (ix*ny + iy)*nz + iz (z fastest), channels minor. */
typedef struct {
    double origin[3];   /* bb_min of getCenters (voxeldescriptors.py:231-243) */
    double voxelsize;   /* isotropic voxel edge, Angstrom */
    int32_t dims[3];    /* nx, ny, nz */
    int32_t reserved;
    int64_t atom_begin; /* rows [atom_begin, atom_end) of coords/sigmas belong to this grid */
    int64_t atom_end;
    int64_t out_offset; /* first voxel of this grid in `out`, in voxels (row = C floats) */
} mkb_grid_desc;

/* K1+K2: batched occupancy on regular grids.
 * Replaces calculate_occupancy (occupancy_utils.pyx:34-61) + the centre materialisation of getCenters for every
 * grid of the batch in one launch sequence (bin atoms -> scan -> scatter -> fill).
 *   coords  [n_atoms,3] float32 device      (reference: coords f32[:,:])
 *   sigmas  [n_atoms,C] float64 device      (reference: sigmas f64[:,:]; 0 = channel off, NaN ignored)
 *   grids   [B] HOST descriptors
 *   out     [sum_b nx*ny*nz, C] float32 device (the reference's float64 results; the host wrapper upcasts)
 * 1 <= C <= 32. */
int mkb_occupancy_grid_batch(mkb_handle_t h, void *stream, const float *coords, const double *sigmas,
                             int64_t n_atoms, int32_t C, const mkb_grid_desc *grids, int32_t B,
                             float *out, uint32_t flags);

/* K1 with device-side channel assembly (SURVEY 8f row 1): the reference builds sigmas = vdw_radius[:, None] *
 * channels.astype(float) on the host (voxeldescriptors.py:332-335); here the (n_atoms,) float64 radii and a per-atom
 * channel bit mask (bit c set = atom belongs to channel c) are the inputs and the (n_atoms, C) float64 matrix never
 * exists -- 12 instead of 8*C bytes per atom over PCIe.  Bit-identical to mkb_occupancy_grid_batch on that matrix. */
int mkb_occupancy_grid_batch_masked(mkb_handle_t h, void *stream, const float *coords, const double *radii,
                                    const uint32_t *chanmask, int64_t n_atoms, int32_t C, const mkb_grid_desc *grids,
                                    int32_t B, float *out, uint32_t flags);

/* K1 with a COMPACT result (end-to-end transfers): ~70 % of a pocket grid is empty, so instead of the dense grid the
 * kernel emits one 4 KB record [4 x][4 y][8 z][8 channels] per 4x4x8-voxel block that has an atom within 5 A, and an
 * index that says which blocks those are.  8 channels, voxel-major.  Block b of grid g (b = ((ix/4)*ceil(ny/4) +
 * iy/4)*ceil(nz/8) + iz/8, grids in batch order) has a record iff blk_rank[b + 1] != blk_rank[b]; the record is
 * records[1024 * blk_rank[b] ...].  records: device, room for mkb_occupancy_compact_blocks(grids, B) records in the
 * worst case; blk_rank: device uint32 [rank_capacity >= blocks + 1].  Exactly one of sigmas / (radii, chanmask) is given.
 * mkb_occupancy_expand_host rebuilds grids [g0, g1) of the dense float32 (sum M, 8) HOST array from host copies of the
 * records (`records` points at record rec0; NULL = only zero-fill the blocks without a record) with n_threads threads;
 * missing blocks are zero-filled; out_f64 != 0 writes
 * float64 (the reference's result dtype).  The result is bit-identical to mkb_occupancy_grid_batch. */
int mkb_occupancy_grid_batch_compact(mkb_handle_t h, void *stream, const float *coords, const double *sigmas,
                                     const double *radii, const uint32_t *chanmask, int64_t n_atoms,
                                     const mkb_grid_desc *grids, int32_t B, float *records, uint32_t *blk_rank,
                                     int64_t rank_capacity);
int64_t mkb_occupancy_compact_blocks(const mkb_grid_desc *grids, int32_t B);
/* K1 straight into the caller's HOST array (end-to-end callers with a page-locked result, e.g. cudaHostAlloc / torch
 * pin_memory: under UVA such memory is device-accessible at the same address).  `out_mapped` is that dense float32
 * (sum M, 8) host array: the kernel stores the blocks that have an atom within 5 A directly into it over PCIe (TMA bulk
 * row copies, ~30 % of the bytes) and does not touch the others; the block index (as for the compact call) is computed before
 * the fill kernel starts and copied to `host_rank` (page-locked, blocks + 1 words) on a side stream, so the host can
 * zero-fill the empty blocks (mkb_occupancy_expand_host with records == NULL) WHILE the GPU computes and writes.
 * mkb_occupancy_wait_index blocks until host_rank has arrived; the caller synchronises `stream` before reading `out`. */
int mkb_occupancy_grid_batch_to_host(mkb_handle_t h, void *stream, const float *coords, const double *sigmas,
                                     const double *radii, const uint32_t *chanmask, int64_t n_atoms,
                                     const mkb_grid_desc *grids, int32_t B, float *out_mapped, uint32_t *blk_rank,
                                     int64_t rank_capacity, uint32_t *host_rank);
int mkb_occupancy_wait_index(mkb_handle_t h);
int mkb_occupancy_expand_host(const mkb_grid_desc *grids, int32_t g0, int32_t g1, const uint32_t *blk_rank,
                              const float *records, int64_t rec0, void *out, int32_t out_f64, int32_t n_threads);

/* Voxel centres on the device (SURVEY 8f row 1), exactly getCenters (voxeldescriptors.py:116-123,243-247):
 * centers[(out_offset_b + v) * 3 + d] = fl(fl(i_d * voxelsize) + origin[d]), v = (ix*ny + iy)*nz + iz; float64 device.
 * K1 itself never needs this array. */
int mkb_grid_centers(mkb_handle_t h, void *stream, const mkb_grid_desc *grids, int32_t B, double *centers);

/* rotateCoordinates (voxeldescriptors.py:78-114), batched (SURVEY 8f row 1): molecule b = atoms [atom_offsets[b],
 * atom_offsets[b+1]) (int64 device, [B+1]) is rotated three times in succession, new = (x - c_b) . R_{b,r}^T + c_b in
 * float64 (row-major 3x3 matrices [B][3][3][3] and centres [B][3], float64 device; the host wrapper builds the matrices
 * with the reference's rotationMatrix formula, util.py:101-117).  Result as float32 (what K1 consumes) and/or float64
 * (what the reference returns); either output may be NULL.  Products and sums individually rounded, left to right
 * (numpy's BLAS order is unspecified: parity is 1e-12 relative, not bitwise). */
int mkb_rotate_coords(mkb_handle_t h, void *stream, const float *coords, int64_t n_atoms, const int64_t *atom_offsets,
                      int32_t B, const double *matrices, const double *centers, float *out_f32, double *out_f64);

/* K1b: occupancy at arbitrary centres (the `usercenters` branch, voxeldescriptors.py:338-340 ->
 * calculate_occupancy).  centers [M,3] float64 device; same arithmetic contract. */
int mkb_occupancy_points(mkb_handle_t h, void *stream, const double *centers, int64_t M,
                         const float *coords, const double *sigmas, int64_t n_atoms, int32_t C,
                         float *out, uint32_t flags);

/* Trajectory view shared by the distance entry points: coords is float32 (n_atoms, 3, F) frame-minor
 * (moleculekit/molecule.py:144-146); element (a, d, f) lives at coords[(a*3 + d)*frame_stride + f], box (3, F) at
 * box[d*frame_stride_box + f].  A frame shard [f0, f1) of a resident trajectory is (coords + f0, n_frames = f1 - f0,
 * frame_stride = F). */
typedef struct {
    const float *coords;
    const float *box;
    int64_t n_atoms;
    int64_t n_frames;
    int64_t frame_stride;     /* elements between consecutive (atom, dim) rows of coords */
    int64_t frame_stride_box; /* elements between consecutive rows of box */
} mkb_traj;

/* K3: dist_trajectory (distance_utils.pyx:126-155) with the truncate / contacts post-ops of
 * pp_calcDistances (projections/util.py:74-84) fused into the store.
 *   sel1 [n1], sel2 [n2], chains [n_atoms] uint32 device; out [n_frames, P] row-major, P = n1*n2 or n1*(n1-1)/2
 *   when selfdist (then sel2 must equal sel1 as in the reference); float32 (mode 0) or uint8 (mode 1).
 *   truncate: NaN = off.  Arithmetic: every float op individually rounded (no FMA), roundf half-away, sqrtf IEEE
 *   -> bit-identical to the reference binary. */
int mkb_dist_trajectory(mkb_handle_t h, void *stream, const mkb_traj *t, const uint32_t *sel1, int64_t n1,
                        const uint32_t *sel2, int64_t n2, const uint32_t *chains, int32_t selfdist, int32_t pbc,
                        int32_t mode, float truncate, float threshold, void *out);

/* K4: contacts_trajectory (distance_utils.pyx:59-93), two calls.
 * count: row_offsets [n_frames*n1 + 1] int64 device receives the exclusive scan of the per-(frame, i) contact
 *        counts; *total_pairs (HOST) receives the grand total (this call synchronises the stream).
 * fill : pairs [total_pairs, 2] uint32 device receives (sel1[i], sel2[j]) in the reference's order: frame-major,
 *        then i ascending, then j ascending -- bit-exact index output.  thr2 = threshold*threshold in float
 *        (pyx:77), compare `<=`.
 * The count call keeps one hit mask per (row, 32 columns) in the handle; a fill call with the SAME arguments (pointers,
 * sizes, flags, threshold) emits the pairs from those masks instead of evaluating the distances again, any other fill call
 * recomputes them.  Either way the pairs are consistent with the row_offsets of the count call. */
int mkb_contacts_count(mkb_handle_t h, void *stream, const mkb_traj *t, const uint32_t *sel1, int64_t n1,
                       const uint32_t *sel2, int64_t n2, const uint32_t *chains, int32_t selfdist, int32_t pbc,
                       float threshold, int64_t *row_offsets, int64_t *total_pairs);
int mkb_contacts_fill(mkb_handle_t h, void *stream, const mkb_traj *t, const uint32_t *sel1, int64_t n1,
                      const uint32_t *sel2, int64_t n2, const uint32_t *chains, int32_t selfdist, int32_t pbc,
                      float threshold, const int64_t *row_offsets, uint32_t *pairs);

/* K5: dist_trajectory_reduction / dist_trajectory_reduction_pairs (distance_utils.pyx:211-350) with the same
 * fused post-ops (projections/util.py:212-223).  Groups are CSR (offsets [G+1] int64, atoms int32), device.
 * gchains1/2 [G1]/[G2] uint32 = chain id of each group's first atom (projections/util.py:174-179).
 * red1/red2: 0 closest, 1 centre of mass (float accumulation in atom order, pyx:160-183).
 * pairs != 0: group g of set 1 against group g of set 2 (G1 == G2), out [n_frames, G1];
 * else out [n_frames, G1*G2] or [n_frames, G1*(G1-1)/2] when selfdist. */
int mkb_dist_reduction(mkb_handle_t h, void *stream, const mkb_traj *t, const int64_t *g1_off,
                       const int32_t *g1_atoms, int64_t G1, const int64_t *g2_off, const int32_t *g2_atoms,
                       int64_t G2, const uint32_t *gchains1, const uint32_t *gchains2, int32_t selfdist,
                       int32_t pbc, const float *masses, int32_t red1, int32_t red2, int32_t pairs, int32_t mode,
                       float truncate, float threshold, void *out);

/* K6: cdist / pdist / squareform / get_collisions (distance_utils.pyx:355-435, 98-121).  Row-major float32. */
int mkb_cdist(mkb_handle_t h, void *stream, const float *a, int64_t n1, const float *b, int64_t n2, int32_t D,
              float *out);
int mkb_pdist(mkb_handle_t h, void *stream, const float *a, int64_t n, int32_t D, float *out);
int mkb_squareform(mkb_handle_t h, void *stream, const float *d, int64_t n, int64_t dim, float *out);
/* get_collisions: single frame, no pbc, LOCAL (i, j) indices; same two-call protocol as K4 with
 * row_offsets [n1 + 1]. */
int mkb_collisions_count(mkb_handle_t h, void *stream, const float *c1, int64_t n1, const float *c2, int64_t n2,
                         float threshold, int64_t *row_offsets, int64_t *total_pairs);
int mkb_collisions_fill(mkb_handle_t h, void *stream, const float *c1, int64_t n1, const float *c2, int64_t n2,
                        float threshold, const int64_t *row_offsets, uint32_t *pairs);

/* K8 (SURVEY 8f row 2): MetricShell radial histogram fused on the distance evaluation; replaces _shells
 * (moleculekit/projections/metricshell.py:183-202) and the (F, P) matrix it consumed.  counts [n_frames, n1, numshells]
 * uint32: partners j of centre sel1[c] with edges[e] < d <= edges[e+1] (edges [numshells+1] float64 device; d = the
 * reference's float32 distance, truncated if truncate is not NaN, compared in float64).  selfdist: sel2 == sel1 and a
 * centre is not its own partner.  1 <= numshells <= 32. */
int mkb_shell_counts(mkb_handle_t h, void *stream, const mkb_traj *t, const uint32_t *sel1, int64_t n1,
                     const uint32_t *sel2, int64_t n2, const uint32_t *chains, int32_t selfdist, int32_t pbc,
                     float truncate, const double *edges, int32_t numshells, uint32_t *counts);

/* K7 (stretch row a13): bond perception, replaces bond_grid_search (moleculekit/bondguesser.py:259-392) +
 * grid_bonds/_is_close (moleculekit/bondguesser_utils/bondguesser_utils.pyx:89-163).  coords [n,3] / radii [n] float32,
 * is_hydrogen [n] uint32, device.  pairdist = final grid box edge (after the caller's max_boxes enlargement loop).
 * Same two-call protocol as K4 with row_offsets [n + 1]; pairs come out as (i < j), unordered inside a row -- the SET
 * equals the reference's (the host wrapper returns it in canonical sorted order). */
int mkb_bonds_count(mkb_handle_t h, void *stream, const float *coords, const float *radii, const uint32_t *is_hydrogen,
                    int64_t n, float pairdist, int64_t *row_offsets, int64_t *total_pairs);
int mkb_bonds_fill(mkb_handle_t h, void *stream, const float *coords, const float *radii, const uint32_t *is_hydrogen,
                   int64_t n, float pairdist, const int64_t *row_offsets, uint32_t *pairs);

/* K11 (SURVEY 8f row 4, second half): XTC compressed coordinates decoded on the device; replaces the frame loop of
 * xtc_read_new / xtc_read_frame (moleculekit/fileformats/xtc/src/xtc_src.cpp:195-258) around xdrfile_decompress_coord_float
 * (src/xdrfile.cpp:750-982) and its host-side scatter into the frame-minor array.  file_bytes = the XTC file on the device;
 * frames[f] (HOST) = one coordinate block as found by walking the XDR frame headers: byte offset and length of the bit stream,
 * precision, minint/maxint, initial smallidx (smallidx < 0: natoms <= 9, the block is 3*natoms big-endian floats).
 * coords (natoms, 3, n_frames) float32 device, element (a, d, f) at coords[(a*3 + d)*frame_stride + f], in nm, or multiplied
 * by `scale` as a second float32 operation (10 = the reference's `coords *= 10`, readers.py:1846).  status [n_frames] int32
 * device: 0 = ok, negative = corrupt block.  Blocks are read as big-endian 32-bit words: file_bytes + data_offset must be
 * 4-byte aligned (XDR guarantees it for a buffer that starts on a word) and readable up to the next multiple of 4 bytes.
 * Bit-identical to the reference reader. */
typedef struct {
    int64_t data_offset;
    int32_t nbytes;
    int32_t natoms;
    float precision;
    int32_t minint[3];
    int32_t maxint[3];
    int32_t smallidx;
} mkb_xtc_frame;
int mkb_xtc_decode(mkb_handle_t h, void *stream, const uint8_t *file_bytes, int64_t file_size, const mkb_xtc_frame *frames,
                   int64_t n_frames, int64_t natoms, float *coords, int64_t frame_stride, float scale, int32_t *status);

/* K10 (SURVEY 8f row 3): the kernel of the `within` / `exwithin` atom selections, replaces within_distance
 * (moleculekit/atomselect_utils/atomselect_utils.pyx:612-653; called from atomselect/atomselect.py:243-251).
 * coords [n_atoms,3] float32 device (one frame, row-major); sel1 [n1] uint32 device = query atoms (NULL = all atoms,
 * n1 == n_atoms); sel2 [n2] uint32 device = source atoms; results [n1] uint8 device: results[ii] is SET to 1 when some
 * source atom lies at float32 squared distance < cutoff*cutoff of query ii and left untouched otherwise (the reference
 * only ever writes True).  Cell list over the source atoms instead of the reference's n1 x n2 loop; identical output. */
int mkb_within_distance(mkb_handle_t h, void *stream, const float *coords, int64_t n_atoms, const uint32_t *sel1,
                        int64_t n1, const uint32_t *sel2, int64_t n2, float cutoff, uint8_t *results);

/* K9 (SURVEY 8f row 4): orthorhombic wrapping of bonded groups, replaces wrap_box
 * (moleculekit/wrapping/wrapping.pyx:91-144; called from Molecule.wrap, moleculekit/molecule.py:2077).  t->coords is
 * MODIFIED IN PLACE like the reference's array.  groups [n_groups] uint32 device: ascending first-atom offsets of
 * consecutive groups, group g = atoms [groups[g], groups[g+1]) -- so n_groups - 1 ranges, the last entry (n_atoms in
 * Molecule.wrap) closes the last one.  centersel [n_centersel] uint32 device: atoms whose running-mean centre is the box
 * centre of each frame; when n_centersel == 0 the fixed `center` (HOST float[3]) is used instead (pyx:106-108).
 * float32 arithmetic with one rounding per operation and roundf half-away: bit-identical to the reference.  Index
 * ranges are the caller's responsibility (the reference compiles with boundscheck off as well). */
int mkb_wrap_box(mkb_handle_t h, void *stream, const mkb_traj *t, const uint32_t *groups, int64_t n_groups,
                 const uint32_t *centersel, int64_t n_centersel, const float *center);

/* K9b: wrapping of bonded groups in triclinic cells, replaces wrap_triclinic_unitcell (moleculekit/wrapping/wrapping.pyx:147-250,
 * unitcell = 2) and wrap_compact_unitcell (pyx:255-344 with get_pbc pyx:357-451 and pbc_dx pyx:454-505; unitcell = 0 is
 * its mode 0 "rectangular", 1 its mode 1 "compact") -- the calls Molecule.wrap makes when a box angle differs from 90
 * (moleculekit/molecule.py:2078-2090).  t->coords is MODIFIED IN PLACE (t->box is not used); boxvectors [3][3][stride]
 * float64 device, row i = box vector i, frame minor like Molecule.boxvectors.  groups / centersel / center as in
 * mkb_wrap_box; every atom is first centred on the wrap centre (also atoms outside all groups), then each group is
 * translated as the reference does it, float32 centres against float64 cell arithmetic: bit-identical coordinates.
 * Returns MKB_ERR_BAD_ARG "Too many triclinic vectors!!" where the reference raises that ValueError (pyx:439-441).  The
 * reference's unbounded while loops are capped at 2^20 iterations (only reached by cells without a positive diagonal). */
int mkb_wrap_triclinic(mkb_handle_t h, void *stream, const mkb_traj *t, const double *boxvectors,
                       int64_t bv_frame_stride, const uint32_t *groups, int64_t n_groups, const uint32_t *centersel,
                       int64_t n_centersel, const float *center, int32_t unitcell);

/* K12: hydrogen bonds over a trajectory, replaces hbonds.calculate (moleculekit/interactions/hbonds/hbonds.pyx:25-134; called
 * by hbonds_calculate, moleculekit/interactions/interactions.py:365-467).  donors [n_donors][2] uint32 device = (heavy atom,
 * hydrogen); acceptors [n_acceptors] uint32 device; sel1 / sel2 [n_atoms] uint32 device 0/1 flags; t->box is the
 * orthorhombic box (3, F).  intra != 0: both atoms in sel1 (pyx:70-73), else one in sel1 and the other in sel2
 * (pyx:74-77).  ignore_hs != 0: the heavy atom's distance is tested, no angle, hydrogen reported as -1 (pyx:101-105).
 * Two calls like K4 -- count: row_offsets [n_frames*n_donors + 1] int64 device = exclusive scan of the per-(frame, donor)
 * hit counts, *total_triples (HOST) the total (synchronises the stream); fill: triples [total][3] int32 device =
 * (heavy, hydrogen | -1, acceptor) in the reference's order (frame, donor, acceptor ascending).  Same booleans as the
 * reference binary (built as C++: round / sqrt / acos on float arguments are the float overloads), the acosf comparison as
 * a precomputed cosine bound. */
int mkb_hbonds_count(mkb_handle_t h, void *stream, const mkb_traj *t, const uint32_t *donors, int64_t n_donors,
                     const uint32_t *acceptors, int64_t n_acceptors, const uint32_t *sel1, const uint32_t *sel2,
                     float dist_threshold, float angle_threshold, int32_t intra, int32_t ignore_hs, int64_t *row_offsets,
                     int64_t *total_triples);
int mkb_hbonds_fill(mkb_handle_t h, void *stream, const mkb_traj *t, const uint32_t *donors, int64_t n_donors,
                    const uint32_t *acceptors, int64_t n_acceptors, const uint32_t *sel1, const uint32_t *sel2,
                    float dist_threshold, float angle_threshold, int32_t intra, int32_t ignore_hs,
                    const int64_t *row_offsets, int32_t *triples);

/* K13: ring-based interaction detectors over a trajectory.  mode 0 replaces pipi.calculate
 * (moleculekit/interactions/pipi/pipi.pyx:86-185), mode 1 cationpi.calculate (interactions/cationpi/cationpi.pyx:91-173),
 * mode 2 sigmahole.calculate (interactions/sigmahole/sigmahole.pyx:91-174); callers pipi_calculate / cationpi_calculate /
 * sigmahole_calculate (moleculekit/interactions/interactions.py:621-946).  rings_atoms uint32 device: concatenated ring atom
 * indexes; starts1 [n_rings1 + 1] uint32 device: ring start indexes of the first set.  second, uint32 device: mode 0 the start
 * indexes [n_second + 1] of the second ring set inside the same rings_atoms; mode 1 cation atom indexes [n_second]; mode 2
 * (halogen, bonded partner) pairs [n_second][2].  p0..p3: mode 0 dist_threshold1, angle_threshold1_max, dist_threshold2,
 * angle_threshold2_min; modes 1 / 2 dist_threshold, angle_threshold_min (p2, p3 unused).  Two calls like K4 -- count:
 * row_offsets [n_frames*n_rings1 + 1] int64 device, *total_pairs (HOST; synchronises the stream); fill: pairs [total][2]
 * int32 device = (ring index, second ring index | cation atom | halogen atom) and distangles [total][2] float32 device =
 * (distance, angle in degrees), in the reference's order (frame, ring, partner ascending).  Pairs and distances are the
 * reference binary's; the reported angle is within a few ulp (it comes from the device's acos, the reference's from glibc's
 * acosf). */
int mkb_ring_pairs_count(mkb_handle_t h, void *stream, int32_t mode, const mkb_traj *t, const uint32_t *rings_atoms,
                         const uint32_t *starts1, int64_t n_rings1, const uint32_t *second, int64_t n_second, float p0,
                         float p1, float p2, float p3, int64_t *row_offsets, int64_t *total_pairs);
int mkb_ring_pairs_fill(mkb_handle_t h, void *stream, int32_t mode, const mkb_traj *t, const uint32_t *rings_atoms,
                        const uint32_t *starts1, int64_t n_rings1, const uint32_t *second, int64_t n_second, float p0,
                        float p1, float p2, float p3, const int64_t *row_offsets, int32_t *pairs, float *distangles);

/* K14: superposition of trajectory frames, replaces the frame loop of _pp_align / _pp_measure_fit (moleculekit/align.py,
 * called from Molecule.align) and util.molRMSD.  frames [n_frames] int64 device: the frames of t to process (indexes into
 * the view t, so a frame shard works as for K3); entry i of transforms / out belongs to frames[i].  sel [n_sel] uint32
 * device; ref float32 device, row j of the selection, dim d, column c at ref[(j*3 + d)*ref_stride + c] (the selected rows,
 * frame-minor like t->coords).  Index ranges are the caller's responsibility.
 * fit  : transforms [n_frames][15] float64 device = R (3x3 row-major), cP, cQ: the proper rotation minimising
 *        sum |(p - cP) R^T + cQ - q|^2 over the selection, p from frame frames[i] of t, q from reference column
 *        matchingframes ? frames[i] : 0.  Centroids and covariance are summed in float64; the rotation is Horn's quaternion
 *        (cyclic Jacobi on the 4x4 key matrix, float64).  It equals the reference's SVD with reflection correction wherever
 *        that is unique (1e-12 relative, not bitwise), and is exactly the identity for a zero covariance (n_sel == 1,
 *        coincident points), where the reference's SVD yields the identity too.
 * apply: every atom of every listed frame of t->coords (MODIFIED IN PLACE): x' = (x - cP) R^T + cQ evaluated in float64
 *        from the float32 input and rounded once to float32.  frames must not repeat.
 * rmsd : out [n_frames] float32 device = sqrt(mean over the selection of |x' - r|^2), summed in float64, where x' is the
 *        float32 value apply would store with transforms[i] (transforms == NULL: the stored coordinate) and r the reference
 *        column ref_frames == 1 ? 0 : frames[i].
 * No atomics: the fit and rmsd sums run in a fixed order that depends only on n_sel and min(32, pow2 >= n_frames), so
 * identical calls return identical bits. */
int mkb_align_fit(mkb_handle_t h, void *stream, const mkb_traj *t, const int64_t *frames, int64_t n_frames,
                  const uint32_t *sel, int64_t n_sel, const float *ref, int64_t ref_stride, int32_t matchingframes,
                  double *transforms);
int mkb_align_apply(mkb_handle_t h, void *stream, const mkb_traj *t, const int64_t *frames, int64_t n_frames,
                    const double *transforms);
int mkb_rmsd(mkb_handle_t h, void *stream, const mkb_traj *t, const int64_t *frames, int64_t n_frames, const uint32_t *sel,
             int64_t n_sel, const float *ref, int64_t ref_stride, int64_t ref_frames, const double *transforms, float *out);

#ifdef __cplusplus
}
#endif
#endif /* MKB200_H */
