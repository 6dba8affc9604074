/*
 * pdbeda_b200.h -- C ABI of libpdbeda_b200.so: pdb_eda's voxel hot path on NVIDIA B200 (sm_100a).
 *
 * This is the drop-in boundary for the reference's only native component, the Cython module
 * pdb_eda/cutils.pyx (bound through `from . import cutils as utils`, pdb_eda/ccp4.py:16-19 and
 * pdb_eda/densityAnalysis.py:26-29).  Every entry point names the reference routine(s) it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types.
 *   - Pointers named d_* are DEVICE pointers owned by the caller (e.g. torch tensors' data_ptr()); the
 *     library never frees them and never allocates behind the caller's back: scratch memory comes from a
 *     caller-supplied workspace whose size is returned by the matching *_workspace_bytes() call.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls only enqueue work;
 *     they do not synchronise unless stated.
 *   - Return value: 0 on success, negative pe_status on failure; pe_last_error() gives the message of the
 *     calling thread's most recent failure.
 *   - Voxel data is the CCP4 mode-2 payload as stored in the file: float32 rho[section][row][column],
 *     column fastest (pdb_eda/ccp4.py:338).  float32 is lossless: the reference's float64 array holds exactly
 *     these values.
 *   - "crs" = (column, row, section) grid indices, "xyz" = orthogonal Angstrom coordinates.
 *   - Canonical voxel order = the reference's itertools.product order: column slowest, section fastest
 *     (pdb_eda/cutils.pyx:199, :241-243).
 */
#ifndef PDBEDA_B200_H
#define PDBEDA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PE_ABI_VERSION 1

typedef enum pe_status {
    PE_OK = 0,
    PE_ERR_ARG = -1,      /* bad argument (null pointer, negative size, unsupported geometry) */
    PE_ERR_CUDA = -2,     /* a CUDA runtime call or launch failed */
    PE_ERR_CAPACITY = -3, /* an output / workspace capacity was too small */
    PE_ERR_NO_DEVICE = -4 /* no CUDA device / not a Blackwell (sm_100) device */
} pe_status;

/* Cell geometry, computed on the host from the 56 header words exactly as DensityHeader.__init__ does
 * (pdb_eda/ccp4.py:158-286).  All arrays of 3 are indexed by crs axis (0 = column, 1 = row, 2 = section)
 * or by xyz axis as noted. */
typedef struct pe_geom {
    int32_t ncrs[3];         /* stored columns, rows, sections (header words 1-3) */
    int32_t crs_start[3];    /* first column, row, section (words 5-7) */
    int32_t xyz_interval[3]; /* sampling intervals along x, y, z (words 8-10) */
    int32_t crs_interval[3]; /* the same, re-indexed by crs axis (pdb_eda/ccp4.py:237) */
    int32_t unique_ncrs[3];  /* min(ncrs, interval) per crs axis: the non-repeating part (pdb_eda/ccp4.py:262-269) */
    int32_t map2xyz[3];      /* xyz axis i is carried by crs axis map2xyz[i] (pdb_eda/ccp4.py:230-234) */
    int32_t map2crs[3];      /* crs axis a carries xyz axis map2crs[a] (pdb_eda/ccp4.py:235) */
    int32_t orthogonal;      /* 1 iff alpha == beta == gamma == 90 exactly (pdb_eda/ccp4.py:297, :313) */
    int32_t mv_perm[3];      /* accumulation order of the host BLAS's 3x3 mat-vec behind np.dot ... */
    int32_t mv_fma;          /* ... and whether it fuses multiply-add (probed at start-up, SURVEY.md A.13) */
    double grid_length[3];   /* cell edge / interval per xyz axis (pdb_eda/ccp4.py:228) */
    double origin[3];        /* xyz of voxel (0,0,0) (pdb_eda/ccp4.py:272-286) */
    double ortho[9];         /* orthogonalisation matrix, row major (pdb_eda/ccp4.py:248-250) */
    double deortho[9];       /* its inverse with |x| < 1e-10 zeroed (pdb_eda/ccp4.py:252-253) */
} pe_geom;

/* ---------------------------------------------------------------- library ---------------------------------- */
int pe_abi_version(void);
const char *pe_last_error(void);
/* Fills sm_count / cc_major / cc_minor of the current device; PE_ERR_NO_DEVICE when there is none. */
int pe_device_info(int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor);

/* Launch accounting.  pe_launch_count: kernels launched by this library since load.  While profiling is enabled
 * every launch is bracketed by CUDA events on its stream; pe_profile_entries() synchronises, folds them and returns
 * the number of distinct kernels seen since the last reset; pe_profile_get(i) gives kernel name, launch count and
 * total device milliseconds.  (No counterpart in the reference; used by bench.py for the roofline line.) */
long long pe_launch_count(void);
void pe_profile_enable(int on);
void pe_profile_reset(void);
int pe_profile_entries(void);
int pe_profile_get(int index, const char **name, long long *count, double *total_ms);

/* SM partition of device `device` (CUDA green contexts): blob_sms SMs with *stream_blob on them, the device's other SMs with
 * *stream_rest; both are non-blocking streams.  Kernels enqueued on one run only on its SMs, so two passes limited by different
 * resources overlap at their full per-SM occupancy.  Every entry point sizes its resident grids (persistent and cooperative
 * kernels) by the SMs of the stream it launches on.  *sms_blob / *sms_rest: the SM counts provisioned.  PE_ERR_ARG for null
 * pointers or a count the driver does not split exactly (from compute capability 9.0 on: a multiple of 8, below the device's
 * SM count), PE_ERR_NO_DEVICE without a device, PE_ERR_CUDA when the driver has no green contexts or refuses; nothing is
 * left behind on failure.  pe_sm_partition_destroy synchronises both streams, then releases streams and contexts. */
int pe_sm_partition_create(int32_t device, int32_t blob_sms, void **stream_blob, void **stream_rest, int32_t *sms_blob,
                           int32_t *sms_rest);
int pe_sm_partition_destroy(void *stream_blob, void *stream_rest);

/* ---------------------------------------------------------------- map statistics --------------------------- */
/* DensityMatrix.meanDensity / stdDensity (pdb_eda/ccp4.py:343-363): population mean and standard deviation of
 * all n stored voxels in float64.  d_out[0] = mean, d_out[1] = std.  d_ws: >= pe_stats_workspace_bytes(). */
int64_t pe_stats_workspace_bytes(void);
int pe_map_mean_std(const float *d_rho, int64_t n, double *d_out, void *d_ws, void *stream);
/* sumOfAbs (pdb_eda/cutils.pyx:28-39) as used by DensityMatrix.getTotalAbsDensity (pdb_eda/ccp4.py:365-376):
 * d_out[0] = sum of |rho| over voxels with |rho| > (double)cutoff. */
int pe_map_sum_abs(const float *d_rho, int64_t n, float cutoff, double *d_out, void *d_ws, void *stream);
/* The same over a float64 array (sumOfAbs accepts any iterable of numbers). */
int pe_sum_abs_f64(const double *d_values, int64_t n, float cutoff, double *d_out, void *d_ws, void *stream);

/* ---------------------------------------------------------------- point lookups ---------------------------- */
/* getPointDensityFromCrs / testValidCrs (pdb_eda/cutils.pyx:125-167), batched.  d_crs: n x 3 int32 un-wrapped
 * indices.  d_rho_out[i] = wrapped density (0 where the cell is not covered), d_valid[i] = testValidCrs.
 * Either output may be NULL. */
int pe_point_density(const pe_geom *g, const float *d_rho, int64_t n, const int32_t *d_crs, float *d_rho_out,
                     uint8_t *d_valid, void *stream);
/* DensityHeader.xyz2crsCoord (pdb_eda/ccp4.py:288-302), batched: d_xyz n x 3 float64 -> d_crs n x 3 int32. */
int pe_xyz2crs(const pe_geom *g, int64_t n, const double *d_xyz, int32_t *d_crs, void *stream);
/* DensityHeader.crs2xyzCoord (pdb_eda/ccp4.py:304-316), batched. */
int pe_crs2xyz(const pe_geom *g, int64_t n, const int32_t *d_crs, double *d_xyz, void *stream);

/* ---------------------------------------------------------------- atom spheres ----------------------------- */
/* One warp per atom.  An atom's candidates are the reference's box range(c-R-1, c+R+1)^3 with
 * R = xyz2crsCoord(origin + [r,r,r]) (pdb_eda/cutils.pyx:238-243); a voxel belongs to the sphere iff
 * sqrt(dx^2+dy^2+dz^2) <= (double)(float)r evaluated in float64 without contraction (pdb_eda/cutils.pyx:218),
 * decided here by the equivalent test dx^2+dy^2+dz^2 <= T(r), T(r) = largest double whose correctly rounded
 * square root is <= r.  Densities come from the periodic-wrapped lookup (pdb_eda/cutils.pyx:136-145).
 *
 * Atoms are given as d_xyz (n x 3 float64; Biopython's float32 coordinates widened exactly) and d_radius
 * (n float32, the Cython `float radius`).  Atoms may be grouped (d_group_start: n_groups+1 int32 CSR offsets
 * into the atom arrays, or NULL for one group per atom): inside a group a voxel is counted once, for the first
 * atom of the group whose sphere holds it -- the set-union semantics of getSphereCrsFromXyzList
 * (pdb_eda/cutils.pyx:250-271).
 *
 * pe_sphere_sums writes, per group, PE_SPHERE_NOUT float64 values (d_out: n_groups x PE_SPHERE_NOUT):
 *   [0] number of voxels in the (union of) sphere(s)              len(getSphereCrsFromXyz(..., 0))
 *   [1] sum of their densities                                    getTotalDensityFromXyz(..., 0)
 *   [2] number with rho > cut_pos   (0 < cut_pos; skipped when cut_pos == 0)
 *   [3] sum of those densities      findAberrantBlobs(+cutoff) total (pdb_eda/densityAnalysis.py:1060-1061,:1183)
 *   [4] number with rho < cut_neg   (cut_neg < 0; skipped when cut_neg == 0)
 *   [5] sum of those densities      findAberrantBlobs(-cutoff) total (pdb_eda/densityAnalysis.py:1184)
 *   [6] 1.0 iff every in-sphere voxel lies inside the stored map   testValidXyzList (pdb_eda/cutils.pyx:273-313)
 *   [7] number of box candidates examined (for throughput accounting)
 * d_ws: >= pe_sphere_workspace_bytes(n_atoms) bytes. */
#define PE_SPHERE_NOUT 8
int64_t pe_sphere_workspace_bytes(int64_t n_atoms);
/* Diagnostic: warp cycles of the grouped (union) kernel by phase -- boxes + bounding box, tile offsets + per-atom tables,
 * membership, gather, reduction + output -- summed over all warps since the last call; synchronises and resets.  All zeros
 * unless the library was built with -DPE_UNION_PHASE_CYCLES=1 (the counters cost the kernel registers). */
int pe_sphere_union_warp_cycles(unsigned long long *out5);
int pe_sphere_sums(const pe_geom *g, const float *d_rho, int32_t n_atoms, const double *d_xyz,
                   const float *d_radius, int32_t n_groups, const int32_t *d_group_start, float cut_pos,
                   float cut_neg, double *d_out, void *d_ws, void *stream);
/* The per-atom and the grouped sums of the same atoms in one call: the results equal those of
 *   pe_sphere_sums(g, d_rho, n_atoms, d_xyz, d_atom_radius, n_atoms, NULL, cut_pos, cut_neg, d_out_atoms, d_ws, stream) and
 *   pe_sphere_sums(g, d_rho, n_atoms, d_xyz, d_group_radius, n_groups, d_group_start, cut_pos, cut_neg, d_out_groups, d_ws, stream),
 * bit for bit, with the same argument checks and status codes and the same workspace (pe_sphere_workspace_bytes(n_atoms)).
 * When the cell is orthogonal and every per-atom box at max_atom_radius is at most 8 voxels wide (the atom-type radii of the
 * cloud pass on a 0.5 A grid), the per-atom sums run as short work items at the end of the grouped kernel: one launch instead
 * of two, and the per-atom work fills the SMs that the last groups leave idle.  Otherwise the call issues the two launches.
 * max_atom_radius is the largest value of d_atom_radius (any larger bound also does; the host cannot read the device array
 * without a synchronisation); an atom whose radius exceeds it gets NaN rows instead of sums. */
int pe_sphere_sums_atoms_and_groups(const pe_geom *g, const float *d_rho, int32_t n_atoms, const double *d_xyz,
                                    const float *d_atom_radius, float max_atom_radius, const float *d_group_radius,
                                    int32_t n_groups, const int32_t *d_group_start, float cut_pos, float cut_neg,
                                    double *d_out_atoms, double *d_out_groups, void *d_ws, void *stream);

/* pe_sphere_sums for the atoms of many structures, each on its own map, in one launch (the region density / discrepancy of a
 * whole batch).  d_maps (device array, n_maps entries): per structure its geometry, the device pointer of its map and its own
 * cutoffs (cut_pos >= 0 >= cut_neg; the caller checks them where it builds the table, an entry that breaks the rule gives NaN
 * rows).  Structure k owns the atoms d_atom_start[k] .. d_atom_start[k+1] (n_maps + 1 offsets; d_xyz n_atoms x 3 float64,
 * d_radius n_atoms float32).  Group g is summed on map d_group_map[g]:
 *   grouped   (d_group_start given): group g is the set-union of the atoms d_group_start[g] .. d_group_start[g+1], one warp
 *             per group as in pe_sphere_sums; d_atom_start may be NULL;
 *   per atom  (d_group_start NULL, n_groups == n_atoms): group a is atom a; atoms are taken four at a time from each
 *             structure's first atom, so a quad never spans two structures.
 * d_out (n_groups x PE_SPHERE_NOUT) holds the values documented for pe_sphere_sums.  Every row is bit-identical to the row
 * pe_sphere_sums gives for the same structure alone (its geometry, map, cutoffs, atoms and group offsets) when the atoms of
 * each structure name one map; it does not depend on the other structures of the call.  A group whose map index is outside
 * [0, n_maps) gives a NaN row.  d_ws: >= pe_batch_sphere_sums_workspace_bytes(n_atoms) bytes. */
typedef struct pe_sums_map {
    pe_geom geom;
    const float *d_rho;
    float cut_pos;
    float cut_neg;
} pe_sums_map;
int64_t pe_batch_sphere_sums_workspace_bytes(int64_t n_atoms);
int pe_batch_sphere_sums(int32_t n_maps, const pe_sums_map *d_maps, int32_t n_atoms, const double *d_xyz, const float *d_radius,
                         int32_t n_groups, const int32_t *d_group_map, const int32_t *d_group_start, const int32_t *d_atom_start,
                         double *d_out, void *d_ws, void *stream);

/* getSphereCrsFromXyz (pdb_eda/cutils.pyx:220-248), batched, as lists.  Two calls:
 *   pe_sphere_count: d_count[a] = len(getSphereCrsFromXyz(dm, xyz[a], radius[a], cutoff)), and
 *                    d_box[a*6 ..] = box low corner (c, r, s) and box extents (nc, nr, ns);
 *   pe_sphere_fill : with d_offset = exclusive prefix sum of d_count (n_atoms+1 entries, int64), writes for
 *                    atom a its voxels in the reference's order (column slowest, section fastest) to
 *                    d_index[d_offset[a] ..]: the voxel's position inside the box in that same order,
 *                    i.e. crs = low + (p / (nr*ns), (p / ns) % nr, p % ns).  Optional per-voxel outputs
 *                    (NULL to skip): d_value = wrapped density; d_label = number of the voxel's 26-connected
 *                    cluster inside this atom's list, numbered in the order createCrsLists creates them
 *                    (pdb_eda/cutils.pyx:44-70) -- this is findAberrantBlobs(atom) (pdb_eda/ccp4.py:437-461).
 * cutoff follows pdb_eda/cutils.pyx:245: > 0 keeps rho > cutoff, < 0 keeps rho < cutoff, 0 keeps all.
 * max_box_voxels bounds nc*nr*ns over the batch (host knows the radii); it sizes shared memory. */
int pe_sphere_count(const pe_geom *g, const float *d_rho, int32_t n_atoms, const double *d_xyz,
                    const float *d_radius, float cutoff, int32_t *d_count, int32_t *d_box, void *stream);
int pe_sphere_fill(const pe_geom *g, const float *d_rho, int32_t n_atoms, const double *d_xyz,
                   const float *d_radius, float cutoff, const int64_t *d_offset, int32_t max_box_voxels,
                   int32_t *d_index, float *d_value, int32_t *d_label, void *stream);

/* ---------------------------------------------------------------- difference-map blobs --------------------- */
/* createFullBlobList (pdb_eda/ccp4.py:463-485) = createFullCrsList (pdb_eda/cutils.pyx:185-203) +
 * createCrsLists (:41-70) + DensityBlob.fromCrsList (pdb_eda/ccp4.py:522-545), for the positive and the negative
 * cutoff in ONE pass over the map (greenBlobList + redBlobList, pdb_eda/densityAnalysis.py:392-412).
 *
 * Class 0 ("green"): rho >= cut_pos (cut_pos > 0).  Class 1 ("red"): rho <= cut_neg (cut_neg < 0).  A class whose
 * cutoff is 0 is skipped (createFullCrsList returns None).  Only the unique sub-volume unique_ncrs is scanned;
 * adjacency is 26-connectivity WITHOUT periodic wrap.
 *
 * Outputs, per class k (all device pointers; capacity `cap_voxels` foreground voxels and `cap_blobs` blobs per class):
 *   d_counts[k*2+0] = number of foreground voxels, d_counts[k*2+1] = number of blobs   (int64, 4 entries)
 *   d_counts[4]     = failure flag (1: a capacity was exceeded -- call again with larger ones; 2: the labelling kernel's blocks
 *                     were not spread evenly over the SMs, part of the map was not scanned; either way results are invalid)
 *   d_key  [k*cap_voxels + p] = canonical index (c*U1 + r)*U2 + s of the p-th foreground voxel, ascending:
 *                               exactly createFullCrsList's list
 *   d_value[k*cap_voxels + p] = its density
 *   d_label[k*cap_voxels + p] = its blob number; blobs are numbered by their smallest canonical member,
 *                               which is the order createCrsLists returns them in
 *   d_stats[(k*cap_blobs + b)*8 ..] = n, sum rho, sum rho*x, sum rho*y, sum rho*z, sum x, sum y, sum z  (float64)
 * d_ws: >= pe_blob_workspace_bytes(g, cap_voxels) bytes. */
int64_t pe_blob_workspace_bytes(const pe_geom *g, int64_t cap_voxels);
/* Diagnostic: device timestamps (ns) at the stage boundaries of the most recent sparse-stage kernel
 * (start, after each of its grid barriers, end); synchronises. */
int pe_blob_stage_times(unsigned long long *out12);
int pe_blob_label(const pe_geom *g, const float *d_rho, float cut_pos, float cut_neg, int64_t cap_voxels,
                  int64_t cap_blobs, int64_t *d_counts, uint32_t *d_key, float *d_value, int32_t *d_label,
                  double *d_stats, void *d_ws, void *stream);

/* ---------------------------------------------------------------- slab-decomposed blob labelling ----------- */
/* One very large map cut into slabs along the section axis (the slowest axis in memory, pdb_eda/ccp4.py:338), one slab per
 * GPU.  The reference cannot run such maps at all (Python float per voxel, N x N cdist: pdb_eda/ccp4.py:123-124,
 * pdb_eda/cutils.pyx:55); the result reproduced is the whole map's createFullBlobList (pdb_eda/ccp4.py:463-485).
 * Every rank labels its slab [s0, s1) with pe_blob_label (geometry = the map's with ncrs[2] / unique_ncrs[2] = the slab's
 * section counts), then:
 *   pe_slab_boundary  fills this rank's exchange buffer (pe_slab_exchange_bytes(cap_blobs, cap_plane) bytes): per sign the
 *                     local blob count, every blob's smallest key in the WHOLE map's canonical order and the (column, row,
 *                     blob) voxels of the slab's first and last section (last_is_cut = 0 for the top slab);
 *   the caller all-gathers the world's buffers into d_gathered (rank-major) -- the halo exchange;
 *   pe_slab_merge     26-adjacency across every cut -> union-find over all ranks' blobs -> d_new_number[k*cap_blobs + b] =
 *                     the whole-map blob number of this rank's local blob b of sign k, d_n_merged[k] = blobs of the whole map;
 *   pe_slab_relabel   rewrites d_label in place and accumulates this rank's part of the per-blob sums (layout of
 *                     pe_blob_label's d_stats, cap_merged rows per sign) with the whole map's geometry; the caller
 *                     all-reduces the table.
 * d_ws: >= pe_slab_workspace_bytes(world, cap_blobs, u0, u1), shared by the three calls; pe_slab_status reads its overflow
 * flag (synchronises).
 * cap_blobs and cap_plane set the layout of the exchange buffers and must be the SAME on every rank (size them from the largest
 * slab).  pe_slab_boundary stamps them into each buffer; pe_slab_merge sets the flag when any rank's buffer carries another
 * stamp or counts beyond them (also when that rank's pe_blob_label or boundary overflowed), and then merges nothing, so every
 * rank sees the failure.  cap_blobs < 2^31, cap_plane < 2^32.
 * Size limits: one SLAB holds fewer than 2^31 stored voxels (32-bit element offsets and keys inside a call); the WHOLE map may
 * be larger -- its keys are 64-bit and g_whole is used for index -> coordinate arithmetic only -- so maps beyond the 1290^3 that
 * one pe_blob_label call takes (1536^3, 2048^3 ...) are labelled slab by slab, on several GPUs or one after another on one. */
int64_t pe_slab_exchange_bytes(int64_t cap_blobs, int64_t cap_plane);
int64_t pe_slab_workspace_bytes(int32_t world, int64_t cap_blobs, int32_t u0, int32_t u1);
int pe_slab_boundary(const pe_geom *g_slab, int32_t u2_whole, int32_t s0, int32_t last_is_cut, const int64_t *d_counts,
                     int64_t cap_voxels, const uint32_t *d_key, const int32_t *d_label, int64_t cap_blobs, int64_t cap_plane,
                     void *d_exchange, void *d_ws, void *stream);
int pe_slab_merge(int32_t world, int32_t rank, const void *d_gathered, int64_t cap_blobs, int64_t cap_plane, int32_t u0,
                  int32_t u1, int32_t *d_new_number, int64_t *d_n_merged, void *d_ws, void *stream);
int pe_slab_relabel(const pe_geom *g_whole, int32_t u2_slab, int32_t s0, const int64_t *d_counts, int64_t cap_voxels,
                    const uint32_t *d_key, const float *d_value, int32_t *d_label, int64_t cap_blobs,
                    const int32_t *d_new_number, const int64_t *d_n_merged, int64_t cap_merged, double *d_stats, void *d_ws,
                    void *stream);
int pe_slab_status(const void *d_ws, void *stream, int32_t *bad);

/* ---------------------------------------------------------------- voxel-list set algebra ------------------- */
/* createCrsLists (pdb_eda/cutils.pyx:41-70) on an arbitrary list of n un-wrapped voxels (d_crs n x 3 int32):
 * d_label[i] = cluster number in the reference's creation order (by first unused input index).
 * d_nclusters: TWO int64: [0] = number of clusters, [1] = non-zero when an index was outside the key range
 * (|index| < 2^20, i.e. -1048575 .. 1048575, without groups; |index| < 2^13, i.e. -8191 .. 8191, and
 * 0 <= group < 2^22 with groups) and the result is invalid.
 * The grouped form clusters every group (d_group[i] >= 0, e.g. the residue a cloud voxel belongs to) on its own
 * -- the residue-cloud merging of aggregateCloud (pdb_eda/densityAnalysis.py:646-677) -- and tolerates repeated
 * voxels: d_first[i] (optional) = 1 iff i is the first entry holding its (group, voxel), which is what turns the
 * list into the SET DensityBlob.merge builds (pdb_eda/ccp4.py:575-586).  d_group may be NULL (one group).
 * d_ws: >= pe_cluster_workspace_bytes(n). */
int64_t pe_cluster_workspace_bytes(int64_t n);
int pe_cluster_crs(int64_t n, const int32_t *d_crs, int32_t *d_label, int64_t *d_nclusters, void *d_ws,
                   void *stream);
int pe_cluster_crs_grouped(int64_t n, const int32_t *d_crs, const int32_t *d_group, int32_t *d_label,
                           uint8_t *d_first, int64_t *d_nclusters, void *d_ws, void *stream);

/* DensityBlob.fromCrsList (pdb_eda/ccp4.py:522-545) for every cluster of a labelled voxel list at once:
 * d_stats[b*8 ..] = n, sum rho, sum rho*x, sum rho*y, sum rho*z, sum x, sum y, sum z over the entries with
 * d_label[i] == b (d_label NULL: one cluster) and d_take[i] != 0 (d_take NULL: all).  rho is the wrapped lookup
 * (pdb_eda/cutils.pyx:125-145), xyz = crs2xyzCoord of the un-wrapped index (pdb_eda/ccp4.py:304-316). */
int pe_crs_stats(const pe_geom *g, const float *d_rho, int64_t n, const int32_t *d_crs, const int32_t *d_label,
                 const uint8_t *d_take, int64_t n_clusters, double *d_stats, void *stream);

/* calculateRsccRsrMetrics (pdb_eda/densityAnalysis.py:860-882) for every group of a labelled voxel list at once, on the
 * Fo map (d_rho_fo = 2Fo-Fc) and the Fc map formed on the fly as fo - 2 * diff in float64 (pdb_eda/densityAnalysis.py:433):
 * d_out[g*8 ..] = n, sum fo, sum fc, sum |fo - fc|, sum |fo + fc|, sum (fo-mean)^2, sum (fc-mean)^2, sum (fo-mean)(fc-mean).
 * RSCC = out[7] / sqrt(out[5] * out[6]), RSR = out[3] / out[4].  Entries with d_take[i] == 0 are skipped. */
int pe_pair_metrics(const pe_geom *g, const float *d_rho_fo, const float *d_rho_diff, int64_t n, const int32_t *d_crs,
                    const int32_t *d_label, const uint8_t *d_take, int64_t n_groups, double *d_out, void *stream);

/* calculateRsccRsrMetrics over the set-union of a group's atom spheres (getSphereCrsFromXyzList, pdb_eda/cutils.pyx:250-271:
 * the reference's box and predicate, float32 radius, un-wrapped indices, a repeated voxel counted once) for the groups of many
 * structures at once -- residueMetrics / atomMetrics (pdb_eda/densityAnalysis.py:803-858) of a whole batch.
 * d_maps (device array, n_maps entries): per structure the geometry and the device pointers of its 2Fo-Fc map (d_fo) and its
 * Fo-Fc map (d_diff) on the same grid; fewer than 2^31 stored voxels per map.  Group g is made of the atoms
 * d_group_start[g] .. d_group_start[g+1] (d_xyz n x 3 float64, d_radius n float32) on map d_group_map[g].
 * d_out[g*8 ..] = the eight sums of pe_pair_metrics over the group's voxel set: n, sum fo, sum fc, sum |fo - fc|,
 * sum |fo + fc|, sum (fo-mean)^2, sum (fc-mean)^2, sum (fo-mean)(fc-mean), with fc = fo - 2 * diff in float64, voxels the map
 * does not cover counted with fo = fc = 0 and the moments centred on the group's own means (two passes).  An empty group
 * gives a zero row, a group whose d_group_map entry is outside [0, n_maps) a NaN row.  The summation order is fixed:
 * results are bit-identical from run to run and do not depend on the other groups of the call.
 * d_ws: >= pe_pair_union_workspace_bytes(n_atoms). */
typedef struct pe_pair_map {
    pe_geom geom;
    const float *d_fo;
    const float *d_diff;
} pe_pair_map;
int64_t pe_pair_union_workspace_bytes(int32_t n_atoms);
int pe_pair_union_metrics(int32_t n_maps, const pe_pair_map *d_maps, int32_t n_groups, const int32_t *d_group_map,
                          const int32_t *d_group_start, const double *d_xyz, const float *d_radius, double *d_out, void *d_ws,
                          void *stream);

/* testOverlap (pdb_eda/cutils.pyx:8-25), all pairs at once: every entry is a voxel of the blob d_owner[i]; two
 * blobs overlap iff some voxel of one is identical or 26-adjacent to some voxel of the other (same group when
 * d_group is given).  Writes each overlapping unordered pair once as (smaller owner, larger owner) to d_pairs
 * (cap_pairs x 2 int32, unordered); d_npairs: TWO int64: [0] = number of pairs found (re-run with a larger
 * cap_pairs when it exceeds it), [1] = key-range overflow flag as above.  d_pairs is complete only when
 * d_npairs[0] <= cap_pairs; otherwise [0] is an upper bound and d_pairs holds some true pairs (possibly none, and
 * not necessarily in its first rows).
 * This is the overlap matrix of pdb_eda/densityAnalysis.py:646-649 and :689-692 in sparse form.
 * d_ws: >= pe_overlap_workspace_bytes(n, cap_pairs). */
int64_t pe_overlap_workspace_bytes(int64_t n, int64_t cap_pairs);
int pe_overlap_pairs(int64_t n, const int32_t *d_crs, const int32_t *d_owner, const int32_t *d_group,
                     int64_t cap_pairs, int64_t *d_npairs, int32_t *d_pairs, void *d_ws, void *stream);

/* ---------------------------------------------------------------- batched cloud aggregation ---------------- */
/* DensityAnalysis.aggregateCloud (pdb_eda/densityAnalysis.py:571-729) for a batch of structures at once: the unit of
 * work of multiple-structures mode (analyzePDBID, pdb_eda/multipleStructures.py:320-356) and of the optimiser's inner
 * loop (processFunction, pdb_eda/optimizeParams.py:410-448).
 *
 * d_maps (device array, n_maps entries): one 2Fo-Fc map per structure -- geometry, device pointer to its voxels, the
 * float32-narrowed densityCutoff (pdb_eda/densityAnalysis.py:131, SURVEY.md App. A.1) and the range of its atoms in the
 * batch arrays.  Atoms (the candidates of pdb_eda/densityAnalysis.py:596-603, in traversal order, structure by structure):
 *   d_atom_map[a]       structure index
 *   d_xyz[a*3..]        float64 coordinates (Biopython's float32 widened exactly), d_radius[a] float32 atom-type radius
 *   d_atom_residue[a]   residue id, unique over the batch; d_atom_local[a] index of the atom inside its residue (< 64)
 *   d_atom_bonded[a]    bit mask of the in-residue indices of its bonded atoms (bonded_atoms table)
 *   d_atom_electrons[a] electrons * occupancy
 *
 * pe_cloud_count:  d_offset (n_atoms + 1 uint32) = exclusive prefix sum of every atom's number of cloud voxels
 *                  (len(getSphereCrsFromXyz(dm, xyz, r, cutoff))); d_totals[0] = total, d_totals[1] = largest candidate box.
 *                  d_scan_ws: >= 256 + 4 * (n_atoms / 1024 + 2) bytes.  d_box_bits (may be NULL; 8 uint32 per atom): the count
 *                  pass leaves the membership bitmap of every candidate box of at most 256 voxels there, and pe_cloud_aggregate,
 *                  given the same pointer, starts from it instead of enumerating the spheres a second time.
 * pe_cloud_aggregate (n_entries = d_totals[0], max_box_voxels = d_totals[1]) writes
 *   d_atom_out[a*8..]  number of clouds, voxels of the best (nearest-centroid) cloud, its centroid distance, its total
 *                      density, its centroid x y z, flags (0: does not contribute, 1: contributes, 3: contributes and is
 *                      completely overlapped, pdb_eda/densityAnalysis.py:623-659)
 *   d_map_out[m*8..]   numVoxelsAggregated, totalAggregatedDensity, totalAggregatedElectrons, domain clouds, domain clouds
 *                      with >= min_cloud_electrons, residue clouds, residue clouds with >= min_cloud_electrons,
 *                      centroidDistanceCutoff (pdb_eda/densityAnalysis.py:609, :681, :712-724)
 * d_ws: >= pe_cloud_workspace_bytes(n_atoms, n_entries, n_residues, n_maps).  pe_cloud_status reads the workspace's error flag
 * (un-wrapped index outside +-8190 or inconsistent counts) and synchronises. */
typedef struct pe_batch_map {
    pe_geom geom;
    const float *d_rho;
    float cutoff;
    int32_t atom_begin, atom_end;
    int32_t reserved;
} pe_batch_map;
int64_t pe_cloud_workspace_bytes(int64_t n_atoms, int64_t n_entries, int64_t n_residues, int64_t n_maps);
int pe_cloud_count(int32_t n_maps, const pe_batch_map *d_maps, int32_t n_atoms, const int32_t *d_atom_map, const double *d_xyz,
                   const float *d_radius, uint32_t *d_offset, int64_t *d_totals, void *d_scan_ws, uint32_t *d_box_bits, void *stream);
int pe_cloud_aggregate(int32_t n_maps, const pe_batch_map *d_maps, int32_t n_atoms, const int32_t *d_atom_map,
                       const double *d_xyz, const float *d_radius, const int32_t *d_atom_residue,
                       const int32_t *d_atom_local, const uint64_t *d_atom_bonded, const double *d_atom_electrons,
                       int32_t n_residues, const uint32_t *d_offset, int64_t n_entries, int32_t max_box_voxels,
                       double min_cloud_electrons, const uint32_t *d_box_bits, double *d_atom_out, double *d_map_out, void *d_ws,
                       void *stream);
int pe_cloud_status(const void *d_ws, void *stream, int32_t *bad);
/* The per-atom-type statistics block of aggregateCloud (pdb_eda/densityAnalysis.py:734-766) for every structure of a batch,
 * from the outputs of pe_cloud_aggregate: the second centroid filter (:746-748), then per (structure, atom type) the medians of
 * num_voxels, density_electron_ratio, centroid_distance, adj_density_electron_ratio, volume, bfactor (> 0), the b-factor slope
 * (scipy.stats.linregress with its p-value test, :729-733), domain_fraction, corrected_fraction and
 * corrected_density_electron_ratio.  d_perm lists the batch's atoms structure by structure and, inside a structure, atom type
 * by atom type; segment s (d_seg_begin[s] .. d_seg_end[s] into d_perm, at most max_segment long) holds the atoms of type
 * d_seg_type[s] of structure d_seg_map[s].  d_atom_static: n_atoms x 3 (electrons, occupancy, bfactor).
 * Outputs: d_seg_out[s*14..] = kept rows, the ten values above in that order, contributing atoms of the type, those completely
 * overlapped (pdb_eda/densityAnalysis.py:653-659), spare; d_map_stats[m*4..] = atoms analysed (len(atomCloudDescriptions)),
 * densityElectronRatio (NaN below min_total_electrons, :726), the centroid cutoff, ok flag.  d_scratch: 9 x n_atoms float64. */
int pe_cloud_statistics(int32_t n_maps, const pe_batch_map *d_maps, int32_t n_atoms, const double *d_atom_out,
                        const double *d_map_out, const double *d_atom_static, const int32_t *d_perm, int32_t n_segments,
                        const int32_t *d_seg_map, const int32_t *d_seg_type, const int32_t *d_seg_begin,
                        const int32_t *d_seg_end, int32_t max_segment, const double *d_unit_volume,
                        const double *d_current_slopes, double min_total_electrons, double *d_scratch, double *d_seg_out,
                        double *d_map_stats, void *stream);

/* ---------------------------------------------------------------- symmetry atoms --------------------------- */
/* createSymmetryAtoms (pdb_eda/cutils.pyx:73-103).  d_xyz: n_atoms x 3 float64; d_rot: n_ops x 12 float64
 * (REMARK 290 3x4 operators, pdb_eda/pdbParser.py:71-77); d_shift: 27 x 3 float64, the lattice translations
 * np.dot(orthoMat, (i,j,k)) with i slowest, formed by the caller; lo/hi (host pointers, 3 doubles each): the
 * circumscribed box already widened by 5 A (pdb_eda/cutils.pyx:101; pdb_eda/densityAnalysis.py:899-903).
 * Kept images are written in the reference's order -- (i,j,k,op) lexicographic, then atom order -- as
 * d_atom[m] (atom index), d_image[m] (= ((i+1)*9 + (j+1)*3 + (k+1))*n_ops + op) and d_out_xyz[m*3..].
 * d_count[0] = number kept (int64); when it exceeds `cap` only the first cap are written and the call still
 * returns PE_OK (re-run with a larger cap).  d_ws: >= pe_symmetry_workspace_bytes(n_atoms, n_ops). */
int64_t pe_symmetry_workspace_bytes(int32_t n_atoms, int32_t n_ops);
int pe_symmetry_expand(const pe_geom *g, int32_t n_atoms, const double *d_xyz, int32_t n_ops, const double *d_rot,
                       const double *d_shift, const double *lo, const double *hi, int64_t cap, int64_t *d_count,
                       int32_t *d_atom, int32_t *d_image, double *d_out_xyz, void *d_ws, void *stream);

/* ---------------------------------------------------------------- atom-to-blob distances ------------------- */
/* The inner loop of calculateAtomSpecificBlobStatistics (pdb_eda/densityAnalysis.py:932-937): for each blob
 * centroid the first nearest of n_atoms coordinates under scipy's euclidean cdist, in float64.
 * d_centroid: n_blobs x 3, d_coords: n_atoms x 3; d_idx[b] = np.argmin index, d_dist[b] = the distance. */
int pe_nearest_atom(int64_t n_blobs, const double *d_centroid, int64_t n_atoms, const double *d_coords,
                    int32_t *d_idx, double *d_dist, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PDBEDA_B200_H */
