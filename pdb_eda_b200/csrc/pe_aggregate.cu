// pe_aggregate.cu -- cloud aggregation (DensityAnalysis.aggregateCloud, pdb_eda/densityAnalysis.py:571-729) for a BATCH of
// structures in one sequence of launches: the unit of multiple-structures mode (analyzePDBID,
// pdb_eda/multipleStructures.py:320-356) and of the optimiser's inner loop (processFunction,
// pdb_eda/optimizeParams.py:410-448).
//
// What the reference does per structure, and what runs here for all structures of the batch at once:
//   pass 1  every candidate atom's clouds = findAberrantBlobs(atom.coord, radius[type], densityCutoff) (:605):
//           sphere voxels with rho > cutoff, 26-connected clusters, per cloud sum rho / centroid / size; the atom's
//           smallest centroid distance (:608)                                   -> cloud_count_kernel, cloud_fill_kernel
//                                                                                  (8 lanes per atom for boxes of <= 256 voxels)
//           centroidDistanceCutoff = nanmedian + 2.5 nanstd per structure (:609) -> cutoff_kernel (radix select)
//   pass 2  an atom contributes unless it has several clouds and even the nearest centroid is beyond the cutoff
//           (:623-634); all clouds of a contributing atom join its residue's pool (:638-639)   -> accept_kernel
//           residue level: clouds of one residue that touch (testOverlap, pdb_eda/cutils.pyx:8-25) are merged; an atom
//           is "completely overlapped" when it touches every bonded atom of its residue that contributes (:646-659)
//           domain level: residue clouds that touch are merged (:689-708); a merged cloud is a voxel SET, so the
//           totals run over each distinct voxel once and over the distinct atoms of the merged cloud (:712-724)
//                                                      -> pair path: atoms binned into a per-structure cell grid
//                                                         (atom_cell_insert_kernel), one warp per atom tests its neighbours'
//                                                         cloud voxels against byte masks of its own clouds in shared memory
//                                                         (cloud_pair_kernel: two union-finds over cloud ids + per-atom
//                                                         adjacency bits + first flags), cloud_roots_kernel,
//                                                         map_summary_kernel; fallback for batches the pair kernel's frame
//                                                         cannot hold (device flag): one hash table of all pool voxels
//                                                         (pool_insert / cloud_merge / cloud_first_kernel)
// The host keeps the per-atom-type statistics (numpy / scipy, pdb_eda/densityAnalysis.py:734-766), vectorised over the
// batch.  Order-dependent descriptions (which atom names a merged cloud, :717) are not produced here; the single
// structure API (DensityAnalysis.aggregateCloud) replays those with Python sets.
//
// Batch layout: atoms of one structure are contiguous (pe_batch_map::atom_begin/end); every atom carries its structure
// index, a residue id that is unique over the batch, its index inside the residue (< 64) and the bit mask of its bonded
// atoms' indices inside the residue.
#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include "pe_select.cuh"
#include "pe_sphere_dev.cuh"

namespace pe {

constexpr int kAggThreads = 256;
constexpr int kSummaryThreads = 1024;        // kernels with one CTA per structure: the largest structure of a batch sets their duration
constexpr uint64_t kAggEmpty = ~0ull;
constexpr uint32_t kAggNil = 0xffffffffu;
constexpr int kKeyBits = 14;                 // per crs axis, offset 2^13: |index| < 8192
constexpr int kKeyOff = 1 << (kKeyBits - 1);
constexpr int kSmallBox = 8;                 // widest box edge of the 8-lanes-per-atom count path
struct SmallTabB {
    double sq[3][kSmallBox];  // per crs axis: fl((coord - atom)^2) of the box's indices
    int off[3][kSmallBox];    // wrapped element offsets, or kInvalidOff
};
static_assert(kSmallBox * kSmallBox * kSmallBox <= 1024, "magic division by dim[1]");
constexpr int kBoxBitWords = 8;              // candidate boxes of up to 256 voxels hand their bitmap from the count pass to the fill pass
constexpr int kPairClouds = 8;               // clouds per atom the pair kernel's byte masks can name
constexpr int kPairWarps = 4;
constexpr int kPairList = 64;                // (cloud, cloud) pairs a warp collects before it unites them
constexpr int kPairCand = 64;                // candidate atoms a warp collects before it walks their entries

// Hash table of the pool voxels.  Every structure owns a REGION of the slot array (twice its number of cloud voxels), so the
// probes of a thread block -- entries are ordered structure by structure -- stay inside a few megabytes that L2 holds, instead of
// scattering over one table of the whole batch (hundreds of megabytes: every probe a DRAM access).  A slot is 16 bytes (key,
// head of the chain of entries at that voxel), read with one load.
struct AggSlot {
    unsigned long long key;
    uint32_t head;
    uint32_t pad;
};
struct AggTable {
    AggSlot *slot;
    const uint32_t *offset;       // n_atoms + 1: first cloud voxel of every atom
    const pe_batch_map *maps;     // atom ranges of the structures
    uint2 *node;                  // per entry: (next entry of the same voxel, owning atom)
};

__device__ __forceinline__ void agg_region(const AggTable &t, uint64_t key, uint64_t &base, uint32_t &size) {
    const pe_batch_map *m = t.maps + (key >> (3 * kKeyBits));
    const uint64_t e0 = t.offset[m->atom_begin], e1 = t.offset[m->atom_end];
    base = 2 * e0 + 16ull * (key >> (3 * kKeyBits));
    size = (uint32_t)(2 * (e1 - e0) + 16);
}
__device__ __forceinline__ uint32_t agg_start(uint64_t key, uint32_t size) {
    const uint32_t h = (uint32_t)((key * 0x9E3779B97F4A7C15ull) >> 32);
    return (uint32_t)(((uint64_t)h * size) >> 32);
}

__device__ __forceinline__ uint32_t agg_lookup(const AggTable &t, uint64_t key) {
    uint64_t base;
    uint32_t size;
    agg_region(t, key, base, size);
    uint32_t h = agg_start(key, size);
    for (;;) {
        const uint4 s = __ldcg(reinterpret_cast<const uint4 *>(t.slot + base + h));
        const unsigned long long k = ((unsigned long long)s.y << 32) | s.x;
        if (k == key) return s.z;
        if (k == kAggEmpty) return kAggNil;
        h = h + 1 == size ? 0 : h + 1;
    }
}

// per-warp copy of a structure's geometry in shared memory (the device helpers take it by reference)
__device__ __forceinline__ void load_geom(pe_geom *dst, const pe_batch_map *m, int lane) {
    static_assert(sizeof(pe_geom) % 8 == 0 && offsetof(pe_batch_map, geom) == 0, "geometry is copied as 64-bit words");
    const unsigned long long *src = reinterpret_cast<const unsigned long long *>(&m->geom);
    unsigned long long *d = reinterpret_cast<unsigned long long *>(dst);
    for (int k = lane; k < (int)(sizeof(pe_geom) / 8); k += 32) d[k] = src[k];
    __syncwarp();
}

// ------------------------------------------------------------------------------------------------ pass 1: counts
// One atom by one warp (boxes wider than 8 voxels, skewed cells): the candidate box in the reference's product order.
__device__ __forceinline__ void count_one_atom(const pe_batch_map *__restrict__ maps, int a, const int32_t *__restrict__ atom_map,
                                               const double *__restrict__ xyz, const float *__restrict__ radius, uint32_t *__restrict__ count,
                                               unsigned long long *__restrict__ d_maxbox, uint32_t *__restrict__ box_bits, AxisTab *tab,
                                               pe_geom *gs, uint32_t *wb, int lane) {
    const pe_batch_map *m = maps + atom_map[a];
    load_geom(gs, m, lane);
    const pe_geom &g = *gs;
    const float *rho = m->d_rho;
    const float cutoff = m->cutoff;
    const double ax = xyz[3 * a], ay = xyz[3 * a + 1], az = xyz[3 * a + 2];
    AtomBox b;
    double T;
    atom_box(g, ax, ay, az, radius[a], b, T);
    int n = 0;
    // boxes of at most 32 * kBoxBitWords candidates also hand their membership bitmap (the reference's product order) to the
    // fill pass, which then neither enumerates the sphere nor reads the candidates' densities a second time
    const int D1 = b.dim[1], D2 = b.dim[2];
    const bool keep = box_bits != nullptr && b.dim[0] * D1 * D2 <= 32 * kBoxBitWords;
    if (keep) {
        if (lane < kBoxBitWords) wb[lane] = 0u;
        __syncwarp();
    }
    for_each_inside(g, rho, b, ax, ay, az, T, tab, lane, [&](int ic, int ir, int is, bool, float v) {
        if (passes(v, cutoff)) {
            ++n;
            if (keep) {
                const int p = (ic * D1 + ir) * D2 + is;
                atomicOr(&wb[p >> 5], 1u << (p & 31));
            }
        }
    });
    n = warp_sum(n);
    if (keep) {
        __syncwarp();
        if (lane < kBoxBitWords) box_bits[(int64_t)a * kBoxBitWords + lane] = wb[lane];
    }
    if (lane == 0) {
        count[a] = (uint32_t)n;
        const unsigned long long vol = (unsigned long long)b.dim[0] * (unsigned long long)b.dim[1] * (unsigned long long)b.dim[2];
        if (vol > *d_maxbox) atomicMax(d_maxbox, vol);  // a cached (possibly stale, i.e. smaller) value only costs a redundant atomic
    }
    __syncwarp();  // the scratch is reused by the warp's next atom
}

// A warp takes kCountAtoms = 4 consecutive atoms.  At the atom-type radii (0.6 - 1.3 A on a 0.5 A grid) a candidate box is 4^3 or
// 6^3 voxels for ~15 cloud voxels, so when all four boxes are at most 8 wide in an orthogonal cell each atom gets 8 lanes (the
// layout of sphere_sums_kernel, pe_sphere.cu): a lane walks box rows (row, section), finds the row's in-sphere columns exactly
// (row_chord) and gathers just those -- a third of the instructions of one warp per atom (ncu: 1,050 warp instructions per atom,
// issue slots 59 % busy).  Every 8-lane group keeps its own copy of its structure's geometry: a warp's atoms may belong to two
// structures.  Otherwise the warp handles its atoms one after the other with all 32 lanes (count_one_atom).
constexpr int kCountAtoms = 4;
template <int MODE>
__device__ __forceinline__ int count_small_rows(const pe_geom &g, const float *__restrict__ rho, const SmallTabB &t, const int *lo, const int *dim,
                                                double ax, double ay, double az, double T, float cutoff, bool keep, uint32_t *wb, int l8) {
    const int ic = g.map2crs[0];  // xyz axis carried by the columns
    const float inv_gl = (float)(1.0 / g.grid_length[ic]);
    const float xc = (float)((sel3(ax, ay, az, ic) - g.origin[ic]) / g.grid_length[ic] - (double)lo[0]);
    const int nC = dim[0], D1 = dim[1], D2 = dim[2];
    const double *sqc = t.sq[0];
    int km = min(max(nC / 2, 0), nC - 1);  // the column nearest the atom: the box's centre column or one of its neighbours
    if (km > 0 && sqc[km - 1] < sqc[km]) --km;
    else if (km + 1 < nC && sqc[km + 1] < sqc[km]) ++km;
    const int rows = D1 * D2;
    const unsigned div_d1 = (1024u + (unsigned)D1 - 1u) / (unsigned)D1;  // exact for row < 64, D1 <= 8
    int n = 0;
    for (int row = l8; row < rows; row += 8) {
        const int is = (int)(((unsigned)row * div_d1) >> 10), ir = row - is * D1;
        const double sr = t.sq[1][ir], ss = t.sq[2][is];
        const double A = (MODE == 0) ? ss : ((MODE == 1) ? sr : __dadd_rn(sr, ss));
        const double B = (MODE == 0) ? sr : ss;
        int kl, kh;
        if (!row_chord<MODE>(sqc, nC, km, xc, inv_gl, A, B, T, kl, kh)) continue;
        const int o1 = t.off[1][ir], o2 = t.off[2][is];
        const int orr = o1 | o2;
        const unsigned osum = (unsigned)o1 + (unsigned)o2;
        float v[kSmallBox];
#pragma unroll
        for (int j = 0; j < kSmallBox; ++j) {  // all loads of the chord first
            const int k = kl + j;
            v[j] = 0.f;
            if (k <= kh) {
                const int oc = t.off[0][k];
                if ((orr | oc) >= 0) v[j] = __ldg(rho + (int)(osum + (unsigned)oc));  // a voxel outside the stored map counts as 0
            }
        }
#pragma unroll
        for (int j = 0; j < kSmallBox; ++j) {
            if (kl + j > kh) break;
            if (passes(v[j], cutoff)) {
                ++n;
                if (keep) {
                    const int p = ((kl + j) * D1 + ir) * D2 + is;
                    atomicOr(&wb[p >> 5], 1u << (p & 31));
                }
            }
        }
    }
    return n;
}

__global__ void __launch_bounds__(kSphereWarps * 32)
    cloud_count_kernel(const pe_batch_map *__restrict__ maps, int n_atoms, const int32_t *__restrict__ atom_map,
                       const double *__restrict__ xyz, const float *__restrict__ radius, uint32_t *__restrict__ count,
                       unsigned long long *__restrict__ d_maxbox, uint32_t *__restrict__ box_bits) {
    __shared__ AxisTab tabs[kSphereWarps][2];
    __shared__ pe_geom geoms[kSphereWarps][kCountAtoms];
    __shared__ SmallTabB stab[kSphereWarps][kCountAtoms];
    __shared__ uint32_t wbits[kSphereWarps][kCountAtoms][kBoxBitWords];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int a0 = (blockIdx.x * kSphereWarps + warp) * kCountAtoms;
    if (a0 >= n_atoms) return;
    const int sub = lane >> 3, l8 = lane & 7;
    const int a = a0 + sub;
    const bool live = a < n_atoms;
    const pe_batch_map *m = maps + (live ? atom_map[a] : 0);
    if (live) {  // the group's copy of its structure's geometry
        const unsigned long long *src = reinterpret_cast<const unsigned long long *>(&m->geom);
        unsigned long long *d = reinterpret_cast<unsigned long long *>(&geoms[warp][sub]);
        for (int k = l8; k < (int)(sizeof(pe_geom) / 8); k += 8) d[k] = src[k];
    }
    __syncwarp();
    const pe_geom &g = geoms[warp][sub];
    int lo[3] = {0, 0, 0}, dim[3] = {0, 0, 0};
    double ax = 0.0, ay = 0.0, az = 0.0, T = -1.0;
    bool small = true;
    if (live) {
        ax = xyz[3 * a];
        ay = xyz[3 * a + 1];
        az = xyz[3 * a + 2];
        AtomBox bb;
        atom_box(g, ax, ay, az, radius[a], bb, T);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            lo[k] = bb.lo[k];
            dim[k] = bb.dim[k];
        }
        small = g.orthogonal && dim[0] <= kSmallBox && dim[1] <= kSmallBox && dim[2] <= kSmallBox;
    }
    if (!__all_sync(kFull, small)) {
        for (int q = 0; q < kCountAtoms && a0 + q < n_atoms; ++q)
            count_one_atom(maps, a0 + q, atom_map, xyz, radius, count, d_maxbox, box_bits, tabs[warp], &geoms[warp][0], wbits[warp][0], lane);
        return;
    }
    const int vol = dim[0] * dim[1] * dim[2];
    const bool keep = box_bits != nullptr && vol <= 32 * kBoxBitWords;
    uint32_t *wb = wbits[warp][sub];
    int n = 0;
    wb[l8] = 0u;  // kBoxBitWords == 8: one word per lane of the group
    if (live && vol > 0) {
        SmallTabB &t = stab[warp][sub];
#pragma unroll
        for (int axis = 0; axis < 3; ++axis) {
            if (l8 < dim[axis]) {
                t.sq[axis][l8] = axis_sq(g, axis, lo[axis] + l8, ax, ay, az);
                t.off[axis][l8] = axis_off(g, axis, lo[axis] + l8);
            }
        }
        __syncwarp(0xffu << (8 * sub));  // the 8 lanes of this atom (they take this branch together)
        const float cutoff = m->cutoff;
        const float *rho = m->d_rho;
        const int mode = g.map2xyz[2] == 1 ? 0 : (g.map2xyz[2] == 2 ? 1 : 2);  // crs axis that carries z
        if (mode == 0)
            n = count_small_rows<0>(g, rho, t, lo, dim, ax, ay, az, T, cutoff, keep, wb, l8);
        else if (mode == 1)
            n = count_small_rows<1>(g, rho, t, lo, dim, ax, ay, az, T, cutoff, keep, wb, l8);
        else
            n = count_small_rows<2>(g, rho, t, lo, dim, ax, ay, az, T, cutoff, keep, wb, l8);
    }
    __syncwarp();
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) n += __shfl_xor_sync(kFull, n, o);
    if (live) {
        if (keep) box_bits[(int64_t)a * kBoxBitWords + l8] = wb[l8];
        if (l8 == 0) {
            count[a] = (uint32_t)n;
            const unsigned long long v = (unsigned long long)(vol > 0 ? vol : 0);
            if (v > *d_maxbox) atomicMax(d_maxbox, v);  // L1-cached read of the one hot address: stale values only cost a redundant atomic
        }
    }
}

// ------------------------------------------------------------------------------------------------ pass 1: clouds
// One warp per atom: membership bitmap in the reference's product order, ordered emission of the voxels (packed key,
// density, cluster number), in-warp 26-connected clustering (numbered in createCrsLists order) and the per-cloud sums of
// DensityBlob.fromCrsList (pdb_eda/ccp4.py:522-545).  Per-atom record (8 doubles): number of clouds, voxels of the best
// cloud, smallest centroid distance, total density of the best cloud, its centroid xyz, [7] is written by later kernels.
// Dynamic shared memory per warp: bits[nw] | pref[nw] | pidx[maxbox] lab[maxbox] rnk[maxbox] (u16).
struct FillArgs {
    const pe_batch_map *maps;
    int n_atoms;
    const int32_t *atom_map;
    const double *xyz;
    const float *radius;
    const uint32_t *offset;
    int max_box;
    unsigned long long *e_key;
    float *e_val;
    uint32_t *e_atom;
    uint16_t *e_lab;
    uint32_t *n_clouds;
    double *atom_out;
    int *d_bad;
    unsigned long long *abox;
    const uint32_t *box_bits;
    int *cell_edge;
    int dil_cap;
};

// the per-atom results every later kernel reads: the atom's record and the bounding box of its cloud voxels
__device__ __forceinline__ void fill_box_record(const FillArgs &A, int a, int map_id, int n, int lo_c, int lo_r, int lo_s, int hi_c, int hi_r,
                                                int hi_s) {
    const int d0 = hi_c - lo_c + 1, d1 = hi_r - lo_r + 1, d2 = hi_s - lo_s + 1;
    const int dmax = max(d0, max(d1, d2));
    if (dmax > A.cell_edge[map_id]) atomicMax(A.cell_edge + map_id, dmax);  // hot addresses, read through L1: only the rare increases go to the atomic unit
    // a batch with a cloud the pair kernel's shared-memory frame cannot hold takes the hash-table path
    if (dmax > 15 || n > 1024 || (d0 + 2) * (d1 + 2) * (d2 + 2) > A.dil_cap) A.d_bad[1] = 1;
    A.abox[a] = ((unsigned long long)(unsigned)(lo_c + kKeyOff) << 40) | ((unsigned long long)(unsigned)(lo_r + kKeyOff) << 26) |
                ((unsigned long long)(unsigned)(lo_s + kKeyOff) << 12) | ((unsigned long long)(d0 & 15) << 8) |
                ((unsigned long long)(d1 & 15) << 4) | (unsigned long long)(d2 & 15);
}

// Shift masks of the flood fill for box positions 32 w .. 32 w + 31 (p = (ic*D1 + ir)*D2 + is): nfs / nls = positions that may
// move -1 / +1 along sections, nfr / nlr = -1 / +1 along rows.  They cover EVERY position, member or not: one dilation step moves
// along sections and then along rows, and a diagonal neighbour is reached through a position that may hold no voxel.  Built row
// by row (a row = D2 consecutive positions), so a word costs at most 32 / D2 + 2 steps.
__device__ __forceinline__ void shift_masks(int w, int vol, int D1, int D2, uint32_t &nfs, uint32_t &nls, uint32_t &nfr, uint32_t &nlr) {
    nfs = nls = nfr = nlr = 0u;
    const int p0 = 32 * w, p1 = min(p0 + 32, vol);
    for (int t = p0 / D2; t * D2 < p1; ++t) {
        const int a = max(t * D2, p0) - p0, e = min((t + 1) * D2, p1) - p0;  // the row's bits a .. e-1 in this word
        const uint32_t row = (e - a >= 32 ? 0xffffffffu : (1u << (e - a)) - 1u) << a;
        const int ir = t % D1;
        if (ir != 0) nfr |= row;
        if (ir != D1 - 1) nlr |= row;
        nfs |= t * D2 >= p0 ? row & ~(1u << a) : row;               // not the row's first position (is = 0)
        nls |= (t + 1) * D2 <= p1 ? row & ~(1u << (e - 1)) : row;    // not its last (is = D2 - 1)
    }
}

// One atom by one warp (boxes of more than 256 candidates, or no bitmap from the count pass).
__device__ __forceinline__ void fill_one_atom(const FillArgs &A, int a, unsigned char *base, AxisTab *tab, pe_geom *gs, int lane) {
    const pe_batch_map *__restrict__ maps = A.maps;
    const int32_t *__restrict__ atom_map = A.atom_map;
    const double *__restrict__ xyz = A.xyz;
    const float *__restrict__ radius = A.radius;
    const uint32_t *__restrict__ offset = A.offset;
    const int max_box = A.max_box;
    unsigned long long *__restrict__ e_key = A.e_key;
    float *__restrict__ e_val = A.e_val;
    uint32_t *__restrict__ e_atom = A.e_atom;
    uint16_t *__restrict__ e_lab = A.e_lab;
    uint32_t *__restrict__ n_clouds = A.n_clouds;
    double *__restrict__ atom_out = A.atom_out;
    int *__restrict__ d_bad = A.d_bad;
    const uint32_t *__restrict__ box_bits = A.box_bits;
    const int nw_max = (max_box + 31) / 32;
    const int box_pad = (max_box + 1) / 2 * 2;
    uint32_t *bits = reinterpret_cast<uint32_t *>(base);
    uint32_t *pref = bits + nw_max;
    uint16_t *pidx = reinterpret_cast<uint16_t *>(pref + nw_max);
    uint16_t *lab = pidx + box_pad;
    uint16_t *rnk = lab + box_pad;

    const int map_id = atom_map[a];
    const pe_batch_map *m = maps + map_id;
    load_geom(gs, m, lane);
    const pe_geom &g = *gs;
    const float *rho = m->d_rho;
    const float cutoff = m->cutoff;
    const double ax = xyz[3 * a], ay = xyz[3 * a + 1], az = xyz[3 * a + 2];
    AtomBox b;
    double T;
    atom_box(g, ax, ay, az, radius[a], b, T);
    const int D1 = b.dim[1], D2 = b.dim[2];
    const int vol = b.dim[0] * D1 * D2;
    double *rec = atom_out + (int64_t)a * 8;
    if (vol > max_box || vol > 65535) {  // cannot happen: max_box comes from the count pass over the same atoms
        if (lane == 0) {
            *d_bad = 1;
            n_clouds[a] = 0;
            for (int k = 0; k < 8; ++k) rec[k] = 0.0;
        }
        return;
    }
    const int nw = (vol + 31) / 32;
    for (int w = lane; w < nw; w += 32) bits[w] = 0u;
    __syncwarp();
    // 1. membership bits in the reference's order: p = (ic*D1 + ir)*D2 + is (from the count pass when it kept them)
    if (box_bits != nullptr && vol <= 32 * kBoxBitWords) {
        if (lane < nw) bits[lane] = box_bits[(int64_t)a * kBoxBitWords + lane];
        __syncwarp();
    } else {
        for_each_inside(g, rho, b, ax, ay, az, T, tab, lane, [&](int ic, int ir, int is, bool, float v) {
            if (passes(v, cutoff)) {
                const int p = (ic * D1 + ir) * D2 + is;
                atomicOr(bits + (p >> 5), 1u << (p & 31));
            }
        });
    }
    // 2. per-word prefix counts
    int running = 0;
    for (int w0 = 0; w0 < nw; w0 += 32) {
        const int w = w0 + lane;
        const int cnt = w < nw ? __popc(bits[w]) : 0;
        const int ex = warp_excl_scan(cnt, lane);
        if (w < nw) pref[w] = (uint32_t)(running + ex);
        running += __shfl_sync(kFull, ex + cnt, 31);
    }
    __syncwarp();
    const int n = running;
    const uint32_t obase = offset[a];
    if ((uint32_t)n != offset[a + 1] - obase) {  // the two passes must agree
        if (lane == 0) *d_bad = 1;
        return;
    }
    // 3. ordered list of box positions
    for (int w = lane; w < nw; w += 32) {
        uint32_t word = bits[w];
        int j = (int)pref[w];
        while (word) {
            const int bit = __ffs(word) - 1;
            word &= word - 1;
            pidx[j++] = (uint16_t)(w * 32 + bit);
        }
    }
    __syncwarp();
    // 4 + 5. 26-connected clusters of the listed voxels, numbered by their first member (the order createCrsLists creates them in)
    int nroots = 0;
    if (nw <= 32) {
        // Bit-parallel flood fill: the box is at most 32 words, one per lane.  A cluster grows from the lowest unlabelled voxel by
        // repeated 3 x 3 x 3 dilation -- three separable +-1 shifts of the whole bit string (multi-word shifts across lanes), with
        // masks that stop a shift from wrapping into the next row / plane -- intersected with the unlabelled voxels, until it stops
        // growing; clusters therefore come out in the order of their first member.  (The min-label propagation this replaces was
        // 56 % of the kernel's instructions: 27 bit tests and label look-ups per voxel and round.)
        uint32_t nfs, nls, nfr, nlr;  // positions that may move -1 / +1 along sections, -1 / +1 along rows
        shift_masks(lane, vol, D1, D2, nfs, nls, nfr, nlr);
        auto shl = [&](uint32_t v, int k) {  // the bit string moved k positions up
            const int q = k >> 5, r = k & 31;
            uint32_t a = __shfl_up_sync(kFull, v, q), c = __shfl_up_sync(kFull, v, q + 1);
            if (lane < q) a = 0u;
            if (lane < q + 1) c = 0u;
            return r ? ((a << r) | (c >> (32 - r))) : a;
        };
        auto shr = [&](uint32_t v, int k) {
            const int q = k >> 5, r = k & 31;
            uint32_t a = __shfl_down_sync(kFull, v, q), c = __shfl_down_sync(kFull, v, q + 1);
            if (lane + q > 31) a = 0u;
            if (lane + q + 1 > 31) c = 0u;
            return r ? ((a >> r) | (c << (32 - r))) : a;
        };
        const uint32_t mine = lane < nw ? bits[lane] : 0u;
        const int mybase = lane < nw ? (int)pref[lane] : 0;
        uint32_t todo = mine;
        const int plane = D1 * D2;
        for (;;) {
            const unsigned has = __ballot_sync(kFull, todo != 0u);
            if (!has) break;
            uint32_t comp = (lane == __ffs((int)has) - 1) ? (todo & (0u - todo)) : 0u;  // the lowest unlabelled voxel
            for (;;) {
                const uint32_t x = comp | shl(comp & nls, 1) | shr(comp & nfs, 1);
                const uint32_t y = x | shl(x & nlr, D2) | shr(x & nfr, D2);
                const uint32_t z = (y | (plane < 1024 ? (shl(y, plane) | shr(y, plane)) : 0u)) & todo;
                const bool grew = z != comp;
                comp = z;
                if (!__any_sync(kFull, grew)) break;
            }
            for (uint32_t c = comp; c;) {
                const int bit = __ffs((int)c) - 1;
                c &= c - 1u;
                const int j = mybase + __popc(mine & ((1u << bit) - 1u));
                lab[j] = (uint16_t)j;
                rnk[j] = (uint16_t)nroots;  // rnk[lab[j]] is the cluster number below
            }
            todo &= ~comp;
            ++nroots;
        }
        __syncwarp();
    } else {
    // min-label propagation with pointer jumping (boxes of more than 1,024 voxels)
    for (int j = lane; j < n; j += 32) lab[j] = (uint16_t)j;
    __syncwarp();
    for (;;) {
        bool changed = false;
        for (int j = lane; j < n; j += 32) {
            const int p = pidx[j];
            const int is = p % D2, t = p / D2, ir = t % D1, ic = t / D1;
            int mn = lab[j];
            for (int dc = -1; dc <= 1; ++dc) {
                const int c2 = ic + dc;
                if (c2 < 0 || c2 >= b.dim[0]) continue;
                for (int dr = -1; dr <= 1; ++dr) {
                    const int r2 = ir + dr;
                    if (r2 < 0 || r2 >= D1) continue;
                    for (int ds = -1; ds <= 1; ++ds) {
                        const int s2 = is + ds;
                        if (s2 < 0 || s2 >= D2) continue;
                        const int q = (c2 * D1 + r2) * D2 + s2;
                        const uint32_t word = bits[q >> 5];
                        if (!((word >> (q & 31)) & 1u)) continue;
                        const int jn = (int)pref[q >> 5] + __popc(word & ((1u << (q & 31)) - 1u));
                        mn = min(mn, (int)lab[jn]);
                    }
                }
            }
            mn = min(mn, (int)lab[mn]);
            if (mn < (int)lab[j]) {
                lab[j] = (uint16_t)mn;
                changed = true;
            }
        }
        __syncwarp();
        if (!__any_sync(kFull, changed)) break;
    }
    // number the clusters by their first member
    for (int j0 = 0; j0 < n; j0 += 32) {
        const int j = j0 + lane;
        const int isroot = (j < n && lab[j] == j) ? 1 : 0;
        const int ex = warp_excl_scan(isroot, lane);
        if (isroot) rnk[j] = (uint16_t)(nroots + ex);
        nroots += __shfl_sync(kFull, ex + isroot, 31);
    }
    __syncwarp();
    }
    // 6. entries: packed key (structure, un-wrapped crs), density, owning atom, cloud number inside the atom
    bool bad = false;
    int lo_c = INT_MAX, lo_r = INT_MAX, lo_s = INT_MAX, hi_c = INT_MIN, hi_r = INT_MIN, hi_s = INT_MIN;
    for (int j = lane; j < n; j += 32) {
        const int p = pidx[j];
        const int is = p % D2, t = p / D2, ir = t % D1, ic = t / D1;
        const int c = b.lo[0] + ic, r = b.lo[1] + ir, s = b.lo[2] + is;
        lo_c = min(lo_c, c);
        hi_c = max(hi_c, c);
        lo_r = min(lo_r, r);
        hi_r = max(hi_r, r);
        lo_s = min(lo_s, s);
        hi_s = max(hi_s, s);
        const unsigned uc = (unsigned)(c + kKeyOff), ur = (unsigned)(r + kKeyOff), us = (unsigned)(s + kKeyOff);
        // neighbours (+-1) must stay inside the field: 1 <= u < 2^14 - 1
        if (uc - 1u >= (1u << kKeyBits) - 2u || ur - 1u >= (1u << kKeyBits) - 2u || us - 1u >= (1u << kKeyBits) - 2u) bad = true;
        const int oc = axis_off(g, 0, c), orr = axis_off(g, 1, r), os = axis_off(g, 2, s);
        e_key[obase + j] = ((unsigned long long)(unsigned)map_id << (3 * kKeyBits)) | ((unsigned long long)uc << (2 * kKeyBits)) |
                           ((unsigned long long)ur << kKeyBits) | (unsigned long long)us;
        e_val[obase + j] = ((oc | orr | os) >= 0) ? __ldg(rho + (oc + orr + os)) : 0.f;
        e_atom[obase + j] = (uint32_t)a;
        e_lab[obase + j] = rnk[lab[j]];
    }
    if (__any_sync(kFull, bad) && lane == 0) *d_bad = 1;
    if (n > 0) {
        // bounding box of the atom's cloud voxels for the pair kernel (key-offset corner, dimensions).  A batch with a cloud the
        // pair kernel's shared-memory frame cannot hold takes the hash-table path (d_bad[1]); cell_edge[structure] = widest bounding box edge
        // of the batch = cell edge of the atom grid.
        lo_c = __reduce_min_sync(kFull, lo_c);
        lo_r = __reduce_min_sync(kFull, lo_r);
        lo_s = __reduce_min_sync(kFull, lo_s);
        hi_c = __reduce_max_sync(kFull, hi_c);
        hi_r = __reduce_max_sync(kFull, hi_r);
        hi_s = __reduce_max_sync(kFull, hi_s);
        if (lane == 0) fill_box_record(A, a, map_id, n, lo_c, lo_r, lo_s, hi_c, hi_r, hi_s);
    }
    // 7. per-cloud sums (fromCrsList) -> centroid distance; the nearest cloud (first minimum, :630-634)
    double best_dist = 0.0, best_sum = 0.0, bcx = 0.0, bcy = 0.0, bcz = 0.0;
    int best_n = 0;
    for (int k = 0; k < nroots; ++k) {
        double sd = 0.0, sx = 0.0, sy = 0.0, sz = 0.0;
        int cn = 0;
        for (int j = lane; j < n; j += 32) {
            if ((int)rnk[lab[j]] != k) continue;
            const int p = pidx[j];
            const int is = p % D2, t = p / D2, ir = t % D1, ic = t / D1;
            const int c = b.lo[0] + ic, r = b.lo[1] + ir, s = b.lo[2] + is;
            const int oc = axis_off(g, 0, c), orr = axis_off(g, 1, r), os = axis_off(g, 2, s);
            const double d = ((oc | orr | os) >= 0) ? (double)__ldg(rho + (oc + orr + os)) : 0.0;
            double x, y, z;
            crs2xyz(g, c, r, s, x, y, z);
            sd += d;
            sx += __dmul_rn(d, x);
            sy += __dmul_rn(d, y);
            sz += __dmul_rn(d, z);
            ++cn;
        }
        sd = warp_sum(sd);
        sx = warp_sum(sx);
        sy = warp_sum(sy);
        sz = warp_sum(sz);
        cn = warp_sum(cn);
        const double cx = sx / sd, cy = sy / sd, cz = sz / sd;
        const double dx = ax - cx, dy = ay - cy, dz = az - cz;
        const double dist = sqrt(dx * dx + dy * dy + dz * dz);  // np.linalg.norm(atom.coord - cloud.centroid)
        if (k == 0 || dist < best_dist) {  // Python's min(): a later value replaces only when strictly smaller
            best_dist = dist;
            best_sum = sd;
            best_n = cn;
            bcx = cx;
            bcy = cy;
            bcz = cz;
        }
    }
    if (lane == 0) {
        if (nroots > kPairClouds) d_bad[1] = 1;
        n_clouds[a] = (uint32_t)nroots;
        rec[0] = (double)nroots;
        rec[1] = (double)best_n;
        rec[2] = best_dist;
        rec[3] = best_sum;
        rec[4] = bcx;
        rec[5] = bcy;
        rec[6] = bcz;
        rec[7] = 0.0;
    }
}

// A warp takes kFillAtoms = 4 consecutive atoms.  When the count pass left a bitmap for all four (candidate boxes of at most 256
// voxels: 8 words) each atom gets 8 lanes, one bitmap word per lane: prefix counts, the bit-parallel flood fill (multi-word
// shifts across the 8 lanes), the entries and the per-cloud sums all run inside the 8-lane group, four atoms side by side --
// the one-warp-per-atom form spent ~1,900 warp instructions per atom with a third of the lanes busy (ncu: issue slots 60 % busy).
// Otherwise the warp handles its atoms one after the other with all 32 lanes (fill_one_atom).
constexpr int kFillAtoms = 4;
struct FillGroupShared {
    pe_geom geom;
    float val[32 * kBoxBitWords];   // density of the listed voxels
    uint8_t lab[32 * kBoxBitWords];  // their cluster numbers
};

__global__ void __launch_bounds__(kSphereWarps * 32) cloud_fill_kernel(const FillArgs A, int warps, size_t per_warp) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    __shared__ AxisTab tabs[kSphereWarps][2];
    __shared__ FillGroupShared fgs[kSphereWarps][kFillAtoms];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int a0 = (blockIdx.x * warps + warp) * kFillAtoms;
    if (a0 >= A.n_atoms) return;
    const int sub = lane >> 3, l8 = lane & 7;
    const unsigned gmask = 0xffu << (8 * sub);
    const int a = a0 + sub;
    const bool live = a < A.n_atoms;
    const int map_id = live ? A.atom_map[a] : 0;
    const pe_batch_map *m = A.maps + map_id;
    FillGroupShared &fg = fgs[warp][sub];
    if (live) {
        const unsigned long long *src = reinterpret_cast<const unsigned long long *>(&m->geom);
        unsigned long long *d = reinterpret_cast<unsigned long long *>(&fg.geom);
        for (int k = l8; k < (int)(sizeof(pe_geom) / 8); k += 8) d[k] = src[k];
    }
    __syncwarp();
    const pe_geom &g = fg.geom;
    AtomBox b;
    double T;
    double ax = 0.0, ay = 0.0, az = 0.0;
    int vol = 0;
    if (live) {
        ax = A.xyz[3 * a];
        ay = A.xyz[3 * a + 1];
        az = A.xyz[3 * a + 2];
        atom_box(g, ax, ay, az, A.radius[a], b, T);
        vol = b.dim[0] * b.dim[1] * b.dim[2];
    }
    const bool small = !live || (A.box_bits != nullptr && vol <= 32 * kBoxBitWords);
    if (!__all_sync(kFull, small)) {
        for (int q = 0; q < kFillAtoms && a0 + q < A.n_atoms; ++q) {
            fill_one_atom(A, a0 + q, dyn_smem + per_warp * warp, tabs[warp], &fgs[warp][0].geom, lane);
            __syncwarp();  // the scratch is reused by the warp's next atom
        }
        return;
    }
    if (!live) return;  // from here on only the 8 lanes of a group synchronise
    const float *rho = m->d_rho;
    const int D1 = b.dim[1], D2 = b.dim[2];
    const int nw = (vol + 31) / 32;
    double *rec = A.atom_out + (int64_t)a * 8;
    // 1 + 2. the bitmap of the count pass, one word per lane; prefix counts
    const uint32_t mine = l8 < nw ? A.box_bits[(int64_t)a * kBoxBitWords + l8] : 0u;
    int mybase, n;
    {
        const int cnt = __popc(mine);
        int x = cnt;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
            const int y = __shfl_up_sync(gmask, x, o, 8);
            if (l8 >= o) x += y;
        }
        mybase = x - cnt;
        n = __shfl_sync(gmask, x, 7, 8);
    }
    const uint32_t obase = A.offset[a];
    if ((uint32_t)n != A.offset[a + 1] - obase) {  // the two passes must agree
        if (l8 == 0) *A.d_bad = 1;
        return;
    }
    // 4 + 5. 26-connected clusters by bit-parallel flood fill, numbered by their first member (createCrsLists order)
    // p / D by multiplication: exact for p < 256, D <= 256
    const uint32_t m2 = (65536u + (uint32_t)max(D2, 1) - 1u) / (uint32_t)max(D2, 1), m1 = (65536u + (uint32_t)max(D1, 1) - 1u) / (uint32_t)max(D1, 1);
    uint32_t nfs, nls, nfr, nlr;  // positions that may move -1 / +1 along sections, -1 / +1 along rows
    shift_masks(l8, vol, D1, D2, nfs, nls, nfr, nlr);
    auto shl = [&](uint32_t v, int k) {  // the group's bit string moved k positions up
        const int q = k >> 5, r = k & 31;
        uint32_t x = __shfl_up_sync(gmask, v, q, 8), y = __shfl_up_sync(gmask, v, q + 1, 8);
        if (l8 < q) x = 0u;
        if (l8 < q + 1) y = 0u;
        return r ? ((x << r) | (y >> (32 - r))) : x;
    };
    auto shr = [&](uint32_t v, int k) {
        const int q = k >> 5, r = k & 31;
        uint32_t x = __shfl_down_sync(gmask, v, q, 8), y = __shfl_down_sync(gmask, v, q + 1, 8);
        if (l8 + q > 7) x = 0u;
        if (l8 + q + 1 > 7) y = 0u;
        return r ? ((x >> r) | (y << (32 - r))) : x;
    };
    int nroots = 0;
    {
        uint32_t todo = mine;
        const int plane = D1 * D2;
        for (;;) {
            const unsigned has = (__ballot_sync(gmask, todo != 0u) >> (8 * sub)) & 0xffu;
            if (!has) break;
            uint32_t comp = (l8 == __ffs((int)has) - 1) ? (todo & (0u - todo)) : 0u;  // the lowest unlabelled voxel
            for (;;) {
                const uint32_t x = comp | shl(comp & nls, 1) | shr(comp & nfs, 1);
                const uint32_t y = x | shl(x & nlr, D2) | shr(x & nfr, D2);
                const uint32_t z = (y | (plane < 32 * kBoxBitWords ? (shl(y, plane) | shr(y, plane)) : 0u)) & todo;
                const bool grew = z != comp;
                comp = z;
                if (!__any_sync(gmask, grew)) break;
            }
            for (uint32_t c = comp; c;) {
                const int bit = __ffs((int)c) - 1;
                c &= c - 1u;
                fg.lab[mybase + __popc(mine & ((1u << bit) - 1u))] = (uint8_t)nroots;
            }
            todo &= ~comp;
            ++nroots;
        }
    }
    __syncwarp(gmask);
    // 6. entries: packed key (structure, un-wrapped crs), density, owning atom, cloud number inside the atom
    bool bad = false;
    int lo_c = INT_MAX, lo_r = INT_MAX, lo_s = INT_MAX, hi_c = INT_MIN, hi_r = INT_MIN, hi_s = INT_MIN;
    {
        int jj = mybase;
        for (uint32_t cb = mine; cb; cb &= cb - 1u, ++jj) {
            const uint32_t p = 32u * (uint32_t)l8 + (uint32_t)(__ffs((int)cb) - 1);
            const uint32_t q = (p * m2) >> 16, ic = (q * m1) >> 16;
            const int c = b.lo[0] + (int)ic, r = b.lo[1] + (int)(q - ic * (uint32_t)D1), s = b.lo[2] + (int)(p - q * (uint32_t)D2);
            lo_c = min(lo_c, c);
            hi_c = max(hi_c, c);
            lo_r = min(lo_r, r);
            hi_r = max(hi_r, r);
            lo_s = min(lo_s, s);
            hi_s = max(hi_s, s);
            const unsigned uc = (unsigned)(c + kKeyOff), ur = (unsigned)(r + kKeyOff), us = (unsigned)(s + kKeyOff);
            // neighbours (+-1) must stay inside the field: 1 <= u < 2^14 - 1
            if (uc - 1u >= (1u << kKeyBits) - 2u || ur - 1u >= (1u << kKeyBits) - 2u || us - 1u >= (1u << kKeyBits) - 2u) bad = true;
            const int oc = axis_off(g, 0, c), orr = axis_off(g, 1, r), os = axis_off(g, 2, s);
            const float v = ((oc | orr | os) >= 0) ? __ldg(rho + (oc + orr + os)) : 0.f;
            fg.val[jj] = v;
            A.e_key[obase + jj] = ((unsigned long long)(unsigned)map_id << (3 * kKeyBits)) | ((unsigned long long)uc << (2 * kKeyBits)) |
                                  ((unsigned long long)ur << kKeyBits) | (unsigned long long)us;
            A.e_val[obase + jj] = v;
            A.e_atom[obase + jj] = (uint32_t)a;
            A.e_lab[obase + jj] = (uint16_t)fg.lab[jj];
        }
    }
    if (__any_sync(gmask, bad) && l8 == 0) *A.d_bad = 1;
    if (n > 0) {
        lo_c = __reduce_min_sync(gmask, lo_c);
        lo_r = __reduce_min_sync(gmask, lo_r);
        lo_s = __reduce_min_sync(gmask, lo_s);
        hi_c = __reduce_max_sync(gmask, hi_c);
        hi_r = __reduce_max_sync(gmask, hi_r);
        hi_s = __reduce_max_sync(gmask, hi_s);
        if (l8 == 0) fill_box_record(A, a, map_id, n, lo_c, lo_r, lo_s, hi_c, hi_r, hi_s);
    }
    // 7. per-cloud sums (fromCrsList) -> centroid distance; the nearest cloud (first minimum, :630-634)
    double best_dist = 0.0, best_sum = 0.0, bcx = 0.0, bcy = 0.0, bcz = 0.0;
    int best_n = 0;
    for (int k = 0; k < nroots; ++k) {
        double sd = 0.0, sx = 0.0, sy = 0.0, sz = 0.0;
        int cn = 0;
        int jj = mybase;
        for (uint32_t cb = mine; cb; cb &= cb - 1u, ++jj) {
            if ((int)fg.lab[jj] != k) continue;
            const uint32_t p = 32u * (uint32_t)l8 + (uint32_t)(__ffs((int)cb) - 1);
            const uint32_t q = (p * m2) >> 16, ic = (q * m1) >> 16;
            const int c = b.lo[0] + (int)ic, r = b.lo[1] + (int)(q - ic * (uint32_t)D1), s = b.lo[2] + (int)(p - q * (uint32_t)D2);
            const double d = (double)fg.val[jj];
            double x, y, z;
            crs2xyz(g, c, r, s, x, y, z);
            sd += d;
            sx += __dmul_rn(d, x);
            sy += __dmul_rn(d, y);
            sz += __dmul_rn(d, z);
            ++cn;
        }
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            sd += __shfl_xor_sync(gmask, sd, o);
            sx += __shfl_xor_sync(gmask, sx, o);
            sy += __shfl_xor_sync(gmask, sy, o);
            sz += __shfl_xor_sync(gmask, sz, o);
            cn += __shfl_xor_sync(gmask, cn, o);
        }
        const double cx = sx / sd, cy = sy / sd, cz = sz / sd;
        const double dx = ax - cx, dy = ay - cy, dz = az - cz;
        const double dist = sqrt(dx * dx + dy * dy + dz * dz);  // np.linalg.norm(atom.coord - cloud.centroid)
        if (k == 0 || dist < best_dist) {  // Python's min(): a later value replaces only when strictly smaller
            best_dist = dist;
            best_sum = sd;
            best_n = cn;
            bcx = cx;
            bcy = cy;
            bcz = cz;
        }
    }
    if (l8 == 0) {
        if (nroots > kPairClouds) A.d_bad[1] = 1;
        A.n_clouds[a] = (uint32_t)nroots;
        rec[0] = (double)nroots;
        rec[1] = (double)best_n;
        rec[2] = best_dist;
        rec[3] = best_sum;
        rec[4] = bcx;
        rec[5] = bcy;
        rec[6] = bcz;
        rec[7] = 0.0;
    }
}

// ------------------------------------------------------------------------------------------------ centroid cutoff
// np.nanmedian(d) + 2.5 * np.nanstd(d) over the smallest centroid distances of a structure's atoms that have clouds
// (pdb_eda/densityAnalysis.py:608-609).  One CTA per structure; exact order statistics by radix select on the bit
// patterns (distances are >= 0, so IEEE order is integer order); fixed-order reductions: deterministic.
__global__ void __launch_bounds__(kSummaryThreads)
    cutoff_kernel(const pe_batch_map *__restrict__ maps, const double *__restrict__ atom_out, double *__restrict__ map_out) {
    __shared__ SelectShared sel;
    __shared__ double scratch[kSummaryThreads / 32];
    const pe_batch_map *m = maps + blockIdx.x;
    const int a0 = m->atom_begin, a1 = m->atom_end;
    double *mo = map_out + (int64_t)blockIdx.x * 8;
    auto valid = [&](int a) { return atom_out[(int64_t)a * 8] > 0.0 && !isnan(atom_out[(int64_t)a * 8 + 2]); };
    double cnt = 0.0, sum = 0.0;
    for (int a = a0 + threadIdx.x; a < a1; a += blockDim.x)
        if (valid(a)) {
            cnt += 1.0;
            sum += atom_out[(int64_t)a * 8 + 2];
        }
    cnt = block_sum_fixed(cnt, scratch);
    sum = block_sum_fixed(sum, scratch);
    const double mean = sum / cnt;
    double sq = 0.0;
    for (int a = a0 + threadIdx.x; a < a1; a += blockDim.x)
        if (valid(a)) {
            const double d = atom_out[(int64_t)a * 8 + 2] - mean;
            sq += d * d;
        }
    sq = block_sum_fixed(sq, scratch);
    const double median = block_nanmedian(a1 - a0, [&](int i) { return valid(a0 + i) ? order_key(atom_out[(int64_t)(a0 + i) * 8 + 2]) : kNoKey; }, sel);
    if (threadIdx.x == 0) mo[7] = median + 2.5 * sqrt(sq / cnt);  // NaN when no atom has a cloud
}

// ------------------------------------------------------------------------------------------------ pass 2: which atoms contribute
__global__ void __launch_bounds__(kAggThreads)
    accept_kernel(const pe_batch_map *__restrict__ maps, int n_atoms, const int32_t *__restrict__ atom_map,
                  const int32_t *__restrict__ atom_residue, const int32_t *__restrict__ atom_local, double *__restrict__ atom_out,
                  const double *__restrict__ map_out, uint32_t *__restrict__ cloud_count, unsigned long long *__restrict__ res_mask) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a > n_atoms) return;
    if (a == n_atoms) {
        cloud_count[a] = 0u;  // the scan wants n_atoms + 1 entries
        return;
    }
    double *rec = atom_out + (int64_t)a * 8;
    const double cutoff = map_out[(int64_t)atom_map[a] * 8 + 7];
    const int nc = (int)rec[0];
    const bool ok = nc > 0 && (nc == 1 || !(rec[2] > cutoff));
    rec[7] = ok ? 1.0 : 0.0;
    cloud_count[a] = ok ? (uint32_t)nc : 0u;
    if (ok) atomicOr(res_mask + atom_residue[a], 1ull << atom_local[a]);
}

// ------------------------------------------------------------------------------------------------ pool voxel table
__global__ void __launch_bounds__(kAggThreads)
    pool_insert_kernel(int64_t n, const unsigned long long *__restrict__ e_key, const uint32_t *__restrict__ e_atom,
                       const double *__restrict__ atom_out, AggTable t, const int *__restrict__ flags) {
    if (!flags[1]) return;  // the pair kernel handles this batch
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t atom = e_atom[i];
        uint32_t next = kAggNil;
        if (atom_out[(int64_t)atom * 8 + 7] != 0.0) {  // the atom contributes
            const unsigned long long key = e_key[i];
            uint64_t base;
            uint32_t size;
            agg_region(t, key, base, size);
            uint32_t h = agg_start(key, size);
            for (;;) {
                AggSlot *sl = t.slot + base + h;
                unsigned long long old = sl->key;
                if (old == kAggEmpty) old = atomicCAS(&sl->key, (unsigned long long)kAggEmpty, key);
                if (old == kAggEmpty || old == key) {
                    next = atomicExch(&sl->head, (uint32_t)i);
                    break;
                }
                h = h + 1 == size ? 0 : h + 1;
            }
        }
        t.node[i] = make_uint2(next, atom);
    }
}

// per atom: (first cloud id, residue, index inside the residue, contributes) in one 16-byte record
__global__ void __launch_bounds__(kAggThreads)
    atom_info_kernel(int n_atoms, const uint32_t *__restrict__ cloud_start, const int32_t *__restrict__ atom_residue,
                     const int32_t *__restrict__ atom_local, const double *__restrict__ atom_out, int4 *__restrict__ info) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n_atoms) return;
    info[a] = make_int4((int)cloud_start[a], atom_residue[a], atom_local[a], atom_out[(int64_t)a * 8 + 7] != 0.0 ? 1 : 0);
}

// Every pool voxel looks at its own position and at 13 of its 26 neighbours (adjacency is symmetric): clouds that share or
// touch a voxel are united in the domain union-find; clouds of one residue also in the residue union-find, and their atoms
// mark each other in the per-atom adjacency masks (the overlap matrix of pdb_eda/densityAnalysis.py:646-649 reduced to
// what the completeness test of :653-659 reads).
__global__ void __launch_bounds__(kAggThreads)
    cloud_merge_kernel(int64_t n, const unsigned long long *__restrict__ e_key, const uint16_t *__restrict__ e_lab,
                       const int4 *__restrict__ info, AggTable t, uint32_t *parent_dom, uint32_t *parent_res, unsigned long long *adj,
                       const int *__restrict__ flags) {
    if (!flags[1]) return;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t ai = t.node[i].y;
        const int4 me = info[ai];
        if (!me.w) continue;
        const unsigned long long key = e_key[i];
        const uint32_t ci = (uint32_t)me.x + e_lab[i];
        uint32_t root_dom = ci;  // a known ancestor of ci in the domain forest, carried from one hook to the next
#pragma unroll 1
        for (int q = 0; q < 14; ++q) {
            // q = 0: the voxel itself; q = 1..13: the neighbours that precede it in (c, r, s) order
            const int p = q - 1;
            const int dc = q == 0 ? 0 : (p < 9 ? -1 : 0);
            const int dr = q == 0 ? 0 : (p < 9 ? (p / 3) - 1 : (p < 12 ? -1 : 0));
            const int ds = q == 0 ? 0 : (p < 9 ? (p % 3) - 1 : (p < 12 ? (p - 9) - 1 : -1));
            const unsigned long long nk = key + (long long)dc * (1ll << (2 * kKeyBits)) + (long long)dr * (1ll << kKeyBits) + (long long)ds;
            for (uint32_t j = agg_lookup(t, nk); j != kAggNil;) {
                const uint2 nd = t.node[j];
                const uint32_t jj = j;
                j = nd.x;
                if (nd.y == ai) continue;  // clouds of one atom are disjoint components: never adjacent
                const int4 other = info[nd.y];
                const uint32_t cj = (uint32_t)other.x + e_lab[jj];
                if (__ldcg(parent_dom + cj) != root_dom || __ldcg(parent_dom + root_dom) != root_dom) {  // cheap "already one set" test
                    uf_union(parent_dom, root_dom, cj);
                    root_dom = __ldcg(parent_dom + root_dom);
                }
                if (other.y == me.y) {
                    uf_union(parent_res, ci, cj);
                    const unsigned long long bi = 1ull << me.z, bj = 1ull << other.z;
                    if (!(adj[ai] & bj)) atomicOr(adj + ai, bj);
                    if (!(adj[nd.y] & bi)) atomicOr(adj + nd.y, bi);
                }
            }
        }
    }
}

// first[i] = 1 iff entry i is the first pool entry of its voxel: the SET semantics of DensityBlob.merge (pdb_eda/ccp4.py:575-586)
__global__ void __launch_bounds__(kAggThreads)
    cloud_first_kernel(int64_t n, const unsigned long long *__restrict__ e_key, const int4 *__restrict__ info, AggTable t,
                       uint8_t *__restrict__ first, const int *__restrict__ flags) {
    if (!flags[1]) return;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        uint8_t f = 0;
        if (info[t.node[i].y].w) {
            uint32_t mn = kAggNil;
            for (uint32_t j = agg_lookup(t, e_key[i]); j != kAggNil; j = t.node[j].x) mn = min(mn, j);
            f = mn == (uint32_t)i ? 1 : 0;
        }
        first[i] = f;
    }
}

// ------------------------------------------------------------------------------------------------ pair path
// The same merge without a voxel table.  Clouds of two atoms can only touch when the atoms' boxes touch, an atom has a handful
// of such neighbours, and a box is a few hundred voxels -- so instead of hashing every cloud voxel of the batch (55 M entries,
// 14 dependent probes each: 45 of the 84 ms of a 256-structure pass) the ATOMS are binned into a grid of cells one box edge wide
// (a hash table of n_atoms entries, one region per structure), and a warp that owns atom j
//   1. lays j's clouds out in shared memory over the box grown by one voxel: per voxel a byte mask of the clouds of j that
//      hold or touch it (27 ORs per cloud voxel) and the number of j's own entry at that voxel;
//   2. looks up the 27 cells around j (one lane each) and, for every contributing atom i < j whose box touches j's, walks i's
//      entries: a voxel that falls on a non-empty mask byte makes (cloud of i, clouds of j) pairs -- collected as a 64-bit
//      mask and united ONCE per pair after the walk -- and a voxel that j holds too is not j's first entry (the SET semantics
//      of DensityBlob.merge, pdb_eda/ccp4.py:575-586).
// Union-find forests, adjacency masks and first flags are what cloud_merge_kernel / cloud_first_kernel produce.  Batches the
// frame cannot hold (a box edge above 15 voxels, more than 1,024 box voxels, more than kPairClouds clouds on an atom) are flagged
// by cloud_fill_kernel (flags[1]) and take the hash-table kernels instead.
__device__ __forceinline__ void atom_region(const pe_batch_map *maps, uint32_t map_id, uint64_t &base, uint32_t &size) {
    const pe_batch_map *m = maps + map_id;
    base = 2ull * (uint64_t)m->atom_begin + 16ull * map_id;
    size = (uint32_t)(2 * (m->atom_end - m->atom_begin) + 16);
}
__device__ __forceinline__ unsigned long long cell_key(uint32_t map_id, uint32_t cc, uint32_t cr, uint32_t cs) {
    return ((unsigned long long)map_id << (3 * kKeyBits)) | ((unsigned long long)cc << (2 * kKeyBits)) | ((unsigned long long)cr << kKeyBits) |
           (unsigned long long)cs;
}

__global__ void __launch_bounds__(kAggThreads)
    atom_cell_insert_kernel(const pe_batch_map *__restrict__ maps, int n_atoms, const int32_t *__restrict__ atom_map,
                            const int4 *__restrict__ info, const unsigned long long *__restrict__ abox, AggSlot *aslot,
                            uint32_t *__restrict__ anext, const int *__restrict__ flags, const int *__restrict__ cell_edge) {
    if (flags[1]) return;
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n_atoms) return;
    uint32_t next = kAggNil;
    if (info[a].w) {
        const uint32_t E = (uint32_t)max(cell_edge[atom_map[a]], 1);
        const unsigned long long bx = abox[a];
        const uint32_t map_id = (uint32_t)atom_map[a];
        const unsigned long long key = cell_key(map_id, (uint32_t)(bx >> 40) / E, (uint32_t)((bx >> 26) & 0x3fffu) / E, (uint32_t)((bx >> 12) & 0x3fffu) / E);
        uint64_t base;
        uint32_t size;
        atom_region(maps, map_id, base, size);
        uint32_t h = agg_start(key, size);
        for (;;) {
            AggSlot *sl = aslot + base + h;
            unsigned long long old = sl->key;
            if (old == kAggEmpty) old = atomicCAS(&sl->key, (unsigned long long)kAggEmpty, key);
            if (old == kAggEmpty || old == key) {
                next = atomicExch(&sl->head, (uint32_t)a);
                break;
            }
            h = h + 1 == size ? 0 : h + 1;
        }
    }
    anext[a] = next;
}

// (56 registers, 9 CTAs per SM.  __launch_bounds__(128, 12) / (128, 16) -- 40 / 32 registers with spills -- ran at 21.2 / 22.4 ms
// against 14.8 ms, and so did (128, 1), which lets ptxas take more registers: profiles/r02_c3_pool.md.)
__global__ void __launch_bounds__(kPairWarps * 32)
    cloud_pair_kernel(const pe_batch_map *__restrict__ maps, int n_atoms, const int32_t *__restrict__ atom_map,
                      const uint32_t *__restrict__ offset, const unsigned long long *__restrict__ e_key, const uint16_t *__restrict__ e_lab,
                      const int4 *__restrict__ info, const unsigned long long *__restrict__ abox, const AggSlot *__restrict__ aslot,
                      const uint32_t *__restrict__ anext, uint32_t *parent_dom, uint32_t *parent_res, unsigned long long *adj,
                      uint8_t *__restrict__ first, const int *__restrict__ flags, int dil_cap, const int *__restrict__ cell_edge) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    if (flags[1]) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int j = blockIdx.x * kPairWarps + warp;
    if (j >= n_atoms) return;
    const int dil_bytes = (dil_cap + 7) & ~7, ent_bytes = 2 * ((dil_cap + 3) & ~3);
    unsigned char *base = dyn_smem + (size_t)(dil_bytes + ent_bytes + 128 + 24 * kPairCand + 8 * kPairList) * warp;
    uint32_t *dil32 = reinterpret_cast<uint32_t *>(base);
    const uint8_t *dil = base;
    uint16_t *ent = reinterpret_cast<uint16_t *>(base + dil_bytes);
    uint32_t *dup = reinterpret_cast<uint32_t *>(base + dil_bytes + ent_bytes);
    const int4 me = info[j];
    const uint32_t e0 = offset[j];
    const int n = (int)(offset[j + 1] - e0);
    if (!me.w) {
        for (int e = lane; e < n; e += 32) first[e0 + e] = 0;
        return;
    }
    const unsigned long long bx = abox[j];
    const int uc0 = (int)(bx >> 40), ur0 = (int)((bx >> 26) & 0x3fffu), us0 = (int)((bx >> 12) & 0x3fffu);
    const int D0 = (int)((bx >> 8) & 15u), D1 = (int)((bx >> 4) & 15u), D2 = (int)(bx & 15u);
    const int G0 = D0 + 2, G1 = D1 + 2, G2 = D2 + 2, gvol = G0 * G1 * G2;
    const int fc = uc0 - 1, fr = ur0 - 1, fs = us0 - 1;  // corner of the grown box
    // the loads of j's own entries are issued first and used after the cell look-up below, whose round trip they share
    unsigned long long own_key = 0ull;
    uint32_t own_lab = 0u;
    if (lane < n) {
        own_key = e_key[e0 + lane];
        own_lab = e_lab[e0 + lane];
    }
    // the 27 cells around j, one lane each: head of the cell's chain of atoms
    uint32_t i = kAggNil;
    if (lane < 27) {
        const int E = max(cell_edge[atom_map[j]], 1);
        const int cc = uc0 / E + lane / 9 - 1, cr = ur0 / E + (lane / 3) % 3 - 1, cs = us0 / E + lane % 3 - 1;
        if (cc >= 0 && cr >= 0 && cs >= 0) {
            const uint32_t map_id = (uint32_t)atom_map[j];
            const unsigned long long key = cell_key(map_id, (uint32_t)cc, (uint32_t)cr, (uint32_t)cs);
            uint64_t rbase;
            uint32_t size;
            atom_region(maps, map_id, rbase, size);
            uint32_t h = agg_start(key, size);
            for (;;) {
                const uint4 sl = __ldg(reinterpret_cast<const uint4 *>(aslot + rbase + h));
                const unsigned long long k = ((unsigned long long)sl.y << 32) | sl.x;
                if (k == key) {
                    i = sl.z;
                    break;
                }
                if (k == kAggEmpty) break;
                h = h + 1 == size ? 0 : h + 1;
            }
        }
    }
    for (int w = lane; w < (gvol + 3) / 4; w += 32) dil32[w] = 0u;
    for (int w = lane; w < (gvol + 1) / 2; w += 32) reinterpret_cast<uint32_t *>(ent)[w] = 0u;
    dup[lane] = 0u;
    __syncwarp();
    for (int e = lane; e < n; e += 32) {
        const unsigned long long key = e < 32 ? own_key : e_key[e0 + e];
        const int x = (int)((key >> (2 * kKeyBits)) & 0x3fffu) - fc, y = (int)((key >> kKeyBits) & 0x3fffu) - fr, z = (int)(key & 0x3fffu) - fs;
        const int p = (x * G1 + y) * G2 + z;
        ent[p] = (uint16_t)(e + 1);
        const uint32_t m = 1u << (e < 32 ? own_lab : (uint32_t)e_lab[e0 + e]);
#pragma unroll
        for (int dc = -1; dc <= 1; ++dc)
#pragma unroll
            for (int dr = -1; dr <= 1; ++dr)
#pragma unroll
                for (int ds = -1; ds <= 1; ++ds) {
                    const int q = p + (dc * G1 + dr) * G2 + ds;
                    atomicOr(dil32 + (q >> 2), m << (8 * (q & 3)));
                }
    }
    __syncwarp();
    // Phase A: the 27 cells around j, one lane each; contributing atoms i < j whose box touches j's go to the warp's candidate
    // list together with what phase B needs of them (all of a chain element's loads are independent: one round trip per element).
    // Phase B: candidates four at a time, lanes over a candidate's entries (coalesced loads, four candidates in flight).
    uint32_t *cand = dup + 32;  // kPairCand x 6 words: atom, first entry, entries, first cloud id, residue, index inside the residue
    int ncand = 0;
    uint2 *plist = reinterpret_cast<uint2 *>(cand + 6 * kPairCand);
    int npair = 0;
    unsigned long long adj_j = 0ull;  // atoms of j's residue whose clouds touch j's (warp-uniform)
    // Pairs are united lane-parallel, two lanes per pair (domain forest / residue forest): a union-find operation is half a dozen
    // dependent loads, and doing them one pair after the other was 4 of the kernel's 19 ms.  (Recording the pairs in a global
    // edge list and uniting them in a kernel of their own, one thread per edge, was slower in total: 10.8 + 5.2 ms against 14.9 ms.)
    auto drain = [&]() {
        __syncwarp();
        // The first pair goes ahead of the others: an atom's pairs mostly lead into ONE set (its residue, the chain so far), and
        // once the first has hooked the atom's cloud under that set's root the others see "same parent" after one round trip
        // instead of walking both trees and colliding on the same atomicMin.
        if (lane < 2 && npair > 0) {
            const uint2 pr = plist[0];
            const uint32_t ci = pr.x & 0x7fffffffu;
            if (lane == 0)
                uf_union_cached(parent_dom, ci, pr.y);
            else if (pr.x >> 31)
                uf_union_cached(parent_res, ci, pr.y);
        }
        __syncwarp();
        for (int t = lane + 2; t < 2 * npair; t += 32) {
            const uint2 pr = plist[t >> 1];
            const uint32_t ci = pr.x & 0x7fffffffu;
            if (!(t & 1))
                uf_union_cached(parent_dom, ci, pr.y);
            else if (pr.x >> 31)
                uf_union_cached(parent_res, ci, pr.y);
        }
        __syncwarp();
        npair = 0;
    };
    auto flush = [&]() {
        __syncwarp();
        for (int c0 = 0; c0 < ncand; c0 += 4) {
            unsigned long long key[4];
            uint32_t lab[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                key[u] = 0ull;
                lab[u] = 0u;
                if (c0 + u < ncand) {
                    const uint32_t ei0 = cand[6 * (c0 + u) + 1], ni = cand[6 * (c0 + u) + 2];
                    if ((uint32_t)lane < ni) {
                        key[u] = e_key[ei0 + lane];
                        lab[u] = e_lab[ei0 + lane];
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (c0 + u >= ncand) break;  // warp-uniform
                const uint32_t *cd = cand + 6 * (c0 + u);
                const uint32_t i = cd[0], ei0 = cd[1], ni = cd[2];
                uint32_t plo = 0u, phi = 0u;  // bit 8 * (cloud of i) + (cloud of j), as two words
                for (uint32_t eb = 0; eb < ni; eb += 32) {
                    unsigned long long k = key[u];
                    uint32_t l = lab[u];
                    const bool live = eb + lane < ni;
                    if (eb > 0 && live) {  // more than 32 entries: the rest is loaded here
                        k = e_key[ei0 + eb + lane];
                        l = e_lab[ei0 + eb + lane];
                    }
                    if (live) {
                        const int x = (int)((k >> (2 * kKeyBits)) & 0x3fffu) - fc, y = (int)((k >> kKeyBits) & 0x3fffu) - fr,
                                  z = (int)(k & 0x3fffu) - fs;
                        if ((unsigned)x < (unsigned)G0 && (unsigned)y < (unsigned)G1 && (unsigned)z < (unsigned)G2) {
                            const int p = (x * G1 + y) * G2 + z;
                            const uint32_t m = dil[p];
                            if (m) {
                                if (l < 4)
                                    plo |= m << (8 * l);
                                else
                                    phi |= m << (8 * (l - 4));
                                const uint32_t en = ent[p];
                                if (en) atomicOr(dup + ((en - 1) >> 5), 1u << ((en - 1) & 31));
                            }
                        }
                    }
                }
                plo = __reduce_or_sync(kFull, plo);
                phi = __reduce_or_sync(kFull, phi);
                if (!(plo | phi)) continue;
                const bool same_res = cd[4] == (uint32_t)me.y;
                // the (cloud of i, cloud of j) pairs go to the warp's pair list; they are united lane-parallel (drain) so that the
                // dependent loads of one union-find operation overlap those of the others instead of following them
                const int nlo = __popc(plo), nhi = __popc(phi);
                if (npair + nlo + nhi > kPairList) drain();
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t w = h ? phi : plo;
                    if ((w >> lane) & 1u) {
                        const int bit = 32 * h + lane;
                        const int at = npair + (h ? nlo : 0) + __popc(w & ((1u << lane) - 1u));
                        plist[at] = make_uint2((cd[3] + (uint32_t)(bit >> 3)) | (same_res ? 0x80000000u : 0u), (uint32_t)me.x + (uint32_t)(bit & 7));
                    }
                }
                npair += nlo + nhi;
                if (same_res) {
                    adj_j |= 1ull << cd[5];
                    if (lane == 0) atomicOr(adj + i, 1ull << me.z);  // result unused: a fire-and-forget reduction
                }
            }
        }
        __syncwarp();
        ncand = 0;
    };
    {
        while (__any_sync(kFull, i != kAggNil)) {
            bool take = false;
            uint32_t cur = i, ei0 = 0u, ei1 = 0u;
            int4 other = make_int4(0, 0, 0, 0);
            if (i != kAggNil) {
                const uint32_t nx = anext[i];
                if ((int)i < j) {
                    other = info[i];
                    const unsigned long long bi = abox[i];
                    ei0 = offset[i];
                    ei1 = offset[i + 1];
                    const int ic0 = (int)(bi >> 40), ir0 = (int)((bi >> 26) & 0x3fffu), is0 = (int)((bi >> 12) & 0x3fffu);
                    take = other.w && !(ic0 > uc0 + D0 || uc0 > ic0 + (int)((bi >> 8) & 15u) || ir0 > ur0 + D1 || ur0 > ir0 + (int)((bi >> 4) & 15u) ||
                                        is0 > us0 + D2 || us0 > is0 + (int)(bi & 15u));
                }
                i = nx;
            }
            const unsigned tm = __ballot_sync(kFull, take);
            if (take) {
                uint32_t *cd = cand + 6 * (ncand + __popc(tm & ((1u << lane) - 1u)));
                cd[0] = cur;
                cd[1] = ei0;
                cd[2] = ei1 - ei0;
                cd[3] = (uint32_t)other.x;
                cd[4] = (uint32_t)other.y;
                cd[5] = (uint32_t)other.z;
            }
            ncand += __popc(tm);
            if (ncand > kPairCand - 32) flush();
        }
        flush();
        drain();  // once per atom (or when the pair list fills): every drain is a chain of dependent union-find loads
    }
    __syncwarp();
    if (lane == 0 && adj_j) atomicOr(adj + j, adj_j);
    for (int e = lane; e < n; e += 32) first[e0 + e] = ((dup[e >> 5] >> (e & 31)) & 1u) ? 0 : 1;
}

__global__ void __launch_bounds__(kAggThreads) slot_clear_kernel(AggSlot *slot, int64_t n, const int *__restrict__ flags) {
    if (!flags[1]) return;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        slot[i].key = kAggEmpty;
        slot[i].head = kAggNil;
    }
}

// Electrons of every merged cloud: the sum over the DISTINCT atoms that have a cloud in it (blob.atoms after merge,
// pdb_eda/ccp4.py:582).  One thread per contributing atom; the atom's clouds are consecutive ids.
__global__ void __launch_bounds__(kAggThreads)
    cloud_roots_kernel(int n_atoms, const double *__restrict__ atom_out, const uint32_t *__restrict__ cloud_start,
                       const double *__restrict__ atom_electrons, uint32_t *parent_dom, uint32_t *parent_res,
                       double *elec_dom, double *elec_res) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n_atoms) return;
    if (atom_out[(int64_t)a * 8 + 7] == 0.0) return;
    const uint32_t c0 = cloud_start[a], c1 = cloud_start[a + 1];
    const double e = atom_electrons[a];
    for (uint32_t c = c0; c < c1; ++c) {
        const uint32_t rd = uf_find(parent_dom, c), rr = uf_find(parent_res, c);
        bool seen_d = false, seen_r = false;
        for (uint32_t p = c0; p < c; ++p) {  // an earlier cloud of this atom already brought the atom into that merged cloud
            seen_d |= uf_find(parent_dom, p) == rd;
            seen_r |= uf_find(parent_res, p) == rr;
        }
        if (!seen_d) atomicAdd(elec_dom + rd, e);
        if (!seen_r) atomicAdd(elec_res + rr, e);
    }
}

// Per structure (one CTA each, fixed-order reductions): distinct pool voxels and their density sum (numVoxelsAggregated,
// totalAggregatedDensity), merged clouds and their electrons (totalAggregatedElectrons; residue / domain clouds with at
// least min_cloud_electrons, pdb_eda/densityAnalysis.py:681, :722), and the completeness flag of every contributing atom.
__global__ void __launch_bounds__(kSummaryThreads)
    map_summary_kernel(const pe_batch_map *__restrict__ maps, const uint32_t *__restrict__ offset, const float *__restrict__ e_val,
                       const uint8_t *__restrict__ first, double *__restrict__ atom_out, const uint32_t *__restrict__ cloud_start,
                       const uint32_t *__restrict__ parent_dom, const uint32_t *__restrict__ parent_res,
                       const double *__restrict__ elec_dom, const double *__restrict__ elec_res,
                       const int32_t *__restrict__ atom_residue, const unsigned long long *__restrict__ atom_bonded,
                       const unsigned long long *__restrict__ adj, const unsigned long long *__restrict__ res_mask,
                       double min_cloud_electrons, double *__restrict__ map_out) {
    __shared__ double scratch[kSummaryThreads / 32];
    const pe_batch_map *m = maps + blockIdx.x;
    const int a0 = m->atom_begin, a1 = m->atom_end;
    double *mo = map_out + (int64_t)blockIdx.x * 8;
    // voxels (both loads of an entry are issued whatever the flag says, four entries per thread in flight: with the density load
    // behind the flag test the largest structure's 2,700 dependent iterations were 2.7 of the kernel's 3 ms)
    double nvox = 0.0, dens = 0.0;
    {
        const uint32_t e1 = offset[a1];
#pragma unroll 4
        for (uint32_t i = offset[a0] + threadIdx.x; i < e1; i += kSummaryThreads) {
            const uint8_t f = first[i];
            const float v = e_val[i];
            nvox += f ? 1.0 : 0.0;
            dens += f ? (double)v : 0.0;
        }
    }
    nvox = block_sum_fixed(nvox, scratch);
    dens = block_sum_fixed(dens, scratch);
    // merged clouds
    double n_dom = 0.0, n_dom_min = 0.0, n_res = 0.0, n_res_min = 0.0, elec = 0.0;
    for (uint32_t c = cloud_start[a0] + threadIdx.x; c < cloud_start[a1]; c += blockDim.x) {
        if (parent_dom[c] == c) {  // a root points at itself whether or not the tree below it is flat
            n_dom += 1.0;
            elec += elec_dom[c];
            if (elec_dom[c] >= min_cloud_electrons) n_dom_min += 1.0;
        }
        if (parent_res[c] == c) {
            n_res += 1.0;
            if (elec_res[c] >= min_cloud_electrons) n_res_min += 1.0;
        }
    }
    n_dom = block_sum_fixed(n_dom, scratch);
    n_dom_min = block_sum_fixed(n_dom_min, scratch);
    n_res = block_sum_fixed(n_res, scratch);
    n_res_min = block_sum_fixed(n_res_min, scratch);
    elec = block_sum_fixed(elec, scratch);
    // completeness (:653-659): every bonded atom of the residue that contributes must touch this atom
    for (int a = a0 + threadIdx.x; a < a1; a += blockDim.x) {
        double *rec = atom_out + (int64_t)a * 8;
        if (rec[7] == 0.0) continue;
        const unsigned long long need = atom_bonded[a] & res_mask[atom_residue[a]];
        rec[7] = (need & ~adj[a]) == 0ull ? 3.0 : 1.0;  // bit 0: contributes, bit 1: completely overlapped
    }
    if (threadIdx.x == 0) {
        mo[0] = nvox;
        mo[1] = dens;
        mo[2] = elec;
        mo[3] = n_dom;
        mo[4] = n_dom_min;
        mo[5] = n_res;
        mo[6] = n_res_min;
    }
}

__global__ void __launch_bounds__(kAggThreads) iota_kernel(int64_t n, uint32_t *a, uint32_t *b) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        a[i] = (uint32_t)i;
        b[i] = (uint32_t)i;
    }
}

static int agg_grid(int64_t n) {
    int64_t blocks = (n + kAggThreads - 1) / kAggThreads;
    const int64_t max_blocks = (int64_t)sm_count() * 16;
    if (blocks < 1) blocks = 1;
    return (int)(blocks < max_blocks ? blocks : max_blocks);
}

struct AggLayout {
    int64_t cloud_count, cloud_start, scan, key, val, atom, lab, node, first, slots, info, parent_dom, parent_res, elec_dom,
        elec_res, adj, res_mask, flags, abox, aslot, anext, cell_edge, total;
};

static AggLayout agg_layout(int64_t n_atoms, int64_t n_entries, int64_t n_residues, int64_t n_maps) {
    AggLayout L;
    int64_t p = 0;
    auto take = [&](int64_t bytes) {
        const int64_t at = p;
        p += align_up(bytes > 0 ? bytes : 1, 256);
        return at;
    };
    const int64_t cap = 2 * n_entries + 16 * n_maps;  // slots: every structure's region is twice its cloud voxels (+ 16)
    L.flags = take(256);
    L.cloud_count = take((n_atoms + 1) * 4);
    L.cloud_start = take((n_atoms + 1) * 4);
    L.scan = take(scan_ws_bytes(n_atoms + 1));
    L.key = take(n_entries * 8);
    L.val = take(n_entries * 4);
    L.atom = take(n_entries * 4);
    L.lab = take(n_entries * 2);
    L.node = take(n_entries * 8);
    L.first = take(n_entries);
    L.slots = take(cap * 16);
    L.info = take(n_atoms * 16);
    L.parent_dom = take(n_entries * 4);
    L.parent_res = take(n_entries * 4);
    L.elec_dom = take(n_entries * 8);
    L.elec_res = take(n_entries * 8);
    L.adj = take(n_atoms * 8);
    L.res_mask = take(n_residues * 8);
    L.abox = take(n_atoms * 8);
    L.aslot = take((2 * n_atoms + 16 * n_maps) * 16);  // atom grid of the pair path: every structure's region is twice its atoms (+ 16)
    L.anext = take(n_atoms * 4);
    L.cell_edge = take(n_maps * 4);  // per structure: widest cloud bounding box edge = edge of its atom grid's cells
    L.total = p;
    return L;
}

}  // namespace pe

using namespace pe;

extern "C" {

int64_t pe_cloud_workspace_bytes(int64_t n_atoms, int64_t n_entries, int64_t n_residues, int64_t n_maps) {
    if (n_atoms < 0 || n_entries < 0 || n_residues < 0 || n_maps < 0) return -1;
    return agg_layout(n_atoms, n_entries, n_residues, n_maps).total;
}

int pe_cloud_count(int32_t n_maps, const pe_batch_map *d_maps, int32_t n_atoms, const int32_t *d_atom_map, const double *d_xyz,
                   const float *d_radius, uint32_t *d_offset, int64_t *d_totals, void *d_scan_ws, uint32_t *d_box_bits, void *stream) {
    PE_CHECK_ARG(n_maps >= 0 && n_atoms >= 0 && d_totals, "pe_cloud_count: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    PE_CUDA(cudaMemsetAsync(d_totals, 0, 2 * sizeof(int64_t), st));
    if (n_atoms == 0) return PE_OK;
    PE_CHECK_ARG(d_maps && d_atom_map && d_xyz && d_radius && d_offset && d_scan_ws, "pe_cloud_count: null pointer");
    PE_CHECK_ARG(n_maps < (1 << 20), "pe_cloud_count: at most 2^20 structures per batch");
    // counts are written into d_offset and scanned in place (n_atoms + 1 entries, the last one zero)
    PE_CUDA(cudaMemsetAsync(d_offset + n_atoms, 0, sizeof(uint32_t), st));
    const int blocks = (n_atoms + kSphereWarps * kCountAtoms - 1) / (kSphereWarps * kCountAtoms);
    PE_LAUNCH("cloud_count_kernel", st, cloud_count_kernel<<<blocks, kSphereWarps * 32, 0, st>>>(
        d_maps, n_atoms, d_atom_map, d_xyz, d_radius, d_offset, (unsigned long long *)(d_totals + 1), d_box_bits));
    PE_LAUNCH_CHECK();
    return exclusive_scan_u32(d_offset, d_offset, (int64_t)n_atoms + 1, nullptr, d_totals, d_scan_ws, st, false);
}

int pe_cloud_aggregate(int32_t n_maps, const pe_batch_map *d_maps, int32_t n_atoms, const int32_t *d_atom_map, const double *d_xyz,
                       const float *d_radius, const int32_t *d_atom_residue, const int32_t *d_atom_local,
                       const uint64_t *d_atom_bonded, const double *d_atom_electrons, int32_t n_residues, const uint32_t *d_offset,
                       int64_t n_entries, int32_t max_box_voxels, double min_cloud_electrons, const uint32_t *d_box_bits,
                       double *d_atom_out, double *d_map_out, void *d_ws, void *stream) {
    PE_CHECK_ARG(n_maps >= 0 && n_atoms >= 0 && n_residues >= 0 && n_entries >= 0, "pe_cloud_aggregate: negative size");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_maps == 0) return PE_OK;
    PE_CHECK_ARG(d_maps && d_map_out && d_ws, "pe_cloud_aggregate: null pointer");
    PE_CUDA(cudaMemsetAsync(d_map_out, 0, (size_t)n_maps * 8 * sizeof(double), st));
    if (n_atoms == 0) return PE_OK;
    PE_CHECK_ARG(d_atom_map && d_xyz && d_radius && d_atom_residue && d_atom_local && d_atom_bonded && d_atom_electrons && d_offset &&
                     d_atom_out,
                 "pe_cloud_aggregate: null pointer");
    PE_CHECK_ARG(n_entries < (1ll << 31), "pe_cloud_aggregate: too many cloud voxels in one batch");
    PE_CHECK_ARG(max_box_voxels > 0 && max_box_voxels <= 16384, "pe_cloud_aggregate: atom boxes of %d voxels are not supported (1..16384)",
                 max_box_voxels);
    const AggLayout L = agg_layout(n_atoms, n_entries, n_residues, n_maps);
    char *ws = (char *)d_ws;
    int *d_bad = (int *)(ws + L.flags);
    uint32_t *cloud_count = (uint32_t *)(ws + L.cloud_count);
    uint32_t *cloud_start = (uint32_t *)(ws + L.cloud_start);
    unsigned long long *e_key = (unsigned long long *)(ws + L.key);
    float *e_val = (float *)(ws + L.val);
    uint32_t *e_atom = (uint32_t *)(ws + L.atom);
    uint16_t *e_lab = (uint16_t *)(ws + L.lab);
    uint8_t *first = (uint8_t *)(ws + L.first);
    AggTable t;
    t.slot = (AggSlot *)(ws + L.slots);
    t.offset = d_offset;
    t.maps = d_maps;
    t.node = (uint2 *)(ws + L.node);
    int4 *info = (int4 *)(ws + L.info);
    uint32_t *parent_dom = (uint32_t *)(ws + L.parent_dom), *parent_res = (uint32_t *)(ws + L.parent_res);
    double *elec_dom = (double *)(ws + L.elec_dom), *elec_res = (double *)(ws + L.elec_res);
    unsigned long long *adj = (unsigned long long *)(ws + L.adj), *res_mask = (unsigned long long *)(ws + L.res_mask);
    const int64_t cap = 2 * n_entries + 16 * (int64_t)n_maps;

    unsigned long long *abox = (unsigned long long *)(ws + L.abox);
    AggSlot *aslot = (AggSlot *)(ws + L.aslot);
    uint32_t *anext = (uint32_t *)(ws + L.anext);
    int *cell_edge = (int *)(ws + L.cell_edge);
    // shared-memory frame of the pair kernel: the largest box grown by one voxel on every side (an atom whose grown box is larger
    // sends the batch down the hash-table path)
    int dil_cap = 5 * max_box_voxels + 64;
    if (dil_cap > 4096) dil_cap = 4096;

    PE_CUDA(cudaMemsetAsync(d_bad, 0, 256, st));
    {
        // PE_CLOUD_FORCE_HASH=1 sends every batch down the hash-table path (tests compare the two paths)
        const char *force = getenv("PE_CLOUD_FORCE_HASH");
        if (force && force[0] == '1') PE_CUDA(cudaMemsetAsync(d_bad + 1, 1, 1, st));
    }
    PE_CUDA(cudaMemsetAsync(cell_edge, 0, (size_t)n_maps * sizeof(int), st));
    PE_CUDA(cudaMemsetAsync(aslot, 0xff, (size_t)(2 * (int64_t)n_atoms + 16 * (int64_t)n_maps) * sizeof(AggSlot), st));
    PE_CUDA(cudaMemsetAsync(elec_dom, 0, (size_t)(n_entries > 0 ? n_entries : 1) * 8, st));
    PE_CUDA(cudaMemsetAsync(elec_res, 0, (size_t)(n_entries > 0 ? n_entries : 1) * 8, st));
    PE_CUDA(cudaMemsetAsync(adj, 0, (size_t)n_atoms * 8, st));
    PE_CUDA(cudaMemsetAsync(res_mask, 0, (size_t)(n_residues > 0 ? n_residues : 1) * 8, st));

    // pass 1: clouds of every atom
    const int nw_max = (max_box_voxels + 31) / 32;
    const size_t per_warp = (size_t)nw_max * 8 + (size_t)((max_box_voxels + 1) / 2 * 2) * 6;
    int warps = (int)((size_t)(160 * 1024) / per_warp);
    if (warps > kSphereWarps) warps = kSphereWarps;
    PE_CHECK_ARG(warps >= 1, "pe_cloud_aggregate: a box of %d voxels needs %zu bytes of shared memory", max_box_voxels, per_warp);
    const size_t smem = per_warp * warps;
    PE_CUDA(cudaFuncSetAttribute(cloud_fill_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    {
        FillArgs fa;
        fa.maps = d_maps;
        fa.n_atoms = n_atoms;
        fa.atom_map = d_atom_map;
        fa.xyz = d_xyz;
        fa.radius = d_radius;
        fa.offset = d_offset;
        fa.max_box = max_box_voxels;
        fa.e_key = e_key;
        fa.e_val = e_val;
        fa.e_atom = e_atom;
        fa.e_lab = e_lab;
        fa.n_clouds = cloud_count;
        fa.atom_out = d_atom_out;
        fa.d_bad = d_bad;
        fa.abox = abox;
        fa.box_bits = d_box_bits;
        fa.cell_edge = cell_edge;
        fa.dil_cap = dil_cap;
        const int per_block = warps * kFillAtoms;
        PE_LAUNCH("cloud_fill_kernel", st, cloud_fill_kernel<<<(n_atoms + per_block - 1) / per_block, warps * 32, smem, st>>>(fa, warps, per_warp));
    }
    PE_LAUNCH("cutoff_kernel", st, cutoff_kernel<<<n_maps, kSummaryThreads, 0, st>>>(d_maps, d_atom_out, d_map_out));
    // pass 2: contributing atoms, cloud ids
    PE_LAUNCH("accept_kernel", st, accept_kernel<<<(n_atoms + 1 + kAggThreads - 1) / kAggThreads, kAggThreads, 0, st>>>(
        d_maps, n_atoms, d_atom_map, d_atom_residue, d_atom_local, d_atom_out, d_map_out, cloud_count, res_mask));
    PE_LAUNCH_CHECK();
    if (int rc = exclusive_scan_u32(cloud_count, cloud_start, (int64_t)n_atoms + 1, nullptr, nullptr, ws + L.scan, st, false)) return rc;
    if (n_entries > 0) {
        const int grid = agg_grid(n_entries);
        PE_LAUNCH("iota_kernel", st, iota_kernel<<<grid, kAggThreads, 0, st>>>(n_entries, parent_dom, parent_res));
        PE_LAUNCH("atom_info_kernel", st, atom_info_kernel<<<(n_atoms + kAggThreads - 1) / kAggThreads, kAggThreads, 0, st>>>(
            n_atoms, cloud_start, d_atom_residue, d_atom_local, d_atom_out, info));
        // pair path (atom grid + one warp per atom); the hash-table kernels return at once unless cloud_fill_kernel flagged the batch
        PE_LAUNCH("atom_cell_insert_kernel", st, atom_cell_insert_kernel<<<(n_atoms + kAggThreads - 1) / kAggThreads, kAggThreads, 0, st>>>(
            d_maps, n_atoms, d_atom_map, info, abox, aslot, anext, d_bad, cell_edge));
        {
            const size_t pair_smem = (size_t)(((dil_cap + 7) & ~7) + 2 * ((dil_cap + 3) & ~3) + 128 + 24 * kPairCand + 8 * kPairList) * kPairWarps;
            PE_CUDA(cudaFuncSetAttribute(cloud_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pair_smem));
            PE_LAUNCH("cloud_pair_kernel", st, cloud_pair_kernel<<<(n_atoms + kPairWarps - 1) / kPairWarps, kPairWarps * 32, pair_smem, st>>>(
                d_maps, n_atoms, d_atom_map, d_offset, e_key, e_lab, info, abox, aslot, anext, parent_dom, parent_res, adj, first, d_bad, dil_cap, cell_edge));
        }
        PE_LAUNCH("slot_clear_kernel", st, slot_clear_kernel<<<grid, kAggThreads, 0, st>>>(t.slot, cap, d_bad));
        PE_LAUNCH("pool_insert_kernel", st, pool_insert_kernel<<<grid, kAggThreads, 0, st>>>(n_entries, e_key, e_atom, d_atom_out, t, d_bad));
        PE_LAUNCH("cloud_merge_kernel", st, cloud_merge_kernel<<<grid, kAggThreads, 0, st>>>(n_entries, e_key, e_lab, info, t, parent_dom,
                                                                                           parent_res, adj, d_bad));
        PE_LAUNCH("cloud_first_kernel", st, cloud_first_kernel<<<grid, kAggThreads, 0, st>>>(n_entries, e_key, info, t, first, d_bad));
    }
    PE_LAUNCH("cloud_roots_kernel", st, cloud_roots_kernel<<<(n_atoms + kAggThreads - 1) / kAggThreads, kAggThreads, 0, st>>>(
        n_atoms, d_atom_out, cloud_start, d_atom_electrons, parent_dom, parent_res, elec_dom, elec_res));
    PE_LAUNCH("map_summary_kernel", st, map_summary_kernel<<<n_maps, kSummaryThreads, 0, st>>>(
        d_maps, d_offset, e_val, first, d_atom_out, cloud_start, parent_dom, parent_res, elec_dom, elec_res, d_atom_residue,
        (const unsigned long long *)d_atom_bonded, adj, res_mask, min_cloud_electrons, d_map_out));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

/* Non-zero when the last pe_cloud_aggregate on this workspace met an index outside the key range or an inconsistent
 * count (synchronises the stream). */
int pe_cloud_status(const void *d_ws, void *stream, int32_t *bad) {
    PE_CHECK_ARG(d_ws && bad, "pe_cloud_status: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const AggLayout L = agg_layout(0, 0, 0, 0);
    PE_CUDA(cudaMemcpyAsync(bad, (const char *)d_ws + L.flags, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaStreamSynchronize(st));
    return PE_OK;
}

}  // extern "C"
