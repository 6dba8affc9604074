// pe_sphere.cu -- per-atom sphere enumeration, density gather-sum and voxel lists.
//
// Replaces (batched over atoms):
//   getSphereCrsFromXyz / getSphereCrsFromXyzList        pdb_eda/cutils.pyx:220-271
//   _testXyzWithinDistance                               pdb_eda/cutils.pyx:205-218
//   testValidXyz / testValidXyzList                      pdb_eda/cutils.pyx:273-313
//   DensityMatrix.getTotalDensityFromXyz                 pdb_eda/ccp4.py:418-435
//   findAberrantBlobs(atom) clustering (createCrsLists)  pdb_eda/ccp4.py:437-461, pdb_eda/cutils.pyx:44-70
//
// Design (B200): the work per in-sphere voxel is one 4-byte gather, so these kernels are bounded by instruction
// issue (float64 membership tests, float64 accumulation) and L2 gathers long before HBM; everything is arranged to
// keep the per-candidate instruction count minimal:
//   * in orthogonal cells the squared distance separates per axis:  d2 = fl(fl(X2 + Y2) + Z2)  where each term
//     is the already-rounded square the reference forms, so the per-axis squares and the wrapped memory offsets
//     are tabulated once per atom in shared memory and a candidate costs one DADD + one DSETP;
//   * sqrt is never evaluated:  sqrt_rn(d2) <= r  <=>  d2 <= T(r)  (sphere_threshold);
//   * along a box row the in-sphere columns are one interval: it is guessed from the sphere's chord in float32 and
//     proved with four exact float64 tests (row_chord), so a box row costs ~4 tests instead of one per candidate;
//   * per-atom kernel: four atoms per warp (8 lanes each, lanes walk box rows) while the boxes are at most 8 wide
//     (atom-type radii); larger boxes take one warp per atom with lanes along the column axis (contiguous in memory);
//   * union kernel (persistent CTAs walk the groups): row chords OR-ed into a shared-memory bitmap, which is then
//     compacted into a list of map offsets and gathered densely, once per voxel of the union (see sphere_union_kernel);
//   * warp-shuffle / fixed-order block reductions make the float64 sums run-to-run deterministic.
// Skewed cells take generic passes that evaluate the reference's 3x3 mat-vec per candidate in the host BLAS's
// accumulation order.
#include <float.h>
#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <stddef.h>
#include <type_traits>
#include "pe_common.cuh"
#include "pe_sphere_dev.cuh"

namespace pe {

int launch_union_warp(const pe_geom *g, const float *d_rho, int n_groups, const int32_t *d_group_start, const double *d_xyz,
                      const float *d_radius, int32_t *box, double *thr, float cut_pos, float cut_neg, int *d_counter, double *d_out,
                      int n_quad_atoms, const float *d_atom_radius, double *d_out_atoms, cudaStream_t st);  // pe_union.cu

// ------------------------------------------------------------------------------------------------ sums kernel
// CASEB: the column axis carries z (the last term of the reference's sum), so fl(X2 + Y2) depends on (row, section).
template <bool CASEB>
__device__ __forceinline__ void sums_ortho(const pe_geom &g, const float *__restrict__ rho, const AtomBox &b, double ax,
                                           double ay, double az, double T, const AxisTab *tab, int lane, float cp,
                                           float cn, SphereAcc &acc) {
    // inner axis = the crs axis that carries z when that is the row or section axis; else sections.
    const int inner = CASEB ? 2 : g.map2xyz[2];       // 1 (rows) or 2 (sections)
    const int outer = 3 - inner;
    const AxisTab &ti = tab[inner - 1];
    const AxisTab &to = tab[outer - 1];
    const int Di = sel3(b.dim[0], b.dim[1], b.dim[2], inner), Do = sel3(b.dim[0], b.dim[1], b.dim[2], outer), D0 = b.dim[0];
    int d0p = 1;
    while (d0p < D0 && d0p < 32) d0p <<= 1;
    const int rpi = 32 / d0p;  // box rows handled per warp iteration
    const int lrow = lane / d0p, lc = lane % d0p;
    for (int cbase = 0; cbase < D0; cbase += 32) {
        const int ic = cbase + lc;
        const bool act = ic < D0;
        const int c = b.lo[0] + ic;
        const double sqc = act ? axis_sq(g, 0, c, ax, ay, az) : 0.0;
        const int offc = act ? axis_off(g, 0, c) : kInvalidOff;
        for (int ko0 = 0; ko0 < Do; ko0 += rpi) {  // warp-uniform trip count (the ballot below needs every lane)
            const int ko = ko0 + lrow;
            const bool rowact = act && ko < Do;
            const double sqo = rowact ? to.sq[ko] : 0.0;
            const int offo = rowact ? to.off[ko] : kInvalidOff;
            const double P = __dadd_rn(sqc, sqo);  // fl(X2 + Y2) when !CASEB
            const int offco = offc | offo;
            const int sumco = (int)((unsigned)offc + (unsigned)offo);
#pragma unroll 2
            for (int ki = 0; ki < Di; ++ki) {
                const double sqi = ti.sq[ki];
                const int offi = ti.off[ki];
                const double d2 = CASEB ? __dadd_rn(__dadd_rn(sqo, sqi), sqc) : __dadd_rn(P, sqi);
                const bool inside = rowact && (d2 <= T);
                if (!__any_sync(kFull, inside)) continue;  // most of a box lies outside its sphere: nothing to gather
                const bool ok = (offco | offi) >= 0;
                float v = 0.f;
                if (inside && ok) v = __ldg(rho + (int)((unsigned)sumco + (unsigned)offi));
                acc.bad |= (inside && !ok) ? 1 : 0;
                acc.add(inside, v, cp, cn);
            }
        }
    }
}

__device__ __forceinline__ void sums_generic(const pe_geom &g, const float *__restrict__ rho, const AtomBox &b, double ax,
                                             double ay, double az, double T, int lane, float cp, float cn, SphereAcc &acc) {
    const int D0 = b.dim[0], D1 = b.dim[1], D2 = b.dim[2];
    const int64_t vol = (int64_t)D0 * D1 * D2;
    for (int64_t m = lane; m < vol; m += 32) {
        const int ic = (int)(m % D0);
        const int64_t t = m / D0;
        const int ir = (int)(t % D1), is = (int)(t / D1);
        const int c = b.lo[0] + ic, r = b.lo[1] + ir, s = b.lo[2] + is;
        double vx, vy, vz;
        crs2xyz(g, c, r, s, vx, vy, vz);
        bool inside = dist2(ax, ay, az, vx, vy, vz) <= T;
        if (!inside) continue;
        const int oc = axis_off(g, 0, c), orr = axis_off(g, 1, r), os = axis_off(g, 2, s);
        const bool ok = (oc | orr | os) >= 0;
        const float v = ok ? __ldg(rho + (oc + orr + os)) : 0.f;
        acc.bad |= (inside && !ok) ? 1 : 0;
        acc.add(inside, v, cp, cn);
    }
}

// One atom by one warp: tabulated separable squares (orthogonal cells) or the generic per-candidate pass.
template <int MODE>
__device__ __forceinline__ void sums_one_atom(const pe_geom &g, const float *__restrict__ rho, int a, const double *__restrict__ xyz,
                                              const float *__restrict__ radius, float cp, float cn, AxisTab *tab, int lane,
                                              double *__restrict__ out) {
    const double ax = xyz[3 * a], ay = xyz[3 * a + 1], az = xyz[3 * a + 2];
    AtomBox b;
    double T;
    atom_box(g, ax, ay, az, radius[a], b, T);
    SphereAcc acc;
    const bool tabulated = g.orthogonal && b.dim[0] <= kDMax * 32 && b.dim[1] <= kDMax && b.dim[2] <= kDMax;
    if (tabulated) {
        fill_tables(g, b, ax, ay, az, tab, lane);
        sums_ortho<MODE == 2>(g, rho, b, ax, ay, az, T, tab, lane, cp, cn, acc);
    } else {
        sums_generic(g, rho, b, ax, ay, az, T, lane, cp, cn, acc);
    }
    const int n_all = warp_sum(acc.n_all), n_pos = warp_sum(acc.n_pos), n_neg = warp_sum(acc.n_neg);
    const int bad = warp_sum(acc.bad);
    const double s_all = warp_sum(acc.s_all), s_pos = warp_sum(acc.s_pos), s_neg = warp_sum(acc.s_neg);
    if (lane == 0) {
        double *o = out + (int64_t)a * PE_SPHERE_NOUT;
        o[0] = (double)n_all;
        o[1] = s_all;
        o[2] = (double)n_pos;
        o[3] = s_pos;
        o[4] = (double)n_neg;
        o[5] = s_neg;
        o[6] = bad ? 0.0 : 1.0;
        o[7] = (double)b.dim[0] * (double)b.dim[1] * (double)b.dim[2];
    }
    __syncwarp();  // the tables are refilled for the warp's next atom
}

// Per-atom sums.  A warp takes kAtomsPerWarp = 4 consecutive atoms: 8 lanes per atom (quad_sums, pe_sphere_dev.cuh) when all four
// boxes are at most kSmallDim wide in an orthogonal cell; otherwise the warp handles its atoms one after the other with all
// 32 lanes (sums_one_atom).
template <int MODE>
__global__ void __launch_bounds__(kSphereWarps * 32)
    sphere_sums_kernel(const __grid_constant__ pe_geom g, const float *__restrict__ rho, int n_atoms,
                       const double *__restrict__ xyz, const float *__restrict__ radius, float cp, float cn,
                       double *__restrict__ out /* n_atoms x PE_SPHERE_NOUT */) {
    __shared__ AxisTab tabs[kSphereWarps][2];
    __shared__ SmallTab stab[kSphereWarps][kAtomsPerWarp];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int a0 = (blockIdx.x * kSphereWarps + warp) * kAtomsPerWarp;
    if (a0 >= n_atoms) return;
    cp = eff_pos(cp);
    cn = eff_neg(cn);
    if (quad_sums<MODE>(g, rho, n_atoms, a0, xyz, radius, cp, cn, stab[warp], lane, out)) return;
    for (int q = 0; q < kAtomsPerWarp && a0 + q < n_atoms; ++q)
        sums_one_atom<MODE>(g, rho, a0 + q, xyz, radius, cp, cn, tabs[warp], lane, out);
}

// ------------------------------------------------------------------------------------------------ union kernel
// Set-union of the spheres of one group of atoms (getSphereCrsFromXyzList, pdb_eda/cutils.pyx:250-271; the region
// density / discrepancy sums of pdb_eda/densityAnalysis.py:1037-1068, :1160-1211).  One CTA per group, two phases
// per tile of the group's bounding box (tiles of 64 columns x 40 rows x 40 sections; a residue at the reference's
// default 3.5 A radius is one tile):
//   1. membership: every warp walks its share of every atom's box rows and ORs the in-sphere columns of a box row
//      into a shared-memory bitmap (two 32-bit words per (row, section)) -- one ballot and one or two atomicOr per
//      warp iteration, no global memory traffic.  OR is commutative, so no ordering between atoms is needed.
//   2. gather: the set bits are compacted into a list of map offsets, which the warps then walk densely
//      (union_gather).  Each voxel of the union is read exactly once however many spheres hold it, and the float64
//      summation order is fixed, so results are run-to-run deterministic.
constexpr int kUnionWarps = 4;
constexpr int kTileC = 64, kTileR = 40, kTileS = 40;

constexpr int kUnionChunk = 8;       // atoms whose tables are resident at once

struct UnionShared {
    uint32_t bits[kTileR * kTileS * 2];
    double sqC[kUnionChunk][kTileC];  // per atom of the chunk: squares along the tile's columns / rows / sections
    double sqR[kUnionChunk][kTileR];  // (only the part of the atom's box that lies inside the tile)
    double sqS[kUnionChunk][kTileS];
    double T[kUnionChunk];
    int offC[kTileC], offR[kTileR], offS[kTileS];  // wrapped element offsets of the tile's indices
    int cLo[kUnionChunk], nC[kUnionChunk], rLo[kUnionChunk], nR[kUnionChunk], sLo[kUnionChunk], nS[kUnionChunk];
    int kMin[kUnionChunk];             // column (index into sqC) nearest the atom: the minimum of its sqC
    float xC[kUnionChunk];             // the atom's fractional column, as an index into sqC (interval guess only)
};

// Membership of one chunk of atoms in one tile: a work item is one box row (row, section) of one atom; its in-sphere
// columns (row_chord: ~4 exact float64 tests per box row instead of one per candidate voxel) are OR-ed into the bitmap.
template <int MODE, bool WIDE>
__device__ __forceinline__ void union_mark_rows(UnionShared &sh, int nchunk, int tid, int nthreads, float inv_gl) {
    for (int j = 0; j < nchunk; ++j) {  // block-uniform
        const int nR = sh.nR[j], nS = sh.nS[j], nC = sh.nC[j];
        if (nR <= 0) continue;
        // items of this atom: its box rows, laid out with the section count padded to a power of two (no division)
        const int shift = nS > 1 ? 32 - __clz(nS - 1) : 0;
        const int total = nR << shift;
        const double T = sh.T[j];
        const double *sqc = sh.sqC[j];
        // the column nearest the atom: the box's centre column or, after rounding, one of its neighbours
        int km = sh.kMin[j];
        if (km > 0 && sqc[km - 1] < sqc[km]) --km;
        else if (km + 1 < nC && sqc[km + 1] < sqc[km]) ++km;
        const float xc = sh.xC[j];
        const int cbit = sh.cLo[j];
        uint32_t *rows = sh.bits + 2 * (sh.rLo[j] * kTileS + sh.sLo[j]);
        for (int li = tid; li < total; li += nthreads) {
            const int is = li & ((1 << shift) - 1), ir = li >> shift;
            if (is >= nS) continue;
            const double sr = sh.sqR[j][ir], ss = sh.sqS[j][is];
            const double A = (MODE == 0) ? ss : ((MODE == 1) ? sr : __dadd_rn(sr, ss));
            const double B = (MODE == 0) ? sr : ss;
            int kl, kh;
            if (!row_chord<MODE>(sqc, nC, km, xc, inv_gl, A, B, T, kl, kh)) continue;  // the row misses the sphere
            const int count = kh - kl + 1;
            uint32_t *word = rows + 2 * (ir * kTileS + is);
            if (WIDE) {
                const unsigned long long run = count >= 64 ? ~0ull : ((1ull << count) - 1ull);
                const unsigned long long wide = run << (cbit + kl);
                const uint32_t wlo = (uint32_t)wide, whi = (uint32_t)(wide >> 32);
                if (wlo) atomicOr(word, wlo);
                if (whi) atomicOr(word + 1, whi);
            } else {  // the tile is at most 32 columns wide
                const uint32_t run = count >= 32 ? ~0u : ((1u << count) - 1u);
                atomicOr(word, run << (cbit + kl));
            }
        }
    }
}

__device__ __forceinline__ void union_mark_generic(const pe_geom &g, const AtomBox &b, double ax, double ay, double az,
                                                   double T, int tid, int nthreads, int tc0, int tr0, int ts0, int tC, int tR,
                                                   int tS, uint32_t *bits) {
    const int c_lo = max(b.lo[0], tc0), c_hi = min(b.lo[0] + b.dim[0], tc0 + tC);
    const int r_lo = max(b.lo[1], tr0), r_hi = min(b.lo[1] + b.dim[1], tr0 + tR);
    const int s_lo = max(b.lo[2], ts0), s_hi = min(b.lo[2] + b.dim[2], ts0 + tS);
    if (c_lo >= c_hi || r_lo >= r_hi || s_lo >= s_hi) return;
    const int nc = c_hi - c_lo, n1 = r_hi - r_lo;
    const int vol = nc * n1 * (s_hi - s_lo);
    for (int m = tid; m < vol; m += nthreads) {
        const int ic = m % nc, t = m / nc;
        const int c = c_lo + ic, r = r_lo + t % n1, s = s_lo + t / n1;
        double vx, vy, vz;
        crs2xyz(g, c, r, s, vx, vy, vz);
        if (!(dist2(ax, ay, az, vx, vy, vz) <= T)) continue;
        const int cb = c - tc0;
        atomicOr(bits + 2 * ((r - tr0) * kTileS + (s - ts0)) + (cb >> 5), 1u << (cb & 31));
    }
}

// Phase 2 of the union kernel: compact, then gather densely.  The bitmap rows of the tile are taken 32 at a time, one
// (row, section) per lane.  Compaction: a warp prefix sum of the popcounts gives every row its place in a per-warp
// list in shared memory, and each lane writes the map offsets of its set bits there -- consecutive entries are
// consecutive columns of a row, then the next row.  Gather: the warp walks the list with every lane busy and
// kGatherLoads independent loads in flight per lane, each load covering a few contiguous runs of the map.  The voxel
// count comes from the popcounts, so the per-voxel work is one conversion, the float64 additions and the class tests.
// The list lives in the storage of the (now dead) membership tables; when a batch holds more voxels than the list,
// its rows are taken in as many rounds as needed (a word never exceeds the list).  64-column tiles pass each batch
// twice, once per 32-column half.  The summation order is fixed, so results are run-to-run deterministic.
// (Tried: 64 bitmap rows per warp iteration -- the warps of a block finish further apart, 173 -> 185 us; batches handed
// out on demand through a shared counter -- no faster, and the summation order is no longer fixed.)
constexpr int kGatherLoads = 8;
constexpr int kListCap = kUnionChunk * (kTileC + kTileR + kTileS) * 2 / kUnionWarps;  // ints per warp

template <bool WIDE, bool CHECKED, bool HASNEG>
__device__ __forceinline__ void union_gather(UnionShared &sh, const float *__restrict__ rho, SphereAcc &acc, float cp, float cn,
                                             int warp, int lane, int tR, int tS) {
    static_assert(offsetof(UnionShared, sqR) == offsetof(UnionShared, sqC) + sizeof(double) * kUnionChunk * kTileC, "table layout");
    static_assert(offsetof(UnionShared, sqS) == offsetof(UnionShared, sqR) + sizeof(double) * kUnionChunk * kTileR, "table layout");
    static_assert(kListCap >= 32, "a word must fit the list");
    int *list = reinterpret_cast<int *>(&sh.sqC[0][0]) + warp * kListCap;
    const int nwords = tR * tS;
    // wi / tS by multiplication: exact for wi < 2^11 and tS <= 2^6 (wi * tS < 2^20, no 32-bit overflow)
    const unsigned div_tS = ((1u << 20) + (unsigned)tS - 1u) / (unsigned)tS;
    static_assert(kTileR * kTileS < (1 << 11) && kTileS <= 64, "magic division by tS");
    for (int w0 = warp * 32; w0 < nwords; w0 += kUnionWarps * 32) {
        const int wi = w0 + lane;
        const int rl = (int)(((unsigned)wi * div_tS) >> 20), sl = wi - rl * tS;
        uint2 mine = make_uint2(0u, 0u);
        uint32_t *wordp = sh.bits + 2 * (rl * kTileS + sl);
        if (wi < nwords) mine = *reinterpret_cast<const uint2 *>(wordp);
        if (!__any_sync(kFull, (mine.x | mine.y) != 0u)) continue;
        if ((mine.x | mine.y) != 0u) *reinterpret_cast<uint2 *>(wordp) = make_uint2(0u, 0u);  // leave the bitmap clear
        int orr = 0, osum = 0;
        if (wi < nwords) {
            const int o1 = sh.offR[rl], o2 = sh.offS[sl];
            orr = o1 | o2;
            osum = (int)((unsigned)o1 + (unsigned)o2);
        }
#pragma unroll
        for (int half = 0; half < (WIDE ? 2 : 1); ++half) {
            uint32_t w = half ? mine.y : mine.x;
            if (WIDE && !__any_sync(kFull, w != 0u)) continue;
            const int *offc = sh.offC + 32 * half;
            const int oc0 = offc[0];
            const int c = __popc(w);
            bool pending = c > 0;
            while (true) {  // one round unless the batch overflows the list
                const int cc = pending ? c : 0;
                const int excl = warp_excl_scan(cc, lane);
                const bool fits = excl + cc <= kListCap;
                const int total = __reduce_max_sync(kFull, fits ? excl + cc : 0);
                if (pending && fits) {
                    int *dst = list + excl;
                    if (CHECKED) {
                        while (w) {
                            const int bcol = __ffs((int)w) - 1;
                            w &= w - 1u;
                            const int oc = offc[bcol];
                            *dst++ = ((orr | oc) < 0) ? -1 : (int)((unsigned)osum + (unsigned)oc);
                        }
                    } else {  // every index of the tile is stored and its columns are adjacent in memory
                        const int rowbase = (int)((unsigned)osum + (unsigned)oc0);
                        while (w) {
                            const int bcol = __ffs((int)w) - 1;
                            w &= w - 1u;
                            *dst++ = rowbase + bcol;
                        }
                    }
                    pending = false;
                }
                __syncwarp();
                if (lane == 0) acc.n_all += total;
                for (int i0 = 0; i0 < total; i0 += 32 * kGatherLoads) {
                    int e[kGatherLoads];
                    float v[kGatherLoads];
#pragma unroll
                    for (int u = 0; u < kGatherLoads; ++u) {
                        const int idx = i0 + 32 * u + lane;
                        e[u] = idx < total ? list[idx] : -2;
                    }
#pragma unroll
                    for (int u = 0; u < kGatherLoads; ++u) {
                        v[u] = 0.f;
                        if (e[u] >= 0) v[u] = __ldg(rho + e[u]);
                        if (CHECKED) acc.bad |= (e[u] == -1) ? 1 : 0;
                    }
#pragma unroll
                    for (int u = 0; u < kGatherLoads; ++u) {
                        if (HASNEG)
                            acc.add(false, v[u], cp, cn);
                        else
                            acc.add_pos(false, v[u], cp);
                    }
                }
                __syncwarp();  // the list is rewritten by the next round / half / batch
                if (!__any_sync(kFull, pending)) break;
            }
        }
    }
}

// Diagnostic: SM cycles spent per phase, summed over all CTAs of the launches since the last read
// (prologue, membership, gather, epilogue); read and reset with pe_sphere_union_cycles().
// Compiled in with -DPE_UNION_PHASE_CYCLES=1 only: the four 64-bit accumulators and the time mark are live across the whole
// kernel, and with 64 registers per thread they cost the hot loops registers (163.2 -> 160.9 us without them; pe_sphere_union_cycles() then reads zeros).
#ifndef PE_UNION_PHASE_CYCLES
#define PE_UNION_PHASE_CYCLES 0
#endif
__device__ unsigned long long g_union_cycles[4];

template <int MODE>
__global__ void __launch_bounds__(kUnionWarps * 32, 7)
    sphere_union_kernel(const __grid_constant__ pe_geom g, const float *__restrict__ rho, int n_groups,
                        const int32_t *__restrict__ group_start, const double *__restrict__ xyz,
                        const float *__restrict__ radius, int32_t *box, double *thr, float cp, float cn,
                        double *__restrict__ out /* n_groups x PE_SPHERE_NOUT */) {
    __shared__ UnionShared sh;
    __shared__ double red_d[kUnionWarps][3];
    __shared__ int red_i[kUnionWarps][4];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#if PE_UNION_PHASE_CYCLES
    long long t_mark = clock64();
    long long t_phase[4] = {0, 0, 0, 0};
#endif
    cp = eff_pos(cp);
    cn = eff_neg(cn);
    const float inv_gl = (float)(1.0 / g.grid_length[g.map2crs[0]]);  // columns per Angstrom (interval guess only)
    // persistent CTAs: the bitmap is cleared once (the gather leaves it clear), then groups are taken round robin
    for (int i = tid; i < kTileR * kTileS * 2; i += blockDim.x) sh.bits[i] = 0u;
    for (int grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
    const int a0 = group_start[grp], a1 = group_start[grp + 1];
    // boxes and distance thresholds of the group's atoms (into the workspace arrays: any group size)
    for (int a = a0 + tid; a < a1; a += blockDim.x) {
        AtomBox bb;
        double tt;
        atom_box(g, xyz[3 * a], xyz[3 * a + 1], xyz[3 * a + 2], radius[a], bb, tt);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            box[6 * a + k] = bb.lo[k];
            box[6 * a + 3 + k] = bb.dim[k];
        }
        thr[a] = tt;
    }
    __syncthreads();  // boxes visible block-wide; the previous group's reduction scratch has been consumed
    // the group's bounding box
    int ulo0 = INT_MAX, ulo1 = INT_MAX, ulo2 = INT_MAX, uhi0 = INT_MIN, uhi1 = INT_MIN, uhi2 = INT_MIN;
    double candidates = 0.0;
    for (int a = a0; a < a1; ++a) {
        const int32_t *bx = box + 6 * a;
        const int d0 = bx[3], d1 = bx[4], d2 = bx[5];
        candidates += (double)d0 * (double)d1 * (double)d2;
        if (d0 <= 0 || d1 <= 0 || d2 <= 0) continue;
        ulo0 = min(ulo0, bx[0]);
        ulo1 = min(ulo1, bx[1]);
        ulo2 = min(ulo2, bx[2]);
        uhi0 = max(uhi0, bx[0] + d0);
        uhi1 = max(uhi1, bx[1] + d1);
        uhi2 = max(uhi2, bx[2] + d2);
    }
    SphereAcc acc;
    if (uhi0 > ulo0) {
        for (int ts0 = ulo2; ts0 < uhi2; ts0 += kTileS)
            for (int tr0 = ulo1; tr0 < uhi1; tr0 += kTileR)
                for (int tc0 = ulo0; tc0 < uhi0; tc0 += kTileC) {
                    const int tC = min(kTileC, uhi0 - tc0), tR = min(kTileR, uhi1 - tr0), tS = min(kTileS, uhi2 - ts0);
                    for (int k = tid; k < tC; k += blockDim.x) sh.offC[k] = axis_off(g, 0, tc0 + k);
                    for (int k = tid; k < tR; k += blockDim.x) sh.offR[k] = axis_off(g, 1, tr0 + k);
                    for (int k = tid; k < tS; k += blockDim.x) sh.offS[k] = axis_off(g, 2, ts0 + k);
                    __syncthreads();  // bitmap is clear, offsets are in place
#if PE_UNION_PHASE_CYCLES
                    {
                        const long long now = clock64();
                        t_phase[0] += now - t_mark;
                        t_mark = now;
                    }
#endif
                    // phase 1: membership
                    if (g.orthogonal) {
                        for (int c0 = a0; c0 < a1; c0 += kUnionChunk) {
                            const int nchunk = min(kUnionChunk, a1 - c0);
                            if (tid < nchunk) {  // the part of each atom's box inside the tile (tile-relative)
                                const int32_t *bx = box + 6 * (c0 + tid);
                                const bool any = bx[3] > 0 && bx[4] > 0 && bx[5] > 0;
                                const int cl = max(bx[0], tc0), ch = min(bx[0] + bx[3], tc0 + tC);
                                const int rl = max(bx[1], tr0), rh = min(bx[1] + bx[4], tr0 + tR);
                                const int sl = max(bx[2], ts0), shh = min(bx[2] + bx[5], ts0 + tS);
                                const bool hit = any && cl < ch && rl < rh && sl < shh;
                                sh.cLo[tid] = cl - tc0;
                                sh.nC[tid] = hit ? ch - cl : 0;
                                sh.rLo[tid] = rl - tr0;
                                sh.nR[tid] = hit ? rh - rl : 0;
                                sh.sLo[tid] = sl - ts0;
                                sh.nS[tid] = hit ? shh - sl : 0;
                                sh.T[tid] = thr[c0 + tid];
                                // centre column of the box (range(c - R - 1, c + R + 1): c = lo + dim / 2), clamped into the tile part
                                sh.kMin[tid] = hit ? min(max(bx[0] + bx[3] / 2 - cl, 0), ch - cl - 1) : 0;
                                const int ic = g.map2crs[0];  // xyz axis carried by the columns
                                sh.xC[tid] = (float)((sel3(xyz[3 * (c0 + tid)], xyz[3 * (c0 + tid) + 1], xyz[3 * (c0 + tid) + 2], ic) -
                                                      g.origin[ic]) / g.grid_length[ic] - (double)cl);
                            }
                            __syncthreads();
                            for (int idx = tid; idx < nchunk * (kTileC + kTileR + kTileS); idx += blockDim.x) {
                                const int j = idx / (kTileC + kTileR + kTileS), e = idx - j * (kTileC + kTileR + kTileS);
                                const int a = c0 + j;
                                const double ax = xyz[3 * a], ay = xyz[3 * a + 1], az = xyz[3 * a + 2];
                                if (e < kTileC) {
                                    if (e < sh.nC[j]) sh.sqC[j][e] = axis_sq(g, 0, tc0 + sh.cLo[j] + e, ax, ay, az);
                                } else if (e < kTileC + kTileR) {
                                    const int k = e - kTileC;
                                    if (k < sh.nR[j]) sh.sqR[j][k] = axis_sq(g, 1, tr0 + sh.rLo[j] + k, ax, ay, az);
                                } else {
                                    const int k = e - kTileC - kTileR;
                                    if (k < sh.nS[j]) sh.sqS[j][k] = axis_sq(g, 2, ts0 + sh.sLo[j] + k, ax, ay, az);
                                }
                            }
                            __syncthreads();
                            if (tC > 32)
                                union_mark_rows<MODE, true>(sh, nchunk, tid, blockDim.x, inv_gl);
                            else
                                union_mark_rows<MODE, false>(sh, nchunk, tid, blockDim.x, inv_gl);
                            __syncthreads();  // tables are reused by the next chunk
                        }
                    } else {
                        for (int a = a0; a < a1; ++a) {
                            AtomBox b;
#pragma unroll
                            for (int k = 0; k < 3; ++k) {
                                b.lo[k] = box[6 * a + k];
                                b.dim[k] = box[6 * a + 3 + k];
                            }
                            if (b.dim[0] <= 0 || b.dim[1] <= 0 || b.dim[2] <= 0) continue;
                            union_mark_generic(g, b, xyz[3 * a], xyz[3 * a + 1], xyz[3 * a + 2], thr[a], tid, blockDim.x, tc0, tr0,
                                               ts0, tC, tR, tS, sh.bits);
                        }
                    }
                    __syncthreads();
#if PE_UNION_PHASE_CYCLES
                    {
                        const long long now = clock64();
                        t_phase[1] += now - t_mark;
                        t_mark = now;
                    }
#endif
                    // phase 2: gather every voxel of the union once (union_gather), specialised on the tile width
                    // (32- or 64-bit bitmap rows), on whether every index of the tile is covered by the stored map
                    // (no validity logic in the loop) and on whether the negative class is in use.
                    {
                        const bool wide = tC > 32;
                        const bool has_neg = cn > __int_as_float(0xff800000);
                        int invalid = 0;
                        for (int k = tid; k < tC + tR + tS; k += blockDim.x) {
                            invalid |= (k < tC ? sh.offC[k] : (k < tC + tR ? sh.offR[k - tC] : sh.offS[k - tC - tR])) < 0 ? 1 : 0;
                            if (k > 0 && k < tC) invalid |= (sh.offC[k] != sh.offC[k - 1] + 1) ? 1 : 0;
                        }
                        // tiles that straddle the periodic boundary (columns not adjacent in memory) take the checked path too
                        const bool checked = __syncthreads_or(invalid) != 0;
                        const int sel = (wide ? 4 : 0) | (checked ? 2 : 0) | (has_neg ? 1 : 0);
                        switch (sel) {
                            case 0: union_gather<false, false, false>(sh, rho, acc, cp, cn, warp, lane, tR, tS); break;
                            case 1: union_gather<false, false, true>(sh, rho, acc, cp, cn, warp, lane, tR, tS); break;
                            case 2: union_gather<false, true, false>(sh, rho, acc, cp, cn, warp, lane, tR, tS); break;
                            case 3: union_gather<false, true, true>(sh, rho, acc, cp, cn, warp, lane, tR, tS); break;
                            case 4: union_gather<true, false, false>(sh, rho, acc, cp, cn, warp, lane, tR, tS); break;
                            case 5: union_gather<true, false, true>(sh, rho, acc, cp, cn, warp, lane, tR, tS); break;
                            case 6: union_gather<true, true, false>(sh, rho, acc, cp, cn, warp, lane, tR, tS); break;
                            default: union_gather<true, true, true>(sh, rho, acc, cp, cn, warp, lane, tR, tS); break;
                        }
                    }
                    __syncthreads();
#if PE_UNION_PHASE_CYCLES
                    {
                        const long long now = clock64();
                        t_phase[2] += now - t_mark;
                        t_mark = now;
                    }
#endif
                }
    }
    const int n_all = warp_sum(acc.n_all), n_pos = warp_sum(acc.n_pos), n_neg = warp_sum(acc.n_neg);
    const int bad = warp_sum(acc.bad);
    const double s_all = warp_sum(acc.s_all), s_pos = warp_sum(acc.s_pos), s_neg = warp_sum(acc.s_neg);
    if (lane == 0) {
        red_i[warp][0] = n_all;
        red_i[warp][1] = n_pos;
        red_i[warp][2] = n_neg;
        red_i[warp][3] = bad;
        red_d[warp][0] = s_all;
        red_d[warp][1] = s_pos;
        red_d[warp][2] = s_neg;
    }
    __syncthreads();
    if (tid == 0) {
        int ni[4] = {0, 0, 0, 0};
        double sd[3] = {0.0, 0.0, 0.0};
        for (int w = 0; w < kUnionWarps; ++w) {  // fixed order: deterministic
            for (int k = 0; k < 4; ++k) ni[k] += red_i[w][k];
            for (int k = 0; k < 3; ++k) sd[k] += red_d[w][k];
        }
        double *o = out + (int64_t)grp * PE_SPHERE_NOUT;
        o[0] = (double)ni[0];
        o[1] = sd[0];
        o[2] = (double)ni[1];
        o[3] = sd[1];
        o[4] = (double)ni[2];
        o[5] = sd[2];
        o[6] = ni[3] ? 0.0 : 1.0;
        o[7] = candidates;
    }
#if PE_UNION_PHASE_CYCLES
    {
        const long long now = clock64();
        t_phase[3] += now - t_mark;
        t_mark = now;
    }
#endif
    }  // next group
#if PE_UNION_PHASE_CYCLES
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) atomicAdd(g_union_cycles + k, (unsigned long long)t_phase[k]);
    }
#endif
}

// ------------------------------------------------------------------------------------------------ list kernels
__global__ void __launch_bounds__(kSphereWarps * 32)
    sphere_count_kernel(const __grid_constant__ pe_geom g, const float *__restrict__ rho, int n_atoms,
                        const double *__restrict__ xyz, const float *__restrict__ radius, float cutoff,
                        int32_t *__restrict__ count, int32_t *__restrict__ box_out) {
    __shared__ AxisTab tabs[kSphereWarps][2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int a = blockIdx.x * kSphereWarps + warp;
    if (a >= n_atoms) return;
    const double ax = xyz[3 * a], ay = xyz[3 * a + 1], az = xyz[3 * a + 2];
    AtomBox b;
    double T;
    atom_box(g, ax, ay, az, radius[a], b, T);
    int n = 0;
    for_each_inside(g, rho, b, ax, ay, az, T, tabs[warp], lane,
                    [&](int, int, int, bool, float v) { n += passes(v, cutoff) ? 1 : 0; });
    n = warp_sum(n);
    if (lane == 0) {
        count[a] = n;
        if (box_out) {
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                box_out[6 * a + k] = b.lo[k];
                box_out[6 * a + 3 + k] = b.dim[k];
            }
        }
    }
}

// Dynamic shared memory per warp: bits[nw] | pref[nw] | (labels only) pidx[maxbox] lab[maxbox] rnk[maxbox] as u16.
template <bool LABELS>
__global__ void sphere_fill_kernel(const __grid_constant__ pe_geom g, const float *__restrict__ rho, int n_atoms,
                                   const double *__restrict__ xyz, const float *__restrict__ radius, float cutoff,
                                   const int64_t *__restrict__ offset, int max_box, int32_t *__restrict__ out_index,
                                   float *__restrict__ out_value, int32_t *__restrict__ out_label) {
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    __shared__ AxisTab tabs[kSphereWarps][2];
    const int warps = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int a = blockIdx.x * warps + warp;
    if (a >= n_atoms) return;
    const int nw_max = (max_box + 31) / 32;
    const size_t per_warp = (size_t)nw_max * 8 + (LABELS ? (size_t)((max_box + 1) / 2 * 2) * 6 : 0);
    unsigned char *base = dyn_smem + per_warp * warp;
    uint32_t *bits = reinterpret_cast<uint32_t *>(base);
    uint32_t *pref = bits + nw_max;
    uint16_t *pidx = reinterpret_cast<uint16_t *>(pref + nw_max);
    uint16_t *lab = pidx + (max_box + 1) / 2 * 2;
    uint16_t *rnk = lab + (max_box + 1) / 2 * 2;

    const double ax = xyz[3 * a], ay = xyz[3 * a + 1], az = xyz[3 * a + 2];
    AtomBox b;
    double T;
    atom_box(g, ax, ay, az, radius[a], b, T);
    const int D1 = b.dim[1], D2 = b.dim[2];
    const int vol = b.dim[0] * D1 * D2;
    if (vol > max_box) return;  // caller's bound was wrong; the count pass reported the real box, nothing is written
    const int nw = (vol + 31) / 32;
    for (int w = lane; w < nw; w += 32) bits[w] = 0u;
    __syncwarp();
    // 1. membership bits in the reference's order: p = (ic*D1 + ir)*D2 + is
    for_each_inside(g, rho, b, ax, ay, az, T, tabs[warp], lane, [&](int ic, int ir, int is, bool, float v) {
        if (passes(v, cutoff)) {
            const int p = (ic * D1 + ir) * D2 + is;
            atomicOr(bits + (p >> 5), 1u << (p & 31));
        }
    });
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
    const int64_t obase = offset[a];
    // 3. ordered emission
    for (int w = lane; w < nw; w += 32) {
        uint32_t word = bits[w];
        int j = (int)pref[w];
        while (word) {
            const int bit = __ffs(word) - 1;
            word &= word - 1;
            const int p = w * 32 + bit;
            out_index[obase + j] = p;
            if (LABELS) pidx[j] = (uint16_t)p;
            if (out_value) {
                const int is = p % D2, t = p / D2, ir = t % D1, ic = t / D1;
                const int oc = axis_off(g, 0, b.lo[0] + ic), orr = axis_off(g, 1, b.lo[1] + ir), os = axis_off(g, 2, b.lo[2] + is);
                out_value[obase + j] = ((oc | orr | os) >= 0) ? __ldg(rho + (oc + orr + os)) : 0.f;
            }
            ++j;
        }
    }
    if (!LABELS) return;
    __syncwarp();
    // 4. 26-connected clusters of the listed voxels: min-label propagation with pointer jumping.
    for (int j = lane; j < n; j += 32) lab[j] = (uint16_t)j;
    __syncwarp();
    for (;;) {
        bool changed = false;
        for (int j = lane; j < n; j += 32) {
            const int p = pidx[j];
            const int is = p % D2, t = p / D2, ir = t % D1, ic = t / D1;
            int m = lab[j];
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
                        m = min(m, (int)lab[jn]);
                    }
                }
            }
            m = min(m, (int)lab[m]);
            if (m < (int)lab[j]) {
                lab[j] = (uint16_t)m;
                changed = true;
            }
        }
        __syncwarp();
        if (!__any_sync(kFull, changed)) break;
    }
    // 5. number the clusters by their first member (the order createCrsLists creates them in)
    int nroots = 0;
    for (int j0 = 0; j0 < n; j0 += 32) {
        const int j = j0 + lane;
        const int isroot = (j < n && lab[j] == j) ? 1 : 0;
        const int ex = warp_excl_scan(isroot, lane);
        if (isroot) rnk[j] = (uint16_t)(nroots + ex);
        nroots += __shfl_sync(kFull, ex + isroot, 31);
    }
    __syncwarp();
    for (int j = lane; j < n; j += 32) out_label[obase + j] = (int32_t)rnk[lab[j]];
}

}  // namespace pe

using namespace pe;

// Round 1's CTA-per-group kernel instead of the warp-per-group one, kept for A/B measurements.
static bool use_union_cta_kernel() {
    static const bool on = getenv("PE_UNION_CTA") != nullptr;
    return on;
}

// Whether every box of an atom whose radius is at most max_radius is at most kSmallDim wide, decided as atom_box decides a
// box: dim = 2 * R + 2 along each crs axis, with R from xyz2crs(origin + r) -- in an orthogonal cell
// rint(fl(fl(origin + r) - origin) / grid_length), which only grows with r.
static bool boxes_are_small(const pe_geom *g, float max_radius) {
    if (!g->orthogonal || !(max_radius <= FLT_MAX)) return false;  // skewed cell, NaN or infinite bound
    const double r = (double)max_radius;
    double R[3];
    for (int i = 0; i < 3; ++i) R[i] = nearbyint(((g->origin[i] + r) - g->origin[i]) / g->grid_length[i]);
    for (int k = 0; k < 3; ++k)
        if (2.0 * R[g->map2crs[k]] + 2.0 > (double)kSmallDim) return false;
    return true;
}

extern "C" {

int pe_sphere_union_cycles(unsigned long long *out4) {
    PE_CHECK_ARG(out4 != nullptr, "pe_sphere_union_cycles: null pointer");
    PE_CUDA(cudaMemcpyFromSymbol(out4, g_union_cycles, sizeof(unsigned long long) * 4));
    unsigned long long zero[4] = {0, 0, 0, 0};
    PE_CUDA(cudaMemcpyToSymbol(g_union_cycles, zero, sizeof(zero)));
    return PE_OK;
}

int64_t pe_sphere_workspace_bytes(int64_t n_atoms) {
    if (n_atoms < 0) n_atoms = 0;
    return align_up(n_atoms * 6 * 4, 256) + align_up(n_atoms * 8, 256) + align_up(n_atoms * 4, 256) +
           align_up(n_atoms * PE_SPHERE_NOUT * 8, 256);
}

int pe_sphere_sums(const pe_geom *g, const float *d_rho, int32_t n_atoms, const double *d_xyz, const float *d_radius,
                   int32_t n_groups, const int32_t *d_group_start, float cut_pos, float cut_neg, double *d_out,
                   void *d_ws, void *stream) {
    if (int rc = check_geom(g)) return rc;
    PE_CHECK_ARG(n_atoms >= 0 && n_groups >= 0, "pe_sphere_sums: negative size");
    if (n_atoms == 0 && n_groups == 0) return PE_OK;
    PE_CHECK_ARG(d_rho && d_xyz && d_radius && d_out && d_ws, "pe_sphere_sums: null pointer");
    PE_CHECK_ARG(d_group_start || n_groups == n_atoms, "pe_sphere_sums: n_groups must equal n_atoms without group offsets");
    PE_CHECK_ARG(!(cut_pos < 0.f) && !(cut_neg > 0.f), "pe_sphere_sums: cut_pos must be >= 0 and cut_neg <= 0");
    cudaStream_t st = (cudaStream_t)stream;
    char *ws = (char *)d_ws;
    int32_t *box = (int32_t *)ws;
    ws += align_up((int64_t)n_atoms * 6 * 4, 256);
    double *thr = (double *)ws;
    ws += align_up((int64_t)n_atoms * 8, 256);
    if (d_group_start == nullptr) {
        const int mode1 = g->map2xyz[2] == 1 ? 0 : (g->map2xyz[2] == 2 ? 1 : 2);  // crs axis that carries z
        const int sblocks = (n_atoms + kSphereWarps * kAtomsPerWarp - 1) / (kSphereWarps * kAtomsPerWarp);
        if (mode1 == 0)
            PE_LAUNCH("sphere_sums_kernel", st, sphere_sums_kernel<0><<<sblocks, kSphereWarps * 32, 0, st>>>(*g, d_rho, n_atoms, d_xyz, d_radius,
                                                                                                  cut_pos, cut_neg, d_out));
        else if (mode1 == 1)
            PE_LAUNCH("sphere_sums_kernel", st, sphere_sums_kernel<1><<<sblocks, kSphereWarps * 32, 0, st>>>(*g, d_rho, n_atoms, d_xyz, d_radius,
                                                                                                  cut_pos, cut_neg, d_out));
        else
            PE_LAUNCH("sphere_sums_kernel", st, sphere_sums_kernel<2><<<sblocks, kSphereWarps * 32, 0, st>>>(*g, d_rho, n_atoms, d_xyz, d_radius,
                                                                                                  cut_pos, cut_neg, d_out));
        PE_LAUNCH_CHECK();
        return PE_OK;
    }
    if (n_groups > 0 && !use_union_cta_kernel()) {
        int *counter = (int *)ws;  // third region of the workspace
        return launch_union_warp(g, d_rho, n_groups, d_group_start, d_xyz, d_radius, box, thr, cut_pos, cut_neg, counter, d_out, 0,
                                 nullptr, nullptr, st);
    }
    if (n_groups > 0) {
        const int mode = g->map2xyz[2] == 1 ? 0 : (g->map2xyz[2] == 2 ? 1 : 2);  // crs axis that carries z
        // persistent CTAs, 7 per SM (72 registers, no spills, 23 KB shared memory each).  Measured on C2: 6 / 7 / 8 per SM (78 / 72 /
        // 64 registers) 174 / 158.6 / 159.8 us; earlier in the round 5 / 6 / 7 / 8 / 9 per SM gave 210 / 189 / 173 / 170 / 175 us
        const int ugrid = min(n_groups, sm_count() * 7);
        if (mode == 0)
            PE_LAUNCH("sphere_union_kernel", st, sphere_union_kernel<0><<<ugrid, kUnionWarps * 32, 0, st>>>(
                *g, d_rho, n_groups, d_group_start, d_xyz, d_radius, box, thr, cut_pos, cut_neg, d_out));
        else if (mode == 1)
            PE_LAUNCH("sphere_union_kernel", st, sphere_union_kernel<1><<<ugrid, kUnionWarps * 32, 0, st>>>(
                *g, d_rho, n_groups, d_group_start, d_xyz, d_radius, box, thr, cut_pos, cut_neg, d_out));
        else
            PE_LAUNCH("sphere_union_kernel", st, sphere_union_kernel<2><<<ugrid, kUnionWarps * 32, 0, st>>>(
                *g, d_rho, n_groups, d_group_start, d_xyz, d_radius, box, thr, cut_pos, cut_neg, d_out));
    }
    PE_LAUNCH_CHECK();
    return PE_OK;
}

int pe_sphere_sums_atoms_and_groups(const pe_geom *g, const float *d_rho, int32_t n_atoms, const double *d_xyz,
                                    const float *d_atom_radius, float max_atom_radius, const float *d_group_radius, int32_t n_groups,
                                    const int32_t *d_group_start, float cut_pos, float cut_neg, double *d_out_atoms,
                                    double *d_out_groups, void *d_ws, void *stream) {
    if (int rc = check_geom(g)) return rc;
    PE_CHECK_ARG(n_atoms >= 0 && n_groups >= 0, "pe_sphere_sums_atoms_and_groups: negative size");
    if (n_atoms == 0 && n_groups == 0) return PE_OK;
    PE_CHECK_ARG(d_rho && d_xyz && d_atom_radius && d_group_radius && d_out_atoms && d_out_groups && d_ws,
                 "pe_sphere_sums_atoms_and_groups: null pointer");
    PE_CHECK_ARG(d_group_start || n_groups == n_atoms,
                 "pe_sphere_sums_atoms_and_groups: n_groups must equal n_atoms without group offsets");
    PE_CHECK_ARG(!(cut_pos < 0.f) && !(cut_neg > 0.f), "pe_sphere_sums_atoms_and_groups: cut_pos must be >= 0 and cut_neg <= 0");
    if (n_atoms > 0 && n_groups > 0 && d_group_start && !use_union_cta_kernel() && boxes_are_small(g, max_atom_radius)) {
        char *ws = (char *)d_ws;
        int32_t *box = (int32_t *)ws;
        ws += align_up((int64_t)n_atoms * 6 * 4, 256);
        double *thr = (double *)ws;
        ws += align_up((int64_t)n_atoms * 8, 256);
        return launch_union_warp(g, d_rho, n_groups, d_group_start, d_xyz, d_group_radius, box, thr, cut_pos, cut_neg, (int *)ws,
                                 d_out_groups, n_atoms, d_atom_radius, d_out_atoms, (cudaStream_t)stream);
    }
    if (int rc = pe_sphere_sums(g, d_rho, n_atoms, d_xyz, d_atom_radius, n_atoms, nullptr, cut_pos, cut_neg, d_out_atoms, d_ws, stream))
        return rc;
    return pe_sphere_sums(g, d_rho, n_atoms, d_xyz, d_group_radius, n_groups, d_group_start, cut_pos, cut_neg, d_out_groups, d_ws, stream);
}

int pe_sphere_count(const pe_geom *g, const float *d_rho, int32_t n_atoms, const double *d_xyz, const float *d_radius,
                    float cutoff, int32_t *d_count, int32_t *d_box, void *stream) {
    if (int rc = check_geom(g)) return rc;
    PE_CHECK_ARG(n_atoms >= 0, "pe_sphere_count: negative size");
    if (n_atoms == 0) return PE_OK;
    PE_CHECK_ARG(d_rho && d_xyz && d_radius && d_count, "pe_sphere_count: null pointer");
    const int blocks = (n_atoms + kSphereWarps - 1) / kSphereWarps;
    PE_LAUNCH("sphere_count_kernel", (cudaStream_t)stream, sphere_count_kernel<<<blocks, kSphereWarps * 32, 0, (cudaStream_t)stream>>>(*g, d_rho, n_atoms, d_xyz, d_radius, cutoff,
                                                                                d_count, d_box));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

int pe_sphere_fill(const pe_geom *g, const float *d_rho, int32_t n_atoms, const double *d_xyz, const float *d_radius,
                   float cutoff, const int64_t *d_offset, int32_t max_box_voxels, int32_t *d_index, float *d_value,
                   int32_t *d_label, void *stream) {
    if (int rc = check_geom(g)) return rc;
    PE_CHECK_ARG(n_atoms >= 0, "pe_sphere_fill: negative size");
    if (n_atoms == 0) return PE_OK;
    PE_CHECK_ARG(d_rho && d_xyz && d_radius && d_offset && d_index, "pe_sphere_fill: null pointer");
    PE_CHECK_ARG(max_box_voxels > 0, "pe_sphere_fill: max_box_voxels must be positive");
    const bool labels = d_label != nullptr;
    PE_CHECK_ARG(!labels || max_box_voxels <= 32768, "pe_sphere_fill: cluster labels need boxes of at most 32768 voxels (got %d)",
                 max_box_voxels);
    PE_CHECK_ARG(max_box_voxels <= (1 << 19), "pe_sphere_fill: boxes of more than 2^19 voxels are not supported (got %d)",
                 max_box_voxels);
    const int nw_max = (max_box_voxels + 31) / 32;
    const size_t per_warp = (size_t)nw_max * 8 + (labels ? (size_t)((max_box_voxels + 1) / 2 * 2) * 6 : 0);
    const size_t budget = 200 * 1024;
    int warps = (int)(budget / per_warp);
    if (warps > kSphereWarps) warps = kSphereWarps;
    PE_CHECK_ARG(warps >= 1, "pe_sphere_fill: box of %d voxels needs %zu bytes of shared memory per warp", max_box_voxels,
                 per_warp);
    const size_t smem = per_warp * warps;
    const int blocks = (n_atoms + warps - 1) / warps;
    cudaStream_t st = (cudaStream_t)stream;
    if (labels) {
        PE_CUDA(cudaFuncSetAttribute(sphere_fill_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        PE_LAUNCH("sphere_fill_kernel", st, sphere_fill_kernel<true><<<blocks, warps * 32, smem, st>>>(*g, d_rho, n_atoms, d_xyz, d_radius, cutoff, d_offset,
                                                                   max_box_voxels, d_index, d_value, d_label));
    } else {
        PE_CUDA(cudaFuncSetAttribute(sphere_fill_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        PE_LAUNCH("sphere_fill_kernel", st, sphere_fill_kernel<false><<<blocks, warps * 32, smem, st>>>(*g, d_rho, n_atoms, d_xyz, d_radius, cutoff, d_offset,
                                                                    max_box_voxels, d_index, d_value, d_label));
    }
    PE_LAUNCH_CHECK();
    return PE_OK;
}

}  // extern "C"
