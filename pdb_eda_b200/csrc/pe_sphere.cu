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
//   * grouped sums (the set-union of a group's spheres): one warp per group, row chords OR-ed into a shared-memory bitmap,
//     which is then compacted into a list of map offsets and gathered densely, once per voxel of the union (pe_union.cu);
//   * warp-shuffle reductions in a fixed order make the float64 sums run-to-run deterministic.
// Skewed cells take generic passes that evaluate the reference's 3x3 mat-vec per candidate in the host BLAS's
// accumulation order.
#include <float.h>
#include <math.h>
#include <stddef.h>
#include <type_traits>
#include "pe_common.cuh"
#include "pe_sphere_dev.cuh"

namespace pe {

int launch_union_warp(const pe_geom *g, const float *d_rho, int n_groups, const int32_t *d_group_start, const double *d_xyz,
                      const float *d_radius, int32_t *box, double *thr, float cut_pos, float cut_neg, int *d_counter, double *d_out,
                      int n_quad_atoms, const float *d_atom_radius, double *d_out_atoms, cudaStream_t st);  // pe_union.cu
int launch_batch_union(int n_maps, const pe_sums_map *d_maps, int n_groups, const int32_t *d_group_map, const int32_t *d_group_start,
                       const double *d_xyz, const float *d_radius, int32_t *box, double *thr, int *d_counter, double *d_out,
                       cudaStream_t st);  // pe_union.cu

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

// Per-atom sums of many structures, each on its own map (pe_batch_sphere_sums without group offsets).  The work items are the
// quads of sphere_sums_kernel counted from each structure's first atom, so that a quad never spans two structures and takes
// the same atoms as it does in a launch for its structure alone; flattened over the structures, they are dealt out to the
// warps in a fixed stride.  A quad whose atoms all name one valid map runs sphere_sums_kernel's code on it (quad_sums, or
// sums_one_atom atom by atom); otherwise every atom is summed alone on its own map, or gets a NaN row when that map index or
// its cutoffs are invalid.  The warp keeps the current map's pe_geom in shared memory.
__device__ __forceinline__ void copy_geom(pe_geom &dst, const pe_geom &src, int lane) {
    static_assert(sizeof(pe_geom) % 4 == 0, "pe_geom is copied as 32-bit words");
    __syncwarp();  // the previous geometry is no longer read
    for (int i = lane; i < (int)(sizeof(pe_geom) / 4); i += 32) reinterpret_cast<int *>(&dst)[i] = reinterpret_cast<const int *>(&src)[i];
    __syncwarp();
}

__device__ __forceinline__ bool sums_map_ok(int m, int n_maps, const pe_sums_map *maps) {
    return m >= 0 && m < n_maps && !(maps[m].cut_pos < 0.f) && !(maps[m].cut_neg > 0.f);
}

__global__ void __launch_bounds__(kSphereWarps * 32)
    batch_sphere_sums_kernel(int n_maps, const pe_sums_map *__restrict__ maps, const int32_t *__restrict__ atom_start,
                             const int32_t *__restrict__ group_map, const double *__restrict__ xyz, const float *__restrict__ radius,
                             double *__restrict__ out /* n_atoms x PE_SPHERE_NOUT */) {
    __shared__ AxisTab tabs[kSphereWarps][2];
    __shared__ SmallTab stab[kSphereWarps][kAtomsPerWarp];
    __shared__ pe_geom geoms[kSphereWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * kSphereWarps + warp, n_warps = (int64_t)gridDim.x * kSphereWarps;
    pe_geom &g = geoms[warp];
    int64_t q_base = 0;  // flattened index of structure k's first quad
    for (int k = 0; k < n_maps; ++k) {
        const int s0 = atom_start[k], s1 = atom_start[k + 1];
        const int64_t nq = s1 > s0 ? (s1 - s0 + kAtomsPerWarp - 1) / kAtomsPerWarp : 0;
        int64_t t = q_base + ((gw - q_base) % n_warps + n_warps) % n_warps;  // this warp's first quad at or after q_base
        for (; t < q_base + nq; t += n_warps) {
            const int a0 = s0 + (int)(t - q_base) * kAtomsPerWarp;
            const int m = group_map[a0];
            const int mq = (lane < kAtomsPerWarp && a0 + lane < s1) ? group_map[a0 + lane] : m;
            if (__all_sync(kFull, mq == m) && sums_map_ok(m, n_maps, maps)) {
                copy_geom(g, maps[m].geom, lane);
                const float *rho = maps[m].d_rho;
                const float cp = eff_pos(maps[m].cut_pos), cn = eff_neg(maps[m].cut_neg);
                const int mode = g.map2xyz[2] == 1 ? 0 : (g.map2xyz[2] == 2 ? 1 : 2);  // z_axis_mode, warp-uniform
                bool done;
                if (mode == 0)
                    done = quad_sums<0>(g, rho, s1, a0, xyz, radius, cp, cn, stab[warp], lane, out);
                else if (mode == 1)
                    done = quad_sums<1>(g, rho, s1, a0, xyz, radius, cp, cn, stab[warp], lane, out);
                else
                    done = quad_sums<2>(g, rho, s1, a0, xyz, radius, cp, cn, stab[warp], lane, out);
                if (done) continue;
            }
            for (int a = a0; a < min(a0 + kAtomsPerWarp, s1); ++a) {
                const int ma = group_map[a];
                if (!sums_map_ok(ma, n_maps, maps)) {
                    if (lane < PE_SPHERE_NOUT) out[(int64_t)a * PE_SPHERE_NOUT + lane] = __longlong_as_double(0x7ff8000000000000ll);
                    continue;
                }
                copy_geom(g, maps[ma].geom, lane);
                const float *rho = maps[ma].d_rho;
                const float cp = eff_pos(maps[ma].cut_pos), cn = eff_neg(maps[ma].cut_neg);
                const int mode = g.map2xyz[2] == 1 ? 0 : (g.map2xyz[2] == 2 ? 1 : 2);
                if (mode == 0)
                    sums_one_atom<0>(g, rho, a, xyz, radius, cp, cn, tabs[warp], lane, out);
                else if (mode == 1)
                    sums_one_atom<1>(g, rho, a, xyz, radius, cp, cn, tabs[warp], lane, out);
                else
                    sums_one_atom<2>(g, rho, a, xyz, radius, cp, cn, tabs[warp], lane, out);
            }
        }
        q_base += nq;
    }
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

// The sphere workspace, in 256-byte aligned regions: the atoms' boxes (6 int32 each: low corner, extents), their distance
// thresholds, and a slot of its own for the union kernel's work-item counter (grouped calls use it even when n_atoms == 0).
struct SphereWs {
    int32_t *box;
    double *thr;
    int *counter;
    static int64_t thr_at(int64_t n_atoms) { return align_up(n_atoms * 6 * 4, 256); }
    static int64_t counter_at(int64_t n_atoms) { return thr_at(n_atoms) + align_up(n_atoms * 8, 256); }
    static int64_t bytes(int64_t n_atoms) { return counter_at(n_atoms) + 256; }
    SphereWs(void *d_ws, int64_t n_atoms)
        : box((int32_t *)d_ws), thr((double *)((char *)d_ws + thr_at(n_atoms))), counter((int *)((char *)d_ws + counter_at(n_atoms))) {}
};

extern "C" {

int64_t pe_sphere_workspace_bytes(int64_t n_atoms) { return SphereWs::bytes(n_atoms < 0 ? 0 : n_atoms); }

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
    if (d_group_start == nullptr) {
        const int mode = z_axis_mode(g);
        const int sblocks = (n_atoms + kSphereWarps * kAtomsPerWarp - 1) / (kSphereWarps * kAtomsPerWarp);
        if (mode == 0)
            PE_LAUNCH("sphere_sums_kernel", st, sphere_sums_kernel<0><<<sblocks, kSphereWarps * 32, 0, st>>>(*g, d_rho, n_atoms, d_xyz, d_radius,
                                                                                                  cut_pos, cut_neg, d_out));
        else if (mode == 1)
            PE_LAUNCH("sphere_sums_kernel", st, sphere_sums_kernel<1><<<sblocks, kSphereWarps * 32, 0, st>>>(*g, d_rho, n_atoms, d_xyz, d_radius,
                                                                                                  cut_pos, cut_neg, d_out));
        else
            PE_LAUNCH("sphere_sums_kernel", st, sphere_sums_kernel<2><<<sblocks, kSphereWarps * 32, 0, st>>>(*g, d_rho, n_atoms, d_xyz, d_radius,
                                                                                                  cut_pos, cut_neg, d_out));
        PE_LAUNCH_CHECK();
        return PE_OK;
    }
    if (n_groups > 0) {
        const SphereWs ws(d_ws, n_atoms);
        return launch_union_warp(g, d_rho, n_groups, d_group_start, d_xyz, d_radius, ws.box, ws.thr, cut_pos, cut_neg, ws.counter, d_out,
                                 0, nullptr, nullptr, st);
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
    if (n_atoms > 0 && n_groups > 0 && d_group_start && boxes_are_small(g, max_atom_radius)) {
        const SphereWs ws(d_ws, n_atoms);
        return launch_union_warp(g, d_rho, n_groups, d_group_start, d_xyz, d_group_radius, ws.box, ws.thr, cut_pos, cut_neg, ws.counter,
                                 d_out_groups, n_atoms, d_atom_radius, d_out_atoms, (cudaStream_t)stream);
    }
    if (int rc = pe_sphere_sums(g, d_rho, n_atoms, d_xyz, d_atom_radius, n_atoms, nullptr, cut_pos, cut_neg, d_out_atoms, d_ws, stream))
        return rc;
    return pe_sphere_sums(g, d_rho, n_atoms, d_xyz, d_group_radius, n_groups, d_group_start, cut_pos, cut_neg, d_out_groups, d_ws, stream);
}

int64_t pe_batch_sphere_sums_workspace_bytes(int64_t n_atoms) { return SphereWs::bytes(n_atoms < 0 ? 0 : n_atoms); }

int pe_batch_sphere_sums(int32_t n_maps, const pe_sums_map *d_maps, int32_t n_atoms, const double *d_xyz, const float *d_radius,
                         int32_t n_groups, const int32_t *d_group_map, const int32_t *d_group_start, const int32_t *d_atom_start,
                         double *d_out, void *d_ws, void *stream) {
    PE_CHECK_ARG(n_maps >= 0 && n_atoms >= 0 && n_groups >= 0, "pe_batch_sphere_sums: negative size");
    if (n_groups == 0) return PE_OK;
    PE_CHECK_ARG(n_maps > 0, "pe_batch_sphere_sums: groups without maps");
    PE_CHECK_ARG(d_maps && d_xyz && d_radius && d_group_map && d_out && d_ws, "pe_batch_sphere_sums: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (d_group_start == nullptr) {
        PE_CHECK_ARG(n_groups == n_atoms, "pe_batch_sphere_sums: n_groups must equal n_atoms without group offsets");
        PE_CHECK_ARG(d_atom_start != nullptr, "pe_batch_sphere_sums: per-atom sums need d_atom_start");
        // every structure adds at most one partial quad; the warps stride over the quads, so the grid only sets the parallelism
        const int64_t quads = (int64_t)n_atoms / kAtomsPerWarp + n_maps;
        int64_t blocks = (quads + kSphereWarps - 1) / kSphereWarps;
        const int64_t max_blocks = (int64_t)sm_count() * 16;
        if (blocks > max_blocks) blocks = max_blocks;
        PE_LAUNCH("batch_sphere_sums_kernel", st, batch_sphere_sums_kernel<<<(int)blocks, kSphereWarps * 32, 0, st>>>(
            n_maps, d_maps, d_atom_start, d_group_map, d_xyz, d_radius, d_out));
        PE_LAUNCH_CHECK();
        return PE_OK;
    }
    const SphereWs ws(d_ws, n_atoms);
    return launch_batch_union(n_maps, d_maps, n_groups, d_group_map, d_group_start, d_xyz, d_radius, ws.box, ws.thr, ws.counter, d_out, st);
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
