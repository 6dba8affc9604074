// pe_union.cu -- set-union sphere sums, one WARP per group of atoms (the grouped form of pe_sphere_sums).
//
// Replaces getSphereCrsFromXyzList (pdb_eda/cutils.pyx:250-271) + the sums of calculateRegionDensity / calculateRegionDiscrepancy
// (pdb_eda/densityAnalysis.py:1037-1068, :1160-1211) for every residue (group) of a structure at once.
//
// A warp owns a group from start to finish -- boxes, bounding box, per-atom tables, membership bitmap, compaction, gather,
// reduction all stay inside the warp (shuffles and __syncwarp only, no block barriers), groups are handed out through one
// atomic counter, and the four warps of a CTA only share the SM:
//   * tile = 32 columns x 32 rows x 32 sections of the group's bounding box (a residue at the default 3.5 A radius on a 0.5 A
//     grid is one tile), one 32-bit bitmap word per (row, section): 4 KB per warp;
//   * atoms are taken one after the other: the warp tabulates the atom's squares along the three axes (one entry per lane),
//     then every lane takes box rows (row, section) of that atom, finds the row's in-sphere columns exactly (row_chord) and ORs
//     the run into its word -- no atomics: within an atom every word belongs to one lane;
//   * gather: the bitmap rows are taken 32 at a time (one per lane); a row's bits are almost always ONE run, which is written
//     to the warp's list of map offsets with a counted loop (runs with holes fall back to bit scanning); the list is then
//     walked densely with 8 independent loads in flight per lane, each voxel of the union read exactly once.
// The float64 summation order is fixed, so results are run-to-run deterministic.  Skewed cells test every candidate voxel of a
// box with the reference's distance instead of tabulated squares; a bounding box larger than one tile is split into more tiles
// (columns included).
#include <limits.h>
#include <stddef.h>
#include "pe_sphere_dev.cuh"

#ifndef PE_UNION_PHASE_CYCLES
#define PE_UNION_PHASE_CYCLES 0
#endif

namespace pe {

// Diagnostic (compiled in with -DPE_UNION_PHASE_CYCLES=1 only): warp cycles by phase, summed over all warps since the last
// read through pe_sphere_union_warp_cycles(): 0 boxes + bounding box, 1 tile offsets + per-atom tables, 2 membership, 3 gather,
// 4 reduction + output.
__device__ unsigned long long g_union_warp_cycles[5];
// The clock of one warp's phases, carried through the work items (every member is empty in the normal build).
struct PhaseClock {
#if PE_UNION_PHASE_CYCLES
    long long mark, t[5];
    // clock64 only exists in the device pass; the host pass parses these bodies as well
    __device__ __forceinline__ static long long now() {
#ifdef __CUDA_ARCH__
        return clock64();
#else
        return 0;
#endif
    }
    __device__ __forceinline__ PhaseClock() : mark(now()), t{0, 0, 0, 0, 0} {}
    __device__ __forceinline__ void lap(int k) {
        const long long now = PhaseClock::now();
        t[k] += now - mark;
        mark = now;
    }
    __device__ __forceinline__ void flush(int lane) {
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < 5; ++k) atomicAdd(g_union_warp_cycles + k, (unsigned long long)t[k]);
        }
    }
#else
    __device__ __forceinline__ void lap(int) {}
    __device__ __forceinline__ void flush(int) {}
#endif
};

constexpr int kUW = 4;        // warps per CTA
constexpr int kUT = 32;       // tile edge
constexpr int kUCtas = 7;     // resident CTAs per SM (6 / 7 / 8 / 9: 165 / 144 / 146-148 / 174 us; spills at 64 registers)
constexpr int kUList = 704;   // list entries per warp: what 7 CTAs per SM leave (448 at 8, 256 at 9)
constexpr int kULoads = 8;    // loads in flight per lane (4: 165 us, 8: 144 us, 12 / 16: 149-153 us on C2's region pass)

struct WarpUnion {
    uint32_t bits[kUT * kUT];     // [row][section]
    int list[kUList];
    double sqC[kUT], sqR[kUT], sqS[kUT];  // an atom item keeps its quad's SmallTabs here (quad_tabs)
    int offC[kUT], offR[kUT], offS[kUT];
};
// 228 KB of shared memory per SM, of which every CTA also takes 1 KB for the system: kUList is as long as kUCtas CTAs allow.
static_assert(kUCtas * (kUW * sizeof(WarpUnion) + 1024) <= 228 * 1024, "kUCtas CTAs per SM do not fit the shared memory");
// At 7 CTAs per SM the shared memory has no room for more: an atom item's tables take the place of a residue item's per-atom
// tables and tile offsets, which are dead between two items.
static_assert(offsetof(WarpUnion, offS) + sizeof(WarpUnion::offS) - offsetof(WarpUnion, sqC) == kAtomsPerWarp * sizeof(SmallTab),
              "the quad's tables fill the residue tables' bytes exactly");
static_assert(offsetof(WarpUnion, sqC) % alignof(SmallTab) == 0, "SmallTab alignment");
__device__ __forceinline__ SmallTab *quad_tabs(WarpUnion &w) { return reinterpret_cast<SmallTab *>(w.sqC); }

// Sums of one step of the gather: kULoads values per lane; the float64 additions form a small tree (fixed shape:
// deterministic) so that no accumulator carries a chain of eight dependent additions.
template <bool HASNEG, int N>
__device__ __forceinline__ void step_sum(const float *v, SphereAcc &acc, float cp, float cn) {
    double d[N], p[N], q[N];
#pragma unroll
    for (int u = 0; u < N; ++u) {
        d[u] = widen(v[u]);
        const bool pos = v[u] > cp;
        p[u] = pos ? d[u] : 0.0;
        acc.n_pos += pos ? 1 : 0;
        if (HASNEG) {
            const bool neg = v[u] < cn;
            q[u] = neg ? d[u] : 0.0;
            acc.n_neg += neg ? 1 : 0;
        }
    }
#pragma unroll
    for (int o = 1; o < N; o <<= 1) {
#pragma unroll
        for (int u = 0; u + o < N; u += 2 * o) {
            d[u] += d[u + o];
            p[u] += p[u + o];
            if (HASNEG) q[u] += q[u + o];
        }
    }
    acc.s_all += d[0];
    acc.s_pos += p[0];
    if (HASNEG) acc.s_neg += q[0];
}

// Gather of one tile: every voxel of the union is read once.  The bitmap rows are taken one tile row (= up to 32 sections, one
// per lane) at a time; a warp prefix sum of the popcounts places every row's voxels in a list of map offsets (a row's bits are
// almost always ONE run, written with a counted loop; rows with holes are bit-scanned), and the list is walked densely, 8
// (or, for short lists, 4) independent loads per lane and step.
// Measured and dropped (profiles/r02_union_phases.md): keeping a batch's loads in flight across the compaction of the next one,
// in registers (146.3 us) or as cp.async copies into the list itself (147.9 us) against 144.4 us for this plain form.  No single
// pipe limits the kernel (issue slots 64 % busy; ALU 38 %, LSU 32 %, XU 20 %, FP64 12 %): it is the length of each warp's
// dependent instruction chains at 28 warps per SM.
template <bool CHECKED, bool HASNEG>
__device__ __forceinline__ void gather_tile(WarpUnion &w, const float *__restrict__ rho, SphereAcc &acc, float cp, float cn, int lane,
                                            int tR, int tS) {
    int *list = w.list;
    const int oc0 = w.offC[0];
    for (int r0 = 0; r0 < tR; ++r0) {  // one tile row = tS (<= 32) words = one batch
        uint32_t wd = lane < tS ? w.bits[r0 * kUT + lane] : 0u;
        if (!__any_sync(kFull, wd != 0u)) continue;
        if (wd != 0u) w.bits[r0 * kUT + lane] = 0u;  // leave the bitmap clear
        int orr = 0, osum = 0;
        if (lane < tS) {
            const int o1 = w.offR[r0], o2 = w.offS[lane];
            orr = o1 | o2;
            osum = (int)((unsigned)o1 + (unsigned)o2);
        }
        const int c = __popc(wd);
        bool pending = c > 0;
        while (true) {  // one round unless the batch overflows the list
            const int cc = pending ? c : 0;
            const int excl = warp_excl_scan(cc, lane);
            const bool fits = excl + cc <= kUList;
            const int total = __reduce_max_sync(kFull, fits ? excl + cc : 0);
            if (pending && fits) {
                int *dst = list + excl;
                if (CHECKED) {
                    uint32_t x = wd;
                    while (x) {
                        const int bcol = __ffs((int)x) - 1;
                        x &= x - 1u;
                        const int oc = w.offC[bcol];
                        *dst++ = ((orr | oc) < 0) ? -1 : (int)((unsigned)osum + (unsigned)oc);
                    }
                } else {
                    const int first = __ffs((int)wd) - 1;
                    const int rowbase = (int)((unsigned)osum + (unsigned)oc0);
                    if (((wd >> first) + 1u) & (wd >> first)) {  // holes: more than one run
                        uint32_t x = wd;
                        while (x) {
                            const int bcol = __ffs((int)x) - 1;
                            x &= x - 1u;
                            *dst++ = rowbase + bcol;
                        }
                    } else {  // one run of c columns starting at `first`
                        const int v0 = rowbase + first;
#pragma unroll 4
                        for (int j = 0; j < c; ++j) dst[j] = v0 + j;
                    }
                }
                pending = false;
            }
            __syncwarp();
            if (lane == 0) acc.n_all += total;
            for (int i0 = 0; i0 < total; i0 += 32 * kULoads) {
                const bool half = total - i0 <= 32 * (kULoads / 2);  // warp-uniform: short lists issue half the loads
                float v[kULoads];
#pragma unroll
                for (int u = 0; u < kULoads; ++u) {
                    v[u] = 0.f;
                    if (u >= kULoads / 2 && half) continue;
                    const int idx = i0 + 32 * u + lane;
                    const int e = idx < total ? list[idx] : -2;
                    if (e >= 0) v[u] = __ldg(rho + e);
                    if (CHECKED) acc.bad |= (e == -1) ? 1 : 0;
                }
                if (half)
                    step_sum<HASNEG, kULoads / 2>(v, acc, cp, cn);
                else
                    step_sum<HASNEG, kULoads>(v, acc, cp, cn);
            }
            __syncwarp();  // the list is rewritten by the next round / batch
            if (!__any_sync(kFull, pending)) break;
        }
    }
}

// One group of atoms [a0, a1) by one warp, from the atom boxes to the output row o (PE_SPHERE_NOUT values, written by lane 0).
// The list capacity kUList, kULoads and the short-list rule of gather_tile fix the summation order, so every kernel that calls
// this gives a group the same bits.  Leaves w.bits clear.  cp / cn: effective cutoffs; icx / inv_gl: the column axis' xyz axis
// and its inverse grid length.
template <int MODE>
__device__ __forceinline__ void union_group(WarpUnion &w, const pe_geom &g, const float *__restrict__ rho, int a0, int a1,
                                            const double *__restrict__ xyz, const float *__restrict__ radius, int32_t *box,
                                            double *thr, float cp, float cn, bool has_neg, int icx, float inv_gl, int lane,
                                            double *__restrict__ o, PhaseClock &clk) {
    // boxes and thresholds of the group's atoms (lanes over atoms), bounding box by warp reductions
    int ulo0 = INT_MAX, ulo1 = INT_MAX, ulo2 = INT_MAX, uhi0 = INT_MIN, uhi1 = INT_MIN, uhi2 = INT_MIN;
    double candidates = 0.0;
    for (int a = a0 + lane; a < a1; a += 32) {
        AtomBox bb;
        double tt;
        atom_box(g, xyz[3 * a], xyz[3 * a + 1], xyz[3 * a + 2], radius[a], bb, tt);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            box[6 * a + k] = bb.lo[k];
            box[6 * a + 3 + k] = bb.dim[k];
        }
        thr[a] = tt;
        candidates += (double)bb.dim[0] * (double)bb.dim[1] * (double)bb.dim[2];
        if (bb.dim[0] > 0 && bb.dim[1] > 0 && bb.dim[2] > 0) {
            ulo0 = min(ulo0, bb.lo[0]);
            ulo1 = min(ulo1, bb.lo[1]);
            ulo2 = min(ulo2, bb.lo[2]);
            uhi0 = max(uhi0, bb.lo[0] + bb.dim[0]);
            uhi1 = max(uhi1, bb.lo[1] + bb.dim[1]);
            uhi2 = max(uhi2, bb.lo[2] + bb.dim[2]);
        }
    }
    __syncwarp();  // boxes visible to the whole warp
    candidates = warp_sum(candidates);
    ulo0 = warp_min(ulo0);
    ulo1 = warp_min(ulo1);
    ulo2 = warp_min(ulo2);
    uhi0 = warp_max(uhi0);
    uhi1 = warp_max(uhi1);
    uhi2 = warp_max(uhi2);
    SphereAcc acc;
    clk.lap(0);
    if (uhi0 > ulo0) {
        for (int ts0 = ulo2; ts0 < uhi2; ts0 += kUT)
            for (int tr0 = ulo1; tr0 < uhi1; tr0 += kUT)
                for (int tc0 = ulo0; tc0 < uhi0; tc0 += kUT) {
                    const int tC = min(kUT, uhi0 - tc0), tR = min(kUT, uhi1 - tr0), tS = min(kUT, uhi2 - ts0);
                    // wrapped element offsets of the tile's indices; is every index stored and are the columns adjacent?
                    int invalid = 0;
                    {
                        const int oc = lane < tC ? axis_off(g, 0, tc0 + lane) : 0;
                        const int orw = lane < tR ? axis_off(g, 1, tr0 + lane) : 0;
                        const int os = lane < tS ? axis_off(g, 2, ts0 + lane) : 0;
                        w.offC[lane] = oc;
                        w.offR[lane] = orw;
                        w.offS[lane] = os;
                        invalid = (oc | orw | os) < 0 ? 1 : 0;
                        const int prev = __shfl_up_sync(kFull, oc, 1);
                        if (lane > 0 && lane < tC && oc != prev + 1) invalid = 1;
                    }
                    const bool checked = __any_sync(kFull, invalid != 0);
                    // membership, atom by atom
                    for (int a = a0; a < a1; ++a) {
                        const int32_t *bx = box + 6 * a;
                        const int b0 = bx[0], b1 = bx[1], b2 = bx[2], d0 = bx[3], d1 = bx[4], d2 = bx[5];
                        if (d0 <= 0 || d1 <= 0 || d2 <= 0) continue;
                        const int cl = max(b0, tc0), ch = min(b0 + d0, tc0 + tC);
                        const int rl = max(b1, tr0), rh = min(b1 + d1, tr0 + tR);
                        const int sl = max(b2, ts0), sh = min(b2 + d2, ts0 + tS);
                        if (cl >= ch || rl >= rh || sl >= sh) continue;
                        const double ax = xyz[3 * a], ay = xyz[3 * a + 1], az = xyz[3 * a + 2];
                        const double T = thr[a];
                        if (g.orthogonal) {
                            const int nC = ch - cl, nR = rh - rl, nS = sh - sl;
                            if (lane < nC) w.sqC[lane] = axis_sq(g, 0, cl + lane, ax, ay, az);
                            if (lane < nR) w.sqR[lane] = axis_sq(g, 1, rl + lane, ax, ay, az);
                            if (lane < nS) w.sqS[lane] = axis_sq(g, 2, sl + lane, ax, ay, az);
                            __syncwarp();
                            clk.lap(1);
                            // centre column of the box (range(c - R - 1, c + R + 1): c = lo + dim / 2), clamped into the tile part
                            const int kmin = min(max(b0 + d0 / 2 - cl, 0), nC - 1);
                            const float xc = (float)((sel3(ax, ay, az, icx) - g.origin[icx]) / g.grid_length[icx] - (double)cl);
                            mark_atom<MODE>(w.bits, w.sqC, w.sqR, w.sqS, lane, cl - tc0, nC, rl - tr0, nR, sl - ts0, nS, T, xc, inv_gl,
                                            kmin);
                            __syncwarp();  // tables are rewritten by the next atom; its rows may share words with this one
                            clk.lap(2);
                        } else {
                            const int nc = ch - cl, n1 = rh - rl;
                            const int vol = nc * n1 * (sh - sl);
                            for (int m = lane; m < vol; m += 32) {
                                const int ic = m % nc, t = m / nc;
                                const int c = cl + ic, r = rl + t % n1, s = sl + t / n1;
                                double vx, vy, vz;
                                crs2xyz(g, c, r, s, vx, vy, vz);
                                if (!(dist2(ax, ay, az, vx, vy, vz) <= T)) continue;
                                atomicOr(&w.bits[(r - tr0) * kUT + (s - ts0)], 1u << (c - tc0));
                            }
                            __syncwarp();
                        }
                    }
                    // gather every voxel of the union once
                    clk.lap(1);
                    if (checked) {
                        if (has_neg)
                            gather_tile<true, true>(w, rho, acc, cp, cn, lane, tR, tS);
                        else
                            gather_tile<true, false>(w, rho, acc, cp, cn, lane, tR, tS);
                    } else {
                        if (has_neg)
                            gather_tile<false, true>(w, rho, acc, cp, cn, lane, tR, tS);
                        else
                            gather_tile<false, false>(w, rho, acc, cp, cn, lane, tR, tS);
                    }
                    __syncwarp();
                    clk.lap(3);
                }
    }
    const int n_all = warp_sum(acc.n_all), n_pos = warp_sum(acc.n_pos), n_neg = warp_sum(acc.n_neg);
    const int bad = warp_sum(acc.bad);
    const double s_all = warp_sum(acc.s_all), s_pos = warp_sum(acc.s_pos), s_neg = warp_sum(acc.s_neg);
    if (lane == 0) {
        o[0] = (double)n_all;
        o[1] = s_all;
        o[2] = (double)n_pos;
        o[3] = s_pos;
        o[4] = (double)n_neg;
        o[5] = s_neg;
        o[6] = bad ? 0.0 : 1.0;
        o[7] = candidates;
    }
    clk.lap(4);
}

// Work items, handed out in order through one counter: [0, n_groups) are groups (the long items), then, when n_quad_atoms > 0,
// one item per quad of atoms [4q, 4q + 4) summed at atom_radius into out_atoms (quad_sums: the short items fill the SMs that
// the last groups would leave idle).  The host hands atoms over only when every box at atom_radius is at most kSmallDim wide;
// a quad that is not writes NaN rows, so that a wrong decision cannot pass for a result.
template <int MODE>
__global__ void __launch_bounds__(kUW * 32, kUCtas)
    sphere_union_warp_kernel(const __grid_constant__ pe_geom g, const float *__restrict__ rho, int n_groups,
                             const int32_t *__restrict__ group_start, const double *__restrict__ xyz, const float *__restrict__ radius,
                             int32_t *box, double *thr, float cp, float cn, int *__restrict__ counter,
                             double *__restrict__ out /* n_groups x PE_SPHERE_NOUT */, int n_quad_atoms,
                             const float *__restrict__ atom_radius, double *__restrict__ out_atoms /* n_quad_atoms x PE_SPHERE_NOUT */) {
    __shared__ WarpUnion wsh[kUW];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    WarpUnion &w = wsh[warp];
    cp = eff_pos(cp);
    cn = eff_neg(cn);
    const bool has_neg = cn > __int_as_float(0xff800000);
    const int icx = g.map2crs[0];  // xyz axis carried by the columns
    const float inv_gl = (float)(1.0 / g.grid_length[icx]);
    for (int i = lane; i < kUT * kUT; i += 32) w.bits[i] = 0u;  // cleared once: the gather leaves it clear
    __syncwarp();
    PhaseClock clk;
    const int n_items = n_groups + (n_quad_atoms + kAtomsPerWarp - 1) / kAtomsPerWarp;
    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(counter, 1);
        item = __shfl_sync(kFull, item, 0);
        if (item >= n_items) break;
        if (item >= n_groups) {
            const int a0 = (item - n_groups) * kAtomsPerWarp;
            if (!quad_sums<MODE>(g, rho, n_quad_atoms, a0, xyz, atom_radius, cp, cn, quad_tabs(w), lane, out_atoms) &&
                lane < min(kAtomsPerWarp, n_quad_atoms - a0) * PE_SPHERE_NOUT)
                out_atoms[(int64_t)a0 * PE_SPHERE_NOUT + lane] = __longlong_as_double(0x7ff8000000000000ll);
            continue;
        }
        const int grp = item;
        union_group<MODE>(w, g, rho, group_start[grp], group_start[grp + 1], xyz, radius, box, thr, cp, cn, has_neg, icx, inv_gl, lane,
                          out + (int64_t)grp * PE_SPHERE_NOUT, clk);
    }
    clk.flush(lane);
}

int launch_union_warp(const pe_geom *g, const float *d_rho, int n_groups, const int32_t *d_group_start, const double *d_xyz,
                      const float *d_radius, int32_t *box, double *thr, float cut_pos, float cut_neg, int *d_counter, double *d_out,
                      int n_quad_atoms, const float *d_atom_radius, double *d_out_atoms, cudaStream_t st) {
    const int mode = z_axis_mode(g);
    PE_CUDA(cudaMemsetAsync(d_counter, 0, sizeof(int), st));
    const int warps_needed = n_groups + (n_quad_atoms + kAtomsPerWarp - 1) / kAtomsPerWarp;
    int grid = (warps_needed + kUW - 1) / kUW;
    const int max_grid = stream_sm_count(st) * kUCtas;
    if (grid > max_grid) grid = max_grid;
    if (mode == 0)
        PE_LAUNCH("sphere_union_kernel", st, sphere_union_warp_kernel<0><<<grid, kUW * 32, 0, st>>>(
            *g, d_rho, n_groups, d_group_start, d_xyz, d_radius, box, thr, cut_pos, cut_neg, d_counter, d_out,
            n_quad_atoms, d_atom_radius, d_out_atoms));
    else if (mode == 1)
        PE_LAUNCH("sphere_union_kernel", st, sphere_union_warp_kernel<1><<<grid, kUW * 32, 0, st>>>(
            *g, d_rho, n_groups, d_group_start, d_xyz, d_radius, box, thr, cut_pos, cut_neg, d_counter, d_out,
            n_quad_atoms, d_atom_radius, d_out_atoms));
    else
        PE_LAUNCH("sphere_union_kernel", st, sphere_union_warp_kernel<2><<<grid, kUW * 32, 0, st>>>(
            *g, d_rho, n_groups, d_group_start, d_xyz, d_radius, box, thr, cut_pos, cut_neg, d_counter, d_out,
            n_quad_atoms, d_atom_radius, d_out_atoms));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

// ------------------------------------------------------------------------------------------------ groups of many structures
// The groups of a whole batch, each on its own map (pe_batch_sphere_sums, grouped form): the work item of
// sphere_union_warp_kernel (union_group) with the geometry, map and cutoffs read from the group's table entry.  A warp keeps
// its group's pe_geom in shared memory next to its WarpUnion, which leaves room for 6 CTAs per SM instead of 7; the order of
// the sums does not depend on the occupancy, so a group's row is the bits sphere_union_warp_kernel gives it.
constexpr int kUBatchCtas = 6;
struct WarpUnionGeom {
    WarpUnion u;
    pe_geom geom;  // the current group's map geometry
};
static_assert(kUBatchCtas * (kUW * sizeof(WarpUnionGeom) + 1024) <= 228 * 1024, "kUBatchCtas CTAs per SM do not fit the shared memory");

__global__ void __launch_bounds__(kUW * 32, kUBatchCtas)
    batch_union_kernel(int n_maps, const pe_sums_map *__restrict__ maps, int n_groups, const int32_t *__restrict__ group_map,
                       const int32_t *__restrict__ group_start, const double *__restrict__ xyz, const float *__restrict__ radius,
                       int32_t *box, double *thr, int *__restrict__ counter, double *__restrict__ out /* n_groups x PE_SPHERE_NOUT */) {
    __shared__ WarpUnionGeom wsh[kUW];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    WarpUnion &w = wsh[warp].u;
    for (int i = lane; i < kUT * kUT; i += 32) w.bits[i] = 0u;  // cleared once: the gather leaves it clear
    __syncwarp();
    PhaseClock clk;
    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(counter, 1);
        item = __shfl_sync(kFull, item, 0);
        if (item >= n_groups) break;
        const int grp = item;
        double *o = out + (int64_t)grp * PE_SPHERE_NOUT;
        const int m = group_map[grp];
        const bool bad_map = m < 0 || m >= n_maps;
        float cp = bad_map ? 0.f : maps[m].cut_pos, cn = bad_map ? 0.f : maps[m].cut_neg;
        if (bad_map || cp < 0.f || cn > 0.f) {  // a group on no valid entry of the table: NaN, so that it cannot pass for a result
            if (lane < PE_SPHERE_NOUT) o[lane] = __longlong_as_double(0x7ff8000000000000ll);
            continue;
        }
        static_assert(sizeof(pe_geom) % 4 == 0, "pe_geom is copied as 32-bit words");
        for (int i = lane; i < (int)(sizeof(pe_geom) / 4); i += 32)
            reinterpret_cast<int *>(&wsh[warp].geom)[i] = reinterpret_cast<const int *>(&maps[m].geom)[i];
        __syncwarp();
        const pe_geom &g = wsh[warp].geom;
        const float *rho = maps[m].d_rho;
        cp = eff_pos(cp);
        cn = eff_neg(cn);
        const bool has_neg = cn > __int_as_float(0xff800000);
        const int icx = g.map2crs[0];
        const float inv_gl = (float)(1.0 / g.grid_length[icx]);
        const int a0 = group_start[grp], a1 = group_start[grp + 1];
        const int mode = g.map2xyz[2] == 1 ? 0 : (g.map2xyz[2] == 2 ? 1 : 2);  // z_axis_mode, warp-uniform
        if (mode == 0)
            union_group<0>(w, g, rho, a0, a1, xyz, radius, box, thr, cp, cn, has_neg, icx, inv_gl, lane, o, clk);
        else if (mode == 1)
            union_group<1>(w, g, rho, a0, a1, xyz, radius, box, thr, cp, cn, has_neg, icx, inv_gl, lane, o, clk);
        else
            union_group<2>(w, g, rho, a0, a1, xyz, radius, box, thr, cp, cn, has_neg, icx, inv_gl, lane, o, clk);
        __syncwarp();  // the geometry is rewritten by the next group
    }
    clk.flush(lane);
}

int launch_batch_union(int n_maps, const pe_sums_map *d_maps, int n_groups, const int32_t *d_group_map, const int32_t *d_group_start,
                       const double *d_xyz, const float *d_radius, int32_t *box, double *thr, int *d_counter, double *d_out,
                       cudaStream_t st) {
    PE_CUDA(cudaMemsetAsync(d_counter, 0, sizeof(int), st));
    int grid = (n_groups + kUW - 1) / kUW;
    const int max_grid = sm_count() * kUBatchCtas;
    if (grid > max_grid) grid = max_grid;
    PE_LAUNCH("batch_union_kernel", st, batch_union_kernel<<<grid, kUW * 32, 0, st>>>(
        n_maps, d_maps, n_groups, d_group_map, d_group_start, d_xyz, d_radius, box, thr, d_counter, d_out));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

}  // namespace pe

extern "C" int pe_sphere_union_warp_cycles(unsigned long long *out5) {
    PE_CHECK_ARG(out5 != nullptr, "pe_sphere_union_warp_cycles: null pointer");
    PE_CUDA(cudaMemcpyFromSymbol(out5, pe::g_union_warp_cycles, sizeof(unsigned long long) * 5));
    unsigned long long zero[5] = {0, 0, 0, 0, 0};
    PE_CUDA(cudaMemcpyToSymbol(pe::g_union_warp_cycles, zero, sizeof(zero)));
    return PE_OK;
}
