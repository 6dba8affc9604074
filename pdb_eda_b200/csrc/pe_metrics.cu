// pe_metrics.cu -- RSCC / RSR sums over the set-union of a group's atom spheres on a 2Fo-Fc / Fo-Fc map pair, for the groups
// of many structures in one launch (pe_pair_union_metrics).
//
// The per-structure chain it replaces for batches -- sphere voxel lists in global memory (pe_sphere_count / pe_sphere_fill),
// a hash table over the whole list for the first occurrence of every (group, voxel) (pe_cluster_crs_grouped), and two passes
// of one float64 atomicAdd per voxel and sum (pe_pair_metrics) -- becomes one warp per group, from the atom boxes to the output
// row, as in sphere_union_warp_kernel (pe_union.cu):
//   * groups are handed out through one atomic counter; a group's geometry and maps come from its entry of the map table, so
//     every group of the batch may sit on a different grid, cell and axis order (the z-axis mode is a warp-uniform switch);
//   * membership: per 32^3 tile of the group's bounding box one bitmap word per (row, section), atoms marked one after the other
//     with tabulated squares and exact row chords (mark_atom) in orthogonal cells, the reference's distance per candidate in
//     skewed cells;
//   * gather: the bitmap is compacted row after row into a list of map offsets (a row's bits are almost always one run), the
//     list is walked densely with kMLoads independent loads per lane and map, each voxel of the union read once from both maps;
//   * two passes, like pe_pair_metrics and scipy's pearsonr: pass 1 sums n, fo, fc, |fo - fc|, |fo + fc|; pass 2 the moments
//     centred on the group's own means.  A group inside one tile keeps its bitmap from pass 1 and clears it in pass 2; a larger
//     group rebuilds every tile's membership in pass 2.
// Every lane adds its list entries in list order and the warp reduction has a fixed shape, so the sums are bit-identical from
// run to run and do not depend on the other groups of the batch.
#include <limits.h>
#include <stddef.h>
#include "pe_sphere_dev.cuh"

namespace pe {

constexpr int kMW = 4;       // warps per CTA
constexpr int kMT = 32;      // tile edge
constexpr int kMCtas = 4;    // resident CTAs per SM: 128 registers without spills (5 and 6 CTAs spill)
constexpr int kMList = 768;  // list entries per warp (>= 32: one bitmap word always fits an empty list)
constexpr int kMLoads = 4;   // loads in flight per lane and map
constexpr int kMRec = 8;     // int32 per atom record of the workspace: box low corner, box extents, threshold (float64)

struct WarpPair {
    uint32_t bits[kMT * kMT];  // [row][section]
    int list[kMList];
    double sqC[kMT], sqR[kMT], sqS[kMT];
    int offC[kMT], offR[kMT], offS[kMT];
    pe_geom geom;  // the current group's map geometry
};
static_assert(kMCtas * (kMW * sizeof(WarpPair) + 1024) <= 228 * 1024, "kMCtas CTAs per SM do not fit the shared memory");

struct PairAcc {
    int n = 0;
    double s_fo = 0.0, s_fc = 0.0, s_dif = 0.0, s_sum = 0.0;  // pass 1
    double s_xx = 0.0, s_yy = 0.0, s_xy = 0.0;                // pass 2
};

// Walks list[0, total): every entry is a map offset, or -1 for a voxel the stored map does not cover (fo = fc = 0, counted).
template <int PASS>
__device__ __forceinline__ void walk_list(const int *list, int total, const float *__restrict__ fo_map,
                                          const float *__restrict__ diff_map, double m_fo, double m_fc, PairAcc &acc, int lane) {
    if (PASS == 0 && lane == 0) acc.n += total;
    for (int i0 = 0; i0 < total; i0 += 32 * kMLoads) {
        float vf[kMLoads], vd[kMLoads];
        bool in[kMLoads];
#pragma unroll
        for (int u = 0; u < kMLoads; ++u) {
            const int idx = i0 + 32 * u + lane;
            in[u] = idx < total;
            const int e = in[u] ? list[idx] : -1;
            vf[u] = 0.f;
            vd[u] = 0.f;
            if (e >= 0) {
                vf[u] = __ldg(fo_map + e);
                vd[u] = __ldg(diff_map + e);
            }
        }
#pragma unroll
        for (int u = 0; u < kMLoads; ++u) {
            if (!in[u]) continue;
            const double fo = (double)vf[u];
            const double fc = __dsub_rn(fo, __dmul_rn((double)vd[u], 2.0));  // densityObj.density - diffDensityObj.density * 2
            if (PASS == 0) {
                acc.s_fo += fo;
                acc.s_fc += fc;
                acc.s_dif += fabs(fo - fc);
                acc.s_sum += fabs(fo + fc);
            } else {
                const double xm = fo - m_fo, ym = fc - m_fc;
                acc.s_xx += xm * xm;
                acc.s_yy += ym * ym;
                acc.s_xy += xm * ym;
            }
        }
    }
}

// Gather of one tile: the bitmap rows (one word per lane) are compacted into the list in order, which is walked whenever the
// next word would not fit and at the end.  CLEAR leaves the bitmap clear.
template <int PASS, bool CHECKED>
__device__ __forceinline__ void gather_pair_tile(WarpPair &w, const float *__restrict__ fo_map, const float *__restrict__ diff_map,
                                                 double m_fo, double m_fc, PairAcc &acc, int lane, int tR, int tS, bool clear) {
    int *list = w.list;
    const int oc0 = w.offC[0];
    int base = 0;  // warp-uniform: entries in the list
    for (int r0 = 0; r0 < tR; ++r0) {
        const uint32_t wd = lane < tS ? w.bits[r0 * kMT + lane] : 0u;
        if (!__any_sync(kFull, wd != 0u)) continue;
        if (clear && wd != 0u) w.bits[r0 * kMT + lane] = 0u;
        int orr = 0, osum = 0;
        if (lane < tS) {
            const int o1 = w.offR[r0], o2 = w.offS[lane];
            orr = o1 | o2;
            osum = (int)((unsigned)o1 + (unsigned)o2);
        }
        const int c = __popc(wd);
        bool pending = c > 0;
        while (true) {
            const int cc = pending ? c : 0;
            const int excl = warp_excl_scan(cc, lane);
            const bool fits = base + excl + cc <= kMList;  // the lanes that fit are a prefix: excl + cc grows with the lane
            const int added = __reduce_max_sync(kFull, fits ? excl + cc : 0);
            if (pending && fits) {
                int *dst = list + base + excl;
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
                        for (int j = 0; j < c; ++j) dst[j] = v0 + j;
                    }
                }
                pending = false;
            }
            base += added;
            if (!__any_sync(kFull, pending)) break;
            __syncwarp();
            walk_list<PASS>(list, base, fo_map, diff_map, m_fo, m_fc, acc, lane);
            __syncwarp();  // the list is rewritten
            base = 0;
        }
    }
    __syncwarp();
    walk_list<PASS>(list, base, fo_map, diff_map, m_fo, m_fc, acc, lane);
    __syncwarp();
}

// Tile offsets and membership of the atoms [a0, a1) in the tile at (tc0, tr0, ts0) of extent (tC, tR, tS).  Returns, warp-
// uniformly, whether the tile needs the checked gather (an index the map does not store, or columns that are not adjacent).
__device__ __forceinline__ bool build_tile(WarpPair &w, const pe_geom &g, int mode, int a0, int a1, const double *__restrict__ xyz,
                                           const int32_t *rec, int tc0, int tr0, int ts0, int tC, int tR, int tS,
                                           int lane) {
    const int icx = g.map2crs[0];  // xyz axis carried by the columns
    const float inv_gl = (float)(1.0 / g.grid_length[icx]);
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
    for (int a = a0; a < a1; ++a) {
        const int32_t *bx = rec + kMRec * a;
        const int b0 = bx[0], b1 = bx[1], b2 = bx[2], d0 = bx[3], d1 = bx[4], d2 = bx[5];
        if (d0 <= 0 || d1 <= 0 || d2 <= 0) continue;
        const int cl = max(b0, tc0), ch = min(b0 + d0, tc0 + tC);
        const int rl = max(b1, tr0), rh = min(b1 + d1, tr0 + tR);
        const int sl = max(b2, ts0), sh = min(b2 + d2, ts0 + tS);
        if (cl >= ch || rl >= rh || sl >= sh) continue;
        const double ax = xyz[3 * a], ay = xyz[3 * a + 1], az = xyz[3 * a + 2];
        const double T = *reinterpret_cast<const double *>(bx + 6);
        if (g.orthogonal) {
            const int nC = ch - cl, nR = rh - rl, nS = sh - sl;
            if (lane < nC) w.sqC[lane] = axis_sq(g, 0, cl + lane, ax, ay, az);
            if (lane < nR) w.sqR[lane] = axis_sq(g, 1, rl + lane, ax, ay, az);
            if (lane < nS) w.sqS[lane] = axis_sq(g, 2, sl + lane, ax, ay, az);
            __syncwarp();
            const int kmin = min(max(b0 + d0 / 2 - cl, 0), nC - 1);
            const float xc = (float)((sel3(ax, ay, az, icx) - g.origin[icx]) / g.grid_length[icx] - (double)cl);
            if (mode == 0)
                mark_atom<0>(w.bits, w.sqC, w.sqR, w.sqS, lane, cl - tc0, nC, rl - tr0, nR, sl - ts0, nS, T, xc, inv_gl, kmin);
            else if (mode == 1)
                mark_atom<1>(w.bits, w.sqC, w.sqR, w.sqS, lane, cl - tc0, nC, rl - tr0, nR, sl - ts0, nS, T, xc, inv_gl, kmin);
            else
                mark_atom<2>(w.bits, w.sqC, w.sqR, w.sqS, lane, cl - tc0, nC, rl - tr0, nR, sl - ts0, nS, T, xc, inv_gl, kmin);
            __syncwarp();  // tables are rewritten by the next atom; its rows may share words with this one
        } else {
            const int nc = ch - cl, n1 = rh - rl;
            const int vol = nc * n1 * (sh - sl);
            for (int m = lane; m < vol; m += 32) {
                const int ic = m % nc, t = m / nc;
                const int c = cl + ic, r = rl + t % n1, s = sl + t / n1;
                double vx, vy, vz;
                crs2xyz(g, c, r, s, vx, vy, vz);
                if (!(dist2(ax, ay, az, vx, vy, vz) <= T)) continue;
                atomicOr(&w.bits[(r - tr0) * kMT + (s - ts0)], 1u << (c - tc0));
            }
            __syncwarp();
        }
    }
    return checked;
}

template <int PASS>
__device__ __forceinline__ void gather_pair(WarpPair &w, bool checked, const float *fo_map, const float *diff_map, double m_fo,
                                            double m_fc, PairAcc &acc, int lane, int tR, int tS, bool clear) {
    if (checked)
        gather_pair_tile<PASS, true>(w, fo_map, diff_map, m_fo, m_fc, acc, lane, tR, tS, clear);
    else
        gather_pair_tile<PASS, false>(w, fo_map, diff_map, m_fo, m_fc, acc, lane, tR, tS, clear);
}

__global__ void __launch_bounds__(kMW * 32, kMCtas)
    pair_union_metrics_kernel(int n_maps, const pe_pair_map *__restrict__ maps, int n_groups, const int32_t *__restrict__ group_map,
                              const int32_t *__restrict__ group_start, const double *__restrict__ xyz,
                              const float *__restrict__ radius, int32_t *rec, int *__restrict__ counter,
                              double *__restrict__ out /* n_groups x 8 */) {
    __shared__ WarpPair wsh[kMW];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    WarpPair &w = wsh[warp];
    for (int i = lane; i < kMT * kMT; i += 32) w.bits[i] = 0u;  // cleared once: every group leaves it clear
    __syncwarp();
    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(counter, 1);
        item = __shfl_sync(kFull, item, 0);
        if (item >= n_groups) break;
        const int grp = item;
        double *o = out + (int64_t)grp * 8;
        const int m = group_map[grp];
        if (m < 0 || m >= n_maps) {  // a group on no map of the table: NaN, so that it cannot pass for a result
            if (lane < 8) o[lane] = __longlong_as_double(0x7ff8000000000000ll);
            continue;
        }
        static_assert(sizeof(pe_geom) % 4 == 0, "pe_geom is copied as 32-bit words");
        for (int i = lane; i < (int)(sizeof(pe_geom) / 4); i += 32)
            reinterpret_cast<int *>(&w.geom)[i] = reinterpret_cast<const int *>(&maps[m].geom)[i];
        __syncwarp();
        const pe_geom &g = w.geom;
        const float *fo_map = maps[m].d_fo, *diff_map = maps[m].d_diff;
        const int mode = g.map2xyz[2] == 1 ? 0 : (g.map2xyz[2] == 2 ? 1 : 2);  // z_axis_mode
        const int a0 = group_start[grp], a1 = group_start[grp + 1];
        int ulo0 = INT_MAX, ulo1 = INT_MAX, ulo2 = INT_MAX, uhi0 = INT_MIN, uhi1 = INT_MIN, uhi2 = INT_MIN;
        for (int a = a0 + lane; a < a1; a += 32) {
            AtomBox bb;
            double tt;
            atom_box(g, xyz[3 * a], xyz[3 * a + 1], xyz[3 * a + 2], radius[a], bb, tt);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                rec[kMRec * a + k] = bb.lo[k];
                rec[kMRec * a + 3 + k] = bb.dim[k];
            }
            *reinterpret_cast<double *>(rec + kMRec * a + 6) = tt;
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
        ulo0 = warp_min(ulo0);
        ulo1 = warp_min(ulo1);
        ulo2 = warp_min(ulo2);
        uhi0 = warp_max(uhi0);
        uhi1 = warp_max(uhi1);
        uhi2 = warp_max(uhi2);
        PairAcc acc;
        double m_fo = 0.0, m_fc = 0.0;
        if (uhi0 > ulo0) {
            const bool one_tile = uhi0 - ulo0 <= kMT && uhi1 - ulo1 <= kMT && uhi2 - ulo2 <= kMT;
            bool checked0 = false;
            // pass 1: n and the first sums
            for (int ts0 = ulo2; ts0 < uhi2; ts0 += kMT)
                for (int tr0 = ulo1; tr0 < uhi1; tr0 += kMT)
                    for (int tc0 = ulo0; tc0 < uhi0; tc0 += kMT) {
                        const int tC = min(kMT, uhi0 - tc0), tR = min(kMT, uhi1 - tr0), tS = min(kMT, uhi2 - ts0);
                        const bool checked = build_tile(w, g, mode, a0, a1, xyz, rec, tc0, tr0, ts0, tC, tR, tS, lane);
                        checked0 = checked;
                        gather_pair<0>(w, checked, fo_map, diff_map, 0.0, 0.0, acc, lane, tR, tS, !one_tile);
                    }
            const int n = warp_sum(acc.n);
            const double s_fo = warp_sum(acc.s_fo), s_fc = warp_sum(acc.s_fc);
            m_fo = s_fo / (double)n;
            m_fc = s_fc / (double)n;
            // pass 2: moments centred on the group's means
            if (one_tile) {
                gather_pair<1>(w, checked0, fo_map, diff_map, m_fo, m_fc, acc, lane, uhi1 - ulo1, uhi2 - ulo2, true);
            } else {
                for (int ts0 = ulo2; ts0 < uhi2; ts0 += kMT)
                    for (int tr0 = ulo1; tr0 < uhi1; tr0 += kMT)
                        for (int tc0 = ulo0; tc0 < uhi0; tc0 += kMT) {
                            const int tC = min(kMT, uhi0 - tc0), tR = min(kMT, uhi1 - tr0), tS = min(kMT, uhi2 - ts0);
                            const bool checked = build_tile(w, g, mode, a0, a1, xyz, rec, tc0, tr0, ts0, tC, tR, tS, lane);
                            gather_pair<1>(w, checked, fo_map, diff_map, m_fo, m_fc, acc, lane, tR, tS, true);
                        }
            }
        }
        const int n = warp_sum(acc.n);
        const double s_fo = warp_sum(acc.s_fo), s_fc = warp_sum(acc.s_fc), s_dif = warp_sum(acc.s_dif), s_sum = warp_sum(acc.s_sum);
        const double s_xx = warp_sum(acc.s_xx), s_yy = warp_sum(acc.s_yy), s_xy = warp_sum(acc.s_xy);
        if (lane == 0) {
            o[0] = (double)n;
            o[1] = s_fo;
            o[2] = s_fc;
            o[3] = s_dif;
            o[4] = s_sum;
            o[5] = s_xx;
            o[6] = s_yy;
            o[7] = s_xy;
        }
        __syncwarp();
    }
}

}  // namespace pe

using namespace pe;

extern "C" {

int64_t pe_pair_union_workspace_bytes(int32_t n_atoms) {
    if (n_atoms < 0) return -1;
    return 256 + (int64_t)n_atoms * kMRec * sizeof(int32_t);
}

int pe_pair_union_metrics(int32_t n_maps, const pe_pair_map *d_maps, int32_t n_groups, const int32_t *d_group_map,
                          const int32_t *d_group_start, const double *d_xyz, const float *d_radius, double *d_out, void *d_ws,
                          void *stream) {
    PE_CHECK_ARG(n_maps >= 0 && n_groups >= 0, "pe_pair_union_metrics: negative size");
    if (n_groups == 0) return PE_OK;
    PE_CHECK_ARG(n_maps > 0, "pe_pair_union_metrics: groups without maps");
    PE_CHECK_ARG(d_maps && d_group_map && d_group_start && d_xyz && d_radius && d_out && d_ws, "pe_pair_union_metrics: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    // workspace: counter, then per atom its box (6 int32) and distance threshold (float64) in one 32-byte record
    int *counter = (int *)d_ws;
    int32_t *rec = (int32_t *)((char *)d_ws + 256);
    PE_CUDA(cudaMemsetAsync(counter, 0, sizeof(int), st));
    int grid = (n_groups + kMW - 1) / kMW;
    const int max_grid = sm_count() * kMCtas;
    if (grid > max_grid) grid = max_grid;
    PE_LAUNCH("pair_union_metrics_kernel", st, pair_union_metrics_kernel<<<grid, kMW * 32, 0, st>>>(
        n_maps, d_maps, n_groups, d_group_map, d_group_start, d_xyz, d_radius, rec, counter, d_out));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

}  // extern "C"
