// pe_sphere_dev.cuh -- device helpers shared by the sphere kernels (pe_sphere.cu) and the batched cloud aggregation
// (pe_aggregate.cu): the candidate box of getSphereCrsFromXyz (pdb_eda/cutils.pyx:238-243), the separable squared
// distance tables of orthogonal cells and the in-sphere enumeration in the reference's order.
#pragma once
#include "pe_common.cuh"

namespace pe {

constexpr int kDMax = 64;        // widest tabulated box edge (2R+2); wider boxes use the generic path
constexpr int kSphereWarps = 4;  // warps (= atoms) per CTA

struct AxisTab {
    double sq[kDMax];  // fl((coord - atom)^2) per index along this axis
    int off[kDMax];    // wrapped element offset contribution, or kInvalidOff
};

struct AtomBox {
    int lo[3];
    int dim[3];
};

// Box of getSphereCrsFromXyz (pdb_eda/cutils.pyx:238-243) and the distance threshold.
__device__ __forceinline__ void atom_box(const pe_geom &g, double ax, double ay, double az, float radius, AtomBox &b,
                                         double &thr) {
    const double r = (double)radius;
    int c0, r0, s0, rc, rr, rs;
    xyz2crs(g, ax, ay, az, c0, r0, s0);
    xyz2crs(g, __dadd_rn(g.origin[0], r), __dadd_rn(g.origin[1], r), __dadd_rn(g.origin[2], r), rc, rr, rs);
    b.lo[0] = c0 - rc - 1;
    b.lo[1] = r0 - rr - 1;
    b.lo[2] = s0 - rs - 1;
    b.dim[0] = max(2 * rc + 2, 0);
    b.dim[1] = max(2 * rr + 2, 0);
    b.dim[2] = max(2 * rs + 2, 0);
    thr = sphere_threshold(r);
}

// Axis term of the separable squared distance for crs axis `axis`, index k (orthogonal cells only).
__device__ __forceinline__ double axis_sq(const pe_geom &g, int axis, int k, double ax, double ay, double az) {
    const int i = g.map2crs[axis];  // xyz axis carried by this crs axis
    const double coord = __dadd_rn(__dmul_rn((double)k, g.grid_length[i]), g.origin[i]);
    const double d = __dsub_rn(coord, sel3(ax, ay, az, i));
    return __dmul_rn(d, d);
}

__device__ __forceinline__ int axis_off(const pe_geom &g, int axis, int k) {
    const int w = wrap_index(k, g.ncrs[axis], g.crs_interval[axis]);
    if (w < 0) return kInvalidOff;
    return axis == 0 ? w : (axis == 1 ? w * g.ncrs[0] : w * g.ncrs[0] * g.ncrs[1]);
}

__device__ __forceinline__ void fill_tables(const pe_geom &g, const AtomBox &b, double ax, double ay, double az,
                                            AxisTab *tab /* [2]: row axis, section axis */, int lane) {
    for (int k = lane; k < b.dim[1]; k += 32) {
        tab[0].sq[k] = axis_sq(g, 1, b.lo[1] + k, ax, ay, az);
        tab[0].off[k] = axis_off(g, 1, b.lo[1] + k);
    }
    for (int k = lane; k < b.dim[2]; k += 32) {
        tab[1].sq[k] = axis_sq(g, 2, b.lo[2] + k, ax, ay, az);
        tab[1].off[k] = axis_off(g, 2, b.lo[2] + k);
    }
    __syncwarp();
}

// Calls f(ic, ir, is, value_is_valid, rho) for every in-sphere voxel of the box, lanes in parallel.
template <class F>
__device__ __forceinline__ void for_each_inside(const pe_geom &g, const float *__restrict__ rho, const AtomBox &b,
                                                double ax, double ay, double az, double T, AxisTab *tab, int lane, F f) {
    const int D0 = b.dim[0], D1 = b.dim[1], D2 = b.dim[2];
    const bool tabulated = g.orthogonal && D1 <= kDMax && D2 <= kDMax;
    if (tabulated) {
        fill_tables(g, b, ax, ay, az, tab, lane);
        const bool caseb = g.map2xyz[2] == 0;
        const int inner = caseb ? 2 : g.map2xyz[2];
        const int outer = 3 - inner;
        const AxisTab &ti = tab[inner - 1];
        const AxisTab &to = tab[outer - 1];
        const int Di = sel3(b.dim[0], b.dim[1], b.dim[2], inner), Do = sel3(b.dim[0], b.dim[1], b.dim[2], outer);
        int d0p = 1;
        while (d0p < D0 && d0p < 32) d0p <<= 1;
        const int rpi = 32 / d0p, lrow = lane / d0p, lc = lane % d0p;
        for (int cbase = 0; cbase < D0; cbase += 32) {
            const int ic = cbase + lc;
            if (ic >= D0) continue;
            const int c = b.lo[0] + ic;
            const double sqc = axis_sq(g, 0, c, ax, ay, az);
            const int offc = axis_off(g, 0, c);
            for (int ko = lrow; ko < Do; ko += rpi) {
                const double sqo = to.sq[ko];
                const int offo = to.off[ko];
                const double P = __dadd_rn(sqc, sqo);
                // membership of the whole line first, then the gathers four at a time: with the load behind the distance test of
                // its own iteration a lane paid one memory round trip per in-sphere voxel (24 % of the count pass's stall samples)
                for (int kb = 0; kb < Di; kb += 32) {
                    uint32_t inside = 0u;
                    const int ke = min(Di - kb, 32);
                    for (int ki = 0; ki < ke; ++ki) {
                        const double sqi = ti.sq[kb + ki];
                        const double d2 = caseb ? __dadd_rn(__dadd_rn(sqo, sqi), sqc) : __dadd_rn(P, sqi);
                        inside |= (d2 <= T ? 1u : 0u) << ki;
                    }
                    while (inside) {
                        int kk[4];
                        float vv[4];
                        bool okk[4], has[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            has[u] = inside != 0u;
                            kk[u] = kb + __ffs((int)inside) - 1;
                            inside &= inside - 1u;
                            vv[u] = 0.f;
                            okk[u] = false;
                            if (has[u]) {
                                const int offi = ti.off[kk[u]];
                                okk[u] = (offc | offo | offi) >= 0;
                                if (okk[u]) vv[u] = __ldg(rho + (offc + offo + offi));
                            }
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            if (!has[u]) continue;
                            const int ir = inner == 1 ? kk[u] : ko, is = inner == 2 ? kk[u] : ko;
                            f(ic, ir, is, okk[u], vv[u]);
                        }
                    }
                }
            }
        }
        __syncwarp();
    } else {
        const int64_t vol = (int64_t)D0 * D1 * D2;
        for (int64_t m = lane; m < vol; m += 32) {
            const int ic = (int)(m % D0);
            const int64_t t = m / D0;
            const int ir = (int)(t % D1), is = (int)(t / D1);
            const int c = b.lo[0] + ic, r = b.lo[1] + ir, s = b.lo[2] + is;
            double vx, vy, vz;
            crs2xyz(g, c, r, s, vx, vy, vz);
            if (!(dist2(ax, ay, az, vx, vy, vz) <= T)) continue;
            const int oc = axis_off(g, 0, c), orr = axis_off(g, 1, r), os = axis_off(g, 2, s);
            const bool ok = (oc | orr | os) >= 0;
            const float v = ok ? __ldg(rho + (oc + orr + os)) : 0.f;
            f(ic, ir, is, ok, v);
        }
        __syncwarp();
    }
}

// Density predicate of getSphereCrsFromXyz (pdb_eda/cutils.pyx:245); all operands are exact float32 values.
__device__ __forceinline__ bool passes(float v, float cut) { return (0.f < cut && cut < v) || (v < cut && cut < 0.f) || cut == 0.f; }

// float -> double widening.  An integer-pipe bit-twiddling version was tried when F2F.F64.F32 showed up as the top
// stall of the first capture (profiles/r01a_first_path.md); once the gather loops kept four independent loads in
// flight the plain conversion (one issue slot, its latency hidden) became the faster one again: 257 -> 231 us on
// the C2 region pass.
__device__ __forceinline__ double widen(float v) { return (double)v; }

// Effective cutoffs: a class whose cutoff is 0 is switched off by an unreachable threshold.
__device__ __forceinline__ float eff_pos(float cp) { return cp > 0.f ? cp : __int_as_float(0x7f800000); }
__device__ __forceinline__ float eff_neg(float cn) { return cn < 0.f ? cn : __int_as_float(0xff800000); }

struct SphereAcc {
    int n_all = 0, n_pos = 0, n_neg = 0, bad = 0;
    double s_all = 0.0, s_pos = 0.0, s_neg = 0.0;
    // v must be 0 when the voxel is not taken; cp / cn are the effective cutoffs (cp > 0 > cn).
    __device__ __forceinline__ void add(bool take, float v, float cp, float cn) {
        const double d = widen(v);
        s_all += d;
        if (take) ++n_all;
        if (v > cp) {
            ++n_pos;
            s_pos += d;
        }
        if (v < cn) {
            ++n_neg;
            s_neg += d;
        }
    }
    // the same with the negative class switched off (cn == -inf): a third less work per voxel
    __device__ __forceinline__ void add_pos(bool take, float v, float cp) {
        const double d = widen(v);
        s_all += d;
        if (take) ++n_all;
        if (v > cp) {
            ++n_pos;
            s_pos += d;
        }
    }
};

// ------------------------------------------------------------------------------------------------ exact chords
// MODE 0: z is carried by the row axis, 1: by the section axis, 2: by the column axis.
inline int z_axis_mode(const pe_geom *g) { return g->map2xyz[2] == 1 ? 0 : (g->map2xyz[2] == 2 ? 1 : 2); }

// Squared distance of column k of a box row exactly as the reference adds it: fl(fl(X2 + Y2) + Z2).
template <int MODE>
__device__ __forceinline__ bool row_pred(const double *sqc, int k, double A, double B, double T) {
    // MODE 0/1: A = square of the non-z axis among (row, section), B = square of the z axis;
    // MODE 2  : A = fl(row square + section square), the column carries z.
    const double d2 = (MODE == 2) ? __dadd_rn(A, sqc[k]) : __dadd_rn(__dadd_rn(sqc[k], A), B);
    return d2 <= T;
}

// In-sphere columns [kl, kh] of one box row, exactly.  Along the columns of a box row the squared distance falls to the
// column nearest the atom (km) and rises again (every rounding step is monotone), so the in-sphere columns are one
// interval around that column.  The interval is GUESSED in float32 from the chord of the sphere along the row
// (half-width sqrt(T - A - B) in columns around the atom's fractional column xc) and then VERIFIED with the exact
// float64 predicate: inside at kl and kh, outside at kl - 1 and kh + 1 -- four independent tests that, by unimodality,
// prove the guess.  A guess that fails (an end within ~1e-5 columns of a grid point, or a row that only just misses the
// sphere) falls back to two binary searches with the same exact predicate.  Rows that miss the sphere leave after one
// exact test without touching the table: every rounding step is monotone and the column term is >= 0, so
// d2 >= fl(A + B) for every column of the row.  Returns false when no column of the row is inside.
// 1 / sqrt(x) for the chord guess only: the bare MUFU.RSQ (rsqrtf() wraps it in denormal scaling, six more instructions
// per box row; a denormal remainder just yields a guess that the exact tests reject)
__device__ __forceinline__ float rsqrt_guess(float x) {
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

template <int MODE>
__device__ __forceinline__ bool row_chord(const double *sqc, int nC, int km, float xc, float inv_gl, double A, double B, double T,
                                          int &kl, int &kh) {
    const double AB = (MODE == 2) ? A : __dadd_rn(A, B);
    if (!(AB <= T)) return false;  // exact: the row misses the sphere
    const float rem = (float)__dsub_rn(T, AB);
    const float h = rem > 0.f ? rem * rsqrt_guess(rem) * inv_gl : 0.f;
    const float xl = xc - h, xr = xc + h;
    const float fl_ = ceilf(xl), fr_ = floorf(xr);
    // The float32 guess is within 2e-5 columns of the real chord ends (|xc|, h <= 64 columns; rsqrt.approx 2^-22 relative), and the
    // reference's rounded float64 predicate moves an end by less than 1e-8 columns once the half chord exceeds 1e-6 columns.  So
    // when both guessed ends are more than kChordEps away from every grid point the interval is PROVEN without evaluating the
    // predicate (the exact tests below only run for the ~0.1 % of ends that fall within kChordEps of a column).
    constexpr float kChordEps = 2.5e-4f;
    if (h > 0.01f && fl_ - xl > kChordEps && xl - (fl_ - 1.f) > kChordEps && xr - fr_ > kChordEps && (fr_ + 1.f) - xr > kChordEps) {
        kl = max((int)fl_, 0);
        kh = min((int)fr_, nC - 1);
        return kl <= kh;
    }
    kl = min(max((int)fl_, 0), km);
    kh = max(min((int)fr_, nC - 1), km);
    const bool in_l = row_pred<MODE>(sqc, kl, A, B, T), in_h = row_pred<MODE>(sqc, kh, A, B, T);
    const bool out_l = kl == 0 || !row_pred<MODE>(sqc, kl - 1, A, B, T);
    const bool out_h = kh == nC - 1 || !row_pred<MODE>(sqc, kh + 1, A, B, T);
    if (in_l && in_h && out_l && out_h) return true;
    if (!row_pred<MODE>(sqc, km, A, B, T)) return false;  // the row misses the sphere
    int lo = 0, hi = km;  // smallest k in [0, km] inside
    while (lo < hi) {
        const int mid = (int)((unsigned)(lo + hi) >> 1);  // lo + hi >= 0, which the compiler does not always prove
        if (row_pred<MODE>(sqc, mid, A, B, T))
            hi = mid;
        else
            lo = mid + 1;
    }
    kl = lo;
    lo = km;
    hi = nC - 1;  // largest k in [km, nC) inside
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (row_pred<MODE>(sqc, mid, A, B, T))
            lo = mid;
        else
            hi = mid - 1;
    }
    kh = lo;
    return true;
}

// ------------------------------------------------------------------------------------------------ tile membership
// Shared by the grouped kernels (pe_union.cu, pe_metrics.cu): a warp owns a 32^3 tile, bits holds one 32-bit word per
// (row, section) (row-major, 32 sections per row).  sqc / sqR / sqS: the atom's squares along the tile part's columns,
// rows and sections.
// Membership of one atom in the warp's tile, exactly: a lane takes (row, section) lines of the atom's box, each on its own --
// row_chord finds the line's in-sphere columns and the lane ORs the run into the line's word.  (A sweep along the
// sections that narrows one interval from line to line needs fewer tests per line, but chains every line to the previous one
// and was slower: profiles/r02_union_phases.md.)
template <int MODE>
__device__ __forceinline__ void mark_atom(uint32_t *bits, const double *sqc, const double *sqR, const double *sqS, int lane, int cl,
                                          int nC, int rl, int nR, int sl, int nS, double T, float xc, float inv_gl, int kmin) {
    int km = kmin;  // the column nearest the atom: the box's centre column or, after rounding, one of its neighbours
    if (km > 0 && sqc[km - 1] < sqc[km]) --km;
    else if (km + 1 < nC && sqc[km + 1] < sqc[km]) ++km;
    const int shift = nS > 1 ? 32 - __clz(nS - 1) : 0;
    const int total = nR << shift;
#pragma unroll 2
    for (int li = lane; li < total; li += 32) {
        const int is = li & ((1 << shift) - 1), ir = li >> shift;
        if (is >= nS) continue;
        const double sr = sqR[ir], ss = sqS[is];
        const double A = (MODE == 0) ? ss : ((MODE == 1) ? sr : __dadd_rn(sr, ss));
        const double B = (MODE == 0) ? sr : ss;
        int kl, kh;
        if (!row_chord<MODE>(sqc, nC, km, xc, inv_gl, A, B, T, kl, kh)) continue;  // the row misses the sphere
        const int count = kh - kl + 1;
        const uint32_t run = count >= 32 ? ~0u : ((1u << count) - 1u);
        bits[(rl + ir) * 32 + (sl + is)] |= run << (cl + kl);  // within an atom this word belongs to this lane alone
    }
}

__device__ __forceinline__ int warp_min(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(kFull, v, o));
    return v;
}
__device__ __forceinline__ int warp_max(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(kFull, v, o));
    return v;
}

// ------------------------------------------------------------------------------------------------ per-atom sums, 4 atoms per warp
// At the atom-type radii of the cloud pass (0.6 - 1.3 A on a 0.5 A grid) a box is 4^3 or 6^3 candidates for ~15 in-sphere
// voxels, so when all four boxes of a warp's quad are at most kSmallDim wide (orthogonal cell) each atom gets 8 lanes: a lane
// walks box rows (row, section), finds the row's in-sphere columns exactly (row_chord) and gathers just those -- a fraction of
// the instructions of one warp per atom (49.7 -> 29.1 us on C2's cloud pass, see DESIGN.md).  One copy of this code serves
// sphere_sums_kernel (pe_sphere.cu) and the atom items of sphere_union_warp_kernel (pe_union.cu), so a per-atom result does
// not depend on which kernel computed it.
constexpr int kSmallDim = 8;
constexpr int kAtomsPerWarp = 4;
struct SmallTab {
    double sq[3][kSmallDim];  // per crs axis: fl((coord - atom)^2) of the box's indices
    int off[3][kSmallDim];    // wrapped element offsets, or kInvalidOff
};

// Sums of the atoms [a0, a0 + 4) (those below n_atoms) into out (PE_SPHERE_NOUT per atom).  cp / cn are the effective cutoffs
// (eff_pos / eff_neg).  Returns false, warp-uniformly and with nothing written, unless the cell is orthogonal and every box of
// the quad is at most kSmallDim wide.  Called by a whole warp; tab: kAtomsPerWarp tables of the warp's own.
template <int MODE>
__device__ __forceinline__ bool quad_sums(const pe_geom &g, const float *__restrict__ rho, int n_atoms, int a0,
                                          const double *__restrict__ xyz, const float *__restrict__ radius, float cp, float cn,
                                          SmallTab *tab, int lane, double *__restrict__ out) {
    const int sub = lane >> 3, l8 = lane & 7;
    const int a = a0 + sub;
    const bool live = a < n_atoms;
    // box and distance threshold of this lane's atom (the 8 lanes of an atom compute the same values: SIMT makes that free,
    // and a separate one-thread-per-atom launch in front of this kernel cost 9 us for C2's 40,000 atoms)
    int lo[3] = {0, 0, 0}, dim[3] = {0, 0, 0};
    double ax = 0.0, ay = 0.0, az = 0.0, T = -1.0;
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
    }
    const bool small = g.orthogonal && dim[0] <= kSmallDim && dim[1] <= kSmallDim && dim[2] <= kSmallDim;
    if (!__all_sync(kFull, small)) return false;
    SphereAcc acc;
    if (live && dim[0] > 0 && dim[1] > 0 && dim[2] > 0) {
        SmallTab &t = tab[sub];
#pragma unroll
        for (int axis = 0; axis < 3; ++axis) {
            if (l8 < dim[axis]) {
                t.sq[axis][l8] = axis_sq(g, axis, lo[axis] + l8, ax, ay, az);
                t.off[axis][l8] = axis_off(g, axis, lo[axis] + l8);
            }
        }
        __syncwarp(0xffu << (8 * sub));  // the 8 lanes of this atom (they take this branch together)
        const int ic = g.map2crs[0];  // xyz axis carried by the columns
        const float inv_gl = (float)(1.0 / g.grid_length[ic]);
        // the atom's fractional column inside the box: formed in float64 and rounded once, so that the guess stays within
        // 1e-5 columns of the real chord ends whatever the size of the map (row_chord's proof needs that)
        const float xc = (float)((sel3(ax, ay, az, ic) - g.origin[ic]) / g.grid_length[ic] - (double)lo[0]);
        const int nC = dim[0];
        const double *sqc = t.sq[0];
        // the column nearest the atom: the box's centre column or, after rounding, one of its neighbours
        int km = min(max(nC / 2, 0), nC - 1);
        if (km > 0 && sqc[km - 1] < sqc[km]) --km;
        else if (km + 1 < nC && sqc[km + 1] < sqc[km]) ++km;
        const int rows = dim[1] * dim[2];
        const unsigned div_d1 = (1024u + (unsigned)dim[1] - 1u) / (unsigned)dim[1];  // exact for row < 64, dim[1] <= 8
        static_assert(kSmallDim * kSmallDim * kSmallDim <= 1024, "magic division by dim[1]");
        for (int row = l8; row < rows; row += 8) {
            const int is = (int)(((unsigned)row * div_d1) >> 10), ir = row - is * dim[1];  // row / dim[1]
            const double sr = t.sq[1][ir], ss = t.sq[2][is];
            const double A = (MODE == 0) ? ss : ((MODE == 1) ? sr : __dadd_rn(sr, ss));
            const double B = (MODE == 0) ? sr : ss;
            int kl, kh;
            if (!row_chord<MODE>(sqc, nC, km, xc, inv_gl, A, B, T, kl, kh)) continue;
            const int o1 = t.off[1][ir], o2 = t.off[2][is];
            const int orr = o1 | o2;
            const unsigned osum = (unsigned)o1 + (unsigned)o2;
            // all loads of the chord first (a chord has at most kSmallDim columns), then the sums.  (Walking the rows of
            // the four atoms in lock step, reconverged every iteration, is slower -- 31.2 against 29.1 us: left to
            // themselves the four groups drift apart and hide each other's latency.)
            float v[kSmallDim];
#pragma unroll
            for (int j = 0; j < kSmallDim; ++j) {
                const int k = kl + j;
                v[j] = 0.f;
                if (k <= kh) {
                    const int oc = t.off[0][k];
                    const bool ok = (orr | oc) >= 0;
                    if (ok) v[j] = __ldg(rho + (int)(osum + (unsigned)oc));
                    acc.bad |= ok ? 0 : 1;
                }
            }
            const bool has_neg = cn > __int_as_float(0xff800000);  // warp-uniform: the negative class is in use
#pragma unroll
            for (int j = 0; j < kSmallDim; ++j) {
                if (kl + j > kh) break;  // chords are ~3 columns long: the sums are not worth issuing for empty slots
                if (has_neg)
                    acc.add(true, v[j], cp, cn);
                else
                    acc.add_pos(true, v[j], cp);
            }
        }
    }
    __syncwarp();  // the tables are free for the warp's next use
    // sums over the 8 lanes of an atom
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
        acc.n_all += __shfl_xor_sync(kFull, acc.n_all, o);
        acc.n_pos += __shfl_xor_sync(kFull, acc.n_pos, o);
        acc.n_neg += __shfl_xor_sync(kFull, acc.n_neg, o);
        acc.bad += __shfl_xor_sync(kFull, acc.bad, o);
        acc.s_all += __shfl_xor_sync(kFull, acc.s_all, o);
        acc.s_pos += __shfl_xor_sync(kFull, acc.s_pos, o);
        acc.s_neg += __shfl_xor_sync(kFull, acc.s_neg, o);
    }
    if (live && l8 == 0) {
        double *o = out + (int64_t)a * PE_SPHERE_NOUT;
        o[0] = (double)acc.n_all;
        o[1] = acc.s_all;
        o[2] = (double)acc.n_pos;
        o[3] = acc.s_pos;
        o[4] = (double)acc.n_neg;
        o[5] = acc.s_neg;
        o[6] = acc.bad ? 0.0 : 1.0;
        o[7] = (double)dim[0] * (double)dim[1] * (double)dim[2];
    }
    return true;
}

}  // namespace pe
