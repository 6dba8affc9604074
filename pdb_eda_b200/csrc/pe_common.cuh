// pe_common.cuh -- shared device helpers of libpdbeda_b200.so (sm_100a).
//
// Geometry arithmetic follows pdb_eda/ccp4.py:288-316 operation by operation in IEEE double with explicit
// round-to-nearest intrinsics (no FMA contraction; the library is also built with -fmad=false), because voxel
// membership has to match the reference bit for bit (SURVEY.md App. A.3).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/pdbeda_b200.h"

namespace pe {

void set_error(const char *fmt, ...);

#define PE_CHECK_ARG(cond, ...)          \
    do {                                 \
        if (!(cond)) {                   \
            pe::set_error(__VA_ARGS__);  \
            return PE_ERR_ARG;           \
        }                                \
    } while (0)

#define PE_CUDA(call)                                                                         \
    do {                                                                                      \
        cudaError_t err__ = (call);                                                           \
        if (err__ != cudaSuccess) {                                                           \
            pe::set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__,                \
                          cudaGetErrorString(err__));                                         \
            return PE_ERR_CUDA;                                                               \
        }                                                                                     \
    } while (0)

#define PE_LAUNCH_CHECK()                                                                     \
    do {                                                                                      \
        cudaError_t err__ = cudaGetLastError();                                               \
        if (err__ != cudaSuccess) {                                                           \
            pe::set_error("kernel launch failed at %s:%d: %s", __FILE__, __LINE__,            \
                          cudaGetErrorString(err__));                                         \
            return PE_ERR_CUDA;                                                               \
        }                                                                                     \
    } while (0)

// Every kernel launch goes through PE_LAUNCH: it counts the launch (pe_launch_count) and, while profiling is enabled
// (pe_profile_enable), brackets it with CUDA events on the launching stream so that bench.py can report per-kernel
// device times measured inside its timed region.
struct ProfScope {
    int slot;
    cudaStream_t stream;
    ProfScope(const char *tag, cudaStream_t st);
    ~ProfScope();
};
#define PE_LAUNCH(tag, stream, ...)                          \
    do {                                                     \
        pe::ProfScope prof_scope__(tag, (cudaStream_t)(stream)); \
        __VA_ARGS__;                                         \
    } while (0)

int sm_count();  // cached SM count of the current device (148 on B200)
// SMs a kernel launched on st can use: those of the stream's green context (pe_sm_partition_create), else sm_count().  Grids
// sized to be resident (persistent and cooperative kernels) take this, so that they fill a partition and never exceed it.
int stream_sm_count(cudaStream_t st);
int check_geom(const pe_geom *g);  // host-side validation shared by the entry points (pe_map.cu)
int check_geom_shape(const pe_geom *g, int64_t *nvox_out);  // the same without the 2^31-voxel limit of one call

static inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kInvalidOff = (int)0x80000000;  // sign bit marks "cell not covered by the stored map"

// ------------------------------------------------------------------------------------------------ small helpers
__device__ __forceinline__ int sel3(int a0, int a1, int a2, int i) { return i == 0 ? a0 : (i == 1 ? a1 : a2); }
__device__ __forceinline__ double sel3(double a0, double a1, double a2, int i) { return i == 0 ? a0 : (i == 1 ? a1 : a2); }

__device__ __forceinline__ int floordiv(int a, int b) {
    int q = a / b;
    if ((a % b != 0) && ((a < 0) != (b < 0))) --q;
    return q;
}

// getPointDensityFromCrs index rule (pdb_eda/cutils.pyx:138-143): returns the stored index or -1.
__device__ __forceinline__ int wrap_index(int k, int n, int interval) {
    if (k < 0 || k >= n) k -= floordiv(k, interval) * interval;
    if ((n <= k && k < interval) || k < 0) return -1;
    return k;
}

// One row of np.dot(M, x) in the accumulation order of the host BLAS (SURVEY.md App. A.13).
__device__ __forceinline__ double mv_row(const double *a, double x0, double x1, double x2, const pe_geom &g) {
    const int p0 = g.mv_perm[0], p1 = g.mv_perm[1], p2 = g.mv_perm[2];
    const double a0 = a[p0], a1 = a[p1], a2 = a[p2];
    const double y0 = sel3(x0, x1, x2, p0), y1 = sel3(x0, x1, x2, p1), y2 = sel3(x0, x1, x2, p2);
    double acc = __dmul_rn(a0, y0);
    if (g.mv_fma) {
        acc = __fma_rn(a1, y1, acc);
        acc = __fma_rn(a2, y2, acc);
    } else {
        acc = __dadd_rn(acc, __dmul_rn(a1, y1));
        acc = __dadd_rn(acc, __dmul_rn(a2, y2));
    }
    return acc;
}

// (int)rint(a / b) with the correctly rounded quotient, as Python's round(a / b) forms it.  A float64 division is ~30 instructions and
// every atom pays six of them; a * (1 / b) is within two ulp of the quotient (< 4e-10 below 1e6), so unless it lands within 1e-9 of a half-integer it
// rounds to the same integer, and only those rare cases (and non-finite ones) take the real division.
__device__ __forceinline__ int round_quotient(double a, double b) {
    const double q = __dmul_rn(a, __drcp_rn(b));
    const double r = rint(q);
    const double d = fabs(__dsub_rn(q, r));
    if (d < 0.499999999 && fabs(q) < 1.0e6) return (int)r;
    return (int)rint(__ddiv_rn(a, b));
}

// DensityHeader.xyz2crsCoord (pdb_eda/ccp4.py:288-302).  rint() == Python round() (half to even).
__device__ __forceinline__ void xyz2crs(const pe_geom &g, double x, double y, double z, int &c, int &r, int &s) {
    int p0, p1, p2;
    if (g.orthogonal) {
        p0 = round_quotient(__dsub_rn(x, g.origin[0]), g.grid_length[0]);
        p1 = round_quotient(__dsub_rn(y, g.origin[1]), g.grid_length[1]);
        p2 = round_quotient(__dsub_rn(z, g.origin[2]), g.grid_length[2]);
    } else {
        const double f0 = mv_row(g.deortho + 0, x, y, z, g);
        const double f1 = mv_row(g.deortho + 3, x, y, z, g);
        const double f2 = mv_row(g.deortho + 6, x, y, z, g);
        p0 = (int)rint(__dmul_rn(f0, (double)g.xyz_interval[0])) - g.crs_start[g.map2xyz[0]];
        p1 = (int)rint(__dmul_rn(f1, (double)g.xyz_interval[1])) - g.crs_start[g.map2xyz[1]];
        p2 = (int)rint(__dmul_rn(f2, (double)g.xyz_interval[2])) - g.crs_start[g.map2xyz[2]];
    }
    c = sel3(p0, p1, p2, g.map2crs[0]);
    r = sel3(p0, p1, p2, g.map2crs[1]);
    s = sel3(p0, p1, p2, g.map2crs[2]);
}

// DensityHeader.crs2xyzCoord (pdb_eda/ccp4.py:304-316).
__device__ __forceinline__ void crs2xyz(const pe_geom &g, int c, int r, int s, double &x, double &y, double &z) {
    const int k0 = sel3(c, r, s, g.map2xyz[0]);
    const int k1 = sel3(c, r, s, g.map2xyz[1]);
    const int k2 = sel3(c, r, s, g.map2xyz[2]);
    if (g.orthogonal) {
        x = __dadd_rn(__dmul_rn((double)k0, g.grid_length[0]), g.origin[0]);
        y = __dadd_rn(__dmul_rn((double)k1, g.grid_length[1]), g.origin[1]);
        z = __dadd_rn(__dmul_rn((double)k2, g.grid_length[2]), g.origin[2]);
    } else {
        const double f0 = __ddiv_rn((double)(k0 + g.crs_start[g.map2xyz[0]]), (double)g.xyz_interval[0]);
        const double f1 = __ddiv_rn((double)(k1 + g.crs_start[g.map2xyz[1]]), (double)g.xyz_interval[1]);
        const double f2 = __ddiv_rn((double)(k2 + g.crs_start[g.map2xyz[2]]), (double)g.xyz_interval[2]);
        x = mv_row(g.ortho + 0, f0, f1, f2, g);
        y = mv_row(g.ortho + 3, f0, f1, f2, g);
        z = mv_row(g.ortho + 6, f0, f1, f2, g);
    }
}

// Squared distance exactly as _testXyzWithinDistance forms it before the sqrt (pdb_eda/cutils.pyx:218).
__device__ __forceinline__ double dist2(double ax, double ay, double az, double bx, double by, double bz) {
    const double dx = __dsub_rn(bx, ax), dy = __dsub_rn(by, ay), dz = __dsub_rn(bz, az);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// Largest double T with sqrt_rn(T) <= r.  sqrt_rn is monotone, so  sqrt_rn(d2) <= r  <=>  d2 <= T.
// (r is a float32 widened to double, so r*r is exact and the search takes a couple of steps.)
__device__ __forceinline__ double sphere_threshold(double r) {
    if (!(r >= 0.0)) return -1.0;  // negative or NaN radius: nothing is within distance
    if (isinf(r)) return r;
    double t = __dmul_rn(r, r);
    while (t > 0.0 && __dsqrt_rn(t) > r) t = __longlong_as_double(__double_as_longlong(t) - 1);
    for (;;) {
        const double u = __longlong_as_double(__double_as_longlong(t) + 1);
        if (__dsqrt_rn(u) <= r)
            t = u;
        else
            break;
    }
    return t;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ int warp_excl_scan(int v, int lane) {
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(kFull, x, o);
        if (lane >= o) x += y;
    }
    return x - v;
}

// ------------------------------------------------------------------------------------------------ union-find
// Lock-free union-find over uint32 node ids; a root is always the smallest id of its set, which is what makes
// the labels canonical (blob number = rank of the blob's first voxel in the reference's scan order).
__device__ __forceinline__ uint32_t uf_find(const uint32_t *parent, uint32_t x) {
    uint32_t p = __ldcg(parent + x);
    while (p != x) {
        x = p;
        p = __ldcg(parent + x);
    }
    return x;
}
// find with path halving: every visited node is re-pointed at its grandparent.  The plain stores race with the
// atomicMin hooks benignly: a node only ever points at a smaller id of its own (eventual) set, and a thread whose
// hook is overwritten carries on uniting the roots it saw (see uf_union).
__device__ __forceinline__ uint32_t uf_find_halve(uint32_t *parent, uint32_t x) {
    uint32_t p = __ldcg(parent + x);
    while (p != x) {
        const uint32_t gp = __ldcg(parent + p);
        if (gp != p) __stcg(parent + x, gp);
        x = p;
        p = gp;
    }
    return x;
}
__device__ __forceinline__ void uf_union(uint32_t *parent, uint32_t a, uint32_t b) {
    {
        // two nodes with the same parent are in one set already: one round trip instead of two finds (the common case once a
        // component's nodes point at its root)
        const uint32_t pa = __ldcg(parent + a), pb = __ldcg(parent + b);
        if (pa == pb || pa == b || pb == a) return;
        a = pa;
        b = pb;
    }
    for (;;) {
        a = uf_find_halve(parent, a);
        b = uf_find_halve(parent, b);
        if (a == b) return;
        if (a < b) {
            const uint32_t t = a;
            a = b;
            b = t;
        }
        const uint32_t old = atomicMin(parent + a, b);  // hook the larger root under the smaller
        if (old == a) return;
        a = old;
    }
}

// The same union with L1-CACHED parent loads.  A stale parent is still an ancestor (pointers only ever move to smaller ids of the
// same set), so finds through stale lines are merely longer, "same ancestor" still proves "same set", and the hook itself is an
// atomicMin whose return value is fresh: a stale "root" that has been hooked meanwhile is found out there and the loop carries on
// from its real parent.  What the cache buys: thousands of warps unite into the same few giant sets, and with ld.cg every one of
// their finds reads the root's line from its one L2 slice.  Only for kernels whose results are read by LATER launches.
__device__ __forceinline__ uint32_t uf_find_halve_cached(uint32_t *parent, uint32_t x) {
    uint32_t p = parent[x];
    while (p != x) {
        const uint32_t gp = parent[p];
        if (gp != p) __stcg(parent + x, gp);
        x = p;
        p = gp;
    }
    return x;
}
__device__ __forceinline__ void uf_union_cached(uint32_t *parent, uint32_t a, uint32_t b) {
    {
        const uint32_t pa = parent[a], pb = parent[b];
        if (pa == pb || pa == b || pb == a) return;
        a = pa;
        b = pb;
    }
    for (;;) {
        a = uf_find_halve_cached(parent, a);
        b = uf_find_halve_cached(parent, b);
        if (a == b) return;
        if (a < b) {
            const uint32_t t = a;
            a = b;
            b = t;
        }
        const uint32_t old = atomicMin(parent + a, b);  // hook the larger root under the smaller
        if (old == a) return;
        a = old;
    }
}

// ------------------------------------------------------------------------------------------------ scans (pe_scan.cu)
// Exclusive prefix sum of n uint32 values (n read from d_n when non-null, else n_host) in three launches.
// d_total (may be null) receives the grand total as int64.  d_block_ws: >= scan_ws_bytes(capacity) bytes.
int64_t scan_ws_bytes(int64_t capacity);
int exclusive_scan_u32(const uint32_t *d_in, uint32_t *d_out, int64_t capacity, const int64_t *d_n, int64_t *d_total,
                       void *d_block_ws, cudaStream_t stream, bool popcount_input);

}  // namespace pe
