// pe_cluster.cu -- set algebra on arbitrary lists of un-wrapped voxels: 26-connected clustering, de-duplication,
// per-cluster sums and pairwise overlap tests.
//
// Replaces
//   createCrsLists            pdb_eda/cutils.pyx:41-70     N x N cdist + breadth-first growth from the first unused
//                                                          index; adjacency = Euclidean index distance <= sqrt(3),
//                                                          i.e. all |delta| <= 1, no periodic wrap
//   DensityBlob.fromCrsList   pdb_eda/ccp4.py:522-545      per-blob sums (also what DensityBlob.merge recomputes, :575-586)
//   testOverlap               pdb_eda/cutils.pyx:8-25      any voxel pair with all |delta| <= 1 (identical voxels count)
// and, built from those, the residue / domain cloud merging of aggregateCloud (pdb_eda/densityAnalysis.py:646-708):
// clouds that overlap transitively are merged into one voxel SET, so a merged cloud is a 26-connected component
// of the union of its members' voxels, and its sums run over each distinct voxel once.
//
// All neighbour queries go through an open-addressing hash table in the caller's workspace (packed 64-bit key ->
// chain of input indices), so memory is O(N) instead of the reference's O(N^2) distance matrix (46 GB at 384^3,
// SURVEY.md section 3.3).  Clusters are numbered by their smallest input index ("root = smallest id" union-find,
// then ranking the roots), which is the order createCrsLists creates them in.
//
// Entries may carry a group id (e.g. the residue a cloud voxel belongs to): voxels only see voxels of their own
// group.  Key layout: without groups 3 x 21 bits (|index| < 2^20, i.e. -1048575 .. 1048575); with groups 22 bits of
// group + 3 x 14 bits (|index| < 2^13, i.e. -8191 .. 8191, and 0 <= group < 2^22) -- checked on the device, anything
// else (including -2^20 / -2^13 and a negative group) raises the overflow flag.
#include "pe_common.cuh"

namespace pe {

constexpr int kClThreads = 256;
constexpr uint64_t kEmptyKey = ~0ull;
constexpr uint32_t kNil = 0xffffffffu;

// An axis field holds index + (2^(bits-1) - 1), i.e. 0 .. 2^bits - 2 for |index| < 2^(bits-1): the all-ones field is never
// used, so no valid key equals kEmptyKey (with groups the key fills all 64 bits).
__device__ __forceinline__ bool pack_crs(int c, int r, int s, int group, bool grouped, uint64_t &key) {
    if (grouped) {
        const int off = (1 << 13) - 1;
        const unsigned top = (1u << 14) - 2u;
        const unsigned uc = (unsigned)(c + off), ur = (unsigned)(r + off), us = (unsigned)(s + off);
        if (uc > top || ur > top || us > top || (unsigned)group >> 22) return false;
        key = ((uint64_t)(unsigned)group << 42) | ((uint64_t)uc << 28) | ((uint64_t)ur << 14) | (uint64_t)us;
    } else {
        const int off = (1 << 20) - 1;
        const unsigned top = (1u << 21) - 2u;
        const unsigned uc = (unsigned)(c + off), ur = (unsigned)(r + off), us = (unsigned)(s + off);
        if (uc > top || ur > top || us > top) return false;
        key = ((uint64_t)uc << 42) | ((uint64_t)ur << 21) | (uint64_t)us;
    }
    return true;
}
__device__ __forceinline__ uint64_t hash_slot(uint64_t key, int log2cap) {
    return (key * 0x9E3779B97F4A7C15ull) >> (64 - log2cap);
}

struct VoxelTable {
    unsigned long long *key;  // cap slots, kEmptyKey when free
    uint32_t *head;           // cap slots: most recently inserted input index of the slot's chain
    uint32_t *next;           // n entries: previous entry with the same key, or kNil
    int log2cap;
};

// Inserts every entry; entries with the same key (same voxel, same group) are chained.
__global__ void __launch_bounds__(kClThreads)
    table_insert_kernel(int64_t n, const int32_t *__restrict__ crs, const int32_t *__restrict__ group, VoxelTable t,
                        int *__restrict__ d_bad) {
    const uint64_t mask = (1ull << t.log2cap) - 1;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        uint64_t key;
        if (!pack_crs(crs[3 * i], crs[3 * i + 1], crs[3 * i + 2], group ? group[i] : 0, group != nullptr, key)) {
            *d_bad = 1;
            t.next[i] = kNil;
            continue;
        }
        uint64_t h = hash_slot(key, t.log2cap);
        for (;;) {
            unsigned long long old = t.key[h];
            if (old == kEmptyKey) old = atomicCAS(t.key + h, (unsigned long long)kEmptyKey, (unsigned long long)key);
            if (old == kEmptyKey || old == key) {
                t.next[i] = atomicExch(t.head + h, (uint32_t)i);
                break;
            }
            h = (h + 1) & mask;
        }
    }
}

// Head of the chain stored for `key`, or kNil.
__device__ __forceinline__ uint32_t table_lookup(const VoxelTable &t, uint64_t key) {
    const uint64_t mask = (1ull << t.log2cap) - 1;
    uint64_t h = hash_slot(key, t.log2cap);
    for (;;) {
        const unsigned long long k = t.key[h];
        if (k == key) return t.head[h];
        if (k == kEmptyKey) return kNil;
        h = (h + 1) & mask;
    }
}

__device__ __forceinline__ uint32_t chain_min(const VoxelTable &t, uint32_t j) {
    uint32_t m = kNil;
    for (; j != kNil; j = t.next[j]) m = min(m, j);
    return m;
}

// first[i] = 1 iff i is the first input entry holding its (group, voxel); duplicates are united with it.
__global__ void __launch_bounds__(kClThreads)
    cluster_first_kernel(int64_t n, const int32_t *__restrict__ crs, const int32_t *__restrict__ group, VoxelTable t,
                         uint32_t *__restrict__ parent, uint8_t *__restrict__ first) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        uint64_t key;
        uint32_t m = (uint32_t)i;
        if (pack_crs(crs[3 * i], crs[3 * i + 1], crs[3 * i + 2], group ? group[i] : 0, group != nullptr, key))
            m = chain_min(t, table_lookup(t, key));
        parent[i] = m;  // m <= i: a valid "smaller id" parent
        if (first) first[i] = m == (uint32_t)i ? 1 : 0;
    }
}

__global__ void __launch_bounds__(kClThreads)
    cluster_merge_kernel(int64_t n, const int32_t *__restrict__ crs, const int32_t *__restrict__ group, VoxelTable t,
                         uint32_t *parent) {
    // 13 of the 26 neighbours suffice: adjacency is symmetric and every voxel looks "backwards".
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int c = crs[3 * i], r = crs[3 * i + 1], s = crs[3 * i + 2];
        const int gi = group ? group[i] : 0;
#pragma unroll
        for (int q = 0; q < 13; ++q) {
            const int dc = q < 9 ? -1 : 0;
            const int dr = q < 9 ? (q / 3) - 1 : (q < 12 ? -1 : 0);
            const int ds = q < 9 ? (q % 3) - 1 : (q < 12 ? (q - 9) - 1 : -1);
            uint64_t key;
            if (!pack_crs(c + dc, r + dr, s + ds, gi, group != nullptr, key)) continue;
            const uint32_t j = table_lookup(t, key);
            if (j != kNil) uf_union(parent, (uint32_t)i, j);  // any entry of the chain: they share one root
        }
    }
}

__global__ void __launch_bounds__(kClThreads)
    cluster_flatten_kernel(int64_t n, uint32_t *parent, uint32_t *__restrict__ flag) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t root = uf_find(parent, (uint32_t)i);
        parent[i] = root;
        flag[i] = root == (uint32_t)i ? 1u : 0u;
    }
}

__global__ void __launch_bounds__(kClThreads)
    cluster_label_kernel(int64_t n, const uint32_t *__restrict__ parent, const uint32_t *__restrict__ rank,
                         int32_t *__restrict__ label) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) label[i] = (int32_t)rank[parent[i]];
}

// ------------------------------------------------------------------------------------------------ per-cluster sums
// DensityBlob.fromCrsList (pdb_eda/ccp4.py:522-545) for every cluster at once.  Consecutive entries of one cluster
// are combined by a segmented warp reduction before the float64 atomics.
__global__ void __launch_bounds__(kClThreads)
    crs_stats_kernel(const __grid_constant__ pe_geom g, const float *__restrict__ rho, int64_t n,
                     const int32_t *__restrict__ crs, const int32_t *__restrict__ label, const uint8_t *__restrict__ take,
                     int64_t n_clusters, double *__restrict__ stats) {
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t start = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t i0 = start - lane; i0 < n; i0 += stride) {
        const int64_t i = i0 + lane;
        int32_t blob = -1;
        double v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (i < n && (!take || take[i])) {
            blob = label ? label[i] : 0;
            if (blob < 0 || blob >= n_clusters) blob = -1;
        }
        if (blob >= 0) {
            const int c = crs[3 * i], r = crs[3 * i + 1], s = crs[3 * i + 2];
            const int wc = wrap_index(c, g.ncrs[0], g.crs_interval[0]);
            const int wr = wrap_index(r, g.ncrs[1], g.crs_interval[1]);
            const int wsx = wrap_index(s, g.ncrs[2], g.crs_interval[2]);
            const double d = ((wc | wr | wsx) >= 0) ? (double)__ldg(rho + ((int64_t)wsx * g.ncrs[1] + wr) * g.ncrs[0] + wc) : 0.0;
            double x, y, z;
            crs2xyz(g, c, r, s, x, y, z);
            v[0] = 1.0;
            v[1] = d;
            v[2] = __dmul_rn(d, x);
            v[3] = __dmul_rn(d, y);
            v[4] = __dmul_rn(d, z);
            v[5] = x;
            v[6] = y;
            v[7] = z;
        }
        const int32_t prev = __shfl_up_sync(kFull, blob, 1);
        const bool head = (lane == 0) || (prev != blob);
        const unsigned heads = __ballot_sync(kFull, head);
        const int seg = __popc(heads & (0xffffffffu >> (31 - lane)));
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int seg_o = __shfl_down_sync(kFull, seg, o);
            const bool add = (lane + o < 32) && (seg_o == seg);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const double other = __shfl_down_sync(kFull, v[q], o);
                if (add) v[q] += other;
            }
        }
        if (blob >= 0 && head) {
            double *st = stats + (int64_t)blob * 8;
#pragma unroll
            for (int q = 0; q < 8; ++q) atomicAdd(st + q, v[q]);
        }
    }
}

// ------------------------------------------------------------------------------------------------ two-map metrics
// Real-space correlation / R factor over voxel sets (calculateRsccRsrMetrics, pdb_eda/densityAnalysis.py:860-882):
// fo = 2Fo-Fc value, fc = fo - 2 * (Fo-Fc) value formed in float64 exactly as the reference's
// `densityObj.density - diffDensityObj.density * 2` (pdb_eda/densityAnalysis.py:433).  Pass 0 accumulates
// n, sum fo, sum fc, sum |fo - fc|, sum |fo + fc|; pass 1 the centred second moments (two-pass, like scipy's pearsonr).
template <int PASS>
__global__ void __launch_bounds__(kClThreads)
    pair_metrics_kernel(const __grid_constant__ pe_geom g, const float *__restrict__ rho_fo, const float *__restrict__ rho_diff,
                        int64_t n, const int32_t *__restrict__ crs, const int32_t *__restrict__ label,
                        const uint8_t *__restrict__ take, int64_t n_groups, double *__restrict__ out) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (take && !take[i]) continue;
        const int grp = label ? label[i] : 0;
        if (grp < 0 || grp >= n_groups) continue;
        const int wc = wrap_index(crs[3 * i], g.ncrs[0], g.crs_interval[0]);
        const int wr = wrap_index(crs[3 * i + 1], g.ncrs[1], g.crs_interval[1]);
        const int wsx = wrap_index(crs[3 * i + 2], g.ncrs[2], g.crs_interval[2]);
        double fo = 0.0, df = 0.0;
        if ((wc | wr | wsx) >= 0) {
            const int64_t off = ((int64_t)wsx * g.ncrs[1] + wr) * g.ncrs[0] + wc;
            fo = (double)__ldg(rho_fo + off);
            df = (double)__ldg(rho_diff + off);
        }
        const double fc = __dsub_rn(fo, __dmul_rn(df, 2.0));
        double *o = out + (int64_t)grp * 8;
        if (PASS == 0) {
            atomicAdd(o + 0, 1.0);
            atomicAdd(o + 1, fo);
            atomicAdd(o + 2, fc);
            atomicAdd(o + 3, fabs(fo - fc));
            atomicAdd(o + 4, fabs(fo + fc));
        } else {
            const double cnt = o[0];
            const double xm = fo - o[1] / cnt, ym = fc - o[2] / cnt;
            atomicAdd(o + 5, xm * xm);
            atomicAdd(o + 6, ym * ym);
            atomicAdd(o + 7, xm * ym);
        }
    }
}

// ------------------------------------------------------------------------------------------------ overlap pairs
// For every entry, every entry of another owner at an identical or 26-adjacent voxel (same group) yields the
// unordered owner pair; pairs are de-duplicated through a second hash set and appended to the output.
__global__ void __launch_bounds__(kClThreads)
    overlap_pairs_kernel(int64_t n, const int32_t *__restrict__ crs, const int32_t *__restrict__ owner,
                         const int32_t *__restrict__ group, VoxelTable t, unsigned long long *pair_set, int pair_log2cap,
                         int64_t cap_pairs, unsigned long long *__restrict__ d_npairs, int32_t *__restrict__ pairs) {
    const uint64_t pmask = (1ull << pair_log2cap) - 1;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int c = crs[3 * i], r = crs[3 * i + 1], s = crs[3 * i + 2];
        const int gi = group ? group[i] : 0;
        const int oi = owner[i];
        for (int q = 0; q < 27; ++q) {
            uint64_t key;
            if (!pack_crs(c + q / 9 - 1, r + (q / 3) % 3 - 1, s + q % 3 - 1, gi, group != nullptr, key)) continue;
            for (uint32_t j = table_lookup(t, key); j != kNil; j = t.next[j]) {
                const int oj = owner[j];
                if (oj <= oi) continue;  // each unordered pair once, from its smaller owner
                const unsigned long long pk = ((unsigned long long)(uint32_t)oi << 32) | (uint32_t)oj;
                uint64_t h = hash_slot(pk, pair_log2cap);
                for (uint64_t probes = 0;; ++probes) {
                    if (probes > pmask) {  // pair set full: far more distinct pairs than cap_pairs
                        atomicAdd(d_npairs, 1ull);
                        break;
                    }
                    unsigned long long old = pair_set[h];
                    if (old == pk) break;
                    if (old == kEmptyKey) {
                        old = atomicCAS(pair_set + h, (unsigned long long)kEmptyKey, pk);
                        if (old == kEmptyKey) {
                            const unsigned long long slot = atomicAdd(d_npairs, 1ull);
                            if ((int64_t)slot < cap_pairs) {
                                pairs[2 * slot] = oi;
                                pairs[2 * slot + 1] = oj;
                            }
                            break;
                        }
                        if (old == pk) break;
                    }
                    h = (h + 1) & pmask;
                }
            }
        }
    }
}

static int table_log2cap(int64_t n) {
    int l = 6;
    while ((1ll << l) < 2 * n + 16) ++l;
    return l;
}

static int grid_for(int64_t n) {
    int64_t blocks64 = (n + kClThreads - 1) / kClThreads;
    const int64_t max_blocks = (int64_t)sm_count() * 16;
    if (blocks64 < 1) blocks64 = 1;
    return (int)(blocks64 < max_blocks ? blocks64 : max_blocks);
}

// Carves the voxel table out of the workspace and fills it.  Returns the bytes consumed.
static int build_table(int64_t n, const int32_t *d_crs, const int32_t *d_group, char *ws, VoxelTable &t, int *d_bad,
                       cudaStream_t st, int64_t &used) {
    t.log2cap = table_log2cap(n);
    const int64_t cap = 1ll << t.log2cap;
    char *p = ws;
    t.key = (unsigned long long *)p;
    p += align_up(cap * 8, 256);
    t.head = (uint32_t *)p;
    p += align_up(cap * 4, 256);
    t.next = (uint32_t *)p;
    p += align_up(n * 4, 256);
    used = p - ws;
    PE_CUDA(cudaMemsetAsync(t.key, 0xff, cap * 8, st));
    PE_CUDA(cudaMemsetAsync(t.head, 0xff, cap * 4, st));
    PE_LAUNCH("table_insert_kernel", st, table_insert_kernel<<<grid_for(n), kClThreads, 0, st>>>(n, d_crs, d_group, t, d_bad));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

static int64_t table_bytes(int64_t n) {
    const int64_t cap = 1ll << table_log2cap(n);
    return align_up(cap * 8, 256) + align_up(cap * 4, 256) + align_up(n * 4, 256);
}

}  // namespace pe

using namespace pe;

extern "C" {

int64_t pe_cluster_workspace_bytes(int64_t n) {
    if (n < 0) return -1;
    return 256 + table_bytes(n) + 3 * align_up(n * 4, 256) + scan_ws_bytes(n);
}

int pe_cluster_crs_grouped(int64_t n, const int32_t *d_crs, const int32_t *d_group, int32_t *d_label, uint8_t *d_first,
                           int64_t *d_nclusters, void *d_ws, void *stream) {
    PE_CHECK_ARG(n >= 0 && d_nclusters, "pe_cluster_crs: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    PE_CUDA(cudaMemsetAsync(d_nclusters, 0, 2 * sizeof(int64_t), st));
    if (n == 0) return PE_OK;
    PE_CHECK_ARG(d_crs && d_label && d_ws, "pe_cluster_crs: null pointer");
    PE_CHECK_ARG(n < (1ll << 31), "pe_cluster_crs: list too long");
    char *ws = (char *)d_ws;
    int *d_bad = (int *)(d_nclusters + 1);  // second int64 of the counter pair: key-range overflow flag
    ws += 256;
    VoxelTable t;
    int64_t used = 0;
    if (int rc = build_table(n, d_crs, d_group, ws, t, d_bad, st, used)) return rc;
    ws += used;
    uint32_t *parent = (uint32_t *)ws;
    ws += align_up(n * 4, 256);
    uint32_t *flag = (uint32_t *)ws;
    ws += align_up(n * 4, 256);
    uint32_t *rank = (uint32_t *)ws;
    ws += align_up(n * 4, 256);
    void *scan_ws = ws;
    const int blocks = grid_for(n);
    PE_LAUNCH("cluster_first_kernel", st, cluster_first_kernel<<<blocks, kClThreads, 0, st>>>(n, d_crs, d_group, t, parent, d_first));
    PE_LAUNCH("cluster_merge_kernel", st, cluster_merge_kernel<<<blocks, kClThreads, 0, st>>>(n, d_crs, d_group, t, parent));
    PE_LAUNCH("cluster_flatten_kernel", st, cluster_flatten_kernel<<<blocks, kClThreads, 0, st>>>(n, parent, flag));
    PE_LAUNCH_CHECK();
    if (int rc = exclusive_scan_u32(flag, rank, n, nullptr, d_nclusters, scan_ws, st, false)) return rc;
    PE_LAUNCH("cluster_label_kernel", st, cluster_label_kernel<<<blocks, kClThreads, 0, st>>>(n, parent, rank, d_label));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

int pe_cluster_crs(int64_t n, const int32_t *d_crs, int32_t *d_label, int64_t *d_nclusters, void *d_ws, void *stream) {
    return pe_cluster_crs_grouped(n, d_crs, nullptr, d_label, nullptr, d_nclusters, d_ws, stream);
}

int pe_crs_stats(const pe_geom *g, const float *d_rho, int64_t n, const int32_t *d_crs, const int32_t *d_label,
                 const uint8_t *d_take, int64_t n_clusters, double *d_stats, void *stream) {
    if (int rc = check_geom(g)) return rc;
    PE_CHECK_ARG(n >= 0 && n_clusters >= 0, "pe_crs_stats: negative size");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_clusters == 0) return PE_OK;
    PE_CHECK_ARG(d_stats, "pe_crs_stats: null output");
    PE_CUDA(cudaMemsetAsync(d_stats, 0, (size_t)n_clusters * 8 * sizeof(double), st));
    if (n == 0) return PE_OK;
    PE_CHECK_ARG(d_rho && d_crs, "pe_crs_stats: null pointer");
    PE_LAUNCH("crs_stats_kernel", st, crs_stats_kernel<<<grid_for(n), kClThreads, 0, st>>>(*g, d_rho, n, d_crs, d_label, d_take, n_clusters, d_stats));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

int pe_pair_metrics(const pe_geom *g, const float *d_rho_fo, const float *d_rho_diff, int64_t n, const int32_t *d_crs,
                    const int32_t *d_label, const uint8_t *d_take, int64_t n_groups, double *d_out, void *stream) {
    if (int rc = check_geom(g)) return rc;
    PE_CHECK_ARG(n >= 0 && n_groups >= 0, "pe_pair_metrics: negative size");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_groups == 0) return PE_OK;
    PE_CHECK_ARG(d_out, "pe_pair_metrics: null output");
    PE_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n_groups * 8 * sizeof(double), st));
    if (n == 0) return PE_OK;
    PE_CHECK_ARG(d_rho_fo && d_rho_diff && d_crs, "pe_pair_metrics: null pointer");
    PE_LAUNCH("pair_metrics_kernel", st, pair_metrics_kernel<0><<<grid_for(n), kClThreads, 0, st>>>(
        *g, d_rho_fo, d_rho_diff, n, d_crs, d_label, d_take, n_groups, d_out));
    PE_LAUNCH("pair_metrics_kernel", st, pair_metrics_kernel<1><<<grid_for(n), kClThreads, 0, st>>>(
        *g, d_rho_fo, d_rho_diff, n, d_crs, d_label, d_take, n_groups, d_out));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

int64_t pe_overlap_workspace_bytes(int64_t n, int64_t cap_pairs) {
    if (n < 0 || cap_pairs < 0) return -1;
    const int64_t pcap = 1ll << table_log2cap(cap_pairs);
    return 256 + table_bytes(n) + align_up(pcap * 8, 256);
}

int pe_overlap_pairs(int64_t n, const int32_t *d_crs, const int32_t *d_owner, const int32_t *d_group, int64_t cap_pairs,
                     int64_t *d_npairs, int32_t *d_pairs, void *d_ws, void *stream) {
    PE_CHECK_ARG(n >= 0 && cap_pairs >= 0 && d_npairs, "pe_overlap_pairs: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    PE_CUDA(cudaMemsetAsync(d_npairs, 0, 2 * sizeof(int64_t), st));
    if (n == 0) return PE_OK;
    PE_CHECK_ARG(d_crs && d_owner && d_ws && (cap_pairs == 0 || d_pairs), "pe_overlap_pairs: null pointer");
    PE_CHECK_ARG(n < (1ll << 31), "pe_overlap_pairs: list too long");
    char *ws = (char *)d_ws + 256;
    int *d_bad = (int *)(d_npairs + 1);
    VoxelTable t;
    int64_t used = 0;
    if (int rc = build_table(n, d_crs, d_group, ws, t, d_bad, st, used)) return rc;
    ws += used;
    const int plog = table_log2cap(cap_pairs);
    unsigned long long *pair_set = (unsigned long long *)ws;
    PE_CUDA(cudaMemsetAsync(pair_set, 0xff, (size_t)(1ll << plog) * 8, st));
    PE_LAUNCH("overlap_pairs_kernel", st, overlap_pairs_kernel<<<grid_for(n), kClThreads, 0, st>>>(n, d_crs, d_owner, d_group, t, pair_set, plog, cap_pairs,
                                                             (unsigned long long *)d_npairs, d_pairs));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

}  // extern "C"
