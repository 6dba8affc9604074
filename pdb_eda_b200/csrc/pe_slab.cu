// pe_slab.cu -- merging the blob labels of a map that is cut into slabs along the section axis, one slab per GPU
// (BASELINE.json config 4).  The reference holds a whole map in one process and clusters with an N x N distance matrix
// (pdb_eda/ccp4.py:123-124, :337-338; pdb_eda/cutils.pyx:41-70), so it has no counterpart of this file; what is reproduced
// is its RESULT on the whole map: 26-connected components without periodic wrap, numbered by their smallest
// (column-slowest) voxel (pdb_eda/cutils.pyx:59-69, SURVEY.md App. A.5), and DensityBlob.fromCrsList's sums per blob
// (pdb_eda/ccp4.py:522-545).
//
// Every rank labels its slab with pe_blob_label, then
//   pe_slab_boundary  packs ONE exchange buffer per rank: per sign the number of local blobs, each blob's smallest GLOBAL
//                     canonical key (ascending in the local blob number) and the voxels (column, row, blob) of the slab's
//                     first and last section;
//   (the caller all-gathers the buffers: the only data-path collective besides the final all-reduce of the sums)
//   pe_slab_merge     on every rank, redundantly and deterministically: for every cut the first plane of the upper slab is
//                     painted into a dense (column, row) plane and the last plane of the lower slab looks at its 9 neighbours
//                     there -> union-find over all ranks' blobs; a merged blob is represented by its member with the smallest
//                     key; the new number of a blob = how many representatives of ALL ranks have a smaller key, found by one
//                     binary search per rank in the gathered (sorted) key arrays -- no global sort;
//   pe_slab_relabel   re-numbers this rank's voxels and accumulates the per-blob sums from the voxels with the WHOLE map's
//                     geometry (global section index), into a table the caller all-reduces.
// No host round trip between the stages; capacities are fixed per call and the same on every rank (the buffer layout follows
// them), overflows and buffers packed with other capacities raise a flag.
#include "pe_common.cuh"

namespace pe {

constexpr int kSlabThreads = 256;

// One sign's block: hdr[0] = local blobs, hdr[1] / hdr[2] = voxels of the first / last plane, hdr[3] = slab_stamp of the
// capacities that laid the block out.  The merge reads every rank's block at the offsets ITS capacities give, so all ranks
// must use the same ones; a block with another stamp sets the error flag and the merge leaves the buffers alone.
struct SlabLayout {  // of one sign's block inside a rank's exchange buffer, in bytes
    int64_t hdr, minkey, first, last, size;
};
__host__ __device__ inline unsigned long long slab_stamp(int64_t cap_blobs, int64_t cap_plane) {  // cap_blobs < 2^31, cap_plane < 2^32
    return ((unsigned long long)cap_blobs << 32) | (unsigned long long)cap_plane;
}
__host__ __device__ inline SlabLayout slab_layout(int64_t cap_blobs, int64_t cap_plane) {
    SlabLayout L;
    L.hdr = 0;
    L.minkey = 32;
    L.first = L.minkey + 8 * cap_blobs;
    const int64_t plane = (12 * cap_plane + 7) / 8 * 8;
    L.last = L.first + plane;
    L.size = L.last + plane;
    return L;
}

static int slab_grid(int64_t n) {
    int64_t blocks = (n + kSlabThreads - 1) / kSlabThreads;
    const int64_t max_blocks = (int64_t)sm_count() * 8;
    if (blocks < 1) blocks = 1;
    return (int)(blocks < max_blocks ? blocks : max_blocks);
}

// ------------------------------------------------------------------------------------------------ boundary
__global__ void __launch_bounds__(kSlabThreads)
    slab_boundary_kernel(const int64_t *__restrict__ counts, int64_t cap_voxels, const uint32_t *__restrict__ key,
                         const int32_t *__restrict__ label, int U1, int Uslab, int U2, int s0, int last_is_cut, int64_t cap_blobs,
                         int64_t cap_plane, char *__restrict__ buf, int *__restrict__ d_bad) {
    const int k = blockIdx.y;  // sign
    const SlabLayout L = slab_layout(cap_blobs, cap_plane);
    char *base = buf + (int64_t)k * L.size;
    unsigned long long *hdr = (unsigned long long *)(base + L.hdr);
    unsigned long long *minkey = (unsigned long long *)(base + L.minkey);
    int32_t *first = (int32_t *)(base + L.first), *last = (int32_t *)(base + L.last);
    const int64_t n = counts[2 * k], nb = counts[2 * k + 1];
    // pe_blob_label failed (its counts may then exceed the capacities): no stamp, so that every rank's merge flags this block
    const bool ok = counts[4] == 0 && n <= cap_voxels && nb <= cap_blobs;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        hdr[0] = (unsigned long long)nb;
        hdr[3] = ok ? slab_stamp(cap_blobs, cap_plane) : 0ull;
    }
    if (!ok) {
        if (blockIdx.x == 0 && threadIdx.x == 0) *d_bad = 1;
        return;
    }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t kk = key[k * cap_voxels + i];
        const int b = label[k * cap_voxels + i];
        const int sl = (int)(kk % (uint32_t)Uslab);
        const uint32_t colrow = kk / (uint32_t)Uslab;
        const unsigned long long gkey = (unsigned long long)colrow * (unsigned long long)U2 + (unsigned long long)(s0 + sl);
        atomicMin(minkey + b, gkey);
        if (sl == 0 || (sl == Uslab - 1 && last_is_cut)) {
            const int r = (int)(colrow % (uint32_t)U1), c = (int)(colrow / (uint32_t)U1);
            if (sl == 0) {
                const unsigned long long at = atomicAdd(hdr + 1, 1ull);
                if ((int64_t)at < cap_plane) {
                    first[3 * at] = c;
                    first[3 * at + 1] = r;
                    first[3 * at + 2] = b;
                } else {
                    *d_bad = 1;
                }
            }
            if (sl == Uslab - 1 && last_is_cut) {
                const unsigned long long at = atomicAdd(hdr + 2, 1ull);
                if ((int64_t)at < cap_plane) {
                    last[3 * at] = c;
                    last[3 * at + 1] = r;
                    last[3 * at + 2] = b;
                } else {
                    *d_bad = 1;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ merge
struct MergeArgs {
    const char *gathered;  // world buffers of buf_bytes each
    int64_t buf_bytes, cap_blobs, cap_plane;
    int world, rank, U0, U1;
    int32_t *planes;       // (2 signs) x (world - 1 cuts) x U0 x U1, -1 = empty
    uint32_t *parent;      // 2 x world x cap_blobs
    unsigned long long *compkey;
    uint32_t *absorbed, *absorbed_scan;
    int *bad;              // the error flag (first word of the workspace): set -> the later merge kernels do nothing
};

__device__ __forceinline__ const char *sign_block(const MergeArgs &a, int rank, int k) {
    return a.gathered + (int64_t)rank * a.buf_bytes + (int64_t)k * slab_layout(a.cap_blobs, a.cap_plane).size;
}
__device__ __forceinline__ int64_t blob_count(const MergeArgs &a, int rank, int k) {
    return (int64_t)((const unsigned long long *)sign_block(a, rank, k))[0];
}

// also checks the header of every rank's blocks before any kernel reads their contents: the stamp of this call's capacities,
// counts within them.  Every rank flags the same blocks, so a failure on one rank stops all ranks before the all-reduce.
__global__ void __launch_bounds__(kSlabThreads) slab_init_kernel(MergeArgs a) {
    const int64_t total = 2ll * a.world * a.cap_blobs;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if (blockIdx.x == 0)
        for (int slot = threadIdx.x; slot < 2 * a.world; slot += blockDim.x) {
            const unsigned long long *hdr = (const unsigned long long *)sign_block(a, slot % a.world, slot / a.world);
            if (hdr[3] != slab_stamp(a.cap_blobs, a.cap_plane) || hdr[0] > (unsigned long long)a.cap_blobs ||
                hdr[1] > (unsigned long long)a.cap_plane || hdr[2] > (unsigned long long)a.cap_plane)
                *a.bad = 1;
        }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        a.parent[i] = (uint32_t)i;
        a.compkey[i] = ~0ull;
        a.absorbed[i] = 0u;
    }
}

// blockIdx.y = sign * (world - 1) + cut: paints the first plane of rank cut + 1
__global__ void __launch_bounds__(kSlabThreads) slab_paint_kernel(MergeArgs a) {
    if (*a.bad) return;
    const int k = blockIdx.y / (a.world - 1), cut = blockIdx.y % (a.world - 1);
    const SlabLayout L = slab_layout(a.cap_blobs, a.cap_plane);
    const char *blk = sign_block(a, cut + 1, k);
    const int64_t n = (int64_t)((const unsigned long long *)blk)[1];
    const int32_t *first = (const int32_t *)(blk + L.first);
    int32_t *plane = a.planes + (int64_t)blockIdx.y * a.U0 * a.U1;
    const uint32_t gbase = (uint32_t)(((int64_t)k * a.world + cut + 1) * a.cap_blobs);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n && i < a.cap_plane; i += stride)
        plane[(int64_t)first[3 * i] * a.U1 + first[3 * i + 1]] = (int32_t)(gbase + (uint32_t)first[3 * i + 2]);
}

// the last plane of rank `cut` against the painted plane: 26-adjacency across the cut = the 9 (column, row) neighbours
__global__ void __launch_bounds__(kSlabThreads) slab_union_kernel(MergeArgs a) {
    if (*a.bad) return;
    const int k = blockIdx.y / (a.world - 1), cut = blockIdx.y % (a.world - 1);
    const SlabLayout L = slab_layout(a.cap_blobs, a.cap_plane);
    const char *blk = sign_block(a, cut, k);
    const int64_t n = (int64_t)((const unsigned long long *)blk)[2];
    const int32_t *last = (const int32_t *)(blk + L.last);
    const int32_t *plane = a.planes + (int64_t)blockIdx.y * a.U0 * a.U1;
    const uint32_t gbase = (uint32_t)(((int64_t)k * a.world + cut) * a.cap_blobs);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n && i < a.cap_plane; i += stride) {
        const int c = last[3 * i], r = last[3 * i + 1];
        const uint32_t me = gbase + (uint32_t)last[3 * i + 2];
        for (int dc = -1; dc <= 1; ++dc) {
            const int c2 = c + dc;
            if (c2 < 0 || c2 >= a.U0) continue;
            for (int dr = -1; dr <= 1; ++dr) {
                const int r2 = r + dr;
                if (r2 < 0 || r2 >= a.U1) continue;
                const int32_t other = plane[(int64_t)c2 * a.U1 + r2];
                if (other >= 0) uf_union(a.parent, me, (uint32_t)other);
            }
        }
    }
}

// smallest key of every merged blob (at its union-find root)
__global__ void __launch_bounds__(kSlabThreads) slab_compkey_kernel(MergeArgs a) {
    if (*a.bad) return;
    const int slot = blockIdx.y;  // sign * world + rank
    const int k = slot / a.world, rank = slot % a.world;
    const char *blk = sign_block(a, rank, k);
    const int64_t nb = min(blob_count(a, rank, k), a.cap_blobs);
    const unsigned long long *minkey = (const unsigned long long *)(blk + slab_layout(a.cap_blobs, a.cap_plane).minkey);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nb; i += stride) {
        const uint32_t gid = (uint32_t)((int64_t)slot * a.cap_blobs + i);
        const uint32_t root = uf_find(a.parent, gid);
        atomicMin(a.compkey + root, minkey[i]);
    }
}

// a blob is absorbed when it is not the member of its merged blob that carries the smallest key
__global__ void __launch_bounds__(kSlabThreads) slab_absorbed_kernel(MergeArgs a) {
    if (*a.bad) return;
    const int slot = blockIdx.y;
    const int k = slot / a.world, rank = slot % a.world;
    const char *blk = sign_block(a, rank, k);
    const int64_t nb = min(blob_count(a, rank, k), a.cap_blobs);
    const unsigned long long *minkey = (const unsigned long long *)(blk + slab_layout(a.cap_blobs, a.cap_plane).minkey);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nb; i += stride) {
        const uint32_t gid = (uint32_t)((int64_t)slot * a.cap_blobs + i);
        a.absorbed[gid] = a.compkey[uf_find(a.parent, gid)] != minkey[i] ? 1u : 0u;
    }
}

// new number of every blob of THIS rank (blockIdx.y = sign) + the number of merged blobs per sign
__global__ void __launch_bounds__(kSlabThreads)
    slab_number_kernel(MergeArgs a, int32_t *__restrict__ new_number /* 2 x cap_blobs */, int64_t *__restrict__ n_merged /* 2 */) {
    if (*a.bad) return;
    const int k = blockIdx.y;
    const SlabLayout L = slab_layout(a.cap_blobs, a.cap_plane);
    const int64_t nb = min(blob_count(a, a.rank, k), a.cap_blobs);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        int64_t total = 0;
        for (int r = 0; r < a.world; ++r) {
            const int64_t n = min(blob_count(a, r, k), a.cap_blobs);
            const int64_t base = ((int64_t)k * a.world + r) * a.cap_blobs;
            // absorbed_scan is an exclusive scan over the whole id space (one spare entry at its end)
            total += n - (int64_t)(a.absorbed_scan[base + n] - a.absorbed_scan[base]);
        }
        n_merged[k] = total;
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nb; i += stride) {
        const uint32_t gid = (uint32_t)(((int64_t)k * a.world + a.rank) * a.cap_blobs + i);
        const unsigned long long ck = a.compkey[uf_find(a.parent, gid)];
        int64_t number = 0;
        for (int r = 0; r < a.world; ++r) {
            const char *blk = sign_block(a, r, k);
            const int64_t n = min((int64_t)((const unsigned long long *)blk)[0], a.cap_blobs);
            const unsigned long long *keys = (const unsigned long long *)(blk + L.minkey);
            int64_t lo = 0, hi = n;  // first position with keys[pos] >= ck
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if (keys[mid] < ck)
                    lo = mid + 1;
                else
                    hi = mid;
            }
            const int64_t base = ((int64_t)k * a.world + r) * a.cap_blobs;
            // pos <= cap_blobs - 1 or pos == n == cap_blobs: the scan array has one spare entry per call (see the layout)
            const uint32_t before = a.absorbed_scan[base + lo] - a.absorbed_scan[base];
            number += lo - (int64_t)before;
        }
        new_number[(int64_t)k * a.cap_blobs + i] = (int32_t)number;
    }
}

// ------------------------------------------------------------------------------------------------ relabel + sums
__global__ void __launch_bounds__(kSlabThreads)
    slab_relabel_kernel(const __grid_constant__ pe_geom g /* whole map */, const int64_t *__restrict__ counts, int64_t cap_voxels,
                        const uint32_t *__restrict__ key, const float *__restrict__ value, int32_t *__restrict__ label, int Uslab,
                        int s0, int64_t cap_blobs, const int32_t *__restrict__ new_number, const int64_t *__restrict__ n_merged,
                        int64_t cap_merged, double *__restrict__ stats /* 2 x cap_merged x 8 */, int *__restrict__ d_bad) {
    if (*d_bad) return;  // the merge did not run: new_number / n_merged are not this call's
    const int k = blockIdx.y;
    const int lane = threadIdx.x & 31;
    const int64_t n = counts[2 * k];
    if (n_merged[k] > cap_merged) {
        if (blockIdx.x == 0 && threadIdx.x == 0) *d_bad = 1;
        return;
    }
    const int U1 = g.unique_ncrs[1];
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t start = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t i0 = start - lane; i0 < n; i0 += stride) {
        const int64_t i = i0 + lane;
        int32_t blob = -1;
        double v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (i < n) {
            const int64_t at = (int64_t)k * cap_voxels + i;
            blob = new_number[(int64_t)k * cap_blobs + label[at]];
            label[at] = blob;
            const uint32_t kk = key[at];
            const int sl = (int)(kk % (uint32_t)Uslab);
            const uint32_t colrow = kk / (uint32_t)Uslab;
            const int r = (int)(colrow % (uint32_t)U1), c = (int)(colrow / (uint32_t)U1);
            double x, y, z;
            crs2xyz(g, c, r, s0 + sl, x, y, z);
            const double d = (double)value[at];
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
        const int segno = __popc(heads & (0xffffffffu >> (31 - lane)));
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int seg_o = __shfl_down_sync(kFull, segno, o);
            const bool take = (lane + o < 32) && (seg_o == segno);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const double other = __shfl_down_sync(kFull, v[q], o);
                if (take) v[q] += other;
            }
        }
        if (blob >= 0 && head) {
            double *st = stats + ((int64_t)k * cap_merged + blob) * 8;
#pragma unroll
            for (int q = 0; q < 8; ++q) atomicAdd(st + q, v[q]);
        }
    }
}

struct MergeWs {
    int64_t flags, planes, parent, compkey, absorbed, absorbed_scan, scan, total;
};
static MergeWs merge_ws(int world, int64_t cap_blobs, int U0, int U1) {
    MergeWs w;
    int64_t p = 0;
    auto take = [&](int64_t bytes) {
        const int64_t at = p;
        p += align_up(bytes > 0 ? bytes : 1, 256);
        return at;
    };
    const int64_t ids = 2ll * world * cap_blobs + 1;
    w.flags = take(256);
    w.planes = take(2ll * (world > 1 ? world - 1 : 1) * U0 * U1 * 4);
    w.parent = take(ids * 4);
    w.compkey = take(ids * 8);
    w.absorbed = take(ids * 4);
    w.absorbed_scan = take(ids * 4);
    w.scan = take(scan_ws_bytes(ids));
    w.total = p;
    return w;
}

}  // namespace pe

using namespace pe;

extern "C" {

int64_t pe_slab_exchange_bytes(int64_t cap_blobs, int64_t cap_plane) {
    if (cap_blobs < 0 || cap_plane < 0) return -1;
    return 2 * slab_layout(cap_blobs, cap_plane).size;
}

int64_t pe_slab_workspace_bytes(int32_t world, int64_t cap_blobs, int32_t u0, int32_t u1) {
    if (world < 1 || cap_blobs < 0 || u0 < 0 || u1 < 0) return -1;
    return merge_ws(world, cap_blobs, u0, u1).total;
}

int pe_slab_boundary(const pe_geom *g_slab, int32_t u2_whole, int32_t s0, int32_t last_is_cut, const int64_t *d_counts, int64_t cap_voxels,
                     const uint32_t *d_key, const int32_t *d_label, int64_t cap_blobs, int64_t cap_plane, void *d_exchange, void *d_ws,
                     void *stream) {
    if (int rc = check_geom(g_slab)) return rc;
    PE_CHECK_ARG(d_counts && d_key && d_label && d_exchange && d_ws, "pe_slab_boundary: null pointer");
    PE_CHECK_ARG(cap_voxels > 0 && cap_blobs > 0 && cap_plane > 0, "pe_slab_boundary: capacities must be positive");
    PE_CHECK_ARG(cap_blobs < (1ll << 31) && cap_plane < (1ll << 32), "pe_slab_boundary: capacities out of range");
    cudaStream_t st = (cudaStream_t)stream;
    const SlabLayout L = slab_layout(cap_blobs, cap_plane);
    char *buf = (char *)d_exchange;
    int *d_bad = (int *)d_ws;  // first word of the merge workspace
    PE_CUDA(cudaMemsetAsync(d_bad, 0, 256, st));
    for (int k = 0; k < 2; ++k) {
        PE_CUDA(cudaMemsetAsync(buf + k * L.size + L.hdr, 0, 32, st));
        PE_CUDA(cudaMemsetAsync(buf + k * L.size + L.minkey, 0xff, (size_t)cap_blobs * 8, st));
    }
    dim3 grid(slab_grid(cap_voxels), 2);
    PE_LAUNCH("slab_boundary_kernel", st, slab_boundary_kernel<<<grid, kSlabThreads, 0, st>>>(
        d_counts, cap_voxels, d_key, d_label, g_slab->unique_ncrs[1], g_slab->unique_ncrs[2], u2_whole, s0, last_is_cut, cap_blobs, cap_plane,
        buf, d_bad));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

int pe_slab_merge(int32_t world, int32_t rank, const void *d_gathered, int64_t cap_blobs, int64_t cap_plane, int32_t u0, int32_t u1,
                  int32_t *d_new_number, int64_t *d_n_merged, void *d_ws, void *stream) {
    PE_CHECK_ARG(world >= 1 && rank >= 0 && rank < world, "pe_slab_merge: bad rank / world");
    PE_CHECK_ARG(d_gathered && d_new_number && d_n_merged && d_ws, "pe_slab_merge: null pointer");
    PE_CHECK_ARG(2ll * world * cap_blobs < (1ll << 31), "pe_slab_merge: too many blobs for 32-bit ids");
    PE_CHECK_ARG(cap_blobs > 0 && cap_plane > 0 && cap_plane < (1ll << 32), "pe_slab_merge: capacities out of range");
    cudaStream_t st = (cudaStream_t)stream;
    const MergeWs w = merge_ws(world, cap_blobs, u0, u1);
    char *ws = (char *)d_ws;
    MergeArgs a;
    a.gathered = (const char *)d_gathered;
    a.buf_bytes = 2 * slab_layout(cap_blobs, cap_plane).size;
    a.cap_blobs = cap_blobs;
    a.cap_plane = cap_plane;
    a.world = world;
    a.rank = rank;
    a.U0 = u0;
    a.U1 = u1;
    a.planes = (int32_t *)(ws + w.planes);
    a.parent = (uint32_t *)(ws + w.parent);
    a.compkey = (unsigned long long *)(ws + w.compkey);
    a.absorbed = (uint32_t *)(ws + w.absorbed);
    a.absorbed_scan = (uint32_t *)(ws + w.absorbed_scan);
    a.bad = (int *)(ws + w.flags);
    const int64_t ids = 2ll * world * cap_blobs + 1;
    PE_LAUNCH("slab_init_kernel", st, slab_init_kernel<<<slab_grid(ids), kSlabThreads, 0, st>>>(a));
    if (world > 1) {
        PE_CUDA(cudaMemsetAsync(a.planes, 0xff, (size_t)2 * (world - 1) * u0 * u1 * 4, st));
        dim3 grid(slab_grid(cap_plane) < 64 ? slab_grid(cap_plane) : 64, 2 * (world - 1));
        PE_LAUNCH("slab_paint_kernel", st, slab_paint_kernel<<<grid, kSlabThreads, 0, st>>>(a));
        PE_LAUNCH("slab_union_kernel", st, slab_union_kernel<<<grid, kSlabThreads, 0, st>>>(a));
    }
    dim3 grid_b(slab_grid(cap_blobs), 2 * world);
    PE_LAUNCH("slab_compkey_kernel", st, slab_compkey_kernel<<<grid_b, kSlabThreads, 0, st>>>(a));
    PE_LAUNCH("slab_absorbed_kernel", st, slab_absorbed_kernel<<<grid_b, kSlabThreads, 0, st>>>(a));
    PE_LAUNCH_CHECK();
    PE_CUDA(cudaMemsetAsync(a.absorbed + (ids - 1), 0, 4, st));
    if (int rc = exclusive_scan_u32(a.absorbed, a.absorbed_scan, ids, nullptr, nullptr, ws + w.scan, st, false)) return rc;
    dim3 grid_n(slab_grid(cap_blobs), 2);
    PE_LAUNCH("slab_number_kernel", st, slab_number_kernel<<<grid_n, kSlabThreads, 0, st>>>(a, d_new_number, d_n_merged));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

/* Error flag of the slab calls on this workspace (a capacity was exceeded); synchronises the stream. */
int pe_slab_status(const void *d_ws, void *stream, int32_t *bad) {
    PE_CHECK_ARG(d_ws && bad, "pe_slab_status: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    PE_CUDA(cudaMemcpyAsync(bad, d_ws, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    PE_CUDA(cudaStreamSynchronize(st));
    return PE_OK;
}

int pe_slab_relabel(const pe_geom *g_whole, int32_t u2_slab, int32_t s0, const int64_t *d_counts, int64_t cap_voxels, const uint32_t *d_key,
                    const float *d_value, int32_t *d_label, int64_t cap_blobs, const int32_t *d_new_number, const int64_t *d_n_merged,
                    int64_t cap_merged, double *d_stats, void *d_ws, void *stream) {
    if (int rc = check_geom_shape(g_whole, nullptr)) return rc;  // only crs -> xyz of the whole map: no 2^31-voxel limit here
    PE_CHECK_ARG(d_counts && d_key && d_value && d_label && d_new_number && d_n_merged && d_stats && d_ws, "pe_slab_relabel: null pointer");
    PE_CHECK_ARG(cap_voxels > 0 && cap_blobs > 0 && cap_merged > 0 && u2_slab > 0, "pe_slab_relabel: capacities must be positive");
    cudaStream_t st = (cudaStream_t)stream;
    PE_CUDA(cudaMemsetAsync(d_stats, 0, (size_t)2 * cap_merged * 8 * sizeof(double), st));
    dim3 grid(slab_grid(cap_voxels), 2);
    PE_LAUNCH("slab_relabel_kernel", st, slab_relabel_kernel<<<grid, kSlabThreads, 0, st>>>(
        *g_whole, d_counts, cap_voxels, d_key, d_value, d_label, u2_slab, s0, cap_blobs, d_new_number, d_n_merged, cap_merged, d_stats,
        (int *)d_ws));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

}  // extern "C"
