// pe_blob.cu -- +/- cutoff thresholding fused with 26-connected component labelling of the difference map.
//
// Replaces  createFullCrsList (pdb_eda/cutils.pyx:185-203) + createCrsLists (pdb_eda/cutils.pyx:41-70) +
// DensityBlob.fromCrsList (pdb_eda/ccp4.py:522-545), i.e. DensityMatrix.createFullBlobList (pdb_eda/ccp4.py:463-485),
// for the green (+cutoff) and red (-cutoff) lists of pdb_eda/densityAnalysis.py:392-412 in one pass over the map.
//
// Design (B200).  The map is read exactly once, by an HBM-bound streaming kernel that thresholds both signs and
// writes two bit planes (1 bit per voxel and class, 1/16 of the bytes read).  The bit planes are stored in the
// REFERENCE'S scan order -- column slowest, section fastest, 32 sections per word -- so that
//   * a popcount prefix sum over the words gives every foreground voxel its position in createFullCrsList's list
//     (deterministic, order-preserving compaction without sorting), and
//   * union-find over those positions with "smaller id wins" makes every blob's root its first voxel in that
//     order, so ranking the roots yields the reference's blob order directly (canonical min-index relabelling).
// Everything after the streaming kernel touches only the bit planes (N/8 bytes) and the sparse foreground.
// Runs of set bits along the section axis are linked at initialisation (parent = first voxel of the run), the
// remaining 12 predecessor neighbours are merged with lock-free atomicMin hooking.  The streaming kernel also
// counts the foreground per 512-word segment of the planes, so the sparse stage knows every voxel's list position
// (and both class totals) without a counting pass of its own.
//
// The transposition (memory order is column-fastest, bit order is section-fastest) costs nothing: a thread owns
// 4 adjacent columns of one row and walks 32 sections, so the 32 loads it issues are independent 16-byte loads
// that are contiguous across the warp (512 B per warp per section), and the word it builds is complete in
// registers.
#include <cooperative_groups.h>
#include "pe_common.cuh"

namespace cg = cooperative_groups;

namespace pe {

constexpr int kBmpTx = 32;         // threads along columns (x VEC columns each)
constexpr int kBmpTy = 8;          // threads along rows
constexpr int kSparseThreads = 512;
constexpr int kSegShift = 9;       // words per counting segment of the bit planes: 512
constexpr int kSegWords = 1 << kSegShift;
constexpr int kChunkShift = 9;     // voxels per root-ranking chunk: 512 (= kSparseThreads)
constexpr int kChunkSmem = 4096;   // chunks whose prefix fits the shared-memory table (2 M voxels)
constexpr int kScanBlocksPerSm = 2;  // blocks per SM that scan the bit planes in P1 (of the 3 resident ones)
constexpr int kQueueCap = 160;     // non-empty words a warp collects before it drains them (P1)
constexpr int kPoolWords = (kSparseThreads / 32) * 3 * kQueueCap > kChunkSmem ? (kSparseThreads / 32) * 3 * kQueueCap : kChunkSmem;
static_assert((1 << kChunkShift) == kSparseThreads, "a ranking chunk is one block of voxels");

struct BlobPlan {
    int U0, U1, U2, W;    // unique columns, rows, sections; words per (column,row)
    int64_t nwords;       // U0*U1*W words per class
    int64_t nwords_pad;   // the same rounded up to a whole segment: distance between the two bit planes
    int64_t nseg;         // counting segments over both planes
    int64_t cap;          // foreground capacity per class
    int64_t nchunk_cap;   // ranking chunks at capacity
    // workspace carve-up
    int64_t off_bmp, off_base, off_parent, off_flags, off_coarse, off_seg, total;
};

static BlobPlan make_plan(const pe_geom *g, int64_t cap) {
    BlobPlan p;
    p.U0 = g->unique_ncrs[0];
    p.U1 = g->unique_ncrs[1];
    p.U2 = g->unique_ncrs[2];
    p.W = ((p.U2 + 31) / 32 + 7) / 8 * 8;  // padded: see threshold_bitmap_kernel
    p.nwords = (int64_t)p.U0 * p.U1 * p.W;
    p.nwords_pad = align_up(p.nwords, kSegWords);
    p.nseg = 2 * p.nwords_pad / kSegWords;
    p.cap = cap;
    p.nchunk_cap = (2 * cap + kSparseThreads - 1) / kSparseThreads + 1;
    int64_t o = 0;
    p.off_bmp = o;
    o += align_up(2 * p.nwords_pad * 4, 256);
    p.off_base = o;
    o += align_up(2 * p.nwords_pad * 4, 256);
    p.off_parent = o;
    o += align_up(2 * cap * 4, 256);
    p.off_flags = o;  // per 32 voxels: root flags + roots before the word inside its chunk
    o += align_up((2 * cap / 32 + 2 * (kSparseThreads / 32)) * 8, 256);  // the last chunk is written whole
    p.off_coarse = o;  // per chunk: roots; then (maps beyond kChunkSmem chunks) their exclusive prefix
    o += align_up(2 * p.nchunk_cap * 4, 256);
    p.off_seg = o;
    o += align_up(p.nseg * 4, 256) + 1024;  // + per-SM block ranks and the count of scanning blocks (zeroed with the counts)
    p.total = o;
    return p;
}

// ------------------------------------------------------------------------------------------------ K1: stream
// W (words per (column, row)) is padded to a multiple of 8, so the kWordsPerThread = 4 words a thread produces for
// one (column, row) are one aligned 16-byte store, and the two thread blocks that share a 32-byte sector are
// neighbours in launch order (the word-group index is blockIdx.x, the fastest-varying block index): every bit-plane
// sector reaches DRAM as one full write.  The kernel also counts the foreground voxels of every 512-word segment of the
// planes (segcount, zeroed by the caller), which is all the sparse stage needs to place every voxel in the list.  Scattered 4-byte word stores cost a read-modify-write per sector once the
// bit planes no longer fit L2 (768^3 ran at 28 % of the HBM peak, tune log in profiles/r01_threshold_tuning.md).
constexpr int kWordsPerThread = 4;

template <int VEC>
__global__ void __launch_bounds__(384)
    threshold_bitmap_kernel(const float *__restrict__ rho, int NC, int NR, int U0, int U1, int U2, int W, float cpos,
                            float cneg, bool use_pos, bool use_neg, uint32_t *__restrict__ bmp_pos,
                            uint32_t *__restrict__ bmp_neg, int64_t nwords_pad, uint32_t *__restrict__ segcount) {
    const int c = (blockIdx.y * blockDim.x + threadIdx.x) * VEC;
    const int r = blockIdx.z * blockDim.y + threadIdx.y;
    if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.y == 0) {  // padding between / after the planes
        const int64_t nwords = (int64_t)U0 * U1 * W;
        for (int64_t i = nwords + threadIdx.x; i < nwords_pad; i += blockDim.x) {
            bmp_pos[i] = 0u;
            bmp_neg[i] = 0u;
        }
    }
    if (c >= U0 || r >= U1) return;
    const int w_begin = blockIdx.x * kWordsPerThread;
    const int64_t plane = (int64_t)NR * NC;
    const float *col = rho + (int64_t)r * NC + c;
    uint32_t accp[VEC][kWordsPerThread], accn[VEC][kWordsPerThread];
#pragma unroll
    for (int q = 0; q < kWordsPerThread; ++q) {
        const int w = w_begin + q;
        uint32_t pos[VEC], neg[VEC];
#pragma unroll
        for (int i = 0; i < VEC; ++i) pos[i] = neg[i] = 0u;
        const int s0 = w * 32;
        const int nbits = min(32, U2 - s0);  // <= 0 in the padding words
        const float *p = col + (int64_t)s0 * plane;
        if (nbits == 32) {
            if (VEC == 4) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {  // two batches of 16 independent 16-byte loads
                    float4 v[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        v[j] = __ldg(reinterpret_cast<const float4 *>(p + (int64_t)(h * 16 + j) * plane));
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float e[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            pos[i] |= (e[i] >= cpos) ? (1u << (h * 16 + j)) : 0u;
                            neg[i] |= (e[i] <= cneg) ? (1u << (h * 16 + j)) : 0u;
                        }
                    }
                }
            } else {
                float v[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = __ldg(p + (int64_t)j * plane);
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    pos[0] |= (v[j] >= cpos) ? (1u << j) : 0u;
                    neg[0] |= (v[j] <= cneg) ? (1u << j) : 0u;
                }
            }
        } else {
            for (int j = 0; j < nbits; ++j) {
#pragma unroll
                for (int i = 0; i < VEC; ++i) {
                    const float e = (i == 0 || c + i < NC) ? __ldg(p + (int64_t)j * plane + i) : 0.f;
                    pos[i] |= (e >= cpos) ? (1u << j) : 0u;
                    neg[i] |= (e <= cneg) ? (1u << j) : 0u;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            accp[i][q] = use_pos ? pos[i] : 0u;
            accn[i][q] = use_neg ? neg[i] : 0u;
        }
    }
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
        if (c + i < U0) {
            const int64_t widx = ((int64_t)(c + i) * U1 + r) * W + w_begin;  // multiple of 4 words: 16-byte aligned
            *reinterpret_cast<uint4 *>(bmp_pos + widx) = make_uint4(accp[i][0], accp[i][1], accp[i][2], accp[i][3]);
            *reinterpret_cast<uint4 *>(bmp_neg + widx) = make_uint4(accn[i][0], accn[i][1], accn[i][2], accn[i][3]);
            // foreground per segment of the concatenated planes (four aligned words never straddle a segment);
            // at +/-3 sigma one store in twenty carries a voxel, so these atomics are rare
            const int np = __popc(accp[i][0]) + __popc(accp[i][1]) + __popc(accp[i][2]) + __popc(accp[i][3]);
            const int nn = __popc(accn[i][0]) + __popc(accn[i][1]) + __popc(accn[i][2]) + __popc(accn[i][3]);
            if (np) atomicAdd(segcount + (widx >> kSegShift), (uint32_t)np);
            if (nn) atomicAdd(segcount + ((nwords_pad + widx) >> kSegShift), (uint32_t)nn);
        }
    }
}

// ------------------------------------------------------------------------------------------------ sparse stage
// Everything after the streaming kernel touches only the bit planes and the sparse foreground, for BOTH signs at
// once: the planes are scanned as one concatenated word array, so green voxels occupy positions [0, n0) and red
// voxels [n0, n0 + n1) of one index space, and one union-find / one root ranking serves both.  ONE cooperative kernel
// (grid = resident blocks), four phases separated by three grid-wide barriers:
//   P1  list positions from the segment counts of K1 (every block sums the few thousand counts itself: no barrier),
//       then keys and initial parents of every foreground voxel -- a voxel points at the first voxel of
//       its run of consecutive sections;
//   P2  density gather and union-find hooking of the 12 predecessor neighbours outside the voxel's own column (all bit-plane and
//       position loads of a voxel are issued together, then hooked with lock-free atomicMin, "smaller id wins", the
//       voxel's current root carried from one hook to the next); the per-blob sums are zeroed on the side;
//   P3  flatten; root flags (one ballot word per 32 voxels) with the root count before each word inside its 512-voxel
//       chunk, and the root count of each chunk;
//   P4  every block scans the chunk counts into shared memory, so that the rank of any root -- the reference's blob
//       number, because a root is its blob's first voxel in scan order -- is two loads and a popcount; labels and
//       per-blob sums (DensityBlob.fromCrsList, pdb_eda/ccp4.py:534-545) with a segmented warp reduction in front of
//       the float64 atomics.
// Barriers were 35 % of the stall samples of the seven-barrier version (profiles/r01_final_c2_step.md).
// Phase boundaries of the last launch (globaltimer ns, written by block 0): pe_blob_stage_times().
__device__ unsigned long long g_stage_ns[12];
__device__ __forceinline__ void stamp(int i) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        g_stage_ns[i] = t;
    }
}

struct SparseArgs {
    const float *rho;
    int NC, NR, U1, U2, W;
    int64_t nwords_pad, cap, cap_blobs;
    int nseg;
    int p1_blocks;             // blocks that take part in P1 (the others go straight to the first barrier)
    int p1_per_sm;             // ... = this many per SM
    int *sm_rank;              // [256] blocks seen per SM, [255] scanning blocks so far (zeroed per launch)
    const uint32_t *bmp;       // two planes, nwords_pad apart
    const uint32_t *segcount;  // foreground voxels per segment (K1)
    uint32_t *base;            // per non-empty word: position of its first set bit in the concatenated voxel list
    uint32_t *parent;          // 2 * cap
    uint2 *flags;              // per 32 voxels: (root flags, roots before this word inside its chunk)
    uint32_t *coarse;          // per chunk: roots; [nchunk_cap ...): exclusive prefix when it does not fit shared memory
    int64_t nchunk_cap;
    int64_t *counts;           // n_fg0, n_blobs0, n_fg1, n_blobs1, overflow
    uint32_t *key;             // outputs, class k at k * cap
    float *value;
    int32_t *label;
    double *stats;             // class k at k * cap_blobs * 8
};

__device__ __forceinline__ uint32_t block_sum_u32(uint32_t v, uint32_t *smem /* >= 32 */) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    v = (uint32_t)warp_sum((int)v);
    __syncthreads();
    if (lane == 0) smem[w] = v;
    __syncthreads();
    uint32_t t = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += smem[i];
    return t;
}

// union that returns the root of the merged set (the smaller of the two roots), starting from a known ancestor
__device__ __forceinline__ uint32_t uf_union_root(uint32_t *parent, uint32_t a, uint32_t b) {
    for (;;) {
        a = uf_find_halve(parent, a);
        b = uf_find_halve(parent, b);
        if (a == b) return a;
        if (a < b) {
            const uint32_t t = a;
            a = b;
            b = t;
        }
        const uint32_t old = atomicMin(parent + a, b);  // hook the larger root under the smaller
        if (old == a) return b;
        a = old;
    }
}

// number of roots with a list position below x (x < n): the rank of x when x is a root
__device__ __forceinline__ uint32_t roots_below(const uint2 *__restrict__ flags, const uint32_t *cpre, uint32_t x) {
    const uint2 f = __ldcg(flags + (x >> 5));
    return cpre[x >> kChunkShift] + f.y + (uint32_t)__popc(f.x & ((1u << (x & 31u)) - 1u));
}

__global__ void __launch_bounds__(kSparseThreads, 3) blob_sparse_kernel(const __grid_constant__ pe_geom g, const SparseArgs a) {
    cg::grid_group grid = cg::this_grid();
    __shared__ uint32_t smem[32];
    __shared__ uint32_t pool[kPoolWords];  // P1: the warps' word queues; P4: the chunk prefix table
    uint32_t *cpre_s = pool;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nb = gridDim.x, b = blockIdx.x;
    const int warps_per_block = kSparseThreads >> 5;
    stamp(0);

    // ---- P1: positions, keys, densities, initial parents
    // contiguous run of segments per warp; the voxels before it are the segment counts before it.  Only the first p1_blocks blocks
    // scan (two per SM: with a third one the same words take longer -- three copies of the count prefix per SM and 48 warps on the
    // ballots and shuffles of the scan, profiles/r01_blob_sizes.md); the others wait at the barrier and read the totals after it.
    uint32_t n0 = 0, n_all = 0;
    // which blocks scan: the first p1_per_sm to arrive on each SM (block indices say nothing about placement); they number
    // themselves densely in arrival order
    __shared__ int scan_index;
    if (threadIdx.x == 0) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        int idx = -1;
        if (a.p1_blocks >= nb) idx = b;  // every block scans
        else if (atomicAdd(a.sm_rank + (smid < 254u ? smid : 254u), 1) < a.p1_per_sm) idx = atomicAdd(a.sm_rank + 255, 1);
        scan_index = idx;
    }
    __syncthreads();
    const int bi = scan_index;
    if (bi >= 0 && bi < a.p1_blocks) {
        const int nwarps = a.p1_blocks * warps_per_block;
        const int spw = (a.nseg + nwarps - 1) / nwarps;  // segments per warp
        const int seg_class1 = (int)(a.nwords_pad >> kSegShift);
        const int sb = min(bi * warps_per_block * spw, a.nseg);  // first segment of this block
        {
            // this warp's words are requested into L2 now (K1 streamed the whole map through L2 after writing them), so the
            // loads below, behind the prefix computation, find them there
            const int seg_begin = min(sb + warp * spw, a.nseg), seg_end = min(seg_begin + spw, a.nseg);
            for (int64_t i = ((int64_t)seg_begin << kSegShift) + 32 * lane; i < ((int64_t)seg_end << kSegShift); i += 32 * 32)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(a.bmp + i));
        }
        uint32_t before;
        {
            uint32_t s_before = 0, s0 = 0, s_all = 0;
            constexpr int kBatch = 8;  // independent loads in flight per thread (one L2 round trip per batch, not per count)
            for (int i0 = threadIdx.x; i0 < a.nseg; i0 += kSparseThreads * kBatch) {
                uint32_t v[kBatch];
#pragma unroll
                for (int j = 0; j < kBatch; ++j) {
                    const int i = i0 + j * kSparseThreads;
                    v[j] = i < a.nseg ? __ldg(a.segcount + i) : 0u;
                }
#pragma unroll
                for (int j = 0; j < kBatch; ++j) {
                    const int i = i0 + j * kSparseThreads;
                    s_all += v[j];
                    if (i < sb) s_before += v[j];
                    if (i < seg_class1) s0 += v[j];
                }
            }
            before = block_sum_u32(s_before, smem);
            n0 = block_sum_u32(s0, smem);
            n_all = block_sum_u32(s_all, smem);
        }
        const bool overflow = (int64_t)n0 > a.cap || (int64_t)(n_all - n0) > a.cap;  // the same in every scanning block
        if (bi == 0 && threadIdx.x == 0) {
            a.counts[0] = (int64_t)n0;
            a.counts[2] = (int64_t)(n_all - n0);
            if (overflow) a.counts[4] = 1;
        }
        if (!overflow) {
            const int seg_begin = min(sb + warp * spw, a.nseg), seg_end = min(seg_begin + spw, a.nseg);
            uint32_t mine = 0;
            for (int i = sb + lane; i < seg_begin; i += 32) mine += a.segcount[i];
            uint32_t run = before + (uint32_t)warp_sum((int)mine);
            uint32_t carry = 0u;  // the word before the current one
            if (seg_begin < seg_end && seg_begin > 0) carry = a.bmp[((int64_t)seg_begin << kSegShift) - 1];
            const int64_t w_end = (int64_t)seg_end << kSegShift;
            uint32_t *queue = pool + warp * (3 * kQueueCap);
            int qn = 0;
            uint4 next = make_uint4(0u, 0u, 0u, 0u);
            if (seg_begin < seg_end) next = __ldcg(reinterpret_cast<const uint4 *>(a.bmp + ((int64_t)seg_begin << kSegShift) + 4 * lane));
            for (int64_t i0 = (int64_t)seg_begin << kSegShift; i0 < w_end; i0 += 128) {
                const int64_t widx0 = i0 + 4 * lane;
                const uint4 wv = next;
                if (i0 + 128 < w_end) next = __ldcg(reinterpret_cast<const uint4 *>(a.bmp + widx0 + 128));  // in flight during this iteration
                const int c4 = __popc(wv.x) + __popc(wv.y) + __popc(wv.z) + __popc(wv.w);
                const int excl = warp_excl_scan(c4, lane);
                uint32_t p = run + (uint32_t)excl;
                run += (uint32_t)__shfl_sync(kFull, excl + c4, 31);
                uint32_t prevw = __shfl_up_sync(kFull, wv.w, 1);
                if (lane == 0) prevw = carry;
                carry = __shfl_sync(kFull, wv.w, 31);
                // non-empty words go to the warp's queue: (word index, position of the word's first voxel | "the word before
                // ends in a set bit" << 31, bits)
                const uint32_t words[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const uint32_t word = words[q];
                    const unsigned act = __ballot_sync(kFull, word != 0u);
                    if (word) {
                        const int slot = qn + __popc(act & ((1u << lane) - 1u));
                        const uint32_t pw = q == 0 ? prevw : words[q > 0 ? q - 1 : 0];
                        queue[slot] = (uint32_t)(widx0 + q);
                        queue[kQueueCap + slot] = p | (pw & 0x80000000u);
                        queue[2 * kQueueCap + slot] = word;
                        p += (uint32_t)__popc(word);
                    }
                    qn += __popc(act);
                }
                const bool last = i0 + 128 >= w_end;
                if (qn <= kQueueCap - 128 && !last) continue;  // room for another 128 words
                // ---- drain: one lane per non-empty word (at +/-3 sigma one word in twenty: draining them as they come would
                // leave two lanes of the warp busy)
                __syncwarp();
                for (int e = lane; e < qn; e += 32) {
                    const uint32_t widx = queue[e], pp = queue[kQueueCap + e], word = queue[2 * kQueueCap + e];
                    const uint32_t p_first = pp & 0x7fffffffu;
                    const int k = (int64_t)widx >= a.nwords_pad ? 1 : 0;
                    const uint32_t local = widx - (k ? (uint32_t)a.nwords_pad : 0u);
                    const uint32_t colrow = local / (uint32_t)a.W;
                    const int w = (int)(local - colrow * (uint32_t)a.W);
                    const int64_t out0 = (int64_t)k * a.cap - (k ? (int64_t)n0 : 0);  // output index = out0 + position
                    const bool prev_last = (w > 0) && (pp >> 31);
                    a.base[widx] = p_first;
                    // bits that start a run of consecutive sections inside this word (a run entering from the previous word
                    // has no start bit here: its voxels point at the previous word's last voxel, one hop from that run's start)
                    const uint32_t starts = word & ~((word << 1) | (prev_last ? 1u : 0u));
                    const uint32_t keybase = colrow * (uint32_t)a.U2 + (uint32_t)w * 32u;
                    uint32_t rest = word, pv = p_first;
                    while (rest) {
                        const int bit = __ffs(rest) - 1;
                        rest &= rest - 1;
                        // parent = first voxel of the run (finds stay O(1) instead of O(run length))
                        const uint32_t below = starts & ((2u << bit) - 1u);
                        uint32_t par;
                        if (below) {
                            const int sbit = 31 - __clz(below);
                            par = p_first + (uint32_t)__popc(word & ((1u << sbit) - 1u));
                        } else {
                            par = p_first - 1;  // the run continues from the previous word (prev_last is set)
                        }
                        a.key[out0 + pv] = keybase + (uint32_t)bit;
                        a.parent[pv] = par;
                        ++pv;
                    }
                }
                qn = 0;
                __syncwarp();
            }
        }
    }  // scanning blocks
    grid.sync();
    stamp(1);
    if (!(bi >= 0 && bi < a.p1_blocks)) {  // the totals the first scanning block left before the barrier
        n0 = (uint32_t)__ldcg(a.counts + 0);
        n_all = n0 + (uint32_t)__ldcg(a.counts + 2);
    }
    if (a.p1_blocks < nb && __ldcg(a.sm_rank + 255) != a.p1_blocks) {
        // not every SM held its share of the scanning blocks (cannot happen while 3 blocks fill an SM; checked, not assumed):
        // part of the planes was never scanned -- fail loudly instead of returning a partial list
        if (b == 0 && threadIdx.x == 0) a.counts[4] = 2;
        return;
    }
    if (__ldcg(a.counts + 4) != 0) return;  // a class overflows its capacity: grid-uniform, nothing has been written
    const int64_t n = (int64_t)n_all;
    const uint32_t n1 = n_all - n0;

    // ---- P2: hook the 12 predecessor neighbours outside the voxel's own column; zero the per-blob sums
    const int64_t gstride = (int64_t)nb * kSparseThreads;
    const int64_t gtid = (int64_t)b * kSparseThreads + threadIdx.x;
    {
        const int64_t rows0 = min((int64_t)n0, a.cap_blobs) * 8, rows1 = min((int64_t)n1, a.cap_blobs) * 8;
        for (int64_t i = gtid; i < rows0; i += gstride) a.stats[i] = 0.0;
        for (int64_t i = gtid; i < rows1; i += gstride) a.stats[a.cap_blobs * 8 + i] = 0.0;
    }
    for (int64_t i = gtid; i < n; i += gstride) {
        const int k = i >= (int64_t)n0 ? 1 : 0;
        const int64_t oi = (int64_t)k * a.cap + (i - (k ? (int64_t)n0 : 0));
        const uint32_t kk = __ldcg(a.key + oi);
        const int s = (int)(kk % (uint32_t)a.U2);
        const uint32_t colrow = kk / (uint32_t)a.U2;
        const int r = (int)(colrow % (uint32_t)a.U1), c = (int)(colrow / (uint32_t)a.U1);
        const int w = s >> 5, bit = s & 31;
        const uint32_t *bmp = a.bmp + (k ? a.nwords_pad : 0);
        const uint32_t *base = a.base + (k ? a.nwords_pad : 0);
        // the density of the voxel: one independent gather per thread, in flight while the neighbours are looked up
        const float dens = __ldg(a.rho + ((int64_t)s * a.NR + r) * a.NC + c);
        // the four neighbour columns (c-1, r-1), (c-1, r), (c-1, r+1), (c, r-1): their words of this voxel's section
        // range, all loads in flight together
        int64_t nw[4];
        bool ok[4];
        ok[0] = c > 0 && r > 0;
        ok[1] = c > 0;
        ok[2] = c > 0 && r + 1 < a.U1;
        ok[3] = r > 0;
        nw[0] = ((int64_t)(c - 1) * a.U1 + r - 1) * a.W + w;
        nw[1] = nw[0] + a.W;
        nw[2] = nw[1] + a.W;
        nw[3] = ((int64_t)c * a.U1 + r - 1) * a.W + w;
        uint32_t B[4], Bm[4], Bp[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            B[j] = ok[j] ? __ldcg(bmp + nw[j]) : 0u;
            Bm[j] = (ok[j] && bit == 0 && w > 0) ? __ldcg(bmp + nw[j] - 1) : 0u;
            Bp[j] = (ok[j] && bit == 31 && w + 1 < a.W) ? __ldcg(bmp + nw[j] + 1) : 0u;
        }
        // adjacent voxels of a neighbour column: the one at the same section if set (its s-1 / s+1 neighbours are chained
        // to it already), else those at s-1 and s+1
        uint32_t sel[4];  // bit 0: same section, bit 1: s-1 in this word, bit 2: s+1 in this word, bit 3: s-1 in the word before, bit 4: s+1 in the word after
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            uint32_t m = 0;
            if ((B[j] >> bit) & 1u) {
                m = 1u;
            } else {
                if (bit > 0 && ((B[j] >> (bit - 1)) & 1u)) m |= 2u;
                if (bit < 31 && ((B[j] >> (bit + 1)) & 1u)) m |= 4u;
                if (Bm[j] >> 31) m |= 8u;
                if (Bp[j] & 1u) m |= 16u;
            }
            sel[j] = m;
        }
        // A neighbour at this voxel's own section is itself 26-adjacent to every other predecessor neighbour within one row
        // and one column of it, and each of those pairs is hooked by whichever of the two comes later in scan order -- so
        // hooking that one neighbour is enough (by induction over the scan order the components come out the same), and the
        // dependent find / atomicMin round trips of the others are saved.  Columns: 0 (c-1, r-1), 1 (c-1, r), 2 (c-1, r+1),
        // 3 (c, r-1); 0 and 2, and 2 and 3, are two rows apart.
        if (sel[1] & 1u) {
            sel[0] = sel[2] = sel[3] = 0u;
        } else if (sel[3] & 1u) {
            sel[0] = sel[1] = 0u;
        } else if (sel[0] & 1u) {
            sel[1] = sel[3] = 0u;
        } else if (sel[2] & 1u) {
            sel[1] = 0u;
        } else {
            // no neighbour at this section: the same argument per side (s-1: bits 1 and 3, s+1: bits 2 and 4) -- the
            // neighbours of one side in columns within one row of each other are adjacent to each other
#pragma unroll
            for (int side = 0; side < 2; ++side) {
                const uint32_t bits = side ? (4u | 16u) : (2u | 8u);
                if (sel[1] & bits) {
                    sel[0] &= ~bits;
                    sel[2] &= ~bits;
                    sel[3] &= ~bits;
                } else if (sel[3] & bits) {
                    sel[0] &= ~bits;
                }
            }
        }
        uint32_t bs[4], bsm[4], bsp[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t m = sel[j];
            bs[j] = (m & 7u) ? __ldcg(base + nw[j]) : 0u;
            bsm[j] = (m & 8u) ? __ldcg(base + nw[j] - 1) : 0u;
            bsp[j] = (m & 16u) ? __ldcg(base + nw[j] + 1) : 0u;
        }
        uint32_t nbr[8];
        int cnt = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t m = sel[j];
            if (m & 1u) nbr[cnt++] = bs[j] + (uint32_t)__popc(B[j] & ((1u << bit) - 1u));
            if (m & 2u) nbr[cnt++] = bs[j] + (uint32_t)__popc(B[j] & ((1u << (bit - 1)) - 1u));
            if (m & 8u) nbr[cnt++] = bsm[j] + (uint32_t)__popc(Bm[j] & 0x7fffffffu);
            if (m & 4u) nbr[cnt++] = bs[j] + (uint32_t)__popc(B[j] & ((1u << (bit + 1)) - 1u));
            if (m & 16u) nbr[cnt++] = bsp[j];
        }
        // one union site for all lanes; the voxel's root is carried from one hook to the next
        uint32_t cur = (uint32_t)i;
#pragma unroll 1
        for (int j = 0; j < cnt; ++j) cur = uf_union_root(a.parent, cur, nbr[j]);
        a.value[oi] = dens;
    }
    grid.sync();
    stamp(2);

    // ---- P3: flatten; root flags per 32 voxels, roots before each word inside its chunk, roots per chunk
    const int64_t nchunks = (n + kSparseThreads - 1) >> kChunkShift;
    __shared__ uint32_t wcnt[32];
    for (int64_t chunk = b; chunk < nchunks; chunk += nb) {
        const int64_t i = (chunk << kChunkShift) + threadIdx.x;
        bool isroot = false;
        if (i < n) {
            const uint32_t root = uf_find(a.parent, (uint32_t)i);
            a.parent[i] = root;  // still a valid ancestor for concurrent finds
            isroot = root == (uint32_t)i;
        }
        const uint32_t fw = __ballot_sync(kFull, isroot);
        if (lane == 0) wcnt[warp] = (uint32_t)__popc(fw);
        __syncthreads();
        uint32_t fine = 0, tot = 0;
        for (int j = 0; j < warps_per_block; ++j) {
            const uint32_t v = wcnt[j];
            if (j < warp) fine += v;
            tot += v;
        }
        if (lane == 0) a.flags[(chunk << (kChunkShift - 5)) + warp] = make_uint2(fw, fine);
        if (threadIdx.x == 0) a.coarse[chunk] = tot;
        __syncthreads();  // wcnt is rewritten by the next chunk
    }
    grid.sync();
    stamp(3);

    // ---- P4: chunk prefix (per block, in shared memory), blob counts, labels + sums
    const uint32_t *cpre = cpre_s;
    uint32_t n_roots;
    if (nchunks <= kChunkSmem) {
        // every thread scans kChunkSmem / kSparseThreads consecutive chunk counts, then a block scan of the partials
        constexpr int kPer = kChunkSmem / kSparseThreads;
        uint32_t v[kPer], sum = 0;
#pragma unroll
        for (int j = 0; j < kPer; ++j) {
            const int64_t ci = (int64_t)threadIdx.x * kPer + j;
            v[j] = ci < nchunks ? __ldcg(a.coarse + ci) : 0u;
            sum += v[j];
        }
        const uint32_t wex = (uint32_t)warp_excl_scan((int)sum, lane);
        __syncthreads();
        if (lane == 31) wcnt[warp] = wex + sum;
        __syncthreads();
        uint32_t off = wex;
        uint32_t all = 0;
        for (int j = 0; j < warps_per_block; ++j) {
            const uint32_t t = wcnt[j];
            if (j < warp) off += t;
            all += t;
        }
#pragma unroll
        for (int j = 0; j < kPer; ++j) {
            cpre_s[threadIdx.x * kPer + j] = off;
            off += v[j];
        }
        n_roots = all;
        __syncthreads();
    } else {
        // very large foreground: block 0 scans the chunk counts into global memory, one more barrier
        uint32_t *gpre = a.coarse + a.nchunk_cap;
        if (b == 0) {
            __shared__ uint32_t carry_s;
            if (threadIdx.x == 0) carry_s = 0u;
            __syncthreads();
            for (int64_t c0 = 0; c0 < nchunks; c0 += kSparseThreads) {
                const int64_t ci = c0 + threadIdx.x;
                const uint32_t v = ci < nchunks ? __ldcg(a.coarse + ci) : 0u;
                const uint32_t wex = (uint32_t)warp_excl_scan((int)v, lane);
                if (lane == 31) wcnt[warp] = wex + v;
                __syncthreads();
                uint32_t off = carry_s + wex, all = 0;
                for (int j = 0; j < warps_per_block; ++j) {
                    const uint32_t t = wcnt[j];
                    if (j < warp) off += t;
                    all += t;
                }
                if (ci < nchunks) gpre[ci] = off;
                __syncthreads();
                if (threadIdx.x == 0) carry_s += all;
                __syncthreads();
            }
            if (threadIdx.x == 0) gpre[nchunks] = carry_s;
        }
        grid.sync();
        cpre = gpre;
        n_roots = __ldcg(gpre + nchunks);
    }
    const uint32_t nb0 = n0 == n_all ? n_roots : roots_below(a.flags, cpre, n0);  // roots among the class-0 voxels
    const uint32_t nb1 = n_roots - nb0;
    if (b == 0 && threadIdx.x == 0) {
        a.counts[1] = (int64_t)nb0;
        a.counts[3] = (int64_t)nb1;
    }
    if ((int64_t)nb0 > a.cap_blobs || (int64_t)nb1 > a.cap_blobs) {  // grid-uniform
        if (b == 0 && threadIdx.x == 0) a.counts[4] = 1;
        return;
    }
    for (int64_t i0 = gtid - lane; i0 < n; i0 += gstride) {  // warp-uniform trip count
        const int64_t i = i0 + lane;
        const bool live = i < n;
        int32_t blob = -1;
        double v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (live) {
            const int k = i >= (int64_t)n0 ? 1 : 0;
            const int64_t oi = (int64_t)k * a.cap + (i - (k ? (int64_t)n0 : 0));
            const uint32_t gr = roots_below(a.flags, cpre, __ldcg(a.parent + i));
            blob = (int32_t)(gr - (k ? nb0 : 0u));
            a.label[oi] = blob;
            blob += k ? (int32_t)a.cap_blobs : 0;  // row of the combined stats table
            const uint32_t kk = __ldcg(a.key + oi);
            const int s = (int)(kk % (uint32_t)a.U2);
            const uint32_t colrow = kk / (uint32_t)a.U2;
            const int r = (int)(colrow % (uint32_t)a.U1), c = (int)(colrow / (uint32_t)a.U1);
            double x, y, z;
            crs2xyz(g, c, r, s, x, y, z);
            const double d = (double)__ldcg(a.value + oi);
            v[0] = 1.0;
            v[1] = d;
            v[2] = __dmul_rn(d, x);
            v[3] = __dmul_rn(d, y);
            v[4] = __dmul_rn(d, z);
            v[5] = x;
            v[6] = y;
            v[7] = z;
        }
        // segmented reduction over runs of equal blob id (runs along the section axis are the common case)
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
        if (live && head) {
            double *st = a.stats + (int64_t)blob * 8;
#pragma unroll
            for (int q = 0; q < 8; ++q) atomicAdd(st + q, v[q]);
        }
    }
    stamp(4);
}

}  // namespace pe

using namespace pe;

extern "C" {

int pe_blob_stage_times(unsigned long long *out12) {
    PE_CHECK_ARG(out12 != nullptr, "pe_blob_stage_times: null pointer");
    PE_CUDA(cudaMemcpyFromSymbol(out12, g_stage_ns, sizeof(unsigned long long) * 12));
    return PE_OK;
}

int64_t pe_blob_workspace_bytes(const pe_geom *g, int64_t cap_voxels) {
    if (!g || cap_voxels < 0) return -1;
    return make_plan(g, cap_voxels).total;
}

int pe_blob_label(const pe_geom *g, const float *d_rho, float cut_pos, float cut_neg, int64_t cap_voxels,
                  int64_t cap_blobs, int64_t *d_counts, uint32_t *d_key, float *d_value, int32_t *d_label,
                  double *d_stats, void *d_ws, void *stream) {
    if (int rc = check_geom(g)) return rc;
    PE_CHECK_ARG(d_rho && d_counts && d_key && d_value && d_label && d_stats && d_ws, "pe_blob_label: null pointer");
    PE_CHECK_ARG(cap_voxels > 0 && cap_blobs > 0, "pe_blob_label: capacities must be positive");
    PE_CHECK_ARG(cap_voxels < (1ll << 30), "pe_blob_label: cap_voxels must be below 2^30");
    PE_CHECK_ARG(!(cut_pos < 0.f) && !(cut_neg > 0.f), "pe_blob_label: cut_pos must be >= 0 and cut_neg <= 0");
    PE_CHECK_ARG(cut_pos == cut_pos && cut_neg == cut_neg, "pe_blob_label: NaN cutoff");
    const BlobPlan p = make_plan(g, cap_voxels);
    PE_CHECK_ARG((int64_t)p.U0 * p.U1 * p.U2 < (1ll << 32), "pe_blob_label: unique volume too large for 32-bit keys");
    PE_CHECK_ARG(p.nwords_pad < (1ll << 31), "pe_blob_label: bit planes too large");
    cudaStream_t st = (cudaStream_t)stream;
    char *ws = (char *)d_ws;
    const int NC = g->ncrs[0], NR = g->ncrs[1];
    uint32_t *bmp = (uint32_t *)(ws + p.off_bmp);
    const bool use_pos = cut_pos > 0.f, use_neg = cut_neg < 0.f;

    PE_CUDA(cudaMemsetAsync(d_counts, 0, 5 * sizeof(int64_t), st));
    uint32_t *segcount = (uint32_t *)(ws + p.off_seg);
    PE_CUDA(cudaMemsetAsync(segcount, 0, (size_t)align_up(p.nseg * 4, 256) + 1024, st));
    // K1: the only pass over the map
    {
        const bool vec4 = (NC % 4 == 0) && (((uintptr_t)d_rho & 15u) == 0);
        const int vec = vec4 ? 4 : 1;
        const int tx = kBmpTx, ty = kBmpTy;  // block shape makes no measurable difference (profiles/r01_threshold_tuning.md)
        dim3 block(tx, ty, 1);
        dim3 grid(p.W / kWordsPerThread, (p.U0 + tx * vec - 1) / (tx * vec), (p.U1 + ty - 1) / ty);
        PE_CHECK_ARG(grid.y <= 65535 && grid.z <= 65535, "pe_blob_label: map too large for the launch grid");
        if (vec4)
            PE_LAUNCH("threshold_bitmap_kernel", st, threshold_bitmap_kernel<4><<<grid, block, 0, st>>>(
                d_rho, NC, NR, p.U0, p.U1, p.U2, p.W, cut_pos, cut_neg, use_pos, use_neg, bmp, bmp + p.nwords_pad, p.nwords_pad, segcount));
        else
            PE_LAUNCH("threshold_bitmap_kernel", st, threshold_bitmap_kernel<1><<<grid, block, 0, st>>>(
                d_rho, NC, NR, p.U0, p.U1, p.U2, p.W, cut_pos, cut_neg, use_pos, use_neg, bmp, bmp + p.nwords_pad, p.nwords_pad, segcount));
        PE_LAUNCH_CHECK();
    }
    // sparse stage: one cooperative kernel for both signs
    SparseArgs a;
    a.rho = d_rho;
    a.NC = NC;
    a.NR = NR;
    a.U1 = p.U1;
    a.U2 = p.U2;
    a.W = p.W;
    a.nwords_pad = p.nwords_pad;
    a.cap = p.cap;
    a.cap_blobs = cap_blobs;
    a.nseg = (int)p.nseg;
    a.bmp = bmp;
    a.segcount = segcount;
    a.base = (uint32_t *)(ws + p.off_base);
    a.parent = (uint32_t *)(ws + p.off_parent);
    a.flags = (uint2 *)(ws + p.off_flags);
    a.coarse = (uint32_t *)(ws + p.off_coarse);
    a.nchunk_cap = p.nchunk_cap;
    a.counts = d_counts;
    a.key = d_key;
    a.value = d_value;
    a.label = d_label;
    a.stats = d_stats;
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        PE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, blob_sparse_kernel, kSparseThreads, 0));
        PE_CHECK_ARG(blocks_per_sm > 0, "pe_blob_label: the sparse kernel does not fit an SM");
    }
    // the SMs of the launching stream: on an SM partition the grid fills exactly the partition's SMs (a larger cooperative grid is
    // a launch error, never a wait), so that "3 blocks on every SM" below still holds there
    const int sms = stream_sm_count(st);
    const int nblocks = sms * (blocks_per_sm < 3 ? blocks_per_sm : 3);
    // P1 runs on two blocks per SM (384^3: 13.7 us against 16.7 us with all three scanning; 768^3 / 1024^3: no difference)
    // -- only when exactly 3 blocks fill an SM, so that every SM is known to hold 3 of the grid's blocks; otherwise every block scans
    a.p1_per_sm = blocks_per_sm == 3 ? kScanBlocksPerSm : (blocks_per_sm < 3 ? blocks_per_sm : 3);
    a.p1_blocks = sms * a.p1_per_sm;
    a.sm_rank = (int *)(ws + p.off_seg + align_up(p.nseg * 4, 256));
    pe_geom geom = *g;
    void *args[] = {(void *)&geom, (void *)&a};
    PE_LAUNCH("blob_sparse_kernel", st,
              PE_CUDA(cudaLaunchCooperativeKernel((const void *)blob_sparse_kernel, dim3(nblocks), dim3(kSparseThreads), args, 0, st)));
    PE_LAUNCH_CHECK();
    return PE_OK;
}

}  // extern "C"
