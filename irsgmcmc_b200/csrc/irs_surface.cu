// irs_surface.cu -- average surface distance per sample and structure, the LabelContour + average Hausdorff distance part of
// the reference's calc_metrics (utils/util.py:151-206, :171-176; host restatement: utils.util.calc_ASD_host):
//   box pass     bounding box of A u B and |A|, |B| for every (sample, label) in one pass over the volumes
//   three passes the exact separable Euclidean distance transform over every box (W, then H, then D), both directions at once:
//                channel 0 = squared distance to the contour of B, channel 1 = to the contour of A
//   reduction    the two directed means over the contour voxels, block partials summed in a fixed order (no float atomics);
//                for the Hausdorff distance it also appends every contour voxel's squared distance to a list per (pair, direction)
//   selection    (Hausdorff distance only) one CTA per list: maximum and the percentile's ranks by an MSB-first radix select
//                over the fp32 bit patterns (irs_select.cuh)
// Contour (ITK LabelContourImageFilter, FullyConnectedOff): a voxel of the set with one of its 6 face neighbours outside the set,
// where outside the volume counts as outside.  The box holds every voxel of A and B, so "outside the box" is "outside the set",
// and an exact transform over the box is exact for every contour voxel: no margin is needed.
#include <float.h>
#include <limits.h>

#include "irs_kernels.cuh"
#include "irs_edt.cuh"
#include "irs_select.cuh"

namespace {

constexpr int kBox = 8;   // per (sample, label): z0 y0 x0 z1 y1 x1 (inclusive), |A|, |B|

__global__ void surface_box_init_kernel(int* __restrict__ boxes, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) boxes[i] = (i % kBox) < 3 ? INT_MAX : ((i % kBox) < 6 ? -1 : 0);
}

__device__ __forceinline__ int label_index(const LabelList& l, int v) {
    if (v == 0) return -1;   // background is never a structure label
    for (int i = 0; i < l.n; ++i)
        if (l.v[i] == v) return i;
    return -1;
}

// the lanes of a warp holding the same label merge their voxels into one shared-memory update (integer min / max / add:
// order independent).  Called by all 32 lanes.
__device__ __forceinline__ void box_add(int* sh, int idx, int count_slot, int z, int y, int x) {
    const unsigned peers = __match_any_sync(0xffffffffu, idx);
    if (idx < 0) return;
    const int z0 = __reduce_min_sync(peers, z), z1 = __reduce_max_sync(peers, z);
    const int y0 = __reduce_min_sync(peers, y), y1 = __reduce_max_sync(peers, y);
    const int x0 = __reduce_min_sync(peers, x), x1 = __reduce_max_sync(peers, x);
    if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) {
        int* b = sh + idx * kBox;
        atomicMin(b + 0, z0); atomicMin(b + 1, y0); atomicMin(b + 2, x0);
        atomicMax(b + 3, z1); atomicMax(b + 4, y1); atomicMax(b + 5, x1);
        atomicAdd(b + count_slot, __popc(peers));
    }
}

__global__ void __launch_bounds__(256)
surface_box_kernel(const short* __restrict__ seg_a, long long a_cs, const short* __restrict__ seg_b, LabelList labels,
                   int* __restrict__ boxes, IrsDims d) {
    __shared__ int sh[32 * kBox];
    for (int i = threadIdx.x; i < 32 * kBox; i += blockDim.x) sh[i] = (i % kBox) < 3 ? INT_MAX : ((i % kBox) < 6 ? -1 : 0);
    __syncthreads();
    const int c = blockIdx.y, lane = threadIdx.x & 31;
    const long long V = d.V();
    const short* a = seg_a + (size_t)c * a_cs;
    const short* b = seg_b + (size_t)c * V;
    // warp-uniform trip count: every lane takes part in the warp-wide merges
    for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x - lane); base < V;
         base += (long long)gridDim.x * blockDim.x) {
        const long long i = base + lane;
        int ia = -1, ib = -1, x = 0, y = 0, z = 0;
        if (i < V) {
            ia = label_index(labels, a[i]);
            ib = label_index(labels, b[i]);
            const long long r = i / d.W;
            x = (int)(i - r * d.W); y = (int)(r % d.H); z = (int)(r / d.H);
        }
        if (!__any_sync(0xffffffffu, ia >= 0 || ib >= 0)) continue;
        box_add(sh, ia, 6, z, y, x);
        box_add(sh, ib, 7, z, y, x);
    }
    __syncthreads();
    int* g = boxes + (size_t)c * labels.n * kBox;
    for (int i = threadIdx.x; i < labels.n * kBox; i += blockDim.x) {
        const int l = i / kBox, k = i % kBox;
        if (sh[l * kBox + 6] == 0 && sh[l * kBox + 7] == 0) continue;
        if (k < 3) atomicMin(g + i, sh[i]);
        else if (k < 6) atomicMax(g + i, sh[i]);
        else if (sh[i]) atomicAdd(g + i, sh[i]);
    }
}

// ---- distance transform over the boxes of one launch group ----------------------------------------------------------------
struct AsdBox {
    long long off;            // first float of the box in the workspace: channel 0 then channel 1, each (nd, nh, nw)
    int c, label, pair;       // sample, label value, index into asd[]
    int z0, y0, x0, nd, nh, nw;
    int cap_a;                // Hausdorff lists after the two channels: |A| floats (contour of A), then |B| floats
};

struct AsdGroup {
    int n;
    long long line0[3][IRS_ASD_MAX_BOXES + 1];   // prefix of the lines per box: pass 0 (rows, both channels), 1 (H), 2 (D)
    AsdBox b[IRS_ASD_MAX_BOXES];
};

IRS_HD long long box_voxels(const AsdBox& B) { return (long long)B.nd * B.nh * B.nw; }

// blocks of the reduction of one box: a function of the box alone, so that the summation order (and the result, to the
// bit) does not depend on which other boxes share the launch
IRS_HD int reduce_blocks(long long nvox) {
    const long long g = (nvox + 2047) / 2048;
    return (int)(g < IRS_ASD_REDUCE_BLOCKS ? g : IRS_ASD_REDUCE_BLOCKS);
}

__device__ __forceinline__ int group_box(const AsdGroup& G, int pass, long long line) {
    int lo = 0, hi = G.n - 1;   // last box whose first line is <= line
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (G.line0[pass][mid] <= line) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

__device__ __forceinline__ bool in_set(const short* s, const AsdBox& B, IrsDims d, int z, int y, int x) {
    if (z < B.z0 || z >= B.z0 + B.nd || y < B.y0 || y >= B.y0 + B.nh || x < B.x0 || x >= B.x0 + B.nw) return false;
    return __ldg(s + ((long long)z * d.H + y) * d.W + x) == B.label;
}

__device__ __forceinline__ bool on_contour(const short* s, const AsdBox& B, IrsDims d, int z, int y, int x) {
    return in_set(s, B, d, z, y, x) &&
           !(in_set(s, B, d, z, y, x - 1) && in_set(s, B, d, z, y, x + 1) && in_set(s, B, d, z, y - 1, x) &&
             in_set(s, B, d, z, y + 1, x) && in_set(s, B, d, z - 1, y, x) && in_set(s, B, d, z + 1, y, x));
}

// pass 0: one thread per box row (z, y): contour flags of both sets, then the two-sweep 1-D distance along W
__global__ void __launch_bounds__(128)
edt_rows_kernel(const short* __restrict__ seg_a, long long a_cs, const short* __restrict__ seg_b, IrsDims d,
                const __grid_constant__ AsdGroup G, float* __restrict__ ws, float w) {
    const long long line = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (line >= G.line0[0][G.n]) return;
    const int bi = group_box(G, 0, line);
    const AsdBox& B = G.b[bi];
    const int j = (int)(line - G.line0[0][bi]);
    const int zz = j / B.nh, yy = j - zz * B.nh;
    float* r0 = ws + B.off + ((long long)zz * B.nh + yy) * B.nw;   // sites: contour of B
    float* r1 = r0 + box_voxels(B);                                 // sites: contour of A
    const short* a = seg_a + (size_t)B.c * a_cs;
    const short* b = seg_b + (size_t)B.c * d.V();
    const int z = B.z0 + zz, y = B.y0 + yy;
    for (int x = 0; x < B.nw; ++x) {
        r0[x] = on_contour(b, B, d, z, y, B.x0 + x) ? 0.0f : INFINITY;
        r1[x] = on_contour(a, B, d, z, y, B.x0 + x) ? 0.0f : INFINITY;
    }
    irs_edt_sites_1d(r0, 1, B.nw, w);
    irs_edt_sites_1d(r1, 1, B.nw, w);
}

// passes 1 (AXIS = 1, lines along H) and 2 (AXIS = 2, lines along D): one thread per line and channel, lower envelope of
// parabolas with its scratch in shared memory (3 * n_max words per thread, interleaved by thread)
template <int AXIS>
__global__ void __launch_bounds__(128)
edt_envelope_kernel(float* __restrict__ ws, const __grid_constant__ AsdGroup G, float w, int n_max) {
    extern __shared__ float smem[];
    const int T = blockDim.x, t = threadIdx.x;
    const long long line = (long long)blockIdx.x * T + t;
    if (line >= G.line0[AXIS][G.n]) return;
    const int bi = group_box(G, AXIS, line);
    const AsdBox& B = G.b[bi];
    const long long j = line - G.line0[AXIS][bi];
    const long long plane = (long long)B.nh * B.nw;
    long long base;
    long long ds;
    int n;
    if (AXIS == 1) {
        const long long per = (long long)B.nd * B.nw, r = j % per, zz = r / B.nw;
        base = B.off + (j / per) * box_voxels(B) + zz * plane + (r - zz * B.nw);
        ds = B.nw;
        n = B.nh;
    } else {
        base = B.off + (j / plane) * box_voxels(B) + j % plane;
        ds = plane;
        n = B.nd;
    }
    int* v = reinterpret_cast<int*>(smem) + t;
    irs_edt_envelope_1d(ws + base, ds, n, w, v, smem + (size_t)T * n_max + t, smem + (size_t)2 * T * n_max + t, T);
}

// ASD = (mean over the contour of A of the distance to the contour of B + the same from B to A) / 2.  A voxel is on the
// contour of B exactly when its channel-0 distance is 0 (spacings are positive), and likewise for A: the flags need no
// second look at the volumes.  Per box: reduce_blocks() blocks, each a fixed-order partial; the last to arrive adds them up.
// LISTS (Hausdorff distance): every contour voxel of A also appends its squared distance to the contour of B to the box's list
// AB, and the same from B to A; the slots come from one integer atomicAdd per warp, so the list order varies from run to run
// while the sums (each thread's sequence of voxels is the same in both variants) and every order statistic do not.
__device__ __forceinline__ void list_append(bool on, float key, float* list, unsigned int* count, int lane) {
    const unsigned m = __ballot_sync(0xffffffffu, on);
    if (m == 0u) return;
    const int leader = __ffs(m) - 1;
    unsigned base = 0u;
    if (lane == leader) base = atomicAdd(count, (unsigned)__popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (on) list[base + __popc(m & ((1u << lane) - 1u))] = key;
}

template <bool LISTS>
__global__ void __launch_bounds__(256)
asd_reduce_kernel(float* __restrict__ ws, const __grid_constant__ AsdGroup G, double* __restrict__ partials,
                  unsigned int* __restrict__ counters, double* __restrict__ asd, double* __restrict__ hd,
                  double* __restrict__ hd_q) {
    __shared__ double sh[4 * 8];
    __shared__ bool last;
    const AsdBox& B = G.b[blockIdx.y];
    const long long nvox = box_voxels(B);
    const int nb = reduce_blocks(nvox);
    if ((int)blockIdx.x >= nb) return;
    const float* d0 = ws + B.off;
    const float* d1 = d0 + nvox;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double v[4] = {0.0, 0.0, 0.0, 0.0};   // sum over cA of d(., cB), |cA|, sum over cB of d(., cA), |cB|
    if (LISTS) {
        float* list_ab = ws + B.off + 2 * nvox;
        float* list_ba = list_ab + B.cap_a;
        unsigned int* n_ab = counters + IRS_ASD_MAX_BOXES + blockIdx.y;
        unsigned int* n_ba = n_ab + IRS_ASD_MAX_BOXES;
        // warp-uniform trip count for the warp-wide slot allocation; each thread visits the voxels of the loop below
        for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x - lane); base < nvox;
             base += (long long)nb * blockDim.x) {
            const long long i = base + lane;
            float a = 1.0f, b = 1.0f;
            if (i < nvox) { a = d0[i]; b = d1[i]; }
            if (b == 0.0f) { v[0] += sqrt((double)a); v[1] += 1.0; }
            if (a == 0.0f) { v[2] += sqrt((double)b); v[3] += 1.0; }
            list_append(b == 0.0f, a, list_ab, n_ab, lane);
            list_append(a == 0.0f, b, list_ba, n_ba, lane);
        }
    } else {
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvox; i += (long long)nb * blockDim.x) {
            const float a = d0[i], b = d1[i];
            if (b == 0.0f) { v[0] += sqrt((double)a); v[1] += 1.0; }
            if (a == 0.0f) { v[2] += sqrt((double)b); v[3] += 1.0; }
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const double s = irs_warp_sum(v[k]);
        if (lane == 0) sh[k * 8 + warp] = s;
    }
    __syncthreads();
    double* p = partials + (size_t)blockIdx.y * 4 * IRS_ASD_REDUCE_BLOCKS;
    if (threadIdx.x == 0) {
        for (int k = 0; k < 4; ++k) {
            double s = 0.0;
            for (int w8 = 0; w8 < (int)(blockDim.x >> 5); ++w8) s += sh[k * 8 + w8];
            p[k * IRS_ASD_REDUCE_BLOCKS + blockIdx.x] = s;
        }
        __threadfence();
        last = atomicAdd(counters + blockIdx.y, 1u) == (unsigned)(nb - 1);
    }
    __syncthreads();
    if (!last || threadIdx.x != 0) return;
    __threadfence();
    double tot[4];
    for (int k = 0; k < 4; ++k) {
        double s = 0.0;
        for (int g = 0; g < nb; ++g) s += __ldcg(p + k * IRS_ASD_REDUCE_BLOCKS + g);
        tot[k] = s;
    }
    asd[B.pair] = 0.5 * (tot[0] / tot[1] + tot[2] / tot[3]);
    if (LISTS) hd[B.pair] = hd_q[B.pair] = 0.0;   // the selection raises them with integer maxima
    counters[blockIdx.y] = 0u;
}

// Hausdorff distance: one CTA per (box, direction) list of n squared distances (blockIdx.x = 0: contour of A to B, 1: B to A).
// Four MSB-first passes of IRS_SELECT_BITS bits find the key at rank i of the percentile (shared-memory histograms, lanes with
// the same digit merged into one integer atomicAdd); rank i + 1 is that key again when more than i + 1 keys are <= it, else the
// smallest key above it (one more pass, a block minimum).  The first pass also takes the list's maximum.  The two directions
// meet in integer atomicMax on the fp64 bit patterns of the non-negative results: HD = max of the maxima, HD_q = max of the
// directed percentiles, independent of which CTA comes first.  The list's count is reset for the next launch group.
constexpr int kSelectThreads = 512;

__global__ void __launch_bounds__(kSelectThreads)
hd_select_kernel(const float* __restrict__ ws, const __grid_constant__ AsdGroup G, unsigned int* __restrict__ counters,
                 double q, double* __restrict__ hd, double* __restrict__ hd_q) {
    __shared__ unsigned int hist[IRS_SELECT_BINS];
    __shared__ unsigned int sh_bin, sh_r, sh_eq, sh_max, sh_min;
    const AsdBox& B = G.b[blockIdx.y];
    const int dir = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const long long nvox = box_voxels(B);
    const unsigned int* keys = reinterpret_cast<const unsigned int*>(ws + B.off + 2 * nvox + (dir ? B.cap_a : 0));
    unsigned int* count = counters + IRS_ASD_MAX_BOXES * (1 + dir) + blockIdx.y;
    const unsigned int n = __ldcg(count);
    if (n == 0u) return;   // not reached: a non-empty set has a contour
    const IrsPercentileRank pr = irs_percentile_rank(n, q);
    if (t == 0) { sh_max = 0u; sh_min = 0xffffffffu; }
    unsigned int prefix = 0u, mask = 0u, r = pr.i, mx = 0u;
    for (int shift = 32 - IRS_SELECT_BITS; shift >= 0; shift -= IRS_SELECT_BITS) {
        for (int k = t; k < IRS_SELECT_BINS; k += kSelectThreads) hist[k] = 0u;
        __syncthreads();
        for (unsigned int base = t - lane; base < n; base += kSelectThreads) {   // warp-uniform: lanes merge below
            const unsigned int k = base + lane;
            int bin = -1;
            if (k < n) {
                const unsigned int v = __ldcg(keys + k);
                if (shift == 32 - IRS_SELECT_BITS) mx = max(mx, v);
                if ((v & mask) == prefix) bin = (int)((v >> shift) & (IRS_SELECT_BINS - 1));
            }
            const unsigned peers = __match_any_sync(0xffffffffu, bin);
            if (bin >= 0 && lane == __ffs(peers) - 1) atomicAdd(hist + bin, (unsigned)__popc(peers));
        }
        __syncthreads();
        if (warp == 0) {   // lane l owns bins [8 l, 8 l + 8): the lane where the cumulative count passes r walks its bins
            constexpr int per = IRS_SELECT_BINS / 32;
            unsigned int s = 0u;
#pragma unroll
            for (int k = 0; k < per; ++k) s += hist[lane * per + k];
            unsigned int incl = s;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned int u = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += u;
            }
            const unsigned int excl = incl - s;
            if (excl <= r && r < incl) {
                unsigned int rr = r - excl;
                const int bin = lane * per + irs_select_bin(hist + lane * per, per, &rr);
                sh_bin = (unsigned)bin;
                sh_r = rr;
                sh_eq = hist[bin];
            }
        }
        __syncthreads();
        prefix |= sh_bin << shift;
        mask |= (unsigned int)(IRS_SELECT_BINS - 1) << shift;
        r = sh_r;
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    if (lane == 0) atomicMax(&sh_max, mx);
    const bool above = !pr.last && pr.i + 1 >= pr.i - r + sh_eq;   // keys <= rank i's key: (i - r) below it, sh_eq equal to it
    if (above) {
        unsigned int m = 0xffffffffu;
        for (unsigned int k = t; k < n; k += kSelectThreads) {
            const unsigned int v = __ldcg(keys + k);
            if (v > prefix) m = min(m, v);
        }
        m = __reduce_min_sync(0xffffffffu, m);
        if (lane == 0) atomicMin(&sh_min, m);
    }
    __syncthreads();
    if (t != 0) return;
    const unsigned int next = above ? sh_min : prefix;
    const double p = irs_percentile_value(__uint_as_float(prefix), __uint_as_float(next), pr);
    const double h = sqrt((double)__uint_as_float(sh_max));
    atomicMax(reinterpret_cast<unsigned long long*>(hd_q + B.pair), (unsigned long long)__double_as_longlong(p));
    atomicMax(reinterpret_cast<unsigned long long*>(hd + B.pair), (unsigned long long)__double_as_longlong(h));
    *count = 0u;
}

__global__ void fill_kernel(double* __restrict__ x, int n, double value) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] = value;
}

bool bad_spacing(float s) { return !(s > 0.0f) || !(s * s >= FLT_MIN) || !(s * s <= FLT_MAX); }

// the Hausdorff outputs of irs_surface_distances; hd == nullptr: the average surface distance alone
struct HdOut {
    double q;
    double* hd;
    double* hd_q;
};

int launch_group(const short* seg_a, long long a_cs, const short* seg_b, IrsDims d, const AsdGroup& G, const float* w,
                 float* ws, double* partials, unsigned int* counters, double* asd, const HdOut& hd, cudaStream_t st) {
    if (G.n == 0) return IRS_OK;
    const long long rows = G.line0[0][G.n];
    edt_rows_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, st>>>(seg_a, a_cs, seg_b, d, G, ws, w[0]);
    IRS_LAUNCH_CHECK();
    for (int pass = 1; pass <= 2; ++pass) {
        int n_max = 1;
        for (int k = 0; k < G.n; ++k) n_max = max(n_max, pass == 1 ? G.b[k].nh : G.b[k].nd);
        const size_t per_thread = (size_t)12 * n_max;
        int T = (int)((200u * 1024u) / per_thread);
        T = T >= 128 ? 128 : (T >= 32 ? T & ~31 : T);
        if (T < 1) return IRS_ERR_UNSUPPORTED;
        const size_t smem = (size_t)T * per_thread;
        const long long lines = G.line0[pass][G.n];
        const unsigned blocks = (unsigned)((lines + T - 1) / T);
        void (*kern)(float*, const AsdGroup, float, int) = pass == 1 ? edt_envelope_kernel<1> : edt_envelope_kernel<2>;
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return (int)e;
        }
        kern<<<blocks, T, smem, st>>>(ws, G, w[pass], n_max);
        IRS_LAUNCH_CHECK();
    }
    int nb = 1;
    for (int k = 0; k < G.n; ++k) nb = max(nb, reduce_blocks(box_voxels(G.b[k])));
    if (!hd.hd) {
        asd_reduce_kernel<false><<<dim3(nb, G.n), 256, 0, st>>>(ws, G, partials, counters, asd, nullptr, nullptr);
        IRS_LAUNCH_CHECK();
        return IRS_OK;
    }
    asd_reduce_kernel<true><<<dim3(nb, G.n), 256, 0, st>>>(ws, G, partials, counters, asd, hd.hd, hd.hd_q);
    IRS_LAUNCH_CHECK();
    hd_select_kernel<<<dim3(2, G.n), kSelectThreads, 0, st>>>(ws, G, counters, hd.q, hd.hd, hd.hd_q);
    IRS_LAUNCH_CHECK();
    return IRS_OK;
}

// both entry points: validation before any CUDA call, then the pairs of the range in launch groups of IRS_ASD_MAX_BOXES boxes
int surface_distances(const short* seg_a, long long a_chain_stride, const short* seg_b, const int* labels_host, int n_labels,
                      const int* boxes_host, const float* spacing_host, int pair_begin, int pair_end, float* workspace,
                      long long workspace_floats, double* partials, unsigned int* counters, double* asd, const HdOut& hd,
                      int C, int D, int H, int W, void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    if (!seg_a || !seg_b || !labels_host || !boxes_host || !spacing_host || !partials || !counters || !asd ||
        n_labels < 1 || n_labels > 32 || pair_begin < 0 || pair_end < pair_begin || pair_end > C * n_labels)
        return IRS_ERR_BAD_ARG;
    for (int i = 0; i < n_labels; ++i)
        if (labels_host[i] == 0) return IRS_ERR_UNSUPPORTED;
    for (int k = 0; k < 3; ++k)
        if (bad_spacing(spacing_host[k])) return IRS_ERR_BAD_ARG;
    const bool lists = hd.hd != nullptr;
    // spacing is (x, y, z): the W axis is weighted by spacing[0]^2
    const float w[3] = {spacing_host[0] * spacing_host[0], spacing_host[1] * spacing_host[1], spacing_host[2] * spacing_host[2]};
    long long need = 0;
    for (int p = pair_begin; p < pair_end; ++p) {
        const int* bx = boxes_host + (size_t)p * kBox;
        if (bx[6] <= 0 || bx[7] <= 0) continue;
        if (bx[0] < 0 || bx[1] < 0 || bx[2] < 0 || bx[0] > bx[3] || bx[1] > bx[4] || bx[2] > bx[5] || bx[3] >= D ||
            bx[4] >= H || bx[5] >= W)
            return IRS_ERR_BAD_ARG;
        need += 2LL * (bx[3] - bx[0] + 1) * (bx[4] - bx[1] + 1) * (bx[5] - bx[2] + 1);
        // the contour of A is a subset of A: |A| + |B| floats hold both lists
        if (lists) need += (long long)bx[6] + bx[7];
    }
    if (need > workspace_floats || (need > 0 && !workspace)) return IRS_ERR_WORKSPACE;
    if (pair_end == pair_begin) return IRS_OK;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(counters, 0, sizeof(unsigned int) * (lists ? IRS_SD_COUNTERS : IRS_ASD_MAX_BOXES), st);
    if (e != cudaSuccess) return (int)e;
    // an empty structure on either side gives inf (the reference's `except: ASD = inf`); the others are overwritten below
    const int n_pairs = pair_end - pair_begin;
    for (double* out : {asd, hd.hd, hd.hd_q}) {
        if (!out) continue;
        fill_kernel<<<(n_pairs + 255) / 256, 256, 0, st>>>(out + pair_begin, n_pairs, (double)INFINITY);
        IRS_LAUNCH_CHECK();
    }
    IrsDims d{D, H, W};
    AsdGroup G;
    G.n = 0;
    long long off = 0;
    for (int p = pair_begin; p < pair_end; ++p) {
        const int* bx = boxes_host + (size_t)p * kBox;
        if (bx[6] <= 0 || bx[7] <= 0) continue;
        if (G.n == 0) G.line0[0][0] = G.line0[1][0] = G.line0[2][0] = 0;
        AsdBox& B = G.b[G.n];
        B.off = off;
        B.c = p / n_labels;
        B.label = labels_host[p % n_labels];
        B.pair = p;
        B.z0 = bx[0]; B.y0 = bx[1]; B.x0 = bx[2];
        B.nd = bx[3] - bx[0] + 1; B.nh = bx[4] - bx[1] + 1; B.nw = bx[5] - bx[2] + 1;
        B.cap_a = bx[6];
        off += 2 * box_voxels(B) + (lists ? (long long)bx[6] + bx[7] : 0LL);
        G.line0[0][G.n + 1] = G.line0[0][G.n] + (long long)B.nd * B.nh;
        G.line0[1][G.n + 1] = G.line0[1][G.n] + 2LL * B.nd * B.nw;
        G.line0[2][G.n + 1] = G.line0[2][G.n] + 2LL * B.nh * B.nw;
        if (++G.n == IRS_ASD_MAX_BOXES) {
            IRS_TRY(launch_group(seg_a, a_chain_stride, seg_b, d, G, w, workspace, partials, counters, asd, hd, st));
            G.n = 0;
        }
    }
    return launch_group(seg_a, a_chain_stride, seg_b, d, G, w, workspace, partials, counters, asd, hd, st);
}

}  // namespace

extern "C" int irs_surface_boxes(const short* seg_a, long long a_chain_stride, const short* seg_b, const int* labels_host,
                                 int n_labels, int* boxes, int C, int D, int H, int W, void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    if (!seg_a || !seg_b || !labels_host || !boxes || n_labels < 1 || n_labels > 32) return IRS_ERR_BAD_ARG;
    LabelList l;
    l.n = n_labels;
    for (int i = 0; i < n_labels; ++i) {
        if (labels_host[i] == 0) return IRS_ERR_UNSUPPORTED;   // label 0 = background
        l.v[i] = labels_host[i];
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int n = C * n_labels * kBox;
    surface_box_init_kernel<<<(n + 255) / 256, 256, 0, st>>>(boxes, n);
    IRS_LAUNCH_CHECK();
    IrsDims d{D, H, W};
    const long long b = (d.V() + 255) / 256;
    surface_box_kernel<<<dim3((unsigned)(b < 296 ? b : 296), C), 256, 0, st>>>(seg_a, a_chain_stride, seg_b, l, boxes, d);
    return (int)cudaGetLastError();
}

extern "C" int irs_average_surface_distance(const short* seg_a, long long a_chain_stride, const short* seg_b,
                                            const int* labels_host, int n_labels, const int* boxes_host,
                                            const float* spacing_host, int pair_begin, int pair_end, float* workspace,
                                            long long workspace_floats, double* partials, unsigned int* counters,
                                            double* asd, int C, int D, int H, int W, void* stream) {
    return surface_distances(seg_a, a_chain_stride, seg_b, labels_host, n_labels, boxes_host, spacing_host, pair_begin,
                             pair_end, workspace, workspace_floats, partials, counters, asd, HdOut{0.0, nullptr, nullptr}, C,
                             D, H, W, stream);
}

extern "C" int irs_surface_distances(const short* seg_a, long long a_chain_stride, const short* seg_b,
                                     const int* labels_host, int n_labels, const int* boxes_host, const float* spacing_host,
                                     double percentile, int pair_begin, int pair_end, float* workspace,
                                     long long workspace_floats, double* partials, unsigned int* counters, double* asd,
                                     double* hd, double* hd_q, int C, int D, int H, int W, void* stream) {
    if (!hd || !hd_q || !(percentile >= 0.0 && percentile <= 100.0)) return IRS_ERR_BAD_ARG;
    return surface_distances(seg_a, a_chain_stride, seg_b, labels_host, n_labels, boxes_host, spacing_host, pair_begin,
                             pair_end, workspace, workspace_floats, partials, counters, asd, HdOut{percentile, hd, hd_q}, C,
                             D, H, W, stream);
}
