// irs_segpost.cu -- posterior of the warped segmentation: a per-voxel histogram of labels over every accumulated sample.
//   update   per kept sample, the C warped segmentations (C, V) int16 are added into counts (L, V) int32: counts[l][v] is the
//            number of segmentations whose voxel v carries labels[l].  The class "other" (0, negative values, any value not
//            in the list) is never stored.  One thread owns VW consecutive voxels of every label row: no atomics, and each
//            counts element is read and written at most once per launch.
//   finish   from the counts of n segmentations: probabilities (float)c / (float)n, the majority label (ties to "other", then
//            to the earlier entry of the list), the label entropy over the L + 1 classes, and exact int64 summaries per label
//            (sum of the counts, the same inside the fixed segmentation's structure, voxels with 0 < count < n) through
//            block sums in shared memory and one 64-bit integer atomicAdd per block and value -- order independent.
// Integer counts make the result independent of how the samples are batched or split over GPUs (parallel.merge_label_counts
// sum-all-reduces them).
#include <cstdint>

#include "irs_kernels.cuh"

namespace {

constexpr unsigned FULL = 0xffffffffu;

// the bit of the list slot holding label value v, 0 for "other" (the compare loop of dice_counts_kernel)
__device__ __forceinline__ unsigned slot_bit(int v, const LabelList& labels) {
    if (v == 0) return 0u;   // background: never a label (the list holds no 0)
    for (int l = 0; l < labels.n; ++l)
        if (v == labels.v[l]) return 1u << l;
    return 0u;
}

template <int VW>
__device__ __forceinline__ void load_shorts(const short* __restrict__ p, short (&x)[VW]) {
    if constexpr (VW == 4) {
        const short4 t = __ldg(reinterpret_cast<const short4*>(p));
        x[0] = t.x; x[1] = t.y; x[2] = t.z; x[3] = t.w;
    } else {
        x[0] = __ldg(p);
    }
}

template <int VW>
__device__ __forceinline__ void load_ints(const int* __restrict__ p, int (&x)[VW]) {
    if constexpr (VW == 4) {
        const int4 t = __ldg(reinterpret_cast<const int4*>(p));
        x[0] = t.x; x[1] = t.y; x[2] = t.z; x[3] = t.w;
    } else {
        x[0] = __ldg(p);
    }
}

// grid: one thread per VW consecutive voxels.  VW = 4: 8-byte segmentation loads and int4 read-modify-writes of the counts
// (V % 4 == 0, aligned buffers); VW = 1 otherwise.
template <int VW>
__global__ void __launch_bounds__(256)
label_counts_kernel(const short* __restrict__ seg, int C, long long V, LabelList labels, int* __restrict__ counts) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= V / VW) return;
    const short* s = seg + q * VW;
    // pass 1: which list slots occur in this thread's voxels in any chain
    unsigned present = 0u;
#pragma unroll 4
    for (int c = 0; c < C; ++c) {
        short x[VW];
        load_shorts<VW>(s + (size_t)c * V, x);
#pragma unroll
        for (int k = 0; k < VW; ++k) present |= slot_bit(x[k], labels);
    }
    // pass 2, per occurring slot: count it over the same (L1-resident) values, then one read-modify-write of its row
    while (present) {
        const int l = __ffs(present) - 1;
        present &= present - 1u;
        const int lab = labels.v[l];
        int add[VW];
#pragma unroll
        for (int k = 0; k < VW; ++k) add[k] = 0;
#pragma unroll 4
        for (int c = 0; c < C; ++c) {
            short x[VW];
            load_shorts<VW>(s + (size_t)c * V, x);
#pragma unroll
            for (int k = 0; k < VW; ++k) add[k] += x[k] == lab ? 1 : 0;
        }
        int* p = counts + (size_t)l * V + q * VW;
        if constexpr (VW == 4) {
            int4 cur = *reinterpret_cast<int4*>(p);
            cur.x += add[0]; cur.y += add[1]; cur.z += add[2]; cur.w += add[3];
            *reinterpret_cast<int4*>(p) = cur;
        } else {
            *p += add[0];
        }
    }
}

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// grid-stride over groups of VW voxels; every thread of a block runs the same number of iterations (warp votes below)
template <int VW>
__global__ void __launch_bounds__(256)
label_posterior_kernel(const int* __restrict__ counts, LabelList labels, int n, long long V,
                       const short* __restrict__ seg_fixed, float* __restrict__ prob, short* __restrict__ majority,
                       float* __restrict__ entropy, unsigned long long* __restrict__ summary) {
    __shared__ unsigned long long acc[32 * 3];   // per label: S, O, U of this block
    for (int i = threadIdx.x; i < 32 * 3; i += blockDim.x) acc[i] = 0ull;
    __syncthreads();
    const float nf = (float)n;
    const long long nq = V / VW;
    const int lane = threadIdx.x & 31;
    for (long long base = (long long)blockIdx.x * blockDim.x; base < nq; base += (long long)gridDim.x * blockDim.x) {
        const long long q = base + threadIdx.x;
        const bool active = q < nq;
        short f[VW];
#pragma unroll
        for (int k = 0; k < VW; ++k) f[k] = 0;
        if (active && seg_fixed != nullptr) load_shorts<VW>(seg_fixed + q * VW, f);
        int total[VW], best[VW], best_slot[VW];
        float H[VW];
#pragma unroll
        for (int k = 0; k < VW; ++k) { total[k] = 0; best[k] = -1; best_slot[k] = 0; H[k] = 0.f; }
        for (int l = 0; l < labels.n; ++l) {
            const int lab = labels.v[l];
            int c[VW];
#pragma unroll
            for (int k = 0; k < VW; ++k) c[k] = 0;
            if (active) load_ints<VW>(counts + (size_t)l * V + q * VW, c);
            float p[VW];
            unsigned long long s = 0ull, o = 0ull, u = 0ull;
#pragma unroll
            for (int k = 0; k < VW; ++k) {
                p[k] = (float)c[k] / nf;
                total[k] += c[k];
                if (c[k] > best[k]) { best[k] = c[k]; best_slot[k] = l; }   // strict: the earlier entry keeps a tie
                if (c[k] > 0) H[k] -= p[k] * logf(p[k]);
                s += (unsigned long long)c[k];
                o += f[k] == lab ? (unsigned long long)c[k] : 0ull;
                u += (c[k] > 0 && c[k] < n) ? 1ull : 0ull;
            }
            if (active) {
                float* pp = prob + (size_t)l * V + q * VW;
                if constexpr (VW == 4) *reinterpret_cast<float4*>(pp) = make_float4(p[0], p[1], p[2], p[3]);
                else *pp = p[0];
            }
            if (__any_sync(FULL, (s | o | u) != 0ull)) {   // most voxels carry no label: skip the reduction there
                s = warp_sum_u64(s);
                o = warp_sum_u64(o);
                u = warp_sum_u64(u);
                if (lane == 0) {
                    if (s) atomicAdd(&acc[3 * l], s);
                    if (o) atomicAdd(&acc[3 * l + 1], o);
                    if (u) atomicAdd(&acc[3 * l + 2], u);
                }
            }
        }
        if (!active) continue;
        short m[VW];
        float h[VW];
#pragma unroll
        for (int k = 0; k < VW; ++k) {
            const int other = n - total[k];
            m[k] = other >= best[k] ? (short)0 : (short)labels.v[best_slot[k]];   // "other" wins ties
            h[k] = H[k];
            if (other > 0) {
                const float po = (float)other / nf;
                h[k] -= po * logf(po);
            }
        }
        if constexpr (VW == 4) {
            *reinterpret_cast<short4*>(majority + q * VW) = make_short4(m[0], m[1], m[2], m[3]);
            *reinterpret_cast<float4*>(entropy + q * VW) = make_float4(h[0], h[1], h[2], h[3]);
        } else {
            majority[q] = m[0];
            entropy[q] = h[0];
        }
    }
    __syncthreads();
    if (threadIdx.x < labels.n * 3 && acc[threadIdx.x]) atomicAdd(summary + threadIdx.x, acc[threadIdx.x]);
}

// the label list of both entry points: 1..32 distinct non-zero int16 values
int make_labels(const int* labels_host, int n_labels, LabelList* out) {
    if (!labels_host || n_labels < 1 || n_labels > 32) return IRS_ERR_BAD_ARG;
    out->n = n_labels;
    for (int i = 0; i < n_labels; ++i) {
        const int v = labels_host[i];
        if (v == 0) return IRS_ERR_UNSUPPORTED;   // label 0 = background, as for irs_dice_counts
        if (v < -32768 || v > 32767) return IRS_ERR_BAD_ARG;
        for (int j = 0; j < i; ++j)
            if (labels_host[j] == v) return IRS_ERR_BAD_ARG;
        out->v[i] = v;
    }
    return IRS_OK;
}

bool aligned(const void* p, unsigned bytes) { return (reinterpret_cast<uintptr_t>(p) & (bytes - 1)) == 0; }

}  // namespace

extern "C" int irs_label_counts_update(const short* seg, int C, long long V, const int* labels_host, int n_labels,
                                       int* counts, void* stream) {
    if (!seg || !counts || C < 1 || V < 1) return IRS_ERR_BAD_ARG;
    LabelList labels;
    IRS_TRY(make_labels(labels_host, n_labels, &labels));
    cudaStream_t st = (cudaStream_t)stream;
    if (V % 4 == 0 && aligned(seg, 8) && aligned(counts, 16))
        label_counts_kernel<4><<<(unsigned)((V / 4 + 255) / 256), 256, 0, st>>>(seg, C, V, labels, counts);
    else
        label_counts_kernel<1><<<(unsigned)((V + 255) / 256), 256, 0, st>>>(seg, C, V, labels, counts);
    return (int)cudaGetLastError();
}

extern "C" int irs_label_posterior(const int* counts, const int* labels_host, int n_labels, long long n, long long V,
                                   const short* seg_fixed, float* prob, short* majority, float* entropy, long long* summary,
                                   void* stream) {
    // n > INT_MAX cannot be the number of segmentations behind int32 counts
    if (!counts || !prob || !majority || !entropy || !summary || n < 1 || n > 0x7fffffffLL || V < 1) return IRS_ERR_BAD_ARG;
    LabelList labels;
    IRS_TRY(make_labels(labels_host, n_labels, &labels));
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(summary, 0, sizeof(long long) * 3 * n_labels, st);
    if (e != cudaSuccess) return (int)e;
    unsigned long long* sm = reinterpret_cast<unsigned long long*>(summary);
    const bool vec = V % 4 == 0 && aligned(counts, 16) && aligned(prob, 16) && aligned(entropy, 16) && aligned(majority, 8) &&
                     aligned(seg_fixed, 8);
    const long long groups = vec ? V / 4 : V;
    const long long b = (groups + 255) / 256;
    const unsigned nb = (unsigned)(b < 148 * 8 ? b : 148 * 8);
    if (vec)
        label_posterior_kernel<4><<<nb, 256, 0, st>>>(counts, labels, (int)n, V, seg_fixed, prob, majority, entropy, sm);
    else
        label_posterior_kernel<1><<<nb, 256, 0, st>>>(counts, labels, (int)n, V, seg_fixed, prob, majority, entropy, sm);
    return (int)cudaGetLastError();
}
