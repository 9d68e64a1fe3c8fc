// irs_metrics.cu -- per-sample evaluation kernels used at kept samples (SURVEY.md section 8f, N2):
//   log det J of the transformation + folded-voxel count   (reference utils/util.py:72-91,209-212)
//   Dice overlap counts for a list of labels                (reference utils/util.py:123-148)
#include "irs_kernels.cuh"

namespace {

// nabla[j][i] = d T_i / d x_j: forward differences with the last one replicated, divided by the spacing 2/(n-1)
// (reference utils/diff_op.py:78-96), then the 3x3 determinant written out as in utils/util.py:72-91
__global__ void __launch_bounds__(256)
log_det_j_kernel(const float* __restrict__ T_all, float* __restrict__ log_det, int* __restrict__ n_folded, IrsDims d) {
    const int V = (int)d.V();
    const int c = blockIdx.y;
    const float* T = T_all + (size_t)c * 3 * V;
    const int sy = d.W, sz = d.W * d.H;
    const float kx = 0.5f * (float)(d.W - 1), ky = 0.5f * (float)(d.H - 1), kz = 0.5f * (float)(d.D - 1);
    int folded = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < V; i += gridDim.x * blockDim.x) {
        const int x = i % d.W, y = (i / d.W) % d.H, z = i / sz;
        const int ix = x < d.W - 1 ? i : i - 1, iy = y < d.H - 1 ? i : i - sy, iz = z < d.D - 1 ? i : i - sz;
        float J[3][3];  // J[j][comp]
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const float* f = T + (size_t)ch * V;
            J[0][ch] = (__ldg(f + ix + 1) - __ldg(f + ix)) * kx;
            J[1][ch] = (__ldg(f + iy + sy) - __ldg(f + iy)) * ky;
            J[2][ch] = (__ldg(f + iz + sz) - __ldg(f + iz)) * kz;
        }
        // nabla_x = J[.][0], nabla_y = J[.][1], nabla_z = J[.][2]
        const float ld = irs_log_det_3x3(J);
        if (log_det != nullptr) log_det[(size_t)c * V + i] = ld;
        folded += (ld != ld) ? 1 : 0;   // NaN: negative determinant
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) folded += __shfl_xor_sync(0xffffffffu, folded, o);
    if ((threadIdx.x & 31) == 0 && folded) atomicAdd(n_folded + c, folded);   // integer: order independent
}

// counts[c][l] = (|A == l|, |B == l|, |A == l and B == l|)
__global__ void __launch_bounds__(256)
dice_counts_kernel(const short* __restrict__ seg_a, long long a_cs, const short* __restrict__ seg_b, LabelList labels,
                   unsigned int* __restrict__ counts, long long V) {
    __shared__ unsigned int sh[32 * 3];
    const int c = blockIdx.y;
    if (threadIdx.x < 96) sh[threadIdx.x] = 0u;
    __syncthreads();
    const short* a = seg_a + (size_t)c * a_cs;
    const short* b = seg_b + (size_t)c * V;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < V; i += (long long)gridDim.x * blockDim.x) {
        const int va = a[i], vb = b[i];
        if (va == 0 && vb == 0) continue;   // background is never a structure label in the reference's dictionary
        for (int l = 0; l < labels.n; ++l) {
            const bool ma = va == labels.v[l], mb = vb == labels.v[l];
            if (ma) atomicAdd(&sh[l * 3], 1u);
            if (mb) atomicAdd(&sh[l * 3 + 1], 1u);
            if (ma && mb) atomicAdd(&sh[l * 3 + 2], 1u);
        }
    }
    __syncthreads();
    if (threadIdx.x < labels.n * 3 && sh[threadIdx.x]) atomicAdd(counts + (size_t)c * labels.n * 3 + threadIdx.x, sh[threadIdx.x]);
}

}  // namespace

extern "C" int irs_log_det_jacobian(const float* T, float* log_det, int* n_folded, int C, int D, int H, int W,
                                    void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    if (!T || !n_folded) return IRS_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(n_folded, 0, sizeof(int) * C, st);
    if (e != cudaSuccess) return (int)e;
    IrsDims d{D, H, W};
    long long b = (d.V() + 255) / 256;
    dim3 grid((unsigned)(b < 1184 ? b : 1184), C);
    log_det_j_kernel<<<grid, 256, 0, st>>>(T, log_det, n_folded, d);
    return (int)cudaGetLastError();
}

extern "C" int irs_dice_counts(const short* seg_a, long long a_chain_stride, const short* seg_b, const int* labels_host,
                               int n_labels, unsigned int* counts, int C, long long V, void* stream) {
    if (!seg_a || !seg_b || !labels_host || !counts || n_labels < 1 || n_labels > 32 || C < 1 || V < 1)
        return IRS_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(counts, 0, sizeof(unsigned int) * C * n_labels * 3, st);
    if (e != cudaSuccess) return (int)e;
    LabelList l;
    l.n = n_labels;
    for (int i = 0; i < n_labels; ++i) {
        if (labels_host[i] == 0) return IRS_ERR_UNSUPPORTED;   // label 0 = background
        l.v[i] = labels_host[i];
    }
    long long b = (V + 255) / 256;
    dim3 grid((unsigned)(b < 592 ? b : 592), C);
    dice_counts_kernel<<<grid, 256, 0, st>>>(seg_a, a_chain_stride, seg_b, l, counts, V);
    return (int)cudaGetLastError();
}
