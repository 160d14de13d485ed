// K1: candidate query grid -- sdf.get_voxel_centers_grid_smaller_pc (source/sdf.py:46-70).
// occupancy scatter -> eps^3 box dilation (any-occupied; the reference's float box sum is only tested
// for != 0) -> ordered compaction (C order == np.nonzero order) with the last index plane dropped.
// HBM/L2-bound byte work: res^3 B written + read, Q*4 B of indices out.
#include "common.cuh"
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

namespace p2s {

// model_space_to_volume_space (source/sdf.py:73-75) in the reference's float32 arithmetic
__device__ __forceinline__ int ms_to_vs(float p, int res) {
    float t = __fdiv_rn(__fadd_rn(p, 1.0f), 2.0f);
    return (int)floorf(__fmul_rn(t, (float)res));
}

__global__ void occupancy_kernel(const float* __restrict__ pts, int64_t N, int res, uint8_t* __restrict__ occ) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    int ix = ms_to_vs(pts[i * 3 + 0], res), iy = ms_to_vs(pts[i * 3 + 1], res), iz = ms_to_vs(pts[i * 3 + 2], res);
    if ((unsigned)ix >= (unsigned)res || (unsigned)iy >= (unsigned)res || (unsigned)iz >= (unsigned)res) return;
    occ[((int64_t)ix * res + iy) * res + iz] = 1;
}

// An occupied voxel i marks outputs i+d, d in [-floor(e/2), ceil(e/2)-1] (scipy.ndimage.convolve with a
// ones kernel, origin 0; SURVEY.md section 10) => output o looks at inputs o-ceil(e/2)+1 .. o+floor(e/2).
// One thread per 4 consecutive z voxels.
__global__ void dilate_flag_kernel(const uint8_t* __restrict__ occ, int res, int lo, int hi, uint8_t* __restrict__ flag) {
    const int zq = (res + 3) / 4;
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t total = (int64_t)res * res * zq;
    if (t >= total) return;
    int z0 = (int)(t % zq) * 4;
    int y = (int)((t / zq) % res);
    int x = (int)(t / ((int64_t)zq * res));
    unsigned any[4] = {0, 0, 0, 0};
    const int x_lo = max(x + lo, 0), x_hi = min(x + hi, res - 1);
    const int y_lo = max(y + lo, 0), y_hi = min(y + hi, res - 1);
    const int z_lo = max(z0 + lo, 0), z_hi = min(z0 + 3 + hi, res - 1);
    for (int xx = x_lo; xx <= x_hi; ++xx)
        for (int yy = y_lo; yy <= y_hi; ++yy) {
            const uint8_t* row = occ + ((int64_t)xx * res + yy) * res;
            for (int zz = z_lo; zz <= z_hi; ++zz) {
                unsigned o = row[zz];
#pragma unroll
                for (int j = 0; j < 4; ++j) any[j] |= (zz >= z0 + j + lo && zz <= z0 + j + hi) ? o : 0u;
            }
        }
    const bool xy_ok = (x < res - 1) && (y < res - 1);   // [:-1,:-1,:-1]  (sdf.py:66)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        int z = z0 + j;
        if (z < res) flag[((int64_t)x * res + y) * res + z] = (xy_ok && z < res - 1 && any[j]) ? 1 : 0;
    }
}

__global__ void query_points_kernel(const int32_t* __restrict__ lin, int64_t Q, int res, float* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Q) return;
    int v = lin[i];
    int iz = v % res, iy = (v / res) % res, ix = v / (res * res);
    // volume_space_to_model_space on int64 -> float64, then astype(float32)   (sdf.py:67-70,78-79)
    out[i * 3 + 0] = (float)(((double)ix + 0.5) / (double)res * 2.0 - 1.0);
    out[i * 3 + 1] = (float)(((double)iy + 0.5) / (double)res * 2.0 - 1.0);
    out[i * 3 + 2] = (float)(((double)iz + 0.5) / (double)res * 2.0 - 1.0);
}

void query_grid(const float* pts, int64_t N, int res, int eps, int32_t* lin_idx, int64_t cap,
                int64_t* count_host, cudaStream_t st) {
    P2S_CHECK(res >= 2 && res <= 1024, "grid resolution out of range");
    P2S_CHECK(eps >= 1 && eps <= 31, "epsilon out of range");
    const int64_t vox = (int64_t)res * res * res;
    size_t cub_bytes = 0;
    cub::CountingInputIterator<int32_t> counting(0);
    int* d_num = nullptr;
    cub::DeviceSelect::Flagged(nullptr, cub_bytes, counting, (uint8_t*)nullptr, (int32_t*)nullptr, d_num, (int)vox, st);
    size_t off_flag = (size_t)vox, off_sel = off_flag + (size_t)vox;
    off_sel = (off_sel + 255) / 256 * 256;
    size_t off_num = off_sel + (size_t)vox * 4;
    size_t off_cub = off_num + 256;
    uint8_t* base = (uint8_t*)device_ctx().grid_ws.get(off_cub + cub_bytes);
    uint8_t* occ = base;
    uint8_t* flag = base + off_flag;
    int32_t* sel = (int32_t*)(base + off_sel);
    d_num = (int*)(base + off_num);
    P2S_CUDA(cudaMemsetAsync(occ, 0, (size_t)vox, st));
    P2S_LAUNCH(occupancy_kernel, (unsigned)cdiv(N, 256), 256, 0, st, pts, N, res, occ);
    const int lo = -((eps + 1) / 2) + 1, hi = eps / 2;
    const int64_t threads = (int64_t)res * res * ((res + 3) / 4);
    P2S_LAUNCH(dilate_flag_kernel, (unsigned)cdiv(threads, 256), 256, 0, st, occ, res, lo, hi, flag);
    P2S_CUDA(cub::DeviceSelect::Flagged(base + off_cub, cub_bytes, counting, flag, sel, d_num, (int)vox, st));
    g_launches.fetch_add(2, std::memory_order_relaxed);  // cub: scan + select kernels
    int h_num = 0;
    P2S_CUDA(cudaMemcpyAsync(&h_num, d_num, sizeof(int), cudaMemcpyDeviceToHost, st));
    P2S_CUDA(cudaStreamSynchronize(st));
    *count_host = h_num;
    int64_t ncopy = h_num < cap ? h_num : cap;
    if (ncopy > 0) P2S_CUDA(cudaMemcpyAsync(lin_idx, sel, (size_t)ncopy * 4, cudaMemcpyDeviceToDevice, st));
}

void query_points(const int32_t* lin_idx, int64_t Q, int res, float* out, cudaStream_t st) {
    if (Q <= 0) return;
    P2S_LAUNCH(query_points_kernel, (unsigned)cdiv(Q, 256), 256, 0, st, lin_idx, Q, res, out);
}

}  // namespace p2s
