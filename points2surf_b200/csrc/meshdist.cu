// K9: the acceptance metric of the reconstruction path on the device -- area-weighted surface sampling and the
// symmetric nearest-neighbour distances behind `_chamfer_distance_single_file` / `_hausdorff_distance_single_file`
// (source/base/evaluation.py:222-304).  The reference samples with trimesh.sample.sample_surface_even and queries
// two cKDTrees; both libraries are absent here (parity unpinned for the sampler, see oracle/p2s_oracle.py:
// sample_mesh_surface), the distance part is pinned against scipy.spatial.cKDTree in the tests.
//   1. face areas (f64) -> inclusive scan (CUB)                 2. sample: Philox -> face by binary search of the
//   cumulative area, uniform barycentric coordinates (reflection rule)
//   3. exhaustive tiled nearest neighbour: every CTA stages a slab of the target cloud in shared memory, one source
//   point per thread, best (d^2, index) merged across slabs with a 64-bit atomicMin
//   4. finalise: sqrt, sum (f64) and max per direction.
// 10^4 x 10^4 samples = 10^8 distance evaluations: compute-trivial, latency-bound; sized to fill the 148 SMs.
#include "common.cuh"
#include <cub/device/device_scan.cuh>

namespace p2s {

namespace {

__global__ void face_area_kernel(const float* __restrict__ verts, const int32_t* __restrict__ faces, int64_t F,
                                 int64_t V, double* __restrict__ area) {
    int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    int32_t a = faces[3 * f], b = faces[3 * f + 1], c = faces[3 * f + 2];
    double out = 0.0;
    if (a >= 0 && b >= 0 && c >= 0 && a < V && b < V && c < V) {
        double ax = verts[3 * (int64_t)a], ay = verts[3 * (int64_t)a + 1], az = verts[3 * (int64_t)a + 2];
        double ux = verts[3 * (int64_t)b] - ax, uy = verts[3 * (int64_t)b + 1] - ay, uz = verts[3 * (int64_t)b + 2] - az;
        double wx = verts[3 * (int64_t)c] - ax, wy = verts[3 * (int64_t)c + 1] - ay, wz = verts[3 * (int64_t)c + 2] - az;
        double cx = uy * wz - uz * wy, cy = uz * wx - ux * wz, cz = ux * wy - uy * wx;
        out = 0.5 * sqrt(cx * cx + cy * cy + cz * cz);
    }
    area[f] = out;
}

__global__ void mesh_sample_kernel(const float* __restrict__ verts, const int32_t* __restrict__ faces, int64_t F,
                                   const double* __restrict__ cum, int64_t n, uint64_t seed,
                                   float* __restrict__ samples, int32_t* __restrict__ face_ids) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t r[4];
    philox4x32_10((uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)i, (uint32_t)(i >> 32), 0u, 0x3e5a11c7u, r);
    // 53-bit uniform in [0,1) for the face pick, 24-bit uniforms for the barycentric coordinates
    double u = (double)((((uint64_t)r[0] << 32) | r[1]) >> 11) * (1.0 / 9007199254740992.0);
    double target = u * cum[F - 1];
    int64_t lo = 0, hi = F - 1;   // first face whose cumulative area exceeds the target
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if (cum[mid] > target) hi = mid; else lo = mid + 1;
    }
    float r1 = (float)(r[2] >> 8) * (1.0f / 16777216.0f), r2 = (float)(r[3] >> 8) * (1.0f / 16777216.0f);
    if (r1 + r2 > 1.0f) { r1 = 1.0f - r1; r2 = 1.0f - r2; }
    int64_t a = faces[3 * lo], b = faces[3 * lo + 1], c = faces[3 * lo + 2];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        float p0 = verts[3 * a + d], p1 = verts[3 * b + d], p2 = verts[3 * c + d];
        samples[3 * i + d] = p0 + r1 * (p1 - p0) + r2 * (p2 - p0);
    }
    if (face_ids) face_ids[i] = (int32_t)lo;
}

constexpr int kNnThreads = 256;
constexpr int kNnTile = 1024;   // target points per shared-memory tile (12 KB as SoA floats)

__global__ void nn_init_kernel(unsigned long long* __restrict__ best, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) best[i] = ~0ull;
}

// grid (ceil(na / 256), slabs): slab s covers targets [s * slab_len, min(nb, (s + 1) * slab_len))
__global__ void __launch_bounds__(kNnThreads)
nn_slab_kernel(const float* __restrict__ a, int64_t na, const float* __restrict__ b, int64_t nb, int64_t slab_len,
               unsigned long long* __restrict__ best) {
    __shared__ float sx[kNnTile], sy[kNnTile], sz[kNnTile];
    int64_t i = (int64_t)blockIdx.x * kNnThreads + threadIdx.x;
    float px = 0.f, py = 0.f, pz = 0.f;
    if (i < na) { px = a[3 * i]; py = a[3 * i + 1]; pz = a[3 * i + 2]; }
    int64_t j0 = (int64_t)blockIdx.y * slab_len, j1 = min(nb, j0 + slab_len);
    float bd = INFINITY;
    int64_t bj = -1;
    for (int64_t t = j0; t < j1; t += kNnTile) {
        int cnt = (int)min((int64_t)kNnTile, j1 - t);
        __syncthreads();
        for (int k = threadIdx.x; k < cnt; k += kNnThreads) {
            sx[k] = b[3 * (t + k)]; sy[k] = b[3 * (t + k) + 1]; sz[k] = b[3 * (t + k) + 2];
        }
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < cnt; ++k) {
            float dx = __fsub_rn(px, sx[k]), dy = __fsub_rn(py, sy[k]), dz = __fsub_rn(pz, sz[k]);
            float d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
            if (d < bd) { bd = d; bj = t + k; }   // strict <: the lowest index wins ties inside a slab
        }
    }
    if (i < na && bj >= 0) {
        // non-negative floats order like their bit patterns; the index in the low word breaks ties towards the lowest j
        unsigned long long key = ((unsigned long long)__float_as_uint(bd) << 32) | (uint32_t)bj;
        atomicMin(best + i, key);
    }
}

// out[0] += sum of distances (f64), out_max (float bits, non-negative) = max distance
__global__ void __launch_bounds__(256)
nn_finalize_kernel(const unsigned long long* __restrict__ best, int64_t na, float* __restrict__ dist,
                   int32_t* __restrict__ idx, double* __restrict__ sum_out, unsigned int* __restrict__ max_out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float d = 0.f;
    if (i < na) {
        unsigned long long key = best[i];
        d = sqrtf(__uint_as_float((uint32_t)(key >> 32)));
        if (dist) dist[i] = d;
        if (idx) idx[i] = (int32_t)(uint32_t)key;
    }
    if (!sum_out) return;
    double s = d;
    float m = d;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    }
    __shared__ double ws[8];
    __shared__ float wm[8];
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { ws[w] = s; wm[w] = m; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < 8; ++k) { s += ws[k]; m = fmaxf(m, wm[k]); }
        atomicAdd(sum_out, s);
        atomicMax(max_out, __float_as_uint(m));
    }
}

void nn_core(const float* a, int64_t na, const float* b, int64_t nb, float* dist, int32_t* idx, double* sum_out,
             unsigned int* max_out, cudaStream_t st) {
    DeviceCtx& ctx = device_ctx();
    unsigned long long* best = ctx.mesh_best.as<unsigned long long>((size_t)na);
    P2S_LAUNCH(nn_init_kernel, (unsigned)cdiv(na, 256), 256, 0, st, best, na);
    int64_t gx = cdiv(na, kNnThreads);
    int64_t max_slabs = cdiv(nb, kNnTile);
    int64_t slabs = std::min<int64_t>(max_slabs, std::max<int64_t>(1, cdiv(4 * (int64_t)ctx.sm_count, gx)));
    slabs = std::min<int64_t>(slabs, 65535);
    int64_t slab_len = cdiv(cdiv(nb, slabs), kNnTile) * kNnTile;
    slabs = cdiv(nb, slab_len);
    P2S_LAUNCH(nn_slab_kernel, dim3((unsigned)gx, (unsigned)slabs), kNnThreads, 0, st, a, na, b, nb, slab_len, best);
    P2S_LAUNCH(nn_finalize_kernel, (unsigned)cdiv(na, 256), 256, 0, st, best, na, dist, idx, sum_out, max_out);
}

}  // namespace

void mesh_sample(const float* verts, int64_t V, const int32_t* faces, int64_t F, int64_t n, uint64_t seed,
                 float* samples, int32_t* face_ids, cudaStream_t st) {
    P2S_CHECK(V > 0 && F > 0, "empty mesh");
    if (n <= 0) return;
    DeviceCtx& ctx = device_ctx();
    double* area = ctx.mesh_area.as<double>((size_t)F);
    double* cum = ctx.mesh_cum.as<double>((size_t)F);
    P2S_LAUNCH(face_area_kernel, (unsigned)cdiv(F, 256), 256, 0, st, verts, faces, F, V, area);
    size_t tmp_bytes = 0;
    P2S_CUDA(cub::DeviceScan::InclusiveSum(nullptr, tmp_bytes, area, cum, (int)F, st));
    void* tmp = ctx.mesh_cub.get(tmp_bytes);
    P2S_CUDA(cub::DeviceScan::InclusiveSum(tmp, tmp_bytes, area, cum, (int)F, st));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    P2S_LAUNCH(mesh_sample_kernel, (unsigned)cdiv(n, 256), 256, 0, st, verts, faces, F, cum, n, seed, samples, face_ids);
}

void nn_distance(const float* a, int64_t na, const float* b, int64_t nb, float* dist, int32_t* idx, cudaStream_t st) {
    P2S_CHECK(nb > 0, "empty target cloud");
    if (na <= 0) return;
    nn_core(a, na, b, nb, dist, idx, nullptr, nullptr, st);
}

// out4 (host): sum a->b, sum b->a, max a->b, max b->a
void chamfer_hausdorff(const float* a, int64_t na, const float* b, int64_t nb, double* out4_host, cudaStream_t st) {
    P2S_CHECK(na > 0 && nb > 0, "empty cloud");
    // [0..1] f64 sums, then 2 x u32 maxima
    double* red = device_ctx().mesh_red.as<double>(3);
    P2S_CUDA(cudaMemsetAsync(red, 0, 3 * sizeof(double), st));
    unsigned int* mx = reinterpret_cast<unsigned int*>(red + 2);
    nn_core(a, na, b, nb, nullptr, nullptr, red + 0, mx + 0, st);
    nn_core(b, nb, a, na, nullptr, nullptr, red + 1, mx + 1, st);
    double h[3];
    P2S_CUDA(cudaMemcpyAsync(h, red, sizeof(h), cudaMemcpyDeviceToHost, st));
    P2S_CUDA(cudaStreamSynchronize(st));
    unsigned int hm[2];
    memcpy(hm, &h[2], sizeof(hm));
    float m0, m1;
    memcpy(&m0, &hm[0], 4);
    memcpy(&m1, &hm[1], 4);
    out4_host[0] = h[0]; out4_host[1] = h[1]; out4_host[2] = m0; out4_host[3] = m1;
}

}  // namespace p2s
