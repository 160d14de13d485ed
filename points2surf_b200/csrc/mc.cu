// K8: marching cubes at `level` + unit-cube transform + orientation fix -- the tail of
// sdf.implicit_surface_to_mesh (source/sdf.py:211-227).  The reference delegates to
// skimage.measure.marching_cubes_lewiner and trimesh.repair.fix_inversion (both absent here: parity
// unpinned, see oracle/mc_oracle.py for the shared conventions).  Ambiguous faces are resolved by the asymptotic decider
// (the face test of Lewiner's algorithm); the interior (tunnel) test of MC33 is not implemented.  HBM-bound: res^3*4 B read (+ L2-resident
// re-reads of neighbours), ~20 B/voxel of scan scratch, V*12 + F*12 B written.
//   1. flag sign-changing grid edges (3 per voxel)      2. exclusive scan -> vertex ids (welded by edge)
//   3. emit vertices (linear interpolation, fp32)       4. per-cell case -> triangle count, scan
//   5. emit faces through the edge -> vertex map        6. signed volume, flip all faces if negative
#include "common.cuh"
#include "mc_tables.cuh"
#include <cub/device/device_scan.cuh>

namespace p2s {

namespace {

__global__ void mc_edge_flags_kernel(const float* __restrict__ vol, int R, float level, uint8_t* __restrict__ flags) {
    int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t V = (int64_t)R * R * R;
    if (v >= V) return;
    int iz = (int)(v % R), iy = (int)((v / R) % R), ix = (int)(v / ((int64_t)R * R));
    bool p = vol[v] > level;
    flags[3 * v + 0] = (ix + 1 < R) && ((vol[v + (int64_t)R * R] > level) != p);
    flags[3 * v + 1] = (iy + 1 < R) && ((vol[v + R] > level) != p);
    flags[3 * v + 2] = (iz + 1 < R) && ((vol[v + 1] > level) != p);
}

__global__ void mc_emit_verts_kernel(const float* __restrict__ vol, int R, float level, const uint8_t* __restrict__ flags,
                                     const int32_t* __restrict__ vid, float* __restrict__ verts, int64_t vcap) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t E = 3 * (int64_t)R * R * R;
    if (e >= E || !flags[e]) return;
    int32_t id = vid[e];
    if (id >= vcap) return;
    int64_t v = e / 3;
    int a = (int)(e % 3);
    int iz = (int)(v % R), iy = (int)((v / R) % R), ix = (int)(v / ((int64_t)R * R));
    int64_t stride = a == 0 ? (int64_t)R * R : (a == 1 ? R : 1);
    float v0 = vol[v], v1 = vol[v + stride];
    float t = __fdiv_rn(__fsub_rn(level, v0), __fsub_rn(v1, v0));
    float p[3] = {(float)ix, (float)iy, (float)iz};
    p[a] = __fadd_rn(p[a], t);
#pragma unroll
    for (int d = 0; d < 3; ++d)   // ((v + 0.5) / res - 0.5) * 2   (sdf.py:224), fp32
        verts[(int64_t)id * 3 + d] = __fmul_rn(__fsub_rn(__fdiv_rn(__fadd_rn(p[d], 0.5f), (float)R), 0.5f), 2.0f);
}

// Table row of a cell: the corner-sign case plus, for every ambiguous face (+-+-), the asymptotic decider -- are the two
// positive corners joined through the face?  The bilinear interpolant's saddle value is (A*C - B*D) / (A + C - B - D) with
// A, C / B, D the two diagonals (values minus level); the denominator's sign is that of the A/C diagonal, so the decision is
// the sign of A*C - B*D, evaluated in float64 with separately rounded products (no FMA contraction) exactly like the CPU
// restatement (oracle/mc_topo.py), so that both sides take identical decisions.
__device__ __forceinline__ int mc_row(const float* __restrict__ vol, int R, float level, int cx, int cy, int cz) {
    int c = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        int dx = k & 1, dy = (k >> 1) & 1, dz = (k >> 2) & 1;
        c |= (vol[((int64_t)(cx + dx) * R + (cy + dy)) * R + (cz + dz)] > level) ? (1 << k) : 0;
    }
    int row = kMcRowBase[c];
    const unsigned amb = kMcAmbMask[c];
    if (amb) {
        int bit = 0;
        for (int f = 0; f < 6; ++f) {
            if (!((amb >> f) & 1u)) continue;
            double d[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int k = kMcFaceRing[f][i];
                d[i] = __dsub_rn((double)vol[((int64_t)(cx + (k & 1)) * R + (cy + ((k >> 1) & 1))) * R + (cz + ((k >> 2) & 1))], (double)level);
            }
            const double num = __dsub_rn(__dmul_rn(d[0], d[2]), __dmul_rn(d[1], d[3]));
            const bool joined = ((c >> kMcFaceRing[f][0]) & 1) ? (num > 0.0) : (num < 0.0);
            row += joined ? (1 << bit) : 0;
            ++bit;
        }
    }
    return row;
}

__global__ void mc_cell_count_kernel(const float* __restrict__ vol, int R, float level, uint8_t* __restrict__ counts) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int C = R - 1;
    if (i >= (int64_t)C * C * C) return;
    int cz = (int)(i % C), cy = (int)((i / C) % C), cx = (int)(i / ((int64_t)C * C));
    counts[i] = kMcTriCount[mc_row(vol, R, level, cx, cy, cz)];
}

__global__ void mc_emit_faces_kernel(const float* __restrict__ vol, int R, float level, const uint8_t* __restrict__ counts,
                                     const int32_t* __restrict__ offs, const int32_t* __restrict__ vid,
                                     int32_t* __restrict__ faces, int64_t fcap) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int C = R - 1;
    if (i >= (int64_t)C * C * C) return;
    int n = counts[i];
    if (n == 0) return;
    int cz = (int)(i % C), cy = (int)((i / C) % C), cx = (int)(i / ((int64_t)C * C));
    int cs = mc_row(vol, R, level, cx, cy, cz);
    int32_t off = offs[i];
    for (int t = 0; t < n; ++t) {
        if (off + t >= fcap) return;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            int e = kMcTriTable[cs][3 * t + j];
            int a = e >> 2, r = e & 3;
            int lo[3] = {0, 0, 0};
            int o0 = a == 0 ? 1 : 0, o1 = a == 2 ? 1 : 2;   // the two axes other than a, ascending
            lo[o0] = r & 1;
            lo[o1] = r >> 1;
            int64_t g = 3 * (((int64_t)(cx + lo[0]) * R + (cy + lo[1])) * R + (cz + lo[2])) + a;
            faces[(int64_t)(off + t) * 3 + j] = vid[g];
        }
    }
}

__global__ void mc_signed_volume_kernel(const float* __restrict__ verts, const int32_t* __restrict__ faces, int64_t F, double* acc) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double v = 0.0;
    if (i < F) {
        const float* a = verts + (int64_t)faces[i * 3 + 0] * 3;
        const float* b = verts + (int64_t)faces[i * 3 + 1] * 3;
        const float* c = verts + (int64_t)faces[i * 3 + 2] * 3;
        double cx = (double)b[1] * c[2] - (double)b[2] * c[1];
        double cy = (double)b[2] * c[0] - (double)b[0] * c[2];
        double cz = (double)b[0] * c[1] - (double)b[1] * c[0];
        v = (double)a[0] * cx + (double)a[1] * cy + (double)a[2] * cz;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v != 0.0) atomicAdd(acc, v);
}

__global__ void mc_flip_kernel(int32_t* __restrict__ faces, int64_t F, const double* acc) {
    if (*acc >= 0.0) return;   // trimesh.repair.fix_inversion: invert only when the volume is negative
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F) return;
    int32_t t = faces[i * 3 + 1];
    faces[i * 3 + 1] = faces[i * 3 + 2];
    faces[i * 3 + 2] = t;
}

}  // namespace

void marching_cubes(const float* vol, int R, float level, float* verts, int64_t vcap, int32_t* faces, int64_t fcap,
                    int64_t* nverts_host, int64_t* nfaces_host, cudaStream_t st) {
    P2S_CHECK(R >= 2 && R <= 1024, "grid resolution out of range");
    const int64_t V = (int64_t)R * R * R, E = 3 * V;
    const int64_t C = (int64_t)(R - 1) * (R - 1) * (R - 1);
    P2S_CHECK(E < (1ll << 31), "volume too large for 32-bit edge ids");
    size_t cub1 = 0, cub2 = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, cub1, (uint8_t*)nullptr, (int32_t*)nullptr, (int)E, st);
    cub::DeviceScan::ExclusiveSum(nullptr, cub2, (uint8_t*)nullptr, (int32_t*)nullptr, (int)C, st);
    size_t cub_bytes = cub1 > cub2 ? cub1 : cub2;
    auto al = [](size_t x) { return (x + 255) / 256 * 256; };
    size_t off_flags = 256, off_vid = off_flags + al(E), off_cnt = off_vid + al(E * 4), off_offs = off_cnt + al(C),
           off_cub = off_offs + al(C * 4);
    uint8_t* base = (uint8_t*)device_ctx().mc_ws.get(off_cub + cub_bytes);
    double* acc = (double*)base;
    uint8_t* flags = base + off_flags;
    int32_t* vid = (int32_t*)(base + off_vid);
    uint8_t* counts = base + off_cnt;
    int32_t* offs = (int32_t*)(base + off_offs);

    P2S_LAUNCH(mc_edge_flags_kernel, (unsigned)cdiv(V, 256), 256, 0, st, vol, R, level, flags);
    P2S_CUDA(cub::DeviceScan::ExclusiveSum(base + off_cub, cub_bytes, flags, vid, (int)E, st));
    P2S_LAUNCH(mc_cell_count_kernel, (unsigned)cdiv(C, 256), 256, 0, st, vol, R, level, counts);
    P2S_CUDA(cub::DeviceScan::ExclusiveSum(base + off_cub, cub_bytes, counts, offs, (int)C, st));
    g_launches.fetch_add(4, std::memory_order_relaxed);  // cub: 2 kernels per scan
    int32_t last_vid = 0, last_off = 0;
    uint8_t last_flag = 0, last_cnt = 0;
    P2S_CUDA(cudaMemcpyAsync(&last_vid, vid + (E - 1), 4, cudaMemcpyDeviceToHost, st));
    P2S_CUDA(cudaMemcpyAsync(&last_flag, flags + (E - 1), 1, cudaMemcpyDeviceToHost, st));
    P2S_CUDA(cudaMemcpyAsync(&last_off, offs + (C - 1), 4, cudaMemcpyDeviceToHost, st));
    P2S_CUDA(cudaMemcpyAsync(&last_cnt, counts + (C - 1), 1, cudaMemcpyDeviceToHost, st));
    P2S_CUDA(cudaStreamSynchronize(st));
    const int64_t nv = (int64_t)last_vid + last_flag, nf = (int64_t)last_off + last_cnt;
    *nverts_host = nv;
    *nfaces_host = nf;
    if (!verts || !faces || vcap < nv || fcap < nf) return;   // counting call (or capacity too small): nothing emitted
    if (nv == 0 || nf == 0) return;
    P2S_LAUNCH(mc_emit_verts_kernel, (unsigned)cdiv(E, 256), 256, 0, st, vol, R, level, flags, vid, verts, vcap);
    P2S_LAUNCH(mc_emit_faces_kernel, (unsigned)cdiv(C, 256), 256, 0, st, vol, R, level, counts, offs, vid, faces, fcap);
    P2S_CUDA(cudaMemsetAsync(acc, 0, sizeof(double), st));
    P2S_LAUNCH(mc_signed_volume_kernel, (unsigned)cdiv(nf, 256), 256, 0, st, verts, faces, nf, acc);
    P2S_LAUNCH(mc_flip_kernel, (unsigned)cdiv(nf, 256), 256, 0, st, faces, nf, acc);
}

}  // namespace p2s
