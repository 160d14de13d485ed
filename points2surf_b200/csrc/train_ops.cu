// K10: primitives of the training step (SURVEY.md section 8a row a14: compute_loss + backward + SGD,
// source/points_to_surf_train.py:441-461,537-563; train-mode BatchNorm of source/points_to_surf_model.py).
// Activations are row-major [rows, C] fp32 (rows = queries x points, channels contiguous), the layout of the fp32
// inference path; the host side (points2surf_b200/train.py) sequences these ops layer by layer like the reference's
// autograd graph.  fp32 FMA throughout (the reference trains in fp32); GEMMs:
//   forward  Z = X W^T            -> launch_gemm_nt (net_fp32.cu)
//   dX = dZ W = dZ (W^T)^T        -> launch_gemm_nt on the transposed weight (transpose_kernel)
//   dW = dZ^T X                   -> gemm_tn_kernel below (contraction over the rows, split over CTAs, atomics)
// Column reductions (BatchNorm statistics, bias / gamma / beta gradients) accumulate in f64.
#include "model.cuh"

namespace p2s {

namespace {

// ---------------------------------------------------------------- C[z][n][k] (+)= sum_m A[z][m][n] * B[z][m][k]
// 128 (n) x 64 (k) output tile, 256 threads, 8 x 4 outputs per thread, 16 rows of m per shared-memory step.
constexpr int kTnN = 128, kTnK = 64, kTnM = 16;

__global__ void __launch_bounds__(256)
gemm_tn_kernel(const float* __restrict__ A, int64_t a_stride_z, int lda, const float* __restrict__ B,
               int64_t b_stride_z, int ldb, float* __restrict__ C, int64_t c_stride_z, int ldc, int M, int N, int K,
               int splits, int rows_per_split, int use_atomics) {
    __shared__ float As[kTnM][kTnN];
    __shared__ float Bs[kTnM][kTnK];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;   // tx -> k (4 each), ty -> n (8 each)
    const int n0 = blockIdx.x * kTnN, k0 = blockIdx.y * kTnK;
    const int z = blockIdx.z / splits, sp = blockIdx.z % splits;
    const float* Az = A + (int64_t)z * a_stride_z;
    const float* Bz = B + (int64_t)z * b_stride_z;
    const int m_begin = sp * rows_per_split, m_end = min(M, m_begin + rows_per_split);
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int m0 = m_begin; m0 < m_end; m0 += kTnM) {
        // A tile: 16 rows x 128 cols = 2048 floats, 8 per thread; B tile: 16 x 64 = 1024, 4 per thread
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int e = tid + i * 256, r = e >> 7, c = e & 127;
            As[r][c] = (m0 + r < m_end && n0 + c < N) ? Az[(int64_t)(m0 + r) * lda + n0 + c] : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = tid + i * 256, r = e >> 6, c = e & 63;
            Bs[r][c] = (m0 + r < m_end && k0 + c < K) ? Bz[(int64_t)(m0 + r) * ldb + k0 + c] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < kTnM; ++r) {
            float a[8], b[4];
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = As[r][ty + 16 * i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[r][tx + 16 * j];
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
    float* Cz = C + (int64_t)z * c_stride_z;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int n = n0 + ty + 16 * i;
        if (n >= N) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + tx + 16 * j;
            if (k >= K) continue;
            if (use_atomics) atomicAdd(Cz + (int64_t)n * ldc + k, acc[i][j]);
            else Cz[(int64_t)n * ldc + k] = acc[i][j];
        }
    }
}

// ---------------------------------------------------------------- out[z][c][r] = in[z][r][c]
__global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int rows, int cols) {
    __shared__ float t[32][33];
    const int z = blockIdx.z;
    const float* iz = in + (int64_t)z * rows * cols;
    float* oz = out + (int64_t)z * rows * cols;
    int c = blockIdx.x * 32 + threadIdx.x, r0 = blockIdx.y * 32;
    for (int j = threadIdx.y; j < 32; j += 8)
        if (r0 + j < rows && c < cols) t[j][threadIdx.x] = iz[(int64_t)(r0 + j) * cols + c];
    __syncthreads();
    int r = r0 + threadIdx.x, c0 = blockIdx.x * 32;
    for (int j = threadIdx.y; j < 32; j += 8)
        if (c0 + j < cols && r < rows) oz[(int64_t)(c0 + j) * rows + r] = t[threadIdx.x][j];
}

// ---------------------------------------------------------------- column reductions over [M, C] (f64 accumulators)
// MODE 0: s1 += sum x, s2 += sum x*x                      (BatchNorm statistics)
// MODE 1: s1 += sum g, s2 += sum g * xhat, g = dy * (y > 0 if y), xhat = (z - mean) * invstd   (BatchNorm backward)
// MODE 2: s1 += sum x                                      (bias gradient)
template <int MODE>
__global__ void __launch_bounds__(256)
col_reduce_kernel(const float* __restrict__ x, const float* __restrict__ z, const float* __restrict__ y,
                  const float* __restrict__ mean, const float* __restrict__ invstd, int64_t M, int C,
                  int64_t rows_per_block, double* __restrict__ s1, double* __restrict__ s2) {
    const int c = blockIdx.x * 32 + threadIdx.x;
    const int64_t r_begin = (int64_t)blockIdx.y * rows_per_block, r_end = min(M, r_begin + rows_per_block);
    float a1 = 0.f, a2 = 0.f;
    if (c < C) {
        float mu = 0.f, is = 0.f;
        if (MODE == 1) { mu = mean[c]; is = invstd[c]; }
#pragma unroll 4
        for (int64_t r = r_begin + threadIdx.y; r < r_end; r += 8) {
            const int64_t e = r * C + c;
            float v = x[e];
            if (MODE == 0) { a1 += v; a2 = fmaf(v, v, a2); }
            else if (MODE == 1) {
                if (y && !(y[e] > 0.f)) v = 0.f;
                a1 += v;
                a2 = fmaf(v, (z[e] - mu) * is, a2);
            } else a1 += v;
        }
    }
    __shared__ float r1[8][32], r2[8][32];
    r1[threadIdx.y][threadIdx.x] = a1;
    r2[threadIdx.y][threadIdx.x] = a2;
    __syncthreads();
    if (threadIdx.y == 0 && c < C) {
        double d1 = 0.0, d2 = 0.0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { d1 += (double)r1[j][threadIdx.x]; d2 += (double)r2[j][threadIdx.x]; }
        atomicAdd(s1 + c, d1);
        if (MODE != 2) atomicAdd(s2 + c, d2);
    }
}

// mean / invstd from the sums; running statistics like torch.nn.BatchNorm1d (momentum 0.1, unbiased running var)
__global__ void bn_finalize_kernel(const double* __restrict__ s1, const double* __restrict__ s2, int64_t M, int C,
                                   float eps, float momentum, float* __restrict__ mean, float* __restrict__ invstd,
                                   float* __restrict__ running_mean, float* __restrict__ running_var) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double mu = s1[c] / (double)M;
    double var = s2[c] / (double)M - mu * mu;
    if (var < 0.0) var = 0.0;
    mean[c] = (float)mu;
    invstd[c] = (float)(1.0 / sqrt(var + (double)eps));
    if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mu;
    if (running_var) {
        double unbiased = M > 1 ? var * (double)M / (double)(M - 1) : var;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
    }
}

// Row-tiled element-wise kernels: blockDim = (tx, 256 / tx) with tx consecutive channels per row, grid = (channel
// blocks, row chunks); every thread keeps the parameters of its channel in registers and walks down the rows, so the
// accesses are coalesced and there is no per-element integer division.
// y = act(gamma * (z - mean) * invstd + beta)
__global__ void __launch_bounds__(256)
bn_apply_kernel(const float* __restrict__ z, int64_t M, int C, int64_t rows_per_block, const float* __restrict__ mean,
                const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ beta,
                int relu, float* __restrict__ y) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float a = gamma[c] * invstd[c], mu = mean[c], bt = beta[c];
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_block, r1 = min(M, r0 + rows_per_block);
#pragma unroll 4
    for (int64_t r = r0 + threadIdx.y; r < r1; r += blockDim.y) {
        const float v = fmaf(a, z[r * C + c] - mu, bt);
        y[r * C + c] = relu ? fmaxf(v, 0.f) : v;
    }
}

// dz = gamma * invstd * (g - s1/M - xhat * s2/M), g = dy masked by the ReLU
__global__ void __launch_bounds__(256)
bn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ z, const float* __restrict__ y, int64_t M,
                    int C, int64_t rows_per_block, const float* __restrict__ mean, const float* __restrict__ invstd,
                    const float* __restrict__ gamma, const double* __restrict__ s1, const double* __restrict__ s2,
                    float* __restrict__ dz) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float is = invstd[c], mu = mean[c], gi = gamma[c] * is;
    const float m1 = (float)(s1[c] / (double)M), m2 = (float)(s2[c] / (double)M);
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_block, r1 = min(M, r0 + rows_per_block);
#pragma unroll 4
    for (int64_t r = r0 + threadIdx.y; r < r1; r += blockDim.y) {
        const int64_t e = r * C + c;
        float g = dy[e];
        if (y && !(y[e] > 0.f)) g = 0.f;
        const float xhat = (z[e] - mu) * is;
        dz[e] = gi * (g - m1 - xhat * m2);
    }
}

// ---- BatchNorm (+ReLU) fused with the max over the points of each query (the conv3 layers: the 1024-channel
// activations are never materialised after the BatchNorm, and the backward never builds the sparse dy)
__global__ void bn_maxpool_fwd_kernel(const float* __restrict__ z, int64_t B, int npts, int C,
                                      const float* __restrict__ mean, const float* __restrict__ invstd,
                                      const float* __restrict__ gamma, const float* __restrict__ beta, int relu,
                                      float* __restrict__ out, int32_t* __restrict__ arg) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t b = blockIdx.y;
    if (c >= C) return;
    const float a = gamma[c] * invstd[c], mu = mean[c], bt = beta[c];
    const float* p = z + b * npts * (int64_t)C + c;
    float best = -INFINITY;
    int bi = 0;
    for (int i = 0; i < npts; ++i) {
        float v = fmaf(a, p[(int64_t)i * C] - mu, bt);
        if (relu) v = fmaxf(v, 0.f);
        if (v > best || i == 0) { best = v; bi = i; }   // first maximum, like torch.max / MaxPool1d
    }
    out[b * C + c] = best;
    arg[b * C + c] = bi;
}

// s1[c] += sum_b g, s2[c] += sum_b g * xhat(b, arg, c); g = dout * (out > 0 if relu)
__global__ void __launch_bounds__(256)
bn_maxpool_bwd_reduce_kernel(const float* __restrict__ dout, const int32_t* __restrict__ arg,
                             const float* __restrict__ out, const float* __restrict__ z,
                             const float* __restrict__ mean, const float* __restrict__ invstd, int64_t B, int npts,
                             int C, int relu, int64_t rows_per_block, double* __restrict__ s1, double* __restrict__ s2) {
    const int c = blockIdx.x * 32 + threadIdx.x;
    const int64_t b0 = (int64_t)blockIdx.y * rows_per_block, b1 = min(B, b0 + rows_per_block);
    float a1 = 0.f, a2 = 0.f;
    if (c < C) {
        const float mu = mean[c], is = invstd[c];
        for (int64_t b = b0 + threadIdx.y; b < b1; b += 8) {
            float g = dout[b * C + c];
            if (relu && !(out[b * C + c] > 0.f)) g = 0.f;
            const float xhat = (z[(b * npts + arg[b * C + c]) * (int64_t)C + c] - mu) * is;
            a1 += g;
            a2 = fmaf(g, xhat, a2);
        }
    }
    __shared__ float r1[8][32], r2[8][32];
    r1[threadIdx.y][threadIdx.x] = a1;
    r2[threadIdx.y][threadIdx.x] = a2;
    __syncthreads();
    if (threadIdx.y == 0 && c < C) {
        double d1 = 0.0, d2 = 0.0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { d1 += (double)r1[j][threadIdx.x]; d2 += (double)r2[j][threadIdx.x]; }
        atomicAdd(s1 + c, d1);
        atomicAdd(s2 + c, d2);
    }
}

// grid (channel blocks, point chunks of 32, B)
__global__ void __launch_bounds__(256)
bn_maxpool_bwd_apply_kernel(const float* __restrict__ dout, const int32_t* __restrict__ arg,
                            const float* __restrict__ out, const float* __restrict__ z, const float* __restrict__ mean,
                            const float* __restrict__ invstd, const float* __restrict__ gamma,
                            const double* __restrict__ s1, const double* __restrict__ s2, int64_t B, int npts, int C,
                            int relu, float* __restrict__ dz) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const int64_t b = blockIdx.z;
    const int64_t M = B * npts;
    const float is = invstd[c], mu = mean[c], gi = gamma[c] * is;
    const float m1 = (float)(s1[c] / (double)M), m2 = (float)(s2[c] / (double)M);
    const int a = arg[b * C + c];
    float g = dout[b * C + c];
    if (relu && !(out[b * C + c] > 0.f)) g = 0.f;
    const int p0 = blockIdx.y * 32, p1 = min(npts, p0 + 32);
    const int64_t base = (b * npts + p0) * (int64_t)C + c;
    const float* zp = z + base;
    float* dp = dz + base;
#pragma unroll 4
    for (int p = p0; p < p1; ++p, zp += C, dp += C) {
        const float xhat = (*zp - mu) * is;
        *dp = gi * ((p == a ? g : 0.f) - m1 - xhat * m2);
    }
}

// ---------------------------------------------------------------- max over the points of each query, with argmax
__global__ void maxpool_fwd_kernel(const float* __restrict__ y, int64_t B, int npts, int C, float* __restrict__ out,
                                   int32_t* __restrict__ arg) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B * C) return;
    int64_t b = e / C;
    int c = (int)(e % C);
    const float* p = y + b * npts * (int64_t)C + c;
    float best = p[0];
    int bi = 0;
    for (int i = 1; i < npts; ++i) {
        float v = p[(int64_t)i * C];
        if (v > best || (v != v && !(best != best))) { best = v; bi = i; }   // first maximum; NaN propagates like torch
    }
    out[e] = best;
    arg[e] = bi;
}

// grid (ceil(C / 256), point chunks, B): no integer division per element
__global__ void maxpool_bwd_kernel(const float* __restrict__ dout, const int32_t* __restrict__ arg, int64_t B, int npts,
                                   int C, float* __restrict__ dy) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const int64_t b = blockIdx.z;
    const int a = arg[b * C + c];
    const float g = dout[b * C + c];
    const int p0 = blockIdx.y * 32, p1 = min(npts, p0 + 32);
    float* d = dy + (b * npts + p0) * (int64_t)C + c;
    for (int p = p0; p < p1; ++p, d += C) *d = (p == a) ? g : 0.f;
}

// ---------------------------------------------------------------- loss (sdf_nn.calc_loss_magnitude / calc_loss_sign)
// loss_out[0] = w_mag * mean((tanh|p0| - tanh|t / r|)^2), loss_out[1] = w_sign * mean(BCEWithLogits(p1, s));
// dpred = d(loss0 + loss1)/dpred.  One block.
__global__ void __launch_bounds__(256)
loss_kernel(const float* __restrict__ pred, const float* __restrict__ target_mag, const float* __restrict__ radius,
            const float* __restrict__ target_sign, int64_t B, float w_mag, float w_sign, int fixed_radius,
            double* __restrict__ loss_out, float* __restrict__ dpred) {
    double l0 = 0.0, l1 = 0.0;
    const float invB = 1.f / (float)B;
    for (int64_t i = threadIdx.x; i < B; i += blockDim.x) {
        float p0 = pred[2 * i], p1 = pred[2 * i + 1];
        float t = target_mag[i];
        if (!fixed_radius) t = t / radius[i];
        float a = tanhf(fabsf(p0)), b = tanhf(fabsf(t));
        float d = a - b;
        l0 += (double)(d * d);
        float sg = p0 > 0.f ? 1.f : (p0 < 0.f ? -1.f : 0.f);
        float s = target_sign[i];
        float ax = fabsf(p1);
        l1 += (double)(fmaxf(p1, 0.f) - p1 * s + log1pf(expf(-ax)));
        if (dpred) {
            dpred[2 * i] = w_mag * 2.f * d * invB * (1.f - a * a) * sg;
            float sig = 1.f / (1.f + expf(-p1));
            dpred[2 * i + 1] = w_sign * (sig - s) * invB;
        }
    }
    __shared__ double r0[256], r1[256];
    r0[threadIdx.x] = l0; r1[threadIdx.x] = l1;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) { r0[threadIdx.x] += r0[threadIdx.x + o]; r1[threadIdx.x] += r1[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        loss_out[0] = (double)w_mag * r0[0] / (double)B;
        loss_out[1] = (double)w_sign * r1[0] / (double)B;
    }
}

// ---------------------------------------------------------------- quaternion -> rotation, backward
// R = I + s * A(q), s = 2 / |q|^2 (utils.batch_quat_to_rotmat, source/base/utils.py:13-46; q is not normalised);
// like the forward kernel, q4 is the raw fc3 output and q = q4 + (1,0,0,0) (points_to_surf_model.py:124-126)
__global__ void quat_to_rot_bwd_kernel(const float* __restrict__ q4, const float* __restrict__ dR, int64_t B,
                                       float* __restrict__ dq) {
    int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float q0 = q4[4 * b] + 1.f, q1 = q4[4 * b + 1], q2 = q4[4 * b + 2], q3 = q4[4 * b + 3];
    const float* g = dR + 9 * b;
    const float n2 = q0 * q0 + q1 * q1 + q2 * q2 + q3 * q3;
    const float s = 2.f / n2;
    // A_ij (row-major)
    const float A[9] = {-(q2 * q2 + q3 * q3), q1 * q2 - q3 * q0, q1 * q3 + q2 * q0,
                        q1 * q2 + q3 * q0, -(q1 * q1 + q3 * q3), q2 * q3 - q1 * q0,
                        q1 * q3 - q2 * q0, q2 * q3 + q1 * q0, -(q1 * q1 + q2 * q2)};
    float gA = 0.f;
#pragma unroll
    for (int i = 0; i < 9; ++i) gA += g[i] * A[i];
    // sum_ij g_ij dA_ij/dq_k
    const float d0 = -q3 * g[1] + q2 * g[2] + q3 * g[3] - q1 * g[5] - q2 * g[6] + q1 * g[7];
    const float d1 = q2 * g[1] + q3 * g[2] + q2 * g[3] - 2.f * q1 * g[4] - q0 * g[5] + q3 * g[6] + q0 * g[7] - 2.f * q1 * g[8];
    const float d2 = -2.f * q2 * g[0] + q1 * g[1] + q0 * g[2] + q1 * g[3] + q3 * g[5] - q0 * g[6] + q3 * g[7] - 2.f * q2 * g[8];
    const float d3 = -2.f * q3 * g[0] - q0 * g[1] + q1 * g[2] + q0 * g[3] - 2.f * q3 * g[4] + q2 * g[5] + q1 * g[6] + q2 * g[7];
    const float ds = -s * s;   // ds/dq_k = -s^2 q_k
    dq[4 * b + 0] = ds * q0 * gA + s * d0;
    dq[4 * b + 1] = ds * q1 * gA + s * d1;
    dq[4 * b + 2] = ds * q2 * gA + s * d2;
    dq[4 * b + 3] = ds * q3 * gA + s * d3;
}

// x[b][c] += v[c] for the identity offsets (quaternion (1,0,0,0); flattened I_64)
__global__ void add_row_kernel(float* __restrict__ x, const float* __restrict__ v, int64_t B, int C) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < B * C) x[e] += v[e % C];
}

// torch.optim.SGD (momentum, dampening 0, no Nesterov, no weight decay): buf = g on the first step, else mu*buf + g
__global__ void sgd_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ buf, int64_t n,
                           float lr, float momentum, int first) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float b = first ? g[i] : fmaf(momentum, buf[i], g[i]);
    buf[i] = b;
    p[i] = fmaf(-lr, b, p[i]);
}

// y += a * x
__global__ void axpy_kernel(float* __restrict__ y, const float* __restrict__ x, float a, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = fmaf(a, x[i], y[i]);
}

// out[b][p][:] = in[b][p][:] - q[b][:]   (points_to_surf_model.py:303)
__global__ void center_kernel(const float* __restrict__ in, const float* __restrict__ q, int64_t B, int npts,
                              float* __restrict__ out) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B * npts * 3) return;
    int64_t b = e / ((int64_t)npts * 3);
    out[e] = in[e] - q[b * 3 + e % 3];
}

}  // namespace

// ---------------------------------------------------------------------------------------------- host launchers
void op_gemm_tn(const float* A, int64_t a_stride_z, int lda, const float* B, int64_t b_stride_z, int ldb, float* C,
                int64_t c_stride_z, int ldc, int M, int N, int K, int batch, bool accumulate, cudaStream_t st) {
    if (N <= 0 || K <= 0 || batch <= 0) return;
    if (batch == 1 && M > 0 && gemm_tn_tc_ok(A, lda, B, ldb, M, N, K)) {
        // large weight gradients: split-precision tensor-core kernel (gemm_tn_tc.cu), partial tiles added atomically
        if (!accumulate) P2S_CUDA(cudaMemset2DAsync(C, sizeof(float) * ldc, 0, sizeof(float) * K, N, st));
        launch_gemm_tn_tc(A, lda, B, ldb, C, ldc, M, N, K, st);
        return;
    }
    const int tiles = (int)(cdiv(N, kTnN) * cdiv(K, kTnK)) * batch;
    int splits = 1;
    if (M > 2048) {
        splits = (int)std::min<int64_t>(cdiv(M, 1024), std::max<int64_t>(1, cdiv(4 * (int64_t)device_ctx().sm_count, tiles)));
    }
    int rows = (int)(cdiv(cdiv(M, splits), kTnM) * kTnM);
    splits = (int)cdiv(M, rows);
    if (splits < 1) splits = 1;
    P2S_CHECK((int64_t)batch * splits <= 65535, "gemm_tn: grid.z too large");
    const bool atomics = accumulate || splits > 1;
    if (atomics && !accumulate) {
        if (c_stride_z == (int64_t)N * ldc && ldc == K) {
            P2S_CUDA(cudaMemsetAsync(C, 0, sizeof(float) * (size_t)batch * N * K, st));
        } else {
            for (int z = 0; z < batch; ++z)
                P2S_CUDA(cudaMemset2DAsync(C + z * c_stride_z, sizeof(float) * ldc, 0, sizeof(float) * K, N, st));
        }
    }
    dim3 g((unsigned)cdiv(N, kTnN), (unsigned)cdiv(K, kTnK), (unsigned)(batch * splits));
    P2S_LAUNCH(gemm_tn_kernel, g, 256, 0, st, A, a_stride_z, lda, B, b_stride_z, ldb, C, c_stride_z, ldc, M, N, K,
               splits, rows, atomics ? 1 : 0);
}

void op_transpose(const float* in, float* out, int rows, int cols, int batch, cudaStream_t st) {
    if (rows <= 0 || cols <= 0 || batch <= 0) return;
    dim3 g((unsigned)cdiv(cols, 32), (unsigned)cdiv(rows, 32), (unsigned)batch);
    P2S_LAUNCH(transpose_kernel, g, dim3(32, 8), 0, st, in, out, rows, cols);
}

static void col_reduce_grid(int64_t M, int C, dim3& g, int64_t& rows_per_block) {
    int64_t cx = cdiv(C, 32);
    int64_t want = std::max<int64_t>(1, cdiv(8 * (int64_t)device_ctx().sm_count, cx));
    rows_per_block = std::max<int64_t>(64, cdiv(M, want));
    rows_per_block = std::min<int64_t>(rows_per_block, 4096);
    rows_per_block = std::max<int64_t>(rows_per_block, cdiv(M, 65535));
    g = dim3((unsigned)cx, (unsigned)cdiv(M, rows_per_block));
}

// blockDim (tx, 256/tx), grid (channel blocks, row chunks) for the row-tiled element-wise kernels
static void rowwise_grid(int64_t M, int C, dim3& blk, dim3& g, int64_t& rows_per_block) {
    const int tx = C >= 128 ? 128 : (C >= 64 ? 64 : 32);
    blk = dim3(tx, 256 / tx);
    const int64_t cx = cdiv(C, tx);
    const int64_t want = std::max<int64_t>(1, cdiv(16 * (int64_t)device_ctx().sm_count, cx));
    rows_per_block = std::max<int64_t>(4 * blk.y, cdiv(M, want));
    rows_per_block = std::max<int64_t>(rows_per_block, cdiv(M, 65535));
    g = dim3((unsigned)cx, (unsigned)cdiv(M, rows_per_block));
}

// s1, s2: f64 [C], zeroed here
void op_col_stats(const float* x, int64_t M, int C, double* s1, double* s2, cudaStream_t st) {
    P2S_CUDA(cudaMemsetAsync(s1, 0, sizeof(double) * C, st));
    P2S_CUDA(cudaMemsetAsync(s2, 0, sizeof(double) * C, st));
    if (M <= 0) return;
    dim3 g; int64_t rpb;
    col_reduce_grid(M, C, g, rpb);
    P2S_LAUNCH(col_reduce_kernel<0>, g, dim3(32, 8), 0, st, x, nullptr, nullptr, nullptr, nullptr, M, C, rpb, s1, s2);
}

void op_col_sum(const float* x, int64_t M, int C, double* s1, cudaStream_t st) {
    P2S_CUDA(cudaMemsetAsync(s1, 0, sizeof(double) * C, st));
    if (M <= 0) return;
    dim3 g; int64_t rpb;
    col_reduce_grid(M, C, g, rpb);
    P2S_LAUNCH(col_reduce_kernel<2>, g, dim3(32, 8), 0, st, x, nullptr, nullptr, nullptr, nullptr, M, C, rpb, s1, (double*)nullptr);
}

void op_bn_finalize(const double* s1, const double* s2, int64_t M, int C, float eps, float momentum, float* mean,
                    float* invstd, float* running_mean, float* running_var, cudaStream_t st) {
    P2S_LAUNCH(bn_finalize_kernel, (unsigned)cdiv(C, 128), 128, 0, st, s1, s2, M, C, eps, momentum, mean, invstd,
               running_mean, running_var);
}

void op_bn_apply(const float* z, int64_t M, int C, const float* mean, const float* invstd, const float* gamma,
                 const float* beta, bool relu, float* y, cudaStream_t st) {
    if (M <= 0) return;
    dim3 blk, g; int64_t rpb;
    rowwise_grid(M, C, blk, g, rpb);
    P2S_LAUNCH(bn_apply_kernel, g, blk, 0, st, z, M, C, rpb, mean, invstd, gamma, beta, relu ? 1 : 0, y);
}

// dz from dy; s1 (= dbeta) and s2 (= dgamma) f64 [C] are outputs
void op_bn_backward(const float* dy, const float* z, const float* y_or_null, int64_t M, int C, const float* mean,
                    const float* invstd, const float* gamma, double* s1, double* s2, float* dz, cudaStream_t st) {
    P2S_CUDA(cudaMemsetAsync(s1, 0, sizeof(double) * C, st));
    P2S_CUDA(cudaMemsetAsync(s2, 0, sizeof(double) * C, st));
    if (M <= 0) return;
    dim3 g; int64_t rpb;
    col_reduce_grid(M, C, g, rpb);
    P2S_LAUNCH(col_reduce_kernel<1>, g, dim3(32, 8), 0, st, dy, z, y_or_null, mean, invstd, M, C, rpb, s1, s2);
    dim3 blk, g2; int64_t rpb2;
    rowwise_grid(M, C, blk, g2, rpb2);
    P2S_LAUNCH(bn_bwd_apply_kernel, g2, blk, 0, st, dy, z, y_or_null, M, C, rpb2, mean, invstd, gamma, s1, s2, dz);
}

void op_maxpool_fwd(const float* y, int64_t B, int npts, int C, float* out, int32_t* arg, cudaStream_t st) {
    if (B <= 0) return;
    P2S_LAUNCH(maxpool_fwd_kernel, (unsigned)cdiv(B * C, 256), 256, 0, st, y, B, npts, C, out, arg);
}

void op_maxpool_bwd(const float* dout, const int32_t* arg, int64_t B, int npts, int C, float* dy, cudaStream_t st) {
    if (B <= 0) return;
    P2S_CHECK(B <= 65535, "maxpool_bwd: batch too large for grid.z");
    P2S_LAUNCH(maxpool_bwd_kernel, dim3((unsigned)cdiv(C, 256), (unsigned)cdiv(npts, 32), (unsigned)B), 256, 0, st, dout, arg, B, npts, C, dy);
}

void op_loss(const float* pred, const float* target_mag, const float* radius, const float* target_sign, int64_t B,
             float w_mag, float w_sign, bool fixed_radius, double* loss_out, float* dpred, cudaStream_t st) {
    P2S_LAUNCH(loss_kernel, 1, 256, 0, st, pred, target_mag, radius, target_sign, B, w_mag, w_sign,
               fixed_radius ? 1 : 0, loss_out, dpred);
}

void op_quat_to_rot_bwd(const float* q4, const float* dR, int64_t B, float* dq, cudaStream_t st) {
    if (B <= 0) return;
    P2S_LAUNCH(quat_to_rot_bwd_kernel, (unsigned)cdiv(B, 128), 128, 0, st, q4, dR, B, dq);
}

void op_add_row(float* x, const float* v, int64_t B, int C, cudaStream_t st) {
    if (B <= 0) return;
    P2S_LAUNCH(add_row_kernel, (unsigned)cdiv(B * C, 256), 256, 0, st, x, v, B, C);
}

void op_sgd(float* p, const float* g, float* buf, int64_t n, float lr, float momentum, bool first, cudaStream_t st) {
    if (n <= 0) return;
    P2S_LAUNCH(sgd_kernel, (unsigned)cdiv(n, 256), 256, 0, st, p, g, buf, n, lr, momentum, first ? 1 : 0);
}

void op_axpy(float* y, const float* x, float a, int64_t n, cudaStream_t st) {
    if (n <= 0) return;
    P2S_LAUNCH(axpy_kernel, (unsigned)cdiv(n, 256), 256, 0, st, y, x, a, n);
}

void op_center(const float* in, const float* q, int64_t B, int npts, float* out, cudaStream_t st) {
    if (B <= 0) return;
    P2S_LAUNCH(center_kernel, (unsigned)cdiv(B * npts * 3, 256), 256, 0, st, in, q, B, npts, out);
}

// BatchNorm(train) (+ReLU) + max over the npts points of each query, without materialising the normalised tensor
void op_bn_maxpool_fwd(const float* z, int64_t B, int npts, int C, const float* mean, const float* invstd,
                       const float* gamma, const float* beta, bool relu, float* out, int32_t* arg, cudaStream_t st) {
    if (B <= 0) return;
    P2S_CHECK(B <= 65535, "bn_maxpool_fwd: batch too large for grid.y");
    P2S_LAUNCH(bn_maxpool_fwd_kernel, dim3((unsigned)cdiv(C, 128), (unsigned)B), 128, 0, st, z, B, npts, C, mean, invstd,
               gamma, beta, relu ? 1 : 0, out, arg);
}

// backward of the above: dout [B,C] -> dz [B*npts, C]; s1 = dbeta, s2 = dgamma (f64 [C])
void op_bn_maxpool_bwd(const float* dout, const int32_t* arg, const float* out, const float* z, int64_t B, int npts, int C,
                       const float* mean, const float* invstd, const float* gamma, bool relu, double* s1, double* s2,
                       float* dz, cudaStream_t st) {
    P2S_CUDA(cudaMemsetAsync(s1, 0, sizeof(double) * C, st));
    P2S_CUDA(cudaMemsetAsync(s2, 0, sizeof(double) * C, st));
    if (B <= 0) return;
    P2S_CHECK(B <= 65535, "bn_maxpool_bwd: batch too large for grid.z");
    const int64_t rpb = std::max<int64_t>(8, cdiv(B, 64));
    P2S_LAUNCH(bn_maxpool_bwd_reduce_kernel, dim3((unsigned)cdiv(C, 32), (unsigned)cdiv(B, rpb)), dim3(32, 8), 0, st, dout, arg,
               out, z, mean, invstd, B, npts, C, relu ? 1 : 0, rpb, s1, s2);
    const int tx = C >= 128 ? 128 : (C >= 64 ? 64 : 32);
    P2S_LAUNCH(bn_maxpool_bwd_apply_kernel, dim3((unsigned)cdiv(C, tx), (unsigned)cdiv(npts, 32), (unsigned)B), tx, 0, st, dout,
               arg, out, z, mean, invstd, gamma, s1, s2, B, npts, C, relu ? 1 : 0, dz);
}

}  // namespace p2s
