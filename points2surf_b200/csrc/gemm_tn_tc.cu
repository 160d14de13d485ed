// Tensor-core weight-gradient GEMM of the training step (SURVEY.md section 8a row a14):
//     C[N][K] += sum_m A[m][n] * B[m][k]          (dW = dZ^T X; A = dZ [M,N], B = X [M,K], both fp32 row-major)
// The contraction runs over the rows m (up to 1.3 M of them), so both operands are "transposed" with respect to the
// K-major layout tcgen05 wants.  The producers do the transposition on the fly: a warp reads whole rows (coalesced),
// every thread ends up with an 8 (m) x 4 (n) block and writes four 16-byte core-matrix rows of the K-major operand
// image (k = m), split into fp16 hi / lo parts; three MMAs per k-step (lo*hi + hi*lo + hi*hi) keep fp32-level accuracy
// (same scheme as fc_tc.cu).  One CTA = one 128 (n) x 128 (k) output tile x one slice of the rows; partial tiles are
// added to C with fp32 atomics (C is zeroed or holds the running gradient).
//   warps 0-3   A-operand producers (dZ tile 32 rows x 128 n), afterwards the epilogue (TMEM -> atomicAdd)
//   warps 4-7   B-operand producers (X tile 32 rows x 128 k)
//   warp  8     tcgen05.mma issue (elect-one), commits free the stage
// HBM-bound by design: every dZ element is read once per k-tile (K <= 128: once), X once per n-tile (L2 hits).
#include "model.cuh"
#include "tc_ptx.cuh"

namespace p2s {

using namespace ptx;

namespace {

constexpr int kStages = 3;
constexpr int kBM = 32;                        // rows of m per stage (two MMA k-steps of 16)
constexpr uint32_t kHalf = 128 * kBM * 2;      // one 128 x 32 fp16 operand image: 8 KB (K-major, LBO 128, SBO 512)
constexpr uint32_t kStageOp = 2 * kHalf;       // hi + lo
constexpr uint32_t kSmem = kStages * 2 * kStageOp + 256;

struct Bars {
    uint64_t full[kStages], empty[kStages], d_full;
    uint32_t tmem_base;
};

// Fill one operand image (hi | lo) from src[m][c0 .. c0+127] (row stride ld), rows m0 .. m0+31 (< m_end), cols < ncols.
// t = thread index within the 128 producers of this operand.
__device__ __forceinline__ void fill_operand(uint8_t* dst, const float* __restrict__ src, int ld, int64_t m0, int64_t m_end,
                                             int c0, int ncols, int t) {
    const int col = c0 + (t & 31) * 4;        // 4 consecutive n (or k)
    const int rg = t >> 5;                    // row group: rows rg*8 .. rg*8+7  == k-chunk rg of the operand
    float4 v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int64_t m = m0 + rg * 8 + j;
        v[j] = (m < m_end && col < ncols) ? *reinterpret_cast<const float4*>(src + m * ld + col) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const int lane = t & 31;
#pragma unroll
    for (int ii = 0; ii < 4; ++ii) {
        const int i = (ii + (lane >> 1)) & 3;                       // rotate to spread the shared-memory banks
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = i == 0 ? v[j].x : (i == 1 ? v[j].y : (i == 2 ? v[j].z : v[j].w));
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            __half2 h = __floats2half2_rn(x[2 * e], x[2 * e + 1]);
            float2 hf = __half22float2(h);
            __half2 l = __floats2half2_rn(x[2 * e] - hf.x, x[2 * e + 1] - hf.y);
            hi[e] = *reinterpret_cast<uint32_t*>(&h);
            lo[e] = *reinterpret_cast<uint32_t*>(&l);
        }
        const int n = (t & 31) * 4 + i;                             // operand row inside the tile
        uint8_t* d = dst + (uint32_t)(n >> 3) * 512u + (uint32_t)rg * 128u + (uint32_t)(n & 7) * 16u;
        *reinterpret_cast<uint4*>(d) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(d + kHalf) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}

__global__ void __launch_bounds__(288)
gemm_tn_tc_kernel(const float* __restrict__ A, int lda, const float* __restrict__ B, int ldb, float* __restrict__ C, int ldc,
                  int64_t M, int N, int K, int64_t rows_per_split) {
    extern __shared__ __align__(1024) uint8_t smem[];
    Bars* bars = reinterpret_cast<Bars*>(smem + kStages * 2 * kStageOp);
    const int tid = threadIdx.x, warp = tid >> 5;
    const int n0 = blockIdx.x * 128, k0 = blockIdx.y * 128;
    const int64_t m_begin = (int64_t)blockIdx.z * rows_per_split;
    const int64_t m_end = m_begin + rows_per_split < M ? m_begin + rows_per_split : M;
    const int nsteps = (int)((m_end - m_begin + kBM - 1) / kBM);
    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&bars->full[s], 256); mbar_init(&bars->empty[s], 1); }
        mbar_init(&bars->d_full, 1);
        fence_mbar_init();
    }
    if (warp == 8) { tmem_alloc(&bars->tmem_base, 128); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = bars->tmem_base;
    uint8_t* opA = smem;                                  // [stage][hi | lo]
    uint8_t* opB = smem + kStages * kStageOp;

    if (warp < 8) {
        const bool isA = warp < 4;
        const int t = tid & 127;
        for (int st = 0; st < nsteps; ++st) {
            const int s = st % kStages;
            const uint32_t use = (uint32_t)(st / kStages);
            mbar_wait_bounded(&bars->empty[s], (use & 1) ^ 1);
            const int64_t m0 = m_begin + (int64_t)st * kBM;
            if (isA) fill_operand(opA + s * kStageOp, A, lda, m0, m_end, n0, N, t);
            else fill_operand(opB + s * kStageOp, B, ldb, m0, m_end, k0, K, t);
            fence_proxy_async_smem();
            mbar_arrive(&bars->full[s]);
        }
        if (isA) {
            // ---- epilogue: TMEM lane = n row of the tile
            mbar_wait_bounded(&bars->d_full, 0);
            tc_fence_after();
            const int n = n0 + warp * 32 + (tid & 31);
            const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
#pragma unroll
            for (int c0 = 0; c0 < 128; c0 += 32) {
                uint32_t r[32];
                tmem_ld_x32(tmem + lane_base + c0, r);
                tmem_ld_wait();
                if (n < N) {
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (k0 + c0 + j < K) atomicAdd(C + (int64_t)n * ldc + k0 + c0 + j, __uint_as_float(r[j]));
                }
            }
        }
    } else {
        const uint32_t idesc = make_idesc_f16(128, 128);
        const uint64_t dsc_a = make_smem_desc(smem_u32(opA), 128, 512);
        const uint64_t dsc_b = make_smem_desc(smem_u32(opB), 128, 512);
        for (int st = 0; st < nsteps; ++st) {
            const int s = st % kStages;
            const uint32_t use = (uint32_t)(st / kStages);
            mbar_wait_bounded(&bars->full[s], use & 1);
            tc_fence_after();
            if (elect_one()) {
                const uint64_t a_hi = dsc_a + (uint64_t)(s * (kStageOp >> 4)), a_lo = a_hi + (uint64_t)(kHalf >> 4);
                const uint64_t b_hi = dsc_b + (uint64_t)(s * (kStageOp >> 4)), b_lo = b_hi + (uint64_t)(kHalf >> 4);
#pragma unroll
                for (int ks = 0; ks < kBM / 16; ++ks) {
                    mma_ss(tmem, a_lo + (uint64_t)(ks * 16), b_hi + (uint64_t)(ks * 16), idesc, (st | ks) > 0);
                    mma_ss(tmem, a_hi + (uint64_t)(ks * 16), b_lo + (uint64_t)(ks * 16), idesc, 1);
                    mma_ss(tmem, a_hi + (uint64_t)(ks * 16), b_hi + (uint64_t)(ks * 16), idesc, 1);
                }
                mma_commit(&bars->empty[s]);
                if (st == nsteps - 1) mma_commit(&bars->d_full);
            }
            __syncwarp();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) tmem_dealloc(tmem, 128);
}

}  // namespace

bool gemm_tn_tc_ok(const float* A, int lda, const float* B, int ldb, int64_t M, int N, int K) {
    return M >= 4096 && N >= 64 && K >= 64 && N % 4 == 0 && K % 4 == 0 && lda % 4 == 0 && ldb % 4 == 0 &&
           ((uintptr_t)A % 16 == 0) && ((uintptr_t)B % 16 == 0);
}

// C must already hold the values the product is added to (zeros or a running gradient)
void launch_gemm_tn_tc(const float* A, int lda, const float* B, int ldb, float* C, int ldc, int64_t M, int N, int K,
                       cudaStream_t st) {
    DeviceCtx& ctx = device_ctx();
    ctx.set_max_dynamic_smem((const void*)gemm_tn_tc_kernel, (int)kSmem);
    const int64_t tiles = cdiv(N, 128) * cdiv(K, 128);
    int64_t splits = std::max<int64_t>(1, cdiv(2 * (int64_t)ctx.sm_count, tiles));
    splits = std::min<int64_t>(splits, cdiv(M, 1024));
    splits = std::min<int64_t>(splits, 65535);
    int64_t rows = cdiv(cdiv(M, splits), kBM) * kBM;
    splits = cdiv(M, rows);
    dim3 grid((unsigned)cdiv(N, 128), (unsigned)cdiv(K, 128), (unsigned)splits);
    P2S_LAUNCH(gemm_tn_tc_kernel, grid, 288, kSmem, st, A, lda, B, ldb, C, ldc, M, N, K, rows);
}

}  // namespace p2s
