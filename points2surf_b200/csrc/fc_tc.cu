// Tensor-core GEMM for the per-query FC tails of the TC path (QSTN/STN heads 1024->512->256->{4,4096} and the
// decoder 1024->512 (x2), 1024->256, 256->128; source/points_to_surf_model.py:62-64,120-122,335,343,348-350) and for
// the training GEMMs:
//     C[M][N] = act( A[M][K] * W[N][K]^T + b ),  W pre-packed operand images, fp32 accumulation in TMEM.
// These layers produce the point rotation, the 64x64 feature transform and the logits, so they keep fp32-level
// accuracy: every fp32 operand x is split into two fp16 numbers x_hi + x_lo (x_hi = fp16(x), x_lo = fp16(x - x_hi))
// and the product is evaluated as A_hi*W_hi + A_lo*W_hi + A_hi*W_lo (the dropped lo*lo term is ~2^-22 relative).
// Three tensor-core passes cost nothing here: the FC tails are 1 % of the network's FLOPs.
// One CTA per 128 x 128 output tile; K streamed in 32-wide stages (3-deep ring):
//   warps 0-3  producers: thread = output row; load 32 fp32 of that row, split, store the two K-major A operands;
//              afterwards the same warps run the epilogue (TMEM -> +bias, ReLU -> global)
//   warp 4     bulk-copies the W stage images (hi + lo, 16 KB) and issues the tcgen05.mma (elect-one issue)
// Two CTAs fit per SM (96 KB smem, 128 TMEM columns each), so one CTA's prologue/epilogue overlaps the other's MMAs.
#include "model.cuh"
#include "tc_ptx.cuh"

namespace p2s {

using namespace ptx;

namespace {

constexpr int kStages = 3;
constexpr int kBK = 32;
constexpr uint32_t kHalf = 128 * kBK * 2;     // one 128 x 32 fp16 operand image: 8 KB (K-major, LBO 128, SBO 512)
constexpr uint32_t kStageA = 2 * kHalf;       // hi + lo
constexpr uint32_t kStageB = 2 * kHalf;       // hi + lo
constexpr uint32_t kFcSmem = kStages * (kStageA + kStageB) + 256;

struct FcBars {
    uint64_t full[kStages], empty[kStages], d_full;
    uint32_t tmem_base;
};

// A operand: fp32 rows (converted by the producer warps, `A`; training GEMMs) or a pre-packed operand image `Aimg`
// ([M/128][K/32][hi | lo][128 x 32 fp16], the W layout; FC tails): then the producers have nothing to do and both operands of
// a k-step arrive by bulk copy.  ncu showed the fp32 mode L1TEX-bound on the FC tails (61-77 % l1tex throughput, 17-19 %
// tensor-active): every A element was loaded and split once per N tile (4x for the 1024->512 layers, 32x for the folded
// 256->4096 layer) through row-per-thread loads.
// out_mode: 0 fp32 rows (ldc), 1 / 2 the pass kernel's per-query operand image (fp16 / hi | lo), 3 the NEXT layer's operand
// image (k-steps out_kt_off.. of out_kt_total).
__global__ void __launch_bounds__(160) fc_tc_kernel(const float* __restrict__ A, int lda, const uint8_t* __restrict__ Wimg,
                                                    const float* __restrict__ bias, float* __restrict__ C, int ldc,
                                                    int M, int N, int K, int relu, int out_mode,
                                                    const uint8_t* __restrict__ Aimg, int out_kt_total, int out_kt_off) {
    extern __shared__ __align__(1024) uint8_t smem[];
    FcBars* bars = reinterpret_cast<FcBars*>(smem + kStages * (kStageA + kStageB));
    const int tid = threadIdx.x, warp = tid >> 5;
    const int m0 = blockIdx.y * 128, nt = blockIdx.x;   // N tiles of one row block are adjacent: A is re-read from L2
    const int nk = K / kBK;
    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&bars->full[s], Aimg ? 1 : 129); mbar_init(&bars->empty[s], 1); }
        mbar_init(&bars->d_full, 1);
        fence_mbar_init();
    }
    if (warp == 4) { tmem_alloc(&bars->tmem_base, 128); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = bars->tmem_base;

    if (warp < 4) {
        // ---- producers: A[m0 + tid][k0 .. k0+31] -> fp16 hi / lo, K-major (LBO 128, SBO 512)
        const int row = m0 + tid;
        const float* src = A + (int64_t)(row < M ? row : 0) * lda;
        // register double buffer: the loads of k-step kt + 1 are in flight while k-step kt is converted and stored (with one
        // stage of loads per thread the producers were latency-bound: ~800 cycles of L2 latency per 384 cycles of MMA)
        float4 v[8], nv[8];
        const bool row_ok = row < M;
        const int nk_prod = Aimg ? 0 : nk;           // operand image: nothing to produce
        if (!Aimg) {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = row_ok ? *reinterpret_cast<const float4*>(src + j * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        for (int kt = 0; kt < nk_prod; ++kt) {
            const int s = kt % kStages;
            const uint32_t use = (uint32_t)(kt / kStages);
            const bool more = row_ok && (kt + 1 < nk);
#pragma unroll
            for (int j = 0; j < 8; ++j) nv[j] = more ? *reinterpret_cast<const float4*>(src + (kt + 1) * kBK + j * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            mbar_wait_bounded(&bars->empty[s], (use & 1) ^ 1);
            uint8_t* dst = smem + s * kStageA + (uint32_t)(tid >> 3) * 512u + (uint32_t)(tid & 7) * 16u;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float x[8] = {v[2 * c].x, v[2 * c].y, v[2 * c].z, v[2 * c].w, v[2 * c + 1].x, v[2 * c + 1].y, v[2 * c + 1].z, v[2 * c + 1].w};
                uint32_t hi[4], lo[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    __half2 h = __floats2half2_rn(x[2 * e], x[2 * e + 1]);
                    float2 hf = __half22float2(h);
                    __half2 l = __floats2half2_rn(x[2 * e] - hf.x, x[2 * e + 1] - hf.y);
                    hi[e] = *reinterpret_cast<uint32_t*>(&h);
                    lo[e] = *reinterpret_cast<uint32_t*>(&l);
                }
                *reinterpret_cast<uint4*>(dst + c * 128) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                *reinterpret_cast<uint4*>(dst + kHalf + c * 128) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            }
            fence_proxy_async_smem();
            mbar_arrive(&bars->full[s]);
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = nv[j];
        }
        // ---- epilogue
        mbar_wait_bounded(&bars->d_full, 0);
        tc_fence_after();
        const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
        float* dstrow = C + (int64_t)row * ldc + nt * 128;
        const float* b = bias + nt * 128;
#pragma unroll
        for (int n0 = 0; n0 < 128; n0 += 32) {
            uint32_t r[32];
            tmem_ld_x32(tmem + lane_base + n0, r);
            tmem_ld_wait();
            if (out_mode == 3) {
                // C as the next layer's A operand image: this 32-column chunk is exactly one k-step of that layer
                uint8_t* blk = reinterpret_cast<uint8_t*>(C) + ((size_t)blockIdx.y * out_kt_total + out_kt_off + nt * 4 + (n0 >> 5)) * (size_t)kStageA +
                               (uint32_t)(tid >> 3) * 512u + (uint32_t)(tid & 7) * 16u;
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    uint32_t hi[4], lo[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        float x0 = __uint_as_float(r[g * 8 + 2 * e]) + b[n0 + g * 8 + 2 * e], x1 = __uint_as_float(r[g * 8 + 2 * e + 1]) + b[n0 + g * 8 + 2 * e + 1];
                        if (relu) { x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); }
                        if (row >= M) { x0 = 0.f; x1 = 0.f; }
                        __half2 h = __floats2half2_rn(x0, x1);
                        float2 hf = __half22float2(h);
                        __half2 l = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
                        hi[e] = *reinterpret_cast<uint32_t*>(&h);
                        lo[e] = *reinterpret_cast<uint32_t*>(&l);
                    }
                    *reinterpret_cast<uint4*>(blk + g * 128) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<uint4*>(blk + kHalf + g * 128) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                }
            } else if (row < M && out_mode) {
                // C is a per-row fp16 operand image of a [64][64] matrix (row-major index = column of this GEMM):
                // K-major, LBO 128, SBO 1024 -- the per-query B operand of the pass kernel
                // out_mode == 2: split precision, 16384 B per row: hi image | lo image
                uint8_t* img = reinterpret_cast<uint8_t*>(C) + (size_t)row * (out_mode == 2 ? 16384 : 8192);
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                    const int col = nt * 128 + n0 + j;
                    const int o = col >> 6, i = col & 63;
                    uint32_t v[4], vl[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float x0 = __uint_as_float(r[j + 2 * e]) + b[n0 + j + 2 * e], x1 = __uint_as_float(r[j + 2 * e + 1]) + b[n0 + j + 2 * e + 1];
                        v[e] = pack_half2(x0, x1);
                        const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&v[e]));
                        vl[e] = pack_half2(x0 - hf.x, x1 - hf.y);
                    }
                    const uint32_t off = (uint32_t)(o >> 3) * 1024u + (uint32_t)(i >> 3) * 128u + (uint32_t)(o & 7) * 16u;
                    *reinterpret_cast<uint4*>(img + off) = make_uint4(v[0], v[1], v[2], v[3]);
                    if (out_mode == 2) *reinterpret_cast<uint4*>(img + 8192 + off) = make_uint4(vl[0], vl[1], vl[2], vl[3]);
                }
            } else if (row < M) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    if (nt * 128 + n0 + j >= N) continue;   // padded tile (N % 128 != 0, N % 4 == 0)
                    float4 o;
                    o.x = __uint_as_float(r[j + 0]) + b[n0 + j + 0];
                    o.y = __uint_as_float(r[j + 1]) + b[n0 + j + 1];
                    o.z = __uint_as_float(r[j + 2]) + b[n0 + j + 2];
                    o.w = __uint_as_float(r[j + 3]) + b[n0 + j + 3];
                    if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                    *reinterpret_cast<float4*>(dstrow + n0 + j) = o;
                }
            }
        }
    } else {
        // ---- W stage copies + MMA issue (warp-uniform loop, one elected lane issues)
        const uint32_t idesc = make_idesc_f16(128, 128);
        const uint64_t dsc_a = make_smem_desc(smem_u32(smem), 128, 512);
        const uint64_t dsc_b = make_smem_desc(smem_u32(smem + kStages * kStageA), 128, 512);
        const uint8_t* wsrc = Wimg + (size_t)nt * nk * kStageB;
        const uint8_t* asrc = Aimg ? Aimg + (size_t)blockIdx.y * nk * kStageA : nullptr;
        // prefetch the first stages of W (and of A in image mode)
        for (int kt = 0; kt < nk && kt < kStages; ++kt) {
            if (elect_one()) {
                mbar_arrive_expect_tx(&bars->full[kt], kStageB + (asrc ? kStageA : 0u));
                bulk_g2s(smem + kStages * kStageA + kt * kStageB, wsrc + (size_t)kt * kStageB, kStageB, &bars->full[kt]);
                if (asrc) bulk_g2s(smem + kt * kStageA, asrc + (size_t)kt * kStageA, kStageA, &bars->full[kt]);
            }
            __syncwarp();
        }
        for (int kt = 0; kt < nk; ++kt) {
            const int s = kt % kStages;
            const uint32_t use = (uint32_t)(kt / kStages);
            mbar_wait_bounded(&bars->full[s], use & 1);
            tc_fence_after();
            if (elect_one()) {
                const uint64_t a_hi = dsc_a + (uint64_t)(s * (kStageA >> 4)), a_lo = a_hi + (uint64_t)(kHalf >> 4);
                const uint64_t b_hi = dsc_b + (uint64_t)(s * (kStageB >> 4)), b_lo = b_hi + (uint64_t)(kHalf >> 4);
#pragma unroll
                for (int ks = 0; ks < kBK / 16; ++ks) {
                    mma_ss(tmem, a_lo + (uint64_t)(ks * 16), b_hi + (uint64_t)(ks * 16), idesc, (kt | ks) > 0);   // small terms first
                    mma_ss(tmem, a_hi + (uint64_t)(ks * 16), b_lo + (uint64_t)(ks * 16), idesc, 1);
                    mma_ss(tmem, a_hi + (uint64_t)(ks * 16), b_hi + (uint64_t)(ks * 16), idesc, 1);
                }
                mma_commit(&bars->empty[s]);
                if (kt == nk - 1) mma_commit(&bars->d_full);
            }
            __syncwarp();
            // refill the slot used one step earlier (its MMAs have had a full stage of time to drain) with the W
            // image of k-step (kt - 1) + kStages
            if (kt >= 1) {
                const int kp = kt - 1, kn = kp + kStages;
                if (kn < nk) {
                    const int sp = kp % kStages;
                    mbar_wait_bounded(&bars->empty[sp], (uint32_t)(kp / kStages) & 1);
                    if (elect_one()) {
                        mbar_arrive_expect_tx(&bars->full[sp], kStageB + (asrc ? kStageA : 0u));
                        bulk_g2s(smem + kStages * kStageA + sp * kStageB, wsrc + (size_t)kn * kStageB, kStageB, &bars->full[sp]);
                        if (asrc) bulk_g2s(smem + sp * kStageA, asrc + (size_t)kn * kStageA, kStageA, &bars->full[sp]);
                    }
                    __syncwarp();
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) tmem_dealloc(tmem, 128);
}

// fp32 activations A[M][K] (+ optional bias / ReLU) -> A operand images [ceil(M/128)][K/32][hi | lo][128 x 32 fp16, K-major,
// LBO 128, SBO 512]; rows >= M are zero.  One CTA per (row tile, k-step): 8 lanes read one row's 128 bytes (coalesced).
__global__ void __launch_bounds__(256) pack_a_kernel(const float* __restrict__ A, int lda, int M, int K, const float* __restrict__ in_bias,
                                                     int in_relu, uint8_t* __restrict__ img) {
    const int kt = blockIdx.x, mt = blockIdx.y, c = threadIdx.x & 7;
    uint8_t* blk = img + ((size_t)mt * (K / kBK) + kt) * (size_t)kStageA;
    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (in_bias) b4 = __ldg(reinterpret_cast<const float4*>(in_bias + kt * kBK + c * 4));
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = (threadIdx.x >> 3) + 32 * i, row = mt * 128 + r;
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row < M) {
            x = *reinterpret_cast<const float4*>(A + (int64_t)row * lda + kt * kBK + c * 4);
            x.x += b4.x; x.y += b4.y; x.z += b4.z; x.w += b4.w;
            if (in_relu) { x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f); }
        }
        const __half2 h0 = __floats2half2_rn(x.x, x.y), h1 = __floats2half2_rn(x.z, x.w);
        const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
        const __half2 l0 = __floats2half2_rn(x.x - f0.x, x.y - f0.y), l1 = __floats2half2_rn(x.z - f1.x, x.w - f1.y);
        const uint32_t off = (uint32_t)(r >> 3) * 512u + (uint32_t)(c >> 1) * 128u + (uint32_t)(r & 7) * 16u + (uint32_t)(c & 1) * 8u;
        *reinterpret_cast<uint2*>(blk + off) = make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
        *reinterpret_cast<uint2*>(blk + kHalf + off) = make_uint2(*reinterpret_cast<const uint32_t*>(&l0), *reinterpret_cast<const uint32_t*>(&l1));
    }
}

// fp32 W[N][K] -> images [Npad/128][K/32][hi | lo][128 x 32 fp16, K-major, LBO 128, SBO 512], rows N..Npad-1 zero
__global__ void pack_fc_pad_kernel(const float* __restrict__ W, int N, int Npad, int K, uint8_t* __restrict__ img) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)Npad * K) return;
    int n = (int)(e / K), k = (int)(e % K);
    int nt = n >> 7, r = n & 127, kt = k / kBK, kk = k % kBK;
    size_t off = ((size_t)nt * (K / kBK) + kt) * kStageB + (size_t)(r >> 3) * 512 + (size_t)(kk >> 3) * 128 + (size_t)(r & 7) * 16 + (size_t)(kk & 7) * 2;
    const float w = n < N ? W[e] : 0.f;
    const __half h = __float2half_rn(w);
    *reinterpret_cast<__half*>(img + off) = h;
    *reinterpret_cast<__half*>(img + off + kHalf) = __float2half_rn(w - __half2float(h));
}

}  // namespace

bool fc_tc_supported(int N, int K) { return (N % 128 == 0) && (K % kBK == 0) && N >= 128 && K >= kBK; }

uint8_t* fc_tc_pack(const Layer& L, std::vector<void*>& allocs) { return fc_tc_pack_raw(L.W, L.cout, L.cin, allocs); }

// A as fp32 rows, C as fp32 rows; N may end in a partial 128-column tile (N % 4 == 0)
void launch_fc_tc(const float* A, int lda, const uint8_t* Wimg, const float* bias, float* C, int ldc,
                  int64_t M, int N, int K, bool relu, cudaStream_t st) {
    if (M <= 0) return;
    P2S_CHECK(N % 4 == 0 && N >= 64 && K % kBK == 0 && K >= kBK && lda % 4 == 0 && ldc % 4 == 0, "bad FC shape for the tensor-core kernel");
    P2S_CHECK(cdiv(M, 128) <= 65535, "too many rows for one launch");
    dim3 grid((unsigned)cdiv(N, 128), (unsigned)cdiv(M, 128), 1);
    device_ctx().set_max_dynamic_smem((const void*)fc_tc_kernel, (int)kFcSmem);
    P2S_LAUNCH(fc_tc_kernel, grid, 160, kFcSmem, st, A, lda, Wimg, bias, C, ldc, (int)M, N, K, relu ? 1 : 0, 0, (const uint8_t*)nullptr, 0, 0);
}

void launch_pack_a(const float* A, int lda, int64_t M, int K, const float* in_bias, bool in_relu, uint8_t* img, cudaStream_t st) {
    if (M <= 0) return;
    P2S_CHECK(K % kBK == 0 && lda % 4 == 0 && cdiv(M, 128) <= 65535, "bad shape for the A operand image");
    dim3 grid((unsigned)(K / kBK), (unsigned)cdiv(M, 128), 1);
    P2S_LAUNCH(pack_a_kernel, grid, 256, 0, st, A, lda, (int)M, K, in_bias, in_relu ? 1 : 0, img);
}

// A given as an operand image (launch_pack_a or a previous layer's out_mode 3).  out_mode: 0 fp32 row-major C (ldc), 1 / 2 the
// per-query operand image of the pass kernel (N == 4096), 3 the next layer's A image (k-steps out_kt_off.. of out_kt_total).
void launch_fc_tc_img(const uint8_t* Aimg, const uint8_t* Wimg, const float* bias, void* C, int ldc, int64_t M, int N, int K,
                      bool relu, cudaStream_t st, int out_mode, int out_kt_total, int out_kt_off) {
    if (M <= 0) return;
    P2S_CHECK(fc_tc_supported(N, K) && Aimg && (out_mode == 0 ? ldc % 4 == 0 : (out_mode == 3 ? out_kt_off + N / 32 <= out_kt_total : N == 4096)),
              "bad FC shape for the tensor-core kernel (operand-image mode)");
    P2S_CHECK(cdiv(M, 128) <= 65535, "too many rows for one launch");
    dim3 grid((unsigned)(N / 128), (unsigned)cdiv(M, 128), 1);
    device_ctx().set_max_dynamic_smem((const void*)fc_tc_kernel, (int)kFcSmem);
    P2S_LAUNCH(fc_tc_kernel, grid, 160, kFcSmem, st, (const float*)nullptr, 0, Wimg, bias, reinterpret_cast<float*>(C), ldc, (int)M, N, K, relu ? 1 : 0,
               out_mode, Aimg, out_kt_total, out_kt_off);
}

// images of a raw fp32 matrix W[N][K] (device pointer)
uint8_t* fc_tc_pack_raw(const float* W, int N, int K, std::vector<void*>& allocs) {
    P2S_CHECK(fc_tc_supported(N, K), "layer shape not supported by the tensor-core FC kernel");
    void* p = nullptr;
    P2S_CUDA(cudaMalloc(&p, (size_t)N * K * 4));
    allocs.push_back(p);
    P2S_LAUNCH(pack_fc_pad_kernel, (unsigned)cdiv((int64_t)N * K, 256), 256, 0, 0, W, N, N, K, (uint8_t*)p);
    return (uint8_t*)p;
}

// Split-precision tensor-core GEMM for weights that change between calls (training): packs W [N][K] into a reusable
// scratch image on `st`, then runs fc_tc_kernel.  Stream order makes the scratch reuse safe.  bias may be null.
bool gemm_nt_tc_ok(const float* A, int lda, const float* C, int ldc, int64_t M, int N, int K) {
    return N % 4 == 0 && N >= 64 && K % kBK == 0 && K >= kBK && N <= 4096 && M >= 128 && M < (int64_t)1 << 31 && lda % 4 == 0 && ldc % 4 == 0 &&
           ((uintptr_t)A % 16 == 0) && ((uintptr_t)C % 16 == 0);
}

void launch_gemm_nt_tc(const float* A, int lda, const float* W, const float* bias, float* C, int ldc, int64_t M, int N,
                       int K, bool relu, cudaStream_t st) {
    DeviceCtx& ctx = device_ctx();
    const int Npad = (int)(cdiv(N, 128) * 128);
    uint8_t* wimg = reinterpret_cast<uint8_t*>(ctx.train_wimg.get((size_t)Npad * K * 4));
    if (!bias) {
        const bool fresh = !ctx.train_zero_bias.p;
        float* z = ctx.train_zero_bias.as<float>(4096);
        if (fresh) P2S_CUDA(cudaMemsetAsync(z, 0, 4096 * sizeof(float), st));
        bias = z;
    }
    P2S_LAUNCH(pack_fc_pad_kernel, (unsigned)cdiv((int64_t)Npad * K, 256), 256, 0, st, W, N, Npad, K, wimg);
    launch_fc_tc(A, lda, wimg, bias, C, ldc, M, N, K, relu, st);
}

}  // namespace p2s
