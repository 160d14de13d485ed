// Tensor-core implementation of PointsToSurfModel.forward (source/points_to_surf_model.py:296-352) for sm_100a.
//
// The per-point Conv1d(k=1) stacks (98 % of the FLOPs, SURVEY.md section 2a) run as tcgen05.mma tiles with fp16
// operands / fp32 accumulation in TMEM; the three dependent max-reductions of the vanilla network become three
// launches of ONE kernel (`pointnet_pass_kernel`):
//   pass A  QSTN        : x(1300 pts) -> 64 (fp32 FMA) -> 128 -> 1024, max          (model.py:100-107)
//   pass B  STN64       : x -> 64 -> 64 | 64 -> 128 -> 1024, max                     (model.py:190-191,41-48)
//   pass C  final       : x -> 64 -> 64 | (W1*T) 64 -> 128 -> 1024 (no ReLU), max    (model.py:190-212)
// The quaternion rotation is folded into the first layer's weights per query (W0*R), the 64x64 feature
// transform into conv1's weights per query (W1*T), both exactly as in the fp32 path up to operation order.
//
// Tile = 128 points of one query (segments are padded with a duplicate of their first point: max-invariant).
// Mid layers: M = 128 points (TMEM lanes), A operand = activations in TMEM (tcgen05.st by the epilogue
// warps), B operand = weights in smem.  Big layer 128 -> 1024: M = 128 channels, A = resident W3 tile in smem,
// B = the tile's 128-channel activations in smem, D[channel lane][point column] so that the max over points is
// a per-thread reduction over TMEM columns (no shuffles).  Each CTA owns 512 of the 1024 channels (its half
// of W3, 128 KB fp16, stays resident in shared memory); CTA 2j and 2j+1 stream the same queries.
//
// Warp roles (576 threads): warps 14-17 compute the first layer (fp32 FMA) of every tile; warps 0-3 and 9-12 are two
// chains (even / odd tiles) running the mid-layer epilogues (thread = point = TMEM lane); warps 4-7 the column-max
// epilogue of the big layer; warp 8 issues the big-layer MMAs (blocking waits), warp 13 the mid-layer MMAs of both
// chains (polling).
//
// The small per-query FC tails between the passes run on the split-precision tensor-core FC kernel (fc_tc.cu) as a chain of
// operand images; only the 256 -> 4 QSTN output layer and the 128 -> 2 logits layer stay on the fp32 FMA GEMM (net_fp32.cu).
#include "model.cuh"
#include "tc_ptx.cuh"

#ifndef P2S_TC_BOUNDED_WAIT
#define P2S_TC_BOUNDED_WAIT 1   // trap instead of hanging if a barrier protocol bug slips in
#endif

namespace p2s {

using namespace ptx;

namespace {

constexpr int kTile = 128;
constexpr int kThreads = 576;   // warps 0-3 chain 0 | 4-7 column-max epilogue | 8 big-layer issuer | 9-12 chain 1 | 13 mid-layer issuer | 14-17 first layer
// shared memory map (bytes).  PRECISE = split-precision variant used for the guard-band recompute: every fp16
// operand x is carried as x_hi + x_lo and every product is evaluated as a_hi*b_hi + a_lo*b_hi + a_hi*b_lo (three MMAs
// per k-step, ~2^-22 relative), so the images are twice as large and a CTA owns one 128-channel chunk instead of four.
constexpr uint32_t kAct2Bytes = 32768;                   // 128 points x 128 channels fp16
constexpr uint32_t kSmallBytes = 192 * 4 + 320 * 4 + 168;  // Wq[3][64], biases[256 mid + 64 first], barriers
template <bool PRECISE>
struct Cfg {
    static constexpr int kChunks = PRECISE ? 1 : 4;                  // 128-channel chunks of the big layer per CTA
    static constexpr int kSplit = 8 / kChunks;                       // CTAs that share one query stream
    static constexpr uint32_t kChunkBytes = PRECISE ? 65536u : 32768u;   // W3 chunk image (hi [+ lo])
    static constexpr uint32_t kW3Bytes = kChunks * kChunkBytes;
    static constexpr uint32_t kMidBytes = (8192u + 8192u + 16384u) * (PRECISE ? 2u : 1u);
    static constexpr uint32_t kOffMid = kW3Bytes;
    static constexpr uint32_t kOffAct2 = kOffMid + kMidBytes;
    static constexpr uint32_t kOffSmall = kOffAct2 + 2 * kAct2Bytes;   // normal: two tile buffers; precise: one buffer, hi | lo
    static constexpr uint32_t kSmemBytes = kOffSmall + kSmallBytes;
    static constexpr uint32_t kACols = PRECISE ? 64u : 32u;          // TMEM columns of one chain's A operand (hi [+ lo])
    static constexpr uint32_t kPerqBytes = PRECISE ? 16384u : 8192u; // per-query conv1*(T+I) image
    static constexpr uint32_t kMidScale = PRECISE ? 2u : 1u;
};
static_assert(Cfg<false>::kSmemBytes <= 232448 && Cfg<true>::kSmemBytes <= 232448, "shared memory budget");
// TMEM map (columns)
constexpr uint32_t kColD3 = 0;      // 2 stages x 128
constexpr uint32_t kColDmid = 256;  // 128 columns: accumulator of the 128-channel mid layers (shared by the chains)
constexpr uint32_t kColDmidB = 448; // 64 columns: accumulator of the 64-channel mid layers (shared by the chains)
constexpr uint32_t kColA = 384;     // 2 chains x 32 (fp16 pairs, K = 64)

struct Seg {
    const float* ptr;   // [B, n, 3]
    int n;              // real points per query
    int tiles;          // ceil(n / 128)
    int center;         // subtract the query point (model.py:303)
};

struct PassParams {
    Seg seg[2];
    const float* query;        // [B,3]
    const float* R;            // [B,9] rotation folded into W0, or null
    int tiles_per_query;
    int B;
    const float* W0;           // [64,3]
    const float* b0;           // [64]
    int num_mid;               // 1 or 3
    int mid_N[3];              // output channels of each mid layer
    const uint8_t* mid_img[3]; // packed fp16 operand images (K-major, LBO 128, SBO 1024)
    const float* mid_bias[3];
    int perq_layer;            // index of the mid layer with per-query weights, or -1
    const uint8_t* perq_img;   // [B] x 8192 B (precise: hi | lo, 16384 B)
    const uint8_t* w3_img;     // [8 chunks][32768 B] (precise: [8][hi | lo])  (K-major, LBO 128, SBO 2048)
    float* out;                // [B,1024] raw max (bias / ReLU applied by the consumer: launch_pack_a adds it while packing)
    long long* wstats;         // diagnostics: per-role barrier wait cycles (null = off)
};

struct Bars {
    uint64_t w_full, wq_full, perq_done;
    uint64_t dmid_free[2];      // [0]: 128-column accumulator, [1]: 64-column accumulator
    uint64_t a_ready[2], a_free[2], dmid_ready[2];
    uint64_t act2_full[2], act2_empty[2], d3_full[2], d3_empty[2];
    uint32_t tmem_base;
};
static_assert(sizeof(Bars) <= 168, "barrier block");

// `acc` (diagnostics, P2S_TC_WAITSTATS=1): cycles this thread spent waiting are added to it
__device__ __forceinline__ void wait_bar(uint64_t* bar, uint32_t parity, long long* acc = nullptr) {
#if P2S_TC_BOUNDED_WAIT
    long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 2000000000LL) {
            printf("p2s: mbarrier timeout block %d thread %d bar %p parity %u\n", blockIdx.x, threadIdx.x, (void*)bar, parity);
            __trap();
        }
    }
    if (acc) *acc += clock64() - t0;
#else
    mbar_wait(bar, parity);
#endif
}
// wait statistics layout: [role 0..5][slot 0..7]; roles: 0 big-layer issuer, 1 mid issuer, 2 chain 0, 3 chain 1, 4 first layer,
// 5 column-max epilogue; slots: 0 act2_full, 1 d3_empty, 2 dmid_free, 3 dmid_ready, 4 act2_empty, 5 a_free, 6 d3_full, 7 role cycles
enum { WS_ACT2_FULL = 0, WS_D3_EMPTY, WS_DMID_FREE, WS_DMID_READY, WS_ACT2_EMPTY, WS_A_FREE, WS_D3_FULL, WS_TOTAL, WS_SLOTS };
__device__ __forceinline__ void ws_flush(long long* g, int role, const long long* ws, long long t_begin) {
    if (!g || (threadIdx.x & 31) != 0) return;
    for (int i = 0; i < WS_TOTAL; ++i) if (ws[i]) atomicAdd((unsigned long long*)&g[role * WS_SLOTS + i], (unsigned long long)ws[i]);
    atomicAdd((unsigned long long*)&g[role * WS_SLOTS + WS_TOTAL], (unsigned long long)(clock64() - t_begin));
}

// relu(a), relu(b) -> packed fp16x2 (low half = a), saturating
__device__ __forceinline__ uint32_t pack_relu(float a, float b) {
    uint32_t r;
    asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
}
// split-precision variant: hi = fp16(relu(x)), lo = fp16(relu(x) - hi)
__device__ __forceinline__ void pack_relu_split(float a, float b, uint32_t& hi, uint32_t& lo) {
    hi = pack_relu(a, b);
    const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
    lo = pack_half2(fmaxf(a, 0.f) - hf.x, fmaxf(b, 0.f) - hf.y);
}

template <bool PRECISE, bool STATS = false>
__global__ void __launch_bounds__(kThreads, 1) pointnet_pass_kernel(const PassParams p) {
    using C = Cfg<PRECISE>;
    constexpr uint32_t kOffMid = C::kOffMid, kOffAct2 = C::kOffAct2, kOffSmall = C::kOffSmall, kOffW3 = 0;
    extern __shared__ __align__(1024) uint8_t smem[];
    float* s_wq = reinterpret_cast<float*>(smem + kOffSmall);             // [3][64]: rows of (W0*R)^T
    float* s_bias = s_wq + 192;                                           // [256] mid biases back to back, [64] first-layer bias
    Bars* bars = reinterpret_cast<Bars*>(s_bias + 320);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int part = blockIdx.x % C::kSplit;                             // which 128-channel chunks this CTA owns
    const int stream = blockIdx.x / C::kSplit, nstreams = gridDim.x / C::kSplit;
    const int nq = (p.B > stream) ? (p.B - stream + nstreams - 1) / nstreams : 0;   // queries of this CTA
    const int tpq = p.tiles_per_query;
    const int ntiles = nq * tpq;

    if (tid == 0) {
        mbar_init(&bars->w_full, 1);
        mbar_init(&bars->wq_full, 1);
        mbar_init(&bars->perq_done, 1);
        mbar_init(&bars->dmid_free[0], 128);
        mbar_init(&bars->dmid_free[1], 128);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars->a_ready[i], 128);
            mbar_init(&bars->a_free[i], 128);
            mbar_init(&bars->dmid_ready[i], 1);
            mbar_init(&bars->act2_full[i], 128);
            mbar_init(&bars->act2_empty[i], 1);
            mbar_init(&bars->d3_full[i], 1);
            mbar_init(&bars->d3_empty[i], 128);
        }
        fence_mbar_init();
    }
    if (warp == 8) { tmem_alloc(&bars->tmem_base, 512); tmem_relinquish(); }
    {
        int off = 0;
        for (int l = 0; l < p.num_mid; ++l) {
            for (int i = tid; i < p.mid_N[l]; i += kThreads) s_bias[off + i] = p.mid_bias[l][i];
            off += p.mid_N[l];
        }
        for (int i = tid; i < 64; i += kThreads) s_bias[256 + i] = p.b0[i];
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = bars->tmem_base;
    long long ws[WS_TOTAL] = {0, 0, 0, 0, 0, 0, 0};
    long long* const wsp = STATS ? ws : nullptr;            // STATS = false: everything below folds away
    const long long t_begin = STATS ? clock64() : 0;

    if (warp == 8) {
        // =============================================================== big-layer MMA issuer (+ resident weight loads)
        // The whole warp runs the warp-uniform loop; one elected lane issues the asynchronous instructions.
        if (ntiles > 0) {
            if (lane == 0) {
                uint32_t bytes = C::kW3Bytes;
                for (int l = 0; l < p.num_mid; ++l) if (l != p.perq_layer) bytes += (uint32_t)p.mid_N[l] * 128u * C::kMidScale;
                mbar_arrive_expect_tx(&bars->w_full, bytes);
                for (uint32_t o = 0; o < C::kW3Bytes; o += 32768u)
                    bulk_g2s(smem + kOffW3 + o, p.w3_img + (size_t)part * C::kW3Bytes + o, 32768, &bars->w_full);
                uint32_t o = 0;
                for (int l = 0; l < p.num_mid; ++l) {
                    const uint32_t lb = (uint32_t)p.mid_N[l] * 128u * C::kMidScale;
                    if (l != p.perq_layer) bulk_g2s(smem + kOffMid + o, p.mid_img[l], lb, &bars->w_full);
                    else {
                        mbar_arrive_expect_tx(&bars->wq_full, C::kPerqBytes);
                        bulk_g2s(smem + kOffMid + o, p.perq_img + (size_t)stream * C::kPerqBytes, C::kPerqBytes, &bars->wq_full);
                    }
                    o += lb;
                }
            }
            __syncwarp();
            wait_bar(&bars->w_full, 0);
            const uint32_t idesc_l3 = make_idesc_f16(128, 128);
            const uint64_t dsc_w3 = make_smem_desc(smem_u32(smem + kOffW3), 128, 2048);
            const uint64_t dsc_act2 = make_smem_desc(smem_u32(smem + kOffAct2), 128, 2048);
            for (int it = 0; it < ntiles; ++it) {
                // normal: tile t uses activation buffer t & 1; precise: one buffer (hi | lo) used by every tile
                const uint32_t buf = PRECISE ? 0u : ((uint32_t)it & 1), buse = PRECISE ? (uint32_t)it : ((uint32_t)it >> 1);
                wait_bar(&bars->act2_full[buf], buse & 1, wsp ? wsp + WS_ACT2_FULL : nullptr);
                const uint64_t db = dsc_act2 + (uint64_t)(buf * (kAct2Bytes >> 4));
#pragma unroll
                for (int c = 0; c < C::kChunks; ++c) {
                    const uint32_t g = (uint32_t)(it * C::kChunks + c);
                    const uint32_t stage = g & 1, use = g >> 1;
                    wait_bar(&bars->d3_empty[stage], (use & 1) ^ 1, wsp ? wsp + WS_D3_EMPTY : nullptr);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint64_t da = dsc_w3 + (uint64_t)((uint32_t)c * (C::kChunkBytes >> 4));
                        const uint32_t d = tmem + kColD3 + stage * 128u;
                        if (PRECISE) {
                            const uint64_t da_lo = da + (uint64_t)(32768u >> 4), db_lo = db + (uint64_t)(32768u >> 4);
#pragma unroll
                            for (int ks = 0; ks < 8; ++ks) {
                                mma_ss(d, da_lo + (uint64_t)(ks * 16), db + (uint64_t)(ks * 16), idesc_l3, ks > 0);   // small terms first
                                mma_ss(d, da + (uint64_t)(ks * 16), db_lo + (uint64_t)(ks * 16), idesc_l3, 1);
                                mma_ss(d, da + (uint64_t)(ks * 16), db + (uint64_t)(ks * 16), idesc_l3, 1);
                            }
                        } else {
#pragma unroll
                            for (int ks = 0; ks < 8; ++ks)
                                mma_ss(d, da + (uint64_t)(ks * 16), db + (uint64_t)(ks * 16), idesc_l3, ks > 0);
                        }
                        mma_commit(&bars->d3_full[stage]);
                        if (c == C::kChunks - 1) mma_commit(&bars->act2_empty[buf]);
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp == 13) {
        // =============================================================== mid-layer MMA issuer (serves the two chains)
        if (ntiles > 0) {
            uint32_t mid_off[3] = {0, 0, 0};
            {
                uint32_t o = 0;
                for (int l = 0; l < p.num_mid; ++l) { mid_off[l] = o; o += (uint32_t)p.mid_N[l] * 128u * C::kMidScale; }
            }
            const bool perq = p.perq_layer >= 0;
            wait_bar(&bars->w_full, 0);
            if (perq) wait_bar(&bars->wq_full, 0);
            const uint64_t dsc_mid0 = make_smem_desc(smem_u32(smem + kOffMid) + mid_off[0], 128, 1024);
            const uint64_t dsc_mid1 = make_smem_desc(smem_u32(smem + kOffMid) + mid_off[1], 128, 1024);
            const uint64_t dsc_mid2 = make_smem_desc(smem_u32(smem + kOffMid) + mid_off[2], 128, 1024);
            const uint32_t idesc_mid0 = make_idesc_f16(128, (uint32_t)p.mid_N[0]);
            const uint32_t idesc_mid1 = make_idesc_f16(128, (uint32_t)(p.num_mid > 1 ? p.mid_N[1] : 64));
            const uint32_t idesc_mid2 = make_idesc_f16(128, (uint32_t)(p.num_mid > 2 ? p.mid_N[2] : 64));
            int it_mid0 = 0, it_mid1 = 1, l_mid0 = 0, l_mid1 = 0;
            uint32_t rnd0 = 0, rnd1 = 0;        // per-chain (tile, layer) round counter
            uint32_t g_mid = 0;                 // mid MMAs issued so far (alternates which chain is polled first)
            uint32_t g_buf0 = 0, g_buf1 = 0;    // MMAs issued into the 128-column / 64-column accumulator
            int loaded_q = 0, perq_count = 0;   // per-query weights resident for local query `loaded_q`
            bool pq_loading = false;
            while (it_mid0 < ntiles || it_mid1 < ntiles) {
                // ---- per-query weight prefetch: once every tile of the resident query has issued its MMA
                if (perq) {
                    if (!pq_loading && perq_count == tpq && loaded_q + 1 < nq && mbar_test_wait_warp(&bars->perq_done, (uint32_t)loaded_q & 1)) {
                        if (elect_one()) {
                            mbar_arrive_expect_tx(&bars->wq_full, C::kPerqBytes);
                            bulk_g2s(smem + kOffMid + mid_off[p.perq_layer],
                                     p.perq_img + ((size_t)stream + (size_t)(loaded_q + 1) * nstreams) * C::kPerqBytes, C::kPerqBytes, &bars->wq_full);
                        }
                        __syncwarp();
                        pq_loading = true;
                    }
                    if (pq_loading && mbar_test_wait_warp(&bars->wq_full, (uint32_t)(loaded_q + 1) & 1)) {
                        ++loaded_q; perq_count = 0; pq_loading = false;
                    }
                }
                auto try_mid = [&](const int c, int& it_m, int& l_m, uint32_t& rn) {
                    if (it_m >= ntiles) return;
                    const int l = l_m;
                    if (l == p.perq_layer && it_m / tpq != loaded_q) return;
                    if (!mbar_test_wait_warp(&bars->a_ready[c], rn & 1)) return;
                    const bool small = !PRECISE && (p.mid_N[l] == 64);   // precise: the A operands occupy the small accumulator's columns
                    uint32_t& g_buf = small ? g_buf1 : g_buf0;
                    if (g_buf > 0) wait_bar(&bars->dmid_free[small ? 1 : 0], (g_buf - 1) & 1, wsp ? wsp + WS_DMID_FREE : nullptr);   // short: the previous read-out
                    tc_fence_after();
                    const uint32_t idesc = l == 0 ? idesc_mid0 : (l == 1 ? idesc_mid1 : idesc_mid2);
                    const uint64_t dsc = l == 0 ? dsc_mid0 : (l == 1 ? dsc_mid1 : dsc_mid2);
                    const uint32_t a_t = tmem + kColA + (uint32_t)c * C::kACols;
                    const uint32_t d_t = tmem + (small ? kColDmidB : kColDmid);
                    const bool pq_last = (l == p.perq_layer) && (perq_count + 1 == tpq);
                    if (elect_one()) {
                        if (PRECISE) {
                            const uint64_t dsc_lo = dsc + (uint64_t)(((uint32_t)p.mid_N[l] * 128u) >> 4);   // lo image follows hi
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                mma_ts(d_t, a_t + 32 + ks * 8, dsc + (uint64_t)(ks * 16), idesc, ks > 0);     // a_lo * b_hi
                                mma_ts(d_t, a_t + ks * 8, dsc_lo + (uint64_t)(ks * 16), idesc, 1);          // a_hi * b_lo
                                mma_ts(d_t, a_t + ks * 8, dsc + (uint64_t)(ks * 16), idesc, 1);             // a_hi * b_hi
                            }
                        } else {
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks)
                                mma_ts(d_t, a_t + ks * 8, dsc + (uint64_t)(ks * 16), idesc, ks > 0);
                        }
                        mma_commit(&bars->dmid_ready[c]);
                        if (pq_last) mma_commit(&bars->perq_done);
                    }
                    __syncwarp();
                    ++g_mid; ++g_buf; ++rn;
                    if (l == p.perq_layer) ++perq_count;
                    if (++l_m == p.num_mid) { l_m = 0; it_m += 2; }
                };
                if (g_mid & 1) { try_mid(1, it_mid1, l_mid1, rnd1); try_mid(0, it_mid0, l_mid0, rnd0); }
                else { try_mid(0, it_mid0, l_mid0, rnd0); try_mid(1, it_mid1, l_mid1, rnd1); }
            }
        }
    } else if (warp < 4 || (warp >= 9 && warp < 13)) {
        // =============================================================== mid-layer epilogues (two chains)
        const int c = (warp < 4) ? 0 : 1;                 // chain c owns tiles c, c+2, ...; act2 buffer c; A columns c
        const int grp = warp & 3;                         // TMEM lane quarter this warp may access
        const int pt = grp * 32 + lane;                   // point (row) of the tile handled by this thread
        const uint32_t lane_base = (uint32_t)(grp * 32) << 16;
        const uint32_t a_col = tmem + lane_base + kColA + (uint32_t)c * C::kACols;
        uint32_t round = 0;
        for (int it = c; it < ntiles; it += 2) {
            const uint32_t ab = PRECISE ? 0u : (uint32_t)c;                              // activation buffer of this tile
            const uint32_t au = PRECISE ? (uint32_t)it : ((uint32_t)it >> 1);           // its use count
            // ---- mid layers
            int boff = 0;
            for (int l = 0; l < p.num_mid; ++l, ++round) {
                wait_bar(&bars->dmid_ready[c], round & 1, wsp ? wsp + WS_DMID_READY : nullptr);
                tc_fence_after();
                const int N = p.mid_N[l];
                const bool last = (l == p.num_mid - 1);
                if (last) {                         // every MMA that reads this chain's A columns has completed:
                    tc_fence_before();              // the first-layer warps may write the next tile's operand
                    mbar_arrive(&bars->a_free[c]);
                }
                const bool small = !PRECISE && (N == 64);
                const uint32_t dcol = small ? kColDmidB : kColDmid;
                for (int n0 = 0; n0 < N; n0 += 32) {
                    uint32_t r[32];
                    tmem_ld_x32(tmem + lane_base + dcol + n0, r);
                    tmem_ld_wait();
                    if (n0 + 32 >= N) {            // accumulator fully read: hand it to the other chain
                        tc_fence_before();
                        mbar_arrive(&bars->dmid_free[small ? 1 : 0]);
                    }
                    uint32_t v[16], vl[16];
#pragma unroll
                    for (int j4 = 0; j4 < 8; ++j4) {
                        const float4 bb = *reinterpret_cast<const float4*>(s_bias + boff + n0 + 4 * j4);
                        const float2 s01 = fadd2(make_float2(__uint_as_float(r[4 * j4]), __uint_as_float(r[4 * j4 + 1])), make_float2(bb.x, bb.y));
                        const float2 s23 = fadd2(make_float2(__uint_as_float(r[4 * j4 + 2]), __uint_as_float(r[4 * j4 + 3])), make_float2(bb.z, bb.w));
                        if (PRECISE) {
                            pack_relu_split(s01.x, s01.y, v[2 * j4], vl[2 * j4]);
                            pack_relu_split(s23.x, s23.y, v[2 * j4 + 1], vl[2 * j4 + 1]);
                        } else {
                            v[2 * j4] = pack_relu(s01.x, s01.y);
                            v[2 * j4 + 1] = pack_relu(s23.x, s23.y);
                        }
                    }
                    if (!last) {
                        // next layer's A operand (K index = channel, columns hold channel pairs); the MMA that read
                        // this chain's A columns has completed (dmid_ready), so they can be overwritten in place
                        uint32_t w[8];
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) w[j] = v[h * 8 + j];
                            tmem_st_x8(a_col + (uint32_t)(n0 / 2 + h * 8), w);
                            if (PRECISE) {
#pragma unroll
                                for (int j = 0; j < 8; ++j) w[j] = vl[h * 8 + j];
                                tmem_st_x8(a_col + 32u + (uint32_t)(n0 / 2 + h * 8), w);
                            }
                        }
                    } else {
                        // big layer's B operand [point row][channel K] K-major, LBO 128, SBO 2048
                        uint8_t* dst = smem + kOffAct2 + ab * kAct2Bytes + (uint32_t)(pt >> 3) * 2048u + (uint32_t)(pt & 7) * 16u;
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            *reinterpret_cast<uint4*>(dst + (uint32_t)(n0 / 8 + j) * 128u) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                            if (PRECISE)   // lo image of the single activation buffer
                                *reinterpret_cast<uint4*>(dst + kAct2Bytes + (uint32_t)(n0 / 8 + j) * 128u) = make_uint4(vl[4 * j], vl[4 * j + 1], vl[4 * j + 2], vl[4 * j + 3]);
                        }
                    }
                }
                if (!last) {
                    tmem_st_wait();
                    if (l == p.num_mid - 2) wait_bar(&bars->act2_empty[ab], (au & 1) ^ 1, wsp ? wsp + WS_ACT2_EMPTY : nullptr);
                    tc_fence_before();
                    mbar_arrive(&bars->a_ready[c]);
                } else {
                    fence_proxy_async_smem();
                    tc_fence_before();
                    mbar_arrive(&bars->act2_full[ab]);
                }
                boff += N;
            }
        }
    } else if (warp >= 14) {
        // =============================================================== first layer (fp32 FMA) for both chains
        // thread = point = TMEM lane; produces the K = 64 fp16 A operand of the first mid layer of tile `it` in the
        // A columns of chain it & 1 as soon as that chain has released them.
        const int grp = warp & 3;
        const int pt = grp * 32 + lane;
        const int ct = tid - 14 * 32;
        const uint32_t lane_base = (uint32_t)(grp * 32) << 16;
        float* wq = s_wq;
        const float* s_b0 = s_bias + 256;
        int cur_q = -1;
        // loads only: the centring subtraction happens at the use site one tile later, so the loads stay in flight
        auto fetch = [&](int it2, float& x, float& y, float& z, float& cx, float& cy, float& cz) {
            const int qi2 = it2 / tpq, tq2 = it2 - qi2 * tpq;
            const size_t q2 = (size_t)stream + (size_t)qi2 * nstreams;
            const int sgi = tq2 < p.seg[0].tiles ? 0 : 1;
            const Seg& sg = p.seg[sgi];
            int local = (tq2 - (sgi ? p.seg[0].tiles : 0)) * kTile + pt;
            if (local >= sg.n) local = 0;                              // duplicate padding
            const float* src = sg.ptr + (q2 * sg.n + local) * 3;
            x = src[0]; y = src[1]; z = src[2];
            cx = cy = cz = 0.f;
            if (sg.center) { cx = p.query[q2 * 3 + 0]; cy = p.query[q2 * 3 + 1]; cz = p.query[q2 * 3 + 2]; }
        };
        float x = 0.f, y = 0.f, z = 0.f, pcx = 0.f, pcy = 0.f, pcz = 0.f;
        if (ntiles > 0) fetch(0, x, y, z, pcx, pcy, pcz);
        for (int it = 0; it < ntiles; ++it) {
            const int c = it & 1;
            const int qi = it / tpq;
            if (qi != cur_q) {
                // (W0 * R)^T for this query
                const size_t q = (size_t)stream + (size_t)qi * nstreams;
                asm volatile("bar.sync 3, 128;" ::: "memory");      // readers of the previous query's copy are done
                if (ct < 64) {
                    float w0 = p.W0[ct * 3 + 0], w1 = p.W0[ct * 3 + 1], w2 = p.W0[ct * 3 + 2];
                    float r[9] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f};
                    if (p.R) {
#pragma unroll
                        for (int i = 0; i < 9; ++i) r[i] = p.R[q * 9 + i];
                    }
                    wq[0 * 64 + ct] = w0 * r[0] + w1 * r[3] + w2 * r[6];
                    wq[1 * 64 + ct] = w0 * r[1] + w1 * r[4] + w2 * r[7];
                    wq[2 * 64 + ct] = w0 * r[2] + w1 * r[5] + w2 * r[8];
                }
                asm volatile("bar.sync 3, 128;" ::: "memory");
                cur_q = qi;
            }
            x -= pcx; y -= pcy; z -= pcz;              // model.py:303
            uint32_t v[32], vl[PRECISE ? 32 : 1];
#pragma unroll
            for (int j4 = 0; j4 < 16; ++j4) {
                const float4 wx = *reinterpret_cast<const float4*>(wq + 0 * 64 + 4 * j4);
                const float4 wy = *reinterpret_cast<const float4*>(wq + 1 * 64 + 4 * j4);
                const float4 wz = *reinterpret_cast<const float4*>(wq + 2 * 64 + 4 * j4);
                const float4 bb = *reinterpret_cast<const float4*>(s_b0 + 4 * j4);
                // same association as the scalar form fma(wx, x, fma(wy, y, fma(wz, z, b))), two channels per FFMA2
                const float2 xx = make_float2(x, x), yy = make_float2(y, y), zz = make_float2(z, z);
                const float2 h01 = ffma2(make_float2(wx.x, wx.y), xx, ffma2(make_float2(wy.x, wy.y), yy, ffma2(make_float2(wz.x, wz.y), zz, make_float2(bb.x, bb.y))));
                const float2 h23 = ffma2(make_float2(wx.z, wx.w), xx, ffma2(make_float2(wy.z, wy.w), yy, ffma2(make_float2(wz.z, wz.w), zz, make_float2(bb.z, bb.w))));
                if (PRECISE) {
                    pack_relu_split(h01.x, h01.y, v[2 * j4], vl[2 * j4]);
                    pack_relu_split(h23.x, h23.y, v[2 * j4 + 1], vl[2 * j4 + 1]);
                } else {
                    v[2 * j4] = pack_relu(h01.x, h01.y);
                    v[2 * j4 + 1] = pack_relu(h23.x, h23.y);
                }
            }
            if (it + 1 < ntiles) fetch(it + 1, x, y, z, pcx, pcy, pcz);     // next tile's point, in flight during the store
            wait_bar(&bars->a_free[c], (((uint32_t)it >> 1) & 1) ^ 1, wsp ? wsp + WS_A_FREE : nullptr);
            tc_fence_after();
            tmem_st_x32(tmem + lane_base + kColA + (uint32_t)c * C::kACols, v);
            if (PRECISE) {
                uint32_t (&vl32)[32] = reinterpret_cast<uint32_t (&)[32]>(vl);
                tmem_st_x32(tmem + lane_base + kColA + (uint32_t)c * C::kACols + 32u, vl32);
            }
            tmem_st_wait();
            // never trigger the last mid layer's MMA before this chain's act2 buffer is free: its epilogue must not
            // hold the shared D_mid accumulator while waiting for the big layer
            if (p.num_mid == 1) wait_bar(&bars->act2_empty[PRECISE ? 0 : c], ((PRECISE ? (uint32_t)it : ((uint32_t)it >> 1)) & 1) ^ 1, wsp ? wsp + WS_ACT2_EMPTY : nullptr);
            tc_fence_before();
            mbar_arrive(&bars->a_ready[c]);
        }
    } else {
        // =============================================================== big-layer epilogue: max over the tile's points
        const int ew = warp - 4;
        const uint32_t lane_base = (uint32_t)(ew * 32) << 16;
        const int ch_lane = ew * 32 + lane;
        int it = 0;
        for (int qi = 0; qi < nq; ++qi) {
            const int q = stream + qi * nstreams;
            float acc[C::kChunks];
#pragma unroll
            for (int c = 0; c < C::kChunks; ++c) acc[c] = -INFINITY;
            for (int tq = 0; tq < tpq; ++tq, ++it) {
#pragma unroll
                for (int c = 0; c < C::kChunks; ++c) {
                    const uint32_t g = (uint32_t)(it * C::kChunks + c);
                    const uint32_t stage = g & 1, use = g >> 1;
                    wait_bar(&bars->d3_full[stage], use & 1, wsp ? wsp + WS_D3_FULL : nullptr);
                    tc_fence_after();
                    const uint32_t d = tmem + lane_base + kColD3 + stage * 128u;
                    float m = acc[c];
#pragma unroll
                    for (int n0 = 0; n0 < 128; n0 += 64) {
                        uint32_t r0[32], r1[32];
                        tmem_ld_x32(d + n0, r0);
                        tmem_ld_x32(d + n0 + 32, r1);
                        tmem_ld_wait();
                        if (n0 == 64) {             // accumulator fully read: release the stage before reducing
                            tc_fence_before();
                            mbar_arrive(&bars->d3_empty[stage]);
                        }
#pragma unroll
                        for (int j = 0; j < 32; j += 2) m = fmax3(m, __uint_as_float(r0[j]), __uint_as_float(r0[j + 1]));
#pragma unroll
                        for (int j = 0; j < 32; j += 2) m = fmax3(m, __uint_as_float(r1[j]), __uint_as_float(r1[j + 1]));
                    }
                    acc[c] = m;
                }
            }
#pragma unroll
            for (int c = 0; c < C::kChunks; ++c) p.out[(size_t)q * 1024 + (part * C::kChunks + c) * 128 + ch_lane] = acc[c];
        }
    }
    if (STATS) ws_flush(p.wstats, warp == 8 ? 0 : (warp == 13 ? 1 : (warp < 4 ? 2 : (warp >= 14 ? 4 : (warp >= 9 ? 3 : 5)))), ws, t_begin);
    tc_fence_before();
    __syncthreads();
    if (warp == 8) tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------------
// weight packing (device side, once per model)
// ------------------------------------------------------------------------------------------------
// fp32 W[rows][K] -> fp16 K-major no-swizzle operand image: (r/8)*sbo + (k/8)*128 + (r%8)*16 + (k%8)*2
// lo = 1 writes the residual fp16(w - fp16(w)) instead (split-precision images)
__global__ void pack_kmajor_kernel(const float* __restrict__ W, int rows, int K, int row0, uint32_t sbo, uint8_t* __restrict__ img, int lo) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= rows * K) return;
    int r = e / K, k = e % K;
    uint32_t off = (uint32_t)(r >> 3) * sbo + (uint32_t)(k >> 3) * 128u + (uint32_t)(r & 7) * 16u + (uint32_t)(k & 7) * 2u;
    const float w = W[(size_t)(row0 + r) * K + k];
    const __half h = __float2half_rn(w);
    *reinterpret_cast<__half*>(img + off) = lo ? __float2half_rn(w - __half2float(h)) : h;
}

// conv1 folded into the STN's last layer: W1*(T+I) with T = view(fc3(f) + b, 64, 64) is linear in f, so
//   (W1*(T+I))[o][i] = sum_k f[k] * G[o*64+i][k] + g0[o*64+i],
//   G[o*64+i][k] = sum_j W1[o][j] * Wfc3[j*64+i][k],   g0[o*64+i] = sum_j W1[o][j] * bfc3[j*64+i] + W1[o][i].
// One FC layer then yields the per-query operand directly (model.py:62-68,196,201).
__global__ void fold_fc3_kernel(const float* __restrict__ W1, const float* __restrict__ Wfc3, const float* __restrict__ bfc3,
                                float* __restrict__ G, float* __restrict__ g0) {
    const int oi = blockIdx.x;                 // o*64 + i
    const int o = oi >> 6, i = oi & 63;
    const int k = threadIdx.x;                 // 0..255 (fc3 input width)
    float acc = 0.f;
    for (int j = 0; j < 64; ++j) acc = fmaf(W1[o * 64 + j], Wfc3[(size_t)(j * 64 + i) * 256 + k], acc);
    G[(size_t)oi * 256 + k] = acc;
    if (k == 0) {
        float b = W1[o * 64 + i];
        for (int j = 0; j < 64; ++j) b = fmaf(W1[o * 64 + j], bfc3[j * 64 + i], b);
        g0[oi] = b;
    }
}

__global__ void guard_flag_kernel(const float* __restrict__ logits, int64_t B, float band, int32_t* __restrict__ list, int* __restrict__ count, int64_t base, int64_t cap) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    if (fabsf(logits[i * 2 + 1]) < band) {
        int slot = atomicAdd(count, 1);
        if (slot < cap) list[slot] = (int32_t)(base + i);
    }
}

}  // namespace

// ------------------------------------------------------------------------------------------------
struct TcStack {           // one conv stack ending in the 128 -> 1024 layer
    uint8_t* w3_img = nullptr;     // 8 x 32768
    uint8_t* mid_img[3] = {nullptr, nullptr, nullptr};
    uint8_t* w3_img_p = nullptr;   // split precision: 8 x (hi 32768 | lo 32768)
    uint8_t* mid_img_p[3] = {nullptr, nullptr, nullptr};   // split precision: hi | lo
    const float* mid_bias[3] = {nullptr, nullptr, nullptr};
    int mid_N[3] = {0, 0, 0};
    int num_mid = 0;
    const float* W0 = nullptr;
    const float* b0 = nullptr;
    const float* b3 = nullptr;
};

struct TcStnFc {              // tensor-core operand images of an STN's fc1 (1024 -> 512) and fc2 (512 -> 256)
    const uint8_t* fc1 = nullptr;
    const uint8_t* fc2 = nullptr;
};

struct TcWeights {
    TcStack qstn;                // pass A
    TcStack stn[2], fin[2];      // [0] local, [1] global: pass B, pass C
    TcStnFc qstn_fc, stn_fc[2];
    // decoder images: fc1_local / fc1_global (1024 -> 512), fc2 (1024 -> 256), fc3 (256 -> 128)
    const uint8_t* head_fc1[2] = {nullptr, nullptr};
    const uint8_t* head_fc2 = nullptr;
    const uint8_t* head_fc3 = nullptr;
    // conv1 folded into stn2.fc3 per branch: images of G [4096 x 256] and bias g0 [4096]
    const uint8_t* fold_img[2] = {nullptr, nullptr};
    const float* fold_bias[2] = {nullptr, nullptr};
    std::vector<void*> allocs;
    // profile of the dominant kernel (bench.py roofline)
    bool prof_on = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
    double prof_flops = 0.0;
    ~TcWeights() {
        for (void* a : allocs) cudaFree(a);
        for (auto& e : prof_events) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    }
};

namespace {

uint8_t* tc_alloc(TcWeights& t, size_t bytes) {
    void* p = nullptr;
    P2S_CUDA(cudaMalloc(&p, bytes));
    P2S_CUDA(cudaMemset(p, 0, bytes));
    t.allocs.push_back(p);
    return (uint8_t*)p;
}

uint8_t* pack_layer(TcWeights& t, const Layer& L, uint32_t sbo, bool split = false) {   // whole layer as one image (hi [| lo])
    const size_t one = (size_t)L.cout * L.cin * 2;
    uint8_t* img = tc_alloc(t, one * (split ? 2 : 1));
    P2S_LAUNCH(pack_kmajor_kernel, (unsigned)cdiv((int64_t)L.cout * L.cin, 256), 256, 0, 0, L.W, L.cout, L.cin, 0, sbo, img, 0);
    if (split) P2S_LAUNCH(pack_kmajor_kernel, (unsigned)cdiv((int64_t)L.cout * L.cin, 256), 256, 0, 0, L.W, L.cout, L.cin, 0, sbo, img + one, 1);
    return img;
}

uint8_t* pack_w3(TcWeights& t, const Layer& L, bool split = false) {   // 8 chunks of 128 rows, each its own image (hi [| lo])
    P2S_CHECK(L.cout == 1024 && L.cin == 128, "big layer must be 128 -> 1024");
    const size_t chunk = split ? 65536 : 32768;
    uint8_t* img = tc_alloc(t, 8 * chunk);
    for (int c = 0; c < 8; ++c) {
        P2S_LAUNCH(pack_kmajor_kernel, (unsigned)cdiv(128 * 128, 256), 256, 0, 0, L.W, 128, 128, c * 128, 2048u, img + (size_t)c * chunk, 0);
        if (split) P2S_LAUNCH(pack_kmajor_kernel, (unsigned)cdiv(128 * 128, 256), 256, 0, 0, L.W, 128, 128, c * 128, 2048u, img + (size_t)c * chunk + 32768, 1);
    }
    return img;
}

void launch_pass(Model& m, const TcStack& s, const Seg& s0, const Seg& s1, const float* query, const float* R,
                 int64_t B, int perq_layer, const uint8_t* perq_img, float* out, cudaStream_t st, bool precise) {
    PassParams p{};
    p.seg[0] = s0; p.seg[1] = s1;
    p.query = query; p.R = R;
    p.tiles_per_query = s0.tiles + s1.tiles;
    p.B = (int)B;
    p.W0 = s.W0; p.b0 = s.b0;
    p.num_mid = s.num_mid;
    for (int l = 0; l < 3; ++l) { p.mid_N[l] = s.mid_N[l]; p.mid_img[l] = precise ? s.mid_img_p[l] : s.mid_img[l]; p.mid_bias[l] = s.mid_bias[l]; }
    p.perq_layer = perq_layer;
    p.perq_img = perq_img;
    p.w3_img = precise ? s.w3_img_p : s.w3_img;
    p.out = out;
    p.wstats = nullptr;
    TcWeights& t = *m.tc;
    DeviceCtx& ctx = device_ctx();
    static int wstats_on = -1;
    if (wstats_on < 0) { const char* e = getenv("P2S_TC_WAITSTATS"); wstats_on = (e && e[0] == '1') ? 1 : 0; }
    long long* wstats_dev = nullptr;
    if (wstats_on && !precise) {
        wstats_dev = ctx.wait_stats.as<long long>(6 * WS_SLOTS);
        P2S_CUDA(cudaMemsetAsync(wstats_dev, 0, 6 * WS_SLOTS * sizeof(long long), st));
        p.wstats = wstats_dev;
    }
    const int split = precise ? Cfg<true>::kSplit : Cfg<false>::kSplit;
    int streams = ctx.sm_count / split;
    if ((int64_t)streams > B) streams = (int)B;
    const int grid = streams * split;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    const bool prof = t.prof_on && !precise;
    if (prof) {
        P2S_CUDA(cudaEventCreate(&e0)); P2S_CUDA(cudaEventCreate(&e1));
        P2S_CUDA(cudaEventRecord(e0, st));
    }
    if (precise) P2S_LAUNCH(pointnet_pass_kernel<true>, grid, kThreads, Cfg<true>::kSmemBytes, st, p);
    else if (wstats_on) {
        ctx.set_max_dynamic_smem((const void*)pointnet_pass_kernel<false, true>, (int)Cfg<false>::kSmemBytes);
        P2S_LAUNCH((pointnet_pass_kernel<false, true>), grid, kThreads, Cfg<false>::kSmemBytes, st, p);
    } else P2S_LAUNCH(pointnet_pass_kernel<false>, grid, kThreads, Cfg<false>::kSmemBytes, st, p);
    if (wstats_on && !precise) {
        // diagnostics: average wait cycles per warp of each role, as a share of the role's lifetime
        long long h[6 * WS_SLOTS];
        P2S_CUDA(cudaMemcpyAsync(h, wstats_dev, sizeof(h), cudaMemcpyDeviceToHost, st));
        P2S_CUDA(cudaStreamSynchronize(st));
        static const char* const roles[6] = {"big-issuer", "mid-issuer", "chain0", "chain1", "first-layer", "colmax"};
        static const char* const slots[WS_TOTAL] = {"act2_full", "d3_empty", "dmid_free", "dmid_ready", "act2_empty", "a_free", "d3_full"};
        fprintf(stderr, "p2s waitstats: pass num_mid=%d perq=%d pts=%d+%d B=%lld precise=%d grid=%d\n", s.num_mid, perq_layer, s0.n, s1.n, (long long)B, (int)precise, grid);
        for (int r = 0; r < 6; ++r) {
            const double tot = (double)h[r * WS_SLOTS + WS_TOTAL];
            if (tot <= 0) continue;
            fprintf(stderr, "   %-12s", roles[r]);
            for (int i = 0; i < WS_TOTAL; ++i) if (h[r * WS_SLOTS + i]) fprintf(stderr, " %s %.1f%%", slots[i], 100.0 * (double)h[r * WS_SLOTS + i] / tot);
            fprintf(stderr, "  (role cycles per warp %.0f)\n", tot / (grid * (r == 0 || r == 1 ? 1.0 : 4.0)));
        }
    }
    if (prof) {
        P2S_CUDA(cudaEventRecord(e1, st));
        t.prof_events.emplace_back(e0, e1);
        // algorithmic FLOPs of this launch: real (un-padded) points, un-duplicated layers (SURVEY.md section 8d)
        double mac_pt = 3.0 * 64 + 128.0 * 1024;
        int prev = 64;
        for (int l = 0; l < s.num_mid; ++l) { mac_pt += (double)prev * s.mid_N[l]; prev = s.mid_N[l]; }
        t.prof_flops += 2.0 * mac_pt * (double)(s0.n + s1.n) * (double)B;
    }
}

Seg make_seg(const float* ptr, int n, int center) { return Seg{ptr, n, n > 0 ? (n + kTile - 1) / kTile : 0, center}; }

}  // namespace

void tc_build(Model& m) {
    P2S_CHECK(m.cfg.net_size == 1024, "tensor-core path needs net_size 1024");
    TcWeights* t = new TcWeights();
    m.tc = t;
    DeviceCtx& ctx = device_ctx();
    ctx.set_max_dynamic_smem((const void*)pointnet_pass_kernel<false>, (int)Cfg<false>::kSmemBytes);
    ctx.set_max_dynamic_smem((const void*)pointnet_pass_kernel<true>, (int)Cfg<true>::kSmemBytes);
    auto build_stn = [&](TcStack& s, const Stn& stn, const Layer* c0a, const Layer* c0b) {
        // QSTN: x -> conv1(3->64) [layer 0] -> conv2 (64->128) -> conv3 ; STN64 on feat: conv0a [layer 0] -> conv0b -> conv1 -> conv2 -> conv3
        if (!c0a) {
            s.W0 = stn.c1.W; s.b0 = stn.c1.b;
            s.num_mid = 1;
            s.mid_img[0] = pack_layer(*t, stn.c2, 1024); s.mid_bias[0] = stn.c2.b; s.mid_N[0] = 128;
            s.mid_img_p[0] = pack_layer(*t, stn.c2, 1024, true);
        } else {
            s.W0 = c0a->W; s.b0 = c0a->b;
            s.num_mid = 3;
            s.mid_img[0] = pack_layer(*t, *c0b, 1024); s.mid_bias[0] = c0b->b; s.mid_N[0] = 64;
            s.mid_img[1] = pack_layer(*t, stn.c1, 1024); s.mid_bias[1] = stn.c1.b; s.mid_N[1] = 64;
            s.mid_img[2] = pack_layer(*t, stn.c2, 1024); s.mid_bias[2] = stn.c2.b; s.mid_N[2] = 128;
            s.mid_img_p[0] = pack_layer(*t, *c0b, 1024, true);
            s.mid_img_p[1] = pack_layer(*t, stn.c1, 1024, true);
            s.mid_img_p[2] = pack_layer(*t, stn.c2, 1024, true);
        }
        s.w3_img_p = pack_w3(*t, stn.c3, true);
        s.w3_img = pack_w3(*t, stn.c3);
        s.b3 = stn.c3.b;
    };
    auto build_fin = [&](TcStack& s, const Feat& f) {
        s.W0 = f.conv0a.W; s.b0 = f.conv0a.b;
        s.num_mid = 3;
        s.mid_img[0] = pack_layer(*t, f.conv0b, 1024); s.mid_bias[0] = f.conv0b.b; s.mid_N[0] = 64;
        s.mid_img[1] = nullptr; s.mid_bias[1] = f.conv1.b; s.mid_N[1] = 64;       // per query: conv1 * T
        s.mid_img[2] = pack_layer(*t, f.conv2, 1024); s.mid_bias[2] = f.conv2.b; s.mid_N[2] = 128;
        s.mid_img_p[0] = pack_layer(*t, f.conv0b, 1024, true);
        s.mid_img_p[2] = pack_layer(*t, f.conv2, 1024, true);
        s.w3_img_p = pack_w3(*t, f.conv3, true);
        s.w3_img = pack_w3(*t, f.conv3);
        s.b3 = f.conv3.b;
    };
    // every FC layer but the QSTN's fc3 (256 -> 4) and fc4 (128 -> 2) runs on the tensor-core FC kernel; fc_tc_pack checks the shape
    auto mk_stn_fc = [&](const Stn& s) { TcStnFc r; r.fc1 = fc_tc_pack(s.fc1, t->allocs); r.fc2 = fc_tc_pack(s.fc2, t->allocs); return r; };
    if (m.shared_qstn) t->qstn_fc = mk_stn_fc(m.point_stn);
    else if (m.global.has_qstn) t->qstn_fc = mk_stn_fc(m.global.stn1);
    t->stn_fc[0] = mk_stn_fc(m.local.stn2);
    t->stn_fc[1] = mk_stn_fc(m.global.stn2);
    for (int br = 0; br < 2; ++br) {
        const Feat& f = br ? m.global : m.local;
        P2S_CHECK(f.stn2.fc3.cout == 4096 && f.stn2.fc3.cin == 256 && f.conv1.cout == 64 && f.conv1.cin == 64, "unexpected STN shape");
        float* G = reinterpret_cast<float*>(tc_alloc(*t, (size_t)4096 * 256 * 4));
        float* g0 = reinterpret_cast<float*>(tc_alloc(*t, 4096 * 4));
        P2S_LAUNCH(fold_fc3_kernel, 4096, 256, 0, 0, f.conv1.W, f.stn2.fc3.W, f.stn2.fc3.b, G, g0);
        t->fold_img[br] = fc_tc_pack_raw(G, 4096, 256, t->allocs);
        t->fold_bias[br] = g0;
    }
    t->head_fc1[0] = fc_tc_pack(m.fc1_local, t->allocs);
    t->head_fc1[1] = fc_tc_pack(m.fc1_global, t->allocs);
    t->head_fc2 = fc_tc_pack(m.fc2, t->allocs);
    t->head_fc3 = fc_tc_pack(m.fc3, t->allocs);
    if (m.shared_qstn) build_stn(t->qstn, m.point_stn, nullptr, nullptr);
    else if (m.global.has_qstn) build_stn(t->qstn, m.global.stn1, nullptr, nullptr);
    build_stn(t->stn[0], m.local.stn2, &m.local.conv0a, &m.local.conv0b);
    build_stn(t->stn[1], m.global.stn2, &m.global.conv0a, &m.global.conv0b);
    build_fin(t->fin[0], m.local);
    build_fin(t->fin[1], m.global);
    P2S_CUDA(cudaDeviceSynchronize());
}

void tc_destroy(Model& m) {
    delete m.tc;
    m.tc = nullptr;
}

void tc_profile_reset(Model& m, bool on) {
    TcWeights& t = *m.tc;
    for (auto& e : t.prof_events) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    t.prof_events.clear();
    t.prof_flops = 0.0;
    t.prof_on = on;
}

void tc_profile_get(Model& m, double* ms, int64_t* launches, double* flops) {
    TcWeights& t = *m.tc;
    double total = 0.0;
    for (auto& e : t.prof_events) {
        P2S_CUDA(cudaEventSynchronize(e.second));
        float x = 0.f;
        P2S_CUDA(cudaEventElapsedTime(&x, e.first, e.second));
        total += x;
    }
    *ms = total;
    *launches = (int64_t)t.prof_events.size();
    *flops = t.prof_flops;
}

// One pass of the network over B queries on tensor cores.  precise = split-precision operands everywhere
// (the accurate path used for the guard band); fp16 operands otherwise.
void forward_tc(Model& m, const float* patch, const float* sub, const float* query, int64_t B,
                float* logits, cudaStream_t st, bool precise) {
    TcWeights& t = *m.tc;
    const int P = m.cfg.points_per_patch, S = m.cfg.sub_sample_size;
    const int64_t Bc_max = 8192;
    // workspace (floats per query): gmax, f2, q4, R, fmax_l, fmax_g, cat, h4, the 16 KB per-query image (hi | lo) and the
    // A operand images of the FC tails (4 B per element: hi + lo fp16) for K = 1024, 512, 256
    const size_t per_q = 1024 + 256 + 4 + 9 + 1024 * 3 + 128 + 4096 + 1024 + 512 + 256;
    float* base = m.ws_net.as<float>(per_q * (size_t)Bc_max + 1024);
    float* pcur = base;
    auto take = [&](size_t n) { float* r = pcur; pcur += (n * (size_t)Bc_max + 63) / 64 * 64; return r; };
    float* gmax = take(1024); float* f2 = take(256); float* q4 = take(4); float* R = take(9);
    float* fmax_l = take(1024); float* fmax_g = take(1024); float* cat = take(1024); float* h4 = take(128);
    uint8_t* perq = reinterpret_cast<uint8_t*>(take(4096));
    // (Bc_max is a multiple of 128, so every image of Bc_max rows fits its slice)
    uint8_t* imgA = reinterpret_cast<uint8_t*>(take(1024)); uint8_t* imgB = reinterpret_cast<uint8_t*>(take(512)); uint8_t* imgC = reinterpret_cast<uint8_t*>(take(256));
    // FC tails as a chain of operand images: the raw max features are packed once (bias + ReLU on the way), every layer reads
    // its A operand by bulk copy and writes its output as the next layer's image -- no per-N-tile re-conversion of A
    // gmax_raw [Bc,1024] -> relu(+b3) -> fc1 -> fc2; f2 as fp32 rows (out_f2) or as an image in imgC
    auto stn_tail_img = [&](const Stn& s, const TcStnFc& f, const float* gmax_raw, int64_t Bc, float* out_f2) {
        launch_pack_a(gmax_raw, 1024, Bc, 1024, s.c3.b, true, imgA, st);
        launch_fc_tc_img(imgA, f.fc1, s.fc1.b, imgB, 0, Bc, 512, 1024, true, st, 3, 16, 0);
        if (out_f2) launch_fc_tc_img(imgB, f.fc2, s.fc2.b, out_f2, 256, Bc, 256, 512, true, st, 0);
        else launch_fc_tc_img(imgB, f.fc2, s.fc2.b, imgC, 0, Bc, 256, 512, true, st, 3, 8, 0);
    };

    for (int64_t b0 = 0; b0 < B; b0 += Bc_max) {
        const int64_t Bc = (B - b0 < Bc_max) ? (B - b0) : Bc_max;
        const float* pa = patch + b0 * P * 3;
        const float* su = sub + b0 * S * 3;
        const float* qu = query + b0 * 3;
        const float* Rq = nullptr;
        if (m.shared_qstn || m.global.has_qstn) {
            // pass A over cat(patch, sub - q) (shared QSTN, model.py:303,325-327) or over the global branch's sub-sample
            const Stn& qs = m.shared_qstn ? m.point_stn : m.global.stn1;
            const Seg s0 = m.shared_qstn ? make_seg(pa, P, 0) : make_seg(su, S, 1);
            const Seg s1 = m.shared_qstn ? make_seg(su, S, 1) : make_seg(nullptr, 0, 0);
            { StageScope ts("net: pass kernels", st); launch_pass(m, t.qstn, s0, s1, qu, nullptr, Bc, -1, nullptr, gmax, st, precise); }
            { StageScope ts("net: fc tails", st);
              stn_tail_img(qs, t.qstn_fc, gmax, Bc, f2);
              launch_gemm_nt(f2, 0, 256, qs.fc3.W, 0, qs.fc3.b, q4, 0, 4, (int)Bc, qs.fc3.cout, qs.fc3.cin, 1, false, st); }
            launch_quat_to_rot(q4, R, Bc, st);
            Rq = R;
        }
        for (int br = 1; br >= 0; --br) {    // global first like the reference, then local
            const Feat& f = br ? m.global : m.local;
            const Seg sg = br ? make_seg(su, S, 1) : make_seg(pa, P, 0);
            float* fmax = br ? fmax_g : fmax_l;
            // pass B: STN64 -> T
            { StageScope ts("net: pass kernels", st); launch_pass(m, t.stn[br], sg, make_seg(nullptr, 0, 0), qu, Rq, Bc, -1, nullptr, gmax, st, precise); }
            {   // fc1, fc2, then the folded last layer writes the per-query fp16 operand images of conv1*(T+I) directly
                StageScope ts("net: fc tails", st);
                stn_tail_img(f.stn2, t.stn_fc[br], gmax, Bc, nullptr);
                launch_fc_tc_img(imgC, t.fold_img[br], t.fold_bias[br], perq, 0, Bc, 4096, 256, false, st, precise ? 2 : 1);
            }
            // pass C: final stack -> max feature (bias, no ReLU: model.py:203,210-212)
            { StageScope ts("net: pass kernels", st); launch_pass(m, t.fin[br], sg, make_seg(nullptr, 0, 0), qu, Rq, Bc, 1, perq, fmax, st, precise); }
        }
        // max features = raw max + conv3 bias, no ReLU (model.py:203,210-212): the bias is added while packing fc1's operand image.
        // cat(local, global) (model.py:335,343,346) is the K = 1024 operand image of fc2: k-steps 0-15 local, 16-31 global
        StageScope ts_head("net: fc tails", st);
        uint8_t* imgCat = reinterpret_cast<uint8_t*>(cat);            // [Bc,1024] x 4 B: same footprint as fp32 rows
        launch_pack_a(fmax_l, 1024, Bc, 1024, m.local.conv3.b, false, imgA, st);
        launch_fc_tc_img(imgA, t.head_fc1[0], m.fc1_local.b, imgCat, 0, Bc, 512, 1024, true, st, 3, 32, 0);
        launch_pack_a(fmax_g, 1024, Bc, 1024, m.global.conv3.b, false, imgA, st);
        launch_fc_tc_img(imgA, t.head_fc1[1], m.fc1_global.b, imgCat, 0, Bc, 512, 1024, true, st, 3, 32, 16);
        if (m.debug_aux) {      // exported features: the bias is added in place once both images are packed
            launch_bias_act(fmax_l, m.local.conv3.b, Bc, 1024, false, st);
            launch_bias_act(fmax_g, m.global.conv3.b, Bc, 1024, false, st);
            debug_aux_copy(m, b0, Bc, Rq, fmax_l, fmax_g, st);
        }
        launch_fc_tc_img(imgCat, t.head_fc2, m.fc2.b, imgC, 0, Bc, 256, 1024, true, st, 3, 8, 0);
        launch_fc_tc_img(imgC, t.head_fc3, m.fc3.b, h4, 128, Bc, 128, 256, true, st, 0);
        launch_gemm_nt(h4, 0, 128, m.fc4.W, 0, m.fc4.b, logits + b0 * 2, 0, 2, (int)Bc, 2, 128, 1, false, st);
    }
}

// appends base + i to list[0..cap) for every query i < B whose |sign logit| < band; *count counts them
void guard_flag(const float* logits, int64_t B, float band, int64_t base, int32_t* list, int* count, int64_t cap, cudaStream_t st) {
    P2S_LAUNCH(guard_flag_kernel, (unsigned)cdiv(B, 256), 256, 0, st, logits, B, band, list, count, base, cap);
}

}  // namespace p2s
