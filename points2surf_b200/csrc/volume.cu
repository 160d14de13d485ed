// K6 / K7: SDF epilogue, scatter into the dense volume, iterative sign propagation.
//   post_process + combine       source/sdf_nn.py:11-21, source/points_to_surf_eval.py:184-196,263-271,205-207
//   add_samples_to_volume        source/sdf.py:82-111 (reconstruction case: one sample per voxel -> scatter)
//   propagate_sign               source/sdf.py:114-178
//   clamp                        source/sdf.py:200-202
// Signs are int8; the box sums are exact integers (the reference's float sums of {-1,0,1} are too), so the
// result is bit-identical to the reference.  Sign propagation is one persistent cooperative kernel over a work list of
// tiles along the propagating front (see propagate_kernel); section 8d counts it as res^3 * 2 B per iteration.
#include "common.cuh"
#include <algorithm>
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

namespace p2s {

namespace {

__global__ void sdf_from_logits_kernel(const float* __restrict__ logits, const float* __restrict__ radius,
                                       int64_t B, float* __restrict__ sdf) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    float t = tanhf(logits[i * 2 + 0]);
    float mag = __fmul_rn(t, t);
    if (radius) mag = __fmul_rn(mag, radius[i]);
    float v = logits[i * 2 + 1] >= 0.0f ? mag : -mag;
    if (isnan(v)) v = 1.0f;  // points_to_surf_eval.py:205-207
    sdf[i] = v;
}


struct Ctrl {
    // every counter that many CTAs update in the same iteration sits on its own 128-byte line (same-line atomics serialise in L2)
    struct alignas(128) Slot { long long dN, dS; unsigned listCount; unsigned pad[27]; unsigned cursor; } slot[3];   // rotating per-iteration accumulators / work-list sizes
    alignas(128) unsigned long long cntS0;   // zero count of the initial sign volume
    int iters;                  // applied iterations (result)
    int final_buf;              // which ping-pong buffer holds the final signs (result)
    int error;                  // 1: iteration cap hit
    unsigned nonzero_seen;      // some sample is not exactly 0 (sdf.py:187-189)
    unsigned bad_index;         // scatter: number of voxel indices outside [0, res^3)
    unsigned long long visits;  // tile evaluations (diagnostics)
    unsigned long long t_total, t_sync, t_first;   // diagnostics (ns, block 0): kernel, time inside grid.sync(), first iteration
};

__global__ void any_nonzero_kernel(const float* __restrict__ sdf, int64_t Q, Ctrl* c) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool nz = (i < Q) && (sdf[i] != 0.0f);
    if (__any_sync(0xffffffffu, nz) && (threadIdx.x & 31) == 0) atomicOr(&c->nonzero_seen, 1u);
}

// block-wide sum of v, ONE atomic per block.  Every thread of the block must call it.
__device__ __forceinline__ void block_count_add(unsigned v, unsigned long long* dst) {
    __shared__ unsigned warp_sum[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
        unsigned t = threadIdx.x < (blockDim.x >> 5) ? warp_sum[threadIdx.x] : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (threadIdx.x == 0 && t) atomicAdd(dst, (unsigned long long)t);
    }
}

// Sign byte: bits 0-1 = sign in two's complement (0, +1 = 1, -1 = 3), bit 2 = "unknown at the start" (U0).
constexpr uint8_t kU0 = 4u;
__device__ __forceinline__ int sign_of(uint8_t b) { return (int)((int8_t)(b << 6)) >> 6; }

// A = (sign(vol), U0 = (sign == 0)), then the six border faces of vol (not of the signs) are set to -1  (sdf.py:144-154)
__global__ void init_sign_kernel(float* __restrict__ vol, int res, uint8_t* __restrict__ A, Ctrl* c) {
    int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t V = (int64_t)res * res * res;
    unsigned z = 0;
    if (v < V) {
        float x = vol[v];
        int s = x > 0.f ? 1 : (x < 0.f ? -1 : 0);
        A[v] = (uint8_t)((s & 3) | (s == 0 ? kU0 : 0));
        z = (s == 0);
        int iz = (int)(v % res), iy = (int)((v / res) % res), ix = (int)(v / ((int64_t)res * res));
        if (ix == 0 || iy == 0 || iz == 0 || ix == res - 1 || iy == res - 1 || iz == res - 1) vol[v] = -1.0f;
    }
    block_count_add(z, &c->cntS0);
}

// iteration 0 evaluates every tile
__global__ void init_tiles_kernel(int* __restrict__ list0, int* __restrict__ voteZeros, int numTiles, Ctrl* c) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < numTiles) { list0[t] = t; voteZeros[t] = 0; }
    if (t == 0) c->slot[0].listCount = (unsigned)numTiles;
}

// ---- iterative sign propagation (sdf.py:156-178) as ONE persistent cooperative kernel -----------------------------------
// The reference recomputes the 5^3 box vote of the whole volume in every iteration (~0.3 res iterations).  A vote only changes
// where a sign inside its box changed in the previous iteration, and signs change only along the propagating front, so the
// kernel keeps a work list of 8x8x32-voxel tiles whose neighbourhood changed and re-evaluates only those; the zero counts
// behind the reference's two stop rules (`unknown_before.sum() == 0`, `unknown_after.sum() >= unknown_before.sum()`) are
// maintained incrementally (per-tile zero count of the vote, deltas of the sign zero count), so decisions and iteration
// counts are identical to the full recomputation.  Signs ping-pong between two byte volumes: a tile that is not on the work
// list has identical content in both (its last evaluation reproduced its input), a listed tile rewrites the output volume
// completely, and a rejected last iteration is discarded by picking the input volume.  One grid-wide barrier per iteration;
// the stop rule never leaves the device.
constexpr int TX = 8, TY = 8, TZ = 32, kPropThreads = 256;

struct PropParams {
    uint8_t* buf[2];
    int* list[3];
    uint8_t* flags[2];
    int* voteZeros;
    Ctrl* ctrl;
    int res, lo, hi, ntx, nty, ntz, maxIters, words, fast, vec;
    float thr;
};

// SIGMA5 = true: the reference's default sigma (lo = -2, hi = 2) with every loop bound a compile-time constant
template <bool SIGMA5>
__global__ void __launch_bounds__(kPropThreads, 4) propagate_kernel(PropParams p) {
    cg::grid_group grid = cg::this_grid();
    extern __shared__ __align__(16) uint8_t smem[];
    const int res = p.res, hl = SIGMA5 ? 2 : -p.lo, hh = SIGMA5 ? 2 : p.hi, W = hl + hh + 1;
    const int X0 = TX + hl + hh, Y0 = TY + hl + hh, Z0 = TZ + hl + hh;
    const int HW = (max(hl, hh) + 3) >> 2, WPR = TZ / 4 + 2 * HW;     // halo words per side, words per row
    const int ZS = 4 * WPR, zoff = 4 * HW - hl;                        // row stride in bytes; smem byte zoff <-> z = bz - hl
    uint8_t* s0 = smem;                                                 // [X0][Y0][ZS] sign bytes (with U0 flag)
    int8_t* t1 = (int8_t*)(smem + ((X0 * Y0 * ZS + 15) & ~15));         // [X0][Y0][TZ] z sums (|.| <= 11)
    int16_t* t2 = (int16_t*)((uint8_t*)t1 + ((X0 * Y0 * TZ + 15) & ~15));   // [X0][TY][TZ] zy sums (|.| <= 121)
    __shared__ int sh[8];   // 0 dS, 1 voteZeros, 2..7 changed bbox (min x,y,z, max x,y,z)
    __shared__ int sh_count, sh_next[2][2];   // [parity][0: list position, 1: tile] of the tile after the current one
    __shared__ uint16_t rowxy[(TX + 10) * (TY + 10)];   // halo row -> (x << 8) | y
    __shared__ long long sh_d[2];
    const int tid = threadIdx.x;
    for (int r = tid; r < X0 * Y0; r += kPropThreads) rowxy[r] = (uint16_t)(((r / Y0) << 8) | (r % Y0));
    const int ithr = p.thr > 0.f ? (int)ceilf(p.thr) : 0;               // |n| < thr  <=>  |n| < ceil(thr) for integer n
    long long totalN = 0;                                               // zero count of the vote (whole volume)
    long long totalS = (long long)__ldcg(&p.ctrl->cntS0);               // zero count of the signs
    int iters = 0, final_buf = 0, error = 0;
    long long ctaN = 0, ctaS = 0;                                        // thread 0: this CTA's share of the iteration's counter changes
    unsigned long long ctaVisits = 0;
    auto now_ns = [] { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; };
    const bool diag = blockIdx.x == 0 && tid == 0;
    const unsigned long long t_begin = diag ? now_ns() : 0ull;
    unsigned long long t_sync = 0;
    for (int it = 0;; ++it) {
        const int cur = it % 3, nxt = (it + 1) % 3;
        if (totalS == 0) { final_buf = it & 1; break; }                 // `if unknown_before.sum() == 0: break`
        if (it >= p.maxIters) { final_buf = it & 1; error = 1; break; }
        if (blockIdx.x == 0 && tid == 0) {                              // recycle the accumulators of iteration it+1 / it+2
            p.ctrl->slot[nxt].dN = 0; p.ctrl->slot[nxt].dS = 0; p.ctrl->slot[(it + 2) % 3].listCount = 0; p.ctrl->slot[(it + 2) % 3].cursor = 0;
        }
        // (selects instead of indexing the parameter struct: a runtime index would spill it to local memory)
        const uint8_t* __restrict__ in = (it & 1) ? p.buf[1] : p.buf[0];
        uint8_t* __restrict__ out = (it & 1) ? p.buf[0] : p.buf[1];
        // one reader per CTA; tiles are handed out dynamically (a static stride left CTAs waiting ~30 % of the time at the
        // barrier): thread 0 draws the next list position while the current tile is being evaluated
        const int* list = cur == 0 ? p.list[0] : (cur == 1 ? p.list[1] : p.list[2]);
        if (tid == 0) {
            const int k0 = (int)atomicAdd(&p.ctrl->slot[cur].cursor, 1u);
            const int cnt = (int)__ldcg(&p.ctrl->slot[cur].listCount);
            sh_count = cnt; sh_next[0][0] = k0; sh_next[0][1] = k0 < cnt ? __ldcg(&list[k0]) : -1;
        }
        __syncthreads();
        const int count = sh_count;
        int* listNext = nxt == 0 ? p.list[0] : (nxt == 1 ? p.list[1] : p.list[2]);
        uint8_t* flagCur = (it & 1) ? p.flags[1] : p.flags[0];
        uint8_t* flagNext = (it & 1) ? p.flags[0] : p.flags[1];
        // Per tile the global-memory round trips that used to be exposed one after the other (list entry, three passes of halo
        // loads, the tile's vote-zero count, the neighbour flags, the list append) are overlapped: thread 0 draws the next list
        // position first, the halo loads go out in one batch, the next tile id and the old zero count are fetched behind them, and
        // warp 0 marks the neighbours while the other warps already load the next tile (double-buffered hand-over slot).
        int par = 0;
        for (int k = sh_next[0][0]; k < count; k = sh_next[par][0]) {
            const int tile = sh_next[par][1];
            int knext = 0, oldvz = 0;
            if (tid == 0) knext = (int)atomicAdd(&p.ctrl->slot[cur].cursor, 1u);
            auto prefetch_next = [&] {      // thread 0, right behind the halo loads
                oldvz = __ldcg(&p.voteZeros[tile]);
                const int tn = knext < count ? __ldcg(&list[knext]) : -1;
                sh_next[par ^ 1][0] = knext; sh_next[par ^ 1][1] = tn;
            };
            const int tz = tile % p.ntz, ty = (tile / p.ntz) % p.nty, tx = tile / (p.ntz * p.nty);
            const int bx = tx * TX, by = ty * TY, bz = tz * TZ;
            if (tid < 8) sh[tid] = tid < 2 ? 0 : (tid < 5 ? 1 << 20 : -1);
            if (tid == 0) flagCur[tile] = 0;
            if (SIGMA5 && p.vec) {
                // ---- row-vector path (sigma 5, res a multiple of 32: every tile is full and rows are 16-byte aligned).
                // The packed-word path below is ISSUE-bound (ncu: 2.6 IPC, 8.8 k warp instructions per tile, the volume in L2):
                // most of its instructions are per-word address arithmetic.  Here one thread owns a whole halo ROW: one address,
                // two 16-byte loads + two halo words, the z sums of the row straight from registers; the y and x sums are
                // sliding windows down a column (2 packed adds per output instead of 5 loads + 4 adds), the vote is evaluated
                // on packed bytes (carry tricks on 16-bit lanes).  ~2 k warp instructions per tile.
                constexpr int kT1X = 104, kT2X = 72;                                // padded x strides (bank-conflict-free)
                uint32_t* sraw = reinterpret_cast<uint32_t*>(smem);                // [TX*TY][8]   raw bytes (sign | U0) of the tile
                uint32_t* t1w = sraw + TX * TY * 8;                                 // [12][kT1X]   sums along z   ([x][y][8])
                uint32_t* t2w = t1w + 12 * kT1X;                                    // [12][kT2X]   sums along z, y ([x][y][8])
                const unsigned rw = (unsigned)(res >> 2);
                if (tid < 144) {
                    const int x = tid / 12, y = tid - 12 * x;
                    const int gx = min(max(bx + x - 2, 0), res - 1), gy = min(max(by + y - 2, 0), res - 1);
                    const uint32_t* rowp = reinterpret_cast<const uint32_t*>(in) + (unsigned)(gx * res + gy) * rw + (unsigned)(bz >> 2);
                    const uint4 a = __ldcg(reinterpret_cast<const uint4*>(rowp));
                    const uint4 b = __ldcg(reinterpret_cast<const uint4*>(rowp) + 1);
                    const bool lft = bz > 0, rgt = bz + TZ < res;
                    uint32_t hl_w = lft ? __ldcg(rowp - 1) : 0u, hr_w = rgt ? __ldcg(rowp + 8) : 0u;
                    if (tid == 0) prefetch_next();
                    if (!lft) hl_w = (a.x & 0xffu) * 0x01010101u;                   // 'nearest': first voxel of the row
                    if (!rgt) hr_w = (b.w >> 24) * 0x01010101u;                     // last voxel of the row
                    if ((unsigned)(x - 2) < (unsigned)TX && (unsigned)(y - 2) < (unsigned)TY) {
                        uint4* d = reinterpret_cast<uint4*>(sraw + ((x - 2) * TY + (y - 2)) * 8);
                        d[0] = a; d[1] = b;
                    }
                    uint32_t c[10] = {hl_w, a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, hr_w};
#pragma unroll
                    for (int i = 0; i < 10; ++i) c[i] = ((c[i] & 0x03030303u) + 0x01010101u) & 0x03030303u;     // 2-bit sign -> sign + 1
                    uint32_t o[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        o[j] = __funnelshift_r(c[j], c[j + 1], 16) + __funnelshift_r(c[j], c[j + 1], 24) + c[j + 1] +
                               __funnelshift_r(c[j + 1], c[j + 2], 8) + __funnelshift_r(c[j + 1], c[j + 2], 16);
                    uint4* d = reinterpret_cast<uint4*>(t1w + x * kT1X + y * 8);
                    d[0] = make_uint4(o[0], o[1], o[2], o[3]); d[1] = make_uint4(o[4], o[5], o[6], o[7]);
                }
                __syncthreads();
                if (tid < 96) {                                                     // sums along y: thread = (x, word), window slides down y
                    const int j = tid & 7, x = tid >> 3;
                    const uint32_t* r = t1w + x * kT1X + j;
                    uint32_t v[12];
#pragma unroll
                    for (int y = 0; y < 12; ++y) v[y] = r[y * 8];
                    uint32_t acc = v[0] + v[1] + v[2] + v[3] + v[4];
                    uint32_t* w = t2w + x * kT2X + j;
                    w[0] = acc;
#pragma unroll
                    for (int y = 1; y < 8; ++y) { acc = acc - v[y - 1] + v[y + 4]; w[y * 8] = acc; }   // bytes never borrow: v[y-1] is part of acc
                }
                __syncthreads();
                {   // sums along x, vote, apply: thread = (x pair, y, word)
                    const int j = tid & 7, y = (tid >> 3) & 7, x0 = (tid >> 6) * 2;
                    const uint32_t* r = t2w + x0 * kT2X + y * 8 + j;
                    const uint32_t v0 = r[0], v1 = r[kT2X], v2 = r[2 * kT2X], v3 = r[3 * kT2X], v4 = r[4 * kT2X], v5 = r[5 * kT2X];
                    const uint32_t sum0 = v0 + v1 + v2 + v3 + v4;
                    const uint32_t sumv[2] = {sum0, sum0 - v0 + v5};
                    // vote per byte: n = sum - 125; +1 iff n >= T, -1 iff n <= -T with T = max(ceil(thr), 1) (|n| < thr or n == 0 -> 0)
                    const int T = min(max(ithr, 1), 126);
                    const uint32_t cpos = (uint32_t)(0x100 - (125 + T)) * 0x00010001u, cneg = (uint32_t)(0x100 + 125 - T) * 0x00010001u;
                    int dS = 0, nz = 0, mnx = 1 << 20, mxx = -1, mny = 1 << 20, mxy = -1, mnz = 1 << 20, mxz = -1;
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        const int x = x0 + u;
                        const uint32_t sum = sumv[u];
                        const uint32_t e = sum & 0x00ff00ffu, o = (sum >> 8) & 0x00ff00ffu;
                        const uint32_t pe = ((e + cpos) >> 8) & 0x00010001u, po = ((o + cpos) >> 8) & 0x00010001u;
                        const uint32_t ne = ((cneg - e) >> 8) & 0x00010001u, no = ((cneg - o) >> 8) & 0x00010001u;
                        nz += 4 - __popc(pe | ne) - __popc(po | no);
                        const uint32_t ve = pe | (ne * 3u), vo = po | (no * 3u);
                        const uint32_t cand = ve | (vo << 8) | 0x04040404u;         // the four votes as sign bytes with the U0 flag
                        const uint32_t raw = sraw[(x * TY + y) * 8 + j];
                        const uint32_t um = ((raw >> 2) & 0x01010101u) * 0xffu;     // 0xff in the bytes that were unknown at the start
                        const uint32_t neww = (raw & ~um) | (cand & um);
                        reinterpret_cast<uint32_t*>(out)[(unsigned)((bx + x) * res + by + y) * rw + (unsigned)((bz >> 2) + j)] = neww;
                        const uint32_t diff = neww ^ raw;
                        if (diff) {                                               // rare: signs change only along the front
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                if ((diff >> (8 * q)) & 0xffu) {
                                    dS += (int)(((neww >> (8 * q)) & 3u) == 0u) - (int)(((raw >> (8 * q)) & 3u) == 0u);
                                    const int z = 4 * j + q;
                                    mnx = min(mnx, x); mxx = max(mxx, x); mny = min(mny, y); mxy = max(mxy, y); mnz = min(mnz, z); mxz = max(mxz, z);
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) { dS += __shfl_xor_sync(0xffffffffu, dS, o); nz += __shfl_xor_sync(0xffffffffu, nz, o); }
                    if (__any_sync(0xffffffffu, mxx >= 0)) {                       // one set of shared atomics per warp, not per voxel
                        mnx = __reduce_min_sync(0xffffffffu, mnx); mxx = __reduce_max_sync(0xffffffffu, mxx);
                        mny = __reduce_min_sync(0xffffffffu, mny); mxy = __reduce_max_sync(0xffffffffu, mxy);
                        mnz = __reduce_min_sync(0xffffffffu, mnz); mxz = __reduce_max_sync(0xffffffffu, mxz);
                        if ((tid & 31) == 0) {
                            atomicMin(&sh[2], mnx); atomicMax(&sh[5], mxx); atomicMin(&sh[3], mny); atomicMax(&sh[6], mxy);
                            atomicMin(&sh[4], mnz); atomicMax(&sh[7], mxz);
                        }
                    }
                    if ((tid & 31) == 0) { if (dS) atomicAdd(&sh[0], dS); if (nz) atomicAdd(&sh[1], nz); }
                }
            } else if (SIGMA5 || p.fast) {
                // ---- fast path (word-aligned rows, sigma <= 5): four voxels per 32-bit word everywhere.  Signs are held BIASED
                // (sign + 1 in {0,1,2}) so that plain integer adds on packed words are exact box sums: no byte ever exceeds
                // 2 * 5^3 = 250, so nothing carries into its neighbour.  (The byte-at-a-time version spent ~24 k warp
                // instructions per tile, 60 per z-sum output, and was issue-bound at 9 ms per 256^3 volume.)
                uint32_t* sb = reinterpret_cast<uint32_t*>(smem);                 // [X0*Y0][WPR] biased signs, tile + halo
                uint32_t* sraw = sb + X0 * Y0 * WPR;                               // [TX*TY][8]   raw bytes (sign | U0) of the tile
                uint32_t* t1w = sraw + TX * TY * 8;                                // [X0*Y0][8]   sums along z
                uint32_t* t2w = t1w + X0 * Y0 * 8;                                 // [X0*TY][8]   sums along z, y
                const int zw0 = (bz >> 2) - HW, lastw = (res >> 2) - 1, rows = X0 * Y0;
                const int lane16 = tid & 15, rsub = tid >> 4;                     // 16 lanes per row, 16 rows per pass
                // tile + halo, edges replicated ('nearest'); .cg loads: other SMs wrote these words in the previous iteration.
                // Row -> (x, y) comes from a table built once per kernel (two runtime divisions per word made this phase half
                // of the kernel's instructions); offsets are 32-bit (res^3 <= 2^30).
                constexpr int kBatch = SIGMA5 ? 9 : 4;                            // sigma 5: all 144 rows of the tile in ONE batch of loads
                for (int r0 = 0; r0 < rows; r0 += 16 * kBatch) {
                    uint32_t v[kBatch];
#pragma unroll
                    for (int u = 0; u < kBatch; ++u) {                            // independent loads in flight
                        const int row = r0 + 16 * u + rsub;
                        v[u] = 0;
                        if (row < rows && lane16 < WPR) {
                            const unsigned xy = rowxy[row];
                            const int gx = min(max(bx + (int)(xy >> 8) - hl, 0), res - 1), gy = min(max(by + (int)(xy & 0xffu) - hl, 0), res - 1);
                            const unsigned wofs = (unsigned)(gx * res + gy) * (unsigned)(res >> 2) + (unsigned)min(max(zw0 + lane16, 0), lastw);
                            v[u] = __ldcg(reinterpret_cast<const uint32_t*>(in) + wofs);
                        }
                    }
                    if (tid == 0 && r0 == 0) prefetch_next();
#pragma unroll
                    for (int u = 0; u < kBatch; ++u) {
                        const int row = r0 + 16 * u + rsub;
                        if (row < rows && lane16 < WPR) {
                            const int gzw = zw0 + lane16;
                            uint32_t raw = v[u];
                            if (gzw < 0) raw = (raw & 0xffu) * 0x01010101u;           // left of the volume: first voxel of the row
                            else if (gzw > lastw) raw = (raw >> 24) * 0x01010101u;    // right of it: last voxel
                            sb[row * WPR + lane16] = ((raw & 0x03030303u) + 0x01010101u) & 0x03030303u;   // 2-bit sign -> sign + 1
                            const unsigned xy = rowxy[row];
                            const unsigned xi = (xy >> 8) - (unsigned)hl, yi = (xy & 0xffu) - (unsigned)hl, wi = (unsigned)(lane16 - HW);
                            if (xi < (unsigned)TX && yi < (unsigned)TY && wi < 8u) sraw[(xi * TY + yi) * 8 + wi] = raw;
                        }
                    }
                }
                __syncthreads();
                {   // sums along z: output word j of a row = sum over t of the word starting at byte zoff + 4 j + t
                    const int s = zoff & 3, jb0 = zoff >> 2;
                    for (int i = tid; i < rows * 8; i += kPropThreads) {
                        const int row = i >> 3, j = (i & 7) + jb0;
                        const uint32_t* r = sb + row * WPR + j;
                        const uint32_t w0 = r[0], w1 = (j + 1 < WPR) ? r[1] : 0u, w2 = (j + 2 < WPR) ? r[2] : 0u;
                        uint32_t acc = 0;
#pragma unroll
                        for (int t = 0; t < W; ++t) {
                            const int k = s + t;
                            acc += __funnelshift_r(k < 4 ? w0 : w1, k < 4 ? w1 : w2, (k & 3) * 8);
                        }
                        t1w[i] = acc;
                    }
                }
                __syncthreads();
                for (int i = tid; i < X0 * TY * 8; i += kPropThreads) {            // sums along y
                    const int j = i & 7, y = (i >> 3) & (TY - 1), x = i >> 6;
                    const uint32_t* r = t1w + ((x * Y0 + y) << 3) + j;
                    uint32_t acc = 0;
#pragma unroll
                    for (int t = 0; t < W; ++t) acc += r[t << 3];
                    t2w[i] = acc;
                }
                __syncthreads();
                {   // sums along x, threshold, apply
                    const int bias = W * W * W;                                 // every tap carries +1
                    int dS = 0, nz = 0, mnx = 1 << 20, mxx = -1, mny = 1 << 20, mxy = -1, mnz = 1 << 20, mxz = -1;
                    for (int i = tid; i < TX * TY * 8; i += kPropThreads) {
                        const int j = i & 7, y = (i >> 3) & (TY - 1), x = i >> 6;
                        const int gx = bx + x, gy = by + y, gzw = (bz >> 2) + j;
                        if (gx >= res || gy >= res || gzw > lastw) continue;
                        const uint32_t* r = t2w + ((x * TY + y) << 3) + j;
                        uint32_t sum = 0;
#pragma unroll
                        for (int t = 0; t < W; ++t) sum += r[(t * TY) << 3];
                        const uint32_t raw = sraw[i];
                        uint32_t cand = 0;                                        // the four votes as sign bytes with the U0 flag
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int n = (int)((sum >> (8 * q)) & 0xffu) - bias;
                            const int vote = (abs(n) < ithr || n == 0) ? 0 : (n > 0 ? 1 : 3);      // 2-bit two's complement
                            nz += (vote == 0);
                            cand |= (uint32_t)(vote | kU0) << (8 * q);
                        }
                        const uint32_t um = ((raw >> 2) & 0x01010101u) * 0xffu;     // 0xff in the bytes that were unknown at the start
                        const uint32_t neww = (raw & ~um) | (cand & um);
                        reinterpret_cast<uint32_t*>(out)[(unsigned)(gx * res + gy) * (unsigned)(res >> 2) + (unsigned)gzw] = neww;
                        const uint32_t diff = neww ^ raw;
                        if (diff) {                                               // rare: signs change only along the front
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                if ((diff >> (8 * q)) & 0xffu) {
                                    dS += (int)(((neww >> (8 * q)) & 3u) == 0u) - (int)(((raw >> (8 * q)) & 3u) == 0u);
                                    const int z = 4 * j + q;
                                    mnx = min(mnx, x); mxx = max(mxx, x); mny = min(mny, y); mxy = max(mxy, y); mnz = min(mnz, z); mxz = max(mxz, z);
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) { dS += __shfl_xor_sync(0xffffffffu, dS, o); nz += __shfl_xor_sync(0xffffffffu, nz, o); }
                    if (__any_sync(0xffffffffu, mxx >= 0)) {                       // one set of shared atomics per warp, not per voxel
                        mnx = __reduce_min_sync(0xffffffffu, mnx); mxx = __reduce_max_sync(0xffffffffu, mxx);
                        mny = __reduce_min_sync(0xffffffffu, mny); mxy = __reduce_max_sync(0xffffffffu, mxy);
                        mnz = __reduce_min_sync(0xffffffffu, mnz); mxz = __reduce_max_sync(0xffffffffu, mxz);
                        if ((tid & 31) == 0) {
                            atomicMin(&sh[2], mnx); atomicMax(&sh[5], mxx); atomicMin(&sh[3], mny); atomicMax(&sh[6], mxy);
                            atomicMin(&sh[4], mnz); atomicMax(&sh[7], mxz);
                        }
                    }
                    if ((tid & 31) == 0) { if (dS) atomicAdd(&sh[0], dS); if (nz) atomicAdd(&sh[1], nz); }
                }
            } else {
                // tile + halo, edges replicated ('nearest'); .cg loads: other SMs wrote these bytes in the previous iteration, L1 may
                // hold stale lines.  Rows are fetched as aligned 32-bit words, four independent loads in flight per thread (a byte
                // per load made the kernel latency-bound at ~0.4 TB/s); resolutions that are not a multiple of 4 take byte loads.
                if (tid == 0) prefetch_next();
                if (p.words) {
                    const int total = X0 * Y0 * WPR, zw0 = (bz >> 2) - HW, lastw = (res >> 2) - 1;
                    uint32_t* s0w = reinterpret_cast<uint32_t*>(s0);
                    for (int base = 0; base < total; base += 4 * kPropThreads) {
                        uint32_t w[4];
                        int gz[4];
    #pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const int i = base + k * kPropThreads + tid;
                            w[k] = 0; gz[k] = 0;
                            if (i < total) {
                                const int row = i / WPR, wi = i - row * WPR, x = row / Y0, y = row - x * Y0;
                                const int gx = min(max(bx + x - hl, 0), res - 1), gy = min(max(by + y - hl, 0), res - 1);
                                gz[k] = zw0 + wi;
                                w[k] = __ldcg(reinterpret_cast<const uint32_t*>(in + ((size_t)gx * res + gy) * res) + min(max(gz[k], 0), lastw));
                            }
                        }
    #pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const int i = base + k * kPropThreads + tid;
                            if (i < total) {
                                uint32_t v = w[k];
                                if (gz[k] < 0) v = (v & 0xffu) * 0x01010101u;            // left of the volume: first voxel of the row
                                else if (gz[k] > lastw) v = (v >> 24) * 0x01010101u;     // right of it: last voxel
                                s0w[i] = v;
                            }
                        }
                    }
                } else {
                    for (int i = tid; i < X0 * Y0 * Z0; i += kPropThreads) {
                        const int z = i % Z0, xy = i / Z0, y = xy % Y0, x = xy / Y0;
                        const int gx = min(max(bx + x - hl, 0), res - 1), gy = min(max(by + y - hl, 0), res - 1), gz = min(max(bz + z - hl, 0), res - 1);
                        s0[xy * ZS + zoff + z] = __ldcg(in + ((size_t)gx * res + gy) * res + gz);
                    }
                }
                __syncthreads();
                for (int i = tid; i < X0 * Y0 * TZ; i += kPropThreads) {       // sum along z
                    const int z = i & (TZ - 1), xy = i >> 5;
                    const uint8_t* r = s0 + xy * ZS + zoff + z;
                    int acc = 0;
                    for (int t = 0; t < W; ++t) acc += sign_of(r[t]);
                    t1[i] = (int8_t)acc;
                }
                __syncthreads();
                for (int i = tid; i < X0 * TZ; i += kPropThreads) {            // sum along y, sliding window
                    const int z = i & (TZ - 1), x = i >> 5;
                    const int8_t* r = t1 + (x * Y0) * TZ + z;
                    int acc = 0;
                    for (int t = 0; t < W; ++t) acc += r[t * TZ];
                    t2[(x * TY) * TZ + z] = (int16_t)acc;
                    for (int y = 1; y < TY; ++y) {
                        acc += r[(y + W - 1) * TZ] - r[(y - 1) * TZ];
                        t2[(x * TY + y) * TZ + z] = (int16_t)acc;
                    }
                }
                __syncthreads();
                {                                                              // sum along x, threshold, apply
                    const int z = tid & (TZ - 1), y = tid >> 5;
                    const int gy = by + y, gz = bz + z;
                    const bool col_ok = gy < res && gz < res;
                    const int16_t* r = t2 + y * TZ + z;
                    int acc = 0;
                    for (int t = 0; t < W; ++t) acc += r[t * TY * TZ];
                    int dS = 0, nz = 0, cminx = 1 << 20, cmaxx = -1;
                    for (int x = 0; x < TX; ++x) {
                        if (x > 0) acc += r[(x + W - 1) * TY * TZ] - r[(x - 1) * TY * TZ];
                        const int gx = bx + x;
                        if (col_ok && gx < res) {
                            int vote = 0;
                            if (!(fabsf((float)acc) < p.thr)) vote = acc > 0 ? 1 : (acc < 0 ? -1 : 0);
                            nz += (vote == 0);
                            const uint8_t b = s0[((x + hl) * Y0 + (y + hl)) * ZS + zoff + hl + z];
                            uint8_t nb = b;
                            if (b & kU0) {
                                const int so = sign_of(b);
                                nb = (uint8_t)((vote & 3) | kU0);
                                if (vote != so) { dS += (vote == 0) - (so == 0); cminx = min(cminx, x); cmaxx = max(cmaxx, x); }
                            }
                            out[((size_t)gx * res + gy) * res + gz] = nb;
                        }
                    }
                    // block totals
                    unsigned ch = __ballot_sync(0xffffffffu, cmaxx >= 0);
    #pragma unroll
                    for (int o = 16; o > 0; o >>= 1) { dS += __shfl_xor_sync(0xffffffffu, dS, o); nz += __shfl_xor_sync(0xffffffffu, nz, o); }
                    if ((tid & 31) == 0) { if (dS) atomicAdd(&sh[0], dS); if (nz) atomicAdd(&sh[1], nz); }
                    if (ch) {                                                  // rare: signs change only along the front
                        if (cmaxx >= 0) {
                            atomicMin(&sh[2], cminx); atomicMax(&sh[5], cmaxx);
                            atomicMin(&sh[3], y); atomicMax(&sh[6], y);
                            atomicMin(&sh[4], z); atomicMax(&sh[7], z);
                        }
                    }
                }
            }
            __syncthreads();
            if (tid == 0) {     // this CTA's contribution to the iteration's counters: one pair of atomics per iteration, below
                const int old = oldvz;
                if (sh[1] != old) { p.voteZeros[tile] = sh[1]; ctaN += sh[1] - old; }
                ctaS += sh[0];
                ++ctaVisits;
            }
            bool fresh = false;
            int nfresh = 0;
            if (tid < 27 && sh[5] >= 0) {
                // a changed sign at local c moves the votes at c-hh .. c+hl: neighbours whose voxels fall in that range
                const int dz = tid % 3 - 1, dy = (tid / 3) % 3 - 1, dx = tid / 9 - 1;
                const bool rx = dx == 0 || (dx < 0 ? sh[2] - hh < 0 : sh[5] + hl >= TX);
                const bool ry = dy == 0 || (dy < 0 ? sh[3] - hh < 0 : sh[6] + hl >= TY);
                const bool rz = dz == 0 || (dz < 0 ? sh[4] - hh < 0 : sh[7] + hl >= TZ);
                const int nx = tx + dx, ny = ty + dy, nzt = tz + dz;
                if (rx && ry && rz && nx >= 0 && ny >= 0 && nzt >= 0 && nx < p.ntx && ny < p.nty && nzt < p.ntz) {
                    const int n = (nx * p.nty + ny) * p.ntz + nzt;
                    // byte flags, word-wide atomic: set our byte, see whether it was clear
                    unsigned* wptr = (unsigned*)(flagNext + (n & ~3));
                    const unsigned bit = 1u << (8 * (n & 3));
                    fresh = !(atomicOr(wptr, bit) & bit);
                    nfresh = n;
                }
            }
            if (tid < 32) {          // (the 27 marking threads are lanes of warp 0) one list-size atomic per tile, not per neighbour
                const unsigned m = __ballot_sync(0xffffffffu, fresh);
                if (m) {
                    unsigned basepos = 0;
                    if (tid == 0) basepos = atomicAdd(&p.ctrl->slot[nxt].listCount, (unsigned)__popc(m));
                    basepos = __shfl_sync(0xffffffffu, basepos, 0);
                    if (fresh) listNext[basepos + __popc(m & ((1u << tid) - 1u))] = nfresh;
                }
            }
            // no barrier here: sh[] is re-initialised by warp 0 itself (program order) and only touched by the other warps
            // behind the next tile's barriers; the hand-over slot alternates
            par ^= 1;
        }
        if (tid == 0) {
            if (ctaN) atomicAdd((unsigned long long*)&p.ctrl->slot[cur].dN, (unsigned long long)ctaN);
            if (ctaS) atomicAdd((unsigned long long*)&p.ctrl->slot[cur].dS, (unsigned long long)ctaS);
            ctaN = 0; ctaS = 0;
        }
        const unsigned long long ts = diag ? now_ns() : 0ull;
        grid.sync();
        if (diag) { t_sync += now_ns() - ts; if (it == 0) p.ctrl->t_first = now_ns() - t_begin; }
        if (tid == 0) { sh_d[0] = __ldcg(&p.ctrl->slot[cur].dN); sh_d[1] = __ldcg(&p.ctrl->slot[cur].dS); }
        __syncthreads();
        totalN += sh_d[0];
        const long long afterS = totalS + sh_d[1];
        if (totalN >= totalS) { final_buf = it & 1; break; }            // `if unknown_after.sum() >= unknown_before.sum(): break`
        totalS = afterS;
        ++iters;
    }
    if (tid == 0 && ctaVisits) atomicAdd(&p.ctrl->visits, ctaVisits);
    if (blockIdx.x == 0 && tid == 0) { p.ctrl->iters = iters; p.ctrl->final_buf = final_buf; p.ctrl->error = error; p.ctrl->t_total = now_ns() - t_begin; p.ctrl->t_sync = t_sync; }
}

// the reference raises IndexError for an index >= res and wraps a negative one (sdf.py:95-111); here both are counted and
// reported as an error by the entry point, nothing is written out of bounds
__global__ void scatter_kernel(const int32_t* __restrict__ lin, const float* __restrict__ sdf, int64_t Q, int64_t V,
                               float* __restrict__ vol, Ctrl* c) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Q) return;
    const int32_t l = lin[i];
    if (l >= 0 && (int64_t)l < V) vol[l] = sdf[i];
    else atomicAdd(&c->bad_index, 1u);
}

// vol[vol == 0] = S[vol == 0]; clamp to [-1, 1]   (sdf.py:179,200-202)
__global__ void finalize_kernel(float* __restrict__ vol, const uint8_t* __restrict__ A, const uint8_t* __restrict__ B,
                                const Ctrl* __restrict__ c, int64_t V) {
    int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= V) return;
    float x = vol[v];
    if (x == 0.0f) x = (float)sign_of((c->final_buf ? B : A)[v]);
    x = x < -1.0f ? -1.0f : (x > 1.0f ? 1.0f : x);
    vol[v] = x;
}

}  // namespace

void sdf_from_logits(const float* logits, const float* radius, int64_t B, float* sdf, cudaStream_t st) {
    if (B <= 0) return;
    P2S_LAUNCH(sdf_from_logits_kernel, (unsigned)cdiv(B, 256), 256, 0, st, logits, radius, B, sdf);
}

void sdf_to_volume(const int32_t* lin_idx, const float* sdf, int64_t Q, int res, int sigma, float thr,
                   float* vol, int* iterations_host, cudaStream_t st) {
    P2S_CHECK(res >= 2 && res <= 1024, "grid resolution out of range");
    P2S_CHECK(sigma >= 1 && sigma <= 11, "sigma out of range [1, 11]");
    const int64_t V = (int64_t)res * res * res;
    const unsigned blocks = (unsigned)cdiv(V, 256);
    PropParams pp{};
    pp.res = res;
    // convolve(ones(sigma^3), mode='nearest'): output o sums inputs o-ceil(s/2)+1 .. o+floor(s/2)
    pp.lo = -((sigma + 1) / 2) + 1; pp.hi = sigma / 2; pp.thr = thr;
    pp.ntx = (int)cdiv(res, TX); pp.nty = (int)cdiv(res, TY); pp.ntz = (int)cdiv(res, TZ);
    pp.maxIters = 64 * res;
    const int numTiles = pp.ntx * pp.nty * pp.ntz;
    const size_t nt4 = ((size_t)numTiles + 3) & ~(size_t)3;
    size_t off = (sizeof(Ctrl) + 255) & ~(size_t)255;
    const size_t off_A = off; off += (V + 255) & ~(size_t)255;
    const size_t off_B = off; off += (V + 255) & ~(size_t)255;
    const size_t off_lists = off; off += 3 * nt4 * sizeof(int);
    const size_t off_vz = off; off += nt4 * sizeof(int);
    const size_t off_flags = off; off += 2 * nt4;
    DeviceCtx& ctx = device_ctx();
    uint8_t* base = (uint8_t*)ctx.vol_ws.get(off);
    Ctrl* ctrl = (Ctrl*)base;
    pp.ctrl = ctrl;
    pp.buf[0] = base + off_A; pp.buf[1] = base + off_B;
    for (int i = 0; i < 3; ++i) pp.list[i] = (int*)(base + off_lists) + (size_t)i * nt4;
    pp.voteZeros = (int*)(base + off_vz);
    pp.flags[0] = base + off_flags; pp.flags[1] = base + off_flags + nt4;

    P2S_CUDA(cudaMemsetAsync(ctrl, 0, sizeof(Ctrl), st));
    P2S_CUDA(cudaMemsetAsync(vol, 0, (size_t)V * sizeof(float), st));
    if (Q > 0) {
        P2S_LAUNCH(any_nonzero_kernel, (unsigned)cdiv(Q, 256), 256, 0, st, sdf, Q, ctrl);
        P2S_LAUNCH(scatter_kernel, (unsigned)cdiv(Q, 256), 256, 0, st, lin_idx, sdf, Q, V, vol, ctrl);
    }
    P2S_LAUNCH(init_sign_kernel, blocks, 256, 0, st, vol, res, pp.buf[0], ctrl);
    P2S_CUDA(cudaMemsetAsync(pp.flags[0], 0, 2 * nt4, st));
    P2S_LAUNCH(init_tiles_kernel, (unsigned)cdiv(numTiles, 256), 256, 0, st, pp.list[0], pp.voteZeros, numTiles, ctrl);

    // persistent cooperative launch: as many CTAs as are co-resident (the runtime refuses a larger grid instead of hanging)
    const int hl = -pp.lo, hh = pp.hi;
    const int X0 = TX + hl + hh, Y0 = TY + hl + hh, Z0 = TZ + hl + hh;
    const int HW = (std::max(hl, hh) + 3) / 4, ZS = TZ + 8 * HW;
    (void)Z0;
    pp.words = (res % 4 == 0) ? 1 : 0;       // aligned 32-bit row loads need word-aligned rows
    pp.fast = (pp.words && sigma <= 5) ? 1 : 0;   // packed biased-byte sums need 2 * sigma^3 <= 255
    pp.vec = (sigma == 5 && res % 32 == 0) ? 1 : 0;   // row-vector path: full tiles, 16-byte aligned rows
    const size_t smem_generic = (size_t)((X0 * Y0 * ZS + 15) & ~15) + (size_t)((X0 * Y0 * TZ + 15) & ~15) + (size_t)X0 * TY * TZ * 2;
    const size_t smem_fast = 4 * ((size_t)X0 * Y0 * (ZS / 4) + (size_t)TX * TY * 8 + (size_t)X0 * Y0 * 8 + (size_t)X0 * TY * 8);
    const size_t smem = pp.fast ? smem_fast : smem_generic;
    int per_sm = 0;
    const bool s5 = pp.fast && sigma == 5;
    const void* kfn = s5 ? (const void*)propagate_kernel<true> : (const void*)propagate_kernel<false>;
    ctx.set_max_dynamic_smem(kfn, (int)smem);
    if (s5) P2S_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, propagate_kernel<true>, kPropThreads, smem));
    else P2S_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, propagate_kernel<false>, kPropThreads, smem));
    P2S_CHECK(per_sm >= 1, "sign propagation kernel does not fit on an SM");
    const unsigned grid = (unsigned)std::max(1, std::min(numTiles, ctx.sm_count * per_sm));
    void* args[] = {&pp};
    P2S_CUDA(cudaLaunchCooperativeKernel(kfn, dim3(grid), dim3(kPropThreads), args, smem, st));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    P2S_LAUNCH(finalize_kernel, blocks, 256, 0, st, vol, pp.buf[0], pp.buf[1], ctrl, V);
    Ctrl h{};
    P2S_CUDA(cudaMemcpyAsync(&h, ctrl, sizeof(Ctrl), cudaMemcpyDeviceToHost, st));
    P2S_CUDA(cudaStreamSynchronize(st));
    P2S_CHECK(h.bad_index == 0, "voxel index outside [0, res^3): query points must lie in [-1, 1)^3 (the reference raises IndexError / wraps)");
    P2S_CHECK(h.error == 0, "sign propagation did not converge");
    if (iterations_host) *iterations_host = h.iters;
    {
        static int stats = -1;
        if (stats < 0) { const char* e = getenv("P2S_VOL_STATS"); stats = (e && e[0] == '1') ? 1 : 0; }
        if (stats) fprintf(stderr, "p2s sign propagation: res %d, %d iterations, %llu tile evaluations over %d tiles (%.1f per tile; a full sweep per iteration would be %d), grid %u x %d threads, %zu B smem; kernel %.3f ms (block 0: %.3f ms inside grid.sync, first iteration %.3f ms)\n",
                           res, h.iters, h.visits, numTiles, (double)h.visits / numTiles, h.iters + 1, grid, kPropThreads, smem,
                           h.t_total * 1e-6, h.t_sync * 1e-6, h.t_first * 1e-6);
    }
    if (Q > 0 && !h.nonzero_seen) {
        // the reference prints a warning and returns without writing anything (sdf.py:187-189)
        if (iterations_host) *iterations_host = -1;
    }
}

}  // namespace p2s
