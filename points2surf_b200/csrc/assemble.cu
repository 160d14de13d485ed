// K2 / K3: per-query patch assembly -- PointcloudPatchDataset.__getitem__ (source/data_loader.py:322-421).
//   K2  exact kNN (k smallest float64 distances on float32 coordinates, i.e. scipy cKDTree semantics,
//       source/base/point_cloud.py:174-175), patch radius and patch-space normalisation in float32
//       exactly like NumPy (source/base/utils.py:62-69,80-88).
//   K3  global sub-sample (source/base/utils.py:196-227): uniform with replacement, or distance-weighted
//       without replacement via exponential clocks (Efraimidis-Spirakis), which realises the same
//       successive-sampling law as RandomState.choice(replace=False, p) (SURVEY.md section 10).
// One CTA per query; the cloud (N*12 B, L1/L2-resident) is streamed twice per selection:
// a histogram pass over the top bits of the (monotone) key, then a collect pass.  All byte/compare work.
#include "common.cuh"
#include <cub/device/device_radix_sort.cuh>

namespace p2s {

namespace {

constexpr int kThreads = 256;
constexpr int kBins = 2048;
constexpr int kCap = 1024;  // boundary-bin candidates that are sorted exactly (sub-sampler, kNN up to 512 neighbours)
constexpr int kCapBig = 2048;   // kNN with 513..1536 neighbours (large_kNN: 1200) and ball-query patches

// ---- key helpers: non-negative doubles order like their bit patterns ----
__device__ __forceinline__ unsigned long long dkey(double v) { return (unsigned long long)__double_as_longlong(v); }
// level-0 bin: sign+exponent+4 mantissa bits, rebased so that 2^-100 .. 2^27 maps to 0..2047
__device__ __forceinline__ int bin0(unsigned long long key) {
    long long b = (long long)(key >> 48) - ((1023 - 100) << 4);
    return (int)(b < 0 ? 0 : (b > kBins - 1 ? kBins - 1 : b));
}

template <int CAP>
struct SelectSmemT {
    unsigned hist[kBins];
    unsigned long long cand_key[CAP];
    int cand_id[CAP];
    int bin_sel[4];       // selected bin per level
    unsigned below;       // number of keys strictly below the boundary bin
    unsigned n_direct;    // slots used by "surely in" members
    unsigned n_cand;      // boundary candidates collected
    int levels;           // refinement levels used (1..3)
};
using SelectSmem = SelectSmemT<kCap>;

// does `key` fall in the boundary bin chain selected so far (levels [0, upto))?
template <int CAP>
__device__ __forceinline__ int chain_cmp(const SelectSmemT<CAP>& s, unsigned long long key, int upto) {
    // returns -1 if key sorts below the chain, 0 if inside, +1 above
    int b = bin0(key);
    if (b != s.bin_sel[0]) return b < s.bin_sel[0] ? -1 : 1;
    for (int l = 1; l < upto; ++l) {
        int bl = (int)((key >> (48 - 11 * l)) & 0x7FF);
        if (bl != s.bin_sel[l]) return bl < s.bin_sel[l] ? -1 : 1;
    }
    return 0;
}

// Block-wide: find the bin chain that contains the k-th smallest key.  KeyFn(i) -> key of item i.
template <int CAP, class KeyFn>
__device__ void find_boundary(SelectSmemT<CAP>& s, int N, int k, int cand_cap, KeyFn keyfn) {
    const int tid = threadIdx.x;
    if (tid == 0) { s.below = 0; s.levels = 0; }
    for (int level = 0; level < 3; ++level) {
        for (int i = tid; i < kBins; i += kThreads) s.hist[i] = 0;
        __syncthreads();
        for (int i = tid; i < N; i += kThreads) {
            unsigned long long key = keyfn(i);
            if (level == 0) atomicAdd(&s.hist[bin0(key)], 1u);
            else if (chain_cmp(s, key, level) == 0) atomicAdd(&s.hist[(int)((key >> (48 - 11 * level)) & 0x7FF)], 1u);
        }
        __syncthreads();
        if (tid < 32) {  // warp 0: locate the bin where the running count crosses k
            unsigned need = (unsigned)k - s.below;  // rank inside the current chain, 1-based
            unsigned run = 0;
            int found = -1;
            unsigned below_add = 0;
            for (int base = 0; base < kBins && found < 0; base += 32) {
                unsigned c = s.hist[base + tid];
                unsigned incl = c;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
                    if (tid >= o) incl += t;
                }
                unsigned excl = incl - c;
                unsigned hit = __ballot_sync(0xffffffffu, run + incl >= need);
                if (hit) {
                    int lane = __ffs(hit) - 1;
                    found = base + lane;
                    below_add = run + __shfl_sync(0xffffffffu, excl, lane);
                }
                run += __shfl_sync(0xffffffffu, incl, 31);
            }
            if (tid == 0) {
                s.bin_sel[level] = found;
                s.below += below_add;
                s.levels = level + 1;
            }
        }
        __syncthreads();
        if (s.hist[s.bin_sel[level]] <= (unsigned)cand_cap) break;  // uniform: same smem value for all threads
        __syncthreads();
    }
}

// bitonic sort of (key, id) ascending over the first P = pow2ceil(n) slots (slots >= n are padded with +inf keys).
// The total order (key, id) is strict, so the result does not depend on the network used.
// P <= 512: two elements per thread live in registers; compare-exchanges at element strides 1 (in-thread) and 2..32 (warp
// shuffles) need no barrier, only the strides >= 64 go through shared memory: 10 block barriers per sort instead of 45
// (the barriers, not the instructions, were what the kNN kernel spent its time on).
template <int CAP>
__device__ void sort_candidates(SelectSmemT<CAP>& s, int n) {
    const int tid = threadIdx.x;
    int P = 64;
    while (P < n) P <<= 1;                       // n <= CAP (checked by the callers), so P <= CAP
    for (int i = tid; i < P; i += kThreads)
        if (i >= n) { s.cand_key[i] = ~0ull; s.cand_id[i] = 0x7fffffff; }
    __syncthreads();
    auto smem_stage = [&](int size, int stride) {
        for (int t = tid; t < P / 2; t += kThreads) {
            int lo = 2 * t - (t & (stride - 1));
            int hi = lo + stride;
            bool up = ((lo & size) == 0);
            unsigned long long ka = s.cand_key[lo], kb = s.cand_key[hi];
            int ia = s.cand_id[lo], ib = s.cand_id[hi];
            bool gt = (ka > kb) || (ka == kb && ia > ib);
            if (gt == up) { s.cand_key[lo] = kb; s.cand_key[hi] = ka; s.cand_id[lo] = ib; s.cand_id[hi] = ia; }
        }
        __syncthreads();
    };
    if (P <= 2 * kThreads) {
        static_assert(kThreads == 256, "register sort assumes 256 threads (2 elements per thread at P = 512)");
        const bool active = 2 * tid < P;          // warp-uniform: P is a multiple of 64
        unsigned long long k0 = 0, k1 = 0;
        int i0 = 0, i1 = 0;
        auto load = [&] { if (active) { k0 = s.cand_key[2 * tid]; k1 = s.cand_key[2 * tid + 1]; i0 = s.cand_id[2 * tid]; i1 = s.cand_id[2 * tid + 1]; } };
        auto store = [&] { if (active) { s.cand_key[2 * tid] = k0; s.cand_key[2 * tid + 1] = k1; s.cand_id[2 * tid] = i0; s.cand_id[2 * tid + 1] = i1; } };
        // strides min(size / 2, 32) .. 1 of the merge of `size`, in registers
        auto reg_stages = [&](int size) {
            if (!active) return;
            for (int stride = (size >> 1) < 32 ? (size >> 1) : 32; stride >= 2; stride >>= 1) {
                const int m = stride >> 1;                              // lane mask of the partner thread
                const bool up = (((2 * tid) & size) == 0);
                const bool keep_min = (((2 * tid) & stride) == 0) == up;
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    unsigned long long& k = b ? k1 : k0;
                    int& id = b ? i1 : i0;
                    const unsigned long long ok = __shfl_xor_sync(0xffffffffu, k, m);
                    const int oi = __shfl_xor_sync(0xffffffffu, id, m);
                    const bool other_less = (ok < k) || (ok == k && oi < id);
                    if (other_less == keep_min) { k = ok; id = oi; }
                }
            }
            {   // stride 1: the thread's own pair
                const bool up = (((2 * tid) & size) == 0);
                const bool gt = (k0 > k1) || (k0 == k1 && i0 > i1);
                if (gt == up) { const unsigned long long tk = k0; k0 = k1; k1 = tk; const int ti = i0; i0 = i1; i1 = ti; }
            }
        };
        load();
        for (int size = 2; size <= 64 && size <= P; size <<= 1) reg_stages(size);
        store();
        __syncthreads();
        for (int size = 128; size <= P; size <<= 1) {
            for (int stride = size >> 1; stride >= 64; stride >>= 1) smem_stage(size, stride);
            load();
            reg_stages(size);
            store();
            __syncthreads();
        }
        return;
    }
    for (int size = 2; size <= P; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) smem_stage(size, stride);
}

__device__ __forceinline__ double dist2_f64(const float* __restrict__ pts, int i, double qx, double qy, double qz) {
    // cKDTree: sum over dimensions of (x-y)^2, float64, sequential, no FMA contraction
    double dx = (double)pts[i * 3 + 0] - qx, dy = (double)pts[i * 3 + 1] - qy, dz = (double)pts[i * 3 + 2] - qz;
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// NumPy float32: np.linalg.norm(q - p) = sqrt((dx*dx + dy*dy) + dz*dz), every op rounded to float32
__device__ __forceinline__ float norm_f32(float dx, float dy, float dz) {
    return __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
}

// ------------------------------------------------------------------------------------------------
// K2
// ------------------------------------------------------------------------------------------------
// One CTA walks kRun consecutive queries of the ordered list.  Consecutive voxel centres are close, so the exact
// k-th distance of query j gives a *guaranteed* bound for query j+1 (triangle inequality:
// kth(j+1) <= kth(j) + |q(j+1) - q(j)|): one pass collects every point within that bound (typically 1.1-1.2 k
// candidates) and an exact sort finishes the job -- no histogram.  The first query of a run, big jumps between
// queries and overflowing candidate lists fall back to the histogram selection.
constexpr int kRun = 8;        // shortest run; the launcher lengthens it so that the grid is one full wave (see knn_patch)

template <int CAP>
__global__ void __launch_bounds__(kThreads)
knn_patch_kernel(const float* __restrict__ pts, int N, const float* __restrict__ queries, int64_t Q, int k,
                 int32_t* __restrict__ ids_out, float* __restrict__ patch_out, float* __restrict__ radius_out,
                 int* __restrict__ err_flag, int run) {
    constexpr int kCap = CAP;                     // shadows the file-level constant inside this kernel
    __shared__ SelectSmemT<CAP> s;
    __shared__ float red[kThreads / 32];
    __shared__ float s_radius;
    __shared__ double s_kth;          // exact k-th squared distance of the previous query (0 = unknown)
    const int tid = threadIdx.x;
    const int64_t q_begin = (int64_t)blockIdx.x * run;
    const int64_t q_end = (q_begin + run < Q) ? (q_begin + run) : Q;
    if (tid == 0) s_kth = 0.0;
    double pqx = 0.0, pqy = 0.0, pqz = 0.0;
    for (int64_t q = q_begin; q < q_end; ++q) {
        __syncthreads();
        const float qxf = queries[q * 3 + 0], qyf = queries[q * 3 + 1], qzf = queries[q * 3 + 2];
        const double qx = qxf, qy = qyf, qz = qzf;
        auto keyfn = [&](int i) { return dkey(dist2_f64(pts, i, qx, qy, qz)); };
        // ---- fast path: bound from the previous query
        bool done = false;
        const double kth_prev = s_kth;
        if (kth_prev > 0.0) {
            const double ddx = qx - pqx, ddy = qy - pqy, ddz = qz - pqz;
            const double delta = sqrt(ddx * ddx + ddy * ddy + ddz * ddz);
            const double rprev = sqrt(kth_prev);
            if (delta < 0.25 * rprev) {
                const double rb = (rprev + delta) * (1.0 + 1e-12);
                const unsigned long long bound = dkey(rb * rb * (1.0 + 1e-12));
                if (tid == 0) s.n_cand = 0;
                __syncthreads();
                // float32 pre-filter (relative error of the fp32 squared distance < 1e-6): only points that can be
                // inside the bound pay for the exact float64 distance
                const float bound_f = (float)(rb * rb) * 1.00001f;
                for (int i = tid; i < N; i += kThreads) {
                    const float fx = pts[i * 3 + 0] - qxf, fy = pts[i * 3 + 1] - qyf, fz = pts[i * 3 + 2] - qzf;
                    if (fmaf(fx, fx, fmaf(fy, fy, fz * fz)) > bound_f) continue;
                    unsigned long long key = keyfn(i);
                    if (key <= bound) {
                        unsigned slot = atomicAdd(&s.n_cand, 1u);
                        if (slot < (unsigned)kCap) { s.cand_key[slot] = key; s.cand_id[slot] = i; }
                    }
                }
                __syncthreads();
                const unsigned n = s.n_cand;
                if (n >= (unsigned)k && n <= (unsigned)kCap) {
                    sort_candidates(s, (int)n);
                    done = true;
                }
            }
        }
        if (!done) {
            // ---- histogram selection
            __syncthreads();
            find_boundary(s, N, k, kCap - (k > 512 ? k : 512), keyfn);
            if (tid == 0) { s.n_direct = 0; s.n_cand = 0; }
            __syncthreads();
            const int levels = s.levels;
            // collect: keys below the boundary chain are members; keys inside it are candidates
            for (int i = tid; i < N; i += kThreads) {
                unsigned long long key = keyfn(i);
                int c = chain_cmp(s, key, levels);
                if (c < 0) {
                    // members go to the tail of the candidate arrays so one sort orders everything
                    unsigned slot = atomicAdd(&s.n_direct, 1u);
                    if (slot < (unsigned)kCap) { s.cand_key[kCap - 1 - slot] = key; s.cand_id[kCap - 1 - slot] = i; }
                } else if (c == 0) {
                    unsigned slot = atomicAdd(&s.n_cand, 1u);
                    if (slot < (unsigned)kCap) { s.cand_key[slot] = key; s.cand_id[slot] = i; }
                }
            }
            __syncthreads();
            const unsigned n_direct = s.n_direct, n_cand = s.n_cand;
            if (n_direct + n_cand > (unsigned)kCap || n_direct != s.below) {
                // more than kCap points tie into the boundary bin even after 3 refinement levels (degenerate cloud)
                if (tid == 0) atomicExch(err_flag, 1);
                return;
            }
            // compact: move the members right behind the candidates, then sort everything exactly
            unsigned long long mk[(kCap + kThreads - 1) / kThreads];
            int mi[(kCap + kThreads - 1) / kThreads];
            int cnt = 0;
            for (unsigned j = tid; j < n_direct; j += kThreads) { mk[cnt] = s.cand_key[kCap - 1 - j]; mi[cnt] = s.cand_id[kCap - 1 - j]; ++cnt; }
            __syncthreads();
            cnt = 0;
            for (unsigned j = tid; j < n_direct; j += kThreads) { s.cand_key[n_cand + j] = mk[cnt]; s.cand_id[n_cand + j] = mi[cnt]; ++cnt; }
            __syncthreads();
            sort_candidates(s, (int)(n_direct + n_cand));
        }
        // exact k-th squared distance -> bound for the next query of the run
        if (tid == 0) s_kth = __longlong_as_double((long long)s.cand_key[k - 1]);
        pqx = qx; pqy = qy; pqz = qz;

        // radius = max float32 norm over the k neighbours (utils.get_patch_radii)
        float r = 0.f;
        for (int j = tid; j < k; j += kThreads) {
            int id = s.cand_id[j];
            r = fmaxf(r, norm_f32(__fsub_rn(qxf, pts[id * 3 + 0]), __fsub_rn(qyf, pts[id * 3 + 1]), __fsub_rn(qzf, pts[id * 3 + 2])));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r = fmaxf(r, __shfl_xor_sync(0xffffffffu, r, o));
        if ((tid & 31) == 0) red[tid >> 5] = r;
        __syncthreads();
        if (tid == 0) {
            float m = red[0];
            for (int w = 1; w < kThreads / 32; ++w) m = fmaxf(m, red[w]);
            s_radius = m;
            radius_out[q] = m;
        }
        __syncthreads();
        const float radius = s_radius;
        for (int j = tid; j < k; j += kThreads) {
            int id = s.cand_id[j];
            if (ids_out) ids_out[q * k + j] = id;
            float* o = patch_out + (q * k + j) * 3;
            // model_space_to_patch_space: (p - q) / r in float32
            o[0] = __fdiv_rn(__fsub_rn(pts[id * 3 + 0], qxf), radius);
            o[1] = __fdiv_rn(__fsub_rn(pts[id * 3 + 1], qyf), radius);
            o[2] = __fdiv_rn(__fsub_rn(pts[id * 3 + 2], qzf), radius);
        }
    }
}

__device__ __forceinline__ float u01_open(uint32_t x) {  // (0,1]
    return ((float)(x >> 8) + 1.0f) * (1.0f / 16777216.0f);
}

// ------------------------------------------------------------------------------------------------
// K2b: ball-query patches (radius ablations) -- point_cloud.get_patch_kdtree with patch_radius > 0
// (source/base/point_cloud.py:176-192) + the padding rule of PointcloudPatchDataset.__getitem__
// (source/data_loader.py:340-350): all points with float64 distance <= r (cKDTree.query_ball_point semantics on
// float32 coordinates); more than k of them -> a uniformly random k-subset without replacement (rng.choice in the
// reference; here the k smallest Philox clocks, same law, different stream); fewer -> padded with the query point itself
// (patch-space origin, id 0).  Normalisation by the FIXED radius in float32.  One CTA per query.
// Output order: ascending point id when nothing is dropped (the reference's order is the kd-tree traversal order; the
// network max-pools over the patch, so order carries no information).
constexpr int kBallMaxK = 1536;

__global__ void __launch_bounds__(kThreads)
ball_patch_kernel(const float* __restrict__ pts, int N, const float* __restrict__ queries, int64_t qbase,
                  const int32_t* __restrict__ qidx, int k, double r2, float rf, uint64_t seed,
                  int32_t* __restrict__ ids_out, float* __restrict__ patch_out, float* __restrict__ radius_out,
                  int32_t* __restrict__ count_out, int* __restrict__ err_flag) {
    constexpr int CAP = kCapBig;
    __shared__ SelectSmemT<CAP> s;
    __shared__ int sel[kBallMaxK];
    const int tid = threadIdx.x;
    const int64_t q = blockIdx.x;
    const float qxf = queries[q * 3 + 0], qyf = queries[q * 3 + 1], qzf = queries[q * 3 + 2];
    const double qx = qxf, qy = qyf, qz = qzf;
    const uint64_t qi = (uint64_t)(qbase + (qidx ? (int64_t)qidx[q] : q));
    const float bound_f = (float)r2 * 1.00001f + 1e-30f;
    auto in_ball = [&](int i) {
        const float fx = pts[i * 3 + 0] - qxf, fy = pts[i * 3 + 1] - qyf, fz = pts[i * 3 + 2] - qzf;
        if (fmaf(fx, fx, fmaf(fy, fy, fz * fz)) > bound_f) return false;       // fp32 pre-filter, exact test below
        return dist2_f64(pts, i, qx, qy, qz) <= r2;
    };
    auto clock_key = [&](int i) {     // Exp(1) clock of point i for this query
        uint32_t r[4];
        philox4x32_10((uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)qi, (uint32_t)(qi >> 32), (uint32_t)(i >> 2), 0x3c6ef372u, r);
        return dkey((double)(-__logf(u01_open(r[i & 3]))));
    };
    if (tid == 0) { s.n_cand = 0; s.n_direct = 0; }
    __syncthreads();
    for (int i = tid; i < N; i += kThreads) {
        if (!in_ball(i)) continue;
        const unsigned slot = atomicAdd(&s.n_cand, 1u);
        if (slot < (unsigned)CAP) { s.cand_key[slot] = (unsigned long long)i; s.cand_id[slot] = i; }
    }
    __syncthreads();
    const int count = (int)s.n_cand;
    if (count_out && tid == 0) count_out[q] = count;
    int n_sel = count < k ? count : k;
    if (count <= k) {
        sort_candidates(s, count);                            // ascending id
        for (int j = tid; j < n_sel; j += kThreads) sel[j] = s.cand_id[j];
    } else if (count <= CAP) {
        for (int j = tid; j < count; j += kThreads) s.cand_key[j] = clock_key(s.cand_id[j]);
        __syncthreads();
        sort_candidates(s, count);
        for (int j = tid; j < k; j += kThreads) sel[j] = s.cand_id[j];
    } else {
        // more points in the ball than the candidate buffer holds: histogram selection of the k smallest clocks
        __syncthreads();
        auto keyfn = [&](int i) { return in_ball(i) ? clock_key(i) : ~0ull; };
        find_boundary(s, N, k, CAP, keyfn);
        if (tid == 0) { s.n_direct = 0; s.n_cand = 0; }
        __syncthreads();
        const int levels = s.levels;
        for (int i = tid; i < N; i += kThreads) {
            const unsigned long long key = keyfn(i);
            if (key == ~0ull) continue;
            const int c = chain_cmp(s, key, levels);
            if (c < 0) {
                const unsigned slot = atomicAdd(&s.n_direct, 1u);
                if (slot < (unsigned)k) sel[slot] = i;
            } else if (c == 0) {
                const unsigned slot = atomicAdd(&s.n_cand, 1u);
                if (slot < (unsigned)CAP) { s.cand_key[slot] = key; s.cand_id[slot] = i; }
            }
        }
        __syncthreads();
        const unsigned n_direct = s.n_direct, n_cand = s.n_cand;
        if (n_cand > (unsigned)CAP || n_direct != s.below || n_direct + n_cand < (unsigned)k) {
            if (tid == 0) atomicExch(err_flag, 3);
            return;
        }
        sort_candidates(s, (int)n_cand);
        for (unsigned j = tid; n_direct + j < (unsigned)k; j += kThreads) sel[n_direct + j] = s.cand_id[j];
    }
    __syncthreads();
    if (tid == 0) radius_out[q] = rf;
    for (int j = tid; j < k; j += kThreads) {
        float* o = patch_out + (q * k + j) * 3;
        if (j < n_sel) {
            const int id = sel[j];
            if (ids_out) ids_out[q * k + j] = id;
            o[0] = __fdiv_rn(__fsub_rn(pts[id * 3 + 0], qxf), rf);
            o[1] = __fdiv_rn(__fsub_rn(pts[id * 3 + 1], qyf), rf);
            o[2] = __fdiv_rn(__fsub_rn(pts[id * 3 + 2], qzf), rf);
        } else {
            if (ids_out) ids_out[q * k + j] = 0;              // -1 -> 0, coordinates <- query point (data_loader.py:341-345)
            o[0] = 0.f; o[1] = 0.f; o[2] = 0.f;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K3
// ------------------------------------------------------------------------------------------------

__global__ void subsample_uniform_kernel(int N, int64_t Q, int64_t qbase, const int32_t* __restrict__ qidx, int S, uint64_t seed, int32_t* __restrict__ out) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int quads = (S + 3) / 4;
    if (t >= Q * quads) return;
    int64_t q = t / quads;
    int j4 = (int)(t % quads);
    uint32_t r[4];
    uint64_t qi = (uint64_t)(qbase + (qidx ? (int64_t)qidx[q] : q));
    philox4x32_10((uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)qi, (uint32_t)(qi >> 32), (uint32_t)j4, 0x5ab5a3e1u, r);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        int j = j4 * 4 + e;
        if (j < S) out[q * S + j] = (int32_t)(((uint64_t)r[e] * (uint64_t)N) >> 32);
    }
}

// CACHE: per-point values live in dynamic shared memory (N floats) so that the distance, the Philox block (shared
// by 4 consecutive points) and the logarithm are evaluated once per point.  With the cache the selection needs no
// histogram: the clock of point i is Exp(1)/w_i, so the expected number of clocks below t is
//   C(t) = sum_i (1 - exp(-w_i t)) = t*S1 - t^2*S2/2 + t^3*S3/6 - ...        (w_i t <~ 0.2 for S/N ~ 0.1)
// Clocks <= t_lo (C = S - 5 sqrt(S)) are members, clocks in (t_lo, t_hi] (C = S + 5 sqrt(S)) are sorted exactly and
// the smallest S - n_members of them complete the draw -- the same S smallest clocks as the histogram selection,
// which takes over whenever the realised counts do not bracket S.
template <bool CACHE>
__global__ void __launch_bounds__(kThreads)
subsample_weighted_kernel(const float* __restrict__ pts, int N, const float* __restrict__ queries,
                          int64_t qbase, const int32_t* __restrict__ qidx, int S, uint64_t seed, int32_t* __restrict__ out, int* __restrict__ err_flag) {
    extern __shared__ float s_val[];     // [N] when CACHE: distance, then weight
    __shared__ SelectSmem s;
    __shared__ float red[3][kThreads / 32];
    __shared__ float s_dmax, s_tlo, s_thi;
    const int tid = threadIdx.x;
    const int64_t q = blockIdx.x;
    const float qx = queries[q * 3 + 0], qy = queries[q * 3 + 1], qz = queries[q * 3 + 2];
    // dist_prob (utils.py:200-208): float32 like NumPy
    float dmax = 0.f;
    for (int i = tid; i < N; i += kThreads) {
        float d = norm_f32(__fsub_rn(qx, pts[i * 3 + 0]), __fsub_rn(qy, pts[i * 3 + 1]), __fsub_rn(qz, pts[i * 3 + 2]));
        if (CACHE) s_val[i] = d;
        dmax = fmaxf(dmax, d);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dmax = fmaxf(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
    if ((tid & 31) == 0) red[0][tid >> 5] = dmax;
    __syncthreads();
    if (tid == 0) {
        float m = red[0][0];
        for (int w = 1; w < kThreads / 32; ++w) m = fmaxf(m, red[0][w]);
        s_dmax = m;
    }
    __syncthreads();
    dmax = s_dmax;
    const uint64_t qi = (uint64_t)(qbase + (qidx ? (int64_t)qidx[q] : q));
    auto weight_of = [&](float d) {
        float dn = __fdiv_rn(d, dmax);
        float w = __fsub_rn(1.0f, __fmul_rn(1.5f, dn));
        return fminf(fmaxf(w, 0.05f), 1.0f);
    };
    // exponential clock with rate w: the S earliest arrivals are a draw without replacement with p ~ w
    auto clock_of = [&](float w, uint32_t rnd) { return __fdividef(-__logf(u01_open(rnd)), w); };
    auto philox_block = [&](int i4, uint32_t (&r)[4]) {
        philox4x32_10((uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)qi, (uint32_t)(qi >> 32), (uint32_t)i4, 0x77f1e2d3u, r);
    };
    if (CACHE) {
        // ---- weights + their first three power sums
        float m1 = 0.f, m2 = 0.f, m3 = 0.f;
        for (int i = tid; i < N; i += kThreads) {
            const float w = weight_of(s_val[i]);
            s_val[i] = w;
            m1 += w; m2 += w * w; m3 += w * w * w;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            m1 += __shfl_xor_sync(0xffffffffu, m1, o);
            m2 += __shfl_xor_sync(0xffffffffu, m2, o);
            m3 += __shfl_xor_sync(0xffffffffu, m3, o);
        }
        if ((tid & 31) == 0) { red[0][tid >> 5] = m1; red[1][tid >> 5] = m2; red[2][tid >> 5] = m3; }
        __syncthreads();
        if (tid == 0) {
            float S1 = 0.f, S2 = 0.f, S3 = 0.f;
            for (int w = 0; w < kThreads / 32; ++w) { S1 += red[0][w]; S2 += red[1][w]; S3 += red[2][w]; }
            auto solve = [&](float target) {
                if (target <= 0.f) return 0.f;
                float t = target / S1;
                for (int it = 0; it < 6; ++it) {
                    float f = t * (S1 - t * (0.5f * S2 - t * (S3 * (1.0f / 6.0f)))) - target;
                    float fp = S1 - t * (S2 - 0.5f * t * S3);
                    if (!(fp > 0.f)) break;
                    t -= f / fp;
                }
                return t > 0.f ? t : 0.f;
            };
            const float sig = 5.0f * sqrtf((float)S);
            s_tlo = solve((float)S - sig);
            s_thi = solve((float)S + sig);
            s.n_direct = 0; s.n_cand = 0;
        }
        __syncthreads();
        const float tlo = s_tlo, thi = s_thi;
        // ---- clocks (one Philox block per 4 consecutive points) and classification
        for (int i4 = tid; i4 * 4 < N; i4 += kThreads) {
            uint32_t r[4];
            philox_block(i4, r);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int i = i4 * 4 + e;
                if (i >= N) break;
                const float c = clock_of(s_val[i], r[e]);
                if (c <= tlo) {
                    unsigned slot = atomicAdd(&s.n_direct, 1u);
                    if (slot < (unsigned)S) out[q * S + slot] = i;
                } else if (c <= thi) {
                    unsigned slot = atomicAdd(&s.n_cand, 1u);
                    if (slot < (unsigned)kCap) { s.cand_key[slot] = dkey((double)c); s.cand_id[slot] = i; }
                }
            }
        }
        __syncthreads();
        const unsigned n_direct = s.n_direct, n_cand = s.n_cand;
        if (n_direct <= (unsigned)S && n_direct + n_cand >= (unsigned)S && n_cand <= (unsigned)kCap) {
            sort_candidates(s, (int)n_cand);
            for (unsigned j = tid; n_direct + j < (unsigned)S; j += kThreads) out[q * S + n_direct + j] = s.cand_id[j];
            return;
        }
        __syncthreads();     // counts did not bracket S: histogram selection below (cache holds the weights)
    }
    auto keyfn = [&](int i) {
        uint32_t r[4];
        philox_block(i >> 2, r);
        const float w = CACHE ? s_val[i]
                              : weight_of(norm_f32(__fsub_rn(qx, pts[i * 3 + 0]), __fsub_rn(qy, pts[i * 3 + 1]), __fsub_rn(qz, pts[i * 3 + 2])));
        return dkey((double)clock_of(w, r[i & 3]));
    };
    find_boundary(s, N, S, kCap, keyfn);
    if (tid == 0) { s.n_direct = 0; s.n_cand = 0; }
    __syncthreads();
    const int levels = s.levels;
    for (int i = tid; i < N; i += kThreads) {
        unsigned long long key = keyfn(i);
        int c = chain_cmp(s, key, levels);
        if (c < 0) {
            unsigned slot = atomicAdd(&s.n_direct, 1u);
            if (slot < (unsigned)S) out[q * S + slot] = i;
        } else if (c == 0) {
            unsigned slot = atomicAdd(&s.n_cand, 1u);
            if (slot < (unsigned)kCap) { s.cand_key[slot] = key; s.cand_id[slot] = i; }
        }
    }
    __syncthreads();
    const unsigned n_direct = s.n_direct, n_cand = s.n_cand;
    if (n_cand > (unsigned)kCap || n_direct != s.below || n_direct + n_cand < (unsigned)S) {
        if (tid == 0) atomicExch(err_flag, 2);
        return;
    }
    sort_candidates(s, (int)n_cand);
    for (unsigned j = tid; n_direct + j < (unsigned)S; j += kThreads) out[q * S + n_direct + j] = s.cand_id[j];
}

// K3 with a cell index, by rejection: the same successive-sampling law with a fraction of the work when N >= 2 S.
// Drawing without replacement with probabilities ~ w_i is: propose a point, accept it so that proposing-and-accepting point i
// has probability ~ w_i, skip points that were already taken, repeat until S points are taken.  Proposal j of query q is a
// fixed function of (seed, q, j) (Philox block j / 2 -> two (slot, uniform) pairs), so the accepted set -- the first S
// distinct accepted proposals in proposal order -- does not depend on how the proposals are spread over threads and rounds,
// and there is no selection or sort.
// The cloud is binned once per shape into kCG^3 cells (points in cell order, a tight box per cell).  Per query, a cell's
// weight bound wq_c >= max_{i in c} w_i follows from the distance to its box (w is non-increasing in the distance); a
// proposal picks a cell with probability ~ count_c * wq_c and a point uniformly inside it -- ONE integer drawn uniformly
// from [0, sum_c count_c * wq_c) gives both -- and is accepted with probability w_i / wq_c.  The probability of proposing and
// accepting point i is then ~ w_i exactly as for uniform proposals, but ~70 % of the proposals are accepted instead of
// ~17 % (mean weight on a surface cloud).  The maximum distance (the weights' normalisation) is exact: only cells whose
// farthest corner beats the best first-point distance are scanned.  Bounds are quantised UP to multiples of 1/65535, so
// every probability above is an exact integer ratio; 40 random bits select the slot (relative error of a point's
// probability <= 2e-7).
constexpr int kRejPer = 8;        // proposals per thread and round (upper bound); even
constexpr int kRejRounds = 256;
constexpr int kCG = 12, kCC = kCG * kCG * kCG;                 // 1728 cells
constexpr int kCPT = (kCC + kThreads - 1) / kThreads;          // consecutive cells per thread (7)

__global__ void __launch_bounds__(1024) ci_bbox_kernel(const float* __restrict__ pts, int N, float* __restrict__ meta) {
    __shared__ float red[6][32];
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = threadIdx.x; i < N; i += 1024)
#pragma unroll
        for (int a = 0; a < 3; ++a) { const float v = pts[i * 3 + a]; lo[a] = fminf(lo[a], v); hi[a] = fmaxf(hi[a], v); }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o)); hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o)); }
        if ((threadIdx.x & 31) == 0) { red[a][threadIdx.x >> 5] = lo[a]; red[3 + a][threadIdx.x >> 5] = hi[a]; }
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        const int a = threadIdx.x;
        float l = red[a][0], h = red[3 + a][0];
        for (int w = 1; w < 32; ++w) { l = fminf(l, red[a][w]); h = fmaxf(h, red[3 + a][w]); }
        meta[a] = l;
        meta[3 + a] = (h > l) ? (float)kCG / (h - l) : 0.f;
    }
}

__device__ __forceinline__ int ci_cell_of(const float* __restrict__ meta, float x, float y, float z) {
    const int ix = min(kCG - 1, max(0, (int)((x - meta[0]) * meta[3])));
    const int iy = min(kCG - 1, max(0, (int)((y - meta[1]) * meta[4])));
    const int iz = min(kCG - 1, max(0, (int)((z - meta[2]) * meta[5])));
    return (ix * kCG + iy) * kCG + iz;
}

__global__ void ci_key_kernel(const float* __restrict__ pts, int N, const float* __restrict__ meta, uint32_t* __restrict__ key, int32_t* __restrict__ val) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    key[i] = (uint32_t)ci_cell_of(meta, pts[i * 3 + 0], pts[i * 3 + 1], pts[i * 3 + 2]);
    val[i] = i;
}

// one thread per cell: its range in the (stably) sorted order, the points in that order, their tight box
__global__ void ci_finish_kernel(const float* __restrict__ pts, int N, const uint32_t* __restrict__ key_s, const int32_t* __restrict__ perm,
                                 int32_t* __restrict__ start, float* __restrict__ spts, float* __restrict__ cbox) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > kCC) return;
    int lo = 0, hi = N;                       // lower bound of key >= c
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (key_s[mid] < (uint32_t)c) lo = mid + 1; else hi = mid; }
    start[c] = lo;
    if (c == kCC) return;
    float bl[3] = {INFINITY, INFINITY, INFINITY}, bh[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = lo; i < N && key_s[i] == (uint32_t)c; ++i) {
        const int id = perm[i];
#pragma unroll
        for (int a = 0; a < 3; ++a) { const float v = pts[id * 3 + a]; spts[i * 3 + a] = v; bl[a] = fminf(bl[a], v); bh[a] = fmaxf(bh[a], v); }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) { cbox[c * 6 + a] = bl[a]; cbox[c * 6 + 3 + a] = bh[a]; }
}

__global__ void __launch_bounds__(kThreads, 4)
subsample_cells_kernel(const CloudIndex ix, int N, const float* __restrict__ queries, int64_t qbase, const int32_t* __restrict__ qidx, int S,
                       uint64_t seed, int32_t* __restrict__ out_ids, float* __restrict__ out_pts, int* __restrict__ err_flag) {
    extern __shared__ int s_first[];             // [N] position of the first accepted proposal of sorted point i
    __shared__ uint32_t s_prefix[kCC];           // inclusive prefix sums of count_c * wq_c
    __shared__ uint16_t s_wq[kCC];
    __shared__ float redf[kThreads / 32];
    __shared__ uint32_t redu[kThreads / 32];
    __shared__ int redi[kThreads / 32];
    __shared__ float s_bcast;
    __shared__ int s_nfar;
    int2* s_far = reinterpret_cast<int2*>(s_prefix);      // far-cell list (start, count); the prefix sums are written later
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t q = blockIdx.x;
    const float qx = queries[q * 3 + 0], qy = queries[q * 3 + 1], qz = queries[q * 3 + 2];
    const uint64_t qi = (uint64_t)(qbase + (qidx ? (int64_t)qidx[q] : q));
    const float* __restrict__ spts = ix.spts;
    auto dist2 = [&](int j) {        // float32 like NumPy: (dx*dx + dy*dy) + dz*dz, every operation rounded
        const float dx = __fsub_rn(qx, spts[j * 3 + 0]), dy = __fsub_rn(qy, spts[j * 3 + 1]), dz = __fsub_rn(qz, spts[j * 3 + 2]);
        return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
    };
    auto block_max = [&](float v) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
        __syncthreads();                       // previous readers of redf / s_bcast are done
        if (lane == 0) redf[warp] = v;
        __syncthreads();
        if (tid == 0) { float m = redf[0]; for (int w = 1; w < kThreads / 32; ++w) m = fmaxf(m, redf[w]); s_bcast = m; }
        __syncthreads();
        return s_bcast;
    };
    for (int i = tid; i < N; i += kThreads) s_first[i] = 0x7fffffff;
    // ---- own cells: distance bounds to the box, first-point distance (a lower bound of the maximum distance)
    const int c0 = tid * kCPT;
    int cst[kCPT], cnt[kCPT];
    float dmin2[kCPT], dfar2[kCPT];
    float lb2 = 0.f;
#pragma unroll
    for (int k = 0; k < kCPT; ++k) {
        const int c = c0 + k;
        cst[k] = 0; cnt[k] = 0; dmin2[k] = 0.f; dfar2[k] = 0.f;
        if (c < kCC) {
            cst[k] = ix.start[c]; cnt[k] = ix.start[c + 1] - cst[k];
            if (cnt[k] > 0) {
                const float* b = ix.cbox + c * 6;
                const float nx = fmaxf(fmaxf(b[0] - qx, qx - b[3]), 0.f), ny = fmaxf(fmaxf(b[1] - qy, qy - b[4]), 0.f), nz = fmaxf(fmaxf(b[2] - qz, qz - b[5]), 0.f);
                const float fx = fmaxf(fabsf(qx - b[0]), fabsf(qx - b[3])), fy = fmaxf(fabsf(qy - b[1]), fabsf(qy - b[4])), fz = fmaxf(fabsf(qz - b[2]), fabsf(qz - b[5]));
                dmin2[k] = nx * nx + ny * ny + nz * nz;
                dfar2[k] = fx * fx + fy * fy + fz * fz;
                lb2 = fmaxf(lb2, dist2(cst[k]));
            }
        }
    }
    if (tid == 0) s_nfar = 0;
    const float best_lb2 = block_max(lb2);
    // ---- exact maximum distance: only cells whose farthest corner can beat the best first-point distance.  The distance to
    // the far side of a surface is flat, so this is still a fifth of the cloud: the cells go to a shared list and are scanned
    // a warp per cell, four cells in flight (a thread walking its own cells was one dependent gather after the other).
    constexpr int kFarCap = kCC / 2;                  // int2 entries that fit into the prefix array
    float m2 = lb2;
#pragma unroll
    for (int k = 0; k < kCPT; ++k)
        if (cnt[k] > 1 && dfar2[k] * 1.00001f >= best_lb2) {
            const int slot = atomicAdd(&s_nfar, 1);
            if (slot < kFarCap) s_far[slot] = make_int2(cst[k] + 1, cnt[k] - 1);        // (the first point is already in lb2)
            else for (int j = cst[k] + 1; j < cst[k] + cnt[k]; ++j) m2 = fmaxf(m2, dist2(j));   // list full: scan in place
        }
    __syncthreads();
    {
        const int L = min(s_nfar, kFarCap);
        for (int it = warp * 4; it < L; it += (kThreads / 32) * 4) {
            int2 rg[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) rg[u] = (it + u < L) ? s_far[it + u] : make_int2(0, 0);
            float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int u = 0; u < 4; ++u) if (lane < rg[u].y) d[u] = dist2(rg[u].x + lane);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                m2 = fmaxf(m2, d[u]);
                for (int j = lane + 32; j < rg[u].y; j += 32) m2 = fmaxf(m2, dist2(rg[u].x + j));     // cells with more than 32 points
            }
        }
    }
    const float dmax = __fsqrt_rn(block_max(m2));    // max of float32 norms = sqrt of the max float32 squared sum (sqrt is monotone)
    auto weight_of = [&](float d) {                  // dist_prob (utils.py:200-208), float32 like NumPy; non-increasing in d
        return fminf(fmaxf(__fsub_rn(1.0f, __fmul_rn(1.5f, __fdiv_rn(d, dmax))), 0.05f), 1.0f);
    };
    // ---- cell weights (bounds rounded UP to multiples of 1/65535) and their prefix sums
    uint32_t wsum = 0, wq[kCPT];
#pragma unroll
    for (int k = 0; k < kCPT; ++k) {
        wq[k] = 0;
        if (cnt[k] > 0) {
            const float wmax = weight_of(sqrtf(dmin2[k]) * 0.99999f);     // distance to the box, shrunk: a safe lower bound of every d_i
            wq[k] = min(65535u, (uint32_t)ceilf(wmax * 65535.0f) + 1u);
            wsum += (uint32_t)cnt[k] * wq[k];
        }
    }
    uint32_t incl = wsum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) redu[warp] = incl;
    __syncthreads();
    uint32_t run = incl - wsum, total = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) { const uint32_t c = redu[w]; if (w < warp) run += c; total += c; }
#pragma unroll
    for (int k = 0; k < kCPT; ++k) {
        const int c = c0 + k;
        if (c < kCC) { run += (uint32_t)cnt[k] * wq[k]; s_prefix[c] = run; s_wq[c] = (uint16_t)wq[k]; }
    }
    __syncthreads();
    // ---- proposal rounds
    int base = 0, pos0 = 0, per = 6;
    for (int round = 0; round < kRejRounds; ++round) {
        const int mypos = pos0 + tid * per;
        int idx[kRejPer];
        unsigned acc = 0;
        // The proposals of a thread are processed in lock step, phase by phase, so that their shared-memory searches and their
        // gathers overlap (one proposal after the other was a chain of ~15 dependent memory accesses each).
        uint32_t xs[kRejPer];
        float us[kRejPer];
#pragma unroll
        for (int e2 = 0; e2 < kRejPer / 2; ++e2) {
            uint32_t r[4] = {0u, 0u, 0u, 0u};
            if (2 * e2 < per)
                philox4x32_10((uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)qi, (uint32_t)(qi >> 32), (uint32_t)((mypos >> 1) + e2), 0x85ebca6bu, r);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                // 40 random bits -> slot x in [0, total)
                const unsigned long long x40 = ((unsigned long long)r[2 * h] << 32) | ((unsigned long long)(r[2 * h + 1] & 0xffu) << 24);
                xs[2 * e2 + h] = (uint32_t)__umul64hi(x40, (unsigned long long)total);
                us[2 * e2 + h] = (2 * e2 < per) ? (float)(r[2 * h + 1] >> 8) * (1.0f / 16777216.0f) : 1e30f;    // [0, 1); 1e30 = never accepted
            }
        }
        int cel[kRejPer];          // number of prefix sums <= x  =  smallest cell with s_prefix[c] > x
#pragma unroll
        for (int e = 0; e < kRejPer; ++e) cel[e] = 0;
#pragma unroll
        for (int step = 1024; step >= 1; step >>= 1) {
#pragma unroll
            for (int e = 0; e < kRejPer; ++e) {
                const int np = cel[e] + step;
                if (np <= kCC && s_prefix[np - 1] <= xs[e]) cel[e] = np;
            }
        }
        float wqf[kRejPer];
#pragma unroll
        for (int e = 0; e < kRejPer; ++e) {
            const int c = cel[e];
            const uint32_t wqc = s_wq[c];
            const uint32_t off = xs[e] - (c ? s_prefix[c - 1] : 0u);
            idx[e] = ix.start[c] + (int)(off / wqc);
            wqf[e] = (float)wqc * (1.0f / 65535.0f);
        }
        float d2[kRejPer];
#pragma unroll
        for (int e = 0; e < kRejPer; ++e) d2[e] = dist2(idx[e]);
#pragma unroll
        for (int e = 0; e < kRejPer; ++e) {
            const float w = weight_of(__fsqrt_rn(d2[e]));
            if (us[e] * wqf[e] < w) { acc |= 1u << e; atomicMin(&s_first[idx[e]], mypos + e); }
        }
        __syncthreads();
        unsigned fresh = 0;
#pragma unroll
        for (int e = 0; e < kRejPer; ++e)
            if (((acc >> e) & 1u) && s_first[idx[e]] == mypos + e) fresh |= 1u << e;
        const int cntf = __popc(fresh);
        int inc = cntf;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        if (lane == 31) redi[warp] = inc;
        __syncthreads();
        int wbase = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < kThreads / 32; ++w) { const int c = redi[w]; if (w < warp) wbase += c; tot += c; }
        int slot = base + wbase + inc - cntf;
#pragma unroll
        for (int e = 0; e < kRejPer; ++e) {
            if ((fresh >> e) & 1u) {
                if (slot < S) {
                    const int j = idx[e];
                    out_ids[q * S + slot] = ix.perm[j];
                    if (out_pts) {
                        float* o = out_pts + (q * S + slot) * 3;
                        o[0] = spts[j * 3 + 0]; o[1] = spts[j * 3 + 1]; o[2] = spts[j * 3 + 2];
                    }
                }
                ++slot;
            }
        }
        base += tot;
        if (base >= S) return;
        pos0 += kThreads * per;
        const long long need = ((long long)(S - base) * (kThreads * per) * 23 / 20) / (tot > 0 ? tot : 1) + 1;
        const long long p2 = (need + 2 * kThreads - 1) / (2 * kThreads);
        per = (int)(p2 < 1 ? 1 : (p2 > kRejPer / 2 ? kRejPer / 2 : p2)) * 2;
        __syncthreads();
    }
    if (tid == 0) atomicExch(err_flag, 2);
}

__global__ void gather_points_kernel(const float* __restrict__ pts, const int32_t* __restrict__ ids, int64_t count, float* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    int id = ids[i];
    out[i * 3 + 0] = pts[id * 3 + 0];
    out[i * 3 + 1] = pts[id * 3 + 1];
    out[i * 3 + 2] = pts[id * 3 + 2];
}

}  // namespace

void gather_points(const float* pts, const int32_t* ids, int64_t count, float* out, cudaStream_t st);

int assemble_error_check(cudaStream_t st) {  // sync; returns and clears the device error flag
    int h = 0;
    int* f = device_ctx().err_flag;
    P2S_CUDA(cudaMemcpyAsync(&h, f, sizeof(int), cudaMemcpyDeviceToHost, st));
    P2S_CUDA(cudaStreamSynchronize(st));
    if (h) P2S_CUDA(cudaMemsetAsync(f, 0, sizeof(int), st));
    return h;
}

void knn_patch(const float* pts, int64_t N, const float* queries, int64_t Q, int k, int32_t* ids,
               float* patch, float* radius, cudaStream_t st) {
    P2S_CHECK(N >= k, "kNN needs N >= k (the reference returns out-of-range ids otherwise)");
    P2S_CHECK(k >= 1 && k <= kBallMaxK, "k must be in [1, 1536]");
    P2S_CHECK(N < (1 << 30), "cloud too large");
    if (Q <= 0) return;
    // Run length: with 8 queries per CTA a batch of 8 192 queries is 1 024 CTAs = 1.4 waves of the 740 co-resident CTAs, i.e.
    // two waves with the second 38 % full.  Lengthen the runs so that the whole batch is ONE wave (longer runs also amortise
    // the histogram selection of a run's first query better).
    DeviceCtx& ctx = device_ctx();
    if (!ctx.knn_slots_small) {
        int a = 0, b = 0;
        P2S_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, knn_patch_kernel<kCap>, kThreads, 0));
        P2S_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, knn_patch_kernel<kCapBig>, kThreads, 0));
        ctx.knn_slots_small = ctx.sm_count * (a > 0 ? a : 1); ctx.knn_slots_big = ctx.sm_count * (b > 0 ? b : 1);
    }
    const int slots = k <= 512 ? ctx.knn_slots_small : ctx.knn_slots_big;
    int run = (int)cdiv(Q, slots);
    if (run < kRun) run = kRun;
    if (run > 64) run = 64;
    if (k <= 512) P2S_LAUNCH(knn_patch_kernel<kCap>, (unsigned)cdiv(Q, run), kThreads, 0, st, pts, (int)N, queries, Q, k, ids, patch, radius, ctx.err_flag, run);
    else P2S_LAUNCH(knn_patch_kernel<kCapBig>, (unsigned)cdiv(Q, run), kThreads, 0, st, pts, (int)N, queries, Q, k, ids, patch, radius, ctx.err_flag, run);
}

// the Philox stream of query q is keyed by qbase + (qidx ? qidx[q] : q), like the sub-sampler's
void ball_patch(const float* pts, int64_t N, const float* queries, int64_t Q, int64_t qbase, int k, double patch_radius,
                uint64_t seed, int32_t* ids, float* patch, float* radius, int32_t* counts, cudaStream_t st, const int32_t* qidx) {
    P2S_CHECK(patch_radius > 0.0, "ball query needs patch_radius > 0");
    P2S_CHECK(k >= 1 && k <= kBallMaxK, "points_per_patch must be in [1, 1536]");
    P2S_CHECK(N >= 1 && N < (1 << 30), "bad cloud size");
    if (Q <= 0) return;
    P2S_LAUNCH(ball_patch_kernel, (unsigned)Q, kThreads, 0, st, pts, (int)N, queries, qbase, qidx, k, patch_radius * patch_radius,
               (float)patch_radius, seed, ids, patch, radius, counts, device_ctx().err_flag);
}

// Cell index of a cloud for the weighted sub-sampler: bounding box -> cell keys -> stable radix sort (points of a cell keep
// their id order, so the result is deterministic) -> per-cell ranges, sorted points, tight boxes.  The index lives in the
// device context and is valid until the next call on this thread and device (stream order).
constexpr size_t kSubsampleCacheBytes = 160 * 1024;   // dynamic shared memory of the cell and cached clock kernels: 4 B per point

bool cloud_index_usable(int64_t N, int S, int mode) {
    return mode == P2S_SUBSAMPLE_WEIGHTED && N >= 2 * (int64_t)S && (size_t)N * 4 <= kSubsampleCacheBytes;
}

const CloudIndex* cloud_index_build(const float* pts, int64_t N, cudaStream_t st) {
    DeviceCtx& ctx = device_ctx();
    const int n = (int)N;
    size_t cub_bytes = 0;
    P2S_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const int32_t*)nullptr, (int32_t*)nullptr, n, 0, 11, st));
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    size_t off = 0;
    const size_t o_meta = off; off += al(6 * 4);
    const size_t o_key = off; off += al((size_t)n * 4);
    const size_t o_val = off; off += al((size_t)n * 4);
    const size_t o_keys = off; off += al((size_t)n * 4);
    const size_t o_perm = off; off += al((size_t)n * 4);
    const size_t o_start = off; off += al((size_t)(kCC + 1) * 4);
    const size_t o_spts = off; off += al((size_t)n * 12);
    const size_t o_cbox = off; off += al((size_t)kCC * 24);
    const size_t o_cub = off; off += al(cub_bytes);
    uint8_t* b = (uint8_t*)ctx.cloud_ws.get(off);
    float* meta = (float*)(b + o_meta);
    uint32_t* key = (uint32_t*)(b + o_key); int32_t* val = (int32_t*)(b + o_val);
    uint32_t* key_s = (uint32_t*)(b + o_keys); int32_t* perm = (int32_t*)(b + o_perm);
    P2S_LAUNCH(ci_bbox_kernel, 1, 1024, 0, st, pts, n, meta);
    P2S_LAUNCH(ci_key_kernel, (unsigned)cdiv(n, 256), 256, 0, st, pts, n, meta, key, val);
    P2S_CUDA(cub::DeviceRadixSort::SortPairs(b + o_cub, cub_bytes, key, key_s, val, perm, n, 0, 11, st));    // kCC = 1728 < 2^11
    g_launches.fetch_add(3, std::memory_order_relaxed);
    P2S_LAUNCH(ci_finish_kernel, (unsigned)cdiv(kCC + 1, 128), 128, 0, st, pts, n, key_s, perm, (int32_t*)(b + o_start), (float*)(b + o_spts), (float*)(b + o_cbox));
    CloudIndex& ci = ctx.cloud_index;
    ci.meta = meta; ci.spts = (const float*)(b + o_spts); ci.perm = perm; ci.start = (const int32_t*)(b + o_start); ci.cbox = (const float*)(b + o_cbox);
    return &ci;
}

// the Philox stream of query q is keyed by qbase + (qidx ? qidx[q] : q).  pts_out (optional): [Q, S, 3] the selected
// points themselves (what gather_points would produce from `out`).  cidx (optional): the cloud's cell index (built here if
// the cell sampler applies and none is given).
void subsample(const float* pts, int64_t N, const float* queries, int64_t Q, int64_t qbase, int S,
               int mode, uint64_t seed, int32_t* out, cudaStream_t st, const int32_t* qidx, float* pts_out, const CloudIndex* cidx) {
    P2S_CHECK(N >= S, "sub-sample needs N >= sub_sample_size (reference zero-pads after an in-place shuffle; unsupported)");
    P2S_CHECK(N < (1 << 30), "cloud too large");
    if (Q <= 0) return;
    bool gathered = false;
    if (mode == P2S_SUBSAMPLE_UNIFORM) {
        int64_t threads = Q * ((S + 3) / 4);
        P2S_LAUNCH(subsample_uniform_kernel, (unsigned)cdiv(threads, 256), 256, 0, st, (int)N, Q, qbase, qidx, S, seed, out);
    } else if (mode == P2S_SUBSAMPLE_WEIGHTED) {
        const size_t cache_bytes = (size_t)N * sizeof(float);
        DeviceCtx& ctx = device_ctx();
        if (cloud_index_usable(N, S, mode)) {
            // rejection over the cell index: cheap when at most half of the cloud is drawn
            if (!cidx) cidx = cloud_index_build(pts, N, st);
            ctx.set_max_dynamic_smem((const void*)subsample_cells_kernel, (int)kSubsampleCacheBytes);
            P2S_LAUNCH(subsample_cells_kernel, (unsigned)Q, kThreads, cache_bytes, st, *cidx, (int)N, queries, qbase, qidx, S, seed, out, pts_out, ctx.err_flag);
            gathered = true;
        } else if (cache_bytes <= kSubsampleCacheBytes) {
            ctx.set_max_dynamic_smem((const void*)subsample_weighted_kernel<true>, (int)kSubsampleCacheBytes);
            P2S_LAUNCH(subsample_weighted_kernel<true>, (unsigned)Q, kThreads, cache_bytes, st, pts, (int)N, queries, qbase, qidx, S, seed, out, ctx.err_flag);
        } else {
            P2S_LAUNCH(subsample_weighted_kernel<false>, (unsigned)Q, kThreads, 0, st, pts, (int)N, queries, qbase, qidx, S, seed, out, ctx.err_flag);
        }
    } else {
        throw Error("unknown sub-sample mode");
    }
    if (pts_out && !gathered) gather_points(pts, out, Q * S, pts_out, st);
}

// rows of `words` 32-bit words: dst[i] = src[rows[i]] (gather), dst[rows[i]] = src[i] (scatter), for i < n
__global__ void gather_rows_kernel(const uint32_t* __restrict__ src, const int32_t* __restrict__ rows, int64_t n, int words, uint32_t* __restrict__ dst) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * words) return;
    const int64_t i = e / words;
    dst[e] = src[(int64_t)rows[i] * words + (e - i * words)];
}
__global__ void scatter_rows_kernel(const uint32_t* __restrict__ src, const int32_t* __restrict__ rows, int64_t n, int words, uint32_t* __restrict__ dst) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * words) return;
    const int64_t i = e / words;
    dst[(int64_t)rows[i] * words + (e - i * words)] = src[e];
}
void gather_rows(const void* src, const int32_t* rows, int64_t n, int words, void* dst, cudaStream_t st) {
    if (n > 0) P2S_LAUNCH(gather_rows_kernel, (unsigned)cdiv(n * words, 256), 256, 0, st, (const uint32_t*)src, rows, n, words, (uint32_t*)dst);
}
void scatter_rows(const void* src, const int32_t* rows, int64_t n, int words, void* dst, cudaStream_t st) {
    if (n > 0) P2S_LAUNCH(scatter_rows_kernel, (unsigned)cdiv(n * words, 256), 256, 0, st, (const uint32_t*)src, rows, n, words, (uint32_t*)dst);
}

void gather_points(const float* pts, const int32_t* ids, int64_t count, float* out, cudaStream_t st) {
    if (count <= 0) return;
    P2S_LAUNCH(gather_points_kernel, (unsigned)cdiv(count, 256), 256, 0, st, pts, ids, count, out);
}

}  // namespace p2s
