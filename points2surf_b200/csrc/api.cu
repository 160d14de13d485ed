// C-ABI entry points of libp2s_b200.so (include/p2s_b200.h) and the fused reconstruction pipeline.
#include "model.cuh"

namespace p2s {

thread_local std::string g_last_error;
std::atomic<uint64_t> g_launches{0};

DeviceCtx& device_ctx() {
    // the device memory of a context is never freed (a thread's exit may come after the CUDA runtime's)
    static thread_local std::vector<std::unique_ptr<DeviceCtx>> table;
    int dev = 0;
    P2S_CUDA(cudaGetDevice(&dev));
    if ((int)table.size() <= dev) table.resize(dev + 1);
    if (!table[dev]) {
        auto c = std::make_unique<DeviceCtx>();
        c->device = dev;
        P2S_CUDA(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, dev));
        P2S_CUDA(cudaMalloc(&c->err_flag, sizeof(int)));
        P2S_CUDA(cudaMemset(c->err_flag, 0, sizeof(int)));
        table[dev] = std::move(c);
    }
    return *table[dev];
}

void DeviceCtx::set_max_dynamic_smem(const void* fn, int bytes) {
    for (auto& f : smem_limits) {
        if (f.first != fn) continue;
        if (f.second < bytes) {
            P2S_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
            f.second = bytes;
        }
        return;
    }
    P2S_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    smem_limits.emplace_back(fn, bytes);
}

// grid.cu / assemble.cu / volume.cu / mc.cu
void query_grid(const float* pts, int64_t N, int res, int eps, int32_t* lin_idx, int64_t cap, int64_t* count_host, cudaStream_t st);
void query_points(const int32_t* lin_idx, int64_t Q, int res, float* out, cudaStream_t st);
void knn_patch(const float* pts, int64_t N, const float* queries, int64_t Q, int k, int32_t* ids, float* patch, float* radius, cudaStream_t st);
void ball_patch(const float* pts, int64_t N, const float* queries, int64_t Q, int64_t qbase, int k, double patch_radius, uint64_t seed, int32_t* ids, float* patch, float* radius, int32_t* counts, cudaStream_t st, const int32_t* qidx = nullptr);
bool cloud_index_usable(int64_t N, int S, int mode);
const CloudIndex* cloud_index_build(const float* pts, int64_t N, cudaStream_t st);
void subsample(const float* pts, int64_t N, const float* queries, int64_t Q, int64_t qbase, int S, int mode, uint64_t seed, int32_t* out, cudaStream_t st, const int32_t* qidx = nullptr, float* pts_out = nullptr, const CloudIndex* cidx = nullptr);
void gather_rows(const void* src, const int32_t* rows, int64_t n, int words, void* dst, cudaStream_t st);
void scatter_rows(const void* src, const int32_t* rows, int64_t n, int words, void* dst, cudaStream_t st);
void gather_points(const float* pts, const int32_t* ids, int64_t count, float* out, cudaStream_t st);
int assemble_error_check(cudaStream_t st);
void sdf_from_logits(const float* logits, const float* radius, int64_t B, float* sdf, cudaStream_t st);
void sdf_to_volume(const int32_t* lin_idx, const float* sdf, int64_t Q, int res, int sigma, float thr, float* vol, int* iterations_host, cudaStream_t st);
void marching_cubes(const float* vol, int res, float level, float* verts, int64_t vcap, int32_t* faces, int64_t fcap, int64_t* nverts_host, int64_t* nfaces_host, cudaStream_t st);

}  // namespace p2s
#include <chrono>
#include <map>
namespace p2s {
static std::map<std::string, std::pair<double, long>> g_stage;
bool StageTimer::enabled() { static int e = -1; if (e < 0) { const char* v = getenv("P2S_STAGE_TIMING"); e = (v && v[0] == '1') ? 1 : 0; } return e == 1; }
void StageTimer::add(const char* label, double ms) { auto& x = g_stage[label]; x.first += ms; x.second += 1; }
void StageTimer::report() {
    if (!enabled() || g_stage.empty()) return;
    double tot = 0; for (auto& kv : g_stage) tot += kv.second.first;
    fprintf(stderr, "p2s stage timing (host wall clock, stream synchronised around each stage):\n");
    for (auto& kv : g_stage) fprintf(stderr, "  %-28s %10.2f ms  %5.1f%%  (%ld calls)\n", kv.first.c_str(), kv.second.first, 100.0 * kv.second.first / tot, kv.second.second);
    g_stage.clear();
}
static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
StageScope::StageScope(const char* l, cudaStream_t s) : label(l), st(s), on(StageTimer::enabled()) { if (on) { cudaStreamSynchronize(st); t0 = now_ms(); } }
StageScope::~StageScope() { if (on) { cudaStreamSynchronize(st); StageTimer::add(label, now_ms() - t0); } }

namespace {

struct BlobCursor {
    const float* p;
    size_t left;
    Layer take(int cout, int cin) {
        size_t need = (size_t)cout * cin + cout;
        P2S_CHECK(left >= need, "weight blob too short");
        Layer L;
        L.W = p; L.b = p + (size_t)cout * cin; L.cout = cout; L.cin = cin;
        p += need; left -= need;
        return L;
    }
};

Stn take_stn(BlobCursor& c, int dim, int out, int net) {
    Stn s;
    s.c1 = c.take(64, dim); s.c2 = c.take(128, 64); s.c3 = c.take(net, 128);
    s.fc1 = c.take(net / 2, net); s.fc2 = c.take(net / 4, net / 2); s.fc3 = c.take(out, net / 4);
    return s;
}

Feat take_feat(BlobCursor& c, bool qstn, int net) {
    Feat f;
    f.has_qstn = qstn;
    if (qstn) f.stn1 = take_stn(c, 3, 4, net);
    f.stn2 = take_stn(c, 64, 4096, net);
    f.conv0a = c.take(64, 3); f.conv0b = c.take(64, 64);
    f.conv1 = c.take(64, 64); f.conv2 = c.take(128, 64); f.conv3 = c.take(net, 128);
    return f;
}

size_t stn_floats(int dim, int out, int net) {
    auto l = [](size_t co, size_t ci) { return co * ci + co; };
    return l(64, dim) + l(128, 64) + l(net, 128) + l(net / 2, net) + l(net / 4, net / 2) + l(out, net / 4);
}
size_t feat_floats(bool qstn, int net) {
    auto l = [](size_t co, size_t ci) { return co * ci + co; };
    return (qstn ? stn_floats(3, 4, net) : 0) + stn_floats(64, 4096, net) + l(64, 3) + l(64, 64) + l(64, 64) + l(128, 64) + l(net, 128);
}
size_t blob_floats(const p2s_model_config& c) {
    auto l = [](size_t co, size_t ci) { return co * ci + co; };
    const int net = c.net_size;
    const bool shared = c.use_point_stn && c.shared_transformer;
    const bool gq = c.use_point_stn && !c.shared_transformer;
    return (shared ? stn_floats(3, 4, net) : 0) + feat_floats(false, net) + feat_floats(gq, net) +
           2 * l(net / 2, net) + l(net / 4, net) + l(net / 8, net / 4) + l(2, net / 8);
}

void check_cfg(const p2s_model_config& c) {
    P2S_CHECK(c.net_size == 1024, "only net_size 1024 is supported");
    P2S_CHECK(c.points_per_patch >= 8 && c.points_per_patch <= 1536, "points_per_patch must be in [8, 1536]");
    P2S_CHECK(c.sub_sample_size >= 8 && c.sub_sample_size <= 4096, "sub_sample_size must be in [8, 4096]");
}

cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// assembled batch buffers for the fused pipeline
struct BatchBufs {
    float *qpts, *patch, *radius, *sub, *logits;
    int32_t* sub_ids;
};

}  // namespace

// the network without the guard band
static void forward_fast(Model& m, const float* patch, const float* sub, const float* query, int64_t B, float* logits, cudaStream_t st) {
    if (m.precision == P2S_PRECISION_TC) forward_tc(m, patch, sub, query, B, logits, st, false);
    else forward_fp32(m, patch, sub, query, B, logits, st);
}

// guard band of the tensor-core path: queries whose |sign logit| < guard_band, too close to 0 for fp16-operand arithmetic,
// are recomputed by the split-precision pass
static bool guard_on(const Model& m) { return m.precision == P2S_PRECISION_TC && m.guard_band > 0.f; }

static void forward(Model& m, const float* patch, const float* sub, const float* query, int64_t B, float* logits, cudaStream_t st) {
    if (B <= 0) return;
    forward_fast(m, patch, sub, query, B, logits, st);
    if (!guard_on(m)) return;
    StageScope ts_guard("net: guard-band split-precision recompute", st);
    int32_t* list = m.ws_guard.as<int32_t>((size_t)B + 64);
    int* count = reinterpret_cast<int*>(list + B);
    P2S_CUDA(cudaMemsetAsync(count, 0, sizeof(int), st));
    guard_flag(logits, B, m.guard_band, 0, list, count, B, st);
    int n = 0;
    P2S_CUDA(cudaMemcpyAsync(&n, count, sizeof(int), cudaMemcpyDeviceToHost, st));
    P2S_CUDA(cudaStreamSynchronize(st));
    m.last_guard_count += n;
    if (n == 0) return;
    const int rowp = m.cfg.points_per_patch * 3, rows = m.cfg.sub_sample_size * 3;
    float* gp = m.ws_misc.as<float>((size_t)n * (rowp + rows + 3 + 2) + 64);
    float* gs = gp + (size_t)n * rowp; float* gq = gs + (size_t)n * rows; float* gl = gq + ((size_t)n * 3 + 3) / 4 * 4;
    gather_rows(patch, list, n, rowp, gp, st);
    gather_rows(sub, list, n, rows, gs, st);
    gather_rows(query, list, n, 3, gq, st);
    forward_tc(m, gp, gs, gq, n, gl, st, true);
    scatter_rows(gl, list, n, 2, logits, st);
}

static void reconstruct(Model& m, const p2s_recon_config& rc, const float* pts, int64_t N, int64_t first_query,
                        int64_t num_queries, int32_t* lin_idx, float* sdf, int64_t cap, int64_t* Q_host, cudaStream_t st) {
    P2S_CHECK(rc.res >= 2 && rc.eps >= 1 && rc.reserved == 0, "bad reconstruction config");
    const bool fixed_radius = rc.patch_radius > 0.f;      // ball-query patches: |d| is not rescaled (points_to_surf_eval.py:364-368)
    const int P = m.cfg.points_per_patch, S = m.cfg.sub_sample_size;
    int64_t Qall = 0;
    const int64_t vox = (int64_t)rc.res * rc.res * rc.res;
    int32_t* all_idx = m.ws_misc.as<int32_t>((size_t)vox + 64);   // worst case candidate list
    { StageScope t("grid", st); query_grid(pts, N, rc.res, rc.eps, all_idx, vox, &Qall, st); }
    if (first_query < 0) first_query = 0;
    if (first_query > Qall) first_query = Qall;
    int64_t Q = (num_queries < 0) ? (Qall - first_query) : num_queries;
    if (first_query + Q > Qall) Q = Qall - first_query;
    *Q_host = Q;
    P2S_CHECK(Q <= cap, "output capacity too small for the query slab");
    if (Q == 0) return;
    P2S_CUDA(cudaMemcpyAsync(lin_idx, all_idx + first_query, (size_t)Q * 4, cudaMemcpyDeviceToDevice, st));
    int64_t batch = rc.batch > 0 ? rc.batch : (m.precision == P2S_PRECISION_TC ? 8192 : 2048);
    if (batch > Q) batch = Q;
    size_t per_q = 3 + (size_t)P * 3 + 1 + (size_t)S * 3 + 2 + (size_t)S;
    float* base = m.ws_io.as<float>(per_q * (size_t)batch + 64);
    BatchBufs b;
    float* p = base;
    auto take = [&](size_t n) { float* r = p; p += (n * (size_t)batch + 3) / 4 * 4; return r; };
    b.qpts = take(3); b.patch = take((size_t)P * 3); b.radius = take(1); b.sub = take((size_t)S * 3); b.logits = take(2);
    b.sub_ids = reinterpret_cast<int32_t*>(take((size_t)S));
    // guard band: flagged queries are collected over the whole slab and recomputed at the end, in batches of the same
    // size (large GEMMs instead of ~80-query slivers per batch).  ws_guard holds the slab-relative indices of the flagged
    // queries [Q], their voxel indices and SDF values of one recompute batch [batch each], and their count.
    const bool guard = guard_on(m);
    int32_t* glist = nullptr;
    int32_t* glin = nullptr;
    float* gsdf = nullptr;
    int* gcount = nullptr;
    if (guard) {
        glist = m.ws_guard.as<int32_t>((size_t)Q + 2 * (size_t)batch + 1);
        glin = glist + Q;
        gsdf = reinterpret_cast<float*>(glin + batch);
        gcount = reinterpret_cast<int*>(gsdf + batch);
        P2S_CUDA(cudaMemsetAsync(gcount, 0, sizeof(int), st));
    }
    // cell index of the cloud for the weighted sub-sampler: once per shape
    const CloudIndex* cidx = cloud_index_usable(N, S, rc.subsample_mode) ? cloud_index_build(pts, N, st) : nullptr;
    auto assemble = [&](const int32_t* lin, int64_t n, int64_t qbase, const int32_t* qidx) {
        query_points(lin, n, rc.res, b.qpts, st);
        { StageScope t("assemble: knn_patch", st);
          if (fixed_radius) ball_patch(pts, N, b.qpts, n, qbase, P, (double)rc.patch_radius, rc.seed, nullptr, b.patch, b.radius, nullptr, st, qidx);
          else knn_patch(pts, N, b.qpts, n, P, nullptr, b.patch, b.radius, st); }
        // the Philox stream is keyed by the query's rank in the whole ordered list -> independent of slabs/batches
        { StageScope t("assemble: subsample+gather", st);
          subsample(pts, N, b.qpts, n, qbase, S, rc.subsample_mode, rc.seed, b.sub_ids, st, qidx, b.sub, cidx); }
    };
    for (int64_t q0 = 0; q0 < Q; q0 += batch) {
        const int64_t n = (Q - q0 < batch) ? (Q - q0) : batch;
        assemble(lin_idx + q0, n, first_query + q0, nullptr);
        forward_fast(m, b.patch, b.sub, b.qpts, n, b.logits, st);
        if (guard) guard_flag(b.logits, n, m.guard_band, q0, glist, gcount, Q, st);
        sdf_from_logits(b.logits, fixed_radius ? nullptr : b.radius, n, sdf + q0, st);
    }
    if (guard) {
        int ng = 0;
        P2S_CUDA(cudaMemcpyAsync(&ng, gcount, sizeof(int), cudaMemcpyDeviceToHost, st));
        P2S_CUDA(cudaStreamSynchronize(st));
        if (ng > Q) ng = (int)Q;
        m.last_guard_count += ng;
        StageScope tg("net: guard-band split-precision recompute", st);
        for (int64_t g0 = 0; g0 < ng; g0 += batch) {
            const int64_t n = (ng - g0 < batch) ? (ng - g0) : batch;
            gather_rows(lin_idx, glist + g0, n, 1, glin, st);
            assemble(glin, n, first_query, glist + g0);
            forward_tc(m, b.patch, b.sub, b.qpts, n, b.logits, st, true);
            sdf_from_logits(b.logits, fixed_radius ? nullptr : b.radius, n, gsdf, st);
            scatter_rows(gsdf, glist + g0, n, 1, sdf, st);
        }
    }
    int err = assemble_error_check(st);
    P2S_CHECK(err == 0, "degenerate cloud: more than 512 points tie at a selection boundary");
}

}  // namespace p2s

using namespace p2s;

extern "C" {

int p2s_abi_version(void) { return P2S_ABI_VERSION; }
const char* p2s_last_error(void) { return g_last_error.c_str(); }
uint64_t p2s_launch_count(void) { return g_launches.load(); }
void p2s_launch_count_reset(void) { g_launches.store(0); }

size_t p2s_model_blob_floats(const p2s_model_config* cfg) {
    if (!cfg) return 0;
    return blob_floats(*cfg);
}

int p2s_model_create(const p2s_model_config* cfg, const float* blob_host, size_t n_floats, int device, p2s_model** out) {
    return guarded([&] {
        P2S_CHECK(cfg && blob_host && out, "null argument");
        check_cfg(*cfg);
        P2S_CHECK(n_floats == blob_floats(*cfg), "weight blob size does not match the model config");
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0) throw Error("no CUDA device available: libp2s_b200 has no CPU fallback");
        P2S_CHECK(device >= 0 && device < ndev, "bad device index");
        P2S_CUDA(cudaSetDevice(device));
        cudaDeviceProp prop;
        P2S_CUDA(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10) throw Error(std::string("libp2s_b200 is built for sm_100a (B200) only; found ") + prop.name);
        Model* m = new Model();
        m->cfg = *cfg;
        m->device = device;
        m->blob_floats = n_floats;
        P2S_CUDA(cudaMalloc(&m->blob, n_floats * sizeof(float)));
        P2S_CUDA(cudaMemcpy(m->blob, blob_host, n_floats * sizeof(float), cudaMemcpyHostToDevice));
        P2S_CUDA(cudaStreamCreateWithFlags(&m->own_stream, cudaStreamNonBlocking));
        BlobCursor c{m->blob, n_floats};
        const int net = cfg->net_size;
        m->shared_qstn = cfg->use_point_stn && cfg->shared_transformer;
        if (m->shared_qstn) m->point_stn = take_stn(c, 3, 4, net);
        m->local = take_feat(c, false, net);
        m->global = take_feat(c, cfg->use_point_stn && !cfg->shared_transformer, net);
        m->fc1_local = c.take(net / 2, net);
        m->fc1_global = c.take(net / 2, net);
        m->fc2 = c.take(net / 4, net);
        m->fc3 = c.take(net / 8, net / 4);
        m->fc4 = c.take(2, net / 8);
        P2S_CHECK(c.left == 0, "weight blob has trailing data");
        tc_build(*m);
        *out = reinterpret_cast<p2s_model*>(m);
    });
}

void p2s_model_destroy(p2s_model* mm) {
    if (!mm) return;
    Model* m = reinterpret_cast<Model*>(mm);
    cudaSetDevice(m->device);
    StageTimer::report();
    tc_destroy(*m);
    if (m->blob) cudaFree(m->blob);
    m->ws_net.release(); m->ws_io.release(); m->ws_misc.release(); m->ws_guard.release(); m->ws_host.release();
    if (m->own_stream) cudaStreamDestroy(m->own_stream);
    delete m;
}

int p2s_model_set_precision(p2s_model* mm, int precision, float guard_band) {
    return guarded([&] {
        P2S_CHECK(mm, "null model");
        P2S_CHECK(precision == P2S_PRECISION_FP32 || precision == P2S_PRECISION_TC, "unknown precision");
        Model* m = reinterpret_cast<Model*>(mm);
        m->precision = precision;
        m->guard_band = guard_band;
        m->last_guard_count = 0;
    });
}

int p2s_model_last_guard_count(p2s_model* mm, int64_t* count) {
    return guarded([&] {
        P2S_CHECK(mm && count, "null argument");
        Model* m = reinterpret_cast<Model*>(mm);
        P2S_CUDA(cudaSetDevice(m->device));
        *count = m->last_guard_count;
        m->last_guard_count = 0;
    });
}

int p2s_model_set_debug_aux(p2s_model* mm, float* aux) {
    return guarded([&] {
        P2S_CHECK(mm, "null model");
        reinterpret_cast<Model*>(mm)->debug_aux = aux;
    });
}

int p2s_profile_enable(p2s_model* mm, int on) {
    return guarded([&] {
        P2S_CHECK(mm, "null model");
        Model* m = reinterpret_cast<Model*>(mm);
        P2S_CUDA(cudaSetDevice(m->device));
        tc_profile_reset(*m, on != 0);
    });
}

int p2s_profile_get(p2s_model* mm, double* ms, int64_t* launches, double* flops) {
    return guarded([&] {
        P2S_CHECK(mm && ms && launches && flops, "null argument");
        Model* m = reinterpret_cast<Model*>(mm);
        P2S_CUDA(cudaSetDevice(m->device));
        tc_profile_get(*m, ms, launches, flops);
    });
}

int p2s_forward_dev(p2s_model* mm, const float* patch, const float* sub, const float* query, int64_t B, float* logits, void* stream) {
    return guarded([&] {
        P2S_CHECK(mm && patch && sub && query && logits, "null argument");
        Model* m = reinterpret_cast<Model*>(mm);
        P2S_CUDA(cudaSetDevice(m->device));
        forward(*m, patch, sub, query, B, logits, as_stream(stream));
    });
}

int p2s_forward_host(p2s_model* mm, const float* patch, const float* sub, const float* query, int64_t B, float* logits) {
    return guarded([&] {
        P2S_CHECK(mm && patch && sub && query && logits, "null argument");
        Model* m = reinterpret_cast<Model*>(mm);
        P2S_CUDA(cudaSetDevice(m->device));
        if (B <= 0) return;
        const size_t P = m->cfg.points_per_patch, S = m->cfg.sub_sample_size;
        cudaStream_t st = m->own_stream;
        float* d = m->ws_host.as<float>((size_t)B * (P * 3 + S * 3 + 3 + 2) + 16);
        float* d_patch = d;
        float* d_sub = d_patch + (size_t)B * P * 3;
        float* d_q = d_sub + (size_t)B * S * 3;
        float* d_out = d_q + ((size_t)B * 3 + 3) / 4 * 4;
        P2S_CUDA(cudaMemcpyAsync(d_patch, patch, (size_t)B * P * 3 * 4, cudaMemcpyHostToDevice, st));
        P2S_CUDA(cudaMemcpyAsync(d_sub, sub, (size_t)B * S * 3 * 4, cudaMemcpyHostToDevice, st));
        P2S_CUDA(cudaMemcpyAsync(d_q, query, (size_t)B * 3 * 4, cudaMemcpyHostToDevice, st));
        forward(*m, d_patch, d_sub, d_q, B, d_out, st);
        P2S_CUDA(cudaMemcpyAsync(logits, d_out, (size_t)B * 2 * 4, cudaMemcpyDeviceToHost, st));
        P2S_CUDA(cudaStreamSynchronize(st));
    });
}

int p2s_sdf_from_logits_dev(const float* logits, const float* radius, int64_t B, float* sdf, void* stream) {
    return guarded([&] {
        P2S_CHECK(logits && sdf, "null argument");
        sdf_from_logits(logits, radius, B, sdf, as_stream(stream));
    });
}

int p2s_query_grid_dev(const float* pts, int64_t N, int res, int eps, int32_t* lin_idx, int64_t cap, int64_t* count_host, void* stream) {
    return guarded([&] {
        P2S_CHECK(pts && count_host && (lin_idx || cap == 0), "null argument");
        query_grid(pts, N, res, eps, lin_idx, cap, count_host, as_stream(stream));
    });
}

int p2s_query_points_dev(const int32_t* lin_idx, int64_t Q, int res, float* out, void* stream) {
    return guarded([&] {
        P2S_CHECK(lin_idx && out, "null argument");
        query_points(lin_idx, Q, res, out, as_stream(stream));
    });
}

int p2s_knn_patch_dev(const float* pts, int64_t N, const float* queries, int64_t Q, int k, int32_t* ids, float* patch, float* radius, void* stream) {
    return guarded([&] {
        P2S_CHECK(pts && queries && patch && radius, "null argument");
        knn_patch(pts, N, queries, Q, k, ids, patch, radius, as_stream(stream));
        int err = assemble_error_check(as_stream(stream));
        P2S_CHECK(err == 0, "degenerate cloud: more than 512 points tie at the k-th neighbour distance");
    });
}

int p2s_ball_patch_dev(const float* pts, int64_t N, const float* queries, int64_t Q, int64_t qbase, int k, double patch_radius,
                       uint64_t seed, int32_t* ids, float* patch, float* radius, int32_t* counts, void* stream) {
    return guarded([&] {
        P2S_CHECK(pts && queries && patch && radius, "null argument");
        ball_patch(pts, N, queries, Q, qbase, k, patch_radius, seed, ids, patch, radius, counts, as_stream(stream));
        int err = assemble_error_check(as_stream(stream));
        P2S_CHECK(err == 0, "degenerate cloud: too many equal random keys at the ball-query selection boundary");
    });
}

int p2s_subsample_dev(const float* pts, int64_t N, const float* queries, int64_t Q, int64_t qbase, int S, int mode, uint64_t seed, int32_t* sub_ids, void* stream) {
    return guarded([&] {
        P2S_CHECK(pts && queries && sub_ids, "null argument");
        subsample(pts, N, queries, Q, qbase, S, mode, seed, sub_ids, as_stream(stream));
        int err = assemble_error_check(as_stream(stream));
        P2S_CHECK(err == 0, "sub-sample selection failed (degenerate key ties)");
    });
}

int p2s_gather_points_dev(const float* pts, const int32_t* ids, int64_t count, float* out, void* stream) {
    return guarded([&] {
        P2S_CHECK(pts && ids && out, "null argument");
        gather_points(pts, ids, count, out, as_stream(stream));
    });
}

int p2s_reconstruct_dev(p2s_model* mm, const p2s_recon_config* rc, const float* pts, int64_t N, int64_t first_query,
                        int64_t num_queries, int32_t* lin_idx, float* sdf, int64_t cap, int64_t* Q_host, void* stream) {
    return guarded([&] {
        P2S_CHECK(mm && rc && pts && lin_idx && sdf && Q_host, "null argument");
        Model* m = reinterpret_cast<Model*>(mm);
        P2S_CUDA(cudaSetDevice(m->device));
        reconstruct(*m, *rc, pts, N, first_query, num_queries, lin_idx, sdf, cap, Q_host, as_stream(stream));
    });
}

int p2s_reconstruct_host(p2s_model* mm, const p2s_recon_config* rc, const float* pts_host, int64_t N,
                         int32_t* lin_idx_host, float* sdf_host, int64_t cap, int64_t* Q_host) {
    return guarded([&] {
        P2S_CHECK(mm && rc && pts_host && lin_idx_host && sdf_host && Q_host, "null argument");
        Model* m = reinterpret_cast<Model*>(mm);
        P2S_CUDA(cudaSetDevice(m->device));
        cudaStream_t st = m->own_stream;
        float* d_pts = m->ws_host.as<float>((size_t)N * 3 + (size_t)cap * 2 + 64);
        int32_t* d_idx = reinterpret_cast<int32_t*>(d_pts + ((size_t)N * 3 + 3) / 4 * 4);
        float* d_sdf = reinterpret_cast<float*>(d_idx + cap);
        P2S_CUDA(cudaMemcpyAsync(d_pts, pts_host, (size_t)N * 12, cudaMemcpyHostToDevice, st));
        reconstruct(*m, *rc, d_pts, N, 0, -1, d_idx, d_sdf, cap, Q_host, st);
        P2S_CUDA(cudaMemcpyAsync(lin_idx_host, d_idx, (size_t)(*Q_host) * 4, cudaMemcpyDeviceToHost, st));
        P2S_CUDA(cudaMemcpyAsync(sdf_host, d_sdf, (size_t)(*Q_host) * 4, cudaMemcpyDeviceToHost, st));
        P2S_CUDA(cudaStreamSynchronize(st));
    });
}

int p2s_sdf_to_volume_dev(const int32_t* lin_idx, const float* sdf, int64_t Q, int res, int sigma, float thr,
                          float* vol, int* iterations_host, void* stream) {
    return guarded([&] {
        P2S_CHECK(lin_idx && sdf && vol, "null argument");
        sdf_to_volume(lin_idx, sdf, Q, res, sigma, thr, vol, iterations_host, as_stream(stream));
    });
}

int p2s_marching_cubes_dev(const float* vol, int res, float level, float* verts, int64_t vcap, int32_t* faces,
                           int64_t fcap, int64_t* nverts_host, int64_t* nfaces_host, void* stream) {
    return guarded([&] {
        P2S_CHECK(vol && nverts_host && nfaces_host, "null argument");
        marching_cubes(vol, res, level, verts, vcap, faces, fcap, nverts_host, nfaces_host, as_stream(stream));
    });
}

int p2s_mesh_sample_dev(const float* verts, int64_t V, const int32_t* faces, int64_t F, int64_t n, uint64_t seed,
                        float* samples, int32_t* face_ids, void* stream) {
    return guarded([&] {
        P2S_CHECK(verts && faces && (samples || n == 0), "null argument");
        mesh_sample(verts, V, faces, F, n, seed, samples, face_ids, as_stream(stream));
    });
}

int p2s_nn_distance_dev(const float* a, int64_t na, const float* b, int64_t nb, float* dist, int32_t* idx,
                        void* stream) {
    return guarded([&] {
        P2S_CHECK((a || na == 0) && b, "null argument");
        nn_distance(a, na, b, nb, dist, idx, as_stream(stream));
    });
}

int p2s_chamfer_hausdorff_dev(const float* a, int64_t na, const float* b, int64_t nb, double* out4_host, void* stream) {
    return guarded([&] {
        P2S_CHECK(a && b && out4_host, "null argument");
        chamfer_hausdorff(a, na, b, nb, out4_host, as_stream(stream));
    });
}

// ---- training-step primitives (train_ops.cu)
#define P2S_OP(name, params, ...)                                   \
    int name params { return guarded([&] { __VA_ARGS__; }); }

P2S_OP(p2s_op_gemm_nt, (const float* A, int64_t a_stride_z, int lda, const float* W, int64_t w_stride_z, const float* bias,
                        float* C, int64_t c_stride_z, int ldc, int M, int N, int K, int batch, int relu, void* stream),
       P2S_CHECK(A && W && C, "null argument");
       // large unbatched shapes run on the tensor cores in split precision (fp32-level accuracy), the rest on fp32 FMA
       if (batch == 1 && gemm_nt_tc_ok(A, lda, C, ldc, M, N, K))
           launch_gemm_nt_tc(A, lda, W, bias, C, ldc, M, N, K, relu != 0, as_stream(stream));
       else
           launch_gemm_nt(A, a_stride_z, lda, W, w_stride_z, bias, C, c_stride_z, ldc, M, N, K, batch, relu != 0, as_stream(stream)))
P2S_OP(p2s_op_gemm_tn, (const float* A, int64_t a_stride_z, int lda, const float* B, int64_t b_stride_z, int ldb, float* C,
                        int64_t c_stride_z, int ldc, int M, int N, int K, int batch, int accumulate, void* stream),
       P2S_CHECK(A && B && C, "null argument");
        op_gemm_tn(A, a_stride_z, lda, B, b_stride_z, ldb, C, c_stride_z, ldc, M, N, K, batch, accumulate != 0, as_stream(stream)))
P2S_OP(p2s_op_transpose, (const float* in, float* out, int rows, int cols, int batch, void* stream),
       P2S_CHECK(in && out, "null argument"); op_transpose(in, out, rows, cols, batch, as_stream(stream)))
P2S_OP(p2s_op_col_stats, (const float* x, int64_t M, int C, double* s1, double* s2, void* stream),
       P2S_CHECK(x && s1 && s2, "null argument"); op_col_stats(x, M, C, s1, s2, as_stream(stream)))
P2S_OP(p2s_op_col_sum, (const float* x, int64_t M, int C, double* s1, void* stream),
       P2S_CHECK(x && s1, "null argument"); op_col_sum(x, M, C, s1, as_stream(stream)))
P2S_OP(p2s_op_bn_finalize, (const double* s1, const double* s2, int64_t M, int C, float eps, float momentum, float* mean,
                            float* invstd, float* running_mean, float* running_var, void* stream),
       P2S_CHECK(s1 && s2 && mean && invstd && M > 0, "bad argument");
        op_bn_finalize(s1, s2, M, C, eps, momentum, mean, invstd, running_mean, running_var, as_stream(stream)))
P2S_OP(p2s_op_bn_apply, (const float* z, int64_t M, int C, const float* mean, const float* invstd, const float* gamma,
                         const float* beta, int relu, float* y, void* stream),
       P2S_CHECK(z && mean && invstd && gamma && beta && y, "null argument");
        op_bn_apply(z, M, C, mean, invstd, gamma, beta, relu != 0, y, as_stream(stream)))
P2S_OP(p2s_op_bn_backward, (const float* dy, const float* z, const float* y, int64_t M, int C, const float* mean,
                            const float* invstd, const float* gamma, double* s1, double* s2, float* dz, void* stream),
       P2S_CHECK(dy && z && mean && invstd && gamma && s1 && s2 && dz, "null argument");
        op_bn_backward(dy, z, y, M, C, mean, invstd, gamma, s1, s2, dz, as_stream(stream)))
P2S_OP(p2s_op_bn_maxpool_fwd, (const float* z, int64_t B, int npts, int C, const float* mean, const float* invstd,
                               const float* gamma, const float* beta, int relu, float* out, int32_t* arg, void* stream),
       P2S_CHECK(z && mean && invstd && gamma && beta && out && arg && npts > 0, "bad argument");
        op_bn_maxpool_fwd(z, B, npts, C, mean, invstd, gamma, beta, relu != 0, out, arg, as_stream(stream)))
P2S_OP(p2s_op_bn_maxpool_bwd, (const float* dout, const int32_t* arg, const float* out, const float* z, int64_t B, int npts, int C,
                               const float* mean, const float* invstd, const float* gamma, int relu, double* s1, double* s2,
                               float* dz, void* stream),
       P2S_CHECK(dout && arg && out && z && mean && invstd && gamma && s1 && s2 && dz && npts > 0, "bad argument");
        op_bn_maxpool_bwd(dout, arg, out, z, B, npts, C, mean, invstd, gamma, relu != 0, s1, s2, dz, as_stream(stream)))
P2S_OP(p2s_op_maxpool_fwd, (const float* y, int64_t B, int npts, int C, float* out, int32_t* arg, void* stream),
       P2S_CHECK(y && out && arg && npts > 0, "bad argument"); op_maxpool_fwd(y, B, npts, C, out, arg, as_stream(stream)))
P2S_OP(p2s_op_maxpool_bwd, (const float* dout, const int32_t* arg, int64_t B, int npts, int C, float* dy, void* stream),
       P2S_CHECK(dout && arg && dy, "null argument"); op_maxpool_bwd(dout, arg, B, npts, C, dy, as_stream(stream)))
P2S_OP(p2s_op_loss, (const float* pred, const float* target_mag, const float* radius, const float* target_sign, int64_t B,
                     float w_mag, float w_sign, int fixed_radius, double* loss_out, float* dpred, void* stream),
       P2S_CHECK(pred && target_mag && target_sign && loss_out && (radius || fixed_radius) && B > 0, "bad argument");
        op_loss(pred, target_mag, radius, target_sign, B, w_mag, w_sign, fixed_radius != 0, loss_out, dpred, as_stream(stream)))
P2S_OP(p2s_op_quat_to_rot, (const float* q4, float* R, int64_t B, void* stream),
       P2S_CHECK(q4 && R, "null argument"); launch_quat_to_rot(q4, R, B, as_stream(stream)))
P2S_OP(p2s_op_quat_to_rot_bwd, (const float* q4, const float* dR, int64_t B, float* dq, void* stream),
       P2S_CHECK(q4 && dR && dq, "null argument"); op_quat_to_rot_bwd(q4, dR, B, dq, as_stream(stream)))
P2S_OP(p2s_op_add_row, (float* x, const float* v, int64_t B, int C, void* stream),
       P2S_CHECK(x && v, "null argument"); op_add_row(x, v, B, C, as_stream(stream)))
P2S_OP(p2s_op_center, (const float* in, const float* q, int64_t B, int npts, float* out, void* stream),
       P2S_CHECK(in && q && out, "null argument"); op_center(in, q, B, npts, out, as_stream(stream)))
P2S_OP(p2s_op_axpy, (float* y, const float* x, float a, int64_t n, void* stream),
       P2S_CHECK(y && x, "null argument"); op_axpy(y, x, a, n, as_stream(stream)))
P2S_OP(p2s_op_sgd, (float* param, const float* grad, float* momentum_buf, int64_t n, float lr, float momentum, int first_step,
                    void* stream),
       P2S_CHECK(param && grad && momentum_buf, "null argument");
        op_sgd(param, grad, momentum_buf, n, lr, momentum, first_step != 0, as_stream(stream)))
#undef P2S_OP

}  // extern "C"
