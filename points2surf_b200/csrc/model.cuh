// Device-resident model: folded fp32 weights (accuracy path) + packed fp16 operand tiles (tensor-core path).
#pragma once
#include "common.cuh"

namespace p2s {

struct Layer {
    const float* W = nullptr;  // [cout][cin] row-major, BN folded
    const float* b = nullptr;  // [cout]
    int cout = 0, cin = 0;
};

struct Stn {  // QSTN (out 4) or STN dim 64 (out 4096): source/points_to_surf_model.py:12-131
    Layer c1, c2, c3, fc1, fc2, fc3;
};

struct Feat {  // PointNetfeat: source/points_to_surf_model.py:134-234
    bool has_qstn = false;
    Stn stn1, stn2;
    Layer conv0a, conv0b, conv1, conv2, conv3;
};

struct TcWeights;  // net_tc.cu

struct Model {
    p2s_model_config cfg{};
    int device = 0;
    float* blob = nullptr;  // device copy of the folded fp32 blob
    size_t blob_floats = 0;
    bool shared_qstn = false;
    Stn point_stn;
    Feat local, global;
    Layer fc1_local, fc1_global, fc2, fc3, fc4;

    int precision = P2S_PRECISION_FP32;
    float guard_band = 0.f;
    TcWeights* tc = nullptr;

    cudaStream_t own_stream = nullptr;  // used by the *_host entry points
    DevBuf ws_net;                       // network activations
    DevBuf ws_io;                        // staged host inputs / assembled query batches
    DevBuf ws_misc;                      // candidate list of the fused pipeline / gathered guard-band rows
    DevBuf ws_guard;                     // guard-band index lists
    DevBuf ws_host;                      // device staging of host-call inputs/outputs
    int64_t last_guard_count = 0;
    float* debug_aux = nullptr;          // optional [B][kAuxStride]: R(9), feat_local_max(1024), feat_global_max(1024)
};
constexpr int kAuxStride = 2064;
void debug_aux_copy(Model& m, int64_t b0, int64_t Bc, const float* R, const float* fl, const float* fg, cudaStream_t st);

// net_fp32.cu
void forward_fp32(Model& m, const float* patch, const float* sub, const float* query, int64_t B,
                  float* logits, cudaStream_t st);
// net_tc.cu
void tc_build(Model& m);
void tc_destroy(Model& m);
void tc_profile_reset(Model& m, bool on);
void tc_profile_get(Model& m, double* ms, int64_t* launches, double* flops);
// precise: split-precision operands (the guard-band recompute); fp16 operands otherwise
void forward_tc(Model& m, const float* patch, const float* sub, const float* query, int64_t B,
                float* logits, cudaStream_t st, bool precise);
void guard_flag(const float* logits, int64_t B, float band, int64_t base, int32_t* list, int* count, int64_t cap, cudaStream_t st);
// fc_tc.cu
bool fc_tc_supported(int N, int K);
uint8_t* fc_tc_pack(const Layer& L, std::vector<void*>& allocs);
void launch_fc_tc(const float* A, int lda, const uint8_t* Wimg, const float* bias, float* C, int ldc,
                  int64_t M, int N, int K, bool relu, cudaStream_t st);
uint8_t* fc_tc_pack_raw(const float* W, int N, int K, std::vector<void*>& allocs);
void launch_pack_a(const float* A, int lda, int64_t M, int K, const float* in_bias, bool in_relu, uint8_t* img, cudaStream_t st);
void launch_fc_tc_img(const uint8_t* Aimg, const uint8_t* Wimg, const float* bias, void* C, int ldc, int64_t M, int N, int K,
                      bool relu, cudaStream_t st, int out_mode, int out_kt_total = 0, int out_kt_off = 0);
bool gemm_nt_tc_ok(const float* A, int lda, const float* C, int ldc, int64_t M, int N, int K);
void launch_gemm_nt_tc(const float* A, int lda, const float* W, const float* bias, float* C, int ldc, int64_t M, int N,
                       int K, bool relu, cudaStream_t st);
// meshdist.cu
void mesh_sample(const float* verts, int64_t V, const int32_t* faces, int64_t F, int64_t n, uint64_t seed,
                 float* samples, int32_t* face_ids, cudaStream_t st);
void nn_distance(const float* a, int64_t na, const float* b, int64_t nb, float* dist, int32_t* idx, cudaStream_t st);
void chamfer_hausdorff(const float* a, int64_t na, const float* b, int64_t nb, double* out4_host, cudaStream_t st);
// gemm_tn_tc.cu
bool gemm_tn_tc_ok(const float* A, int lda, const float* B, int ldb, int64_t M, int N, int K);
void launch_gemm_tn_tc(const float* A, int lda, const float* B, int ldb, float* C, int ldc, int64_t M, int N, int K,
                       cudaStream_t st);
// train_ops.cu
void op_gemm_tn(const float* A, int64_t a_stride_z, int lda, const float* B, int64_t b_stride_z, int ldb, float* C,
                int64_t c_stride_z, int ldc, int M, int N, int K, int batch, bool accumulate, cudaStream_t st);
void op_transpose(const float* in, float* out, int rows, int cols, int batch, cudaStream_t st);
void op_col_stats(const float* x, int64_t M, int C, double* s1, double* s2, cudaStream_t st);
void op_col_sum(const float* x, int64_t M, int C, double* s1, cudaStream_t st);
void op_bn_finalize(const double* s1, const double* s2, int64_t M, int C, float eps, float momentum, float* mean,
                    float* invstd, float* running_mean, float* running_var, cudaStream_t st);
void op_bn_apply(const float* z, int64_t M, int C, const float* mean, const float* invstd, const float* gamma,
                 const float* beta, bool relu, float* y, cudaStream_t st);
void op_bn_backward(const float* dy, const float* z, const float* y_or_null, int64_t M, int C, const float* mean,
                    const float* invstd, const float* gamma, double* s1, double* s2, float* dz, cudaStream_t st);
void op_bn_maxpool_fwd(const float* z, int64_t B, int npts, int C, const float* mean, const float* invstd,
                       const float* gamma, const float* beta, bool relu, float* out, int32_t* arg, cudaStream_t st);
void op_bn_maxpool_bwd(const float* dout, const int32_t* arg, const float* out, const float* z, int64_t B, int npts, int C,
                       const float* mean, const float* invstd, const float* gamma, bool relu, double* s1, double* s2,
                       float* dz, cudaStream_t st);
void op_maxpool_fwd(const float* y, int64_t B, int npts, int C, float* out, int32_t* arg, cudaStream_t st);
void op_maxpool_bwd(const float* dout, const int32_t* arg, int64_t B, int npts, int C, float* dy, cudaStream_t st);
void op_loss(const float* pred, const float* target_mag, const float* radius, const float* target_sign, int64_t B,
             float w_mag, float w_sign, bool fixed_radius, double* loss_out, float* dpred, cudaStream_t st);
void op_quat_to_rot_bwd(const float* q4, const float* dR, int64_t B, float* dq, cudaStream_t st);
void op_add_row(float* x, const float* v, int64_t B, int C, cudaStream_t st);
void op_sgd(float* p, const float* g, float* buf, int64_t n, float lr, float momentum, bool first, cudaStream_t st);
void op_axpy(float* y, const float* x, float a, int64_t n, cudaStream_t st);
void op_center(const float* in, const float* q, int64_t B, int npts, float* out, cudaStream_t st);

// small shared kernels (net_fp32.cu), also used by the TC path for the per-query FC tails
void launch_gemm_nt(const float* A, int64_t a_stride_z, int lda, const float* W, int64_t w_stride_z,
                    const float* bias, float* C, int64_t c_stride_z, int ldc, int M, int N, int K,
                    int batch, bool relu, cudaStream_t st);
void launch_gemm_nt_colmax(const float* A, int64_t a_stride_z, int lda, const float* W, float* out,
                           int M, int N, int K, int batch, cudaStream_t st);
void launch_fill(float* p, int64_t n, float v, cudaStream_t st);
void launch_bias_act(float* x, const float* bias, int64_t rows, int cols, bool relu, cudaStream_t st);
void launch_quat_to_rot(const float* q4, float* R, int64_t B, cudaStream_t st);
void launch_add_identity64(float* T, int64_t B, cudaStream_t st);

}  // namespace p2s
