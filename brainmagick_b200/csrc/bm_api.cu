// C-ABI entry points of libbm_b200.so (see include/bm_b200.h for the contract and the reference citations).
#include <algorithm>
#include "../../include/bm_b200.h"
#include "common.cuh"
#include "elementwise.cuh"
#include "gemm_simt.cuh"
#include "tc_conv.cuh"
#include "tc_wgrad.cuh"
#include "tc_clip.cuh"
#include "tc_convp.cuh"
#include "tc_convh.cuh"
#include "tc_wgradh.cuh"
#include "tc_wgradp.cuh"
#include "tc_gemm_nt.cuh"
#include "retrieval.cuh"
#include "prep.cuh"
#include "convseq.cuh"
#include "regression.cuh"

namespace bm {
thread_local char g_last_error[512] = "";
unsigned long long g_launches = 0;
int g_debug_flags = 0;
long long* g_debug_buf = nullptr;
}
using namespace bm;

#define ST(s) reinterpret_cast<cudaStream_t>(s)

extern "C" const char* bm_last_error(void) { return bm::g_last_error; }
extern "C" int bm_abi_version(void) { return 1; }
extern "C" unsigned long long bm_launch_count(void) { return bm::g_launches; }
extern "C" int bm_set_debug_buffer(long long* buf) { bm::g_debug_buf = buf; return 0; }
extern "C" int bm_set_debug_flags(int flags) { int old = bm::g_debug_flags; bm::g_debug_flags = flags; return old; }

namespace {

// number of z-chunks so that a reduction GEMM with `tiles` output tiles fills the machine ~2x
inline int pick_chunks(int Z, int tiles) {
    int want = (2 * num_sms() + tiles - 1) / tiles;
    if (want < 1) want = 1;
    if (want > Z) want = Z;
    return want;
}
inline int tiles_of(int M, int N) { return ((M + GBM - 1) / GBM) * ((N + GBN - 1) / GBN); }

}  // namespace

// =================================================================================================
// K1
// =================================================================================================
extern "C" int bm_attention_weights_fwd(const float* positions, const float* freq, const float* heads,
                                        const float* ban_centre, float radius, int R, int C, int O, int P,
                                        float* emb, float* weights, bm_stream_t stream) {
    BM_CHECK_ARG(positions && freq && heads && emb && weights);
    BM_CHECK_ARG(R > 0 && C > 0 && O > 0 && P > 0 && P % 2 == 0);
    int n = 0;
    while ((n + 1) * (n + 1) * 2 <= P) ++n;
    BM_CHECK_ARG(n * n * 2 == P);
    cudaStream_t st = ST(stream);
    fourier_emb_kernel<<<ew_grid((long long)R * C * n * n), 256, 0, st>>>(positions, freq, 0.2f, R * C, n, emb);
    BM_CHECK_LAUNCH();
    // scores[r][o][c] = <emb[r][c][:], heads[o][:]>
    GemmP g = gemm_defaults();
    g.M = C; g.N = O; g.K = P;
    g.Z = R; g.nseg = R; g.zchunk = 1; g.kchunk = P;
    g.A = emb; g.lda_z = (long long)C * P; g.lda_m = P; g.lda_k = 1; g.a_mcontig = 0;
    g.B = heads; g.ldb_z = 0; g.ldb_n = P; g.ldb_k = 1; g.b_ncontig = 0;
    g.D = weights; g.ldd_z = (long long)O * C; g.ldd_m = 1; g.ldd_n = C;
    BM_CUDA(launch_gemm(g, st));
    int rows = R * O;
    masked_softmax_kernel<<<(rows + 7) / 8, 256, 0, st>>>(weights, positions, ban_centre, radius, -0.1f, R, O, C);
    BM_CHECK_LAUNCH();
    return 0;
}

extern "C" int bm_attention_weights_bwd(const float* dweights, const float* weights, const float* emb, int R,
                                        int C, int O, int P, float* dscores, float* dheads, bm_stream_t stream) {
    BM_CHECK_ARG(dweights && weights && emb && dscores && dheads);
    cudaStream_t st = ST(stream);
    int rows = R * O;
    softmax_bwd_kernel<<<(rows + 7) / 8, 256, 0, st>>>(weights, dweights, dscores, rows, C);
    BM_CHECK_LAUNCH();
    // dheads[o][p] = sum_{r,c} ds[r][o][c] emb[r][c][p]
    BM_CUDA(cudaMemsetAsync(dheads, 0, sizeof(float) * O * P, st));
    GemmP g = gemm_defaults();
    g.M = O; g.N = P; g.K = C; g.kchunk = C;
    g.Z = R; g.zchunk = 1; g.nseg = R;
    g.A = dscores; g.lda_z = (long long)O * C; g.lda_m = C; g.lda_k = 1; g.a_mcontig = 0;
    g.B = emb; g.ldb_z = (long long)C * P; g.ldb_n = 1; g.ldb_k = P; g.b_ncontig = 1;
    g.D = dheads; g.ldd_z = 0; g.ldd_m = P; g.ldd_n = 1; g.atomic = 1;
    BM_CUDA(launch_gemm(g, st));
    return 0;
}

// =================================================================================================
// K2
// =================================================================================================
// ---- pieces (leading dimensions explicit so that u / v / x0 may be kept channel-padded for the tensor-core layers) ----
extern "C" int bm_sensor_mix_fwd(const float* meg, const float* weights, const int* rec_of_sample, int B, int C, int T,
                                 int O, int ld_u, float* u, bm_stream_t stream) {
    BM_CHECK_ARG(meg && weights && rec_of_sample && u && ld_u >= O);
    // u[b][t][o] = sum_c meg[b][c][t] w[rec_b][o][c]
    GemmP g = gemm_defaults();
    g.M = T; g.N = O; g.K = C; g.kchunk = C;
    g.Z = B; g.nseg = B; g.zchunk = 1;
    g.A = meg; g.lda_z = (long long)C * T; g.lda_m = 1; g.lda_k = T; g.a_mcontig = 1;
    g.B = weights; g.bsel = rec_of_sample; g.ldb_z = (long long)O * C; g.ldb_n = C; g.ldb_k = 1; g.b_ncontig = 0;
    g.D = u; g.ldd_z = (long long)T * ld_u; g.ldd_m = ld_u; g.ldd_n = 1;
    BM_CUDA(launch_gemm(g, ST(stream)));
    return 0;
}

extern "C" int bm_initial_linear_fwd(const float* u, int ld_u, const float* il_w, const float* il_b, int B, int T, int O,
                                     int IL, int ld_v, float* v, bm_stream_t stream) {
    BM_CHECK_ARG(u && il_w && il_b && v && ld_u >= O && ld_v >= IL);
    // v[row][p] = il_b[p] + sum_o u[row][o] il_w[p][o]
    GemmP g = gemm_defaults();
    g.M = B * T; g.N = IL; g.K = O; g.kchunk = O;
    g.A = u; g.lda_m = ld_u; g.lda_k = 1;
    g.B = il_w; g.ldb_n = O; g.ldb_k = 1;
    g.D = v; g.ldd_m = ld_v; g.ldd_n = 1;
    g.bias = il_b;
    BM_CUDA(launch_gemm(g, ST(stream)));
    return 0;
}

extern "C" int bm_subject_layers_fwd(const float* v, int ld_v, const float* subj_w, const int* subject, int B, int T,
                                     int IL, int D, int ld_x0, float* x0, bm_stream_t stream) {
    BM_CHECK_ARG(v && subj_w && subject && x0 && ld_v >= IL && ld_x0 >= D);
    // x0[b][t][d] = sum_p v[b][t][p] M[s_b][p][d]
    GemmP g = gemm_defaults();
    g.M = T; g.N = D; g.K = IL; g.kchunk = IL;
    g.Z = B; g.nseg = B; g.zchunk = 1;
    g.A = v; g.lda_z = (long long)T * ld_v; g.lda_m = ld_v; g.lda_k = 1;
    g.B = subj_w; g.bsel = subject; g.ldb_z = (long long)IL * D; g.ldb_n = 1; g.ldb_k = D; g.b_ncontig = 1;
    g.D = x0; g.ldd_z = (long long)T * ld_x0; g.ldd_m = ld_x0; g.ldd_n = 1;
    BM_CUDA(launch_gemm(g, ST(stream)));
    return 0;
}

extern "C" int bm_sensor_chain_fwd(const float* meg, const float* weights, const int* rec_of_sample,
                                   const float* il_w, const float* il_b, const float* subj_w, const int* subject,
                                   int B, int C, int T, int O, int IL, int D, int ld_x0, float* u, float* v,
                                   float* x0, bm_stream_t stream) {
    BM_CHECK_ARG(meg && weights && rec_of_sample && il_w && il_b && subj_w && subject && u && v && x0);
    BM_CHECK_ARG(ld_x0 >= D);
    int rc = bm_sensor_mix_fwd(meg, weights, rec_of_sample, B, C, T, O, O, u, stream);
    if (!rc) rc = bm_initial_linear_fwd(u, O, il_w, il_b, B, T, O, IL, IL, v, stream);
    if (!rc) rc = bm_subject_layers_fwd(v, IL, subj_w, subject, B, T, IL, D, ld_x0, x0, stream);
    return rc;
}

extern "C" int bm_subject_layers_bwd(const float* dx0, int ld_x0, const float* v, int ld_v, const float* subj_w,
                                     const int* subject, const int* subj_order, const int* subj_off, int B, int T, int IL,
                                     int D, int S, int ld_dv, float* dv, float* d_subj_w, bm_stream_t stream) {
    BM_CHECK_ARG(dx0 && v && subj_w && subject && subj_order && subj_off && dv && d_subj_w);
    BM_CHECK_ARG(ld_x0 >= D && ld_v >= IL && ld_dv >= IL);
    cudaStream_t st = ST(stream);
    {   // dv[b][t][p] = sum_d g[b][t][d] M[s_b][p][d]
        GemmP g = gemm_defaults();
        g.M = T; g.N = IL; g.K = D; g.kchunk = D;
        g.Z = B; g.nseg = B; g.zchunk = 1;
        g.A = dx0; g.lda_z = (long long)T * ld_x0; g.lda_m = ld_x0; g.lda_k = 1;
        g.B = subj_w; g.bsel = subject; g.ldb_z = (long long)IL * D; g.ldb_n = D; g.ldb_k = 1;
        g.D = dv; g.ldd_z = (long long)T * ld_dv; g.ldd_m = ld_dv; g.ldd_n = 1;
        BM_CUDA(launch_gemm(g, st));
    }
    {   // dM[s][p][d] = sum_{b in s} sum_t v[b][t][p] g[b][t][d]
        GemmP g = gemm_defaults();
        g.M = IL; g.N = D; g.K = T; g.kchunk = T;
        g.Z = B; g.nseg = S; g.seg_off = subj_off; g.zlist = subj_order;
        g.A = v; g.lda_z = (long long)T * ld_v; g.lda_m = 1; g.lda_k = ld_v; g.a_mcontig = 1;
        g.B = dx0; g.ldb_z = (long long)T * ld_x0; g.ldb_n = 1; g.ldb_k = ld_x0; g.b_ncontig = 1;
        g.D = d_subj_w; g.ldd_z = (long long)IL * D; g.ldd_m = D; g.ldd_n = 1;
        BM_CUDA(launch_gemm(g, st));
    }
    return 0;
}

extern "C" int bm_initial_linear_bwd(const float* dv, int ld_dv, const float* u, int ld_u, const float* il_w, int B, int T,
                                     int O, int IL, int ld_du, float* du, float* d_il_w, float* d_il_b,
                                     bm_stream_t stream) {
    BM_CHECK_ARG(dv && u && il_w && du && d_il_w && d_il_b && ld_dv >= IL && ld_u >= O && ld_du >= O);
    cudaStream_t st = ST(stream);
    {   // d_il_w[p][o] = sum_{b,t} dv[b][t][p] u[b][t][o]
        BM_CUDA(cudaMemsetAsync(d_il_w, 0, sizeof(float) * IL * O, st));
        GemmP g = gemm_defaults();
        g.M = IL; g.N = O; g.K = T; g.kchunk = T;
        g.Z = B; g.nseg = pick_chunks(B, tiles_of(IL, O)); g.zchunk = (B + g.nseg - 1) / g.nseg;
        g.nseg = (B + g.zchunk - 1) / g.zchunk;
        g.A = dv; g.lda_z = (long long)T * ld_dv; g.lda_m = 1; g.lda_k = ld_dv; g.a_mcontig = 1;
        g.B = u; g.ldb_z = (long long)T * ld_u; g.ldb_n = 1; g.ldb_k = ld_u; g.b_ncontig = 1;
        g.D = d_il_w; g.ldd_z = 0; g.ldd_m = O; g.ldd_n = 1; g.atomic = 1;
        BM_CUDA(launch_gemm(g, st));
    }
    {   // d_il_b[p] = sum dv
        BM_CUDA(cudaMemsetAsync(d_il_b, 0, sizeof(float) * IL, st));
        GemmP g = gemm_defaults();                      // column sums as a 1-row GEMM would waste a tile: dedicated kernel
        (void)g;
        long long rows = (long long)B * T;
        dim3 grid((unsigned)((rows + 255) / 256), (IL + 127) / 128);
        colsum_strided_kernel<<<grid, 128, 0, st>>>(dv, d_il_b, rows, IL, ld_dv, 256);
        BM_CHECK_LAUNCH();
    }
    {   // du[row][o] = sum_p dv[row][p] il_w[p][o]
        GemmP g = gemm_defaults();
        g.M = B * T; g.N = O; g.K = IL; g.kchunk = IL;
        g.A = dv; g.lda_m = ld_dv; g.lda_k = 1;
        g.B = il_w; g.ldb_n = 1; g.ldb_k = O; g.b_ncontig = 1;
        g.D = du; g.ldd_m = ld_du; g.ldd_n = 1;
        BM_CUDA(launch_gemm(g, st));
    }
    return 0;
}

extern "C" int bm_sensor_mix_bwd(const float* du, int ld_du, const float* meg, const int* rec_order, const int* rec_off,
                                 int B, int C, int T, int O, int R, float* d_weights, bm_stream_t stream) {
    BM_CHECK_ARG(du && meg && rec_order && rec_off && d_weights && ld_du >= O);
    // dw[r][o][c] = sum_{b in r} sum_t du[b][t][o] meg[b][c][t]
    GemmP g = gemm_defaults();
    g.M = O; g.N = C; g.K = T; g.kchunk = T;
    g.Z = B; g.nseg = R; g.seg_off = rec_off; g.zlist = rec_order;
    g.A = du; g.lda_z = (long long)T * ld_du; g.lda_m = 1; g.lda_k = ld_du; g.a_mcontig = 1;
    g.B = meg; g.ldb_z = (long long)C * T; g.ldb_n = T; g.ldb_k = 1; g.b_ncontig = 0;
    g.D = d_weights; g.ldd_z = (long long)O * C; g.ldd_m = C; g.ldd_n = 1;
    BM_CUDA(launch_gemm(g, ST(stream)));
    return 0;
}

extern "C" int bm_sensor_chain_bwd(const float* dx0, const float* meg, const float* il_w, const float* subj_w,
                                   const int* subject, const float* u, const float* v, const int* subj_order,
                                   const int* subj_off, const int* rec_order, const int* rec_off, int B, int C,
                                   int T, int O, int IL, int D, int ld_x0, int S, int R, float* dv, float* du,
                                   float* d_subj_w, float* d_il_w, float* d_il_b, float* d_weights,
                                   bm_stream_t stream) {
    BM_CHECK_ARG(dx0 && meg && il_w && subj_w && subject && u && v && subj_order && subj_off && rec_order && rec_off);
    BM_CHECK_ARG(dv && du && d_subj_w && d_il_w && d_il_b && d_weights);
    BM_CHECK_ARG(ld_x0 >= D);
    int rc = bm_subject_layers_bwd(dx0, ld_x0, v, IL, subj_w, subject, subj_order, subj_off, B, T, IL, D, S, IL, dv,
                                   d_subj_w, stream);
    if (!rc) rc = bm_initial_linear_bwd(dv, IL, u, O, il_w, B, T, O, IL, O, du, d_il_w, d_il_b, stream);
    if (!rc) rc = bm_sensor_mix_bwd(du, O, meg, rec_order, rec_off, B, C, T, O, R, d_weights, stream);
    return rc;
}

// =================================================================================================
// K3 / K4
// =================================================================================================
extern "C" int bm_conv_weight_prep(const float* w, int Cout, int Cin, int Kw, float* wf, float* wb,
                                   bm_stream_t stream) {
    BM_CHECK_ARG(w && (wf || wb) && Cout > 0 && Cin > 0 && Kw > 0);
    weight_prep_kernel<<<ew_grid((long long)Cout * Cin * Kw), 256, 0, ST(stream)>>>(w, wf, wb, Cout, Cin, Kw);
    BM_CHECK_LAUNCH();
    return 0;
}

static int conv_gemm(const float* x, const float* wmat, const float* bias, const float* addend, int B, int T,
                     int K, int N, int Kw, int dilation, int sign, float* y, double* stats, int glu, float* glu_out,
                     cudaStream_t st) {
    BM_CHECK_ARG(Kw >= 1 && Kw <= 3 && (Kw % 2) == 1);
    GemmP g = gemm_defaults();
    g.M = T; g.N = N; g.K = K; g.kchunk = K; g.taps = Kw;
    g.Z = B; g.nseg = B; g.zchunk = 1;
    g.A = x; g.lda_z = (long long)T * K; g.lda_m = K; g.lda_k = 1;
    for (int j = 0; j < Kw; ++j) g.a_shift_m[j] = sign * (j - Kw / 2) * dilation;
    g.B = wmat; g.ldb_z = 0; g.ldb_tap = (long long)K * N; g.ldb_k = N; g.ldb_n = 1; g.b_ncontig = 1;
    g.D = y; g.ldd_z = (long long)T * N; g.ldd_m = N; g.ldd_n = 1;
    g.bias = bias; g.addend = addend; g.stats = stats;
    if (glu) {
        g.glu = 1; g.glu_out = glu_out;
        g.ldg_z = (long long)T * (N / 2); g.ldg_m = N / 2; g.ldg_n = 1;
    }
    BM_CUDA(launch_gemm(g, st));
    return 0;
}

extern "C" int bm_conv1d_fwd(const float* x, const float* wf, const float* bias, int B, int T, int Cin, int Cout,
                             int Kw, int dilation, float* y, double* stats, bm_stream_t stream) {
    BM_CHECK_ARG(x && wf && y && B > 0 && T > 0 && Cin > 0 && Cout > 0 && dilation >= 1);
    cudaStream_t st = ST(stream);
    if (stats) BM_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * 2 * Cout, st));
    return conv_gemm(x, wf, bias, nullptr, B, T, Cin, Cout, Kw, dilation, +1, y, stats, 0, nullptr, st);
}

extern "C" int bm_bn_stats_finalize(const double* stats, long long n, float eps, float momentum,
                                    float* running_mean, float* running_var, float* mean, float* invstd, int C,
                                    bm_stream_t stream) {
    BM_CHECK_ARG(stats && mean && invstd && C > 0 && n > 0);
    BM_CHECK_ARG((running_mean == nullptr) == (running_var == nullptr));
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, ST(stream)>>>(stats, (double)n, eps, momentum, running_mean,
                                                               running_var, mean, invstd, C);
    BM_CHECK_LAUNCH();
    return 0;
}

extern "C" int bm_bn_eval_stats(const float* running_mean, const float* running_var, float eps, float* mean,
                                float* invstd, int C, bm_stream_t stream) {
    BM_CHECK_ARG(running_mean && running_var && mean && invstd && C > 0);
    bn_eval_stats_kernel<<<(C + 127) / 128, 128, 0, ST(stream)>>>(running_mean, running_var, eps, mean, invstd, C);
    BM_CHECK_LAUNCH();
    return 0;
}

// amax_out (nullable, every producer below): a device float that receives max |output| -- the scale source of the F16-pipe
// conv that consumes the tensor next (bm_tc_conv1d_f16's x_amax), folded into the producing kernel instead of a bm_amax pass
static int amax_begin(float* amax_out, cudaStream_t st) {
    if (amax_out) BM_CUDA(cudaMemsetAsync(amax_out, 0, sizeof(float), st));
    return 0;
}

extern "C" int bm_bn_gelu_skip_fwd(const float* y, const float* mean, const float* invstd, const float* gamma,
                                   const float* beta, const float* x_old, float* x_new, long long rows, int C,
                                   float* amax_out, bm_stream_t stream) {
    BM_CHECK_ARG(y && mean && invstd && gamma && beta && x_new && rows > 0 && C > 0);
    long long total = rows * C;
    if (int rc = amax_begin(amax_out, ST(stream))) return rc;
    bool vec = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(x_new) |
                                 reinterpret_cast<uintptr_t>(x_old)) % 16 == 0);
    if (vec && C / 4 <= 256 && aligned16(mean, invstd, gamma) && aligned16(beta)) {
        const int cx = C / 4, ry = std::max(1, 320 / cx);
        const unsigned nblk = (unsigned)((rows + CS_ROWS_PER_BLOCK - 1) / CS_ROWS_PER_BLOCK);
        bn_gelu_skip_fwd_cs_kernel<<<nblk, dim3(cx, ry), 0, ST(stream)>>>(y, mean, invstd, gamma, beta, x_old, x_new, rows, C,
                                                                          reinterpret_cast<unsigned int*>(amax_out));
        BM_CHECK_LAUNCH();
        return 0;
    }
    if (vec)
        bn_gelu_skip_fwd_kernel<4><<<ew_grid(total, 256, 4), 256, 0, ST(stream)>>>(y, mean, invstd, gamma, beta,
                                                                                 x_old, x_new, total, C);
    else
        bn_gelu_skip_fwd_kernel<1><<<ew_grid(total), 256, 0, ST(stream)>>>(y, mean, invstd, gamma, beta, x_old,
                                                                          x_new, total, C);
    BM_CHECK_LAUNCH();
    if (amax_out) return tc::launch_amax(x_new, total, amax_out, ST(stream));
    return 0;
}

extern "C" int bm_bn_gelu_skip_bwd(const float* g, const float* y, const float* mean, const float* invstd,
                                   const float* gamma, const float* beta, int batch_stats, long long rows, int C,
                                   double* sums, float* dy, float* dgamma, float* dbeta, float* amax_out,
                                   bm_stream_t stream) {
    BM_CHECK_ARG(g && y && mean && invstd && gamma && beta && sums && dy && dgamma && dbeta && rows > 0 && C > 0);
    cudaStream_t st = ST(stream);
    BM_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * 2 * C, st));
    if (int rc = amax_begin(amax_out, st)) return rc;
    const long long total = rows * C;
    const bool vec = (C % 4 == 0) && aligned16(g, y, dy) && aligned16(mean, invstd, gamma) && aligned16(beta);
    if (vec && C / 4 <= 256 && aligned16(dgamma, dbeta)) {
        const int cx = C / 4, ry = std::max(1, 320 / cx);
        const unsigned nblk = (unsigned)((rows + CS_ROWS_PER_BLOCK - 1) / CS_ROWS_PER_BLOCK);
        bn_gelu_bwd_reduce_cs_kernel<<<nblk, dim3(cx, ry), sizeof(float) * 2 * C * ry, st>>>(g, y, mean, invstd, gamma, beta,
                                                                                          sums, rows, C);
        BM_CHECK_LAUNCH();
        bn_param_grad_kernel<<<(C + 127) / 128, 128, 0, st>>>(sums, dgamma, dbeta, C);
        BM_CHECK_LAUNCH();
        bn_gelu_bwd_apply_cs_kernel<<<nblk, dim3(cx, ry), 0, st>>>(g, y, mean, invstd, gamma, beta, dgamma, dbeta,
                                                                   (float)(1.0 / (double)rows), batch_stats, dy, rows, C,
                                                                   reinterpret_cast<unsigned int*>(amax_out));
        BM_CHECK_LAUNCH();
        return 0;
    }
    {   // generic shapes: one thread per column, 128 rows per block
        const int rpb = 128;
        dim3 grid((unsigned)((rows + rpb - 1) / rpb), (C + 127) / 128);
        bn_gelu_bwd_reduce_kernel<<<grid, 128, 0, st>>>(g, y, mean, invstd, gamma, beta, sums, rows, C, rpb);
    }
    BM_CHECK_LAUNCH();
    bn_param_grad_kernel<<<(C + 127) / 128, 128, 0, st>>>(sums, dgamma, dbeta, C);
    BM_CHECK_LAUNCH();
    if (vec)
        bn_gelu_bwd_apply_v4_kernel<<<ew_grid(total / 4), 256, 0, st>>>(
            reinterpret_cast<const float4*>(g), reinterpret_cast<const float4*>(y), reinterpret_cast<const float4*>(mean),
            reinterpret_cast<const float4*>(invstd), reinterpret_cast<const float4*>(gamma),
            reinterpret_cast<const float4*>(beta), sums, (double)rows, batch_stats, reinterpret_cast<float4*>(dy),
            total / 4, C);
    else
        bn_gelu_bwd_apply_kernel<<<ew_grid(total), 256, 0, st>>>(g, y, mean, invstd, gamma, beta, sums, (double)rows,
                                                               batch_stats, dy, total, C);
    BM_CHECK_LAUNCH();
    if (amax_out) return tc::launch_amax(dy, total, amax_out, st);
    return 0;
}

extern "C" int bm_conv1d_bwd_data(const float* dy, const float* wb, const float* addend, int B, int T, int Cin,
                                  int Cout, int Kw, int dilation, float* dx, bm_stream_t stream) {
    BM_CHECK_ARG(dy && wb && dx && B > 0 && T > 0 && Cin > 0 && Cout > 0 && dilation >= 1);
    return conv_gemm(dy, wb, nullptr, addend, B, T, Cout, Cin, Kw, dilation, -1, dx, nullptr, 0, nullptr,
                     ST(stream));
}

extern "C" int bm_conv1d_bwd_weight(const float* dy, const float* x, int B, int T, int Cin, int Cout, int Kw,
                                    int dilation, float* dw, float* dbias, bm_stream_t stream) {
    BM_CHECK_ARG(dy && x && dw && B > 0 && T > 0 && Cin > 0 && Cout > 0 && Kw >= 1 && Kw <= 3);
    cudaStream_t st = ST(stream);
    BM_CUDA(cudaMemsetAsync(dw, 0, sizeof(float) * (size_t)Cout * Cin * Kw, st));
    int nseg = pick_chunks(B, tiles_of(Cout, Cin) * Kw);
    int zchunk = (B + nseg - 1) / nseg;
    nseg = (B + zchunk - 1) / zchunk;
    for (int j = 0; j < Kw; ++j) {
        GemmP g = gemm_defaults();
        g.M = Cout; g.N = Cin; g.K = T; g.kchunk = T;
        g.Z = B; g.nseg = nseg; g.zchunk = zchunk;
        g.A = dy; g.lda_z = (long long)T * Cout; g.lda_m = 1; g.lda_k = Cout; g.a_mcontig = 1;
        g.B = x; g.ldb_z = (long long)T * Cin; g.ldb_n = 1; g.ldb_k = Cin; g.b_ncontig = 1;
        g.b_shift_k[0] = (j - Kw / 2) * dilation;
        g.D = dw + j; g.ldd_z = 0; g.ldd_m = (long long)Cin * Kw; g.ldd_n = Kw; g.atomic = 1;
        BM_CUDA(launch_gemm(g, st));
    }
    if (dbias) {
        BM_CUDA(cudaMemsetAsync(dbias, 0, sizeof(float) * Cout, st));
        long long rows = (long long)B * T;
        dim3 grid((unsigned)((rows + 255) / 256), (Cout + 127) / 128);
        colsum_cl_kernel<<<grid, 128, 0, st>>>(dy, dbias, rows, Cout, 256);
        BM_CHECK_LAUNCH();
    }
    return 0;
}

extern "C" int bm_conv1d_glu_fwd(const float* x, const float* wf, const float* bias, int B, int T, int Cin, int H,
                                 int Kw, float* h, float* out, bm_stream_t stream) {
    BM_CHECK_ARG(x && wf && out && B > 0 && T > 0 && Cin > 0 && H > 0);
    return conv_gemm(x, wf, bias, nullptr, B, T, Cin, 2 * H, Kw, 1, +1, h, nullptr, 1, out, ST(stream));
}

extern "C" int bm_glu_bwd(const float* g, const float* h, long long rows, int H, float* dh, float* dbias,
                          float* amax_out, bm_stream_t stream) {
    BM_CHECK_ARG(g && h && dh && rows > 0 && H > 0);
    cudaStream_t st = ST(stream);
    if (dbias) BM_CUDA(cudaMemsetAsync(dbias, 0, sizeof(float) * 2 * H, st));
    if (int rc = amax_begin(amax_out, st)) return rc;
    if (H % 4 == 0 && H / 4 <= 256 && aligned16(g, h, dh)) {
        const int cx = H / 4, ry = std::max(1, 320 / cx);
        const unsigned nblk = (unsigned)((rows + CS_ROWS_PER_BLOCK - 1) / CS_ROWS_PER_BLOCK);
        glu_bwd_cs_kernel<<<nblk, dim3(cx, ry), dbias ? sizeof(float) * 2 * H * ry : 0, st>>>(
            g, h, dh, dbias, rows, H, reinterpret_cast<unsigned int*>(amax_out));
        BM_CHECK_LAUNCH();
        return 0;
    }
    if (H % 4 == 0 && aligned16(g, h, dh))
        glu_bwd_v4_kernel<<<ew_grid(rows * H / 4), 256, 0, st>>>(
            reinterpret_cast<const float4*>(g), reinterpret_cast<const float4*>(h), reinterpret_cast<float4*>(dh), rows, H);
    else
        glu_bwd_kernel<<<ew_grid(rows * H), 256, 0, st>>>(g, h, dh, rows, H);
    BM_CHECK_LAUNCH();
    if (dbias) {
        dim3 grid((unsigned)((rows + 255) / 256), (2 * H + 127) / 128);
        colsum_cl_kernel<<<grid, 128, 0, st>>>(dh, dbias, rows, 2 * H, 256);
        BM_CHECK_LAUNCH();
    }
    if (amax_out) return tc::launch_amax(dh, rows * 2 * H, amax_out, st);
    return 0;
}

// =================================================================================================
// K5
// =================================================================================================
extern "C" int bm_head_fwd(const float* x, const float* w0, const float* b0, const float* w2, const float* b2,
                           int B, int T, int H, int F, float* h1, float* q, float* est, bm_stream_t stream) {
    BM_CHECK_ARG(x && w0 && b0 && w2 && b2 && q && est && B > 0 && T > 0 && H > 0 && F > 0);
    cudaStream_t st = ST(stream);
    const int H2 = 2 * H;
    {   // h1 = x w0^T + b0 ; q = GELU(h1)
        GemmP g = gemm_defaults();
        g.M = B * T; g.N = H2; g.K = H; g.kchunk = H;
        g.A = x; g.lda_m = H; g.lda_k = 1;
        g.B = w0; g.ldb_n = H; g.ldb_k = 1;
        g.D = q; g.ldd_m = H2; g.ldd_n = 1;
        g.bias = b0; g.aux = h1; g.act = 1;
        BM_CUDA(launch_gemm(g, st));
    }
    {   // est[b][f][t] = b2[f] + sum_i q[b][t][i] w2[i][f]
        GemmP g = gemm_defaults();
        g.M = T; g.N = F; g.K = H2; g.kchunk = H2;
        g.Z = B; g.nseg = B; g.zchunk = 1;
        g.A = q; g.lda_z = (long long)T * H2; g.lda_m = H2; g.lda_k = 1;
        g.B = w2; g.ldb_n = 1; g.ldb_k = F; g.b_ncontig = 1;
        g.D = est; g.ldd_z = (long long)F * T; g.ldd_m = 1; g.ldd_n = T;
        g.bias = b2;
        BM_CUDA(launch_gemm(g, st));
    }
    return 0;
}

// dW2, db2, dh1 = dq*GELU'(h1) (in place in dq), dW0, db0 -- the parameter-gradient half of the head backward
extern "C" int bm_head_bwd_params(const float* dest, const float* x, const float* h1, const float* q, int B, int T,
                                  int H, int F, float* dq, float* dw0, float* db0, float* dw2, float* db2,
                                  bm_stream_t stream) {
    BM_CHECK_ARG(dest && x && h1 && q && dq && dw0 && db0 && dw2 && db2);
    cudaStream_t st = ST(stream);
    const int H2 = 2 * H;
    const long long rows = (long long)B * T;
    {   // dw2[i][f] = sum_{b,t} q[b][t][i] dest[b][f][t]
        BM_CUDA(cudaMemsetAsync(dw2, 0, sizeof(float) * (size_t)H2 * F, st));
        GemmP g = gemm_defaults();
        g.M = H2; g.N = F; g.K = T; g.kchunk = T;
        g.Z = B; g.nseg = pick_chunks(B, tiles_of(H2, F)); g.zchunk = (B + g.nseg - 1) / g.nseg;
        g.nseg = (B + g.zchunk - 1) / g.zchunk;
        g.A = q; g.lda_z = (long long)T * H2; g.lda_m = 1; g.lda_k = H2; g.a_mcontig = 1;
        g.B = dest; g.ldb_z = (long long)F * T; g.ldb_n = T; g.ldb_k = 1; g.b_ncontig = 0;
        g.D = dw2; g.ldd_m = F; g.ldd_n = 1; g.atomic = 1;
        BM_CUDA(launch_gemm(g, st));
    }
    {   // db2[f] = sum_{b,t} dest[b][f][t]
        BM_CUDA(cudaMemsetAsync(db2, 0, sizeof(float) * F, st));
        long long nrows = (long long)B * F;
        rowsum_cm_kernel<<<(unsigned)((nrows + 7) / 8), 256, 0, st>>>(dest, db2, B, F, T);
        BM_CHECK_LAUNCH();
    }
    gelu_bwd_kernel<<<ew_grid(rows * H2), 256, 0, st>>>(dq, h1, dq, rows * H2);   // dq <- dh1
    BM_CHECK_LAUNCH();
    {   // dw0[n][k] = sum_rows dh1[row][n] x[row][k]
        BM_CUDA(cudaMemsetAsync(dw0, 0, sizeof(float) * (size_t)H2 * H, st));
        GemmP g = gemm_defaults();
        g.M = H2; g.N = H; g.K = T; g.kchunk = T;
        g.Z = B; g.nseg = pick_chunks(B, tiles_of(H2, H)); g.zchunk = (B + g.nseg - 1) / g.nseg;
        g.nseg = (B + g.zchunk - 1) / g.zchunk;
        g.A = dq; g.lda_z = (long long)T * H2; g.lda_m = 1; g.lda_k = H2; g.a_mcontig = 1;
        g.B = x; g.ldb_z = (long long)T * H; g.ldb_n = 1; g.ldb_k = H; g.b_ncontig = 1;
        g.D = dw0; g.ldd_m = H; g.ldd_n = 1; g.atomic = 1;
        BM_CUDA(launch_gemm(g, st));
    }
    {   // db0
        BM_CUDA(cudaMemsetAsync(db0, 0, sizeof(float) * H2, st));
        dim3 grid((unsigned)((rows + 255) / 256), (H2 + 127) / 128);
        colsum_cl_kernel<<<grid, 128, 0, st>>>(dq, db0, rows, H2, 256);
        BM_CHECK_LAUNCH();
    }
    return 0;
}

extern "C" int bm_head_bwd(const float* dest, const float* x, const float* w0, const float* w2, const float* h1,
                           const float* q, int B, int T, int H, int F, float* dq, float* dx, float* dw0,
                           float* db0, float* dw2, float* db2, bm_stream_t stream) {
    BM_CHECK_ARG(dest && x && w0 && w2 && h1 && q && dq && dx && dw0 && db0 && dw2 && db2);
    cudaStream_t st = ST(stream);
    const int H2 = 2 * H;
    const long long rows = (long long)B * T;
    {   // dq[b][t][i] = sum_f dest[b][f][t] w2[i][f]
        GemmP g = gemm_defaults();
        g.M = T; g.N = H2; g.K = F; g.kchunk = F;
        g.Z = B; g.nseg = B; g.zchunk = 1;
        g.A = dest; g.lda_z = (long long)F * T; g.lda_m = 1; g.lda_k = T; g.a_mcontig = 1;
        g.B = w2; g.ldb_n = F; g.ldb_k = 1;
        g.D = dq; g.ldd_z = (long long)T * H2; g.ldd_m = H2; g.ldd_n = 1;
        BM_CUDA(launch_gemm(g, st));
    }
    int rc = bm_head_bwd_params(dest, x, h1, q, B, T, H, F, dq, dw0, db0, dw2, db2, stream);
    if (rc) return rc;
    {   // dx[row][k] = sum_n dh1[row][n] w0[n][k]
        GemmP g = gemm_defaults();
        g.M = (int)rows; g.N = H; g.K = H2; g.kchunk = H2;
        g.A = dq; g.lda_m = H2; g.lda_k = 1;
        g.B = w0; g.ldb_n = 1; g.ldb_k = H; g.b_ncontig = 1;
        g.D = dx; g.ldd_m = H; g.ldd_n = 1;
        BM_CUDA(launch_gemm(g, st));
    }
    return 0;
}

// =================================================================================================
// K6
// =================================================================================================
// Scratch (caller-owned, passed to every call): bm_clip_workspace() floats.  Tensor-core path: split-K partial score
// tiles + fp64 partial sums of squares + the finalize ticket (csrc/tc_clip.cuh); FP32-FMA path: fp64 sums of squares.
extern "C" long long bm_clip_workspace(int Bn, int Bc, long long KT) {
    if (Bn <= 0 || Bc <= 0 || KT <= 0) return 0;
    if (tc::clip_tc_supported(Bn, Bc, KT)) return tc::clip_ws_floats(Bn, Bc, KT);
    return 2ll * Bc + 2;
}

extern "C" int bm_candidate_inv_norms(const float* cand, int Bc, long long KT, double* ss, float* inv_norm,
                                      bm_stream_t stream) {
    BM_CHECK_ARG(cand && ss && inv_norm && Bc > 0 && KT > 0);
    cudaStream_t st = ST(stream);
    BM_CUDA(cudaMemsetAsync(ss, 0, sizeof(double) * Bc, st));
    int splits = (int)((KT + 65535) / 65536);
    if (splits > 32) splits = 32;
    row_sumsq_kernel<<<dim3(Bc, splits), 256, 0, st>>>(cand, ss, KT);
    BM_CHECK_LAUNCH();
    inv_norm_kernel<<<(Bc + 127) / 128, 128, 0, st>>>(ss, inv_norm, Bc);
    BM_CHECK_LAUNCH();
    return 0;
}

namespace {
// scores (+ probs / row_loss / loss) on whichever kernel the shape allows
int clip_forward(const float* est, const float* cand, int Bn, int Bc, long long KT, int norms_given, int target_offset,
                 float* inv_norm, float* scores, float* probs, float* row_loss, float* loss, float* ws,
                 long long ws_floats, int* status, cudaStream_t st) {
    BM_CHECK_ARG(est && cand && inv_norm && scores && ws && Bn > 0 && Bc > 0 && KT > 0);
    BM_CHECK_ARG(KT < (1ll << 31));
    BM_CHECK_ARG(ws_floats >= bm_clip_workspace(Bn, Bc, KT));
    BM_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & 7) == 0);
    if (tc::clip_tc_supported(Bn, Bc, KT))
        return tc::launch_clip_scores(est, cand, Bn, Bc, KT, norms_given, target_offset, inv_norm, scores, probs, row_loss,
                                      loss, ws, status, st);
    // FP32-FMA GEMM (feature sizes not a multiple of 4 floats: no TMA row pitch)
    if (!norms_given) {
        int rc = bm_candidate_inv_norms(cand, Bc, KT, reinterpret_cast<double*>(ws), inv_norm, st);
        if (rc) return rc;
    }
    BM_CUDA(cudaMemsetAsync(scores, 0, sizeof(float) * (size_t)Bn * Bc, st));
    GemmP g = gemm_defaults();
    g.M = Bn; g.N = Bc; g.K = (int)KT;
    int tiles = tiles_of(Bn, Bc);
    int ks = (2 * num_sms() + tiles - 1) / tiles;
    long long kchunk = (KT + ks - 1) / ks;
    kchunk = ((kchunk + GBK - 1) / GBK) * GBK;
    ks = (int)((KT + kchunk - 1) / kchunk);
    g.ksplit = ks; g.kchunk = (int)kchunk;
    g.A = est; g.lda_m = KT; g.lda_k = 1;
    g.B = cand; g.ldb_n = KT; g.ldb_k = 1;
    g.D = scores; g.ldd_m = Bc; g.ldd_n = 1; g.atomic = 1;
    g.colscale = inv_norm;
    BM_CUDA(launch_gemm(g, st));
    if (probs || row_loss) {
        clip_ce_rows_kernel<<<Bn, 256, 0, st>>>(scores, Bn, Bc, target_offset, row_loss, probs);
        BM_CHECK_LAUNCH();
    }
    if (loss) {
        mean_kernel<<<1, 256, 0, st>>>(row_loss, Bn, loss);
        BM_CHECK_LAUNCH();
    }
    return 0;
}
}  // namespace

extern "C" int bm_clip_scores(const float* est, const float* cand, int Bn, int Bc, long long KT, int norms_given,
                              float* inv_norm, float* scores, float* probs, float* workspace,
                              long long workspace_floats, int* status, bm_stream_t stream) {
    return clip_forward(est, cand, Bn, Bc, KT, norms_given, 0, inv_norm, scores, probs, nullptr, nullptr, workspace,
                        workspace_floats, status, ST(stream));
}

extern "C" int bm_clip_loss_fwd(const float* est, const float* cand, int Bn, int Bc, long long KT,
                                int target_offset, float* inv_norm, float* scores, float* probs, float* row_loss,
                                float* loss, float* workspace, long long workspace_floats, int* status,
                                bm_stream_t stream) {
    BM_CHECK_ARG(probs && row_loss && loss);
    BM_CHECK_ARG(target_offset >= 0 && target_offset + Bn <= Bc);
    return clip_forward(est, cand, Bn, Bc, KT, 0, target_offset, inv_norm, scores, probs, row_loss, loss, workspace,
                        workspace_floats, status, ST(stream));
}

extern "C" int bm_clip_loss_bwd(const float* probs, const float* inv_norm, const float* cand, const float* gout,
                                int Bn, int Bc, long long KT, int target_offset, float* G, float* dest,
                                int* status, bm_stream_t stream) {
    BM_CHECK_ARG(probs && inv_norm && cand && gout && G && dest && Bn > 0 && Bc > 0 && KT > 0);
    BM_CHECK_ARG(KT < (1ll << 31));
    cudaStream_t st = ST(stream);
    if (tc::gemm_nt_pp_supported(Bn, (int)KT, Bc) && Bn >= 192) {
        // persistent CTA pairs (csrc/tc_gemm_nt.cuh): dE = G C with G [Bn][Bc], C [Bc][KT].  Its M tile is 256 rows: with
        // fewer than 192 estimates (cfg3 / cfg5 per-rank batches of 64 / 128) the padding costs more than the single-CTA
        // kernel below loses (measured 0.47 vs 0.32 ms at 64 x 512, 0.75 vs 0.59 ms at 128 x 1024)
        clip_ce_bwd_kernel<<<ew_grid((long long)Bn * Bc), 256, 0, st>>>(probs, inv_norm, gout, Bn, Bc, target_offset, G, 0);
        BM_CHECK_LAUNCH();
        return tc::launch_gemm_nt_pp(G, cand, dest, Bn, (int)KT, Bc, status, st);
    }
    if (tc::wgrad_tc_supported(Bn, (int)KT)) {
        // tensor cores: dE[b][k] = sum_o G^T[o][b] C[o][k]  == weight-gradient GEMM with "positions" = candidates
        clip_ce_bwd_kernel<<<ew_grid((long long)Bn * Bc), 256, 0, st>>>(probs, inv_norm, gout, Bn, Bc, target_offset, G, 1);
        BM_CHECK_LAUNCH();
        return tc::launch_wgrad_tc(G, cand, 1, Bc, Bn, (int)KT, (int)KT, 1, 1, dest, dest, status, st);   // direct mode: no workspace
    }
    clip_ce_bwd_kernel<<<ew_grid((long long)Bn * Bc), 256, 0, st>>>(probs, inv_norm, gout, Bn, Bc, target_offset, G, 0);
    BM_CHECK_LAUNCH();
    GemmP g = gemm_defaults();
    g.M = Bn; g.N = (int)KT; g.K = Bc; g.kchunk = Bc;
    g.A = G; g.lda_m = Bc; g.lda_k = 1;
    g.B = cand; g.ldb_n = 1; g.ldb_k = KT; g.b_ncontig = 1;
    g.D = dest; g.ldd_m = KT; g.ldd_n = 1;
    BM_CUDA(launch_gemm(g, st));
    return 0;
}

// =================================================================================================
// Stand-alone ConvSequence epilogues + candidate-side ClipLoss gradient (SURVEY 8(f) row 3: DeepMel)
// =================================================================================================
extern "C" int bm_bn_act_skip_fwd(const float* y, const float* mean, const float* invstd, const float* gamma,
                                  const float* beta, const float* x_old, float* x_new, long long rows, int C, int act,
                                  float slope, bm_stream_t stream) {
    BM_CHECK_ARG(y && x_new && rows > 0 && C > 0 && act >= 0 && act <= 2);
    BM_CHECK_ARG(!mean || (invstd && gamma && beta));
    bn_act_skip_fwd_kernel<<<ew_grid(rows * C), 256, 0, ST(stream)>>>(y, mean, invstd, gamma, beta, x_old, x_new,
                                                                      rows * C, C, act, slope);
    BM_CHECK_LAUNCH();
    return 0;
}

extern "C" int bm_bn_act_skip_bwd(const float* g, const float* y, const float* mean, const float* invstd,
                                  const float* gamma, const float* beta, int batch_stats, long long rows, int C,
                                  int act, float slope, double* sums, float* dy, float* dgamma, float* dbeta,
                                  bm_stream_t stream) {
    BM_CHECK_ARG(g && y && dy && rows > 0 && C > 0 && act >= 0 && act <= 2);
    BM_CHECK_ARG(!mean || (invstd && gamma && beta && sums && dgamma && dbeta));
    cudaStream_t st = ST(stream);
    if (mean) {
        BM_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * 2 * C, st));
        const int rpb = 128;
        dim3 grid((unsigned)((rows + rpb - 1) / rpb), (C + 127) / 128);
        bn_act_bwd_reduce_kernel<<<grid, 128, 0, st>>>(g, y, mean, invstd, gamma, beta, sums, rows, C, rpb, act, slope);
        BM_CHECK_LAUNCH();
        bn_param_grad_kernel<<<(C + 127) / 128, 128, 0, st>>>(sums, dgamma, dbeta, C);
        BM_CHECK_LAUNCH();
    }
    bn_act_bwd_apply_kernel<<<ew_grid(rows * C), 256, 0, st>>>(g, y, mean, invstd, gamma, beta, sums, (double)rows,
                                                               batch_stats, dy, rows * C, C, act, slope);
    BM_CHECK_LAUNCH();
    return 0;
}

extern "C" int bm_clip_loss_bwd_cand(const float* probs, const float* scores, const float* inv_norm, const float* est,
                                     const float* cand, const float* gout, int Bn, int Bc, long long KT,
                                     int target_offset, float* G, float* coef, float* dcand, int* status,
                                     bm_stream_t stream) {
    BM_CHECK_ARG(probs && scores && inv_norm && est && cand && gout && G && coef && dcand);
    BM_CHECK_ARG(Bn > 0 && Bc > 0 && KT > 0 && KT < (1ll << 31));
    cudaStream_t st = ST(stream);
    clip_ce_bwd_kernel<<<ew_grid((long long)Bn * Bc), 256, 0, st>>>(probs, inv_norm, gout, Bn, Bc, target_offset, G, 0);
    BM_CHECK_LAUNCH();
    clip_cand_coef_kernel<<<(Bc + 127) / 128, 128, 0, st>>>(G, scores, inv_norm, Bn, Bc, coef);     // needs G as [Bn][Bc]
    BM_CHECK_LAUNCH();
    // dcand[o][k] = sum_b G[b][o] est[b][k]
    if (tc::gemm_nt_pp_supported(Bc, (int)KT, Bn)) {
        // persistent CTA pairs (csrc/tc_gemm_nt.cuh): A = G^T [Bc][Bn] (rewritten into the same scratch), B = est [Bn][KT]
        clip_ce_bwd_kernel<<<ew_grid((long long)Bn * Bc), 256, 0, st>>>(probs, inv_norm, gout, Bn, Bc, target_offset, G, 1);
        BM_CHECK_LAUNCH();
        int rc = tc::launch_gemm_nt_pp(G, est, dcand, Bc, (int)KT, Bn, status, st);
        if (rc) return rc;
    } else if (tc::wgrad_tc_supported(Bc, (int)KT)) {
        int rc = tc::launch_wgrad_tc(G, est, 1, Bn, Bc, (int)KT, (int)KT, 1, 1, dcand, dcand, status, st);   // direct mode
        if (rc) return rc;
    } else {
        GemmP g = gemm_defaults();
        g.M = Bc; g.N = (int)KT; g.K = Bn; g.kchunk = Bn;
        g.A = G; g.lda_m = 1; g.lda_k = Bc; g.a_mcontig = 1;
        g.B = est; g.ldb_n = 1; g.ldb_k = KT; g.b_ncontig = 1;
        g.D = dcand; g.ldd_m = KT; g.ldd_n = 1;
        BM_CUDA(launch_gemm(g, st));
    }
    clip_cand_correct_kernel<<<ew_grid((long long)Bc * KT), 256, 0, st>>>(cand, coef, KT, (long long)Bc * KT, dcand);
    BM_CHECK_LAUNCH();
    return 0;
}

// =================================================================================================
// Retrieval evaluation (SURVEY 8(f) row 1)
// =================================================================================================
extern "C" int bm_retrieval_topk(const float* vals, long long ld, int Bn, int n_cols, const float* own_values,
                                 int own_col, int is_prob, int k, const long long* labels,
                                 const long long* own_labels, const long long* targets, long long* top_idx,
                                 float* top_prob, int* hit, float* soft, float* row_max, float* row_sum,
                                 bm_stream_t stream) {
    BM_CHECK_ARG(vals && Bn > 0 && n_cols > 0 && ld >= n_cols && k >= 0);
    BM_CHECK_ARG(!own_values || (own_col >= 0 && own_col < n_cols));
    BM_CHECK_ARG(!own_labels || (labels && own_col >= 0 && own_col < n_cols));
    BM_CHECK_ARG(!(hit || soft) || (labels && targets));
    BM_CHECK_ARG(k == 0 || top_idx || top_prob || hit);
    int threads = n_cols >= 4096 ? 512 : 256;
    retrieval_topk_kernel<<<Bn, threads, 0, ST(stream)>>>(vals, ld, n_cols, own_values, own_col, is_prob, k, labels,
                                                          own_labels, targets, top_idx, top_prob, hit, soft, row_max,
                                                          row_sum);
    BM_CHECK_LAUNCH();
    return 0;
}

extern "C" int bm_retrieval_probs(const float* scores, long long ld, int Bn, int n_cols, float* probs,
                                  bm_stream_t stream) {
    BM_CHECK_ARG(scores && probs && Bn > 0 && n_cols > 0 && ld >= n_cols);
    softmax_rows_ld_kernel<<<Bn, 256, 0, ST(stream)>>>(scores, ld, n_cols, probs);
    BM_CHECK_LAUNCH();
    return 0;
}

extern "C" int bm_retrieval_vocab_probs(const float* scores, long long ld, int Bn, const float* own_scores,
                                        const float* row_max, const float* row_sum, const int* perm, const int* seg,
                                        int V, const int* own_word, float* vocab, bm_stream_t stream) {
    BM_CHECK_ARG(scores && row_max && row_sum && perm && seg && vocab && Bn > 0 && V > 0);
    BM_CHECK_ARG(!own_scores || own_word);
    vocab_probs_kernel<<<Bn, 256, 0, ST(stream)>>>(scores, ld, own_scores, row_max, row_sum, perm, seg, V, own_word,
                                                   vocab);
    BM_CHECK_LAUNCH();
    return 0;
}

extern "C" int bm_rowdot_scaled(const float* a, const float* c, int Bn, long long K, float* own,
                                bm_stream_t stream) {
    BM_CHECK_ARG(a && c && own && Bn > 0 && K > 0);
    rowdot_scaled_kernel<<<Bn, 512, 0, ST(stream)>>>(a, c, K, own);
    BM_CHECK_LAUNCH();
    return 0;
}

// =================================================================================================
// Batch preparation (SURVEY 8(f) row 2)
// =================================================================================================
extern "C" int bm_scale_clamp_crop(const float* x, const int* slot, const float* center, const float* scale, int B,
                                   int C, int T, int t0, int T_out, float limit, int clip, int inverse, float* y,
                                   unsigned int* peak_bits, bm_stream_t stream) {
    BM_CHECK_ARG(x && center && scale && y && B > 0 && C > 0 && T > 0);
    BM_CHECK_ARG(t0 >= 0 && T_out > 0 && t0 + T_out <= T);
    BM_CHECK_ARG(!clip || limit >= 0.f);
    cudaStream_t st = ST(stream);
    if (peak_bits) BM_CUDA(cudaMemsetAsync(peak_bits, 0, sizeof(unsigned) * B, st));
    long long rows = (long long)B * C;
    long long blocks = (rows + 7) / 8;                       // 8 warps (rows) per block
    long long cap = (long long)num_sms() * 8;                // one full wave of 2048-thread SMs, grid-stride beyond
    if (blocks > cap) blocks = cap;
    scale_clamp_crop_kernel<<<(unsigned)blocks, 256, 0, st>>>(x, slot, center, scale, B, C, T, t0, T_out, limit, clip,
                                                             inverse, y, peak_bits);
    BM_CHECK_LAUNCH();
    return 0;
}

extern "C" int bm_reject_compact(const unsigned int* peak_bits, const unsigned char* mask, long long mask_elems,
                                 float limit, int B, unsigned char* keep, int* keep_rows, int* n_keep,
                                 bm_stream_t stream) {
    BM_CHECK_ARG(peak_bits && keep && keep_rows && n_keep && B > 0);
    BM_CHECK_ARG(!mask || mask_elems > 0);
    reject_compact_kernel<<<1, 1024, 0, ST(stream)>>>(peak_bits, mask, mask_elems, limit, B, keep, keep_rows, n_keep);
    BM_CHECK_LAUNCH();
    return 0;
}

extern "C" int bm_gather_rows(const float* x, const int* rows, int n_rows, long long row_elems, float* y,
                              bm_stream_t stream) {
    BM_CHECK_ARG(x && rows && y && n_rows > 0 && row_elems > 0);
    gather_rows_kernel<<<ew_grid((long long)n_rows * row_elems), 256, 0, ST(stream)>>>(x, rows, n_rows, row_elems, y);
    BM_CHECK_LAUNCH();
    return 0;
}

// =================================================================================================
// Regression objectives (L1Loss / L2Loss, bm/losses.py:11-26)
// =================================================================================================
extern "C" int bm_regression_loss_fwd(const float* est, const float* out, const unsigned char* mask, int B, int F, int Fm,
                                      int T, int p, double* workspace, float* loss, bm_stream_t stream) {
    BM_CHECK_ARG(est && out && mask && workspace && loss);
    BM_CHECK_ARG(B > 0 && F > 0 && T > 0 && (Fm == 1 || Fm == F) && (p == 1 || p == 2));
    const long long rows = (long long)B * F;
    const int grid = regression_grid(rows * T);
    const bool vec = T % 4 == 0 && reg_aligned(est, 16) && reg_aligned(out, 16) && reg_aligned(mask, 4);
    cudaStream_t st = ST(stream);
    BM_CUDA(cudaMemsetAsync(workspace + REG_WS_TICKET, 0, sizeof(unsigned int), st));
    if (p == 1)
        launch_regression_fwd_p<1>(vec, grid, est, out, mask, rows, F, Fm == F, T, workspace, loss, st);
    else
        launch_regression_fwd_p<2>(vec, grid, est, out, mask, rows, F, Fm == F, T, workspace, loss, st);
    BM_CHECK_LAUNCH();
    return 0;
}

extern "C" int bm_regression_loss_bwd(const float* est, const float* out, const unsigned char* mask, const float* gout,
                                      const double* workspace, int B, int F, int Fm, int T, int p, float* dest, float* dout,
                                      bm_stream_t stream) {
    BM_CHECK_ARG(est && out && mask && gout && workspace && (dest || dout));
    BM_CHECK_ARG(B > 0 && F > 0 && T > 0 && (Fm == 1 || Fm == F) && (p == 1 || p == 2));
    const long long rows = (long long)B * F;
    const int grid = regression_grid(rows * T);
    const bool vec = T % 4 == 0 && reg_aligned(est, 16) && reg_aligned(out, 16) && reg_aligned(mask, 4) &&
                     reg_aligned(dest, 16) && reg_aligned(dout, 16);
    cudaStream_t st = ST(stream);
    if (p == 1)
        launch_regression_bwd_p<1>(vec, grid, est, out, mask, rows, F, Fm == F, T, gout, workspace, dest, dout, st);
    else
        launch_regression_bwd_p<2>(vec, grid, est, out, mask, rows, F, Fm == F, T, gout, workspace, dest, dout, st);
    BM_CHECK_LAUNCH();
    return 0;
}

// =================================================================================================
// tcgen05 (tensor-core) versions of K3/K4
// =================================================================================================
extern "C" int bm_tc_conv_supported(int T, int Cin, int Ntot, int Kw, int glu) {
    return tc::conv_tc_supported(T, Cin, Ntot, Kw, glu) ? 1 : 0;
}

extern "C" int bm_tc_weight_split(const float* w, int Cout, int Cin, int Kw, float* f_hi, float* f_lo, float* g_hi,
                                  float* g_lo, bm_stream_t stream) {
    BM_CHECK_ARG(w && Cout > 0 && Cin > 0 && Kw > 0);
    BM_CHECK_ARG((f_hi || g_hi) && !(f_lo && !f_hi) && !(g_lo && !g_hi));
    tc::weight_split_kernel<<<ew_grid((long long)Cout * Cin * Kw), 256, 0, ST(stream)>>>(w, f_hi, f_lo, g_hi, g_lo,
                                                                                       Cout, Cin, Kw);
    BM_CHECK_LAUNCH();
    return 0;
}

extern "C" int bm_tc_conv1d(const float* x, const float* w_hi, const float* w_lo, const float* bias,
                            const float* addend, int B, int T, int Cin, int Ntot, int Kw, int dilation, int sign,
                            int glu, int act, int out_tmajor, float* y, float* aux, float* glu_out, double* stats,
                            int* status, bm_stream_t stream) {
    BM_CHECK_ARG(stats == nullptr);      // only the CTA-pair kernel produces BatchNorm statistics in its epilogue
    BM_CHECK_ARG(x && w_hi && w_lo && B > 0 && T > 0 && dilation >= 1 && (sign == 1 || sign == -1));
    BM_CHECK_ARG(glu ? (glu_out != nullptr) : (y != nullptr));
    BM_CHECK_ARG(B <= 65535);
    BM_CHECK_ARG(!(glu && (act || out_tmajor || aux)));
    BM_CHECK_ARG(tc::conv_tc_supported(T, Cin, Ntot, Kw, glu));
    tc::ConvTcP p;
    p.B = B; p.T = T; p.Cin = Cin; p.Ntot = Ntot; p.taps = Kw; p.dilation = dilation; p.sign = sign; p.glu = glu;
    p.bias = bias; p.addend = addend; p.y = y; p.glu_out = glu_out; p.err = status;
    p.act = act; p.out_tmajor = out_tmajor; p.aux = aux; p.bn = 0; p.wsel = nullptr; p.n_wsets = 1;
    BM_CHECK_ARG(!(glu && (act || out_tmajor || aux)));
    return tc::launch_conv_tc(x, w_hi, w_lo, p, ST(stream));
}

// per-column sum / sum of squares of a channels-last matrix (BatchNorm batch statistics after the tcgen05 conv)
extern "C" int bm_col_stats(const float* y, long long rows, int C, double* stats, bm_stream_t stream) {
    BM_CHECK_ARG(y && stats && rows > 0 && C > 0);
    cudaStream_t st = ST(stream);
    BM_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * 2 * C, st));
    {
        const int rpb = 128;
        dim3 grid((unsigned)((rows + rpb - 1) / rpb), (C + 127) / 128);
        col_stats_kernel<<<grid, 128, 0, st>>>(y, stats, rows, C, rpb);
    }
    BM_CHECK_LAUNCH();
    return 0;
}

// y = x * mask[c] over [B, C, T] (SimpleConv's subsample_meg_channels, simpleconv.py:97-102,200-203); y may alias x
extern "C" int bm_channel_mask(const float* x, const float* mask, int B, int C, int T, float* y, bm_stream_t stream) {
    BM_CHECK_ARG(x && mask && y && B > 0 && C > 0 && T > 0);
    const long long total = (long long)B * C * T;
    channel_mask_kernel<<<ew_grid(total), 256, 0, ST(stream)>>>(x, mask, y, C, T, total);
    BM_CHECK_LAUNCH();
    return 0;
}

// [Z, N, T] (channel-major) -> [Z, T, N] (channels-last)
extern "C" int bm_transpose_nt(const float* in, int Z, int N, int T, float* out, bm_stream_t stream) {
    BM_CHECK_ARG(in && out && Z > 0 && N > 0 && T > 0 && Z <= 65535);
    dim3 grid((T + 31) / 32, (N + 31) / 32, Z);
    transpose_nt_kernel<<<grid, dim3(32, 8), 0, ST(stream)>>>(in, out, N, T, N, N);
    BM_CHECK_LAUNCH();
    return 0;
}

// same with an output row stride ld_out >= N; the pad columns N..ld_out-1 are written as zeros
extern "C" int bm_transpose_nt_ld(const float* in, int Z, int N, int T, int ld_out, float* out, bm_stream_t stream) {
    BM_CHECK_ARG(in && out && Z > 0 && N > 0 && T > 0 && Z <= 65535 && ld_out >= N);
    dim3 grid((T + 31) / 32, (ld_out + 31) / 32, Z);
    transpose_nt_kernel<<<grid, dim3(32, 8), 0, ST(stream)>>>(in, out, N, T, ld_out, ld_out);
    BM_CHECK_LAUNCH();
    return 0;
}

// weight gradient of a (dilated) conv / pointwise layer on the tensor cores: dW[m][n][tap] = sum_{b,t} dY[b,t,m] X[b,t+s,n]
extern "C" int bm_tc_wgrad_supported(int M, int N) { return tc::wgrad_tc_supported(M, N) ? 1 : 0; }
extern "C" long long bm_tc_wgrad_workspace(int B, int M, int N, int Kw) {
    return (long long)tc::wgrad_workspace_floats(B, M, N, Kw);
}
extern "C" int bm_tc_wgrad(const float* dy, const float* x, int B, int T, int M, int N, int Ntrue, int Kw,
                           int dilation, float* workspace, float* dw, float* dbias, int* status, bm_stream_t stream) {
    BM_CHECK_ARG(dy && x && workspace && dw && B > 0 && T > 0 && Kw >= 1 && Kw <= 3 && dilation >= 1);
    BM_CHECK_ARG(tc::wgrad_tc_supported(M, N) && Ntrue > 0 && Ntrue <= N);
    return tc::launch_wgrad_tc(dy, x, B, T, M, N, Ntrue, Kw, dilation, workspace, dw, status, ST(stream), dbias);
}

// CTA-pair weight gradient of a k-tap conv (csrc/tc_wgradp.cuh): output rows = (tap, x channel), reduction over the
// flattened rows; no bias gradient (use bm_col_sum on dy where the layer's bias gradient is not exactly zero)
extern "C" int bm_tc_wgrad_conv_supported(int T, int M, int N, int Kw) {
    return tc::wgradp_supported(T, M, N, Kw) ? 1 : 0;
}
extern "C" long long bm_tc_wgrad_conv_workspace(int B, int T, int M, int N, int Kw) {
    return (long long)tc::wgradp_workspace_floats(B, T, M, N, Kw);
}
extern "C" int bm_tc_wgrad_conv(const float* dy, const float* x, int B, int T, int M, int N, int Ntrue, int Kw,
                                int dilation, float* workspace, float* dw, int* status, bm_stream_t stream) {
    BM_CHECK_ARG(dy && x && workspace && dw && B > 0 && T > 0 && dilation >= 1);
    BM_CHECK_ARG(tc::wgradp_supported(T, M, N, Kw) && Ntrue > 0 && Ntrue <= N);
    return tc::launch_wgrad_pp(dy, x, B, T, M, N, Ntrue, Kw, dilation, workspace, dw, status, ST(stream));
}

// the same weight gradient on the F16 pipe (csrc/tc_wgradh.cuh): dy_amax / x_amax = device floats with max |dy|, max |x|
// (bm_amax, or the amax_out of the kernels that produced the tensors); same shape gate and workspace as bm_tc_wgrad_conv
extern "C" int bm_tc_wgrad_conv_f16(const float* dy, const float* dy_amax, const float* x, const float* x_amax, int B, int T,
                                    int M, int N, int Ntrue, int Kw, int dilation, float* workspace, float* dw, int* status,
                                    bm_stream_t stream) {
    BM_CHECK_ARG(dy && dy_amax && x && x_amax && workspace && dw && B > 0 && T > 0 && dilation >= 1);
    BM_CHECK_ARG(tc::wgradp_supported(T, M, N, Kw) && Ntrue > 0 && Ntrue <= N);
    return tc::launch_wgrad_hp(dy, dy_amax, x, x_amax, B, T, M, N, Ntrue, Kw, dilation, workspace, dw, status, ST(stream));
}

extern "C" int bm_col_sum(const float* x, long long rows, int C, float* out, bm_stream_t stream) {
    BM_CHECK_ARG(x && out && rows > 0 && C > 0);
    cudaStream_t st = ST(stream);
    BM_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * C, st));
    {
        dim3 grid((unsigned)((rows + 255) / 256), (C + 127) / 128);
        colsum_cl_kernel<<<grid, 128, 0, st>>>(x, out, rows, C, 256);
    }
    BM_CHECK_LAUNCH();
    return 0;
}

// dh = dq * GELU'(h)  (elementwise; dh may alias dq)
extern "C" int bm_gelu_bwd(const float* dq, const float* h, long long n, float* dh, bm_stream_t stream) {
    BM_CHECK_ARG(dq && h && dh && n > 0);
    if (n % 4 == 0 && aligned16(dq, h, dh))
        gelu_bwd_v4_kernel<<<ew_grid(n / 4), 256, 0, ST(stream)>>>(
            reinterpret_cast<const float4*>(dq), reinterpret_cast<const float4*>(h), reinterpret_cast<float4*>(dh), n / 4);
    else
        gelu_bwd_kernel<<<ew_grid(n), 256, 0, ST(stream)>>>(dq, h, dh, n);
    BM_CHECK_LAUNCH();
    return 0;
}

extern "C" int bm_tc_conv1d_persistent_supported(int T, int Cin, int Ntot, int Kw, int glu) {
    return tc::conv_pp_supported(T, Cin, Ntot, Kw, glu) ? 1 : 0;
}
// persistent CTA-pair kernel (csrc/tc_convp.cuh): w_raw = the RAW fp32 weights re-laid K-major [Kw][Ntot][Cin]
// (bm_tc_weight_split with f_lo / g_lo = NULL); accumulate=1: y += conv (in place, TMA reduce-add)
extern "C" int bm_tc_conv1d_persistent(const float* x, const float* w_raw, const float* bias, int accumulate, int B, int T,
                                       int Cin, int Ntot, int Kw, int dilation, int sign, int glu, int act,
                                       int out_tmajor, float* y, float* aux, float* glu_out, double* stats, int* status,
                                       bm_stream_t stream) {
    BM_CHECK_ARG(x && w_raw && B > 0 && T > 0 && dilation >= 1 && (sign == 1 || sign == -1));
    BM_CHECK_ARG(glu ? (glu_out != nullptr) : (y != nullptr));
    BM_CHECK_ARG(tc::conv_pp_supported(T, Cin, Ntot, Kw, glu));
    tc::ConvPPArgs a;
    a.x = x; a.w_raw = w_raw; a.bias = bias; a.B = B; a.T = T; a.Cin = Cin; a.Ntot = Ntot; a.taps = Kw;
    a.dilation = dilation; a.sign = sign; a.glu = glu; a.act = act; a.out_tmajor = out_tmajor; a.accumulate = accumulate;
    a.y = y; a.aux = aux; a.glu_out = glu_out; a.stats = stats; a.err = status;
    return tc::launch_conv_pp(a, ST(stream));
}

// ---- the same conv on the F16 tensor pipe (csrc/tc_convh.cuh): fp32 operands as two fp16 pieces of a power-of-two-scaled
// tensor.  bm_amax writes the largest magnitude of a tensor into a device float; bm_f16_split prepares the weights
// (w_raw [Kw][Ntot][Cin] -> fp16 hi / lo copies of w_raw * scale(amax)); the kernel scales x itself.
extern "C" int bm_amax(const float* x, long long n, float* amax, bm_stream_t stream) {
    BM_CHECK_ARG(x && amax && n > 0);
    return tc::launch_amax(x, n, amax, ST(stream));
}
extern "C" int bm_f16_split(const float* src, long long n, const float* amax, void* hi, void* lo, bm_stream_t stream) {
    BM_CHECK_ARG(src && amax && hi && lo && n > 0);
    return tc::launch_f16_split(src, n, amax, hi, lo, ST(stream));
}
extern "C" int bm_tc_weight_split_f16(const float* w, const float* w_amax, int Cout, int Cin, int Kw, void* f_hi, void* f_lo,
                                      void* g_hi, void* g_lo, bm_stream_t stream) {
    BM_CHECK_ARG(w && w_amax && Cout > 0 && Cin > 0 && Kw > 0);
    BM_CHECK_ARG((f_hi || g_hi) && (!f_hi == !f_lo) && (!g_hi == !g_lo));
    tc::weight_split_f16_kernel<<<ew_grid((long long)Cout * Cin * Kw), 256, 0, ST(stream)>>>(
        w, w_amax, reinterpret_cast<__half*>(f_hi), reinterpret_cast<__half*>(f_lo), reinterpret_cast<__half*>(g_hi),
        reinterpret_cast<__half*>(g_lo), Cout, Cin, Kw);
    BM_CHECK_LAUNCH();
    return 0;
}
extern "C" int bm_tc_conv1d_f16(const float* x, const float* x_amax, const void* w_hi, const void* w_lo, const float* w_amax,
                                const float* bias, int accumulate, int B, int T, int Cin, int Ntot, int Kw, int dilation,
                                int sign, int glu, int act, int out_tmajor, float* y, float* aux, float* glu_out,
                                double* stats, float* amax_out, int* status, bm_stream_t stream) {
    BM_CHECK_ARG(x && x_amax && w_hi && w_lo && w_amax && B > 0 && T > 0 && dilation >= 1 && (sign == 1 || sign == -1));
    BM_CHECK_ARG(glu ? (glu_out != nullptr) : (y != nullptr));
    BM_CHECK_ARG(tc::conv_pp_supported(T, Cin, Ntot, Kw, glu));
    tc::ConvHPArgs h;
    tc::ConvPPArgs& a = h.c;
    a.x = x; a.w_raw = nullptr; a.bias = bias; a.B = B; a.T = T; a.Cin = Cin; a.Ntot = Ntot; a.taps = Kw;
    a.dilation = dilation; a.sign = sign; a.glu = glu; a.act = act; a.out_tmajor = out_tmajor; a.accumulate = accumulate;
    a.y = y; a.aux = aux; a.glu_out = glu_out; a.stats = stats; a.err = status;
    h.x_amax = x_amax; h.w_hi = w_hi; h.w_lo = w_lo; h.w_amax = w_amax; h.out_amax = amax_out;
    BM_CHECK_ARG(!amax_out || ((glu || act) && !out_tmajor));      // the outputs another conv consumes: GLU out, GELU out
    if (int rc = amax_begin(amax_out, ST(stream))) return rc;
    return tc::launch_conv_hp(h, ST(stream));
}

// pointwise (1x1) contraction with a per-sample weight set (SubjectLayers.forward / its data gradient, common.py:55-58):
//   y[b,t,n] = sum_k x[b,t,k] W[wsel[b]][n][k];  w_hi/w_lo are the tf32-split K-major weight sets [S][Ntot][Cin]
extern "C" int bm_tc_pointwise_sel(const float* x, const float* w_hi, const float* w_lo, const int* wsel, int n_sets,
                                   int B, int T, int Cin, int Ntot, float* y, int* status, bm_stream_t stream) {
    BM_CHECK_ARG(x && w_hi && w_lo && wsel && y && n_sets > 0 && B > 0 && B <= 65535 && T > 0);
    BM_CHECK_ARG(tc::conv_tc_supported(T, Cin, Ntot, 1, 0));
    tc::ConvTcP p;
    p.B = B; p.T = T; p.Cin = Cin; p.Ntot = Ntot; p.taps = 1; p.dilation = 1; p.sign = 1; p.glu = 0;
    p.bias = nullptr; p.addend = nullptr; p.y = y; p.glu_out = nullptr; p.err = status;
    p.act = 0; p.out_tmajor = 0; p.aux = nullptr; p.bn = 0; p.wsel = wsel; p.n_wsets = n_sets;
    return tc::launch_conv_tc(x, w_hi, w_lo, p, ST(stream));
}

// per-group pointwise weight gradient (SubjectLayers: dM[s] = sum over the samples of subject s), tensor cores:
//   out[g][m][n] = sum_{b in group g} sum_t dy[b,t,m] x[b,t,n];  out is [G][ceil(M/128)*128][N]
extern "C" int bm_tc_wgrad_grouped(const float* dy, const float* x, const int* order, const int* seg_off, int G, int B,
                                   int T, int M, int N, float* out, int* status, bm_stream_t stream) {
    BM_CHECK_ARG(dy && x && order && seg_off && out && G > 0 && B > 0 && T > 0);
    BM_CHECK_ARG(tc::wgrad_tc_supported(M, N));
    return tc::launch_wgrad_tc_grouped(dy, x, order, seg_off, G, B, T, M, N, out, status, ST(stream));
}

// ---- K1 pieces, for callers that run the two attention contractions on the tensor cores -------------------------
extern "C" int bm_fourier_emb(const float* positions, const float* freq, int R, int C, int P, float* emb,
                              bm_stream_t stream) {
    BM_CHECK_ARG(positions && freq && emb && R > 0 && C > 0 && P > 0 && P % 2 == 0);
    int n = 0;
    while ((n + 1) * (n + 1) * 2 <= P) ++n;
    BM_CHECK_ARG(n * n * 2 == P);
    fourier_emb_kernel<<<ew_grid((long long)R * C * n * n), 256, 0, ST(stream)>>>(positions, freq, 0.2f, R * C, n, emb);
    BM_CHECK_LAUNCH();
    return 0;
}
// in-place: weights[r][o][:] = softmax_c(scores + mask), mask = -inf on INVALID / banned sensors (common.py:339-357)
extern "C" int bm_masked_softmax(float* weights, const float* positions, const float* ban_centre, float radius, int R,
                                 int O, int C, bm_stream_t stream) {
    BM_CHECK_ARG(weights && positions && R > 0 && O > 0 && C > 0);
    int rows = R * O;
    masked_softmax_kernel<<<(rows + 7) / 8, 256, 0, ST(stream)>>>(weights, positions, ban_centre, radius, -0.1f, R, O, C);
    BM_CHECK_LAUNCH();
    return 0;
}
// dscores = w * (dw - sum_c w dw), rows of length C
extern "C" int bm_softmax_bwd(const float* weights, const float* dweights, long long rows, int C, float* dscores,
                              bm_stream_t stream) {
    BM_CHECK_ARG(weights && dweights && dscores && rows > 0 && C > 0);
    softmax_bwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, ST(stream)>>>(weights, dweights, dscores, (int)rows, C);
    BM_CHECK_LAUNCH();
    return 0;
}
