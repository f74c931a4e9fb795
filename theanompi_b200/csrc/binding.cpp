// pybind11 bindings of the sm_100a extension.  Torch-free on purpose: tensors cross the boundary as raw device
// pointers (tensor.data_ptr()) and streams as cudaStream_t handles (torch.cuda.current_stream().cuda_stream); the
// Python wrappers in theanompi_b200/ops/cuda_impl.py and parallel/symmetric.py own shape / dtype / contiguity checks.
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <cstring>
#include <memory>
#include <vector>

#include "api.h"
#include "peer_arena.h"

namespace py = pybind11;
using namespace tmpi;
typedef uintptr_t ptr_t;

static inline void* P(ptr_t p) { return reinterpret_cast<void*>(p); }
static inline cudaStream_t S(ptr_t s) { return reinterpret_cast<cudaStream_t>(s); }
static inline cudaStream_t S_(ptr_t s) { return reinterpret_cast<cudaStream_t>(s); }

static GroupTable make_table(const std::vector<float>& lr_mult, const std::vector<float>& wd, const std::vector<int>& exch) {
  GroupTable t;
  for (int i = 0; i < kMaxGroups; ++i) {
    t.lr_mult[i] = i < (int)lr_mult.size() ? lr_mult[i] : 1.f;
    t.wd[i] = i < (int)wd.size() ? wd[i] : 0.f;
    t.exch[i] = i < (int)exch.size() ? exch[i] : 1;
  }
  return t;
}

struct PyComm {   // shared_ptr-held wrapper so kernels always see a live mapping
  std::unique_ptr<PeerArena> pa;
};

PYBIND11_MODULE(_tmpi_native, m) {
  m.doc() = "theanompi_b200 native sm_100a kernels and peer-memory runtime";
  m.def("launch_count", [] { return (unsigned long long)g_launch_count.load(); });
  m.def("reset_launch_count", [] { g_launch_count.store(0); });
  m.def("capture_status", [](ptr_t st) {
    cudaStreamCaptureStatus s = cudaStreamCaptureStatusNone;
    cudaError_t e = cudaStreamIsCapturing(S(st), &s);
    return py::make_tuple((int)e, (int)s);
  });
  m.attr("ARENA_BLOCK") = kArenaBlock;
  m.attr("MAX_RANKS") = kMaxRanks;
  m.attr("MAX_COMM_BLOCKS") = kMaxCommBlocks;

  // ---------------------------------------------------------------- GEMM
  m.def("gemm_set_debug", &gemm_set_debug);
  m.def("gemm_set_bulk", &gemm_set_bulk);
  m.def("gemm_rs_add_range", [](ptr_t c_lo, ptr_t c_hi, long long blo, long long per) { gemm_rs_add_range(P(c_lo), P(c_hi), blo, per); });
  m.def("gemm_rs_clear", &gemm_rs_clear);
  m.def("gemm_plan_splits", &gemm_plan_splits);
  m.def("gemm_plan_tall", &gemm_plan_tall);
  m.def("gemm_bf16", [](ptr_t A, ptr_t B, ptr_t C, ptr_t bias, int M, int N, int K, long long lda, long long ldb, long long ldc,
                        int a_mn, int b_mn, int out_bf16, int bias_mode, int relu, float alpha, int bn_hint, int splitk, ptr_t st, int tf32) {
    gemm_bf16(P(A), P(B), P(C), (const float*)P(bias), M, N, K, lda, ldb, ldc, a_mn, b_mn, out_bf16, bias_mode, relu, alpha, bn_hint,
              splitk, S(st), tf32);
  }, py::arg("A"), py::arg("B"), py::arg("C"), py::arg("bias"), py::arg("M"), py::arg("N"), py::arg("K"), py::arg("lda"), py::arg("ldb"),
     py::arg("ldc"), py::arg("a_mn"), py::arg("b_mn"), py::arg("out_bf16"), py::arg("bias_mode"), py::arg("relu"), py::arg("alpha"),
     py::arg("bn_hint"), py::arg("splitk"), py::arg("st"), py::arg("tf32") = 0);

  m.def("conv_fprop", [](ptr_t x, ptr_t w, ptr_t y, ptr_t bias, int N, int H, int W, int Ctot, int c_off, int Cg, int KH, int KW, int Ho, int Wo,
                         int S, int Pd, int O, long long ldc, int relu, int out_bf16, int dgrad, ptr_t st, int tf32) {
    conv_fprop_bf16(P(x), P(w), P(y), (const float*)P(bias), N, H, W, Ctot, c_off, Cg, KH, KW, Ho, Wo, S, Pd, O, ldc, relu, out_bf16, dgrad,
                    S_(st), tf32);
  }, py::arg("x"), py::arg("w"), py::arg("y"), py::arg("bias"), py::arg("N"), py::arg("H"), py::arg("W"), py::arg("Ctot"), py::arg("c_off"),
     py::arg("Cg"), py::arg("KH"), py::arg("KW"), py::arg("Ho"), py::arg("Wo"), py::arg("S"), py::arg("P"), py::arg("O"), py::arg("ldc"),
     py::arg("relu"), py::arg("out_bf16"), py::arg("dgrad"), py::arg("st"), py::arg("tf32") = 0);
  m.def("conv_wgrad", [](ptr_t dy, ptr_t x, ptr_t dw, int N, int H, int W, int Ctot, int c_off, int Cg, int KH, int KW, int Ho, int Wo, int S,
                         int Pd, int O, long long ldy, ptr_t st, int tf32) {
    conv_wgrad_bf16(P(dy), P(x), P(dw), N, H, W, Ctot, c_off, Cg, KH, KW, Ho, Wo, S, Pd, O, ldy, S_(st), tf32);
  }, py::arg("dy"), py::arg("x"), py::arg("dw"), py::arg("N"), py::arg("H"), py::arg("W"), py::arg("Ctot"), py::arg("c_off"), py::arg("Cg"),
     py::arg("KH"), py::arg("KW"), py::arg("Ho"), py::arg("Wo"), py::arg("S"), py::arg("P"), py::arg("O"), py::arg("ldy"), py::arg("st"),
     py::arg("tf32") = 0);
  m.def("conv_fprop2", [](ptr_t x, ptr_t w0, ptr_t w1, ptr_t y0, ptr_t y1, ptr_t b0, ptr_t b1, int N, int H, int W, int Ctot, int c_off0, int c_off1,
                          int Cg, int KH, int KW, int Ho, int Wo, int S, int Pd, int O, long long ldc, int relu, int out_bf16, int dgrad, ptr_t st,
                          int tf32) {
    conv_fprop2_bf16(P(x), P(w0), P(w1), P(y0), P(y1), (const float*)P(b0), (const float*)P(b1), N, H, W, Ctot, c_off0, c_off1, Cg, KH, KW, Ho,
                     Wo, S, Pd, O, ldc, relu, out_bf16, dgrad, S_(st), tf32);
  }, py::arg("x"), py::arg("w0"), py::arg("w1"), py::arg("y0"), py::arg("y1"), py::arg("b0"), py::arg("b1"), py::arg("N"), py::arg("H"),
     py::arg("W"), py::arg("Ctot"), py::arg("c_off0"), py::arg("c_off1"), py::arg("Cg"), py::arg("KH"), py::arg("KW"), py::arg("Ho"),
     py::arg("Wo"), py::arg("S"), py::arg("P"), py::arg("O"), py::arg("ldc"), py::arg("relu"), py::arg("out_bf16"), py::arg("dgrad"),
     py::arg("st"), py::arg("tf32") = 0);
  m.def("conv_wgrad2", [](ptr_t dy0, ptr_t dy1, ptr_t x, ptr_t dw0, ptr_t dw1, int N, int H, int W, int Ctot, int c_off0, int c_off1, int Cg,
                          int KH, int KW, int Ho, int Wo, int S, int Pd, int O, long long ldy, ptr_t st, int tf32) {
    conv_wgrad2_bf16(P(dy0), P(dy1), P(x), P(dw0), P(dw1), N, H, W, Ctot, c_off0, c_off1, Cg, KH, KW, Ho, Wo, S, Pd, O, ldy, S_(st), tf32);
  }, py::arg("dy0"), py::arg("dy1"), py::arg("x"), py::arg("dw0"), py::arg("dw1"), py::arg("N"), py::arg("H"), py::arg("W"), py::arg("Ctot"),
     py::arg("c_off0"), py::arg("c_off1"), py::arg("Cg"), py::arg("KH"), py::arg("KW"), py::arg("Ho"), py::arg("Wo"), py::arg("S"),
     py::arg("P"), py::arg("O"), py::arg("ldy"), py::arg("st"), py::arg("tf32") = 0);
  m.def("space_to_depth", [](ptr_t x, ptr_t y, int N, int H, int W, int C, int S, int Hs, int Ws, int Cp, int Pd, ptr_t st) {
    space_to_depth(P(x), P(y), N, H, W, C, S, Hs, Ws, Cp, Pd, S_(st)); });
  m.def("s2d_filter", [](ptr_t src, ptr_t dst, int O, int KH, int KW, int C, int S, int KHs, int KWs, int Cp, int dir, ptr_t st) {
    s2d_filter(P(src), P(dst), O, KH, KW, C, S, KHs, KWs, Cp, dir, S_(st)); });
  m.def("conv_weight_flip", [](ptr_t w, ptr_t wt, int O, int KH, int KW, int Cg, ptr_t st) { conv_weight_flip(P(w), P(wt), O, KH, KW, Cg, S_(st)); });

  // ---------------------------------------------------------------- layer kernels
  m.def("lrn_fwd", [](ptr_t x, ptr_t y, long long rows, int C, int n, float k, float alpha, float beta, ptr_t st) {
    lrn_fwd(P(x), P(y), rows, C, n, k, alpha, beta, S(st)); });
  m.def("lrn_bwd", [](ptr_t x, ptr_t dy, ptr_t dx, long long rows, int C, int n, float k, float alpha, float beta, ptr_t st) {
    lrn_bwd(P(x), P(dy), P(dx), rows, C, n, k, alpha, beta, S(st)); });
  m.def("pool_fwd", [](ptr_t x, ptr_t y, ptr_t arg, int N, int H, int W, int C, int Ho, int Wo, int k, int s, int p, int is_max, ptr_t st) {
    pool_fwd(P(x), P(y), P(arg), N, H, W, C, Ho, Wo, k, s, p, is_max, S(st)); });
  m.def("pool_bwd", [](ptr_t dy, ptr_t arg, ptr_t dx, int N, int H, int W, int C, int Ho, int Wo, int k, int s, int p, int is_max, ptr_t st) {
    pool_bwd(P(dy), P(arg), P(dx), N, H, W, C, Ho, Wo, k, s, p, is_max, S(st)); });
  m.def("dropout_fwd", [](ptr_t x, ptr_t y, ptr_t mask, long long n, float p, unsigned long long seed, int layer, ptr_t step, ptr_t st) {
    dropout_fwd(P(x), P(y), P(mask), n, p, seed, layer, P(step), S(st)); });
  m.def("dropout_bwd", [](ptr_t dy, ptr_t mask, ptr_t dx, long long n, ptr_t st) { dropout_bwd(P(dy), P(mask), P(dx), n, S(st)); });
  m.def("advance_step", [](ptr_t step, ptr_t st) { advance_step(P(step), S(st)); });
  m.def("softmax_xent", [](ptr_t logits, ptr_t labels, ptr_t dlogits, ptr_t rowstat, ptr_t out3, int B, int C, float weight, ptr_t st) {
    softmax_xent(P(logits), P(labels), P(dlogits), P(rowstat), P(out3), B, C, weight, S(st)); });
  m.def("maxpool_relu_bias_bwd", [](ptr_t dyp, ptr_t arg, ptr_t y, ptr_t dym, ptr_t db0, ptr_t db1, int c_split, int N, int H, int W, int C,
                                    int Ho, int Wo, int k, int s, int p, ptr_t st) {
    maxpool_relu_bias_bwd(P(dyp), P(arg), P(y), P(dym), P(db0), P(db1), c_split, N, H, W, C, Ho, Wo, k, s, p, S(st)); });
  m.def("relu_bias_bwd2", [](ptr_t dy, ptr_t y, ptr_t dym, ptr_t db, ptr_t db1, int c_split, long long R, int C, long long ld, int relu, ptr_t st) {
    relu_bias_bwd2(P(dy), P(y), P(dym), P(db), P(db1), c_split, R, C, ld, relu, S(st)); });
  m.def("relu_bias_bwd", [](ptr_t dy, ptr_t y, ptr_t dym, ptr_t db, long long R, int C, long long ld, int relu, ptr_t st) {
    relu_bias_bwd(P(dy), P(y), P(dym), P(db), R, C, ld, relu, S(st)); });
  m.def("im2col", [](ptr_t x, ptr_t col, int N, int H, int W, int Ctot, int c_off, int Cg, int KH, int KW, int Ho, int Wo, int s, int p,
                     long long ldcol, ptr_t st) { im2col(P(x), P(col), N, H, W, Ctot, c_off, Cg, KH, KW, Ho, Wo, s, p, ldcol, S(st)); });
  m.def("col2im", [](ptr_t dcol, ptr_t dx, int N, int H, int W, int Ctot, int c_off, int Cg, int KH, int KW, int Ho, int Wo, int s, int p,
                     long long ldcol, ptr_t st) { col2im(P(dcol), P(dx), N, H, W, Ctot, c_off, Cg, KH, KW, Ho, Wo, s, p, ldcol, S(st)); });
  m.def("pad_rows", [](ptr_t src, ptr_t dst, long long rows, int cols, long long src_ld, long long dst_ld, ptr_t st) {
    pad_rows(P(src), P(dst), rows, cols, src_ld, dst_ld, S(st)); });
  m.def("transpose_bf16", [](ptr_t src, ptr_t dst, int R, int C, ptr_t st) { transpose_bf16(P(src), P(dst), R, C, S(st)); });
  m.def("crop_mirror_norm", [](ptr_t x, int in_kind, ptr_t mean, int mean_mode, float scale, ptr_t cscale, ptr_t out, int out_bf16, ptr_t offs,
                               ptr_t flips, int N, int H, int W, int C, int ch, int cw, int Cout, ptr_t st) {
    crop_mirror_norm(P(x), in_kind, P(mean), mean_mode, scale, P(cscale), P(out), out_bf16, P(offs), P(flips), N, H, W, C, ch, cw, Cout, S(st)); });

  // ---------------------------------------------------------------- fp32-storage layer kernels (tf32 precision mode)
  m.def("lrn_fwd_f32", [](ptr_t x, ptr_t y, long long rows, int C, int n, float k, float alpha, float beta, ptr_t st) {
    lrn_fwd_f32(P(x), P(y), rows, C, n, k, alpha, beta, S(st)); });
  m.def("lrn_bwd_f32", [](ptr_t x, ptr_t dy, ptr_t dx, long long rows, int C, int n, float k, float alpha, float beta, ptr_t st) {
    lrn_bwd_f32(P(x), P(dy), P(dx), rows, C, n, k, alpha, beta, S(st)); });
  m.def("pool_fwd_f32", [](ptr_t x, ptr_t y, ptr_t arg, int N, int H, int W, int C, int Ho, int Wo, int k, int s, int p, int is_max, ptr_t st) {
    pool_fwd_f32(P(x), P(y), P(arg), N, H, W, C, Ho, Wo, k, s, p, is_max, S(st)); });
  m.def("pool_bwd_f32", [](ptr_t dy, ptr_t arg, ptr_t dx, int N, int H, int W, int C, int Ho, int Wo, int k, int s, int p, int is_max, ptr_t st) {
    pool_bwd_f32(P(dy), P(arg), P(dx), N, H, W, C, Ho, Wo, k, s, p, is_max, S(st)); });
  m.def("dropout_fwd_f32", [](ptr_t x, ptr_t y, ptr_t mask, long long n, float p, unsigned long long seed, int layer, ptr_t step, ptr_t st) {
    dropout_fwd_f32(P(x), P(y), P(mask), n, p, seed, layer, P(step), S(st)); });
  m.def("dropout_bwd_f32", [](ptr_t dy, ptr_t mask, ptr_t dx, long long n, ptr_t st) { dropout_bwd_f32(P(dy), P(mask), P(dx), n, S(st)); });
  m.def("softmax_xent_f32", [](ptr_t logits, ptr_t labels, ptr_t dlogits, ptr_t rowstat, ptr_t out3, int B, int C, float weight, ptr_t st) {
    softmax_xent_f32(P(logits), P(labels), P(dlogits), P(rowstat), P(out3), B, C, weight, S(st)); });
  m.def("relu_bias_bwd2_f32", [](ptr_t dy, ptr_t y, ptr_t dym, ptr_t db, ptr_t db1, int c_split, long long R, int C, long long ld, int relu, ptr_t st) {
    relu_bias_bwd2_f32(P(dy), P(y), P(dym), P(db), P(db1), c_split, R, C, ld, relu, S(st)); });
  m.def("bias_act_f32", [](ptr_t acc, ptr_t bias, ptr_t y, int R, int C, int relu, ptr_t st) { bias_act_f32(P(acc), P(bias), P(y), R, C, relu, S(st)); });
  m.def("im2col_f32", [](ptr_t x, ptr_t col, int N, int H, int W, int Ctot, int c_off, int Cg, int KH, int KW, int Ho, int Wo, int s, int p,
                         long long ldcol, ptr_t st) { im2col_f32(P(x), P(col), N, H, W, Ctot, c_off, Cg, KH, KW, Ho, Wo, s, p, ldcol, S(st)); });
  m.def("col2im_f32", [](ptr_t dcol, ptr_t dx, int N, int H, int W, int Ctot, int c_off, int Cg, int KH, int KW, int Ho, int Wo, int s, int p,
                         long long ldcol, ptr_t st) { col2im_f32(P(dcol), P(dx), N, H, W, Ctot, c_off, Cg, KH, KW, Ho, Wo, s, p, ldcol, S(st)); });
  m.def("pad_rows_f32", [](ptr_t src, ptr_t dst, long long rows, int cols, long long src_ld, long long dst_ld, ptr_t st) {
    pad_rows_f32(P(src), P(dst), rows, cols, src_ld, dst_ld, S(st)); });
  m.def("space_to_depth_f32", [](ptr_t x, ptr_t y, int N, int H, int W, int C, int S, int Hs, int Ws, int Cp, int Pd, ptr_t st) {
    space_to_depth_f32(P(x), P(y), N, H, W, C, S, Hs, Ws, Cp, Pd, S_(st)); });
  m.def("s2d_filter_pack_f32", [](ptr_t src, ptr_t dst, int O, int KH, int KW, int C, int S, int KHs, int KWs, int Cp, ptr_t st) {
    s2d_filter_pack_f32(P(src), P(dst), O, KH, KW, C, S, KHs, KWs, Cp, S_(st)); });

  // ---------------------------------------------------------------- batch norm / residual
  m.def("bn_forward", [](ptr_t x, ptr_t res, ptr_t y, ptr_t gamma, ptr_t beta, ptr_t mean, ptr_t rstd, ptr_t run_mean, ptr_t run_var, ptr_t scratch,
                         long long R, int C, float momentum, float eps, int training, int relu, int f32, ptr_t st) {
    bn_forward(P(x), P(res), P(y), P(gamma), P(beta), P(mean), P(rstd), P(run_mean), P(run_var), P(scratch), R, C, momentum, eps, training, relu,
               f32, S(st)); });
  m.def("bn_backward", [](ptr_t x, ptr_t dy, ptr_t y, ptr_t dx, ptr_t dres, ptr_t gamma, ptr_t mean, ptr_t rstd, ptr_t dgamma, ptr_t dbeta,
                          ptr_t scratch, long long R, int C, int relu, int f32, ptr_t st) {
    bn_backward(P(x), P(dy), P(y), P(dx), P(dres), P(gamma), P(mean), P(rstd), P(dgamma), P(dbeta), P(scratch), R, C, relu, f32, S(st)); });
  m.def("add4_tensors", [](ptr_t a, ptr_t b, ptr_t c, ptr_t d, ptr_t y, long long n, int f32, ptr_t st) {
    add4_tensors(P(a), P(b), P(c), P(d), P(y), n, f32, S(st)); });
  m.def("add_tensors", [](ptr_t a, ptr_t b, ptr_t y, long long n, int f32, ptr_t st) { add_tensors(P(a), P(b), P(y), n, f32, S(st)); });

  // ---------------------------------------------------------------- recurrent / embedding
  m.def("lstm_cell_fwd", [](ptr_t gx, ptr_t gh, ptr_t c_prev, ptr_t h_prev, ptr_t mask, ptr_t act, ptr_t c_out, ptr_t h_out, int B, int H, int f32,
                            ptr_t st) { lstm_cell_fwd(P(gx), P(gh), P(c_prev), P(h_prev), P(mask), P(act), P(c_out), P(h_out), B, H, f32, S(st)); });
  m.def("lstm_cell_bwd", [](ptr_t dh_out, ptr_t dh_rec, ptr_t dh_pass_in, ptr_t dc_next, ptr_t act, ptr_t c, ptr_t c_prev, ptr_t mask, ptr_t dG,
                            ptr_t dc_prev, ptr_t dh_pass, int B, int H, int f32, ptr_t st) {
    lstm_cell_bwd(P(dh_out), P(dh_rec), P(dh_pass_in), P(dc_next), P(act), P(c), P(c_prev), P(mask), P(dG), P(dc_prev), P(dh_pass), B, H, f32, S(st)); });
  m.def("embedding_fwd", [](ptr_t ids, ptr_t W, ptr_t out, long long n, int D, int f32, ptr_t st) { embedding_fwd(P(ids), P(W), P(out), n, D, f32, S(st)); });
  m.def("embedding_bwd", [](ptr_t ids, ptr_t dout, ptr_t dW, long long n, int D, long long V, int f32, ptr_t st) {
    embedding_bwd(P(ids), P(dout), P(dW), n, D, V, f32, S(st)); });
  m.def("masked_mean_fwd", [](ptr_t h, ptr_t mask, ptr_t out, int Tn, int B, int H, int f32, ptr_t st) { masked_mean_fwd(P(h), P(mask), P(out), Tn, B, H, f32, S(st)); });
  m.def("masked_mean_bwd", [](ptr_t dout, ptr_t mask, ptr_t dh, int Tn, int B, int H, int f32, ptr_t st) { masked_mean_bwd(P(dout), P(mask), P(dh), Tn, B, H, f32, S(st)); });

  // ---------------------------------------------------------------- optimizer / legacy kernels
  m.def("sgd_flat", [](ptr_t W, ptr_t G, ptr_t U, ptr_t H, ptr_t block_group, std::vector<float> lr_mult, std::vector<float> wd,
                       std::vector<int> exch, ptr_t lr_ptr, float mu, int nesterov, float inv_k, long long lo, long long hi, int filter,
                       ptr_t st) {
    sgd_flat(P(W), P(G), P(U), P(H), P(block_group), make_table(lr_mult, wd, exch), P(lr_ptr), mu, nesterov, inv_k, lo, hi, filter, S(st)); });
  m.def("adam_flat", [](ptr_t W, ptr_t G, ptr_t M, ptr_t V, ptr_t H, ptr_t block_group, std::vector<float> lr_mult, std::vector<float> wd,
                        std::vector<int> exch, ptr_t lr_ptr, ptr_t step, float b1, float b2, float eps, long long lo, long long hi, ptr_t st,
                        float inv_k, int filter, int advance) {
    adam_flat(P(W), P(G), P(M), P(V), P(H), P(block_group), make_table(lr_mult, wd, exch), P(lr_ptr), P(step), b1, b2, eps, lo, hi, inv_k,
              filter, advance, S(st)); },
    py::arg("W"), py::arg("G"), py::arg("M"), py::arg("V"), py::arg("H"), py::arg("block_group"), py::arg("lr_mult"), py::arg("wd"),
    py::arg("exch"), py::arg("lr_ptr"), py::arg("step"), py::arg("b1"), py::arg("b2"), py::arg("eps"), py::arg("lo"), py::arg("hi"),
    py::arg("st"), py::arg("inv_k") = 1.f, py::arg("filter") = 0, py::arg("advance") = 1);
  m.def("adam_advance", [](ptr_t step, ptr_t st) { adam_advance(P(step), S(st)); });
  m.def("easgd_elastic", [](ptr_t w, ptr_t h, ptr_t center, float alpha, long long n, int max_blocks, ptr_t st, int lockfree) {
    easgd_elastic(P(w), P(h), P(center), alpha, n, max_blocks, lockfree, S(st)); },
    py::arg("w"), py::arg("h"), py::arg("center"), py::arg("alpha"), py::arg("n"), py::arg("max_blocks"), py::arg("st"), py::arg("lockfree") = 0);
  m.def("copy_flat", [](ptr_t dst, ptr_t dst_h, ptr_t src, long long n, int max_blocks, ptr_t st) {
    copy_flat(P(dst), P(dst_h), P(src), n, max_blocks, nullptr, S(st)); });
  m.def("gosgd_merge", [](ptr_t w, ptr_t h, ptr_t b, float a_self, float a_src, long long n, int max_blocks, ptr_t st) {
    gosgd_merge(P(w), P(h), P(b), a_self, a_src, n, max_blocks, S(st)); });
  m.def("bias_act_cast", [](ptr_t acc, ptr_t bias, ptr_t y, int R, int C, int relu, ptr_t st) { bias_act_cast(P(acc), P(bias), P(y), R, C, relu, S(st)); });
  m.def("cast_flat", [](ptr_t src, ptr_t dst, long long n, int kind, ptr_t st) { cast_flat(P(src), P(dst), n, kind, S(st)); });
  m.def("sum_chunks", [](ptr_t src, ptr_t dst, long long chunk, int nchunks, int is_half, ptr_t st) {
    sum_chunks(P(src), P(dst), chunk, nchunks, is_half, S(st)); });
  m.def("vecadd", [](ptr_t cur, ptr_t tmp, long long n, int is_half, ptr_t st) { vecadd(P(cur), P(tmp), n, is_half, S(st)); });

  // ---------------------------------------------------------------- peer memory + fused collectives
  py::class_<PyComm, std::shared_ptr<PyComm>>(m, "PeerArena")
      .def(py::init([](int rank, int world, int device, unsigned long long bytes, const std::string& job, bool force_ipc) {
        auto c = std::make_shared<PyComm>();
        c->pa.reset(new PeerArena(rank, world, device, (size_t)bytes, job, force_ipc));
        return c;
      }), py::arg("rank"), py::arg("world"), py::arg("device"), py::arg("bytes"), py::arg("job"), py::arg("force_ipc") = false)
      .def("send_handles_to", [](PyComm& c, int peer) { py::gil_scoped_release r; c.pa->send_handles_to(peer); })
      .def("recv_handles", [](PyComm& c) { py::gil_scoped_release r; c.pa->recv_handles(); })
      .def("ipc_handles", [](PyComm& c) { return py::bytes(c.pa->ipc_handles()); })
      .def("ipc_open", [](PyComm& c, int peer, const std::string& h) { c.pa->ipc_open(peer, h); })
      .def("multicast_supported", [](PyComm& c) { return c.pa->multicast_supported(); })
      .def("mc_create_and_send", [](PyComm& c) { py::gil_scoped_release r; c.pa->mc_create_and_send(); })
      .def("mc_recv", [](PyComm& c) { py::gil_scoped_release r; c.pa->mc_recv(); })
      .def("mc_add_device", [](PyComm& c) { c.pa->mc_add_device(); })
      .def("mc_bind_and_map", [](PyComm& c) { c.pa->mc_bind_and_map(); })
      .def("arena_ptr", [](PyComm& c, int p) { return (ptr_t)c.pa->arena_ptr(p); })
      .def("sig_ptr", [](PyComm& c, int p) { return (ptr_t)c.pa->sig_ptr(p); })
      .def("mc_ptr", [](PyComm& c) { return (ptr_t)c.pa->mc_ptr(); })
      .def("arena_bytes", [](PyComm& c) { return (unsigned long long)c.pa->arena_bytes(); })
      .def("mode", [](PyComm& c) { return c.pa->mode(); })
      .def("vmm_error", [](PyComm& c) { return c.pa->vmm_error(); })
      .def("device_barrier", [](PyComm& c, ptr_t st) { device_barrier(c.pa->ctx(), S(st)); })
      .def("ticket_acquire", [](PyComm& c, int owner, ptr_t local_state, ptr_t st) { ticket_acquire(c.pa->ctx(), owner, P(local_state), S(st)); })
      .def("ticket_release", [](PyComm& c, int owner, ptr_t local_state, ptr_t st) { ticket_release(c.pa->ctx(), owner, P(local_state), S(st)); })
      .def("gosgd_push", [](PyComm& c, ptr_t state, int dest, long long w_off, long long snap_off, long long n, int max_blocks, ptr_t st) {
             gosgd_push(c.pa->ctx(), P(state), dest, w_off, snap_off, n, max_blocks, S(st)); })
      .def("gosgd_poll_merge", [](PyComm& c, ptr_t state, long long w_off, long long h_off, long long snap_off, long long n, int max_blocks,
                                  ptr_t st) { gosgd_poll_merge(c.pa->ctx(), P(state), w_off, h_off, snap_off, n, max_blocks, S(st)); })
      .def("proto_words_offset", [](PyComm&) { return (long long)((size_t)kMaxCommBlocks * kMaxRanks + kMaxCommBlocks) * 4; })
      .def("fused_allreduce_sgd",
           [](PyComm& c, long long w_off, long long g_off, long long u_off, long long h_off, long long wire_off, ptr_t block_group,
              std::vector<float> lr_mult, std::vector<float> wd, std::vector<int> exch, ptr_t lr_ptr, float mu, int nesterov, float inv_k,
              long long lo, long long hi, int wire16, int algo, int max_blocks, ptr_t st, int pre_reduced, int push_master) {
             FusedArgs a;
             a.pre_reduced = pre_reduced;
             a.push_master = push_master;
             a.ctx = c.pa->ctx();
             a.w_off = w_off; a.g_off = g_off; a.u_off = u_off; a.h_off = h_off; a.wire_off = wire_off;
             a.block_group = (const uint8_t*)P(block_group);
             a.tab = make_table(lr_mult, wd, exch);
             a.lr_ptr = (const float*)P(lr_ptr); a.mu = mu; a.nesterov = nesterov; a.inv_k = inv_k; a.lo = lo; a.hi = hi; a.wire16 = wire16;
             fused_allreduce_sgd(a, algo, max_blocks, S(st));
           }, py::arg("w_off"), py::arg("g_off"), py::arg("u_off"), py::arg("h_off"), py::arg("wire_off"), py::arg("block_group"),
           py::arg("lr_mult"), py::arg("wd"), py::arg("exch"), py::arg("lr_ptr"), py::arg("mu"), py::arg("nesterov"), py::arg("inv_k"),
           py::arg("lo"), py::arg("hi"), py::arg("wire16"), py::arg("algo"), py::arg("max_blocks"), py::arg("st"), py::arg("pre_reduced") = 0,
           py::arg("push_master") = 1)
      .def("fused_allreduce_adam",
           [](PyComm& c, long long w_off, long long g_off, long long m_off, long long v_off, long long h_off, long long wire_off,
              ptr_t block_group, std::vector<float> lr_mult, std::vector<float> wd, std::vector<int> exch, ptr_t lr_ptr, ptr_t step,
              float b1, float b2, float eps, float inv_k, long long lo, long long hi, int wire16, int algo, int max_blocks, ptr_t st,
              int push_master) {
             FusedArgs a;
             a.pre_reduced = 0;
             a.push_master = push_master;
             a.ctx = c.pa->ctx();
             a.w_off = w_off; a.g_off = g_off; a.u_off = m_off; a.h_off = h_off; a.wire_off = wire_off;
             a.block_group = (const uint8_t*)P(block_group);
             a.tab = make_table(lr_mult, wd, exch);
             a.lr_ptr = (const float*)P(lr_ptr); a.mu = 0.f; a.nesterov = 0; a.inv_k = inv_k; a.lo = lo; a.hi = hi; a.wire16 = wire16;
             a.adam.v_off = v_off; a.adam.b1 = b1; a.adam.b2 = b2; a.adam.eps = eps;
             a.adam.step = (const unsigned long long*)P(step);
             fused_allreduce_adam(a, algo, max_blocks, S(st));
           }, py::arg("w_off"), py::arg("g_off"), py::arg("m_off"), py::arg("v_off"), py::arg("h_off"), py::arg("wire_off"),
           py::arg("block_group"), py::arg("lr_mult"), py::arg("wd"), py::arg("exch"), py::arg("lr_ptr"), py::arg("step"), py::arg("b1"),
           py::arg("b2"), py::arg("eps"), py::arg("inv_k"), py::arg("lo"), py::arg("hi"), py::arg("wire16"), py::arg("algo"),
           py::arg("max_blocks"), py::arg("st"), py::arg("push_master") = 1)
      .def("push_region_slices",
           [](PyComm& c, long long off, ptr_t block_group, std::vector<float> lr_mult, std::vector<float> wd, std::vector<int> exch,
              long long lo, long long hi, int max_blocks, ptr_t st) {
             FusedArgs a;
             a.pre_reduced = 0; a.ctx = c.pa->ctx();
             a.w_off = a.g_off = a.u_off = a.wire_off = 0; a.h_off = -1;
             a.block_group = (const uint8_t*)P(block_group);
             a.tab = make_table(lr_mult, wd, exch);
             a.lr_ptr = nullptr; a.mu = 0.f; a.nesterov = 0; a.inv_k = 1.f; a.lo = lo; a.hi = hi; a.wire16 = 0;
             push_region_slices(a, off, max_blocks, S(st));
           })
      .def("configure_gemm_rs", [](PyComm& c, long long g_off) {
             // peer views of the gradient region for the reduce-scatter GEMM epilogue
             const CommCtx x = c.pa->ctx();
             const void* peers[kMaxRanks];
             for (int p = 0; p < x.world; ++p) peers[p] = reinterpret_cast<const char*>(x.arena[p]) + g_off;
             gemm_rs_configure(x.world, peers, peers[x.rank]);
           })
      .def("allreduce_flat",
           [](PyComm& c, long long src_off, long long dst_off, long long h_off, ptr_t block_group, std::vector<float> lr_mult,
              std::vector<float> wd, std::vector<int> exch, float scale, long long lo, long long hi, int skip_local, int algo,
              int max_blocks, ptr_t st) {
             ReduceArgs a;
             a.ctx = c.pa->ctx();
             a.src_off = src_off; a.dst_off = dst_off; a.h_off = h_off;
             a.block_group = (const uint8_t*)P(block_group);
             a.tab = make_table(lr_mult, wd, exch);
             a.scale = scale; a.lo = lo; a.hi = hi; a.skip_local_groups = skip_local;
             allreduce_flat(a, algo, max_blocks, S(st));
           });
}
