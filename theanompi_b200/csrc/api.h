// Host-visible API of the sm_100a extension (implemented in the .cu / .cpp files of this directory).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"

namespace tmpi {

constexpr int kMaxRanks = 8;
constexpr int kMaxCommBlocks = 1024;     // signal-pad rows

struct CommCtx {
  void* arena[kMaxRanks];                // base of rank p's arena as mapped in THIS process
  uint32_t* sig[kMaxRanks];              // signal pad of rank p: uint32 [kMaxCommBlocks][kMaxRanks]
  uint32_t* epoch;                       // local: per-block barrier epoch counters [kMaxCommBlocks]
  void* mc_arena;                        // multicast mapping of the arena (NVLS) or nullptr
  int rank, world;
  long long spin_limit;                  // clock64 cycles a flag barrier may spin before it traps (TMPI_BARRIER_TIMEOUT_S)
};

struct FusedArgs {
  CommCtx ctx;
  long long w_off, g_off, u_off, h_off, wire_off;   // byte offsets of the regions inside the arena (h_off < 0: no shadow)
  const uint8_t* block_group;
  GroupTable tab;
  const float* lr_ptr;                               // device scalar (CUDA-graph friendly)
  float mu;
  int nesterov;
  float inv_k;
  long long lo, hi;                                  // element range, multiples of kArenaBlock
  int wire16;                                        // gradients travel as bf16 (cast into the wire region first)
  int pre_reduced;                                   // the range's gradients were already reduce-scattered into their owner's G by the
                                                     // wgrad GEMM epilogues (gemm_rs_*): skip the gather, zero G after use
  int push_master = 1;                               // two-shot: 1 = push the updated fp32 master slice AND the bf16 shadow to every peer;
                                                     // 0 = owner keeps the master of WEIGHT blocks (group 0): peers receive only their bf16
                                                     // compute shadow — a third of the all-gather bytes; bias blocks (read in fp32 by the
                                                     // forward pass) are always pushed; push_region_slices() re-synchronises W on demand
  struct Adam {                                      // fused_allreduce_adam only: the M moment lives in the U region (u_off)
    long long v_off = -1;                            // second moment region
    float b1 = 0.9f, b2 = 0.999f, eps = 1e-8f;
    const unsigned long long* step = nullptr;        // device bias-correction counter: steps taken so far, advanced once per step
  } adam;
};

struct ReduceArgs {
  CommCtx ctx;
  long long src_off, dst_off, h_off;     // h_off >= 0: also refresh the bf16 shadow from the result (weight averaging)
  const uint8_t* block_group;
  GroupTable tab;
  float scale;
  long long lo, hi;
  int skip_local_groups;                 // leave non-exchanged blocks untouched
};

// ---- gemm_tcgen05.cu
void gemm_set_debug(int flags);
void gemm_set_bulk(int mask);      // epilogue through the bulk copy engine: bit0 stores, bit1 split-K adds, bit2 reduce-scatter adds; -1 = env
// Reduce-scatter fused into the wgrad GEMM epilogue: register the peer views of the gradient region and the tensors whose
// fp32 GEMM output (C pointer inside [c_lo, c_hi)) must be red.add-ed into the OWNER rank's G instead of stored locally.
// Ownership = the two-shot exchange kernel's partition of the bucket [blo, blo + world * per) in 1024-element blocks.
void gemm_rs_configure(int world, const void* const* peer_g /*[world]*/, const void* local_g);
void gemm_rs_add_range(const void* c_lo, const void* c_hi, long long blo, long long per);
void gemm_rs_clear();
int gemm_plan_splits(int tiles, int num_kb, int sms);          // split-K factor the launcher would pick
int gemm_plan_tall(long long M, int nt, int out_bf16, int sms);   // 1 = 256-row CTA tiles   // bottleneck probe knobs of the tcgen05 GEMM (see Params::dbg)
void gemm_bf16(const void* A, const void* B, void* C, const float* bias, int M, int N, int K, long long lda, long long ldb,
               long long ldc, int a_mn, int b_mn, int out_bf16, int bias_mode, int relu, float alpha, int bn_hint, int splitk,
               cudaStream_t st, int tf32 = 0);     // tf32 = 1: fp32 operands / fp32 output through tcgen05 kind::tf32

void conv_fprop_bf16(const void* x, const void* w, void* y, const float* bias, int N, int H, int W, int Ctot, int c_off, int Cg, int KH,
                     int KW, int Ho, int Wo, int S, int P, int O, long long ldc, int relu, int out_bf16, int dgrad, cudaStream_t st, int tf32 = 0);
void conv_wgrad_bf16(const void* dy, const void* x, void* dw, int N, int H, int W, int Ctot, int c_off, int Cg, int KH, int KW, int Ho,
                     int Wo, int S, int P, int O, long long ldy, cudaStream_t st, int tf32 = 0);
// both groups of a 2-group convolution in one persistent launch (see gemm_tcgen05.cu)
void conv_fprop2_bf16(const void* x, const void* w0, const void* w1, void* y0, void* y1, const float* bias0, const float* bias1, int N, int H,
                      int W, int Ctot, int c_off0, int c_off1, int Cg, int KH, int KW, int Ho, int Wo, int S, int P, int O, long long ldc,
                      int relu, int out_bf16, int dgrad, cudaStream_t st, int tf32 = 0);
void conv_wgrad2_bf16(const void* dy0, const void* dy1, const void* x, void* dw0, void* dw1, int N, int H, int W, int Ctot, int c_off0,
                      int c_off1, int Cg, int KH, int KW, int Ho, int Wo, int S, int P, int O, long long ldy, cudaStream_t st, int tf32 = 0);

// ---- nn_kernels.cu
void space_to_depth(const void* x, void* y, int N, int H, int W, int C, int S, int Hs, int Ws, int Cp, int P, cudaStream_t st);
void s2d_filter(const void* src, void* dst, int O, int KH, int KW, int C, int S, int KHs, int KWs, int Cp, int dir, cudaStream_t st);
void conv_weight_flip(const void* w, void* wt, int O, int KH, int KW, int Cg, cudaStream_t st);
void lrn_fwd(const void* x, void* y, long long rows, int C, int n, float k, float alpha, float beta, cudaStream_t st);
void lrn_bwd(const void* x, const void* dy, void* dx, long long rows, int C, int n, float k, float alpha, float beta, cudaStream_t st);
void pool_fwd(const void* x, void* y, void* arg, int N, int H, int W, int C, int Ho, int Wo, int k, int s, int p, int is_max, cudaStream_t st);
void pool_bwd(const void* dy, const void* arg, void* dx, int N, int H, int W, int C, int Ho, int Wo, int k, int s, int p, int is_max, cudaStream_t st);
void dropout_fwd(const void* x, void* y, void* mask, long long n, float p_drop, unsigned long long seed, int layer, const void* step, cudaStream_t st);
void dropout_bwd(const void* dy, const void* mask, void* dx, long long n, cudaStream_t st);
void advance_step(void* step, cudaStream_t st);
void softmax_xent(const void* logits, const void* labels, void* dlogits, void* rowstat, void* out3, int B, int C, float weight, cudaStream_t st);
void relu_bias_bwd(const void* dy, const void* y, void* dym, void* db, long long R, int C, long long ld, int relu, cudaStream_t st);
void relu_bias_bwd2(const void* dy, const void* y, void* dym, void* db, void* db1, int c_split, long long R, int C, long long ld, int relu,
                    cudaStream_t st);
void maxpool_relu_bias_bwd(const void* dyp, const void* arg, const void* y, void* dym, void* db0, void* db1, int c_split, int N, int H,
                           int W, int C, int Ho, int Wo, int k, int s, int p, cudaStream_t st);
void im2col(const void* x, void* col, int N, int H, int W, int Ctot, int c_off, int Cg, int KH, int KW, int Ho, int Wo, int s, int p,
            long long ldcol, cudaStream_t st);
void col2im(const void* dcol, void* dx, int N, int H, int W, int Ctot, int c_off, int Cg, int KH, int KW, int Ho, int Wo, int s, int p,
            long long ldcol, cudaStream_t st);
void pad_rows(const void* src, void* dst, long long rows, int cols, long long src_ld, long long dst_ld, cudaStream_t st);
void transpose_bf16(const void* src, void* dst, int R, int C, cudaStream_t st);
void crop_mirror_norm(const void* x, int in_kind, const void* mean, int mean_mode, float scale, const void* cscale, void* out, int out_bf16, const void* offs,
                      const void* flips, int N, int H, int W, int C, int ch, int cw, int Cout, cudaStream_t st);

// ---- nn_kernels_f32.cu: fp32-storage variants for the tf32 precision mode (same semantics, C % 4 == 0)
void lrn_fwd_f32(const void* x, void* y, long long rows, int C, int n, float k, float alpha, float beta, cudaStream_t st);
void lrn_bwd_f32(const void* x, const void* dy, void* dx, long long rows, int C, int n, float k, float alpha, float beta, cudaStream_t st);
void pool_fwd_f32(const void* x, void* y, void* arg, int N, int H, int W, int C, int Ho, int Wo, int k, int s, int p, int is_max, cudaStream_t st);
void pool_bwd_f32(const void* dy, const void* arg, void* dx, int N, int H, int W, int C, int Ho, int Wo, int k, int s, int p, int is_max,
                  cudaStream_t st);
void dropout_fwd_f32(const void* x, void* y, void* mask, long long n, float p_drop, unsigned long long seed, int layer, const void* step,
                     cudaStream_t st);
void dropout_bwd_f32(const void* dy, const void* mask, void* dx, long long n, cudaStream_t st);
void softmax_xent_f32(const void* logits, const void* labels, void* dlogits, void* rowstat, void* out3, int B, int C, float weight, cudaStream_t st);
void relu_bias_bwd2_f32(const void* dy, const void* y, void* dym, void* db, void* db1, int c_split, long long R, int C, long long ld, int relu,
                        cudaStream_t st);
void bias_act_f32(const void* acc, const void* bias, void* y, int R, int C, int relu, cudaStream_t st);
void im2col_f32(const void* x, void* col, int N, int H, int W, int Ctot, int c_off, int Cg, int KH, int KW, int Ho, int Wo, int s, int p,
                long long ldcol, cudaStream_t st);
void col2im_f32(const void* dcol, void* dx, int N, int H, int W, int Ctot, int c_off, int Cg, int KH, int KW, int Ho, int Wo, int s, int p,
                long long ldcol, cudaStream_t st);
void pad_rows_f32(const void* src, void* dst, long long rows, int cols, long long src_ld, long long dst_ld, cudaStream_t st);
void space_to_depth_f32(const void* x, void* y, int N, int H, int W, int C, int S, int Hs, int Ws, int Cp, int P, cudaStream_t st);
void s2d_filter_pack_f32(const void* src, void* dst, int O, int KH, int KW, int C, int S, int KHs, int KWs, int Cp, cudaStream_t st);

// ---- bn_kernels.cu: batch norm (+ residual)(+ ReLU) forward / backward, residual add  (f32: fp32 activations, else bf16)
void bn_forward(const void* x, const void* res, void* y, const void* gamma, const void* beta, void* mean, void* rstd, void* run_mean,
                void* run_var, void* scratch, long long R, int C, float momentum, float eps, int training, int relu, int f32, cudaStream_t st);
void bn_backward(const void* x, const void* dy, const void* y, void* dx, void* dres, const void* gamma, const void* mean, const void* rstd,
                 void* dgamma, void* dbeta, void* scratch, long long R, int C, int relu, int f32, cudaStream_t st);
void add_tensors(const void* a, const void* b, void* y, long long n, int f32, cudaStream_t st);
void add4_tensors(const void* a, const void* b, const void* c, const void* d, void* y, long long n, int f32, cudaStream_t st);

// ---- rnn_kernels.cu: LSTM cell fwd / bwd, embedding gather / scatter, masked mean pooling  (f32: fp32 activations, else bf16)
void lstm_cell_fwd(const void* gx, const void* gh, const void* c_prev, const void* h_prev, const void* mask, void* act, void* c_out, void* h_out,
                   int B, int H, int f32, cudaStream_t st);
void lstm_cell_bwd(const void* dh_out, const void* dh_rec, const void* dh_pass_in, const void* dc_next, const void* act, const void* c,
                   const void* c_prev, const void* mask, void* dG, void* dc_prev, void* dh_pass, int B, int H, int f32, cudaStream_t st);
void embedding_fwd(const void* ids, const void* W, void* out, long long n, int D, int f32, cudaStream_t st);
void embedding_bwd(const void* ids, const void* dout, void* dW, long long n, int D, long long V, int f32, cudaStream_t st);
void masked_mean_fwd(const void* h, const void* mask, void* out, int Tn, int B, int H, int f32, cudaStream_t st);
void masked_mean_bwd(const void* dout, const void* mask, void* dh, int Tn, int B, int H, int f32, cudaStream_t st);

// ---- comm_kernels.cu
void sgd_flat(void* W, const void* G, void* U, void* H, const void* block_group, const GroupTable& tab, const void* lr_ptr, float mu,
              int nesterov, float inv_k, long long lo, long long hi, int filter, cudaStream_t st);
// G: the gradient source (G or R region); filter as sgd_flat; advance = 1: bump the step counter after the update
void adam_flat(void* W, const void* G, void* M, void* V, void* H, const void* block_group, const GroupTable& tab, const void* lr_ptr, void* step,
               float b1, float b2, float eps, long long lo, long long hi, float inv_k, int filter, int advance, cudaStream_t st);
void adam_advance(void* step, cudaStream_t st);
void fused_allreduce_sgd(const FusedArgs& a, int algo, int max_blocks, cudaStream_t st);
void fused_allreduce_adam(const FusedArgs& a, int algo, int max_blocks, cudaStream_t st);
// every rank pushes the slice it owns in the two-shot partition of [lo, hi) of the fp32 region at byte offset `off` to all peers
void push_region_slices(const FusedArgs& a, long long off, int max_blocks, cudaStream_t st);
void allreduce_flat(const ReduceArgs& a, int algo, int max_blocks, cudaStream_t st);
void device_barrier(const CommCtx& c, cudaStream_t st);
void easgd_elastic(void* w, void* h, void* center, float alpha, long long n, int max_blocks, int lockfree, cudaStream_t st);
// device-side ticket lock in rank `owner`'s signal pad (EASGD: the center); local_state = >= 1 uint32 of local device memory
void ticket_acquire(const CommCtx& c, int owner, void* local_state, cudaStream_t st);
void ticket_release(const CommCtx& c, int owner, void* local_state, cudaStream_t st);
void copy_flat(void* dst, void* dst_h, const void* src, long long n, int max_blocks, const void* gate, cudaStream_t st);
// device-side gossip (GOSGD): state = 64 uint32 of local device memory, [0] holds the push-sum weight (float)
void gosgd_push(const CommCtx& c, void* state, int dest, long long w_off, long long snap_off, long long n, int max_blocks, cudaStream_t st);
void gosgd_poll_merge(const CommCtx& c, void* state, long long w_off, long long h_off, long long snap_off, long long n, int max_blocks,
                      cudaStream_t st);
void gosgd_merge(void* w, void* h, const void* b, float a_self, float a_src, long long n, int max_blocks, cudaStream_t st);
void bias_act_cast(const void* acc, const void* bias, void* y, int R, int C, int relu, cudaStream_t st);
void cast_flat(const void* src, void* dst, long long n, int kind, cudaStream_t st);
void sum_chunks(const void* src, void* dst, long long chunk, int nchunks, int is_half, cudaStream_t st);
void vecadd(void* cur, const void* tmp, long long n, int is_half, cudaStream_t st);

}  // namespace tmpi
