// Internal (non-ABI) declarations shared by the stemgnn_b200 translation units.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace sg {

// ---- TMA tensor maps (tensor_map.cu) ------------------------------------------------------------------------------------
// 2-D tiled map of a row-major `rows` x `cols` tensor with row pitch `pitch_bytes` (anything outside reads as zero), box =
// box_rows x box_cols elements.  false when the driver has no encoder or rejects the map (callers then return -1).
bool make_tensor_map_2d(CUtensorMap* map, CUtensorMapDataType dtype, const void* base, uint64_t rows, uint64_t cols,
                        uint64_t pitch_bytes, uint32_t box_rows, uint32_t box_cols, CUtensorMapSwizzle swizzle);

// ---- GRU (gru.cu) --------------------------------------------------------------------------------
struct GruArgs {
  const float* xs;     // (N, B, W) sequence-major input
  const float* w_ih;   // (3N, W)
  const float* w_hh;   // (3N, N)
  const float* b_ih;   // (3N)
  const float* b_hh;   // (3N)
  const float* wk;     // (N)  weight_key   (indexed by step)
  const float* wq;     // (N)  weight_query
  float* key;          // (B, N)
  float* query;        // (B, N)
  float* h_all;        // (N, B, N) or null
  float* gi;           // (N, B, 3N) scratch: input projection of every step
  float* g_r; float* g_z; float* g_n; float* g_hn;   // (N, B, N) gate values saved for BPTT (or null)
  int B, N, W;
  int xrep;            // measurement knob: redundant DSMEM sends per step (1 = normal)
  int tc_reuse;        // 1: the packed fp16 hi/lo W_hh images at the start of `gi` are still valid (frozen weights)
};
// tensor-core recurrence (gru_tc.cu): 0 launched, -1 outside its envelope (caller falls back), >0 error
int gru_tc_forward(const GruArgs& a, uint8_t* img, int reuse_img, cudaStream_t st);
size_t gru_tc_image_bytes(int N, int W);
const char* gru_tc_kernel_name();
// per-step tensor-core path for N beyond the cluster envelope (gru_step_tc.cu): W_hh images streamed from L2 by TMA
size_t gru_step_tc_scratch_bytes(int B, int N);
int gru_step_tc_forward(const GruArgs& a, uint8_t* scratch, size_t scratch_bytes, int reuse_img, cudaStream_t st);
int gru_keyquery_forward(const GruArgs& a, int path, float* scratch, cudaStream_t st);
// persistent-cluster BPTT (one launch); -1 = unsupported here, use the per-step kernels
int gru_bwd_cluster(const float* w_hh, const float* wk, const float* wq, const float* d_key,
                    const float* d_query, const float* h_all, const float* g_r, const float* g_z,
                    const float* g_n, const float* g_hn, float* dgh, float* dgi, int B, int N,
                    cudaStream_t st);

// ---- attention / Laplacian (latent.cu) ----------------------------------------------------------------
struct AttnArgs {
  const float* key;      // (B,N)
  const float* query;    // (B,N)
  const float* qmax;     // (B)
  float* a_raw;          // (N,N) batch mean of (dropped-out) softmax rows, NOT symmetrised
  float* deg;            // (N)   row sums of a_raw (base_model.py:141)
  float* row_m;          // (B,N) softmax row max   (saved for backward; may be null)
  float* row_zinv;       // (B,N) 1 / softmax denominator
  const uint8_t* mask;   // optional explicit keep mask (B,N,N)
  uint64_t seed, offset;
  const unsigned long long* offset_dev;   // optional device counter added to `offset` (graph replays)
  float alpha, p;
  int use_dropout;       // 0: eval
  int B, N;
};
// x_pad (optional): (B*W, ld_pad) copy of x with a TMA-able row pitch (ld_pad % 4 == 0), operand of the tcgen05 GFT
int launch_prep_layouts(const float* x, float* xs, float* x_bnw, int B, int W, int N, cudaStream_t st,
                        float* x_pad = nullptr, int ld_pad = 0);
int launch_attention(const AttnArgs& a, float* qmax, cudaStream_t st);
// L_pad (optional): row i of mul_L[1] is also written to row 3*i of L_pad (pitch ld_pad): interleaved Chebyshev stack
int launch_laplacian(const float* a_raw, const float* deg, float* attention, float* mul_L, int N,
                     cudaStream_t st, float* L_pad = nullptr, int ld_pad = 0);

// ---- fused Laplacian + Jacobi eigensolver (eig.cu), opt-in graph mode ---------------------------------------------------
int laplacian_eig(const float* a_raw, const float* deg, int N, float* lambda, float* U, int* info, int max_sweeps,
                  float tol, cudaStream_t st);
int eig_poly_stack(const float* lambda, const float* U, int N, float* scratch, float* mul_L, cudaStream_t st);

// ---- spectral block helpers (spectral.cu) -----------------------------------------------------------
struct HeadArgs {
  const float* pre; int ldp;
  const float* x_bnw;          // (R, W) block input
  const float* bf; const float* wfr; const float* bfr;
  const float* bb; const float* wsc; const float* bsc;   // null for block 1
  float* forecast;             // (R, W)
  float* backcast_bnw;         // (R, W)    or null
  float* backcast_bwn;         // (B, W, N) or null
  float* save_fs;              // (R, T) or null (training)
  int R, N, T, W;
};
int launch_gft(const float* mul_L, const float* x_bwn, float* G, float* skbuf, int B, int N, int W,
               cudaStream_t st, unsigned short* g_img = nullptr, int ldh = 0, int bf16 = 0, int* g_ready = nullptr);
int launch_block_head(const HeadArgs& a, cudaStream_t st);
int launch_model_head(const float* f0, const float* f1, const float* w0, const float* b0,
                      const float* w2, const float* b2, float* out, int B, int N, int W, int H,
                      cudaStream_t st);
int launch_fold_in(const float* w_in, float* w_out, int d, int W, int chain, int kfirst, int nk,
                   cudaStream_t st);
int launch_irfft_table(float* ic, int T, cudaStream_t st);
int launch_irfft_rows(const float* act3, const float* ic, float* iffted, int B, int N, int T,
                      cudaStream_t st);
int launch_gfted_to_rows(const float* gfted, float* G4, int B, int N, int W, cudaStream_t st);

// ---- tcgen05 TF32 GLU GEMM (glu_tc.cu): returns 0 ok, -1 unsupported shape/device, >0 error ----------
int glu_gemm_tc(int M, int N, int K, const float* A, int lda, const float* Wl, const float* bl,
                const float* Wr, const float* br, float* out, int ldo, float* save_l, float* save_s,
                int lds, cudaStream_t st);

// fused 3-layer GLU chain on tcgen05 (glu_tc.cu); -1 = unsupported shape (use the per-layer kernels)
int glu_chain_tc(int M, int N, int K1, const float* G, int ldg, const float* const w[3][2],
                 const float* const bias[3][2], float* out3, int ldo3, float* const act[2],
                 float* const save_l[3], float* const save_s[3], cudaStream_t st);

// fused 3-layer GLU chain on tcgen05 kind::f16 (glu_h.cu): mode 0 = fp16 hi/lo split operands (fp32 parity), 1 = bf16
size_t glu_chain_h_scratch_halves(int M, int N, int K1);
int glu_chain_h(int mode, int M, int N, int K1, const float* G, int ldg, const float* const w[3][2],
                const float* const bias[3][2], float* out3, int ldo3, float* const act[2], float* const save_l[3],
                float* const save_s[3], unsigned short* scratch, int reuse_w, const unsigned short* g_shared,
                cudaStream_t st, int g_ready = 0);

// generic tcgen05 TF32 GEMM (glu_tc.cu): C0/C1 (+)= alpha A[M,K] B[N,K]^T; rows m >= msplit go to C1.
// split_ops: 1 = 3xTF32 split operands (spec_tc.cu, fp32-level), 0 = one truncated-TF32 pass, -1 = default (split unless
// STEMGNN_TC_NOSPLIT is set)
int tc_gemm(int M, int N, int K, float alpha, const float* A, int lda, const float* B, int ldb, int n_rows_b,
            float* C0, float* C1, int msplit, int ldc, int n_store, int atomic, int splits, cudaStream_t st,
            int split_ops = -1);

// ---- spectral-block GEMMs on tcgen05 with 3xTF32 split operands (spec_tc.cu): 0 ok, -1 unsupported, >0 error -------------
// padded (TMA-able) copy with an optional row permutation (spec_tc.cu); row_mul = 3, stack_n = N: the three stacked Chebyshev
// terms interleaved as row n*3 + k'
int launch_pad_rows(const float* src, long long rows, int cols, int ld_src, float* dst, int ld_dst, cudaStream_t st,
                    int row_mul = 1, int row_add = 0, int stack_n = 0);
int tc3_gemm(int M, int N, int K, float alpha, const float* A, int lda, const float* B, int ldb, int n_rows_b, float* C0,
             float* C1, int msplit, int ldc, int n_store, int atomic, int splits, int split_ops, cudaStream_t st);
int gft_tc(const float* mul_Lp, int ldl, const float* xp, int ldx, float* G, unsigned short* g_img, int ldh, int bf16,
           int B, int N, int W, int split_ops, cudaStream_t st);
int out_head_tc(const float* act3, int K, const float* woutT, int PWp, const HeadArgs& h, float* bc_pad, int ld_pad,
                int split_ops, cudaStream_t st);

// ---- workspace ---------------------------------------------------------------------------------------
struct BlockWs {
  float* G;        // (R, 3W | 4W) graph-Fourier rows
  float* w1f;      // [chain][side](d, ncol) DFT-folded first-layer weights
  float* ic;       // [2](T,T) inverse real DFT table
  float* ri;       // [2](4T, T) irfft o weight[k]
  float* wout;     // woutT (round16(T+W), 8T): folded output map, K-major for the tensor-core GEMM
  float* act1;     // [chain](R, d)
  float* act2;     // [chain](R, d)
  float* act3;     // (R, 2d) = [real3 | imag3]
  float* pre;      // (R, T+W)
  float* forecast; // (R, W)
  float* bc_bnw;   // (R, W) backcast, block-input layout
  float* bc_bwn;   // (B, W, N) backcast, GFT operand layout
  float* bc_pad;   // (B*W, pad4(N)) the same with a TMA-able row pitch (operand of the tcgen05 GFT of the next block)
  float* save_l[6]; float* save_s[6];   // training: GLU left pre-activation / gate per GLU index
  float* fs;       // training: forecast_source (R, T)
  float* hscratch[2];   // per chain: 16-bit operand images of the kind::f16 GLU chain (G hi/lo + weight hi/lo)
};
// scratch of the backward pass (training workspaces only)
struct BwdWs {
  float *h_fsum, *h_act, *h_dhj, *h_dout, *d_fsum;      // model head
  float *d_pre, *negdz, *d_act3, *d_wout, *d_ri, *d_w1f, *dlr, *d_act[2], *d_G, *d_Gp;   // block (reused)
  float *dlrT, *inT, *wsT;   // K-major operands of the tcgen05 backward GEMMs: (2d, R), (d, R), (d, 2d)
  float *d_bc, *d_x0, *d_mul_L, *dAsym, *ddeg, *dA, *dots, *d_key, *d_query;
  float *dgh, *dh[2], *d_xs;
  float *dghT, *hT;          // (3N, S*B) and (N, S*B): K-major operands of the tensor-core dW_hh GEMM
};
struct Workspace {
  float *xs, *x_bnw, *key, *query, *qmax, *a_raw, *deg, *mul_L, *attention, *gru_scratch, *gi;
  float* skbuf;    // split-K partial products (8 x max(N*N, 3N*B*W) floats)
  float *mul_Lp, *x_pad;   // (3N, pad4(N)): row n*3 + k' = mul_L[k'+1][n][:], and (B*W, pad4(N)) = x; TMA-able row pitches
  float *row_m, *row_zinv, *h_all, *g_r, *g_z, *g_n, *g_hn;
  float *eig_lambda, *eig_U, *eig_S;   // eig graph mode: eigenvalues (n), eigenvectors (n,n), scaled copy (N,n)
  int* eig_info;
  BwdWs bwd;
  BlockWs blk[STEMGNN_MAX_STACK];
  size_t floats;
};
Workspace carve_workspace(const stemgnn_dims_t& dm, int training, float* base);

int model_backward(const stemgnn_dims_t* dims, const stemgnn_params_t* params,
                   const stemgnn_fwd_opts_t* opts, const float* x, const float* d_forecast,
                   const float* d_attention, const stemgnn_grads_t* grads, float* d_x,
                   void* workspace, size_t workspace_bytes, cudaStream_t st);

}  // namespace sg
