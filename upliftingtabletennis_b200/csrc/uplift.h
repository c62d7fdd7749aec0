// Uplifting transformer internals shared by uplift.cu (fp32 path) and uplift_tc.cu (bf16 tcgen05 path).
#pragma once
#include <string>
#include <vector>

#include "ttk_internal.h"

struct LayerW {
  const float *ln1w, *ln1b, *qkvw, *qkvb, *projw, *invf, *fc1w, *fc1b, *fc2w, *fc2b, *ln2w, *ln2b;
};
struct HeadW {
  const float *w1, *b1, *w2, *b2, *w3, *b3;
};


struct UpliftParam {
  std::string name;
  int numel;
  float* dev = nullptr;
  bool set = false;
};

struct ttk_uplift {
  int dim, heads, depth, skip;
  int device = -1;                 // device of the parameters (ttk_bind_device)
  std::vector<UpliftParam> params;
  LayerW* layers_dev = nullptr;    // [4 pos + (depth-4) temporal + 4 second]
  bool layers_ready = false;
  int launches = 0;
  // bf16 tensor-core path: every layer's [qkv(384) | proj(128) | fc1(128) | fc2(128)] x 128 weight rows, K-major
  __nv_bfloat16* wmat_dev = nullptr;
  bool wmat_ready = false;
  // fp32-class tensor-core path (3xTF32): hi / lo halves of every layer's [qkv | proj | fc1 | fc2] weight rows, fp32 [layers*768][128] each
  float *w3_hi = nullptr, *w3_lo = nullptr;
  bool w3_ready = false;
  int find(const std::string& n) const {
    for (size_t i = 0; i < params.size(); ++i)
      if (params[i].name == n) return (int)i;
    return -1;
  }
  const float* dev(const std::string& n) const { return params[find(n)].dev; }
};

struct UpliftIO {
  const float *ball, *table, *mask, *times;
  int batch, T;
  float *rot_out, *pos_out;
  float *X, *table_emb, *second_emb;     // workspace slices
  void* attn_rows;                       // bf16 [batch*T][128]: attention output of the ball tokens in the last table-token layer
  int mask_additive;                     // mask holds additive values ({-1e9, 0}) instead of {0, 1}
};

// gemm3_umma.cu: C = act(A' W^T + bias) (+ R) with K = 128, fp32 in / out, three TF32 tensor-core products per term (fp32-level results).
struct Gemm3Args {
  const float* A;          // [M][128]
  const float *W_hi, *W_lo; // [N][128]: W = W_hi + W_lo, W_hi = tf32(W) (split on the host, ttk_uplift3_prepare)
  const float* bias;       // [N] or null
  const float* R;          // [M][N] residual or null (may alias C)
  float* C;                // [M][N]
  int M, N;                // N a multiple of 128
  int relu;
  const float* ln_stats;   // [M][2] (mean, rstd) of A's rows: A' = LayerNorm(A) with ln_gamma / ln_beta [128]; null: A' = A
  const float *ln_gamma, *ln_beta;
  float* out_stats;        // [M][2] mean / rstd (eps 1e-5) of the rows of C, for the next LayerNorm (N = 128 only); null: not needed
};
int ttk_gemm3(const Gemm3Args& g, cudaStream_t st);
// uplift3.cu: the transformer on ttk_gemm3 + fp32 attention ("tf32x3" arithmetic class)
size_t ttk_uplift3_workspace_bytes(const ttk_uplift* h, int batch, int T);
int ttk_uplift3_prepare(ttk_uplift* h);
int ttk_uplift3_stage(ttk_uplift* h, int mode, const UpliftIO& io, void* ws, cudaStream_t st);

// uplift_tc.cu
int ttk_uplift_tc_prepare(ttk_uplift* h);
int ttk_uplift_tc_stage(ttk_uplift* h, int mode, const UpliftIO& io, cudaStream_t st);
