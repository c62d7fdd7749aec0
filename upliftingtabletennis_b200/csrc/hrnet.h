// HRNet executor internals shared between hrnet.cu (plan + SIMT kernels) and conv_umma.cu (tcgen05 path).
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "ttk_internal.h"

struct TtkConv {
  std::string name, bn;
  int cin, cout, k, stride;     // logical sizes (reference)
  int cin_p, cout_p;            // padded to multiples of 16
  bool set = false;
  float* w_f32 = nullptr;       // device, [k*k][cin_p][cout_p] float32 (SIMT path)
  float* w_bfr = nullptr;       // device, same layout, values rounded to bf16 (SIMT path on bf16 storage)
  float* w_hfr = nullptr;       // device, same layout, values rounded to fp16 (SIMT path on fp16 storage)
  float* bias = nullptr;        // device, [cout_p] float32
  __nv_bfloat16* w_umma = nullptr;  // device, tcgen05 B-operand image, bf16 (see ttk_conv_umma_pack)
  __half* w_umma_f16 = nullptr;     // device, the same image in fp16
  float* w_umma32 = nullptr;        // device, tcgen05 B-operand image for kind::tf32: fp32 containers, values rounded to TF32
  float* w_x3 = nullptr;            // device, 3xTF32 B-operand images: W_hi = tf32(w), then W_lo = w - W_hi, in the x3 layout
  std::vector<float> w_host, b_host; // folded weights as set by the host (used to build fused variants)
};

struct TtkTensor {
  int c;        // channels (padded)
  int shift;    // resolution = (H >> shift, W >> shift)
  int first, last;   // op indices of first write / last read (liveness)
  size_t offset;     // byte offset in the workspace (per forward plan)
};

enum { OP_CONV = 0, OP_SUM = 1, OP_FINAL = 2 };

struct TtkOp {
  int type;
  int conv = -1;
  int in = -1, out = -1;
  int nres = 0;
  int res[3] = {-1, -1, -1};   // residual / summand tensors
  bool relu = false;
};

struct ConvLaunch {
  const void* in;
  void* out;
  const void* res[3];
  int res_shift[3];
  int nres;
  int n, hin, win, hout, wout;
  int cin, cout;       // padded
  int relu;
  const void* in2 = nullptr;   // second input of a K-concatenated 1x1 convolution (fused projection shortcut)
  int cin2 = 0;
};

struct ttk_hrnet {
  int in_ch, out_ch, out_first, out_count;
  int device = -1;              // device of the packed weights (ttk_bind_device)
  std::vector<TtkConv> convs;
  std::vector<TtkTensor> tensors;
  std::vector<TtkOp> ops;
  int input_tensor = -1;
  int dead_ops = 0;             // ops of the reference's graph whose outputs nothing reads (removed from the plan)
  int subbatch = 16;
  int launches = 0;
  int force_simt = 0;           // 16-bit / TF32 storage through the SIMT kernels (debug / cross-check of the tcgen05 path)
  // final 1x1 conv weights: [out_count][16] + bias[out_count], float32 device
  float* final_w = nullptr;
  float* final_b = nullptr;
  // bottleneck fusion: conv3 (1x1, 32->128) and the projection shortcut (1x1, 64->128) as ONE K-concatenated GEMM
  int dual_ds_op = -1, dual_c3_op = -1;
  void* w_dual = nullptr;           // bf16 image
  void* w_dual_f16 = nullptr;       // fp16 image
  void* w_dual32 = nullptr;         // TF32 image
  float* bias_dual = nullptr;
  bool dual_ready = false;
  int use_dual = 1;
  int cur_esz = 0;              // element size of the tensor-core path the running forward uses (0: SIMT), for the profile records
  bool cur_x3 = false;          // ... and whether it is the 3xTF32 path
  int use_block_fusion = 1;     // BasicBlocks as one kernel (block_umma.cu): the 16- and 32-channel branches in bf16 / fp16, the 16-channel branch
                                // in TF32.  Round 1 measured break-even in bf16 because the thin MMAs were issue bound (16 instructions per
                                // tcgen05.mma); with the warp-uniform issue loop the fused blocks win (DESIGN.md section 4.2)
  // optional per-launch timing (ttk_hrnet_set_profile): events bracket every launch on the caller's stream
  int profile = 0;
  std::vector<cudaEvent_t> events;     // pool, events[i] precedes launch i
  struct Rec { int op; int n; double flops, bytes; bool simt_fallback = false; };
  std::vector<Rec> recs;
};

// conv_umma.cu: implicit-GEMM convolution on tcgen05/TMEM fed by TMA.  esz = bytes per activation element: 2 = bf16 (kind::f16; f16:
// IEEE fp16 instead), 4 = fp32 activations multiplied as TF32 (kind::tf32); x3 (esz 4 only): every product as three TF32 products of
// split operands.  Returns TTK_ERR_UNSUPPORTED when the shape has no tensor-core kernel (caller falls back to SIMT on the same storage
// type).
int ttk_conv_umma_launch(const TtkConv& cv, const ConvLaunch& a, cudaStream_t st, int esz = 2, bool x3 = false, bool f16 = false);
int ttk_conv_umma_pack(TtkConv& cv, const float* w_host);
// out = relu(W3 a + Wd x + bias): a.in = a (32 ch), a.in2 = x (64 ch); returns TTK_ERR_UNSUPPORTED if the driver rejects the maps
int ttk_conv_umma_launch_dual(const void* w_dual, const float* bias_dual, const ConvLaunch& a, cudaStream_t st, int esz = 2, bool f16 = false);
void ttk_conv_umma_pack_dual(const float* w3, const float* wd, int esz, std::vector<uint8_t>& out, bool f16 = false);

// block_umma.cu: y = relu(conv2(relu(conv1(x))) + x) for the 3x3 stride-1 pairs of a BasicBlock with 16 or 32 (padded) channels.
int ttk_block_umma_launch(const TtkConv& c1, const TtkConv& c2, const void* x, void* y, int n, int h, int w, cudaStream_t st, int esz = 2,
                          bool f16 = false);
