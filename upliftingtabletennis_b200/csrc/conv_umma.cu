// Implicit-GEMM convolution (3x3 stride 1/2, 1x1) on the 5th-generation tensor cores:
// tcgen05.mma with TMEM accumulators, operands staged by TMA, fused bias / residual / ReLU epilogue.
// Two arithmetic classes share the kernel (template parameter ESZ = bytes per activation element):
//   ESZ 2: 16-bit activations and weights, kind::f16: bf16, or IEEE fp16 with template parameter H = 1 (umma_prims.h: Fmt16 holds
//          everything that differs between the two; tiles, dispatch and fusion are the same);
//   ESZ 4: fp32 activations in HBM, kind::tf32 -- the class cuDNN uses for the reference's convolutions on a GPU (torch enables
//          TF32 for cuDNN by default).  The tensor map of the input has data type TFLOAT32, so TMA rounds every element to TF32
//          (nearest-even) on its way into shared memory; the weights are rounded once on the host; kind::tf32 ignores the low 13
//          mantissa bits, which are zero by then (tools/tf32_probe.cu, profiles/r02_tf32_probe.log).  Accumulation, bias,
//          residual adds and ReLU are fp32, and the stored activations are full fp32 like the reference's.
// Reference ops: the Conv2d + BatchNorm2d(eval) + ReLU (+ residual / fuse sum) groups of
// balldetection/models/wasb.py:35-105, :179-245, :383-416.
//
// Mapping (NHWC bf16 activations):
//   M = 128 consecutive output pixels of one image row, N = Cout (or a 64-wide slice of it), K = taps x Cin.
//   A CTA tile is R output rows x 128 pixels.  ONE TMA box brings the (R+2) x 130 pixel halo of a
//   K-chunk (<= 128 bytes of channels = one swizzled row of 32/64/128 bytes per pixel) into shared memory;
//   the 9 taps are NOT re-loaded: tap (ky,kx) of output row r is the same staged tile with the
//   matrix descriptor's start address moved by ((r+ky)*130 + kx) pixel rows.  tools/umma_probe.cu
//   established on a B200 that the 32/64/128-byte swizzles are applied to absolute shared-memory
//   address bits, so row-shifted descriptors (base_offset 0) read exactly what TMA wrote.
//   Stride 2: the input is addressed as four parity sub-grids (even/odd rows x even/odd columns, one
//   tensor map each, strides doubled); every tap then reads one sub-grid with unit pixel stride.
//   Image borders come for free from TMA's zero fill of out-of-bounds coordinates.
//   Vertical tap fusion (3x3 stride 1, Cout <= 64): an MMA costs at least the shared-memory read of its
//   128 x 16 A slab, so N = Cout = 16..64 leaves the tensor pipe mostly fetching.  The accumulators of a
//   tile's R output rows sit side by side in TMEM in REVERSE row order; input row yi and horizontal tap kx
//   are then multiplied ONCE with B = [W(ky=0,kx) | W(ky=1,kx) | W(ky=2,kx)] (N = 3 Cout), which lands in
//   the column blocks of output rows yi+1, yi, yi-1.  3(R+2) wide MMAs replace 9R narrow ones.
//   Accumulators are zeroed by the epilogue after it drains them, so every MMA accumulates.
// Roles (persistent CTA, static tile round-robin): warp 0 = TMA producer, warp 1 = MMA issuer
// (one elected thread), warps 2-5 = epilogue (TMEM -> registers -> bias/residual/ReLU -> bf16 -> global).
// Pipelines: smem full/empty ring over load units, double-buffered TMEM accumulators (tmem full/empty).
//
// 3xTF32 (template flag X3, fp32 elements): fp32-level products on the same tensor cores.  Every operand is split into two TF32
// numbers, x = x_hi + x_lo with x_hi = tf32(x) and x_lo = x - x_hi, and each MMA of the TF32 kernel becomes three into the same
// accumulator: A_hi W_hi + A_lo W_hi + A_hi W_lo (the dropped A_lo W_lo and kind::tf32 truncating the lo terms are 2^-22 of a product
// each, as in gemm3_umma.cu).  The input map has type FLOAT32, so TMA stages the raw values; four transform warps (6-9) split a
// staged unit element by element -- hi in place, lo into a second plane behind it with the same swizzle -- before the MMA warp may
// read it, so HBM traffic is that of the TF32 kernel.  W_hi and W_lo are split once by the host and both stay resident.  Both
// planes double the shared memory of the weights and of a stage, so the x3 tiles are sized separately (see kc_of / cout_tile).
#include <cuda.h>

#include <string.h>

#include <algorithm>
#include <vector>

#include "hrnet.h"
#include "umma_prims.h"

namespace {

using namespace umma;

constexpr int BW = 128;          // output pixels per tile row = MMA M
constexpr int THREADS = 192;         // TMA warp, MMA warp, 4 epilogue warps
constexpr int THREADS_HF = 320;      // horizontal tap fusion: 8 epilogue warps (two per TMEM lane quarter, alternating output rows)
constexpr int THREADS_X3 = 320;      // 3xTF32: TMA warp, MMA warp, 4 epilogue warps, 4 transform warps

constexpr int pow2_cols(int c) { return c <= 32 ? 32 : c <= 64 ? 64 : c <= 128 ? 128 : c <= 256 ? 256 : 512; }
constexpr int al1024(int b) { return (b + 1023) & ~1023; }

// KS: 1 or 3; S: stride 1 or 2 (3x3 only); CIN: padded input channels; COUT: output channels handled by one CTA
// (blockIdx.y selects the slice when the layer has more); R: output rows per tile; STAGES: smem ring depth;
// RB: reserve shared memory for TMA-staged residual tiles (double buffered with the accumulators);
// KCO: channels per K-chunk when not the default (a narrower chunk buys a taller tile for the same shared memory);
// X3: 3xTF32 (hi and lo planes of every staged unit and of the weights).
template <int KS, int S, int CIN, int COUT, int R, int STAGES, int RB, int KCO = 0, int ESZ = 2, int HF = 0, int X3 = 0>
struct Cfg {
  static constexpr int KCMAX = 128 / ESZ;                           // a swizzled smem row holds at most 128 bytes
  static constexpr int KC = KCO ? KCO : (CIN < KCMAX ? CIN : KCMAX);      // channels per K-chunk = one swizzled smem row
  static constexpr int NKC = CIN / KC;
  static constexpr int ROWB = KC * ESZ;
  static constexpr int KSTEPS = ROWB / 32;                          // MMAs per row: K = 16 bf16 or 8 tf32 = 32 bytes each
  static constexpr int PAD = KS / 2;
  static constexpr bool FUSE = KS == 3 && S == 1 && 3 * COUT <= 256;   // vertical tap fusion
  static constexpr int NPY = S == 2 ? 2 : 1;            // row-parity units per K-chunk
  static constexpr int NBOX = S == 2 ? 2 : 1;           // TMA boxes per unit (column parities)
  static constexpr int TW = S == 2 ? BW + 1 : (HF ? BW : BW + 2 * PAD);
  static constexpr int OUTW = HF ? BW - 2 : BW;          // output pixels per tile row (horizontal tap fusion: the edge lanes are halo only)
  static constexpr int TR = S == 2 ? R + 1 : R + 2 * PAD;
  static constexpr int BOX_BYTES = TR * TW * ROWB;
  static constexpr int BOX_AL = al1024(BOX_BYTES);
  static constexpr int NPLANE = X3 ? 2 : 1;
  static constexpr int A_BYTES = NBOX * BOX_AL;         // one plane of a stage (X3: hi; lo follows)
  static constexpr int STAGE_BYTES = NPLANE * A_BYTES;
  static constexpr int UNITS = NKC * NPY;               // load units per tile
  static constexpr int TAPS = KS * KS;
  static constexpr int W_BYTES = TAPS * NKC * COUT * ROWB;
  static constexpr int W_BYTES_AL = al1024(W_BYTES);      // one plane of the weights (X3: W_hi; W_lo follows)
  static constexpr int ACC_COLS = (HF ? 3 : 1) * R * COUT;      // HF: three accumulator sets (one per horizontal tap) per output row
  static constexpr int TMEM_COLS = pow2_cols(2 * ACC_COLS);
  // residual staging: boxes of CB channels (<= 128 swizzled bytes per pixel) x 128 px x R rows
  static constexpr int CB = COUT < KCMAX ? COUT : KCMAX;
  static constexpr int NRB = COUT / CB;
  static constexpr int RROWB = CB * ESZ;
  static constexpr int RBOX_BYTES = R * BW * RROWB;     // multiple of 1024
  static constexpr int RES_BYTES = RB ? 2 * NRB * RBOX_BYTES : 0;
  static constexpr uint32_t RSWZ = RROWB == 32 ? 1u : RROWB == 64 ? 3u : 7u;
  static constexpr int XCH_BYTES = HF ? 4 * 2 * R * COUT * 4 : 0;      // HF: edge-lane exchange between the four epilogue warps
  static constexpr int SMEM_BASE = 1024 + NPLANE * W_BYTES_AL + STAGES * STAGE_BYTES + RES_BYTES + COUT * 4 + XCH_BYTES + 256;
  // STG (fp32 layers with >= 32 output channels per CTA, where shared memory allows): a column group (32 channels = 128 contiguous
  // bytes of a pixel) is staged per warp in shared memory and written out row-contiguous -- 8 pixels x 128 bytes per store
  // instruction instead of 32 pixels x 32 bytes, a quarter of the L1 wavefronts.  The wide layers' epilogues are bound by exactly
  // those: stem conv1 ran at 64 % of the HBM rate with l1tex 95 % busy.
  static constexpr int STG_WARP_BYTES = 32 * 128;
  static constexpr bool STG_WANTED = S == 1 && !RB && !HF && ESZ == 4 && COUT % 32 == 0 && R * COUT >= 64;
  static constexpr bool STG = STG_WANTED && SMEM_BASE + 128 + 4 * STG_WARP_BYTES <= 232448;
  static constexpr int SMEM_BYTES = SMEM_BASE + (STG ? 128 + 4 * STG_WARP_BYTES : 0);
  static constexpr uint32_t LAYOUT = ROWB == 32 ? 6u : ROWB == 64 ? 4u : 2u;     // SWIZZLE_32B / 64B / 128B
  static constexpr uint32_t SWZ = ROWB == 32 ? 1u : ROWB == 64 ? 3u : 7u;
  static_assert(S == 1 || KS == 3, "stride 2 is implemented for 3x3 only");
  static_assert(!HF || (KS == 3 && S == 1 && 9 * COUT <= 256 && COUT == 16 && !RB), "horizontal tap fusion: 3x3 stride 1, 16 output channels, no staged residual");
  static_assert(2 * ACC_COLS <= 512, "accumulators exceed TMEM");
  // software-pipelined epilogue (see the kernel): stride-1 layers without TMA-staged residual tiles, whose shared-memory reads have no
  // latency to hide (the full-resolution 16 -> 16 layers ran at 6.5 TB/s without it, 5.7 TB/s with it).  TF32: all of them; bf16: the
  // wide layers (64+ output channels per CTA), whose epilogue -- one warp per scheduler -- is what bounds them
  static constexpr bool PIPE = S == 1 && !RB && !HF && ACC_COLS >= 64 && (ESZ == 4 || COUT >= 64);
  static constexpr int GMAX = (ESZ == 2 && !PIPE) ? 64 : 32;
  static constexpr int GCOLS = ACC_COLS < GMAX ? ACC_COLS : GMAX;     // accumulator columns fetched per TMEM wait
  static_assert(ESZ == 2 || ESZ == 4, "bf16 or tf32-in-fp32 elements");
  static_assert(!X3 || (ESZ == 4 && !HF), "3xTF32: fp32 elements, no horizontal tap fusion");
  static_assert(3 * STAGES + 6 <= 31, "barriers and the TMEM slot share 256 bytes");
  static_assert(ACC_COLS % GCOLS == 0, "the epilogue drains whole groups of accumulator columns");
  static_assert(ROWB == 32 || ROWB == 64 || ROWB == 128, "a K-chunk is one 32/64/128-byte swizzled row");
  static_assert(COUT % 16 == 0 && COUT <= 256 && CIN % 16 == 0, "bad channel counts");
  static_assert(SMEM_BYTES <= 232448, "shared memory budget");
};

struct KMaps {
  CUtensorMap m[4];            // stride 1: m[0]; stride 2: m[py * 2 + px] (parity sub-grids)
  CUtensorMap res;             // residual tensor (same shape as the output), when staged by TMA
};

struct KArgs {
  const void* w;               // packed weights, see ttk_conv_umma_pack
  const void* w_lo;            // X3: the W_lo image (same layout)
  const float* bias;
  void* out;
  const void* res[3];
  int rsh[3];
  int nres;
  int res_tma;                 // res[0] (shift 0) arrives through shared memory
  int dual;                    // 1x1 only, two K-concatenated inputs: the first `dual` K-chunks come from tensor map m[0], the rest from m[1]
  int n, h, w_img, cout_total;
  int relu;
  int tiles_x, tiles_y, total;
};

template <int KS, int S, int CIN, int COUT, int R, int STAGES, int RB, int KCO = 0, int ESZ = 2, int HF = 0, int X3 = 0, int H = 0>
__global__ void __launch_bounds__(HF ? THREADS_HF : X3 ? THREADS_X3 : THREADS, 1) conv_umma_kernel(const __grid_constant__ KMaps maps, const KArgs a) {
  constexpr int NTHR = HF ? THREADS_HF : X3 ? THREADS_X3 : THREADS;
  using C = Cfg<KS, S, CIN, COUT, R, STAGES, RB, KCO, ESZ, HF, X3>;
  using F = Fmt16<H>;                                   // ESZ 2: bf16 (H 0) or fp16 (H 1)
  static_assert(!H || (ESZ == 2 && !X3), "fp16 is a 16-bit element format");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sW = smem;
  uint8_t* sA = smem + C::NPLANE * C::W_BYTES_AL;
  uint8_t* sR = sA + STAGES * C::STAGE_BYTES;           // [acc][box][row][px][CB] swizzled (1024-aligned)
  float* sBias = reinterpret_cast<float*>(sR + C::RES_BYTES);
  float* sXch = sBias + COUT;                           // HF: [warp][set 0 of lane 31 | set 2 of lane 0][R][COUT]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sXch + C::XCH_BYTES / 4);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * STAGES + 6);
  // STG: per-warp staging rows of 128 bytes, 128-byte aligned (behind the barriers' 256 bytes)
  uint8_t* sStage = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(bars) + 256 + 127) & ~(uintptr_t)127);
  const uint32_t bar_full = smem_u32(bars), bar_empty = bar_full + 8 * STAGES, bar_tfull = bar_empty + 8 * STAGES,
                 bar_tempty = bar_tfull + 16, bar_rfull = bar_tempty + 16,
                 bar_ready = bar_rfull + 16;      // X3: unit split into hi / lo by the transform warps
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_off = blockIdx.y * COUT;                  // output-channel slice of this CTA
  const bool res_tma = RB && a.res_tma;

  // ---- one-time setup: weights (software swizzle on absolute address bits, as TMA does), bias, barriers, TMEM ----
  {
    constexpr int WV = C::W_BYTES / 16, CPR = C::ROWB / 16;
    const uint32_t wbase = smem_u32(sW);
    for (int i = tid; i < C::NPLANE * WV; i += NTHR) {
      const int p = i / WV, j = i - p * WV;             // plane (X3: 0 = W_hi, 1 = W_lo), 16-byte piece within it
      const uint4* wsrc = reinterpret_cast<const uint4*>(p ? a.w_lo : a.w) + (size_t)blockIdx.y * WV;
      uint32_t addr = wbase + p * C::W_BYTES_AL + (j / CPR) * C::ROWB + (j % CPR) * 16;
      addr ^= ((addr >> 7) & C::SWZ) << 4;
      *reinterpret_cast<uint4*>(sW + (addr - wbase)) = __ldg(wsrc + j);
    }
    for (int i = tid; i < COUT; i += NTHR) sBias[i] = a.bias[n_off + i];
  }
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
      if (X3) mbar_init(bar_ready + 8 * s, 4);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_tfull + 8 * i, 1);
      mbar_init(bar_tempty + 8 * i, HF ? 8 : 4);
      mbar_init(bar_rfull + 8 * i, 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  fence_async_smem();              // weights: generic-proxy writes -> async proxy (tensor core)
  if (warp == 2) tmem_alloc(smem_u32(tmem_slot), C::TMEM_COLS);
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      uint32_t it = 0, tcount = 0;
      for (int tile = blockIdx.x; tile < a.total; tile += gridDim.x, ++tcount) {
        const int tx = tile % a.tiles_x, ty = (tile / a.tiles_x) % a.tiles_y, img = tile / (a.tiles_x * a.tiles_y);
        for (int u = 0; u < C::UNITS; ++u, ++it) {
          const int kc = u / C::NPY, py = u % C::NPY;
          const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
          mbar_wait(bar_empty + 8 * s, ph ^ 1);
          mbar_expect_tx(bar_full + 8 * s, C::NBOX * C::BOX_BYTES);
          const uint32_t dst = smem_u32(sA + s * C::STAGE_BYTES);
          if (S == 1) {
            if (KS == 1 && a.dual)     // channels beyond the first tensor are zero filled
              tma_load_4d(dst, &maps.m[kc < a.dual ? 0 : 1], bar_full + 8 * s, (kc < a.dual ? kc : kc - a.dual) * C::KC, tx * BW, ty * R, img);
            else
              tma_load_4d(dst, &maps.m[0], bar_full + 8 * s, kc * C::KC, tx * C::OUTW - C::PAD, ty * R - C::PAD, img);
          } else {
#pragma unroll
            for (int px = 0; px < 2; ++px)
              tma_load_4d(dst + px * C::BOX_AL, &maps.m[py * 2 + px], bar_full + 8 * s, kc * C::KC, tx * BW - px, ty * R - py, img);
          }
        }
        if (res_tma) {
          // the residual buffer pairs with the accumulator buffer: free once the epilogue of tile-2 has finished
          const uint32_t acc = tcount & 1, aph = (tcount >> 1) & 1;
          mbar_wait(bar_tempty + 8 * acc, aph);
          mbar_expect_tx(bar_rfull + 8 * acc, C::NRB * C::RBOX_BYTES);
#pragma unroll
          for (int b = 0; b < C::NRB; ++b)
            tma_load_4d(smem_u32(sR + (acc * C::NRB + b) * C::RBOX_BYTES), &maps.res, bar_rfull + 8 * acc, n_off + b * C::CB, tx * BW,
                        ty * R, img);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    // The WHOLE warp walks the loops with warp-uniform values and one elected lane issues: addresses, descriptors and the TMEM
    // column then live in uniform registers and consecutive tcgen05.mma are 1-3 instructions apart.  With `if (lane == 0)` around
    // the loops the compiler treated every operand as divergent and wrapped each MMA in an ELECT / R2UR.BROADCAST loop (16
    // instructions, ~80 clk per MMA against the tensor pipe's 45 clk for a thin one -- the thin layers were issue bound).
    {
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
      const bool leader = elect_one();
      const uint32_t wbase = smem_u32(sW) >> 4;
      // operands as 16-byte shared-memory addresses of A and B; every MMA accumulates (the epilogue zeroes what it drains)
      auto issue = [leader](uint32_t d, uint32_t a16, uint32_t b16, uint32_t idesc) {
        const uint64_t da = make_desc16<8 * C::ROWB, C::LAYOUT>(a16), db = make_desc16<8 * C::ROWB, C::LAYOUT>(b16);
        if (X3) {      // the lo planes sit one plane behind the hi planes
          const uint64_t da_lo = make_desc16<8 * C::ROWB, C::LAYOUT>(a16 + C::A_BYTES / 16);
          const uint64_t db_lo = make_desc16<8 * C::ROWB, C::LAYOUT>(b16 + C::W_BYTES_AL / 16);
          if (leader) {
            mma_tf32(d, da_lo, db, idesc, 1u);
            mma_tf32(d, da, db_lo, idesc, 1u);
          }
        }
        if (leader) {
          if (ESZ == 2) mma(d, da, db, idesc, 1u);
          else mma_tf32(d, da, db, idesc, 1u);
        }
      };
      uint32_t it = 0, tcount = 0;
      for (int tile = blockIdx.x; tile < a.total; tile += gridDim.x, ++tcount) {
        const uint32_t acc = tcount & 1, aph = (tcount >> 1) & 1;
        mbar_wait(bar_tempty + 8 * acc, aph);      // accumulators drained and zeroed by the epilogue
        fence_after();
        const uint32_t d_acc = tmem_u + acc * C::ACC_COLS;
        for (int u = 0; u < C::UNITS; ++u, ++it) {
          const int kc = u / C::NPY, py = u % C::NPY;
          const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
          mbar_wait((X3 ? bar_ready : bar_full) + 8 * s, ph);
          fence_after();
          const uint32_t abase = smem_u32(sA + s * C::STAGE_BYTES) >> 4;      // 16-byte units from here on (make_desc16)
          constexpr uint32_t RB16 = C::ROWB / 16;
          if (HF) {
            // horizontal + vertical tap fusion: input row hr (lane = input pixel, no shift) times [W(ky, kx) for all kx, ky in k0..k1]:
            // N = 3 (k1 - k0 + 1) Cout lands in the accumulator sets [row block][kx][Cout]; the epilogue adds the three sets of a row
            // with a lane shift of kx - 1
#pragma unroll 1
            for (int hr = 0; hr < R + 2; ++hr) {
              const int yi = hr - 1;
              const int k0 = yi + 2 - R > 0 ? yi + 2 - R : 0;
              const int k1 = yi + 1 < 2 ? yi + 1 : 2;
              const uint32_t idesc = ESZ == 2 ? make_idesc(128, (k1 - k0 + 1) * 3 * COUT, 0, H) : make_idesc_tf32(128, (k1 - k0 + 1) * 3 * COUT);
              const uint32_t d_tmem = d_acc + (R - 2 - yi + k0) * 3 * COUT;
              const uint32_t arow = abase + hr * C::TW * RB16;
              const uint32_t brow = wbase + ((kc * 3 + k0) * 3 * COUT) * RB16;
#pragma unroll
              for (int ks = 0; ks < C::KSTEPS; ++ks)
                issue(d_tmem, arow + ks * 2, brow + ks * 2, idesc);
            }
          } else if (C::FUSE) {
            // input (halo) row hr = yi + 1 feeds output rows yo = yi + 1 - ky; row yo lives in column block R-1-yo
#pragma unroll 1
            for (int hr = 0; hr < R + 2; ++hr) {
              const int yi = hr - 1;
              const int k0 = yi + 2 - R > 0 ? yi + 2 - R : 0;
              const int k1 = yi + 1 < 2 ? yi + 1 : 2;
              const uint32_t idesc = ESZ == 2 ? make_idesc(128, (k1 - k0 + 1) * COUT, 0, H) : make_idesc_tf32(128, (k1 - k0 + 1) * COUT);
              const uint32_t d_tmem = d_acc + (R - 2 - yi + k0) * COUT;
#pragma unroll
              for (int kx = 0; kx < 3; ++kx) {
                const uint32_t arow = abase + (hr * C::TW + kx) * RB16;
                const uint32_t brow = wbase + (((kc * 3 + kx) * 3 + k0) * COUT) * RB16;
#pragma unroll
                for (int ks = 0; ks < C::KSTEPS; ++ks)
                  issue(d_tmem, arow + ks * 2, brow + ks * 2, idesc);
              }
            }
          } else {
            constexpr uint32_t idesc = ESZ == 2 ? make_idesc(128, COUT, 0, H) : make_idesc_tf32(128, COUT);
#pragma unroll 1
            for (int r = 0; r < R; ++r) {
              const uint32_t d_tmem = d_acc + (R - 1 - r) * COUT;
#pragma unroll
              for (int tap = 0; tap < C::TAPS; ++tap) {
                const int ky = tap / KS, kx = tap % KS;
                uint32_t arow;
                if (S == 1) {
                  arow = abase + ((r + ky) * C::TW + kx) * RB16;
                } else {
                  if ((ky != 1 ? 1 : 0) != py) continue;     // this unit holds the other row parity
                  const int px = kx != 1 ? 1 : 0;
                  arow = abase + px * (C::BOX_AL / 16) + ((r + (ky == 2 ? 1 : 0)) * C::TW + (kx == 2 ? 1 : 0)) * RB16;
                }
                const uint32_t brow = wbase + ((tap * C::NKC + kc) * COUT) * RB16;
#pragma unroll
                for (int ks = 0; ks < C::KSTEPS; ++ks)
                  issue(d_tmem, arow + ks * 2, brow + ks * 2, idesc);
              }
            }
          }
          if (leader) commit(bar_empty + 8 * s);          // smem stage reusable once these MMAs have read it
        }
        if (leader) commit(bar_tfull + 8 * acc);          // accumulators complete
        __syncwarp();
      }
    }
  } else if (X3 && warp >= 6) {
    // ===== transform warps 6..9: raw fp32 unit -> hi = tf32(x) in place, lo = x - hi into the second plane =====
    // element-wise at the same offsets: both planes are 1024-byte aligned, so the swizzle TMA applied holds for both
    const int t = tid - 6 * 32;
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < a.total; tile += gridDim.x) {
      for (int u = 0; u < C::UNITS; ++u, ++it) {
        const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
        mbar_wait(bar_full + 8 * s, ph);
#pragma unroll
        for (int b = 0; b < C::NBOX; ++b) {
          uint8_t* hi = sA + s * C::STAGE_BYTES + b * C::BOX_AL;
          uint8_t* lo = hi + C::A_BYTES;
#pragma unroll 4
          for (int i = t; i < C::BOX_BYTES / 16; i += 128) {
            const float4 v = *reinterpret_cast<const float4*>(hi + i * 16);
            float4 h, l;
            split_tf32(v.x, h.x, l.x);
            split_tf32(v.y, h.y, l.y);
            split_tf32(v.z, h.z, l.z);
            split_tf32(v.w, h.w, l.w);
            *reinterpret_cast<float4*>(hi + i * 16) = h;
            *reinterpret_cast<float4*>(lo + i * 16) = l;
          }
        }
        fence_async_smem();              // generic-proxy writes -> visible to the tensor core
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_ready + 8 * s);
      }
    }
  } else {
    // ===== epilogue warps 2..5: TMEM lane quarter (warp % 4) =====
    const int q = warp & 3;
    const int m = q * 32 + lane;                   // pixel within the tile row = TMEM lane
    constexpr int GCOLS = C::GCOLS;                // accumulator columns fetched per TMEM wait
    constexpr int NSUB = GCOLS / 16;
    constexpr int RW = 4 * ESZ;                    // 32-bit words of the 16 channels of a pixel: 8 (bf16, one sector) or 16 (fp32, two)
    const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
    const int eg = (warp - 2) >> 2;                // HF: epilogue group 0 / 1 takes the even / odd output rows of a tile
    // zero both accumulator buffers, then open them for the MMA warp
    if (eg == 0)
      for (int c = 0; c < 2 * C::ACC_COLS; c += 16) tmem_zero16(lane_base + c);
    tmem_wait_st();
    fence_before();
    __syncwarp();
    if (lane == 0) {
      mbar_arrive(bar_tempty);
      mbar_arrive(bar_tempty + 8);
    }
    // f += the 16 channels held in w (16-bit pairs widened by Fmt16: bf16 by bit placement, fp16 converted)
    auto add_words = [](float* f, const uint32_t* w) {
      if (ESZ == 2) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          f[2 * j] += F::lo(w[j]);
          f[2 * j + 1] += F::hi(w[j]);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) f[j] += __uint_as_float(w[j]);
      }
    };
    uint32_t tcount = 0;
    for (int tile = blockIdx.x; tile < a.total; tile += gridDim.x, ++tcount) {
      const int tx = tile % a.tiles_x, ty = (tile / a.tiles_x) % a.tiles_y, img = tile / (a.tiles_x * a.tiles_y);
      const uint32_t acc = tcount & 1, aph = (tcount >> 1) & 1;
      const int ox = HF ? tx * C::OUTW + m - 1 : tx * BW + m;      // HF: lane m is input pixel tx OUTW - 1 + m and output pixel of the same index
      if (res_tma) mbar_wait(bar_rfull + 8 * acc, aph);
      mbar_wait(bar_tfull + 8 * acc, aph);
      fence_after();
      if constexpr (HF != 0) {
        // ---- horizontal tap fusion: out[r][x] = set0[r][x - 1] + set1[r][x] + set2[r][x + 1]; lanes 0 and 127 are halo only ----
        const uint32_t tbase = lane_base + acc * C::ACC_COLS;
        float* xme = sXch + (q * 2) * R * COUT;
        // pass 1: the edge lanes publish what their neighbours in the adjacent warps need
#pragma unroll 1
        for (int r = eg; r < R; r += 2) {
          uint32_t e0[16], e2[16];
          tmem_ld16(tbase + (R - 1 - r) * 3 * COUT, e0);
          tmem_ld16(tbase + (R - 1 - r) * 3 * COUT + 2 * COUT, e2);
          tmem_wait_ld();
          if (lane == 31) {
#pragma unroll
            for (int j = 0; j < 16; ++j) xme[r * COUT + j] = __uint_as_float(e0[j]);
          }
          if (lane == 0) {
#pragma unroll
            for (int j = 0; j < 16; ++j) xme[R * COUT + r * COUT + j] = __uint_as_float(e2[j]);
          }
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        const float* xprev = sXch + ((q > 0 ? q - 1 : 0) * 2) * R * COUT;              // set 0 of the previous warp's lane 31
        const float* xnext = sXch + ((q < 3 ? q + 1 : 3) * 2 + 1) * R * COUT;          // set 2 of the next warp's lane 0
#pragma unroll 1
        for (int r = eg; r < R; r += 2) {
          uint32_t v0[16], v1[16], v2[16];
          const uint32_t ta = tbase + (R - 1 - r) * 3 * COUT;
          tmem_ld16(ta, v0);
          tmem_ld16(ta + COUT, v1);
          tmem_ld16(ta + 2 * COUT, v2);
          tmem_wait_ld();
          tmem_zero16(ta);
          tmem_zero16(ta + COUT);
          tmem_zero16(ta + 2 * COUT);
          const int oy = ty * R + r;
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            float left = __shfl_up_sync(0xffffffffu, __uint_as_float(v0[j]), 1);
            float right = __shfl_down_sync(0xffffffffu, __uint_as_float(v2[j]), 1);
            if (lane == 0) left = xprev[r * COUT + j];
            if (lane == 31) right = xnext[r * COUT + j];
            f[j] = (left + __uint_as_float(v1[j])) + right + sBias[j];
          }
          const bool live = m >= 1 && m <= C::OUTW && ox < a.w_img && oy < a.h;
          for (int rr = 0; rr < a.nres; ++rr) {            // (the layer this path serves has no residual; kept for the one-conv test hook)
            if (!live) break;
            const int sh = a.rsh[rr];
            const char* rp = (const char*)a.res[rr] +
                             ((((size_t)img * (a.h >> sh) + (oy >> sh)) * (a.w_img >> sh) + (ox >> sh)) * a.cout_total + n_off) * ESZ;
            uint32_t rw[RW];
#pragma unroll
            for (int i = 0; i < RW / 8; ++i) ldg256(rp + 32 * i, &rw[8 * i]);
            add_words(f, rw);
          }
          if (a.relu) {
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
          }
          if (live) {
            char* op = (char*)a.out + ((((size_t)img * a.h + oy) * a.w_img + ox) * a.cout_total + n_off) * ESZ;
            if (ESZ == 2) {
              uint32_t o[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) o[j] = F::pack(f[2 * j], f[2 * j + 1]);
              stg256(op, o);
            } else {
              uint32_t o[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) o[j] = __float_as_uint(f[j]);
              stg256(op, o);
              stg256(op + 32, o + 8);
            }
          }
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");        // the exchange buffer is free for the next tile
      } else if constexpr (C::PIPE) {
        // Software-pipelined drain (stride-1 layers without staged residual tiles, at most one residual): the TMEM load and the residual loads of column
        // group g + 1 are in flight while group g is added up and stored, so neither latency is exposed per group (stem conv1 ran at
        // 59 % of the HBM rate waiting for one tcgen05.ld at a time; residuals read from global memory cost ~1 us per group).
        constexpr int G = C::ACC_COLS / GCOLS;
        uint32_t v[2][NSUB][16], rv[2][NSUB][RW];
        const int nres = a.nres;
        const uint32_t tbase = lane_base + acc * C::ACC_COLS;
        auto fetch = [&](int g, uint32_t (&vv)[NSUB][16], uint32_t (&rr)[NSUB][RW]) {
#pragma unroll
          for (int sb = 0; sb < NSUB; ++sb) tmem_ld16(tbase + g * GCOLS + sb * 16, vv[sb]);
#pragma unroll
          for (int sb = 0; sb < NSUB; ++sb) {
            const int col = g * GCOLS + sb * 16, r = R - 1 - col / COUT, c0 = col % COUT;
            const int oy = ty * R + r;
#pragma unroll
            for (int j = 0; j < RW; ++j) rr[sb][j] = 0;
            if (nres > 0) {
              if (res_tma) {
                const uint32_t row = smem_u32(sR + (acc * C::NRB + c0 / C::CB) * C::RBOX_BYTES) + (r * BW + m) * C::RROWB;
                const uint32_t swz = ((row >> 7) & C::RSWZ) << 4;
#pragma unroll
                for (int i = 0; i < RW / 4; ++i) lds128((row + (c0 % C::CB) * ESZ + 16 * i) ^ swz, &rr[sb][4 * i]);
              } else if (ox < a.w_img && oy < a.h) {
                const int sh = a.rsh[0];
                const char* rp = (const char*)a.res[0] +
                                 ((((size_t)img * (a.h >> sh) + (oy >> sh)) * (a.w_img >> sh) + (ox >> sh)) * a.cout_total + n_off + c0) * ESZ;
#pragma unroll
                for (int i = 0; i < RW / 8; ++i) ldg256(rp + 32 * i, &rr[sb][8 * i]);
              }
            }
          }
        };
        fetch(0, v[0], rv[0]);
        tmem_wait_ld();
#pragma unroll
        for (int sb = 0; sb < NSUB; ++sb) tmem_zero16(tbase + sb * 16);
#pragma unroll
        for (int g = 0; g < G; ++g) {
          if (g + 1 < G) fetch(g + 1, v[(g + 1) & 1], rv[(g + 1) & 1]);
          if (C::STG && nres == 0) {         // (with a residual the staged form measured slower: 0.74 vs 0.60 ms for the half-resolution conv2 layers)
            // the group's 32 channels of this lane's pixel -> staging row `lane` (16-byte chunk c at slot c ^ (lane & 7): conflict free),
            // then 4 store instructions of 8 pixels x 128 contiguous bytes each (lane = pixel it * 8 + lane / 4, 32-byte piece lane % 4)
            const int col = g * GCOLS, r = R - 1 - col / COUT, c0 = col % COUT;
            const int oy = ty * R + r;
            const uint32_t srow = smem_u32(sStage) + (warp - 2) * C::STG_WARP_BYTES;
#pragma unroll
            for (int sb = 0; sb < NSUB; ++sb) {
              float f[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[g & 1][sb][j]) + sBias[c0 + sb * 16 + j];
              if (nres > 0) add_words(f, rv[g & 1][sb]);
              if (a.relu) {
#pragma unroll
                for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
              }
#pragma unroll
              for (int u = 0; u < 4; ++u)
                asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(srow + lane * 128 + (((sb * 4 + u) ^ (lane & 7)) << 4)), "f"(f[4 * u]),
                             "f"(f[4 * u + 1]), "f"(f[4 * u + 2]), "f"(f[4 * u + 3])
                             : "memory");
            }
            __syncwarp();
            const int pq = lane & 3;
#pragma unroll
            for (int it = 0; it < 4; ++it) {
              const int p = it * 8 + (lane >> 2);
              uint32_t o[8];
              lds128(srow + p * 128 + (((2 * pq) ^ (p & 7)) << 4), o);
              lds128(srow + p * 128 + (((2 * pq + 1) ^ (p & 7)) << 4), o + 4);
              const int oxp = tx * BW + (warp & 3) * 32 + p;
              if (oxp < a.w_img && oy < a.h)
                stg256((char*)a.out + ((((size_t)img * a.h + oy) * a.w_img + oxp) * a.cout_total + n_off + c0) * 4 + pq * 32, o);
            }
            __syncwarp();
          } else
#pragma unroll
          for (int sb = 0; sb < NSUB; ++sb) {
            const int col = g * GCOLS + sb * 16, r = R - 1 - col / COUT, c0 = col % COUT;
            const int oy = ty * R + r;
            if (!(ox < a.w_img && oy < a.h)) continue;
            float f[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[g & 1][sb][j]) + sBias[c0 + j];
            if (nres > 0) add_words(f, rv[g & 1][sb]);
            if (a.relu) {
#pragma unroll
              for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
            }
            char* op = (char*)a.out + ((((size_t)img * a.h + oy) * a.w_img + ox) * a.cout_total + n_off + c0) * ESZ;
            if (ESZ == 2) {
              uint32_t o[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) o[j] = F::pack(f[2 * j], f[2 * j + 1]);
              stg256(op, o);
            } else {
              uint32_t o[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) o[j] = __float_as_uint(f[j]);
              stg256(op, o);
              stg256(op + 32, o + 8);
            }
          }
          if (g + 1 < G) {
            tmem_wait_ld();
#pragma unroll
            for (int sb = 0; sb < NSUB; ++sb) tmem_zero16(tbase + (g + 1) * GCOLS + sb * 16);     // leave the columns zeroed for the next tile
          }
        }
      } else {
#pragma unroll 1
      for (int g0 = 0; g0 < C::ACC_COLS; g0 += GCOLS) {
        uint32_t v[NSUB][16];
        const uint32_t taddr = lane_base + acc * C::ACC_COLS + g0;
#pragma unroll
        for (int sb = 0; sb < NSUB; ++sb) tmem_ld16(taddr + sb * 16, v[sb]);
        // residual operands for the same columns, all fetched before the TMEM wait so that the latencies overlap (the
        // lower-resolution fuse terms used to be loaded one by one at their point of use: 0.25 ms per stage-3/4 fuse conv)
        uint32_t rv[NSUB][RW], rx[NSUB][2][RW];
        const int nres = a.nres;
#pragma unroll
        for (int sb = 0; sb < NSUB; ++sb) {
          const int col = g0 + sb * 16, r = R - 1 - col / COUT, c0 = col % COUT;
          const int oy = ty * R + r;
          const bool live = ox < a.w_img && oy < a.h;
#pragma unroll
          for (int j = 0; j < RW; ++j) rv[sb][j] = 0;
          if (nres > 0) {
            if (res_tma) {
              const uint32_t row = smem_u32(sR + (acc * C::NRB + c0 / C::CB) * C::RBOX_BYTES) + (r * BW + m) * C::RROWB;
              const uint32_t swz = ((row >> 7) & C::RSWZ) << 4;       // a pixel row never crosses a 128-byte line: one XOR for all its chunks
#pragma unroll
              for (int i = 0; i < RW / 4; ++i) lds128((row + (c0 % C::CB) * ESZ + 16 * i) ^ swz, &rv[sb][4 * i]);
            } else if (live) {
              const int sh = a.rsh[0];
              const char* rp = (const char*)a.res[0] +
                               ((((size_t)img * (a.h >> sh) + (oy >> sh)) * (a.w_img >> sh) + (ox >> sh)) * a.cout_total + n_off + c0) * ESZ;
#pragma unroll
              for (int i = 0; i < RW / 8; ++i) ldg256(rp + 32 * i, &rv[sb][8 * i]);
            }
#pragma unroll
            for (int rr = 1; rr < 3; ++rr) {
              if (rr < nres && live) {
                const int sh = a.rsh[rr];
                const char* rp = (const char*)a.res[rr] +
                                 ((((size_t)img * (a.h >> sh) + (oy >> sh)) * (a.w_img >> sh) + (ox >> sh)) * a.cout_total + n_off + c0) * ESZ;
#pragma unroll
                for (int i = 0; i < RW / 8; ++i) ldg256(rp + 32 * i, &rx[sb][rr - 1][8 * i]);
              }
            }
          }
        }
        tmem_wait_ld();
#pragma unroll
        for (int sb = 0; sb < NSUB; ++sb) tmem_zero16(taddr + sb * 16);     // leave the columns zeroed for the next tile
#pragma unroll
        for (int sb = 0; sb < NSUB; ++sb) {
          const int col = g0 + sb * 16, r = R - 1 - col / COUT, c0 = col % COUT;
          const int oy = ty * R + r;
          if (!(ox < a.w_img && oy < a.h)) continue;
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[sb][j]) + sBias[c0 + j];
          if (nres > 0) {
            add_words(f, rv[sb]);
#pragma unroll
            for (int rr = 1; rr < 3; ++rr) {
              if (rr >= nres) break;
              add_words(f, rx[sb][rr - 1]);
            }
          }
          if (a.relu) {
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
          }
          // 256-bit stores: the 16 channels of a pixel are one (bf16) or two (fp32) whole 32-byte sectors
          char* op = (char*)a.out + ((((size_t)img * a.h + oy) * a.w_img + ox) * a.cout_total + n_off + c0) * ESZ;
          if (ESZ == 2) {
            uint32_t o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = F::pack(f[2 * j], f[2 * j + 1]);
            stg256(op, o);
          } else {
            uint32_t o[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) o[j] = __float_as_uint(f[j]);
            stg256(op, o);
            stg256(op + 32, o + 8);
          }
        }
      }
      }
      tmem_wait_st();
      fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
    }
  }
  fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem, C::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
// output channels one CTA handles: 128-wide 3x3 layers with 64+ input channels are split so the weights fit in shared memory
// 3xTF32 (x3): W_hi and W_lo of a 3x3 slice are 72 cin_p cout_tile bytes; cin_p cout_tile <= 2048 keeps them at <= 144 KB
int cout_tile(const TtkConv& cv, int esz, bool x3 = false) {
  if (x3) return cv.k == 3 ? std::min(cv.cout_p, 2048 / cv.cin_p) : cv.cout_p;
  return (cv.k == 3 && cv.cout_p == 128 && cv.cin_p >= 64) ? (esz == 2 ? 64 : 32) : cv.cout_p;
}
bool fused_ky(const TtkConv& cv, int esz, bool x3 = false) { return cv.k == 3 && cv.stride == 1 && 3 * cout_tile(cv, esz, x3) <= 256; }
// horizontal + vertical tap fusion (one MMA per input row and K step, N = 9 Cout): the thin layer that is bound by its MMA count
// -- TF32 only: with K = 8 per instruction it has twice the MMAs of the bf16 kernel (4.48 -> 3.50 ms per 32 stacks); in bf16 the extra
// epilogue work (three accumulator sets, two shuffles per value, edge-lane exchange) outweighs the saved MMAs (1.74 -> 3.00 ms)
bool fused_h(const TtkConv& cv, int esz, bool x3 = false) { return esz == 4 && !x3 && cv.k == 3 && cv.stride == 1 && cv.cin_p == 128 && cv.cout_p == 16; }
// channels per K-chunk (one swizzled shared-memory row).  The stride-1 3x3 layers with 64+ input channels are bound by their MMA
// count (a 128-pixel x 32-byte MMA holds the tensor pipe 45.5 clk at N <= 48 and N / 2 clk from N = 96 on, tools/tf32_probe.cu) and
// the halo rows of a tile are pure overhead: 3 (R + 2) / R MMAs per K step and output row.  Narrow chunks shrink the staging boxes so
// that taller tiles fit: bf16 transition1.0 R = 3 -> 8, the 64 -> 64 layers R = 2 -> 4, and the 128 -> 128 layers get a second
// pipeline stage.  With fp32 elements the 3x3 weights of the wide layers take up to 147 KB, which leaves room for 8-channel chunks.
// x3: the narrowest chunk for every 3x3 layer (one 32-byte row, one MMA K step): the MMA count does not depend on it, and the
// staging boxes -- two planes each -- stay small enough for two stages next to up to 144 KB of weights.
int kc_of(const TtkConv& cv, int esz, bool x3 = false) {
  if (x3) return cv.k == 3 ? 8 : std::min(cv.cin_p, 32);
  if (esz == 2) {
    if (cv.k == 3 && cv.stride == 1 && cv.cin_p >= 64) return 32;
    // stride 2 with 64+ input channels (transition1.1 1.74 -> 1.49 ms): two-row tiles and a third pipeline stage in the same shared memory
    if (cv.k == 3 && cv.stride == 2 && cv.cin_p >= 64) return 32;
    return cv.cin_p < 64 ? cv.cin_p : 64;
  }
  if (cv.k == 3 && cv.stride == 1 && cv.cin_p == 128 && cv.cout_p == 16) return 16;      // transition1.0: 64-byte rows fill faster than 32-byte ones
  if (cv.k == 3 && cv.cin_p >= 64) return 8;
  if (cv.k == 3 && cv.stride == 2 && cv.cin_p == 32 && cv.cout_p == 128) return 8;
  if (cv.k == 3) return 16;
  return 32;
}

CUtensorMapSwizzle swizzle_for(int row_bytes) {
  return row_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
}

float round_tf32(float v) {      // nearest-even on the 13 dropped mantissa bits (finite inputs)
  uint32_t u;
  memcpy(&u, &v, 4);
  u += 0xfffu + ((u >> 13) & 1u);
  u &= ~0x1fffu;
  memcpy(&v, &u, 4);
  return v;
}

template <int KS, int S, int CIN, int COUT, int R, int STAGES, int RB, int KCO = 0, int ESZ = 2, int HF = 0, int X3 = 0, int H = 0>
int launch(const TtkConv& cv, const ConvLaunch& a, cudaStream_t st) {
  using C = Cfg<KS, S, CIN, COUT, R, STAGES, RB, KCO, ESZ, HF, X3>;
  if (C::KC != kc_of(cv, ESZ, X3) || COUT != cout_tile(cv, ESZ, X3) || (HF != 0) != fused_h(cv, ESZ, X3)) {
    ttk_set_error("conv %s: kernel K-chunk %d / output slice %d differ from the packed weights' %d / %d", cv.name.c_str(), C::KC, COUT,
                  kc_of(cv, ESZ, X3), cout_tile(cv, ESZ, X3));
    return TTK_ERR_STATE;
  }
  EncodeFn encode = get_encode();
  if (!encode) {
    ttk_set_error("cuTensorMapEncodeTiled is not available from the driver");
    return TTK_ERR_CUDA;
  }
  static TtkPerDevice attr;
  if (attr.first()) {
    TTK_CUDA(cudaFuncSetAttribute(conv_umma_kernel<KS, S, CIN, COUT, R, STAGES, RB, KCO, ESZ, HF, X3, H>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  C::SMEM_BYTES));
  }
  if (S == 2 && ((a.hin & 1) || (a.win & 1))) return TTK_ERR_UNSUPPORTED;
  // the input map's TFLOAT32 type makes TMA round fp32 to TF32 (nearest-even) while it fills shared memory; 3xTF32 needs the raw values
  const CUtensorMapDataType in_type =
      ESZ == 2 ? Fmt16<H>::MAP : X3 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_TFLOAT32;
  const CUtensorMapDataType res_type = ESZ == 2 ? Fmt16<H>::MAP : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  KMaps maps;
  cuuint32_t box[4] = {(cuuint32_t)C::KC, (cuuint32_t)C::TW, (cuuint32_t)C::TR, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  for (int i = 0; i < (S == 2 ? 4 : 1); ++i) {
    const int py = i >> 1, px = i & 1;
    cuuint64_t dims[4] = {(cuuint64_t)CIN, (cuuint64_t)(a.win / S), (cuuint64_t)(a.hin / S), (cuuint64_t)a.n};
    cuuint64_t strides[3] = {(cuuint64_t)CIN * ESZ * S, (cuuint64_t)a.win * CIN * ESZ * S, (cuuint64_t)a.hin * a.win * CIN * ESZ};
    void* base = (char*)const_cast<void*>(a.in) + ((size_t)py * a.win + px) * CIN * ESZ;
    const CUresult r = encode(&maps.m[i], in_type, 4, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(C::ROWB),
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      ttk_set_error("cuTensorMapEncodeTiled failed (%d) for conv %s", (int)r, cv.name.c_str());
      return TTK_ERR_CUDA;
    }
  }
  for (int i = (S == 2 ? 4 : 1); i < 4; ++i) maps.m[i] = maps.m[0];
  const bool res_tma = RB && a.nres > 0 && a.res_shift[0] == 0;
  maps.res = maps.m[0];
  if (res_tma) {
    cuuint64_t dims[4] = {(cuuint64_t)a.cout, (cuuint64_t)a.wout, (cuuint64_t)a.hout, (cuuint64_t)a.n};
    cuuint64_t strides[3] = {(cuuint64_t)a.cout * ESZ, (cuuint64_t)a.wout * a.cout * ESZ, (cuuint64_t)a.hout * a.wout * a.cout * ESZ};
    cuuint32_t rbox[4] = {(cuuint32_t)C::CB, (cuuint32_t)BW, (cuuint32_t)R, 1};
    const CUresult r = encode(&maps.res, res_type, 4, const_cast<void*>(a.res[0]), dims, strides, rbox, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              swizzle_for(C::RROWB), CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      ttk_set_error("cuTensorMapEncodeTiled (residual) failed (%d) for conv %s", (int)r, cv.name.c_str());
      return TTK_ERR_CUDA;
    }
  }
  KArgs k;
  k.w = ESZ == 2 ? (H ? (const void*)cv.w_umma_f16 : (const void*)cv.w_umma) : X3 ? (const void*)cv.w_x3 : (const void*)cv.w_umma32;
  k.w_lo = X3 ? (const void*)(cv.w_x3 + (size_t)cv.k * cv.k * cv.cin_p * cv.cout_p) : nullptr;      // [W_hi image | W_lo image]
  k.bias = cv.bias;
  k.out = a.out;
  for (int i = 0; i < 3; ++i) {
    k.res[i] = a.res[i];
    k.rsh[i] = a.res_shift[i];
  }
  k.nres = a.nres;
  k.res_tma = res_tma ? 1 : 0;
  k.dual = 0;
  k.n = a.n;
  k.h = a.hout;
  k.w_img = a.wout;
  k.cout_total = a.cout;
  k.relu = a.relu;
  k.tiles_x = ttk_cdiv(a.wout, C::OUTW);
  k.tiles_y = ttk_cdiv(a.hout, R);
  k.total = k.tiles_x * k.tiles_y * a.n;
  const int nsplit = a.cout / COUT;
  // persistent CTAs: as many as fit per SM (shared memory and TMEM columns), never more than there are tiles
  int occ = std::min(232448 / (C::SMEM_BYTES + 1024), 512 / C::TMEM_COLS);
  occ = std::max(1, std::min(occ, 2));
  const int gx = std::max(1, std::min(k.total, ttk_num_sms() * occ / nsplit));
  dim3 grid(gx, nsplit);
  conv_umma_kernel<KS, S, CIN, COUT, R, STAGES, RB, KCO, ESZ, HF, X3, H><<<grid, HF ? THREADS_HF : X3 ? THREADS_X3 : THREADS, C::SMEM_BYTES, st>>>(maps, k);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

// Bottleneck tail: out = relu(W3 a + Wd x + bias) with a (32 channels) and x (64 channels) K-concatenated.  bf16 / fp16: two 64-channel
// K-chunks (the first box reaches past the 32-channel tensor, TMA zero fills); tf32: three 32-channel chunks (a | x[0:32] | x[32:64]).
template <int ESZ, int H = 0>
int launch_dual(const void* w_dual, const float* bias_dual, const ConvLaunch& a, cudaStream_t st) {
  constexpr int R = 2, STAGES = 3, KC = 128 / ESZ, CINK = ESZ == 2 ? 128 : 96;
  using C = Cfg<1, 1, CINK, 128, R, STAGES, 0, 0, ESZ>;
  EncodeFn encode = get_encode();
  if (!encode) return TTK_ERR_UNSUPPORTED;
  static TtkPerDevice attr;
  if (attr.first()) {
    TTK_CUDA(cudaFuncSetAttribute(conv_umma_kernel<1, 1, CINK, 128, R, STAGES, 0, 0, ESZ, 0, 0, H>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  C::SMEM_BYTES));
  }
  KMaps maps;
  cuuint32_t box[4] = {(cuuint32_t)KC, (cuuint32_t)BW, (cuuint32_t)R, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  const void* ins[2] = {a.in, a.in2};
  const int cins[2] = {a.cin, a.cin2};
  for (int i = 0; i < 2; ++i) {
    cuuint64_t dims[4] = {(cuuint64_t)cins[i], (cuuint64_t)a.win, (cuuint64_t)a.hin, (cuuint64_t)a.n};
    cuuint64_t strides[3] = {(cuuint64_t)cins[i] * ESZ, (cuuint64_t)a.win * cins[i] * ESZ, (cuuint64_t)a.hin * a.win * cins[i] * ESZ};
    const CUresult r = encode(&maps.m[i], ESZ == 2 ? Fmt16<H>::MAP : CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 4, const_cast<void*>(ins[i]),
                              dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return TTK_ERR_UNSUPPORTED;      // e.g. a driver that rejects a box wider than the tensor
  }
  maps.m[2] = maps.m[3] = maps.res = maps.m[0];
  KArgs k;
  k.w = w_dual;
  k.w_lo = nullptr;
  k.bias = bias_dual;
  k.out = a.out;
  for (int i = 0; i < 3; ++i) {
    k.res[i] = nullptr;
    k.rsh[i] = 0;
  }
  k.nres = 0;
  k.res_tma = 0;
  k.dual = 1;
  k.n = a.n;
  k.h = a.hout;
  k.w_img = a.wout;
  k.cout_total = a.cout;
  k.relu = a.relu;
  k.tiles_x = ttk_cdiv(a.wout, BW);
  k.tiles_y = ttk_cdiv(a.hout, R);
  k.total = k.tiles_x * k.tiles_y * a.n;
  const int gx = std::max(1, std::min(k.total, ttk_num_sms()));
  conv_umma_kernel<1, 1, CINK, 128, R, STAGES, 0, 0, ESZ, 0, 0, H><<<gx, THREADS, C::SMEM_BYTES, st>>>(maps, k);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

}  // namespace

int ttk_conv_umma_launch_dual(const void* w_dual, const float* bias_dual, const ConvLaunch& a, cudaStream_t st, int esz, bool f16) {
  if (a.cin != 32 || a.cin2 != 64 || a.cout != 128) return TTK_ERR_UNSUPPORTED;
  if (esz == 2) return f16 ? launch_dual<2, 1>(w_dual, bias_dual, a, st) : launch_dual<2>(w_dual, bias_dual, a, st);
  return launch_dual<4>(w_dual, bias_dual, a, st);
}

// Host image of the fused bottleneck tail's B operand: [k-chunk][cout 128][KC], chunk 0 = conv3 (32 input channels, zero padded to KC),
// then the projection shortcut's 64 input channels.  bf16 / fp16 (f16): KC = 64 (2 chunks); tf32: KC = 32 (3 chunks), values rounded
// to TF32.
void ttk_conv_umma_pack_dual(const float* w3, const float* wd, int esz, std::vector<uint8_t>& out, bool f16) {
  const int KC = 128 / esz, nk = esz == 2 ? 2 : 3;
  out.assign((size_t)nk * 128 * KC * esz, 0);
  auto put = [&](int kc, int co, int c, float v) {
    const size_t i = ((size_t)kc * 128 + co) * KC + c;
    if (esz == 2 && f16) reinterpret_cast<__half*>(out.data())[i] = Fmt16<1>::round(v);
    else if (esz == 2) reinterpret_cast<__nv_bfloat16*>(out.data())[i] = Fmt16<0>::round(v);
    else reinterpret_cast<float*>(out.data())[i] = round_tf32(v);
  };
  for (int co = 0; co < 128; ++co) {
    for (int ci = 0; ci < 32; ++ci) put(0, co, ci, w3[(size_t)co * 32 + ci]);
    for (int ci = 0; ci < 64; ++ci) put(1 + ci / KC, co, ci % KC, wd[(size_t)co * 64 + ci]);
  }
}

// Weights for the tensor-core path: rows of KC input channels (K-major), zero padded, per output-channel slice:
//   fused 3x3 stride 1 : [slice][k-chunk][kx][ky][cout_tile][KC]   (B = the three vertical taps side by side)
//   transition1.0      : [k-chunk][ky][kx][cout][KC]               (B = all nine taps: horizontal + vertical fusion)
//   otherwise          : [slice][tap][k-chunk][cout_tile][KC]
// bf16 (w_umma), TF32-rounded fp32 (w_umma32), 3xTF32 (w_x3: the W_hi = tf32(w) image, then the W_lo = w - W_hi image) and fp16
// (w_umma_f16, the bf16 layout) are all kept; the 2- and 4-byte images differ in KC and in the slice width of the wide layers.
int ttk_conv_umma_pack(TtkConv& cv, const float* w_host) {
  const int kk = cv.k * cv.k;
  for (int mode = 0; mode < 4; ++mode) {
    const int esz = mode == 0 || mode == 3 ? 2 : 4;
    const bool x3 = mode == 2, f16 = mode == 3;
    const int KC = kc_of(cv, esz, x3);
    const int nkc = cv.cin_p / KC;
    const int ct = cout_tile(cv, esz, x3);
    const bool fused = fused_ky(cv, esz, x3);
    const size_t count = (size_t)kk * cv.cin_p * cv.cout_p;
    std::vector<uint8_t> w(count * esz * (x3 ? 2 : 1), 0);
    for (int co = 0; co < cv.cout; ++co)
      for (int ci = 0; ci < cv.cin; ++ci)
        for (int t = 0; t < kk; ++t) {
          const int kc = ci / KC, c = ci % KC, sl = co / ct, cl = co % ct;
          size_t row;
          if (fused_h(cv, esz, x3)) {
            const int ky = t / 3, kx = t % 3;
            row = (((size_t)sl * nkc + kc) * 3 + ky) * 3 + kx;      // [k-chunk][ky][kx][cout]: B of one input row = all nine taps
          } else if (fused) {
            const int ky = t / 3, kx = t % 3;
            row = (((size_t)sl * nkc + kc) * 3 + kx) * 3 + ky;
          } else {
            row = ((size_t)sl * kk + t) * nkc + kc;
          }
          const float v = w_host[((size_t)co * cv.cin + ci) * kk + t];
          const size_t i = (row * ct + cl) * KC + c;
          if (f16) {
            reinterpret_cast<__half*>(w.data())[i] = Fmt16<1>::round(v);
          } else if (esz == 2) {
            reinterpret_cast<__nv_bfloat16*>(w.data())[i] = Fmt16<0>::round(v);
          } else {
            const float hi = round_tf32(v);
            reinterpret_cast<float*>(w.data())[i] = hi;
            if (x3) reinterpret_cast<float*>(w.data())[count + i] = v - hi;      // exact
          }
        }
    void** dst = f16 ? (void**)&cv.w_umma_f16 : esz == 2 ? (void**)&cv.w_umma : x3 ? (void**)&cv.w_x3 : (void**)&cv.w_umma32;
    if (!*dst) TTK_CUDA(cudaMalloc(dst, w.size()));
    TTK_CUDA(cudaMemcpy(*dst, w.data(), w.size(), cudaMemcpyHostToDevice));
  }
  return TTK_OK;
}

namespace {
// 16-bit elements (H = 0: bf16, 1: fp16): one dispatch table for both formats
template <int H>
int launch16(const TtkConv& cv, const ConvLaunch& a, cudaStream_t st) {
  const int ci = cv.cin_p, co = cout_tile(cv, 2);
  const int k = cv.k, s = cv.stride;
#define TTK_UMMA(KS_, S_, CI_, CO_, R_, ST_, RB_) \
  if (k == KS_ && s == S_ && ci == CI_ && co == CO_) return launch<KS_, S_, CI_, CO_, R_, ST_, RB_, 0, 2, 0, 0, H>(cv, a, st);
#define TTK_UMMA_KC(KS_, S_, CI_, CO_, R_, ST_, KC_) \
  if (k == KS_ && s == S_ && ci == CI_ && co == CO_) return launch<KS_, S_, CI_, CO_, R_, ST_, 0, KC_, 2, 0, 0, H>(cv, a, st);
  // 3x3 stride 1
  TTK_UMMA(3, 1, 16, 64, 4, 3, 0)     // stem conv1 (9 -> 64, input padded to 16 channels)
  TTK_UMMA_KC(3, 1, 64, 64, 4, 3, 32)      // stem conv2, quarter-resolution branch
  if (k == 3 && s == 1 && ci == 32 && co == 32 && a.nres == 0) return launch<3, 1, 32, 32, 8, 2, 0, 0, 2, 0, 0, H>(cv, a, st);   // no residual tiles to stage: taller tile
  TTK_UMMA(3, 1, 32, 32, 4, 2, 1)     // bottleneck conv2, half-resolution branch
  TTK_UMMA(3, 1, 16, 16, 8, 3, 1)     // full-resolution branch
  TTK_UMMA_KC(3, 1, 128, 16, 8, 2, 32)     // transition1.0
  TTK_UMMA_KC(3, 1, 128, 64, 2, 2, 32)     // eighth-resolution branch (128 -> 128 as two 64-channel output slices)
  // 3x3 stride 2 (transitions and fuse down-paths)
  TTK_UMMA_KC(3, 2, 128, 32, 2, 3, 32)
  TTK_UMMA(3, 2, 16, 16, 4, 3, 0)
  TTK_UMMA(3, 2, 16, 32, 4, 3, 0)
  TTK_UMMA(3, 2, 16, 64, 4, 3, 0)
  TTK_UMMA(3, 2, 16, 128, 2, 3, 0)
  TTK_UMMA(3, 2, 32, 32, 4, 2, 0)
  TTK_UMMA(3, 2, 32, 64, 4, 2, 0)
  TTK_UMMA(3, 2, 32, 128, 2, 2, 0)
  TTK_UMMA_KC(3, 2, 64, 64, 2, 3, 32)      // 64 -> 128 as two output slices
  // 1x1
  TTK_UMMA(1, 1, 64, 32, 4, 2, 0)     // bottleneck conv1, fuse 64 -> 32
  TTK_UMMA(1, 1, 32, 128, 2, 3, 1)    // bottleneck conv3 (+ projection shortcut as residual)
  TTK_UMMA(1, 1, 64, 128, 2, 3, 0)    // bottleneck projection shortcut
  TTK_UMMA(1, 1, 32, 16, 4, 3, 0)     // fuse layers (low -> high resolution)
  TTK_UMMA(1, 1, 64, 16, 4, 3, 0)
  TTK_UMMA(1, 1, 128, 16, 4, 2, 0)
  TTK_UMMA(1, 1, 128, 32, 4, 2, 0)
  TTK_UMMA(1, 1, 128, 64, 2, 2, 0)
#undef TTK_UMMA_KC
#undef TTK_UMMA
  return TTK_ERR_UNSUPPORTED;
}
}  // namespace

int ttk_conv_umma_launch(const TtkConv& cv, const ConvLaunch& a, cudaStream_t st, int esz, bool x3, bool f16) {
  if (esz == 2) return f16 ? launch16<1>(cv, a, st) : launch16<0>(cv, a, st);
  const int ci = cv.cin_p, co = cout_tile(cv, esz, x3);
  const int k = cv.k, s = cv.stride;
  if (x3) {
    // ---- 3xTF32: shared memory = 1 KB + 2 planes x (weights + STAGES x box) + bias + barriers (+ 16 KB store staging where it fits) ----
    // 3x3 boxes of 8 channels: stride 1 (R + 2) x 130 px x 32 B, stride 2 two boxes of (R + 1) x 129 px x 32 B, each 1024-aligned.
#define TTK_UMMA3(KS_, S_, CI_, CO_, R_, ST_, KC_) \
  if (k == KS_ && s == S_ && ci == CI_ && co == CO_) return launch<KS_, S_, CI_, CO_, R_, ST_, 0, KC_, 4, 0, 1>(cv, a, st);
    // 3x3 stride 1 (vertical tap fusion throughout)
    TTK_UMMA3(3, 1, 16, 64, 4, 2, 8)      // stem conv1: 72 KB weights + 2 x 50 KB stages + 16 KB staging = 190 KB
    TTK_UMMA3(3, 1, 64, 32, 2, 2, 8)      // stem conv2, quarter-resolution branch (two 32-channel slices): 144 KB + 2 x 34 KB = 213 KB
    TTK_UMMA3(3, 1, 32, 32, 4, 2, 8)      // half-resolution branch: 72 KB + 2 x 50 KB + 16 KB = 190 KB
    TTK_UMMA3(3, 1, 16, 16, 8, 2, 8)      // full-resolution branch: 18 KB + 2 x 82 KB = 183 KB
    TTK_UMMA3(3, 1, 128, 16, 2, 2, 8)     // transition1.0, eighth-resolution branch (eight 16-channel slices): 144 KB + 2 x 34 KB = 213 KB
    // 3x3 stride 2
    TTK_UMMA3(3, 2, 16, 16, 2, 3, 8)      // 18 KB + 3 x 52 KB = 175 KB
    TTK_UMMA3(3, 2, 16, 32, 2, 3, 8)      // 36 KB + 3 x 52 KB = 193 KB
    TTK_UMMA3(3, 2, 16, 64, 2, 2, 8)      // 72 KB + 2 x 52 KB = 177 KB
    TTK_UMMA3(3, 2, 16, 128, 1, 2, 8)     // 144 KB + 2 x 36 KB = 218 KB
    TTK_UMMA3(3, 2, 32, 32, 2, 2, 8)      // 72 KB + 2 x 52 KB = 177 KB
    TTK_UMMA3(3, 2, 32, 64, 1, 2, 8)      // 32 -> 64 and 32 -> 128 (two slices): 144 KB + 2 x 36 KB = 218 KB
    TTK_UMMA3(3, 2, 64, 32, 1, 2, 8)      // 64 -> 128 (four slices): 144 KB + 2 x 36 KB = 218 KB
    TTK_UMMA3(3, 2, 128, 16, 1, 2, 8)     // 128 -> 32 (two slices): 144 KB + 2 x 36 KB = 218 KB
    // 1x1: 2 x 64 KB per stage of 2 rows x 128 px x 128 B
    TTK_UMMA3(1, 1, 64, 32, 2, 2, 32)
    TTK_UMMA3(1, 1, 32, 128, 2, 2, 32)
    TTK_UMMA3(1, 1, 64, 128, 2, 2, 32)
    TTK_UMMA3(1, 1, 32, 16, 2, 3, 32)
    TTK_UMMA3(1, 1, 64, 16, 2, 3, 32)
    TTK_UMMA3(1, 1, 128, 16, 2, 3, 32)
    TTK_UMMA3(1, 1, 128, 32, 2, 2, 32)
    TTK_UMMA3(1, 1, 128, 64, 2, 2, 32)
#undef TTK_UMMA3
    return TTK_ERR_UNSUPPORTED;
  }
  // ---- TF32 (fp32 activations): same tiles, re-sized for 4-byte elements (shared memory: weights + STAGES boxes + residual tiles) ----
#define TTK_UMMA32(KS_, S_, CI_, CO_, R_, ST_, RB_, KC_) \
  if (k == KS_ && s == S_ && ci == CI_ && co == CO_) return launch<KS_, S_, CI_, CO_, R_, ST_, RB_, KC_, 4>(cv, a, st);
  // 3x3 stride 1
  TTK_UMMA32(3, 1, 16, 64, 4, 3, 0, 16)      // stem conv1
  TTK_UMMA32(3, 1, 64, 64, 4, 3, 0, 8)       // stem conv2, quarter-resolution branch: 147 KB of weights + three 25 KB boxes (no room for store staging; two boxes + staging measured slower: 3.80 vs 3.66 ms)
  if (k == 3 && s == 1 && ci == 32 && co == 32 && a.nres == 0) return launch<3, 1, 32, 32, 8, 2, 0, 16, 4>(cv, a, st);
  TTK_UMMA32(3, 1, 32, 32, 4, 3, 0, 16)      // half-resolution branch (residual read from global memory: no room for staged tiles)
  if (k == 3 && s == 1 && ci == 16 && co == 16 && a.nres == 0) return launch<3, 1, 16, 16, 8, 2, 0, 16, 4>(cv, a, st);     // taller tile (R = 4 with four stages: 0.77 vs 0.66 ms)
  TTK_UMMA32(3, 1, 16, 16, 4, 3, 1, 16)      // full-resolution branch, residual tiles staged by TMA
  if (k == 3 && s == 1 && ci == 128 && co == 16) return launch<3, 1, 128, 16, 4, 3, 0, 16, 4, 1>(cv, a, st);     // transition1.0: nine taps per MMA
  TTK_UMMA32(3, 1, 128, 32, 4, 3, 0, 8)      // eighth-resolution branch (128 -> 128 as four 32-channel output slices)
  // 3x3 stride 2
  TTK_UMMA32(3, 2, 128, 32, 2, 3, 0, 8)
  TTK_UMMA32(3, 2, 16, 16, 4, 2, 0, 16)
  TTK_UMMA32(3, 2, 16, 32, 4, 2, 0, 16)
  TTK_UMMA32(3, 2, 16, 64, 4, 2, 0, 16)
  TTK_UMMA32(3, 2, 16, 128, 2, 2, 0, 16)
  TTK_UMMA32(3, 2, 32, 32, 4, 2, 0, 16)
  TTK_UMMA32(3, 2, 32, 64, 2, 3, 0, 16)
  TTK_UMMA32(3, 2, 32, 128, 2, 3, 0, 8)
  TTK_UMMA32(3, 2, 64, 32, 2, 3, 0, 8)       // 64 -> 128 as four output slices
  // 1x1
  TTK_UMMA32(1, 1, 64, 32, 4, 3, 0, 32)
  TTK_UMMA32(1, 1, 32, 128, 2, 3, 0, 32)
  TTK_UMMA32(1, 1, 64, 128, 2, 3, 0, 32)
  TTK_UMMA32(1, 1, 32, 16, 4, 3, 0, 32)
  TTK_UMMA32(1, 1, 64, 16, 4, 3, 0, 32)
  TTK_UMMA32(1, 1, 128, 16, 4, 3, 0, 32)
  TTK_UMMA32(1, 1, 128, 32, 4, 3, 0, 32)
  TTK_UMMA32(1, 1, 128, 64, 2, 3, 0, 32)
#undef TTK_UMMA32
  return TTK_ERR_UNSUPPORTED;
}
