// Fused BasicBlock of the HRNet branches on tcgen05 (bf16 / fp16: 16- and 32-channel branches; TF32 on fp32 activations: the 16-channel
// full-resolution branch, whose two convolutions are HBM bound on their own -- 320 bytes per pixel conv by conv, 128 fused):
//   y = relu(conv2(relu(conv1(x) + b1)) + b2 + x)              balldetection/models/wasb.py:35-64 (BasicBlock.forward, BN folded)
// The two 3x3 convolutions of a block run in ONE kernel: the intermediate tensor never leaves the SM and the residual is taken
// from the staged input tile, so a block reads x once and writes y once (conv by conv it is read x, write t, read t, read x,
// write y: 5 tensor passes instead of 2 -- the branch layers are HBM bound, DESIGN.md section 4.2).
//
// Tile = R output rows x 126 output pixels.  One TMA box brings the (R+4) x 130 pixel input halo (zero fill outside the image).
//   M1: conv1 on tensor cores for the (R+2) x 128 intermediate pixels the tile needs (vertical tap fusion as in conv_umma.cu:
//       one MMA per input row and horizontal tap against [W(ky=0) | W(ky=1) | W(ky=2)], accumulators in reverse row order)
//   E1: accumulators -> + b1, ReLU, zero outside the image (conv2 pads the intermediate TENSOR with zeros) -> bf16 / fp16 -> shared
//       memory in the same swizzled pixel-row layout TMA produces, so conv2 addresses it with the same descriptors
//   M2: conv2 from that tile,  E2: + b2 + x (from the staged input tile) -> ReLU -> global.
// Roles (persistent CTA): warp 0 TMA producer (input ring), warp 1 MMA issuer, warps 2-5 / 6-9 the epilogue groups of slot 0 / 1.
// With 16 channels two tiles are in flight per CTA (slot = accumulators + intermediate tile): the MMA issuer polls the slots'
// barriers and issues whichever convolution is ready, so the tensor pipe works on one tile while the other is in an epilogue.
// The accumulators are zeroed by the epilogue that drains them (every MMA accumulates).
#include <algorithm>

#include "hrnet.h"
#include "umma_prims.h"

namespace {

using namespace umma;

constexpr int BW = 128, WO = 126, TW = 130, THREADS = 320;      // TMA warp, MMA warp, 8 epilogue warps
constexpr int al1024(int b) { return (b + 1023) & ~1023; }


// GRES (TF32): the residual x is read from global memory (L2: TMA fetched the same lines a moment ago) in fp32 instead of from the
// staged tile, which TMA rounded to TF32 -- the block then computes what the two separate convolutions compute -- and the input tile is
// free as soon as conv1 has read it, so two buffers serve two slots.
template <int C, int R, int SLOTS, int ESZ = 2, int GRES = 0>
struct BCfg {
  static constexpr int ROWB = ESZ * C;                 // bytes per pixel row of a tile (32 or 64)
  static constexpr int R1 = R + 2, RX = R + 4;         // intermediate rows, input rows
  static constexpr int NX = GRES ? 2 : SLOTS + 1;      // input tile ring: one tile per slot in flight plus one being loaded
  static constexpr int NSG = SLOTS == 1 ? 2 : 1;       // epilogue warp groups per slot: with one slot both groups drain it, half the rows each
  static constexpr int X_BYTES = RX * TW * ROWB, X_AL = al1024(X_BYTES);
  static constexpr int T_BYTES = R1 * TW * ROWB, T_AL = al1024(T_BYTES);
  static constexpr int W_BYTES = 9 * C * ROWB, W_AL = al1024(W_BYTES);
  static constexpr int ACC1 = R1 * C, ACC2 = R * C, ACC = ACC1 + ACC2;
  static constexpr int TMEM_COLS = 512;
  static constexpr int SMEM_BYTES = 1024 + 2 * W_AL + NX * X_AL + SLOTS * T_AL + 2 * C * 4 + 256;
  static constexpr uint32_t LAYOUT = ROWB == 32 ? 6u : 4u;     // SWIZZLE_32B / 64B
  static constexpr uint32_t SWZ = ROWB == 32 ? 1u : 3u;
  static_assert((C == 16 || C == 32) && (ROWB == 32 || ROWB == 64), "channel counts of the fused block");
  static_assert(SLOTS * ACC <= 512, "accumulators exceed TMEM");
  static_assert(SMEM_BYTES <= 232448, "shared memory budget");
};

struct BlockArgs {
  const void *w1, *w2;               // packed like ttk_conv_umma_pack (fused 3x3: [kx][ky][cout][cin])
  const float *b1, *b2;
  const void* x;                     // the block's input (GRES: residual source)
  void* out;
  int n, h, w;
  int tiles_x, tiles_y, total;
};

// RR output rows from RR + 2 staged rows at `abase`, weights at `wbase`, accumulators at `d_acc` (row yo in column block RR-1-yo).
// Called by the whole MMA warp with warp-uniform arguments; the elected lane issues (see conv_umma.cu).
template <int C, int RR, uint32_t LAYOUT, int ESZ, int H>
__device__ __forceinline__ void issue_conv(uint32_t abase, uint32_t wbase, uint32_t d_acc, bool leader) {
  constexpr int ROWB = ESZ * C;
  constexpr uint32_t RB16 = ROWB / 16;
  const uint32_t a16 = abase >> 4, w16 = wbase >> 4;
#pragma unroll 1
  for (int hr = 0; hr < RR + 2; ++hr) {
    const int yi = hr - 1;
    const int k0 = yi + 2 - RR > 0 ? yi + 2 - RR : 0;
    const int k1 = yi + 1 < 2 ? yi + 1 : 2;
    const uint32_t idesc = ESZ == 2 ? make_idesc(128, (k1 - k0 + 1) * C, 0, H) : make_idesc_tf32(128, (k1 - k0 + 1) * C);
    const uint32_t d = d_acc + (RR - 2 - yi + k0) * C;
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const uint32_t arow = a16 + (hr * TW + kx) * RB16;
      const uint32_t brow = w16 + ((kx * 3 + k0) * C) * RB16;
#pragma unroll
      for (int ks = 0; ks < ROWB / 32; ++ks)
        if (leader) {
          if (ESZ == 2) mma(d, make_desc16<8 * ROWB, LAYOUT>(arow + ks * 2), make_desc16<8 * ROWB, LAYOUT>(brow + ks * 2), idesc, 1u);
          else mma_tf32(d, make_desc16<8 * ROWB, LAYOUT>(arow + ks * 2), make_desc16<8 * ROWB, LAYOUT>(brow + ks * 2), idesc, 1u);
        }
    }
  }
}

// Tiles of a CTA are numbered t = 0, 1, 2, ... in the order it takes them; tile t lives in input buffer t % NX and in slot t % SLOTS
// (slot = its own accumulators and intermediate tile, served by its own group of four epilogue warps), so with two slots the MMAs of
// one tile run under the epilogues of the other.  H: the 16-bit format (0 bf16, 1 fp16; umma_prims.h: Fmt16).
template <int C, int R, int SLOTS, int ESZ = 2, int GRES = 0, int H = 0>
__global__ void __launch_bounds__(THREADS, 1) block_umma_kernel(const __grid_constant__ CUtensorMap xmap, const BlockArgs a) {
  using K = BCfg<C, R, SLOTS, ESZ, GRES>;
  using F = Fmt16<H>;
  static_assert(!H || ESZ == 2, "fp16 is a 16-bit element format");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sW1 = smem;
  uint8_t* sW2 = sW1 + K::W_AL;
  uint8_t* sX = sW2 + K::W_AL;                         // NX input tiles
  uint8_t* sT = sX + K::NX * K::X_AL;                  // one intermediate tile per slot
  float* sB1 = reinterpret_cast<float*>(sT + SLOTS * K::T_AL);
  float* sB2 = sB1 + C;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB2 + C);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  const uint32_t bar_xfull = smem_u32(bars), bar_xempty = bar_xfull + 8 * 3, bar_m1 = bar_xempty + 8 * 3, bar_st = bar_m1 + 8 * 2, bar_m2 = bar_st + 8 * 2,
                 bar_init = bar_m2 + 8 * 2;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int my_tiles = a.total > (int)blockIdx.x ? (a.total - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

  // ---- one-time setup: weights (software swizzle on absolute address bits, as TMA does), biases, zeroed intermediate tiles ----
  {
    constexpr int CPR = K::ROWB / 16;
    for (int which = 0; which < 2; ++which) {
      const uint4* src = reinterpret_cast<const uint4*>(which ? a.w2 : a.w1);
      uint8_t* dstb = which ? sW2 : sW1;
      const uint32_t wb = smem_u32(dstb);
      for (int i = tid; i < K::W_BYTES / 16; i += THREADS) {
        uint32_t addr = wb + (i / CPR) * K::ROWB + (i % CPR) * 16;
        addr ^= ((addr >> 7) & K::SWZ) << 4;
        *reinterpret_cast<uint4*>(dstb + (addr - wb)) = __ldg(src + i);
      }
    }
    for (int i = tid; i < C; i += THREADS) sB1[i] = a.b1[i], sB2[i] = a.b2[i];
    for (int i = tid; i < SLOTS * K::T_AL / 16; i += THREADS) reinterpret_cast<uint4*>(sT)[i] = make_uint4(0, 0, 0, 0);
  }
  if (tid == 0) {
    for (int s = 0; s < K::NX; ++s) {
      mbar_init(bar_xfull + 8 * s, 1);
      mbar_init(bar_xempty + 8 * s, GRES ? 1 : 4 * K::NSG);
    }
    for (int k = 0; k < SLOTS; ++k) {
      mbar_init(bar_m1 + 8 * k, 1);
      mbar_init(bar_st + 8 * k, 4 * K::NSG);
      mbar_init(bar_m2 + 8 * k, 1);
    }
    mbar_init(bar_init, 4 * SLOTS * K::NSG);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  fence_async_smem();                                  // weights / zeros: generic-proxy writes -> async proxy (tensor core)
  if (warp == 2) tmem_alloc(smem_u32(tmem_slot), K::TMEM_COLS);
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int t = 0; t < my_tiles; ++t) {
        const int tile = blockIdx.x + t * gridDim.x;
        const int tx = tile % a.tiles_x, ty = (tile / a.tiles_x) % a.tiles_y, img = tile / (a.tiles_x * a.tiles_y);
        const uint32_t s = t % K::NX, ph = (t / K::NX) & 1;
        mbar_wait(bar_xempty + 8 * s, ph ^ 1);
        mbar_expect_tx(bar_xfull + 8 * s, K::X_BYTES);
        tma_load_4d(smem_u32(sX + s * K::X_AL), &xmap, bar_xfull + 8 * s, 0, tx * WO - 2, ty * R - 2, img);
      }
    }
  } else if (warp == 1) {
    {
      const bool leader = elect_one();
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
      mbar_wait(bar_init, 0);                          // accumulators zeroed
      fence_after();
      // per slot: next tile number and whether its conv1 has been issued; a slot advances whenever its barrier has flipped
      int nxt[SLOTS], stage[SLOTS], live = 0;
      for (int k = 0; k < SLOTS; ++k) nxt[k] = k, stage[k] = 0, live += k < my_tiles ? 1 : 0;
      while (live > 0) {
#pragma unroll
        for (int k = 0; k < SLOTS; ++k) {
          const int t = nxt[k];
          if (t >= my_tiles) continue;
          const uint32_t acc1 = tmem_u + k * K::ACC, acc2 = acc1 + K::ACC1;
          if (stage[k] == 0) {
            const uint32_t s = t % K::NX;
            if (!mbar_test(bar_xfull + 8 * s, (t / K::NX) & 1)) continue;
            fence_after();
            issue_conv<C, K::R1, K::LAYOUT, ESZ, H>(smem_u32(sX + s * K::X_AL), smem_u32(sW1), acc1, leader);
            if (leader) commit(bar_m1 + 8 * k);
            if (GRES && leader) commit(bar_xempty + 8 * s);      // nothing else reads the input tile
            __syncwarp();
            stage[k] = 1;
          } else {
            if (!mbar_test(bar_st + 8 * k, (t / SLOTS) & 1)) continue;       // intermediate tile written (and acc1 zeroed again)
            fence_after();
            issue_conv<C, R, K::LAYOUT, ESZ, H>(smem_u32(sT + k * K::T_AL), smem_u32(sW2), acc2, leader);
            if (leader) commit(bar_m2 + 8 * k);
            __syncwarp();
            stage[k] = 0;
            nxt[k] = t + SLOTS;
            if (nxt[k] >= my_tiles) --live;
          }
        }
      }
    }
  } else {
    // epilogue group (warp - 2) / 4 serves slot k (two slots), or half the rows of the only slot; TMEM lane quarter q = warp % 4,
    // thread = pixel of a tile row.  Rows are drained G at a time (64 accumulator columns per TMEM wait) so that the load latency is
    // paid once per group.
    const int q = warp & 3, ge = (warp - 2) >> 2;
    const int k = SLOTS == 1 ? 0 : ge, sg = SLOTS == 1 ? ge : 0;
    constexpr int E1_ROWS = K::R1 / K::NSG, E2_ROWS = R / K::NSG;
    static_assert(K::R1 % K::NSG == 0 && R % K::NSG == 0, "rows split evenly between the epilogue groups");
    const int e1_lo = sg * E1_ROWS, e1_hi = e1_lo + E1_ROWS, e2_lo = sg * E2_ROWS, e2_hi = e2_lo + E2_ROWS;
    const int m = q * 32 + lane;                       // pixel within the tile row = TMEM lane
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    const uint32_t acc1 = tmem + k * K::ACC, acc2 = acc1 + K::ACC1;
    constexpr int G = 64 / C;                          // rows per group
    for (int c = sg * 16; c < K::ACC; c += 16 * K::NSG) tmem_zero16(acc1 + lane_base + c);
    tmem_wait_st();
    float b1r[C], b2r[C];                               // biases in registers (TF32 instantiation; the bf16 ones read shared memory)
    if (ESZ == 4) {
#pragma unroll
      for (int j = 0; j < C; ++j) b1r[j] = sB1[j], b2r[j] = sB2[j];
    }
    fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_init);
    const uint32_t st_base = smem_u32(sT + k * K::T_AL);
    for (int t = k; t < my_tiles; t += SLOTS) {
      const int tile = blockIdx.x + t * gridDim.x;
      const int tx = tile % a.tiles_x, ty = (tile / a.tiles_x) % a.tiles_y, img = tile / (a.tiles_x * a.tiles_y);
      const uint32_t s = t % K::NX, tp = (t / SLOTS) & 1;
      const int x0 = tx * WO, y0 = ty * R;
      // ---- E1: intermediate pixel (y0 - 1 + ri, x0 - 1 + m) ----
      mbar_wait(bar_m1 + 8 * k, tp);
      fence_after();
      const int ix = x0 - 1 + m;
      const bool col_in = ix >= 0 && ix < a.w;
#pragma unroll 1
      for (int r0 = e1_lo; r0 < e1_hi; r0 += G) {
        uint32_t v[G][C];
#pragma unroll
        for (int g = 0; g < G; ++g)
          if (r0 + g < e1_hi) {
#pragma unroll
            for (int c = 0; c < C; c += 16) tmem_ld16(acc1 + lane_base + (K::R1 - 1 - (r0 + g)) * C + c, v[g] + c);
          }
        tmem_wait_ld();
#pragma unroll
        for (int g = 0; g < G; ++g)
          if (r0 + g < e1_hi) {
#pragma unroll
            for (int c = 0; c < C; c += 16) tmem_zero16(acc1 + lane_base + (K::R1 - 1 - (r0 + g)) * C + c);
          }
#pragma unroll
        for (int g = 0; g < G; ++g) {
          const int ri = r0 + g;
          if (ri < e1_hi) {
            const int iy = y0 - 1 + ri;
            const bool inside = col_in && iy >= 0 && iy < a.h;
            uint32_t pk[C * ESZ / 4];
            if (ESZ == 2) {
#pragma unroll
              for (int j = 0; j < C / 2; ++j) {
                const float f0 = inside ? fmaxf(__uint_as_float(v[g][2 * j]) + sB1[2 * j], 0.f) : 0.f;
                const float f1 = inside ? fmaxf(__uint_as_float(v[g][2 * j + 1]) + sB1[2 * j + 1], 0.f) : 0.f;
                pk[j] = F::pack(f0, f1);
              }
            } else {
              // the intermediate is an operand of kind::tf32, which truncates: round it here (to nearest; the integer form of
              // cvt.rna.tf32.f32, exact for these non-negative finite values and a quarter of its instructions)
#pragma unroll
              for (int j = 0; j < C; ++j) {
                const float f0 = inside ? fmaxf(__uint_as_float(v[g][j]) + b1r[j], 0.f) : 0.f;
                pk[j] = (__float_as_uint(f0) + 0x1000u) & 0xFFFFE000u;
              }
            }
            const uint32_t row_ad = st_base + (ri * TW + m) * K::ROWB;
#pragma unroll
            for (int u = 0; u < K::ROWB / 16; ++u) {
              uint32_t ad = row_ad + u * 16;
              ad ^= ((ad >> 7) & K::SWZ) << 4;
              asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(ad), "r"(pk[4 * u]), "r"(pk[4 * u + 1]), "r"(pk[4 * u + 2]), "r"(pk[4 * u + 3]) : "memory");
            }
          }
        }
      }
      tmem_wait_st();
      fence_before();
      fence_async_smem();                              // intermediate tile visible to the tensor core
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_st + 8 * k);
      // ---- E2: output pixel (y0 + r, x0 + m), residual from the staged input tile at (r + 2, m + 2) ----
      const int ox = x0 + m;
      const bool col_ok = m < WO && ox < a.w;
      const uint32_t sx_base = smem_u32(sX + s * K::X_AL);
      // GRES: the fp32 residual rows are requested from global memory (L2) BEFORE the wait for conv2, whose ~1400 clk cover the latency
      // (one row group holds all of E2's rows: R <= G)
      static_assert(!GRES || E2_ROWS <= G, "one residual prefetch per tile");
      uint32_t rv[G][C * ESZ / 4];
      if (GRES) {
#pragma unroll
        for (int g = 0; g < G; ++g) {
          const int oy = y0 + e2_lo + g;
          if (g < E2_ROWS && col_ok && oy < a.h) {
            const char* rp = (const char*)a.x + (((size_t)img * a.h + oy) * a.w + ox) * C * ESZ;
#pragma unroll
            for (int u = 0; u < K::ROWB / 32; ++u) ldg256(rp + 32 * u, rv[g] + 8 * u);
          }
        }
      }
      mbar_wait(bar_m2 + 8 * k, tp);
      fence_after();
#pragma unroll 1
      for (int r0 = e2_lo; r0 < e2_hi; r0 += G) {
        uint32_t v[G][C];
#pragma unroll
        for (int g = 0; g < G; ++g)
          if (r0 + g < e2_hi) {
#pragma unroll
            for (int c = 0; c < C; c += 16) tmem_ld16(acc2 + lane_base + (R - 1 - (r0 + g)) * C + c, v[g] + c);
            if (!GRES) {
              const uint32_t row_ad = sx_base + ((r0 + g + 2) * TW + (m + 2)) * K::ROWB;
#pragma unroll
              for (int u = 0; u < K::ROWB / 16; ++u) {
                uint32_t ad = row_ad + u * 16;
                ad ^= ((ad >> 7) & K::SWZ) << 4;
                asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(rv[g][4 * u]), "=r"(rv[g][4 * u + 1]), "=r"(rv[g][4 * u + 2]), "=r"(rv[g][4 * u + 3]) : "r"(ad));
              }
            }
          }
        tmem_wait_ld();
#pragma unroll
        for (int g = 0; g < G; ++g)
          if (r0 + g < e2_hi) {
#pragma unroll
            for (int c = 0; c < C; c += 16) tmem_zero16(acc2 + lane_base + (R - 1 - (r0 + g)) * C + c);
          }
#pragma unroll
        for (int g = 0; g < G; ++g) {
          const int r = r0 + g;
          const int oy = y0 + r;
          if (r < e2_hi && col_ok && oy < a.h) {
            uint32_t o[C * ESZ / 4];
            if (ESZ == 2) {
#pragma unroll
              for (int j = 0; j < C / 2; ++j) {
                const float f0 = fmaxf(__uint_as_float(v[g][2 * j]) + sB2[2 * j] + F::lo(rv[g][j]), 0.f);
                const float f1 = fmaxf(__uint_as_float(v[g][2 * j + 1]) + sB2[2 * j + 1] + F::hi(rv[g][j]), 0.f);
                o[j] = F::pack(f0, f1);
              }
            } else {
              // the residual is the staged input tile, i.e. x as TMA rounded it to TF32 (2^-12 relative: inside the path's class)
#pragma unroll
              for (int j = 0; j < C; ++j) o[j] = __float_as_uint(fmaxf(__uint_as_float(v[g][j]) + b2r[j] + __uint_as_float(rv[g][j]), 0.f));
            }
            uint4* op = reinterpret_cast<uint4*>((char*)a.out + (((size_t)img * a.h + oy) * a.w + ox) * C * ESZ);
#pragma unroll
            for (int u = 0; u < K::ROWB / 16; ++u) op[u] = make_uint4(o[4 * u], o[4 * u + 1], o[4 * u + 2], o[4 * u + 3]);
          }
        }
      }
      tmem_wait_st();
      fence_before();
      __syncwarp();
      if (!GRES && lane == 0) mbar_arrive(bar_xempty + 8 * s);  // the input tile (residual source) is free
    }
  }
  fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem, K::TMEM_COLS);
}

template <int C, int R, int SLOTS, int ESZ = 2, int GRES = 0, int H = 0>
int launch(const TtkConv& c1, const TtkConv& c2, const void* x, void* y, int n, int h, int w, cudaStream_t st) {
  using K = BCfg<C, R, SLOTS, ESZ, GRES>;
  EncodeFn encode = get_encode();
  if (!encode) {
    ttk_set_error("cuTensorMapEncodeTiled is not available from the driver");
    return TTK_ERR_CUDA;
  }
  static TtkPerDevice attr;
  if (attr.first()) {
    TTK_CUDA(cudaFuncSetAttribute(block_umma_kernel<C, R, SLOTS, ESZ, GRES, H>, cudaFuncAttributeMaxDynamicSharedMemorySize, K::SMEM_BYTES));
  }
  CUtensorMap map;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
  cuuint64_t strides[3] = {(cuuint64_t)C * ESZ, (cuuint64_t)w * C * ESZ, (cuuint64_t)h * w * C * ESZ};
  cuuint32_t box[4] = {(cuuint32_t)C, (cuuint32_t)TW, (cuuint32_t)K::RX, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  if (encode(&map, ESZ == 2 ? Fmt16<H>::MAP : CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 4, const_cast<void*>(x), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
             K::ROWB == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
    ttk_set_error("cuTensorMapEncodeTiled failed for the fused block %s", c1.name.c_str());
    return TTK_ERR_CUDA;
  }
  BlockArgs a;
  if (ESZ == 2 && H) a.w1 = c1.w_umma_f16, a.w2 = c2.w_umma_f16;
  else a.w1 = ESZ == 2 ? (const void*)c1.w_umma : (const void*)c1.w_umma32, a.w2 = ESZ == 2 ? (const void*)c2.w_umma : (const void*)c2.w_umma32;
  a.b1 = c1.bias, a.b2 = c2.bias, a.x = x, a.out = y;
  a.n = n, a.h = h, a.w = w;
  a.tiles_x = ttk_cdiv(w, WO), a.tiles_y = ttk_cdiv(h, R);
  a.total = a.tiles_x * a.tiles_y * n;
  const int grid = std::max(1, std::min(a.total, ttk_num_sms()));
  block_umma_kernel<C, R, SLOTS, ESZ, GRES, H><<<grid, THREADS, K::SMEM_BYTES, st>>>(map, a);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

}  // namespace

// y = relu(conv2(relu(conv1(x))) + x) for two 3x3 stride-1 convolutions with cin = cout = 16 or 32 (padded), NHWC bf16 (esz 2; f16: fp16)
// or, for 16 channels, NHWC fp32 multiplied as TF32 (esz 4).
int ttk_block_umma_launch(const TtkConv& c1, const TtkConv& c2, const void* x, void* y, int n, int h, int w, cudaStream_t st, int esz, bool f16) {
  if (c1.k != 3 || c2.k != 3 || c1.stride != 1 || c2.stride != 1 || c1.cin_p != c1.cout_p || c2.cin_p != c1.cin_p || c2.cout_p != c1.cin_p)
    return TTK_ERR_UNSUPPORTED;
  // TF32 (64-byte rows): two 3-row tiles in flight with the fp32 residual from global memory (esz 4), or one 4-row tile with the residual
  // from the staged tile (esz 5: the first version, kept for comparison)
  if (esz == 4) return c1.cin_p == 16 ? launch<16, 3, 2, 4, 1>(c1, c2, x, y, n, h, w, st) : TTK_ERR_UNSUPPORTED;
  if (esz == 5) return c1.cin_p == 16 ? launch<16, 4, 1, 4, 0>(c1, c2, x, y, n, h, w, st) : TTK_ERR_UNSUPPORTED;
  if (c1.cin_p == 16) return f16 ? launch<16, 6, 2, 2, 0, 1>(c1, c2, x, y, n, h, w, st) : launch<16, 6, 2>(c1, c2, x, y, n, h, w, st);      // two tiles in flight (2 x 224 TMEM columns)
  if (c1.cin_p == 32) return f16 ? launch<32, 4, 1, 2, 0, 1>(c1, c2, x, y, n, h, w, st) : launch<32, 4, 1>(c1, c2, x, y, n, h, w, st);      // 320 TMEM columns per tile: one slot
  return TTK_ERR_UNSUPPORTED;
}
