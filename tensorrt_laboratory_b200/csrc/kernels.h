// Host-visible launch API of the sm_100a kernels (implemented in kernels.cu).
// Internal to libb200infer.so -- the public boundary is include/b200infer.h.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace b2k {

// ---------------------------------------------------------------------------------------------
// implicit-GEMM convolution on tcgen05 tensor cores
//   D[M = batch*Ho*Wo, N = Cout] = A[M, K = taps*Cin] * B[N, K]^T,  fp16 in, fp32 accumulate in TMEM,
//   epilogue: + bias[n] (+ residual[m][n]) -> relu -> fp16 -> NHWC store.
// ---------------------------------------------------------------------------------------------
enum { A_TILED = 0, A_IM2COL = 1 };

struct ConvArgs {
    const float* bias;       // [Cout_phys] fp32 (BN/Scale folded)
    const __half* residual;  // [M][Cout_phys] or nullptr
    __half* out;             // [M][Cout_phys]
    int M;                   // valid output pixels (batch*Ho*Wo)
    int Cout;                // physical output channels = row pitch of out/residual
    int num_kblocks;         // k-blocks of 64 K-elements
    int cblocks;             // KB==64: Cin_phys/64 channel blocks per tap
    int taps;                // real filter taps (kh*kw)
    int taps_phys;           // taps incl. zero-weight padding (even for KB==8)
    int kw;                  // filter width (tap -> (r, s))
    int HoWo, Wo;            // output plane, output width (m -> (img, p, q))
    int stride_h, stride_w;  // conv strides
    int pad_h, pad_w;        // top / left padding
    int relu;
    int a_mode;              // A_TILED (1x1 stride-1: plain 2-D TMA) or A_IM2COL (TMA im2col mode)
    int splits;              // split-K factor (gridDim.z); 1 = none
    int kb_per_split;        // k-blocks per split
    float* workspace;        // splits > 1: [tile][split][128][BN] fp32 partial tiles
    int* tile_counters;      // splits > 1: one arrival counter per output tile (zero between launches)
    int pdl_trigger;         // 0: release the dependent kernel right after the prologue, 1: after the main loop
    const uint8_t* wpacked;  // KB==64: weights as pre-swizzled 4 KiB blocks [num_kblocks][Cout/32][32][128 B]; the BN-wide
                             // tile of one k-block is one contiguous cp.async.bulk (nullptr: fetch through mapB)
    int halo_rows;           // halo variant: output rows R per tile (tile = R rows x (Wo+2) padded columns of one image)
    int cn;                  // CTAs per cluster along N sharing one activation tile by TMA multicast (1 = no cluster)
    int tiles_m, tiles_n;    // persistent variant: output tile grid (128-row x BN-column tiles)
    int dbg_mode;            // bottleneck isolation (debug only): bit0 skip MMA issue, bit1 skip A loads, bit2 skip B loads
    long long* dbg;          // optional per-CTA phase timestamps (16 x int64 per CTA), nullptr in production
};

struct ConvLaunch {
    CUtensorMap mapA;  // activations: 2-D tiled [M, Cin] or 4-D im2col (C, W, H, N)
    CUtensorMap mapB;  // weights: 2-D tiled [Cout_phys, Ktot]
    CUtensorMap mapOut;  // output tile store: 2-D tiled [M, Cout_phys], box 128 x min(64, BN), swizzled
    CUtensorMap mapRes;  // residual tile load: same geometry over the residual tensor (unused when no residual)
    ConvArgs args;
    int bn;            // N tile: 32 / 64 / 128 / 256
    int kb;            // K elements per TMA sub-tile: 64 (SWIZZLE_128B), 32 (SWIZZLE_64B: stem with the filter
                       // row folded into "channels" through an overlapping pixel stride) or 8 (no swizzle)
    int stages;        // smem pipeline depth: 1 / 2 / 4 / 8
    int sps;           // 64-wide K sub-blocks per pipeline stage: 1 or 2 (KB == 64 only)
    int grid_m, grid_n;
    int cn;            // cluster size along N (1, 2 or 4; KB == 64 only): mapA's box is then 128/cn rows
    int halo;          // 1: conv3x3_halo_tcgen05 (3x3 s1 p1; mapA / mapOut are 4-D tiled {C, W, H, N} maps; grid_m = N * ceil(H/R))
    int ws_ctas;       // > 0: persistent warp-specialised variant with this many CTAs (0: one tile per CTA)
};

// returns 0 or a cudaError_t
int launch_conv_f16_tcgen05(const ConvLaunch& L, cudaStream_t stream);
// one-time: opt in to large dynamic shared memory for every instantiation
int init_conv_kernels();
bool conv_config_exists(int bn, int kb, int stages, int sps = 1);  // is this configuration instantiated?
int conv_smem_bytes(int bn, int stages, bool residual, int sps = 1);  // dynamic shared memory of one CTA
bool conv_cluster_config_exists(int bn, int stages, int sps, int cn);  // cluster-multicast instantiations
bool conv_halo_config_exists(int bn);                                // 3x3 halo variant
int conv_halo_smem(int bn, int w, int r, int cblocks);
bool conv_ws_config_exists(int bn, int stages, int sps);             // persistent warp-specialised variant
int conv_ws_smem(int bn, int stages, int sps, bool residual);
// programmatic dependent launch on/off for every kernel of this library (default on)
void set_pdl(bool on);
bool get_pdl();

// ---------------------------------------------------------------------------------------------
// net_f16_tcgen05 -- ONE persistent kernel for a whole run of consecutive convolution layers (net_kernel.cu).
//   The tiles (128 output pixels x BN output channels) of every layer of the run form one ordered work list; CTAs draw
//   tickets from it.  A tile of layer L+1 starts as soon as the 128-row tiles of layer L that it reads are stored
//   (per-(layer, M-tile) arrival counters in global memory) instead of waiting for the whole layer.
// ---------------------------------------------------------------------------------------------
constexpr int kNetMaxLayers = 160;   // layer descriptors are copied to shared memory

struct NetLayerInfo {
    const uint8_t* wpacked;   // pre-swizzled weights [num_kblocks][Cout/32][32][128 B]
    const float* bias;        // [Cout]
    __half* out;              // [M][Cout] NHWC
    const __half* residual;   // [M][Cout] or nullptr
    int M, Cout, num_kblocks, cblocks;
    int kw, HoWo, Wo, stride_h;
    int stride_w, pad_h, pad_w, relu;
    int a_mode, bn, tiles_m, tiles_n;
    int tile_begin, total_tiles;
    int in_flag_off;         // first M-tile counter of the layer that produces the input (-1: produced before this kernel)
    int in_need;             // N tiles per M tile of that layer = value of a complete counter
    int res_flag_off, res_need;  // same for the residual input
    int out_flag_off;        // first M-tile counter of this layer
    int dep_off;             // first entry of this layer in NetArgs::deps
    int war_upto;            // every layer of the run up to this index must be COMPLETE before this layer may store: its output
                             // buffer is recycled arena memory those layers read or wrote (-1: none)
    int pad_[3];
};
static_assert(sizeof(NetLayerInfo) % 16 == 0, "NetLayerInfo is copied to shared memory in 16-byte words");
struct alignas(64) NetLayer {
    CUtensorMap mapA;    // activations: 2-D tiled [M, Cin] (box 128 x 64) or 4-D im2col
    NetLayerInfo info;
};
struct NetArgs {
    const NetLayer* layers;  // device memory
    const short2* deps;      // device: per (layer, M tile) first / last M tile of the input it reads
    int* mt_done;            // device: per (layer, M tile) finished-tile counters (zero between launches)
    int* layer_done;         // device: per layer finished-tile counters (zero between launches)
    int* ctrl;               // device: [0] ticket counter, [1] exited CTAs (zero between launches)
    int n_layers, total_tiles, n_flags;
    int stages;              // shared-memory ring depth (2..4 stages of one 64-wide K-block: 16 KiB of activations + 16 KiB of weights)
    long long* dbg;          // optional (debug instantiation): 8 roles x 8 int64 counters per CTA
};
int init_net_kernel();
int net_smem_bytes(int n_layers, int stages);
// persistent launch with `ctas` CTAs (up to two per SM when the ring is shallow enough); returns 0 or a cudaError_t
int launch_net_f16_tcgen05(const NetArgs& a, int ctas, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// INT8 path (i8_kernels.cu): tcgen05.mma.kind::i8 convolution with a requantising epilogue + its SIMT helpers
// ---------------------------------------------------------------------------------------------
struct I8ConvArgs {
    const uint8_t* wpacked;  // int8 weights as pre-swizzled blocks [num_kblocks][Cout/32][32][128 B] (K-block = 128 bytes)
    const float* m;          // [Cout] fl(s_in * s_w[c] / s_out)
    const float* b;          // [Cout] fl(bias[c] / s_out)
    float r;                 // fl(s_res / s_out) (fused residual)
    int has_res, relu;
    int M, Cout, num_kblocks, cblocks;  // cblocks = Cin_phys / 128
    int kw, HoWo, Wo, stride_h, stride_w, pad_h, pad_w, a_mode;
    // padding that need not be computed: the LAST 128-channel block of every tap holds `last_cb_mmas` (1..4) 32-byte MMA
    // slices of real input channels (the rest is zero), and output channels >= cout_real are padding whose result is zero
    int last_cb_mmas, cout_real;
};
struct I8ConvLaunch {
    CUtensorMap mapA;    // int8 activations: 2-D tiled [M, Cin] (box 128 rows x 128 B) or 4-D im2col
    CUtensorMap mapOut;  // int8 output store: 2-D tiled [M, Cout], box 128 x 128 B, 128B swizzle
    CUtensorMap mapRes;  // int8 residual load, same geometry
    I8ConvArgs args;
    int bn, stages, grid_m, grid_n;  // N tile 128 / 256, shared-memory ring depth 2..4
};
int init_conv_i8_kernels();
bool conv_i8_config_exists(int bn, int stages);
int conv_i8_smem_bytes(int bn, int stages, bool residual);
int launch_conv_i8_tcgen05(const I8ConvLaunch& L, cudaStream_t stream);
// fp16 NHWC -> int8 NHWC, q = clip(rint(fl(float(h) * inv_s)), +-127); channels >= C are written as zeros
int launch_quantize_h_to_i8(const void* src, void* dst, long long pixels, int C, int C_in_phys, int C_out_phys, float inv_s,
                            cudaStream_t stream);
// global average pool int8 NHWC -> fp16 [N][C_out_phys]: h = fp16(fl(float(sum q) * k))
int launch_avgpool_i8(const void* src, void* dst, int N, int HW, int C, int C_in_phys, int C_out_phys, float k, cudaStream_t stream);
// int8 NHWC -> fp32 NCHW binding: y = fl(float(q) * s)
int launch_output_cast_i8(const void* src, float* dst, int N, int C, int H, int W, int C_phys, float s, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// SIMT kernels (reference/fp32 engine path, and the non-GEMM operators of the fp16 path)
// ---------------------------------------------------------------------------------------------
struct SimtConvArgs {
    const void* in;        // NHWC [N,H,W,Cin_phys]
    const void* w;         // [Cout_phys][taps_phys][Cin_phys]
    const float* bias;     // [Cout_phys]
    const void* residual;  // NHWC out-shaped or nullptr
    void* out;             // NHWC [N,Ho,Wo,Cout_phys]
    int N, H, W, Cin, Cin_phys, Ho, Wo, Cout, Cout_phys;
    int kh, kw, taps_phys, stride_h, stride_w, pad_h, pad_w, relu;
    int w_packed;          // 1: `w` uses the pre-swizzled block layout (fp16 engines)
};
int launch_conv_simt(const SimtConvArgs& a, bool half_storage, cudaStream_t stream);

// fp32 NCHW binding -> NHWC activations (zero-filled channel padding)
// (`src_half`: the binding holds fp16 instead of fp32 -- plans built with input_dtype="f16")
// max_blocks > 0 caps the grid (the kernels are grid-stride loops): a cast that reads its source over PCIe (zero-copy
// pinned input) lives for the length of the transfer and must not occupy every thread slot of the machine meanwhile
int launch_input_cast(const void* src, bool src_half, void* dst, int N, int C, int H, int W, int C_phys,
                      bool half_storage, int max_blocks, cudaStream_t stream);
// fp32 NCHW binding -> fp16 [N, H, pad_l + W/2 + pad_r, 8] with channel = dw*4 + c (horizontal space-to-depth, C <= 4;
// border pixels zero)
int launch_input_cast_s2d(const void* src, bool src_half, void* dst, int N, int C, int H, int W, int pad_l, int pad_r,
                          int max_blocks, cudaStream_t stream);
// uint8 HWC image binding: source geometry, crop and normalisation (plan_format.h InputNormRec).  Passed BY VALUE as a
// kernel argument, so the cast reads nothing but the image bytes.
struct U8Norm {
    float mean[4];
    float inv_std[4];
    int C;             // source channels, 1..4
    int src_h, src_w;  // source image
    int top, left;     // crop origin; the crop size is the engine tensor's H x W
    int perm[4];       // output channel c reads source channel perm[c]
};
// uint8 [N, src_h, src_w, C] -> fp16 [N, H, pad_l + W/2 + pad_r, 8], the layout of launch_input_cast_s2d
int launch_input_cast_u8_s2d(const void* src, void* dst, int N, int H, int W, int pad_l, int pad_r, const U8Norm& nrm,
                             int max_blocks, cudaStream_t stream);
// uint8 [N, src_h, src_w, C] -> fp16 NHWC [N, H, W, 8] (zero-filled channels C..7)
int launch_input_cast_u8_c8(const void* src, void* dst, int N, int H, int W, const U8Norm& nrm, int max_blocks,
                            cudaStream_t stream);
// NHWC activations -> fp32 NCHW binding
int launch_output_cast(const void* src, float* dst, int N, int C, int H, int W, int C_phys,
                       bool half_storage, cudaStream_t stream);
int launch_maxpool(const void* src, void* dst, int N, int H, int W, int C_phys, int Ho, int Wo, int k,
                   int stride, int pad, bool half_storage, cudaStream_t stream);
// global average pool: NHWC [N,HW,C] -> [N,1,1,C]
int launch_avgpool(const void* src, void* dst, int N, int HW, int C_phys, bool half_storage,
                   cudaStream_t stream);
// out[n][j] = bias[j] + sum_k in[n][k]*w[j][k]   (in: activations, K = HW*C_phys; out fp32 [N][Cout])
int launch_fc(const void* in, const void* w, const float* bias, float* out, int N, int K, int Cout,
              bool half_storage, cudaStream_t stream);
int launch_softmax(const float* in, float* out, int N, int C, cudaStream_t stream);

// global average pool + FC + bias + softmax in one launch (fp16 engines; tail_f16_kernel in kernels.cu)
struct TailArgs {
    const __half* in;     // [N][HW][C] NHWC activations
    const __half* w;      // [Cout][C]
    const float* bias;    // [Cout]
    float* out;           // [N][Cout] softmax (the output binding)
    __half* pooled;       // [N][C] scratch (the pooled activation tensor of the plan)
    float* logits;        // [N][Cout] scratch (the FC output vector of the plan)
    int* ctrl;            // 4 ints, zero between launches: ticket, finished pool items, finished FC items, exited CTAs
    int N, HW, C, Cout;
};
bool tail_f16_applies(int N, int HW, int C, int Cout);
int launch_tail_f16(const TailArgs& a, cudaStream_t stream);

}  // namespace b2k
