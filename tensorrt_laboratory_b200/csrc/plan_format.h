// On-disk / in-memory layout of a B2ENGINE plan ("serialized engine").
// Written by tensorrt_laboratory_b200/builder.py, read by engine.cu.  Little-endian, fixed-size records.
// It plays the role of the TensorRT plan file the reference reads in
// trtlab/tensorrt/src/runtime.cc:62-95 (file -> deserializeCudaEngine).
#pragma once
#include <stdint.h>

namespace b2plan {

constexpr char kMagic[8] = {'B', '2', 'E', 'N', 'G', 'I', 'N', 'E'};
constexpr uint32_t kVersion = 1;

enum OpType : uint32_t {
    OP_INPUT_CAST = 0,   // fp32 NCHW binding -> NHWC activation tensor
    OP_CONV = 1,         // conv + folded BN/Scale bias (+ residual) (+ ReLU)
    OP_MAXPOOL = 2,
    OP_AVGPOOL = 3,      // global average pool
    OP_FC = 4,           // inner product -> fp32 vector
    OP_SOFTMAX = 5,      // fp32 vector -> fp32 vector
    OP_OUTPUT_CAST = 6,  // NHWC activation tensor -> fp32 NCHW binding (dequantised when the tensor is int8)
    OP_QUANTIZE = 7,     // fp16 NHWC tensor -> int8 NHWC tensor (INT8 engines: in front of the first int8 convolution)
};

enum TensorKind : uint32_t { T_ACT = 0 /* NHWC, engine precision */, T_VEC = 1 /* [N, c] fp32 */ };

#pragma pack(push, 1)
struct Header {  // 128 bytes
    char magic[8];
    uint32_t version;
    uint32_t precision;  // B2_PREC_*
    uint32_t max_batch;
    uint32_t n_tensors;
    uint32_t n_ops;
    uint32_t n_bindings;
    uint64_t payload_offset;  // from blob start, 256-byte aligned
    uint64_t payload_bytes;
    char name[64];
    // optional tactic table (the role of the tactics a TensorRT plan carries): n_tactics TacticRec records at
    // tactics_offset from the blob start, behind the weight payload.  0 / 0 = none (tune at load, or cost model)
    uint32_t n_tactics;
    uint32_t reserved;
    uint64_t tactics_offset;
};
struct TacticRec {  // 40 bytes: the measured-best kernel configuration of one (conv op, batch)
    uint32_t op, batch, bn, stages, splits, sps, ws, cn, halo, reserved;
};
struct TensorRec {  // 96 bytes
    char name[64];
    uint32_t kind;
    uint32_t h, w, c, c_phys;
    int32_t binding;  // >= 0: storage is bindings[binding] (T_VEC only), -1: activation arena
    float scale;      // INT8 engines: > 0 marks an int8 tensor (1 byte per element, real value = q * scale); 0 = fp16 / fp32
    uint8_t pad[4];
};
struct OpRec {  // 176 bytes
    char name[64];
    uint32_t type;
    int32_t in, res, out;  // tensor indices (-1 = none)
    int32_t binding;       // cast ops: binding index
    uint32_t k, stride, pad_;
    uint32_t relu;         // bit 0: fused ReLU.  bit 2 (convs): INT8 convolution -- int8 weights in 128-byte K blocks, and the
                           // "bias" region holds [m: cout_phys fp32][b: cout_phys fp32][r, 0, 0, 0] (quantize.py).
                           // bit 1 (convs): weights are stored as pre-swizzled 4 KiB blocks
                           // [K/64][Cout/32][32 rows][128 B] (builder.pack_weights_sw128) instead of row-major [Cout][K]
    uint32_t ceil_mode;    // pools: Caffe ceil mode.  convs: algorithmic K (Cin*kh*kw of the ORIGINAL conv) when the
                           // builder re-expressed the layer (0 = cin*taps)
    uint32_t cin, cout, cin_phys, cout_phys, taps, taps_phys;
    uint64_t w_off, w_bytes, b_off, b_bytes;  // payload-relative
    // rectangular / anisotropic convs (0 = square: kw=k, stride_w=stride, pad_w_*=pad_).  `k`, `stride`, `pad_`
    // then describe the H direction.  INPUT_CAST: k = horizontal space-to-depth factor (0/1 = none, 2 = pack pixel
    // pairs into channels [dw*4 + c]).  INPUT_CAST of a B2_DT_UINT8 binding: b_off / b_bytes address its InputNormRec
    // (b_bytes = 48); 0 / 0 for every other input binding.
    uint32_t kw, stride_w, pad_w_lo, pad_w_hi;
};
// Normalisation of a uint8 HWC image binding (C <= 4), per item:
//     y[c][h][w] = (float(x[crop_top + h][crop_left + w][perm[c]]) - mean[c]) * inv_std[c]      (fp32: one sub, one mul)
// (H, W) is the crop = the engine tensor's geometry.  Entries c >= C are 0.
struct InputNormRec {  // 48 bytes
    float mean[4];
    float inv_std[4];
    uint32_t crop_top, crop_left;
    uint8_t perm[4];
    uint8_t pad[4];
};
struct BindingRec {  // 128 bytes
    char name[64];
    uint32_t is_input;
    uint32_t dtype;   // B2_DT_*
    int32_t tensor;   // tensor it feeds / is fed by
    uint32_t nd;
    int32_t dims[8];  // per batch item
    uint8_t pad[16];
};
#pragma pack(pop)

static_assert(sizeof(Header) == 128, "Header size");
static_assert(sizeof(TacticRec) == 40, "TacticRec size");
static_assert(sizeof(TensorRec) == 96, "TensorRec size");
static_assert(sizeof(OpRec) == 176, "OpRec size");
static_assert(sizeof(BindingRec) == 128, "BindingRec size");
static_assert(sizeof(InputNormRec) == 48, "InputNormRec size");

}  // namespace b2plan
