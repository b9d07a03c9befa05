// sm_100a kernels of the B200-native inference engine.
//
//  * conv_f16_tcgen05 -- implicit-GEMM convolution: TMA (tiled or im2col mode) -> 128B-swizzled smem ->
//    tcgen05.mma (UMMA 128xBNx16, fp16 x fp16 -> fp32 in TMEM) -> tcgen05.ld epilogue with
//    bias / residual / ReLU fused -> 128-bit NHWC stores.  One 128xBN output tile per CTA,
//    warp 0 = TMA producer, warp 1 = MMA issuer, warp 2 = TMEM allocator, all 4 warps = epilogue.
//  * SIMT kernels -- fp32-engine reference path (fp64 accumulate) and the non-GEMM operators
//    (layout casts, max/avg pool, FC, softmax).
//
// Replaces the forward pass the reference delegates to TensorRT:
// trtlab/tensorrt/src/workspace.cc:47,52 (enqueueV2) / examples/10_Internals/README.md:50-52.
#include "kernels.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "ptx_sm100.cuh"

namespace b2k {

// SPS = 64-wide K sub-blocks per pipeline stage (1 or 2): one mbarrier round trip (~150-200 cycles of wait +
// commit on the single issuing thread) is then amortised over 128 K-elements instead of 64.
template <int BN, int STAGES, int SPS = 1>
struct ConvCfg {
    static constexpr int A_SUBBLK = 128 * 64 * 2;  // 16 KiB: 128 rows x 64 K-elements
    static constexpr int B_SUBBLK = BN * 64 * 2;
    static constexpr int A_STAGE = SPS * A_SUBBLK;
    static constexpr int B_STAGE = SPS * B_SUBBLK;
    static constexpr int TMEM_COLS = BN < 32 ? 32 : BN;
    static constexpr int PIPE_BYTES = STAGES * (A_STAGE + B_STAGE);
    static constexpr int TILE_BYTES = 128 * BN * 2;  // one fp16 output (or residual) tile
    static_assert(TILE_BYTES <= PIPE_BYTES, "the output staging tile reuses the pipeline buffers");
};

// smem: [A stages][B stages][residual tile (optional)][barriers 256 B][bias BN x 4 B]; +1 KiB alignment slack
__host__ __device__ constexpr int conv_smem_layout_bytes(int bn, int stages, bool residual, int sps = 1) {
    return stages * sps * (128 * 64 * 2 + bn * 64 * 2) + (residual ? 128 * bn * 2 : 0) + 256 + bn * 4 + 1024;
}

// AV resolves the operand paths at compile time for the production instantiations: 1 = im2col-mode activations + packed
// weights, 2 = tiled activations + packed weights, 0 = decided at run time from ConvArgs (thin-K paths, unpacked plans,
// clusters, debug).
template <int BN, int KB, int STAGES, int SPS, int CN = 1, bool DBG = false, int AV = 0>
__global__ void __launch_bounds__(128)
conv_f16_tcgen05(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                 const __grid_constant__ CUtensorMap mapOut, const __grid_constant__ CUtensorMap mapRes,
                 const ConvArgs p) {
    static_assert(SPS == 1 || KB == 64, "multi-sub-block stages exist for the 64-wide K path only");
    using Cfg = ConvCfg<BN, STAGES, SPS>;
    constexpr int TPS = 64 / KB;            // TMA sub-tiles per stage: 1 (KB=64), 2 (KB=32 row-folded stem), 8 (KB=8)
    constexpr int A_SUB = 128 * KB * 2;     // bytes of one A sub-tile
    constexpr int B_SUB = BN * KB * 2;
    constexpr int NG = BN / 32;             // 32-column groups of the accumulator
    constexpr int OW = BN >= 64 ? 64 : 32;  // columns per output TMA box
    constexpr int OROWB = OW * 2;           // bytes per staged output row (128 or 64)
    constexpr int NBOX = BN / OW;
    constexpr uint32_t IDESC = make_idesc_f16(128, BN);

    extern __shared__ uint8_t smem_raw[];
    // 1 KiB alignment by OFFSETTING the __shared__ array (a uintptr_t round trip would turn every later access into a
    // generic LD.E / ST.E instead of LDS / STS)
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const bool has_res = p.residual != nullptr;
    uint8_t* sA = smem;
    uint8_t* sB = smem + STAGES * Cfg::A_STAGE;
    uint8_t* sOut = smem;                    // output staging reuses the (drained) pipeline buffers
    uint8_t* sRes = smem + Cfg::PIPE_BYTES;  // residual tile, only when has_res
    uint8_t* tail = sRes + (has_res ? Cfg::TILE_BYTES : 0);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* accum_bar = empty_bar + STAGES;
    uint64_t* res_bar = accum_bar + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bar + 1);
    uint32_t* last_flag = tmem_slot + 1;
    float* s_bias = reinterpret_cast<float*>(tail + 256);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN;
    const int m0 = blockIdx.y * 128;
    // phase timestamps / bottleneck-isolation switches exist only in the DBG instantiations: even never-taken uniform
    // branches inside the single-thread producer and MMA loops are measurable (see profiles/README.md, A/B runs)
    long long* dbg = (DBG && p.dbg) ? p.dbg + 16ll * ((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) : nullptr;
    if (dbg && threadIdx.x == 0) {
        dbg[0] = clock64();
        unsigned long long gt;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
        dbg[8] = static_cast<long long>(gt);
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        dbg[10] = smid;
    }
    const int kb_begin = blockIdx.z * p.kb_per_split;
    const int kb_end = min(p.num_kblocks, kb_begin + p.kb_per_split);
    const int nk = (kb_end - kb_begin + SPS - 1) / SPS;  // pipeline steps (each covers up to SPS 64-wide K-blocks)
    auto subs_in_step = [&](int i) -> int {            // 64-wide K-blocks in pipeline step i
        const int rem = (kb_end - kb_begin) - i * SPS;
        return rem < SPS ? rem : SPS;
    };
    const bool split = p.splits > 1;
    static_assert(AV == 0 || (KB == 64 && CN == 1 && !DBG), "resolved operand paths exist for the plain 64-wide K kernels");
    const bool a_tiled = AV == 2 ? true : (AV == 1 ? false : p.a_mode == A_TILED);
    const bool w_packed = AV != 0 ? true : p.wpacked != nullptr;
    // Cluster of `cn` CTAs along N (same 128 output pixels, different output-channel tiles): every CTA fetches 1/cn of
    // each activation sub-block and multicasts it to all of them, so L2 serves the tile once per cluster instead of once
    // per CTA.  A stage may be refilled only when EVERY CTA has consumed it -> the MMA warps multicast their stage
    // release and the empty barriers count cn arrivals.
    // (compile-time: the one-CTA instantiations carry none of the cluster code in their loops)
    static_assert(CN == 1 || KB == 64, "clusters exist for the 64-wide K path only");
    constexpr int cn = CN;
    const uint32_t crank = cn > 1 ? cluster_ctarank() : 0u;
    constexpr uint16_t cmask = static_cast<uint16_t>((1u << cn) - 1u);

    // ---------------- prologue: nothing here depends on the previous kernel's output ----------------
    if (threadIdx.x == 0) {
        tma_prefetch_desc(&mapA);
        tma_prefetch_desc(&mapB);
        tma_prefetch_desc(&mapOut);
        if (has_res) tma_prefetch_desc(&mapRes);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], static_cast<uint32_t>(cn));
        }
        mbar_init(accum_bar, 1);
        mbar_init(res_bar, 1);
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 2) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    if (cn > 1) cluster_sync_all();  // peers' barriers exist before anything is multicast at them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 3) {  // bias -> smem while the pipeline spins up; published by the pre-epilogue barrier
#pragma unroll
        for (int i = 0; i < BN / 32; ++i) s_bias[lane + 32 * i] = __ldg(p.bias + n0 + lane + 32 * i);
    }
    if (p.pdl_trigger == 0) pdl_launch_dependents();
    if (dbg && threadIdx.x == 0) dbg[1] = clock64();

    auto sub_tiles = [&](int kb) -> int {  // TMA sub-tiles (filter taps / tap rows) in k-block kb
        if (KB == 64) return 1;
        const int n = p.taps_phys - kb * TPS;
        return n > TPS ? TPS : n;
    };
    const bool skip_mma = DBG && (p.dbg_mode & 1), skip_a = DBG && KB == 64 && (p.dbg_mode & 2),
               skip_b = DBG && KB == 64 && (p.dbg_mode & 4);
    // step i of the pipeline covers K-blocks kb_begin + i*SPS ... ; `kb` below is always the FIRST K-block of a step
    auto stage_bytes = [&](int kb) -> uint32_t {
        if (KB == 64) {
            const int ns = subs_in_step((kb - kb_begin) / SPS);
            return static_cast<uint32_t>(ns * ((skip_a ? 0 : Cfg::A_SUBBLK) + (skip_b ? 0 : Cfg::B_SUBBLK)));
        }
        return static_cast<uint32_t>(sub_tiles(kb) * (A_SUB + B_SUB));
    };
    auto load_b = [&](int kb, int s) {  // weights: constant data, legal before pdl_wait()
        if (skip_b) return;
        uint8_t* b_dst = sB + s * Cfg::B_STAGE;
        if (KB == 64) {
            const int ns = subs_in_step((kb - kb_begin) / SPS);
            for (int u = 0; u < ns; ++u) {
                if (w_packed) {  // one contiguous run of BN/32 pre-swizzled 4 KiB blocks
                    bulk_load_1d(&full_bar[s], b_dst + u * Cfg::B_SUBBLK,
                                 p.wpacked + (static_cast<size_t>(kb + u) * (p.Cout >> 5) + (n0 >> 5)) * 4096, BN * 128);
                } else {
                    tma_load_2d(&mapB, &full_bar[s], b_dst + u * Cfg::B_SUBBLK, (kb + u) * 64, n0);
                }
            }
        } else {
            const int nt = sub_tiles(kb);
            for (int t = 0; t < nt; ++t) tma_load_2d(&mapB, &full_bar[s], b_dst + t * B_SUB, (kb * TPS + t) * KB, n0);
        }
    };
    auto load_residual = [&]() {  // residual tile -> smem, same box geometry as the output store
        mbar_expect_tx(res_bar, Cfg::TILE_BYTES);
#pragma unroll
        for (int b = 0; b < NBOX; ++b) tma_load_2d(&mapRes, res_bar, sRes + b * (128 * OROWB), n0 + b * OW, m0);
    };

    if (warp == 0) {
        {
            // ================= TMA producer (whole warp converged, one elected lane issues) =================
            int img0 = 0, p0 = 0, q0 = 0;
            const int slice_rows = 128 / cn;                 // rows of the A tile this CTA fetches (all of them: cn == 1)
            int ms = m0 + static_cast<int>(crank) * slice_rows;  // first output pixel of the slice
            const uint32_t slice_off = crank * static_cast<uint32_t>(slice_rows) * 128u;  // 128-byte swizzled rows
            if (!a_tiled) {
                if (ms >= p.M) ms = 0;  // slice entirely past the last pixel: its rows are never stored, fetch valid ones
                img0 = ms / p.HoWo;
                const int rem = ms - img0 * p.HoWo;
                p0 = rem / p.Wo;
                q0 = rem - p0 * p.Wo;
            }
            const int base_w = q0 * p.stride_w - p.pad_w;
            const int base_h = p0 * p.stride_h - p.pad_h;
            // K-block -> (filter row r, filter column sx, channel block cb), advanced incrementally: integer division
            // by a run-time value costs ~100 cycles and this thread's issue rate paces the whole main loop
            int cur_cb = 0, cur_r = 0, cur_sx = 0;
            if (KB == 64) {
                const int tap0 = kb_begin / p.cblocks;
                cur_cb = kb_begin - tap0 * p.cblocks;
                cur_r = tap0 / p.kw;
                cur_sx = tap0 - cur_r * p.kw;
            }
            auto load_a = [&](int kb, int s) {  // must be called with consecutive kb starting at kb_begin
                if (skip_a) return;
                uint8_t* a_dst = sA + s * Cfg::A_STAGE;
                if (KB == 64) {
                    const int ns = subs_in_step((kb - kb_begin) / SPS);
                    for (int u = 0; u < ns; ++u) {
                        if (cn > 1) {
                            if (a_tiled) {
                                tma_load_2d_mc(&mapA, &full_bar[s], a_dst + u * Cfg::A_SUBBLK + slice_off, cur_cb * 64, ms, cmask);
                            } else {
                                tma_load_im2col_4d_mc(&mapA, &full_bar[s], a_dst + u * Cfg::A_SUBBLK + slice_off, cur_cb * 64, base_w,
                                                      base_h, img0, static_cast<uint16_t>(cur_sx), static_cast<uint16_t>(cur_r), cmask);
                            }
                        } else if (a_tiled) {
                            tma_load_2d(&mapA, &full_bar[s], a_dst + u * Cfg::A_SUBBLK, cur_cb * 64, m0);
                        } else {
                            tma_load_im2col_4d(&mapA, &full_bar[s], a_dst + u * Cfg::A_SUBBLK, cur_cb * 64, base_w, base_h, img0,
                                               static_cast<uint16_t>(cur_sx), static_cast<uint16_t>(cur_r));
                        }
                        if (++cur_cb == p.cblocks) {
                            cur_cb = 0;
                            if (++cur_sx == p.kw) {
                                cur_sx = 0;
                                ++cur_r;
                            }
                        }
                    }
                } else {
                    const int nt = sub_tiles(kb);
                    for (int t = 0; t < nt; ++t) {
                        const int tap = kb * TPS + t;
                        const int tap_a = tap < p.taps ? tap : p.taps - 1;  // padded tap: weights are zero
                        const int r = tap_a / p.kw;
                        const int sx = tap_a - r * p.kw;
                        tma_load_im2col_4d(&mapA, &full_bar[s], a_dst + t * A_SUB, 0, base_w, base_h, img0,
                                           static_cast<uint16_t>(sx), static_cast<uint16_t>(r));
                    }
                }
            };
            // For 64-wide K-blocks the weights have their own issuing thread (warp 3): one thread needs ~200 cycles
            // per TMA instruction, which is what paces the main loop.
            constexpr bool kSplitProducers = KB == 64;
            const int npre = nk < STAGES ? nk : STAGES;
            if (elect_one_sync()) {
                for (int i = 0; i < npre; ++i) {  // first ring pass: weights fly while the previous kernel drains
                    mbar_expect_tx(&full_bar[i], stage_bytes(kb_begin + i * SPS));
                    if (!kSplitProducers) load_b(kb_begin + i * SPS, i);
                }
            }
            __syncwarp();
            pdl_wait();
            if (dbg && lane == 0) dbg[2] = clock64();
            if (elect_one_sync()) {
                for (int i = 0; i < npre; ++i) load_a(kb_begin + i * SPS, i);
                if (has_res && !split) load_residual();
            }
            __syncwarp();
            long long tw = 0, te = 0, tl = 0;
            for (int i = npre; i < nk; ++i) {
                const int s = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                long long c0 = 0, c1 = 0, c3 = 0;
                if (dbg) c0 = clock64();
                mbar_wait(&empty_bar[s], ph ^ 1);
                if (dbg) c1 = clock64();
                if (elect_one_sync()) {
                    mbar_expect_tx(&full_bar[s], stage_bytes(kb_begin + i * SPS));
                    load_a(kb_begin + i * SPS, s);
                    if (!kSplitProducers) load_b(kb_begin + i * SPS, s);
                }
                __syncwarp();
                if (dbg) {
                    c3 = clock64();
                    tw += c1 - c0, tl += c3 - c1;
                }
            }
            if (dbg && lane == 0) dbg[11] = tw, dbg[12] = te, dbg[13] = tl;
        }
        __syncwarp();
    } else if (warp == 1) {
        {
            // ================= MMA issuer (whole warp converged, one elected lane issues) =================
            long long mw = 0, mi = 0;
            for (int i = 0; i < nk; ++i) {
                const int s = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                long long m0c = 0, m1c = 0;
                if (dbg) m0c = clock64();
                mbar_wait(&full_bar[s], ph);
                tc_fence_after();
                if (dbg) m1c = clock64(), mw += m1c - m0c;
                if (dbg && i == 0 && lane == 0) dbg[3] = clock64();
                const uint32_t a_addr = smem_u32(sA + s * Cfg::A_STAGE);
                const uint32_t b_addr = smem_u32(sB + s * Cfg::B_STAGE);
                if (elect_one_sync()) {
                if (skip_mma) {
                } else if (KB == 64) {
                    const int ns = subs_in_step(i);
#pragma unroll
                    for (int u = 0; u < SPS; ++u) {
                        if (u < ns) {
#pragma unroll
                            for (int j = 0; j < 4; ++j) {  // 4 x (K = 16) inside one 128-byte swizzle row
                                const uint64_t ad = make_smem_desc(a_addr + u * Cfg::A_SUBBLK + j * 32, 16, 1024, 2);
                                const uint64_t bd = make_smem_desc(b_addr + u * Cfg::B_SUBBLK + j * 32, 16, 1024, 2);
                                umma_f16(tmem_base, ad, bd, IDESC, (i > 0 || u > 0 || j > 0) ? 1u : 0u);
                            }
                        }
                    }
                } else if (KB == 32) {
                    // row-folded stem: each sub-tile is one filter row = 32 K-elements in 64-byte swizzled rows
                    const int nt = sub_tiles(kb_begin + i);
                    for (int t = 0; t < nt; ++t) {
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            const uint64_t ad = make_smem_desc(a_addr + t * A_SUB + j * 32, 16, 512, 4);
                            const uint64_t bd = make_smem_desc(b_addr + t * B_SUB + j * 32, 16, 512, 4);
                            umma_f16(tmem_base, ad, bd, IDESC, (i > 0 || t > 0 || j > 0) ? 1u : 0u);
                        }
                    }
                } else {
                    const int nt = sub_tiles(kb_begin + i);
                    for (int j = 0; j < nt / 2; ++j) {  // one K=16 step = two 8-channel taps
                        const uint64_t ad = make_smem_desc(a_addr + 2 * j * A_SUB, A_SUB, 128, 0);
                        const uint64_t bd = make_smem_desc(b_addr + 2 * j * B_SUB, B_SUB, 128, 0);
                        umma_f16(tmem_base, ad, bd, IDESC, (i > 0 || j > 0) ? 1u : 0u);
                    }
                }
                if (cn > 1) umma_commit_mc(&empty_bar[s], cmask);  // every producer of the cluster hears it
                else umma_commit(&empty_bar[s]);                   // frees the smem stage when these MMAs retire
                }
                __syncwarp();
                if (dbg) mi += clock64() - m1c;
            }
            if (elect_one_sync()) umma_commit(accum_bar);  // accumulator complete
            __syncwarp();
            if (dbg && lane == 0) dbg[4] = clock64(), dbg[14] = mw, dbg[15] = mi;
        }
        __syncwarp();
    }

    else if (warp == 3 && KB == 64) {
        // ================= weight producer: constants, so no dependency wait; only the ring's empty barriers ====
        for (int i = 0; i < nk; ++i) {
            const int s = i % STAGES;
            if (i >= STAGES) mbar_wait(&empty_bar[s], ((i / STAGES) & 1) ^ 1);
            if (elect_one_sync()) load_b(kb_begin + i * SPS, s);
            __syncwarp();
        }
    }

    // ====== epilogue: TMEM -> registers -> bias/residual/ReLU -> fp16 -> swizzled smem tile -> TMA store ======
    pdl_wait();  // every global access below depends on the previous kernel
    const int row = warp * 32 + lane;

    mbar_wait(accum_bar, 0);  // all MMAs retired: the pipeline buffers are free to become the output staging tile
    tc_fence_after();
    __syncthreads();          // s_bias visible; every role has left its loop
    if (dbg && threadIdx.x == 64) dbg[5] = clock64();
    if (p.pdl_trigger == 1) pdl_launch_dependents();
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);

    // bias + residual + relu for 32 columns of this thread's row, packed into the staging tile
    auto finish_group = [&](int g, float (&f)[32]) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int col = g * 32 + q * 8;       // column inside the BN-wide tile
            const int box = col / OW;             // which 64- (or 32-) column TMA box
            const int chunk = (col % OW) / 8;     // 16-byte chunk inside the box row
            const uint32_t so = static_cast<uint32_t>(box * (128 * OROWB)) + swz_off<OROWB>(row, chunk);
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = f[q * 8 + i] + s_bias[col + i];
            if (has_res) {
                const uint4 rv = *reinterpret_cast<const uint4*>(sRes + so);
                const __half2* r2 = reinterpret_cast<const __half2*>(&rv);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float2 rf = __half22float2(r2[i]);
                    v[2 * i] += rf.x;
                    v[2 * i + 1] += rf.y;
                }
            }
            if (p.relu) {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = fmaxf(v[i], 0.0f);
            }
            uint4 o;
            __half2* o2 = reinterpret_cast<__half2*>(&o);
#pragma unroll
            for (int i = 0; i < 4; ++i) o2[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
            *reinterpret_cast<uint4*>(sOut + so) = o;
        }
    };

    bool do_store = true;
    if (!split) {
        if (has_res) mbar_wait(res_bar, 0);
        constexpr int GP = NG >= 2 ? 2 : 1;  // groups per TMEM round trip
#pragma unroll
        for (int g0 = 0; g0 < NG; g0 += GP) {
            uint32_t acc[GP][32];
#pragma unroll
            for (int j = 0; j < GP; ++j) tmem_ld32(taddr + (g0 + j) * 32, acc[j]);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < GP; ++j) {
                float f[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(acc[j][i]);
                finish_group(g0 + j, f);
            }
        }
    } else {
        // ---- split-K: publish the fp32 partial tile, the last CTA of the tile reduces IN FIXED ORDER ----
        const int tile = blockIdx.y * gridDim.x + blockIdx.x;
        float* ws_tile = p.workspace + static_cast<size_t>(tile) * p.splits * (128 * BN);
        float* mine = ws_tile + static_cast<size_t>(blockIdx.z) * (128 * BN) + static_cast<size_t>(row) * BN;
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            uint32_t acc[32];
            tmem_ld32(taddr + g * 32, acc);
            tmem_wait_ld();
#pragma unroll
            for (int q = 0; q < 8; ++q)
                __stcg(reinterpret_cast<uint4*>(mine + g * 32) + q, make_uint4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]));
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();  // cumulative: orders the whole CTA's partial-tile stores before the arrival
            const int prev = atomicAdd(p.tile_counters + tile, 1);
            const uint32_t last = (prev == p.splits - 1) ? 1u : 0u;
            if (last) {
                p.tile_counters[tile] = 0;  // re-arm for the next launch
                if (has_res) load_residual();
            }
            *last_flag = last;
        }
        __syncthreads();
        do_store = *last_flag != 0;
        if (do_store) {
            __threadfence();
            if (has_res) mbar_wait(res_bar, 0);
#pragma unroll
            for (int g = 0; g < NG; ++g) {
                float f[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) f[i] = 0.f;
                for (int sp = 0; sp < p.splits; sp += 2) {  // two partial tiles (16 x 16 B) in flight per step
                    const float4* s0 = reinterpret_cast<const float4*>(ws_tile + static_cast<size_t>(sp) * (128 * BN) +
                                                                       static_cast<size_t>(row) * BN + g * 32);
                    const bool two = sp + 1 < p.splits;
                    const float4* s1 = two ? s0 + (128 * BN) / 4 : s0;
                    float4 t0[8], t1[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) t0[q] = __ldcg(s0 + q);
#pragma unroll
                    for (int q = 0; q < 8; ++q) t1[q] = two ? __ldcg(s1 + q) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int q = 0; q < 8; ++q) {  // fixed order: split sp, then split sp+1
                        f[4 * q] = (f[4 * q] + t0[q].x) + t1[q].x;
                        f[4 * q + 1] = (f[4 * q + 1] + t0[q].y) + t1[q].y;
                        f[4 * q + 2] = (f[4 * q + 2] + t0[q].z) + t1[q].z;
                        f[4 * q + 3] = (f[4 * q + 3] + t0[q].w) + t1[q].w;
                    }
                }
                finish_group(g, f);
            }
        }
    }
    if (dbg && threadIdx.x == 64) dbg[6] = clock64();
    if (p.pdl_trigger == 2) pdl_launch_dependents();  // latest useful point: only the output store is left
    fence_proxy_async();  // generic-proxy smem writes -> visible to the TMA (async proxy)
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
    if (threadIdx.x == 0 && do_store) {
        // rows >= M and nothing else are clipped by the tensor map; one bulk store per 64-column box
#pragma unroll
        for (int b = 0; b < NBOX; ++b) tma_store_2d(&mapOut, sOut + b * (128 * OROWB), n0 + b * OW, m0);
        tma_store_commit_and_wait_read();  // smem must stay alive until the TMA has read it
    }
    if (cn > 1) {
        // peers arrive on THIS CTA's empty barriers when their MMAs retire: hear the last release of every stage before
        // the shared memory can go to another CTA, then leave together
        if (warp == 1) {
            const int first = nk > STAGES ? nk - STAGES : 0;
            for (int i = first; i < nk; ++i) mbar_wait(&empty_bar[i % STAGES], (i / STAGES) & 1);
        }
        __syncthreads();
        cluster_sync_all();
    }
    if (dbg && threadIdx.x == 64) {
        dbg[7] = clock64();
        unsigned long long gt;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
        dbg[9] = static_cast<long long>(gt);
    }
}

// =================================================================================================
// conv_f16_tcgen05_ws -- persistent, warp-specialised variant (a TACTIC next to the one-tile-per-CTA kernel).
//   gridDim.x CTAs walk the tile list with a static stride.  12 warps:
//     warp 0  activation producer (TMA)                              warp 1  MMA issuer
//     warp 2  weight producer (cp.async.bulk) + TMEM owner           warp 3  residual producer (TMA)
//     warps 4-7   epilogue group 0: the CTA's even tiles, accumulator 0, staging / residual buffer 0
//     warps 8-11  epilogue group 1: the odd tiles, accumulator 1, staging / residual buffer 1
//   (TMEM lane quadrant of an epilogue warp = warp % 4.)
//   Everything a tile needs is double-buffered, so the stream never drains: while group g turns tile i into fp16
//   (TMEM -> regs -> +bias +residual, ReLU -> swizzled smem -> TMA store), the other group does the same for tile i+1,
//   the MMA warp fills the accumulator of tile i+2's parity as soon as it is drained, the producers run STAGES K-blocks
//   and one residual tile ahead, and the TMA store of a staging buffer is awaited only right before that buffer is
//   written again (two tiles later).  For the wide, short-K 1x1 convolutions with a residual -- memory-shaped layers
//   whose roofline is the L2 read+write stream (tools/micro/l2_stream.cu) -- this keeps loads, math and stores of
//   three tiles in flight per CTA.  The prologue (barrier init, TMEM alloc) and the first TMA round trip are paid once
//   per CTA instead of once per tile.  64-channel K-blocks with packed weights only; no split-K.
// =================================================================================================
__host__ __device__ constexpr int conv_ws_smem_bytes(int bn, int stages, int sps, bool residual) {
    return stages * sps * (128 * 64 * 2 + bn * 64 * 2) + 2 * 128 * bn * 2 + (residual ? 2 * 128 * bn * 2 : 0) + 256 + 1024;
}

template <int BN, int STAGES, int SPS>
__global__ void __launch_bounds__(384)
conv_f16_tcgen05_ws(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapOut,
                    const __grid_constant__ CUtensorMap mapRes, const ConvArgs p) {
    constexpr int A_SUBBLK = 128 * 64 * 2;
    constexpr int B_SUBBLK = BN * 64 * 2;
    constexpr int A_STAGE = SPS * A_SUBBLK;
    constexpr int B_STAGE = SPS * B_SUBBLK;
    constexpr int PIPE_BYTES = STAGES * (A_STAGE + B_STAGE);
    constexpr int TILE_BYTES = 128 * BN * 2;
    constexpr int NG = BN / 32;
    constexpr int OW = BN >= 64 ? 64 : 32;
    constexpr int OROWB = OW * 2;
    constexpr int NBOX = BN / OW;
    constexpr int TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;  // two accumulators (power of two for BN in {32..256})
    constexpr uint32_t IDESC = make_idesc_f16(128, BN);

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const bool has_res = p.residual != nullptr;
    uint8_t* sA = smem;
    uint8_t* sB = smem + STAGES * A_STAGE;
    uint8_t* sOut = smem + PIPE_BYTES;           // [2][TILE_BYTES]
    uint8_t* sRes = sOut + 2 * TILE_BYTES;       // [2][TILE_BYTES] when the layer has a residual
    uint8_t* tail = sRes + (has_res ? 2 * TILE_BYTES : 0);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* acc_full = empty_bar + STAGES;   // [2]
    uint64_t* acc_empty = acc_full + 2;        // [2]
    uint64_t* res_full = acc_empty + 2;        // [2]
    uint64_t* res_empty = res_full + 2;        // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_empty + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int num_tiles = p.tiles_m * p.tiles_n;
    const int nsteps = (p.num_kblocks + SPS - 1) / SPS;  // pipeline steps per tile
    auto subs_in_step = [&](int i) -> int {
        const int rem = p.num_kblocks - i * SPS;
        return rem < SPS ? rem : SPS;
    };

    if (threadIdx.x == 0) {
        if (p.dbg) p.dbg[static_cast<size_t>(blockIdx.x) * 16] = clock64();
        tma_prefetch_desc(&mapA);
        tma_prefetch_desc(&mapOut);
        if (has_res) tma_prefetch_desc(&mapRes);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&acc_full[b], 1);
            mbar_init(&acc_empty[b], 1);
            mbar_init(&res_full[b], 1);
            mbar_init(&res_empty[b], 1);
        }
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 2) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (p.pdl_trigger == 0) pdl_launch_dependents();
    // optional phase accounting (debug aid, b2_context_debug_conv_timing): 16 int64 per CTA
    //  0 start  1 roles begin  2 epilogue group 0 done  3 tiles of group 0   group 0, summed over its tiles: 4 wait accumulator
    //  5 wait residual  6 wait own previous store + barrier A  7 TMEM -> regs -> smem  8 barrier B + store issue
    //  9 MMA warp: wait accumulator free  10 MMA warp: wait operands  11 producer: wait residual buffer  12 producer: wait stage
    //  13 MMA warp done
    long long* const dbg = p.dbg ? p.dbg + static_cast<size_t>(blockIdx.x) * 16 : nullptr;
    if (dbg && threadIdx.x == 0) dbg[1] = clock64();

    if (warp == 0) {
        // ================= activation producer =================
        pdl_wait();
        long long w_stage = 0;
        int g = 0;   // global pipeline step counter of this CTA (across tiles)
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int mt = tile / p.tiles_n;
            const int m0 = mt * 128;
            int img0 = 0, p0 = 0, q0 = 0;
            if (p.a_mode == A_IM2COL) {
                img0 = m0 / p.HoWo;
                const int rem = m0 - img0 * p.HoWo;
                p0 = rem / p.Wo;
                q0 = rem - p0 * p.Wo;
            }
            const int base_w = q0 * p.stride_w - p.pad_w;
            const int base_h = p0 * p.stride_h - p.pad_h;
            int cur_cb = 0, cur_r = 0, cur_sx = 0;
            for (int i = 0; i < nsteps; ++i, ++g) {
                const int s = g % STAGES;
                const long long t1 = dbg ? clock64() : 0;
                mbar_wait(&empty_bar[s], ((g / STAGES) & 1) ^ 1);
                if (dbg) w_stage += clock64() - t1;
                if (elect_one_sync()) {
                    const int ns = subs_in_step(i);
                    mbar_expect_tx(&full_bar[s], static_cast<uint32_t>(ns * (A_SUBBLK + B_SUBBLK)));
                    uint8_t* a_dst = sA + s * A_STAGE;
                    for (int u = 0; u < ns; ++u) {
                        if (p.a_mode == A_TILED)
                            tma_load_2d(&mapA, &full_bar[s], a_dst + u * A_SUBBLK, cur_cb * 64, m0);
                        else
                            tma_load_im2col_4d(&mapA, &full_bar[s], a_dst + u * A_SUBBLK, cur_cb * 64, base_w, base_h, img0,
                                               static_cast<uint16_t>(cur_sx), static_cast<uint16_t>(cur_r));
                        if (++cur_cb == p.cblocks) {
                            cur_cb = 0;
                            if (++cur_sx == p.kw) {
                                cur_sx = 0;
                                ++cur_r;
                            }
                        }
                    }
                }
                __syncwarp();
            }
        }
        if (dbg && lane == 0) dbg[12] = w_stage;
    } else if (warp == 3) {
        // ================= residual producer: its waits never hold back the operand stream =================
        if (has_res) {
            pdl_wait();
            long long w_res = 0;
            int lt = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++lt) {
                const int mt = tile / p.tiles_n;
                const int nt = tile - mt * p.tiles_n;
                const int m0 = mt * 128, n0 = nt * BN;
                const int rb = lt & 1;  // buffer lt&1 is free once the epilogue of tile lt-2 has read it
                const long long t0 = dbg ? clock64() : 0;
                mbar_wait(&res_empty[rb], ((lt >> 1) & 1) ^ 1);
                if (dbg) w_res += clock64() - t0;
                if (elect_one_sync()) {
                    mbar_expect_tx(&res_full[rb], TILE_BYTES);
#pragma unroll
                    for (int b = 0; b < NBOX; ++b)
                        tma_load_2d(&mapRes, &res_full[rb], sRes + rb * TILE_BYTES + b * (128 * OROWB), n0 + b * OW, m0);
                }
                __syncwarp();
            }
            if (dbg && lane == 0) dbg[11] = w_res;
        }
    } else if (warp == 2) {
        // ================= weight producer (constants: no dependency wait) =================
        int g = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int nt = tile % p.tiles_n;
            const int n0 = nt * BN;
            for (int i = 0; i < nsteps; ++i, ++g) {
                const int s = g % STAGES;
                if (g >= STAGES) mbar_wait(&empty_bar[s], ((g / STAGES) & 1) ^ 1);
                if (elect_one_sync()) {
                    const int ns = subs_in_step(i);
                    for (int u = 0; u < ns; ++u)
                        bulk_load_1d(&full_bar[s], sB + s * B_STAGE + u * B_SUBBLK,
                                     p.wpacked + (static_cast<size_t>(i * SPS + u) * (p.Cout >> 5) + (n0 >> 5)) * 4096, BN * 128);
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        int g = 0, lt = 0;
        long long w_acc = 0, w_ops = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++lt) {
            const int b = lt & 1;
            const long long t0 = dbg ? clock64() : 0;
            mbar_wait(&acc_empty[b], ((lt >> 1) & 1) ^ 1);  // the epilogue has drained this accumulator
            if (dbg) w_acc += clock64() - t0;
            tc_fence_after();
            const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(b * BN);
            for (int i = 0; i < nsteps; ++i, ++g) {
                const int s = g % STAGES;
                const long long t1 = dbg ? clock64() : 0;
                mbar_wait(&full_bar[s], (g / STAGES) & 1);
                if (dbg) w_ops += clock64() - t1;
                tc_fence_after();
                const uint32_t a_addr = smem_u32(sA + s * A_STAGE);
                const uint32_t b_addr = smem_u32(sB + s * B_STAGE);
                if (elect_one_sync()) {
                    const int ns = subs_in_step(i);
#pragma unroll
                    for (int u = 0; u < SPS; ++u) {
                        if (u < ns) {
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const uint64_t ad = make_smem_desc(a_addr + u * A_SUBBLK + j * 32, 16, 1024, 2);
                                const uint64_t bd = make_smem_desc(b_addr + u * B_SUBBLK + j * 32, 16, 1024, 2);
                                umma_f16(tmem_d, ad, bd, IDESC, (i > 0 || u > 0 || j > 0) ? 1u : 0u);
                            }
                        }
                    }
                    umma_commit(&empty_bar[s]);
                    if (i == nsteps - 1) umma_commit(&acc_full[b]);
                }
                __syncwarp();
            }
        }
        if (p.pdl_trigger == 1) pdl_launch_dependents();
        if (dbg && lane == 0) dbg[9] = w_acc, dbg[10] = w_ops, dbg[13] = clock64();
    } else if (warp >= 4) {
        // ================= epilogue: two groups of 4 warps (128 threads, one accumulator row each) =================
        pdl_wait();
        const int grp = (warp - 4) >> 2;  // == accumulator / staging / residual buffer index == parity of the local tile
        const int q = warp & 3;           // TMEM lane quadrant this warp may access
        const int row = q * 32 + lane;
        const bool e0 = (threadIdx.x == 128 + grp * 128);
        uint8_t* const my_out = sOut + grp * TILE_BYTES;
        const uint8_t* const my_res = sRes + grp * TILE_BYTES;
        const uint32_t bar_a = 1 + 2 * grp, bar_b = 2 + 2 * grp;
        int lt = grp;
        const bool rec = dbg && e0 && grp == 0;
        long long d_acc = 0, d_res = 0, d_a = 0, d_math = 0, d_b = 0, d_tiles = 0;
        for (int tile = blockIdx.x + grp * static_cast<int>(gridDim.x); tile < num_tiles; tile += 2 * gridDim.x, lt += 2) {
            const int mt = tile / p.tiles_n;
            const int nt = tile - mt * p.tiles_n;
            const int m0 = mt * 128, n0 = nt * BN;
            const uint32_t par = (lt >> 1) & 1;
            const long long c0 = rec ? clock64() : 0;
            mbar_wait(&acc_full[grp], par);
            tc_fence_after();
            const long long c1 = rec ? clock64() : 0;
            if (has_res) mbar_wait(&res_full[grp], par);
            const long long c2 = rec ? clock64() : 0;
            // (A) this group's previous TMA store has finished READING the staging buffer
            if (e0) tma_store_wait_read0();
            named_bar_sync(bar_a, 128);
            const long long c3 = rec ? clock64() : 0;
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(grp * BN);
            const float4* bias4 = reinterpret_cast<const float4*>(p.bias + n0);
            constexpr int GP = NG >= 2 ? 2 : 1;
#pragma unroll
            for (int g0 = 0; g0 < NG; g0 += GP) {
                uint32_t acc[GP][32];
#pragma unroll
                for (int j = 0; j < GP; ++j) tmem_ld32(taddr + (g0 + j) * 32, acc[j]);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < GP; ++j) {
#pragma unroll
                    for (int qq = 0; qq < 4; ++qq) {
                        const int col = (g0 + j) * 32 + qq * 8;
                        const int box = col / OW;
                        const int chunk = (col % OW) / 8;
                        const uint32_t so = static_cast<uint32_t>(box * (128 * OROWB)) + swz_off<OROWB>(row, chunk);
                        const float4 b0 = __ldg(bias4 + col / 4), b1 = __ldg(bias4 + col / 4 + 1);
                        float v[8];
                        v[0] = __uint_as_float(acc[j][qq * 8 + 0]) + b0.x;
                        v[1] = __uint_as_float(acc[j][qq * 8 + 1]) + b0.y;
                        v[2] = __uint_as_float(acc[j][qq * 8 + 2]) + b0.z;
                        v[3] = __uint_as_float(acc[j][qq * 8 + 3]) + b0.w;
                        v[4] = __uint_as_float(acc[j][qq * 8 + 4]) + b1.x;
                        v[5] = __uint_as_float(acc[j][qq * 8 + 5]) + b1.y;
                        v[6] = __uint_as_float(acc[j][qq * 8 + 6]) + b1.z;
                        v[7] = __uint_as_float(acc[j][qq * 8 + 7]) + b1.w;
                        if (has_res) {
                            const uint4 rv = *reinterpret_cast<const uint4*>(my_res + so);
                            const __half2* r2 = reinterpret_cast<const __half2*>(&rv);
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const float2 rf = __half22float2(r2[i]);
                                v[2 * i] += rf.x;
                                v[2 * i + 1] += rf.y;
                            }
                        }
                        if (p.relu) {
#pragma unroll
                            for (int i = 0; i < 8; ++i) v[i] = fmaxf(v[i], 0.0f);
                        }
                        uint4 o;
                        __half2* o2 = reinterpret_cast<__half2*>(&o);
#pragma unroll
                        for (int i = 0; i < 4; ++i) o2[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
                        *reinterpret_cast<uint4*>(my_out + so) = o;
                    }
                }
            }
            tc_fence_before();
            fence_proxy_async();
            const long long c4 = rec ? clock64() : 0;
            // (B) every thread of the group has drained its TMEM rows, read its residual row and staged its output row
            named_bar_sync(bar_b, 128);
            if (e0) {
                mbar_arrive(&acc_empty[grp]);              // the accumulator may be overwritten by tile lt+2
                if (has_res) mbar_arrive(&res_empty[grp]);  // the residual buffer may be refilled
#pragma unroll
                for (int bx = 0; bx < NBOX; ++bx) tma_store_2d(&mapOut, my_out + bx * (128 * OROWB), n0 + bx * OW, m0);
                tma_store_commit();  // awaited at (A) of this group's next tile, or below before the CTA retires
            }
            if (rec) {
                const long long c5 = clock64();
                d_acc += c1 - c0, d_res += c2 - c1, d_a += c3 - c2, d_math += c4 - c3, d_b += c5 - c4, ++d_tiles;
            }
        }
        if (e0) tma_store_wait_read0();  // shared memory must outlive the last bulk store's read
        if (rec) dbg[2] = clock64(), dbg[3] = d_tiles, dbg[4] = d_acc, dbg[5] = d_res, dbg[6] = d_a, dbg[7] = d_math, dbg[8] = d_b;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

// =================================================================================================
// conv3x3_halo_tcgen05 -- 3x3 / stride 1 / pad 1 convolution that brings every input pixel into shared memory ONCE per
//   (tile, 64-channel block) instead of once per filter tap.
//
//   The tile is R whole output rows of one image in PADDED coordinates: accumulator row m' = hh*(W+2) + ww.  One 4-D
//   TMA box {64 ch, W+2, R+2, 1} starting at (w = -1, h = h0-1) lands the halo block in smem as (R+2)*(W+2) pixel rows
//   of 128 B (SWIZZLE_128B); out-of-image pixels are zero-filled by the TMA, which IS the convolution's padding.  The A
//   operand of tap (r, s) is the same block read from pixel row r*(W+2)+s on: a start-address offset in the UMMA
//   descriptor (the 128B swizzle is a function of the absolute smem address, so a row shift keeps it consistent).
//   Columns ww = W, W+1 of every row compute garbage that the output TMA store (box {BN, W+2, R, 1} at w = 0) clips.
//   A traffic per tile and channel block: (R+2)(W+2) pixel rows instead of 9 x 128.
//
//   warp 0 = halo producer, warp 1 = MMA issuer, warp 2 = TMEM owner, warp 3 = weight producer, all 4 = epilogue.
//   The halo blocks of ALL channel blocks stay resident, so the K loop runs tap outer / channel block inner exactly
//   like the im2col kernel: same products in the same fp32 summation order -> bit-identical results, whichever of the
//   two tactics the tuner picks.
// =================================================================================================
constexpr int kHaloMaxCBlocks = 8;
__host__ __device__ constexpr int halo_b_stages(int bn) { return bn >= 256 ? 3 : 4; }
// bytes of one A stage: the loaded halo block, but never less than what the farthest tap's 128-row window touches
__host__ __device__ constexpr int halo_a_stage_bytes(int w, int r) {
    const int loaded = (r + 2) * (w + 2);
    const int touched = 128 + 2 * (w + 2) + 2;
    const int rows = loaded > touched ? loaded : touched;
    return (rows * 128 + 1023) / 1024 * 1024;
}
__host__ __device__ constexpr int halo_smem_bytes(int bn, int w, int r, int cblocks) {
    return cblocks * halo_a_stage_bytes(w, r) + halo_b_stages(bn) * bn * 128 + 256 + bn * 4 + 1024;
}

template <int BN>
__global__ void __launch_bounds__(128)
conv3x3_halo_tcgen05(const __grid_constant__ CUtensorMap mapIn, const __grid_constant__ CUtensorMap mapOut, const ConvArgs p) {
    constexpr int NB = halo_b_stages(BN);
    constexpr int B_BLK = BN * 128;  // one tap of one 64-channel block: BN rows of 128 B (pre-swizzled)
    constexpr int NG = BN / 32;
    constexpr int OW = 64;
    constexpr int NBOX = BN / OW;
    constexpr uint32_t IDESC = make_idesc_f16(128, BN);

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const int W = p.Wo, Wp = p.Wo + 2, R = p.halo_rows;
    const int a_stage = halo_a_stage_bytes(W, R);
    const int cblocks = p.cblocks;
    uint8_t* sA = smem;
    uint8_t* sB = smem + cblocks * a_stage;
    uint8_t* sOut = smem;  // staging reuses the drained buffers
    uint8_t* tail = sB + NB * B_BLK;
    uint64_t* a_full = reinterpret_cast<uint64_t*>(tail);
    uint64_t* b_full = a_full + kHaloMaxCBlocks;
    uint64_t* b_empty = b_full + NB;
    uint64_t* accum_bar = b_empty + NB;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);
    float* s_bias = reinterpret_cast<float*>(tail + 256);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN;
    const int Ho = p.HoWo / p.Wo;
    const int tiles_per_img = (Ho + R - 1) / R;
    const int img = blockIdx.y / tiles_per_img;
    const int h0 = (blockIdx.y - img * tiles_per_img) * R;
    const int nsteps = cblocks * 9;  // weight blocks, in (tap, cb) order = the packed layout's K order

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&mapIn);
        tma_prefetch_desc(&mapOut);
        for (int s = 0; s < cblocks; ++s) mbar_init(&a_full[s], 1);
        for (int s = 0; s < NB; ++s) {
            mbar_init(&b_full[s], 1);
            mbar_init(&b_empty[s], 1);
        }
        mbar_init(accum_bar, 1);
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 2) tmem_alloc(tmem_slot, BN);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (p.pdl_trigger == 0) pdl_launch_dependents();

    if (warp == 0) {
        // ================= halo producer =================
        const uint32_t halo_bytes = static_cast<uint32_t>((R + 2) * Wp * 128);
        pdl_wait();
        if (elect_one_sync()) {
            for (int cb = 0; cb < cblocks; ++cb) {
                mbar_expect_tx(&a_full[cb], halo_bytes);
                tma_load_4d(&mapIn, &a_full[cb], sA + cb * a_stage, cb * 64, -1, h0 - 1, img);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================= MMA issuer =================
        int i = 0;
#pragma unroll 1
        for (int tap = 0; tap < 9; ++tap) {
            const int r = tap / 3, sx = tap - r * 3;
            const uint32_t tap_off = static_cast<uint32_t>((r * Wp + sx) * 128);
#pragma unroll 1
            for (int cb = 0; cb < cblocks; ++cb, ++i) {
                const int sb = i % NB;
                if (tap == 0) mbar_wait(&a_full[cb], 0);
                mbar_wait(&b_full[sb], (i / NB) & 1);
                tc_fence_after();
                const uint32_t a_addr = smem_u32(sA + cb * a_stage) + tap_off;
                const uint32_t b_addr = smem_u32(sB + sb * B_BLK);
                if (elect_one_sync()) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        // descriptor "base offset" stays 0: the swizzle pattern is anchored at the 1024-aligned stage base
                        // (measured: setting it to (addr >> 7) & 7 for the shifted start gives wrong results)
                        const uint64_t ad = make_smem_desc(a_addr + j * 32, 16, 1024, 2);
                        const uint64_t bd = make_smem_desc(b_addr + j * 32, 16, 1024, 2);
                        umma_f16(tmem_base, ad, bd, IDESC, (i > 0 || j > 0) ? 1u : 0u);
                    }
                    umma_commit(&b_empty[sb]);
                }
                __syncwarp();
            }
        }
        if (elect_one_sync()) umma_commit(accum_bar);
        __syncwarp();
    } else if (warp == 3) {
        // ================= weight producer (constants: no dependency wait) =================
        for (int i = lane; i < BN; i += 32) s_bias[i] = __ldg(p.bias + n0 + i);
        for (int i = 0; i < nsteps; ++i) {
            const int sb = i % NB;
            if (i >= NB) mbar_wait(&b_empty[sb], ((i / NB) & 1) ^ 1);
            if (elect_one_sync()) {
                mbar_expect_tx(&b_full[sb], B_BLK);
                bulk_load_1d(&b_full[sb], sB + sb * B_BLK, p.wpacked + (static_cast<size_t>(i) * (p.Cout >> 5) + (n0 >> 5)) * 4096,
                             B_BLK);
            }
            __syncwarp();
        }
    }

    // ====== epilogue: TMEM -> registers -> bias/ReLU -> fp16 -> swizzled smem tile -> 4-D TMA store ======
    pdl_wait();
    const int row = warp * 32 + lane;
    mbar_wait(accum_bar, 0);
    tc_fence_after();
    __syncthreads();
    if (p.pdl_trigger == 1) pdl_launch_dependents();
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
#pragma unroll
    for (int g = 0; g < NG; ++g) {
        uint32_t acc[32];
        tmem_ld32(taddr + g * 32, acc);
        tmem_wait_ld();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int col = g * 32 + q * 8;
            const int box = col / OW;
            const int chunk = (col % OW) / 8;
            const uint32_t so = static_cast<uint32_t>(box * (128 * 128)) + swz_off<128>(row, chunk);
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                v[i] = __uint_as_float(acc[q * 8 + i]) + s_bias[col + i];
                if (p.relu) v[i] = fmaxf(v[i], 0.0f);
            }
            uint4 o;
            __half2* o2 = reinterpret_cast<__half2*>(&o);
#pragma unroll
            for (int i = 0; i < 4; ++i) o2[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
            *reinterpret_cast<uint4*>(sOut + so) = o;
        }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, BN);
    if (threadIdx.x == 0) {
        // box {64 ch, W+2, R, 1} at w = 0: the two garbage columns of every row and rows past H are clipped
#pragma unroll
        for (int b = 0; b < NBOX; ++b) tma_store_4d(&mapOut, sOut + b * (128 * 128), n0 + b * OW, 0, h0, img);
        tma_store_commit_and_wait_read();
    }
}

static bool g_use_pdl = true;
void set_pdl(bool on) { g_use_pdl = on; }
bool get_pdl() { return g_use_pdl; }

template <typename Kern, typename... Args>
static int launch_kernel_cluster(Kern kern, dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl, unsigned cluster_x,
                                 Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    unsigned n = 0;
    if (pdl && g_use_pdl) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    if (cluster_x > 1) {
        attr[n].id = cudaLaunchAttributeClusterDimension;
        attr[n].val.clusterDim.x = cluster_x;
        attr[n].val.clusterDim.y = 1;
        attr[n].val.clusterDim.z = 1;
        ++n;
    }
    cfg.attrs = attr;
    cfg.numAttrs = n;
    return static_cast<int>(cudaLaunchKernelEx(&cfg, kern, args...));
}
template <typename Kern, typename... Args>
static int launch_kernel(Kern kern, dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl, Args... args) {
    return launch_kernel_cluster(kern, grid, block, smem, stream, pdl, 1u, args...);
}

template <int BN, int KB, int STAGES, int SPS, int CN = 1>
static int launch_one(const ConvLaunch& L, cudaStream_t stream) {
    dim3 grid(L.grid_n, L.grid_m, L.args.splits);
    const size_t smem = size_t(conv_smem_layout_bytes(BN, STAGES, L.args.residual != nullptr, SPS));
    if (CN > 1 && (KB != 64 || L.grid_n % CN != 0 || L.args.cn != CN)) return static_cast<int>(cudaErrorInvalidValue);
    if (CN == 1 && (L.args.dbg != nullptr || L.args.dbg_mode != 0))
        return launch_kernel_cluster(conv_f16_tcgen05<BN, KB, STAGES, SPS, 1, true>, grid, dim3(128), smem, stream, true, 1u, L.mapA,
                                     L.mapB, L.mapOut, L.mapRes, L.args);
    if constexpr (CN == 1 && KB == 64) {
        if (L.args.wpacked != nullptr) {
            if (L.args.a_mode == A_TILED)
                return launch_kernel_cluster(conv_f16_tcgen05<BN, KB, STAGES, SPS, 1, false, 2>, grid, dim3(128), smem, stream, true, 1u,
                                             L.mapA, L.mapB, L.mapOut, L.mapRes, L.args);
            return launch_kernel_cluster(conv_f16_tcgen05<BN, KB, STAGES, SPS, 1, false, 1>, grid, dim3(128), smem, stream, true, 1u,
                                         L.mapA, L.mapB, L.mapOut, L.mapRes, L.args);
        }
    }
    return launch_kernel_cluster(conv_f16_tcgen05<BN, KB, STAGES, SPS, CN>, grid, dim3(128), smem, stream, true,
                                 static_cast<unsigned>(CN), L.mapA, L.mapB, L.mapOut, L.mapRes, L.args);
}

template <int BN, int KB, int STAGES, int SPS, int CN = 1>
static int init_one() {
    const int want = conv_smem_layout_bytes(BN, STAGES, true, SPS);
    const int bytes = want > 227 * 1024 ? conv_smem_layout_bytes(BN, STAGES, false, SPS) : want;
    if (CN == 1) {
        int e = static_cast<int>(cudaFuncSetAttribute(conv_f16_tcgen05<BN, KB, STAGES, SPS, 1, true>,
                                                      cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        if (e) return e;
        if constexpr (KB == 64) {
            if ((e = static_cast<int>(cudaFuncSetAttribute(conv_f16_tcgen05<BN, KB, STAGES, SPS, 1, false, 1>,
                                                           cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)))) return e;
            if ((e = static_cast<int>(cudaFuncSetAttribute(conv_f16_tcgen05<BN, KB, STAGES, SPS, 1, false, 2>,
                                                           cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)))) return e;
        }
    }
    return static_cast<int>(cudaFuncSetAttribute(conv_f16_tcgen05<BN, KB, STAGES, SPS, CN>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
}

int conv_smem_bytes(int bn, int stages, bool residual, int sps) { return conv_smem_layout_bytes(bn, stages, residual, sps); }

// instantiated (BN, KB, STAGES, SPS) configurations
#define B2_FOR_EACH_CONV(X) \
    X(32, 64, 1, 1) X(32, 64, 2, 1) X(32, 64, 4, 1) X(32, 64, 8, 1) \
    X(64, 64, 1, 1) X(64, 64, 2, 1) X(64, 64, 4, 1) X(64, 64, 8, 1) \
    X(128, 64, 1, 1) X(128, 64, 2, 1) X(128, 64, 4, 1) X(256, 64, 2, 1) X(256, 64, 4, 1) \
    X(32, 64, 2, 2) X(32, 64, 4, 2) X(64, 64, 2, 2) X(64, 64, 4, 2) X(128, 64, 2, 2) X(256, 64, 2, 2) \
    X(32, 8, 2, 1) X(32, 8, 4, 1) X(64, 8, 2, 1) X(64, 8, 4, 1) X(64, 8, 8, 1) X(128, 8, 4, 1) \
    X(32, 32, 2, 1) X(32, 32, 4, 1) X(64, 32, 1, 1) X(64, 32, 2, 1) X(64, 32, 4, 1) X(128, 32, 2, 1) X(128, 32, 4, 1)

int conv_halo_smem(int bn, int w, int r, int cblocks) { return halo_smem_bytes(bn, w, r, cblocks); }
bool conv_halo_config_exists(int bn) { return bn == 64 || bn == 128 || bn == 256; }
static int init_conv_halo_kernels() {
    int e;
    if ((e = static_cast<int>(cudaFuncSetAttribute(conv3x3_halo_tcgen05<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)))) return e;
    if ((e = static_cast<int>(cudaFuncSetAttribute(conv3x3_halo_tcgen05<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)))) return e;
    if ((e = static_cast<int>(cudaFuncSetAttribute(conv3x3_halo_tcgen05<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)))) return e;
    return 0;
}
static int launch_conv_halo(const ConvLaunch& L, cudaStream_t stream) {
    const int R = L.args.halo_rows;
    const size_t smem = size_t(halo_smem_bytes(L.bn, L.args.Wo, R, L.args.cblocks));
    if (smem > 227 * 1024 || R < 1 || R * (L.args.Wo + 2) > 128 || L.args.cblocks > kHaloMaxCBlocks) return static_cast<int>(cudaErrorInvalidValue);
    dim3 grid(L.grid_n, L.grid_m, 1);
    switch (L.bn) {
        case 64: return launch_kernel(conv3x3_halo_tcgen05<64>, grid, dim3(128), smem, stream, true, L.mapA, L.mapOut, L.args);
        case 128: return launch_kernel(conv3x3_halo_tcgen05<128>, grid, dim3(128), smem, stream, true, L.mapA, L.mapOut, L.args);
        case 256: return launch_kernel(conv3x3_halo_tcgen05<256>, grid, dim3(128), smem, stream, true, L.mapA, L.mapOut, L.args);
    }
    return static_cast<int>(cudaErrorInvalidValue);
}

// cluster-multicast instantiations (BN, STAGES, SPS, CN): an experiment-only tactic (never won a timing), kept small
#define B2_FOR_EACH_CONV_CLUSTER(X) \
    X(32, 4, 1, 2) X(32, 4, 1, 4) X(64, 1, 1, 2) X(64, 2, 1, 2) X(64, 2, 1, 4) X(64, 2, 2, 2) X(64, 4, 2, 2) X(64, 4, 2, 4) \
    X(128, 2, 1, 2) X(128, 2, 1, 4) X(128, 2, 2, 2)

int init_conv_ws_kernels();
int launch_conv_f16_tcgen05_ws(const ConvLaunch& L, cudaStream_t stream);

int init_conv_kernels() {
    int e = init_conv_ws_kernels();
    if (e) return e;
    if ((e = init_conv_halo_kernels())) return e;
#define B2_INIT(BN_, KB_, ST_, SPS_) \
    if ((e = init_one<BN_, KB_, ST_, SPS_>())) return e;
    B2_FOR_EACH_CONV(B2_INIT)
#undef B2_INIT
#define B2_INIT_CL(BN_, ST_, SPS_, CN_) \
    if ((e = init_one<BN_, 64, ST_, SPS_, CN_>())) return e;
    B2_FOR_EACH_CONV_CLUSTER(B2_INIT_CL)
#undef B2_INIT_CL
    return 0;
}

int launch_conv_f16_tcgen05(const ConvLaunch& L, cudaStream_t stream) {
    if (L.halo) return launch_conv_halo(L, stream);
    if (L.ws_ctas > 0) return launch_conv_f16_tcgen05_ws(L, stream);
    if (L.cn > 1) {
#define B2_CASE_CL(BN_, ST_, SPS_, CN_) \
    if (L.bn == BN_ && L.kb == 64 && L.stages == ST_ && L.sps == SPS_ && L.cn == CN_) return launch_one<BN_, 64, ST_, SPS_, CN_>(L, stream);
        B2_FOR_EACH_CONV_CLUSTER(B2_CASE_CL)
#undef B2_CASE_CL
        return static_cast<int>(cudaErrorInvalidValue);
    }
#define B2_CASE(BN_, KB_, ST_, SPS_) \
    if (L.bn == BN_ && L.kb == KB_ && L.stages == ST_ && L.sps == SPS_) return launch_one<BN_, KB_, ST_, SPS_>(L, stream);
    B2_FOR_EACH_CONV(B2_CASE)
#undef B2_CASE
    return static_cast<int>(cudaErrorInvalidValue);
}

// instantiated persistent (BN, STAGES, SPS) configurations
#define B2_FOR_EACH_CONV_WS(X) \
    X(32, 4, 1) X(64, 2, 1) X(64, 4, 1) X(64, 2, 2) X(64, 4, 2) X(128, 2, 1) X(128, 4, 1) X(128, 2, 2) X(256, 2, 1)

template <int BN, int STAGES, int SPS>
static int launch_one_ws(const ConvLaunch& L, cudaStream_t stream) {
    const size_t smem = size_t(conv_ws_smem_bytes(BN, STAGES, SPS, L.args.residual != nullptr));
    return launch_kernel(conv_f16_tcgen05_ws<BN, STAGES, SPS>, dim3(L.ws_ctas), dim3(384), smem, stream, true, L.mapA, L.mapOut,
                         L.mapRes, L.args);
}

int init_conv_ws_kernels() {
    int e = 0;
#define B2_INIT_WS(BN_, ST_, SPS_)                                                                                        \
    {                                                                                                                     \
        const int want = conv_ws_smem_bytes(BN_, ST_, SPS_, true);                                                        \
        e = static_cast<int>(cudaFuncSetAttribute(conv_f16_tcgen05_ws<BN_, ST_, SPS_>,                                    \
                                                  cudaFuncAttributeMaxDynamicSharedMemorySize,                            \
                                                  want > 227 * 1024 ? conv_ws_smem_bytes(BN_, ST_, SPS_, false) : want)); \
        if (e) return e;                                                                                                  \
    }
    B2_FOR_EACH_CONV_WS(B2_INIT_WS)
#undef B2_INIT_WS
    return 0;
}

int launch_conv_f16_tcgen05_ws(const ConvLaunch& L, cudaStream_t stream) {
#define B2_CASE_WS(BN_, ST_, SPS_) \
    if (L.bn == BN_ && L.stages == ST_ && L.sps == SPS_) return launch_one_ws<BN_, ST_, SPS_>(L, stream);
    B2_FOR_EACH_CONV_WS(B2_CASE_WS)
#undef B2_CASE_WS
    return static_cast<int>(cudaErrorInvalidValue);
}

bool conv_ws_config_exists(int bn, int stages, int sps) {
#define B2_HAS_WS(BN_, ST_, SPS_) \
    if (bn == BN_ && stages == ST_ && sps == SPS_) return true;
    B2_FOR_EACH_CONV_WS(B2_HAS_WS)
#undef B2_HAS_WS
    return false;
}

int conv_ws_smem(int bn, int stages, int sps, bool residual) { return conv_ws_smem_bytes(bn, stages, sps, residual); }

bool conv_cluster_config_exists(int bn, int stages, int sps, int cn) {
#define B2_HAS_CL(BN_, ST_, SPS_, CN_) \
    if (bn == BN_ && stages == ST_ && sps == SPS_ && cn == CN_) return true;
    B2_FOR_EACH_CONV_CLUSTER(B2_HAS_CL)
#undef B2_HAS_CL
    return false;
}

bool conv_config_exists(int bn, int kb, int stages, int sps) {
#define B2_HAS(BN_, KB_, ST_, SPS_) \
    if (bn == BN_ && kb == KB_ && stages == ST_ && sps == SPS_) return true;
    B2_FOR_EACH_CONV(B2_HAS)
#undef B2_HAS
    return false;
}

// =================================================================================================
// SIMT kernels
// =================================================================================================
static thread_local int B2_LAUNCH_RC = 0;

template <typename T>
struct Acc;
template <>
struct Acc<float> {
    using type = double;  // fp32 engine: fp64 accumulate -> order-independent to ~1e-12
};
template <>
struct Acc<__half> {
    using type = float;
};
__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
template <typename T>
__device__ __forceinline__ T from_f(float v);
template <>
__device__ __forceinline__ float from_f<float>(float v) { return v; }
template <>
__device__ __forceinline__ __half from_f<__half>(float v) { return __float2half_rn(v); }

// direct convolution, one thread per output element (co fastest)
template <typename T>
__global__ void conv_simt_kernel(SimtConvArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    using acc_t = typename Acc<T>::type;
    const long long total = static_cast<long long>(a.N) * a.Ho * a.Wo * a.Cout_phys;
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= total) return;
    const int co = static_cast<int>(idx % a.Cout_phys);
    long long pix = idx / a.Cout_phys;
    const int wo = static_cast<int>(pix % a.Wo);
    pix /= a.Wo;
    const int ho = static_cast<int>(pix % a.Ho);
    const int n = static_cast<int>(pix / a.Ho);
    T* out = reinterpret_cast<T*>(a.out);
    if (co >= a.Cout) {
        out[idx] = from_f<T>(0.0f);
        return;
    }
    const T* in = reinterpret_cast<const T*>(a.in);
    const T* w = reinterpret_cast<const T*>(a.w) + static_cast<size_t>(co) * a.taps_phys * a.Cin_phys;
    acc_t acc = 0;
    for (int r = 0; r < a.kh; ++r) {
        const int hi = ho * a.stride_h - a.pad_h + r;
        if (hi < 0 || hi >= a.H) continue;
        for (int s = 0; s < a.kw; ++s) {
            const int wi = wo * a.stride_w - a.pad_w + s;
            if (wi < 0 || wi >= a.W) continue;
            const T* ip = in + ((static_cast<size_t>(n) * a.H + hi) * a.W + wi) * a.Cin_phys;
            const T* wp = w + static_cast<size_t>(r * a.kw + s) * a.Cin_phys;
            if (a.w_packed) {
                const size_t kbase = static_cast<size_t>(r * a.kw + s) * a.Cin_phys;
                for (int c = 0; c < a.Cin; ++c) {
                    const size_t k = kbase + c;
                    const size_t kk = k & 63;
                    const size_t off = (((k >> 6) * static_cast<size_t>(a.Cout_phys >> 5) + static_cast<size_t>(co >> 5)) << 11) + (static_cast<size_t>(co & 31) << 6) +
                                       ((((kk >> 3) ^ (co & 7))) << 3) + (kk & 7);  // in T (= 2-byte) elements
                    acc += static_cast<acc_t>(to_f(ip[c])) * static_cast<acc_t>(to_f(reinterpret_cast<const T*>(a.w)[off]));
                }
            } else {
                for (int c = 0; c < a.Cin; ++c)
                    acc += static_cast<acc_t>(to_f(ip[c])) * static_cast<acc_t>(to_f(wp[c]));
            }
        }
    }
    acc_t v = acc + static_cast<acc_t>(a.bias[co]);
    if (a.residual) v += static_cast<acc_t>(to_f(reinterpret_cast<const T*>(a.residual)[idx]));
    if (a.relu && v < 0) v = 0;
    out[idx] = from_f<T>(static_cast<float>(v));
}

int launch_conv_simt(const SimtConvArgs& a, bool half_storage, cudaStream_t stream) {
    const long long total = static_cast<long long>(a.N) * a.Ho * a.Wo * a.Cout_phys;
    const int threads = 128;
    const long long blocks = (total + threads - 1) / threads;
    if (blocks <= 0) return 0;
    if (half_storage)
        B2_LAUNCH_RC = launch_kernel(conv_simt_kernel<__half>, dim3(static_cast<unsigned>(blocks)), dim3(threads), 0, stream, true, a);
    else
        B2_LAUNCH_RC = launch_kernel(conv_simt_kernel<float>, dim3(static_cast<unsigned>(blocks)), dim3(threads), 0, stream, true, a);
    return B2_LAUNCH_RC;
}

// fp32 NCHW -> NHWC (channel-padded).  One thread per pixel: reads are coalesced per channel plane,
// the write is one contiguous C_phys-element row.
__device__ __forceinline__ float ld_in(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_in(const __half* p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ float2 ld_in2(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }
__device__ __forceinline__ float2 ld_in2(const __half* p) { return __half22float2(__ldg(reinterpret_cast<const __half2*>(p))); }

// S = element type of the input BINDING (fp32, or fp16 for plans built with input_dtype="f16")
template <typename T, typename S>
__global__ void input_cast_kernel(const S* __restrict__ src, T* __restrict__ dst, int N, int C, int HW,
                                  int C_phys) {
    pdl_launch_dependents();
    pdl_wait();
    const long long total = static_cast<long long>(N) * HW, step = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total; idx += step) {
        const int n = static_cast<int>(idx / HW);
        const int px = static_cast<int>(idx - static_cast<long long>(n) * HW);
        const S* s = src + static_cast<size_t>(n) * C * HW + px;
        T* d = dst + static_cast<size_t>(idx) * C_phys;
        for (int c = 0; c < C_phys; ++c) d[c] = from_f<T>(c < C ? ld_in(s + static_cast<size_t>(c) * HW) : 0.0f);
    }
}

// specialisation used by the fp16 path when C_phys == 8: one 16-byte store per pixel
template <typename S>
__global__ void input_cast_c8_kernel(const S* __restrict__ src, uint4* __restrict__ dst, int N, int C, int HW) {
    pdl_launch_dependents();
    pdl_wait();
    const long long total = static_cast<long long>(N) * HW, step = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total; idx += step) {
        const int n = static_cast<int>(idx / HW);
        const int px = static_cast<int>(idx - static_cast<long long>(n) * HW);
        const S* s = src + static_cast<size_t>(n) * C * HW + px;
        float f[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) f[c] = c < C ? ld_in(s + static_cast<size_t>(c) * HW) : 0.0f;
        uint4 o;
        __half2* o2 = reinterpret_cast<__half2*>(&o);
#pragma unroll
        for (int i = 0; i < 4; ++i) o2[i] = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
        dst[idx] = o;
    }
}

template <typename S>
static int launch_input_cast_t(const S* src, void* dst, int N, int C, int H, int W, int C_phys, bool half_storage,
                               int max_blocks, cudaStream_t stream) {
    const long long total = static_cast<long long>(N) * H * W;
    const int threads = 256;
    unsigned blocks = static_cast<unsigned>((total + threads - 1) / threads);
    if (max_blocks > 0 && blocks > static_cast<unsigned>(max_blocks)) blocks = static_cast<unsigned>(max_blocks);  // grid-stride
    if (half_storage && C_phys == 8 && C <= 8)
        B2_LAUNCH_RC = launch_kernel(input_cast_c8_kernel<S>, dim3(blocks), dim3(threads), 0, stream, false, src, reinterpret_cast<uint4*>(dst), N, C, H * W);
    else if (half_storage)
        B2_LAUNCH_RC = launch_kernel(input_cast_kernel<__half, S>, dim3(blocks), dim3(threads), 0, stream, false, src, reinterpret_cast<__half*>(dst), N, C, H * W, C_phys);
    else
        B2_LAUNCH_RC = launch_kernel(input_cast_kernel<float, S>, dim3(blocks), dim3(threads), 0, stream, false, src, reinterpret_cast<float*>(dst), N, C, H * W, C_phys);
    return B2_LAUNCH_RC;
}
int launch_input_cast(const void* src, bool src_half, void* dst, int N, int C, int H, int W, int C_phys, bool half_storage,
                      int max_blocks, cudaStream_t stream) {
    if (src_half) return launch_input_cast_t(static_cast<const __half*>(src), dst, N, C, H, W, C_phys, half_storage, max_blocks, stream);
    return launch_input_cast_t(static_cast<const float*>(src), dst, N, C, H, W, C_phys, half_storage, max_blocks, stream);
}

// fp32 NCHW -> fp16 [N, H, pad_l + W/2 + pad_r, 8], channel = dw*4 + c: one 16-byte store per PAIR of input pixels;
// the pad_l / pad_r border pixels are written as zeros (the stem's horizontal padding made physical)
template <typename S>
__global__ void input_cast_s2d_kernel(const S* __restrict__ src, uint4* __restrict__ dst, int N, int C, int H, int W,
                                      int pad_l, int pad_r) {
    pdl_launch_dependents();
    pdl_wait();
    const int W2 = W >> 1;
    const int Wp = W2 + pad_l + pad_r;
    const long long total = static_cast<long long>(N) * H * Wp, step = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total; idx += step) {
        const int wp = static_cast<int>(idx % Wp);
        const long long t = idx / Wp;
        const int h = static_cast<int>(t % H);
        const int n = static_cast<int>(t / H);
        const int w2 = wp - pad_l;
        uint4 o = make_uint4(0u, 0u, 0u, 0u);
        if (w2 >= 0 && w2 < W2) {
            const S* s = src + (static_cast<size_t>(n) * C * H + h) * W + 2 * w2;
            float f[8];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                float2 v = make_float2(0.f, 0.f);
                if (c < C) v = ld_in2(s + static_cast<size_t>(c) * H * W);
                f[c] = v.x;
                f[4 + c] = v.y;
            }
            __half2* o2 = reinterpret_cast<__half2*>(&o);
#pragma unroll
            for (int i = 0; i < 4; ++i) o2[i] = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
        }
        dst[idx] = o;
    }
}

int launch_input_cast_s2d(const void* src, bool src_half, void* dst, int N, int C, int H, int W, int pad_l, int pad_r,
                          int max_blocks, cudaStream_t stream) {
    const long long total = static_cast<long long>(N) * H * (W / 2 + pad_l + pad_r);
    const int threads = 256;
    unsigned blocks = static_cast<unsigned>((total + threads - 1) / threads);
    if (max_blocks > 0 && blocks > static_cast<unsigned>(max_blocks)) blocks = static_cast<unsigned>(max_blocks);  // grid-stride
    if (src_half)
        B2_LAUNCH_RC = launch_kernel(input_cast_s2d_kernel<__half>, dim3(blocks), dim3(threads), 0, stream, false,
                                     static_cast<const __half*>(src), reinterpret_cast<uint4*>(dst), N, C, H, W, pad_l, pad_r);
    else
        B2_LAUNCH_RC = launch_kernel(input_cast_s2d_kernel<float>, dim3(blocks), dim3(threads), 0, stream, false,
                                     static_cast<const float*>(src), reinterpret_cast<uint4*>(dst), N, C, H, W, pad_l, pad_r);
    return B2_LAUNCH_RC;
}

// uint8 HWC images -> normalised fp32 -> fp16 (round to nearest).  (x - mean) * inv_std is one rounded subtract and one
// rounded multiply, never contracted into an FMA, so the values equal builder.preprocess_u8 bit for bit and the engine
// computes exactly what its fp32 binding computes on the preprocessed batch.
__device__ __forceinline__ float u8_norm(unsigned char v, float mean, float inv_std) {
    return __fmul_rn(__fsub_rn(static_cast<float>(v), mean), inv_std);
}

// One thread per packed output pixel (a PAIR of crop pixels): consecutive threads read consecutive 2*C-byte runs of the
// same source row, so a warp reads one contiguous span (no alignment assumed: crop_left * C may be odd).
__global__ void input_cast_u8_s2d_kernel(const unsigned char* __restrict__ src, uint4* __restrict__ dst, int N, int H, int W,
                                         int pad_l, int pad_r, U8Norm nrm) {
    pdl_launch_dependents();
    pdl_wait();
    const int W2 = W >> 1;
    const int Wp = W2 + pad_l + pad_r;
    const long long total = static_cast<long long>(N) * H * Wp, step = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total; idx += step) {
        const int wp = static_cast<int>(idx % Wp);
        const long long t = idx / Wp;
        const int h = static_cast<int>(t % H);
        const int n = static_cast<int>(t / H);
        const int w2 = wp - pad_l;
        uint4 o = make_uint4(0u, 0u, 0u, 0u);
        if (w2 >= 0 && w2 < W2) {
            const unsigned char* s =
                src + ((static_cast<size_t>(n) * nrm.src_h + nrm.top + h) * nrm.src_w + nrm.left + 2 * w2) * nrm.C;
            float f[8];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                f[c] = f[4 + c] = 0.f;
                if (c < nrm.C) {
                    f[c] = u8_norm(__ldg(s + nrm.perm[c]), nrm.mean[c], nrm.inv_std[c]);
                    f[4 + c] = u8_norm(__ldg(s + nrm.C + nrm.perm[c]), nrm.mean[c], nrm.inv_std[c]);
                }
            }
            __half2* o2 = reinterpret_cast<__half2*>(&o);
#pragma unroll
            for (int i = 0; i < 4; ++i) o2[i] = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
        }
        dst[idx] = o;
    }
}

// One thread per crop pixel, one 16-byte store of 8 fp16 channels; a warp reads 32 * C contiguous source bytes.
__global__ void input_cast_u8_c8_kernel(const unsigned char* __restrict__ src, uint4* __restrict__ dst, int N, int H, int W,
                                        U8Norm nrm) {
    pdl_launch_dependents();
    pdl_wait();
    const long long total = static_cast<long long>(N) * H * W, step = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total; idx += step) {
        const int w = static_cast<int>(idx % W);
        const long long t = idx / W;
        const int h = static_cast<int>(t % H);
        const int n = static_cast<int>(t / H);
        const unsigned char* s = src + ((static_cast<size_t>(n) * nrm.src_h + nrm.top + h) * nrm.src_w + nrm.left + w) * nrm.C;
        float f[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) f[c] = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c)
            if (c < nrm.C) f[c] = u8_norm(__ldg(s + nrm.perm[c]), nrm.mean[c], nrm.inv_std[c]);
        uint4 o;
        __half2* o2 = reinterpret_cast<__half2*>(&o);
#pragma unroll
        for (int i = 0; i < 4; ++i) o2[i] = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
        dst[idx] = o;
    }
}

int launch_input_cast_u8_s2d(const void* src, void* dst, int N, int H, int W, int pad_l, int pad_r, const U8Norm& nrm,
                             int max_blocks, cudaStream_t stream) {
    const long long total = static_cast<long long>(N) * H * (W / 2 + pad_l + pad_r);
    const int threads = 256;
    unsigned blocks = static_cast<unsigned>((total + threads - 1) / threads);
    if (max_blocks > 0 && blocks > static_cast<unsigned>(max_blocks)) blocks = static_cast<unsigned>(max_blocks);  // grid-stride
    B2_LAUNCH_RC = launch_kernel(input_cast_u8_s2d_kernel, dim3(blocks), dim3(threads), 0, stream, false,
                                 static_cast<const unsigned char*>(src), reinterpret_cast<uint4*>(dst), N, H, W, pad_l, pad_r, nrm);
    return B2_LAUNCH_RC;
}

int launch_input_cast_u8_c8(const void* src, void* dst, int N, int H, int W, const U8Norm& nrm, int max_blocks,
                            cudaStream_t stream) {
    const long long total = static_cast<long long>(N) * H * W;
    const int threads = 256;
    unsigned blocks = static_cast<unsigned>((total + threads - 1) / threads);
    if (max_blocks > 0 && blocks > static_cast<unsigned>(max_blocks)) blocks = static_cast<unsigned>(max_blocks);  // grid-stride
    B2_LAUNCH_RC = launch_kernel(input_cast_u8_c8_kernel, dim3(blocks), dim3(threads), 0, stream, false,
                                 static_cast<const unsigned char*>(src), reinterpret_cast<uint4*>(dst), N, H, W, nrm);
    return B2_LAUNCH_RC;
}

template <typename T>
__global__ void output_cast_kernel(const T* __restrict__ src, float* __restrict__ dst, int N, int C, int HW,
                                   int C_phys) {
    pdl_launch_dependents();
    pdl_wait();
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(N) * C * HW) return;
    const int px = static_cast<int>(idx % HW);
    const long long t = idx / HW;
    const int c = static_cast<int>(t % C);
    const int n = static_cast<int>(t / C);
    dst[idx] = to_f(src[(static_cast<size_t>(n) * HW + px) * C_phys + c]);
}

int launch_output_cast(const void* src, float* dst, int N, int C, int H, int W, int C_phys, bool half_storage,
                       cudaStream_t stream) {
    const long long total = static_cast<long long>(N) * C * H * W;
    const int threads = 256;
    const unsigned blocks = static_cast<unsigned>((total + threads - 1) / threads);
    if (half_storage)
        B2_LAUNCH_RC = launch_kernel(output_cast_kernel<__half>, dim3(blocks), dim3(threads), 0, stream, true, reinterpret_cast<const __half*>(src), dst, N, C, H * W, C_phys);
    else
        B2_LAUNCH_RC = launch_kernel(output_cast_kernel<float>, dim3(blocks), dim3(threads), 0, stream, true, reinterpret_cast<const float*>(src), dst, N, C, H * W, C_phys);
    return B2_LAUNCH_RC;
}

// max pool, NHWC, windows clipped to the image (Caffe ceil mode produces partial windows)
template <typename T>
__global__ void maxpool_kernel(const T* __restrict__ src, T* __restrict__ dst, int N, int H, int W, int C, int Ho,
                               int Wo, int k, int stride, int pad) {
    pdl_launch_dependents();
    pdl_wait();
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(N) * Ho * Wo * C) return;
    const int c = static_cast<int>(idx % C);
    long long t = idx / C;
    const int wo = static_cast<int>(t % Wo);
    t /= Wo;
    const int ho = static_cast<int>(t % Ho);
    const int n = static_cast<int>(t / Ho);
    float m = -INFINITY;
    for (int r = 0; r < k; ++r) {
        const int hi = ho * stride - pad + r;
        if (hi < 0 || hi >= H) continue;
        for (int s = 0; s < k; ++s) {
            const int wi = wo * stride - pad + s;
            if (wi < 0 || wi >= W) continue;
            m = fmaxf(m, to_f(src[((static_cast<size_t>(n) * H + hi) * W + wi) * C + c]));
        }
    }
    dst[idx] = from_f<T>(m);
}

// fp16 NHWC, 8 channels (16 bytes) per thread
__global__ void maxpool_h8_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int N, int H, int W,
                                  int C8, int Ho, int Wo, int k, int stride, int pad) {
    pdl_launch_dependents();
    pdl_wait();
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(N) * Ho * Wo * C8) return;
    const int c = static_cast<int>(idx % C8);
    long long t = idx / C8;
    const int wo = static_cast<int>(t % Wo);
    t /= Wo;
    const int ho = static_cast<int>(t % Ho);
    const int n = static_cast<int>(t / Ho);
    const __half2 ninf = __float2half2_rn(-INFINITY);
    __half2 m[4] = {ninf, ninf, ninf, ninf};
    for (int r = 0; r < k; ++r) {
        const int hi = ho * stride - pad + r;
        if (hi < 0 || hi >= H) continue;
        for (int s = 0; s < k; ++s) {
            const int wi = wo * stride - pad + s;
            if (wi < 0 || wi >= W) continue;
            const uint4 v = __ldg(src + ((static_cast<size_t>(n) * H + hi) * W + wi) * C8 + c);
            const __half2* v2 = reinterpret_cast<const __half2*>(&v);
#pragma unroll
            for (int i = 0; i < 4; ++i) m[i] = __hmax2(m[i], v2[i]);
        }
    }
    uint4 o;
    __half2* o2 = reinterpret_cast<__half2*>(&o);
#pragma unroll
    for (int i = 0; i < 4; ++i) o2[i] = m[i];
    dst[idx] = o;
}

int launch_maxpool(const void* src, void* dst, int N, int H, int W, int C_phys, int Ho, int Wo, int k, int stride,
                   int pad, bool half_storage, cudaStream_t stream) {
    const int threads = 256;
    if (half_storage && C_phys % 8 == 0) {
        const long long total = static_cast<long long>(N) * Ho * Wo * (C_phys / 8);
        B2_LAUNCH_RC = launch_kernel(maxpool_h8_kernel, dim3(static_cast<unsigned>((total + threads - 1) / threads)), dim3(threads), 0, stream, true, 
            reinterpret_cast<const uint4*>(src), reinterpret_cast<uint4*>(dst), N, H, W, C_phys / 8, Ho, Wo, k, stride, pad);
    } else {
        const long long total = static_cast<long long>(N) * Ho * Wo * C_phys;
        const unsigned blocks = static_cast<unsigned>((total + threads - 1) / threads);
        if (half_storage)
            B2_LAUNCH_RC = launch_kernel(maxpool_kernel<__half>, dim3(blocks), dim3(threads), 0, stream, true, reinterpret_cast<const __half*>(src), reinterpret_cast<__half*>(dst), N, H, W, C_phys, Ho, Wo, k, stride, pad);
        else
            B2_LAUNCH_RC = launch_kernel(maxpool_kernel<float>, dim3(blocks), dim3(threads), 0, stream, true, reinterpret_cast<const float*>(src), reinterpret_cast<float*>(dst), N, H, W, C_phys, Ho, Wo, k, stride, pad);
    }
    return B2_LAUNCH_RC;
}

template <typename T>
__global__ void avgpool_kernel(const T* __restrict__ src, T* __restrict__ dst, int N, int HW, int C) {
    pdl_launch_dependents();
    pdl_wait();
    using acc_t = typename Acc<T>::type;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= N * C) return;
    const int c = idx % C;
    const int n = idx / C;
    acc_t acc = 0;
    for (int i = 0; i < HW; ++i) acc += static_cast<acc_t>(to_f(src[(static_cast<size_t>(n) * HW + i) * C + c]));
    dst[idx] = from_f<T>(static_cast<float>(acc / static_cast<acc_t>(HW)));
}

// fp16 global average pool, 16 bytes per load: block = 32 channel groups (8 channels each) x 8 pixel slices; every slice
// sums its pixels (stride 8), the slices are added in fixed order through smem -> deterministic, ~7 loads per thread for
// the 7x7 plane instead of 49 dependent 2-byte loads
__global__ void __launch_bounds__(256) avgpool_h8_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int N, int HW, int C8) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float part[8][32][8];
    const int lane_cg = threadIdx.x & 31, slice = threadIdx.x >> 5;
    const int groups_per_img = (C8 + 31) / 32;
    const int n = blockIdx.x / groups_per_img;
    const int cg = (blockIdx.x - n * groups_per_img) * 32 + lane_cg;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    if (cg < C8) {
        const uint4* base = src + static_cast<size_t>(n) * HW * C8 + cg;
        for (int px = slice; px < HW; px += 8) {
            const uint4 v = __ldg(base + static_cast<size_t>(px) * C8);
            const __half2* h2 = reinterpret_cast<const __half2*>(&v);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 f = __half22float2(h2[i]);
                acc[2 * i] += f.x;
                acc[2 * i + 1] += f.y;
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) part[slice][lane_cg][i] = acc[i];
    __syncthreads();
    if (slice == 0 && cg < C8) {
        const float inv = 1.0f / static_cast<float>(HW);
        float tot[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float t = part[0][lane_cg][i];
#pragma unroll
            for (int sl = 1; sl < 8; ++sl) t += part[sl][lane_cg][i];
            tot[i] = t * inv;
        }
        uint4 o;
        __half2* o2 = reinterpret_cast<__half2*>(&o);
#pragma unroll
        for (int i = 0; i < 4; ++i) o2[i] = __floats2half2_rn(tot[2 * i], tot[2 * i + 1]);
        dst[static_cast<size_t>(n) * C8 + cg] = o;
    }
}

int launch_avgpool(const void* src, void* dst, int N, int HW, int C_phys, bool half_storage, cudaStream_t stream) {
    if (half_storage && C_phys % 8 == 0) {
        const int c8 = C_phys / 8;
        const unsigned blocks = static_cast<unsigned>(N * ((c8 + 31) / 32));
        B2_LAUNCH_RC = launch_kernel(avgpool_h8_kernel, dim3(blocks), dim3(256), 0, stream, true, reinterpret_cast<const uint4*>(src),
                                     reinterpret_cast<uint4*>(dst), N, HW, c8);
        return B2_LAUNCH_RC;
    }
    const int threads = 128;
    const unsigned blocks = static_cast<unsigned>((N * C_phys + threads - 1) / threads);
    if (half_storage)
        B2_LAUNCH_RC = launch_kernel(avgpool_kernel<__half>, dim3(blocks), dim3(threads), 0, stream, true, reinterpret_cast<const __half*>(src), reinterpret_cast<__half*>(dst), N, HW, C_phys);
    else
        B2_LAUNCH_RC = launch_kernel(avgpool_kernel<float>, dim3(blocks), dim3(threads), 0, stream, true, reinterpret_cast<const float*>(src), reinterpret_cast<float*>(dst), N, HW, C_phys);
    return B2_LAUNCH_RC;
}

// fully connected: one warp per output neuron, all batch rows (<= 8 per pass) share each weight read
template <typename T>
__global__ void fc_kernel(const T* __restrict__ in, const T* __restrict__ w, const float* __restrict__ bias,
                          float* __restrict__ out, int N, int K, int Cout) {
    pdl_launch_dependents();
    pdl_wait();
    using acc_t = typename Acc<T>::type;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= Cout) return;
    const T* wr = w + static_cast<size_t>(warp) * K;
    for (int nb = 0; nb < N; nb += 8) {
        acc_t acc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = 0;
        for (int kk = lane; kk < K; kk += 32) {
            const acc_t wv = static_cast<acc_t>(to_f(wr[kk]));
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (nb + i < N) acc[i] += wv * static_cast<acc_t>(to_f(in[static_cast<size_t>(nb + i) * K + kk]));
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            acc_t v = acc[i];
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0 && nb + i < N)
                out[static_cast<size_t>(nb + i) * Cout + warp] = static_cast<float>(v + static_cast<acc_t>(bias[warp]));
        }
    }
}

// fp16 fast path (K == 256 * KV, KV <= 8): one warp per output neuron; each lane first pulls its slice of the
// weight row into registers -- weights are constants, so this happens BEFORE the PDL wait and overlaps the
// previous kernel -- then up to 8 batch rows are staged in shared memory and reduced with warp shuffles.
template <int ROWS>
__global__ void __launch_bounds__(256)
fc_h8_kernel(const __half* __restrict__ in, const __half* __restrict__ w, const float* __restrict__ bias,
             float* __restrict__ out, int N, int K, int Cout) {
    extern __shared__ uint4 s_in[];  // [ROWS][K/8]
    const int kv = K / 8;            // uint4 per row
    const int per_lane = kv / 32;    // <= 8
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int j = blockIdx.x * (blockDim.x >> 5) + warp;
    uint4 wreg[8];
    if (j < Cout) {
        const uint4* wr = reinterpret_cast<const uint4*>(w + static_cast<size_t>(j) * K);
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (i < per_lane) wreg[i] = __ldg(wr + lane + 32 * i);
    }
    pdl_launch_dependents();
    pdl_wait();
    for (int nb = 0; nb < N; nb += ROWS) {
        const int rows = min(ROWS, N - nb);
        __syncthreads();
        for (int i = threadIdx.x; i < rows * kv; i += blockDim.x)
            s_in[i] = __ldg(reinterpret_cast<const uint4*>(in + static_cast<size_t>(nb) * K) + i);
        __syncthreads();
        if (j < Cout) {
            float acc[ROWS];
#pragma unroll
            for (int r = 0; r < ROWS; ++r) acc[r] = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (i < per_lane) {
                    const __half2* w2 = reinterpret_cast<const __half2*>(&wreg[i]);
                    float2 wf[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) wf[q] = __half22float2(w2[q]);
#pragma unroll
                    for (int r = 0; r < ROWS; ++r) {
                        if (r < rows) {
                            const uint4 xv = s_in[r * kv + lane + 32 * i];
                            const __half2* x2 = reinterpret_cast<const __half2*>(&xv);
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                const float2 xf = __half22float2(x2[q]);
                                acc[r] = fmaf(wf[q].x, xf.x, acc[r]);
                                acc[r] = fmaf(wf[q].y, xf.y, acc[r]);
                            }
                        }
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < ROWS; ++r) {
                float v = acc[r];
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (lane == 0 && r < rows) out[static_cast<size_t>(nb + r) * Cout + j] = v + bias[j];
            }
        }
    }
}

int launch_fc(const void* in, const void* w, const float* bias, float* out, int N, int K, int Cout, bool half_storage,
              cudaStream_t stream) {
    if (half_storage && K % 256 == 0 && K <= 2048) {
        const int threads = 128;  // 4 warps -> 4 neurons per block (250 blocks for the 1000-way classifier)
        const unsigned blocks = static_cast<unsigned>((Cout + 3) / 4);
        const size_t smem = static_cast<size_t>(K) * 2 * 8;
        static bool attr_set = false;
        if (!attr_set) {
            cudaFuncSetAttribute(fc_h8_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
            attr_set = true;
        }
        B2_LAUNCH_RC = launch_kernel(fc_h8_kernel<8>, dim3(blocks), dim3(threads), smem, stream, true, reinterpret_cast<const __half*>(in), reinterpret_cast<const __half*>(w), bias, out, N, K, Cout);
        return B2_LAUNCH_RC;
    }
    const int threads = 128;  // 4 warps
    const unsigned blocks = static_cast<unsigned>((Cout + 3) / 4);
    if (half_storage)
        B2_LAUNCH_RC = launch_kernel(fc_kernel<__half>, dim3(blocks), dim3(threads), 0, stream, true, reinterpret_cast<const __half*>(in), reinterpret_cast<const __half*>(w), bias, out, N, K, Cout);
    else
        B2_LAUNCH_RC = launch_kernel(fc_kernel<float>, dim3(blocks), dim3(threads), 0, stream, true, reinterpret_cast<const float*>(in), reinterpret_cast<const float*>(w), bias, out, N, K, Cout);
    return B2_LAUNCH_RC;
}

// row softmax, one 256-thread block per row
__global__ void softmax_kernel(const float* __restrict__ in, float* __restrict__ out, int C) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float red[32];
    const float* x = in + static_cast<size_t>(blockIdx.x) * C;
    float* y = out + static_cast<size_t>(blockIdx.x) * C;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    float m = -INFINITY;
    for (int i = threadIdx.x; i < C; i += blockDim.x) m = fmaxf(m, x[i]);
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) red[warp] = m;
    __syncthreads();
    m = red[0];
    for (int i = 1; i < nwarp; ++i) m = fmaxf(m, red[i]);
    __syncthreads();
    float s = 0.f;
    for (int i = threadIdx.x; i < C; i += blockDim.x) s += expf(x[i] - m);
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    s = 0.f;
    for (int i = 0; i < nwarp; ++i) s += red[i];
    const float inv = 1.0f / s;
    for (int i = threadIdx.x; i < C; i += blockDim.x) y[i] = expf(x[i] - m) * inv;
}

int launch_softmax(const float* in, float* out, int N, int C, cudaStream_t stream) {
    if (N <= 0) return 0;
    B2_LAUNCH_RC = launch_kernel(softmax_kernel, dim3(N), dim3(256), 0, stream, true, in, out, C);
    return B2_LAUNCH_RC;
}


// =================================================================================================
// tail_f16_kernel -- global average pool + fully connected + bias + softmax in ONE launch (fp16 engines).
//   The three operators are a dependency chain over tiny tensors (RN50, batch 8: 1.6 MB in, 4.1 MB of weights, 32 KB
//   out), so as separate kernels they are three launch + drain latencies.  Here the work is one ordered ticket list
//   -- pool items, then FC items (8 neurons each, one per warp), then one softmax item per image -- drawn by the CTAs of
//   a single grid; an FC item pulls its weight rows into registers BEFORE it waits for the pooled vector, a softmax item
//   waits for the logits.  In-order tickets drawn by running CTAs only make the waits deadlock-free without any
//   co-residency assumption.  The arithmetic (summation orders, fp16 rounding of the pooled vector, expf) is exactly
//   that of avgpool_h8_kernel / fc_h8_kernel / softmax_kernel: results are bit-identical to the unfused path.
//   Reference ops: models/ResNet-50-deploy.prototxt:2292-2302 (pool5) + InnerProduct + Softmax.
// =================================================================================================
__device__ __forceinline__ int tail_ld_relaxed(const int* p) {
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// A POLITE wait: relaxed loads with back-off while the counter is short, ONE acquire fence once it is not.  (An
// acquire load per iteration costs an L1 invalidation each time -- on an SM this CTA shares with other streams' kernels.)
__device__ __forceinline__ void tail_wait_counter(const int* p, int need) {
    uint32_t spins = 0;
    long long t0 = 0;
    while (tail_ld_relaxed(p) < need) {
        __nanosleep(64);
        if ((++spins & 0xFFFu) == 0) {
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000LL) __trap();
        }
    }
    asm volatile("fence.acq_rel.gpu;" ::: "memory");
}

// (256, 2): at most 128 registers per thread.  Unbounded the kernel took 154, i.e. 39 K registers per CTA -- more than an SM
// that already hosts three conv CTAs of OTHER contexts has left, so the tail's CTAs queued for emptier SMs and a forward pass
// at 4 contexts paid ~24 us for it (fused 51.1 k img/s against 53.1 k unfused; 52.4 k with the cap, 50.2 k at 80 registers where
// the spills cost more than the residency wins).  With the weight rows in shared memory the kernel needs 116 and spills nothing.
__global__ void __launch_bounds__(256, 2) tail_f16_kernel(const TailArgs a) {
    extern __shared__ uint4 s_dyn[];  // FC: [8][K/8] staged pooled rows
    __shared__ float part[8][32][8];
    __shared__ float red[32];
    __shared__ int s_ticket;
    __shared__ __align__(8) uint64_t wbar;  // the FC item's weight rows have landed in s_w (one bulk copy per item)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int C8 = a.C / 8;
    const int groups_per_img = (C8 + 31) / 32;
    const int n_pool = a.N * groups_per_img;
    const int n_fc = (a.Cout + 7) / 8;
    // counters: [0] FC tickets  [1] pool items done  [2] FC items done  [3] CTAs gone  [4] pool tickets  [5] softmax tickets
    // Order of work in a CTA: take an FC item and pull its weight rows into registers (constants: no dependency), THEN help
    // with the pooling until no pool ticket is left, then wait for the pooling, compute, and finally take softmax rows.
    // With one CTA per FC item (the default grid) the 4 MB of weights stream in while the pooling runs and the FC phase is a
    // single wave.  Deadlock-free for any grid: a CTA only ever waits for items whose tickets are held by RUNNING CTAs, and
    // those wait on nothing (pool) or on pool items only (FC).
    auto take = [&](int* counter, int limit) -> int {
        __syncthreads();
        if (threadIdx.x == 0) s_ticket = tail_ld_relaxed(counter) < limit ? atomicAdd(counter, 1) : limit;
        __syncthreads();
        return s_ticket;
    };
    const int K = a.C;
    const int kv = K / 8, per_lane = kv / 32;  // uint4 per row / per lane (<= 8)
    uint4* const s_w = s_dyn + 8 * kv;         // [8 neurons][K/8]: this item's weight rows
    if (threadIdx.x == 0) {
        mbar_init(&wbar, 1);
        fence_barrier_init();
        fence_proxy_async();
    }
    uint32_t wphase = 0;
    pdl_launch_dependents();
    bool waited = false;  // griddepcontrol.wait executed (before the first read of the previous kernel's output)
    for (;;) {
        const int f = take(a.ctrl + 0, n_fc);  // (its barriers also publish wbar's initialisation and retire the previous item)
        const bool have_fc = f < n_fc;
        const int j = f * 8 + warp;
        if (have_fc && threadIdx.x == 0) {
            // constants: ONE bulk copy (<= 8 consecutive rows = 32 KB) started before the dependency wait, in flight during the
            // pooling -- no registers held meanwhile (the kernel used to park the rows in 32 registers per thread)
            const int rows_w = min(8, a.Cout - f * 8);
            const uint32_t bytes = static_cast<uint32_t>(rows_w) * static_cast<uint32_t>(K) * 2u;
            mbar_expect_tx(&wbar, bytes);
            bulk_load_1d(&wbar, s_w, a.w + static_cast<size_t>(f) * 8 * K, bytes);
        }
        // ---------------- global average pool: (image, 256-channel group) items until none is left ----------------
        for (;;) {
            const int t = take(a.ctrl + 4, n_pool);
            if (t >= n_pool) break;
            if (!waited) pdl_wait(), waited = true;
            const int n = t / groups_per_img;
            const int cg = (t - n * groups_per_img) * 32 + lane;
            const int slice = warp;
            float acc[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = 0.f;
            if (cg < C8) {
                const uint4* base = reinterpret_cast<const uint4*>(a.in) + static_cast<size_t>(n) * a.HW * C8 + cg;
                // up to 8 of this slice's pixels are requested before the first is consumed (the loop was one L2 round trip
                // per pixel); they are still ADDED in ascending pixel order, so the sums keep their bits
                for (int px0 = slice; px0 < a.HW; px0 += 64) {
                    uint4 v[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        if (px0 + 8 * k < a.HW) v[k] = __ldg(base + static_cast<size_t>(px0 + 8 * k) * C8);
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        if (px0 + 8 * k < a.HW) {
                            const __half2* h2 = reinterpret_cast<const __half2*>(&v[k]);
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const float2 f = __half22float2(h2[i]);
                                acc[2 * i] += f.x;
                                acc[2 * i + 1] += f.y;
                            }
                        }
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) part[slice][lane][i] = acc[i];
            __syncthreads();
            if (slice == 0 && cg < C8) {
                const float inv = 1.0f / static_cast<float>(a.HW);
                float tot[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    float tt = part[0][lane][i];
#pragma unroll
                    for (int sl = 1; sl < 8; ++sl) tt += part[sl][lane][i];
                    tot[i] = tt * inv;
                }
                uint4 o;
                __half2* o2 = reinterpret_cast<__half2*>(&o);
#pragma unroll
                for (int i = 0; i < 4; ++i) o2[i] = __floats2half2_rn(tot[2 * i], tot[2 * i + 1]);
                reinterpret_cast<uint4*>(a.pooled)[static_cast<size_t>(n) * C8 + cg] = o;
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                __threadfence();
                atomicAdd(a.ctrl + 1, 1);
            }
        }
        if (have_fc) {
            // ---------------- fully connected: 8 neurons (one per warp) x all images ----------------
            if (!waited) pdl_wait(), waited = true;
            if (threadIdx.x == 0) tail_wait_counter(a.ctrl + 1, n_pool);
            __syncthreads();
            mbar_wait(&wbar, wphase);
            wphase ^= 1u;
            for (int nb = 0; nb < a.N; nb += 8) {
                const int rows = min(8, a.N - nb);
                __syncthreads();
                for (int i = threadIdx.x; i < rows * kv; i += blockDim.x)
                    s_dyn[i] = __ldcg(reinterpret_cast<const uint4*>(a.pooled + static_cast<size_t>(nb) * K) + i);
                __syncthreads();
                if (j < a.Cout) {
                    float acc[8];
#pragma unroll
                    for (int r = 0; r < 8; ++r) acc[r] = 0.f;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        if (i < per_lane) {
                            const uint4 wv = s_w[warp * kv + lane + 32 * i];
                            const __half2* w2 = reinterpret_cast<const __half2*>(&wv);
                            float2 wf[4];
#pragma unroll
                            for (int q = 0; q < 4; ++q) wf[q] = __half22float2(w2[q]);
#pragma unroll
                            for (int r = 0; r < 8; ++r) {
                                if (r < rows) {
                                    const uint4 xv = s_dyn[r * kv + lane + 32 * i];
                                    const __half2* x2 = reinterpret_cast<const __half2*>(&xv);
#pragma unroll
                                    for (int q = 0; q < 4; ++q) {
                                        const float2 xf = __half22float2(x2[q]);
                                        acc[r] = fmaf(wf[q].x, xf.x, acc[r]);
                                        acc[r] = fmaf(wf[q].y, xf.y, acc[r]);
                                    }
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int r = 0; r < 8; ++r) {
                        float v = acc[r];
                        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                        if (lane == 0 && r < rows) a.logits[static_cast<size_t>(nb + r) * a.Cout + j] = v + a.bias[j];
                    }
                }
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                __threadfence();
                atomicAdd(a.ctrl + 2, 1);
            }
            continue;  // another FC item, if the grid is smaller than the item list
        }
        // ---------------- softmax: one image per ticket, once every FC item is in ----------------
        for (;;) {
            const int n = take(a.ctrl + 5, a.N);
            if (n >= a.N) break;
            if (!waited) pdl_wait(), waited = true;
            if (threadIdx.x == 0) tail_wait_counter(a.ctrl + 2, n_fc);
            __syncthreads();
            const float* x = a.logits + static_cast<size_t>(n) * a.Cout;
            float* y = a.out + static_cast<size_t>(n) * a.Cout;
            const int nwarp = blockDim.x >> 5;
            // the row is read ONCE (<= 8 logits per thread stay in registers through max, sum and normalisation: three L2 round
            // trips became one); rows wider than 8 x blockDim fall back to re-reading.  Same operations in the same order.
            constexpr int kKeep = 8;
            const bool keep = a.Cout <= kKeep * static_cast<int>(blockDim.x);
            float xv[kKeep];
            float m = -INFINITY;
            if (keep) {
#pragma unroll
                for (int k = 0; k < kKeep; ++k) {
                    const int i = threadIdx.x + k * blockDim.x;
                    xv[k] = i < a.Cout ? __ldcg(x + i) : -INFINITY;
                }
#pragma unroll
                for (int k = 0; k < kKeep; ++k) m = fmaxf(m, xv[k]);
            } else {
                for (int i = threadIdx.x; i < a.Cout; i += blockDim.x) m = fmaxf(m, __ldcg(x + i));
            }
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            if (lane == 0) red[warp] = m;
            __syncthreads();
            m = red[0];
            for (int i = 1; i < nwarp; ++i) m = fmaxf(m, red[i]);
            __syncthreads();
            float sum = 0.f;
            if (keep) {
#pragma unroll
                for (int k = 0; k < kKeep; ++k) {
                    const int i = threadIdx.x + k * blockDim.x;
                    if (i < a.Cout) {
                        xv[k] = expf(xv[k] - m);
                        sum += xv[k];
                    }
                }
            } else {
                for (int i = threadIdx.x; i < a.Cout; i += blockDim.x) sum += expf(__ldcg(x + i) - m);
            }
            for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            if (lane == 0) red[warp] = sum;
            __syncthreads();
            sum = 0.f;
            for (int i = 0; i < nwarp; ++i) sum += red[i];
            const float inv = 1.0f / sum;
            if (keep) {
#pragma unroll
                for (int k = 0; k < kKeep; ++k) {
                    const int i = threadIdx.x + k * blockDim.x;
                    if (i < a.Cout) y[i] = xv[k] * inv;
                }
            } else {
                for (int i = threadIdx.x; i < a.Cout; i += blockDim.x) y[i] = expf(__ldcg(x + i) - m) * inv;
            }
        }
        break;
    }
    // the last CTA to leave re-arms the counters for the next launch
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(a.ctrl + 3, 1) == static_cast<int>(gridDim.x) - 1) {
            a.ctrl[0] = 0, a.ctrl[1] = 0, a.ctrl[2] = 0, a.ctrl[4] = 0, a.ctrl[5] = 0;
            __threadfence();
            a.ctrl[3] = 0;
        }
    }
}

bool tail_f16_applies(int N, int HW, int C, int Cout) { return N >= 1 && HW >= 1 && C % 256 == 0 && C <= 2048 && Cout >= 1; }

int launch_tail_f16(const TailArgs& a, cudaStream_t stream) {
    if (!tail_f16_applies(a.N, a.HW, a.C, a.Cout)) return static_cast<int>(cudaErrorInvalidValue);
    const int items = a.N * ((a.C / 8 + 31) / 32) + (a.Cout + 7) / 8 + a.N;
    static int cap = -1, use_pdl = -1;
    if (cap < 0) {
        const char* v = getenv("B2_TAIL_CTAS");
        cap = v ? atoi(v) : 148;  // one wave: every FC item (8 neurons) gets its own CTA, so the weight rows stream in one round
        if (cap < 1) cap = 1;
        v = getenv("B2_TAIL_PDL");
        use_pdl = v ? atoi(v) : 1;
    }
    const unsigned blocks = static_cast<unsigned>(items < cap ? items : cap);
    const size_t smem = static_cast<size_t>(a.C) * 2 * 8 * 2;  // pooled rows of 8 images + the weight rows of 8 neurons
    static bool attr_set = false;
    if (!attr_set) {
        cudaFuncSetAttribute(tail_f16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        attr_set = true;
    }
    B2_LAUNCH_RC = launch_kernel(tail_f16_kernel, dim3(blocks), dim3(256), smem, stream, use_pdl != 0, a);
    return B2_LAUNCH_RC;
}

}  // namespace b2k
