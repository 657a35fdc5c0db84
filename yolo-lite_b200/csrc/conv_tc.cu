// Implicit-GEMM convolution on the 5th-gen tensor cores (tcgen05 + TMEM), operands fed AND results drained by
// TMA.
//
//   D[M = 128 output pixels, N = co_tile] = sum over taps (r,s) and channel blocks of
//       A[pixels shifted by the tap, kblk channels]  x  W[co_tile, kblk]
//
// * activations are NHWC bf16; the A tile of one tap is a TH x TW spatial patch of TN images fetched by a
//   single 4-D TMA box {kblk, TW, TH, TN}; the conv halo and ragged image edges are TMA out-of-bounds
//   zero fill (signed coordinates), so there is no im2col buffer and no padding pass;
// * stride-2 convs read one of four "parity planes" (h%2, w%2) of the input, each its own 4-D tensor map,
//   so a tap is again a dense box;
// * 1x1 convs run in flat mode: the whole (n,h,w) extent is one axis and tiles are 128 consecutive pixels;
// * weights are packed [co][tap][ci] bf16 (K-major), fetched by a 2-D TMA box {kblk, co_tile};
// * both tiles land in the canonical K-major swizzled layout (SW128/64/32 for kblk 64/32/16) that
//   tcgen05.mma reads through shared-memory descriptors; accumulation is fp32 in TMEM;
// * epilogue: two groups of 4 warps, group g owns TMEM accumulator stage g (tiles alternate between the
//   groups).  Per 32-column chunk: tcgen05.ld -> +bias (smem) -> SiLU (1 MUFU) -> +residual -> bf16/f32 ->
//   swizzled staging tile in smem -> ONE TMA store of the {chunk, TW, TH, TN} box into the channel slice of
//   the destination (concat = aliasing; ragged rows / channel tails are clipped by the tensor map).  The
//   nearest-2x upsample is four more TMA stores of the same staging tile into the parity planes of the
//   upsampled destination, so a result that feeds both a Concat and an Upsample->Concat is computed once.
//
// Warp roles: warp 0 = TMA producer (one lane), warp 1 = TMEM owner + MMA issuer (one lane),
// warps 2..9 = epilogue.  Pipeline: `stages`-deep smem ring with full/empty mbarriers; tcgen05.commit
// releases a stage back to the producer and finally signals the epilogue group of that accumulator.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "conv_tc.cuh"

namespace yl {


// Persistent: gridDim.x CTAs each walk tiles blockIdx.x, +gridDim.x, ...  The TMA producer runs ahead across
// tile boundaries (the smem ring never drains), and with two TMEM accumulator stages the epilogue of tile i
// overlaps the loads and MMAs of tiles i+1, i+2.
// B2B = true: the back-to-back instantiation (a second 1x1 GEMM + Detect decode behind the conv, see conv_tc.cuh); a
// separate instantiation so that the production kernel's code and register allocation stay exactly what they were.
template <bool DBG, bool B2B = false>
__global__ void __launch_bounds__(kConvTcThreads, 2) conv_tc_kernel(const __grid_constant__ ConvTcParams p) {
    extern __shared__ uint8_t smem_raw[];
    // broadcast from lane 0 so the compiler treats the warp index (and every role / tile index derived from it)
    // as warp-uniform
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;

    // ---- shared memory carve-up (1024-B aligned: required by the 128-B swizzle atom)
    const uint32_t raw = smem_u32(smem_raw);
    uint8_t* base = smem_raw + (((raw + 1023u) & ~1023u) - raw);
    uint8_t* sA = base;
    uint8_t* sB = sA + (size_t)p.stages * p.a_bytes;
    uint8_t* sStg = sB + (size_t)p.b_region;  // [2 groups][stg_bufs][stg_bytes]
    float* sbias = reinterpret_cast<float*>(sStg + 2 * (size_t)p.stg_bufs * p.stg_bytes);
    const int nbias = p.n_tiles * p.co_tile + 32;                          // chunk tails read past co_tile
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(sbias + ((nbias + 3) & ~3));
    uint64_t* empty_bar = full_bar + p.stages;
    uint64_t* tfull_bar = empty_bar + p.stages;   // [2] accumulator ready for its epilogue group
    uint64_t* tempty_bar = tfull_bar + 2;         // [2] accumulator drained
    uint64_t* w_bar = tempty_bar + 2;             // patch mode: resident weights landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_bar + 1);
    // back-to-back mode: second GEMM's weight tiles, bias and barriers live behind everything else
    uint8_t* sB3 = nullptr;
    float* sbias3 = nullptr;
    uint64_t *a2_full = nullptr, *a2_empty = nullptr, *tfull2_bar = nullptr, *tempty2_bar = nullptr, *w3_bar = nullptr;
    if constexpr (B2B) {
        const uint32_t t = smem_u32(tmem_slot + 1);
        sB3 = reinterpret_cast<uint8_t*>(tmem_slot + 1) + (((t + 1023u) & ~1023u) - t);
        sbias3 = reinterpret_cast<float*>(sB3 + (size_t)p.k2blocks * p.b3_bytes);
        a2_full = reinterpret_cast<uint64_t*>(sbias3 + ((p.co_tile3 + 32 + 3) & ~3));
        a2_empty = a2_full + 2;
        tfull2_bar = a2_empty + 2;
        tempty2_bar = tfull2_bar + 2;
        w3_bar = tempty2_bar + 2;
    }

    // programmatic dependent launch: let the next kernel of the stream start its prologue as our CTAs retire
    griddep_launch_dependents();
    if (threadIdx.x == 0) YL_STAMP(0);
    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&tfull_bar[s], 1);
            mbar_init(&tempty_bar[s], 4);  // one arrive per epilogue warp of the group
        }
        mbar_init(w_bar, 1);
        if constexpr (B2B) {
            for (int s = 0; s < 2; ++s) {
                mbar_init(&a2_full[s], 1);
                mbar_init(&a2_empty[s], 1);
                mbar_init(&tfull2_bar[s], 1);
                mbar_init(&tempty2_bar[s], 4);
            }
            mbar_init(w3_bar, 1);
        }
        mbar_fence_init();
    }
    if (warp == 1) {
        tmem_alloc(tmem_slot, p.tmem_cols);
        tmem_relinquish();
    }
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tmA[0]);
        tma_prefetch_desc(&p.tmB);
        if (p.store_y) tma_prefetch_desc(&p.tmY[p.y_map_first]);
    }
    {
        const float bs = p.act ? 0.5f : 1.0f;   // activated convs stage b / 2 (the epilogue works on h = x / 2)
        for (int i = threadIdx.x; i < nbias; i += blockDim.x) sbias[i] = i < p.n_bias ? bs * __ldg(p.bias + i) : 0.f;
        if constexpr (B2B)
            for (int i = threadIdx.x; i < p.co_tile3 + 32; i += blockDim.x) sbias3[i] = i < p.n_bias3 ? __ldg(p.bias3 + i) : 0.f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) YL_STAMP(1);
    const int taps = p.ksize * p.ksize;
    const int kiters = taps * p.cin_blocks;
    if constexpr (B2B) {
        // the second GEMM's weights are constants: fetched before the dependency wait
        if (warp == 0 && elect_one()) {
            mbar_expect_tx(w3_bar, (uint32_t)p.k2blocks * (uint32_t)p.co_tile3 * 128u);
            for (int kb = 0; kb < p.k2blocks; ++kb) tma_load_2d(sB3 + (size_t)kb * p.b3_bytes, &p.tmB3, w3_bar, kb * 64, 0);
        }
    }
    // resident weights are constants too: their TMA loads are issued before the dependency wait, so they fly
    // while the previous kernel of the stream is still draining
    if (warp == 0 && p.wearly && (p.patch || p.wres) && elect_one()) {
        mbar_expect_tx(w_bar, p.w_bytes);
        if (p.patch) {
            tma_load_3d(sB, &p.tmW3, w_bar, 0, 0, 0);
        } else {
            int ki = 0;
            for (int tap = 0; tap < taps; ++tap)
                for (int cb = 0; cb < p.cin_blocks; ++cb, ++ki)
                    tma_load_2d(sB + (size_t)ki * p.b_bytes, &p.tmB, w_bar, tap * p.ci_pad + cb * p.kblk, 0);
        }
    }
    // everything above touched only constants (weights, bias, tensor maps); activations written by the
    // previous kernel of the stream are read / overwritten only after it has completed
    griddep_wait();
    if (threadIdx.x == 0) YL_STAMP(2);
    if (warp == 0 && !p.wearly && (p.patch || p.wres) && elect_one()) {
        mbar_expect_tx(w_bar, p.w_bytes);
        if (p.patch) {
            tma_load_3d(sB, &p.tmW3, w_bar, 0, 0, 0);
        } else {
            int ki = 0;
            for (int tap = 0; tap < taps; ++tap)
                for (int cb = 0; cb < p.cin_blocks; ++cb, ++ki)
                    tma_load_2d(sB + (size_t)ki * p.b_bytes, &p.tmB, w_bar, tap * p.ci_pad + cb * p.kblk, 0);
        }
    }

    // Producer and MMA warps run their loops warp-uniformly (all 32 lanes wait on the mbarriers and compute the
    // same coordinates / descriptors, so they live in uniform registers) and one elected lane issues the TMA /
    // tcgen05 instructions: a `lane == 0` branch instead makes every operand "possibly divergent" and costs a
    // register->uniform waterfall loop per issued instruction.
    if (warp == 0) {
        // ================= TMA producer =================
        const bool leader = elect_one();
        int st = 0;
        uint32_t ph = 0;  // ring position / phase of the stage being filled
        if (p.patch) {
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
                int wt, ht;
                const int mt = fast_divmod(tile, p.fd_tiles_w, &wt);
                const int i0 = fast_divmod(mt, p.fd_tiles_h, &ht);
                const int w0 = wt * p.TW, h0 = ht * p.TH;
                mbar_wait(&empty_bar[st], ph ^ 1u);
                if (leader) {
                    mbar_expect_tx(&full_bar[st], p.tx_bytes);
                    tma_load_4d(sA + (size_t)st * p.a_bytes, &p.tmA[0], &full_bar[st], 0, w0 - 1, h0 - 1, i0);
                }
                if (++st == p.stages) {
                    st = 0;
                    ph ^= 1u;
                }
            }
        } else {
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
                int nt, wt, ht;
                int mt = fast_divmod(tile, p.fd_ntiles, &nt);
                mt = fast_divmod(mt, p.fd_tiles_w, &wt);
                const int it = fast_divmod(mt, p.fd_tiles_h, &ht);
                const int w0 = wt * p.TW, h0 = ht * p.TH, i0 = it * p.TN;
                const int n0 = nt * p.co_tile;
                int tap = 0;
                for (int r = 0; r < p.ksize; ++r) {
                    for (int s2 = 0; s2 < p.ksize; ++s2, ++tap) {
                        const int offh = r - p.pad, offw = s2 - p.pad;
                        int map = 0, dh = offh, dw = offw;
                        if (p.stride == 2) {
                            const int ph2 = offh & 1, pw2 = offw & 1;
                            map = ph2 * 2 + pw2;
                            dh = (offh - ph2) >> 1;
                            dw = (offw - pw2) >> 1;
                        }
                        for (int cb = 0; cb < p.cin_blocks; ++cb) {
                            mbar_wait(&empty_bar[st], ph ^ 1u);
                            if (leader) {
                                mbar_expect_tx(&full_bar[st], p.tx_bytes);
                                tma_load_4d(sA + (size_t)st * p.a_bytes, &p.tmA[map], &full_bar[st], cb * p.kblk,
                                            w0 + dw, h0 + dh, i0);
                                if (!p.wres)
                                    tma_load_2d(sB + (size_t)st * p.b_bytes, &p.tmB, &full_bar[st],
                                                tap * p.ci_pad + cb * p.kblk, n0);
                            }
                            if (++st == p.stages) {
                                st = 0;
                                ph ^= 1u;
                            }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        const bool leader = elect_one();
        const uint32_t idesc = umma_idesc_bf16(128, (uint32_t)p.co_tile);
        const uint32_t rb = (uint32_t)p.kblk * 2u;  // operand row bytes = swizzle span
        const int ksteps = p.kblk / 16;
        int st = 0;
        uint32_t ph = 0;
        int acc = 0;
        uint32_t acc_ph = 0;
        if (p.patch || p.wres) {
            mbar_wait(w_bar, 0);
            tc_fence_after();
        }
        // back-to-back: D2[g] = A2[g] (this CTA's j-th tile, written by epilogue group g = j & 1) x W3^T, issued one tile
        // behind the first GEMM so that neither waits for the other's epilogue
        int ntile = 0;
        auto mma2 = [&](int j) {
            const int g2 = j & 1;
            const uint32_t ph2 = (uint32_t)(j >> 1) & 1u;
            mbar_wait(&a2_full[g2], ph2);
            mbar_wait(&tempty2_bar[g2], ph2 ^ 1u);
            tc_fence_after();
            if (leader) {
                const uint32_t idesc2 = umma_idesc_bf16(128, (uint32_t)p.co_tile3);
                const uint32_t d2 = tmem_base + (uint32_t)(2 * p.acc_stride + g2 * p.acc3_stride);
                for (int kb = 0; kb < p.k2blocks; ++kb) {
                    const int ks2 = (min(64, p.c2_ch - kb * 64) + 15) >> 4;
                    const uint64_t da2 = umma_desc_kmajor(smem_u32(sStg + (size_t)g2 * p.stg_bufs * p.stg_bytes + (size_t)kb * 16384), 128u);
                    const uint64_t db2 = umma_desc_kmajor(smem_u32(sB3 + (size_t)kb * p.b3_bytes), 128u);
                    for (int k = 0; k < ks2; ++k)
                        umma_bf16(d2, da2 + (uint64_t)(2 * k), db2 + (uint64_t)(2 * k), idesc2, (kb > 0 || k > 0) ? 1u : 0u);
                }
                umma_commit(&a2_empty[g2]);
                umma_commit(&tfull2_bar[g2]);
            }
        };
        if constexpr (B2B) {
            mbar_wait(w3_bar, 0);
            tc_fence_after();
        }
        if (p.patch) {
            const uint32_t sbo = (uint32_t)p.patch_pw * rb;       // next 8-row group = next patch row (TW == 8)
            const uint32_t wtap = (uint32_t)p.co_tile * rb;       // bytes of one tap's weight tile
            const uint32_t b0 = smem_u32(sB);
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
                mbar_wait(&tempty_bar[acc], acc_ph ^ 1u);
                mbar_wait(&full_bar[st], ph);
                tc_fence_after();
                if (leader && tile == (int)blockIdx.x) YL_STAMP(3);
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.acc_stride);
                const uint32_t a0 = smem_u32(sA + (size_t)st * p.a_bytes);
                if (leader) {
                    uint32_t first = 0;
                    uint32_t arow = a0;
                    uint32_t bt = b0;
                    for (int r = 0; r < 3; ++r, arow += (uint32_t)p.patch_pw * rb) {
                        for (int s2 = 0; s2 < 3; ++s2, bt += wtap) {
                            const uint32_t astart = arow + (uint32_t)s2 * rb;
                            const uint32_t bo = p.patch_bo ? ((astart >> 7) & 7u) : 0u;
                            const uint64_t da = umma_desc_kmajor_ex(astart, rb, sbo, bo);
                            const uint64_t db = umma_desc_kmajor(bt, rb);
                            for (int k = 0; k < ksteps; ++k) {
                                umma_bf16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, first);
                                first = 1u;
                            }
                        }
                    }
                    umma_commit(&empty_bar[st]);
                    umma_commit(&tfull_bar[acc]);
                }
                if (++st == p.stages) {
                    st = 0;
                    ph ^= 1u;
                }
                acc ^= 1;
                if (acc == 0) acc_ph ^= 1u;
                if constexpr (B2B) {
                    if (ntile > 0) mma2(ntile - 1);
                    ++ntile;
                }
            }
        } else {
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
                mbar_wait(&tempty_bar[acc], acc_ph ^ 1u);  // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.acc_stride);
                for (int ki = 0; ki < kiters; ++ki) {
                    mbar_wait(&full_bar[st], ph);
                    tc_fence_after();
                    if (leader && tile == (int)blockIdx.x && ki == 0) YL_STAMP(3);
                    if (leader) {
                        const uint64_t da = umma_desc_kmajor(smem_u32(sA + (size_t)st * p.a_bytes), rb);
                        const uint64_t db = umma_desc_kmajor(smem_u32(sB + (size_t)(p.wres ? ki : st) * p.b_bytes), rb);
                        for (int k = 0; k < ksteps; ++k) {
                            // advance 16 bf16 (32 B) along K inside the swizzle atom: +2 in the (addr >> 4) field
                            umma_bf16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc,
                                      (ki > 0 || k > 0) ? 1u : 0u);
                        }
                        umma_commit(&empty_bar[st]);
                    }
                    if (++st == p.stages) {
                        st = 0;
                        ph ^= 1u;
                    }
                }
                if (leader) umma_commit(&tfull_bar[acc]);
                acc ^= 1;
                if (acc == 0) acc_ph ^= 1u;
                if constexpr (B2B) {
                    if (ntile > 0) mma2(ntile - 1);
                    ++ntile;
                }
            }
        }
        if constexpr (B2B) {
            if (ntile > 0) mma2(ntile - 1);
        }
    } else {
        // ================= epilogue =================
        const int e = warp - 2;
        const int g = e >> 2;    // epilogue group = accumulator stage
        const int q = warp & 3;  // TMEM lane quadrant this warp may read
        const int gtid = (e & 3) * 32 + lane;
        uint8_t* stg = sStg + (size_t)g * p.stg_bufs * p.stg_bytes;
        const TileRange tr = {(int)blockIdx.x, p.total_tiles, (int)gridDim.x};
        uint32_t acc_uses = 0;
        // epi_kind: 0 / 1 = the hot instantiations (32-column chunks, bf16 NHWC store, SiLU, without / with residual),
        // 2 = every other combination
        // epi_kind (host side, plan_conv_tc): the hot combinations get their own instantiation (32-column chunks):
        //   0 / 1  SiLU, bf16 store, without / with residual        2 / 3  no activation, bf16 store, without / with residual
        //   4 / 5 / 6  Detect box decode / class decode / class filter WITHOUT an NHWC store (engine path head convs)
        //   7  everything else (fp32 destination, decode + raw store, 16-column chunks)
#define YL_EPI(CW_, ACT_, RES_, DET_, GEN_) \
    conv_tc_epilogue<CW_, ACT_, RES_, DET_, GEN_, DBG>(p, p, tr, acc_uses, g, q, lane, gtid, tmem_base, tfull_bar, tempty_bar, \
                                                       stg, sbias)
        if constexpr (B2B) {
            uint8_t* a2 = sStg + (size_t)g * p.stg_bufs * p.stg_bytes;
            if (p.act)
                conv_tc_epilogue_b2b<true>(p, tr, g, q, lane, gtid, tmem_base, tfull_bar, tempty_bar, a2_full, a2_empty,
                                           tfull2_bar, tempty2_bar, a2, sbias, sbias3);
            else
                conv_tc_epilogue_b2b<false>(p, tr, g, q, lane, gtid, tmem_base, tfull_bar, tempty_bar, a2_full, a2_empty,
                                            tfull2_bar, tempty2_bar, a2, sbias, sbias3);
        } else {
        const int kind = DBG ? 7 : p.epi_kind;     // the timeline build keeps only the generic code
        if (kind == 0) YL_EPI(32, true, false, 0, false);
        else if (kind == 1) YL_EPI(32, true, true, 0, false);
        else if (kind == 2) YL_EPI(32, false, false, 0, false);
        else if (kind == 3) YL_EPI(32, false, true, 0, false);
        else if (kind == 4) YL_EPI(32, false, false, YL_DET_BOX, false);
        else if (kind == 5) YL_EPI(32, false, false, YL_DET_CLS, false);
        else if (kind == 6) YL_EPI(32, false, false, YL_DET_CLS_FILTER, false);
        else if (p.cw == 32) YL_EPI(32, false, false, 0, true);
        else YL_EPI(16, false, false, 0, true);
        }
#undef YL_EPI
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, p.tmem_cols);
    if (threadIdx.x == 0) YL_STAMP(7);
}

// ------------------------------------------------------------------------------------------------ host side
// yl_debug_timeline: device buffer of [capacity][16] timestamps; state of the CALLING THREAD (the thread that arms it
// is the one whose launches are stamped), so concurrent users of the library are unaffected
static thread_local unsigned long long* g_dbg_buf = nullptr;
static thread_local int g_dbg_cap = 0, g_dbg_next = 0;
static int g_max_dyn_smem = 0;
static int g_num_sms = 148;

static void read_knobs();

int init_conv_tc() {
    read_knobs();
    int dev = 0;
    YL_CUDA(cudaGetDevice(&dev));
    int max_optin = 0;
    YL_CUDA(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    g_max_dyn_smem = max_optin;
    YL_CUDA(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
    YL_CUDA(cudaFuncSetAttribute(conv_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin));
    YL_CUDA(cudaFuncSetAttribute(conv_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin));
    YL_CUDA((cudaFuncSetAttribute(conv_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin)));
    return YL_OK;
}

bool encode_map(CUtensorMap* m, CUtensorMapDataType dt, void* base, int rank, const uint64_t* dims,
                       const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle sw) {
    EncodeTiledFn enc = get_encode_tiled();
    if (!enc) {
        set_error("yl_init() was not called (TMA encoder unresolved)");
        return false;
    }
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(m, dt, (cuuint32_t)rank, base, dims, strides_bytes, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d): rank %d dims [%llu,%llu,%llu,%llu] box [%u,%u,%u,%u]", (int)r,
                  rank, (unsigned long long)dims[0], (unsigned long long)dims[1],
                  (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0), box[0],
                  box[1], rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0);
        return false;
    }
    return true;
}

CUtensorMapSwizzle swizzle_for_bytes(int row_bytes) {
    return row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                            : (row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}

// A-tile box (TW, TH, TN) with TW*TH*TN <= 128 output pixels, possibly spanning images: minimise the number
// of 128-row MMA tiles needed to cover (Wo, Ho, N); ties prefer wide boxes (longer contiguous runs).
static void choose_patch(int Ho, int Wo, int N, int* TH, int* TW, int* TN) {
    long long best = -1;
    int bw = 1, bh = 1, bn = 1;
    for (int tw = Wo < 128 ? Wo : 128; tw >= 1; --tw) {
        if (tw != Wo && (tw & (tw - 1))) continue;  // full width or a power of two
        for (int th = 1; th * tw <= 128 && th <= Ho; ++th) {
            int tn = 128 / (tw * th);
            if (tn > N) tn = N;
            // TN > 1 stacks the same (tw, th) window of consecutive images: the box is a 4-D hyper-rectangle
            const long long tiles = (long long)ceil_div(Wo, tw) * ceil_div(Ho, th) * ceil_div(N, tn);
            if (best < 0 || tiles < best) {
                best = tiles;
                bw = tw;
                bh = th;
                bn = tn;
            }
        }
    }
    *TW = bw;
    *TH = bh;
    *TN = bn;
}

static bool conv_tc_supported_ex(const yl_conv_args* a, char* why, size_t why_len, bool allow_no_output);
bool conv_tc_supported(const yl_conv_args* a, char* why, size_t why_len) {
    return conv_tc_supported_ex(a, why, why_len, false);
}
static bool conv_tc_supported_ex(const yl_conv_args* a, char* why, size_t why_len, bool allow_no_output) {
#define NOPE(msg)                                   \
    do {                                            \
        if (why) snprintf(why, why_len, "%s", msg); \
        return false;                               \
    } while (0)
    const yl_tensor& x = a->x;
    const yl_tensor& y = a->y;
    if (x.dtype != YL_BF16) NOPE("input must be bf16");
    if (!(a->k == 1 || a->k == 3)) NOPE("k must be 1 or 3");
    if (!(a->stride == 1 || a->stride == 2)) NOPE("stride must be 1 or 2");
    if (x.c % 8 || x.coff % 8 || x.cstride % 8) NOPE("input channels/offset/stride must be multiples of 8");
    if (y.c % 8 || y.coff % 8 || y.cstride % 8) NOPE("output channels/offset/stride must be multiples of 8");
    if (a->ci_pad % 8 || a->ci_pad < x.c) NOPE("ci_pad must be a multiple of 8 and >= x.c");
    if (a->co_pad % 8 || a->co_pad < y.c) NOPE("co_pad must be a multiple of 8 and >= y.c");
    if (a->stride == 2 && ((x.h | x.w) & 1)) NOPE("stride 2 needs even input dims");
    if (a->res.data && (a->res.c % 8 || a->res.coff % 8 || a->res.cstride % 8 || a->res.dtype != YL_BF16))
        NOPE("residual must be bf16 with 8-channel alignment");
    if (a->y_up.data && (a->y_up.c != y.c || a->y_up.coff % 8 || a->y_up.cstride % 8 || a->y_up.dtype != y.dtype))
        NOPE("y_up must match y's channels and dtype with 8-channel alignment");
    if (a->y_up.data && a->upsample2x) NOPE("y_up and upsample2x are mutually exclusive");
    if (((uintptr_t)x.data | (uintptr_t)y.data | (uintptr_t)a->w | (uintptr_t)a->bias | (uintptr_t)a->res.data |
         (uintptr_t)a->y_up.data) & 15)
        NOPE("pointers must be 16-byte aligned");
    if (a->det.pred) {
        const yl_det_epilogue& d = a->det;
        if (a->k != 1 || a->stride != 1 || a->upsample2x || a->y_up.data || a->res.data || a->act)
            NOPE("Detect-decode epilogue needs a plain 1x1 stride-1 conv without activation / residual / upsample");
        if (d.mode == YL_DET_BOX) {
            if (d.reg_max != 16 || y.c != 64) NOPE("Detect box decode is built for reg_max == 16 (64 channels)");
        } else if (d.mode == YL_DET_CLS) {
            if (y.c != d.nc || y.c > 256) NOPE("Detect class decode needs co == nc <= 256");
        } else if (d.mode == YL_DET_CLS_FILTER) {
            if (y.c != d.nc || y.c > 256) NOPE("Detect class filter needs co == nc <= 256");
            if (!d.cand_ws || !(d.conf >= 0.f && d.conf <= 1.f)) NOPE("Detect class filter needs a workspace and conf in [0,1]");
            if ((long long)d.A * d.nc >= (1ll << 32)) NOPE("A * nc must fit 32 bits");
        } else {
            NOPE("bad Detect-decode mode");
        }
        if (d.nc < 1 || d.A < 1 || d.anchor0 < 0 || d.anchor0 + x.h * x.w > d.A) NOPE("bad Detect-decode anchor range");
    } else if (!y.data && !allow_no_output) {
        NOPE("null output");
    }
    return true;
#undef NOPE
}

// Tensor maps of a destination of conv-output resolution (Ho, Wo) [up == 0, one map] or of the 2x-upsampled
// resolution [up == 1, four parity-plane maps]; flat mode describes the pixel axis as one dimension.
bool encode_out_maps(CUtensorMap* maps, const yl_tensor& y, int Ho, int Wo, int N, bool flat, bool up,
                            const uint32_t* box, CUtensorMapSwizzle sw) {
    const uint64_t es = (y.dtype == YL_F32) ? 4 : 2;
    const CUtensorMapDataType dt = (y.dtype == YL_F32) ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    uint8_t* yb = reinterpret_cast<uint8_t*>(y.data) + (size_t)y.coff * es;
    const uint64_t cs = (uint64_t)y.cstride * es;
    if (!up) {
        if (flat) {
            const uint64_t M = (uint64_t)N * Ho * Wo;
            uint64_t dims[4] = {(uint64_t)y.c, M, 1, 1};
            uint64_t str[3] = {cs, cs * M, cs * M};
            return encode_map(&maps[0], dt, yb, 4, dims, str, box, sw);
        }
        uint64_t dims[4] = {(uint64_t)y.c, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
        uint64_t str[3] = {cs, cs * Wo, cs * Wo * Ho};
        return encode_map(&maps[0], dt, yb, 4, dims, str, box, sw);
    }
    const uint64_t W2 = 2ull * Wo, H2 = 2ull * Ho;
    for (int dy = 0; dy < 2; ++dy)
        for (int dx = 0; dx < 2; ++dx) {
            uint64_t dims[4] = {(uint64_t)y.c, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
            uint64_t str[3] = {2 * cs, 2 * cs * W2, cs * W2 * H2};
            if (!encode_map(&maps[dy * 2 + dx], dt, yb + ((size_t)dy * W2 + dx) * cs, 4, dims, str, box, sw)) return false;
        }
    return true;
}

static int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

// Tuning knobs (A/B switches used by tools/): read from the environment ONCE, in yl_init; launches never touch getenv.
struct ConvTcKnobs {
    int nsplit = 1, patch = 1, patch_k64 = 0, patch_wmax_kb = 80, small_nsplit = 1, patch_pitch = 10, patch_bo = 0;
    int chain_nsplit = 1, chain_patch = 1, chain_bres = 1;
    int wres = 1, stg_sub = 2, stg_bufs = 2, wearly = 1, grid_ctas = 2, patch_eff_pct = 60;
};
static ConvTcKnobs g_knobs;
static void read_knobs() {
    ConvTcKnobs k;
    k.nsplit = env_int("YL_NSPLIT", k.nsplit);
    k.patch = env_int("YL_PATCH", k.patch);
    k.patch_k64 = env_int("YL_PATCH_K64", k.patch_k64);
    k.patch_wmax_kb = env_int("YL_PATCH_WMAX_KB", k.patch_wmax_kb);
    k.small_nsplit = env_int("YL_SMALL_NSPLIT", k.small_nsplit);
    k.patch_pitch = env_int("YL_PATCH_PITCH", k.patch_pitch);
    k.patch_bo = env_int("YL_PATCH_BO", k.patch_bo);
    k.wres = env_int("YL_WRES", k.wres);
    k.stg_sub = env_int("YL_STG_SUB", k.stg_sub);
    k.stg_bufs = env_int("YL_STG_BUFS", k.stg_bufs);
    k.wearly = env_int("YL_WEARLY", k.wearly);
    k.grid_ctas = env_int("YL_GRID_CTAS", k.grid_ctas);
    k.patch_eff_pct = env_int("YL_PATCH_EFF", k.patch_eff_pct);
    k.chain_nsplit = env_int("YL_CHAIN_NSPLIT", k.chain_nsplit);
    k.chain_patch = env_int("YL_CHAIN_PATCH", k.chain_patch);
    k.chain_bres = env_int("YL_CHAIN_BRES", k.chain_bres);
    g_knobs = k;
}

// Everything of a launch that is decided on the host: tiling, mode (flat / halo patch / resident weights / N split),
// smem carve-up and the tensor maps.  Shared by the launch and by yl_conv_tc_info (tests assert which path ran).
int plan_conv_tc(const yl_conv_args* a, ConvTcParams& p, int* grid_out, size_t* smem_out, const ConvTcPlanOpts* opts) {
    char why[128];
    const yl_conv_args* head = opts ? opts->head : nullptr;
    YL_CHECK(conv_tc_supported_ex(a, why, sizeof(why), head != nullptr), YL_ERR_UNSUPPORTED, "tcgen05 conv unsupported: %s", why);
    if (head) {
        const yl_det_epilogue& d = head->det;
        YL_CHECK(!a->det.pred && !a->y.data && !a->res.data && !a->y_up.data && !a->upsample2x && a->y.dtype == YL_BF16,
                 YL_ERR_UNSUPPORTED, "back-to-back: the first conv is a plain bf16 conv whose result is not stored");
        YL_CHECK(head->k == 1 && head->stride == 1 && !head->act && !head->res.data && !head->y_up.data && !head->upsample2x &&
                     !head->y.data && d.pred && (d.mode == YL_DET_BOX || d.mode == YL_DET_CLS),
                 YL_ERR_UNSUPPORTED, "back-to-back: the head conv is a plain 1x1 with a box / class decode epilogue, not stored");
        YL_CHECK(head->x.c == a->y.c && a->y.c <= 128 && head->y.c <= 128 && head->y.c % 8 == 0 && head->ci_pad >= head->x.c &&
                     head->ci_pad % 8 == 0 && head->co_pad >= head->y.c && head->co_pad % 8 == 0,
                 YL_ERR_UNSUPPORTED, "back-to-back: channel counts (<= 128, head input = conv output)");
        YL_CHECK(d.mode == YL_DET_BOX ? (d.reg_max == 16 && head->y.c == 64) : (head->y.c == d.nc), YL_ERR_UNSUPPORTED,
                 "back-to-back: box decode needs reg_max 16 (64 channels), class decode co == nc");
        YL_CHECK(d.nc >= 1 && d.A >= 1 && d.anchor0 >= 0, YL_ERR_ARG, "bad Detect-decode anchor range");
        YL_CHECK((((uintptr_t)head->w | (uintptr_t)head->bias) & 15) == 0, YL_ERR_ARG, "pointers must be 16-byte aligned");
    }
    const yl_tensor& x = a->x;
    const yl_tensor& y = a->y;
    const int pad = a->k / 2;
    const int Ho = (x.h + 2 * pad - a->k) / a->stride + 1;
    const int Wo = (x.w + 2 * pad - a->k) / a->stride + 1;
    const int up = a->upsample2x ? 2 : 1;
    YL_CHECK(y.n == x.n && y.h == Ho * up && y.w == Wo * up, YL_ERR_ARG,
             "conv output dims mismatch: got (%d,%d,%d) expected (%d,%d,%d)", y.n, y.h, y.w, x.n, Ho * up, Wo * up);
    if (a->y_up.data)
        YL_CHECK(a->y_up.n == x.n && a->y_up.h == 2 * Ho && a->y_up.w == 2 * Wo, YL_ERR_ARG,
                 "y_up dims mismatch: got (%d,%d,%d) expected (%d,%d,%d)", a->y_up.n, a->y_up.h, a->y_up.w, x.n, 2 * Ho,
                 2 * Wo);

    const bool chain = opts && opts->chain;
    if (chain)
        YL_CHECK(!a->det.pred && y.data && y.dtype == YL_BF16, YL_ERR_UNSUPPORTED,
                 "a conv chain takes bf16 -> bf16 layers without a Detect epilogue");
    memset(&p, 0, sizeof(p));
    p.ksize = a->k;
    p.stride = a->stride;
    p.pad = pad;
    p.ci_pad = a->ci_pad;
    // channel block = TMA box row: one 128-B row costs the TMA unit about as much as a 32-B row, so round the
    // channel count up (48 -> one 64-wide block whose tail is OOB zero fill) rather than splitting it
    p.kblk = x.c > 32 ? 64 : (x.c > 16 ? 32 : 16);
    p.cin_blocks = ceil_div(x.c, p.kblk);
    const CUtensorMapSwizzle sw = swizzle_for_bytes(p.kblk * 2);
    const CUtensorMapDataType bf = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;

    // N tiling
    const int co16 = ceil_div(y.c, 16) * 16;
    int n_tiles = ceil_div(co16, chain ? 128 : 256);
    // A 129..256-wide tile needs all 512 TMEM columns for its two accumulator stages, i.e. one CTA per SM.  When the
    // M tiling then yields between one and two waves of CTAs (20x20 maps at bs = 64: 200 tiles on 148 SMs), the
    // second wave runs almost alone; halving the tile (2 CTAs/SM, 256 columns each) keeps every tile resident at once.
    {
        const long long m_est = ceil_div64((long long)x.n * Ho * Wo, 128);
        // (a Detect epilogue runs as one N tile, see below)
        if (!chain && n_tiles == 1 && co16 > 128 && m_est > g_num_sms && m_est <= 2ll * g_num_sms && g_knobs.nsplit &&
            !a->det.pred)
            n_tiles = 2;
    }
    // The epilogue drains and stores whole cw-column chunks (32 whenever n_tiles > 1), so every N tile but the last must
    // be a multiple of 32 wide: a tile ending mid-chunk (co 144 as two 80-wide tiles) would store its out-of-tile
    // accumulator columns over the first channels of the next tile.
    p.co_tile = n_tiles > 1 ? ceil_div(ceil_div(co16, n_tiles), 32) * 32 : co16;

    // halo-patch mode: 3x3 stride-1 convs on thin inputs are L2->SM bound when every tap is fetched separately
    // (9 narrow TMA boxes per tile); fetch the (TH+2) x (TW+2) patch once instead and slide the A descriptor
    bool patch = false;
    if (!chain && a->k == 3 && a->stride == 1 && x.c <= 64 && n_tiles == 1 && g_knobs.patch) {
        const int kb = g_knobs.patch_k64 ? 64 : p.kblk;
        const double eff = (double)Ho * Wo / ((double)ceil_div(Wo, 8) * 8 * ceil_div(Ho, 16) * 16);
        if (9 * p.co_tile * kb * 2 <= g_knobs.patch_wmax_kb * 1024 && eff * 100.0 >= (double)g_knobs.patch_eff_pct) {
            patch = true;
            p.kblk = kb;
            p.cin_blocks = 1;
        }
    }
    // Small problems (bs = 1 latency): with far fewer 128-pixel tiles than SMs a CTA's epilogue walks its N / 32 column
    // chunks serially (~0.45 us each, tools/timeline.py) while most of the GPU idles.  Split N down to 32-column tiles:
    // the chunks become parallel CTAs (the A tile is re-read from L2 by each, which is free at this size).
    if (!chain && !patch && g_knobs.small_nsplit && !a->det.pred) {
        const long long m_est = ceil_div64((long long)x.n * Ho * Wo, 128);
        int nt = n_tiles;
        while (m_est * nt * 2 <= g_num_sms && co16 % (64 * nt) == 0 && co16 / (2 * nt) >= 32) nt *= 2;
        if (nt != n_tiles) {
            n_tiles = nt;
            p.co_tile = co16 / nt;
        }
    }
    // Detect epilogues take every channel of a pixel in ONE N tile: the box decode (four DFL sides) and the class filter
    // (running best class) keep per-pixel state across the chunks, and the decode addresses prediction rows by the chunk
    // index inside the tile.  (Splitting the class conv would only help nc % 64 == 0 or nc > 128 at small batches; a
    // tile-aware decode measured ~0.2 % slower at bs = 64 on a B200 at 1000 W: it changes the register allocation of the
    // whole production kernel.)
    YL_CHECK(n_tiles == 1 || !a->det.pred, YL_ERR_UNSUPPORTED, "a Detect epilogue needs one N tile (got %d)", n_tiles);
    const CUtensorMapSwizzle swp = swizzle_for_bytes(p.kblk * 2);

    // M tiling + activation tensor maps
    __nv_bfloat16* xb = reinterpret_cast<__nv_bfloat16*>(x.data) + x.coff;
    const uint64_t es = 2;
    const bool flat = (!chain && a->k == 1 && a->stride == 1 && !a->upsample2x && !a->y_up.data);
    if (patch) {
        p.patch = 1;
        p.patch_pw = g_knobs.patch_pitch;
        p.patch_bo = g_knobs.patch_bo;  // measured: the swizzle XOR uses absolute smem address bits
        YL_CHECK(p.patch_pw >= 10 && p.patch_pw <= 16, YL_ERR_ARG, "YL_PATCH_PITCH must be in [10, 16]");
        p.Ho = Ho;
        p.Wo = Wo;
        p.Nimg = x.n;
        p.TW = 8;
        p.TH = 16;
        p.TN = 1;
        p.tiles_w = ceil_div(Wo, 8);
        p.tiles_h = ceil_div(Ho, 16);
        p.tiles_n = x.n;
        uint32_t box[4] = {(uint32_t)p.kblk, (uint32_t)p.patch_pw, 18u, 1u};
        uint64_t dims[4] = {(uint64_t)x.c, (uint64_t)x.w, (uint64_t)x.h, (uint64_t)x.n};
        uint64_t str[3] = {(uint64_t)x.cstride * es, (uint64_t)x.cstride * es * x.w,
                           (uint64_t)x.cstride * es * x.w * x.h};
        if (!encode_map(&p.tmA[0], bf, xb, 4, dims, str, box, swp)) return YL_ERR_CUDA;
        // weights [co_pad][9][ci_pad] viewed as {ci, co, tap}
        const uint64_t K = 9ull * a->ci_pad;
        uint64_t wd[3] = {(uint64_t)a->ci_pad, (uint64_t)a->co_pad, 9};
        uint64_t ws[2] = {K * es, (uint64_t)a->ci_pad * es};
        uint32_t wb[3] = {(uint32_t)p.kblk, (uint32_t)p.co_tile, 9u};
        if (!encode_map(&p.tmW3, bf, const_cast<void*>(a->w), 3, wd, ws, wb, swp)) return YL_ERR_CUDA;
        p.tmB = p.tmW3;  // (prefetched by the producer; unused otherwise)
    } else if (flat) {
        const uint64_t M = (uint64_t)x.n * x.h * x.w;
        YL_CHECK(M < (1ull << 31), YL_ERR_ARG, "too many pixels");
        p.Ho = 1;
        p.Wo = (int)M;
        p.Nimg = 1;
        p.TH = 1;
        p.TW = 128;
        p.TN = 1;
        p.tiles_h = 1;
        p.tiles_n = 1;
        p.tiles_w = ceil_div((int)M, 128);
        uint64_t dims[4] = {(uint64_t)x.c, M, 1, 1};
        uint64_t str[3] = {(uint64_t)x.cstride * es, (uint64_t)x.cstride * es * M, (uint64_t)x.cstride * es * M};
        uint32_t box[4] = {(uint32_t)p.kblk, 128, 1, 1};
        if (!encode_map(&p.tmA[0], bf, xb, 4, dims, str, box, sw)) return YL_ERR_CUDA;
    } else {
        p.Ho = Ho;
        p.Wo = Wo;
        p.Nimg = x.n;
        choose_patch(Ho, Wo, chain ? 1 : x.n, &p.TH, &p.TW, &p.TN);
        if (chain && g_knobs.chain_nsplit) {
            // a cluster of `chain_cluster` CTAs owns one image: give every CTA (at least) two tiles per layer when the
            // channel count allows, so both epilogue groups of a CTA drain an accumulator at the same time
            const int tm = ceil_div(Ho, p.TH) * ceil_div(Wo, p.TW);
            // (1x1 only: every extra N tile of a 3x3 re-reads the nine shifted A boxes, and those layers are bound by
            // L2 -> SM traffic, tools/chain_timeline.py)
            // ... unless the cluster is large (tiny batches: the image must be spread over many SMs and L2 is idle)
            while ((a->k == 1 || opts->chain_cluster > 4) && tm * n_tiles < 2 * opts->chain_cluster &&
                   co16 % (64 * n_tiles) == 0 && co16 / (2 * n_tiles) >= 32)
                n_tiles *= 2;
            p.co_tile = ceil_div(ceil_div(co16, n_tiles), 16) * 16;
        }
        // chain, 3x3 stride 1: "full-width patch".  The M rows of a tile are (TW = Wo + 2) x TH consecutive positions of a
        // zero-padded (Wo + 2)-wide image, so tap (r, s) of the whole tile is the SAME shared-memory patch read from a start
        // address shifted by r * TW + s rows: ONE TMA box {kblk, Wo + 2, TH + 2} per tile and channel block instead of nine
        // (these layers are bound by L2 -> SM bytes and by the TMA box-row rate, not by math).  The two surplus columns of
        // every row compute junk that the destination tensor map clips (columns Wo, Wo + 1 are out of bounds).
        if (chain && a->k == 3 && a->stride == 1 && Wo + 2 <= 128 && p.cin_blocks <= 2 && g_knobs.chain_patch) {
            p.ch_mode = 1;
            p.TW = Wo + 2;
            p.TH = 128 / p.TW < Ho ? 128 / p.TW : Ho;
            p.TN = 1;
        }
        p.tiles_h = ceil_div(Ho, p.TH);
        p.tiles_w = ceil_div(Wo, p.TW);
        p.tiles_n = ceil_div(x.n, p.TN);
        uint32_t box[4] = {(uint32_t)p.kblk, (uint32_t)p.TW, (uint32_t)(p.ch_mode ? p.TH + 2 : p.TH), (uint32_t)p.TN};
        if (a->stride == 1) {
            uint64_t dims[4] = {(uint64_t)x.c, (uint64_t)x.w, (uint64_t)x.h, (uint64_t)x.n};
            uint64_t str[3] = {(uint64_t)x.cstride * es, (uint64_t)x.cstride * es * x.w,
                               (uint64_t)x.cstride * es * x.w * x.h};
            if (!encode_map(&p.tmA[0], bf, xb, 4, dims, str, box, sw)) return YL_ERR_CUDA;
        } else {
            for (int ph = 0; ph < 2; ++ph)
                for (int pw = 0; pw < 2; ++pw) {
                    uint64_t dims[4] = {(uint64_t)x.c, (uint64_t)x.w / 2, (uint64_t)x.h / 2, (uint64_t)x.n};
                    uint64_t str[3] = {(uint64_t)x.cstride * es * 2, (uint64_t)x.cstride * es * x.w * 2,
                                       (uint64_t)x.cstride * es * x.w * x.h};
                    __nv_bfloat16* b = xb + ((size_t)ph * x.w + pw) * x.cstride;
                    if (!encode_map(&p.tmA[ph * 2 + pw], bf, b, 4, dims, str, box, sw)) return YL_ERR_CUDA;
                }
        }
    }
    // weights: [co_pad][k*k*ci_pad] bf16
    if (!patch) {
        const uint64_t K = (uint64_t)a->k * a->k * a->ci_pad;
        uint64_t dims[2] = {K, (uint64_t)a->co_pad};
        uint64_t str[1] = {K * es};
        uint32_t box[2] = {(uint32_t)p.kblk, (uint32_t)p.co_tile};
        if (!encode_map(&p.tmB, bf, const_cast<void*>(a->w), 2, dims, str, box, sw)) return YL_ERR_CUDA;
    }

    // epilogue chunking
    p.y_f32 = (y.dtype == YL_F32);
    const int oes = p.y_f32 ? 4 : 2;
    p.cw = p.co_tile >= 32 ? 32 : 16;
    p.nchunks = ceil_div(p.co_tile, p.cw);
    p.acc_stride = p.nchunks * p.cw;

    p.a_bytes = 128u * p.kblk * 2u;
    p.b_bytes = ((uint32_t)p.co_tile * p.kblk * 2u + 1023u) & ~1023u;
    p.tx_bytes = (uint32_t)(p.TW * p.TH * p.TN) * p.kblk * 2u + (uint32_t)p.co_tile * p.kblk * 2u;
    if (patch) {
        p.tx_bytes = (uint32_t)p.patch_pw * 18u * p.kblk * 2u;
        p.a_bytes = (p.tx_bytes + 1023u) & ~1023u;
        p.w_bytes = 9u * p.co_tile * p.kblk * 2u;
        p.b_bytes = (p.w_bytes + 1023u) & ~1023u;
    }
    if (chain) {
        const uint32_t rb = (uint32_t)p.kblk * 2u;
        p.ch_a_tx = (uint32_t)(p.TW * (p.ch_mode ? p.TH + 2 : p.TH) * p.TN) * rb;
        p.ch_b_tx = (uint32_t)p.co_tile * rb;
        // the last tap of accumulator row 127 reads patch row 127 + 2 * TW + 2
        if (p.ch_mode) p.a_bytes = ((uint32_t)(130 + 2 * p.TW) * rb + 1023u) & ~1023u;
    }
    p.m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
    p.n_tiles = n_tiles;
    p.total_tiles = p.m_tiles * n_tiles;
    YL_CHECK((long long)p.m_tiles * n_tiles < (1ll << 31), YL_ERR_ARG, "too many tiles");
    p.fd_ntiles = make_fastdiv(n_tiles);
    p.fd_tiles_w = make_fastdiv(p.tiles_w);
    p.fd_tiles_h = make_fastdiv(p.tiles_h);
    // two accumulator stages (one per epilogue group); two CTAs per SM when TMEM and smem allow
    uint32_t cols = 32;
    while ((int)cols < 2 * p.acc_stride) cols <<= 1;
    YL_CHECK(cols <= 512, YL_ERR_UNSUPPORTED, "accumulator needs %u TMEM columns", cols);
    if (head) {
        YL_CHECK(n_tiles == 1 && p.cw == 32, YL_ERR_UNSUPPORTED, "back-to-back needs one N tile of 32-column chunks");
        p.b2b = 1;
        p.c2_ch = y.c;
        p.k2blocks = ceil_div(p.co_tile, 64);
        p.co_tile3 = ceil_div(head->y.c, 16) * 16;
        p.nchunks3 = ceil_div(p.co_tile3, 32);
        p.acc3_stride = p.nchunks3 * 32;
        p.b3_bytes = ((uint32_t)p.co_tile3 * 128u + 1023u) & ~1023u;
        p.bias3 = head->bias;
        p.n_bias3 = head->co_pad;
        while ((int)cols < 2 * p.acc_stride + 2 * p.acc3_stride) cols <<= 1;
        YL_CHECK(cols <= 512, YL_ERR_UNSUPPORTED, "back-to-back accumulators need %u TMEM columns", cols);
        uint64_t dims[2] = {(uint64_t)head->ci_pad, (uint64_t)head->co_pad};
        uint64_t str[1] = {(uint64_t)head->ci_pad * 2};
        uint32_t box[2] = {64u, (uint32_t)p.co_tile3};
        if (!encode_map(&p.tmB3, bf, const_cast<void*>(head->w), 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B)) return YL_ERR_CUDA;
    }
    p.tmem_cols = cols;
    int ctas_per_sm = (cols <= 256) ? 2 : 1;
    if (chain) YL_CHECK(cols <= 256, YL_ERR_UNSUPPORTED, "chain layer needs %u TMEM columns (two CTAs share an SM)", cols);
    if (patch && p.b_bytes > 40u * 1024u) ctas_per_sm = 1;  // big resident 9-tap weights: one CTA owns the SM
    const int kiters_total = a->k * a->k * p.cin_blocks;
    const size_t wres_bytes = (size_t)kiters_total * p.b_bytes;
    if (!chain && !patch && n_tiles == 1 && g_knobs.wres &&
        wres_bytes <= (size_t)(ctas_per_sm == 2 ? 48 : 120) * 1024) {
        p.wres = 1;
        p.w_bytes = (uint32_t)kiters_total * (uint32_t)p.co_tile * p.kblk * 2u;
        p.tx_bytes = (uint32_t)(p.TW * p.TH * p.TN) * p.kblk * 2u;
    }
    const int nbias = n_tiles * p.co_tile + 32;
    const uint32_t stage_bytes = (patch || p.wres) ? p.a_bytes : p.a_bytes + p.b_bytes;
    const size_t fixed_b = patch ? p.b_bytes : (p.wres ? wres_bytes : 0);
    // (a chain CTA also keeps two copies of the parameter block and its barriers in front of the operand ring)
    const size_t cta_smem = chain ? (size_t)(112 * 1024 - 5632) : (size_t)(ctas_per_sm == 2 ? 112 * 1024 : 224 * 1024);

    // staging: prefer 128-B pixel rows per TMA store (two TMEM chunks of bf16) and two staging tiles per
    // epilogue group (the store of chunk k overlaps chunk k+1); fall back when the operand ring would get
    // too shallow to cover the HBM latency
    int sub_pref = (!p.y_f32 && p.cw == 32 && p.nchunks >= 2) ? 2 : 1;
    if (n_tiles > 1 && (p.nchunks & 1)) sub_pref = 1;  // a half-filled store row would spill into the next N tile
    sub_pref = g_knobs.stg_sub >= 2 ? sub_pref : 1;
    const int bufs_pref = g_knobs.stg_bufs >= 2 ? 2 : 1;
    const int cand[4][2] = {{sub_pref, bufs_pref}, {1, bufs_pref}, {sub_pref, 1}, {1, 1}};
    size_t fixed = 0;
    int stages = 0;
    for (int ci = 0; ci < 4; ++ci) {
        p.stg_sub = cand[ci][0];
        p.stg_bufs = cand[ci][1];
        p.stg_row_bytes = p.stg_sub * p.cw * oes;
        p.stg_bytes = (128u * (uint32_t)p.stg_row_bytes + 1023u) & ~1023u;  // 128 rows; 1024-B swizzle atoms
        fixed = 1024 + 2 * (size_t)p.stg_bufs * p.stg_bytes + (size_t)((nbias + 3) & ~3) * 4 + 16;
        if (head) {
            // the staging tiles double as the second GEMM's A tiles: a group needs k2blocks tiles of 128 rows x 128 B
            if ((size_t)p.stg_bufs * p.stg_bytes < (size_t)p.k2blocks * 16384) continue;
            fixed += 1024 + (size_t)p.k2blocks * p.b3_bytes + (size_t)((p.co_tile3 + 32 + 3) & ~3) * 4 + 9 * 8 + 64;
        }
        const long long budget = (long long)cta_smem - (long long)fixed - (long long)fixed_b - 16 * 24 - 64;
        if (chain) {
            // two rings: activations (ring A: one stage per k-iteration, or per (tile, channel block) patch) and weights
            // (ring B: one stage per k-iteration, or RESIDENT for the layer: a CTA of the cluster only ever sees one N
            // tile when n_tiles divides the cluster size, so its k-iterations' weight tiles are loaded once per layer)
            const int cs = opts->chain_cluster;
            const int kit = a->k * a->k * p.cin_blocks;
            const int a_set = p.ch_mode ? p.cin_blocks : 1;
            const int tiles_cta = ceil_div(p.tiles_w * p.tiles_h * n_tiles, cs);
            const long long ab = p.a_bytes, bb = p.b_bytes;
            int na = 0, nb = 0, bres = 0;
            if (g_knobs.chain_bres && cs % n_tiles == 0 && (long long)kit * bb + a_set * ab <= budget) {
                bres = 1;
                nb = kit;
                na = (int)((budget - (long long)kit * bb) / ab);
                const int sets = tiles_cta > 1 ? 2 : 1;
                if (p.ch_mode) na = (na / a_set < sets ? na / a_set : sets) * a_set;
                else if (na > 6) na = 6;
                if (!p.ch_mode && na < 2 && tiles_cta * kit > 1) bres = 0;   // a one-deep activation ring would serialise the loads
            }
            if (bres) {
            } else if (p.ch_mode) {
                na = a_set * ((tiles_cta > 1 && 2 * a_set * ab + 3 * bb <= budget) ? 2 : 1);
                nb = (int)((budget - na * ab) / bb);
                if (nb > 12) nb = 12;
            } else {
                na = nb = (int)(budget / (ab + bb));
                if (na > 6) na = nb = 6;
            }
            const bool ok = na >= a_set && na >= 1 && (bres || nb >= 2) && (p.ch_mode || bres || na >= 2);
            p.ch_na = na;
            p.ch_nb = nb;
            p.ch_bres = bres;
            stages = ok ? (na > 2 ? na : 2) : 0;
            if (ok) break;
            continue;
        }
        stages = budget > 0 ? (int)(budget / stage_bytes) : 0;
        if (stages >= 3 || (stages >= 2 && (size_t)stages * stage_bytes >= 40 * 1024)) break;
    }
    p.nstore = ceil_div(p.nchunks, p.stg_sub);
    if (chain) YL_CHECK(stages > 0, YL_ERR_UNSUPPORTED, "chain layer does not fit the shared-memory budget");
    if (head)
        YL_CHECK((size_t)p.stg_bufs * p.stg_bytes >= (size_t)p.k2blocks * 16384, YL_ERR_UNSUPPORTED,
                 "back-to-back: no shared memory left for the second GEMM's A tiles");
    if (stages > 12) stages = 12;
    if (stages < 2) stages = 2;
    p.stages = stages;
    p.b_region = (uint32_t)((patch || p.wres) ? fixed_b : (size_t)stages * p.b_bytes);
    const size_t smem = chain ? fixed + (size_t)p.ch_na * p.a_bytes + (size_t)p.ch_nb * p.b_bytes + 64
                              : fixed + fixed_b + (size_t)stages * stage_bytes + (2 * stages + 5) * 8 + 16;
    YL_CHECK((int)smem <= g_max_dyn_smem, YL_ERR_UNSUPPORTED, "conv tile needs %zu B smem (max %d)", smem,
             g_max_dyn_smem);

    // destination tensor maps: box = one store chunk of one tile
    if (y.data) {
        const CUtensorMapSwizzle osw = swizzle_for_bytes(p.stg_row_bytes);
        uint32_t obox[4] = {(uint32_t)(p.stg_sub * p.cw), (uint32_t)p.TW, (uint32_t)p.TH, (uint32_t)p.TN};
        if (a->upsample2x) {
            if (!encode_out_maps(&p.tmY[1], y, Ho, Wo, x.n, false, true, obox, osw)) return YL_ERR_CUDA;
            p.y_map_first = 1;
            p.y_map_last = 5;
        } else {
            if (!encode_out_maps(&p.tmY[0], y, Ho, Wo, x.n, flat, false, obox, osw)) return YL_ERR_CUDA;
            p.y_map_first = 0;
            p.y_map_last = 1;
            if (a->y_up.data) {
                if (!encode_out_maps(&p.tmY[1], a->y_up, Ho, Wo, x.n, false, true, obox, osw)) return YL_ERR_CUDA;
                p.y_map_last = 5;
            }
        }
    }

    p.store_y = y.data != nullptr;
    if (head) {
        p.det_mode = head->det.mode;
        p.det_pred = head->det.pred;
        p.det_nc = head->det.nc;
        p.det_A = head->det.A;
        p.det_anchor0 = head->det.anchor0;
        p.det_hw = Ho * Wo;
        p.det_w = Wo;
        p.det_stride = head->det.stride;
        p.det_M = (long long)x.n * Ho * Wo;
        YL_CHECK(head->det.anchor0 + Ho * Wo <= head->det.A, YL_ERR_ARG, "bad Detect-decode anchor range");
    }
    if (a->det.pred) {
        p.det_mode = a->det.mode;
        p.det_pred = a->det.pred;
        p.det_nc = a->det.nc;
        p.det_A = a->det.A;
        p.det_anchor0 = a->det.anchor0;
        p.det_hw = x.h * x.w;
        p.det_w = x.w;
        p.det_stride = a->det.stride;
        p.det_M = (long long)x.n * x.h * x.w;
        if (a->det.mode == YL_DET_CLS_FILTER) {
            p.det_conf = a->det.conf;
            p.det_cand_counts = reinterpret_cast<uint32_t*>(a->det.cand_ws);
            p.det_cand_keys = reinterpret_cast<unsigned long long*>(
                reinterpret_cast<char*>(a->det.cand_ws) + ((size_t)x.n * 4 + 255) / 256 * 256);
        }
    }
    p.wearly = g_knobs.wearly;
    p.bias = a->bias;
    p.n_bias = a->co_pad;
    p.act = a->act;
    p.res = reinterpret_cast<const __nv_bfloat16*>(a->res.data);
    p.res_cstride = a->res.cstride;
    p.res_coff = a->res.coff;
    p.res_c = a->res.c;
    p.epi_kind = 7;
    if (p.cw == 32 && !p.y_f32 && p.store_y && !p.det_mode)
        p.epi_kind = (p.act ? 0 : 2) + (p.res ? 1 : 0);
    else if (p.cw == 32 && !p.store_y && !p.act && !p.res && p.det_mode)
        p.epi_kind = p.det_mode == YL_DET_BOX ? 4 : (p.det_mode == YL_DET_CLS ? 5 : 6);

    int grid = g_num_sms * (ctas_per_sm < g_knobs.grid_ctas ? ctas_per_sm : g_knobs.grid_ctas);
    if (grid > p.total_tiles) grid = p.total_tiles;
    *grid_out = grid;
    *smem_out = smem;
    return YL_OK;
}

int launch_conv_b2b(const yl_conv_args* a, const yl_conv_args* head, cudaStream_t stream) {
    ConvTcParams p;
    int grid = 0;
    size_t smem = 0;
    ConvTcPlanOpts o;
    o.head = head;
    const int rc = plan_conv_tc(a, p, &grid, &smem, &o);
    if (rc != YL_OK) return rc;
    YL_CUDA(launch_kernel(conv_tc_kernel<false, true>, dim3(grid), dim3(kConvTcThreads), smem, stream, p));
    YL_LAUNCH_OK("conv_tc_kernel<b2b>");
    return YL_OK;
}

bool conv_b2b_supported(const yl_conv_args* a, const yl_conv_args* head) {
    ConvTcParams p;
    int grid = 0;
    size_t smem = 0;
    ConvTcPlanOpts o;
    o.head = head;
    return a && head && plan_conv_tc(a, p, &grid, &smem, &o) == YL_OK;
}

int launch_conv_tc(const yl_conv_args* a, cudaStream_t stream) {
    ConvTcParams p;
    int grid = 0;
    size_t smem = 0;
    const int rc = plan_conv_tc(a, p, &grid, &smem);
    if (rc != YL_OK) return rc;
    if (g_dbg_buf && g_dbg_next < g_dbg_cap) {
        p.dbg = g_dbg_buf + 16ll * g_dbg_next++;
        YL_CUDA(launch_kernel(conv_tc_kernel<true>, dim3(grid), dim3(kConvTcThreads), smem, stream, p));
    } else {
        YL_CUDA(launch_kernel(conv_tc_kernel<false>, dim3(grid), dim3(kConvTcThreads), smem, stream, p));
    }
    YL_LAUNCH_OK("conv_tc_kernel");
    return YL_OK;
}

int conv_tc_info(const yl_conv_args* a, yl_conv_tc_plan* out) {
    ConvTcParams p;
    int grid = 0;
    size_t smem = 0;
    const int rc = plan_conv_tc(a, p, &grid, &smem);
    if (rc != YL_OK) return rc;
    out->flat = (p.Ho == 1 && p.Nimg == 1 && p.TW == 128 && !p.patch) ? 1 : 0;
    out->patch = p.patch;
    out->wres = p.wres;
    out->tile_w = p.TW;
    out->tile_h = p.TH;
    out->tile_n = p.TN;
    out->m_tiles = p.m_tiles;
    out->n_tiles = p.n_tiles;
    out->co_tile = p.co_tile;
    out->kblk = p.kblk;
    out->stages = p.stages;
    out->grid = grid;
    out->smem_bytes = (int)smem;
    out->tmem_cols = (int)p.tmem_cols;
    out->cw = p.cw;
    out->stg_sub = p.stg_sub;
    out->epi_kind = p.epi_kind;
    return YL_OK;
}

}  // namespace yl

// Debug aid (tools/timeline.py): subsequent conv_tc launches get consecutive 8-slot rows of `device_buf`
// ([capacity][16] uint64) into which CTA 0 writes %globaltimer at: kernel start, prologue done, dependency wait
// done, first operands landed, first accumulator ready, last store issued, staging drained, exit.
extern "C" int yl_debug_timeline(unsigned long long* device_buf, int capacity) {
    yl::g_dbg_buf = device_buf;
    yl::g_dbg_cap = device_buf ? capacity : 0;
    yl::g_dbg_next = 0;
    return YL_OK;
}
