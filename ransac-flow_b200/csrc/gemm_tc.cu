// tcgen05 / TMEM / TMA tensor-core engine (sm_100a).
//
// One warp-specialised kernel, two epilogues:
//   MODE_CONV : implicit-GEMM convolution (stride 1) over a ragged NHWC batch, TF32 operands,
//               fp32 accumulation in TMEM, epilogue = folded-BN bias + residual + ReLU
//               (model/model.py:27-56,59-125,167-322; torchvision ResNet-50 conv1..layer3);
//   MODE_CORR : utils/outil.py:34-37 score = featA^T featB as 3xTF32 (hi*hi + lo*hi + hi*lo, fp32-grade
//               accuracy so the arg-max agrees with an fp32 GEMM) with the row / column arg-max fused
//               into the epilogue; the NA x NB matrix never leaves the SM.
//
// Data path per CTA (one 128-pixel x BN-channel output tile):
//   warp 0  : TMA producer.  A tile = 3-D box (32 channels, tw, th) of the NHWC image at the tap's
//             offset (out-of-bounds = zero padding for free), B tile = 2-D box (32 k, BN rows) of the
//             K-major weight matrix; both land in 128B-swizzled shared memory, mbarrier complete_tx.
//   warp 1  : allocates TMEM, issues tcgen05.mma.kind::tf32 (M=128, N=BN, K=8) x4 per stage from one
//             thread, tcgen05.commit releases the stage / publishes the accumulator.
//   warps 2-5: epilogue, tcgen05.ld 32 lanes x 32 columns at a time straight from TMEM.
#include <cuda.h>
#include <cuda_fp16.h>

#include <cstdlib>
#include <mutex>
#include <unordered_map>

#include "common.cuh"
#include "tc_common.cuh"

namespace rf {

struct alignas(64) TcParams {
    CUtensorMap mapA[RF_MAX_IMGS];        // per image: (C, W, H) fp32, box (32, tw, th)
    CUtensorMap mapY[RF_MAX_IMGS];        // per image: output (Cout, Wo, Ho), box (32, tw, th)   [TMA-store epilogue]
    CUtensorMap mapR[RF_MAX_IMGS];        // per image: residual, same geometry                   [TMA-load in the epilogue]
    CUtensorMap mapAlo;                   // MODE_CORR: low part of A
    CUtensorMap mapB;                     // (K, Cout) fp32, box (32, BN)
    CUtensorMap mapBlo;                   // MODE_CORR: low part of B
    int nimg;
    int tile_start[RF_MAX_IMGS + 1];      // prefix sums of tiles per image
    int tiles_x[RF_MAX_IMGS];
    int tw[RF_MAX_IMGS];                  // tile width (tile height = 128 / tw)
    int Ho[RF_MAX_IMGS], Wo[RF_MAX_IMGS];
    long long out_pix[RF_MAX_IMGS + 1];
    int R, S, pad, stride, Cin, Cout, relu, round_out, tma_epi;
    int stages;                           // fp16 tap-streaming kernel: ring depth chosen per layer on the host
    int res_pf;                           // fp16 tap-streaming kernel: residual tile prefetched into its own staging at CTA start
    int raster_n;                         // convolutions: channel tiles fastest in the grid (CTAs of one pixel tile run together)
    const float* bias;
    const float* residual;
    float* y;
    unsigned long long* rowbest;          // MODE_CORR
    unsigned long long* colbest;
    int NA, NB;
};


constexpr int MODE_CONV = 0, MODE_CORR = 1;

// Convolution epilogue shared by the tap-streaming and the halo kernels (warps 2..5 = 128 threads, thread m owns
// accumulator row m = pixel m of the tile): + folded-BN bias, + residual, ReLU, TF32 rounding, store.
// fp16 epilogue core (engine 2): thread m's accumulator row -> + bias, + residual, ReLU, saturate -> fp16 into the
// 128-byte-swizzled staging boxes (64 channels x 128 pixels x 2 B = 16 KB each; the residual boxes were TMA-loaded into
// the same place).  32 accumulator columns = 64 bytes = four 16-byte chunks of the pixel's 128-byte row.
template <int BN>
__device__ __forceinline__ void epi_rows_f16(const float* __restrict__ bias, int Cout, int relu, bool has_res, int n0, int m,
                                             uint32_t trow, uint8_t* stg) {
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
        uint32_t v[32];
        tmem_ld32(trow + c * 32, v);
        const int n = n0 + c * 32;
        uint8_t* rowp = stg + (c >> 1) * TC_A_BYTES + m * 128;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int chunk = (c & 1) * 4 + j;
            uint4* sp = reinterpret_cast<uint4*>(rowp + ((chunk ^ (m & 7)) << 4));
            float o[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = __uint_as_float(v[8 * j + e]);
            if (bias && n + 8 * j < Cout) {
                const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + n + 8 * j));
                const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + n + 8 * j + 4));
                o[0] += b0.x; o[1] += b0.y; o[2] += b0.z; o[3] += b0.w; o[4] += b1.x; o[5] += b1.y; o[6] += b1.z; o[7] += b1.w;
            }
            if (has_res) {
                const uint4 rr = *sp;
                const __half2* h = reinterpret_cast<const __half2*>(&rr);
#pragma unroll
                for (int e = 0; e < 4; ++e) { const float2 f = __half22float2(h[e]); o[2 * e] += f.x; o[2 * e + 1] += f.y; }
            }
            if (relu) {
#pragma unroll
                for (int e = 0; e < 8; ++e) o[e] = fmaxf(o[e], 0.f);
            }
            uint4 out;
            __half2* ho = reinterpret_cast<__half2*>(&out);
#pragma unroll
            for (int e = 0; e < 4; ++e)         // saturate instead of overflowing to inf
                ho[e] = __floats2half2_rn(fminf(fmaxf(o[2 * e], -65504.f), 65504.f), fminf(fmaxf(o[2 * e + 1], -65504.f), 65504.f));
            *sp = out;
        }
    }
}

template <int BN, bool F16 = false>
__device__ __forceinline__ void conv_epilogue(const TcParams& p, int img, int ox0, int oy0, int tw, int n0, int m, uint32_t trow,
                                              uint8_t* smem, uint64_t* res_full, int warp, int lane, bool res_issued = false) {
    if constexpr (F16) {
        // engine 2: always the bulk path (the host requires Cout % 8 == 0); boxes of 64 fp16 channels.  `smem` is the
        // staging area: the idle pipeline stages, or the dedicated residual staging when the producer warp already
        // issued the residual loads at CTA start (res_issued)
        constexpr int NBOX = BN / 64;
        uint8_t* stg = smem;
        const bool has_res = p.residual != nullptr;
        if (has_res) {
            if (!res_issued && warp == 2 && lane == 0) {
                mbar_expect_tx(res_full, NBOX * TC_A_BYTES);
#pragma unroll
                for (int b = 0; b < NBOX; ++b) tma_load_3d(stg + b * TC_A_BYTES, &p.mapR[img], res_full, n0 + b * 64, ox0, oy0);
            }
            mbar_wait(res_full, 0);
        }
        epi_rows_f16<BN>(p.bias, p.Cout, p.relu, has_res, n0, m, trow, stg);
        fence_proxy_async();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (warp == 2 && lane == 0) {
#pragma unroll
            for (int b = 0; b < NBOX; ++b)
                if (n0 + b * 64 < p.Cout) tma_store_3d(&p.mapY[img], stg + b * TC_A_BYTES, n0 + b * 64, ox0, oy0);
            tma_store_commit_and_wait_read();
        }
        return;
    }
    if (p.tma_epi) {
        // ---- bulk epilogue: residual tile in by TMA, result tile out by TMA; the pipeline stages are idle now and
        // serve as staging: BN/32 boxes of (32 channels x tw x th) = 128 rows x 128 B, 128-byte swizzled ----
        uint8_t* stg = smem;
        const bool has_res = p.residual != nullptr;
        if (has_res) {
            if (warp == 2 && lane == 0) {
                mbar_expect_tx(res_full, (BN / 32) * TC_A_BYTES);
#pragma unroll
                for (int c = 0; c < BN / 32; ++c) tma_load_3d(stg + c * TC_A_BYTES, &p.mapR[img], res_full, n0 + c * 32, ox0, oy0);
            }
            mbar_wait(res_full, 0);
        }
#pragma unroll 1
        for (int c = 0; c < BN / 32; ++c) {
            uint32_t v[32];
            tmem_ld32(trow + c * 32, v);
            const int n = n0 + c * 32;
            uint8_t* rowp = stg + c * TC_A_BYTES + m * 128;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float4* sp = reinterpret_cast<float4*>(rowp + ((j ^ (m & 7)) << 4));
                float4 o = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
                if (p.bias && n + 4 * j < p.Cout) { float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + n + 4 * j)); o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w; }
                if (has_res) { float4 rr = *sp; o.x += rr.x; o.y += rr.y; o.z += rr.z; o.w += rr.w; }
                if (p.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                if (p.round_out) { o.x = round_tf32(o.x); o.y = round_tf32(o.y); o.z = round_tf32(o.z); o.w = round_tf32(o.w); }
                *sp = o;
            }
        }
        fence_proxy_async();                        // generic-proxy smem writes -> visible to the TMA (async proxy)
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (warp == 2 && lane == 0) {
#pragma unroll
            for (int c = 0; c < BN / 32; ++c)
                if (n0 + c * 32 < p.Cout) tma_store_3d(&p.mapY[img], stg + c * TC_A_BYTES, n0 + c * 32, ox0, oy0);
            tma_store_commit_and_wait_read();       // smem must stay valid until the bulk stores have read it
        }
    } else {
        const int py = m / tw, px = m - py * tw;
        const int oy = oy0 + py, ox = ox0 + px;
        const bool valid = (oy < p.Ho[img]) && (ox < p.Wo[img]);
        const long long pix = p.out_pix[img] + (long long)oy * p.Wo[img] + ox;
#pragma unroll 1
        for (int c = 0; c < BN / 32; ++c) {
            uint32_t v[32];
            tmem_ld32(trow + c * 32, v);
            const int n = n0 + c * 32;
            if (valid && n < p.Cout) {
                float* dst = p.y + pix * p.Cout + n;
                const float* res = p.residual ? p.residual + pix * p.Cout + n : nullptr;
                if (n + 32 <= p.Cout && (p.Cout & 3) == 0) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        float4 o = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                        if (p.bias) { float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + n + j)); o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w; }
                        if (res) { float4 rr = __ldg(reinterpret_cast<const float4*>(res + j)); o.x += rr.x; o.y += rr.y; o.z += rr.z; o.w += rr.w; }
                        if (p.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                        if (p.round_out) { o.x = round_tf32(o.x); o.y = round_tf32(o.y); o.z = round_tf32(o.z); o.w = round_tf32(o.w); }
                        *reinterpret_cast<float4*>(dst + j) = o;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (n + j < p.Cout) {
                            float o = __uint_as_float(v[j]);
                            if (p.bias) o += __ldg(p.bias + n + j);
                            if (res) o += __ldg(res + j);
                            if (p.relu) o = fmaxf(o, 0.f);
                            if (p.round_out) o = round_tf32(o);
                            dst[j] = o;
                        }
                }
            }
        }
    }
}


template <int BN, int MODE, bool DEEP = false>
struct TcCfg {
    static constexpr int NSPLIT = (MODE == MODE_CORR) ? 2 : 1;
    static constexpr int B_BYTES = BN * 128;
    static constexpr int STAGE_BYTES = NSPLIT * (TC_A_BYTES + B_BYTES);
    // three CTAs per SM (so one tile's epilogue / prologue overlaps the others' main loops): <= 73 KB of stages each;
    // the 3xTF32 correlation needs 64 KB per stage and keeps one CTA per SM with 3 stages
    // measured in sequence (profiles/): co-resident CTAs matter more than ring depth (one tile's prologue /
    // epilogue hides behind the others' main loops, and the loop itself is L2->SM bandwidth bound).  K-deep layers
    // (3x3, wide 1x1): 2 CTAs x 3 stages; short-K layers (1x1 expansions with residual): 3 CTAs x 2 stages
    static constexpr int BUDGET = (MODE == MODE_CORR) ? 200 * 1024 : (DEEP ? 100 * 1024 : 73 * 1024);
    static constexpr int STAGES = BUDGET / STAGE_BYTES > 8 ? 8 : BUDGET / STAGE_BYTES;
    static constexpr int CTAS_PER_SM = (MODE == MODE_CORR) ? 1 : (DEEP ? 2 : 3);
    static constexpr int TMEM_COLS = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

template <int BN, int MODE, bool DEEP, bool F16 = false>
__global__ void __launch_bounds__(TC_THREADS, TcCfg<BN, MODE, DEEP>::CTAS_PER_SM)
tc_kernel(const __grid_constant__ TcParams p) {
    using Cfg = TcCfg<BN, MODE, DEEP>;
    constexpr int STAGES = Cfg::STAGES, NSPLIT = Cfg::NSPLIT;
    constexpr int BK = tc_bk<F16>();              // channels per 128-byte K block
    constexpr int TMEM_COLS = Cfg::TMEM_COLS;
    static_assert(!(F16 && MODE == MODE_CORR), "the fp16-split correlation is tc_corr_pipe_kernel");
    // fp16 convolutions: ring depth per layer (<= STAGES) and, for layers with a residual, a dedicated staging area
    // behind the ring that the producer fills at CTA start (more bytes in flight per SM, one DRAM latency less per CTA)
    const int NST = (F16 && MODE == MODE_CONV) ? p.stages : STAGES;
    const bool res_pf = F16 && MODE == MODE_CONV && p.res_pf;
    constexpr int RES_BYTES = (BN / 64) * TC_A_BYTES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);      // pointer arithmetic keeps the shared address space (LDS / STS, not generic LD / ST)
    uint8_t* res_stg = smem + NST * Cfg::STAGE_BYTES;
    uint64_t* full = reinterpret_cast<uint64_t*>(res_stg + (res_pf ? RES_BYTES : 0));
    uint64_t* empty = full + STAGES;
    uint64_t* tmem_full = empty + STAGES;
    uint64_t* res_full = tmem_full + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // ---- tile decode ----
    // conv: blockIdx.x = pixel tile, blockIdx.y = channel tile.  corr: swapped, so that the CTAs sharing one 128-row
    // slab of featA (1 MB of hi+lo) are co-resident and the slab is fetched from DRAM once
    const bool nfast = (MODE == MODE_CORR) || p.raster_n;
    const int mtile = nfast ? blockIdx.y : blockIdx.x;
    const int ntile = nfast ? blockIdx.x : blockIdx.y;
    int img = 0;
#pragma unroll
    for (int j = 1; j < RF_MAX_IMGS; ++j) img += (j < p.nimg && mtile >= p.tile_start[j]) ? 1 : 0;
    const int tloc = mtile - p.tile_start[img];
    const int tw = p.tw[img], th = 128 / tw;
    const int tyi = tloc / p.tiles_x[img], txi = tloc - tyi * p.tiles_x[img];
    const int ox0 = txi * tw, oy0 = tyi * th;
    const int n0 = ntile * BN;
    const int kc = p.Cin / BK;                    // K blocks (32 fp32 / 64 fp16 channels) per tap
    const int KI = p.R * p.S * kc;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NST; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(tmem_full, 1);
        mbar_init(res_full, 1);
        fence_barrier_init();
    }
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.mapA[img]);
        tma_prefetch_desc(&p.mapB);
        if (NSPLIT == 2) { tma_prefetch_desc(&p.mapAlo); tma_prefetch_desc(&p.mapBlo); }
    }
    if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // =============================== TMA producer ===============================
        if (lane == 0) {
            for (int it = 0; it < KI; ++it) {
                const int st = it % NST, ph = (it / NST) & 1;
                mbar_wait(&empty[st], ph ^ 1);
                uint8_t* sbase = smem + st * Cfg::STAGE_BYTES;
                mbar_expect_tx(&full[st], Cfg::STAGE_BYTES);
                const int tap = it / kc, cc = it - tap * kc;
                const int r = tap / p.S, s = tap - r * p.S;
                const int c0 = cc * BK, x = ox0 * p.stride + s - p.pad, y = oy0 * p.stride + r - p.pad;
                const int kcol = tap * p.Cin + c0;
                tma_load_3d(sbase, &p.mapA[img], &full[st], c0, x, y);
                tma_load_2d(sbase + NSPLIT * TC_A_BYTES, &p.mapB, &full[st], kcol, n0);
                if (NSPLIT == 2) {
                    tma_load_3d(sbase + TC_A_BYTES, &p.mapAlo, &full[st], c0, x, y);
                    tma_load_2d(sbase + 2 * TC_A_BYTES + Cfg::B_BYTES, &p.mapBlo, &full[st], kcol, n0);
                }
                if (F16 && it == 0 && res_pf) {       // right behind the first operand tiles: the residual tile
                    mbar_expect_tx(res_full, RES_BYTES);
#pragma unroll
                    for (int b = 0; b < BN / 64; ++b) tma_load_3d(res_stg + b * TC_A_BYTES, &p.mapR[img], res_full, n0 + b * 64, ox0, oy0);
                }
            }
        }
    } else if (warp == 1) {
        // =============================== MMA issuer ===============================
        {   // whole warp, warp-uniform control flow; umma_* elect the issuing lane
            constexpr uint32_t idesc = make_idesc<F16>(BN);
            for (int it = 0; it < KI; ++it) {
                const int st = it % NST, ph = (it / NST) & 1;
                mbar_wait(&full[st], ph);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + st * Cfg::STAGE_BYTES);
                const uint32_t sb = sa + NSPLIT * TC_A_BYTES;
                const uint64_t da = make_desc_sw128(sa), db = make_desc_sw128(sb);
                if (NSPLIT == 2) {
                    umma_3xtf32_x4(tmem_base, da, make_desc_sw128(sa + TC_A_BYTES), db, make_desc_sw128(sb + Cfg::B_BYTES), idesc, it != 0 ? 1u : 0u);
                } else {
                    umma_x4<F16>(tmem_base, da, db, idesc, it != 0 ? 1u : 0u);      // 4 x (UMMA_K = 8 tf32 / 16 fp16 = 32 bytes)
                }
                umma_commit(&empty[st]);            // stage free once these MMAs have read it
            }
            umma_commit(tmem_full);                 // accumulator complete
        }
    } else {
        // =============================== epilogue (warps 2..5) ===============================
        const int q = warp & 3;                     // TMEM lane quarter this warp may access
        const int m = q * 32 + lane;                // accumulator row = pixel inside the tile
        mbar_wait(tmem_full, 0);
        tc_fence_after();
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
        if (MODE == MODE_CONV) {
            conv_epilogue<BN, F16>(p, img, ox0, oy0, tw, n0, m, trow, res_pf ? res_stg : smem, res_full, warp, lane, res_pf);
        } else {
            // utils/outil.py:36-37: row arg-max (thread-local over this tile's columns), column arg-max via an
            // smem transpose of the score tile (the pipeline stages are idle by now)
            float* sS = reinterpret_cast<float*>(smem);
            constexpr int LD = BN + 1;
            const int row = ox0 + m;                // corr "image" is 1 x NA: tile = 128 consecutive rows of featA
            const bool rvalid = row < p.NA;
            unsigned long long best = 0ull;
#pragma unroll 1
            for (int c = 0; c < BN / 32; ++c) {
                uint32_t v[32];
                tmem_ld32(trow + c * 32, v);
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int col = n0 + c * 32 + j;
                    const float s = __uint_as_float(v[j]);
                    sS[m * LD + c * 32 + j] = s;
                    if (col < p.NB) {
                        unsigned long long k = pack_key(s, (uint32_t)col);
                        best = k > best ? k : best;
                    }
                }
            }
            if (rvalid && best != 0ull) atomicMax(p.rowbest + row, best);
            asm volatile("bar.sync 1, 128;" ::: "memory");
            const int t = (warp - 2) * 32 + lane;
            const int rmax = min(128, p.NA - ox0);
            for (int cidx = t; cidx < BN; cidx += 128) {
                const int col = n0 + cidx;
                if (col >= p.NB) continue;
                unsigned long long cb = 0ull;
                for (int rr = 0; rr < rmax; ++rr) {
                    unsigned long long k = pack_key(sS[rr * LD + cidx], (uint32_t)(ox0 + rr));
                    cb = k > cb ? k : cb;
                }
                if (cb != 0ull) atomicMax(p.colbest + col, cb);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}


// ------------------------------------------------------------------------------------------------------------
// 3x3 / stride-1 convolutions with HALO REUSE.  The tap-streaming kernel above fetches the A tile nine times per
// 32-channel chunk (once per tap, shifted by one pixel) and is bound by L2->SM operand bandwidth.  Here the CTA
// owns an 8 x 16 pixel tile, loads its (8+2) x (16+2) halo ONCE per chunk (180 rows x 128 B, one TMA box) and the
// nine taps are nine UMMA descriptors into the same shared memory: tap (r, s) starts (r*10 + s) rows into the halo
// and its sixteen 8-row core groups are 10 rows (1280 B) apart - the descriptor's stride-byte-offset.  Two rings:
// A (halo chunks) and B (one K-major weight tile per tap).
// ------------------------------------------------------------------------------------------------------------
constexpr int HALO_TW = 8, HALO_TH = 16;
constexpr int HALO_LD = HALO_TW + 2;                                   // halo row pitch in pixels
constexpr int HALO_A_BYTES = HALO_LD * (HALO_TH + 2) * 128;            // 23040
constexpr int HALO_A_SLOT = 23 * 1024;                                 // 1024-byte aligned slot

template <int BN>
struct HaloCfg {
    static constexpr int B_BYTES = BN * 128;
    static constexpr int NA = 2;
    static constexpr int NB = (BN == 128) ? 3 : 4;
    static constexpr int RING_BYTES = NA * HALO_A_SLOT + NB * B_BYTES;
    static constexpr int STG_BYTES = BN * 512;
    static constexpr int DATA_BYTES = RING_BYTES > STG_BYTES ? RING_BYTES : STG_BYTES;
    static constexpr int SMEM_BYTES = DATA_BYTES + 1024 + 256;
    static constexpr int TMEM_COLS = BN <= 64 ? 64 : 128;
};

__device__ __forceinline__ uint64_t make_desc_halo(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)(saddr >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((HALO_LD * 128) >> 4) << 32;                       // 8-row core groups are one halo row pitch apart
    d |= (uint64_t)1 << 46;
    // The start address is NOT 1024-byte aligned and the groups are 1280 B apart.  Measured on B200 (round 1): the
    // 128-byte swizzle of tcgen05.mma is a pure function of the shared-memory address bits (it matches what the TMA
    // wrote for any row phase) and the descriptor's base-offset field must stay 0; setting it to (addr >> 7) & 7, as the
    // PTX text suggests for unaligned starts, double-applies the phase and gives wrong results.
    d |= (uint64_t)2 << 61;
    return d;
}

// OUT32 (with F16): fp16 operands, fp32 output through the fp32 epilogue (the layer feeding a TF32 / fp32 consumer)
template <int BN, bool F16 = false, bool OUT32 = false>
__global__ void __launch_bounds__(TC_THREADS, 2)
tc_halo_kernel(const __grid_constant__ TcParams p) {
    using Cfg = HaloCfg<BN>;
    constexpr int NA = Cfg::NA, NB = Cfg::NB;
    constexpr int BK = tc_bk<F16>();
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);      // pointer arithmetic keeps the shared address space (LDS / STS, not generic LD / ST)
    uint8_t* sA = smem;
    uint8_t* sB = smem + NA * HALO_A_SLOT;
    uint64_t* fullA = reinterpret_cast<uint64_t*>(smem + Cfg::DATA_BYTES);
    uint64_t* emptyA = fullA + NA;
    uint64_t* fullB = emptyA + NA;
    uint64_t* emptyB = fullB + NB;
    uint64_t* tmem_full = emptyB + NB;
    uint64_t* res_full = tmem_full + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_full + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    int img = 0;
#pragma unroll
    for (int j = 1; j < RF_MAX_IMGS; ++j) img += (j < p.nimg && (int)blockIdx.x >= p.tile_start[j]) ? 1 : 0;
    const int tloc = blockIdx.x - p.tile_start[img];
    const int tyi = tloc / p.tiles_x[img], txi = tloc - tyi * p.tiles_x[img];
    const int ox0 = txi * HALO_TW, oy0 = tyi * HALO_TH;
    const int n0 = blockIdx.y * BN;
    const int kc = p.Cin / BK;

    if (threadIdx.x == 0) {
        for (int i = 0; i < NA; ++i) { mbar_init(&fullA[i], 1); mbar_init(&emptyA[i], 1); }
        for (int i = 0; i < NB; ++i) { mbar_init(&fullB[i], 1); mbar_init(&emptyB[i], 1); }
        mbar_init(tmem_full, 1);
        mbar_init(res_full, 1);
        fence_barrier_init();
    }
    if (warp == 0 && lane == 0) { tma_prefetch_desc(&p.mapA[img]); tma_prefetch_desc(&p.mapB); }
    if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int ib = 0;
            for (int cc = 0; cc < kc; ++cc) {
                const int sa = cc % NA, pha = (cc / NA) & 1;
                mbar_wait(&emptyA[sa], pha ^ 1);
                mbar_expect_tx(&fullA[sa], HALO_A_BYTES);
                tma_load_3d(sA + sa * HALO_A_SLOT, &p.mapA[img], &fullA[sa], cc * BK, ox0 - 1, oy0 - 1);
                for (int tap = 0; tap < 9; ++tap, ++ib) {
                    const int sb = ib % NB, phb = (ib / NB) & 1;
                    mbar_wait(&emptyB[sb], phb ^ 1);
                    mbar_expect_tx(&fullB[sb], Cfg::B_BYTES);
                    tma_load_2d(sB + sb * Cfg::B_BYTES, &p.mapB, &fullB[sb], tap * p.Cin + cc * BK, n0);
                }
            }
        }
    } else if (warp == 1) {
        {   // whole warp, warp-uniform control flow; umma_* elect the issuing lane
            constexpr uint32_t idesc = make_idesc<F16>(BN);
            int ib = 0;
            for (int cc = 0; cc < kc; ++cc) {
                const int sa = cc % NA, pha = (cc / NA) & 1;
                mbar_wait(&fullA[sa], pha);
                tc_fence_after();
                const uint32_t abase = smem_u32(sA + sa * HALO_A_SLOT);
                for (int tap = 0; tap < 9; ++tap, ++ib) {
                    const int sb = ib % NB, phb = (ib / NB) & 1;
                    mbar_wait(&fullB[sb], phb);
                    tc_fence_after();
                    const int r = tap / 3, sx = tap - r * 3;
                    const uint32_t aaddr = abase + (uint32_t)((r * HALO_LD + sx) * 128);
                    const uint64_t db = make_desc_sw128(smem_u32(sB + sb * Cfg::B_BYTES));
                    umma_x4<F16>(tmem_base, make_desc_halo(aaddr), db, idesc, (cc | tap) != 0 ? 1u : 0u);
                    umma_commit(&emptyB[sb]);
                }
                umma_commit(&emptyA[sa]);
            }
            umma_commit(tmem_full);
        }
    } else {
        const int q = warp & 3;
        const int m = q * 32 + lane;
        mbar_wait(tmem_full, 0);
        tc_fence_after();
        conv_epilogue<BN, F16 && !OUT32>(p, img, ox0, oy0, HALO_TW, n0, m, tmem_base + ((uint32_t)(q * 32) << 16), smem, res_full, warp, lane);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}


// Tile decode of the persistent convolution kernels (tc_resb_kernel, tc_pipe_kernel): tile t of tiles_m pixel tiles x
// (Cout / BN) channel tiles.
struct TileCoord { int img, ox0, oy0, tw, n0; };

template <bool HALO>
__device__ __forceinline__ TileCoord decode_tile(const TcParams& p, int t, int tiles_m, int BN) {
    TileCoord c;
    int nt = t / tiles_m, mt = t - nt * tiles_m;            // pixel tiles fastest: co-running CTAs share the weight tile
    if (p.raster_n) {                                       // channel tiles fastest: co-running CTAs share the pixel tile
        const int tiles_n = (p.Cout + BN - 1) / BN;
        mt = t / tiles_n;
        nt = t - mt * tiles_n;
    }
    int img = 0;
#pragma unroll
    for (int j = 1; j < RF_MAX_IMGS; ++j) img += (j < p.nimg && mt >= p.tile_start[j]) ? 1 : 0;
    const int tloc = mt - p.tile_start[img];
    c.img = img;
    c.tw = HALO ? HALO_TW : p.tw[img];
    const int th = 128 / c.tw;
    const int tyi = tloc / p.tiles_x[img], txi = tloc - tyi * p.tiles_x[img];
    c.ox0 = txi * c.tw;
    c.oy0 = tyi * th;
    c.n0 = nt * BN;
    return c;
}

// ------------------------------------------------------------------------------------------------------------
// 3x3 / stride-1 / 64 -> 64 channel convolutions (ResNet-50 layer1 conv2, FeatureExtractor layer1): K is only two
// 32-channel chunks, so a tile is ~1.2 us of MMA work and one-tile CTAs live mostly in launch / TMA / epilogue
// latency.  All 18 weight tiles (9 taps x 2 chunks x 8 KB = 144 KB) fit in shared memory: this persistent kernel loads
// them ONCE per CTA, then streams halo tiles (2 x 23 KB) through a two-slot ring while two TMEM accumulators let the
// epilogue of tile i overlap the MMAs of tile i+1.  Per tile only the 46 KB halo crosses L2->SM.
// ------------------------------------------------------------------------------------------------------------
// fp16 (engine 2): 64 channels are ONE 128-byte K block, so the weights are 72 KB and the halo ring gets four slots
template <bool F16>
struct ResBCfg {
    static constexpr int BN = 64, KC = F16 ? 1 : 2, NTAP = 9, NA = F16 ? 4 : 2;
    static constexpr int B_TILE = BN * 128;                                 // 8 KB
    static constexpr int B_BYTES = KC * NTAP * B_TILE;                      // 144 KB (72 KB fp16)
    static constexpr int OFF_A = B_BYTES;
    static constexpr int OFF_STG = OFF_A + NA * HALO_A_SLOT;
    static constexpr int STG = F16 ? BN * 256 : BN * 512;                   // 32 KB (16 KB fp16)
    static constexpr int DATA_BYTES = OFF_STG + STG;
    static constexpr int SMEM_BYTES = DATA_BYTES + 1024 + 256;
    static constexpr int TMEM_COLS = 128;                                   // two 64-column accumulators
};

template <bool F16 = false>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_resb_kernel(const __grid_constant__ TcParams p, int tiles_m) {
    using Cfg = ResBCfg<F16>;
    constexpr int BN = Cfg::BN, NA = Cfg::NA;
    constexpr int BK = tc_bk<F16>();
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);      // pointer arithmetic keeps the shared address space (LDS / STS, not generic LD / ST)
    uint8_t* sB = smem;
    uint8_t* sA = smem + Cfg::OFF_A;
    uint8_t* sStg = smem + Cfg::OFF_STG;
    uint64_t* fullA = reinterpret_cast<uint64_t*>(smem + Cfg::DATA_BYTES);
    uint64_t* emptyA = fullA + NA;
    uint64_t* fullB = emptyA + NA;              // [1]
    uint64_t* tmem_full = fullB + 1;            // [2]
    uint64_t* tmem_empty = tmem_full + 2;       // [2]
    uint64_t* res_full = tmem_empty + 2;        // [1]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_full + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total = tiles_m;                  // Cout = 64: a single channel tile

    if (threadIdx.x == 0) {
        for (int i = 0; i < NA; ++i) { mbar_init(&fullA[i], 1); mbar_init(&emptyA[i], 1); }
        mbar_init(fullB, 1);
        for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 128); }
        mbar_init(res_full, 1);
        fence_barrier_init();
    }
    if (warp == 0 && lane == 0) { tma_prefetch_desc(&p.mapA[0]); tma_prefetch_desc(&p.mapB); tma_prefetch_desc(&p.mapY[0]); }
    if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            // the whole weight set, once: tile (cc, tap) at sB + (cc * 9 + tap) * 8 KB
            mbar_expect_tx(fullB, Cfg::B_BYTES);
            for (int cc = 0; cc < Cfg::KC; ++cc)
                for (int tap = 0; tap < Cfg::NTAP; ++tap)
                    tma_load_2d(sB + (cc * Cfg::NTAP + tap) * Cfg::B_TILE, &p.mapB, fullB, tap * p.Cin + cc * BK, 0);
            uint32_t ia = 0;
            for (int t = blockIdx.x; t < total; t += gridDim.x) {
                const TileCoord c = decode_tile<true>(p, t, tiles_m, BN);
                for (int cc = 0; cc < Cfg::KC; ++cc, ++ia) {
                    const int sa = ia % NA;
                    mbar_wait(&emptyA[sa], ((ia / NA) & 1) ^ 1);
                    mbar_expect_tx(&fullA[sa], HALO_A_BYTES);
                    tma_load_3d(sA + sa * HALO_A_SLOT, &p.mapA[c.img], &fullA[sa], cc * BK, c.ox0 - 1, c.oy0 - 1);
                }
            }
        }
    } else if (warp == 1) {
        {   // whole warp, warp-uniform control flow; umma_* elect the issuing lane
            constexpr uint32_t idesc = make_idesc<F16>(BN);
            mbar_wait(fullB, 0);
            tc_fence_after();
            uint32_t ia = 0, ti = 0;
            for (int t = blockIdx.x; t < total; t += gridDim.x, ++ti) {
                const uint32_t buf = ti & 1;
                mbar_wait(&tmem_empty[buf], ((ti >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t tacc = tmem_base + buf * BN;
                for (int cc = 0; cc < Cfg::KC; ++cc, ++ia) {
                    const int sa = ia % NA;
                    mbar_wait(&fullA[sa], (ia / NA) & 1);
                    tc_fence_after();
                    const uint32_t abase = smem_u32(sA + sa * HALO_A_SLOT);
#pragma unroll
                    for (int tap = 0; tap < Cfg::NTAP; ++tap) {
                        const int r = tap / 3, sx = tap - r * 3;
                        const uint32_t aaddr = abase + (uint32_t)((r * HALO_LD + sx) * 128);
                        const uint64_t db = make_desc_sw128(smem_u32(sB + (cc * Cfg::NTAP + tap) * Cfg::B_TILE));
                        umma_x4<F16>(tacc, make_desc_halo(aaddr), db, idesc, (cc | tap) != 0 ? 1u : 0u);
                    }
                    umma_commit(&emptyA[sa]);
                }
                umma_commit(&tmem_full[buf]);
            }
        }
    } else {
        const int q = warp & 3;
        const int m = q * 32 + lane;
        const bool leader = (warp == 2 && lane == 0);
        const bool has_res = p.residual != nullptr;
        constexpr int NBOX = Cfg::STG / TC_A_BYTES;                 // staging boxes of 128 bytes per pixel: 2 (fp32) / 1 (fp16)
        uint32_t ti = 0;
        for (int t = blockIdx.x; t < total; t += gridDim.x, ++ti) {
            const uint32_t buf = ti & 1;
            const TileCoord c = decode_tile<true>(p, t, tiles_m, BN);
            if (leader) {
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");          // staging buffer has been read out
                if (has_res) {
                    mbar_expect_tx(res_full, NBOX * TC_A_BYTES);
#pragma unroll
                    for (int cb = 0; cb < NBOX; ++cb) tma_load_3d(sStg + cb * TC_A_BYTES, &p.mapR[c.img], res_full, cb * BK, c.ox0, c.oy0);
                }
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            mbar_wait(&tmem_full[buf], (ti >> 1) & 1);
            tc_fence_after();
            if (has_res) mbar_wait(res_full, ti & 1);
            const uint32_t trow = tmem_base + buf * BN + ((uint32_t)(q * 32) << 16);
            if constexpr (F16) epi_rows_f16<BN>(p.bias, p.Cout, p.relu, has_res, 0, m, trow, sStg);
#pragma unroll 1
            for (int cb = 0; cb < (F16 ? 0 : BN / 32); ++cb) {
                uint32_t v[32];
                tmem_ld32(trow + cb * 32, v);
                const int n = cb * 32;
                uint8_t* rowp = sStg + cb * TC_A_BYTES + m * 128;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float4* sp = reinterpret_cast<float4*>(rowp + ((j ^ (m & 7)) << 4));
                    float4 o = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
                    if (p.bias) { float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + n + 4 * j)); o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w; }
                    if (has_res) { float4 rr = *sp; o.x += rr.x; o.y += rr.y; o.z += rr.z; o.w += rr.w; }
                    if (p.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                    if (p.round_out) { o.x = round_tf32(o.x); o.y = round_tf32(o.y); o.z = round_tf32(o.z); o.w = round_tf32(o.w); }
                    *sp = o;
                }
            }
            tc_fence_before();
            mbar_arrive(&tmem_empty[buf]);
            fence_proxy_async();
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (leader) {
#pragma unroll
                for (int cb = 0; cb < NBOX; ++cb) tma_store_3d(&p.mapY[c.img], sStg + cb * TC_A_BYTES, cb * BK, c.ox0, c.oy0);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
        if (leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------------------
// PIPELINED persistent fp16 convolution (tap streaming: 1x1 of any stride, 3x3 / stride 2).  ncu on the one-tile-per-CTA
// kernel (profiles/r1_f16_layers_ncu.json) shows every such layer latency bound - DRAM <= 55 %, L2 <= 32 %, tensor
// pipe <= 28 %, a CTA lives ~10 us for ~1 us of work: operand load -> MMA -> residual load -> epilogue -> store drain
// are serial inside a CTA and at most four CTAs fit an SM.  Here one CTA per SM software-pipelines tiles:
//   warp 0     : TMA producer - residual tile of tile i (into staging buffer i & 1, as soon as the store of tile i-2
//                has read it out) and the K blocks of tile i into an NS-deep ring; runs ahead across tiles;
//   warp 1     : MMA issuer - accumulator i & 1 of two, so tile i+1 multiplies while tile i drains;
//   warps 2-5  : epilogue group 0 (even tiles), warps 6-9: epilogue group 1 (odd tiles) - TMEM -> + bias, + residual,
//                ReLU -> fp16 swizzled staging -> TMA store; two groups so that two epilogues overlap.
// ------------------------------------------------------------------------------------------------------------
template <int BN>
struct PipeCfg {
    static constexpr int B_BYTES = BN * 128;
    static constexpr int STAGE_BYTES = TC_A_BYTES + B_BYTES;
    static constexpr int NS = BN == 128 ? 4 : 6;
    static constexpr int STG = (BN / 64) * TC_A_BYTES;                      // fp16 staging: BN / 64 boxes of 16 KB
    static constexpr int OFF_STG = NS * STAGE_BYTES;
    static constexpr int DATA_BYTES = OFF_STG + 2 * STG;
    static constexpr int SMEM_BYTES = DATA_BYTES + 1024 + 512;
    static constexpr int TMEM_COLS = 2 * BN;
    static constexpr int THREADS = 320;
};

template <int BN>
__global__ void __launch_bounds__(PipeCfg<BN>::THREADS, 1)
tc_pipe_kernel(const __grid_constant__ TcParams p, int tiles_m, int tiles_n) {
    using Cfg = PipeCfg<BN>;
    constexpr int NS = Cfg::NS, NBOX = BN / 64, BK = TC_BK_F16;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);      // pointer arithmetic keeps the shared address space (LDS / STS, not generic LD / ST)
    uint8_t* sStg = smem + Cfg::OFF_STG;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + Cfg::DATA_BYTES);
    uint64_t* empty = full + NS;
    uint64_t* tmem_full = empty + NS;           // [2]
    uint64_t* tmem_empty = tmem_full + 2;       // [2] 128 arrivals
    uint64_t* res_full = tmem_empty + 2;        // [2]
    uint64_t* stg_free = res_full + 2;          // [2] the group's leader: the TMA store has read the staging buffer
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(stg_free + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total = tiles_m * tiles_n;
    const int kc = p.Cin / BK;
    const int KI = p.R * p.S * kc;
    const bool has_res = p.residual != nullptr;

    if (threadIdx.x == 0) {
        for (int i = 0; i < NS; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 128); mbar_init(&res_full[i], 1); mbar_init(&stg_free[i], 1); }
        fence_barrier_init();
    }
    if (warp == 0 && lane == 0) { tma_prefetch_desc(&p.mapA[0]); tma_prefetch_desc(&p.mapB); tma_prefetch_desc(&p.mapY[0]); }
    if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // =============================== TMA producer ===============================
        if (lane == 0) {
            uint32_t cnt = 0, ti = 0;
            for (int t = blockIdx.x; t < total; t += gridDim.x, ++ti) {
                const TileCoord c = decode_tile<false>(p, t, tiles_m, BN);
                if (has_res) {
                    const uint32_t g = ti & 1;
                    mbar_wait(&stg_free[g], ((ti >> 1) & 1) ^ 1);        // tile ti-2's store has read this buffer (passes at once for ti < 2)
                    mbar_expect_tx(&res_full[g], Cfg::STG);
#pragma unroll
                    for (int b = 0; b < NBOX; ++b)
                        tma_load_3d(sStg + g * Cfg::STG + b * TC_A_BYTES, &p.mapR[c.img], &res_full[g], c.n0 + b * 64, c.ox0, c.oy0);
                }
                for (int it = 0; it < KI; ++it, ++cnt) {
                    const int st = cnt % NS;
                    mbar_wait(&empty[st], ((cnt / NS) & 1) ^ 1);
                    uint8_t* sbase = smem + st * Cfg::STAGE_BYTES;
                    mbar_expect_tx(&full[st], Cfg::STAGE_BYTES);
                    const int tap = it / kc, cc = it - tap * kc;
                    const int r = tap / p.S, sx = tap - r * p.S;
                    tma_load_3d(sbase, &p.mapA[c.img], &full[st], cc * BK, c.ox0 * p.stride + sx - p.pad, c.oy0 * p.stride + r - p.pad);
                    tma_load_2d(sbase + TC_A_BYTES, &p.mapB, &full[st], tap * p.Cin + cc * BK, c.n0);
                }
            }
        }
    } else if (warp == 1) {
        // =============================== MMA issuer (whole warp, warp-uniform) ===============================
        constexpr uint32_t idesc = make_idesc_f16(BN);
        uint32_t cnt = 0, ti = 0;
        for (int t = blockIdx.x; t < total; t += gridDim.x, ++ti) {
            const uint32_t buf = ti & 1;
            mbar_wait(&tmem_empty[buf], ((ti >> 1) & 1) ^ 1);               // the epilogue has drained this accumulator
            tc_fence_after();
            const uint32_t tacc = tmem_base + buf * BN;
            for (int it = 0; it < KI; ++it, ++cnt) {
                const int st = cnt % NS;
                mbar_wait(&full[st], (cnt / NS) & 1);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + st * Cfg::STAGE_BYTES);
                umma_f16_x4(tacc, make_desc_sw128(sa), make_desc_sw128(sa + TC_A_BYTES), idesc, it != 0 ? 1u : 0u);
                umma_commit(&empty[st]);
            }
            umma_commit(&tmem_full[buf]);
        }
    } else {
        // =============================== epilogue groups ===============================
        const uint32_t g = (uint32_t)(warp - 2) >> 2;                       // 0: warps 2-5, 1: warps 6-9
        const int q = warp & 3;                                             // TMEM lane quarter this warp may access
        const int m = q * 32 + lane;
        const bool leader = ((warp - 2) & 3) == 0 && lane == 0;
        uint8_t* stg = sStg + g * Cfg::STG;
        uint32_t k = 0;                                                     // this group's tile counter
        for (int t = blockIdx.x + (int)g * (int)gridDim.x; t < total; t += 2 * gridDim.x, ++k) {
            const TileCoord c = decode_tile<false>(p, t, tiles_m, BN);
            // the leader comes here only after the previous store has read the staging buffer
            if (g == 0) asm volatile("bar.sync 1, 128;" ::: "memory"); else asm volatile("bar.sync 2, 128;" ::: "memory");
            mbar_wait(&tmem_full[g], k & 1);
            tc_fence_after();
            if (has_res) mbar_wait(&res_full[g], k & 1);
            const uint32_t trow = tmem_base + g * BN + ((uint32_t)(q * 32) << 16);
            epi_rows_f16<BN>(p.bias, p.Cout, p.relu, has_res, c.n0, m, trow, stg);
            tc_fence_before();
            mbar_arrive(&tmem_empty[g]);                                    // accumulator drained (128 arrivals)
            fence_proxy_async();
            if (g == 0) asm volatile("bar.sync 1, 128;" ::: "memory"); else asm volatile("bar.sync 2, 128;" ::: "memory");
            if (leader) {
#pragma unroll
                for (int b = 0; b < NBOX; ++b)
                    if (c.n0 + b * 64 < p.Cout) tma_store_3d(&p.mapY[c.img], stg + b * TC_A_BYTES, c.n0 + b * 64, c.ox0, c.oy0);
                tma_store_commit_and_wait_read();
                if (has_res) mbar_arrive(&stg_free[g]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------------------
// PERSISTENT correlation + mutual-NN kernel (utils/outil.py:34-37, precision 2 = fp16 split).  ncu on the former
// one-tile-per-CTA kernel (profiles/r1_corr_f16_ncu.json): 17.8 us per 128 x 128 score tile for 6.3 us of MMAs - one
// CTA per SM (192 KB of stages), so TMEM allocation, the first TMA round trip and the whole arg-max epilogue are
// serial with the K loop.  Here one CTA per SM walks its tiles (N-tiles fastest: the CTAs sharing a featA slab run
// together) with the three roles decoupled:
//   warp 0    : TMA producer, 3-stage ring of (A hi, A lo, B hi, B lo) K blocks, runs ahead into the next tile;
//   warp 1    : MMA issuer, TWO accumulator pairs (hi*hi | cross terms) x 128 columns = all 512 TMEM columns: tile
//               i+1 multiplies while tile i drains;
//   warps 2-5 : epilogue.  Row arg-max thread-local straight from TMEM; column arg-max 32 columns at a time through
//               a 128 x 33 float transposition buffer of its own (the stages are busy), four row quarters combined
//               through 1 KB of keys, one atomicMax per column and per row of the tile as before.
// Per score: hi*hi into the main accumulator, lo*hi + hi*lo (at 2^11 scale) into the cross one, combined with one fma;
// ties go to the smallest index.
// ------------------------------------------------------------------------------------------------------------
struct CorrPipeCfg {
    static constexpr int BN = 128;
    static constexpr int B_BYTES = BN * 128;
    static constexpr int STAGE_BYTES = 2 * (TC_A_BYTES + B_BYTES);            // 64 KB
    static constexpr int NS = 3;
    static constexpr int LD = 33;                                             // transposition pitch: conflict-free both ways
    static constexpr int OFF_T = NS * STAGE_BYTES;
    static constexpr int T_BYTES = 128 * LD * 4;
    static constexpr int OFF_P = OFF_T + T_BYTES;
    static constexpr int P_BYTES = 4 * 32 * 8;
    static constexpr int DATA_BYTES = OFF_P + P_BYTES;
    static constexpr int SMEM_BYTES = DATA_BYTES + 1024 + 256;
    static constexpr int TMEM_COLS = 512;
};
static_assert(CorrPipeCfg::SMEM_BYTES <= 227 * 1024, "shared memory");
static_assert((CorrPipeCfg::OFF_P % 8) == 0 && (CorrPipeCfg::DATA_BYTES % 8) == 0, "alignment");


__device__ __forceinline__ unsigned long long pack_ord(uint32_t ord, uint32_t idx) {
    return ((unsigned long long)ord << 32) | (unsigned long long)(0xFFFFFFFFu - idx);
}

__global__ void __launch_bounds__(TC_THREADS, 1)
tc_corr_pipe_kernel(const __grid_constant__ TcParams p, int tiles_m, int tiles_n) {
    using Cfg = CorrPipeCfg;
    constexpr int NS = Cfg::NS, BN = Cfg::BN, BK = TC_BK_F16, LD = Cfg::LD;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);      // pointer arithmetic keeps the shared address space (LDS / STS, not generic LD / ST)
    float* sT = reinterpret_cast<float*>(smem + Cfg::OFF_T);
    unsigned long long* sP = reinterpret_cast<unsigned long long*>(smem + Cfg::OFF_P);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + Cfg::DATA_BYTES);
    uint64_t* empty = full + NS;
    uint64_t* tmem_full = empty + NS;           // [2]
    uint64_t* tmem_empty = tmem_full + 2;       // [2] 128 arrivals
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total = tiles_m * tiles_n;
    const int KI = p.Cin / BK;

    if (threadIdx.x == 0) {
        for (int i = 0; i < NS; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 128); }
        fence_barrier_init();
    }
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.mapA[0]); tma_prefetch_desc(&p.mapAlo); tma_prefetch_desc(&p.mapB); tma_prefetch_desc(&p.mapBlo);
    }
    if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // =============================== TMA producer ===============================
        if (lane == 0) {
            uint32_t cnt = 0;
            for (int t = blockIdx.x; t < total; t += gridDim.x) {
                const int mt = t / tiles_n, nt = t - mt * tiles_n;
                const int row0 = mt * 128, n0 = nt * BN;
                for (int it = 0; it < KI; ++it, ++cnt) {
                    const int st = cnt % NS;
                    mbar_wait(&empty[st], ((cnt / NS) & 1) ^ 1);
                    uint8_t* sbase = smem + st * Cfg::STAGE_BYTES;
                    mbar_expect_tx(&full[st], Cfg::STAGE_BYTES);
                    const int c0 = it * BK;
                    tma_load_3d(sbase, &p.mapA[0], &full[st], c0, row0, 0);
                    tma_load_2d(sbase + 2 * TC_A_BYTES, &p.mapB, &full[st], c0, n0);
                    tma_load_3d(sbase + TC_A_BYTES, &p.mapAlo, &full[st], c0, row0, 0);
                    tma_load_2d(sbase + 2 * TC_A_BYTES + Cfg::B_BYTES, &p.mapBlo, &full[st], c0, n0);
                }
            }
        }
    } else if (warp == 1) {
        // =============================== MMA issuer (whole warp, warp-uniform) ===============================
        constexpr uint32_t idesc = make_idesc_f16(BN);
        uint32_t cnt = 0, ti = 0;
        for (int t = blockIdx.x; t < total; t += gridDim.x, ++ti) {
            const uint32_t buf = ti & 1;
            mbar_wait(&tmem_empty[buf], ((ti >> 1) & 1) ^ 1);               // the epilogue has drained this accumulator pair
            tc_fence_after();
            const uint32_t td = tmem_base + buf * (2 * BN);
            for (int it = 0; it < KI; ++it, ++cnt) {
                const int st = cnt % NS;
                mbar_wait(&full[st], (cnt / NS) & 1);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + st * Cfg::STAGE_BYTES);
                const uint32_t sb = sa + 2 * TC_A_BYTES;
                // [B hi | B lo] are adjacent in the stage, [main | cross] in TMEM: one N = 256 instruction + A lo x B hi
                umma_f16split2_x4(td, BN, make_desc_sw128(sa), make_desc_sw128(sa + TC_A_BYTES), make_desc_sw128(sb),
                                  make_idesc_f16(2 * BN), idesc, it != 0 ? 1u : 0u);
                umma_commit(&empty[st]);
            }
            umma_commit(&tmem_full[buf]);
        }
    } else {
        // =============================== epilogue (warps 2..5) ===============================
        const int q = warp & 3;                     // TMEM lane quarter this warp may access
        const int m = q * 32 + lane;                // accumulator row = featA row inside the tile
        const int tid = (warp - 2) * 32 + lane;     // 0..127 for the column pass
        const int cj = tid & 31, qq = tid >> 5;
        uint32_t ti = 0;
        for (int t = blockIdx.x; t < total; t += gridDim.x, ++ti) {
            const uint32_t buf = ti & 1;
            const int mt = t / tiles_n, nt = t - mt * tiles_n;
            const int row0 = mt * 128, n0 = nt * BN;
            const int rmax = min(128, p.NA - row0);
            mbar_wait(&tmem_full[buf], (ti >> 1) & 1);
            tc_fence_after();
            const uint32_t trow = tmem_base + buf * (2 * BN) + ((uint32_t)(q * 32) << 16);
            uint32_t rbo = 0u, rbi = 0u;            // row best: ordered score (0 = none yet), column
#pragma unroll 1
            for (int c = 0; c < BN / 32; ++c) {
                uint32_t v[32], x[32];
                tmem_ld32x2(trow + c * 32, v, trow + BN + c * 32, x);
                if (c == BN / 32 - 1) {             // last TMEM read of this tile: hand the accumulators back
                    tc_fence_before();
                    mbar_arrive(&tmem_empty[buf]);
                }
                const int colbase = n0 + c * 32;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float s = fmaf(__uint_as_float(x[j]), 0.00048828125f, __uint_as_float(v[j]));     // + cross terms * 2^-11
                    sT[m * LD + j] = s;
                    const uint32_t o = f2ord(s);
                    if (colbase + j < p.NB && o > rbo) { rbo = o; rbi = (uint32_t)(colbase + j); }
                }
                asm volatile("bar.sync 1, 128;" ::: "memory");
                // column arg-max of this 128 x 32 block: thread (qq, cj) scans rows qq*32 .. +31 of column cj
                uint32_t cbo = 0u, cbi = 0u;
#pragma unroll 8
                for (int rr = 0; rr < 32; ++rr) {
                    const int r = qq * 32 + rr;
                    const uint32_t o = f2ord(sT[r * LD + cj]);
                    if (r < rmax && o > cbo) { cbo = o; cbi = (uint32_t)(row0 + r); }
                }
                sP[qq * 32 + cj] = cbo ? pack_ord(cbo, cbi) : 0ull;
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (tid < 32) {
                    unsigned long long k0 = sP[tid], k1 = sP[32 + tid], k2 = sP[64 + tid], k3 = sP[96 + tid];
                    k0 = k1 > k0 ? k1 : k0;
                    k2 = k3 > k2 ? k3 : k2;
                    k0 = k2 > k0 ? k2 : k0;
                    if (colbase + tid < p.NB && k0 != 0ull) atomicMax(p.colbest + colbase + tid, k0);
                }
            }
            if (m < rmax && rbo != 0u) atomicMax(p.rowbest + row0 + m, pack_ord(rbo, rbi));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------------------
// ResNet-50 stem, fused (engine 2): conv 7x7 / stride 2 / pad 3 on the 3-channel fp32 image + folded BN + ReLU ->
// fp16 NHWC, without materialising the im2col matrix (350 MB written and read back per pair at 480x640 x 8 images).
// One CTA = 16 x 8 output pixels x 64 channels:
//   warps 0-3 : stage the 37 x 21 x 3 input window in shared memory (coalesced, zero padded), then each thread builds
//               ITS pixel's 147-long (r, s, c) patch as fp16 directly in the 128-byte-swizzled K-major layout the
//               UMMA descriptors expect (three K blocks of 64; 148..191 are zeros), fence.proxy.async, arrive;
//   warp 4    : TMA-loads the 64 x 192 fp16 weights, issues 12 tcgen05.mma kind::f16 (M 128, N 64, K 16), commits;
//   warps 0-3 : epilogue - TMEM -> + bias, ReLU -> fp16 swizzled staging (the A tile's first block) -> one TMA store.
// ------------------------------------------------------------------------------------------------------------
constexpr int STEM_TW = 16, STEM_TH = 8, STEM_K = 7, STEM_C = 3, STEM_KK = 147, STEM_KB = 3;
constexpr int STEM_IN_W = ((STEM_TW - 1) * 2 + STEM_K) * STEM_C;          // 111 floats per staged input row
constexpr int STEM_IN_H = (STEM_TH - 1) * 2 + STEM_K;                     // 21 rows
constexpr int STEM_IN_LD = 112;
constexpr int STEM_B_TILE = 64 * 128;                                     // 8 KB per K block
constexpr int STEM_OFF_B = STEM_KB * TC_A_BYTES;                          // 48 KB
constexpr int STEM_OFF_IN = STEM_OFF_B + STEM_KB * STEM_B_TILE;           // 72 KB
constexpr int STEM_OFF_BAR = STEM_OFF_IN + STEM_IN_H * STEM_IN_LD * 4;    // + 9408 B
constexpr int STEM_SMEM = STEM_OFF_BAR + 64 + 1024;
constexpr int STEM_THREADS = 160;

struct alignas(64) StemParams {
    CUtensorMap mapB;                     // weights fp16 [64][192], box (64, 64)
    CUtensorMap mapY[RF_MAX_IMGS];        // output fp16 (64, Wo, Ho), box (64, 16, 8)
    int nimg;
    int tile_start[RF_MAX_IMGS + 1];
    int tiles_x[RF_MAX_IMGS];
    int H[RF_MAX_IMGS], W[RF_MAX_IMGS];
    long long in_pix[RF_MAX_IMGS];
    const float* x;
    const float* bias;
};

__global__ void __launch_bounds__(STEM_THREADS, 2)
stem7_f16_kernel(const __grid_constant__ StemParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);      // pointer arithmetic keeps the shared address space (LDS / STS, not generic LD / ST)
    uint8_t* sA = smem;
    uint8_t* sB = smem + STEM_OFF_B;
    float* sIn = reinterpret_cast<float*>(smem + STEM_OFF_IN);
    uint64_t* bar_b = reinterpret_cast<uint64_t*>(smem + STEM_OFF_BAR);
    uint64_t* bar_a = bar_b + 1;
    uint64_t* bar_mma = bar_a + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_mma + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    int img = 0;
#pragma unroll
    for (int j = 1; j < RF_MAX_IMGS; ++j) img += (j < p.nimg && (int)blockIdx.x >= p.tile_start[j]) ? 1 : 0;
    const int tloc = blockIdx.x - p.tile_start[img];
    const int tyi = tloc / p.tiles_x[img], txi = tloc - tyi * p.tiles_x[img];
    const int ox0 = txi * STEM_TW, oy0 = tyi * STEM_TH;

    if (threadIdx.x == 0) {
        mbar_init(bar_b, 1);
        mbar_init(bar_a, 128);
        mbar_init(bar_mma, 1);
        fence_barrier_init();
    }
    if (warp == 4) {
        if (lane == 0) { tma_prefetch_desc(&p.mapB); tma_prefetch_desc(&p.mapY[img]); }
        tmem_alloc(tmem_slot, 64);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 4) {
        if (lane == 0) {
            mbar_expect_tx(bar_b, STEM_KB * STEM_B_TILE);
#pragma unroll
            for (int kb = 0; kb < STEM_KB; ++kb) tma_load_2d(sB + kb * STEM_B_TILE, &p.mapB, bar_b, kb * 64, 0);
        }
        mbar_wait(bar_b, 0);
        mbar_wait(bar_a, 0);
        tc_fence_after();
        constexpr uint32_t idesc = make_idesc_f16(64);
#pragma unroll
        for (int kb = 0; kb < STEM_KB; ++kb)
            umma_f16_x4(tmem_base, make_desc_sw128(smem_u32(sA + kb * TC_A_BYTES)), make_desc_sw128(smem_u32(sB + kb * STEM_B_TILE)), idesc, kb != 0 ? 1u : 0u);
        umma_commit(bar_mma);
    } else {
        const int m = threadIdx.x;                              // 0..127: output pixel inside the tile = accumulator row
        // ---- stage the input window: rows 2*oy0-3 .. +20, float columns (2*ox0-3)*3 .. +110 ----
        const int H = p.H[img], WC = p.W[img] * STEM_C;
        const float* src = p.x + p.in_pix[img] * STEM_C;
        const int iy0 = oy0 * 2 - 3, col0 = (ox0 * 2 - 3) * STEM_C;
        // all loads first (independent, one DRAM latency), then the shared-memory stores
        constexpr int NLD = (STEM_IN_H * STEM_IN_W + 127) / 128;         // 19 per thread
        float stage[NLD];
#pragma unroll
        for (int i = 0; i < NLD; ++i) {
            const int idx = m + i * 128;
            const int r = idx / STEM_IN_W, j = idx - r * STEM_IN_W;
            const int iy = iy0 + r, col = col0 + j;
            stage[i] = (idx < STEM_IN_H * STEM_IN_W && iy >= 0 && iy < H && col >= 0 && col < WC) ? __ldg(src + (long long)iy * WC + col) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < NLD; ++i) {
            const int idx = m + i * 128;
            const int r = idx / STEM_IN_W, j = idx - r * STEM_IN_W;
            if (idx < STEM_IN_H * STEM_IN_W) sIn[r * STEM_IN_LD + j] = stage[i];
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        // ---- this pixel's patch, (r, s, c) order: element k = r*21 + s*3 + c sits at sIn[2*py + r][6*px + (k % 21)] ----
        const int py = m >> 4, px = m & 15;
        const float* base = sIn + (2 * py) * STEM_IN_LD + 6 * px;
#pragma unroll
        for (int kb = 0; kb < STEM_KB; ++kb) {
#pragma unroll
            for (int c8 = 0; c8 < 8; ++c8) {
                uint4 o;
                __half2* ho = reinterpret_cast<__half2*>(&o);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int k0 = kb * 64 + c8 * 8 + 2 * e, k1 = k0 + 1;
                    const float a = k0 < STEM_KK ? base[(k0 / 21) * STEM_IN_LD + (k0 % 21)] : 0.f;
                    const float b = k1 < STEM_KK ? base[(k1 / 21) * STEM_IN_LD + (k1 % 21)] : 0.f;
                    ho[e] = __floats2half2_rn(a, b);
                }
                *reinterpret_cast<uint4*>(sA + kb * TC_A_BYTES + m * 128 + ((c8 ^ (m & 7)) << 4)) = o;
            }
        }
        fence_proxy_async();                                    // generic-proxy writes -> visible to the tensor core (async proxy)
        mbar_arrive(bar_a);
        // ---- epilogue ----
        mbar_wait(bar_mma, 0);
        tc_fence_after();
        const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
        epi_rows_f16<64>(p.bias, 64, 1, false, 0, m, trow, sA);
        fence_proxy_async();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (m == 0) {
            tma_store_3d(&p.mapY[img], sA, 0, ox0, oy0);
            tma_store_commit_and_wait_read();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) tmem_dealloc(tmem_base, 64);
}

// hi = x with the 13 low mantissa bits cleared (exactly representable in TF32), lo = x - hi (exact in fp32)
__global__ void split_tf32_kernel(const float4* __restrict__ x, float4* __restrict__ hi, float4* __restrict__ lo, long long n4) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    float4 v = __ldg(x + i), h, l;
    h.x = __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u); l.x = v.x - h.x;
    h.y = __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u); l.y = v.y - h.y;
    h.z = __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u); l.z = v.z - h.z;
    h.w = __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u); l.w = v.w - h.w;
    hi[i] = h;
    lo[i] = l;
}

// fp16 split for the correlation (precision 2) of both feature matrices in ONE launch: hi = fp16(x), lo = fp16((x - hi) * 2^11);
// hi/lo of A then hi/lo of B are consecutive in the workspace, and the arg-max keys are zeroed by the first threads.
__global__ void split_f16_all_kernel(const float4* __restrict__ A, const float4* __restrict__ B, uint2* __restrict__ Ahi, uint2* __restrict__ Alo,
                                     uint2* __restrict__ Bhi, uint2* __restrict__ Blo, long long na4, long long nb4,
                                     unsigned long long* __restrict__ keys, long long nkeys) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nkeys) keys[i] = 0ull;
    if (i >= na4 + nb4) return;
    const bool isA = i < na4;
    const long long k = isA ? i : i - na4;
    const float4 v = __ldg((isA ? A : B) + k);
    const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
    const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
    const __half2 l0 = __floats2half2_rn((v.x - f0.x) * 2048.f, (v.y - f0.y) * 2048.f);
    const __half2 l1 = __floats2half2_rn((v.z - f1.x) * 2048.f, (v.w - f1.y) * 2048.f);
    uint2 ho, lo2;
    ho.x = *reinterpret_cast<const uint32_t*>(&h0); ho.y = *reinterpret_cast<const uint32_t*>(&h1);
    lo2.x = *reinterpret_cast<const uint32_t*>(&l0); lo2.y = *reinterpret_cast<const uint32_t*>(&l1);
    (isA ? Ahi : Bhi)[k] = ho;
    (isA ? Alo : Blo)[k] = lo2;
}

// ------------------------------------------------------------------ host side: tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    return fn;
}

struct MapKey {
    const void* ptr;
    unsigned long long d0, d1, d2, d3, plane;
    unsigned b0, b1, b2, b3, es, esize;
    bool operator==(const MapKey& o) const {
        return ptr == o.ptr && d0 == o.d0 && d1 == o.d1 && d2 == o.d2 && d3 == o.d3 && plane == o.plane && b0 == o.b0 && b1 == o.b1 && b2 == o.b2 &&
               b3 == o.b3 && es == o.es && esize == o.esize;
    }
};
struct MapKeyHash {
    size_t operator()(const MapKey& k) const {
        size_t h = std::hash<const void*>()(k.ptr);
        auto mix = [&](unsigned long long v) { h ^= std::hash<unsigned long long>()(v) + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2); };
        mix(k.d0); mix(k.d1); mix(k.d2); mix(k.d3); mix(k.plane); mix(k.b0); mix(k.b1); mix(k.b2); mix(k.b3); mix(k.es); mix(k.esize);
        return h;
    }
};
static std::mutex g_map_mu;
static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_maps;

// fp32 (esize 4) or fp16 (esize 2) tensor (d0 innermost, d1, d2[, d3]), dense strides (the 4-D form: d3 planes `plane_bytes`
// apart), box of (b0, b1, b2[, b3]) ELEMENTS LOADED, traversal stride `es` on d1 / d2 (strided convolutions: every es-th
// pixel), 128B swizzle, zero fill out of bounds
int get_map4(CUtensorMap* out, const void* ptr, unsigned long long d0, unsigned long long d1, unsigned long long d2, unsigned long long d3,
             unsigned long long plane_bytes, unsigned b0, unsigned b1, unsigned b2, unsigned b3, unsigned es_, unsigned esize) {
    MapKey key{ptr, d0, d1, d2, d3, plane_bytes, b0, b1, b2, b3, es_, esize};
    std::lock_guard<std::mutex> g(g_map_mu);
    auto it = g_maps.find(key);
    if (it != g_maps.end()) { *out = it->second; return 0; }
    EncodeTiledFn enc = get_encode();
    if (!enc) return fail_msg("cuTensorMapEncodeTiled is not available from this driver");
    cuuint64_t dims[4] = {d0, d1, d2, d3};
    cuuint64_t strides[3] = {d0 * (unsigned long long)esize, d0 * d1 * (unsigned long long)esize, plane_bytes};
    cuuint32_t box[4] = {b0, b1 * es_, b2 * es_, b3};      // bounding box in tensor coordinates; ceil(box / stride) elements are loaded
    cuuint32_t es[4] = {1, es_, es_, 1};
    int rank = d3 > 0 ? 4 : (d2 > 0 ? 3 : 2);
    CUresult r = enc(out, esize == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, rank, const_cast<void*>(ptr), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled failed with CUresult %d (dims %llu,%llu,%llu,%llu box %u,%u,%u,%u)", (int)r, d0, d1, d2, d3, b0, b1, b2, b3);
        return 3;
    }
    if (g_maps.size() > 8192) g_maps.clear();
    g_maps[key] = *out;
    return 0;
}

int get_map(CUtensorMap* out, const void* ptr, unsigned long long d0, unsigned long long d1, unsigned long long d2,
            unsigned b0, unsigned b1, unsigned b2, unsigned es_, unsigned esize) {
    return get_map4(out, ptr, d0, d1, d2, 0, 0, b0, b1, b2, 0, es_, esize);
}

int pick_tw(int Ho, int Wo) {
    // tile = tw x (128/tw) output pixels: minimise the padded area
    int best = 16;
    long long best_area = -1;
    const int cands[5] = {16, 32, 8, 64, 128};
    for (int i = 0; i < 5; ++i) {
        int tw = cands[i], th = 128 / tw;
        long long area = (long long)((Wo + tw - 1) / tw) * ((Ho + th - 1) / th);
        if (best_area < 0 || area < best_area) { best_area = area; best = tw; }
    }
    return best;
}

// Off by default: measured -2 % end to end (profiles/README.md), the extra staging costs a resident CTA.  Kept because
// the kernel without this path compiles worse: ptxas moves the one-tile fp16 kernel's prologue off the uniform datapath
// (80 -> 84 registers) and those kernels run 12 % slower.
static int respf_mode() {
    const char* e = getenv("RF_TC_RESPF");    // fp16 1x1 convs with a residual: prefetch the residual tile at CTA start
    return e ? atoi(e) : 0;
}

template <bool F16>
static int launch_resb(const TcParams& p, int tiles_m, cudaStream_t st) {
    static bool attr[64] = {false};
    const int dev = current_device();
    if (!attr[dev]) {
        RF_CUDA(cudaFuncSetAttribute(tc_resb_kernel<F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, ResBCfg<F16>::SMEM_BYTES));
        attr[dev] = true;
    }
    const int grid = tiles_m < num_sms() ? tiles_m : num_sms();
    tc_resb_kernel<F16><<<grid, TC_THREADS, ResBCfg<F16>::SMEM_BYTES, st>>>(p, tiles_m);
    RF_LAUNCHED();
    return 0;
}

template <int BN>
static int launch_pipe(const TcParams& p, int tiles_m, int tiles_n, cudaStream_t st) {
    using Cfg = PipeCfg<BN>;
    static bool attr[64] = {false};
    const int dev = current_device();
    if (!attr[dev]) {
        RF_CUDA(cudaFuncSetAttribute(tc_pipe_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        attr[dev] = true;
    }
    const int total = tiles_m * tiles_n;
    const int grid = total < num_sms() ? total : num_sms();
    tc_pipe_kernel<BN><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, st>>>(p, tiles_m, tiles_n);
    RF_LAUNCHED();
    return 0;
}

template <int BN, bool F16 = false, bool OUT32 = false>
static int launch_halo(const TcParams& p, int tiles, int ntiles_n, cudaStream_t st) {
    using Cfg = HaloCfg<BN>;
    static bool attr[64] = {false};
    const int dev = current_device();
    if (!attr[dev]) {
        RF_CUDA(cudaFuncSetAttribute(tc_halo_kernel<BN, F16, OUT32>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        attr[dev] = true;
    }
    tc_halo_kernel<BN, F16, OUT32><<<dim3(tiles, ntiles_n), TC_THREADS, Cfg::SMEM_BYTES, st>>>(p);
    RF_LAUNCHED();
    return 0;
}

template <int BN, int MODE, bool DEEP, bool F16 = false>
static int launch_tc(const TcParams& p, int tiles, int ntiles_n, cudaStream_t st) {
    using Cfg = TcCfg<BN, MODE, DEEP>;
    static bool attr[64] = {false};
    const int dev = current_device();
    if (!attr[dev]) {
        RF_CUDA(cudaFuncSetAttribute(tc_kernel<BN, MODE, DEEP, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     Cfg::SMEM_BYTES + (F16 ? (BN / 64) * TC_A_BYTES : 0)));
        attr[dev] = true;
    }
    dim3 grid = (MODE == MODE_CORR || p.raster_n) ? dim3(ntiles_n, tiles) : dim3(tiles, ntiles_n);
    if (F16 && MODE == MODE_CONV) {
        // ring depth: never more stages than K blocks; with a prefetched residual two stages (+ its staging) keep two or
        // three CTAs resident per SM
        TcParams q = p;
        const int KI = p.R * p.S * (p.Cin / TC_BK_F16);
        q.res_pf = (p.residual != nullptr && respf_mode()) ? 1 : 0;
        int stages = KI < Cfg::STAGES ? KI : Cfg::STAGES;
        if (q.res_pf && stages > 2) stages = 2;
        q.stages = stages;
        const int smem = stages * Cfg::STAGE_BYTES + (q.res_pf ? (BN / 64) * TC_A_BYTES : 0) + 1024 + 256;
        tc_kernel<BN, MODE, DEEP, F16><<<grid, TC_THREADS, smem, st>>>(q);
        RF_LAUNCHED();
        return 0;
    }
    tc_kernel<BN, MODE, DEEP, F16><<<grid, TC_THREADS, Cfg::SMEM_BYTES, st>>>(p);
    RF_LAUNCHED();
    return 0;
}

}  // namespace rf

using namespace rf;

bool rf_conv2d_tc_supported(const ConvParams& p) {
    return (p.stride == 1 || p.stride == 2) && (p.Cin % TC_BK) == 0 && p.Cout >= 1 && p.R == p.S && (p.R == 1 || p.R == 3);
}
// engine 2: fp16 activations / weights; every layer must fit (there is no fp16 SIMT path to fall back to)
bool rf_conv2d_f16_supported(const ConvParams& p) {
    return (p.stride == 1 || p.stride == 2) && (p.Cin % TC_BK_F16) == 0 && p.Cout >= 8 && (p.Cout % 8) == 0 && p.R == p.S && (p.R == 1 || p.R == 3);
}

// f16 = false: x / residual / y fp32, w_tc fp32 [Cout][K] (TF32-rounded).  f16 = true: the same pointers hold IEEE fp16.
// out32 (with f16): y is fp32 (3x3 / stride 1 layers only, no residual) - the hand-over from fp16 layers to a TF32 consumer.
int rf_conv2d_tc(const ImgSet& set, const ConvParams& cp, const void* w_tc, cudaStream_t st, bool f16, bool out32) {
    RF_REQUIRE(w_tc != nullptr, "rf_conv2d_nhwc: tensor-core engines need w_tc ([Cout][R*S*Cin])");
    RF_REQUIRE(f16 ? rf_conv2d_f16_supported(cp) : rf_conv2d_tc_supported(cp),
               "rf_conv2d_nhwc: tensor-core engines need stride 1 or 2, 1x1 or 3x3, Cin % 32 == 0 (fp16: Cin % 64 == 0, Cout % 8 == 0)");
    TcParams p;
    memset(&p, 0, sizeof(p));
    const int BN = cp.Cout > 64 ? 128 : 64;
    const unsigned esz = f16 ? 2u : 4u;
    const unsigned bk = f16 ? TC_BK_F16 : TC_BK;
    const unsigned esz_y = (f16 && !out32) ? 2u : 4u;                // output (and residual) element size
    const unsigned bk_y = (f16 && !out32) ? TC_BK_F16 : TC_BK;
    RF_REQUIRE(!out32 || (f16 && cp.R == 3 && cp.stride == 1 && cp.pad == 1 && cp.residual == nullptr),
               "rf_conv2d_nhwc: engine 3 (fp16 operands, fp32 output) covers 3x3 / stride 1 / pad 1 layers without residual");
    const char* xb = reinterpret_cast<const char*>(cp.x);
    const char* rb = reinterpret_cast<const char*>(cp.residual);
    char* yb = reinterpret_cast<char*>(cp.y);
    p.nimg = set.n;
    const bool halo = cp.R == 3 && cp.stride == 1 && cp.pad == 1;      // halo reuse (tc_halo_kernel, tc_resb_kernel)
    int tiles = 0;
    for (int i = 0; i < set.n; ++i) {
        int tw = halo ? HALO_TW : pick_tw(set.Ho[i], set.Wo[i]), th = 128 / tw;
        p.tw[i] = tw;
        p.tiles_x[i] = (set.Wo[i] + tw - 1) / tw;
        p.tile_start[i] = tiles;
        tiles += p.tiles_x[i] * ((set.Ho[i] + th - 1) / th);
        p.Ho[i] = set.Ho[i]; p.Wo[i] = set.Wo[i];
        p.out_pix[i] = set.out_pix[i];
        int rc = get_map(&p.mapA[i], xb + set.in_pix[i] * cp.Cin * esz, (unsigned long long)cp.Cin, (unsigned long long)set.W[i],
                         (unsigned long long)set.H[i], bk, (unsigned)(halo ? tw + 2 : tw), (unsigned)(halo ? th + 2 : th), (unsigned)cp.stride, esz);
        if (rc) return rc;
    }
    // bulk (TMA) epilogue whenever the output rows are 16-byte aligned (fp32: Cout % 4 == 0; fp16: Cout % 8 == 0, required)
    p.tma_epi = (((cp.Cout * esz_y) & 15) == 0 && ((uintptr_t)cp.y % 16) == 0 && ((uintptr_t)cp.residual % 16) == 0) ? 1 : 0;
    RF_REQUIRE(!f16 || out32 || p.tma_epi, "rf_conv2d_nhwc: engine 2 needs 16-byte aligned y / residual");
    if (p.tma_epi) {
        for (int i = 0; i < set.n; ++i) {
            const unsigned tw = (unsigned)p.tw[i], th = 128u / tw;
            int rc = get_map(&p.mapY[i], yb + set.out_pix[i] * cp.Cout * esz_y, (unsigned long long)cp.Cout, (unsigned long long)set.Wo[i],
                             (unsigned long long)set.Ho[i], bk_y, tw, th, 1, esz_y);
            if (!rc && cp.residual)
                rc = get_map(&p.mapR[i], rb + set.out_pix[i] * cp.Cout * esz_y, (unsigned long long)cp.Cout, (unsigned long long)set.Wo[i],
                             (unsigned long long)set.Ho[i], bk_y, tw, th, 1, esz_y);
            if (rc) return rc;
        }
    }
    for (int i = set.n; i <= RF_MAX_IMGS; ++i) p.tile_start[i] = tiles;
    p.out_pix[set.n] = set.out_pix[set.n];
    int rc = get_map(&p.mapB, w_tc, (unsigned long long)cp.K, (unsigned long long)cp.Cout, 0, bk, (unsigned)BN, 0, 1, esz);
    if (rc) return rc;
    p.R = cp.R; p.S = cp.S; p.pad = cp.pad; p.stride = cp.stride; p.Cin = cp.Cin; p.Cout = cp.Cout; p.relu = cp.relu; p.round_out = cp.round_out;
    p.bias = cp.bias; p.residual = cp.residual; p.y = cp.y;
    const int nt = (cp.Cout + BN - 1) / BN;
    // channel tiles fastest for the tap-streaming kernels: the CTAs of one pixel tile run together (A once from HBM, whole
    // output rows; +2 % per pair); the grid's y dimension holds at most 65535 pixel tiles
    p.raster_n = tiles <= 65535 ? 1 : 0;
    const bool deep = cp.K >= 512;                                   // >= 16 K-steps of 32 fp32 channels (8 of 64 fp16)
    // the weights-resident persistent kernel for 64 -> 64 3x3 convs (a 3-slot / direct-store variant measured no faster:
    // 332 vs 320 us per pair)
    const bool resb = halo && cp.Cin == 64 && cp.Cout == 64;
    if (f16 && out32) return BN == 128 ? launch_halo<128, true, true>(p, tiles, nt, st) : launch_halo<64, true, true>(p, tiles, nt, st);
    if (f16) {
        if (resb) return launch_resb<true>(p, tiles, st);
        if (halo) return BN == 128 ? launch_halo<128, true>(p, tiles, nt, st) : launch_halo<64, true>(p, tiles, nt, st);
        // the pipelined persistent kernel where it measured faster: >= 4 K blocks and >= 2 tiles per SM
        if (cp.K >= 4 * TC_BK_F16 && (long long)tiles * nt >= 2ll * num_sms())
            return BN == 128 ? launch_pipe<128>(p, tiles, nt, st) : launch_pipe<64>(p, tiles, nt, st);
        if (BN == 128) return deep ? launch_tc<128, MODE_CONV, true, true>(p, tiles, nt, st) : launch_tc<128, MODE_CONV, false, true>(p, tiles, nt, st);
        return deep ? launch_tc<64, MODE_CONV, true, true>(p, tiles, nt, st) : launch_tc<64, MODE_CONV, false, true>(p, tiles, nt, st);
    }
    if (resb && p.tma_epi) return launch_resb<false>(p, tiles, st);
    if (halo) return BN == 128 ? launch_halo<128>(p, tiles, nt, st) : launch_halo<64>(p, tiles, nt, st);
    if (BN == 128) return deep ? launch_tc<128, MODE_CONV, true>(p, tiles, nt, st) : launch_tc<128, MODE_CONV, false>(p, tiles, nt, st);
    return deep ? launch_tc<64, MODE_CONV, true>(p, tiles, nt, st) : launch_tc<64, MODE_CONV, false>(p, tiles, nt, st);
}

// engine 2: fused ResNet-50 stem (see stem7_f16_kernel).  x fp32 [sum HW][3], w_f16 [64][192] ((r, s, c) order, zero
// padded), bias fp32 [64], y fp16 [sum HoWo][64]
int rf_stem7_f16_impl(const float* x, int nimg, const int* hw_host, const void* w_f16, const float* bias, void* y_f16, void* stream) {
    RF_REQUIRE(x != nullptr && w_f16 != nullptr && y_f16 != nullptr, "rf_stem7: null pointer");
    RF_REQUIRE(((uintptr_t)y_f16 % 16) == 0 && ((uintptr_t)w_f16 % 16) == 0, "rf_stem7: pointers must be 16-byte aligned");
    ImgSet set;
    RF_REQUIRE(make_imgset(set, nimg, hw_host, 7, 2, 3) == 0, "rf_stem7: bad image set");
    StemParams p;
    memset(&p, 0, sizeof(p));
    p.nimg = nimg;
    int tiles = 0;
    for (int i = 0; i < nimg; ++i) {
        p.tiles_x[i] = (set.Wo[i] + STEM_TW - 1) / STEM_TW;
        p.tile_start[i] = tiles;
        tiles += p.tiles_x[i] * ((set.Ho[i] + STEM_TH - 1) / STEM_TH);
        p.H[i] = set.H[i]; p.W[i] = set.W[i];
        p.in_pix[i] = set.in_pix[i];
        int rc = get_map(&p.mapY[i], static_cast<char*>(y_f16) + set.out_pix[i] * 64 * 2, 64ull, (unsigned long long)set.Wo[i],
                         (unsigned long long)set.Ho[i], 64, STEM_TW, STEM_TH, 1, 2);
        if (rc) return rc;
    }
    for (int i = nimg; i <= RF_MAX_IMGS; ++i) p.tile_start[i] = tiles;
    int rc = get_map(&p.mapB, w_f16, 192ull, 64ull, 0, 64, 64, 0, 1, 2);
    if (rc) return rc;
    p.x = x; p.bias = bias;
    static bool attr[64] = {false};
    const int dev = current_device();
    if (!attr[dev]) {
        RF_CUDA(cudaFuncSetAttribute(stem7_f16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, STEM_SMEM));
        attr[dev] = true;
    }
    stem7_f16_kernel<<<tiles, STEM_THREADS, STEM_SMEM, as_stream(stream)>>>(p);
    RF_LAUNCHED();
    return 0;
}

size_t rf_corr_tc_workspace(int NA, int NB, int C) { return 2ull * ((size_t)NA + NB) * C * sizeof(float) + 1024; }

static int launch_corr_pipe(const TcParams& p, int tiles_m, int tiles_n, cudaStream_t st) {
    using Cfg = CorrPipeCfg;
    static bool attr[64] = {false};
    const int dev = current_device();
    if (!attr[dev]) {
        RF_CUDA(cudaFuncSetAttribute(tc_corr_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        attr[dev] = true;
    }
    const long long total = (long long)tiles_m * tiles_n;
    const int grid = total < num_sms() ? (int)total : num_sms();
    tc_corr_pipe_kernel<<<grid, TC_THREADS, Cfg::SMEM_BYTES, st>>>(p, tiles_m, tiles_n);
    RF_LAUNCHED();
    return 0;
}

// precision 1: 3xTF32 one-tile-per-CTA kernel; the caller has zeroed rowbest / colbest.
// precision 2: the persistent fp16-split kernel.  presplit (nullable): {A hi, A lo, B hi, B lo} fp16 planes written by the
// producer of the features (rf_l2norm_split_nhwc): no split launch, the caller has zeroed the keys.  Without presplit the
// split launch zeroes rowbest / colbest (contiguous, NA + NB keys).
int rf_corr_argmax_tc(const float* featA, int NA, const float* featB, int NB, int C,
                      unsigned long long* rowbest, unsigned long long* colbest, void* ws, cudaStream_t st, int precision,
                      const void* const* presplit) {
    const bool f16 = precision == 2;
    RF_REQUIRE(presplit == nullptr || f16, "rf_corr_mutual_nn: pre-split operands go with the persistent fp16-split kernel");
    RF_REQUIRE((C % (f16 ? TC_BK_F16 : TC_BK)) == 0, "rf_corr_mutual_nn: precision 1 needs C % 32 == 0, precision 2 C % 64 == 0");
    uintptr_t base = (reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255;
    const size_t esz = f16 ? 2 : 4;
    char* Ahi = reinterpret_cast<char*>(base);
    char* Alo = Ahi + (size_t)NA * C * esz;
    char* Bhi = Alo + (size_t)NA * C * esz;
    char* Blo = Bhi + (size_t)NB * C * esz;
    long long na4 = (long long)NA * C / 4, nb4 = (long long)NB * C / 4;
    if (presplit != nullptr) {
        Ahi = const_cast<char*>(static_cast<const char*>(presplit[0]));
        Alo = const_cast<char*>(static_cast<const char*>(presplit[1]));
        Bhi = const_cast<char*>(static_cast<const char*>(presplit[2]));
        Blo = const_cast<char*>(static_cast<const char*>(presplit[3]));
        for (int i = 0; i < 4; ++i) RF_REQUIRE(presplit[i] != nullptr && ((uintptr_t)presplit[i] % 16) == 0, "rf_corr_mutual_nn_presplit: planes must be 16-byte aligned");
    } else if (f16) {
        RF_REQUIRE(colbest == rowbest + NA, "rf_corr_mutual_nn: arg-max keys must be contiguous");
        const long long nkeys = (long long)NA + NB, n = na4 + nb4 > nkeys ? na4 + nb4 : nkeys;
        split_f16_all_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const float4*)featA, (const float4*)featB, (uint2*)Ahi, (uint2*)Alo,
                                                                            (uint2*)Bhi, (uint2*)Blo, na4, nb4, rowbest, nkeys);
        RF_LAUNCHED();
    } else {
        split_tf32_kernel<<<(unsigned)((na4 + 255) / 256), 256, 0, st>>>((const float4*)featA, (float4*)Ahi, (float4*)Alo, na4);
        RF_LAUNCHED();
        split_tf32_kernel<<<(unsigned)((nb4 + 255) / 256), 256, 0, st>>>((const float4*)featB, (float4*)Bhi, (float4*)Blo, nb4);
        RF_LAUNCHED();
    }
    const int BN = 128;
    const unsigned bk = f16 ? TC_BK_F16 : TC_BK, es = (unsigned)esz;
    TcParams p;
    memset(&p, 0, sizeof(p));
    p.nimg = 1;
    p.tw[0] = 128;
    p.tiles_x[0] = (NA + 127) / 128;
    p.tile_start[0] = 0;
    for (int i = 1; i <= RF_MAX_IMGS; ++i) p.tile_start[i] = p.tiles_x[0];
    p.Ho[0] = 1; p.Wo[0] = NA;
    int rc = get_map(&p.mapA[0], Ahi, (unsigned long long)C, (unsigned long long)NA, 1, bk, 128, 1, 1, es);
    if (!rc) rc = get_map(&p.mapAlo, Alo, (unsigned long long)C, (unsigned long long)NA, 1, bk, 128, 1, 1, es);
    if (!rc) rc = get_map(&p.mapB, Bhi, (unsigned long long)C, (unsigned long long)NB, 0, bk, BN, 0, 1, es);
    if (!rc) rc = get_map(&p.mapBlo, Blo, (unsigned long long)C, (unsigned long long)NB, 0, bk, BN, 0, 1, es);
    if (rc) return rc;
    p.R = 1; p.S = 1; p.pad = 0; p.stride = 1; p.Cin = C; p.Cout = NB;
    p.rowbest = rowbest; p.colbest = colbest; p.NA = NA; p.NB = NB;
    if (f16) return launch_corr_pipe(p, p.tiles_x[0], (NB + BN - 1) / BN, st);
    return launch_tc<BN, MODE_CORR, false>(p, p.tiles_x[0], (NB + BN - 1) / BN, st);
}
