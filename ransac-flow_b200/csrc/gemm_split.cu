// Engine 4 ("f16x3"): fp32-GRADE convolutions on the tcgen05 tensor cores.
//
// The reference runs its networks in fp32 (quick_start/coarseAlignFeatMatch.py:34-52,106; model/model.py:59-125,167-322)
// and the mutual-nearest-neighbour arg-max of utils/outil.py:34-43 is decided by score gaps of a few 1e-7, so 10-bit
// tensor-core operands (TF32 / fp16 activations) do not reproduce its match set.  Here every activation and weight is
// carried as TWO fp16 planes, x = hi + lo * 2^-11 with hi = fp16(x), lo = fp16((x - hi) * 2^11) (22 significand bits), and
// every MAC is three kind::f16 MMAs: hi*hi into one TMEM accumulator, hi*lo + lo*hi (at 2^11 scale) into a second one; the
// epilogue adds them with one fma, applies folded-BN bias / residual / ReLU in fp32 and writes the result split again.
//
// Data layout: a split tensor is [2][P][C] fp16 (plane 0 = hi, plane 1 = lo * 2^11; 4 bytes per element like fp32).  Every
// TMA tensor map is 4-D (C, W, H, plane) with a box of 2 planes, so ONE bulk copy brings the hi and the lo tile of a K block
// into consecutive shared memory ([hi tile | lo tile], both 128-byte swizzled), one copy stores both output planes, one
// loads both residual planes.  Weights are (K, Cout, plane) with a 3-D box.
//
// One persistent kernel, one CTA per SM, 320 threads:
//   warp 0    : TMA producer.  Tap streaming (1x1 of any stride, 3x3 / stride 2): A = (64 ch, tw, th, 2) box at the tap's
//               offset (zero padding by out-of-bounds fill), B = (64 k, 64 rows, 2) box.  HALO (3x3 / stride 1): A = the
//               (8+2) x (16+2) halo of one 64-channel block once, the nine taps are nine UMMA descriptors into it (see
//               tc_halo_kernel in gemm_tc.cu), B = nine weight boxes.  Runs ahead across tiles, never waits for an epilogue.
//   warp 1    : MMA issuer.  Two accumulator PAIRS (main | cross) x 64 columns x 2 buffers = 256 TMEM columns: tile i+1
//               multiplies while tile i drains.
//   warps 2-5 : epilogue group 0 (even tiles), warps 6-9: group 1 (odd tiles): TMEM -> main + cross * 2^-11 + bias
//               (+ residual hi + lo * 2^-11, TMA-loaded into the group's staging buffer by its own leader) -> ReLU -> split ->
//               swizzled staging [hi box | lo box] -> one TMA store.
//               `out32`: fp32 rows straight to global memory instead (the 49- / 1-channel outputs of the heads).

#include "common.cuh"
#include "tc_common.cuh"

namespace rf {

constexpr int SP_BN = 64;
constexpr int SP_EPW = 8;                                                   // warps per epilogue group
constexpr int SP_THREADS = 64 + 2 * 32 * SP_EPW;                            // producer warp + MMA warp + two epilogue groups
constexpr int SP_HALO_TW = 8, SP_HALO_TH = 16, SP_HALO_LD = SP_HALO_TW + 2;
constexpr int SP_HALO_PLANE = SP_HALO_LD * (SP_HALO_TH + 2) * 128;          // 23040 B: one plane of a halo block

struct alignas(64) SplitParams {
    CUtensorMap mapA[RF_MAX_IMGS];        // per image: input (Cin, W, H, 2) fp16
    CUtensorMap mapY[RF_MAX_IMGS];        // per image: output (Cout, Wo, Ho, 2), box (64, tw, th, 2)
    CUtensorMap mapR[RF_MAX_IMGS];        // per image: residual, same geometry as the output
    CUtensorMap mapB;                     // weights (K, Cout, 2), box (64, 64, 2)
    int nimg;
    int tile_start[RF_MAX_IMGS + 1];
    int tiles_x[RF_MAX_IMGS];
    float inv_tiles_x[RF_MAX_IMGS];       // 1 / tiles_x, 1 / tiles_n: tile decoding without integer divisions (sp_fast_div)
    float inv_tiles_n;
    int tw[RF_MAX_IMGS];
    int tw_shift[RF_MAX_IMGS];            // log2(tw): tiles are tw x (128 / tw) pixels, tw a power of two
    int Ho[RF_MAX_IMGS], Wo[RF_MAX_IMGS];
    long long out_pix[RF_MAX_IMGS + 1];
    int R, S, pad, stride, Cin, Cout, relu, has_res, out32;
    int tiles_m, tiles_n;
    int kc1, stride2;                     // dual-input 1x1: K blocks [0, kc1) come from mapA, the rest from mapR (second input, its own stride)
    const float* bias;
    float* y32;                           // out32: fp32 [P][Cout]
};

// BN = 64: the two epilogue groups take alternate tiles.  BN = 128 (tap streaming only): each group takes one 64-channel half of
// EVERY tile - twice the work per operand byte fetched from L2 (the tap-streaming layers are L2-bandwidth bound at BN = 64:
// 48 KB per K block for 12 MMAs) and N = 128 MMAs, which the shared-memory read port can feed at the full tensor rate.
// RES2 (tap streaming, BN = 64, layers with a residual): TWO staging buffers per epilogue group, so that the residual tile of
// the group's next tile is in flight while the current one is combined and stored; paid for with a 2-deep operand ring (these
// layers have K <= 256: one to four K blocks per tile).
template <bool HALO, int BN_, bool RES2_ = false>
struct SplitCfg {
    static constexpr int BN = BN_;
    static constexpr bool RES2 = RES2_;
    static constexpr int B_PLANE = BN * 128;                                  // 8 / 16 KB
    static constexpr int B_TILE = 2 * B_PLANE;                                // hi + lo planes of one weight tile
    static constexpr int A_LO = HALO ? SP_HALO_PLANE : TC_A_BYTES;            // offset of the lo plane inside an A slot
    static constexpr int A_TX = 2 * A_LO;
    static constexpr int A_SLOT = HALO ? 46 * 1024 : 2 * TC_A_BYTES;          // 1024-byte aligned slots
    static constexpr int NA = HALO ? 2 : ((BN == 128 || RES2) ? 2 : 3);
    static constexpr int NB = HALO ? (BN == 128 ? 2 : 4) : (RES2 ? 2 : 3);
    static constexpr int NSB = RES2 ? 2 : 1;                                  // staging buffers per epilogue group
    static constexpr int TB = HALO ? 9 : 1;                                   // B tiles consumed per A slot
    static constexpr int STG = 2 * TC_A_BYTES;                                // per epilogue group: [hi box | lo box] of 64 channels
    static constexpr int OFF_B = NA * A_SLOT;
    static constexpr int OFF_STG = OFF_B + NB * B_TILE;
    static constexpr int DATA_BYTES = OFF_STG + 2 * NSB * STG;
    static constexpr int SMEM_BYTES = DATA_BYTES + 1024 + 512;
    static constexpr int TMEM_COLS = 4 * BN;                                  // 2 buffers x (main | cross)
    static_assert(!RES2 || (!HALO && BN == 64), "double-buffered staging: tap streaming, 64-channel tiles");
};
static_assert(SplitCfg<true, 128>::SMEM_BYTES <= 227 * 1024, "shared memory");
static_assert(SplitCfg<true, 64>::SMEM_BYTES <= 227 * 1024 && SplitCfg<false, 64>::SMEM_BYTES <= 227 * 1024 &&
              SplitCfg<false, 128>::SMEM_BYTES <= 227 * 1024 && SplitCfg<false, 64, true>::SMEM_BYTES <= 227 * 1024, "shared memory");
static_assert(SplitCfg<true, 64>::A_TX <= SplitCfg<true, 64>::A_SLOT, "halo slot");

__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(smem_u32(smem_dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"((uint64_t)map), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}

// K-major, 128-byte swizzle, 8-row core groups one HALO row pitch (10 pixels = 1280 B) apart; base offset 0 (the
// swizzle of tcgen05.mma is a function of the shared-memory address: gemm_tc.cu make_desc_halo, measured in round 1)
__device__ __forceinline__ uint64_t sp_desc_halo(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)(saddr >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((SP_HALO_LD * 128) >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

static_assert(sizeof(SplitParams) <= 32764, "kernel parameter space (CUDA 12.1+ large kernel parameters)");

struct SpTile { int img, ox0, oy0, tw, n0, tw_shift; };

// a / d for 0 <= a < 2^24 with inv = 1.0f / d: the float quotient is within one of the exact one, one correction step makes it exact
// (an integer division is ~25 instructions; the tile decode runs once per tile in every warp of the kernel)
__device__ __forceinline__ int sp_fast_div(int a, int d, float inv) {
    int q = __float2int_rz(__int2float_rn(a) * inv);
    const int r = a - q * d;
    q += (r >= d) ? 1 : 0;
    q -= (r < 0) ? 1 : 0;
    return q;
}


template <bool HALO, int BN = SP_BN>
__device__ __forceinline__ SpTile sp_decode(const SplitParams& p, int t) {
    SpTile c;
    const int mt = sp_fast_div(t, p.tiles_n, p.inv_tiles_n), nt = t - mt * p.tiles_n;      // channel tiles fastest: co-running CTAs share the pixel tile
    int img = 0;
#pragma unroll
    for (int j = 1; j < RF_MAX_IMGS; ++j) img += (j < p.nimg && mt >= p.tile_start[j]) ? 1 : 0;
    const int tloc = mt - p.tile_start[img];
    c.img = img;
    c.tw = HALO ? SP_HALO_TW : p.tw[img];
    c.tw_shift = HALO ? 3 : p.tw_shift[img];
    const int th = 128 >> c.tw_shift;
    const int tyi = sp_fast_div(tloc, p.tiles_x[img], p.inv_tiles_x[img]), txi = tloc - tyi * p.tiles_x[img];
    c.ox0 = txi * c.tw;
    c.oy0 = tyi * th;
    c.n0 = nt * BN;
    return c;
}

// split one fp32 value pair into (hi, lo * 2^11) half2 pairs, saturating like the fp16 engine
// (cvt.rn.satfinite: one instruction per pair converts, packs and clamps to +-65504; an overflowing value gets hi = lo = 65504)
__device__ __forceinline__ __half2 sp_pack_sat(float a, float b) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));     // first source -> upper half
    return *reinterpret_cast<__half2*>(&r);
}
__device__ __forceinline__ void sp_split2(float a, float b, __half2& hi, __half2& lo) {
    hi = sp_pack_sat(a, b);
    const float2 f = __half22float2(hi);
    lo = sp_pack_sat((a - f.x) * 2048.f, (b - f.y) * 2048.f);
}

template <bool HALO, int BN_, bool RES2 = false>
__global__ void __launch_bounds__(SP_THREADS, 1)
tc_split_kernel(const __grid_constant__ SplitParams p) {
    using Cfg = SplitCfg<HALO, BN_, RES2>;
    constexpr int GT = 32 * SP_EPW;             // threads of one epilogue group
    constexpr int NSB = Cfg::NSB;
    constexpr int BN = Cfg::BN, NA = Cfg::NA, NB = Cfg::NB, TB = Cfg::TB, BK = TC_BK_F16;
    constexpr bool WIDE = BN == 128;            // both epilogue groups work on every tile (one 64-channel half each)
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);      // pointer arithmetic keeps the shared address space (LDS / STS, not generic LD / ST)
    uint8_t* sA = smem;
    uint8_t* sB = smem + Cfg::OFF_B;
    uint8_t* sStg = smem + Cfg::OFF_STG;
    uint64_t* fullA = reinterpret_cast<uint64_t*>(smem + Cfg::DATA_BYTES);
    uint64_t* emptyA = fullA + NA;
    uint64_t* fullB = emptyA + NA;
    uint64_t* emptyB = fullB + NB;
    uint64_t* tmem_full = emptyB + NB;          // [2]
    uint64_t* tmem_empty = tmem_full + 2;       // [2] 128 arrivals
    uint64_t* res_full = tmem_empty + 2;        // [2 groups][2 buffers] the residual tile has landed in that staging buffer
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_full + 4);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total = p.tiles_m * p.tiles_n;
    const int kc = p.Cin / BK;
    const int NAI = HALO ? kc : p.R * p.S * kc;             // A slots per tile
    const bool has_res = p.has_res != 0;

    if (threadIdx.x == 0) {
        for (int i = 0; i < NA; ++i) { mbar_init(&fullA[i], 1); mbar_init(&emptyA[i], 1); }
        for (int i = 0; i < NB; ++i) { mbar_init(&fullB[i], 1); mbar_init(&emptyB[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], WIDE ? 2 * GT : GT); }
        for (int i = 0; i < 4; ++i) mbar_init(&res_full[i], 1);
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
            uint32_t ia_cnt = 0, ib_cnt = 0, ti = 0;
            for (int t = blockIdx.x; t < total; t += gridDim.x, ++ti) {
                const SpTile c = sp_decode<HALO, BN>(p, t);
                for (int ia = 0; ia < NAI; ++ia, ++ia_cnt) {
                    const int sa = ia_cnt % NA;
                    mbar_wait(&emptyA[sa], ((ia_cnt / NA) & 1) ^ 1);
                    int tap = 0, cc = ia;
                    if (HALO) {
                        mbar_expect_tx(&fullA[sa], Cfg::A_TX);
                        tma_load_4d(sA + sa * Cfg::A_SLOT, &p.mapA[c.img], &fullA[sa], ia * BK, c.ox0 - 1, c.oy0 - 1, 0);
                    } else {
                        mbar_expect_tx(&fullA[sa], Cfg::A_TX);
                        tap = ia / kc;
                        cc = ia - tap * kc;
                        const int r = tap / p.S, sx = tap - r * p.S;
                        if (cc < p.kc1)
                            tma_load_4d(sA + sa * Cfg::A_SLOT, &p.mapA[c.img], &fullA[sa], cc * BK, c.ox0 * p.stride + sx - p.pad,
                                        c.oy0 * p.stride + r - p.pad, 0);
                        else                                                // second input of a dual 1x1 (the fused down-sampling branch)
                            tma_load_4d(sA + sa * Cfg::A_SLOT, &p.mapR[c.img], &fullA[sa], (cc - p.kc1) * BK, c.ox0 * p.stride2, c.oy0 * p.stride2, 0);
                    }
                    for (int jb = 0; jb < TB; ++jb, ++ib_cnt) {
                        const int sb = ib_cnt % NB;
                        mbar_wait(&emptyB[sb], ((ib_cnt / NB) & 1) ^ 1);
                        mbar_expect_tx(&fullB[sb], Cfg::B_TILE);
                        const int btap = HALO ? jb : tap;
                        tma_load_3d(sB + sb * Cfg::B_TILE, &p.mapB, &fullB[sb], btap * p.Cin + cc * BK, c.n0, 0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // =============================== MMA issuer (whole warp, warp-uniform) ===============================
        constexpr uint32_t idesc = make_idesc_f16(BN);
        uint32_t ia_cnt = 0, ib_cnt = 0, ti = 0;
        for (int t = blockIdx.x; t < total; t += gridDim.x, ++ti) {
            const uint32_t buf = ti & 1;
            mbar_wait(&tmem_empty[buf], ((ti >> 1) & 1) ^ 1);               // the epilogue has drained this accumulator pair
            tc_fence_after();
            const uint32_t td = tmem_base + buf * (2 * BN);
            for (int ia = 0; ia < NAI; ++ia, ++ia_cnt) {
                const int sa = ia_cnt % NA;
                mbar_wait(&fullA[sa], (ia_cnt / NA) & 1);
                tc_fence_after();
                const uint32_t abase = smem_u32(sA + sa * Cfg::A_SLOT);
                for (int jb = 0; jb < TB; ++jb, ++ib_cnt) {
                    const int sb = ib_cnt % NB;
                    mbar_wait(&fullB[sb], (ib_cnt / NB) & 1);
                    tc_fence_after();
                    const uint32_t bb = smem_u32(sB + sb * Cfg::B_TILE);
                    uint32_t aaddr = abase;
                    if (HALO) { const int r = jb / 3, sx = jb - r * 3; aaddr += (uint32_t)((r * SP_HALO_LD + sx) * 128); }
                    const uint64_t ahi = HALO ? sp_desc_halo(aaddr) : make_desc_sw128(aaddr);
                    const uint64_t alo = HALO ? sp_desc_halo(aaddr + Cfg::A_LO) : make_desc_sw128(aaddr + Cfg::A_LO);
                    // [B hi | B lo] as one 2N-wide instruction + A lo x B hi
                    umma_f16split2_x4(td, BN, ahi, alo, make_desc_sw128(bb), make_idesc_f16(2 * BN), idesc, (ia | jb) != 0 ? 1u : 0u);
                    umma_commit(&emptyB[sb]);
                }
                umma_commit(&emptyA[sa]);
            }
            umma_commit(&tmem_full[buf]);
        }
    } else {
        // =============================== epilogue groups ===============================
        // A group is eight warps: two warps per TMEM lane quarter, 32 columns each - the epilogue is ~11 fp32 instructions per
        // output element (combine, bias, residual hi + lo, ReLU, split) in dependent chains, and with K <= 256 it, not the MMAs
        // or HBM, sets the tile rate (ncu: 2.5 warps per scheduler, 6.2 cycles between issues); sixteen epilogue warps halve the
        // drain time of an accumulator pair against one warp per quarter.
        const uint32_t g = (uint32_t)(warp - 2) / SP_EPW;                   // group 0 / 1
        const int idx = (warp - 2) % SP_EPW;
        const int q = warp & 3;                                             // TMEM lane quarter this warp may access
        const int m = q * 32 + lane;
        const bool leader = idx == 0 && lane == 0;
        const int cb = idx >> 2;                                            // this warp's 32-column block
        uint8_t* stg_base = sStg + g * NSB * Cfg::STG;
        uint32_t k = 0;                                                     // this group's tile counter
        const int t_first = blockIdx.x + (WIDE ? 0 : (int)g * (int)gridDim.x), t_step = (WIDE ? 1 : 2) * (int)gridDim.x;
        auto group_sync = [&]() {
            if (g == 0) asm volatile("bar.sync 1, %0;" ::"n"(GT) : "memory"); else asm volatile("bar.sync 2, %0;" ::"n"(GT) : "memory");
        };
        // Residual tiles come in by TMA into the group's OWN staging buffer, issued by the group's leader: the first one here,
        // the next one as soon as the store of the current tile has read the buffer out.  (First version: the producer warp
        // issued them and had to wait for the staging buffer of tile i-2 - that wait stalled the operand loads of tile i behind
        // the epilogue of tile i-2; second version: each thread loaded its residual row from global memory into registers -
        // 16 uncoalesced 16-byte loads per thread through an L1 squeezed to ~28 KB by the 220 KB of shared memory: 1.3-1.5x slower.)
        // RES2: two buffers per group - the residual of tile k + 1 is issued while tile k is being combined, a whole group
        // cycle ahead of its use, and the store of tile k needs no wait before the group moves on.
        if (leader && has_res && t_first < total) {
            const SpTile c0 = sp_decode<HALO, BN>(p, t_first);
            mbar_expect_tx(&res_full[2 * g], Cfg::STG);
            tma_load_4d(stg_base, &p.mapR[c0.img], &res_full[2 * g], c0.n0 + (WIDE ? 64 * (int)g : 0), c0.ox0, c0.oy0, 0);
        }
        const bool bias_vec = p.bias != nullptr && (p.Cout & 3) == 0;
        for (int t = t_first; t < total; t += t_step, ++k) {
            const SpTile c = sp_decode<HALO, BN>(p, t);
            const uint32_t buf = WIDE ? (k & 1) : g;                        // accumulator pair of this tile
            const uint32_t fph = WIDE ? ((k >> 1) & 1) : (k & 1);           // phase of its tmem_full barrier
            const int nbase = c.n0 + (WIDE ? 64 * (int)g : 0);              // first output channel of this group's 64-wide slice
            const int py = m >> c.tw_shift, px = m - (py << c.tw_shift);
            const bool pvalid = (c.oy0 + py < p.Ho[c.img]) && (c.ox0 + px < p.Wo[c.img]);
            const long long pix = p.out_pix[c.img] + (long long)(c.oy0 + py) * p.Wo[c.img] + (c.ox0 + px);
            // the leader comes here only after the previous store has read the staging buffer (two buffers, no residual: the
            // store of tile k - 2 used this tile's buffer; the one of tile k - 1 may still be reading the other)
            if (RES2 && !has_res && leader) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            group_sync();
            const uint32_t sb = RES2 ? (k & 1) : 0;                         // staging buffer of this tile
            uint8_t* stg = stg_base + sb * Cfg::STG;
            mbar_wait(&tmem_full[buf], fph);
            tc_fence_after();
            if (has_res) mbar_wait(&res_full[2 * g + sb], RES2 ? ((k >> 1) & 1) : (k & 1));
            if (RES2 && has_res && leader) {
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");      // the other buffer's store (tile k - 1) has read it out
                if (t + t_step < total) {
                    const SpTile cn = sp_decode<HALO, BN>(p, t + t_step);
                    mbar_expect_tx(&res_full[2 * g + (sb ^ 1)], Cfg::STG);
                    tma_load_4d(stg_base + (sb ^ 1) * Cfg::STG, &p.mapR[cn.img], &res_full[2 * g + (sb ^ 1)], cn.n0, cn.ox0, cn.oy0, 0);
                }
            }
            const uint32_t trow = tmem_base + buf * (2 * BN) + (WIDE ? 64 * g : 0) + ((uint32_t)(q * 32) << 16);
            float* yrow = p.out32 ? p.y32 + pix * p.Cout : nullptr;
            {
                uint32_t v[32], x[32];
                tmem_ld32x2(trow + cb * 32, v, trow + BN + cb * 32, x);
                const int n = nbase + cb * 32;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float o[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) o[e] = fmaf(__uint_as_float(x[8 * j + e]), 0.00048828125f, __uint_as_float(v[8 * j + e]));
                    if (p.bias != nullptr) {
                        if (bias_vec && n + 8 * j + 8 <= p.Cout) {
                            const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + n + 8 * j));
                            const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + n + 8 * j + 4));
                            o[0] += b0.x; o[1] += b0.y; o[2] += b0.z; o[3] += b0.w; o[4] += b1.x; o[5] += b1.y; o[6] += b1.z; o[7] += b1.w;
                        } else {
#pragma unroll
                            for (int e = 0; e < 8; ++e) if (n + 8 * j + e < p.Cout) o[e] += __ldg(p.bias + n + 8 * j + e);
                        }
                    }
                    if (p.out32) {
                        if (pvalid) {
#pragma unroll
                            for (int e = 0; e < 8; ++e)
                                if (n + 8 * j + e < p.Cout) yrow[n + 8 * j + e] = p.relu ? fmaxf(o[e], 0.f) : o[e];
                        }
                        continue;
                    }
                    const int chunk = cb * 4 + j;
                    uint4* hp = reinterpret_cast<uint4*>(stg + m * 128 + ((chunk ^ (m & 7)) << 4));
                    uint4* lp = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(hp) + TC_A_BYTES);
                    if (has_res) {
                        const uint4 rh = *hp, rl = *lp;
                        const __half2* h = reinterpret_cast<const __half2*>(&rh);
                        const __half2* l = reinterpret_cast<const __half2*>(&rl);
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float2 fh = __half22float2(h[e]), fl = __half22float2(l[e]);
                            o[2 * e] += fmaf(fl.x, 0.00048828125f, fh.x);
                            o[2 * e + 1] += fmaf(fl.y, 0.00048828125f, fh.y);
                        }
                    }
                    if (p.relu) {
#pragma unroll
                        for (int e = 0; e < 8; ++e) o[e] = fmaxf(o[e], 0.f);
                    }
                    uint4 oh, ol;
                    __half2* ph = reinterpret_cast<__half2*>(&oh);
                    __half2* pl = reinterpret_cast<__half2*>(&ol);
#pragma unroll
                    for (int e = 0; e < 4; ++e) sp_split2(o[2 * e], o[2 * e + 1], ph[e], pl[e]);
                    *hp = oh;
                    *lp = ol;
                }
            }
            tc_fence_before();
            mbar_arrive(&tmem_empty[buf]);                                  // accumulator pair drained (GT arrivals per group)
            if (!p.out32) {
                fence_proxy_async();
                group_sync();
                if (leader) {
                    if (nbase < p.Cout) tma_store_4d(&p.mapY[c.img], stg, nbase, c.ox0, c.oy0, 0);
                    if (RES2) {
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");   // read out while the group works on its next tile
                    } else {
                        tma_store_commit_and_wait_read();
                        if (has_res && t + t_step < total) {                // the group's next residual tile, into the buffer just read out
                            const SpTile cn = sp_decode<HALO, BN>(p, t + t_step);
                            mbar_expect_tx(&res_full[2 * g], Cfg::STG);
                            tma_load_4d(stg, &p.mapR[cn.img], &res_full[2 * g], cn.n0 + (WIDE ? 64 * (int)g : 0), cn.ox0, cn.oy0, 0);
                        }
                    }
                }
            }
        }
        if (RES2 && leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------------------
// ResNet-50 stem, fused, split operands: conv 7x7 / stride 2 / pad 3 on the 3-channel fp32 image + folded BN + ReLU ->
// split NHWC, without an im2col matrix in HBM.  PERSISTENT and warp specialised, one CTA per SM, 416 threads:
//   warps 0-7 : builders (two threads per output pixel, half a patch each).  Stage the 37 x 21 x 3 input window of the tile in shared memory (the NEXT tile's window is
//               already in flight in registers), then build the tile's 147-long (r, s, c) patches as hi / lo planes
//               straight in the 128-byte-swizzled K-major layout (3 + 3 K blocks of 64), fence.proxy.async, arrive;
//   warp 8    : loads the split weights ONCE per CTA (48 KB), then per tile nine MMA groups into accumulator pair
//               (tile & 1); one commit hands the patch buffer back to the builders, one publishes the accumulators;
//   warps 9-12: epilogue.  TMEM -> + bias, ReLU, split -> [hi box | lo box] staging -> one TMA store of both planes,
//               overlapped with the builders' next tile.
// History (config 2, 7132 tiles): one tile per CTA, everything serial, 155 KB: 358 us; persistent with a single reused K-block
// slot and two CTAs per SM: 408 us (three build -> MMA -> commit round trips per tile); this version: see profiles/.
// ------------------------------------------------------------------------------------------------------------
constexpr int SS_TW = 16, SS_TH = 8, SS_K = 7, SS_C = 3, SS_KK = 147, SS_KB = 3;
constexpr int SS_IN_W = ((SS_TW - 1) * 2 + SS_K) * SS_C;                  // 111 floats per staged input row
constexpr int SS_IN_H = (SS_TH - 1) * 2 + SS_K;                           // 21 rows
constexpr int SS_IN_LD = 112;
constexpr int SS_B_TILE = 2 * 64 * 128;                                   // [hi | lo] weights of one K block: 16 KB
constexpr int SS_OFF_ALO = SS_KB * TC_A_BYTES;                            // 48 KB: lo planes of the patches
constexpr int SS_OFF_B = 2 * SS_KB * TC_A_BYTES;                          // 96 KB
constexpr int SS_OFF_STG = SS_OFF_B + SS_KB * SS_B_TILE;                  // 144 KB
constexpr int SS_OFF_IN = SS_OFF_STG + 2 * TC_A_BYTES;                    // 176 KB
constexpr int SS_OFF_BAR = SS_OFF_IN + SS_IN_H * SS_IN_LD * 4;
constexpr int SS_SMEM = SS_OFF_BAR + 128 + 1024;
constexpr int SS_BUILD = 256;                                             // builder threads: two per output pixel (half a patch each)
constexpr int SS_EPI = 256;                                               // epilogue threads: two warps per TMEM lane quarter, 32 columns each
constexpr int SS_THREADS = SS_BUILD + 32 + SS_EPI;                        // + MMA warp + 8 epilogue warps
constexpr int SS_NLD = (SS_IN_H * SS_IN_W + SS_BUILD - 1) / SS_BUILD;      // window floats per builder thread
static_assert(SS_SMEM <= 227 * 1024, "stem shared memory");

struct alignas(64) StemSplitParams {
    CUtensorMap mapB;                     // weights (192, 64, 2) fp16, box (64, 64, 2)
    CUtensorMap mapY[RF_MAX_IMGS];        // output (64, Wo, Ho, 2), box (64, 16, 8, 2)
    int nimg, total;
    int tile_start[RF_MAX_IMGS + 1];
    int tiles_x[RF_MAX_IMGS];
    float inv_tiles_x[RF_MAX_IMGS];
    int H[RF_MAX_IMGS], W[RF_MAX_IMGS];
    long long in_pix[RF_MAX_IMGS];
    const float* x;
    const float* bias;
};

struct StemTile { int img, ox0, oy0; };
__device__ __forceinline__ StemTile stem_decode(const StemSplitParams& p, int t) {
    StemTile c;
    int img = 0;
#pragma unroll
    for (int j = 1; j < RF_MAX_IMGS; ++j) img += (j < p.nimg && t >= p.tile_start[j]) ? 1 : 0;
    const int tloc = t - p.tile_start[img];
    const int tyi = sp_fast_div(tloc, p.tiles_x[img], p.inv_tiles_x[img]), txi = tloc - tyi * p.tiles_x[img];
    c.img = img;
    c.ox0 = txi * SS_TW;
    c.oy0 = tyi * SS_TH;
    return c;
}
// the (zero padded) 21 x 111 input window of a tile, SS_BUILD threads x SS_NLD floats
__device__ __forceinline__ void stem_load_window(const StemSplitParams& p, const StemTile& c, int m, float (&stage)[SS_NLD]) {
    const int H = p.H[c.img], WC = p.W[c.img] * SS_C;
    const float* src = p.x + p.in_pix[c.img] * SS_C;
    const int iy0 = c.oy0 * 2 - 3, col0 = (c.ox0 * 2 - 3) * SS_C;
#pragma unroll
    for (int i = 0; i < SS_NLD; ++i) {
        const int idx = m + i * SS_BUILD;
        const int r = idx / SS_IN_W, j = idx - r * SS_IN_W;
        const int iy = iy0 + r, col = col0 + j;
        stage[i] = (idx < SS_IN_H * SS_IN_W && iy >= 0 && iy < H && col >= 0 && col < WC) ? __ldg(src + (long long)iy * WC + col) : 0.f;
    }
}

// one staged window element: (hi, lo * 2^11) fp16 pair packed in 32 bits (hi in the low half).  The window is split ONCE when it is
// staged (2 331 values per tile); the patches (24 576 values per tile, every input pixel sits in ~12 of them) are then pure
// byte shuffles: 2 LDS + 2 PRMT per element pair instead of 2 LDS + ~12 conversions / subtractions / multiplications.
__device__ __forceinline__ uint32_t stem_pack_split(float v) {
    __half2 hi, lo;
    sp_split2(v, 0.f, hi, lo);
    return (*reinterpret_cast<uint32_t*>(&hi) & 0xFFFFu) | (*reinterpret_cast<uint32_t*>(&lo) << 16);
}

// half a patch: the 16-byte chunks 4 * HALF .. 4 * HALF + 3 of each of the three K blocks of pixel m, hi and lo planes
template <int HALF, int kb>
__device__ __forceinline__ void stem_build_half(const uint32_t* __restrict__ base, uint8_t* sA, int m) {
    {
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            const int c8 = HALF * 4 + cc;
            uint4 oh, ol;
            uint32_t* ph = reinterpret_cast<uint32_t*>(&oh);
            uint32_t* pl = reinterpret_cast<uint32_t*>(&ol);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int k0 = kb * 64 + c8 * 8 + 2 * e, k1 = k0 + 1;
                const uint32_t a = k0 < SS_KK ? base[(k0 / 21) * SS_IN_LD + (k0 % 21)] : 0u;
                const uint32_t b = k1 < SS_KK ? base[(k1 / 21) * SS_IN_LD + (k1 % 21)] : 0u;
                ph[e] = __byte_perm(a, b, 0x5410);          // (hi(a), hi(b))
                pl[e] = __byte_perm(a, b, 0x7632);          // (lo(a), lo(b))
            }
            uint8_t* dst = sA + kb * TC_A_BYTES + m * 128 + ((c8 ^ (m & 7)) << 4);
            *reinterpret_cast<uint4*>(dst) = oh;
            *reinterpret_cast<uint4*>(dst + SS_OFF_ALO) = ol;
        }
    }
}

__global__ void __launch_bounds__(SS_THREADS, 1)
stem7_split_kernel(const __grid_constant__ StemSplitParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);      // pointer arithmetic keeps the shared address space (LDS / STS, not generic LD / ST)
    uint8_t* sA = smem;
    uint8_t* sB = smem + SS_OFF_B;
    uint8_t* sStg = smem + SS_OFF_STG;
    uint32_t* sIn = reinterpret_cast<uint32_t*>(smem + SS_OFF_IN);      // the staged window as packed (hi, lo) pairs
    uint64_t* bar_b = reinterpret_cast<uint64_t*>(smem + SS_OFF_BAR);
    uint64_t* bar_a = bar_b + 1;          // [3] SS_BUILD arrivals: K block kb of the tile's patches is in shared memory
    uint64_t* bar_free = bar_a + SS_KB;   // [3] commit: the MMAs reading K block kb are done
    uint64_t* tmem_full = bar_free + SS_KB;   // [2] commit: accumulator pair complete
    uint64_t* tmem_empty = tmem_full + 2; // [2] 128 arrivals: the epilogue has drained it
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        mbar_init(bar_b, 1);
        for (int i = 0; i < SS_KB; ++i) { mbar_init(&bar_a[i], SS_BUILD); mbar_init(&bar_free[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], SS_EPI); }
        fence_barrier_init();
    }
    constexpr int WMMA = SS_BUILD / 32;                         // the MMA warp sits right behind the builders
    if (warp == WMMA) {
        if (lane == 0) { tma_prefetch_desc(&p.mapB); tma_prefetch_desc(&p.mapY[0]); }
        tmem_alloc(tmem_slot, 256);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp < WMMA) {
        // =============================== builders ===============================
        const int bt = threadIdx.x;                             // 0..255
        const int m = bt & 127, half = bt >> 7;                 // output pixel inside the tile = A row; which half of each K block
        const int py = m >> 4, px = m & 15;
        const uint32_t* base = sIn + (2 * py) * SS_IN_LD + 6 * px;
        float stage[SS_NLD];
        StemTile c = stem_decode(p, (int)blockIdx.x < p.total ? (int)blockIdx.x : 0);
        if ((int)blockIdx.x < p.total) stem_load_window(p, c, bt, stage);
        uint32_t ti = 0;
        for (int t = blockIdx.x; t < p.total; t += gridDim.x, ++ti) {
            asm volatile("bar.sync 1, 256;" ::: "memory");      // everybody has finished reading the previous window
#pragma unroll
            for (int i = 0; i < SS_NLD; ++i) {
                const int idx = bt + i * SS_BUILD;
                const int r = idx / SS_IN_W, j = idx - r * SS_IN_W;
                if (idx < SS_IN_H * SS_IN_W) sIn[r * SS_IN_LD + j] = stem_pack_split(stage[i]);
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (t + (int)gridDim.x < p.total) {                 // next tile's window: in flight while this tile is built
                c = stem_decode(p, t + gridDim.x);
                stem_load_window(p, c, bt, stage);
            }
            // the three K blocks of the patch buffer are a ring between the builders and the MMA warp: block kb of this tile is
            // built as soon as the previous tile's MMAs on block kb are done, while its blocks kb + 1.. are still being multiplied
            // (one barrier pair for the whole buffer serialised build and MMAs: 2.3 k + 2.7 k cycles per tile)
            // ---- this pixel's patch, (r, s, c) order: element k = r*21 + s*3 + c sits at sIn[2*py + r][6*px + (k % 21)] ----
            // (thread `half` of the pixel builds the 16-byte chunks 4 * half .. 4 * half + 3 of each K block; warp-uniform branch, so
            // that every (k / 21, k % 21) stays a compile-time constant)
#define RF_STEM_BLOCK(KB)                                                                                              \
            if (ti > 0) mbar_wait(&bar_free[KB], (ti - 1) & 1);                                                          \
            if (half == 0) stem_build_half<0, KB>(base, sA, m); else stem_build_half<1, KB>(base, sA, m);                \
            fence_proxy_async();            /* generic-proxy writes -> visible to the tensor core (async proxy) */      \
            mbar_arrive(&bar_a[KB]);
            RF_STEM_BLOCK(0)
            RF_STEM_BLOCK(1)
            RF_STEM_BLOCK(2)
#undef RF_STEM_BLOCK
        }
    } else if (warp == WMMA) {
        // =============================== weights once, then the MMA issuer ===============================
        if (lane == 0) {
            mbar_expect_tx(bar_b, SS_KB * SS_B_TILE);
#pragma unroll
            for (int kb = 0; kb < SS_KB; ++kb) tma_load_3d(sB + kb * SS_B_TILE, &p.mapB, bar_b, kb * 64, 0, 0);
        }
        mbar_wait(bar_b, 0);
        constexpr uint32_t idesc = make_idesc_f16(64);
        uint32_t ti = 0;
        for (int t = blockIdx.x; t < p.total; t += gridDim.x, ++ti) {
            const uint32_t buf = ti & 1;
            mbar_wait(&tmem_empty[buf], ((ti >> 1) & 1) ^ 1);
            tc_fence_after();
            const uint32_t td = tmem_base + buf * 128;
#pragma unroll
            for (int kb = 0; kb < SS_KB; ++kb) {
                mbar_wait(&bar_a[kb], ti & 1);
                tc_fence_after();
                const uint32_t a = smem_u32(sA + kb * TC_A_BYTES), b = smem_u32(sB + kb * SS_B_TILE);
                // [B hi | B lo] are adjacent (SS_B_TILE), main | cross accumulators too: two MMAs per K step
                umma_f16split2_x4(td, 64, make_desc_sw128(a), make_desc_sw128(a + SS_OFF_ALO), make_desc_sw128(b), make_idesc_f16(128), idesc,
                                  kb != 0 ? 1u : 0u);
                umma_commit(&bar_free[kb]);
            }
            umma_commit(&tmem_full[buf]);
        }
    } else {
        // =============================== epilogue (8 warps) ===============================
        // one 4-warp group drained an accumulator pair in ~5 k cycles - the tile rate of the whole kernel (the builders and the
        // MMAs need ~2.5 k each); two warps per lane quarter, 32 of the 64 columns each
        const int q = warp & 3;                                 // TMEM lane quarter this warp may access
        const int m = q * 32 + lane;
        const int cb = (warp - (WMMA + 1)) >> 2;                // this warp's 32-column block
        const bool leader = (warp == WMMA + 1 && lane == 0);
        uint32_t ti = 0;
        for (int t = blockIdx.x; t < p.total; t += gridDim.x, ++ti) {
            const uint32_t buf = ti & 1;
            const StemTile c = stem_decode(p, t);
            asm volatile("bar.sync 2, %0;" ::"n"(SS_EPI) : "memory");      // the leader's previous store has read the staging buffer
            mbar_wait(&tmem_full[buf], (ti >> 1) & 1);
            tc_fence_after();
            const uint32_t trow = tmem_base + buf * 128 + ((uint32_t)(q * 32) << 16);
            {
                uint32_t v[32], x[32];
                tmem_ld32x2(trow + cb * 32, v, trow + 64 + cb * 32, x);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float o[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) o[e] = fmaf(__uint_as_float(x[8 * j + e]), 0.00048828125f, __uint_as_float(v[8 * j + e]));
                    if (p.bias != nullptr) {
                        const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + cb * 32 + 8 * j));
                        const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + cb * 32 + 8 * j + 4));
                        o[0] += b0.x; o[1] += b0.y; o[2] += b0.z; o[3] += b0.w; o[4] += b1.x; o[5] += b1.y; o[6] += b1.z; o[7] += b1.w;
                    }
                    uint4 oh, ol;
                    __half2* ph = reinterpret_cast<__half2*>(&oh);
                    __half2* pl = reinterpret_cast<__half2*>(&ol);
#pragma unroll
                    for (int e = 0; e < 4; ++e) sp_split2(fmaxf(o[2 * e], 0.f), fmaxf(o[2 * e + 1], 0.f), ph[e], pl[e]);
                    const int chunk = cb * 4 + j;
                    uint8_t* dst = sStg + m * 128 + ((chunk ^ (m & 7)) << 4);
                    *reinterpret_cast<uint4*>(dst) = oh;
                    *reinterpret_cast<uint4*>(dst + TC_A_BYTES) = ol;
                }
            }
            tc_fence_before();
            mbar_arrive(&tmem_empty[buf]);
            fence_proxy_async();
            asm volatile("bar.sync 2, %0;" ::"n"(SS_EPI) : "memory");
            if (leader) {
                tma_store_4d(&p.mapY[c.img], sStg, 0, c.ox0, c.oy0, 0);
                tma_store_commit_and_wait_read();
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == WMMA) tmem_dealloc(tmem_base, 256);
}

}  // namespace rf

using namespace rf;

bool rf_conv2d_split_supported(const ConvParams& p) {
    return (p.stride == 1 || p.stride == 2) && (p.Cin % TC_BK_F16) == 0 && p.Cout >= 1 && p.R == p.S && (p.R == 1 || p.R == 3);
}

// x / residual / y: split tensors ([2][P][C] fp16, planes `P * C` elements apart); w_split: [2][Cout][K] fp16; out32: y is
// fp32 [P][Cout] (no residual).
// dual: a second input (x2, its own per-image sizes hw2, Cin2 channels, sampled with stride2) whose channels continue the K axis
// of a 1x1 convolution: y = act(W[:, :Cin] x + W[:, Cin:] x2[::stride2] + bias) - a bottleneck's conv3 and its down-sampling
// branch in one GEMM (the branch's output never goes to HBM and comes back as a residual).
struct SplitDual { const void* x2; const int* hw2; int Cin2, stride2; };

static int rf_conv2d_split_impl(const ImgSet& set, const ConvParams& cp, const void* w_split, cudaStream_t st, bool out32, const SplitDual* dual);

int rf_conv2d_split(const ImgSet& set, const ConvParams& cp, const void* w_split, cudaStream_t st, bool out32) {
    return rf_conv2d_split_impl(set, cp, w_split, st, out32, nullptr);
}

static int rf_conv2d_split_impl(const ImgSet& set, const ConvParams& cp, const void* w_split, cudaStream_t st, bool out32, const SplitDual* dual) {
    RF_REQUIRE(w_split != nullptr, "rf_conv2d_nhwc: engine 4 needs the split weights ([2][Cout][R*S*Cin] fp16)");
    RF_REQUIRE(rf_conv2d_split_supported(cp), "rf_conv2d_nhwc: engine 4 needs stride 1 or 2, 1x1 or 3x3, Cin % 64 == 0");
    RF_REQUIRE(out32 || (cp.Cout % 8) == 0, "rf_conv2d_nhwc: engine 4 needs Cout % 8 == 0 for split outputs");
    RF_REQUIRE(!out32 || cp.residual == nullptr, "rf_conv2d_nhwc: engine 4 fp32 outputs take no residual");
    RF_REQUIRE(((uintptr_t)cp.x % 16) == 0 && ((uintptr_t)cp.y % 16) == 0 && ((uintptr_t)cp.residual % 16) == 0 && ((uintptr_t)w_split % 16) == 0,
               "rf_conv2d_nhwc: engine 4 needs 16-byte aligned pointers");
    SplitParams p;
    memset(&p, 0, sizeof(p));
    const bool halo = (cp.R == 3 && cp.stride == 1 && cp.pad == 1);
    const char* xb = reinterpret_cast<const char*>(cp.x);
    const char* rb = reinterpret_cast<const char*>(cp.residual);
    char* yb = reinterpret_cast<char*>(cp.y);
    const unsigned long long in_plane = (unsigned long long)set.in_pix[set.n] * cp.Cin * 2ull;
    const unsigned long long out_plane = (unsigned long long)set.out_pix[set.n] * cp.Cout * 2ull;
    long long in2_pix[RF_MAX_IMGS + 1] = {0};
    if (dual) {
        RF_REQUIRE(!halo && cp.R == 1 && cp.stride == 1 && cp.pad == 0 && cp.residual == nullptr && !out32 && dual->x2 != nullptr &&
                   (dual->Cin2 % TC_BK_F16) == 0 && (dual->stride2 == 1 || dual->stride2 == 2) && ((uintptr_t)dual->x2 % 16) == 0,
                   "rf_conv1x1_dual_split: 1x1 / stride 1 on the first input, no residual, Cin2 % 64 == 0, stride2 1 or 2");
        for (int i = 0; i < set.n; ++i) {
            RF_REQUIRE((dual->hw2[2 * i] - 1) / dual->stride2 + 1 == set.Ho[i] && (dual->hw2[2 * i + 1] - 1) / dual->stride2 + 1 == set.Wo[i],
                       "rf_conv1x1_dual_split: the second input, sampled with stride2, must have the first input's size");
            in2_pix[i + 1] = in2_pix[i] + (long long)dual->hw2[2 * i] * dual->hw2[2 * i + 1];
        }
    }
    const unsigned long long in2_plane = dual ? (unsigned long long)in2_pix[set.n] * dual->Cin2 * 2ull : 0ull;
    p.nimg = set.n;
    int tiles = 0;
    for (int i = 0; i < set.n; ++i) {
        const int tw = halo ? SP_HALO_TW : pick_tw(set.Ho[i], set.Wo[i]), th = 128 / tw;
        p.tw[i] = tw;
        p.tw_shift[i] = 0;
        while ((1 << p.tw_shift[i]) < tw) ++p.tw_shift[i];
        RF_REQUIRE((1 << p.tw_shift[i]) == tw, "rf_conv2d_nhwc: tile width must be a power of two");
        p.tiles_x[i] = (set.Wo[i] + tw - 1) / tw;
        p.inv_tiles_x[i] = 1.0f / (float)p.tiles_x[i];
        p.tile_start[i] = tiles;
        tiles += p.tiles_x[i] * ((set.Ho[i] + th - 1) / th);
        p.Ho[i] = set.Ho[i]; p.Wo[i] = set.Wo[i];
        p.out_pix[i] = set.out_pix[i];
        int rc = get_map4(&p.mapA[i], xb + set.in_pix[i] * cp.Cin * 2, (unsigned long long)cp.Cin, (unsigned long long)set.W[i], (unsigned long long)set.H[i], 2,
                          in_plane, TC_BK_F16, (unsigned)(halo ? tw + 2 : tw), (unsigned)(halo ? th + 2 : th), 2, (unsigned)cp.stride, 2);
        if (rc) return rc;
        if (!out32) {
            rc = get_map4(&p.mapY[i], yb + set.out_pix[i] * cp.Cout * 2, (unsigned long long)cp.Cout, (unsigned long long)set.Wo[i], (unsigned long long)set.Ho[i], 2,
                          out_plane, TC_BK_F16, (unsigned)tw, (unsigned)th, 2, 1, 2);
            if (!rc && dual) {
                const long long off2 = in2_pix[i];
                rc = get_map4(&p.mapR[i], static_cast<const char*>(dual->x2) + off2 * dual->Cin2 * 2, (unsigned long long)dual->Cin2,
                              (unsigned long long)dual->hw2[2 * i + 1], (unsigned long long)dual->hw2[2 * i], 2, in2_plane, TC_BK_F16, (unsigned)tw,
                              (unsigned)th, 2, (unsigned)dual->stride2, 2);
            }
            if (!rc && cp.residual)
                rc = get_map4(&p.mapR[i], rb + set.out_pix[i] * cp.Cout * 2, (unsigned long long)cp.Cout, (unsigned long long)set.Wo[i], (unsigned long long)set.Ho[i], 2,
                              out_plane, TC_BK_F16, (unsigned)tw, (unsigned)th, 2, 1, 2);
            if (rc) return rc;
        }
    }
    for (int i = set.n; i <= RF_MAX_IMGS; ++i) p.tile_start[i] = tiles;
    p.out_pix[set.n] = set.out_pix[set.n];
    // measured per layer (profiles/r2_*): wide tiles pay for deep-K layers with >= 2 channel tiles and no residual (ResNet
    // down-sampling 1x1s, bottleneck c1 of layer 3, the stride-2 3x3s): -7 .. -15 %; the residual layers and 128-channel outputs
    // are faster with narrow tiles taken alternately by the two epilogue groups
    // ONE K block per tile and no residual (two K blocks - the fused conv3 + down-sampling of layer1 - need both operand slots of
    // that variant for one tile, which serialises load latency and MMAs: 116 us against 85 us with the wide tile): the epilogue sets the tile rate, and the double-buffered-staging variant
    // (64-channel tiles, store read-out off the critical path) beats the wide tile (ResNet layer1 down-sampling 1x1: 79 -> 75 us)
    const bool shallow = !halo && cp.R == 1 && cp.K <= 64;
    // halo reuse with 128-channel tiles (N = 128 MMAs: less issue overhead per MAC, half the halo-block traffic; two-deep weight ring)
    const bool halo_wide = halo && cp.Cout >= 128 && (cp.Cout % 128) == 0;
    const bool tap_wide = !halo && !shallow && (cp.Cout % 128) == 0 && (cp.residual == nullptr ? cp.Cout >= 256 : cp.K > 128);
    const int BN = (halo_wide || tap_wide) ? 128 : 64;
    int rc = get_map(&p.mapB, w_split, (unsigned long long)cp.K, (unsigned long long)cp.Cout, 2, TC_BK_F16, (unsigned)BN, 2, 1, 2);
    if (rc) return rc;
    p.R = cp.R; p.S = cp.S; p.pad = cp.pad; p.stride = cp.stride; p.Cin = cp.Cin; p.Cout = cp.Cout; p.relu = cp.relu;
    p.kc1 = cp.Cin / TC_BK_F16;
    p.stride2 = 1;
    if (dual) { p.Cin = cp.Cin + dual->Cin2; p.stride2 = dual->stride2; }      // the kernel's K axis: both inputs
    p.has_res = cp.residual != nullptr ? 1 : 0;
    p.out32 = out32 ? 1 : 0;
    p.bias = cp.bias;
    p.y32 = out32 ? cp.y : nullptr;

    p.tiles_m = tiles;
    p.tiles_n = (cp.Cout + BN - 1) / BN;
    p.inv_tiles_n = 1.0f / (float)p.tiles_n;
    const long long total = (long long)p.tiles_m * p.tiles_n;
    RF_REQUIRE(total < (1ll << 24), "rf_conv2d_nhwc: too many tiles");          // sp_fast_div is exact below 2^24
    const int grid = total < num_sms() ? (int)total : num_sms();
    // double-buffered staging pays for the HBM-bound residual layers with one or two K blocks per tile (ResNet layer 1 / 2
    // c3 + residual: 147 -> 121 us, 81 -> 64 us); with four K blocks (layer 3) the 2-deep operand ring costs more than the
    // residual prefetch gains (45 -> 52 us): measured, profiles/README.md
    const int which = halo ? (halo_wide ? 4 : 1) : (BN == 128 ? 2 : (((cp.residual != nullptr && cp.K <= 128) || shallow) ? 3 : 0));
    const int dev = current_device();
    static bool attr[64][5] = {{false}};
    auto launch = [&](auto kernel, int smem, int slot) {
        if (!attr[dev][slot]) {
            RF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            attr[dev][slot] = true;
        }
        kernel<<<grid, SP_THREADS, smem, st>>>(p);
        return 0;
    };
    int lrc;
    if (which == 4) lrc = launch(tc_split_kernel<true, 128>, SplitCfg<true, 128>::SMEM_BYTES, 4);
    else if (which == 1) lrc = launch(tc_split_kernel<true, 64>, SplitCfg<true, 64>::SMEM_BYTES, 0);
    else if (which == 2) lrc = launch(tc_split_kernel<false, 128>, SplitCfg<false, 128>::SMEM_BYTES, 1);
    else if (which == 3) lrc = launch(tc_split_kernel<false, 64, true>, SplitCfg<false, 64, true>::SMEM_BYTES, 2);
    else lrc = launch(tc_split_kernel<false, 64>, SplitCfg<false, 64>::SMEM_BYTES, 3);
    if (lrc) return lrc;
    RF_LAUNCHED();
    return 0;
}

extern "C" int rf_conv1x1_dual_split(const void* x1, const void* x2, int nimg, const int* hw1_host, const int* hw2_host, int Cin1, int Cin2,
                                     int stride2, const void* w_split, const float* bias, int Cout, int relu, void* y, void* stream) {
    RF_REQUIRE(x1 != nullptr && x2 != nullptr && y != nullptr && hw1_host != nullptr && hw2_host != nullptr, "rf_conv1x1_dual_split: null pointer");
    RF_REQUIRE(Cin1 >= 1 && Cin2 >= 1 && Cout >= 1, "rf_conv1x1_dual_split: bad channel counts");
    ImgSet set;
    RF_REQUIRE(make_imgset(set, nimg, hw1_host, 1, 1, 0) == 0, "rf_conv1x1_dual_split: bad image set");
    ConvParams p;
    p.x = static_cast<const float*>(x1); p.w = nullptr; p.bias = bias; p.residual = nullptr; p.y = static_cast<float*>(y);
    p.Cin = Cin1; p.Cout = Cout; p.R = 1; p.S = 1; p.stride = 1; p.pad = 0; p.relu = relu;
    p.round_out = 0;
    p.Mtot = set.out_pix[nimg];
    p.K = Cin1 + Cin2;
    SplitDual dual{x2, hw2_host, Cin2, stride2};
    return rf_conv2d_split_impl(set, p, w_split, as_stream(stream), false, &dual);
}

// engine 4: fused ResNet-50 stem.  x fp32 [sum HW][3], w_split [2][64][192] fp16 ((r, s, c) order, zero padded), bias fp32 [64],
// y split [2][sum HoWo][64]
int rf_stem7_split_impl(const float* x, int nimg, const int* hw_host, const void* w_split, const float* bias, void* y_split, void* stream) {
    RF_REQUIRE(x != nullptr && w_split != nullptr && y_split != nullptr, "rf_stem7: null pointer");
    RF_REQUIRE(((uintptr_t)y_split % 16) == 0 && ((uintptr_t)w_split % 16) == 0, "rf_stem7: pointers must be 16-byte aligned");
    ImgSet set;
    RF_REQUIRE(make_imgset(set, nimg, hw_host, 7, 2, 3) == 0, "rf_stem7: bad image set");
    StemSplitParams p;
    memset(&p, 0, sizeof(p));
    p.nimg = nimg;
    const unsigned long long out_plane = (unsigned long long)set.out_pix[nimg] * 64ull * 2ull;
    int tiles = 0;
    for (int i = 0; i < nimg; ++i) {
        p.tiles_x[i] = (set.Wo[i] + SS_TW - 1) / SS_TW;
        p.inv_tiles_x[i] = 1.0f / (float)p.tiles_x[i];
        p.tile_start[i] = tiles;
        tiles += p.tiles_x[i] * ((set.Ho[i] + SS_TH - 1) / SS_TH);
        p.H[i] = set.H[i]; p.W[i] = set.W[i];
        p.in_pix[i] = set.in_pix[i];
        int rc = get_map4(&p.mapY[i], static_cast<char*>(y_split) + set.out_pix[i] * 64 * 2, 64ull, (unsigned long long)set.Wo[i],
                          (unsigned long long)set.Ho[i], 2, out_plane, 64, SS_TW, SS_TH, 2, 1, 2);
        if (rc) return rc;
    }
    for (int i = nimg; i <= RF_MAX_IMGS; ++i) p.tile_start[i] = tiles;
    int rc = get_map(&p.mapB, w_split, 192ull, 64ull, 2, 64, 64, 2, 1, 2);
    if (rc) return rc;
    p.x = x; p.bias = bias;
    static bool attr[64] = {false};
    const int dev = current_device();
    if (!attr[dev]) {
        RF_CUDA(cudaFuncSetAttribute(stem7_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SS_SMEM));
        attr[dev] = true;
    }
    p.total = tiles;
    const int grid = tiles < num_sms() ? tiles : num_sms();
    stem7_split_kernel<<<grid, SS_THREADS, SS_SMEM, as_stream(stream)>>>(p);
    RF_LAUNCHED();
    return 0;
}
