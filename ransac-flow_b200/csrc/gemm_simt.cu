// Exact-fp32 (FMA, SIMT) GEMM-shaped kernels: the precise engine of the library.
//
//  * corr_argmax_kernel  - utils/outil.py:34-41: score = featA^T featB with the
//    row/column arg-max fused into the epilogue; the NA x NB matrix is never written.
//  * conv_kernel         - implicit-GEMM convolution over a ragged NHWC batch with
//    folded BatchNorm bias, residual add and ReLU in the epilogue
//    (model/model.py:27-56,59-125,167-322; torchvision ResNet-50 conv1..layer3).
//
// Both use the same 128 x (16*TN) x 16 register-tiled main loop: 256 threads,
// 8 x TN accumulators per thread, K-slices staged through shared memory
// (transposed on the store so fragment reads are 128-bit and conflict free),
// global loads of slice k+1 in flight while slice k is multiplied.
// The tcgen05 tensor-core engine (gemm_tc.cu) replaces these where TF32 is allowed.

#include "common.cuh"

namespace rf {

constexpr int BM = 128;          // rows (A feature vectors / output pixels) per tile
constexpr int BK = 16;           // K slice
constexpr int LDS_A = BM + 4;    // padded leading dimension of the transposed A slice

// ---------------------------------------------------------------------------
// shared main-loop pieces
// ---------------------------------------------------------------------------
template <int TN>
struct Frag {
    float acc[8][TN];
};

template <int TN>
__device__ __forceinline__ void mma_slice(const float* __restrict__ sA, const float* __restrict__ sB, int ldb,
                                          int ty, int tx, Frag<TN>& f) {
    // sA[k][m] (ld LDS_A), sB[k][n] (ld ldb).  Thread rows: ty*4..+3 and 64+ty*4..+3; cols: tx*4.. (and BN/2+tx*4.. if TN==8)
#pragma unroll
    for (int k = 0; k < BK; ++k) {
        float a[8], b[TN];
        float4 a0 = *reinterpret_cast<const float4*>(sA + k * LDS_A + ty * 4);
        float4 a1 = *reinterpret_cast<const float4*>(sA + k * LDS_A + 64 + ty * 4);
        a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
        float4 b0 = *reinterpret_cast<const float4*>(sB + k * ldb + tx * 4);
        b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w;
        if (TN == 8) {
            float4 b1 = *reinterpret_cast<const float4*>(sB + k * ldb + 64 + tx * 4);
            b[4 % TN] = b1.x; b[5 % TN] = b1.y; b[6 % TN] = b1.z; b[7 % TN] = b1.w;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < TN; ++j) f.acc[i][j] = fmaf(a[i], b[j], f.acc[i][j]);
    }
}

// transposed store of one float4 (4 consecutive k of one row m) into sT[k][m]
__device__ __forceinline__ void store_T(float* sT, int ld, int k4, int m, float4 v) {
    sT[(k4 + 0) * ld + m] = v.x;
    sT[(k4 + 1) * ld + m] = v.y;
    sT[(k4 + 2) * ld + m] = v.z;
    sT[(k4 + 3) * ld + m] = v.w;
}

// ---------------------------------------------------------------------------
// correlation + row/column arg-max
// ---------------------------------------------------------------------------
// grid: (ceil(NB/128), ceil(NA/128)); block 256.  rowbest[NA], colbest[NB]: packed keys, zero-initialised.
__global__ void __launch_bounds__(256, 2)
corr_argmax_kernel(const float* __restrict__ A, int NA, const float* __restrict__ B, int NB, int C,
                   unsigned long long* __restrict__ rowbest, unsigned long long* __restrict__ colbest) {
    __shared__ __align__(16) float sA[2][BK * LDS_A];
    __shared__ __align__(16) float sB[2][BK * LDS_A];
    __shared__ unsigned long long sCol[8][128];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ty = tid >> 4, tx = tid & 15;
    const int row0 = blockIdx.y * BM, col0 = blockIdx.x * 128;

    // loader mapping: 16 (row-group, k-quad) combos per operand, 2 per warp; lanes along rows
    float4 ra[2], rb[2];
    auto gload = [&](int k0) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            int combo = warp * 2 + q;
            int rg = combo >> 2, kq = combo & 3;
            int k = k0 + kq * 4;
            int ar = row0 + rg * 32 + lane, br = col0 + rg * 32 + lane;
            ra[q] = (ar < NA && k < C) ? __ldg(reinterpret_cast<const float4*>(A + (long long)ar * C + k)) : make_float4(0, 0, 0, 0);
            rb[q] = (br < NB && k < C) ? __ldg(reinterpret_cast<const float4*>(B + (long long)br * C + k)) : make_float4(0, 0, 0, 0);
        }
    };
    auto sstore = [&](int buf) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            int combo = warp * 2 + q;
            int rg = combo >> 2, kq = combo & 3;
            store_T(sA[buf], LDS_A, kq * 4, rg * 32 + lane, ra[q]);
            store_T(sB[buf], LDS_A, kq * 4, rg * 32 + lane, rb[q]);
        }
    };
    Frag<8> f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) f.acc[i][j] = 0.f;

    const int nk = (C + BK - 1) / BK;
    gload(0);
    sstore(0);
    __syncthreads();
    for (int kt = 0; kt < nk; ++kt) {
        int buf = kt & 1;
        if (kt + 1 < nk) gload((kt + 1) * BK);
        mma_slice<8>(sA[buf], sB[buf], LDS_A, ty, tx, f);
        if (kt + 1 < nk) sstore(buf ^ 1);
        __syncthreads();
    }

    // ---- epilogue: fused arg-max (utils/outil.py:36-37) ----
    int rows[8], cols[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) rows[i] = row0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
#pragma unroll
    for (int j = 0; j < 8; ++j) cols[j] = col0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
    // row max over this tile's 128 columns: thread-local, then across the 16 lanes sharing ty
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        unsigned long long best = 0ull;
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (cols[j] < NB) {
                unsigned long long k = pack_key(f.acc[i][j], (uint32_t)cols[j]);
                best = k > best ? k : best;
            }
#pragma unroll
        for (int d = 8; d >= 1; d >>= 1) {
            unsigned long long o = __shfl_xor_sync(0xffffffffu, best, d);
            best = o > best ? o : best;
        }
        if (tx == 0 && rows[i] < NA && best != 0ull) atomicMax(rowbest + rows[i], best);
    }
    // column max over this tile's 128 rows: thread-local, across the two ty of a warp, then across warps via smem
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        unsigned long long best = 0ull;
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (rows[i] < NA) {
                unsigned long long k = pack_key(f.acc[i][j], (uint32_t)rows[i]);
                best = k > best ? k : best;
            }
        unsigned long long o = __shfl_xor_sync(0xffffffffu, best, 16);
        best = o > best ? o : best;
        if (lane < 16) sCol[warp][(j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4))] = best;
    }
    __syncthreads();
    if (tid < 128) {
        unsigned long long best = 0ull;
#pragma unroll
        for (int w = 0; w < 8; ++w) { unsigned long long o = sCol[w][tid]; best = o > best ? o : best; }
        if (col0 + tid < NB && best != 0ull) atomicMax(colbest + col0 + tid, best);
    }
}

// mutual test (utils/outil.py:38-42), fully parallel: rowbest[i] is overwritten with (1 << 63 | j) when (i, j) is a
// mutual nearest-neighbour pair with non-zero score, else 0
__global__ void mutual_flag_kernel(unsigned long long* __restrict__ rowbest, const unsigned long long* __restrict__ colbest, int NA) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= NA) return;
    unsigned long long rk = rowbest[i], out = 0ull;
    if (rk != 0ull) {
        uint32_t j = key_index(rk);
        float v = key_value(rk);
        unsigned long long ck = __ldg(colbest + j);
        if (key_index(ck) == (uint32_t)i && (__fmul_rn(v, v) > 0.f)) out = (1ull << 63) | (unsigned long long)j;     // keepMax > 0
    }
    rowbest[i] = out;
}

// single CTA: order-preserving compaction of the flagged rows (utils/outil.py:43-44: nonzero() is row-major)
__global__ void __launch_bounds__(1024)
mutual_compact_kernel(const unsigned long long* __restrict__ flagged, int NA, long long* __restrict__ idx1, long long* __restrict__ idx2,
                      int* __restrict__ count) {
    __shared__ int s_scan[32];
    __shared__ int s_off;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_off = 0;
    __syncthreads();
    for (int base = 0; base < NA; base += 1024) {
        int i = base + tid;
        unsigned long long f = (i < NA) ? flagged[i] : 0ull;
        int keep = (f >> 63) ? 1 : 0;
        int incl = keep;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        if (lane == 31) s_scan[warp] = incl;
        __syncthreads();
        int wofs = 0, total = 0;
        for (int w = 0; w < 32; ++w) { int v = s_scan[w]; if (w < warp) wofs += v; total += v; }
        int off = s_off;
        if (keep) {
            int o = off + wofs + incl - 1;
            idx1[o] = i;
            idx2[o] = (long long)(f & 0xFFFFFFFFull);
        }
        __syncthreads();
        if (tid == 0) s_off = off + total;
        __syncthreads();
    }
    if (tid == 0) *count = s_off;
}

// mutual test + order-preserving compaction in ONE single-CTA kernel (the two kernels above fused; used behind the
// persistent correlation kernel).  Warp w owns a contiguous block of rows; pass 1 counts its mutual pairs with coalesced
// loads and ballots, the 32 warp totals are scanned, pass 2 recomputes the flags (L1 / L2 hits) and writes the pairs in
// row order.  rowbest / colbest are left untouched.
__device__ __forceinline__ bool mutual_pair(const unsigned long long* __restrict__ rowbest, const unsigned long long* __restrict__ colbest,
                                            int i, int NA, uint32_t& j) {
    if (i >= NA) return false;
    const unsigned long long rk = __ldg(rowbest + i);
    if (rk == 0ull) return false;
    j = key_index(rk);
    const float v = key_value(rk);
    const unsigned long long ck = __ldg(colbest + j);
    return key_index(ck) == (uint32_t)i && (__fmul_rn(v, v) > 0.f);              // keepMax > 0 (utils/outil.py:41-42)
}

__global__ void __launch_bounds__(1024)
mutual_flag_compact_kernel(const unsigned long long* __restrict__ rowbest, const unsigned long long* __restrict__ colbest, int NA,
                           long long* __restrict__ idx1, long long* __restrict__ idx2, int* __restrict__ count) {
    __shared__ int s_cnt[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int chunk = (((NA + 31) / 32) + 31) / 32 * 32;          // rows per warp, a multiple of 32
    const int begin = warp * chunk;
    int cnt = 0;
#pragma unroll 4
    for (int b = 0; b < chunk; b += 32) {
        uint32_t j = 0;
        const bool f = mutual_pair(rowbest, colbest, begin + b + lane, NA, j);
        cnt += __popc(__ballot_sync(0xffffffffu, f));
    }
    if (lane == 0) s_cnt[warp] = cnt;
    __syncthreads();
    int off = 0, total = 0;
    for (int w = 0; w < 32; ++w) { const int v = s_cnt[w]; off += (w < warp) ? v : 0; total += v; }
#pragma unroll 4
    for (int b = 0; b < chunk; b += 32) {
        uint32_t j = 0;
        const int i = begin + b + lane;
        const bool f = mutual_pair(rowbest, colbest, i, NA, j);
        const uint32_t bal = __ballot_sync(0xffffffffu, f);
        if (f) {
            const int o = off + __popc(bal & ((1u << lane) - 1u));
            idx1[o] = i;
            idx2[o] = (long long)j;
        }
        off += __popc(bal);
    }
    if (tid == 0) *count = total;
}

// Column-driven form of the kernel above: a mutual pair is one per COLUMN at most (<= NB of them), so the dependent
// rowbest[i] -> colbest[j] chain is walked for the NB columns only (one or two independent loads per thread); the matches
// are scattered into a row-indexed table in shared memory and compacted from there in row order (= the reference's
// nonzero() order, utils/outil.py:43) with ballots.  dynamic smem: NA ints.  ~3 us instead of ~12 us at config 2.
__global__ void __launch_bounds__(1024)
mutual_cols_compact_kernel(const unsigned long long* __restrict__ rowbest, const unsigned long long* __restrict__ colbest, int NA, int NB,
                           long long* __restrict__ idx1, long long* __restrict__ idx2, int* __restrict__ count) {
    extern __shared__ int sRow[];                 // 0 = unmatched row, j + 1 = matched with column j
    __shared__ int s_cnt[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < NA; i += 1024) sRow[i] = 0;
    __syncthreads();
    for (int j = tid; j < NB; j += 1024) {
        const unsigned long long ck = __ldg(colbest + j);
        if (ck == 0ull) continue;
        const uint32_t i = key_index(ck);
        if (i >= (uint32_t)NA) continue;
        const unsigned long long rk = __ldg(rowbest + i);
        const float v = key_value(rk);
        if (rk != 0ull && key_index(rk) == (uint32_t)j && (__fmul_rn(v, v) > 0.f)) sRow[i] = j + 1;     // keepMax > 0 (utils/outil.py:41-42)
    }
    __syncthreads();
    const int chunk = (((NA + 31) / 32) + 31) / 32 * 32;          // rows per warp, a multiple of 32
    const int begin = warp * chunk;
    int cnt = 0;
    for (int b = 0; b < chunk; b += 32) {
        const int i = begin + b + lane;
        cnt += __popc(__ballot_sync(0xffffffffu, i < NA && sRow[i] != 0));
    }
    if (lane == 0) s_cnt[warp] = cnt;
    __syncthreads();
    int off = 0, total = 0;
    for (int w = 0; w < 32; ++w) { const int v = s_cnt[w]; off += (w < warp) ? v : 0; total += v; }
    for (int b = 0; b < chunk; b += 32) {
        const int i = begin + b + lane;
        const int f = (i < NA) ? sRow[i] : 0;
        const uint32_t bal = __ballot_sync(0xffffffffu, f != 0);
        if (f) {
            const int o = off + __popc(bal & ((1u << lane) - 1u));
            idx1[o] = i;
            idx2[o] = (long long)(f - 1);
        }
        off += __popc(bal);
    }
    if (tid == 0) *count = total;
}

static int launch_mutual_compact(const unsigned long long* rowbest, const unsigned long long* colbest, int NA, int NB, long long* idx1, long long* idx2,
                                 int* count, cudaStream_t st) {
    const size_t smem = (size_t)NA * sizeof(int);
    if (smem <= 200 * 1024) {                                      // the row table fits in shared memory: column-driven compaction
        static bool attr[64] = {false};
        const int dev = current_device();
        if (!attr[dev]) {
            RF_CUDA(cudaFuncSetAttribute(mutual_cols_compact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            attr[dev] = true;
        }
        mutual_cols_compact_kernel<<<1, 1024, smem, st>>>(rowbest, colbest, NA, NB, idx1, idx2, count);
    } else {
        mutual_flag_compact_kernel<<<1, 1024, 0, st>>>(rowbest, colbest, NA, idx1, idx2, count);
    }
    RF_LAUNCHED();
    return 0;
}

// ---------------------------------------------------------------------------
// implicit-GEMM convolution
// ---------------------------------------------------------------------------

// TN = 8: tile 128 x 128; TN = 4: tile 128 x 64.  VEC: Cin % 16 == 0 (a K slice never straddles a tap).
template <int TN, bool VEC>
__global__ void __launch_bounds__(256, 2)
conv_kernel(const __grid_constant__ ImgSet set, const ConvParams p) {
    constexpr int BN = 16 * TN;
    constexpr int LDB = BN + 4;
    __shared__ __align__(16) float sA[2][BK * LDS_A];
    __shared__ __align__(16) float sB[2][BK * LDB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ty = tid >> 4, tx = tid & 15;
    const long long m0 = (long long)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;

    // ---- per-thread pixel bookkeeping for the A loader: rows lane + 32*rg ----
    // VEC: 16 (rg, kq) combos, 2 per warp -> this thread touches 2 (pixel, k-quad) pairs per slice.
    // !VEC: thread loads 8 scalars: row = tid & 127, k = (tid >> 7) + 2*e.
    constexpr int NPIX = VEC ? 2 : 1;
    int pimg[NPIX], poy[NPIX], pox[NPIX];
    bool pok[NPIX];
#pragma unroll
    for (int q = 0; q < NPIX; ++q) {
        int r = VEC ? (((warp * 2 + q) >> 2) * 32 + lane) : (tid & 127);
        long long pm = m0 + r;
        pok[q] = pm < p.Mtot;
        int im = 0, oy = 0, ox = 0;
        if (pok[q]) {
            im = find_img(set, pm);
            int local = (int)(pm - set.out_pix[im]);
            oy = local / set.Wo[im];
            ox = local - oy * set.Wo[im];
        }
        pimg[q] = im; poy[q] = oy; pox[q] = ox;
    }

    float4 ra[2];
    float ras[8];
    float4 rb[TN == 8 ? 2 : 1];
    auto gload = [&](int k0) {
        if (VEC) {
            int tap = k0 / p.Cin;
            int c0 = k0 - tap * p.Cin;
            int r = tap / p.S, s = tap - r * p.S;
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                int kq = (warp * 2 + q) & 3;
                float4 v = make_float4(0, 0, 0, 0);
                if (pok[q]) {
                    int im = pimg[q];
                    int iy = poy[q] * p.stride - p.pad + r, ix = pox[q] * p.stride - p.pad + s;
                    if (iy >= 0 && iy < set.H[im] && ix >= 0 && ix < set.W[im])
                        v = __ldg(reinterpret_cast<const float4*>(p.x + (set.in_pix[im] + (long long)iy * set.W[im] + ix) * p.Cin + c0 + kq * 4));
                }
                ra[q] = v;
            }
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                int k = k0 + (tid >> 7) + 2 * e;
                float v = 0.f;
                if (pok[0] && k < p.K) {
                    int tap = k / p.Cin;
                    int c = k - tap * p.Cin;
                    int r = tap / p.S, s = tap - r * p.S;
                    int im = pimg[0];
                    int iy = poy[0] * p.stride - p.pad + r, ix = pox[0] * p.stride - p.pad + s;
                    if (iy >= 0 && iy < set.H[im] && ix >= 0 && ix < set.W[im])
                        v = __ldg(p.x + (set.in_pix[im] + (long long)iy * set.W[im] + ix) * p.Cin + c);
                }
                ras[e] = v;
            }
        }
        // B slice: BK rows x BN cols, float4 along Cout when aligned
#pragma unroll
        for (int q = 0; q < (TN == 8 ? 2 : 1); ++q) {
            int f4 = tid + q * 256;                 // float4 index in the slice: BK * BN/4 of them
            int kr = f4 / (BN / 4), c4 = (f4 - kr * (BN / 4)) * 4;
            int k = k0 + kr, n = n0 + c4;
            float4 v = make_float4(0, 0, 0, 0);
            if (k < p.K) {
                const float* src = p.w + (long long)k * p.Cout + n;
                if (((p.Cout & 3) == 0) && n + 3 < p.Cout) v = __ldg(reinterpret_cast<const float4*>(src));
                else {
                    if (n + 0 < p.Cout) v.x = __ldg(src + 0);
                    if (n + 1 < p.Cout) v.y = __ldg(src + 1);
                    if (n + 2 < p.Cout) v.z = __ldg(src + 2);
                    if (n + 3 < p.Cout) v.w = __ldg(src + 3);
                }
            }
            rb[q] = v;
        }
    };
    auto sstore = [&](int buf) {
        if (VEC) {
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                int combo = warp * 2 + q;
                store_T(sA[buf], LDS_A, (combo & 3) * 4, (combo >> 2) * 32 + lane, ra[q]);
            }
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) sA[buf][((tid >> 7) + 2 * e) * LDS_A + (tid & 127)] = ras[e];
        }
#pragma unroll
        for (int q = 0; q < (TN == 8 ? 2 : 1); ++q) {
            int f4 = tid + q * 256;
            int kr = f4 / (BN / 4), c4 = (f4 - kr * (BN / 4)) * 4;
            *reinterpret_cast<float4*>(&sB[buf][kr * LDB + c4]) = rb[q];
        }
    };

    Frag<TN> f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) f.acc[i][j] = 0.f;

    const int nk = (p.K + BK - 1) / BK;
    gload(0);
    sstore(0);
    __syncthreads();
    for (int kt = 0; kt < nk; ++kt) {
        int buf = kt & 1;
        if (kt + 1 < nk) gload((kt + 1) * BK);
        // B fragment columns: tx*4 (+ 64 + tx*4 for TN == 8)
        mma_slice<TN>(sA[buf], sB[buf], LDB, ty, tx, f);
        if (kt + 1 < nk) sstore(buf ^ 1);
        __syncthreads();
    }

    // ---- epilogue: + bias (folded BN), + residual, ReLU ----
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        long long pm = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (pm >= p.Mtot) continue;
#pragma unroll
        for (int h = 0; h < TN / 4; ++h) {
            int n = n0 + h * 64 + tx * 4;
            if (n >= p.Cout) continue;
            float v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = f.acc[i][h * 4 + j];
            long long o = pm * p.Cout + n;
            if (((p.Cout & 3) == 0) && n + 3 < p.Cout) {
                if (p.bias) {
                    float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + n));
                    v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w;
                }
                if (p.residual) {
                    float4 r = __ldg(reinterpret_cast<const float4*>(p.residual + o));
                    v[0] += r.x; v[1] += r.y; v[2] += r.z; v[3] += r.w;
                }
                if (p.relu) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[j] = fmaxf(v[j], 0.f);
                }
                if (p.round_out) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[j] = round_tf32(v[j]);
                }
                *reinterpret_cast<float4*>(p.y + o) = make_float4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (n + j < p.Cout) {
                        float t = v[j];
                        if (p.bias) t += __ldg(p.bias + n + j);
                        if (p.residual) t += __ldg(p.residual + o + j);
                        if (p.relu) t = fmaxf(t, 0.f);
                        if (p.round_out) t = round_tf32(t);
                        p.y[o + j] = t;
                    }
                }
            }
        }
    }
}

}  // namespace rf

using namespace rf;

// tensor-core engines live in gemm_tc.cu
int rf_corr_argmax_tc(const float* featA, int NA, const float* featB, int NB, int C,
                      unsigned long long* rowbest, unsigned long long* colbest, void* ws, cudaStream_t st, int precision,
                      const void* const* presplit = nullptr);
size_t rf_corr_tc_workspace(int NA, int NB, int C);
int rf_conv2d_tc(const ImgSet& set, const ConvParams& p, const void* w_tc, cudaStream_t st, bool f16, bool out32);
bool rf_conv2d_tc_supported(const ConvParams& p);
int rf_conv2d_split(const ImgSet& set, const ConvParams& p, const void* w_split, cudaStream_t st, bool out32);

static size_t keys_bytes(int NA, int NB) {
    return (((size_t)(NA > 0 ? NA : 0) + (size_t)(NB > 0 ? NB : 0)) * sizeof(unsigned long long) + 255) / 256 * 256;
}

extern "C" size_t rf_corr_mutual_nn_workspace(int NA, int NB, int C, int precision) {
    size_t b = keys_bytes(NA, NB) + 256;
    if (precision == 1 || precision == 2) b += rf_corr_tc_workspace(NA > 0 ? NA : 0, NB > 0 ? NB : 0, C);
    return b;
}

extern "C" int rf_corr_mutual_nn_launches(int precision) {
    if (precision == 2) return 3;                                    // split+zero, persistent correlation, flag+compact
    return precision == 0 ? 4 : 6;                                   // memset, [split, split,] correlation, flag, compact
}

extern "C" int rf_corr_mutual_nn(const float* featA, int NA, const float* featB, int NB, int C,
                                 int64_t* idx1_out, int64_t* idx2_out, int* count_out,
                                 void* ws, size_t ws_bytes, int precision, void* stream) {
    RF_REQUIRE(NA >= 0 && NB >= 0 && C > 0 && (C % 4) == 0, "rf_corr_mutual_nn: bad sizes (C must be a multiple of 4)");
    RF_REQUIRE(ws != nullptr && ws_bytes >= rf_corr_mutual_nn_workspace(NA, NB, C, precision), "rf_corr_mutual_nn: workspace too small");
    RF_REQUIRE(((uintptr_t)featA % 16) == 0 && ((uintptr_t)featB % 16) == 0, "rf_corr_mutual_nn: features must be 16-byte aligned");
    cudaStream_t st = as_stream(stream);
    unsigned long long* rowbest = reinterpret_cast<unsigned long long*>(ws);
    unsigned long long* colbest = rowbest + NA;
    // precision 2: persistent correlation kernel; its split launch zeroes the keys, and the mutual test and the compaction
    // are one kernel.  Empty inputs take the memset / flag / compact path below (count 0).
    const bool pipe = precision == 2 && NA > 0 && NB > 0;
    if (!pipe) RF_CUDA(cudaMemsetAsync(ws, 0, ((size_t)NA + NB) * sizeof(unsigned long long), st));
    if (NA > 0 && NB > 0) {
        RF_REQUIRE(precision >= 0 && precision <= 2, "rf_corr_mutual_nn: precision is 0 (fp32 SIMT), 1 (3xTF32) or 2 (fp16 split)");
        if (precision >= 1) {
            int rc = rf_corr_argmax_tc(featA, NA, featB, NB, C, rowbest, colbest, static_cast<unsigned char*>(ws) + keys_bytes(NA, NB), st, precision);
            if (rc) return rc;
        } else {
            dim3 grid((NB + 127) / 128, (NA + BM - 1) / BM);
            corr_argmax_kernel<<<grid, 256, 0, st>>>(featA, NA, featB, NB, C, rowbest, colbest);
            RF_LAUNCHED();
        }
    }
    if (pipe) return launch_mutual_compact(rowbest, colbest, NA, NB, (long long*)idx1_out, (long long*)idx2_out, count_out, st);
    if (NA > 0) {
        mutual_flag_kernel<<<(NA + 255) / 256, 256, 0, st>>>(rowbest, colbest, NA);
        RF_LAUNCHED();
    }
    mutual_compact_kernel<<<1, 1024, 0, st>>>(rowbest, NA, (long long*)idx1_out, (long long*)idx2_out, count_out);
    RF_LAUNCHED();
    return 0;
}

// utils/outil.py:32-45 with operands the producer already split (rf_l2norm_split_nhwc: hi = fp16(x), lo = fp16((x - hi) * 2^11)):
// memset of the keys, the persistent fp16-split correlation kernel, the column-driven compaction.  ws: (NA + NB) keys.
extern "C" size_t rf_corr_mutual_nn_presplit_workspace(int NA, int NB) { return keys_bytes(NA, NB) + 256; }

extern "C" int rf_corr_mutual_nn_presplit(const void* A_hi, const void* A_lo, int NA, const void* B_hi, const void* B_lo, int NB, int C,
                                          int64_t* idx1_out, int64_t* idx2_out, int* count_out, void* ws, size_t ws_bytes, void* stream) {
    RF_REQUIRE(NA >= 0 && NB >= 0 && C > 0 && (C % 64) == 0, "rf_corr_mutual_nn_presplit: bad sizes (C must be a multiple of 64)");
    RF_REQUIRE(ws != nullptr && ws_bytes >= rf_corr_mutual_nn_presplit_workspace(NA, NB), "rf_corr_mutual_nn_presplit: workspace too small");
    cudaStream_t st = as_stream(stream);
    unsigned long long* rowbest = reinterpret_cast<unsigned long long*>(ws);
    unsigned long long* colbest = rowbest + NA;
    RF_CUDA(cudaMemsetAsync(ws, 0, ((size_t)NA + NB) * sizeof(unsigned long long), st));
    if (NA == 0 || NB == 0) {
        RF_CUDA(cudaMemsetAsync(count_out, 0, sizeof(int), st));
        return 0;
    }
    const void* planes[4] = {A_hi, A_lo, B_hi, B_lo};
    int rc = rf_corr_argmax_tc(nullptr, NA, nullptr, NB, C, rowbest, colbest, nullptr, st, 2, planes);
    if (rc) return rc;
    return launch_mutual_compact(rowbest, colbest, NA, NB, (long long*)idx1_out, (long long*)idx2_out, count_out, st);
}

extern "C" int rf_conv2d_nhwc(const float* x, int nimg, const int* hw_host, int Cin,
                              const float* w, const float* w_tc, const float* bias, const float* residual,
                              int Cout, int R, int S, int stride, int pad, int relu, int engine,
                              float* y, void* stream) {
    RF_REQUIRE(R == S && R >= 1 && stride >= 1 && pad >= 0 && Cin >= 1 && Cout >= 1, "rf_conv2d_nhwc: bad conv geometry");
    ImgSet set;
    RF_REQUIRE(make_imgset(set, nimg, hw_host, R, stride, pad) == 0, "rf_conv2d_nhwc: bad image set");
    ConvParams p;
    p.x = x; p.w = w; p.bias = bias; p.residual = residual; p.y = y;
    p.Cin = Cin; p.Cout = Cout; p.R = R; p.S = S; p.stride = stride; p.pad = pad; p.relu = relu;
    p.Mtot = set.out_pix[nimg];
    p.K = R * S * Cin;
    // tensor-core engine: ReLU'd activations are the next conv's MMA operand; store them rounded to nearest TF32
    // (the MMA truncates), which removes the truncation bias.  The fp32 engine never rounds.
    p.round_out = ((engine == RF_ENGINE_TF32 || engine == RF_ENGINE_F16_OUT32) && relu) ? 1 : 0;
    cudaStream_t st = as_stream(stream);
    RF_REQUIRE(engine >= RF_ENGINE_FP32 && engine <= RF_ENGINE_SPLIT_OUT32, "rf_conv2d_nhwc: unknown engine");
    // engine 2 = tcgen05 with fp16 activations and weights (x, residual, y, w_tc hold IEEE halves); no SIMT fallback.
    // engine 3 = the same with an fp32 (TF32-rounded after ReLU) output: the hand-over to a TF32 layer
    if (engine == RF_ENGINE_F16) return rf_conv2d_tc(set, p, w_tc, st, true, false);
    if (engine == RF_ENGINE_F16_OUT32) return rf_conv2d_tc(set, p, w_tc, st, true, true);
    // engine 4 = tcgen05 with fp16 hi / lo split operands (fp32-grade, gemm_split.cu): x, residual, y are split tensors
    // ([2][P][C] fp16), w_tc = [2][Cout][K] fp16.  engine 5 = the same with an fp32 [P][Cout] output (no residual)
    if (engine == RF_ENGINE_SPLIT) return rf_conv2d_split(set, p, w_tc, st, false);
    if (engine == RF_ENGINE_SPLIT_OUT32) return rf_conv2d_split(set, p, w_tc, st, true);
    // engine 1 = tcgen05 TF32 where the layer shape allows it (stride 1, Cin % 32 == 0); other layers
    // (3-channel stems, stride-2 convs, 49-channel heads) run on the exact-fp32 SIMT engine below
    if (engine == 1 && w_tc != nullptr && rf_conv2d_tc_supported(p)) return rf_conv2d_tc(set, p, w_tc, st, false, false);
    RF_REQUIRE(((uintptr_t)x % 16) == 0 && ((uintptr_t)w % 16) == 0 && ((uintptr_t)y % 16) == 0, "rf_conv2d_nhwc: pointers must be 16-byte aligned");
    const bool vec = (Cin % 16) == 0;
    const bool wide = Cout >= 128;
    unsigned gx = (unsigned)((p.Mtot + BM - 1) / BM);
    if (wide) {
        dim3 grid(gx, (Cout + 127) / 128);
        if (vec) conv_kernel<8, true><<<grid, 256, 0, st>>>(set, p);
        else conv_kernel<8, false><<<grid, 256, 0, st>>>(set, p);
    } else {
        dim3 grid(gx, (Cout + 63) / 64);
        if (vec) conv_kernel<4, true><<<grid, 256, 0, st>>>(set, p);
        else conv_kernel<4, false><<<grid, 256, 0, st>>>(set, p);
    }
    RF_LAUNCHED();
    return 0;
}
