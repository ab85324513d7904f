// Score-map loss of a supervised call (nets/pips.py:58-90 score_map_loss + :14-37 balanced_ce_loss, on the score maps
// of :502-511) without the dense score maps.
//
// Bilinear interpolation with align_corners=True is linear, so the reference's score map of track (b,s,n) at the start
// of an iteration,
//     fcp[y,x] = sum_l interpolate_l( <f, F_l> / sqrt(C) ),      f = ffeats[b,n,s]
// equals <f, Gr[b*S+s, y, x, :]> with Gr = sum_l interpolate(F_l -> H8 x W8) / sqrt(C), a channels-last map of the size
// of pyramid level 0.  Gr is built once per forward (score_grid_kernel); the score maps of one iteration are then one
// GEMM per frame (M = the frame's queries, N = its H8*W8 pixels, K = 128), and the loss needs two numbers per
// (track, iteration): the sum of softplus(fcp) over every pixel but the target g, and fcp[g].  The GEMM epilogue
// (score_loss_kernel) emits exactly those; no score map is stored.  The fp64 finalize turns them into the scalar
//     ce = sum_pos softplus(-fcp[g]) / (1e-6 + K*I) + sum_neg softplus(fcp) / (1e-6 + K*I*(H8*W8 - 1)).
//
// The GEMM runs on tcgen05 with bf16x3 operands (hi*hi + lo*hi + hi*lo, fp32 accumulation): |fcp| reaches ~50, where
// a plain bf16 product is off by ~0.1.
#include "ptx.cuh"
#include "common.cuh"

namespace pips {
namespace {

constexpr int C = PIPS_C;
constexpr int L = PIPS_LEVELS;
constexpr int SBM = 128;                          // queries per tile (MMA M; one epilogue thread per row)
constexpr int SBN = PIPS_SCORE_TILE;              // pixels per tile (MMA N), 256
constexpr int SBK = 64;                           // one 128-byte swizzle row of bf16
constexpr int SUB = 128;                          // pixels per partial (one epilogue warp's half of a tile)
constexpr int THREADS = 384;                      // warp 0 TMA, warp 1 MMA, warp 2 TMEM, warps 4..11 epilogue
constexpr int EPI_THREADS = 256;
constexpr uint32_t A_PART = SBM * SBK * 2;        // 16 KB: one (hi|lo, kb) slice of the A tile
constexpr uint32_t A_BYTES = 4 * A_PART;          // hi kb0, hi kb1, lo kb0, lo kb1
constexpr uint32_t B_PART = SBN * SBK * 2;        // 32 KB
constexpr uint32_t STAGE_BYTES = 2 * B_PART;      // hi + lo of one K-block of the pixel tile
constexpr int STAGES = 2;
constexpr uint32_t SMEM_BYTES = 1024 + A_BYTES + STAGES * STAGE_BYTES + 256;
constexpr float SCALE = 0.08838834764831845f;     // 1 / sqrt(128), nets/pips.py:396

__host__ __device__ inline int padded_pixels(int H8, int W8) { return (H8 * W8 + SBN - 1) / SBN * SBN; }

struct GridLevels {
    const float* lvl[L];
    int H[L], W[L];
};

// Gr[f, p, c] = (sum_l interpolate(F_l)[f, p, c]) / sqrt(C) as a (hi, lo) bf16 pair: hi plane (frames, Ppad, 128), then
// the lo plane.  Rows p in [H8*W8, Ppad) are zero.  ATen's upsample_bilinear2d index arithmetic (as heat_upsample_kernel):
// src = dst * (in-1)/(out-1), i0 = (int)src, second tap i0 + (i0 < in-1); the levels are added in the order 0, 1, 2, 3.
__global__ void __launch_bounds__(256) score_grid_kernel(GridLevels lv, int frames, int H8, int W8, int Ppad,
                                                         __nv_bfloat16* __restrict__ grid) {
    const size_t total = static_cast<size_t>(frames) * Ppad * (C / 4);
    const size_t plane = static_cast<size_t>(frames) * Ppad * C;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int c4 = static_cast<int>(i % (C / 4));
        const size_t fp = i / (C / 4);
        const int p = static_cast<int>(fp % Ppad);
        const size_t f = fp / Ppad;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p < H8 * W8) {
            const int y = p / W8, x = p - y * W8;
            acc = reinterpret_cast<const float4*>(lv.lvl[0] + (f * H8 * W8 + p) * C)[c4];      // level 0: exact copy
#pragma unroll
            for (int l = 1; l < L; ++l) {
                const int h = lv.H[l], w = lv.W[l];
                const float sy = H8 > 1 ? static_cast<float>(h - 1) / static_cast<float>(H8 - 1) : 0.0f;
                const float sx = W8 > 1 ? static_cast<float>(w - 1) / static_cast<float>(W8 - 1) : 0.0f;
                const float fy = sy * y, fx = sx * x;
                const int y0 = static_cast<int>(fy), x0 = static_cast<int>(fx);
                const int yp = y0 < h - 1 ? 1 : 0, xp = x0 < w - 1 ? 1 : 0;
                const float ly = fy - y0, lx = fx - x0;
                const float hy = 1.0f - ly, hx = 1.0f - lx;
                const float4* m = reinterpret_cast<const float4*>(lv.lvl[l] + f * h * w * C);
                const float4 v00 = m[(y0 * w + x0) * (C / 4) + c4], v01 = m[(y0 * w + x0 + xp) * (C / 4) + c4];
                const float4 v10 = m[((y0 + yp) * w + x0) * (C / 4) + c4], v11 = m[((y0 + yp) * w + x0 + xp) * (C / 4) + c4];
                acc.x += hy * (hx * v00.x + lx * v01.x) + ly * (hx * v10.x + lx * v11.x);
                acc.y += hy * (hx * v00.y + lx * v01.y) + ly * (hx * v10.y + lx * v11.y);
                acc.z += hy * (hx * v00.z + lx * v01.z) + ly * (hx * v10.z + lx * v11.z);
                acc.w += hy * (hx * v00.w + lx * v01.w) + ly * (hx * v10.w + lx * v11.w);
            }
            acc.x *= SCALE; acc.y *= SCALE; acc.z *= SCALE; acc.w *= SCALE;
        }
        const uint32_t h01 = cvt_bf16x2(acc.x, acc.y), h23 = cvt_bf16x2(acc.z, acc.w);
        const uint32_t l01 = cvt_bf16x2(acc.x - __uint_as_float(h01 << 16), acc.y - __uint_as_float(h01 & 0xffff0000u));
        const uint32_t l23 = cvt_bf16x2(acc.z - __uint_as_float(h23 << 16), acc.w - __uint_as_float(h23 & 0xffff0000u));
        const size_t o = fp * C + c4 * 4;
        *reinterpret_cast<uint2*>(grid + o) = make_uint2(h01, h23);
        *reinterpret_cast<uint2*>(grid + plane + o) = make_uint2(l01, l23);
    }
}

struct LossArgs {
    const float* ffeats;          // (B*nc, S, 128) of this call's particles
    const int* target;            // (B, S, n_total): pixel index y*W8 + x, or -1
    float* neg;                   // [iter][tile128][rows]
    float* pos;                   // [iter][rows]
    int S, nc, n_offset, n_total, rows;
    int P, Ppad, frames, mtiles, ptiles, pchunk_tiles, pchunks, units, iter;
};

__device__ __forceinline__ float ex2_approx(float v) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float lg2_approx(float v) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}

// Persistent over work units (frame, 128-query tile, run of pixel tiles).  The A tile (the frame's queries, fp32 ffeats
// split into hi/lo) is written into shared memory by the epilogue warps in the 128-byte-swizzled K-major layout TMA would
// produce; the pixel tiles of Gr stream through a 2-stage TMA ring; the accumulator is double-buffered in TMEM.
__global__ void __launch_bounds__(THREADS, 1) score_loss_kernel(const __grid_constant__ CUtensorMap map_g, const LossArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint8_t* a_tile = smem;
    uint8_t* ring = smem + A_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + STAGES * STAGE_BYTES);
    // barriers: full[STAGES], empty[STAGES], tfull[2], tempty[2], a_full, a_empty
    const uint32_t full0 = smem_u32(bars);
    const uint32_t empty0 = full0 + 8 * STAGES;
    const uint32_t tfull0 = empty0 + 8 * STAGES;
    const uint32_t tempty0 = tfull0 + 16;
    const uint32_t a_full = tempty0 + 16;
    const uint32_t a_empty = a_full + 8;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 6);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) tma_prefetch_desc(&map_g);
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full0 + 8 * s, 1);
            mbar_init(empty0 + 8 * s, 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(tfull0 + 8 * s, 1);
            mbar_init(tempty0 + 8 * s, EPI_THREADS);
        }
        mbar_init(a_full, EPI_THREADS);
        mbar_init(a_empty, 1);
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc(smem_u32(tmem_slot), 512);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer (pixel tiles of Gr, hi and lo)
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int u = blockIdx.x; u < a.units; u += gridDim.x) {
                const int pc = u % a.pchunks;
                const int f = u / (a.pchunks * a.mtiles);
                const int t0 = pc * a.pchunk_tiles;
                const int t1 = min(a.ptiles, t0 + a.pchunk_tiles);
                for (int t = t0; t < t1; ++t) {
                    const int grow = f * a.Ppad + t * SBN;
                    for (int kb = 0; kb < C / SBK; ++kb) {
                        mbar_wait(empty0 + 8 * stage, phase ^ 1);
                        const uint32_t fb = full0 + 8 * stage;
                        mbar_arrive_expect_tx(fb, STAGE_BYTES);
                        const uint32_t base = smem_u32(ring + stage * STAGE_BYTES);
                        tma_load_2d(base, &map_g, fb, kb * SBK, grow);
                        tma_load_2d(base + B_PART, &map_g, fb, kb * SBK, a.frames * a.Ppad + grow);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer: whole warp, one elected lane issues
        const bool elected = elect_one();
        constexpr uint32_t idesc = umma_idesc_bf16(SBM, SBN);
        uint32_t stage = 0, phase = 0;
        int it = 0, ui = 0;
        for (int u = blockIdx.x; u < a.units; u += gridDim.x, ++ui) {
            const int pc = u % a.pchunks;
            const int t0 = pc * a.pchunk_tiles;
            const int t1 = min(a.ptiles, t0 + a.pchunk_tiles);
            mbar_wait(a_full, ui & 1);                          // the epilogue warps have written this unit's A tile
            tc_fence_after();
            const uint32_t abase = smem_u32(a_tile);
            for (int t = t0; t < t1; ++t, ++it) {
                const uint32_t as = it & 1, aphase = (it >> 1) & 1;
                mbar_wait(tempty0 + 8 * as, aphase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + as * SBN;
                for (int kb = 0; kb < C / SBK; ++kb) {
                    mbar_wait(full0 + 8 * stage, phase);
                    tc_fence_after();
                    const uint32_t base = smem_u32(ring + stage * STAGE_BYTES);
                    const uint64_t a_hi = umma_desc_sw128(abase + kb * A_PART);
                    const uint64_t a_lo = umma_desc_sw128(abase + (2 + kb) * A_PART);
                    const uint64_t b_hi = umma_desc_sw128(base);
                    const uint64_t b_lo = umma_desc_sw128(base + B_PART);
#pragma unroll
                    for (int k = 0; k < SBK / 16; ++k) {
                        const uint64_t adv = static_cast<uint64_t>((k * 16 * 2) >> 4);
                        if (elected) umma_f16(d_tmem, a_hi + adv, b_hi + adv, idesc, (kb | k) != 0);
                        if (elected) umma_f16(d_tmem, a_lo + adv, b_hi + adv, idesc, 1);
                        if (elected) umma_f16(d_tmem, a_hi + adv, b_lo + adv, idesc, 1);
                    }
                    if (elected) umma_commit(empty0 + 8 * stage);
                    if (elected && kb == C / SBK - 1) umma_commit(tfull0 + 8 * as);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
            if (elected) umma_commit(a_empty);                  // A tile reusable once this unit's MMAs retire
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ------------------------------------------------------------ A loader + epilogue (256 threads)
        const int et = threadIdx.x - 128;
        const int q = warp & 3;                                 // TMEM lane quadrant of this warp
        const int half = (warp - 4) >> 2;                       // which 128 pixels of the 256-pixel tile
        int it = 0, ui = 0;
        for (int u = blockIdx.x; u < a.units; u += gridDim.x, ++ui) {
            const int pc = u % a.pchunks;
            const int mt = (u / a.pchunks) % a.mtiles;
            const int f = u / (a.pchunks * a.mtiles);
            const int b = f / a.S, s = f - b * a.S;
            const int m0 = mt * SBM;
            const int t0 = pc * a.pchunk_tiles;
            const int t1 = min(a.ptiles, t0 + a.pchunk_tiles);

            mbar_wait(a_empty, (ui & 1) ^ 1);                   // the previous unit's MMAs are done with the A tile
            for (int i = et; i < SBM * (C / 8); i += EPI_THREADS) {
                const int r = i >> 4, c8 = i & 15;              // row, 8-channel (16-byte bf16) piece
                const int n = m0 + r;
                float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
                if (n < a.nc) {
                    const float4* src = reinterpret_cast<const float4*>(a.ffeats + ((static_cast<size_t>(b) * a.nc + n) * a.S + s) * C + c8 * 8);
                    v0 = src[0];
                    v1 = src[1];
                }
                const float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
                uint32_t hw[4], lw[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    hw[e] = cvt_bf16x2(v[2 * e], v[2 * e + 1]);
                    lw[e] = cvt_bf16x2(v[2 * e] - __uint_as_float(hw[e] << 16), v[2 * e + 1] - __uint_as_float(hw[e] & 0xffff0000u));
                }
                const int kb = c8 >> 3, piece = c8 & 7;
                const uint32_t off = kb * A_PART + (r >> 3) * 1024 + (r & 7) * 128 + ((piece ^ (r & 7)) << 4);
                *reinterpret_cast<uint4*>(a_tile + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
                *reinterpret_cast<uint4*>(a_tile + 2 * A_PART + off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
            }
            fence_proxy_async_smem();                           // generic-proxy smem writes -> visible to tcgen05.mma
            mbar_arrive(a_full);

            const int n = m0 + q * 32 + lane;
            const int row = f * a.n_total + a.n_offset + n;     // (b, s, n) in the caller's full particle range
            int g = n < a.nc ? __ldg(a.target + row) : -1;
            if (g >= a.P) g = -1;                               // not a pixel: excluded (as in the finalize)
            const bool warp_active = __any_sync(0xffffffffu, g >= 0);   // rows without a target skip the softplus work
            for (int t = t0; t < t1; ++t, ++it) {
                const uint32_t as = it & 1, aphase = (it >> 1) & 1;
                mbar_wait(tfull0 + 8 * as, aphase);
                tc_fence_after();
                if (warp_active) {
                    const uint32_t taddr = tmem_base + as * SBN + half * SUB + (static_cast<uint32_t>(q * 32) << 16);
                    const int col0 = t * SBN + half * SUB;
                    const int gl = g - col0;                    // target column inside this half tile (may be outside)
                    const int lim = a.P - col0;                 // valid columns
                    float smax = 0.f, slog = 0.f, vg = 0.f;
#pragma unroll 1
                    for (int c = 0; c < SUB; c += 64) {
                        uint32_t va[32], vb[32];
                        tmem_ld_32x32(taddr + c, va);
                        tmem_ld_32x32(taddr + c + 32, vb);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 64; ++j) {
                            const float v = __uint_as_float(j < 32 ? va[j] : vb[j - 32]);
                            // softplus(v) = max(v, 0) + log(1 + exp(-|v|)), the log taken in base 2 and scaled once
                            const float l = lg2_approx(1.0f + ex2_approx(fabsf(v) * -1.4426950408889634f));
                            const int col = c + j;
                            const bool ok = col < lim && col != gl;
                            smax += ok ? fmaxf(v, 0.f) : 0.f;
                            slog += ok ? l : 0.f;
                            vg = col == gl ? v : vg;
                        }
                    }
                    if (g >= 0) {
                        a.neg[(static_cast<size_t>(a.iter) * (a.Ppad / SUB) + col0 / SUB) * a.rows + row] =
                            fmaf(slog, 0.6931471805599453f, smax);
                        if (gl >= 0 && gl < SUB) a.pos[static_cast<size_t>(a.iter) * a.rows + row] = vg;
                    }
                }
                tc_fence_before();
                mbar_arrive(tempty0 + 8 * as);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, 512);
}

constexpr int FIN_ROWS = 1024;                    // rows per finalize block: fixes the reduction tree
constexpr int FIN_THREADS = 256;

__device__ __forceinline__ double softplus_d(double v) { return fmax(v, 0.0) + log1p(exp(-fabs(v))); }

// fixed-order block reduction of three fp64 values
__device__ void block_sum3(double (&v)[3], double (*sh)[FIN_THREADS]) {
    for (int k = 0; k < 3; ++k) sh[k][threadIdx.x] = v[k];
    __syncthreads();
    for (int o = FIN_THREADS / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o)
            for (int k = 0; k < 3; ++k) sh[k][threadIdx.x] += sh[k][threadIdx.x + o];
        __syncthreads();
    }
    for (int k = 0; k < 3; ++k) v[k] = sh[k][0];
}

// per block of FIN_ROWS rows: (sum of negative terms, sum of positive terms, kept rows) in fp64
__global__ void __launch_bounds__(FIN_THREADS) score_finalize_rows(const int* __restrict__ target, int rows, int iters,
                                                                   int P, int tiles, const float* __restrict__ neg,
                                                                   const float* __restrict__ pos, double* __restrict__ out) {
    __shared__ double sh[3][FIN_THREADS];
    double v[3] = {0.0, 0.0, 0.0};
    for (int j = 0; j < FIN_ROWS / FIN_THREADS; ++j) {
        const int r = blockIdx.x * FIN_ROWS + j * FIN_THREADS + threadIdx.x;
        if (r >= rows || target[r] < 0 || target[r] >= P) continue;
        v[2] += 1.0;
        for (int i = 0; i < iters; ++i) {
            v[1] += softplus_d(-static_cast<double>(pos[static_cast<size_t>(i) * rows + r]));
            for (int t = 0; t < tiles; ++t) v[0] += neg[(static_cast<size_t>(i) * tiles + t) * rows + r];
        }
    }
    block_sum3(v, sh);
    if (threadIdx.x == 0)
        for (int k = 0; k < 3; ++k) out[blockIdx.x * 3 + k] = v[k];
}

__global__ void __launch_bounds__(FIN_THREADS) score_finalize_total(const double* __restrict__ part, int blocks, int iters,
                                                                    int P, float* __restrict__ ce) {
    __shared__ double sh[3][FIN_THREADS];
    double v[3] = {0.0, 0.0, 0.0};
    for (int b = threadIdx.x; b < blocks; b += FIN_THREADS)
        for (int k = 0; k < 3; ++k) v[k] += part[b * 3 + k];
    block_sum3(v, sh);
    if (threadIdx.x == 0) {
        const double ki = v[2] * iters;                   // kept (track, iteration) pairs: one positive each
        ce[0] = static_cast<float>(v[1] / (1e-6 + ki) + v[0] / (1e-6 + ki * (P - 1.0)));
    }
}

size_t finalize_offset(int rows, int iters, int H8, int W8) {      // floats before the fp64 block partials
    const size_t tiles = padded_pixels(H8, W8) / SUB;
    const size_t n = static_cast<size_t>(iters) * rows * (tiles + 1);
    return (n + 1) / 2 * 2;
}

}  // namespace
}  // namespace pips

using namespace pips;

extern "C" int pips_score_grid(const float* const* lvl_f32, int frames, int H8, int W8, void* grid, void* stream) {
    if (!lvl_f32 || !grid) return fail("pips_score_grid: null pointer");
    if (frames <= 0) return fail("pips_score_grid: empty problem");
    if ((H8 >> (L - 1)) < 1 || (W8 >> (L - 1)) < 1) return fail("pips_score_grid: feature map too small for 4 levels");
    GridLevels lv;
    int h = H8, w = W8;
    for (int l = 0; l < L; ++l) {
        if (!lvl_f32[l]) return fail("pips_score_grid: null pyramid level");
        lv.lvl[l] = lvl_f32[l];
        lv.H[l] = h;
        lv.W[l] = w;
        h /= 2;
        w /= 2;
    }
    const int Ppad = padded_pixels(H8, W8);
    const size_t total = static_cast<size_t>(frames) * Ppad * (C / 4);
    const size_t blocks = (total + 255) / 256;
    const size_t cap = static_cast<size_t>(sm_count()) * 16;
    score_grid_kernel<<<static_cast<unsigned>(blocks < cap ? blocks : cap), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        lv, frames, H8, W8, Ppad, static_cast<__nv_bfloat16*>(grid));
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail_cuda("pips_score_grid", e);
}

extern "C" size_t pips_score_loss_scratch_floats(int rows, int iters, int H8, int W8) {
    if (rows <= 0 || iters <= 0 || H8 <= 0 || W8 <= 0) return 0;
    const size_t blocks = (static_cast<size_t>(rows) + FIN_ROWS - 1) / FIN_ROWS;
    return finalize_offset(rows, iters, H8, W8) + 2 * 3 * blocks;
}

extern "C" int pips_score_loss(const void* grid, int B, int S, int N, int H8, int W8, const float* ffeats, const int* target,
                               int n_offset, int n_total, int iter, int iters, float* partial, void* stream) {
    if (!grid || !ffeats || !target || !partial) return fail("pips_score_loss: null pointer");
    if (B <= 0 || S <= 0 || N <= 0 || H8 <= 0 || W8 <= 0 || iters <= 0) return fail("pips_score_loss: empty problem");
    if (n_offset < 0 || n_offset + N > n_total) return fail("pips_score_loss: particle slice outside n_total");
    if (iter < 0 || iter >= iters) return fail("pips_score_loss: iteration outside [0, iters)");
    const long long rows_ll = static_cast<long long>(B) * S * n_total;
    if (rows_ll > (1LL << 31) - 1 || static_cast<long long>(B) * S * padded_pixels(H8, W8) * 2 > (1LL << 31) - 1)
        return fail("pips_score_loss: problem too large for 32-bit indexing");
    LossArgs a;
    a.ffeats = ffeats;
    a.target = target;
    a.rows = static_cast<int>(rows_ll);
    a.neg = partial;
    a.Ppad = padded_pixels(H8, W8);
    a.pos = partial + static_cast<size_t>(iters) * (a.Ppad / SUB) * a.rows;
    a.S = S; a.nc = N; a.n_offset = n_offset; a.n_total = n_total;
    a.P = H8 * W8;
    a.frames = B * S;
    a.mtiles = (N + SBM - 1) / SBM;
    a.ptiles = a.Ppad / SBN;
    a.iter = iter;
    // split each frame's pixel tiles into runs so that every SM gets a work unit; which CTA computes a (row, tile)
    // partial does not change its value
    const int sms = sm_count();
    const int per_frame = a.frames * a.mtiles;
    int want = (sms + per_frame - 1) / per_frame;
    if (want > a.ptiles) want = a.ptiles;
    a.pchunk_tiles = (a.ptiles + want - 1) / want;
    a.pchunks = (a.ptiles + a.pchunk_tiles - 1) / a.pchunk_tiles;
    a.units = per_frame * a.pchunks;

    CUtensorMap map;
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(2) * a.frames * a.Ppad};
    cuuint64_t gstride[1] = {static_cast<cuuint64_t>(C) * 2};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(SBK), static_cast<cuuint32_t>(SBN)};
    cuuint32_t estr[2] = {1, 1};
    if (!encode_tiled(&map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(grid), gdim, gstride, box, estr,
                      CU_TENSOR_MAP_SWIZZLE_128B))
        return fail("pips_score_loss: tensor map failed");
    static bool attr[kMaxDevices] = {};
    cudaError_t e = ensure_dyn_smem(score_loss_kernel, attr, SMEM_BYTES);
    if (e != cudaSuccess) return fail_cuda("pips_score_loss: smem attribute", e);
    const int grid_x = a.units < sms ? a.units : sms;
    score_loss_kernel<<<grid_x, THREADS, SMEM_BYTES, static_cast<cudaStream_t>(stream)>>>(map, a);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail_cuda("pips_score_loss", e);
}

extern "C" int pips_score_loss_finalize(const int* target, int rows, int iters, int H8, int W8, float* partial, float* ce,
                                        void* stream) {
    if (!target || !partial || !ce) return fail("pips_score_loss_finalize: null pointer");
    if (rows <= 0 || iters <= 0 || H8 <= 0 || W8 <= 0) return fail("pips_score_loss_finalize: empty problem");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int tiles = padded_pixels(H8, W8) / SUB;
    const int blocks = (rows + FIN_ROWS - 1) / FIN_ROWS;
    double* part = reinterpret_cast<double*>(partial + finalize_offset(rows, iters, H8, W8));
    score_finalize_rows<<<blocks, FIN_THREADS, 0, st>>>(target, rows, iters, H8 * W8, tiles, partial,
                                                        partial + static_cast<size_t>(iters) * tiles * rows, part);
    score_finalize_total<<<1, FIN_THREADS, 0, st>>>(part, blocks, iters, H8 * W8, ce);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail_cuda("pips_score_loss_finalize", e);
}
