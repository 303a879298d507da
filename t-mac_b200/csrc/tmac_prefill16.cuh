// tmac_prefill16.cuh -- the prefill tile of the fp path (N >= 64): both scales folded into fp16 operands, fp32 accumulation over the
// whole K in TMEM, stream-K over the SMs when there are fewer tiles than SMs.
//
//   C[m][n] = sum_{g,e} (0.5*scale[m][wg(g)] * S[m][g][e]) * (lut_scale[n][ag(g)] * T8[n][g][e])            (main term)
//           + sum_wg (0.5*scale[m][wg] + zero[m][wg]) * (lut_bias[n][2wg] + lut_bias[n][2wg+1])            (bias term)
//
// The int8 tile (tmac_prefill.cuh) keeps the reference's integer sums exact but has to drain and rescale the accumulator
// after every activation group (256 cycles of MMA against ~2800 CUDA-core warp-instructions per step).  Here both factors
// ride in the operands: A = fp16(0.5*s*S) is expanded by the producers from the packed codes, B = fp16(ls*T8) is laid out
// once per call by lut_tile16_kernel, the accumulator lives in TMEM for the whole K and is read once.  The bias term is one
// more contraction step with exact operands: A columns (0.5s, 0.5s, z, z) against B columns (LBhi, LBlo, LBhi, LBlo), LB
// split into two fp16 so that their sum carries 22 bits.  Both operands are normalised per token and per row by powers of two
// (see p16_exp below), so fp16's range never clips them.  Operand rounding (2^-11 per entry) keeps every output within
// 2.5e-4 x sum_k |x_k| |W_mk| of the CPU kernel -- NOT inside the 2e-5 the exact paths hold, so this tile has its own
// tolerance and never serves the int32 (BitNet) path.
//
// Tile: 128 weight rows x 256 tokens per CTA, tcgen05.mma kind::f16 (M 128, N 256, K 16), 8 MMAs per activation group.
//   warps 0..15 : producers (thread = weight row x 4 of the step's 16 groups): code byte -> 8 unit fp16 from a 256-entry
//                 table, x (0.5*s) by HMUL2, one 16-byte store into the K-major canonical A tile; afterwards the epilogue.
//   warp  16    : MMA issuer; tcgen05.commit releases the stage, the last commit publishes the accumulator.
//   warp  17    : TMA issuer: one 64 KB bulk copy (the B tile of the step) per step.
// Supported: W2 (PB 2), chunk 128, act group 64, per-row scales (+ zero points), symmetric LUT -- as the int8 tile.
#pragma once
#include "tmac_prefill.cuh"

namespace tmac_b200 {

constexpr int kP16NT = 256;                          // tokens per CTA (MMA N)
constexpr int kP16ABytes = 128 * 128 * 2;            // A tile: 128 rows x 128 contraction entries, fp16
constexpr int kP16BBytes = kP16NT * 128 * 2;         // B tile: 256 tokens x 128 entries, fp16 = one record
constexpr int kP16SubA = kP16ABytes, kP16SubB = kP16BBytes;   // the pipeline moves whole steps: 16 K-groups = 8 MMAs
constexpr int kP16NA = 2, kP16NB = 2;                // ring depths.  (Measured at N = 256: half-step rings 3 x 16 KB + 5 x 32 KB: 110 us; TMA multicast
                                                     // of B over CTA pairs: 101 us; stream-K over all SMs: 121 us; this: 102 us.)
constexpr int kP16ProdWarps = 16, kP16WarpMma = 16, kP16WarpTma = 17;
constexpr int kP16Threads = 18 * 32;

struct Prefill16Params {
    const unsigned char *W;
    void *C;
    int N, K, Mout, ldc, out_f16;
    int nchunk, zp, sd, blk_bytes;
    int nmain, nextra;                               // activation-group steps, bias steps (128 columns = 32 weight groups each)
    size_t rsb_stride;
    const unsigned char *tiles;                      // lut_tile16_kernel output: [token tile][nmain + nextra][kP16BBytes]
    int nrsb, ntiles, streamk;                       // row super-blocks, tiles = nrsb * token tiles, stream-K split (see the kernel)
    float *scratch;                                  // [grid][256 tokens][128 rows] fp32 partial tiles (stream-K)
    int *flags;                                      // [grid] partial tile ready
    const int *texp;                                 // [N] token exponents e_n (p16_token_exp_kernel)
    const int *rexp;                                 // [nrsb * 128] row exponents f_m (p16_row_exp, computed at upload)
};

// Range handling.  fp16 holds 2^-14 .. 65504 at full precision, the inputs do not come in that range: a token's LUT biases
// reach 128 x its activations (inf past 65504), small scales or activations fall into fp16's subnormals.  So both operands are
// normalised by exact powers of two: token n's B entries and biases by 2^-e_n (its largest entry lands in [2^14, 2^15)), row
// m's 0.5*scale and zero by 2^-f_m (largest in [2^13, 2^14), so that the A entry 3 * 0.5*scale stays below 65504); the
// epilogue multiplies by 2^(e_n + f_m).  Scaling a token or a row by 2^k then shifts e_n or f_m by k and leaves every operand
// bit unchanged: the tile's output scales by exactly 2^k, as the exact paths' does.  Exponents are clamped to +-64 so that every
// factor 2^e is an fp32 normal and the epilogue's val * 2^e_n * 2^f_m is exact (|val| < 2^47 after normalisation); the clamp
// binds only for token or row magnitudes beyond 2^+-49.
__host__ __device__ inline int p16_exp(float m, int top) {   // e with m * 2^-e in [2^(top-1), 2^top); 0 for 0, inf, NaN
    if (!(m > 0.f) || m > 3.4e38f) return 0;
    int e;
    frexpf(m, &e);
    return e - top < -64 ? -64 : (e - top > 64 ? 64 : e - top);
}

__device__ __forceinline__ float p16_pow2(int e) { return __int_as_float((e + 127) << 23); }   // 2^e, -126 <= e <= 127

inline int p16_row_exp(const float *scales, const float *zeros, int ng) {     // f_m of one row: ng groups
    float m = 0.f;
    for (int g = 0; g < ng; ++g) {
        m = std::max(m, 0.5f * std::fabs(scales[g]));
        if (zeros) m = std::max(m, std::fabs(zeros[g]));
    }
    return p16_exp(m, 14);
}

// e_n of every token: one warp per token scans its K/64 LUT scales and K/128 bias pairs (the same sums lut_tile16_kernel forms).
__global__ void __launch_bounds__(256) p16_token_exp_kernel(const float *ls, const float *lb, int *texp, int N, int nag) {
    const int n = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    pdl_wait();                                      // ls / lb: the preprocessor (or the caller's work) before this launch
    pdl_launch_dependents();                         // lut_tile16_kernel loads its LUT entries meanwhile, then waits for texp
    if (n >= N) return;
    const float *l = ls + (size_t)n * nag, *b = lb + (size_t)n * nag;
    float m = 0.f;
    for (int i = lane; i < nag; i += 32) m = fmaxf(m, 128.f * fabsf(l[i]));
    for (int i = lane; i < nag / 2; i += 32) m = fmaxf(m, fabsf(b[2 * i] + b[2 * i + 1]));
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) texp[n] = p16_exp(m, 15);
}

__device__ __forceinline__ uint64_t p16_desc(uint32_t saddr, uint32_t lbo) {
    uint64_t d = (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)(lbo >> 4) << 16;                 // byte distance between the two 16-byte K chunks of one MMA
    d |= (uint64_t)(128u >> 4) << 32;                // 8-row groups are 128 B apart
    d |= (uint64_t)1 << 46;
    return d;
}

// B tiles.  grid = (nmain + nextra, token tiles of 256), block = 256 (thread = token).
//   step < nmain : entries (lut_scale[n][step] * 2^-e_n * T8[n][16*step + g][e]) as fp16, token t, group g at ((g*32 + t/8)*128 + (t%8)*16)
//   bias steps   : column 4*wg + {0,1,2,3} = {LBhi, LBlo, LBhi, LBlo}, LB = (lut_bias[n][2wg] + lut_bias[n][2wg+1]) * 2^-e_n; 8 columns per chunk
__global__ void __launch_bounds__(256) lut_tile16_kernel(const int8_t *qlut, const float *ls, const float *lb, const int *texp, unsigned char *out,
                                                         int N, int K, int nmain, int nextra) {
    const int step = blockIdx.x, tile = blockIdx.y, t = threadIdx.x, n = tile * kP16NT + t;
    const int nag = K / 64, nwg = K / 128;
    unsigned char *rec = out + ((size_t)tile * (nmain + nextra) + step) * kP16BBytes;
    if (step < nmain) {
        const uint2 *src = reinterpret_cast<const uint2 *>(qlut) + ((size_t)n * (K / 4) + (size_t)step * 16) * 2;
        uint2 q[16];
        float l = 0.f;
#pragma unroll
        for (int g = 0; g < 16; ++g) q[g] = (n < N) ? __ldg(src + g * 2) : make_uint2(0, 0);   // the 8 stored entries of each group
        if (n < N) l = ls[(size_t)n * nag + step];
        pdl_wait();                                  // texp: p16_token_exp_kernel, launched just before as the primary grid
        if (n < N) l *= p16_pow2(-texp[n]);
#pragma unroll
        for (int g = 0; g < 16; ++g) {
            uint32_t o[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t word = k < 2 ? q[g].x : q[g].y;
                const float a = (float)(int)(int8_t)((word >> (16 * (k & 1))) & 0xff) * l;
                const float b = (float)(int)(int8_t)((word >> (16 * (k & 1) + 8)) & 0xff) * l;
                const __half2 h = __floats2half2_rn(a, b);
                o[k] = *reinterpret_cast<const uint32_t *>(&h);
            }
            *reinterpret_cast<uint4 *>(rec + ((size_t)(g * 32 + (t >> 3)) * 128 + (t & 7) * 16)) = make_uint4(o[0], o[1], o[2], o[3]);
        }
    } else {
        const int e = step - nmain;                  // bias step: weight groups 32e .. 32e+31, two per 16-byte chunk
        pdl_wait();
        const float sn = p16_pow2((n < N) ? -texp[n] : 0);
#pragma unroll
        for (int kc = 0; kc < 16; ++kc) {
            uint32_t o[4];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int wg = e * 32 + kc * 2 + u;
                float LB = 0.f;
                if (n < N && wg < nwg) LB = (lb[(size_t)n * nag + 2 * wg] + lb[(size_t)n * nag + 2 * wg + 1]) * sn;
                const __half hi = __float2half_rn(LB);
                const __half lo = __float2half_rn(LB - __half2float(hi));
                const __half2 h = __halves2half2(hi, lo);
                o[2 * u] = o[2 * u + 1] = *reinterpret_cast<const uint32_t *>(&h);
            }
            *reinterpret_cast<uint4 *>(rec + ((size_t)(kc * 32 + (t >> 3)) * 128 + (t & 7) * 16)) = make_uint4(o[0], o[1], o[2], o[3]);
        }
    }
}

// One CTA walks a contiguous run [L0, L1) of the linear (tile, step) sequence -- tile = (row super-block, token tile), nsteps
// contraction steps per tile.  streamk == 0: L0 = cta * nsteps, one whole tile per CTA (grid = tiles).  streamk == 1: grid = SMs,
// [L0, L1) = [S*cta/G, S*(cta+1)/G): at most the tail of one tile and the head of the next (two TMEM accumulators); a tile cut by
// CTA boundaries is finished by the CTA that holds its LAST step, the others store their fp32 partial tile to `scratch[cta]` and
// raise `flags[cta]`; the finisher adds the partials in ascending K order (deterministic), stores C and clears the flags.
//
// Pipeline.  A (16 producer warps) and B (TMA, 64 KB per step) have their own 2-deep rings; each step's 8 MMAs release one slot
// of each.
__global__ void __launch_bounds__(kP16Threads, 1) prefill16_w2_kernel(const Prefill16Params p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char *sA = smem;                                              // [NA][16 KB]
    unsigned char *sB = sA + kP16NA * kP16SubA;                            // [NB][32 KB]
    unsigned char *raw = sB + kP16NB * kP16SubB;                           // [2][blk] packed block (codes + scales)
    const int rawsz = (p.blk_bytes + 127) & ~127;
    uint64_t *bars = reinterpret_cast<uint64_t *>(raw + 2 * rawsz);
    uint64_t *fullA = bars, *emptyA = fullA + kP16NA, *fullB = emptyA + kP16NA, *emptyB = fullB + kP16NB, *accfull = emptyB + kP16NB;   // accfull[2]
    __shared__ uint32_t tmem_base_s;
    __shared__ float tok_scale[2][kP16NT];                                  // 2^e_n of each fragment's tokens (epilogue)

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nsteps = p.nmain + p.nextra;
    const int G = gridDim.x, cta = blockIdx.x;
    const long long Stot = (long long)p.ntiles * nsteps;
    const int L0 = p.streamk ? (int)(Stot * cta / G) : cta * nsteps, L1 = p.streamk ? (int)(Stot * (cta + 1) / G) : (cta + 1) * nsteps;
    // fragments: f = 0 -> [L0, min(L1, end of L0's tile)), f = 1 -> the rest (head of the next tile)
    int ft[2], fs0[2], fs1[2], nfrag = 0;
    for (int L = L0; L < L1 && nfrag < 2;) {
        const int t = L / nsteps, s0 = L - t * nsteps, s1 = min(nsteps, s0 + (L1 - L));
        ft[nfrag] = t; fs0[nfrag] = s0; fs1[nfrag] = s1; ++nfrag;
        L += s1 - s0;
    }

    if (tid == 0) {
        for (int i = 0; i < kP16NA; ++i) { pf_mbar_init(fullA + i, kP16ProdWarps); pf_mbar_init(emptyA + i, 1); }
        for (int i = 0; i < kP16NB; ++i) { pf_mbar_init(fullB + i, 1); pf_mbar_init(emptyB + i, 1); }
        pf_mbar_init(accfull, 1); pf_mbar_init(accfull + 1, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kP16WarpMma) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(pf_s32(&tmem_base_s)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;

    if (warp < kP16ProdWarps) {
        // ======================= A producers: thread = (weight row, 4 of the step's 16 K-groups) =======================
        const int r = tid & 127, gq = tid >> 7;
        const int wl = r >> 2, wi = r & 3;           // lane / row-in-lane of the stream layout (RW = 4)
        const int n16 = p.blk_bytes >> 4;
        int it = 0;                                  // running step counter over both fragments
        for (int f = 0; f < nfrag; ++f) {
            const int rsb = ft[f] % p.nrsb;
            const unsigned char *rsb_base = p.W + (size_t)rsb * p.rsb_stride;
            const int f_m = p.rexp[rsb * 128 + r];
            const float zsc = p16_pow2(-f_m), hsc = 0.5f * zsc;           // z * 2^-f_m, 0.5 * scale * 2^-f_m: exact
            const int s0 = fs0[f], s1m = min(fs1[f], p.nmain);
            if (s0 < s1m) {
                const int c_first = s0 >> 1, c_last = (s1m - 1) >> 1;
                asm volatile("bar.sync 1, 512;" ::: "memory");             // the previous fragment's last block is dead
                for (int i = tid; i < n16; i += kP16ProdWarps * 32) cp_async16_plain(raw + (size_t)(c_first & 1) * rawsz + i * 16, rsb_base + (size_t)c_first * p.blk_bytes + i * 16);
                cp_async_commit();
                for (int c = c_first; c <= c_last; ++c) {
                    unsigned char *rb = raw + (size_t)(c & 1) * rawsz;
                    cp_async_wait_all();
                    asm volatile("bar.sync 1, 512;" ::: "memory");         // block c visible to all producers; block c-1 dead
                    if (c + 1 <= c_last) {
                        unsigned char *nb = raw + (size_t)((c + 1) & 1) * rawsz;
                        const unsigned char *src = rsb_base + (size_t)(c + 1) * p.blk_bytes;
                        for (int i = tid; i < n16; i += kP16ProdWarps * 32) cp_async16_plain(nb + i * 16, src + i * 16);
                        cp_async_commit();
                    }
                    const uint32_t *words = reinterpret_cast<const uint32_t *>(rb);
                    // the row's 8 A entries of one K-group: +-hs at entry j0 (plane 0) plus +-2hs at entry j1 (plane 1), hs = fp16(0.5 * scale),
                    // built in registers: (+-hs) + (+-2hs) is one fp16 rounding of the exact k * hs; hs = fp16(0.5 * scale * 2^-f_m)
                    const __half hsh = __float2half_rn(load_scale(rb + 4096, p.sd, wl * 4 + wi) * hsc);
                    const uint32_t c1 = __half_as_ushort(hsh), c2 = __half_as_ushort(__hadd(hsh, hsh));
                    const int u0 = (c == c_first) ? (s0 & 1) : 0, u1 = (c == c_last) ? ((s1m - 1) & 1) : 1;   // steps of this chunk
#pragma unroll 1
                    for (int u = u0; u <= u1; ++u, ++it) {
                        const int s = it % kP16NA;
                        pf_mbar_wait(emptyA + s, ((it / kP16NA) & 1) ^ 1);     // the MMAs that read this slot have completed
                        unsigned char *a_dst = sA + (size_t)s * kP16SubA;
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            const int gl = gq * 4 + kk;                        // group within the step = 16-byte chunk index
                            const int gqc = u * 16 + gl;                       // group within the chunk (0..31)
                            const int q = gqc >> 2, k = gqc & 3;
                            const uint32_t *w4 = words + ((size_t)q * 32 + wl) * 4;
                            const uint32_t jb = (w4[k] >> (8 * wi)) & 0x77u;                                   // j0 | j1 << 4
                            const uint32_t ng = (w4[2 * (k >> 1) + (wi >> 1)] >> (16 * (wi & 1) + 8 * (k & 1) + 3)) & 0x11u;   // neg0 | neg1 << 4
                            const uint32_t j0 = jb & 7u, j1 = jb >> 4;
                            const uint32_t v0 = (c1 ^ ((ng & 1u) << 15)) << ((j0 & 1u) * 16), v1 = (c2 ^ ((ng & 0x10u) << 11)) << ((j1 & 1u) * 16);
                            uint32_t o4[4];
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                const uint32_t a = (j0 >> 1) == (uint32_t)e ? v0 : 0u, b = (j1 >> 1) == (uint32_t)e ? v1 : 0u;
                                const __half2 x = __hadd2(*reinterpret_cast<const __half2 *>(&a), *reinterpret_cast<const __half2 *>(&b));
                                o4[e] = *reinterpret_cast<const uint32_t *>(&x);
                            }
                            *reinterpret_cast<uint4 *>(a_dst + ((size_t)(gl * 16 + (r >> 3)) * 128 + (r & 7) * 16)) = make_uint4(o4[0], o4[1], o4[2], o4[3]);
                        }
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) pf_mbar_arrive(fullA + s);
                        __syncwarp();
                    }
                }
            }
            // bias steps: A columns 4*wg + {0,1,2,3} = {0.5s, 0.5s, z, z} of weight group wg (= chunk index), 2 groups per 16-byte chunk
            for (int step = max(fs0[f], p.nmain); step < fs1[f]; ++step, ++it) {
                {
                    const int e = step - p.nmain, s = it % kP16NA;
                    pf_mbar_wait(emptyA + s, ((it / kP16NA) & 1) ^ 1);
                    unsigned char *a_dst = sA + (size_t)s * kP16SubA;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const int gl = gq * 4 + kk, kc = gl;
                        uint32_t o[4];
#pragma unroll
                        for (int u = 0; u < 2; ++u) {
                            const int wg = e * 32 + kc * 2 + u;
                            float hs = 0.f, zz = 0.f;
                            if (wg < p.nchunk) {
                                const unsigned char *sp = rsb_base + (size_t)wg * p.blk_bytes + 4096;
                                hs = load_scale(sp, p.sd, wl * 4 + wi) * hsc;
                                if (p.zp) zz = load_scale(sp + (size_t)128 * p.sd, p.sd, wl * 4 + wi) * zsc;
                            }
                            const __half2 a = __floats2half2_rn(hs, hs), b = __floats2half2_rn(zz, zz);
                            o[2 * u] = *reinterpret_cast<const uint32_t *>(&a); o[2 * u + 1] = *reinterpret_cast<const uint32_t *>(&b);
                        }
                        *reinterpret_cast<uint4 *>(a_dst + ((size_t)(gl * 16 + (r >> 3)) * 128 + (r & 7) * 16)) = make_uint4(o[0], o[1], o[2], o[3]);
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) pf_mbar_arrive(fullA + s);
                    __syncwarp();
                }
            }
        }
        // ======================= epilogue: thread = (weight row, 64-token column group) =======================
        // partial tiles first (another CTA waits for them), then the tile this CTA finishes
        const int lq = warp & 3, cg = warp >> 2;     // TMEM lane quarter of this warp, columns 64*cg .. 64*cg+63
        const int er = lq * 32 + lane;
        for (int i = tid; i < nfrag * kP16NT; i += kP16ProdWarps * 32) {
            const int fi = i / kP16NT, n = ((fi ? ft[1] : ft[0]) / p.nrsb) * kP16NT + i % kP16NT;   // (no dynamic index: ft stays in registers)
            tok_scale[fi][i % kP16NT] = p16_pow2(n < p.N ? p.texp[n] : 0);
        }
        asm volatile("bar.sync 1, 512;" ::: "memory");
        for (int pass = 0; pass < 2; ++pass)
            for (int f = 0; f < nfrag; ++f) {
                const bool whole = fs0[f] == 0 && fs1[f] == nsteps, last = fs1[f] == nsteps;
                if ((pass == 0) == last) continue;   // pass 0: fragments that do not hold the tile's last step
                const int rsb = ft[f] % p.nrsb, tile = ft[f] / p.nrsb, n0 = tile * kP16NT, ntok = min(kP16NT, p.N - n0);
                const int row = rsb * 128 + er, f_m = p.rexp[row];
                const float rf = p16_pow2(f_m);
                pf_mbar_wait(accfull + f, 0);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                int c_first = cta;
                if (last && !whole) {                // wait for the CTAs that hold steps [0, s0) of this tile
                    const long long lin0 = (long long)ft[f] * nsteps;
                    c_first = (int)(lin0 * G / Stot);
                    while ((int)(Stot * (c_first + 1) / G) <= lin0) ++c_first;
                    while ((int)(Stot * c_first / G) > lin0) --c_first;
                    if (tid == 0)
                        for (int c2 = c_first; c2 < cta; ++c2) {
                            int v, spins = 0;
                            do { asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p.flags + c2) : "memory"); } while (v == 0 && ++spins < (1 << 24));
                        }
                    asm volatile("bar.sync 1, 512;" ::: "memory");
                }
#pragma unroll 1
                for (int hh = 0; hh < 2; ++hh) {
                    uint32_t v[32];
                    PF_TMEM_LD32(v, tmem + ((uint32_t)(lq * 32) << 16) + f * 256 + cg * 64 + hh * 32);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int t = cg * 64 + hh * 32 + j;
                        float val = __uint_as_float(v[j]);
                        if (!last) {                 // partial tile -> scratch[cta][t][row]
                            p.scratch[((size_t)cta * kP16NT + t) * 128 + er] = val;
                            continue;
                        }
                        if (!whole) {
                            float acc = 0.f;         // ascending K order: earlier CTAs first, this CTA's part last
                            for (int c2 = c_first; c2 < cta; ++c2) acc += __ldcg(p.scratch + ((size_t)c2 * kP16NT + t) * 128 + er);
                            val = acc + val;
                        }
                        if (t < ntok && row < p.Mout) {
                            val = val * tok_scale[f][t] * rf;   // undo the normalisation (exact, see p16_exp)
                            const size_t o = (size_t)(n0 + t) * p.ldc + row;
                            if (p.out_f16) reinterpret_cast<__half *>(p.C)[o] = __float2half_rn(val);
                            else reinterpret_cast<float *>(p.C)[o] = val;
                        }
                    }
                }
                if (!last) {                         // publish: every thread's stores, then the flag
                    __threadfence();
                    asm volatile("bar.sync 1, 512;" ::: "memory");
                    if (tid == 0) asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p.flags + cta), "r"(1) : "memory");
                } else if (!whole) {
                    asm volatile("bar.sync 1, 512;" ::: "memory");             // all partial reads done: the flags can be reused by the next launch
                    if (tid == 0) for (int c2 = c_first; c2 < cta; ++c2) asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(p.flags + c2), "r"(0) : "memory");
                }
            }
    } else if (warp == kP16WarpTma) {
        if (lane == 0) {
            int it = 0;
            for (int f = 0; f < nfrag; ++f) {
                const unsigned char *src = p.tiles + (size_t)(ft[f] / p.nrsb) * nsteps * kP16BBytes;
                for (int u = fs0[f]; u < fs1[f]; ++u, ++it) {
                    const int s = it % kP16NB;
                    pf_mbar_wait(emptyB + s, ((it / kP16NB) & 1) ^ 1);
                    pf_expect_tx(fullB + s, kP16SubB);
                    pf_bulk_g2s(sB + (size_t)s * kP16SubB, src + (size_t)u * kP16SubB, kP16SubB, fullB + s);
                }
            }
        }
    } else if (warp == kP16WarpMma) {
        if (lane == 0) {
            // kind::f16: fp16 x fp16 -> fp32; instruction descriptor: D format F32 (1 << 4), A/B format F16 (0), N >> 3 at bit 17, M >> 4 at bit 24
            const uint32_t idesc = (1u << 4) | ((uint32_t)(kP16NT >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            int it = 0;
            for (int f = 0; f < nfrag; ++f) {
                for (int u = fs0[f]; u < fs1[f]; ++u, ++it) {
                    const int sa = it % kP16NA, sb = it % kP16NB;
                    pf_mbar_wait(fullA + sa, (it / kP16NA) & 1);
                    pf_mbar_wait(fullB + sb, (it / kP16NB) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a0 = pf_s32(sA + (size_t)sa * kP16SubA), b0 = pf_s32(sB + (size_t)sb * kP16SubB);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {    // K = 16 entries = two 16-byte chunks per MMA
                        const uint64_t da = p16_desc(a0 + i * 2 * 2048, 2048), db = p16_desc(b0 + i * 2 * 4096, 4096);
                        const uint32_t acc = (u > fs0[f] || i > 0) ? 1u : 0u;
                        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                                     ::"r"(tmem + f * 256), "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
                    }
                    pf_commit(emptyA + sa);          // both slots are free once these MMAs have read them
                    pf_commit(emptyB + sb);
                }
                pf_commit(accfull + f);              // all MMAs of the fragment complete: its accumulator may be read
            }
        }
    }
    __syncwarp();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == kP16WarpMma) {
        __syncwarp();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
    }
}

}  // namespace tmac_b200
