// K1t: PCM -> spectrum for 256-point frames (8 kHz telephone speech: 20-32 ms windows), the specialised front end of the
// general path.  Same arithmetic as the 512-point front end k_frames2 (rawIN::get_frame, src/io/in.cc:305-419:
// pre-emphasis, Hamming, mean of the windowed frame removed inside the window, real FFT, power, P[0] = 1e-10, optional
// square root), organised the same way -- registers, one shared-memory transpose between two passes -- for half the
// length:
//   256 real points = 128 complex = 16 x 8.  A GROUP OF 8 THREADS owns a frame (four frames per warp); thread g holds the
//   16 complex points z[8 n1 + g]: pass 1 is one 16-point DFT per thread over n1 (dft16, ctu_fft.cuh), the twiddle
//   W128^(g k1), a transpose through a padded exchange tile; pass 2 is two 8-point DFTs per thread (k1 = g and g + 8) over
//   the 8 threads' values; the real-input split reads Z[k] and Z[128 - k] from the tile and each thread finishes 17 of the
//   129 bins.
// The general kernel (k_frames_any: one WARP per frame, radix-4 passes in shared memory, a warp barrier per pass) needs
// 14.7 ms per 8 M frames for this step; see DESIGN 11 for what this one measures.
// Work unit: a tile of 16 consecutive frames of one utterance (the 16-frame tile list), 128 threads = 16 groups = one pass;
// persistent CTAs with the next tile's samples prefetched (cp.async), like k_frames2.
// The transform runs on packed FP32 instructions (ctu_fft.cuh); the windowing stays scalar: as 8-byte loads and packed
// multiplies (what k_frames2 does, with its window in registers) it measured 9.84 ms against 9.23 ms per 19.98 M frames
// (all scalar: 9.54 ms; tools/gpu_jobs/r2_job44.sh, r2_job45.sh).
#ifndef CTU_FRAMES256_CUH
#define CTU_FRAMES256_CUH

#include "ctu_kernels.cuh"

namespace ctu {

constexpr int F256_THREADS = 128;
constexpr int F256_TILE = 16;                 // frames per CTA = groups per CTA
constexpr int F256_M = 128;                   // complex points
constexpr int F256_XP = 9;                    // pitch (complex) of a row of the 16 x 8 exchange tile
constexpr int F256_GRP = 16 * F256_XP + 8;    // complex elements of a group's exchange tile: 144 (>= the 128 of the linear Z) + 8, so that
                                              // the two groups of a half warp start 16 banks apart

struct Tables256 {
    const float2 *tw128;     // [16][8]: W128^(g k1) at [k1 * 8 + g]
    const float2 *twsplit;   // -i/2 e^{-2 pi i k / 256}, k <= 128
    const float *win;        // analysis window [window]
};

// floats of the tile's pre-emphasised samples / of the raw int16 prefetch buffer (8-sample chunks, 16-byte phase kept)
__host__ __device__ inline int smem256_samples(int window, int wshift) { return ((F256_TILE - 1) * wshift + window + 7) & ~7; }
__host__ __device__ inline int smem256_raw(int window, int wshift) { return (((F256_TILE - 1) * wshift + window + 1 + 8 + 7) / 8) * 4; }
__host__ __device__ inline size_t smem256_floats(int window, int wshift) {
    return (size_t)2 * F256_TILE * F256_GRP + 2 * 128 + 2 * 130 + 256 + smem256_samples(window, wshift) + smem256_raw(window, wshift) +
           TILE_AHEAD_FLOATS;
}

// (dft8 and the index algebra of the 16 x 8 decomposition: ctu_fft.cuh, emulated on the CPU by tests/emu/emu_fft.cpp)
__device__ __forceinline__ float group_sum8(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v;
}

// five resident CTAs per SM (at most 96 registers, no spills); left to itself ptxas takes 117 registers, which leaves four
__global__ void __launch_bounds__(F256_THREADS, 5)
k_frames256(const __grid_constant__ FrameParams P, BatchDesc bd, Tables256 tb, const int16_t *__restrict__ pcm, float *__restrict__ dst, int nbins,
            int ntiles) {
    extern __shared__ __align__(16) float sm[];
    const int tid = threadIdx.x, g = tid & 7, grp = tid >> 3;
    const int w = P.window, s = P.wshift;
    cpx<float> *sX = reinterpret_cast<cpx<float> *>(sm);                                // [16 groups][F256_GRP]
    cpx<float> *sTw = sX + F256_TILE * F256_GRP;                                        // 128
    cpx<float> *sTs = sTw + 128;                                                        // 129 (+1)
    float *sW = reinterpret_cast<float *>(sTs + 130);                                   // 256
    float *sD = sW + 256;                                                               // the tile's pre-emphasised samples
    int16_t *raw = reinterpret_cast<int16_t *>(sD + smem256_samples(w, s));             // int16 prefetch buffer
    TileAhead *ahead = reinterpret_cast<TileAhead *>(sD + smem256_samples(w, s) + smem256_raw(w, s));
    // persistent CTAs: the next tile's PCM travels HBM -> shared memory (cp.async) while this one is transformed
    int tile = blockIdx.x;
    if (tile >= ntiles) return;
    TileMeta cur = load_tile_meta(bd, tile, s, F256_TILE);
    tile_ahead_init(ahead, bd, tile, ntiles);
    int edge = 0;
    prefetch_pcm<F256_THREADS>(raw, pcm, cur, (cur.nf - 1) * s + w + 1, edge);
    for (int i = tid; i < 128; i += F256_THREADS) sTw[i] = mk<float>(tb.tw128[i].x, tb.tw128[i].y);
    for (int i = tid; i < 129; i += F256_THREADS) sTs[i] = mk<float>(tb.twsplit[i].x, tb.twsplit[i].y);
    for (int i = tid; i < 256; i += F256_THREADS) sW[i] = (i < w) ? tb.win[i] : 0.f;
    cpx<float> *xch = sX + grp * F256_GRP;
#pragma unroll 1
    for (int j = 0; tile < ntiles; tile += gridDim.x, j ^= 1) {
    const int next = tile + gridDim.x;
    const int nf = cur.nf;
    finish_pcm<F256_THREADS>(raw, sD, pcm, cur, (nf - 1) * s + w + 1, edge, P.preem);   // pre-emphasis once per sample
    __syncthreads();                                       // samples (and, the first time, the tables) staged; raw is free again
    const TileMeta nxt = tile_ahead_next(ahead, j, bd, tile, ntiles, s, F256_TILE);   // used only when next < ntiles
    if (next < ntiles) prefetch_pcm<F256_THREADS>(raw, pcm, nxt, (nxt.nf - 1) * s + w + 1, edge);
    // a group past the end of the tile recomputes the tile's last frame and stores nothing (shuffles name the full warp)
    const bool store = grp < nf;
    const int f = min(grp, nf - 1);
    const float *d = sD + f * s;
    cpx<float> a[16];
    float sum = 0.f;
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++) {
        const int i0 = 16 * n1 + 2 * g;                    // complex point 8 n1 + g = real samples i0, i0 + 1
        const float y0 = (i0 < w) ? sW[i0] * d[i0] : 0.f;
        const float y1 = (i0 + 1 < w) ? sW[i0 + 1] * d[i0 + 1] : 0.f;
        a[n1] = mk<float>(y0, y1);
        sum += y0 + y1;
    }
    if (P.remove_dc) {
        // mean of the WINDOWED frame, subtracted from the window's samples only (src/io/in.cc:375-382)
        const float mean = group_sum8(sum) / (float)w;
#pragma unroll
        for (int n1 = 0; n1 < 16; n1++) {
            const int i0 = 16 * n1 + 2 * g;
            if (i0 < w) a[n1].x -= mean;
            if (i0 + 1 < w) a[n1].y -= mean;
        }
    }
    // pass 1: over n1; a[k1] = sum_n1 z[8 n1 + g] W16^(n1 k1), times W128^(g k1), to the tile at [k1][g]
    fft128_pass1(a, g, sTw, xch, F256_XP);
    __syncwarp();
    // pass 2: k1 = g and g + 8, over the 8 threads' values: Z[k1 + 16 k2]
    cpx<float> b0[8], b1[8];
    fft128_pass2(b0, b1, g, xch, F256_XP);
    __syncwarp();                                          // every read of the transposed tile is done: it becomes the linear Z
#pragma unroll
    for (int k2 = 0; k2 < 8; k2++) { xch[g + 16 * k2] = b0[k2]; xch[g + 8 + 16 * k2] = b1[k2]; }
    __syncwarp();
    // real-input split (X[k] = (Z[k] + conj Z[128-k]) / 2 + twsplit[k] (Z[k] - conj Z[128-k])), power / magnitude
    if (store) {
        float *grow = dst + (cur.row0 + f) * nbins;
#pragma unroll
        for (int j = 0; j < 17; j++) {
            const int k = g + 8 * j;
            if (k > F256_M) break;
            const cpx<float> X = rfft256_bin(xch, sTs, k);
            float p = X.x * X.x + X.y * X.y;
            if (k == 0 && P.remove_dc) p = 1e-10f;         // fixed floor (src/io/in.cc:390)
            grow[k] = P.take_sqrt ? sqrtf(p) : p;
        }
    }
    __syncthreads();                                       // sD is re-staged by the next iteration
    cur = nxt;
    }
}

}  // namespace ctu
#endif
