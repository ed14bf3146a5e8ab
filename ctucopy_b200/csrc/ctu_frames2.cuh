// K1s: PCM -> spectrum with a GROUP-LOCAL pipeline (the front end of every chain in which a
// cross-frame stage follows: noise-reduction scans, Burg detector, synthesis).
//
// A CTA of 128 threads = 8 groups of 16 threads works on a tile of 16 consecutive frames of
// one utterance.  The CTA synchronises once, after staging the tile's pre-emphasised samples
// (four per thread, finish_pcm) and the (small) tables in shared memory; the descriptors of
// the next tiles arrive ahead in shared memory (TileAhead); from then on each group takes a frame through
//   window, DC removal -> 256-point complex FFT (16 points per thread, ctu_fft.cuh) -> real
//   split by register shuffles -> power / magnitude
// on its own, synchronising only inside its half warp, and stores its 257 bins from the
// registers straight to HBM (every store instruction covers 64 contiguous bytes).
// No [frames x 257] tile in shared memory: 39.0 KB per CTA; persistent CTAs, twiddles in registers, complex arithmetic on
// packed FP32 instructions (ctu_fft.cuh).  Five resident CTAs (20 warps) per SM at 94 registers for 25 ms windows (window
// values read from shared memory), four at up to 128 registers otherwise (window values in registers), against two CTAs
// (16 warps) for the 32-frame tile kernel k_frames it replaced, which needed that tile for its lane = frame filter bank.
// Measured on 9.98 M frames: 5.63 ms here (first version: 7.3), 8.4 ms (persistent, prefetching) / 9.5 ms (plain) with k_frames.
// Replaces rawIN::get_frame (src/io/in.cc:305-419).
#ifndef CTU_FRAMES2_CUH
#define CTU_FRAMES2_CUH

#include "ctu_kernels.cuh"

namespace ctu {

constexpr int F2_THREADS = 128;
constexpr int F2_GROUPS = F2_THREADS / GROUP;   // 8 frames in flight per CTA
constexpr int F2_TILE = 16;                     // frames per CTA: two passes
constexpr int F2_ROWF = 2 * XPAD * 16;          // floats in a group's exchange area (544)

struct Smem2 {
    int oX, oTw, oTs, oW, oD, oRaw, oA, total;  // float offsets
};
__host__ __device__ inline Smem2 smem2_layout(int window, int wshift) {
    Smem2 L;
    int o = 0;
    L.oX = o; o += F2_GROUPS * F2_ROWF;
    L.oTw = o; o += 256 * 2;
    L.oTs = o; o += 130 * 2;
    L.oW = o; o += (window + 3) & ~3;
    L.oD = o; o += ((F2_TILE - 1) * wshift + window + 7) & ~7;
    L.oRaw = o; o += (((F2_TILE - 1) * wshift + window + 1 + 8 + 7) / 8) * 4;   // int16 prefetch buffer: 8-sample chunks
    L.oA = o; o += TILE_AHEAD_FLOATS;
    L.total = o;
    return L;
}

// CPLX: also store the complex spectrum X (float2 per bin) for the synthesis (k_synth_c): the phase then never has to be
// recomputed from the samples.
// WSM: the thread's 32 window values come from shared memory (16 eight-byte loads per frame) instead of living in
// registers.  With packed arithmetic the kernel is latency bound at four CTAs per SM (ncu: issue slots 54 %, FP32 pipe 29 %,
// shared-memory wavefronts 61 %, 16 warps per SM); without the 32 registers the 25 ms window fits five CTAs (92 registers,
// no spills; 94 since the descriptor and staging changes): 6.19 -> 6.05 ms per 9.98 M frames (tools/gpu_jobs/r2_job46.sh).
// The other instantiations would spill at 102 registers (32 ms window, stored complex spectrum: 5.80 -> 6.33 ms) and keep
// the window in registers at four CTAs.
template <int WT, bool CPLX> struct F2Cfg {
    static constexpr bool wsm = (WT == 400) && !CPLX;
    static constexpr int minb = wsm ? 5 : 4;
};
template <int WT, bool CPLX = false>
__global__ void __launch_bounds__(F2_THREADS, F2Cfg<WT, CPLX>::minb)
k_frames2(const __grid_constant__ FrameParams P, BatchDesc bd, FftTables tb, const int16_t *__restrict__ pcm, float *__restrict__ dst,
          int ntiles, float2 *__restrict__ cdst = nullptr) {
    extern __shared__ __align__(16) float sm[];
    const Smem2 L = smem2_layout(P.window, P.wshift);
    const int tid = threadIdx.x;
    const int w = WT ? WT : P.window, s = P.wshift;
    float *sD = sm + L.oD, *sW = sm + L.oW;
    int16_t *raw = reinterpret_cast<int16_t *>(sm + L.oRaw);
    cpx<float> *sTw = reinterpret_cast<cpx<float> *>(sm + L.oTw);
    cpx<float> *sTs = reinterpret_cast<cpx<float> *>(sm + L.oTs);
    // persistent CTAs: the next tile's PCM is prefetched with cp.async while this one is transformed
    int tile = blockIdx.x;
    if (tile >= ntiles) return;
    TileMeta cur = load_tile_meta(bd, tile, s, F2_TILE);
    TileAhead *ahead = reinterpret_cast<TileAhead *>(sm + L.oA);
    tile_ahead_init(ahead, bd, tile, ntiles);
    int edge = 0;
    prefetch_pcm<F2_THREADS>(raw, pcm, cur, (cur.nf - 1) * s + w + 1, edge);
    for (int i = tid; i < w; i += F2_THREADS) sW[i] = tb.win[i];
    for (int i = tid; i < 256; i += F2_THREADS) sTw[i] = mk<float>(tb.tw256[i].x, tb.tw256[i].y);
    for (int i = tid; i < 129; i += F2_THREADS) sTs[i] = mk<float>(tb.twsplit[i].x, tb.twsplit[i].y);

    const int c = tid & (GROUP - 1), grp = tid / GROUP;
    cpx<float> *xch = reinterpret_cast<cpx<float> *>(sm + L.oX + grp * F2_ROWF);
    const float inv_w = 1.0f / (float)w;
    // a thread windows the same 2 x 16 sample positions of every frame it ever sees: its window values live in
    // registers for the whole (persistent) kernel instead of being re-read from shared memory per frame
    __syncthreads();
    constexpr bool WSM = F2Cfg<WT, CPLX>::wsm;
    float wr[WSM ? 2 : 32];
    if constexpr (!WSM) {
#pragma unroll
        for (int n1 = 0; n1 < 16; n1++) {
            const int i0 = 32 * n1 + 2 * c;
            wr[2 * n1] = (i0 < w) ? sW[i0] : 0.f;
            wr[2 * n1 + 1] = (i0 + 1 < w) ? sW[i0 + 1] : 0.f;
        }
    }
    // window value i of this thread (i = 2 n1, 2 n1 + 1 <-> sample 32 n1 + 2 c, + 1; the caller keeps the index inside the window)
    auto wv = [&](int i) -> float { if constexpr (WSM) return sW[32 * (i >> 1) + 2 * c + (i & 1)]; else return wr[i]; };
    // so do its twiddles: the six inter-pass ones it used to load per frame, and twsplit[c] (the other seven split
    // twiddles are that value times compile-time constants) -- 14 shared-memory loads per frame off the LSU pipe
    cpx<float> twr[6];
    twr[0] = sTw[16 + c]; twr[1] = sTw[32 + c]; twr[2] = sTw[48 + c];
    twr[3] = sTw[64 + c]; twr[4] = sTw[128 + c]; twr[5] = sTw[192 + c];
    const cpx<float> ts_c = sTs[c];
#pragma unroll 1
    for (int j = 0; tile < ntiles; tile += gridDim.x, j ^= 1) {
    const int next = tile + gridDim.x;
    const int nf = cur.nf;
    const int64_t row0 = cur.row0;
    finish_pcm<F2_THREADS>(raw, sD, pcm, cur, (nf - 1) * s + w + 1, edge, P.preem);
    __syncthreads();                                          // samples staged; the raw buffer is free again
    const TileMeta nxt = tile_ahead_next(ahead, j, bd, tile, ntiles, s, F2_TILE);   // used only when next < ntiles
    if (next < ntiles) prefetch_pcm<F2_THREADS>(raw, pcm, nxt, (nxt.nf - 1) * s + w + 1, edge);
    // the two groups of a warp walk the tile in step (frames grp, grp + 8): with an odd number of frames the last group
    // recomputes the tile's last frame and stores nothing -- every shuffle can then name the full warp (bare SHFL)
    const int nf_even = (nf + 1) & ~1;
#pragma unroll 1
    for (int f0 = grp; f0 < nf_even; f0 += F2_GROUPS) {
        const bool store = f0 < nf;
        const int f = min(f0, nf - 1);
        cpx<float> a[16];
        // sample pairs as 8-byte loads: a half warp covers 128 contiguous bytes, so the two frames of a warp (whose rows
        // start on the same bank when the shift is a multiple of 32 samples) no longer collide (ncu: 16 of the 105
        // wavefronts per frame were these conflicts).  Needs an even shift; odd shifts take scalar loads.
        const float *d = sD + f * s;
        const bool pair = (s & 1) == 0;
        // two samples and their two window values are register pairs: windowing, the sum for the mean and its
        // subtraction are packed instructions (ctu_fft.cuh); the sum runs over even and odd samples separately
        cpx<float> sum2 = mk<float>(0.f, 0.f);
#pragma unroll
        for (int n1 = 0; n1 < 16; n1++) {
            const int i0 = 32 * n1 + 2 * c;
            if (i0 + 1 < w && pair) {
                const float2 dd = *reinterpret_cast<const float2 *>(d + i0);
                if constexpr (WSM) {
                    const float2 ww = *reinterpret_cast<const float2 *>(sW + i0);
                    a[n1] = pmul(mk<float>(ww.x, ww.y), mk<float>(dd.x, dd.y));
                } else {
                    a[n1] = pmul(mk<float>(wr[2 * n1], wr[2 * n1 + 1]), mk<float>(dd.x, dd.y));
                }
            } else {
                float y0 = 0.f, y1 = 0.f;
                if (i0 < w) y0 = wv(2 * n1) * d[i0];
                if (i0 + 1 < w) y1 = wv(2 * n1 + 1) * d[i0 + 1];
                a[n1] = mk<float>(y0, y1);
            }
            if (32 * n1 < w) sum2 = sum2 + a[n1];
        }
        if (P.remove_dc) {
            // mean of the WINDOWED frame, subtracted from the window's samples only (src/io/in.cc:375-382)
            const float mean = group_sum16_all(sum2.x + sum2.y) * inv_w;
#pragma unroll
            for (int n1 = 0; n1 < 16; n1++) {
                const int i0 = 32 * n1 + 2 * c;
                if (32 * n1 < w) a[n1] = a[n1] - mk<float>(i0 < w ? mean : 0.f, i0 + 1 < w ? mean : 0.f);
            }
        }
        fft256_pass1_reg(a, c, twr, xch);
        __syncwarp();
        fft256_pass2(a, c, xch);
        cpx<float> lo[8], hi[8], mid;
        rfft_split_shfl_rec(a, c, ts_c, lo, hi, mid);
        __syncwarp();                                         // all reads of the exchange tile are done
        if (!store) continue;
        float *g = dst + (row0 + f) * SPITCH;
        if (CPLX) {
            float2 *gc = cdst + (row0 + f) * NBIN;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                gc[c + 16 * j] = make_float2(lo[j].x, lo[j].y);
                gc[NC - c - 16 * j] = make_float2(hi[j].x, hi[j].y);
            }
            if (c == 0) gc[128] = make_float2(mid.x, mid.y);
        }
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const int k = c + 16 * j;
            float pl = lo[j].x * lo[j].x + lo[j].y * lo[j].y;
            float ph = hi[j].x * hi[j].x + hi[j].y * hi[j].y;
            if (k == 0 && P.remove_dc) pl = 1e-10f;           // fixed floor (src/io/in.cc:390)
            if (P.take_sqrt) { pl = sqrtf(pl); ph = sqrtf(ph); }
            g[k] = pl;
            g[NC - k] = ph;
        }
        if (c == 0) {
            const float pm = mid.x * mid.x + mid.y * mid.y;
            g[128] = P.take_sqrt ? sqrtf(pm) : pm;
        } else if (c <= SPITCH - NBIN) {
            g[NBIN - 1 + c] = 0.f;                             // pad columns: read (times zero weights) by the 16-byte loads of k_bank
        }
    }
    __syncthreads();                                          // sD is re-staged by the next iteration
    cur = nxt;
    }
}

}  // namespace ctu
#endif
