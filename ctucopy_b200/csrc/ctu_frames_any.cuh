// K1g: the frame kernel for FFT sizes other than 512 (8 kHz telephone speech: 256 points;
// 22-48 kHz audio: 1024 / 2048 points).  Same chain, same arithmetic conventions as k_frames2 + k_bank
// (rawIN::get_frame src/io/in.cc:305-419, FB::project_frame src/fea/fb.cc:72-86, specFEA /
// logspecFEA / dctcFEA src/fea/fea_impl.cc:37-131), written for generality rather than speed:
// one WARP per frame, the real transform as an in-place radix-2 complex FFT of half the length
// in shared memory, filter-bank weights and twiddles read from global memory (no size limit of
// the kernel-parameter block).  Every BASELINE configuration is 16 kHz / 512 points and takes
// the specialised kernels; this one exists so that other sampling rates work at all.
#ifndef CTU_FRAMES_ANY_CUH
#define CTU_FRAMES_ANY_CUH

#include "ctu_kernels.cuh"

namespace ctu {

constexpr int ANY_THREADS = 256;              // 8 warps = 8 frames in flight
constexpr int ANY_TILE = 16;                  // frames per CTA (the 16-frame tile list)
constexpr int ANY_MAX_NFFT = 2048;
constexpr int ANY_DC1_MAX = 18;               // frames a sample can be part of (+1), -remove_dc1

struct AnyTables {
    const float2 *tw;        // e^{-2 pi i k / M}, k < M/2           (M = nfft/2)
    const float2 *twsplit;   // -i/2 e^{-2 pi i k / nfft}, k <= M
    const float *win;        // analysis window [window]
    const float *fbw;        // packed filter-bank taps (scaled like FrameParams::w), bands 16-byte aligned
    const int4 *bands;       // [nb] {lo, ntaps, woff, 0}
    int nfft, log2m;
    // CTA-level copies in shared memory behind the per-warp areas (float offsets, -1 = read from global): every butterfly,
    // window multiply and filter-bank tap used to be a dependent global load; the host stages what fits without costing a
    // resident CTA (any_stage_layout)
    int o_tw, o_ts, o_win, o_fbw, nfbw;
    int o_m2, nm2;           // the second-stage matrix (DCT + lifter), TRANSPOSED: [nb][nrows]
    int o_pcm, npcm;         // the tile's pre-emphasised samples as floats (plain configurations: no dither, no -remove_dc1)
};

__host__ __device__ inline size_t any_smem_floats_per_warp(int nfft) { return (size_t)nfft /* M complex */ + (nfft / 2 + 4) /* bins */ + MAXB + 4; }

// which tables go to shared memory: in the order twiddles, split twiddles, window, filter-bank taps, as long as the CTA keeps
// the residency its per-warp areas alone would have (at most 8 CTAs of 256 threads per SM)
inline size_t any_stage_layout(AnyTables &tb, int window) {
    const size_t base = any_smem_floats_per_warp(tb.nfft) * (256 / 32);
    const size_t cap = (227 * 1024 - 8 * 1024) / sizeof(float);                       // per SM, minus the per-CTA reservations
    const size_t ctas = std::max<size_t>(1, std::min<size_t>(8, cap / base));
    const size_t budget = cap / ctas;
    const int M = tb.nfft / 2;
    size_t o = base;
    auto take = [&](int &off, size_t n) { n = (n + 3) & ~(size_t)3; if (o + n <= budget) { off = (int)o; o += n; } else off = -1; };
    take(tb.o_m2, (size_t)tb.nm2);         // first: read with a per-lane index, which the constant bank serialises (13 x 26
                                           // replays per frame: the DCT alone took half the time of an 8 kHz MFCC frame)
    take(tb.o_pcm, (size_t)tb.npcm);       // the 16 frames of a tile overlap 2-3 times: one coalesced pass instead of two 2-byte
                                           // global loads and two conversions per sample and frame
    take(tb.o_tw, (size_t)M);              // M/2 float2
    take(tb.o_ts, (size_t)2 * (M + 1));
    take(tb.o_win, (size_t)window);
    take(tb.o_fbw, (size_t)tb.nfbw);
    return o * sizeof(float);
}

// -remove_dc1 (src/io/in.cc:343-350): mean of the ring at frame t, m_t = mean(raw frame t) - sum_d m_{t-d} (w - d s) / w
// (the overlap with frame t-d has already lost m_{t-d}).  One warp per utterance, frames in order, fp64.
__global__ void __launch_bounds__(128)
k_dc1_means(const int *__restrict__ nframes, const int64_t *__restrict__ row_off, const int64_t *__restrict__ pcm_off, int u0, int n_utts,
            int w, int s, const int16_t *__restrict__ pcm, double *__restrict__ m) {
    const int u = u0 + blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (u >= u0 + n_utts) return;
    const int lane = threadIdx.x & 31;
    const int T = nframes[u];
    const int16_t *x = pcm + pcm_off[u];
    double *mu = m + row_off[u];
    for (int t = 0; t < T; t++) {
        int acc = 0;
        for (int i = lane; i < w; i += 32) acc += (int)x[(int64_t)t * s + i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) {
            double v = (double)acc / (double)w;
            for (int d = 1; d * s < w && d <= t; d++) v -= mu[t - d] * (double)(w - d * s) / (double)w;
            mu[t] = v;
        }
        __syncwarp();
    }
}

template <int SRC, int DST, int KIND>
__global__ void __launch_bounds__(ANY_THREADS)
k_frames_any(const __grid_constant__ FrameParams P, BatchDesc bd, AnyTables tb, const int16_t *__restrict__ pcm,
             const float *__restrict__ src, float *__restrict__ dst) {
    extern __shared__ __align__(16) float sm[];
    const int lane = threadIdx.x & 31, wv = threadIdx.x >> 5;
    const int nfft = tb.nfft, M = nfft >> 1, nbins = M + 1;
    float *base = sm + (size_t)wv * any_smem_floats_per_warp(nfft);
    cpx<float> *z = reinterpret_cast<cpx<float> *>(base);              // M complex
    float *row = base + nfft;                                          // nbins (+pad)
    float *sY = row + (M + 4);                                         // MAXB (+pad)
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int nf = min(ANY_TILE, bd.nframes[u] - t0);
    const int64_t row0 = bd.row_off[u] + t0;
    const int w = P.window, s = P.wshift, nb = P.nb;
    // tables: shared-memory copies where the host found room for them
    const float2 *twp = tb.tw, *tsp = tb.twsplit;
    const float *winp = tb.win, *fbwp = tb.fbw;
    if (tb.o_tw >= 0) { float2 *d = reinterpret_cast<float2 *>(sm + tb.o_tw); for (int i = threadIdx.x; i < (M >> 1); i += ANY_THREADS) d[i] = tb.tw[i]; twp = d; }
    if (tb.o_ts >= 0) { float2 *d = reinterpret_cast<float2 *>(sm + tb.o_ts); for (int i = threadIdx.x; i <= M; i += ANY_THREADS) d[i] = tb.twsplit[i]; tsp = d; }
    if (tb.o_win >= 0 && SRC == SRC_PCM) { float *d = sm + tb.o_win; for (int i = threadIdx.x; i < w; i += ANY_THREADS) d[i] = tb.win[i]; winp = d; }
    const float *spcm = nullptr;
    if (SRC == SRC_PCM && tb.o_pcm >= 0 && tb.npcm > 0 && !P.dither && !P.dc1) {
        float *d = sm + tb.o_pcm;
        const int16_t *x = pcm + bd.pcm_off[u] + (int64_t)t0 * s;
        const int ns = (nf - 1) * s + w;
        for (int i = threadIdx.x; i < ns; i += ANY_THREADS) {
            const float xi = (float)x[i], xp = (i == 0 && t0 == 0) ? 0.f : (float)x[i - 1];
            d[i] = fmaf(-P.preem, xp, xi);
        }
        spcm = d;
    }
    const float *m2t = nullptr;
    if (tb.o_m2 >= 0 && DST == DST_FEA && KIND == KIND_DCTC) {
        float *d = sm + tb.o_m2;
        for (int i = threadIdx.x; i < P.nrows * nb; i += ANY_THREADS) d[(i % nb) * P.nrows + i / nb] = P.m2[(i / nb) * P.nbp + i % nb];
        m2t = d;
    }
    if (tb.o_fbw >= 0 && DST != DST_SPEC) { float *d = sm + tb.o_fbw; for (int i = threadIdx.x; i < tb.nfbw; i += ANY_THREADS) d[i] = tb.fbw[i]; fbwp = d; }
    __syncthreads();
    constexpr bool WANT_LOG = (DST == DST_FEA) && (KIND == KIND_DCTC || KIND == KIND_LOGSPEC || KIND == KIND_TRAPLOG);
    for (int f = wv; f < nf; f += ANY_THREADS / 32) {
        // ---- A: frame -> spectrum row ------------------------------------------------------------
        if (SRC == SRC_PCM) {
            const int16_t *x = pcm + bd.pcm_off[u] + (int64_t)(t0 + f) * s;
            const float *dn = P.dither ? P.dither + bd.pcm_off[u] + (int64_t)(t0 + f) * s : nullptr;
            const bool at_start = (t0 + f) == 0;
            float *y = reinterpret_cast<float *>(z);                   // the frame as nfft reals, natural order first
            float sum = 0.f;
            // -remove_dc1: frame t subtracts the mean of the whole ring from the ring, so a sample that is in frames
            // t-d .. t has lost m[t-d] + .. + m[t] by the time frame t reads it (m from k_dc1_means)
            float md[ANY_DC1_MAX];
            const int nd = P.dc1 ? min(ANY_DC1_MAX, w / s + 1) : 0;
            for (int d = 0; d < nd; d++) md[d] = (t0 + f - d >= 0) ? (float)P.dc1[row0 + f - d] : 0.f;
            auto ring_off = [&](int i, int d0) {        // what sample i of the frame has lost, counting frames t-d0, t-d0-1, ...
                float c = 0.f;
                for (int d = d0; d < nd; d++) if (i + (d - d0) * s < w) c += md[d];
                return c;
            };
            // Large frames go straight to their bit-reversed places (complex point n = i / 2 lands at rev(n)); small ones are
            // stored in natural order and permuted in a pass of their own.  Measured: the scattered store lands 16 consecutive
            // points in two banks at M = 128 (8 kHz: 14.7 -> 16.1 ms per 8 M frames), while at M >= 512 the saved pass wins
            // (22.05 kHz: 36.8 -> 34.9 ms per 2.9 M frames, 44.1 kHz: 45.0 -> 41.0 ms per 1.4 M).
            const bool fold = nfft >= 1024;
            const int rsh = 32 - tb.log2m;
            auto place = [&](int i) { return fold ? 2 * (int)(__brev((unsigned)(i >> 1)) >> rsh) + (i & 1) : i; };
            for (int i = lane; i < nfft; i += 32) {
                float v = 0.f;
                if (i < w) {
                    if (spcm) v = winp[i] * spcm[f * s + i];
                    else {
                        float xi = (float)x[i];
                        float xp = (i == 0 && at_start) ? 0.f : (float)x[i - 1];
                        if (dn) { xi += dn[i]; if (!(i == 0 && at_start)) xp += dn[i - 1]; }
                        if (P.dc1) {
                            xi -= ring_off(i, 0);
                            // the sample before the frame was remembered at the end of frame t-1 (src/io/in.cc:384)
                            if (i > 0) xp -= ring_off(i - 1, 0);
                            else if (!at_start) xp -= ring_off(s - 1, 1);
                        }
                        v = winp[i] * fmaf(-P.preem, xp, xi);
                    }
                }
                y[place(i)] = v;
                sum += v;
            }
            if (P.remove_dc) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
                const float mean = sum / (float)w;                    // of the windowed frame, subtracted inside the window only
                __syncwarp();
                for (int i = lane; i < w; i += 32) y[place(i)] -= mean;
            }
            __syncwarp();
            if (!fold) {
                // bit-reversal permutation of the M complex points (z[n] = y[2n] + i y[2n+1])
                for (int n = lane; n < M; n += 32) {
                    const int r = (int)(__brev((unsigned)n) >> rsh);
                    if (r > n) { const cpx<float> t = z[n]; z[n] = z[r]; z[r] = t; }
                }
                __syncwarp();
            }
            // decimation in time on the bit-reversed points: one radix-2 stage when log2(M) is odd, then radix-4 passes (two
            // radix-2 stages of half lengths h and 2h fused: the four points p, p+h, p+2h, p+3h are read and written once, the
            // second stage's odd twiddle is -i times the even one).  A third of the shared-memory passes and warp barriers
            // of the radix-2 loop this replaces.
            int h = 1, sh = tb.log2m - 1;                             // first stage: half length h, twiddle tw[j << sh]
            if (tb.log2m & 1) {
                for (int b = lane; b < (M >> 1); b += 32) {
                    const cpx<float> a = z[2 * b], t = z[2 * b + 1];
                    z[2 * b] = a + t;
                    z[2 * b + 1] = a - t;
                }
                __syncwarp();
                h = 2; sh--;
            }
            for (; 4 * h <= M; h <<= 2, sh -= 2) {
                for (int q = lane; q < (M >> 2); q += 32) {
                    const int j = q & (h - 1), p0 = ((q - j) << 2) + j;
                    const float2 w1 = twp[(size_t)j << sh], w2 = twp[(size_t)j << (sh - 1)];
                    const cpx<float> z0 = z[p0], t1 = cmul(z[p0 + h], mk<float>(w1.x, w1.y));
                    const cpx<float> z2 = z[p0 + 2 * h], t3 = cmul(z[p0 + 3 * h], mk<float>(w1.x, w1.y));
                    const cpx<float> a0 = z0 + t1, a1 = z0 - t1;
                    const cpx<float> u2 = cmul(z2 + t3, mk<float>(w2.x, w2.y)), u3 = cmul(z2 - t3, mk<float>(w2.x, w2.y));
                    const cpx<float> v3 = mk<float>(u3.y, -u3.x);     // -i u3
                    z[p0] = a0 + u2;
                    z[p0 + 2 * h] = a0 - u2;
                    z[p0 + h] = a1 + v3;
                    z[p0 + 3 * h] = a1 - v3;
                }
                __syncwarp();
            }
            // real-input split, power / magnitude
            for (int k = lane; k <= M; k += 32) {
                const cpx<float> A = z[k == M ? 0 : k], B = conj(z[k == 0 ? 0 : M - k]);
                const float2 ts = tsp[k];
                const cpx<float> X = mk<float>(0.5f * (A.x + B.x), 0.5f * (A.y + B.y)) + cmul(mk<float>(ts.x, ts.y), A - B);
                float p = X.x * X.x + X.y * X.y;
                if (k == 0 && P.remove_dc) p = 1e-10f;                // fixed floor (src/io/in.cc:390)
                row[k] = P.take_sqrt ? sqrtf(p) : p;
            }
        } else {
            const float *g = src + (row0 + f) * nbins;
            for (int k = lane; k < nbins; k += 32) row[k] = g[k];
        }
        __syncwarp();
        if (DST == DST_SPEC) {
            float *g = dst + (row0 + f) * nbins;
            for (int k = lane; k < nbins; k += 32) g[k] = row[k];
            __syncwarp();
            continue;
        }
        if (P.energy_mode == EN_NR || P.energy_mode == EN_IN) {
            const float e = half_spectrum_energy(row, nbins, (P.energy_mode == EN_NR) || P.take_sqrt);
            if (lane == 0) P.energy[row0 + f] = e;
        }
        // ---- B: filter bank, one band per lane -----------------------------------------------------
        const bool late_log = (KIND == KIND_LOGSPEC && P.energy_mode == EN_BANDS && DST == DST_FEA);
        for (int b = lane; b < nb; b += 32) {
            const int4 bs = __ldg(tb.bands + b);
            const float *r = row + bs.x;
            const float *wq = fbwp + bs.z;
            float acc = 0.f;
            for (int k = 0; k < bs.y; k++) acc = fmaf(r[k], wq[k], acc);   // the reference's summation order
            const bool lg = WANT_LOG && !late_log;
            float yv;
            if (P.inld) { yv = powf(acc, 0.33f) * P.inld_scale; if (lg) yv = logf(yv); }
            else yv = lg ? logf(acc) + P.log_offset : acc * P.lin_scale;
            sY[b] = yv;
        }
        for (int b = nb + lane; b < P.nbp; b += 32) sY[b] = 0.f;
        __syncwarp();
        if (DST == DST_FB) {
            float *g = dst + (row0 + f) * nb;
            for (int b = lane; b < nb; b += 32) g[b] = sY[b];
            __syncwarp();
            continue;
        }
        // ---- C: features ---------------------------------------------------------------------------
        float *g = dst + (row0 + f) * P.out_stride;
        if (KIND == KIND_DCTC) {
            for (int i = lane; i < P.nrows; i += 32) {
                float acc = 0.f;
                if (m2t) {
                    for (int k = 0; k < nb; k++) acc = fmaf(sY[k], m2t[k * P.nrows + i], acc);      // lanes read consecutive words
                } else {
                    const float *m = P.m2 + i * P.nbp;
                    for (int k = 0; k < nb; k++) acc = fmaf(sY[k], m[k], acc);
                }
                g[i] = acc;
            }
        } else {
            if (P.energy_mode == EN_BANDS && lane == 0) {
                double acc = 0.5 * (double)sY[0] * (double)sY[0];
                for (int b = 1; b < nb - 1; b++) acc += (double)sY[b] * (double)sY[b];
                acc += 0.5 * (double)sY[nb - 1] * (double)sY[nb - 1];
                P.energy[row0 + f] = (float)log(acc * 2.0);
            }
            for (int b = lane; b < nb; b += 32) g[b] = late_log ? logf(sY[b]) : sY[b];
        }
        __syncwarp();
    }
}

}  // namespace ctu
#endif
