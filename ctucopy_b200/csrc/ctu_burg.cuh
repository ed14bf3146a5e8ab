// K4 / K5: the Burg cepstral detector (sm_100a), compiled in its own translation unit (ctu_burg.cu):
//   k_burg / k_burg_any  per frame, fp64: forward FFT -> (|X|^a, phase) -> unnormalised inverse FFT -> [Hann] -> Burg
//                        lattice -> LPC cepstrum (src/nr/nr.cc:281-292, src/vad/vad.cc:222-237, src/vdet/Burg.h:49-152)
//   k_cepdet             per utterance: adaptive-threshold cepstral detector (src/vdet/CepstralDet.h:134-194)
#ifndef CTU_BURG_CUH
#define CTU_BURG_CUH

#include "ctu_nr_params.cuh"

namespace ctu {

// ------------------------------------------------------------------------------------------
// K4: Burg cepstrum per frame (fp64 throughout so that detector decisions are reproducible)
// 128 threads = 8 frames per pass; a CTA takes HALF of a 32-frame tile (two passes), so that its staged samples, the
// tables and the eight exchange areas fit four CTAs per SM.
//   * the half tile's PCM is staged once into shared memory as int16 (16-byte loads);
//   * forward FFT -> per-bin gain (|X|^a or the post-NR magnitude, over |X|) -> inverse FFT.  Real split, gain and the
//     inverse pre-split run IN PLACE on the 16 complex registers of a thread, pair by pair (bins k and 256-k): the
//     partner's value arrives by shuffle, the rebuilt pair is written back over the registers it came from.  (Round 1
//     materialised lo[8] / hi[8] / zn[8] next to a[16]: 236 registers, two CTAs per SM, FP64 pipe 41 % busy.)
//   * lattice: sample i = c*CH + j lives in thread c's registers.  All updates and sums are unconditional; the elements the
//     reference no longer reads (i < ik, src/vdet/Burg.h:64-68) are driven to exact zeros instead of being masked, and where
//     the window fills the threads exactly the denominator is carried from stage to stage (see the stage loop).
//   * the predictor coefficients are distributed (thread i holds a_i; one shuffle per stage).
// CH: samples per thread; EXACT: window == 16*CH (no tail masking in the energy sums); GENA: the spectral exponent is not 1
// or 2 (-nr_a): only that instantiation carries pow() -- inlined at the 17 bin sites of a thread it costs the common paths
// registers and instruction-cache space for nothing.
// ------------------------------------------------------------------------------------------
constexpr int BURG_THREADS = 128;
constexpr int BURG_GROUPS = BURG_THREADS / GROUP;
constexpr int BURG_HALF = TILE_F / 2;                     // frames per CTA

// Shuffles inside a 16-lane group with the FULL member mask: both groups of a warp always execute them together (a group
// without a frame of its own recomputes the tile's last frame and skips the stores).  With the per-group masks of round 1
// every shuffle was wrapped in BSSY / WARPSYNC / ENDCOLLECTIVE / BSYNC: a fifth of the kernel's instructions.
__device__ __forceinline__ double shfl16d(double v, int src) { return __shfl_sync(0xffffffffu, v, src, 16); }
// num / den without the IEEE division sequence (range checks, a slow-path call: ~16 instructions and a branch, eleven times
// per frame): hardware reciprocal seed, two Newton steps, one correction of the quotient -- within an ulp of the rounded
// quotient; 0 / 0 and x / 0 come out NaN / inf as the reference's division gives them
__device__ __forceinline__ double fast_div(double n, double d) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    r = fma(fma(-d, r, 1.0), r, r);
    r = fma(fma(-d, r, 1.0), r, r);
    const double q = n * r;
    return fma(fma(-d, q, n), r, q);
}
__device__ __forceinline__ double group_sum16d_all(double v) {
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v;
}

template <int CH, bool EXACT, int MINB, bool GENA, bool REC = EXACT>
__global__ void __launch_bounds__(BURG_THREADS, MINB)
k_burg(const __grid_constant__ BurgParams B, int src_mode, BatchDesc bd, int nhalf, const int16_t *__restrict__ pcm, const float *__restrict__ spec,
       double *__restrict__ ceps, const double2 *__restrict__ g_tw256, const double2 *__restrict__ g_twsplit,
       const double2 *__restrict__ g_twinv, const double *__restrict__ g_win, const double *__restrict__ g_hann) {
    extern __shared__ __align__(16) double smd[];
    const int tid = threadIdx.x;
    const int w = EXACT ? 16 * CH : B.window, s = B.wshift;
    const int wp = (w + 1) & ~1;
    cpx<double> *sTw = reinterpret_cast<cpx<double> *>(smd);            // 256
    cpx<double> *sTs = sTw + 256;                                      // 129 (+1 pad)
    cpx<double> *sTi = sTs + 130;                                      // 129 (+1 pad)
    cpx<double> *sX = sTi + 130;                                       // BURG_GROUPS * 16*17 (also the time signal)
    double *sWin = reinterpret_cast<double *>(sX + BURG_GROUPS * XPAD * 16);   // w: analysis window
    double *sHann = sWin + wp;                                         // w: detector's Hann (NR source)
    int16_t *sPcm = reinterpret_cast<int16_t *>(sHann + wp);           // 8 + (BURG_HALF-1)*s + w + 1 + 8
    for (int i = tid; i < 256; i += BURG_THREADS) sTw[i] = mk<double>(g_tw256[i].x, g_tw256[i].y);
    for (int i = tid; i < 129; i += BURG_THREADS) { sTs[i] = mk<double>(g_twsplit[i].x, g_twsplit[i].y); sTi[i] = mk<double>(g_twinv[i].x, g_twinv[i].y); }
    for (int i = tid; i < wp; i += BURG_THREADS) {
        sWin[i] = (i < w) ? g_win[i] : 0.0;
        sHann[i] = (i < w) ? ((src_mode == BURG_SRC_NR) ? g_hann[i] : 1.0) : 0.0;
    }
    {
    const int ht = blockIdx.x;
    const int2 tile = bd.tiles[ht >> 1];
    const int u = tile.x, t0 = tile.y + (ht & 1) * BURG_HALF;
    const int nf = min(BURG_HALF, bd.nframes[u] - t0);
    if (nf <= 0) return;                                     // (uniform over the CTA)
    const int64_t row0 = bd.row_off[u] + t0;
    // samples [first-1, first + nsamp): the one before the tile feeds the first pre-emphasis
    const int nsamp = (nf - 1) * s + w + 1;
    const bool at_start = (t0 == 0);
    const int16_t *src = pcm + bd.pcm_off[u] + (int64_t)t0 * s - 1;
    const int phase = (int)((reinterpret_cast<uintptr_t>(src) & 15) >> 1);      // same 16-byte phase in shared memory
    int16_t *dpcm = sPcm + phase;
    for (int k0 = tid * 8 - phase; k0 < nsamp; k0 += BURG_THREADS * 8) {
        if (k0 >= (at_start ? 1 : 0) && k0 + 8 <= nsamp) {
            *reinterpret_cast<int4 *>(dpcm + k0) = __ldg(reinterpret_cast<const int4 *>(src + k0));
        } else {
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int k = k0 + j;
                if (k >= 0 && k < nsamp) dpcm[k] = (k == 0 && at_start) ? (int16_t)0 : src[k];
            }
        }
    }
    __syncthreads();
    const int c = tid & (GROUP - 1), grp = tid / GROUP;
    const int partner = (16 - c) & 15;
    cpx<double> *xch = sX + grp * (XPAD * 16);
    double *xt = reinterpret_cast<double *>(xch);
    const int ncoef = (src_mode == BURG_SRC_NR) ? B.ncoef_nr : B.ncoef_vad;
    const double inv_w = 1.0 / (double)w;
#pragma unroll 1
    for (int pass = 0; pass < BURG_HALF / BURG_GROUPS; pass++) {
        // a group whose frame number is past the end of the tile recomputes the tile's last frame and stores nothing
        const bool active = pass * BURG_GROUPS + grp < nf;
        const int f = min(pass * BURG_GROUPS + grp, nf - 1);
        {
            cpx<double> a[16];
            {
                const int16_t *x = dpcm + f * s + 1;                  // x[-1] is the sample before the frame
                double sum = 0;
#pragma unroll
                for (int n1 = 0; n1 < 16; n1++) {
                    const int i0 = 32 * n1 + 2 * c;
                    double y0 = 0, y1 = 0;
                    if (i0 < w) {                                     // w is even for every supported window
                        const double xm = (double)x[i0 - 1], x0 = (double)x[i0], x1 = (double)x[i0 + 1];
                        y0 = sWin[i0] * (x0 - B.preem * xm);
                        y1 = sWin[i0 + 1] * (x1 - B.preem * x0);
                    }
                    a[n1] = mk<double>(y0, y1);
                    sum += y0 + y1;
                }
                if (B.remove_dc) {
                    const double mean = group_sum16d_all(sum) * inv_w;
#pragma unroll
                    for (int n1 = 0; n1 < 16; n1++) {
                        const int i0 = 32 * n1 + 2 * c;
                        if (i0 < w) a[n1].x -= mean;
                        if (i0 + 1 < w) a[n1].y -= mean;
                    }
                }
                fft256_pass1(a, c, sTw, xch);
            }
            __syncwarp();
            {
                fft256_pass2(a, c, xch);
                // (|X|^a or the post-NR spectrum) with the phase of X: every bin is scaled by
                // E/|X| -- what Xa*cos(phi), Xa*sin(phi) amount to (src/nr/nr.cc:281-292,
                // src/vad/vad.cc:222-233) -- with the reference's conventions for bin 0
                // (phase 0, src/io/in.cc:398), the Nyquist bin (real) and atan(0/0) = -pi/2
                const float *srow = (src_mode == BURG_SRC_VAD && B.use_spec_gain) ? spec + (row0 + f) * B.spitch : nullptr;
                const bool expand = (src_mode == BURG_SRC_NR && B.expand);
                auto scale_bin = [&](cpx<double> X, int k) -> cpx<double> {
                    double m2 = X.x * X.x + X.y * X.y;
                    const bool edge = (k == 0 || k == NC);
                    if (k == 0) { if (B.remove_dc) m2 = 1e-10; X = mk<double>(sqrt(m2), 0.0); }
                    const double rm = (m2 > 0.0) ? rsqrt(m2) : 0.0;          // 1/|X|
                    const double m = m2 * rm;                                // |X|
                    double E, g;
                    if (srow) { E = (double)srow[k]; g = E * rm; }
                    else {
                        // E = Xa^a with Xa = |X|^2 (fb_power) or |X|;  g = E/|X| without the division
                        // where the exponents are small integers
                        const int ak = expand ? B.a_kind : 1;
                        if (GENA && ak == 0) { E = pow(B.fb_power ? m2 : m, B.a); g = E * rm; }
                        else if (B.fb_power) { E = (ak == 2) ? m2 * m2 : m2; g = (ak == 2) ? m2 * m : m; }
                        else { E = (ak == 2) ? m2 : m; g = (ak == 2) ? m : 1.0; }
                    }
                    if (m2 == 0.0) return edge ? mk<double>(E, 0.0) : mk<double>(0.0, -E);
                    return mk<double>(X.x * g, edge ? 0.0 : X.y * g);
                };
                // real split (rfft_split_pairs), gain, inverse pre-split (irfft_presplit_local / _place), one bin pair at a
                // time and in place: thread c needs Z[256-k] = a[15-j] of thread 16-c (thread 0: its own a[16-j]) and hands
                // conj(Zc[256-k]) back to the same thread, which stores it where the value it lent came from
                const cpx<double> x128 = conj(a[8]);                       // X[128], meaningful for c == 0
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const int k = c + 16 * j;
                    const cpx<double> prov = (c == 0) ? a[(16 - j) & 15] : a[15 - j];
                    cpx<double> Z;
                    Z.x = __shfl_sync(0xffffffffu, prov.x, partner, 16);
                    Z.y = __shfl_sync(0xffffffffu, prov.y, partner, 16);
                    const cpx<double> A = a[j];
                    cpx<double> lo, hi;
                    if (j == 0 && c == 0) {
                        lo = mk<double>(A.x + A.y, 0.0);
                        hi = mk<double>(A.x - A.y, 0.0);
                    } else {
                        const cpx<double> Bc = conj(Z);
                        const cpx<double> E = mk<double>(0.5 * (A.x + Bc.x), 0.5 * (A.y + Bc.y));
                        const cpx<double> Tt = cmul(sTs[k], A - Bc);
                        lo = E + Tt;
                        hi = conj(E - Tt);
                    }
                    lo = scale_bin(lo, k);
                    hi = scale_bin(hi, NC - k);
                    cpx<double> zn;
                    if (j == 0 && c == 0) {
                        a[0] = conj(mk<double>(lo.x + hi.x, lo.x - hi.x));
                        zn = mk<double>(0.0, 0.0);
                    } else {
                        const cpx<double> S = lo + conj(hi);
                        const cpx<double> U = cmul(lo - conj(hi), sTi[k]);
                        a[j] = conj(mk<double>(S.x - U.y, S.y + U.x));           // conj(Zc[k])
                        zn = conj(mk<double>(S.x + U.y, -S.y + U.x));           // conj(Zc[256-k])
                    }
                    cpx<double> back;
                    back.x = __shfl_sync(0xffffffffu, zn.x, partner, 16);
                    back.y = __shfl_sync(0xffffffffu, zn.y, partner, 16);
                    if (c == 0) { if (j >= 1) a[(16 - j) & 15] = back; }
                    else a[15 - j] = back;
                }
                if (c == 0) {
                    // Zc[128] pairs with itself: S = 2 Re(mid), U = 2i Im(mid) * twinv[128]
                    const cpx<double> mid = scale_bin(x128, 128);
                    const cpx<double> Um = cmul(mk<double>(0.0, 2.0 * mid.y), sTi[128]);
                    a[8] = conj(mk<double>(2.0 * mid.x - Um.y, Um.x));
                }
            }
            __syncwarp();                                             // pass-2 reads of the exchange tile are done
            fft256_pass1(a, c, sTw, xch);
            __syncwarp();
            fft256_pass2(a, c, xch);
            __syncwarp();                                             // xch is re-used for the time signal
            {
#pragma unroll
                for (int k2 = 0; k2 < 16; k2++) {
                    const int n = c + 16 * k2;
                    xt[2 * n] = a[k2].x;
                    xt[2 * n + 1] = -a[k2].y;
                }
            }
            __syncwarp();
        }
        {
            // ---- Burg lattice (src/vdet/Burg.h:49-95) on the first w samples ------------------
            double ef[CH], eb[CH];
            double en = 0;
#pragma unroll
            for (int j = 0; j < CH; j++) {
                const int i = c * CH + j;
                double v = (EXACT || i < w) ? xt[i < NFFT ? i : 0] * sHann[i < w ? i : 0] : 0.0;
                if (!EXACT && i >= w) v = 0.0;
                ef[j] = eb[j] = v;
                en += v * v;
            }
            const double en_all = group_sum16d_all(en);
            double alpha = en_all * inv_w;
            // The reference's sums run over i >= ik (src/vdet/Burg.h:64-68).  Elements below ik can only belong to thread 0
            // (ik <= 15 < CH); they are kept at exact zeros instead of being masked out of the sums: thread 0 starts with
            // ef[0] = 0 and takes `below` = 0, which makes eb[ik-1] come out 0 by itself, and ef[ik] is cleared after stage
            // ik by a select chain over the 15 candidates.  (Measured alternatives, 3.99 M frames, k_burg alone: masking the
            // 16 candidates in every stage's sums 20.5 ms, a jump on the stage number 22.6 ms, the select chain 18.7 ms;
            // persistent CTAs lost 2 ms in each case.  DESIGN 10 has the later attempt with one "head" sample per thread.)
            //
            // REC: the denominator is carried from stage to stage instead of being summed again.  With
            //   ef'[i] = ef[i] + rc eb[i-1],  eb'[i] = eb[i-1] + rc ef[i],  rc = -2 num / den:
            //   sum_{i>=ik} (ef'[i]^2 + eb'[i]^2) = (1 + rc^2) den + 4 rc num = (1 - rc^2) den,   so
            //   den_{ik+1} = sum_{i>=ik+1} ef'[i]^2 + sum_{i>=ik} eb'[i]^2 - eb'[N-1]^2 = (1 - rc^2) den_ik - ef'[ik]^2 - eb'[N-1]^2
            // (Andersen 1978): one sum (num) instead of three per sample and stage, 3 DFMA instead of 5.  A rounding error of
            // num or den is amplified by ~2 rc^2 / (1 - rc^2) per stage, i.e. the carried value drifts from the direct sum by
            // ~1e-16 / (accumulated prediction gain); when that gain since the last direct sum passes 1e3 the stage sums den
            // directly again (warp-uniform branch), which bounds the drift at ~1e-13.
            const double v_first = shfl16d(ef[0], 0), v_last = shfl16d(ef[CH - 1], 15);
            double den_c = 2.0 * en_all - v_first * v_first - v_last * v_last;       // stage 1: ef = eb = v
            double gain_c = 1.0;
            if (c == 0) ef[0] = 0.0;
            double a_c = (c == 0) ? 1.0 : 0.0, aa_c = a_c;            // thread i holds a_i
            // the stage loop stays rolled: unrolled 15 times the kernel was 14 k instructions and stalled on instruction fetch
#pragma unroll 1
            for (int ik = 1; ik < ncoef; ik++) {
                double below = shfl16d(eb[CH - 1], (c + 15) & 15);         // eb of sample i-1 across the thread boundary
                if (c == 0) below = 0.0;
                double num, den;
                if (!REC || __any_sync(0xffffffffu, gain_c < 1e-3)) {
                    // three independent chains per parity: the sums are latency-bound otherwise
                    double nu[2] = {0, 0}, df[2] = {0, 0}, db[2] = {0, 0};
#pragma unroll
                    for (int j = 0; j < CH; j++) {
                        const double pv = (j > 0) ? eb[j > 0 ? j - 1 : 0] : below;
                        if (EXACT || c * CH + j < w) {
                            df[j & 1] = fma(ef[j], ef[j], df[j & 1]);
                            db[j & 1] = fma(pv, pv, db[j & 1]);
                            nu[j & 1] = fma(ef[j], pv, nu[j & 1]);
                        }
                    }
                    num = group_sum16d_all(nu[0] + nu[1]) * 2.0;
                    den = group_sum16d_all((df[0] + df[1]) + (db[0] + db[1]));
                    gain_c = 1.0;
                } else {
                    double nu[4] = {0, 0, 0, 0};
#pragma unroll
                    for (int j = 0; j < CH; j++) {
                        const double pv = (j > 0) ? eb[j > 0 ? j - 1 : 0] : below;
                        nu[j & 3] = fma(ef[j], pv, nu[j & 3]);
                    }
                    num = group_sum16d_all((nu[0] + nu[1]) + (nu[2] + nu[3])) * 2.0;
                    den = den_c;
                }
                const double rc = -fast_div(num, den);
                const double om = 1 - rc * rc;
                alpha *= om;
#pragma unroll
                for (int j = CH - 1; j >= 0; j--) {
                    const double pv = (j > 0) ? eb[j > 0 ? j - 1 : 0] : below;
                    const double e0 = ef[j];
                    ef[j] = e0 + rc * pv;
                    eb[j] = pv + rc * e0;
                }
                // ef[ik] leaves the sums (its value is what the carried denominator loses)
                double gone = 0.0;
#pragma unroll
                for (int j = 1; j < BURG_MAXC && j < CH; j++) if (c == 0 && j == ik) { gone = ef[j]; ef[j] = 0.0; }
                if (REC) {
                    const double e_first = shfl16d(gone, 0), b_last = shfl16d(eb[CH - 1], 15);
                    den_c = om * den - e_first * e_first - b_last * b_last;
                    gain_c *= om;
                }
                // a_i = aa_i + rc * aa_{ik-i} (0 < i < ik), a_ik = rc
                const double other = shfl16d(aa_c, (ik - c) & 15);
                if (c == ik) a_c = rc;
                else if (c >= 1 && c < ik) a_c = aa_c + rc * other;
                aa_c = a_c;
            }
            // LPC -> cepstrum (src/vdet/Burg.h:141-152), thread 0 of the group
            double av[BURG_MAXC];
#pragma unroll
            for (int k = 0; k < BURG_MAXC; k++) av[k] = shfl16d(a_c, k);
            if (c == 0 && active) {
                double cc[BURG_MAXC];
                double *o = ceps + (row0 + f) * BURG_MAXC;
#pragma unroll
                for (int n = 1; n < BURG_MAXC; n++) {
                    double sum = 0;
#pragma unroll
                    for (int k = 1; k < BURG_MAXC; k++) if (k < n) sum += (double)(n - k) * cc[(n - k) & (BURG_MAXC - 1)] * av[k];
                    cc[n] = -av[n] - sum * (1.0 / n);                 // (1 / n is a compile-time constant: the loop is unrolled)
                    if (n < ncoef) o[n] = cc[n];
                }
                o[0] = log(alpha);
            }
        }
        __syncwarp();
    }
    }
}

// ------------------------------------------------------------------------------------------
// K4g: the Burg front end for FFT sizes other than 512 (fwss / hwss / 2fwss and the LPC cepstral-distance criterion at
// 8 kHz, 22-48 kHz).  Same arithmetic as k_burg, one WARP per frame, everything in shared memory:
//   frame -> FFT -> per-bin gain (|X|^a or the post-NR magnitude, on the phase of X) -> unnormalised inverse -> first
//   `window` samples [x Hann for the NR detector] -> Burg lattice (src/vdet/Burg.h:49-95) -> cepstrum (:141-152).
// The lattice keeps ef (aliasing the time signal) and eb in shared memory; a stage updates them in chunks of 32 samples
// from the END of the frame, so that eb[i-1] is still the old value when sample i is updated.
// ------------------------------------------------------------------------------------------
// doubles of shared memory per warp of k_burg_any: z (padded), Y, eb
__host__ __device__ inline size_t burg_any_doubles(int M) { return (size_t)2 * any64_zslots(M) + 2 * (M + 2) + 2 * M; }

// DC1: -remove_dc1, the frame is built from the de-meaned ring (B.dc1)
template <bool DC1>
__global__ void __launch_bounds__(ANY64_THREADS)
k_burg_any(const __grid_constant__ BurgParams B, int src_mode, BatchDesc bd, AnyTables64 tb, const int16_t *__restrict__ pcm,
           const float *__restrict__ spec, double *__restrict__ ceps, const double *__restrict__ g_hann) {
    extern __shared__ __align__(16) double smd[];
    const int lane = threadIdx.x & 31, wv = threadIdx.x >> 5;
    const int nfft = tb.nfft, M = nfft >> 1, nbins = M + 1;
    cpx<double> *z = reinterpret_cast<cpx<double> *>(smd + (size_t)wv * burg_any_doubles(M));   // M complex = nfft reals, padded (ctu_any64.cuh)
    cpx<double> *Y = z + any64_zslots(M);                                                      // M + 1 complex (+ pad)
    double *eb = reinterpret_cast<double *>(Y + M + 2);                                         // nfft reals
    double *ef = reinterpret_cast<double *>(Y);                                                 // the lattice's forward errors: Y is dead by then
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int nf = min(TILE_F, bd.nframes[u] - t0);
    const int64_t row0 = bd.row_off[u] + t0;
    const int w = B.window, s = B.wshift;
    const int ncoef = (src_mode == BURG_SRC_NR) ? B.ncoef_nr : B.ncoef_vad;
    for (int f = wv; f < nf; f += ANY64_THREADS / 32) {
        any64_analysis<DC1>(z, tb, pcm + bd.pcm_off[u] + (int64_t)(t0 + f) * s, (t0 + f) == 0, w, B.preem, B.remove_dc, lane, DC1 ? B.dc1 + row0 + f : nullptr, t0 + f, s);
        // (|X|^a or the post-NR spectrum) with the phase of X -- see k_burg for the conventions (bin 0: phase 0 and the fixed
        // 1e-10 floor under -remove_dc, src/io/in.cc:390-398; Nyquist real; atan(0/0) = -pi/2)
        const float *srow = (src_mode == BURG_SRC_VAD && B.use_spec_gain) ? spec + (row0 + f) * B.spitch : nullptr;
        const bool expand = (src_mode == BURG_SRC_NR && B.expand);
        for (int k = lane; k <= M; k += 32) {
            cpx<double> X = any64_bin(z, tb, k);
            double m2 = X.x * X.x + X.y * X.y;
            const bool edge = (k == 0 || k == M);
            if (k == 0) { if (B.remove_dc) m2 = 1e-10; X = mk<double>(sqrt(m2), 0.0); }
            const double rm = (m2 > 0.0) ? rsqrt(m2) : 0.0;
            const double m = m2 * rm;
            double E, g;
            if (srow) { E = (double)srow[k]; g = E * rm; }
            else {
                const int ak = expand ? B.a_kind : 1;
                if (ak == 0) { E = pow(B.fb_power ? m2 : m, B.a); g = E * rm; }
                else if (B.fb_power) { E = (ak == 2) ? m2 * m2 : m2; g = (ak == 2) ? m2 * m : m; }
                else { E = (ak == 2) ? m2 : m; g = (ak == 2) ? m : 1.0; }
            }
            Y[k] = (m2 == 0.0) ? (edge ? mk<double>(E, 0.0) : mk<double>(0.0, -E)) : mk<double>(X.x * g, edge ? 0.0 : X.y * g);
        }
        __syncwarp();
        any64_inverse(z, Y, tb, lane);
        // ---- Burg lattice on the first w samples ------------------------------------------------------------------
        double en = 0.0;
        for (int i = lane; i < w; i += 32) {
            const double v = any64_real(z, i) * ((src_mode == BURG_SRC_NR) ? g_hann[i] : 1.0);
            ef[i] = v; eb[i] = v;
            en += v * v;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) en += __shfl_xor_sync(0xffffffffu, en, o);
        double alpha = en / (double)w;
        __syncwarp();
        double a_c = (lane == 0) ? 1.0 : 0.0, aa_c = a_c;              // lane i holds a_i
#pragma unroll 1
        for (int ik = 1; ik < ncoef; ik++) {
            double num = 0.0, den = 0.0;
            for (int i = ik + lane; i < w; i += 32) {
                const double e1 = ef[i], e2 = eb[i - 1];
                num = fma(e1, e2, num);
                den += e1 * e1 + e2 * e2;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { num += __shfl_xor_sync(0xffffffffu, num, o); den += __shfl_xor_sync(0xffffffffu, den, o); }
            const double rc = -(2.0 * num) / den;
            alpha *= 1 - rc * rc;
            for (int base = (w - 1) & ~31; base >= 0; base -= 32) {
                const int i = base + lane;
                const bool ok = i >= 1 && i < w;
                double e0 = 0.0, pv = 0.0;
                if (ok) { e0 = ef[i]; pv = eb[i - 1]; }
                __syncwarp();
                if (ok) { ef[i] = e0 + rc * pv; eb[i] = pv + rc * e0; }
                __syncwarp();
            }
            const double other = __shfl_sync(0xffffffffu, aa_c, (ik - lane) & 31);
            if (lane == ik) a_c = rc;
            else if (lane >= 1 && lane < ik) a_c = aa_c + rc * other;
            aa_c = a_c;
        }
        double av[BURG_MAXC];
#pragma unroll
        for (int k = 0; k < BURG_MAXC; k++) av[k] = __shfl_sync(0xffffffffu, a_c, k);
        if (lane == 0) {
            double cc[BURG_MAXC];
            double *o = ceps + (row0 + f) * BURG_MAXC;
#pragma unroll
            for (int n = 1; n < BURG_MAXC; n++) {
                double sum = 0;
#pragma unroll
                for (int k = 1; k < BURG_MAXC; k++) if (k < n) sum += (double)(n - k) * cc[(n - k) & (BURG_MAXC - 1)] * av[k];
                cc[n] = -av[n] - sum / n;
                if (n < ncoef) o[n] = cc[n];
            }
            o[0] = log(alpha);
        }
        __syncwarp();
    }
}

static inline size_t burg_smem_bytes(int w, int s) {
    return sizeof(double) * (2 * (256 + 130 + 130 + BURG_GROUPS * XPAD * 16) + 2 * ((w + 1) & ~1)) + sizeof(int16_t) * (size_t)(8 + (BURG_HALF - 1) * s + w + 1 + 8 + 8);
}

int launch_burg(const BurgParams &B, int src_mode, const BatchDesc &bd, int64_t ntiles, const int16_t *pcm, const float *spec,
                              double *ceps, const double2 *tw, const double2 *ts, const double2 *ti, const double *win, const double *hann,
                              cudaStream_t s, LaunchCtx *lc, std::string &err) {
    if (ntiles <= 0) return CTU_OK;
    if (B.nfft) {                                        // FFT sizes other than 512: the general kernel
        const int M = B.nfft / 2;
        const size_t bytes_any = (size_t)(ANY64_THREADS / 32) * burg_any_doubles(M) * sizeof(double);
        AnyTables64 tb{B.any_tw, B.any_ts, win, B.nfft, B.log2m};
        auto ka = B.dc1 ? k_burg_any<true> : k_burg_any<false>;
        cudaError_t e2 = cudaFuncSetAttribute(ka, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes_any);
        lc->begin("k_burg_any", s);
        if (e2 == cudaSuccess) ka<<<(unsigned)ntiles, ANY64_THREADS, bytes_any, s>>>(B, src_mode, bd, tb, pcm, spec, ceps, hann);
        lc->end(s);
        if (e2 == cudaSuccess) e2 = cudaGetLastError();
        if (e2 != cudaSuccess) { err = std::string("CUDA: ") + cudaGetErrorString(e2) + " (k_burg_any)"; return CTU_ERR_CUDA; }
        return CTU_OK;
    }
    if (B.window & 1) { err = "CTU: the Burg detector path needs an even window length"; return CTU_ERR_UNSUPPORTED; }
    size_t bytes = burg_smem_bytes(B.window, B.wshift);
    if (bytes > 227 * 1024) { err = "CTU: window shift too large for the Burg detector kernel"; return CTU_ERR_UNSUPPORTED; }
    cudaError_t e;
    lc->begin("k_burg", s);
#define CTU_BURG_LAUNCH2(CH, EX, MB, GA)                                                                               \
    e = cudaFuncSetAttribute(k_burg<CH, EX, MB, GA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);           \
    if (e == cudaSuccess)                                                                                                  \
        k_burg<CH, EX, MB, GA><<<(unsigned)(2 * ntiles), BURG_THREADS, bytes, s>>>(B, src_mode, bd, (int)(2 * ntiles), pcm, spec, ceps, tw, ts, ti, win, hann)
#define CTU_BURG_LAUNCH(CH, EX, MB)                                                                                    \
    if (gena) { CTU_BURG_LAUNCH2(CH, EX, 2, true); } else { CTU_BURG_LAUNCH2(CH, EX, MB, false); }
    // the general exponent only matters where the detector's input is expanded (NR source, hwss / fwss)
    const bool gena = (src_mode == BURG_SRC_NR && B.expand && B.a_kind == 0);
    // 25 samples per thread: 128 registers = four CTAs per SM; 32 samples per thread (window up to 512): three
    if (B.window == 400) { CTU_BURG_LAUNCH(25, true, 4); }
    else if (B.window == 512) { CTU_BURG_LAUNCH(32, true, 2); }
    else if (B.window <= 400) { CTU_BURG_LAUNCH(25, false, 3); }
    else { CTU_BURG_LAUNCH(32, false, 2); }
#undef CTU_BURG_LAUNCH2
#undef CTU_BURG_LAUNCH
    lc->end(s);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { err = std::string("CUDA: ") + cudaGetErrorString(e) + " (k_burg)"; return CTU_ERR_CUDA; }
    return CTU_OK;
}

// ------------------------------------------------------------------------------------------
// K5: cepstral detector (src/vdet/CepstralDet.h:134-194), sequential per utterance
// ------------------------------------------------------------------------------------------
// One WARP per utterance: the warp stages blocks of 32 frames of cepstra in shared memory (coalesced, all loads
// in flight at once) and lane 0 runs the sequential state machine out of shared memory.  With one thread per
// utterance every frame waited for its own HBM / L2 round trip (2 ms per launch whatever the batch size, which
// dominated the chunked host path).
constexpr int CEPDET_WARPS = 4;
__global__ void __launch_bounds__(32 * CEPDET_WARPS)
k_cepdet(const __grid_constant__ BurgParams B, const int *__restrict__ nframes, const int64_t *__restrict__ row_off, int u0,
         int n_utts, const double *__restrict__ ceps, uint8_t *__restrict__ flags) {
    __shared__ double stage[CEPDET_WARPS][32 * BURG_MAXC];
    __shared__ uint8_t sflag[CEPDET_WARPS][32];
    const int wv = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * CEPDET_WARPS + wv;
    if (i >= n_utts) return;
    const int u = u0 + i;
    const int T = nframes[u];
    const int nc = B.ncoef_nr;
    const double *cp0 = ceps + row_off[u] * BURG_MAXC;
    uint8_t *fl = flags + row_off[u];
    double c0[BURG_MAXC];
    double dMean = 0, dMean2 = 0, dVar = 0, thr = 0;
    for (int tb = 0; tb < T; tb += 32) {
        const int nb = min(32, T - tb);
        for (int k = lane; k < nb * BURG_MAXC; k += 32) stage[wv][k] = cp0[(int64_t)tb * BURG_MAXC + k];
        __syncwarp();
        if (lane == 0) {
            // c0[] stays in registers: every loop over the coefficients is unrolled to BURG_MAXC with k < nc as a predicate (with
            // the run-time bound the array lived in local memory and every access was a dependent L1 round trip: the kernel
            // took 2.7 ms per 10 000 utterances, two thirds of it in those)
            for (int j = 0; j < nb; j++) {
                const int t = tb + j;
                const double *cp = stage[wv] + j * BURG_MAXC;
                bool res = false;
                if (t == 0) {
#pragma unroll
                    for (int k = 0; k < BURG_MAXC; k++) if (k < nc) c0[k] = cp[k];
                } else {
                    if (t == 1) {
#pragma unroll
                        for (int k = 0; k < BURG_MAXC; k++) if (k < nc) c0[k] = (c0[k] + cp[k]) / 2.0;
                    }
                    double sum = 0;
#pragma unroll
                    for (int k = 1; k < BURG_MAXC; k++) if (k < nc) { double d = cp[k] - c0[k]; sum += d * d; }
                    const double dist = 4.3429 * sqrt(2 * sum);
                    if (t == 1) { dMean = dist; dMean2 = dist * dist; thr = dMean; }
                    else {
                        res = (t > B.ninit) && (dist >= thr);
                        if (!res) {
#pragma unroll
                            for (int k = 0; k < BURG_MAXC; k++) if (k < nc) c0[k] = B.P * c0[k] + (1 - B.P) * cp[k];
                            dMean = B.Q * dMean + (1 - B.Q) * dist;
                            dMean2 = B.Q * dMean2 + (1 - B.Q) * dist * dist;
                            dVar = dMean2 - dMean * dMean;
                            thr = dMean + 2.0 * sqrt(dVar);
                        }
                    }
                }
                sflag[wv][j] = res ? 1 : 0;
            }
        }
        __syncwarp();
        if (lane < nb) fl[tb + lane] = sflag[wv][lane];
        __syncwarp();
    }
}

int launch_cepdet(const BurgParams &B, const int *d_nframes, const int64_t *d_row_off, int u0, int u1, const double *ceps,
                                uint8_t *flags, cudaStream_t s, LaunchCtx *lc, std::string &err) {
    int n = u1 - u0;
    if (n <= 0) return CTU_OK;
    lc->begin("k_cepdet", s);
    k_cepdet<<<(n + CEPDET_WARPS - 1) / CEPDET_WARPS, 32 * CEPDET_WARPS, 0, s>>>(B, d_nframes, d_row_off, u0, n, ceps, flags);
    lc->end(s);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { err = std::string("CUDA: ") + cudaGetErrorString(e) + " (k_cepdet)"; return CTU_ERR_CUDA; }
    return CTU_OK;
}

}  // namespace ctu
#endif
