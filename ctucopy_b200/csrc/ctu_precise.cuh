// fp64 variant of the frame pipeline for the configurations whose REFERENCE arithmetic
// cancels many digits, so that fp32 intermediates cannot reach the parity tolerance:
//   * noise reduction applied to filter-bank outputs (-nr_when afterFB): |Y - b*Navg| and
//     exten's Yavg = |Y - Navg| lose 3-5 digits on stationary segments (src/nr/nr.cc:110-132,
//     245-249, 352-356);
//   * LPC from squared band powers (lpa / lpc without the ^0.33 law, src/fea/fea_impl.cc:
//     165-169): the autocorrelation matrix is ill-conditioned.
// B200 issues FP64 FMAs at half the FP32 rate, so this path costs ~3x, not 30x.
// Layout: 16 threads per frame (ctu_fft.cuh in double), 8 frames per pass, everything a
// frame needs stays inside its group: FB bands, cepstral rows and autocorrelation lags are
// dealt round-robin to the group's 16 threads.
#ifndef CTU_PRECISE_CUH
#define CTU_PRECISE_CUH

#include "ctu_kernels.cuh"
#include "ctu_nr_params.cuh"

namespace ctu {

constexpr int P64_THREADS = 128;
constexpr int P64_GROUPS = P64_THREADS / GROUP;
constexpr int P64_ROW = 264;          // doubles per spectrum row
enum { SRC64_PCM = 0, SRC64_FB = 1, SRC64_SPEC = 2 };
enum { DST64_FB = 0, DST64_FEA = 1 };

struct Tables64 {
    const double2 *tw256, *twsplit;
    const double *win;
    const double *w;       // packed filter-bank taps (true scale)
    const double *m2;      // second-stage matrix [nrows][nb]
    const double *lift;    // lpc lifter [ncep+1]
    // FFT sizes other than 512: k_frames64_any (nfft == 0: the specialised kernel)
    int nfft, log2m;
    const double2 *any_tw, *any_ts;
    int spitch;            // floats per row of the fp32 spectrum matrix (SRC64_SPEC)
};

// non-template entry points (defined in ctu_precise.cu, where the kernels below are compiled)
int launch_frames64(int src_kind, int dst_kind, int kind, const FrameParams &P, const BatchDesc &bd, const Tables64 &tb, int64_t ntiles, const int16_t *pcm,
                    const double *src64, const float *spec, double *dst64, float *dst, cudaStream_t stream, LaunchCtx *lc, std::string &err);
int launch_nr_scan64(const NrParams &N, const int *d_nframes, const int64_t *d_row_off, int u0, int u1, int size, double *X,
                     const uint8_t *flags, double *carry, cudaStream_t s, LaunchCtx *lc, std::string &err);

#ifdef CTU_PRECISE_IMPL
template <int LANES> __device__ __forceinline__ double lanes_sum_d(double v) {
    if (LANES == 16) return group_sum16d(v);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Everything after the spectrum row (energies, filter bank, features) for one frame held by LANES threads: shared by the
// 512-point kernel (16 threads per frame) and the general one (a warp per frame).  pr: spectrum row [nbins] (fp64).
template <int SRC, int DST, int KIND, int LANES>
__device__ __forceinline__ void frames64_tail(const FrameParams &P, const Tables64 &tb, int nbins, const double *pr, double *sY, double *sR, int c,
                                              bool active, int64_t row, const double *__restrict__ src, double *__restrict__ dst64,
                                              float *__restrict__ dst) {
    const int nb = P.nb;
    if ((SRC == SRC64_PCM || SRC == SRC64_SPEC) && (P.energy_mode == EN_NR || P.energy_mode == EN_IN)) {
        // energy of the half spectrum (src/nr/nr.cc:36-45 squares the stored values; src/io/in.cc:403-413 sums power)
        const bool square = (P.energy_mode == EN_NR) || P.take_sqrt;
        double acc = 0;
        if (active) for (int k = c; k < nbins; k += LANES) {
            double v = pr[k];
            if (square) v *= v;
            if (k == 0 || k == nbins - 1) v *= 0.5;
            acc += v;
        }
        acc = lanes_sum_d<LANES>(acc);
        if (active && c == 0) P.energy[row] = (float)log(acc * 2.0);
    }
    if (SRC == SRC64_PCM || SRC == SRC64_SPEC) {
        // filter bank: bands dealt round-robin to the group's threads, sequential sum
        // over the taps in the reference's order (src/fea/fb.cc:76-83)
        if (active) {
            for (int b = c; b < nb; b += LANES) {
                const int lo_ = P.lo[b], hi_ = P.hi[b];
                const double *wp = tb.w + P.woff[b] - lo_;
                double acc = 0;
                for (int k = lo_; k <= hi_; k++) acc += pr[k] * wp[k];
                if (P.inld) acc = pow(acc, 0.33);
                sY[b] = acc;
            }
        }
    } else {
        if (active) for (int b = c; b < nb; b += LANES) sY[b] = src[row * nb + b];
    }
    __syncwarp();
    if (DST == DST64_FB) {
        if (active) for (int b = c; b < nb; b += LANES) dst64[row * nb + b] = sY[b];
        __syncwarp();
        return;
    }
    // ---- features --------------------------------------------------------------------------
    float *orow = dst + row * P.out_stride;
    double *orow64 = dst64 ? dst64 + row * P.out_stride : nullptr;
    if (KIND == KIND_SPEC || KIND == KIND_LOGSPEC || KIND == KIND_TRAPLOG) {
        if (P.energy_mode == EN_BANDS && active && c == 0) {
            double acc = 0.5 * sY[0] * sY[0];
            for (int b = 1; b < nb - 1; b++) acc += sY[b] * sY[b];
            acc += 0.5 * sY[nb - 1] * sY[nb - 1];
            P.energy[row] = (float)log(acc * 2.0);
        }
        if (active) for (int b = c; b < nb; b += LANES) {
            double v = (KIND == KIND_SPEC) ? sY[b] : log(sY[b]);
            orow[b] = (float)v;
            if (orow64) orow64[b] = v;
        }
    } else if (KIND == KIND_DCTC) {
        if (active) for (int b = c; b < nb; b += LANES) sY[b] = log(sY[b]);
        __syncwarp();
        if (active) for (int i = c; i < P.nrows; i += LANES) {
            const double *m = tb.m2 + i * nb;
            double acc = 0;
            for (int k = 0; k < nb; k++) acc += sY[k] * m[k];
            orow[i] = (float)acc;
            if (orow64) orow64[i] = acc;
        }
    } else {
        const int p = P.lporder;
        if (active && P.lpa_square) for (int b = c; b < nb; b += LANES) sY[b] = sY[b] * sY[b];
        __syncwarp();
        if (active) for (int k = c; k <= p; k += LANES) {
            const double *m = tb.m2 + k * nb;
            double acc = 0;
            for (int n = 0; n < nb; n++) acc += sY[n] * m[n];
            sR[k] = acc;
        }
        __syncwarp();
        if (active && c == 0) {
            if (P.energy_mode == EN_LPC) P.energy[row] = (float)log(sR[0]);
            double a[MAXR], aa[MAXR];
            double Pe = sR[0];
            double rc = -sR[1] / sR[0];
            Pe = Pe * (1 - rc * rc);
            a[0] = aa[0] = 1.0; a[1] = aa[1] = rc;
            for (int ik = 2; ik <= p; ik++) {
                double dm = sR[ik];
                for (int n = 1; n <= ik - 1; n++) dm += aa[n] * sR[ik - n];
                rc = -dm / Pe;
                a[ik] = rc;
                for (int n = 1; n <= ik - 1; n++) a[n] = aa[n] + rc * aa[ik - n];
                for (int n = 1; n <= ik; n++) aa[n] = a[n];
                Pe = Pe * (1 - rc * rc);
            }
            if (KIND == KIND_LPA) {
                for (int i = 1; i <= p; i++) { orow[i - 1] = (float)a[i]; if (orow64) orow64[i - 1] = a[i]; }
            } else {
                double cc[MAXR];
                const int N = P.ncep;
                cc[0] = log(Pe);
                for (int n = 1; n <= N; n++) {
                    double sum = 0;
                    if (n <= p) {
                        for (int k = 1; k <= n - 1; k++) sum += (n - k) * cc[n - k] * a[k];
                        cc[n] = -a[n] - sum / n;
                    } else {
                        for (int k = 1; k <= p; k++) sum += (n - k) * cc[n - k] * a[k];
                        cc[n] = -sum / n;
                    }
                }
                for (int n = 1; n <= N; n++) { double v = cc[n] * tb.lift[n]; orow[n - 1] = (float)v; if (orow64) orow64[n - 1] = v; }
                if (P.c0_last) { orow[N] = (float)cc[0]; if (orow64) orow64[N] = cc[0]; }
            }
        }
    }
    __syncwarp();
}

template <int SRC, int DST, int KIND>
__global__ void __launch_bounds__(P64_THREADS)
k_frames64(const __grid_constant__ FrameParams P, BatchDesc bd, Tables64 tb, const int16_t *__restrict__ pcm, const double *__restrict__ src,
           const float *__restrict__ spec, double *__restrict__ dst64, float *__restrict__ dst) {
    extern __shared__ __align__(16) double smd[];
    const int tid = threadIdx.x;
    const int w = P.window, s = P.wshift, nb = P.nb;
    cpx<double> *sTw = reinterpret_cast<cpx<double> *>(smd);          // 256
    cpx<double> *sTs = sTw + 256;                                    // 130
    cpx<double> *sX = sTs + 130;                                     // groups * 272
    double *sP = reinterpret_cast<double *>(sX + P64_GROUPS * XPAD * 16);   // groups * P64_ROW
    double *sYa = sP + P64_GROUPS * P64_ROW;                         // groups * 64
    double *sRa = sYa + P64_GROUPS * 64;                             // groups * 64
    if (SRC == SRC64_PCM) {
        for (int i = tid; i < 256; i += P64_THREADS) sTw[i] = mk<double>(tb.tw256[i].x, tb.tw256[i].y);
        for (int i = tid; i < 129; i += P64_THREADS) sTs[i] = mk<double>(tb.twsplit[i].x, tb.twsplit[i].y);
    }
    __syncthreads();
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int nf = min(TILE_F, bd.nframes[u] - t0);
    const int64_t row0 = bd.row_off[u] + t0;
    const int64_t g0 = bd.pcm_off[u];
    const int c = tid & (GROUP - 1), grp = tid / GROUP;
    cpx<double> *xch = sX + grp * (XPAD * 16);
    double *pr = sP + grp * P64_ROW;
    double *sY = sYa + grp * 64;
    double *sR = sRa + grp * 64;
#pragma unroll 1
    for (int pass = 0; pass < TILE_F / P64_GROUPS; pass++) {
        const int f = pass * P64_GROUPS + grp;
        const bool active = f < nf;
        if (SRC == SRC64_SPEC) {
            // (noise-reduced) fp32 spectrum from HBM, widened
            if (active) for (int k = c; k < NBIN; k += GROUP) pr[k] = (double)spec[(row0 + f) * tb.spitch + k];
            __syncwarp();
        }
        if (SRC == SRC64_PCM) {
            cpx<double> a[16];
            if (active) {
                const int64_t fs0 = g0 + (int64_t)(t0 + f) * s;
                const bool at_start = (t0 + f) == 0;
                double sum = 0;
#pragma unroll
                for (int n1 = 0; n1 < 16; n1++) {
                    int i0 = 32 * n1 + 2 * c;
                    double y0 = 0, y1 = 0;
                    if (i0 < w) {
                        double xm = (i0 == 0) ? (at_start ? 0.0 : (double)pcm[fs0 - 1]) : (double)pcm[fs0 + i0 - 1];
                        double x0 = (double)pcm[fs0 + i0];
                        y0 = tb.win[i0] * (x0 - (double)P.preem * xm);
                        if (i0 + 1 < w) y1 = tb.win[i0 + 1] * ((double)pcm[fs0 + i0 + 1] - (double)P.preem * x0);
                    }
                    a[n1] = mk<double>(y0, y1);
                    sum += y0 + y1;
                }
                if (P.remove_dc) {
                    double mean = group_sum16d(sum) / (double)w;
#pragma unroll
                    for (int n1 = 0; n1 < 16; n1++) {
                        int i0 = 32 * n1 + 2 * c;
                        if (i0 < w) a[n1].x -= mean;
                        if (i0 + 1 < w) a[n1].y -= mean;
                    }
                }
                fft256_pass1(a, c, sTw, xch);
            }
            __syncwarp();
            if (active) fft256_pass2(a, c, xch);
            __syncwarp();
            if (active) fft256_store_linear(a, c, xch);
            __syncwarp();
            if (active) {
                cpx<double> lo[8], hi[8], mid;
                rfft_split(xch, c, sTs, lo, hi, mid);
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    int k = c + 16 * j;
                    double pl = lo[j].x * lo[j].x + lo[j].y * lo[j].y;
                    double ph = hi[j].x * hi[j].x + hi[j].y * hi[j].y;
                    if (k == 0 && P.remove_dc) pl = 1e-10;
                    if (P.take_sqrt) { pl = sqrt(pl); ph = sqrt(ph); }
                    pr[k] = pl;
                    pr[NC - k] = ph;
                }
                if (c == 0) {
                    double pm = mid.x * mid.x + mid.y * mid.y;
                    pr[128] = P.take_sqrt ? sqrt(pm) : pm;
                }
            }
            __syncwarp();
        }
        frames64_tail<SRC, DST, KIND, GROUP>(P, tb, NBIN, pr, sY, sR, c, active, row0 + f, src, dst64, dst);
    }
}

// The same chain for FFT sizes other than 512 (and for -remove_dc1 at any size): one warp per frame, front end from
// ctu_any64.cuh.  DC1: PCM source under -remove_dc1, the frame is built from the de-meaned ring (P.dc1).
template <int SRC, int DST, int KIND, bool DC1 = false>
__global__ void __launch_bounds__(ANY64_THREADS)
k_frames64_any(const __grid_constant__ FrameParams P, BatchDesc bd, Tables64 tb, const int16_t *__restrict__ pcm, const double *__restrict__ src,
               const float *__restrict__ spec, double *__restrict__ dst64, float *__restrict__ dst) {
    extern __shared__ __align__(16) double smd[];
    const int lane = threadIdx.x & 31, wv = threadIdx.x >> 5;
    const int nfft = tb.nfft, M = nfft >> 1, nbins = M + 1;
    double *base = smd + (size_t)wv * (2 * any64_zslots(M) + (M + 4) + 64 + 64);
    cpx<double> *z = reinterpret_cast<cpx<double> *>(base);                    // padded (ctu_any64.cuh)
    double *pr = base + 2 * any64_zslots(M);
    double *sY = pr + (M + 4);
    double *sR = sY + 64;
    const AnyTables64 at{tb.any_tw, tb.any_ts, tb.win, nfft, tb.log2m};
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int nf = min(TILE_F, bd.nframes[u] - t0);
    const int64_t row0 = bd.row_off[u] + t0;
    for (int f = wv; f < nf; f += ANY64_THREADS / 32) {
        if (SRC == SRC64_SPEC) {
            for (int k = lane; k < nbins; k += 32) pr[k] = (double)spec[(row0 + f) * tb.spitch + k];
            __syncwarp();
        }
        if (SRC == SRC64_PCM) {
            any64_analysis<DC1>(z, at, pcm + bd.pcm_off[u] + (int64_t)(t0 + f) * P.wshift, (t0 + f) == 0, P.window, (double)P.preem, P.remove_dc, lane,
                                DC1 ? P.dc1 + row0 + f : nullptr, t0 + f, P.wshift);
            for (int k = lane; k <= M; k += 32) {
                const cpx<double> X = any64_bin(z, at, k);
                double pw = X.x * X.x + X.y * X.y;
                if (k == 0 && P.remove_dc) pw = 1e-10;                 // fixed floor (src/io/in.cc:390)
                pr[k] = P.take_sqrt ? sqrt(pw) : pw;
            }
            __syncwarp();
        }
        frames64_tail<SRC, DST, KIND, 32>(P, tb, nbins, pr, sY, sR, lane, true, row0 + f, src, dst64, dst);
    }
}

static inline size_t p64_smem_bytes() {
    return sizeof(double) * (2 * (256 + 130 + P64_GROUPS * XPAD * 16) + P64_GROUPS * (P64_ROW + 64 + 64));
}

template <int SRC, int DST, int KIND>
static int launch_frames64_t(const FrameParams &P, const BatchDesc &bd, const Tables64 &tb, int64_t ntiles, const int16_t *pcm,
                             const double *src, const float *spec, double *dst64, float *dst, cudaStream_t s, LaunchCtx *lc,
                             std::string &err) {
    if (ntiles <= 0) return CTU_OK;
    if (tb.nfft) {
        const size_t bytes_any = (size_t)(ANY64_THREADS / 32) * (2 * any64_zslots(tb.nfft / 2) + tb.nfft / 2 + 4 + 128) * sizeof(double);
        auto ka = k_frames64_any<SRC, DST, KIND>;
        if constexpr (SRC == SRC64_PCM) { if (P.dc1) ka = k_frames64_any<SRC, DST, KIND, true>; }
        cudaError_t e2 = cudaFuncSetAttribute(ka, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes_any);
        if (e2 == cudaSuccess) {
            lc->begin(SRC == SRC64_PCM ? (DST == DST64_FB ? "k_frames64_any<pcm,fb>" : "k_frames64_any<pcm,fea>")
                      : SRC == SRC64_SPEC ? (DST == DST64_FB ? "k_frames64_any<spec,fb>" : "k_frames64_any<spec,fea>") : "k_frames64_any<fb,fea>", s);
            ka<<<(unsigned)ntiles, ANY64_THREADS, bytes_any, s>>>(P, bd, tb, pcm, src, spec, dst64, dst);
            lc->end(s);
            e2 = cudaGetLastError();
        }
        if (e2 != cudaSuccess) { err = std::string("CUDA: ") + cudaGetErrorString(e2) + " (k_frames64_any)"; return CTU_ERR_CUDA; }
        return CTU_OK;
    }
    size_t bytes = p64_smem_bytes();
    auto kern = k_frames64<SRC, DST, KIND>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) {
        lc->begin(SRC == SRC64_PCM ? (DST == DST64_FB ? "k_frames64<pcm,fb>" : "k_frames64<pcm,fea>")
                  : SRC == SRC64_SPEC ? (DST == DST64_FB ? "k_frames64<spec,fb>" : "k_frames64<spec,fea>") : "k_frames64<fb,fea>", s);
        kern<<<(unsigned)ntiles, P64_THREADS, bytes, s>>>(P, bd, tb, pcm, src, spec, dst64, dst);
        lc->end(s);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) { err = std::string("CUDA: ") + cudaGetErrorString(e) + " (k_frames64)"; return CTU_ERR_CUDA; }
    return CTU_OK;
}

template <int SRC, int DST>
static int launch_frames64_k(int kind, const FrameParams &P, const BatchDesc &bd, const Tables64 &tb, int64_t nt, const int16_t *pcm,
                             const double *src, const float *spec, double *dst64, float *dst, cudaStream_t s, LaunchCtx *lc,
                             std::string &err) {
    switch (kind) {
        case KIND_SPEC: return launch_frames64_t<SRC, DST, KIND_SPEC>(P, bd, tb, nt, pcm, src, spec, dst64, dst, s, lc, err);
        case KIND_LOGSPEC: return launch_frames64_t<SRC, DST, KIND_LOGSPEC>(P, bd, tb, nt, pcm, src, spec, dst64, dst, s, lc, err);
        case KIND_DCTC: return launch_frames64_t<SRC, DST, KIND_DCTC>(P, bd, tb, nt, pcm, src, spec, dst64, dst, s, lc, err);
        case KIND_LPA: return launch_frames64_t<SRC, DST, KIND_LPA>(P, bd, tb, nt, pcm, src, spec, dst64, dst, s, lc, err);
        case KIND_LPC: return launch_frames64_t<SRC, DST, KIND_LPC>(P, bd, tb, nt, pcm, src, spec, dst64, dst, s, lc, err);
        case KIND_TRAPLOG: return launch_frames64_t<SRC, DST, KIND_TRAPLOG>(P, bd, tb, nt, pcm, src, spec, dst64, dst, s, lc, err);
    }
    err = "CTU: bad kind";
    return CTU_ERR_CONFIG;
}

// ---- fp64 noise-reduction scan over band values (same recursions as k_nr_scan, written as
// the reference writes them; cancellation is harmless at 53 bits) ----------------------------
__global__ void __launch_bounds__(128)
k_nr_scan64(const __grid_constant__ NrParams N, const int *__restrict__ nframes, const int64_t *__restrict__ row_off, int u0, int n_utts,
            int size, double *X, const uint8_t *__restrict__ flags, double *__restrict__ carry) {
    // carry (opt-in list semantics of hwss / fwss / 2fwss, see k_nr_scan_carry): one thread per bin walks the utterances of the
    // range in order, a file's noise estimate starts from the enhanced last frame of the file before it
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (carry ? (int64_t)size : (int64_t)n_utts * size)) return;
    const int bin = (int)(gid % size);
    const int ufirst = carry ? u0 : u0 + (int)(gid / size), ulast = carry ? u0 + n_utts : ufirst + 1;
    const double p = N.pd, a = N.ad, b = (double)N.b;
    double cv = carry ? carry[bin] : 0.0;
    for (int u = ufirst; u < ulast; u++) {
    const int T = nframes[u];
    if (T <= 0) continue;
    double *x = X + row_off[u] * size + bin;
    const uint8_t *fl = flags ? flags + row_off[u] : nullptr;
    double Navg = (N.mode == NR_EXTEN) ? 0.95 : 0.0, Yavg = 0.05, Nravg = 0.0;
    if (carry && N.mode != NR_EXTEN) Navg = (N.mode == NR_2FWSS || N.a_kind == 1) ? cv : (N.a_kind == 2) ? __dmul_rn(cv, cv) : pow(cv, a);
    // Every product and sum below is rounded on its own (__dmul_rn / __dadd_rn / __dsub_rn: no FMA contraction), in the
    // reference's order (src/nr/nr.cc:95-140, 224-261, 331-369, 397-442).  This path exists for fidelity: where the
    // subtraction cancels almost everything (x - H x with H = 1 - 1e-13) the reference's result IS its rounding pattern --
    // a fused x - H x gives the mathematically better value, 1 % away from what the reference writes (found by the
    // 200-set sweep: TRAP-DCT of a band that exten takes from 21.9 to 1.9e-12).
    const double omp = __dsub_rn(1.0, p);
    for (int t = 0; t < T; t++) {
        double xi = x[(int64_t)t * size];
        if (N.mode == NR_EXTEN) {
            double H;
            if (N.a_kind == 1) H = Navg / __dadd_rn(Navg, Yavg);
            else if (N.a_kind == 2) H = Navg / sqrt(__dadd_rn(__dmul_rn(Navg, Navg), __dmul_rn(Yavg, Yavg)));
            else H = Navg / pow(__dadd_rn(pow(Navg, a), pow(Yavg, a)), 1. / a);
            const double Nn = __dmul_rn(H, xi);
            Navg = __dadd_rn(__dmul_rn(p, Navg), __dmul_rn(omp, Nn));
            Yavg = (xi > Navg) ? __dsub_rn(xi, Navg) : __dsub_rn(Navg, xi);
            xi = __dsub_rn(xi, Nn);
        } else {
            const int ninit = (N.mode == NR_HWSS) ? N.initsegs - (t + 1) : N.initsegs - t;
            const bool upd = (fl[t] == 0) || ninit > 0;
            if (N.mode == NR_2FWSS) {
                if (upd) Navg = __dadd_rn(__dmul_rn(p, Navg), __dmul_rn(omp, xi));
                xi = __dsub_rn(xi, Navg); if (xi < 0.) xi = -xi;
                if (upd) Nravg = __dadd_rn(__dmul_rn(p, Nravg), __dmul_rn(omp, xi));
                xi = __dsub_rn(xi, Nravg); if (xi < 0.) xi = -xi;
            } else {
                if (N.a_kind == 2) xi = __dmul_rn(xi, xi); else if (N.a_kind == 0) xi = pow(xi, a);
                if (upd) Navg = __dadd_rn(__dmul_rn(p, Navg), __dmul_rn(omp, xi));
                xi = __dsub_rn(xi, __dmul_rn(b, Navg));
                if (xi < 0.) xi = (N.mode == NR_HWSS) ? 0. : -xi;
                if (N.a_kind == 2) xi = sqrt(xi); else if (N.a_kind == 0) xi = pow(xi, 1.0 / a);
            }
        }
        x[(int64_t)t * size] = xi;
        cv = xi;
    }
    if (N.carry_xform == 1) cv = log(cv); else if (N.carry_xform == 2) cv = __dmul_rn(cv, cv);
    }
    if (carry) carry[bin] = cv;
}

int launch_nr_scan64(const NrParams &N, const int *d_nframes, const int64_t *d_row_off, int u0, int u1, int size, double *X,
                                   const uint8_t *flags, double *carry, cudaStream_t s, LaunchCtx *lc, std::string &err) {
    int64_t n = carry ? (int64_t)size : (int64_t)(u1 - u0) * size;
    if (n <= 0 || u1 <= u0) return CTU_OK;
    lc->begin("k_nr_scan64", s);
    k_nr_scan64<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(N, d_nframes, d_row_off, u0, u1 - u0, size, X, flags, carry);
    lc->end(s);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { err = std::string("CUDA: ") + cudaGetErrorString(e) + " (k_nr_scan64)"; return CTU_ERR_CUDA; }
    return CTU_OK;
}

int launch_frames64(int src_kind, int dst_kind, int kind, const FrameParams &P, const BatchDesc &bd, const Tables64 &tb, int64_t nt, const int16_t *pcm,
                    const double *src64, const float *spec, double *dst64, float *dst, cudaStream_t s, LaunchCtx *lc, std::string &err) {
    const int src = src_kind, dst_k = dst_kind;
    if (src == SRC64_PCM && dst_k == DST64_FB) return launch_frames64_t<SRC64_PCM, DST64_FB, KIND_SPEC>(P, bd, tb, nt, pcm, src64, spec, dst64, dst, s, lc, err);
    if (src == SRC64_FB && dst_k == DST64_FEA) return launch_frames64_k<SRC64_FB, DST64_FEA>(kind, P, bd, tb, nt, pcm, src64, spec, dst64, dst, s, lc, err);
    if (src == SRC64_SPEC && dst_k == DST64_FEA) return launch_frames64_k<SRC64_SPEC, DST64_FEA>(kind, P, bd, tb, nt, pcm, src64, spec, dst64, dst, s, lc, err);
    if (src == SRC64_PCM && dst_k == DST64_FEA) return launch_frames64_k<SRC64_PCM, DST64_FEA>(kind, P, bd, tb, nt, pcm, src64, spec, dst64, dst, s, lc, err);
    err = "CTU: internal: unsupported fp64 chain";
    return CTU_ERR_CONFIG;
}
#endif  // CTU_PRECISE_IMPL

}  // namespace ctu
#endif
