// Cross-frame kernels of the CtuCopy hot path (sm_100a), compiled in their own translation unit (ctu_nr.cu):
//   K2/K3 k_nr_scan / k_nr_scan4   extended spectral subtraction and the VAD-driven hwss / fwss / 2fwss recursions as
//                        standalone kernels (src/nr/nr.cc:86-140, 212-261, 331-369, 397-442): used where the enhanced
//                        spectrum itself is needed in HBM (waveform output, VAD module, general FFT sizes); feature
//                        chains run the same recursion inside k_bank (ctu_bank.cuh)
//   K6    k_vad_*        VAD module: criterion, threshold state machines, majority filter, drop compaction
//                        (src/vad/vad.cc:96-107, 220-294, 329-625, 692-745; src/vad/vad.h:126-175)
//   K9    k_synth_c      (|X|enh, phase of X) -> inverse FFT -> overlap-add in frame order -> floor(x/correction) ->
//                        clip -> int16 (src/io/out.cc:346-451)
// Parameter blocks, the per-frame recursion step (nr_step) and the launcher prototypes: ctu_nr_params.cuh.
#ifndef CTU_NR_KERNELS_CUH
#define CTU_NR_KERNELS_CUH

#include "ctu_nr_params.cuh"

namespace ctu {

// SIZE: row length known at compile time (257 spectrum bins) so that the SCAN_UNROLL loads of
// a block share one base register with immediate offsets; 0 = runtime (band domain)
template <int MODE, int AKIND, int SIZE>
__global__ void __launch_bounds__(256)
k_nr_scan(const __grid_constant__ NrParams N, const int *__restrict__ nframes, const int64_t *__restrict__ row_off, int u0, int n_utts,
          int size_rt, float *X, const uint8_t *__restrict__ flags) {
    const int size = SIZE ? SIZE : size_rt;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (int64_t)n_utts * size) return;
    const int u = u0 + (int)(gid / size), bin = (int)(gid % size);
    const int T = nframes[u];
    float *x = X + row_off[u] * size + bin;
    const uint8_t *fl = (MODE != NR_EXTEN) ? flags + row_off[u] : nullptr;
    // exten: smoothed noise Navg / smoothed speech Yavg start at 0.95 / 0.05 (src/nr/nr.cc:86-93);
    // *ss: the noise estimate of a standalone file starts at 0 (src/nr/nr.cc:212-222)
    ScanState S;
    S.Navg = (MODE == NR_EXTEN) ? 0.95f : 0.f; S.Yavg = 0.05f; S.Nravg = 0.f; S.Nd = 0.95; S.Yd = 0.05;
    int t0 = 0;
    for (; t0 + SCAN_UNROLL <= T; t0 += SCAN_UNROLL) {
        float v[SCAN_UNROLL];
        uint8_t f[SCAN_UNROLL];
        float *xr = x + (int64_t)t0 * size;
#pragma unroll
        for (int j = 0; j < SCAN_UNROLL; j++) {
            v[j] = xr[j * size];
            f[j] = (MODE != NR_EXTEN) ? fl[t0 + j] : 0;
        }
#pragma unroll
        for (int j = 0; j < SCAN_UNROLL; j++) v[j] = nr_step<MODE, AKIND>(N, S, v[j], t0 + j, f[j]);
#pragma unroll
        for (int j = 0; j < SCAN_UNROLL; j++) xr[j * size] = v[j];
    }
    for (; t0 < T; t0++) {
        float *xr = x + (int64_t)t0 * size;
        *xr = nr_step<MODE, AKIND>(N, S, *xr, t0, (MODE != NR_EXTEN) ? fl[t0] : 0);
    }
}

// The 512-point spectrum (rows of SPITCH = 260 floats, 16-byte aligned): a thread owns FOUR consecutive bins and moves
// them with 16-byte loads / stores, SCAN4_UNROLL frames in flight -- 65 threads per utterance.  The last thread's bins
// 257..259 are the pad columns: kept zero.
constexpr int SCAN4_UNROLL = 8;
constexpr int SCAN4_TPU = SPITCH / 4;           // threads per utterance

template <int MODE, int AKIND>
__global__ void __launch_bounds__(256)
k_nr_scan4(const __grid_constant__ NrParams N, const int *__restrict__ nframes, const int64_t *__restrict__ row_off, int u0, int n_utts,
           float *X, const uint8_t *__restrict__ flags) {
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (int64_t)n_utts * SCAN4_TPU) return;
    const int u = u0 + (int)(gid / SCAN4_TPU), q = (int)(gid % SCAN4_TPU);
    const int T = nframes[u];
    float4 *x = reinterpret_cast<float4 *>(X + row_off[u] * SPITCH) + q;
    const uint8_t *fl = (MODE != NR_EXTEN) ? flags + row_off[u] : nullptr;
    const bool last = (q == SCAN4_TPU - 1);       // bins 256 | pad pad pad
    ScanState S[4];
#pragma unroll
    for (int i = 0; i < 4; i++) { S[i].Navg = (MODE == NR_EXTEN) ? 0.95f : 0.f; S[i].Yavg = 0.05f; S[i].Nravg = 0.f; S[i].Nd = 0.95; S[i].Yd = 0.05; }
    int t0 = 0;
    for (; t0 + SCAN4_UNROLL <= T; t0 += SCAN4_UNROLL) {
        float4 v[SCAN4_UNROLL];
        uint8_t f[SCAN4_UNROLL];
        float4 *xr = x + (int64_t)t0 * SCAN4_TPU;
#pragma unroll
        for (int j = 0; j < SCAN4_UNROLL; j++) {
            v[j] = xr[j * SCAN4_TPU];
            f[j] = (MODE != NR_EXTEN) ? fl[t0 + j] : 0;
        }
#pragma unroll
        for (int j = 0; j < SCAN4_UNROLL; j++) {
            v[j].x = nr_step<MODE, AKIND>(N, S[0], v[j].x, t0 + j, f[j]);
            if (!last) {
                v[j].y = nr_step<MODE, AKIND>(N, S[1], v[j].y, t0 + j, f[j]);
                v[j].z = nr_step<MODE, AKIND>(N, S[2], v[j].z, t0 + j, f[j]);
                v[j].w = nr_step<MODE, AKIND>(N, S[3], v[j].w, t0 + j, f[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < SCAN4_UNROLL; j++) xr[j * SCAN4_TPU] = v[j];
    }
    for (; t0 < T; t0++) {
        float4 *xr = x + (int64_t)t0 * SCAN4_TPU;
        float4 v = *xr;
        const uint8_t f = (MODE != NR_EXTEN) ? fl[t0] : 0;
        v.x = nr_step<MODE, AKIND>(N, S[0], v.x, t0, f);
        if (!last) {
            v.y = nr_step<MODE, AKIND>(N, S[1], v.y, t0, f);
            v.z = nr_step<MODE, AKIND>(N, S[2], v.z, t0, f);
            v.w = nr_step<MODE, AKIND>(N, S[3], v.w, t0, f);
        }
        *xr = v;
    }
}

template <int MODE>
static inline void launch_nr_scan_a(const NrParams &N, unsigned grid, cudaStream_t s, const int *d_nframes, const int64_t *d_row_off, int u0,
                                    int n, int size, float *X, const uint8_t *flags, bool vec4) {
    const int ak = (N.a_kind == 1 || MODE == NR_2FWSS) ? 1 : N.a_kind;
    if (vec4) {
        if (ak == 1) k_nr_scan4<MODE, 1><<<grid, 256, 0, s>>>(N, d_nframes, d_row_off, u0, n, X, flags);
        else if (ak == 2) k_nr_scan4<MODE, 2><<<grid, 256, 0, s>>>(N, d_nframes, d_row_off, u0, n, X, flags);
        else k_nr_scan4<MODE, 0><<<grid, 256, 0, s>>>(N, d_nframes, d_row_off, u0, n, X, flags);
        return;
    }
    if (ak == 1) k_nr_scan<MODE, 1, 0><<<grid, 256, 0, s>>>(N, d_nframes, d_row_off, u0, n, size, X, flags);
    else if (ak == 2) k_nr_scan<MODE, 2, 0><<<grid, 256, 0, s>>>(N, d_nframes, d_row_off, u0, n, size, X, flags);
    else k_nr_scan<MODE, 0, 0><<<grid, 256, 0, s>>>(N, d_nframes, d_row_off, u0, n, size, X, flags);
}

// K2c: hwss / fwss / 2fwss with the reference's LIST semantics (opt-in: ctu_set_option "ss_carry").  hwssNR / dfwssNR::new_file
// (src/nr/nr.cc:212-222, 397-408) start a file's noise estimate from whatever the shared spectrum buffer holds: the ENHANCED
// last frame of the file before it (zeros for the first file of a process).  That chains every utterance to the one before, so
// the only parallelism left is the bins: one thread per bin walks the utterances of the range in list order, `carry` holds the
// buffer between ranges, plans and calls.  Waveform output: sigOUT::save_frame negates the Nyquist bin in that buffer when
// its phase is not 0 (src/io/out.cc:414) -- cspec (the stored complex spectrum) gives the sign.
constexpr int CARRY_UNROLL = 8;
template <int MODE, int AKIND>
__global__ void __launch_bounds__(128)
k_nr_scan_carry(const __grid_constant__ NrParams N, const int *__restrict__ nframes, const int64_t *__restrict__ row_off, int u0, int n_utts,
                int size, int pitch, float *X, const uint8_t *__restrict__ flags, float *__restrict__ carry, const float2 *__restrict__ cspec) {
    const int bin = blockIdx.x * blockDim.x + threadIdx.x;
    if (bin >= size) return;
    float cv = carry[bin];
    for (int i = 0; i < n_utts; i++) {
        const int u = u0 + i, T = nframes[u];
        if (T <= 0) continue;
        ScanState S;
        S.Navg = (MODE == NR_2FWSS || AKIND == 1) ? cv : (AKIND == 2) ? cv * cv : powf(cv, N.a);
        S.Yavg = 0.05f; S.Nravg = 0.f; S.Nd = 0.95; S.Yd = 0.05;
        float *x = X + row_off[u] * pitch + bin;
        const uint8_t *fl = flags + row_off[u];
        for (int t0 = 0; t0 < T; t0 += CARRY_UNROLL) {
            float v[CARRY_UNROLL];
            uint8_t f[CARRY_UNROLL];
#pragma unroll
            for (int j = 0; j < CARRY_UNROLL; j++) {
                const int t = min(t0 + j, T - 1);
                v[j] = x[(int64_t)t * pitch];
                f[j] = fl[t];
            }
#pragma unroll
            for (int j = 0; j < CARRY_UNROLL; j++)
                if (t0 + j < T) {
                    cv = nr_step<MODE, AKIND>(N, S, v[j], t0 + j, f[j]);
                    x[(int64_t)(t0 + j) * pitch] = cv;
                }
        }
        if (cspec && bin == size - 1 && cspec[(row_off[u] + T - 1) * (int64_t)size + bin].x < 0.f) cv = -cv;
    }
    carry[bin] = cv;
}

template <int MODE>
static inline void launch_nr_scan_carry_a(const NrParams &N, cudaStream_t s, const int *d_nframes, const int64_t *d_row_off, int u0, int n, int size,
                                          int pitch, float *X, const uint8_t *flags, float *carry, const float2 *cspec) {
    const int ak = (N.a_kind == 1 || MODE == NR_2FWSS) ? 1 : N.a_kind;
    const unsigned grid = (unsigned)((size + 127) / 128);
    if (ak == 1) k_nr_scan_carry<MODE, 1><<<grid, 128, 0, s>>>(N, d_nframes, d_row_off, u0, n, size, pitch, X, flags, carry, cspec);
    else if (ak == 2) k_nr_scan_carry<MODE, 2><<<grid, 128, 0, s>>>(N, d_nframes, d_row_off, u0, n, size, pitch, X, flags, carry, cspec);
    else k_nr_scan_carry<MODE, 0><<<grid, 128, 0, s>>>(N, d_nframes, d_row_off, u0, n, size, pitch, X, flags, carry, cspec);
}

int launch_nr_scan_carry(const NrParams &N, const int *d_nframes, const int64_t *d_row_off, int u0, int u1, int size, int pitch, float *X,
                         const uint8_t *flags, float *carry, const float2 *cspec, cudaStream_t s, LaunchCtx *lc, std::string &err) {
    if (u1 <= u0) return CTU_OK;
    lc->begin("k_nr_scan_carry", s);
    switch (N.mode) {
        case NR_HWSS: launch_nr_scan_carry_a<NR_HWSS>(N, s, d_nframes, d_row_off, u0, u1 - u0, size, pitch, X, flags, carry, cspec); break;
        case NR_FWSS: launch_nr_scan_carry_a<NR_FWSS>(N, s, d_nframes, d_row_off, u0, u1 - u0, size, pitch, X, flags, carry, cspec); break;
        default: launch_nr_scan_carry_a<NR_2FWSS>(N, s, d_nframes, d_row_off, u0, u1 - u0, size, pitch, X, flags, carry, cspec); break;
    }
    lc->end(s);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { err = std::string("CUDA: ") + cudaGetErrorString(e) + " (k_nr_scan_carry)"; return CTU_ERR_CUDA; }
    return CTU_OK;
}

// size: bins per row; pitch: floats per row (SPITCH for the 512-point spectrum, else = size)
int launch_nr_scan(const NrParams &N, const int *d_nframes, const int64_t *d_row_off, int u0, int u1, int size, int pitch, float *X,
                                 const uint8_t *flags, cudaStream_t s, LaunchCtx *lc, std::string &err) {
    const bool vec4 = (size == NBIN && pitch == SPITCH);
    if (!vec4 && pitch != size) { err = "CTU: spectrum pitch not supported by the scan"; return CTU_ERR_CONFIG; }
    int64_t n = (int64_t)(u1 - u0) * (vec4 ? SCAN4_TPU : size);
    if (n <= 0) return CTU_OK;
    const unsigned grid = (unsigned)((n + 255) / 256);
    lc->begin("k_nr_scan", s);
    switch (N.mode) {
        case NR_EXTEN: launch_nr_scan_a<NR_EXTEN>(N, grid, s, d_nframes, d_row_off, u0, u1 - u0, size, X, flags, vec4); break;
        case NR_HWSS: launch_nr_scan_a<NR_HWSS>(N, grid, s, d_nframes, d_row_off, u0, u1 - u0, size, X, flags, vec4); break;
        case NR_FWSS: launch_nr_scan_a<NR_FWSS>(N, grid, s, d_nframes, d_row_off, u0, u1 - u0, size, X, flags, vec4); break;
        default: launch_nr_scan_a<NR_2FWSS>(N, grid, s, d_nframes, d_row_off, u0, u1 - u0, size, X, flags, vec4); break;
    }
    lc->end(s);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { err = std::string("CUDA: ") + cudaGetErrorString(e) + " (k_nr_scan)"; return CTU_ERR_CUDA; }
    return CTU_OK;
}

// ------------------------------------------------------------------------------------------
// K6: VAD module
// ------------------------------------------------------------------------------------------
// energy criterion: one warp per frame over the (post-NR) spectrum
__global__ void k_vad_energy(const __grid_constant__ VadParams V, const float *__restrict__ spec, int64_t row0, int64_t nrows,
                             double *__restrict__ cri) {
    const int64_t r = row0 + (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= row0 + nrows) return;
    const int lane = threadIdx.x & 31;
    const float *x = spec + r * V.spitch;
    double e = 0;
    for (int k = lane; k < V.nbins; k += 32) { double v = (double)x[k]; e += v * v; }
    for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
    if (lane == 0) cri[r] = V.energy_db ? 10.0 * log10(DBL_MIN + e) : e;
}

// thresholds + background update + majority filter (src/vad/vad.cc:249-276, 300-420, src/vad/vad.h:126-175).
// One WARP per utterance, like k_cepdet: the warp stages the criterion inputs of 32 frames in shared memory (coalesced, all
// loads in flight at once), lane 0 runs the sequential state machines out of shared memory -- same operations in the same
// order as before -- and the majority filter runs one row per lane.  With one thread per utterance every frame waited for
// its own memory round trip: 1-3 ms per launch whatever the batch size, which the chunked host path paid per chunk.
constexpr int VADSCAN_WARPS = 4;
__global__ void __launch_bounds__(VADSCAN_WARPS * 32)
k_vad_scan(const __grid_constant__ VadParams V, const int *__restrict__ nframes, const int64_t *__restrict__ row_off, int u0,
           int n_utts, const double *__restrict__ cri_frame, const double *__restrict__ ceps,
           const double *__restrict__ fea, int fea_dim /* row pitch */, uint8_t *__restrict__ vad0_tmp, uint8_t *__restrict__ vad_out,
           uint8_t *__restrict__ keep) {
    extern __shared__ __align__(16) double sm_vs[];
    const int lane = threadIdx.x & 31, wv = threadIdx.x >> 5;
    const int i = blockIdx.x * VADSCAN_WARPS + wv;
    if (i >= n_utts) return;
    const int u = u0 + i;
    const int T = nframes[u];
    const int64_t R0 = row_off[u];
    const int cn = (V.cri == VCRI_ENERGY) ? 1 : V.cep_n;
    double *sc = sm_vs + (size_t)wv * (32 * cn + 64 + 4);      // [32][cn] staged criterion inputs
    double *c0 = sc + 32 * cn;                                // [64] running background (cepstral criteria)
    uint8_t *sv = reinterpret_cast<uint8_t *>(c0 + 64);       // [32] decisions of the block
    double s_min = 0, s_max = 0, mean = 0, mean2 = 0, var = 0, dmin = 0, dmax = 0, dyn = 0;
    for (int base = 0; base < T; base += 32) {
        const int n = min(32, T - base);
        if (V.cri == VCRI_ENERGY) {
            if (lane < n) sc[lane] = cri_frame[R0 + min(base + lane + V.latency, T - 1)];
        } else {
            for (int idx = lane; idx < n * cn; idx += 32) {
                const int j = idx / cn, k = idx - j * cn;
                const int64_t fidx = R0 + min(base + j + V.latency, T - 1);   // spectrum frame this row is paired with
                sc[idx] = (V.cri == VCRI_CEPDIST_LPC) ? ceps[fidx * BURG_MAXC + k] : fea[(R0 + base + j) * fea_dim + k];
            }
        }
        __syncwarp();
        if (lane == 0) {
            for (int j = 0; j < n; j++) {
                const int r = base + j;
                const double *ci_row = sc + j * cn;
                double c;
                if (V.cri == VCRI_ENERGY) {
                    c = ci_row[0];
                } else {
                    // cepstral distance to the running background c0 (src/vad/vad.cc:249-276)
                    double sum = 0;
                    if (r == 0) {
                        for (int k = 0; k < cn; k++) c0[k] = ci_row[k];
                        c = 0.0;
                    } else {
                        for (int k = 0; k < cn; k++) {
                            const double ci = ci_row[k];
                            if (r == 1) c0[k] = (c0[k] + ci) / 2.0;
                            if ((V.cri == VCRI_CEPDIST_LPC) ? (k >= 1) : (k != V.fea_skip)) { double d = ci - c0[k]; sum += d * d; }
                        }
                        c = 4.3429 * sqrt(2 * sum);
                    }
                }
                bool v;
                double th = 0.0;                     // the threshold as the reference's debug file holds it after this step
                if (V.thr == VTHR_ABSOLUTE) {
                    th = V.abs_thr;
                    v = c >= V.abs_thr;
                } else if (V.thr == VTHR_PERC) {
                    if (r == 0 || (double)r < (double)V.perc_init) { s_min = c; s_max = c; }
                    else { s_min = (c < s_min) ? c : s_min; s_max = (c > s_max) ? c : s_max; }
                    th = s_min + (V.perc_thr / 100.0) * (s_max - s_min);
                    v = c >= th;
                } else if (V.thr == VTHR_ADAPT) {
                    if (r == 0) { mean = c; mean2 = c * c; var = 0.0; v = false; th = c; }
                    else {
                        th = mean + V.adapt_za * sqrt(var);
                        if ((c < th) || (r <= V.adapt_init)) {
                            mean = V.adapt_q * mean + (1.0 - V.adapt_q) * c;
                            mean2 = V.adapt_q * mean2 + (1.0 - V.adapt_q) * c * c;
                            var = mean2 - mean * mean;
                            v = false;
                        } else v = true;
                    }
                } else {
                    const int i0 = max(1, V.dyn_init);
                    if (r < i0) { dmax = c; dmin = c; dyn = 0.0; v = false; th = c; }
                    else if (r == i0) {
                        dmax = fmax(dmax, c) + V.dyn_min / 10.0;
                        dmin = fmin(dmin, c) - V.dyn_min / 10.0;
                        dyn = dmax - dmin; v = false; th = c;
                    } else {
                        if (dmax < c) dmax = V.qmaxinc * dmax + (1.0 - V.qmaxinc) * c; else dmax = V.qmaxdec * dmax + (1.0 - V.qmaxdec) * c;
                        if (dmin > c) dmin = V.qmindec * dmin + (1.0 - V.qmindec) * c; else dmin = V.qmininc * dmin + (1.0 - V.qmininc) * c;
                        dyn = dmax - dmin;
                        th = dmin + (V.dyn_perc / 100.0) * dyn;
                        v = (c > th) && (dyn > V.dyn_min);
                    }
                }
                sv[j] = v ? 1 : 0;
                if (V.dbg) {
                    // what VAD::save_frame would write after this step (src/vad/vad.cc:109-111, 278-286, 333-335, 400-404,
                    // 497-508, 627-634); the host pairs row i with step min(i + (order-1)/2, T-1)
                    double *d = V.dbg + (R0 + r) * VAD_DBG;
                    d[0] = c; d[1] = th;
                    if (V.thr == VTHR_PERC) { d[2] = s_min; d[3] = s_max; d[4] = 0.0; }
                    else if (V.thr == VTHR_ADAPT) { d[2] = mean; d[3] = mean2; d[4] = var; }
                    else if (V.thr == VTHR_DYN) { d[2] = dmin; d[3] = dmax; d[4] = dyn; }
                    else { d[2] = d[3] = d[4] = 0.0; }
                }
                if (V.cri != VCRI_ENERGY && !(v && r > V.cep_init)) {
                    for (int k = 0; k < cn; k++) c0[k] = V.cep_p * c0[k] + (1.0 - V.cep_p) * ci_row[k];
                }
            }
        }
        __syncwarp();
        if (lane < n) vad0_tmp[R0 + base + lane] = sv[lane];
        __syncwarp();
    }
    // majority vote over `order` decisions centred on the row; zeros beyond both ends
    const int h = (V.order - 1) / 2;
    for (int r = lane; r < T; r += 32) {
        int sum = 0;
        for (int q = r + h - V.order + 1; q <= r + h; q++)
            if (q >= 0 && q < T) sum += vad0_tmp[R0 + q];
        bool dec = ((double)sum / (double)V.order) >= 0.5;
        if (vad_out) vad_out[R0 + r] = dec ? 1 : 0;
        keep[R0 + r] = (dec || !V.drop) ? 1 : 0;
    }
}

// drop mode: compact the kept rows of each utterance towards its first row (one CTA per
// utterance, chunks of 32 rows staged through shared memory so in-place moves are safe)
__global__ void __launch_bounds__(256)
k_vad_compact(const int *__restrict__ nframes, const int64_t *__restrict__ row_off, int u0, const uint8_t *__restrict__ keep, float *fea,
              int dim, int *__restrict__ rows_out) {
    extern __shared__ __align__(16) float smc[];
    __shared__ int s_pos[33];
    const int u = u0 + blockIdx.x;
    const int T = nframes[u];
    const int64_t R0 = row_off[u];
    int written = 0;
    for (int base = 0; base < T; base += 32) {
        const int n = min(32, T - base);
        for (int i = threadIdx.x; i < n * dim; i += blockDim.x) smc[i] = fea[(R0 + base) * dim + i];
        if (threadIdx.x == 0) {
            int pos = 0;
            for (int j = 0; j < n; j++) { s_pos[j] = keep[R0 + base + j] ? pos++ : -1; }
            s_pos[32] = pos;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < n * dim; i += blockDim.x) {
            int j = i / dim, col = i - j * dim;
            int pos = s_pos[j];
            if (pos >= 0) fea[(R0 + written + pos) * dim + col] = smc[i];
        }
        written += s_pos[32];
        __syncthreads();
    }
    if (threadIdx.x == 0) rows_out[u] = written;
}

// ------------------------------------------------------------------------------------------
// K9: synthesis.  One CTA = one tile of the plan's synthesis tile list: SYN_FRAMES - hh output hops of one utterance
// plus the hh frames before them that still overlap the tile's first sample, one frame per 16-thread group, a single
// pass.  Every frame's time signal goes to its own shared-memory slot; the overlap-add then sums the slots in frame
// order, exactly the order in which the reference accumulates (src/io/out.cc:427-429), so the result is deterministic.
// ------------------------------------------------------------------------------------------
// The frame's complex spectrum X is the one k_frames2 stores next to |X| when a waveform is wanted, so the synthesis
// needs no second forward transform -- no PCM staging, no window, no forward FFT -- only the enhanced magnitude on the
// stored phase, the inverse transform and the overlap-add.  Storing X costs 2 x 2056 B of HBM traffic per frame (write +
// read) and saves about 40 % of the instructions of a synthesis that transforms every frame again (DESIGN.md, k_synth_c).
// WT / ST: window and shift known at compile time (0 = runtime) -- turns the divisions of the overlap-add index
// arithmetic into shifts / multiplies and prunes the zero padding.
template <int WT, int ST>
#ifndef CTU_SYNC_MINB
#define CTU_SYNC_MINB 3
#endif
__global__ void __launch_bounds__(SYN_THREADS, CTU_SYNC_MINB)
k_synth_c(const __grid_constant__ SynthParams S, int window, int wshift, BatchDesc bd, int tile_frames, int ntiles,
          const int64_t *__restrict__ osamp_off, const float2 *__restrict__ cspec, const float *__restrict__ spec, int16_t *__restrict__ out,
          const float2 *__restrict__ g_tw256, const float2 *__restrict__ g_twinv) {
    extern __shared__ __align__(16) float sm[];
    const int tid = threadIdx.x;
    const int w = WT ? WT : window, s = ST ? ST : wshift, hh = S.hh;
    cpx<float> *sTw = reinterpret_cast<cpx<float> *>(sm);                 // 256
    cpx<float> *sTi = sTw + 256;                                         // 130
    cpx<float> *sX = sTi + 130;                                          // SYN_GROUPS * 16*17
    float *sYt = reinterpret_cast<float *>(sX + SYN_GROUPS * XPAD * 16); // SYN_FRAMES * w
    for (int i = tid; i < 256; i += SYN_THREADS) sTw[i] = mk<float>(g_tw256[i].x, g_tw256[i].y);
    for (int i = tid; i < 129; i += SYN_THREADS) sTi[i] = mk<float>(g_twinv[i].x, g_twinv[i].y);
    __syncthreads();
    const int c = tid & (GROUP - 1), grp = tid / GROUP;
    const unsigned hm = 0xffffu << (tid & 16);
    cpx<float> *xch = sX + grp * (XPAD * 16);
    // (fetching a tile's inputs one tile ahead, before the overlap-add of the current one, was tried: 11.0 ms at two CTAs
    // per SM against 10.8 ms with three and no prefetch -- the kernel is bound by the transform and the overlap-add)
    struct SynMeta { int u, t0, T, nf, tfirst, nfr; };
    auto meta_of = [&](int tile) {
        SynMeta m;
        const int2 tl = bd.tiles[tile];
        m.u = tl.x; m.t0 = tl.y; m.T = bd.nframes[m.u];
        m.nf = min(tile_frames, m.T - m.t0); m.tfirst = max(m.t0 - hh, 0); m.nfr = m.t0 + m.nf - m.tfirst;
        return m;
    };
    cpx<float> lo[8], hi[8], mid;
    float Alo[8], Ahi[8], Amid = 0.f;
    auto fetch = [&](const SynMeta &m) {
        if (grp < m.nfr) {
            const int64_t row = bd.row_off[m.u] + m.tfirst + grp;
            const float *srow = spec + row * SPITCH;
            const float2 *xrow = cspec + row * NBIN;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                Alo[j] = __ldg(srow + c + 16 * j); Ahi[j] = __ldg(srow + NC - c - 16 * j);
                const float2 xl = __ldg(xrow + c + 16 * j), xh = __ldg(xrow + NC - c - 16 * j);
                lo[j] = mk<float>(xl.x, xl.y); hi[j] = mk<float>(xh.x, xh.y);
            }
            Amid = __ldg(srow + 128);
            const float2 xm = __ldg(xrow + 128);
            mid = mk<float>(xm.x, xm.y);
        }
    };
    int tile = blockIdx.x;
    if (tile >= ntiles) return;
#pragma unroll 1
    for (; tile < ntiles; tile += gridDim.x) {
        const SynMeta cur = meta_of(tile);
        fetch(cur);
        const int u = cur.u, t0 = cur.t0, T = cur.T, nf = cur.nf, tfirst = cur.tfirst, nfr = cur.nfr;
        if (grp < nfr) {
            const int f = grp;
            cpx<float> a[16];
            // enhanced magnitude with the ORIGINAL phase: scale X by |X|enh / (|X| nfft); bin 0 has phase 0, the Nyquist
            // bin is always written non-negative (src/io/out.cc:417-424)
            const float invn = 1.0f / (float)NFFT;
            auto scale_bin = [&](cpx<float> X, float A, bool edge) -> cpx<float> {
                A *= invn;
                if (edge) return mk<float>(A, 0.f);
                float m2 = X.x * X.x + X.y * X.y;
                if (m2 == 0.f) return mk<float>(0.f, -A);
                float g = A * rsqrtf(m2);
                return cscale(X, g);
            };
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const bool edge = (c == 0 && j == 0);               // k == 0 pairs with k == 256
                lo[j] = scale_bin(lo[j], Alo[j], edge);
                hi[j] = scale_bin(hi[j], Ahi[j], edge);
            }
            mid = scale_bin(mid, Amid, false);
            irfft_presplit_shfl(a, c, sTi, lo, hi, mid);
            fft256_pass1_rec(a, c, sTw, xch);
            __syncwarp(hm);
            fft256_pass2(a, c, xch);
            __syncwarp(hm);
            float *yt = sYt + f * w;
#pragma unroll
            for (int k2 = 0; k2 < 16; k2++) {
                int n = c + 16 * k2;
                if (2 * n + 1 < w) *reinterpret_cast<float2 *>(yt + 2 * n) = make_float2(a[k2].x, -a[k2].y);
                else if (2 * n < w) yt[2 * n] = a[k2].x;
            }
        }
        __syncthreads();
        // overlap-add in frame order (fp64 accumulator like the reference's cbuffer), floor(x / correction), clip
        // (src/io/out.cc:427-451)
        const bool last = (t0 + nf == T);
        const int nout = nf * s + (last ? (w - s) : 0);
        int16_t *o = out + osamp_off[u] + (int64_t)t0 * s;
        const int base = (t0 - tfirst) * s;
        const double inv_corr = 1.0 / S.correction;
        if (!((w | s) & 3) && !(reinterpret_cast<uintptr_t>(o) & 7)) {
            // four samples per thread where window and shift are multiples of four (16-byte slot reads, one 8-byte store)
            for (int i = 4 * tid; i < nout; i += 4 * SYN_THREADS) {
                const int pos = base + i;
                const int fa = (pos < w) ? 0 : (pos - w) / s + 1;
                const int fb = min(pos / s, nfr - 1);
                double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
                for (int f = fa; f <= fb; f++) {
                    const float4 y = *reinterpret_cast<const float4 *>(sYt + f * w + (pos - f * s));
                    a0 += (double)y.x; a1 += (double)y.y; a2 += (double)y.z; a3 += (double)y.w;
                }
                int v0 = (int)floor(a0 * inv_corr), v1 = (int)floor(a1 * inv_corr), v2 = (int)floor(a2 * inv_corr), v3 = (int)floor(a3 * inv_corr);
                v0 = max(-32767, min(32767, v0)); v1 = max(-32767, min(32767, v1));
                v2 = max(-32767, min(32767, v2)); v3 = max(-32767, min(32767, v3));
                uint2 pk;
                pk.x = (unsigned)(uint16_t)(int16_t)v0 | ((unsigned)(uint16_t)(int16_t)v1 << 16);
                pk.y = (unsigned)(uint16_t)(int16_t)v2 | ((unsigned)(uint16_t)(int16_t)v3 << 16);
                *reinterpret_cast<uint2 *>(o + i) = pk;
            }
        } else if (!((w | s) & 1) && !(reinterpret_cast<uintptr_t>(o) & 3)) {
            // two samples per thread: with an even window and shift an even-aligned pair has the same contributing frames,
            // so the index arithmetic is shared, the slots are read 8 bytes at a time and the pair leaves as one 32-bit store
            // (the overlap-add was ~45 % of this kernel's instructions)
            for (int i = 2 * tid; i < nout; i += 2 * SYN_THREADS) {
                const int pos = base + i;
                const int fa = (pos < w) ? 0 : (pos - w) / s + 1;
                const int fb = min(pos / s, nfr - 1);
                double a0 = 0.0, a1 = 0.0;
                for (int f = fa; f <= fb; f++) {
                    const float2 y = *reinterpret_cast<const float2 *>(sYt + f * w + (pos - f * s));
                    a0 += (double)y.x; a1 += (double)y.y;
                }
                int v0 = (int)floor(a0 * inv_corr), v1 = (int)floor(a1 * inv_corr);
                v0 = max(-32767, min(32767, v0)); v1 = max(-32767, min(32767, v1));
                *reinterpret_cast<unsigned *>(o + i) = (unsigned)(uint16_t)(int16_t)v0 | ((unsigned)(uint16_t)(int16_t)v1 << 16);
            }
        } else
        for (int i = tid; i < nout; i += SYN_THREADS) {
            const int pos = base + i;
            const int fa = (pos < w) ? 0 : (pos - w) / s + 1;
            const int fb = min(pos / s, nfr - 1);
            double acc = 0.0;
            for (int f = fa; f <= fb; f++) acc += (double)sYt[f * w + (pos - f * s)];
            int v = (int)floor(acc * inv_corr);
            v = max(-32767, min(32767, v));
            o[i] = (int16_t)v;
        }
        __syncthreads();                                      // the slots are re-used by the next tile
    }
}

int launch_synth_c(const SynthParams &S, const FrameParams &F, const BatchDesc &bd, int tile_frames, int64_t ntiles,
                                 const int64_t *d_osamp_off, const float2 *cspec, const float *spec, int16_t *out, const float2 *tw,
                                 const float2 *ti, cudaStream_t s, LaunchCtx *lc, std::string &err) {
    if (ntiles <= 0) return CTU_OK;
    if (F.window & 1) { err = "CTU: synthesis needs an even window length"; return CTU_ERR_UNSUPPORTED; }
    const size_t bytes = sizeof(float) * (2 * (256 + 130 + SYN_GROUPS * XPAD * 16) + (size_t)SYN_FRAMES * F.window);
    if (bytes > 227 * 1024 || tile_frames < 1) { err = "CTU: window/shift combination needs too much shared memory for synthesis"; return CTU_ERR_UNSUPPORTED; }
    cudaError_t e;
    int per_sm = 1, num_sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    lc->begin("k_synth_c", s);
#define CTU_SYNTHC_LAUNCH(WT, ST)                                                                                                    \
    e = cudaFuncSetAttribute(k_synth_c<WT, ST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);                          \
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_synth_c<WT, ST>, SYN_THREADS, bytes);         \
    if (e == cudaSuccess)                                                                                                            \
        k_synth_c<WT, ST><<<(unsigned)std::min<int64_t>(ntiles, (int64_t)std::max(per_sm, 1) * num_sms), SYN_THREADS, bytes, s>>>(  \
            S, F.window, F.wshift, bd, tile_frames, (int)ntiles, d_osamp_off, cspec, spec, out, tw, ti)
    if (F.window == 512 && F.wshift == 256) { CTU_SYNTHC_LAUNCH(512, 256); }
    else if (F.window == 400 && F.wshift == 160) { CTU_SYNTHC_LAUNCH(400, 160); }
    else { CTU_SYNTHC_LAUNCH(0, 0); }
#undef CTU_SYNTHC_LAUNCH
    lc->end(s);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { err = std::string("CUDA: ") + cudaGetErrorString(e) + " (k_synth_c)"; return CTU_ERR_CUDA; }
    return CTU_OK;
}

int launch_vad_module(VadParams V, const BurgParams &B, const BatchDesc &bd32, int64_t nt32, const int *d_nframes,
                                    const int64_t *d_row_off, int u0, int u1, int64_t row0, int64_t nrows, const int16_t *d_pcm,
                                    const float *d_spec, float *d_fea, const double *d_fea64, int fea_dim, double *d_ceps, double *d_cri,
                                    uint8_t *d_vad0,
                                    uint8_t *d_vadout, uint8_t *d_keep, int *d_rows, const double2 *tw, const double2 *ts,
                                    const double2 *ti, const double *win, cudaStream_t s, LaunchCtx *lc, std::string &err) {
    const int n = u1 - u0;
    if (n <= 0) return CTU_OK;
    cudaError_t e = cudaSuccess;
    if (V.cri == VCRI_ENERGY) {
        if (nrows > 0) {
            lc->begin("k_vad_energy", s);
            k_vad_energy<<<(unsigned)((nrows + 7) / 8), 256, 0, s>>>(V, d_spec, row0, nrows, d_cri);
            lc->end(s);
            e = cudaGetLastError();
        }
        V.cep_n = 0;
    } else if (V.cri == VCRI_CEPDIST_LPC) {
        V.cep_n = B.ncoef_vad;
        if (V.cep_n > BURG_MAXC || V.cep_n < 2) { err = "CTU: -vad_lpc_coefs must be 2..16"; return CTU_ERR_UNSUPPORTED; }
        int st = launch_burg(B, BURG_SRC_VAD, bd32, nt32, d_pcm, d_spec, d_ceps, tw, ts, ti, win, nullptr, s, lc, err);
        if (st) return st;
    } else {
        V.cep_n = fea_dim - V.has_E;      // the reference's vector does not hold the energy
        if (!d_fea64) { err = "CTU: internal: fp64 feature matrix missing for the cepstral-distance VAD"; return CTU_ERR_CONFIG; }
    }
    if (V.cep_n > 64) { err = "CTU: cepstral-distance VAD supports vectors of up to 64 values"; return CTU_ERR_UNSUPPORTED; }
    if (e == cudaSuccess) {
        lc->begin("k_vad_scan", s);
        const int cn_s = (V.cri == VCRI_ENERGY) ? 1 : V.cep_n;
        const size_t vs_bytes = (size_t)VADSCAN_WARPS * (32 * cn_s + 64 + 4) * sizeof(double);
        e = cudaFuncSetAttribute(k_vad_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)vs_bytes);
        k_vad_scan<<<(n + VADSCAN_WARPS - 1) / VADSCAN_WARPS, VADSCAN_WARPS * 32, vs_bytes, s>>>(V, d_nframes, d_row_off, u0, n, d_cri, d_ceps, d_fea64, fea_dim, d_vad0, d_vadout, d_keep);
        lc->end(s);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && V.drop) {
        size_t bytes = (size_t)32 * fea_dim * sizeof(float);
        e = cudaFuncSetAttribute(k_vad_compact, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(bytes, 1024));
        if (e == cudaSuccess) {
            lc->begin("k_vad_compact", s);
            k_vad_compact<<<n, 256, bytes, s>>>(d_nframes, d_row_off, u0, d_keep, d_fea, fea_dim, d_rows);
            lc->end(s);
            e = cudaGetLastError();
        }
    }
    if (e != cudaSuccess) { err = std::string("CUDA: ") + cudaGetErrorString(e) + " (vad module)"; return CTU_ERR_CUDA; }
    return CTU_OK;
}

}  // namespace ctu
#endif
