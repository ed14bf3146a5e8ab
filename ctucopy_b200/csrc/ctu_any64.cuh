// fp64 building blocks of the GENERAL kernels (FFT sizes other than 512): one warp owns a frame, the transform is an
// in-place FFT (radix-4 passes) of nfft/2 complex points in shared memory.  Used by the general synthesis (ctu_synth_any.cuh) and
// by the general Burg front end below.  Speed is secondary here (every BASELINE configuration takes the 512-point
// kernels); the arithmetic conventions are those of k_synth_c / k_burg, restated from the same reference lines.
#ifndef CTU_ANY64_CUH
#define CTU_ANY64_CUH

#include "ctu_kernels.cuh"

namespace ctu {

struct AnyTables64 {
    const double2 *tw;       // e^{-2 pi i k / M}, k < M/2           (M = nfft/2)
    const double2 *twsplit;  // -i/2 e^{-2 pi i k / nfft}, k <= M
    const double *win;       // analysis window [window]
    int nfft, log2m;
    int spitch;              // floats per row of the fp32 spectrum matrix
};

constexpr int ANY64_THREADS = 128;            // 4 warps per CTA

// The M complex points of a frame live at PADDED positions zp(n) = n + n / 16: 16-byte elements at power-of-two strides (bit
// reversal: M/2, M/4, ...; radix-4 passes: h, 2h, 3h) put a warp's accesses into one or two banks -- ncu on 8 kHz runs showed
// the general synthesis at 99.5 % of the LSU wavefront peak with 5.5e8 conflicts in 1.26e9 wavefronts (profiles/
// r02_ncu_general_fp64_8k.txt).  One slot of padding every 16 spreads them.  any64_zslots(M) = slots to reserve for z.
__host__ __device__ __forceinline__ int zp(int n) { return n + (n >> 4); }
__host__ __device__ inline int any64_zslots(int M) { return M + (M >> 4) + 1; }
// real sample i of the frame (z[n] = y[2n] + i y[2n+1]) in the padded layout
__device__ __forceinline__ double &any64_real(cpx<double> *z, int i) { return reinterpret_cast<double *>(z)[2 * zp(i >> 1) + (i & 1)]; }

// in-place decimation-in-time FFT of M complex points held by one warp in shared memory
__device__ __forceinline__ void warp_fft_radix2(cpx<double> *z, int M, int log2m, const double2 *__restrict__ tw, int lane) {
    for (int n = lane; n < M; n += 32) {
        const int r = (int)(__brev((unsigned)n) >> (32 - log2m));
        if (r > n) { const cpx<double> t = z[zp(n)]; z[zp(n)] = z[zp(r)]; z[zp(r)] = t; }
    }
    __syncwarp();
    // one radix-2 stage when log2(M) is odd, then radix-4 passes (two radix-2 stages of half lengths h and 2h fused: the four
    // points p, p+h, p+2h, p+3h are read and written once; the second stage's odd twiddle is -i times the even one)
    int h = 1, sh = log2m - 1;
    if (log2m & 1) {
        for (int b = lane; b < (M >> 1); b += 32) {
            const cpx<double> a = z[zp(2 * b)], t = z[zp(2 * b + 1)];
            z[zp(2 * b)] = a + t;
            z[zp(2 * b + 1)] = a - t;
        }
        __syncwarp();
        h = 2; sh--;
    }
    for (; 4 * h <= M; h <<= 2, sh -= 2) {
        for (int q = lane; q < (M >> 2); q += 32) {
            const int j = q & (h - 1), p0 = ((q - j) << 2) + j;
            const double2 w1 = __ldg(tw + ((size_t)j << sh)), w2 = __ldg(tw + ((size_t)j << (sh - 1)));
            const int q0 = zp(p0), q1 = zp(p0 + h), q2 = zp(p0 + 2 * h), q3 = zp(p0 + 3 * h);
            const cpx<double> z0 = z[q0], t1 = cmul(z[q1], mk<double>(w1.x, w1.y));
            const cpx<double> z2 = z[q2], t3 = cmul(z[q3], mk<double>(w1.x, w1.y));
            const cpx<double> a0 = z0 + t1, a1 = z0 - t1;
            const cpx<double> u2 = cmul(z2 + t3, mk<double>(w2.x, w2.y)), u3 = cmul(z2 - t3, mk<double>(w2.x, w2.y));
            const cpx<double> v3 = mk<double>(u3.y, -u3.x);           // -i u3
            z[q0] = a0 + u2;
            z[q2] = a0 - u2;
            z[q1] = a1 + v3;
            z[q3] = a1 - v3;
        }
        __syncwarp();
    }
}

// the frame exactly as rawIN::get_frame builds it (pre-emphasis, window, mean of the windowed frame removed inside the
// window, src/io/in.cc:362-388), transformed: z holds FFT_M of the even/odd packed frame afterwards
__device__ __forceinline__ void any64_analysis(cpx<double> *z, const AnyTables64 &tb, const int16_t *__restrict__ x, bool at_start, int w,
                                               double preem, int remove_dc, int lane) {
    const int nfft = tb.nfft;
    double sum = 0.0;
    for (int i = lane; i < nfft; i += 32) {
        double v = 0.0;
        if (i < w) {
            const double xi = (double)x[i];
            const double xp = (i == 0 && at_start) ? 0.0 : (double)x[i - 1];
            v = tb.win[i] * (xi - preem * xp);
        }
        any64_real(z, i) = v;
        sum += v;
    }
    if (remove_dc) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        const double mean = sum / (double)w;
        __syncwarp();
        for (int i = lane; i < w; i += 32) any64_real(z, i) -= mean;
    }
    __syncwarp();
    warp_fft_radix2(z, nfft >> 1, tb.log2m, tb.tw, lane);
}

// bin k of the real-input spectrum from the packed transform
__device__ __forceinline__ cpx<double> any64_bin(const cpx<double> *z, const AnyTables64 &tb, int k) {
    const int M = tb.nfft >> 1;
    const cpx<double> a = z[zp(k == M ? 0 : k)], b = conj(z[zp(k == 0 ? 0 : M - k)]);
    const double2 ts = __ldg(tb.twsplit + k);
    return mk<double>(0.5 * (a.x + b.x), 0.5 * (a.y + b.y)) + cmul(mk<double>(ts.x, ts.y), a - b);
}

// UNNORMALISED inverse real transform (what FFTW's HC2R gives, src/io/out.cc:425, src/nr/nr.cc:291, src/vad/vad.cc:232) of
// the half spectrum Y[0..M] into the nfft reals that alias z:  Z[k] = E[k] + i O[k], E = (Y[k] + conj Y[M-k]) / 2,
// O = e^{+2 pi i k / nfft} (Y[k] - conj Y[M-k]) / 2;  z[n] = 2 sum_k Z[k] e^{+2 pi i k n / M} = 2 conj(FFT_M(conj Z))[n];
// y[2n] = Re z[n], y[2n+1] = Im z[n] (read them with any64_real: z is padded).
__device__ __forceinline__ void any64_inverse(cpx<double> *z, const cpx<double> *Y, const AnyTables64 &tb, int lane) {
    const int M = tb.nfft >> 1;
    for (int k = lane; k < M; k += 32) {
        const cpx<double> a = Y[k], b = conj(Y[M - k]);
        const double2 ts = __ldg(tb.twsplit + k);                      // (-sin/2, -cos/2)  ->  e^{+i th}/2 = (-ts.y, -ts.x)
        const cpx<double> E = mk<double>(0.5 * (a.x + b.x), 0.5 * (a.y + b.y));
        const cpx<double> O = cmul(mk<double>(-ts.y, -ts.x), a - b);
        z[zp(k)] = mk<double>(E.x - O.y, -(E.y + O.x));                // conj(Z[k])
    }
    __syncwarp();
    warp_fft_radix2(z, M, tb.log2m, tb.tw, lane);
    for (int n = lane; n < M; n += 32) {                               // in place: z[n] occupies reals 2n, 2n+1
        const cpx<double> v = z[zp(n)];
        z[zp(n)] = mk<double>(2.0 * v.x, -2.0 * v.y);
    }
    __syncwarp();
}

}  // namespace ctu
#endif
