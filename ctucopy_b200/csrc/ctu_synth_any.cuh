// K9g: synthesis for FFT sizes other than 512 (enhanced waveforms at 8 kHz: 256 points; 22-48 kHz: 1024 / 2048).
// Same chain as k_synth_c (sigOUT::save_frame, src/io/out.cc:374-451): the frame's own spectrum, transformed here again
// from the PCM, gives the phase, the noise-reduced magnitude replaces its modulus, inverse real FFT, overlap-add in frame order, floor(x / correction),
// clip.  Written for generality like k_frames_any -- one WARP per frame, radix-2 in shared memory -- and in fp64
// throughout: the specialised kernel reaches +-1 LSB with an fp32 16x16 transform, a 10-stage fp32 radix-2 would not
// stay there for loud frames.  Two kernels: frames -> time-domain segments in a workspace [frames x window] (fp64),
// then one thread per output sample adds the overlapping segments in frame order like the reference's ring.
#ifndef CTU_SYNTH_ANY_CUH
#define CTU_SYNTH_ANY_CUH

#include "ctu_frames_any.cuh"
#include "ctu_any64.cuh"

namespace ctu {

constexpr int SYNANY_THREADS = ANY64_THREADS;  // 4 warps: 4 x (2 zslots(M) + 2M + 4) doubles of shared memory, 135 KB at 2048 points

// DC1: -remove_dc1, the frame is built from the de-meaned ring (dc1 = the ring means of k_dc1_means, one per frame)
template <bool DC1>
__global__ void __launch_bounds__(SYNANY_THREADS)
k_synth_frames_any(int window, int wshift, double preem, int remove_dc, BatchDesc bd, AnyTables64 tb, const int16_t *__restrict__ pcm,
                   const float *__restrict__ spec, double *__restrict__ yt, const double *__restrict__ dc1) {
    extern __shared__ __align__(16) double smd[];
    const int lane = threadIdx.x & 31, wv = threadIdx.x >> 5;
    const int nfft = tb.nfft, M = nfft >> 1, nbins = M + 1;
    cpx<double> *z = reinterpret_cast<cpx<double> *>(smd + (size_t)wv * (2 * any64_zslots(M) + 2 * (M + 2)));   // M complex, padded
    cpx<double> *Y = z + any64_zslots(M);                                                                        // M + 1 complex (+ pad)
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int nf = min(ANY_TILE, bd.nframes[u] - t0);
    const int64_t row0 = bd.row_off[u] + t0;
    const int w = window, s = wshift;
    for (int f = wv; f < nf; f += SYNANY_THREADS / 32) {
        any64_analysis<DC1>(z, tb, pcm + bd.pcm_off[u] + (int64_t)(t0 + f) * s, (t0 + f) == 0, w, preem, remove_dc, lane, DC1 ? dc1 + row0 + f : nullptr, t0 + f, s);
        // ---- real-input split; enhanced magnitude on the original phase, scaled by 1/nfft (src/io/out.cc:417-424) ---
        const float *A = spec + (row0 + f) * tb.spitch;
        const double invn = 1.0 / (double)nfft;
        for (int k = lane; k <= M; k += 32) {
            const cpx<double> X = any64_bin(z, tb, k);
            const double mag = (double)__ldg(A + k) * invn;
            cpx<double> Yk;
            if (k == 0 || k == M) Yk = mk<double>(mag, 0.0);            // bin 0: phase 0; Nyquist: written non-negative
            else {
                const double m2 = X.x * X.x + X.y * X.y;
                if (m2 == 0.0) Yk = mk<double>(0.0, -mag);
                else { const double g = mag / sqrt(m2); Yk = mk<double>(X.x * g, X.y * g); }
            }
            Y[k] = Yk;
        }
        __syncwarp();
        any64_inverse(z, Y, tb, lane);
        double *o = yt + (row0 + f) * w;
        for (int i = lane; i < w; i += 32) o[i] = any64_real(z, i);
        __syncwarp();
    }
}

// overlap-add in frame order with an fp64 accumulator (the reference's cbuffer), floor(x / correction), clip to +-32767
// (src/io/out.cc:427-451).  One CTA per 16-hop tile of the output (the last tile of a file also writes the window's tail).
__global__ void __launch_bounds__(256)
k_ola_any(int window, int wshift, double inv_corr, BatchDesc bd, const int64_t *__restrict__ osamp_off, const double *__restrict__ yt,
          int16_t *__restrict__ out) {
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int T = bd.nframes[u];
    const int nf = min(ANY_TILE, T - t0);
    const int w = window, s = wshift;
    const int nout = nf * s + ((t0 + nf == T) ? (w - s) : 0);
    const double *y = yt + bd.row_off[u] * w;
    int16_t *o = out + osamp_off[u] + (int64_t)t0 * s;
    for (int i = threadIdx.x; i < nout; i += blockDim.x) {
        const int64_t pos = (int64_t)t0 * s + i;
        const int64_t fa = (pos < w) ? 0 : (pos - w) / s + 1;          // first frame with fa*s + w > pos
        const int64_t fb = min(pos / s, (int64_t)T - 1);
        double acc = 0.0;
        for (int64_t f = fa; f <= fb; f++) acc += y[f * w + (pos - f * s)];
        int v = (int)floor(acc * inv_corr);
        v = max(-32767, min(32767, v));
        o[i] = (int16_t)v;
    }
}

}  // namespace ctu
#endif
