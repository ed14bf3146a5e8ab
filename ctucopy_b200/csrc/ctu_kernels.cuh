// Device code of the CtuCopy hot path for sm_100a shared by the frame kernels and the row kernels behind them:
//   * the parameter blocks and tile descriptors of the frame kernels (FrameParams, BatchDesc, FftTables), the PCM
//     staging of a tile (prefetch_pcm / finish_pcm: cp.async one tile ahead, pre-emphasis once per sample) and the
//     16-lane helpers of the group-per-frame 512-point transform (ctu_fft.cuh);
//   * the row kernels: LPC epilogue (k_lpc), exponential CMS and CMVN, energies, deltas, TRAP-DCT, column gather /
//     context stacking, container rows, G.711 expansion.
// The frame kernels themselves: ctu_frames2.cuh (PCM -> spectrum), ctu_bank.cuh (spectrum -> band values / features),
// ctu_frames256.cuh (256-point PCM -> spectrum) and ctu_frames_any.cuh (every other FFT size).
#ifndef CTU_KERNELS_CUH
#define CTU_KERNELS_CUH

#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "ctu_fft.cuh"

namespace ctu {

// host-side launch bookkeeping: counts kernel launches and, when profiling is switched on
// (ctu_profile_enable), brackets every kernel with CUDA events on its own stream
struct LaunchCtx {
    struct Rec { const char *name; cudaEvent_t a, b; };
    uint64_t launches = 0;
    bool prof_on = false;
    std::vector<Rec> recs;
    void begin(const char *name, cudaStream_t s) {
        launches++;
        if (!prof_on) return;
        Rec r; r.name = name;
        cudaEventCreate(&r.a); cudaEventCreate(&r.b);
        cudaEventRecord(r.a, s);
        recs.push_back(r);
    }
    void end(cudaStream_t s) { if (prof_on) cudaEventRecord(recs.back().b, s); }
    void clear() { for (auto &r : recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); } recs.clear(); }
};

constexpr int TILE_F = 32;        // frames per CTA tile
constexpr int MAXB = 64;          // filter-bank bands
constexpr int MAXW = 2560;        // packed filter-bank taps
constexpr int MAXR = 40;          // rows of the second-stage matrix (cepstra / autocorrelation lags)
constexpr int MAXM2 = 2048;       // second-stage matrix entries (rows x nb)
constexpr int DELTA_ROWS_C = 64;   // rows per tile of the 64-row tile list (= DELTA_ROWS)

enum Src { SRC_PCM = 0, SRC_SPEC = 1 };
enum Dst { DST_SPEC = 0, DST_FB = 1, DST_FEA = 2 };
enum Kind { KIND_SPEC = 1, KIND_LOGSPEC = 2, KIND_DCTC = 3, KIND_LPA = 4, KIND_LPC = 5, KIND_TRAPLOG = 6 };

// kernel parameter block (lives in the constant bank: warp-uniform indexed loads)
struct FrameParams {
    int window, wshift;
    float preem;
    int remove_dc;
    int take_sqrt;         // !fb_power: magnitude instead of power (src/io/in.cc:415-417)
    // filter bank
    int nb;
    int inld;              // ^0.33 (src/fea/fb.cc:81-83)
    float inld_scale;      // S^-0.33 where the packed weights carry a factor S
    float lin_scale;       // 1/S
    float log_offset;      // -ln S
    short lo[MAXB], hi[MAXB];
    int woff[MAXB];        // multiples of 4: each band's taps start 16-byte aligned
    alignas(16) float w[MAXW];
    // second stage
    int nrows;             // rows of m2 (dctc: output columns in writer order; lpc/lpa: lporder+1 lags)
    int nbp;               // row pitch of m2: nb rounded up to a multiple of 4 (zero padded)
    alignas(16) float m2[MAXM2];       // [nrows][nbp]
    int lporder, ncep;     // lpc/lpa
    int lpa_square;        // lpa/lpc without inld: square the band values first (src/fea/fea_impl.cc:165-169)
    int c0_last;           // lpc: write c1..cN then c0 (fea_c0 on) else c1..cN
    float lift[MAXR];      // lpc lifter for c1..cN (1 when fea_lifter <= 1)
    // output geometry
    int out_dim;           // values this kernel writes per row
    int out_stride;        // floats per row of the destination matrix
    // optional _E column (SURVEY 8a a22): which stage's energy the writer points at
    // (BATCH::init_out, src/io/batch.cc:98-118); written per frame into `energy`
    int energy_mode;       // EnergyMode
    float *energy;         // [total frames] log energies (device), nullptr when unused
    // -remove_dc1 (src/io/in.cc:343-350): per-frame means of the repeatedly de-meaned sample ring, nullptr when off
    const double *dc1;
    // -dither: (2*rand()/RAND_MAX - 1)*dither per loaded sample, same indexing as the PCM buffer, nullptr when off
    const float *dither;
};
enum EnergyMode {
    EN_NONE = 0,
    EN_NR = 1,             // _NR::compute_E (src/nr/nr.cc:36-45): sum of SQUARES of the spectrum handed to the filter bank
    EN_IN = 2,             // rawIN::get_frame (src/io/in.cc:403-413): sum of the POWER spectrum
    EN_BANDS = 3,          // specFEA / logspecFEA (src/fea/fea_impl.cc:45-50, 69-74): sum of squares of the band values
    EN_LPC = 4,            // lpaFEA (src/fea/fea_impl.cc:177): log R0
    EN_RAW = 5             // raw energy (src/io/in.cc:353-361), own kernel
};

struct BatchDesc {
    const int64_t *pcm_off;   // [n_utts] first sample of each utterance in the PCM buffer
    const int *nframes;       // [n_utts]
    const int64_t *row_off;   // [n_utts] first global frame index
    const int2 *tiles;        // [n_tiles] (utterance, first frame)
};

struct FftTables {            // device pointers
    const float2 *tw256, *twsplit, *twinv;
    const float *win;
};

// sum over the 16 lanes of this thread's half warp, for code in which both halves of a warp always arrive together: the
// FULL member mask.  A shuffle whose mask is not a compile-time constant is wrapped in BSSY / WARPSYNC / ENDCOLLECTIVE /
// BSYNC by the compiler (four extra instructions and a convergence barrier each); with 0xffffffff it is the bare SHFL.
__device__ __forceinline__ float group_sum16_all(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v;
}

// real-input split / inverse pre-split with the partner values fetched by register shuffles between
// thread c and thread (16-c)%16 of the group (arithmetic: ctu_fft.cuh, emulated in tests/emu).  The split
// forms its twiddles from the thread-constant twsplit[c] (rfft_split_pairs_rec) and uses the full member
// mask: both groups of the warp call it together.
template <class T>
__device__ __forceinline__ void rfft_split_shfl_rec(const cpx<T> (&a)[16], int c, cpx<T> ts_c, cpx<T> (&lo)[8], cpx<T> (&hi)[8], cpx<T> &mid) {
    const unsigned m = 0xffffffffu;
    const int src = (16 - c) & 15;
    cpx<T> Zp[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        Zp[j].x = __shfl_sync(m, a[15 - j].x, src, 16);
        Zp[j].y = __shfl_sync(m, a[15 - j].y, src, 16);
    }
    rfft_split_pairs_rec(a, Zp, c, ts_c, lo, hi, mid);
}

template <class T>
__device__ __forceinline__ void irfft_presplit_shfl(cpx<T> (&a)[16], int c, const cpx<T> *twinv, const cpx<T> (&lo)[8], const cpx<T> (&hi)[8],
                                                    cpx<T> mid) {
    const unsigned m = 0xffffu << (threadIdx.x & 16);
    const int src = (16 - c) & 15;
    cpx<T> zn[8], znp[8], z128;
    irfft_presplit_local(a, zn, z128, c, twinv, lo, hi, mid);
#pragma unroll
    for (int r = 0; r < 8; r++) {
        znp[r].x = __shfl_sync(m, zn[r].x, src, 16);
        znp[r].y = __shfl_sync(m, zn[r].y, src, 16);
    }
    irfft_presplit_place(a, c, zn, znp, z128);
}

// E = log(2 * (t_0/2 + t_last/2 + sum of the inner terms)) over one row of n values, term = v or
// v*v; one warp per row, `lane` strided.  The reference's formula for the energy of a
// half spectrum (src/io/in.cc:403-413, src/nr/nr.cc:36-45).
__device__ __forceinline__ float half_spectrum_energy(const float *row, int n, bool square) {
    const int lane = threadIdx.x & 31;
    float acc = 0.f;
    for (int k = lane; k < n; k += 32) {
        float v = row[k];
        if (square) v *= v;
        if (k == 0 || k == n - 1) v *= 0.5f;
        acc += v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    return logf(acc * 2.f);
}

// int16 -> float without the (quarter-rate) conversion pipe: 1.5*2^23 + x is exact
__device__ __forceinline__ float s16_to_f32(int x) { return __int_as_float(0x4B400000 + x) - 12582912.0f; }
// two int16 (a little-endian pair: element 2j in the low half) -> two floats, exactly: with the sign bits flipped the halves are
// v + 32768 in 0..65535, which PRMT places under the exponent of 2^23 (no sign extension); one packed subtraction of
// 2^23 + 2^15 leaves v
__device__ __forceinline__ cpx<float> s16x2_to_f32x2(uint32_t p) {
    const uint32_t q = p ^ 0x80008000u;
    const cpx<float> b = mk<float>(__uint_as_float(__byte_perm(q, 0x4B000000u, 0x7610)), __uint_as_float(__byte_perm(q, 0x4B000000u, 0x7632)));
    return b - mk<float>(8421376.0f, 8421376.0f);
}

// ---- PCM prefetch: the next tile's samples travel HBM -> shared memory with cp.async while the
// current tile is being transformed (the CTAs are persistent).  The raw int16 buffer keeps the
// 16-byte phase of the source address so that whole 16-byte chunks can be copied; the (at most
// two) partial chunks at the ends go through a register.
struct TileMeta { int t0, nf; int64_t row0, g0; };

// a tile's list entry resolved against its utterance, as loaded; tile_meta turns it into the TileMeta
struct TileDesc { int t0, nfu; int64_t roff, poff; };

__device__ __forceinline__ TileDesc load_tile_desc(const BatchDesc &bd, int2 t) {
    TileDesc d;
    d.t0 = t.y;
    d.nfu = bd.nframes[t.x];
    d.roff = bd.row_off[t.x];
    d.poff = bd.pcm_off[t.x];
    return d;
}

__device__ __forceinline__ TileMeta tile_meta(const TileDesc &d, int wshift, int tile_frames) {
    TileMeta m;
    m.t0 = d.t0;
    m.nf = min(tile_frames, d.nfu - d.t0);
    m.row0 = d.roff + d.t0;
    m.g0 = d.poff + (int64_t)d.t0 * wshift;
    return m;
}

__device__ __forceinline__ TileMeta load_tile_meta(const BatchDesc &bd, int tile, int wshift, int tile_frames) {
    return tile_meta(load_tile_desc(bd, bd.tiles[tile]), wshift, tile_frames);
}

// Descriptors of the tiles a persistent CTA takes next (tile + G, tile + 2G, ...; G = gridDim.x), fetched ahead by thread 0
// with cp.async into shared memory: in the iteration of `tile`, the per-utterance values of tile + 2G and the list entry of
// tile + 3G.  They land by the cp.async wait of the next iteration, so no load is consumed in the iteration that issues it.
// (The values are warp uniform, and the compiler moves a loaded one into a uniform register as soon as its load returns:
// with global loads the whole CTA waited there for two dependent load latencies per tile, and holding the values in
// ordinary registers across the transform costs the registers of the fifth CTA.)  Two slots, alternating by iteration.
struct TileAhead {
    int64_t roff[2], poff[2];
    int2 t[2];
    int nfu[2], t0[2];
};
constexpr int TILE_AHEAD_FLOATS = (int)(sizeof(TileAhead) / 4);   // 16: a multiple of four keeps what follows 16-byte aligned

__device__ __forceinline__ void cp_async_small(void *dst, const void *src, int bytes) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    if (bytes == 8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(src) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(src) : "memory");
}

// thread 0: the per-utterance values of list entry e into slot j
__device__ __forceinline__ void tile_ahead_desc(TileAhead *A, int j, const BatchDesc &bd, int2 e) {
    A->t0[j] = e.y;
    cp_async_small(&A->nfu[j], bd.nframes + e.x, 4);
    cp_async_small(&A->roff[j], bd.row_off + e.x, 8);
    cp_async_small(&A->poff[j], bd.pcm_off + e.x, 8);
}

// before the first tile (the copies join the first PCM prefetch's group)
__device__ __forceinline__ void tile_ahead_init(TileAhead *A, const BatchDesc &bd, int tile, int ntiles) {
    const int G = gridDim.x;
    if (threadIdx.x != 0) return;
    if (tile + G < ntiles) tile_ahead_desc(A, 0, bd, bd.tiles[tile + G]);
    if (tile + 2 * G < ntiles) cp_async_small(&A->t[0], bd.tiles + tile + 2 * G, 8);
}

// in the iteration of `tile` (slot j = its parity), after the cp.async wait and a barrier: the descriptor of tile + G
// (meaningful when tile + G < ntiles); thread 0 then issues the copies that the next iteration reads from slot j ^ 1
__device__ __forceinline__ TileMeta tile_ahead_next(TileAhead *A, int j, const BatchDesc &bd, int tile, int ntiles, int wshift,
                                                    int tile_frames) {
    const TileDesc d = TileDesc{A->t0[j], A->nfu[j], A->roff[j], A->poff[j]};
    if (threadIdx.x == 0) {
        const int G = gridDim.x;
        if (tile + 2 * G < ntiles) tile_ahead_desc(A, j ^ 1, bd, A->t[j]);
        if (tile + 3 * G < ntiles) cp_async_small(&A->t[j ^ 1], bd.tiles + tile + 3 * G, 8);
    }
    return tile_meta(d, wshift, tile_frames);
}

// element k of the tile's sample run is sample (k - 1): k = 0 is the sample before the tile
// (pre-emphasis memory), valid only when the tile is not at the start of its utterance
template <int NT>
__device__ __forceinline__ void prefetch_pcm(int16_t *raw, const int16_t *__restrict__ pcm, const TileMeta &m, int n, int &edge) {
    const int16_t *S0 = pcm + m.g0 - 1;
    const int phase = (int)((reinterpret_cast<uintptr_t>(S0) & 15) >> 1);
    const int kmin = (m.t0 == 0) ? 1 : 0;
    const int nchunks = (phase + n + 7) >> 3;
    for (int j = threadIdx.x; j < nchunks; j += NT) {
        const int k0 = 8 * j - phase;
        if (k0 >= kmin && k0 + 8 <= n) {
            const unsigned dst = (unsigned)__cvta_generic_to_shared(raw + 8 * j);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(S0 + k0) : "memory");
        }
    }
    // partial chunks: the first one (j = 0) and the last one; thread t < 8 takes element t of the
    // first, thread 8 + t element t of the last
    edge = 0;
    if (threadIdx.x < 16) {
        const int j = (threadIdx.x < 8) ? 0 : nchunks - 1;
        const int k0 = 8 * j - phase, k = k0 + (threadIdx.x & 7);
        const bool partial = !(k0 >= kmin && k0 + 8 <= n) && (threadIdx.x < 8 || nchunks > 1);
        if (partial && k >= kmin && k < n) edge = (int)S0[k];
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}

// after the copies have landed: partial-chunk elements from the registers, then raw -> float with
// pre-emphasis (src/io/in.cc:364-372), every sample converted once for all the frames it is in
template <int NT>
__device__ __forceinline__ void finish_pcm(int16_t *raw, float *__restrict__ sD, const int16_t *__restrict__ pcm, const TileMeta &m, int n,
                                           int edge, float alpha) {
    const int16_t *S0 = pcm + m.g0 - 1;
    const int phase = (int)((reinterpret_cast<uintptr_t>(S0) & 15) >> 1);
    const int kmin = (m.t0 == 0) ? 1 : 0;
    const int nchunks = (phase + n + 7) >> 3;
    asm volatile("cp.async.wait_all;" ::: "memory");
    if (threadIdx.x < 16) {
        const int j = (threadIdx.x < 8) ? 0 : nchunks - 1;
        const int k0 = 8 * j - phase, k = k0 + (threadIdx.x & 7);
        const bool partial = !(k0 >= kmin && k0 + 8 <= n) && (threadIdx.x < 8 || nchunks > 1);
        if (partial && k >= 0 && k < n) raw[phase + k] = (k >= kmin) ? (int16_t)edge : (int16_t)0;
    }
    __syncthreads();
    const int16_t *x = raw + phase;                       // x[k]: element k
    const int nsamp = n - 1;
    int i0 = 0;
    if (phase & 1) {
        // x + 1 is 4-byte aligned: a thread takes four consecutive samples -- two int16 pairs, the sample before them and
        // one 16-byte store.  Consecutive threads take consecutive runs, so a warp's pair loads cover 256 contiguous bytes
        // (two wavefronts each), the loads of the sample before (stride 8 bytes) two, and its store 512 contiguous bytes
        // (four): 10 wavefronts per 128 samples against 12 for four rounds of the scalar loop below, in a quarter of the
        // loop iterations.  (An earlier 8-samples-per-thread layout lost to the scalar loop: it cost four wavefronts per
        // load; ncu, profiles/.  Here no access spans more bytes than it moves.)
        const int nq = nsamp >> 2;
#pragma unroll 2   // fully unrolled, the loop costs the 32-register-window instantiations of k_frames2 a spill
        for (int q = threadIdx.x; q < nq; q += NT) {
            const int i = 4 * q;
            const uint32_t *xp = reinterpret_cast<const uint32_t *>(x + i + 1);
            const cpx<float> a = s16x2_to_f32x2(xp[0]), b = s16x2_to_f32x2(xp[1]);
            const float p = s16_to_f32((int)x[i]);
            *reinterpret_cast<float4 *>(sD + i) =
                make_float4(fmaf(-alpha, p, a.x), fmaf(-alpha, a.x, a.y), fmaf(-alpha, a.y, b.x), fmaf(-alpha, b.x, b.y));
        }
        i0 = 4 * nq;
    }
    // even phases (odd utterance offsets or shifts), and the last nsamp % 4 samples of odd ones: one sample per thread
    for (int i = i0 + threadIdx.x; i < nsamp; i += NT) {
        const float prev = s16_to_f32((int)x[i]);
        const float xi = s16_to_f32((int)x[i + 1]);
        sD[i] = fmaf(-alpha, prev, xi);
    }
}

// ------------------------------------------------------------------------------------------
// Exponential cepstral mean subtraction (cms_POST::process_frame, src/fea/post_impl.cc:203-209):
// per utterance and per static coefficient  m = m*Z + c*(1-Z);  c -= m  with a FLOAT running mean
// and a float coefficient, applied to the finished rows (the deltas were taken from the
// un-normalised statics, src/io/batch.cc:159-163).  One thread per (utterance, column).
// ------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(128)
k_cms_exp(const int *__restrict__ nframes, const int64_t *__restrict__ row_off, int u0, int n_utts, int ncols, int stride, float Z,
          float *__restrict__ fea) {
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n_utts * ncols) return;
    const int u = u0 + gid / ncols, col = gid % ncols;
    const int T = nframes[u];
    float *x = fea + row_off[u] * stride + col;
    const float omZ = 1.0f - Z;
    float m = 0.f;
    // the recurrence is serial in t but its loads are not: eight rows are fetched before the chain advances
    int t = 0;
    for (; t + 8 <= T; t += 8, x += 8 * (int64_t)stride) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; i++) v[i] = x[(int64_t)i * stride];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const double c = (double)v[i];
            m = (float)((double)(m * Z) + c * (double)omZ);
            x[(int64_t)i * stride] = (float)(c - (double)m);
        }
    }
    for (; t < T; t++, x += stride) {
        const double c = (double)*x;
        m = (float)((double)(m * Z) + c * (double)omZ);
        *x = (float)(c - (double)m);
    }
}

// ------------------------------------------------------------------------------------------
// CMVN, device half (cmvn_POST::sum_fea / sum_cv / process_frame, src/fea/post_impl.cc:52-118):
// per-utterance column sums (of the values, or of squared deviations from a centre) in a fixed
// order -- the host adds the utterances of a speaker in list order, so the statistics are
// reproducible -- and the normalisation (F - mean) / var of every row.
// ------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(128)
k_colsums(const int *__restrict__ nframes, const int64_t *__restrict__ row_off, int n_utts, int dim, int stride,
          const float *__restrict__ fea, const double *__restrict__ center, double *__restrict__ sums) {
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n_utts * dim) return;
    const int u = gid / dim, col = gid - u * dim;
    const int T = nframes[u];
    const float *x = fea + row_off[u] * stride + col;
    const double c = center ? center[gid] : 0.0;
    double acc = 0.0;
    if (center) for (int t = 0; t < T; t++, x += stride) { const double d = (double)*x - c; acc += d * d; }
    else for (int t = 0; t < T; t++, x += stride) acc += (double)*x;
    sums[gid] = acc;
}

static __global__ void __launch_bounds__(256)
k_normalise(BatchDesc bd, int dim, int stride, const double *__restrict__ mean, const double *__restrict__ scale, float *__restrict__ fea) {
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int nr = min(DELTA_ROWS_C, bd.nframes[u] - t0);
    float *base = fea + (bd.row_off[u] + t0) * stride;
    const double *m = mean + (int64_t)u * dim, *v = scale + (int64_t)u * dim;
    for (int i = threadIdx.x; i < nr * dim; i += blockDim.x) {
        const int r = i / dim, col = i - r * dim;
        float *x = base + r * stride + col;
        *x = (float)(((double)*x - m[col]) / v[col]);
    }
}

// ------------------------------------------------------------------------------------------
// raw energy (src/io/in.cc:353-361): log of the sum of squares of the frame's raw samples 1..w-1
// (the first one is skipped).  One warp per frame.
// ------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256)
k_rawenergy(BatchDesc bd, int window, int wshift, const int16_t *__restrict__ pcm, float *__restrict__ energy) {
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int nf = min(DELTA_ROWS_C, bd.nframes[u] - t0);
    const int lane = threadIdx.x & 31;
    for (int f = threadIdx.x >> 5; f < nf; f += 8) {
        const int16_t *x = pcm + bd.pcm_off[u] + (int64_t)(t0 + f) * wshift;
        double acc = 0;
        for (int i = 1 + lane; i < window; i += 32) { const double v = (double)x[i]; acc += v * v; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) energy[bd.row_off[u] + t0 + f] = (float)log(acc);
    }
}

// The writer reads *E when a row leaves the delta / VAD delay lines (src/io/out.cc:183-202), so
// row t carries the energy of frame min(t + latency, T-1): last column of the feature matrix.
static __global__ void __launch_bounds__(256)
k_place_energy(BatchDesc bd, int latency, int stride, const float *__restrict__ energy, float *__restrict__ fea) {
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int T = bd.nframes[u];
    const int64_t row0 = bd.row_off[u];
    for (int t = t0 + threadIdx.x; t < min(t0 + DELTA_ROWS_C, T); t += blockDim.x)
        fea[(row0 + t) * stride + stride - 1] = energy[row0 + min(t + latency, T - 1)];
}

// ------------------------------------------------------------------------------------------
// K1c: LPC epilogue as its own kernel, one THREAD per frame (src/fea/fea_impl.cc:163-284:
// band values -> autocorrelation by cosine transform -> Levinson-Durbin -> [cepstrum,
// lifter]).  The recursion is a ~1000-instruction dependent fp64 chain per frame; run by one
// warp inside a frame kernel it stalls the whole CTA, here 128 independent frames
// per CTA and many CTAs per SM hide it.  PORD / NCEP compile-time (0 = runtime) keeps the
// coefficient arrays in registers.
// in: band values (true scale, after ^0.33) [rows x nb]; out: rows of the feature matrix.
// ------------------------------------------------------------------------------------------
constexpr int LPC_THREADS = 128;

template <int PORD, int NCEP, bool CEPS>
__global__ void __launch_bounds__(LPC_THREADS)
k_lpc(const __grid_constant__ FrameParams P, int64_t row0, int64_t nrows, const float *__restrict__ fb, float *__restrict__ out) {
    extern __shared__ __align__(16) float sm[];
    const int nb = P.nb, ld = nb | 1;
    const int64_t r0 = row0 + (int64_t)blockIdx.x * LPC_THREADS;
    const int nr = (int)min((int64_t)LPC_THREADS, row0 + nrows - r0);
    for (int i = threadIdx.x; i < nr * nb; i += LPC_THREADS) {
        int r = i / nb, b = i - r * nb;
        float v = fb[r0 * nb + i];
        sm[r * ld + b] = P.lpa_square ? v * v : v;
    }
    __syncthreads();
    if ((int)threadIdx.x >= nr) return;
    const float *y = sm + threadIdx.x * ld;
    const int p = PORD ? PORD : P.lporder;
    constexpr int NA = PORD ? PORD + 1 : MAXR;
    double R[NA], a[NA], aa[NA];
    // autocorrelation lags R[k] = sum_n y[n] m[k][n]: bands in the outer loop, so that a band value is converted to fp64 once
    // instead of once per lag (the conversions were a third of the kernel's instructions); every R[k] still adds its terms in
    // band order
#pragma unroll
    for (int k = 0; k < NA; k++) R[k] = 0.0;
    for (int n = 0; n < nb; n++) {
        const double yn = (double)y[n];
#pragma unroll
        for (int k = 0; k < NA; k++) if (k <= p) R[k] += yn * (double)P.m2[k * P.nbp + n];
    }
    if (P.energy_mode == EN_LPC) P.energy[r0 + threadIdx.x] = (float)log(R[0]);
    double Pe = R[0];
    double rc = -R[1] / R[0];
    Pe = Pe * (1 - rc * rc);
    a[0] = aa[0] = 1.0; a[1] = aa[1] = rc;
#pragma unroll
    for (int ik = 2; ik < NA; ik++) {
        if (ik <= p) {
            double dm = R[ik];
#pragma unroll
            for (int n = 1; n < NA; n++) if (n <= ik - 1) dm += aa[n] * R[ik - n];
            rc = -dm / Pe;
            a[ik] = rc;
#pragma unroll
            for (int n = 1; n < NA; n++) if (n <= ik - 1) a[n] = aa[n] + rc * aa[ik - n];
#pragma unroll
            for (int n = 1; n < NA; n++) if (n <= ik) aa[n] = a[n];
            Pe = Pe * (1 - rc * rc);
        }
    }
    float *o = out + (r0 + threadIdx.x) * P.out_stride;
    if (!CEPS) {
#pragma unroll
        for (int i = 1; i < NA; i++) if (i <= p) o[i - 1] = (float)a[i];       // a0 is not written
        return;
    }
    const int N = NCEP ? NCEP : P.ncep;
    constexpr int NC_ = NCEP ? NCEP + 1 : MAXR;
    double cc[NC_];
    cc[0] = log(Pe);
#pragma unroll
    for (int n = 1; n < NC_; n++) {
        if (n <= N) {
            double sum = 0;
#pragma unroll
            for (int k = 1; k < NA; k++) if (k <= p && k <= n - 1) sum += (double)(n - k) * cc[(n - k) > 0 ? (n - k) : 0] * a[k];
            cc[n] = (n <= p ? -a[n < NA ? n : 0] : 0.0) - sum * (1.0 / n);            // (compile-time reciprocal: the loop is unrolled)
            o[n - 1] = (float)(cc[n] * (double)P.lift[n]);
        }
    }
    if (P.c0_last) o[N] = (float)cc[0];
}

// Container rows on the device (SURVEY 8f.1): what pfileOUT / htkOUT do per value on the host (src/io/pfile.cc:470-539:
// rows of big-endian u32 sentence, u32 frame, float32 x dim; src/io/out.cc:189-213: byte-swapped floats for -endian_out
// big).  One CTA per 64-row tile; `out` may alias `fea` when only the byte order changes (same row pitch).
//   pfile != 0: out rows are dim + 2 words, sentence = sent0 + utterance index, frame = row index within the utterance
static __global__ void __launch_bounds__(256)
k_format_rows(BatchDesc bd, int dim, int pfile, uint32_t sent0, const float *fea, uint32_t *out) {
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int nr = min(DELTA_ROWS_C, bd.nframes[u] - t0);
    const int64_t row0 = bd.row_off[u] + t0;
    const int od = dim + (pfile ? 2 : 0);
    const uint32_t *src = reinterpret_cast<const uint32_t *>(fea) + row0 * dim;
    uint32_t *dst = out + row0 * od;
    for (int i = threadIdx.x; i < nr * od; i += blockDim.x) {
        const int r = i / od, col = i - r * od;
        uint32_t v;
        if (pfile && col == 0) v = sent0 + (uint32_t)u;
        else if (pfile && col == 1) v = (uint32_t)(t0 + r);
        else v = src[r * dim + col - (pfile ? 2 : 0)];
        dst[i] = __byte_perm(v, 0, 0x0123);
    }
}

// one thread per utterance writes that utterance's tile descriptors
// (the non-template kernels of this header are `static`: it is included by several translation units)
static __global__ void k_build_tiles(const int *__restrict__ nframes, const int64_t *__restrict__ tile_off, int n_utts, int tile_f,
                              int2 *__restrict__ tiles) {
    int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n_utts) return;
    int T = nframes[u];
    int64_t o = tile_off[u];
    for (int t = 0, i = 0; t < T; t += tile_f, i++) tiles[o + i] = make_int2(u, t);
}

// ------------------------------------------------------------------------------------------
// K7 deltas: regression over +-win rows with replicated edges, chained per order, the whole
// chain in one kernel over a tile of rows with halo (src/fea/fea_delta.cc:146-164 and the
// edge logic :70-130, :178-206 in its regular regime, see oracle fea_delta_block).
// Reads block 0 (static) of the output matrix, writes blocks 1..n_order in place.
// ------------------------------------------------------------------------------------------
struct DeltaParams {
    int n_order;
    int win[3];
    float inv_den[3];
    double inv_den64[3];
    int blk;          // columns per block (ncep+1 incl. c0 position)
    int stride;       // floats per row
    int span_max;     // tile_rows + 2 * sum(win): rows of one staging buffer
};
constexpr int DELTA_ROWS = 64;

template <class E>
__global__ void __launch_bounds__(256)
k_delta(const __grid_constant__ DeltaParams D, BatchDesc bd, int tile_rows, E *__restrict__ fea, const E *__restrict__ src = nullptr,
        int src_stride = 0) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    E *sm = reinterpret_cast<E *>(sm_raw);
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int T = bd.nframes[u];
    const int nr = min(tile_rows, T - t0);
    const int64_t row0 = bd.row_off[u];
    const int blk = D.blk;
    // thread = (column cx of 16, row ry of 16): no divisions in the loops
    const int cx = threadIdx.x & 15, ry = threadIdx.x >> 4;
    int halo = 0;
    for (int k = 0; k < D.n_order; k++) halo += D.win[k];
    const int span = nr + 2 * halo;                       // rows t0-halo .. t0+nr+halo-1 (clamped)
    E *cur = sm;                                          // [span][blk]
    E *nxt = sm + D.span_max * blk;
    // src != nullptr: the static block comes from another matrix (the first blk columns of its rows: feature-file input,
    // spectral vectors) and is written to the output rows here as well -- gather and deltas in one pass
    for (int r = ry; r < span; r += 16) {
        const int ta = t0 - halo + r, t = min(max(ta, 0), T - 1);
        const E *g = src ? src + (row0 + t) * src_stride : fea + (row0 + t) * D.stride;
        const bool own = src && ta >= t0 && ta < t0 + nr;
        for (int col = cx; col < blk; col += 16) {
            const E v = g[col];
            cur[r * blk + col] = v;
            if (own) fea[(row0 + t) * D.stride + col] = v;
        }
    }
    __syncthreads();
    int h = halo;                                         // halo still valid around `cur`
    for (int k = 0; k < D.n_order; k++) {
        const int W = D.win[k];
        const int hn = h - W;                             // halo of the next block
        const int rows_n = nr + 2 * hn;
        const E scale = (sizeof(E) == 8) ? (E)D.inv_den64[k] : (E)D.inv_den[k];
        for (int r = ry; r < rows_n; r += 16) {           // r: index into next (offset hn)
            const int t = t0 - hn + r;                    // absolute row of this output
            const int tc = min(max(t, 0), T - 1);         // replicated edge: value of the clamped row
            const bool own = (t >= t0 && t < t0 + nr);
            for (int col = cx; col < blk; col += 16) {
                // window rows around tc, each clamped to [0, T-1]; position in `cur` = row - (t0 - h)
                E acc = 0;
                for (int j = 1; j <= W; j++) {
                    const int tp = min(tc + j, T - 1), tm = max(tc - j, 0);
                    acc += (E)j * (cur[(tp - (t0 - h)) * blk + col] - cur[(tm - (t0 - h)) * blk + col]);
                }
                E v = acc * scale;
                if (W == 1 && tc == T - 1) v = 0;         // reference quirk for win == 1 (see oracle)
                nxt[r * blk + col] = v;
                if (own) fea[(row0 + t) * D.stride + (k + 1) * blk + col] = v;
            }
        }
        __syncthreads();
        E *tmp = cur; cur = nxt; nxt = tmp;
        h = hn;
    }
}

// Fast path for the standard configuration (delta + acceleration, both windows 2, at most 16
// columns per block): a thread owns one column and four consecutive rows of a 64-row tile and
// keeps the whole chain in registers.  Replicated edges: the staged tile already holds c at
// clamped rows, and a delta "at" a row outside the file is the delta of the clamped row
// (src/fea/fea_delta.cc:70-130, 178-206).
template <class E>
__global__ void __launch_bounds__(256)
k_delta22(const __grid_constant__ DeltaParams D, BatchDesc bd, E *__restrict__ fea, const E *__restrict__ src = nullptr, int src_stride = 0) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    E *cur = reinterpret_cast<E *>(sm_raw);               // [DELTA_ROWS + 8][blk]
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int T = bd.nframes[u];
    const int nr = min(DELTA_ROWS, T - t0);
    const int64_t row0 = bd.row_off[u];
    const int blk = D.blk;
    const int cx = threadIdx.x & 15, seg = threadIdx.x >> 4;
    const int span = nr + 8;                              // rows t0-4 .. t0+nr+3 (clamped)
    if (cx < blk)
        for (int r = seg; r < span; r += 16) {
            const int t = min(max(t0 - 4 + r, 0), T - 1);
            cur[r * blk + cx] = src ? src[(row0 + t) * src_stride + cx] : fea[(row0 + t) * D.stride + cx];
        }
    __syncthreads();
    const int r0 = seg * 4;                               // first of this thread's rows, relative to t0
    if (cx >= blk || r0 >= nr) return;
    const E s1 = (sizeof(E) == 8) ? (E)D.inv_den64[0] : (E)D.inv_den[0];
    const E s2 = (sizeof(E) == 8) ? (E)D.inv_den64[1] : (E)D.inv_den[1];
    // delta at rows t0+r0-2 .. t0+r0+5, each taken at the clamped row
    E d[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int tc = min(max(t0 + r0 - 2 + i, 0), T - 1);
        const E *c = cur + (tc - (t0 - 4)) * blk + cx;    // position of row tc in the staged tile
        d[i] = ((c[blk] - c[-blk]) + (E)2 * (c[2 * blk] - c[-2 * blk])) * s1;     // same order as the reference sum
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int t = t0 + r0 + i;
        if (t >= t0 + nr) break;
        const E a = ((d[i + 3] - d[i + 1]) + (E)2 * (d[i + 4] - d[i])) * s2;
        E *o = fea + (row0 + t) * D.stride + cx;
        if (src) o[0] = cur[(r0 + i + 4) * blk + cx];     // static block from the external source (see k_delta)
        o[blk] = d[i + 2];
        o[2 * blk] = a;
    }
}

// ------------------------------------------------------------------------------------------
// K8 TRAP-DCT: per (row, band) a `traplen`-row trajectory of log band energies, mean
// removal + Hamming + DCT-II folded into one [ndct x traplen] matrix on the host
// (src/fea/fea_trap.cc:84-108; context replication :63-69, :111-127).
// in: logfb [rows x nb]; out: [rows x nb*ndct] band-major.
// ------------------------------------------------------------------------------------------
constexpr int TRAP_ROWS = 64;
constexpr int TRAP_MAXL = 128;
constexpr int TRAP_MAXN = 16;
struct TrapParams {
    int L, ndct, nb, h;         // h = (L+1)/2
    int out_stride, pad[3];     // m starts on a 16-byte boundary of the parameter bank
    float m[TRAP_MAXN * TRAP_MAXL];   // [L][ndct], m[j * ndct + k-1] = 2*hamm[j]*cos(pi (j+.5) k / L) with the mean removal folded in:
                                      // the coefficients of one trajectory position are neighbours (pairs for the packed FMA)
};

// LT / NT: trajectory length and coefficient count known at compile time (0 = runtime).
// With both fixed the j and k loops unroll completely and the matrix entries come out of the constant bank four at a time
// (LDCU.128 into uniform registers) as operands of packed FMAs (FFMA2, ctu_fft.cuh): the folded pair (dj, sj) times the
// entries of an even and an odd coefficient, into their two partial sums -- half the issue slots of one FFMA per entry
// (4.73 -> 4.16 ms per 9.98 M frames).  Four consecutive rows of a band per thread with sliding pairs -- 12.5 shared-memory
// loads per output instead of 51, the constants fetched once for four outputs, 250 instead of 370 instructions per output --
// measured 4.26 ms (tools/gpu_jobs/r2_job45.sh): the kernel is not bound by its instruction count.
template <int LT, int NT>
__global__ void __launch_bounds__(256)
k_trapdct(const __grid_constant__ TrapParams Tp, BatchDesc bd, int tile_rows, const float *__restrict__ logfb,
          float *__restrict__ out) {
    extern __shared__ __align__(16) float sm[];
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int T = bd.nframes[u];
    const int nr = min(tile_rows, T - t0);
    const int64_t row0 = bd.row_off[u];
    const int nb = Tp.nb, L = LT ? LT : Tp.L, h = (L + 1) / 2, ND = NT ? NT : Tp.ndct;
    const bool regular = T >= h - 1;
    // rows needed: t0-(h-1) .. t0+nr-1+(h-1), clamped (replicated context)
    const int span = nr + L - 1;
    if (regular) {
        for (int i = threadIdx.x; i < span * nb; i += blockDim.x) {
            int r = i / nb, b = i - r * nb;
            int t = min(max(t0 - (h - 1) + r, 0), T - 1);
            sm[i] = logfb[(row0 + t) * nb + b];
        }
    } else {
        // fewer than h-1 frames: all T rows live in the tile (T < h-1 <= tile_rows)
        for (int i = threadIdx.x; i < T * nb; i += blockDim.x) sm[i] = logfb[row0 * nb + i];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nr * nb; i += blockDim.x) {
        int r = i / nb, b = i - r * nb;
        constexpr int NA = NT ? NT : TRAP_MAXN;
        float acc[NA];
#pragma unroll
        for (int k = 0; k < NA; k++) acc[k] = 0.f;
        // the rows of m sum to zero (mean removal is folded in), so any constant may be
        // subtracted first: take the centre value to keep the fp32 products small
        if (regular) {
            const float *v = sm + r * nb + b;
            const float ref = v[(h - 1) * nb];
            if (LT && NT) {
                // Hamming x DCT-II rows are symmetric (even k) or antisymmetric (odd k) about the
                // centre of the odd-length trajectory, and removing the mean keeps that: fold
                // x[j] +- x[L-1-j] first, half the multiplies.  The centre sample is `ref`, so its
                // own term is zero.
                constexpr int LH = (LT ? LT : 1) / 2;
                static_assert(NA % 2 == 0, "coefficient pairs");
                cpx<float> ac[NA / 2];
#pragma unroll
                for (int k = 0; k < NA / 2; k++) ac[k] = mk<float>(0.f, 0.f);
#pragma unroll
                for (int j = 0; j < LH; j++) {
                    const cpx<float> x = mk<float>(v[j * nb], v[((LT ? LT : 1) - 1 - j) * nb]) - mk<float>(ref, ref);
                    const cpx<float> ds = x + mk<float>(-x.y, x.x);               // (xa - xb, xb + xa): the swap and the sign are operand modifiers
#pragma unroll
                    for (int k = 0; k < NA / 2; k++)                                                       // entry k holds DCT index k+1
                        ac[k] = pfma(ds, mk<float>(Tp.m[j * NA + 2 * k], Tp.m[j * NA + 2 * k + 1]), ac[k]);
                }
#pragma unroll
                for (int k = 0; k < NA / 2; k++) { acc[2 * k] = ac[k].x; acc[2 * k + 1] = ac[k].y; }
            } else {
                for (int j = 0; j < L; j++) {
                    const float x = v[j * nb] - ref;
#pragma unroll
                    for (int k = 0; k < NA; k++)
                        if (k < ND) acc[k] = fmaf(x, Tp.m[j * ND + k], acc[k]);
                }
            }
        } else {
            // flush r of a short file sees Z never-written (zero) ring rows first
            const int Z = h - T - (r + 1);
            const float ref = sm[b];
            for (int j = 0; j < L; j++) {
                float x = -ref;
                if (j >= Z) x = sm[min(max(j - Z - (h - 1), 0), T - 1) * nb + b] - ref;
#pragma unroll
                for (int k = 0; k < NA; k++)
                    if (k < ND) acc[k] = fmaf(x, Tp.m[j * ND + k], acc[k]);
            }
        }
        float *o = out + (row0 + t0 + r) * Tp.out_stride + b * ND;
#pragma unroll
        for (int k = 0; k < NA; k++)
            if (k < ND) o[k] = acc[k];
    }
}

// ------------------------------------------------------------------------------------------
// K9: column gather / context stacking.  Three uses, one kernel:
//   * `-fea_trap N` (deltaFEA::trap, src/fea/fea_delta.cc:166-176): out[t][i*L + j] = C[t + j - win][i], L = N = 2 win + 1,
//     rows clamped to the utterance, with the reference's start-up and flush behaviour (closed form and its derivation:
//     oracle/ctu_oracle.py trap_stack_closed_form -- first row stacks rows 0 x win, 1, 1, 2, .., win; with win == 1 the last
//     row stacks row T-1 three times; the first row and the last `win` rows then carry C[t][0..fea_c) in their first fea_c
//     elements, src/fea/fea_delta.cc:88-90, 197-199);
//   * deltas of spec / logspec vectors: the delta chain works on the first fea_ncepcoefs+1 elements (L = 1);
//   * feature-file input (htkIN, src/io/in.cc:682-690): the first fea_c columns of the input rows (L = 1).
// C is in the reference's INTERNAL order; `rot` says the source block is stored in writer order (c1..cN, c0).
// One CTA per tile of DELTA_ROWS rows; consecutive threads write consecutive output elements.
// ------------------------------------------------------------------------------------------
struct StackParams {
    int L, win;          // context length (1 = plain gather) and half width
    int fea_c;           // coefficients taken from every source row
    int rot;             // source column of internal coefficient i: rot ? (i == 0 ? fea_c-1 : i-1) : i
    int src_stride, dst_stride;
};

// STAGE: the tile's source rows t0-win .. t0+nr-1+win (all src_stride columns: one contiguous block of memory) are copied to
// shared memory with coalesced loads, and the tile's output -- also one contiguous block -- is written element by element in
// memory order.  Without STAGE (rows too wide for shared memory) the gather reads global memory directly.
template <bool STAGE>
__global__ void __launch_bounds__(256)
k_stack(const StackParams S, BatchDesc bd, int tile_rows, const float *__restrict__ src, float *__restrict__ dst) {
    extern __shared__ __align__(16) float sm_stack[];
    const int2 tile = bd.tiles[blockIdx.x];
    const int u = tile.x, t0 = tile.y;
    const int T = bd.nframes[u];
    const int nr = min(tile_rows, T - t0);
    const int64_t row0 = bd.row_off[u];
    const int L = S.L, win = S.win, fc = S.fea_c;
    const int W = fc * L, ss = S.src_stride, ds = S.dst_stride;
    // staged rows: [lo, hi]; the first row of a file also reads row 1 (start-up priming), the last one row T-1
    const int lo = max(t0 - win, 0), hi = min(max(t0 + nr - 1 + win, L > 1 ? 1 : 0), T - 1);
    if (STAGE) {
        const float *g = src + (row0 + lo) * ss;
        const int n = (hi - lo + 1) * ss;
        for (int i = threadIdx.x; i < n; i += 256) sm_stack[i] = __ldg(g + i);
        __syncthreads();
    }
    float *o = dst + (row0 + t0) * ds;
    // a thread owns one output column e (a few when a row has more than 256 of them) and walks down the rows of its row
    // group: the column's (coefficient, context position) pair is worked out once, and consecutive threads write
    // consecutive floats of a row
    const int RG = (W >= 256) ? 1 : 256 / W;
    const int rg = (W >= 256) ? 0 : threadIdx.x / W;
    if (rg >= RG) return;
    for (int e = threadIdx.x - rg * W; e < W; e += 256) {
        const int i = e / L, j = e - i * L;
        const int col = S.rot ? (i == 0 ? fc - 1 : i - 1) : i;
        const int col_own = S.rot ? (e == 0 ? fc - 1 : e - 1) : e;        // column e of the row itself (edge rows, e < fc)
        // interior rows: source offset and destination pointer advance by constants (the kernel is issue-bound, not
        // memory-bound: 83 % of the issue slots with the index arithmetic redone per element)
        int so = (t0 + rg + j - win - lo) * ss + col;
        const int so_step = RG * ss;
        float *op = o + (int64_t)rg * ds + e;
        const int64_t op_step = (int64_t)RG * ds;
        const int t_hi = T - 1 - win;
        for (int f = rg; f < nr; f += RG, so += so_step, op += op_step) {
            const int t = t0 + f;
            if (L > 1 && (t < win || t > t_hi)) {                        // start-up / flush rows
                int k = t + j - win, c = col;
                if (t == 0) k = (j < win) ? 0 : (j <= win + 1 ? 1 : j - win);
                k = min(max(k, 0), T - 1);
                if (win == 1 && t == T - 1) k = T - 1;
                if ((t == 0 || t >= T - win) && e < fc) { k = t; c = col_own; }
                *op = STAGE ? sm_stack[(k - lo) * ss + c] : __ldg(src + (row0 + k) * ss + c);
            } else {
                *op = STAGE ? sm_stack[so] : __ldg(src + (row0 + lo) * ss + so);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// G.711 expansion on the device (alaw2lin, src/io/amulaw.h): 8-bit codes -> int16 PCM through a 256-entry table.
// Both buffers are indexed by the same absolute sample index and allocated 256-byte aligned, so a thread takes the
// 8 samples [8i, 8i+8) of the range rounded down to a multiple of 8: one 8-byte load, one 16-byte store.
// ------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256)
k_g711_expand(const uint8_t *__restrict__ codes, int16_t *__restrict__ pcm, int64_t first, int64_t count, const int16_t *__restrict__ table) {
    __shared__ int16_t lut[256];
    lut[threadIdx.x] = table[threadIdx.x];
    __syncthreads();
    const int64_t a0 = first & ~(int64_t)7;
    const int64_t end = first + count;
    for (int64_t i = a0 + 8 * ((int64_t)blockIdx.x * blockDim.x + threadIdx.x); i < end; i += 8 * (int64_t)gridDim.x * blockDim.x) {
        if (i >= first && i + 8 <= end) {
            const uint2 c = *reinterpret_cast<const uint2 *>(codes + i);
            int4 o;
            o.x = (int)(uint16_t)lut[c.x & 255] | ((int)(uint16_t)lut[(c.x >> 8) & 255] << 16);
            o.y = (int)(uint16_t)lut[(c.x >> 16) & 255] | ((int)(uint16_t)lut[c.x >> 24] << 16);
            o.z = (int)(uint16_t)lut[c.y & 255] | ((int)(uint16_t)lut[(c.y >> 8) & 255] << 16);
            o.w = (int)(uint16_t)lut[(c.y >> 16) & 255] | ((int)(uint16_t)lut[c.y >> 24] << 16);
            *reinterpret_cast<int4 *>(pcm + i) = o;
        } else {
            for (int64_t k = max(i, first); k < min(i + 8, end); k++) pcm[k] = lut[codes[k]];
        }
    }
}

}  // namespace ctu
#endif
