// K1b: spectrum -> [noise-reduction scan] -> filter bank -> log / DCT / band values, one kernel.
//
// The second half of every 512-point feature chain: the PCM -> spectrum kernel (k_frames2) leaves [frames x SPITCH]
// rows in HBM (257 bins padded to 260 floats = 16-byte aligned rows); this kernel takes them through
//   NR::process_frame      exten / hwss / fwss / 2fwss on the linear spectrum (src/nr/nr.cc:95-140, 212-261, 331-369,
//                          397-442) -- fused: the recursion runs on the tile in shared memory, the enhanced spectrum
//                          never goes back to HBM (it used to cross HBM three more times: scan read + write, then read)
//   FB::project_frame      banded projection, ^0.33 (src/fea/fb.cc:72-86)
//   FEA::process_frame     spec / logspec / dctc, or band values for the LPC kernel / log bands for TRAP-DCT
//                          (src/fea/fea_impl.cc:37-131)
// and writes each frame's result once.
//
// Work unit: a tile of 32 consecutive frames of one utterance = ONE contiguous run of nf * 1040 bytes, fetched by a
// single bulk asynchronous copy (cp.async.bulk + mbarrier: no load instructions, no LSU traffic, no registers).  A CTA
// holds ONE tile (44 KB of shared memory in all, 64 registers: four CTAs = 32 warps per SM) and asks for its next tile
// as soon as the filter bank has consumed the current one, so the copy overlaps its own second stage and store and the
// other three CTAs' work.  (First version: two tile buffers per CTA, two CTAs per SM -- every phase between two
// barriers then had 16 warps to hide its latencies with, and the fused scan, a 32-step dependent chain per bin, ran at a
// third of the speed of the standalone scan kernel.)  CTAs are persistent.  Without a scan they stride over the plan's
// 32-frame tile list; with a scan each CTA owns whole utterances (u = blockIdx.x, += gridDim.x) and walks their tiles
// in time order with the recursion state of its 257 bins in registers.
//
// Filter bank: lane == frame.  A lane reads its frame's row with 16-byte loads (row pitch 260 floats = 4 mod 32 banks:
// the eight lanes of a quarter warp cover all 32 banks, so a 128-bit load costs its minimum of four wavefronts) and the
// weights with 16-byte BROADCAST loads from a shared-memory copy whose bands start at multiples of four bins (zero
// padded).  Per four taps: 2 loads + 4 FMAs.  The kernel this replaces (k_frames<spec,..>) indexed the weights in the
// kernel-parameter bank with a per-thread register: one LDC + one 4-byte LDS + one FMA per tap, 5x the instructions.
#ifndef CTU_BANK_CUH
#define CTU_BANK_CUH

#include "ctu_kernels.cuh"
#include "ctu_nr_params.cuh"

namespace ctu {

constexpr int BANK_THREADS = 256;
constexpr int BANK_TILE_FLOATS = TILE_F * SPITCH;          // 8320 floats = 33 280 bytes

struct BankParams {
    int nb, nbp;               // bands, rounded up to a multiple of 4
    int ypitch;                // floats per row of the band tile: multiple of 4, = 4 mod 32
    int inld;
    float inld_scale, lin_scale, log_offset;
    int nrows;                 // dctc: output columns
    int out_dim, out_stride;
    int energy_mode;
    float *energy;
    int take_sqrt;
    int wtot4;                 // float4 groups of packed weights
    const int4 *bands;         // [nb]: (first bin / 4, float4 groups, offset into w4, -)
    const float4 *w4;          // weights, every band padded to whole groups of four bins
    const float *m2;           // [nrows][nbp] second-stage matrix (dctc), zero padded
    NrParams nr;               // fused scan
    const uint8_t *flags;      // detector decisions per frame (hwss / fwss / 2fwss)
};

struct BankSmem { int oTile, oY, oO, oW, oM, oBands, oFlags, oBar, total; };     // float offsets
__host__ __device__ inline BankSmem bank_smem(int nb, int nbp, int ypitch, int wtot4, int nrows, int out_dim) {
    BankSmem L;
    int o = 0;
    L.oTile = o; o += BANK_TILE_FLOATS;
    L.oY = o; o += TILE_F * ypitch;
    L.oO = o; o += (TILE_F * out_dim + 3) & ~3;            // output staging (the tile itself is being refilled by then)
    L.oW = o; o += 4 * wtot4;
    L.oM = o; o += (nrows * nbp + 3) & ~3;
    L.oBands = o; o += 4 * nb;
    L.oFlags = o; o += TILE_F / 4 * 2;                     // 32 bytes + pad
    L.oBar = o; o += 2;                                    // one 8-byte mbarrier
    L.total = o;
    return L;
}

// ---- bulk asynchronous copy + mbarrier (sm_90+ PTX; SASS: UBLKCP / SYNCS) -------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
    unsigned ok;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
    } while (!ok);
}

// the tiles a CTA works through, in order
struct BankWalk {
    int u, t0, T;              // current tile: utterance, first frame, frames of the utterance
    int64_t row0;              // first global row of the utterance
    int tile;                  // tile-list mode: index into the list
    bool valid;
};

template <bool NR>
__device__ __forceinline__ BankWalk bank_first(const BatchDesc &bd, int ntiles, int u0, int n_utts) {
    BankWalk w;
    w.tile = blockIdx.x; w.u = 0; w.t0 = 0; w.T = 0; w.row0 = 0; w.valid = false;
    if (NR) {
        int i = blockIdx.x;
        while (i < n_utts && bd.nframes[u0 + i] <= 0) i += gridDim.x;
        if (i < n_utts) { w.u = u0 + i; w.tile = i; w.t0 = 0; w.T = bd.nframes[w.u]; w.row0 = bd.row_off[w.u]; w.valid = true; }
    } else if (w.tile < ntiles) {
        const int2 t = bd.tiles[w.tile];
        w.u = t.x; w.t0 = t.y; w.T = bd.nframes[w.u]; w.row0 = bd.row_off[w.u]; w.valid = true;
    }
    return w;
}
template <bool NR>
__device__ __forceinline__ BankWalk bank_next(const BankWalk &c, const BatchDesc &bd, int ntiles, int u0, int n_utts) {
    BankWalk w = c;
    if (NR) {
        if (c.t0 + TILE_F < c.T) { w.t0 = c.t0 + TILE_F; return w; }
        int i = c.tile + gridDim.x;
        while (i < n_utts && bd.nframes[u0 + i] <= 0) i += gridDim.x;
        w.valid = i < n_utts;
        if (w.valid) { w.u = u0 + i; w.tile = i; w.t0 = 0; w.T = bd.nframes[w.u]; w.row0 = bd.row_off[w.u]; }
        return w;
    }
    w.tile = c.tile + gridDim.x;
    w.valid = w.tile < ntiles;
    if (w.valid) { const int2 t = bd.tiles[w.tile]; w.u = t.x; w.t0 = t.y; w.T = bd.nframes[w.u]; w.row0 = bd.row_off[w.u]; }
    return w;
}

// one tile of the recursion: 32 frames in shared memory, in place.  Threads 0-127 own the bin pairs (2t, 2t + 1) and run
// nr_step2 on packed FP32 with 8-byte loads and stores (SPITCH is even, so every pair is aligned); thread 128 carries bin
// 256 on the scalar nr_step, in the x half of its state; warps 5-7 have no scan work.
constexpr int BANK_SCAN_CHUNK = 8;
constexpr int BANK_SCAN_PAIRS = 128;
template <int MODE, int AKIND, bool FULL>
__device__ __forceinline__ void bank_scan_chunk(const NrParams &N, ScanState2 &S, float *tile, const uint8_t *fl, int f0, int nf, int t0) {
    cpx<float> *x = reinterpret_cast<cpx<float> *>(tile) + threadIdx.x;
    // the values come into registers first (independent loads, all in flight at once); in place, every step would wait for
    // its own shared-memory load behind the previous step's store
    cpx<float> v[BANK_SCAN_CHUNK];
#pragma unroll
    for (int j = 0; j < BANK_SCAN_CHUNK; j++) v[j] = x[(f0 + j) * (SPITCH / 2)];
#pragma unroll
    for (int j = 0; j < BANK_SCAN_CHUNK; j++)
        if (FULL || f0 + j < nf) v[j] = nr_step2<MODE, AKIND>(N, S, v[j], t0 + f0 + j, (MODE != NR_EXTEN) ? fl[f0 + j] : 0);
#pragma unroll
    for (int j = 0; j < BANK_SCAN_CHUNK; j++) x[(f0 + j) * (SPITCH / 2)] = v[j];
}
template <int MODE, int AKIND, bool FULL>
__device__ __forceinline__ void bank_scan_chunk_last(const NrParams &N, ScanState2 &S2, float *tile, const uint8_t *fl, int f0, int nf, int t0) {
    float *x = tile + 2 * BANK_SCAN_PAIRS;
    ScanState S;
    S.Navg = S2.Navg.x; S.Yavg = S2.Yavg.x; S.Nravg = S2.Nravg.x;
    float v[BANK_SCAN_CHUNK];
#pragma unroll
    for (int j = 0; j < BANK_SCAN_CHUNK; j++) v[j] = x[(f0 + j) * SPITCH];
#pragma unroll
    for (int j = 0; j < BANK_SCAN_CHUNK; j++)
        if (FULL || f0 + j < nf) v[j] = nr_step<MODE, AKIND>(N, S, v[j], t0 + f0 + j, (MODE != NR_EXTEN) ? fl[f0 + j] : 0);
#pragma unroll
    for (int j = 0; j < BANK_SCAN_CHUNK; j++) x[(f0 + j) * SPITCH] = v[j];
    S2.Navg.x = S.Navg; S2.Yavg.x = S.Yavg; S2.Nravg.x = S.Nravg;
}

template <int MODE, int AKIND>
__device__ __forceinline__ void bank_scan_tile(const NrParams &N, ScanState2 &S, float *tile, const uint8_t *fl, int nf, int t0) {
    // eight frames at a time; the loop over the chunks stays rolled (unrolled over all 32 frames, seven mode variants made
    // the kernel 240 KB of code).  Whole chunks take the branch-free body.
    if (threadIdx.x < BANK_SCAN_PAIRS) {
#pragma unroll 1
        for (int f0 = 0; f0 < nf; f0 += BANK_SCAN_CHUNK) {
            if (f0 + BANK_SCAN_CHUNK <= nf) bank_scan_chunk<MODE, AKIND, true>(N, S, tile, fl, f0, nf, t0);
            else bank_scan_chunk<MODE, AKIND, false>(N, S, tile, fl, f0, nf, t0);
        }
    } else if (threadIdx.x == BANK_SCAN_PAIRS) {
#pragma unroll 1
        for (int f0 = 0; f0 < nf; f0 += BANK_SCAN_CHUNK) {
            if (f0 + BANK_SCAN_CHUNK <= nf) bank_scan_chunk_last<MODE, AKIND, true>(N, S, tile, fl, f0, nf, t0);
            else bank_scan_chunk_last<MODE, AKIND, false>(N, S, tile, fl, f0, nf, t0);
        }
    }
}

template <int KIND, int DST, bool NR>
__global__ void __launch_bounds__(BANK_THREADS, 4)
k_bank(const __grid_constant__ BankParams B, BatchDesc bd, int ntiles, int u0, int n_utts, const float *__restrict__ spec, float *__restrict__ dst) {
    extern __shared__ __align__(16) float sm[];
    const BankSmem L = bank_smem(B.nb, B.nbp, B.ypitch, B.wtot4, B.nrows, B.out_dim);
    const int tid = threadIdx.x, lane = tid & 31, wv = tid >> 5;
    float *tile = sm + L.oTile, *sO = sm + L.oO;
    float *sY = sm + L.oY;
    float4 *sW4 = reinterpret_cast<float4 *>(sm + L.oW);
    float *sM = sm + L.oM;
    int4 *sBands = reinterpret_cast<int4 *>(sm + L.oBands);
    uint8_t *sFlags = reinterpret_cast<uint8_t *>(sm + L.oFlags);
    uint64_t *bar = reinterpret_cast<uint64_t *>(sm + L.oBar);

    BankWalk cur = bank_first<NR>(bd, ntiles, u0, n_utts);
    if (!cur.valid) return;
    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < B.wtot4; i += BANK_THREADS) sW4[i] = B.w4[i];
    for (int i = tid; i < B.nrows * B.nbp; i += BANK_THREADS) sM[i] = B.m2[i];
    for (int i = tid; i < B.nb; i += BANK_THREADS) sBands[i] = B.bands[i];
    // pad columns of the band tile (read by the 4-wide second-stage loop) stay zero for the whole kernel
    for (int i = tid; i < TILE_F * B.ypitch; i += BANK_THREADS) sY[i] = 0.f;
    __syncthreads();
    // the i-th tile of this CTA completes phase i & 1 of the mbarrier
    if (tid == 0) {
        const int nf = min(TILE_F, cur.T - cur.t0);
        const unsigned bytes = (unsigned)nf * SPITCH * sizeof(float);
        mbar_expect_tx(bar, bytes);
        bulk_g2s(tile, spec + (cur.row0 + cur.t0) * SPITCH, bytes, bar);
    }
    ScanState2 S;
    S.Navg = S.Yavg = S.Nravg = mk(0.f, 0.f);
#pragma unroll 1
    for (int it = 0; cur.valid; it++) {
        const BankWalk nxt = bank_next<NR>(cur, bd, ntiles, u0, n_utts);
        const int nf = min(TILE_F, cur.T - cur.t0);
        const int64_t row0 = cur.row0 + cur.t0;
        if (NR && B.nr.mode != NR_EXTEN && tid < TILE_F) sFlags[tid] = (tid < nf) ? B.flags[row0 + tid] : 0;
        mbar_wait(bar, (unsigned)it & 1u);
        if (NR) {
            if (cur.t0 == 0) {
                // exten: smoothed noise / speech start at 0.95 / 0.05 (src/nr/nr.cc:86-93); *ss: the noise estimate of a
                // standalone file starts at 0 (src/nr/nr.cc:212-222)
                const float n0 = (B.nr.mode == NR_EXTEN) ? 0.95f : 0.f;
                S.Navg = mk(n0, n0); S.Yavg = mk(0.05f, 0.05f); S.Nravg = mk(0.f, 0.f);
            }
            if (B.nr.mode != NR_EXTEN) __syncthreads();                      // flags staged
            const bool a2 = B.nr.a_kind == 2;
            switch (B.nr.mode) {
                case NR_EXTEN: if (a2) bank_scan_tile<NR_EXTEN, 2>(B.nr, S, tile, sFlags, nf, cur.t0); else bank_scan_tile<NR_EXTEN, 1>(B.nr, S, tile, sFlags, nf, cur.t0); break;
                case NR_HWSS: if (a2) bank_scan_tile<NR_HWSS, 2>(B.nr, S, tile, sFlags, nf, cur.t0); else bank_scan_tile<NR_HWSS, 1>(B.nr, S, tile, sFlags, nf, cur.t0); break;
                case NR_FWSS: if (a2) bank_scan_tile<NR_FWSS, 2>(B.nr, S, tile, sFlags, nf, cur.t0); else bank_scan_tile<NR_FWSS, 1>(B.nr, S, tile, sFlags, nf, cur.t0); break;
                default: bank_scan_tile<NR_2FWSS, 1>(B.nr, S, tile, sFlags, nf, cur.t0); break;
            }
            __syncthreads();
        }
        // ---- energy of the spectrum handed to the filter bank (modes EN_NR / EN_IN), one warp per frame
        if (B.energy_mode == EN_NR || B.energy_mode == EN_IN) {
            const bool square = (B.energy_mode == EN_NR) || B.take_sqrt;
            for (int f = wv; f < nf; f += BANK_THREADS / 32) {
                const float e = half_spectrum_energy(tile + f * SPITCH, NBIN, square);
                if (lane == 0) B.energy[row0 + f] = e;
            }
        }
        // ---- filter bank, lane == frame; bands dealt to the warps in snake order (band widths grow with the band number)
        {
            const float4 *row4 = reinterpret_cast<const float4 *>(tile + lane * SPITCH);
            const bool want_log = (DST == DST_FEA) && (KIND == KIND_DCTC || KIND == KIND_TRAPLOG || (KIND == KIND_LOGSPEC && B.energy_mode != EN_BANDS));
            for (int i = 0;; i++) {
                const int b = i * (BANK_THREADS / 32) + ((i & 1) ? (BANK_THREADS / 32 - 1 - wv) : wv);
                if (i * (BANK_THREADS / 32) >= B.nb) break;
                if (b >= B.nb) continue;
                const int4 bnd = sBands[b];
                const float4 *r = row4 + bnd.x;
                const float4 *wq = sW4 + bnd.z;
                // four partial sums as two register pairs: one packed FMA (FFMA2, ctu_fft.cuh) per two taps, the same values
                cpx<float> a01 = mk<float>(0.f, 0.f), a23 = a01;
#pragma unroll 4
                for (int q = 0; q < bnd.y; q++) {
                    const float4 x = r[q], w = wq[q];
                    a01 = pfma(mk<float>(x.x, x.y), mk<float>(w.x, w.y), a01);
                    a23 = pfma(mk<float>(x.z, x.w), mk<float>(w.z, w.w), a23);
                }
                const float acc = (a01.x + a01.y) + (a23.x + a23.y);
                float y;
                if (B.inld) {
                    y = powf(acc, 0.33f) * B.inld_scale;
                    if (want_log) y = logf(y);
                } else {
                    y = want_log ? logf(acc) + B.log_offset : acc * B.lin_scale;
                }
                sY[lane * B.ypitch + b] = y;
            }
        }
        __syncthreads();                                                       // band tile complete; the spectrum tile is dead
        // ... so the next tile can come in while the second stage runs and the result is stored
        if (tid == 0 && nxt.valid) {
            const int nfn = min(TILE_F, nxt.T - nxt.t0);
            const unsigned bytes = (unsigned)nfn * SPITCH * sizeof(float);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy accesses to the tile (scan) before the async-proxy write
            mbar_expect_tx(bar, bytes);
            bulk_g2s(tile, spec + (nxt.row0 + nxt.t0) * SPITCH, bytes, bar);
        }
        const int od = B.out_dim;
        if (DST == DST_FB) {
            float *g = dst + row0 * B.nb;
            for (int i = tid; i < nf * B.nb; i += BANK_THREADS) {
                const int f = i / B.nb, b = i - f * B.nb;
                g[i] = sY[f * B.ypitch + b];
            }
        } else {
            const float *y = sY + lane * B.ypitch;
            if (KIND == KIND_DCTC) {
                // rows i and i + 8 in one pass over the band vector: each 16-byte read of y (four wavefronts: every lane its
                // own frame) feeds two rows, whose matrix reads are broadcasts; pad taps are zero, pad y entries are zero
                const float4 *y4 = reinterpret_cast<const float4 *>(y);
                constexpr int NW = BANK_THREADS / 32;
                for (int i = wv; i < B.nrows; i += 2 * NW) {
                    const float4 *m4 = reinterpret_cast<const float4 *>(sM + i * B.nbp);
                    cpx<float> a01 = mk<float>(0.f, 0.f), a23 = a01;
                    if (i + NW < B.nrows) {                                    // warp-uniform
                        const float4 *n4 = reinterpret_cast<const float4 *>(sM + (i + NW) * B.nbp);
                        cpx<float> b01 = a01, b23 = a01;
                        // unrolled four times, k_bank<dctc, fea, nr> spills
#pragma unroll 2
                        for (int q = 0; q < B.nbp / 4; q++) {
                            const float4 v = y4[q], m = m4[q], n = n4[q];
                            a01 = pfma(mk<float>(v.x, v.y), mk<float>(m.x, m.y), a01);
                            a23 = pfma(mk<float>(v.z, v.w), mk<float>(m.z, m.w), a23);
                            b01 = pfma(mk<float>(v.x, v.y), mk<float>(n.x, n.y), b01);
                            b23 = pfma(mk<float>(v.z, v.w), mk<float>(n.z, n.w), b23);
                        }
                        sO[lane * od + i + NW] = (b01.x + b01.y) + (b23.x + b23.y);
                    } else {
#pragma unroll 4
                        for (int q = 0; q < B.nbp / 4; q++) {
                            const float4 v = y4[q], m = m4[q];
                            a01 = pfma(mk<float>(v.x, v.y), mk<float>(m.x, m.y), a01);
                            a23 = pfma(mk<float>(v.z, v.w), mk<float>(m.z, m.w), a23);
                        }
                    }
                    sO[lane * od + i] = (a01.x + a01.y) + (a23.x + a23.y);
                }
            } else {
                // with the energy of the band values wanted, logspec arrives here in true scale
                const bool late_log = (KIND == KIND_LOGSPEC && B.energy_mode == EN_BANDS);
                for (int b = wv; b < B.nb; b += BANK_THREADS / 32) sO[lane * od + b] = late_log ? logf(y[b]) : y[b];
                if (B.energy_mode == EN_BANDS && wv == 0 && lane < nf) {
                    // fp64: with equal-loudness weights the band values are ~1e-20 and their squares leave the fp32 range
                    double acc = 0.5 * (double)y[0] * (double)y[0];
                    for (int b = 1; b < B.nb - 1; b++) acc += (double)y[b] * (double)y[b];
                    acc += 0.5 * (double)y[B.nb - 1] * (double)y[B.nb - 1];
                    B.energy[row0 + lane] = (float)log(acc * 2.0);
                }
            }
            __syncthreads();
            if (od == B.out_stride) {
                float *g = dst + row0 * od;                                    // whole rows: one contiguous run
                for (int i = tid; i < nf * od; i += BANK_THREADS) g[i] = sO[i];
            } else {
                for (int i = tid; i < nf * od; i += BANK_THREADS) {
                    const int f = i / od, col = i - f * od;
                    dst[(row0 + f) * B.out_stride + col] = sO[i];
                }
            }
        }
        // Band values written straight from the band tile: the next filter bank must wait for these reads.  The feature path
        // needs no barrier here: every read of the band tile (second stage) lies before the barrier in front of the store
        // loop, and the staging area is next written after the NEXT tile's band-tile barrier, which every thread reaches
        // only after its own stores -- one barrier per tile fewer for the early warps to wait at (ncu: 17-25 % of this
        // kernel's stall samples were barrier waits).
        if (DST == DST_FB) __syncthreads();
        cur = nxt;
    }
}

// ---- host side -------------------------------------------------------------------------------------------------------
struct BankTables {                      // device copies, built once per handle
    int4 *d_bands = nullptr;
    float4 *d_w4 = nullptr;
    float *d_m2 = nullptr;
    int wtot4 = 0, ypitch = 0;
};

// packs the fp32 weights of FrameParams (true weights x the power-of-two scale S) so that every band starts at a multiple
// of four bins: host vectors for upload
static inline void bank_pack(const FrameParams &P, std::vector<int4> &bands, std::vector<float> &w) {
    bands.clear(); w.clear();
    for (int b = 0; b < P.nb; b++) {
        const int lo = P.lo[b], hi = P.hi[b];
        const int k0 = lo & ~3, k1 = (hi + 4) & ~3;                           // [k0, k1) covers lo..hi; k1 <= 260 = SPITCH
        bands.push_back(make_int4(k0 / 4, (k1 - k0) / 4, (int)w.size() / 4, 0));
        for (int k = k0; k < k1; k++) w.push_back((k >= lo && k <= hi) ? P.w[P.woff[b] + k - lo] : 0.f);
    }
}

template <int KIND, int DST>
static inline int launch_bank_t(const BankParams &B, bool nr, const BatchDesc &bd, int64_t ntiles, int u0, int n_utts, int num_sms, const float *spec,
                                float *dst, cudaStream_t s, LaunchCtx *lc, std::string &err) {
    const BankSmem L = bank_smem(B.nb, B.nbp, B.ypitch, B.wtot4, B.nrows, B.out_dim);
    const size_t bytes = (size_t)L.total * sizeof(float);
    const int64_t units = nr ? n_utts : ntiles;
    if (units <= 0) return CTU_OK;
    cudaError_t e;
    int per_sm = 2;
    static const char *const names[2][2] = {{"k_bank<fb>", "k_bank<fea>"}, {"k_bank<nr,fb>", "k_bank<nr,fea>"}};
    lc->begin(names[nr ? 1 : 0][DST == DST_FEA ? 1 : 0], s);
    if (nr) {
        auto kern = k_bank<KIND, DST, true>;
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, BANK_THREADS, bytes);
        const unsigned grid = (unsigned)std::min<int64_t>(units, (int64_t)std::max(per_sm, 1) * num_sms);
        if (e == cudaSuccess) kern<<<grid, BANK_THREADS, bytes, s>>>(B, bd, (int)ntiles, u0, n_utts, spec, dst);
    } else {
        auto kern = k_bank<KIND, DST, false>;
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, BANK_THREADS, bytes);
        const unsigned grid = (unsigned)std::min<int64_t>(units, (int64_t)std::max(per_sm, 1) * num_sms);
        if (e == cudaSuccess) kern<<<grid, BANK_THREADS, bytes, s>>>(B, bd, (int)ntiles, u0, n_utts, spec, dst);
    }
    lc->end(s);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { err = std::string("CUDA: ") + cudaGetErrorString(e) + " (k_bank)"; return CTU_ERR_CUDA; }
    return CTU_OK;
}

// kind: KIND_* of the feature chain; to_fb: write band values (LPC epilogue / precise consumers) instead of features
static inline int launch_bank(const BankParams &B, int kind, bool to_fb, bool nr, const BatchDesc &bd, int64_t ntiles, int u0, int n_utts, int num_sms,
                              const float *spec, float *dst, cudaStream_t s, LaunchCtx *lc, std::string &err) {
    if (to_fb) return launch_bank_t<KIND_SPEC, DST_FB>(B, nr, bd, ntiles, u0, n_utts, num_sms, spec, dst, s, lc, err);
    switch (kind) {
        case KIND_SPEC: return launch_bank_t<KIND_SPEC, DST_FEA>(B, nr, bd, ntiles, u0, n_utts, num_sms, spec, dst, s, lc, err);
        case KIND_LOGSPEC: return launch_bank_t<KIND_LOGSPEC, DST_FEA>(B, nr, bd, ntiles, u0, n_utts, num_sms, spec, dst, s, lc, err);
        case KIND_DCTC: return launch_bank_t<KIND_DCTC, DST_FEA>(B, nr, bd, ntiles, u0, n_utts, num_sms, spec, dst, s, lc, err);
        case KIND_TRAPLOG: return launch_bank_t<KIND_TRAPLOG, DST_FEA>(B, nr, bd, ntiles, u0, n_utts, num_sms, spec, dst, s, lc, err);
    }
    err = "CTU: bad kind";
    return CTU_ERR_CONFIG;
}

}  // namespace ctu
#endif
