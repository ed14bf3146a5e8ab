// Parameter blocks of the cross-frame stages (noise-reduction scans, Burg detector, VAD module, synthesis), the
// per-frame recursion step shared by the standalone scan kernels and k_bank, and the prototypes of the launchers whose
// kernels are compiled in their own translation units (ctu_nr.cu, ctu_burg.cu).
#ifndef CTU_NR_PARAMS_CUH
#define CTU_NR_PARAMS_CUH

#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>

#include "ctu_internal.h"
#include "ctu_kernels.cuh"
#include "ctu_any64.cuh"

namespace ctu {

constexpr int BURG_MAXC = 16;     // cepstral coefficients kept per frame (pitch of d_ceps)
enum { BURG_SRC_NR = 0, BURG_SRC_VAD = 1 };

struct NrParams {
    int mode;            // CtuNrMode
    float a, b, p;
    double ad, pd;
    int a_kind;          // 1: a == 1, 2: a == 2, 0: general
    int initsegs;
    int carry_xform;     // list semantics on the band path: what FEA does IN PLACE to the band vector that the next file's noise
                         // estimate starts from -- 1: log (dctcFEA, src/fea/fea_impl.cc:108), 2: square (lpaFEA without the
                         // cube-root law, :166-169), 0: nothing
};

struct SynthParams {
    double correction;   // max over offsets of the summed overlapping Hamming windows
    int hh;              // frames before a tile that still overlap its first sample
};

struct BurgParams {
    int window, wshift, remove_dc;
    double preem;
    int fb_power;        // spectrum handed to NR is power (else magnitude)
    int a_kind; double a;  // expansion applied before the detector (hwss/fwss); 2fwss: none
    int expand;          // 0 for 2fwss
    int ncoef_nr;        // fea_ncepcoefs (src/nr/nr.cc:266-270)
    int ncoef_vad;       // vad_lpc_coefs
    int ninit; double P, Q;   // detector options <- (nr_initsegs, nr_p, nr_q)
    int use_spec_gain;   // VAD source: post-NR spectrum present (gain from d_spec) else own spectrum
    // FFT sizes other than 512: the general kernel k_burg_any (nfft == 0: the specialised k_burg)
    int nfft, log2m;
    const double2 *any_tw, *any_ts;
    int spitch;          // floats per row of the spectrum matrix
};

struct VadParams {
    int cri, thr, drop;
    int energy_db;
    int latency;         // rows between a feature row and the spectrum frame the VAD sees
    int order;           // majority filter length
    int cep_n;           // length of the cepstral vector (lpc: vad_lpc_coefs, fea: feature dim)
    int nbins;           // spectrum bins per frame (wfft/2 + 1)
    int spitch;          // floats per row of the spectrum matrix
    int has_E;           // last column of the feature rows is the _E column
    int fea_skip;        // fea criterion: WRITER column holding the reference's internal element 0 (left out of the
                         // distance, src/vad/vad.cc:262-272), or -1 when that element is not written at all
    int cep_init; double cep_p;
    double abs_thr;
    int perc_init; double perc_thr;
    int adapt_init; double adapt_q, adapt_za;
    int dyn_init; double dyn_perc, dyn_min, qmaxinc, qmaxdec, qmindec, qmininc;
    // -vad_out_mode debug: per step VAD_DBG doubles (criterion, threshold, three values of the threshold's state), else null
    double *dbg;
};
constexpr int VAD_DBG = 5;

// ------------------------------------------------------------------------------------------
static inline int build_nr_params(const ctu_config &c, int nr_mode, int vad_src, bool signal_out, int nb, NrParams &N, SynthParams &S,
                                  BurgParams &B, VadParams &V, std::string &err) {
    std::memset(&N, 0, sizeof(N)); std::memset(&S, 0, sizeof(S)); std::memset(&B, 0, sizeof(B)); std::memset(&V, 0, sizeof(V));
    N.mode = nr_mode;
    N.a = (float)c.nr_a; N.b = (float)c.nr_b; N.p = (float)c.nr_p; N.ad = c.nr_a; N.pd = c.nr_p;
    N.a_kind = (c.nr_a == 1.0) ? 1 : (c.nr_a == 2.0) ? 2 : 0;
    N.initsegs = c.nr_initsegs;
    // OLA correction (src/io/out.cc:346-372)
    {
        const int s = c.wshift, w = c.window;
        double pi = 2. * asin(1.), corr = 0.;
        for (int i = 0; i < s; i++) {
            int x = i; double y = 0.;
            while (x < w) { y += 0.54 - (1 - 0.54) * cos(2 * pi * (double)x / (w - 1.)); x += s; }
            if (y > corr) corr = y;
        }
        S.correction = corr;
        S.hh = (w + s - 1) / s - 1;
    }
    B.window = c.window; B.wshift = c.wshift; B.remove_dc = c.remove_dc; B.preem = (double)c.preem;
    B.fb_power = c.fb_power;
    B.a = c.nr_a; B.a_kind = N.a_kind; B.expand = (nr_mode != NR_2FWSS);
    B.ncoef_nr = c.fea_ncepcoefs; B.ncoef_vad = c.vad_lpc_coefs;
    B.ninit = c.nr_initsegs; B.P = c.nr_p; B.Q = c.nr_q;
    B.use_spec_gain = (nr_mode != NR_NONE && c.nr_when == 0);
    if (nr_mode >= NR_HWSS && vad_src == VADSRC_BURG && (c.fea_ncepcoefs > BURG_MAXC || c.fea_ncepcoefs < 2)) {
        err = "CTU: Burg detector supports 2..16 cepstral coefficients"; return CTU_ERR_UNSUPPORTED;
    }
    V.energy_db = c.vad_energy_db;
    V.order = c.vad_filter_order;
    V.cep_init = c.vad_cepdist_init; V.cep_p = c.vad_cepdist_p;
    V.abs_thr = c.vad_absolute_thr;
    V.perc_init = c.vad_perc_init; V.perc_thr = c.vad_perc_thr;
    V.adapt_init = c.vad_adapt_init; V.adapt_q = c.vad_adapt_q; V.adapt_za = c.vad_adapt_za;
    V.dyn_init = c.vad_dyn_init; V.dyn_perc = c.vad_dyn_perc; V.dyn_min = c.vad_dyn_min;
    V.qmaxinc = c.vad_dyn_qmaxinc; V.qmaxdec = c.vad_dyn_qmaxdec; V.qmindec = c.vad_dyn_qmindec; V.qmininc = c.vad_dyn_qmininc;
    // latency of the feature chain as BATCH::save_frame sees it (src/io/batch.cc:172-204)
    V.latency = 0;
    std::string kind(c.fea_kind);
    if (kind != "trapdct" && kind != "lpa" && c.fea_delta) {      // deltas, or one stage used as the -fea_trap window
        int wins[3] = {c.d_win, c.a_win, c.t_win};
        for (int k = 0; k < c.n_order; k++) V.latency += wins[k];
    }
    if (kind == "trapdct") V.latency = (c.fea_trapdct_traplen + 1) / 2 - 1;
    (void)signal_out; (void)nb;
    return CTU_OK;
}

// ------------------------------------------------------------------------------------------
// K2 / K3: noise-reduction scans
// ------------------------------------------------------------------------------------------
// One thread per (utterance, bin), frames walked in blocks of SCAN_UNROLL: all loads of a
// block are issued before the (sequentially dependent) recursion touches them and all
// stores after it, so each thread keeps SCAN_UNROLL x 4 B of reads in flight.  MODE / AKIND
// are compile-time so the hot loop carries only the state it needs (register count decides
// how many bytes per SM are in flight, and this kernel is HBM-bound).
constexpr int SCAN_UNROLL = 16;

struct ScanState { float Navg, Yavg, Nravg; double Nd, Yd; };

__device__ __forceinline__ float fast_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float fast_rsqrt(float x) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

// one frame of the recursion for one bin
template <int MODE, int AKIND>
__device__ __forceinline__ float nr_step(const NrParams &N, ScanState &S, float xi, int t, uint8_t flag) {
    const float p = N.p, q = 1.f - N.p;
    if (MODE == NR_EXTEN) {
        if (AKIND == 0) {                   // general exponent: fp64, as the reference writes it
            double Hd = S.Nd / pow(pow(S.Nd, N.ad) + pow(S.Yd, N.ad), 1. / N.ad);
            double xd = (double)xi, Nn = Hd * xd;
            S.Nd = N.pd * S.Nd + (1 - N.pd) * Nn;
            S.Yd = fabs(xd - S.Nd);
            return (float)(xd - Nn);
        }
        // H = Navg/(Navg+Yavg) (a=1) or Navg/hypot(Navg,Yavg) (a=2); the output X-H*X is formed
        // as X*(1-H) with 1-H written without cancellation.  Reciprocal and reciprocal square root are the hardware
        // approximations (MUFU, <= 2 ulp): the IEEE-rounded forms wrap each of them in a range check, two fix-up FMAs and
        // a slow-path branch -- 10 of the 25 instructions of a step in the fused scan (ncu, profiles/r02_*), which is issue
        // bound -- and the recursion is a contraction (p < 1), so the extra ulp does not accumulate
        float H, omH;
        if (AKIND == 1) {
            const float r = fast_rcp(S.Navg + S.Yavg);
            H = S.Navg * r; omH = S.Yavg * r;
        } else {
            const float h2 = fmaf(S.Navg, S.Navg, S.Yavg * S.Yavg);
            const float ri = fast_rsqrt(h2);                  // 1 / hypot
            const float hh = h2 * ri;                         // hypot
            H = S.Navg * ri;
            omH = S.Yavg * S.Yavg * fast_rcp(hh * (hh + S.Navg));
        }
        const float Nn = H * xi;
        S.Navg = fmaf(p, S.Navg, q * Nn);
        S.Yavg = fabsf(xi - S.Navg);
        return xi * omH;
    }
    // hwss decrements its counter before use, fwss / 2fwss after (src/nr/nr.cc:226, 367, 440)
    const int ninit = (MODE == NR_HWSS) ? N.initsegs - (t + 1) : N.initsegs - t;
    const bool upd = (flag == 0) || ninit > 0;
    if (MODE == NR_2FWSS) {
        if (upd) S.Navg = fmaf(p, S.Navg, q * xi);
        xi = fabsf(xi - S.Navg);
        if (upd) S.Nravg = fmaf(p, S.Nravg, q * xi);
        return fabsf(xi - S.Nravg);
    }
    if (AKIND == 2) xi = xi * xi;
    else if (AKIND == 0) xi = powf(xi, N.a);
    if (upd) S.Navg = fmaf(p, S.Navg, q * xi);
    xi = xi - N.b * S.Navg;
    if (MODE == NR_HWSS) { if (xi < 0.f) xi = 0.f; }
    else if (xi < 0.f) xi = -xi;
    if (AKIND == 2) xi = sqrtf(xi);
    else if (AKIND == 0) xi = powf(xi, 1.f / N.a);
    return xi;
}

// ------------------------------------------------------------------------------------------
// shared front end in double precision for one frame held by a 16-thread group
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double group_sum16d(double v) {
    const unsigned m = 0xffffu << (threadIdx.x & 16);
    v += __shfl_xor_sync(m, v, 8);
    v += __shfl_xor_sync(m, v, 4);
    v += __shfl_xor_sync(m, v, 2);
    v += __shfl_xor_sync(m, v, 1);
    return v;
}

// geometry shared with the host orchestration (the kernels live in ctu_nr_kernels.cuh / ctu_burg.cuh, each its own
// translation unit)
constexpr int SYN_THREADS = 256;
constexpr int SYN_GROUPS = SYN_THREADS / GROUP;
constexpr int SYN_FRAMES = SYN_GROUPS;

// ---- launchers defined in ctu_nr.cu / ctu_burg.cu -------------------------------------------------------------------
int launch_nr_scan(const NrParams &N, const int *d_nframes, const int64_t *d_row_off, int u0, int u1, int size, int pitch, float *X,
                   const uint8_t *flags, cudaStream_t s, LaunchCtx *lc, std::string &err);
int launch_nr_scan_carry(const NrParams &N, const int *d_nframes, const int64_t *d_row_off, int u0, int u1, int size, int pitch, float *X,
                         const uint8_t *flags, float *carry, const float2 *cspec, cudaStream_t s, LaunchCtx *lc, std::string &err);
int launch_burg(const BurgParams &B, int src_mode, const BatchDesc &bd, int64_t ntiles, const int16_t *pcm, const float *spec,
                double *ceps, const double2 *tw, const double2 *ts, const double2 *ti, const double *win, const double *hann,
                cudaStream_t s, LaunchCtx *lc, std::string &err);
int launch_cepdet(const BurgParams &B, const int *d_nframes, const int64_t *d_row_off, int u0, int u1, const double *ceps,
                  uint8_t *flags, cudaStream_t s, LaunchCtx *lc, std::string &err);
int launch_synth_c(const SynthParams &S, const FrameParams &F, const BatchDesc &bd, int tile_frames, int64_t ntiles,
                   const int64_t *d_osamp_off, const float2 *cspec, const float *spec, int16_t *out, const float2 *tw,
                   const float2 *ti, cudaStream_t s, LaunchCtx *lc, std::string &err);
int launch_vad_module(VadParams V, const BurgParams &B, const BatchDesc &bd32, int64_t nt32, const int *d_nframes,
                      const int64_t *d_row_off, int u0, int u1, int64_t row0, int64_t nrows, const int16_t *d_pcm,
                      const float *d_spec, float *d_fea, const double *d_fea64, int fea_dim, double *d_ceps, double *d_cri,
                      uint8_t *d_vad0, uint8_t *d_vadout, uint8_t *d_keep, int *d_rows, const double2 *tw, const double2 *ts,
                      const double2 *ti, const double *win, cudaStream_t s, LaunchCtx *lc, std::string &err);

}  // namespace ctu
#endif
