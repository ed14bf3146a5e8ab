// Host orchestration behind the C ABI (include/ctucopy_b200.h): table design in fp64,
// plan (frame/tile bookkeeping, workspaces), kernel sequencing per configuration, and the
// chunked H2D / compute / D2H pipeline of the end-to-end entry point.
// This is the GPU replacement of BATCH::process / process_frame / flush_fea
// (src/io/batch.cc:205-422).  There is NO CPU fallback anywhere in this file: without a
// CUDA device ctu_create fails with CTU_ERR_CUDA.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "ctu_internal.h"
#include "ctu_kernels.cuh"
#include "ctu_frames2.cuh"
#include "ctu_frames_any.cuh"
#include "ctu_nr_params.cuh"
#include "ctu_precise.cuh"
#include "ctu_tdiir.cuh"
#include "ctu_frames256.cuh"
#include "ctu_bank.cuh"
#include "ctu_synth_any.cuh"

using namespace ctu;

// glibc's rand() after srand(1) (random_r TYPE_3: r[i] = r[i-3] + r[i-31] mod 2^32, output r[i] >> 1, 310 values
// discarded after seeding), which the reference draws once per loaded sample (src/io/in.cc:205, 452-455)
struct GlibcRand {
    uint32_t r[34];
    int i = 0;
    GlibcRand() {
        int64_t v = 1;
        uint32_t init[34];
        init[0] = 1;
        for (int k = 1; k < 31; k++) { v = (16807 * (int64_t)init[k - 1]) % 2147483647; if (v < 0) v += 2147483647; init[k] = (uint32_t)v; }
        for (int k = 31; k < 34; k++) init[k] = init[k - 31];
        for (int k = 0; k < 34; k++) r[k] = init[k];
        i = 0;                                   // r[(i + k) % 34] holds element (count + k) of the sequence, k < 34
        for (int k = 0; k < 310; k++) step();
    }
    inline uint32_t step() {                      // element n = element n-31 + element n-3; the window holds n-34 .. n-1
        const uint32_t v = r[(i + 3) % 34] + r[(i + 31) % 34];
        r[i] = v;
        i = (i + 1) % 34;
        return v;
    }
    inline uint32_t next() { return step() >> 1; }
};

// ------------------------------------------------------------------------------------------
struct ctu_handle {
    ctu_config cfg;
    int device = 0, num_sms = 148;
    std::string err;
    LaunchCtx lc;
    CtuFbDesign fb;
    int fea_kind = FEA_NONE, nr_mode = NR_NONE, vad_src = VADSRC_NONE;
    bool signal_out = false, do_vad = false, vad_drop = false;
    int vad_cri = VCRI_ENERGY, vad_thr = VTHR_PERC;
    int static_dim = 0, feature_dim = 0;
    int energy_mode = 0, energy_latency = 0;   // optional _E column (last column of every row)
    // context stacking / deltas of non-cepstral vectors / feature-file input: the static block is gathered from a
    // separate matrix by k_stack (the frame kernels' output, or the caller's feature rows)
    bool gather = false, fea_in = false;
    StackParams skp;
    int in_dim = 0;                            // floats per input row (feature input)
    int work_dim = 0;                          // row width the chain computes (= feature_dim + columns the writer cuts)
    int cms_cols = 0;                          // leading columns -fea_Z_exp normalises
    FrameParams fp;      // filter bank + second stage tables
    DeltaParams dp;
    TrapParams tp;
    NrParams nrp{};
    SynthParams sp{};
    BurgParams bp{};
    VadParams vp{};
    // device tables
    float2 *d_tw256 = nullptr, *d_twsplit = nullptr, *d_twinv = nullptr;
    float *d_win = nullptr;
    // FFT sizes other than 512 (ctu_frames_any.cuh)
    bool generic = false;
    int nbins = NBIN;
    int spitch = SPITCH;                       // floats per row of the spectrum matrix (general FFT sizes: = nbins)
    BankTables bank;                           // k_bank's packed filter bank (512-point feature chains)
    BankParams bkp{};
    float2 *d_any_tw = nullptr, *d_any_ts = nullptr;
    float2 *d_tw128 = nullptr;                 // 256-point front end (ctu_frames256.cuh): W128^(g k1)
    double2 *d_any_tw64 = nullptr, *d_any_ts64 = nullptr;     // fp64 copies for the general synthesis (ctu_synth_any.cuh)
    float *d_any_fbw = nullptr;
    int4 *d_any_bands = nullptr;
    std::vector<float> fbw_all;
    std::vector<int4> bands_all;
    double2 *d_tw256d = nullptr, *d_twsplitd = nullptr, *d_twinvd = nullptr;
    double *d_wind = nullptr, *d_hann = nullptr;
    // fp64 tables of the precise path (ctu_precise.cuh)
    bool precise = false;
    std::vector<double> w64, m264, lift64;
    double *d_w64 = nullptr, *d_m264 = nullptr, *d_lift64 = nullptr;
    // -fea_kind td-iir-mfcc (ctu_tdiir.cuh)
    TdiirParams tdp{};
    double *d_td_coefs = nullptr, *d_td_win = nullptr, *d_td_dct = nullptr;
    cudaStream_t streams[3] = {nullptr, nullptr, nullptr};
    // device blocks of destroyed plans, kept for the next plan: a list is processed as a sequence of plans of
    // similar size, and cudaMalloc / cudaFree of gigabytes cost more than the kernels that use them
    int16_t *d_g711[2] = {nullptr, nullptr};   // expansion tables (mu-law, A-law), uploaded on first use
    uint64_t rand_pos = 0;               // -dither: values of the process-wide rand() stream drawn by earlier plans
    GlibcRand rand_gen;                  // generator state after rand_gen_pos values (a list is a sequence of plans: the next
    uint64_t rand_gen_pos = 0;           // plan resumes here instead of stepping from the seed again)
    // run-time knobs outside the reference's option set (ctu_set_option; the environment gives the defaults)
    int copy_only = 0;                   // host entry points: copies only, kernels skipped (control measurement)
    int chunk_mb = 32;                   // MB of PCM per pipeline chunk of the host entry points
    int fuse_nr = 1;                     // 1: the noise-reduction scan runs inside k_bank (tile in shared memory) where it can
    int front256 = 1;                    // 1: 256-point frames take k_frames256 for PCM -> spectrum; 0: the general kernel throughout
    int compact_static = 1;              // 1: cepstra behind a delta chain are written as compact rows and the delta kernel writes the whole output row
    // hwss / fwss / 2fwss with the reference's LIST semantics (a file's noise estimate starts from the enhanced last frame of
    // the file before it, src/nr/nr.cc:212-222, 397-408): opt-in, one handle = one list walked in order on one GPU
    int ss_carry = 0;
    float *d_carry = nullptr;            // the shared spectrum buffer between utterances, ranges, plans and calls
    double *d_carry64 = nullptr;         // ... on the fp64 band path (noise reduction after the filter bank)
    cudaEvent_t carry_ev = nullptr;      // orders the chained scans of consecutive chunks, which run on different streams
    bool carry_ev_set = false;
    struct PoolBlock { void *p; size_t bytes; bool used; };
    std::vector<PoolBlock> pool;
};

struct ctu_plan {
    ctu_handle *h = nullptr;
    int n_utts = 0;
    std::vector<int64_t> offsets;        // n_utts+1 sample offsets
    std::vector<int> nframes;
    std::vector<int64_t> row_off;        // n_utts+1
    std::vector<int64_t> osamp_off;      // n_utts+1 (signal output)
    std::vector<int64_t> tile32_off, tile64_off, tileS_off, tileF_off;   // n_utts+1 (S: synthesis tiles of syn_tile hops)
    int syn_tile = 0;
    std::vector<int64_t> rows_per_utt;
    int64_t total_frames = 0, total_osamp = 0, total_samples = 0;
    // device bookkeeping
    int64_t *d_pcm_off = nullptr, *d_row_off = nullptr, *d_osamp_off = nullptr, *d_t32_off = nullptr, *d_t64_off = nullptr;
    int *d_nframes = nullptr;
    int2 *d_tiles32 = nullptr, *d_tiles64 = nullptr, *d_tilesS = nullptr, *d_tilesF = nullptr;
    int64_t *d_tS_off = nullptr, *d_tF_off = nullptr;
    // workspaces (whole batch)
    float *d_spec = nullptr, *d_fb = nullptr, *d_log = nullptr;
    float *d_static = nullptr;           // static block before k_stack (gather modes)
    float *d_work = nullptr;             // full-width rows when the writer cuts the last column (feature input)
    float *d_in = nullptr;               // feature input rows (host entry point)
    float2 *d_cspec = nullptr;           // complex spectrum kept for the synthesis (k_synth_c)
    double *d_yt = nullptr;              // synthesised frames [frames x window] of the general synthesis
    double *d_fb64 = nullptr;            // band values of the precise path
    double *d_fea64 = nullptr;           // fp64 copy of the feature matrix (feature-vector VAD criterion)
    float *d_E = nullptr;                // log energy per frame (-fea_E)
    double *d_dc1 = nullptr;             // ring means per frame (-remove_dc1)
    float *d_dither = nullptr;           // dither noise per sample (-dither), generated on first use
    uint64_t rand_base = 0;
    bool dither_ready = false;
    double *d_ceps = nullptr;            // Burg cepstra [frames x ncoef]
    double *d_tdseg = nullptr;           // td-iir-mfcc: windowed band energies per segment of gcd(window, shift) samples
    double *d_cri = nullptr;             // VAD criterion per frame
    double *d_vdbg = nullptr;            // -vad_out_mode debug: VAD_DBG doubles per VAD step
    uint8_t *d_flags = nullptr;          // NR-internal detector decisions
    uint8_t *d_keep = nullptr;           // VAD module: row kept
    uint8_t *d_vad0 = nullptr;           // VAD module: unfiltered decisions
    int *d_rows = nullptr;               // rows written per utterance (drop mode)
    int64_t workspace_bytes = 0;
    // buffers owned for the host entry point
    int16_t *d_pcm = nullptr, *d_wave = nullptr;
    uint8_t *d_codes = nullptr;          // G.711 codes as uploaded (ctu_plan_run_host_g711)
    float *d_fea = nullptr;
    uint8_t *d_ext = nullptr, *d_vadnr_out = nullptr, *d_vad_out = nullptr;
    bool host_bufs = false;
    int row_format = 0;                  // CTU_ROWS_*: layout of the rows the host entry points hand back
    uint32_t sent0 = 0;                  // pfile rows: sentence number of the plan's first utterance
    uint32_t *d_fmt = nullptr;           // pfile rows on the device [rows x (dim + 2)]
    std::vector<void *> blocks;          // this plan's blocks of the handle's pool
};

static thread_local std::string g_create_err;

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            h->err = std::string("CUDA: ") + cudaGetErrorString(e_) + " at " #call;                \
            return CTU_ERR_CUDA;                                                                   \
        }                                                                                          \
    } while (0)

static int fail(ctu_handle *h, int code, const std::string &m) {
    h->err = m;
    return code;
}

const char *ctu_last_error(const ctu_handle *h) { return h ? h->err.c_str() : g_create_err.c_str(); }
int ctu_feature_dim(const ctu_handle *h) { return h ? h->feature_dim : 0; }
int ctu_input_dim(const ctu_handle *h) { return (h && h->fea_in) ? h->in_dim : 0; }
int ctu_is_signal_output(const ctu_handle *h) { return h && h->signal_out; }
int ctu_num_bands(const ctu_handle *h) { return h ? h->fb.nb : 0; }
uint64_t ctu_launch_count(const ctu_handle *h) { return h ? h->lc.launches : 0; }

int ctu_profile_enable(ctu_handle *h, int on) {
    if (!h) return CTU_ERR_CONFIG;
    h->lc.clear();
    h->lc.prof_on = on != 0;
    return CTU_OK;
}
int ctu_profile_count(const ctu_handle *h) { return h ? (int)h->lc.recs.size() : 0; }
int ctu_profile_get(ctu_handle *h, int idx, const char **name, float *ms) {
    if (!h || idx < 0 || idx >= (int)h->lc.recs.size()) return CTU_ERR_CONFIG;
    auto &r = h->lc.recs[idx];
    CK(cudaEventSynchronize(r.b));
    float t = 0;
    CK(cudaEventElapsedTime(&t, r.a, r.b));
    if (name) *name = r.name;
    if (ms) *ms = t;
    return CTU_OK;
}

int ctu_design_filter_bank(const ctu_config *cfg, double *mat, int32_t *lo, int32_t *hi, int32_t *nb) {
    CtuFbDesign d;
    std::string e = ctu_design_fb(*cfg, d);
    if (!e.empty()) { g_create_err = e; return CTU_ERR_CONFIG; }
    if (nb) *nb = d.nb;
    if (mat) std::copy(d.mat.begin(), d.mat.end(), mat);
    if (lo) std::copy(d.lo.begin(), d.lo.end(), lo);
    if (hi) std::copy(d.hi.begin(), d.hi.end(), hi);
    return CTU_OK;
}

int ctu_fb_matrix(const ctu_handle *h, double *mat, int32_t *lo, int32_t *hi) {
    if (!h || h->fb.nb == 0) return CTU_ERR_CONFIG;
    if (mat) std::copy(h->fb.mat.begin(), h->fb.mat.end(), mat);
    if (lo) std::copy(h->fb.lo.begin(), h->fb.lo.end(), lo);
    if (hi) std::copy(h->fb.hi.begin(), h->fb.hi.end(), hi);
    return CTU_OK;
}

int64_t ctu_num_frames(const ctu_handle *h, int64_t n) {
    if (!h) return -1;
    if (h->fea_in) return n;                        // feature input: a row is a frame
    const int w = h->cfg.window, s = h->cfg.wshift;
    if (n < w - s) return -1;                       // "IO: Signal shorter than one frame!"
    return (n - (w - s)) / s;
}

int64_t ctu_num_output_samples(const ctu_handle *h, int64_t n) {
    int64_t T = ctu_num_frames(h, n);
    if (T < 0) return -1;
    if (h->fea_in) return 0;
    return T * h->cfg.wshift + (h->cfg.window - h->cfg.wshift);
}

// ------------------------------------------------------------------------------------------
// table construction (host, fp64)
// ------------------------------------------------------------------------------------------
template <class T> static int upload(ctu_handle *h, T **dst, const std::vector<T> &v) {
    CK(cudaMalloc((void **)dst, std::max<size_t>(1, v.size()) * sizeof(T)));
    // pageable source: cudaMemcpy may return once the data is staged, and the consumers run on cudaStreamNonBlocking
    // streams that do not order against the legacy stream -- wait for the DMA itself
    if (!v.empty()) { CK(cudaMemcpy(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice)); CK(cudaDeviceSynchronize()); }
    return CTU_OK;
}

static int build_fft_tables(ctu_handle *h) {
    const double PI = 3.14159265358979323846264338327950288;
    std::vector<float2> tw(256), ts(129), ti(129);
    std::vector<double2> twd(256), tsd(129), tid_(129);
    for (int k1 = 0; k1 < 16; k1++)
        for (int c = 0; c < 16; c++) {
            double a = -2 * PI * (double)(c * k1) / 256.0;
            twd[k1 * 16 + c] = make_double2(cos(a), sin(a));
            tw[k1 * 16 + c] = make_float2((float)cos(a), (float)sin(a));
        }
    for (int k = 0; k <= 128; k++) {
        double th = 2 * PI * k / 512.0;
        tsd[k] = make_double2(-sin(th) / 2, -cos(th) / 2);
        ts[k] = make_float2((float)(-sin(th) / 2), (float)(-cos(th) / 2));
        tid_[k] = make_double2(cos(th), sin(th));
        ti[k] = make_float2((float)cos(th), (float)sin(th));
    }
    // analysis window: Hamming, pi = 2*asin(1) (src/io/in.cc:139-144)
    const int w = h->cfg.window;
    std::vector<float> win(w);
    std::vector<double> wind(w), hann(w);
    double pi = 2. * asin(1.);
    for (int j = 0; j < w; j++) {
        wind[j] = 0.54 - (1 - 0.54) * cos(2 * pi * j / (w - 1.));
        win[j] = (float)wind[j];
        // Hann of the cepstral detector, its own 10-digit pi (src/vdet/CepstralDet.h:126-131)
        hann[j] = 0.5 * (1 - cos((2 * 3.141592653 / w) * j));
    }
    int st;
    if ((st = upload(h, &h->d_tw256, tw))) return st;
    if ((st = upload(h, &h->d_twsplit, ts))) return st;
    if ((st = upload(h, &h->d_twinv, ti))) return st;
    if ((st = upload(h, &h->d_win, win))) return st;
    if ((st = upload(h, &h->d_tw256d, twd))) return st;
    if ((st = upload(h, &h->d_twsplitd, tsd))) return st;
    if ((st = upload(h, &h->d_twinvd, tid_))) return st;
    if ((st = upload(h, &h->d_wind, wind))) return st;
    if ((st = upload(h, &h->d_hann, hann))) return st;
    return CTU_OK;
}

static int build_frame_params(ctu_handle *h) {
    const ctu_config &c = h->cfg;
    FrameParams &P = h->fp;
    std::memset(&P, 0, sizeof(P));
    P.window = c.window; P.wshift = c.wshift;
    P.preem = c.preem;
    P.remove_dc = c.remove_dc;
    P.take_sqrt = !c.fb_power;
    P.inld_scale = 1.f; P.lin_scale = 1.f; P.log_offset = 0.f;
    if (h->signal_out || h->fea_in) return CTU_OK;
    const CtuFbDesign &fb = h->fb;
    if (fb.nb > MAXB) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: more than 64 filter-bank bands");
    P.nb = fb.nb;
    P.inld = fb.inld;
    // Equal-loudness weights are ~1e-30 above 10 kHz sampling (src/fea/fb.cc:157-164): carry
    // an exact power-of-two factor S in the packed fp32 weights and undo it after the
    // non-linearity, so that quiet frames do not go denormal.
    double wmax = 0;
    for (double v : fb.mat) if (std::isfinite(v)) wmax = std::max(wmax, std::fabs(v));
    int e = 0;
    if (wmax > 0 && wmax < 1e-6) { std::frexp(wmax, &e); e = -e; }
    const double S = std::ldexp(1.0, e);
    P.inld_scale = (float)std::pow(S, -0.33);
    P.lin_scale = (float)(1.0 / S);
    P.log_offset = (float)(-std::log(S));
    int off = 0;
    for (int b = 0; b < fb.nb; b++) {
        int n = fb.hi[b] - fb.lo[b] + 1;
        if (!h->generic && off + n > MAXW) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: filter bank has too many taps");
        off = (off + 3) & ~3;
        if (!h->generic && off + n > MAXW) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: filter bank has too many taps");
        P.lo[b] = (short)fb.lo[b]; P.hi[b] = (short)fb.hi[b]; P.woff[b] = off;
        h->w64.resize(off + n, 0.0);            // same (4-aligned) offsets as the fp32 copy
        h->fbw_all.resize(off + n, 0.f);
        h->bands_all.push_back(make_int4(fb.lo[b], n, off, 0));
        for (int k = 0; k < n; k++) {
            const float wv = (float)(fb.mat[(size_t)b * fb.bins + fb.lo[b] + k] * S);
            if (off + k < MAXW) P.w[off + k] = wv;           // the general kernel reads its taps from global memory
            h->fbw_all[off + k] = wv;
            h->w64[off + k] = fb.mat[(size_t)b * fb.bins + fb.lo[b] + k];
        }
        off += n;
    }
    // second stage
    const int nb = fb.nb;
    const int nbp = (nb + 3) & ~3;
    P.nbp = nbp;
    const int N = c.fea_ncepcoefs;
    std::vector<double> lift(N + 1, 1.0);
    if (c.fea_lifter > 1)
        for (int n = 1; n <= N; n++) lift[n] = 1 + ((double)c.fea_lifter) / 2 * sin(3.141592653589793 * (double)n / ((double)c.fea_lifter));
    switch (h->fea_kind) {
        case FEA_SPEC: case FEA_LOGSPEC: case FEA_TRAPDCT:
            h->static_dim = nb;
            break;
        case FEA_DCTC: {
            // c[i] = sqrt(2/N) sum_k ln Y_k cos(pi i (k-1/2)/N), lifter on i >= 1, pi = 3.1415926535898
            // (src/fea/fea_impl.cc:81-131); rows stored in WRITER order c1..cN, c0 (src/io/out.cc:189-201)
            int rows = N + (c.fea_c0 ? 1 : 0);
            if (rows > MAXR || rows * nbp > MAXM2) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: cepstral matrix too large");
            double norm = sqrt(2.0 / nb);
            auto wd = [&](int id) { return cos(3.1415926535898 * (double)id / (2 * nb)); };
            for (int r = 0; r < rows; r++) {
                int i = (r < N) ? r + 1 : 0;
                for (int k = 1; k <= nb; k++) {
                    int id = ((2 * k - 1) * i) % (4 * nb);
                    P.m2[r * nbp + k - 1] = (float)(wd(id) * norm * (i >= 1 ? lift[i] : 1.0));
                    h->m264.push_back(wd(id) * norm * (i >= 1 ? lift[i] : 1.0));
                }
            }
            P.nrows = rows;
            h->static_dim = rows;
            break;
        }
        case FEA_LPA: case FEA_LPC: {
            const int p = c.fea_lporder;
            if (p + 1 > MAXR || (p + 1) * nbp > MAXM2 || N + 1 > MAXR) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: LP order too large");
            if (nb < 2) return fail(h, CTU_ERR_CONFIG, "CTU: LPC needs at least two bands");
            const int Nf = (nb - 1) * 2;
            for (int k = 0; k <= p; k++)
                for (int n = 0; n < nb; n++) {
                    double v;
                    if (n == 0) v = 0.5;
                    else if (n == nb - 1) v = (1 - 2 * (k % 2)) * 0.5;
                    else v = cos(2 * 3.141592653589793 * ((n * k) % Nf) / Nf);
                    P.m2[k * nbp + n] = (float)(v / ((double)Nf / 2));
                    h->m264.push_back(v / ((double)Nf / 2));
                }
            P.nrows = p + 1;
            P.lporder = p; P.ncep = N;
            P.lpa_square = !fb.inld;
            P.c0_last = c.fea_c0;
            for (int n = 0; n <= N; n++) P.lift[n] = (float)lift[n];
            h->lift64 = lift;
            if (!fb.inld) h->precise = true;      // LPC from squared band powers: ill-conditioned
            if (h->fea_kind == FEA_LPA) {
                // htkOUT writes a[1..ncep] with the cepstral loop bounds (src/io/out.cc:189-201):
                // only lporder == ncepcoefs is memory-safe in the reference
                if (p != N) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: -fea_kind lpa needs fea_lporder == fea_ncepcoefs (the reference overruns its buffers otherwise)");
                h->static_dim = p;
            } else {
                h->static_dim = N + (c.fea_c0 ? 1 : 0);
            }
            break;
        }
        default: break;
    }
    return CTU_OK;
}


static int build_delta_trap_params(ctu_handle *h) {
    const ctu_config &c = h->cfg;
    DeltaParams &D = h->dp;
    StackParams &S = h->skp;
    std::memset(&D, 0, sizeof(D));
    std::memset(&S, 0, sizeof(S));
    S.L = 1;
    // deltaFEA works on the first fea_ncepcoefs+1 elements of whatever vector it is given (src/fea/fea_delta.cc:23, 31);
    // -fea_trap reuses its first stage as a context window (src/io/opts.cc:694-704)
    const int fea_c = c.fea_ncepcoefs + 1;
    const bool chain = c.fea_delta && c.n_order > 0;
    const bool trap = chain && c.fea_trap;
    const bool cepstral = (h->fea_kind == FEA_DCTC || h->fea_kind == FEA_LPC);
    int n_order = (chain && !trap) ? c.n_order : 0;
    int blk = h->static_dim;
    if (h->fea_in) {
        h->in_dim = c.nfeacoefs;
        if (h->in_dim < 1) return fail(h, CTU_ERR_CONFIG, "IN: -nfeacoefs must be positive");
        if (chain && h->in_dim < fea_c) return fail(h, CTU_ERR_CONFIG, "IN: -nfeacoefs is smaller than fea_ncepcoefs+1, the columns the delta chain reads");
        h->gather = true;
        blk = chain ? fea_c : h->in_dim;
        S.fea_c = blk; S.rot = 0; S.src_stride = h->in_dim;
        h->static_dim = blk;
    } else if (chain) {
        if (h->fea_kind == FEA_LPA) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: deltas / stacking with -fea_kind lpa (the reference's delta chain and writer disagree on the vector layout)");
        if (h->fea_kind == FEA_TRAPDCT) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: deltas / stacking with trapdct (the reference never flushes the TRAP ring then, src/io/batch.cc:253: the last rows are lost)");
        if (cepstral && !c.fea_c0)
            return fail(h, CTU_ERR_UNSUPPORTED, trap ? "CTU: -fea_trap with -fea_c0 off (the reference writes past its output buffer, src/io/out.cc:184)"
                                                     : "CTU: deltas with -fea_c0 off (the reference writes uninitialised columns there, src/io/out.cc:189-201)");
        if (!cepstral && h->fb.nb < fea_c) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: deltas / stacking read fea_ncepcoefs+1 elements, more than the filter bank has bands");
        if (!cepstral || trap) {
            h->gather = true;
            blk = fea_c;
            S.fea_c = fea_c; S.rot = cepstral ? 1 : 0; S.src_stride = h->static_dim;
        } else if (h->compact_static && h->fea_kind == FEA_DCTC && !h->do_vad && !(h->nr_mode != NR_NONE && c.nr_when == 1)) {
            // MFCC + deltas: the cepstra go to a compact [rows x static_dim] matrix (whole rows, coalesced) and the delta kernel
            // takes its static block from there (the plain column gather above, no rotation: the block is in writer order
            // already) and writes c | delta | delta-delta as whole output rows.  In place, the filter-bank kernel wrote 52 of
            // every 156 bytes and the delta kernel 104, both as partial sectors: the delta kernel read 156 B per frame to
            // use 52 and ran at a third of the HBM rate (profiles/r02_ncu_mfcc_exten.txt).  Not with the VAD module (its
            // feature criterion reads the rows) nor on the fp64 band path.
            h->gather = true;
            S.fea_c = blk; S.rot = 0; S.src_stride = h->static_dim;
        }
    }
    if (trap) {
        if (c.d_win < 1) return fail(h, CTU_ERR_CONFIG, "FEA: Trap window size must be >= 3!");
        S.win = c.d_win; S.L = 2 * c.d_win + 1;
    }
    if (h->gather && h->do_vad && h->vad_cri == VCRI_CEPDIST_FEA)
        return fail(h, CTU_ERR_UNSUPPORTED, "CTU: the feature-vector VAD criterion together with stacking / deltas of spectral vectors");
    D.n_order = n_order;
    int wins[3] = {c.d_win, c.a_win, c.t_win};
    int halo = 0;
    for (int k = 0; k < n_order; k++) {
        if (wins[k] < 1) return fail(h, CTU_ERR_CONFIG, "FEA: Delta window size must be > 1!");
        D.win[k] = wins[k];
        double den = 0;
        for (int i = 1; i <= wins[k]; i++) den += i * i;
        D.inv_den[k] = (float)(1.0 / (2 * den));
        D.inv_den64[k] = 1.0 / (2 * den);
        halo += wins[k];
    }
    D.blk = blk;
    h->work_dim = (trap ? blk * S.L : blk * (n_order + 1)) + (c.fea_E ? 1 : 0);
    h->feature_dim = h->work_dim;
    if (h->fea_in) {
        // htkOUT::get_fea_size (src/io/out.cc:95-112) cuts one element for lpa, and for lpc / dctc without c0; the
        // writer then copies the first fea_size elements as they come (src/io/out.cc:177-179)
        if (h->fea_kind == FEA_LPA || (cepstral && !c.fea_c0)) h->feature_dim = h->work_dim - 1;
        if (h->feature_dim < 1) return fail(h, CTU_ERR_CONFIG, "OUT: empty feature vector");
    }
    if ((c.stat_cmvn || c.apply_cmvn) && h->work_dim != h->feature_dim)
        return fail(h, CTU_ERR_UNSUPPORTED, "CTU: CMVN on feature files whose last column the writer cuts (lpa, lpc / dctc without c0)");
    D.stride = h->work_dim;
    S.dst_stride = h->work_dim;
    D.span_max = DELTA_ROWS + 2 * halo;
    // -fea_Z_exp normalises the first fea_ncepcoefs+1 elements of the finished vector (src/fea/post_impl.cc:203-209): the
    // whole static block of cepstral rows (c0 included, wherever the writer puts it), the leading columns otherwise
    h->cms_cols = h->gather ? ((h->fea_in && !chain) ? 0 : fea_c) : h->static_dim;
    if (h->fea_kind == FEA_TRAPDCT) {
        TrapParams &T = h->tp;
        std::memset(&T, 0, sizeof(T));
        const int L = c.fea_trapdct_traplen, n = c.fea_trapdct_ndct;
        if (L % 2 == 0) return fail(h, CTU_ERR_CONFIG, "FEA: TRAP length must be odd!");
        if (n >= L) return fail(h, CTU_ERR_CONFIG, "FEA: Number of DCT coeffs must be less than TRAP length (c0 is not output)!");
        if (L > TRAP_MAXL || n > TRAP_MAXN || n < 1) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: TRAP-DCT supports traplen <= 127, ndct <= 16");
        T.L = L; T.ndct = n; T.nb = h->fb.nb; T.h = (L + 1) / 2;
        const double PI = 3.14159265358979323846264338327950288;
        for (int k = 1; k <= n; k++) {
            std::vector<double> row(L);
            double sum = 0;
            for (int j = 0; j < L; j++) {
                double hamm = 0.54 - (1 - 0.54) * cos(2 * 3.14159265359 * j / (L - 1.));
                row[j] = 2.0 * hamm * cos(PI * (j + 0.5) * k / L);
                sum += row[j];
            }
            for (int j = 0; j < L; j++) T.m[j * n + (k - 1)] = (float)(row[j] - sum / L);
        }
        h->feature_dim = h->work_dim = h->fb.nb * n;
        T.out_stride = h->feature_dim;
    }
    if (c.fea_E) {
        // which stage's E the writer points at: BATCH::init_out (src/io/batch.cc:98-118)
        if (h->fea_kind == FEA_TRAPDCT) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: -fea_E with trapdct (the reference never sets that energy)");
        if (!std::strcmp(c.format_out, "pfile")) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: -fea_E with pfile output (the reference declares the pfile without the energy column, src/io/out.cc:252)");
        const bool lp = (h->fea_kind == FEA_LPA || h->fea_kind == FEA_LPC);
        // with the VAD module init_out never looks at fea_rawenergy (src/io/batch.cc:74-96): lpc/lpa still get log R0,
        // dctc after the FB gets IN's (raw) energy, the other stages leave their E unset
        if (c.fea_rawenergy && h->do_vad && !lp && !(h->fea_kind == FEA_DCTC && c.nr_when == 1))
            return fail(h, CTU_ERR_UNSUPPORTED, "CTU: -fea_rawenergy with the VAD module: the reference writes an energy that was never computed (src/io/batch.cc:74-96)");
        if (c.fea_rawenergy && !(h->do_vad && lp)) h->energy_mode = EN_RAW;
        else if (h->fea_kind == FEA_DCTC) h->energy_mode = (c.nr_when == 1) ? EN_IN : EN_NR;
        else if (h->fea_kind == FEA_LPA || h->fea_kind == FEA_LPC) h->energy_mode = EN_LPC;
        else h->energy_mode = EN_BANDS;
        // the row is written `latency` frames after its energy was current (deltas, VAD majority filter)
        int lat = trap ? c.d_win : 0;
        for (int k = 0; k < n_order; k++) lat += wins[k];
        if (h->do_vad) lat += (c.vad_filter_order - 1) / 2;
        h->energy_latency = lat;
    }
    return CTU_OK;
}

// FFT size other than the specialised 512 points (the fp64 Burg / synthesis kernels then take their general form)
static bool c_wfft_is_general(const ctu_handle *h) { return h->cfg.wfft != NFFT; }
// 8 kHz-sized frames take the specialised 256-point front end (ctu_frames256.cuh) and the general kernel from the spectrum on
static bool fast256(const ctu_handle *h) {
    return h->generic && !h->fea_in && h->cfg.wfft == 256 && h->cfg.wshift <= h->cfg.window && h->cfg.dither == 0.0 && !h->cfg.remove_dc1 && h->front256;
}

static int resolve_modes(ctu_handle *h) {
    const ctu_config &c = h->cfg;
    std::string fo(c.format_out), kind(c.fea_kind), nr(c.nr_mode), vm(c.vadmode);
    h->signal_out = (fo == "raw" || fo == "wave");
    if (!h->signal_out && fo != "htk" && fo != "pfile" && fo != "ark") return fail(h, CTU_ERR_CONFIG, "OUT: Unknown output file format!");
    if (h->signal_out) h->fea_kind = FEA_NONE;
    else if (kind == "spec") h->fea_kind = FEA_SPEC;
    else if (kind == "logspec") h->fea_kind = FEA_LOGSPEC;
    else if (kind == "dctc") h->fea_kind = FEA_DCTC;
    else if (kind == "lpa") h->fea_kind = FEA_LPA;
    else if (kind == "lpc") h->fea_kind = FEA_LPC;
    else if (kind == "trapdct") h->fea_kind = FEA_TRAPDCT;
    else if (kind == "td-iir-mfcc") h->fea_kind = FEA_TDIIR;
    else return fail(h, CTU_ERR_CONFIG, "FEA: Unknown feature kind!");
    if (kind == "td-iir-mfcc") {
        // BATCH::BATCH, src/io/batch.cc:28, 61-62: no NR, no FB, no FEA, no deltaFEA, no POST, no VAD object -- IN's 13-element
        // vector goes straight to the writer (process_frame :221-222).  What the reference does NOT survive is refused:
        if (h->signal_out) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: td-iir-mfcc with waveform output (the reference hands its 13 cepstra to the synthesis)");
        if (c.fea_in) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: td-iir-mfcc with feature-file input");
        if (c.fea_ncepcoefs != 12)
            return fail(h, CTU_ERR_UNSUPPORTED, "CTU: td-iir-mfcc needs -fea_ncepcoefs 12 (the reference writes 13 coefficients into a vector of fea_ncepcoefs+1, src/io/in.cc:168-170, 328)");
        if (!c.fea_c0) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: td-iir-mfcc with -fea_c0 off (the writer's last column is never set, src/io/out.cc:95-112, 189-200)");
        if (c.fea_E) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: td-iir-mfcc with -fea_E (no energy is computed on this branch, src/io/in.cc:317-340)");
        if (c.fea_delta && c.n_order > 0)
            return fail(h, CTU_ERR_UNSUPPORTED, "CTU: td-iir-mfcc with deltas / stacking (the reference calls a deltaFEA it never built, src/io/batch.cc:217-218)");
        if (c.stat_cmvn || c.apply_cmvn) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: td-iir-mfcc with CMVN (no POST object exists on this branch)");
        if (std::string(c.vad_apply_mode) != "none" || std::string(c.vad_out_mode) != "none")
            return fail(h, CTU_ERR_UNSUPPORTED, "CTU: td-iir-mfcc with the VAD module (the reference dereferences a VAD it never built, src/io/batch.cc:230-232)");
        if (c.window > 4096) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: td-iir-mfcc with a window longer than 4096 samples");
        // noise reduction, dither, DC removal, pre-emphasis and CMS never run on this branch (src/io/in.cc:430-436): ignored
        h->nr_mode = NR_NONE; h->vad_src = VADSRC_NONE; h->do_vad = false; h->fea_in = false;
        h->nbins = c.wfftby2; h->spitch = h->nbins;
        return CTU_OK;
    }
    if (nr == "none") h->nr_mode = NR_NONE;
    else if (nr == "exten") h->nr_mode = NR_EXTEN;
    else if (nr == "hwss") h->nr_mode = NR_HWSS;
    else if (nr == "fwss") h->nr_mode = NR_FWSS;
    else if (nr == "2fwss") h->nr_mode = NR_2FWSS;
    else return fail(h, CTU_ERR_CONFIG, "NR: Unknown noise reduction mode!");
    h->vad_src = vm == "burg" ? VADSRC_BURG : vm == "file" ? VADSRC_FILE : VADSRC_NONE;
    if (h->nr_mode >= NR_HWSS) {
        if (h->vad_src == VADSRC_NONE) return fail(h, CTU_ERR_CONFIG, "NR: Please specify Voice Activity Detector!");
        if (h->vad_src == VADSRC_BURG && c.nr_when == 1 && !h->signal_out)
            return fail(h, CTU_ERR_CONFIG, "NR: Cannot use Burg detector after filter bank!");
    }
    h->fea_in = c.fea_in != 0;
    if (h->fea_in) {
        // BATCH::BATCH, src/io/batch.cc:55-60: no IN spectrum, no NR, no FB, no FEA -- only deltaFEA / POST / OUT
        if (h->signal_out) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: feature-file input with waveform output");
        if (c.fea_E) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: -fea_E with feature-file input (no energy is ever computed; the reference reads past its vector, src/io/out.cc:177-179)");
        if (h->fea_kind == FEA_DCTC && !c.fea_rawenergy)
            return fail(h, CTU_ERR_UNSUPPORTED, "CTU: feature-file input with -fea_kind dctc needs -fea_rawenergy on (the reference dereferences a null NR otherwise, src/io/batch.cc:108)");
        if (h->fea_kind == FEA_TRAPDCT) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: feature-file input with -fea_kind trapdct");
        h->nr_mode = NR_NONE; h->vad_src = VADSRC_NONE;
    }
    std::string am(c.vad_apply_mode), om(c.vad_out_mode);
    h->do_vad = (am != "none" || om != "none");
    if (h->do_vad && h->fea_in) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: the VAD module with feature-file input (there is no spectrum to decide on)");
    h->vad_drop = (am == "drop");
    if (h->do_vad && h->signal_out)
        return fail(h, CTU_ERR_UNSUPPORTED, "CTU: the VAD module with waveform output (the reference dereferences an uninitialised pointer there, src/io/batch.cc:63-65,230-241)");
    if (h->do_vad) {
        std::string cm(c.vad_cri_mode), tm(c.vad_thr_mode), dm(c.vad_cepdist_mode);
        if (cm == "energy") h->vad_cri = VCRI_ENERGY;
        else if (cm == "cepdist") {
            if (dm == "lpc") {
                h->vad_cri = VCRI_CEPDIST_LPC;
                if (!c.phase_needed) return fail(h, CTU_ERR_CONFIG, "VADcri_cepdist: cannot perform iFFT!");
            } else if (dm == "fea" || dm == "in") h->vad_cri = VCRI_CEPDIST_FEA;
            else return fail(h, CTU_ERR_CONFIG, "VADcri_cepdist: unknown vad_cepdist_mode!");
        } else return fail(h, CTU_ERR_CONFIG, "VAD: unknown vad_cri_mode!");
        if (tm == "absolute") h->vad_thr = VTHR_ABSOLUTE;
        else if (tm == "perc") h->vad_thr = VTHR_PERC;
        else if (tm == "adapt") h->vad_thr = VTHR_ADAPT;
        else if (tm == "dyn") h->vad_thr = VTHR_DYN;
        else return fail(h, CTU_ERR_CONFIG, "VAD: unknown vad_thr_mode!");
        if (c.vad_filter_order < 1 || c.vad_filter_order % 2 == 0)
            return fail(h, CTU_ERR_CONFIG, "medianFilter: filter order must be positive, odd number!");
    }
    // post-processing (SURVEY 8f.2)
    if (c.stat_cmvn || c.apply_cmvn) {
        // the host drives the passes (ctu_plan_colsums / ctu_plan_normalise); what the device half supports:
        if (h->signal_out || h->do_vad || h->fea_kind == FEA_LPA || h->fea_kind == FEA_TRAPDCT ||
            ((h->fea_kind == FEA_DCTC || h->fea_kind == FEA_LPC) && !c.fea_c0))
            return fail(h, CTU_ERR_UNSUPPORTED, "CTU: CMVN is built for dctc / lpc (with c0), spec and logspec features without the VAD module");
        if (c.cms_exp_coef > 0 || c.fea_Z_block > 0)
            return fail(h, CTU_ERR_CONFIG, "OPTS: CMN or CMVN can not be set together with CMS option (exp or block CMS normalisations)!");
    }
    if (c.fea_Z_block > 0)
        return fail(h, CTU_ERR_UNSUPPORTED, "CTU: -fea_Z_block: the reference dies with SIGSEGV in this mode (ring of row pointers allocated with sizeof(float), src/fea/post_impl.cc:179); nothing to match");
    if (c.cms_exp_coef > 0) {
        const bool chain = c.fea_delta && c.n_order > 0;
        if (h->signal_out || (h->fea_kind != FEA_DCTC && h->fea_kind != FEA_LPC && !chain && !h->fea_in))
            return fail(h, CTU_ERR_UNSUPPORTED, "CTU: -fea_Z_exp is built for cepstral features (dctc, lpc) and for delta / stacking chains");
        if (h->do_vad) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: -fea_Z_exp together with the VAD module");
    }
    // -remove_dc1 needs per-frame ring offsets: only the general kernels apply them
    // dither (src/io/in.cc:452-455): glibc's rand() stream restated on the host, one value per loaded sample in list
    // order; applied by the general kernel
    h->generic = !h->fea_in && ((c.wfft != NFFT) || c.remove_dc1 || c.dither != 0.0);
    if (h->fea_in) { h->nbins = c.wfftby2; h->spitch = h->nbins; return CTU_OK; }
    if (c.dither != 0.0 && (c.remove_dc1 || (c.fea_E && c.fea_rawenergy)))
        return fail(h, CTU_ERR_UNSUPPORTED, "CTU: -dither together with -remove_dc1 or -fea_rawenergy");
    h->nbins = c.wfftby2;
    h->spitch = h->generic ? h->nbins : SPITCH;      // 512-point path: rows padded to 260 floats (16-byte aligned)
    if (c.remove_dc1 && c.window / c.wshift + 1 > ANY_DC1_MAX) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: -remove_dc1 with a window longer than 17 shifts");
    if (h->generic) {
        // other sampling rates / window lengths, -remove_dc1, -dither: the general (slower) frame kernel; synthesis, the Burg
        // detector and the fp64 path have general siblings too (ctu_any64.cuh), which apply the ring offsets of -remove_dc1
        // but not the noise of -dither
        if (c.wfft < 64 || c.wfft > ANY_MAX_NFFT) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: FFT sizes from 64 to 2048 points are built (window of 33..2048 samples)");
        if (h->signal_out && c.dither != 0.0) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: waveform output together with -dither");
        if ((h->vad_src == VADSRC_BURG || (h->do_vad && h->vad_cri == VCRI_CEPDIST_LPC)) && c.dither != 0.0)
            return fail(h, CTU_ERR_UNSUPPORTED, "CTU: the Burg detector together with -dither");
    }
    return CTU_OK;
}

// rawIN::loadf_filters (src/io/in.cc:242-262): one filter per line, ten TAB-separated numbers parsed with atof; the
// reference reads lines until the file ends (past its 24 rows when there are more) and hands strtok's NULL to atof when a
// line is short -- both refused here.  Host tables of the td-iir-mfcc path (ctu_tdiir.cuh).
static int build_tdiir(ctu_handle *h, std::vector<double> &coefs, std::vector<double> &win, std::vector<double> &dct) {
    const ctu_config &c = h->cfg;
    FILE *f = std::fopen(c.filters, "r");
    if (!f) return fail(h, CTU_ERR_INPUT, std::string("IN: Cannot open the filter coefficient file '") + c.filters + "' (-filters)");
    coefs.assign(TDIIR_BANDS * 10, 0.0);
    char line[1000];
    int nf = 0;
    while (nf < TDIIR_BANDS && std::fgets(line, sizeof(line), f)) {
        char *save = nullptr;
        char *tok = strtok_r(line, "\t", &save);
        for (int i = 0; i < 10; i++) {
            if (!tok) { std::fclose(f); return fail(h, CTU_ERR_INPUT, "IN: a line of the filter coefficient file has fewer than 10 TAB-separated numbers"); }
            coefs[nf * 10 + i] = std::atof(tok);
            tok = strtok_r(nullptr, "\t", &save);
        }
        nf++;
    }
    std::fclose(f);
    if (nf < TDIIR_BANDS) return fail(h, CTU_ERR_INPUT, "IN: the filter coefficient file holds fewer than 24 filters");
    const int w = c.window, s = c.wshift;
    win.resize(w);
    const double pi = 2. * asin(1.);
    for (int j = 0; j < w; j++) win[j] = 0.54 - (1 - 0.54) * cos(2 * pi * j / (w - 1.));       // src/io/in.cc:139-144
    // wdct[i] = cos(pi i / 48), used at index (2k-1) i % 96 (src/io/in.cc:236-237, 330-333)
    dct.resize(TDIIR_NCEP * TDIIR_BANDS);
    for (int i = 0; i < TDIIR_NCEP; i++)
        for (int k = 1; k <= TDIIR_BANDS; k++)
            dct[i * TDIIR_BANDS + (k - 1)] = cos(3.14159265358979 * (double)(((2 * k - 1) * i) % (4 * TDIIR_BANDS)) / (2 * TDIIR_BANDS));
    int a = w, b = s;
    while (b) { const int t = a % b; a = b; b = t; }
    TdiirParams &P = h->tdp;
    P.window = w; P.wshift = s; P.seg = a; P.spf = w / a; P.sps = s / a;
    // samples staged per step: the largest length up to TDIIR_CHUNK that is a multiple or a divisor of the segment
    int L = TDIIR_CHUNK;
    while (L > 1 && (L % a) != 0 && (a % L) != 0) L--;
    P.chunk = L; P.run = std::min(a, L);
    P.weight = (double)c.weight_of_td_iir_mfcc_bank;
    h->static_dim = h->feature_dim = h->work_dim = TDIIR_NCEP;
    return CTU_OK;
}

int ctu_create(const ctu_config *cfg, int device, ctu_handle **out) {
    if (!cfg || !out) { g_create_err = "CTU: null argument"; return CTU_ERR_CONFIG; }
    *out = nullptr;
    if (cfg->abi_version != CTU_ABI_VERSION) { g_create_err = "CTU: ABI version mismatch"; return CTU_ERR_CONFIG; }
    ctu_handle *h = new ctu_handle;
    h->cfg = *cfg;
    h->device = device;
    if (const char *e = getenv("CTU_FUSE_NR")) h->fuse_nr = atoi(e);
    if (const char *e = getenv("CTU_FRONT256")) h->front256 = atoi(e);
    if (const char *e = getenv("CTU_COMPACT_STATIC")) h->compact_static = atoi(e);
    if (const char *e = getenv("CTU_CHUNK_MB")) h->chunk_mb = std::max(1, atoi(e));
    auto bail = [&](int st) { g_create_err = h->err; delete h; return st; };
    int st = ctu_config_finalize(&h->cfg);
    if (st) { h->err = ctu_config_error(); return bail(st); }
    if ((st = resolve_modes(h))) return bail(st);
    if (h->fea_kind == FEA_TDIIR) {
        std::vector<double> coefs, win, dct;
        std::memset(&h->fp, 0, sizeof(h->fp)); std::memset(&h->dp, 0, sizeof(h->dp)); std::memset(&h->skp, 0, sizeof(h->skp));
        h->skp.L = 1;                                // no delta chain, no stacking on this branch
        if ((st = build_tdiir(h, coefs, win, dct))) return bail(st);
        int ndev = 0;
        cudaError_t ce = cudaGetDeviceCount(&ndev);
        if (ce != cudaSuccess || ndev == 0 || device >= ndev) {
            h->err = std::string("CUDA: no usable device (") + (ce != cudaSuccess ? cudaGetErrorString(ce) : "device index out of range") +
                     "); libctucopy_b200 has no CPU fallback";
            return bail(CTU_ERR_CUDA);
        }
        if (cudaSetDevice(device) != cudaSuccess) { h->err = "CUDA: cudaSetDevice failed"; return bail(CTU_ERR_CUDA); }
        cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device);
        if ((st = upload(h, &h->d_td_coefs, coefs)) || (st = upload(h, &h->d_td_win, win)) || (st = upload(h, &h->d_td_dct, dct))) return bail(st);
        h->tdp.coefs = h->d_td_coefs; h->tdp.win = h->d_td_win; h->tdp.dct = h->d_td_dct;
        for (int i = 0; i < 3; i++)
            if (cudaStreamCreateWithFlags(&h->streams[i], cudaStreamNonBlocking) != cudaSuccess) { h->err = "CUDA: stream creation failed"; return bail(CTU_ERR_CUDA); }
        *out = h;
        return CTU_OK;
    }
    if (!h->signal_out && !h->fea_in) {
        std::string e = ctu_design_fb(h->cfg, h->fb);
        if (!e.empty()) { h->err = e; return bail(CTU_ERR_CONFIG); }
    }
    if ((st = build_frame_params(h))) return bail(st);
    if ((st = build_delta_trap_params(h))) return bail(st);
    if (!h->fea_in && (st = build_nr_params(h->cfg, h->nr_mode, h->vad_src, h->signal_out, h->fb.nb, h->nrp, h->sp, h->bp, h->vp, h->err))) return bail(st);
    h->nrp.carry_xform = (h->cfg.nr_when == 1 && !h->signal_out) ? (h->fea_kind == FEA_DCTC ? 1 : ((h->fea_kind == FEA_LPA || h->fea_kind == FEA_LPC) && !h->fb.inld) ? 2 : 0) : 0;
    h->vp.cri = h->vad_cri; h->vp.thr = h->vad_thr; h->vp.drop = h->vad_drop;
    h->vp.has_E = h->energy_mode ? 1 : 0;
    h->vp.nbins = h->nbins; h->vp.spitch = h->spitch; h->bp.spitch = h->spitch;
    // the reference's vector is in internal order (c0 first, a0 first); rows here are in writer order
    if (h->fea_kind == FEA_DCTC || h->fea_kind == FEA_LPC) h->vp.fea_skip = h->cfg.fea_c0 ? h->static_dim - 1 : -1;
    else if (h->fea_kind == FEA_LPA) h->vp.fea_skip = -1;
    else h->vp.fea_skip = 0;
    // the device: fail loudly, there is no CPU path
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0 || device >= ndev) {
        h->err = std::string("CUDA: no usable device (") + (ce != cudaSuccess ? cudaGetErrorString(ce) : "device index out of range") +
                 "); libctucopy_b200 has no CPU fallback";
        return bail(CTU_ERR_CUDA);
    }
    if (cudaSetDevice(device) != cudaSuccess) { h->err = "CUDA: cudaSetDevice failed"; return bail(CTU_ERR_CUDA); }
    cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device);
    if (!h->fea_in && (st = build_fft_tables(h))) return bail(st);
    if (h->nr_mode != NR_NONE && h->cfg.nr_when == 1 && !h->signal_out) h->precise = true;   // subtraction on band values
    // VAD criterion = distance between feature vectors, fed to threshold state machines whose
    // decisions must match the reference bit for bit: features in fp64 like the reference's
    if (h->do_vad && h->vad_cri == VCRI_CEPDIST_FEA) h->precise = true;
    // the fp64 general kernels (ctu_any64.cuh) also take the 512-point frames whose window length is odd (e.g. 32 ms at
    // 11.025 kHz = 353 samples): the specialised synthesis / Burg kernels pair samples two by two.  They take -remove_dc1
    // at every size too: k_synth_c and k_burg read X from k_frames2, which applies no ring offsets, and k_frames_any
    // (the spectrum under -remove_dc1) does not store X.  The spectrum that feeds the noise reduction and the features
    // stays on k_frames_any.
    const bool any64 = c_wfft_is_general(h) || (h->cfg.window & 1) || h->cfg.remove_dc1;
    if (h->generic || any64) {
        if (h->generic && h->precise && h->cfg.dither != 0.0) {
            h->err = "CTU: -dither together with a configuration that needs the fp64 path (band-domain noise reduction, LPC without the cube-root law, feature-vector VAD)";
            return bail(CTU_ERR_UNSUPPORTED);
        }
        const int N = h->cfg.wfft, M = N / 2;
        const double PI = 3.14159265358979323846264338327950288;
        const bool burg = h->vad_src == VADSRC_BURG || (h->do_vad && h->vad_cri == VCRI_CEPDIST_LPC);
        if (any64 && (h->signal_out || burg || h->precise)) {
            std::vector<double2> twd(std::max(1, M / 2)), tsd(M + 1);
            for (int k = 0; k < M / 2; k++) twd[k] = make_double2(cos(-2 * PI * k / M), sin(-2 * PI * k / M));
            for (int k = 0; k <= M; k++) { const double th = 2 * PI * k / N; tsd[k] = make_double2(-sin(th) / 2, -cos(th) / 2); }
            if ((st = upload(h, &h->d_any_tw64, twd)) || (st = upload(h, &h->d_any_ts64, tsd))) return bail(st);
            int lg = 0;
            while ((1 << lg) < M) lg++;
            h->bp.nfft = N; h->bp.log2m = lg; h->bp.any_tw = h->d_any_tw64; h->bp.any_ts = h->d_any_ts64;
        }
        if (h->generic && N == 256) {
            std::vector<float2> t128(128);
            for (int k1 = 0; k1 < 16; k1++)
                for (int g = 0; g < 8; g++) t128[k1 * 8 + g] = make_float2((float)cos(-2 * PI * (g * k1) / 128.0), (float)sin(-2 * PI * (g * k1) / 128.0));
            if ((st = upload(h, &h->d_tw128, t128))) return bail(st);
        }
        if (h->generic) {
            std::vector<float2> tw(std::max(1, M / 2)), ts(M + 1);
            for (int k = 0; k < M / 2; k++) tw[k] = make_float2((float)cos(-2 * PI * k / M), (float)sin(-2 * PI * k / M));
            for (int k = 0; k <= M; k++) { const double th = 2 * PI * k / N; ts[k] = make_float2((float)(-sin(th) / 2), (float)(-cos(th) / 2)); }
            if ((st = upload(h, &h->d_any_tw, tw)) || (st = upload(h, &h->d_any_ts, ts)) || (st = upload(h, &h->d_any_fbw, h->fbw_all)) ||
                (st = upload(h, &h->d_any_bands, h->bands_all))) return bail(st);
        }
    }
    if (h->precise) {
        if ((st = upload(h, &h->d_w64, h->w64)) || (st = upload(h, &h->d_m264, h->m264)) || (st = upload(h, &h->d_lift64, h->lift64))) return bail(st);
    }
    if (!h->generic && !h->fea_in && !h->signal_out && !h->precise && h->fea_kind != FEA_NONE) {
        // k_bank's copy of the filter bank: bands aligned to groups of four bins, second-stage matrix, geometry
        std::vector<int4> bands; std::vector<float> w;
        bank_pack(h->fp, bands, w);
        std::vector<float4> w4(w.size() / 4);
        for (size_t i = 0; i < w4.size(); i++) w4[i] = make_float4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
        std::vector<float> m2((size_t)std::max(1, h->fp.nrows * h->fp.nbp));
        if (h->fea_kind == FEA_DCTC) for (int i = 0; i < h->fp.nrows * h->fp.nbp; i++) m2[i] = h->fp.m2[i];
        if ((st = upload(h, &h->bank.d_bands, bands)) || (st = upload(h, &h->bank.d_w4, w4)) || (st = upload(h, &h->bank.d_m2, m2))) return bail(st);
        h->bank.wtot4 = (int)w4.size();
        h->bank.ypitch = ((h->fp.nbp + 31) / 32) * 32 + 4;
        BankParams &B = h->bkp;
        B.nb = h->fp.nb; B.nbp = h->fp.nbp; B.ypitch = h->bank.ypitch;
        B.inld = h->fp.inld; B.inld_scale = h->fp.inld_scale; B.lin_scale = h->fp.lin_scale; B.log_offset = h->fp.log_offset;
        B.nrows = (h->fea_kind == FEA_DCTC) ? h->fp.nrows : 0;
        B.take_sqrt = h->fp.take_sqrt;
        B.wtot4 = h->bank.wtot4; B.bands = h->bank.d_bands; B.w4 = h->bank.d_w4; B.m2 = h->bank.d_m2;
        B.nr = h->nrp;
    }
    for (int i = 0; i < 3; i++)
        if (cudaStreamCreateWithFlags(&h->streams[i], cudaStreamNonBlocking) != cudaSuccess) { h->err = "CUDA: stream creation failed"; return bail(CTU_ERR_CUDA); }
    *out = h;
    return CTU_OK;
}

void ctu_destroy(ctu_handle *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaFree(h->d_tw256); cudaFree(h->d_twsplit); cudaFree(h->d_twinv); cudaFree(h->d_win);
    cudaFree(h->d_w64); cudaFree(h->d_m264); cudaFree(h->d_lift64);
    cudaFree(h->d_tw256d); cudaFree(h->d_twsplitd); cudaFree(h->d_twinvd); cudaFree(h->d_wind); cudaFree(h->d_hann);
    cudaFree(h->d_any_tw64); cudaFree(h->d_any_ts64);
    cudaFree(h->d_g711[0]); cudaFree(h->d_g711[1]);
    cudaFree(h->d_any_tw); cudaFree(h->d_any_ts); cudaFree(h->d_any_fbw); cudaFree(h->d_any_bands);
    cudaFree(h->bank.d_bands); cudaFree(h->bank.d_w4); cudaFree(h->bank.d_m2);
    cudaFree(h->d_td_coefs); cudaFree(h->d_td_win); cudaFree(h->d_td_dct);
    cudaFree(h->d_carry); cudaFree(h->d_carry64); cudaFree(h->d_tw128);
    if (h->carry_ev) cudaEventDestroy(h->carry_ev);
    for (auto &b : h->pool) cudaFree(b.p);
    for (int i = 0; i < 3; i++) if (h->streams[i]) cudaStreamDestroy(h->streams[i]);
    h->lc.clear();
    delete h;
}

// ------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------
template <class T> static int dev_alloc(ctu_handle *h, ctu_plan *p, T **ptr, size_t n) {
    const size_t bytes = (std::max<size_t>(n, 1) * sizeof(T) + 255) & ~size_t(255);
    p->workspace_bytes += (int64_t)bytes;
    int best = -1;
    for (int i = 0; i < (int)h->pool.size(); i++) {
        const auto &b = h->pool[i];
        if (!b.used && b.bytes >= bytes && b.bytes <= 2 * bytes + 4096 && (best < 0 || b.bytes < h->pool[best].bytes)) best = i;
    }
    if (best >= 0) {
        h->pool[best].used = true;
        *ptr = (T *)h->pool[best].p;
    } else {
        void *q = nullptr;
        cudaError_t e = cudaMalloc(&q, bytes);
        if (e != cudaSuccess) {
            // out of memory: give the cached blocks back and try once more
            for (auto &b : h->pool) if (!b.used) { cudaFree(b.p); b.p = nullptr; }
            h->pool.erase(std::remove_if(h->pool.begin(), h->pool.end(), [](const ctu_handle::PoolBlock &b) { return b.p == nullptr; }), h->pool.end());
            cudaGetLastError();
            CK(cudaMalloc(&q, bytes));
        }
        h->pool.push_back({q, bytes, true});
        *ptr = (T *)q;
    }
    p->blocks.push_back((void *)*ptr);
    return CTU_OK;
}

int ctu_plan_create(ctu_handle *h, const int64_t *off, int32_t n, ctu_plan **out) {
    if (!h || !off || !out || n < 0) return CTU_ERR_CONFIG;
    *out = nullptr;
    CK(cudaSetDevice(h->device));
    ctu_plan *p = new ctu_plan;
    p->h = h; p->n_utts = n;
    p->offsets.assign(off, off + n + 1);
    p->nframes.resize(n); p->row_off.resize(n + 1); p->osamp_off.resize(n + 1);
    p->tile32_off.resize(n + 1); p->tile64_off.resize(n + 1); p->tileS_off.resize(n + 1); p->tileF_off.resize(n + 1);
    p->syn_tile = std::max(1, SYN_FRAMES - h->sp.hh);
    if (h->signal_out && !h->bp.nfft && h->sp.hh >= SYN_FRAMES) { delete p; return fail(h, CTU_ERR_UNSUPPORTED, "CTU: window / shift ratio too large for synthesis"); }
    p->rows_per_utt.assign(n, 0);
    const int w = h->cfg.window, s = h->cfg.wshift;
    int64_t rows = 0, osamp = 0, t32 = 0, t64 = 0, tS = 0, tF = 0;
    for (int u = 0; u < n; u++) {
        int64_t N = off[u + 1] - off[u];
        if (!h->fea_in && N < w - s) { delete p; return fail(h, CTU_ERR_INPUT, "IO: Signal shorter than one frame!"); }
        int64_t T = h->fea_in ? N : (N - (w - s)) / s;                 // feature input: one row = one frame
        if (T > 0x7fffffff) { delete p; return fail(h, CTU_ERR_INPUT, "CTU: utterance too long"); }
        p->nframes[u] = (int)T;
        p->row_off[u] = rows; p->osamp_off[u] = osamp; p->tile32_off[u] = t32; p->tile64_off[u] = t64; p->tileS_off[u] = tS; p->tileF_off[u] = tF;
        tF += (T + F2_TILE - 1) / F2_TILE;
        tS += (T + p->syn_tile - 1) / p->syn_tile;
        rows += T; osamp += T * s + (w - s);
        t32 += (T + TILE_F - 1) / TILE_F; t64 += (T + DELTA_ROWS - 1) / DELTA_ROWS;
        p->rows_per_utt[u] = T;
        // the delta / TRAP closed forms need win+2 rows; shorter files take the reference's
        // start-up path whose output depends on never-written ring memory
        if (h->dp.n_order > 0) {
            int mw = 0;
            for (int k = 0; k < h->dp.n_order; k++) mw = std::max(mw, h->dp.win[k]);
            if (T < mw + 2) { delete p; return fail(h, CTU_ERR_UNSUPPORTED, "CTU: utterance shorter than delta window + 2 frames"); }
        }
        if (h->skp.L > 1 && T < h->skp.win + 2) { delete p; return fail(h, CTU_ERR_UNSUPPORTED, "CTU: utterance shorter than half the stacking window + 2 frames"); }
    }
    if (h->cfg.dither != 0.0 && !h->fea_in) {
        p->rand_base = h->rand_pos;
        h->rand_pos += (uint64_t)rows * (uint64_t)s + (uint64_t)n * (uint64_t)(w - s);     // one rand() per LOADED sample
    }
    p->row_off[n] = rows; p->osamp_off[n] = osamp; p->tile32_off[n] = t32; p->tile64_off[n] = t64; p->tileS_off[n] = tS; p->tileF_off[n] = tF;
    p->total_frames = rows; p->total_osamp = osamp; p->total_samples = off[n] - off[0];
    int st = 0;
    auto up64 = [&](int64_t **d, const std::vector<int64_t> &v) -> int {
        if ((st = dev_alloc(h, p, d, v.size()))) return st;
        CK(cudaMemcpy(*d, v.data(), v.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
        return CTU_OK;
    };
    std::vector<int64_t> pcm_off(p->offsets.begin(), p->offsets.end());   // same indexing as the caller's buffer
    if ((st = up64(&p->d_pcm_off, pcm_off)) || (st = up64(&p->d_row_off, p->row_off)) || (st = up64(&p->d_osamp_off, p->osamp_off)) ||
        (st = up64(&p->d_t32_off, p->tile32_off)) || (st = up64(&p->d_t64_off, p->tile64_off))) { ctu_plan_destroy(p); return st; }
    if ((st = dev_alloc(h, p, &p->d_nframes, n))) { ctu_plan_destroy(p); return st; }
#define CKP(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            h->err = std::string("CUDA: ") + cudaGetErrorString(e_) + " at " #call;                \
            ctu_plan_destroy(p);                                                                   \
            return CTU_ERR_CUDA;                                                                   \
        }                                                                                          \
    } while (0)
    if (n) CKP(cudaMemcpy(p->d_nframes, p->nframes.data(), n * sizeof(int), cudaMemcpyHostToDevice));
    if ((st = dev_alloc(h, p, &p->d_tiles32, t32)) || (st = dev_alloc(h, p, &p->d_tiles64, t64))) { ctu_plan_destroy(p); return st; }
    if ((st = up64(&p->d_tF_off, p->tileF_off)) || (st = dev_alloc(h, p, &p->d_tilesF, tF))) { ctu_plan_destroy(p); return st; }
    if (h->signal_out && ((st = up64(&p->d_tS_off, p->tileS_off)) || (st = dev_alloc(h, p, &p->d_tilesS, tS)))) { ctu_plan_destroy(p); return st; }
    if (n) {
        k_build_tiles<<<(n + 127) / 128, 128>>>(p->d_nframes, p->d_t32_off, n, TILE_F, p->d_tiles32);
        k_build_tiles<<<(n + 127) / 128, 128>>>(p->d_nframes, p->d_t64_off, n, DELTA_ROWS, p->d_tiles64);
        k_build_tiles<<<(n + 127) / 128, 128>>>(p->d_nframes, p->d_tF_off, n, F2_TILE, p->d_tilesF);
        if (h->signal_out) k_build_tiles<<<(n + 127) / 128, 128>>>(p->d_nframes, p->d_tS_off, n, p->syn_tile, p->d_tilesS);
        h->lc.launches += h->signal_out ? 4 : 3;
        CKP(cudaGetLastError());
    }
    // the tables above came from pageable memory and the tile lists from the legacy stream; everything that consumes them
    // runs on non-blocking streams, which do not order against either
    CKP(cudaDeviceSynchronize());
#undef CKP
    // workspaces by configuration
    if (h->gather && !h->fea_in && (st = dev_alloc(h, p, &p->d_static, (size_t)rows * h->static_dim))) { ctu_plan_destroy(p); return st; }
    if (h->work_dim != h->feature_dim && (st = dev_alloc(h, p, &p->d_work, (size_t)rows * h->work_dim))) { ctu_plan_destroy(p); return st; }
    if (h->fea_in) { *out = p; return CTU_OK; }
    if (h->fea_kind == FEA_TDIIR) {
        const size_t nseg = (size_t)(rows * h->tdp.sps + (int64_t)n * (h->tdp.spf - h->tdp.sps));
        if ((st = dev_alloc(h, p, &p->d_tdseg, nseg * TDIIR_BANDS + 1)) || (st = dev_alloc(h, p, &p->d_flags, (size_t)rows + 1))) { ctu_plan_destroy(p); return st; }
        *out = p;
        return CTU_OK;
    }
    const bool nr_on = h->nr_mode != NR_NONE;
    // the fp32 512-point feature chains always go PCM -> spectrum (k_frames2) -> k_bank
    const bool need_spec = h->signal_out || (nr_on && h->cfg.nr_when == 0) || (h->do_vad && h->vad_cri != VCRI_CEPDIST_FEA) ||
                           (!h->precise && !h->generic && h->fea_kind != FEA_NONE) ||
                           (fast256(h) && !h->precise && h->fea_kind != FEA_NONE);
    const bool lpc_kind = (h->fea_kind == FEA_LPA || h->fea_kind == FEA_LPC);
    const bool need_fb = !h->signal_out && ((nr_on && h->cfg.nr_when == 1) || lpc_kind);
    if (need_spec && (st = dev_alloc(h, p, &p->d_spec, (size_t)rows * h->spitch))) { ctu_plan_destroy(p); return st; }
    if (h->signal_out && h->bp.nfft && (st = dev_alloc(h, p, &p->d_yt, (size_t)rows * h->cfg.window))) { ctu_plan_destroy(p); return st; }
    if (h->signal_out && !h->bp.nfft && (st = dev_alloc(h, p, &p->d_cspec, (size_t)rows * NBIN))) { ctu_plan_destroy(p); return st; }
    if (need_fb && !h->precise && (st = dev_alloc(h, p, &p->d_fb, (size_t)rows * h->fb.nb))) { ctu_plan_destroy(p); return st; }
    if (need_fb && h->precise && (st = dev_alloc(h, p, &p->d_fb64, (size_t)rows * h->fb.nb))) { ctu_plan_destroy(p); return st; }
    if (h->do_vad && h->vad_cri == VCRI_CEPDIST_FEA && (st = dev_alloc(h, p, &p->d_fea64, (size_t)rows * h->feature_dim))) { ctu_plan_destroy(p); return st; }
    if (h->energy_mode && (st = dev_alloc(h, p, &p->d_E, (size_t)rows))) { ctu_plan_destroy(p); return st; }
    if (h->cfg.remove_dc1 && (st = dev_alloc(h, p, &p->d_dc1, (size_t)rows))) { ctu_plan_destroy(p); return st; }
    if (h->cfg.dither != 0.0 && (st = dev_alloc(h, p, &p->d_dither, (size_t)p->total_samples + 8))) { ctu_plan_destroy(p); return st; }
    if (h->fea_kind == FEA_TRAPDCT && (st = dev_alloc(h, p, &p->d_log, (size_t)rows * h->fb.nb))) { ctu_plan_destroy(p); return st; }
    const bool burg_nr = h->nr_mode >= NR_HWSS && h->vad_src == VADSRC_BURG;
    const bool burg_vad = h->do_vad && h->vad_cri == VCRI_CEPDIST_LPC;
    if ((burg_nr || burg_vad) && (st = dev_alloc(h, p, &p->d_ceps, (size_t)rows * BURG_MAXC))) { ctu_plan_destroy(p); return st; }
    if ((st = dev_alloc(h, p, &p->d_flags, (size_t)rows))) { ctu_plan_destroy(p); return st; }
    if (h->do_vad) {
        if ((st = dev_alloc(h, p, &p->d_cri, (size_t)rows)) || (st = dev_alloc(h, p, &p->d_keep, (size_t)rows)) || (st = dev_alloc(h, p, &p->d_vad0, (size_t)rows)) ||
            (st = dev_alloc(h, p, &p->d_rows, (size_t)n))) { ctu_plan_destroy(p); return st; }
        if (!std::strcmp(h->cfg.vad_out_mode, "debug") && (st = dev_alloc(h, p, &p->d_vdbg, (size_t)rows * VAD_DBG))) { ctu_plan_destroy(p); return st; }
    }
    *out = p;
    return CTU_OK;
}

void ctu_plan_destroy(ctu_plan *p) {
    if (!p) return;
    cudaSetDevice(p->h->device);
    cudaDeviceSynchronize();                 // what cudaFree would have done: nothing of this plan is in flight any more
    for (void *q : p->blocks)
        for (auto &b : p->h->pool) if (b.p == q) { b.used = false; break; }
    delete p;
}

int64_t ctu_plan_total_frames(const ctu_plan *p) { return p ? p->total_frames : 0; }
int64_t ctu_plan_max_rows(const ctu_plan *p) { return p ? p->total_frames : 0; }
int64_t ctu_plan_total_output_samples(const ctu_plan *p) { return p ? p->total_osamp : 0; }
int64_t ctu_plan_workspace_bytes(const ctu_plan *p) { return p ? p->workspace_bytes : 0; }
int ctu_plan_frames_per_utt(const ctu_plan *p, int64_t *f) {
    if (!p || !f) return CTU_ERR_CONFIG;
    for (int u = 0; u < p->n_utts; u++) f[u] = p->nframes[u];
    return CTU_OK;
}
int ctu_plan_rows_per_utt(const ctu_plan *p, int64_t *r) {
    if (!p || !r) return CTU_ERR_CONFIG;
    for (int u = 0; u < p->n_utts; u++) r[u] = p->rows_per_utt[u];
    return CTU_OK;
}

// ------------------------------------------------------------------------------------------
// kernel sequencing
// ------------------------------------------------------------------------------------------
struct Range {          // a contiguous run of utterances = contiguous tiles and rows
    int u0, u1;
    int64_t t32_0, t32_n, t64_0, t64_n, tS_0, tS_n, tF_0, tF_n, row0, nrows;
};

static Range make_range(const ctu_plan *p, int u0, int u1) {
    Range r;
    r.u0 = u0; r.u1 = u1;
    r.t32_0 = p->tile32_off[u0]; r.t32_n = p->tile32_off[u1] - r.t32_0;
    r.t64_0 = p->tile64_off[u0]; r.t64_n = p->tile64_off[u1] - r.t64_0;
    r.tS_0 = p->tileS_off[u0]; r.tS_n = p->tileS_off[u1] - r.tS_0;
    r.tF_0 = p->tileF_off[u0]; r.tF_n = p->tileF_off[u1] - r.tF_0;
    r.row0 = p->row_off[u0]; r.nrows = p->row_off[u1] - r.row0;
    return r;
}

struct Range;
// tile list of one contiguous run of utterances for the frame kernels
struct FrameTiles {
    const int2 *t16; int64_t n16;     // 16-frame tiles
    float2 *cplx = nullptr;           // PCM -> spectrum: also store the complex spectrum here (synthesis)
};

template <int SRC, int DST, int KIND, int WT>
static int launch_frames_w(ctu_handle *h, const FrameParams &P, const ctu_plan *p, const FrameTiles &ft, const int16_t *pcm,
                           const float *src, float *dst, cudaStream_t s) {
    static const char *const names[2][3] = {{"k_frames<pcm,spec>", "k_frames<pcm,fb>", "k_frames<pcm,fea>"},
                                            {"k_frames<spec,spec>", "k_frames<spec,fb>", "k_frames<spec,fea>"}};
    if constexpr (SRC == SRC_PCM && DST == DST_SPEC) {
        if (fast256(h) && !P.dither && !P.dc1) {
            if (ft.n16 <= 0) return CTU_OK;
            const size_t bytes = smem256_floats(P.window, P.wshift) * sizeof(float);
            CK(cudaFuncSetAttribute(k_frames256, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
            BatchDesc bd{p->d_pcm_off, p->d_nframes, p->d_row_off, ft.t16};
            Tables256 tb{h->d_tw128, h->d_any_ts, h->d_win};
            h->lc.begin(names[SRC][DST], s);
            int per_sm = 1;
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_frames256, F256_THREADS, bytes));
            const unsigned grid = (unsigned)std::min<int64_t>(ft.n16, (int64_t)std::max(per_sm, 1) * h->num_sms);
            k_frames256<<<grid, F256_THREADS, bytes, s>>>(P, bd, tb, pcm, dst, h->nbins, (int)ft.n16);
            h->lc.end(s);
            CK(cudaGetLastError());
            return CTU_OK;
        }
    }
    if (h->generic) {
        if (ft.n16 <= 0) return CTU_OK;
        int log2m = 0;
        while ((1 << (log2m + 1)) <= h->cfg.wfft / 2) log2m++;
        AnyTables tb{h->d_any_tw, h->d_any_ts, h->d_win, h->d_any_fbw, h->d_any_bands, h->cfg.wfft, log2m, -1, -1, -1, -1, (int)h->fbw_all.size(), -1,
                     (DST == DST_FEA && KIND == KIND_DCTC) ? P.nrows * P.nb : 0, -1,
                     (SRC == SRC_PCM && !P.dither && !P.dc1) ? (ANY_TILE - 1) * P.wshift + P.window : 0};
        const size_t bytes = any_stage_layout(tb, h->cfg.window);
        auto kern = k_frames_any<SRC, DST, KIND>;
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        BatchDesc bd{p->d_pcm_off, p->d_nframes, p->d_row_off, ft.t16};
        h->lc.begin(names[SRC][DST], s);
        kern<<<(unsigned)ft.n16, ANY_THREADS, bytes, s>>>(P, bd, tb, pcm, src, dst);
        h->lc.end(s);
        CK(cudaGetLastError());
        return CTU_OK;
    }
    if constexpr (SRC == SRC_PCM && DST == DST_SPEC) {
        if (ft.n16 <= 0) return CTU_OK;
        Smem2 L = smem2_layout(P.window, P.wshift);
        size_t bytes = (size_t)L.total * sizeof(float);
        auto kern = ft.cplx ? k_frames2<WT, true> : k_frames2<WT, false>;
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        FftTables tb{h->d_tw256, h->d_twsplit, h->d_twinv, h->d_win};
        BatchDesc bd{p->d_pcm_off, p->d_nframes, p->d_row_off, ft.t16};
        // persistent CTAs: exactly as many as are resident at once (five per SM at 25/10 ms, four at 32/16 ms)
        int per_sm = 1;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, F2_THREADS, bytes));
        const unsigned grid = (unsigned)std::min<int64_t>(ft.n16, std::max(per_sm, 1) * (int64_t)h->num_sms);
        h->lc.begin(names[SRC][DST], s);
        kern<<<grid, F2_THREADS, bytes, s>>>(P, bd, tb, pcm, dst, (int)ft.n16, ft.cplx);
        h->lc.end(s);
        CK(cudaGetLastError());
        return CTU_OK;
    } else {
        // 512-point band values and features come from the spectrum in k_bank (ctu_bank.cuh)
        return fail(h, CTU_ERR_CONFIG, "CTU: internal: 512-point band values or features outside k_bank");
    }
}

template <int SRC, int DST, int KIND>
static int launch_frames_t(ctu_handle *h, const FrameParams &P, const ctu_plan *p, const FrameTiles &ft, const int16_t *pcm,
                           const float *src, float *dst, cudaStream_t s) {
    // the PCM front end is specialised for the two standard window lengths (25 ms and 32 ms
    // at 16 kHz); every other length takes the generic instantiation
    if constexpr (SRC == SRC_PCM && DST == DST_SPEC) {
        if (P.window == 400) return launch_frames_w<SRC, DST, KIND, 400>(h, P, p, ft, pcm, src, dst, s);
        if (P.window == 512) return launch_frames_w<SRC, DST, KIND, 512>(h, P, p, ft, pcm, src, dst, s);
    }
    return launch_frames_w<SRC, DST, KIND, 0>(h, P, p, ft, pcm, src, dst, s);
}

template <int SRC, int DST>
static int launch_frames_k(ctu_handle *h, int kind, const FrameParams &P, const ctu_plan *p, const FrameTiles &ft, const int16_t *pcm,
                           const float *src, float *dst, cudaStream_t s) {
    switch (kind) {
        case KIND_SPEC: return launch_frames_t<SRC, DST, KIND_SPEC>(h, P, p, ft, pcm, src, dst, s);
        case KIND_LOGSPEC: return launch_frames_t<SRC, DST, KIND_LOGSPEC>(h, P, p, ft, pcm, src, dst, s);
        case KIND_DCTC: return launch_frames_t<SRC, DST, KIND_DCTC>(h, P, p, ft, pcm, src, dst, s);
        case KIND_TRAPLOG: return launch_frames_t<SRC, DST, KIND_TRAPLOG>(h, P, p, ft, pcm, src, dst, s);
    }
    return fail(h, CTU_ERR_CONFIG, "CTU: bad kind");
}

// LPC epilogue kernel over rows [row0, row0+nrows) of the band matrix
static int launch_lpc(ctu_handle *h, const FrameParams &P, bool ceps, int64_t row0, int64_t nrows, const float *fb, float *out, cudaStream_t s) {
    if (nrows <= 0) return CTU_OK;
    const unsigned grid = (unsigned)((nrows + LPC_THREADS - 1) / LPC_THREADS);
    const size_t bytes = (size_t)LPC_THREADS * (P.nb | 1) * sizeof(float);
    h->lc.begin("k_lpc", s);
    if (ceps && P.lporder == 12 && P.ncep == 12) k_lpc<12, 12, true><<<grid, LPC_THREADS, bytes, s>>>(P, row0, nrows, fb, out);
    else if (ceps) k_lpc<0, 0, true><<<grid, LPC_THREADS, bytes, s>>>(P, row0, nrows, fb, out);
    else if (P.lporder == 12) k_lpc<12, 0, false><<<grid, LPC_THREADS, bytes, s>>>(P, row0, nrows, fb, out);
    else k_lpc<0, 0, false><<<grid, LPC_THREADS, bytes, s>>>(P, row0, nrows, fb, out);
    h->lc.end(s);
    CK(cudaGetLastError());
    return CTU_OK;
}

static int kind_of(const ctu_handle *h) {
    switch (h->fea_kind) {
        case FEA_SPEC: return KIND_SPEC;
        case FEA_LOGSPEC: return KIND_LOGSPEC;
        case FEA_DCTC: return KIND_DCTC;
        case FEA_LPA: return KIND_LPA;
        case FEA_LPC: return KIND_LPC;
        case FEA_TRAPDCT: return KIND_TRAPLOG;
    }
    return KIND_SPEC;
}

static int prepare_dither(ctu_plan *p) {
    ctu_handle *h = p->h;
    if (!p->d_dither || p->dither_ready) return CTU_OK;
    const int w = h->cfg.window, s = h->cfg.wshift;
    std::vector<float> noise((size_t)p->total_samples + 8, 0.f);
    // resume from the state the previous plan left (only a shard offset set behind it, ctu_set_rand_offset, or plans
    // prepared out of order make the generator step from the seed)
    if (p->rand_base < h->rand_gen_pos) { h->rand_gen = GlibcRand(); h->rand_gen_pos = 0; }
    GlibcRand &g = h->rand_gen;
    for (uint64_t k = h->rand_gen_pos; k < p->rand_base; k++) g.step();
    uint64_t drawn = 0;
    const double d = h->cfg.dither;
    for (int u = 0; u < p->n_utts; u++) {
        const int64_t o = p->offsets[u] - p->offsets[0];
        const int64_t nloaded = (int64_t)p->nframes[u] * s + (w - s);
        for (int64_t k = 0; k < nloaded; k++) noise[(size_t)(o + k)] = (float)((2. * (double)g.next() / 2147483647. - 1.) * d);
        drawn += (uint64_t)nloaded;
    }
    h->rand_gen_pos = p->rand_base + drawn;
    // pageable source, consumers on non-blocking streams: wait for the DMA itself (see upload())
    CK(cudaMemcpy(p->d_dither, noise.data(), noise.size() * sizeof(float), cudaMemcpyHostToDevice));
    CK(cudaDeviceSynchronize());
    p->dither_ready = true;
    return CTU_OK;
}

// Runs utterances [u0,u1) of the plan on stream s.  All pointers are whole-batch device
// buffers (rows / samples are addressed through the plan's global offsets).
// ---- the delta / stacking / CMS chain on rows of work_dim floats (deltaFEA src/fea/fea_delta.cc:70-206, cms_POST
// src/fea/post_impl.cc:203-209); `src` = the matrix k_stack gathers the static block from (gather modes)
static int run_chain(ctu_plan *p, const Range &r, const BatchDesc &bd64, const float *src, float *d_fea, cudaStream_t s) {
    ctu_handle *h = p->h;
    // deltas of a plain column gather (feature-file input, spectral vectors): the delta kernel reads the static block from
    // the source itself; only stacking and the plain copy need k_stack
    const bool fused = h->gather && h->dp.n_order > 0 && h->skp.L == 1 && !h->skp.rot;
    if (h->gather && !fused && r.t64_n > 0) {
        const StackParams &S = h->skp;
        const size_t bytes = (size_t)(DELTA_ROWS + 2 * S.win + 1) * S.src_stride * sizeof(float);
        h->lc.begin("k_stack", s);
        if (bytes <= 96 * 1024) {
            CK(cudaFuncSetAttribute(k_stack<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
            k_stack<true><<<(unsigned)r.t64_n, 256, bytes, s>>>(S, bd64, DELTA_ROWS, src, d_fea);
        } else {
            k_stack<false><<<(unsigned)r.t64_n, 256, 0, s>>>(S, bd64, DELTA_ROWS, src, d_fea);
        }
        h->lc.end(s);
        CK(cudaGetLastError());
    }
    const float *dsrc = fused ? src : nullptr;
    const int dss = fused ? h->skp.src_stride : 0;
    if (h->dp.n_order > 0 && r.t64_n > 0) {
        const bool fast = (h->dp.n_order == 2 && h->dp.win[0] == 2 && h->dp.win[1] == 2 && h->dp.blk <= 16);
        size_t bytes = fast ? (size_t)(DELTA_ROWS + 8) * h->dp.blk * sizeof(float) : (size_t)2 * h->dp.span_max * h->dp.blk * sizeof(float);
        h->lc.begin("k_delta", s);
        if (fast) {
            k_delta22<float><<<(unsigned)r.t64_n, 256, bytes, s>>>(h->dp, bd64, d_fea, dsrc, dss);
        } else {
            CK(cudaFuncSetAttribute(k_delta<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
            k_delta<float><<<(unsigned)r.t64_n, 256, bytes, s>>>(h->dp, bd64, DELTA_ROWS, d_fea, dsrc, dss);
        }
        h->lc.end(s);
        CK(cudaGetLastError());
        if (p->d_fea64) {
            h->lc.begin("k_delta64", s);
            if (fast) {
                k_delta22<double><<<(unsigned)r.t64_n, 256, 2 * bytes, s>>>(h->dp, bd64, p->d_fea64);
            } else {
                CK(cudaFuncSetAttribute(k_delta<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * bytes)));
                k_delta<double><<<(unsigned)r.t64_n, 256, 2 * bytes, s>>>(h->dp, bd64, DELTA_ROWS, p->d_fea64);
            }
            h->lc.end(s);
            CK(cudaGetLastError());
        }
    }
    if (h->cfg.cms_exp_coef > 0 && h->cms_cols > 0 && r.nrows > 0) {
        // static block in writer order: c1..cN [c0]; c0 is normalised in the reference even when it is not written
        const int ncols = h->cms_cols, n = (r.u1 - r.u0) * ncols;
        h->lc.begin("k_cms_exp", s);
        k_cms_exp<<<(n + 127) / 128, 128, 0, s>>>(p->d_nframes, p->d_row_off, r.u0, r.u1 - r.u0, ncols, h->work_dim, h->cfg.cms_exp_coef, d_fea);
        h->lc.end(s);
        CK(cudaGetLastError());
    }
    return CTU_OK;
}

static int run_range(ctu_plan *p, const Range &r, const int16_t *d_pcm, const uint8_t *d_ext, float *d_fea, int16_t *d_wave,
                     uint8_t *d_vadnr, uint8_t *d_vadout, cudaStream_t s) {
    ctu_handle *h = p->h;
    if (r.nrows <= 0 && !h->signal_out) return CTU_OK;
    BatchDesc bd32{p->d_pcm_off, p->d_nframes, p->d_row_off, p->d_tiles32 + r.t32_0};
    BatchDesc bd64{p->d_pcm_off, p->d_nframes, p->d_row_off, p->d_tiles64 + r.t64_0};
    FrameTiles ft{p->d_tilesF + r.tF_0, r.tF_n};
    int st;
    if (h->fea_kind == FEA_TDIIR)        // time-domain IIR filter bank -> band energies -> log -> DCT (ctu_tdiir.cuh)
        return launch_tdiir(h->tdp, bd64, r.t64_n, p->d_pcm_off, p->d_nframes, p->d_row_off, r.u0, r.u1, d_pcm, p->d_tdseg, d_fea, h->feature_dim, s,
                            &h->lc, h->err);
    const int kind = kind_of(h);
    uint8_t *flags = d_vadnr ? d_vadnr : p->d_flags;

    // ---- stage 1: spectrum / band values, noise reduction ---------------------------------
    const bool nr_on = h->nr_mode != NR_NONE;
    const bool before = h->cfg.nr_when == 0 || h->signal_out;
    const bool need_spec = p->d_spec != nullptr;
    FrameParams P = h->fp;
    BurgParams BP = h->bp;
    BP.dc1 = p->d_dc1;
    if (p->d_dc1 && r.u1 > r.u0) {
        h->lc.begin("k_dc1_means", s);
        k_dc1_means<<<(unsigned)((r.u1 - r.u0 + 3) / 4), 128, 0, s>>>(p->d_nframes, p->d_row_off, p->d_pcm_off, r.u0, r.u1 - r.u0, h->cfg.window,
                                                                    h->cfg.wshift, d_pcm, p->d_dc1);
        h->lc.end(s);
        CK(cudaGetLastError());
        P.dc1 = p->d_dc1;
    }
    P.dither = p->d_dither ? p->d_dither - p->offsets[0] : nullptr;
    if (need_spec) {
        P.out_dim = h->nbins; P.out_stride = h->nbins;
        ft.cplx = p->d_cspec;                 // waveform output: X itself is kept for the synthesis
        if ((st = launch_frames_t<SRC_PCM, DST_SPEC, KIND_SPEC>(h, P, p, ft, d_pcm, nullptr, p->d_spec, s))) return st;
        ft.cplx = nullptr;
    }
    // the scan runs inside k_bank, on the tile in shared memory, whenever nothing but the filter bank consumes the enhanced
    // spectrum (the enhanced spectrum then never exists in HBM)
    const bool bank_path = need_spec && !h->generic && !h->precise && !h->signal_out && h->fea_kind != FEA_NONE;
    const bool carry = h->ss_carry && h->nr_mode >= NR_HWSS;
    const bool fuse_scan = bank_path && nr_on && before && h->fuse_nr && !h->do_vad && h->nrp.a_kind != 0 && !carry;
    if (nr_on && before) {
        if (h->nr_mode >= NR_HWSS && h->vad_src == VADSRC_BURG) {
            if ((st = launch_burg(BP, BURG_SRC_NR, bd32, r.t32_n, d_pcm, nullptr, p->d_ceps, h->d_tw256d, h->d_twsplitd, h->d_twinvd, h->d_wind,
                                  h->d_hann, s, &h->lc, h->err))) return st;
            if ((st = launch_cepdet(h->bp, p->d_nframes, p->d_row_off, r.u0, r.u1, p->d_ceps, flags, s, &h->lc, h->err))) return st;
        }
        const uint8_t *fl = (h->nr_mode >= NR_HWSS) ? (h->vad_src == VADSRC_FILE ? d_ext : flags) : nullptr;
        if (h->nr_mode >= NR_HWSS && !fl) return fail(h, CTU_ERR_INPUT, "NR: Unable to open VAD file!\n");
        if (carry) {
            if (h->carry_ev_set) CK(cudaStreamWaitEvent(s, h->carry_ev, 0));
            if ((st = launch_nr_scan_carry(h->nrp, p->d_nframes, p->d_row_off, r.u0, r.u1, h->nbins, h->spitch, p->d_spec, fl, h->d_carry,
                                           h->signal_out ? p->d_cspec : nullptr, s, &h->lc, h->err))) return st;
            CK(cudaEventRecord(h->carry_ev, s));
            h->carry_ev_set = true;
        } else
        if (!fuse_scan && (st = launch_nr_scan(h->nrp, p->d_nframes, p->d_row_off, r.u0, r.u1, h->nbins, h->spitch, p->d_spec, fl, s, &h->lc, h->err))) return st;
        if (h->vad_src == VADSRC_FILE && d_vadnr && h->nr_mode >= NR_HWSS)
            CK(cudaMemcpyAsync(d_vadnr + r.row0, d_ext + r.row0, r.nrows, cudaMemcpyDeviceToDevice, s));
    }
    if (h->signal_out && h->bp.nfft) {
        // other FFT sizes / odd window lengths: frames -> segments (fp64, one warp per frame), then overlap-add per 16-hop tile
        if (r.tF_n <= 0) return CTU_OK;
        BatchDesc bdF{p->d_pcm_off, p->d_nframes, p->d_row_off, p->d_tilesF + r.tF_0};
        const int N = h->cfg.wfft, M = N / 2;
        int lg = 0;
        while ((1 << lg) < M) lg++;
        AnyTables64 tb{h->d_any_tw64, h->d_any_ts64, h->d_wind, N, lg, h->spitch};
        const size_t bytes = (size_t)(SYNANY_THREADS / 32) * (2 * any64_zslots(M) + 2 * (M + 2)) * sizeof(double);
        auto ks = p->d_dc1 ? k_synth_frames_any<true> : k_synth_frames_any<false>;
        CK(cudaFuncSetAttribute(ks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        h->lc.begin("k_synth_frames_any", s);
        ks<<<(unsigned)r.tF_n, SYNANY_THREADS, bytes, s>>>(h->cfg.window, h->cfg.wshift, (double)h->cfg.preem, h->cfg.remove_dc, bdF, tb, d_pcm, p->d_spec, p->d_yt,
                                                          p->d_dc1);
        h->lc.end(s);
        CK(cudaGetLastError());
        h->lc.begin("k_ola_any", s);
        k_ola_any<<<(unsigned)r.tF_n, 256, 0, s>>>(h->cfg.window, h->cfg.wshift, 1.0 / h->sp.correction, bdF, p->d_osamp_off, p->d_yt, d_wave);
        h->lc.end(s);
        CK(cudaGetLastError());
        return CTU_OK;
    }
    if (h->signal_out) {
        BatchDesc bdS{p->d_pcm_off, p->d_nframes, p->d_row_off, p->d_tilesS + r.tS_0};
        return launch_synth_c(h->sp, h->fp, bdS, p->syn_tile, r.tS_n, p->d_osamp_off, p->d_cspec, p->d_spec, d_wave, h->d_tw256, h->d_twinv, s, &h->lc, h->err);
    }

    // ---- stage 2: features ------------------------------------------------------------------
    float *fea_dst = d_fea;
    int od = h->static_dim, ostride = h->feature_dim;
    if (kind == KIND_TRAPLOG) { fea_dst = p->d_log; od = h->fb.nb; ostride = h->fb.nb; }
    if (h->gather) { fea_dst = p->d_static; ostride = h->static_dim; }        // k_stack builds the rows from it
    P = h->fp; P.out_dim = od; P.out_stride = ostride;
    P.energy_mode = h->energy_mode; P.energy = p->d_E;
    P.dc1 = p->d_dc1;
    P.dither = p->d_dither ? p->d_dither - p->offsets[0] : nullptr;
    BankParams BK = h->bkp;
    BK.energy_mode = h->energy_mode; BK.energy = p->d_E;
    BK.flags = (h->nr_mode >= NR_HWSS) ? (h->vad_src == VADSRC_FILE ? d_ext : flags) : nullptr;
    if (h->precise) {
        // fp64 path (ctu_precise.cuh): band-domain noise reduction / ill-conditioned LPC /
        // features that feed VAD decisions
        Tables64 t64{h->d_tw256d, h->d_twsplitd, h->d_wind, h->d_w64, h->d_m264, h->d_lift64, h->bp.nfft, h->bp.log2m, h->bp.any_tw, h->bp.any_ts, h->spitch};
        double *f64 = (kind == KIND_TRAPLOG) ? nullptr : p->d_fea64;
        if (nr_on && !before) {
            const uint8_t *fl = (h->nr_mode >= NR_HWSS) ? d_ext : nullptr;
            if (h->nr_mode >= NR_HWSS && !fl) return fail(h, CTU_ERR_INPUT, "NR: Unable to open VAD file!\n");
            if ((st = launch_frames64(SRC64_PCM, DST64_FB, KIND_SPEC, P, bd32, t64, r.t32_n, d_pcm, nullptr, nullptr, p->d_fb64, nullptr, s, &h->lc, h->err))) return st;
            if (carry && h->carry_ev_set) CK(cudaStreamWaitEvent(s, h->carry_ev, 0));
            if ((st = launch_nr_scan64(h->nrp, p->d_nframes, p->d_row_off, r.u0, r.u1, h->fb.nb, p->d_fb64, fl, carry ? h->d_carry64 : nullptr, s, &h->lc, h->err))) return st;
            if (carry) { CK(cudaEventRecord(h->carry_ev, s)); h->carry_ev_set = true; }
            if (d_vadnr && fl) CK(cudaMemcpyAsync(d_vadnr + r.row0, d_ext + r.row0, r.nrows, cudaMemcpyDeviceToDevice, s));
            if ((st = launch_frames64(SRC64_FB, DST64_FEA, kind, P, bd32, t64, r.t32_n, nullptr, p->d_fb64, nullptr, f64, fea_dst, s, &h->lc, h->err))) return st;
        } else if (nr_on && before) {
            // noise-reduced fp32 spectrum (stage 1) is the source
            if ((st = launch_frames64(SRC64_SPEC, DST64_FEA, kind, P, bd32, t64, r.t32_n, nullptr, nullptr, p->d_spec, f64, fea_dst, s, &h->lc, h->err))) return st;
        } else {
            if ((st = launch_frames64(SRC64_PCM, DST64_FEA, kind, P, bd32, t64, r.t32_n, d_pcm, nullptr, nullptr, f64, fea_dst, s, &h->lc, h->err))) return st;
        }
    } else if (kind == KIND_LPA || kind == KIND_LPC) {
        // band values to HBM (76 B per frame for PLP), then one thread per frame for the recursion
        FrameParams Pf = h->fp; Pf.out_dim = h->fb.nb; Pf.out_stride = h->fb.nb;   // (its energy comes from k_lpc: log R0)
        Pf.dc1 = p->d_dc1; Pf.dither = P.dither;
        if (bank_path) {
            BK.out_dim = h->fb.nb; BK.out_stride = h->fb.nb; BK.energy_mode = EN_NONE;      // (log R0 comes from k_lpc)
            if ((st = launch_bank(BK, kind, true, fuse_scan, bd32, r.t32_n, r.u0, r.u1 - r.u0, h->num_sms, p->d_spec, p->d_fb, s, &h->lc, h->err))) return st;
        } else if (need_spec) { if ((st = launch_frames_t<SRC_SPEC, DST_FB, KIND_SPEC>(h, Pf, p, ft, nullptr, p->d_spec, p->d_fb, s))) return st; }
        else if ((st = launch_frames_t<SRC_PCM, DST_FB, KIND_SPEC>(h, Pf, p, ft, d_pcm, nullptr, p->d_fb, s))) return st;
        if ((st = launch_lpc(h, P, kind == KIND_LPC, r.row0, r.nrows, p->d_fb, fea_dst, s))) return st;
    } else if (bank_path) {
        BK.out_dim = od; BK.out_stride = ostride;
        if ((st = launch_bank(BK, kind, false, fuse_scan, bd32, r.t32_n, r.u0, r.u1 - r.u0, h->num_sms, p->d_spec, fea_dst, s, &h->lc, h->err))) return st;
    } else if (need_spec) {
        if ((st = launch_frames_k<SRC_SPEC, DST_FEA>(h, kind, P, p, ft, nullptr, p->d_spec, fea_dst, s))) return st;
    } else {
        if ((st = launch_frames_k<SRC_PCM, DST_FEA>(h, kind, P, p, ft, d_pcm, nullptr, fea_dst, s))) return st;
    }
    // ---- stage 3: long-context ------------------------------------------------------------
    if (kind == KIND_TRAPLOG && r.t64_n > 0) {
        size_t bytes = (size_t)(TRAP_ROWS + h->tp.L - 1) * h->tp.nb * sizeof(float);
        h->lc.begin("k_trapdct", s);
        if (h->tp.L == 51 && h->tp.ndct == 8) {
            CK(cudaFuncSetAttribute(k_trapdct<51, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
            k_trapdct<51, 8><<<(unsigned)r.t64_n, 256, bytes, s>>>(h->tp, bd64, TRAP_ROWS, p->d_log, d_fea);
        } else {
            CK(cudaFuncSetAttribute(k_trapdct<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
            k_trapdct<0, 0><<<(unsigned)r.t64_n, 256, bytes, s>>>(h->tp, bd64, TRAP_ROWS, p->d_log, d_fea);
        }
        h->lc.end(s);
        CK(cudaGetLastError());
    }
    if ((st = run_chain(p, r, bd64, p->d_static, d_fea, s))) return st;
    if (h->energy_mode && r.t64_n > 0) {
        if (h->energy_mode == EN_RAW) {
            h->lc.begin("k_rawenergy", s);
            if (p->d_dc1) k_rawenergy<true><<<(unsigned)r.t64_n, 256, 0, s>>>(bd64, h->cfg.window, h->cfg.wshift, d_pcm, p->d_E, p->d_dc1);
            else k_rawenergy<false><<<(unsigned)r.t64_n, 256, 0, s>>>(bd64, h->cfg.window, h->cfg.wshift, d_pcm, p->d_E, nullptr);
            h->lc.end(s);
        }
        h->lc.begin("k_place_energy", s);
        k_place_energy<<<(unsigned)r.t64_n, 256, 0, s>>>(bd64, h->energy_latency, h->feature_dim, p->d_E, d_fea);
        h->lc.end(s);
        CK(cudaGetLastError());
    }
    // ---- stage 4: VAD module -----------------------------------------------------------------
    if (h->do_vad) {
        VadParams VP = h->vp;
        VP.dbg = p->d_vdbg;
        if ((st = launch_vad_module(VP, BP, bd32, r.t32_n, p->d_nframes, p->d_row_off, r.u0, r.u1, r.row0, r.nrows, d_pcm, p->d_spec, d_fea,
                                    p->d_fea64, h->feature_dim, p->d_ceps, p->d_cri, p->d_vad0, d_vadout, p->d_keep, p->d_rows, h->d_tw256d, h->d_twsplitd,
                                    h->d_twinvd, h->d_wind, s, &h->lc, h->err))) return st;
    }
    return CTU_OK;
}

static int fetch_rows(ctu_plan *p, cudaStream_t s) {
    ctu_handle *h = p->h;
    if (!h->do_vad || !h->vad_drop) {
        for (int u = 0; u < p->n_utts; u++) p->rows_per_utt[u] = p->nframes[u];
        return CTU_OK;
    }
    std::vector<int> rows(p->n_utts);
    CK(cudaMemcpyAsync(rows.data(), p->d_rows, p->n_utts * sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    for (int u = 0; u < p->n_utts; u++) p->rows_per_utt[u] = rows[u];
    return CTU_OK;
}

int ctu_plan_run_device(ctu_plan *p, const int16_t *d_pcm, const uint8_t *d_ext_vad, float *d_features, int16_t *d_waveform,
                        uint8_t *d_vad_nr, uint8_t *d_vad_out, void *stream) {
    if (!p) return CTU_ERR_CONFIG;
    ctu_handle *h = p->h;
    CK(cudaSetDevice(h->device));
    if (h->fea_in) return fail(h, CTU_ERR_CONFIG, "CTU: this handle takes feature rows (-format_in htk): use ctu_plan_run_device_fea / ctu_plan_run_host_fea");
    if (!h->signal_out && !d_features) return fail(h, CTU_ERR_CAPACITY, "CTU: features buffer is NULL");
    if (h->signal_out && !d_waveform) return fail(h, CTU_ERR_CAPACITY, "CTU: waveform buffer is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    { int st0 = prepare_dither(p); if (st0) return st0; }
    Range r = make_range(p, 0, p->n_utts);
    if (h->signal_out) CK(cudaMemsetAsync(d_waveform, 0, (size_t)p->total_osamp * sizeof(int16_t), s));
    int st = run_range(p, r, d_pcm, d_ext_vad, d_features, d_waveform, d_vad_nr, d_vad_out, s);
    if (st) return st;
    return fetch_rows(p, s);
}

// G.711 expansion values, 16-bit (ITU-T G.711 tables scaled to 16 bits, which is what alaw2lin computes bit by bit,
// src/io/amulaw.h:19-56): segment number in bits 4-6, step in bits 0-3, sign in bit 7 (set = positive).
int ctu_g711_table(int alaw, int16_t *t) {
    if (!t) return CTU_ERR_CONFIG;
    for (int code = 0; code < 256; code++) {
        int v;
        if (alaw) {
            const int a = code ^ 0x55;                      // even bits are inverted on the line
            const int seg = (a >> 4) & 7, step = a & 15;
            v = (step << 4) + 8;                            // segment 0: linear, 16 per step
            if (seg >= 1) v = ((step << 4) + 0x108) << (seg - 1);
            if (!(a & 0x80)) v = -v;
        } else {
            const int u = ~code & 0xff;                     // mu-law codes are stored inverted
            const int seg = (u >> 4) & 7, step = u & 15;
            v = (((step << 3) + 0x84) << seg) - 0x84;
            if (u & 0x80) v = -v;
        }
        t[code] = (int16_t)v;
    }
    return CTU_OK;
}

static int run_host_impl(ctu_plan *p, const int16_t *pcm, const uint8_t *ext_vad, float *features, int16_t *waveform, uint8_t *vad_nr,
                         uint8_t *vad_out, bool keep, const uint8_t *codes = nullptr, int alaw = 0) {
    if (!p) return CTU_ERR_CONFIG;
    ctu_handle *h = p->h;
    CK(cudaSetDevice(h->device));
    if (h->fea_in) return fail(h, CTU_ERR_CONFIG, "CTU: this handle takes feature rows (-format_in htk): use ctu_plan_run_device_fea / ctu_plan_run_host_fea");
    if (!keep && !h->signal_out && !features) return fail(h, CTU_ERR_CAPACITY, "CTU: features buffer is NULL");
    if (!keep && h->signal_out && !waveform) return fail(h, CTU_ERR_CAPACITY, "CTU: waveform buffer is NULL");
    int st;
    if ((st = prepare_dither(p))) return st;
    if (!p->host_bufs) {
        if ((st = dev_alloc(h, p, &p->d_pcm, (size_t)p->total_samples + 8))) return st;
        if (!h->signal_out && (st = dev_alloc(h, p, &p->d_fea, (size_t)p->total_frames * h->feature_dim))) return st;
        if (h->signal_out && (st = dev_alloc(h, p, &p->d_wave, (size_t)p->total_osamp))) return st;
        if ((st = dev_alloc(h, p, &p->d_ext, (size_t)p->total_frames))) return st;
        if ((st = dev_alloc(h, p, &p->d_vadnr_out, (size_t)p->total_frames))) return st;
        if ((st = dev_alloc(h, p, &p->d_vad_out, (size_t)p->total_frames))) return st;
        p->host_bufs = true;
    }
    if (p->row_format == CTU_ROWS_PFILE && !p->d_fmt && !h->signal_out &&
        (st = dev_alloc(h, p, &p->d_fmt, (size_t)p->total_frames * (h->feature_dim + 2) + 8))) return st;
    if (codes) {
        if (!p->d_codes && (st = dev_alloc(h, p, &p->d_codes, (size_t)p->total_samples + 16))) return st;
        int16_t *&tab = h->d_g711[alaw ? 1 : 0];
        if (!tab) {
            std::vector<int16_t> t(256);
            ctu_g711_table(alaw, t.data());
            if ((st = upload(h, &tab, t))) return st;
        }
    }
    // chunks of utterances of roughly 32 MB of PCM, round-robin over three streams so that
    // H2D of chunk i+1, the kernels of chunk i and D2H of chunk i-1 overlap
    const int64_t chunk_samples = (int64_t)h->chunk_mb << 19;
    // the NR-internal detector's decisions exist only for hwss / fwss / 2fwss; otherwise the caller gets zeros
    const bool have_vadnr = h->nr_mode >= NR_HWSS;
    if (vad_nr && !have_vadnr && !keep) std::memset(vad_nr, 0, (size_t)p->total_frames);
    int u0 = 0, ci = 0;
    const int64_t base = p->offsets[0];
    st = CTU_OK;
    // an error in the middle of the loop must not return while copies into the caller's buffers are in flight
#define CKL(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            h->err = std::string("CUDA: ") + cudaGetErrorString(e_) + " at " #call;                \
            st = CTU_ERR_CUDA;                                                                     \
            goto drain;                                                                            \
        }                                                                                          \
    } while (0)
    while (u0 < p->n_utts) {
        int u1 = u0 + 1;
        while (u1 < p->n_utts && p->offsets[u1 + 1] - p->offsets[u0] <= chunk_samples) u1++;
        // td-iir-mfcc: the filter recurrence is sequential along an utterance, its parallelism is utterances x 24 bands --
        // a chunk must hold enough utterances to fill the device (five CTAs of four utterances per SM), whatever their size
        if (h->fea_kind == FEA_TDIIR) u1 = std::max(u1, std::min(p->n_utts, u0 + 20 * h->num_sms));
        cudaStream_t s = h->streams[ci % 3];
        Range r = make_range(p, u0, u1);
        int64_t so = p->offsets[u0] - base, sn = p->offsets[u1] - p->offsets[u0];
        if (codes) {
            // one byte per sample over PCIe; expanded next to the PCM buffer's own indexing
            CKL(cudaMemcpyAsync(p->d_codes + so, codes + p->offsets[u0], (size_t)sn, cudaMemcpyHostToDevice, s));
            if (sn > 0 && !h->copy_only) {
                h->lc.begin("k_g711_expand", s);
                k_g711_expand<<<(unsigned)std::min<int64_t>((sn / 8 + 256) / 256, 148 * 8), 256, 0, s>>>(p->d_codes, p->d_pcm, so, sn, h->d_g711[alaw ? 1 : 0]);
                h->lc.end(s);
                CKL(cudaGetLastError());
            }
        } else {
            CKL(cudaMemcpyAsync(p->d_pcm + so, pcm + p->offsets[u0], sn * sizeof(int16_t), cudaMemcpyHostToDevice, s));
        }
        if (ext_vad && r.nrows) CKL(cudaMemcpyAsync(p->d_ext + r.row0, ext_vad + r.row0, r.nrows, cudaMemcpyHostToDevice, s));
        // copy_only (ctu_set_option): the same chunk schedule with the kernels left out -- the control measurement that
        // says how much of the end-to-end time is the host <-> device copies themselves (bench.py e2e.copy_only_ms)
        if (!h->copy_only) {
            if (h->signal_out) CKL(cudaMemsetAsync(p->d_wave + p->osamp_off[u0], 0, (size_t)(p->osamp_off[u1] - p->osamp_off[u0]) * sizeof(int16_t), s));
            if ((st = run_range(p, r, p->d_pcm - base, ext_vad ? p->d_ext : nullptr, p->d_fea, p->d_wave, p->d_vadnr_out, p->d_vad_out, s))) goto drain;
        }
        if (keep) { u0 = u1; ci++; continue; }             // results stay on the device (ctu_plan_fetch brings them back)
        if (!h->signal_out && r.nrows) {
            const void *srcp = p->d_fea + r.row0 * h->feature_dim;
            size_t row_bytes = (size_t)h->feature_dim * sizeof(float);
            if (p->row_format != CTU_ROWS_NATIVE && r.t64_n > 0 && !h->copy_only) {
                // container rows formatted on the device: the host writer is left with one fwrite per utterance (or batch)
                const bool pf = p->row_format == CTU_ROWS_PFILE;
                BatchDesc bd64{p->d_pcm_off, p->d_nframes, p->d_row_off, p->d_tiles64 + r.t64_0};
                h->lc.begin("k_format_rows", s);
                k_format_rows<<<(unsigned)r.t64_n, 256, 0, s>>>(bd64, h->feature_dim, pf ? 1 : 0, p->sent0, p->d_fea, pf ? p->d_fmt : reinterpret_cast<uint32_t *>(p->d_fea));
                h->lc.end(s);
                CKL(cudaGetLastError());
            }
            if (p->row_format == CTU_ROWS_PFILE) { row_bytes += 8; srcp = p->d_fmt + r.row0 * (h->feature_dim + 2); }
            CKL(cudaMemcpyAsync(reinterpret_cast<char *>(features) + (size_t)r.row0 * row_bytes, srcp, (size_t)r.nrows * row_bytes, cudaMemcpyDeviceToHost, s));
        }
        if (h->signal_out) {
            int64_t o0 = p->osamp_off[u0], on = p->osamp_off[u1] - o0;
            CKL(cudaMemcpyAsync(waveform + o0, p->d_wave + o0, on * sizeof(int16_t), cudaMemcpyDeviceToHost, s));
        }
        if (vad_nr && r.nrows && have_vadnr) CKL(cudaMemcpyAsync(vad_nr + r.row0, p->d_vadnr_out + r.row0, r.nrows, cudaMemcpyDeviceToHost, s));
        if (vad_out && r.nrows && h->do_vad) CKL(cudaMemcpyAsync(vad_out + r.row0, p->d_vad_out + r.row0, r.nrows, cudaMemcpyDeviceToHost, s));
        u0 = u1; ci++;
    }
#undef CKL
drain:
    for (int i = 0; i < 3; i++) {
        cudaError_t e = cudaStreamSynchronize(h->streams[i]);
        if (e != cudaSuccess && st == CTU_OK) { h->err = std::string("CUDA: ") + cudaGetErrorString(e) + " (stream synchronize)"; st = CTU_ERR_CUDA; }
    }
    if (st) return st;
    return fetch_rows(p, h->streams[0]);
}

int ctu_plan_run_host(ctu_plan *p, const int16_t *pcm, const uint8_t *ext_vad, float *features, int16_t *waveform, uint8_t *vad_nr,
                      uint8_t *vad_out) {
    return run_host_impl(p, pcm, ext_vad, features, waveform, vad_nr, vad_out, false);
}

int ctu_plan_run_host_g711(ctu_plan *p, const uint8_t *codes, int alaw, const uint8_t *ext_vad, float *features, int16_t *waveform,
                           uint8_t *vad_nr, uint8_t *vad_out) {
    if (!codes) return CTU_ERR_CONFIG;
    return run_host_impl(p, nullptr, ext_vad, features, waveform, vad_nr, vad_out, false, codes, alaw);
}

int ctu_plan_run_host_keep(ctu_plan *p, const int16_t *pcm, const uint8_t *ext_vad) {
    return run_host_impl(p, pcm, ext_vad, nullptr, nullptr, nullptr, nullptr, true);
}

int ctu_plan_fetch(ctu_plan *p, float *features, int16_t *waveform, uint8_t *vad_nr, uint8_t *vad_out) {
    if (!p || !p->host_bufs) return CTU_ERR_CONFIG;
    ctu_handle *h = p->h;
    CK(cudaSetDevice(h->device));
    if (features && p->d_fea) CK(cudaMemcpy(features, p->d_fea, (size_t)p->total_frames * h->feature_dim * sizeof(float), cudaMemcpyDeviceToHost));
    if (waveform && p->d_wave) CK(cudaMemcpy(waveform, p->d_wave, (size_t)p->total_osamp * sizeof(int16_t), cudaMemcpyDeviceToHost));
    if (vad_nr && p->d_vadnr_out) CK(cudaMemcpy(vad_nr, p->d_vadnr_out, (size_t)p->total_frames, cudaMemcpyDeviceToHost));
    if (vad_out && h->do_vad) CK(cudaMemcpy(vad_out, p->d_vad_out, (size_t)p->total_frames, cudaMemcpyDeviceToHost));
    return CTU_OK;
}

// ---- feature-file input: rows in, rows out (htkIN -> deltaFEA -> cms_POST -> OUT, src/io/batch.cc:55-60, 217-218) -----
static int run_range_fea(ctu_plan *p, const Range &r, const float *d_in, float *d_fea, cudaStream_t s) {
    ctu_handle *h = p->h;
    if (r.nrows <= 0) return CTU_OK;
    BatchDesc bd64{p->d_pcm_off, p->d_nframes, p->d_row_off, p->d_tiles64 + r.t64_0};
    float *work = p->d_work ? p->d_work : d_fea;
    int st = run_chain(p, r, bd64, d_in, work, s);
    if (st) return st;
    if (p->d_work)      // the writer drops the last element of every row (htkOUT::get_fea_size, src/io/out.cc:95-112)
        CK(cudaMemcpy2DAsync(d_fea + r.row0 * h->feature_dim, (size_t)h->feature_dim * sizeof(float), work + r.row0 * h->work_dim,
                             (size_t)h->work_dim * sizeof(float), (size_t)h->feature_dim * sizeof(float), (size_t)r.nrows, cudaMemcpyDeviceToDevice, s));
    return CTU_OK;
}

int ctu_plan_run_device_fea(ctu_plan *p, const float *d_fea_in, float *d_features, void *stream) {
    if (!p) return CTU_ERR_CONFIG;
    ctu_handle *h = p->h;
    CK(cudaSetDevice(h->device));
    if (!h->fea_in) return fail(h, CTU_ERR_CONFIG, "CTU: this handle takes PCM: use ctu_plan_run_device / ctu_plan_run_host");
    if (!d_fea_in || !d_features) return fail(h, CTU_ERR_CAPACITY, "CTU: feature buffer is NULL");
    int st = run_range_fea(p, make_range(p, 0, p->n_utts), d_fea_in + p->offsets[0] * h->in_dim, d_features, (cudaStream_t)stream);
    if (st) return st;
    return fetch_rows(p, (cudaStream_t)stream);
}

int ctu_plan_run_host_fea(ctu_plan *p, const float *fea_in, float *features) {
    if (!p) return CTU_ERR_CONFIG;
    ctu_handle *h = p->h;
    CK(cudaSetDevice(h->device));
    if (!h->fea_in) return fail(h, CTU_ERR_CONFIG, "CTU: this handle takes PCM: use ctu_plan_run_device / ctu_plan_run_host");
    if (!fea_in) return fail(h, CTU_ERR_CAPACITY, "CTU: feature buffer is NULL");
    int st;
    if (!p->host_bufs) {
        if ((st = dev_alloc(h, p, &p->d_in, (size_t)p->total_frames * h->in_dim + 8))) return st;
        if ((st = dev_alloc(h, p, &p->d_fea, (size_t)p->total_frames * h->feature_dim + 8))) return st;
        p->host_bufs = true;
    }
    // the same three-stream pipeline as the PCM entry point: chunks of utterances of about 32 MB of input
    const int64_t chunk_rows = std::max<int64_t>(1, ((int64_t)h->chunk_mb << 20) / ((int64_t)h->in_dim * (int64_t)sizeof(float)));
    const float *in0 = fea_in + p->offsets[0] * h->in_dim;
    int u0 = 0, ci = 0;
    st = CTU_OK;
    cudaError_t ce = cudaSuccess;
    while (u0 < p->n_utts && st == CTU_OK && ce == cudaSuccess) {
        int u1 = u0 + 1;
        while (u1 < p->n_utts && p->row_off[u1 + 1] - p->row_off[u0] <= chunk_rows) u1++;
        cudaStream_t s = h->streams[ci % 3];
        Range r = make_range(p, u0, u1);
        if (r.nrows) {
            ce = cudaMemcpyAsync(p->d_in + r.row0 * h->in_dim, in0 + r.row0 * h->in_dim, (size_t)r.nrows * h->in_dim * sizeof(float), cudaMemcpyHostToDevice, s);
            if (ce == cudaSuccess && !h->copy_only) st = run_range_fea(p, r, p->d_in, p->d_fea, s);
            if (ce == cudaSuccess && st == CTU_OK && features)
                ce = cudaMemcpyAsync(features + r.row0 * h->feature_dim, p->d_fea + r.row0 * h->feature_dim,
                                     (size_t)r.nrows * h->feature_dim * sizeof(float), cudaMemcpyDeviceToHost, s);
        }
        u0 = u1; ci++;
    }
    // also on an error: nothing may still be copying into the caller's buffer when this returns
    for (int i = 0; i < 3; i++) { cudaError_t e = cudaStreamSynchronize(h->streams[i]); if (ce == cudaSuccess) ce = e; }
    if (st) return st;
    CK(ce);
    return fetch_rows(p, h->streams[0]);
}

// ---- per-utterance column statistics and normalisation of the device-resident feature rows: the device
// half of CMVN (cmvn_POST::sum_fea / sum_cv / process_frame, src/fea/post_impl.cc:52-118).  The host
// groups utterances by speaker and owns the statistics file.
int ctu_cmvn_dim(const ctu_handle *h) { return h ? h->feature_dim - (h->energy_mode ? 1 : 0) : 0; }

int ctu_plan_colsums(ctu_plan *p, const double *center, double *sums) {
    if (!p || !sums || !p->host_bufs || !p->d_fea) return CTU_ERR_CONFIG;
    ctu_handle *h = p->h;
    CK(cudaSetDevice(h->device));
    const int dim = ctu_cmvn_dim(h);
    const size_t n = (size_t)p->n_utts * dim;
    if (n == 0) return CTU_OK;
    double *d_c = nullptr, *d_s = nullptr;
    int st;
    if ((st = dev_alloc(h, p, &d_s, n))) return st;
    if (center) {
        if ((st = dev_alloc(h, p, &d_c, n))) return st;
        CK(cudaMemcpyAsync(d_c, center, n * sizeof(double), cudaMemcpyHostToDevice, h->streams[0]));
    }
    h->lc.begin("k_colsums", h->streams[0]);
    k_colsums<<<(unsigned)((n + 127) / 128), 128, 0, h->streams[0]>>>(p->d_nframes, p->d_row_off, p->n_utts, dim, h->feature_dim, p->d_fea, d_c, d_s);
    h->lc.end(h->streams[0]);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(sums, d_s, n * sizeof(double), cudaMemcpyDeviceToHost, h->streams[0]));
    CK(cudaStreamSynchronize(h->streams[0]));
    return CTU_OK;
}

int ctu_plan_normalise(ctu_plan *p, const double *mean, const double *scale) {
    if (!p || !mean || !scale || !p->host_bufs || !p->d_fea) return CTU_ERR_CONFIG;
    ctu_handle *h = p->h;
    CK(cudaSetDevice(h->device));
    const int dim = ctu_cmvn_dim(h);
    const size_t n = (size_t)p->n_utts * dim;
    if (n == 0) return CTU_OK;
    double *d_m = nullptr, *d_v = nullptr;
    int st;
    if ((st = dev_alloc(h, p, &d_m, n)) || (st = dev_alloc(h, p, &d_v, n))) return st;
    // stream-ordered on the stream that runs k_normalise (a pageable source makes the call itself synchronous)
    CK(cudaMemcpyAsync(d_m, mean, n * sizeof(double), cudaMemcpyHostToDevice, h->streams[0]));
    CK(cudaMemcpyAsync(d_v, scale, n * sizeof(double), cudaMemcpyHostToDevice, h->streams[0]));
    const int64_t t64 = p->tile64_off[p->n_utts];
    if (t64 > 0) {
        BatchDesc bd64{p->d_pcm_off, p->d_nframes, p->d_row_off, p->d_tiles64};
        h->lc.begin("k_normalise", h->streams[0]);
        k_normalise<<<(unsigned)t64, 256, 0, h->streams[0]>>>(bd64, dim, h->feature_dim, d_m, d_v, p->d_fea);
        h->lc.end(h->streams[0]);
        CK(cudaGetLastError());
    }
    CK(cudaStreamSynchronize(h->streams[0]));
    return CTU_OK;
}

int ctu_run(ctu_handle *h, const int16_t *pcm, const int64_t *off, int32_t n, const uint8_t *ext_vad, float *features,
            int64_t fcap_rows, int16_t *waveform, int64_t wcap, uint8_t *vad_nr, uint8_t *vad_out, int64_t *frames_per_utt,
            int64_t *rows_per_utt) {
    ctu_plan *p = nullptr;
    int st = ctu_plan_create(h, off, n, &p);
    if (st) return st;
    if (!h->signal_out && fcap_rows < p->total_frames) { ctu_plan_destroy(p); return fail(h, CTU_ERR_CAPACITY, "CTU: features buffer too small"); }
    if (h->signal_out && wcap < p->total_osamp) { ctu_plan_destroy(p); return fail(h, CTU_ERR_CAPACITY, "CTU: waveform buffer too small"); }
    st = ctu_plan_run_host(p, pcm + 0, ext_vad, features, waveform, vad_nr, vad_out);
    if (!st && frames_per_utt) ctu_plan_frames_per_utt(p, frames_per_utt);
    if (!st && rows_per_utt) ctu_plan_rows_per_utt(p, rows_per_utt);
    ctu_plan_destroy(p);
    return st;
}

int ctu_plan_set_row_format(ctu_plan *p, int format, uint32_t first_sentence) {
    if (!p) return CTU_ERR_CONFIG;
    ctu_handle *h = p->h;
    if (format != CTU_ROWS_NATIVE && format != CTU_ROWS_BE && format != CTU_ROWS_PFILE) return fail(h, CTU_ERR_CONFIG, "CTU: unknown row format");
    if (format != CTU_ROWS_NATIVE && (h->signal_out || h->fea_in)) return fail(h, CTU_ERR_UNSUPPORTED, "CTU: row formats apply to feature output from sample input");
    p->row_format = format;
    p->sent0 = first_sentence;
    return CTU_OK;
}
int64_t ctu_plan_row_bytes(const ctu_plan *p) {
    if (!p) return 0;
    return (int64_t)sizeof(float) * (p->h->feature_dim + (p->row_format == CTU_ROWS_PFILE ? 2 : 0));
}

int ctu_plan_fetch_vad_debug(ctu_plan *p, double *steps, uint8_t *vad0) {
    if (!p) return CTU_ERR_CONFIG;
    ctu_handle *h = p->h;
    if (!p->d_vdbg) return fail(h, CTU_ERR_CONFIG, "CTU: the handle was not created with -vad_out_mode debug");
    CK(cudaSetDevice(h->device));
    CK(cudaDeviceSynchronize());
    if (steps) CK(cudaMemcpy(steps, p->d_vdbg, (size_t)p->total_frames * VAD_DBG * sizeof(double), cudaMemcpyDeviceToHost));
    if (vad0) CK(cudaMemcpy(vad0, p->d_vad0, (size_t)p->total_frames, cudaMemcpyDeviceToHost));
    return CTU_OK;
}

int ctu_set_option(ctu_handle *h, const char *name, int64_t value) {
    if (!h || !name) return CTU_ERR_CONFIG;
    const std::string n(name);
    if (n == "copy_only") h->copy_only = value != 0;
    else if (n == "chunk_mb") h->chunk_mb = (int)std::max<int64_t>(1, value);
    else if (n == "ss_carry") {
        // (re)starts a list: the buffer is zero before the first file of a reference process (Vec's constructor, src/base/types.h:35-38)
        if (value && h->nr_mode >= NR_HWSS) {
            if (h->signal_out && h->bp.nfft)
                return fail(h, CTU_ERR_UNSUPPORTED, "CTU: ss_carry with waveform output on the general synthesis (FFT sizes other than 512, odd window lengths, -remove_dc1)");
            CK(cudaSetDevice(h->device));
            const size_t nmax = (size_t)std::max(h->nbins, h->fb.nb) + 8;
            if (!h->d_carry) CK(cudaMalloc(&h->d_carry, nmax * sizeof(float)));
            if (!h->d_carry64) CK(cudaMalloc(&h->d_carry64, nmax * sizeof(double)));
            if (!h->carry_ev) CK(cudaEventCreateWithFlags(&h->carry_ev, cudaEventDisableTiming));
            CK(cudaMemset(h->d_carry, 0, nmax * sizeof(float)));
            CK(cudaMemset(h->d_carry64, 0, nmax * sizeof(double)));
            CK(cudaDeviceSynchronize());
            h->carry_ev_set = false;
        }
        h->ss_carry = value != 0;
    }
    else if (n == "fuse_nr") h->fuse_nr = value != 0;
    else if (n == "front256") h->front256 = value != 0;                   // takes effect for plans created afterwards
    else return fail(h, CTU_ERR_CONFIG, "CTU: unknown run-time option " + n);
    return CTU_OK;
}

int ctu_set_rand_offset(ctu_handle *h, uint64_t drawn) {
    if (!h) return CTU_ERR_CONFIG;
    h->rand_pos = drawn;
    return CTU_OK;
}

int ctu_host_alloc(void **ptr, uint64_t bytes) {
    if (!ptr) return CTU_ERR_CONFIG;
    *ptr = nullptr;
    cudaError_t e = cudaHostAlloc(ptr, (size_t)std::max<uint64_t>(bytes, 1), cudaHostAllocDefault);
    if (e != cudaSuccess) { g_create_err = std::string("CUDA: ") + cudaGetErrorString(e) + " (cudaHostAlloc)"; return CTU_ERR_CUDA; }
    return CTU_OK;
}
void ctu_host_free(void *ptr) { if (ptr) cudaFreeHost(ptr); }
int ctu_device_count(void) { int n = 0; return cudaGetDeviceCount(&n) == cudaSuccess ? n : 0; }

int ctu_debug_spectrum(ctu_plan *p, const int16_t *d_pcm, float *d_spec, void *stream) {
    if (!p) return CTU_ERR_CONFIG;
    ctu_handle *h = p->h;
    CK(cudaSetDevice(h->device));
    const FrameTiles ft{p->d_tilesF, p->tileF_off[p->n_utts]};
    FrameParams P = h->fp; P.out_dim = h->nbins; P.out_stride = h->nbins;
    // the kernels write rows of h->spitch floats (260 on the 512-point path); the tap hands out compact rows
    float *tmp = d_spec;
    int st;
    if (h->spitch != h->nbins) {
        tmp = p->d_spec;
        if (!tmp && (st = dev_alloc(h, p, &p->d_spec, (size_t)p->total_frames * h->spitch))) return st;
        tmp = p->d_spec;
    }
    st = launch_frames_t<SRC_PCM, DST_SPEC, KIND_SPEC>(h, P, p, ft, d_pcm, nullptr, tmp, (cudaStream_t)stream);
    if (st) return st;
    if (tmp != d_spec && p->total_frames > 0)
        CK(cudaMemcpy2DAsync(d_spec, (size_t)h->nbins * sizeof(float), tmp, (size_t)h->spitch * sizeof(float), (size_t)h->nbins * sizeof(float),
                             (size_t)p->total_frames, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    return CTU_OK;
}
