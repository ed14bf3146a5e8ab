/*
 * ctucopy_b200.h -- C ABI of the B200-native CtuCopy hot path.
 *
 * The reference (pmizera/ctucopy 4.0.2) has no plugin / FFI seam: its hot path is the
 * per-file, per-frame loop of BATCH::process (src/io/batch.cc:297-422) calling
 * IN::get_frame (src/io/in.cc:305-419), NR::process_frame (src/nr/nr.cc), FB::project_frame
 * (src/fea/fb.cc:72-86), FEA::process_frame (src/fea/fea_impl.cc, fea_trap.cc),
 * deltaFEA (src/fea/fea_delta.cc), VAD (src/vad/vad.cc) and sigOUT::save_frame
 * (src/io/out.cc:405-451), one frame at a time through shared Vec<double> buffers.
 * A GPU cannot be fed frame by frame, so this ABI replaces that loop at BATCH granularity:
 * a whole list of utterances in, per-utterance frame counts + a feature matrix in the
 * WRITER's column order (src/io/out.cc:183-202) or an int16 waveform out.  What stays on
 * the host is what the reference does outside the loop: option parsing, file decoding,
 * the HTK / pfile / ark / raw / wave writers and list iteration (host/ in this repo).
 *
 * Plain C types only; no exceptions cross the boundary; every function returns a
 * ctu_status (0 = OK) and ctu_last_error() gives the reference's own message text where
 * the reference would have thrown one (src/main.cpp:31-60 maps those to exit status 255).
 * A handle is single-owner and not thread-safe: one handle per GPU / host thread.
 */
#ifndef CTUCOPY_B200_H
#define CTUCOPY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CTU_ABI_VERSION 4
#define CTU_STR 40
#define CTU_FBDEF 1024

typedef enum ctu_status {
    CTU_OK = 0,
    CTU_ERR_CONFIG = 1,      /* option error (the reference throws "OPTS: ...", "FB: ...", "NR: ...") */
    CTU_ERR_INPUT = 2,       /* e.g. "IO: Signal shorter than one frame!" (src/io/in.cc:277)          */
    CTU_ERR_UNSUPPORTED = 3, /* not built here, or undefined behaviour in the reference (message says) */
    CTU_ERR_CUDA = 4,        /* CUDA runtime failure, or no usable device: there is NO CPU fallback   */
    CTU_ERR_CAPACITY = 5     /* caller's output buffer too small                                      */
} ctu_status;

/* The hot-path subset of `class opts` (src/io/opts.h:36-166), same names, same meaning,
 * same defaults (src/io/opts.cc:34-146).  Strings are NUL-terminated; booleans are 0/1. */
typedef struct ctu_config {
    int32_t abi_version;             /* CTU_ABI_VERSION                                          */
    /* IO */
    char    format_out[CTU_STR];     /* htk|pfile|ark -> features; raw|wave -> enhanced waveform  */
    int32_t fs;
    float   preem;                   /* stored as float like the reference (src/io/opts.h:47)     */
    double  dither;                  /* amplitude of the uniform dither (code default 0, src/io/opts.cc:38) */
    int32_t remove_dc, remove_dc1;
    double  window_ms, wshift_ms;
    /* filter bank */
    char    fb_scale[CTU_STR], fb_shape[CTU_STR];
    int32_t fb_norm, fb_power, fb_eqld, fb_inld;
    char    fb_definition[CTU_FBDEF];
    /* noise reduction */
    char    vadmode[CTU_STR];        /* none|burg|file                                           */
    char    nr_mode[CTU_STR];        /* none|exten|hwss|fwss|2fwss                               */
    double  nr_p, nr_q, nr_a, nr_b;
    int32_t nr_initsegs;
    int32_t nr_when;                 /* 0 = beforeFB, 1 = afterFB (opts::NRwhen)                  */
    /* parametrisation */
    char    fea_kind[CTU_STR];       /* spec|logspec|dctc|lpa|lpc|trapdct|td-iir-mfcc            */
    int32_t fea_lporder, fea_ncepcoefs, fea_c0, fea_E, fea_rawenergy, fea_lifter;
    int32_t fea_trapdct_traplen, fea_trapdct_ndct;
    int32_t fea_delta, n_order, d_win, a_win, t_win;
    /* VAD module */
    char    vad_apply_mode[CTU_STR]; /* none|silence|drop                                        */
    char    vad_out_mode[CTU_STR];   /* none|vad|debug                                           */
    char    vad_cri_mode[CTU_STR];   /* energy|cepdist                                           */
    char    vad_thr_mode[CTU_STR];   /* absolute|perc|adapt|dyn                                  */
    int32_t vad_energy_db;
    char    vad_cepdist_mode[CTU_STR]; /* lpc|fea|in                                             */
    double  vad_cepdist_p;
    int32_t vad_cepdist_init, vad_lpc_coefs;
    double  vad_absolute_thr;
    int32_t vad_perc_init;
    double  vad_perc_thr;
    int32_t vad_adapt_init;
    double  vad_adapt_q, vad_adapt_za;
    int32_t vad_dyn_init;
    double  vad_dyn_perc, vad_dyn_min, vad_dyn_qmaxinc, vad_dyn_qmaxdec, vad_dyn_qmindec, vad_dyn_qmininc;
    int32_t vad_filter_order;
    /* derived by ctu_config_finalize (opts::check_config, src/io/opts.cc:255-325) */
    int32_t window, wshift, wfft, wfftby2, phase_needed;
    /* post-processing (src/fea/post_impl.cc): cepstral mean subtraction.  Time constants in ms, -1 = off
     * (floats like the reference, src/io/opts.h); cms_exp_coef = 1 - 2*wshift_ms/fea_Z_exp is derived.   */
    float   fea_Z_exp, fea_Z_block;
    float   cms_exp_coef;
    int32_t stat_cmvn, apply_cmvn;   /* CMVN passes: the host drives them (ctu_plan_colsums / _normalise)  */
    /* context stacking and feature-file input (src/io/opts.cc:694-704, 786; src/io/in.cc:623-690)         */
    int32_t fea_trap, trap_win;      /* -fea_trap N: rows t-(N-1)/2 .. t+(N-1)/2 stacked per coefficient     */
    int32_t fea_in;                  /* 1 = -format_in htk: the input is a feature matrix, not PCM           */
    int32_t nfeacoefs;               /* -nfeacoefs: floats per input feature row                             */
    /* -fea_kind td-iir-mfcc (src/io/in.cc:242-262, 281-340): coefficient file of the 24 time-domain IIR band filters, one
     * filter per line, ten TAB-separated numbers (b0..b4, input gain, a1..a4); read by ctu_create like rawIN::loadf_filters */
    char    filters[CTU_FBDEF];
    float   weight_of_td_iir_mfcc_bank;   /* float like the reference (src/io/opts.h:164), default 2.026          */
} ctu_config;

typedef struct ctu_handle ctu_handle;
typedef struct ctu_plan ctu_plan;

/* ---- configuration (replaces opts::opts / set_preset / parse / check_config) ---------- */
int ctu_config_init(ctu_config *cfg);                         /* defaults, src/io/opts.cc:34-146   */
int ctu_config_sizeof(void);                                  /* sizeof(ctu_config) of this build: lets a binding check its mirror */
/* One option exactly as opts::parse takes it (src/io/opts.cc:644-846): `value` may be NULL.
 * Options outside the hot path (-S -i -o -C -v ... -format_in -endian_*) are accepted and
 * ignored here; the host CLI owns them.  Unknown option -> CTU_ERR_CONFIG.               */
int ctu_config_set(ctu_config *cfg, const char *option, const char *value);
/* argv-style list with the reference's rule that a token starting with '-' is never a
 * value (src/io/opts.cc:185-192); then ctu_config_finalize.                              */
int ctu_config_parse(ctu_config *cfg, int argc, const char *const *argv);
int ctu_config_finalize(ctu_config *cfg);
const char *ctu_config_error(void);                           /* message of the last config error (thread local) */

/* ---- handle: designs the filter bank and all tables in fp64 on the host, uploads them -- */
int ctu_create(const ctu_config *cfg, int device, ctu_handle **out);
void ctu_destroy(ctu_handle *h);
const char *ctu_last_error(const ctu_handle *h);              /* h may be NULL: error of a failed ctu_create */

/* Host-only filter-bank design in fp64 (FB::FB and helpers, src/fea/fb.cc:20-66, 100-457),
 * usable without a GPU: nb bands out; mat[nb*wfftby2] (caller sizes it for 999 bands at
 * most, or passes NULL to query nb), lo/hi = first / last tap of each band.              */
int ctu_design_filter_bank(const ctu_config *cfg, double *mat, int32_t *lo, int32_t *hi, int32_t *nb);

int ctu_feature_dim(const ctu_handle *h);      /* floats per output row, writer order (0 in waveform mode) */
int ctu_input_dim(const ctu_handle *h);        /* floats per INPUT row of a feature-input handle (-format_in htk), else 0 */
int ctu_is_signal_output(const ctu_handle *h); /* 1 when format_out is raw|wave                             */
int ctu_num_bands(const ctu_handle *h);        /* FB::size                                                  */
/* FB::mat as designed (src/fea/fb.cc:255-457): mat[nb*wfftby2] row-major, lo/hi[nb].     */
int ctu_fb_matrix(const ctu_handle *h, double *mat, int32_t *lo, int32_t *hi);
/* rawIN::new_file/get_frame framing (src/io/in.cc:264-279, 314): frames for an utterance
 * of n samples; -1 when the reference would throw "IO: Signal shorter than one frame!".  */
int64_t ctu_num_frames(const ctu_handle *h, int64_t nsamples);
int64_t ctu_num_output_samples(const ctu_handle *h, int64_t nsamples); /* T*s + (w-s)     */
uint64_t ctu_launch_count(const ctu_handle *h); /* CUDA kernels launched by this handle so far */

/* Per-kernel timing for the benchmark's roofline line: when enabled, every kernel this
 * handle launches is bracketed by CUDA events on its stream.  ctu_profile_get waits for
 * record idx and returns the kernel's name (static string) and duration.              */
int ctu_profile_enable(ctu_handle *h, int on);     /* also clears previous records      */
int ctu_profile_count(const ctu_handle *h);
int ctu_profile_get(ctu_handle *h, int idx, const char **name, float *ms);

/* ---- plan: a list of utterances (sample offsets into one concatenated PCM buffer; for a
 * feature-input handle, ROW offsets into one concatenated [rows x ctu_input_dim] matrix) ---- */
int ctu_plan_create(ctu_handle *h, const int64_t *utt_offsets /* n_utts+1 */, int32_t n_utts, ctu_plan **out);
void ctu_plan_destroy(ctu_plan *p);
int64_t ctu_plan_total_frames(const ctu_plan *p);   /* sum of T_u                                 */
int64_t ctu_plan_max_rows(const ctu_plan *p);       /* rows the feature buffer must hold (= total frames) */
int64_t ctu_plan_total_output_samples(const ctu_plan *p);
int ctu_plan_frames_per_utt(const ctu_plan *p, int64_t *frames /* n_utts */);
int64_t ctu_plan_workspace_bytes(const ctu_plan *p);

/* What one run produced, per utterance (host arrays owned by the plan, valid until the
 * next run): rows written for utterance u (differs from frames only with -vad_apply_mode
 * drop) and its first row in the output matrix.                                          */
int ctu_plan_rows_per_utt(const ctu_plan *p, int64_t *rows /* n_utts */);

/* Device-resident run: every pointer is a DEVICE pointer, work is enqueued on `stream`
 * (a cudaStream_t passed as void*) and not synchronised.  Outputs that do not apply may
 * be NULL.  ext_vad: one byte per frame in list order, any non-zero byte = speech
 * (src/nr/nr.cc:297-302) -- only for vadmode "file".
 *   features : float32 [max_rows x feature_dim]  writer column order
 *   waveform : int16   [total_output_samples]    (signal output)
 *   vad_nr   : uint8   [total_frames]            decisions of the NR-internal detector
 *   vad_out  : uint8   [total_frames]            VAD-module decisions after the median filter
 * With -vad_apply_mode drop the kept rows are compacted per utterance and
 * ctu_plan_rows_per_utt reports the counts (this call then synchronises the stream).   */
int ctu_plan_run_device(ctu_plan *p, const int16_t *d_pcm, const uint8_t *d_ext_vad, float *d_features,
                        int16_t *d_waveform, uint8_t *d_vad_nr, uint8_t *d_vad_out, void *stream);

/* End-to-end run with HOST buffers: H2D, kernels and D2H are pipelined over chunks of
 * utterances on internal streams; returns when the outputs are complete.               */
int ctu_plan_run_host(ctu_plan *p, const int16_t *pcm, const uint8_t *ext_vad, float *features,
                      int16_t *waveform, uint8_t *vad_nr, uint8_t *vad_out);

/* Feature-file input (-format_in htk; htkIN::get_frame src/io/in.cc:682-690 -> deltaFEA src/fea/fea_delta.cc:70-206
 * -> cms_POST src/fea/post_impl.cc:203-209 -> htkOUT::save_frame src/io/out.cc:177-179): rows of ctu_input_dim()
 * floats in, rows of ctu_feature_dim() floats out (file column order, no reordering).  Device / host variants as
 * above; `keep` leaves the result on the device for ctu_plan_colsums / _normalise / _fetch.                       */
int ctu_plan_run_device_fea(ctu_plan *p, const float *d_fea_in, float *d_features, void *stream);
int ctu_plan_run_host_fea(ctu_plan *p, const float *fea_in, float *features /* NULL = keep on the device */);

/* G.711 input (-format_in alaw | mulaw; rawIN::loadframe + alaw2lin, src/io/in.cc:470-500, src/io/amulaw.h): the caller
 * hands over the 8-bit codes as they are in the file and the expansion to 16-bit PCM runs on the device, so only ONE byte
 * per sample crosses PCIe (the end-to-end rate of this path is bound by the host-to-device copy).  Offsets of the plan
 * count samples = bytes.  ctu_g711_table gives the 256 expansion values (law: 1 = A-law, 0 = mu-law) for hosts that
 * decode themselves.                                                                                                   */
int ctu_g711_table(int alaw, int16_t *table /* 256 */);
int ctu_plan_run_host_g711(ctu_plan *p, const uint8_t *codes, int alaw, const uint8_t *ext_vad, float *features,
                           int16_t *waveform, uint8_t *vad_nr, uint8_t *vad_out);

/* The same in steps, for callers that post-process on the device before fetching: run with the results
 * left on the device, [ctu_plan_colsums / ctu_plan_normalise], then ctu_plan_fetch.                  */
int ctu_plan_run_host_keep(ctu_plan *p, const int16_t *pcm, const uint8_t *ext_vad);
int ctu_plan_fetch(ctu_plan *p, float *features, int16_t *waveform, uint8_t *vad_nr, uint8_t *vad_out);

/* CMVN, device half (cmvn_POST::sum_fea / sum_cv / process_frame, src/fea/post_impl.cc:52-118), on the
 * feature rows ctu_plan_run_host_keep left on the device.  dim = ctu_cmvn_dim(): the row without the _E
 * column, in WRITER column order.  Arrays are host arrays [n_utts x dim].
 *   ctu_plan_colsums  : sums[u][c] = sum over the rows of utterance u of F[c]            (center == NULL)
 *                                  = sum of (F[c] - center[u][c])^2                      (center != NULL)
 *   ctu_plan_normalise: F[c] = (F[c] - mean[u][c]) / scale[u][c]   (the reference divides by the VARIANCE)
 * The host groups utterances by speaker and owns the statistics file (src/io/out.cc:591-615).          */
int ctu_cmvn_dim(const ctu_handle *h);
int ctu_plan_colsums(ctu_plan *p, const double *center, double *sums);
int ctu_plan_normalise(ctu_plan *p, const double *mean, const double *scale);

/* Convenience: plan + run_host + destroy.  frames_per_utt/rows_per_utt may be NULL.     */
int ctu_run(ctu_handle *h, const int16_t *pcm, const int64_t *utt_offsets, int32_t n_utts, const uint8_t *ext_vad,
            float *features, int64_t features_capacity_rows, int16_t *waveform, int64_t waveform_capacity,
            uint8_t *vad_nr, uint8_t *vad_out, int64_t *frames_per_utt, int64_t *rows_per_utt);

/* -dither draws one value of the process-wide glibc rand() stream (srand(1), src/io/in.cc:205, 452-455) per loaded
 * sample, in list order.  A handle continues the stream from plan to plan like the reference process does from file to
 * file; a shard that starts in the middle of a list sets how many values the files before it have drawn
 * ((window - wshift) + frames * wshift per file).                                                                  */
int ctu_set_rand_offset(ctu_handle *h, uint64_t values_drawn);

/* Container rows formatted on the device (SURVEY 8f.1): what the reference's writers do value by value on the host.
 *   CTU_ROWS_NATIVE  float32 rows in host byte order (default)
 *   CTU_ROWS_BE      byte-swapped float32 rows: HTK -endian_out big (src/io/out.cc:189-213)
 *   CTU_ROWS_PFILE   pfile rows (src/io/pfile.cc:470-539): big-endian u32 sentence, u32 frame, float32 x dim; the sentence
 *                    number of the plan's first utterance is first_sentence, frames count from 0 per utterance (rows kept
 *                    by -vad_apply_mode drop are numbered as written)
 * Applies to the `features` buffer of ctu_plan_run_host / _run_host_g711, which must then hold ctu_plan_max_rows() x
 * ctu_plan_row_bytes() bytes; row r of utterance u starts at byte (first row of u + r) x row_bytes.                    */
#define CTU_ROWS_NATIVE 0
#define CTU_ROWS_BE 1
#define CTU_ROWS_PFILE 2
int ctu_plan_set_row_format(ctu_plan *p, int format, uint32_t first_sentence);
int64_t ctu_plan_row_bytes(const ctu_plan *p);

/* -vad_out_mode debug (FileWriter and the save_frame members of the criterion / threshold classes, src/vad/vad.h:39-76,
 * src/vad/vad.cc:91-111, 212-286, 324-335, 375-404, 456-508, 565-634): the values behind the reference's side files
 * <vadfile>_vad0, _energy | _cepdist (+ _c0init), _thr and the threshold's own files.  Per VAD step of every utterance
 * (= per frame, list order) CTU_VAD_DEBUG_COLS doubles -- criterion, threshold, then the threshold's state: perc crimin,
 * crimax, -; adapt crimean, crimean2, crivar; dyn dmin, dmax, dyn; absolute -, -, - -- and the unfiltered decision vad0.
 * The reference writes a row once the majority filter has decided it, AFTER the state has advanced: row i of a side file
 * holds step min(i + (vad_filter_order - 1) / 2, T - 1) (the rows written by the flush repeat the last step), and its
 * *init flag files compare that step + 1 with the init length.  Valid after a run of this plan; needs a handle created
 * with -vad_out_mode debug.                                                                                          */
#define CTU_VAD_DEBUG_COLS 5
int ctu_plan_fetch_vad_debug(ctu_plan *p, double *steps /* [total_frames x CTU_VAD_DEBUG_COLS] */, uint8_t *vad0 /* [total_frames] */);

/* Run-time knobs that are not reference options (the reference has no counterpart: it has one code path):
 *   "copy_only"      1 = the host entry points do their H2D / D2H copies with the kernels left out: the control
 *                        measurement behind bench.py's e2e.copy_only_ms
 *   "chunk_mb"       MB of PCM per pipeline chunk of the host entry points (default 32)
 * Unknown name -> CTU_ERR_CONFIG.                                                                                  */
int ctu_set_option(ctu_handle *h, const char *name, int64_t value);

/* Page-locked host memory for the buffers handed to ctu_plan_run_host / ctu_run: pageable memory
 * makes every chunk copy synchronous and several times slower.  (What rawIN's fread buffer and the
 * writers' obuffer are to the reference, src/io/in.cc:434-460, src/io/out.cc:95-106.)            */
int ctu_host_alloc(void **ptr, uint64_t bytes);
int ctu_device_count(void);                      /* CUDA devices visible to this process (0 = none: nothing can run)  */
void ctu_host_free(void *ptr);

/* Debug / test taps (device-resident, synchronous): intermediate stages of one plan run. */
int ctu_debug_spectrum(ctu_plan *p, const int16_t *d_pcm, float *d_spec /* [frames x wfftby2] */, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* CTUCOPY_B200_H */
