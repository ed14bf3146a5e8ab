"""ctypes binding of include/ctucopy_b200.h.

Mirrors the reference's surface for this path: option strings go in exactly as on the
`ctucopy` command line (opts::parse, src/io/opts.cc:644-846), a list of utterances goes
through the chain BATCH builds (src/io/batch.cc:24-69) and per-utterance feature matrices
(writer column order) or enhanced waveforms come out.  All compute happens in
libctucopy_b200.so on the GPU; this module fails loudly when the library is missing.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

CTU_STR = 40
CTU_FBDEF = 1024
ABI_VERSION = 4


class CtuError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__("ctucopy_b200 status %d: %s" % (status, message))
        self.status = status
        self.message = message


class Config(C.Structure):
    """struct ctu_config (include/ctucopy_b200.h) == hot-path subset of `class opts`."""
    _fields_ = [
        ("abi_version", C.c_int32),
        ("format_out", C.c_char * CTU_STR),
        ("fs", C.c_int32),
        ("preem", C.c_float),
        ("dither", C.c_double),
        ("remove_dc", C.c_int32), ("remove_dc1", C.c_int32),
        ("window_ms", C.c_double), ("wshift_ms", C.c_double),
        ("fb_scale", C.c_char * CTU_STR), ("fb_shape", C.c_char * CTU_STR),
        ("fb_norm", C.c_int32), ("fb_power", C.c_int32), ("fb_eqld", C.c_int32), ("fb_inld", C.c_int32),
        ("fb_definition", C.c_char * CTU_FBDEF),
        ("vadmode", C.c_char * CTU_STR),
        ("nr_mode", C.c_char * CTU_STR),
        ("nr_p", C.c_double), ("nr_q", C.c_double), ("nr_a", C.c_double), ("nr_b", C.c_double),
        ("nr_initsegs", C.c_int32),
        ("nr_when", C.c_int32),
        ("fea_kind", C.c_char * CTU_STR),
        ("fea_lporder", C.c_int32), ("fea_ncepcoefs", C.c_int32), ("fea_c0", C.c_int32), ("fea_E", C.c_int32),
        ("fea_rawenergy", C.c_int32), ("fea_lifter", C.c_int32),
        ("fea_trapdct_traplen", C.c_int32), ("fea_trapdct_ndct", C.c_int32),
        ("fea_delta", C.c_int32), ("n_order", C.c_int32), ("d_win", C.c_int32), ("a_win", C.c_int32), ("t_win", C.c_int32),
        ("vad_apply_mode", C.c_char * CTU_STR), ("vad_out_mode", C.c_char * CTU_STR),
        ("vad_cri_mode", C.c_char * CTU_STR), ("vad_thr_mode", C.c_char * CTU_STR),
        ("vad_energy_db", C.c_int32),
        ("vad_cepdist_mode", C.c_char * CTU_STR),
        ("vad_cepdist_p", C.c_double),
        ("vad_cepdist_init", C.c_int32), ("vad_lpc_coefs", C.c_int32),
        ("vad_absolute_thr", C.c_double),
        ("vad_perc_init", C.c_int32),
        ("vad_perc_thr", C.c_double),
        ("vad_adapt_init", C.c_int32),
        ("vad_adapt_q", C.c_double), ("vad_adapt_za", C.c_double),
        ("vad_dyn_init", C.c_int32),
        ("vad_dyn_perc", C.c_double), ("vad_dyn_min", C.c_double), ("vad_dyn_qmaxinc", C.c_double),
        ("vad_dyn_qmaxdec", C.c_double), ("vad_dyn_qmindec", C.c_double), ("vad_dyn_qmininc", C.c_double),
        ("vad_filter_order", C.c_int32),
        ("window", C.c_int32), ("wshift", C.c_int32), ("wfft", C.c_int32), ("wfftby2", C.c_int32), ("phase_needed", C.c_int32),
        ("fea_Z_exp", C.c_float), ("fea_Z_block", C.c_float), ("cms_exp_coef", C.c_float),
        ("stat_cmvn", C.c_int32), ("apply_cmvn", C.c_int32),
        ("fea_trap", C.c_int32), ("trap_win", C.c_int32), ("fea_in", C.c_int32), ("nfeacoefs", C.c_int32),
        ("filters", C.c_char * 1024), ("weight_of_td_iir_mfcc_bank", C.c_float),
    ]


def lib_path() -> str:
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "libctucopy_b200.so")


_lib = None


def lib() -> C.CDLL:
    """Loads libctucopy_b200.so (built in-tree by __graft_entry__.build() / csrc/Makefile)."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise ImportError("%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no Python/CPU fallback for the CtuCopy hot path)" % p)
    L = C.CDLL(p)
    vp, i32, i64, cp = C.c_void_p, C.c_int32, C.c_int64, C.c_char_p
    P = C.POINTER
    L.ctu_config_sizeof.argtypes = []; L.ctu_config_sizeof.restype = C.c_int
    if L.ctu_config_sizeof() != C.sizeof(Config):
        raise ImportError("ctucopy_b200.api.Config (%d bytes) does not mirror struct ctu_config of %s (%d bytes)" % (C.sizeof(Config), p, L.ctu_config_sizeof()))
    L.ctu_config_init.argtypes = [P(Config)]; L.ctu_config_init.restype = C.c_int
    L.ctu_config_set.argtypes = [P(Config), cp, cp]; L.ctu_config_set.restype = C.c_int
    L.ctu_config_parse.argtypes = [P(Config), C.c_int, P(cp)]; L.ctu_config_parse.restype = C.c_int
    L.ctu_config_finalize.argtypes = [P(Config)]; L.ctu_config_finalize.restype = C.c_int
    L.ctu_config_error.argtypes = []; L.ctu_config_error.restype = cp
    L.ctu_create.argtypes = [P(Config), C.c_int, P(vp)]; L.ctu_create.restype = C.c_int
    L.ctu_destroy.argtypes = [vp]; L.ctu_destroy.restype = None
    L.ctu_last_error.argtypes = [vp]; L.ctu_last_error.restype = cp
    L.ctu_design_filter_bank.argtypes = [P(Config), vp, vp, vp, P(i32)]; L.ctu_design_filter_bank.restype = C.c_int
    L.ctu_feature_dim.argtypes = [vp]; L.ctu_feature_dim.restype = C.c_int
    L.ctu_input_dim.argtypes = [vp]; L.ctu_input_dim.restype = C.c_int
    L.ctu_plan_run_device_fea.argtypes = [vp, vp, vp, vp]; L.ctu_plan_run_device_fea.restype = C.c_int
    L.ctu_plan_run_host_fea.argtypes = [vp, vp, vp]; L.ctu_plan_run_host_fea.restype = C.c_int
    L.ctu_g711_table.argtypes = [C.c_int, vp]; L.ctu_g711_table.restype = C.c_int
    L.ctu_plan_run_host_g711.argtypes = [vp, vp, C.c_int, vp, vp, vp, vp, vp]; L.ctu_plan_run_host_g711.restype = C.c_int
    L.ctu_is_signal_output.argtypes = [vp]; L.ctu_is_signal_output.restype = C.c_int
    L.ctu_num_bands.argtypes = [vp]; L.ctu_num_bands.restype = C.c_int
    L.ctu_fb_matrix.argtypes = [vp, vp, vp, vp]; L.ctu_fb_matrix.restype = C.c_int
    L.ctu_num_frames.argtypes = [vp, i64]; L.ctu_num_frames.restype = i64
    L.ctu_num_output_samples.argtypes = [vp, i64]; L.ctu_num_output_samples.restype = i64
    L.ctu_launch_count.argtypes = [vp]; L.ctu_launch_count.restype = C.c_uint64
    L.ctu_profile_enable.argtypes = [vp, C.c_int]; L.ctu_profile_enable.restype = C.c_int
    L.ctu_profile_count.argtypes = [vp]; L.ctu_profile_count.restype = C.c_int
    L.ctu_profile_get.argtypes = [vp, C.c_int, P(cp), P(C.c_float)]; L.ctu_profile_get.restype = C.c_int
    L.ctu_plan_create.argtypes = [vp, vp, i32, P(vp)]; L.ctu_plan_create.restype = C.c_int
    L.ctu_plan_destroy.argtypes = [vp]; L.ctu_plan_destroy.restype = None
    for f in ("ctu_plan_total_frames", "ctu_plan_max_rows", "ctu_plan_total_output_samples", "ctu_plan_workspace_bytes"):
        getattr(L, f).argtypes = [vp]; getattr(L, f).restype = i64
    L.ctu_plan_frames_per_utt.argtypes = [vp, vp]; L.ctu_plan_frames_per_utt.restype = C.c_int
    L.ctu_plan_rows_per_utt.argtypes = [vp, vp]; L.ctu_plan_rows_per_utt.restype = C.c_int
    L.ctu_plan_run_device.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]; L.ctu_plan_run_device.restype = C.c_int
    L.ctu_plan_run_host.argtypes = [vp, vp, vp, vp, vp, vp, vp]; L.ctu_plan_run_host.restype = C.c_int
    L.ctu_run.argtypes = [vp, vp, vp, i32, vp, vp, i64, vp, i64, vp, vp, vp, vp]; L.ctu_run.restype = C.c_int
    L.ctu_debug_spectrum.argtypes = [vp, vp, vp, vp]; L.ctu_debug_spectrum.restype = C.c_int
    L.ctu_plan_run_host_keep.argtypes = [vp, vp, vp]; L.ctu_plan_run_host_keep.restype = C.c_int
    L.ctu_plan_fetch.argtypes = [vp, vp, vp, vp, vp]; L.ctu_plan_fetch.restype = C.c_int
    L.ctu_cmvn_dim.argtypes = [vp]; L.ctu_cmvn_dim.restype = C.c_int
    L.ctu_plan_colsums.argtypes = [vp, vp, vp]; L.ctu_plan_colsums.restype = C.c_int
    L.ctu_plan_normalise.argtypes = [vp, vp, vp]; L.ctu_plan_normalise.restype = C.c_int
    L.ctu_set_rand_offset.argtypes = [vp, C.c_uint64]; L.ctu_set_rand_offset.restype = C.c_int
    L.ctu_set_option.argtypes = [vp, cp, i64]; L.ctu_set_option.restype = C.c_int
    L.ctu_plan_fetch_vad_debug.argtypes = [vp, vp, vp]; L.ctu_plan_fetch_vad_debug.restype = C.c_int
    L.ctu_host_alloc.argtypes = [P(vp), C.c_uint64]; L.ctu_host_alloc.restype = C.c_int
    L.ctu_host_free.argtypes = [vp]; L.ctu_host_free.restype = None
    _lib = L
    return L


def parse_config(argv: Sequence[str]) -> Config:
    """ctu_config_init + ctu_config_parse: same option strings as the reference's CLI."""
    L = lib()
    cfg = Config()
    L.ctu_config_init(C.byref(cfg))
    arr = (C.c_char_p * len(argv))(*[a.encode() for a in argv])
    st = L.ctu_config_parse(C.byref(cfg), len(argv), arr)
    if st:
        raise CtuError(st, L.ctu_config_error().decode())
    return cfg


def design_filter_bank(cfg: Config):
    """Host-only fp64 filter-bank design (no GPU needed): (mat [nb, bins], lo, hi)."""
    L = lib()
    nb = C.c_int32(0)
    st = L.ctu_design_filter_bank(C.byref(cfg), None, None, None, C.byref(nb))
    if st:
        raise CtuError(st, L.ctu_last_error(None).decode())
    mat = np.zeros((nb.value, cfg.wfftby2), dtype=np.float64)
    lo = np.zeros(nb.value, dtype=np.int32)
    hi = np.zeros(nb.value, dtype=np.int32)
    L.ctu_design_filter_bank(C.byref(cfg), mat.ctypes.data, lo.ctypes.data, hi.ctypes.data, C.byref(nb))
    return mat, lo, hi


def _ptr(a) -> Optional[int]:
    if a is None:
        return None
    if isinstance(a, int):
        return a
    return a.ctypes.data


@dataclass
class Result:
    frames_per_utt: np.ndarray
    rows_per_utt: np.ndarray
    row_offsets: np.ndarray                 # first row of each utterance in `features`
    features: Optional[np.ndarray] = None   # float32 [total_frames, dim]
    waveform: Optional[np.ndarray] = None   # int16 [total_output_samples]
    wave_offsets: Optional[np.ndarray] = None
    vad_nr: Optional[np.ndarray] = None
    vad_out: Optional[np.ndarray] = None

    def utt_features(self, u: int) -> np.ndarray:
        r0 = int(self.row_offsets[u])
        return self.features[r0: r0 + int(self.rows_per_utt[u])]

    def utt_waveform(self, u: int) -> np.ndarray:
        return self.waveform[int(self.wave_offsets[u]): int(self.wave_offsets[u + 1])]


class Handle:
    def __init__(self, cfg_or_argv, device: int = 0):
        self.L = lib()
        self.cfg = cfg_or_argv if isinstance(cfg_or_argv, Config) else parse_config(list(cfg_or_argv))
        h = C.c_void_p()
        st = self.L.ctu_create(C.byref(self.cfg), device, C.byref(h))
        if st:
            raise CtuError(st, self.L.ctu_last_error(None).decode())
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.L.ctu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st: int):
        if st:
            raise CtuError(st, self.L.ctu_last_error(self.h).decode())

    @property
    def feature_dim(self) -> int:
        return self.L.ctu_feature_dim(self.h)

    @property
    def signal_output(self) -> bool:
        return bool(self.L.ctu_is_signal_output(self.h))

    @property
    def num_bands(self) -> int:
        return int(self.L.ctu_num_bands(self.h))

    @property
    def launch_count(self) -> int:
        return int(self.L.ctu_launch_count(self.h))

    def set_option(self, name: str, value: int):
        """Run-time knobs outside the reference's option set (ctu_set_option): copy_only, chunk_mb."""
        self._check(self.L.ctu_set_option(self.h, name.encode(), int(value)))

    def profile(self, on: bool):
        self._check(self.L.ctu_profile_enable(self.h, 1 if on else 0))

    def profile_records(self):
        """[(kernel name, milliseconds)] for every launch since profile(True)."""
        out = []
        for i in range(self.L.ctu_profile_count(self.h)):
            name = C.c_char_p(); ms = C.c_float()
            self._check(self.L.ctu_profile_get(self.h, i, C.byref(name), C.byref(ms)))
            out.append((name.value.decode(), float(ms.value)))
        return out

    def num_frames(self, nsamples: int) -> int:
        return int(self.L.ctu_num_frames(self.h, nsamples))

    def fb_matrix(self):
        nb = self.L.ctu_num_bands(self.h)
        mat = np.zeros((nb, self.cfg.wfftby2)); lo = np.zeros(nb, np.int32); hi = np.zeros(nb, np.int32)
        self._check(self.L.ctu_fb_matrix(self.h, mat.ctypes.data, lo.ctypes.data, hi.ctypes.data))
        return mat, lo, hi

    @property
    def input_dim(self) -> int:
        return int(self.L.ctu_input_dim(self.h))

    def plan(self, lengths: Sequence[int]) -> "Plan":
        return Plan(self, lengths)


class Plan:
    """A list of utterances laid end to end in one PCM buffer (ctu_plan)."""

    def __init__(self, handle: Handle, lengths: Sequence[int]):
        self.hd = handle
        self.L = handle.L
        self.lengths = np.asarray(lengths, dtype=np.int64)
        self.offsets = np.concatenate([[0], np.cumsum(self.lengths)]).astype(np.int64)
        p = C.c_void_p()
        handle._check(self.L.ctu_plan_create(handle.h, self.offsets.ctypes.data, len(self.lengths), C.byref(p)))
        self.p = p
        n = len(self.lengths)
        self.frames_per_utt = np.zeros(n, dtype=np.int64)
        self.L.ctu_plan_frames_per_utt(self.p, self.frames_per_utt.ctypes.data)
        self.row_offsets = np.concatenate([[0], np.cumsum(self.frames_per_utt)]).astype(np.int64)
        self.total_frames = int(self.L.ctu_plan_total_frames(self.p))
        self.total_output_samples = int(self.L.ctu_plan_total_output_samples(self.p))
        w, s = handle.cfg.window, handle.cfg.wshift
        self.wave_offsets = np.concatenate([[0], np.cumsum(self.frames_per_utt * s + (w - s))]).astype(np.int64)

    def close(self):
        if getattr(self, "p", None):
            self.L.ctu_plan_destroy(self.p)
            self.p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def workspace_bytes(self) -> int:
        return int(self.L.ctu_plan_workspace_bytes(self.p))

    def rows_per_utt(self) -> np.ndarray:
        r = np.zeros(len(self.lengths), dtype=np.int64)
        self.L.ctu_plan_rows_per_utt(self.p, r.ctypes.data)
        return r

    def fetch_vad_debug(self):
        """-vad_out_mode debug: (steps float64 [total_frames, 5], vad0 uint8 [total_frames]) of the last run
        (ctu_plan_fetch_vad_debug); vad_debug_files() turns one utterance's slice into the reference's side files."""
        steps = np.zeros((self.total_frames, 5), dtype=np.float64)
        vad0 = np.zeros(self.total_frames, dtype=np.uint8)
        self.hd._check(self.L.ctu_plan_fetch_vad_debug(self.p, steps.ctypes.data, vad0.ctypes.data))
        return steps, vad0

    def run_device(self, d_pcm: int, d_features: Optional[int] = None, d_waveform: Optional[int] = None,
                   d_ext_vad: Optional[int] = None, d_vad_nr: Optional[int] = None, d_vad_out: Optional[int] = None,
                   stream: int = 0):
        """All arguments are raw device addresses (e.g. torch.Tensor.data_ptr()); enqueues on `stream`."""
        self.hd._check(self.L.ctu_plan_run_device(self.p, d_pcm, d_ext_vad, d_features, d_waveform, d_vad_nr, d_vad_out, stream))

    def run_host_fea(self, fea_in: np.ndarray, *, features: Optional[np.ndarray] = None) -> Result:
        """Feature-file input (-format_in htk): rows of Handle.input_dim floats in, rows of feature_dim floats out."""
        hd = self.hd
        assert fea_in.dtype == np.float32 and fea_in.flags.c_contiguous and fea_in.shape == (int(self.offsets[-1]), hd.input_dim)
        if features is None:
            features = np.empty((self.total_frames, hd.feature_dim), dtype=np.float32)
        hd._check(self.L.ctu_plan_run_host_fea(self.p, _ptr(fea_in), _ptr(features)))
        return Result(self.frames_per_utt.copy(), self.rows_per_utt(), self.row_offsets, features)

    def run_device_fea(self, d_fea_in: int, d_features: int, stream: int = 0):
        self.hd._check(self.L.ctu_plan_run_device_fea(self.p, d_fea_in, d_features, stream))

    def run_host(self, pcm: np.ndarray, ext_vad: Optional[np.ndarray] = None, *, features: Optional[np.ndarray] = None,
                 waveform: Optional[np.ndarray] = None, want_vad: bool = True, g711: Optional[str] = None) -> Result:
        """End to end with host buffers (numpy, ideally pinned): H2D + kernels + D2H.  g711 = "alaw" | "mulaw": `pcm` holds
        the 8-bit codes of the files, expanded on the device (ctu_plan_run_host_g711)."""
        hd = self.hd
        assert pcm.dtype == (np.uint8 if g711 else np.int16) and pcm.flags.c_contiguous and len(pcm) == int(self.offsets[-1])
        dim = hd.feature_dim
        if hd.signal_output:
            if waveform is None:
                waveform = np.empty(self.total_output_samples, dtype=np.int16)
        elif features is None:
            features = np.empty((self.total_frames, dim), dtype=np.float32)
        vnr = np.zeros(self.total_frames, dtype=np.uint8) if want_vad else None
        vout = np.zeros(self.total_frames, dtype=np.uint8) if want_vad else None
        if ext_vad is not None:
            ext_vad = np.ascontiguousarray(ext_vad, dtype=np.uint8)
            assert len(ext_vad) == self.total_frames
        if g711:
            hd._check(self.L.ctu_plan_run_host_g711(self.p, _ptr(pcm), 1 if g711 == "alaw" else 0, _ptr(ext_vad), _ptr(features), _ptr(waveform),
                                                    _ptr(vnr), _ptr(vout)))
        else:
            hd._check(self.L.ctu_plan_run_host(self.p, _ptr(pcm), _ptr(ext_vad), _ptr(features), _ptr(waveform), _ptr(vnr), _ptr(vout)))
        return Result(self.frames_per_utt.copy(), self.rows_per_utt(), self.row_offsets, features, waveform, self.wave_offsets, vnr, vout)


def extract(argv: Sequence[str], utterances: List[np.ndarray], ext_vad: Optional[List[np.ndarray]] = None, device: int = 0,
            options: Optional[dict] = None) -> Result:
    """One-call convenience used by the parity tests: what `ctucopy <argv> -S list` computes
    for the listed utterances (each processed as its own file).  options: run-time knobs (Handle.set_option)."""
    hd = Handle(argv, device)
    try:
        for k, v in (options or {}).items():
            hd.set_option(k, v)
        plan = hd.plan([len(u) for u in utterances])
        try:
            pcm = np.ascontiguousarray(np.concatenate(utterances).astype(np.int16)) if utterances else np.zeros(0, np.int16)
            ev = np.concatenate(ext_vad).astype(np.uint8) if ext_vad is not None else None
            return plan.run_host(pcm, ev)
        finally:
            plan.close()
    finally:
        hd.close()


def vad_debug_files(cfg: Config, steps: np.ndarray, vad0: np.ndarray) -> dict:
    """The side files `-vad_out_mode debug` writes next to <vadfile> for ONE utterance, suffix -> bytes (native doubles, or
    '0' / '1' characters), from that utterance's rows of Plan.fetch_vad_debug().  Same rule as host/ctucopy_main.cc: row i
    holds VAD step min(i + (vad_filter_order - 1) / 2, T - 1) (VAD::save_frame runs after the state has advanced and the
    flush rows repeat the last step, src/vad/vad.cc:710-725, src/io/batch.cc:243-249)."""
    T = len(vad0)
    h = (cfg.vad_filter_order - 1) // 2
    if T <= h:
        return {}
    step = np.minimum(np.arange(T) + h, T - 1)
    ch = lambda b: np.where(b, ord("1"), ord("0")).astype(np.uint8).tobytes()
    col = lambda k: np.ascontiguousarray(steps[step, k], dtype="<f8").tobytes()
    out = {"vad0": ch(vad0[step] != 0)}
    if cfg.vad_cri_mode.decode() == "energy":
        out["energy"] = col(0)
    else:
        out["cepdist"] = col(0)
        out["c0init"] = ch((step + 1) <= cfg.vad_cepdist_init)
    m = cfg.vad_thr_mode.decode()
    if m == "absolute":
        out["thr"] = np.full(T, cfg.vad_absolute_thr, dtype="<f8").tobytes()
    elif m == "perc":
        out.update(crimin=col(2), crimax=col(3), thr=col(1))
    elif m == "adapt":
        out.update(init=ch((step + 1) <= cfg.vad_adapt_init), crimean=col(2), crimean2=col(3), crivar=col(4), thr=col(1))
    else:
        out.update(dmin=col(2), dmax=col(3), dyn=col(4), dynmin=np.full(T, cfg.vad_dyn_min, dtype="<f8").tobytes(), thr=col(1))
    return out


def g711_table(alaw: bool) -> np.ndarray:
    """The 256 expansion values the library uses (host-only call, no GPU needed)."""
    t = np.zeros(256, dtype=np.int16)
    lib().ctu_g711_table(1 if alaw else 0, t.ctypes.data)
    return t


def extract_g711(argv: Sequence[str], code_streams: List[np.ndarray], alaw: bool, device: int = 0) -> Result:
    """`ctucopy -format_in alaw|mulaw <argv> -S list`: the 8-bit codes go to the GPU as they are."""
    hd = Handle(argv, device)
    try:
        plan = hd.plan([len(u) for u in code_streams])
        try:
            return plan.run_host(np.ascontiguousarray(np.concatenate(code_streams).astype(np.uint8)), g711="alaw" if alaw else "mulaw")
        finally:
            plan.close()
    finally:
        hd.close()


def extract_features(argv: Sequence[str], matrices: List[np.ndarray], device: int = 0) -> Result:
    """`ctucopy -format_in htk <argv> -S list` for the listed feature matrices (each its own file): deltas, context
    stacking, CMS on existing features.  Every matrix must have Handle.input_dim (= -nfeacoefs) columns."""
    hd = Handle(argv, device)
    try:
        plan = hd.plan([m.shape[0] for m in matrices])
        try:
            x = np.ascontiguousarray(np.concatenate(matrices, axis=0).astype(np.float32))
            return plan.run_host_fea(x)
        finally:
            plan.close()
    finally:
        hd.close()
