"""-remove_dc1 (the reference's ring that is de-meaned on every frame, src/io/in.cc:343-350) on the chains that build the frame
again in fp64: waveform output (k_synth_frames_any), the Burg detector and the VAD module's cepdist/lpc criterion (k_burg_any),
the fp64 feature path (k_frames64_any), and -fea_rawenergy (k_rawenergy).

Every input carries a DC bias (+-2500, a slow ramp, a signal close to clipping), and for every case the oracle's output with
-remove_dc1 on differs from its output with the option off by more than the bar the library is held to: a library that ignored
the option would fail."""
import os
import subprocess

import numpy as np
import pytest

import ctu_oracle as co
import golden_util as gu
import ctucopy_b200 as cb
import test_gpu_parity as tp
from ctucopy_b200 import synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "host", "ctucopy_b200")
DC1 = ["-remove_dc1", "on"]


def biased(u, kind):
    x = np.asarray(u, dtype=np.float64)
    if kind == "plus":
        x = x + 2500.0
    elif kind == "minus":
        x = x - 2500.0
    elif kind == "ramp":
        x = x + np.linspace(-4000.0, 4000.0, len(x))
    elif kind == "clip":
        x = x * (29000.0 / max(1.0, float(np.abs(x).max()))) + 3500.0
    return np.clip(np.round(x), -32768, 32767).astype(np.int16)


def signals(fs):
    if fs == 16000:
        ins = gu.inputs()
        base = [ins[0], ins[1], ins[4], ins[5]]
    else:
        base = [synthetic.utterance(k, sec, fs) for k, sec in ((0, 1.0), (1, 1.0), (2, 2.0), (7, 1.0))]
    return [biased(b, k) for b, k in zip(base, ("plus", "minus", "ramp", "clip"))]


def raw(fs):
    return ["-fs", str(fs), "-format_in", "raw", "-dither", "0"]


MF = ["-preset", "mfcc", "-preem", "0.97"]
BENCH_FWSS_BURG = ["-preset", "mfcc", "-preem", "0.97", "-nr_mode", "fwss", "-vad", "burg", "-nr_when", "beforeFB", "-format_out", "pfile=out.pfile"]
# name: (fs, args without -remove_dc1, external VAD stream)
CASES = {
    # waveforms: 512 / 256 / 2048 points, and 353 samples (odd) at 11.025 kHz / 32 ms
    "exten_raw_16k": (16000, ["-preset", "exten", "-format_out", "raw"], False),
    "exten_raw_8k": (8000, ["-preset", "exten", "-format_out", "raw"], False),
    "exten_wave_44k": (44100, ["-preset", "exten", "-format_out", "wave"], False),
    "exten_raw_11k_w32": (11025, ["-preset", "exten", "-w", "32", "-s", "16", "-format_out", "raw"], False),
    "fwss_burg_raw": (16000, ["-w", "32", "-s", "16", "-nr_mode", "fwss", "-nr_b", "1.5", "-vad", "burg", "-format_out", "raw"], False),
    "hwss_file_raw": (16000, ["-nr_mode", "hwss", "-vad", "file=vadin.bin", "-format_out", "raw"], True),
    # the Burg detector
    "fwss_burg_16k": (16000, BENCH_FWSS_BURG, False),
    "fwss_burg_8k": (8000, BENCH_FWSS_BURG, False),
    "2fwss_burg": (16000, MF + ["-nr_mode", "2fwss", "-vad", "burg", "-nr_initsegs", "5", "-format_out", "htk"], False),
    # the VAD module
    "vad_cepdist_lpc": (16000, MF + ["-format_out", "htk", "-vad_out_mode", "vad", "-vad_thr_mode", "adapt", "-vad_cri_mode", "cepdist",
                                     "-vad_cepdist_mode", "lpc", "-vad", "burg"], False),
    "vad_cepdist_fea": (16000, MF + ["-format_out", "htk", "-vad_out_mode", "vad", "-vad_thr_mode", "adapt", "-vad_cri_mode", "cepdist",
                                     "-vad_cepdist_mode", "fea", "-vad_filter_order", "5"], False),
    # the fp64 path
    "fwss_file_afterFB": (16000, MF + ["-nr_mode", "fwss", "-vad", "file=vadin.bin", "-nr_when", "afterFB", "-format_out", "htk"], True),
    "lpc_no_inld": (16000, ["-format_out", "htk", "-fb_scale", "mel", "-fea_kind", "lpc", "-fb_inld", "off", "-fea_lporder", "12",
                            "-fea_ncepcoefs", "12"], False),
    # raw energy
    "mfcc_E_raw": (16000, MF + ["-fea_E", "on", "-fea_rawenergy", "on", "-format_out", "htk"], False),
    "mfcc_E_D_A_raw": (16000, MF + ["-fea_E", "on", "-fea_rawenergy", "on", "-fea_delta", "d_a", "-format_out", "htk"], False),
}


def case_args(name, dc1=True):
    fs, extra, _ = CASES[name]
    return raw(fs) + extra + (DC1 if dc1 else [])


def ext_vad_for(o, utts, seed):
    """a VAD byte stream for -vad file=: one 0/1 byte per frame, runs of speech and pauses"""
    rng = np.random.default_rng(seed)
    out = []
    for u in utts:
        T = co.num_frames(len(u), o)
        out.append((np.repeat(rng.integers(0, 2, T // 7 + 1), 7)[:T]).astype(np.uint8))
    return out


def is_wave(o):
    return o.format_out in ("raw", "wave")


def wave_ok(got, want):
    if got.shape != want.shape:
        return False
    d = np.abs(got.astype(np.int32) - want.astype(np.int32))
    return d.size == 0 or (d.max() <= 1 and (d > 0).mean() < tp.WAVE_MAX_FRAC)


def features_ok(name, j, got, want, kind, sens):
    try:
        tp.check_features(name, j, got, want, kind, sens)
        return True
    except AssertionError:
        return False


def case_inputs(name):
    fs, _, has_ev = CASES[name]
    utts = signals(fs)
    o = co.parse_args(case_args(name))
    return o, utts, (ext_vad_for(o, utts, 7) if has_ev else None)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def ring_closed_form(x, w, s, T):
    """k_dc1_means' recurrence and the accumulated offsets, restated: m_t = mean(raw frame t) - sum_d m_{t-d} (w - d s) / w;
    sample i of frame t has lost m_{t-d} for every d <= t with i + d s < w.  Returns the ring's frames [T, w] and the sample
    before each frame as pre-emphasis reads it (sample s-1 of frame t-1)."""
    x = np.asarray(x, dtype=np.float64)
    m = np.zeros(T)
    for t in range(T):
        v = float(np.sum(x[t * s: t * s + w])) / w
        for d in range(1, t + 1):
            if d * s >= w:
                break
            v -= m[t - d] * (w - d * s) / w
        m[t] = v
    fr = np.empty((T, w))
    prev = np.zeros(T)
    for t in range(T):
        for i in range(w):
            v = x[t * s + i]
            for d in range((w - 1 - i) // s, -1, -1):
                if d <= t:
                    v -= m[t - d]
            fr[t, i] = v
        if t > 0:
            prev[t] = fr[t - 1, s - 1]
    return fr, prev


@pytest.mark.parametrize("ws", [("25", "10"), ("32", "8"), ("17", "1")], ids=["w/s=2.5", "w/s=4", "w/s=17"])
def test_ring_closed_form_reproduces_the_oracle_ring(ws):
    """The oracle de-means its sample ring frame after frame (front_end); the GPU computes the ring means once per utterance
    and subtracts the accumulated offsets.  The oracle's ring frames, read back from its spectra (no pre-emphasis, no window
    DC removal: the frame is irfft / window), and the sample before each frame (from the pre-emphasised spectra) agree with
    the closed form within 1e-9."""
    base = raw(16000) + ["-w", ws[0], "-s", ws[1], "-preset", "mfcc", "-format_out", "htk", "-remove_dc", "off"] + DC1
    x = biased(synthetic.utterance(3, 0.25), "ramp").astype(np.float64)
    x = np.clip(np.round(x + 3000.0 * np.sin(np.arange(len(x)) / 700.0)), -32768, 32767)      # DC that wanders
    o0 = co.parse_args(base + ["-preem", "0"])
    o1 = co.parse_args(base + ["-preem", "0.97"])
    w, s, T = o0.window, o0.wshift, co.num_frames(len(x), o0)
    assert w // s + 1 == {"25": 3, "32": 5, "17": 18}[ws[0]]
    W = co.hamming(w)
    fe0, fe1 = co.front_end(x, o0), co.front_end(x, o1)
    fr_o = np.fft.irfft(fe0.spec, o0.wfft)[:, :w] / W
    fr_c, prev_c = ring_closed_form(x, w, s, T)
    assert np.abs(fr_o - fr_c).max() < 1e-9, np.abs(fr_o - fr_c).max()
    a = float(np.float32(o1.preem))
    y0 = np.fft.irfft(fe1.spec, o1.wfft)[:, 0] / W[0]
    prev_o = (fr_o[:, 0] - y0) / a
    assert np.abs(prev_o - prev_c).max() < 1e-9, np.abs(prev_o - prev_c).max()
    # and the ring actually moved the samples: the raw frames are far from it
    assert np.abs(fr_c - np.stack([x[t * s: t * s + w] for t in range(T)])).max() > 1000


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_output_depends_on_remove_dc1(name):
    """For every GPU case below, the oracle with -remove_dc1 off is outside the bar the library is held to."""
    o, utts, ev = case_inputs(name)
    o_off = co.parse_args(case_args(name, dc1=False))
    differs = 0
    for j, u in enumerate(utts):
        e = None if ev is None else ev[j]
        on, off = co.run_pipeline(u, o, e), co.run_pipeline(u, o_off, e)
        if is_wave(o):
            differs += not wave_ok(off.waveform, on.waveform)
        else:
            differs += not features_ok(name, j, off.features, on.features, o.fea_kind, tp._sensitivity(case_args(name), o, u, e))
    assert differs == len(utts), (name, differs)


NEWLY_ACCEPTED = ["exten_raw_16k", "exten_raw_8k", "exten_wave_44k", "exten_raw_11k_w32", "fwss_burg_raw", "hwss_file_raw", "fwss_burg_16k",
                  "fwss_burg_8k", "2fwss_burg", "vad_cepdist_lpc", "vad_cepdist_fea", "fwss_file_afterFB", "lpc_no_inld", "mfcc_E_raw",
                  "mfcc_E_D_A_raw"]


def test_newly_accepted_configurations_pass_validation():
    """Each configuration that -remove_dc1 used to refuse now gets as far as the device: without a GPU the handle fails for
    the missing device (status 4), with one it is created."""
    import torch
    gpu = torch.cuda.is_available()
    for name in NEWLY_ACCEPTED + ["mulaw_exten_8k"]:
        args = case_args(name) if name in CASES else ["-fs", "8000", "-format_in", "mulaw", "-dither", "0", "-preset", "exten", "-format_out", "raw"] + DC1
        if gpu:
            cb.Handle(args).close()
            continue
        with pytest.raises(cb.CtuError) as e:
            cb.Handle(args)
        assert e.value.status == 4 and "no CPU fallback" in e.value.message, (name, e.value.status, e.value.message)


def test_remaining_refusals():
    """-dither stays refused on the chains that build the frame again, and together with -remove_dc1; a ring of more than
    17 shifts stays refused (status 3, before any device is touched).  The -dither messages name -dither alone."""
    cases = [
        (raw(16000)[:-2] + ["-dither", "1", "-preset", "exten", "-format_out", "raw"], "-dither"),
        (raw(16000)[:-2] + ["-dither", "1"] + BENCH_FWSS_BURG, "-dither"),
        (raw(16000)[:-2] + ["-dither", "1"] + MF + ["-format_out", "htk", "-vad_out_mode", "vad", "-vad_cri_mode", "cepdist",
                                                   "-vad_cepdist_mode", "lpc", "-vad", "burg"], "-dither"),
        (raw(16000)[:-2] + ["-dither", "1", "-preset", "mfcc", "-format_out", "htk"] + DC1, "-dither together with -remove_dc1"),
        (raw(16000) + ["-w", "18", "-s", "1", "-preset", "mfcc", "-format_out", "htk"] + DC1, "longer than 17 shifts"),
        (raw(16000) + ["-preset", "exten", "-w", "18", "-s", "1", "-format_out", "raw"] + DC1, "longer than 17 shifts"),
    ]
    for args, msg in cases:
        with pytest.raises(cb.CtuError) as e:
            cb.Handle(args)
        assert e.value.status == 3 and msg in e.value.message, (args, e.value.message)
        if msg == "-dither":
            assert "-remove_dc1" not in e.value.message, e.value.message


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def check_case(name, args, o, res, utts, ev, j0=0):
    """library result `res` (utterances from j0 on) against the oracle: waveforms within 1 LSB, features within the parity
    bar plus the subtraction sensitivity term, detector and VAD decisions bit for bit"""
    for j, u in enumerate(utts):
        e = None if ev is None else ev[j]
        ref = co.run_pipeline(u, o, e)
        k = j0 + j
        if is_wave(o):
            got = res.utt_waveform(k)
            d = np.abs(got.astype(np.int32) - ref.waveform.astype(np.int32))
            assert got.shape == ref.waveform.shape and (d.size == 0 or (d.max() <= 1 and (d > 0).mean() < tp.WAVE_MAX_FRAC)), \
                (name, j, got.shape, ref.waveform.shape, d.max() if d.size else 0)
        else:
            assert int(res.frames_per_utt[k]) == ref.nframes, (name, j)
            tp.check_features(name, j, res.utt_features(k), ref.features, o.fea_kind, tp._sensitivity(args, o, u, e))
        r0 = int(res.row_offsets[k])
        if ref.vad_nr is not None and o.vadmode == "burg":
            got = res.vad_nr[r0: r0 + ref.nframes].astype(bool)
            assert np.array_equal(got, ref.vad_nr), (name, j, "detector decisions differ at %d frames" % int((got != ref.vad_nr).sum()))
        if ref.vad is not None:
            v = ref.vad.vad
            got = res.vad_out[r0: r0 + len(v)].astype(bool)
            assert np.array_equal(got, v), (name, j, "VAD decisions differ at %d frames" % int((got != v).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_cuda_matches_oracle_with_remove_dc1(name):
    o, utts, ev = case_inputs(name)
    args = case_args(name)
    res = cb.extract(args, utts, ev)
    check_case(name, args, o, res, utts, ev)


@pytest.mark.gpu
def test_mulaw_8k_exten_waveform():
    """G.711 input: the 8-bit codes go to the device as they are, the ring is built from their expansion"""
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(gu.GOLDEN, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    args = ["-fs", "8000", "-format_in", "mulaw", "-dither", "0", "-preset", "exten", "-format_out", "raw"] + DC1
    o = co.parse_args(args)
    o_off = co.parse_args(args[:-2])
    codes = [mg.g711_encode(u, False) for u in signals(8000)]
    res = cb.extract_g711(args, codes, alaw=False)
    for j, c in enumerate(codes):
        pcm = co.g711_expand(c, False)
        ref = co.run_pipeline(pcm, o)
        assert wave_ok(res.utt_waveform(j), ref.waveform), j
        assert not wave_ok(co.run_pipeline(pcm, o_off).waveform, ref.waveform), j


def _chunks_of(lengths, chunk_mb):
    """chunks ctu_plan_run_host cuts the list into (utterances up to chunk_mb << 19 samples, at least one)"""
    lim, n, u0, offs = chunk_mb << 19, 0, 0, np.concatenate([[0], np.cumsum(lengths)])
    while u0 < len(lengths):
        u1 = u0 + 1
        while u1 < len(lengths) and offs[u1 + 1] - offs[u0] <= lim:
            u1 += 1
        u0, n = u1, n + 1
    return n


LONG_CHAINS = {"exten_raw_16k": False, "fwss_burg_16k": False, "mfcc_E_D_A_raw": True}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(LONG_CHAINS))
def test_long_ragged_batches_and_entry_points(name):
    """10 s utterances (about 60 16-frame tiles each: the ring means cross every tile boundary) in a ragged list with
    zero-frame and one-frame entries where the chain takes them (no deltas; a delta chain gets the shortest utterance it
    accepts), so the ring restarts at every utterance.  run_device, run_host and run_host in 1 MB chunks (several chunks on
    three streams) agree bit for bit."""
    import torch
    args = case_args(name)
    o = co.parse_args(args)
    w = o.window
    deltas = LONG_CHAINS[name]
    s = o.wshift
    longs = [biased(synthetic.utterance(k, 10.0), kind) for k, kind in zip(range(20, 28), ("plus", "ramp", "minus", "clip") * 2)]
    if deltas:
        # a delta chain refuses utterances shorter than its window + 2 frames (zero frames included): the shortest it takes
        shorts = [biased(synthetic.utterance(40 + k, 0.2)[: w + 3 * s + 7 * k], "plus") for k in range(3)]
    else:
        shorts = [biased(synthetic.utterance(40 + k, 0.1)[: w - s + 13 * k], "plus") for k in range(3)]         # zero frames
        shorts += [biased(synthetic.utterance(50 + k, 0.1)[: w + 5 * k], "minus") for k in range(3)]           # one frame
    utts = []
    for k, u in enumerate(longs):
        utts += [u, shorts[k % len(shorts)]]
    lens = [len(u) for u in utts]
    hd = cb.Handle(args)
    plan = hd.plan(lens)
    pcm = np.ascontiguousarray(np.concatenate(utts))
    sig = hd.signal_output
    nfr = plan.total_frames
    d_pcm = torch.from_numpy(pcm).cuda()
    d_vnr = torch.zeros(max(nfr, 1), dtype=torch.uint8, device="cuda")
    if sig:
        d_out = torch.empty(plan.total_output_samples, dtype=torch.int16, device="cuda")
        plan.run_device(d_pcm.data_ptr(), d_waveform=d_out.data_ptr(), d_vad_nr=d_vnr.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    else:
        d_out = torch.empty((nfr, hd.feature_dim), dtype=torch.float32, device="cuda")
        plan.run_device(d_pcm.data_ptr(), d_features=d_out.data_ptr(), d_vad_nr=d_vnr.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    out, vnr = d_out.cpu().numpy(), d_vnr.cpu().numpy()[:nfr]

    def bits(a):
        return a.view(np.uint32) if a.dtype == np.float32 else a

    results = []
    for chunk_mb in (None, 1):
        if chunk_mb:
            hd.set_option("chunk_mb", chunk_mb)
        res = plan.run_host(pcm)
        got = res.waveform if sig else res.features
        assert np.array_equal(bits(got), bits(out)), (name, chunk_mb, "run_host differs from run_device")
        if o.vadmode == "burg":
            assert np.array_equal(res.vad_nr, vnr), (name, chunk_mb, "detector decisions")
        results.append(res)
    fpu = plan.frames_per_utt
    assert deltas or (int((fpu == 0).sum()) >= 3 and int((fpu == 1).sum()) >= 3), fpu
    assert _chunks_of(lens, 1) >= 2
    # the oracle: two long utterances and every short one that has frames
    pick = [0, 2] + [j for j, u in enumerate(utts) if len(u) < 2 * w + 3 * s and fpu[j] > 0]
    for j in pick:
        check_case(name, args, o, results[1], [utts[j]], None, j0=j)
    plan.close()
    hd.close()


@pytest.mark.gpu
def test_cli_wave_files_equal_the_library_waveform(tmp_path):
    """host/ctucopy_b200 -remove_dc1 on -format_out wave -S list: every file is the library's waveform behind the 44-byte header"""
    args = case_args("exten_wave_44k")
    utts = signals(44100)
    for i, u in enumerate(utts):
        np.asarray(u).astype("<i2").tofile(str(tmp_path / ("u%d.raw" % i)))
    with open(tmp_path / "list.scp", "w") as fh:
        for i in range(len(utts)):
            fh.write("%s/u%d.raw %s/u%d.wav\n" % (tmp_path, i, tmp_path, i))
    pr = subprocess.run([EXE] + args + ["-S", str(tmp_path / "list.scp")], capture_output=True, cwd=str(tmp_path))
    assert pr.returncode == 0, pr.stderr.decode()
    res = cb.extract(args, utts)
    for i in range(len(utts)):
        b = open(tmp_path / ("u%d.wav" % i), "rb").read()
        assert b[:4] == b"RIFF" and len(b) == 44 + 2 * len(res.utt_waveform(i)), i
        assert np.array_equal(np.frombuffer(b[44:], dtype="<i2"), res.utt_waveform(i)), i
