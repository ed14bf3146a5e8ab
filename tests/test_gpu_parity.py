"""Parity of the CUDA path (through the C ABI) against the reference binary's committed
outputs (tests/golden) and against the numpy oracle on fresh seeded inputs.

Bars (BASELINE.json north_star): bit-exact frame counts, row counts and VAD decisions;
payload within 1e-4 relative or 1e-3 absolute in the log domain; int16 waveforms within
1 LSB (on fewer than 0.5 % of the samples; measured 0.11 % on 10 s utterances: floor() boundaries,
SURVEY App. C-16); non-finite positions identical.
"""
import numpy as np
import pytest

import ctu_oracle as co
import golden_util as gu
import ctucopy_b200 as cb
from ctucopy_b200 import synthetic

pytestmark = pytest.mark.gpu

# log-domain feature kinds compare with an absolute floor of 1e-3.  Linear ones (band values, LP coefficients) at 1e-4
# relative plus 1e-5 of the row maximum: north_star's "1e-3 absolute in the log domain" is 1e-3 RELATIVE for the linear
# value, so this is the tighter reading for every entry within 40 dB of the frame's peak, and the floor only matters for
# bands 100 dB below it (a sum of fp32 products cannot resolve those: the reference carries them in fp64)
LOG_KINDS = ("dctc", "lpc", "logspec", "trapdct", "td-iir-mfcc")
ILL_CONDITIONED = {"lpa_mel"}   # lpa from SQUARED mel band powers: see tests/test_oracle_vs_golden.py; the well-conditioned
                                # lpa case (PLP bank, cube-root compressed) is the golden plpc_lpa, held to the full bar
# hwss zeroes bins by half-wave rectification.  In the LOG domain, log(0) = -inf positions depend on the sign of quantities
# that are 0 +- rounding (the reference is not reproducible against itself across FFT libraries there): for this one golden
# only the finite entries that agree are compared.  The mode itself is pinned at the full tolerance in the LINEAR domain by
# the goldens hwss_burg_spec_mag / hwss_burg_spec_pow (below, through check_features' normal path), and its detector
# decisions bit for bit.
HALFWAVE = {"hwss_burg_a2"}
WAVE_MAX_FRAC = 0.005           # share of samples allowed to differ by one LSB


def check_features(name, i, got, want, kind, sens=None):
    assert got.shape == want.shape, (name, i, got.shape, want.shape)
    if name in HALFWAVE:
        both = np.isfinite(got) & np.isfinite(want)
        assert both.mean() > 0.5 * np.isfinite(want).mean()
        np.testing.assert_allclose(got[both], want[both], rtol=1e-3, atol=5e-2)
        return
    assert gu.same_nonfinite(got, want), (name, i, "non-finite positions differ")
    fin = np.isfinite(want)
    if name in ILL_CONDITIONED:
        np.testing.assert_allclose(got[fin], want[fin], rtol=5e-2, atol=5e-2)
        return
    err = np.abs(got - want)[fin]
    if kind in LOG_KINDS:
        tol = 1e-4 * np.abs(want) + 1e-3
    else:
        rowmax = np.max(np.where(fin, np.abs(want), 0), axis=1, keepdims=True)
        tol = 1e-4 * np.abs(want) + 1e-5 * rowmax
    if sens is not None:
        # behind a spectral subtraction: plus four times the oracle's own response to one front-end rounding error of its
        # input spectrum (tools/parity_sweep.py: sensitivity) -- where |X| - b N cancels k digits no implementation that
        # computes the spectrum in fp32 can agree to better than 1e-7 x 10^k of the result
        tol = tol + 4.0 * sens
    tol = tol[fin]
    bad = err > tol
    assert not bad.any(), (name, i, "max err %.3g (tol %.3g) at %d entries" % (err.max(), tol[np.argmax(err)], bad.sum()))


def _sweep_module():
    import importlib.util, os
    spec = importlib.util.spec_from_file_location("parity_sweep", os.path.join(gu.GOLDEN, "..", "..", "tools", "parity_sweep.py"))
    ps = importlib.util.module_from_spec(spec); spec.loader.exec_module(ps)
    return ps


def _sensitivity(args, o, pcm, ext_vad=None):
    return _sweep_module().sensitivity(args, o, pcm, None, ext_vad)


@pytest.mark.parametrize("name", gu.case_names())
def test_cuda_matches_reference_golden(name):
    c = gu.Case(name)
    args = c.oracle_args()
    o = co.parse_args(args)
    ins = gu.inputs()
    idx = list(range(len(ins)))
    if o.n_order > 0:
        # utterances shorter than delta window + 2 frames take the reference's start-up path
        # (ring memory never written); the library refuses them explicitly
        mw = max([o.d_win, o.a_win, o.t_win][: o.n_order])
        short = [i for i in idx if co.num_frames(len(ins[i]), o) < mw + 2]
        for i in short:
            with pytest.raises(cb.CtuError):
                cb.extract(args, [ins[i]])
        idx = [i for i in idx if i not in short]
    ev = [c.extvad[i] for i in idx] if c.extvad[idx[0]] is not None else None
    res = cb.extract(args, [ins[i] for i in idx], ev)
    for j, i in enumerate(idx):
        if o.dither != 0.0:
            # the goldens are one reference process per utterance: every file starts the rand() stream afresh,
            # while a batch continues it from utterance to utterance (test_dither_stream_continues_through_a_list)
            res, j = cb.extract(args, [ins[i]]), 0
        want = c.payload(i)
        if c.kind in ("raw", "wave"):
            got = res.utt_waveform(j)
            assert got.shape == want.shape, (name, i)
            d = np.abs(got.astype(np.int32) - want.astype(np.int32))
            assert d.max() <= 1, (name, i, d.max())
            assert (d > 0).mean() < WAVE_MAX_FRAC, (name, i, (d > 0).mean())
        else:
            got = res.utt_features(j)
            assert int(res.frames_per_utt[j]) == co.num_frames(len(ins[i]), o)
            check_features(name, i, got, want, o.fea_kind, _sensitivity(args, o, ins[i], c.extvad[i]))
        if c.aux[i] is not None and c.kind != "ark":
            v = np.frombuffer(c.aux[i], dtype=np.uint8) - 48
            r0 = int(res.row_offsets[j])
            gotv = res.vad_out[r0: r0 + len(v)]
            assert np.array_equal(gotv, v), (name, i, "VAD decisions differ at %d frames" % int((gotv != v).sum()))


@pytest.mark.parametrize("name", gu.carry_case_names())
def test_cuda_list_carry_matches_reference_golden(name):
    """ss_carry (opt-in): hwss / fwss / 2fwss with the reference's LIST semantics -- a file's noise estimate starts from the
    enhanced last frame of the file before it (src/nr/nr.cc:212-222, 397-408).  The goldens are the files of ONE reference
    process; detector decisions bit for bit.  (The carried value itself has the tolerance of the previous file's last row,
    so the conditioning probe starts from the oracle's carry.)"""
    args, kind, idx, outs, ev = gu.carry_case(name)
    o = co.parse_args(args)
    ins = [gu.inputs()[i] for i in idx]
    res = cb.extract(args, ins, ev, options={"ss_carry": 1})
    refs = co.run_list_carry(ins, o, ev)
    ps = _sweep_module()
    for j, u in enumerate(ins):
        if kind == "raw":
            want = np.frombuffer(outs[j], dtype="<i2")
            got = res.utt_waveform(j)
            assert got.shape == want.shape, (name, j)
            d = np.abs(got.astype(np.int32) - want.astype(np.int32))
            assert d.max() <= 1 and (d > 0).mean() < WAVE_MAX_FRAC, (name, j, d.max(), (d > 0).mean())
        else:
            want = gu.rr.parse_htk(outs[j])[1]
            sens = ps.sensitivity(args, o, u, refs[j], None if ev is None else ev[j], refs[j].navg0)
            check_features(name, j, res.utt_features(j), want, o.fea_kind, sens)
        if refs[j].vad_nr is not None and o.vadmode == "burg":
            r0 = int(res.row_offsets[j])
            assert np.array_equal(res.vad_nr[r0: r0 + refs[j].nframes].astype(bool), refs[j].vad_nr), (name, j)
    # and a second call on a fresh handle without the option gives the per-utterance result again
    solo = cb.extract(args, ins[1:2], None if ev is None else ev[1:2])
    ref1 = co.run_pipeline(ins[1], o, None if ev is None else ev[1])
    if kind == "raw":
        assert np.abs(solo.utt_waveform(0).astype(np.int32) - ref1.waveform.astype(np.int32)).max() <= 1
    else:
        check_features(name, 1, solo.utt_features(0), ref1.features, o.fea_kind, ps.sensitivity(args, o, ins[1], ref1, None if ev is None else ev[1]))


PARITY_SET = [synthetic.utterance(k, sec) for k, sec in [(0, 1.0), (1, 2.5), (2, 1.0), (3, 2.5), (4, 1.0), (5, 1.0), (6, 2.5), (7, 1.0),
                                                         (8, 1.0), (9, 2.5), (10, 1.0), (11, 1.0), (12, 1.0), (13, 2.5), (14, 1.0)]]
B = ["-fs", "16000", "-format_in", "raw", "-dither", "0"]
ORACLE_CASES = {
    "mfcc_d_a": B + ["-preset", "mfcc", "-preem", "0.97", "-fb_definition", "23filters", "-format_out", "htk", "-fea_delta", "d_a"],
    "plp": B + ["-preset", "plpc", "-format_out", "ark=x.ark"],
    "trapdct": B + ["-format_out", "htk", "-fb_definition", "23filters", "-fb_eqld", "off", "-fb_inld", "off", "-preem", "0.97",
                    "-fea_kind", "trapdct,51,8"],
    "exten_raw": B + ["-preset", "exten", "-format_out", "raw"],
    "mfcc_exten": B + ["-preset", "mfcc", "-preem", "0.97", "-nr_mode", "exten", "-format_out", "htk", "-fea_delta", "d_a"],
    "fwss_burg": B + ["-preset", "mfcc", "-preem", "0.97", "-nr_mode", "fwss", "-vad", "burg", "-format_out", "pfile=x.pfile"],
    # SURVEY 8f.4: time-domain IIR filter bank (25 / 10 ms: five 80-sample segments per frame, two per shift)
    "tdiir": B + ["-format_out", "htk", "-w", "25", "-s", "10", "-fea_kind", "td-iir-mfcc", "-filters", gu.rr.TDIIR_FILTERS, "-fea_ncepcoefs", "12"],
}


@pytest.mark.parametrize("name", list(ORACLE_CASES))
def test_cuda_matches_oracle_on_parity_set(name):
    """Fresh seeded inputs (tones / chirps / pink noise at several SNRs), whole batch in one
    call, each utterance compared with the oracle run on it alone."""
    args = ORACLE_CASES[name]
    o = co.parse_args(args)
    res = cb.extract(args, PARITY_SET)
    for j, u in enumerate(PARITY_SET):
        ref = co.run_pipeline(u, o)
        if o.format_out == "raw":
            d = np.abs(res.utt_waveform(j).astype(np.int32) - ref.waveform.astype(np.int32))
            assert d.max() <= 1 and (d > 0).mean() < WAVE_MAX_FRAC, (name, j, d.max(), (d > 0).mean())
        else:
            check_features(name, j, res.utt_features(j), ref.features, o.fea_kind)
        if ref.vad_nr is not None:
            r0 = int(res.row_offsets[j])
            got = res.vad_nr[r0: r0 + ref.nframes]
            assert np.array_equal(got.astype(bool), ref.vad_nr), (name, j, "detector decisions differ at %d frames" % int((got.astype(bool) != ref.vad_nr).sum()))


# every alternative kernel path of the BASELINE configurations (run-time options, ctu_set_option): the standalone scan
# instead of the one fused into k_bank
ALT_PATHS = [("mfcc_exten", {"fuse_nr": 0}), ("mfcc_exten", {"fuse_nr": 1}), ("fwss_burg", {"fuse_nr": 0}), ("fwss_burg", {"fuse_nr": 1})]


@pytest.mark.parametrize("name,options", ALT_PATHS, ids=["%s-%s" % (n, "+".join("%s=%d" % kv for kv in o.items())) for n, o in ALT_PATHS])
def test_alternative_kernel_paths_match_oracle(name, options):
    args = ORACLE_CASES[name]
    o = co.parse_args(args)
    res = cb.extract(args, PARITY_SET, options=options)
    for j, u in enumerate(PARITY_SET):
        ref = co.run_pipeline(u, o)
        if o.format_out == "raw":
            d = np.abs(res.utt_waveform(j).astype(np.int32) - ref.waveform.astype(np.int32))
            assert d.max() <= 1 and (d > 0).mean() < WAVE_MAX_FRAC, (name, j, d.max(), (d > 0).mean())
        else:
            check_features(name, j, res.utt_features(j), ref.features, o.fea_kind)
        if ref.vad_nr is not None:
            r0 = int(res.row_offsets[j])
            assert np.array_equal(res.vad_nr[r0: r0 + ref.nframes].astype(bool), ref.vad_nr), (name, j)


@pytest.mark.parametrize("front256", [1, 0])
def test_8khz_front_ends_match_oracle(front256):
    """256-point frames (8 kHz): the specialised front end k_frames256 (default) and the general kernel k_frames_any, on a
    ragged batch, plain MFCC_0_D_A and MFCC behind exten (the spectrum goes through the scan in between)."""
    for extra in ([], ["-nr_mode", "exten"]):
        args = ["-fs", "8000", "-format_in", "raw", "-dither", "0", "-preset", "mfcc", "-preem", "0.97"] + extra + ["-fea_delta", "d_a", "-format_out", "htk"]
        o = co.parse_args(args)
        utts = PARITY_SET[:6] + [PARITY_SET[1][:4000 + 37], PARITY_SET[3][:200 + 80 * 6]]
        res = cb.extract(args, utts, options={"front256": front256})
        for j, u in enumerate(utts):
            ref = co.run_pipeline(u, o)
            assert int(res.frames_per_utt[j]) == ref.nframes
            check_features("mfcc8k", j, res.utt_features(j), ref.features, o.fea_kind, _sensitivity(args, o, u) if extra else None)


def test_fused_and_standalone_scan_agree_bit_for_bit():
    """k_bank's in-tile scan and the standalone k_nr_scan4 run the same recursion step (nr_step): identical features."""
    for name in ("mfcc_exten", "fwss_burg"):
        a = cb.extract(ORACLE_CASES[name], PARITY_SET, options={"fuse_nr": 1})
        b = cb.extract(ORACLE_CASES[name], PARITY_SET, options={"fuse_nr": 0})
        assert np.array_equal(a.features, b.features), name


def test_compact_and_in_place_cepstra_agree_bit_for_bit(monkeypatch):
    """MFCC + deltas: the cepstra as a compact matrix with the delta kernel writing whole rows (default) and the in-place layout
    (CTU_COMPACT_STATIC=0, read when the handle is created) run the same arithmetic on the same values: identical features, on a
    ragged batch, with and without a noise-reduction scan in front."""
    utts = PARITY_SET[:5] + [PARITY_SET[1][:4000 + 37], PARITY_SET[3][:400 + 160 * 6]]
    for name in ("mfcc_d_a", "mfcc_exten"):
        monkeypatch.delenv("CTU_COMPACT_STATIC", raising=False)
        a = cb.extract(ORACLE_CASES[name], utts)
        monkeypatch.setenv("CTU_COMPACT_STATIC", "0")
        b = cb.extract(ORACLE_CASES[name], utts)
        assert a.features.shape == b.features.shape and np.array_equal(a.features, b.features), name
    monkeypatch.delenv("CTU_COMPACT_STATIC", raising=False)


@pytest.mark.parametrize("name", [n for n in gu.case_names() if n.startswith("vaddbg_")])
def test_vad_debug_side_files_match_reference(name):
    """-vad_out_mode debug: the side files next to the decision file (criterion, threshold and its state per written row,
    init flags, unfiltered decisions), assembled from ctu_plan_fetch_vad_debug like the CLI does, against the files the
    reference binary wrote.  Characters bit for bit; doubles to 1e-9 relative (the criterion of the energy mode is a sum
    over an fp32 spectrum on the device, fp64 in the reference: 1e-6 of the undecibeled value; dB values ~1e-8)."""
    c = gu.Case(name)
    args = c.oracle_args()
    ins = gu.inputs()
    o = co.parse_args(args)
    mw = max([o.d_win, o.a_win, o.t_win][: o.n_order]) if o.n_order > 0 else 0
    # (utterances shorter than delta window + 2 frames are refused, see test_cuda_matches_reference_golden)
    idx = [i for i in range(len(ins)) if c.debug[i] and co.num_frames(len(ins[i]), o) >= mw + 2]
    hd = cb.Handle(args)
    plan = hd.plan([len(ins[i]) for i in idx])
    res = plan.run_host(np.ascontiguousarray(np.concatenate([ins[i] for i in idx]).astype(np.int16)))
    steps, vad0 = plan.fetch_vad_debug()
    for j, i in enumerate(idx):
        r0, r1 = int(res.row_offsets[j]), int(res.row_offsets[j + 1])
        files = cb.vad_debug_files(hd.cfg, steps[r0:r1], vad0[r0:r1])
        want = c.debug[i]
        assert sorted(files) == sorted(want), (name, i, sorted(files), sorted(want))
        for suf, wb in want.items():
            gb = files[suf]
            assert len(gb) == len(wb), (name, i, suf, len(gb), len(wb))
            if suf in ("vad0", "c0init", "init"):
                assert gb == wb, (name, i, suf, "flags differ")
            else:
                g, w_ = np.frombuffer(gb, dtype="<f8"), np.frombuffer(wb, dtype="<f8")
                np.testing.assert_allclose(g, w_, rtol=2e-5, atol=1e-6, err_msg="%s input %d file _%s" % (name, i, suf))
    plan.close(); hd.close()


def test_batch_position_independence_and_ragged_lengths():
    """An utterance's output does not depend on where it sits in the list (what makes
    utterance sharding exact, SURVEY.md finding 4), including ragged lengths and a
    zero-frame entry."""
    args = ORACLE_CASES["mfcc_d_a"]
    utts = [PARITY_SET[3][:16000 + 37], PARITY_SET[0], PARITY_SET[1][:4000], PARITY_SET[2]]
    a = cb.extract(args, utts)
    b = cb.extract(args, utts[::-1])
    for j in range(len(utts)):
        assert np.array_equal(a.utt_features(j), b.utt_features(len(utts) - 1 - j))
    single = cb.extract(args, [utts[2]])
    assert np.array_equal(single.utt_features(0), a.utt_features(2))
    # zero-frame utterance (w-s <= N < w) yields zero rows, shorter input is refused like the reference
    args0 = B + ["-preset", "mfcc", "-format_out", "htk"]
    r = cb.extract(args0, [PARITY_SET[0][:399], PARITY_SET[0][:400]])
    assert list(r.frames_per_utt) == [0, 1]
    with pytest.raises(cb.CtuError) as e:
        cb.extract(args0, [PARITY_SET[0][:239]])
    assert "Signal shorter than one frame" in e.value.message


def test_full_size_properties():
    """At BASELINE's full utterance size (10 s, 998 frames) and a few hundred utterances:
    frame counts, linearity of the spectrum stage in the input scale (power scales by 4 ->
    log-mel features shift by ln 4 on c0 only), and determinism."""
    args = B + ["-preset", "mfcc", "-preem", "0.97", "-format_out", "htk", "-fea_lifter", "0"]
    base = [synthetic.utterance(k, 10.0) for k in range(4)]
    utts = [base[i % 4] for i in range(64)]
    r1 = cb.extract(args, utts)
    assert np.all(r1.frames_per_utt == 998) and r1.features.shape == (64 * 998, 13)
    r2 = cb.extract(args, utts)
    assert np.array_equal(r1.features, r2.features)
    for j in range(4, 64):
        assert np.array_equal(r1.utt_features(j), r1.utt_features(j % 4))
    half = [(u // 2 * 2 // 2).astype(np.int16) for u in base]            # exact halves of even samples
    even = [(u // 2 * 2).astype(np.int16) for u in base]
    fe = cb.extract(args, even).features
    fh = cb.extract(args, half).features
    d = fe - fh
    c0_shift = np.sqrt(2.0 / 26) * 26 * np.log(4.0)
    assert np.allclose(d[:, :12], 0, atol=2e-3)
    assert np.allclose(d[:, 12], c0_shift, atol=2e-3)


def test_spectrum_tap_matches_numpy_fft():
    import torch
    args = B + ["-preset", "mfcc", "-preem", "0.97", "-format_out", "htk"]
    hd = cb.Handle(args)
    u = PARITY_SET[1]
    plan = hd.plan([len(u)])
    d_pcm = torch.from_numpy(u.copy()).cuda()
    d_spec = torch.empty((plan.total_frames, 257), dtype=torch.float32, device="cuda")
    st = hd.L.ctu_debug_spectrum(plan.p, d_pcm.data_ptr(), d_spec.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert st == 0
    o = co.parse_args(args)
    want = co.front_end(u, o).Xabs
    got = d_spec.cpu().numpy().astype(np.float64)
    rowmax = want.max(axis=1, keepdims=True)
    assert np.all(np.abs(got - want) <= 1e-4 * want + 2e-6 * rowmax)
    plan.close(); hd.close()


def test_energy_column_with_vad_delay_matches_oracle():
    """-fea_E rows written through the VAD module carry the energy of the frame that is
    (delta latency + majority-filter delay) ahead (checked against the reference binary when
    the oracle was extended; here CUDA vs oracle)."""
    args = B + ["-preset", "mfcc", "-preem", "0.97", "-fea_E", "on", "-fea_delta", "d_a", "-format_out", "htk",
                "-vad_out_mode", "vad", "-vad_filter_order", "5"]
    o = co.parse_args(args)
    res = cb.extract(args, PARITY_SET[:4])
    for j, u in enumerate(PARITY_SET[:4]):
        ref = co.run_pipeline(u, o)
        check_features("mfcc_E_vad", j, res.utt_features(j), ref.features, "dctc")


@pytest.mark.parametrize("name", ["mfcc_exten", "fwss_burg", "exten_raw", "plp", "trapdct", "tdiir"])
def test_full_length_utterances_match_oracle(name):
    """BASELINE's utterance size (10 s = 998 frames): the cross-frame recursions (noise estimates,
    detector thresholds, overlap-add) run their full length; every detector decision must match."""
    args = ORACLE_CASES[name]
    o = co.parse_args(args)
    utts = [synthetic.utterance(k, 10.0) for k in (3, 6)]
    res = cb.extract(args, utts)
    for j, u in enumerate(utts):
        ref = co.run_pipeline(u, o)
        if o.format_out == "raw":
            d = np.abs(res.utt_waveform(j).astype(np.int32) - ref.waveform.astype(np.int32))
            assert d.max() <= 1 and (d > 0).mean() < WAVE_MAX_FRAC, (name, j, d.max(), (d > 0).mean())
        else:
            assert int(res.frames_per_utt[j]) == 998
            check_features(name, j, res.utt_features(j), ref.features, o.fea_kind)
        if ref.vad_nr is not None:
            r0 = int(res.row_offsets[j])
            got = res.vad_nr[r0: r0 + ref.nframes]
            assert np.array_equal(got.astype(bool), ref.vad_nr), (name, j, int((got.astype(bool) != ref.vad_nr).sum()))


def test_randomised_option_sweep_matches_oracle():
    """A fixed draw of 30 option sets from tools/parity_sweep.py (filter-bank scales / shapes, feature kinds,
    orders, lifters, deltas, noise-reduction modes, energy, CMS), CUDA vs oracle at the north_star tolerance.
    hwss is left out: half-wave rectification makes the reference irreproducible against itself."""
    import random
    import importlib.util
    spec = importlib.util.spec_from_file_location("parity_sweep", __import__("os").path.join(gu.GOLDEN, "..", "..", "tools", "parity_sweep.py"))
    ps = importlib.util.module_from_spec(spec); spec.loader.exec_module(ps)
    rng = random.Random(5)
    ins = [gu.inputs()[i] for i in (0, 5)]
    done = 0
    while done < 30:
        args = ps.draw(rng)
        if "hwss" in args:
            continue
        o = co.parse_args(args)
        try:
            res = cb.extract(args, ins)
        except cb.CtuError as e:
            assert e.status == 3, (args, e.message)          # only "not built" refusals are acceptable
            continue
        for i, u in enumerate(ins):
            ref = co.run_pipeline(u, o)
            ok, why = ps.tol_ok(res.utt_features(i), ref.features, o.fea_kind, ps.sensitivity(args, o, u, ref))
            assert ok, (why, " ".join(args))
            if ref.vad_nr is not None:
                r0 = int(res.row_offsets[i])
                assert np.array_equal(res.vad_nr[r0: r0 + ref.nframes].astype(bool), ref.vad_nr), " ".join(args)
        done += 1


@pytest.mark.parametrize("n, seed, signal_share, other_fs_share", [(200, 23, 0.0, 0.0), (200, 61, 0.3, 1.0), (200, 63, 0.5, 0.7)])
def test_option_sweeps_of_200_sets_have_no_miss_outside_log_domain_hwss(n, seed, signal_share, other_fs_share):
    """The three draws of tools/parity_sweep.py that left non-hwss misses open at the end of round 1 (profiles/
    r01_parity_sweeps.txt), as the tool itself runs them: waveform draws (<= 1 LSB), other sampling rates, the VAD module,
    detector and VAD decisions bit for bit.  Every option set without -nr_mode hwss must pass."""
    import random
    ps = _sweep_module()
    ps.SIGNAL_SHARE, ps.OTHER_FS_SHARE = signal_share, other_fs_share
    rng = random.Random(seed)
    ins = [gu.inputs()[i] for i in (0, 5)]
    bad = []
    for _ in range(n):
        args = ps.draw(rng)
        try:
            o = co.parse_args(args)
            refs = [co.run_pipeline(u, o) for u in ins]
        except Exception:
            continue                                         # invalid for the reference too
        if o.nr_mode == "hwss":
            continue
        try:
            res = cb.extract(args, ins)
        except cb.CtuError as e:
            assert e.status == 3, (" ".join(args), e.message)
            continue
        for i, u in enumerate(ins):
            if o.format_out == "raw":
                g, w_ = res.utt_waveform(i).astype(np.int32), refs[i].waveform.astype(np.int32)
                ok = g.shape == w_.shape and np.abs(g - w_).max() <= 1 and (g != w_).mean() < 0.02
                why = "waveform"
            else:
                ok, why = ps.tol_ok(res.utt_features(i), refs[i].features, o.fea_kind, ps.sensitivity(args, o, u, refs[i]))
            r0 = int(res.row_offsets[i])
            if refs[i].vad_nr is not None:
                ok = ok and np.array_equal(res.vad_nr[r0: r0 + refs[i].nframes].astype(bool), refs[i].vad_nr)
            if refs[i].vad is not None:
                ok = ok and np.array_equal(res.vad_out[r0: r0 + refs[i].nframes].astype(bool), refs[i].vad.vad)
            if not ok:
                bad.append((i, why, " ".join(args)))
    assert not bad, bad


def test_dither_stream_continues_through_a_list():
    """-dither: the second and third utterances of a batch take their noise from where the first one stopped in the
    process-wide rand() stream, exactly like the files of a reference list (src/io/in.cc:205, 452-455)."""
    args = ["-fs", "16000", "-format_in", "raw", "-dither", "1.0", "-preset", "mfcc", "-preem", "0.97", "-fea_delta", "d_a", "-format_out", "htk"]
    o = co.parse_args(args)
    utts = [PARITY_SET[0], PARITY_SET[1], PARITY_SET[2]]
    res = cb.extract(args, utts)
    off = 0
    for j, u in enumerate(utts):
        ref = co.run_pipeline(u, o, rand_offset=off)
        off += (o.window - o.wshift) + ref.nframes * o.wshift
        check_features("dither", j, res.utt_features(j), ref.features, "dctc")


# ---- SURVEY 8f.3: context stacking, deltas of spectral vectors, feature-file input ---------------------------------------

@pytest.mark.parametrize("name", gu.feain_case_names())
def test_cuda_feature_input_matches_reference_golden(name):
    """-format_in htk: rows of an existing feature file through deltas / stacking / CMS (ctu_plan_run_host_fea).  Gathers
    (copy, stacking) are bit-exact; the delta regression is fp32 on the device, fp64 in the reference."""
    c = gu.Case(name)
    args = c.oracle_args()
    o = co.parse_args(args)
    src = gu.Case(c.source)
    mats = [np.ascontiguousarray(src.payload(i), dtype=np.float32) for i in range(len(gu.inputs()))]
    idx = list(range(len(mats)))
    if o.fea_delta and o.n_order > 0:
        mw = max([o.d_win, o.a_win, o.t_win][: o.n_order])
        short = [i for i in idx if mats[i].shape[0] < mw + 2]
        for i in short:
            with pytest.raises(cb.CtuError):
                cb.extract_features(args, [mats[i]])
        idx = [i for i in idx if i not in short]
    res = cb.extract_features(args, [mats[i] for i in idx])
    exact = o.fea_trap or not o.fea_delta
    for j, i in enumerate(idx):
        got, want = res.utt_features(j), c.payload(i)
        if exact and not (o.cms_exp_coef > 0):
            assert got.shape == want.shape and np.array_equal(got, want), (name, i)
        else:
            check_features(name, i, got, want, "dctc")


def test_stacking_large_batch_matches_closed_form_bit_exactly():
    """-fea_trap on feature input, 300 ragged utterances in one plan, windows from 3 to 31 rows: a pure gather, so the
    device result must equal the oracle's closed form (= the reference's state machine) bit for bit.  Also through the
    device-resident entry point."""
    import torch
    rng = np.random.default_rng(5)
    for N, dim in ((3, 13), (9, 13), (31, 20)):
        w = (N - 1) // 2
        mats = [rng.standard_normal((int(rng.integers(w + 2, 400)), dim)).astype(np.float32) for _ in range(300)]
        args = ["-fs", "16000", "-format_in", "htk", "-nfeacoefs", str(dim), "-fea_ncepcoefs", str(dim - 1), "-fea_kind", "spec",
                "-fea_trap", str(N), "-format_out", "htk"]
        res = cb.extract_features(args, mats)
        for j, m in enumerate(mats):
            want = co.trap_stack_closed_form(m.astype(np.float64), w).astype(np.float32)
            assert np.array_equal(res.utt_features(j), want), (N, j)
        hd = cb.Handle(args)
        plan = hd.plan([m.shape[0] for m in mats])
        x = torch.from_numpy(np.concatenate(mats)).cuda()
        y = torch.empty((plan.total_frames, hd.feature_dim), dtype=torch.float32, device="cuda")
        plan.run_device_fea(x.data_ptr(), y.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(y.cpu().numpy(), res.features)
        plan.close(); hd.close()


def test_feature_input_refusals():
    """Configurations in which the reference crashes or reads memory it never wrote are refused, not imitated."""
    B_ = ["-fs", "16000", "-format_in", "htk", "-format_out", "htk"]
    for extra in (["-fea_kind", "dctc"],                                   # null NR dereferenced, src/io/batch.cc:108
                  ["-fea_kind", "lpc", "-fea_E", "on"],                    # no energy exists
                  ["-fea_kind", "lpc", "-vad_out_mode", "vad"],            # no spectrum for the VAD module
                  ["-fea_kind", "lpc", "-fea_delta", "d", "-fea_ncepcoefs", "20"]):   # the chain reads 21 of 13 columns
        with pytest.raises(cb.CtuError):
            cb.Handle(B_ + extra)
    with pytest.raises(cb.CtuError):
        cb.Handle(B[:2] + ["-format_in", "raw", "-preset", "mfcc", "-fea_kind", "trapdct,11,3", "-fea_delta", "d", "-format_out", "htk"])
    with pytest.raises(cb.CtuError):
        cb.Handle(B + ["-preset", "mfcc", "-fea_trap", "5", "-fea_c0", "off", "-format_out", "htk"])


@pytest.mark.parametrize("name", ["g711_alaw_mfcc_8k", "g711_mulaw_exten_raw_8k", "g711_alaw_plp_16k"])
def test_cuda_g711_input_matches_reference_golden(name):
    """8-bit A-law / mu-law files: the codes are uploaded as they are (one byte per sample over PCIe) and expanded on the
    device (k_g711_expand); results against the reference binary run on the same files."""
    args, alaw, codes = gu.g711_case(name)
    c = gu.Case(name)
    o = co.parse_args(args)
    idx = [i for i in range(len(codes)) if co.num_frames(len(codes[i]), o) >= (4 if o.n_order else 0)]
    res = cb.extract_g711(args, [codes[i] for i in idx], alaw)
    for j, i in enumerate(idx):
        want = c.payload(i)
        if c.kind == "raw":
            got = res.utt_waveform(j)
            d = np.abs(got.astype(np.int32) - want.astype(np.int32))
            assert got.shape == want.shape and d.max() <= 1 and (d > 0).mean() < 0.02, (name, i)
        else:
            check_features(name, i, res.utt_features(j), want, o.fea_kind)


def test_feature_input_random_chains_match_oracle():
    """Random delta / stacking / CMS chains on random feature matrices (dims 5..40, windows 1..4, stacking 3..15 rows, with
    and without the writer's column cut), ragged row counts, 40 option sets: the device against the oracle's state machine."""
    rng = np.random.default_rng(11)
    for it in range(40):
        dim = int(rng.integers(5, 41))
        ncep = int(rng.integers(2, dim))                       # the chain reads ncep+1 <= dim columns
        kind = ["lpc", "spec", "logspec", "lpa"][int(rng.integers(0, 4))]
        args = ["-fs", "16000", "-format_in", "htk", "-nfeacoefs", str(dim), "-fea_ncepcoefs", str(ncep), "-fea_kind", kind, "-format_out", "htk"]
        mode = int(rng.integers(0, 4))
        need = 1
        if mode == 1:
            order = ["d", "d_a", "d_a_t"][int(rng.integers(0, 3))]
            wins = [int(rng.integers(1, 5)) for _ in range(3)]
            args += ["-fea_delta", order, "-d_win", str(wins[0]), "-a_win", str(wins[1]), "-t_win", str(wins[2])]
            need = max(wins[: len(order.split("_"))]) + 2
        elif mode == 2:
            N = int(rng.choice([3, 5, 7, 9, 11, 15]))
            args += ["-fea_trap", str(N)]
            need = (N - 1) // 2 + 2
        elif mode == 3:
            args += ["-fea_delta", "d_a"]
            need = 4
        if mode in (1, 3) and rng.random() < 0.4:
            args += ["-fea_Z_exp", str(int(rng.choice([200, 500, 1500])))]
        if kind == "lpc" and rng.random() < 0.3:
            args += ["-fea_c0", "off"]
        o = co.parse_args(args)
        mats = [rng.standard_normal((int(rng.integers(need, need + 200)), dim)).astype(np.float32) * 3 for _ in range(int(rng.integers(1, 12)))]
        res = cb.extract_features(args, mats)
        for j, m in enumerate(mats):
            want = co.run_features(m, o)
            got = res.utt_features(j)
            assert got.shape == want.shape, (args, j, got.shape, want.shape)
            if mode in (0, 2):
                assert np.array_equal(got, want), (args, j)
            else:
                assert np.all(np.abs(got - want) <= 1e-4 * np.abs(want) + 1e-3), (args, j, float(np.abs(got - want).max()))
