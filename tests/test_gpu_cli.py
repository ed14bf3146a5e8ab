"""The C++ command-line host (host/ctucopy_b200) against the reference binary's FILES:
headers, frame counts and container layout byte-exact; payload within the parity
tolerance; and for the fp64 band-domain path the whole container byte-identical."""
import os
import subprocess

import numpy as np
import pytest

import golden_util as gu
import ref_runner as rr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "host", "ctucopy_b200")


def run_cli(tmp, args, utts, vad_out=False, ext_vad=None):
    for i, u in enumerate(utts):
        np.asarray(u).astype("<i2").tofile(os.path.join(tmp, "u%d.raw" % i))
    if ext_vad is not None:
        open(os.path.join(tmp, "vadin.bin"), "wb").write(ext_vad)
    with open(os.path.join(tmp, "list.scp"), "w") as fh:
        for i in range(len(utts)):
            fh.write("%s/u%d.raw %s/u%d.out%s\n" % (tmp, i, tmp, i, (" spk %s/u%d.vad" % (tmp, i)) if vad_out else ""))
    a = [s.replace("{ARK}", os.path.join(tmp, "o.ark")).replace("{PFILE}", os.path.join(tmp, "o.pfile")).replace("{VADIN}", os.path.join(tmp, "vadin.bin"))
         .replace("{FILTERS}", rr.TDIIR_FILTERS) for s in args]
    pr = subprocess.run([EXE] + a + ["-S", os.path.join(tmp, "list.scp")], capture_output=True, cwd=tmp)
    assert pr.returncode == 0, pr.stderr.decode()
    return pr


def test_cli_htk_files(tmp_path):
    for name, be in (("mfcc30_d_a", "<"), ("mfcc26_be", ">")):
        c = gu.Case(name)
        idx = [0, 4, 5]
        run_cli(str(tmp_path), c.args, [gu.inputs()[i] for i in idx])
        for j, i in enumerate(idx):
            got = open(tmp_path / ("u%d.out" % j), "rb").read()
            want = c.raw[i]
            assert len(got) == len(want) and got[:12] == want[:12], (name, i)       # header byte-exact
            a, b = rr.parse_htk(got, be)[1], rr.parse_htk(want, be)[1]
            assert np.all(np.abs(a - b) <= 1e-4 * np.abs(b) + 1e-3)


def test_cli_td_iir_mfcc_files(tmp_path):
    """-fea_kind td-iir-mfcc (SURVEY 8f.4) through the CLI: HTK header byte-exact (parmKind 9 | _0), rows within tolerance.
    Every golden is the FIRST file of a reference process: the reference carries the filter state from file to file, this
    path is defined per utterance (DESIGN 9), so each file of the list below must equal its own one-file golden."""
    c = gu.Case("tdiir_w30s10")
    idx = [0, 4, 5]
    run_cli(str(tmp_path), c.args, [gu.inputs()[i] for i in idx])
    for j, i in enumerate(idx):
        got = open(tmp_path / ("u%d.out" % j), "rb").read()
        want = c.raw[i]
        assert len(got) == len(want) and got[:12] == want[:12], i
        a, b = rr.parse_htk(got)[1], rr.parse_htk(want)[1]
        assert np.all(np.abs(a - b) <= 1e-4 * np.abs(b) + 1e-3), (i, np.abs(a - b).max())


def test_cli_ss_carry_reproduces_the_reference_list_run(tmp_path):
    """-ss_carry on: fwss over a three-file list as ONE reference process writes it (every file's noise estimate starts from
    the enhanced last frame of the file before, src/nr/nr.cc:212-222); without the option the second file differs grossly."""
    args, kind, idx, outs, ev = gu.carry_case("carry_fwss_burg")
    ins = [gu.inputs()[i] for i in idx]
    run_cli(str(tmp_path), args + ["-ss_carry", "on"], ins)
    for j in range(len(idx)):
        got = open(tmp_path / ("u%d.out" % j), "rb").read()
        assert len(got) == len(outs[j]) and got[:12] == outs[j][:12], j
        a, b = rr.parse_htk(got)[1], rr.parse_htk(outs[j])[1]
        assert np.all(np.abs(a - b) <= 1e-4 * np.abs(b) + 2e-3), (j, np.abs(a - b).max())
    run_cli(str(tmp_path), args, ins)
    a, b = rr.parse_htk(open(tmp_path / "u1.out", "rb").read())[1], rr.parse_htk(outs[1])[1]
    assert np.abs(a - b).max() > 1.0
    pr = subprocess.run([EXE] + args + ["-ss_carry", "on", "-gpus", "2", "-S", str(tmp_path / "list.scp")], capture_output=True)
    assert pr.returncode != 0 and b"-ss_carry" in pr.stderr


def test_cli_pfile_band_domain_path_is_byte_identical(tmp_path):
    c = gu.Case("fwss_file_afterFB_pfile")
    for i in (0, 4):
        run_cli(str(tmp_path), c.args, [gu.inputs()[i]], ext_vad=c.extvad[i].tobytes())
        assert open(tmp_path / "o.pfile", "rb").read() == c.raw[i]


def test_cli_ark_scp_and_multi_sentence_pfile(tmp_path):
    c = gu.Case("plpc_ark")
    ins = [gu.inputs()[i] for i in (0, 1, 4)]
    run_cli(str(tmp_path), c.args, ins)
    ark = open(tmp_path / "o.ark", "rb").read()
    mats = rr.parse_ark(ark)
    assert list(mats) == [str(tmp_path / ("u%d.out" % j)) for j in range(3)]
    scp = open(tmp_path / "o.scp").read().splitlines()
    for line, key in zip(scp, mats):
        k, loc = line.split(" ")
        off = int(loc.rsplit(":", 1)[1])
        assert k == key and ark[off: off + 5] == b"\x00BFM "
    for j, i in enumerate((0, 1, 4)):
        want = c.payload(i)
        got = mats[str(tmp_path / ("u%d.out" % j))]
        assert got.shape == want.shape and np.all(np.abs(got - want) <= 1e-4 * np.abs(want) + 1e-3)
    c = gu.Case("fwss_burg_pfile")
    run_cli(str(tmp_path), c.args, ins)
    meta, feat = rr.parse_pfile(open(tmp_path / "o.pfile", "rb").read())
    T = [c.payload(i).shape[0] for i in (0, 1, 4)]
    assert list(meta["table"]) == [0, T[0], T[0] + T[1], sum(T)]
    assert np.array_equal(meta["sent_id"], np.repeat([0, 1, 2], T))
    want = np.concatenate([c.payload(i) for i in (0, 1, 4)])
    assert np.all(np.abs(feat - want) <= 1e-4 * np.abs(want) + 1e-3)
    assert "-num_sentences 3\n" in meta["header"] and ("-num_frames %d\n" % sum(T)) in meta["header"]


def test_cli_vad_debug_side_files(tmp_path):
    """-vad_out_mode debug through the CLI: the same set of side files as the reference binary (names = <vadfile>_<suffix>),
    flag files byte-identical, doubles within the device's resolution."""
    for name in ("vaddbg_perc", "vaddbg_adapt_cepdist_lpc"):
        c = gu.Case(name)
        idx = [0, 4, 5]
        run_cli(str(tmp_path), c.args, [gu.inputs()[i] for i in idx], vad_out=True)
        for j, i in enumerate(idx):
            want = c.debug[i]
            have = sorted(f[len("u%d.vad_" % j):] for f in os.listdir(tmp_path) if f.startswith("u%d.vad_" % j))
            assert have == sorted(want), (name, i, have)
            assert open(tmp_path / ("u%d.vad" % j), "rb").read() == c.aux[i], (name, i, "decision file")
            for suf, wb in want.items():
                gb = open(tmp_path / ("u%d.vad_%s" % (j, suf)), "rb").read()
                assert len(gb) == len(wb), (name, i, suf)
                if suf in ("vad0", "c0init", "init"):
                    assert gb == wb, (name, i, suf)
                else:
                    np.testing.assert_allclose(np.frombuffer(gb, "<f8"), np.frombuffer(wb, "<f8"), rtol=2e-5, atol=1e-6)
        for f in os.listdir(tmp_path):
            os.remove(tmp_path / f)


def test_cli_waveform_and_vad_files(tmp_path):
    for name in ("exten_raw", "exten_wave_a1"):
        c = gu.Case(name)
        run_cli(str(tmp_path), c.args, [gu.inputs()[1]])
        got = open(tmp_path / "u0.out", "rb").read()
        want = c.raw[1]
        assert len(got) == len(want)
        hdr = 44 if c.kind == "wave" else 0
        assert got[:hdr] == want[:hdr]
        d = np.abs(np.frombuffer(got[hdr:], "<i2").astype(int) - np.frombuffer(want[hdr:], "<i2").astype(int))
        assert d.max() <= 1
    c = gu.Case("vad_energy_dyn_drop")
    run_cli(str(tmp_path), c.args, [gu.inputs()[4]], vad_out=True)
    assert open(tmp_path / "u0.vad", "rb").read() == c.aux[4]                     # '0'/'1' per frame, byte-exact
    got = open(tmp_path / "u0.out", "rb").read()
    assert got[:12] == c.raw[4][:12]                                              # nSamples after drop


def test_cli_errors_like_the_reference(tmp_path):
    pr = subprocess.run([EXE, "-fs", "16000", "-preset", "mfcc", "-format_in", "raw", "-format_out", "htk", "-S", "/nonexistent"], capture_output=True)
    assert pr.returncode == 255 and b"BATCH: Cannot open list file!" in pr.stderr
    np.zeros(100, "<i2").tofile(tmp_path / "s.raw")
    (tmp_path / "l.scp").write_text("%s/s.raw %s/s.out\n" % (tmp_path, tmp_path))
    pr = subprocess.run([EXE, "-fs", "16000", "-preset", "mfcc", "-format_in", "raw", "-format_out", "htk", "-S", str(tmp_path / "l.scp")], capture_output=True)
    assert pr.returncode == 255 and b"IO: Signal shorter than one frame!" in pr.stderr


def test_cli_sharded_run_merges_to_the_single_process_files(tmp_path):
    """-shard r/N (one process per GPU; both shards on device 0 here) + -merge N gives the
    same ark / scp / pfile bytes and the same per-utterance HTK files as one process."""
    ins = [gu.inputs()[i] for i in (0, 4, 1, 5, 2)]
    for fmt in ("ark={ARK}", "pfile={PFILE}"):
        args = ["-fs", "16000", "-format_in", "raw", "-dither", "0", "-preset", "plpc", "-format_out", fmt]
        one, two = tmp_path / ("one_" + fmt[:3]), tmp_path / ("two_" + fmt[:3])
        one.mkdir(); two.mkdir()
        run_cli(str(one), args, ins)
        for r in range(2):
            run_cli(str(two), args + ["-shard", "%d/2" % r, "-device", "0"], ins)
        a = [s.replace("{ARK}", str(two / "o.ark")).replace("{PFILE}", str(two / "o.pfile")) for s in args]
        pr = subprocess.run([EXE] + a + ["-merge", "2"], capture_output=True)
        assert pr.returncode == 0, pr.stderr.decode()
        for fn in ("o.ark", "o.scp", "o.pfile"):
            if (one / fn).exists():
                got = open(two / fn, "rb").read().replace(str(two).encode(), b"@")
                want = open(one / fn, "rb").read().replace(str(one).encode(), b"@")
                assert got == want, fn
        assert not [f for f in os.listdir(two) if f.startswith("shard")]


def _stat_numbers(text):
    names, vals = [], []
    for ln in text.splitlines():
        tok = ln.split()
        if tok and tok[0] in ("mean", "var"):
            vals.append([float(x) for x in tok[1:]])
        elif tok:
            names.append(tok[0])
    return names, np.array(vals)


@pytest.mark.parametrize("name", ["cmvn_3stage_d_a", "cmvn_stat_plp", "cmvn_3stage_trap3", "cmvn_3stage_logspec_d",
                                  "cmvnfea_3stage_d", "cmvnfea_3stage_copy", "cmvnfea_stat_trap3"])
def test_cli_cmvn_statistics_and_normalised_features(tmp_path, name):
    """List-mode CMVN through the CLI against the reference binary's statistics file and feature files (sample input, and
    HTK feature files in: the cmvnfea_* cases)."""
    args, idx, spk, stat, outs = gu.cmvn_case(name)
    ins = gu.inputs()
    src = gu.Case("mfcc30_static") if name.startswith("cmvnfea") else None
    for i in idx:
        if src is not None:
            open(tmp_path / ("u%d.raw" % i), "wb").write(src.raw[i])      # an HTK parameter file, whatever its name
        else:
            ins[i].astype("<i2").tofile(tmp_path / ("u%d.raw" % i))
    with open(tmp_path / "list.scp", "w") as fh:
        for i, sp in zip(idx, spk):
            fh.write("%s/u%d.raw %s/u%d.htk %s\n" % (tmp_path, i, tmp_path, i, sp))
    a = [x.replace("{STAT}", str(tmp_path / "cmvn.stat")) for x in args]
    pr = subprocess.run([EXE] + a + ["-S", str(tmp_path / "list.scp")], capture_output=True)
    assert pr.returncode == 0, pr.stderr.decode()
    names, vals = _stat_numbers(open(tmp_path / "cmvn.stat").read())
    rnames, rvals = _stat_numbers(stat)
    assert names == rnames and vals.shape == rvals.shape
    np.testing.assert_allclose(vals, rvals, rtol=2e-4, atol=2e-4)
    for i in idx:
        if i in outs:
            got = open(tmp_path / ("u%d.htk" % i), "rb").read()
            assert got[:12] == outs[i][:12]
            g, w = rr.parse_htk(got)[1], rr.parse_htk(outs[i])[1]
            # north_star tolerance for log-domain features; the division by a small variance (deltas) scales absolute errors up
            assert np.all(np.abs(g - w) <= 1e-4 * np.abs(w) + 1e-3), float(np.abs(g - w).max())
        else:
            assert not (tmp_path / ("u%d.htk" % i)).exists()
    # applying from an existing statistics file is refused (the reference writes +-inf there)
    if "-apply_cmvn" in args:
        pr = subprocess.run([EXE] + a + ["-S", str(tmp_path / "list.scp")], capture_output=True)
        assert pr.returncode == 255 and b"existing statistics file" in pr.stderr


def test_cli_cmvn_under_gpus_is_the_single_process_result(tmp_path):
    """CMVN with -gpus 2 (two worker threads and handles; both on device 0 when the box has one GPU): per-utterance column
    sums are added on the host in list order, so the statistics file and the normalised feature files are BYTE-identical
    to the one-GPU run, whatever the split."""
    args, idx, spk, stat, outs = gu.cmvn_case("cmvn_3stage_d_a")
    ins = gu.inputs()
    many = idx * 6                                   # 24 utterances, 4 speakers' worth of repeats
    res = {}
    for g in (1, 2):
        d = tmp_path / ("g%d" % g); d.mkdir()
        for n, i in enumerate(many):
            ins[i].astype("<i2").tofile(d / ("u%d.raw" % n))
        with open(d / "list.scp", "w") as fh:
            for n, i in enumerate(many):
                fh.write("%s/u%d.raw %s/u%d.htk %s\n" % (d, n, d, n, spk[idx.index(i)] + str(n % 3)))
        a = [x.replace("{STAT}", str(d / "cmvn.stat")) for x in args]
        env = dict(os.environ, CTU_CMVN_BATCH_SAMPLES="60000")       # several batches, so that both workers get some
        pr = subprocess.run([EXE] + a + ["-S", str(d / "list.scp")] + (["-gpus", "2"] if g == 2 else []), capture_output=True, env=env)
        assert pr.returncode == 0, pr.stderr.decode()
        res[g] = (open(d / "cmvn.stat", "rb").read(), [open(d / ("u%d.htk" % n), "rb").read() for n in range(len(many))])
    assert res[1][0] == res[2][0], "statistics text differs between -gpus 1 and -gpus 2"
    assert res[1][1] == res[2][1], "normalised features differ between -gpus 1 and -gpus 2"


def test_cli_feature_file_input_and_stacking_headers(tmp_path):
    """-format_in htk through the command line: stacked rows byte-identical to the reference's files (a pure gather), delta
    rows within tolerance with byte-exact headers -- including the reference's parmKind quirks (the decimal "T bit", and
    "spec" as the kind of every file after the first with -fea_trap on sample input)."""
    tmp = str(tmp_path)
    for name in ("feain_spec_trap5", "feain_trap3_be", "feain_copy", "feain_dctc_d_a_t_noc0", "feain_lpc_d_cms"):
        c = gu.Case(name)
        src = gu.Case(c.source)
        idx = [0, 4, 5]
        with open(os.path.join(tmp, "list.scp"), "w") as fh:
            for j, i in enumerate(idx):
                open(os.path.join(tmp, "f%d.htk" % j), "wb").write(src.raw[i])
                fh.write("%s/f%d.htk %s/g%d.htk\n" % (tmp, j, tmp, j))
        pr = subprocess.run([EXE] + c.args + ["-S", os.path.join(tmp, "list.scp")], capture_output=True, cwd=tmp)
        assert pr.returncode == 0, pr.stderr.decode()
        be = ">" if c.kind == "htk_be" else "<"
        for j, i in enumerate(idx):
            got, want = open(os.path.join(tmp, "g%d.htk" % j), "rb").read(), c.raw[i]
            assert len(got) == len(want) and got[:12] == want[:12], (name, i)
            if "trap" in name or name == "feain_copy":
                assert got == want, (name, i)
            else:
                a, b = rr.parse_htk(got, be)[1], rr.parse_htk(want, be)[1]
                assert np.all(np.abs(a - b) <= 1e-4 * np.abs(b) + 1e-3), (name, i)
    # sample input + stacking, several files in one list: the reference writes each file's rows as a one-file run does
    # (the mfcc_trap5 golden), and base kind 8 ("spec") into the header of every file after the first, which its own list
    # run with -fea_trap in the cmvn_3stage_trap3 golden records
    _, lidx, _, _, louts = gu.cmvn_case("cmvn_3stage_trap3")
    kinds = [rr.parse_htk(louts[i])[0]["kind"] for i in lidx]
    assert kinds[0] & 0x3f == 6 and all(k & 0x3f == 8 for k in kinds[1:]), kinds
    c = gu.Case("mfcc_trap5")
    idx = [0, 4, 5]
    run_cli(tmp, c.args, [gu.inputs()[i] for i in idx])
    for j, i in enumerate(idx):
        got, want = open(os.path.join(tmp, "u%d.out" % j), "rb").read(), c.raw[i]
        meta, a = rr.parse_htk(got)
        wmeta, b = rr.parse_htk(want)
        assert len(got) == len(want) and got[:10] == want[:10], (j, got[:12], want[:12])
        assert meta["kind"] == (wmeta["kind"] if j == 0 else (wmeta["kind"] & ~0x3f) | 8), ("parmKind of file %d" % j, meta["kind"])
        assert np.all(np.abs(a - b) <= 1e-4 * np.abs(b) + 1e-3)


def test_cli_g711_files(tmp_path):
    """-format_in alaw / mulaw through the command line (codes expanded on the GPU) against the reference's files."""
    tmp = str(tmp_path)
    for name in ("g711_alaw_mfcc_8k", "g711_mulaw_exten_raw_8k"):
        args, alaw, codes = gu.g711_case(name)
        c = gu.Case(name)
        idx = [0, 4, 5]
        with open(os.path.join(tmp, "list.scp"), "w") as fh:
            for j, i in enumerate(idx):
                codes[i].tofile(os.path.join(tmp, "c%d.al" % j))
                fh.write("%s/c%d.al %s/c%d.out\n" % (tmp, j, tmp, j))
        pr = subprocess.run([EXE] + args + ["-S", os.path.join(tmp, "list.scp")], capture_output=True, cwd=tmp)
        assert pr.returncode == 0, pr.stderr.decode()
        for j, i in enumerate(idx):
            got, want = open(os.path.join(tmp, "c%d.out" % j), "rb").read(), c.raw[i]
            assert len(got) == len(want), (name, i)
            if c.kind == "raw":
                d = np.abs(np.frombuffer(got, "<i2").astype(np.int32) - np.frombuffer(want, "<i2").astype(np.int32))
                assert d.max() <= 1
            else:
                assert got[:12] == want[:12]
                a, b = rr.parse_htk(got)[1], rr.parse_htk(want)[1]
                assert np.all(np.abs(a - b) <= 1e-4 * np.abs(b) + 1e-3)
