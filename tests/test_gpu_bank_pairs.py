"""k_bank's fused noise-reduction scan on bin pairs.

Inside k_bank the recursion runs on two bins per thread (nr_step2: packed FP32, one MUFU per lane) and bin 256 on the scalar
nr_step; the standalone scan k_nr_scan4 (fuse_nr = 0) runs the scalar nr_step on every bin.  Both are meant to give the same
bits, so every fused configuration -- exten with a = 1 and a = 2, hwss / fwss with a = 1 and a = 2 and 2fwss from a VAD file,
each with MFCC and log-spectrum output -- is run both ways and compared bit for bit.  The batch is ragged: utterances of 1, 7,
8, 31, 32, 33 and 998 frames put partial chunks of eight frames, partial and whole 32-frame tiles through the scan, and with
more utterances than resident CTAs every CTA walks several of them, so the scan state is reset at each utterance's first tile.
One exten case is also held to the oracle."""
import numpy as np
import pytest

import ctu_oracle as co
import ctucopy_b200 as cb
import test_gpu_parity as tp
from ctucopy_b200 import synthetic

RAW = ["-fs", "16000", "-format_in", "raw", "-dither", "0"]
MF = ["-preset", "mfcc", "-preem", "0.97"]
OUTPUTS = {"mfcc": ["-format_out", "htk"], "logspec": ["-fea_kind", "logspec", "-format_out", "htk"]}
SCANS = {
    "exten_a1": ["-nr_mode", "exten", "-nr_a", "1"],
    "exten_a2": ["-nr_mode", "exten", "-nr_a", "2"],
    "hwss_a1": ["-nr_mode", "hwss", "-nr_a", "1", "-vad", "file=vadin.bin"],
    "hwss_a2": ["-nr_mode", "hwss", "-nr_a", "2", "-vad", "file=vadin.bin"],
    "fwss_a1": ["-nr_mode", "fwss", "-nr_a", "1", "-nr_b", "1.5", "-vad", "file=vadin.bin"],
    "fwss_a2": ["-nr_mode", "fwss", "-nr_a", "2", "-vad", "file=vadin.bin"],
    "2fwss": ["-nr_mode", "2fwss", "-nr_initsegs", "5", "-vad", "file=vadin.bin"],
}
CASES = {"%s-%s" % (s, k): RAW + MF + SCANS[s] + OUTPUTS[k] for s in SCANS for k in OUTPUTS}

FRAMES = [1, 7, 8, 31, 32, 33, 998]
COPIES = 100          # 700 utterances: more than the 4 x 148 CTAs of k_bank that are resident on a B200


def ragged_batch():
    """COPIES rounds of the FRAMES lengths, each utterance a different stretch of one of eight 10 s signals"""
    base = [synthetic.utterance(k, 10.0) for k in range(8)]
    utts = []
    for c in range(COPIES):
        for i, T in enumerate(FRAMES):
            n = 400 + 160 * (T - 1)
            b = base[(c + i) % len(base)]
            off = (97 * (7 * c + i)) % (len(b) - n + 1)
            utts.append(b[off: off + n])
    return utts


def ext_vad_for(o, utts, seed):
    """a VAD byte stream for -vad file=: one 0/1 byte per frame, runs of speech and pauses"""
    rng = np.random.default_rng(seed)
    return [np.repeat(rng.integers(0, 2, co.num_frames(len(u), o) // 5 + 1), 5)[: co.num_frames(len(u), o)].astype(np.uint8) for u in utts]


def run(args, utts, ev, fuse):
    hd = cb.Handle(args)
    try:
        hd.set_option("fuse_nr", fuse)
        plan = hd.plan([len(u) for u in utts])
        try:
            hd.profile(True)
            res = plan.run_host(np.ascontiguousarray(np.concatenate(utts)), None if ev is None else np.concatenate(ev))
            names = {n for n, _ in hd.profile_records()}
            hd.profile(False)
            return res, names
        finally:
            plan.close()
    finally:
        hd.close()


# ---- CPU -------------------------------------------------------------------------------------------------------------

def test_ragged_batch_geometry():
    """The batch has the frame counts it is meant to have, and the VAD stream has speech and pauses."""
    o = co.parse_args(CASES["exten_a1-mfcc"])
    utts = ragged_batch()
    assert [co.num_frames(len(u), o) for u in utts] == FRAMES * COPIES
    ev = np.concatenate(ext_vad_for(o, utts, 3))
    assert 0.3 < ev.mean() < 0.7


@pytest.mark.parametrize("name", list(CASES))
def test_fused_configurations_reach_the_device(name):
    """Every configuration here is accepted: without a GPU the handle fails for the missing device only (status 4)."""
    import torch
    if torch.cuda.is_available():
        cb.Handle(CASES[name]).close()
        return
    with pytest.raises(cb.CtuError) as e:
        cb.Handle(CASES[name])
    assert e.value.status == 4, (name, e.value.status, e.value.message)


# ---- GPU -------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_fused_and_standalone_scan_agree_bit_for_bit_on_a_ragged_batch(name):
    args = CASES[name]
    o = co.parse_args(args)
    utts = ragged_batch()
    ev = ext_vad_for(o, utts, 3) if o.vadmode == "file" else None
    a, ka = run(args, utts, ev, 1)
    b, kb = run(args, utts, ev, 0)
    # the two runs took the two paths
    assert "k_bank<nr,fea>" in ka and not any(k.startswith("k_nr_scan") for k in ka), sorted(ka)
    assert "k_nr_scan" in kb and "k_bank<nr,fea>" not in kb, sorted(kb)
    assert list(a.frames_per_utt) == FRAMES * COPIES
    assert a.features.shape == b.features.shape
    diff = a.features.view(np.uint32) != b.features.view(np.uint32)
    assert not diff.any(), (name, "%d of %d values differ, first in row %d" % (diff.sum(), diff.size, int(np.argwhere(diff)[0][0])))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["exten_a1-mfcc", "exten_a2-logspec"])
def test_fused_exten_matches_oracle_on_a_ragged_batch(name):
    """One round of the ragged lengths through the fused scan against the oracle, at the parity bar with the subtraction
    sensitivity term."""
    args = CASES[name]
    o = co.parse_args(args)
    utts = ragged_batch()[: 2 * len(FRAMES)]
    res, names = run(args, utts, None, 1)
    assert "k_bank<nr,fea>" in names
    for j, u in enumerate(utts):
        ref = co.run_pipeline(u, o)
        assert int(res.frames_per_utt[j]) == ref.nframes
        tp.check_features(name, j, res.utt_features(j), ref.features, o.fea_kind, tp._sensitivity(args, o, u))
