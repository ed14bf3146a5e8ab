"""The persistent frame kernels past their first tile.

k_frames2, k_frames256 and k_bank are launched with as many CTAs as are resident at once, and every CTA then walks the
tile list (or, for k_bank, the utterance list) with a stride of the grid size.  What only happens from a CTA's second tile
on -- the descriptors fetched ahead (TileAhead), the cp.async prefetch of the next tile's samples with the pre-emphasis
memory in a register, k_bank's mbarrier phases and the reset of its scan state at each utterance -- is exercised here on
batches of several tiles per CTA:
  * a vectorised fp64 restatement of rawIN::get_frame, held to the oracle's per-frame loop (no GPU needed);
  * every PCM -> spectrum front end through the kernel tap ctu_debug_spectrum, on ragged batches that put every utterance
    offset phase, every last-tile length, full-scale samples and single impulses at tile edges through the staging, with
    the device PCM starting at each of the eight 2-byte phases of a 16-byte chunk;
  * the bench.py workloads on benchmark-scale ragged batches through ctu_plan_run_device: repeated utterances must come
    out bit for bit alike, the three entry points must agree bit for bit, and one copy of each distinct signal must match
    the oracle.
"""
import importlib.util
import os

import numpy as np
import pytest

import ctu_oracle as co
import ctucopy_b200 as cb
import test_gpu_parity as tp
from ctucopy_b200 import synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- 1. fp64 reference front end -------------------------------------------------------------------------------------

def ref_spectrum(pcm, o):
    """rawIN::get_frame (src/io/in.cc:305-419) for a whole utterance at once: framing, pre-emphasis with memory 0 at the
    utterance start, the reference's Hamming window, removal of the windowed frame's mean with the 1e-10 floor on bin 0,
    zero padding to wfft, power or (-fb_power off) magnitude.  Same as co.front_end(...).Xabs without its per-frame loop;
    -dither and -remove_dc1 are not covered."""
    assert o.dither == 0.0 and not o.remove_dc1
    w, s = o.window, o.wshift
    x = np.asarray(pcm, dtype=np.float64)
    T = co.num_frames(len(x), o)
    fr = x[np.arange(T)[:, None] * s + np.arange(w)[None, :]]
    alpha = float(np.float32(o.preem))
    if alpha > 0.0:
        prev = np.empty_like(fr)
        prev[:, 1:] = fr[:, :-1]
        prev[:, 0] = np.concatenate([[0.0], x[np.arange(1, T) * s - 1]]) if T else 0.0
        fr = fr - alpha * prev
    y = co.hamming(w)[None, :] * fr
    if o.remove_dc:
        y = y - y.sum(axis=1, keepdims=True) / w
    F = np.fft.rfft(y, n=o.wfft, axis=1)
    P = F.real * F.real + F.imag * F.imag
    if o.remove_dc:
        P[:, 0] = 1e-10
    return P if o.fb_power else np.sqrt(P)


# geometry -> kernel (ctu_api.cu: launch_frames_t picks the 400 / 512 specialisation by window length, launch_frames_w takes
# k_frames256 when fast256() holds and k_frames_any for every FFT size other than 512 points)
GEOMETRIES = {
    "400_160": ["-fs", "16000", "-w", "25", "-s", "10"],        # k_frames2<400,false>, window values in shared memory
    "400_159": ["-fs", "16000", "-w", "25", "-s", "9.9375"],    # k_frames2<400,false>, odd shift: scalar sample loads
    "512_256": ["-fs", "16000", "-w", "32", "-s", "16"],        # k_frames2<512,false>
    "512_128": ["-fs", "16000", "-w", "32", "-s", "8"],         # k_frames2<512,false>
    "320_160": ["-fs", "16000", "-w", "20", "-s", "10"],        # k_frames2<0,false>
    "480_160": ["-fs", "16000", "-w", "30", "-s", "10"],        # k_frames2<0,false>
    "441_221": ["-fs", "22050", "-w", "20", "-s", "10"],        # k_frames2<0,false>, odd window and shift
    "353_176": ["-fs", "11025", "-w", "32", "-s", "16"],        # k_frames2<0,false>, odd window
    "200_80": ["-fs", "8000", "-w", "25", "-s", "10"],          # k_frames256 (front256=1) / k_frames_any (front256=0)
    "1103_441": ["-fs", "44100", "-w", "25", "-s", "10"],       # k_frames_any, 2048 points
}
BASE = ["-format_in", "raw", "-dither", "0", "-preset", "mfcc", "-format_out", "htk"]


def _onoff(v):
    return "on" if v else "off"


def spectrum_args(geom, preem, remove_dc, fb_power):
    return BASE + GEOMETRIES[geom] + ["-preem", str(preem), "-remove_dc", _onoff(remove_dc), "-fb_power", _onoff(fb_power)]


def full_scale_signal(n, rng, fs):
    """Runs of -32768, runs of 32767, alternating +-full scale, uniform int16 over the whole range and speech-like
    synthetic audio, in random order and lengths."""
    out = np.empty(n, dtype=np.int16)
    i = 0
    while i < n:
        m = min(n - i, int(rng.integers(30, 700)))
        kind = int(rng.integers(0, 5))
        if kind == 0:
            out[i:i + m] = -32768
        elif kind == 1:
            out[i:i + m] = 32767
        elif kind == 2:
            out[i:i + m] = np.where(np.arange(m) % 2 == int(rng.integers(0, 2)), 32767, -32768)
        elif kind == 3:
            out[i:i + m] = rng.integers(-32768, 32768, m)
        else:
            out[i:i + m] = synthetic.utterance(int(rng.integers(0, 30)), (m + 1) / fs, fs)[:m]
        i += m
    return out


@pytest.mark.parametrize("geom", list(GEOMETRIES))
def test_reference_front_end_matches_oracle(geom):
    """The vectorised reference against co.front_end (the oracle's frame-by-frame restatement of the reference binary),
    with and without pre-emphasis and DC removal, power and magnitude, to 1e-12 relative (plus 1e-12 of the row maximum:
    the two sum the frame in different orders)."""
    rng = np.random.default_rng(7)
    for preem, dc, power in ((0.97, True, True), (0.0, True, False), (0.97, False, False), (0.0, False, True)):
        o = co.parse_args(spectrum_args(geom, preem, dc, power))
        w, s = o.window, o.wshift
        ins = [synthetic.utterance(3, 0.25, o.fs)[: w - s + 11 * s + 5],
               full_scale_signal(w - s + 7 * s + s - 1, rng, o.fs),
               np.zeros(w - s + 3 * s, np.int16)]
        for u in ins:
            want = co.front_end(u, o).Xabs
            got = ref_spectrum(u, o)
            assert got.shape == want.shape and want.shape[0] == co.num_frames(len(u), o)
            rowmax = want.max(axis=1, keepdims=True)
            assert np.all(np.abs(got - want) <= 1e-12 * (want + rowmax)), (geom, preem, dc, power)


# ---- 2. staging phases of every PCM -> spectrum front end ---------------------------------------------------------------

# (geometry, -preem, -remove_dc, -fb_power, front256): a covering set of the options over the kernel instantiations
STAGING = [
    ("400_160", 0.97, True, True, 1),
    ("400_159", 0.97, False, False, 1),
    ("512_256", 0.97, True, False, 1),
    ("512_128", 0.0, True, True, 1),
    ("320_160", 0.97, False, True, 1),
    ("480_160", 0.0, False, False, 1),
    ("441_221", 0.97, True, True, 1),
    ("353_176", 0.97, True, False, 1),
    ("200_80", 0.97, True, True, 1),
    ("200_80", 0.0, False, False, 0),
    ("1103_441", 0.97, False, True, 1),
]


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def staging_batch(o, min_tiles, rng):
    """A ragged list for the front end's tile walk.  Zero-frame spacers of w-s .. w-1 random samples put the next utterance
    at a chosen offset mod 8 (the 2-byte phase of its samples in a 16-byte chunk, before the buffer's own phase is added).
    Each round takes every (offset mod 8, frames in the last 16-frame tile) pair once, with random whole tiles in front and
    0 .. s-1 samples after the last frame; the content is full-scale mixes or speech-like audio.  Then all-zero utterances
    with one full-scale impulse: on the last sample before a tile (t0 s - 1), on the first sample of a tile (t0 s) or on the
    last sample of a frame.  Returns (utterances, impulse position or None per utterance)."""
    w, s = o.window, o.wshift
    utts, imp = [], []
    off = [0]

    def add(u, p=None):
        utts.append(u); imp.append(p); off[0] += len(u)

    def phase_to(ph):
        add(rng.integers(-32768, 32768, w - s + (ph - off[0] - (w - s)) % 8).astype(np.int16))

    tiles = 0
    while tiles < min_tiles:
        for r in range(1, 17):
            for ph in rng.permutation(8):
                nf = 16 * int(rng.integers(0, 8)) + r
                n = w - s + nf * s + int(rng.integers(0, s))
                phase_to(ph)
                if rng.random() < 0.5:
                    add(full_scale_signal(n, rng, o.fs))
                else:
                    add(synthetic.utterance(int(rng.integers(0, 60)), (n + 1) / o.fs, o.fs)[:n])
                tiles += (nf + 15) // 16
    for kind in range(3):
        for ph in range(8):
            nf = 40 + 3 * ph
            if kind == 0:
                p = 16 * s * (1 + ph % 2) - 1
            elif kind == 1:
                p = 16 * s * (1 + ph % 2)
            else:
                p = (15 if ph % 2 else nf - 1) * s + w - 1
            u = np.zeros(w - s + nf * s + int(rng.integers(0, s)), np.int16)
            u[p] = 32767 if (ph + kind) % 2 else -32768
            phase_to(ph)
            add(u, p)
    return utts, imp


@pytest.mark.gpu
@pytest.mark.parametrize("geom,preem,dc,power,front256", STAGING, ids=["%s-preem%g-dc%d-pow%d-f256_%d" % c for c in STAGING])
def test_front_end_staging_phases_match_reference(geom, preem, dc, power, front256):
    import torch
    args = spectrum_args(geom, preem, dc, power)
    o = co.parse_args(args)
    w, s = o.window, o.wshift
    rng = np.random.default_rng(sum(map(ord, geom)) + 17 * front256)
    min_tiles = 3 * 8 * _sms()
    utts, imp = staging_batch(o, min_tiles, rng)
    hd = cb.Handle(args)
    hd.set_option("front256", front256)
    plan = hd.plan([len(u) for u in utts])
    fpu = plan.frames_per_utt
    # several tiles per persistent CTA: at least three times as many 16-frame tiles as the largest grid (eight CTAs per SM)
    assert int(((fpu + 15) // 16).sum()) >= min_tiles
    assert (fpu == 0).sum() >= 128 + 24 and set(((fpu + 15) % 16 + 1)[fpu > 0]) == set(range(1, 17))
    pcm = np.concatenate(utts)
    total = len(pcm)
    d_pcm = torch.from_numpy(pcm).cuda()
    stream = torch.cuda.current_stream().cuda_stream
    nb = o.wfftby2
    first = None
    for k in range(8):
        # the device samples start at element k of the buffer: the 16-byte phase comes from the real address
        buf = torch.zeros(total + 16, dtype=torch.int16, device="cuda")
        buf[k:k + total].copy_(d_pcm)
        d_spec = torch.full((plan.total_frames, nb), float("nan"), dtype=torch.float32, device="cuda")
        assert buf.data_ptr() % 16 == 0
        assert hd.L.ctu_debug_spectrum(plan.p, buf.data_ptr() + 2 * k, d_spec.data_ptr(), stream) == 0
        if first is None:
            first = d_spec
        else:
            # every phase stages the same values with the same arithmetic: bit-identical spectra
            same = torch.equal(d_spec.view(torch.int32), first.view(torch.int32))
            assert same, (geom, "buffer phase %d differs from phase 0 at %d values" % (k, int((d_spec != first).sum())))
    got_all = first.cpu().numpy()
    # bin 0 of a frame of zeros: the 1e-10 floor in fp32 (its square root for magnitudes), or 0 without DC removal
    floor = (np.float32(1e-10) if power else np.sqrt(np.float32(1e-10))) if dc else np.float32(0.0)
    for j, u in enumerate(utts):
        r0, T = int(plan.row_offsets[j]), int(fpu[j])
        if T == 0:
            continue
        got, want = got_all[r0:r0 + T], ref_spectrum(u, o)
        if imp[j] is not None:
            # frames that hold neither the impulse nor (pre-emphasis) the sample after it are exactly zero but for the floor
            p = imp[j]
            t = np.arange(T)
            hit = (t * s <= p) & (p < t * s + w)
            if preem > 0:
                hit |= (t * s <= p + 1) & (p + 1 < t * s + w)
            quiet = got[~hit]
            wrong = np.any(quiet[:, 1:] != 0, axis=1) | (quiet[:, 0] != floor)
            assert not wrong.any(), (geom, j, "impulse at %d: frames %s are not zero" % (p, np.nonzero(~hit)[0][wrong][:8]))
        # magnitude domain
        got = got.astype(np.float64)
        if power:
            got, want = np.sqrt(got), np.sqrt(want)
        rowmax = want.max(axis=1, keepdims=True)
        err = np.abs(got - want)
        bad = ~(err <= 1e-4 * want + 2e-6 * rowmax)                 # (a NaN, from a row never written, is bad too)
        assert not bad.any(), (geom, j, "offset %d mod 8, %d frames: %d values off, first frame %d" %
                               (int(plan.offsets[j]) % 8, T, int(bad.sum()), int(np.nonzero(bad.any(axis=1))[0][0])))
    plan.close(); hd.close()


# ---- 3. benchmark-scale ragged batches through ctu_plan_run_device -------------------------------------------------------

def _bench_module():
    spec = importlib.util.spec_from_file_location("ctu_bench", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


BENCH_NAMES = ["mfcc_exten", "mfcc_d_a", "plp", "trapdct", "exten", "fwss_burg", "tdiir", "mfcc_trap5"]
MFCC_EXTEN_8K = ["-fs", "8000", "-format_in", "raw", "-dither", "0", "-preset", "mfcc", "-preem", "0.97", "-nr_mode", "exten",
                 "-fea_delta", "d_a", "-format_out", "htk"]


def _workload_args(name):
    return MFCC_EXTEN_8K if name == "mfcc_exten_8k" else list(_bench_module().WORKLOADS[name][0])


N_BASE = 24


def bench_batch(o, sms, rng):
    """About 1300 utterances (0.3 .. 1.5 s, ragged) with spacers.  N_BASE distinct base signals (two of them 10 s long)
    appear three times each: once in every third of the list, the first copy at an even offset, the second at an odd one,
    the third at either.  Spacers are zero-frame entries, or in chains with deltas / stacking the shortest utterances they
    accept; a spacer of odd or even length in front of a copy sets the parity of its offset.  Returns (utterances,
    {base: [list index of each copy]})."""
    w, s, fs = o.window, o.wshift, o.fs
    mw = max([o.d_win, o.a_win, o.t_win][: o.n_order]) if o.n_order > 0 else -2
    spacer0 = w - s + (mw + 2) * s                        # zero frames, or delta window + 2 frames

    def slen():
        return int(rng.integers(int(0.3 * fs), int(1.5 * fs)))

    bases = [synthetic.utterance(200 + b, 10.0 if b < 2 else 1.6, fs)[: 10 * fs - int(rng.integers(0, s)) if b < 2 else slen()]
             for b in range(N_BASE)]
    pool = [synthetic.utterance(300 + k, 30.0, fs) for k in range(4)]
    thirds = []
    for c in range(3):
        items = [("f", None)] * 410 + [("c", b) for b in range(N_BASE)]
        thirds.append([items[i] for i in rng.permutation(len(items))])
    utts, where, off = [], {b: [] for b in range(N_BASE)}, 0
    for c, items in enumerate(thirds):
        for kind, b in items:
            if kind == "c":
                want = (0, 1, b % 2)[c]
                sp = spacer0 + ((off + spacer0) % 2 != want)           # odd extra sample flips the parity
                utts.append(rng.integers(-3000, 3000, sp).astype(np.int16)); off += sp
                where[b].append(len(utts))
                utts.append(bases[b]); off += len(bases[b])
            else:
                if rng.random() < 0.45:
                    sp = spacer0 + int(rng.integers(0, 2))
                    utts.append(rng.integers(-3000, 3000, sp).astype(np.int16)); off += sp
                n = slen()
                src = pool[int(rng.integers(0, len(pool)))]
                a = int(rng.integers(0, len(src) - n))
                utts.append(src[a:a + n]); off += n
    return utts, where


def _chunks_of(lengths, chunk_mb):
    """Number of chunks ctu_plan_run_host cuts the list into (utterances up to chunk_mb << 19 samples, at least one)."""
    lim, n, u0, offs = chunk_mb << 19, 0, 0, np.concatenate([[0], np.cumsum(lengths)])
    while u0 < len(lengths):
        u1 = u0 + 1
        while u1 < len(lengths) and offs[u1 + 1] - offs[u0] <= lim:
            u1 += 1
        u0, n = u1, n + 1
    return n


@pytest.mark.gpu
@pytest.mark.parametrize("name", BENCH_NAMES + ["mfcc_exten_8k"])
def test_benchmark_scale_ragged_batch_through_run_device(name):
    import torch
    args = _workload_args(name)
    o = co.parse_args(args)
    sms = _sms()
    rng = np.random.default_rng(sum(map(ord, name)))
    utts, where = bench_batch(o, sms, rng)
    lens = [len(u) for u in utts]
    hd = cb.Handle(args)
    plan = hd.plan(lens)
    fpu = plan.frames_per_utt
    # every k_bank CTA (four per SM) owns several utterances and 32-frame tiles: several mbarrier phases and scan resets
    assert len(utts) >= 3 * 4 * sms and int(((fpu + 31) // 32).sum()) >= 3 * 4 * sms
    assert int((fpu > 0).sum()) >= 2 * 4 * sms
    pcm = np.ascontiguousarray(np.concatenate(utts))
    sig = hd.signal_output
    nfr = plan.total_frames
    d_pcm = torch.from_numpy(pcm).cuda()
    d_vnr = torch.zeros(nfr, dtype=torch.uint8, device="cuda")
    d_vout = torch.zeros(nfr, dtype=torch.uint8, device="cuda")
    if sig:
        d_out = torch.empty(plan.total_output_samples, dtype=torch.int16, device="cuda")
        plan.run_device(d_pcm.data_ptr(), d_waveform=d_out.data_ptr(), d_vad_nr=d_vnr.data_ptr(), d_vad_out=d_vout.data_ptr(),
                        stream=torch.cuda.current_stream().cuda_stream)
    else:
        d_out = torch.empty((nfr, hd.feature_dim), dtype=torch.float32, device="cuda")
        plan.run_device(d_pcm.data_ptr(), d_features=d_out.data_ptr(), d_vad_nr=d_vnr.data_ptr(), d_vad_out=d_vout.data_ptr(),
                        stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    out, vnr, vout = d_out.cpu().numpy(), d_vnr.cpu().numpy(), d_vout.cpu().numpy()
    have_vadnr = o.nr_mode in ("hwss", "fwss", "2fwss")
    do_vad = o.vad_apply_mode != "none" or o.vad_out_mode != "none"
    rows = plan.rows_per_utt()
    ro = np.concatenate([[0], np.cumsum(rows)])

    def utt_out(res_out, j):
        if sig:
            return res_out[int(plan.wave_offsets[j]): int(plan.wave_offsets[j + 1])]
        return res_out[int(ro[j]): int(ro[j + 1])]

    def bits(a):
        return a.view(np.uint32) if a.dtype == np.float32 else a

    # 1. copies: the same samples at offsets of either parity, anywhere in the list, give the same bits
    for b, js in where.items():
        j0 = js[0]
        f0 = slice(int(plan.row_offsets[j0]), int(plan.row_offsets[j0]) + int(fpu[j0]))
        for j in js[1:]:
            assert fpu[j] == fpu[j0] and np.array_equal(bits(utt_out(out, j)), bits(utt_out(out, j0))), (name, b, j0, j)
            f = slice(int(plan.row_offsets[j]), int(plan.row_offsets[j]) + int(fpu[j]))
            assert np.array_equal(vnr[f], vnr[f0]) and np.array_equal(vout[f], vout[f0]), (name, b, j0, j, "decisions")
    # 2. entry points: the host entry point in one chunk and, with chunk_mb=1, in many chunks on three streams
    assert name == "tdiir" or _chunks_of(lens, 1) >= 6             # (td-iir-mfcc keeps 20 utterances per SM in a chunk)
    for chunk_mb in (None, 1):
        if chunk_mb:
            hd.set_option("chunk_mb", chunk_mb)
        res = plan.run_host(pcm)
        got = res.waveform if sig else res.features
        assert np.array_equal(bits(got), bits(out)), (name, chunk_mb, "run_host differs from run_device")
        # (the detector's decisions exist for hwss / fwss / 2fwss, the VAD module's when it is on)
        assert not have_vadnr or np.array_equal(res.vad_nr, vnr), (name, chunk_mb, "detector decisions")
        assert not do_vad or np.array_equal(res.vad_out, vout), (name, chunk_mb, "VAD decisions")
    # 3. the oracle, on the copy in the last third of the list
    for b, js in where.items():
        j = js[2]
        u = utts[j]
        ref = co.run_pipeline(u, o)
        assert int(fpu[j]) == ref.nframes, (name, j)
        got = utt_out(out, j)
        if sig:
            d = np.abs(got.astype(np.int32) - ref.waveform.astype(np.int32))
            assert got.shape == ref.waveform.shape and d.max() <= 1 and (d > 0).mean() < tp.WAVE_MAX_FRAC, (name, j, d.max(), (d > 0).mean())
        else:
            tp.check_features(name, j, got, ref.features, o.fea_kind, tp._sensitivity(args, o, u))
        f = slice(int(plan.row_offsets[j]), int(plan.row_offsets[j]) + ref.nframes)
        if ref.vad_nr is not None:
            assert np.array_equal(vnr[f].astype(bool), ref.vad_nr), (name, j, "detector decisions differ at %d frames" % int((vnr[f].astype(bool) != ref.vad_nr).sum()))
        if ref.vad is not None:
            assert np.array_equal(vout[f].astype(bool), ref.vad.vad), (name, j, "VAD decisions differ")
    plan.close(); hd.close()
