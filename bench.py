#!/usr/bin/env python
"""bench.py -- feature frames/s of the CtuCopy hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--utts U] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic 16 kHz utterances
(10 000 x 10 s per GPU by default = 9.98 M frames, SURVEY.md 8(d) throughput set; inputs
3.2 GB, far larger than L2, so no cache flush is needed between timed steps).
  value : whole-job frames/s with the PCM already resident in HBM (CUDA events on the
          launching stream, max over ranks)
  e2e   : the same metric through the public C-ABI call with HOST (pinned) buffers:
          H2D of the PCM and D2H of the features inside the timed region
          e2e.copy_only_ms = the same chunk schedule with the kernels left out (control: what the
          host <-> device copies alone cost on this box at this N); e2e.frac_of_copy_only = copy_only_ms / ms_per_step
  roofline / cpu_baseline : see DESIGN.md "Measurement"
  workloads : the other BASELINE configs (PLP, MFCC_0_D_A, exten -> waveform, TRAP-DCT, fwss + Burg) measured the
          same way with fewer steps, each with its own roofline / e2e / selfcheck
  selfcheck : after the timed region the output of the LAST utterance of the batch is compared bit for bit with
          the output of the identical utterance near the start of the batch (past 2^31 elements in between), and
          with the CPU oracle within the parity tolerance
Multi-GPU: one process per GPU (torchrun), utterances sharded by rank, no collective on the
data path (weak scaling: every rank gets its own 10 000 utterances).
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B = ["-fs", "16000", "-format_in", "raw", "-dither", "0"]
WORKLOADS = {
    # name: (args, algorithmic bytes per frame of the whole step, ~flops per frame)
    # mfcc_exten is the headline: MFCC_0_D_A features at the metric's 10 ms hop with extended spectral subtraction on
    # the linear spectrum in front (north_star target "MFCC+exten ... pipelines"; BASELINE configs[1]'s algorithm, configs[0]'s
    # feature kind).  configs[1] verbatim (exten -> waveform, 16 ms hop, no features) is the "exten" workload.
    "mfcc_exten": (B + ["-preset", "mfcc", "-preem", "0.97", "-nr_mode", "exten", "-format_out", "htk", "-fea_delta", "d_a"], 476, 19000),
    "mfcc_d_a": (B + ["-format_out", "htk", "-w", "25", "-s", "10", "-preem", "0.97", "-fb_scale", "mel", "-fb_shape", "triang",
                      "-fb_power", "on", "-fb_definition", "30filters", "-nr_mode", "none", "-fb_eqld", "off", "-fb_inld", "off",
                      "-fea_kind", "dctc", "-fea_ncepcoefs", "12", "-fea_c0", "on", "-fea_E", "off", "-fea_lifter", "22",
                      "-fea_rawenergy", "off", "-fea_delta", "d_a", "-d_win", "2", "-a_win", "2", "-t_win", "2"], 476, 18000),
    "plp": (B + ["-preset", "plpc", "-format_out", "ark=out.ark"], 372, 19000),
    "trapdct": (B + ["-format_out", "htk", "-fb_definition", "23filters", "-fb_eqld", "off", "-fb_inld", "off", "-preem", "0.97",
                     "-fea_kind", "trapdct,51,8"], 1056, 40000),
    "exten": (B + ["-preset", "exten", "-format_out", "raw"], 1024, 30000),
    "fwss_burg": (B + ["-preset", "mfcc", "-preem", "0.97", "-nr_mode", "fwss", "-vad", "burg", "-nr_when", "beforeFB",
                       "-format_out", "pfile=out.pfile"], 380, 70000),
    # SURVEY 8f.3: MFCC_0 with +-2 frames of context stacked per coefficient (13 -> 65 columns)
    "mfcc_trap5": (B + ["-preset", "mfcc", "-preem", "0.97", "-fea_trap", "5", "-format_out", "htk"], 320 + 260, 18000),
    # SURVEY 8f.4 (egs/conf/20): 24 time-domain IIR band filters -> windowed band energies -> log -> DCT; 30 ms / 10 ms; the
    # coefficient file is the committed test fixture (the reference ships none)
    "tdiir": (B + ["-format_out", "htk", "-w", "30", "-s", "10", "-nr_mode", "none", "-fea_kind", "td-iir-mfcc",
                   "-filters", os.path.join(ROOT, "tests", "golden", "tdiir_filters.asc"), "-fea_ncepcoefs", "12"], 320 + 52, 160 * 24 * 22),
}
DEFAULT_WORKLOAD = "mfcc_exten"


def kernel_alg_bytes(name, hop, dim, nb):
    """ALGORITHMIC bytes one frame costs in each kernel (DESIGN.md section 3): what the kernel must read and write once."""
    pcm = 2 * hop
    return {
        "k_frames<pcm,fea>": pcm + 4 * dim, "k_frames<pcm,spec>": pcm + 4 * 257, "k_frames<pcm,fb>": pcm + 4 * nb,
        "k_frames<spec,fea>": 4 * 257 + 4 * dim, "k_frames<spec,fb>": 4 * 257 + 4 * nb,
        # k_bank: one spectrum row in (257 bins; the three pad floats per row are overhead, not algorithmic bytes), one
        # feature / band row out; with the scan fused nothing else moves
        "k_bank<fea>": 4 * 257 + 4 * dim, "k_bank<nr,fea>": 4 * 257 + 4 * dim, "k_bank<fb>": 4 * 257 + 4 * nb, "k_bank<nr,fb>": 4 * 257 + 4 * nb,
        "k_nr_scan": 2 * 4 * 257, "k_delta": 4 * dim + 12 * dim,   # compact static block in, c | delta | delta-delta out (whole rows)
        "k_lpc": 4 * nb + 4 * dim, "k_trapdct": 4 * nb + 4 * dim,
        "k_synth": pcm + 4 * 257 + pcm, "k_burg": pcm + 8 * 16, "k_cepdet": 8 * 16 + 1,
        "k_stack": 4 * 13 + 4 * dim,          # static block read once, stacked row written once
        "k_synth_c": 8 * 257 + 4 * 257 + pcm,  # stored complex spectrum + enhanced magnitudes in, one hop of int16 out
        "k_tdiir_filter": pcm + 8 * 24, "k_tdiir_frames": 3 * 8 * 24 + 4 * dim,   # one segment of 24 band energies per hop (30 / 10 ms)
    }.get(name)


METRIC = "feature frames/sec (16 kHz, 10 ms hop)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6553.3), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region: sampled every 20 ms from before
    the warm-up; stop(t0, t1) keeps the samples whose timestamps fall inside the timed window (all
    samples under load if the window is too short to hold two)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        import datetime
        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[1]), float(f[2]), [n for n, v in zip(names, f[5:9]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        window = "timed region"
        sel = [r for r in rows if t0 is not None and t0 <= r[0] <= t1]
        if len(sel) < 2:
            sel, window = rows, "warm-up + timed region (timed region shorter than two samples)"
        sm = [r[1] for r in sel]
        reasons = sorted({n for r in sel for n in r[3]})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(r[2] for r in sel) if sel else None,
                "reasons": reasons, "samples": len(sm), "window": window}


def cpu_reference_run(workload, utt_files, per_proc, cores, tmp, opt="O2"):
    """Times the reference's own CPU implementation (oracle/_ref/ctucopy4_<opt>, unmodified
    sources + FFT shim) on `cores` processes, each walking a list of `per_proc` 10 s
    utterances.  Returns (frames/s, frames, seconds)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "ctucopy4_" + opt)
    if not os.path.exists(exe):
        raise FileNotFoundError("oracle/_ref/ctucopy4_%s missing (run oracle/build_ref.sh in the build container)" % opt)
    args = [a for a in WORKLOADS[workload][0]]
    args = [a.replace("out.ark", os.path.join(tmp, "o.ark")).replace("out.pfile", os.path.join(tmp, "o.pfile")) for a in args]
    procs = []
    for p in range(cores):
        lst = os.path.join(tmp, "l%d.scp" % p)
        with open(lst, "w") as fh:
            for i in range(per_proc):
                fh.write("%s %s/o%d.out\n" % (utt_files[(p + i) % len(utt_files)], tmp, p))
        a = [x.replace(os.path.join(tmp, "o.ark"), os.path.join(tmp, "o%d.ark" % p)).replace(os.path.join(tmp, "o.pfile"),
             os.path.join(tmp, "o%d.pfile" % p)) for x in args]
        procs.append([exe] + a + ["-S", lst])
    t0 = time.perf_counter()
    running = [subprocess.Popen(c, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, cwd=tmp) for c in procs]
    rc = [r.wait() for r in running]
    dt = time.perf_counter() - t0
    if any(rc):
        raise RuntimeError("reference binary failed: exit codes %s" % sorted(set(rc)))
    return None, dt


def frames_per_utt(workload, nsamp=160000):
    w, s = (512, 256) if workload == "exten" else (480, 160) if workload == "tdiir" else (400, 160)
    return (nsamp - (w - s)) // s


def write_utts(tmp, n_unique):
    from ctucopy_b200 import synthetic
    files = []
    for k in range(n_unique):
        p = os.path.join(tmp, "u%d.raw" % k)
        synthetic.utterance(k, 10.0).astype("<i2").tofile(p)
        files.append(p)
    return files


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = len(os.sched_getaffinity(0))
    tmp = tempfile.mkdtemp(prefix="ctu_ref_")
    try:
        files = write_utts(tmp, 8)
        fpu = frames_per_utt(a.workload)
        per_proc = max(4, int(a.ref_seconds * 60000 / fpu))     # ~a.ref_seconds of work per core per step at ~60 k frames/s/core
        for _ in range(max(a.warmup, 0) and 1):
            cpu_reference_run(a.workload, files, max(2, per_proc // 8), cores, tmp)
        times = []
        for _ in range(a.steps):
            _, dt = cpu_reference_run(a.workload, files, per_proc, cores, tmp)
            times.append(dt)
        frames = cores * per_proc * fpu
        total = sum(times)
        val = frames * len(times) / total
        line = {
            "impl": "reference", "metric": METRIC, "value": val, "unit": "frames/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1000.0 * total / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": a.workload, "utterances_per_step": cores * per_proc, "seconds_per_utt": 10.0,
                       "args": " ".join(WORKLOADS[a.workload][0])},
            "cpu_baseline": {"value": val, "unit": "frames/s", "cores": cores, "kind": "reference",
                             "sample": "%d processes x %d utterances of 10 s per step, oracle/_ref/ctucopy4_O2 (unmodified reference sources, "
                                       "-O2, FFT shim instead of FFTW), list mode, file I/O on local disk" % (cores, per_proc)},
            "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return 0


def cli_run(workload, n_utts):
    """File -> file through the command-line host (host/ctucopy_b200: decode -> pinned buffers -> library -> writers, three
    overlapped stages) on /dev/shm: SURVEY 8f.1.  Returns the wall-clock rate of a whole process run (CUDA start-up
    included), and the steady-state rate from the stage times the host prints under CTU_TIMING=1."""
    import re
    from ctucopy_b200 import synthetic
    exe = os.path.join(ROOT, "host", "ctucopy_b200")
    base = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    d = tempfile.mkdtemp(prefix="ctu_cli_", dir=base)
    try:
        os.makedirs(d + "/in"); os.makedirs(d + "/out")
        uniq = [synthetic.utterance(k, 10.0).astype("<i2").tobytes() for k in range(16)]
        for i in range(n_utts):
            with open("%s/in/u%05d.raw" % (d, i), "wb") as fh:
                fh.write(uniq[i % 16])
        args = [a.replace("out.ark", d + "/o.ark").replace("out.pfile", d + "/o.pfile") for a in WORKLOADS[workload][0]]
        with open(d + "/list.scp", "w") as fh:
            for i in range(n_utts):
                fh.write("%s/in/u%05d.raw %s/out/u%05d.out\n" % (d, i, d, i))
        fpu = frames_per_utt(workload)
        runs = []
        for rep in range(2):
            t0 = time.perf_counter()
            pr = subprocess.run([exe] + args + ["-S", d + "/list.scp"], capture_output=True, text=True, env=dict(os.environ, CTU_TIMING="1"))
            dt = time.perf_counter() - t0
            if pr.returncode != 0:
                return {"error": "CLI exit %d: %s" % (pr.returncode, pr.stderr.strip()[-200:])}
            st = {}
            for m in re.finditer(r"\[ctu timing\] (.+?)\s+([0-9.]+) s", pr.stderr):
                st.setdefault(m.group(1).strip(), []).append(float(m.group(2)))
            runs.append((dt, st))
        dt, st = runs[-1]
        nb = len(st.get("batch ctu_run", [])) or 1
        # steady state: the slowest of the three overlapped stages, per batch (the first batch, which pays the allocations,
        # left out when there are several)
        per_stage = {k: (statistics.median(v[1:]) if len(v) > 2 else statistics.median(v)) for k, v in st.items() if k.startswith("batch")}
        slow = max(per_stage.values()) if per_stage else None
        return {"workload": workload, "files": n_utts, "frames": n_utts * fpu, "where": base, "wall_s": dt, "frames_per_s_whole_run": n_utts * fpu / dt,
                "startup_s": (st.get("ctu_create (CUDA init)") or [None])[0], "batches": nb, "stage_s_per_batch": per_stage,
                "frames_per_s_steady": (n_utts * fpu / nb) / slow if slow else None, "first_run_wall_s": runs[0][0],
                "note": "second of two runs; steady = frames per batch / slowest overlapped stage (read+decode | library call | write)"}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def selfcheck(workload, args, plan, hd, d_out, lens, uniq, first, sig):
    """Correctness at bench scale, outside the timed region: (1) utterance n-1 holds the same samples as utterance
    (n-1) % uniq, so their outputs must be bit-identical although they sit at opposite ends of the batch (2.56e9
    spectrum elements apart: 64-bit indexing, tile lists, persistent-CTA strides); (2) that utterance against the CPU
    oracle (test infrastructure, the checker only) within the parity tolerance of tests/test_gpu_parity.py."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ctu_oracle as co
    from ctucopy_b200 import synthetic
    n = len(lens)
    a_i, b_i = n - 1, (n - 1) % uniq
    if sig:
        off = plan.wave_offsets
        ya = d_out[int(off[a_i]): int(off[a_i + 1])].cpu().numpy()
        yb = d_out[int(off[b_i]): int(off[b_i + 1])].cpu().numpy()
    else:
        ro = plan.row_offsets
        ya = d_out[int(ro[a_i]): int(ro[a_i + 1])].cpu().numpy()
        yb = d_out[int(ro[b_i]): int(ro[b_i + 1])].cpu().numpy()
    out = {"identical_utts": [a_i, b_i]}
    if ya.shape != yb.shape or ya.tobytes() != yb.tobytes():
        out["status"] = "FAILED: outputs of identical utterances %d and %d differ" % (a_i, b_i)
        return out
    o = co.parse_args([x for x in args])
    ref = co.run_pipeline(synthetic.utterance(first + b_i, 10.0), o)
    if sig:
        d = np.abs(ya.astype(np.int32) - ref.waveform.astype(np.int32))
        out["oracle_max_lsb"] = int(d.max())
        out["oracle_frac_off_by_one"] = float((d > 0).mean())
        ok = d.max() <= 1 and (d > 0).mean() < 0.005
    else:
        fin = np.isfinite(ref.features)
        same_nf = np.array_equal(np.isfinite(ya), fin)
        err = np.abs(ya - ref.features)[fin]
        tol = (1e-4 * np.abs(ref.features) + 1e-3)[fin]
        out["oracle_max_err_over_tol"] = float((err / tol).max()) if err.size else 0.0
        ok = same_nf and bool((err <= tol).all())
    out["tolerance"] = "waveform: <= 1 LSB on < 0.5 % of samples" if sig else "1e-4 relative + 1e-3 absolute (log-domain features)"
    out["status"] = "ok" if ok else "FAILED: differs from the oracle beyond the parity tolerance"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=list(WORKLOADS))
    ap.add_argument("--utts", type=int, default=10000, help="utterances of 10 s per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--ref-seconds", type=float, default=4.0, help="CPU work per core per step of the reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--others", default="auto", choices=["auto", "all", "none"],
                    help="the other BASELINE configs under 'workloads': auto = all of them on one GPU, PLP only under torchrun")
    ap.add_argument("--no-selfcheck", action="store_true")
    ap.add_argument("--cli-utts", type=int, default=20000, help="10 s files for the file -> file run of the command-line host (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's output to DIR/*.npy (rank 0's shard under torchrun)")
    a = ap.parse_args()
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    if a.impl == "reference":
        return run_reference_arm(a)

    import torch
    import torch.distributed as dist
    import ctucopy_b200 as cb
    from ctucopy_b200 import synthetic

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the CtuCopy hot path has no CPU fallback"}))
        return 1
    torch.cuda.set_device(local)
    numa = None
    if world > 1:
        # one process per GPU: run on (and, by first touch, allocate the pinned buffers from) the CPU cores next to this
        # rank's GPU -- the end-to-end number is bound by host <-> device copies, which cross the socket link otherwise
        try:
            import pynvml
            pynvml.nvmlInit()
            hnd = pynvml.nvmlDeviceGetHandleByIndex(local)
            words = pynvml.nvmlDeviceGetCpuAffinity(hnd, (os.cpu_count() + 63) // 64)
            cpus = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1} & os.sched_getaffinity(0)
            if cpus and os.environ.get("CTU_BENCH_NO_AFFINITY") is None:
                os.sched_setaffinity(0, cpus)
                numa = "%d cpus next to GPU %d" % (len(cpus), local)
        except Exception as e:      # affinity is an optimisation, never fatal
            numa = "unavailable (%s)" % type(e).__name__
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # each rank's shard of the utterance list (weak scaling: a.utts per rank): 16 distinct utterances tiled, and every
    # rank synthesises its OWN 16 (utterance numbers 16*rank .. 16*rank+15), so no two ranks hold the same samples
    uniq = min(16, a.utts)
    first = uniq * rank
    pcm_np, lens = synthetic.batch(a.utts, 10.0, unique=uniq, first=first)
    h_pcm = torch.empty(len(pcm_np), dtype=torch.int16).pin_memory()
    h_pcm.numpy()[:] = pcm_np
    del pcm_np
    d_pcm = h_pcm.cuda(non_blocking=True)
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream().cuda_stream

    def dump_outputs(d, plan, d_out, sig, lens):
        """The output of the last timed step as a caller receives it, for comparing two builds output for output: a fixed,
        seeded sample of whole utterances (features [utt, frame, dim] or waveform [utt, sample], float32) within 64 MB,
        and the batch positions of the sampled utterances (float64).  An utterance larger than the whole budget is cut to
        its leading rows."""
        os.makedirs(d, exist_ok=True)
        off = plan.wave_offsets if sig else plan.row_offsets
        budget = (60 << 20) // (4 * (1 if sig else d_out.shape[1]))          # rows of float32 within 60 MiB
        longest = max(int(off[i + 1] - off[i]) for i in range(len(lens)))
        k = min(len(lens), 256, max(1, budget // longest))
        keep = min(longest, budget // k)
        sel = np.sort(np.random.default_rng(0).choice(len(lens), k, replace=False))
        rows = [d_out[int(off[i]): min(int(off[i + 1]), int(off[i]) + keep)].float().cpu().numpy() for i in sel]
        np.save(os.path.join(d, "waveform.npy" if sig else "features.npy"), np.stack(rows))
        np.save(os.path.join(d, "utterances.npy"), sel.astype(np.float64))

    def measure(workload, steps, warmup, e2e_steps, with_clocks, check, dump=None):
        args, bytes_step, flops = WORKLOADS[workload]
        hd = cb.Handle(args, device=local)
        plan = hd.plan(lens)
        frames = plan.total_frames
        dim = hd.feature_dim
        sig = hd.signal_output
        if sig:
            d_out = torch.empty(plan.total_output_samples, dtype=torch.int16, device="cuda")
            h_out = torch.empty(plan.total_output_samples, dtype=torch.int16).pin_memory()
        else:
            d_out = torch.empty((frames, dim), dtype=torch.float32, device="cuda")
            h_out = torch.empty((frames, dim), dtype=torch.float32).pin_memory()

        def step():
            if sig:
                plan.run_device(d_pcm.data_ptr(), d_waveform=d_out.data_ptr(), stream=stream)
            else:
                plan.run_device(d_pcm.data_ptr(), d_features=d_out.data_ptr(), stream=stream)

        sampler = ClockSampler(local) if with_clocks else None
        if sampler:
            sampler.start()
            step(); torch.cuda.synchronize()
            time.sleep(0.25)                               # nvidia-smi needs a moment before its first sample
        for _ in range(warmup):
            step()
        barrier()
        t_begin = time.time()
        l0 = hd.launch_count
        hd.profile(True)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            step()
        ev1.record()
        barrier()
        t_end = time.time()
        ms = ev0.elapsed_time(ev1)
        launches = hd.launch_count - l0
        recs = hd.profile_records()
        hd.profile(False)
        clocks = sampler.stop(t_begin, t_end) if sampler else None
        ms = max_over_ranks(ms)
        if dump and rank == 0:
            dump_outputs(dump, plan, d_out, sig, lens)
        # per-kernel average duration over the timed region; the dominant kernel is the one with the largest share
        by = {}
        for n, t in recs:
            by.setdefault(n, []).append(t)
        kern_ms = {n: sum(v) / steps for n, v in by.items()}
        dom = max(kern_ms, key=kern_ms.get) if kern_ms else None
        hop = 256 if workload == "exten" else 160
        sdim = dim // 3 if ("-fea_delta" in args and dim % 3 == 0) else dim      # static block of a _D_A vector
        kinfo = {}
        for n, ms_k in kern_ms.items():
            if workload == "mfcc_trap5":
                sdim = 13
            d = {"k_delta": sdim, "k_frames<pcm,fea>": sdim if workload != "trapdct" else hd.num_bands,
                 "k_frames<spec,fea>": sdim, "k_lpc": sdim,
                 "k_bank<fea>": sdim if workload != "trapdct" else hd.num_bands,
                 "k_bank<nr,fea>": sdim if workload != "trapdct" else hd.num_bands}.get(n, dim)
            ab = kernel_alg_bytes(n, hop, d, hd.num_bands)
            if ab:
                gbs = frames * ab / (ms_k / 1000.0) / 1e9
                kinfo[n] = {"ms": ms_k, "alg_bytes_per_frame": ab, "achieved_gbs": gbs}
        chk = None
        if check:
            try:
                chk = selfcheck(workload, args, plan, hd, d_out, lens, uniq, first, sig)
            except Exception as e:      # a broken checker must not hide the measurement; it is reported as such
                chk = {"status": "FAILED: selfcheck raised %s: %s" % (type(e).__name__, e)}
        # ---- end to end through the public host-buffer call, and the same chunk schedule with the kernels left out
        e2e = None
        if e2e_steps > 0:
            pcm_host = h_pcm.numpy()
            out_host = h_out.numpy()
            kw = {"waveform": out_host} if sig else {"features": out_host}

            def timed(nsteps):
                plan.run_host(pcm_host, want_vad=False, **kw)       # warm-up (the first call allocates the plan's device buffers)
                barrier()
                t0 = time.perf_counter()
                for _ in range(nsteps):
                    plan.run_host(pcm_host, want_vad=False, **kw)
                torch.cuda.synchronize()
                return max_over_ranks(time.perf_counter() - t0)

            dt = timed(e2e_steps)
            hd.set_option("copy_only", 1)
            dtc = timed(e2e_steps)
            hd.set_option("copy_only", 0)
            h2d, d2h = int(h_pcm.numel() * 2), int(h_out.numel() * h_out.element_size())
            e2e = {"value": world * frames * e2e_steps / dt, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "ms_per_step": 1000 * dt / e2e_steps, "copy_only_ms": 1000 * dtc / e2e_steps, "frac_of_copy_only": dtc / dt,
                   "copy_only_gbs_per_gpu": (h2d + d2h) / 1e9 / (dtc / e2e_steps),
                   "note": "copy_only = the same ctu_plan_run_host chunk schedule (32 MB of PCM per chunk, three streams) with every kernel "
                           "skipped: frac_of_copy_only close to 1 means the end-to-end time IS the host <-> device copy time of this box at this N"}
        res = dict(frames=frames, ms=ms, launches=launches, kern_ms=kern_ms, dom=dom, clocks=clocks, e2e=e2e,
                   bytes_step=bytes_step, kinfo=kinfo, flops=flops, dim=dim, args=args, selfcheck=chk)
        plan.close(); hd.close()
        del d_out, h_out
        torch.cuda.empty_cache()
        return res

    hbm, peak_src = peaks()

    def roofline_of(workload, r, value):
        for k in r["kinfo"].values():
            k["frac"] = k["achieved_gbs"] / hbm
        if r["dom"] not in r["kinfo"]:
            return None
        ki = r["kinfo"][r["dom"]]
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            t = json.load(open(tp)).get(workload + ":" + r["dom"])
            if t:   # measured DRAM bytes per frame (ncu --set full) x frames of this launch
                traffic = t["dram_bytes_per_frame"] * r["frames"]
        return {"bound": "hbm", "kernel": r["dom"], "achieved": ki["achieved_gbs"], "peak": hbm, "unit": "GB/s", "frac": ki["frac"],
                "traffic": traffic, "peak_source": peak_src, "kernel_ms": ki["ms"], "alg_bytes_per_frame": ki["alg_bytes_per_frame"],
                "alg_bytes_per_launch": ki["alg_bytes_per_frame"] * r["frames"],
                "step_alg_bytes_per_frame": r["bytes_step"],
                "step_hbm_frac": (value / world) * r["bytes_step"] / 1e9 / hbm,
                "fp32_frac_of_74TF": (value / world) * r["flops"] / 74e12,
                "kernels": r["kinfo"]}

    check = not a.no_selfcheck
    r = measure(a.workload, a.steps, a.warmup, a.e2e_steps, True, check, a.dump_outputs)
    value = world * r["frames"] * a.steps / (r["ms"] / 1000.0)
    roof = roofline_of(a.workload, r, value)
    if roof:
        roof["note"] = ("dominant kernel = largest share of the step; the FFT front end is FP32 / shared-memory-pipe bound, not HBM "
                        "bound (DESIGN.md 3); the noise-reduction scan is the HBM-bound piece of this path")
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": r["ms"] / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": a.workload, "utterances_per_gpu": a.utts, "seconds_per_utt": 10.0, "frames_per_gpu": r["frames"],
                   "feature_dim": r["dim"], "args": " ".join(r["args"]), "l2": "inputs (3.2 GB PCM per GPU) exceed L2; no flush needed",
                   "sharding": "utterances by rank (rank r holds synthetic utterances 16r .. 16r+15, tiled), no collective",
                   "cpu_affinity": numa},
        "gpu_launches": r["launches"], "kernel_ms_per_step": r["kern_ms"], "clocks": r["clocks"], "e2e": r["e2e"], "roofline": roof,
        "selfcheck": (r["selfcheck"] or {}).get("status", "skipped"), "selfcheck_detail": r["selfcheck"],
    }
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        tmp = tempfile.mkdtemp(prefix="ctu_cpu_")
        try:
            cores = len(os.sched_getaffinity(0))
            files = write_utts(tmp, 8)
            fpu = frames_per_utt(a.workload)
            per_proc = max(4, int(6.0 * 60000 / fpu))
            _, dt = cpu_reference_run(a.workload, files, per_proc, cores, tmp)
            line["cpu_baseline"] = {"value": cores * per_proc * fpu / dt, "unit": "frames/s", "cores": cores, "kind": "reference",
                                    "sample": "%d processes x %d utterances of 10 s (%.1f s wall), oracle/_ref/ctucopy4_O2 = unmodified "
                                              "reference sources at -O2 with the FFT shim (no FFTW in the image)" % (cores, per_proc, dt)}
        except Exception as e:  # the baseline is a reported extra, never fatal for the GPU numbers
            line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference", "sample": "failed: %s" % e}
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    if rank == 0 and world == 1 and a.cli_utts > 0:
        try:
            line["cli"] = cli_run(a.workload, a.cli_utts)
            cb_ = line.get("cpu_baseline") or {}
            if cb_.get("value") and line["cli"].get("frames_per_s_whole_run"):
                line["cli"]["vs_cpu_reference_whole_run"] = line["cli"]["frames_per_s_whole_run"] / cb_["value"]
        except Exception as e:      # reported, never fatal for the headline
            line["cli"] = {"error": "%s: %s" % (type(e).__name__, e)}
    # ---- the other BASELINE configs, measured the same way with fewer steps (BASELINE.json configs 1, 2, 3, 4, 5)
    names = []
    if a.others == "all" or (a.others == "auto" and world == 1):
        names = [w for w in ("plp", "mfcc_d_a", "exten", "trapdct", "fwss_burg", "tdiir") if w != a.workload]
    elif a.others == "auto":
        names = [w for w in ("plp",) if w != a.workload]
    others = {}
    for w in names:
        try:
            k = max(3, min(5, a.steps // 4))
            x = measure(w, k, 3, 2, False, check)
            v = world * x["frames"] * k / (x["ms"] / 1000.0)
            others[w] = {"value": v, "unit": "frames/s", "steps": k, "warmup": 3, "frames_per_gpu": x["frames"], "ms_per_step": x["ms"] / k,
                         "args": " ".join(x["args"]), "gpu_launches": x["launches"], "kernel_ms_per_step": x["kern_ms"], "e2e": x["e2e"],
                         "roofline": roofline_of(w, x, v), "selfcheck": (x["selfcheck"] or {}).get("status", "skipped"),
                         "selfcheck_detail": x["selfcheck"]}
        except Exception as e:
            others[w] = {"error": "%s: %s" % (type(e).__name__, e)}
    if others:
        line["workloads"] = others
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    # ONE JSON line on stdout: libraries that write to file descriptor 1 from native code (NCCL prints its
    # version banner there) are sent to stderr; only our own print() reaches the real stdout
    sys.stdout.flush()
    _real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = _real
    rc = main()
    _real.flush()
    sys.exit(rc)
