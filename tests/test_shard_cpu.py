"""Host-side multi-GPU logic on CPU: list partitioning and the ordered merge of per-rank
containers (SURVEY.md 8e).  The per-rank containers are the ones one process writes for each
rank's list range, stored in tests/golden/shard_containers.npz (tests/golden/make_shard_golden.py),
so the check is exact: the merged ark+scp / pfile must equal, byte for byte, what one process
writes for the whole list.  A world_size-2 gloo run covers the plumbing bench.py uses under
torchrun (rank ranges, barrier, max-over-ranks, gather to rank 0)."""
import os
import subprocess
import sys

import numpy as np

import golden_util as gu
import ref_runner as rr
from ctucopy_b200 import shard

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "host", "ctucopy_b200")
B = ["-fs", "16000", "-format_in", "raw", "-dither", "0"]


def test_partition_is_contiguous_balanced_and_total():
    rng = np.random.default_rng(3)
    for n_utts, world in ((1, 2), (2, 2), (7, 2), (100, 8), (1000, 8), (5, 8)):
        s = rng.integers(1000, 200000, n_utts).tolist()
        cut = shard.partition(s, world)
        assert cut[0] == 0 and cut[-1] == n_utts and all(a <= b for a, b in zip(cut, cut[1:]))
        if n_utts >= 100:
            per = [sum(s[cut[r]:cut[r + 1]]) for r in range(world)]
            assert max(per) - min(per) <= 2 * max(s)
    assert shard.partition([10, 10, 10, 10], 2) == [0, 2, 4]
    assert shard.rank_range([10, 10, 10, 10], 1, 2) == (2, 4)
    ev = bytes(range(10))
    assert shard.split_ext_vad(ev, [3, 3, 4], [0, 2, 3]) == [ev[:6], ev[6:]]


def _containers(name, tag, d):
    """stored containers of list `name` (make_shard_golden.SHARD_LISTS) for `tag` -> (ark, scp, pfile) bytes, scp paths under d"""
    z = np.load(os.path.join(gu.GOLDEN, "shard_containers.npz"))
    out = {kind: z["%s_%s_%s" % (name, tag, kind)].tobytes() for kind in ("ark", "pfile")}
    out["scp"] = z["%s_%s_scp" % (name, tag)].tobytes().decode().replace("{D}", d)
    return out


def test_stored_containers_hold_the_reference_matrices(tmp_path):
    """The stored plpc containers against what the reference wrote for each utterance with the same options (the plpc_ark
    golden, one utterance per run): same keys in list order, the same matrix header bytes at every scp offset, matrices
    within the parity tolerance."""
    c = gu.Case("plpc_ark")
    whole = _containers("plpc", "whole", str(tmp_path))
    got = rr.parse_ark(whole["ark"])
    order = (0, 4, 1, 5, 2, 3)
    assert list(got) == ["utt%d" % i for i in order]
    offs = [int(ln.rsplit(":", 1)[1]) for ln in whole["scp"].splitlines()]
    for i, off in zip(order, offs):
        ref_off = int(c.aux[i].decode().split()[1].rsplit(":", 1)[1])
        assert whole["ark"][off:off + 15] == c.raw[i][ref_off:ref_off + 15], i
        a, b = got["utt%d" % i], c.payload(i)
        assert a.shape == b.shape and np.all(np.abs(a - b) <= 1e-4 * np.abs(b) + 1e-3), i


def test_merged_containers_equal_the_single_process_reference(tmp_path):
    d = str(tmp_path)
    ins = gu.inputs()
    utts = [("utt%d" % i, ins[i]) for i in (0, 4, 1, 5, 2, 3)]
    args = ["-preset", "mfcc", "-preem", "0.97"]
    whole = _containers("mfcc", "whole", d)
    for world in (2, 3):
        cut = shard.partition([len(u) for _, u in utts], world)
        parts = [_containers("mfcc", "w%dr%d" % (world, r), d) for r in range(world)]
        for r, p in enumerate(parts):
            assert [ln.split()[0] for ln in p["scp"].splitlines()] == [n for n, _ in utts[cut[r]:cut[r + 1]]]
        # python merge
        assert shard.merge_pfile([p["pfile"] for p in parts]) == whole["pfile"]
        scps = [p["scp"].replace("/w%dr%d/" % (world, r), "/whole/") for r, p in enumerate(parts)]
        ark, scp = shard.merge_ark([p["ark"] for p in parts], scps)
        assert ark == whole["ark"] and scp == whole["scp"]
        # C++ host merge (-merge N works on files named shard<r>of<N>_<name>; no GPU involved)
        if os.path.exists(EXE):
            m = os.path.join(d, "m%d" % world)
            os.makedirs(m)
            for r, p in enumerate(parts):
                open(os.path.join(m, "shard%dof%d_o.pfile" % (r, world)), "wb").write(p["pfile"])
                open(os.path.join(m, "shard%dof%d_o.ark" % (r, world)), "wb").write(p["ark"])
                open(os.path.join(m, "shard%dof%d_o.scp" % (r, world)), "w").write(scps[r].replace("/whole/", "/m%d/" % world))
            for kind in ("pfile", "ark"):
                pr = subprocess.run([EXE] + B + args + ["-format_out", "%s=%s/o.%s" % (kind, m, kind), "-merge", str(world)], capture_output=True)
                assert pr.returncode == 0, pr.stderr.decode()
            assert open(os.path.join(m, "o.pfile"), "rb").read() == whole["pfile"]
            assert open(os.path.join(m, "o.ark"), "rb").read() == whole["ark"]
            assert open(os.path.join(m, "o.scp")).read() == whole["scp"].replace("/whole/", "/m%d/" % world)
            assert not [f for f in os.listdir(m) if f.startswith("shard")]


WORKER = r"""
import os, sys, pickle
sys.path[:0] = [%(root)r, os.path.join(%(root)r, "oracle"), os.path.join(%(root)r, "tests")]
import numpy as np
import torch, torch.distributed as dist
import golden_util as gu
from ctucopy_b200 import shard
import test_shard_cpu as T
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo")
ins = gu.inputs()
utts = [("utt%%d" %% i, ins[i]) for i in (0, 4, 1, 5, 2, 3)]
lo, hi = shard.rank_range([len(u) for _, u in utts], rank, world)
d = sys.argv[1]
part = T._containers("plpc", "r%%d" %% rank, d)
assert [ln.split()[0] for ln in part["scp"].splitlines()] == [n for n, _ in utts[lo:hi]]
part["scp"] = part["scp"].replace("/r%%d/" %% rank, "/whole/")
dist.barrier()
t = torch.tensor([float(rank + 1)], dtype=torch.float64)
dist.all_reduce(t, op=dist.ReduceOp.MAX)               # the max-over-ranks bench.py takes of its timings
assert t.item() == world
gathered = [None] * world if rank == 0 else None
dist.gather_object(part, gathered, dst=0)
if rank == 0:
    whole = T._containers("plpc", "whole", d)
    assert shard.merge_pfile([g["pfile"] for g in gathered]) == whole["pfile"]
    ark, scp = shard.merge_ark([g["ark"] for g in gathered], [g["scp"] for g in gathered])
    assert ark == whole["ark"] and scp == whole["scp"]
    open(os.path.join(d, "ok"), "w").write("ok")
dist.destroy_process_group()
"""


def test_world_size_2_gloo_shards_merge_to_the_single_process_result(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER % {"root": ROOT})
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29631", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script), str(tmp_path)], env=dict(env, RANK=str(r), LOCAL_RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=300)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(outs)
    assert (tmp_path / "ok").exists()
