#!/usr/bin/env python
"""Writes tests/golden/shard_containers.npz, the Kaldi ark+scp and ICSI pfile containers that tests/test_shard_cpu.py
merges and compares: for each list of SHARD_LISTS, the container one process writes for the whole list and the ones it
writes for each rank's range of the list.  They are written by the command-line host (host/ctucopy_b200, needs a CUDA
device), whose container layout tests/test_gpu_cli.py compares with the reference's files.  Paths inside the scp files
are stored with the output directory replaced by {D}.

    python tests/golden/make_shard_golden.py          # after __graft_entry__.build(), on a GPU machine
"""
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import golden_util as gu  # noqa: E402
from ctucopy_b200 import shard  # noqa: E402

EXE = os.path.join(ROOT, "host", "ctucopy_b200")
B = ["-fs", "16000", "-format_in", "raw", "-dither", "0"]
ORDER = (0, 4, 1, 5, 2, 3)                     # golden inputs, in list order
# name: (options, {world sizes: tag of rank r})
SHARD_LISTS = {
    "mfcc": (["-preset", "mfcc", "-preem", "0.97"], {2: "w2r%d", 3: "w3r%d"}),
    "plpc": (["-preset", "plpc"], {2: "r%d"}),
}


def containers(args, utts, d, tag):
    """one process of the host on `utts` -> {"ark", "scp", "pfile"} bytes, containers under d/tag"""
    os.makedirs(os.path.join(d, tag), exist_ok=True)
    lst = os.path.join(d, tag, "list.scp")
    with open(lst, "w") as fh:
        for name, u in utts:
            p = os.path.join(d, name + ".raw")
            if not os.path.exists(p):
                np.asarray(u).astype("<i2").tofile(p)
            fh.write("%s %s\n" % (p, name))
    out = {}
    for kind in ("ark", "pfile"):
        tgt = os.path.join(d, tag, "o." + kind)
        pr = subprocess.run([EXE] + B + args + ["-format_out", "%s=%s" % (kind, tgt), "-S", lst], capture_output=True, cwd=d)
        assert pr.returncode == 0, pr.stderr.decode()
        out[kind] = open(tgt, "rb").read()
    out["scp"] = open(os.path.join(d, tag, "o.scp"), "rb").read().replace(d.encode(), b"{D}")
    return out


def main():
    ins = gu.inputs()
    utts = [("utt%d" % i, ins[i]) for i in ORDER]
    res = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, (args, worlds) in SHARD_LISTS.items():
            d = os.path.join(tmp, name)
            parts = {"whole": utts}
            for world, tag in worlds.items():
                cut = shard.partition([len(u) for _, u in utts], world)
                parts.update({tag % r: utts[cut[r]:cut[r + 1]] for r in range(world)})
            for tag, sub in parts.items():
                for kind, b in containers(args, sub, d, tag).items():
                    res["%s_%s_%s" % (name, tag, kind)] = np.frombuffer(b, dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, "shard_containers.npz"), **res)
    print("shard_containers.npz:", len(res), "arrays,", sum(v.size for v in res.values()), "bytes")


if __name__ == "__main__":
    main()
