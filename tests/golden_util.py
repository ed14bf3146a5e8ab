"""Loads tests/golden/*.npz (written by tests/golden/make_golden.py from the reference binary)."""
import json
import os

import numpy as np

import ref_runner as rr

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

_inputs = None


def inputs():
    global _inputs
    if _inputs is None:
        z = np.load(os.path.join(GOLDEN, "inputs.npz"))
        _inputs = [z["in%d" % i] for i in range(len(z.files))]
    return _inputs


def case_names():
    return sorted(f[:-4] for f in os.listdir(GOLDEN) if f.endswith(".npz") and f not in ("inputs.npz", "fb_design.npz", "shard_containers.npz") and not f.startswith("cmvn") and not f.startswith("feain_") and not f.startswith("g711_") and not f.startswith("carry_"))


def g711_case(name):
    """8-bit input golden: (args, law, [codes per input], Case-like payload access through Case(name))."""
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    n = len(inputs())
    return json.loads(str(z["args"])), str(z["law"]) == "alaw", [z["codes%d" % i] for i in range(n)]


def feain_case_names():
    """Feature-file input goldens (-format_in htk): Case(name).source names the golden whose payloads are the inputs."""
    return sorted(f[:-4] for f in os.listdir(GOLDEN) if f.startswith("feain_") and f.endswith(".npz"))


def carry_case_names():
    """*ss modes over a list in one reference process (the opt-in "ss_carry" semantics)"""
    return sorted(f[:-4] for f in os.listdir(GOLDEN) if f.startswith("carry_") and f.endswith(".npz"))


def carry_case(name):
    """(args, kind, input indices in list order, [output bytes per file], [external VAD flags per file] or None)"""
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    idx = [int(i) for i in z["idx"]]
    outs = [z["out%d" % j].tobytes() for j in range(len(idx))]
    ev = [z["extvad%d" % j] for j in range(len(idx))] if "extvad0" in z.files else None
    args = [a.replace("{VADIN}", "vadin.bin") for a in json.loads(str(z["args"]))]
    return args, str(z["kind"]), idx, outs, ev


def cmvn_case(name):
    """A list-mode CMVN golden: (args with {STAT}, input indices, speakers, statistics text, {index: HTK bytes})."""
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    idx = [int(i) for i in z["idx"]]
    outs = {i: z["out%d" % i].tobytes() for i in idx if ("out%d" % i) in z.files}
    return json.loads(str(z["args"])), idx, json.loads(str(z["spk"])), z["stat"].tobytes().decode(), outs


class Case:
    def __init__(self, name):
        z = np.load(os.path.join(GOLDEN, name + ".npz"))
        self.name = name
        self.args = json.loads(str(z["args"]))
        self.kind = str(z["kind"])
        self.source = str(z["source"]) if "source" in z.files else None
        self.n = len(inputs())
        self.raw = [z["out%d" % i].tobytes() for i in range(self.n)]
        self.aux = [z["aux%d" % i].tobytes() if ("aux%d" % i) in z.files else None for i in range(self.n)]
        self.extvad = [z["extvad%d" % i] if ("extvad%d" % i) in z.files else None for i in range(self.n)]
        # -vad_out_mode debug side files: per input, suffix -> raw bytes (native doubles, or '0' / '1' characters)
        self.debug = [{f[4:f.rindex("_")]: z[f].tobytes() for f in z.files if f.startswith("dbg_") and f.endswith("_%d" % i)} for i in range(self.n)]

    def oracle_args(self):
        """args as given to the reference, with container placeholders made harmless"""
        return [a.replace("{ARK}", "out.ark").replace("{PFILE}", "out.pfile").replace("{VADIN}", "vadin.bin").replace("{FILTERS}", rr.TDIIR_FILTERS) for a in self.args]

    def payload(self, i):
        """golden payload of utterance i as an array (features float32 [T,dim] or int16 PCM)"""
        b = self.raw[i]
        if self.kind == "htk":
            return rr.parse_htk(b)[1]
        if self.kind == "htk_be":
            return rr.parse_htk(b, ">")[1].astype("<f4")
        if self.kind == "ark":
            return list(rr.parse_ark(b).values())[0]
        if self.kind == "pfile":
            return rr.parse_pfile(b)[1]
        if self.kind == "raw":
            return np.frombuffer(b, dtype="<i2")
        if self.kind == "wave":
            return np.frombuffer(b[44:], dtype="<i2")
        raise ValueError(self.kind)


def same_nonfinite(a, b):
    return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(np.isposinf(a), np.isposinf(b)) and \
        np.array_equal(np.isneginf(a), np.isneginf(b))
