"""Shared helpers for the parity tests, smoke() and bench.py's cpu_baseline leg: locate models, run the oracle
(oracle/_ref = the reference's own CPU path when its prebuilt binary is present, else the C++ restatement in
oracle/), run the CUDA path through the C ABI, and compare u8 frames.  TEST INFRASTRUCTURE."""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
sys.path.insert(0, os.path.join(ROOT, "rife-ncnn-vulkan_b200"))
import synth  # noqa: E402

FAMILY = {"rife-v4.6": "v4", "rife-v4": "v4", "rife-v2.3": "v2", "rife-v2": "v2", "rife-v2.4": "v2", "rife-v3.0": "v2", "rife-v3.1": "v2",
          "rife": "v1", "rife-HD": "v1", "rife-UHD": "v1", "rife-anime": "v1"}


def model_dir(name):
    d = os.path.join(REF_DIR, "models", name)
    if os.path.isdir(d):
        return d
    d = os.path.join(ROOT, "tests", "models", name)  # synthetic-weight models (tests/make_synth_model.py)
    if os.path.isdir(d):
        return d
    import make_synth_model
    if name in make_synth_model.SEEDS:
        # the reference's model files did not travel: seeded random weights in the same file format and interface
        # (tests/make_synth_model.py), written once per process to a temporary directory (the tree may be read-only)
        if name not in _SYNTH:
            if "root" not in _SYNTH:
                import atexit
                import shutil
                _SYNTH["root"] = tempfile.mkdtemp(prefix="rife-b200-synth-")
                atexit.register(shutil.rmtree, _SYNTH["root"], True)
            _SYNTH[name] = make_synth_model.write_model(os.path.join(_SYNTH["root"], name), make_synth_model.SEEDS[name], name)
        return _SYNTH[name]
    return None


_SYNTH = {}
GOLD_DIR = os.path.join(ROOT, "tests", "golden")


def _sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for chunk in iter(lambda: f.read(1 << 20), b""):
            h.update(chunk)
    return h.hexdigest()


def golden_frame(name):
    """The committed golden frame of case `name` (tests/golden/golden.json) for the model files model_dir() finds, or None
    when there is none for them.  golden.npz holds the reference's CPU path on the reference's model files;
    golden_synth.npz holds the C++ restatement (oracle/) on the seeded synthetic rife-v4.6 weights of
    tests/make_synth_model.py, which stand in where the reference's files are absent.  The synthetic set is chosen only
    when the flownet.bin in use is byte for byte the one it was made with."""
    m = json.load(open(os.path.join(GOLD_DIR, "golden.json")))[name]
    md = model_dir(m["model"])
    if md is None:
        return None
    synth = json.load(open(os.path.join(GOLD_DIR, "golden_synth.json"))).get(name)
    if synth is not None and _sha256(os.path.join(md, "flownet.bin")) == synth["model_sha256"]:
        return np.load(os.path.join(GOLD_DIR, "golden_synth.npz"))[name]
    if md == _SYNTH.get(m["model"]):  # a generated stand-in without committed frames of its own
        return None
    return np.load(os.path.join(GOLD_DIR, "golden.npz"))[name]


def _cpu_flags():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("flags"):
                return set(line.split(":", 1)[1].split())
    except OSError:
        pass
    return set()


def ref_binary():
    """Path of the reference-oracle executable usable on this host, or None."""
    fl = _cpu_flags()
    forced = os.environ.get("RIFE_ORACLE_ISA")
    if forced:
        p = os.path.join(REF_DIR, "ref_rife_" + forced)
        return p if os.path.exists(p) else None
    cands = []
    if {"avx512f", "avx512bw", "avx512vl", "avx512dq", "avx512cd"} <= fl:
        cands.append("ref_rife_avx512")
    if "avx2" in fl and "fma" in fl:
        cands.append("ref_rife_avx2")
    for c in cands:
        p = os.path.join(REF_DIR, c)
        if os.path.exists(p) and os.access(p, os.X_OK):
            return p
    return None


def port_binary():
    p = os.path.join(ROOT, "oracle", "build", "oracle_rife")
    return p if os.path.exists(p) else None


def run_oracle(model, in0, in1, timestep=0.5, tta=False, tta_temporal=False, uhd=False, threads=None, repeat=1, warmup=0, which="auto", modeldir=None,
               crop_padded=False):
    """Returns (out u8 array, info dict).  which: 'ref' | 'port' | 'auto' (ref if present else port).
    modeldir overrides the lookup of `model` (the family flags still come from the name).
    crop_padded (port only): crop the padded output rows like the reference's GPU path instead of reproducing the CPU path's
    contiguous read (src/rife.cpp:4375-4387); the two differ only when w % 32 != 0 and no spatial TTA is used."""
    if crop_padded:
        which = "port"
    exe = None
    kind = None
    if which in ("auto", "ref"):
        exe = ref_binary()
        kind = "reference"
    if exe is None and which in ("auto", "port"):
        exe = port_binary()
        kind = "port"
    if exe is None:
        raise RuntimeError("no oracle executable available (oracle/_ref/ref_rife_* or oracle/build/oracle_rife)")
    md = modeldir or model_dir(model)
    if md is None:
        raise RuntimeError("model %s not available" % model)
    h, w = in0.shape[:2]
    with tempfile.TemporaryDirectory() as td:
        a, b, o = (os.path.join(td, n) for n in ("a.rgb", "b.rgb", "o.rgb"))
        np.ascontiguousarray(in0).tofile(a)
        np.ascontiguousarray(in1).tofile(b)
        cmd = [exe, "--model", md, "--family", FAMILY[model], "--w", str(w), "--h", str(h), "--in0", a, "--in1", b, "--out", o,
               "--t", repr(float(timestep)), "--repeat", str(repeat), "--warmup", str(warmup)]
        if crop_padded:
            cmd.append("--crop-padded")
        if tta:
            cmd.append("--tta")
        if tta_temporal:
            cmd.append("--tta-temporal")
        if uhd:
            cmd.append("--uhd")
        # small frames on a many-core host: cap the OpenMP team (128 threads on a 96x64 image crawl)
        cmd += ["--threads", str(threads or min(os.cpu_count() or 1, 16))]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        if r.returncode != 0:
            raise RuntimeError("oracle failed: %s\n%s" % (" ".join(cmd), r.stderr[-2000:]))
        info = json.loads(r.stdout.strip().splitlines()[-1])
        info["kind"] = kind
        out = np.fromfile(o, np.uint8).reshape(h, w, 3)
    return out, info


def compare(a, b):
    d = np.abs(a.astype(np.int16) - b.astype(np.int16))
    mse = float(np.mean(d.astype(np.float64) ** 2))
    return {"max_abs_diff": int(d.max()), "share_ne": float(np.mean(d > 0)), "share_ge2": float(np.mean(d >= 2)),
            "psnr_db": float("inf") if mse == 0 else float(10 * np.log10(255.0 ** 2 / mse))}


def run_gpu(pkg, model, in0, in1, timestep=0.5, tta=False, tta_temporal=False, uhd=False, gpuid=0, options=None):
    v2, v4 = pkg.family_flags(model)
    r = pkg.RIFE(gpuid, tta, tta_temporal, uhd, 1, v2, v4)
    try:
        r.load(model_dir(model))
        for k, v in (options or {}).items():
            r.set_option(k, v)
        return r.process(in0, in1, timestep)
    finally:
        r.close()


def check_case(pkg, model="rife-v4.6", w=256, h=192, timestep=0.5, tta=False, tta_temporal=False, uhd=False, dx=3, dy=2, seed=0, options=None, crop="reference"):
    """crop (matters only when w % 32 != 0 and no spatial TTA): "reference" compares with the reference's own CPU path, whose
    contiguous read of the padded output the library reproduces under option cpu_crop_quirk = 1; "padded" compares the
    library's default (the crop of the padded rows, as the reference's GPU path does) with the restatement run with --crop-padded."""
    in0, in1 = synth.pair(w, h, dx=dx, dy=dy, seed=seed)
    options = dict(options or {})
    if crop == "reference":
        if w % 32 and not tta:
            options["cpu_crop_quirk"] = 1
        ref, info = run_oracle(model, in0, in1, timestep, tta, tta_temporal, uhd)
    else:
        ref, info = run_oracle(model, in0, in1, timestep, tta, tta_temporal, uhd, crop_padded=True)
    out = run_gpu(pkg, model, in0, in1, timestep, tta, tta_temporal, uhd, options=options)
    res = compare(out, ref)
    res["oracle"] = info["kind"]
    # sanity: the interpolated frame must be a real image, not a constant
    res["out_std"] = float(out.std())
    return res
