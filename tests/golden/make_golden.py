#!/usr/bin/env python3
"""Regenerates tests/golden/golden.npz from oracle/_ref (the reference's own CPU functions + vendored ncnn, built by
oracle/build_ref.py from the reference's source tree; avx2 build, the ISA every x86 CI host has), where that build and the
reference's model files are present.  Inputs are synth.pair(w, h, dx, dy, seed).

--synthetic regenerates tests/golden/golden_synth.npz instead: the rife-v4.6 cases on the seeded synthetic weights of
tests/make_synth_model.py (the model a checkout without the reference's files runs on), computed by the C++ restatement
(oracle/build/oracle_rife), with the sha256 of the flownet.bin they were made with."""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import parity  # noqa: E402

CASES = [
    # name, model, w, h, kwargs for run_oracle, synth kwargs
    ("v46_plain_128x96", "rife-v4.6", 128, 96, {}, {}),
    ("v46_plain_100x70_cpu_crop_quirk", "rife-v4.6", 100, 70, {}, {}),
    ("v46_t025_128x96", "rife-v4.6", 128, 96, {"timestep": 0.25}, {}),
    ("v46_tta_96x64", "rife-v4.6", 96, 64, {"tta": True}, {}),
    ("v46_temporal_96x64", "rife-v4.6", 96, 64, {"tta_temporal": True}, {}),
    ("v46_tta_temporal_96x64", "rife-v4.6", 96, 64, {"tta": True, "tta_temporal": True}, {}),
    ("v46_large_motion_160x96", "rife-v4.6", 160, 96, {}, {"dx": 12, "dy": 8}),
    ("v4_t075_128x96", "rife-v4", 128, 96, {"timestep": 0.75}, {}),
    ("v23_plain_128x96", "rife-v2.3", 128, 96, {}, {}),
    ("v23_tta_temporal_96x64", "rife-v2.3", 96, 64, {"tta": True, "tta_temporal": True}, {}),
    ("v23_uhd_128x128", "rife-v2.3", 128, 128, {"uhd": True}, {}),
    ("anime_plain_128x96", "rife-anime", 128, 96, {}, {}),
    ("anime_tta_temporal_96x64", "rife-anime", 96, 64, {"tta": True, "tta_temporal": True}, {}),
]


def main(synthetic=False):
    os.environ["RIFE_ORACLE_ISA"] = "avx2"
    arrays, manifest = {}, {}
    td = tempfile.TemporaryDirectory()
    synth_model = None
    if synthetic:
        import make_synth_model
        synth_model = make_synth_model.write_model(os.path.join(td.name, "rife-v4.6"), seed=0)
    for name, model, w, h, kw, skw in CASES:
        if synthetic and model != "rife-v4.6":
            continue
        a, b = parity.synth.pair(w, h, **skw)
        out, info = parity.run_oracle(model, a, b, which="port" if synthetic else "ref", modeldir=synth_model, **kw)
        arrays[name] = out
        manifest[name] = {"model": model, "w": w, "h": h, "oracle_kwargs": kw, "synth_kwargs": skw,
                          "in_sha256": hashlib.sha256(a.tobytes() + b.tobytes()).hexdigest(),
                          "out_sha256": hashlib.sha256(out.tobytes()).hexdigest()}
        if synthetic:
            manifest[name]["model_sha256"] = parity._sha256(os.path.join(synth_model, "flownet.bin"))
        print(name, out.mean())
    base = os.path.join(HERE, "golden_synth" if synthetic else "golden")
    np.savez_compressed(base + ".npz", **arrays)
    json.dump(manifest, open(base + ".json", "w"), indent=1, sort_keys=True)
    td.cleanup()


if __name__ == "__main__":
    main(synthetic="--synthetic" in sys.argv[1:])
