"""Pins the oracle (no GPU): the C++ restatement in oracle/ must reproduce the committed golden frames, which
were produced by oracle/_ref = the reference's own CPU functions + its vendored ncnn (tests/golden/make_golden.py), or --
where the reference's model files are absent and rife-v4.6 runs on the seeded synthetic weights -- by the restatement
itself on those weights (tests/golden/golden_synth.*, parity.golden_frame).
Two valid CPU builds of the reference differ by 1 LSB on ~1e-4 of the values (BASELINE.md section 5), hence the tolerance."""
import hashlib
import json
import os

import numpy as np
import pytest

import parity

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MANIFEST = json.load(open(os.path.join(GOLD, "golden.json")))
ARRAYS = np.load(os.path.join(GOLD, "golden.npz"))

FAST = ["v46_plain_128x96", "v46_plain_100x70_cpu_crop_quirk", "v46_t025_128x96", "v46_tta_96x64", "v46_temporal_96x64",
        "v46_tta_temporal_96x64", "v46_large_motion_160x96", "v4_t075_128x96", "v23_plain_128x96", "v23_uhd_128x128", "anime_plain_128x96"]


def _inputs(name):
    m = MANIFEST[name]
    a, b = parity.synth.pair(m["w"], m["h"], **m["synth_kwargs"])
    assert hashlib.sha256(a.tobytes() + b.tobytes()).hexdigest() == m["in_sha256"], "synthetic frame generator drifted"
    return m, a, b


def test_golden_file_is_intact():
    for name, m in MANIFEST.items():
        assert hashlib.sha256(ARRAYS[name].tobytes()).hexdigest() == m["out_sha256"], name
    synth = json.load(open(os.path.join(GOLD, "golden_synth.json")))
    synth_arrays = np.load(os.path.join(GOLD, "golden_synth.npz"))
    for name, m in synth.items():
        assert {k: v for k, v in m.items() if k not in ("out_sha256", "model_sha256")} == \
            {k: v for k, v in MANIFEST[name].items() if k != "out_sha256"}, name
        assert hashlib.sha256(synth_arrays[name].tobytes()).hexdigest() == m["out_sha256"], name


@pytest.mark.parametrize("name", FAST)
def test_port_reproduces_golden(name):
    if parity.port_binary() is None:
        pytest.skip("oracle/build/oracle_rife not built")
    m, a, b = _inputs(name)
    gold = parity.golden_frame(name)
    if gold is None:
        pytest.skip("model not available")
    out, _ = parity.run_oracle(m["model"], a, b, which="port", **m["oracle_kwargs"])
    res = parity.compare(out, gold)
    assert res["max_abs_diff"] <= 1 and res["share_ne"] < 2e-3, res


@pytest.mark.parametrize("name", ["v46_plain_128x96", "v23_plain_128x96", "anime_tta_temporal_96x64"])
def test_reference_binary_reproduces_golden(name):
    if parity.ref_binary() is None:
        pytest.skip("oracle/_ref not built on this host")
    m, a, b = _inputs(name)
    out, _ = parity.run_oracle(m["model"], a, b, which="ref", **m["oracle_kwargs"])
    res = parity.compare(out, ARRAYS[name])
    assert res["max_abs_diff"] <= 1 and res["share_ne"] < 2e-3, res


def test_synthetic_model_loads_in_both_oracles(tmp_path):
    """tests/make_synth_model.py writes the rife-v4.6 architecture in the reference's file format: the reference binary
    (real ncnn parser) must accept it and agree with the restatement."""
    import make_synth_model
    import subprocess
    d = make_synth_model.write_model(str(tmp_path / "rife-v4.6"), seed=1)
    assert os.path.getsize(os.path.join(d, "flownet.bin")) == 10614320  # same byte count as the reference's file
    a, b = parity.synth.pair(96, 64)
    (tmp_path / "a.rgb").write_bytes(a.tobytes())
    (tmp_path / "b.rgb").write_bytes(b.tobytes())
    outs = []
    for exe in (parity.ref_binary(), parity.port_binary()):
        if exe is None:
            continue
        o = str(tmp_path / ("o%d.rgb" % len(outs)))
        subprocess.run([exe, "--model", d, "--family", "v4", "--w", "96", "--h", "64", "--in0", str(tmp_path / "a.rgb"), "--in1", str(tmp_path / "b.rgb"),
                        "--out", o, "--threads", "4"], check=True, stdout=subprocess.PIPE)
        outs.append(np.fromfile(o, np.uint8))
    if len(outs) < 1:
        pytest.skip("no oracle executable")
    assert outs[0].std() > 5
    if len(outs) == 2:
        assert np.abs(outs[0].astype(int) - outs[1].astype(int)).max() <= 1


ALL_FAMILIES = ["rife", "rife-HD", "rife-UHD", "rife-anime", "rife-v2", "rife-v2.3", "rife-v2.4", "rife-v3.0", "rife-v3.1", "rife-v4", "rife-v4.6"]


@pytest.mark.parametrize("model", ALL_FAMILIES)
def test_port_matches_reference_binary_for_every_model_directory(model):
    """Every model directory the reference ships (SURVEY.md section 8f, N2), read from the reference tree where it is
    mounted: the C++ restatement against the reference's own CPU path.  Build-container only (the GPU box has neither the
    tree nor a need for it)."""
    md = os.path.join("/root/reference/models", model)
    if not os.path.isdir(md):
        pytest.skip("reference tree not mounted")
    if parity.ref_binary() is None or parity.port_binary() is None:
        pytest.skip("oracle executables not built")
    a, b = parity.synth.pair(96, 64)
    t = 0.25 if parity.FAMILY[model] == "v4" else 0.5
    ref, _ = parity.run_oracle(model, a, b, t, which="ref", modeldir=md, threads=4)
    port, _ = parity.run_oracle(model, a, b, t, which="port", modeldir=md, threads=4)
    res = parity.compare(port, ref)
    assert ref.std() > 5
    assert res["max_abs_diff"] <= 1 and res["share_ne"] < 2e-3, res
