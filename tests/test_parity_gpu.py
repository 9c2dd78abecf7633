"""GPU parity: CUDA path (through the C ABI) vs the oracle on seeded synthetic frame pairs.
Tolerance (BASELINE.json north_star): <= 1 LSB per RGB channel, PSNR > 50 dB.
precision 0 = fp32 CUDA-core kernels for every layer ("exact" tier); 1 = tcgen05 tensor-core convolutions with
split-fp16 (hi+lo) activations; 2 = tcgen05 with plain fp16 activations."""
import json
import os

import numpy as np
import pytest

import parity

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _need(model):
    if parity.model_dir(model) is None:
        pytest.skip("model %s not shipped to this box" % model)


def _ok(res):
    assert res["max_abs_diff"] <= 1 and res["psnr_db"] > 50, res
    assert res["out_std"] > 5, res


@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("w,h", [(256, 256), (640, 360), (96, 64)])
def test_v46_plain(pkg, w, h, precision):
    _need("rife-v4.6")
    _ok(parity.check_case(pkg, "rife-v4.6", w, h, options={"precision": precision}))


@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("t", [0.25, 0.75])
def test_v4_timesteps(pkg, t, precision):
    _need("rife-v4")
    _ok(parity.check_case(pkg, "rife-v4", 256, 192, timestep=t, options={"precision": precision}))


@pytest.mark.parametrize("precision", [0, 1])
def test_v23_config1(pkg, precision):
    _need("rife-v2.3")
    _ok(parity.check_case(pkg, "rife-v2.3", 256, 256, options={"precision": precision}))


def test_anime_plain(pkg):
    _need("rife-anime")
    _ok(parity.check_case(pkg, "rife-anime", 256, 192, options={"precision": 0}))


@pytest.mark.parametrize("model,tta,ttat,precision", [("rife-v4.6", True, False, 0), ("rife-v4.6", False, True, 1), ("rife-v4.6", True, True, 1),
                                                       ("rife-anime", True, True, 0), ("rife-v2.3", True, True, 0), ("rife-v2.3", False, True, 0)])
def test_tta_modes(pkg, model, tta, ttat, precision):
    _need(model)
    _ok(parity.check_case(pkg, model, 160, 96, tta=tta, tta_temporal=ttat, options={"precision": precision}))


@pytest.mark.parametrize("model", ["rife-v2.3", "rife-anime"])
def test_uhd_mode(pkg, model):
    _need(model)
    _ok(parity.check_case(pkg, model, 256, 192, uhd=True, options={"precision": 0}))


def test_timestep_edges_copy_inputs(pkg):
    _need("rife-v4.6")
    a, b = parity.synth.pair(64, 64)
    assert np.array_equal(parity.run_gpu(pkg, "rife-v4.6", a, b, 0.0), a)
    assert np.array_equal(parity.run_gpu(pkg, "rife-v4.6", a, b, 1.0), b)


@pytest.mark.parametrize("precision", [0, 1])
def test_large_motion(pkg, precision):
    _need("rife-v4.6")
    _ok(parity.check_case(pkg, "rife-v4.6", 640, 352, dx=24, dy=16, options={"precision": precision}))


def test_golden_frames(pkg):
    """Committed golden frames (made by oracle/_ref, or by the restatement on the synthetic rife-v4.6 weights where the
    reference's model files are absent: parity.golden_frame): no oracle execution needed here."""
    manifest = json.load(open(os.path.join(GOLD, "golden.json")))
    checked = 0
    for name, m in manifest.items():
        gold = parity.golden_frame(name)
        if gold is None:
            continue
        a, b = parity.synth.pair(m["w"], m["h"], **m["synth_kwargs"])
        kw = dict(m["oracle_kwargs"])
        # the goldens are outputs of the reference's CPU path: ragged widths carry its contiguous-read quirk (rife.cpp:4375-4387)
        opts = {"cpu_crop_quirk": 1} if m["w"] % 32 and not kw.get("tta", False) else None
        out = parity.run_gpu(pkg, m["model"], a, b, kw.pop("timestep", 0.5), kw.get("tta", False), kw.get("tta_temporal", False), kw.get("uhd", False), options=opts)
        res = parity.compare(out, gold)
        assert res["max_abs_diff"] <= 1 and res["psnr_db"] > 50, (name, res)
        checked += 1
    assert checked > 0


def test_batch_and_device_entry_points_match_process(pkg):
    _need("rife-v4.6")
    import ctypes
    w, h = 256, 192
    frames = [parity.synth.frame(k, w, h) for k in range(4)]
    v2, v4 = pkg.family_flags("rife-v4.6")
    r = pkg.RIFE(0, False, False, False, 1, v2, v4)
    r.load(parity.model_dir("rife-v4.6"))
    singles = [r.process(frames[i], frames[i + 1], 0.5) for i in range(3)]
    outs = [np.empty_like(frames[0]) for _ in range(3)]
    r.process_batch_ptr([f.ctypes.data for f in frames[:3]], [f.ctypes.data for f in frames[1:]], w, h, [0.5] * 3, [o.ctypes.data for o in outs])
    for s, o in zip(singles, outs):
        assert np.array_equal(s, o)
    # more lanes than pairs, fewer lanes than pairs, timestep edge inside a batch
    r.set_option("lanes", 3)
    outs2 = [np.empty_like(frames[0]) for _ in range(3)]
    r.process_batch_ptr([f.ctypes.data for f in frames[:3]], [f.ctypes.data for f in frames[1:]], w, h, [0.5, 1.0, 0.5], [o.ctypes.data for o in outs2])
    assert np.array_equal(outs2[0], singles[0]) and np.array_equal(outs2[1], frames[2]) and np.array_equal(outs2[2], singles[2])
    r.close()


@pytest.mark.parametrize("w,h", [(256, 256), (640, 360), (100, 70), (1920, 1080)])
def test_v46_fused_fast_path(pkg, w, h):
    """The hand-scheduled rife-v4.6 path (fused head / update / tail kernels + tcgen05 convs): active after its
    load-time self-check, equal to the generic executor up to fp32 rounding, and within tolerance of the oracle."""
    _need("rife-v4.6")
    a, b = parity.synth.pair(w, h)
    v2, v4 = pkg.family_flags("rife-v4.6")
    r = pkg.RIFE(0, False, False, False, 1, v2, v4)
    r.load(parity.model_dir("rife-v4.6"))
    assert r.get_option("fast_active") == 1
    fast = r.process(a, b, 0.5)
    r.set_option("fast", 0)
    assert r.get_option("fast_active") == 0
    generic = r.process(a, b, 0.5)
    r.close()
    d = parity.compare(fast, generic)
    assert d["max_abs_diff"] <= 1 and d["share_ne"] < 5e-3, d
    if w % 32 == 0:  # ragged widths: see test_ragged_widths_crop_the_padded_output
        ref, _ = parity.run_oracle("rife-v4.6", a, b, 0.5)
        res = parity.compare(fast, ref)
        assert res["max_abs_diff"] <= 1 and res["psnr_db"] > 50, res


@pytest.mark.parametrize("mask", [0, 12, 15])
@pytest.mark.parametrize("case", ["synth", "large_motion", "readme_images"])
def test_v46_precision_choices_stay_within_one_lsb(pkg, mask, case):
    """plain_blocks: which IFBlocks run their residual chain on plain fp16 activations (default 12 = blocks 2,3).
    The all-split tier (0) and the shipped default (12) must stay within 1 LSB / 50 dB of the oracle; the opt-in
    all-plain tier (15) is allowed a 2-LSB difference on at most 1e-4 of the values (it sits at the edge: a handful of
    pixels of the README frames reach 2)."""
    _need("rife-v4.6")
    if case == "synth":
        a, b = parity.synth.pair(640, 360)
    elif case == "large_motion":
        a, b = parity.synth.pair(640, 352, dx=24, dy=16)
    else:
        try:
            from PIL import Image
            d = os.path.join(parity.REF_DIR, "images")
            a = np.array(Image.open(os.path.join(d, "0.png")).convert("RGB"))
            b = np.array(Image.open(os.path.join(d, "1.png")).convert("RGB"))
        except Exception:
            pytest.skip("README frames or PIL not available")
    ref, _ = parity.run_oracle("rife-v4.6", a, b, 0.5)
    out = parity.run_gpu(pkg, "rife-v4.6", a, b, 0.5, options={"plain_blocks": mask})
    res = parity.compare(out, ref)
    if mask == 15:
        assert res["max_abs_diff"] <= 2 and res["share_ge2"] < 1e-4 and res["psnr_db"] > 50 and res["share_ne"] < 0.02, res
    else:
        assert res["max_abs_diff"] <= 1 and res["psnr_db"] > 50 and res["share_ne"] < 0.02, res


def test_concurrent_process_calls_on_one_handle(pkg):
    """The reference calls RIFE::process from several proc threads on one object (src/main.cpp:346-366)."""
    _need("rife-v4.6")
    import threading
    w, h = 320, 192
    frames = [parity.synth.frame(k, w, h) for k in range(5)]
    v2, v4 = pkg.family_flags("rife-v4.6")
    r = pkg.RIFE(0, False, False, False, 1, v2, v4)
    r.load(parity.model_dir("rife-v4.6"))
    expect = [r.process(frames[i], frames[i + 1], 0.5) for i in range(4)]
    got = [None] * 4
    errs = []

    def work(i):
        try:
            for _ in range(3):
                got[i] = r.process(frames[i], frames[i + 1], 0.5)
        except Exception as e:  # pragma: no cover
            errs.append(e)

    ts = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    r.close()
    assert not errs, errs
    for e, g_ in zip(expect, got):
        assert np.array_equal(e, g_)


def test_batched_lockstep_equals_single_pair_path(pkg):
    """8 pairs in one lock-step batch (TMA 4D tensor maps, blockIdx.z image index) vs the same pairs one at a time."""
    _need("rife-v4.6")
    w, h = 256, 160
    frames = [parity.synth.frame(k, w, h, dx=5, dy=3) for k in range(9)]
    v2, v4 = pkg.family_flags("rife-v4.6")
    r = pkg.RIFE(0, False, False, False, 1, v2, v4)
    r.load(parity.model_dir("rife-v4.6"))
    r.set_option("lanes", 1)
    singles = [r.process(frames[i], frames[i + 1], 0.25 + 0.0625 * i) for i in range(8)]
    outs = [np.empty_like(frames[0]) for _ in range(8)]
    r.set_option("batch", 8)
    r.process_batch_ptr([f.ctypes.data for f in frames[:8]], [f.ctypes.data for f in frames[1:]], w, h, [0.25 + 0.0625 * i for i in range(8)],
                        [o.ctypes.data for o in outs])
    r.close()
    for s_, o in zip(singles, outs):
        assert np.array_equal(s_, o)


@pytest.mark.parametrize("w,h", [(256, 160), (100, 70), (1920, 1080)])
def test_v46_recompute_fm_modes_are_bit_identical(pkg, w, h):
    """recompute_fm 1 / 2: the full-resolution flow / mask planes are rebuilt from the per-block flow tensors instead of
    being stored and re-read (fused_v46.cu).  Same operations in the same order, so the frames must be identical -- for a
    single pair, for a lock-step batch with different timesteps, and for a ragged size (w % 32 != 0), there with and without
    the contiguous-read quirk of src/rife.cpp:4375-4387."""
    _need("rife-v4.6")
    nb = 3 if w * h > 1000000 else 8
    frames = [parity.synth.frame(k, w, h, dx=5, dy=3) for k in range(nb + 1)]
    ts = [0.25 + 0.0625 * i for i in range(nb)]
    v2, v4 = pkg.family_flags("rife-v4.6")
    r = pkg.RIFE(0, False, False, False, 1, v2, v4)
    r.load(parity.model_dir("rife-v4.6"))
    assert r.get_option("fast_active") == 1
    r.set_option("lanes", 1)
    r.set_option("batch", nb)
    r.set_option("cpu_crop_quirk", 1 if (w, h) == (100, 70) else 0)
    results = {}
    for mode in (0, 1, 2):
        r.set_option("recompute_fm", mode)
        assert r.get_option("recompute_fm") == mode
        single = r.process(frames[0], frames[1], 0.5)
        outs = [np.empty_like(frames[0]) for _ in range(nb)]
        r.process_batch_ptr([f.ctypes.data for f in frames[:nb]], [f.ctypes.data for f in frames[1:]], w, h, ts, [o.ctypes.data for o in outs])
        results[mode] = [single] + outs
    r.close()
    assert results[0][0].std() > 5
    for mode in (1, 2):
        for a_, b_ in zip(results[0], results[mode]):
            assert np.array_equal(a_, b_), (mode, parity.compare(a_, b_))


def test_concurrent_process_calls_are_combined_into_batches(pkg):
    """Option "combine": process() calls arriving from several threads while another call is being served run as one
    lock-step batch (csrc/combiner.h) -- the reference CLI's `-j load:proc:save` threading (src/main.cpp:346-366).
    Results must equal the one-at-a-time results bit for bit, and some batching must actually have happened."""
    _need("rife-v4.6")
    import threading
    w, h = 320, 192
    frames = [parity.synth.frame(k, w, h) for k in range(9)]
    v2, v4 = pkg.family_flags("rife-v4.6")
    r = pkg.RIFE(0, False, False, False, 1, v2, v4)
    r.load(parity.model_dir("rife-v4.6"))
    r.set_option("combine", 0)
    expect = [r.process(frames[i], frames[i + 1], 0.5) for i in range(8)]
    r.set_option("combine", 1)
    nb0, nr0 = r.get_option("combined_batches"), r.get_option("combined_requests")
    got = [None] * 8
    errs = []
    gate = threading.Barrier(8)

    def work(i):
        try:
            gate.wait()
            for _ in range(4):
                got[i] = r.process(frames[i], frames[i + 1], 0.5)
        except Exception as e:  # pragma: no cover
            errs.append(e)

    ts = [threading.Thread(target=work, args=(i,)) for i in range(8)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    nb, nr = r.get_option("combined_batches") - nb0, r.get_option("combined_requests") - nr0
    r.close()
    assert not errs, errs
    for e, g_ in zip(expect, got):
        assert np.array_equal(e, g_)
    assert nr == 32 and nb < nr, (nb, nr)


# ---- round 2: the resolutions the metric is quoted on, the other model directories, the boundary options ------------------------

def _batch_vs_oracle(pkg, model, w, h, ts, lanes=2, threads=None):
    """len(ts) consecutive pairs of the synthetic stream through ONE process_batch call (lock-step batches on the fused path),
    each pair with its own timestep, every output compared with the oracle's frame for that pair."""
    n = len(ts)
    frames = [parity.synth.frame(k, w, h) for k in range(n + 1)]
    v2, v4 = pkg.family_flags(model)
    r = pkg.RIFE(0, False, False, False, 1, v2, v4)
    r.load(parity.model_dir(model))
    r.set_option("lanes", lanes)
    fast = r.get_option("fast_active")
    outs = [np.empty_like(frames[0]) for _ in range(n)]
    r.process_batch_ptr([f.ctypes.data for f in frames[:n]], [f.ctypes.data for f in frames[1:]], w, h, ts, [o.ctypes.data for o in outs])
    r.close()
    worst = None
    for i in range(n):
        ref, info = parity.run_oracle(model, frames[i], frames[i + 1], ts[i], threads=threads)
        res = parity.compare(outs[i], ref)
        assert res["max_abs_diff"] <= 1 and res["psnr_db"] > 50, (model, w, h, i, ts[i], res)
        assert outs[i].std() > 5
        if worst is None or res["psnr_db"] < worst["psnr_db"]:
            worst = res
    return fast, worst


def test_v46_1080p_lockstep_batch_vs_oracle(pkg):
    """BASELINE configs[1] at its own resolution: 8 pairs of 1920x1080 in one lock-step batch, distinct timesteps, vs the oracle."""
    _need("rife-v4.6")
    fast, worst = _batch_vs_oracle(pkg, "rife-v4.6", 1920, 1080, [0.5, 0.25, 0.75, 0.5, 0.125, 0.625, 0.5, 0.875])
    assert fast == 1
    print("1080p worst pair:", worst)


def test_v46_4k_lockstep_batch_vs_oracle(pkg):
    """BASELINE configs[2] at its own resolution: 3840x2160 (padded to 3840x2176), two pairs per lock-step batch, vs the oracle."""
    _need("rife-v4.6")
    fast, worst = _batch_vs_oracle(pkg, "rife-v4.6", 3840, 2160, [0.5, 0.25])
    assert fast == 1
    print("4K worst pair:", worst)


def test_v4_1080p_timestep_sweep_vs_oracle(pkg):
    """BASELINE configs[4]: rife-v4, the -n 4x schedule t = 0.25, 0.5, 0.75 at 1080p, on the fused path of the rife-v4 layout."""
    _need("rife-v4")
    fast, worst = _batch_vs_oracle(pkg, "rife-v4", 1920, 1080, [0.25, 0.5, 0.75])
    assert fast == 1
    print("rife-v4 1080p worst pair:", worst)


@pytest.mark.parametrize("w,h", [(256, 256), (640, 360), (100, 70)])
def test_v4_fused_path_matches_generic_executor(pkg, w, h):
    """The hand-scheduled path of the rife-v4 layout (PReLU, one residual per chain, 5-channel flow heads at half the block
    resolution): active after the load-time self-check, equal to the generic executor up to fp32 rounding, within tolerance
    of the oracle."""
    _need("rife-v4")
    a, b = parity.synth.pair(w, h)
    r = pkg.RIFE(0, False, False, False, 1, False, True)
    r.load(parity.model_dir("rife-v4"))
    assert r.get_option("fast_active") == 1
    fast = r.process(a, b, 0.3)
    r.set_option("fast", 0)
    generic = r.process(a, b, 0.3)
    r.close()
    d = parity.compare(fast, generic)
    assert d["max_abs_diff"] <= 1 and d["share_ne"] < 5e-3, d
    if w % 32 == 0:
        ref, _ = parity.run_oracle("rife-v4", a, b, 0.3)
        res = parity.compare(fast, ref)
        assert res["max_abs_diff"] <= 1 and res["psnr_db"] > 50, res


ALL_MODELS = ["rife", "rife-HD", "rife-UHD", "rife-anime", "rife-v2", "rife-v2.3", "rife-v2.4", "rife-v3.0", "rife-v3.1", "rife-v4", "rife-v4.6"]


@pytest.mark.parametrize("model", ALL_MODELS)
def test_every_model_directory_vs_oracle(pkg, model):
    """SURVEY.md section 8f, N2: every model directory the reference ships (src/main.cpp:658-683 sniffs them all), default
    precision tier, against the oracle."""
    _need(model)
    t = 0.5 if parity.FAMILY[model] != "v4" else 0.4
    _ok(parity.check_case(pkg, model, 256, 192, timestep=t))


@pytest.mark.parametrize("model,uhd", [("rife-UHD", True), ("rife-v3.1", True), ("rife-HD", False)])
def test_more_models_with_tta(pkg, model, uhd):
    """UHD cases use a size whose halves are multiples of 32: the reference's CPU path pads to 32 also in UHD mode
    (rife.cpp:1238-1240), halves the padded frame and runs the flownet on it (rife.cpp:2212-2228); at 160x96 the 80x48 input makes
    the flownet's pyramid levels disagree in size and the reference binary (and the restatement, faithfully) corrupts its heap --
    there is no reference output to compare with."""
    _need(model)
    w, h = (192, 128) if uhd else (160, 96)
    _ok(parity.check_case(pkg, model, w, h, tta=True, tta_temporal=True, uhd=uhd))


@pytest.mark.parametrize("model,fast", [("rife-v4.6", 1), ("rife-v4.6", 0), ("rife-v4", 1), ("rife-v2.3", 0)])
@pytest.mark.parametrize("w,h", [(100, 70), (90, 50)])
def test_ragged_widths_crop_the_padded_output(pkg, model, fast, w, h):
    """w % 32 != 0.  Default: the frame is the crop of the padded result (what the reference's GPU path produces,
    rife_postproc.comp:42) -- checked against the restatement run with --crop-padded AND through a size-independent property:
    it must equal the crop of the result for the same frames zero-padded to the padded size by the caller (same arithmetic,
    bit for bit).  Option cpu_crop_quirk = 1: the reference CPU path's sheared frame (rife.cpp:4375-4387), checked against the
    reference binary itself."""
    _need(model)
    a, b = parity.synth.pair(w, h)
    opts = {"fast": fast}
    v2, v4 = pkg.family_flags(model)
    t = 0.5
    r = pkg.RIFE(0, False, False, False, 1, v2, v4)
    r.load(parity.model_dir(model))
    r.set_option("fast", fast)
    out = r.process(a, b, t)
    wp, hp = (w + 31) // 32 * 32, (h + 31) // 32 * 32
    ap, bp = np.zeros((hp, wp, 3), np.uint8), np.zeros((hp, wp, 3), np.uint8)
    ap[:h, :w], bp[:h, :w] = a, b
    full = r.process(ap, bp, t)
    r.set_option("cpu_crop_quirk", 1)
    quirk = r.process(a, b, t)
    r.close()
    assert np.array_equal(out, full[:h, :w])
    res = parity.compare(out, parity.run_oracle(model, a, b, t, crop_padded=True)[0])
    assert res["max_abs_diff"] <= 1 and res["psnr_db"] > 50, res
    res = parity.compare(quirk, parity.run_oracle(model, a, b, t)[0])
    assert res["max_abs_diff"] <= 1 and res["psnr_db"] > 50, res
    assert not np.array_equal(out, quirk)
    del opts


@pytest.mark.parametrize("model,tta", [("rife-v4.6", False), ("rife-v4.6", True), ("rife-v2.3", False)])
def test_bgr_frames(pkg, model, tta):
    """Option "bgr" (the reference's Windows build hands over B,G,R frames, rife_preproc.comp:13,53-56): processing the
    channel-swapped frames with the option on must give the channel-swapped result, bit for bit."""
    _need(model)
    a, b = parity.synth.pair(160, 96)
    v2, v4 = pkg.family_flags(model)
    r = pkg.RIFE(0, tta, False, False, 1, v2, v4)
    r.load(parity.model_dir(model))
    rgb = r.process(a, b, 0.5)
    r.set_option("bgr", 1)
    bgr = r.process(np.ascontiguousarray(a[:, :, ::-1]), np.ascontiguousarray(b[:, :, ::-1]), 0.5)
    r.close()
    assert np.array_equal(bgr[:, :, ::-1], rgb)


def test_frame_cache_reuses_uploads_across_calls(pkg):
    """Option "frame_cache" (SURVEY.md 8f, N1): frame k+1 of pair (k, k+1) is found on the device when pair (k+1, k+2) arrives."""
    _need("rife-v4.6")
    w, h = 320, 192
    frames = [parity.synth.frame(k, w, h) for k in range(6)]
    r = pkg.RIFE(0, False, False, False, 1, False, True)
    r.load(parity.model_dir("rife-v4.6"))
    expect = [r.process(frames[i], frames[i + 1], 0.5) for i in range(5)]
    assert r.get_option("frame_cache_hits") == 0
    h2d0 = pkg.copy_bytes()[0]
    r.set_option("frame_cache", 1)
    got = [r.process(frames[i], frames[i + 1], 0.5) for i in range(5)]
    hits = r.get_option("frame_cache_hits")
    h2d = pkg.copy_bytes()[0] - h2d0
    # a buffer whose content changed must be announced
    frames[5][:] = frames[0]
    r.forget_frames()
    again = r.process(frames[4], frames[5], 0.5)
    fresh = pkg.RIFE(0, False, False, False, 1, False, True)
    fresh.load(parity.model_dir("rife-v4.6"))
    want = fresh.process(frames[4], frames[5], 0.5)
    fresh.close()
    r.close()
    for e, g_ in zip(expect, got):
        assert np.array_equal(e, g_)
    assert hits == 4 and h2d == 6 * w * h * 3, (hits, h2d)
    assert np.array_equal(again, want)


def test_long_stream_recycles_the_frame_table(pkg):
    """One process_batch call with more distinct frames (141) than the frame table holds (66): entries are recycled while lanes
    still read earlier chunks (an upload into a recycled entry waits for the lane that read it).  Every result must equal the
    single-call result for the same pair, bit for bit; then a call with a larger frame size on the same handle (the table drops
    its undersized buffers in one go), and the first size again."""
    _need("rife-v4.6")
    w, h = 160, 96
    n = 140
    frames = parity.synth.stream(0, n + 1, w, h)
    r = pkg.RIFE(0, False, False, False, 1, False, True)
    r.load(parity.model_dir("rife-v4.6"))
    outs = [np.empty_like(frames[0]) for _ in range(n)]
    ts = [0.5 if i % 3 else 0.25 for i in range(n)]
    h2d0 = pkg.copy_bytes()[0]
    r.process_batch_ptr([f.ctypes.data for f in frames[:n]], [f.ctypes.data for f in frames[1:]], w, h, ts, [o.ctypes.data for o in outs])
    assert pkg.copy_bytes()[0] - h2d0 == (n + 1) * w * h * 3  # every frame of the stream went up exactly once
    for i in (0, 1, 7, 8, 63, 64, 65, 66, 67, 100, 131, 132, n - 1):
        assert np.array_equal(outs[i], r.process(frames[i], frames[i + 1], ts[i])), i
    w2, h2 = 256, 192
    big = parity.synth.stream(0, 12, w2, h2)
    outs2 = [np.empty_like(big[0]) for _ in range(11)]
    r.process_batch_ptr([f.ctypes.data for f in big[:11]], [f.ctypes.data for f in big[1:]], w2, h2, [0.5] * 11, [o.ctypes.data for o in outs2])
    for i in (0, 5, 10):
        assert np.array_equal(outs2[i], r.process(big[i], big[i + 1], 0.5)), i
    outs3 = [np.empty_like(frames[0]) for _ in range(n)]
    r.process_batch_ptr([f.ctypes.data for f in frames[:n]], [f.ctypes.data for f in frames[1:]], w, h, ts, [o.ctypes.data for o in outs3])
    r.close()
    for a_, b_ in zip(outs, outs3):
        assert np.array_equal(a_, b_)


def test_failed_reload_leaves_the_engine_usable(pkg):
    """load_packed with a damaged blob on a loaded engine must fail without touching the loaded model (transactional load)."""
    _need("rife-v4.6")
    a, b = parity.synth.pair(256, 160)
    r = pkg.RIFE(0, False, False, False, 1, False, True)
    r.load(parity.model_dir("rife-v4.6"))
    before = r.process(a, b, 0.5)
    blob = r.export_weights().copy()
    bad = blob[: len(blob) // 2]
    with pytest.raises(pkg.RifeError):
        r.load_packed(bad)
    bad2 = blob.copy()
    bad2[12:20] = 255  # param length = 2^64 - 1: must be rejected, not wrapped around
    with pytest.raises(pkg.RifeError):
        r.load_packed(bad2)
    assert r.get_option("fast_active") == 1
    assert np.array_equal(r.process(a, b, 0.5), before)
    r.load_packed(blob)
    assert np.array_equal(r.process(a, b, 0.5), before)
    r.close()


def test_null_frame_in_a_batch_is_rejected_before_anything_is_queued(pkg):
    _need("rife-v4.6")
    w, h = 128, 96
    frames = [parity.synth.frame(k, w, h) for k in range(4)]
    r = pkg.RIFE(0, False, False, False, 1, False, True)
    r.load(parity.model_dir("rife-v4.6"))
    outs = [np.full_like(frames[0], 7) for _ in range(3)]
    with pytest.raises(pkg.RifeError):
        r.process_batch_ptr([frames[0].ctypes.data, frames[1].ctypes.data, None], [f.ctypes.data for f in frames[1:]], w, h, [0.5] * 3, [o.ctypes.data for o in outs])
    assert all((o == 7).all() for o in outs)  # nothing was written
    ok = r.process(frames[0], frames[1], 0.5)
    r.close()
    assert ok.std() > 5


@pytest.mark.parametrize("model", ["rife-v4.6", "rife-v4"])
@pytest.mark.parametrize("case", ["synth", "large_motion", "readme_images"])
def test_packed_head_tensors_are_an_opt_in_approximation(pkg, model, case):
    """Option "head_pack" (default OFF): the block-head tensors as ONE fp16 plane whose slots 12..15 carry the lo parts of the
    four flow channels (fused_v46_kernels.cuh: 32 instead of 64 bytes per pixel, half the tensor work in the first stride-2
    conv, +6.7 % fps).  Measured in round 2 (profiles/r2_s2): the synthetic rife-v4.6 pairs stay within 1 LSB, but the README
    frames reach 7 LSB on 0.03 % of the values and rife-v4 2-3 LSB -- the warped frames / mask need their lo parts too -- so it
    does NOT meet the +-1 LSB bar and is not the default.  This test pins what the option does deliver (PSNR > 60 dB, fewer
    than 0.1 % of the values off by 2 or more) and that the default, on the same pair, stays within 1 LSB."""
    _need(model)
    if case == "synth":
        a, b = parity.synth.pair(640, 360)
    elif case == "large_motion":
        a, b = parity.synth.pair(640, 352, dx=24, dy=16)
    else:
        try:
            from PIL import Image
            d = os.path.join(parity.REF_DIR, "images")
            a = np.array(Image.open(os.path.join(d, "0.png")).convert("RGB"))
            b = np.array(Image.open(os.path.join(d, "1.png")).convert("RGB"))
        except Exception:
            pytest.skip("README frames or PIL not available")
    base = {"cpu_crop_quirk": 1} if a.shape[1] % 32 else {}
    ref, _ = parity.run_oracle(model, a, b, 0.5)
    res = parity.compare(parity.run_gpu(pkg, model, a, b, 0.5, options=dict(base, head_pack=1)), ref)
    assert res["max_abs_diff"] <= 8 and res["psnr_db"] > 60 and res["share_ge2"] < 1e-3, res
    res0 = parity.compare(parity.run_gpu(pkg, model, a, b, 0.5, options=base), ref)
    assert res0["max_abs_diff"] <= 1 and res0["psnr_db"] > 50, res0
