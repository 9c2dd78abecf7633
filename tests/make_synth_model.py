#!/usr/bin/env python3
"""Writes a model directory with the rife-v4.6 IFNet architecture (SURVEY.md Appendix B) and seeded random weights in
the reference's on-disk format (ncnn .param text + .bin with fp16 conv weights, SURVEY.md section 3.5).

Used only when the reference's model files did not travel (no oracle/_ref/models): bench.py then reports
`"weights": "synthetic"` and the parity tests compare the CUDA path with the oracle restatement on this model.
write_model() also writes stand-ins for the other model directories (build_v4, build_3net): the same interface blobs and
layouts the engine and the oracle address, seeded weights.
The graph is written from the architecture description (blocks of conv3x3 s2, conv3x3 s2, 8 x residual conv3x3,
deconv4x4 s2 + PixelShuffle; bilinear resampling, warps, flow / mask accumulation, sigmoid blend); blob and layer
names are ours except the interface blobs in0, in1, in2, flow0..flow3, out0 that the engine addresses by name."""
import os
import struct
import sys

import numpy as np


class Graph:
    def __init__(self):
        self.layers = []   # (type, name, bottoms, tops, params-string)
        self.weights = []  # per layer: list of ("fp16"|"f32", ndarray)
        self.n = 0

    def uid(self, prefix):
        self.n += 1
        return "%s_%d" % (prefix, self.n)

    def add(self, typ, bottoms, ntop=1, params="", weights=None, top_names=None, name=None):
        name = name or self.uid(typ.lower().replace(".", "_"))
        tops = top_names or [self.uid("b") for _ in range(ntop)]
        self.layers.append([typ, name, list(bottoms), tops, params])
        self.weights.append(weights or [])
        return tops[0] if ntop == 1 else tops

    def finalize(self):
        """Insert ncnn-style Split layers for blobs with several consumers."""
        consumers = {}
        for li, L in enumerate(self.layers):
            for bi, b in enumerate(L[2]):
                consumers.setdefault(b, []).append((li, bi))
        out_layers, out_weights = [], []
        rename = {}  # (layer index, bottom index) -> new blob name
        for li, L in enumerate(self.layers):
            bottoms = [rename.get((li, bi), b) for bi, b in enumerate(L[2])]
            out_layers.append([L[0], L[1], bottoms, L[3], L[4]])
            out_weights.append(self.weights[li])
            for t in L[3]:
                cs = consumers.get(t, [])
                if len(cs) > 1:
                    names = ["%s_s%d" % (t, k) for k in range(len(cs))]
                    out_layers.append(["Split", "split_" + t, [t], names, ""])
                    out_weights.append([])
                    for (cl, cb), nn in zip(cs, names):
                        rename[(cl, cb)] = nn
        blobs = set()
        for L in out_layers:
            blobs.update(L[2])
            blobs.update(L[3])
        return out_layers, out_weights, len(blobs)


def build_v46(seed=0):
    rng = np.random.default_rng(seed)
    g = Graph()

    def conv(x, cin, cout, stride, act_leaky):
        w = (rng.standard_normal((cout, cin, 9)) * np.sqrt(2.0 / (9 * cin)) * 0.7).astype(np.float16)
        b = (rng.standard_normal(cout) * 0.02).astype(np.float32)
        p = "0=%d 1=3 %s4=1 5=1 6=%d" % (cout, "3=2 " if stride == 2 else "", w.size)
        if act_leaky:
            p += " 9=2 -23310=1,2.000000e-01"
        return g.add("Convolution", [x], params=p, weights=[("fp16", w), ("f32", b)])

    def deconv(x, cin):
        w = (rng.standard_normal((24, cin, 16)) * np.sqrt(1.0 / (4 * cin)) * 0.15).astype(np.float16)
        b = (rng.standard_normal(24) * 0.01).astype(np.float32)
        return g.add("Deconvolution", [x], params="0=24 1=4 3=2 4=1 5=1 6=%d" % w.size, weights=[("fp16", w), ("f32", b)])

    def interp(x, s):
        return g.add("Interp", [x], params="0=2 1=%e 2=%e" % (s, s))

    def crop(x, a, b):
        return g.add("Crop", [x], params="-23309=1,%d -23310=1,%d -23311=1,0" % (a, b))

    in0 = g.add("Input", [], top_names=["in0"], name="in0")
    in1 = g.add("Input", [], top_names=["in1"], name="in1")
    in2 = g.add("Input", [], top_names=["in2"], name="in2")
    widths, scales = [192, 128, 96, 64], [8, 4, 2, 1]
    F = M = None
    for k in range(4):
        c, s = widths[k], scales[k]
        if k == 0:
            x = interp(g.add("Concat", [in0, in1, in2]), 1.0 / s)
            cin = 7
        else:
            w1 = g.add("rife.Warp", [in1, crop(F, 2, 4)])
            w0 = g.add("rife.Warp", [in0, crop(F, 0, 2)])
            x = g.add("Concat", [w0, w1, in2, M])
            if s != 1:
                x = interp(x, 1.0 / s)
                fd = g.add("BinaryOp", [interp(F, 1.0 / s)], params="0=3 1=1 2=%e" % float(s))
            else:
                fd = F
            x = g.add("Concat", [x, fd])
            cin = 12
        y = conv(x, cin, c // 2, 2, True)
        y = conv(y, c // 2, c, 2, True)
        for _ in range(8):
            t = conv(y, c, c, 1, False)
            t = g.add("BinaryOp", [t, y], params="")
            y = g.add("ReLU", [t], params="0=2.000000e-01")
        d = g.add("PixelShuffle", [deconv(y, c)], params="0=2", top_names=["flow%d" % k])
        u = interp(d, float(s)) if s != 1 else d
        uf, um = crop(u, 0, 4), crop(u, 4, 5)
        if k == 0:
            F = g.add("BinaryOp", [uf], params="0=2 1=1 2=%e" % float(s))
            M = um
        elif s != 1:
            F = g.add("Eltwise", [F, uf], params="0=1 -23301=2,1.000000e+00,%e" % float(s))
            M = g.add("BinaryOp", [M, um], params="")
        else:
            F = g.add("BinaryOp", [F, uf], params="")
            M = g.add("BinaryOp", [M, um], params="")
    m = g.add("Sigmoid", [M])
    om = g.add("BinaryOp", [m], params="0=7 1=1 2=1.000000e+00")
    t1 = g.add("BinaryOp", [g.add("rife.Warp", [in1, crop(F, 2, 4)]), om], params="0=2")
    t0 = g.add("BinaryOp", [g.add("rife.Warp", [in0, crop(F, 0, 2)]), m], params="0=2")
    g.add("BinaryOp", [t0, t1], params="", top_names=["out0"])
    return g


class Ops:
    """Seeded layers on a Graph: convolutions with fp16 weights, per-channel PReLU, resampling, channel crops."""

    def __init__(self, g, rng):
        self.g, self.rng = g, rng

    def conv(self, x, cin, cout, k=3, stride=1, gain=0.7):
        w = (self.rng.standard_normal((cout, cin, k * k)) * np.sqrt(2.0 / (k * k * cin)) * gain).astype(np.float16)
        b = (self.rng.standard_normal(cout) * 0.02).astype(np.float32)
        p = "0=%d 1=%d %s4=%d 5=1 6=%d" % (cout, k, "3=2 " if stride == 2 else "", k // 2, w.size)
        return self.g.add("Convolution", [x], params=p, weights=[("fp16", w), ("f32", b)])

    def prelu(self, x, c):
        a = (0.2 + 0.1 * self.rng.random(c)).astype(np.float32)
        return self.g.add("PReLU", [x], params="0=%d" % c, weights=[("f32", a)])

    def cp(self, x, cin, cout, k=3, stride=1):
        return self.prelu(self.conv(x, cin, cout, k, stride), cout)

    def deconv(self, x, cin, cout, gain=0.15, **kw):
        w = (self.rng.standard_normal((cout, cin, 16)) * np.sqrt(1.0 / (4 * cin)) * gain).astype(np.float16)
        b = (self.rng.standard_normal(cout) * 0.01).astype(np.float32)
        return self.g.add("Deconvolution", [x], params="0=%d 1=4 3=2 4=1 5=1 6=%d" % (cout, w.size), weights=[("fp16", w), ("f32", b)], **kw)

    def interp(self, x, s):
        return self.g.add("Interp", [x], params="0=2 1=%e 2=%e" % (s, s))

    def mul(self, x, s, **kw):
        return self.g.add("BinaryOp", [x], params="0=2 1=1 2=%e" % s, **kw)

    def crop(self, x, a, b):
        return self.g.add("Crop", [x], params="-23309=1,%d -23310=1,%d -23311=1,0" % (a, b))


def build_v4(seed=0):
    """The rife-v4 layout (SURVEY.md Appendix B): per-channel PReLU after every convolution, one residual around the eight chain
    convolutions (from the second stride-2 conv's activation to after the last one), a 5-channel flow head at half the block
    resolution (blob flowK), up-sampled by 2s; the flow fed to block k is scaled by 1/s."""
    g = Graph()
    o = Ops(g, np.random.default_rng(seed))
    in0 = g.add("Input", [], top_names=["in0"], name="in0")
    in1 = g.add("Input", [], top_names=["in1"], name="in1")
    in2 = g.add("Input", [], top_names=["in2"], name="in2")
    widths, scales = [192, 128, 96, 64], [8, 4, 2, 1]
    F = M = None
    for k in range(4):
        c, s = widths[k], scales[k]
        if k == 0:
            x = o.interp(g.add("Concat", [in0, in1, in2]), 1.0 / s)
            cin = 7
        else:
            w1 = g.add("rife.Warp", [in1, o.crop(F, 2, 4)])
            w0 = g.add("rife.Warp", [in0, o.crop(F, 0, 2)])
            x = g.add("Concat", [w0, w1, in2, M])
            fd = F
            if s != 1:
                x = o.interp(x, 1.0 / s)
                fd = o.mul(o.interp(F, 1.0 / s), 1.0 / s)
            x = g.add("Concat", [x, fd])
            cin = 12
        y = o.cp(x, cin, c // 2, stride=2)
        y1 = o.cp(y, c // 2, c, stride=2)
        t = y1
        for _ in range(8):
            t = o.cp(t, c, c)
        t = g.add("BinaryOp", [t, y1], params="")
        d = o.deconv(t, c, 5, top_names=["flow%d" % k])
        u = o.interp(d, 2.0 * s)
        uf, um = o.crop(u, 0, 4), o.crop(u, 4, 5)
        if k == 0:
            F = o.mul(uf, 2.0 * s)
            M = um
        else:
            F = g.add("Eltwise", [F, uf], params="0=1 -23301=2,1.000000e+00,%e" % (2.0 * s))
            M = g.add("BinaryOp", [M, um], params="")
    m = g.add("Sigmoid", [M])
    om = g.add("BinaryOp", [m], params="0=7 1=1 2=1.000000e+00")
    t1 = g.add("BinaryOp", [g.add("rife.Warp", [in1, o.crop(F, 2, 4)]), om], params="0=2")
    t0 = g.add("BinaryOp", [g.add("rife.Warp", [in0, o.crop(F, 0, 2)]), m], params="0=2")
    g.add("BinaryOp", [t0, t1], params="", top_names=["out0"])
    return g


def build_3net(v2, seed=0):
    """flownet / contextnet / fusionnet with the interface blobs of the reference's v1 (rife, rife-HD, rife-UHD, rife-anime) and
    v2 (rife-v2 .. rife-v3.1) families -- input0, input1 -> flow (half resolution; 4 channels for v2, 2 for v1); input.1 + flow.0
    (v1: flow.1 = -flow.0, injectable) -> f1..f4 at 1/2..1/16; img0, img1, flow, 3..6, 7..10 -> output -- and a small seeded body
    (5x5 convolutions in the v1 flownet, per-channel PReLU, warps, a sigmoid blend)."""
    rng = np.random.default_rng(seed)
    nf = 4 if v2 else 2
    # flownet
    g = Graph()
    o = Ops(g, rng)
    a = g.add("Input", [], top_names=["input0"], name="input0")
    b = g.add("Input", [], top_names=["input1"], name="input1")
    x = o.cp(g.add("Concat", [a, b]), 6, 32, k=3 if v2 else 5, stride=2)
    x = o.cp(x, 32, 48, stride=2)
    x = o.cp(x, 48, 48)
    o.mul(o.deconv(x, 48, nf, gain=0.3), 4.0, top_names=["flow"])
    flownet = g
    # contextnet
    g = Graph()
    o = Ops(g, rng)
    img = g.add("Input", [], top_names=["input.1"], name="input.1")
    fl = g.add("Input", [], top_names=["flow.0"], name="flow.0")
    if not v2:
        fl = g.add("UnaryOp", [fl], params="0=1", top_names=["flow.1"])
    widths = [8, 16, 16, 16]
    x, cin = img, 3
    for k in range(4):
        x = o.cp(x, cin, widths[k], stride=2)
        cin = widths[k]
        if k:
            fl = o.mul(o.interp(fl, 0.5), 0.5)
        g.add("rife.Warp", [x, fl], top_names=["f%d" % (k + 1)])
    contextnet = g
    # fusionnet
    g = Graph()
    o = Ops(g, rng)
    i0 = g.add("Input", [], top_names=["img0"], name="img0")
    i1 = g.add("Input", [], top_names=["img1"], name="img1")
    fl = g.add("Input", [], top_names=["flow"], name="flow")
    feats = [(g.add("Input", [], top_names=[str(3 + k)], name=str(3 + k)), g.add("Input", [], top_names=[str(7 + k)], name=str(7 + k))) for k in range(4)]
    fu = o.mul(o.interp(fl, 2.0), 2.0)
    w0 = g.add("rife.Warp", [i0, o.crop(fu, 0, 2)])
    w1 = g.add("rife.Warp", [i1, o.crop(fu, 2, 4) if v2 else g.add("UnaryOp", [fu], params="0=1")])
    x, cin = g.add("Concat", [w0, w1, fu]), 6 + nf
    skips = []
    for k in range(4):
        x = o.cp(x, cin, 16, stride=2)
        x = o.cp(g.add("Concat", [x, feats[k][0], feats[k][1]]), 16 + 2 * widths[k], 16)
        skips.append(x)
        cin = 16
    x = skips[3]
    for k in (2, 1, 0):
        x = o.prelu(o.deconv(x, 16, 16, gain=1.0), 16)
        x = g.add("Concat", [x, skips[k]])
        x = o.cp(x, 32, 16)
    x = o.deconv(x, 16, 4, gain=0.5)
    m = g.add("Sigmoid", [o.crop(x, 3, 4)])
    om = g.add("BinaryOp", [m], params="0=7 1=1 2=1.000000e+00")
    r = o.mul(g.add("Sigmoid", [o.crop(x, 0, 3)]), 0.1)
    blend = g.add("BinaryOp", [g.add("BinaryOp", [w0, m], params="0=2"), g.add("BinaryOp", [w1, om], params="0=2")], params="")
    g.add("BinaryOp", [blend, r], params="", top_names=["output"])
    return {"flownet": flownet, "contextnet": contextnet, "fusionnet": g}


# one seed per model directory, so that directories of one family do not share weights
SEEDS = {"rife-v4.6": 0, "rife-v4": 1, "rife": 2, "rife-HD": 3, "rife-UHD": 4, "rife-anime": 5, "rife-v2": 6, "rife-v2.3": 7, "rife-v2.4": 8,
         "rife-v3.0": 9, "rife-v3.1": 10}


def _write_net(dirpath, name, graph):
    layers, weights, nblobs = graph.finalize()
    with open(os.path.join(dirpath, name + ".param"), "w") as f:
        f.write("7767517\n%d %d\n" % (len(layers), nblobs))
        for typ, lname, bottoms, tops, params in layers:
            f.write("%-24s %-24s %d %d %s %s\n" % (typ, lname, len(bottoms), len(tops), " ".join(bottoms + tops), params))
    with open(os.path.join(dirpath, name + ".bin"), "wb") as f:
        for ws in weights:
            for kind, arr in ws:
                if kind == "fp16":
                    f.write(struct.pack("<I", 0x01306B47))
                    raw = np.ascontiguousarray(arr, dtype=np.float16).tobytes()
                    f.write(raw)
                    f.write(b"\0" * ((-len(raw)) % 4))
                else:
                    f.write(np.ascontiguousarray(arr, dtype=np.float32).tobytes())


def write_model(dirpath, seed=0, model="rife-v4.6"):
    """Writes the synthetic model directory `model` (one of SEEDS) with the given seed."""
    os.makedirs(dirpath, exist_ok=True)
    if model == "rife-v4.6":
        nets = {"flownet": build_v46(seed)}
    elif model == "rife-v4":
        nets = {"flownet": build_v4(seed)}
    else:
        nets = build_3net(model.startswith("rife-v"), seed)
    for name, graph in nets.items():
        _write_net(dirpath, name, graph)
    return dirpath


if __name__ == "__main__":
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.abspath(__file__)), "models", "rife-v4.6")
    print(write_model(out))
