"""-m gpu: every layer of loaded CUNet / UpCUNet engines against float64 torch.nn.functional on the CPU.

Each layer is fed the engine's own input tensors for that layer (w2x_layer_tensor, include/w2x_dev.h), so errors do not compound and a
failure names one layer.  The wiring (each layer's producer, the skip tensors and their crops, the SE producers) is nunif's, restated from
oracle/models.py; the weights are those of the torch model, rounded the way the pack stores them (fp16 RN, or TF32 RN for tf32 engines).

Checked per engine: every conv layer (bound from the magnitude sum), the fused RGB first layer, the squeeze-excite channel sums, the
excite gate (against the engine's own sums, tight, and against the mean of the engine's output, end to end), the per-image folded
weights (bit-exact), the SE consumers, the final layer with its clamp.  Besides: the kernel variants the planner picked across all
audited engines (pinned), partial batches, slot permutation, the render path's last, partial batch against infer, a model whose SE gates
reach below 1e-3 and above 0.999, and power checks showing that each bar rejects the fault it exists for.

Engines (name: precision, scale, tile, batch, images given to infer) and why each is here:
- f16_2x_t38:  the smallest 2x tile; odd intermediate extents (17, 15, 13), pixel tiles partial on both edges, fewer tiles than SMs.
- f16_2x_t66:  partial batch (3 of 4 slots); odd extents (31, 29, 27); also the slot-permutation and render engine.
- f16_2x_t130: mid size: the down-sampled UNet1 extent is 63 (odd), several pixel-tile shapes.
- f16_2x_t256: the production tile; more pixel tiles than SMs, so the persistent loops wrap; odd UNet2 bottom extents (117, 115, 113);
  the largest SE extent (234 x 234).
- f16_1x_t60:  the smallest 1x tile.
- f16_1x_t168: 1x whose UNet2 bottom extents are odd (35, 33, 31), and a partial batch (2 of 3 slots).
- tf32_2x_t38, tf32_2x_t130 (more tiles than SMs), tf32_2x_t98 (partial batch, 2 of 3), tf32_1x_t104 (odd UNet2 bottom extents 19, 17, 15; also
  the permutation and render engine).
- wide_f16_2x_t66, wide_tf32_1x_t60: the model with wide SE gates (fp16 subnormal folded weights).
"""
import os

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import onnx_io, tiling
from oracle.models import make_model

pytestmark = pytest.mark.gpu

# name -> (model, precision, scale, tile, batch, images given to infer)
ENGINES = {
    "f16_2x_t38": ("base", "fp16", 2, 38, 3, 3),
    "f16_2x_t66": ("base", "fp16", 2, 66, 4, 3),
    "f16_2x_t130": ("base", "fp16", 2, 130, 2, 2),
    "f16_2x_t256": ("base", "fp16", 2, 256, 2, 2),
    "f16_1x_t60": ("base", "fp16", 1, 60, 3, 3),
    "f16_1x_t168": ("base", "fp16", 1, 168, 3, 2),
    "tf32_2x_t38": ("base", "tf32", 2, 38, 2, 2),
    "tf32_2x_t98": ("base", "tf32", 2, 98, 3, 2),
    "tf32_2x_t130": ("base", "tf32", 2, 130, 2, 2),
    "tf32_1x_t104": ("base", "tf32", 1, 104, 2, 2),
    "wide_f16_2x_t66": ("wide", "fp16", 2, 66, 3, 3),
    "wide_tf32_1x_t60": ("wide", "tf32", 1, 60, 3, 3),
}

SE = {4: "unet1.conv2.se", 12: "unet2.conv2.se", 15: "unet2.conv3.se", 18: "unet2.conv4.se"}
FOLD = {5: 4, 13: 12, 16: 15, 19: 18}        # consumer -> the SE layer whose gate is folded into its weights
DOWN, UP2 = (2, 10, 13), (5, 16, 19)
WIDE_SE_FACTOR = 8.0                           # SE fc2 weights x 8: gates from below 1e-3 to above 0.999
MIN_SLOT_SPREAD = 0.05                          # some channel of every SE block differs by this much between two slots

# The kernel variants the planner picks for CUNet across the audited engines (layer_kernel, reduced to the fields that select code).
# A planner change that adds or removes a path fails test_kernel_variants_are_pinned; update this list on purpose.
PINNED_VARIANTS = [
    "first-layer fp32",                                             # tf32: layers 0, 8
    "fused into the next layer",                                    # fp16: layers 0, 8
    "head kernel, taps in N",                                       # fp16 2x: layers 7, 21; 1x: 21
    "igemm bn=128 kc=64 epilogue=tma-skip nbuf=3",                  # fp16: 5, 16, 19 (convT 2x2 + skip)
    "igemm bn=128 kc=64 epilogue=two-group nbuf=2",                 # fp16: 13, 15
    "igemm bn=64 kc=64 epilogue=two-group nbuf=2",                  # fp16: 2, 10
    "igemm-tf32 bn=128",
    "igemm-tf32 bn=16",
    "igemm-tf32 bn=256",
    "igemm-tf32 bn=64",
    "patch3x3 bn=16 kc=64 epilogue=direct nbuf=1",                  # fp16 1x: layer 7
    "patch3x3 bn=64 kc=64 epilogue=two-group nbuf=2",               # fp16: 3, 4, 6, 11, 12, 14, 17, 18, 20
    "patch3x3+rgb-first-layer bn=64 kc=32 epilogue=two-group nbuf=2",  # fp16: 1, 9
]


# ---- rounding as the engine stores values -------------------------------------------------------------------------------------
def _tf32(a):
    u = np.ascontiguousarray(a, np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0xFFF + ((u >> 13) & 1)) & 0xFFFFE000).astype(np.uint32).view(np.float32)


def _f16(a):
    return np.asarray(a, np.float32).astype(np.float16)


def _t(a):
    """engine NHWC -> float64 NCHW"""
    return torch.from_numpy(np.asarray(a, np.float64)).permute(0, 3, 1, 2)


def _np(t):
    return t.permute(0, 2, 3, 1).numpy()


def _crop(t, c):
    return t[:, :, c:-c, c:-c]


# ---- models and engines ---------------------------------------------------------------------------------------------------------
def _widen(model):
    with torch.no_grad():
        for name in SE.values():
            dict(model.named_modules())[name].conv2.weight.mul_(WIDE_SE_FACTOR)
    return model


@pytest.fixture(scope="session")
def audit_models(tmp_path_factory):
    """The seed-1234 cunet/art models and their wide-gate variant, in directories of their own (engine files are written beside them)."""
    import w2x
    root = str(tmp_path_factory.mktemp("audit_models"))
    out = {}
    for key in ("base", "wide"):
        for scale in (1, 2):
            m = make_model("cunet", scale, 1234)
            if key == "wide":
                _widen(m)
            path = w2x.model_path(os.path.join(root, key), "cunet/art", 0, scale)
            os.makedirs(os.path.dirname(path), exist_ok=True)
            onnx_io.export_cunet(m, path)
            out[(key, scale)] = (m, path)
    return out


def _load(path, precision, scale, tile, batch):
    import w2x
    prec = w2x.PRECISION_TF32 if precision == "tf32" else w2x.PRECISION_FP16
    e = w2x.Img2Img()
    msgs = []
    e.setMessageCallback(lambda s, m: msgs.append(m))
    assert e.build(path, w2x.BuildConfig.fixed(batch, tile, precision=prec)), msgs
    assert e.load(path, w2x.RenderConfig(precision=prec, batchSize=batch, height=tile, width=tile, scaling=scale)), msgs
    return e


def _inputs(n, tile, seed=0):
    """n strongly different tiles, NCHW f32 on the u8 grid: a synthetic_frame crop, black, white, noise, horizontal and vertical ramps"""
    rng = np.random.default_rng(seed)
    r = np.linspace(0, 1, tile, dtype=np.float32)
    fr = tiling.synthetic_frame(3 * tile, 2 * tile, seed)[..., ::-1].transpose(2, 0, 1).astype(np.float32) / 255
    xs = [fr[:, :tile, :tile], np.zeros((3, tile, tile)), np.ones((3, tile, tile)), rng.random((3, tile, tile)),
          np.broadcast_to(r[None, None, :], (3, tile, tile)), np.broadcast_to(r[None, :, None], (3, tile, tile)), fr[:, tile:, tile:2 * tile]]
    return np.stack([np.rint(np.asarray(x, np.float64) * 255) / 255 for x in xs[:n]]).astype(np.float32)


def _dump(e):
    """every tensor w2x_layer_tensor exposes, as the last batch left it"""
    d = {"kernel": [], "out": [], "sums": [], "gate": [], "wimg": []}
    for i in range(22):
        d["kernel"].append(e.layer_kernel(i))
        for key, which in (("out", 0), ("sums", 2), ("gate", 3), ("wimg", 4)):
            d[key].append(e.layer_tensor(i, which))
    d["x"] = e.layer_tensor(0, 1)
    return d


class Audit:
    def __init__(self, name, spec, model, x, y, dump):
        self.name = name
        self.key, self.precision, self.scale, self.tile, self.batch, self.n = spec
        self.model, self.x, self.y, self.d = model, x, y, dump
        self.tf32 = self.precision == "tf32"
        mods = [(nm, m) for nm, m in model.named_modules() if isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)) and ".se." not in nm]
        assert len(mods) == 22
        rnd = _tf32 if self.tf32 else _f16
        self.w32 = [rnd(m.weight.detach().numpy()) for _, m in mods]           # the stored weights (fp16 or TF32 values)
        self.W = [torch.from_numpy(w.astype(np.float64)) for w in self.w32]
        self.b = [torch.from_numpy(m.bias.detach().numpy().astype(np.float64)) for _, m in mods]
        self.se = {i: dict(model.named_modules())[nm] for i, nm in SE.items()}

    def out(self, i):
        return self.d["out"][i][:self.n]

    def gate(self, i):
        return self.d["gate"][i][:self.n]


@pytest.fixture(scope="session")
def audits(audit_models, built_lib):
    """name -> Audit, built on first use: one engine, one infer on _inputs, every layer tensor dumped, engine closed."""
    cache = {}

    def get(name):
        if name not in cache:
            spec = ENGINES[name]
            key, precision, scale, tile, batch, n = spec
            model, path = audit_models[(key, scale)]
            e = _load(path, precision, scale, tile, batch)
            x = _inputs(n, tile)
            y = e.infer(x)
            assert y is not None, e.last_error
            cache[name] = Audit(name, spec, model, x, y, _dump(e))
            e.close()
        return cache[name]
    return get


# ---- float64 references ---------------------------------------------------------------------------------------------------------
def _op(a, i, x, w, b):
    if i in DOWN:
        return F.conv2d(x, w, b, stride=2)
    if i in UP2:
        return F.conv_transpose2d(x, w, b, stride=2)
    if i == 7 and a.scale == 2:
        return F.conv_transpose2d(x, w, b, stride=2, padding=3)
    return F.conv2d(x, w, b)


def _ones_like_one_output(i, w):
    """a one-output-channel kernel of ones: _op with it sums |input| over everything that feeds one output element"""
    return torch.ones_like(w[:, :1]) if isinstance(w, torch.Tensor) and (i in UP2 or i == 7) else torch.ones_like(w[:1])


def _layer_inputs(a, i, gate=None):
    """-> (input, skip or None) of layer i in float64 NCHW, from the engine's own tensors; gate: the SE gates to apply (default the engine's)"""
    g = (lambda j: torch.from_numpy(np.asarray(gate[j] if gate and j in gate else a.gate(j), np.float64))[:, :, None, None])
    if i == 0:
        x = _t(a.d["x"][:a.n, :, :, :3])
    elif i == 8:
        x = _t(a.out(7)[..., :3])
    elif i in FOLD:
        x = _t(a.out(FOLD[i])) * g(FOLD[i])
    else:
        x = _t(a.out(i - 1))
    skip = None
    if i == 5:
        skip = _crop(_t(a.out(1)), 4)
    elif i == 16:
        skip = _crop(_t(a.out(12)) * g(12), 4)
    elif i == 19:
        skip = _crop(_t(a.out(9)), 16)
    elif i == 21:
        skip = _crop(_t(a.out(7)[..., :3]), 20)
    return x, skip


def _act(i, t):
    if i == 21:
        return torch.clamp(t, 0, 1)
    return t if i == 7 else F.leaky_relu(t, 0.1)


def layer_ratio(a, i, gate=None):
    """max over the layer's elements of |engine - float64| / bound (<= 1 passes); the output of layer i from the engine's inputs"""
    W, b = a.W[i], a.b[i]
    fusedFirst = not a.tf32 and i in (1, 9)
    if i == 21:
        got = torch.from_numpy(a.y.astype(np.float64))
    else:
        got = _t(a.out(i))
        if i == 7:
            assert (a.out(7)[..., 3] == 0).all(), "padding channel of the NHWC4 head is not zero"
            got = got[:, :3]
    if fusedFirst:
        # layers 0 / 8 run inside 1 / 9: the 32-channel tensor between them is computed from the model input and rounded to fp16 in the kernel
        assert a.d["out"][i - 1] is None
        x0 = _t(a.d["x"][:a.n, :, :, :3]) if i == 1 else _t(a.out(7)[..., :3])
        a0 = F.leaky_relu(F.conv2d(x0, a.W[i - 1], a.b[i - 1]), 0.1)
        m0 = F.conv2d(x0.abs(), a.W[i - 1].abs(), a.b[i - 1].abs())
        x, skip = a0, None
        d0 = 2.0 ** -11 * a0.abs() + 2.0 ** -15 * m0 + 2.0 ** -25      # the fp16 intermediate's error
    else:
        x, skip = _layer_inputs(a, i, gate)
    pre = _op(a, i, x, W, b)
    mag = _op(a, i, x.abs(), W.abs(), b.abs())
    if skip is not None:
        pre = _act(i, pre) + skip if i != 21 else pre + skip
        mag = mag + skip.abs()
        ref = pre if i != 21 else torch.clamp(pre, 0, 1)
    else:
        ref = _act(i, pre)
    if a.tf32 and i in (0, 8):          # fp32 FMA on the CUDA cores
        tol = 2.0 ** -15 * mag + 2.0 ** -22 * ref.abs()
    elif a.tf32:                        # the tensor core drops the low 13 bits of the fp32 activations: 2^-10 relative per term
        tol = (2.0 ** -10 + 2.0 ** -15) * mag + 2.0 ** -22 * ref.abs()
        if i in FOLD:                   # the folded weights are rounded to TF32
            tol = tol + 2.0 ** -10 * mag
    else:                               # fp16 output rounding + fp32 accumulation
        tol = 2.0 ** -11 * ref.abs() + 2.0 ** -15 * mag + 2.0 ** -24
        if i in FOLD:                   # the folded weights are rounded to fp16 (subnormals included)
            tol = tol + 2.0 ** -11 * mag + 2.0 ** -25 * _op(a, i, x.abs(), _ones_like_one_output(i, W), None)
        if fusedFirst:
            tol = tol + F.conv2d(d0, W.abs())
    tol = tol + 1e-30
    assert got.shape == ref.shape, (got.shape, ref.shape)
    r = ((got - ref).abs() / tol).amax()
    return float(r)


def sum_ratio(a, i, sums=None):
    """SE channel sums against the engine's own output: exact in a tf32 engine, within the fp16 rounding otherwise.  -> max |err| / bound"""
    out = a.out(i).astype(np.float64)
    s = (a.d["sums"][i] if sums is None else sums)[:a.n]
    hw = out.shape[1] * out.shape[2]
    if a.tf32:
        want = np.rint(out * 1024).astype(np.int64).sum(axis=(1, 2))
        return float(np.abs(s - want).max()) * 1e30      # any difference fails
    err = np.abs(s / 1024.0 - out.sum(axis=(1, 2)))
    tol = np.abs(out).sum(axis=(1, 2)) * 2.0 ** -11 + hw * (2.0 ** -11 + 2.0 ** -25)
    return float((err / tol).max())


def _se_ref(a, i, mean):
    """float64 excite of SE block i from per-image channel means -> (gate, its fp32 evaluation bound)"""
    se = a.se[i]
    W1 = se.conv1.weight.detach().double().flatten(1).numpy()
    b1 = se.conv1.bias.detach().double().numpy()
    W2 = se.conv2.weight.detach().double().flatten(1).numpy()
    b2 = se.conv2.bias.detach().double().numpy()
    c, r = W1.shape[1], W1.shape[0]
    u = 2.0 ** -24
    h = np.maximum(mean @ W1.T + b1, 0)
    A1 = np.abs(mean) @ np.abs(W1).T + np.abs(b1)
    eh = (c + 4) * u * A1                                        # the mean's three roundings and fp32 FMA over c terms
    s = h @ W2.T + b2
    es = (r + 2) * u * (h @ np.abs(W2).T + np.abs(b2)) + eh @ np.abs(W2).T
    g = 1 / (1 + np.exp(-s))
    dg = g * (1 - g)
    tol = 2 * (dg * (es + 2.0 ** -21) + 2.0 ** -22 * g) + 2.0 ** -30   # expf, the add and the division; a factor 2 of slack
    return g, tol, (np.abs(W1), np.abs(W2))


def gate_ratio(a, i, end_to_end=False):
    """SE gate of layer i: from the engine's sums (isolates the excite kernel) or from the float64 mean of its output (the whole block)"""
    out = a.out(i).astype(np.float64)
    hw = out.shape[1] * out.shape[2]
    got = a.gate(i).astype(np.float64)
    if not end_to_end:
        g, tol, _ = _se_ref(a, i, a.d["sums"][i][:a.n] / 1024.0 / hw)
    else:
        g, tol, (aW1, aW2) = _se_ref(a, i, out.mean(axis=(1, 2)))
        dmean = (2.0 ** -11 + 2.0 ** -25) if a.tf32 else (np.abs(out).sum(axis=(1, 2)) * 2.0 ** -11 + hw * (2.0 ** -11 + 2.0 ** -25)) / hw
        dmean = np.broadcast_to(dmean, g.shape)
        tol = tol + 1.01 * 0.25 * ((dmean @ aW1.T) @ aW2.T)       # ReLU 1-Lipschitz, sigmoid' <= 1/4
    return float((np.abs(got - g) / tol).max())


def float64_gates(a, i):
    out = a.out(i).astype(np.float64)
    return _se_ref(a, i, out.mean(axis=(1, 2)))[0]


def _packed(a, i):
    """the stored GEMM operand B [npad][ktot] of a folded layer, restated from the torch weights (fp16 or TF32 values as float32)"""
    w = a.w32[i].astype(np.float32)
    if i in UP2:                                                 # row = (dy*2+dx)*cout + co, k = ci
        cin, cout = w.shape[:2]
        return np.ascontiguousarray(w.transpose(2, 3, 1, 0).reshape(4 * cout, cin))
    cout, cin = w.shape[:2]                                      # down 2x2: k = (dy*2+dx)*cin + ci
    return np.ascontiguousarray(w.transpose(0, 2, 3, 1).reshape(cout, 4 * cin))


def fold_mismatches(a, i, wimg=None):
    """per-image folded weights of layer i against RN(float32(W) * float32(gate[img][k % cin])), bit for bit -> number of differing elements"""
    wp = _packed(a, i)
    cin = a.w32[i].shape[0] if i in UP2 else a.w32[i].shape[1]
    k = np.arange(wp.shape[1]) % cin
    g = a.gate(FOLD[i]).astype(np.float32)[:, None, k]
    prod = wp[None] * g
    got = (a.d["wimg"][i] if wimg is None else wimg)[:a.n]
    assert got.shape == prod.shape, (got.shape, prod.shape)
    if a.tf32:
        want = _tf32(prod)
        return int((got.view(np.uint32) != want.view(np.uint32)).sum())
    want = prod.astype(np.float16)
    return int((got.view(np.uint16) != want.view(np.uint16)).sum())


# ---- the audit ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(ENGINES))
def test_every_layer_matches_float64(name, audits):
    a = audits(name)
    assert a.d["x"].shape == (a.batch, a.tile, a.tile, 4) and (a.d["x"][:a.n, :, :, 3] == 0).all()
    bad = {}
    for i in range(22):
        if a.d["out"][i] is None:
            assert i == 21 or (not a.tf32 and i in (0, 8)), (i, a.d["kernel"][i])
        if not a.tf32 and i in (0, 8):
            continue
        r = layer_ratio(a, i)
        if not r <= 1:
            bad[i] = (r, a.d["kernel"][i])
    assert not bad, bad


@pytest.mark.parametrize("name", list(ENGINES))
def test_squeeze_excite_sums_gates_and_folded_weights(name, audits):
    a = audits(name)
    bad = {}
    for i in SE:
        assert a.d["sums"][i] is not None and a.d["gate"][i] is not None
        for what, r in (("sums", sum_ratio(a, i)), ("gate", gate_ratio(a, i)), ("gate end to end", gate_ratio(a, i, end_to_end=True))):
            if not r <= 1:
                bad[(i, what)] = r
        spread = np.ptp(float64_gates(a, i), axis=0).max()
        assert spread >= MIN_SLOT_SPREAD, (i, spread)         # the inputs tell the slots apart
    for i in FOLD:
        mism = fold_mismatches(a, i)
        if mism:
            bad[(i, "folded weights")] = mism
    for i in range(22):                                        # exactly the SE layers / folded consumers have these tensors
        assert (a.d["sums"][i] is not None) == (i in SE) and (a.d["gate"][i] is not None) == (i in SE)
        assert (a.d["wimg"][i] is not None) == (i in FOLD), i
    assert not bad, bad


def test_wide_gates_reach_both_ends(audits):
    """the wide-gate model really has gates below 1e-3 and above 0.999, and fp16 engines see subnormal folded weights"""
    for name in ("wide_f16_2x_t66", "wide_tf32_1x_t60"):
        a = audits(name)
        g = np.concatenate([float64_gates(a, i).ravel() for i in SE])
        assert g.min() < 1e-3 and g.max() > 0.999, (g.min(), g.max())
    a = audits("wide_f16_2x_t66")
    w = np.concatenate([np.abs(a.d["wimg"][i][:a.n].astype(np.float32)).ravel() for i in FOLD])
    assert ((w > 0) & (w < 2.0 ** -14)).any()


def _variant(desc):
    """the fields of a layer_kernel description that select code: kernel, N tile, epilogue"""
    head = desc.split(" bn=")[0]
    if "bn=" not in desc:
        return desc.split(" (")[0]
    f = dict(kv.split("=") for kv in desc.split()[1:] if "=" in kv)
    if head == "igemm-tf32":
        return f"igemm-tf32 bn={f['bn']}"
    grouped = f["tma"] == "1" and f["skip"] == "0" and f["nbuf"] == "2" and int(f["bn"]) <= 128
    epi = "two-group" if grouped else "tma-skip" if f["skip"] == "1" else "tma" if f["tma"] == "1" else "staged" if f["staged"] == "1" else "direct"
    return f"{head} bn={f['bn']} kc={f['kc']} epilogue={epi} nbuf={f['nbuf']}"


def test_kernel_variants_are_pinned(audits):
    seen = {}
    for name in ENGINES:
        for i, k in enumerate(audits(name).d["kernel"]):
            seen.setdefault(_variant(k), set()).add(i)
    if sorted(seen) != sorted(PINNED_VARIANTS):
        pytest.fail("kernel variants (layers) differ from PINNED_VARIANTS:\n" + "\n".join(f"{v!r}: {sorted(seen[v])}" for v in sorted(seen)))


@pytest.mark.parametrize("name", ["f16_2x_t66", "tf32_1x_t104"])
def test_permuted_batch_gives_permuted_result(name, audit_models, built_lib):
    """tiles are independent and the SE sums exact integers: a permuted batch is the permuted result, bit for bit"""
    key, precision, scale, tile, batch, _ = ENGINES[name]
    e = _load(audit_models[(key, scale)][1], precision, scale, tile, batch)
    x = _inputs(batch, tile, seed=3)
    perm = np.roll(np.arange(batch), 1)
    y = e.infer(x)
    yp = e.infer(x[perm])
    assert y is not None and yp is not None, e.last_error
    assert np.array_equal(yp.view(np.uint32), y[perm].view(np.uint32))
    e.close()


@pytest.mark.parametrize("name", ["f16_2x_t66", "tf32_1x_t104"])
def test_render_last_batch_equals_infer(name, audit_models, built_lib):
    """render's last, partial batch (fused first layer on the frame-wide unpack buffer, the padding slots skipped) leaves every layer
    tensor of its slots byte-identical to infer of the same tiles on a fresh engine"""
    key, precision, scale, tile, batch, _ = ENGINES[name]
    path = audit_models[(key, scale)][1]
    e = _load(path, precision, scale, tile, batch)
    ot = e.output_tile_size
    for w in range(90, 400):
        g = tiling.calculate_tiles(w, 70, w * scale, 70 * scale, tile, tile, ot, ot, scale, 1 / 16, 1 / 16)
        if g.count % batch and g.count > batch:
            break
    src = tiling.synthetic_frame(w, 70, 11)
    assert e.render(src) is not None, e.last_error
    got = _dump(e)
    e.close()
    first = (g.count - 1) // batch * batch
    n = g.count - first
    rgb = src[..., ::-1]
    tiles = []
    for q in range(first, g.count):            # row-major processing order
        j, i = divmod(q, g.nx)
        tiles.append(tiling.normalize_u8(tiling.pad_roi(rgb, g.in_rects[i * g.ny + j])).transpose(2, 0, 1))
    f = _load(path, precision, scale, tile, batch)
    assert f.infer(np.stack(tiles)) is not None, f.last_error
    want = _dump(f)
    f.close()
    assert got["kernel"] == want["kernel"]
    for key_ in ("out", "sums", "gate", "wimg"):
        for i in range(22):
            a, b = got[key_][i], want[key_][i]
            assert (a is None) == (b is None), (key_, i)
            if a is not None:
                assert a[:n].tobytes() == b[:n].tobytes(), (key_, i, n)


def test_layer_tensor_refusals(audit_models, built_lib, tmp_path):
    import __graft_entry__
    e = _load(audit_models[("base", 2)][1], "fp16", 2, 38, 1)
    for index, which, msg in ((22, 0, "out of range"), (-1, 3, "out of range"), (3, 5, "unknown tensor")):
        with pytest.raises(RuntimeError, match=msg):
            e.layer_tensor(index, which)
    assert e.layer_tensor(3, 2) is None and e.layer_tensor(4, 4) is None    # no SE on layer 3, no folded weights on layer 4
    e.close()
    _, path = __graft_entry__.make_synthetic_model(str(tmp_path), 2, 0, model="swin_unet/art")
    s = _load(path, "fp16", 2, 64, 1)
    with pytest.raises(RuntimeError, match="not a CUNet engine"):
        s.layer_tensor(0, 0)
    s.close()


# ---- power checks: each bar rejects the fault it exists for --------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["f16_2x_t66", "tf32_2x_t98"])
def test_consumer_check_rejects_swapped_gates(name, audits):
    a = audits(name)
    for i in FOLD:
        g = a.gate(FOLD[i])
        swapped = {FOLD[i]: g[[1, 0] + list(range(2, len(g)))]}
        assert layer_ratio(a, i) <= 1
        assert layer_ratio(a, i, gate=swapped) > 1, i


@pytest.mark.parametrize("name", ["f16_2x_t256", "tf32_2x_t130"])
def test_sum_check_rejects_a_dropped_row(name, audits):
    """one output row missing from the squeeze, at the largest SE extent audited"""
    a = audits(name)
    i = max(SE, key=lambda j: a.out(j).shape[1] * a.out(j).shape[2])
    row = np.rint(a.out(i)[:, -1].astype(np.float64) * 1024).astype(np.int64).sum(axis=1)
    sums = a.d["sums"][i].copy()
    sums[:a.n] -= row
    assert sum_ratio(a, i) <= 1
    assert sum_ratio(a, i, sums) > 1, (i, a.out(i).shape)


@pytest.mark.parametrize("name", ["f16_2x_t66", "tf32_2x_t98"])
def test_fold_check_rejects_one_ulp(name, audits):
    a = audits(name)
    for i in FOLD:
        w = a.d["wimg"][i].copy()
        bits = w.view(np.uint32 if a.tf32 else np.uint16).reshape(-1)
        bits[bits.size // (2 * a.batch) + 7] += 0x2000 if a.tf32 else 1      # slot 0, one element, 1 ulp of the stored format
        assert fold_mismatches(a, i) == 0
        assert fold_mismatches(a, i, w) == 1, i
