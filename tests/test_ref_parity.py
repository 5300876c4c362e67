"""The NumPy oracle and the product's host logic against THE REFERENCE'S OWN CODE.

oracle/_ref/libw2xref.so = /root/reference/src/tensorrt/*.cpp compiled unmodified against CPU mocks of OpenCV-CUDA /
TensorRT / CUDA / nlohmann-json (oracle/Makefile, oracle/ref_shim/).  `live` tests call it directly and are skipped where it
is not built (no /root/reference); `golden` tests use the vectors tests/golden/make_ref_goldens.py generated from it.
Everything here is integer / byte / exactly-specified IEEE f32 work: comparisons are bit-exact."""
import ctypes as C
import json
import os
import shutil

import numpy as np
import pytest
from hypothesis import assume, given, settings, strategies as st

import refcases
from oracle import ref, tiling

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = np.load(os.path.join(HERE, "golden", "ref_goldens.npz"))
GRIDS = json.load(open(os.path.join(HERE, "golden", "tile_grid.json")))
HASHES = json.load(open(os.path.join(HERE, "golden", "ref_hashes.json")))
live = pytest.mark.skipif(not ref.available(), reason="oracle/_ref is not built: needs the upstream waifu2x-tensorrt sources "
                          "(make -C oracle REF=<checkout>); the golden tests cover the cases stored under tests/golden")


# ---------------------------------------------------------------------------------------------------------------------
# calculateTiles (img2img_render.cpp:7-66)
# ---------------------------------------------------------------------------------------------------------------------
@live
@pytest.mark.parametrize("name", sorted(refcases.GRID_CASES))
def test_live_grid_equals_committed_golden(name):
    W, H, T, OT, S, B = refcases.GRID_CASES[name]
    n, ins, outs = ref.calculate_tiles(W, H, W * S, H * S, T, T, OT, OT, S, B, B)
    g = GRIDS[name]
    assert n == g["count"] and [list(r) for r in ins] == g["in_rects"] and [list(r) for r in outs] == g["out_rects"]


@live
@settings(max_examples=300, deadline=None)
@given(W=st.integers(1, 5000), H=st.integers(1, 3000), T=st.sampled_from([64, 112, 128, 256, 400, 640]), S=st.sampled_from([1, 2, 4]),
       B=st.sampled_from([0.0, 1 / 32, 1 / 16, 1 / 8, 1 / 4]), fam=st.sampled_from(["cunet", "swin"]))
def test_oracle_and_product_grid_equal_reference_on_random_frames(W, H, T, S, B, fam, built_lib):
    import w2x
    OT = (T - 16) * S if fam == "swin" else (2 * T - 72 if S == 2 else T - 56)
    assume(fam == "swin" or S in (1, 2))
    assume(OT > 0)
    # an overlap that swallows the whole effective tile divides by <= 0 in the reference (:32-33: inf / negative counts); the
    # product rejects it ("overlap too large"), see test_degenerate_overlap_is_rejected
    assume(tiling.lround(OT / (T * S) * T) - tiling.lround(T * B) > 0)
    n, ins, outs = ref.calculate_tiles(W, H, W * S, H * S, T, T, OT, OT, S, B, B)
    g = tiling.calculate_tiles(W, H, W * S, H * S, T, T, OT, OT, S, B, B)
    if g.nx < 1 or g.ny < 1:
        # frame smaller than the input overlap: the reference's tiling.x / tiling.y go non-positive and its loops do not run
        # a negative tileCount makes the reference's vector::reserve throw (render() then fails): reported as INT_MIN by the driver
        assert ins == [] and (n == g.nx * g.ny or (n == -(1 << 31) and g.nx * g.ny < 0))
        n2, _, ir2, _ = w2x.calculate_tiles(W, H, W * S, H * S, T, T, OT, OT, S, B, B)
        assert n2 == 0 and ir2 == []  # the product reports an empty grid (the reference's tileCount may be garbage here)
        return
    assert n == g.count and ins == g.in_rects and outs == g.out_rects
    n2, grid, ir2, or2 = w2x.calculate_tiles(W, H, W * S, H * S, T, T, OT, OT, S, B, B)
    assert n2 == n and ir2 == ins and or2 == outs


def test_degenerate_overlap_is_rejected(built_lib):
    import w2x
    with pytest.raises(ValueError):
        w2x.calculate_tiles(36, 36, 36, 36, 64, 64, 8, 8, 1, 0.25, 0.25)   # cunet 1x tile 64: effective tile 8 < overlap 16
    with pytest.raises(ValueError):
        w2x.calculate_tiles(36, 36, 36, 36, 64, 64, 8, 8, 1, 0.125, 0.125)  # effective tile 8 == overlap 8: division by zero


# ---------------------------------------------------------------------------------------------------------------------
# createTileWeights (img2img_load.cpp:29-52) and applyWeights (img2img_render.cpp:107-121)
# ---------------------------------------------------------------------------------------------------------------------
def _check_weights(ox, oy, size, top, right, bottom, left, built_lib):
    import w2x
    wo = tiling.create_tile_weights(ox, oy, size, size)
    assert np.array_equal(wo[0][:, 0], top) and np.array_equal(wo[1][0, :], right)
    assert np.array_equal(wo[2][:, 0], bottom) and np.array_equal(wo[3][0, :], left)
    # the product keeps two ramps: ramp[i] = weights[3] column i (left) / weights[0] row i (top), i < overlap
    rx, ry = w2x.blend_ramp(ox), w2x.blend_ramp(oy)
    assert np.array_equal(np.asarray(rx, np.float32), left[:ox]) and np.array_equal(np.asarray(ry, np.float32), top[:oy])
    assert (left[ox:] == 1).all() and (top[oy:] == 1).all()
    assert np.array_equal(right, left[::-1]) and np.array_equal(bottom, top[::-1])


@pytest.mark.parametrize("ox,oy,size", refcases.WEIGHT_CASES)
def test_weights_golden(ox, oy, size, built_lib):
    k = f"weights_{ox}_{oy}_{size}"
    _check_weights(ox, oy, size, GOLD[k + "_top_col0"], GOLD[k + "_right_row0"], GOLD[k + "_bottom_col0"], GOLD[k + "_left_row0"], built_lib)


@live
@pytest.mark.parametrize("ox,oy,size", refcases.WEIGHT_CASES + [(1, 1, 8), (5, 2, 24)])
def test_weights_live(ox, oy, size, built_lib):
    w = ref.create_tile_weights(ox, oy, size, size)
    wo = tiling.create_tile_weights(ox, oy, size, size)
    for i in range(4):
        for c in range(3):
            assert np.array_equal(w[i][..., c], wo[i])
    _check_weights(ox, oy, size, w[0, :, 0, 0], w[1, 0, :, 0], w[2, :, 0, 0], w[3, 0, :, 0], built_lib)


@live
def test_apply_weights_live():
    rng = np.random.default_rng(3)
    size, ov = 24, 5
    weights = tiling.create_tile_weights(ov, ov, size, size)
    cw, ch = 60, 50
    for rect in [(0, 0, 24, 24), (19, 0, 24, 24), (38, 0, 22, 24), (0, 19, 24, 24), (19, 19, 24, 24), (38, 38, 22, 12), (0, 38, 24, 12), (36, 26, 24, 24)]:
        t = rng.uniform(-0.2, 1.2, size=(size, size, 3)).astype(np.float32)
        assert np.array_equal(ref.apply_weights(t, ov, ov, rect, cw, ch), tiling.apply_weights(t, rect, cw, ch, weights)), rect


# ---------------------------------------------------------------------------------------------------------------------
# padRoi, applyAugmentation / reverseAugmentation, blobFromImages
# ---------------------------------------------------------------------------------------------------------------------
@live
def test_pad_roi_live():
    img = refcases.frame(37, 29, 7)
    for rect in [(0, 0, 16, 16), (-5, -3, 16, 16), (30, 20, 16, 16), (-18, -18, 64, 64), (10, -2, 8, 40), (-4, 5, 50, 8), (21, 13, 16, 16)]:
        assert np.array_equal(ref.pad_roi(img, rect), tiling.pad_roi(img, rect)), rect


@live
@pytest.mark.parametrize("k", range(8))
def test_augmentations_live(k):
    n = 12
    t8 = refcases.frame(n, n, 8 + k)
    assert np.array_equal(ref.apply_augmentation(t8, k), tiling.augment(t8, k))
    tf = np.random.default_rng(k).uniform(0, 1, size=(n, n, 3)).astype(np.float32)
    inv = ref.reverse_augmentation(tf, k, aliased=False)
    assert np.array_equal(inv, tiling.reverse_augment(tf, k))
    # round trip through the reference's own pair: reverse(apply(x)) == x
    fwd = ref.apply_augmentation(t8, k).astype(np.float32)
    assert np.array_equal(ref.reverse_augmentation(fwd, k), t8.astype(np.float32))
    # closed forms the CUDA kernels implement
    a = tiling.augment(t8, k)
    for r, c in [(0, 0), (3, 7), (11, 2)]:
        rr, cc = tiling.augment_src_index(k, r, c, n)
        assert (a[r, c] == t8[rr, cc]).all()
        rr, cc = tiling.reverse_src_index(k, r, c, n)
        assert (inv[r, c] == tf[rr, cc]).all()


@live
def test_blob_from_images_live():
    tiles = np.stack([refcases.frame(16, 16, 30 + i) for i in range(3)])
    ref.set_pitch_align(1)
    try:
        blob = ref.blob_from_images(tiles)
    finally:
        ref.set_pitch_align(512)
    want = np.stack([tiling.normalize_u8(t).transpose(2, 0, 1) for t in tiles])
    assert np.array_equal(blob, want)


@live
def test_blob_pitch_bug_q4_is_reproduced_by_the_mock():
    """README 'batch sizes > 1 produce wrong tiles' (SURVEY q4): with cudaMallocPitch-like rows the blob of a batch whose
    3*T*T is not pitch-aligned is read back shifted.  Shows the mock keeps the allocation semantics that matter."""
    tiles = np.stack([refcases.frame(20, 20, 40 + i) for i in range(2)])  # 3*20*20 = 1200 B per image, not a 512 multiple
    want = np.stack([tiling.normalize_u8(t).transpose(2, 0, 1) for t in tiles])
    blob = ref.blob_from_images(tiles)
    assert np.array_equal(blob[0], want[0]) and not np.array_equal(blob[1], want[1])


@pytest.mark.parametrize("name", sorted(refcases.UNPACK_CASES))
def test_unpack_golden_equals_oracle(name):
    W, H, T, OT, S, B, seed = refcases.UNPACK_CASES[name]
    src = refcases.frame(W, H, seed)
    rgb = src[..., ::-1]
    g = tiling.calculate_tiles(W, H, W * S, H * S, T, T, OT, OT, S, B, B)
    gold = GOLD["unpack_" + name]
    assert gold.shape[0] == g.count
    for i, r in enumerate(g.in_rects):
        want = tiling.normalize_u8(tiling.augment(tiling.pad_roi(rgb, r), i % 8)).transpose(2, 0, 1).astype(np.float16)
        assert np.array_equal(gold[i].view(np.uint16), np.ascontiguousarray(want).view(np.uint16)), i


# ---------------------------------------------------------------------------------------------------------------------
# Img2Img::build + load + render with an analytic network
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_render(name):
    W, H, T, OT, S, B, batch, tta, seed = refcases.RENDER_CASES[name]
    src = refcases.frame(W, H, seed)
    model = refcases.posdep_model(S, T, OT)
    return src, model, dict(tile=T, out_tile=OT, scaling=S, overlap=B, batch=batch, tta=tta)


@pytest.mark.parametrize("name", sorted(refcases.RENDER_CASES))
def test_render_golden_equals_oracle(name):
    src, model, kw = _oracle_render(name)
    got = tiling.render(src, model, tta_mode="reference_q1", **kw)
    assert np.array_equal(got, GOLD["render_" + name])
    if kw["tta"]:
        # the product implements the mean (documented deviation, SURVEY q1); with a non-equivariant network it differs
        assert not np.array_equal(tiling.render(src, model, tta_mode="mean", **kw), got)


@live
@pytest.mark.parametrize("name", sorted(refcases.RENDER_CASES))
def test_render_live_equals_golden(name):
    src, model, kw = _oracle_render(name)
    assert np.array_equal(ref.render(src, model, **kw), GOLD["render_" + name])


@live
def test_render_live_batch_size_does_not_change_the_result():
    src, model, kw = _oracle_render("cunet2x_t64_b2")
    a = ref.render(src, model, **{**kw, "batch": 1})
    for b in (2, 3, 5):
        assert np.array_equal(ref.render(src, model, **{**kw, "batch": b}), a), b


@pytest.mark.parametrize("name", sorted(refcases.STITCH_CASES))
def test_stitch_golden_equals_oracle(name):
    W, H, T, OT, S, B, seed = refcases.STITCH_CASES[name]
    g = tiling.calculate_tiles(W, H, W * S, H * S, T, T, OT, OT, S, B, B)
    tiles = refcases.stitch_tiles(g.count, OT, seed)
    got = tiling.render(np.zeros((H, W, 3), np.uint8), refcases.replay_model(tiles, OT), T, OT, S, B, batch=1)
    assert np.array_equal(got, GOLD["stitch_" + name])


# ---------------------------------------------------------------------------------------------------------------------
# getConfigHash / serializeConfig (img2img_build.cpp:8-50), isCompatible / isOptimized / getEnginePath (img2img_load.cpp:9-27,79-114)
# ---------------------------------------------------------------------------------------------------------------------
def _w2x_build_cfg(ints):
    import w2x
    c = w2x.BuildConfig()
    for k, v in zip(("deviceId", "precision", "minBatchSize", "optBatchSize", "maxBatchSize", "minChannels", "optChannels", "maxChannels",
                     "minWidth", "optWidth", "maxWidth", "minHeight", "optHeight", "maxHeight"), ints):
        setattr(c, k, v)
    return c


@pytest.mark.parametrize("i", range(len(HASHES)))
def test_config_hash_and_sidecar_equal_reference(i, built_lib, tmp_path):
    import w2x
    h = HASHES[i]
    assert w2x.config_hash(h["device"], _w2x_build_cfg(h["cfg"])) == h["sha256"]
    if ref.available():
        ref.set_device_name(h["device"])
        try:
            assert ref.config_hash(ref.CBuild(*h["cfg"])) == h["sha256"]
        finally:
            ref.set_device_name("NVIDIA B200")
    # the sidecar the product writes for this config parses to the same key order and values
    want = json.loads(h["sidecar"])
    assert list(want) == ["deviceName", "precision", "minBatchSize", "optBatchSize", "maxBatchSize", "minChannels", "optChannels", "maxChannels",
                          "minWidth", "optWidth", "maxWidth", "minHeight", "optHeight", "maxHeight"]
    assert want["deviceName"] == h["device"] and want["precision"] == ("FP16" if h["cfg"][1] == 1 else "TF32")


@live
def test_engine_selection_equals_reference(built_lib, tmp_path):
    """getEnginePath over a directory of sidecars: reference (.trt) and product (.w2x) pick the same stem in every scenario."""
    import w2x
    dev = "NVIDIA B200"
    ref.set_device_name(dev)
    model = tmp_path / "noise3_scale2x.onnx"
    model.write_bytes(b"x")
    profiles = {
        "fixed8_256": (0, 1, 8, 8, 8, 3, 3, 3, 256, 256, 256, 256, 256, 256),
        "range": (0, 1, 1, 1, 4, 3, 3, 3, 64, 256, 640, 64, 256, 640),
        "tf32": (0, 0, 1, 1, 4, 3, 3, 3, 64, 256, 640, 64, 256, 640),
        "fixed4_400": (0, 1, 4, 4, 4, 3, 3, 3, 400, 400, 400, 400, 400, 400),
    }
    stems = {}
    for name, ints in profiles.items():
        cfg = ref.CBuild(*ints)
        stem = "noise3_scale2x_" + ref.config_hash(cfg)[:16]
        stems[name] = stem
        ref.serialize_config(str(tmp_path / (stem + ".json")), cfg)
        (tmp_path / (stem + ".trt")).write_bytes(b"W2XSHIMENGINE 2 72\n")
        (tmp_path / (stem + ".w2x")).write_bytes(b"placeholder")
    scenarios = [
        dict(batch=8, tile=256, precision=1),   # optimized profile wins
        dict(batch=2, tile=128, precision=1),   # only the range profile is compatible
        dict(batch=1, tile=256, precision=1),   # range profile, optimized
        dict(batch=4, tile=400, precision=1),   # fixed4_400 optimized; range compatible
        dict(batch=1, tile=256, precision=0),   # tf32 profile
        dict(batch=16, tile=256, precision=1),  # nothing fits
        dict(batch=1, tile=1024, precision=1),  # nothing fits
    ]
    for sc in scenarios:
        r = ref.render_config(batch=sc["batch"], tile=sc["tile"], scaling=2, precision=sc["precision"])
        ok_ref, path_ref = ref.get_engine_path(str(model), r)
        rc = w2x.RenderConfig(batchSize=sc["batch"], height=sc["tile"], width=sc["tile"], scaling=2, precision=sc["precision"])
        try:
            ok_w2x, path_w2x = True, w2x.select_engine(str(model), rc, dev)
        except RuntimeError as ex:
            ok_w2x, path_w2x = False, str(ex)
        assert ok_ref == ok_w2x, (sc, path_ref, path_w2x)
        if ok_ref:
            stem_ref, stem_w2x = os.path.basename(path_ref)[:-4], os.path.basename(path_w2x)[:-4]
            opt_ref = [n for n, ints in profiles.items() if ref.is_optimized(r, ref.CBuild(*ints)) and ref.is_compatible(r, ref.CBuild(*ints))]
            if opt_ref:
                # an optimized profile exists: both must pick it (directory order cannot matter)
                assert stem_ref == stem_w2x == stems[opt_ref[0]], sc
            else:
                # no optimized profile: the reference takes the first compatible file in directory order, the product in name
                # order (documented deviation) -- both must be compatible ones
                compat = {stems[n] for n, ints in profiles.items() if ref.is_compatible(r, ref.CBuild(*ints))}
                assert stem_ref in compat and stem_w2x in compat, sc
        else:
            assert path_ref == "could not satisfy render configuration" and "could not satisfy render configuration" in path_w2x
