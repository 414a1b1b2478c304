"""SuperPoint extractor, CPU side: the oracle pinned to outputs of the unmodified reference module
(tests/golden/superpoint_*.npz), the device algorithms' design checked in numpy against the oracle
(tests/sp_emulation.py mirrors the index arithmetic of csrc/superpoint.cu), and the host logic of the module."""
import inspect
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import superpoint_oracle as O
from onepose_b200 import SuperPoint, _lib, synthetic
from tests import sp_emulation as E
from tests.golden_util import GOLDEN_DIR, SUPERPOINT_CASES, golden_threads, load_superpoint_case


@pytest.mark.parametrize("name", SUPERPOINT_CASES)
def test_oracle_matches_reference_module(name):
    g, sd, conf, img = load_superpoint_case(name)
    p = O.params_from_numpy(sd)
    every = int(g["meta_every"])
    for ac, tag in ((False, "ac0"), (True, "ac1")):
        with golden_threads():
            out = O.forward(p, img, conf, align_corners=ac)
        for b in range(img.shape[0]):
            np.testing.assert_array_equal(out["keypoints"][b].numpy(), g[f"keypoints_{b}"])         # bit-exact key points
            np.testing.assert_allclose(out["scores"][b].numpy(), g[f"scores_{b}"], atol=1e-7)
            np.testing.assert_allclose(out["descriptors"][b].numpy()[:, ::every], g[f"descriptors_{tag}_{b}"], atol=2e-6)


def test_released_config_keeps_the_default_threshold():
    """extract_features.py:19-24 spells the key 'keypoints_threshold'; the module reads 'keypoint_threshold' (superpoint.py:164)."""
    m = SuperPoint(synthetic.SUPERPOINT_CONF)
    assert m.config["keypoint_threshold"] == 0.005 and m.config["keypoints_threshold"] == 0.6
    assert m.config["nms_radius"] == 3 and m.config["max_keypoints"] == 4096 and m.config["remove_borders"] == 4


def test_module_surface_matches_reference():
    spec = json.load(open(os.path.join(GOLDEN_DIR, "superpoint_state_dict_spec.json")))
    m = SuperPoint({})
    sd = m.state_dict()
    assert list(sd.keys()) == list(spec.keys())
    for k, shape in spec.items():
        assert list(sd[k].shape) == shape, k
    syn = synthetic.make_superpoint_state_dict(0)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in syn.items()}, strict=True)
    assert list(inspect.signature(SuperPoint.forward).parameters) == ["self", "inp"]           # superpoint.py:140
    assert SuperPoint.default_config == O.DEFAULT_CONFIG
    for bad in (0, -2):
        with pytest.raises(ValueError, match="max_keypoints"):
            SuperPoint({"max_keypoints": bad})                                                  # superpoint.py:133-135
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(torch.zeros(1, 1, 64, 64))


def test_sp_config_struct_matches_header():
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "onepose_b200.h")).read()
    body = re.search(r"typedef struct opb_sp_config \{(.*?)\} opb_sp_config;", header, re.S).group(1)
    assert re.findall(r"(?:int32_t|float)\s+(\w+);", body) == [f[0] for f in _lib.OpbSpConfig._fields_]


def test_no_gpu_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import ctypes as C
    lib = _lib.load()
    cfg = _lib.OpbSpConfig(256, 3, 0.005, 4096, 4, 1, 0)
    h = C.c_void_p()
    assert lib.opb_sp_create(C.byref(cfg), C.byref(h)) == -2
    cfg = _lib.OpbSpConfig(256, 3, 0.005, 0, 4, 1, 0)
    assert lib.opb_sp_create(C.byref(cfg), C.byref(h)) == -1 and b"max_keypoints" in lib.opb_sp_last_error(None)


# ---------------------------------------------------------------------------------------------
# design of the device path, in numpy, against the oracle
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def small():
    sd = synthetic.make_superpoint_state_dict(0, 4.0)
    H, W = 64, 80
    img = np.stack([synthetic.make_image(i, H, W) for i in (1, 2)], 0)
    return sd, O.params_from_numpy(sd), torch.from_numpy(img), H, W


def test_pixel_grid_convolution_is_nine_shifted_gemms(small):
    sd, p, x, H, W = small
    B = x.shape[0]
    h, w, P = E.stage(H, W, 0)
    rows = E.to_grid(O.encoder(p, x, upto=0).numpy())
    out = E.conv_grid(rows, E.pack_conv(sd["conv1b.weight"]), sd["conv1b.bias"], h, w, P, 64)
    assert np.abs(E.from_grid(out, B, 64, h, w) - O.encoder(p, x, upto=1).numpy()).max() < 1e-5
    q = np.arange(out.shape[0]) % P
    yy, xx = q // (w + 2), q % (w + 2)
    border = (yy < 1) | (yy > h) | (xx < 1) | (xx > w)
    assert not out[border].any()                                  # the output is again a zero-bordered grid
    pooled = E.pool_grid(out, B, 64, h, w)
    assert np.abs(E.from_grid(pooled, B, 64, h // 2, w // 2) - O.encoder(p, x, upto=2).numpy()).max() < 1e-5
    # fused heads: [convPa | convDa] side by side, then the 1x1 layers on column windows
    feat = O.encoder(p, x)
    h3, w3, P3 = E.stage(H, W, 3)
    wpd = np.concatenate([E.pack_conv(sd["convPa.weight"]), E.pack_conv(sd["convDa.weight"])], 0)
    bpd = np.concatenate([sd["convPa.bias"], sd["convDa.bias"]])
    head = E.conv_grid(E.to_grid(feat.numpy()), wpd, bpd, h3, w3, P3, 128)
    logits = head[:, :256] @ E.pack_conv(sd["convPb.weight"]).T + sd["convPb.bias"]
    ref = O._conv(p, "convPb", O._conv(p, "convPa", feat), relu=False).numpy()
    assert np.abs(E.from_grid(logits.astype(np.float32), B, 65, h3, w3) - ref).max() < 2e-4


@pytest.mark.parametrize("r", [0, 1, 3, 4, 6])
def test_tiled_nms_equals_simple_nms(small, r):
    sd, p, x, H, W = small
    sc = O.dense_scores(p, O.encoder(p, x))
    ref = O.simple_nms(sc, r).numpy()
    for b in range(x.shape[0]):
        np.testing.assert_array_equal(E.nms_tiled(sc[b].numpy(), r), ref[b])
    flat = torch.full((1, 40, 48), 0.25)                          # plateau: every pixel ties, all survive in the reference
    np.testing.assert_array_equal(E.nms_tiled(flat[0].numpy(), r), O.simple_nms(flat, r)[0].numpy())


@pytest.mark.parametrize("k", [4096, 50, -1])
def test_ordered_selection_and_rank_topk(small, k):
    sd, p, x, H, W = small
    nms = O.simple_nms(O.dense_scores(p, O.encoder(p, x)), 3)
    cfg = {**O.DEFAULT_CONFIG, "nms_radius": 3, "max_keypoints": k}
    kk, ss = O.select_keypoints(nms[0], cfg)
    ek, es = E.select(nms[0].numpy(), cfg["keypoint_threshold"], cfg["remove_borders"], k)
    np.testing.assert_array_equal(kk.numpy(), ek)
    np.testing.assert_array_equal(ss.numpy(), es)


@pytest.mark.parametrize("ac", [True, False])
def test_descriptor_sampling(small, ac):
    sd, p, x, H, W = small
    feat = O.encoder(p, x)
    nms = O.simple_nms(O.dense_scores(p, feat), 3)
    kk, _ = O.select_keypoints(nms[0], {**O.DEFAULT_CONFIG, "max_keypoints": 60})
    raw = O._conv(p, "convDb", O._conv(p, "convDa", feat), relu=False)
    h3, w3, P3 = E.stage(H, W, 3)
    ref = O.sample_descriptors(kk, F.normalize(raw[0], p=2, dim=0), 8, ac).numpy()
    em = E.sample(E.to_grid(raw.numpy())[:P3], h3, w3, P3, kk.numpy(), ac)
    assert np.abs(em - ref).max() < 1e-6
