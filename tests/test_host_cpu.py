"""CPU-side checks: the C-ABI library loads and exports every declared symbol, the module is
state-dict compatible with the reference, host logic that needs no GPU."""
import json
import os
import re

import numpy as np
import pytest
import torch

from onepose_b200 import GATsSuperGlue, LitModelGATsSPG, _lib, synthetic
from tests.golden_util import GOLDEN_DIR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "onepose_b200.h")).read()
    declared = set(re.findall(r"\b(opb_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name)


def test_header_is_plain_c(tmp_path):
    """The drop-in boundary is a C ABI: the header must compile as C99 with no C++/torch types (cgo / ctypes / JNI bind it)."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "hdr.c"
    src.write_text('#include "onepose_b200.h"\nint main(void) { opb_config c; (void)c; return 0; }\n')
    inc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-I", inc, str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_config_struct_matches_header():
    header = open(os.path.join(ROOT, "include", "onepose_b200.h")).read()
    body = re.search(r"typedef struct opb_config \{(.*?)\} opb_config;", header, re.S).group(1)
    fields = re.findall(r"(?:int32_t|float)\s+(\w+);", body)
    assert fields == [f[0] for f in _lib.OpbConfig._fields_]


def test_no_gpu_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import ctypes as C
    lib = _lib.load()
    cfg = _lib.OpbConfig(256, 4, 0.07, 0.2, 1, 0, 0, 0)
    h = C.c_void_p()
    rc = lib.opb_create(C.byref(cfg), C.byref(h))
    assert rc == -2 and b"no CPU path" in lib.opb_last_error(None)


def test_state_dict_keys_and_shapes_match_reference():
    spec = json.load(open(os.path.join(GOLDEN_DIR, "state_dict_spec.json")))
    m = GATsSuperGlue(dict(synthetic.DEFAULT_HPARAMS))
    sd = m.state_dict()
    assert list(sd.keys()) == list(spec.keys())
    for k, shape in spec.items():
        assert list(sd[k].shape) == shape, k
    # the seeded synthetic state dict (reference key names) loads strictly
    syn = synthetic.make_state_dict(0)
    m.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in syn.items()}, strict=True)


def test_empty_input_returns_reference_style_dict():
    g = np.load(os.path.join(GOLDEN_DIR, "empty_n0_m96.npz"))
    m = GATsSuperGlue(dict(synthetic.DEFAULT_HPARAMS))
    data = {k: torch.from_numpy(v) for k, v in synthetic.make_batch(1, [11], 0, 96, 8).items()}
    out = m(data)
    assert isinstance(out, dict) and sorted(out.keys()) == list(g["keys"])
    assert out["matches0"].dtype == torch.int32 and tuple(out["matches1"].shape) == g["matches1"].shape
    assert (out["matches1"].numpy() == g["matches1"]).all() and out["skip_train"] is True


def test_cpu_tensors_are_rejected():
    m = GATsSuperGlue(dict(synthetic.DEFAULT_HPARAMS))
    data = {k: torch.from_numpy(v) for k, v in synthetic.make_batch(1, [11], 16, 32, 8).items()}
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(data)


def test_unsupported_match_type():
    hp = dict(synthetic.DEFAULT_HPARAMS, match_type="sinkhorn")
    m = GATsSuperGlue(hp)
    data = {k: torch.from_numpy(v) for k, v in synthetic.make_batch(1, [11], 16, 32, 8).items()}
    with pytest.raises(NotImplementedError):
        m(data)


def test_lightning_checkpoint_standin(tmp_path):
    hp = dict(synthetic.DEFAULT_HPARAMS, lr=1e-3)
    syn = synthetic.make_state_dict(3)
    ckpt = {"state_dict": {"matcher." + k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in syn.items()},
            "hyper_parameters": hp}
    ckpt["state_dict"]["extractor.conv1a.weight"] = torch.zeros(1)
    path = tmp_path / "GATsSPG.ckpt"
    torch.save(ckpt, path)
    model = LitModelGATsSPG.load_from_checkpoint(str(path)).eval().freeze()
    assert torch.equal(model.matcher.final_proj.weight, torch.from_numpy(syn["final_proj.weight"]))
    assert not any(p.requires_grad for p in model.parameters())


def test_forward_signature_and_module_surface_match_reference():
    """Same constructor argument, same forward(data) entry, same attribute names the reference callers touch."""
    import inspect
    sig = inspect.signature(GATsSuperGlue.__init__)
    assert list(sig.parameters) == ["self", "hparams"]                      # GATs_SuperGlue.py:145
    assert list(inspect.signature(GATsSuperGlue.forward).parameters) == ["self", "data"]   # :179
    m = GATsSuperGlue(dict(synthetic.DEFAULT_HPARAMS))
    assert m.match_type == "softmax" and hasattr(m, "gnn") and hasattr(m, "final_proj") and hasattr(m, "bin_score")


def test_features3d_module_mirrors_reference_names():
    from onepose_b200 import features3d
    import inspect
    assert list(inspect.signature(features3d.pad_features3d_random).parameters)[:3] == ["descriptors", "scores", "n_target_shape"]
    assert list(inspect.signature(features3d.build_features3d_leaves).parameters)[:5] == [
        "descriptors", "scores", "idxs", "n_target_shape", "num_leaf"]                # data_utils.py:143, :163
    assert list(inspect.signature(features3d.mean_descriptors).parameters)[:2] == ["descriptors", "idxs"]   # feature_process.py:297
    assert list(inspect.signature(features3d.mean_scores).parameters)[:2] == ["scores", "idxs"]
    with pytest.raises(RuntimeError, match="no CPU path"):
        features3d.pad_features3d_random(np.ones((4, 3), np.float32), np.ones((3, 1), np.float32), 5, device="cpu")


def test_caller_supplied_result_buffers_are_viewed_not_copied():
    """match_frames(out=...): results land in views of the caller's flat buffers (a serving loop allocates once)."""
    from onepose_b200.matcher import _out_view
    dev = torch.device("cpu")
    pool = {"matches0": torch.zeros(100, dtype=torch.int64), "conf_matrix": torch.zeros(1000)}
    v = _out_view(pool, "matches0", (3, 20), torch.int64, dev)
    assert tuple(v.shape) == (3, 20) and v.data_ptr() == pool["matches0"].data_ptr() and v.is_contiguous()
    c = _out_view(pool, "conf_matrix", (2, 10, 30), torch.float32, dev)
    assert tuple(c.shape) == (2, 10, 30) and c.data_ptr() == pool["conf_matrix"].data_ptr()
    fresh = _out_view(pool, "matches1", (2, 5), torch.int64, dev)             # not in the pool: allocated
    assert tuple(fresh.shape) == (2, 5)
    assert tuple(_out_view(None, "matches0", (4, 4), torch.int64, dev).shape) == (4, 4)
    with pytest.raises(ValueError):
        _out_view(pool, "conf_matrix", (2, 10, 60), torch.float32, dev)         # too small
    with pytest.raises(ValueError):
        _out_view(pool, "matches0", (3, 20), torch.float32, dev)                # wrong dtype


def test_plain_c_client_links_and_runs(tmp_path):
    """The boundary is a C ABI: a C99 program (tests/c_abi/client.c) compiles against the header alone, links the in-tree library and
    gets status codes + messages, no exceptions (here, without a GPU: OPB_E_CUDA from both constructors)."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    _lib.load()
    libdir = os.path.join(ROOT, "onepose_b200")
    exe = tmp_path / "client"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c_abi", "client.c"),
                        "-L", libdir, "-l:libonepose_b200.so", f"-Wl,-rpath,{libdir}", "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "opb_create ->" in r.stdout and "opb_sp_create ->" in r.stdout


def test_calls_without_a_handle_report_their_own_error():
    """opb_last_error(NULL) is the message of this thread's last failed call without a handle: after a failed opb_create, each
    handle-less entry point that rejects its arguments (before any CUDA work) leaves a message naming itself."""
    import ctypes as C
    lib = _lib.load()
    buf = C.create_string_buffer(1024)
    p = C.cast(buf, C.c_void_p)
    calls = {
        "opb_gather_features3d": lambda: lib.opb_gather_features3d(p, p, 0, 1, p, 1, p, p, 1, None),
        "opb_segmented_mean_f64": lambda: lib.opb_segmented_mean_f64(p, p, 0, 256, p, None),
        "opb_segmented_mean_scores_f64": lambda: lib.opb_segmented_mean_scores_f64(p, p, 0, p, None),
        "opb_ransac_pnp": lambda: lib.opb_ransac_pnp(p, p, p, p, 0, 128, 8.0, 0, p, p, p, p, None),
        "opb_debug_gemm": lambda: lib.opb_debug_gemm(p, p, p, p, p, 1, 256, 64, 0, None),
        "opb_forward": lambda: lib.opb_forward(None, p, None, 1, 1, p, p, p, p, p, None),
    }
    for name, call in calls.items():
        bad = _lib.OpbConfig(128, 4, 0.07, 0.2, 1, 0, 0, 0)          # rejected before any CUDA call
        h = C.c_void_p()
        assert lib.opb_create(C.byref(bad), C.byref(h)) == -1
        assert b"descriptor_dim" in lib.opb_last_error(None)
        assert call() == -1, name
        msg = lib.opb_last_error(None)
        assert name.encode() in msg and b"descriptor_dim" not in msg, (name, msg)
        assert lib.opb_sp_last_error(None) == msg                    # one slot for both handle types
