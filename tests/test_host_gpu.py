"""Host runtime of the two handle types on the GPU (run with -m gpu): launch counts and profile entries, status codes of the weight
look-up, and handles that live on a device other than the current one."""
import numpy as np
import pytest
import torch

from onepose_b200 import GATsSuperGlue, SuperPoint, _lib, synthetic

pytestmark = pytest.mark.gpu

# the profile prefixes bench.py reads
BENCH_PREFIXES = ("gemm epi1 ", "gemm epi5 ", "gemm epi6 ", "gemm epi7 ", "gats_aggregate", "kv_state_h", "score_sums_finalize",
                  "mutual_match")
# one launch each, in launch order, of SuperPoint.forward_padded
SP_LAUNCHES = ["sp_conv1a", "conv1b", "sp_pool2x2", "conv2a", "conv2b", "sp_pool2x2", "conv3a", "conv3b", "sp_pool2x2", "conv4a", "conv4b",
               "convPa|convDa", "convPb", "convDb", "sp_scores", "sp_nms", "sp_count", "sp_compact", "sp_emit", "sp_sample"]
SP_CONF = {"nms_radius": 3, "max_keypoints": 128}


def _matcher(device="cuda:0"):
    m = GATsSuperGlue(dict(synthetic.DEFAULT_HPARAMS)).eval()
    m.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in synthetic.make_state_dict(0).items()})
    return m.to(device)


def _extractor(device="cuda:0"):
    sp = SuperPoint(SP_CONF).eval()
    sp.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in synthetic.make_superpoint_state_dict(0, 4.0).items()})
    return sp.to(device)


def test_matcher_launch_counts_and_profile():
    """One frame: 85 launches (48 GEMMs) on the first call after set_object, which runs the object prologue, and 75 (43 GEMMs) on
    a later call, through the device and the host entry alike; every prefix bench.py reads has launches."""
    data = synthetic.make_batch(1, [3], 200, 500, 8)
    m = _matcher()
    d3, d2 = (torch.from_numpy(data[k][0]).cuda() for k in ("descriptors3d_db", "descriptors2d_db"))
    q = torch.from_numpy(data["descriptors2d_query"])
    m.set_object(d3, d2)
    m.set_profiling(True)
    for call in (lambda: m.match_frames(q.cuda()), lambda: m.match_frames_host(q.pin_memory())):
        m.set_object(d3, d2)
        for launches, gemms in ((85, 48), (75, 43)):
            call()
            assert m.launch_count() == launches
            assert m.get_profile()["gemm_launches"] == gemms
            for prefix in BENCH_PREFIXES:
                assert m.get_profile_entry(prefix)["launches"] > 0, prefix
    m.set_profiling(False)


def test_extractor_launches_and_profile_names():
    sp = _extractor()
    img = torch.from_numpy(synthetic.make_image(1, 96, 128)[None]).cuda()
    sp.forward_padded(img)
    sp.set_profiling(True)
    sp.forward_padded(img)
    assert sp.launch_count() == len(SP_LAUNCHES)
    prof = sp.get_profile()
    assert [name for name, _, _ in prof] == SP_LAUNCHES
    assert all(fl > 0 for name, _, fl in prof if name.startswith("conv"))
    sp.set_profiling(False)


def test_wrong_size_weight_is_invalid():
    lib = _lib.load()
    short = np.zeros(10, np.float32)
    m = _matcher()
    m.set_object(torch.zeros(256, 4, device="cuda"), torch.zeros(256, 32, device="cuda"))    # creates the handle, loads weights
    assert lib.opb_load_weight(m._handle, b"final_proj.bias", short.ctypes.data, short.size) == 0
    assert lib.opb_finalize_weights(m._handle) == -1
    assert b"final_proj.bias" in lib.opb_last_error(m._handle)
    sp = _extractor()
    sp.forward_padded(torch.zeros(1, 1, 64, 64, device="cuda"))
    assert lib.opb_sp_load_weight(sp._handle, b"convDb.bias", short.ctypes.data, short.size) == 0
    assert lib.opb_sp_finalize_weights(sp._handle) == -1
    assert b"convDb.bias" in lib.opb_sp_last_error(sp._handle)


def test_handles_on_a_device_other_than_the_current_one():
    """Modules on cuda:1 called while cuda:0 is current: every handle entry point makes its own device current, and kernel
    attributes are set on each device.  Same results, bit for bit, as on cuda:0."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    data = synthetic.make_batch(2, [1, 2], 200, 500, 8)
    img = synthetic.make_image(2, 96, 128)[None]

    def run(dev):
        m, sp = _matcher(dev), _extractor(dev)
        outs = []
        for _ in range(2):
            m({k: torch.from_numpy(v).to(dev) for k, v in data.items()})
            outs.append({k: v.cpu() for k, v in m.last_batched.items()})
            outs.append({k: v.cpu() for k, v in sp.forward_padded(torch.from_numpy(img).to(dev)).items()})
        torch.cuda.synchronize(dev)
        return outs

    ref = run("cuda:0")
    with torch.cuda.device(0):
        other = run("cuda:1")
    for a, b in zip(ref, other):
        for k in a:
            assert torch.equal(a[k], b[k]), k
