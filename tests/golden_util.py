"""Load a golden fixture (tests/golden/*.npz, made by make_golden.py from the
reference module) and regenerate its seeded inputs."""
import contextlib
import glob
import os

import numpy as np
import torch

from onepose_b200 import synthetic

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FORWARD_CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz"))
                       if not os.path.basename(p).startswith(("empty", "mean_", "features3d", "dustbin", "pnp_", "superpoint")))
RELEASED_CASES = [c for c in FORWARD_CASES if not c.startswith(("noself", "lintrans", "additional"))]
# make_golden.py records the fixtures on this many torch CPU threads.  How torch's fp32 convolutions split their sums depends on
# the thread count: on 32 or 128 threads the SuperPoint scores move by ~1e-6 (up to 20 ulp), so a CPU recomputation that is
# held to a fixture at fp32 rounding runs on the same count.
GOLDEN_THREADS = 8


@contextlib.contextmanager
def golden_threads():
    """Run the enclosed CPU computation on the thread count the fixtures were recorded with."""
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(n)


def load_case(name):
    g = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))
    hp = dict(synthetic.DEFAULT_HPARAMS)
    for k, v in zip(g["meta_hp_keys"], g["meta_hp_vals"]):
        hp[str(k)] = bool(v)
    sd = synthetic.make_state_dict(int(g["meta_wseed"]), damped=bool(g["meta_damped"]), hparams=hp)
    data = synthetic.make_batch(int(g["meta_obj"]), [int(f) for f in g["meta_frames"]],
                                int(g["meta_N"]), int(g["meta_M"]), int(g["meta_L"]))
    return g, hp, sd, data


def conf_reference_view(g, conf):
    """(reference conf values, same-shaped view of ``conf``) -- full or the stored sample."""
    if "conf_matrix" in g:
        return g["conf_matrix"], conf
    return g["conf_sample"], conf[:, ::7, ::5]


def load_dustbin_case():
    """Forward on an object built by the reference's pad_features3d_random / build_features3d_leaves (all-ones dustbin leaves,
    duplicate all-ones padded 3D points): inputs are stored in the fixture (they come from the reference functions)."""
    g = dict(np.load(os.path.join(GOLDEN_DIR, "dustbin_n64_m96.npz"), allow_pickle=False))
    hp = dict(synthetic.DEFAULT_HPARAMS)
    sd = synthetic.make_state_dict(0, damped=True, hparams=hp)
    N, M = g["query"].shape[1], g["desc3d"].shape[1]
    data = {"keypoints2d": np.zeros((1, N, 2), np.float32), "keypoints3d": np.zeros((1, M, 3), np.float32),
            "descriptors2d_query": g["query"][None], "descriptors3d_db": g["desc3d"][None], "descriptors2d_db": g["desc2d"][None]}
    return g, hp, sd, data


SUPERPOINT_CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "superpoint_*.npz")))


def load_superpoint_case(name):
    """(fixture, state dict, config, images [B,1,H,W]) of a SuperPoint golden (inputs regenerated from the recorded seeds)."""
    g = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))
    sd = synthetic.make_superpoint_state_dict(int(g["meta_wseed"]), float(g["meta_gain"]))
    conf = {}
    for k, v in zip(g["meta_conf_keys"], g["meta_conf_vals"]):
        k = str(k)
        conf[k] = float(v) if "threshold" in k else int(v)
    img = np.stack([synthetic.make_image(int(i), int(g["meta_H"]), int(g["meta_W"])) for i in g["meta_images"]], 0)
    return g, sd, conf, img
