"""Drop-in boundary (SURVEY.md §8b): a trainer of the reference, imported with ``dropin/`` ahead of it on sys.path
(scnerf_b200.launch), must bind every hot-path name to this repository.  CPU only.

The same checks run on two trees.  The stand-in tree is written by the test: the reference's directory layout and
import statements (NeRF/run_nerf.py:50-62, nerfplusplus/ddp_train_nerf.py:17-26), the samplers the NeRF++ trainer
defines itself, stubs of the out-of-scope modules (matching, data loading), and hot-path modules that raise when
imported, so a name that is not shadowed by a shim fails the test.  The reference's own unmodified trainers are
checked when ``SCNERF_REFERENCE`` names a checkout of the original SCNeRF project."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("SCNERF_REFERENCE")
needs_ref = pytest.mark.skipif(not (REF and os.path.isfile(os.path.join(REF, "NeRF", "run_nerf.py"))),
                               reason="SCNERF_REFERENCE does not name a checkout of the original SCNeRF project")

_SHADOWED = 'raise ImportError("stand-in hot-path module: a drop-in shim must answer this import")\n'
STANDIN = {
    "NeRF/run_nerf.py": '''
import os
import sys
import numpy as np
import torch
sys.path.insert(0, "..")
from render import *
from get_rays import *
from create_nerf import *
from run_nerf_helpers import *
from model.camera_model import *
from model.ray_dist_loss import proj_ray_dist_loss_single, preprocess_match
from model.reprojection import *


def train():
    fix_seeds(0)
    kw = create_nerf, render, render_path, img2mse, mse2psnr, get_rays_np, reprojection_error
    rays = (get_rays_full_image_no_camera, get_rays_full_image_use_camera, get_rays_kps_no_camera,
            get_rays_kps_use_camera)
    cams = PinholeModelRotNoiseLearning10kRayoRayd, PinholeModelRotNoiseLearning10kRayoRaydDistortion
    return kw, rays, cams, proj_ray_dist_loss_single, preprocess_match, np, torch, os
''',
    "NeRF/render.py": _SHADOWED,
    "NeRF/get_rays.py": _SHADOWED,
    "NeRF/create_nerf.py": _SHADOWED,
    "NeRF/run_nerf_helpers.py": _SHADOWED,
    "model/camera_model.py": _SHADOWED,
    "model/camera_dict.py": _SHADOWED,
    "model/ray_dist_loss.py": _SHADOWED,
    "model/reprojection.py": "def reprojection_error(*a):\n    return None\n",
    "nerfplusplus/ddp_train_nerf.py": '''
import os
import sys
import numpy as np
import torch
sys.path.insert(0, "..")
from nerf_sample_ray_split import RaySamplerSingleImage, render_ray_from_camera
from data_loader_split import load_data_split
from create_nerf import create_nerf
from model.ray_dist_loss import proj_ray_dist_loss_single, preprocess_match


def intersect_sphere(ray_o, ray_d):
    raise RuntimeError("stand-in sampler: must be rebound")


def perturb_samples(z_vals):
    raise RuntimeError("stand-in sampler: must be rebound")


def sample_pdf(bins, weights, N_samples, det=False):
    raise RuntimeError("stand-in sampler: must be rebound")


def render_single_image(rank, world_size, models, ray_sampler, chunk_size):
    raise RuntimeError("stand-in renderer: must be rebound")


def setup_logger():
    pass


def train():
    return (create_nerf, RaySamplerSingleImage, render_ray_from_camera, load_data_split, proj_ray_dist_loss_single,
            preprocess_match, intersect_sphere, perturb_samples, sample_pdf, render_single_image, np, torch, os)
''',
    "nerfplusplus/nerf_sample_ray_split.py": '''
def render_ray_from_camera(*a, **k):
    raise RuntimeError("stand-in ray generator: must be rebound")


class RaySamplerSingleImage:
    def random_sample(self, N_rand):
        return render_ray_from_camera(N_rand)
''',
    "nerfplusplus/data_loader_split.py": "def load_data_split(*a, **k):\n    return None\n",
    "nerfplusplus/create_nerf.py": _SHADOWED,
    "nerfplusplus/ddp_model.py": _SHADOWED,
    "nerfplusplus/nerf_network.py": _SHADOWED,
}


def _standin_tree(tmp_path):
    for rel, src in STANDIN.items():
        f = tmp_path / rel
        f.parent.mkdir(parents=True, exist_ok=True)
        f.write_text(src.lstrip("\n"))
    return str(tmp_path)


def _report(kind, ref):
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1", CUDA_VISIBLE_DEVICES="")
    env.pop("PYTHONPATH", None)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_check.py"), kind, ref],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("REPORT")][-1]
    return json.loads(line[len("REPORT"):])


def _check_run_nerf(ref):
    """NeRF/run_nerf.py:1-70: render / get_rays / create_nerf / run_nerf_helpers / model.camera_model /
    model.ray_dist_loss."""
    r = _report("nerf", ref)
    assert r["trainer"] == os.path.join(ref, "NeRF", "run_nerf.py")           # the tree's own trainer file ran
    for name, owner in r["names"].items():
        assert owner is not None and owner.startswith("scnerf_b200."), (name, owner)
    for m in ("render", "get_rays", "create_nerf", "run_nerf_helpers", "camera_model", "model.camera_model",
              "model.ray_dist_loss"):
        assert r["modules"][m]["impl"] == "scnerf_b200." + m.split(".")[-1], (m, r["modules"][m])
    # out-of-scope modules still come from the trainer's tree (matching, evaluation)
    assert r["modules"]["model.reprojection"]["file"].startswith(ref)
    # every name the trainer takes from its star imports exists behind the shim
    missing = [n for n, (ok, _) in r["star_names"].items() if not ok]
    assert not missing, missing


def _check_ddp_train_nerf(ref):
    """nerfplusplus/ddp_train_nerf.py:17,25-26 imports + the samplers it defines itself (:50-132,135-256)."""
    r = _report("nerfpp", ref)
    assert r["trainer"] == os.path.join(ref, "nerfplusplus", "ddp_train_nerf.py")
    want = {"create_nerf": "scnerf_b200.nerfplusplus.create_nerf",
            "render_ray_from_camera": "scnerf_b200.nerfplusplus.nerf_sample_ray_split",
            "intersect_sphere": "scnerf_b200.nerfplusplus.ddp_train_nerf",
            "perturb_samples": "scnerf_b200.nerfplusplus.ddp_train_nerf",
            "sample_pdf": "scnerf_b200.nerfplusplus.ddp_train_nerf",
            "render_single_image": "scnerf_b200.nerfplusplus.ddp_train_nerf",
            "proj_ray_dist_loss_single": "scnerf_b200.ray_dist_loss"}
    for name, owner in want.items():
        assert r["names"][name] == owner, (name, r["names"][name])
    # the dataset sampler (kept from the trainer's tree) reaches the CUDA ray generator through its own globals
    assert r["names"]["RaySamplerSingleImage.random_sample -> render_ray_from_camera"].startswith("scnerf_b200.")
    assert r["modules"]["nerf_sample_ray_split"]["wraps"] == os.path.join(ref, "nerfplusplus", "nerf_sample_ray_split.py")
    assert r["modules"]["data_loader_split"]["file"].startswith(ref)
    assert not [n for n, (ok, _) in r["star_names"].items() if not ok]


@needs_ref
def test_unmodified_run_nerf_binds_to_this_repo():
    _check_run_nerf(REF)


@needs_ref
def test_unmodified_ddp_train_nerf_binds_to_this_repo():
    _check_ddp_train_nerf(REF)


def test_standin_run_nerf_binds_to_this_repo(tmp_path):
    _check_run_nerf(_standin_tree(tmp_path))


def test_standin_ddp_train_nerf_binds_to_this_repo(tmp_path):
    _check_ddp_train_nerf(_standin_tree(tmp_path))


def test_patch_trainer_rebinds_a_namespace():
    """create_nerf() patches the calling trainer's globals in spawned processes (create_nerf.py:_patch_calling_trainer)."""
    sys.path.insert(0, ROOT)
    from scnerf_b200.nerfplusplus.create_nerf import patch_trainer
    ns = {"intersect_sphere": len, "perturb_samples": len, "sample_pdf": len, "unrelated": 1}
    done = patch_trainer(ns)
    assert sorted(done) == ["intersect_sphere", "perturb_samples", "sample_pdf"]
    assert ns["sample_pdf"].__module__ == "scnerf_b200.nerfplusplus.ddp_train_nerf" and ns["unrelated"] == 1
    assert patch_trainer(ns) == []          # idempotent
