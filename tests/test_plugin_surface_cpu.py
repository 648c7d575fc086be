"""The nerfstudio plugin surface (SURVEY §8b): `dn_config.method_specifications()` must hand nerfstudio exactly what the
reference's dn_config.py does — same trainer arguments, optimizer groups and model overrides for the three methods —
with this package's pipeline / model configs.  nerfstudio is absent from the image, so both sides run against stand-in
classes that record constructor arguments: the reference's side was recorded by tests/golden/make_golden_config.py
(executing the reference file unmodified), ours is recorded here."""
import dataclasses
import importlib
import json
import os
import sys

import pytest

from tests.golden.make_golden_config import NERFSTUDIO, Rec, recording_modules


@pytest.fixture()
def fake_nerfstudio():
    before = set(sys.modules)
    recording_modules(NERFSTUDIO)
    yield
    for k in set(sys.modules) - before:
        del sys.modules[k]


def test_method_specifications_match_the_reference(fake_nerfstudio, golden_dir):
    import dn_splatter_b200.dn_config as C
    from dn_splatter_b200.dn_model import DNSplatterModelConfig
    from dn_splatter_b200.dn_pipeline import DNSplatterPipelineConfig

    want = json.load(open(os.path.join(golden_dir, "dn_config_specs.json")))
    dm = Rec(dataparser=Rec(load_3D_points=True))
    specs = C.method_specifications(datamanager_config=dm)
    assert sorted(specs) == sorted(want) == ["ags-mesh", "dn-splatter", "dn-splatter-big"]
    defaults = DNSplatterModelConfig()
    ours_only = {"exact_isect_lists", "sync_free", "fused_ssim", "fuse_loss_backward", "list_shift"}
    for name, spec in specs.items():
        w = want[name]
        assert spec.kw["description"] == w["description"]
        got_tr, want_tr = spec.kw["config"].kw, w["config"]
        plain = lambda d: {k: v for k, v in d.items() if k not in ("pipeline", "optimizers", "viewer", "__class__")}  # noqa: E731
        assert plain(got_tr) == plain(want_tr), name
        assert got_tr["viewer"].kw == {k: v for k, v in want_tr["viewer"].items() if k != "__class__"}
        # optimizer groups: same names, lr / eps, schedules
        assert sorted(got_tr["optimizers"]) == sorted(want_tr["optimizers"])
        for grp, o in got_tr["optimizers"].items():
            wo = want_tr["optimizers"][grp]
            assert o["optimizer"].kw == {k: v for k, v in wo["optimizer"].items() if k != "__class__"}, (name, grp)
            if wo["scheduler"] is None:
                assert o["scheduler"] is None
            else:
                assert o["scheduler"].kw == {k: v for k, v in wo["scheduler"].items() if k != "__class__"}, (name, grp)
        # pipeline: our config class, the caller's datamanager, the reference's model overrides and nothing else
        pipe = got_tr["pipeline"]
        assert isinstance(pipe, DNSplatterPipelineConfig) and pipe.datamanager is not dm and pipe.datamanager.kw.keys() == dm.kw.keys()
        overrides = {k: v for k, v in want_tr["pipeline"]["model"].items() if k != "__class__"}
        model = pipe.model
        assert isinstance(model, DNSplatterModelConfig)
        for k, v in overrides.items():
            assert getattr(model, k) == v, (name, k)
        changed = {f.name for f in dataclasses.fields(model)
                   if f.name != "_target" and getattr(model, f.name) != getattr(defaults, f.name)}
        assert changed - ours_only <= set(overrides), (name, changed)
    # module attributes for the entry points ('dn_splatter_b200.dn_config:dn_splatter', ...)
    with pytest.raises(AttributeError):
        C.no_such_method


def test_config_keeps_the_reference_field_names(golden_dir):
    """Every field of the reference's DNSplatterModelConfig exists here with the same default (SURVEY §8b, a14)."""
    import ast

    from dn_splatter_b200.dn_model import CameraOptimizerConfig, DNSplatterModelConfig

    cfg = DNSplatterModelConfig()
    # every `name: type = default` of the reference's config class, recorded by tests/golden/make_golden_config.py
    ref = json.load(open(os.path.join(golden_dir, "dn_model_config_fields.json")))
    expect = {"regularization_strategy": "dn-splatter", "use_depth_loss": False, "depth_tolerance": 0.1, "depth_lambda": 0.0,
              "use_depth_smooth_loss": False, "smooth_loss_lambda": 0.1, "predict_normals": True, "use_normal_loss": True,
              "use_normal_cosine_loss": False, "use_normal_tv_loss": True, "normal_supervision": "mono", "normal_lambda": 0.1,
              "use_sparse_loss": False, "sparse_lambda": 0.1, "sparse_loss_steps": 10, "use_binary_opacities": False,
              "binary_opacities_threshold": 0.9, "two_d_gaussians": True, "warmup_length": 500, "num_downscales": 0,
              "use_scale_regularization": False, "max_gauss_ratio": 5.0, "stop_split_at": 15000,
              "output_depth_during_training": True, "pearson_lambda": 0}
    assert set(ref) - {"_target"} == set(expect) | {"depth_loss_type", "smooth_loss_type", "camera_optimizer"}
    for k, v in expect.items():
        assert ast.literal_eval(ref[k]) == v, k
        assert getattr(cfg, k) == v, k
    assert ref["depth_loss_type"] == "DepthLossType.EdgeAwareLogL1" and ref["smooth_loss_type"] == "DepthLossType.TV"
    assert "CameraOptimizerConfig(mode='off')" in ref["camera_optimizer"]
    assert isinstance(cfg.camera_optimizer, CameraOptimizerConfig) and cfg.camera_optimizer.mode == "off"
    assert cfg.depth_loss_type.value == "EdgeAwareLogL1" and cfg.smooth_loss_type.value == "TV"
