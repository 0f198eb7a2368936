"""Drop-in check at the plugin boundary (SURVEY.md 8b): the REFERENCE's own plugin sources -- PseudoLabRPN / DARPN,
SourceFreeAdaptiveTeacherStandardROIHeads (+ Eval, AdaptiveTeacher variants), SourceFreeFastRCNNOutputLayers, vgg_backbone --
import unchanged against ``sfod_b200.d2shim`` (a ``detectron2`` namespace backed by this package) and build from the
reference's config keys on top of the B200 base classes.  Reads a checkout of the original project named by $SFOD_REFERENCE_ROOT
and is skipped without one.  No reference source is copied into the repository."""
import importlib
import os
import sys
import types

import pytest
import torch

REF_ROOT = os.environ.get("SFOD_REFERENCE_ROOT", "")
REF = os.path.join(REF_ROOT, "daod", "modeling")
pytestmark = pytest.mark.skipif(not (REF_ROOT and os.path.isdir(REF)), reason="original project sources not available (SFOD_REFERENCE_ROOT)")


@pytest.fixture(scope="module")
def ref():
    import sfod_b200  # noqa: F401
    from sfod_b200 import d2shim
    had = {k: v for k, v in sys.modules.items() if k.split(".")[0] == "detectron2"}
    assert d2shim.install(force=True)
    pkgs = {}
    for name, sub in (("refdaod_pg", "proposal_generator"), ("refdaod_rh", "roi_heads"), ("refdaod_ma", "meta_arch")):
        m = types.ModuleType(name)
        m.__path__ = [os.path.join(REF, sub)]          # the package's real __init__ (which pulls unrelated baselines) is not executed
        sys.modules[name] = m
        pkgs[sub] = name
    mods = {
        "rpn": importlib.import_module("refdaod_pg.rpn"),
        "fast": importlib.import_module("refdaod_rh.source_free_fast_rcnn"),
        "heads": importlib.import_module("refdaod_rh.source_free_adaptive_teacher_roi_heads"),
        "heads_eval": importlib.import_module("refdaod_rh.source_free_adaptive_teacher_roi_heads_eval"),
        "heads_at": importlib.import_module("refdaod_rh.adaptive_teacher_roi_heads"),
        "vgg": importlib.import_module("refdaod_ma.vgg"),
    }
    yield mods, sys.modules["detectron2"].registries
    d2shim.uninstall()
    for k in [k for k in sys.modules if k.startswith("refdaod_")]:
        del sys.modules[k]
    sys.modules.update(had)


def test_reference_plugin_sources_import_and_register(ref):
    mods, regs = ref
    from sfod_b200 import modeling
    for name in ("PseudoLabRPN", "DARPN"):
        assert name in regs["PROPOSAL_GENERATOR"]
    for name in ("SourceFreeAdaptiveTeacherStandardROIHeads", "SourceFreeAdaptiveTeacherEvalStandardROIHeads", "AdaptiveTeacherStandardROIHeads"):
        assert name in regs["ROI_HEADS"]
    for name in ("build_vgg_backbone", "build_vgg_fpn_backbone"):
        assert name in regs["BACKBONE"]
    # the reference classes are the reference's code (defined under REF_ROOT) on top of THIS package's bases
    assert mods["rpn"].PseudoLabRPN.__module__ == "refdaod_pg.rpn" and issubclass(mods["rpn"].PseudoLabRPN, modeling.RPN)
    assert issubclass(mods["fast"].SourceFreeFastRCNNOutputLayers, modeling.FastRCNNOutputLayers)
    assert mods["heads"].__file__.startswith(REF_ROOT)
    # the rest of the detectron2.layers census of SURVEY.md 8(b) (reference box_head.py:9, trainers/base.py:22)
    from detectron2.layers import Conv2d, FrozenBatchNorm2d, get_norm
    assert isinstance(get_norm("BN", 8), torch.nn.BatchNorm2d) and isinstance(get_norm("FrozenBN", 8), FrozenBatchNorm2d)
    assert get_norm("", 8) is None and issubclass(Conv2d, torch.nn.Conv2d)


def test_reference_plugins_build_from_cfg_and_reach_the_kernel_boundary(ref):
    mods, regs = ref
    import detectron2.modeling as d2m                      # the shim
    from sfod_b200 import config, modeling
    from sfod_b200.structures import Boxes, ImageList, Instances
    cfg = config.vgg_source_free_cfg(); cfg.MODEL.DEVICE = "cpu"
    torch.manual_seed(0)
    backbone = d2m.build_backbone(cfg)                     # reference vgg_backbone (nn.BatchNorm2d layers)
    ours = modeling.vgg_backbone(cfg)
    assert type(backbone).__module__ == "refdaod_ma.vgg"
    assert list(backbone.state_dict().keys()) == list(ours.state_dict().keys())          # identical checkpoint layout
    assert backbone.output_shape()["vgg4"].stride == 32 and backbone.output_shape()["vgg4"].channels == 512
    rpn = d2m.build_proposal_generator(cfg, backbone.output_shape())
    heads = d2m.build_roi_heads(cfg, backbone.output_shape())
    assert type(rpn).__module__ == "refdaod_pg.rpn" and type(heads).__module__ == "refdaod_rh.source_free_adaptive_teacher_roi_heads"
    assert type(heads.box_predictor).__module__ == "refdaod_rh.source_free_fast_rcnn"
    assert isinstance(heads.box_pooler, modeling.ROIPooler) and heads.box_pooler.pooler_type == "ROIAlignV2"
    assert rpn.pre_nms_topk == {True: 12000, False: 6000} and rpn.post_nms_topk == {True: 2000, False: 1000}
    # the reference's forward runs its own Python and lands in libsfod_b200 at the operator boundary: on CPU tensors the
    # library refuses (no CPU fallback) -- exactly at predict_proposals / the box pooler
    feats = {"vgg4": torch.randn(1, 512, 6, 8)}
    images = ImageList(torch.zeros(1, 3, 192, 256), [(192, 256)])
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        rpn(images, feats, None, compute_loss=False)
    prop = Instances((192, 256)); prop.proposal_boxes = Boxes(torch.tensor([[4.0, 4, 100, 90]])); prop.objectness_logits = torch.zeros(1)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        heads(images, feats, [prop], targets=None, compute_loss=False, branch="unsup_data_weak")
    # the reference's label_and_sample_proposals (its own override) runs on the shimmed helpers
    tgt = Instances((192, 256)); tgt.gt_boxes = Boxes(torch.tensor([[0.0, 0, 110, 100]])); tgt.gt_classes = torch.tensor([3])
    from sfod_b200.utils.events import EventStorage
    with EventStorage() as st:
        out = heads.label_and_sample_proposals([prop], [tgt], branch="supervised_target")
    assert len(out[0]) == 2 and sorted(out[0].gt_classes.tolist()) == [3, 3]            # proposal + appended GT, both foreground
    assert "roi_head/num_target_fg_samples_supervised_target" in st.latest()


def test_reference_meta_arch_source_builds_on_the_shim(ref):
    """One level up: the reference's own META-ARCHITECTURE source (daod/modeling/meta_arch/source_free_adaptive_teacher_rcnn.py,
    `@configurable` + `from_config`, its `dann` and `bpc_loss` imports) loads unchanged, builds from the config through the
    shim's registries -- i.e. out of the reference's own backbone / RPN / ROI-head plugin classes on the B200 bases -- has the
    checkpoint layout of this package's mirror, and its forward reaches the kernel boundary."""
    mods, regs = ref
    import types as _types
    from sfod_b200 import config, modeling
    ref_root = os.path.dirname(REF)                                  # <REF_ROOT>/daod
    stubs = {"daod": [ref_root], "daod.modeling": [REF], "daod.loss": [os.path.join(ref_root, "loss")]}
    saved = {k: sys.modules.get(k) for k in list(stubs) + ["daod.modeling.dann", "daod.loss.bpc_loss"]}
    try:
        for name, path in stubs.items():                              # namespace stubs: the packages' real __init__ files are not run
            m = _types.ModuleType(name); m.__path__ = path; sys.modules[name] = m
        ma = importlib.import_module("refdaod_ma.source_free_adaptive_teacher_rcnn")
        assert ma.__file__.startswith(REF_ROOT)
        # the other meta-architectures the reference registers (daod/modeling/meta_arch/__init__.py:1-5) stay importable too
        for other in ("adaptive_teacher_rcnn", "da_faster_rcnn", "cda_faster_rcnn", "ts_ensemble"):
            importlib.import_module("refdaod_ma." + other)
        for name in ("AdaptiveTeacherGeneralizedRCNN", "MeanTeacherGeneralizedRCNN", "DAFasterRCNN", "CDAFasterRCNN"):
            assert name in regs["META_ARCH"], name
        cls = regs["META_ARCH"].get("SourceFreeAdaptiveTeacherGeneralizedRCNN")
        assert cls is ma.SourceFreeAdaptiveTeacherGeneralizedRCNN and cls.__module__ == "refdaod_ma.source_free_adaptive_teacher_rcnn"
        cfg = config.vgg_source_free_cfg(); cfg.MODEL.DEVICE = "cpu"
        torch.manual_seed(0)
        model = cls(cfg)                                              # detectron2's `configurable` protocol: cfg -> from_config -> __init__
        assert type(model.backbone).__module__ == "refdaod_ma.vgg"
        assert type(model.proposal_generator).__module__ == "refdaod_pg.rpn"
        assert type(model.roi_heads).__module__ == "refdaod_rh.source_free_adaptive_teacher_roi_heads"
        mirror = modeling.SourceFreeAdaptiveTeacherGeneralizedRCNN(cfg)
        ref_sd, our_sd = model.state_dict(), mirror.state_dict()
        assert list(ref_sd.keys()) == list(our_sd.keys())             # same checkpoint: names, order
        assert all(ref_sd[k].shape == our_sd[k].shape and ref_sd[k].dtype == our_sd[k].dtype for k in ref_sd)
        mirror.load_state_dict(ref_sd)                                # and loadable both ways
        model.load_state_dict(mirror.state_dict())
        # the reference's forward (its own Python) on a CPU batch runs its torch backbone and stops at the first native operator
        model.train()
        batch = [{"image": torch.randint(0, 256, (3, 96, 128), dtype=torch.uint8).float()}]
        with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA tensors only"):
            model(batch, branch="unsup_data_weak")
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_reference_hook_runs_on_the_trainer_protocol(ref):
    """The reference's own ValLossHook (daod/engine/hooks/val_loss.py) subclasses detectron2's HookBase; on the shim it runs
    unchanged on this package's TrainerBase: same callbacks, `trainer.iter` / `max_iter` / `storage`."""
    import types as _types
    from sfod_b200.engine import HookBase, TrainerBase
    m = _types.ModuleType("refdaod_hooks"); m.__path__ = [os.path.join(REF_ROOT, "daod", "engine", "hooks")]; sys.modules["refdaod_hooks"] = m
    try:
        vl = importlib.import_module("refdaod_hooks.val_loss")
        assert vl.__file__.startswith(REF_ROOT) and issubclass(vl.ValLossHook, HookBase)

        class Model:
            def __call__(self, data):
                return {"loss_cls": torch.tensor(0.5) * data, "loss_box_reg": 0.25 * data, "num_fg": 3.0}, [], []

        class Loop(TrainerBase):
            steps = 0
            def run_step(self):
                self.steps += 1

        order = []
        class Probe(HookBase):
            def before_train(self): order.append("before_train")
            def before_step(self): order.append(f"before_step{self.trainer.iter}")
            def after_step(self): order.append(f"after_step{self.trainer.iter}")
            def after_train(self): order.append("after_train")

        loop = Loop()
        loop.register_hooks([Probe(), None, vl.ValLossHook(2, Model(), [1.0, 3.0], model_name="_student")])
        loop.train(0, 5)
        assert loop.steps == 5 and loop.iter == 5
        assert order[0] == "before_train" and order[-1] == "after_train" and order[1:3] == ["before_step0", "after_step0"]
        # evaluated after iterations 1, 3 (period 2) and 4 (final): mean over the loader of each loss_* entry
        hist = loop.storage.history("total_loss_student_val")
        assert len(hist) == 3 and abs(hist[-1] - (0.5 * 2.0 + 0.25 * 2.0)) < 1e-6
        assert abs(loop.storage.latest()["loss_cls_student_val"] - 1.0) < 1e-6 and "num_fg_student_val" not in loop.storage.latest()
    finally:
        for k in [k for k in sys.modules if k.startswith("refdaod_hooks")]:
            del sys.modules[k]
