"""The reference's own config files (configs/rsprompter/*-nwpu*.py) build the B200 modules through the registry
surface.  tests/golden/reference_configs.pt holds each file resolved through its ``_base_`` chain (``model`` and
``custom_imports``; tests/golden/make_golden.py configs)."""
import copy
import os

import pytest
import torch

FX = torch.load(os.path.join(os.path.dirname(__file__), "golden", "reference_configs.pt"), weights_only=False)


def _load(name):
    """The resolved reference config file `name` as a Config."""
    from rsprompter_b200.registry import Config
    return Config(copy.deepcopy(FX[name]), filename=name)


def _strip_init(cfg):
    """Pretrained checkpoints do not exist offline: drop init_cfg (random init is loaded instead)."""
    if isinstance(cfg, dict):
        cfg.pop("init_cfg", None)
        for v in cfg.values():
            _strip_init(v)
    elif isinstance(cfg, (list, tuple)):
        for v in cfg:
            _strip_init(v)
    return cfg


def test_base_config_inheritance_and_delete(tmp_path):
    """Config.fromfile merges a child over its ``_base_`` the way rsprompter_anchor-nwpu-peft-512.py sits on
    _base_/rsprompter_anchor.py: ``backbone`` and ``neck.feature_aggregator`` are replaced (``_delete_=True``), the rest
    of the model, ``neck.feature_spliter`` included, is inherited."""
    from rsprompter_b200.registry import Config
    base, peft = FX["rsprompter_anchor-nwpu.py"], FX["rsprompter_anchor-nwpu-peft-512.py"]
    assert "extra_config" in base["model"]["backbone"]
    (tmp_path / "_base_").mkdir()
    (tmp_path / "_base_" / "base.py").write_text(
        f"custom_imports = {base['custom_imports']!r}\nmodel = {base['model']!r}\n")
    child = dict(backbone=dict(_delete_=True, **peft["model"]["backbone"]),
                 neck=dict(feature_aggregator=dict(_delete_=True, **peft["model"]["neck"]["feature_aggregator"])))
    (tmp_path / "child.py").write_text(f"_base_ = ['_base_/base.py']\nmodel = {child!r}\n")
    cfg = Config.fromfile(str(tmp_path / "child.py"))
    m = cfg.model
    assert m.type == "RSPrompterAnchor"                                   # from _base_
    assert m.backbone.type == "MMPretrainSamVisionEncoder" and "extra_config" not in m.backbone  # _delete_
    assert m.neck.feature_aggregator.type == "PseudoFeatureAggregator"
    assert m.neck.feature_spliter.type == "RSSimpleFPN"                   # merged, not replaced
    assert m.roi_head.bbox_head.num_classes == 10
    assert m.test_cfg.rcnn.max_per_img == 100
    assert cfg.custom_imports["imports"] == ["mmdet.rsprompter"]
    ref = _load("rsprompter_anchor-nwpu-peft-512.py").model
    assert m.backbone == ref.backbone and m.neck == ref.neck


@pytest.mark.parametrize("name,enc_cls", [("rsprompter_anchor-nwpu.py", "RSSamVisionEncoder"),
                                          ("rsprompter_anchor-nwpu-peft-512.py", "MMPretrainSamVisionEncoder")])
def test_reference_anchor_configs_build(name, enc_cls):
    from rsprompter_b200 import synthetic
    from rsprompter_b200.registry import MODELS
    cfg = _load(name)
    model_cfg = _strip_init(cfg.to_dict()["model"])
    model = MODELS.build(model_cfg)
    assert type(model).__name__ == "RSPrompterAnchor"
    assert type(model.backbone).__name__ == enc_cls
    arch = model.backbone.vision_encoder.arch
    assert arch.name == "base" and arch.hidden_size == 768
    if enc_cls == "MMPretrainSamVisionEncoder":
        assert arch.image_size == 512 and arch.grid == 32
        assert model.backbone.vision_encoder.layers[2].attn.rel_pos_h.shape == (63, 64)
        sd = synthetic.anchor_detector_state_dict(arch, 10, 0, seed=0, pseudo_neck=True)
    else:
        sd = synthetic.anchor_detector_state_dict(arch, 10, 6, seed=0)
    assert set(model.state_dict()) == set(sd)
    model.load_state_dict(sd, strict=True)
    assert model.roi_head.test_cfg.score_thr == 0.05 and model.rpn_head.test_cfg.nms_pre == 1000


@pytest.mark.parametrize("name,enc_cls,nq", [("rsprompter_query-nwpu.py", "RSSamVisionEncoder", 70),
                                             ("rsprompter_query-nwpu-peft-512.py", "MMPretrainSamVisionEncoder", 70)])
def test_reference_query_configs_build(name, enc_cls, nq):
    from rsprompter_b200 import synthetic
    from rsprompter_b200.registry import MODELS
    cfg = _load(name)
    model_cfg = _strip_init(cfg.to_dict()["model"])
    model = MODELS.build(model_cfg)
    assert type(model).__name__ == "RSPrompterQuery" and type(model.backbone).__name__ == enc_cls
    head = model.panoptic_head
    assert head.num_queries == nq and head.num_classes == 10 and head.per_pointset_point == 5
    assert head.pixel_decoder.num_encoder_levels == 3 and head.pixel_decoder.num_points == 4 and head.num_layers == 6
    assert model.panoptic_fusion_head.test_cfg.max_per_image == nq and model.test_cfg.instance_on
    arch = model.backbone.vision_encoder.arch
    pseudo = enc_cls == "MMPretrainSamVisionEncoder"
    sd = synthetic.query_detector_state_dict(arch, 10, 0 if pseudo else 6, nq=nq, seed=0, pseudo_neck=pseudo)
    assert set(model.state_dict()) == set(sd)
    model.load_state_dict(sd, strict=True)


def test_reference_samdet_config_builds_the_segmentor():
    """configs/rsprompter/samdet-nwpu.py: type SAMDet with a stock mmdet FasterRCNN detector (outside this package) and
    an RSSamModel segmentor (SURVEY 8(f4), M:718-741, 1060-1215): the segmentor entry builds the B200 SamModel
    (ViT-B: samdet-nwpu.py:25 points at sam_vit_base) with HF SamModel's parameter names; SAMDet is in the registry."""
    from rsprompter_b200.registry import MODELS
    cfg = _load("samdet-nwpu.py")
    m = cfg.to_dict()["model"]
    assert m["type"] == "SAMDet" and MODELS.get("SAMDet") is not None
    assert m["segmentor"]["type"] == "RSSamModel" and m["detector"]["type"] == "FasterRCNN"
    seg = MODELS.build(_strip_init(dict(m["segmentor"])))
    sam = seg.sam_model
    assert sam.varch.name == "base" and sam.varch.num_layers == 12
    keys = set(sam.state_dict())
    for k in ("vision_encoder.layers.11.attn.qkv.weight", "prompt_encoder.point_embed.3.weight",
              "prompt_encoder.shared_embedding.positional_embedding", "shared_image_embedding.positional_embedding",
              "mask_decoder.transformer.layers.1.cross_attn_image_to_token.out_proj.weight",
              "mask_decoder.output_hypernetworks_mlps.3.proj_out.weight"):
        assert k in keys, k


def test_reference_samseg_maskrcnn_config_builds():
    """configs/rsprompter/samseg-maskrcnn-nwpu.py (SURVEY 8(f4); M:1218-1244): SAMSegMaskRCNN with the stock
    StandardRoIHead / Shared2FCBBoxHead / FCNMaskHead builds from the reference's own config file and takes a state dict
    with mmdet's parameter names (fcn_mask_head.py:68-126: convs.N.conv, upsample, conv_logits)."""
    from rsprompter_b200 import synthetic
    from rsprompter_b200.registry import MODELS
    cfg = _load("samseg-maskrcnn-nwpu.py")
    model = MODELS.build(_strip_init(cfg.to_dict()["model"]))
    assert type(model).__name__ == "SAMSegMaskRCNN" and type(model.roi_head).__name__ == "StandardRoIHead"
    assert type(model.roi_head.mask_head).__name__ == "FCNMaskHead" and model.roi_head.mask_head.num_classes == 10
    assert model.rpn_head.prior_generator.num_base_priors[0] == 3            # scales=[8] x 3 ratios
    arch = model.backbone.vision_encoder.arch
    assert arch.name == "base"
    sd = synthetic.maskrcnn_detector_state_dict(arch, 10, 6, seed=0)
    assert set(model.state_dict()) == set(sd)
    model.load_state_dict(sd, strict=True)
    assert sd["roi_head.mask_head.upsample.weight"].shape == (256, 256, 2, 2)
    assert sd["roi_head.mask_head.conv_logits.weight"].shape == (10, 256, 1, 1)
    assert model.test_cfg.rcnn.mask_thr_binary == 0.5 and not hasattr(model, "shared_image_embedding")


def test_reference_samseg_mask2former_config_builds():
    """configs/rsprompter/samseg-mask2former-nwpu.py (SURVEY 8(f4); M:1247-1274): SAMSegMask2Former with the stock
    Mask2FormerHead (feat_channels 256, 9 decoder layers, FFN 2048) / MaskFormerFusionHead builds from the reference's
    own config file and takes a state dict with mmdet's parameter names."""
    from rsprompter_b200 import synthetic
    from rsprompter_b200.registry import MODELS
    cfg = _load("samseg-mask2former-nwpu.py")
    model = MODELS.build(_strip_init(cfg.to_dict()["model"]))
    assert type(model).__name__ == "SAMSegMask2Former" and type(model.panoptic_head).__name__ == "Mask2FormerHead"
    assert type(model.panoptic_fusion_head).__name__ == "MaskFormerFusionHead"
    head = model.panoptic_head
    assert head.feat_channels == 256 and head.num_layers == 9 and head.num_queries == 70 and head.num_classes == 10
    assert head.pixel_decoder.E == 256 and head.pixel_decoder.num_encoder_levels == 3
    arch = model.backbone.vision_encoder.arch
    sd = synthetic.mask2former_detector_state_dict(arch, 10, 6, nq=70, seed=0)          # nwpu: num_queries = 70
    assert set(model.state_dict()) == set(sd)
    model.load_state_dict(sd, strict=True)
    assert sd["panoptic_head.cls_embed.weight"].shape == (11, 256)
    assert sd["panoptic_head.transformer_decoder.layers.8.ffn.layers.0.0.weight"].shape == (2048, 256)
    assert sd["panoptic_head.pixel_decoder.encoder.layers.2.ffn.layers.1.weight"].shape == (256, 1024)
    assert model.test_cfg.instance_on and not model.test_cfg.panoptic_on
