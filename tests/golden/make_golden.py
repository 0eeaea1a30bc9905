"""Generates tests/golden/reference_functions.pt by EXECUTING the reference's own in-tree source
(read from /root/reference at generation time; nothing is copied into this repo).

The reference package cannot be imported here (mmcv / mmengine / peft are absent), so the pure
tensor functions / methods on the hot path are pulled out of their files with `ast` and executed
in a namespace that only provides torch / numpy / math; methods get a SimpleNamespace `self`.
Run in the build container:   python tests/golden/make_golden.py
The fixtures pin oracle/restate*.py in tests/test_golden_cpu.py (no /root/reference at test time).
"""
import ast
import math
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch
import torch.nn.functional as F

REF = "/root/reference"
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_functions.pt")


def load_defs(relpath, names, cls=None):
    """Compile the named top-level functions (or methods of class `cls`) of a reference file."""
    src = open(os.path.join(REF, relpath)).read()
    tree = ast.parse(src)
    body = tree.body
    if cls is not None:
        body = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == cls).body
    ns = dict(torch=torch, F=F, np=np, math=math, Tensor=torch.Tensor, Tuple=tuple, Optional=None,
              Sequence=None, Union=None, List=list)
    for node in body:
        if isinstance(node, ast.FunctionDef) and node.name in names:
            node.decorator_list = []
            node.returns = None
            for a in node.args.args + node.args.kwonlyargs:
                a.annotation = None
            mod = ast.Module(body=[node], type_ignores=[])
            exec(compile(ast.fix_missing_locations(mod), relpath, "exec"), ns)
    missing = [n for n in names if n not in ns]
    assert not missing, f"{relpath}: {missing} not found"
    return ns


def main():
    g = torch.Generator().manual_seed(1234)
    fx = {}

    # ---- mmpretrain/models/backbones/vit_sam.py:17-157
    vs = load_defs("mmpretrain/models/backbones/vit_sam.py",
                   ["window_partition", "window_unpartition", "get_rel_pos", "add_decomposed_rel_pos"])
    x = torch.randn(2, 20, 23, 8, generator=g)
    win, pad_hw = vs["window_partition"](x, 14)
    fx["window_partition"] = dict(x=x, ws=14, windows=win, pad_hw=tuple(pad_hw),
                                  back=vs["window_unpartition"](win, 14, pad_hw, (20, 23)))
    table = torch.randn(27, 16, generator=g)
    fx["get_rel_pos_same"] = dict(q=14, k=14, table=table, out=vs["get_rel_pos"](14, 14, table))
    table2 = torch.randn(127, 16, generator=g)
    fx["get_rel_pos_resized"] = dict(q=32, k=32, table=table2, out=vs["get_rel_pos"](32, 32, table2))
    S, hd, nb = 6, 16, 3
    q = torch.randn(nb, S * S, hd, generator=g)
    rh, rw = torch.randn(2 * S - 1, hd, generator=g), torch.randn(2 * S - 1, hd, generator=g)
    attn = torch.zeros(nb, S * S, S * S)
    fx["decomposed_rel_pos"] = dict(q=q, rel_h=rh, rel_w=rw, S=S,
                                    bias=vs["add_decomposed_rel_pos"](attn, q, rh, rw, (S, S), (S, S)))

    # ---- mmdet/models/task_modules/coders/delta_xywh_bbox_coder.py:262-359
    dc = load_defs("mmdet/models/task_modules/coders/delta_xywh_bbox_coder.py", ["delta2bbox"])
    rois = torch.rand(40, 4, generator=g) * 200
    rois[:, 2:] = rois[:, :2] + torch.rand(40, 2, generator=g) * 300 + 1
    deltas = torch.randn(40, 12, generator=g) * 2
    fx["delta2bbox"] = dict(rois=rois, deltas=deltas, stds=(0.1, 0.1, 0.2, 0.2), max_shape=(256, 320),
                            out=dc["delta2bbox"](rois, deltas, (0., 0., 0., 0.), (0.1, 0.1, 0.2, 0.2), (256, 320)))
    d1 = torch.randn(40, 4, generator=g)
    fx["delta2bbox_rpn"] = dict(rois=rois, deltas=d1, stds=(1., 1., 1., 1.), max_shape=(256, 320),
                                out=dc["delta2bbox"](rois, d1, (0., 0., 0., 0.), (1., 1., 1., 1.), (256, 320)))

    # ---- mmdet/models/task_modules/prior_generators/anchor_generator.py:161-301
    ag = load_defs("mmdet/models/task_modules/prior_generators/anchor_generator.py",
                   ["gen_single_level_base_anchors", "_meshgrid", "single_level_grid_priors"], cls="AnchorGenerator")
    self_ = SimpleNamespace(center_offset=0.0, scale_major=True, strides=[(8, 8)], use_box_type=False)
    self_._meshgrid = lambda x, y, row_major=True: ag["_meshgrid"](self_, x, y, row_major)
    base = ag["gen_single_level_base_anchors"](self_, 8, torch.tensor([4., 8.]), torch.tensor([0.5, 1.0, 2.0]))
    self_.base_anchors = [base]
    fx["anchors"] = dict(base_size=8, scales=[4, 8], ratios=[0.5, 1.0, 2.0], base=base, featmap=(3, 5), stride=8,
                         grid=ag["single_level_grid_priors"](self_, (3, 5), 0, torch.float32, "cpu"))

    # ---- mmdet/models/layers/positional_encoding.py:60-110
    pe = load_defs("mmdet/models/layers/positional_encoding.py", ["forward"], cls="SinePositionalEncoding")
    self_ = SimpleNamespace(num_feats=8, temperature=10000, normalize=True, scale=2 * math.pi, eps=1e-6, offset=0.0)
    fx["sine_pe"] = dict(B=2, H=5, W=7, num_feats=8, out=pe["forward"](self_, torch.zeros(2, 5, 7, dtype=torch.bool)))

    # ---- mmdet/models/roi_heads/roi_extractors/single_level_roi_extractor.py:40-62
    re_ = load_defs("mmdet/models/roi_heads/roi_extractors/single_level_roi_extractor.py", ["map_roi_levels"],
                    cls="SingleRoIExtractor")
    r5 = torch.cat([torch.zeros(40, 1), rois * torch.rand(40, 1, generator=g) * 4], dim=1)
    fx["map_roi_levels"] = dict(rois=r5, num_levels=4,
                                out=re_["map_roi_levels"](SimpleNamespace(finest_scale=56), r5, 4))

    # ---- mmdet/structures/mask/utils.py:56-77
    mu = load_defs("mmdet/structures/mask/utils.py", ["mask2bbox"])
    masks = torch.rand(6, 20, 30, generator=g) > 0.9
    masks[2] = False
    fx["mask2bbox"] = dict(masks=masks, out=mu["mask2bbox"](masks))

    # ---- mmdet/rsprompter/models.py:45-50 LN2d.forward
    ln = load_defs("mmdet/rsprompter/models.py", ["forward"], cls="LN2d")
    w, b = torch.randn(8, generator=g), torch.randn(8, generator=g)
    xx = torch.randn(2, 8, 4, 5, generator=g)
    fx["ln2d"] = dict(x=xx, weight=w, bias=b, eps=1e-6,
                      out=ln["forward"](SimpleNamespace(weight=w, bias=b, eps=1e-6), xx))

    # ---- mmdet/models/seg_heads/panoptic_fusion_heads/maskformer_fusion_head.py:126-182 instance_postprocess
    class _Inst(SimpleNamespace):
        pass
    fh = load_defs("mmdet/models/seg_heads/panoptic_fusion_heads/maskformer_fusion_head.py", ["instance_postprocess"],
                   cls="MaskFormerFusionHead")
    fh["instance_postprocess"].__globals__.update(mask2bbox=mu["mask2bbox"], InstanceData=_Inst)
    nq, ncls = 12, 5
    mask_cls = torch.randn(nq, ncls + 1, generator=g) * 2
    yy, xx2 = torch.meshgrid(torch.arange(40), torch.arange(48), indexing="ij")
    cy, cx, rr = torch.rand(nq, 1, 1, generator=g) * 40, torch.rand(nq, 1, 1, generator=g) * 48, torch.rand(nq, 1, 1, generator=g) * 12
    mask_pred = (rr + 2 - ((yy - cy) ** 2 + (xx2 - cx) ** 2).sqrt()) * 1.3 + 0.1 * torch.randn(nq, 40, 48, generator=g)
    self_ = SimpleNamespace(test_cfg=dict(max_per_image=7), num_classes=ncls, num_things_classes=ncls)
    res = fh["instance_postprocess"](self_, mask_cls, mask_pred)
    fx["instance_postprocess"] = dict(mask_cls=mask_cls, mask_pred=mask_pred, num_classes=ncls, max_per_image=7,
                                      bboxes=res.bboxes, labels=res.labels, scores=res.scores, masks=res.masks)

    # ---- mmdet/rsprompter/models.py:661-715 RSMaskFormerFusionHead.predict (crop to the resized image + rescale)
    rf = load_defs("mmdet/rsprompter/models.py", ["predict"], cls="RSMaskFormerFusionHead")
    meta = dict(img_shape=(60, 96), ori_shape=(50, 80), scale_factor=(1.2, 1.2), batch_input_shape=(96, 96))
    self_ = SimpleNamespace(test_cfg=dict(panoptic_on=False, semantic_on=False, instance_on=True, max_per_image=7),
                            num_classes=ncls, num_things_classes=ncls)
    self_.instance_postprocess = lambda c, m: fh["instance_postprocess"](self_, c, m)
    mp_b = torch.randn(1, nq, 96, 96, generator=g) * 2
    out = rf["predict"](self_, mask_cls[None], mp_b, [SimpleNamespace(metainfo=meta)], rescale=True)[0]["ins_results"]
    fx["fusion_predict_rescale"] = dict(mask_cls=mask_cls, mask_pred=mp_b[0], meta=meta, num_classes=ncls, max_per_image=7,
                                        bboxes=out.bboxes, labels=out.labels, scores=out.scores, masks=out.masks)

    # ---- mmdet/rsprompter/models.py:1746-1784 RSPrompterAnchorMaskHead._predict_by_feat_single (rescale=True)
    mh = load_defs("mmdet/rsprompter/models.py", ["_predict_by_feat_single"], cls="RSPrompterAnchorMaskHead")
    meta2 = dict(ori_shape=(50, 80), scale_factor=(1.2, 1.2), batch_input_shape=(96, 96))
    logits = torch.randn(5, 1, 24, 24, generator=g) * 3
    boxes = torch.rand(5, 4, generator=g) * 90
    b_in = boxes.clone()
    im = mh["_predict_by_feat_single"](SimpleNamespace(), logits, b_in, torch.zeros(5, dtype=torch.long), meta2,
                                       SimpleNamespace(mask_thr_binary=0.5), rescale=True)
    fx["anchor_mask_rescale"] = dict(logits=logits, boxes=boxes, meta=meta2, masks=im, boxes_out=b_in)

    # ---- mmpretrain checkpoint resize at load time (VS:611-662, mmpretrain/models/utils/embed.py:16-59)
    import types
    fake_log = types.ModuleType("mmengine.logging")
    fake_log.MMLogger = SimpleNamespace(get_current_instance=lambda: SimpleNamespace(info=lambda *a, **k: None))
    sys.modules.setdefault("mmengine", types.ModuleType("mmengine"))
    sys.modules["mmengine.logging"] = fake_log
    em = load_defs("mmpretrain/models/utils/embed.py", ["resize_pos_embed"])
    vsl = load_defs("mmpretrain/models/backbones/vit_sam.py", ["_prepare_pos_embed", "_prepare_relative_position"],
                    cls="ViTSAM")
    vsl["_prepare_pos_embed"].__globals__.update(resize_pos_embed=em["resize_pos_embed"])
    ck_pos = torch.randn(1, 8, 8, 12, generator=g)
    ck_rel = torch.randn(15, 6, generator=g)
    ck_win = torch.randn(5, 6, generator=g)
    own = {"layers.0.attn.rel_pos_h": torch.zeros(7, 6), "layers.1.attn.rel_pos_w": torch.zeros(5, 6)}
    self_ = SimpleNamespace(pos_embed=torch.zeros(1, 4, 4, 12), patch_embed=SimpleNamespace(init_out_size=(4, 4)),
                            interpolate_mode="bicubic", embed_dims=12, state_dict=lambda: own)
    sd_ck = {"pos_embed": ck_pos.clone(), "layers.0.attn.rel_pos_h": ck_rel.clone(), "layers.1.attn.rel_pos_w": ck_win.clone()}
    vsl["_prepare_pos_embed"](self_, sd_ck, "")
    vsl["_prepare_relative_position"](self_, sd_ck, "")
    fx["ckpt_resize"] = dict(pos_embed=ck_pos, rel_pos=ck_rel, rel_win=ck_win, pos_embed_out=sd_ck["pos_embed"],
                             rel_pos_out=sd_ck["layers.0.attn.rel_pos_h"], rel_win_out=sd_ck["layers.1.attn.rel_pos_w"])

    torch.save(fx, OUT)
    print("wrote", OUT, {k: list(v.keys()) for k, v in fx.items()})


def main_maskrcnn():
    """tests/golden/reference_maskrcnn.pt: FCNMaskHead's paste path (SAMSegMaskRCNN), a file of its own so that the
    first fixture file stays byte-identical."""
    g = torch.Generator().manual_seed(4321)
    fx = {}
    rel = "mmdet/models/roi_heads/mask_heads/fcn_mask_head.py"
    pm = load_defs(rel, ["_do_paste_mask"])
    n, hm, H, W = 9, 28, 72, 100
    probs = torch.rand(n, 1, hm, hm, generator=g)
    boxes = torch.rand(n, 4, generator=g) * torch.tensor([60., 40., 60., 40.])
    boxes[:, 2:] = boxes[:, :2] + torch.rand(n, 2, generator=g) * 50 + 0.5
    boxes[0] = torch.tensor([-8.0, -3.5, 30.0, 90.0])          # sticks out of the canvas
    boxes[1] = torch.tensor([40.0, 10.0, 40.0, 30.0])          # zero width: inf -> 0 rule
    boxes[2] = torch.tensor([0.0, 0.0, float(W), float(H)])    # the whole canvas
    out, _ = pm["_do_paste_mask"](probs, boxes, H, W, skip_empty=False)
    fx["do_paste_mask"] = dict(probs=probs, boxes=boxes, hw=(H, W), out=out)

    mh = load_defs(rel, ["_predict_by_feat_single"], cls="FCNMaskHead")
    mh["_predict_by_feat_single"].__globals__.update(_do_paste_mask=pm["_do_paste_mask"], BYTES_PER_FLOAT=4,
                                                     GPU_MEM_LIMIT=1024 ** 3)
    C = 3
    logits = torch.randn(n, C, hm, hm, generator=g) * 3
    labels = torch.randint(0, C, (n,), generator=g)
    self_ = SimpleNamespace(class_agnostic=False)
    for name, rescale in (("fcn_predict_rescale", True), ("fcn_predict_norescale", False)):
        meta = dict(ori_shape=(60, 84), scale_factor=(1.25, 1.2))
        b_in = boxes.clone()
        im = mh["_predict_by_feat_single"](self_, logits.clone(), b_in, labels, meta,
                                           SimpleNamespace(mask_thr_binary=0.5), rescale=rescale)
        fx[name] = dict(logits=logits, boxes=boxes, labels=labels, meta=meta, rescale=rescale, masks=im, boxes_out=b_in)
    out_path = os.path.join(os.path.dirname(OUT), "reference_maskrcnn.pt")
    torch.save(fx, out_path)
    print("wrote", out_path, {k: list(v.keys()) for k, v in fx.items()})


def _exec_class(relpath, name, ns):
    """Execute one top-level class definition of a reference file (decorators and annotations stripped) in `ns`."""
    tree = ast.parse(open(os.path.join(REF, relpath)).read())
    node = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == name)
    node.decorator_list = []
    for sub in ast.walk(node):
        if isinstance(sub, ast.FunctionDef):
            sub.returns = None
            for a in sub.args.args + sub.args.kwonlyargs:
                a.annotation = None
    exec(compile(ast.fix_missing_locations(ast.Module(body=[node], type_ignores=[])), relpath, "exec"), ns)
    return ns[name]


def _self_assign(relpath, cls, attr, self_ns, ns):
    """Evaluate the right-hand side of `self.<attr> = ...` (last occurrence) inside `cls.__init__` of a reference file
    with `self` bound to `self_ns`; for constructors whose base classes (mmdet / mmcv) cannot be instantiated here."""
    tree = ast.parse(open(os.path.join(REF, relpath)).read())
    cnode = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == cls)
    init = next(n for n in cnode.body if isinstance(n, ast.FunctionDef) and n.name == "__init__")
    rhs = None
    for n in ast.walk(init):
        if isinstance(n, ast.Assign) and len(n.targets) == 1 and isinstance(n.targets[0], ast.Attribute) \
                and n.targets[0].attr == attr and getattr(n.targets[0].value, "id", None) == "self":
            rhs = n.value
    assert rhs is not None, (cls, attr)
    return eval(compile(ast.fix_missing_locations(ast.Expression(body=rhs)), relpath, "eval"), dict(ns, self=self_ns))


def main_state_keys():
    """tests/golden/reference_state_keys.json: parameter / buffer names and shapes produced by the reference's OWN
    constructors for the RSPrompter-specific modules (mmdet/rsprompter/models.py), executed here with torch only.
    mmengine's BaseModule is replaced by nn.Module; mmcv's ConvModule / build_norm_layer cannot be imported (mmcv is
    neither in the image nor under /root/reference), so sub-modules built through them (RSSimpleFPN's lateral / fpn
    convs and its LN2d) are recorded from a 12-line stand-in that follows mmcv's documented naming (conv under `.conv`,
    the norm under infer_abbr(LN2d) = `norm_layer`): those entries are marked "stub": true."""
    import json
    from torch import nn
    rel = "mmdet/rsprompter/models.py"

    class BaseModule(nn.Module):
        def __init__(self, init_cfg=None):
            super().__init__()

    ln_ns = dict(torch=torch, nn=nn, F=F)
    LayerNorm2d = _exec_class("mmpretrain/models/utils/norm.py", "LayerNorm2d", dict(ln_ns))
    ns = dict(torch=torch, nn=nn, F=F, BaseModule=BaseModule, LayerNorm2d=LayerNorm2d, List=list, Tensor=torch.Tensor)
    LN2d = _exec_class(rel, "LN2d", ns)

    def build_norm_layer(cfg, num_features, postfix=""):
        assert cfg["type"] == "LN2d"
        return "norm_layer" + str(postfix), LN2d(num_features, **{k: v for k, v in cfg.items() if k not in ("type", "requires_grad")})

    class ConvModule(nn.Module):      # stand-in, see the docstring
        def __init__(self, cin, cout, k, padding=0, conv_cfg=None, norm_cfg=None, act_cfg=None, inplace=False):
            super().__init__()
            self.conv = nn.Conv2d(cin, cout, k, padding=padding, bias=norm_cfg is None)
            if norm_cfg is not None:
                name, layer = build_norm_layer(norm_cfg, cout)
                self.add_module(name, layer)

    ns.update(build_norm_layer=build_norm_layer, ConvModule=ConvModule)
    out = {}

    def record(name, module, stub_prefixes=()):
        out[name] = {k: dict(shape=list(v.shape), **({"stub": True} if k.startswith(tuple(stub_prefixes)) and stub_prefixes else {}))
                     for k, v in module.state_dict().items()}

    agg = _exec_class(rel, "RSFeatureAggregator", ns)
    record("RSFeatureAggregator[base,hidden32,range(1,13,2)]",
           agg("work_dirs/sam_cache/sam_vit_base", hidden_channels=32, out_channels=256, select_layers=range(1, 13, 2)))
    record("RSFeatureAggregator[huge,hidden32,range(1,33,2)]",
           agg("facebook/sam-vit-huge", hidden_channels=32, out_channels=256, select_layers=range(1, 33, 2)))
    pagg = _exec_class(rel, "PseudoFeatureAggregator", ns)
    record("PseudoFeatureAggregator[256,512,256]", pagg(256, hidden_channels=512, out_channels=256))
    fpn = _exec_class(rel, "RSSimpleFPN", ns)
    record("RSSimpleFPN[256,[64,128,256,256],256,5,LN2d]",
           fpn(256, [64, 128, 256, 256], 256, 5, norm_cfg=dict(type="LN2d", requires_grad=True)),
           stub_prefixes=("lateral_convs.", "fpn_convs."))
    # statements of constructors whose bases are mmdet classes
    pe = _self_assign(rel, "RSPrompterAnchorMaskHead", "point_emb", SimpleNamespace(),
                      dict(nn=nn, in_channels=256, roi_feat_size=14, num_sincos=2, per_pointset_point=5))
    record("RSPrompterAnchorMaskHead.point_emb[256,14,sincos,5]", pe)
    self_q = SimpleNamespace(feat_channels=128, out_channels=256, num_classes=10)
    record("RSMask2FormerHead.point_emb[128,256,sincos,5]",
           _self_assign(rel, "RSMask2FormerHead", "point_emb", self_q, dict(nn=nn, num_sincos=2, per_pointset_point=5)))
    record("RSMask2FormerHead.cls_embed[128,10]", _self_assign(rel, "RSMask2FormerHead", "cls_embed", self_q, dict(nn=nn)))
    # stock heads used by the SAM-seg detectors (plain torch statements of their constructors)
    m2f = "mmdet/models/dense_heads/mask2former_head.py"
    self_m = SimpleNamespace(num_classes=10, num_queries=100, num_transformer_feat_level=3)
    record("Mask2FormerHead.mask_embed[256,256]",
           _self_assign(m2f, "Mask2FormerHead", "mask_embed", self_m, dict(nn=nn, feat_channels=256, out_channels=256)))
    record("Mask2FormerHead.cls_embed[256,10]",
           _self_assign(m2f, "Mask2FormerHead", "cls_embed", self_m, dict(nn=nn, feat_channels=256)))
    path = os.path.join(os.path.dirname(OUT), "reference_state_keys.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print("wrote", path, {k: len(v) for k, v in out.items()})


def main_necks():
    """tests/golden/reference_necks.pt: inputs, seeded state dicts and outputs of the reference's OWN forward() of
    RSFeatureAggregator, PseudoFeatureAggregator and RSSimpleFPN (mmdet/rsprompter/models.py), executed with torch only
    (BaseModule -> nn.Module; RSSimpleFPN's ConvModule / build_norm_layer through the stand-ins documented in
    main_state_keys: conv -> LN2d, no activation, as ConvModule(norm_cfg=LN2d, act_cfg=None) orders them).  Small
    channel counts keep the file small; the layer structure is the shipped one."""
    import einops
    from torch import nn
    rel = "mmdet/rsprompter/models.py"

    class BaseModule(nn.Module):
        def __init__(self, init_cfg=None):
            super().__init__()

    LayerNorm2d = _exec_class("mmpretrain/models/utils/norm.py", "LayerNorm2d", dict(torch=torch, nn=nn, F=F))
    ns = dict(torch=torch, nn=nn, F=F, einops=einops, BaseModule=BaseModule, LayerNorm2d=LayerNorm2d, List=list,
              Tensor=torch.Tensor)
    LN2d = _exec_class(rel, "LN2d", ns)

    def build_norm_layer(cfg, num_features, postfix=""):
        return "norm_layer" + str(postfix), LN2d(num_features)

    class ConvModule(nn.Module):
        def __init__(self, cin, cout, k, padding=0, conv_cfg=None, norm_cfg=None, act_cfg=None, inplace=False):
            super().__init__()
            assert norm_cfg is not None and act_cfg is None
            self.conv = nn.Conv2d(cin, cout, k, padding=padding, bias=False)
            self.add_module("norm_layer", build_norm_layer(norm_cfg, cout)[1])

        def forward(self, x):
            return self.norm_layer(self.conv(x))

    ns.update(build_norm_layer=build_norm_layer, ConvModule=ConvModule)
    g = torch.Generator().manual_seed(777)
    fx = {}

    def randomise(m):
        with torch.no_grad():
            for n, t in m.state_dict().items():
                if n.endswith("num_batches_tracked"):
                    continue
                if n.endswith("running_var"):
                    t.copy_(1.0 + torch.rand(t.shape, generator=g))
                elif t.dim() == 1:
                    t.copy_((1.0 if n.endswith("weight") else 0.0) + 0.2 * torch.randn(t.shape, generator=g))
                else:
                    t.copy_(torch.randn(t.shape, generator=g) * (1.5 / (t[0].numel() ** 0.5)))
        return m.eval()

    sel = range(1, 13, 2)
    agg = randomise(_exec_class(rel, "RSFeatureAggregator", ns)("sam_vit_base", hidden_channels=8, out_channels=16,
                                                                select_layers=sel))
    used = {i: torch.randn(1, 3, 4, 768, generator=g) for i in sel}
    hidden = [used.get(i, torch.zeros(1, 3, 4, 768)) for i in range(13)]
    with torch.no_grad():
        out = agg(hidden)
    fx["feature_aggregator"] = dict(state_dict={k: v.clone() for k, v in agg.state_dict().items()}, select_layers=list(sel),
                                    hidden={i: used[i] for i in sel}, out=out)
    pagg = randomise(_exec_class(rel, "PseudoFeatureAggregator", ns)(24, hidden_channels=16, out_channels=8))
    x = torch.randn(2, 24, 7, 9, generator=g)
    with torch.no_grad():
        out = pagg((x,))
    fx["pseudo_feature_aggregator"] = dict(state_dict={k: v.clone() for k, v in pagg.state_dict().items()}, x=x, out=out)
    fpn = randomise(_exec_class(rel, "RSSimpleFPN", ns)(16, [4, 8, 16, 16], 8, 5, norm_cfg=dict(type="LN2d", requires_grad=True)))
    x = torch.randn(2, 16, 6, 8, generator=g)
    with torch.no_grad():
        outs = fpn(x)
    fx["simple_fpn"] = dict(state_dict={k: v.clone() for k, v in fpn.state_dict().items()}, x=x, outs=list(outs))
    path = os.path.join(os.path.dirname(OUT), "reference_necks.pt")
    torch.save(fx, path)
    print("wrote", path, os.path.getsize(path), {k: list(v.keys()) for k, v in fx.items()})


CONFIG_NAMES = ("rsprompter_anchor-nwpu.py", "rsprompter_anchor-nwpu-peft-512.py", "rsprompter_query-nwpu.py",
                "rsprompter_query-nwpu-peft-512.py", "samdet-nwpu.py", "samseg-maskrcnn-nwpu.py",
                "samseg-mask2former-nwpu.py")


def main_configs():
    """tests/golden/reference_configs.pt: the reference's own configs/rsprompter/*-nwpu*.py resolved through their
    ``_base_`` chains by rsprompter_b200.registry.Config (mmengine's merge rules), per file the ``model`` dict and
    ``custom_imports`` as plain dicts (tuples and ranges kept).  Needs the built package."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    from rsprompter_b200.registry import Config

    def plain(o):
        if isinstance(o, dict):
            return {k: plain(v) for k, v in o.items()}
        if isinstance(o, (list, tuple)):
            return type(o)(plain(v) for v in o)
        return o

    fx = {}
    for name in CONFIG_NAMES:
        cfg = Config.fromfile(os.path.join(REF, "configs", "rsprompter", name)).to_dict()
        fx[name] = dict(model=plain(cfg["model"]), custom_imports=plain(cfg["custom_imports"]))
    path = os.path.join(os.path.dirname(OUT), "reference_configs.pt")
    torch.save(fx, path)
    print("wrote", path, os.path.getsize(path), sorted(fx))


if __name__ == "__main__":
    if not os.path.isdir(REF):
        sys.exit("/root/reference not mounted")
    if "maskrcnn" in sys.argv[1:]:
        main_maskrcnn()
    elif "configs" in sys.argv[1:]:
        main_configs()
    elif "state_keys" in sys.argv[1:]:
        main_state_keys()
    elif "necks" in sys.argv[1:]:
        main_necks()
    else:
        main()
