"""TEST INFRASTRUCTURE ONLY -- never imported by the product path.

Loader that imports the *unmodified* reference hot-path files straight from the
checkout ``$CMT_REFERENCE_ROOT`` names (read-only) so that their CPU/fp32 output can be dumped as
golden vectors (``oracle/make_golden.py``) and used to pin the restatement in
``oracle/cmt_oracle.py``.

The reference needs mmcv-full 1.6.2 / mmdet 2.28.2 / mmdet3d 1.0.0rc6 /
flash-attn 0.2.2 (reference ``Dockerfile:47-70``), none of which is installed
and none of which lives in the reference tree.  The handful of entry points
the seven hot-path files import are restated here from those packages'
published behaviour (SURVEY.md appendix B lists every name).  Because that
third-party arithmetic is a restatement, parity for it is "unpinned by a
reference test" -- the reference ships no tests at all (SURVEY.md section 4).

The reference tree is not part of this repository; nothing under ``tests -m gpu``,
``bench.py`` or ``__graft_entry__.smoke`` may import this module.
"""
from __future__ import annotations

import copy
import importlib
import os
import sys
import types

import torch
import torch.nn as nn

# a checkout of the original CMT-Cooperative-Perception project; unset: the tests that run it are skipped
REFERENCE_ROOT = os.environ.get("CMT_REFERENCE_ROOT", "")


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "projects", "mmdet3d_plugin"))


# --------------------------------------------------------------------------
# registries (mmcv.utils.Registry, build_from_cfg)
# --------------------------------------------------------------------------
class Registry:
    def __init__(self, name):
        self.name = name
        self.module_dict = {}

    def register_module(self, name=None, force=False, module=None):
        def deco(cls):
            self.module_dict[name or cls.__name__] = cls
            return cls
        if module is not None:
            return deco(module)
        return deco

    def get(self, key):
        return self.module_dict[key]

    def build(self, cfg, default_args=None):
        cfg = dict(cfg)
        if default_args:
            for k, v in default_args.items():
                cfg.setdefault(k, v)
        typ = cfg.pop("type")
        cls = self.module_dict[typ] if isinstance(typ, str) else typ
        return cls(**cfg)


class ConfigDict(dict):
    """mmcv.utils.ConfigDict: attribute access, nested dicts wrapped."""

    def __init__(self, *a, **kw):
        super().__init__()
        for k, v in dict(*a, **kw).items():
            self[k] = v

    @staticmethod
    def _wrap(v):
        if isinstance(v, dict) and not isinstance(v, ConfigDict):
            return ConfigDict(v)
        if isinstance(v, (list, tuple)):
            return type(v)(ConfigDict._wrap(x) for x in v)
        return v

    def __setitem__(self, k, v):
        super().__setitem__(k, ConfigDict._wrap(v))

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v

    def update(self, *a, **kw):
        for k, v in dict(*a, **kw).items():
            self[k] = v

    def __deepcopy__(self, memo):
        return ConfigDict({k: copy.deepcopy(v, memo) for k, v in self.items()})


ATTENTION = Registry("attention")
FEEDFORWARD_NETWORK = Registry("ffn")
TRANSFORMER_LAYER = Registry("transformer layer")
TRANSFORMER_LAYER_SEQUENCE = Registry("transformer layer sequence")
TRANSFORMER = Registry("transformer")
HEADS = Registry("heads")
BBOX_CODERS = Registry("bbox coders")


# --------------------------------------------------------------------------
# mmcv.runner
# --------------------------------------------------------------------------
class BaseModule(nn.Module):
    def __init__(self, init_cfg=None):
        super().__init__()
        self._is_init = False
        self.init_cfg = copy.deepcopy(init_cfg)

    def init_weights(self):
        for m in self.children():
            if hasattr(m, "init_weights"):
                m.init_weights()
        self._is_init = True


class Sequential(BaseModule, nn.Sequential):
    def __init__(self, *args, init_cfg=None):
        BaseModule.__init__(self, init_cfg)
        nn.Sequential.__init__(self, *args)


class ModuleList(BaseModule, nn.ModuleList):
    def __init__(self, modules=None, init_cfg=None):
        BaseModule.__init__(self, init_cfg)
        nn.ModuleList.__init__(self, modules)


def _identity_decorator_factory(*a, **kw):
    def deco(fn):
        return fn
    return deco


# --------------------------------------------------------------------------
# mmcv.cnn
# --------------------------------------------------------------------------
class ConvModule(nn.Module):
    """conv (bias off when a norm follows) -> bn -> relu; attrs .conv/.bn."""

    def __init__(self, in_channels, out_channels, kernel_size, padding=0,
                 conv_cfg=None, norm_cfg=None, **kw):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size,
                              padding=padding, bias=norm_cfg is None)
        self.bn = nn.BatchNorm2d(out_channels) if norm_cfg is not None else None
        self.activate = nn.ReLU(inplace=True)

    def forward(self, x):
        x = self.conv(x)
        if self.bn is not None:
            x = self.bn(x)
        return self.activate(x)


def build_norm_layer(cfg, num_features, postfix=""):
    assert cfg["type"] == "LN"
    return "ln" + str(postfix), nn.LayerNorm(num_features, eps=cfg.get("eps", 1e-5))


def xavier_init(module, gain=1, bias=0, distribution="normal"):
    if hasattr(module, "weight") and module.weight is not None:
        if distribution == "uniform":
            nn.init.xavier_uniform_(module.weight, gain=gain)
        else:
            nn.init.xavier_normal_(module.weight, gain=gain)
    if hasattr(module, "bias") and module.bias is not None:
        nn.init.constant_(module.bias, bias)


def build_dropout(cfg, default_args=None):
    return nn.Dropout(cfg.get("drop_prob", 0.0))


class FFN(BaseModule):
    """mmcv.cnn.bricks.transformer.FFN (mmcv-full 1.6.2)."""

    def __init__(self, embed_dims=256, feedforward_channels=1024, num_fcs=2,
                 act_cfg=dict(type="ReLU", inplace=True), ffn_drop=0.0,
                 dropout_layer=None, add_identity=True, init_cfg=None, **kw):
        super().__init__(init_cfg)
        self.embed_dims = embed_dims
        layers = []
        in_channels = embed_dims
        for _ in range(num_fcs - 1):
            layers.append(Sequential(nn.Linear(in_channels, feedforward_channels),
                                     nn.ReLU(inplace=True), nn.Dropout(ffn_drop)))
            in_channels = feedforward_channels
        layers.append(nn.Linear(feedforward_channels, embed_dims))
        layers.append(nn.Dropout(ffn_drop))
        self.layers = Sequential(*layers)
        self.dropout_layer = build_dropout(dropout_layer) if dropout_layer else nn.Identity()
        self.add_identity = add_identity

    def forward(self, x, identity=None):
        out = self.layers(x)
        if not self.add_identity:
            return self.dropout_layer(out)
        if identity is None:
            identity = x
        return identity + self.dropout_layer(out)


FEEDFORWARD_NETWORK.register_module(name="FFN")(FFN)


class BaseTransformerLayer(BaseModule):
    """mmcv.cnn.bricks.transformer.BaseTransformerLayer (mmcv-full 1.6.2)."""

    def __init__(self, attn_cfgs=None,
                 ffn_cfgs=dict(type="FFN", embed_dims=256, feedforward_channels=1024,
                               num_fcs=2, ffn_drop=0.0, act_cfg=dict(type="ReLU", inplace=True)),
                 operation_order=None, norm_cfg=dict(type="LN"), init_cfg=None,
                 batch_first=False, **kwargs):
        deprecated = dict(feedforward_channels="feedforward_channels",
                          ffn_dropout="ffn_drop", ffn_num_fcs="num_fcs")
        ffn_cfgs = copy.deepcopy(dict(ffn_cfgs))
        for ori, new in deprecated.items():
            if ori in kwargs:
                ffn_cfgs[new] = kwargs[ori]
        super().__init__(init_cfg)
        self.batch_first = batch_first
        num_attn = operation_order.count("self_attn") + operation_order.count("cross_attn")
        if isinstance(attn_cfgs, dict):
            attn_cfgs = [copy.deepcopy(attn_cfgs) for _ in range(num_attn)]
        self.num_attn = num_attn
        self.operation_order = operation_order
        self.norm_cfg = norm_cfg
        self.pre_norm = operation_order[0] == "norm"
        self.attentions = ModuleList()
        index = 0
        for name in operation_order:
            if name in ("self_attn", "cross_attn"):
                cfg = copy.deepcopy(dict(attn_cfgs[index]))
                cfg["batch_first"] = self.batch_first
                self.attentions.append(ATTENTION.build(cfg))
                index += 1
        self.embed_dims = self.attentions[0].embed_dims
        self.ffns = ModuleList()
        num_ffns = operation_order.count("ffn")
        if isinstance(ffn_cfgs, dict):
            ffn_cfgs = [copy.deepcopy(ffn_cfgs) for _ in range(num_ffns)]
        for i in range(num_ffns):
            cfg = dict(ffn_cfgs[i])
            cfg.setdefault("embed_dims", self.embed_dims)
            self.ffns.append(FEEDFORWARD_NETWORK.build(cfg))
        self.norms = ModuleList()
        for _ in range(operation_order.count("norm")):
            self.norms.append(build_norm_layer(norm_cfg, self.embed_dims)[1])

    def forward(self, query, key=None, value=None, query_pos=None, key_pos=None,
                attn_masks=None, query_key_padding_mask=None, key_padding_mask=None, **kwargs):
        norm_index = attn_index = ffn_index = 0
        identity = query
        if attn_masks is None:
            attn_masks = [None for _ in range(self.num_attn)]
        elif isinstance(attn_masks, torch.Tensor):
            attn_masks = [copy.deepcopy(attn_masks) for _ in range(self.num_attn)]
        for layer in self.operation_order:
            if layer == "self_attn":
                temp_key = temp_value = query
                query = self.attentions[attn_index](
                    query, temp_key, temp_value, identity if self.pre_norm else None,
                    query_pos=query_pos, key_pos=query_pos, attn_mask=attn_masks[attn_index],
                    key_padding_mask=query_key_padding_mask, **kwargs)
                attn_index += 1
                identity = query
            elif layer == "norm":
                query = self.norms[norm_index](query)
                norm_index += 1
            elif layer == "cross_attn":
                query = self.attentions[attn_index](
                    query, key, value, identity if self.pre_norm else None,
                    query_pos=query_pos, key_pos=key_pos, attn_mask=attn_masks[attn_index],
                    key_padding_mask=key_padding_mask, **kwargs)
                attn_index += 1
                identity = query
            elif layer == "ffn":
                query = self.ffns[ffn_index](query, identity if self.pre_norm else None)
                ffn_index += 1
        return query


class TransformerLayerSequence(BaseModule):
    def __init__(self, transformerlayers=None, num_layers=None, init_cfg=None):
        super().__init__(init_cfg)
        if isinstance(transformerlayers, dict):
            transformerlayers = [copy.deepcopy(transformerlayers) for _ in range(num_layers)]
        self.num_layers = num_layers
        self.layers = ModuleList()
        for i in range(num_layers):
            self.layers.append(TRANSFORMER_LAYER.build(transformerlayers[i]))
        self.embed_dims = self.layers[0].embed_dims
        self.pre_norm = self.layers[0].pre_norm

    def forward(self, query, key, value, query_pos=None, key_pos=None, attn_masks=None,
                query_key_padding_mask=None, key_padding_mask=None, **kwargs):
        for layer in self.layers:
            query = layer(query, key, value, query_pos=query_pos, key_pos=key_pos,
                          attn_masks=attn_masks, query_key_padding_mask=query_key_padding_mask,
                          key_padding_mask=key_padding_mask, **kwargs)
        return query


def build_transformer_layer_sequence(cfg, default_args=None):
    return TRANSFORMER_LAYER_SEQUENCE.build(cfg, default_args)


# --------------------------------------------------------------------------
# mmdet
# --------------------------------------------------------------------------
def inverse_sigmoid(x, eps=1e-5):
    """mmdet.models.utils.transformer.inverse_sigmoid (mmdet 2.28.2)."""
    x = x.clamp(min=0, max=1)
    x1 = x.clamp(min=eps)
    x2 = (1 - x).clamp(min=eps)
    return torch.log(x1 / x2)


def multi_apply(func, *args, **kwargs):
    from functools import partial
    pfunc = partial(func, **kwargs) if kwargs else func
    map_results = map(pfunc, *args)
    return tuple(map(list, zip(*map_results)))


def _dummy(*a, **kw):
    return None


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


_INSTALLED = False


def install_stubs():
    """Seed sys.modules with the stub packages + namespace packages that point
    into REFERENCE_ROOT (skipping its heavy __init__.py files)."""
    global _INSTALLED
    if _INSTALLED:
        return
    if not reference_available():
        raise RuntimeError(f"reference tree not found at CMT_REFERENCE_ROOT={REFERENCE_ROOT!r}")
    plug = os.path.join(REFERENCE_ROOT, "projects", "mmdet3d_plugin")

    def ns(name, path):
        m = types.ModuleType(name)
        m.__path__ = [path]
        sys.modules[name] = m

    ns("projects", os.path.join(REFERENCE_ROOT, "projects"))
    ns("projects.mmdet3d_plugin", plug)
    ns("projects.mmdet3d_plugin.models", os.path.join(plug, "models"))
    ns("projects.mmdet3d_plugin.models.utils", os.path.join(plug, "models", "utils"))
    ns("projects.mmdet3d_plugin.models.dense_heads", os.path.join(plug, "models", "dense_heads"))
    ns("projects.mmdet3d_plugin.core", os.path.join(plug, "core"))
    ns("projects.mmdet3d_plugin.core.bbox", os.path.join(plug, "core", "bbox"))
    ns("projects.mmdet3d_plugin.core.bbox.coders", os.path.join(plug, "core", "bbox", "coders"))

    if "turtle" not in sys.modules:
        _mod("turtle", down=_dummy)

    _mod("mmcv")
    _mod("mmcv.cnn", ConvModule=ConvModule, build_norm_layer=build_norm_layer,
         xavier_init=xavier_init, build_conv_layer=_dummy, constant_init=_dummy,
         kaiming_init=_dummy, build_activation_layer=_dummy)
    _mod("mmcv.cnn.bricks")
    _mod("mmcv.cnn.bricks.transformer", FFN=FFN, BaseTransformerLayer=BaseTransformerLayer,
         TransformerLayerSequence=TransformerLayerSequence,
         build_transformer_layer_sequence=build_transformer_layer_sequence,
         build_positional_encoding=_dummy)
    _mod("mmcv.cnn.bricks.drop", build_dropout=build_dropout)
    _mod("mmcv.cnn.bricks.registry", ATTENTION=ATTENTION, TRANSFORMER_LAYER=TRANSFORMER_LAYER,
         TRANSFORMER_LAYER_SEQUENCE=TRANSFORMER_LAYER_SEQUENCE)
    _mod("mmcv.runner", BaseModule=BaseModule, force_fp32=_identity_decorator_factory,
         auto_fp16=_identity_decorator_factory)
    _mod("mmcv.runner.base_module", BaseModule=BaseModule)
    _mod("mmcv.utils", ConfigDict=ConfigDict, deprecated_api_warning=_identity_decorator_factory,
         build_from_cfg=_dummy, to_2tuple=_dummy)

    _mod("mmdet")
    _mod("mmdet.core", multi_apply=multi_apply, build_bbox_coder=lambda cfg: BBOX_CODERS.build(cfg),
         bbox_cxcywh_to_xyxy=_dummy, bbox_xyxy_to_cxcywh=_dummy, build_assigner=_dummy,
         build_sampler=_dummy, reduce_mean=_dummy)
    _mod("mmdet.core.bbox", BaseBBoxCoder=object)
    _mod("mmdet.core.bbox.builder", BBOX_CODERS=BBOX_CODERS)
    _mod("mmdet.models", HEADS=HEADS, build_loss=_dummy)
    _mod("mmdet.models.utils", build_transformer=lambda cfg: TRANSFORMER.build(cfg),
         NormedLinear=_dummy, inverse_sigmoid=inverse_sigmoid)
    _mod("mmdet.models.utils.builder", TRANSFORMER=TRANSFORMER)
    _mod("mmdet.models.utils.transformer", inverse_sigmoid=inverse_sigmoid)
    _mod("mmdet.models.dense_heads")
    _mod("mmdet.models.dense_heads.anchor_free_head", AnchorFreeHead=object)

    builder = types.SimpleNamespace(build_head=lambda cfg: HEADS.build(cfg))
    _mod("mmdet3d")
    _mod("mmdet3d.core", limit_period=_dummy, circle_nms=_dummy, draw_heatmap_gaussian=_dummy,
         gaussian_radius=_dummy, xywhr2xyxyr=_dummy)
    _mod("mmdet3d.models", builder=builder)
    _mod("mmdet3d.models.utils")
    _mod("mmdet3d.models.utils.clip_sigmoid", clip_sigmoid=_dummy)

    # flash-attn 0.2.2 entry points: only imported, never called by the oracle
    # (the north star's oracle is the nn.MultiheadAttention path).
    if "flash_attn" in sys.modules:
        for k in [k for k in sys.modules if k == "flash_attn" or k.startswith("flash_attn.")]:
            del sys.modules[k]
    _mod("flash_attn")
    _mod("flash_attn.flash_attn_interface", flash_attn_unpadded_kvpacked_func=_dummy)
    _mod("flash_attn.bert_padding", unpad_input=_dummy, pad_input=_dummy, index_first_axis=_dummy)
    _INSTALLED = True


def load_reference():
    """Import the reference hot-path modules verbatim.  Returns a namespace."""
    install_stubs()
    pre = "projects.mmdet3d_plugin."
    util = importlib.import_module(pre + "core.bbox.util")
    coder = importlib.import_module(pre + "core.bbox.coders.multi_task_bbox_coder")
    attention = importlib.import_module(pre + "models.utils.attention")
    petr = importlib.import_module(pre + "models.utils.petr_transformer")
    cmt_tr = importlib.import_module(pre + "models.utils.cmt_transformer")
    head = importlib.import_module(pre + "models.dense_heads.cmt_head")
    head_coop = importlib.import_module(pre + "models.dense_heads.cmt_head_coop")
    # configs name mmcv's own MultiheadAttention for self-attention; its code is
    # identical to the reference's PETRMultiheadAttention (petr_transformer.py:37-177).
    ATTENTION.module_dict.setdefault("MultiheadAttention", petr.PETRMultiheadAttention)
    return types.SimpleNamespace(util=util, coder=coder, attention=attention, petr=petr,
                                 cmt_transformer=cmt_tr, head=head, head_coop=head_coop,
                                 HEADS=HEADS, ConfigDict=ConfigDict)


def build_reference_head(head_type: str, cfg: dict):
    """Instantiate a reference head class from a (reference-config-shaped) dict,
    with cross-attention switched to the nn.MultiheadAttention oracle path."""
    ref = load_reference()
    cfg = ConfigDict(copy.deepcopy(cfg))
    for a in cfg["transformer"]["decoder"]["transformerlayers"]["attn_cfgs"]:
        if a["type"] == "PETRMultiheadFlashAttention":
            a["type"] = "PETRMultiheadAttention"
    cfg.pop("type", None)
    head = ref.HEADS.get(head_type)(**cfg)
    head.eval()
    return head
