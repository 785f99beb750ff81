"""TEST INFRASTRUCTURE — run the reference itself (s3prl) on a fabricated checkpoint.

Used by oracle/make_golden.py (fixtures) and by bench.py's `--impl reference` / cpu_baseline legs. The reference is
the s3prl checkout beside this repository (../reference, or S3PRL_REFERENCE), else the copy installed under
oracle/_ref (see oracle/build_ref.py).
Nothing in the product package imports this module.
"""
from __future__ import annotations

import os
import sys
import tempfile
from pathlib import Path
from typing import Optional

import torch

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from s3prl_b200.upstream.configs import ARCHS  # noqa: E402
from s3prl_b200.upstream.convert import reference_model_cfg  # noqa: E402


def reference_root() -> Optional[Path]:
    from build_ref import REFERENCE, TARGET, exists

    for cand in (REFERENCE, TARGET):
        if exists(cand / "s3prl" / "upstream" / "hubert" / "expert.py"):
            return cand
    return None


def activate() -> Path:
    """Put the reference on sys.path (once) and register the import shims it needs in this image."""
    root = reference_root()
    if root is None:
        raise RuntimeError("the reference (s3prl) is neither checked out at ../reference (or S3PRL_REFERENCE) nor installed under oracle/_ref")
    if str(root) not in sys.path:
        sys.path.insert(0, str(root))
    from s3prl_b200.run_downstream import install_shims

    install_shims()
    return root


def reference_expert(name: str, sd):
    """The reference's UpstreamExpert (reference constructors, reference load_state_dict, reference forward and hooks)
    on the fabricated state dict `sd` of architecture `name`."""
    activate()
    cfg = ARCHS[name]
    model_cfg = dict(reference_model_cfg(cfg), dropout=0.1, attention_dropout=0.1, encoder_layerdrop=0.05)
    tmp = tempfile.NamedTemporaryFile(suffix=".pt", delete=False)
    tmp.close()
    try:
        if cfg.family == "distiller":
            from s3prl.upstream.distiller.expert import UpstreamExpert
            from s3prl.upstream.distiller.model import DistillerConfig, DistillerModel

            from s3prl_b200.upstream.convert import distiller_config

            dcfg = distiller_config(cfg)
            skeleton = DistillerModel(DistillerConfig(dcfg))
            full = skeleton.state_dict()
            full.update(sd)
            torch.save({"Config": {"distiller": dcfg}, "Distiller": full}, tmp.name)
        elif cfg.family == "hubert":
            from s3prl.upstream.hubert.expert import UpstreamExpert
            from s3prl.upstream.hubert.hubert_model import HubertConfig, HubertModel, HubertPretrainingConfig
            from s3prl.upstream.utils import merge_with_parent

            model_cfg.update(label_rate=50.0, final_dim=256, untie_final_proj=True)
            task_cfg = dict(normalize=cfg.normalize, sample_rate=16000, label_rate=50.0)
            symbols = [[str(i) for i in range(504)]]
            skeleton = HubertModel(
                merge_with_parent(HubertConfig, model_cfg), merge_with_parent(HubertPretrainingConfig, task_cfg), symbols
            )
            full = skeleton.state_dict()
            full.update(sd)
            torch.save(
                {"task_cfg": task_cfg, "model_cfg": model_cfg, "model_weight": full, "dictionaries_symbols": symbols},
                tmp.name,
            )
        elif cfg.family == "data2vec":
            from s3prl.upstream.data2vec.data2vec_model import Data2VecAudioConfig, Data2VecAudioModel
            from s3prl.upstream.data2vec.expert import UpstreamExpert
            from s3prl.upstream.utils import merge_with_parent

            task_cfg = dict(normalize=cfg.normalize, sample_rate=16000)
            skeleton = Data2VecAudioModel(merge_with_parent(Data2VecAudioConfig, model_cfg))
            skeleton.remove_pretraining_modules()  # what load_converted_model does before load_state_dict
            full = skeleton.state_dict()
            full.update(sd)
            full["_ema"] = {}  # deleted unconditionally by the reference loader (data2vec/convert.py:48-49)
            torch.save({"task_cfg": task_cfg, "model_cfg": model_cfg, "model_weight": full}, tmp.name)
        elif cfg.family == "wav2vec2":
            from s3prl.upstream.utils import merge_with_parent
            from s3prl.upstream.wav2vec2.expert import UpstreamExpert
            from s3prl.upstream.wav2vec2.wav2vec2_model import Wav2Vec2Config, Wav2Vec2Model

            model_cfg.update(quantize_targets=True, final_dim=768 if cfg.encoder_embed_dim == 1024 else 256)
            task_cfg = dict(normalize=cfg.normalize, sample_rate=16000)
            skeleton = Wav2Vec2Model(merge_with_parent(Wav2Vec2Config, model_cfg))
            full = skeleton.state_dict()
            full.update(sd)
            torch.save({"task_cfg": task_cfg, "model_cfg": model_cfg, "model_weight": full}, tmp.name)
        else:
            if name.startswith("unispeech_sat"):
                from s3prl.upstream.unispeech_sat.expert import UpstreamExpert
            else:
                from s3prl.upstream.wavlm.expert import UpstreamExpert
            from s3prl.upstream.wavlm.WavLM import WavLM, WavLMConfig

            skeleton = WavLM(WavLMConfig(model_cfg))
            full = skeleton.state_dict()
            full.update(sd)
            torch.save({"cfg": model_cfg, "model": full}, tmp.name)
        missing = set(sd) - set(skeleton.state_dict())
        assert not missing, f"fabricated keys unknown to the reference model: {sorted(missing)[:5]}"
        expert = UpstreamExpert(tmp.name)
    finally:
        os.unlink(tmp.name)
    expert.eval()
    return expert


def reference_featurizer(expert):
    """The reference's Featurizer over `expert` (s3prl/upstream/interfaces.py:134-272), CPU."""
    activate()
    from s3prl.upstream.interfaces import Featurizer

    return Featurizer(expert, "hidden_states", upstream_device="cpu")
