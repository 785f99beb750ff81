"""Padded-tensor interface to the B200 upstreams: the counterpart of ``s3prl.nn`` for this package.

Same public surface as the reference's new-style wrappers (s3prl/nn/upstream.py) — class names, constructor
arguments, properties, return conventions — resolved against ``s3prl_b200.hub`` instead of ``s3prl.hub``:

    model = S3PRLUpstream("hubert_base").cuda()
    all_hs, all_lens = model(wavs_padded, wavs_len)     # wavs_padded [B, Lmax] fp32 CUDA, wavs_len [B] long
    hs, hs_len = Featurizer(model).cuda()(all_hs, all_lens)

What has to agree with the reference bit for bit is the integer bookkeeping (SURVEY App. A.3-5), restated here from
its definition rather than from the reference's code:

* a layer with stride ``s`` is presented with ``ceil(Lmax / s)`` frames (``nn/upstream.py:208-214``): the conv stack
  yields ``floor((Lmax - 400) / 320) + 1``, so one frame is usually missing and the last one is repeated; a longer
  sequence is cut. Only an off-by-less-than-2x mismatch is legal (``:166-179``);
* ``h_len = floor((len - 1) / s) + 1`` per utterance, from the lengths the caller passed (``:223``), and the batch is
  cut to ``max(h_len)`` frames;
* inputs shorter than 0.05 s are zero-extended to 0.05 s first (``:196-206``).

``Featurizer`` (``:234-349``) and ``UpstreamDownstreamModel`` (``:352-384``) are the reference's reduction and
composition wrappers; the weighted layer sum runs in the fused CUDA kernel ``s3b_weighted_sum`` (+ its backward).
Parity: ``tests/test_host_cpu.py::test_nn_featurizer_matches_reference_logic`` checks these classes on the CPU
against what the reference's own returned (tests/golden/nn_upstream.pt); ``tests/test_api_gpu.py`` covers the device path.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import hub

SAMPLE_RATE = 16000
MIN_SAMPLES = int(0.05 * SAMPLE_RATE)  # MIN_SECOND of the reference


def _fit_frames(h: torch.Tensor, frames: int) -> torch.Tensor:
    """[B, T, D] -> [B, frames, D]: cut, or extend by repeating the last frame."""
    have = h.shape[1]
    if have == frames:
        return h
    small, large = sorted((have, frames))
    assert large // small == 1, f"{have}, {frames}"  # a 2x mismatch means a wrong stride, not a rounding frame
    if have > frames:
        return h[:, :frames]
    tail = h[:, have - 1 : have].expand(-1, frames - have, -1)
    return torch.cat([h, tail], dim=1)


class S3PRLUpstream(nn.Module):
    """``s3prl.nn.S3PRLUpstream``: ``forward(wavs [B, L(,1)], wavs_len [B]) -> (list of [B, T', D], list of [B])``."""

    @classmethod
    def available_names(cls, only_registered_ckpt: bool = False) -> List[str]:
        return hub.options()

    def __init__(
        self,
        name: str,
        path_or_url: str = None,
        refresh: bool = False,
        normalize: bool = False,
        extra_conf: dict = None,
        randomize: bool = False,
    ):
        super().__init__()
        kwargs = dict(extra_conf or {}, refresh=refresh)
        if path_or_url is not None:
            kwargs["ckpt"] = path_or_url
        if randomize:
            # The reference re-initialises the loaded model in place (nn/upstream.py:119-122). These upstreams own their
            # weights on the device, so fresh ones are fabricated instead — for the checkpoint's architecture when a
            # path is given — from a seed drawn off the default generator: reproducible under torch.manual_seed and
            # without reseeding the global RNG.
            kwargs["randomize_seed"] = int(torch.randint(0, 2**31 - 1, ()).item())
        self.upstream = hub.ENTRIES[name](**kwargs)
        self.normalize = normalize
        # Static facts. The reference finds them with a pseudo forward (nn/upstream.py:124-128); that would need a GPU
        # at construction time, and they follow from the architecture anyway.
        arch = getattr(self.upstream, "arch", None)
        if arch is not None:  # NL + 1 hidden states; feat_final + layers + prediction heads for the Distiller
            count, width = arch.num_outputs, self.upstream.hidden_size
        elif hasattr(self.upstream, "num_layers"):
            count, width = self.upstream.num_layers + 1, self.upstream.hidden_size
        else:  # fbank / mel / linear: one feature sequence
            count, width = 1, self.upstream.output_dim
        stride = self.upstream.get_downsample_rates("hidden_states")
        self._hidden_sizes = [width] * count
        self._downsample_rates = [stride] * count

    @property
    def num_layers(self) -> int:
        return len(self._hidden_sizes)

    @property
    def hidden_sizes(self) -> List[int]:
        return self._hidden_sizes

    @property
    def downsample_rates(self) -> List[int]:
        return self._downsample_rates

    def forward(self, wavs: torch.Tensor, wavs_len: torch.Tensor) -> Tuple[List[torch.Tensor], List[torch.Tensor]]:
        if wavs.dim() == 3:
            wavs = wavs.squeeze(-1)
        given_len = wavs_len
        shortfall = MIN_SAMPLES - int(given_len.max())
        if shortfall > 0:
            wavs = F.pad(wavs, (0, shortfall))
            wavs_len = wavs_len + shortfall
        utterances = [w[: int(n)] for w, n in zip(wavs, wavs_len)]
        layers = self.upstream(utterances)["hidden_states"]
        assert len(layers) == self.num_layers, f"{len(layers)}, {self.num_layers}"
        longest = int(wavs_len.max())
        all_hs, all_lens = [], []
        for h, stride in zip(layers, self._downsample_rates):
            h = _fit_frames(h, -(-longest // stride))
            frames = torch.div(given_len - 1, stride, rounding_mode="floor") + 1
            h = h[:, : int(frames.max())]
            all_hs.append(F.layer_norm(h, h.shape[-1:]) if self.normalize else h)
            all_lens.append(frames)
        return all_hs, all_lens


class Featurizer(nn.Module):
    """``s3prl.nn.Featurizer``: reduce the upstream's layers to one sequence. A single layer is passed through; several
    get a trainable softmax-weighted sum (``weights``, initial zeros) over ``layer_selections`` — all layers when None —
    optionally after ``F.layer_norm`` over the hidden dimension of every layer."""

    def __init__(self, upstream: S3PRLUpstream, layer_selections: Optional[Sequence[int]] = None, normalize: bool = False):
        super().__init__()
        widths, strides = set(upstream.hidden_sizes), set(upstream.downsample_rates)
        assert len(widths) == 1 and len(strides) == 1, "every layer must share one hidden size and one stride"
        self._output_size, self._downsample_rate = widths.pop(), strides.pop()
        self.normalize = normalize
        total = upstream.num_layers
        if total > 1:
            if layer_selections is None:
                layer_selections = range(total)
            assert len(layer_selections) <= total
            self.layer_selections = sorted(layer_selections)
            self.weights = nn.Parameter(torch.zeros(len(self.layer_selections)))

    @property
    def output_size(self) -> int:
        return self._output_size

    @property
    def downsample_rate(self) -> int:
        return self._downsample_rate

    def forward(self, all_hs: List[torch.Tensor], all_lens: List[torch.Tensor]) -> Tuple[torch.Tensor, torch.Tensor]:
        if len(all_hs) == 1:
            return all_hs[0], all_lens[0]
        from ..upstream import featurizer as fused  # the CUDA weighted sum (no CPU fallback)

        keep = set(self.layer_selections)
        picked = [(h, n) for i, (h, n) in enumerate(zip(all_hs, all_lens)) if i in keep]
        assert len(picked) > 1
        layers = [F.layer_norm(h, h.shape[-1:]) if self.normalize else h for h, _ in picked]
        return fused.weighted_sum(layers, F.softmax(self.weights, dim=-1)), picked[0][1]


class UpstreamDownstreamModel(nn.Module):
    """``s3prl.nn.UpstreamDownstreamModel``: upstream -> featurizer -> downstream(h, h_len, *args, **kwargs). The
    upstreams of this package are frozen (no autograd through the CUDA forward), so ``upstream_trainable=True`` is
    refused instead of training silently on constants."""

    def __init__(self, upstream: S3PRLUpstream, featurizer: Featurizer, downstream, upstream_trainable: bool = False):
        super().__init__()
        if upstream_trainable:
            raise NotImplementedError("s3prl_b200 upstreams are frozen: upstream_trainable=True is not supported")
        self.upstream, self.featurizer, self.downstream = upstream, featurizer, downstream
        self.upstream_trainable = False

    input_size = 1  # a waveform

    @property
    def downsample_rate(self) -> int:
        return self.featurizer.downsample_rate

    @property
    def output_size(self) -> int:
        return self.downstream.output_size

    def forward(self, wav, wav_len, *args, **kwargs):
        self.upstream.eval()
        with torch.no_grad():
            hidden, hidden_len = self.upstream(wav, wav_len)
        return self.downstream(*self.featurizer(hidden, hidden_len), *args, **kwargs)
