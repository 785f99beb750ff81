"""TEST INFRASTRUCTURE — generates tests/golden/* by EXECUTING THE REFERENCE (s3prl, see oracle/ref_runtime.py).

Only where an s3prl checkout is at hand; the tests read the stored results and never need the reference:

    python oracle/make_golden.py [--only hubert_base]     # reference at ../reference, or S3PRL_REFERENCE=/path/to/s3prl

For every architecture it
  1. fabricates the deterministic checkpoint (s3prl_b200.upstream.weights.fabricate_state_dict, seed 0),
  2. writes it in the reference's converted-checkpoint format and loads it with the reference's own
     ``UpstreamExpert`` (s3prl/upstream/{hubert,wav2vec2,wavlm}/expert.py) — reference constructors, reference
     ``load_state_dict``, reference forward and hooks,
  3. runs ``expert(wavs)`` on seeded waveforms (equal-length and ragged batches, incl. a 0.05 s utterance),
  4. stores a strided sub-sample of every hidden state plus per-layer norms (fixtures stay < ~1 MB each).
Integer rules (frame masks, WavLM buckets, Featurizer lengths) are recorded exhaustively.
"""
from __future__ import annotations

import argparse
import os
import sys
import tempfile
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))
GOLDEN = ROOT / "tests" / "golden"

from s3prl_b200.upstream.configs import ARCHS, CONV_LAYERS  # noqa: E402
from s3prl_b200.upstream.weights import fabricate_state_dict  # noqa: E402

# (architecture, list of waveform lengths per case, channel stride of the stored sub-sample)
CASES = {
    "hubert_base": ([[16000, 12345, 800], [8000, 8000]], 7),
    "wav2vec2_base_960": ([[16000, 12345, 800], [8000, 8000]], 7),
    "wavlm_base_plus": ([[16000, 12345, 800], [8000, 8000]], 7),
    "wav2vec2_large_ll60k": ([[12000, 7001]], 13),
    "wav2vec2_large_960": ([[12000, 7001]], 13),
    "wavlm_large": ([[12000, 7001]], 13),
    "hubert_large_ll60k": ([[12000, 7001]], 13),
    "unispeech_sat_base_plus": ([[16000, 12345, 800], [8000, 8000]], 7),
    "unispeech_sat_large": ([[12000, 7001]], 13),
    "distilhubert_base": ([[16000, 12345, 3200], [8000, 8000]], 7),
    "data2vec_base_960": ([[16000, 12345, 800], [8000, 8000]], 7),
    "data2vec_large_ll60k": ([[12000, 7001]], 13),
}


# BASELINE.json sizes (SURVEY §8: C3 = wav2vec2_large 20 s -> T = 999, C4 = wavlm_base_plus 10 s -> T = 499) on a batch
# the CPU reference can afford: fixture name -> (architecture, cases, channel stride, time stride of the sub-sample)
FULL_SIZE = {
    "c3_wav2vec2_large_960": ("wav2vec2_large_960", [[320000, 320000]], 13, 8),
    "c3_wav2vec2_large_ll60k": ("wav2vec2_large_ll60k", [[320000, 271828]], 13, 8),
    "c4_wavlm_base_plus": ("wavlm_base_plus", [[160000, 160000], [160000, 100003]], 7, 4),
}


def seeded_wavs(lens, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(n, generator=g) for n in lens]


from ref_runtime import activate, reference_expert  # noqa: E402  (the reference itself on a fabricated checkpoint)


def make_model_fixture(name: str, fixture: str = None):
    if fixture is None:
        (lens_cases, cstride), tstride, fixture = CASES[name], 1, name
    else:
        name, lens_cases, cstride, tstride = FULL_SIZE[fixture]
    sd = fabricate_state_dict(ARCHS[name], seed=0)
    expert = reference_expert(name, sd)
    out = {"arch": name, "weight_seed": 0, "channel_stride": cstride, "time_stride": tstride, "cases": []}
    for ci, lens in enumerate(lens_cases):
        wavs = seeded_wavs(lens, seed=100 + ci)
        with torch.no_grad():
            res = expert(wavs)
        hs = [h.float() for h in res["hidden_states"]]
        out["cases"].append(
            {
                "lens": lens,
                "wav_seed": 100 + ci,
                "shape": tuple(hs[0].shape),
                "num_hidden": len(hs),
                # time sub-sample anchored at the LAST frame so that the end of the sequence is always covered
                "sub": torch.stack([h[:, (h.shape[1] - 1) % tstride :: tstride, ::cstride].contiguous() for h in hs]),
                "norms": torch.tensor([h.double().norm().item() for h in hs]),
                "abs_max": torch.tensor([h.abs().max().item() for h in hs]),
            }
        )
        print(f"{fixture} case {ci}: lens={lens} -> {len(hs)} x {tuple(hs[0].shape)}", flush=True)
    torch.save(out, GOLDEN / f"{fixture}.pt")


def make_integer_fixture():
    """Frame-mask rules, WavLM buckets and length rules straight from the reference code."""
    from s3prl.upstream.hubert.hubert_model import HubertModel
    from s3prl.upstream.interfaces import Featurizer  # noqa: F401  (rule restated below, see tolist)
    from s3prl.upstream.wav2vec2.wav2vec2_model import Wav2Vec2Config, Wav2Vec2Model
    from s3prl.upstream.wavlm.modules import MultiheadAttention as WavLMAttention

    g = torch.Generator().manual_seed(7)
    batches, short_batches = [], []
    w2v = Wav2Vec2Model(Wav2Vec2Config(encoder_layers=1, quantize_targets=False))
    # 60 random batches, then batches holding utterances SHORTER than the 400-sample receptive field (the wav2vec2
    # rule's unclamped floor arithmetic goes to 0 / negative there and the mask index wraps around)
    short = [[16000, 50], [16000, 5], [8000, 399, 55, 56, 57, 1], [16000, 400, 401, 719, 720, 721], [4000, 10, 9, 14, 15, 16]]
    g2 = torch.Generator().manual_seed(11)
    for _ in range(12):
        short.append([int(torch.randint(2000, 40000, (1,), generator=g2))] + torch.randint(1, 400, (4,), generator=g2).tolist())
    for it in range(60 + len(short)):
        if it >= 60:
            lens = short[it - 60]
            B = len(lens)
        else:
            B = int(torch.randint(1, 7, (1,), generator=g))
            lens = torch.randint(400, 170000, (B,), generator=g).tolist()
            if torch.rand(1, generator=g).item() < 0.3:
                lens = [max(lens)] * B  # no padding at all
        Lmax = max(lens)
        pad = ~torch.lt(torch.arange(Lmax).unsqueeze(0), torch.tensor(lens).unsqueeze(1))
        n = Lmax
        for _d, k, s in CONV_LAYERS:
            n = (n - k) // s + 1
        T = n
        feats = torch.zeros(B, T, 1)
        hub_mask = HubertModel.forward_padding_mask(None, feats, pad)
        # wav2vec2 rule: replay the statements of Wav2Vec2Model.forward (wav2vec2_model.py:2652-2671)
        if pad.any():
            input_lengths = (1 - pad.long()).sum(-1)
            output_lengths = w2v._get_feat_extract_output_lengths(input_lengths)
            m = torch.zeros((B, T), dtype=torch.float32)
            m[(torch.arange(B), output_lengths - 1)] = 1
            w2v_mask = (1 - m.flip([-1]).cumsum(-1).flip([-1])).bool()
            w2v_valid = [int((~r).sum()) for r in w2v_mask]
        else:
            w2v_valid = [T] * B
        (batches if it < 60 else short_batches).append(
            {
                "lens": lens,
                "T": T,
                "hubert_valid": [int((~r).sum()) for r in hub_mask],
                "hubert_prefix": bool(all((r[: int((~r).sum())] == False).all() for r in hub_mask)),  # noqa: E712
                "wav2vec2_valid": w2v_valid,
                "featurizer_len": [round(n_ / 320) for n_ in lens],
                "s3prl_upstream_len": [(n_ - 1) // 320 + 1 for n_ in lens],
            }
        )
    att = WavLMAttention(768, 12, has_relative_attention_bias=True, num_buckets=320, max_distance=800)
    rel = torch.arange(-2100, 2101, dtype=torch.long)
    buckets = att._relative_positions_bucket(rel.unsqueeze(0), bidirectional=True)[0]
    torch.save({"batches": batches, "short_batches": short_batches, "wavlm_rel": rel, "wavlm_bucket": buckets},
               GOLDEN / "integer_rules.pt")
    print(f"integer rules: {len(batches)} + {len(short_batches)} batches, {len(rel)} relative positions")


def make_fbank_fixture():
    """s3prl.upstream.baseline fbank (config 1: 4 x 1 s, seed 0) + a ragged batch."""
    from s3prl.upstream.baseline.hubconf import fbank

    expert = fbank()
    expert.eval()
    out = {"cases": []}
    torch.manual_seed(0)
    c1 = [torch.randn(16000) for _ in range(4)]  # BASELINE.md C1
    for name, wavs in (("c1_4x1s_seed0", c1), ("ragged", seeded_wavs([16000, 9999, 4000, 480], 321))):
        with torch.no_grad():
            hs = expert(wavs)["hidden_states"][0]
        out["cases"].append({"name": name, "lens": [len(w) for w in wavs], "out": hs.float().clone()})
        print(f"fbank {name}: {tuple(hs.shape)}")
    torch.save(out, GOLDEN / "fbank.pt")


def make_spectrogram_fixture():
    """s3prl.upstream.baseline mel / linear entries (torch.stft path) on equal-length and ragged batches."""
    from s3prl.upstream.baseline.hubconf import linear, mel

    out = {"cases": []}
    for name, factory in (("mel", mel), ("linear", linear)):
        expert = factory()
        expert.eval()
        torch.manual_seed(0)
        c1 = [torch.randn(16000) for _ in range(4)]
        ragged = seeded_wavs([16000, 9999, 4000, 1234], 654)
        ragged[1][-37:] = 0.0  # trailing exact zeros exercise the non-zero trimming rule
        for cname, wavs in (("4x1s_seed0", c1), ("ragged", ragged)):
            with torch.no_grad():
                hs = expert(wavs)["hidden_states"][0]
            out["cases"].append({"feat": name, "name": cname, "lens": [len(w) for w in wavs], "out": hs.float().clone()})
            print(f"{name} {cname}: {tuple(hs.shape)}")
    torch.save(out, GOLDEN / "spectrogram.pt")


class FakeUpstream:
    """The static facts s3prl.nn.Featurizer reads from an upstream: n layers of width 16 at stride 320."""

    def __init__(self, n):
        self.num_layers, self.hidden_sizes, self.downsample_rates = n, [16] * n, [320] * n


def fake_s3prl_upstream(cls):
    """An S3PRLUpstream (the reference's class or s3prl_b200.nn's) around a fake three-layer upstream with the conv
    stack's frame rule, built without the constructor (which would load a model)."""

    class Fake(torch.nn.Module):
        def forward(self, wavs):
            frames = max((len(w) - 400) // 320 + 1 if len(w) >= 400 else 0 for w in wavs)
            base = torch.arange(len(wavs) * frames * 2, dtype=torch.float32).view(len(wavs), frames, 2)
            return {"hidden_states": [base + k for k in range(3)]}

    obj = cls.__new__(cls)
    torch.nn.Module.__init__(obj)
    obj.upstream, obj.normalize = Fake(), False
    obj._hidden_sizes, obj._downsample_rates = [2] * 3, [320] * 3
    obj._num_layers = 3  # read by the reference's num_layers property
    return obj


# the cases of tests/test_host_cpu.py that nn_upstream.pt answers
FEATURIZER_CASES = ((None, False), ([4, 0, 2], False), (None, True), ([1, 3], True))
S3PRL_UPSTREAM_LENS = ([16000, 9000, 3200], [16001, 480], [700, 500], [32000, 31999], [1281, 1280, 1279], [48000])
S3PRL_UPSTREAM_REFUSED_LENS = ([960, 961], [1000, 900])  # 2 frames from the conv rule where ceil(L / 320) = 4


def make_nn_fixture():
    """The reference's s3prl.nn wrappers (s3prl/nn/upstream.py:166-384) on the CPU: Featurizer outputs and weight
    gradients (layer selection, normalize), UpstreamDownstreamModel plumbing, S3PRLUpstream length bookkeeping on a
    fake upstream, and which inputs the latter refuses."""
    from s3prl.nn.upstream import Featurizer, S3PRLUpstream, UpstreamDownstreamModel

    g = torch.Generator().manual_seed(0)
    hs = [torch.randn(3, 7, 16, generator=g) for _ in range(5)]
    lens = [torch.tensor([7, 5, 2])] * 5
    featurizer = []
    for sel, norm in FEATURIZER_CASES:
        f = Featurizer(FakeUpstream(5), sel, norm)
        w = torch.randn(len(f.weights), generator=g)
        with torch.no_grad():
            f.weights.copy_(w)
        h, h_len = f(hs, lens)
        h.square().sum().backward()
        featurizer.append({"layer_selections": list(f.layer_selections), "weights": w, "hs": h.detach(), "hs_len": h_len,
                           "grad": f.weights.grad.clone(), "output_size": f.output_size,
                           "downsample_rate": f.downsample_rate})
    single = Featurizer(FakeUpstream(1))

    class Up(torch.nn.Module):
        num_layers, hidden_sizes, downsample_rates = 5, [16] * 5, [320] * 5

        def forward(self, wav, wav_len):
            return hs, lens

    class Down(torch.nn.Module):
        output_size = 3

        def forward(self, h, h_len, scale=1.0):
            return h[..., :3] * scale, h_len

    udm = UpstreamDownstreamModel(Up(), Featurizer(Up()), Down())
    udm_hs, udm_len = udm(None, None, scale=2.0)

    ref, cases = fake_s3prl_upstream(S3PRLUpstream), []
    for case_lens in S3PRL_UPSTREAM_LENS:
        for normalize in (False, True):
            ref.normalize = normalize
            wavs = torch.zeros(len(case_lens), max(case_lens) + 37)  # the padded tensor may be wider than the longest
            for i, n in enumerate(case_lens):
                wavs[i, :n] = torch.randn(n, generator=g)
            a_hs, a_len = ref(wavs, torch.tensor(case_lens))
            b_hs, b_len = ref(wavs.unsqueeze(-1), torch.tensor(case_lens))
            assert all(torch.equal(x, y) for x, y in zip(a_hs + a_len, b_hs + b_len))
            cases.append({"lens": case_lens, "normalize": normalize, "hs": a_hs, "hs_len": a_len})
    refused = []
    for case_lens in S3PRL_UPSTREAM_REFUSED_LENS:
        try:
            ref(torch.zeros(len(case_lens), max(case_lens)), torch.tensor(case_lens))
            refused.append(False)
        except AssertionError:
            refused.append(True)
    torch.save({"inputs": {"hs": hs, "lens": lens}, "featurizer": featurizer,
                "single_layer_has_weights": hasattr(single, "weights"),
                "udm": {"hs": udm_hs.detach(), "hs_len": udm_len, "input_size": udm.input_size,
                        "downsample_rate": udm.downsample_rate, "output_size": udm.output_size},
                "s3prl_upstream": cases, "s3prl_upstream_refused": refused},
               GOLDEN / "nn_upstream.pt")
    print(f"nn: {len(featurizer)} featurizer cases, {len(cases)} S3PRLUpstream cases, refused {refused}")


def make_hub_fixture():
    """The entry names of the reference's s3prl.hub (s3prl/hub.py:40-54 options()), which the Runner resolves with
    getattr(hub, name) and s3prl_b200.hub.install overrides."""
    import json

    import s3prl.hub as hub

    names = sorted(hub.options())
    (GOLDEN / "hub_entries.json").write_text(json.dumps(names, indent=0) + "\n")
    print(f"hub: {len(names)} entries")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None)
    args = ap.parse_args()
    GOLDEN.mkdir(parents=True, exist_ok=True)
    activate()
    torch.manual_seed(0)
    if args.only in (None, "integer"):
        make_integer_fixture()
    if args.only in (None, "nn"):
        make_nn_fixture()
    if args.only in (None, "hub"):
        make_hub_fixture()
    if args.only in (None, "fbank"):
        make_fbank_fixture()
    if args.only in (None, "spectrogram"):
        make_spectrogram_fixture()
    for name in CASES:
        if args.only in (None, name):
            make_model_fixture(name)
    for fixture in FULL_SIZE:
        if args.only in (None, fixture, "full_size"):
            make_model_fixture(None, fixture)


if __name__ == "__main__":
    main()
