"""CPU tests of the host-side logic: C-ABI symbol export, loud failure without a GPU, hub injection into s3prl.hub,
the s3prl.nn mirrors against the reference's results (tests/golden), utterance sharding + gather over gloo with
world_size 2."""
import os
import re
import sys
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]
GOLDEN = ROOT / "tests" / "golden"


def test_cabi_exports_every_declared_symbol(s3b_lib):
    from s3prl_b200 import lib

    header = (ROOT / "include" / "s3prl_b200.h").read_text()
    declared = set(re.findall(r"\b(s3b_[a-z0-9_]+)\s*\(", header))
    declared -= {"s3b_model", "s3b_config"}
    assert declared, "no declarations parsed"
    for sym in sorted(declared):
        assert hasattr(s3b_lib, sym), f"{sym} declared in include/s3prl_b200.h but not exported"
    assert declared == set(lib.EXPORTED_SYMBOLS)
    assert s3b_lib.s3b_version() >= 100
    assert s3b_lib.s3b_fbank_num_frames(16000) == 98


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the GPU-less behaviour")
def test_no_cpu_fallback(s3b_lib):
    from s3prl_b200 import lib
    from s3prl_b200.hub import fbank
    from s3prl_b200.upstream.expert import UpstreamExpert

    assert s3b_lib.s3b_device_count() == 0
    expert = UpstreamExpert(name="hubert_base", state_dict={})
    with pytest.raises(lib.S3BError):
        expert([torch.randn(16000)])
    with pytest.raises(lib.S3BError):
        fbank()([torch.randn(16000)])


def test_model_create_validates_the_architecture(s3b_lib):
    """s3b_model_create needs no device: unsupported shapes are refused with a message instead of failing later."""
    import ctypes as C

    from s3prl_b200 import lib
    from s3prl_b200.upstream.configs import ARCHS
    from s3prl_b200.upstream.expert import _c_config

    def create(cfg, **over):
        c = _c_config(cfg)
        for k, v in over.items():
            setattr(c, k, v)
        h = C.c_void_p()
        rc = s3b_lib.s3b_model_create(C.byref(c), C.byref(h))
        if rc == 0:
            s3b_lib.s3b_model_destroy(h)
        return rc, s3b_lib.s3b_last_error().decode()

    for name in ("hubert_base", "wav2vec2_large_ll60k", "wavlm_large", "distilhubert_base", "data2vec_base_960",
                 "data2vec_large_ll60k"):
        assert create(ARCHS[name])[0] == 0, name
    rc, msg = create(ARCHS["hubert_base"], num_heads=16)  # 48-wide heads
    assert rc != 0 and "head dim" in msg
    rc, msg = create(ARCHS["data2vec_base_960"], family=lib.FAMILY_HUBERT)  # conv blocks go with the wav2vec2 mask rule
    assert rc != 0 and "pos_conv_depth" in msg
    rc, msg = create(ARCHS["data2vec_base_960"], pos_conv_depth=9)
    assert rc != 0 and "pos_conv_depth" in msg
    rc, msg = create(ARCHS["hubert_base"], pos_conv_kernel=127)  # the weight-normed conv needs an even kernel here
    assert rc != 0 and "even" in msg
    rc, msg = create(ARCHS["hubert_base"], pred_heads=3)  # prediction heads without the distiller front end: fine
    assert rc == 0
    rc, msg = create(ARCHS["hubert_base"], no_feature_layer_norm=1)
    assert rc != 0 and "distiller" in msg


def test_default_lanes_rule(s3b_lib):
    """Scheduling only (results are bit-identical, tests/test_upstream_gpu.py::test_lanes_are_bit_identical): two
    utterance lanes from 12 k frames per call on, one below — the measured crossover (profiles/README.md r2p / r2q)."""
    if os.environ.get("S3B_LANES") or os.environ.get("S3B_LANE_MIN_FRAMES"):
        pytest.skip("lane override set in the environment")
    f = s3b_lib.s3b_default_lanes
    assert f(None, 32, 160000) == 2 and f(None, 16, 320000) == 2   # BASELINE C2 / C3 on one GPU
    assert f(None, 16, 160000) == 1 and f(None, 8, 160000) == 1 and f(None, 4, 160000) == 1  # their 2 / 4 / 8-GPU shards
    assert f(None, 1, 16000000) == 1  # a single utterance cannot be split
    assert f(None, 0, 160000) == -1 and f(None, 4, 100) == -1


def test_config_from_reference_cfg_dict():
    from s3prl_b200.upstream.configs import ARCHS, arch_from_reference_cfg

    cfg = arch_from_reference_cfg(
        "wav2vec2",
        dict(extractor_mode="layer_norm", conv_bias=True, layer_norm_first=True, encoder_layers=24,
             encoder_embed_dim=1024, encoder_ffn_embed_dim=4096, encoder_attention_heads=16,
             conv_feature_layers="[(512, 10, 5)] + [(512, 3, 2)] * 4 + [(512,2,2)] + [(512,2,2)]"),
        dict(normalize=True),
    )
    assert cfg == ARCHS["wav2vec2_large_ll60k"]
    with pytest.raises(ValueError):
        arch_from_reference_cfg("hubert", dict(conv_feature_layers="[(512, 10, 5)]"))


def test_fabricated_state_dict_is_deterministic_and_loadable_layout():
    from s3prl_b200.upstream.configs import ARCHS
    from s3prl_b200.upstream.weights import fabricate_state_dict

    a = fabricate_state_dict(ARCHS["wavlm_base_plus"], 0)
    b = fabricate_state_dict(ARCHS["wavlm_base_plus"], 0)
    assert a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)
    assert a["encoder.pos_conv.0.weight_v"].shape == (768, 48, 128)
    assert a["encoder.layers.0.self_attn.relative_attention_bias.weight"].shape == (320, 12)
    assert a["feature_extractor.conv_layers.0.2.weight"].shape == (512,)
    c = fabricate_state_dict(ARCHS["wav2vec2_large_ll60k"], 0)
    assert c["feature_extractor.conv_layers.3.2.1.weight"].shape == (512,)
    assert c["feature_extractor.conv_layers.3.0.bias"].shape == (512,)


def test_hub_injection_into_reference(tmp_path):
    """`getattr(s3prl.hub, name)` — what Runner._get_upstream does (runner.py:141) — yields our expert after
    run_downstream.inject(), every other entry of the reference hub stays as it was, and the Featurizer the Runner
    instantiates is ours. Runs against the reference's own s3prl when it is available (oracle/build_ref.py), else against
    a stand-in package with the layout inject() touches and the reference hub's entry names (tests/golden/hub_entries.json,
    recorded from the reference by oracle/make_golden.py)."""
    import json
    import subprocess

    names = json.loads((GOLDEN / "hub_entries.json").read_text())
    assert {"hubert_base", "wavlm_base_plus", "fbank"} <= set(names)
    reference = _reference_install()
    if reference is None:
        reference = tmp_path
        pkg = tmp_path / "s3prl"
        for sub in ("upstream", "downstream"):
            (pkg / sub).mkdir(parents=True)
            (pkg / sub / "__init__.py").write_text("")
        (pkg / "__init__.py").write_text("")
        (pkg / "hub.py").write_text("".join(f"def {n}(*args, **kwargs):\n    raise RuntimeError('stand-in')\n" for n in names))
        (pkg / "upstream" / "interfaces.py").write_text("class Featurizer:\n    pass\n")
        (pkg / "downstream" / "runner.py").write_text("from s3prl.upstream.interfaces import Featurizer\n\n\nclass Runner:\n    pass\n")
    code = (
        "import json\n"
        "from s3prl_b200 import run_downstream as R\n"
        "R.install_shims()\n"
        "import s3prl.hub as hub\n"
        f"reference = json.loads(open({str(GOLDEN / 'hub_entries.json')!r}).read())\n"
        "before = {n: getattr(hub, n) for n in reference}\n"
        "names = R.inject()\n"
        "from s3prl_b200 import hub as ours\n"
        "from s3prl_b200.upstream.expert import UpstreamExpert\n"
        "from s3prl_b200.upstream.baseline import FbankExpert\n"
        "from s3prl_b200.upstream.featurizer import Featurizer\n"
        "e = getattr(hub, 'hubert_base')(ckpt=None, model_config=None, refresh=False)\n"
        "assert isinstance(e, UpstreamExpert) and e.get_downsample_rates('hidden_states') == 320\n"
        "assert isinstance(hub.fbank(), FbankExpert)\n"
        "assert isinstance(hub.wavlm_base_plus(), UpstreamExpert)\n"
        "assert all(getattr(hub, n) is ours.ENTRIES[n] for n in reference if n in ours.ENTRIES)\n"
        "assert all(getattr(hub, n) is before[n] for n in reference if n not in ours.ENTRIES)\n"
        "from s3prl.downstream.runner import Runner\n"
        "import s3prl.downstream.runner as runner, s3prl.upstream.interfaces as interfaces\n"
        "assert runner.Featurizer is Featurizer and interfaces.Featurizer is Featurizer\n"
        "print('OK', len(names), hub.__file__)\n"
    )
    env = dict(os.environ, PYTHONPATH=f"{reference}:{ROOT}")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=600)
    assert r.returncode == 0 and "OK" in r.stdout, r.stderr[-2000:]
    print(r.stdout.strip())


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under s3prl_b200/ (Python or CUDA) may import, include or execute it."""
    pat = re.compile(r"^\s*(from|import)\s+\S*oracle|sys\.path\S*oracle|#include\s+\S*oracle", re.M)
    for f in list((ROOT / "s3prl_b200").rglob("*.py")) + list((ROOT / "s3prl_b200" / "csrc").glob("*.cu*")):
        assert not pat.search(f.read_text()), f


def test_header_is_plain_c_and_links(s3b_lib, tmp_path):
    """include/s3prl_b200.h compiles as C99 (-Wall -Werror) and every entry point links from a plain-C program
    (examples/cabi_smoke.c); the integer frame rule runs through the ABI without a GPU."""
    import shutil
    import subprocess

    from s3prl_b200 import lib as L

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    exe = tmp_path / "cabi_smoke"
    libdir = L.lib_path().parent
    r = subprocess.run(
        [gcc, "-std=c99", "-Wall", "-Werror", f"-I{ROOT / 'include'}", str(ROOT / "examples" / "cabi_smoke.c"),
         f"-L{libdir}", "-ls3prl_b200", f"-Wl,-rpath,{libdir}", "-o", str(exe)],
        capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, (r.stdout, r.stderr)
    from s3prl_b200 import lib as L2

    assert f"{len(L2.EXPORTED_SYMBOLS)} entry points" in r.stdout and "49 3" in r.stdout


def test_hub_covers_the_same_skeleton_relatives():
    """Every wav2vec2 / HuBERT / WavLM / UniSpeech-SAT hub entry of the reference whose model is the 7-conv +
    post-/pre-LN Transformer skeleton with 64-wide heads (SURVEY §8(f) N3) has an entry here with the right family and
    shape; the entries outside the skeleton (conformer, 1B/2B XLS-R with 80/120-wide heads) are absent on purpose."""
    from s3prl_b200 import hub
    from s3prl_b200.upstream.configs import get_arch

    names = set(hub.options())
    for n in ("hubert_base", "hubert_large_ll60k", "hubert_base_robust_mgr", "mhubert_base_vp_en_es_fr_it3",
              "contentvec", "contentvec_km100", "contentvec_km500", "ms_hubert", "wav2vec2_base_960",
              "wav2vec2_large_960", "wav2vec2_large_ll60k", "wav2vec2_large_lv60_cv_swbd_fsh", "xlsr_53",
              "xls_r_300m", "wavlm_base", "wavlm_base_plus", "wavlm_large", "unispeech_sat_base",
              "unispeech_sat_base_plus", "unispeech_sat_large", "hubert_local", "wav2vec2_local", "wavlm_local",
              "unispeech_sat_local", "distilhubert", "distilhubert_base", "distiller_local", "data2vec", "data2vec_base_960",
              "data2vec_large_ll60k", "data2vec_local", "hubert_custom", "hubert_url", "wav2vec2_custom", "wav2vec2_url",
              "wavlm_url", "unispeech_sat_url", "distiller_url", "data2vec_custom", "data2vec_url", "fbank", "mel", "linear"):
        assert n in names, n
    for n in ("xls_r_1b", "xls_r_2b", "wav2vec2_conformer_relpos"):
        assert n not in names
    assert get_arch("xlsr_53") == get_arch("wav2vec2_large_ll60k")
    u = get_arch("unispeech_sat_base_plus")
    assert u.family == "wavlm" and not u.relative_position_embedding and not u.gru_rel_pos
    ul = get_arch("unispeech_sat_large")
    assert ul.layer_norm_first and ul.extractor_mode == "layer_norm" and ul.encoder_layers == 24
    assert get_arch("unispeech_sat") == u
    d = get_arch("data2vec")  # five k = 19 conv blocks instead of the weight-normed k = 128 conv (data2vec/hubconf.py:25-52)
    assert d.family == "data2vec" and d.family_id == 1 and d.pos_conv_depth == 5 and d.pos_conv_kernel == 19
    assert d.extractor_mode == "layer_norm" and d.normalize and not d.layer_norm_first
    assert get_arch("data2vec_large_ll60k").encoder_layers == 24


def _gloo_worker(rank, world, port, tmpdir):
    import torch.distributed as dist

    from s3prl_b200 import parallel as P

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        n_items, T, D = 7, 5, 4
        lens_all = [1000 + 37 * i for i in range(n_items)]
        full = torch.arange(n_items * T * D, dtype=torch.float32).view(n_items, T, D)
        lo, hi = P.shard_bounds(n_items, rank, world)
        my_lens = P.shard_batch(lens_all, rank, world)
        assert my_lens == lens_all[lo:hi]
        assert P.global_max_len(my_lens) == max(lens_all)
        out = P.gather_features(full[lo:hi].clone(), n_items)
        assert torch.equal(out, full)
        even = torch.arange(8 * T * D, dtype=torch.float32).view(8, T, D)
        lo, hi = P.shard_bounds(8, rank, world)
        assert torch.equal(P.gather_features(even[lo:hi].clone(), 8), even)
        (Path(tmpdir) / f"ok{rank}").write_text("ok")
    finally:
        dist.destroy_process_group()


def test_shard_and_gather_gloo_world2(tmp_path):
    import torch.multiprocessing as mp

    from s3prl_b200 import parallel as P

    # pure partition logic
    for n in (1, 7, 32, 33):
        for world in (1, 2, 3, 8):
            spans = [P.shard_bounds(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()


def test_converted_checkpoint_layouts_roundtrip(tmp_path):
    """N4: every converted layout the reference's *_local entries read (hubert/convert.py:37-56,
    wav2vec2/convert.py:26-39, wavlm/expert.py:37-40) is written by save_converted_checkpoint and read back by
    load_reference_checkpoint into the same ArchConfig and tensors; a file with a missing key raises the reference's
    ValueError text."""
    from s3prl_b200 import hub
    from s3prl_b200.upstream.configs import ARCHS
    from s3prl_b200.upstream.convert import converted_checkpoint, save_converted_checkpoint
    from s3prl_b200.upstream.weights import fabricate_state_dict, load_reference_checkpoint

    for name in ("hubert_base", "wav2vec2_large_ll60k", "wavlm_base_plus", "unispeech_sat_base_plus", "wavlm_large",
                 "distilhubert_base", "data2vec_base_960"):
        cfg = ARCHS[name]
        sd = fabricate_state_dict(cfg, 0)
        path = tmp_path / f"{name}.pt"
        save_converted_checkpoint(path, cfg, sd)
        got_cfg, got_sd = load_reference_checkpoint(str(path), cfg.family)
        assert got_cfg == cfg, name
        assert got_sd.keys() == sd.keys() and all(torch.equal(got_sd[k], sd[k]) for k in sd)
        # the hub's *_local entry builds an expert from the file (no GPU needed until the first forward)
        local = {"hubert": "hubert_local", "wav2vec2": "wav2vec2_local", "wavlm": "wavlm_local",
                 "distiller": "distiller_local", "data2vec": "data2vec_local"}[cfg.family]
        e = hub.ENTRIES[local](str(path))
        assert e.arch == cfg and e.num_layers == cfg.encoder_layers
        url_entry = hub.ENTRIES[local.replace("_local", "_url")]  # *_url / *_custom: a path works, a URL is refused
        assert url_entry(str(path), refresh=True).arch == cfg
        with pytest.raises(ValueError, match="not reachable"):
            url_entry("https://huggingface.co/s3prl/converted_ckpts/resolve/main/x.pt")
    with pytest.raises(ValueError, match="legacy"):
        hub.ENTRIES["hubert_custom"](str(tmp_path / "hubert_base.pt"), legacy=True)
    layout = converted_checkpoint(ARCHS["hubert_base"], {})
    assert set(layout) == {"task_cfg", "model_cfg", "model_weight", "dictionaries_symbols"}
    assert set(converted_checkpoint(ARCHS["wav2vec2_base_960"], {})) == {"task_cfg", "model_cfg", "model_weight"}
    assert set(converted_checkpoint(ARCHS["wavlm_base"], {})) == {"cfg", "model"}
    bad = tmp_path / "bad.pt"
    torch.save({"model_cfg": {}, "model_weight": {}}, bad)
    with pytest.raises(ValueError, match="required key: task_cfg is missing"):
        load_reference_checkpoint(str(bad), "hubert")


def test_fairseq_state_conversion():
    """convert_fairseq_state == load_and_convert_fairseq_ckpt minus the I/O (hubert/convert.py:17-34,
    wav2vec2/convert.py:14-23): cfg.task / cfg.model / model / dictionaries are re-keyed, nothing else."""
    from s3prl_b200.upstream.configs import arch_from_reference_cfg
    from s3prl_b200.upstream.convert import convert_fairseq_state

    class Dictionary:  # stand-in for fairseq.data.dictionary.Dictionary (only .symbols is read)
        def __init__(self, n):
            self.symbols = [str(i) for i in range(n)]

    w = {"layer_norm.weight": torch.ones(512)}
    state = {"cfg": {"task": {"normalize": False, "label_rate": 50.0}, "model": {"encoder_layers": 12, "extractor_mode": "default"}},
             "model": w, "task_state": {"dictionaries": [Dictionary(504)]}}
    out = convert_fairseq_state(state, "hubert")
    assert set(out) == {"task_cfg", "model_cfg", "model_weight", "dictionaries_symbols"}
    assert out["model_weight"] is w and len(out["dictionaries_symbols"][0]) == 504
    assert arch_from_reference_cfg("hubert", out["model_cfg"], out["task_cfg"]).encoder_layers == 12
    out2 = convert_fairseq_state({"cfg": state["cfg"], "model": w}, "wav2vec2")
    assert set(out2) == {"task_cfg", "model_cfg", "model_weight"}
    with pytest.raises(ValueError):
        convert_fairseq_state({"model": w}, "hubert")
    with pytest.raises(ValueError):
        convert_fairseq_state({"cfg": state["cfg"], "model": w}, "hubert")  # no dictionaries


@pytest.mark.parametrize("kind,kw", [
    ("hubert", {}),
    ("hubert", dict(feat_extract_norm="layer", do_stable_layer_norm=True, conv_bias=True)),
    ("wav2vec2", {}),
    ("wavlm", {}),
    ("data2vec", {}),
])
def test_huggingface_second_oracle(kind, kw):
    """N4: the HF -> fairseq parameter-name map (upstream/convert.py) against an INDEPENDENT implementation: a random
    transformers Hubert/Wav2Vec2/WavLM model (the reference's hf_* experts run these, hf_hubert/expert.py:12-41)
    evaluated by transformers' own forward must agree with oracle/upstream_oracle.py on the renamed weights
    (equal-length batch: HF's "group-norm" models ignore the attention mask). Also pins WavLM's gated relative
    position bias in the oracle against a second code base."""
    transformers = pytest.importorskip("transformers")
    import dataclasses

    sys.path.insert(0, str(ROOT / "oracle"))
    import upstream_oracle as O
    from s3prl_b200.upstream.convert import hf_to_fairseq_key, load_hf_model

    Cfg = {"hubert": transformers.HubertConfig, "wav2vec2": transformers.Wav2Vec2Config, "wavlm": transformers.WavLMConfig,
           "data2vec": transformers.Data2VecAudioConfig}[kind]
    Mod = {"hubert": transformers.HubertModel, "wav2vec2": transformers.Wav2Vec2Model, "wavlm": transformers.WavLMModel,
           "data2vec": transformers.Data2VecAudioModel}[kind]
    torch.manual_seed(0)
    cfg = Cfg(num_hidden_layers=2, **kw)
    cfg.layerdrop = 0.0
    model = Mod(cfg).eval()
    with torch.no_grad():
        for _n, p in model.named_parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn_like(p))
    arch, sd = load_hf_model(model)
    assert [k for k in model.state_dict() if hf_to_fairseq_key(k, arch.extractor_mode) is None] == ["masked_spec_embed"]
    x = torch.randn(2, 6000)
    with torch.no_grad():
        hf = model(x, output_hidden_states=True).hidden_states
        ref, _ = O.upstream_forward(list(x), {k: v.detach() for k, v in sd.items()}, dataclasses.replace(arch, normalize=False))
    assert len(hf) == len(ref) == 3
    for a, b in zip(hf, ref):
        assert ((a - b).norm() / b.norm()).item() < 5e-6


def _nn_golden():
    """What the reference's s3prl.nn classes returned on the inputs below (oracle/make_golden.py make_nn_fixture)."""
    return torch.load(GOLDEN / "nn_upstream.pt", weights_only=False)


def test_nn_featurizer_matches_reference_logic(monkeypatch):
    """s3prl_b200.nn.Featurizer / UpstreamDownstreamModel against the reference's own classes (s3prl/nn/upstream.py:234-384)
    on the CPU: layer selection, normalize, single-layer pass-through, weights and their gradient. The fused CUDA sum is
    replaced by its torch definition for this host-logic test (the kernel itself is pinned in tests/test_api_gpu.py)."""
    sys.path.insert(0, str(ROOT / "oracle"))
    from make_golden import FakeUpstream

    import s3prl_b200.upstream.featurizer as fused
    from s3prl_b200.nn import Featurizer, UpstreamDownstreamModel

    def torch_sum(feature, norm_weights):
        return (norm_weights.view(-1, 1, 1, 1) * torch.stack(list(feature), 0)).sum(0)

    with pytest.raises(fused._lib.S3BError):  # the product path has no CPU fallback
        fused.weighted_sum([torch.zeros(1, 4, 8)] * 2, torch.ones(2) / 2)
    monkeypatch.setattr(fused, "weighted_sum", torch_sum)

    fx = _nn_golden()
    hs, lens = fx["inputs"]["hs"], fx["inputs"]["lens"]
    cases = ((None, False), ([4, 0, 2], False), (None, True), ([1, 3], True))
    assert len(fx["featurizer"]) == len(cases)
    for (sel, norm), ref in zip(cases, fx["featurizer"]):
        ours = Featurizer(FakeUpstream(5), sel, norm)
        with torch.no_grad():
            ours.weights.copy_(ref["weights"])
        assert ours.layer_selections == ref["layer_selections"]
        a, al = ours(hs, lens)
        assert torch.allclose(a, ref["hs"], atol=1e-6) and torch.equal(al, ref["hs_len"])
        a.square().sum().backward()
        assert torch.allclose(ours.weights.grad, ref["grad"], rtol=1e-5, atol=1e-6)
        assert ours.output_size == ref["output_size"] == 16 and ours.downsample_rate == ref["downsample_rate"] == 320
    one = Featurizer(FakeUpstream(1))
    assert not hasattr(one, "weights") and not fx["single_layer_has_weights"]
    assert one(hs[:1], lens[:1])[0] is hs[0]

    class Up(torch.nn.Module):
        num_layers, hidden_sizes, downsample_rates = 5, [16] * 5, [320] * 5

        def forward(self, wav, wav_len):
            return hs, lens

    class Down(torch.nn.Module):  # no reduction: the stored result is exact on any CPU
        output_size = 3

        def forward(self, h, h_len, scale=1.0):
            return h[..., :3] * scale, h_len

    f = Featurizer(Up())
    ours, ref = UpstreamDownstreamModel(Up(), f, Down()), fx["udm"]
    a, al = ours(None, None, scale=2.0)
    assert torch.equal(a, ref["hs"]) and torch.equal(al, ref["hs_len"])
    assert (ours.input_size, ours.downsample_rate, ours.output_size) == (ref["input_size"], ref["downsample_rate"], ref["output_size"])
    with pytest.raises(NotImplementedError):
        UpstreamDownstreamModel(Up(), f, Down(), upstream_trainable=True)


def test_s3prl_upstream_bookkeeping_matches_reference_class():
    """The length bookkeeping of s3prl_b200.nn.S3PRLUpstream.forward (frame count per layer, last-frame repeat / cut,
    h_len, the 0.05 s minimum, normalize) against what the reference's own class (s3prl/nn/upstream.py:166-231) returned
    on the same fake upstream: identical tensors, and an AssertionError where the reference refuses a 2x frame mismatch."""
    sys.path.insert(0, str(ROOT / "oracle"))
    from make_golden import fake_s3prl_upstream

    from s3prl_b200.nn import S3PRLUpstream as Ours

    fx = _nn_golden()
    ours = fake_s3prl_upstream(Ours)
    # the fake upstream reads only the lengths, so these waveforms need not be the ones the reference was given
    g = torch.Generator().manual_seed(0)
    cases = [(lens, normalize) for lens in ([16000, 9000, 3200], [16001, 480], [700, 500], [32000, 31999],
                                            [1281, 1280, 1279], [48000]) for normalize in (False, True)]
    assert [(c["lens"], c["normalize"]) for c in fx["s3prl_upstream"]] == cases
    for ref in fx["s3prl_upstream"]:
        lens = ref["lens"]
        ours.normalize = ref["normalize"]
        width = max(lens) + 37  # the padded tensor may be wider than the longest utterance
        wavs = torch.zeros(len(lens), width)
        for i, n in enumerate(lens):
            wavs[i, :n] = torch.randn(n, generator=g)
        for w in (wavs, wavs.unsqueeze(-1)):
            b_hs, b_len = ours(w, torch.tensor(lens))
            assert len(ref["hs"]) == len(b_hs) == 3
            assert all(torch.equal(x, y) for x, y in zip(ref["hs"], b_hs)), lens
            assert all(torch.equal(x, y) for x, y in zip(ref["hs_len"], b_len)), lens
    # 2 frames from the conv rule where ceil(L / 320) = 4: refused by the reference, and here
    assert fx["s3prl_upstream_refused"] == [True, True]
    for lens in ([960, 961], [1000, 900]):
        with pytest.raises(AssertionError):
            ours(torch.zeros(len(lens), max(lens)), torch.tensor(lens))


def test_s3prl_upstream_wrapper_layer_counts():
    """S3PRLUpstream's static facts without a device: NL + 1 entries for the encoders, feat_final + layers + prediction
    heads for DistilHuBERT (s3prl/upstream/distiller/expert.py:44-63), one for fbank."""
    from s3prl_b200.nn import S3PRLUpstream

    assert S3PRLUpstream("hubert_base").num_layers == 13
    assert S3PRLUpstream("data2vec_large_ll60k").num_layers == 25
    d = S3PRLUpstream("distilhubert_base")
    assert d.num_layers == 6 and d.hidden_sizes == [768] * 6 and d.downsample_rates == [320] * 6


def _reference_install():
    """The s3prl checkout beside the repository (or S3PRL_REFERENCE), else the install under oracle/_ref that build()
    makes from it (oracle/build_ref.py), else None."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import ref_runtime

    return ref_runtime.reference_root()


# This test runs the reference's own training loop, so no stored result can stand in for the reference here.
@pytest.mark.skipif(_reference_install() is None, reason="needs the reference (s3prl): check it out at ../reference (or set S3PRL_REFERENCE) before build()")
def test_launcher_runs_reference_runner_on_synthetic_librispeech(tmp_path):
    """BASELINE config 5 plumbing without a GPU: the launcher's synthetic LibriSpeech-shaped dataloader
    (s3prl_b200/synthetic.py, replacing ctc/data.py:73-86 load_dataset) drives the reference's UNMODIFIED Runner.train
    (runner.py:227-429) and CTC DownstreamExpert for one optimisation step; S3B_NO_INJECT keeps the reference's own CPU
    fbank upstream so that the test needs no device. -f/--upstream_trainable is refused."""
    import subprocess

    env = dict(os.environ, PYTHONPATH=f"{ROOT}:{_reference_install()}", S3B_NO_INJECT="1")
    cmd = [sys.executable, "-m", "s3prl_b200.run_downstream", "--synthetic_data", "-m", "train", "-u", "fbank", "-d", "ctc",
           "-c", "downstream/ctc/librispeech.yaml", "-p", str(tmp_path / "exp"), "--device", "cpu", "-o",
           "config.runner.total_steps=1,,config.runner.eval_step=100000,,config.runner.save_step=100000,,"
           "config.runner.log_step=1,,config.downstream_expert.corpus.batch_size=2,,"
           "config.downstream_expert.model.RNNs.dim=[64,64,64],,config.downstream_expert.model.project_dim=64"]
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "train loss:" in r.stdout and "synthetic LibriSpeech-shaped" in r.stderr
    r2 = subprocess.run(cmd[:3] + ["-f"] + cmd[3:], capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=300)
    assert r2.returncode != 0 and "upstream_trainable is not supported" in r2.stderr


def test_synthetic_batches_follow_collect_audio_batch_rules():
    """Host batch assembly (ctc/data.py:11-43): descending length inside a batch, bucket halved when the first
    utterance exceeds 300 000 samples, float32 waveforms, integer label arrays."""
    import numpy as np

    from s3prl_b200 import synthetic as syn

    class Tok:
        vocab_size = 31

    dl = syn.load_dataset("train", Tok(), {"batch_size": 32, "bucketing": True, "num_workers": 0})
    seen_half = seen_full = False
    for i, (wavs, labels, files) in enumerate(dl):
        lens = [len(w) for w in wavs]
        assert lens == sorted(lens, reverse=True)
        assert all(w.dtype == np.float32 for w in wavs) and all(l.dtype == np.int64 for l in labels)
        assert len(wavs) == len(labels) == len(files)
        if len(wavs) == 16:
            seen_half = True
            assert max(lens) <= 24 * 16000
        if len(wavs) == 32:
            seen_full = True
            # (the rule looks at the bucket's FIRST utterance, which need not be its longest)
            assert max(lens) <= 24 * 16000 and min(lens) >= 2 * 16000
        assert len(wavs) in (16, 32)
        if i > 200:
            break
    assert seen_full and seen_half
