"""CPU: `dropin.load_reference_weights` / `attach` / `attach_v1` against the reference's own modules and call sites, as
recorded in tests/golden/reference_interfaces.json (oracle/make_goldens_interfaces.py): for small modules built by the
reference's own classes, the name / shape / dtype of every state-dict entry and the plain attributes the drop-in reads;
and every call `infer_v2_5.py` / `infer.py` make at the rebound seams.  Stand-ins rebuilt from the record go through the
drop-in, a recording stand-in replaces the engine, and the test checks that every hyper-parameter the drop-in derives
from the state dicts equals what the modules were constructed with, that every tensor name the engine will ask for
(`gpt.…`, `s2mel.…`, `codec.…`, `bigvgan.…`) is present, and that the reference's calls bind to the rebound seams."""
import json
import os
import types

import torch

GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference_interfaces.json")


def _golden():
    with open(GOLD) as f:
        return json.load(f)


def _module(rec):
    """Stand-in for a recorded reference module: its state dict, placeholder values under the reference's names,
    shapes and dtypes."""
    sd = {k: torch.ones(shape, dtype=getattr(torch, dt)) for k, (shape, dt) in rec["state_dict"].items()}
    return types.SimpleNamespace(state_dict=lambda: sd)


def _gpt(rec):
    """Stand-in for a reference `UnifiedVoice` (v2 or v1) with the attributes the drop-in reads."""
    a = rec["attrs"]
    m = _module(rec)
    m.gpt = types.SimpleNamespace(h=[None] * a["blocks"])
    for k in ("model_dim", "heads", "number_mel_codes", "start_mel_token", "stop_mel_token", "max_mel_tokens"):
        setattr(m, k, a[k])
    if a.get("emo_input_size") is not None:
        m.emo_input_size = a["emo_input_size"]
    if "emo_perceiver_encoder.latents" in m.state_dict():
        m.emo_perceiver_encoder = types.SimpleNamespace(latents=m.state_dict()["emo_perceiver_encoder.latents"])
        if a.get("emo_perceiver_heads") is not None:
            m.emo_perceiver_encoder.heads = a["emo_perceiver_heads"]
    if "kv_cache" in a:
        m.inference_model = types.SimpleNamespace(kv_cache=a["kv_cache"])
    return m


def _bigvgan(rec):
    m = _module(rec)
    m.h = rec["h"]
    return m


def _reference_tts():
    """The modules of a reference IndexTTS2 (infer_v2_5) that `attach` reads and rebinds."""
    mods = _golden()["modules"]
    s2 = _module(mods["s2mel"])
    s2.models = {name: types.SimpleNamespace() for name in mods["s2mel"]["models"]}
    s2.models["cfm"].in_channels = mods["s2mel"]["attrs"]["cfm_in_channels"]
    return types.SimpleNamespace(gpt=_gpt(mods["gpt"]), s2mel=s2, semantic_codec=_module(mods["semantic_codec"]),
                                 bigvgan=_bigvgan(mods["bigvgan"]))


class RecordingEngine:
    device = 0

    def __init__(self):
        self.weights, self.calls = {}, {}

    def load_state_dict(self, prefix, sd):
        for k, v in sd.items():
            self.weights[prefix + k] = tuple(v.shape)

    def gpt_init(self, *a, **k):
        self.calls["gpt_init"] = (a, k)

    def emo_init(self, c):
        self.calls["emo_init"] = dict(c)
        self.emo_cfg = types.SimpleNamespace(**c)

    def s2mel_init(self, c):
        self.calls["s2mel_init"] = dict(c)

    def codec_init(self, c):
        self.calls["codec_init"] = dict(c)

    def bigvgan_init(self, h):
        self.calls["bigvgan_init"] = dict(h)


def test_config_derivation_from_real_reference_modules():
    from indextts_b200 import synth
    from indextts_b200.dropin import load_reference_weights
    from oracle.validate_gpt_vs_hf import small_case

    cfg, _, _, _ = small_case()
    h = synth.small_config()
    tts = _reference_tts()
    gpt = tts.gpt
    eng = RecordingEngine()
    load_reference_weights(eng, tts, max_batch=4)

    a, k = eng.calls["gpt_init"]
    assert a[:6] == (cfg["layers"], cfg["model_dim"], cfg["heads"], cfg["number_mel_codes"], cfg["start_mel_token"],
                     cfg["stop_mel_token"])
    assert a[6] == cfg["max_mel_tokens"] + 2 + 1            # mel_pos rows (model_v2.py:398-400)
    assert k["max_batch"] == 4 and k["weights_bf16"] is True
    emo = eng.calls["emo_init"]
    assert (emo["idim"], emo["odim"], emo["linear_units"], emo["heads"], emo["blocks"]) == (1024, 32, 48, 2, 1)
    assert emo["model_dim"] == cfg["model_dim"] and emo["p_dim"] == gpt.emo_perceiver_encoder.latents.shape[-1]
    s = eng.calls["s2mel_init"]
    assert (s["hidden"], s["heads"], s["depth"], s["wn_hidden"], s["wn_layers"], s["wn_kernel"]) == (64, 1, 3, 64, 2, 5)
    assert (s["in_channels"], s["content_dim"], s["style_dim"], s["lr_in"], s["lr_convs"]) == (80, 64, 24, 96, 4)
    c = eng.calls["codec_init"]
    assert c == dict(codebook_size=64, hidden_size=96, codebook_dim=8, vocos_dim=48, vocos_intermediate_dim=64,
                     vocos_num_layers=2)
    assert eng.calls["bigvgan_init"]["upsample_rates"] == list(h["upsample_rates"])
    # the tensors the C++ side looks up by name exist under the names the reference uses
    need = ["gpt.gpt.h.0.attn.c_attn.weight", "gpt.mel_head.weight", "gpt.final_norm.weight", "gpt.spk_emb_proj.weight",
            "gpt.lang_embedding.weight", "gpt.text_pos_embedding.emb.weight", "gpt.emovec_layer.weight",
            "gpt.emo_conditioning_encoder.embed.out.0.weight", "gpt.emo_perceiver_encoder.latents",
            "s2mel.cfm.estimator.cond_projection.weight", "s2mel.cfm.estimator.wavenet.in_layers.0.conv.conv.weight",
            "s2mel.length_regulator.content_in_proj.weight", "codec.quantizer.quantizers.0.codebook.weight",
            "codec.decoder.1.weight", "bigvgan.conv_pre.weight", "bigvgan.ups.0.0.weight",
            "bigvgan.resblocks.0.convs1.0.weight", "bigvgan.conv_post.weight"]
    missing = [n for n in need if n not in eng.weights]
    assert not missing, missing
    assert not any(".weight_g" in n or ".weight_v" in n or "parametrizations" in n for n in eng.weights), \
        "weight-norm pairs must be folded before they reach the engine"


def test_rebound_seams_accept_the_reference_call_sites():
    """Every call `infer_v2_5.py` makes at a seam binds to the callable `attach` installs there (same positional
    arity, same keyword names) — the drop-in claim of INTEGRATION.md, checked against the reference's call sites
    ((positional count, keyword names, **kwargs passed) per call, read from its source with ast)."""
    import inspect

    from indextts_b200.dropin import attach

    tts = _reference_tts()
    gpt, bv = tts.gpt, tts.bigvgan
    eng = RecordingEngine()
    attach(tts, engine=eng)
    seams = {"merge_emovec": tts.gpt.merge_emovec, "inference_speech": tts.gpt.inference_speech,
             "codec_decode": tts.semantic_codec.decode, "length_regulator": tts.s2mel.models["length_regulator"].forward,
             "cfm_inference": tts.s2mel.models["cfm"].inference, "bigvgan": tts.bigvgan.forward}
    sites = _golden()["call_sites"]["infer_v2_5"]
    assert set(sites) == set(seams), (sorted(sites), sorted(seams))
    for name, calls in sites.items():
        sig = inspect.signature(seams[name])
        for npos, kws, star in calls:
            try:
                sig.bind(*([None] * npos), **{k: None for k in kws})
            except TypeError as e:
                raise AssertionError(f"{name}: reference call ({npos} positional, keywords {kws}) does not bind to {sig}: {e}")
    # the rebound objects are the reference's own module objects: infer_generator reaches them unchanged
    assert tts.gpt is gpt and tts.bigvgan is bv and tts._b200_engine is eng


def test_attach_v1_on_real_reference_v1_modules():
    """v1 / v1.5 drop-in (row a13): `attach_v1` on the reference's own v1 `UnifiedVoice` and `BigVGAN` classes — the derived
    prompt-encoder / vocoder configuration equals what the modules were built with, and the calls `indextts/infer.py` makes
    at the three seams bind to the rebound callables."""
    import inspect

    from indextts_b200 import synth
    from indextts_b200.dropin import attach_v1
    from oracle.validate_gpt_vs_hf import small_case

    cfg, _, _, _ = small_case()
    ccfg = synth.small_v1_cond_cfg(cfg["model_dim"])
    h = synth.small_v1_config()
    doc = _golden()
    gpt, bv = _gpt(doc["modules"]["v1_gpt"]), _bigvgan(doc["modules"]["v1_bigvgan"])
    tts = types.SimpleNamespace(gpt=gpt, bigvgan=bv)

    class Rec(RecordingEngine):
        def v1_cond_init(self, c, n):
            self.calls["v1_cond_init"] = (dict(c), n)

        def v1_vocoder_init(self, hh):
            self.calls["v1_vocoder_init"] = dict(hh)

    eng = Rec()
    attach_v1(tts, engine=eng)
    c, n = eng.calls["v1_cond_init"]
    assert n == 32
    for k in ("idim", "odim", "linear_units", "heads", "blocks", "cnn_kernel", "p_dim", "p_heads", "p_dim_head", "p_depth", "p_ff_mult"):
        assert c[k] == ccfg[k], (k, c[k], ccfg[k])
    a, kw = eng.calls["gpt_init"]
    assert a[:3] == (cfg["layers"], cfg["model_dim"], cfg["heads"]) and kw["weights_bf16"] is False
    assert eng.calls["v1_vocoder_init"]["gpt_dim"] == h["gpt_dim"]
    assert "bigvgan_v1.speaker_encoder.blocks.0.conv.conv.weight" in eng.weights and "bigvgan_v1.cond_layer.weight" in eng.weights
    assert "gpt.conditioning_encoder.embed.out.0.weight" in eng.weights and "gpt.perceiver_encoder.latents" in eng.weights
    # call sites of indextts/infer.py
    want = {"self.gpt.inference_speech": tts.gpt.inference_speech, "self.gpt": tts.gpt.forward, "self.bigvgan": tts.bigvgan.forward}
    sites = doc["call_sites"]["infer"]
    assert set(sites) == set(want)
    for name, calls in sites.items():
        for npos, kws, _star in calls:
            inspect.signature(want[name]).bind(*([None] * npos), **{k: None for k in kws})
