"""Mint tests/golden/reference_interfaces.json: what the drop-in (index-tts_b200/dropin.py) and the entry-point classes
(index-tts_b200/infer_v2_5.py, infer.py) rely on from the reference, recorded as data so that the tests that check
them run without the reference tree.

Stored:
  modules     the small reference modules of tests/test_dropin_cpu.py, built by the reference's own classes: the name,
              shape and dtype of every state-dict entry, plus the plain attributes `attach` / `attach_v1` read;
  call_sites  every call `infer_v2_5.py` (`infer_generator`) and `infer.py` make at the rebound seams: the number of
              positional arguments, the keyword names, and whether `**kwargs` is passed;
  signatures  the parameter names and literal defaults of `IndexTTS2` / `IndexTTS` `__init__` and `infer`.

Build container only (needs the reference tree, oracle/refimport.py).
    python -m oracle.make_goldens_interfaces
"""
import ast
import json
import os
import re

from indextts_b200 import synth
from oracle import refimport
from oracle.gpt import make_gpt_weights
from oracle.make_goldens_v1 import reference_module
from oracle.validate_gpt_vs_hf import small_case

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                   "reference_interfaces.json")

# the seams `attach` rebinds, under the expression `infer_generator` calls them by
SEAMS_V2 = {"self.gpt.merge_emovec": "merge_emovec", "self.gpt.inference_speech": "inference_speech",
            "self.semantic_codec.decode": "codec_decode", "self.s2mel.models['length_regulator']": "length_regulator",
            "self.s2mel.models['cfm'].inference": "cfm_inference", "self.bigvgan": "bigvgan"}
SEAMS_V1 = ("self.gpt.inference_speech", "self.gpt", "self.bigvgan")


def state_dict_layout(m):
    return {k: [list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in m.state_dict().items()}


def modules():
    cfg, _, _, _ = small_case()
    cfg = dict(cfg, n_langs=106)
    gpt = refimport.gpt_module(cfg, make_gpt_weights(cfg, seed=1, bf16=False))
    s2 = refimport.s2mel_module(refimport.s2mel_args(hidden=64, heads=1, depth=3, wn_hidden=64, wn_layers=2,
                                                     content_dim=64, lr_in=96, style_dim=24))
    codec = refimport.codec_module(codebook_size=64, hidden_size=96, codebook_dim=8, vocos_dim=48,
                                   vocos_intermediate_dim=64, vocos_num_layers=2)
    bv = refimport.bigvgan_module(synth.small_config())
    per = getattr(gpt, "emo_perceiver_encoder", None)
    out = {
        "gpt": {"state_dict": state_dict_layout(gpt),
                "attrs": {"blocks": len(gpt.gpt.h), "model_dim": gpt.model_dim, "heads": gpt.heads,
                          "number_mel_codes": gpt.number_mel_codes, "start_mel_token": gpt.start_mel_token,
                          "stop_mel_token": gpt.stop_mel_token, "max_mel_tokens": gpt.max_mel_tokens,
                          "emo_input_size": getattr(gpt, "emo_input_size", None),
                          "emo_perceiver_heads": getattr(per, "heads", None)}},
        "s2mel": {"state_dict": state_dict_layout(s2), "models": sorted(s2.models.keys()),
                  "attrs": {"cfm_in_channels": s2.models["cfm"].in_channels}},
        "semantic_codec": {"state_dict": state_dict_layout(codec)},
        "bigvgan": {"state_dict": state_dict_layout(bv), "h": dict(bv.h)},
    }
    cfg, _, _, _ = small_case()
    ccfg = synth.small_v1_cond_cfg(cfg["model_dim"])
    gpt1 = refimport.gpt_module_v1(cfg, ccfg, synth.make_gpt_v1_weights(cfg, ccfg, seed=3), kv_cache=False)
    h1 = synth.small_v1_config()
    bv1 = reference_module(h1, synth.make_bigvgan_v1_weights(h1, seed=5))
    out["v1_gpt"] = {"state_dict": state_dict_layout(gpt1),
                     "attrs": {"blocks": len(gpt1.gpt.h), "model_dim": gpt1.model_dim, "heads": gpt1.heads,
                               "number_mel_codes": gpt1.number_mel_codes, "start_mel_token": gpt1.start_mel_token,
                               "stop_mel_token": gpt1.stop_mel_token, "max_mel_tokens": gpt1.max_mel_tokens,
                               "kv_cache": bool(getattr(gpt1.inference_model, "kv_cache", False))}}
    out["v1_bigvgan"] = {"state_dict": state_dict_layout(bv1), "h": dict(bv1.h)}
    return out


def _source(rel):
    return ast.parse(open(os.path.join(refimport.REF, "indextts", rel)).read())


def call_sites():
    v2 = {}
    for node in ast.walk(_source("infer_v2_5.py")):
        if isinstance(node, ast.Call) and ast.unparse(node.func) in SEAMS_V2:
            v2.setdefault(SEAMS_V2[ast.unparse(node.func)], []).append(
                [len(node.args), [k.arg for k in node.keywords if k.arg is not None],
                 any(k.arg is None for k in node.keywords)])
    v1 = {}
    for node in ast.walk(_source("infer.py")):
        if isinstance(node, ast.Call) and ast.unparse(node.func) in SEAMS_V1:
            v1.setdefault(ast.unparse(node.func), []).append(
                [len(node.args), [k.arg for k in node.keywords if k.arg is not None],
                 any(k.arg is None for k in node.keywords)])
    return {"infer_v2_5": v2, "infer": v1}


def signatures():
    out = {}
    for rel, cls_name in (("infer_v2_5.py", "IndexTTS2"), ("infer.py", "IndexTTS")):
        cls = next(n for n in _source(rel).body if isinstance(n, ast.ClassDef) and n.name == cls_name)
        fns = {f.name: f for f in cls.body if isinstance(f, ast.FunctionDef)}
        out[cls_name] = {name: {"args": [a.arg for a in fns[name].args.args],
                                "kwarg": fns[name].args.kwarg.arg if fns[name].args.kwarg else None,
                                "defaults": [ast.literal_eval(d) for d in fns[name].args.defaults]}
                         for name in ("__init__", "infer")}
    return out


def main():
    refimport.setup()
    doc = {"modules": modules(), "call_sites": call_sites(), "signatures": signatures()}
    text = json.dumps(doc, sort_keys=True, indent=1)
    # one line per state-dict entry / call site: lists without (then with one level of) nested lists go on one line
    flat = lambda m: re.sub(r"\s*\n\s*", " ", m.group(0)).replace("[ ", "[").replace(" ]", "]")  # noqa: E731
    text = re.sub(r"\[[^\[\]{}]*\]", flat, text)
    text = re.sub(r"\[[^\[\]{}]*(?:\[[^\[\]{}]*\][^\[\]{}]*)+\]", flat, text)
    assert json.loads(text) == json.loads(json.dumps(doc))
    with open(OUT, "w") as f:
        f.write(text + "\n")
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
