"""The entry-point classes keep the reference's constructor / .infer() signatures (SURVEY §8b): parameter names and literal
defaults as recorded from the reference source in tests/golden/reference_interfaces.json (oracle/make_goldens_interfaces.py).
Building a live reference IndexTTS2 additionally needs checkpoints and the w2v-BERT / CAMPPlus / BigVGAN downloads of
infer_v2_5.py:170-260, which do not exist offline — that is what blocks an end-to-end `.infer()` test here, not anything
in this package."""
import inspect
import json
import os

GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference_interfaces.json")


def _reference_signatures(cls_name):
    with open(GOLD) as f:
        return json.load(f)["signatures"][cls_name]


def _params(fn, drop=()):
    return [(n, p.default) for n, p in inspect.signature(fn).parameters.items() if n not in drop]


def test_indextts2_signatures_match_the_reference():
    fns = _reference_signatures("IndexTTS2")
    from indextts_b200.infer_v2_5 import IndexTTS2
    for name, drop in (("__init__", ("engine_device",)), ("infer", ())):
        ref_args = list(fns[name]["args"])
        mine = [n for n, _ in _params(getattr(IndexTTS2, name), drop)]
        if fns[name]["kwarg"]:
            ref_args.append(fns[name]["kwarg"])
        assert mine == ref_args, (name, mine, ref_args)
        ref_defaults = fns[name]["defaults"]
        my_defaults = [d for n, d in _params(getattr(IndexTTS2, name), drop) if d is not inspect.Parameter.empty]
        assert my_defaults == ref_defaults, (name, my_defaults, ref_defaults)


def test_indextts_v1_signatures_match_the_reference():
    fns = _reference_signatures("IndexTTS")
    from indextts_b200.infer import IndexTTS
    for name, drop in (("__init__", ("engine_device",)), ("infer", ())):
        ref_args = fns[name]["args"] + ([fns[name]["kwarg"]] if fns[name]["kwarg"] else [])
        mine = [n for n, _ in _params(getattr(IndexTTS, name), drop)]
        assert mine == ref_args, (name, mine, ref_args)
