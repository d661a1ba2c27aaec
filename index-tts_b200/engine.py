"""ctypes shim over libidxtts.so (include/idxtts.h).

The library is the product; this file only marshals pointers.  Tensors may be torch tensors
(CPU or CUDA) or numpy arrays — the library accepts host or device pointers.  There is no CPU
fallback: `Engine()` raises RuntimeError when no sm_100 device is visible or the library is
missing.
"""
import ctypes as C
import os
import re

import numpy as np

try:  # torch is only a tensor container here
    import torch
except Exception:  # pragma: no cover
    torch = None

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
LIB_PATH = os.path.join(_PKG, "libidxtts.so")
HEADER_PATH = os.path.join(_ROOT, "include", "idxtts.h")

IDX_F32, IDX_BF16, IDX_F16, IDX_I32, IDX_I64 = 0, 1, 2, 3, 4

_lib = None


class GptConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "layers", "model_dim", "heads", "number_mel_codes", "start_mel_token", "stop_mel_token",
        "max_mel_positions", "max_prompt", "max_batch", "weights_bf16")]


class Sampling(C.Structure):
    _fields_ = [("do_sample", C.c_int32), ("num_beams", C.c_int32), ("top_k", C.c_int32),
                ("top_p", C.c_float), ("temperature", C.c_float),
                ("repetition_penalty", C.c_float), ("length_penalty", C.c_float),
                ("max_new_tokens", C.c_int32), ("seed", C.c_uint64),
                ("forbid_stop_before", C.c_int32), ("mel_pos_mode", C.c_int32)]


class GptRequest(C.Structure):
    _fields_ = [("prompt_emb", C.c_void_p), ("prompt_len", C.c_int32),
                ("codes_out", C.c_void_p), ("n_codes_out", C.c_void_p),
                ("logits_out", C.c_void_p), ("forced_codes", C.c_void_p)]


class BigvganConfig(C.Structure):
    _fields_ = [("num_mels", C.c_int32), ("upsample_initial_channel", C.c_int32),
                ("num_upsamples", C.c_int32), ("upsample_rates", C.c_int32 * 8),
                ("upsample_kernel_sizes", C.c_int32 * 8), ("num_kernels", C.c_int32),
                ("resblock_kernel_sizes", C.c_int32 * 4),
                ("resblock_dilations", (C.c_int32 * 3) * 4),
                ("use_tanh_at_final", C.c_int32), ("use_bias_at_final", C.c_int32),
                ("snake_logscale", C.c_int32)]


class S2melConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("hidden", "heads", "depth", "wn_hidden", "wn_layers", "wn_kernel",
                                         "in_channels", "content_dim", "style_dim", "lr_in", "lr_convs")]


class CodecConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("codebook_size", "hidden_size", "codebook_dim", "vocos_dim",
                                         "vocos_intermediate_dim", "vocos_num_layers")]


class EmoConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("idim", "odim", "linear_units", "heads", "blocks", "cnn_kernel", "p_dim",
                                         "p_heads", "p_dim_head", "p_depth", "p_ff_mult", "model_dim")]


class VocodeRequest(C.Structure):
    _fields_ = [("codes", C.c_void_p), ("n_codes", C.c_int32), ("prompt_condition", C.c_void_p),
                ("ref_mel", C.c_void_p), ("P", C.c_int32), ("style", C.c_void_p), ("z", C.c_void_p),
                ("F", C.c_int32), ("wav_out", C.c_void_p), ("pcm16_out", C.c_void_p), ("mel_out", C.c_void_p)]


def fold_weight_norm(sd):
    """torch weight_norm (dim=0) folded into a plain `.weight`: w = g * v / ||v|| — what
    remove_weight_norm() / the parametrisation computes on the fly in the reference."""
    out = {}
    for k, v in sd.items():
        if k.endswith("weight_g"):
            base = k[: -len("weight_g")]
            vv = sd[base + "weight_v"].float()
            norm = vv.reshape(vv.shape[0], -1).norm(dim=1).reshape(-1, *([1] * (vv.dim() - 1)))
            out[base + "weight"] = v.float() * vv / norm
        elif k.endswith("weight_v"):
            continue
        else:
            out[k] = v
    return out


def declared_symbols():
    """Every function the C-ABI header declares (used by the symbol-export test)."""
    src = open(HEADER_PATH).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(idx_[a-z0-9_]+)\s*\(", src)))


def load_library(path: str = None):
    """dlopen the library and check that it exports everything include/idxtts.h declares."""
    global _lib
    if _lib is not None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} not found: build it with `python __graft_entry__.py` — there is no "
            "CPU/PyTorch fallback for the hot path")
    lib = C.CDLL(path)
    missing = [s for s in declared_symbols() if not hasattr(lib, s)]
    if missing:
        raise RuntimeError(f"libidxtts.so does not export: {missing}")
    lib.idx_last_error.restype = C.c_char_p
    lib.idx_last_error.argtypes = [C.c_void_p]
    lib.idx_version.restype = C.c_char_p
    lib.idx_launch_count.restype = C.c_int64
    lib.idx_launch_count.argtypes = [C.c_void_p]
    lib.idx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.idx_destroy.argtypes = [C.c_void_p]
    lib.idx_sync.argtypes = [C.c_void_p]
    lib.idx_wait_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.idx_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    lib.idx_event_record.argtypes = [C.c_void_p, C.c_int]
    lib.idx_event_elapsed_ms.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double)]
    lib.idx_load_weight.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int, C.c_int,
                                    C.POINTER(C.c_int64)]
    lib.idx_gpt_init.argtypes = [C.c_void_p, C.POINTER(GptConfig)]
    lib.idx_gpt_generate.argtypes = [C.c_void_p, C.POINTER(GptRequest), C.c_int,
                                     C.POINTER(Sampling)]
    lib.idx_gpt_prepare_inputs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_int, C.c_int, C.c_void_p]
    lib.idx_gpt_last_timing.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    lib.idx_gpt_profile.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
    lib.idx_gpt_profile_fine.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    lib.idx_v1_cond_init.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    lib.idx_v1_get_conditioning.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.idx_gpt_prepare_inputs_v1.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    lib.idx_gpt_latents_v1.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    lib.idx_v1_vocoder_init.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.idx_v1_speaker_embedding.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.idx_v1_vocode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    lib.idx_gpt_beam_trace.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.idx_bigvgan_init.argtypes = [C.c_void_p, C.POINTER(BigvganConfig)]
    lib.idx_bigvgan_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.idx_antialias_snake.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.idx_bigvgan_last_ms.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    lib.idx_debug_conv_gemm.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                        C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                        C.c_float, C.c_longlong, C.c_int, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p]
    lib.idx_debug_gemm_pair_epilogue.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                                 C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                                 C.c_int, C.c_float, C.c_void_p]
    lib.idx_debug_flash_attention.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                              C.c_void_p]
    lib.idx_debug_attention_rope.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.idx_s2mel_init.argtypes = [C.c_void_p, C.POINTER(S2melConfig)]
    lib.idx_codec_init.argtypes = [C.c_void_p, C.POINTER(CodecConfig)]
    lib.idx_codec_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.idx_length_regulate.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.idx_dit_forward.argtypes = [C.c_void_p] + [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_void_p]
    lib.idx_cfm_solve.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_int, C.c_float, C.c_void_p]
    lib.idx_s2mel_last_ms.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    lib.idx_emo_init.argtypes = [C.c_void_p, C.POINTER(EmoConfig)]
    lib.idx_merge_emovec.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_float, C.c_void_p]
    lib.idx_codes_to_wav.argtypes = [C.c_void_p, C.POINTER(VocodeRequest), C.c_int, C.c_float]
    _lib = lib
    return lib


def _ptr(x):
    """Raw pointer of a contiguous torch tensor / numpy array (host or device)."""
    if x is None:
        return None
    if torch is not None and isinstance(x, torch.Tensor):
        assert x.is_contiguous(), "tensor must be contiguous"
        return x.data_ptr()
    assert isinstance(x, np.ndarray) and x.flags["C_CONTIGUOUS"]
    return x.ctypes.data


def _as_f32(x):
    if torch is not None and isinstance(x, torch.Tensor):
        return x.detach().to(torch.float32).contiguous()
    return np.ascontiguousarray(x, dtype=np.float32)


def _is_cuda(x):
    return torch is not None and isinstance(x, torch.Tensor) and x.is_cuda


def _empty_like_src(src, shape, np_dtype=np.float32):
    """Output container that lives where `src` lives: a torch CUDA tensor for a CUDA input (the library then writes
    device-to-device, nothing bounces through the host), a numpy array otherwise."""
    if _is_cuda(src):
        return torch.empty(shape, dtype=getattr(torch, np.dtype(np_dtype).name), device=src.device)
    return np.empty(shape, dtype=np_dtype)


class _OrderedLib:
    """Proxy over the ctypes library that honours the stream contract of include/idxtts.h: before every call the
    engine stream is ordered (idx_wait_stream: event + cudaStreamWaitEvent, no host block) after torch's current
    stream, so device tensors still being produced by pending torch kernels are complete when the engine reads them."""
    _PLAIN = ("idx_last_error", "idx_destroy", "idx_launch_count", "idx_version", "idx_wait_stream", "idx_create")

    def __init__(self, lib, eng):
        self._lib, self._eng = lib, eng

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if name in self._PLAIN:
            return fn
        eng, raw = self._eng, self._lib

        def call(*a):
            if torch is not None and torch.cuda.is_available() and torch.cuda.is_initialized():
                raw.idx_wait_stream(eng.h, C.c_void_p(torch.cuda.current_stream(eng.device).cuda_stream))
            return fn(*a)
        return call


class Engine:
    """One engine = one CUDA device = one caller thread at a time (include/idxtts.h)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.idx_create(int(device), C.byref(h))
        if rc != 0:
            raise RuntimeError(f"idx_create failed ({rc}): {self.lib.idx_last_error(None).decode()}")
        self.h = h
        self.device = device
        self._keep = []
        self.lib = _OrderedLib(self.lib, self)

    def close(self):
        if getattr(self, "h", None):
            self.lib.idx_destroy(self.h)
            self.h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"{what} failed ({rc}): {self.lib.idx_last_error(self.h).decode()}")

    @property
    def launches(self) -> int:
        return int(self.lib.idx_launch_count(self.h))

    def sync(self):
        self._check(self.lib.idx_sync(self.h), "idx_sync")

    def set_option(self, name: str, value: int):
        self._check(self.lib.idx_set_option(self.h, name.encode(), int(value)), f"idx_set_option({name})")

    def event_record(self, slot: int):
        self._check(self.lib.idx_event_record(self.h, int(slot)), "idx_event_record")

    def event_elapsed_ms(self, a: int, b: int) -> float:
        t = C.c_double()
        self._check(self.lib.idx_event_elapsed_ms(self.h, int(a), int(b), C.byref(t)), "idx_event_elapsed_ms")
        return t.value

    # ------------------------------------------------------------------ weights --
    def load_weight(self, name: str, t):
        t = _as_f32(t)
        shape = (C.c_int64 * max(1, t.ndim))(*[int(s) for s in t.shape])
        self._check(self.lib.idx_load_weight(self.h, name.encode(), _ptr(t), IDX_F32, t.ndim, shape),
                    f"idx_load_weight({name})")

    def load_state_dict(self, prefix: str, sd: dict):
        """Mirror of load_checkpoint (indextts/utils/checkpoint.py:22-35): every tensor of the
        state dict is registered under `prefix + key`."""
        for k, v in sd.items():
            if hasattr(v, "dtype") and (getattr(v, "is_floating_point", lambda: True)()):
                self.load_weight(prefix + k, v)

    # ---------------------------------------------------------------------- GPT --
    def gpt_init(self, layers, model_dim, heads, number_mel_codes=8194, start_mel_token=8192,
                 stop_mel_token=8193, max_mel_positions=0, max_prompt=640, max_batch=1,
                 weights_bf16=True):
        cfg = GptConfig(layers, model_dim, heads, number_mel_codes, start_mel_token,
                        stop_mel_token, max_mel_positions, max_prompt, max_batch,
                        1 if weights_bf16 else 0)
        self._check(self.lib.idx_gpt_init(self.h, C.byref(cfg)), "idx_gpt_init")
        self.gpt_cfg = cfg

    def gpt_prepare_inputs(self, style, emo_vec, text_ids, lang: int):
        """prepare_gpt_inputs (gpt/model_v2.py:648-714): returns [3+L+2, D] float32 (numpy)."""
        dev_src = style if _is_cuda(style) else (emo_vec if _is_cuda(emo_vec) else None)
        style = _as_f32(style).reshape(-1)
        emo_vec = _as_f32(emo_vec).reshape(-1)
        if torch is not None and isinstance(text_ids, torch.Tensor):
            text_ids = text_ids.detach().cpu().numpy()       # a few dozen ids: the valid_mask below is host logic
        ids = np.ascontiguousarray(np.asarray(text_ids, dtype=np.int32).reshape(-1))
        # valid_mask of model_v2.py:674: start/stop text tokens inside the padded ids are dropped
        ids = np.ascontiguousarray(ids[(ids != 0) & (ids != 1)])
        D = self.gpt_cfg.model_dim
        out = _empty_like_src(dev_src, (3 + len(ids) + 2, D))
        self._check(self.lib.idx_gpt_prepare_inputs(self.h, _ptr(style), _ptr(emo_vec), _ptr(ids),
                                                    len(ids), int(lang), _ptr(out)),
                    "idx_gpt_prepare_inputs")
        return out

    def gpt_generate(self, prompts, max_new_tokens, repetition_penalty=10.0, do_sample=False,
                     num_beams=1, top_k=0, top_p=1.0, temperature=1.0, length_penalty=0.0,
                     seed=0, forbid_stop_before=0, forced_codes=None, return_logits=False, mel_pos_mode=0):
        """Mirror of UnifiedVoice.inference_speech → generate (gpt/model_v2.py:716-825).
        prompts: list of [S_i, D] float32 arrays (the [cond][text] embeddings, no padding).
        Returns list of int32 code arrays (stop token included when produced) and, optionally,
        the raw per-step fp32 logits."""
        n = len(prompts)
        V = self.gpt_cfg.number_mel_codes
        reqs = (GptRequest * n)()
        keep = []
        codes = [np.zeros(max_new_tokens, dtype=np.int32) for _ in range(n)]
        ncodes = [np.zeros(1, dtype=np.int32) for _ in range(n)]
        lshape = (max_new_tokens, V) if num_beams == 1 else (max_new_tokens, num_beams, V)
        logits = [np.zeros(lshape, dtype=np.float32) if return_logits else None for _ in range(n)]
        for i, pr in enumerate(prompts):
            pr = _as_f32(pr)
            keep.append(pr)
            reqs[i].prompt_emb = _ptr(pr)
            reqs[i].prompt_len = int(pr.shape[0])
            reqs[i].codes_out = _ptr(codes[i])
            reqs[i].n_codes_out = _ptr(ncodes[i])
            reqs[i].logits_out = _ptr(logits[i])
            if forced_codes is not None:
                fc = np.zeros(max_new_tokens, dtype=np.int32)
                src = np.asarray(forced_codes[i], dtype=np.int32)[:max_new_tokens]
                fc[:len(src)] = src
                keep.append(fc)
                reqs[i].forced_codes = _ptr(fc)
        sp = Sampling(int(do_sample), int(num_beams), int(top_k), float(top_p), float(temperature),
                      float(repetition_penalty), float(length_penalty), int(max_new_tokens),
                      int(seed), int(forbid_stop_before), int(mel_pos_mode))
        self._check(self.lib.idx_gpt_generate(self.h, reqs, n, C.byref(sp)), "idx_gpt_generate")
        out = [codes[i][: int(ncodes[i][0])].copy() for i in range(n)]
        if return_logits:
            if num_beams > 1:
                steps = self.gpt_last_timing()["steps"]
                return out, [logits[i][:steps] for i in range(n)]
            return out, [logits[i][: int(ncodes[i][0])] for i in range(n)]
        return out

    # ------------------------------------------------------- v1 / v1.5 GPT side (row a13) --
    def v1_cond_init(self, c: dict, n_latents=32):
        cfg = EmoConfig(*[c[k] for k in ("idim", "odim", "linear_units", "heads", "blocks", "cnn_kernel", "p_dim",
                                         "p_heads", "p_dim_head", "p_depth", "p_ff_mult", "model_dim")])
        self._check(self.lib.idx_v1_cond_init(self.h, C.byref(cfg), int(n_latents)), "idx_v1_cond_init")
        self.v1_cond_cfg, self._v1_nlat = cfg, int(n_latents)

    def v1_get_conditioning(self, mel):
        """UnifiedVoice.get_conditioning (gpt/model.py:493-503): mel [T, 100] → conds [32, model_dim]."""
        m = _as_f32(mel)
        out = np.empty((self._v1_nlat, self.v1_cond_cfg.model_dim), dtype=np.float32)
        self._check(self.lib.idx_v1_get_conditioning(self.h, _ptr(m), int(m.shape[0]), _ptr(out)), "idx_v1_get_conditioning")
        return out

    def gpt_prepare_inputs_v1(self, conds, text_ids):
        """prepare_gpt_inputs of v1 (gpt/model.py:597-660): [conds][start_text, text.., stop_text] rows."""
        cd = _as_f32(conds)
        ids = np.ascontiguousarray(np.asarray(text_ids, dtype=np.int32).reshape(-1))
        ids = np.ascontiguousarray(ids[(ids != 0) & (ids != 1)])
        out = np.empty((cd.shape[0] + len(ids) + 2, self.gpt_cfg.model_dim), dtype=np.float32)
        self._check(self.lib.idx_gpt_prepare_inputs_v1(self.h, _ptr(cd), int(cd.shape[0]), _ptr(ids), len(ids), _ptr(out)),
                    "idx_gpt_prepare_inputs_v1")
        return out

    def gpt_latents_v1(self, conds, text_ids, codes):
        """UnifiedVoice.forward(return_latent=True) (gpt/model.py:526-589) → latents [n_codes, model_dim]."""
        cd = _as_f32(conds)
        ids = np.ascontiguousarray(np.asarray(text_ids, dtype=np.int32).reshape(-1))
        cs = np.ascontiguousarray(np.asarray(codes, dtype=np.int32).reshape(-1))
        out = np.empty((len(cs), self.gpt_cfg.model_dim), dtype=np.float32)
        self._check(self.lib.idx_gpt_latents_v1(self.h, _ptr(cd), int(cd.shape[0]), _ptr(ids), len(ids), _ptr(cs), len(cs),
                                                _ptr(out)), "idx_gpt_latents_v1")
        return out

    def gpt_beam_trace(self, utterance=0, max_steps=4096, num_beams=3):
        """(parents [steps, m], tokens [steps, m], scores [steps, m], final_score) of the last beam-search call."""
        pt = np.zeros((max_steps, num_beams, 2), dtype=np.int32)
        sc = np.zeros((max_steps, num_beams), dtype=np.float32)
        steps, fs = C.c_int32(0), C.c_double(0)
        self._check(self.lib.idx_gpt_beam_trace(self.h, int(utterance), _ptr(pt), _ptr(sc), max_steps,
                                                C.byref(steps), C.byref(fs)), "idx_gpt_beam_trace")
        k = min(steps.value, max_steps)
        return pt[:k, :, 0].copy(), pt[:k, :, 1].copy(), sc[:k].copy(), fs.value

    def gpt_last_timing(self):
        t = (C.c_double * 4)()
        self._check(self.lib.idx_gpt_last_timing(self.h, t), "idx_gpt_last_timing")
        return {"prefill_ms": t[0], "decode_ms": t[1], "steps": int(t[2]), "launches": int(t[3])}

    def gpt_profile(self, enable=True, read=False):
        """Phase-boundary %globaltimer stamps (ns) of CTA 0 for the last step of the last launch."""
        buf = np.zeros(320, dtype=np.int64)
        self._check(self.lib.idx_gpt_profile(self.h, int(enable), _ptr(buf) if read else None, 320 if read else 0),
                    "idx_gpt_profile")
        return buf

    def gpt_profile_fine(self, num_sms=148):
        """[num_sms][64] sub-phase %globaltimer stamps (ns) of every CTA, middle layer of the last decode step."""
        buf = np.zeros((num_sms, 64), dtype=np.int64)
        self._check(self.lib.idx_gpt_profile_fine(self.h, _ptr(buf), buf.size), "idx_gpt_profile_fine")
        return buf

    # ------------------------------------------------------------------ BigVGAN --
    @staticmethod
    def _bigvgan_cfg(h: dict, num_mels):
        cfg = BigvganConfig()
        cfg.num_mels = num_mels
        cfg.upsample_initial_channel = h["upsample_initial_channel"]
        rates, ks = h["upsample_rates"], h["upsample_kernel_sizes"]
        cfg.num_upsamples = len(rates)
        for i, (r, k) in enumerate(zip(rates, ks)):
            cfg.upsample_rates[i] = r
            cfg.upsample_kernel_sizes[i] = k
        rk, rd = h["resblock_kernel_sizes"], h["resblock_dilation_sizes"]
        cfg.num_kernels = len(rk)
        for j, (k, ds) in enumerate(zip(rk, rd)):
            cfg.resblock_kernel_sizes[j] = k
            for m, d in enumerate(ds):
                cfg.resblock_dilations[j][m] = d
        cfg.use_tanh_at_final = int(h.get("use_tanh_at_final", True))
        cfg.use_bias_at_final = int(h.get("use_bias_at_final", True))
        cfg.snake_logscale = int(h.get("snake_logscale", True))
        return cfg

    def bigvgan_init(self, h: dict):
        cfg = self._bigvgan_cfg(h, h.get("num_mels", 80))
        self._check(self.lib.idx_bigvgan_init(self.h, C.byref(cfg)), "idx_bigvgan_init")
        self.bigvgan_cfg = cfg
        self._bigvgan_up = int(np.prod(h["upsample_rates"]))

    # ------------------------------------------------------- v1 / v1.5 vocoder (row a13) --
    def v1_vocoder_init(self, h: dict):
        """indextts/BigVGAN/models.py:129-199 — tensors registered under "bigvgan_v1."."""
        cfg = self._bigvgan_cfg(dict(h, use_tanh_at_final=True), h["gpt_dim"])
        self._check(self.lib.idx_v1_vocoder_init(self.h, C.byref(cfg), int(h["num_mels"]), int(h["speaker_embedding_dim"]),
                                                 int(h.get("cond_d_vector_in_each_upsampling_layer", True))),
                    "idx_v1_vocoder_init")
        self.v1_cfg = dict(h)
        self._v1_up = int(np.prod(h["upsample_rates"]))

    def v1_speaker_embedding(self, mel_ref):
        """ECAPA_TDNN.forward (ECAPA_TDNN.py:543-582): mel_ref [Tm, n_mels] → [speaker_embedding_dim]."""
        m = _as_f32(mel_ref)
        out = np.empty(self.v1_cfg["speaker_embedding_dim"], dtype=np.float32)
        self._check(self.lib.idx_v1_speaker_embedding(self.h, _ptr(m), int(m.shape[0]), _ptr(out)), "idx_v1_speaker_embedding")
        return out

    def v1_vocode(self, latent, mel_ref):
        """BigVGAN.forward(latent, mel_ref) (BigVGAN/models.py:201-249): latent [T, gpt_dim], mel_ref [Tm, n_mels] → wav [T*up]."""
        x, m = _as_f32(latent), _as_f32(mel_ref)
        out = np.empty(x.shape[0] * self._v1_up, dtype=np.float32)
        self._check(self.lib.idx_v1_vocode(self.h, _ptr(x), int(x.shape[0]), _ptr(m), int(m.shape[0]), _ptr(out)), "idx_v1_vocode")
        return out

    def bigvgan_forward(self, mel, out=None):
        """BigVGAN.forward (s2mel/modules/bigvgan/bigvgan.py:360-386): mel [B,80,F] f32 →
        wav [B,1,F*256] f32.  Accepts numpy (host) or torch (host/cuda) buffers."""
        mel = _as_f32(mel)
        B, _, F = mel.shape
        n = F * self._bigvgan_up
        if out is None:
            if torch is not None and isinstance(mel, torch.Tensor):
                out = torch.empty((B, 1, n), dtype=torch.float32, device=mel.device)
            else:
                out = np.empty((B, 1, n), dtype=np.float32)
        self._check(self.lib.idx_bigvgan_forward(self.h, _ptr(mel), B, F, _ptr(out)),
                    "idx_bigvgan_forward")
        return out

    def bigvgan_last_ms(self):
        t = C.c_double()
        self._check(self.lib.idx_bigvgan_last_ms(self.h, C.byref(t)), "idx_bigvgan_last_ms")
        return t.value

    def antialias_snake(self, x, alpha, beta, logscale=True):
        """Activation1d(SnakeBeta) (alias_free_activation/torch/act.py:8-30) on x [B,C,T]."""
        x = _as_f32(x)
        alpha, beta = _as_f32(alpha), _as_f32(beta)
        B, Cc, T = x.shape
        if torch is not None and isinstance(x, torch.Tensor):
            y = torch.empty_like(x)
        else:
            y = np.empty_like(x)
        self._check(self.lib.idx_antialias_snake(self.h, _ptr(x), _ptr(alpha), _ptr(beta), B, Cc, T,
                                                 int(logscale), _ptr(y)), "idx_antialias_snake")
        return y

    # ------------------------------------------------------------- s2mel + codec --
    def s2mel_init(self, c: dict):
        cfg = S2melConfig(c["hidden"], c["heads"], c["depth"], c["wn_hidden"], c["wn_layers"], c["wn_kernel"],
                          c["in_channels"], c["content_dim"], c["style_dim"], c["lr_in"], c["lr_convs"])
        self._check(self.lib.idx_s2mel_init(self.h, C.byref(cfg)), "idx_s2mel_init")
        self.s2mel_cfg = cfg

    def codec_init(self, c: dict):
        cfg = CodecConfig(c["codebook_size"], c["hidden_size"], c["codebook_dim"], c["vocos_dim"],
                          c["vocos_intermediate_dim"], c["vocos_num_layers"])
        self._check(self.lib.idx_codec_init(self.h, C.byref(cfg)), "idx_codec_init")
        self.codec_cfg = cfg

    def codec_decode(self, codes):
        """EnhancedCodec.decode (codec/models.py:205-231): codes [n] → S_infer [2n, hidden]."""
        if _is_cuda(codes):
            codes = codes.detach().reshape(-1).to(torch.int32).contiguous()
        else:
            codes = np.ascontiguousarray(np.asarray(codes, dtype=np.int32).reshape(-1))
        out = _empty_like_src(codes, (2 * int(codes.shape[0]), self.codec_cfg.hidden_size))
        self._check(self.lib.idx_codec_decode(self.h, _ptr(codes), int(codes.shape[0]), _ptr(out)), "idx_codec_decode")
        return out

    def length_regulate(self, S, ylen):
        """InterpolateRegulator.forward (length_regulator.py:90-141): S [n, in] → [ylen, C]."""
        S = _as_f32(S)
        out = _empty_like_src(S, (int(ylen), self.s2mel_cfg.content_dim))
        self._check(self.lib.idx_length_regulate(self.h, _ptr(S), int(S.shape[0]), int(ylen), _ptr(out)),
                    "idx_length_regulate")
        return out

    def dit_forward(self, x, prompt_x, t, style, cond):
        """DiT.forward (diffusion_transformer.py:186-257) for full-length sequences."""
        x, prompt_x, t, style, cond = (_as_f32(a) for a in (x, prompt_x, t, style, cond))
        B, _, T = x.shape
        out = _empty_like_src(x, (B, self.s2mel_cfg.in_channels, T))
        self._check(self.lib.idx_dit_forward(self.h, _ptr(x), _ptr(prompt_x), _ptr(t), _ptr(style), _ptr(cond),
                                             B, T, _ptr(out)), "idx_dit_forward")
        return out

    def cfm_solve(self, mu, prompt, style, z, n_steps=25, cfg_rate=0.7):
        """BASECFM.inference (flow_matching.py:30-115) with caller-supplied noise z [80, T]."""
        mu, prompt, style, z = (_as_f32(a) for a in (mu, prompt, style, z))
        T = mu.shape[0]
        P = prompt.shape[-1]
        out = _empty_like_src(z, (self.s2mel_cfg.in_channels, T))
        self._check(self.lib.idx_cfm_solve(self.h, _ptr(mu), T, _ptr(prompt), P, _ptr(style), _ptr(z),
                                           int(n_steps), float(cfg_rate), _ptr(out)), "idx_cfm_solve")
        return out

    def s2mel_last_ms(self):
        t = (C.c_double * 3)()
        self._check(self.lib.idx_s2mel_last_ms(self.h, t), "idx_s2mel_last_ms")
        return {"codec_ms": t[0], "length_regulator_ms": t[1], "cfm_ms": t[2]}

    def codes_to_wav(self, codes, prompt_condition, ref_mel, style, z, F, n_steps=25, cfg_rate=0.7,
                     want_wav=True, want_pcm16=False, want_mel=False, out=None):
        """infer_v2_5.py:827-856 for one segment.  Host or device (torch.cuda) buffers.
        Returns dict(wav=[F*256] f32, pcm16=..., mel=[80,F])."""
        on_dev = torch is not None and isinstance(z, torch.Tensor) and z.is_cuda
        if on_dev and isinstance(codes, torch.Tensor):
            codes_t = codes.to(torch.int32).contiguous()
        else:      # host codes are fine next to device buffers: every ABI pointer may be host or device
            codes_t = np.ascontiguousarray(np.asarray(codes, dtype=np.int32).reshape(-1))
        pc, rm, st, zz = (_as_f32(a) for a in (prompt_condition, ref_mel, style, z))
        P = int(rm.shape[-1])
        up = self._bigvgan_up
        res = {}

        def mk(shape, dtype_np, dtype_t):
            if on_dev:
                return torch.empty(shape, dtype=dtype_t, device=z.device)
            return np.empty(shape, dtype=dtype_np)
        if want_wav:
            res["wav"] = mk((F * up,), np.float32, torch.float32 if torch else None)
        if want_pcm16:
            res["pcm16"] = mk((F * up,), np.int16, torch.int16 if torch else None)
        if want_mel:
            res["mel"] = mk((80, F), np.float32, torch.float32 if torch else None)
        r = VocodeRequest(_ptr(codes_t), int(codes_t.shape[0]), _ptr(pc), _ptr(rm), P, _ptr(st), _ptr(zz), int(F),
                          _ptr(res.get("wav")), _ptr(res.get("pcm16")), _ptr(res.get("mel")))
        self._check(self.lib.idx_codes_to_wav(self.h, C.byref(r), int(n_steps), float(cfg_rate)), "idx_codes_to_wav")
        return res

    # --------------------------------------------------------------- diagnostics --
    def debug_conv_gemm(self, A, wk, taps=1, dil=1, pad=0, M=None, bias=None, act=0, res=None, accum=False,
                        scale=1.0, out_off=0, ldo=None, out_valid=None, out_rows=None, backend=0, out_init=None,
                        biasN=0):
        """One channels-last multi-tap GEMM through a chosen back end (1 SIMT, 2 tcgen05)."""
        A = np.ascontiguousarray(A, dtype=np.float32)
        wk = np.ascontiguousarray(wk, dtype=np.float32)
        B, Tin, K = A.shape
        N = wk.shape[0]
        M = Tin if M is None else M
        ldo = N if ldo is None else ldo
        out_rows = M if out_rows is None else out_rows
        per = out_rows * ldo if out_valid is None else int(out_valid)
        out_valid = per
        out = np.zeros((B, per), dtype=np.float32) if out_init is None else np.ascontiguousarray(out_init, dtype=np.float32).reshape(B, per).copy()
        b_ = None if bias is None else np.ascontiguousarray(bias, dtype=np.float32)
        r_ = None if res is None else np.ascontiguousarray(res, dtype=np.float32).reshape(B, per)
        self._check(self.lib.idx_debug_conv_gemm(self.h, _ptr(A), B, Tin, K, _ptr(wk), taps, dil, pad, M, N, _ptr(b_),
                                                 biasN, act, _ptr(r_), int(accum), float(scale), int(out_off), ldo,
                                                 int(out_valid), int(per), int(backend), _ptr(out)),
                    "idx_debug_conv_gemm")
        return out

    def debug_gemm_pair_epilogue(self, A, wk, epi, taps=1, dil=1, pad=0, M=None, bias=None, aux=None, aux_stride=0,
                                 scale=1.0):
        """fp16 tensor-core GEMM with a fused pair epilogue (1 SwiGLU, 2 WaveNet gate, 3 RoPE; aux_stride = heads).
        A [B][Tin][K] and wk [N][taps*K] in fp32, module row order.  Returns float16: [B][M][N/2] for epi 1 / 2, and
        Qr | Kr | Vb as [3][B*H][M][64] for epi 3."""
        A = np.ascontiguousarray(A, dtype=np.float32)
        wk = np.ascontiguousarray(wk, dtype=np.float32)
        B, Tin, K = A.shape
        N = wk.shape[0]
        M = Tin if M is None else M
        b_ = None if bias is None else np.ascontiguousarray(bias, dtype=np.float32)
        g_ = None if aux is None else np.ascontiguousarray(aux, dtype=np.float32)
        if epi == 3:
            H = max(int(aux_stride), 1)
            out = np.zeros((3, B * H, M, 64), np.float16) if N == 192 * H else np.zeros(B * M * N, np.float16)
        else:
            out = np.zeros((B, M, max(N // 2, 1)), np.float16)
        self._check(self.lib.idx_debug_gemm_pair_epilogue(self.h, _ptr(A), B, Tin, K, _ptr(wk), taps, dil, pad, M, N,
                                                          _ptr(b_), int(epi), _ptr(g_), int(aux_stride), float(scale),
                                                          _ptr(out)),
                    "idx_debug_gemm_pair_epilogue")
        return out

    def debug_flash_attention(self, qkv16, B, T, H, kernel, want_out=True, want_out16=True):
        """Flash attention on fp16 Qr | Kr | Vb ([3][B*H][T][64]) through kernel 1 (mma.sync) or 2 (tcgen05).
        Returns (out f32 [B][T][H*64] or None, out16 float16 [B][T][H*64] or None)."""
        q = np.ascontiguousarray(qkv16, dtype=np.float16)
        assert q.size == 3 * B * H * T * 64
        out = np.zeros((B, T, H * 64), np.float32) if want_out else None
        out16 = np.zeros((B, T, H * 64), np.float16) if want_out16 else None
        self._check(self.lib.idx_debug_flash_attention(self.h, _ptr(q), B, T, H, int(kernel), _ptr(out), _ptr(out16)),
                    "idx_debug_flash_attention")
        return out, out16

    def debug_attention_rope(self, qkv, H, backend):
        """The DiT attention with RoPE on fp32 qkv [B][T][3*H*64]: backend 1 SIMT fp32, 0 fp16 mma.sync flash."""
        qkv = np.ascontiguousarray(qkv, dtype=np.float32)
        B, T, _ = qkv.shape
        out = np.zeros((B, T, H * 64), np.float32)
        self._check(self.lib.idx_debug_attention_rope(self.h, _ptr(qkv), B, T, H, int(backend), _ptr(out)),
                    "idx_debug_attention_rope")
        return out

    # ------------------------------------------------------------------- emotion --
    def emo_init(self, c: dict):
        cfg = EmoConfig(*[c[k] for k in ("idim", "odim", "linear_units", "heads", "blocks", "cnn_kernel", "p_dim",
                                         "p_heads", "p_dim_head", "p_depth", "p_ff_mult", "model_dim")])
        self._check(self.lib.idx_emo_init(self.h, C.byref(cfg)), "idx_emo_init")
        self.emo_cfg = cfg

    def merge_emovec(self, spk_feats, emo_feats=None, alpha=1.0):
        """UnifiedVoice.merge_emovec (gpt/model_v2.py:833-838): feats [T, 1024] → emo_vec [model_dim]."""
        sf = _as_f32(spk_feats)
        ef = None if emo_feats is None else _as_f32(emo_feats)
        out = _empty_like_src(sf, (self.emo_cfg.model_dim,))
        self._check(self.lib.idx_merge_emovec(self.h, _ptr(sf), int(sf.shape[0]), _ptr(ef),
                                              0 if ef is None else int(ef.shape[0]), float(alpha), _ptr(out)),
                    "idx_merge_emovec")
        return out
