#!/usr/bin/env python
"""bench.py — the IndexTTS-2.5 per-segment hot path on B200 (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--quick] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One "step" = one utterance through the whole per-segment pipeline of IndexTTS2.infer
(infer_v2_5.py:749-864): prompt embeddings → GPT prefill + 256 greedy speech tokens (stop masked
until step 256, repetition_penalty 10) → semantic-codec decode → length regulator (F = 880) →
cat 10 s reference (P = 861) → CFM 25 Euler steps, CFG 0.7 (T = 1741) → BigVGAN (225 280 samples,
10.22 s of 22.05 kHz audio) → pcm16.  Speaker conditioning (w2v-BERT / CAMPPlus / mel of the
reference audio, SURVEY §8f "next") and the emotion vector are cached per speaker exactly as the
reference caches them (infer_v2_5.py:620-667; trap P11) and are inputs here.

Metric: whole-job speech-tokens/s (higher is better) with RTF alongside.  `value` is measured with
all inputs resident in HBM; `e2e` through the same public API with HOST buffers (H2D of the
request, D2H of codes + pcm16 inside the timed region).  Synthetic seeded weights at the
[ASSUMED] IndexTTS-2.5 shapes (no checkpoints offline) — `data: synthetic`.

N > 1: one process per GPU, utterances shard embarrassingly (weak scaling); NCCL broadcasts the
speaker latents once and gathers the finished pcm16 waveforms on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_TOKENS = 256
P_FRAMES = 861          # 10 s reference at 22.05 kHz / hop 256
N_TEXT = 32
CFM_STEPS, CFG_RATE = 25, 0.7
AUDIO_S_PER_TOKEN = 2 * 1.72 * 256 / 22050.0


def ncu_traffic():
    """DRAM bytes per decode step of the dominant kernel, from the committed ncu capture summary (tests/tools/ncu_metrics.py
    turns the .ncu-rep of `ncu --set full` into this JSON); null when no capture has been committed for this kernel."""
    p = os.path.join(ROOT, "profiles", "r02_gpt_decode1_ncu.json")
    try:
        d = json.load(open(p))
        return float(d["dram_bytes_per_step"]), (f"dram__bytes_read.sum + dram__bytes_write.sum of one gpt_decode1_kernel launch / "
                                                 f"{d['steps_per_launch']} steps, ncu --set full, profiles/r02_gpt_decode1_ncu.json")
    except Exception:
        return None, "no committed ncu capture of this kernel"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
                for nm, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------- workload --
def make_inputs(seed, cfg_gpt, w_gpt):
    """Synthetic request of the named shape; conditioning tensors are what the reference caches."""
    from indextts_b200.synth import r16
    g = torch.Generator().manual_seed(seed)
    style = torch.randn(192, generator=g)
    emo = r16(torch.randn(cfg_gpt["model_dim"], generator=g) * 0.5)
    text = torch.randint(2, 12000, (N_TEXT,), generator=g)
    prompt_condition = torch.randn(P_FRAMES, 512, generator=g)
    ref_mel = torch.randn(80, P_FRAMES, generator=g) * 1.5 - 4.0
    F = int(2 * N_TOKENS * 1.72)
    z = torch.randn(80, P_FRAMES + F, generator=g)     # the cfm.inference noise (trap P6)
    return dict(style=style, emo=emo, text=text, prompt_condition=prompt_condition, ref_mel=ref_mel, z=z, F=F)


def build_engine(device, max_batch=1):
    from indextts_b200.engine import Engine, fold_weight_norm
    from indextts_b200 import synth
    t0 = time.time()
    e = Engine(device)
    cfg = synth.gpt_config()
    wg = synth.make_gpt_weights(cfg, seed=2025, bf16=True)
    e.load_state_dict("gpt.", wg)
    e.gpt_init(cfg["layers"], cfg["model_dim"], cfg["heads"], cfg["number_mel_codes"], cfg["start_mel_token"],
               cfg["stop_mel_token"], cfg["max_mel_positions"], max_prompt=80 if max_batch > 1 else 64, max_batch=max_batch, weights_bf16=True)
    c, cc = dict(synth.S2MEL_CFG), dict(synth.CODEC_CFG)
    ws = fold_weight_norm(synth.make_s2mel_weights(c, seed=1234))
    e.load_state_dict("s2mel.", {k: v for k, v in ws.items() if v.is_floating_point()})
    e.load_state_dict("codec.", fold_weight_norm(synth.make_codec_weights(cc, seed=4321)))
    e.s2mel_init(c)
    e.codec_init(cc)
    h = dict(synth.BIGVGAN_V2_22K)
    e.load_state_dict("bigvgan.", synth.make_bigvgan_weights(h, seed=1234))
    e.bigvgan_init(h)
    return e, cfg, wg, time.time() - t0


def run_utterance(e, inp, prompt_emb, host: bool):
    """The public-API call sequence of one segment.  host=True: numpy inputs/outputs (H2D/D2H inside)."""
    (codes,) = e.gpt_generate([prompt_emb], N_TOKENS, 10.0, forbid_stop_before=N_TOKENS)
    if host:
        res = e.codes_to_wav(codes, inp["prompt_condition"], inp["ref_mel"], inp["style"], inp["z"], inp["F"],
                             CFM_STEPS, CFG_RATE, want_wav=False, want_pcm16=True)
    else:
        dcodes = torch.from_numpy(codes).to(inp["z_d"].device)
        res = e.codes_to_wav(dcodes, inp["pc_d"], inp["mel_d"], inp["style_d"], inp["z_d"], inp["F"],
                             CFM_STEPS, CFG_RATE, want_wav=False, want_pcm16=True)
    return codes, res["pcm16"]


DUMP_LIMIT_BYTES = 64 << 20
PCM_SAMPLE = 1 << 20      # samples kept of a job's concatenated pcm16 (a whole config-5 job has ~1e8)


def dump_outputs(out_dir, arrays):
    """`--dump-outputs`: one DIR/<name>.npy per array, float32 or float64 (codes and pcm16 are integers, exact in
    either), so that two builds of the project can be compared output for output on the same seeded inputs."""
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, f"dump of {total} bytes exceeds {DUMP_LIMIT_BYTES}"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def stage_breakdown(e):
    g = e.gpt_last_timing()
    s = e.s2mel_last_ms()
    return g, s


WORKLOAD = ("IndexTTS-2.5 infer_v2_5 batch=1 per GPU: 10 s reference (P=861), 32 text tokens, "
            "256 greedy speech tokens, codec->length-regulator->CFM 25 steps CFG 0.7 (T=1741)->BigVGAN "
            "(225280 samples); speaker/emotion conditioning cached per speaker as in the reference")


# -------------------------------------------------------------------------- cpu arm --
DTYPE = ("bf16 GPT (bf16 weights/activations, fp32 accumulate, fp32 residual stream = the reference's use_bf16 autocast) + "
         "tail on tcgen05 with fp16 operands (kind::f16: DiT / WaveNet / BigVGAN-resblock GEMMs and the DiT flash attention; "
         "fp32 accumulate, fp32 softmax, fp32 residual streams and pointwise math) and tf32 over fp32 storage for the small "
         "rest (codec, length regulator, K=80 input convs, ConvTranspose upsamplers)")


def config_block(world):
    """Identical for both arms: the driver compares it to decide `same_config`."""
    return {"workload": WORKLOAD, "utterances_per_gpu_per_step": 1,
            "parallelism": f"dp{world} (utterance sharding)" if world > 1 else "dp1",
            "l2": "working set >> L2 (0.97 GB of GPT weights streamed per token, 112 M vocoder weights)"}


def cpu_reference_full(threads):
    """The reference's per-segment path restated by the oracle port, on the host cores, at the FULL config-2 size
    (the same WORKLOAD the GPU arm times): fp32 like the reference on a CPU (use_bf16 needs CUDA autocast),
    GPT prefill + 256 cached greedy steps at 24 x 1280, codec decode, length regulator (F = 880), CFM 25 Euler steps
    CFG 0.7 at T = 1741, BigVGAN 225 280 samples.  Returns a callable that runs one utterance and returns
    (seconds, per-stage seconds)."""
    from indextts_b200 import synth
    from oracle.gpt import GptOracle, prepare_gpt_inputs
    from oracle.s2mel import cfm_inference, codec_decode, fold_weight_norm, length_regulate
    from oracle.bigvgan import bigvgan_forward
    torch.set_num_threads(threads)
    cfg = synth.gpt_config()
    wg = synth.make_gpt_weights(cfg, seed=2025, bf16=False)
    c, cc, h = dict(synth.S2MEL_CFG), dict(synth.CODEC_CFG), dict(synth.BIGVGAN_V2_22K)
    ws = fold_weight_norm(synth.make_s2mel_weights(c, seed=1234))
    wc = fold_weight_norm(synth.make_codec_weights(cc, seed=4321))
    wb = synth.make_bigvgan_weights(h, seed=1234)
    inp = make_inputs(1000, cfg, wg)
    prompt = prepare_gpt_inputs(wg, inp["style"], inp["emo"], inp["text"], lang=1, bf16=False)
    F = inp["F"]
    pc, ref_mel, z = inp["prompt_condition"][None], inp["ref_mel"][None], inp["z"][None]
    oracle = GptOracle(cfg, wg, bf16=False)

    def once():
        t0 = time.perf_counter()
        with torch.no_grad():
            codes, _ = oracle.generate(prompt, N_TOKENS, 10.0, N_TOKENS)
            assert len(codes) == N_TOKENS
            t1 = time.perf_counter()
            S = codec_decode(wc, torch.from_numpy(np.asarray(codes, dtype=np.int64))[None])
            cond = length_regulate(ws, S, F)
            mu = torch.cat([pc, cond], 1)
            mel = cfm_inference(ws, c, mu, torch.LongTensor([P_FRAMES + F]), ref_mel, inp["style"][None], z, CFM_STEPS, CFG_RATE)
            t2 = time.perf_counter()
            wav = bigvgan_forward(h, wb, mel[:, :, P_FRAMES:])
            assert wav.shape[-1] == F * 256
        t3 = time.perf_counter()
        return t3 - t0, {"gpt": t1 - t0, "s2mel": t2 - t1, "bigvgan": t3 - t2}
    return once


def host_threads():
    """Threads for the CPU arm: the cores this process may run on (cgroup / affinity aware), at most 32 — the r1/r2 boxes
    showed 64 torch threads on a 128-logical-core host SLOWER than 8 real cores for this workload."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return max(1, min(n, 32))


def run_reference(args, rank, world):
    """`--impl reference`: the reference's own (CPU, fp32) implementation of the path — the oracle port; the reference
    itself cannot be built offline (DESIGN.md section 6) — on the box's host cores, SAME config, metric and unit as the
    B200 arm.  Every step is the FULL config-2 utterance (~1 minute of CPU work), so --steps / --warmup are honoured only
    as far as IDX_REF_BUDGET_S allows (default 300 s: "the whole run ends within a few minutes"); the line reports the
    steps that actually ran and says that the request was cut."""
    if rank != 0:
        return
    threads = host_threads()
    once = cpu_reference_full(threads)
    budget = float(os.environ.get("IDX_REF_BUDGET_S", "300"))
    t_start = time.perf_counter()
    W, K = max(0, args.warmup), max(1, args.steps)
    t_first, _ = once()                                   # first warm-up step doubles as the cost probe
    fit = int((budget - (time.perf_counter() - t_start)) / max(t_first, 1e-3))
    w_run = 1
    if W == 0:
        ts, stages = [t_first], [_]
        k_run, w_run = 1, 0
    else:
        w_left = max(0, min(W - 1, fit - 1))
        for _i in range(w_left):
            once()
        w_run += w_left
        fit = int((budget - (time.perf_counter() - t_start)) / max(t_first, 1e-3))
        k_run = max(1, min(K, fit))
        ts, stages = [], []
        for _i in range(k_run):
            t, st = once()
            ts.append(t)
            stages.append(st)
    t = float(np.mean(ts))
    val = N_TOKENS / t
    audio_s = N_TOKENS * AUDIO_S_PER_TOKEN
    sample = (f"the full config-2 utterance per step ({N_TOKENS} speech tokens, P={P_FRAMES}, T={P_FRAMES + int(2 * N_TOKENS * 1.72)}, "
              f"CFM {CFM_STEPS} steps, {int(2 * N_TOKENS * 1.72) * 256} samples): oracle port, torch CPU fp32, {threads} threads of "
              f"{os.cpu_count()} host cores; {k_run} timed + {w_run} warm-up steps"
              + ("" if (k_run == K and w_run == W) else f" (requested {K} + {W}: cut to fit {budget:.0f} s)"))
    line = {"impl": "reference", "metric": "speech_tokens_per_s", "value": val, "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": k_run, "warmup": w_run, "ms_per_step": t * 1000, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "rtf": t / audio_s,
            "config": config_block(world),
            "stage_ms_per_step": {k: float(np.mean([st[k] for st in stages])) * 1000 for k in ("gpt", "s2mel", "bigvgan")},
            "cpu_baseline": {"value": val, "unit": "tokens/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------- batch jobs: BASELINE configs 3 and 5 --
JOBS = {
    "config3": ("IndexTTS-2.5 batch=32 on one GPU per rank-share: 32 utterances of one speaker, 512 speech tokens each, full "
                "gpt->codec->length-regulator->CFM 25 steps (T=861+1761)->BigVGAN pipeline"),
    "config5": ("IndexTTS-2.5 batch=256 mixed-length utterances (speech tokens U[128,768], seed 0; 4 speakers, 10 s references) "
                "sharded over the ranks by longest-processing-time-first; NCCL broadcast of the speaker latents, gather of the wavs"),
}


def make_job(name):
    """The fixed utterance list of a batch workload: (n_tokens, speaker, text_len) per utterance, seeded."""
    g = torch.Generator().manual_seed(0)
    if name == "config3":
        n, toks, spk = 32, [512] * 32, [0] * 32
    else:
        n = 256
        toks = [int(x) for x in torch.randint(128, 769, (n,), generator=g)]
        spk = [i % 4 for i in range(n)]
    tl = [int(x) for x in torch.randint(24, 61, (n,), generator=g)]
    return [dict(idx=i, n=toks[i], spk=spk[i], L=tl[i]) for i in range(n)]


def run_job(args, rank, world, local):
    """`--workload config3|config5` as the whole run: sets up the process group and the engine, runs the job, prints its line."""
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
    if rank != 0:
        ge.build()
    e, cfg, wg, t_load = build_engine(local, max_batch=8)
    outputs = {} if args.dump_outputs else None
    line = job_line(args.workload, e, cfg, wg, dist, rank, world, local, outputs)
    if rank == 0:
        print(json.dumps(line))
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
    if dist is not None:
        dist.destroy_process_group()


def job_line(workload, e, cfg, wg, dist, rank, world, local, outputs=None):
    """The whole fixed job once (after a warm-up mini-job), strong scaling over the ranks; returns the JSON line on rank 0.
    GPT decodes up to 8 utterances per group (sorted by length so a group's rows finish together; a row that reached its
    own length keeps decoding until the group's longest is done — those extra tokens are not counted); the tail runs
    per utterance.  Reports useful speech-tokens/s and RTF of the whole job, per-stage device time and the per-rank
    busy time (LPT imbalance).  `outputs` (a dict) receives this rank's results of the timed job: the codes of its
    utterances in utterance order, concatenated, and a seeded sample of their concatenated pcm16."""
    from indextts_b200.sharding import broadcast_latents, gather_wavs, lpt_assign
    dev = torch.device("cuda", local)
    job = make_job(workload)
    nspk = 1 + max(u["spk"] for u in job)
    # speaker latents: made on rank 0, broadcast once per speaker
    lats = []
    for sp in range(nspk):
        inp = make_inputs(100 + sp, cfg, wg)
        lat = {k: inp[k].to(dev).contiguous() for k in ("prompt_condition", "ref_mel", "style", "emo")}
        if dist is not None:
            broadcast_latents(dist, lat, src=0)
        lats.append(lat)
    share = lpt_assign([u["n"] for u in job], world)[rank]
    mine = sorted((job[i] for i in share), key=lambda u: -u["n"])
    gtxt = torch.Generator().manual_seed(1234)
    texts = {u["idx"]: torch.randint(2, 12000, (u["L"],), generator=torch.Generator().manual_seed(5000 + u["idx"])) for u in job}
    gz = torch.Generator(device=dev).manual_seed(77 + rank)

    def process(utts):
        t_g = t_c = t_v = 0.0
        wavs, kept, ntok = [], [], 0
        for g0 in range(0, len(utts), 8):
            grp = utts[g0:g0 + 8]
            prompts = [e.gpt_prepare_inputs(lats[u["spk"]]["style"], lats[u["spk"]]["emo"], texts[u["idx"]], 1) for u in grp]
            nmax = max(u["n"] for u in grp)
            outs = e.gpt_generate(prompts, nmax, 10.0, forbid_stop_before=nmax)
            t = e.gpt_last_timing()
            t_g += t["prefill_ms"] + t["decode_ms"]
            for u, codes in zip(grp, outs):
                n = u["n"]
                F = int(2 * n * 1.72)
                lat = lats[u["spk"]]
                z = torch.randn(80, P_FRAMES + F, device=dev, generator=gz)          # cfm.inference draws it per utterance (P6)
                res = e.codes_to_wav(np.minimum(codes[:n], 8191), lat["prompt_condition"], lat["ref_mel"], lat["style"], z, F,
                                     CFM_STEPS, CFG_RATE, want_wav=False, want_pcm16=True)
                t_c += e.s2mel_last_ms()["cfm_ms"]
                t_v += e.bigvgan_last_ms()
                wavs.append(res["pcm16"])
                kept.append(codes[:n])
                ntok += n
        return wavs, kept, ntok, (t_g, t_c, t_v)

    def barrier():
        e.sync()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    process([dict(u, n=64) for u in mine[:3]])                  # warm-up mini-job (allocations, NCCL channels)
    if dist is not None:
        gather_wavs(dist, torch.zeros(16, dtype=torch.int16, device=dev), rank, world, dst=0)
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    l0 = e.launches
    t0 = time.perf_counter()
    wavs, kept, ntok, (t_g, t_c, t_v) = process(mine)
    e.sync()
    torch.cuda.synchronize()
    t_busy = time.perf_counter() - t0
    if dist is not None:
        gather_wavs(dist, torch.cat([w.reshape(-1) for w in wavs]) if wavs else torch.zeros(0, dtype=torch.int16, device=dev), rank, world, dst=0)
    barrier()
    t_job = time.perf_counter() - t0
    clocks = sampler.stop()
    launches = e.launches - l0
    if outputs is not None and mine:
        order = sorted(range(len(mine)), key=lambda i: mine[i]["idx"])
        pcm = torch.cat([wavs[i].reshape(-1) for i in order])
        sel = np.sort(np.random.default_rng(0).integers(0, pcm.numel(), min(PCM_SAMPLE, pcm.numel())))
        outputs["codes"] = np.concatenate([kept[i] for i in order]).astype(np.float64)
        outputs["pcm16_sample"] = pcm[torch.from_numpy(sel).to(dev)].float().cpu().numpy()
    stats = torch.tensor([t_job, t_busy, t_g, t_c, t_v, float(ntok), float(launches)], device=dev, dtype=torch.float64)
    if dist is not None:
        allst = [torch.zeros_like(stats) for _ in range(world)]
        dist.all_gather(allst, stats)
    else:
        allst = [stats]
    if rank == 0:
        A = torch.stack(allst).cpu().numpy()
        t = float(A[:, 0].max())
        tokens = int(A[:, 5].sum())
        audio_s = tokens * AUDIO_S_PER_TOKEN
        line = {"metric": "speech_tokens_per_s", "value": tokens / t, "unit": "tokens/s", "n_gpus": world, "steps": 1, "warmup": 1,
                "ms_per_step": t * 1000, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": DTYPE,
                "data": "synthetic", "rtf": t / audio_s,
                "config": {"workload": JOBS[workload], "utterances": len(job), "speech_tokens": tokens, "audio_s": audio_s,
                           "parallelism": f"dp{world} (LPT utterance sharding)", "gpt_rows_per_group": 8,
                           "l2": "working set >> L2"},
                "per_rank": {"busy_s": [float(x) for x in A[:, 1]], "gpt_s": [float(x) / 1000 for x in A[:, 2]],
                             "cfm_s": [float(x) / 1000 for x in A[:, 3]], "bigvgan_s": [float(x) / 1000 for x in A[:, 4]],
                             "tokens": [int(x) for x in A[:, 5]]},
                "lpt_imbalance": float(A[:, 1].max() / max(A[:, 1].mean(), 1e-9)),
                "e2e": {"value": tokens / t, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                        "note": "device-resident latents; codes cross the host once per group; pcm16 gathered on rank 0 over NCCL"},
                "gpu_launches": int(A[:, 6].sum()), "clocks": clocks}
        return line
    return None


# ---------------------------------------------------------------------------- main --
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config5", action="store_true", help="skip the config-5 job block of the default run")
    ap.add_argument("--workload", default="config2", choices=["config2", "config3", "config5"],
                    help="config2 (default): the batch-1 headline; config3 / config5: the fixed batch jobs, run once")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32 / "
                         "float64, <= 64 MB): codes and pcm16 of the headline utterance and, when it runs, codes and a "
                         "seeded pcm16 sample of the batch job; rank 0's results")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the B200 path computed; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload != "config2":
        run_job(args, rank, world, local)
        return
    W = max(3, args.warmup)
    K = args.steps

    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
    if rank != 0:
        ge.build()
    dev = torch.device("cuda", local)
    e, cfg, wg, t_load = build_engine(local, max_batch=8)      # one engine serves the batch-1 line and the config-5 job

    # speaker latents: produced on rank 0, broadcast over NCCL (north-star multi-GPU plumbing)
    inp = make_inputs(100, cfg, wg)
    lat = {k: inp[k].to(dev).contiguous() for k in ("prompt_condition", "ref_mel", "style", "emo")}
    if dist is not None:
        from indextts_b200.sharding import broadcast_latents
        broadcast_latents(dist, lat, src=0)
    # per-rank utterance: own text and noise
    mine = make_inputs(1000 + rank, cfg, wg)
    mine.update({k: lat[k].cpu() for k in lat})
    prompt_emb = e.gpt_prepare_inputs(mine["style"].numpy(), mine["emo"].numpy(), mine["text"].numpy(), 1)
    mine["pc_d"], mine["mel_d"], mine["style_d"] = lat["prompt_condition"], lat["ref_mel"], lat["style"]
    mine["z_d"] = mine["z"].to(dev).contiguous()
    prompt_emb_d = torch.from_numpy(prompt_emb).to(dev)
    host_in = {k: np.ascontiguousarray(mine[k].numpy()) for k in ("prompt_condition", "ref_mel", "style", "z")}
    host_in["F"] = mine["F"]

    def barrier():
        e.sync()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    # ---- device-resident timing ----
    for _ in range(W):
        codes, pcm = run_utterance(e, mine, prompt_emb_d, host=False)
    assert len(codes) == N_TOKENS and pcm.shape[0] == mine["F"] * 256
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    l0 = e.launches
    e.event_record(0)
    g_ms = c_ms = v_ms = 0.0
    gpt_launch_ms, gpt_launches = 0.0, 0
    for _ in range(K):
        codes, pcm = run_utterance(e, mine, prompt_emb_d, host=False)
        g, s = stage_breakdown(e)
        g_ms += g["prefill_ms"] + g["decode_ms"]
        gpt_launch_ms += g["decode_ms"]
        gpt_launches += max(1, g["launches"] - 1)
        c_ms += s["cfm_ms"]
        v_ms += e.bigvgan_last_ms()
    e.event_record(1)
    barrier()
    clocks = sampler.stop()
    t_dev = e.event_elapsed_ms(0, 1) / 1000.0
    launches = e.launches - l0
    outputs = {"codes": codes.astype(np.float64), "pcm16": pcm.float().cpu().numpy()} if args.dump_outputs else None
    # ---- end to end: host buffers in, pcm16 out, gather on rank 0 ----
    if dist is not None:
        from indextts_b200.sharding import gather_wavs
    for _ in range(2):
        _, pcm_w = run_utterance(e, host_in, prompt_emb, host=True)
        if dist is not None:      # warm the gather too: NCCL sets its point-to-point channels up on first use
            gather_wavs(dist, torch.from_numpy(pcm_w).to(dev), rank, world, dst=0)
    barrier()
    t0 = time.perf_counter()
    e.event_record(2)
    for _ in range(K):
        codes_h, pcm_h = run_utterance(e, host_in, prompt_emb, host=True)
        if dist is not None:
            gather_wavs(dist, torch.from_numpy(pcm_h).to(dev), rank, world, dst=0)
    e.event_record(3)
    barrier()
    t_e2e_wall = time.perf_counter() - t0
    t_e2e = max(e.event_elapsed_ms(2, 3) / 1000.0, 0.0)
    t_e2e = max(t_e2e, t_e2e_wall if dist is None else t_e2e)
    h2d = int(prompt_emb.nbytes + sum(host_in[k].nbytes for k in ("prompt_condition", "ref_mel", "style", "z")) + N_TOKENS * 4)
    d2h = int(N_TOKENS * 4 + mine["F"] * 256 * 2)

    if dist is not None:
        t = torch.tensor([t_dev, t_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_dev, t_e2e = float(t[0]), float(t[1])
    # BASELINE config 5 (the fixed 256-utterance mixed-length job, strong scaling over the ranks) measured in the same run,
    # after the timed regions of the headline: reported as an extra block, the headline stays config 2 (VERDICT r1 item 6)
    job5 = None
    if not args.no_config5:
        job_out = {} if outputs is not None else None
        job5 = job_line("config5", e, cfg, wg, dist, rank, world, local, job_out)
        if job_out:
            outputs.update({"config5_" + k: v for k, v in job_out.items()})
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    tokens = world * K * N_TOKENS
    value = tokens / t_dev
    audio_s = N_TOKENS * AUDIO_S_PER_TOKEN
    hbm_peak, tc_peak, which = peaks()
    # roofline of the dominant HBM-bound kernel: the fused GPT decode step (DESIGN.md §kernels)
    L, D, V = cfg["layers"], cfg["model_dim"], cfg["number_mel_codes"]
    w_bytes = (L * (12 * D * D) + D * V) * 2                       # streamed bf16 weights per step
    ctx = 3 + N_TEXT + 2 + 1 + N_TOKENS / 2.0                      # mean context over the decode
    kv_bytes = 2 * L * ctx * D * 2 + 2 * L * D * 2
    step_us = gpt_launch_ms / (K * N_TOKENS) * 1000.0
    achieved = (w_bytes + kv_bytes) / (step_us * 1e-6) / 1e9
    cfm_flop = CFM_STEPS * 0.64e12
    line = {
        "metric": "speech_tokens_per_s", "value": value, "unit": "tokens/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": t_dev / K * 1000.0, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": DTYPE, "data": "synthetic",
        "rtf": (t_dev / K) / audio_s, "e2e_rtf": (t_e2e / K) / audio_s,
        "config": config_block(world),
        "stage_ms_per_step": {"gpt": g_ms / K, "cfm": c_ms / K, "bigvgan": v_ms / K,
                              "other": (t_dev * 1000 - g_ms - c_ms - v_ms) / K},
        "roofline": {"kernel": "gpt_decode1_kernel (one decode step of the batch-1 decode kernel)", "bound": "hbm", "achieved": achieved, "peak": hbm_peak,
                     "unit": "GB/s", "frac": achieved / hbm_peak,
                     "traffic": ncu_traffic()[0], "traffic_note": ncu_traffic()[1],
                     "peak_source": which,
                     "us_per_decode_step": step_us,
                     "algorithmic_bytes_per_step": w_bytes + kv_bytes},
        "roofline_cfm": {"bound": "tensor", "achieved": cfm_flop / (c_ms / K * 1e-3) / 1e12, "peak": tc_peak,
                         "unit": "TFLOP/s", "frac": cfm_flop / (c_ms / K * 1e-3) / 1e12 / tc_peak,
                         "note": "0.64 TFLOP per Euler step at T=1741 (SURVEY §8d); peak is the bf16 figure"},
        "roofline_bigvgan": {"bound": "tensor", "achieved": 1.8037e9 * mine["F"] / (v_ms / K * 1e-3) / 1e12, "peak": tc_peak,
                             "unit": "TFLOP/s", "frac": 1.8037e9 * mine["F"] / (v_ms / K * 1e-3) / 1e12 / tc_peak,
                             "note": "1.8037 GFLOP per mel frame (SURVEY §8d)"},
        "e2e": {"value": tokens / t_e2e, "unit": "tokens/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches), "clocks": clocks, "weights_load_s": t_load,
    }
    if job5 is not None:
        line["config5"] = {k: job5[k] for k in ("value", "unit", "scaling", "rtf", "ms_per_step", "config", "per_rank", "lpt_imbalance",
                                                "gpu_launches")}
    if not args.no_cpu_baseline and world == 1:          # the CPU leg is reported at N = 1 only (tier contract ④)
        try:
            threads = host_threads()
            tcpu, st = cpu_reference_full(threads)()
            line["cpu_baseline"] = {"value": N_TOKENS / tcpu, "unit": "tokens/s", "cores": threads, "kind": "port",
                                    "rtf": tcpu / audio_s,
                                    "sample": f"ONE full config-2 utterance (the same workload: {N_TOKENS} tokens, P={P_FRAMES}, "
                                              f"T={P_FRAMES + mine['F']}, CFM {CFM_STEPS} steps, BigVGAN {mine['F'] * 256} samples), no warm-up, "
                                              f"oracle port on torch CPU fp32, {tcpu:.1f} s wall (gpt {st['gpt']:.1f}, s2mel {st['s2mel']:.1f}, "
                                              f"bigvgan {st['bigvgan']:.1f}), {threads} threads of {os.cpu_count()} cores"}
        except Exception as ex:  # the bench line must survive a CPU-leg hiccup
            line["cpu_baseline"] = {"value": None, "unit": "tokens/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": f"failed: {ex}"}
    print(json.dumps(line))
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
