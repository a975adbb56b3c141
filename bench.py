#!/usr/bin/env python
"""Benchmark of the hot path.  Default workload = BASELINE.json configs[1]: VGGish FAD on
10 000 x 10 s synthetic 16 kHz clips per GPU.  The other BASELINE configurations run at their per-GPU size:

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model M]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --model clap-laion-audio --clips 6250          # configs[2]: 50 000 clips over 8 GPUs
    python bench.py --model encodec-emb --clips 1250 --indiv       # configs[3]: 5 000 songs over 4 GPUs, per-song FAD
    python bench.py --model whisper-small --clips 3125 --inf       # configs[4]: 25 000 clips over 8 GPUs, FAD-inf sweep
    python bench.py --dump-outputs DIR                             # also write the last timed step's results as DIR/*.npy

One "step" = one pass of the whole hot path over the eval set: PCM16 -> front-end -> embedder ->
fp16 embeddings -> (n, sum, outer-product) statistics -> [all-reduce] -> Frechet distance against
fixed baseline statistics.  Records of one line:
  value / ms_per_step   device-resident: PCM already in HBM, CUDA events, max over ranks, per-kernel profiling OFF
  e2e                   the same step through the reference-facing plugin calls with HOST buffers:
                        ModelLoader.embed_pcm_batch_flat (pinned int16 PCM in, fp16 embeddings back on the host, what
                        cache_embedding_files writes) -> utils.DeviceStatistics -> calc_frechet_distance (float out)
  e2e_fused             the repo's in-memory pipeline (EvalSetFAD.run_host): same host PCM, embeddings stay in HBM
  e2e_files             (N = 1) .wav directories -> cache_embedding_files -> FrechetAudioDistance.score, the `fadtk`
                        command line's calls, files on local disk
  strong_scaling        BASELINE's fixed-size job (the model's default clip count IN TOTAL) sharded over the N ranks:
                        end-to-end FAD wall-clock including the all-reduce
  roofline              dominant kernel, from a SEPARATE profiled pass (CUDA events around every kernel group)
`--impl reference` times the reference's CPU implementation of the path (torch-CPU fp32 restatement of the third-party
model + reference-pinned numpy statistics/Frechet, oracle/) on a bounded sample of the same workload, on every host
core this process may use (affinity and cgroup quota; torchrun's OMP_NUM_THREADS=1 is overridden).
`--dump-outputs DIR` (rank 0) writes, after the timing, what the last timed step handed its caller, as float64 .npy:
  frechet.npy        EvalSetFAD.run_device's fp64[8] (FAD, tr sqrt(C1 C2), residual, iterations, |mu1-mu2|^2, tr C1, tr C2, 0)
  indiv_scores.npy   with --indiv: every song's FAD, in clip order
  inf_fit.npy        with --inf: FAD-inf score, slope, r^2
The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path


def host_cores() -> int:
    """CPU cores this process may really use: scheduler affinity, capped by the cgroup CPU quota (a container with a
    64-core affinity mask and an 8-CPU quota thrashes on 64 threads - round 1's reference arm moved 6x between runs)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = Path(path).read_text().split()
            if path.endswith("cpu.max"):
                quota, period = txt[0], float(txt[1])
            else:
                quota, period = txt[0], float(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            if quota not in ("max", "-1") and period > 0:
                n = max(1, min(n, int(math.ceil(float(quota) / period))))
            break
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n)


HOST_CORES = host_cores()
if "--impl" in sys.argv and "reference" in sys.argv:
    # before numpy / torch load their thread pools: the CPU arm uses every core it may, whoever launched it
    for _v in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[_v] = str(HOST_CORES)
os.environ.setdefault("FADTK_SYNTHETIC", "1")      # benchmarks run the real architectures on seeded random weights (no checkpoints offline)

import numpy as np      # noqa: E402
import torch            # noqa: E402

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

CLIP_SECONDS = 10.0
ROWS_PER_CLIP = 10
# tensor-core layers of VGGish (conv1's 7.1 MFLOP run on the CUDA cores): 2*M*N*K per example
UMMA_LAYER_FLOP = {
    "conv2": 2 * 48 * 32 * 128 * 576, "conv3_1": 2 * 24 * 16 * 256 * 1152, "conv3_2": 2 * 24 * 16 * 256 * 2304,
    "conv4_1": 2 * 12 * 8 * 512 * 2304, "conv4_2": 2 * 12 * 8 * 512 * 4608,
    "fc1": 2 * 12288 * 4096, "fc2": 2 * 4096 * 4096, "fc3": 2 * 4096 * 128,
}


# HTSAT-tiny GEMMs per 10-s window: 24 T C^2 per Swin block + 3 patch-merging reductions
def _htsat_gemm_flop(embed, depths):
    dims = [(d, 4096 >> (2 * i), embed << i) for i, d in enumerate(depths)]
    return sum(d * 24 * t * c * c for d, t, c in dims) + sum(2 * (t // 4) * 4 * c * 2 * c for _, t, c in dims[:3])


def _whisper_gemm_flop(d, n_enc, n_dec):
    """tensor-core GEMM FLOPs per clip (30-s padded input): conv stem (as 3-tap GEMMs), encoder layers,
    cross-attention K/V projections; the 2-token decoder GEMMs are negligible."""
    f = 4 * d
    stem = 2 * 3000 * d * 240 + 2 * 1500 * d * 3 * d
    enc = n_enc * 2 * 1500 * (4 * d * d + 2 * d * f)
    ckv = n_dec * 2 * 1500 * 2 * d * d
    return stem + enc + ckv


CLAP_GEMM_FLOP = _htsat_gemm_flop(96, (2, 2, 6, 2))
WHISPER_SMALL_GEMM_FLOP = _whisper_gemm_flop(768, 12, 12)


def _encodec_gemm_flop(T=240000):
    """algorithmic conv + LSTM FLOPs of the 24 kHz SEANet encoder per clip of T samples (2*M*N*K, no padding)"""
    fl, ch, t = 2 * T * 32 * 7, 32, T
    for r in (2, 4, 5, 8):
        fl += 2 * t * (ch // 2) * 3 * ch + 2 * t * ch * (ch // 2) + 2 * t * ch * ch     # conv3, conv1, shortcut
        t = -(-t // r)
        fl += 2 * t * 2 * ch * 2 * r * ch                                               # down conv
        ch *= 2
    fl += 2 * (2 * t * 2048 * 512 * 2)                                                 # LSTM: input + recurrent, 2 layers
    fl += 2 * t * 128 * 7 * 512
    return fl


ENCODEC_GEMM_FLOP = _encodec_gemm_flop()


def _w2v_gemm_flop(L=160000, d=768, layers=12, ffn=3072):
    """conv feature encoder + projection + positional conv + transformer GEMMs per clip of L samples"""
    t, fl, cin = L, 0, 1
    for k, s_ in zip((10, 3, 3, 3, 3, 2, 2), (5, 2, 2, 2, 2, 2, 2)):
        t = (t - k) // s_ + 1
        fl += 2 * t * 512 * k * cin
        cin = 512
    fl += 2 * t * d * 512 + 2 * t * d * (d // 16) * 128
    return fl + layers * 2 * t * (4 * d * d + 2 * d * ffn)


W2V2_BASE_GEMM_FLOP = _w2v_gemm_flop()
CLAP_MUSIC_GEMM_FLOP = _htsat_gemm_flop(128, (2, 2, 12, 2))

# units_per_clip: rows_flop is the algorithmic GEMM work of ONE unit (VGGish example, CLAP window, clip otherwise)
MODELS = {
    "vggish": dict(sr=16000, clips=10000, baseline_clips=1000, chunk_clips=1000, d=128, units_per_clip=ROWS_PER_CLIP,
                   workload="VGGish FAD, {clips} x 10 s synthetic 16 kHz clips per GPU vs {base}-clip baseline (BASELINE.json configs[1])",
                   rows_flop=sum(UMMA_LAYER_FLOP.values())),
    "clap-laion-audio": dict(sr=48000, clips=500, baseline_clips=100, chunk_clips=50, d=512, units_per_clip=ROWS_PER_CLIP,
                             workload="clap-laion-audio (HTSAT-tiny) FAD, {clips} x 10 s synthetic 48 kHz clips per GPU vs {base}-clip "
                                      "baseline (BASELINE.json configs[2]: 6250 clips per GPU = 50 000 over 8 GPUs)",
                             rows_flop=CLAP_GEMM_FLOP),
    "clap-laion-music": dict(sr=48000, clips=250, baseline_clips=50, chunk_clips=25, d=512, units_per_clip=ROWS_PER_CLIP,
                             workload="clap-laion-music (HTSAT-base) FAD, {clips} x 10 s synthetic 48 kHz clips per GPU vs {base}-clip baseline",
                             rows_flop=CLAP_MUSIC_GEMM_FLOP),
    "encodec-emb": dict(sr=24000, clips=512, baseline_clips=64, chunk_clips=512, d=128, units_per_clip=1,
                        workload="encodec-emb (24 kHz SEANet encoder) FAD, {clips} x 10 s synthetic 24 kHz clips per GPU (750 rows per clip) "
                                 "vs {base}-clip baseline (BASELINE.json configs[3]: 1250 songs per GPU = 5 000 over 4 GPUs, --indiv)",
                        rows_flop=ENCODEC_GEMM_FLOP),
    "w2v2-base": dict(sr=16000, clips=256, baseline_clips=32, chunk_clips=32, d=768, units_per_clip=1,
                      workload="w2v2-base (hidden_states[12]) FAD, {clips} x 10 s synthetic 16 kHz clips per GPU (499 rows per clip) vs {base}-clip baseline",
                      rows_flop=W2V2_BASE_GEMM_FLOP),
    "whisper-small": dict(sr=16000, clips=256, baseline_clips=64, chunk_clips=64, d=768, units_per_clip=1,
                          workload="whisper-small FAD, {clips} x 10 s synthetic 16 kHz clips per GPU (each padded to 30 s, 2 rows per clip) "
                                   "vs {base}-clip baseline (BASELINE.json configs[4]: 3125 clips per GPU = 25 000 over 8 GPUs, --inf)",
                          rows_flop=WHISPER_SMALL_GEMM_FLOP),
}


def cpu_scoring_indiv(mu_b, cov_b, songs):
    """cpu_baseline leg of benchmarks/scoring.py --mode indiv: the reference arithmetic (oracle) per song.
    -> (scores, seconds)"""
    from oracle import fad_oracle as fo
    t0 = time.perf_counter()
    want = [fo.frechet_distance(mu_b, cov_b, *fo.embd_statistics(s)) for s in songs]
    return want, time.perf_counter() - t0


def cpu_scoring_inf(mu_b, cov_b, rows, steps, k):
    """cpu_baseline leg of benchmarks/scoring.py --mode inf: the first k bootstrap sizes on the oracle, consuming the
    global numpy RNG exactly like the reference (seeded 0 here).  -> (scores, seconds in gather+cov, seconds in Frechet, sizes)"""
    from oracle import fad_oracle as fo
    sizes = fo.inf_sample_sizes(len(rows), steps, 500)
    np.random.seed(0)
    pts, t_stats, t_fr = [], 0.0, 0.0
    for n in sizes[:k]:
        t0 = time.perf_counter()
        pick = np.random.choice(rows.shape[0], size=n, replace=True)
        st = fo.embd_statistics(rows[pick])
        t1 = time.perf_counter()
        pts.append(fo.frechet_distance(mu_b, cov_b, *st))
        t_stats += t1 - t0
        t_fr += time.perf_counter() - t1
    return pts, t_stats, t_fr, sizes


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d.get("bf16_tflops_sustained", 1443.3), d.get("hbm_gbs", 6567.7), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    FIELDS = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        rows = [r.split(",") for r in Path(self.tmp.name).read_text().strip().splitlines() if r.count(",") >= 6]
        os.unlink(self.tmp.name)
        if not rows:
            return out
        sm = [float(r[0]) for r in rows if r[0].strip().replace(".", "").isdigit()]
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_max_mhz"] = float(rows[0][1])
        pw = [float(r[2]) for r in rows if r[2].strip().replace(".", "").isdigit()]
        if pw:
            out["power_w_median"] = float(np.median(pw))
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for i, n in enumerate(names):
            if any("Active" in r[3 + i] and "Not" not in r[3 + i] for r in rows):
                out["reasons"].append(n)
        out["samples"] = len(rows)
        return out


def oracle_embed_fn(model: str, state):
    if model == "vggish":
        from oracle import vggish_oracle as vo
        return lambda pcm: vo.embed(vo.load_wav_semantics(pcm), state)
    if model == "encodec-emb":
        from oracle import encodec_oracle as eo
        return lambda pcm: eo.embed(pcm / 32768.0, state)
    if model == "w2v2-base":
        from oracle import w2v_oracle as wv
        hf, fe = wv.build(state, "w2v2")
        return lambda pcm: wv.embed(pcm / 32768.0, hf, fe, 12)
    if model.startswith("whisper-"):
        from fadtk_b200 import weights_whisper
        from oracle import whisper_oracle as wo
        hf, fe = wo.build(state, weights_whisper.SYNTH_START)
        return lambda pcm: wo.embed(pcm / 32768.0, hf, fe, weights_whisper.SYNTH_START)
    from oracle import clap_oracle as co
    return lambda pcm: co.embed(pcm / 32768.0, state)


def cpu_reference_leg(model, pcm_clips: np.ndarray, base_stats, state, budget_s: float = 15.0):
    """Reference CPU path on a bounded sample: per-clip loop (fad_batch.py semantics), fp32 torch
    restatement of the model, fp16 cache rounding, per-file statistics + Chan merge (utils.py:13-46),
    eig-route Frechet, on HOST_CORES threads.  -> dict"""
    from oracle import fad_oracle as fo
    torch.set_num_threads(HOST_CORES)
    embed = oracle_embed_fn(model, state)
    threads = torch.get_num_threads()
    t0 = time.perf_counter()
    embs = []
    used = 0
    for i in range(pcm_clips.shape[0]):
        embs.append(embed(pcm_clips[i]))
        used += 1
        if time.perf_counter() - t0 > budget_s and used >= 4:
            break
    t_embed = time.perf_counter() - t0
    t1 = time.perf_counter()
    mu, cov = fo.online_statistics(embs)          # one clip = one file: utils.py:19-46 semantics
    t_stats = time.perf_counter() - t1
    t2 = time.perf_counter()
    fad = fo.frechet_distance(base_stats[0], base_stats[1], mu, cov)
    t_fr = time.perf_counter() - t2
    total = t_embed + t_stats + t_fr
    return {"value": used * CLIP_SECONDS / total, "unit": "audio-s/s", "cores": threads, "kind": "port",
            "host": {"affinity_cores": len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else None,
                     "usable_cores": HOST_CORES, "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS")},
            "sample": f"{used} of the eval clips ({used * CLIP_SECONDS:.0f} audio-s): embed {t_embed:.2f}s, "
                      f"stats {t_stats:.3f}s, frechet {t_fr:.3f}s; "
                      + ("transformers WhisperFeatureExtractor + WhisperModel on CPU (the reference's own dependency, "
                         "driven as model_loader.py:663-669) + numpy/scipy" if model.startswith("whisper-") else
                         f"oracle/ torch-CPU fp32 {model} + numpy/scipy (reference third-party model is not installable offline)"),
            "fad": float(fad), "clips": used, "seconds": total}


def synthetic_state(model: str):
    from fadtk_b200 import weights, weights_clap
    if model == "vggish":
        return weights.synthetic_vggish_state(0)
    if model == "encodec-emb":
        from fadtk_b200 import weights_encodec
        return weights_encodec.synthetic_encodec_state(0)
    if model == "w2v2-base":
        from fadtk_b200 import weights_w2v
        return weights_w2v.synthetic_w2v_state(0)
    if model.startswith("whisper-"):
        from fadtk_b200 import weights_whisper
        return weights_whisper.synthetic_whisper_state(0, model.split("-", 1)[1])
    return weights_clap.synthetic_clap_state(0, "base" if model == "clap-laion-music" else "tiny")


def make_loader(model: str, chunk_clips: int):
    """The registry's plugin object for ``model`` (seed-0 synthetic weights under FADTK_SYNTHETIC=1: byte-identical to
    synthetic_state()), sized so one forward takes ``chunk_clips`` clips."""
    from fadtk_b200 import model_loader as mlm
    if model == "vggish":
        return mlm.VGGishModel()
    if model in ("clap-laion-audio", "clap-laion-music"):
        return mlm.CLAPLaionModel(model.rsplit("-", 1)[1], max_chunks=chunk_clips * ROWS_PER_CLIP)
    if model == "encodec-emb":
        return mlm.EncodecEmbModel("24k", max_chunk_samples=16 * int(CLIP_SECONDS * 24000))
    if model == "w2v2-base":
        return mlm.W2V2Model("base", 12, max_clips=chunk_clips)
    if model.startswith("whisper-"):
        return mlm.WhisperModel(model.split("-", 1)[1], max_clips=chunk_clips)
    raise ValueError(model)


def reference_arm(args, spec, config, state, rank):
    if rank != 0:
        return
    from fadtk_b200 import synth
    sr = spec["sr"]
    torch.set_num_threads(HOST_CORES)
    embed = oracle_embed_fn(args.model, state)
    n_base, n_eval = (16, 64) if args.model == "vggish" else (4, 16)
    base = np.concatenate([embed(synth.musiclike_clip(i, CLIP_SECONDS, sr, True)) for i in range(n_base)])
    base_stats = (base.astype(np.float64).mean(0), np.cov(base.astype(np.float64), rowvar=False))
    sample = np.stack([synth.musiclike_clip(i, CLIP_SECONDS, sr) for i in range(n_eval)])
    per_step = max(4.0, 40.0 / max(1, args.steps + args.warmup))
    for _ in range(max(1, args.warmup)):          # at least one untimed pass: thread pools, oneDNN primitives, page faults
        cpu_reference_leg(args.model, sample, base_stats, state, budget_s=min(per_step, 6.0))
    legs = [cpu_reference_leg(args.model, sample, base_stats, state, budget_s=per_step) for _ in range(args.steps)]
    secs = sum(l["seconds"] for l in legs)
    clips = sum(l["clips"] for l in legs)
    val = clips * CLIP_SECONDS / secs
    cb = dict(legs[-1])
    cb["value"] = val
    cb["per_step_values"] = [l["value"] for l in legs]
    for k in ("fad", "clips", "seconds"):
        cb.pop(k)
    print(json.dumps({"impl": "reference", "metric": "audio_seconds_embedded_per_second", "value": val,
                      "unit": "audio-s/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": 1000.0 * secs / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                      "cpu_baseline": cb,
                      "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="vggish", choices=list(MODELS))
    ap.add_argument("--clips", type=int, default=0, help="eval clips per GPU (0 = the model's default)")
    ap.add_argument("--baseline-clips", type=int, default=0)
    ap.add_argument("--chunk-clips", type=int, default=0)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --clips per GPU (the headline); strong: --clips IN TOTAL, sharded over the ranks")
    ap.add_argument("--indiv", action="store_true", help="per-song FAD of every eval clip after the embedding (configs[3])")
    ap.add_argument("--inf", action="store_true", help="FAD-inf sweep over the gathered embeddings (configs[4])")
    ap.add_argument("--files-clips", type=int, default=2000, help="eval clips of the e2e_files record (N = 1, vggish; 0 = skip)")
    ap.add_argument("--profile-steps", type=int, default=1, help="steps of the separate per-kernel profiling pass")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path, default=None,
                    help="after the timing, write the last timed step's results as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path's results (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    spec = MODELS[args.model]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    total_default = spec["clips"]
    args.clips = args.clips or spec["clips"]
    total_clips = world * args.clips
    if args.scaling == "strong":                              # --clips is the whole job; this rank's share
        total_clips = args.clips
        base_n, extra = divmod(total_clips, world)
        args.clips = base_n + (1 if rank < extra else 0)
    args.baseline_clips = args.baseline_clips or spec["baseline_clips"]
    args.chunk_clips = min(args.chunk_clips or spec["chunk_clips"], max(1, args.clips))
    sr = spec["sr"]
    clip_samples = int(sr * CLIP_SECONDS)

    pcm_gb = args.clips * clip_samples * 2 / 1e9
    config = {"workload": spec["workload"].format(clips=args.clips, base=args.baseline_clips),
              "model": f"{args.model} (seeded synthetic weights, real architecture)", "clips_per_gpu": args.clips,
              "clip_seconds": CLIP_SECONDS, "chunk_clips": args.chunk_clips,
              "l2": f"inputs ({pcm_gb:.1f} GB PCM per GPU) exceed L2; no explicit flush", "parallelism": f"dp{world}"}
    state = synthetic_state(args.model)

    if args.impl == "reference":
        return reference_arm(args, spec, config, state, rank)

    # ------------------------------------------------------------------------ our arm
    from fadtk_b200 import _native, dist, synth
    from fadtk_b200.fad import calc_frechet_distance
    from fadtk_b200.pipeline import EvalSetFAD
    from fadtk_b200.utils import DeviceStatistics
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_from_env("nccl")
    dev = torch.device("cuda", local_rank)
    # ONE engine per process: the plugin object below loads its weights into it, the in-memory pipeline drives it
    eng = _native.engine(local_rank, max_examples=args.chunk_clips * ROWS_PER_CLIP)
    ml = make_loader(args.model, args.chunk_clips)
    ml.load_model()
    assert ml._engine is eng

    # baseline statistics (identical on every rank), outside the timed region
    d = spec["d"]
    zero_mu, eye = torch.zeros(d, dtype=torch.float64), torch.eye(d, dtype=torch.float64)
    helper = EvalSetFAD(eng, zero_mu, eye, clip_samples, clips_per_chunk=args.chunk_clips, model=args.model)
    base_pcm = synth.musiclike_device(args.baseline_clips, CLIP_SECONDS, sr, seed=30_000, device=dev,
                                      fmax=1500.0, noise=0.08)
    base_emb = torch.cat([helper.embed(base_pcm[s:s + args.chunk_clips]) for s in range(0, args.baseline_clips, args.chunk_clips)])
    shift = base_emb[:4096].float().mean(0).to(torch.float16)
    acc = eng.stats_accumulate(base_emb, shift, eng.stats_new(d))
    mu_b, cov_b = eng.stats_finalize(acc, shift, d)
    mu_b_host, cov_b_host = mu_b.cpu().numpy(), cov_b.cpu().numpy()
    del base_pcm

    pcm = synth.musiclike_device(args.clips, CLIP_SECONDS, sr, seed=20_000 + rank, device=dev)
    job = EvalSetFAD(eng, mu_b, cov_b, clip_samples, clips_per_chunk=args.chunk_clips, model=args.model)
    rows_per_clip = job.rows_per_clip

    def sync_all():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warm):
        """``steps`` calls of fn between barrier + synchronize on both sides; CUDA events AND the host clock (a step
        that ends with a device->host read is bounded by both); max over ranks.  -> (event ms, wall ms, last result)"""
        res = None
        for _ in range(warm):
            res = fn()
        sync_all()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            res = fn()
        e1.record()
        sync_all()
        return dist.max_over_ranks(e0.elapsed_time(e1)), dist.max_over_ranks((time.perf_counter() - t0) * 1000.0), res

    # ---- device-resident timing (value): per-kernel profiling OFF
    eng.profile(False)
    for _ in range(args.warmup):
        job.run_device(pcm)
    sync_all()
    launches0 = eng.launches
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms, _, res = timed(lambda: job.run_device(pcm), args.steps, 0)
    clocks = sampler.stop() if sampler else None
    launches = eng.launches - launches0
    outputs = {"frechet": res.cpu().numpy()}
    fad_value = float(res[0].item())
    audio_s = total_clips * CLIP_SECONDS * args.steps
    value = audio_s / (ms / 1000.0)

    # ---- separate profiled pass -> roofline of the dominant kernel (tcgen05 conv / FC GEMM)
    peak_tf, peak_hbm, peak_src = measured_peaks()
    eng.profile_collect()
    eng.profile(True)
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    pe0.record()
    for _ in range(max(1, args.profile_steps)):
        job.run_device(pcm)
    pe1.record()
    torch.cuda.synchronize()
    prof_ms = pe0.elapsed_time(pe1)
    prof = eng.profile_collect()
    eng.profile(False)
    units = args.clips * spec["units_per_clip"] * max(1, args.profile_steps)   # examples (VGGish) / windows (CLAP) / clips
    forward_keys = [k for k in prof if k not in ("frechet", "stats", "stats_reduce")]
    gemm_keys = [k for k in UMMA_LAYER_FLOP if k in prof] if args.model == "vggish" else [k for k in ("clap_gemm",) if k in prof]
    gemm_ms = sum(prof[k][0] for k in gemm_keys)
    gemm_launch = sum(prof[k][1] for k in gemm_keys)
    forward_ms = sum(prof[k][0] for k in forward_keys)
    flop = spec["rows_flop"] * units
    wlo_fp8 = os.environ.get("FADTK_WLO") == "fp8"
    if args.model == "vggish":
        # every GEMM of the forward is timed by layer: the kernel's own rate
        denom_ms, basis = gemm_ms, "CUDA events around each layer's launch (separate profiled pass)"
        split_mask = 0xFF                                     # weights.ALL_LAYERS_SPLIT: what VGGishModel packs
        per_layer_factor = 1.5 if wlo_fp8 else 2.0            # an fp8 low-part MMA takes half the tensor-pipe time of an fp16 one
        issued_factor = sum(UMMA_LAYER_FLOP[k] * (per_layer_factor if (split_mask >> i) & 1 else 1.0)
                            for i, k in enumerate(UMMA_LAYER_FLOP)) / sum(UMMA_LAYER_FLOP.values())
        pair_env = os.environ.get("FADTK_PAIR", "auto")
        pairs = {"auto": "CTA pairs (cta_group::2, M = 256) on conv3_2, conv4_1, conv4_2, fc1, fc2", "1": "CTA pairs (cta_group::2) on every layer",
                 "0": "single-CTA MMAs"}.get(pair_env, f"CTA pairs mask {pair_env}")
        kernel = (f"fad::conv_gemm_kernel<128, STAGES, {2 if wlo_fp8 else 1}, PAIR> (tcgen05 kind::f16, {pairs}; fp16 hi/lo split weights on "
                  f"{bin(split_mask).count('1')}/8 layers: " + ("low parts as kind::f8f6f4 E4M3 MMAs)" if wlo_fp8 else "2 fp16 MMAs per K slice into one TMEM accumulator)"))
    else:
        # the GEMM category does not cover every GEMM of these forwards (front-end convolutions are timed with the
        # front end): rate over the WHOLE forward - a lower bound of the kernel's own rate that cannot exceed the peak
        denom_ms = forward_ms
        basis = "algorithmic GEMM FLOPs / whole forward time of the profiled pass (lower bound of the kernel's own rate)"
        issued_factor = None
        kernel = "fad::conv_gemm_kernel (tcgen05 kind::f16; every Linear / convolution-as-GEMM of the forward)"
    achieved = flop / (denom_ms / 1000.0) / 1e12 if denom_ms > 0 else 0.0
    per_layer = {k: {"ms_per_launch": prof[k][0] / prof[k][1], "tflops": UMMA_LAYER_FLOP[k] * units / (prof[k][0] / 1000.0) / 1e12}
                 for k in UMMA_LAYER_FLOP if k in prof and prof[k][0] > 0} if args.model == "vggish" else None
    other = {k: {"ms_total": v[0], "launches": v[1]} for k, v in prof.items() if k not in gemm_keys}
    traffic, traffic_src = None, None
    tf = ROOT / "profiles" / "roofline_traffic.json"
    if tf.exists() and gemm_launch:
        t = json.loads(tf.read_text()).get(args.model)
        if t:
            traffic = t["dram_gb_per_row"] * units / gemm_launch
            traffic_src = t["source"]
    roofline = {"kernel": kernel, "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": achieved / peak_tf, "peak_source": peak_src, "basis": basis,
                "traffic": traffic, "traffic_unit": "GB per launch", "traffic_source": traffic_src,
                "issued_factor": issued_factor,
                "issued_tflops": issued_factor * achieved if issued_factor else None,
                "issued_frac": issued_factor * achieved / peak_tf if issued_factor else None,
                "note": "achieved counts ALGORITHMIC FLOPs (2*M*N*K once); issued_factor = tensor-pipe time issued per algorithmic FLOP (hi/lo weight split)",
                "launches": gemm_launch, "avg_launch_ms": gemm_ms / max(1, gemm_launch),
                "algorithmic_gflop_per_unit": spec["rows_flop"] / 1e9,
                "share_of_step": gemm_ms / prof_ms if prof_ms > 0 else None,
                "profiled_pass_ms_per_step": prof_ms / max(1, args.profile_steps),
                "per_layer": per_layer, "other_kernels": other}

    # ---- scoring modes of configs[3] / configs[4], on the embeddings of one more (untimed) forward
    scoring = None
    if args.indiv or args.inf:
        emb_all = torch.cat([job.embed(pcm[s:s + args.chunk_clips]).clone() for s in range(0, args.clips, args.chunk_clips)])
        base_obj = _native.Baseline(eng, mu_b, cov_b)
        base_obj.mu_host = mu_b_host
        if args.indiv:
            offs = torch.arange(0, args.clips + 1, device=dev, dtype=torch.int64) * rows_per_clip

            def indiv_step():
                out = base_obj.frechet_batched(emb_all, offs)[:, 0].contiguous()
                if world > 1:
                    parts = [torch.empty_like(out) for _ in range(world)]
                    torch.distributed.all_gather(parts, out)
                    out = torch.cat(parts)
                return out.cpu().numpy()                       # the scores the csv is written from
            ms_i, wall_i, scores = timed(indiv_step, args.steps, 1)
            outputs["indiv_scores"] = scores
            ms_i = max(ms_i, wall_i) / args.steps
            scoring = {"mode": "indiv (score_individual arithmetic: fad_frechet_batched, all songs in lock-step; scores gathered to every rank)",
                       "songs": int(len(scores)), "rows_per_song": rows_per_clip, "d": d,
                       "ms_per_pass": ms_i, "songs_per_s": len(scores) / (ms_i / 1000.0),
                       "finite": bool(np.isfinite(scores).all()), "median_fad": float(np.median(scores))}
        else:
            from fadtk_b200.fad import _device_score
            if world > 1:
                parts = [torch.empty_like(emb_all) for _ in range(world)]
                torch.distributed.all_gather(parts, emb_all)
                emb_inf = torch.cat(parts)
            else:
                emb_inf = emb_all
            n_rows = emb_inf.shape[0]
            sizes = [int(n) for n in np.linspace(min(500, n_rows), n_rows, 25)]

            def inf_step():
                np.random.seed(0)
                pts = []
                for step, n in enumerate(sizes):               # rank 0 owns the RNG stream (fad.py:333), steps are sharded
                    idx = np.random.choice(n_rows, size=n, replace=True) if rank == 0 else np.empty(n, dtype=np.int64)
                    idx = dist.broadcast_int64(idx)
                    if step % world == rank:
                        pts.append([n, _device_score(base_obj, emb_inf, eng, torch.from_numpy(idx).to(dev))])
                if world > 1:
                    pts = sorted((p for part in dist.allgather_objects(pts) for p in part), key=lambda p: p[0])
                ys = np.array(pts)
                xs = 1 / np.array(sizes)
                slope, intercept = np.polyfit(xs, ys[:, 1], 1)
                r2 = 1 - np.sum((ys[:, 1] - (slope * xs + intercept)) ** 2) / np.sum((ys[:, 1] - np.mean(ys[:, 1])) ** 2)
                return intercept, slope, r2
            ms_f, wall_f, (inf_score, inf_slope, inf_r2) = timed(inf_step, args.steps, 1)
            outputs["inf_fit"] = np.array([inf_score, inf_slope, inf_r2])
            ms_f = max(ms_f, wall_f) / args.steps
            scoring = {"mode": "inf (score_inf arithmetic: host RNG indices, gather + exact Gram + Frechet per size on the GPU, sizes sharded over ranks)",
                       "rows": int(n_rows), "d": d, "sizes": 25, "ms_per_sweep": ms_f, "fad_inf": float(inf_score),
                       "slope": float(inf_slope), "r2": float(inf_r2),
                       "gram_tflops_over_sweep": sum(2.0 * n * d * d for n in sizes) / (ms_f / 1000.0) / 1e12}
        del emb_all

    # ---- end to end from pinned host memory
    e2e = e2e_fused = None
    if not args.no_e2e:
        host = torch.empty((args.clips, clip_samples), dtype=torch.int16, pin_memory=True)
        host.copy_(pcm)
        torch.cuda.synchronize()
        host_np = host.numpy()
        chunks = [[host_np[i] for i in range(s, min(s + args.chunk_clips, args.clips))] for s in range(0, args.clips, args.chunk_clips)]
        emb_bytes = args.clips * rows_per_clip * d * 2

        def plugin_step():
            """the reference-facing calls: plugin embeds host PCM and hands fp16 embeddings back on the host (what the
            batch driver writes to .npy), statistics of those host arrays, Frechet distance of host statistics"""
            st = DeviceStatistics(d, eng, reduce_ranks=world > 1)
            for part in chunks:
                flat, _rows = ml.embed_pcm_batch_flat(part)
                st.add(flat)
            st.allreduce()
            mu_e, cov_e = st.finalize()
            return float(calc_frechet_distance(mu_b_host, cov_b_host, mu_e.cpu().numpy(), cov_e.cpu().numpy()))

        ms_p, wall_p, fad_p = timed(plugin_step, args.steps, 2)
        ms_p = max(ms_p, wall_p)
        e2e = {"value": audio_s / (ms_p / 1000.0), "unit": "audio-s/s", "ms_per_step": ms_p / args.steps,
               "h2d_bytes_per_step": int(args.clips * clip_samples * 2 + emb_bytes + 2 * (d * d + d) * 8),
               "d2h_bytes_per_step": int(emb_bytes + (d * d + d) * 8 + 64), "fad": fad_p,
               "api": f"{type(ml).__name__}.embed_pcm_batch_flat (ModelLoader plugin: pinned int16 PCM in, fp16 embeddings out on the host) "
                      "-> utils.DeviceStatistics.add/allreduce/finalize -> fad.calc_frechet_distance (host mu/cov in, float out)"}

        ms_e, wall_e, fad_h = timed(lambda: job.run_host(host), args.steps, 2)
        ms_e = max(ms_e, wall_e)
        e2e_fused = {"value": audio_s / (ms_e / 1000.0), "unit": "audio-s/s", "ms_per_step": ms_e / args.steps,
                     "h2d_bytes_per_step": int(args.clips * clip_samples * 2), "d2h_bytes_per_step": 8, "fad": fad_h,
                     "api": "fadtk_b200.pipeline.EvalSetFAD.run_host (pinned int16 PCM in, embeddings stay in HBM, FAD float out)"}
        del host, host_np, chunks

    # ---- strong scaling: the model's default job size IN TOTAL, sharded over the ranks (BASELINE target: 10 000 clips)
    strong = None
    if args.scaling == "strong" or world == 1:
        strong = {"total_clips": int(total_clips), "clips_per_gpu": int(args.clips), "fad_wallclock_s": ms / args.steps / 1000.0,
                  "value": value, "unit": "audio-s/s", "what": "the headline step (this run IS the fixed-size job)",
                  "e2e_wallclock_s": e2e_fused["ms_per_step"] / 1000.0 if e2e_fused else None}
    elif not args.no_strong:
        job_total = min(total_default, world * args.clips)
        base_n, extra = divmod(job_total, world)
        mine = base_n + (1 if rank < extra else 0)
        sub = pcm[:mine].contiguous()
        job_s = EvalSetFAD(eng, mu_b, cov_b, clip_samples, clips_per_chunk=min(args.chunk_clips, max(1, mine)), model=args.model)
        ms_s, _, res_s = timed(lambda: job_s.run_device(sub), args.steps, 2)
        strong = {"total_clips": int(job_total), "clips_per_gpu": int(mine),
                  "fad_wallclock_s": ms_s / args.steps / 1000.0, "value": job_total * CLIP_SECONDS * args.steps / (ms_s / 1000.0),
                  "unit": "audio-s/s", "fad": float(res_s[0].item()),
                  "what": "device-resident step (embed shard -> exact Gram -> ONE all-reduce -> Newton-Schulz Frechet), CUDA events, max over ranks"}
        if not args.no_e2e:
            hs = torch.empty((mine, clip_samples), dtype=torch.int16, pin_memory=True)
            hs.copy_(sub)
            torch.cuda.synchronize()
            ms_h, wall_h, _ = timed(lambda: job_s.run_host(hs), args.steps, 2)
            strong["e2e_wallclock_s"] = max(ms_h, wall_h) / args.steps / 1000.0

    # ---- the directory flow (N = 1): .wav files -> cache_embedding_files -> FrechetAudioDistance.score
    e2e_files = None
    if world == 1 and args.files_clips > 0 and args.model == "vggish" and not args.no_e2e:
        try:
            e2e_files = files_flow(ml, args.files_clips, max(64, args.files_clips // 8), sr)
        except Exception as e:                                  # a full /tmp must not cost the headline
            e2e_files = {"error": repr(e)[:300]}

    if rank != 0:
        dist.shutdown()
        return
    if args.dump_outputs is not None:
        write_outputs(args.dump_outputs, outputs)

    # ---- CPU baseline + parity sample (rank 0, N = 1 only)
    cpu = None
    parity = None
    if world == 1 and not args.no_cpu_baseline:
        n_sample = 64 if args.model == "vggish" else 24
        sample = pcm[:n_sample].cpu().numpy()
        cpu = cpu_reference_leg(args.model, sample, (mu_b_host, cov_b_host), state, budget_s=15.0)
        n = cpu["clips"]
        # same clips through the GPU path -> FAD vs the CPU oracle's FAD on identical audio
        sub = EvalSetFAD(eng, mu_b, cov_b, clip_samples, clips_per_chunk=args.chunk_clips, model=args.model)
        sub.shift = job.shift
        fad_gpu_sample = float(sub.run_device(pcm[:n].contiguous())[0].item())
        parity = {"clips": n, "fad_gpu": fad_gpu_sample, "fad_cpu_oracle": cpu["fad"],
                  "rel_err": abs(fad_gpu_sample - cpu["fad"]) / abs(cpu["fad"])}
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "host")}

    line = {"metric": "audio_seconds_embedded_per_second", "value": value, "unit": "audio-s/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f16",
            "data": "synthetic", "config": config, "fad": fad_value, "fad_wallclock_s": ms / args.steps / 1000.0,
            "clocks": clocks, "e2e": e2e, "e2e_fused": e2e_fused, "e2e_files": e2e_files, "strong_scaling": strong,
            "scoring": scoring, "gpu_launches": int(launches), "roofline": roofline,
            "cpu_baseline": cpu, "parity_sample": parity}
    print(json.dumps(line))
    dist.shutdown()


DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(directory: Path, outputs: dict) -> None:
    """Each array of ``outputs`` as float64 ``directory/<name>.npy``."""
    arrays = {name: np.asarray(a, dtype=np.float64) for name, a in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes of results exceed the {DUMP_LIMIT_BYTES}-byte limit")
    directory.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(directory / f"{name}.npy", a)


def files_flow(ml, clips: int, baseline_clips: int, sr: int, workers: int = 16) -> dict:
    """`fadtk vggish <baseline dir> <eval dir>` as the command line runs it (fadtk/__main__.py:39-70): directories of PCM16
    .wav files -> cache_embedding_files (convert cache, .npy caches) -> FrechetAudioDistance.score.  Wall clock."""
    import shutil
    from fadtk_b200 import _io_native, synth
    from fadtk_b200.fad import FrechetAudioDistance
    from fadtk_b200.fad_batch import cache_embedding_files
    root = Path(tempfile.mkdtemp(prefix="fadtk_bench_files_"))
    try:
        def write_set(sub, count, seed, **kw):
            (root / sub).mkdir(parents=True, exist_ok=True)
            pcm = synth.musiclike_device(count, CLIP_SECONDS, sr, seed, torch.device("cuda", torch.cuda.current_device()), **kw).cpu().numpy()
            paths = [root / sub / f"clip{i:06d}.wav" for i in range(count)]
            st = _io_native.wav_write(paths, pcm.reshape(-1), np.arange(count) * pcm.shape[1], np.full(count, pcm.shape[1]), sr, workers)
            assert not st.any()
        write_set("eval", clips, 1)
        write_set("base", baseline_clips, 2, fmax=1500.0, noise=0.08)
        write_set("warm", 64, 3)
        cache_embedding_files(root / "warm", ml, workers=workers)          # pinned staging, workspaces
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        cache_embedding_files(root / "base", ml, workers=workers)
        cache_embedding_files(root / "eval", ml, workers=workers)
        t1 = time.perf_counter()
        score = FrechetAudioDistance(ml, audio_load_worker=workers, load_model=False).score(root / "base", root / "eval")
        t2 = time.perf_counter()
        n = clips + baseline_clips
        return {"value": n * CLIP_SECONDS / (t2 - t0), "unit": "audio-s/s", "files": n, "seconds_total": t2 - t0,
                "embed_seconds": t1 - t0, "stats_and_frechet_seconds": t2 - t1, "fad": float(score), "io_threads": workers,
                "api": "fadtk_b200.fad_batch.cache_embedding_files x2 + FrechetAudioDistance.score (the fadtk command line's calls), files on local disk"}
    finally:
        shutil.rmtree(root, ignore_errors=True)


if __name__ == "__main__":
    main()
