"""End-to-end parity of the reference-facing Python API (which calls the CUDA path through the
C ABI) against the CPU oracle and the reference-generated golden vectors."""
import numpy as np
import pytest
import torch

import fadtk_b200 as fk
from fadtk_b200 import synth
from oracle import fad_oracle as fo
from oracle import vggish_oracle as vo
from oracle.make_golden import spectrum_cov

pytestmark = pytest.mark.gpu


class GoldLoader(fk.ModelLoader):
    """A plugin with no forward pass: statistics / scoring only (like make_golden's fake loader)."""

    def __init__(self):
        super().__init__("gold", 128, 16000)

    def load_model(self):
        pass

    def _get_embedding(self, audio):
        raise NotImplementedError


def test_calc_embd_statistics_golden(engine, golden_dir):
    g = np.load(golden_dir / "stats_cases.npz")
    mu, cov = fk.calc_embd_statistics(g["cat"])
    assert mu.dtype == np.float16                                       # fad.py:48 dtype behaviour
    assert np.abs(mu.astype(np.float64) - g["mu_cat"].astype(np.float64)).max() <= 2 ** -9   # <= 1 fp16 ulp near 2
    ref = g["cov_cat"]
    assert np.abs(cov - ref).max() < 3e-5 * np.abs(ref).max()
    with pytest.raises(AssertionError):
        fk.calc_embd_statistics(g["cat"][:1])                           # fad.py:46


def test_online_statistics_from_npy_files(engine, golden_dir, tmp_path):
    g = np.load(golden_dir / "stats_cases.npz")
    files = np.split(g["cat"], np.cumsum(g["sizes"])[:-1])
    paths = []
    for i, f in enumerate(files):
        np.save(tmp_path / f"{i}.npy", f)
        paths.append(tmp_path / f"{i}.npy")
    mu, cov = fk.calculate_embd_statistics_online(paths)
    # golden = the reference's calculate_embd_statistics_online on the same files, including its
    # fp16 per-file means (6e-5 away from the exact covariance of the concatenation)
    assert np.abs(mu - g["mu_online"]).max() < 1e-12
    assert np.abs(cov - g["cov_online"]).max() < 1e-10 * np.abs(cov).max()


def test_frechet_golden_real_statistics(engine, golden_dir):
    g = np.load(golden_dir / "frechet_fma_pop_128.npz")
    got = fk.calc_frechet_distance(g["mu1"], g["cov1"], g["mu2"], g["cov2"])
    assert got == pytest.approx(float(g["fad"]), rel=1e-7)
    with pytest.raises(AssertionError):
        fk.calc_frechet_distance(g["mu1"][:5], g["cov1"], g["mu2"], g["cov2"])


@pytest.mark.parametrize("i", [0, 1, 2])
def test_frechet_golden_ill_conditioned_spectra(engine, golden_dir, i):
    g = np.load(golden_dir / "frechet_spectra.npz")
    c1 = spectrum_cov(g[f"evals1_{i}"], 100 + i)
    c2 = spectrum_cov(g[f"evals2_{i}"], 200 + i)
    got = fk.calc_frechet_distance(g[f"mu1_{i}"], c1, g[f"mu2_{i}"], c2)
    assert got == pytest.approx(float(g[f"fad_{i}"]), rel=1e-6)


def test_fad_of_identical_statistics_is_zero(engine):
    rng = np.random.default_rng(0)
    x = rng.normal(size=(2000, 128))
    mu, cov = x.mean(0), np.cov(x, rowvar=False)
    assert abs(fk.calc_frechet_distance(mu, cov, mu, cov)) < 1e-8 * np.trace(cov)


def _write_stats_npz(path, mu, cov, name="gold"):
    np.savez(path, **{f"{name}.mu": mu, f"{name}.cov": cov})


def test_score_inf_matches_reference_with_seeded_rng(engine, golden_dir, tmp_path):
    g = np.load(golden_dir / "inf_case.npz")
    mu_b, cov_b = fo.embd_statistics(g["base"])
    _write_stats_npz(tmp_path / "base.npz", mu_b, cov_b)
    np.save(tmp_path / "eval.npy", g["eval"])
    fad = fk.FrechetAudioDistance(GoldLoader(), audio_load_worker=1, load_model=False)
    np.random.seed(0)
    res = fad.score_inf(tmp_path / "base.npz", [tmp_path / "eval.npy"], steps=int(g["steps"]), min_n=int(g["min_n"]))
    pts = np.array(res.points)
    assert np.array_equal(pts[:, 0], g["points"][:, 0])
    assert np.allclose(pts[:, 1], g["points"][:, 1], rtol=1e-4)          # the project's FAD tolerance
    assert res.score == pytest.approx(float(g["score"]), rel=2e-4)
    assert res.r2 == pytest.approx(float(g["r2"]), abs=1e-4)


def test_score_individual_matches_reference_csv(engine, golden_dir, tmp_path):
    g = np.load(golden_dir / "indiv_case.npz")
    _write_stats_npz(tmp_path / "base.npz", g["mu_base"], g["cov_base"])
    ev = tmp_path / "ev"
    (ev / "embeddings" / "gold").mkdir(parents=True)
    for k in g.files:
        if k.startswith("song"):
            (ev / f"{k}.wav").write_bytes(b"")
            np.save(ev / "embeddings" / "gold" / f"{k}.npy", g[k])
    fad = fk.FrechetAudioDistance(GoldLoader(), audio_load_worker=1, load_model=False)
    csv = fad.score_individual(tmp_path / "base.npz", ev, tmp_path / "out.csv")
    rows = [ln.split(",") for ln in csv.read_text().splitlines()]
    names = [r[0].split("/")[-1] for r in rows]
    scores = np.array([float(r[1]) for r in rows])
    assert names == list(g["names"])                                     # |score| order, short song dropped
    assert np.allclose(scores, g["scores"], rtol=1e-4)


@pytest.mark.parametrize("d,lens", [(128, [750, 2, 1, 130, 40, 750, 333]), (512, [300, 700, 17])])
def test_frechet_batched_matches_oracle_per_item(engine, d, lens):
    """fad_frechet_batched == per-item reference arithmetic (fad.py:42-48 + :51-120), ragged items,
    rank-deficient items (n < d), and an item with a single row (reference: AssertionError -> NaN here)."""
    from fadtk_b200 import _native
    rng = np.random.default_rng(5)
    mix = rng.standard_normal((d, d)) * (1.0 / np.sqrt(d))
    base_rows = (rng.standard_normal((4 * d, d)) @ mix).astype(np.float16)
    mu_b, cov_b = fo.embd_statistics(base_rows)
    mu_b = mu_b.astype(np.float64)        # load_stats returns fp64 baselines (fad.py:286-288); fp16 - fp16 would stay fp16 (fad.py:83)
    items = [((rng.standard_normal((n, d)) @ mix) * (0.5 + 0.3 * i) + 0.1 * i).astype(np.float16) for i, n in enumerate(lens)]
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    base = _native.Baseline(engine, mu_b, cov_b)
    dev = engine.torch_device
    out = base.frechet_batched(torch.from_numpy(np.concatenate(items)).to(dev), torch.from_numpy(offs).to(dev)).cpu().numpy()
    assert out.shape == (len(lens), 8) and [int(v) for v in out[:, 7]] == lens
    for k, rows in enumerate(items):
        if len(rows) < 2:
            assert np.isnan(out[k, 0])
            continue
        want = fo.frechet_distance(mu_b, cov_b, *fo.embd_statistics(rows))
        assert out[k, 0] == pytest.approx(want, rel=2e-6, abs=1e-7 * (out[k, 5] + out[k, 6])), (k, len(rows), out[k, 0], want)


def _make_dir(root, kind, count, seconds):
    root.mkdir(parents=True)
    clips = []
    for i in range(count):
        pcm = synth.musiclike_clip(i, seconds, 16000, baseline=(kind == "base"))
        synth.write_wav(root / f"clip{i:03d}.wav", pcm, 16000)
        clips.append(pcm)
    return clips


def test_directory_flow_layout_and_score(vgg_engine, vgg_state, tmp_path):
    """fadtk <model> <baseline> <eval> flow: convert/ + embeddings/ + stats/ layout, then FAD."""
    base = _make_dir(tmp_path / "base", "base", 14, 10.0)
    evl = _make_dir(tmp_path / "eval", "eval", 14, 10.0)
    ml = fk.VGGishModel()
    for d in (tmp_path / "base", tmp_path / "eval"):
        fk.cache_embedding_files(d, ml, workers=4)
    assert (tmp_path / "eval" / "convert" / "16000" / "clip000.wav").exists()      # fad.py:143-160
    e0 = np.load(tmp_path / "eval" / "embeddings" / "vggish" / "clip000.npy")       # utils.py:60-68
    assert e0.dtype == np.float16 and e0.shape == (10, 128)                         # model_loader.py:47-48
    want0 = vo.embed(vo.load_wav_semantics(evl[0]), vgg_state)
    rel = np.sqrt(((e0.astype(np.float64) - want0) ** 2).mean() / (want0.astype(np.float64) ** 2).mean())
    assert rel < 3e-3
    fad = fk.FrechetAudioDistance(ml, audio_load_worker=2, load_model=False)
    score = fad.score(tmp_path / "base", tmp_path / "eval")
    assert (tmp_path / "eval" / "stats" / "vggish" / "cov.npy").exists()            # fad.py:286-288
    # same embeddings through the reference-pinned numpy oracle: per-file statistics + Chan merge
    # (utils.py:13-46, incl. its fp16 per-file means) is what the reference does for a directory
    def files(d):
        return [np.load(p) for p in sorted((d / "embeddings" / "vggish").glob("*.npy"))]
    want = fo.frechet_distance(*fo.online_statistics(files(tmp_path / "base")),
                               *fo.online_statistics(files(tmp_path / "eval")))
    assert score == pytest.approx(want, rel=1e-6)
    # second call is served from the caches
    fk.cache_embedding_files(tmp_path / "eval", ml, workers=4)
    assert fad.score(tmp_path / "base", tmp_path / "eval") == pytest.approx(score, rel=1e-12)


def test_plugin_get_embedding_single_clip(vgg_engine, vgg_state):
    ml = fk.VGGishModel()
    ml.load_model()
    pcm = synth.noise_clip(4, 0.5, 16000)                        # shorter than min_len: zero padded
    wav = ml.enforce_min_len(pcm / 32768.0)
    got = ml.get_embedding(wav)
    want = vo.embed(vo.load_wav_semantics(pcm), vgg_state)
    assert got.dtype == np.float16 and got.shape == want.shape == (1, 128)
    assert np.abs(got.astype(np.float32) - want.astype(np.float32)).max() < 5e-2 * np.abs(want.astype(np.float32)).max()


def test_fad_parity_1e4_on_identical_audio(vgg_engine, vgg_state):
    """north_star: FAD within 1e-4 relative of the reference CPU path on identical synthetic audio.
    100 + 100 ten-second clips -> 1000 + 1000 frames; CPU oracle = fp32 torch VGGish + fp16 cache
    rounding + numpy statistics + eig-route Frechet."""
    n = 100
    sets = {"base": [synth.musiclike_clip(i, 10.0, 16000, baseline=True) for i in range(n)],
            "eval": [synth.musiclike_clip(i, 10.0, 16000) for i in range(n)]}
    ml = fk.VGGishModel()
    ml.load_model()
    gpu = {k: np.concatenate(ml.embed_pcm_batch(v)) for k, v in sets.items()}
    cpu = {k: np.concatenate([vo.embed(vo.load_wav_semantics(c), vgg_state) for c in v]) for k, v in sets.items()}
    fad_gpu = fk.calc_frechet_distance(*fk.calc_embd_statistics(gpu["base"]), *fk.calc_embd_statistics(gpu["eval"]))
    fad_cpu = fo.frechet_distance(*fo.embd_statistics(cpu["base"]), *fo.embd_statistics(cpu["eval"]))
    rel = abs(fad_gpu - fad_cpu) / abs(fad_cpu)
    assert rel < 1e-4, f"FAD gpu {fad_gpu} vs cpu reference path {fad_cpu}: rel {rel}"


@pytest.mark.parametrize("name,seconds", [("encodec-emb", 2.0), ("whisper-tiny", 2.0), ("hubert-base-2", 2.0), ("clap-laion-music", 1.5)])
def test_directory_flow_for_every_embedder_family(engine, tmp_path, name, seconds):
    """cache_embedding_files (batched, fad_batch.py:25-48) must write what the plugin contract
    (load_wav -> get_embedding, model_loader.py:40-70) gives file by file, in the reference's cache layout."""
    ml = {m.name: m for m in fk.get_all_models()}[name]
    d = tmp_path / "set"
    d.mkdir()
    clips = []
    for i in range(3):
        pcm = synth.musiclike_clip(i, seconds + 0.25 * i, ml.sr)
        synth.write_wav(d / f"c{i}.wav", pcm, ml.sr)
        clips.append(pcm)
    fk.cache_embedding_files(d, ml, workers=2)
    for i, pcm in enumerate(clips):
        e = np.load(d / "embeddings" / name / f"c{i}.npy")
        assert e.dtype == np.float16 and e.ndim == 2 and e.shape[1] == ml.num_features
        one = ml.get_embedding(ml.load_wav(d / "convert" / str(ml.sr) / f"c{i}.wav"))
        assert np.array_equal(e, one), (name, i)
    mu, cov = fk.FrechetAudioDistance(ml, load_model=False).load_stats(d)
    assert mu.shape == (ml.num_features,) and cov.shape == (ml.num_features, ml.num_features) and np.isfinite(cov).all()


def test_baseline_config0_sine_vs_noise_one_second_clips(vgg_engine, vgg_state, tmp_path, monkeypatch):
    """BASELINE.json configs[0]: VGGish FAD of 32 x 1 s sine tones vs 32 x 1 s white noise.  One second = exactly ONE
    VGGish frame per file, so (a) the DIRECTORY path of the reference yields an all-NaN covariance (np.cov of one row,
    fadtk/utils.py:16) and the score fails - mirrored; (b) the plumbing check is the CONCATENATED path
    (calc_embd_statistics on the 32 x 128 matrix, rank <= 31: a singular product for fad.py:88-106), compared with
    the reference-pinned oracle on the same embeddings and with the full CPU oracle."""
    monkeypatch.delenv("FADTK_SINGLE_FRAME_FILES", raising=False)
    sets = {"sine": [synth.sine_clip(i, 1.0, 16000) for i in range(32)],
            "noise": [synth.noise_clip(i, 1.0, 16000) for i in range(32)]}
    ml = fk.VGGishModel()
    ml.load_model()
    gpu = {k: ml.embed_pcm_batch(v) for k, v in sets.items()}
    assert all(e.shape == (1, 128) and e.dtype == np.float16 for v in gpu.values() for e in v)

    # (b) concatenated path
    cat = {k: np.concatenate(v) for k, v in gpu.items()}
    fad_gpu = fk.calc_frechet_distance(*fk.calc_embd_statistics(cat["sine"]), *fk.calc_embd_statistics(cat["noise"]))
    fad_same = fo.frechet_distance(*fo.embd_statistics(cat["sine"]), *fo.embd_statistics(cat["noise"]))
    assert fad_gpu == pytest.approx(fad_same, rel=1e-6)
    cpu = {k: np.concatenate([vo.embed(vo.load_wav_semantics(c), vgg_state) for c in v]) for k, v in sets.items()}
    fad_cpu = fo.frechet_distance(*fo.embd_statistics(cpu["sine"]), *fo.embd_statistics(cpu["noise"]))
    print(f"config0: gpu {fad_gpu:.6f} oracle-on-gpu-embeddings {fad_same:.6f} cpu {fad_cpu:.6f} rel {abs(fad_gpu - fad_cpu) / fad_cpu:.2e}")
    assert fad_gpu == pytest.approx(fad_cpu, rel=1e-3)            # 32 rows in 128-d: ill-posed, looser than the 1e-4 of real sizes

    # (a) directory path: per-file caches with one row each
    paths = {}
    for k, v in gpu.items():
        d = tmp_path / k / "embeddings" / "vggish"
        d.mkdir(parents=True)
        paths[k] = []
        for i, e in enumerate(v):
            np.save(d / f"clip{i:03d}.npy", e)
            paths[k].append(d / f"clip{i:03d}.npy")
    mu, cov = fk.calculate_embd_statistics_online(paths["sine"])
    mu_ref, cov_ref = fo.online_statistics(gpu["sine"])
    assert np.isnan(cov).all() and np.isnan(cov_ref).all()        # the reference's behaviour, utils.py:16
    assert np.abs(mu - mu_ref).max() < 1e-12
    fad = fk.FrechetAudioDistance(ml, audio_load_worker=2, load_model=False)
    with pytest.raises(ValueError):                               # scipy's sqrtm refuses NaN input in the reference too (fad.py:88)
        fad.score(tmp_path / "sine", tmp_path / "noise")
    # extension: let single-frame files contribute their row -> the concatenated statistics
    monkeypatch.setenv("FADTK_SINGLE_FRAME_FILES", "keep")
    mu_k, cov_k = fk.calculate_embd_statistics_online(paths["sine"])
    x = cat["sine"].astype(np.float64)
    assert np.abs(mu_k - x.mean(0)).max() < 1e-12 and np.abs(cov_k - np.cov(x, rowvar=False)).max() < 1e-10 * np.abs(cov_k).max()


def test_bench_dumps_what_the_last_timed_step_returned(tmp_path):
    """bench.py --dump-outputs DIR: frechet.npy is the fp64[8] result of the last timed EvalSetFAD.run_device step,
    the vector the reported FAD is read from."""
    import json
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    r = subprocess.run([sys.executable, str(root / "bench.py"), "--clips", "16", "--baseline-clips", "16", "--steps", "2",
                        "--warmup", "0", "--no-cpu-baseline", "--no-e2e", "--files-clips", "0",
                        "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    got = np.load(tmp_path / "out" / "frechet.npy")
    assert got.dtype == np.float64 and got.shape == (8,)
    assert got[0] == line["fad"] and np.isfinite(got).all()
    assert sorted(p.name for p in (tmp_path / "out").iterdir()) == ["frechet.npy"]
