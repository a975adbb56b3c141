"""Regenerate tests/golden/*.npz by running the REAL reference (imported unchanged from
/root/reference through oracle/ref_shims.py).  Build-container only; the outputs are committed
because /root/reference does not exist on the GPU box.

    python -m oracle.make_golden

Fixtures
--------
frechet_fma_pop_128.npz    vggish vs encodec-emb statistics of fadtk/stats/fma_pop.npz (d=128,
                           real covariances, cond 2e3 / 5e4) -> calc_frechet_distance
frechet_spectra.npz        covariances with the REAL eigen-spectra of fma_pop's clap-laion-audio /
                           clap-laion-music (512), MERT-v1-95M-1/-4 (768) and clap-2023 / dac-44kHz
                           (1024) statistics, rotated by a seeded orthogonal matrix (keeps the file
                           small while keeping cond up to 1e9) -> calc_frechet_distance
stats_cases.npz            seeded fp16 embeddings -> calc_embd_statistics,
                           calculate_embd_statistics_online (incl. the n=1 NaN behaviour)
inf_case.npz               seeded fp16 embeddings, np.random.seed(0) -> score_inf
indiv_case.npz             per-song embeddings -> score_individual CSV rows
"""
from __future__ import annotations

import tempfile
from pathlib import Path

import numpy as np

from oracle.ref_shims import load_reference, REFERENCE_ROOT

OUT = Path(__file__).resolve().parent.parent / "tests" / "golden"


def spectrum_cov(evals: np.ndarray, seed: int) -> np.ndarray:
    """Q diag(evals) Q^T with Q from a seeded QR - reproducible from (evals, seed)."""
    d = evals.shape[0]
    q, r = np.linalg.qr(np.random.default_rng(seed).normal(size=(d, d)))
    q = q * np.sign(np.diag(r))
    c = (q * evals) @ q.T
    return 0.5 * (c + c.T)


class _FakeLoader:
    def __init__(self, name):
        self.name = name


def main():
    ref = load_reference()
    OUT.mkdir(parents=True, exist_ok=True)
    fma = np.load(REFERENCE_ROOT / "fadtk" / "stats" / "fma_pop.npz")

    # 1. real 128-d statistics
    a, b = "vggish", "encodec-emb"
    fad = ref.calc_frechet_distance(fma[a + ".mu"], fma[a + ".cov"], fma[b + ".mu"], fma[b + ".cov"])
    np.savez_compressed(OUT / "frechet_fma_pop_128.npz", mu1=fma[a + ".mu"], cov1=fma[a + ".cov"],
                        mu2=fma[b + ".mu"], cov2=fma[b + ".cov"], fad=np.float64(fad),
                        names=np.array([a, b]))
    print("fma_pop 128:", fad)

    # 2. real spectra, seeded rotations
    spec = {}
    for i, (a, b) in enumerate([("clap-laion-audio", "clap-laion-music"),
                                ("MERT-v1-95M-1", "MERT-v1-95M-4"), ("clap-2023", "dac-44kHz")]):
        ea = np.clip(np.linalg.eigvalsh(fma[a + ".cov"])[::-1], 0, None)
        eb = np.clip(np.linalg.eigvalsh(fma[b + ".cov"])[::-1], 0, None)
        c1, c2 = spectrum_cov(ea, 100 + i), spectrum_cov(eb, 200 + i)
        mu1, mu2 = fma[a + ".mu"], fma[b + ".mu"]
        fad = ref.calc_frechet_distance(mu1, c1, mu2, c2)
        spec[f"evals1_{i}"], spec[f"evals2_{i}"] = ea, eb
        spec[f"mu1_{i}"], spec[f"mu2_{i}"] = mu1, mu2
        spec[f"fad_{i}"] = np.float64(fad)
        spec[f"names_{i}"] = np.array([a, b])
        print("spectra", a, b, ea.shape, "cond", ea[0] / max(ea[-1], 1e-300), fad)
    np.savez_compressed(OUT / "frechet_spectra.npz", **spec)

    # 3. statistics
    rng = np.random.default_rng(1234)
    files = [(rng.normal(0.3, 1.5, (n, 128)) * rng.uniform(0.5, 2, 128)).astype(np.float16)
             for n in (10, 7, 2, 33, 10, 5)]
    cat = np.concatenate(files)
    mu_c, cov_c = ref.calc_embd_statistics(cat)
    with tempfile.TemporaryDirectory() as tmp:
        paths = []
        for i, f in enumerate(files):
            p = Path(tmp) / f"{i}.npy"
            np.save(p, f)
            paths.append(p)
        mu_o, cov_o = ref.calculate_embd_statistics_online(paths)
        p1 = Path(tmp) / "one.npy"
        np.save(p1, files[0][:1])
        with np.errstate(all="ignore"):
            mu_n, cov_n = ref.calculate_embd_statistics_online(paths + [p1])
    np.savez_compressed(OUT / "stats_cases.npz", sizes=np.array([f.shape[0] for f in files]), cat=cat,
                        mu_cat=mu_c, cov_cat=cov_c, mu_online=mu_o, cov_online=cov_o,
                        cov_with_single_frame_file_is_nan=np.array(bool(np.isnan(cov_n).all())))
    print("stats: mu dtype", mu_c.dtype, "online mu dtype", mu_o.dtype, "nan-case", np.isnan(cov_n).all())

    # 4. FAD-inf (fad.py:304-351) with the global RNG seeded; few rows keep the fixture small (about 250 kB)
    rng = np.random.default_rng(77)
    base = (rng.normal(0, 1, (256, 128)) * rng.uniform(0.5, 2, 128)).astype(np.float16)
    evl = (rng.normal(0.1, 1.1, (800, 128)) * rng.uniform(0.5, 2, 128)).astype(np.float16)
    mu_b, cov_b = ref.calc_embd_statistics(base)
    with tempfile.TemporaryDirectory() as tmp:
        np.savez(Path(tmp) / "base.npz", **{"gold.mu": mu_b, "gold.cov": cov_b})
        p = Path(tmp) / "eval.npy"
        np.save(p, evl)
        fad_obj = ref.FrechetAudioDistance(_FakeLoader("gold"), audio_load_worker=1, load_model=False)
        np.random.seed(0)
        res = fad_obj.score_inf(Path(tmp) / "base.npz", [p], steps=10, min_n=500)
    np.savez_compressed(OUT / "inf_case.npz", base=base, eval=evl, score=res.score, slope=res.slope,
                        r2=res.r2, points=np.array(res.points), steps=10, min_n=500)
    print("inf:", res.score, res.slope, res.r2)

    # 5. per-song (fad.py:353-395): 12 songs x (n_i, 128), one too short (dropped)
    rng = np.random.default_rng(99)
    songs = [(rng.normal(0.05 * i, 1 + 0.05 * i, (n, 128))).astype(np.float16)
             for i, n in enumerate((10, 10, 40, 10, 1, 10, 25, 10, 10, 130, 10, 10))]
    with tempfile.TemporaryDirectory() as tmp:
        tmp = Path(tmp)
        np.savez(tmp / "base.npz", **{"gold.mu": mu_b, "gold.cov": cov_b})
        (tmp / "ev" / "embeddings" / "gold").mkdir(parents=True)
        for i, s in enumerate(songs):
            (tmp / "ev" / f"song{i:02d}.wav").write_bytes(b"")
            np.save(tmp / "ev" / "embeddings" / "gold" / f"song{i:02d}.npy", s)
        fad_obj = ref.FrechetAudioDistance(_FakeLoader("gold"), audio_load_worker=1, load_model=False)
        import contextlib, io
        with contextlib.redirect_stderr(io.StringIO()):
            csv = fad_obj.score_individual(tmp / "base.npz", tmp / "ev", tmp / "out.csv")
        rows = [ln.split(",") for ln in Path(csv).read_text().splitlines()]
    names = np.array([Path(r[0]).name for r in rows])
    scores = np.array([float(r[1]) for r in rows])
    np.savez_compressed(OUT / "indiv_case.npz", mu_base=mu_b, cov_base=cov_b, names=names, scores=scores,
                        **{f"song{i:02d}": s for i, s in enumerate(songs)})
    print("indiv:", list(zip(names, scores))[:3], "... kept", len(rows), "of", len(songs))


def registry():
    """names / num_features / sample rates of the reference's get_all_models() (model_loader.py:676-701) ->
    tests/golden/registry.json.  Only the constructors run (no model code); laion_clap's version probe
    (model_loader.py:317) is answered with the locked version."""
    import importlib.metadata as md
    import json
    load_reference()
    real = md.version
    md.version = lambda name: "1.1.7" if name == "laion_clap" else real(name)
    try:
        from fadtk.model_loader import get_all_models
        rows = [[m.name, int(m.num_features), int(m.sr)] for m in get_all_models()]
    finally:
        md.version = real
    OUT.mkdir(parents=True, exist_ok=True)
    (OUT / "registry.json").write_text(json.dumps(rows, indent=0))
    print(f"registry.json: {len(rows)} models")


if __name__ == "__main__":
    main()
    registry()
