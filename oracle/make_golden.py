"""Generate tests/golden/*.npz from the UNMODIFIED reference (build container only).

    python -m oracle.make_golden

Every array below is an output of the reference's own modules imported from
/root/reference (see oracle/refshim.py); the weights are the reference's own
random init (``torch.manual_seed``), stored so the fixtures travel to the GPU box.
Configs are reduced (nf=16, 3 levels, F=64) so that the fixtures stay small; the
full-size reference outputs of tests/test_oracle_vs_reference.py are reference_live.npz.

    python -m oracle.make_golden reference_live    # reference_live.npz only
TEST INFRASTRUCTURE – see oracle/__init__.py.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import refshim, sde as sde_mod
from .arch import NetConfig, state_dict_manifest

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

SMALL = dict(nf=16, ch_mult=(1, 2, 2), image_size=64, num_res_blocks=2)


def _np(t):
    return t.detach().cpu().numpy()


def golden_network(name, backbone, cfg: NetConfig, seed):
    model = refshim.make_score_model(backbone=backbone, seed=seed, nf=cfg.nf, ch_mult=cfg.ch_mult,
                                     image_size=cfg.image_size, attn_resolutions=cfg.attn_resolutions,
                                     n_fft=126, hop_length=32)
    sd = model.dnn.state_dict()
    assert [k for k, _ in state_dict_manifest(cfg)] == list(sd.keys())
    g = torch.Generator().manual_seed(seed + 100)
    B, F, T = 2, 64, 64
    x = torch.complex(torch.randn(B, 1, F, T, generator=g), torch.randn(B, 1, F, T, generator=g)) * 0.3
    y = torch.complex(torch.randn(B, 1, F, T, generator=g), torch.randn(B, 1, F, T, generator=g)) * 0.3
    t = torch.tensor([0.83, 0.11])
    with torch.no_grad():
        dnn_out = model.dnn(torch.cat([x, y], dim=1), t)
        score = model(x, y, t)

    # PC sampler with injected noise.  'euler_maruyama' is not reachable through pc_sampler in the
    # reference: predictors.py:49 forwards `stepsize` into OUVESDE.sde() -> TypeError.
    samples = {}
    N = 3
    for pred, corr in [("reverse_diffusion", "ald"), ("reverse_diffusion", "langevin"), ("none", "ald"),
                       ("reverse_diffusion", "none")]:
        nd = sde_mod.n_noise_draws(N, pred, corr, 1)
        draws = sde_mod.make_noise((B, 1, F, T), nd, seed=7)
        with refshim.injected_noise(draws):
            smp, nfe = model.get_pc_sampler(pred, corr, y, N=N, corrector_steps=1, snr=0.5)()
        samples[f"pc_{pred}_{corr}"] = _np(smp)
        samples[f"nfe_{pred}_{corr}"] = np.int64(nfe)

    # full enhancement chain (enhancement.py:75-96 sequence on CPU)
    from sgmse.util.other import pad_spec
    L = 2000
    wav = 0.1 * torch.randn(B, L, generator=g)
    outs, Ys = [], []
    for b in range(B):
        yb = wav[b:b + 1]
        norm = yb.abs().max()
        Y = torch.unsqueeze(model._forward_transform(model._stft(yb / norm)), 0)
        Y = pad_spec(Y)
        draws = [d[b:b + 1] for d in sde_mod.make_noise((B, 1, F, Y.shape[-1]), sde_mod.n_noise_draws(N, "reverse_diffusion", "ald", 1), seed=11)]
        with refshim.injected_noise(draws):
            smp, _ = model.get_pc_sampler("reverse_diffusion", "ald", Y, N=N, corrector_steps=1, snr=0.5)()
        xh = model.to_audio(smp.squeeze(), L) * norm
        outs.append(_np(xh)); Ys.append(_np(Y[0]))
    np.savez_compressed(
        os.path.join(OUT, f"{name}.npz"),
        **{"w/" + k: _np(v) for k, v in sd.items()},
        x=_np(x), y=_np(y), t=_np(t), dnn_out=_np(dnn_out), score=_np(score),
        wav=_np(wav), enh=np.stack(outs), Y=np.stack(Ys), **samples)
    print(name, "params", sum(v.numel() for v in sd.values()))


PRECOND = {
    "plain": dict(loss_type="data_prediction", network_scaling=None, c_in="1", c_out="1", c_skip="0", sigma_data=0.1),
    "edm": dict(loss_type="data_prediction", network_scaling="1/sigma", c_in="edm", c_out="edm", c_skip="edm", sigma_data=0.1),
}


def golden_v2(name, cfg: NetConfig, seed):
    """SURVEY.md §8f-1: backbone 'ncsnpp_v2' behind ScoreModel.forward's preconditioning (model.py:283-304) with the
    Schroedinger-bridge SDE and both SB samplers (sampling/__init__.py:145-249), plus the OUVE predictor-corrector
    sampler driven by a score-matching v2 model.  One set of weights, several ScoreModel wrappers."""
    kw = dict(nf=cfg.nf, ch_mult=cfg.ch_mult, image_size=cfg.image_size, attn_resolutions=cfg.attn_resolutions,
              n_fft=126, hop_length=32)
    base = refshim.make_score_model(backbone="ncsnpp_v2", seed=seed, sde="sbve", k=2.6, c=0.4, N=3, **kw, **PRECOND["plain"])
    sd = base.dnn.state_dict()
    assert [k for k, _ in state_dict_manifest(cfg)] == list(sd.keys())
    g = torch.Generator().manual_seed(seed + 100)
    B, F, T = 2, 64, 64
    x = torch.complex(torch.randn(B, 1, F, T, generator=g), torch.randn(B, 1, F, T, generator=g)) * 0.3
    y = torch.complex(torch.randn(B, 1, F, T, generator=g), torch.randn(B, 1, F, T, generator=g)) * 0.3
    t = torch.tensor([0.83, 0.11])
    out = {}
    with torch.no_grad():
        out["dnn_out"] = _np(base.dnn(x, y, t))
        for tag, pre in PRECOND.items():
            m = refshim.make_score_model(backbone="ncsnpp_v2", seed=seed, sde="sbve", k=2.6, c=0.4, N=3, **kw, **pre)
            m.dnn.load_state_dict(sd)
            out[f"fwd_{tag}"] = _np(m(x, y, t))
            for st in ("sde", "ode"):
                draws = sde_mod.make_noise((B, 1, F, T), 3, seed=13)
                with refshim.injected_noise(draws):
                    smp, n = m.get_sb_sampler(m.sde, y, sampler_type=st)()
                out[f"sb_{st}_{tag}"] = _np(smp)
                out[f"sb_n_{st}_{tag}"] = np.int64(n)
        # OUVE + PC sampler on a score-matching v2 model (c_skip = 0, c_out = 1/sigma, network output unscaled)
        pre = dict(loss_type="score_matching", network_scaling=None, c_in="1", c_out="1/sigma", c_skip="0", sigma_data=0.1)
        m = refshim.make_score_model(backbone="ncsnpp_v2", seed=seed, **kw, **pre)
        m.dnn.load_state_dict(sd)
        out["fwd_ouve_score"] = _np(m(x, y, t))
        N = 3
        draws = sde_mod.make_noise((B, 1, F, T), sde_mod.n_noise_draws(N, "reverse_diffusion", "ald", 1), seed=7)
        with refshim.injected_noise(draws):
            smp, nfe = m.get_pc_sampler("reverse_diffusion", "ald", y, N=N, corrector_steps=1, snr=0.5)()
        out["pc_ouve_score"] = _np(smp)
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), **{"w/" + k: _np(v) for k, v in sd.items()},
                        x=_np(x), y=_np(y), t=_np(t), **out)
    print(name, "params", sum(v.numel() for v in sd.values()))


def golden_ops():
    """Op-level outputs of the reference layer library (FIR resamplers, STFT chain)."""
    refshim.import_reference()
    from sgmse.backbones.ncsnpp_utils import up_or_down_sampling as uds
    from sgmse.data_module import SpecsDataModule
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, 3, 8, 12, generator=g)
    dm = SpecsDataModule(base_dir="/nonexistent", n_fft=126, hop_length=32)
    dm48 = SpecsDataModule(base_dir="/nonexistent", n_fft=1534, hop_length=384, spec_factor=0.065,
                           spec_abs_exponent=0.667)
    wav = 0.1 * torch.randn(2, 2000, generator=g)
    wav48 = 0.1 * torch.randn(1, 6000, generator=g)
    S = dm.stft(wav)
    S48 = dm48.stft(wav48)
    np.savez_compressed(
        os.path.join(OUT, "ops.npz"),
        fir_x=_np(x), fir_down=_np(uds.downsample_2d(x, (1, 3, 3, 1), factor=2)),
        fir_up=_np(uds.upsample_2d(x, (1, 3, 3, 1), factor=2)),
        wav=_np(wav), stft=_np(S), spec_fwd=_np(dm.spec_fwd(S)), spec_back=_np(dm.spec_back(dm.spec_fwd(S))),
        istft=_np(dm.istft(S, 2000)),
        wav48=_np(wav48), stft48=_np(S48), spec_fwd48=_np(dm48.spec_fwd(S48)), istft48=_np(dm48.istft(S48, 6000)))


def golden_ode(name, src_name, backbone, cfg: NetConfig, seed):
    """SURVEY.md §8f-4: the probability-flow ODE sampler (sampling/__init__.py:72-143; scipy RK45 through host numpy
    round trips) of the unmodified reference, prior draw injected, ``denoise=False`` (``denoise=True`` raises TypeError in
    the reference, predictors.py:60).  The network is the one of ``src_name``.npz (same seed -> same init; asserted)."""
    model = refshim.make_score_model(backbone=backbone, seed=seed, nf=cfg.nf, ch_mult=cfg.ch_mult,
                                     image_size=cfg.image_size, attn_resolutions=cfg.attn_resolutions,
                                     n_fft=126, hop_length=32)
    z = np.load(os.path.join(OUT, src_name + ".npz"))
    for k, v in model.dnn.state_dict().items():
        assert np.array_equal(z["w/" + k], _np(v)), k
    y = torch.from_numpy(z["y"])
    out = {}
    for tag, tol in (("loose", 1e-3), ("default", 1e-5)):
        draws = sde_mod.make_noise(tuple(y.shape), 1, seed=17)
        with refshim.injected_noise(draws):
            smp, nfe = model.get_ode_sampler(y, denoise=False, device="cpu", rtol=tol, atol=tol)()
        out[f"x_{tag}"] = _np(smp)
        out[f"nfe_{tag}"] = np.int64(nfe)
        out[f"tol_{tag}"] = np.float64(tol)
        print(name, tag, "nfe", nfe)
    try:
        with refshim.injected_noise(sde_mod.make_noise(tuple(y.shape), 1, seed=17)):
            model.get_ode_sampler(y, device="cpu", rtol=1e-3, atol=1e-3)()
        out["denoise_default_raises"] = np.int64(0)
    except TypeError as exc:
        out["denoise_default_raises"] = np.int64(1)
        print("denoise=True ->", type(exc).__name__, exc)
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), y=_np(y), prior_seed=np.int64(17), **out)


def golden_full_n30(name="full_n30"):
    """BASELINE.json configs[0] through the UNMODIFIED reference: one 4-s 16 kHz clip, full-size NCSN++ (65.6 M
    parameters), OUVE SDE, predictor-corrector sampler reverse_diffusion + ald, N = 30, snr = 0.5 -- the sequence of
    model.enhance (model.py:433-459) / enhancement.py:75-96 on CPU, ~5 minutes on 8 cores.  The weights are the oracle's
    seeded init (oracle/weights.py, seed 0) loaded into the reference model, the clip is bench.py's synthetic utterance 0
    and the 61 noise draws come from seeds -- all three are regenerated on the GPU box, only the reference's OUTPUT is
    stored (enhanced waveform + final spectrogram, 1.3 MB)."""
    import time
    from . import weights as o_w
    from sgmse_b200.synth import synthetic_speech
    cfg = NetConfig.ncsnpp()
    model = refshim.make_score_model("ncsnpp", seed=0)
    from sgmse.util.other import pad_spec
    model.dnn.load_state_dict(o_w.make_state_dict(cfg, seed=0))
    L, N = 64000, 30
    wav = synthetic_speech(1, L)                                   # 0.1 * randn, torch.manual_seed(1000)
    t0 = time.time()
    norm = wav.abs().max()
    Y = torch.unsqueeze(model._forward_transform(model._stft(wav / norm)), 0)
    Y = pad_spec(Y)
    draws = sde_mod.make_noise(tuple(Y.shape), sde_mod.n_noise_draws(N, "reverse_diffusion", "ald", 1), seed=2000)
    with refshim.injected_noise(draws), torch.no_grad():
        sample, nfe = model.get_pc_sampler("reverse_diffusion", "ald", Y, N=N, corrector_steps=1, snr=0.5)()
    x_hat = model.to_audio(sample.squeeze(), L) * norm
    print(name, "reference CPU run", round(time.time() - t0, 1), "s, nfe", nfe, "threads", torch.get_num_threads())
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), enh=_np(x_hat.reshape(-1)), sample=_np(sample[0, 0]),
                        nfe=np.int64(nfe), N=np.int64(N), L=np.int64(L), wav_seed=np.int64(1000), weight_seed=np.int64(0),
                        noise_seed=np.int64(2000), snr=np.float64(0.5), cpu_seconds=np.float64(time.time() - t0),
                        cpu_threads=np.int64(torch.get_num_threads()))


V2_ODE_PRECOND = {
    "score": dict(loss_type="score_matching", network_scaling=None, c_in="1", c_out="1/sigma", c_skip="0", sigma_data=0.1),
    "denoiser_edm_in": dict(loss_type="denoiser", network_scaling="1/t", c_in="edm", c_out="1", c_skip="0", sigma_data=0.1),
}


def golden_ode_v2(name="ode_v2_small"):
    """The probability-flow ODE sampler on preconditioned 'ncsnpp_v2' score models with the OUVE SDE (get_ode_sampler calls
    ScoreModel.forward(x, y, t), i.e. model.py:283-304): the weights of ncsnpp_v2_small.npz under two ScoreModel wrappers --
    a plain score-matching model, and a 'denoiser' model with c_in = 'edm' and 1/t network scaling (every evaluation
    rescales the network input)."""
    cfg = NetConfig.ncsnpp_v2(attn_resolutions=(16,), **SMALL)
    kw = dict(nf=cfg.nf, ch_mult=cfg.ch_mult, image_size=cfg.image_size, attn_resolutions=cfg.attn_resolutions,
              n_fft=126, hop_length=32)
    z = np.load(os.path.join(OUT, "ncsnpp_v2_small.npz"))
    sd = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w/")}
    y = torch.from_numpy(z["y"])
    out = {}
    for tag, pre in V2_ODE_PRECOND.items():
        m = refshim.make_score_model(backbone="ncsnpp_v2", seed=3, **kw, **pre)
        m.dnn.load_state_dict(sd)
        with refshim.injected_noise(sde_mod.make_noise(tuple(y.shape), 1, seed=19)):
            smp, nfe = m.get_ode_sampler(y, denoise=False, device="cpu", rtol=1e-3, atol=1e-3)()
        out[f"x_{tag}"] = _np(smp)
        out[f"nfe_{tag}"] = np.int64(nfe)
        print(name, tag, "nfe", nfe, "finite", bool(torch.isfinite(torch.view_as_real(smp)).all()))
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), y=_np(y), prior_seed=np.int64(19), tol=np.float64(1e-3), **out)


MID = dict(nf=64, ch_mult=(1, 2, 2), image_size=64, attn_resolutions=(16,), num_res_blocks=1)


def golden_mid_tc(name="ncsnpp_mid"):
    """Reference-generated sampler / enhancement fixtures on a config whose layers are tcgen05-tileable (64..128 channels),
    so that the PRODUCT mode (fp16_tc) -- not only the fp32 validation mode -- is compared with outputs of the unmodified
    reference (VERDICT r1, weak #1).  Like full_n30: weights (oracle/weights.py seed 5, loaded into the reference model),
    inputs and noise are regenerated from seeds on the GPU box; only the reference's OUTPUTS are stored.
    Sampler: the four predictor/corrector pairs at N = 3, the default pair also at N = 12 (24 evaluations: drift over a
    longer chain); chain: enhancement.py:75-96 at N = 6 on two clips."""
    from . import weights as o_w
    cfg = NetConfig.ncsnpp(**MID)
    model = refshim.make_score_model("ncsnpp", seed=0, n_fft=126, hop_length=32, **MID)
    from sgmse.util.other import pad_spec
    model.dnn.load_state_dict(o_w.make_state_dict(cfg, seed=5))
    g = torch.Generator().manual_seed(105)
    B, F, T = 2, 64, 128
    y = torch.complex(torch.randn(B, 1, F, T, generator=g), torch.randn(B, 1, F, T, generator=g)) * 0.3
    x = y + 0.2 * torch.complex(torch.randn(B, 1, F, T, generator=g), torch.randn(B, 1, F, T, generator=g))
    t = torch.tensor([0.83, 0.11])
    out = {}
    with torch.no_grad():
        out["score"] = _np(model(x, y, t))
    for pred, corr, N in [("reverse_diffusion", "ald", 3), ("reverse_diffusion", "langevin", 3), ("none", "ald", 3),
                          ("reverse_diffusion", "none", 3), ("reverse_diffusion", "ald", 12)]:
        draws = sde_mod.make_noise((B, 1, F, T), sde_mod.n_noise_draws(N, pred, corr, 1), seed=7)
        with refshim.injected_noise(draws):
            smp, nfe = model.get_pc_sampler(pred, corr, y, N=N, corrector_steps=1, snr=0.5)()
        out[f"pc_{pred}_{corr}_N{N}"] = _np(smp)
        out[f"nfe_{pred}_{corr}_N{N}"] = np.int64(nfe)
    # BASELINE config 4 sampler settings (README.md:43: dereverberation checkpoint, --N 50 --snr 0.33): 100 evaluations
    draws = sde_mod.make_noise((B, 1, F, T), sde_mod.n_noise_draws(50, "reverse_diffusion", "ald", 1), seed=9)
    with refshim.injected_noise(draws):
        smp, nfe = model.get_pc_sampler("reverse_diffusion", "ald", y, N=50, corrector_steps=1, snr=0.33)()
    out["pc_dereverb_N50_snr033"] = _np(smp)
    out["nfe_dereverb_N50_snr033"] = np.int64(nfe)
    L, N = 4000, 6
    wav = 0.1 * torch.randn(B, L, generator=g)
    enh = []
    for b in range(B):
        yb = wav[b:b + 1]
        norm = yb.abs().max()
        Y = pad_spec(torch.unsqueeze(model._forward_transform(model._stft(yb / norm)), 0))
        draws = [d[b:b + 1] for d in sde_mod.make_noise((B, 1, F, Y.shape[-1]), sde_mod.n_noise_draws(N, "reverse_diffusion", "ald", 1), seed=11)]
        with refshim.injected_noise(draws):
            smp, _ = model.get_pc_sampler("reverse_diffusion", "ald", Y, N=N, corrector_steps=1, snr=0.5)()
        enh.append(_np(model.to_audio(smp.squeeze(), L) * norm))
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), x=_np(x), y=_np(y), t=_np(t), wav=_np(wav), enh=np.stack(enh),
                        weight_seed=np.int64(5), input_seed=np.int64(105), **out)
    print(name, "params", sum(v.numel() for v in model.dnn.state_dict().values()))


def score_model_skeleton(model) -> dict:
    """Everything ``sgmse_b200.config_from_score_model`` / ``install`` read from a live ScoreModel, as plain data: the
    NCSN++ attributes, the type name (and ``out_ch``) of every entry of ``dnn.all_modules``, the data module's STFT
    settings and window, the SDE and the state_dict layout.  tests/test_oracle_vs_reference.py rebuilds a stand-in from it."""
    dnn, dm, sde = model.dnn, model.data_module, model.sde
    d = {"backbone": model.backbone, "t_eps": float(model.t_eps), "sr": int(getattr(model, "sr", 16000)),
         "dnn": {a: getattr(dnn, a) for a in ("nf", "num_resolutions", "num_res_blocks", "progressive", "progressive_input",
                                             "resblock_type", "embedding_type", "skip_rescale", "conditional", "centered",
                                             "scale_by_sigma") if hasattr(dnn, a)},
         "all_modules": [[type(m).__name__, getattr(m, "out_ch", None)] for m in dnn.all_modules],
         "data_module": {"transform_type": dm.transform_type, "n_fft": dm.n_fft, "hop_length": dm.hop_length,
                         "spec_factor": float(dm.spec_factor), "spec_abs_exponent": float(dm.spec_abs_exponent),
                         "window": dm.window.float().tolist()},
         "sde": {"type": type(sde).__name__, "N": sde.N,
                 **{a: float(getattr(sde, a)) for a in ("theta", "sigma_min", "sigma_max", "k", "c", "eps") if hasattr(sde, a)},
                 **({"sampler_type": sde.sampler_type} if hasattr(sde, "sampler_type") else {})},
         "state_dict": [[k, list(v.shape)] for k, v in dnn.state_dict().items()]}
    d["dnn"]["attn_resolutions"] = list(dnn.attn_resolutions)
    d["dnn"]["all_resolutions"] = list(dnn.all_resolutions)
    for a in ("loss_type", "network_scaling", "c_in", "c_out", "c_skip", "sigma_data"):
        if hasattr(model, a):
            d[a] = getattr(model, a)
    return d


REF_48K = dict(n_fft=1534, hop_length=384, spec_factor=0.065, spec_abs_exponent=0.667, theta=2.0, sigma_min=0.1, sigma_max=1.0)
REF_V2_SBVE = dict(sde="sbve", k=2.6, c=0.4, sampler_type="sde", N=50, loss_type="data_prediction", network_scaling="1/sigma",
                   c_in="edm", c_out="edm", c_skip="edm")
# (theta, sigma_min, sigma_max), N, snr: BASELINE configs 2, 4 and 3
SCHEDULES = [((1.5, 0.05, 0.5), 30, 0.5), ((1.5, 0.05, 0.5), 50, 0.33), ((2.0, 0.1, 1.0), 30, 0.5)]
DROPIN_MID = dict(nf=64, ch_mult=(1, 2, 2), image_size=64, attn_resolutions=(16,), num_res_blocks=1, n_fft=126, hop_length=32)
DROPIN_LENGTHS = [4000, 1900, 3100, 2000]


def golden_reference_live(name="reference_live"):
    """What tests/test_oracle_vs_reference.py and the batched-service test of tests/test_gpu_dropin.py compare with: outputs
    of the unmodified reference at full size (NCSN++ forward, the enhancement.py:75-96 chain at N = 1), its SDE scalars and
    sampler schedules, its probability-flow ODE sampler on a 48 kHz configuration, its per-file enhancement loop on a
    tcgen05-tileable configuration, and the attribute skeletons of three live ScoreModels (JSON, key 'score_models').  Weights are
    the oracle's seeded init (oracle/weights.py) loaded into the reference model; inputs and noise come from seeds."""
    import json
    from . import weights as o_w
    refshim.import_reference()
    from sgmse.util.other import pad_spec
    from sgmse.sdes import OUVESDE
    from sgmse_b200 import Engine, EngineConfig
    out, skel = {}, {}
    cfg = NetConfig.ncsnpp()
    m16 = refshim.make_score_model("ncsnpp", seed=0)
    skel["ncsnpp"] = score_model_skeleton(m16)
    out["fwd_keys"] = np.array(list(m16.dnn.state_dict().keys()))
    m16.dnn.load_state_dict(o_w.make_state_dict(cfg, seed=0))
    g = torch.Generator().manual_seed(0)
    x = torch.complex(torch.randn(1, 2, 256, 64, generator=g), torch.randn(1, 2, 256, 64, generator=g)) * 0.3
    with torch.no_grad():
        out["fwd_out"] = _np(m16.dnn(x, torch.tensor([0.4])))
    ts = torch.tensor([1.0, 0.5, 0.03])
    out["sde_t"] = _np(ts)
    out["sde_std"] = np.array([float(m16.sde._std(t[None])) for t in ts])
    out["sde_diffusion"] = np.array([float(m16.sde.sde(torch.zeros(1), torch.zeros(1), t[None])[1]) for t in ts])
    # enhancement.py:75-96, N = 1, full-size network, one 0.5-s clip (63 frames -> padded to 64)
    g = torch.Generator().manual_seed(4)
    L = 8000
    wav = 0.1 * torch.randn(1, L, generator=g)
    draws = sde_mod.make_noise((1, 1, 256, 64), 3, seed=5)
    norm = wav.abs().max()
    Y = pad_spec(torch.unsqueeze(m16._forward_transform(m16._stft(wav / norm)), 0))
    with refshim.injected_noise(draws):
        smp, nfe = m16.get_pc_sampler("reverse_diffusion", "ald", Y, N=1, corrector_steps=1, snr=0.5)()
    out["chain_enh"] = _np(m16.to_audio(smp.squeeze(), L) * norm)
    out["chain_nfe"] = np.int64(nfe)
    # get_ode_sampler's default denoise=True fails inside the reference (predictors.py:60)
    try:
        m16.get_ode_sampler(torch.zeros(1, 1, 256, 64, dtype=torch.complex64), device="cpu", rtol=1e-1, atol=1e-1)()
        out["ode_default_error"] = np.array("")
    except TypeError as exc:
        out["ode_default_error"] = np.array(str(exc))
    # sampler schedules: the reference's scalars on the engine's own fp32 time steps
    for i, ((theta, smin, smax), N, snr) in enumerate(SCHEDULES):
        sde = OUVESDE(theta=theta, sigma_min=smin, sigma_max=smax, N=N)
        eng = Engine(EngineConfig(theta=theta, sigma_min=smin, sigma_max=smax, t_eps=0.03))
        ets = eng.sampler_schedule(N=N, predictor="reverse_diffusion", corrector="ald", corrector_steps=1, snr=snr)[0]
        eng.close()
        x0 = torch.zeros(1, 1, 1, 1, dtype=torch.complex64)
        y0 = torch.ones(1, 1, 1, 1, dtype=torch.complex64)
        std, f, G = [], [], []
        for j in range(N):
            t = ets[j:j + 1]
            stepsize = ets[j] - ets[j + 1] if j != N - 1 else ets[-1]
            std.append(float(sde._std(t)))
            fj, Gj = sde.discretize(x0, y0, t, stepsize)
            f.append(float(fj.real))
            G.append(float(Gj))
        out[f"sched{i}_linspace"] = _np(torch.linspace(sde.T, 0.03, N))
        out[f"sched{i}_ts"] = _np(ets)
        out[f"sched{i}_std1"] = np.float64(float(sde._std(torch.ones(1))))
        out[f"sched{i}_std"], out[f"sched{i}_f"], out[f"sched{i}_G"] = np.array(std), np.array(f), np.array(G)
    # probability-flow ODE, 48 kHz SDE parameters, eps = 0.05, batch of 2 = one coupled ODE system
    small = dict(nf=16, ch_mult=(1, 2, 2), image_size=64, num_res_blocks=2)
    m = refshim.make_score_model("ncsnpp_48k", seed=5, n_fft=126, hop_length=32, theta=2.0, sigma_min=0.1, sigma_max=1.0, **small)
    m.dnn.load_state_dict(o_w.make_state_dict(NetConfig.ncsnpp_48k(**small), seed=5))
    g = torch.Generator().manual_seed(3)
    y = torch.complex(torch.randn(2, 1, 64, 64, generator=g), torch.randn(2, 1, 64, 64, generator=g)) * 0.3
    with refshim.injected_noise(sde_mod.make_noise(tuple(y.shape), 1, seed=23)):
        smp, nfe = m.get_ode_sampler(y, denoise=False, device="cpu", rtol=1e-3, atol=1e-3, eps=0.05)()
    out["ode_x"], out["ode_nfe"] = _np(smp), np.int64(nfe)
    # the reference's per-file loop (enhancement.py:58-99) over clips of four lengths, N = 3
    mcfg = {k: v for k, v in DROPIN_MID.items() if k not in ("n_fft", "hop_length")}
    m = refshim.make_score_model("ncsnpp", seed=7, **DROPIN_MID)
    m.dnn.load_state_dict(o_w.make_state_dict(NetConfig.ncsnpp(**mcfg), seed=7))
    g = torch.Generator().manual_seed(8)
    nd = sde_mod.n_noise_draws(3, "reverse_diffusion", "ald", 1)
    for i, n in enumerate(DROPIN_LENGTHS):
        clip = (0.1 * torch.randn(n, generator=g) * (1.0 + 0.5 * i))[None]
        norm = clip.abs().max()
        Y = pad_spec(torch.unsqueeze(m._forward_transform(m._stft(clip / norm)), 0), mode="zero_pad")
        with refshim.injected_noise(sde_mod.make_noise((1, 1, 64, Y.shape[-1]), nd, seed=40 + i)):
            smp, _ = m.get_pc_sampler("reverse_diffusion", "ald", Y, N=3, corrector_steps=1, snr=0.5)()
        out[f"files_enh{i}"] = _np((m.to_audio(smp.squeeze(), n) * norm).squeeze())
    skel["ncsnpp_48k"] = score_model_skeleton(refshim.make_score_model("ncsnpp_48k", seed=0, **REF_48K))
    skel["ncsnpp_v2_sbve"] = score_model_skeleton(refshim.make_score_model("ncsnpp_v2", seed=0, **REF_V2_SBVE))
    out["score_models"] = np.array(json.dumps(skel, separators=(",", ":")))
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), **out)


def main():
    os.makedirs(OUT, exist_ok=True)
    golden_ops()
    golden_network("ncsnpp_small", "ncsnpp", NetConfig.ncsnpp(attn_resolutions=(16,), **SMALL), seed=1)
    golden_network("ncsnpp48k_small", "ncsnpp_48k", NetConfig.ncsnpp_48k(**SMALL), seed=2)
    golden_v2("ncsnpp_v2_small", NetConfig.ncsnpp_v2(attn_resolutions=(16,), **SMALL), seed=3)
    golden_ode("ode_small", "ncsnpp_small", "ncsnpp", NetConfig.ncsnpp(attn_resolutions=(16,), **SMALL), seed=1)
    golden_ode("ode48k_small", "ncsnpp48k_small", "ncsnpp_48k", NetConfig.ncsnpp_48k(**SMALL), seed=2)
    golden_ode_v2()
    golden_mid_tc()
    golden_full_n30()            # ~2.5 minutes: the full-size reference run
    golden_reference_live()


if __name__ == "__main__":
    import sys
    if sys.argv[1:] == ["reference_live"]:        # this fixture alone: leaves the others untouched
        os.makedirs(OUT, exist_ok=True)
        golden_reference_live()
    else:
        main()
