"""The oracle and the host-side boundary against the UNMODIFIED reference.

What the reference computed -- full-size outputs, SDE scalars, sampler schedules, the ODE sampler, and the attribute skeletons
of live ScoreModels -- is stored in tests/golden/reference_live.npz (oracle/make_golden.py: golden_reference_live), so these tests run from the repository alone.  The weights are the
oracle's seeded init loaded into the reference model, regenerated here from the same seed.  The two tests that need the
reference's ScoreModel class itself (its EMA swap in train / eval, the staged copy) run only where the reference is importable."""
import json
import os
import types

import numpy as np
import pytest
import torch

from oracle import refshim, ncsnpp as o_net, sde as o_sde, spec as o_spec, pipeline as o_pipe, weights as o_w
from oracle.arch import NetConfig, state_dict_manifest

live = pytest.mark.skipif(not refshim.reference_available(), reason="reference checkout not present")


@pytest.fixture(scope="module")
def ref(golden_dir):
    return np.load(os.path.join(golden_dir, "reference_live.npz"))


@pytest.fixture(scope="module")
def skeletons(ref):
    return json.loads(str(ref["score_models"]))


class RecordedScoreModel:
    """Stand-in for a live ScoreModel, rebuilt from the attributes recorded from one (oracle/make_golden.py:
    score_model_skeleton): every value config_from_score_model reads, the module types of dnn.all_modules, and a
    zero-filled state_dict with the reference's names, order and shapes."""

    def __init__(self, d):
        kinds = {}

        def instance(type_name, **attrs):
            cls = kinds.setdefault(type_name, type(type_name, (), {}))
            obj = cls()
            obj.__dict__.update(attrs)
            return obj

        layout = [(k, tuple(s)) for k, s in d["state_dict"]]
        self.backbone, self.t_eps, self.sr = d["backbone"], d["t_eps"], d["sr"]
        self.dnn = types.SimpleNamespace(**d["dnn"], all_modules=[instance(n, **({} if oc is None else {"out_ch": oc}))
                                                                   for n, oc in d["all_modules"]],
                                         state_dict=lambda: {k: torch.zeros(s) for k, s in layout})
        dm = dict(d["data_module"])
        dm["window"] = torch.tensor(dm["window"])
        self.data_module = types.SimpleNamespace(**dm)
        self.sde = instance(d["sde"]["type"], **{k: v for k, v in d["sde"].items() if k != "type"})
        for a in ("loss_type", "network_scaling", "c_in", "c_out", "c_skip", "sigma_data"):
            if a in d:
                setattr(self, a, d[a])


@pytest.fixture(scope="module")
def recorded16k(skeletons):
    return RecordedScoreModel(skeletons["ncsnpp"])


@pytest.fixture(scope="module")
def model16k():
    return refshim.make_score_model("ncsnpp", seed=0)


def test_full_size_forward_matches_reference(ref):
    cfg = NetConfig.ncsnpp()
    assert [k for k, _ in state_dict_manifest(cfg)] == ref["fwd_keys"].tolist()
    sd = o_w.make_state_dict(cfg, seed=0)
    g = torch.Generator().manual_seed(0)
    x = torch.complex(torch.randn(1, 2, 256, 64, generator=g), torch.randn(1, 2, 256, 64, generator=g)) * 0.3
    t = torch.tensor([0.4])
    with torch.no_grad():
        got = o_net.forward(sd, cfg, x, t)
    r = torch.from_numpy(ref["fwd_out"])
    assert ((r - got).abs().max() / r.abs().max()).item() < 1e-5


def test_sde_scalars_match_reference(ref):
    o = o_sde.OUVE()
    for t, std, diffusion in zip(ref["sde_t"].tolist(), ref["sde_std"], ref["sde_diffusion"]):
        assert abs(std - o.std(t)) < 1e-6
        assert abs(diffusion - o.diffusion(t)) < 1e-6
    assert abs(o.std(1.0) - 0.38898) < 1e-4          # SURVEY.md §8a


def test_config_is_recovered_from_a_live_score_model(recorded16k):
    from sgmse_b200 import config_from_score_model, Engine
    cfg = config_from_score_model(recorded16k, mode="fp16_tc", max_batch=4)
    assert cfg.backbone == "ncsnpp" and cfg.nf == 128 and tuple(cfg.ch_mult) == (1, 1, 2, 2, 2, 2, 2)
    assert tuple(cfg.attn_resolutions) == (16,) and cfg.image_size == 256 and cfg.num_res_blocks == 2
    assert (cfg.n_fft, cfg.hop_length, cfg.window) == (510, 128, "hann")
    assert abs(cfg.theta - 1.5) < 1e-9 and abs(cfg.t_eps - 0.03) < 1e-9
    eng = Engine(cfg)
    sd = recorded16k.dnn.state_dict()
    blob = eng.flatten_state_dict(sd)      # names, order and sizes all agree
    assert blob.numel() == sum(p.numel() for p in sd.values())
    eng.close()


def test_config_48k(skeletons):
    from sgmse_b200 import config_from_score_model, Engine
    m = RecordedScoreModel(skeletons["ncsnpp_48k"])
    cfg = config_from_score_model(m)
    assert cfg.backbone == "ncsnpp_48k" and cfg.progressive == "none" and cfg.progressive_input == "none"
    assert tuple(cfg.attn_resolutions) == () and cfg.n_fft == 1534
    eng = Engine(cfg)
    assert eng.flatten_state_dict(m.dnn.state_dict()).numel() == eng.weights_numel()
    eng.close()


def test_enhance_chain_matches_reference_sequence(ref):
    """Oracle pipeline vs the enhancement.py:75-96 sequence of the reference, N=1, injected noise, short clip."""
    g = torch.Generator().manual_seed(4)
    L = 8000                                   # 63 frames -> padded to 64
    wav = 0.1 * torch.randn(1, L, generator=g)
    draws = o_sde.make_noise((1, 1, 256, 64), 3, seed=5)
    cfg = NetConfig.ncsnpp()
    got = o_pipe.enhance(o_w.make_state_dict(cfg, seed=0), cfg, o_spec.SpecConfig(), o_sde.OUVE(), wav, draws, N=1)
    r = torch.from_numpy(ref["chain_enh"])
    assert int(ref["chain_nfe"]) == 2
    assert ((r - got[0]).abs().max() / r.abs().max()).item() < 1e-3


SCHEDULES = [(1.5, 30, 0.5), (1.5, 50, 0.33), (2.0, 30, 0.5)]      # order of oracle/make_golden.py SCHEDULES


@pytest.mark.parametrize("sde_kw,N,snr", [
    (dict(theta=1.5, sigma_min=0.05, sigma_max=0.5), 30, 0.5),      # config 2 (VoiceBank-DEMAND), model.py:426 defaults
    (dict(theta=1.5, sigma_min=0.05, sigma_max=0.5), 50, 0.33),     # config 4 (WSJ0-REVERB, README.md:43)
    (dict(theta=2.0, sigma_min=0.1, sigma_max=1.0), 30, 0.5),       # config 3 (EARS-WHAM 48 kHz, README.md:89)
])
def test_sampler_schedule_matches_reference_scalars(ref, sde_kw, N, snr):
    """Every per-step scalar the captured launch sequence bakes in (engine.cu: make_tables, exported through
    sgmse_b200_sampler_schedule) against the reference's own objects: OUVESDE._std / .sde / .discretize
    (sdes.py:188-219,72-89), the step sizes of sampling/__init__.py:56-62, AnnealedLangevinDynamics' step size
    (correctors.py:69-81) and ReverseDiffusionPredictor (predictors.py:60-65).  Host-only: runs without a GPU."""
    from sgmse_b200 import Engine, EngineConfig
    k = f"sched{SCHEDULES.index((sde_kw['theta'], N, snr))}_"
    eng = Engine(EngineConfig(**sde_kw, t_eps=0.03))
    ts, std1, coef = eng.sampler_schedule(N=N, predictor="reverse_diffusion", corrector="ald", corrector_steps=1, snr=snr)
    eng.close()
    ref_ts = torch.from_numpy(ref[k + "linspace"])
    # the engine follows the CUDA linspace kernel the reference runs on a GPU (one rounding per element); the vectorised
    # CPU kernel rounds twice (base + step * lane) and may differ in the last bit
    assert torch.allclose(ts, ref_ts, rtol=2.5e-7, atol=0.0)
    assert abs(std1 - float(ref[k + "std1"])) < 1e-6 * std1 + 1e-7
    assert coef.shape == (2 * N, 3)
    # step sizes are differences of neighbouring fp32 time steps (sampling/__init__.py:59-62): a last-bit difference
    # in the linspace is 3e-6 of dt, so the reference's formulas were evaluated on the engine's own time steps
    assert torch.equal(ts, torch.from_numpy(ref[k + "ts"]))
    for i in range(N):
        eps = 2 * (snr * float(ref[k + "std"][i])) ** 2
        cy, cs, cz = coef[2 * i].tolist()                      # corrector row
        assert cy == 0.0 and abs(cs - eps) <= 2e-6 * eps and abs(cz - (2 * eps) ** 0.5) <= 2e-6 * (2 * eps) ** 0.5
        f, G = float(ref[k + "f"][i]), float(ref[k + "G"][i])  # f = theta (y - x) dt with y - x = 1, G = g sqrt(dt)
        cy, cs, cz = coef[2 * i + 1].tolist()                  # predictor row: x_mean = x - (f - G^2 score)
        assert abs(cy + f) <= 2e-6 * abs(f)
        assert abs(cz - G) <= 2e-6 * G and abs(cs - G ** 2) <= 4e-6 * G ** 2


def test_config_v2_sbve_is_recovered_and_rebound(skeletons):
    """SURVEY.md §8f-1: a ScoreModel(backbone='ncsnpp_v2', sde='sbve') is read back completely (architecture, SB
    parameters, preconditioning attributes) and install() rebinds forward / get_sb_sampler / enhance (host side only)."""
    import sgmse_b200
    from sgmse_b200 import config_from_score_model, Engine
    m = RecordedScoreModel(skeletons["ncsnpp_v2_sbve"])
    cfg = config_from_score_model(m)
    assert cfg.backbone == "ncsnpp_v2" and not cfg.scale_by_sigma and cfg.sde == "sbve"
    assert (cfg.sb_k, cfg.sb_c) == (2.6, 0.4) and cfg.nf == 128 and tuple(cfg.ch_mult) == (1, 1, 2, 2, 2, 2, 2)
    assert (cfg.loss_type, cfg.network_scaling, cfg.c_in, cfg.c_out, cfg.c_skip) == ("data_prediction", "1/sigma", "edm", "edm", "edm")
    eng = Engine(cfg)
    assert eng.flatten_state_dict(m.dnn.state_dict()).numel() == eng.weights_numel()
    ts, _, rows = eng.sampler_schedule(N=m.sde.N, kind="sb_sde")
    assert ts.shape == (50,) and rows.shape == (50, 3) and abs(float(ts[-1]) - 1e-4) < 1e-9
    sgmse_b200.install(m, engine=eng)
    assert m.get_sb_sampler.__func__.__name__ == "get_sb_sampler" and "_sgmse_b200_engine" in m.__dict__
    sgmse_b200.uninstall(m)
    assert "get_sb_sampler" not in m.__dict__
    eng.close()


@live
def test_install_for_in_training_evaluation(model16k):
    """SURVEY.md §8f-3: with rebind_forward=False the differentiable torch forward stays in place (training steps), the
    samplers and enhance() go to the engine, and every model.eval() re-snapshots model.dnn (EMA swap, model.py:111-122)."""
    import sgmse_b200
    from sgmse_b200 import config_from_score_model, Engine
    eng = Engine(config_from_score_model(model16k))
    loads = []
    eng.load_blob = lambda blob: loads.append((blob.numel(), float(blob[0])))      # no GPU here: record instead of uploading
    sgmse_b200.install(model16k, engine=eng, rebind_forward=False, refresh_on_eval=True)
    try:
        assert "forward" not in model16k.__dict__ and "enhance" in model16k.__dict__ and "get_pc_sampler" in model16k.__dict__
        with torch.no_grad():
            model16k.dnn.output_layer.weight.view(-1)[0] = 0.25                      # "an optimiser step"
        model16k.eval()
        assert loads and loads[-1] == (eng.weights_numel(), 0.25)                    # output_layer.weight leads the blob
        model16k.train(True)                                                         # ScoreModel.train(mode, no_ema=False), model.py:98-109
        model16k.eval(no_ema=True)
        assert len(loads) == 2
        # Lightning + DDP never call ScoreModel.eval(): nn.Module.eval(wrapper) -> child.train(False) (ADVICE r1)
        model16k.train(True)
        torch.nn.Module.eval(torch.nn.Sequential(model16k))
        assert len(loads) == 3
    finally:
        sgmse_b200.uninstall(model16k)
        model16k.eval()
    assert "train" not in model16k.__dict__ and "eval" not in model16k.__dict__ and "enhance" not in model16k.__dict__
    eng.close()


def test_install_rebinds_the_ode_sampler(ref, recorded16k):
    """SURVEY.md §8f-4: install() routes ScoreModel.get_ode_sampler (model.py:370-390) to the engine for the OUVE SDE;
    the default call fails with the reference's own TypeError (denoise=True, predictors.py:60) before any GPU work, on
    the reference and on the engine alike."""
    import sgmse_b200
    from sgmse_b200 import config_from_score_model, Engine
    y = torch.zeros(1, 1, 256, 64, dtype=torch.complex64)
    assert "stepsize" in str(ref["ode_default_error"])                              # the unmodified reference
    eng = Engine(config_from_score_model(recorded16k))
    sgmse_b200.install(recorded16k, engine=eng)
    try:
        assert recorded16k.get_ode_sampler.__func__.__name__ == "get_ode_sampler" and "get_ode_sampler" in recorded16k.__dict__
        with pytest.raises(TypeError, match="stepsize"):
            recorded16k.get_ode_sampler(y)()
        with pytest.raises(RuntimeError, match="CUDA tensor"):                      # no CPU path behind the boundary
            recorded16k.get_ode_sampler(y, denoise=False, minibatch=1)()
    finally:
        sgmse_b200.uninstall(recorded16k)
    assert "get_ode_sampler" not in recorded16k.__dict__
    eng.close()


def test_ode_oracle_matches_reference_live(ref):
    """oracle/ode.py against the unmodified get_ode_sampler on a config the other fixtures do not hold (48 kHz SDE
    parameters, eps = 0.05, batch of 2 = one coupled ODE system)."""
    from oracle import ode as o_ode
    SMALL = dict(nf=16, ch_mult=(1, 2, 2), image_size=64, num_res_blocks=2)
    cfg = NetConfig.ncsnpp_48k(**SMALL)
    sd = o_w.make_state_dict(cfg, seed=5)
    g = torch.Generator().manual_seed(3)
    y = torch.complex(torch.randn(2, 1, 64, 64, generator=g), torch.randn(2, 1, 64, 64, generator=g)) * 0.3
    draws = o_sde.make_noise(tuple(y.shape), 1, seed=23)
    sde = o_sde.OUVE(theta=2.0, sigma_min=0.1, sigma_max=1.0)
    got, nfe = o_ode.ode_sample(lambda a, b, c: o_net.score(sd, cfg, a, b, c), y, sde, eps=0.05, rtol=1e-3, atol=1e-3,
                                prior_noise=draws[0])
    r = torch.from_numpy(ref["ode_x"])
    assert nfe == int(ref["ode_nfe"])
    assert ((r - got).abs().max() / r.abs().max()).item() < 1e-6


def test_staged_reference_is_unmodified():
    """oracle/_ref/ (what the GPU box and bench.py's reference arm import) is a byte-for-byte copy of /root/reference:
    every staged file matches its manifest hash, and where the live checkout is present, the live file."""
    import os
    from oracle import build_ref
    if not os.path.isdir("/root/reference/sgmse"):
        pytest.skip("live checkout not present")
    dst = build_ref.build()
    assert dst and build_ref.staged() and build_ref.verify() == []
    import json
    man = json.load(open(os.path.join(dst, "MANIFEST.json")))
    assert "sgmse/model.py" in man["files"] and "enhancement.py" in man["files"] and len(man["files"]) >= 25
    for rel in man["files"]:
        assert open(os.path.join(dst, rel), "rb").read() == open(os.path.join("/root/reference", rel), "rb").read(), rel
