"""The drop-in itself on hardware (SURVEY.md §8b, §8f-3): a live, UNMODIFIED reference ``ScoreModel`` (imported from the staged
copy ``oracle/_ref`` -- see oracle/build_ref.py -- or from /root/reference where that exists), ``sgmse_b200.install(model)``,
then the reference's own public calls: ``model.enhance(y)``, ``model.get_pc_sampler(...)()``, ``model(x_t, y, t)``
(/root/reference/sgmse/model.py:264-310,348-368,426-465), compared with the same model before installation, run on the CPU
with the same injected noise.  Second half: the in-training evaluation flow (model.py:205-257, util/inference.py:16-63):
``install(rebind_forward="no_grad", refresh_on_eval=True)``, weights change, the EMA swap of ``eval()`` -- reached the way
Lightning + DDP reach it, through ``nn.Module.eval(wrapper)`` -- and ``enhance`` must follow the swapped-in weights.

Run on the B200 box: ``pytest -m gpu``.  The tests that install on a live ScoreModel are skipped when neither /root/reference
nor oracle/_ref is present; the batched file service is compared with the reference's per-file loop as stored in
tests/golden/reference_live.npz and runs from the repository alone.
"""
import os

import numpy as np
import pytest
import torch

from oracle import refshim, sde as o_sde, pipeline as o_pipe

pytestmark = pytest.mark.gpu
live = pytest.mark.skipif(not refshim.reference_available(), reason="reference not staged (oracle/_ref) and no live checkout")

# mid-size config: 64..128 channels -> the tcgen05 convolutions run in fp16_tc mode (same as MID_E in test_gpu_parity.py)
MID = dict(nf=64, ch_mult=(1, 2, 2), image_size=64, attn_resolutions=(16,), num_res_blocks=1, n_fft=126, hop_length=32)
L, N = 4000, 3

# measured on a B200 (profiles/r02_parity.txt): fp32 sampler 1.6e-6 / waveform 1.5e-6 / forward 3.3e-6; fp16_tc 1.30e-3 /
# 1.08e-3 (SI-SDR 59.4 dB) / 2.66e-3; bounds = 2x measured
TOL = {"fp32": dict(spec=3.3e-6, wav=3e-6, fwd=6.7e-6), "fp16_tc": dict(spec=2.6e-3, wav=2.2e-3, fwd=5.4e-3)}


def rel_l2(a, b):
    a, b = torch.as_tensor(a).detach().cpu(), torch.as_tensor(b).detach().cpu()
    if a.is_complex():
        a, b = torch.view_as_real(a), torch.view_as_real(b)
    return (torch.linalg.vector_norm((a - b).reshape(-1)) / torch.linalg.vector_norm(b.reshape(-1))).item()


def make_model(seed=3):
    return refshim.make_score_model("ncsnpp", seed=seed, **MID)


def reference_run(model, wav, draws, n=N):
    """enhancement.py:68-99 on the CPU with the unmodified reference; returns (Y, sample, waveform)."""
    from sgmse.util.other import pad_spec
    T_orig = wav.size(1)
    norm = wav.abs().max()
    Y = torch.unsqueeze(model._forward_transform(model._stft(wav / norm)), 0)
    Y = pad_spec(Y, mode="zero_pad")
    with refshim.injected_noise(list(draws)):
        sample, nfe = model.get_pc_sampler("reverse_diffusion", "ald", Y, N=n, corrector_steps=1, snr=0.5)()
    x_hat = model.to_audio(sample.squeeze(), T_orig) * norm
    return Y, sample, x_hat.squeeze().numpy(), nfe


@live
@pytest.mark.parametrize("mode", ["fp32", "fp16_tc"])
def test_install_on_a_live_reference_score_model(mode):
    import sgmse_b200
    model = make_model()
    g = torch.Generator().manual_seed(5)
    wav = 0.1 * torch.randn(1, L, generator=g)
    Tp = 128                                                   # 126 frames -> padded to 128
    draws = o_sde.make_noise((1, 1, 64, Tp), o_sde.n_noise_draws(N, "reverse_diffusion", "ald", 1), seed=17)
    Y, ref_sample, ref_wav, ref_nfe = reference_run(model, wav, draws)
    assert tuple(Y.shape) == (1, 1, 64, Tp)
    x_t = Y + 0.3 * draws[0]
    t = torch.tensor([0.6])
    with torch.no_grad():
        ref_score = model(x_t, Y, t)                           # ScoreModel.forward, legacy branch (model.py:307-310)

    eng = sgmse_b200.install(model, mode=mode, max_batch=2)
    try:
        noise = torch.stack(draws).cuda()
        sample, nfe = model.get_pc_sampler("reverse_diffusion", "ald", Y.cuda(), N=N, corrector_steps=1, snr=0.5, noise=noise)()
        assert nfe == ref_nfe == 2 * N and sample.is_cuda and sample.dtype == torch.complex64 and sample.shape == ref_sample.shape
        e_spec = rel_l2(sample, ref_sample)
        x_hat = model.enhance(wav, N=N, noise=noise)           # the reference's one-call API (model.py:426-465), rebound
        assert isinstance(x_hat, np.ndarray) and x_hat.shape == (L,) and x_hat.dtype == np.float32
        e_wav = rel_l2(x_hat, ref_wav)
        sdr = o_pipe.si_sdr(ref_wav, x_hat)
        with torch.no_grad():
            e_fwd = rel_l2(model(x_t.cuda(), Y.cuda(), t.cuda()), ref_score)
        if mode == "fp16_tc":
            assert eng.counter("tc_convs_last_forward") > 0, "tcgen05 path not taken"
        print(f"drop-in {mode}: sampler rel-L2 {e_spec:.3e}, waveform rel-L2 {e_wav:.3e}, SI-SDR(ref, engine) {sdr:.1f} dB, "
              f"forward rel-L2 {e_fwd:.3e}")
        tol = TOL[mode]
        assert e_spec < tol["spec"] and e_wav < tol["wav"] and e_fwd < tol["fwd"]
        # timeit variant: (x_hat, nfe, rtf) as model.py:460-463; Philox noise path: finite and seed-reproducible
        a, nfe_t, rtf = model.enhance(wav, N=N, timeit=True, seed=9)
        b = model.enhance(wav, N=N, seed=9)
        assert nfe_t == 2 * N and rtf > 0 and np.isfinite(a).all() and np.array_equal(a, b)
        # minibatch loop of get_pc_sampler (model.py:354-368): list of nfe, same samples
        Y2 = torch.cat([Y, Y], 0).cuda()
        n2 = torch.cat([noise, noise], 1)
        s2, ns = model.get_pc_sampler("reverse_diffusion", "ald", Y2, N=N, minibatch=1, corrector_steps=1, snr=0.5, noise=n2)()
        assert ns == [2 * N, 2 * N] and torch.equal(s2[0], sample[0]) and torch.equal(s2[1], sample[0])
    finally:
        sgmse_b200.uninstall(model)
        eng.close()
    # uninstalled: the reference's own torch path is back, bit-for-bit
    _, again, _, _ = reference_run(model, wav, draws)
    assert torch.equal(again, ref_sample)


class TinyEMA:
    """A working stand-in for torch_ema.ExponentialMovingAverage (store / copy_to / restore are what ScoreModel.train()
    uses, model.py:111-122); refshim's stub is inert, this one really swaps weights."""

    def __init__(self, params, seed):
        g = torch.Generator().manual_seed(seed)
        self.shadow = [p.detach().clone() * 0.95 + 0.02 * torch.randn(p.shape, generator=g) * p.detach().abs().mean() for p in params]
        self.collected_params = None

    def store(self, params):
        self.collected_params = [p.detach().clone() for p in params]

    def copy_to(self, params):
        for s, p in zip(self.shadow, params):
            p.data.copy_(s)

    def restore(self, params):
        for c, p in zip(self.collected_params, params):
            p.data.copy_(c)
        self.collected_params = None

    def to(self, *a, **k):
        pass


@live
def test_in_training_evaluation_follows_the_ema_swap():
    """validation_step (model.py:205-257) calls self.enhance per file with whatever weights eval() swapped into self.dnn;
    evaluate_model (util/inference.py:47-50) calls model.get_pc_sampler the same way.  The engine must see the EMA
    weights after every swap, also when the swap is reached through the DDP wrapper's nn.Module.eval()."""
    import sgmse_b200
    model = make_model(seed=4)
    model.train(True)
    model.ema = TinyEMA(list(model.dnn.parameters()), seed=1)
    g = torch.Generator().manual_seed(6)
    wav = 0.1 * torch.randn(1, L, generator=g)
    draws = o_sde.make_noise((1, 1, 64, 128), o_sde.n_noise_draws(N, "reverse_diffusion", "ald", 1), seed=19)
    noise = torch.stack(draws)

    # what the reference computes: training weights W (no_ema) and EMA weights S
    model.eval(no_ema=True)
    _, _, ref_W, _ = reference_run(model, wav, draws)
    model.train(True)
    model.eval()
    Y, _, ref_S, _ = reference_run(model, wav, draws)
    x_t, t = Y + 0.2 * draws[1], torch.tensor([0.4])
    with torch.no_grad():
        ref_fwd_S = model(x_t, Y, t)
    model.train(True)
    assert rel_l2(ref_S, ref_W) > 1e-2                          # the swap matters for the output

    eng = sgmse_b200.install(model, mode="fp32", max_batch=2, rebind_forward="no_grad", refresh_on_eval=True)
    try:
        noise_d = noise.cuda()
        got_W = model.enhance(wav, N=N, noise=noise_d)          # installed in train mode: the training weights
        assert rel_l2(got_W, ref_W) < 1e-5
        wrapper = torch.nn.Sequential(model)                    # stands for DistributedDataParallel(model) (train.py:104)
        torch.nn.Module.eval(wrapper)                           # Lightning: on_validation_model_eval -> trainer.model.eval()
        got_S = model.enhance(wav, N=model.sde.N if False else N, noise=noise_d)
        e = rel_l2(got_S, ref_S)
        print(f"in-training evaluation: after the EMA swap rel-L2 {e:.3e} vs the reference on the swapped weights "
              f"({rel_l2(got_S, ref_W):.3e} vs the training weights)")
        assert e < 3e-6 and rel_l2(got_S, ref_W) > 5e-3                # measured 1.44e-6
        # the validation loss route: _step -> self(x_t, y, t) under torch.no_grad() goes to the engine (EMA weights) ...
        with torch.no_grad():
            out = model(x_t.cuda(), Y.cuda(), t.cuda())
        assert out.is_cuda and rel_l2(out, ref_fwd_S) < 1e-5
        # ... while a forward with autograd stays on the torch modules (CPU tensors in, autograd graph out)
        out_t = model(x_t, Y, t)
        assert out_t.requires_grad and not out_t.is_cuda
        # back to training (EMA restore), an "optimizer step", next validation epoch: the engine follows again
        wrapper.train()
        with torch.no_grad():
            for p in model.dnn.parameters():
                p.mul_(1.01)
        model.ema.shadow = [s * 0.9 for s in model.ema.shadow]
        torch.nn.Module.eval(wrapper)
        got_S2 = model.enhance(wav, N=N, noise=noise_d)
        sgmse_b200.uninstall(model)
        _, _, ref_S2, _ = reference_run(model, wav, draws)      # model is still in eval(): dnn holds the new EMA weights
        assert rel_l2(got_S2, ref_S2) < 1e-5 and rel_l2(got_S2, ref_S) > 5e-3
    finally:
        sgmse_b200.uninstall(model)
        eng.close()


def test_batched_file_service_against_the_reference_file_loop(golden_dir):
    """SURVEY.md §8f-2 against the REFERENCE (not against the engine itself): clips of three different lengths -- two padded
    frame counts, so two buckets -- through the unmodified reference's per-file loop (enhancement.py:58-99 on the CPU, injected
    noise; stored by oracle/make_golden.py: golden_reference_live, weights = oracle init seed 7) and through BatchedEnhancer
    with the same weights and per-clip noise; every clip individually, in both engine modes."""
    from oracle import weights as o_w
    from oracle.arch import NetConfig
    from sgmse_b200 import BatchedEnhancer, Engine, EngineConfig
    gold = np.load(os.path.join(golden_dir, "reference_live.npz"))
    net = {k: v for k, v in MID.items() if k not in ("n_fft", "hop_length")}
    sd = o_w.make_state_dict(NetConfig.ncsnpp(**net), seed=7)
    g = torch.Generator().manual_seed(8)
    lengths = [4000, 1900, 3100, 2000]                      # 126, 60, 97, 63 frames -> padded to 128, 64, 128, 64
    clips = [0.1 * torch.randn(n, generator=g) * (1.0 + 0.5 * i) for i, n in enumerate(lengths)]
    nd = o_sde.n_noise_draws(N, "reverse_diffusion", "ald", 1)
    draws = {i: o_sde.make_noise((1, 1, 64, 128 if lengths[i] > 2048 else 64), nd, seed=40 + i) for i in range(len(clips))}
    refs = [gold[f"files_enh{i}"] for i in range(len(clips))]
    for mode, tol in (("fp32", 1e-5), ("fp16_tc", 2.2e-3)):
        eng = Engine(EngineConfig(**MID, mode=mode, max_batch=2))
        eng.load_state_dict(sd)
        outs, ids = BatchedEnhancer(eng)(clips, seed=0, N=N, predictor="reverse_diffusion", corrector="ald", corrector_steps=1, snr=0.5,
                                         noise_for=lambda i, tp: torch.stack(draws[i]))
        errs = [rel_l2(o, r) for o, r in zip(outs, refs)]
        print(f"batched file service vs the reference file loop, {mode}: per-clip waveform rel-L2 " + ", ".join(f"{e:.2e}" for e in errs))
        assert all(o.shape[0] == n for o, n in zip(outs, lengths)) and sorted(ids) == [0, 1, 2, 3]
        assert max(errs) < tol
        eng.close()
