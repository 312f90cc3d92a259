"""yume_b200/sampler.py against the reference's own code, on CPU: the sigma schedule is compared with what `get_sampling_sigmas`,
EXTRACTED from fastvideo/sample/sample_5b.py, returned (tests/golden/sampling_sigmas.json, tools/make_golden_install.py), the SDE update
with the statements of sample_tts.py:726-744 restated verbatim, and the Euler / CFG loops with an explicit unrolled restatement of
sample_5b.py:941-1034 and sample.py:755-790 over a toy `transformer`."""
import json
import math

import torch

from yume_b200 import sampler


def test_sigma_schedule_equals_the_reference_function(golden_dir):
    for case in json.loads((golden_dir / "sampling_sigmas.json").read_text()):
        steps, shift, want = case["steps"], case["shift"], case["sigmas"]
        got = sampler.sampling_sigmas(steps, shift)
        assert len(got) == len(want) == steps and max(abs(a - float(b)) for a, b in zip(got, want)) < 1e-12


def test_sde_update_equals_the_reference_statements():
    g = torch.Generator().manual_seed(0)
    latent_new, noise_pred = torch.randn(4, 2, 3, 5, generator=g), torch.randn(4, 2, 3, 5, generator=g)
    for sigma, sigma_next, last in ((0.9, 0.7, False), (0.3, 0.0, True), (0.5, 0.6, False)):
        temp_x0 = latent_new + ((0.0 if last else sigma_next) - sigma) * noise_pred
        # sample_tts.py:726-744, names kept
        eta = 0.3
        pred_original_sample = latent_new + (0 - sigma) * noise_pred
        delta_t = 0 if last else (sigma - sigma_next)
        if delta_t < 0:
            delta_t = 0
        dsigma = (0 - sigma) if last else (sigma_next - sigma)
        std_dev_t = eta * math.sqrt(delta_t)
        score_estimate = -(latent_new - pred_original_sample * (1 - sigma)) / sigma ** 2
        prev_sample_mean = temp_x0 + (-0.5 * eta ** 2 * score_estimate) * dsigma
        noise = torch.randn(prev_sample_mean.shape, generator=torch.Generator().manual_seed(5))
        want = prev_sample_mean + noise * std_dev_t
        got = sampler.sde_update(latent_new, noise_pred, temp_x0, sigma, sigma_next, last, 0.3, torch.Generator().manual_seed(5))
        assert torch.allclose(got, want, rtol=0, atol=1e-6)


def _toy(scale):
    """A deterministic stand-in for WanModel.forward with the reference's call shapes (5B returns a list, 14B a tuple)."""
    def f5(x, t, latent_frame_zero=8, context=None, seq_len=0):
        return [torch.tanh(x[0] * scale + t.float().mean() * 1e-3 + context[0].float().mean())]

    def f14(x, t, rand_num_img=None, latent_frame_zero=8, context=None, **_):
        return torch.tanh(x[0] * scale - t.float().mean() * 1e-3 + context[0].float().mean()), None
    return f5, f14


def test_5b_loop_equals_the_unrolled_reference_loop():
    f5, _ = _toy(0.7)
    g = torch.Generator().manual_seed(1)
    hist, noise = torch.randn(6, 5, 4, 4, generator=g), torch.randn(6, 2, 4, 4, generator=g)
    ctx = torch.randn(3, 8, generator=g)
    lfz, steps, shift = 2, 4, 7.0
    got = sampler.denoise_chunk_5b(f5, torch.cat([hist, noise], 1), hist, lfz, steps, dict(context=[ctx], seq_len=0), shift=shift)
    # sample_5b.py:941-1034 (i2v branch), unrolled: per-token t = [0 for history, sigma*1000 for new]; Euler; history re-attached
    sig = sampler.sampling_sigmas(steps, shift)
    latent = torch.cat([hist, noise], 1)
    for i in range(steps):
        pred = f5([latent], torch.tensor([[0.0, sig[i] * 1000.0]]), latent_frame_zero=lfz, context=[ctx], seq_len=0)[0][:, -lfz:]
        step = (0 - sig[i]) if i + 1 == steps else (sig[i + 1] - sig[i])
        latent = torch.cat([hist, latent[:, -lfz:] + step * pred], dim=1)
    assert torch.equal(got, latent)


def test_14b_cfg_loop_equals_the_unrolled_reference_loop():
    _, f14 = _toy(0.4)
    g = torch.Generator().manual_seed(2)
    noise, model_input = torch.randn(4, 7, 4, 4, generator=g), torch.randn(4, 7, 4, 4, generator=g)
    ctx_c, ctx_n = torch.randn(3, 8, generator=g), torch.randn(3, 8, generator=g)
    lfz, steps, shift, cfg = 2, 6, 3.0, 5.0
    got = sampler.denoise_chunk_14b(f14, noise, model_input, lfz, steps, dict(context=[ctx_c]), dict(context=[ctx_n]), rand_num_img=0.6,
                                    shift=shift, guidance=cfg)
    sliced = sampler.denoise_chunk_14b(f14, noise, model_input, lfz, steps, dict(context=[ctx_c]), dict(context=[ctx_n]), rand_num_img=0.6,
                                       shift=shift, guidance=cfg, first_steps=2)
    # sample.py:755-790, unrolled: cond + uncond at the same latent / t, guidance, Euler on the new frames, history re-noised to the next sigma
    sig = sampler.sampling_sigmas(steps, shift)
    latent, after2 = noise, None
    for i in range(steps):
        t = torch.tensor([sig[i] * 1000.0])
        cond, _ = f14([latent], t, rand_num_img=0.6, latent_frame_zero=lfz, context=[ctx_c])
        uncond, _ = f14([latent], t, rand_num_img=0.6, latent_frame_zero=lfz, context=[ctx_n])
        pred = (uncond + cfg * (cond - uncond))[:, -lfz:]
        step = (0 - sig[i]) if i + 1 == steps else (sig[i + 1] - sig[i])
        x0 = latent[:, -lfz:] + step * pred
        s1 = sig[min(steps - 1, i + 1)]
        latent = torch.cat([noise[:, :-lfz] * s1 + (1 - s1) * model_input[:, :-lfz], x0], dim=1)
        if i == 1:
            after2 = latent
    assert torch.equal(got, latent) and torch.equal(sliced, after2)
