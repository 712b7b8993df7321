"""The product's host loops against the REFERENCE's loops over a full 50-step schedule, on a CPU double of the engine.

`DirectInversion.invert` (ddim_loop + offset_calculate, models/p2p/inversion.py:308-319,375-403) and
`direct_inversion_p2p_guidance_forward` (models/p2p/p2p_guidance_forward.py:103-116,135-173) of the reference run unmodified
(oracle/ref_shim.py) on a cheap fake UNet; the product's `pnpinversion_b200/inversion.py` and `p2p_guidance_forward.py` run
on the same fake UNet with `fused_step` replaced by tests/cpu_engine_double.cpu_fused_step.  What this pins is everything
the GPU fixtures cannot cover at 4 steps: the index arithmetic of all 50 + 50 + 50 steps (which latent is the target of
which offset step, which noise_loss rectifies which step, the timestep order in both directions).
The reference's results are recorded in tests/golden/reference_host_loops.npz (tests/reference_golden.py; re-record
with PNP_RECORD_REFERENCE=1 where the reference tree is available)."""
import types

import torch

from oracle import ref_shim
from pnpinversion_b200 import synth
from tests.cpu_engine_double import FakeUNet, cpu_fused_step
from tests.reference_golden import recorded_fixture

golden = recorded_fixture("host_loops")


class _Vae:  # image2latent passes 4-D tensors through (utils/utils.py:73-74); decode only feeds the unused image_rec
    def decode(self, z):
        return {"sample": torch.zeros(z.shape[0], 3, 8, 8, dtype=z.dtype)}


def _calls(model):
    """the fake UNet's call log (batch shape, timestep) as rows of integers"""
    return [list(shape) + [t] for shape, t in model.unet.calls]


def _models(recording):
    """(reference model or None when replaying, product model) on the fake UNet"""
    from pnpinversion_b200.scheduler import DDIMSchedulerDev

    tok = synth.FakeTokenizer()
    common = dict(tokenizer=tok, text_encoder=synth.SynthTextEncoder(), device=torch.device("cpu"))
    ref_model = None
    if recording:
        md = ref_shim.load_my_diffusers()
        ref_sched = md.DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                                     clip_sample=False, set_alpha_to_one=False)
        ref_sched.set_timesteps(50)
        ref_model = types.SimpleNamespace(unet=FakeUNet(), scheduler=ref_sched, vae=_Vae(), **common)
    my_sched = DDIMSchedulerDev(engine=None, table_dtype="float64")  # the vendored scheduler's table is float64
    my_sched.set_timesteps(50)
    my_model = types.SimpleNamespace(unet=FakeUNet(), scheduler=my_sched, vae=None, **common)
    return ref_model, my_model


def test_inversion_offset_and_rectified_forward_loops_follow_the_reference_for_50_steps(monkeypatch, golden):
    from pnpinversion_b200 import inversion as my_inv
    from pnpinversion_b200 import p2p_guidance_forward as my_fwd
    from pnpinversion_b200 import scheduler as my_sched_mod
    from pnpinversion_b200.attention_control import EmptyControl

    for mod in (my_inv, my_fwd, my_sched_mod):
        monkeypatch.setattr(mod, "fused_step", cpu_fused_step)
    ref = ref_shim.load_reference_p2p() if golden.recording else None
    ref_model, my_model = _models(golden.recording)
    prompts = list(synth.CAT_PROMPTS)
    z = synth.synth_latent(3)
    torch.set_grad_enabled(False)

    if golden.recording:
        _, _, xs_r, nl_r = ref.inversion.DirectInversion(model=ref_model, num_ddim_steps=50).invert(
            image_gt=z, prompt=prompts, guidance_scale=7.5)
    _, _, xs_m, nl_m = my_inv.DirectInversion(model=my_model, num_ddim_steps=50).invert(
        image_gt=z, prompt=prompts, guidance_scale=7.5)
    calls_r = golden.value("invert/calls", lambda: _calls(ref_model)).tolist()
    assert calls_r == _calls(my_model)  # same batch shapes and timesteps, in the same order
    assert len(calls_r) == 100 and calls_r[0] == [1, 4, 64, 64, 0] and calls_r[50] == [4, 4, 64, 64, 980]
    assert golden.value("invert/lens", lambda: [len(xs_r), len(nl_r)]).tolist() == [len(xs_m), len(nl_m)] == [51, 50]
    for i, b in enumerate(xs_m):
        assert golden.equal(f"invert/x_star/{i}", b, lambda: xs_r[i])  # inverse steps: bit for bit
    for i, b in enumerate(nl_m):
        assert golden.close(f"invert/noise_loss/{i}", b, lambda: nl_r[i], atol=2e-6), i

    # the forward pass starts from the inverted latent (bit-identical in both, asserted above); each side is rectified
    # with its own noise_loss list (equal within 2e-6, asserted above)
    x_t = xs_m[-1]
    if golden.recording:
        lat_r, _ = ref.p2p_guidance_forward.direct_inversion_p2p_guidance_forward(
            model=ref_model, prompt=prompts, controller=ref.attention_control.EmptyControl(), latent=xs_r[-1],
            noise_loss_list=nl_r, num_inference_steps=50, guidance_scale=7.5, generator=None)
    lat_m, _ = my_fwd.direct_inversion_p2p_guidance_forward(
        model=my_model, prompt=prompts, controller=EmptyControl(), latent=x_t, noise_loss_list=nl_m,
        num_inference_steps=50, guidance_scale=7.5, generator=None)
    assert golden.value("forward/calls", lambda: _calls(ref_model)).tolist() == _calls(my_model)
    assert len(my_model.unet.calls) == 150
    assert golden.close("forward/latents", lat_m, lambda: lat_r, atol=5e-5, k=64)
    # the invariant of the method: the rectified source branch lands on the inverted image
    assert float((lat_m[0] - xs_m[0][0]).abs().max()) < 1e-4
    assert golden.value("forward/source_vs_inverted",
                        lambda: float((lat_r[0] - xs_r[0][0]).abs().max())) < 1e-4


def test_plain_p2p_forward_and_add_target_ablation_follow_the_reference(monkeypatch, golden):
    """`p2p_guidance_forward` (:21-62, the ddim+p2p baseline: no rectification) and
    `direct_inversion_p2p_guidance_forward_add_target` (:119-132,175-213: both branches rectified)."""
    from pnpinversion_b200 import p2p_guidance_forward as my_fwd
    from pnpinversion_b200 import scheduler as my_sched_mod
    from pnpinversion_b200.attention_control import EmptyControl

    for mod in (my_fwd, my_sched_mod):
        monkeypatch.setattr(mod, "fused_step", cpu_fused_step)
    ref = ref_shim.load_reference_p2p() if golden.recording else None
    ref_model, my_model = _models(golden.recording)
    prompts = list(synth.CAT_PROMPTS)
    torch.set_grad_enabled(False)
    g = torch.Generator().manual_seed(21)
    x_t = torch.randn(1, 4, 64, 64, generator=g)
    nl = [torch.randn(2, 4, 64, 64, generator=g) * 0.01 for _ in range(50)]

    b, _ = my_fwd.p2p_guidance_forward(model=my_model, prompt=prompts, controller=EmptyControl(), latent=x_t,
                                       num_inference_steps=50, guidance_scale=7.5, generator=None)
    assert golden.close("plain/latents", b, lambda: ref.p2p_guidance_forward.p2p_guidance_forward(
        model=ref_model, prompt=prompts, controller=ref.attention_control.EmptyControl(), latent=x_t,
        num_inference_steps=50, guidance_scale=7.5, generator=None)[0], atol=5e-5, k=64)
    assert golden.value("plain/calls", lambda: _calls(ref_model)).tolist() == _calls(my_model)
    assert len(my_model.unet.calls) == 50

    b, _ = my_fwd.direct_inversion_p2p_guidance_forward_add_target(
        model=my_model, prompt=prompts, controller=EmptyControl(), latent=x_t, noise_loss_list=nl,
        num_inference_steps=50, guidance_scale=7.5, generator=None)
    assert golden.close("add_target/latents", b, lambda: ref.p2p_guidance_forward.direct_inversion_p2p_guidance_forward_add_target(
        model=ref_model, prompt=prompts, controller=ref.attention_control.EmptyControl(), latent=x_t, noise_loss_list=nl,
        num_inference_steps=50, guidance_scale=7.5, generator=None)[0], atol=5e-5, k=64)
    assert golden.value("add_target/calls", lambda: _calls(ref_model)).tolist() == _calls(my_model)
    assert len(my_model.unet.calls) == 100


def test_edict_coupled_loop_follows_the_reference_for_40_plus_40_steps(monkeypatch, golden):
    """`pnpinversion_b200.edict.coupled_stablediffusion` against the reference's own `coupled_stablediffusion`
    (edict_functions.py:707-956, compiled from its source by oracle/ref_shim.load_reference_edict) on the fake UNet:
    deterministic noising over 40 of 50 steps (init_image_strength 0.8), then generation from that pair with a
    prompt_edit.  Checks the timestep order in both directions, the leapfrog alternation, the mixing layers, the step
    algebra and which prediction plays 'cond' under Prompt-to-Prompt.  The reference computes in fp64, the product loop in
    fp32, and the un-mixing layers amplify rounding by (1/0.93^2) per step: hence the tolerances."""
    from pnpinversion_b200 import edict as my_edict
    from pnpinversion_b200 import scheduler as my_sched_mod
    from pnpinversion_b200.scheduler import DDIMSchedulerDev
    from tests.cpu_engine_double import FakeLib

    monkeypatch.setattr(my_edict, "fused_step", cpu_fused_step)
    monkeypatch.setattr(my_sched_mod, "fused_step", cpu_fused_step)
    monkeypatch.setattr(my_edict._lib, "load", lambda: FakeLib())
    monkeypatch.setattr(my_edict._lib, "current_stream_ptr", lambda: 0)
    torch.set_grad_enabled(False)
    tok, te = synth.FakeTokenizer(), synth.SynthTextEncoder(dtype=torch.float64)
    src, tgt = synth.CAT_PROMPTS

    class Tok:
        model_max_length = tok.model_max_length

        def __call__(self, text, padding="max_length", max_length=77, truncation=True, return_tensors="pt",
                     return_overflowing_tokens=True):
            return tok(text, padding=padding, max_length=max_length, truncation=truncation, return_tensors=return_tensors)

    class Clip:
        def __call__(self, ids):
            return types.SimpleNamespace(last_hidden_state=te(ids)[0])

    class RefUNet(FakeUNet):
        def named_modules(self):
            return []

        def __call__(self, x, t, encoder_hidden_states=None):
            out = super().__call__(x, t, encoder_hidden_states)["sample"].to(x.dtype)
            return types.SimpleNamespace(sample=out)

    ref_unet = RefUNet()
    z = synth.synth_latent(4)
    kw = dict(init_image_strength=0.8, steps=50, mix_weight=0.93, guidance_scale=3.0)
    if golden.recording:
        ns = ref_shim.load_reference_edict(ref_unet, Clip(), Tok(), "cpu")
        lat_r = ns["coupled_stablediffusion"](src, reverse=True, init_image=[z.double(), z.double().clone()], **kw)
        out_r = ns["coupled_stablediffusion"](src, tgt, fixed_starting_latent=lat_r, return_latents=True, **kw)

    my_sched = DDIMSchedulerDev(engine=None, table_dtype="float64")
    my_model = types.SimpleNamespace(unet=FakeUNet(), scheduler=my_sched, vae=None, tokenizer=tok,
                                     text_encoder=synth.SynthTextEncoder(), device=torch.device("cpu"))
    lat_m = my_edict.coupled_stablediffusion(my_model, src, reverse=True, init_image=[z, z.clone()], **kw)
    out_m = my_edict.coupled_stablediffusion(my_model, src, tgt, fixed_starting_latent=lat_m, **kw)

    # the reference makes 2 (3 with prompt_edit) single-row calls per sub-step, the product one batched call
    t_ref = golden.value("edict/timesteps", lambda: [t for _, t in ref_unet.calls]).tolist()
    t_mine = [t for _, t in my_model.unet.calls]
    assert t_ref[0:160:2] == t_mine[0:80] and t_ref[160::3] == t_mine[80:]
    assert t_mine[0] == 0 and t_mine[79] == 780 and t_mine[80] == 780 and t_mine[-1] == 0  # t = 0 .. 780 up, then down
    assert my_model.unet.calls[0][0] == (2, 4, 64, 64) and my_model.unet.calls[-1][0] == (3, 4, 64, 64)

    for i in range(2):  # relative L2 distance on a fixed sample of 256 of the 16384 elements
        e_lat = golden.rel(f"edict/noised/{i}", lat_m[i], lambda: lat_r[i])
        e_out = golden.rel(f"edict/edited/{i}", out_m[i], lambda: out_r[i])
        assert e_lat < 2e-3 and e_out < 2e-3, (i, e_lat, e_out)


def test_inversion_variants_follow_the_reference(monkeypatch, golden):
    """The guidance / ablation family of `models/p2p/inversion.py::DirectInversion`: CFG inversion
    (`invert_with_guidance_scale_vary_guidance` :412-419 - the reference's two B=1 calls per step are the two rows of one
    B=2 call here), the scaled offset (`invert_not_full` :478-499), the skipped offset (`invert_skip_step` :501-526), and
    `NegativePromptInversion.invert` (:78-101, with and without the slerp interpolation) - over 50 steps on the fake UNet."""
    from pnpinversion_b200 import inversion as my_inv
    from pnpinversion_b200 import scheduler as my_sched_mod

    for mod in (my_inv, my_sched_mod):
        monkeypatch.setattr(mod, "fused_step", cpu_fused_step)
    ref = ref_shim.load_reference_p2p() if golden.recording else None
    prompts = list(synth.CAT_PROMPTS)
    z = synth.synth_latent(5)
    torch.set_grad_enabled(False)

    def both(call_ref, call_mine):
        ref_model, my_model = _models(golden.recording)
        r = call_ref(ref.inversion.DirectInversion(model=ref_model, num_ddim_steps=50)) if golden.recording else None
        m = call_mine(my_inv.DirectInversion(model=my_model, num_ddim_steps=50))
        return r, m, ref_model, my_model

    # CFG inversion at 2.5, offsets at 7.5
    r, m, rm, mm = both(lambda inv: inv.invert_with_guidance_scale_vary_guidance(z, prompts, 2.5, 7.5),
                        lambda inv: inv.invert_with_guidance_scale_vary_guidance(z, prompts, 2.5, 7.5))
    t_ref = golden.value("cfg/timesteps", lambda: [t for _, t in rm.unet.calls]).tolist()
    t_mine = [t for _, t in mm.unet.calls]
    assert t_ref[0:100:2] == t_mine[:50] and t_ref[100:] == t_mine[50:]  # 2 x B=1 calls per step there, 1 x B=2 here
    assert mm.unet.calls[0][0] == (2, 4, 64, 64)
    assert golden.value("cfg/lens", lambda: [len(r[2]), len(r[3])]).tolist() == [len(m[2]), len(m[3])]
    for i, b in enumerate(m[2]):
        assert golden.close(f"cfg/x_star/{i}", b, lambda: r[2][i], atol=2e-5), i
    for i, b in enumerate(m[3]):
        assert golden.close(f"cfg/noise_loss/{i}", b, lambda: r[3][i], atol=5e-5), i

    # loss * 0.8 and loss on every 5th step only
    for kw_name, kw in (("invert_not_full", dict(scale=0.8)), ("invert_skip_step", dict(skip_step=5))):
        r, m, rm, mm = both(lambda inv: getattr(inv, kw_name)(image_gt=z, prompt=prompts, guidance_scale=7.5, **kw),
                            lambda inv: getattr(inv, kw_name)(image_gt=z, prompt=prompts, guidance_scale=7.5, **kw))
        assert golden.value(f"{kw_name}/calls", lambda: _calls(rm)).tolist() == _calls(mm)
        assert golden.value(f"{kw_name}/len", lambda: len(r[3])) == len(m[3])
        for i, b in enumerate(m[3]):
            assert golden.close(f"{kw_name}/noise_loss/{i}", b, lambda: r[3][i], atol=5e-6), (kw_name, i)
        if kw_name == "invert_skip_step":
            assert float(m[3][1].abs().max()) == 0.0 and float(m[3][5].abs().max()) > 0.0

    # negative-prompt inversion
    for interp in (0.0, 0.3):
        ref_model, my_model = _models(golden.recording)
        if golden.recording:
            ri = ref.inversion.NegativePromptInversion(model=ref_model, num_ddim_steps=50).invert(z, prompts[0],
                                                                                                 npi_interp=interp)
        mi = my_inv.NegativePromptInversion(model=my_model, num_ddim_steps=50).invert(z, prompts[0], npi_interp=interp)
        assert golden.value(f"npi_{interp}/calls", lambda: _calls(ref_model)).tolist() == _calls(my_model)
        assert len(my_model.unet.calls) == 50
        assert golden.value(f"npi_{interp}/lens", lambda: [len(ri[2]), len(ri[3])]).tolist() == [len(mi[2]), len(mi[3])]
        for i, b in enumerate(mi[2]):
            assert golden.equal(f"npi_{interp}/x_star/{i}", b, lambda: ri[2][i])
        dtype = golden.value(f"npi_{interp}/noise_loss_dtype", lambda: str(ri[3][0].dtype).split(".")[-1]).item()
        assert len(mi[3]) == 50 and golden.close(f"npi_{interp}/noise_loss/0", mi[3][0].to(getattr(torch, dtype)),
                                                 lambda: ri[3][0], atol=1e-6)


def test_schedule_with_a_step_count_that_does_not_divide_1000(monkeypatch):
    """30 steps: diffusers 0.10's `(arange(0, n) * (1000 // n)).round()[::-1]` gives 30 timesteps from 957 (the vendored
    0.3.0 scheduler would give 31 from 990); inversion, offsets and the rectified forward pass run over exactly 30 steps
    and the source branch still lands on the inverted latent."""
    from pnpinversion_b200 import inversion as my_inv
    from pnpinversion_b200 import p2p_guidance_forward as my_fwd
    from pnpinversion_b200 import scheduler as my_sched_mod
    from pnpinversion_b200.attention_control import EmptyControl

    for mod in (my_inv, my_fwd, my_sched_mod):
        monkeypatch.setattr(mod, "fused_step", cpu_fused_step)
    _, my_model = _models(recording=False)
    my_model.scheduler.set_timesteps(30)
    assert my_model.scheduler.timesteps.tolist() == [33 * i for i in range(29, -1, -1)]
    prompts = list(synth.CAT_PROMPTS)
    z = synth.synth_latent(2)
    torch.set_grad_enabled(False)
    _, _, xs, nl = my_inv.DirectInversion(model=my_model, num_ddim_steps=30).invert(image_gt=z, prompt=prompts,
                                                                                   guidance_scale=7.5)
    assert len(xs) == 31 and len(nl) == 30
    lat, _ = my_fwd.direct_inversion_p2p_guidance_forward(model=my_model, prompt=prompts, controller=EmptyControl(),
                                                          latent=xs[-1], noise_loss_list=nl, num_inference_steps=30,
                                                          guidance_scale=7.5, generator=None)
    assert [t for _, t in my_model.unet.calls[:30]] == [33 * i for i in range(30)]
    assert float((lat[0] - xs[0][0]).abs().max()) < 1e-4


def test_proximal_guidance_forward_follows_the_reference(monkeypatch, golden):
    """`proximal_guidance_forward` (models/p2p/proximal_guidance_forward.py:20-170) as the negative-prompt-inversion
    methods call it (p2p_editor.py:350-410): reconstruction pass (prox None), edit pass with prox 'l0' / 'l1', with and
    without the reconstruction guidance on the predicted x0 (scheduler_dev.py:61-70)."""
    from pnpinversion_b200 import p2p_guidance_forward as my_fwd
    from pnpinversion_b200 import scheduler as my_sched_mod
    from pnpinversion_b200.attention_control import EmptyControl

    for mod in (my_fwd, my_sched_mod):
        monkeypatch.setattr(mod, "fused_step", cpu_fused_step)
    import importlib
    import sys
    # models/p2p/scheduler_dev.py subclasses `diffusers.DDIMScheduler` (0.10, absent here).  The harness offers it the
    # vendored 0.3.0 scheduler under that name, with the one config field step() reads that 0.3.0 lacks; the
    # reference's DDIMSchedulerDev.step (:10-121) itself runs unmodified.
    if golden.recording:
        ref = ref_shim.load_reference_p2p()
        ref_prox = importlib.import_module("models.p2p.proximal_guidance_forward")
        md = ref_shim.load_my_diffusers()

        class _Sched(md.DDIMScheduler):
            @property
            def config(self):
                return types.SimpleNamespace(**dict(super().config), prediction_type="epsilon")

        class _Out(dict):
            def __init__(self, **kw):
                super().__init__(**kw)
                self.__dict__.update(kw)

    if golden.recording and "diffusers" not in sys.modules:
        d = types.ModuleType("diffusers")
        d.__path__ = []
        d.DDIMScheduler = _Sched
        ds = types.ModuleType("diffusers.schedulers")
        ds.__path__ = []
        dd = types.ModuleType("diffusers.schedulers.scheduling_ddim")
        dd.DDIMScheduler, dd.DDIMSchedulerOutput = _Sched, _Out
        monkeypatch.setitem(sys.modules, "diffusers", d)
        monkeypatch.setitem(sys.modules, "diffusers.schedulers", ds)
        monkeypatch.setitem(sys.modules, "diffusers.schedulers.scheduling_ddim", dd)
    if golden.recording:
        sys.modules.pop("models.p2p.scheduler_dev", None)
        ref_sd = importlib.import_module("models.p2p.scheduler_dev")
    prompts = list(synth.CAT_PROMPTS)
    torch.set_grad_enabled(False)
    g = torch.Generator().manual_seed(33)
    x_t = torch.randn(1, 4, 64, 64, generator=g)
    enc = torch.randn(1, 4, 64, 64, generator=g)
    x_stars = [torch.randn(1, 4, 64, 64, generator=g) for _ in range(51)]
    te, tok = synth.SynthTextEncoder(), synth.FakeTokenizer()
    uncond = [te(tok([prompts[0]]).input_ids)[0]] * 50
    for prox, guided in ((None, False), ("l0", False), ("l1", True)):
        ref_model, my_model = _models(golden.recording)
        if golden.recording:
            # the reference's proximal path needs scheduler.step(..., ref_image=, recon_lr=, recon_mask=): DDIMSchedulerDev
            ref_model.scheduler = ref_sd.DDIMSchedulerDev(beta_start=0.00085, beta_end=0.012,
                                                          beta_schedule="scaled_linear", clip_sample=False,
                                                          set_alpha_to_one=False)
            ref_model.scheduler.set_timesteps(50)
        kw = dict(guidance_scale=7.5, generator=None, uncond_embeddings=uncond, edit_stage=True, prox=prox, quantile=0.7,
                  image_enc=enc if guided else None, recon_lr=0.1 if guided else 0, recon_t=400 if guided else 1000,
                  x_stars=x_stars, dilate_mask=1)
        b, _ = my_fwd.proximal_guidance_forward(model=my_model, prompt=prompts, controller=EmptyControl(), latent=x_t, **kw)
        assert golden.close(f"prox_{prox}_{guided}/latents", b, lambda: ref_prox.proximal_guidance_forward(
            model=ref_model, prompt=prompts, controller=ref.attention_control.EmptyControl(), latent=x_t, **kw)[0],
            atol=1e-4, k=64), (prox, guided)
        assert golden.value(f"prox_{prox}_{guided}/calls", lambda: _calls(ref_model)).tolist() == _calls(my_model)
        assert len(my_model.unet.calls) == 50
