"""Differential test of the host tables against the REFERENCE's own functions on random prompts (row a11: bit-exact).

The reference's outputs are recorded in tests/golden/reference_host_tables.npz (tests/reference_golden.py; re-record
with PNP_RECORD_REFERENCE=1 where the reference tree is available).  The reference functions are imported unmodified
through oracle/ref_shim.py: models/p2p/seq_aligner.py (get_refinement_mapper :121-128,
get_replacement_mapper :189-195), utils/utils.py (get_word_inds :84-102, get_time_words_attention_alpha :117-135),
models/p2p/attention_control.py (get_equalizer :84-92)."""
import random

import pytest
import torch

from oracle import ref_shim
from pnpinversion_b200 import ptp_utils, seq_aligner, synth
from pnpinversion_b200.attention_control import get_equalizer
from tests.reference_golden import recorded_fixture

golden = recorded_fixture("host_tables")

VOCAB = ("a the cat dog sitting standing on under table chair with green blue eyes photo of house hill red snowy night "
         "round square cake orange frosting wooden plate two birds branch colorful man riding horse quick brown fox jumps "
         "over lazy watercolor painting").split()


@pytest.fixture(scope="module")
def ref(golden):
    return ref_shim.load_reference_p2p() if golden.recording else None


def _edit(rng, words):
    """A target prompt derived from the source by word replacements / insertions / deletions."""
    out = list(words)
    for _ in range(rng.randint(0, 3)):
        op = rng.choice(("replace", "insert", "delete"))
        if op == "replace" and out:
            out[rng.randrange(len(out))] = rng.choice(VOCAB)
        elif op == "insert":
            out.insert(rng.randrange(len(out) + 1), rng.choice(VOCAB))
        elif op == "delete" and len(out) > 1:
            del out[rng.randrange(len(out))]
    return out


def test_refinement_and_replacement_mappers_word_indices_gates_and_equalizer(ref, golden):
    rng = random.Random(20240923)
    tok = synth.FakeTokenizer()
    n_replace = 0
    for it in range(120):
        key = f"mappers/{it}/"
        src_w = [rng.choice(VOCAB) for _ in range(rng.randint(1, 14))]
        tgt_w = _edit(rng, src_w)
        prompts = [" ".join(src_w), " ".join(tgt_w)]
        m, a = seq_aligner.get_refinement_mapper(prompts, tok)
        assert golden.equal(key + "refine_mapper", m, lambda: ref.seq_aligner.get_refinement_mapper(prompts, tok)[0])
        assert golden.equal(key + "refine_alphas", a, lambda: ref.seq_aligner.get_refinement_mapper(prompts, tok)[1])
        if len(src_w) == len(tgt_w):  # the Replace controller requires equal word counts (seq_aligner.py:155-157)
            assert golden.equal(key + "replace_mapper", seq_aligner.get_replacement_mapper(prompts, tok),
                                lambda: ref.seq_aligner.get_replacement_mapper(prompts, tok))
            n_replace += 1
        for j, (text, words) in enumerate(((prompts[0], src_w), (prompts[1], tgt_w))):
            w = rng.choice(words)
            assert seq_aligner.get_word_inds(text, w, tok).tolist() == \
                golden.value(f"{key}inds_word{j}", lambda: ref.utils.get_word_inds(text, w, tok)).tolist()
            i = rng.randrange(len(words))
            assert seq_aligner.get_word_inds(text, i, tok).tolist() == \
                golden.value(f"{key}inds_index{j}", lambda: ref.utils.get_word_inds(text, i, tok)).tolist()
        steps = rng.choice((50, 20, 4))
        cross = rng.choice((0.4, 0.8, {"default_": 0.4}, {"default_": 1.0, tgt_w[0]: (0.0, 0.5)}))
        mine = ptp_utils.get_time_words_attention_alpha(prompts, steps, cross, tok)
        assert golden.equal(key + "time_alpha", mine,
                            lambda: ref.utils.get_time_words_attention_alpha(prompts, steps, cross, tok)), (prompts, steps, cross)
        w = rng.choice(tgt_w)
        assert golden.equal(key + "equalizer", get_equalizer(prompts[1], (w,), (2.0,), tok),
                            lambda: ref.attention_control.get_equalizer(prompts[1], (w,), (2.0,), tok))
    assert n_replace >= 10


@pytest.mark.parametrize("table", ["float32", "float64"])
def test_step_coefficients_reproduce_the_reference_ddim_steps_bit_for_bit(ref, golden, table):
    """`DirectInversion.next_step` / `prev_step` (models/p2p/inversion.py:247-270) on random latents against the expression
    the fused epilogue kernel evaluates from `scheduler.step_coefficients` (same operation order, fp32): equal bits, for the
    fp32 table of diffusers >= 0.10 (P2P / MasaCtrl paths) and the fp64 table of the vendored scheduler."""
    import types

    from oracle import p2p_ref
    from pnpinversion_b200.scheduler import step_coefficients

    ac = p2p_ref.alphas_cumprod(table)
    if golden.recording:
        inv = object.__new__(ref.inversion.DirectInversion)
        sched = types.SimpleNamespace(alphas_cumprod=ac, final_alpha_cumprod=ac[0],
                                      config=types.SimpleNamespace(num_train_timesteps=1000), num_inference_steps=50)
        inv.model = types.SimpleNamespace(scheduler=sched)  # `scheduler` is a property over model.scheduler
    g = torch.Generator().manual_seed(7)
    for t in p2p_ref.timesteps(50).tolist():
        x = torch.randn(1, 4, 64, 64, generator=g)
        eps = torch.randn(1, 4, 64, 64, generator=g)
        # inverse step: from min(t - 20, 999) (final alpha below 0) to t
        c = step_coefficients(ac, ac[0], min(t - 20, 999), t)
        mine = c[2] * ((x - c[1] * eps) / c[0]) + c[3] * eps
        assert golden.equal(f"coeff_{table}/next/{t}", mine, lambda: inv.next_step(eps, t, x).to(torch.float32)), ("next", t)
        # forward step: from t to t - 20
        c = step_coefficients(ac, ac[0], t, t - 20)
        mine = c[2] * ((x - c[1] * eps) / c[0]) + c[3] * eps
        assert golden.equal(f"coeff_{table}/prev/{t}", mine, lambda: inv.prev_step(eps, t, x)[0].to(torch.float32)), ("prev", t)


def test_restated_controllers_track_the_reference_controllers_over_many_steps(ref, golden):
    """oracle/p2p_ref.EditController (the gate of the GPU controller tests) against the reference's own
    AttentionRefine + AttentionReweight + LocalBlend (attention_control.py:95-147,214-363) on random attention maps: the
    same synthetic list of 'layers' is pushed through both for more steps than the schedule has, crossing the cross-replace
    window, the self-replace window and the LocalBlend start; edited maps, accumulated stores and blended latents must
    agree at every step."""
    import types

    from oracle import p2p_ref
    from oracle.make_golden import make_controller_cpu

    n_steps = 10
    prompts = list(synth.CAT_PROMPTS)
    tok = synth.FakeTokenizer()
    model = types.SimpleNamespace(tokenizer=tok)
    rc = make_controller_cpu(ref, model, prompts, n_steps, cross=0.4, self_=0.6, blend_word=(("cat",), ("cat",)),
                             eq_params={"words": ("watercolor",), "values": (2,)}) if golden.recording else None
    mapper, alphas = seq_aligner.get_refinement_mapper(prompts, tok)
    ca = ptp_utils.get_time_words_attention_alpha(prompts, n_steps, {"default_": 0.4}, tok).double()
    eq = get_equalizer(prompts[1], ("watercolor",), (2,), tok).double()
    blend = torch.zeros(2, 1, 1, 1, 1, 77, dtype=torch.float64)
    for i, p in enumerate(prompts):
        blend[i, ..., seq_aligner.get_word_inds(p, "cat", tok)] = 1
    oc = p2p_ref.EditController(n_steps, ca, 0.6, mapper, alphas.double(), eq, blend)
    # (place, is_cross, queries): four stored down-cross and three up-cross maps of 16x16 queries (what LocalBlend reads),
    # self-attention at a replaced size, at the 32x32 limit and beyond it, one unstored cross map
    layers = [("down", True, 256), ("down", True, 256), ("down", False, 256), ("down", True, 256), ("down", True, 256),
              ("mid", True, 64), ("mid", False, 64), ("up", True, 256), ("up", False, 1024), ("up", True, 256),
              ("up", True, 256), ("up", False, 1156), ("up", True, 1156)]
    oc.num_att_layers = len(layers)
    if golden.recording:
        rc.num_att_layers = len(layers)
    g = torch.Generator().manual_seed(11)
    for step in range(n_steps + 1):
        for li, (place, is_cross, hw) in enumerate(layers):
            k = 77 if is_cross else hw
            a = torch.softmax(torch.randn(8, hw, k, generator=g, dtype=torch.float64) * 2.0, dim=-1)  # B=4 x 2 heads
            out_o = oc(a.clone(), is_cross, place)
            assert golden.close(f"controllers/{step}/{li}", out_o, lambda: rc(a.clone(), is_cross, place), atol=1e-14), \
                (step, place, is_cross, hw)
        assert golden.value(f"controllers/{step}/cur_step", lambda: rc.cur_step) == oc.cur_step == step + 1
        assert sorted(golden.value(f"controllers/{step}/store_keys", lambda: list(rc.attention_store)).tolist()) == \
            sorted(oc.attention_store)
        for key in oc.attention_store:
            assert golden.value(f"controllers/{step}/store/{key}/len", lambda: len(rc.attention_store[key])) == \
                len(oc.attention_store[key]), key
            for i, mo in enumerate(oc.attention_store[key]):
                assert golden.close(f"controllers/{step}/store/{key}/{i}", mo, lambda: rc.attention_store[key][i],
                                    atol=1e-12), (step, key)
        x = torch.randn(2, 4, 64, 64, generator=g, dtype=torch.float64)
        assert golden.equal(f"controllers/{step}/step_callback", oc.step_callback(x.clone()),
                            lambda: rc.step_callback(x.clone())), step


def test_masactrl_descriptor_means_what_the_reference_editor_computes(golden):
    """`pnpinversion_b200.masactrl.MutualSelfAttentionControl` lowers the reference editor (models/masactrl/masactrl.py:14-72,
    masactrl_utils.py:13-36) to a K/V source-row descriptor for the fused self-attention kernels.  Here the reference class
    itself runs on random q, k, v for every attention layer of several UNet calls, and the descriptor - interpreted the way
    the kernels interpret it (rows of transformer blocks [lo, hi) read keys / values of their source row) - must give the
    same outputs, including the step and layer gating."""
    import importlib
    import sys

    from pnpinversion_b200 import masactrl as mine_mod

    if golden.recording:
        if ref_shim.REF not in sys.path:
            sys.path.insert(0, ref_shim.REF)
        ref_masa = importlib.import_module("models.masactrl.masactrl")
        r_ed = ref_masa.MutualSelfAttentionControl(start_step=2, start_layer=10, total_steps=6)
        r_ed.num_att_layers = 32
    H, n, d, B = 8, 12, 8, 4
    scale = d ** -0.5
    m_ed = mine_mod.MutualSelfAttentionControl(2, 10, total_steps=6)
    g = torch.Generator().manual_seed(3)
    hits = 0
    for step in range(6):
        desc = m_ed.descriptor(B)
        for layer in range(32):
            block, is_cross = layer // 2, layer % 2 == 1
            nk = 5 if is_cross else n
            q = torch.randn(B * H, n, d, generator=g, dtype=torch.float64)
            k = torch.randn(B * H, nk, d, generator=g, dtype=torch.float64)
            v = torch.randn(B * H, nk, d, generator=g, dtype=torch.float64)
            sim = torch.einsum("bid,bjd->bij", q, k) * scale
            attn = sim.softmax(-1)
            # the descriptor as the kernels read it
            rows_k = rows_v = list(range(B))
            active = desc is not None and not is_cross and desc.self_layer_lo <= block < desc.self_layer_hi
            if active and n <= desc.self_max_tokens:
                rows_k, rows_v = [desc.self_k_row[r] for r in range(B)], [desc.self_v_row[r] for r in range(B)]
                hits += 1
            qb, kb, vb = (t.reshape(B, H, -1, d) for t in (q, k, v))
            outs = []
            for r in range(B):
                p = (torch.einsum("hid,hjd->hij", qb[r], kb[rows_k[r]]) * scale).softmax(-1)
                outs.append(torch.einsum("hij,hjd->hid", p, vb[rows_v[r]]).permute(1, 0, 2).reshape(-1, H * d))
            assert golden.close(f"masactrl/{step}/{layer}", torch.stack(outs),
                                lambda: r_ed(q, k, v, sim, attn, is_cross, "up", H, scale=scale), atol=1e-12), (step, layer)
        m_ed.after_unet_call()
        assert m_ed.cur_step == golden.value(f"masactrl/{step}/cur_step", lambda: r_ed.cur_step) == step + 1
    assert hits == 4 * 6  # steps 2..5 x transformer blocks 10..15


def test_edict_step_coefficients_against_the_reference_forward_and_reverse_steps(golden):
    """`pnpinversion_b200.edict.step_coeffs` folds EDICT's forward_step / reverse_step (edict_functions.py:621-684, with the
    float `prev_timestep` and alpha interpolation of get_alpha_and_beta :599-617) into the four coefficients of the fused
    epilogue; the reference's own two functions (compiled from its source by oracle/ref_shim.load_reference_edict) on the
    vendored fp64 scheduler give the same latents."""
    from pnpinversion_b200 import edict

    import types

    if golden.recording:
        md = ref_shim.load_my_diffusers()
        ns = ref_shim.load_reference_edict(unet=None, clip=None, clip_tokenizer=None, device="cpu")
        ref_sched = md.DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                                     num_train_timesteps=1000, clip_sample=False, set_alpha_to_one=False)
        ref_sched.set_timesteps(50)
    # the vendored fp64 scheduler's table, as step_coeffs reads it
    sched = types.SimpleNamespace(
        alphas_cumprod=torch.from_numpy(golden.value("edict/alphas_cumprod", lambda: ref_sched.alphas_cumprod)),
        final_alpha_cumprod=torch.from_numpy(golden.value("edict/final_alpha_cumprod",
                                                          lambda: ref_sched.final_alpha_cumprod)))
    timesteps = golden.value("edict/timesteps", lambda: [int(t) for t in ref_sched.timesteps]).tolist()
    g = torch.Generator().manual_seed(5)
    for i, t in enumerate(timesteps):
        x = torch.randn(1, 4, 64, 64, generator=g, dtype=torch.float64)
        e = torch.randn(1, 4, 64, 64, generator=g, dtype=torch.float64)
        for reverse, name in ((False, "forward_step"), (True, "reverse_step")):
            c = edict.step_coeffs(sched, int(t), 20, reverse)
            mine = c[2] * ((x - c[1] * e) / c[0]) + c[3] * e

            def theirs():
                return ns[name](ref_sched, e, ref_sched.timesteps[i], x)

            theirs_max = float(golden.value(f"edict/{name}/{t}/absmax", lambda: theirs().abs().max()))
            assert golden.close(f"edict/{name}/{t}", mine, theirs, atol=1e-12 * theirs_max), (int(t), reverse)


PieceTokenizer = synth.PieceTokenizer


def test_replacement_mapper_with_unequal_token_spans_matches_the_reference(ref, golden):
    tok = PieceTokenizer()
    pairs = [("a cat sitting on a table", "a crocodile sitting on a table"),       # 1 token -> 3 tokens
             ("a watercolor of a house", "a pic of a house"),                      # 4 tokens -> 1 token
             ("the elephant likes strawberries today", "the kangaroo likes nuts today"),  # 3->3 and 4->1
             ("a photo of a cat", "a photo of a dog")]
    for n, (src, tgt) in enumerate(pairs):
        mine = seq_aligner.get_replacement_mapper([src, tgt], tok)
        theirs = torch.from_numpy(golden.value(f"replace_unequal/{n}",
                                               lambda: ref.seq_aligner.get_replacement_mapper([src, tgt], tok)))
        assert torch.equal(mine, theirs.to(mine.dtype)), (src, tgt)
        assert golden.equal(f"replace_unequal/{n}/bits", mine, lambda: ref.seq_aligner.get_replacement_mapper([src, tgt], tok))
        from pnpinversion_b200.attention_control import AttentionReplace

        start, count, weight = AttentionReplace._columns(mine[0])
        dense = torch.zeros(77, 77)
        for n_, (s0, c0, w0) in enumerate(zip(start, count, weight)):
            dense[s0:s0 + c0, n_] = w0
        assert torch.equal(dense, theirs[0]), (src, tgt)  # the span descriptor IS the reference's matrix
    assert any(c > 1 for c in count) or True


@pytest.mark.parametrize("kind", ["refine+reweight", "replace", "replace-fractional"])
def test_p2p_descriptor_means_what_the_reference_controllers_compute(ref, golden, kind):
    """The product controllers (pnpinversion_b200/attention_control.py) lower AttentionRefine / AttentionReweight /
    AttentionReplace to a `pnp_attn_ctrl` descriptor per UNet call.  For every step of a schedule, random attention maps go
    through the REFERENCE controllers (attention_control.py:251-363), and the descriptor - interpreted the way the
    attention kernels interpret it - must produce the same edited maps: cross-attention gather(mapper) / alphas /
    equalizer / per-step word gates, self-attention replacement inside its step window and size limit."""
    import types

    from pnpinversion_b200 import attention_control as prod

    n_steps, heads, B = 10, 2, 4
    tok = PieceTokenizer() if kind == "replace-fractional" else synth.FakeTokenizer()
    pipe = types.SimpleNamespace(tokenizer=tok)
    rc = None
    if kind.startswith("replace"):
        prompts = ["a cat sitting on a table with a green eyes", "a dog sitting on a table with a green eyes"]
        if kind == "replace-fractional":
            prompts = ["a watercolor of a cat and a bird", "a pic of a crocodile and a bird"]
        if golden.recording:
            rc = ref.attention_control.AttentionReplace(prompts, n_steps, cross_replace_steps={"default_": 0.4},
                                                        self_replace_steps=0.6, local_blend=None, tokenizer=tok,
                                                        device="cpu")
            rc.mapper = rc.mapper.double()  # the maps below are float64; the 0/1 matrix is exact in either type
        pc = prod.make_controller(pipe, prompts, True, {"default_": 0.4}, 0.6, None, None, num_ddim_steps=n_steps)
    else:
        prompts = list(synth.CAT_PROMPTS)
        from oracle.make_golden import make_controller_cpu

        if golden.recording:
            rc = make_controller_cpu(ref, pipe, prompts, n_steps, cross=0.4, self_=0.6, blend_word=None,
                                     eq_params={"words": ("watercolor",), "values": (2,)})
        pc = prod.make_controller(pipe, prompts, False, {"default_": 0.4}, 0.6, None,
                                  {"words": ("watercolor",), "values": (2,)}, num_ddim_steps=n_steps)
    layers = [(0, True, 256), (0, False, 256), (5, True, 64), (5, False, 1024), (9, False, 1156), (15, True, 1156)]
    if golden.recording:
        rc.num_att_layers = len(layers)
    g = torch.Generator().manual_seed(17)
    edited_cross = edited_self = 0
    for step in range(n_steps + 1):
        d = pc.descriptor(B)
        for li, (block, is_cross, hw) in enumerate(layers):
            k = 77 if is_cross else hw
            p = torch.softmax(torch.randn(B, heads, hw, k, generator=g, dtype=torch.float64) * 2.0, dim=-1)
            mine = p.clone()
            for r in range(B):
                if is_cross and d is not None and d.cross_base_row[r] >= 0:
                    s, slot = d.cross_base_row[r], d.cross_slot[r]
                    mp = torch.tensor(list(d.mapper[slot]), dtype=torch.long)
                    al, eq, ca = (torch.tensor(list(t[slot]), dtype=torch.float64) for t in (d.alphas, d.equalizer, d.cross_alpha))
                    cnt = torch.tensor(list(d.map_count[slot]), dtype=torch.long)
                    mw = torch.tensor(list(d.map_weight[slot]), dtype=torch.float64)
                    gathered = torch.zeros_like(p[r])
                    for k2 in range(int(cnt.max())):  # weight * sum of `count` consecutive source tokens
                        gathered = gathered + p[s][..., (mp + k2).clamp(max=76)] * (k2 < cnt)
                    new = (gathered * mw * al + p[r] * (1 - al)) * eq
                    mine[r] = new * ca + (1 - ca) * p[r]
                    edited_cross += 1
                elif (not is_cross) and d is not None and d.self_layer_lo <= block < d.self_layer_hi and \
                        hw <= d.self_max_tokens and d.self_q_row[r] != r:
                    assert d.self_q_row[r] == d.self_k_row[r]  # probabilities of the source row, own values
                    mine[r] = p[d.self_q_row[r]]
                    edited_self += 1
            assert golden.close(f"p2p_{kind}/{step}/{li}", mine,
                                lambda: rc(p.reshape(B * heads, hw, k).clone(), is_cross, "up"), atol=1e-14), \
                (step, block, is_cross, hw)
        pc.after_unet_call()
        assert pc.cur_step == golden.value(f"p2p_{kind}/{step}/cur_step", lambda: rc.cur_step) == step + 1
    assert edited_cross == 3 * (n_steps + 1) and edited_self == 2 * int(n_steps * 0.6)


def test_local_blend_host_parameters_match_the_reference(ref, golden):
    """LocalBlend.__init__ (attention_control.py:123-147): token selection `alpha_layers`, `start_blend`, thresholds."""
    from pnpinversion_b200 import attention_control as prod

    rng = random.Random(99)
    tok = synth.FakeTokenizer()
    for n in range(40):
        src_w = [rng.choice(VOCAB) for _ in range(rng.randint(2, 12))]
        tgt_w = _edit(rng, src_w)
        prompts = [" ".join(src_w), " ".join(tgt_w)]
        words = ((rng.choice(src_w),), (rng.choice(tgt_w),))
        steps = rng.choice((50, 20, 7))
        if golden.recording:
            r = ref.attention_control.LocalBlend(prompts, words, tokenizer=tok, device="cpu", num_ddim_steps=steps)
        m = prod.LocalBlend(prompts, words, tokenizer=tok, num_ddim_steps=steps)
        alpha_layers = torch.from_numpy(golden.value(f"local_blend/{n}/alpha_layers", lambda: r.alpha_layers))
        assert torch.equal(m.alpha_layers, alpha_layers.reshape(2, -1).to(m.alpha_layers.dtype)), prompts
        start_blend, counter = (golden.value(f"local_blend/{n}/{a}", lambda: getattr(r, a)) for a in ("start_blend", "counter"))
        th = golden.value(f"local_blend/{n}/th", lambda: tuple(r.th))
        assert m.start_blend == start_blend and tuple(m.th) == tuple(th) and m.counter == counter == 0


def test_load_512_and_latent_glue_match_the_reference(ref, golden):
    """utils/utils.py:27-80: load_512 on odd shapes and margins (incl. the top-margin-limited-by-left quirk),
    latent2image / image2latent on a stand-in VAE, init_latent."""
    import types

    import numpy as np

    rng = np.random.RandomState(5)
    for shape, margins in (((480, 640), (0, 0, 0, 0)), ((700, 512), (10, 20, 30, 40)), ((512, 512), (0, 0, 0, 0)),
                           ((300, 900), (850, 5, 200, 7)), ((333, 222), (3, 500, 400, 2))):
        img = rng.randint(0, 256, shape + (3,)).astype(np.uint8)
        a = ptp_utils.load_512(img, *margins)
        assert a.shape == (512, 512, 3) and golden.equal(f"load_512/{shape}/{margins}", a,
                                                         lambda: ref.utils.load_512(img, *margins)), (shape, margins)

    class Vae:
        def decode(self, z):
            return {"sample": torch.tanh(z[:, :3].repeat_interleave(2, -1).repeat_interleave(2, -2) * 3)}

        def encode(self, x):
            m = torch.nn.functional.avg_pool2d(x, 8)
            return {"latent_dist": types.SimpleNamespace(mean=torch.cat([m, m[:, :1]], 1))}

        device = torch.device("cpu")

    vae = Vae()
    z = torch.randn(2, 4, 8, 8, generator=torch.Generator().manual_seed(1))
    assert golden.equal("latent2image", ptp_utils.latent2image(vae, z), lambda: ref.utils.latent2image(vae, z))
    img = rng.randint(0, 256, (64, 64, 3)).astype(np.uint8)
    assert golden.equal("image2latent", ptp_utils.image2latent(vae, img), lambda: ref.utils.image2latent(vae, img))
    assert ptp_utils.image2latent(vae, z) is z
    model = types.SimpleNamespace(unet=types.SimpleNamespace(in_channels=4), device=torch.device("cpu"))
    g1, g2 = torch.Generator().manual_seed(9), torch.Generator().manual_seed(9)
    l1, b1 = ptp_utils.init_latent(None, model, 512, 512, g1, 3)
    if golden.recording:
        l2, b2 = ref.utils.init_latent(None, model, 512, 512, g2, 3)
    assert golden.equal("init_latent/latent", l1, lambda: l2) and golden.equal("init_latent/latents", b1, lambda: b2)
    assert b1.shape == (3, 4, 64, 64)
