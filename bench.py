#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: 512x512, 50-step DDIM-inversion + PnP-rectified P2P edit, images/sec.

    python bench.py --gpus N --steps K --warmup W            # this repo (libpnpinv.so, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on the host cores

A "step" is `--lanes` x `--batch` whole images per GPU, each through `P2PEditor.edit_batch` ("directinversion+p2p") on
its own synthetic 4x64x64 latent with the cat prompt pair, i.e. the faithful 650 UNet sample-forwards per image
(50 inversion + 3 x 50 x 4 offset / reconstruction / edit) + 200 fused epilogues (BASELINE.md section 2).  `--batch L`
images share every UNet call (batch L for the inversion, 4 L afterwards; the four 50-step loops run inside
libpnpinv.so, `pnp_run_loop`); `--lanes N` such passes are in flight concurrently on one GPU (parallel.EditLanes: one
CUDA stream, engine handle and host thread per lane, all lanes SHARING one copy of the weights through `pnp_clone`).
`--batch 1 --lanes 1` is the single-image latency configuration (BASELINE config 2 as worded).  Weak scaling: every rank
edits its own K steps (image-parallel, SURVEY.md section 8e); NCCL only broadcasts the inputs and gathers the outputs.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

UNET_GFLOP = 803.27          # per sample-forward, SURVEY.md section 8d
FWD_PER_IMAGE = 650          # faithful directinversion+p2p
N_B4_CALLS, N_B1_CALLS = 150, 50
BLEND = (("cat",), ("cat",))
EQ = {"words": ("watercolor",), "values": (2,)}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["bf16_tflops_sustained"]), float(p["bf16_tflops"]), float(p["hbm_gbs"]), "measured"
    except Exception:
        return 1400.0, 1590.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()  # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 8 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) >= 8 and r[2].isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_outputs(results, limit=60 << 20):
    """{name: float32 array} of the tensors the timed path returned for its last step (one result per lane, the fields of
    BatchEditResult / MasaCtrlBatchResult / the EDICT latents), at most `limit` bytes in all (under 64 MB with the .npy
    headers): an array larger than its share of what is left keeps every s-th entry of its first axis (s fixed by the
    sizes), smaller arrays are kept whole.  The inputs are seeded, so two builds can be compared output for output."""
    fields = {}
    for ln, r in enumerate(results):
        for k, v in vars(r).items():
            if isinstance(v, torch.Tensor) and v.is_floating_point():
                fields[k if len(results) == 1 else f"lane{ln}_{k}"] = v
    out, left = {}, limit
    for i, (k, v) in enumerate(sorted(fields.items(), key=lambda kv: kv[1].numel())):
        share = left // (len(fields) - i)
        stride = -(-v.numel() * 4 // share)
        a = v.detach()[::stride] if stride > 1 else v.detach()
        out[k] = a.float().cpu().numpy()
        left -= out[k].nbytes
    return out


def cpu_unet_times(state_dict, threads, reps=1, which=("b4", "b1")):
    """Times the CPU oracle port (oracle/unet_ref.py, fp32 like the reference's P2P path) on the host cores."""
    from oracle import unet_ref
    from pnpinversion_b200 import synth

    torch.set_num_threads(threads)
    ref = unet_ref.UNetRef(state_dict, dtype=torch.float32)
    tok, te = synth.FakeTokenizer(), synth.SynthTextEncoder()
    prompts = list(synth.CAT_PROMPTS)
    ctx = torch.cat([te(tok([""] * 2).input_ids)[0], te(tok(prompts).input_ids)[0]])
    lat = torch.cat([synth.synth_latent(0), synth.synth_latent(1)])
    out = {}
    with torch.no_grad():
        for name, x, c in (("b4", torch.cat([lat] * 2), ctx), ("b1", lat[:1], ctx[2:3])):
            if name not in which:
                continue
            if reps > 0 and name == "b1":
                ref(x, 501, c)  # warm-up (page-in, thread pool); the B=4 call is too long to repeat
            t0 = time.perf_counter()
            for _ in range(max(reps, 1)):
                ref(x, 501, c)
            out[name] = (time.perf_counter() - t0) / max(reps, 1)
    return out


def run_reference(args, rank, world):
    """The reference arm: the reference's own algorithm on the host CPU (oracle port, there is no compiled reference).
    Each step = one B=4 and one B=1 UNet forward (a bounded sample of the 150 + 50 calls one image needs); images/sec
    is the extrapolation 1 / (150 t_b4 + 50 t_b1).  The fused epilogues are negligible on the CPU as well."""
    if rank != 0:
        return
    from pnpinversion_b200 import synth

    threads = max(1, (os.cpu_count() or 2) // 2)  # physical cores (measured faster than all hyper-threads)
    sd = synth.synth_unet_state_dict(0)
    # Bounded sample: a B=4 fp32 UNet forward of the port takes about a minute on 64 cores, so it is measured ONCE (it
    # also serves as the warm-up of the thread pool); every step then times one B=1 forward and scales the B=4 time by
    # the B=4 : B=1 ratio of that first measurement.  K = 3 steps ~ 2 minutes, K = 10 ~ 3-4 minutes.
    first = cpu_unet_times(sd, threads)
    ratio = first["b4"] / first["b1"]
    # BASELINE config 1 timed IN FULL (BASELINE.md section 3): the 20-step DDIM inversion of one latent through the
    # oracle port's UNet and inverse step, 20 B=1 forwards
    cfg1_s = None
    if not args.no_config1:
        from oracle import p2p_ref, unet_ref

        ref = unet_ref.UNetRef(sd, dtype=torch.float32)
        tok, te = synth.FakeTokenizer(), synth.SynthTextEncoder()
        ctx1 = te(tok([synth.CAT_PROMPTS[0]]).input_ids)[0]
        sch = p2p_ref.Schedule(20, "float32")
        x = synth.synth_latent(0)
        t0 = time.perf_counter()
        with torch.no_grad():
            for t in [50 * i for i in range(20)]:
                x = sch.next_step(ref(x, t, ctx1).float(), t, x)
        cfg1_s = time.perf_counter() - t0
    vals = []
    t_all0 = time.perf_counter()
    for i in range(args.steps):
        b1 = cpu_unet_times(sd, threads, reps=0, which=("b1",))["b1"]
        vals.append(1.0 / (N_B4_CALLS * ratio * b1 + N_B1_CALLS * b1))
    wall = time.perf_counter() - t_all0
    v = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": "images_per_sec_512x512_50step_invert_edit", "value": v, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * wall / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "directinversion+p2p 50 steps, 1 image (B=4 edit batch), faithful 650 UNet forwards",
                   "timing": "host wall clock; extrapolated from 1xB4 + 1xB1 UNet forward per step"},
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": threads, "kind": "port",
                         "sample": f"per step: one B=1 fp32 UNet forward of oracle/unet_ref.py ({1000 * wall / max(args.steps, 1):.0f} ms); "
                                   f"B=4 forward measured once ({first['b4']:.1f} s = {ratio:.2f} x B=1); x150 / x50 "
                                   "extrapolation to one image (650 UNet sample-forwards)",
                         "config1_20_step_inversion_s": cfg1_s},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-image-path", action="store_true", help="skip the image-path (VAE) end-to-end measurement")
    ap.add_argument("--no-single-image", action="store_true", help="skip the one-image-per-pass (batch=1) measurement")
    ap.add_argument("--no-config1", action="store_true", help="reference arm: skip the full 20-step config-1 timing")
    ap.add_argument("--workload", default="p2p", choices=["p2p", "masactrl", "edict"],
                    help="p2p: directinversion+p2p (BASELINE configs 2/3, the headline); masactrl: directinversion+masactrl "
                         "(config 4, default batch 4 -> UNet batch 16); edict: edict+p2p (config 5, default batch 8)")
    ap.add_argument("--batch", type=int, default=0, help="images that share every UNet call (0 = the workload's default)")
    ap.add_argument("--minimal", action="store_true",
                    help="p2p only: the 450-forward variant (no reconstruction pass: its decoded row is the inverted latent "
                         "by the rectification invariant) as the timed workload; the default run reports it beside the "
                         "faithful number")
    ap.add_argument("--text-encoder", default="clip", choices=["synth", "clip"],
                    help="synth: seeded embedding-table stand-in evaluated on the host; clip: the fused CLIP text encoder of "
                         "libpnpinv.so (csrc/clip.cu, random-init SD-1.x text tower) - the prompts are then encoded on the GPU "
                         "inside every pass")
    ap.add_argument("--lanes", type=int, default=1,
                    help="passes in flight per GPU (own CUDA stream / engine handle / host thread, shared weights)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3  # timing rule: W >= 3

    from pnpinversion_b200 import _lib, synth
    from pnpinversion_b200.model import FusedModel
    from pnpinversion_b200.p2p_editor import P2PEditor

    assert torch.cuda.is_available(), "bench.py needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    from pnpinversion_b200.parallel import EditLanes

    WL = {"p2p": dict(batch=8, fwd=650, rows=4, name="directinversion+p2p",
                      what="UNet batch L for the inversion, 4L for the offset / reconstruction / edit loops"),
          "masactrl": dict(batch=4, fwd=550, rows=4, name="directinversion+masactrl",
                           what="UNet batch L inversion, 4L offsets, 2L direct synthesis, 4L mutual self-attention pass"),
          "edict": dict(batch=8, fwd=800, rows=3, name="edict+p2p",
                        what="coupled pair: 2 x (50 + 50 + 40) steps at UNet batch 2L, 2 x 40 P2P steps at 3L")}[args.workload]
    FWD = 450 if (args.minimal and args.workload == "p2p") else WL["fwd"]
    sd = synth.synth_unet_state_dict(0)
    NB = max(1, args.batch or WL["batch"])  # images per pass
    NL = max(1, args.lanes)          # concurrent passes
    L = NB * NL                      # images per step and GPU
    text_encoder = synth.SynthTextEncoder()
    if args.text_encoder == "clip":
        from pnpinversion_b200.clip import FusedCLIPTextEncoder

        text_encoder = FusedCLIPTextEncoder(synth.synth_clip_state_dict(0), device=str(dev))
    parent = FusedModel(sd, device=str(dev), max_batch=WL["rows"] * NB, tokenizer=synth.FakeTokenizer(),
                        text_encoder=text_encoder)
    made = []

    def make_editor():
        m = parent if not made else parent.clone()  # lanes share ONE copy of the weights (pnp_clone)
        made.append(m)
        return P2PEditor(["directinversion+p2p"], dev, num_ddim_steps=50, model=m)

    lanes = EditLanes(make_editor, NL, dev)
    model = parent
    src, tgt = synth.CAT_PROMPTS

    from types import SimpleNamespace

    minimal_now = [bool(args.minimal)]

    def edit_on(editor, z):
        """z: (NB,1,4,64,64) or (NB,4,64,64) latents of one pass -> object with .latents (the edited latents)"""
        zz = z.reshape(NB, 4, 64, 64).to(dev, non_blocking=True)
        if args.workload == "p2p":
            return editor.edit_batch(zz, [src] * NB, [tgt] * NB, guidance_scale=7.5, cross_replace_steps=0.4,
                                     self_replace_steps=0.6, blend_word=BLEND, eq_params=EQ, minimal=minimal_now[0])
        if args.workload == "masactrl":
            from pnpinversion_b200.masactrl import MasaCtrlEditor

            me = MasaCtrlEditor(["directinversion+masactrl"], dev, num_ddim_steps=50, model=editor.ldm_stable)
            return me.edit_batch(zz, [tgt] * NB, guidance_scale=7.5, step=4, layper=10)
        from pnpinversion_b200.edict import edit_image_edict_p2p

        recon, edit = edit_image_edict_p2p(editor.ldm_stable, zz, [src] * NB, [tgt] * NB, use_p2p=True, steps=50)
        return SimpleNamespace(latents=torch.cat([recon[0], edit[0]]))

    def edit_step(zs):
        """One bench step = NL passes of NB images, one pass per lane, through the public editor call."""
        return lanes.run([(lambda ed, z=z: edit_on(ed, z)) for z in zs])

    total = (args.warmup + args.steps) * L
    # inputs: rank 0 draws the seeded latents for everybody and broadcasts them (the image-parallel scatter)
    z_all = torch.empty(world, total, 1, 4, 64, 64, device=dev)
    if rank == 0:
        for r in range(world):
            for i in range(total):
                z_all[r, i] = synth.synth_latent(r * total + i).to(dev)
    if dist is not None:
        dist.broadcast(z_all, src=0)
    z_dev = z_all[rank]

    # ---------------- warm-up: the first pass of every lane alone (plans, GEMM autotuning, graphs), then concurrently
    z_pass = z_dev.reshape(-1, NB, 1, 4, 64, 64)  # [(warmup+steps) * NL passes][NB]
    for ln in range(NL):
        edit_on(lanes.editors[ln], z_pass[ln])
        torch.cuda.synchronize()
    for i in range(1, args.warmup):
        edit_step([z_pass[i * NL + ln] for ln in range(NL)])
    torch.cuda.synchronize()
    lib = _lib.load()
    def launches_now():
        n = sum(ed.ldm_stable.unet.kernel_launches() for ed in lanes.editors)
        return n + (text_encoder.kernel_launches() if hasattr(text_encoder, "kernel_launches") else 0)

    l0 = launches_now()
    first = args.warmup * NL

    # ---------------- timed region 1: inputs resident in HBM
    sampler = ClockSampler(local)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    outs = []
    for i in range(args.steps):
        last = edit_step([z_pass[first + i * NL + ln] for ln in range(NL)])
        outs.extend(r.latents for r in last)
    e1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # copied now: the passes measured below may reuse the buffers these results live in
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, a in host_outputs(last).items():
            np.save(os.path.join(args.dump_outputs, f"{k}.npy"), a)
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        gathered = [torch.empty_like(torch.stack(outs)) for _ in range(world)]
        dist.all_gather(gathered, torch.stack(outs))  # the image-parallel gather of the edited latents
    ms = float(ms.item())
    launches = launches_now() - l0
    value = world * args.steps * L / (ms / 1000.0)

    # ---------------- timed region 2: end to end through the public API with HOST buffers
    z_host = [z_pass[first + i].cpu().pin_memory() for i in range(args.steps * NL)]
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    host_results = []
    for i in range(args.steps):
        # H2D of the latents + context embeddings and D2H of the result latents happen inside each lane's job
        host_results.extend(lanes.run([(lambda ed, z=z: edit_on(ed, z).latents.cpu())
                                       for z in z_host[i * NL:(i + 1) * NL]]))
    t1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    ms2 = torch.tensor([t0.elapsed_time(t1)], device=dev)
    if dist is not None:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = world * args.steps * L / (float(ms2.item()) / 1000.0)
    # the disclosed shortcut, measured beside the faithful number (same inputs, device-resident, 2 steps)
    minimal_line = None
    if args.workload == "p2p" and not args.minimal:
        minimal_now[0] = True
        edit_step([z_pass[first + ln] for ln in range(NL)])
        torch.cuda.synchronize()
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ksteps = min(2, args.steps)
        m0.record()
        for i in range(ksteps):
            edit_step([z_pass[first + i * NL + ln] for ln in range(NL)])
        m1.record()
        torch.cuda.synchronize()
        minimal_now[0] = False
        msm = torch.tensor([m0.elapsed_time(m1)], device=dev)
        if dist is not None:
            dist.all_reduce(msm, op=dist.ReduceOp.MAX)
        minimal_line = {"value": world * ksteps * L / (float(msm.item()) / 1000.0), "unit": "images/s", "steps": ksteps,
                        "unet_forwards_per_image": 450,
                        "what": "same outputs for directinversion+p2p without the reconstruction pass (its decoded row is "
                                "the inverted latent by the rectification invariant; bit-identical edit, "
                                "tests/test_gpu_batched.py)"}
    # the image-path API end to end (P2PEditor.edit_batch on HWC uint8 host arrays -> 2048x512 PIL strips): VAE encode,
    # the four loops, VAE decodes of the reconstruction and edit latents, panel assembly on the host; one step, rank 0
    def side_measurement(fn):
        """The figures beside the headline (rank 0, no collective inside) must not take the headline down with them: an
        exception is recorded in the line instead."""
        try:
            return fn()
        except Exception as e:  # noqa: BLE001
            return {"error": f"{type(e).__name__}: {e}"[:300]}

    def measure_image_path():
        import numpy as np

        from pnpinversion_b200.vae import FusedVAE

        parent.vae = FusedVAE(synth.synth_vae_state_dict(0), device=str(dev))
        try:
            rng = np.random.RandomState(7)
            imgs = [rng.randint(0, 256, (512, 512, 3)).astype(np.uint8) for _ in range(NB)]
            ed0 = lanes.editors[0]
            ed0.edit_batch(imgs[:1], [src], [tgt], blend_word=BLEND, eq_params=EQ)  # VAE plans (B = 1, 2) built outside the timing
            torch.cuda.synchronize()
            w0 = time.perf_counter()
            strips = ed0.edit_batch(imgs, [src] * NB, [tgt] * NB, guidance_scale=7.5, cross_replace_steps=0.4,
                                    self_replace_steps=0.6, blend_word=BLEND, eq_params=EQ)
            torch.cuda.synchronize()
            wall = time.perf_counter() - w0
            assert len(strips) == NB and strips[0].size == (2048, 512)
            return {"value": NB / wall, "unit": "images/s", "images": NB, "seconds": wall,
                    "h2d_bytes": NB * 512 * 512 * 3, "d2h_bytes": NB * 4 * 3 * 512 * 512 * 4,
                    "what": "host wall clock around P2PEditor.edit_batch(list of HWC uint8 arrays) -> PIL strips: VAE encode + "
                            "650 UNet forwards + 4 VAE decodes per image + panel assembly (synthetic VAE weights)"}
        finally:
            parent.vae = None

    image_line = None
    if args.workload == "p2p" and not args.minimal and rank == 0 and not args.no_image_path:
        image_line = side_measurement(measure_image_path)
    # BASELINE config 2 as worded ("batch=1"): one image at a time through the same editor (UNet batch 1 / 4), two images
    # after one warm-up image that builds the plans of those batch sizes; device-resident input, rank 0
    def measure_single_image():
        ed0 = lanes.editors[0]

        def one(i):
            return ed0.edit_batch(z_pass[first][i:i + 1].reshape(1, 4, 64, 64).to(dev), [src], [tgt], guidance_scale=7.5,
                                  cross_replace_steps=0.4, self_replace_steps=0.6, blend_word=BLEND, eq_params=EQ)

        one(0)
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(2):
            one(i % NB)
        s1.record()
        torch.cuda.synchronize()
        sec = s0.elapsed_time(s1) / 1000.0 / 2
        return {"value": 1.0 / sec, "unit": "images/s", "seconds_per_image": sec, "images": 2,
                "what": "one image per pass (UNet batch 1 for the inversion, 4 for the guided loops), faithful 650 "
                        "forwards, same handle and weights; CUDA events"}

    single_line = None
    if args.workload == "p2p" and not args.minimal and rank == 0 and not args.no_single_image and NB > 1:
        single_line = side_measurement(measure_single_image)
    ctx_rows = {"p2p": 4, "masactrl": 4, "edict": 9}[args.workload] * NB  # edict: 4 coupled passes encode 2+2+2+3 rows per image
    # per pass: NB latents from pinned memory + the prompts: token ids ([rows,77] int32) when the fused CLIP text encoder runs
    # on the GPU, the [rows,77,768] fp32 context rows when the host stand-in computes them
    h2d = NL * (NB * 4 * 64 * 64 * 4 + ctx_rows * 77 * (4 if args.text_encoder == "clip" else 768 * 4))
    d2h = NL * 2 * NB * 4 * 64 * 64 * 4

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (tcgen05 GEMM / implicit conv), CUDA events around every op
    sustained, burst, hbm, peak_src = peaks()
    maxops = 1024
    ms_op = (C.c_float * maxops)()
    kind = (C.c_int32 * maxops)()
    fl = (C.c_double * maxops)()
    n = C.c_int()
    kinds = {0: "tcgen05_gemm_conv", 1: "groupnorm", 2: "layernorm", 3: "self_attention", 4: "cross_attention",
             5: "other"}
    agg = {k: [0.0, 0.0, 0] for k in kinds.values()}
    reps = 3
    per_op = None
    PB = WL["rows"] * NB  # the UNet batch of the guided loops
    if model.unet._ctx_batch != PB or True:
        # pnp_unet_profile needs the context of that batch size installed on this handle
        ctxp = torch.zeros(PB, 77, 768, device=dev)
        _lib.check(lib.pnp_set_context(model.unet.handle, C.c_void_p(ctxp.data_ptr()), PB, _lib.current_stream_ptr()))
        model.unet._ctx_ref = None
    for _ in range(reps):
        _lib.check(lib.pnp_unet_profile(model.unet.handle, PB, 501, 10, ms_op, kind, fl, maxops, C.byref(n)))
        if per_op is None:
            per_op = [[kind[i], fl[i], 0.0] for i in range(n.value)]
        for i in range(n.value):
            per_op[i][2] += ms_op[i] / reps
        for i in range(n.value):
            a = agg[kinds[kind[i]]]
            a[0] += ms_op[i] / reps
            a[1] += fl[i] / reps
            a[2] += 1
    dump = os.environ.get("PNP_PROFILE_DUMP")
    if dump:
        with open(dump, "w") as f:
            json.dump(per_op, f)
    tot_ms = sum(a[0] for a in agg.values())
    g = agg["tcgen05_gemm_conv"]
    n_gemm = g[2] // reps
    achieved = g[1] / (g[0] * 1e-3) / 1e12 if g[0] > 0 else 0.0
    roofline = {
        "bound": "tensor",
        "kernel": f"gemm_tcgen05_kernel<BN> (all GEMM / implicit-conv launches of one B={PB} UNet call)",
        "achieved": achieved, "peak": burst, "unit": "TFLOP/s", "frac": achieved / burst,
        "peak_source": f"{peak_src} bf16_tflops (burst: every op is timed alone, 10 launches back to back between two "
                       f"CUDA events); sustained {sustained}",
        "frac_of_sustained_peak": achieved / sustained,
        "launches_per_unet_call": n_gemm, "gflop_per_launch_avg": g[1] / max(n_gemm, 1) / 1e9,
        "avg_launch_us": 1000.0 * g[0] / max(n_gemm, 1), "share_of_unet_time": g[0] / tot_ms if tot_ms else None,
        "traffic": None,
        "unet_batch": PB,
        "by_kernel_ms_per_unet_call": {k: round(v[0], 4) for k, v in agg.items()},
        "unet_sum_of_kernels_ms": tot_ms,
        "unet_tflops_sum_of_kernels": PB * UNET_GFLOP / tot_ms if tot_ms else None,
        "whole_job_tflops": value * FWD * UNET_GFLOP / 1e3,
        "whole_job_frac_of_sustained_peak": value * FWD * UNET_GFLOP / 1e3 / (sustained * world),
    }
    # `traffic`: DRAM bytes per GEMM launch cannot be measured inside a timed bench; it comes from the committed ncu
    # capture of this build at the same UNet batch (profiles/r2_traffic.json, made by tools/traffic_from_ncu.py from a
    # WARM-cache launch list, `--cache-control none`, one whole forward in its real order) - null for any other batch
    tj = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r2_traffic.json")
    if os.path.exists(tj):
        with open(tj) as f:
            tr = json.load(f).get(str(PB))
        if tr:
            roofline["traffic"] = tr["gemm_dram_bytes_per_launch"]
            roofline["traffic_unit"] = "DRAM bytes (read + write) per GEMM launch, ncu warm-cache capture of one forward"
            roofline["traffic_source"] = tr["source"]
    ab, nl = C.c_double(0.0), C.c_int(0)
    _lib.check(lib.pnp_unet_gemm_bytes(model.unet.handle, PB, C.byref(ab), C.byref(nl)))
    # compulsory bytes of the same launches (activations, weights, residual read once; output written once)
    roofline["algorithmic_bytes_per_launch"] = ab.value / max(nl.value, 1)

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        threads = max(1, (os.cpu_count() or 2) // 2)  # physical cores: hyper-threads slow the CPU convolutions down
        t = cpu_unet_times(sd, threads)
        v = 1.0 / (N_B4_CALLS * t["b4"] + N_B1_CALLS * t["b1"])
        cpu = {"value": v, "unit": "images/s", "cores": threads, "kind": "port", "dtype": "f32",
               "sample": f"one B=4 ({t['b4']:.2f} s) and one B=1 ({t['b1']:.2f} s) UNet forward of oracle/unet_ref.py "
                         f"on {threads} host threads; extrapolated x150 / x50 to one image"}

    line = {
        "metric": "images_per_sec_512x512_50step_invert_edit", "value": value, "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": f"{WL['name']} 50 steps, {L} image(s) per step and GPU = {NL} concurrent pass(es) x "
                               f"{NB} image(s) per pass ({WL['what']}), "
                               + ("faithful " if FWD == WL["fwd"] else "MINIMAL (no reconstruction pass) ") +
                               f"{FWD} UNet sample-forwards per image, "
                               "SD-1.x random-init UNet, cat prompts"
                               + (", step loops inside libpnpinv.so (pnp_run_loop)" if args.workload != "edict" else ""),
                   "images_per_step_per_gpu": L, "lanes_per_gpu": NL, "images_per_pass": NB,
                   "weights": "one fp16 copy per GPU shared by all lanes (pnp_clone)",
                   "parallelism": f"image-parallel x{world} GPUs x {NL} concurrent passes (CUDA streams) x {NB} images "
                                  "per UNet call",
                   "l2": "each step streams 1.72 GB of fp16 weights per UNet call (> 126 MB L2), no flush needed",
                   "text_encoder": ("fused CLIP text encoder on the GPU (csrc/clip.cu, random-init)" if args.text_encoder == "clip"
                                    else "seeded embedding-table stand-in on the host"),
                   "accumulate": "fp32"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "roofline": roofline,
    }
    if minimal_line is not None:
        line["minimal_450"] = minimal_line
    if image_line is not None:
        line["image_path_e2e"] = image_line
    if single_line is not None:
        line["single_image"] = single_line
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
