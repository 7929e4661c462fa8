"""bench.py — headline benchmark of the FateZero hot path on B200.

metric  : edited frames/sec = F / (T_inversion + T_edit) for one 512x512x8-frame clip, 50 DDIM steps, one target prompt
          (BASELINE.json / SURVEY.md §8(d)); one "step" of this script = ONE full clip edit (50 inversion UNet forwards with the
          attention-map STORE + 50 CFG edit forwards with INJECT), random-init SD-1.4-geometry UNet, synthetic latents.
value   : inputs already resident in HBM when the timed region starts.
e2e     : the same edit through the reference-facing API with HOST buffers: per step the clean latents are copied from pinned host
          memory and the edited latents are read back to the host inside the timed region.
roofline: the dominant kernel is the tcgen05 tap-GEMM (convs + linears + temporal LoRA, 86% of the FLOPs): algorithmic FLOPs of all its
          launches in one clip edit / the sum of their CUDA-event durations (instrumented extra pass), against the measured bf16 peak.
st_attn : ST-attn TFLOPS = sum over the spatio-temporal attention launches of a clip of 4*BF*heads*S*T*d / sum of their CUDA-event durations.
vae     : the VAE bracket (encode + decode of the clip's frames on the tap-GEMM), reported next to the metric, not inside it.
Launch:  python bench.py [--gpus N --steps K --warmup W] [--config style|attribute|long24|shape768]
         N>1 under torch.distributed.run, one rank per GPU: the frames of ONE clip are split over the ranks with the same weights as N=1
         ("strong" scaling; exchanges = peer-memory push/flag kernels, DESIGN.md §6); --shard clips = independent clips per rank (replicas)
         python bench.py --impl reference ...   (CPU arm: the oracle port of the reference on the host cores, one full-frame step pair per step)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

DDIM_STEPS = 50
SRC = "a silver jeep driving down a curvy road in the countryside"
# BASELINE.json configs #2..#5 (SURVEY.md §8(d)); the default (`style`) is the configuration the metric is quoted on
CONFIGS = {
    "style": dict(  # config/style/jeep_watercolor.yaml p2p_config[1]
        frames=8, size=64, model_config=dict(lora=160, SparseCausalAttention_index=["mid"], least_sc_channel=640),
        tgt="watercolor painting of " + SRC,
        p2p=dict(is_replace_controller=False, cross_replace_steps={"default_": 0.8}, self_replace_steps=0.8,
                 eq_params={"words": ["watercolor"], "values": [10, 10]}),
        workload="style edit (config/style): 512x512x8f, 50 DDIM steps, Refine+Reweight, SD-1.4 UNet geometry, synthetic weights/latents"),
    "attribute": dict(  # config/attribute/bear_tiger_lion_leopard.yaml:65-69 + config/teaser/jeep_posche_local_latent_blend.yaml:29-39
        frames=8, size=64, model_config=dict(lora=160, SparseCausalAttention_index=["mid"], least_sc_channel=640),
        tgt="a Porsche car driving down a curvy road in the countryside",
        p2p=dict(is_replace_controller=True, cross_replace_steps={"default_": 0.7}, self_replace_steps=0.7,
                 blend_words=[["silver", "jeep"], ["Porsche", "car"]], blend_self_attention=True, blend_latents=True, blend_th=[0.3, 0.3]),
        workload="attribute edit (config/attribute + teaser blend): 512x512x8f, 50 DDIM steps, Replace + self-attention mask blend + latent blend"),
    "long24": dict(  # BASELINE config #4; precedent config/style/train_shinkai.yaml:6 (32 frames, ['mid'])
        frames=24, size=64, model_config=dict(lora=160, SparseCausalAttention_index=["mid"], least_sc_channel=640),
        tgt="watercolor painting of " + SRC,
        p2p=dict(is_replace_controller=False, cross_replace_steps={"default_": 0.8}, self_replace_steps=0.8,
                 eq_params={"words": ["watercolor"], "values": [10, 10]}),
        workload="long clip: 512x512x24f, 50 DDIM steps, Refine+Reweight, frames sharded over the GPUs (109 GiB of maps per clip)"),
    "shape768": dict(  # config/shape/jeep_posche.yaml p2p_config[1] semantics: default [-1,'first'] K/V frames, ST-attn at every resolution
        frames=16, size=96, model_config=dict(lora=160),
        tgt="a Porsche car driving down a curvy road in the countryside",
        p2p=dict(is_replace_controller=True, cross_replace_steps={"default_": 0.5}, self_replace_steps=0.5,
                 blend_words=[["silver", "jeep"], ["Porsche", "car"]], blend_self_attention=True, blend_th=[0.3, 0.3]),
        workload="shape edit (config/shape): 768x768x16f, 50 DDIM steps, Replace + self-attention mask blend, [-1,'first'] ST-attn at r=96..12"),
}
CFG = dict(CONFIGS["style"], name="style")


def select_config(name: str):
    CFG.clear()
    CFG.update(CONFIGS[name], name=name)
    if os.environ.get("FZ_BENCH_FRAMES"):  # development: e.g. 1 frame on one GPU = what one rank of an 8-GPU frame-sharded run computes
        CFG["frames"] = int(os.environ["FZ_BENCH_FRAMES"])
        CFG["workload"] += f" [frames overridden: {CFG['frames']}]"


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return dict(bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, hbm_gbs=6650.0), "fallback"


# ------------------------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i",
                                          str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=(max(mx) if mx else None), reasons=sorted(reasons),
                    samples=len(sm))


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
def build_pipe(device, degenerate_temporal: bool = False):
    from fatezero_b200 import DDIMScheduler, P2pDDIMSpatioTemporalPipeline, UNetPseudo3DConditionModel, synth
    from fatezero_b200.unet import unet_param_spec
    cfg = synth.SD14_UNET_CONFIG
    unet = UNetPseudo3DConditionModel(**cfg, **CFG["model_config"])
    spec = unet_param_spec(dict(cfg), CFG["model_config"])
    # non-degenerate temporal weights: nothing on the path is an identity that could be skipped (SURVEY.md §8(d))
    unet.load_state_dict(synth.synth_state_dict({k: v[0] for k, v in spec.items()}, seed=0, degenerate_temporal=degenerate_temporal))
    unet.to(device)
    te = synth.ToyTextEncoder(cfg["cross_attention_dim"]).to(device)
    pipe = P2pDDIMSpatioTemporalPipeline(synth.VaeStub(), te, synth.ToyTokenizer(), unet, DDIMScheduler())
    pipe.scheduler.set_timesteps(DDIM_STEPS)
    pipe.prepare_before_train_loop()
    return pipe


def edit_clip(pipe, x0_dev, emb_src):
    """One full clip edit through the reference-facing API: inversion with STORE, then edit_type='swap'.  Returns the inverted latents
    the edit starts from and the pipeline call's result dict."""
    from fatezero_b200 import controllers
    pipe.scheduler.set_timesteps(DDIM_STEPS)
    old = getattr(pipe, "store_controller", None)
    pipe.store_controller = controllers.AttentionStore()
    controllers.register_attention_control(pipe, pipe.store_controller)  # also drops the previous clip's edit controller
    if old is not None:
        old.reset()  # the previous clip's 36 GiB map cache goes back to the caching allocator BEFORE this clip allocates its own
    del old
    pipe.store_controller.LOW_RESOURCE = True
    inv = pipe.ddim_clean2noisy_loop(x0_dev, emb_src, pipe.store_controller)
    pipe.store_controller.LOW_RESOURCE = False
    save_path = None
    if CFG["p2p"].get("blend_words"):
        import tempfile
        save_path = tempfile.mkdtemp()  # attention_util.py:339,348: blending needs a save_path (nothing is written on this path)
    out = pipe(prompt=CFG["tgt"], source_prompt=SRC, edit_type="swap", image=None, strength=None, generator=None,
               num_inference_steps=DDIM_STEPS, clip_length=x0_dev.shape[2], guidance_scale=7.5, num_images_per_prompt=1, latents=inv[-1],
               uncond_embeddings_list=None, save_path=save_path, height=8 * CFG["size"], width=8 * CFG["size"], output_type="latent",
               use_inversion_attention=True, save_self_attention=False, **CFG["p2p"])
    return inv[-1], out


FRAME_AXIS = {"inverted_latents": 2, "edited_latents": 2, "mask_list": 1}


def dump_outputs(dirname, inv_latents, out, world, shard_frames):
    """--dump-outputs: what one clip edit returned to its caller, as float32 DIR/<name>.npy (a few MB: the latents, plus the per-step
    latent-blend masks of the configs that blend latents).  Inputs and weights are seeded, so two builds can be compared file by file.
    N > 1: gathered on rank 0, the ranks' frames joined along the frame axis (--shard frames) or stacked as a leading clip axis."""
    import numpy as np
    import torch.distributed as dist
    arrays = {"inverted_latents": inv_latents, "edited_latents": out["sdimage_output"].images}
    if out["mask_list"]:
        arrays["mask_list"] = torch.stack(out["mask_list"])
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = world * sum(a.nbytes for a in arrays.values())  # every rank holds equal shapes: all ranks decide alike, before the gather
    if total > 64 << 20:
        raise SystemExit(f"--dump-outputs: {total / 2**20:.1f} MiB exceeds the 64 MiB bound")
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, arrays)
        arrays = {k: np.concatenate([p[k] for p in parts], axis=FRAME_AXIS[k]) if shard_frames else np.stack([p[k] for p in parts])
                  for k in arrays}
        if dist.get_rank() != 0:
            return
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(dirname, f"{k}.npy"), a)


def instrument(pipe, x0_dev, emb_src):
    """Extra (untimed) EAGER clip edit with CUDA events around every tap-GEMM and every ST-attention launch:
    returns dict(gemm=(algorithmic FLOPs, seconds, launches, algorithmic bytes), st_attn=(FLOPs, seconds, launches))."""
    from fatezero_b200 import ops
    rec, att = [], []
    stream = torch.cuda.current_stream()

    def timed(fn, on_done):
        def inner(*a, **k):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(stream)
            out = fn(*a, **k)
            e.record(stream)
            on_done(a, k, out, s, e)
            return out
        return inner

    def nbytes(*ts):
        return sum(t.numel() * t.element_size() for t in ts if t is not None)

    def on_gemm(a, k, out, s, e):
        M, K = a[0].shape
        N = a[1].shape[0]
        rec.append((2.0 * M * N * K, nbytes(a[0], a[1], out), s, e, ("gemm", M, N, K)))

    def on_conv(a, k, out, s, e):
        rows = out.numel() / out.shape[-1]
        co = 4 if a[1].shape[1] == 16 else a[1].shape[1]  # conv_out: 4 real output channels in a 16-wide tile
        rec.append((2.0 * rows * co * a[1].shape[2] * 9, nbytes(a[0], a[1], out), s, e, ("conv3x3", tuple(a[0].shape), a[1].shape[1])))

    def on_tconv(a, k, out, s, e):
        rows = out.numel() / out.shape[-1]
        rec.append((2.0 * rows * a[1].shape[1] * a[1].shape[2] * 3, nbytes(a[0], a[1], out), s, e, ("tconv3", tuple(a[0].shape), a[1].shape[1])))

    def on_attn(a, k, out, s, e):
        if k["keys_per_slot"] == 77:
            return  # text cross-attention
        T = len(k["src_index"]) * k["keys_per_slot"]
        att.append((4.0 * k["BF"] * k["heads"] * k["S_q"] * T * k["d"], s, e, (k["S_q"], T, k["d"], k.get("row_mode", 0))))

    saved = (ops.gemm, ops.conv3x3, ops.tconv3, ops.attention)
    ops.gemm, ops.conv3x3, ops.tconv3, ops.attention = (timed(ops.gemm, on_gemm), timed(ops.conv3x3, on_conv), timed(ops.tconv3, on_tconv),
                                                        timed(ops.attention, on_attn))
    mode = pipe.graph_mode
    pipe.graph_mode = "off"  # the instrumented pass needs the Python-level launches (a graph replay does not pass through ops.*)
    try:
        edit_clip(pipe, x0_dev, emb_src)
        torch.cuda.synchronize()
    finally:
        ops.gemm, ops.conv3x3, ops.tconv3, ops.attention = saved
        pipe.graph_mode = mode
    g_flops, g_bytes = sum(r[0] for r in rec), sum(r[1] for r in rec)
    g_secs = sum(r[2].elapsed_time(r[3]) for r in rec) / 1e3
    a_flops = sum(r[0] for r in att)
    a_secs = sum(r[1].elapsed_time(r[2]) for r in att) / 1e3
    if os.environ.get("FZ_SHAPE_REPORT"):
        agg = {}
        for fl, by, s, e, key in rec:
            d = agg.setdefault(str(key), [0, 0.0, 0.0])
            d[0] += 1
            d[1] += s.elapsed_time(e)
            d[2] += fl
        for fl, s, e, key in att:
            d = agg.setdefault("st_attn" + str(key), [0, 0.0, 0.0])
            d[0] += 1
            d[1] += s.elapsed_time(e)
            d[2] += fl
        rows = sorted(([k, v[0], v[1], v[2] / max(v[1], 1e-9) / 1e9] for k, v in agg.items()), key=lambda r: -r[2])
        with open(os.environ["FZ_SHAPE_REPORT"], "w") as f:
            json.dump([dict(shape=r[0], launches=r[1], ms_total=round(r[2], 2), tflops=round(r[3], 1)) for r in rows], f, indent=1)
    return dict(gemm=(g_flops, g_secs, len(rec), g_bytes), st_attn=(a_flops, a_secs, len(att)))


def vae_bracket(device, frames: int, px: int):
    """The VAE bracket of the path (SURVEY.md §8(f) rank 1), outside the headline metric like in SURVEY §8(d): encode `frames` RGB frames and
    decode `frames` latents with fatezero_b200.vae.VaeEngine (SD-1.x VAE geometry, synthetic weights), CUDA-event timed after a warm-up."""
    from fatezero_b200 import synth
    from fatezero_b200 import vae as fzvae
    cfg = dict(fzvae.SD14_VAE_CONFIG)
    eng = fzvae.VaeEngine(synth.synth_state_dict(dict(fzvae.vae_param_spec(cfg)), seed=3), cfg, device)
    img = (torch.rand(frames, 3, px, px, generator=torch.Generator().manual_seed(5)) * 2 - 1).to(device)
    z = torch.randn(frames, 4, px // 8, px // 8, generator=torch.Generator().manual_seed(6)).to(device)
    out = {}
    for name, fn in (("encode_ms", lambda: eng.encode_moments(img)), ("decode_ms", lambda: eng.decode(z))):
        fn()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        out[name] = round(s.elapsed_time(e), 2)
    out.update(frames=frames, resolution=f"{px}x{px}", note="AutoencoderKL geometry of SD-1.x on the tap-GEMM; not part of the frames/s metric")
    del eng
    torch.cuda.empty_cache()
    return out


def run_gpu(args):
    import torch.distributed as dist
    # stdout carries exactly ONE JSON line: libraries that print to fd 1 (NCCL's version banner) are redirected to stderr for the run
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    from fatezero_b200 import _lib, synth
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    FRAMES, SIZE = CFG["frames"], CFG["size"]
    # N > 1: the frames of ONE clip are split over the ranks (north_star split, strong scaling) with the SAME non-identity weights as N = 1:
    # K/V push, GroupNorm statistics exchange, temporal-conv halos and the temporal-attention frames<->pixels exchange run over peer
    # memory (fatezero_b200/csrc/fz_p2p.cu).  --shard clips = independent clips per rank (replicas, weak scaling).
    shard_frames = world > 1 and args.shard == "frames"
    if shard_frames and FRAMES % world:
        raise SystemExit(f"{FRAMES} frames do not split over {world} GPUs")
    pipe = build_pipe(device)
    if shard_frames:
        from fatezero_b200 import dist as fzdist
        pipe.unet.set_frame_shard(rank, world)
        x_full = synth.synth_latents(FRAMES, SIZE, SIZE, seed=1) * 0.5
        x0_host = fzdist.frame_slice(x_full, rank, world).pin_memory()
    else:
        x0_host = (synth.synth_latents(FRAMES, SIZE, SIZE, seed=1 + rank) * 0.5).pin_memory()
    if args.graphs == "off" or (CFG["name"] == "long24" and world < 2):
        pipe.graph_mode = "off"  # 24 frames on one GPU: 109 GiB of maps, no room for an eager copy next to the graph pool
    out_host = torch.empty_like(x0_host).pin_memory()
    x0_dev = x0_host.to(device)
    emb_src = pipe._encode_prompt(SRC, device, 1, True, None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_ms = []

    def timed(fn, n):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(n):
            t0 = time.perf_counter()
            fn()
            host_ms.append((time.perf_counter() - t0) * 1e3)
        e.record()
        barrier()
        ms = s.elapsed_time(e)
        if world > 1:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    last = {}

    def step_resident():
        last["inv"], last["out"] = edit_clip(pipe, x0_dev, emb_src)

    def step_e2e():
        xd = x0_host.to(device, non_blocking=True)
        _, out = edit_clip(pipe, xd, emb_src)
        out_host.copy_(out["sdimage_output"].images.float(), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    # W >= 3 (timing rule); with cuda_graphs=auto the first clip runs eagerly, the second is captured, the third is the first pure replay
    args.warmup = max(args.warmup, 3)
    for _ in range(args.warmup):
        step_resident()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.kernel_launches
    host_ms.clear()
    ms = timed(step_resident, args.steps)
    launches = _lib.kernel_launches - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:  # before the next pass reuses the buffers (graph replays write the same masks in place)
        dump_outputs(args.dump_outputs, last["inv"], last["out"], world, shard_frames)
    last.clear()
    ms_e2e = timed(step_e2e, args.steps)
    frames_total = FRAMES * (1 if (shard_frames or world == 1) else world) * args.steps
    value = frames_total / (ms / 1e3)
    e2e_value = frames_total / (ms_e2e / 1e3)
    pk, pk_kind = peaks()
    roof = cpu = st = None
    inst = None
    if not args.no_instrument:
        if shard_frames and rank != 0:
            instrument(pipe, x0_dev, emb_src)  # the sharded forward exchanges with every rank: all of them run the instrumented clip
        if rank == 0:
            inst = instrument(pipe, x0_dev, emb_src)
    if rank == 0 and inst is not None:
        flops, secs, n_launch, abytes = inst["gemm"]
        peak = float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops", 1400.0)))
        ach = flops / secs / 1e12
        # DRAM bytes per tap-GEMM launch from the committed ncu capture of one step pair of THIS round, if present
        traffic = traffic_src = None
        for cand in ("r02_tapgemm_traffic.json",):
            try:
                tj = json.load(open(os.path.join(ROOT, "profiles", cand)))
                traffic, traffic_src = round(tj["tapgemm_dram_bytes_per_launch"]), f"profiles/{cand}: {tj.get('how', 'ncu dram__bytes_read+write per launch')}"
                break
            except Exception:  # noqa: BLE001
                pass
        roof = dict(kernel="tapgemm_kernel (conv3x3 / linear / temporal-LoRA, tcgen05)", bound="tensor", achieved=round(ach, 1), peak=peak,
                    unit="TFLOP/s", frac=round(ach / peak, 4), traffic=traffic, traffic_source=traffic_src,
                    algorithmic_bytes_per_launch=round(abytes / max(n_launch, 1)), peak_source=f"{pk_kind} sustained bf16 (MEASURED_PEAKS.json)",
                    launches_per_clip=n_launch, algorithmic_tflop_per_clip=round(flops / 1e12, 1),
                    kernel_seconds_per_clip=round(secs, 4), share_of_step=round(secs / (ms / 1e3 / args.steps), 3),
                    how="CUDA events around every launch of an extra eager clip (per rank: this rank's frames)")
        af, asec, an = inst["st_attn"]
        st = dict(value=round(af / max(asec, 1e-9) / 1e12, 1), unit="TFLOP/s", launches_per_clip=an, algorithmic_tflop_per_clip=round(af / 1e12, 1),
                  kernel_seconds_per_clip=round(asec, 4), share_of_step=round(asec / (ms / 1e3 / args.steps), 3),
                  definition="sum over ST-attn launches of 4*BF*heads*S*T*d / sum of their CUDA-event durations (rank 0's frames)")
    vae_line = None
    if rank == 0 and not args.no_instrument:
        vae_line = vae_bracket(device, FRAMES, 8 * SIZE)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_sample()
    if rank == 0:
        par = ("single GPU" if world == 1 else
               (f"frames of ONE clip over {world} GPUs ({FRAMES // world} per GPU): peer-memory push/flag exchange over NVLink (K/V, GroupNorm "
                f"statistics, temporal-conv halos, temporal-attention frames<->pixels); NCCL only for the timing all-reduce" if shard_frames
                else f"{world} independent clips (replicas)"))
        line = dict(metric="edited frames/sec (512x512x8f, 50 DDIM steps: inversion + attention-fused edit)", value=round(value, 4),
                    unit="frames/s", n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=round(ms / args.steps, 2),
                    higher_is_better=True, scaling=("strong" if shard_frames else "weak"), vs_baseline=None, dtype="f16 (fp32 accumulate)",
                    data="synthetic",
                    config=dict(workload=CFG["workload"], name=CFG["name"], frames=FRAMES, latent=f"{SIZE}x{SIZE}", ddim_steps=DDIM_STEPS,
                                model_config=CFG["model_config"], parallelism=par, cuda_graphs=pipe.graph_mode,
                                l2="working set (map cache of the clip + activations) far exceeds the 126 MB L2; no explicit flush"),
                    clocks=clocks, e2e=dict(value=round(e2e_value, 4), unit="frames/s", h2d_bytes_per_step=x0_host.numel() * 4,
                                            d2h_bytes_per_step=out_host.numel() * 4),
                    gpu_launches=int(launches), st_attn_tflops=st, vae=vae_line, roofline=roof,
                    cpu_baseline=cpu)
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------
# CPU arm (the oracle port of the reference on the host cores)
# ------------------------------------------------------------------------------------------------------------------
def cpu_sample_seconds(frames: int):
    """One inversion step (STORE) + one CFG edit step (INJECT) of the configured workload on `frames` frames, fp32, all host threads."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from fatezero_b200 import synth
    from fatezero_b200.unet import unet_param_spec
    from oracle import fz_oracle as fo
    cfg = synth.SD14_UNET_CONFIG
    mc = CFG["model_config"]
    spec = unet_param_spec(dict(cfg), mc)
    ou = fo.OracleUNet(synth.synth_state_dict({k: v[0] for k, v in spec.items()}), cfg, mc)
    tok, te = synth.ToyTokenizer(), synth.ToyTextEncoder(cfg["cross_attention_dim"])
    emb_src, emb_tgt = fo.encode_prompts(tok, te, SRC), fo.encode_prompts(tok, te, CFG["tgt"])
    x0 = synth.synth_latents(frames, CFG["size"], CFG["size"]) * 0.5
    p = CFG["p2p"]
    t0 = time.perf_counter()
    store = fo.OracleStore()
    inv = fo.invert(ou, x0, emb_src[1:], 1, store)
    t1 = time.perf_counter()
    plan = fo.EditPlan(tok, SRC, CFG["tgt"], 1, p["cross_replace_steps"], 1.0, p.get("is_replace_controller", True), p.get("eq_params"))
    ctrl = fo.OracleEdit(plan, store)
    fo.edit(ou, inv[-1], emb_tgt, 1, ctrl)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1


def cpu_threads() -> int:
    """Thread count for the CPU arm: PyTorch's CPU kernels stop scaling (and regress) far below the core count of a 128-core GPU host
    (measured: 222 s per sample with 128 threads vs 14 s with 8), so the arm uses the best of a small sweep's range: min(cores, 32)."""
    return max(1, min(os.cpu_count() or 1, int(os.environ.get("FZ_CPU_THREADS", "32"))))


def cpu_baseline_sample():
    """Bounded in-line sample of the GPU arm (N = 1): 2 of the clip's frames, one DDIM step pair."""
    cores = cpu_threads()
    torch.set_num_threads(cores)
    nf = 2
    t_inv, t_edit = cpu_sample_seconds(nf)
    per_frame_pair = (t_inv + t_edit) / nf
    value = 1.0 / (DDIM_STEPS * per_frame_pair)
    return dict(value=round(value, 6), unit="frames/s", cores=cores, kind="port",
                sample=f"1 of 50 DDIM step pairs (inversion STORE step + CFG edit INJECT step) on {nf} of {CFG['frames']} frames, fp32, {cores} threads; "
                       f"measured {t_inv:.1f}s + {t_edit:.1f}s, scaled linearly in frames and steps (the reference arm times the full-frame step pair)")


def run_reference(args):
    """Reference arm: the oracle port of the reference (the Python reference cannot travel: DESIGN.md §7) on the host cores.  One step =
    ONE FULL step pair of the workload (all frames: inversion STORE step + CFG edit INJECT step), i.e. 1/50 of a clip; frames/s follows."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = cpu_threads()
    torch.set_num_threads(cores)
    F = int(os.environ.get("FZ_REF_FRAMES", CFG["frames"]))  # fewer frames than the clip: a quick check of the arm, not its number
    warmup = min(args.warmup, 1)  # at most one untimed pass: every pass costs the better part of a minute
    for _ in range(warmup):
        cpu_sample_seconds(F)
    times = [sum(cpu_sample_seconds(F)) for _ in range(args.steps)]
    pair = sum(times) / len(times)
    value = F / (DDIM_STEPS * pair)  # frames/s of the sampled frames (== the clip's when F is the clip length)
    sample = (f"each step = 1 of 50 DDIM step pairs on all {F} frames (oracle port of the reference, fp32, {cores} threads), "
              f"{len(times)} timed after {warmup} untimed; scaled linearly in steps only")
    line = dict(impl="reference", metric="edited frames/sec (512x512x8f, 50 DDIM steps: inversion + attention-fused edit)",
                value=round(value, 6), unit="frames/s", n_gpus=int(os.environ.get("WORLD_SIZE", "1")), steps=len(times), warmup=warmup,
                ms_per_step=round(pair * 1e3 * DDIM_STEPS, 1), higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f32",
                data="synthetic", config=dict(workload=CFG["workload"], name=CFG["name"], frames=F, latent=f"{CFG['size']}x{CFG['size']}",
                                             ddim_steps=DDIM_STEPS, model_config=CFG["model_config"]),
                cpu_baseline=dict(value=round(value, 6), unit="frames/s", cores=cores, kind="port", sample=sample),
                e2e=dict(value=round(value, 6), unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3,
                    help="timed steps; a step is one full clip edit (50 inversion + 50 edit DDIM steps) in the GPU arm, one DDIM step pair "
                         "(inversion + edit) on all frames in the reference arm")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="style", choices=sorted(CONFIGS), help="BASELINE.json configs #2..#5 (default: the metric's own)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-instrument", action="store_true", help="skip the extra instrumented clip (roofline / ST-attn TFLOPS)")
    ap.add_argument("--graphs", default="auto", choices=["auto", "off"])
    ap.add_argument("--shard", default="frames", choices=["clips", "frames"],
                    help="N > 1: the frames of ONE clip over the ranks (default, strong scaling) or independent clips per rank (replicas)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs")
    select_config(args.config)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
