"""CPU-side checks: the C-ABI library loads and exports every declared symbol, the parameter spec equals the reference's state dict,
the reference-facing surface exists and refuses to run without CUDA, and the N>1 plumbing works under gloo (world_size 2)."""
import gzip
import json
import os
import re
import subprocess
import sys

import pytest
import torch

from _helpers import ROOT


def test_library_exports_every_header_symbol():
    from fatezero_b200 import _lib
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "fatezero_b200.h")).read()
    syms = sorted(set(re.findall(r"\b(fz_[a-z0-9_]+)\s*\(", hdr)))
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in the header but not exported"
        assert s in _lib.SIGNATURES or s == "fz_last_error"
    assert lib.fz_version() >= 100


def test_no_compute_without_cuda():
    """The product path fails loudly without a GPU (no CPU fallback)."""
    from fatezero_b200 import UNetPseudo3DConditionModel, synth
    unet = UNetPseudo3DConditionModel(**synth.MINI_UNET_CONFIG, lora=160)
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(RuntimeError, match="CUDA"):
        unet(torch.zeros(1, 4, 2, 16, 16), 10, torch.zeros(1, 77, 128))


def test_spec_counts():
    from fatezero_b200 import synth
    from fatezero_b200.unet import unet_param_spec
    spec = unet_param_spec(dict(synth.SD14_UNET_CONFIG), dict(synth.DEFAULT_MODEL_CONFIG))
    assert len(spec) == 902
    n = sum(int(torch.tensor(v[0]).prod()) for v in spec.values())
    assert abs(n - 953.36e6) < 0.01e6
    spec2 = unet_param_spec(dict(synth.SD14_UNET_CONFIG), {})  # no lora: full temporal convs (SURVEY App. E3: 1 060 M params)
    n2 = sum(int(torch.tensor(v[0]).prod()) for v in spec2.values())
    assert abs(n2 - 1060e6) < 2e6


def test_spec_equals_reference_state_dict():
    """unet_param_spec == the reference UNet's state dict (names and shapes, pinned by `python -m oracle.make_ref_pins ref_unet_spec`)."""
    from fatezero_b200 import synth
    from fatezero_b200.unet import unet_param_spec
    g = json.load(gzip.open(os.path.join(ROOT, "tests", "golden", "ref_unet_spec.json.gz")))
    assert g["unet_config"] == json.loads(json.dumps(synth.MINI_UNET_CONFIG))
    assert [c["model_config"] for c in g["configs"]] == [dict(lora=160, SparseCausalAttention_index=["mid"], least_sc_channel=128), {},
                                                         dict(lora=8)]
    for c in g["configs"]:
        ref = c["shapes"]
        spec = unet_param_spec(dict(synth.MINI_UNET_CONFIG), c["model_config"])
        assert set(ref.keys()) == set(spec.keys()), (set(ref) ^ set(spec))  # module registration order differs, names do not
        for k, v in ref.items():
            assert tuple(v) == tuple(spec[k][0]), k


def test_alias_package_paths():
    """The reference's dotted import paths (YAML `target:` strings, test_fatezero.py:24-30) resolve to the B200 classes."""
    code = ("import video_diffusion.pipelines.p2p_ddim_spatial_temporal as p, video_diffusion.prompt_attention.attention_util as a, "
            "video_diffusion.models.unet_3d_condition as u, video_diffusion.prompt_attention.spatial_blend as sb; "
            "import fatezero_b200 as f; assert p.P2pDDIMSpatioTemporalPipeline is f.P2pDDIMSpatioTemporalPipeline; "
            "assert a.make_controller is f.make_controller and a.AttentionStore is f.AttentionStore; "
            "assert u.UNetPseudo3DConditionModel is f.UNetPseudo3DConditionModel and sb.SpatialBlender is f.SpatialBlender; print('OK')")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert out.returncode == 0 and "OK" in out.stdout, out.stderr[-2000:]


def test_pipeline_surface_and_errors(tmp_path):
    from fatezero_b200 import DDIMScheduler, P2pDDIMSpatioTemporalPipeline, UNetPseudo3DConditionModel, controllers, synth
    unet = UNetPseudo3DConditionModel(**synth.MINI_UNET_CONFIG, lora=160)
    pipe = P2pDDIMSpatioTemporalPipeline(synth.VaeStub(), synth.ToyTextEncoder(128), synth.ToyTokenizer(), unet, DDIMScheduler(steps_offset=0, clip_sample=True))
    assert pipe.scheduler.config.steps_offset == 1 and pipe.scheduler.config.clip_sample is False  # stable_diffusion.py:56-81
    assert pipe.vae_scale_factor == 8
    pipe.scheduler.set_timesteps(50)
    assert [int(t) for t in pipe.scheduler.timesteps[:3]] == [981, 961, 941] and int(pipe.scheduler.timesteps[-1]) == 1
    emb = pipe._encode_prompt("a jeep", torch.device("cpu"), 1, True, None)
    assert emb.shape == (2, 77, 128)
    with pytest.raises(ValueError):
        pipe.check_inputs(3, 512, 512, 1)
    with pytest.raises(ValueError):
        pipe.check_inputs("x", 500, 512, 1)
    with pytest.raises(AssertionError):
        pipe(edit_type="bogus")
    n = controllers.register_attention_control(pipe, pipe.store_controller)
    assert n == 32 and pipe.store_controller.num_att_layers == 32  # 16 transformers x (self, cross)
    import numpy as np
    pil = pipe.numpy_to_pil(np.zeros((1, 2, 8, 8, 3), dtype=np.float32))
    assert len(pil) == 1 and len(pil[0]) == 2
    with pytest.raises(ValueError):  # Replace controller needs equal word counts (seq_aligner.py:155-157)
        controllers.make_controller(synth.ToyTokenizer(), ["a b c", "a b c d"], True, {"default_": 0.8}, 0.5, NUM_DDIM_STEPS=10,
                                    additional_attention_store=controllers.AttentionStore())
    with pytest.raises(TypeError):  # blend words need save_path (attention_util.py:339)
        controllers.make_controller(synth.ToyTokenizer(), ["a b c", "a b d"], True, {"default_": 0.8}, 0.5, NUM_DDIM_STEPS=10,
                                    blend_words=[["c"], ["d"]], blend_self_attention=True,
                                    additional_attention_store=controllers.AttentionStore())


def _gloo_worker(rank, world, port, q):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    from fatezero_b200 import dist as fzd
    r, w = fzd.init("gloo")
    fzd.barrier()
    mx = fzd.max_over_ranks(10.0 + 5 * rank, torch.device("cpu"))
    frames = fzd.shard_frames(8, w, r)
    clips = fzd.shard_clips(5, w, r)
    import torch.distributed as dist
    # the exchange pattern of the frame-sharded path: all-gather of per-rank K/V blocks + a SUM all-reduce of GroupNorm partial statistics
    kv = torch.full((len(frames), 3), float(r))
    gathered = [torch.zeros_like(kv) for _ in range(w)]
    dist.all_gather(gathered, kv)
    stats = torch.tensor([1.0 + r, 2.0 * (1 + r)], dtype=torch.float64)
    dist.all_reduce(stats)
    q.put((r, mx, frames, clips, torch.cat(gathered).sum().item(), stats.tolist()))
    dist.destroy_process_group()


def test_gloo_world_size_2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 500)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert res[0][1] == 15.0 and res[1][1] == 15.0            # max over ranks
    assert res[0][2] == [0, 1, 2, 3] and res[1][2] == [4, 5, 6, 7]
    assert res[0][3] == [0, 2, 4] and res[1][3] == [1, 3]
    assert res[0][4] == 12.0 and res[0][5] == [3.0, 6.0]


def _shard_worker(rank, world, port, q):
    """Frame-sharded exchange logic on CPU tensors (gloo): the all-gathered K rows picked through gathered_source_rows and the
    all-reduced GroupNorm sums must equal what the unsharded clip computes."""
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    from fatezero_b200 import dist as fzd
    from fatezero_b200.engine import sc_frame_indices
    fzd.init("gloo")
    B, F, S, C, G = 2, 6, 5, 4, 2
    Fl = F // world
    g = torch.Generator().manual_seed(0)
    k_full = torch.randn(B, F, S, C, generator=g)          # K of the whole clip, (b f) order like the engine
    x_full = torch.randn(B, F, 7, G * 3, generator=g)      # activations for the GroupNorm statistics
    frames = fzd.shard_frames(F, world, rank)
    k_loc = k_full[:, frames].reshape(B * Fl * S, C).contiguous()
    gathered = torch.empty(world * B * Fl * S, C)
    dist.all_gather_into_tensor(gathered, k_loc)
    ok = True
    for index in (["mid"], [-1, "first"], [1, "last"]):
        for fi in sc_frame_indices(index, F):
            rows = fzd.gathered_source_rows(fi, rank, world, Fl, B)
            i = 0
            for b in range(B):
                for f in range(Fl):
                    want = k_full[b, fi[rank * Fl + f]]
                    got = gathered.view(world * B * Fl, S, C)[rows[i]]
                    ok = ok and torch.equal(want, got)
                    i += 1
    xl = x_full[:, frames].reshape(B * Fl, 7, G, 3)
    image_sums = torch.stack([xl.sum((1, 3)), (xl * xl).sum((1, 3))], -1)      # [B*Fl, G, 2]
    s = fzd.allreduce_set_sums(image_sums.contiguous(), Fl)
    xf = x_full.reshape(B, F * 7, G, 3)
    want = torch.stack([xf.sum((1, 3)), (xf * xf).sum((1, 3))], -1)
    ok = ok and torch.allclose(s, want, rtol=1e-5, atol=1e-5)
    sl = fzd.frame_slice(x_full.permute(0, 3, 1, 2), rank, world, dim=2)       # [B, C, F, H] style tensor
    back = fzd.gather_frames(sl, world, dim=2)
    ok = ok and torch.equal(back, x_full.permute(0, 3, 1, 2))
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_frame_shard_exchange_gloo_world_size_2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29100 + (os.getpid() % 500)
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert res == [(0, True), (1, True)]


def test_vae_spec_is_the_published_sd_vae():
    """The AutoencoderKL layout the VAE engine expects: 248 tensors, 83 653 863 parameters (the SD-1.x VAE) — the one fact about diffusers'
    model that can be checked without the package (DESIGN.md §5: the VAE restatement is otherwise unpinned)."""
    from fatezero_b200 import vae
    spec = vae.vae_param_spec(vae.SD14_VAE_CONFIG)
    assert len(spec) == 248
    assert sum(int(torch.tensor(v).prod()) for v in spec.values()) == 83_653_863
    assert spec["encoder.mid_block.attentions.0.query.weight"] == (512, 512) and spec["quant_conv.weight"] == (8, 8, 1, 1)


def test_disk_store_hands_out_paths_and_releases(tmp_path, monkeypatch):
    """attention_store.py:103-106: with disk_store the per-step dict goes to a .pt file and the list holds its PATH (the maps are not kept)."""
    from fatezero_b200 import controllers
    monkeypatch.chdir(tmp_path)
    s = controllers.AttentionStore(disk_store=True)
    m = torch.rand(2, 8, 16, 80).half()
    s.step_store["down_cross"].append(m[..., :77])
    s.cur_step = 1
    s.between_steps()
    assert isinstance(s.attention_store_all_step[0], str) and s.attention_store_paths == s.attention_store_all_step
    loaded = torch.load(s.attention_store_all_step[0])
    assert torch.equal(loaded["down_cross"][0], m[..., :77]) and s.step_store == s.get_empty_store()
    assert s.graph_signature() is None  # disk-backed stores always take the eager loops


def test_controller_state_adoption():
    """graphs.py: after a replay the caller's fresh controller adopts the captured controller's end-of-loop state (shallow list copies of
    the same slabs), so mutating one object's lists never changes the other's."""
    from fatezero_b200 import controllers
    a, b = controllers.AttentionStore(), controllers.AttentionStore()
    assert b.is_pristine() and b.graph_signature() == ("store", True, False)
    a.cur_step = 3
    a.attention_store_all_step = [{"down_cross": [torch.zeros(1)]}] * 3
    a.latents_store = [torch.zeros(1)] * 3
    a._acc = {"down_cross": [torch.ones(1)]}
    a._graph_plan_id = 42
    b.adopt_from(a)
    assert b.cur_step == 3 and b._graph_plan_id == 42 and not b.is_pristine()
    assert b.attention_store_all_step is not a.attention_store_all_step and b.attention_store_all_step[0] is a.attention_store_all_step[0]
    b.latents_store.append(torch.zeros(1))
    assert len(a.latents_store) == 3 and b._acc["down_cross"][0] is a._acc["down_cross"][0] and b._acc["down_cross"] is not a._acc["down_cross"]
