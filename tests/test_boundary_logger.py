"""Drop-in boundary (SURVEY.md §8(b)): the reference's UNCHANGED `P2pSampleLogger.log_sample_images`
(video_diffusion/pipelines/p2p_validation_loop.py:68-131) must be able to drive this repo's pipeline.

Two halves:
  * CPU: the reference's logger, imported THROUGH this repo's `video_diffusion` alias package (modules the alias does not provide fall
    through to the reference tree), ran `log_sample_images` against a recording pipeline (oracle/make_ref_pins.py, pinned in
    tests/golden/ref_logger.json.gz); every recorded call must bind to the signature of our `sd_ddim_pipeline` / `make_controller`, and
    the alias must still fall through for modules it does not provide;
  * GPU: the same call sequence (kwargs as recorded there, cited line by line) against the real CUDA pipeline with stub VAE / tokenizer."""
import gzip
import inspect
import json
import os
import sys

import numpy as np
import pytest
import torch

from _helpers import ROOT, build_product
from fatezero_b200 import synth
from oracle.cases import LOGGER_EDITS as EDITS, LOGGER_P2P as P2P, SRC



def logger_kwargs(idx, prompt, image, latents, save_dir, steps, clip_length):
    """The keyword arguments of the pipeline call in p2p_validation_loop.py:112-131 (use_inversion_attention=True => edit_type 'swap', :99-104)."""
    cfg = dict(P2P[idx])
    cfg.update({"save_self_attention": False, "use_inversion_attention": True})
    return dict(prompt=prompt, source_prompt=SRC, edit_type="swap", image=image, strength=None, generator=torch.Generator(device="cpu").manual_seed(0),
                num_inference_steps=steps, clip_length=clip_length, guidance_scale=7.5, num_images_per_prompt=1, latents=latents,
                uncond_embeddings_list=None, save_path=save_dir, **cfg)


def _replay(v, save_dir):
    """A recorded keyword value of ref_logger.json.gz back as the object the reference logger passed."""
    if isinstance(v, dict) and "__tensor__" in v:
        return torch.zeros(v["__tensor__"])
    if isinstance(v, dict) and "__generator__" in v:
        return torch.Generator(device=v["__generator__"]).manual_seed(0)
    if isinstance(v, dict) and "__save_dir__" in v:
        return save_dir
    return v


def test_unchanged_reference_logger_binds_to_our_pipeline(tmp_path):
    """The pipeline calls of the reference's log_sample_images (pinned by `python -m oracle.make_ref_pins ref_logger`) bind to our
    pipeline and make_controller, and the alias package still lets the reference's own modules (the logger among them) fall through."""
    fake = tmp_path / "ref" / "video_diffusion" / "pipelines"
    fake.mkdir(parents=True)
    (fake / "p2p_validation_loop.py").write_text("P2pSampleLogger = 'reference logger'\n")
    code = r'''
import sys
sys.path.insert(0, %(root)r); sys.path.append(%(ref)r)
import video_diffusion                                        # THIS repo's alias package ...
import video_diffusion.pipelines.p2p_validation_loop as m    # ... falling through to the reference's own file
assert m.__file__.startswith(%(ref)r), m.__file__
from video_diffusion.pipelines.p2p_ddim_spatial_temporal import P2pDDIMSpatioTemporalPipeline as Ours
assert Ours.__module__ == "fatezero_b200.pipeline", Ours.__module__
print("OK")
''' % dict(root=ROOT, ref=str(tmp_path / "ref"))
    import subprocess
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout[-1500:] + r.stderr[-3000:]

    from fatezero_b200 import P2pDDIMSpatioTemporalPipeline as Ours
    from fatezero_b200 import controllers
    g = json.load(gzip.open(os.path.join(ROOT, "tests", "golden", "ref_logger.json.gz")))
    calls = [{k: _replay(v, str(tmp_path)) for k, v in kw.items()} for kw in g["calls"]]
    assert len(calls) == 2
    sig_call = inspect.signature(Ours.sd_ddim_pipeline)
    mk = inspect.signature(controllers.make_controller)
    for kw in calls:
        assert kw["edit_type"] == "swap" and kw["use_inversion_attention"] is True and kw["save_self_attention"] is False
        sig_call.bind(None, controller=None, **kw)     # **args swallows what sd_ddim_pipeline does not name (p2p_ddim_spatial_temporal.py:280)
        # p2preplace_edit (p2p_ddim_spatial_temporal.py:172-222) forwards these keys to make_controller under these names
        mk.bind(None, [kw["source_prompt"], kw["prompt"]], NUM_DDIM_STEPS=kw["num_inference_steps"], is_replace_controller=kw.get("is_replace_controller", True),
                cross_replace_steps=kw["cross_replace_steps"], self_replace_steps=kw["self_replace_steps"], blend_words=kw.get("blend_words"),
                equilizer_params=kw.get("eq_params"), additional_attention_store=None, use_inversion_attention=kw["use_inversion_attention"],
                blend_th=kw.get("blend_th", (0.3, 0.3)), blend_self_attention=kw.get("blend_self_attention"), blend_latents=kw.get("blend_latents"),
                save_path=kw.get("save_path"), save_self_attention=kw.get("save_self_attention", True), disk_store=kw.get("disk_store", False))
    recorded = set(calls[1].keys())
    mine = set(logger_kwargs(1, EDITS[1], None, None, None, 3, 2).keys())
    assert recorded == mine, (recorded ^ mine)   # the GPU half below replays exactly the keyword set the reference logger sends


@pytest.mark.gpu
def test_logger_flow_on_the_cuda_pipeline(tmp_path, report):
    """log_sample_images' call sequence (inversion once, then every editing prompt against the stored maps) on the CUDA pipeline."""
    mc = dict(lora=160, SparseCausalAttention_index=["mid"], least_sc_channel=128)
    pipe = build_product("mini", mc)
    steps, F, size = 3, 2, 32
    pipe.scheduler.set_timesteps(steps)
    pipe.set_progress_bar_config(disable=True)
    dev = pipe.unet.device

    class Vae(synth.VaeStub):  # encode(): the latent-level stand-in of AutoencoderKL.encode (test_fatezero.py:211-222 path)
        def encode(self, x):
            lat = torch.nn.functional.avg_pool2d(x.float(), 8)
            lat = torch.cat([lat, lat[:, :1]], 1)
            return type("O", (), {"latent_dist": type("D", (), {"sample": staticmethod(lambda g=None: lat)})()})()
    pipe.vae = Vae().to(dev)
    images = (torch.rand(F, 3, 8 * size, 8 * size, generator=torch.Generator().manual_seed(3)) * 2 - 1).to(dev)
    emb = pipe._encode_prompt(SRC, dev, 1, True, None)
    # test_fatezero.py:211-222: inversion with the attention store
    lat_all = pipe.prepare_latents_ddim_inverted(images, batch_size=1, num_images_per_prompt=1, text_embeddings=emb, prompt=SRC, store_attention=True,
                                                 LOW_RESOURCE=True, save_path=None)
    assert len(lat_all) == steps + 1 and lat_all[-1].shape == (1, 4, F, size, size)
    assert len(pipe.store_controller.attention_store_all_step) == steps
    outs = []
    for idx, prompt in enumerate(EDITS):
        ret = pipe(**logger_kwargs(idx, prompt, images, lat_all[-1], None, steps, F))
        seq = ret["sdimage_output"].images[0]               # p2p_validation_loop.py:133
        assert len(seq) == F and seq[0].size == (8 * size, 8 * size)
        assert ret["attention_output"] is None or isinstance(ret["attention_output"], list)
        outs.append(np.stack([np.asarray(im) for im in seq]))
    assert np.isfinite(outs[0].astype(np.float32)).all() and (outs[0] != outs[1]).any()
    report["logger_flow"] = dict(frames=F, steps=steps, edits=len(outs), diff=float(np.abs(outs[0].astype(np.float32) - outs[1]).mean()))
