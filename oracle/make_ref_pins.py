"""Generate the small gzipped JSON pins tests/golden/ref_*.json.gz by running pieces of the UNMODIFIED reference (needs a checkout of
it, see REFERENCE_ROOT in oracle/ref_harness.py; the tests read only the pins).  Usage: python -m oracle.make_ref_pins [pin ...]; each
pin runs in its own interpreter because the tables and spec pins import the reference's `video_diffusion` package while the logger pin
imports this repo's alias of it.

  ref_unet_spec   state-dict names and shapes of the reference UNet (mini geometry, three model configs)  -> tests/test_cpu_misc.py
  ref_tables_clip edit tables of ptp_utils / seq_aligner with the real CLIP BPE, plus every encode / decode
                  answer of that tokenizer the tables need (the BPE vocabulary itself is not stored)      -> tests/test_tables.py
  ref_logger      keyword arguments P2pSampleLogger.log_sample_images passes to the pipeline              -> tests/test_boundary_logger.py
"""
import gzip
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

from oracle import ref_harness as rh  # noqa: E402

SPEC_MODEL_CONFIGS = [dict(lora=160, SparseCausalAttention_index=["mid"], least_sc_channel=128), dict(), dict(lora=8)]


def _write(name, obj):
    path = os.path.join(GOLDEN, f"{name}.json.gz")
    with open(path, "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as f:  # mtime=0: same pin, same bytes
        f.write(json.dumps(obj, separators=(",", ":"), sort_keys=True).encode())
    print(name, "->", path, f"{os.path.getsize(path) / 1e3:.1f} kB")


def table(t):
    return dict(dtype=str(t.dtype).replace("torch.", ""), data=t.tolist())


def pin_ref_unet_spec():
    rh._prepare_imports()
    from video_diffusion.models.unet_3d_condition import UNetPseudo3DConditionModel as Ref
    from fatezero_b200 import synth
    out = []
    for mc in SPEC_MODEL_CONFIGS:
        sd = Ref(**synth.MINI_UNET_CONFIG, **mc).state_dict()
        out.append(dict(model_config=mc, shapes={k: list(v.shape) for k, v in sd.items()}))
    _write("ref_unet_spec", dict(unet_config=synth.MINI_UNET_CONFIG, configs=out))


def clip_tokenizer():
    """transformers' CLIPTokenizer over the reference's own BPE merges (CLIP/clip/bpe_simple_vocab_16e6.txt.gz), vocabulary built the
    way CLIP's SimpleTokenizer builds it."""
    from transformers import CLIPTokenizer
    bpe = os.path.join(rh.REFERENCE_ROOT, "CLIP", "clip", "bpe_simple_vocab_16e6.txt.gz")
    lines = gzip.open(bpe).read().decode("utf-8").split("\n")
    merges = [tuple(m.split()) for m in lines[1:49152 - 256 - 2 + 1]]
    bs = list(range(ord("!"), ord("~") + 1)) + list(range(ord("\xa1"), ord("\xac") + 1)) + list(range(ord("\xae"), ord("\xff") + 1))
    cs = bs[:]
    n = 0
    for b in range(2 ** 8):
        if b not in bs:
            bs.append(b)
            cs.append(2 ** 8 + n)
            n += 1
    vocab = [chr(c) for c in cs]
    vocab = vocab + [v + "</w>" for v in vocab]
    vocab += ["".join(m) for m in merges] + ["<|startoftext|>", "<|endoftext|>"]
    tok = CLIPTokenizer(vocab=dict(zip(vocab, range(len(vocab)))), merges=merges, model_max_length=77)
    assert tok.encode("a")[1] == 320 and tok.encode("a")[0] == 49406
    return tok


class RecordingTokenizer:
    """Passes encode / decode through to a real tokenizer and keeps every answer."""

    def __init__(self, tok):
        self.tok, self.encoded, self.decoded = tok, {}, {}

    def encode(self, text):
        ids = self.encoded[text] = list(self.tok.encode(text))
        return ids

    def decode(self, ids):
        assert len(ids) == 1, ids
        s = self.decoded[str(int(ids[0]))] = self.tok.decode(ids)
        return s


def pin_ref_tables_clip():
    rh._prepare_imports()
    import video_diffusion.prompt_attention.ptp_utils as rp
    import video_diffusion.prompt_attention.seq_aligner as rs
    from oracle.cases import PROMPT_PAIRS
    tok = RecordingTokenizer(clip_tokenizer())
    cases = []
    for src, tgt in PROMPT_PAIRS:
        crs = {"default_": 0.8, tgt.split(" ")[1]: 0.3}
        mapper, alphas = rs.get_refinement_mapper([src, tgt], tok)
        c = dict(source=src, target=tgt, cross_replace_steps=crs, num_steps=50,
                 alpha=table(rp.get_time_words_attention_alpha([src, tgt], 50, dict(crs), tok)),
                 refinement_mapper=table(mapper), refinement_alphas=table(alphas),
                 word_inds={w: [int(i) for i in rp.get_word_inds(tgt, w, tok)] for w in tgt.split(" ")})
        if len(src.split(" ")) == len(tgt.split(" ")):
            c["replacement_mapper"] = table(rs.get_replacement_mapper([src, tgt], tok))
        cases.append(c)
    _write("ref_tables_clip", dict(cases=cases, tokenizer=dict(encode=tok.encoded, decode=tok.decoded)))


def pin_ref_logger():
    """The reference's unchanged P2pSampleLogger (imported through this repo's alias package, which falls through to the reference for
    modules it does not provide) drives a pipeline that records its keyword arguments."""
    import types
    import numpy as np
    import torch
    from PIL import Image
    sys.path.insert(0, os.path.join(ROOT, "oracle", "shim"))
    sys.path.append(rh.REFERENCE_ROOT)
    import video_diffusion  # noqa: F401  (this repo's alias package)
    import video_diffusion.pipelines.p2p_validation_loop as m
    from video_diffusion.pipelines.p2p_validation_loop import P2pSampleLogger
    assert m.__file__.startswith(rh.REFERENCE_ROOT), m.__file__
    from fatezero_b200 import P2pDDIMSpatioTemporalPipeline as Ours
    from oracle.cases import LOGGER_EDITS, LOGGER_P2P, SRC

    calls = []

    class Recorder:
        @staticmethod
        def numpy_to_pil(x):
            return Ours.numpy_to_pil(x)

        def __call__(self, **kw):
            calls.append(kw)
            frames = [Image.fromarray(np.zeros((16, 16, 3), np.uint8)) for _ in range(2)]
            return {"sdimage_output": types.SimpleNamespace(images=[frames]), "attention_output": None, "mask_list": None}

    tmp = tempfile.mkdtemp()
    lg = P2pSampleLogger(editing_prompts=LOGGER_EDITS, clip_length=2, logdir=os.path.join(tmp, "log"), num_inference_steps=3,
                         guidance_scale=7.5, sample_seeds=[0], prompt2prompt_edit=True, p2p_config=LOGGER_P2P, use_inversion_attention=True,
                         source_prompt=SRC)
    lg.log_sample_images(pipeline=Recorder(), device=torch.device("cpu"), step=0, image=torch.zeros(2, 3, 16, 16),
                         latents=torch.zeros(1, 4, 2, 4, 4), save_dir=tmp)

    def enc(v):
        if isinstance(v, torch.Tensor):
            return {"__tensor__": list(v.shape)}
        if isinstance(v, torch.Generator):
            return {"__generator__": str(v.device)}
        if v == tmp:
            return {"__save_dir__": True}
        if isinstance(v, dict):
            return {k: enc(x) for k, x in v.items()}
        if isinstance(v, (list, tuple)):
            return [enc(x) for x in v]
        return v

    _write("ref_logger", dict(calls=[{k: enc(v) for k, v in kw.items()} for kw in calls]))


PINS = {"ref_unet_spec": pin_ref_unet_spec, "ref_tables_clip": pin_ref_tables_clip, "ref_logger": pin_ref_logger}

if __name__ == "__main__":
    names = sys.argv[1:] or list(PINS)
    if len(names) == 1:
        PINS[names[0]]()
    else:
        for n in names:
            subprocess.check_call([sys.executable, "-m", "oracle.make_ref_pins", n], cwd=ROOT)
