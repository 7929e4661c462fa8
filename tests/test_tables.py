"""Host-side edit tables: product (fatezero_b200.tables / controllers) == oracle restatement == reference (pinned)."""
import gzip
import json
import os

import pytest
import torch

from _helpers import ROOT
from fatezero_b200 import controllers, synth, tables
from oracle import fz_oracle as fo
from oracle.cases import CASES, PROMPT_PAIRS


@pytest.mark.parametrize("src,tgt", PROMPT_PAIRS)
def test_tables_match_oracle(src, tgt):
    tok = synth.ToyTokenizer()
    N = 10
    crs = {"default_": 0.8, tgt.split(" ")[1]: 0.3}
    al = tables.get_time_words_attention_alpha([src, tgt], N, crs, tok)
    assert torch.equal(al[:, 0, 0, 0, :], fo.cross_replace_alpha_table([src, tgt], N, crs, tok))
    mp, a = tables.get_refinement_mapper([src, tgt], tok)
    omp, oa = fo.refinement_tables([src, tgt], tok)
    assert torch.equal(mp[0], omp) and torch.equal(a[0], oa)
    if len(src.split(" ")) == len(tgt.split(" ")):
        assert torch.equal(tables.get_replacement_mapper([src, tgt], tok)[0], fo.replacement_matrix([src, tgt], tok))
    else:
        with pytest.raises(ValueError):
            tables.get_replacement_mapper([src, tgt], tok)
    word = tgt.split(" ")[1]
    assert torch.equal(tables.get_equalizer(tgt, [word], [10])[0] if False else tables.get_equalizer(tgt, [word], [10], tok)[0],
                       fo.equalizer_row(tgt, [word], [10], tok))


@pytest.mark.parametrize("name", list(CASES))
def test_make_controller_tables(name, tmp_path):
    """make_controller builds the kernel tables the oracle's EditPlan describes."""
    c = CASES[name]
    tok = synth.ToyTokenizer()
    p = c["p2p"]
    inv = controllers.AttentionStore()
    n_src, n_tgt = len(c["source"].split(" ")), len(c["target"].split(" "))
    ctrl = controllers.make_controller(tok, [c["source"], c["target"]], NUM_DDIM_STEPS=c["steps"],
                                       is_replace_controller=p.get("is_replace_controller", True) and n_src == n_tgt,
                                       cross_replace_steps=p["cross_replace_steps"], self_replace_steps=p["self_replace_steps"],
                                       blend_words=p.get("blend_words"), equilizer_params=p.get("eq_params"),
                                       additional_attention_store=inv, use_inversion_attention=True, blend_th=p.get("blend_th", (0.3, 0.3)),
                                       blend_self_attention=p.get("blend_self_attention"), blend_latents=p.get("blend_latents"),
                                       save_path=str(tmp_path), save_self_attention=False)
    plan = fo.EditPlan(tok, c["source"], c["target"], c["steps"], p["cross_replace_steps"], p["self_replace_steps"],
                       p.get("is_replace_controller", True), p.get("eq_params"), p.get("blend_words"),
                       bool(p.get("blend_self_attention")), bool(p.get("blend_latents")), p.get("blend_th", (0.3, 0.3)))
    tab = ctrl._build_xedit("cpu")
    assert tab.shape == (c["steps"] + 1, 8 + 4 * 80 + 6400)
    assert torch.equal(tab[:, 8:85], plan.alpha)
    assert int(tab[0, 0]) == (1 if plan.mode == "replace" else 0)
    if plan.mode == "replace":
        assert torch.equal(tab[0, 328:].reshape(80, 80)[:77, :77], plan.M)
    else:
        assert torch.equal(tab[0, 168:245], plan.a) and torch.equal(tab[0, 248:325], plan.mapper.float())
    eq = plan.eq if plan.eq is not None else torch.ones(77)
    assert torch.equal(tab[0, 88:165], eq)
    assert ctrl.num_self_replace == plan.self_window
    if plan.blend_src is not None:
        blender = ctrl.attention_blend or ctrl.latent_blend
        assert torch.equal(blender.word_row(0), plan.blend_src) and torch.equal(blender.word_row(1), plan.blend_tgt)
        if ctrl.latent_blend is not None:
            assert (ctrl.latent_blend.start_blend, ctrl.latent_blend.end_blend) == plan.lat_window


GOLDEN_TABLES = os.path.join(ROOT, "tests", "golden", "ref_tables_clip.json.gz")  # python -m oracle.make_ref_pins ref_tables_clip


class ReplayTokenizer:
    """The real CLIP BPE tokenizer's answers, as recorded while the reference computed the pinned tables."""

    def __init__(self, rec):
        self.encoded, self.decoded = rec["encode"], rec["decode"]

    def encode(self, text):
        assert text in self.encoded, f"encode({text!r}) was not recorded: regenerate the pin"
        return list(self.encoded[text])

    def decode(self, ids):
        assert len(ids) == 1 and str(int(ids[0])) in self.decoded, f"decode({ids!r}) was not recorded: regenerate the pin"
        return self.decoded[str(int(ids[0]))]


def test_tables_match_reference_with_clip_tokenizer():
    """The tables of the reference's own ptp_utils / seq_aligner with the real CLIP BPE (pinned) == this repo's tables."""
    g = json.load(gzip.open(GOLDEN_TABLES))
    tok = ReplayTokenizer(g["tokenizer"])

    def ref(name):
        return torch.tensor(c[name]["data"], dtype=getattr(torch, c[name]["dtype"]))

    assert [(c["source"], c["target"]) for c in g["cases"]] == [tuple(p) for p in PROMPT_PAIRS]
    for c in g["cases"]:
        src, tgt = c["source"], c["target"]
        crs = c["cross_replace_steps"]
        assert torch.equal(ref("alpha"), tables.get_time_words_attention_alpha([src, tgt], c["num_steps"], dict(crs), tok))
        m2, a2 = tables.get_refinement_mapper([src, tgt], tok)
        assert torch.equal(ref("refinement_mapper"), m2) and torch.equal(ref("refinement_alphas"), a2)
        assert ("replacement_mapper" in c) == (len(src.split(" ")) == len(tgt.split(" ")))
        if "replacement_mapper" in c:
            assert torch.equal(ref("replacement_mapper"), tables.get_replacement_mapper([src, tgt], tok))
        for w in tgt.split(" "):
            assert list(tables.get_word_inds(tgt, w, tok)) == c["word_inds"][w], (tgt, w)
