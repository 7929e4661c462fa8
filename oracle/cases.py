"""Parity cases shared by oracle/make_golden.py (reference run, build container) and the tests (oracle / CUDA runs).
Each case fixes geometry, model_config, prompts, steps and the p2p_config of one edit; inputs come from fatezero_b200.synth."""
SRC = "a silver jeep driving down a curvy road in the countryside"

CASES = {
    # config #1-like: Refine + Reweight (config/low_resource_teaser/jeep_watercolor_ddim_10_steps.yaml), small geometry
    "mini_refine": dict(
        unet="mini", model_config=dict(lora=160, SparseCausalAttention_index=["mid"], least_sc_channel=128),
        frames=3, size=32, steps=4, source=SRC, target="watercolor painting of " + SRC,
        p2p=dict(is_replace_controller=False, cross_replace_steps={"default_": 0.8}, self_replace_steps=0.8,
                 eq_params={"words": ["watercolor"], "values": [10, 10]})),
    # config #3-like: Replace + self-attention mask blend + latent blend (config/teaser/jeep_posche_local_latent_blend.yaml)
    "mini_replace_blend": dict(
        unet="mini", model_config=dict(lora=160, SparseCausalAttention_index=["mid"], least_sc_channel=128),
        frames=2, size=64, steps=5, source=SRC, target="a Porsche car driving down a curvy road in the countryside",
        p2p=dict(is_replace_controller=True, cross_replace_steps={"default_": 0.5}, self_replace_steps=0.6,
                 blend_words=[["silver", "jeep"], ["Porsche", "car"]], blend_self_attention=True, blend_latents=True,
                 blend_th=[0.985, 0.985])),
    # config #5-like semantics: default [-1, 'first'] K/V (two slots) at every level, no least_sc_channel
    "mini_shape": dict(
        unet="mini", model_config=dict(lora=160),
        frames=3, size=32, steps=3, source="a silver jeep driving down a curvy road", target="a red jeep driving down a curvy road",
        p2p=dict(is_replace_controller=True, cross_replace_steps={"default_": 0.7, "red": 0.4}, self_replace_steps=0.7)),
    # Replace + Reweight (equalizer on a swapped word) with ['first', +1] K/V frames (a forward-looking relative index) on 4 frames
    "mini_reweight_next": dict(
        unet="mini", model_config=dict(lora=160, SparseCausalAttention_index=["first", 1], least_sc_channel=128),
        frames=4, size=32, steps=4, source=SRC, target="a silver jeep driving down a snowy road in the countryside",
        p2p=dict(is_replace_controller=True, cross_replace_steps={"default_": 0.6}, self_replace_steps=0.5,
                 eq_params={"words": ["snowy"], "values": [3.0]})),
    # ---- oracle-pinning only (gpu=False: the CUDA parity tests skip them; they widen what the CPU oracle is held to) ----
    # Refine + latent blend WITHOUT self-attention blend, ['last', -1] K/V frames (the blender needs the 16x16 maps: 64x64 latents)
    "pin_refine_latent_blend": dict(
        gpu=False, unet="mini", model_config=dict(lora=160, SparseCausalAttention_index=["last", -1], least_sc_channel=128),
        frames=2, size=64, steps=3, source=SRC, target="a silver jeep driving down a curvy road in the snowy countryside",
        p2p=dict(is_replace_controller=False, cross_replace_steps={"default_": 0.7}, self_replace_steps=0.4,
                 blend_words=[["jeep"], ["jeep"]], blend_latents=True, blend_th=[0.9, 0.9])),
    # Replace on the wider 'mid' UNet geometry (attention at more channel counts), default [-1, 'first'] frames
    "pin_mid_replace": dict(
        gpu=False, unet="mid", model_config=dict(lora=160, least_sc_channel=320),
        frames=2, size=32, steps=3, source="a silver jeep driving down a curvy road", target="a silver tank driving down a curvy road",
        p2p=dict(is_replace_controller=True, cross_replace_steps={"default_": 0.8}, self_replace_steps=0.6,
                 eq_params={"words": ["silver", "tank"], "values": [2.0, 4.0]})),
    # BASELINE config #4 semantics (long clip, 'mid' source frame = frame 11 of 24, B*F = 48 rows in the CFG pass) at the mini geometry
    "pin_long24": dict(
        gpu=False, unet="mini", model_config=dict(lora=160, SparseCausalAttention_index=["mid"], least_sc_channel=128),
        frames=24, size=32, steps=1, source=SRC, target="watercolor painting of " + SRC,
        p2p=dict(is_replace_controller=False, cross_replace_steps={"default_": 0.8}, self_replace_steps=0.8,
                 eq_params={"words": ["watercolor"], "values": [10, 10]})),
    # ---- SD-1.4 geometry (head dims 40/80/160): too slow for the CPU oracle inside the suites, so these goldens are compared with
    # the CUDA product directly (tests/test_gpu_golden_sd14.py); big=True -> make_golden keeps map slices + checksums only ----
    # BASELINE config #1: config/low_resource_teaser/jeep_watercolor_ddim_10_steps.yaml (Refine + Reweight x10, ['mid'] / 640)
    "sd14_config1": dict(
        gpu=False, big=True, unet="sd14", model_config=dict(lora=160, SparseCausalAttention_index=["mid"], least_sc_channel=640),
        frames=8, size=64, steps=10, source=SRC, target="watercolor painting of " + SRC,
        p2p=dict(is_replace_controller=False, cross_replace_steps={"default_": 0.8}, self_replace_steps=0.8,
                 eq_params={"words": ["watercolor"], "values": [10, 10]})),
    # BASELINE config #3 semantics at SD-1.4 geometry: Replace + self-attention mask blend + latent blend
    # (config/attribute/bear_tiger_lion_leopard.yaml:65-69 + config/teaser/jeep_posche_local_latent_blend.yaml:29-39)
    "sd14_replace_blend": dict(
        gpu=False, big=True, unet="sd14", model_config=dict(lora=160, SparseCausalAttention_index=["mid"], least_sc_channel=640),
        frames=2, size=64, steps=4, source=SRC, target="a Porsche car driving down a curvy road in the countryside",
        p2p=dict(is_replace_controller=True, cross_replace_steps={"default_": 0.7}, self_replace_steps=0.7,
                 blend_words=[["silver", "jeep"], ["Porsche", "car"]], blend_self_attention=True, blend_latents=True,
                 blend_th=[0.985, 0.985])),
}
GPU_CASES = [k for k, v in CASES.items() if v.get("gpu", True)]
BIG_CASES = [k for k, v in CASES.items() if v.get("big")]
SMALL_CASES = [k for k, v in CASES.items() if not v.get("big")]

# host-side edit tables: tests/test_tables.py, pinned against the reference by oracle/make_ref_pins.py (ref_tables_clip)
PROMPT_PAIRS = [
    (SRC, "watercolor painting of " + SRC),
    (SRC, "a Porsche car driving down a curvy road in the countryside"),
    ("a silver jeep driving down a curvy road", "a red jeep driving down a curvy road"),
    ("a cat sitting next to a mirror", "a silver cat sculpture sitting next to a mirror"),
    ("a photorealistic squirrel eating a burger", "a photorealistic lion eating a burger"),
    ("a bear walking", "a extraordinarily fluffy bear is walking"),
]

# the reference's sample logger: tests/test_boundary_logger.py, pinned by oracle/make_ref_pins.py (ref_logger)
LOGGER_EDITS = [SRC, "watercolor painting of " + SRC]
LOGGER_P2P = {0: dict(is_replace_controller=False, cross_replace_steps={"default_": 0.8}, self_replace_steps=0.9, blend_self_attention=True),
              1: dict(is_replace_controller=False, cross_replace_steps={"default_": 0.8}, self_replace_steps=0.8,
                      eq_params={"words": ["watercolor"], "values": [10, 10]})}  # config/style/jeep_watercolor.yaml:36-68
