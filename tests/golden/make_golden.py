"""Generate the golden vectors under tests/golden/ from the REAL reference stack.

Run once in the build container (needs /root/reference and transformers; neither is used at test time):

    python tests/golden/make_golden.py

What is pinned (the reference has no tests / fixtures of its own, SURVEY.md §4):
  * ``transformers.CLIPModel`` (the third-party code the reference's hot path delegates to, plip.py:26,50,68)
    loaded with ``oracle.weights.make_state_dict(0)``: image / text features, normalised embeds,
    logits_per_image, and slices of the per-layer hidden states, on ``oracle.synth`` inputs;
  * the reference's own ``plip.PLIP`` class (from /root/reference/plip.py, with the two transformers>=5
    compatibility shims of SURVEY.md §8c) on cfg1: ``encode_images`` of 32 synthetic tiles, and its numpy
    heads ``_cosine_similarity`` / ``_nearest_neighbours``;
  * ``CLIPImageProcessor`` on non-224 images (resize + centre-crop + normalise).
Weights are regenerated from the seed at test time (bit-reproducible torch CPU generator), so only
outputs are stored, plus one of the processor's two input images (the other is regenerated from its seed).
"""
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, "/root/reference")

from oracle import synth, weights  # noqa: E402


def main():
    import transformers
    from transformers import CLIPConfig, CLIPImageProcessor, CLIPModel

    torch.set_grad_enabled(False)
    sd = weights.make_state_dict(0, "rich")
    hf = CLIPModel(CLIPConfig()).eval()
    hf.load_state_dict(sd, strict=True)
    out = {"transformers_version": np.array(transformers.__version__), "torch_version": np.array(torch.__version__)}

    # ---- HF CLIPModel on synthetic inputs -------------------------------------------------------
    n = 8
    px = synth.pixel_values(n)
    ids, mask = synth.token_ids(n)
    vo = hf.vision_model(pixel_values=px, output_hidden_states=True)
    to = hf.text_model(input_ids=ids, attention_mask=mask, output_hidden_states=True)
    full = hf(input_ids=ids, pixel_values=px, attention_mask=mask)
    out["image_features"] = hf.get_image_features(pixel_values=px).pooler_output.numpy()
    out["text_features"] = hf.get_text_features(input_ids=ids, attention_mask=mask).pooler_output.numpy()
    out["text_features_nomask"] = hf.get_text_features(input_ids=ids).pooler_output.numpy()
    out["image_embeds"] = full.image_embeds.numpy()
    out["text_embeds"] = full.text_embeds.numpy()
    out["logits_per_image"] = full.logits_per_image.numpy()
    out["logit_scale_exp"] = np.array(float(hf.logit_scale.exp()))
    for l in (0, 1, 6, 12):
        out[f"vision_hidden_{l}"] = vo.hidden_states[l][:2, :5, :].numpy()   # 2 images, first 5 tokens
        out[f"text_hidden_{l}"] = to.hidden_states[l][:2, :9, :].numpy()     # 2 captions, first 9 tokens
    out["vision_pooled"] = vo.pooler_output.numpy()
    out["text_pooled"] = to.pooler_output.numpy()
    # full-length captions (the headline "77-tok" shape)
    ids_f, mask_f = synth.token_ids(4, seed=77, full_length=True)
    out["text_features_full77"] = hf.get_text_features(input_ids=ids_f, attention_mask=mask_f).pooler_output.numpy()

    # ---- the reference's own PLIP class (shimmed) on cfg1 ------------------------------------------
    import PIL.Image
    import plip as ref_plip  # /root/reference/plip.py

    tmp = tempfile.mkdtemp(prefix="plip_golden_")
    hf.save_pretrained(tmp)
    CLIPImageProcessor().save_pretrained(tmp)

    def _strip(fn):
        def wrapped(name, *a, **kw):
            kw.pop("use_auth_token", None)
            return fn(name, *a, **kw)
        return wrapped

    ref_plip.CLIPModel.from_pretrained = _strip(ref_plip.CLIPModel.from_pretrained)       # shim 1
    ref_plip.CLIPProcessor.from_pretrained = _strip(ref_plip.CLIPProcessor.from_pretrained)
    ref = ref_plip.PLIP(tmp)
    _gif = ref.model.get_image_features
    ref.model.get_image_features = lambda **kw: _gif(**kw).pooler_output                  # shim 2
    tiles = synth.tiles_u8(32, seed=0)
    pil = [PIL.Image.fromarray(t) for t in tiles]
    out["ref_plip_encode_images_bs8"] = ref.encode_images(pil, batch_size=8).astype(np.float32)
    rng = np.random.default_rng(5)
    key = rng.standard_normal((6, 512)).astype(np.float32)
    space = rng.standard_normal((40, 512)).astype(np.float32)
    out["heads_key"], out["heads_space"] = key, space
    out["ref_cosine_similarity"] = ref._cosine_similarity(key, space)
    out["ref_nearest_neighbours_k5"] = ref._nearest_neighbours(5, key, space).astype(np.int64)

    # ---- CLIPImageProcessor on non-224 inputs --------------------------------------------------------
    proc = ref.preprocess.image_processor if hasattr(ref.preprocess, "image_processor") else CLIPImageProcessor()
    rng = np.random.default_rng(9)
    big = [rng.integers(0, 256, (300, 260, 3), dtype=np.uint8), rng.integers(0, 256, (224, 512, 3), dtype=np.uint8)]
    pv = proc(images=[PIL.Image.fromarray(b) for b in big], return_tensors="pt")["pixel_values"].numpy()
    out["proc_input_1"] = big[1]                    # big[0] is regenerated from the seed at test time (file < 1 MB)
    out["proc_pixel_values_sub"] = pv[:, :, ::8, ::8].copy()   # 28x28 subsample of the processor output
    out["proc_pixel_values_mean"] = pv.mean(axis=(2, 3))
    out["proc_class"] = np.array(type(proc).__name__)

    path = os.path.join(ROOT, "tests", "golden", "clip_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, {k: getattr(v, "shape", None) for k, v in out.items()})


if __name__ == "__main__":
    main()
