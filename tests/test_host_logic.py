"""Host-side logic that needs no GPU: validation, preprocessing, sharding maths, loud failure without CUDA."""
import numpy as np
import PIL.Image
import pytest
import torch

from plip_b200 import distributed as D
from plip_b200 import engine as E
from plip_b200 import preprocess as P


def test_pixel_format_validation_mirrors_hf_errors():
    assert E._pixel_format(torch.zeros(2, 3, 224, 224)) == E.PIX_F32_NCHW
    assert E._pixel_format(torch.zeros(2, 3, 224, 224, dtype=torch.bfloat16)) == E.PIX_BF16_NCHW
    assert E._pixel_format(np.zeros((2, 224, 224, 3), np.uint8)) == E.PIX_U8_NHWC
    with pytest.raises(ValueError, match=r"Input image size \(256\*256\) doesn't match model \(224\*224\)"):
        E._pixel_format(torch.zeros(1, 3, 256, 256))          # TF:modeling_clip.py:204-207
    with pytest.raises(ValueError):
        E._pixel_format(np.zeros((1, 3, 224, 224), np.uint8))  # uint8 must be NHWC
    with pytest.raises(TypeError):
        E._pixel_format(torch.zeros(1, 3, 224, 224, dtype=torch.float64))


def test_ids_validation():
    assert E._check_ids(torch.zeros(3, 77, dtype=torch.long), None) == (3, 77)
    with pytest.raises(ValueError, match="Sequence length must be less than max_position_embeddings"):
        E._check_ids(torch.zeros(3, 78, dtype=torch.long), None)   # TF:243-247
    with pytest.raises(ValueError, match="attention_mask"):
        E._check_ids(torch.zeros(3, 77, dtype=torch.long), torch.zeros(3, 76))
    with pytest.raises(TypeError):
        E._ids_dtype(torch.float32)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_silent_cpu_fallback(state_dict):
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        E.Engine(state_dict)
    from plip_b200.plip import PLIP
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        PLIP("whatever")


def test_preprocess_identity_on_224_tiles():
    rng = np.random.default_rng(0)
    tiles = rng.integers(0, 256, (3, 224, 224, 3), dtype=np.uint8)
    out = P.to_uint8_tiles([PIL.Image.fromarray(t) for t in tiles])
    assert out.dtype == np.uint8 and np.array_equal(out, tiles)
    assert np.array_equal(P.to_uint8_tiles(list(tiles)), tiles)   # arrays accepted too
    assert np.array_equal(P.to_uint8_tiles(list(tiles), workers=3), tiles)   # threaded decode keeps the order
    gray = PIL.Image.fromarray(tiles[0, :, :, 0])
    assert P.to_uint8_tiles([gray]).shape == (1, 224, 224, 3)     # convert_rgb


def test_preprocess_resize_crop_matches_clip_image_processor(golden):
    """Non-224 inputs: shortest-edge-224 bicubic + centre crop, then the device-side (x/255-mean)/std.
    Compared with the reference's CLIPImageProcessor output stored in the golden file."""
    from oracle import clip_oracle as O
    # the first input is regenerated from its seed (tests/golden/make_golden.py), the second is stored
    imgs = [np.random.default_rng(9).integers(0, 256, (300, 260, 3), dtype=np.uint8), golden["proc_input_1"]]
    tiles = P.to_uint8_tiles(imgs)
    assert tiles.shape == (2, 224, 224, 3)
    pv = O.preprocess_u8(torch.from_numpy(tiles)).numpy()
    ref_sub, ref_mean = golden["proc_pixel_values_sub"], golden["proc_pixel_values_mean"]
    # geometry (resize + crop window) must agree; interpolation kernels of PIL vs the processor backend
    # differ in the last bits of uint8 rounding -> compare with a small tolerance in normalised units
    assert np.abs(pv.mean(axis=(2, 3)) - ref_mean).max() < 5e-3
    diff = np.abs(pv[:, :, ::8, ::8] - ref_sub)
    assert np.median(diff) < 0.03 and np.mean(diff) < 0.06


def test_shard_counts_and_ranges():
    assert D.shard_counts(10, 4) == [3, 3, 2, 2]
    assert D.shard_counts(100000, 8) == [12500] * 8
    assert D.shard_counts(3, 8) == [1, 1, 1, 0, 0, 0, 0, 0]
    spans = [D.shard_range(10, r, 4) for r in range(4)]
    assert spans == [(0, 3), (3, 6), (6, 8), (8, 10)]
    assert D.world() == (0, 1)
    x = torch.arange(6.).view(3, 2)
    assert D.all_gather_rows(x) is x   # single process: identity


def test_non_rgb_images_follow_the_openai_transform_order():
    """reproducibility/embedders/transform.py:45-52 resizes and crops BEFORE convert("RGB"): for palette / bilevel
    images Pillow then resamples with NEAREST, for RGBA / LA it resamples premultiplied — converting first (what the
    HF processor of plip.py does, and what the RGB fast path does) would give different tiles (ADVICE r1)."""
    import numpy as np
    import PIL.Image
    from plip_b200.preprocess import decode_native_then_rgb, resize_plan

    rng = np.random.default_rng(3)
    pal = PIL.Image.fromarray(rng.integers(0, 256, (260, 300), dtype=np.uint8), mode="P")
    pal.putpalette(rng.integers(0, 256, 768, dtype=np.uint8).tobytes())
    rgba = PIL.Image.fromarray(rng.integers(0, 256, (300, 250, 4), dtype=np.uint8), mode="RGBA")
    rgb = PIL.Image.fromarray(rng.integers(0, 256, (240, 320, 3), dtype=np.uint8))
    got = decode_native_then_rgb([pal, rgba, rgb], crop="round")
    for im, out in zip((pal, rgba), got[:2]):
        nw, nh, left, top = resize_plan(*im.size, 224, "round")
        ref = im.resize((nw, nh), resample=PIL.Image.BICUBIC).crop((left, top, left + 224, top + 224)).convert("RGB")
        assert out.shape == (224, 224, 3) and np.array_equal(out, np.asarray(ref))
        first = np.asarray(im.convert("RGB").resize((nw, nh), resample=PIL.Image.BICUBIC).crop((left, top, left + 224, top + 224)))
        assert not np.array_equal(out, first)                        # the order really matters for these modes
    assert got[2].shape == (240, 320, 3)                             # RGB images stay un-resized for the device kernel
