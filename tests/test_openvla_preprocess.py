"""OpenVLA image preprocessing (Pillow bicubic resize, center crop, per-tower normalisation) and `OpenVlaPolicy`.

CPU (-m "not gpu"): the oracle against Pillow and the full torchvision pipeline bit for bit; the library's host-side
coefficient builder against the oracle; `resize_geometry` against what torchvision produces; argument checks.
GPU (-m gpu): the kernel against Pillow + torchvision bit for bit (batched, strided, padded rows), malformed calls,
and `OpenVlaPolicy.predict_action` from frames against the hand composition from torchvision-prepared pixels."""

import ctypes as C

import numpy as np
import pytest
import torch
import torchvision.transforms.functional as TVF
from PIL import Image

from blurr_b200 import capi, openvla
from oracle import openvla_preprocess_oracle as O

DEV = "cuda:0"
BICUBIC = TVF.InterpolationMode.BICUBIC
MEANS, STDS = (O.DINOV2_MEAN, O.SIGLIP_MEAN), (O.DINOV2_STD, O.SIGLIP_STD)
# (h, w, size): landscape / portrait, identity, square downscale, upscale (crop offset 33.5 -> 34), crop offsets
# 0.5 -> 0 and 1.5 -> 2, odd sizes, HD frames, and the "resize-naive" (h, w) size of the released checkpoint
GEOMS = [(480, 640, 224), (640, 480, 224), (224, 224, 224), (256, 256, 224), (100, 130, 224), (224, 225, 224),
         (224, 227, 224), (181, 224, 224), (333, 517, 224), (720, 1280, 224), (1080, 1920, 224), (480, 640, (224, 224))]
KINDS = ["noise", "smooth", "checker"]


def _gid(g):
    return f"{g[0]}x{g[1]}-{'x'.join(map(str, g[2])) if isinstance(g[2], tuple) else g[2]}"


def frame(seed, h, w, kind):
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    if kind == "checker":                   # 0/255 edges: bicubic overshoot reaches both clip bounds
        c = ((yy // (1 + seed % 3) + xx // 2) % 2) * 255
        return np.stack([c, 255 - c, c], -1).astype(np.uint8)
    base = 127 + 100 * np.sin(xx / (13.0 + seed) + seed) * np.cos(yy / 19.0)
    return np.clip(np.stack([base, 0.6 * base + 60, 255 - base], -1), 0, 255).astype(np.uint8)


def torchvision_pixels(img, size=224, crop=224):
    """What OpenVLA's processor computes per image: resize + crop + to_tensor + normalize per tower, vstack, bf16."""
    pil = Image.fromarray(img)
    outs = []
    for m, s in zip(MEANS, STDS):
        x = TVF.center_crop(TVF.resize(pil, size, interpolation=BICUBIC), crop)
        outs.append(TVF.normalize(TVF.to_tensor(x), m, s))
    return torch.vstack(outs).to(torch.bfloat16)


def torchvision_resized(img, size=224, crop=224):
    return np.asarray(TVF.center_crop(TVF.resize(Image.fromarray(img), size, interpolation=BICUBIC), crop))


def _bits(t):
    return t.contiguous().view(torch.int16)


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("geom", GEOMS, ids=_gid)
def test_oracle_equals_pillow_and_torchvision(geom, kind):
    h, w, size = geom
    img = frame(h + w, h, w, kind)
    rh, rw, _, _ = O.resize_geometry(h, w, size)
    ref = np.asarray(Image.fromarray(img).resize((rw, rh), Image.BICUBIC))
    assert np.array_equal(O.resize_bicubic_u8(img, rh, rw), ref)
    px, small = O.preprocess(img, size)
    assert np.array_equal(small, torchvision_resized(img, size))
    assert torch.equal(_bits(px), _bits(torchvision_pixels(img, size)))


@pytest.mark.parametrize("src,dst", [(53, 24), (24, 53), (640, 298), (480, 224), (640, 224), (517, 347), (333, 224),
                                     (1280, 398), (720, 224), (1920, 398), (1080, 224), (1920, 224), (100, 224),
                                     (130, 291), (224, 224), (225, 224), (227, 224), (1, 3), (3, 1)])
def test_library_coefficients_equal_oracle(src, dst):
    """The C++ table builder (host code of the library, no GPU needed) against the oracle's Pillow restatement."""
    bounds, weights = openvla.pillow_bicubic_coefficients(src, dst)
    o_bounds, o_weights = O.coefficients(src, dst)
    assert np.array_equal(bounds, o_bounds) and np.array_equal(weights, o_weights)
    assert (weights.astype(np.int64).sum(1) - (1 << 22)).__abs__().max() <= weights.shape[1]     # ~1.0 in Q22
    # a wider weight table is zero past ksize
    lib = capi.load_library()
    b2 = np.zeros((dst, 2), np.int32)
    w2 = np.full((dst, weights.shape[1] + 3), -7, np.int32)
    assert lib.blurr_vla_preproc_build_coeffs(src, dst, b2.ctypes.data_as(C.POINTER(C.c_int32)),
                                              w2.ctypes.data_as(C.POINTER(C.c_int32)), w2.shape[1]) == weights.shape[1]
    assert np.array_equal(w2[:, :weights.shape[1]], weights) and not w2[:, weights.shape[1]:].any()


@pytest.mark.parametrize("geom", GEOMS, ids=_gid)
def test_resize_geometry_matches_torchvision(geom):
    h, w, size = geom
    img = frame(1, h, w, "noise")
    resized = TVF.resize(Image.fromarray(img), size, interpolation=BICUBIC)
    rh, rw, top, left = openvla.resize_geometry(h, w, size)
    assert (rh, rw, top, left) == O.resize_geometry(h, w, size)
    assert (resized.height, resized.width) == (rh, rw)
    arr = np.asarray(resized)
    assert np.array_equal(np.asarray(TVF.center_crop(resized, 224)), arr[top:top + 224, left:left + 224])


def test_resize_geometry_rejects_crop_larger_than_resize():
    with pytest.raises(ValueError):
        openvla.resize_geometry(480, 640, (200, 300), 224)


def _create(*args, mean=(0.5,) * 6, std=(0.5,) * 6):
    lib = capi.load_library()
    h = C.c_void_p()
    st = lib.blurr_vla_preproc_create(0, *args, (C.c_float * 6)(*mean), (C.c_float * 6)(*std), C.byref(h))
    if st == 0:
        lib.blurr_vla_preproc_destroy(h)
    return st


@pytest.mark.parametrize("args", [
    (0, 640, 224, 298, 0, 37, 224, 224, 2),           # empty source
    (480, 640, 224, -298, 0, 37, 224, 224, 2),        # negative resize
    (480, 640, 224, 298, 0, 37, 0, 224, 2),           # empty crop
    (480, 640, 224, 298, 1, 37, 224, 224, 2),         # crop below the resize
    (480, 640, 224, 298, 0, 75, 224, 224, 2),         # crop right of the resize
    (480, 640, 224, 298, -1, 37, 224, 224, 2),        # negative offset
    (480, 640, 224, 298, 0, 37, 224, 224, 0),         # n_norms 0
    (480, 640, 224, 298, 0, 37, 224, 224, 3),         # n_norms 3
    (40000, 640, 224, 298, 0, 37, 224, 224, 2),       # larger than 32768
    (30000, 640, 224, 298, 0, 37, 224, 224, 2),       # one row's 535-row window does not fit in shared memory
], ids=["src0", "resize-neg", "crop0", "crop-bottom", "crop-right", "offset-neg", "norms0", "norms3", "huge", "smem"])
def test_create_rejects_invalid_arguments(args):
    """Rejected before any device is touched, so this holds with and without a GPU."""
    assert _create(*args) == -1


def test_create_rejects_zero_std_and_coeffs_reject_bad_sizes():
    std = (0.229, 0.224, 0.225, 0.5, 0.0, 0.5)
    assert _create(480, 640, 224, 298, 0, 37, 224, 224, 2, std=std) == -1
    lib = capi.load_library()
    assert lib.blurr_vla_preproc_build_coeffs(0, 224, None, None, 0) == -1
    assert lib.blurr_vla_preproc_build_coeffs(640, -1, None, None, 0) == -1
    b = np.zeros((224, 2), np.int32)
    w = np.zeros((224, 5), np.int32)                # 640 -> 224 needs 11 taps
    assert lib.blurr_vla_preproc_build_coeffs(640, 224, b.ctypes.data_as(C.POINTER(C.c_int32)),
                                              w.ctypes.data_as(C.POINTER(C.c_int32)), 5) == -1


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("geom", GEOMS, ids=_gid)
def test_gpu_kernel_bit_exact(geom):
    h, w, size = geom
    pre = openvla.ImagePreprocessor(h, w, size, device=DEV)
    (xb, xw), (yb, yw) = pre.coefficients()
    assert np.array_equal(xw, O.coefficients(w, pre.resize_w)[1]) and np.array_equal(yb, O.coefficients(h, pre.resize_h)[0])
    frames = np.stack([frame(b + 5, h, w, kind) for b, kind in enumerate(KINDS)])        # batch 3, one kind per slot
    px, small = pre(torch.as_tensor(frames).to(DEV), return_resized=True)
    torch.cuda.synchronize()
    assert px.shape == (3, 6, 224, 224) and small.shape == (3, 224, 224, 3)
    for b in range(3):
        assert np.array_equal(small[b].cpu().numpy(), torchvision_resized(frames[b], size)), b
        assert torch.equal(_bits(px[b].cpu()), _bits(torchvision_pixels(frames[b], size))), b
    pre.close()


@pytest.mark.gpu
def test_gpu_strided_frames_and_padded_rows():
    h, w = 333, 517
    pre = openvla.ImagePreprocessor(h, w, device=DEV)
    host = np.stack([frame(40 + b, h, w, KINDS[b % 3]) for b in range(6)])
    ref = torch.stack([torchvision_pixels(f) for f in host[::2]])
    dense = torch.as_tensor(host).to(DEV)
    every_other = dense[::2]                                      # frame stride of two frames
    assert not every_other.is_contiguous()
    padded = torch.zeros((3, h, w + 7, 3), dtype=torch.uint8, device=DEV)
    padded[:, :, :w] = every_other
    rows = padded[:, :, :w]                                       # row stride 3 * (w + 7)
    assert rows.stride(1) == 3 * (w + 7)
    for frames in (every_other, rows):
        px = pre(frames)
        torch.cuda.synchronize()
        assert torch.equal(_bits(px.cpu()), _bits(ref))
    out = torch.empty((3, 6, 224, 224), device=DEV, dtype=torch.bfloat16)
    assert pre(rows, out=out) is out
    with pytest.raises(ValueError):
        pre(dense[:, :, :w - 1])
    pre.close()


@pytest.mark.gpu
def test_gpu_malformed_calls_raise():
    with pytest.raises(capi.BlurrError):
        openvla.ImagePreprocessor(480, 640, means=(O.DINOV2_MEAN,) * 3, stds=(O.DINOV2_STD,) * 3, device=DEV)
    with pytest.raises(capi.BlurrError):
        openvla.ImagePreprocessor(480, 640, means=(O.DINOV2_MEAN,), stds=((0.2, 0.0, 0.2),), device=DEV)
    assert _create(1080, 1920, 224, 398, 0, 87, 224, 224, 2) == 0          # a 21-row window per output row fits
    pre = openvla.ImagePreprocessor(480, 640, device=DEV)
    lib = pre.lib
    f = torch.zeros((2, 480, 640, 3), dtype=torch.uint8, device=DEV)
    px = torch.empty((2, 6, 224, 224), dtype=torch.bfloat16, device=DEV)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    fp, pp = C.c_void_p(f.data_ptr()), C.c_void_p(px.data_ptr())
    for args in [(fp, 640 * 3 - 1, 2, f.stride(0), pp),       # row stride below 3 * width
                 (fp, 640 * 3, 0, f.stride(0), pp),           # empty batch
                 (fp, 640 * 3, 65536, f.stride(0), pp),       # batch beyond the grid
                 (None, 640 * 3, 2, f.stride(0), pp),         # null frames
                 (fp, 640 * 3, 2, f.stride(0), None)]:        # null output
        with pytest.raises(capi.BlurrError):
            capi.check(lib.blurr_vla_preproc_frame(pre.handle, stream, *args, None))
    with pytest.raises(capi.BlurrError):
        capi.check(lib.blurr_vla_preproc_frame(None, stream, fp, 640 * 3, 2, f.stride(0), pp, None))
    pre(f, out=px)                                                # the handle still works
    torch.cuda.synchronize()
    pre.close()


@pytest.mark.gpu
def test_gpu_predict_action_from_frames_equals_hand_composition():
    """Shrunk towers (depth 3) and a 2-layer 4096-wide decoder: `predict_action(frames)` == torchvision pixels ->
    towers on contiguous copies -> projector -> prompt -> generate -> de-tokenise, token ids and actions equal."""
    B = 2
    dino = openvla.VitEncoder.synthetic(openvla.dinov2_large_reg4_config(depth=3), DEV, max_batch=B, seed=3)
    sig = openvla.VitEncoder.synthetic(openvla.siglip_so400m_config(depth=3), DEV, max_batch=B, seed=4)
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], DEV, max_rows=B * 256)
    g = torch.Generator(device=DEV).manual_seed(5)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=DEV, generator=g) * 0.02).to(torch.bfloat16),
                       (torch.randn(n_out, device=DEV, generator=g) * 0.02).to(torch.bfloat16))
    backbone = openvla.FusedVisionBackbone(dino, sig, proj)
    cfg = openvla.LlamaShapedConfig(num_layers=2)
    dec = openvla.LlamaDecoder.from_state_dict(cfg, openvla.synthetic_llama_state_dict(cfg, DEV, 0), DEV, max_batch=B)
    pre = openvla.ImagePreprocessor(480, 640, device=DEV)
    policy = openvla.OpenVlaPolicy(pre, backbone, dec)
    frames = np.stack([frame(60, 480, 640, "smooth"), frame(61, 480, 640, "noise")])
    ids_in = torch.randint(3, 32000, (B, 1 + 24), device=DEV, generator=g)
    ids_in[:, 0] = 1
    q01 = np.array([-0.03, -0.04, -0.02, -0.1, -0.1, -0.2, 0.0])
    q99 = np.array([0.03, 0.04, 0.03, 0.1, 0.1, 0.2, 1.0])
    mask = np.array([True] * 6 + [False])

    px_ref = torch.stack([torchvision_pixels(f) for f in frames]).to(DEV)
    feats = torch.cat([dino.forward(px_ref[:, :3].contiguous()), sig.forward(px_ref[:, 3:].contiguous())], dim=-1)
    embeds = openvla.build_prompt_embeds(dec, ids_in, proj.forward(feats))
    ids_ref = dec.generate(embeds, 7)
    act_ref = torch.from_numpy(openvla.ActionDetokenizer().actions(ids_ref.cpu().numpy(), q01, q99, mask))

    for source in (frames, torch.as_tensor(frames).to(DEV)):              # host frames and device-resident frames
        actions, ids = policy.predict_action(source, ids_in, q01, q99, mask, return_token_ids=True)
        assert torch.equal(ids, ids_ref)
        assert actions.shape == (B, 7) and actions.dtype == torch.float64
        assert torch.equal(actions, act_ref)
    one = policy.predict_action(frames[0], ids_in[:1], q01, q99, mask)     # a single [H, W, 3] frame
    assert torch.equal(one, act_ref[:1])

    # the two halves of one 6-channel pixel tensor feed the towers as strided views: same features as copies
    px = pre(torch.as_tensor(frames).to(DEV))
    assert torch.equal(px, px_ref)
    assert torch.equal(dino.forward(px[:, :3]), dino.forward(px[:, :3].contiguous()))
    assert torch.equal(sig.forward(px[:, 3:]), sig.forward(px[:, 3:].contiguous()))
    assert torch.equal(backbone.forward(px[:, :3], px[:, 3:]), backbone.forward(px[:, :3].contiguous(), px[:, 3:].contiguous()))
    torch.cuda.synchronize()
    dec.check()
    for m in (pre, dino, sig, proj, dec):
        m.close()
