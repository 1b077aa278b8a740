"""OpenVLA-OFT's FiLM language conditioning of the vision towers: `blurr_vit_forward_film` (the conditioning GEMM and the
FiLM consumers), `VitEncoder` / `FusedVisionBackbone` with `film_cond`, `film_language_rows` /
`film_language_embedding` and `OftPolicy` with `use_film`.  The specification is oracle/openvla_oft_film_oracle.py.

CPU (-m "not gpu"): the oracle with zero FiLM weights is transformers' own tower (bitwise, fp32 and bf16), the oracle's
FiLMed block is the block in functional ops, the averaged rows for every prompt form, the config's ctypes field, the ABI
version and the new symbol.
GPU (-m gpu): FiLM towers against the oracle with fp32 as the tie-breaker in each consumer regime; zero FiLM weights
give the plain tower bit for bit; isolation of sequences, shared cameras and graph replays (bitwise); rejected calls;
the FiLM policy on a shrunk stack with one and two cameras."""

import os
import re

import numpy as np
import pytest
import torch

from blurr_b200 import capi, openvla
from llama_helpers import Q01, Q99, instructions
from oracle import openvla_oft_film_oracle as OF

DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def _hf_dinov2(hidden, heads, depth, seed):
    from transformers import Dinov2WithRegistersConfig, Dinov2WithRegistersModel
    hc = Dinov2WithRegistersConfig(hidden_size=hidden, num_hidden_layers=depth, num_attention_heads=heads, mlp_ratio=4,
                                   image_size=224, patch_size=14, num_register_tokens=4, layerscale_value=1.0,
                                   attn_implementation="eager")
    torch.manual_seed(seed)
    model = Dinov2WithRegistersModel(hc).eval()
    with torch.no_grad():
        for name, p in model.named_parameters():
            if "lambda1" in name:
                p.copy_(0.5 + torch.rand_like(p))
            elif "cls_token" in name or "register_tokens" in name or "position_embeddings" in name:
                p.copy_(0.5 * torch.randn_like(p))
            elif name.endswith("weight") and p.dim() == 2:
                p.mul_(1.5)
    return model


def _hf_siglip(hidden, inter, heads, depth, seed):
    from transformers import SiglipVisionConfig, SiglipVisionModel
    hc = SiglipVisionConfig(hidden_size=hidden, intermediate_size=inter, num_hidden_layers=depth, num_attention_heads=heads,
                            image_size=224, patch_size=14, attn_implementation="eager")
    torch.manual_seed(seed)
    model = SiglipVisionModel(hc).eval()
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith("weight") and p.dim() == 2 and "position" not in name:
                p.mul_(1.5)
    return model


def _films(n_blocks, llm_dim, vision_dim, seed, zero=False):
    torch.manual_seed(seed)
    films = OF.film_modules(n_blocks, llm_dim, vision_dim).eval()
    with torch.no_grad():
        for f in films:
            for lin in (f.scale, f.shift):
                if zero:
                    lin.weight.zero_()
                    lin.bias.zero_()
                else:                        # |gamma| around 0.5 for a unit-scale language vector
                    lin.weight.copy_(torch.randn_like(lin.weight) * 0.5 / llm_dim ** 0.5)
                    lin.bias.copy_(torch.randn_like(lin.bias) * 0.1)
    return films


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("tower", ["dinov2", "siglip"])
def test_oracle_with_zero_film_is_the_transformers_tower(tower, dtype):
    model = _hf_dinov2(64, 2, 3, 0) if tower == "dinov2" else _hf_siglip(64, 112, 2, 3, 1)
    model = model.to(dtype)
    films = _films(2, 32, 64, 2, zero=True).to(dtype)
    px = (torch.rand((3, 3, 224, 224)) * 2 - 1).to(dtype)
    lang = torch.randn((3, 32)).to(dtype)
    prefix = 5 if tower == "dinov2" else 0
    with torch.inference_mode():
        ref = model(pixel_values=px, output_hidden_states=True).hidden_states[-2][:, prefix:]
        got = OF.film_tower(model, px, films, lang)
    assert torch.equal(got, ref)


@pytest.mark.parametrize("tower", ["dinov2", "siglip"])
def test_oracle_film_block_is_the_functional_block(tower):
    F = torch.nn.functional
    model = (_hf_dinov2(64, 2, 2, 3) if tower == "dinov2" else _hf_siglip(64, 112, 2, 2, 4)).to(torch.bfloat16)
    layer = model.encoder.layer[0] if tower == "dinov2" else model.vision_model.encoder.layers[0]
    g = torch.Generator().manual_seed(5)
    x = torch.randn((2, 261, 64), generator=g).to(torch.bfloat16)
    gamma = (torch.randn((2, 64), generator=g) * 0.5).to(torch.bfloat16)
    beta = (torch.randn((2, 64), generator=g) * 0.1).to(torch.bfloat16)
    sd = {k: v for k, v in layer.state_dict().items()}
    H, nh = 64, 2
    if tower == "dinov2":
        n1, n2, q, k, v, o = "norm1", "norm2", "attention.attention.query", "attention.attention.key", \
            "attention.attention.value", "attention.output.dense"
        f1, f2 = "mlp.fc1", "mlp.fc2"
    else:
        n1, n2, q, k, v, o = "layer_norm1", "layer_norm2", "self_attn.q_proj", "self_attn.k_proj", "self_attn.v_proj", \
            "self_attn.out_proj"
        f1, f2 = "mlp.fc1", "mlp.fc2"
    lin = lambda t, name: F.linear(t, sd[name + ".weight"], sd[name + ".bias"])
    eps = model.config.layer_norm_eps

    def attn(t):
        N, T, _ = t.shape
        heads = lambda u: u.view(N, T, nh, H // nh).transpose(1, 2)
        qh, kh, vh = heads(lin(t, q)), heads(lin(t, k)), heads(lin(t, v))
        w = torch.matmul(qh, kh.transpose(2, 3)) * (H // nh) ** -0.5
        w = F.softmax(w, dim=-1, dtype=torch.float32).to(t.dtype)
        return lin(torch.matmul(w, vh).transpose(1, 2).reshape(N, T, H), o)

    h = attn(F.layer_norm(x, (H,), sd[n1 + ".weight"], sd[n1 + ".bias"], eps))
    if tower == "dinov2":
        h = h * sd["layer_scale1.lambda1"]
    y = x + h
    y = y * (1 + gamma[:, None]) + beta[:, None]
    m = lin(F.layer_norm(y, (H,), sd[n2 + ".weight"], sd[n2 + ".bias"], eps), f1)
    m = lin(F.gelu(m) if tower == "dinov2" else F.gelu(m, approximate="tanh"), f2)
    if tower == "dinov2":
        m = m * sd["layer_scale2.lambda1"]
    ref = y + m
    with torch.inference_mode():
        got = OF.film_block(layer, x, gamma, beta)
    assert torch.equal(got, ref)


def _padded(rows, left: bool, pad_id: int = 7):
    S = max(r.numel() for r in rows)
    ids = torch.full((len(rows), S), pad_id, dtype=torch.int64)
    mask = torch.zeros((len(rows), S), dtype=torch.int64)
    for b, r in enumerate(rows):
        sl = slice(S - r.numel(), S) if left else slice(0, r.numel())
        ids[b, sl] = r
        mask[b, sl] = 1
    return ids, mask


def test_film_language_rows_for_every_prompt_form():
    rows = instructions([9, 4, 13], 0)
    rows[1] = torch.cat([rows[1], torch.tensor([29871])])        # already ends with the empty token: nothing appended
    lay = openvla.oft_prompt_layout(rows, n_patches=256)
    got = openvla.film_language_rows(lay)
    for b, r in enumerate(rows):
        prompt = r.tolist() + ([] if r[-1] == 29871 else [29871])
        want = OF.language_rows(prompt, lay.n_rows)
        assert got[b].tolist() == want == prompt + [2]
        assert len(want) == int(lay.text_lens[b]) + 1        # no pad and no action slot is averaged
    for left in (True, False):
        ids, m = _padded(rows, left)
        lay2 = openvla.oft_prompt_layout(ids, attention_mask=m, n_patches=256)
        assert [t.tolist() for t in openvla.film_language_rows(lay2)] == [t.tolist() for t in got]
    eq = torch.stack(instructions([6, 6], 1))
    lay3 = openvla.oft_prompt_layout(eq, n_patches=513, cfg=openvla.oft_libero_config())
    assert [t.tolist() for t in openvla.film_language_rows(lay3)] == [r.tolist() + [29871, 2] for r in eq]
    # the oracle's rows are OFT's input ids where the action mask is False; the placeholders are the masked ones
    ids, mask = OF.oft_input_ids([1, 5, 29871], 56)
    assert len(ids) == 60 and sum(mask) == 56 and not mask[0] and not mask[-1] and ids[-1] == 2


def test_oracle_language_embedding_is_the_per_sequence_mean():
    g = torch.Generator().manual_seed(2)
    emb = torch.randint(-8, 8, (2, 10, 16), generator=g).to(torch.bfloat16)       # exact sums in any order
    mask = torch.zeros((2, 10), dtype=torch.bool)
    mask[:, 3:8] = True
    got = OF.language_embedding(emb, mask)
    ref = torch.cat([emb[:, :3], emb[:, 8:]], dim=1).float().sum(dim=1) / 5
    assert got.dtype == torch.bfloat16 and torch.equal(got, ref.to(torch.bfloat16))


def test_vit_config_has_film_dim_abi_version_2_and_the_film_symbol():
    assert [f[0] for f in capi.VitConfigC._fields_][-1] == "film_dim"
    header = open(os.path.join(ROOT, "include", "blurr_vit.h")).read()
    assert re.search(r"#define BLURR_VIT_ABI_VERSION (\d+)", header).group(1) == str(capi.VIT_ABI_VERSION) == "2"
    assert "blurr_vit_forward_film" in capi.DECLARED_SYMBOLS and "blurr_vit_forward_film(" in header
    assert openvla.VitShapedConfig(1, 1024, 16, 4096).film_dim == 0 and not openvla.OftConfig().use_film


# ---------------------------------------------------------------------------------------------------------------------
# GPU: FiLM towers
# ---------------------------------------------------------------------------------------------------------------------
def _check_against_fp32(name, got, ref16, ref32):
    e_ours = (got.float() - ref32).abs()
    e_ref = (ref16.float() - ref32).abs()
    rms = ref32.pow(2).mean().sqrt().item()
    print(f"{name}: vs fp32 ours max {e_ours.max().item():.3e} mean {e_ours.mean().item():.3e} | transformers bf16 max "
          f"{e_ref.max().item():.3e} mean {e_ref.mean().item():.3e} (ref rms {rms:.3f})")
    assert e_ours.mean().item() <= 1.5 * e_ref.mean().item() + 1e-4 * rms
    assert e_ours.max().item() <= 2.5 * e_ref.max().item() + 1e-2 * rms


def _pixels(batch, seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return (torch.rand((batch, 3, 224, 224), device=DEV, generator=g) * 2 - 1).to(torch.bfloat16)


def _lang(n, dim, seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return torch.randn((n, dim), device=DEV, generator=g).to(torch.bfloat16)


FILM_DIM = 512


# batch 1: split-K partials; 3 and 5 images: the bf16 hand-off; 8 images (>= 2048 rows): the streaming consumers
@pytest.mark.gpu
@pytest.mark.parametrize("batch,ipc", [(1, 1), (3, 1), (4, 2), (8, 2)])
@pytest.mark.parametrize("tower", ["dinov2", "siglip"])
def test_film_tower_matches_the_oracle(tower, batch, ipc):
    if tower == "dinov2":
        model, H = _hf_dinov2(1024, 16, 3, 0), 1024
    else:
        model, H = _hf_siglip(1152, 4304, 16, 3, 1), 1152
    films = _films(2, FILM_DIM, H, 7)
    model = model.to(torch.bfloat16).to(DEV)
    films = films.to(torch.bfloat16).to(DEV)
    ctor = openvla.VitEncoder.from_hf_dinov2 if tower == "dinov2" else openvla.VitEncoder.from_hf_siglip
    enc = ctor(model, DEV, max_batch=batch, films=films.state_dict())
    px = _pixels(batch, 1)
    lang = _lang(batch // ipc, FILM_DIM, 2)
    with torch.inference_mode():
        ref = OF.film_tower(model, px, films, lang, ipc)
        ref32 = OF.film_tower(model.float(), px.float(), films.float(), lang.float(), ipc)
        gam = films[0].float().scale(lang.float())
    print(f"|gamma| of block 0: mean {gam.abs().mean().item():.3f}")
    got = enc.forward(px, film_cond=lang, images_per_cond=ipc)
    torch.cuda.synchronize()
    _check_against_fp32(f"{tower} FiLM tower B={batch} ipc={ipc} ({enc.last_launch_count} launches)", got, ref, ref32)
    assert not torch.equal(ref, model.to(torch.bfloat16)(pixel_values=px, output_hidden_states=True).hidden_states[-2][
        :, 5 if tower == "dinov2" else 0:])
    enc.close()


def _tower_pair(tower, max_batch):
    cfg = openvla.dinov2_large_reg4_config(depth=3) if tower == "dinov2" else openvla.siglip_so400m_config(depth=3)
    plain = openvla.VitEncoder.synthetic(cfg, DEV, max_batch=max_batch, seed=11)
    cfg_f = openvla.VitShapedConfig(**{**cfg.__dict__, "film_dim": FILM_DIM})
    film = openvla.VitEncoder.synthetic(cfg_f, DEV, max_batch=max_batch, seed=11)
    return plain, film


@pytest.mark.gpu
@pytest.mark.parametrize("tower", ["dinov2", "siglip"])
def test_zero_film_weights_give_the_plain_tower_bitwise(tower):
    plain, film = _tower_pair(tower, 8)
    H = plain.cfg.hidden
    z = torch.zeros((H, FILM_DIM), device=DEV, dtype=torch.bfloat16)
    for l in range(film.cfg.num_layers):
        for name in ("film_scale", "film_shift"):
            film.set_weight(f"layers.{l}.{name}.weight", z)
            film.set_weight(f"layers.{l}.{name}.bias", z[:, 0])
    film.finalize()
    for batch, ipc in ((1, 1), (3, 3), (8, 4)):
        px = _pixels(batch, batch)
        lang = _lang(batch // ipc, FILM_DIM, 3)
        ref = plain.forward(px)
        for graph in (1, 0):
            film.set_option("use_cuda_graph", graph)
            got = film.forward(px, film_cond=lang, images_per_cond=ipc)
            torch.cuda.synchronize()
            assert torch.equal(got, ref), (batch, graph)
        film.set_option("use_cuda_graph", 1)
    plain.close()
    film.close()


@pytest.mark.gpu
@pytest.mark.parametrize("tower", ["dinov2", "siglip"])
def test_film_isolation_shared_cameras_and_graph_replay(tower):
    plain, film = _tower_pair(tower, 8)
    plain.close()
    px = _pixels(8, 4)
    lang = _lang(4, FILM_DIM, 5)
    out = film.forward(px, film_cond=lang, images_per_cond=2).clone()
    # another condition for sequence 2 changes its two images only
    lang2 = lang.clone()
    lang2[2] = _lang(1, FILM_DIM, 6)[0]
    out2 = film.forward(px, film_cond=lang2, images_per_cond=2)
    keep = [0, 1, 2, 3, 6, 7]
    assert torch.equal(out2[keep], out[keep]) and not torch.equal(out2[4:6], out[4:6])
    # permuting sequences permutes the outputs
    perm = [2, 0, 3, 1]
    img = [2 * p + c for p in perm for c in range(2)]
    outp = film.forward(px[img].contiguous(), film_cond=lang[perm].contiguous(), images_per_cond=2)
    assert torch.equal(outp, out[img])
    # the cameras of a sequence share its condition: the same as one condition row per image
    out1 = film.forward(px, film_cond=lang.repeat_interleave(2, dim=0).contiguous(), images_per_cond=1)
    assert torch.equal(out1, out)
    # a condition with a row stride wider than film_dim
    wide = torch.zeros((4, FILM_DIM + 64), device=DEV, dtype=torch.bfloat16)
    wide[:, :FILM_DIM] = lang
    assert torch.equal(film.forward(px, film_cond=wide[:, :FILM_DIM], images_per_cond=2), out)
    # a graph replay with a new condition equals an eager run, with the same launch count
    lang3 = _lang(4, FILM_DIM, 7)
    rep = film.forward(px, film_cond=lang3, images_per_cond=2).clone()
    n_graph = film.last_launch_count
    film.set_option("use_cuda_graph", 0)
    eager = film.forward(px, film_cond=lang3, images_per_cond=2)
    torch.cuda.synchronize()
    assert torch.equal(rep, eager) and film.last_launch_count == n_graph
    film.close()


@pytest.mark.gpu
def test_rejected_film_calls_leave_the_handle_working():
    import ctypes as C
    plain, film = _tower_pair("siglip", 4)
    lib = capi.load_library()
    px = _pixels(4, 8)
    lang = _lang(2, FILM_DIM, 9)
    good = film.forward(px, film_cond=lang, images_per_cond=2).clone()
    out = torch.empty_like(good)
    strides = (C.c_int64 * 4)(*px.stride())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    pxp, cp, op = C.c_void_p(px.data_ptr()), C.c_void_p(lang.data_ptr()), C.c_void_p(out.data_ptr())
    H = film.cfg.hidden
    assert lib.blurr_vit_forward_film(film.handle, st, 4, pxp, strides, cp, FILM_DIM, 3, op, H) == -1       # 3 does not divide 4
    assert lib.blurr_vit_forward_film(film.handle, st, 4, pxp, strides, cp, FILM_DIM, 0, op, H) == -1
    assert lib.blurr_vit_forward_film(film.handle, st, 4, pxp, strides, None, FILM_DIM, 2, op, H) == -1     # NULL cond
    assert lib.blurr_vit_forward_film(film.handle, st, 4, pxp, strides, cp, FILM_DIM - 64, 2, op, H) == -1  # cond_ld
    assert lib.blurr_vit_forward(film.handle, st, 4, pxp, strides, op, H) == -3                            # FiLM handle
    assert lib.blurr_vit_forward_film(plain.handle, st, 4, pxp, strides, cp, FILM_DIM, 2, op, H) == -3     # plain handle
    with pytest.raises(ValueError):
        film.forward(px)
    with pytest.raises(ValueError):
        plain.forward(px, film_cond=lang, images_per_cond=2)
    with pytest.raises(ValueError):
        film.forward(px, film_cond=lang, images_per_cond=3)
    assert torch.equal(film.forward(px, film_cond=lang, images_per_cond=2), good)
    cfg = openvla.VitShapedConfig(**{**film.cfg.__dict__, "film_dim": 100})
    with pytest.raises(capi.BlurrError):
        openvla.VitEncoder(cfg, DEV)
    cfg = openvla.VitShapedConfig(num_layers=1, hidden=256, num_heads=4, mlp_dim=512, film_dim=256)
    with pytest.raises(capi.BlurrError):
        openvla.VitEncoder(cfg, DEV)
    plain.close()
    film.close()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the FiLM policy on a shrunk stack
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def film_stack():
    B = 4
    towers = {}
    for film_dim in (0, 4096):
        d = openvla.dinov2_large_reg4_config(depth=3)
        s = openvla.siglip_so400m_config(depth=3)
        d.film_dim = s.film_dim = film_dim
        towers[film_dim] = (openvla.VitEncoder.synthetic(d, DEV, max_batch=2 * B, seed=3),
                            openvla.VitEncoder.synthetic(s, DEV, max_batch=2 * B, seed=4))
    proj = openvla.MlpProjector([2176, 8704, 4096, 4096], DEV, max_rows=2 * B * 256)
    g = torch.Generator(device=DEV).manual_seed(5)
    for i, (n_out, n_in) in enumerate(((8704, 2176), (4096, 8704), (4096, 4096))):
        proj.set_layer(i, (torch.randn((n_out, n_in), device=DEV, generator=g) * 0.02).to(torch.bfloat16),
                       (torch.randn(n_out, device=DEV, generator=g) * 0.02).to(torch.bfloat16))
    oft = openvla.oft_libero_config()
    cfg = openvla.openvla_oft_7b_config(oft)
    cfg.num_layers = 2
    dec = openvla.LlamaDecoder.from_state_dict(cfg, openvla.synthetic_llama_state_dict(cfg, DEV, 0), DEV, max_batch=B)
    head = openvla.L1RegressionHead.synthetic(oft, 4096, DEV, max_batch=B, seed=6)
    pp = openvla.ProprioProjector.synthetic(8, 4096, DEV, max_rows=B, seed=8)
    cam = torch.device("cuda", torch.cuda.current_device())        # the frames' device, index included
    pres = [openvla.ImagePreprocessor(480, 640, device=cam), openvla.ImagePreprocessor(256, 256, device=cam)]
    frames = [torch.randint(0, 256, (B, 480, 640, 3), device=DEV, dtype=torch.uint8, generator=g),
              torch.randint(0, 256, (B, 256, 256, 3), device=DEV, dtype=torch.uint8, generator=g)]
    backbones = {k: openvla.FusedVisionBackbone(*towers[k], proj) for k in towers}
    yield dict(backbones=backbones, proj=proj, dec=dec, head=head, pp=pp, pres=pres, frames=frames, oft=oft)
    torch.cuda.synchronize()
    dec.check()
    head.check()
    for m in (*pres, *towers[0], *towers[4096], proj, dec, head, pp):
        m.close()


def _policy(st, cameras, film):
    oft = st["oft"] if cameras == 2 else openvla.OftConfig()
    oft = openvla.OftConfig(**{**oft.__dict__, "use_film": film})
    pres = st["pres"] if cameras == 2 else st["pres"][0]
    return openvla.OftPolicy(pres, st["backbones"][4096 if film else 0], st["dec"], st["head"], oft,
                             proprio_projector=st["pp"] if cameras == 2 else None)


def _oracle_language(dec, lay):
    out = []
    for b in range(lay.ids.shape[0]):
        ids, mask = OF.oft_input_ids(lay.ids[b, :int(lay.text_lens[b])].tolist(), lay.n_rows)
        emb = dec.embed(torch.tensor(ids))[None]
        out.append(OF.language_embedding(emb, torch.tensor(mask, device=emb.device)[None]))
    return torch.cat(out)


RAW = np.random.default_rng(1).uniform(-1.5, 2.5, size=(4, 8))
PQ01, PQ99 = np.linspace(-1.0, 0.0, 8), np.linspace(0.5, 2.0, 8)


@pytest.mark.gpu
@pytest.mark.parametrize("cameras", [1, 2])
def test_film_policy_is_the_hand_composition_and_rows_match_batch_one(film_stack, cameras):
    st = film_stack
    pol = _policy(st, cameras, True)
    frames = st["frames"] if cameras == 2 else st["frames"][0]
    kw = dict(proprio=RAW, proprio_q01=PQ01, proprio_q99=PQ99) if cameras == 2 else {}
    rows = instructions([34, 12, 40, 25], 0)
    act, norm = pol.predict_action_chunk(frames, rows, Q01, Q99, return_normalized=True, **kw)
    # oracle mean -> towers -> projector -> forward_rows -> head
    P = 256 * cameras + (1 if cameras == 2 else 0)
    lay = openvla.oft_prompt_layout(rows, n_patches=P, cfg=pol.cfg)
    lang = _oracle_language(pol.decoder, lay)
    assert torch.equal(lang, openvla.film_language_embedding(pol.decoder, lay))
    px = pol.pixel_values(frames)
    px2 = px.reshape(4 * cameras, 6, 224, 224)
    patches = pol.backbone.forward(px2[:, :3], px2[:, 3:], film_cond=lang, images_per_cond=cameras)
    p = patches.reshape(4, 256 * cameras, 4096)
    if cameras == 2:
        state = torch.from_numpy(openvla.normalize_proprio(RAW, PQ01, PQ99).astype(np.float32)).to(DEV, torch.bfloat16)
        p = torch.cat([p, pol.proprio_projector.forward(state)[:, None]], dim=1)
    x = openvla.build_oft_embeds(pol.decoder, lay, p)
    n2 = pol.head.forward(pol.decoder.forward_rows(x, lay.seq_lens, lay.block_starts, lay.row_starts, lay.n_rows))
    assert torch.equal(norm, n2)
    scale = norm.abs().max().item()
    for b, r in enumerate(rows):
        f1 = [f[b] for f in frames] if cameras == 2 else frames[b]
        kw1 = dict(proprio=RAW[b], proprio_q01=PQ01, proprio_q99=PQ99) if cameras == 2 else {}
        _, n1 = pol.predict_action_chunk(f1, r[None].to(DEV), Q01, Q99, return_normalized=True, **kw1)
        d = (n1[0] - norm[b]).abs().max().item()
        print(f"cameras {cameras} row {b}: batch-1 vs batch-4 max_abs {d:.3e} (scale {scale:.3e})")
        assert d <= 0.05 * scale + 1e-2, (b, d, scale)


@pytest.mark.gpu
@pytest.mark.parametrize("cameras", [1, 2])
def test_instruction_moves_the_patch_rows_only_with_film(film_stack, cameras):
    st = film_stack
    frames = st["frames"] if cameras == 2 else st["frames"][0]
    film, plain = _policy(st, cameras, True), _policy(st, cameras, False)
    px = film.pixel_values(frames)
    state = film.proprio_state(RAW, PQ01, PQ99) if cameras == 2 else None
    P = 256 * cameras + (1 if cameras == 2 else 0)
    conds = [openvla.film_language_embedding(film.decoder, openvla.oft_prompt_layout(instructions([20] * 4, s), n_patches=P,
                                                                                   cfg=film.cfg)) for s in (0, 1)]
    a, b = (film.patch_embeds(px, state, c) for c in conds)
    torch.cuda.synchronize()
    assert not torch.equal(a[:, :256 * cameras], b[:, :256 * cameras])
    a0, b0 = (plain.patch_embeds(px, state, c) for c in conds)
    assert torch.equal(a0, b0) and torch.equal(a0, plain.patch_embeds(px, state))


@pytest.mark.gpu
def test_film_policy_rejects_mismatched_towers(film_stack):
    st = film_stack
    oft = openvla.OftConfig(use_film=True)
    with pytest.raises(ValueError, match="film_dim"):
        openvla.OftPolicy(st["pres"][0], st["backbones"][0], st["dec"], st["head"], oft)
    with pytest.raises(ValueError, match="film_dim"):
        openvla.OftPolicy(st["pres"][0], st["backbones"][4096], st["dec"], st["head"], openvla.OftConfig())
    pol = _policy(st, 1, True)
    with pytest.raises(ValueError, match="language"):
        pol.patch_embeds(pol.pixel_values(st["frames"][0]))
