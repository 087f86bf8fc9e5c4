"""End-to-end `sample` flow on the GPU with tiny models (reference src/bin/sample/main.rs:225-285): text -> Embedder ->
Conditioning -> Diffuser::sample_latent -> LatentDecoder::latent_to_image, plus the inpainting branch
(image_to_latent -> sample_latent_with_inpainting), each stage checked against the oracle chain."""
import os

import numpy as np
import pytest
import torch

from sdxl_b200 import (TINY, TINY_CLIP, TINY_OPEN_CLIP, TINY_VAE, ClipConfig, ClipTextEncoder, Diffuser, Embedder, LatentDecoder,
                       OpenClipTokenizer, UNetConfig, synth_weights)
from oracle import clip_oracle as CO
from oracle import tokenizer_oracle as TO
from oracle import unet_oracle as O
from oracle import vae_oracle as VO

pytestmark = pytest.mark.gpu
MINI = os.path.join(os.path.dirname(__file__), "golden", "mini_bpe")

# text encoders whose widths add up to the tiny UNet's context_dim (24 is not reachable with head dim 64): use a UNet
# config sized for them instead — context 128+192, label 64 + 6*256
CLIP_A = TINY_CLIP
CLIP_B = TINY_OPEN_CLIP
UNET = UNetConfig(adm_in_channels=CLIP_B.embed_dim + 6 * 256, model_channels=64, channel_mults=(1, 2, 4), transformer_depths=(0, 1, 1),
                  context_dim=CLIP_A.n_state + CLIP_B.n_state)


def rel_err(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def test_text_to_image_and_inpaint(ctx):
    wa, wb, wu, wv = (synth_weights(c, seed=s) for c, s in ((CLIP_A, 1), (CLIP_B, 2), (UNET, 3), (TINY_VAE, 0)))
    ea, eb = ClipTextEncoder(ctx, CLIP_A, wa), ClipTextEncoder(ctx, CLIP_B, wb)
    tok = OpenClipTokenizer(os.path.join(MINI, "mini_merges.txt"), os.path.join(MINI, "mini_vocab.txt"))
    emb = Embedder(ctx, ea, eb, tok, tok)
    dif = Diffuser(ctx, UNET, wu)
    vae = LatentDecoder(ctx, TINY_VAE, wv)
    text, res = "a photo of a cat", (64, 64)

    cond = emb.text_to_conditioning(text, res, (0, 0), res)
    noise = torch.randn(1, 4, 8, 8, generator=torch.Generator().manual_seed(0))
    latent = dif.sample_latent(cond, 5.0, 6, noise=noise)
    rgb = vae.latent_to_image(latent)
    assert rgb.shape == (1, 32, 32, 3) and rgb.dtype == torch.uint8

    # oracle chain on the same inputs
    otok = TO.OpenClipTokenizer(os.path.join(MINI, "mini_merges.txt"), os.path.join(MINI, "mini_vocab.txt"))
    oc = CO.text_to_conditioning(CLIP_A, O.to_f32(wa), CLIP_B, O.to_f32(wb), otok, otok, TO.tokenize_text, text, res, (0, 0), res)
    h16 = lambda t: t.to(torch.float16).float()  # Conditioning::convert
    ocond = O.OracleConditioning(context_full=h16(oc["context_full"]), unconditional_context_full=h16(oc["unconditional_context_full"]),
                                 channel_context=h16(oc["channel_context"]),
                                 unconditional_channel_context=h16(oc["unconditional_channel_context"]), resolution=res)
    from sdxl_b200 import alphas_cumprod
    olat = O.sample_latent(UNET, O.to_f32(wu), alphas_cumprod(), noise, ocond, 5.0, 6)
    e = rel_err(latent, olat)
    print("pipeline latent rel err", e)
    assert e <= 5e-3
    oimg = VO.latent_to_image(TINY_VAE, O.to_f32(wv), olat).numpy().astype(np.int32)
    diff = np.abs(rgb.cpu().numpy().astype(np.int32) - oimg)
    print("pipeline image max diff", diff.max(), "equal fraction", (diff == 0).mean())
    assert diff.max() <= 3 and (diff <= 1).mean() >= 0.99

    # inpainting branch: reference image -> latent -> sample_latent_with_inpainting (mask true = keep generated)
    ref_rgb = torch.randint(0, 256, (1, 32, 32, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(1))
    ref_lat = vae.image_to_latent(ref_rgb)
    assert ref_lat.shape == (1, 4, 8, 8)
    mask = torch.zeros(1, 4, 8, 8, dtype=torch.bool)
    mask[:, :, :3] = True
    out = dif.sample_latent_with_inpainting(cond, 5.0, 6, ref_lat, mask, seed=7)
    assert out.shape == (1, 4, 8, 8) and torch.isfinite(out).all()

    # the `sample` flow as one call (sdxl_b200.pipeline.sample == main.rs:128-285): same latent path -> same image; the inpainting
    # branch builds the mask from the crop window (here rows 0..24 px = latent rows 0..3 of 8: scale = 32 / 8 = 4)
    import sdxl_b200
    img2 = sdxl_b200.sample(emb, dif, vae, text, guidance=5.0, n_steps=6, resolution=res, noise=noise)
    assert torch.equal(img2, rgb)
    m = sdxl_b200.make_inpaint_mask((32, 32), (8, 8), None, None, None, 12)
    assert torch.equal(m, mask)
    img3 = sdxl_b200.sample(emb, dif, vae, text, guidance=5.0, n_steps=6, reference_rgb=ref_rgb, crop=(None, None, None, 12), seed=7)
    assert img3.shape == (1, 32, 32, 3) and img3.dtype == torch.uint8

    # the reference's shipped format: <name>.mpk + <name>.cfg -> Diffuser, bit-identical to the direct load
    import tempfile
    from sdxl_b200 import burn_record as BR
    with tempfile.TemporaryDirectory() as td:
        BR.save_diffuser(os.path.join(td, "diffuser"), UNET, wu)
        cfg2, w2 = BR.load_diffuser(os.path.join(td, "diffuser"))
    dif2 = Diffuser(ctx, cfg2, w2)
    assert torch.equal(dif2.sample_latent(cond, 5.0, 6, noise=noise), latent)
    dif2.close()
    # a whole model directory as the reference's `sample` reads it (embedder / diffuser / latent_decoder records) -> same image
    with tempfile.TemporaryDirectory() as td:
        BR.save_embedder(os.path.join(td, "embedder"), CLIP_A, wa, CLIP_B, wb)
        BR.save_diffuser(os.path.join(td, "diffuser"), UNET, wu)
        BR.save_latent_decoder(os.path.join(td, "latent_decoder"), TINY_VAE, wv)
        emb3, dif3, ref3, vae3 = sdxl_b200.load_models(ctx, td, tokenizers=(tok, tok))
    assert ref3 is None
    img4 = sdxl_b200.sample(emb3, dif3, vae3, text, guidance=5.0, n_steps=6, resolution=res, noise=noise)
    assert torch.equal(img4, rgb)
    for o in (emb3.clip, emb3.open_clip, dif3, vae3):
        o.close()
    for o in (ea, eb, dif, vae):
        o.close()


def test_unet_load_broadcast_two_gpus():
    """sdxl_unet_load_broadcast at world size 2 (one rank per GPU, torchrun): needs two devices."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29577", os.path.join(root, "tests", "mp", "load_broadcast.py")], cwd=root, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "LOAD_BROADCAST_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])


def _tiny_forward_inputs(seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(2, 4, 16, 16, generator=g), torch.randn(2, 5, TINY.context_dim, generator=g).half().float(),
            torch.randn(2, TINY.adm_in_channels, generator=g).half().float())


def test_two_contexts_two_threads():
    """include/sdxl_b200.h: "one sdxl_ctx per (device, stream) ... independent ctxs are fully concurrent". Two contexts on one
    device, two models, driven from two host threads at once (ctypes releases the GIL): every result equals the sequential one
    bit for bit (no process-global mutable state on the path)."""
    import threading
    import sdxl_b200
    ctxs = [sdxl_b200.Context(0) for _ in range(2)]
    ds = [Diffuser(c, TINY, synth_weights(TINY, seed=s)) for c, s in zip(ctxs, (0, 1))]
    ins = [_tiny_forward_inputs(10), _tiny_forward_inputs(11)]
    ts = [[999, 500, 1], [250, 749, 3]]
    seq = [[ds[i].unet_forward(ins[i][0], [t], ins[i][1], ins[i][2]).cpu() for t in ts[i]] for i in range(2)]
    out = [[None] * 3, [None] * 3]
    errors = []

    def work(i):
        try:
            torch.cuda.set_device(0)
            for rep in range(5):
                for k, t in enumerate(ts[i]):
                    out[i][k] = ds[i].unet_forward(ins[i][0], [t], ins[i][1], ins[i][2]).cpu()
        except Exception as ex:  # noqa: BLE001
            errors.append(ex)
    th = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errors, errors
    for i in range(2):
        for k in range(3):
            assert torch.equal(out[i][k], seq[i][k])
    for d in ds:
        d.close()
    for c in ctxs:
        c.close()


def test_two_devices_one_process():
    """Per-device launch state (shared-memory opt-in, SM count, cluster occupancy): a second device in the same process works."""
    import sdxl_b200
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    w = synth_weights(TINY, seed=0)
    x, c, y = _tiny_forward_inputs(12)
    ref = O.unet_forward(TINY, O.to_f32(w), x, torch.tensor([400]), c, y)
    for dev in (0, 1, 0):
        ctx = sdxl_b200.Context(dev)
        d = Diffuser(ctx, TINY, w)
        out = d.unet_forward(x, [400], c, y).cpu()
        e = float((out - ref).norm() / ref.norm())
        print(f"device {dev}: tiny forward rel err {e:.3e}")
        assert e < 2e-3
        d.close()
        ctx.close()
