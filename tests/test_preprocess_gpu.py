"""GPU: es3_preprocess_images (antialiased resize + normalise + pad) against torch on the CPU, the predictor's SAM2Transforms
path, and the stage-1 loops fed raw decoded images."""
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from efficientsam3_b200 import ops
from efficientsam3_b200.stage1.transforms import ImagePreprocessor, get_preprocess_shape
from helpers import rel_l2

pytestmark = pytest.mark.gpu

MEAN = torch.tensor([123.675, 116.28, 103.53]).view(3, 1, 1)
STD = torch.tensor([58.395, 57.12, 57.375]).view(3, 1, 1)


def _resize(x, size):
    """torch CPU antialiased bilinear of a [3,h,w] fp32 image.  With a width-1 input or output, torch's CPU kernel on an
    NCHW-contiguous tensor returns one value repeated down the column (torch 2.11); the channels-last tensor takes the
    path that evaluates the filter, so the reference uses it there."""
    x = x[None]
    if x.shape[-1] == 1 or size[1] == 1:
        x = x.contiguous(memory_format=torch.channels_last)
    return F.interpolate(x, size, mode="bilinear", align_corners=False, antialias=True)[0]


def _reference(img_chw, S):
    """The stage-1 loader chain: resize to the longest side, norm, pad (sa1b_dataset.py:163-171, 216-227)."""
    h, w = get_preprocess_shape(img_chw.shape[1], img_chw.shape[2], S)
    r = (_resize(img_chw.float(), (h, w)) - MEAN) / STD
    return F.pad(r, (0, S - w, 0, S - h)), (3, h, w)


def _image(h, w, seed, dtype=torch.uint8):
    g = torch.Generator().manual_seed(seed)
    x = torch.randint(0, 256, (3, h, w), generator=g, dtype=torch.uint8)
    return x if dtype == torch.uint8 else x.float() + torch.rand(3, h, w, generator=g)


def _check(got, imgs_chw, S, sizes):
    for i, img in enumerate(imgs_chw):
        ref, sz = _reference(img, S)
        assert tuple(sizes[i]) == sz
        g = got[i].cpu()
        err = (g - ref).abs().max().item()
        print(f"image {i} {tuple(img.shape)} -> {sz}: max |d| = {err:.2e}")
        assert err <= 1e-5, (i, err)
        assert torch.all(g[:, sz[1]:, :] == 0) and torch.all(g[:, :, sz[2]:] == 0)   # pad region: exact zeros


@pytest.mark.parametrize("h,w,S", [(1500, 2250, 1024), (1500, 2250, 1008), (2250, 1500, 1024), (6000, 4000, 1024), (17, 9, 1024),
                                   (768, 1024, 1024), (300, 1, 256)])
@pytest.mark.parametrize("layout", ["chw", "hwc"])
@pytest.mark.parametrize("dtype", [torch.uint8, torch.float32])
@pytest.mark.parametrize("where", ["host", "pinned", "cuda"])
def test_single_image_matches_torch(cuda, h, w, S, layout, dtype, where):
    if (h, w) == (6000, 4000) and (dtype == torch.float32 or where != "host"):
        pytest.skip("the largest image runs once, uint8 from the host (CPU reference time)")
    img = _image(h, w, h + w, dtype)
    x = img if layout == "chw" else img.permute(1, 2, 0).contiguous()
    if where == "cuda":
        x = x.to(cuda)
    elif where == "pinned":
        x = x.pin_memory()                # copied straight from its own memory
    elif layout == "hwc":
        x = x.numpy()                     # numpy HWC, as PIL / cv2 decode it
    got, sizes = ImagePreprocessor(S)([x])
    assert got.shape == (1, 3, S, S) and got.dtype == torch.float32 and got.is_cuda
    _check(got, [img], S, sizes)


def test_mixed_batch_one_call(cuda):
    """Five sizes, both layouts, both dtypes, pinned / pageable host and device images in one es3_preprocess_images call."""
    S = 512
    imgs = [_image(600, 900, 1), _image(900, 600, 2, torch.float32), _image(31, 47, 3), _image(512, 384, 4), _image(2000, 3, 5)]
    inputs = [imgs[0].pin_memory(), imgs[1].permute(1, 2, 0).contiguous().numpy(), imgs[2].to(cuda), imgs[3].permute(1, 2, 0).to(cuda),
              imgs[4].permute(1, 2, 0).contiguous()]
    n0 = ops.launch_count
    got, sizes = ImagePreprocessor(S)(inputs)
    assert ops.launch_count - n0 == ops.KERNELS_PER_CALL["es3_preprocess_images"]
    _check(got, imgs, S, sizes)


def test_strided_cuda_view_and_out_buffer(cuda):
    """A crop of a larger device image is read in place through its strides, into a caller's buffer."""
    big = _image(700, 900, 7).to(cuda)
    crop = big[:, 50:650, 100:850]
    out = torch.full((1, 3, 320, 320), 7.0, device=cuda)
    got, sizes = ImagePreprocessor(320)([crop], out=out)
    assert got.data_ptr() == out.data_ptr()
    _check(got, [crop.cpu().contiguous()], 320, sizes)


@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
def test_predictor_to_input_matches_sam2_transforms(cuda, dtype):
    """ToTensor -> Resize((S,S)) antialias -> Normalize(0.5, 0.5) on the CPU; set_image_batch is one preprocessing call."""
    from efficientsam3_b200.model.sam1_task import SAM3InteractiveImagePredictor
    S = 1008
    dev_model = types.SimpleNamespace(image_size=S, no_mem_embed=torch.zeros(1, device=cuda), _features=None)
    pred = SAM3InteractiveImagePredictor(dev_model)
    rng = np.random.default_rng(0)
    arrs = [rng.integers(0, 256, size=hw + (3,)).astype(np.uint8) for hw in [(300, 420), (1500, 1100), (1008, 1008)]]
    if dtype == np.float32:
        arrs = [(a / 255.0).astype(np.float32) for a in arrs]
    for a in arrs:
        x, hw = pred._to_input(a)
        t = torch.from_numpy(a).permute(2, 0, 1).float()
        if dtype == np.uint8:
            t = t / 255.0
        ref = (_resize(t, (S, S)) - 0.5) / 0.5
        err = (x.cpu() - ref).abs().max().item()
        print(f"predictor {a.shape} {a.dtype}: max |d| = {err:.2e}")
        assert hw == a.shape[:2] and x.shape == (3, S, S) and err <= 1e-5
    calls = []
    dev_model.set_image_batch = lambda x: calls.append(x.shape)
    n0 = ops.launch_count
    pred.set_image_batch(arrs)
    assert ops.launch_count - n0 == ops.KERNELS_PER_CALL["es3_preprocess_images"]
    assert calls == [(3, 3, S, S)] and pred._orig_hw == [a.shape[:2] for a in arrs]


# ------------------------------------------------------------------------------------------ stage 1
def _student(img, embed, seed=3):
    from types import SimpleNamespace as NS
    from efficientsam3_b200.stage1.model import build_image_student_model
    from oracle.weights import fill_state_dict
    cfg = NS(MODEL=NS(BACKBONE="efficientvit_b1"), DATA=NS(IMG_SIZE=img), DISTILL=NS(EMBED_DIM=1024, EMBED_SIZE=embed))
    m = build_image_student_model(cfg)
    m.load_state_dict(fill_state_dict(m.state_dict(), seed))
    return m


def _raw_batch(seed, B=2):
    return [_image(300 + 37 * i, 420 - 29 * i, seed * 10 + i) for i in range(B)]


def test_eval_embedding_of_raw_images(cuda):
    img, embed = 256, 16
    m = _student(img, embed).to(cuda).eval()
    raw = _raw_batch(1)
    x, sizes = ImagePreprocessor(img)(raw)
    ref_x = torch.stack([_reference(r, img)[0] for r in raw]).to(cuda)
    print(f"input max |d| = {(x - ref_x).abs().max().item():.2e}")
    # the strict (fp32) forward (measured on a B200: 8e-7).  The bf16 forward of this random-weight fixture is deterministic
    # (the same input twice is bit-identical) but inputs ~1e-7 apart move it by ~5e-3 rel-L2, about its own error against
    # strict (~7e-3), so it gets the bf16 tolerance
    with ops.strict_precision():
        e, ref = m(x).clone(), m(ref_x).clone()
    assert rel_l2(e.cpu(), ref.cpu()) <= 1e-3
    e16, ref16, again16 = m(x).clone(), m(ref_x).clone(), m(ref_x).clone()
    print(f"strict rel-L2 {rel_l2(e.cpu(), ref.cpu()):.2e}; bf16 rel-L2 {rel_l2(e16.cpu(), ref16.cpu()):.2e} "
          f"(same input twice: {rel_l2(again16.cpu(), ref16.cpu()):.2e}; bf16 vs strict {rel_l2(ref16.cpu(), ref.cpu()):.2e})")
    assert rel_l2(e16.cpu(), ref16.cpu()) <= 2e-2


def test_train_one_epoch_with_raw_samples(cuda):
    from types import SimpleNamespace as NS
    from efficientsam3_b200.stage1.optim import FlatAdamW
    from efficientsam3_b200.stage1.train import train_one_epoch
    img, embed, iters = 256, 16, 2
    cfg = NS(TRAIN=NS(EVAL_BN_WHEN_TRAINING=True, ACCUMULATION_STEPS=1, EPOCHS=1, WARMUP_EPOCHS=0, MIN_LR=1e-6, WARMUP_LR=1e-7,
                      CLIP_GRAD=5.0), DISTILL=NS(EMBED_DIM=1024, EMBED_SIZE=embed, COSINE=1.0), DATA=NS(IMG_SIZE=img))
    raws = [_raw_batch(10 + i) for i in range(iters)]
    teach = [[(np.random.RandomState(10 * i + b).randn(1024 * embed * embed) * 0.5).astype(np.float16) for b in range(2)]
             for i in range(iters)]

    def run(loader, **kw):
        m = _student(img, embed).to(cuda)
        opt = FlatAdamW(m, lr=1e-4, weight_decay=0.01)
        return torch.stack(train_one_epoch(cfg, m, loader, opt, epoch=0, **kw)).cpu()

    raw_loader = [((raws[i], {}), (teach[i], [i, i])) for i in range(iters)]
    ref_loader = []
    for i in range(iters):
        pairs = [_reference(r, img) for r in raws[i]]
        ref_loader.append((([p[0] for p in pairs], {"img_size_before_pad": [p[1] for p in pairs]}), (teach[i], [i, i])))
    got = run(raw_loader, preprocess=ImagePreprocessor(img))
    ref = run(ref_loader)
    print("losses", got.tolist(), ref.tolist())
    torch.testing.assert_close(got, ref, rtol=1e-3, atol=0)


def test_save_embeddings_with_raw_samples(cuda, tmp_path):
    from efficientsam3_b200.stage1 import embeddings as E
    img, embed = 256, 16
    m = _student(img, embed).to(cuda)
    raws = [_raw_batch(20 + i) for i in range(2)]
    keys = [[f"k{b}_{i}" for i in range(2)] for b in range(2)]
    seeds = [np.array([b, b + 10], dtype=np.int32) for b in range(2)]
    # the strict (fp32) forward: inputs that agree to ~1e-6 give embeddings that agree far below the store's fp16 rounding
    with ops.strict_precision():
        E.save_embeddings_one_epoch(m, [((raws[b], None), (keys[b], seeds[b])) for b in range(2)], str(tmp_path / "a"),
                                    preprocess=ImagePreprocessor(img))
        E.save_embeddings_one_epoch(m, [(([_reference(r, img)[0] for r in raws[b]], None), (keys[b], seeds[b])) for b in range(2)],
                                    str(tmp_path / "b"))
    ra = E.EmbeddingStoreReader(str(tmp_path / "a"), E.item_size(1024, embed * embed))
    rb = E.EmbeddingStoreReader(str(tmp_path / "b"), E.item_size(1024, embed * embed))
    for b in range(2):
        for k in keys[b]:
            (sa, ea), (sb, eb) = ra.read_embedding(k), rb.read_embedding(k)
            assert sa == sb
            # one fp16 step apart at most (a value next to a rounding boundary may round either way), plus the fp32 forward's
            # response to inputs that differ by ~1e-7, which matters only for values near zero
            ea, eb = ea.astype(np.float32), eb.astype(np.float32)
            tol = np.spacing(np.abs(eb).astype(np.float16)).astype(np.float32) + 1e-5 * np.abs(eb).max()
            assert np.all(np.abs(ea - eb) <= tol), np.abs(ea - eb).max()


def test_rotating_out_buffers_under_cuda_graphs(cuda):
    img, embed = 256, 16
    m = _student(img, embed).to(cuda).eval()
    pre = ImagePreprocessor(img)
    bufs = [torch.empty(2, 3, img, img, device=cuda) for _ in range(2)]
    batches = [_raw_batch(30 + i) for i in range(4)]
    ref = [m.forward_uncaptured(pre(b)[0]).clone() for b in batches]
    m.enable_cuda_graphs()
    try:
        for i, b in enumerate(batches):
            x, _ = pre(b, out=bufs[i % 2])
            assert x.data_ptr() == bufs[i % 2].data_ptr()
            e = m(x)
            torch.testing.assert_close(e, ref[i], rtol=0, atol=0)
    finally:
        m.enable_cuda_graphs(False)
