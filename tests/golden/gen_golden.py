"""Generate golden fixtures by running the UNMODIFIED reference modules (CPU fp32) in the build container.

    python tests/golden/gen_golden.py [evm|teacher|decoder|all]

Needs /root/reference (absent on the GPU box -- fixtures are committed).  Weights come from
oracle.weights.fill_state_dict(seed) so they are reproducible without being stored.
"""
from __future__ import annotations

import os
import sys
from types import SimpleNamespace as NS

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "ref_shim"))

import install  # noqa: E402  (oracle/ref_shim/install.py)

install.install()
from oracle.weights import fill_state_dict  # noqa: E402

torch.set_grad_enabled(False)


def keyshapes(sd):
    return np.array([f"{k}|{','.join(map(str, v.shape))}|{str(v.dtype).replace('torch.', '')}" for k, v in sd.items()])


def stats(t):
    t = t.double()
    return np.array([t.mean().item(), t.abs().mean().item(), t.std().item()])


def gen_student(backbone, tag, img, embed, seed_w, seed_x, batch=1):
    import model as stage1_model  # /root/reference/stage1/model.py

    cfg = NS(MODEL=NS(BACKBONE=backbone), DATA=NS(IMG_SIZE=img), DISTILL=NS(EMBED_DIM=1024, EMBED_SIZE=embed))
    m = stage1_model.build_image_student_model(cfg).eval()
    sd = fill_state_dict(m.state_dict(), seed_w)
    m.load_state_dict(sd)
    m.train(); m.eval()   # TinyViT's Attention caches `ab` (bias table) inside train(False): refresh after loading weights
    x = torch.randn(batch, 3, img, img, generator=torch.Generator().manual_seed(seed_x))
    out = m(x)
    extra = {}
    if backbone.startswith("efficientvit"):
        st = m.backbone.model(x)
        for k in ("stage0", "stage1", "stage2", "stage3", "stage4"):
            extra[f"stats_{k}"] = stats(st[k])
            extra[f"shape_{k}"] = np.array(st[k].shape)
    path = os.path.join(HERE, f"{tag}.npz")
    np.savez_compressed(path, out=out.numpy(), keys=keyshapes(m.state_dict()), img=img, embed=embed, seed_w=seed_w,
                        seed_x=seed_x, batch=batch, n_params=sum(p.numel() for p in m.parameters()), **extra)
    print(tag, "out", tuple(out.shape), "absmean %.4f" % out.abs().mean().item(), "->", path,
          "%.1f KB" % (os.path.getsize(path) / 1024))


def _ref_loss_functions():
    """build_valid_mask / masked_mse / masked_cosine_loss, executed from the reference's own source
    (stage1/train_image_encoder_stage1.py:271-307).  The script itself is not importable here (yacs, timm.scheduler, ...),
    so only these three function definitions are compiled from its AST -- nothing is copied into the repo."""
    import ast
    import torch.nn.functional as F
    path = "/root/reference/stage1/train_image_encoder_stage1.py"
    tree = ast.parse(open(path).read())
    ns = {"torch": torch, "F": F}
    want = ("build_valid_mask", "masked_mse", "masked_cosine_loss")
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in want:
            exec(compile(ast.Module([node], []), path, "exec"), ns)
    return tuple(ns[k] for k in want)


def gen_student_train(backbone, tag, img, embed, seed_w, seed_x, batch=2, cosine=1.0):
    """One stage-1 training iteration of the UNMODIFIED reference student in .train() (batch-statistics BatchNorm), fp64:
    preds = model(x); loss = masked_mse + COSINE * masked_cosine (the reference's own functions); loss.backward().
    Records the output, the losses, every parameter gradient (norm, sum, first 4 entries) and the updated BN buffers.
    fp64 because the random-weight batch-BN network is ill-conditioned in fp32 (2.5e-3 between fp32 and fp64 gradients)."""
    import model as stage1_model
    build_valid_mask, masked_mse, masked_cosine_loss = _ref_loss_functions()
    cfg = NS(MODEL=NS(BACKBONE=backbone), DATA=NS(IMG_SIZE=img), DISTILL=NS(EMBED_DIM=1024, EMBED_SIZE=embed))
    m = stage1_model.build_image_student_model(cfg)
    m.load_state_dict(fill_state_dict(m.state_dict(), seed_w))
    m = m.double().train()
    g = torch.Generator().manual_seed(seed_x)
    x = torch.randn(batch, 3, img, img, generator=g).double()
    teacher = torch.randn(batch, 1024, embed, embed, generator=g).double()
    sizes = [(3, img, img * 3 // 4) if i % 2 == 0 else (3, img * 2 // 3, img) for i in range(batch)]
    with torch.enable_grad():
        out = m(x)
        mask = build_valid_mask(cfg, sizes, out.shape, out.device).double()
        mse = masked_mse(out, teacher, mask)
        cos = masked_cosine_loss(out, teacher, mask)
        loss = mse + cosine * cos
        loss.backward()
    names, gstat = [], []
    for k, p in m.named_parameters():
        gr = p.grad.reshape(-1)
        first = torch.zeros(4, dtype=torch.float64)
        first[:min(4, gr.numel())] = gr[:4]
        names.append(k)
        gstat.append(torch.cat([gr.norm().reshape(1), gr.sum().reshape(1), first]).numpy())
    bufs = {k: v.detach().numpy() for k, v in m.state_dict().items() if "running_" in k and ("input_stem" in k or "head." in k or "stages.3.op_list.4" in k)}
    path = os.path.join(HERE, f"{tag}.npz")
    np.savez_compressed(path, out=out.detach()[:, ::8].numpy(), loss=np.array([loss.item(), mse.item(), cos.item()]), grad_names=np.array(names),
                        grad_stats=np.stack(gstat), buf_names=np.array(list(bufs.keys())), **{f"buf{i}": v for i, v in enumerate(bufs.values())},
                        keys=keyshapes(m.float().state_dict()), img=img, embed=embed, seed_w=seed_w, seed_x=seed_x, batch=batch, cosine=cosine,
                        sizes=np.array(sizes))
    print(tag, "loss %.6f" % loss.item(), "->", path, "%.1f KB" % (os.path.getsize(path) / 1024))


VIT_SMALL = dict(img_size=112, pretrain_img_size=56, patch_size=14, embed_dim=256, depth=4, num_heads=4, mlp_ratio=4.625,
                 window_size=4, global_att_blocks=(1, 3))


def gen_vit(tag, cfg, seed_w, seed_x, batch):
    """Reference ViT class (sam3/sam3/model/vitdet.py) in the SAM3 configuration family, small dims."""
    from sam3.model.vitdet import ViT

    m = ViT(norm_layer="LayerNorm", drop_path_rate=0.1, qkv_bias=True, use_abs_pos=True, tile_abs_pos=True,
            rel_pos_blocks=(), use_rope=True, use_interp_rope=True, pretrain_use_cls_token=True, retain_cls_token=False,
            ln_pre=True, ln_post=False, return_interm_layers=False, bias_patch_embed=False, **cfg).eval()
    sd = fill_state_dict(m.state_dict(), seed_w)
    m.load_state_dict(sd)
    x = torch.randn(batch, 3, cfg["img_size"], cfg["img_size"], generator=torch.Generator().manual_seed(seed_x))
    out = m(x)[-1]
    path = os.path.join(HERE, f"{tag}.npz")
    np.savez_compressed(path, out=out.numpy(), keys=keyshapes(m.state_dict()), seed_w=seed_w, seed_x=seed_x, batch=batch,
                        n_params=sum(p.numel() for p in m.parameters()), cfg=np.array(repr(cfg)))
    print(tag, "out", tuple(out.shape), "absmean %.4f" % out.abs().mean().item(), "->", path,
          "%.1f KB" % (os.path.getsize(path) / 1024))


def build_ref_sam_heads(E, S):
    """PromptEncoder + MaskDecoder exactly as Sam3TrackerBase._build_sam_heads builds them (:179-218)."""
    from sam3.sam.mask_decoder import MaskDecoder
    from sam3.sam.prompt_encoder import PromptEncoder
    from sam3.sam.transformer import TwoWayTransformer

    pe = PromptEncoder(embed_dim=256, image_embedding_size=(E, E), input_image_size=(S, S), mask_in_chans=16).eval()
    md = MaskDecoder(num_multimask_outputs=3, transformer=TwoWayTransformer(depth=2, embedding_dim=256, mlp_dim=2048, num_heads=8),
                     transformer_dim=256, iou_head_depth=3, iou_head_hidden_dim=256, use_high_res_features=True,
                     iou_prediction_use_sigmoid=True, pred_obj_scores=True, pred_obj_scores_mlp=True,
                     use_multimask_token_for_obj_ptr=True).eval()
    return pe, md


def sam_heads_inputs(B, E, S, seed):
    g = torch.Generator().manual_seed(seed)
    feat = torch.randn(B, 256, E, E, generator=g)
    f288 = torch.randn(B, 256, 4 * E, 4 * E, generator=g)
    f144 = torch.randn(B, 256, 2 * E, 2 * E, generator=g)
    coords = torch.rand(B, 1, 2, generator=g) * S
    labels = torch.ones(B, 1, dtype=torch.int32)
    return feat, f288, f144, coords, labels


def gen_sam_heads(tag, E, S, B, seed_pe, seed_md, seed_x):
    pe, md = build_ref_sam_heads(E, S)
    sd_pe = fill_state_dict(pe.state_dict(), seed_pe)
    sd_md = fill_state_dict(md.state_dict(), seed_md)
    pe.load_state_dict(sd_pe)
    md.load_state_dict(sd_md)
    feat, f288, f144, coords, labels = sam_heads_inputs(B, E, S, seed_x)
    hr = [md.conv_s0(f288), md.conv_s1(f144)]
    sp, de = pe(points=(coords, labels), boxes=None, masks=None)
    dpe = pe.get_dense_pe()
    out = {}
    for mm in (True, False):
        m, iou, tok, obj = md(image_embeddings=feat, image_pe=dpe, sparse_prompt_embeddings=sp, dense_prompt_embeddings=de,
                              multimask_output=mm, repeat_image=False, high_res_features=hr)
        sfx = "mm" if mm else "single"
        out.update({f"masks_{sfx}": m.numpy(), f"iou_{sfx}": iou.numpy(), f"tok_{sfx}": tok.numpy(), f"obj_{sfx}": obj.numpy()})
    q, k = md.transformer(feat, dpe.expand(B, -1, -1, -1), torch.cat([sp, sp], dim=1))
    path = os.path.join(HERE, f"{tag}.npz")
    np.savez_compressed(path, sparse=sp.numpy(), dense_pe=dpe.numpy()[:, :, ::4, ::4], twoway_q=q.numpy(),
                        twoway_k_stats=stats(k), keys_pe=keyshapes(pe.state_dict()), keys_md=keyshapes(md.state_dict()),
                        E=E, S=S, B=B, seed_pe=seed_pe, seed_md=seed_md, seed_x=seed_x, **out)
    print(tag, "masks", out["masks_mm"].shape, "absmean %.4f" % np.abs(out["masks_mm"]).mean(), "obj", out["obj_mm"].ravel(),
          "->", path, "%.1f KB" % (os.path.getsize(path) / 1024))


def gen_sam_prompts(tag, E, S, seed_pe, seed_md, seed_x):
    """Box + point + mask prompts, several prompts on ONE image (repeat_image=True), and SAM2Transforms.postprocess_masks
    (hole / sprinkle filling through the reference's CPU connected-components backend + resize) -- the pieces of
    SAM3InteractiveImagePredictor._predict (sam1_task_predictor.py:329-430) beyond the single-point path."""
    from sam3.model.utils.sam1_utils import SAM2Transforms

    pe, md = build_ref_sam_heads(E, S)
    pe.load_state_dict(fill_state_dict(pe.state_dict(), seed_pe))
    md.load_state_dict(fill_state_dict(md.state_dict(), seed_md))
    g = torch.Generator().manual_seed(seed_x)
    P = 3
    feat = torch.randn(1, 256, E, E, generator=g)
    f288 = torch.randn(1, 256, 4 * E, 4 * E, generator=g)
    f144 = torch.randn(1, 256, 2 * E, 2 * E, generator=g)
    coords = torch.rand(P, 2, 2, generator=g) * S
    labels = torch.tensor([[1, 0], [1, 1], [0, 1]], dtype=torch.int32)
    xy0 = torch.rand(P, 2, generator=g) * S * 0.5
    boxes = torch.cat([xy0, xy0 + 8 + torch.rand(P, 2, generator=g) * S * 0.4], dim=1)
    mask_in = torch.randn(P, 1, 4 * E, 4 * E, generator=g) * 4
    hr = [md.conv_s0(f288), md.conv_s1(f144)]
    dpe = pe.get_dense_pe()
    out = {}
    # (a) PromptEncoder.forward with a direct `boxes` argument (no padding point) and a mask
    sp_a, de_a = pe(points=(coords, labels), boxes=boxes, masks=mask_in)
    out["sparse_pts_boxes"], out["dense_mask0"] = sp_a.numpy(), de_a.numpy()[:1]     # first prompt's map + stats of all
    out["dense_mask_stats"] = np.stack([stats(de_a[i]) for i in range(P)])
    # (b) the predictor's merge: boxes in front as label-2/3 points, boxes=None -> padding point appended
    cc = torch.cat([boxes.reshape(-1, 2, 2), coords], dim=1)
    cl = torch.cat([torch.tensor([[2, 3]], dtype=torch.int32).repeat(P, 1), labels], dim=1)
    sp_b, de_b = pe(points=(cc, cl), boxes=None, masks=mask_in)
    out["sparse_merged"] = sp_b.numpy()
    for mm in (True, False):
        m, iou, tok, obj = md(image_embeddings=feat, image_pe=dpe, sparse_prompt_embeddings=sp_b, dense_prompt_embeddings=de_b,
                              multimask_output=mm, repeat_image=True, high_res_features=hr)
        sfx = "mm" if mm else "single"
        out.update({f"masks_{sfx}": m.numpy(), f"iou_{sfx}": iou.numpy(), f"obj_{sfx}": obj.numpy()})
    # (c) postprocess_masks: holes <= 12 px filled (+10), sprinkles <= 5 px removed (-10), bilinear to a non-square size
    tr = SAM2Transforms(resolution=S, mask_threshold=0.0, max_hole_area=12.0, max_sprinkle_area=5.0)
    low = torch.from_numpy(out["masks_mm"]).clone()
    gm = torch.Generator().manual_seed(seed_x + 1)
    low = low + torch.randn(low.shape, generator=gm) * low.abs().mean() * 1.5       # speckle: many small components
    post = tr.postprocess_masks(low, (50, 70))
    tr0 = SAM2Transforms(resolution=S, mask_threshold=0.0, max_hole_area=0.0, max_sprinkle_area=0.0)
    plain = tr0.postprocess_masks(low, (50, 70))
    assert not torch.equal(post, plain), "hole filling did not change anything: fixture would not pin it"
    out["post_in"], out["post_out"] = low.numpy(), post.numpy()
    out["post_changed_px"] = int(((post > 0) != (plain > 0)).sum())
    path = os.path.join(HERE, f"{tag}.npz")
    np.savez_compressed(path, E=E, S=S, P=P, seed_pe=seed_pe, seed_md=seed_md, seed_x=seed_x, keys_pe=keyshapes(pe.state_dict()),
                        keys_md=keyshapes(md.state_dict()), **out)
    print(tag, "masks", out["masks_mm"].shape, "changed px", out["post_changed_px"], "->", path, "%.1f KB" % (os.path.getsize(path) / 1024))


def gen_neck(tag, dim, d_model, hw, B, seed_w, seed_x):
    from sam3.model.necks import Sam3DualViTDetNeck

    class _Trunk(torch.nn.Module):          # test double: the neck only needs channel_list and a callable trunk
        channel_list = [dim]

        def forward(self, x):
            return [x]

    m = Sam3DualViTDetNeck(trunk=_Trunk(), position_encoding=lambda t: torch.zeros_like(t), d_model=d_model,
                           scale_factors=[4.0, 2.0, 1.0, 0.5], add_sam2_neck=True).eval()
    sd = fill_state_dict(m.state_dict(), seed_w)
    m.load_state_dict(sd)
    x = torch.randn(B, dim, hw, hw, generator=torch.Generator().manual_seed(seed_x))
    s3, _, s2, _ = m(x)
    path = os.path.join(HERE, f"{tag}.npz")
    np.savez_compressed(path, keys=keyshapes(m.state_dict()), dim=dim, d_model=d_model, hw=hw, B=B, seed_w=seed_w, seed_x=seed_x,
                        **{f"sam3_{i}": t.numpy() for i, t in enumerate(s3)}, **{f"sam2_{i}": t.numpy() for i, t in enumerate(s2)})
    print(tag, [tuple(t.shape) for t in s3], "->", path, "%.1f KB" % (os.path.getsize(path) / 1024))


def gen_store(tag, n_rank=2, embed_dim=8, num_embedding=6):
    """A tiny teacher-embedding store written by the reference's TxtManager (stage1/data/augmentation/manager.py),
    including a duplicate key (first occurrence wins).  Committed as a directory of keys.txt / values.bin files."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_manager", "/root/reference/stage1/data/augmentation/manager.py")
    ref_manager = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_manager)   # the file on its own: the package __init__ pulls in mmengine
    TxtManager = ref_manager.TxtManager

    path = os.path.join(HERE, tag)
    if os.path.isdir(path):
        import shutil
        shutil.rmtree(path)
    isz = embed_dim * 2 * num_embedding + 4
    rng = np.random.default_rng(99)
    for r in range(n_rank):
        m = TxtManager(path, isz, r)
        for i in range(4):
            key = f"sa_{r}_{i:03d}"
            emb = rng.standard_normal(embed_dim * num_embedding).astype(np.float16)
            m.write(key, np.int32(1000 * r + i).tobytes() + emb.tobytes())
            if i == 1:   # duplicate: must be ignored
                m.write(key, np.int32(-1).tobytes() + (emb * 0).tobytes())
        m.writer.__del__()
        m.writer.worker = None
    print(tag, sorted(os.listdir(path)))


def gen_student_neck(tag="student_neck_evm_160", img=160, seed_w=81, seed_x=82):
    """EfficientSAM3 image encoder as the reference builds it (`_create_student_vision_backbone`, model_builder.py:789-941):
    state_dict signatures of all nine student variants (sha256 of the key|shape|dtype list) and, for efficientvit b1 with
    re-randomised weights, the FPN outputs of both branches on one small image (strided sub-samples + statistics)."""
    import hashlib
    from sam3 import model_builder as MB
    sigs = {}
    for bt, names in [("efficientvit", ["b0", "b1", "b2"]), ("repvit", ["m0.9", "m1.1", "m2.3"]), ("tinyvit", ["5m", "11m", "21m"])]:
        for mn in names:
            m = MB._create_student_vision_backbone(bt, mn, enable_inst_interactivity=True)
            ks = keyshapes(m.state_dict())
            sigs[f"{bt}:{mn}"] = f"{len(ks)}:{hashlib.sha256(chr(10).join(ks).encode()).hexdigest()}"
    m = MB._create_student_vision_backbone("efficientvit", "b1", enable_inst_interactivity=True).eval()
    m.load_state_dict(fill_state_dict(m.state_dict(), seed_w))
    x = torch.randn(1, 3, img, img, generator=torch.Generator().manual_seed(seed_x))
    s3, _, s2, _ = m(x)
    rec = {}
    for name, outs in (("sam3", s3), ("sam2", s2)):
        for i, t in enumerate(outs):
            rec[f"{name}_{i}_shape"] = np.array(t.shape)
            rec[f"{name}_{i}_stats"] = stats(t)
            rec[f"{name}_{i}_sub"] = t[:, ::16, ::(6 if t.shape[-1] > 36 else 3), ::(6 if t.shape[-1] > 36 else 3)].numpy()
    path = os.path.join(HERE, f"{tag}.npz")
    np.savez_compressed(path, keys=keyshapes(m.state_dict()), sig_names=np.array(list(sigs.keys())), sig_values=np.array(list(sigs.values())),
                        img=img, seed_w=seed_w, seed_x=seed_x, **rec)
    print(tag, "->", path, "%.1f KB" % (os.path.getsize(path) / 1024))


def gen_sampler_cases():
    """Index plans of the reference's MyDistributedSampler (stage1/data/sampler.py) -> sampler_cases.json."""
    import importlib.util
    import json
    spec = importlib.util.spec_from_file_location("ref_sampler", "/root/reference/stage1/data/sampler.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    cases = []
    for n, world, kw in [(10, 4, {}), (256, 8, {}), (7, 2, dict(drop_last=True)), (13, 4, dict(shuffle=False)), (5, 8, {}), (3, 8, {}),
                         (12, 3, dict(pair=True)), (11, 2, dict(pair=True)), (9, 4, dict(padding=False)), (100, 8, dict(seed=5))]:
        for epoch in (0, 3):
            for rank in range(world):
                s = mod.MyDistributedSampler(list(range(n)), num_replicas=world, rank=rank, **kw)
                s.set_epoch(epoch)
                cases.append(dict(n=n, world=world, rank=rank, epoch=epoch, kw=kw, indices=list(iter(s)), length=len(s)))
    json.dump(cases, open(os.path.join(HERE, "sampler_cases.json"), "w"))
    print("sampler_cases.json", len(cases), "cases")


CONVERT_STUDENT = {"module.backbone.model.input_stem.op_list.0.conv.weight": 0.0, "student_trunk.head.0.weight": 1.0,
                   "detector.backbone.vision_backbone.trunk.model.head.3.bias": 2.0, "head.1.running_mean": 3.0}
CONVERT_SAM3 = {"detector.backbone.vision_backbone.trunk.blocks.0.attn.qkv.weight": 9.0,
                "detector.backbone.vision_backbone.convs.0.conv_1x1.weight": 4.0, "detector.transformer.decoder.x": 5.0,
                "tracker.sam_mask_decoder.y": 6.0, "detector.backbone.language_backbone.z": 7.0}
CONVERT_SKIP = ["detector.backbone.language_backbone"]


def gen_convert():
    """The reference's stage1/convert_image_encoder_weights_stage1.py, run as a script on two tiny synthetic checkpoints
    (one-element tensors) -> convert_merge.json: the inputs and the merged checkpoint's keys in order with their values."""
    import json
    import subprocess
    import tempfile
    script = os.path.join(install.REFERENCE_ROOT, "stage1", "convert_image_encoder_weights_stage1.py")
    with tempfile.TemporaryDirectory() as tmp:
        s, t, o = (os.path.join(tmp, n) for n in ("s.pth", "t.pth", "o.pth"))
        torch.save({"model": {k: torch.full((1,), v) for k, v in CONVERT_STUDENT.items()}}, s)
        torch.save({"model": {k: torch.full((1,), v) for k, v in CONVERT_SAM3.items()}}, t)
        cmd = [sys.executable, script, "--student-ckpt", s, "--sam3-ckpt", t, "--output", o]
        for p in CONVERT_SKIP:
            cmd += ["--skip-teacher-prefix", p]
        subprocess.run(cmd, check=True, capture_output=True)
        merged = torch.load(o, weights_only=False)["model"]
    rec = {"student": list(CONVERT_STUDENT.items()), "sam3": list(CONVERT_SAM3.items()), "skip_teacher_prefixes": CONVERT_SKIP,
           "merged": [[k, float(v)] for k, v in merged.items()]}
    json.dump(rec, open(os.path.join(HERE, "convert_merge.json"), "w"), indent=1)
    print("convert_merge.json", len(rec["merged"]), "keys")


def main(which):
    if which in ("convert", "all"):
        gen_convert()
    if which in ("sampler", "all"):
        gen_sampler_cases()
    if which in ("student_neck", "all"):
        gen_student_neck()
    if which in ("train", "all"):
        gen_student_train("efficientvit_b1", "evm_train_160", img=160, embed=12, seed_w=71, seed_x=72)
    if which in ("tvm", "all"):
        gen_student("tiny_vit_11m", "tvm_160", img=160, embed=12, seed_w=61, seed_x=62, batch=1)
    if which in ("store", "all"):
        gen_store("store_small")
    if which in ("variants", "all"):
        # the other six names build_image_student_model accepts (stage1/model.py:386-417); small embeds keep the files small
        gen_student("repvit_m0_9", "rv_m0_9_128", img=128, embed=6, seed_w=71, seed_x=72, batch=1)
        gen_student("repvit_m2_3", "rv_m2_3_128", img=128, embed=6, seed_w=73, seed_x=74, batch=1)
        gen_student("tiny_vit_5m", "tv_5m_160", img=160, embed=6, seed_w=75, seed_x=76, batch=1)
        gen_student("tiny_vit_21m", "tv_21m_160", img=160, embed=6, seed_w=77, seed_x=78, batch=1)
        gen_student("efficientvit_b0", "ev_b0_160", img=160, embed=6, seed_w=79, seed_x=80, batch=1)
        gen_student("efficientvit_b2", "ev_b2_192", img=192, embed=6, seed_w=81, seed_x=82, batch=1)   # 6x6 = 36 > dim 32
    if which in ("rvm", "all"):
        gen_student("repvit_m1_1", "rvm_160", img=160, embed=12, seed_w=51, seed_x=52, batch=1)
    if which in ("neck", "all"):
        gen_neck("neck_small", dim=128, d_model=64, hw=6, B=2, seed_w=31, seed_x=32)
    if which in ("prompts", "all"):
        gen_sam_prompts("sam_prompts_12", E=12, S=168, seed_pe=5, seed_md=6, seed_x=41)
    if which in ("heads", "all"):
        gen_sam_heads("sam_heads_16", E=16, S=224, B=2, seed_pe=5, seed_md=6, seed_x=1)
    if which in ("vit", "all"):
        gen_vit("vit_small_112", VIT_SMALL, seed_w=21, seed_x=3, batch=2)
    if which in ("evm", "all"):
        # 160x160: stage3 10x10, stage4 5x5 (> dim=16 pixels so the linear-attention branch runs, odd size
        # exercises the stride-2 padding), head 5x5 -> bilinear to 12x12.
        gen_student("efficientvit_b1", "evm_160", img=160, embed=12, seed_w=11, seed_x=12, batch=1)
        # 64x64: stage4 is 2x2 = 4 <= dim -> the quadratic-attention branch (oracle only).
        gen_student("efficientvit_b1", "evm_64_quadratic", img=64, embed=2, seed_w=13, seed_x=14, batch=2)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "all")
