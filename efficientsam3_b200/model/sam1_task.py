"""Point-prompt segmentation pipeline (BASELINE config 3): SAM3 ViT trunk -> SAM2-branch FPN -> SAM heads, batched.

Native counterpart of the reference call chain
  SAM3InteractiveImagePredictor.set_image_batch   sam3/sam3/model/sam1_task_predictor.py:121-166
  Sam3TrackerBase.forward_image (conv_s0/conv_s1)  sam3/sam3/model/sam3_tracker_base.py:445-466
  SAM3InteractiveImagePredictor._predict           sam1_task_predictor.py:329-430
  Sam3TrackerBase._forward_sam_heads               sam3_tracker_base.py:220-389
with the reference's per-image Python loop (sam1_task_predictor.py:168-228) replaced by one batched pass
(B images x 1 prompt each, `repeat_image=False` semantics).  Parameter names follow the reference tracker
(`sam_prompt_encoder.*`, `sam_mask_decoder.*`, `no_mem_embed`, `backbone.vision_backbone.{trunk,convs,sam2_convs}.*`).
SAM3InteractiveImagePredictor mirrors the reference predictor API (set_image / set_image_batch / predict / predict_batch)
on top of it: box and mask prompts, several prompts per image, hole filling (es3_fill_small_components) and the resize
to the original size.  Not built: tracker memory (obj_ptr).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .. import ops
from ..sam import MaskDecoder, PromptEncoder, TwoWayTransformer
from ..stage1.transforms import ImagePreprocessor
from .necks import Sam3DualViTDetNeck
from .vitdet import create_sam3_vit_backbone

NO_OBJ_SCORE = -1024.0


class _Holder(nn.Module):
    pass


class Sam3PointPromptSegmenter(nn.Module):
    def __init__(self, image_size=1008, backbone_stride=14, hidden_dim=256, vit_overrides=None, vision_backbone=None):
        """vision_backbone: an already built Sam3DualViTDetNeck (with the SAM2 branch), e.g. the EfficientSAM3 student encoder of
        efficientsam3_b200.model_builder.create_student_vision_backbone; default: the SAM3 ViT trunk + neck."""
        super().__init__()
        self.image_size, self.hidden_dim = image_size, hidden_dim
        e = image_size // backbone_stride
        self.backbone = _Holder()
        if vision_backbone is None:
            trunk = create_sam3_vit_backbone(**(vit_overrides or {}))
            vision_backbone = Sam3DualViTDetNeck(trunk=trunk, position_encoding=None, d_model=hidden_dim,
                                                 scale_factors=[4.0, 2.0, 1.0, 0.5], add_sam2_neck=True)
        assert vision_backbone.sam2_convs is not None, "the SAM heads read the SAM2 branch of the neck (enable_inst_interactivity)"
        self.backbone.vision_backbone = vision_backbone
        self.no_mem_embed = nn.Parameter(torch.zeros(1, 1, hidden_dim))
        nn.init.trunc_normal_(self.no_mem_embed, std=0.02)
        self.sam_prompt_encoder = PromptEncoder(embed_dim=hidden_dim, image_embedding_size=(e, e),
                                                input_image_size=(image_size, image_size), mask_in_chans=16)
        self.sam_mask_decoder = MaskDecoder(
            num_multimask_outputs=3, transformer=TwoWayTransformer(depth=2, embedding_dim=hidden_dim, mlp_dim=2048, num_heads=8),
            transformer_dim=hidden_dim, iou_head_depth=3, iou_head_hidden_dim=256, use_high_res_features=True,
            iou_prediction_use_sigmoid=True, pred_obj_scores=True, pred_obj_scores_mlp=True,
            use_multimask_token_for_obj_ptr=True)
        self._features = None
        self.eval()

    @torch.no_grad()
    def set_image_batch(self, images: torch.Tensor):
        """images [B,3,S,S] fp32 CUDA, already resized / normalised (mean 0.5, std 0.5 as Sam3Processor does)."""
        neck = self.backbone.vision_backbone
        strict = ops.precision() == "strict"
        if hasattr(neck.trunk, "forward_tokens"):       # SAM3 ViT trunk: fp32 token stream -> bf16 NHWC (strict: stays fp32)
            tok, (B, h, w) = neck.trunk.forward_tokens(images)
            feats = (tok if strict else ops.add_rows(tok, None, out_bf16=True, out_f32=False)[0]).view(B, h, w, -1)
        else:                                           # EfficientSAM3 student encoder (model_builder.ListWrapper)
            feats = neck.trunk.forward_nhwc(images)
            B, h, w, _ = feats.shape
        l288, l144, l72 = neck.forward_nhwc(feats, "sam2", (0, 1, 2), f32_levels=(2,))
        md = self.sam_mask_decoder
        feat_s0, feat_s1 = md.project_high_res(l288, l144)
        # image_embed = 72^2 level + no_mem_embed (sam1_task_predictor.py:157) + no_mask dense embedding (mask_decoder.py:189)
        addc = (self.no_mem_embed.detach().reshape(-1) + self.sam_prompt_encoder.no_mask_embed.weight.detach().reshape(-1)).float().contiguous()
        C = l72.shape[-1]
        keys_b16, keys_f32 = ops.add_rows(l72.view(-1, C), addc.view(1, C), out_bf16=not strict, out_f32=True)
        if strict:
            keys_b16 = keys_f32
        # the same level with no_mem_embed only: the base a mask prompt's dense embedding is added to
        _, base_f32 = ops.add_rows(l72.view(-1, C), self.no_mem_embed.detach().reshape(1, C).float().contiguous(), out_f32=True)
        self._features = dict(B=B, h=h, w=w, keys_f32=keys_f32, keys_b16=keys_b16, base_f32=base_f32, feat_s0=feat_s0,
                              feat_s1=feat_s1, pe=self.sam_prompt_encoder.pe_layer.tokens((h, w)))
        return self

    @torch.no_grad()
    def decode_prompts(self, img_idx, points=None, boxes=None, mask_input=None, multimask_output=True, obj_gate=False):
        """P prompts on image `img_idx` of the current batch (the reference's repeat_image=True decoding,
        sam1_task_predictor.py:386-404).  points = (coords [P,N,2], labels [P,N]) in model-input pixels, boxes [P,4] are
        merged in front as label-2/3 corner points, mask_input [P,1,4h,4w] logits.  -> (low-res logits [P,K,4h,4w], iou [P,K])."""
        f = self._features
        assert f is not None, "call set_image_batch first"
        h, w, hw = f["h"], f["w"], f["h"] * f["w"]
        pts = None
        if points is not None:
            pts = (points[0].float(), points[1].to(torch.int32))
        if boxes is not None:
            bc = boxes.float().reshape(-1, 2, 2)
            bl = torch.tensor([[2, 3]], dtype=torch.int32, device=bc.device).repeat(bc.shape[0], 1)
            pts = (torch.cat([bc, pts[0]], dim=1), torch.cat([bl, pts[1]], dim=1)) if pts is not None else (bc, bl)
        pe = self.sam_prompt_encoder
        if pts is not None:
            sparse = pe.embed_sparse(pts, None)
            P = sparse.shape[0]
        else:
            P = mask_input.shape[0] if mask_input is not None else 1
            sparse = torch.empty((P, 0, self.hidden_dim), device=f["keys_f32"].device, dtype=torch.float32)
        sl = slice(img_idx * hw, (img_idx + 1) * hw)
        if mask_input is not None:
            assert mask_input.shape[0] == P and tuple(mask_input.shape[1:]) == (1, 4 * h, 4 * w), tuple(mask_input.shape)
            wts, eps = pe.mask_weights()
            kb, kf = ops.mask_downscale_tokens(mask_input.float(), wts, f["base_f32"][sl].contiguous(), eps,
                                               out_bf16=ops.precision() != "strict")
            kb = kf if kb is None else kb
        else:
            kf = f["keys_f32"][sl].unsqueeze(0).expand(P, -1, -1).reshape(P * hw, -1)
            kb = f["keys_b16"][sl].unsqueeze(0).expand(P, -1, -1).reshape(P * hw, -1)
        s0 = f["feat_s0"][img_idx:img_idx + 1].expand(P, -1, -1, -1).contiguous()
        s1 = f["feat_s1"][img_idx:img_idx + 1].expand(P, -1, -1, -1).contiguous()
        low, iou, _, obj = self.sam_mask_decoder.predict_tokens(kf, kb, f["pe"], sparse, P, h, w, s0, s1, obj_gate=obj_gate,
                                                                multimask_output=multimask_output)
        return low, iou, obj

    @torch.no_grad()
    def predict_batch(self, point_coords, point_labels, multimask_output=True, return_logits=False):
        """point_coords [B,P,2] (x,y in input-image pixels), point_labels [B,P] -> dict with low-res logits
        [B,K,4h,4w], high-res logits or bool masks [B,K,S,S], ious [B,K], object logits [B,1], best index [B]."""
        f = self._features
        assert f is not None, "call set_image_batch first"
        sparse, _ = self.sam_prompt_encoder(points=(point_coords, point_labels), boxes=None, masks=None)
        low, iou, toks, obj = self.sam_mask_decoder.predict_tokens(
            f["keys_f32"], f["keys_b16"], f["pe"], sparse, f["B"], f["h"], f["w"], f["feat_s0"], f["feat_s1"],
            obj_gate=True, multimask_output=multimask_output)
        S = self.image_size
        high, binm = ops.bilinear_nchw(low, S, S, binarize_thr=None if return_logits else 0.0, want_float=return_logits)
        best = torch.argmax(iou, dim=-1)
        return dict(low_res_multimasks=low, high_res=high if return_logits else binm.bool(), ious=iou,
                    object_score_logits=obj, best=best, sam_tokens=toks)


class SAM3InteractiveImagePredictor:
    """sam3/sam3/model/sam1_task_predictor.py:18-120, 168-430 on the native segmenter.  `sam_model` is a
    Sam3PointPromptSegmenter (the reference takes the tracker model with the same sub-module names)."""

    def __init__(self, sam_model: Sam3PointPromptSegmenter, mask_threshold=0.0, max_hole_area=256.0, max_sprinkle_area=0.0):
        self.model = sam_model
        self.mask_threshold = mask_threshold
        self.max_hole_area, self.max_sprinkle_area = max_hole_area, max_sprinkle_area
        self._preprocess = None
        self.reset_predictor()

    @property
    def device(self):
        return self.model.no_mem_embed.device

    def reset_predictor(self):
        self._is_image_set = self._is_batch = False
        self._orig_hw = None
        self.model._features = None

    def _to_inputs(self, images):
        """HWC uint8 / float ndarrays or PIL images -> ([B,3,S,S] fp32 on the device, [(h, w), ...]), resized and normalised like
        SAM2Transforms (ToTensor -> Resize((S,S)) bilinear antialias -> Normalize(0.5, 0.5); sam1_utils.py:17-41) by one
        es3_preprocess_images call for the whole list.  ToTensor leaves float arrays unscaled: they are taken as [0, 1]."""
        import numpy as np
        arrs = []
        for image in images:
            arr = np.asarray(image)
            if arr.ndim != 3 or arr.shape[2] != 3:
                raise NotImplementedError("Image format not supported")
            arrs.append(arr)
        if self._preprocess is None:
            S = self.model.image_size
            self._preprocess = ImagePreprocessor(S, (127.5,) * 3, (127.5,) * 3, square=True, float_scale=255.0, device=self.device)
        x, _ = self._preprocess(arrs)
        return x, [tuple(a.shape[:2]) for a in arrs]

    def _to_input(self, image):
        """One image -> ([3,S,S] fp32 on the device, (h, w)); see _to_inputs."""
        x, hw = self._to_inputs([image])
        return x[0], hw[0]

    @torch.no_grad()
    def set_image(self, image):
        self.reset_predictor()
        x, self._orig_hw = self._to_inputs([image])
        self.model.set_image_batch(x)
        self._is_image_set = True

    @torch.no_grad()
    def set_image_batch(self, image_list):
        self.reset_predictor()
        assert isinstance(image_list, list)
        x, self._orig_hw = self._to_inputs(image_list)
        self.model.set_image_batch(x)
        self._is_image_set = self._is_batch = True

    def get_image_embedding(self):
        """[B,C,h,w] fp32: the 72^2 level + no_mem_embed (what the reference stores as image_embed, :157)."""
        if not self._is_image_set:
            raise RuntimeError("An image must be set with .set_image(...) to generate an embedding.")
        f = self.model._features
        return f["base_f32"].view(f["B"], f["h"], f["w"], -1).permute(0, 3, 1, 2)

    # ---- prompts ------------------------------------------------------------------------------------------------------
    def _transform_coords(self, coords, normalize, orig_hw):
        if normalize:
            h, w = orig_hw
            coords = coords.clone()
            coords[..., 0] = coords[..., 0] / w
            coords[..., 1] = coords[..., 1] / h
        return coords * self.model.image_size

    def _prep_prompts(self, point_coords, point_labels, box, mask_logits, normalize_coords, img_idx=-1):
        unnorm_coords = labels = unnorm_box = mask_input = None
        dev = self.device
        if point_coords is not None:
            assert point_labels is not None, "point_labels must be supplied if point_coords is supplied."
            pc = torch.as_tensor(point_coords, dtype=torch.float, device=dev)
            unnorm_coords = self._transform_coords(pc, normalize_coords, self._orig_hw[img_idx])
            labels = torch.as_tensor(point_labels, dtype=torch.int, device=dev)
            if unnorm_coords.dim() == 2:
                unnorm_coords, labels = unnorm_coords[None], labels[None]
        if box is not None:
            b = torch.as_tensor(box, dtype=torch.float, device=dev)
            unnorm_box = self._transform_coords(b.reshape(-1, 2, 2), normalize_coords, self._orig_hw[img_idx])
        if mask_logits is not None:
            mask_input = torch.as_tensor(mask_logits, dtype=torch.float, device=dev)
            if mask_input.dim() == 3:
                mask_input = mask_input[None]
        return mask_input, unnorm_coords, labels, unnorm_box

    @torch.no_grad()
    def _predict(self, point_coords, point_labels, boxes=None, mask_input=None, multimask_output=True, return_logits=False,
                 img_idx=-1):
        if not self._is_image_set:
            raise RuntimeError("An image must be set with .set_image(...) before mask prediction.")
        idx = img_idx if img_idx >= 0 else len(self._orig_hw) + img_idx
        pts = (point_coords, point_labels) if point_coords is not None else None
        low, iou, _ = self.model.decode_prompts(idx, pts, boxes.reshape(-1, 4) if boxes is not None else None, mask_input,
                                                multimask_output=multimask_output)
        masks = low
        if self.max_hole_area > 0 or self.max_sprinkle_area > 0:
            masks = ops.fill_small_components(low, self.mask_threshold, self.max_hole_area, self.max_sprinkle_area)
        oh, ow = self._orig_hw[idx]
        if return_logits:
            masks, _ = ops.bilinear_nchw(masks, oh, ow)
        else:
            _, binm = ops.bilinear_nchw(masks, oh, ow, binarize_thr=self.mask_threshold, want_float=False)
            masks = binm.bool()
        return masks, iou, torch.clamp(low, -32.0, 32.0)

    def predict(self, point_coords=None, point_labels=None, box=None, mask_input=None, multimask_output=True,
                return_logits=False, normalize_coords=True):
        """-> (masks CxHxW, iou C, low-res logits Cx4hx4w) numpy, for ONE prompt on the current image (:230-296)."""
        if not self._is_image_set:
            raise RuntimeError("An image must be set with .set_image(...) before mask prediction.")
        mask_input, coords, labels, ubox = self._prep_prompts(point_coords, point_labels, box, mask_input, normalize_coords)
        masks, iou, low = self._predict(coords, labels, ubox, mask_input, multimask_output, return_logits=return_logits)
        return masks[0].float().cpu().numpy(), iou[0].float().cpu().numpy(), low[0].float().cpu().numpy()

    def predict_batch(self, point_coords_batch=None, point_labels_batch=None, box_batch=None, mask_input_batch=None,
                      multimask_output=True, return_logits=False, normalize_coords=True):
        """Per-image prompt lists for the images given to set_image_batch (:168-228) -> three lists of numpy arrays."""
        assert self._is_batch, "This function should only be used when in batched mode"
        if not self._is_image_set:
            raise RuntimeError("An image must be set with .set_image_batch(...) before mask prediction.")
        all_masks, all_ious, all_low = [], [], []
        pick = lambda lst, i: lst[i] if lst is not None else None
        for i in range(len(self._orig_hw)):
            mask_input, coords, labels, ubox = self._prep_prompts(pick(point_coords_batch, i), pick(point_labels_batch, i),
                                                                  pick(box_batch, i), pick(mask_input_batch, i),
                                                                  normalize_coords, img_idx=i)
            masks, iou, low = self._predict(coords, labels, ubox, mask_input, multimask_output, return_logits=return_logits,
                                            img_idx=i)
            all_masks.append(masks.squeeze(0).float().cpu().numpy())
            all_ious.append(iou.squeeze(0).float().cpu().numpy())
            all_low.append(low.squeeze(0).float().cpu().numpy())
        return all_masks, all_ious, all_low
