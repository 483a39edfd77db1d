"""Drop-in for the loop body of the reference's stage-1 trainer (stage1/train_image_encoder_stage1.py:154-268, 310-314):
`train_one_epoch` with the reference's loader contract -- batches of ((samples, annos), (saved_embeddings, seeds)) as
`build_loader` yields them, teacher embeddings read from the store -- on the native student, KD loss, backward and optimiser.
Logging / TensorBoard / checkpointing stay with the caller (out of scope, SURVEY.md section 2)."""
from __future__ import annotations

import numpy as np
import torch

from .losses import kd_train_step
from .optim import cosine_lr


def set_bn_state(config, model):
    """train_image_encoder_stage1.py:310-314: with TRAIN.EVAL_BN_WHEN_TRAINING every BatchNorm stays in eval mode (the native
    training graph then uses the running statistics and still produces the BN weight / bias gradients)."""
    if config.TRAIN.EVAL_BN_WHEN_TRAINING:
        for m in model.modules():
            if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
                m.eval()


def train_one_epoch(config, model, data_loader, optimizer, epoch, lr_at=None, on_step=None, preprocess=None):
    """One epoch of stage-1 distillation.  `optimizer`: stage1.optim.FlatAdamW over `model`.  `lr_at(update_index) -> lr`
    replaces `lr_scheduler.step_update` (default: the reference's cosine schedule built from config.TRAIN).  `on_step(idx, loss)`
    is called after every iteration with the detached device loss (call `.item()` there only when you log: it syncs).
    `preprocess`: a stage1.transforms.ImagePreprocessor; `samples` are then decoded images of any size, resized, normalised
    and padded on the device, and img_size_before_pad comes from it.
    Returns the list of per-iteration losses (device scalars)."""
    model.train()
    set_bn_state(config, model)
    optimizer.zero_grad()
    num_steps = len(data_loader)
    accum = int(config.TRAIN.ACCUMULATION_STEPS)
    embed_shape = (config.DISTILL.EMBED_DIM, config.DISTILL.EMBED_SIZE, config.DISTILL.EMBED_SIZE)
    if lr_at is None:
        n_iter = num_steps // accum                  # build_scheduler(config, optimizer, len(loader) // ACCUMULATION_STEPS), :80-84
        total = int(config.TRAIN.EPOCHS * n_iter)
        warm = int(config.TRAIN.WARMUP_EPOCHS * n_iter)
        base = getattr(optimizer, "base_lr", optimizer.lr)     # never optimizer.lr: step(lr=...) overwrites it every update

        def lr_at(t):
            return cosine_lr(t, base, total, config.TRAIN.MIN_LR, warm, config.TRAIN.WARMUP_LR)

    # The reference applies update u with the LR the PREVIOUS `step_update` call left in the optimiser (the scheduler is stepped
    # after optimizer.step(), :216-229); the very first update runs at the scheduler's initial value, which is lr_at(0).
    def lr_for_update(idx):
        prev = idx - accum                               # iteration index of the previous update inside this epoch
        if prev >= 0:
            return lr_at((epoch * num_steps + prev) // accum)
        last = (num_steps // accum) * accum - 1          # last updating iteration of the previous epoch
        if epoch > 0 and last >= 0:
            return lr_at(((epoch - 1) * num_steps + last) // accum)
        return lr_at(0)

    cosine_w = float(config.DISTILL.COSINE)
    dev = next(model.parameters()).device
    losses = []
    for idx, ((samples, annos), (saved_embeddings, seeds)) in enumerate(data_loader):
        if preprocess is not None:
            samples, sizes = preprocess(list(samples))
        else:
            samples, sizes = torch.stack(list(samples), dim=0).to(dev, non_blocking=True), annos["img_size_before_pad"]
        saved = torch.from_numpy(np.stack(saved_embeddings, axis=0)).float()
        saved = saved.view(samples.size(0), *embed_shape).to(dev, non_blocking=True)
        update = (idx + 1) % accum == 0
        loss = kd_train_step(model, optimizer, samples, saved, sizes, cosine_weight=cosine_w,
                             clip_grad=config.TRAIN.CLIP_GRAD, lr=lr_for_update(idx) if update else None,
                             accumulation_steps=accum, update=update)
        losses.append(loss)
        if on_step is not None:
            on_step(idx, loss)
        if getattr(config.DATA, "DEBUG", False):
            break
    return losses
