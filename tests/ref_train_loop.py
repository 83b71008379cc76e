"""Transcription of the reference's training / validation loops (TEST INFRASTRUCTURE ONLY).

Follows the reference's ``train.py:80-152`` (``train_one_epoch``) and ``:26-77`` (``eval_one_epoch``) statement by
statement, quirks included, so that BASELINE configs[4] ("loss-curve parity") is judged against the reference's
loop and not against this repository's own:

* the perceptual model is a GLOBAL in ``eval_one_epoch`` (``train.py:62``) -- here an argument;
* validation ``perceptual_loss`` is ASSIGNED, not accumulated (``train.py:74``), then divided by the number of
  minibatches (``:77``): the logged value is "last batch / count";
* ``scheduler.step()`` runs per minibatch (``train.py:133``);
* SSIM / PSNR come from torchmetrics in the reference (not installed here: SURVEY.md 8c); ``metrics`` is any
  object with the same two functions (``waternet_b200.metrics``, checked separately against hand-computed values);
* tqdm progress bars are dropped.

``model`` is whatever module the caller passes: ``tests/golden/make_golden.py`` runs the unmodified reference
``WaterNet`` through it and stores the curve that the GPU test holds this repository's loop to.
"""
import torch

TRAIN_METRICS_NAMES = ["mse", "ssim", "psnr", "perceptual_loss", "loss"]   # train.py:20
VAL_METRICS_NAMES = ["mse", "ssim", "psnr", "perceptual_loss"]             # train.py:21


def _imagenet_normalize(x):
    """``TF.normalize(x, mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])`` (train.py:111-116)."""
    mean = torch.as_tensor([0.485, 0.456, 0.406], dtype=x.dtype, device=x.device).view(-1, 1, 1)
    std = torch.as_tensor([0.229, 0.224, 0.225], dtype=x.dtype, device=x.device).view(-1, 1, 1)
    return (x - mean) / std


def eval_one_epoch(model, val_dataloader, vgg_model, device, metrics):
    """train.py:26-77."""
    model.eval()
    epoch_metrics = {i: 0 for i in VAL_METRICS_NAMES}
    minibatches_per_epoch = len(val_dataloader)
    with torch.no_grad():
        for _, next_data in enumerate(val_dataloader):
            rgb_ten = next_data["raw"].to(device)
            wb_ten = next_data["wb"].to(device)
            he_ten = next_data["he"].to(device)
            gc_ten = next_data["gc"].to(device)
            ref_ten = next_data["ref"].to(device)
            out = model(rgb_ten, wb_ten, he_ten, gc_ten)
            x = _imagenet_normalize(out)
            y = _imagenet_normalize(ref_ten)
            perceptual_dist = torch.square(255 * (vgg_model(x) - vgg_model(y)))
            perceptual_loss = torch.mean(perceptual_dist)
            epoch_metrics["mse"] += torch.mean(torch.square(255 * (out - ref_ten))).item()
            epoch_metrics["ssim"] += metrics.ssim(out, ref_ten).item()
            epoch_metrics["psnr"] += metrics.psnr(out, ref_ten, 1 - 0).item()
            epoch_metrics["perceptual_loss"] = perceptual_loss.item()   # sic: assignment (train.py:74)
    epoch_metrics = {i: j / minibatches_per_epoch for i, j in epoch_metrics.items()}
    model.train()
    return epoch_metrics


def train_one_epoch(model, train_dataloader, optimizer, scheduler, vgg_model, device, metrics):
    """train.py:80-152."""
    model.train()
    epoch_metrics = {i: 0 for i in TRAIN_METRICS_NAMES}
    minibatches_per_epoch = len(train_dataloader)
    for idx, next_data in enumerate(train_dataloader):
        rgb_ten = next_data["raw"].to(device)
        wb_ten = next_data["wb"].to(device)
        he_ten = next_data["he"].to(device)
        gc_ten = next_data["gc"].to(device)
        ref_ten = next_data["ref"].to(device)
        out = model(rgb_ten, wb_ten, he_ten, gc_ten)
        x = _imagenet_normalize(out)
        y = _imagenet_normalize(ref_ten)
        perceptual_dist = torch.square(255 * (vgg_model(x) - vgg_model(y)))
        perceptual_loss = torch.mean(perceptual_dist)
        mse = torch.mean(torch.square(255 * (out - ref_ten)))
        loss = (0.05 * perceptual_loss) + mse
        optimizer.zero_grad()
        loss.backward()
        optimizer.step()
        scheduler.step()
        epoch_metrics["loss"] += loss.item()
        epoch_metrics["perceptual_loss"] += perceptual_loss.item()
        epoch_metrics["mse"] += mse.item()
        with torch.no_grad():
            epoch_metrics["ssim"] += metrics.ssim(out, ref_ten).item()
            epoch_metrics["psnr"] += metrics.psnr(out, ref_ten, 1 - 0).item()
    epoch_metrics = {i: j / minibatches_per_epoch for i, j in epoch_metrics.items()}
    return epoch_metrics
