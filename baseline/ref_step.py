"""The reference's training / eval step driven through the reference's OWN modules (oracle/_ref mirror of the
checkout: models.preprocess.AugmentMelSTFT, models.mn.model.get_model, models.dymn.model.get_model, helpers.utils.mixup)
-- measurement infrastructure for bench.py's reference arms, never imported by the product.

  * device "cpu":  `bench.py --impl reference` / `cpu_baseline` (kind "reference"): the reference's CPU PyTorch path;
  * device "cuda": `bench.py --impl reference-gpu` / `gpu_baseline`: the reference's cuFFT / cuDNN / cuBLAS path on the
    same B200 -- the bar BASELINE.md section 3 names -- in fp32 (stock defaults: TF32 convolutions, fp32 matmuls) or
    under `torch.autocast(bfloat16)`, `cudnn.benchmark = True`, DistributedDataParallel when world > 1.

The loop body restates ex_audioset.py:135-199 (mel -> mixup -> model -> hard + distillation BCE with the
unknown-teacher mask -> backward -> Adam), including its three per-step loss read-backs (:192-194)."""
import contextlib
import io
import os
import sys

import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(os.path.dirname(HERE), "oracle", "_ref")


def available():
    return os.path.isfile(os.path.join(REF, "models", "mn", "model.py"))


def _import_reference():
    """import the reference packages from the mirror; helpers/utils.py opens metadata/ relative to the CWD (:38)"""
    if REF not in sys.path:
        sys.path.insert(0, REF)
    cwd = os.getcwd()
    os.chdir(REF)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            import warnings
            warnings.filterwarnings("ignore")
            from helpers.utils import mixup
            from models.dymn.model import get_model as get_dymn
            from models.mn.model import get_model as get_mn
            from models.preprocess import AugmentMelSTFT
    finally:
        os.chdir(cwd)
    return get_mn, get_dymn, AugmentMelSTFT, mixup


WIDTH = {"mn04": 0.4, "mn10": 1.0, "mn20": 2.0, "mn40": 4.0, "dymn04": 0.4, "dymn10": 1.0, "dymn20": 2.0}


def build(model_name, device, state_seed=7):
    """-> (model, mel) reference modules on `device`, synthetic state (efficientat_b200.synth recipe)"""
    from efficientat_b200.synth import synth_state_
    get_mn, get_dymn, AugmentMelSTFT, _ = _import_reference()
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        factory = get_dymn if model_name.startswith("dymn") else get_mn
        model = synth_state_(factory(width_mult=WIDTH[model_name]), seed=state_seed).to(device)
        mel = AugmentMelSTFT(freqm=0, timem=0).to(device)                 # ex_audioset.py defaults
    return model, mel


def make_train_step(model_name, wave, y, teacher, known, device, amp=None, ddp=False, lr=8e-4, kd_lambda=0.1,
                    mixup_alpha=0.3):
    """-> step() running ONE iteration of the reference loop on the given (device-resident) batch; returns the loss"""
    _, _, _, mixup = _import_reference()
    model, mel = build(model_name, device)
    net = model
    if ddp:
        net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[device.index] if device.type == "cuda" else None)
    opt = torch.optim.Adam(model.parameters(), lr=lr)
    distillation_loss = torch.nn.BCEWithLogitsLoss(reduction="none")
    model.train()
    mel.train()
    bs = wave.shape[0]
    unknown = ~known if known is not None else None

    def step():
        ctx = torch.autocast(device_type=device.type, dtype=amp) if amp is not None else contextlib.nullcontext()
        with ctx:
            x = mel(wave.reshape(bs, -1)).unsqueeze(1)
            rn, lam = mixup(bs, mixup_alpha)
            lam = lam.to(x.device)
            x = x * lam.reshape(bs, 1, 1, 1) + x[rn] * (1. - lam.reshape(bs, 1, 1, 1))
            y_hat, _ = net(x)
            y_hat = y_hat.float()
            y_mix = y * lam.reshape(bs, 1) + y[rn] * (1. - lam.reshape(bs, 1))
            label_loss = F.binary_cross_entropy_with_logits(y_hat, y_mix, reduction="none").mean()
            soft = distillation_loss(y_hat, teacher).mean(dim=1) * lam.reshape(bs) + \
                distillation_loss(y_hat, teacher[rn]).mean(dim=1) * (1. - lam.reshape(bs))
            if unknown is not None:
                soft[unknown] = soft[unknown] * 0
            label_loss = kd_lambda * label_loss
            soft = (1 - kd_lambda) * soft.mean()
            loss = label_loss + soft
        stats = (loss.detach().cpu().numpy(), label_loss.detach().cpu().numpy(), soft.detach().cpu().numpy())   # :192-194
        loss.backward()
        opt.step()
        opt.zero_grad()
        return float(stats[0])
    return step


def make_eval_step(model_name, wave, device, amp=None):
    model, mel = build(model_name, device)
    model.eval()
    mel.eval()
    bs = wave.shape[0]

    def step():
        ctx = torch.autocast(device_type=device.type, dtype=amp) if amp is not None else contextlib.nullcontext()
        with torch.no_grad(), ctx:
            y_hat, _ = model(mel(wave.reshape(bs, -1)).unsqueeze(1))
        return float(y_hat[:, :2].float().sum().cpu())
    return step
