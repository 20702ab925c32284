"""Generate the committed golden vectors by running the UNMODIFIED reference modules.

Run in the build container only (needs /root/reference, read-only):
    python tests/golden/make_golden.py
Writes tests/golden/*.npz.  The GPU box never runs this; tests read the .npz files.
Inputs and model state come from efficientat_b200.synth (seeded, order-independent), so the
oracle and the CUDA path can regenerate identical inputs without the reference.
"""
import contextlib
import io
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.path.insert(0, REPO)
from efficientat_b200.synth import (bn_modules, get_bn_stats, synth_labels, synth_state_,  # noqa: E402
                                    synth_waveform)

os.chdir(REF)            # helpers/utils.py opens metadata/ relative to CWD
sys.path.insert(0, REF)
with contextlib.redirect_stdout(io.StringIO()):
    from models.dymn.model import get_model as ref_dymn
    from models.mn.model import get_model as ref_mn
    from models.preprocess import AugmentMelSTFT as RefMel

import warnings
warnings.filterwarnings("ignore")
torch.set_num_threads(8)


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def fmap_digest(fmaps):
    """mean / abs-max / 8 strided samples per feature map."""
    out = []
    for f in fmaps:
        flat = f.flatten()
        idx = torch.linspace(0, flat.numel() - 1, 8).long()
        out.append(torch.cat([f.mean().view(1), f.abs().max().view(1), flat[idx]]))
    return torch.stack(out).numpy()


def golden_mel():
    mel = quiet(RefMel)
    mel.eval()
    x = synth_waveform(2, 32000, seed=11)
    with torch.no_grad():
        y = mel(x)
    x2 = synth_waveform(1, 5000, seed=12)      # ragged length: 1 + 4999 // 320 = 16 frames
    with torch.no_grad():
        y2 = mel(x2)
    # non-default geometry (mn10_as_mels_64 / hop variants exist upstream)
    mel3 = quiet(RefMel, n_mels=64, hopsize=500, fmin=50.0, fmax=14000.0)
    mel3.eval()
    with torch.no_grad():
        y3 = mel3(synth_waveform(1, 16000, seed=13))
    # loud, strongly coloured signal: sum of decaying sinusoids (exercises dynamic range)
    t = torch.arange(32000) / 32000.0
    x4 = (0.8 * torch.sin(2 * np.pi * 440 * t) * torch.exp(-3 * t) + 0.05 * torch.sin(2 * np.pi * 9000 * t)
          + 1e-3 * synth_waveform(1, 32000, seed=14)[0] * 10).unsqueeze(0)
    with torch.no_grad():
        y4 = mel(x4)
    np.savez_compressed(os.path.join(HERE, "mel.npz"), y_noise=y.numpy(), y_ragged=y2.numpy(),
                        y_geom=y3.numpy(), x_tone=x4.numpy(), y_tone=y4.numpy())
    print("mel", y.shape, y2.shape, y3.shape, y4.shape)


def run_net(tag, factory, width, n_samples, batch, train=True):
    torch.manual_seed(0)
    model = quiet(factory, width_mult=width)
    synth_state_(model, seed=7)
    # network input: a synthetic "spectrogram" drawn directly (same tensor on both sides, independent of
    # the mel front end, whose parity is pinned separately in mel.npz)
    frames = 1 + (n_samples - 1) // 320
    spec = synth_waveform(batch, 128 * frames, seed=21, std=0.7).view(batch, 1, 128, frames)
    # calibrate BatchNorm running statistics with one training-mode pass (momentum 1 -> running = batch
    # statistics), so that the frozen-BN eval network neither saturates nor loses its input dependence;
    # the calibrated buffers are part of the golden file and are installed by tests/util.build_model.
    model.train()
    for _, m in bn_modules(model):
        m.momentum = 1.0
    with torch.no_grad():
        model(spec)
    for _, m in bn_modules(model):
        m.momentum = 0.01
        m.num_batches_tracked.zero_()
    cal_rm, cal_rv = get_bn_stats(model)
    res = {"spec_digest": fmap_digest([spec]), "cal_rm": cal_rm.numpy(), "cal_rv": cal_rv.numpy()}
    import json
    with open(os.path.join(HERE, f"statedict_{tag.split('_')[0]}.json"), "w") as fh:      # on-disk checkpoint contract
        json.dump({k: list(v.shape) for k, v in model.state_dict().items()}, fh, indent=0)
    # ---- eval
    model.eval()
    with torch.no_grad():
        if tag.startswith("dymn"):
            logits, feat = model(spec)
            _, fmaps = model(spec, return_fmaps=True)
        else:
            logits, feat = model(spec)
            _, fmaps = model._forward_impl(spec, return_fmaps=True)
    res.update(eval_logits=logits.numpy(), eval_feat=feat.numpy(), eval_fmaps=fmap_digest(fmaps))
    if not train:
        np.savez_compressed(os.path.join(HERE, f"{tag}.npz"), **res)
        print(tag, "eval logits absmax", logits.abs().max().item())
        return
    # ---- train: batch-stat BN, dropout disabled (p=0) so the result is deterministic
    model.train()
    for m in model.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    y = synth_labels(batch, 527, seed=5)
    logits_t, _ = model(spec)
    loss = torch.nn.functional.binary_cross_entropy_with_logits(logits_t, y)
    loss.backward()
    names, gnorm, gsamp = [], [], []
    for n, p in model.named_parameters():
        names.append(n)
        g = p.grad.flatten()
        gnorm.append(g.double().norm().item())
        idx = torch.linspace(0, g.numel() - 1, 4).long()
        gsamp.append(g[idx].numpy())
    bn_names, bn_rm, bn_rv = [], [], []
    for n, m in model.named_modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            bn_names.append(n)
            bn_rm.append(m.running_mean[:4].numpy().copy())
            bn_rv.append(m.running_var[:4].numpy().copy())
    res.update(train_logits=logits_t.detach().numpy(), train_loss=np.float64(loss.item()),
               grad_names=np.array(names), grad_norm=np.array(gnorm), grad_samples=np.stack(gsamp),
               bn_names=np.array(bn_names), bn_rm4=np.stack(bn_rm), bn_rv4=np.stack(bn_rv))
    np.savez_compressed(os.path.join(HERE, f"{tag}.npz"), **res)
    print(tag, "eval logits absmax", logits.abs().max().item(), "train loss", loss.item())


def state_digest(sd):
    """per-tensor L2 norm + 4 strided samples of a state_dict (floating tensors only)"""
    out = {}
    for k, v in sd.items():
        if not torch.is_floating_point(v):
            out[k] = {"int": int(v)}
            continue
        f = v.detach().flatten().double()
        idx = torch.linspace(0, f.numel() - 1, 4).long()
        out[k] = {"norm": f.norm().item(), "samples": [float(x) for x in f[idx]]}
    return out


def golden_script():
    """The reference's OWN scripts, unchanged, with the reference's own modules on CPU (scripts/run_reference_script.py
    --side reference): ex_audioset.py --train (mixup, hard + distillation loss with the unknown-teacher mask, Adam,
    LambdaLR schedule, validation; ex_audioset.py:120-222) and inference.py on the wav fixture.  The GPU test
    (tests/test_gpu_refscripts.py) runs the same scripts with `--side ours --cuda` and compares what they log/print."""
    import json
    import re
    import tempfile
    from tests import refscripts as R
    os.chdir(REPO)
    with tempfile.TemporaryDirectory() as wd:
        env = R.make_workdir(wd, checkpoints=("mn04_as", "mn10_as"))
        log, ck = os.path.join(wd, "log.json"), os.path.join(wd, "final.pt")
        r = R.run_script(wd, "reference", "ex_audioset.py", R.SCRIPT_ARGS, env, log_json=log, keep_checkpoint=ck)
        assert r.returncode == 0, r.stderr[-3000:]
        sd = torch.load(ck, map_location="cpu")
        res = {"args": R.SCRIPT_ARGS, "env": R.SCRIPT_ENV, "epochs": R.read_log(log), "final_state": state_digest(sd)}
        r = R.run_script(wd, "reference", "inference.py", ["--model_name", "mn10_as", "--audio_path", R.WAV],
                         env, no_dropout=False)
        assert r.returncode == 0, r.stderr[-3000:]
        rows = re.findall(r"^(.+): (\d\.\d{3})$", r.stdout, flags=re.M)
        assert len(rows) == 10, r.stdout
        res["inference_top10"] = [[a, float(b)] for a, b in rows]
    with open(os.path.join(HERE, "script_mn04.json"), "w") as fh:
        json.dump(res, fh, indent=0)
    print("script: epochs", [e["train_loss"] for e in res["epochs"]], "top1", res["inference_top10"][0])


def golden_script_f4():
    """SURVEY section 8 row f4 (ensemble + windowed inference), reference modules on CPU, fp32:
      * `inference.py --ensemble mn04_as mn10_as` on the wav fixture, unchanged (models/ensemble.py: mean of the logits);
        (an ensemble with a DyMN member is pinned at the synthetic golden inputs instead, tests/test_gpu_zz_f4.py: on this
        recording the synthetic DyMN states overflow -- logits of 1e20 with the reference's own modules -- and pin nothing);
      * `windowed_inference.py` (2 s windows, 1 s hop -> 9 windows of the 10 s fixture): the script's own printout and,
        through tests/golden/windowed_driver.py, EATagger's full-precision result for mn10_as and for the mn04 + mn10 ensemble.
    windowed_inference.py:8 cannot be imported against the reference's own package (it asks models.mn.model for
    get_ensemble_model, which lives in models/ensemble.py); the launcher binds that name on the imported module."""
    import json
    import re
    import tempfile
    from tests import refscripts as R
    os.chdir(REPO)
    wav = R.WAV
    res = {"window_s": 2.0, "hop_s": 1.0, "ensemble": ["mn04_as", "mn10_as"]}
    with tempfile.TemporaryDirectory() as wd:
        env = R.make_workdir(wd, checkpoints=("mn04_as", "mn10_as"))
        r = R.run_script(wd, "reference", "inference.py", ["--ensemble"] + res["ensemble"] + ["--audio_path", wav], env,
                         no_dropout=False)
        assert r.returncode == 0, r.stderr[-3000:]
        rows = re.findall(r"^(.+): (\d\.\d{3})$", r.stdout, flags=re.M)
        assert len(rows) == 10, r.stdout
        res["inference_ensemble_top10"] = [[a, float(b)] for a, b in rows]
        r = R.run_script(wd, "reference", "windowed_inference.py",
                         ["--model", "mn10_as", "--audio_path", wav, "--window_size", "2", "--hop_length", "1"], env,
                         no_dropout=False, extra=["--export-ensemble-in-mn-model"])
        assert r.returncode == 0, r.stderr[-3000:]
        res["windowed_stdout"] = R.parse_windowed_stdout(r.stdout)
        assert len(res["windowed_stdout"]) == 9, r.stdout
        for key, names in (("windowed_mn10", ["mn10_as"]), ("windowed_ensemble", res["ensemble"])):
            out = os.path.join(wd, key + ".json")
            r = R.run_script(wd, "reference", os.path.join(HERE, "windowed_driver.py"),
                             [out, wav, "2", "1", "cpu"] + names, env, no_dropout=False,
                             extra=["--export-ensemble-in-mn-model"])
            assert r.returncode == 0, r.stderr[-3000:]
            res[key] = json.load(open(out))
            assert len(res[key]) == 9
    with open(os.path.join(HERE, "script_f4.json"), "w") as fh:
        json.dump(res, fh, indent=0)
    print("script_f4: ensemble top1", res["inference_ensemble_top10"][0], "windowed[0]", res["windowed_mn10"][0]["tags"][0], "windowed ensemble[0]", res["windowed_ensemble"][0]["tags"][0])


JOBS = {
    "mel": golden_mel,
    "mn10": lambda: run_net("mn10", ref_mn, 1.0, 64000, 2),
    "mn04": lambda: run_net("mn04", ref_mn, 0.4, 32000, 2),
    "mn20": lambda: run_net("mn20", ref_mn, 2.0, 32000, 1),
    "dymn10": lambda: run_net("dymn10", ref_dymn, 1.0, 64000, 2),
    "dymn04": lambda: run_net("dymn04", ref_dymn, 0.4, 32000, 2),
    # the shapes the benchmark times (10 s clips -> 1000 frames) and the widths BASELINE.json names (C4: dymn20, C5: mn40)
    "mn10_10s": lambda: run_net("mn10_10s", ref_mn, 1.0, 320000, 2),
    "dymn20_10s": lambda: run_net("dymn20_10s", ref_dymn, 2.0, 320000, 2),
    "dymn20": lambda: run_net("dymn20", ref_dymn, 2.0, 64000, 2),
    "mn40_10s": lambda: run_net("mn40_10s", ref_mn, 4.0, 320000, 1, train=False),
    "script": golden_script,
    "script_f4": golden_script_f4,
}

if __name__ == "__main__":
    for name in (sys.argv[1:] or list(JOBS)):
        JOBS[name]()
