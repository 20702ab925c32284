#!/usr/bin/env python
"""Run one of the reference's own entry scripts (ex_audioset.py, inference.py) UNCHANGED, either against this
package (`--side ours`: `dropin/` shadows `models.*`, `helpers.utils`, `datasets.audioset`) or against the reference's
own modules (`--side reference`, used to produce golden numbers on CPU and the cuDNN baseline on GPU).

    python scripts/run_reference_script.py --side ours --ref-root oracle/_ref --log-json out.json \
        ex_audioset.py -- --train --cuda --pretrained --model_name mn04_as --batch_size 4 --num_workers 0 ...

The script file itself is executed with runpy from `--ref-root`; nothing in it is edited.  What the launcher sets up
is the ENVIRONMENT the script expects and this container does not have:
  * sys.path: [dropin, repo] + ref-root for everything not shadowed (models.ensemble, helpers.init, metadata/...);
  * `datasets.audioset`: the synthetic AudioSet of dropin/datasets/audioset.py on BOTH sides (the real one needs
    the AudioSet HDF5 files, h5py and PyAV);
  * `librosa.core.load` (librosa is not installed): scipy wav read + polyphase resampling to the requested rate;
  * wandb in disabled mode: the run directory is created (ex_audioset.py saves the checkpoint there) and every
    `wandb.log` payload is appended to `--log-json`;
  * `--seed`: torch / numpy / random seeds before the script starts; `--no-dropout`: nn.Dropout(p) -> p = 0, because the
    CPU generator (reference) and the device generator (this package) cannot produce the same mask.
"""
import argparse
import importlib.util
import json
import os
import random
import runpy
import sys
import types

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _install_librosa_shim():
    try:
        import librosa  # noqa: F401
        return
    except Exception:
        pass
    import numpy as np
    from math import gcd
    from scipy.io import wavfile
    from scipy.signal import resample_poly

    def load(path, sr=22050, mono=True, **_):
        rate, x = wavfile.read(path)
        if x.dtype.kind == "i":
            x = x.astype(np.float32) / float(np.iinfo(x.dtype).max + 1)
        elif x.dtype.kind == "u":
            x = (x.astype(np.float32) - 128.0) / 128.0
        else:
            x = x.astype(np.float32)
        if x.ndim == 2:
            x = x.mean(axis=1) if mono else x.T
        if sr is not None and sr != rate:
            g = gcd(int(sr), int(rate))
            x = resample_poly(x, int(sr) // g, int(rate) // g, axis=-1).astype(np.float32)
            rate = sr
        return np.ascontiguousarray(x, dtype=np.float32), rate

    lib = types.ModuleType("librosa")
    core = types.ModuleType("librosa.core")
    core.load = load
    lib.core = core
    lib.load = load
    lib.__doc__ = "stand-in for librosa.core.load (scipy wav read + resample_poly); librosa is not installed here"
    sys.modules["librosa"] = lib
    sys.modules["librosa.core"] = core


def _install_datasets(ref_root):
    """`datasets` = a package whose search path is the reference's datasets/ directory, with `datasets.audioset`
    replaced by the synthetic stand-in (site-packages also has an unrelated `datasets` distribution)."""
    pkg = types.ModuleType("datasets")
    pkg.__path__ = [os.path.join(REPO, "dropin", "datasets"), os.path.join(ref_root, "datasets")]
    sys.modules["datasets"] = pkg
    spec = importlib.util.spec_from_file_location("datasets.audioset", os.path.join(REPO, "dropin", "datasets", "audioset.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["datasets.audioset"] = mod
    spec.loader.exec_module(mod)
    pkg.audioset = mod


def _install_wandb(log_json):
    os.environ.setdefault("WANDB_MODE", "disabled")
    os.environ.setdefault("WANDB_SILENT", "true")
    import wandb
    orig_init = wandb.init
    records = []

    def init(*a, **k):
        run = orig_init(*a, **k)
        try:
            os.makedirs(wandb.run.dir, exist_ok=True)
        except Exception:
            pass
        orig_log = wandb.log                      # wandb.init rebinds the module-level log to the run's

        def log(payload, *la, **lk):
            rec = {}
            for key, v in payload.items():
                try:
                    rec[key] = float(v)
                except Exception:
                    rec[key] = str(v)
            records.append(rec)
            if log_json:
                with open(log_json, "w") as f:
                    json.dump(records, f)
            return orig_log(payload, *la, **lk)
        wandb.log = log
        return run

    wandb.init = init
    return wandb


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", choices=["ours", "reference"], required=True)
    ap.add_argument("--ref-root", default=os.path.join(REPO, "oracle", "_ref"))
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--no-dropout", action="store_true")
    ap.add_argument("--log-json", default=None)
    ap.add_argument("--keep-checkpoint", default=None, help="copy the last checkpoint the script saved to this path")
    ap.add_argument("--export-ensemble-in-mn-model", action="store_true",
                    help="--side reference only: windowed_inference.py:8 imports get_ensemble_model from models.mn.model, "
                         "which the reference defines in models/ensemble.py only; bind the reference's own function under "
                         "that name on the imported module (no file is edited) so the script can run for golden numbers")
    ap.add_argument("script")
    ap.add_argument("rest", nargs=argparse.REMAINDER)
    a = ap.parse_args()
    ref_root = os.path.abspath(a.ref_root)
    script = os.path.join(ref_root, a.script)          # an absolute path (a driver under tests/golden/) is taken as is
    if not os.path.isfile(script):
        raise SystemExit(f"{script} not found (run `python oracle/make_ref.py` where the reference checkout exists)")
    rest = a.rest[1:] if a.rest and a.rest[0] == "--" else a.rest

    # import resolution: the script's own directory is NOT put first (runpy.run_path does not do it), so `models.*`
    # resolves to dropin/ for --side ours and to the reference checkout otherwise
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or ".") not in (ref_root,)]
    if a.side == "ours":
        sys.path.insert(0, REPO)
        sys.path.insert(0, os.path.join(REPO, "dropin"))
        sys.path.append(ref_root)
    else:
        sys.path.insert(0, ref_root)
    _install_datasets(ref_root)
    _install_librosa_shim()
    wandb = _install_wandb(a.log_json)

    import numpy as np
    import torch
    if a.no_dropout:
        _orig = torch.nn.Dropout.__init__

        def _init(self, p=0.5, inplace=False):
            _orig(self, 0.0, inplace)
        torch.nn.Dropout.__init__ = _init
    if a.seed is not None:
        torch.manual_seed(a.seed)
        np.random.seed(a.seed)
        random.seed(a.seed)

    if a.export_ensemble_in_mn_model and a.side == "reference":
        import models.ensemble
        import models.mn.model
        if not hasattr(models.mn.model, "get_ensemble_model"):
            models.mn.model.get_ensemble_model = models.ensemble.get_ensemble_model

    sys.argv = [script] + rest
    runpy.run_path(script, run_name="__main__")

    if a.keep_checkpoint and wandb.run is not None and os.path.isdir(wandb.run.dir):
        import glob
        import shutil
        pts = sorted(glob.glob(os.path.join(wandb.run.dir, "*.pt")), key=os.path.getmtime)
        if pts:
            shutil.copy2(pts[-1], a.keep_checkpoint)


if __name__ == "__main__":
    main()
