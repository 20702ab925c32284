"""Test harness around scripts/run_reference_script.py: builds the working directory the reference scripts expect
(resources/ with a checkpoint under its release file name, the teacher files, metadata/) and runs a script in it."""
import json
import os
import shutil
import subprocess
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAUNCHER = os.path.join(REPO, "scripts", "run_reference_script.py")
RELEASE_FILE = {"mn04_as": "mn04_as_mAP_432.pt", "mn10_as": "mn10_as_mAP_471.pt", "dymn04_as": "dymn04_as.pt",
                "dymn10_as": "dymn10_as.pt"}            # models/mn/model.py:18-70, models/dymn/model.py:18-33

# the script-level golden configuration (tests/golden/make_golden.py::golden_script and tests/test_gpu_refscripts.py)
SCRIPT_ENV = {"EAT_SYNTH_CLIP_SECONDS": "1", "EAT_SYNTH_TRAIN_CLIPS": "40", "EAT_SYNTH_TEST_CLIPS": "527"}
SCRIPT_ARGS = ["--train", "--pretrained", "--model_name", "mn04_as", "--batch_size", "8", "--num_workers", "0",
               "--n_epochs", "3", "--epoch_len", "24", "--warm_up_len", "2", "--ramp_down_start", "1",
               "--ramp_down_len", "4", "--last_lr_value", "0.1", "--max_lr", "0.0004"]


# recording and AudioSet label table the scripts read (resources/, metadata/ of the original project; the recording is
# stored resampled to 32 kHz, the rate every consumer reads it at, 16-bit; the goldens were produced from this file)
WAV = os.path.join(REPO, "tests", "golden", "metro_station-paris.wav")
METADATA = os.path.join(REPO, "tests", "golden", "metadata")


def ref_root():
    """the mirror of the original EfficientAT project that build() makes (oracle/make_ref.py), or None"""
    p = os.path.join(REPO, "oracle", "_ref")
    return p if os.path.isfile(os.path.join(p, "ex_audioset.py")) else None


def make_workdir(path, checkpoints=("mn04_as",), env=None):
    """-> env dict for the subprocess.  `checkpoints`: release names whose synthetic state (tests/util.build_model:
    seeded weights + calibrated BatchNorm buffers) is stored under the reference's file name in resources/."""
    from tests.util import build_model
    os.makedirs(os.path.join(path, "resources"), exist_ok=True)
    if not os.path.exists(os.path.join(path, "metadata")):
        shutil.copytree(METADATA, os.path.join(path, "metadata"))
    for name in checkpoints:
        m = build_model(name.split("_")[0])
        torch.save({k: v.clone() for k, v in m.state_dict().items()}, os.path.join(path, "resources", RELEASE_FILE[name]))
    e = dict(os.environ)
    e.update(SCRIPT_ENV)
    if env:
        e.update(env)
    sys.path.insert(0, os.path.join(REPO, "dropin", "datasets"))
    try:
        import importlib.util
        spec = importlib.util.spec_from_file_location("_synth_audioset", os.path.join(REPO, "dropin", "datasets", "audioset.py"))
        mod = importlib.util.module_from_spec(spec)
        old = {k: os.environ.get(k) for k in SCRIPT_ENV}
        os.environ.update({k: e[k] for k in SCRIPT_ENV})
        spec.loader.exec_module(mod)
        mod.write_teacher_files(os.path.join(path, "resources"))
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    finally:
        sys.path.pop(0)
    return e


def run_script(workdir, side, script, args, env, seed=0, no_dropout=True, log_json=None, keep_checkpoint=None, timeout=1200,
               extra=()):
    root = ref_root()
    cmd = [sys.executable, LAUNCHER, "--side", side, "--ref-root", root, "--seed", str(seed)] + list(extra)
    if no_dropout:
        cmd.append("--no-dropout")
    if log_json:
        cmd += ["--log-json", log_json]
    if keep_checkpoint:
        cmd += ["--keep-checkpoint", keep_checkpoint]
    cmd += [script, "--"] + list(args)
    r = subprocess.run(cmd, cwd=workdir, env=env, capture_output=True, text=True, timeout=timeout)
    return r


def read_log(path):
    with open(path) as f:
        return json.load(f)


def parse_windowed_stdout(text):
    """windowed_inference.py:144-148 prints `Window: s - e` followed by five `\t<tag>: <p:.2f>` lines per window
    -> [{"start": s, "end": e, "tags": [[tag, p], ...]}]"""
    import re
    out = []
    for line in text.splitlines():
        m = re.match(r"^Window: (\d+\.\d+) - (\d+\.\d+)$", line.strip())
        if m:
            out.append({"start": float(m.group(1)), "end": float(m.group(2)), "tags": []})
            continue
        m = re.match(r"^\t(.+): (\d\.\d{2})$", line)
        if m and out:
            out[-1]["tags"].append([m.group(1), float(m.group(2))])
    return out
