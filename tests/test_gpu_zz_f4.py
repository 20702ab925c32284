"""SURVEY.md section 8 row f4: ensemble + windowed inference.  (Named zz_ so that it is collected after the older files.)

  * the reference's inference.py (`--ensemble`) and windowed_inference.py run UNCHANGED on this package (launcher and
    workdir as in tests/test_gpu_refscripts.py) and print what the reference-modules run printed;
  * the native, window-batched `efficientat_b200.windowed.EATagger` returns the reference EATagger's windows, labels and
    probabilities (full precision, from tests/golden/windowed_driver.py run with the reference's own modules on CPU);
  * an ensemble with a DyMN member equals the mean of the members' golden logits.

Expected numbers: tests/golden/script_f4.json (tests/golden/make_golden.py script_f4)."""
import json
import os
import sys

import numpy as np
import pytest
import torch

from tests import refscripts as R
from tests.util import GOLDEN, build_model, golden, net_inputs, report

pytestmark = pytest.mark.gpu
needs_ref = pytest.mark.skipif(R.ref_root() is None, reason="oracle/_ref (mirror of the reference checkout that build() "
                               "makes) not present")


def _golden():
    with open(os.path.join(GOLDEN, "script_f4.json")) as f:
        return json.load(f)


def _wav():
    return R.WAV


def _same_ranking(got, want, tol):
    """got / want: [[label, probability], ...] in printed order.  The r-th probability must agree within `tol`; a label may
    differ from the reference's only where the reference itself separates the two classes by less than `tol`."""
    assert len(got) == len(want), (got, want)
    ref_prob = {a: b for a, b in want}
    for r, ((lab, prob), (wlab, wprob)) in enumerate(zip(got, want)):
        assert abs(float(prob) - wprob) <= tol, (r, lab, prob, wlab, wprob)
        if lab != wlab:
            assert lab in ref_prob and abs(ref_prob[lab] - wprob) <= tol, (r, lab, wlab)


@needs_ref
def test_inference_py_ensemble_runs_unchanged(tmp_path):
    """inference.py --cuda --ensemble mn04_as mn10_as: `models.ensemble.get_ensemble_model` resolves to this package's
    EnsemblerModel, both members load through the reference's release-file path."""
    import re
    g = _golden()
    wd = str(tmp_path)
    env = R.make_workdir(wd, checkpoints=tuple(g["ensemble"]))
    r = R.run_script(wd, "ours", "inference.py", ["--cuda", "--ensemble"] + g["ensemble"] + ["--audio_path", _wav()], env,
                     no_dropout=False)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    rows = [[a, float(b)] for a, b in re.findall(r"^(.+): (\d\.\d{3})$", r.stdout, flags=re.M)]
    report(f"[parity] inference.py --ensemble {' '.join(g['ensemble'])} top-10 (ours): {rows}")
    _same_ranking(rows, g["inference_ensemble_top10"], 2e-3)


@needs_ref
def test_windowed_inference_py_runs_unchanged(tmp_path):
    """windowed_inference.py --cuda, 2 s windows / 1 s hop over the 10 s fixture = 9 windows.  The script imports
    get_ensemble_model from models.mn.model (windowed_inference.py:8); dropin/models/mn/model.py exports it."""
    g = _golden()
    wd = str(tmp_path)
    env = R.make_workdir(wd, checkpoints=("mn10_as",))
    r = R.run_script(wd, "ours", "windowed_inference.py",
                     ["--cuda", "--model", "mn10_as", "--audio_path", _wav(), "--window_size", str(g["window_s"]),
                      "--hop_length", str(g["hop_s"])], env, no_dropout=False)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    got = R.parse_windowed_stdout(r.stdout)
    assert len(got) == len(g["windowed_stdout"]) == 9, r.stdout
    for w, (a, b) in enumerate(zip(got, g["windowed_stdout"])):
        assert (a["start"], a["end"]) == (b["start"], b["end"])
        _same_ranking(a["tags"], b["tags"], 0.0101)              # the script prints two decimals
    report(f"[parity] windowed_inference.py: 9 windows, first {got[0]['tags'][:2]} (reference {g['windowed_stdout'][0]['tags'][:2]})")


def _shim_loader():
    """the launcher's stand-in for librosa.core.load (scipy wav read + polyphase resampling), as the golden run used it"""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_eat_launcher", R.LAUNCHER)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    saved = {k: sys.modules.get(k) for k in ("librosa", "librosa.core")}
    mod._install_librosa_shim()
    load = sys.modules["librosa"].load
    for k, v in saved.items():
        if v is None:
            sys.modules.pop(k, None)
        else:
            sys.modules[k] = v
    return load


@pytest.mark.parametrize("which", ["windowed_mn10", "windowed_ensemble"])
def test_native_batched_tagger_matches_reference_eatagger(tmp_path, monkeypatch, which):
    """efficientat_b200.windowed.EATagger: all 9 windows through ONE mel launch and ONE forward at batch 9, top-k on the
    device -- against the reference EATagger's per-window loop (reference modules, CPU fp32, full precision)."""
    from efficientat_b200.windowed import EATagger
    g = _golden()
    names = ["mn10_as"] if which == "windowed_mn10" else g["ensemble"]
    R.make_workdir(str(tmp_path), checkpoints=tuple(names))
    monkeypatch.chdir(tmp_path)                                    # resources/<release file>, metadata/ relative to the CWD
    tagger = EATagger(model_name=names[0]) if len(names) == 1 else EATagger(ensemble=names)
    wave, sr = _shim_loader()(_wav(), sr=32000, mono=True)
    assert sr == 32000
    tags = tagger.tag_waveform(wave, window_size=g["window_s"], hop_length=g["hop_s"])
    want = g[which]
    assert len(tags) == len(want) == 9
    worst = 0.0
    for a, b in zip(tags, want):
        assert (a["start"], a["end"]) == (b["start"], b["end"])
        got = [[t["tag"], t["probability"]] for t in a["tags"]]
        assert len(got) == 10
        _same_ranking(got, b["tags"], 5e-4)
        worst = max(worst, max(abs(x[1] - y[1]) for x, y in zip(got, b["tags"])))
    report(f"[parity] native batched EATagger {which}: 9 windows x top-10, worst probability err {worst:.2e}")
    # chunked batches (4 + 4 + 1 windows) against one batch of 9: the same probabilities.  Not bit-identical: a 1x1
    # convolution runs on the tensor cores (bf16x3 products, 2^-16 each) from 1024 rows on and on the exact-fp32 CUDA-core
    # GEMM below, and the row count scales with the batch -- the bound is the parity bound of the two routes (1e-4 on logits)
    p_full, _, _ = tagger.window_probabilities(wave, window_size=g["window_s"], hop_length=g["hop_s"])
    tagger.max_batch = 4
    p_chunk, _, _ = tagger.window_probabilities(wave, window_size=g["window_s"], hop_length=g["hop_s"])
    assert p_full.shape == p_chunk.shape == (9, 527)
    assert torch.isfinite(p_full).all() and torch.isfinite(p_chunk).all()
    diff = (p_full - p_chunk).abs().max().item()
    report(f"[parity] native batched EATagger {which}: batches of 4 vs one batch of 9, max probability diff {diff:.2e}")
    assert diff <= 1e-4
    again = tagger.tag_waveform(wave, window_size=g["window_s"], hop_length=g["hop_s"])
    for a, b in zip(again, want):                                 # and the chunked run meets the reference like the full one
        _same_ranking([[t["tag"], t["probability"]] for t in a["tags"]], b["tags"], 5e-4)


def test_ensemble_with_dymn_member_is_the_mean_of_the_golden_logits():
    """models/ensemble.py:14-23 with an MN and a DyMN member at the synthetic golden inputs (mn04 and dymn04 goldens share
    the input spectrogram): mean of the two reference logit vectors, returned twice."""
    from efficientat_b200.models.ensemble import EnsemblerModel
    spec, _ = net_inputs("mn04")
    spec2, _ = net_inputs("dymn04")
    assert torch.equal(spec, spec2)
    ens = EnsemblerModel([build_model("mn04"), build_model("dymn04")]).cuda().eval()
    with torch.no_grad():
        a, b = ens(spec.cuda())
    assert a is b
    want = (golden("mn04")["eval_logits"] + golden("dymn04")["eval_logits"]) / 2
    err = np.abs(a.cpu().numpy() - want).max()
    report(f"[parity] ensemble mn04 + dymn04: logit max-abs err {err:.3e}")
    assert err < 1e-3
