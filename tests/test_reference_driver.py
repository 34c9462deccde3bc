"""Drop-in proof: the reference's UNMODIFIED quick-start driver (example/00_quick_start/sequential.py:435-522) runs end to end
against this repository - its imports resolve through compat/, its absl flags and prepare_hparams kwargs are accepted, and
fit_step -> tf.train.latest_checkpoint -> load_model -> run_weighted_eval -> predict complete on synthetic wechat-shaped files.

The driver file belongs to the reference project and is not part of this repository, so this test runs only where
PAMREC_REFERENCE names a checkout of it: on a machine with a GPU the real engine runs the device steps, on one without
`StubEngine` (tests/test_host_loops.py) stands in for them - everything between the driver and the C ABI (hparams, iterator,
host loops, checkpoints, metrics) is the product code either way.
tests/test_gpu_quickstart.py runs the same flow on the GPU through compat/'s own copy of the flag set."""
import os
import runpy
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("PAMREC_REFERENCE")
REF_DRIVER = os.path.join(REF, "example", "00_quick_start", "sequential.py") if REF else ""

pytestmark = pytest.mark.skipif(not os.path.isfile(REF_DRIVER), reason="PAMREC_REFERENCE does not name a reference checkout")


@pytest.mark.parametrize("model_flag", ["PAMREC", "MMOE_ORIGINAL", "PLE", "SHAREBOTTOM", "SASREC"])
def test_unmodified_reference_driver_runs(tmp_path, monkeypatch, capsys, lib_built, model_flag):
    from pamrec_b200 import models as M
    from pamrec_b200 import synth
    if not torch.cuda.is_available():
        from test_host_loops import StubEngine
        monkeypatch.setattr(M, "Engine", StubEngine)
    data = tmp_path / "data"
    synth.generate(str(data), "wechat", n_users=120, n_items=600, n_cates=15, mean_len=40, seed=11, eval_per_user=2)
    compat = os.path.join(ROOT, "compat")
    monkeypatch.syspath_prepend(compat)
    monkeypatch.chdir(os.path.join(compat, "example", "00_quick_start"))       # the driver opens ../../reco_utils/.../config/mmoe.yaml
    argv = [REF_DRIVER, "--dataset", "wechat", "--data_path", str(data), "--save_path", str(tmp_path / "ranking"), "--epochs", "1",
            "--batch_size", "100", "--eval_step", "5", "--show_step", "5", "--write_prediction_to_file", "--model", model_flag]
    monkeypatch.setattr(sys, "argv", argv)
    for name in [m for m in sys.modules if m == "reco_utils" or m.startswith("reco_utils.") or m == "tensorflow" or m.startswith("tensorflow.")]:
        monkeypatch.delitem(sys.modules, name)
    with pytest.raises(SystemExit) as done:                                    # absl.app.run ends with sys.exit(main(...))
        runpy.run_path(REF_DRIVER, run_name="__main__")
    assert done.value.code in (None, 0)
    out = capsys.readouterr().out
    assert "start experiment" in out and "Time cost for training is" in out
    # the driver prints the experiment name, then the dict run_weighted_eval returned (QS:517-519)
    lines = out.strip().splitlines()
    last = next(ln for ln in reversed(lines) if ln.startswith("{"))
    res = eval(last, {"__builtins__": {}, "np": np})                           # numpy 2 prints its scalars as np.float64(...)
    for key in ("auc", "logloss", "wauc", "wmrr", "wndcg@2", "whit@10"):       # QS:100-101 metric lists for wechat
        assert key in res and np.isfinite(res[key]), (key, res)
    ckpt_dir = tmp_path / "ranking" / model_flag / "try" / "model"
    assert (ckpt_dir / "checkpoint").exists(), "fit_step saved no checkpoint for tf.train.latest_checkpoint to find"
    preds = np.loadtxt(data / "wechat" / "output.txt")
    n_test = sum(1 for _ in open(data / "wechat" / "test_data"))
    assert preds.shape == (n_test,) and np.isfinite(preds).all()
