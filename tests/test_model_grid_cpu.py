"""Model grid searches without a GPU: checkpoint fingerprints and the refusals that come before any GPU work."""
import numpy as np
import pytest


def test_lsq_fingerprint_unchanged_and_model_parameters_change_it():
    from helicon_b200.checkpoint import fingerprint
    from helicon_b200.engine import model_params
    from helicon_b200.grid import model_fingerprint

    img = np.arange(64, dtype=np.float32).reshape(8, 8)
    axes = (np.array([1.0]), np.array([2.0, 3.0]), np.array([4.0]))
    base = dict(apix=1.0, positive_constraint=-1)
    lsq = fingerprint(img, axes, **base)
    for alg in (None, dict(model="lsq")):
        assert fingerprint(img, axes, **base, **model_fingerprint(model_params(alg))) == lsq
    fps = {fingerprint(img, axes, **base, **model_fingerprint(model_params(a)))
           for a in (dict(model="elasticnet"), dict(model="elasticnet", alpha=1e-3), dict(model="elasticnet", l1_ratio=0.7),
                     dict(model="lasso"), dict(model="ridge"))}
    assert len(fps) == 5 and lsq not in fps


@pytest.mark.parametrize("alg,interp,exc", [
    (dict(model="lreg"), "nn", NotImplementedError),
    (dict(model="ard"), "nn", NotImplementedError),
    (dict(model="no_such_model"), "nn", NotImplementedError),
    (dict(model="elasticnet"), "linear", NotImplementedError),
    (dict(model="elasticnet", alpha=-1.0), "nn", ValueError),
    (dict(model="ridge", alpha=0.0), "nn", ValueError),
])
def test_search_grid_and_cli_refuse_before_gpu_work(alg, interp, exc, tmp_path):
    from helicon_b200 import denovo3DBatch
    from helicon_b200.grid import search_grid

    with pytest.raises(exc):
        search_grid(np.ones((16, 16), np.float32), 1.0, [10.0], [3.0], interpolation=interp, algorithm=alg)
    if alg["model"] in ("lreg", "ard", "no_such_model"):
        with pytest.raises(SystemExit):  # argparse choices
            denovo3DBatch.main(["x.mrc", "--twist", "10", "--rise", "3", "--model", alg["model"]])
        return
    args = ["x.mrc", "--apix", "1", "--twist", "10", "--rise", "3", "--model", alg["model"], "--interpolation", interp]
    if "alpha" in alg:
        args += ["--alpha", str(alg["alpha"])]
    with pytest.raises(exc):
        denovo3DBatch.main(args)
