"""B200Inference.from_train_config against the fields of a real reference TrainConfig: the attribute names it reads
from an initialised TrainConfig -- f_in[1].{depth_range, max_depth, z_near, z_far, z_sampler.threshold, n_ray_samples},
dataset_info.view.{view_cell_center, view_cell_size, fov} (src/features.py:343-360, 747-767; src/train_data.py:60-110)
-- exist on the real objects and carry the values the renderer needs.  tests/golden/train_config_fields.json holds
those attributes as the unmodified reference set them (oracle/gen_golden.py).  No GPU: only the extraction is exercised."""
import json
import os
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import adanerf_oracle as orc


def _namespace(d):
    return SimpleNamespace(**{k: _namespace(v) if isinstance(v, dict) else v for k, v in d.items()})


def _recorded(K, thr):
    with open(os.path.join(GOLDEN, "train_config_fields.json")) as f:
        return next(c for c in json.load(f)["cases"] if c["K"] == K and c["thr"] == thr)


@pytest.mark.parametrize("K,thr", [(8, 0.2), (16, 0.15)])
def test_scene_and_sampler_fields_from_live_train_config(K, thr):
    from adanerf_b200.adapter import B200Inference
    scene = orc.SCENE_PAVILLON
    rec = _recorded(K, thr)
    models = [object(), object()]
    tc = SimpleNamespace(f_in=[None, _namespace(rec["f_in_1"])], dataset_info=SimpleNamespace(view=_namespace(rec["view"])),
                         models=models)
    got, got_models, got_thr, got_k = B200Inference.args_from_train_config(tc)
    assert got_k == K and abs(got_thr - thr) < 1e-7
    assert got_models[0] is models[0] and got_models[1] is models[1]
    np.testing.assert_allclose(got["view_cell_center"], scene["view_cell_center"], rtol=0, atol=0)
    np.testing.assert_allclose(got["view_cell_size"], scene["view_cell_size"], rtol=0, atol=0)
    np.testing.assert_allclose(got["depth_range"], scene["depth_range"], rtol=1e-7)    # the WARPED range (features.py:355)
    assert abs(got["max_depth"] - scene["max_depth"]) < 1e-6 * scene["max_depth"]
    assert abs(got["fov"] - scene["fov"]) < 1e-7
    assert got["z_near"] == pytest.approx(0.001) and got["z_far"] == pytest.approx(1.0)
    assert not got.get("use_ndc", False)
    # the state_dict names the packer expects (src/models.py:18-82, 200-250)
    assert "layers.7.weight" in rec["state_dict_keys"][0] and "pts_linears.5.weight" in rec["state_dict_keys"][1]
