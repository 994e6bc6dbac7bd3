"""TrainConfig.inference drop-in (adanerf_b200.adapter) against the golden output of the reference's own
inference() call on the same batch."""
import numpy as np
import pytest
import torch

from conftest import case_weights, load_golden

pytestmark = pytest.mark.gpu


class _Batch:   # what SampleDataWrapper.get_batch_input returns (src/datasets.py:70-80)
    def __init__(self, d):
        self.d = d

    def get_batch_input(self, i):
        return self.d


@pytest.mark.parametrize("case", ["pav_k8_t0.5", "shaped_k8_t0.2"])
def test_inference_adapter_matches_reference(case):
    from adanerf_b200.adapter import B200Inference
    from oracle import adanerf_oracle as orc
    g = load_golden(case)
    m = g["meta"]
    sd0, sd1 = case_weights(case)
    inf = B200Inference(m["scene_params"], sd0, sd1, m["thr"], m["K"])
    batch = _Batch({"ImagePose": torch.from_numpy(g["pose"]).reshape(1, 3).cuda(),
                    "ImageRotation": torch.from_numpy(g["rot"]).reshape(1, 3, 3).cuda(),
                    "RayDirectionsSamples": torch.from_numpy(g["dirs"]).reshape(1, -1, 3).cuda()})
    outs, dicts = inf.inference(batch, gradient=False, is_inference=True)
    rgb = outs[-1][:, :3].cpu().numpy()
    np.testing.assert_array_equal(dicts[-1]["AdaptiveSamplePositions"].cpu().numpy(), g["asp"])
    assert orc.psnr(rgb, g["rgb"]) >= 49.4
    assert torch.equal(dicts[-1]["PostProcessedNetworkOutput"], outs[-1])
    with pytest.raises(NotImplementedError):
        inf.inference(batch, gradient=True)


def test_inference_adapter_dense_returns_oracle_weights():
    from adanerf_b200.adapter import B200Inference
    g = load_golden("rand_dense_k128")
    m = g["meta"]
    sd0, sd1 = case_weights("rand_dense_k128")
    inf = B200Inference(m["scene_params"], sd0, sd1, 0.0, 128)
    batch = _Batch({"ImagePose": torch.from_numpy(g["pose"]).reshape(1, 3), "ImageRotation": torch.from_numpy(g["rot"]).reshape(1, 3, 3),
                    "RayDirectionsSamples": torch.from_numpy(g["dirs"]).reshape(1, -1, 3)})
    outs, dicts = inf.inference(batch, gradient=False, is_inference=True)
    ow = dicts[1]["OracleWeights"].cpu().numpy()
    np.testing.assert_allclose(ow, g["raw0"], rtol=0, atol=2e-4 * np.abs(g["raw0"]).max())
    assert "AdaptiveSamplePositions" not in dicts[1]


def test_inference_adapter_auxiliary_dict_entries():
    """want_aux=True: the keys plots.render_all_imgs / the depth export read (src/plots.py:272-306)."""
    g = load_golden("pav_k8_t0.2")
    m = g["meta"]
    sd0, sd1 = case_weights("pav_k8_t0.2")
    from adanerf_b200.adapter import B200Inference
    inf = B200Inference(m["scene_params"], sd0, sd1, m["thr"], m["K"], want_aux=True)
    batch = _Batch({"ImagePose": torch.from_numpy(g["pose"]).reshape(1, 3).cuda(),
                    "ImageRotation": torch.from_numpy(g["rot"]).reshape(1, 3, 3).cuda(),
                    "RayDirectionsSamples": torch.from_numpy(g["dirs"]).reshape(1, -1, 3).cuda()})
    outs, dicts = inf.inference(batch, gradient=False, is_inference=True)
    d1 = dicts[1]
    n, K = g["dirs"].shape[0], m["K"]
    assert d1["NeRFWeightsOutput"].shape == (n, K) and d1["NeRFAlphaOutput"].shape == (n, K)
    assert d1["NeRFInputFeatureZVals"].shape == (n, K) and d1["NeRFOutputDepth"].shape == (n, 1)
    same = np.round(d1["AdaptiveSamplePositions"].cpu().numpy() * K) == np.round(g["asp"] * K)
    np.testing.assert_allclose(d1["NeRFOutputDepth"].cpu().numpy()[same], g["depth_est"][same], rtol=0, atol=2e-2)
    np.testing.assert_allclose(d1["NeRFWeightsOutput"].cpu().numpy()[same], g["weights"][same], rtol=0, atol=2e-2)


class _NS:
    def __init__(self, **kw):
        self.__dict__.update(kw)


def _duck_train_config(m, sd0, sd1, K, thr):
    """An object with exactly the attributes B200Inference.from_train_config reads from an initialised reference
    TrainConfig (tests/test_adapter_config.py pins those names against the fields of a reference TrainConfig)."""
    sp = m["scene_params"]
    view = _NS(view_cell_center=sp["view_cell_center"], view_cell_size=sp["view_cell_size"], fov=sp["fov"], focal=None)
    f1 = _NS(depth_range=sp["depth_range"], max_depth=sp["max_depth"], z_near=0.001, z_far=1.0, useNDC=False,
             z_sampler=_NS(threshold=thr), n_ray_samples=K)
    return _NS(f_in=[None, f1], dataset_info=_NS(view=view), models=[sd0, sd1])


def test_from_train_config_renders_like_the_reference():
    """The line INTEGRATION.md tells a maintainer to paste: B200Inference.from_train_config(train_config)."""
    from adanerf_b200.adapter import B200Inference
    from oracle import adanerf_oracle as orc
    g = load_golden("pav_k8_t0.2")
    m = g["meta"]
    sd0, sd1 = case_weights("pav_k8_t0.2")
    inf = B200Inference.from_train_config(_duck_train_config(m, sd0, sd1, m["K"], m["thr"]))
    assert inf.K == m["K"] and abs(inf.threshold - m["thr"]) < 1e-7
    batch = _Batch({"ImagePose": torch.from_numpy(g["pose"]).reshape(1, 3).cuda(),
                    "ImageRotation": torch.from_numpy(g["rot"]).reshape(1, 3, 3).cuda(),
                    "RayDirectionsSamples": torch.from_numpy(g["dirs"]).reshape(1, -1, 3).cuda()})
    outs, dicts = inf.inference(batch, gradient=False, is_inference=True)
    np.testing.assert_array_equal(dicts[-1]["AdaptiveSamplePositions"].cpu().numpy(), g["asp"])
    assert orc.psnr(outs[-1][:, :3].cpu().numpy(), g["rgb"]) >= 49.4
