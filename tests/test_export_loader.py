"""Export-directory format (config.ini + dataset_info.txt + model{0,1}.onnx): Python and C++ readers, CPU only."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from conftest import ROOT
from adanerf_b200 import onnx_weights as ow
from oracle import adanerf_oracle as orc


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from adanerf_b200 import load_library
    return load_library()


def test_onnx_round_trip(tmp_path):
    sd0, sd1 = orc.make_weights("rand", seed=4)
    p = tmp_path / "m.onnx"
    ow.write_onnx_initializers(str(p), {k: v.numpy() for k, v in sd1.items()})
    back = ow.read_onnx_initializers(str(p))
    assert list(back) == list(sd1)
    for k, v in sd1.items():
        np.testing.assert_array_equal(back[k], v.numpy())


def test_cxx_loader_reads_export_dir(lib, tmp_path):
    from adanerf_b200._lib import Scene
    scene = orc.SCENE_PAVILLON
    sd0, sd1 = orc.make_weights("rand", seed=1)
    d = tmp_path / "export"
    ow.write_export_dir(str(d), scene, sd0, sd1, 0.15, 16)
    sc, thr, k, n = Scene(), C.c_float(), C.c_int(), (C.c_int * 2)()
    st = lib.adn_probe_export_dir(str(d).encode(), C.byref(sc), C.byref(thr), C.byref(k), n)
    assert st == 0
    assert abs(thr.value - 0.15) < 1e-7 and k.value == 16
    assert list(n) == [16, 24]                     # initialiser counts of model0 / model1 (SURVEY 8b)
    np.testing.assert_allclose(list(sc.view_cell_center), scene["view_cell_center"], rtol=1e-6)
    np.testing.assert_allclose(list(sc.depth_range), scene["depth_range"], rtol=1e-6)
    assert abs(sc.fov - scene["fov"]) < 1e-6 and abs(sc.max_depth - scene["max_depth"]) < 1e-5
    assert (sc.n_freq_pos, sc.n_freq_dir) == (10, 4)


def test_cxx_loader_errors(lib, tmp_path):
    assert lib.adn_probe_export_dir(str(tmp_path / "missing").encode(), None, None, None, None) == 5   # ADN_ERR_IO
    d = tmp_path / "bad"
    os.makedirs(d)
    (d / "config.ini").write_text("numRaymarchSamples = [8, 8]\n")
    (d / "dataset_info.txt").write_text("fov = 1.0\n")
    assert lib.adn_probe_export_dir(str(d).encode(), None, None, None, None) == 5


def test_cxx_loader_reads_shipped_sample(lib):
    """The export directory the reference's viewer ships (adanerf_real_time_viewer/sample): config.ini and
    dataset_info.txt verbatim, model{0,1}.onnx as exported with every initialiser cut to its leading 4 x 4 block."""
    from adanerf_b200._lib import Scene
    sc, thr, k, n = Scene(), C.c_float(), C.c_int(), (C.c_int * 2)()
    d = os.path.join(ROOT, "tests", "golden", "viewer_sample")
    st = lib.adn_probe_export_dir(d.encode(), C.byref(sc), C.byref(thr), C.byref(k), n)
    assert st == 0 and k.value == 4 and abs(thr.value - 0.15) < 1e-7 and list(n) == [16, 24]
    np.testing.assert_allclose(list(sc.view_cell_center), [2.25, 7.75, 1.5])


@pytest.mark.gpu
def test_render_from_export_dir_matches_state_dict(tmp_path):
    from adanerf_b200 import Renderer
    scene = orc.SCENE_BARBERSHOP
    sd0, sd1 = orc.make_weights("shaped", seed=0)
    d = tmp_path / "export"
    ow.write_export_dir(str(d), scene, sd0, sd1, 0.2, 8)
    r1, thr, K = Renderer.from_export_dir(str(d))
    assert (K, round(thr, 4)) == (8, 0.2)
    r2 = Renderer(scene, sampling_net=sd0, shading_net=sd1)
    pose, rot = torch.tensor(scene["view_cell_center"]), torch.eye(3)
    a = r1.render_camera(pose, rot, 200, 200, thr, K)["rgb"]
    b = r2.render_camera(pose, rot, 200, 200, 0.2, 8)["rgb"]
    assert torch.equal(a, b)
    r1.close()
    r2.close()


def test_weights_checkpoints_to_export_dir(lib, tmp_path):
    """`.weights` (torch.save(state_dict), src/models.py:87-90) -> export directory -> C++ loader."""
    import ctypes as C
    import torch
    from adanerf_b200 import convert
    from adanerf_b200._lib import Scene
    sd0, sd1 = orc.make_weights("rand", seed=5)
    torch.save(sd0, tmp_path / "Net0_opt.weights")
    torch.save(sd1, tmp_path / "Net1_opt.weights")
    scene = orc.SCENE_PAVILLON
    with open(tmp_path / "dataset_info.txt", "w") as f:
        for k in ("view_cell_center", "view_cell_size", "depth_range", "fov", "max_depth"):
            f.write(f"{k} = {scene[k]}\n")
    out = tmp_path / "export"
    convert.main(["--weights0", str(tmp_path / "Net0_opt.weights"), "--weights1", str(tmp_path / "Net1_opt.weights"),
                  "--dataset-info", str(tmp_path / "dataset_info.txt"), "--threshold", "0.15", "--samples", "16", "--out", str(out)])
    sc, thr, K, nt = Scene(), C.c_float(), C.c_int(), (C.c_int * 2)()
    assert lib.adn_probe_export_dir(str(out).encode(), C.byref(sc), C.byref(thr), C.byref(K), nt) == 0
    assert abs(thr.value - 0.15) < 1e-7 and K.value == 16 and list(nt) == [len(sd0), len(sd1)]
    assert abs(sc.max_depth - scene["max_depth"]) < 1e-6
    back = ow.read_onnx_initializers(str(out / "model1.onnx"))
    np.testing.assert_array_equal(back["rgb_linear.weight"], sd1["rgb_linear.weight"].numpy())
    # wrong architecture is rejected with a message
    bad = dict(sd1)
    del bad["views_linears.0.weight"]
    torch.save(bad, tmp_path / "bad.weights")
    with pytest.raises(ValueError, match="views_linears"):
        convert.weights_to_export_dir(tmp_path / "Net0_opt.weights", tmp_path / "bad.weights", tmp_path / "x", scene, 0.2, 8)


def test_cxx_loader_reads_ndc_export(lib, tmp_path):
    """configs/fine_training_ndc.ini exports: useNDC, [2-2, 10-4], NoDepthRange sampler, normalisation None."""
    sd0, sd1 = orc.make_weights("ndc", seed=0)
    d = tmp_path / "ndc"
    ow.write_export_dir(str(d), orc.SCENE_PAVILLON_NDC, sd0, sd1, 0.15, 16)
    from adanerf_b200._lib import Scene
    sc, thr, K, nt = Scene(), C.c_float(), C.c_int(), (C.c_int * 2)()
    assert lib.adn_probe_export_dir(str(d).encode(), C.byref(sc), C.byref(thr), C.byref(K), nt) == 0
    assert (sc.use_ndc, sc.n_freq_pos0, sc.n_freq_dir0, sc.n_freq_pos, sc.n_freq_dir) == (1, 2, 2, 10, 4)
    assert (sc.ndc_w, sc.ndc_h, K.value) == (800, 800, 16)
    # an NDC flag with the depth-range sampler is inconsistent -> rejected
    cfg = (d / "config.ini").read_text().replace("FromClassifiedDepthAdaptiveNoDepthRange", "FromClassifiedDepthAdaptive")
    (d / "config.ini").write_text(cfg)
    assert lib.adn_probe_export_dir(str(d).encode(), C.byref(sc), C.byref(thr), C.byref(K), nt) == 5


@pytest.mark.gpu
def test_render_from_ndc_export_dir_matches_state_dict(tmp_path):
    from adanerf_b200 import Renderer
    scene = orc.SCENE_PAVILLON_NDC
    sd0, sd1 = orc.make_weights("ndc", seed=0)
    d = tmp_path / "export_ndc"
    ow.write_export_dir(str(d), scene, sd0, sd1, 0.15, 16)
    r1, thr, K = Renderer.from_export_dir(str(d))
    r2 = Renderer(scene, sampling_net=sd0, shading_net=sd1)
    pose, rot = torch.tensor(scene["view_cell_center"]), torch.eye(3)
    a = r1.render_camera(pose, rot, 200, 160, thr, K)["rgb"]
    b = r2.render_camera(pose, rot, 200, 160, 0.15, 16)["rgb"]
    assert torch.isfinite(a).all() and torch.equal(a, b)
    r1.close()
    r2.close()


def test_truncated_onnx_is_an_error_not_a_short_model(lib, tmp_path):
    """A model file cut in the middle of a field must fail loading (ADN_ERR_IO / ValueError), not parse as a model with
    fewer initialisers (ADVICE r1: next_field advanced past the end on fixed-width fields)."""
    scene = orc.SCENE_PAVILLON
    sd0, sd1 = orc.make_weights("rand", seed=2)
    d = tmp_path / "export"
    ow.write_export_dir(str(d), scene, sd0, sd1, 0.2, 8)
    whole = (d / "model1.onnx").read_bytes()
    for cut in (len(whole) - 1, len(whole) - 3, len(whole) // 2, 37):
        (d / "model1.onnx").write_bytes(whole[:cut])
        assert lib.adn_probe_export_dir(str(d).encode(), None, None, None, None) == 5, cut   # ADN_ERR_IO
        with pytest.raises(ValueError):
            ow.read_onnx_initializers(str(d / "model1.onnx"))
    # a fixed-width field (wire type 1 / 5) whose payload is missing
    (d / "model1.onnx").write_bytes(whole + bytes([0x09, 0x01, 0x02]))      # field 1, wire type 1, 2 of 8 bytes
    assert lib.adn_probe_export_dir(str(d).encode(), None, None, None, None) == 5
    with pytest.raises(ValueError):
        ow.read_onnx_initializers(str(d / "model1.onnx"))


def test_pickled_module_checkpoints_need_an_explicit_flag(tmp_path):
    """`.weights` files are plain state_dicts (src/models.py:87-90); anything that needs unpickling is refused unless
    the caller opts in (ADVICE r1)."""
    from adanerf_b200 import convert
    net = torch.nn.Linear(3, 2)
    torch.save(net, tmp_path / "module.weights")            # a pickled nn.Module
    with pytest.raises(ValueError, match="allow_pickle"):
        convert.load_weights_file(tmp_path / "module.weights")
    sd = convert.load_weights_file(tmp_path / "module.weights", allow_pickle=True)
    assert set(sd) == {"weight", "bias"}
    torch.save(net.state_dict(), tmp_path / "plain.weights")
    assert set(convert.load_weights_file(tmp_path / "plain.weights")) == {"weight", "bias"}
