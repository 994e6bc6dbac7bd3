"""Pins oracle/adanerf_oracle.py against fixtures produced by the unmodified reference
(oracle/gen_golden.py)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_golden, case_weights
from oracle import adanerf_oracle as orc

CASES = ["pav_k8_t0.2", "pav_k8_t0.5", "pav_k16_t0.15", "shaped_k8_t0.2", "rand_k8_t0.2", "ndc_k16_t0.15"]


def _run(case):
    g = load_golden(case)
    m = g["meta"]
    sd0, sd1 = case_weights(case)
    out = orc.render_rays(torch.from_numpy(g["pose"]), torch.from_numpy(g["rot"]), torch.from_numpy(g["dirs"]),
                          sd0, sd1, m["scene_params"], m["thr"], m["K"], return_stages=True)
    return g, m, out


@pytest.mark.parametrize("case", CASES)
def test_geometry_and_features_match_reference(case):
    g, m, o = _run(case)
    # elementwise fp32 ops: identical on any IEEE host
    np.testing.assert_array_equal(o["ray_d"].numpy(), g["ray_d"])
    np.testing.assert_allclose(o["ray_o"].numpy(), g["ray_o"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(o["x0"].numpy(), g["x0"], rtol=0, atol=2e-4)


@pytest.mark.parametrize("case", CASES)
def test_stage2_bit_exact_on_reference_raw0(case):
    """Feed the reference's own raw0: counts, cells, order and z must match bit for bit."""
    g = load_golden(case)
    m = g["meta"]
    s2 = orc.stage2_sample(torch.from_numpy(g["raw0"]), m["thr"], m["K"], m["scene_params"]["depth_range"],
                           no_depth_range=bool(m["scene_params"].get("use_ndc")))
    z = s2["z"].numpy().copy()
    z[~np.isfinite(z)] = np.nan
    np.testing.assert_array_equal(z, g["z_nan"])
    np.testing.assert_array_equal((s2["count"].numpy() / m["K"]).astype(np.float32), g["asp"])


@pytest.mark.parametrize("case", CASES)
def test_end_to_end_matches_reference(case):
    g, m, o = _run(case)
    # GEMM rounding may differ between hosts (oneMKL kernel selection), so raw0 is close, not equal;
    # a borderline cell may flip, which changes single rays -> compare robustly.
    np.testing.assert_allclose(o["raw0"].numpy(), g["raw0"], rtol=0, atol=5e-4)
    same = (o["asp"].numpy() == g["asp"])
    assert same.mean() > 0.98
    diff = np.abs(o["rgb"].numpy() - g["rgb"])[same]
    assert diff.max() < 2e-3
    assert orc.psnr(o["rgb"].numpy()[same], g["rgb"][same]) > 60.0


@pytest.mark.parametrize("case", ["pav_k8_t0.2", "pav_k8_t0.5", "shaped_k8_t0.2"])
def test_auxiliary_outputs_match_reference(case):
    """NeRFWeightsOutput / NeRFAlphaOutput / NeRFOutputDepth of the reference's inference dict (features.py:566-577)
    on the rays whose sample set the host's GEMM rounding did not change."""
    g, m, o = _run(case)
    same = (o["asp"].numpy() == g["asp"])
    assert same.mean() > 0.98
    np.testing.assert_allclose(o["weights"].numpy()[same], g["weights"][same], rtol=0, atol=2e-3)
    np.testing.assert_allclose(o["alpha"].numpy()[same], g["alpha"][same], rtol=0, atol=2e-3)
    np.testing.assert_allclose(o["depth_est"].numpy()[same], g["depth_est"][same, 0], rtol=0, atol=2e-3)
    # and exactly, given the reference's own per-sample network output: composite + log warp are elementwise fp32
    K, n = m["K"], g["weights"].shape[0]
    mapping = torch.from_numpy(np.isfinite(g["z_nan"]).reshape(-1))
    raw1 = torch.from_numpy(g["raw1_pad"].reshape(-1, 4))[mapping]
    zs = torch.from_numpy(g["z_nan"].reshape(-1))[mapping]
    s2 = orc.stage2_sample(torch.from_numpy(g["raw0"]), m["thr"], K, m["scene_params"]["depth_range"],
                           no_depth_range=bool(m["scene_params"].get("use_ndc")))
    comp = orc.stage5_composite(raw1, zs, s2["zp"], mapping, n, K)
    np.testing.assert_allclose(comp["weights"].numpy(), g["weights"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(comp["alpha"].numpy(), g["alpha"], rtol=0, atol=1e-6)
    de = orc.log_from_world(comp["depth_map"], m["scene_params"]["depth_range"]).numpy()
    np.testing.assert_allclose(de, g["depth_est"][:, 0], rtol=0, atol=1e-6)


def test_dense_config1_matches_reference():
    """BASELINE config 1: 1024 rays, dense 128 samples, random init (chunked like evaluate.py:216-235)."""
    g = load_golden("rand_dense_k128")
    m = g["meta"]
    sd0, sd1 = case_weights("rand_dense_k128")
    o = orc.render_rays(torch.from_numpy(g["pose"]), torch.from_numpy(g["rot"]), torch.from_numpy(g["dirs"]),
                        sd0, sd1, m["scene_params"], 0.0, 128, return_stages=True)
    np.testing.assert_allclose(o["raw0"].numpy(), g["raw0"], rtol=0, atol=5e-4)   # OracleWeights
    np.testing.assert_array_equal(o["z"].numpy(), g["z"])
    # random-init nets drive alpha*zp far outside [0,1] (SURVEY 7c): compare with a relative tolerance
    scale = np.abs(g["rgb"]).max()
    assert np.abs(o["rgb"].numpy() - g["rgb"]).max() <= 2e-3 * max(scale, 1.0)


def test_stage2_stress_vectors():
    """Crafted rows through the reference sampler.  torch.sort(descending=True) in the reference
    (nerf_raymarch_common.py:726) is NOT a stable sort, so its choice among exactly tied values is
    implementation-defined; the oracle (and the CUDA path) define ties as lower-cell-index-first.
    Rows without duplicate values must match bit for bit; rows with ties must agree on everything
    that does not depend on the tie order (count, multiset of selected values)."""
    g = load_golden("stage2_stress")
    raw0 = torch.from_numpy(g["raw0"])
    dr = g["meta"]["depth_range"]
    srt = -np.sort(-g["raw0"], axis=1)
    for K in (1, 4, 8, 16, 128):
        for thr in (0.2, 0.5):
            s2 = orc.stage2_sample(raw0, thr, K, dr)
            z, zp = s2["z"].numpy(), s2["zp"].numpy()
            gz, gzp = g[f"z_K{K}_t{thr}"], g[f"zp_K{K}_t{thr}"]
            cnt = (srt >= np.float32(thr)).sum(1)
            # a tie only matters at the arg-max fallback or across the K-th/K+1-th boundary
            has_ties = ((cnt == 0) & (srt[:, 0] == srt[:, 1])) | \
                       ((cnt > K) & (srt[:, min(K, 127) - 1] == srt[:, min(K, 127)]))
            assert (~has_ties).sum() >= 45
            np.testing.assert_array_equal(z[~has_ties], gz[~has_ties])
            np.testing.assert_array_equal(zp[~has_ties], gzp[~has_ties])
            np.testing.assert_array_equal(np.isfinite(z).sum(1), np.isfinite(gz).sum(1))
            np.testing.assert_array_equal(np.sort(zp, 1), np.sort(gzp, 1))
            # ties resolved lower-index-first: z ascending and unique per row
            zz = np.where(np.isfinite(z), z, np.float32(1e30))
            assert (np.diff(zz, axis=1) >= 0).all()


def test_weight_init_is_reproducible():
    a0, a1 = orc.make_weights("rand", seed=3)
    b0, b1 = orc.make_weights("rand", seed=3)
    assert all(torch.equal(a0[k], b0[k]) for k in a0) and all(torch.equal(a1[k], b1[k]) for k in a1)
    assert a0["layers.0.weight"].shape == (256, 90) and a1["pts_linears.5.weight"].shape == (256, 319)
    assert a1["views_linears.0.weight"].shape == (128, 283)


@pytest.mark.parametrize("seed,K,thr", [(11, 8, 0.2), (12, 4, 0.05), (13, 16, 0.3)])
def test_live_reference_fresh_seed(seed, K, thr):
    """The reference initialised from a fresh seed by its own initialisers, then run on 512 random rays with a sampling
    net shaped for ragged counts (oracle/gen_golden.py: fresh_seeds).  Exact: the initial weights and the sample
    selection on the reference's own raw0.  To GEMM rounding, which differs between hosts (oneMKL picks its kernels by
    instruction set): raw0, the sample counts, rgb and the compositing weights."""
    from oracle.gen_golden import state_dict_digest
    z = np.load(os.path.join(GOLDEN, "fresh_seeds.npz"), allow_pickle=False)
    ref = {k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(f"s{seed}/")}
    scene = orc.SCENE_BARBERSHOP
    sd0, sd1 = orc.make_weights("rand", seed=seed)
    assert [state_dict_digest(sd0), state_dict_digest(sd1)] == ref["init_digest"].tolist()
    # shape the sampling net so counts are ragged (the reference ran on the same weights)
    sd0["layers.7.weight"] *= 0.15
    sd0["layers.7.bias"] = sd0["layers.7.bias"] * 0.15 - 0.2
    dirs = torch.from_numpy(orc.generate_ray_directions(800, 800, scene["fov"]).reshape(-1, 3)).float()
    dirs = dirs[torch.from_numpy(ref["pix"]).long()]
    pose, rot = torch.from_numpy(ref["pose"]), torch.from_numpy(ref["rot"])
    s2 = orc.stage2_sample(torch.from_numpy(ref["raw0"]), thr, K, scene["depth_range"])
    np.testing.assert_array_equal((s2["count"].numpy() / K).astype(np.float32), ref["asp"][ref["raw0_rows"]])
    o = orc.render_rays(pose, rot, dirs, sd0, sd1, scene, thr, K, return_stages=True)
    np.testing.assert_allclose(o["raw0"].numpy()[ref["raw0_rows"]], ref["raw0"], rtol=0, atol=5e-4)
    same = o["asp"].numpy() == ref["asp"]
    assert same.mean() > 0.98
    np.testing.assert_allclose(o["rgb"].numpy()[same], ref["rgb"][same], rtol=0, atol=2e-4)
    np.testing.assert_allclose(o["weights"].numpy()[same], ref["weights"][same], rtol=0, atol=2e-4)
