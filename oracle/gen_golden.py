"""TEST INFRASTRUCTURE -- generates tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference/src, imported through oracle/ref_harness.py) on CPU in the build container.

    python oracle/gen_golden.py            # rewrites tests/golden/
    python oracle/gen_golden.py NAME...    # only the fixtures written by the named functions

The fixtures pin oracle/adanerf_oracle.py (tests/test_oracle_golden.py) and are what the `-m gpu`
parity tests compare the CUDA path with on the GPU box, where /root/reference does not exist.
Every file records torch version + thread count (the reference's GEMMs are ATen/oneMKL calls).
"""
import hashlib
import json
import os
import shutil
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_harness as rh          # noqa: E402
from oracle import adanerf_oracle as orc      # noqa: E402
from adanerf_b200.onnx_weights import read_onnx_initializers, _enc_varint, _field, _fields, _varint  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
RX = torch.tensor([[1, 0, 0], [0, 0, -1], [0, 1, 0]], dtype=torch.float32)  # camera -z -> world +y


def meta(**kw):
    kw.update(torch_version=torch.__version__, threads=torch.get_num_threads(),
              generator="oracle/gen_golden.py via oracle/ref_harness.py (unmodified reference)")
    return np.array(json.dumps(kw))


def save(name, **arrays):
    path = os.path.join(OUT, name)
    np.savez_compressed(path, **arrays)
    print(f"wrote {path}  ({os.path.getsize(path) / 1e6:.2f} MB)")


def stage_case(name, scene_name, scene, sd0, sd1, K, thr, n_rays, stride, pose_off, rot, keep_x1, w=800, h=800, ndc=False):
    dirs_all = torch.from_numpy(rh.generate_ray_directions(
        w, h, scene["fov"], 0.5 * w / np.tan(0.5 * scene["fov"])).reshape(-1, 3)).float()
    pix = (torch.arange(n_rays) * stride) % (w * h)
    dirs = dirs_all[pix]
    pose = torch.tensor(scene["view_cell_center"], dtype=torch.float32) + torch.tensor(pose_off, dtype=torch.float32)
    r = rh.RefRenderer(scene, K=K, thr=thr, w=w, h=h, ndc=ndc)
    r.load_state_dicts(sd0, sd1)
    st = r.stages(pose, rot, dirs)
    arrays = dict(meta=meta(case=name, scene=scene_name, K=K, thr=thr, w=w, h=h, scene_params=scene),
                  pix=pix.numpy().astype(np.int64), dirs=dirs.numpy(), pose=pose.numpy(), rot=rot.numpy(),
                  x0=st["x0"], raw0=st["raw0"], ray_o=st["ray_o"], ray_d=st["ray_d"], rgb=st["rgb"],
                  weights=st["weights"], alpha=st["alpha"], depth_est=st["depth_est"])
    if thr > 0:
        z = st["z_nan"]
        arrays.update(z_nan=z, asp=st["asp"], raw1_pad=st["raw1_pad"])
        cnt = np.isfinite(z).sum(1)
        print(f"  {name}: mean spr {cnt.mean():.2f} hist {np.bincount(cnt, minlength=K + 1).tolist()} "
              f"rays with no cell>=thr: {int((st['raw0'] >= thr).sum(1).__eq__(0).sum())}")
        if keep_x1:
            arrays["x1_nan"] = st["x1_nan"]
    else:
        arrays.update(z=st["z"], raw1=st["raw1"] if keep_x1 else st["raw1"][:4096])
    save(name + ".npz", **arrays)


def stage2_stress():
    """Crafted raw0 rows through the reference sampler itself (nerf_raymarch_common.py:699-757)."""
    rh._install_stubs()
    from nerf_raymarch_common import FromClassifiedDepthAdaptive
    from util.depth_transformations import LogTransform
    g = torch.Generator().manual_seed(7)
    rows = []
    base = torch.rand(128, generator=g)
    rows.append(base.clone())                                   # generic
    rows.append(torch.full((128,), 0.1))                        # all equal, all below -> argmax tie -> cell 0
    rows.append(torch.full((128,), 0.7))                        # all equal, all above -> first K cells
    r = torch.full((128,), -1.0); r[17] = 0.2; rows.append(r)   # exactly == thr (>=)
    r = torch.full((128,), -1.0); r[5] = 0.19999999; rows.append(r)   # just below -> fallback to argmax
    r = torch.zeros(128); r[[3, 9, 40, 41, 42, 100, 127]] = 0.5; rows.append(r)   # ties among survivors
    r = torch.zeros(128); r[::2] = 0.3; r[1::2] = 0.3; r[64] = 0.9; rows.append(r)  # 128 survivors, ties
    r = torch.linspace(-1, 1, 128); rows.append(r)              # ascending values
    r = torch.linspace(1, -1, 128); rows.append(r)              # descending values
    r = torch.full((128,), -5.0); r[127] = -4.0; rows.append(r)  # nothing survives, argmax last cell
    r = torch.full((128,), -5.0); r[0] = 3.0; rows.append(r)    # single survivor, cell 0
    for _ in range(53):                                          # quantised values => many exact ties
        rows.append(torch.round(torch.rand(128, generator=g) * 8) / 8 - 0.3)
    for i in range(40):                                          # generic tie-free rows, various spreads
        rows.append((torch.rand(128, generator=g) - 0.5) * (0.5 + 0.1 * i) + 0.2)
    raw0 = torch.stack(rows).float()
    dr = orc.SCENE_BARBERSHOP["depth_range"]
    arrays = dict(meta=meta(case="stage2_stress", depth_range=dr), raw0=raw0.numpy())
    for K in (1, 4, 8, 16, 128):
        for thr in (0.2, 0.5):
            cfg = rh.make_config(K=K, thr=thr)
            s = FromClassifiedDepthAdaptive(0.001, 1.0, K, z_step=1.0 / 128, noise_amplitude=0.0, config=cfg, net_idx=1)
            z, zp = s.generate(raw0.shape[0], "cpu", depth=raw0.clone(), depth_range=dr, depth_transform=LogTransform)
            arrays[f"z_K{K}_t{thr}"] = z.numpy()
            arrays[f"zp_K{K}_t{thr}"] = zp.numpy()
    save("stage2_stress.npz", **arrays)


FRESH_SEEDS = [(11, 8, 0.2), (12, 4, 0.05), (13, 16, 0.3)]


def state_dict_digest(sd):
    """sha256 over the names and fp32 bytes of a state_dict, in its own order."""
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(np.ascontiguousarray(v.detach().cpu().numpy(), dtype="<f4").tobytes())
    return h.hexdigest()


def fresh_seeds(n_rays=512, n_raw0=64):
    """The reference initialised from fresh seeds (its own initialisers), then run on a ragged-count variant of those
    weights.  Stored per case: the digests of the initial weights, the inputs, and the outputs of one inference call
    (raw0 only for a seeded sample of the rays)."""
    scene = orc.SCENE_BARBERSHOP
    dirs_all = torch.from_numpy(orc.generate_ray_directions(800, 800, scene["fov"]).reshape(-1, 3)).float()
    arrays = dict(meta=meta(case="fresh_seeds", cases=FRESH_SEEDS, scene_params=scene))
    for seed, K, thr in FRESH_SEEDS:
        ref = rh.RefRenderer(scene, K=K, thr=thr, seed=seed)
        sd0 = {k: v.clone() for k, v in ref.models[0].state_dict().items()}
        sd1 = {k: v.clone() for k, v in ref.models[1].state_dict().items()}
        tag = f"s{seed}"
        arrays[tag + "/init_digest"] = np.array([state_dict_digest(sd0), state_dict_digest(sd1)])
        sd0["layers.7.weight"] *= 0.15                  # ragged sample counts
        sd0["layers.7.bias"] = sd0["layers.7.bias"] * 0.15 - 0.2
        ref.load_state_dicts(sd0, sd1)
        g = torch.Generator().manual_seed(seed)
        pix = torch.randperm(dirs_all.shape[0], generator=g)[:n_rays]
        pose = torch.tensor(scene["view_cell_center"]) + 0.1 * torch.randn(3, generator=g)
        rot = orc.rotation_yaw(float(seed * 17))
        st = ref.stages(pose, rot, dirs_all[pix])
        rows = np.sort(np.random.default_rng(seed).choice(n_rays, n_raw0, replace=False))
        arrays.update({tag + "/pix": pix.numpy().astype(np.int32), tag + "/pose": pose.numpy(), tag + "/rot": rot.numpy(),
                       tag + "/raw0_rows": rows.astype(np.int32), tag + "/raw0": st["raw0"][rows], tag + "/asp": st["asp"],
                       tag + "/rgb": st["rgb"], tag + "/weights": st["weights"]})
    save("fresh_seeds.npz", **arrays)


def train_config_fields():
    """The attributes B200Inference.args_from_train_config reads, as an initialised reference TrainConfig carries them."""
    scene = orc.SCENE_PAVILLON
    cases = []
    for K, thr in ((8, 0.2), (16, 0.15)):
        ref = rh.RefRenderer(scene, K=K, thr=thr)
        f1, view = ref.tc.f_in[1], ref.dataset_info.view
        fields = {a: getattr(f1, a) for a in ("depth_range", "max_depth", "z_near", "z_far", "n_ray_samples", "useNDC", "w", "h")
                  if hasattr(f1, a)}
        cases.append(dict(K=K, thr=thr, f_in_1=dict(fields, z_sampler=dict(threshold=f1.z_sampler.threshold)),
                          view={a: getattr(view, a) for a in ("view_cell_center", "view_cell_size", "fov", "focal")},
                          state_dict_keys=[list(m.state_dict()) for m in ref.tc.models]))
    path = os.path.join(OUT, "train_config_fields.json")
    with open(path, "w") as f:
        json.dump(dict(source="reference TrainConfig (FeatureSet.initialize + ModelSelection.getModel, CPU)",
                       torch_version=torch.__version__, cases=cases), f, indent=1)
        f.write("\n")
    print(f"wrote {path}")


def shrink_onnx(src, dst, keep=4):
    """Copies an ONNX model field for field, except that every fp32 initialiser keeps only its leading
    keep x keep block (dims rewritten to match): the exporter's layout at a few kB."""
    buf = memoryview(open(src, "rb").read())

    def copy(fn, wt, v):
        if wt == 0:
            return _field(fn, 0, v)
        if wt == 2:
            return _field(fn, 2, bytes(buf[v[0]:v[1]]))
        return _enc_varint((fn << 3) | wt) + bytes(buf[v[0]:v[1]])     # fixed-width payload, no length

    def tensor(s, e):
        fields = list(_fields(buf, s, e))
        dims = []
        for fn, wt, v in fields:
            if fn == 1 and wt == 0:
                dims.append(v)
            elif fn == 1:
                p = v[0]
                while p < v[1]:
                    d, p = _varint(buf, p)
                    dims.append(d)
        if not any(fn == 2 and v == 1 for fn, _, v in fields):      # not FLOAT: unchanged
            return bytes(buf[s:e])
        raw = next(v for fn, _, v in fields if fn == 9)
        arr = np.frombuffer(buf, dtype="<f4", count=(raw[1] - raw[0]) // 4, offset=raw[0]).reshape(dims)
        small = np.ascontiguousarray(arr[tuple(slice(0, keep) for _ in dims)])
        out, dims_done = b"", False
        for fn, wt, v in fields:
            if fn == 1:
                if not dims_done:
                    out += b"".join(_field(1, 0, d) for d in small.shape)
                    dims_done = True
            elif fn == 9:
                out += _field(9, 2, small.tobytes())
            else:
                out += copy(fn, wt, v)
        return out

    def graph(s, e):
        return b"".join(_field(5, 2, tensor(*v)) if fn == 5 and wt == 2 else copy(fn, wt, v) for fn, wt, v in _fields(buf, s, e))

    model = b"".join(_field(7, 2, graph(*v)) if fn == 7 and wt == 2 else copy(fn, wt, v) for fn, wt, v in _fields(buf, 0, len(buf)))
    with open(dst, "wb") as f:
        f.write(model)
    print(f"wrote {dst}  ({len(model)} bytes, from {len(buf)})")


def shipped_sample():
    """The viewer's shipped export directory: config.ini and dataset_info.txt verbatim, model{0,1}.onnx shrunk."""
    src = os.path.join(rh.REF_ROOT, "adanerf_real_time_viewer", "sample")
    dst = os.path.join(OUT, "viewer_sample")
    os.makedirs(dst, exist_ok=True)
    for name in ("config.ini", "dataset_info.txt"):
        shutil.copyfile(os.path.join(src, name), os.path.join(dst, name))
    for i in range(2):
        shrink_onnx(os.path.join(src, f"model{i}.onnx"), os.path.join(dst, f"model{i}.onnx"))


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    d = os.path.join(rh.REF_ROOT, "adanerf_real_time_viewer", "sample_pavillon_16")
    w0 = read_onnx_initializers(os.path.join(d, "model0.onnx"))
    w1 = read_onnx_initializers(os.path.join(d, "model1.onnx"))
    save("weights_pavillon.npz", meta=meta(source="adanerf_real_time_viewer/sample_pavillon_16/model{0,1}.onnx initialisers"),
         **{"sd0/" + k: v for k, v in w0.items()}, **{"sd1/" + k: v for k, v in w1.items()})
    sd0 = {k: torch.from_numpy(v) for k, v in w0.items()}
    sd1 = {k: torch.from_numpy(v) for k, v in w1.items()}
    pav = orc.SCENE_PAVILLON
    stage_case("pav_k8_t0.2", "pavillon", pav, sd0, sd1, 8, 0.2, 256, 2503, [0.05, -0.03, 0.02], RX, True)
    stage_case("pav_k8_t0.5", "pavillon", pav, sd0, sd1, 8, 0.5, 256, 2503, [0.05, -0.03, 0.02], RX, False)
    stage_case("pav_k16_t0.15", "pavillon", pav, sd0, sd1, 16, 0.15, 256, 2503, [0.0, 0.0, 0.0], orc.rotation_yaw(90.0) @ RX, False)
    s0, s1 = orc.make_weights("shaped", seed=0)
    bar = orc.SCENE_BARBERSHOP
    stage_case("shaped_k8_t0.2", "barbershop", bar, s0, s1, 8, 0.2, 256, 2503, [0.0, 0.0, 0.0], torch.eye(3), True)
    r0, r1 = orc.make_weights("rand", seed=0)
    stage_case("rand_k8_t0.2", "barbershop", bar, r0, r1, 8, 0.2, 256, 2503, [0.0, 0.0, 0.0], torch.eye(3), False)
    # BASELINE config 1: first 1024 rays of the 800x800 grid, dense 128 samples/ray, random init
    stage_case("rand_dense_k128", "barbershop", bar, r0, r1, 128, 0.0, 1024, 1, [0.0, 0.0, 0.0], torch.eye(3), False)
    # NDC / LLFF variant (configs/fine_training_ndc.ini): 30-feature sampling net, NoDepthRange sampler, ndc_rays
    n0, n1 = orc.make_weights("ndc", seed=0)
    stage_case("ndc_k16_t0.15", "pavillon_ndc", orc.SCENE_PAVILLON_NDC, n0, n1, 16, 0.15, 256, 2501, [0.1, -0.05, 0.02],
               orc.rotation_yaw(20.0), True, ndc=True)
    stage2_stress()
    fresh_seeds()
    train_config_fields()
    shipped_sample()


if __name__ == "__main__":
    if len(sys.argv) > 1:               # e.g. `python oracle/gen_golden.py fresh_seeds`: only the named fixtures
        torch.set_num_threads(8)
        for name in sys.argv[1:]:
            globals()[name]()
    else:
        main()
