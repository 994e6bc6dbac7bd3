"""Drop-in for `TrainConfig.inference` (thomasneff/AdaNeRF src/train_data.py:278-299).

`B200Inference.inference(batch, gradient=False, is_inference=True)` has the reference's signature and return
shape -- `(postprocessed_outs, inference_dicts)` -- so `src/evaluate.py:216-235`, `src/plots.py:51-52,237,353`
and `src/export.py:64` can call it unchanged (INTEGRATION.md shows the two-line patch that installs it on an
existing TrainConfig).  Only the entries those callers read are produced:

    outs[-1][:, :3]                          rgb                                (evaluate.py:228)
    dicts[-1]["AdaptiveSamplePositions"]     samples per ray / K                 (evaluate.py:223-224)
    dicts[1]["OracleWeights"]                raw sampling-net output, thr == 0   (evaluate.py:279-280)
    dicts[i]["PostProcessedNetworkOutput"]   = outs[i]                           (util/helper.py:79-130)

The batch keys are the reference's DatasetKeyConstants (src/datasets.py:24-38)."""
import torch

from .renderer import Renderer

# src/datasets.py:29-35 and src/features.py:20-40
KEY_POSE, KEY_ROT, KEY_DIRS = "ImagePose", "ImageRotation", "RayDirectionsSamples"
KEY_POST, KEY_NET_OUT = "PostProcessedNetworkOutput", "NetworkOutputBatch"
KEY_ASP, KEY_ORACLE = "AdaptiveSamplePositions", "OracleWeights"
# FeatureSetKeyConstants (src/features.py:20-40) of the auxiliary tensors RayMarchFromPoses.postprocess stores
KEY_WEIGHTS, KEY_ALPHA, KEY_ZVALS, KEY_DEPTH = "NeRFWeightsOutput", "NeRFAlphaOutput", "NeRFInputFeatureZVals", "NeRFOutputDepth"


class B200Inference:
    """scene: dict (view_cell_center, view_cell_size, depth_range [warped], max_depth, fov) -- the fields
    FeatureSet.initialize reads from DatasetInfo (src/features.py:343-360, :747-767)."""

    def __init__(self, scene, sampling_net, shading_net, threshold, num_samples, device=0, want_oracle_weights=None,
                 want_aux=False):
        self.renderer = Renderer(scene, device=device, sampling_net=sampling_net, shading_net=shading_net)
        self.threshold = float(threshold)
        self.K = int(num_samples)
        self.want_oracle_weights = (self.threshold == 0.0) if want_oracle_weights is None else bool(want_oracle_weights)
        # plots.render_all_imgs / the depth export read NeRFWeightsOutput, NeRFAlphaOutput, NeRFOutputDepth (src/plots.py:272-306)
        self.want_aux = bool(want_aux)

    @staticmethod
    def args_from_train_config(train_config):
        """(scene, [sampling_net, shading_net], threshold, K) read from an initialised reference TrainConfig -- no device
        needed (tests/test_adapter_config.py runs this on the fields of a reference TrainConfig)."""
        f1 = train_config.f_in[1]
        info = train_config.dataset_info
        scene = dict(view_cell_center=list(info.view.view_cell_center), view_cell_size=list(info.view.view_cell_size),
                     depth_range=list(f1.depth_range), max_depth=float(f1.max_depth), fov=float(info.view.fov),
                     z_near=f1.z_near, z_far=f1.z_far)
        if getattr(f1, "useNDC", False):    # configs/*_ndc.ini: ndc_rays(self.h, self.w, self.view.focal, 1., ...) (features.py:430)
            scene.update(use_ndc=True, w=int(f1.w), h=int(f1.h), focal=float(info.view.focal))
        return scene, [train_config.models[0], train_config.models[1]], float(f1.z_sampler.threshold), int(f1.n_ray_samples)

    @classmethod
    def from_train_config(cls, train_config, device=0):
        """Builds the renderer from an initialised reference TrainConfig (models, feature sets, dataset_info)."""
        scene, models, thr, k = cls.args_from_train_config(train_config)
        return cls(scene, models[0], models[1], thr, k, device=device)

    def inference(self, batch_idx, gradient=False, **kwargs):
        if gradient:
            raise NotImplementedError("adanerf_b200 is an inference renderer (src/train.py is out of scope)")
        b = batch_idx.get_batch_input(1) if hasattr(batch_idx, "get_batch_input") else batch_idx
        pose, rot, dirs = b[KEY_POSE], b[KEY_ROT], b[KEY_DIRS]
        if pose.shape[0] != 1:
            raise ValueError("one image per inference call (evaluate.py / plots.py batch a single image)")
        out = self.renderer.render_rays(pose[0], rot[0], dirs.reshape(-1, 3), self.threshold, self.K,
                                        want_nsamples=True, want_oracle_weights=self.want_oracle_weights,
                                        want_aux=("weights", "alpha", "z_vals", "depth_est") if self.want_aux else False)
        rgb = out["rgb"]
        raw0 = out["oracle_weights"]
        d0 = {KEY_POST: raw0, KEY_NET_OUT: raw0}
        d1 = {KEY_POST: rgb}
        if self.threshold > 0.0:
            d1[KEY_ASP] = out["n_samples"].to(torch.float32) / self.K
        if raw0 is not None:
            d1[KEY_ORACLE] = raw0
        if self.want_aux:
            d1[KEY_WEIGHTS], d1[KEY_ALPHA], d1[KEY_ZVALS] = out["weights"], out["alpha"], out["z_vals"]
            d1[KEY_DEPTH] = out["depth_est"].reshape(-1, 1)   # features.py:576-577
        return [raw0, rgb], [d0, d1]

    __call__ = inference
