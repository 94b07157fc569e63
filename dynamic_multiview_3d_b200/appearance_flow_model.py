"""Model-level drop-in surface: the single-view appearance-flow models.

Mirrors dyn_mult_view/multi_view_model/appearance_flow_model.py:17-130 (AppearanceFlowModel),
highdim_angle.py:5-10, lowdim_angle.py:5-8 and appearance_flow_tinghui.py:5-49: same class
names, constructor ``(conf, load_tfrec=True, build_loss=True)``, same ``conf`` keys, same
variable names, same layer sequence (via the reference-named ops in tf_utils.py), same
attributes for the last step's tensors (image0, image1, disp, flow_field, warp_pts, gen, loss).

There is no TF session here, so where the reference builds a graph once and ``sess.run``s it,
these classes expose ``forward(image0, disp)``, ``train_step(image0, image1, disp)`` and a
CUDA-graph-captured ``GraphedTrainStep`` (train.py).  The reference is hard-wired to 128x128
(appearance_flow_model.py:26,53-56); here every 128-derived constant follows the shape rule
of SURVEY.md 8(a) (side H multiple of 32, bottleneck H/32), so conf['image_size']=128
reproduces the reference shapes and 224 gives BASELINE's.

Extra conf keys (all optional): image_size (128), viewpoint_dim (2), loss ('l2' = reference,
'l1' = north-star), grid_order ('ref_yx' = the reference's transposing (Y,X) grid, 'xy'),
algo ('auto'|'simt'|'tcgen05'), seed (0), num_targets (1), num_views (1).

Several targets per source: a batch with disp [B, T, viewpoint_dim] and image1 [B, T, H, H, 3] trains B sources x T
targets.  The encoder runs once per source, fc1 / e_fc1 hands each source's features to its T targets
(functional.linear(group=T)), the decoder runs at B*T rows and the warp reads each source in place.  The loss is the
mean over all B*T target images.  conf['num_targets'] only shapes input_spec(); batch_size is the number of sources.

Several source views per target (conf['num_views'] = Vw > 1, Zhou et al.'s multi-view appearance flow, the batch layout
of MultiViewFusionAppFlow): image0 [Vw, B, H, H, 3], disp [Vw, B, viewpoint_dim] (source v's viewpoint change to the
target), image1 [B, H, H, 3].  Every view runs the same network (encoder and decoder at Vw*B rows); the flow head has a
third channel, a per-pixel confidence logit, and the prediction is  sum_v softmax_v(logit) * warp(src_v, flow_v).  The
warps, the fusion, the loss and the head gradient are one kernel (functional.fused_views_warp_loss).  gen is the fused
[B, H, H, 3]; flow_field [Vw, B, H, H, 2] and confidence [Vw, B, H, H] are views of the head.
"""
import os

import torch

from . import functional as F
from .model_base import ModelBase
from .optimizer import TFAdam
from .tf_utils import conv2d_msra, coords, deconv2d_msra, flow_resample_layer, linear_msra, warp_pts_layer
from .variables import VariableStore, use_store

MAX_VIEWS = 8          # dmv_sampler_fuse_views_loss fuses up to 8 source views


class AppearanceFlowModel(ModelBase):
    ACT = "lrelu"
    INPUT_KEYS = ("image0", "image1", "disp")

    def __init__(self, conf, load_tfrec=True, build_loss=True, device=None):
        self.conf = conf
        self.batch_size = int(conf["batch_size"])
        H = int(conf.get("image_size", 128))
        if H % 32:
            raise ValueError("image_size must be a multiple of 32")
        self.image_shape = [H, H, 3]
        self.viewpoint_dim = int(conf.get("viewpoint_dim", 2))
        self.num_targets = int(conf.get("num_targets", 1))
        if self.num_targets < 1:
            raise ValueError("num_targets must be >= 1")
        self.num_views = int(conf.get("num_views", 1))
        if not 1 <= self.num_views <= MAX_VIEWS:
            raise ValueError("%s: num_views must be 1 .. %d (the fused multi-view kernel's limit), got %d"
                             % (type(self).__name__, MAX_VIEWS, self.num_views))
        if self.num_views > 1 and self.num_targets > 1:
            raise ValueError("%s trains several source views of one target (num_views = %d) or several targets of one source "
                             "(num_targets = %d), not both" % (type(self).__name__, self.num_views, self.num_targets))
        self.head_channels = 3 if self.num_views > 1 else 2      # flow, plus the confidence logit with several views
        self.confidence = None
        self.loss_mode = conf.get("loss", "l2")
        self.grid_order = conf.get("grid_order", "ref_yx")
        self.algo = conf.get("algo", None)
        self.max_iter = 1000000
        self.start_iter = 0
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.store = VariableStore(self.device, seed=int(conf.get("seed", 0)))
        self.build_loss_flag = build_loss
        self.world_size = 1          # data_parallel.attach() raises this; the loss mean is global
        self.image0 = self.image1 = self.disp = None
        self.flow_field = self.gen = self.loss = None
        self.optimizer = None
        # "graph build": one forward on zeros creates every variable in reference order
        z_img, z_disp = self._zeros_for_build()
        if self.device.type == "meta":
            with torch.no_grad(), F.meta_mode():
                self.forward(z_img, z_disp)
        else:
            with torch.no_grad():
                self.forward(z_img, z_disp)
        self.store.finalize(trainable=self._trainable)
        self.t_vars = self.store.trainable_vars()
        if build_loss and self.device.type != "meta":
            self.optimizer = TFAdam(self.store, conf["learning_rate"])

    def _zeros_for_build(self):
        lead = [self.batch_size] if self.num_views == 1 else [self.num_views, self.batch_size]
        return (torch.zeros(lead + self.image_shape, dtype=torch.float32, device=self.device),
                torch.zeros(lead + [self.viewpoint_dim], dtype=torch.float32, device=self.device))

    def input_spec(self):
        B = self.batch_size
        if self.num_views > 1:
            Vw = self.num_views
            return {"image0": (Vw, B) + tuple(self.image_shape), "image1": (B,) + tuple(self.image_shape), "disp": (Vw, B, self.viewpoint_dim)}
        T = () if self.num_targets == 1 else (self.num_targets,)
        return {"image0": tuple([B] + self.image_shape), "image1": tuple([B] + list(T) + self.image_shape),
                "disp": (B,) + T + (self.viewpoint_dim,)}

    # dead variables of the high-dim viewpoint encoder receive no gradient (TF skips None grads)
    def _trainable(self, name):
        return True

    # -- graph ------------------------------------------------------------------------------
    def decodeAngle(self, disp):
        """appearance_flow_model.py:63-66"""
        a0 = linear_msra(disp, 64, "a0", act="lrelu", algo=self.algo)
        a1 = linear_msra(a0, 64, "a1", act="lrelu", algo=self.algo)
        return linear_msra(a1, 64, "a2", act="lrelu", algo=self.algo)

    def _viewpoint_fork(self, disp):
        """decodeAngle on a branch stream, started BEFORE the image encoder is enqueued (it is independent of it until the
        concat): returns a callable that joins the branch and yields the viewpoint code (functional.branch)."""
        if os.environ.get("DMV_VIEW_BRANCH", "1") != "1" or disp.device.type != "cuda":
            return lambda: self.decodeAngle(disp)
        with F.branch(disp.device, disp) as br:
            code = self.decodeAngle(disp)
        return lambda: br.join(code)

    def buildModel(self, image0, disp, group=1):
        """appearance_flow_model.py:83-127 with the shape rule; activations fused into the layers.  The viewpoint branch
        is forked before the encoder is enqueued.  group > 1: disp holds ``group`` consecutive viewpoints per source."""
        viewpoint_code = self._viewpoint_fork(disp)
        return self._decode(self.encode(image0, group), viewpoint_code)

    def encode(self, image0, group=1):
        """The image side: e0 .. e4_0 and fc1 -> features [B * group, 4096] bf16 (each source's row repeated ``group``
        times)."""
        B, H = image0.shape[0], image0.shape[1]
        h5 = H // 32
        a, g = self.ACT, self.algo
        e0 = conv2d_msra(image0, 32, 5, 5, 2, 2, "e0", act=a, algo=g)
        e0_0 = conv2d_msra(e0, 32, 5, 5, 1, 1, "e0_0", act=a, algo=g)
        e1 = conv2d_msra(e0_0, 32, 5, 5, 2, 2, "e1", act=a, algo=g)
        e1_0 = conv2d_msra(e1, 32, 5, 5, 1, 1, "e1_0", act=a, algo=g)
        e2 = conv2d_msra(e1_0, 64, 5, 5, 2, 2, "e2", act=a, algo=g)
        e2_0 = conv2d_msra(e2, 64, 5, 5, 1, 1, "e2_0", act=a, algo=g)
        e3 = conv2d_msra(e2_0, 128, 3, 3, 2, 2, "e3", act=a, algo=g)
        e3_0 = conv2d_msra(e3, 128, 3, 3, 1, 1, "e3_0", act=a, algo=g)
        e4 = conv2d_msra(e3_0, 256, 3, 3, 2, 2, "e4", act=a, algo=g)
        e4_0 = conv2d_msra(e4, 256, 3, 3, 1, 1, "e4_0", act=a, algo=g)
        e4r = F.reshape(e4_0, (B, h5 * h5 * 256))                       # NHWC flatten, (h, w, c) order
        return linear_msra(e4r, 4096, "fc1", act=a, algo=g, group=group)

    def decode(self, features, viewpoint):
        """features [N, 4096] (encode), viewpoint [N, viewpoint_dim] bf16 -> flow field [N, H, H, 2] fp32: the viewpoint
        code, the joint FCs, the decoder and the flow head."""
        return self._decode(features, self._viewpoint_fork(viewpoint))

    def _decode(self, e5, viewpoint_code):
        B, H = e5.shape[0], self.image_shape[0]
        h5 = H // 32
        a, g = self.ACT, self.algo
        concated = torch.cat([e5, viewpoint_code()], dim=1)

        a3 = linear_msra(concated, 4096, "a3", act=a, algo=g)
        a4 = linear_msra(a3, 4096, "a4", act=a, algo=g)
        a5 = linear_msra(a4, h5 * h5 * 256, "a5", act=a, algo=g)
        a5r = F.reshape(a5, (B, h5, h5, 256))

        d4 = deconv2d_msra(a5r, [B, 2 * h5, 2 * h5, 128], 3, 3, 2, 2, "d4", act=a, algo=g)
        d4_0 = conv2d_msra(d4, 128, 3, 3, 1, 1, "d4_0", act=a, algo=g)
        d3 = deconv2d_msra(d4_0, [B, 4 * h5, 4 * h5, 64], 3, 3, 2, 2, "d3", act=a, algo=g)
        d3_0 = conv2d_msra(d3, 64, 5, 5, 1, 1, "d3_0", act=a, algo=g)
        d2 = deconv2d_msra(d3_0, [B, 8 * h5, 8 * h5, 32], 5, 5, 2, 2, "d2", act=a, algo=g)
        d2_0 = conv2d_msra(d2, 64, 5, 5, 1, 1, "d2_0", act=a, algo=g)
        d1 = deconv2d_msra(d2_0, [B, 16 * h5, 16 * h5, 32], 5, 5, 2, 2, "d1", act=a, algo=g)
        d1_0 = conv2d_msra(d1, 32, 5, 5, 1, 1, "d1_0", act=a, algo=g)
        self._last_decoder = d1_0            # subclasses hang further heads here (multi-view confidence)
        # flow head: no activation (appearance_flow_model.py:125); fp32 out for the sampler
        return deconv2d_msra(d1_0, [B, H, H, self.head_channels], 5, 5, 2, 2, "flow_field", act=None, algo=g, out_dtype=torch.float32)

    def forward(self, image0, disp, keep=None):
        """image0 [B,H,H,3] fp32 in [0,1], disp [B,V] fp32 -> dict(flow_field, gen); sets the
        reference's attribute names.  warp_pts is formed inside the sampler; read
        ``self.warp_pts`` to materialise it.  disp [B,T,V]: T targets per source, outputs [B,T,...]."""
        # drop the previous step's tape before building the next one (see VariableStore.new_anchor)
        self.flow_field = self.gen = self.loss = None
        self.store.new_anchor()
        self.image0, self.disp = image0, disp
        if self.num_views > 1:
            with use_store(self.store):
                head = self._views_head(image0, disp)
            self._set_views(head, F.fused_views_warp(_flat_views(image0), head, self.num_views, self.grid_order))
            return {"flow_field": self.flow_field, "gen": self.gen}
        if disp.dim() == 3:
            with use_store(self.store):
                flow, T = self._grouped_flow(image0, disp)
                gen = F.flow_resampler_grouped(image0, flow, T, self.grid_order)
            self.flow_field, self.gen = _per_source(flow, T), _per_source(gen, T)
            return {"flow_field": self.flow_field, "gen": self.gen}
        with use_store(self.store):
            self.flow_field = self.buildModel(image0, F.to_bf16(disp))
            self.gen = flow_resample_layer(image0, self.flow_field, self.grid_order)
        return {"flow_field": self.flow_field, "gen": self.gen}

    def _grouped_flow(self, image0, disp):
        """disp [B, T, V] -> (flow [B*T, H, H, 2], T): each source encoded once, decoded at its T viewpoints."""
        B, T = int(disp.shape[0]), int(disp.shape[1])
        if image0.shape[0] != B:
            raise ValueError("image0 holds %d sources, disp %d" % (image0.shape[0], B))
        return self.buildModel(image0, F.to_bf16(disp.reshape(B * T, disp.shape[2])), T), T

    def _views_head(self, image0, disp):
        """image0 [Vw,B,H,H,3], disp [Vw,B,V] -> the 3-channel head [Vw*B,H,H,3]: every view through the network."""
        Vw, B = self.num_views, int(image0.shape[1]) if image0.dim() == 5 else -1
        if image0.dim() != 5 or disp.dim() != 3 or tuple(image0.shape[:2]) != (Vw, B) or tuple(disp.shape[:2]) != (Vw, B):
            raise ValueError("%s with num_views = %d takes image0 [%d, B, H, H, 3] and disp [%d, B, V], got %s and %s"
                             % (type(self).__name__, Vw, Vw, Vw, tuple(image0.shape), tuple(disp.shape)))
        return self.buildModel(_flat_views(image0), F.to_bf16(disp.reshape(Vw * B, disp.shape[2])))

    def _set_views(self, head, fused):
        Vw = self.num_views
        lead = (Vw, head.shape[0] // Vw) + tuple(head.shape[1:3])
        self.flow_field = head[..., :2].reshape(lead + (2,))
        self.confidence = head[..., 2].reshape(lead)
        self.gen = fused

    @property
    def warp_pts(self):
        """warp_pts_layer(flow_field) (appearance_flow_model.py:126), materialised on demand."""
        f = self.flow_field.detach()
        f = f.reshape((-1,) + tuple(f.shape[-3:]))
        if self.grid_order == "ref_yx":
            return warp_pts_layer(f)
        return f + coords(f.shape[1], f.shape[2], f.shape[0], f.device).flip(-1)

    def build_loss(self, image1):
        """appearance_flow_model.py:68-73: euclidean_loss(gen, image1) (conf['loss']='l1' for L1).
        The mean runs over the GLOBAL batch under data parallelism."""
        self.image1 = image1
        n = image1.numel() // image1.shape[-1] * self.world_size       # every target pixel: B*H*W (B*T*H*W with T targets)
        self.loss = F.reconstruction_loss(self.gen, image1, self.loss_mode, inv_count=1.0 / n, unit_upstream=True)
        return self.loss

    def forward_and_loss(self, image0, image1, disp):
        """forward + build_loss with the warp, the loss and the flow gradient fused into one kernel (the training
        path).  Falls back to the separate calls for shapes the fused kernel does not cover."""
        if type(self).forward is not AppearanceFlowModel.forward or type(self).build_loss is not AppearanceFlowModel.build_loss \
                or self.device.type == "meta":
            self.forward(image0, disp)
            return self.build_loss(image1)
        if self.num_views > 1:
            return self._views_forward_and_loss(image0, image1, disp)
        if disp.dim() == 3:
            return self._grouped_forward_and_loss(image0, image1, disp)
        self.flow_field = self.gen = self.loss = None
        self.store.new_anchor()
        self.image0, self.disp, self.image1 = image0, disp, image1
        with use_store(self.store):
            self.flow_field = self.buildModel(image0, F.to_bf16(disp))
        if not F.warp_loss_supported(image0, self.flow_field, image1) or os.environ.get("DMV_NO_WARP_LOSS"):
            with use_store(self.store):
                self.gen = flow_resample_layer(image0, self.flow_field, self.grid_order)
            return self.build_loss(image1)
        n = image1.shape[0] * image1.shape[1] * image1.shape[2] * self.world_size
        self.loss, self.gen = F.flow_resample_loss(image0, self.flow_field, image1, self.loss_mode, inv_count=1.0 / n,
                                                   grid_order=self.grid_order, unit_upstream=True)
        return self.loss

    def _grouped_forward_and_loss(self, image0, image1, disp):
        """forward_and_loss with T targets per source (image1 [B,T,H,H,3], disp [B,T,V]): the warp of each source by its T
        flows, the loss over all B*T targets and the flow gradient in one kernel (dmv_sampler_loss_fused_shared_src)."""
        self.flow_field = self.gen = self.loss = None
        self.store.new_anchor()
        self.image0, self.disp, self.image1 = image0, disp, image1
        with use_store(self.store):
            flow, T = self._grouped_flow(image0, disp)
        target = image1.reshape((flow.shape[0],) + tuple(image1.shape[2:]))
        if not F.warp_loss_supported(image0, flow, target) or os.environ.get("DMV_NO_WARP_LOSS"):
            self.flow_field = _per_source(flow, T)
            self.gen = _per_source(F.flow_resampler_grouped(image0, flow, T, self.grid_order), T)
            return self.build_loss(image1)
        n = target.numel() // target.shape[-1] * self.world_size
        self.loss, gen = F.flow_resample_loss(image0, flow, target, self.loss_mode, inv_count=1.0 / n, grid_order=self.grid_order,
                                              unit_upstream=True, group=T)
        self.flow_field, self.gen = _per_source(flow, T), _per_source(gen, T)
        return self.loss

    def _views_forward_and_loss(self, image0, image1, disp):
        """forward_and_loss with Vw source views per target: every view's warp, the confidence fusion, the loss and the
        gradient wrt the 3-channel head in one kernel (dmv_sampler_fuse_views_loss); under no_grad the loss alone."""
        self.flow_field = self.gen = self.loss = self.confidence = None
        self.store.new_anchor()
        self.image0, self.disp, self.image1 = image0, disp, image1
        with use_store(self.store):
            head = self._views_head(image0, disp)
        n = image1.shape[0] * image1.shape[1] * image1.shape[2] * self.world_size
        self.loss, fused = F.fused_views_warp_loss(_flat_views(image0), head, image1, self.num_views, self.loss_mode, inv_count=1.0 / n,
                                                   grid_order=self.grid_order, unit_upstream=True)
        self._set_views(head, fused)
        return self.loss

    def step_loss(self, batch):
        return self.forward_and_loss(batch["image0"], batch["image1"], batch["disp"])

    def render_sources(self):
        if self.num_views > 1:
            raise NotImplementedError(
                "%s with num_views = %d has no render(): each view it predicts fuses the warps of %d source views by predicted "
                "confidences, and rendering decodes one source per sample" % (type(self).__name__, self.num_views, self.num_views))
        return ("image0",)

    def _render_encode(self, sources):
        return self.encode(sources["image0"])

    def _render_decode(self, sources, features, viewpoint, group):
        flow = self.decode(features, viewpoint)
        return {"gen": F.flow_resampler_shared(sources["image0"], flow, group, self.grid_order), "flow": flow}

    def visualize(self, image0, image1, disp, iter_num=None):
        """appearance_flow_model.py:132-179: output / ground-truth / input grids, the flow image and the
        correspondence probes (visualize.py).  The TF session argument becomes the batch itself."""
        from .visualize import visualize
        if self.num_views > 1:               # several source views: source frame 0, the fused prediction, the target
            return visualize(self, image0, image1, disp, iter_num, source=image0[0])
        if disp.dim() == 3:                  # several targets per source: each source's first
            image1, disp = image1[:, 0], disp[:, 0]
        return visualize(self, image0, image1, disp, iter_num)


def _flat_views(x):
    """[Vw, B, ...] -> [Vw*B, ...] (view-major rows, no copy)"""
    return x.reshape((x.shape[0] * x.shape[1],) + tuple(x.shape[2:]))


def _per_source(x, T):
    """[B*T, ...] -> [B, T, ...]"""
    return x.reshape((x.shape[0] // T, T) + tuple(x.shape[1:]))


class AppFlowHighDimAngle(AppearanceFlowModel):
    """highdim_angle.py:5-10.  a0 (V->19) and a1 (V->128) are created but unused."""

    def decodeAngle(self, disp):
        store = self.store
        V = int(disp.shape[-1])
        import math
        with store.scope("a0"):        # dead variables: created for checkpoint compatibility only
            store.get("Matrix", [V, 19], "normal", math.sqrt(2.0 / V)); store.get("b", [19], "zeros")
        with store.scope("a1"):
            store.get("Matrix", [V, 128], "normal", math.sqrt(2.0 / V)); store.get("b", [128], "zeros")
        return linear_msra(disp, 256, "a2", act="lrelu", algo=self.algo)

    def _trainable(self, name):
        return not (name.startswith("a0/") or name.startswith("a1/"))


class AppFlowLowDimAngle(AppearanceFlowModel):
    """lowdim_angle.py:5-8."""

    def decodeAngle(self, disp):
        return linear_msra(disp, 10, "a0", act="lrelu", algo=self.algo)


class AppearanceFlowTinghui(AppearanceFlowModel):
    """appearance_flow_tinghui.py:5-49 (Zhou et al.-style lighter net, relu trunk)."""

    def buildModel(self, image0, disp, group=1):
        viewpoint_code = self._viewpoint_fork(disp)
        return self._decode(self.encode(image0, group), viewpoint_code)

    def encode(self, image0, group=1):
        """e0 .. e4, e_fc0, e_fc1 -> features [B * group, 2048] bf16 (each source's row repeated ``group`` times)."""
        B, H = image0.shape[0], image0.shape[1]
        g = self.algo
        e = image0
        for name, c in [("e0", 16), ("e1", 32), ("e2", 64), ("e3", 128), ("e4", 256)]:
            e = conv2d_msra(e, c, 3, 3, 2, 2, name, act="relu", algo=g)
        e4r = F.reshape(e, (B, (H // 32) ** 2 * 256))
        e_fc0 = linear_msra(e4r, 2048, "e_fc0", act="relu", algo=g)
        return linear_msra(e_fc0, 2048, "e_fc1", act="relu", algo=g, group=group)

    def _decode(self, e_fc1, viewpoint_code):
        B, H = e_fc1.shape[0], self.image_shape[0]
        g = self.algo
        concated = torch.cat([e_fc1, viewpoint_code()], dim=1)
        d_fc0 = linear_msra(concated, 2048, "a3", act="relu", algo=g)
        d_fc1 = linear_msra(d_fc0, (H // 16) ** 2 * 32, "a4", act="relu", algo=g)
        d = F.reshape(d_fc1, (B, H // 16, H // 16, 32))
        d = deconv2d_msra(d, [B, H // 8, H // 8, 128], 3, 3, 2, 2, "d3", act="relu", algo=g)
        d = deconv2d_msra(d, [B, H // 4, H // 4, 64], 3, 3, 2, 2, "d2", act="relu", algo=g)
        d = deconv2d_msra(d, [B, H // 2, H // 2, 32], 3, 3, 2, 2, "d1", act="relu", algo=g)
        d = deconv2d_msra(d, [B, H, H, 16], 3, 3, 2, 2, "d0", act="relu", algo=g)
        return deconv2d_msra(d, [B, H, H, self.head_channels], 3, 3, 1, 1, "flow_field", act=None, algo=g, out_dtype=torch.float32)
