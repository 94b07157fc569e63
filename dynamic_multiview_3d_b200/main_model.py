"""Model-level drop-in surface: the colour / depth / colour+depth prediction model.

Mirrors dyn_mult_view/multi_view_model/main_model.py:12-154 (``Base_Prediction_Model``; BASELINE config 4,
conf ``tensorflowdata/cars_colordepth/conf.py``): one 5-conv pre-encoder per input modality
(``image_preprocessing`` :57-65, scopes ``pre_image0`` / ``pre_dimage0``), channel concat, shared trunk
(:105-121), ``d3_0`` widened to ``64 * num_decode`` and split (:123-137, ``split_list.pop()`` hands the
LAST group to the colour head), one decoder per output (``decode`` :68-81) with a tanh head, and
loss = L(colour) + depth_lr_factor * L(depth) (:144-154).

Feature switches are key-presence tests on ``conf`` as in the reference (``'use_color' in conf``).
Extensions (optional conf keys): image_size (128), viewpoint_dim (2), loss ('l2' reference | 'l1' per-channel L1,
tf_utils.py:22 | 'ssim' SSIM + L1 with weight ssim_alpha (0.85) on SSIM, functional.ssim_l1_loss), head ('tanh' reference |
'flow': each head emits a 2-channel flow and the output is the bilinear
warp of its source modality -- the north-star's "warped RGB/depth"; precedent: multiobject_appflow.py:191-209),
grid_order, algo, seed, num_targets (1).  The reference ignores conf['batch_size'] (main_model.py:19 hard-codes 64); here
conf wins.  Several targets per source (disp [B, T, V], image1 / depth1 [B, T, H, H, C]) train as the appearance-flow
models do (appearance_flow_model.py): one encoding per source, B*T decoded targets, the loss over all of them.
"""
import torch

from . import functional as F
from .model_base import ModelBase
from .optimizer import TFAdam
from .tf_utils import conv2d_msra, deconv2d_msra, flow_resample_layer, linear_msra
from .variables import VariableStore, use_store


class Base_Prediction_Model(ModelBase):
    INPUT_KEYS = ("image0", "depth0", "image1", "depth1", "disp")      # train_step(image0, dimage0, image1, dimage1, disp)

    def __init__(self, conf, load_tfrec=True, build_loss=True, device=None):
        self.conf = conf
        self.batch_size = int(conf.get("batch_size", 64))
        H = int(conf.get("image_size", 128))
        if H % 32:
            raise ValueError("image_size must be a multiple of 32")
        self.image_shape = [H, H, 3]
        self.viewpoint_dim = int(conf.get("viewpoint_dim", 2))
        self.loss_mode = conf.get("loss", "l2")
        self.ssim_alpha = float(conf.get("ssim_alpha", 0.85))
        self.head = conf.get("head", "tanh")
        self.num_targets = int(conf.get("num_targets", 1))
        if self.num_targets < 1:
            raise ValueError("num_targets must be >= 1")
        if int(conf.get("num_views", 1)) > 1:
            raise ValueError("%s takes one source view per target (num_views = %s): its colour and depth heads have "
                             "no confidence channel to fuse several views by" % (type(self).__name__, conf["num_views"]))
        self.grid_order = conf.get("grid_order", "ref_yx")
        self.algo = conf.get("algo", None)
        self.use_color = "use_color" in conf
        self.use_depth = "use_depth" in conf
        if not (self.use_color or self.use_depth):
            raise ValueError("conf needs 'use_color' and/or 'use_depth'")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.store = VariableStore(self.device, seed=int(conf.get("seed", 0)))
        self.world_size = 1
        self.gen_image1 = self.gen_dimage1 = self.loss = None
        self.optimizer = None
        B = self.batch_size
        z = lambda c: torch.zeros((B, H, H, c), dtype=torch.float32, device=self.device)
        zd = torch.zeros((B, self.viewpoint_dim), dtype=torch.float32, device=self.device)
        if self.device.type == "meta":
            with torch.no_grad(), F.meta_mode():
                self.forward(z(3), z(1), zd)
        else:
            with torch.no_grad():
                self.forward(z(3), z(1), zd)
        self.store.finalize()
        self.t_vars = self.store.trainable_vars()
        if build_loss and self.device.type != "meta":
            self.optimizer = TFAdam(self.store, conf["learning_rate"])

    # -- graph ---------------------------------------------------------------------------------
    def image_preprocessing(self, x, scope):
        """main_model.py:57-65"""
        g = self.algo
        with self.store.scope(scope):
            e0 = conv2d_msra(x, 32, 5, 5, 2, 2, "e0", act="lrelu", algo=g)
            e0_0 = conv2d_msra(e0, 32, 5, 5, 1, 1, "e0_0", act="lrelu", algo=g)
            e1 = conv2d_msra(e0_0, 32, 5, 5, 2, 2, "e1", act="lrelu", algo=g)
            e1_0 = conv2d_msra(e1, 32, 5, 5, 1, 1, "e1_0", act="lrelu", algo=g)
            return conv2d_msra(e1_0, 64, 5, 5, 2, 2, "e2", act="lrelu", algo=g)

    def decode_output(self, x, scope, num_channels, warp=None):
        """main_model.py:68-81 (``decode``: tanh head) or, with head='flow', a 2-channel flow head and ``warp(flow)``, the
        warp of the output's source modality."""
        g = self.algo
        B, H = x.shape[0], self.image_shape[0]
        h5 = H // 32
        with self.store.scope(scope):
            d2 = deconv2d_msra(x, [B, 8 * h5, 8 * h5, 32], 5, 5, 2, 2, "d2", act="lrelu", algo=g)
            d2_0 = conv2d_msra(d2, 64, 5, 5, 1, 1, "d2_0", act="lrelu", algo=g)
            d1 = deconv2d_msra(d2_0, [B, 16 * h5, 16 * h5, 32], 5, 5, 2, 2, "d1", act="lrelu", algo=g)
            d1_0 = conv2d_msra(d1, 32, 5, 5, 1, 1, "d1_0", act="lrelu", algo=g)
            if self.head == "flow":
                flow = deconv2d_msra(d1_0, [B, H, H, 2], 5, 5, 2, 2, "d0", act=None, algo=g, out_dtype=torch.float32)
                return warp(flow), flow
            gen = deconv2d_msra(d1_0, [B, H, H, num_channels], 5, 5, 2, 2, "d0", act="tanh", algo=g, out_dtype=torch.float32)
            return gen, None

    def buildModel(self, image0, dimage0, disp, group=1):
        """main_model.py:83-142.  group > 1: disp holds ``group`` consecutive viewpoints per source."""
        srcs = {"image0": image0, "depth0": dimage0}
        if group == 1:
            warp = lambda key, flow: flow_resample_layer(srcs[key], flow, self.grid_order)
        else:
            warp = lambda key, flow: F.flow_resampler_grouped(srcs[key], flow, group, self.grid_order)
        out = self.decode(self.encode(image0, dimage0, group), disp, warp)
        self.gen_image1, self.flow_image1 = out.get("gen_image1"), out.get("flow_image1")
        self.gen_dimage1, self.flow_dimage1 = out.get("gen_dimage1"), out.get("flow_dimage1")

    def encode(self, image0, dimage0, group=1):
        """The per-modality pre-encoders, e2_0 .. e4_0 and fc1 -> features [B * group, 4096] bf16 (each source's row repeated
        ``group`` times)."""
        g = self.algo
        x = image0 if image0 is not None else dimage0
        B, H = x.shape[0], x.shape[1]
        h5 = H // 32
        concat_list = []
        if self.use_color:
            concat_list.append(self.image_preprocessing(image0, "pre_image0"))
        if self.use_depth:
            concat_list.append(self.image_preprocessing(dimage0, "pre_dimage0"))
        comb_enc = torch.cat(concat_list, dim=3) if len(concat_list) > 1 else concat_list[0]
        a = "lrelu"
        e2_0 = conv2d_msra(comb_enc, 64, 5, 5, 1, 1, "e2_0", act=a, algo=g)
        e3 = conv2d_msra(e2_0, 128, 3, 3, 2, 2, "e3", act=a, algo=g)
        e3_0 = conv2d_msra(e3, 128, 3, 3, 1, 1, "e3_0", act=a, algo=g)
        e4 = conv2d_msra(e3_0, 256, 3, 3, 2, 2, "e4", act=a, algo=g)
        e4_0 = conv2d_msra(e4, 256, 3, 3, 1, 1, "e4_0", act=a, algo=g)
        return linear_msra(F.reshape(e4_0, (B, h5 * h5 * 256)), 4096, "fc1", act=a, algo=g, group=group)

    def decode(self, e5, disp, warp=None):
        """features [N, 4096] (encode), disp [N, viewpoint_dim] bf16 -> {gen_image1, gen_dimage1} [N, H, H, C] and, with
        head='flow', {flow_image1, flow_dimage1}: the viewpoint FCs, the joint FCs, the decoder and the heads.
        ``warp(source_key, flow)`` warps the source modality ("image0" / "depth0") of a flow head."""
        g, a = self.algo, "lrelu"
        B, H = e5.shape[0], self.image_shape[0]
        h5 = H // 32
        a0 = linear_msra(disp, 64, "a0", act=a, algo=g)
        a1 = linear_msra(a0, 64, "a1", act=a, algo=g)
        a2 = linear_msra(a1, 64, "a2", act=a, algo=g)
        a3 = linear_msra(torch.cat([e5, a2], dim=1), 4096, "a3", act=a, algo=g)
        a4 = linear_msra(a3, 4096, "a4", act=a, algo=g)
        a5 = linear_msra(a4, h5 * h5 * 256, "a5", act=a, algo=g)
        a5r = F.reshape(a5, (B, h5, h5, 256))
        d4 = deconv2d_msra(a5r, [B, 2 * h5, 2 * h5, 128], 3, 3, 2, 2, "d4", act=a, algo=g)
        d4_0 = conv2d_msra(d4, 128, 3, 3, 1, 1, "d4_0", act=a, algo=g)
        d3 = deconv2d_msra(d4_0, [B, 4 * h5, 4 * h5, 64], 3, 3, 2, 2, "d3", act=a, algo=g)
        num_decode = int(self.use_color) + int(self.use_depth)
        d3_0 = conv2d_msra(d3, 64 * num_decode, 5, 5, 1, 1, "d3_0", act=a, algo=g)
        split_list = list(torch.chunk(d3_0, num_decode, dim=3))
        out = {}
        if self.use_color:       # split_list.pop(): the colour head takes the LAST channel group (main_model.py:131-133)
            out["gen_image1"], out["flow_image1"] = self.decode_output(split_list.pop(), "dec_image1", 3, lambda f: warp("image0", f))
        if self.use_depth:
            out["gen_dimage1"], out["flow_dimage1"] = self.decode_output(split_list.pop(), "dec_dimage1", 1, lambda f: warp("depth0", f))
        assert split_list == []
        return {k: v for k, v in out.items() if v is not None}

    def forward(self, image0, dimage0, disp):
        """image0 [B,H,H,3], dimage0 [B,H,H,1] fp32 in [0,1], disp [B,V] -> dict(gen_image1, gen_dimage1).
        disp [B,T,V]: T targets per source, outputs [B,T,H,H,C]."""
        self.gen_image1 = self.gen_dimage1 = self.loss = None
        self.store.new_anchor()
        self.image0, self.dimage0, self.disp = image0, dimage0, disp
        if disp.dim() == 3:
            B, T = int(disp.shape[0]), int(disp.shape[1])
            with use_store(self.store):
                self.buildModel(image0, dimage0, F.to_bf16(disp.reshape(B * T, disp.shape[2])), T)
            for k in ("gen_image1", "flow_image1", "gen_dimage1", "flow_dimage1"):
                v = getattr(self, k)
                if v is not None:
                    setattr(self, k, v.reshape((B, T) + tuple(v.shape[1:])))
        else:
            with use_store(self.store):
                self.buildModel(image0, dimage0, F.to_bf16(disp))
        out = {}
        if self.use_color:
            out["gen_image1"] = self.gen_image1
        if self.use_depth:
            out["gen_dimage1"] = self.gen_dimage1
        return out

    def build_loss(self, image1, dimage1):
        """main_model.py:144-154: loss = L(colour) + L(depth) * depth_lr_factor; mean over the global batch."""
        n = image1.numel() // image1.shape[-1] * self.world_size       # every target pixel: B*H*W (B*T*H*W with T targets)
        loss = None
        if self.use_color:
            loss = F.reconstruction_loss(self.gen_image1, image1, self.loss_mode, inv_count=1.0 / n, unit_upstream=True,
                                         **self._ssim_kw())
        if self.use_depth:
            f = float(self.conf["depth_lr_factor"])
            ld = F.reconstruction_loss(self.gen_dimage1, dimage1, self.loss_mode, weights=[f], inv_count=1.0 / n, unit_upstream=True,
                                       **self._ssim_kw())
            loss = ld if loss is None else loss + ld
        self.image1, self.dimage1, self.loss = image1, dimage1, loss
        return loss

    def input_spec(self):
        B, H = self.batch_size, self.image_shape[0]
        T = () if self.num_targets == 1 else (self.num_targets,)
        return {"image0": (B, H, H, 3), "depth0": (B, H, H, 1), "image1": (B,) + T + (H, H, 3), "depth1": (B,) + T + (H, H, 1),
                "disp": (B,) + T + (self.viewpoint_dim,)}

    def step_loss(self, batch):
        self.forward(batch["image0"], batch["depth0"], batch["disp"])
        return self.build_loss(batch["image1"], batch["depth1"])

    def render_sources(self):
        return (("image0",) if self.use_color else ()) + (("depth0",) if self.use_depth else ())

    def _render_encode(self, sources):
        return self.encode(sources.get("image0"), sources.get("depth0"))

    def _render_decode(self, sources, features, viewpoint, group):
        return self.decode(features, viewpoint, lambda key, flow: F.flow_resampler_shared(sources[key], flow, group, self.grid_order))
