"""Model-level drop-in surface, "next" rows of SURVEY 8(f)-3.

``MultiObjectAppFlow`` mirrors dyn_mult_view/multi_view_model/multiobject_appflow.py:14-286: one pre-encoder per
input (colour ``pre_image0_f``, depth ``pre_dimage0_f``, the two object masks ``pre_mask0_ob0/1``, :80-132), the
shared trunk with the FC bottleneck or the ``fully_conv`` viewpoint smear (:134-166), ``d3_0`` widened to
``64 * num_decode`` and split, ``split_list.pop()`` handing out the LAST group first (:168-218), flow decoders that
all sample ``image0`` (:89-102, 193-198), tanh decoders for depth and masks (:104-120), and the loss of :223-283
(euclidean terms, ``masked_image_loss``, ``use_depth`` / ``predict_target_masks`` factors).  Feature switches are
key-presence tests on ``conf`` as in the reference.

``MultiViewFusionAppFlow`` is BASELINE config 5, which the reference does not contain (SURVEY 8(0) row 5, definition
8(f)-3): ``num_views`` source frames of a multi-object scene per sample.  Every source frame runs the MULTI-OBJECT trunk
above (its colour image, its depth map when ``use_depth`` is set, its two object masks -- the pre-encoders of
multiobject_appflow.py:123-134 -- and its own viewpoint change to the target; shared weights), and ONE decoder
(``dec_image1``) ends in a single 3-channel head ``d0``: channels 0-1 are the flow that warps that frame's colour image,
channel 2 is its per-pixel confidence logit.  The prediction is  sum_v softmax_v(logit)_v * warp(src_v, flow_v)  (after
Zhou et al. 2016); the fusion, the loss and both gradients are one fused kernel (dmv_loss_fused_fwd_bwd).  The views are
a batch dimension for every layer.
"""
import torch

from . import functional as F
from .model_base import ModelBase
from .optimizer import TFAdam
from .tf_utils import conv2d_msra, deconv2d_msra, flow_resample_layer, linear_msra
from .variables import VariableStore, use_store

INPUTS = [("use_color", "image0", "pre_image0_f", 3), ("use_depth", "depth0", "pre_dimage0_f", 1),
          (None, "image0_mask0", "pre_mask0_ob0", 1), (None, "image0_mask1", "pre_mask0_ob1", 1)]
BATCH_KEYS = ["image0", "image0_mask0", "image0_mask1", "image1", "image1_only0", "image1_only1", "image1_mask0", "image1_mask1",
              "depth0", "depth1", "depth1_only0", "depth1_only1", "displacement"]


def decoder_heads(conf):
    """(attribute, scope, kind) in the order multiobject_appflow.py:189-218 pops the channel groups."""
    heads = []
    if "use_color" in conf:
        if "combination_image" in conf:
            heads.append(("gen_image1", "dec_image1", "flow"))
        if "gen_sep_images" in conf:
            heads += [("gen_image1_only0", "dec_image1_only0", "flow"), ("gen_image1_only1", "dec_image1_only1", "flow")]
    if "use_depth" in conf:
        if "combination_image" in conf:
            heads.append(("gen_depth1", "dec_dimage1_f", "tanh"))
        if "gen_sep_images" in conf:
            heads += [("gen_depth1_only0", "dec_depth1_only0", "tanh"), ("gen_depth1_only1", "dec_depth1_only1", "tanh")]
    if "predict_target_masks" in conf:
        heads += [("gen_image1_mask0", "dec_image1_mask0", "tanh"), ("gen_image1_mask1", "dec_image1_mask1", "tanh")]
    return heads


class MultiObjectAppFlow(ModelBase):
    INPUT_KEYS = tuple(BATCH_KEYS)

    def __init__(self, conf, load_tfrec=True, build_loss=True, device=None):
        if int(conf.get("num_targets", 1)) > 1:
            raise ValueError(
                "%s trains one target per sample (num_targets = %s): its targets are per-object renders, masks and depths of "
                "a multi-object scene, not viewpoints of one source image" % (type(self).__name__, conf["num_targets"]))
        self.conf = conf
        self.batch_size = int(conf["batch_size"])
        H = int(conf.get("image_size", 128))
        if H % 32:
            raise ValueError("image_size must be a multiple of 32")
        self.image_shape = [H, H, 3]
        self.scalar_imshape = [H, H, 1]
        self.viewpoint_dim = int(conf.get("viewpoint_dim", 2))
        self.grid_order = conf.get("grid_order", "ref_yx")
        self.algo = conf.get("algo", None)
        self.max_iter, self.start_iter = 1000000, 0
        self.heads = self._heads(conf)
        if not self.heads:
            raise ValueError("conf selects no decoder output")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.store = VariableStore(self.device, seed=int(conf.get("seed", 0)))
        self.world_size = 1
        self.loss = None
        self.optimizer = None
        zeros = {k: torch.zeros(shp, dtype=torch.float32, device=self.device) for k, shp in self.input_spec().items()}
        if self.device.type == "meta":
            with torch.no_grad(), F.meta_mode():
                self.forward(zeros)
        else:
            with torch.no_grad():
                self.forward(zeros)
        self.store.finalize()
        self.t_vars = self.store.trainable_vars()
        if build_loss and self.device.type != "meta":
            self.optimizer = TFAdam(self.store, conf["learning_rate"])

    def _heads(self, conf):
        return decoder_heads(conf)

    def input_spec(self):
        B, H = self.batch_size, self.image_shape[0]
        spec = {k: (B, H, H, 3 if (k.startswith("image") and "mask" not in k) else 1) for k in BATCH_KEYS if k != "displacement"}
        spec["displacement"] = (B, self.viewpoint_dim)
        return spec

    def step_loss(self, batch):
        self.forward(batch)
        return self.build_loss(batch)

    def render(self, sources, viewpoints):
        raise NotImplementedError(
            "MultiObjectAppFlow has no render(): its encoder takes the image, the depth and the object masks of a scene of "
            "several objects and its heads predict per-object outputs, so a view is not a warp of one source image")

    def visualize(self, *args, **kw):
        """multiobject_appflow.py:289-393: imgdata.pkl with every clipped input / output (+ PNG panels)."""
        from .visualize import visualize_multiobject
        return visualize_multiobject(self, self._as_batch(args), **kw)

    # -- graph ---------------------------------------------------------------------------------
    def image_preprocessing(self, x, scope):
        """multiobject_appflow.py:80-87"""
        g = self.algo
        with self.store.scope(scope):
            e0 = conv2d_msra(x, 32, 5, 5, 2, 2, "e0", act="lrelu", algo=g)
            e0_0 = conv2d_msra(e0, 32, 5, 5, 1, 1, "e0_0", act="lrelu", algo=g)
            e1 = conv2d_msra(e0_0, 32, 5, 5, 2, 2, "e1", act="lrelu", algo=g)
            e1_0 = conv2d_msra(e1, 32, 5, 5, 1, 1, "e1_0", act="lrelu", algo=g)
            return conv2d_msra(e1_0, 64, 5, 5, 2, 2, "e2", act="lrelu", algo=g)

    def _decode_trunk(self, x, scope_unused=None):
        g = self.algo
        B, H = x.shape[0], self.image_shape[0]
        h5 = H // 32
        d2 = deconv2d_msra(x, [B, 8 * h5, 8 * h5, 32], 5, 5, 2, 2, "d2", act="lrelu", algo=g)
        d2_0 = conv2d_msra(d2, 64, 5, 5, 1, 1, "d2_0", act="lrelu", algo=g)
        d1 = deconv2d_msra(d2_0, [B, 16 * h5, 16 * h5, 32], 5, 5, 2, 2, "d1", act="lrelu", algo=g)
        return conv2d_msra(d1, 32, 5, 5, 1, 1, "d1_0", act="lrelu", algo=g)

    def decode_flow(self, src_img, x, scope):
        """multiobject_appflow.py:89-102: 2-channel flow head, warp of src_img (always image0)."""
        B, H = x.shape[0], self.image_shape[0]
        with self.store.scope(scope):
            d1_0 = self._decode_trunk(x)
            flow = deconv2d_msra(d1_0, [B, H, H, 2], 5, 5, 2, 2, "d0", act=None, algo=self.algo, out_dtype=torch.float32)
            return flow_resample_layer(src_img, flow, self.grid_order)

    def decode_direct(self, x, scope, num_outputs=1):
        """multiobject_appflow.py:104-120: one-channel tanh head."""
        B, H = x.shape[0], self.image_shape[0]
        with self.store.scope(scope):
            d1_0 = self._decode_trunk(x)
            return deconv2d_msra(d1_0, [B, H, H, 1], 5, 5, 2, 2, "d0", act="tanh", algo=self.algo, out_dtype=torch.float32)

    def buildModel(self, batch):
        """multiobject_appflow.py:123-221"""
        g, a = self.algo, "lrelu"
        B, H = batch["image0"].shape[0], self.image_shape[0]
        h5 = H // 32
        concat_list = [self.image_preprocessing(batch[attr], scope) for key, attr, scope, _ in INPUTS if key is None or key in self.conf]
        comb_enc = torch.cat(concat_list, dim=3)
        e2_0 = conv2d_msra(comb_enc, 64, 5, 5, 1, 1, "e2_0", act=a, algo=g)
        e3 = conv2d_msra(e2_0, 128, 3, 3, 2, 2, "e3", act=a, algo=g)
        e3_0 = conv2d_msra(e3, 128, 3, 3, 1, 1, "e3_0", act=a, algo=g)
        e4 = conv2d_msra(e3_0, 256, 3, 3, 2, 2, "e4", act=a, algo=g)
        e4_0 = conv2d_msra(e4, 256, 3, 3, 1, 1, "e4_0", act=a, algo=g)
        disp = F.to_bf16(batch["displacement"])
        a0 = linear_msra(disp, 64, "a0", act=a, algo=g)
        a1 = linear_msra(a0, 64, "a1", act=a, algo=g)
        a2 = linear_msra(a1, 64, "a2", act=a, algo=g)
        if "fully_conv" in self.conf:        # :147-153: the viewpoint code is tiled over the bottleneck and convolved
            smear = a2.reshape(B, 1, 1, a2.shape[1]).expand(B, h5, h5, a2.shape[1])
            concated = torch.cat([e4_0, smear], dim=3)
            e4_1 = conv2d_msra(concated, 256, 3, 3, 1, 1, "e4_1", act=a, algo=g)
            a5r = conv2d_msra(e4_1, 256, 3, 3, 1, 1, "e4_2", act=a, algo=g)
        else:
            e5 = linear_msra(F.reshape(e4_0, (B, h5 * h5 * 256)), 4096, "fc1", act=a, algo=g)
            a3 = linear_msra(torch.cat([e5, a2], dim=1), 4096, "a3", act=a, algo=g)
            a4 = linear_msra(a3, 4096, "a4", act=a, algo=g)
            a5 = linear_msra(a4, h5 * h5 * 256, "a5", act=a, algo=g)
            a5r = F.reshape(a5, (B, h5, h5, 256))
        d4 = deconv2d_msra(a5r, [B, 2 * h5, 2 * h5, 128], 3, 3, 2, 2, "d4", act=a, algo=g)
        d4_0 = conv2d_msra(d4, 128, 3, 3, 1, 1, "d4_0", act=a, algo=g)
        d3 = deconv2d_msra(d4_0, [B, 4 * h5, 4 * h5, 64], 3, 3, 2, 2, "d3", act=a, algo=g)
        num_decode = len(self.heads)
        d3_0 = conv2d_msra(d3, 64 * num_decode, 5, 5, 1, 1, "d3_0", act=a, algo=g)
        split_list = [t.contiguous() for t in torch.chunk(d3_0, num_decode, dim=3)]
        out = {}
        for attr, scope, kind in self.heads:
            x = split_list.pop()
            if kind == "flow":
                out[attr] = self.decode_flow(batch["image0"], x, scope)
            elif kind == "flowconf":
                out[attr] = self.decode_flowconf(batch["image0"], x, scope)
            else:
                out[attr] = self.decode_direct(x, scope)
        assert split_list == []
        return out

    def forward(self, batch):
        """batch: dict of NHWC fp32 tensors under the reference's attribute names (BATCH_KEYS)."""
        self.loss = None
        self.store.new_anchor()
        self.batch = batch
        with use_store(self.store):
            self.out = self.buildModel(batch)
        for k, v in self.out.items():
            setattr(self, k, v)
        return self.out

    def build_loss(self, batch=None):
        """multiobject_appflow.py:223-283; every mean runs over the global batch."""
        b = batch or self.batch
        n = b["image1"].shape[0] * b["image1"].shape[1] * b["image1"].shape[2] * self.world_size
        conf, out = self.conf, self.out
        terms = []

        def term(gen, tgt, factor=1.0, mask=None):
            Cc = out[gen].shape[-1]
            terms.append(F.reconstruction_loss(out[gen], b[tgt], "l2", weights=[float(factor)] * Cc, inv_count=1.0 / n,
                                               mask=b[mask] if mask else None, unit_upstream=True))

        masked = "masked_image_loss" in conf
        if "use_color" in conf:
            if "combination_image" in conf:
                term("gen_image1", "image1")
            if "gen_sep_images" in conf:
                term("gen_image1_only0", "image1_only0", 1.0, "image1_mask0" if masked else None)
                term("gen_image1_only1", "image1_only1", 1.0, "image1_mask1" if masked else None)
        if "use_depth" in conf:
            f = float(conf["use_depth"])
            if "combination_image" in conf:
                term("gen_depth1", "depth1")
            if "gen_sep_images" in conf:
                term("gen_depth1_only0", "depth1_only0", f, "image1_mask0" if masked else None)
                term("gen_depth1_only1", "depth1_only1", f, "image1_mask1" if masked else None)
        if "predict_target_masks" in conf:
            f = float(conf["predict_target_masks"])
            term("gen_image1_mask0", "image1_mask0", f)
            term("gen_image1_mask1", "image1_mask1", f)
        loss = terms[0]
        for t in terms[1:]:
            loss = loss + t
        self.loss = loss
        return loss


class MultiViewFusionAppFlow(MultiObjectAppFlow):
    """BASELINE config 5: ``num_views`` source frames per sample on the multi-object trunk, one 3-channel
    flow + confidence head per frame, softmax fusion (module docstring)."""
    SRC_KEYS = ("image0", "depth0", "image0_mask0", "image0_mask1")

    def render(self, sources, viewpoints):
        raise NotImplementedError(
            "MultiViewFusionAppFlow has no render(): each view it predicts fuses the warps of num_views source frames of "
            "a multi-object scene by predicted confidences, and rendering covers one source image per sample")

    def __init__(self, conf, load_tfrec=True, build_loss=True, device=None):
        self.num_views = int(conf.get("num_views", 4))
        self.loss_mode = conf.get("loss", "l2")
        if self.loss_mode == "ssim":
            raise ValueError("%s has no 'ssim' loss: its kernel fuses the views before the loss and has no SSIM form; use 'l2' "
                             "or 'l1'" % type(self).__name__)
        self.gens = self.logits = self.fused = self.flow_field = None
        conf = dict(conf)
        conf.setdefault("use_color", "")
        super().__init__(conf, load_tfrec, build_loss, device)

    def _heads(self, conf):
        return [("gen_image1", "dec_image1", "flowconf")]

    @property
    def INPUT_KEYS(self):
        return tuple(k for k in self.SRC_KEYS if k != "depth0" or "use_depth" in self.conf) + ("displacement", "image1")

    def input_spec(self):
        B, H, Vw = self.batch_size, self.image_shape[0], self.num_views
        spec = {"image0": (Vw, B, H, H, 3)}
        if "use_depth" in self.conf:
            spec["depth0"] = (Vw, B, H, H, 1)
        spec.update(image0_mask0=(Vw, B, H, H, 1), image0_mask1=(Vw, B, H, H, 1), displacement=(Vw, B, self.viewpoint_dim),
                    image1=(B, H, H, 3))
        return spec

    def visualize(self, *args, **kw):
        from .visualize import visualize_multiview
        return visualize_multiview(self, self._as_batch(args), **kw)

    def decode_flowconf(self, src_img, x, scope):
        """One 3-channel head: flow (channels 0-1) + confidence logit (channel 2), SURVEY 8(f)-3."""
        B, H = x.shape[0], self.image_shape[0]
        with self.store.scope(scope):
            d1_0 = self._decode_trunk(x)
            head = deconv2d_msra(d1_0, [B, H, H, 3], 5, 5, 2, 2, "d0", act=None, algo=self.algo, out_dtype=torch.float32)
        flow, logit = head[..., :2].contiguous(), head[..., 2].contiguous()
        return flow_resample_layer(src_img, flow, self.grid_order), flow, logit

    def forward(self, batch):
        """batch: image0 [Vw,B,H,H,3], (depth0,) image0_mask0/1 [Vw,B,H,H,1], displacement [Vw,B,V] (each frame's
        viewpoint change to the target), image1 [B,H,H,3] -> dict(flow_field [Vw,B,H,H,2], gens, logits)."""
        self.loss = self.gens = self.logits = self.fused = self.flow_field = None
        self.store.new_anchor()
        self.batch = batch
        Vw, B, H = batch["image0"].shape[0], batch["image0"].shape[1], batch["image0"].shape[2]
        flat = {k: batch[k].reshape((Vw * B,) + tuple(batch[k].shape[2:])) for k in self.SRC_KEYS + ("displacement",) if k in batch}
        with use_store(self.store):
            out = self.buildModel(flat)
        gen, flow, logit = out["gen_image1"]
        self.flow_field = flow.reshape(Vw, B, H, H, 2)
        self.gens = gen.reshape(Vw, B, H, H, 3)
        self.logits = logit.reshape(Vw, B, H, H)
        self.out = {"flow_field": self.flow_field, "gens": self.gens, "logits": self.logits}
        return self.out

    def build_loss(self, batch=None):
        image1 = (batch or self.batch)["image1"]
        n = image1.shape[0] * image1.shape[1] * image1.shape[2] * self.world_size
        self.loss, self.fused = F.fused_views_loss(self.gens, self.logits, image1, self.loss_mode, inv_count=1.0 / n)
        self.gen_image1 = self.fused
        return self.loss
