"""What every model class of the path shares: the step interface the driver and the CUDA-graph step use, and the
checkpoint surface.

The reference's driver touches a model only through ``Model(conf, load_tfrec, build_loss)``, ``model.loss``,
``model.train_op`` and the savers (dyn_mult_view/multi_view_model/train.py:57-65,117-136).  There is no TF session
here, so the same contract is:

  INPUT_KEYS            names of the tensors one ``sess.run`` consumes (the TFRecord feature names where they exist)
  input_spec()          name -> shape of one batch (float32 NHWC, values in [0,1]; viewpoint rows float32)
  train_step(batch)     one ``sess.run([loss, train_op])``: forward, backward, exchange (data parallel), Adam
  eval_loss(batch)      one ``sess.run([loss], {train_cond: 0})``: the validation pass (train.py:128-132), no update
  state_dict()/load_state_dict()   tf.train.Saver over all global variables incl. the Adam slots (train.py:70-71)

``train_step`` also accepts the class's positional form (``train_step(image0, image1, disp)`` etc.).

Novel views (the single-view classes): ``render(sources, viewpoints)`` encodes each source once and decodes every
viewpoint from the same features; ``train.GraphedRender`` is its CUDA-graph form.
"""
import torch


class ModelBase(object):
    INPUT_KEYS = ()

    # -- step interface ------------------------------------------------------------------------------------
    def input_spec(self):
        raise NotImplementedError

    def _as_batch(self, args):
        if len(args) == 1 and isinstance(args[0], dict):
            return args[0]
        if len(args) != len(self.INPUT_KEYS):
            raise TypeError("%s.train_step takes a batch dict or %d tensors %s" % (type(self).__name__, len(self.INPUT_KEYS), self.INPUT_KEYS))
        return dict(zip(self.INPUT_KEYS, args))

    def step_loss(self, batch):
        """forward + loss on the training path; returns the scalar loss tensor (with its tape)."""
        raise NotImplementedError

    def _ssim_kw(self):
        """Extra keyword of the loss calls under conf['loss'] = 'ssim' (the weight of the SSIM term); 'l2' / 'l1' take none."""
        return {"alpha": self.ssim_alpha} if self.loss_mode == "ssim" else {}

    def train_step(self, *args):
        """One sess.run([loss, train_op]) of train.py:122: forward, backward, (gradient exchange,) Adam."""
        dp = getattr(self, "_dp", None)
        if dp is not None and hasattr(dp, "apply_deferred"):
            dp.apply_deferred()    # the late FC matrices take the previous step's update next to this step's encoder forward
        pp = getattr(self.store, "prepack", None)
        if pp is not None:
            pp.begin()             # every layer's packed weights for this step, on a side stream (functional.Prepack)
        try:
            return self._train_step_body(args)
        finally:
            if pp is not None:
                pp.end()

    def _train_step_body(self, args):
        loss = self.step_loss(self._as_batch(args))
        opt = self.optimizer
        opt.begin_step()           # single process: the big FC matrices are updated inside backward (optimizer.py)
        try:
            loss.backward()
        finally:
            opt.end_backward()
        if getattr(self, "_dp", None) is not None:
            self._dp.finish()
        opt.step()
        return loss.detach()

    def flush_updates(self):
        """Make every parameter reflect the completed steps (a deferred optimizer update may still be pending after
        train_step returns; forward passes and state_dict() do this themselves)."""
        dp = getattr(self, "_dp", None)
        if dp is not None and hasattr(dp, "flush"):
            dp.flush()

    def eval_loss(self, *args):
        """The validation pass of train.py:128-132 (val_summ_op): loss only, no gradient, no update."""
        with torch.no_grad():
            return self.step_loss(self._as_batch(args)).detach()

    # -- rendering -----------------------------------------------------------------------------------------------------
    def render_sources(self):
        """Names of the source inputs ``render`` takes."""
        raise NotImplementedError("%s does not implement render()" % type(self).__name__)

    def render(self, sources, viewpoints):
        """Novel views of each source.  ``sources``: dict name -> [B, ...] fp32 (``render_sources()``: image0, and depth0
        for the depth models); ``viewpoints``: [B, V, viewpoint_dim], or [V, viewpoint_dim] for every source.  The
        encoder runs once per source (batch B), the decoder once per view (batch B * V), and each warp reads its source
        in place (functional.flow_resampler_shared).  Returns a dict of [B, V, H, W, C] fp32: gen and flow for the flow
        models; gen_image1 / gen_dimage1 (and flow_image1 / flow_dimage1 with head='flow') for Base_Prediction_Model.
        Inference only (no_grad); reads no training state and leaves every training buffer where it is."""
        self.flush_updates()
        return self._render(sources, viewpoints)

    def _render(self, sources, viewpoints, role="render"):
        keys = self.render_sources()
        missing = [k for k in keys if k not in sources]
        if missing:
            raise KeyError("%s.render needs sources %s (missing %s)" % (type(self).__name__, keys, missing))
        B = int(sources[keys[0]].shape[0])
        if any(int(sources[k].shape[0]) != B for k in keys):
            raise ValueError("sources differ in batch size: %s" % {k: tuple(sources[k].shape) for k in keys})
        vp = viewpoints
        if vp.dim() == 2:
            vp = vp.unsqueeze(0).expand(B, vp.shape[0], vp.shape[1])
        if vp.dim() != 3 or vp.shape[0] != B or vp.shape[2] != self.viewpoint_dim:
            raise ValueError("viewpoints must be [B, V, %d] or [V, %d] with B = %d, got %s"
                             % (self.viewpoint_dim, self.viewpoint_dim, B, tuple(viewpoints.shape)))
        V = int(vp.shape[1])
        from . import functional as F
        from .variables import use_store
        with torch.no_grad(), F.render_scope(role), use_store(self.store):
            self.store._pass_uses = set()           # a fresh pass over the variables (VariableStore.get)
            feats = self._render_encode(sources).repeat_interleave(V, dim=0)
            out = self._render_decode(sources, feats, F.to_bf16(vp.reshape(B * V, self.viewpoint_dim)), V)
        return {k: v.reshape((B, V) + tuple(v.shape[1:])) for k, v in out.items()}

    def visualize(self, *a, **k):
        raise NotImplementedError("%s has no visualize(); the reference's own is broken for this class (SURVEY 3.3)" % type(self).__name__)

    # -- checkpoint surface (tf.train.Saver over GLOBAL_VARIABLES, train.py:70-71) --------------------------------
    def state_dict(self):
        """Every variable under its TF name, plus Adam's slots ``<name>/Adam`` (m), ``<name>/Adam_1`` (v) and the
        step state (beta powers, t).  Under sharded data parallelism this is a COLLECTIVE call: the fp32 masters and
        the moments live with their owning rank and are gathered first, so every rank must call it."""
        dp = getattr(self, "_dp", None)
        if dp is not None and hasattr(dp, "gather_full_state"):
            dp.gather_full_state()
        sd = self.store.state_dict()
        if self.optimizer is not None:
            for k, v in self.store.vars.items():
                if v.trainable:
                    sd[k + "/Adam"] = v.m.detach().cpu().clone()
                    sd[k + "/Adam_1"] = v.v.detach().cpu().clone()
            sd["__adam_state__"] = self.optimizer.state.detach().cpu().clone()
        return sd

    def load_state_dict(self, sd):
        dp = getattr(self, "_dp", None)
        if dp is not None and hasattr(dp, "reset_deferred"):
            dp.flush()
        self.store.load_state_dict({k: v for k, v in sd.items() if k in self.store.vars})
        if self.optimizer is not None:
            for k, v in self.store.vars.items():
                if k + "/Adam" in sd:
                    v.m.copy_(torch.as_tensor(sd[k + "/Adam"]).to(self.device))
                    v.v.copy_(torch.as_tensor(sd[k + "/Adam_1"]).to(self.device))
            if "__adam_state__" in sd:
                self.optimizer.state.copy_(torch.as_tensor(sd["__adam_state__"]).to(self.device))
