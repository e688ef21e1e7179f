"""Drop-in for the reference's ``sampling/collaborator.py`` (graph refiner of the image path).

Same names as ``sampling/collaborator.py:7-88``: ``Refiner(rollout_steps, rollout_rate, rollout_method)``,
``set_env(discriminator, feature_to_data, func_loss)``, ``set_constraints(vmin, vmax)``,
``compute_forward_logits_and_grad(feature)``, ``build_refiner(fake_feature, real_batch, mode)`` and the result
attributes ``default_logit / optimal_logit / optimal_step / optimal_feature / current_feature / current_logit``.

Semantic shift (SURVEY.md §8b): the reference builds a symbolic TF graph from python callables; here
``discriminator`` / ``feature_to_data`` are network specs (``cgs.nets.discriminator_spec(spec)`` /
``feature_to_data_spec(spec)``) and ``build_refiner`` runs eagerly and returns the refined batch.
``func_loss`` must be the BCE-with-ones marker ``cgs.nets.loss_refine`` (nsgan/GAN.py:176-177).
D's BatchNorm runs in inference mode (folded) by default; ``discriminator_spec(spec, is_training=True)`` selects the
reference's training mode (statistics of the refined batch, nsgan/GAN.py:175), see DESIGN.md.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

try:
    from . import _paths  # noqa: F401
    from .policy import PolicyAdaptive
except ImportError:
    import _paths  # noqa: F401
    from policy import PolicyAdaptive
from cgs import lib as L
from cgs import nets as N
from cgs import runtime as R


class Refiner():
    def __init__(self, rollout_steps, rollout_rate, rollout_method="momentum", math=None, cuda_graph=False):
        self.forward_steps = rollout_steps
        self.optimizer = PolicyAdaptive(rollout_rate, rollout_method)
        self.log = False
        self.vmin = None
        self.vmax = None
        self.math = math
        self.early_exit_logit = None      # opt-in (README.md:13); None = reference behaviour (best of K)
        self.cuda_graph = cuda_graph      # capture the K-step launch sequence once per batch shape and replay it
        self.chunk_rows = None            # refine at most this many rows per launch sequence (bounds the workspace)
        self._graphs = {}
        self.replayed_launches = 0        # kernels executed through graph replays (cgs_launch_count sees captures only)
        self._ws = R.Workspace()
        self.real_logits = None
        self.real_logits_mean = None
        self.forward_grad = None

    def set_env(self, discriminator, feature_to_data, func_loss):
        spec_d = discriminator.spec if isinstance(discriminator, N._Role) else discriminator
        spec_g = feature_to_data.spec if isinstance(feature_to_data, N._Role) else feature_to_data
        if not isinstance(spec_d, N.NetSpec) or not isinstance(spec_g, N.NetSpec):
            raise TypeError("discriminator / feature_to_data must be cgs.nets specs (python callables cannot be fused)")
        if not getattr(func_loss, "is_bce_with_ones", False):
            raise NotImplementedError("only the reference's BCE-with-ones refinement loss is built (nsgan/GAN.py:176-177)")
        if getattr(feature_to_data, "is_training", False):
            raise NotImplementedError("G's tail runs in inference mode, as in the reference (nsgan/GAN.py:94)")
        self.discriminator = discriminator
        self.feature_to_data = feature_to_data
        self.func_loss = func_loss
        # captured graphs hold the weight / bias pointers of the previous environment by value: never replay them
        # against another one (their cache entries also keep the specs they were captured with alive)
        self._graphs = {}
        self._batch_bn = bool(getattr(discriminator, "is_training", False))
        self._d = spec_d.d_batch if self._batch_bn else spec_d.d
        self._bn = C.byref(self._d.bn_desc) if self._batch_bn else None     # NULL: inference mode
        self._g = spec_g.gtail
        self._spec = spec_g
        self._cimg = spec_g.image_shape[2]
        if self.math is None:
            self.math = spec_g.math
        if spec_g.math != spec_d.math or self.math != spec_g.math:
            raise ValueError("math mode of the refiner and of both specs must agree (weights are packed per mode)")

    def set_constraints(self, vmin, vmax):
        self.vmin = vmin
        self.vmax = vmax
        print("set_constraints: self.vmin = {:.2f}, self.vmax = {:.2f}".format(self.vmin, self.vmax))

    # ------------------------------------------------------------------------------------------
    def _workspace(self, B, dev):
        nbytes = L.load().cgs_refine_workspace_bytes_bn(C.byref(self._g.desc), C.byref(self._d.desc), self._bn, B)
        if nbytes == 0:
            L.check(-1 if not L.last_error() else -2)
        return self._ws.get(nbytes, dev)

    def _max_rows_per_launch(self):
        return int(L.check(L.load().cgs_refine_max_batch(C.byref(self._g.desc), C.byref(self._d.desc))))

    def _img_shape(self, B):
        h, w, c = self._spec.image_shape
        return (B, h, w, N.cstride(c))

    def compute_forward_logits_and_grad(self, current_feature):
        """collaborator.py:26-39 -> (per-sample logit [B], d sum(loss) / d feature)."""
        dev = self._spec.device
        feat, _ = R.to_device(current_feature, torch.float32, dev)
        B = feat.shape[0]
        logit = torch.empty(B, dtype=torch.float32, device=dev)
        grad = torch.empty_like(feat)
        ws = self._workspace(B, dev)
        L.check(L.load().cgs_forward_logits_and_grad_bn(C.byref(self._g.desc), C.byref(self._d.desc), self._bn,
                                                        L.MATH_IDS[self.math], B, L.ptr(feat), L.ptr(logit), L.ptr(grad),
                                                        None, L.ptr(ws), ws.numel(), L.stream_ptr()))
        return logit, grad

    def feature_to_image(self, feature):
        """feature_to_data(feature) (nsgan/GAN.py:94-101) -> [B,h,w,c] and its logit."""
        dev = self._spec.device
        feat, _ = R.to_device(feature, torch.float32, dev)
        B = feat.shape[0]
        logit = torch.empty(B, dtype=torch.float32, device=dev)
        img = torch.empty(self._img_shape(B), dtype=torch.float32, device=dev)
        ws = self._workspace(B, dev)
        L.check(L.load().cgs_forward_logits_and_grad_bn(C.byref(self._g.desc), C.byref(self._d.desc), self._bn,
                                                        L.MATH_IDS[self.math], B, L.ptr(feat), L.ptr(logit), None,
                                                        L.ptr(img), L.ptr(ws), ws.numel(), L.stream_ptr()))
        return img[..., :self._cimg], logit

    def prefetch(self, fake_feature):
        """Start the host-to-device copy of the NEXT proposal batch on a side stream and return the device tensor to
        hand to `build_refiner` later: the upload then overlaps the refinement of the current batch (the fill-up loop
        knows its next proposals one batch ahead).  `fake_feature`: numpy array or (ideally pinned) host tensor."""
        dev = self._spec.device
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        with torch.cuda.stream(self._copy_stream):
            t, _ = R.to_device(fake_feature, torch.float32, dev)
            ready = torch.cuda.Event()
            ready.record(self._copy_stream)
        t._cgs_ready = ready                                     # build_refiner orders its stream after the copy
        return t

    def build_refiner(self, fake_feature, real_batch=None, mode='deterministic', prob_indices=None,
                      keep_optimal_feature=False):
        if mode not in ('deterministic', 'probabilistic'):
            raise NotImplementedError(mode)
        ready = getattr(fake_feature, "_cgs_ready", None)
        if ready is not None:                                    # a batch staged by prefetch()
            torch.cuda.current_stream().wait_event(ready)
            fake_feature.record_stream(torch.cuda.current_stream())
        method = self.optimizer.method
        if method == 'ladam':
            # the reference calls apply_gradient without a loss here (collaborator.py:66) -> policy.py:51 fails
            raise TypeError("unsupported operand type(s) for +: 'NoneType' and 'float'")
        if method not in ('sgd', 'momentum'):
            raise NotImplementedError(method)                     # policy.py:64
        dev = self._spec.device
        lib = L.load()
        feat_in, was_np = R.to_device(fake_feature, torch.float32, dev)
        if tuple(feat_in.shape[1:]) != self._spec.feature_shape:
            raise ValueError("feature shape %s does not match the spec %s" % (tuple(feat_in.shape[1:]), self._spec.feature_shape))
        B = feat_in.shape[0]
        # the kernels index rows with 32 bits: very large batches are refined in independent chunks (samples are
        # independent under inference-mode BN, so chunking does not change a single bit)
        limit = self._max_rows_per_launch()
        if self.chunk_rows:
            limit = max(1, min(limit, int(self.chunk_rows)))
        if self._batch_bn:
            # training-mode BN normalises over the whole batch: chunks or leaving rows would change the statistics
            if B > limit:
                raise ValueError("a training-mode discriminator refines one batch of at most %d rows in one call "
                                 "(chunking would change the batch statistics)" % limit)
            if self.early_exit_logit is not None:
                raise ValueError("early exit changes the batch the training-mode BN statistics run over")
        if B > limit:
            if prob_indices is None and mode == 'probabilistic':
                prob_indices = np.random.randint(self.forward_steps + 1, size=B)
            outs, attrs = [], []
            for lo in range(0, B, limit):
                pi = None if prob_indices is None else np.asarray(prob_indices)[lo:lo + limit]
                outs.append(self.build_refiner(feat_in[lo:lo + limit], None, mode, pi, keep_optimal_feature))
                attrs.append((self.current_feature, self.default_logit, self.optimal_logit, self.optimal_step, self.optimal_feature))
            cat = lambda i: None if attrs[0][i] is None else torch.cat([a[i] for a in attrs])
            self.current_feature, self.default_logit, self.optimal_logit = cat(0), cat(1), cat(2)
            self.optimal_step, self.optimal_feature = cat(3), cat(4)
            refined = torch.cat(outs)
            return refined.cpu().numpy() if was_np else refined
        idx_host = None
        if mode == 'probabilistic':
            if prob_indices is None:
                prob_indices = np.random.randint(self.forward_steps + 1, size=B)      # collaborator.py:56
            idx_host = np.asarray(prob_indices, dtype=np.int32)
        cfg = L.RefineCfg()
        cfg.steps = int(self.forward_steps)
        cfg.rate = float(self.optimizer.lambda_)
        cfg.method = L.POLICY_IDS[method]
        cfg.alpha = float(self.optimizer.alpha_)
        cfg.mode = L.MODE_PROBABILISTIC if mode == 'probabilistic' else L.MODE_DETERMINISTIC
        cfg.clip = 1 if (self.vmin and self.vmax) else 0           # collaborator.py:69 (truthiness, sic)
        cfg.vmin = float(self.vmin) if cfg.clip else 0.0
        cfg.vmax = float(self.vmax) if cfg.clip else 0.0
        cfg.math = L.MATH_IDS[self.math]
        cfg.early_exit = 0 if self.early_exit_logit is None else 1
        cfg.exit_logit = float(self.early_exit_logit or 0.0)

        def buffers():
            b = dict(feat=torch.empty_like(feat_in),
                     best_img=torch.empty(self._img_shape(B), dtype=torch.float32, device=dev),
                     best_logit=torch.empty(B, dtype=torch.float32, device=dev),
                     best_step=torch.empty(B, dtype=torch.float32, device=dev),
                     default_logit=torch.empty(B, dtype=torch.float32, device=dev),
                     best_feat=torch.empty_like(feat_in) if keep_optimal_feature else None,
                     idx=torch.empty(B, dtype=torch.int32, device=dev) if mode == 'probabilistic' else None)
            return b

        def launch(b, ws):
            L.check(lib.cgs_refine_conv_bn(C.byref(self._g.desc), C.byref(self._d.desc), self._bn, C.byref(cfg), B,
                                           L.ptr(b["feat"]), L.ptr(b["best_img"]), L.ptr(b["best_logit"]),
                                           L.ptr(b["best_step"]), L.ptr(b["default_logit"]), L.ptr(b["idx"]),
                                           L.ptr(b["best_feat"]), L.ptr(ws), ws.numel(), L.stream_ptr()))

        if not self.cuda_graph:
            b = buffers()
            b["feat"].copy_(feat_in)                                  # tf.identity (collaborator.py:48,58)
            if idx_host is not None:
                b["idx"].copy_(torch.from_numpy(idx_host))
            launch(b, self._workspace(B, dev))
        else:
            # the launch sequence depends only on (shapes, config): capture it once, replay afterwards
            key = (B, mode, cfg.steps, cfg.rate, cfg.method, cfg.alpha, cfg.clip, cfg.vmin, cfg.vmax, cfg.math,
                   cfg.early_exit, cfg.exit_logit, keep_optimal_feature, self._batch_bn, id(self._g), id(self._d), str(dev))
            ent = self._graphs.get(key)
            if ent is None:
                b = buffers()
                nbytes = lib.cgs_refine_workspace_bytes_bn(C.byref(self._g.desc), C.byref(self._d.desc), self._bn, B)
                ws = torch.empty(int(nbytes), dtype=torch.uint8, device=dev)
                b["feat"].copy_(feat_in)
                if idx_host is not None:
                    b["idx"].copy_(torch.from_numpy(idx_host))
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):
                    launch(b, ws)                                     # warm-up outside capture (one-time attribute setup)
                torch.cuda.current_stream(dev).wait_stream(side)
                graph = torch.cuda.CUDAGraph()
                n0 = lib.cgs_launch_count()
                with torch.cuda.graph(graph):
                    launch(b, ws)
                ent = self._graphs[key] = (graph, b, ws, int(lib.cgs_launch_count() - n0), (self._g, self._d))
            graph, sb, _, n_kernels, _ = ent
            self.replayed_launches += n_kernels
            sb["feat"].copy_(feat_in)
            if idx_host is not None:
                sb["idx"].copy_(torch.from_numpy(idx_host))
            graph.replay()
            b = {k: (v.clone() if v is not None else None) for k, v in sb.items()}   # results outlive the next replay
        feat, best_img, best_logit, best_step = b["feat"], b["best_img"], b["best_logit"], b["best_step"]
        default_logit, best_feat = b["default_logit"], b["best_feat"]
        self.optimizer.reset_moving_average()                       # collaborator.py:86
        self.current_feature = feat
        self.default_logit = default_logit
        self.optimal_logit = best_logit
        self.optimal_step = best_step
        self.optimal_feature = best_feat
        self.current_logit = None
        refined = best_img[..., :self._cimg]                        # == feature_to_data(optimal_feature), :88
        if was_np:
            return refined.cpu().numpy()
        return refined
