"""Drop-in `InterfacePhysics` for the hot path (reference: DeepPhysiNet/interface/interface_physics.py).

Keeps the constructor (:33-50), `place_one_batch` (:271-320, canonical argument order = the DDP call
site :1033-1035), `encoding_coord` (:322-332), `inverse_norm` (:232-262) and the checkpoint format of
`save_model` / `load_model` (:53-88).  The trainer loops, dataset, logging and visualisation of the
reference are out of scope (SURVEY.md section 2, rows 2/8/10).
"""
import os
import shutil

import torch
import torch.nn as nn

from . import functional as Fn
from .config import FACTOR_KEYS, TERM_NAMES, VAR_ORDER, PhysicsConsts
from .pe import SineCosPE
from .physics_net import PhysicsNet


class InterfacePhysics(nn.Module):
    def __init__(self, meta_cfg: dict, net_cfg: dict, obs_norm_cfg: dict, variable_cfg: dict = None,
                 train_cfg: dict = None, test_cfg=None, inference_cfg: dict = None, **kwargs):
        super().__init__()
        self.net_cfg, self.obs_norm_cfg, self.variable_cfg = net_cfg, obs_norm_cfg, variable_cfg
        self.train_cfg, self.test_cfg, self.inference_cfg = train_cfg or {}, test_cfg, inference_cfg
        self.physics_net = PhysicsNet(meta_cfg, net_cfg)
        self.pe = SineCosPE(3, include_input=False)
        img_size = self.train_cfg.get("img_size", (145, 257))
        if isinstance(img_size, (int, float)):
            self.lat_size, self.lon_size = img_size, img_size
        elif isinstance(img_size, (list, tuple)) and len(img_size) == 2:
            self.lat_size, self.lon_size = img_size
        else:
            raise NotImplementedError
        # set by run_train_interface in the reference (:339-342, :418, :438); given defaults from the config here
        self.dx = float(self.train_cfg.get("dx", 27000))
        self.dy = float(self.train_cfg.get("dy", 27000))
        self.dt = 3600.0
        self.pred_t_span = 86400
        self.with_clip = True
        self.mode = None            # None -> functional.default_mode()
        self.last_terms = None      # per-sample loss terms [B,6] (float64) of the last place_one_batch call

    # ---- checkpoints (:53-88) -------------------------------------------------------------------
    def save_model(self, checkpoint_path, epoch, global_step, prefix="physics", **kwargs):
        os.makedirs(checkpoint_path, exist_ok=True)
        checkpoint_file = os.path.join(checkpoint_path, "%s_%d.pth" % (prefix, epoch))
        state = {"model": self.physics_net.state_dict(), "epoch": epoch, "gobal_step": global_step}
        state.update(kwargs)
        torch.save(state, checkpoint_file)
        shutil.copy(checkpoint_file, os.path.join(checkpoint_path, "%s_latest.pth" % prefix))

    def load_model(self, checkpoint_path, current_epoch=None, prefix="downscale", map_location="cpu"):
        if os.path.isfile(checkpoint_path):
            model_file = checkpoint_path
        elif current_epoch is None:
            model_file = os.path.join(checkpoint_path, "%s_latest.pth" % prefix)
        else:
            model_file = os.path.join(checkpoint_path, "%s_%d.pth" % (prefix, current_epoch))
        if not os.path.exists(model_file):
            print("warning:%s does not exist!" % model_file)
            return None, 0, 0
        state = torch.load(model_file, map_location=map_location)
        step = state.pop("gobal_step", 0)
        epoch = state.pop("epoch", 0)
        return state, epoch + 1, step

    # ---- small PyTorch helpers kept for surface compatibility -------------------------------------
    def encoding_coord(self, x, y, t, pred_t_span):
        x = x / self.dx / (self.lon_size - 1)
        y = y / self.dy / (self.lat_size - 1)
        t = t / pred_t_span
        z = torch.stack([x, y, t], dim=1) if x.dim() == 1 else torch.cat([x, y, t], dim=1)
        return self.pe(z)

    def inverse_norm(self, u, v, P, T, q, rio, obs_norm_cfg, with_clip=False):
        outs = []
        for i, (data, key) in enumerate(zip((u, v, P, T, q, rio), VAR_ORDER)):
            cfg = obs_norm_cfg[key]
            if cfg.get("use_norm", True):
                if cfg.get("norm_type", "mean_norm").lower() != "mean_norm":
                    raise NotImplementedError("only mean_norm is supported on this path")
                data = data * cfg["norm_factor"][1] + cfg["norm_factor"][0]
                if i >= 2 and self.with_clip:      # :256-261 - the argument is shadowed by self.with_clip
                    data = torch.clip(data, cfg["bound"][0], cfg["bound"][1])
            outs.append(data)
        return tuple(outs)

    def consts(self, loss_factor) -> PhysicsConsts:
        return PhysicsConsts.from_cfg(self.obs_norm_cfg, loss_factor, dx=self.dx, dy=self.dy,
                                      lat_size=int(self.lat_size), lon_size=int(self.lon_size),
                                      pred_t_span=float(self.pred_t_span), with_clip=bool(self.with_clip))

    # ---- the hot path ---------------------------------------------------------------------------
    def place_one_batch(self, x, y, t, f, field_data, input_data, forecast_h, criterion, loss_factor,
                        global_step, local_rank, device, summary=None, prefix="inter", log_step=100):
        """Same contract as interface_physics.py:271-320: returns the scalar PDE loss (sum of the six weighted
        residual MSEs) whose .backward() reaches every physics_net parameter.  Host tensors are moved to
        `device` exactly as the reference does (:273-276); batches of samples ([B,N,...]) are allowed and
        give the mean over samples."""
        if not isinstance(criterion, nn.MSELoss) or getattr(criterion, "reduction", "mean") != "mean":
            raise NotImplementedError("the fused residual kernel implements nn.MSELoss() (losses/builder.py:10); got %r" % (criterion,))
        dev = torch.device(device)
        f, x, y, t = (a.to(dev, non_blocking=True) for a in (f, x, y, t))
        field_data = field_data.to(dev, non_blocking=True)
        input_data = input_data.to(dev, non_blocking=True)
        forecast_h = forecast_h.to(dev, non_blocking=True)
        B = field_data.shape[0]
        W = self.physics_net.decoder_weights(field_data, forecast_h)
        shp = (B, -1)
        total, terms = Fn.pde_residual(x.reshape(shp), y.reshape(shp), t.reshape(shp), f.reshape(shp),
                                       input_data.reshape(B, -1, 6), W, consts=self.consts(loss_factor), mode=self.mode)
        self.last_terms = terms
        if global_step % log_step == 1 and local_rank == 0:
            vals = terms.mean(dim=0).tolist()            # .item()-style sync, as in the reference's logging branch
            if summary is not None:
                summary.add_scalar("%s/total_loss" % prefix, float(sum(vals)), global_step)
                for name, v in zip(TERM_NAMES, vals):
                    summary.add_scalar("%s/%s" % (prefix, name), v, global_step)
            print("%s:" % prefix + ",".join("%s:%f" % (n, v) for n, v in zip(TERM_NAMES, vals)))
        return total.float()

    # ---- rows N1 / N3 / N4 of SURVEY 8(f): the callers either side of the hot path --------------------------------
    def margin_loss(self, W, x, y, t, input_data, target, beta=0.1, factor=1.0e6):
        """Supervised data loss of the train loop (interface_physics.py:464-474): values of the six nets at the label
        points against the observations, WeightSmoothL1Loss(beta) (losses/weights_loss.py:12-20) times margin_factor.
        W = physics_net.decoder_weights(...) so the encoder runs once per step instead of three times."""
        B = W.W1.shape[0]
        o = Fn.decoder_values(None, input_data.reshape(B, -1, 6), W, xyz=(x.reshape(B, -1), y.reshape(B, -1), t.reshape(B, -1)),
                              consts=self.consts(self._last_factor()), mode=self.mode)
        return torch.nn.functional.smooth_l1_loss(o, target.reshape(o.shape).to(o.dtype), beta=beta, reduction="none").mean() * factor

    def _last_factor(self):
        from .config import DEFAULT_LOSS_FACTOR
        return getattr(self, "_loss_factor", DEFAULT_LOSS_FACTOR)

    def training_losses(self, batch, loss_factor, with_pde=True, beta=0.1, fuse_margin=True):
        """One training step's loss exactly as interface_physics.py:464-501 composes it (margin data loss + interior PDE loss +
        PDE loss on the margin points), with ONE encoder / hyper-network pass shared by the three terms (the reference re-runs
        MetaNet for each, physics_net.py:42) and - SURVEY 8(f) N1 - ONE library call for the margin points: the reference sends
        them through the decoder twice (values for WeightSmoothL1Loss :467-474, then place_one_batch :489-496); here
        `functional.pde_margin_residual` returns both losses from one forward / reverse sweep / backward.
        `batch` holds device tensors: field_data [B,159,2405], forecast_h [B,1,1], margin_{x,y,t,f} [B,M],
        margin_input_data [B,M,6], margin_data [B,M,6], inter_{x,y,t,f} [B,N], inter_data [B,N,6].
        Returns (train_loss, parts dict).  fuse_margin=False keeps the two separate calls (cross-check)."""
        self._loss_factor = loss_factor
        W = self.physics_net.decoder_weights(batch["field_data"], batch["forecast_h"])
        consts = self.consts(loss_factor)
        mfac = loss_factor.get("margin_factor", 1.0e6)
        parts = {}
        if not (with_pde and fuse_margin):
            parts["margin_loss"] = self.margin_loss(W, batch["margin_x"], batch["margin_y"], batch["margin_t"],
                                                    batch["margin_input_data"], batch["margin_data"], beta=beta, factor=mfac)
            total = parts["margin_loss"]
        if with_pde:
            tot, terms = Fn.pde_residual(batch["inter_x"], batch["inter_y"], batch["inter_t"], batch["inter_f"], batch["inter_data"],
                                         W, consts=consts, mode=self.mode)
            parts["inter_pde_loss"], parts["inter_terms"] = tot, terms
            if fuse_margin:
                B = W.W1.shape[0]
                both, mterms, mloss, _ = Fn.pde_margin_residual(
                    batch["margin_x"], batch["margin_y"], batch["margin_t"], batch["margin_f"], batch["margin_input_data"],
                    batch["margin_data"].reshape(B, -1, 6), W, beta=beta, factor=mfac, consts=consts, mode=self.mode)
                # logging split (no gradient of its own: `both` carries it)
                parts["margin_loss"] = mloss.mean().float()
                parts["margin_pde_loss"] = mterms.sum(dim=1).mean().float()
                parts["margin_terms"] = mterms
                total = tot + both
            else:
                mt, mterms = Fn.pde_residual(batch["margin_x"], batch["margin_y"], batch["margin_t"], batch["margin_f"],
                                             batch["margin_input_data"], W, consts=consts, mode=self.mode)
                parts["margin_pde_loss"], parts["margin_terms"] = mt, mterms
                total = total + tot + mt
        return total, parts

    @torch.no_grad()
    def predict_grid(self, field_data, coarse, forecast_h, time_ids, dt=3600.0, weights=None):
        """Dense-grid continuous-time forward (the working inference of the reference, interface_physics.py:538-606):
        every node of the lat_size x lon_size grid at each lead time `time_ids[i] * dt`, x-major node order (:541-545),
        coord_data from the coarse field by the on-GPU trilinear sampler (dataset.get_margin_grid :528-588), values only,
        inverse_norm WITHOUT clip (:533).  Returns physical fields [len(time_ids), lat_size, lon_size, 6]."""
        dev = field_data.device
        Hh, Ww = int(self.lat_size), int(self.lon_size)
        # the generated weights depend on (field_data, forecast_h) only: a lead-time sweep over one encoded field passes the
        # DecoderWeights of its first call back in (`weights=`) and skips encoder + hyper-network (SURVEY 8(f) N4)
        W = weights if weights is not None else self.physics_net.decoder_weights(field_data[:1], forecast_h[:1])
        xs, ys = torch.meshgrid(torch.arange(Ww, device=dev, dtype=torch.float32),
                                torch.arange(Hh, device=dev, dtype=torch.float32), indexing="ij")
        x = (xs.reshape(1, -1) * self.dx).repeat(1, len(time_ids))
        y = (ys.reshape(1, -1) * self.dy).repeat(1, len(time_ids))
        t = torch.tensor(list(time_ids), device=dev, dtype=torch.float32).repeat_interleave(Hh * Ww).reshape(1, -1) * dt
        consts = self.consts(self._last_factor())
        cd, _ = Fn.sample_field(coarse[:1], x, y, t, consts=consts, want_coriolis=False)
        o = Fn.decoder_values(None, cd, W, xyz=(x, y, t), consts=consts, mode=self.mode)[0]      # [T*W*H, 6]
        mean = torch.tensor(consts.mean, device=dev, dtype=o.dtype)
        std = torch.tensor(consts.std, device=dev, dtype=o.dtype)
        phys = o * std + mean
        return phys.reshape(len(time_ids), Ww, Hh, 6).permute(0, 2, 1, 3).contiguous()

    @torch.no_grad()
    def predict_lattice(self, field_data, coarse, forecast_h, lattice, weights=None):
        """Lattice inference for B samples at once: physical fields [B, nt, ny, nx, 6] of every sample on `lattice`
        (functional.Lattice; Lattice.domain(self.consts(...), refine, ...) covers the whole grid at `refine` times the training
        spacing), coord_data from its own coarse stack coarse[b] [Tt,Hc,Wc,6], inverse_norm without clip as predict_grid.
        The encoder and hyper-network run once for all samples (or not at all with cached `weights`), then one library call
        evaluates every node; the workspace holds a values-only pass (dpn_lattice_workspace_bytes)."""
        W = weights if weights is not None else self.physics_net.decoder_weights(field_data, forecast_h)
        return Fn.decoder_lattice(coarse, W, lattice, consts=self.consts(self._last_factor()), mode=self.mode)
