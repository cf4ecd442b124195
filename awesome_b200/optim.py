"""Drop-in optimizers for ``AwesomeConfig.optimizer_type`` (``awesome/run/awesome_runner.py:263-267``;
created at ``awesome/agent/torch_agent.py:833-834``): ``torch.optim.Adam`` / ``Adamax`` semantics, with every
parameter that lives in a prior module's arena updated by ONE native pass (``awb_optim_step``: moments, bias
correction, L2, update and the ``enforce_convexity`` clamp, SURVEY K10 + K11) instead of per-tensor foreach
kernels plus one clamp launch per tensor.  Parameters outside a prior arena (the segmentation UNet in joint
training) are delegated to the stock torch optimizer of the same kind, so a mixed ``WrapperModule`` works."""
from __future__ import annotations

import ctypes as C
import weakref
from typing import Dict, List, Optional

import torch

from . import _lib as L

_ARENA_MODULES: "weakref.WeakSet" = weakref.WeakSet()     # filled by ArenaPriorModule.__init__


def _owner_of(p: torch.Tensor):
    """The registered prior module whose arena storage holds ``p`` (or None)."""
    try:
        sp = p.untyped_storage().data_ptr()
    except Exception:
        return None
    for m in list(_ARENA_MODULES):
        a = getattr(m, "_arena", None)
        if a is None or a.device != p.device:
            continue
        if a.untyped_storage().data_ptr() == sp and a.data_ptr() <= p.data_ptr() < a.data_ptr() + 4 * a.numel():
            # prefer the outermost module (a PathConnectedNet owns its ConvexNextNet's parameters)
            best = m
            for m2 in list(_ARENA_MODULES):
                a2 = getattr(m2, "_arena", None)
                if a2 is not None and a2.device == p.device and a2.untyped_storage().data_ptr() == sp \
                        and a2.data_ptr() <= a.data_ptr() and a2.numel() > best._arena.numel() \
                        and a2.data_ptr() + 4 * a2.numel() >= a.data_ptr() + 4 * a.numel():
                    best = m2
            return best
    return None


class _FusedBase(torch.optim.Optimizer):
    _kind = "adam"

    def __init__(self, params, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0,
                 **kwargs):
        if lr < 0 or eps < 0 or weight_decay < 0:
            raise ValueError("lr, eps and weight_decay must be non-negative")
        defaults = dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay)
        super().__init__(params, defaults)
        self._plan = None
        self._inner: Optional[torch.optim.Optimizer] = None

    # ---- planning: which parameters are covered by a native arena pass
    def _build_plan(self) -> None:
        by_mod: Dict[int, dict] = {}
        rest: List[dict] = []
        for gi, group in enumerate(self.param_groups):
            others = []
            for p in group["params"]:
                m = _owner_of(p) if p.is_cuda else None
                if m is None:
                    others.append(p)
                else:
                    by_mod.setdefault(id(m), {"module": m, "params": {}})["params"][id(p)] = (p, gi)
            if others:
                rest.append({"params": others, "group": gi})
        native = []
        for ent in by_mod.values():
            m = ent["module"]
            aparams = m._arena_params()
            ok = all(id(p) in ent["params"] for p in aparams)
            if ok:
                # per native group (0 flow_net, 1 convex_net, 2 linear): hyper-parameters must be uniform
                gid = m._optimizer_group_ids()
                hyper = {}
                for p, g in zip(aparams, gid):
                    grp = self.param_groups[ent["params"][id(p)][1]]
                    key = (grp["betas"], grp["eps"])
                    cur = hyper.setdefault(g, {"gi": ent["params"][id(p)][1], "key": key})
                    if cur["key"] != key or (self.param_groups[cur["gi"]]["weight_decay"] != grp["weight_decay"]):
                        ok = False
                if ok and len({h["key"] for h in hyper.values()}) > 1:
                    ok = False
                if ok:
                    native.append({"module": m, "hyper": hyper, "state": None})
            if not ok:
                for p, gi in ent["params"].values():
                    rest.append({"params": [p], "group": gi})
        self._plan = {"native": native, "rest": rest}
        if rest:
            cls = torch.optim.Adam if self._kind == "adam" else torch.optim.Adamax
            groups = []
            for r in rest:
                g = self.param_groups[r["group"]]
                groups.append(dict(params=r["params"], lr=g["lr"], betas=g["betas"], eps=g["eps"],
                                   weight_decay=g["weight_decay"], _src=r["group"]))
            self._inner = cls(groups)

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        if self._plan is None:
            self._build_plan()
        for ent in self._plan["native"]:
            m = ent["module"]
            arena = m._ensure_flat()
            prior = m._prior_for(arena.device)
            aparams = m._arena_params()
            active = self._active_groups(m, aparams)
            if active is None:
                continue
            grads = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1).float()
                               for p in aparams])
            lrs = [0.0] * L.AWB_MAX_GROUPS
            wds = [0.0] * L.AWB_MAX_GROUPS
            betas, eps = (0.9, 0.999), 1e-8
            for g, h in ent["hyper"].items():
                grp = self.param_groups[h["gi"]]
                lrs[g], wds[g] = float(grp["lr"]), float(grp["weight_decay"])
                betas, eps = grp["betas"], grp["eps"]
            with torch.cuda.device(arena.device):
                lr_c = (C.c_double * L.AWB_MAX_GROUPS)(*lrs)
                if ent["state"] is None:
                    ent["state"] = torch.empty(prior.opt_state_bytes(), dtype=torch.uint8, device=arena.device)
                    L.check(prior.lib.awb_opt_state_init(prior.handle, ent["state"].data_ptr(), lr_c, L.stream_ptr()))
                else:
                    L.check(prior.lib.awb_opt_set_lr(prior.handle, ent["state"].data_ptr(), lr_c, L.stream_ptr()))
                kind = L.AWB_OPT_ADAM if self._kind == "adam" else L.AWB_OPT_ADAMAX
                hy = L.OptHyper(kind, betas[0], betas[1], eps, (C.c_float * L.AWB_MAX_GROUPS)(*wds), 0, 0, 0.0, 0.0,
                                0.0, 0.0, active)
                L.check(prior.lib.awb_optim_step(prior.handle, arena.data_ptr(), grads.data_ptr(),
                                                 ent["state"].data_ptr(), C.byref(hy), L.stream_ptr()))
        if self._inner is not None:
            for g in self._inner.param_groups:
                g["lr"] = self.param_groups[g["_src"]]["lr"]
            self._inner.step()
        return loss

    @staticmethod
    def _active_groups(m, aparams) -> Optional[int]:
        """``active_groups`` mask of one native step, like torch, which skips a parameter whose ``.grad`` is None (its
        moments, weight decay and step count stay put): 0 when every native group has grads, the groups that have them
        otherwise, None when none has.  A group is stepped as a whole, so one with only some grads raises."""
        gids = m._optimizer_group_ids()
        has: Dict[int, List[bool]] = {}
        for p, g in zip(aparams, gids):
            has.setdefault(g, []).append(p.grad is not None)
        for p, g in zip(aparams, gids):
            if p.grad is None and any(has[g]):
                name = next(n for n, q in m.named_parameters() if q is p)
                raise ValueError(f"{type(m).__name__}.{name} has no grad while other parameters of its optimizer group "
                                 f"{g} do; the fused step updates a group as a whole")
        on = [g for g, h in has.items() if h[0]]
        if not on:
            return None
        return 0 if len(on) == len(has) else sum(1 << g for g in on)

    def add_param_group(self, param_group):
        super().add_param_group(param_group)
        self._plan = None
        self._inner = None

    # ---- checkpointing: the agent saves ``optimizer.state_dict()`` (torch_agent.py:1009) and, with keep_device=False,
    # frees and recreates the optimizer around every best-model save (``_free_optimizer`` / ``_get_optimizer`` +
    # ``load_state_dict``, torch_agent.py:356, 808, 836).  The moments live outside ``self.state`` (stock optimizer of the
    # non-arena parameters, native blob per arena module), so both are carried in an extra key.
    def _flat_index(self) -> Dict[int, int]:
        out, i = {}, 0
        for g in self.param_groups:
            for p in g["params"]:
                out[id(p)] = i
                i += 1
        return out

    def state_dict(self):
        sd = super().state_dict()
        extra = {"kind": self._kind, "inner": None, "native": []}
        if self._plan is not None:
            idx = self._flat_index()
            if self._inner is not None:
                import copy
                extra["inner"] = copy.deepcopy(self._inner.state_dict())     # a snapshot, like the native blob below
            for ent in self._plan["native"]:
                first = ent["module"]._arena_params()[0]
                blob = ent["state"].detach().cpu().clone() if ent["state"] is not None else None
                extra["native"].append({"first_param": idx[id(first)], "n_params": len(ent["module"]._arena_params()),
                                        "blob": blob})
        sd["awb_fused"] = extra
        return sd

    def load_state_dict(self, state_dict):
        extra = state_dict.get("awb_fused") if isinstance(state_dict, dict) else None
        super().load_state_dict({k: v for k, v in state_dict.items() if k != "awb_fused"})
        self._plan, self._inner = None, None
        if not extra:
            return
        if extra.get("kind") != self._kind:
            raise ValueError(f"optimizer state of kind {extra.get('kind')!r} loaded into {self._kind!r}")
        self._build_plan()
        if extra.get("inner") is not None:
            if self._inner is None:
                raise ValueError("saved state holds non-arena parameters, this optimizer has none")
            self._inner.load_state_dict(extra["inner"])
        idx = self._flat_index()
        saved = {e["first_param"]: e for e in extra.get("native", [])}
        for ent in self._plan["native"]:
            m = ent["module"]
            e = saved.get(idx[id(m._arena_params()[0])])
            if e is None or e["blob"] is None:
                continue
            arena = m._ensure_flat()
            prior = m._prior_for(arena.device)
            if e["blob"].numel() != prior.opt_state_bytes() or e["n_params"] != len(m._arena_params()):
                raise ValueError("saved native optimizer state does not match this prior's layout")
            ent["state"] = e["blob"].to(arena.device).clone()


class FusedAdam(_FusedBase):
    """``torch.optim.Adam`` (single-tensor arithmetic) + fused non-negativity clamp for prior arenas."""
    _kind = "adam"


class FusedAdamax(_FusedBase):
    """``torch.optim.Adamax`` + fused clamp (``betas`` / ``eps`` defaults as torch: (0.9, 0.999), 1e-8)."""
    _kind = "adamax"

    def __init__(self, params, lr: float = 2e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0,
                 **kwargs):
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
