"""The optimiser step of the Gaussian parameters in one launch (SURVEY.md section 8f rank 2).

``FusedAdam`` is a ``torch.optim.Adam`` whose ``step()`` runs csrc/adam.cu through the C ABI (``ogs_adam_step``):
every parameter tensor of every group -- the seven groups ``GaussianModel.training_setup`` builds
(scene/gaussian_model.py:215-230: xyz, f_dc, f_rest, opacity, scaling, rotation, ins_feat) -- is updated by ONE
kernel, 28 B of HBM traffic per element.  Everything else is inherited, so the reference's code that edits the
optimiser keeps working unchanged: ``param_groups[i]["lr"]`` updates (``update_learning_rate``, :236-247),
``state[p]["exp_avg"] / ["exp_avg_sq"]`` surgery in ``replace_tensor_to_optimizer`` / ``_prune_optimizer`` /
``cat_tensors_to_optimizer`` (:357-425), ``state_dict`` / ``load_state_dict`` (:98, :120).

    self.optimizer = FusedAdam(l, lr=0.0, eps=1e-15)        # instead of torch.optim.Adam(l, lr=0.0, eps=1e-15)

Arithmetic: torch/optim/adam.py::_single_tensor_adam (torch 2.11) without weight decay / amsgrad / maximize;
those options raise.  Parameters whose ``.grad`` is None are skipped, exactly like torch (the reference freezes
``_xyz`` that way for ScanNet, :226-227).
"""
import ctypes as C

import torch

from . import _lib


class FusedAdam(torch.optim.Adam):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0, amsgrad=False):
        if weight_decay != 0 or amsgrad:
            raise NotImplementedError("FusedAdam: weight_decay / amsgrad are not used by OpenGaussian and not built")
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=0, amsgrad=False, foreach=False, fused=False)

    def _entries(self):
        """Bumps the step counters and returns (device, [AdamTensor fields + the tensors kept alive])."""
        per_device = {}
        for group in self.param_groups:
            if group.get("weight_decay", 0) != 0 or group.get("amsgrad", False) or group.get("maximize", False):
                raise NotImplementedError("FusedAdam: weight_decay / amsgrad / maximize are not built")
            beta1, beta2 = group["betas"]
            lr = float(group["lr"])
            eps = float(group["eps"])
            for p in group["params"]:
                if p.grad is None:
                    continue
                if not p.is_cuda:
                    raise _lib.OgsError("FusedAdam needs CUDA parameters (no CPU path)")
                if p.grad.is_sparse or p.dtype != torch.float32 or not p.is_contiguous():
                    raise _lib.OgsError("FusedAdam: parameters must be dense contiguous float32")
                state = self.state[p]
                if len(state) == 0:                       # torch/optim/adam.py::_init_group
                    state["step"] = torch.tensor(0.0, dtype=torch.float32)
                    state["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    state["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                state["step"] += 1
                step = float(state["step"])
                m, v = state["exp_avg"], state["exp_avg_sq"]
                if not (m.is_contiguous() and v.is_contiguous()):
                    m, v = m.contiguous(), v.contiguous()
                    state["exp_avg"], state["exp_avg_sq"] = m, v
                g = p.grad.detach()
                if g.dtype != torch.float32 or not g.is_contiguous():
                    g = g.float().contiguous()
                bias_correction1 = 1 - beta1 ** step
                bias_correction2 = 1 - beta2 ** step
                per_device.setdefault(p.device, []).append(
                    (p, g, m, v, lr / bias_correction1, bias_correction2 ** 0.5, beta1, beta2, eps))
        return per_device

    @torch.no_grad()
    def step(self, closure=None, grad_scale: float = 1.0):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        for dev, items in self._entries().items():
            arr = (_lib.AdamTensor * len(items))()
            for a, (p, g, m, v, step_size, bc2s, beta1, beta2, eps) in zip(arr, items):
                a.param, a.grad, a.exp_avg, a.exp_avg_sq = p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr()
                a.n = p.numel()
                a.step_size, a.bias_correction2_sqrt, a.beta1, a.beta2, a.eps = step_size, bc2s, beta1, beta2, eps
                a.one_minus_beta1, a.one_minus_beta2 = 1 - beta1, 1 - beta2
            _lib.launch("ogs_adam_step", dev, len(items), C.cast(arr, C.c_void_p), float(grad_scale))
        return loss
