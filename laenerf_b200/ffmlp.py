"""Drop-in for the reference's `ffmlp` package (ffmlp/ffmlp.py:15-168) on liblaenerf_b200.so (tcgen05 kernels).

Same `FFMLP(input_dim, output_dim, hidden_dim, num_layers, activation)` module, same flat fp32 `weights` parameter
(layout ffmlp.py:121: [hidden,in] + (num_layers-1) x [hidden,hidden] + [16,hidden]), same seed-42 initialisation,
same "always pad the batch to the next multiple of 128" rule and `custom_fwd(cast_inputs=half)` AMP contract.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
from torch.autograd import Function
from torch.amp import custom_bwd, custom_fwd

from . import _native as N


class _ffmlp_forward(Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.half)
    def forward(ctx, inputs, weights, input_dim, output_dim, hidden_dim, num_layers, activation, output_activation,
                inference=False, calc_grad_inputs=False):
        B = inputs.shape[0]
        inputs = inputs.contiguous().half()  # outside autocast the reference would fail CHECK_IS_HALF; be lenient
        weights = weights.contiguous().half()
        outputs = torch.empty(B, output_dim, device=inputs.device, dtype=inputs.dtype)
        lib = N.lib()
        if not inference:
            forward_buffer = torch.empty(num_layers, B, hidden_dim, device=inputs.device, dtype=inputs.dtype)
            N.check(lib.lnrf_ffmlp_forward(N.ptr(inputs), N.ptr(weights), B, input_dim, output_dim, hidden_dim, num_layers,
                                           activation, output_activation, N.ptr(forward_buffer), N.ptr(outputs), N.stream()))
            ctx.save_for_backward(inputs, weights, outputs, forward_buffer)
            ctx.dims = (input_dim, output_dim, hidden_dim, num_layers, activation, output_activation, calc_grad_inputs)
        else:
            N.check(lib.lnrf_ffmlp_inference(N.ptr(inputs), N.ptr(weights), B, input_dim, output_dim, hidden_dim, num_layers,
                                             activation, output_activation, None, N.ptr(outputs), N.stream()))
        return outputs

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, grad):
        B = grad.shape[0]
        grad = grad.contiguous().half()
        inputs, weights, outputs, forward_buffer = ctx.saved_tensors
        input_dim, output_dim, hidden_dim, num_layers, activation, output_activation, calc_grad_inputs = ctx.dims
        lib = N.lib()
        if torch.are_deterministic_algorithms_enabled() and not backward_deterministic(input_dim, output_dim, hidden_dim, num_layers,
                                                                                      activation, output_activation):
            N.alert_not_deterministic(f"FFMLP backward of a {input_dim}-{hidden_dim}x{num_layers}-{output_dim} net with activation "
                                      f"{activation} (lnrf_ffmlp_backward, float-atomics weight gradient)")
        grad_inputs = torch.empty_like(inputs) if calc_grad_inputs else None
        grad_weights = torch.empty_like(weights)
        nbytes = lib.lnrf_ffmlp_wgrad_scratch_bytes(input_dim, output_dim, hidden_dim, num_layers)
        scratch = torch.empty(nbytes // 4, dtype=torch.float32, device=grad.device)
        N.check(lib.lnrf_ffmlp_backward(N.ptr(grad), N.ptr(inputs), N.ptr(weights), N.ptr(forward_buffer), B, input_dim,
                                        output_dim, hidden_dim, num_layers, activation, output_activation,
                                        int(bool(calc_grad_inputs)), None, N.ptr(grad_inputs), N.ptr(grad_weights),
                                        N.ptr(scratch), nbytes, N.stream()))
        return grad_inputs, grad_weights, None, None, None, None, None, None, None, None


ffmlp_forward = _ffmlp_forward.apply


def backward_deterministic(input_dim, output_dim, hidden_dim, num_layers, activation, output_activation=6) -> bool:
    """Whether lnrf_ffmlp_backward sums this net's weight gradient in a fixed order (the two-tile ReLU kernel) rather than with
    float atomics."""
    r = N.lib().lnrf_ffmlp_backward_deterministic(input_dim, output_dim, hidden_dim, num_layers, activation, output_activation)
    N.check(min(r, 0))
    return r == 1


def convert_activation(act):  # ffmlp.py:89-96
    return {"relu": 0, "exponential": 1, "sine": 2, "sigmoid": 3, "squareplus": 4, "softplus": 5}.get(act, 6)


class FFMLP(nn.Module):
    def __init__(self, input_dim, output_dim, hidden_dim, num_layers, activation="relu"):
        super().__init__()
        self.input_dim = input_dim
        self.output_dim = output_dim
        self.hidden_dim = hidden_dim
        self.num_layers = num_layers
        self.activation = convert_activation(activation)
        self.output_activation = convert_activation("none")
        self.tensorcore_width = 16
        assert hidden_dim in [16, 32, 64, 128, 256], f"FFMLP only support hidden_dim in [16, 32, 64, 128, 256], but got {hidden_dim}"
        assert input_dim > 0 and input_dim % 16 == 0, f"FFMLP input_dim should be 16 * m (m  > 0), but got {input_dim}"
        assert output_dim <= 16, f"FFMLP current only supports output dim <= 16, but got {output_dim}"
        assert num_layers >= 2, f"FFMLP num_layers should be larger than 2 (3 matmuls), but got {num_layers}"
        self.padded_output_dim = int(math.ceil(output_dim / 16)) * 16
        self.num_parameters = hidden_dim * (input_dim + hidden_dim * (num_layers - 1) + self.padded_output_dim)
        self.weights = nn.Parameter(torch.zeros(self.num_parameters))
        self.reset_parameters()
        N.check(N.lib().lnrf_allocate_splitk(self.num_layers + 1))  # no-op here; kept for binding parity (ffmlp.py:126)

    def cleanup(self):
        N.check(N.lib().lnrf_free_splitk())

    def __repr__(self):
        return (f"FFMLP: input_dim={self.input_dim} output_dim={self.output_dim} hidden_dim={self.hidden_dim} "
                f"num_layers={self.num_layers} activation={self.activation}")

    def reset_parameters(self):
        torch.manual_seed(42)  # the reference reseeds the global RNG here (ffmlp.py:142); kept because it is observable
        std = math.sqrt(3 / self.hidden_dim)
        self.weights.data.uniform_(-std, std)

    def forward(self, inputs):
        B, C = inputs.shape
        pad = 128 - (B % 128)  # ffmlp.py:157: always > 0, a full 128 rows when B is already aligned
        if pad > 0:
            inputs = torch.cat([inputs, torch.zeros(pad, C, dtype=inputs.dtype, device=inputs.device)], dim=0)
        outputs = ffmlp_forward(inputs, self.weights, self.input_dim, self.padded_output_dim, self.hidden_dim, self.num_layers,
                                self.activation, self.output_activation, not self.training, inputs.requires_grad)
        if B != outputs.shape[0] or self.padded_output_dim != self.output_dim:
            outputs = outputs[:B, :self.output_dim]
        return outputs
