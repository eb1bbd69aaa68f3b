"""PSFNet network container (mirror of the reference's deeplens/psfnet_arch.py:24-47, 251-264).

``MLP`` only *holds* the parameters, under the same ``net.{0,2,4,...}`` state_dict keys as the
reference so checkpoints round-trip; evaluating it goes to the CUDA library.  There is no
PyTorch forward path here on purpose.  Under autograd (grad mode on, and the input or a parameter
requiring grad) the evaluation is differentiable in the input and the parameters, with backward
kernels of the same library.
"""
import torch
import torch.nn as nn


def initialize_weights(m):
    """Reference initialiser for Linear layers: kaiming-uniform weights, zero bias
    (psfnet_arch.py:251-264; the other branches there concern layer types PSFNet never builds)."""
    if isinstance(m, nn.Linear):
        nn.init.kaiming_uniform_(m.weight.data)
        nn.init.constant_(m.bias.data, 0)


class MLP(nn.Module):
    """in -> hidden/4 -> hidden -> (hidden x hidden_layers) -> out, ReLU between, Sigmoid head,
    L1-normalised output.  Same constructor signature and parameter names as the reference."""

    def __init__(self, in_features, out_features, hidden_features=64, hidden_layers=3):
        super().__init__()
        widths = [in_features, hidden_features // 4, hidden_features] + [hidden_features] * hidden_layers
        mods = []
        for a, b in zip(widths[:-1], widths[1:]):
            mods += [nn.Linear(a, b, bias=True), nn.ReLU(inplace=True)]
        mods += [nn.Linear(widths[-1], out_features, bias=True), nn.Sigmoid()]
        self.net = nn.Sequential(*mods)
        self.net.apply(initialize_weights)
        self._evaluator = None      # set by PSFNet: callable([..., in]) -> [..., out] on the GPU

    def linear_layers(self):
        return [m for m in self.net if isinstance(m, nn.Linear)]

    def forward(self, x):
        if self._evaluator is None:
            raise RuntimeError("MLP has no CUDA evaluator attached; use PSFNet.pred / PSFNet.render "
                               "(this build has no PyTorch-eager forward path)")
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            return self._evaluator(x, layers=self.linear_layers())
        return self._evaluator(x)
