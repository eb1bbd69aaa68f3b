"""Focus-distance selection (mirror of the reference's dff/utils.py:4-51).

Same results as the reference for mode='linear', but without its per-image Python loop and the
host synchronisation it implies: on CUDA tensors one kernel (one CTA per image) produces the [B, num]
focus distances; CPU tensors (host-side logic, tests) take the loop-free torch formulation below.
"""
import numpy as np
import torch

import aadff_native as _nat


def select_focus_dist(depth, num, mode='linear', center=True):
    """depth [B,1,H,W] (metres, 0 = invalid) -> focus distances [B,num], ascending."""
    assert num > 3, 'Focal stack size is too small'
    B = depth.shape[0]
    if depth.is_cuda and mode == 'linear' and depth.dtype == torch.float32:
        flat = depth.detach().reshape(B, -1).contiguous()
        out = torch.empty(B, num, device=depth.device, dtype=torch.float32)
        if B:
            _nat.call("aadff_select_focus_f32", flat.data_ptr(), B, flat.shape[1], num, out.data_ptr(),
                      device=depth.device)
        return out
    flat = depth.reshape(B, -1)
    valid = flat > 0
    depth_max = flat.amax(dim=1)
    depth_min = torch.where(valid, flat, torch.full_like(flat, float('inf'))).amin(dim=1)
    if mode == 'linear':
        steps = [depth_min + i * (depth_max - depth_min) / (num - 1) for i in range(num)]
    elif mode == 'importance':
        avg_depth = flat.sum(dim=1) / valid.sum(dim=1)
        steps = [depth_max, depth_min]
        num = num - 2
        while len(steps) < num:
            cand = np.random.rand() * (depth_max - depth_min) + depth_min
            if cand > avg_depth:
                rate = (depth_max - cand) / (depth_max - avg_depth)
            else:
                rate = (cand - depth_min) / (avg_depth - depth_min)
            if np.random.rand() < rate:
                steps.append(cand)
    else:
        raise NotImplementedError
    return torch.sort(torch.stack(steps, dim=1), dim=-1)[0]
