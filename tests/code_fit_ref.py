"""fp64 statement of the frame-code gradient of code fitting (danbo_ray_bias_codes_bwd), shared by the CPU and GPU
tests: the view layer's per-ray bias is W_v[:, 256:283] PE(d) + W_v[:, 283:411] code[row(cam)] + b_v, so
d code[c] = sum over the rays whose cam maps to row c of W_v[:, 283:411]^T d ray_bias.  Row rule of danbo_ray_bias:
cam < 0 reads the mean code (no gradient to the table), cam > rows - 1 reads the last row."""
import torch


def code_rows(cam, n_codes):
    """cam (n,) -> the fitted row each ray reads, -1 for the mean code."""
    cam = cam.long()
    return torch.where(cam < 0, torch.full_like(cam, -1), cam.clamp(max=n_codes - 1))


def codes_grad_fp64(cam, w_view, d_ray_bias, n_codes):
    """Scatter-add of d_ray_bias @ W_v[:, 283:411] over the rows the rays read -> (n_codes,128) fp64."""
    rows = code_rows(cam.cpu(), n_codes)
    per_ray = d_ray_bias.detach().cpu().double() @ w_view.detach().cpu().double()[:, 283:411]
    keep = rows >= 0
    out = torch.zeros(n_codes, 128, dtype=torch.float64)
    return out.index_add_(0, rows[keep], per_ray[keep])


def view_encoding(d):
    """The 27 view columns danbo_ray_bias encodes from a direction d (n,3): d, then sin / cos of 2^f d, f < 4."""
    parts = [d]
    for f in range(4):
        parts += [torch.sin(d * 2. ** f), torch.cos(d * 2. ** f)]
    return torch.cat(parts, -1)


def folded_view_bias(dirs, cam, w_view, b_view, codes, mean_code):
    """The per-ray bias of the folded view layer, as torch ops (differentiable in codes): table = [codes; mean]."""
    table = torch.cat([codes, mean_code[None]], 0)
    idx = code_rows(cam, codes.shape[0])
    idx = torch.where(idx < 0, torch.full_like(idx, codes.shape[0]), idx)
    return view_encoding(dirs) @ w_view[:, 256:283].t() + table[idx] @ w_view[:, 283:411].t() + b_view
