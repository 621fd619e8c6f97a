"""TEST INFRASTRUCTURE — NOT PRODUCT CODE.

Plain-PyTorch restatement of the reference's SSIM (utils/loss_utils.py: gaussian, create_window, ssim, _ssim — the 3DGS
formulation), operator for operator, parameterised on dtype so that tests can run it in float64:
  * gaussian / create_window: the 1-D taps come from Python floats rounded to float32 and normalised in float32, the
    2-D window is their float32 outer product; the window is then cast to the images' dtype (`window.type_as(img1)`)
  * ssim: five grouped conv2d with zero padding (window_size // 2), C1 = 0.01**2, C2 = 0.03**2;
    size_average=True -> map.mean(), False -> one value per image (map.mean(1).mean(1).mean(1))
Pinned: tests/test_ssim_parity.py checks it against scipy.ndimage.correlate and an explicit 2-D loop, and its gradient with
torch.autograd.gradcheck.
"""
from math import exp

import torch
import torch.nn.functional as F


def gaussian(window_size, sigma):
    gauss = torch.tensor([exp(-(x - window_size // 2) ** 2 / float(2 * sigma ** 2)) for x in range(window_size)], dtype=torch.float32)
    return gauss / gauss.sum()


def create_window(window_size, channel):
    g = gaussian(window_size, 1.5).unsqueeze(1)
    return g.mm(g.t()).float().unsqueeze(0).unsqueeze(0).expand(channel, 1, window_size, window_size).contiguous()


def ssim_map(img1, img2, window_size=11):
    """The SSIM map, same shape as the inputs ([N,C,H,W] or [C,H,W]), in the inputs' dtype."""
    channel = img1.size(-3)
    window = create_window(window_size, channel).to(img1.device).type_as(img1)
    pad = window_size // 2
    mu1 = F.conv2d(img1, window, padding=pad, groups=channel)
    mu2 = F.conv2d(img2, window, padding=pad, groups=channel)
    mu1_sq, mu2_sq, mu1_mu2 = mu1.pow(2), mu2.pow(2), mu1 * mu2
    sigma1_sq = F.conv2d(img1 * img1, window, padding=pad, groups=channel) - mu1_sq
    sigma2_sq = F.conv2d(img2 * img2, window, padding=pad, groups=channel) - mu2_sq
    sigma12 = F.conv2d(img1 * img2, window, padding=pad, groups=channel) - mu1_mu2
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    return ((2 * mu1_mu2 + C1) * (2 * sigma12 + C2)) / ((mu1_sq + mu2_sq + C1) * (sigma1_sq + sigma2_sq + C2))


def ssim(img1, img2, window_size=11, size_average=True):
    m = ssim_map(img1, img2, window_size)
    return m.mean() if size_average else m.mean(1).mean(1).mean(1)


def ssim_and_grad(img1, img2, dtype=torch.float64):
    """(per-image SSIM [N], d(sum of the whole map)/d img1) of [N,C,H,W] inputs, evaluated in `dtype` on the inputs' device."""
    x = img1.detach().to(dtype).requires_grad_(True)
    m = ssim_map(x, img2.detach().to(dtype))
    m.sum().backward()
    return m.mean(dim=(1, 2, 3)).detach(), x.grad.detach()
