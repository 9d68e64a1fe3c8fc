"""
Synthetic "brain-MRI-shaped" image pairs (SURVEY.md §8d) with the dict layout of the reference's data loader
(`data_loader/datasets.py:117,128,135` in the reference: ``{'im': f32 (1,1,D,H,W), 'mask': bool, 'seg': int16}`` plus
the variational parameters ``{'mu','log_var','u'}`` of `datasets.py:57-68`).

This is the stand-in for the reference's BiobankDataset (file I/O through SimpleITK, out of scope).  It runs on the host
like the reference's loader does; it is not on the SGLD hot path.
"""
import math

import torch
import torch.nn.functional as F

# label IDs of the 15 structures the reference evaluates (parse_config.py:54-58 in the reference)
STRUCTURE_LABELS = (10, 11, 12, 13, 16, 17, 18, 26, 49, 50, 51, 52, 53, 54, 58)


def _gauss_1d(sigma):
    r = max(1, int(math.ceil(3.0 * sigma)))
    x = torch.arange(-r, r + 1, dtype=torch.float32)
    k = torch.exp(-0.5 * (x / sigma) ** 2)
    return k / k.sum(), r


def _smooth(vol, sigma):
    """separable Gaussian low-pass of a (N,C,D,H,W) tensor, replicate boundary"""
    k, r = _gauss_1d(sigma)
    k = k.to(vol.device)
    C = vol.shape[1]
    for axis in (2, 3, 4):
        shape = [1, 1, 1, 1, 1]
        shape[axis] = -1
        w = k.view(shape).repeat(C, 1, 1, 1, 1)
        pad = [0, 0, 0, 0, 0, 0]
        pad[2 * (4 - axis)] = pad[2 * (4 - axis) + 1] = r
        vol = F.conv3d(F.pad(vol, pad, mode='replicate'), w, groups=C)
    return vol


def _ellipsoid(n, centre, semi_axes, device=None):
    ax = torch.linspace(-1.0, 1.0, n).to(device or 'cpu')
    z, y, x = torch.meshgrid(ax, ax, ax, indexing='ij')
    cz, cy, cx = centre
    az, ay, ax_ = semi_axes
    return ((z - cz) / az) ** 2 + ((y - cy) / ay) ** 2 + ((x - cx) / ax_) ** 2 <= 1.0


def _identity_grid(n, device=None):
    ax = torch.linspace(-1.0, 1.0, n).to(device or 'cpu')
    z, y, x = torch.meshgrid(ax, ax, ax, indexing='ij')
    return torch.stack((x, y, z), -1).unsqueeze(0)  # (1,D,H,W,3), last dim (x,y,z) as F.grid_sample expects


def _exp_velocity(v, no_steps=6):
    """scaling and squaring of a voxel-unit velocity (1,3,n,n,n); returns the normalised sampling grid"""
    n = v.shape[-1]
    d = v * (2.0 / (n - 1)) / float(2 ** no_steps)
    grid = _identity_grid(n, v.device)
    for _ in range(no_steps):
        d = d + F.grid_sample(d, grid + d.permute(0, 2, 3, 4, 1), padding_mode='border', align_corners=True)
    return grid + d.permute(0, 2, 3, 4, 1)


def _texture_and_velocity(n, seed, max_velocity, dev):
    """the generator of make_pair after its first two draws, the smoothed texture noise and the velocity (1,3,n,n,n) in voxels
    with max |v| = max_velocity: the draws of make_pair in its order (the texture first), so that make_landmarks replays the
    same velocity"""
    g = torch.Generator().manual_seed(seed)
    texture = _smooth(torch.randn(1, 1, n, n, n, generator=g).to(dev), n / 32.0)
    v = _smooth(torch.randn(1, 3, n, n, n, generator=g).to(dev), n / 16.0)
    return g, texture, v * (max_velocity / v.abs().max())


def make_pair(n, seed=123, max_velocity=3.0, noise_std=0.02, sigma_v_init=0.5, u_v_init=0.1, device=None):
    """
    returns (fixed, moving, var_params_q_v) on the host, deterministic in (n, seed)
    `device`: where the filtering / resampling of the generator runs (the random numbers always come from the host
    generator; a 256^3 pair takes ~25 s of host convolutions, a second on a GPU); the result is returned on the host

    fixed['im']:  ellipsoidal head, three nested smooth ellipsoids (0.35/0.6/0.85) + low-pass texture + noise, in [0,1]
    moving['im']: fixed warped by exp(v) of a smooth random velocity with max |v| = max_velocity voxels + fresh noise
    mask:         head ellipsoid (about 29 % of the cube);  seg: 15 small labelled ellipsoids, int16
    """
    dev = device or 'cpu'
    g, texture, v = _texture_and_velocity(n, seed, max_velocity, dev)
    E = lambda c, a: _ellipsoid(n, c, a, dev)
    head = E((0.0, 0.0, 0.0), (0.74, 0.92, 0.80))

    im = torch.zeros(n, n, n, device=dev)
    for val, sc in ((0.35, 1.0), (0.6, 0.72), (0.85, 0.4)):
        im = torch.where(E((0.0, 0.02, -0.03), (0.74 * sc, 0.92 * sc, 0.80 * sc)), torch.tensor(val, device=dev), im)
    im = _smooth(im.view(1, 1, n, n, n), max(0.5, n / 64.0))

    texture = 0.08 * texture / texture.abs().max()
    clean = (im + texture) * head

    def finish(vol):
        vol = vol + noise_std * torch.randn(vol.shape, generator=g).to(dev) * head
        lo, hi = vol.min(), vol.max()
        return ((vol - lo) / (hi - lo)).contiguous().cpu()

    seg = torch.zeros(n, n, n, dtype=torch.int16, device=dev)
    for i, label in enumerate(STRUCTURE_LABELS):
        ang = 2.0 * math.pi * i / len(STRUCTURE_LABELS)
        c = (0.25 * math.sin(2.0 * ang), 0.45 * math.sin(ang), 0.4 * math.cos(ang))
        seg[E(c, (0.09, 0.11, 0.10))] = label

    grid = _exp_velocity(v)

    moving_clean = F.grid_sample(clean, grid, mode='bilinear', padding_mode='border', align_corners=True)
    moving_mask = F.grid_sample(head.float().view(1, 1, n, n, n), grid, mode='nearest', padding_mode='border',
                                align_corners=True).bool()
    moving_seg = F.grid_sample(seg.float().view(1, 1, n, n, n), grid, mode='nearest', padding_mode='border',
                               align_corners=True).short()

    fixed = {'im': finish(clean), 'mask': head.view(1, 1, n, n, n).contiguous().cpu(), 'seg': seg.view(1, 1, n, n, n).cpu()}
    moving = {'im': finish(moving_clean), 'mask': moving_mask.cpu(), 'seg': moving_seg.cpu()}

    dims_v = (1, 3, n, n, n)
    var_params_q_v = {'mu': torch.zeros(dims_v), 'log_var': torch.full(dims_v, math.log(sigma_v_init ** 2)),
                      'u': torch.full(dims_v, u_v_init)}
    return fixed, moving, var_params_q_v


def make_landmarks(n, seed=123, max_velocity=3.0, no_landmarks=300, device=None):
    """
    Corresponding landmarks of make_pair(n, seed, max_velocity): (fixed_landmarks, moving_landmarks), (P,3) float64 host
    tensors of zero-based (x, y, z) voxel coordinates, P = no_landmarks, row i of one corresponding to row i of the other.

    make_pair builds moving = fixed o phi with phi = exp(v) (voxel units here).  The moving landmarks q are moving-mask voxels
    drawn with a generator of their own (make_pair's draws are unchanged), kept where phi(q) lies in [1, n - 2] on every
    axis; the fixed landmarks are p = phi(q) from the same sampling grid, so the fixed image at p shows what the moving image
    shows at q.  A registration of the pair estimates T ~ phi^-1, which carries p back to q: the TRE of the true
    transformation is 0 up to the grid's rounding.  ValueError when fewer than no_landmarks voxels qualify.
    """
    dev = device or 'cpu'
    _, _, v = _texture_and_velocity(n, seed, max_velocity, dev)
    grid = _exp_velocity(v)                                               # (1,D,H,W,3) normalised (x, y, z)
    phi = (grid[0].double() + 1.0) * ((n - 1) / 2.0)                      # fixed voxel coordinates (x, y, z)
    head = _ellipsoid(n, (0.0, 0.0, 0.0), (0.74, 0.92, 0.80), dev)
    moving_mask = F.grid_sample(head.float().view(1, 1, n, n, n), grid, mode='nearest', padding_mode='border',
                                align_corners=True).bool()[0, 0]          # make_pair's moving['mask']
    ok = moving_mask & ((phi >= 1.0) & (phi <= n - 2.0)).all(-1)
    idx = torch.nonzero(ok.flatten().cpu()).flatten()
    if idx.numel() < no_landmarks:
        raise ValueError(f'only {idx.numel()} moving-mask voxels map inside [1, n - 2]: fewer than {no_landmarks} landmarks')
    g = torch.Generator().manual_seed(seed + 1)
    pick = idx[torch.randperm(idx.numel(), generator=g)[:no_landmarks]]
    z, y, x = pick // (n * n), (pick // n) % n, pick % n
    q = torch.stack((x, y, z), -1).double()
    p = phi.cpu().reshape(-1, 3)[pick]
    return p.contiguous(), q.contiguous()
