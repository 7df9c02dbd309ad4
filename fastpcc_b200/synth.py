"""Seeded synthetic inputs and parameters for the codec hot path (SURVEY.md 8d).

No datasets or trained checkpoints exist offline, so measurement and parity both run on:
  * `lidar_frame`  -- S2 "lidar-120k": a 64-beam spinning-LiDAR model voxelised with exactly the
    dataset transform of the reference (lib/datasets/KITTIOdometry/dataset.py:90-102).
  * `surface_cloud` -- S1/S3 style voxelised shell surfaces on a 2^bits grid.
  * `colored_surface` -- S4 style: a surface cloud with a smooth, noisy uint8 RGB field.
  * `make_lossl_int_state_dict` -- random int8 parameters for models/convolutional/lossl_coord_int,
    produced with the reference's own PTQ formulas (lib/int_sparse_conv/cuda_ops.py:223-301,
    487-503, 541-607) from seeded float weights and fixed activation scales, under the reference's
    state-dict key names.

Pure numpy; imported by the product's bench/tests and by the oracle's tests (never by oracle/ itself).
"""
import zlib

import numpy as np

SharedFxpShift = 23
WeightRange = 127


# ------------------------------------------------------------------------------------------------
# point clouds
# ------------------------------------------------------------------------------------------------

def lidar_points(seed: int, n_boxes: int = 40, azimuths: int = 2048, beams: int = 64):
    """One KITTI-shaped scan as the sensor delivers it: float32 [N,3] metres (the rows of a velodyne .bin)."""
    rng = np.random.default_rng(seed)
    elev = np.deg2rad(np.linspace(-24.8, 2.0, beams))
    azim = np.linspace(0, 2 * np.pi, azimuths, endpoint=False)
    el, az = np.meshgrid(elev, azim, indexing='ij')
    d = np.stack([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), np.sin(el)], -1).reshape(-1, 3)
    h = 1.73
    t = np.full(d.shape[0], np.inf)
    down = d[:, 2] < -1e-6
    t[down] = -h / d[down, 2]  # ground plane z = -h
    for _ in range(n_boxes):  # axis-aligned boxes standing on the ground
        c = np.array([rng.uniform(-60, 60), rng.uniform(-60, 60)])
        if np.hypot(*c) < 4:
            continue
        half = rng.uniform(0.5, 4.0, 2)
        top = rng.uniform(0.5, 4.0) - h
        lo = np.array([c[0] - half[0], c[1] - half[1], -h])
        hi = np.array([c[0] + half[0], c[1] + half[1], top])
        with np.errstate(divide='ignore', invalid='ignore'):
            t1, t2 = lo[None] / d, hi[None] / d
        tn = np.nanmax(np.minimum(t1, t2), 1)
        tf = np.nanmin(np.maximum(t1, t2), 1)
        hit = (tn <= tf) & (tn > 0)
        t = np.where(hit & (tn < t), tn, t)
    keep = np.isfinite(t) & (t < 120.0) & (rng.random(t.shape[0]) > 0.08)
    return (d[keep] * t[keep, None] * (1 + rng.normal(0, 0.002, (int(keep.sum()), 1)))).astype(np.float32)


def lidar_frame(seed: int, resolution: int = 65536, n_boxes: int = 40, azimuths: int = 2048, beams: int = 64):
    """One KITTI-shaped scan -> int32 [N,3] unique voxels (N ~ 115-125k at the defaults): the dataset transform of
    lib/datasets/KITTIOdometry/dataset.py:90-102 applied to `lidar_points`."""
    xyz = lidar_points(seed, n_boxes, azimuths, beams)
    xyz -= xyz.min(0)
    xyz *= np.float32((resolution - 1) / 400)
    return np.unique(np.round(xyz).astype(np.int32), axis=0)


def surface_cloud(seed: int, bits: int = 10, n_target: int = 200000):
    """Union of voxelised ellipsoid shells on a 2^bits grid, sized to ~n_target unique voxels."""
    rng = np.random.default_rng(seed)
    size = float((1 << bits) - 1)
    pts = []
    n_shapes = 3
    for _ in range(n_shapes):
        centre = rng.uniform(0.35, 0.65, 3) * size
        radii = rng.uniform(0.12, 0.30, 3) * size
        m = int(n_target * 2.2 / n_shapes)
        u = rng.normal(size=(m, 3))
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        pts.append(centre + u * radii)
    xyz = np.unique(np.clip(np.round(np.concatenate(pts)), 0, size).astype(np.int32), axis=0)
    if xyz.shape[0] > n_target:
        xyz = xyz[np.sort(rng.choice(xyz.shape[0], n_target, replace=False))]
    return xyz


def colored_surface(seed: int, bits: int = 10, n_target: int = 200000):
    """S4 "8iVFB-color" style: `surface_cloud` plus uint8 RGB = a low-frequency sinusoid field of position + N(0, 8)
    noise, clipped to 0..255.  -> (xyz int32 [N,3], rgb uint8 [N,3])."""
    xyz = surface_cloud(seed, bits, n_target)
    rng = np.random.default_rng([seed, 404])
    u = xyz.astype(np.float64) / float(1 << bits)                       # position in [0, 1)
    freq = rng.uniform(1.0, 3.0, (3, 3))                                # cycles over the grid, per channel and axis
    phase = rng.uniform(0.0, 2 * np.pi, (3, 3))
    field = 128.0 + 40.0 * np.sin(2 * np.pi * u[:, None, :] * freq[None] + phase[None]).sum(2)
    rgb = np.clip(np.rint(field + rng.normal(0.0, 8.0, field.shape)), 0, 255).astype(np.uint8)
    return xyz, rgb


def with_batch(xyz: np.ndarray, b: int = 0) -> np.ndarray:
    return np.concatenate([np.full((xyz.shape[0], 1), b, np.int32), xyz.astype(np.int32)], 1)


# ------------------------------------------------------------------------------------------------
# parameters
# ------------------------------------------------------------------------------------------------

def _rng(seed, name):
    return np.random.default_rng([seed, zlib.crc32(name.encode())])


def _requant_fxp(sd, prefix, scale_out, guard=2):
    """RequantFxpToScaledInt8.import_parameters (cuda_ops.py:487-503), zero_point 0."""
    shift = int(np.floor(np.log2((1 << (32 - guard)) * scale_out)))
    assert shift >= 0
    sd[prefix + 'requant_mul'] = np.array([round((2.0 ** shift) / scale_out)], dtype=np.uint32)
    sd[prefix + 'requant_shift'] = np.array([shift], dtype=np.int32)
    sd[prefix + 'int_zero_point_out'] = np.zeros(1, dtype=np.int64)


def _quant_affine(sd, prefix, w_float, bias_float, scale_in, scale_out, slope, guard):
    """Shared tail of SparseConvIn8Out8.import_parameters / LinearIn8W8.import_parameters
    (cuda_ops.py:250-301, 565-607) for symmetric (zero-point 0) observers.
    w_float: [..., out_ch, in_ch] already permuted to the int layout."""
    red = tuple(i for i in range(w_float.ndim) if i != w_float.ndim - 2)
    scale_w = np.maximum(np.abs(w_float).max(axis=red) / WeightRange, np.finfo(np.float32).eps)
    shape = [1] * w_float.ndim
    shape[-2] = -1
    sd[prefix + 'weight'] = np.clip(np.round(w_float / scale_w.reshape(shape)), -WeightRange, WeightRange).astype(np.int8)
    sd[prefix + 'bias'] = np.round(bias_float / (scale_in * scale_w)).astype(np.int32)
    if slope is not None:
        sd[prefix + 'slope'] = np.array([round(slope * (1 << 25))], dtype=np.int32)
    mul = scale_in * scale_w / scale_out if scale_out is not None else scale_in * scale_w
    shift = int(np.floor(np.log2((1 << (32 - guard)) / mul).min()))
    assert shift >= (0 if scale_out is not None else SharedFxpShift), shift
    sd[prefix + 'requant_mul'] = np.round(mul * 2.0 ** shift).astype(np.uint32)
    sd[prefix + 'requant_shift'] = np.array([shift], dtype=np.int32)
    sd[prefix + 'int_zero_point_out'] = np.zeros(1, dtype=np.int64)


def _conv(sd, prefix, seed, cin, cout, ks, scale_in, scale_out, prelu, gain=1.0):
    kv = ks ** 3
    r = _rng(seed, prefix)
    eff = cin * (min(kv, 4.0))  # ~4 occupied neighbours per voxel on LiDAR data
    w = r.normal(0, gain / np.sqrt(eff), (kv, cout, cin)).astype(np.float32)
    b = r.normal(0, 0.05, cout).astype(np.float32)
    _quant_affine(sd, prefix, w, b, scale_in, scale_out, 0.25 if prelu else None, guard=10)


def _linear(sd, prefix, seed, cin, cout, scale_in, scale_out, prelu, gain=1.0):
    r = _rng(seed, prefix)
    w = r.normal(0, gain / np.sqrt(cin), (cout, cin)).astype(np.float32)
    b = r.normal(0, 0.05, cout).astype(np.float32)
    _quant_affine(sd, prefix, w, b, scale_in, scale_out, 0.25 if prelu else None, guard=7)


S_ACT = 4.0 / 127  # per-tensor scale of every "scaled int8" activation


def _resblock(sd, prefix, seed, ch):
    _requant_fxp(sd, prefix + 'input_requant.', S_ACT)
    _conv(sd, prefix + 'conv_prelu.', seed, ch, ch, 3, S_ACT, S_ACT, True)
    _conv(sd, prefix + 'conv2.', seed, ch, ch, 3, S_ACT, None, False, gain=0.5)
    sd[prefix + 'prelu.slope'] = np.array([round(0.25 * (1 << 25))], dtype=np.int32)


def _one_scale(sd, prefix, seed, ch, if_upsample, allow_single_ch):
    if allow_single_ch:
        _conv(sd, prefix + 'dec_init.', seed, 1, ch, 3, 1.0, None, False)
    _resblock(sd, prefix + 'dec.', seed, ch)
    _requant_fxp(sd, prefix + 'pred.0.', S_ACT)
    _conv(sd, prefix + 'pred.1.', seed, ch, ch, 3, S_ACT, S_ACT, True)
    _linear(sd, prefix + 'pred.2.', seed, ch, 255, S_ACT, None, False, gain=2.0)
    if if_upsample:
        _requant_fxp(sd, prefix + 'upsample.0.', S_ACT)
        _linear(sd, prefix + 'upsample.1.', seed, ch + 8, ch, S_ACT, None, True)
        _resblock(sd, prefix + 'upsample.2.', seed, ch)
        _requant_fxp(sd, prefix + 'upsample.3.', S_ACT)
        _linear(sd, prefix + 'upsample.4.', seed, ch, ch * 8, S_ACT, None, False)


def _multi_step(sd, prefix, seed, ch, steps, use_more):
    if steps == 2:
        out_ch = ch
        _requant_fxp(sd, prefix + 'dec.0.', S_ACT)
        _linear(sd, prefix + 'dec.1.', seed, ch + 8, out_ch, S_ACT, None, True)
        _resblock(sd, prefix + 'dec.2.', seed, out_ch)
    else:
        k = 2 ** (steps - 2)
        _requant_fxp(sd, prefix + 'embed.0.', 1.0 / 127)
        if use_more:
            emb = 64 if steps == 3 else 512
            cin = (ch if steps == 3 else round(ch * 1.25)) + emb
            out_ch = round(ch * 1.25) if steps == 3 else ch * 2
            _conv(sd, prefix + 'embed.1.', seed, 8, emb, k, 1.0 / 127, None, True)
        else:
            emb, cin, out_ch = ch, 2 * ch, ch
            _conv(sd, prefix + 'embed.1.', seed, 8, emb, k, 1.0 / 127, None, ch >= 256)
        if cin != out_ch:
            _requant_fxp(sd, prefix + 'dec.0.', S_ACT)
            _linear(sd, prefix + 'dec.1.', seed, cin, out_ch, S_ACT, None, True)
            _resblock(sd, prefix + 'dec.2.', seed, out_ch)
        else:
            _resblock(sd, prefix + 'dec.', seed, out_ch)
    for i in range(steps):
        q = f'{prefix}pred.{i}.'
        if i == 0:
            _requant_fxp(sd, q + '0.', S_ACT)
            _conv(sd, q + '1.', seed, out_ch, out_ch, 3, S_ACT, S_ACT, True)
            _linear(sd, q + '2.', seed, out_ch, ch * 8, S_ACT, None, False)
        elif i != steps - 1:
            sd[q + '0.slope'] = np.array([round(0.25 * (1 << 25))], dtype=np.int32)
            _requant_fxp(sd, q + '1.', S_ACT)
            _linear(sd, q + '2.', seed, ch + 8, ch, S_ACT, S_ACT, True)
            _conv(sd, q + '3.', seed, ch, ch, 3, S_ACT, S_ACT, True)
            _linear(sd, q + '4.', seed, ch, ch * 8, S_ACT, None, False)
        else:
            _requant_fxp(sd, q + '0.', S_ACT)
            _conv(sd, q + '1.', seed, ch, ch, 3, S_ACT, S_ACT, True)
            _linear(sd, q + '2.', seed, ch, 255, S_ACT, None, False, gain=2.0)


def make_lossl_int_state_dict(channels=256, max_stride_wo_recurrent=2048, max_stride=8192, fea_stride=16,
                              use_more_ch_for_multi_step_pred=False, seed=7):
    """Random integer parameters for lossl_coord_int.Model under the reference's key names
    (module tree: lossl_coord_int/model.py:28-51, 95-154, 228-238)."""
    sd = {}
    n_wo = int(np.log2(max_stride_wo_recurrent))
    for i in range(n_wo):
        steps = int(np.log2(fea_stride)) - i
        p = f'blocks_dec.{i}.'
        if steps < 1:
            _one_scale(sd, p, seed, channels, True, False)
        elif steps == 1:
            _one_scale(sd, p, seed, channels, False, False)
        else:
            _multi_step(sd, p, seed, channels, steps, use_more_ch_for_multi_step_pred)
    _one_scale(sd, 'block_dec_recurrent.', seed, channels, True, True)
    return sd
