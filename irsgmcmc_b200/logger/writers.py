"""
Sample persistence with the reference's function names and on-disk formats (reference logger/logger.py:35-102,215-238):
images as NIfTI-1 (.nii / .nii.gz), vector fields as legacy-VTK structured points with a 3-component VECTORS array named
'field', grids as legacy-VTK structured grids.  The reference goes through nibabel and tvtk; neither is a dependency here --
both formats are a fixed header plus the raw array, written with numpy and the standard library, readable by nibabel /
SimpleITK / vtkStructuredPointsReader / ParaView.  Host-side I/O: not on the GPU path (SURVEY.md section 8f, row N4).
"""
import gzip
import os
import struct

import numpy as np

_NIFTI_DTYPES = {np.dtype('uint8'): (2, 8), np.dtype('int16'): (4, 16), np.dtype('int32'): (8, 32),
                 np.dtype('float32'): (16, 32), np.dtype('float64'): (64, 64)}


def _to_numpy(x):
    if hasattr(x, 'detach'):
        x = x.detach().cpu().numpy()
    return np.asarray(x)


def save_im_to_disk(im, file_path, spacing=(1, 1, 1)):
    """3-D image -> single-file NIfTI-1 (reference logger/logger.py:83-102: nib.Nifti1Image(im, eye(4)), units mm, zooms =
    spacing).  Array axes are (i, j, k) as given; data are stored in NIfTI (Fortran) order like nibabel does."""
    im = _to_numpy(im)
    if im.dtype == np.bool_:
        im = im.astype(np.uint8)
    if im.dtype not in _NIFTI_DTYPES:
        im = im.astype(np.float32)
    if im.ndim != 3:
        raise ValueError('save_im_to_disk expects a 3-D array')
    code, bitpix = _NIFTI_DTYPES[im.dtype]
    spacing = [float(s) for s in _to_numpy(spacing).reshape(-1)[:3]]
    hdr = bytearray(348)
    struct.pack_into('<i', hdr, 0, 348)                                   # sizeof_hdr
    struct.pack_into('<8h', hdr, 40, 3, im.shape[0], im.shape[1], im.shape[2], 1, 1, 1, 1)   # dim
    struct.pack_into('<h', hdr, 70, code)                                 # datatype
    struct.pack_into('<h', hdr, 72, bitpix)
    struct.pack_into('<8f', hdr, 76, 1.0, spacing[0], spacing[1], spacing[2], 1.0, 1.0, 1.0, 1.0)   # pixdim (qfac = 1)
    struct.pack_into('<f', hdr, 108, 352.0)                               # vox_offset
    struct.pack_into('<f', hdr, 112, 1.0)                                 # scl_slope
    hdr[123] = 2                                                          # xyzt_units: millimetres (header.set_xyzt_units(2))
    struct.pack_into('<h', hdr, 252, 0)                                   # qform_code
    struct.pack_into('<h', hdr, 254, 2)                                   # sform_code: aligned (what nibabel sets for a given affine)
    struct.pack_into('<4f', hdr, 280, spacing[0], 0.0, 0.0, 0.0)          # srow_x .. srow_z: affine with the zooms on the diagonal
    struct.pack_into('<4f', hdr, 296, 0.0, spacing[1], 0.0, 0.0)
    struct.pack_into('<4f', hdr, 312, 0.0, 0.0, spacing[2], 0.0)
    hdr[344:348] = b'n+1\0'
    payload = bytes(hdr) + b'\0\0\0\0' + np.asfortranarray(im).astype(im.dtype.newbyteorder('<')).tobytes(order='F')
    opener = gzip.open if str(file_path).endswith('.gz') else open
    with opener(file_path, 'wb') as f:
        f.write(payload)


def load_im_from_disk(file_path):
    """(array, spacing) of a NIfTI-1 file written by save_im_to_disk (round-trip check; not a general reader)"""
    opener = gzip.open if str(file_path).endswith('.gz') else open
    with opener(file_path, 'rb') as f:
        raw = f.read()
    if struct.unpack_from('<i', raw, 0)[0] != 348 or raw[344:347] != b'n+1':
        raise ValueError('not a little-endian single-file NIfTI-1')
    dim = struct.unpack_from('<8h', raw, 40)
    code = struct.unpack_from('<h', raw, 70)[0]
    dtype = next(k for k, v in _NIFTI_DTYPES.items() if v[0] == code)
    off = int(struct.unpack_from('<f', raw, 108)[0])
    shape = tuple(dim[1:1 + dim[0]])
    arr = np.frombuffer(raw, dtype=dtype.newbyteorder('<'), count=int(np.prod(shape)), offset=off).reshape(shape, order='F')
    return arr.copy(), struct.unpack_from('<8f', raw, 76)[1:4]


def _vtk_header(title, dataset):
    return f'# vtk DataFile Version 3.0\n{title}\nBINARY\nDATASET {dataset}\n'.encode('ascii')


def save_field_to_disk(field, file_path, spacing=(1, 1, 1)):
    """vector field (3, n0, n1, n2) -> legacy VTK structured points, VECTORS 'field' (reference logger/logger.py:35-61: tvtk
    ImageData(dimensions = field_x.shape) with the vectors transposed so that the first array axis varies fastest)"""
    field = _to_numpy(field).astype(np.float32)
    spacing = [float(s) for s in _to_numpy(spacing).reshape(-1)[:3]]
    n0, n1, n2 = field.shape[1:]
    vec = np.stack((field[0], field[1], field[2]), -1).transpose(2, 1, 0, 3).reshape(-1, 3)
    with open(file_path, 'wb') as f:
        f.write(_vtk_header('irsgmcmc_b200 vector field', 'STRUCTURED_POINTS'))
        f.write(f'DIMENSIONS {n0} {n1} {n2}\nORIGIN 0 0 0\nSPACING {spacing[0]} {spacing[1]} {spacing[2]}\n'.encode('ascii'))
        f.write(f'POINT_DATA {n0 * n1 * n2}\nVECTORS field float\n'.encode('ascii'))
        f.write(vec.astype('>f4').tobytes())
        f.write(b'\n')


def save_grid_to_disk(grid, file_path):
    """transformation grid (3, n0, n1, n2) -> legacy VTK structured grid (reference logger/logger.py:64-80)"""
    grid = _to_numpy(grid).astype(np.float32)
    n0, n1, n2 = grid.shape[1:]
    pts = np.stack((grid[0], grid[1], grid[2]), -1).transpose(2, 1, 0, 3).reshape(-1, 3)
    with open(file_path, 'wb') as f:
        f.write(_vtk_header('irsgmcmc_b200 structured grid', 'STRUCTURED_GRID'))
        f.write(f'DIMENSIONS {n0} {n1} {n2}\nPOINTS {n0 * n1 * n2} float\n'.encode('ascii'))
        f.write(pts.astype('>f4').tobytes())
        f.write(b'\n')


def load_field_from_disk(file_path):
    """(field (3, n0, n1, n2), spacing) of a file written by save_field_to_disk (round-trip check; the reference's
    tests/test_utils.py:153-159 does the same through vtkStructuredPointsReader)"""
    with open(file_path, 'rb') as f:
        raw = f.read()
    head, _, rest = raw.partition(b'VECTORS field float\n')
    lines = head.decode('ascii').split('\n')
    dims = [int(x) for x in next(l for l in lines if l.startswith('DIMENSIONS')).split()[1:]]
    spacing = [float(x) for x in next(l for l in lines if l.startswith('SPACING')).split()[1:]]
    n = dims[0] * dims[1] * dims[2]
    vec = np.frombuffer(rest, dtype='>f4', count=3 * n).reshape(dims[2], dims[1], dims[0], 3)
    return np.ascontiguousarray(vec.transpose(3, 2, 1, 0)).astype(np.float32), spacing


def save_sample(save_dir, spacing, sample_no, im_moving_warped_batch, displacement_batch, log_det_J_batch=None, model='MCMC',
                chain_no=None):
    """one kept sample -> <save_dir>/..._im_moving_warped.nii.gz, ..._displacement.vtk, ..._log_det_J.nii.gz with the
    reference's file names (logger/logger.py:215-238; the displacement is scaled by spacing[0] like there)"""
    os.makedirs(save_dir, exist_ok=True)
    prefix = f'chain_{chain_no}_sample_{sample_no:07}' if model == 'MCMC' else f'sample_{sample_no:07}'
    sp = [float(s) for s in _to_numpy(spacing).reshape(-1)[:3]]
    paths = {'im_moving_warped': os.path.join(save_dir, prefix + '_im_moving_warped.nii.gz'),
             'displacement': os.path.join(save_dir, prefix + '_displacement.vtk')}
    save_im_to_disk(_to_numpy(im_moving_warped_batch)[0, 0], paths['im_moving_warped'], sp)
    save_field_to_disk(_to_numpy(displacement_batch)[0] * sp[0], paths['displacement'], sp)
    if log_det_J_batch is not None:
        paths['log_det_J'] = os.path.join(save_dir, prefix + '_log_det_J.nii.gz')
        save_im_to_disk(_to_numpy(log_det_J_batch)[0], paths['log_det_J'], sp)
    return paths


def save_displacement_mean_and_std_dev(save_dir, spacing, displacement_mean, displacement_std_dev, mask, model):
    """sample mean / standard deviation of the displacement (3, D, H, W), scaled by spacing[0], with and without the moving mask
    (1, 1, D, H, W): <model>_sample_mean.vtk, _mean_masked.vtk, _std_dev.vtk, _std_dev_masked.vtk -- the reference's four files
    (logger/logger.py:110-131)"""
    os.makedirs(save_dir, exist_ok=True)
    sp = [float(s) for s in _to_numpy(spacing).reshape(-1)[:3]]
    m = None if mask is None else _to_numpy(mask)[0].astype(np.float32)
    paths = {}
    for tag, field in (('mean', displacement_mean), ('std_dev', displacement_std_dev)):
        f = _to_numpy(field).astype(np.float32) * np.float32(sp[0])
        paths[tag] = os.path.join(save_dir, f'{model}_sample_{tag}.vtk')
        save_field_to_disk(f, paths[tag], sp)
        if m is not None:
            paths[tag + '_masked'] = os.path.join(save_dir, f'{model}_sample_{tag}_masked.vtk')
            save_field_to_disk(f * m, paths[tag + '_masked'], sp)
    return paths


def save_variational_posterior_mean(save_dir, spacing, im_moving_warped, displacement):
    """registration at the mean of q(v): im_moving_warped_mu.nii.gz and displacement_mu.vtk (reference logger/logger.py:198-208)"""
    os.makedirs(save_dir, exist_ok=True)
    sp = [float(s) for s in _to_numpy(spacing).reshape(-1)[:3]]
    paths = {'im_moving_warped_mu': os.path.join(save_dir, 'im_moving_warped_mu.nii.gz'),
             'displacement_mu': os.path.join(save_dir, 'displacement_mu.vtk')}
    save_im_to_disk(_to_numpy(im_moving_warped)[0, 0], paths['im_moving_warped_mu'], sp)
    save_field_to_disk(_to_numpy(displacement)[0] * sp[0], paths['displacement_mu'], sp)
    return paths


def save_landmarks_to_disk(file_path, points, covariance=None, scalars=None):
    """landmarks -> legacy VTK POLYDATA (one vertex per point, readable by vtkPolyDataReader / ParaView): points (P, 3) in mm,
    covariance (P, 6) = (xx, xy, xz, yy, yz, zz) as a symmetric 3x3 TENSORS array 'covariance', scalars {name: (P,)} as one
    SCALARS array each (NaN stays NaN)"""
    pts = _to_numpy(points).astype(np.float64).reshape(-1, 3)
    P = pts.shape[0]
    with open(file_path, 'wb') as f:
        f.write(_vtk_header('irsgmcmc_b200 landmarks', 'POLYDATA'))
        f.write(f'POINTS {P} float\n'.encode('ascii'))
        f.write(pts.astype('>f4').tobytes())
        f.write(f'\nVERTICES {P} {2 * P}\n'.encode('ascii'))
        f.write(np.stack((np.ones(P), np.arange(P)), -1).astype('>i4').tobytes())
        f.write(f'\nPOINT_DATA {P}\n'.encode('ascii'))
        if covariance is not None:
            c = _to_numpy(covariance).astype(np.float64).reshape(P, 6)
            full = c[:, [0, 1, 2, 1, 3, 4, 2, 4, 5]]
            f.write(b'TENSORS covariance float\n')
            f.write(full.astype('>f4').tobytes())
            f.write(b'\n')
        for name, values in (scalars or {}).items():
            f.write(f'SCALARS {name} float 1\nLOOKUP_TABLE default\n'.encode('ascii'))
            f.write(_to_numpy(values).astype('>f4').reshape(P).tobytes())
            f.write(b'\n')


def load_landmarks_from_disk(file_path):
    """(points (P, 3), {array name: values}) of a file written by save_landmarks_to_disk (round-trip check; not a general
    reader): tensors come back as (P, 3, 3), scalars as (P,)"""
    with open(file_path, 'rb') as f:
        raw = f.read()
    pos = raw.index(b'POINTS ')
    line_end = raw.index(b'\n', pos)
    P = int(raw[pos:line_end].split()[1])
    points = np.frombuffer(raw, dtype='>f4', count=3 * P, offset=line_end + 1).reshape(P, 3).astype(np.float64)
    arrays, pos = {}, raw.index(b'POINT_DATA')
    pos = raw.index(b'\n', pos) + 1
    while pos < len(raw):
        line_end = raw.index(b'\n', pos)
        head = raw[pos:line_end].split()
        if head[0] == b'TENSORS':
            arrays[head[1].decode()] = np.frombuffer(raw, dtype='>f4', count=9 * P, offset=line_end + 1).reshape(P, 3, 3)
            pos = line_end + 1 + 36 * P + 1
        else:   # SCALARS name float 1 / LOOKUP_TABLE default
            lut_end = raw.index(b'\n', line_end + 1)
            arrays[head[1].decode()] = np.frombuffer(raw, dtype='>f4', count=P, offset=lut_end + 1).copy()
            pos = lut_end + 1 + 4 * P + 1
    return points, arrays
