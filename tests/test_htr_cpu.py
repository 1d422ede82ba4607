"""The float64 word-augmentation reference (tests/_htr_ref.py) against scipy.ndimage, its exact cases, and the u -> parameter
mapping with its morphology thresholds.  No GPU involved."""
import numpy as np
import pytest
from scipy import ndimage

import _htr_ref as H


def _scipy_augment(img, u_row, rotation, shear, scale, translate, p_morph):
    """One word through scipy: affine_transform maps output (row, col) to input matrix @ (row, col) + offset."""
    h, wb = img.shape
    prm = H.aug_params(u_row[None], rotation, shear, scale, translate, p_morph)
    m = H.inverse_matrix(prm["theta"][0], prm["k"][0], prm["sx"][0], prm["sy"][0])
    m_rc = np.array([[m[1, 1], m[1, 0]], [m[0, 1], m[0, 0]]])
    c = np.array([h / 2.0, wb / 2.0])
    t = np.array([prm["ty"][0], prm["tx"][0]])
    out = ndimage.affine_transform(img, m_rc, offset=c - m_rc @ (c + t), order=1, mode="nearest")
    if prm["morph"][0] < 0:
        out = ndimage.grey_erosion(out, size=3, mode="nearest")
    elif prm["morph"][0] > 0:
        out = ndimage.grey_dilation(out, size=3, mode="nearest")
    return out


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_reference_matches_scipy(seed):
    rng = np.random.default_rng(seed)
    n, h, w = 12, 32, 96
    images = rng.uniform(-1, 1, (n, h, w))
    widths = rng.integers(1, 7, n) * 16
    u = rng.uniform(-1, 1, (n, 7))
    kw = dict(rotation=8.0, shear=0.4, scale=0.2, translate=3.0, p_morph=0.3)
    got = H.augment(images, u, widths, **kw)
    for b in range(n):
        wb = widths[b]
        exp = _scipy_augment(images[b, :, :wb], u[b], **kw)
        np.testing.assert_allclose(got[b, :, :wb], exp, rtol=0, atol=1e-12)
        np.testing.assert_array_equal(got[b, :, wb:], images[b, :, wb:])


def test_identity_and_integer_translation():
    rng = np.random.default_rng(3)
    images = rng.uniform(-1, 1, (3, 32, 48))
    u = rng.uniform(-1, 1, (3, 7))
    np.testing.assert_array_equal(H.augment(images, u), images)                        # all ranges zero
    u = np.zeros((3, 7))
    u[:, 4], u[:, 5] = 0.5, -0.5                                                         # tx = +2, ty = -2 pixels
    got = H.augment(images, u, translate=4.0)
    exp = np.empty_like(images)
    rows = np.clip(np.arange(32) + 2, 0, 31)                                            # dst(x, y) = src(x - 2, y + 2)
    cols = np.clip(np.arange(48) - 2, 0, 47)
    exp[:] = images[:, rows][:, :, cols]
    np.testing.assert_array_equal(got, exp)


def test_parameter_mapping_and_morph_thresholds():
    u = np.array([[1.0, -0.5, 0.25, -1.0, 0.5, -0.25, 0.0]])
    p = H.aug_params(u, rotation=4.0, shear=0.2, scale=0.1, translate=2.0, p_morph=0.25)
    assert np.isclose(p["theta"][0], np.deg2rad(4.0))
    assert np.isclose(p["k"][0], -0.1)
    assert np.isclose(p["sx"][0], 1.025) and np.isclose(p["sy"][0], 0.9)
    assert np.isclose(p["tx"][0], 1.0) and np.isclose(p["ty"][0], -0.5)
    u6 = np.array([-1.0, -0.51, -0.5, 0.0, 0.5, 0.51, 0.99])
    rows = np.zeros((len(u6), 7))
    rows[:, 6] = u6
    assert H.aug_params(rows, 0, 0, 0, 0, 0.25)["morph"].tolist() == [-1, -1, 0, 0, 0, 1, 1]
    assert H.aug_params(rows, 0, 0, 0, 0, 0.0)["morph"].tolist() == [0] * 7          # u in [-1, 1): never
    assert H.aug_params(rows, 0, 0, 0, 0, 0.5)["morph"].tolist() == [-1, -1, -1, 0, 1, 1, 1]
    # the forward map is Rot Shear Scale: its inverse undoes a sheared, scaled, rotated point
    m = H.inverse_matrix(0.3, 0.2, 1.1, 0.9)
    rot = np.array([[np.cos(0.3), -np.sin(0.3)], [np.sin(0.3), np.cos(0.3)]])
    v = np.array([2.0, -3.0])
    np.testing.assert_allclose(m @ (rot @ (np.array([[1, 0.2], [0, 1]]) @ (np.diag([1.1, 0.9]) @ v))), v, atol=1e-12)
