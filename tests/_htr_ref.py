"""Float64 restatements for training R on its own (scrabble-gan_b200/htr.py): the word augmentation of sg_word_augment and R's
forward pass with training-mode BatchNorm, built from the oracle's pieces (oracle/sgan_oracle.py is not changed)."""
import numpy as np
import torch

import sgan_oracle as O


def aug_params(u, rotation, shear, scale, translate, p_morph):
    """Row b of u (n, 7) in [-1, 1) -> word b's parameters: theta (radians; u0 * rotation degrees), shear k, scales sx / sy,
    translations tx / ty, morph (-1 minimum, +1 maximum, 0 none).  The morphology thresholds -1 + 2 p and 1 - 2 p are
    formed in fp32 as the kernel forms them."""
    u = np.asarray(u, np.float64).reshape(-1, 7)
    p = np.float32(p_morph)
    lo, hi = np.float32(-1) + np.float32(2) * p, np.float32(1) - np.float32(2) * p
    return {"theta": np.deg2rad(u[:, 0] * rotation), "k": u[:, 1] * shear, "sx": 1 + u[:, 2] * scale, "sy": 1 + u[:, 3] * scale,
            "tx": u[:, 4] * translate, "ty": u[:, 5] * translate,
            "morph": np.where(u[:, 6] < lo, -1, np.where(u[:, 6] > hi, 1, 0))}


def inverse_matrix(theta, k, sx, sy):
    """Inverse of the forward map Rot(theta) Shear(k) Scale(sx, sy) in (x, y) = (column, row) coordinates."""
    rot = np.array([[np.cos(theta), -np.sin(theta)], [np.sin(theta), np.cos(theta)]])
    fwd = rot @ np.array([[1.0, k], [0.0, 1.0]]) @ np.diag([sx, sy])
    return np.linalg.inv(fwd)


def bilinear_replicate(img, xs, ys):
    """Bilinear samples of img (h, w) at (xs, ys), coordinates clamped to the image (border replicate)."""
    h, w = img.shape
    xs, ys = np.clip(xs, 0, w - 1), np.clip(ys, 0, h - 1)
    x0, y0 = np.floor(xs).astype(np.int64), np.floor(ys).astype(np.int64)
    x1, y1 = np.minimum(x0 + 1, w - 1), np.minimum(y0 + 1, h - 1)
    ax, ay = xs - x0, ys - y0
    top = img[y0, x0] * (1 - ax) + img[y0, x1] * ax
    bot = img[y1, x0] * (1 - ax) + img[y1, x1] * ax
    return top * (1 - ay) + bot * ay


def warp(img, m_inv, tx, ty):
    """The word img (h, wb) warped: output (x, y) samples img at c + m_inv ((x, y) - c - t), c = (wb / 2, h / 2)."""
    h, wb = img.shape
    ys, xs = np.mgrid[0:h, 0:wb].astype(np.float64)
    cx, cy = wb / 2.0, h / 2.0
    dx, dy = xs - cx - tx, ys - cy - ty
    return bilinear_replicate(img, cx + m_inv[0, 0] * dx + m_inv[0, 1] * dy, cy + m_inv[1, 0] * dx + m_inv[1, 1] * dy)


def grey_3x3(img, kind):
    """3x3 grey minimum (kind < 0) or maximum (kind > 0); neighbours outside the image are left out."""
    pad = np.pad(img, 1, mode="edge")            # replicating the border leaves the outside out of a min / max
    h, w = img.shape
    stack = np.stack([pad[i:i + h, j:j + w] for i in range(3) for j in range(3)])
    return stack.min(0) if kind < 0 else stack.max(0)


def augment(images, u, widths=None, rotation=0.0, shear=0.0, scale=0.0, translate=0.0, p_morph=0.0):
    """images (n, h, w); word b occupies columns [0, widths[b]) and the columns right of it are copied."""
    images = np.asarray(images, np.float64)
    n, h, w = images.shape
    widths = np.full(n, w) if widths is None else np.asarray(widths)
    prm = aug_params(u, rotation, shear, scale, translate, p_morph)
    out = images.copy()
    for b in range(n):
        wb = int(widths[b])
        m_inv = inverse_matrix(prm["theta"][b], prm["k"][b], prm["sx"][b], prm["sy"][b])
        word = warp(images[b, :, :wb], m_inv, prm["tx"][b], prm["ty"][b])
        if prm["morph"][b] != 0:
            word = grey_3x3(word, prm["morph"][b])
        out[b, :, :wb] = word
    return out


def recognizer_train(x, labels, input_length, label_length, p):
    """make_recognizer's model output with BOTH BatchNorms in training mode (Keras trainable=True, training=True): batch
    statistics, moving averages updated.  Returns (per-sample CTC losses (B,), {bn*.moving_mean / var: new value}).  The
    operand rounding of O.set_operand_rounding applies as in O.recognizer_probs."""
    new = {}

    def bn(net, name):
        xh, mm, mv = O.batchnorm_train(net, p[name + ".moving_mean"], p[name + ".moving_var"])
        new[name + ".moving_mean"], new[name + ".moving_var"] = mm.detach(), mv.detach()
        return xh * p[name + ".gamma"] + p[name + ".beta"]
    net = O._stored(torch.relu(O.conv2d(x, p["conv1.w"], p["conv1.b"])))
    net = O.max_pool(net, 2, 2)
    net = O._stored(torch.relu(O.conv2d(net, p["conv2.w"], p["conv2.b"])))
    net = O.max_pool(net, 2, 2)
    net = torch.relu(O.conv2d(net, p["conv3.w"], p["conv3.b"]))
    net = O._stored(torch.relu(O.conv2d(net, p["conv4.w"], p["conv4.b"])))
    net = O.max_pool(net, 2, 1)
    net = bn(torch.relu(O.conv2d(net, p["conv5.w"], p["conv5.b"])), "bn5")
    net = O._stored(bn(torch.relu(O.conv2d(net, p["conv6.w"], p["conv6.b"])), "bn6"))
    net = O.max_pool(net, 2, 1)
    net = torch.relu(O.conv2d(net, p["conv7.w"], p["conv7.b"], padding="valid")).squeeze(1)
    probs = torch.softmax(O.dense(net, p["dense.w"], p["dense.b"]), dim=-1)
    return O.ctc_batch_cost(labels, probs, input_length, label_length).view(-1), new

