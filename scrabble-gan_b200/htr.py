"""Training the recogniser on its own: the handwriting-recognition (HTR) side of ScrabbleGAN's main experiment -- train R on
real words, on real plus generated words, with or without classic augmentation, and compare CER / word accuracy
(decode.evaluate_recognizer).

- augment_words: the word augmentation of sg_word_augment (affine warp + 3x3 grey min / max) with parameters drawn by the
  Philox kernel: two libsgan calls, no host synchronisation.
- train_recognizer_step: one update of R alone with Keras `trainable=True, training=True` semantics -- BatchNorm on batch
  statistics, moving averages updated -- unlike inside the GAN step, where R's BatchNorm runs in inference mode (SURVEY Q5).
- generated_word_batches / mixed_word_batches: batch sources of G's words, alone or appended to real batches.

The arithmetic is libsgan kernels; torch only allocates and copies.  There is no host fallback."""
from __future__ import annotations

import random

import numpy as np
import torch

from . import ops
from ._abi import SganError
from .bigacgan.net_architecture import _as_tensor, _nhwc, to_device_f32, to_device_i32


def _host_ints(x):
    """x as a host int array when it lives on the host (list / numpy / CPU tensor), else None."""
    if isinstance(x, torch.Tensor):
        return x.numpy().astype(np.int64).reshape(-1) if not x.is_cuda else None
    if isinstance(x, (np.ndarray, list, tuple)):
        return np.asarray(x, np.int64).reshape(-1)
    return None


def augment_words(images, widths=None, rotation=2.0, shear=0.3, scale=0.1, translate=2.0, p_morph=0.25):
    """Randomly augmented copies of word images (B, 32, W[, 1]) (host buffer, device tensor or DLPack producer), returned as
    new device images (B, 32, W, 1) fp32.  Every word gets its own rotation in [-rotation, rotation] degrees, horizontal
    shear (slant) in [-shear, shear], x / y scales in [1 - scale, 1 + scale], translations in [-translate, translate] pixels,
    and with probability p_morph each (p_morph <= 0.5) a 3x3 grey minimum or maximum -- thinner or thicker strokes for
    bright ink on a dark background, the other way round for dark ink.  widths (B,): each word's columns (ragged batches);
    columns right of a word are copied unchanged.  The parameters come from the runtime's Philox stream.

    The defaults are values typical of word-level HTR augmentation; they have not been tuned on this code base."""
    from .runtime import get_runtime
    rt = get_runtime()
    x = _nhwc(to_device_f32(rt, images))
    w_dev = None
    if widths is not None:
        host = _host_ints(widths)
        if host is not None and ((host < 1) | (host > x.shape[2])).any():
            raise SganError("augment_words: widths must lie in [1, {}], got {}".format(x.shape[2], host.tolist()))
        w_dev = to_device_i32(rt, widths).reshape(-1)
    u = ops.random_(rt, rt.empty((x.shape[0], 7)), normal=False)
    return ops.word_augment(rt, x, u, w_dev, rotation, shear, scale, translate, p_morph)


def train_recognizer_step(recognizer, optimizer, images, labels, input_length=None, label_length=None, augment=None):
    """One training update of R alone: forward with BatchNorm on batch statistics (moving averages updated: epsilon 1e-3,
    momentum 0.99), the gradient of the SUM of the per-sample CTC losses (SURVEY Q7), then
    optimizer.apply_gradients(zip(grads, trainable_variables)) -- an Adam or RMSprop of optim.setup_optimizer.

    images (B, 32, W[, 1]) and labels (B, L) as load_prepare_data yields them (one length bucket), or a ragged batch with
    input_length / label_length (B,) as R's model takes them (frames 4 len - 1, label counts).  augment: None, or a dict of
    augment_words keyword arguments; a ragged batch's words are augmented within their own 4 (input_length + 1) = 16 len
    columns.  recognizer.bn_training is True only for the duration of the step.  Returns the mean loss, a 0-d device
    tensor: the step does not synchronise with the host."""
    rt = recognizer.rt
    if rt.world_size > 1:
        raise NotImplementedError("train_recognizer_step runs on one replica; data-parallel HTR training is not supported")
    x = _nhwc(to_device_f32(rt, images))
    y = to_device_i32(rt, labels)
    il = None if input_length is None else to_device_i32(rt, input_length).reshape(-1)
    ll = None if label_length is None else to_device_i32(rt, label_length).reshape(-1)
    if augment is not None:
        widths = None
        if il is not None:
            host = _host_ints(input_length)
            if host is not None and ((host < 0) | (4 * (host + 1) > x.shape[2])).any():
                raise SganError("train_recognizer_step: input_length {} does not fit {} columns".format(host.tolist(), x.shape[2]))
            widths = 4 * (il + 1)                                  # the reference's width rule, 16 len
        x = augment_words(x, widths, **augment)
    prev = recognizer.bn_training
    recognizer.bn_training = True
    try:
        # R is prepared as the GAN step prepares it (data_utils._step_device)
        recognizer.store.zero_grad()
        recognizer.sn_forward(rt, update_u=True)
        if rt.use_tc:
            recognizer.prepack(rt)
        loss, cache = recognizer.forward(rt, x, y, want_grad=True, input_length=il, label_length=ll)
        recognizer.backward(rt, cache, None, wgrad=True, want_dx=False)
        recognizer.sn_backward(rt)
        tv = recognizer.store.trainable_variables
        optimizer.apply_gradients(zip([v.grad for v in tv], tv))
    finally:
        recognizer.bn_training = prev
    mean = rt.empty((1,))
    ops.colsum_into(rt, loss.view(-1, 1), 1, mean, accumulate=0)
    ops.axpby(rt, 1.0 / loss.shape[0], mean, out=mean)
    return mean.view(())


def _check_generator(generator):
    if generator.style is not None:
        raise ValueError("a style-encoder generator needs style images, not z: it cannot serve as a source of random words")


def _words(random_words, length):
    words = random_words[length - 1] if 1 <= length <= len(random_words) else []
    if len(words) == 0:
        raise ValueError("random_words has no word of length {}".format(length))
    return words


def generated_word_batches(generator, random_words, batch_size, bucket_weights=None, seed=0):
    """Endless generator of (images (B, 32, 16 L, 1), labels (B, L) int32), both on the device: ONE length bucket per batch,
    drawn from bucket_weights (uniform if None; the reference's rule, data_utils.py:64), words drawn from random_words[L - 1]
    as in train_step, z from the runtime's Philox stream, G in inference mode (training=False).  `seed` seeds the host
    choices of lengths and words."""
    _check_generator(generator)
    rt = generator.rt
    rng = np.random.RandomState(seed)
    p = None
    if bucket_weights is not None:
        p = np.asarray(bucket_weights, np.float64)
        p = p / p.sum()
    while True:
        length = int(rng.choice(len(random_words), 1, p=p)[0]) + 1
        words = _words(random_words, length)
        y = to_device_i32(rt, np.array([words[i] for i in rng.randint(0, len(words), size=batch_size)], np.int32))
        z = ops.random_(rt, rt.empty((batch_size, generator.latent_dim)))
        yield generator([z, y], training=False, ragged=False), y


def mixed_word_batches(real_batches, generator, random_words, n_generated):
    """For every (images (B, 32, 16 L[, 1]), labels (B, L)) of real_batches: one device batch of B + n_generated words -- the
    real rows (one copy), then n_generated words of the SAME length L drawn from random_words[L - 1] (Python's `random`, as
    train_step draws its fake words), generated by G in inference mode straight into their rows (img_out).  Yields
    (images (B + n_generated, 32, 16 L, 1), labels (B + n_generated, L) int32)."""
    _check_generator(generator)
    rt = generator.rt
    for batch in real_batches:
        labels = _as_tensor(batch[1], np.int32)
        b, length = labels.shape[0], labels.shape[1]
        words = _words(random_words, length)
        fake = np.array([random.choice(words) for _ in range(n_generated)], np.int32).reshape(n_generated, length)
        n = b + n_generated
        x = rt.empty((n, 32, 16 * length, 1))
        x[:b].copy_(_as_tensor(batch[0], np.float32).reshape(b, 32, 16 * length, 1), non_blocking=True)
        y = torch.empty((n, length), device=rt.device, dtype=torch.int32)
        y[:b].copy_(labels, non_blocking=True)
        y[b:].copy_(torch.from_numpy(fake), non_blocking=True)
        if n_generated > 0:
            z = ops.random_(rt, rt.empty((n_generated, generator.latent_dim)))
            generator.sn_forward(rt, update_u=False)
            generator.forward(rt, z, y[b:], training=False, img_out=x[b:])
        yield x, y
