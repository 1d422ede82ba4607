"""Host-side logic that needs no GPU: the gin-subset reader on the reference's own configuration text, the TF SAME /
transposed-conv phase descriptors, the Keras Adam step size, the channel tables and the step's FLOP model."""
import importlib
import math

import pytest

gin = importlib.import_module("scrabble-gan_b200.gin_lite")

# the bindings of /root/reference/src/scrabble_gan.gin (quoted here: the GPU box has no /root/reference)
GIN_TEXT = """
# Loss and Optimizer (AdamOptimizer for both G, D and R)
setup_optimizer.g_lr = 2E-4
setup_optimizer.d_lr = 2E-4
setup_optimizer.r_lr = 2E-4
setup_optimizer.w_lr = 2E-4
setup_optimizer.beta_1 = 0.0
setup_optimizer.beta_2 = 0.999
setup_optimizer.loss_fn = @hinge                #@not_saturating       #@hinge
setup_optimizer.disc_iters=1                    #2
setup_optimizer.apply_gradient_balance=0        #1      #0
setup_optimizer.rmsprop=0                       #0      #1
shared_specs.latent_dim = 128
shared_specs.embed_y = (32, 8192)
shared_specs.kernel_reg = @spectral_norm
shared_specs.g_bw_attention = 'B3'              #'B_skip'
io.input_dim = (32, 160, 1)
io.seq_len = None
io.char_vec = 'abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ'
"""


def test_gin_subset_reader_parses_the_reference_config():
    gin.clear_config()

    def hinge(a, b, c, d):
        return "hinge"

    def spectral_norm(w, power_iteration=1):
        return w
    gin.external_configurable(hinge)
    gin.external_configurable(spectral_norm)

    @gin.configurable
    def setup_optimizer(g_lr, d_lr, r_lr, w_lr, beta_1, beta_2, loss_fn, disc_iters, apply_gradient_balance, rmsprop):
        return g_lr, beta_1, beta_2, loss_fn, disc_iters, apply_gradient_balance, rmsprop

    @gin.configurable("shared_specs")
    def get_shared_specs(latent_dim, embed_y, kernel_reg, g_bw_attention):
        return latent_dim, embed_y, kernel_reg, g_bw_attention

    gin.parse_config(GIN_TEXT)
    g_lr, b1, b2, loss_fn, disc_iters, agb, rms = setup_optimizer()
    assert (g_lr, b1, b2, disc_iters, agb, rms) == (2e-4, 0.0, 0.999, 1, 0, 0) and loss_fn is hinge
    latent, embed_y, reg, attn = get_shared_specs()
    assert latent == 128 and embed_y == (32, 8192) and reg is spectral_norm and attn == "B3"
    assert gin.query_parameter("io.input_dim") == (32, 160, 1) and gin.query_parameter("io.seq_len") is None
    assert len(gin.query_parameter("io.char_vec")) == 52
    assert setup_optimizer(g_lr=1.0)[0] == 1.0            # explicit arguments win over bindings
    with pytest.raises(ValueError):
        gin.parse_config("not a binding")
    gin.clear_config()


def test_conv_descriptors_follow_tf_padding_rules():
    ops = importlib.import_module("scrabble-gan_b200.ops")
    d = ops.desc_conv_fwd(2, 8, 20, 64, 128, 3, 3, "same")
    assert (d.out_h, d.out_w, d.ntaps) == (8, 20, 9) and (d.tap_dy[0], d.tap_dx[0]) == (-1, -1) and d.w_co_stride == 1
    d = ops.desc_conv_fwd(2, 2, 19, 512, 512, 2, 2, "valid")
    assert (d.out_h, d.out_w, d.ntaps) == (1, 18, 4) and (d.tap_dy[3], d.tap_dx[3]) == (1, 1)
    # Conv2DTranspose 3x3 stride (2,2) SAME: out y = 2 i + kh, cropped -> phases with 1, 2, 2, 4 taps; (2,1): 3 and 6 taps
    taps = sorted(ops.desc_convT_phase(1, 4, 4, 64, 64, 3, 2, 2, py, px).ntaps for (py, px) in ops.convT_phases(3, 2, 2))
    assert taps == [1, 2, 2, 4]
    taps = sorted(ops.desc_convT_phase(1, 4, 4, 64, 64, 3, 2, 1, py, px).ntaps for (py, px) in ops.convT_phases(3, 2, 1))
    assert taps == [3, 6]
    # the 1x1 stride-2 shortcut only reaches even output positions
    assert ops.convT_phases(1, 2, 2) == [(0, 0)] and ops.convT_phases(1, 2, 1) == [(0, 0)]
    dd = ops.desc_conv_dgrad(2, 8, 20, 64, 128, 3, 3, "same")
    assert (dd.c_in, dd.c_out, dd.w_ci_stride, dd.w_co_stride) == (128, 64, 1, 128)


def test_keras_adam_step_size_and_channel_tables():
    optim = importlib.import_module("scrabble-gan_b200.optim")
    na = importlib.import_module("scrabble-gan_b200.bigacgan.net_architecture")
    a = optim.Adam(2e-4, 0.0, 0.999)
    a.iterations = 1
    assert math.isclose(a._lr_t(), 2e-4 * math.sqrt(1 - 0.999), rel_tol=1e-12)
    a.iterations = 1000
    assert math.isclose(a._lr_t(), 2e-4 * math.sqrt(1 - 0.999 ** 1000), rel_tol=1e-12)
    a.advance_for_replay()
    assert a.iterations == 1001
    assert na.get_in_out_channels_gen(32) == ([512, 256, 128], [256, 128, 64])
    assert na.get_in_out_channels_disc(1, 32) == ([1, 64, 512, 1024], [64, 512, 1024, 1024])
    with pytest.raises(ValueError):
        na.get_in_out_channels_gen(64)
    g_opt, d_opt, r_opt, w_opt, loss_fn, disc_iters, agb = optim.setup_optimizer(2e-4, 2e-4, 2e-4, 2e-4, 0.0, 0.999, "hinge", 2, 1, 1)
    assert type(r_opt).__name__ == "RMSprop" and type(g_opt).__name__ == "Adam" and (disc_iters, agb) == (2, 1)


def test_bench_flop_model_matches_the_survey():
    import bench
    # SURVEY.md section 8d: Mode A step = 79.71 GF/img at L=5/5 and 160.32 at L=10/10
    assert abs(bench.step_gflop_per_image(5, 5, executed=False) - 79.714) < 0.01
    assert abs(bench.step_gflop_per_image(10, 10, executed=False) - 160.32) < 0.05
    # executed FLOPs: the merged D backward does not run the reference's frozen D pass over the fake images (one D forward's worth)
    assert abs(bench.step_gflop_per_image(5, 5) - (79.714 - 9.938)) < 0.01


def test_bench_dump_outputs_is_reproducible_and_bounded(tmp_path):
    """bench.py --dump-outputs on host-side parameter stores: the same step output and weights give byte-identical files
    (the weight sample is fixed), float32, every BN moving statistic in full, a large network sampled, 64 MB at most."""
    import types
    import numpy as np
    import torch
    import bench
    params = importlib.import_module("scrabble-gan_b200.params")
    nets = []
    for name, n in (("G", 3 * bench.DUMP_WEIGHT_SAMPLE), ("D", 1000), ("R", 7)):
        store = params.ParamStore(types.SimpleNamespace(device="cpu"), name, seed=len(nets))
        store.add("conv.w", (n, 1), params.init_glorot_uniform)
        if name != "D":
            store.add("bn.moving_mean", (8,), params.init_zeros, trainable=False)
            store.add("bn.moving_var", (8,), params.init_ones, trainable=False)
        store.finalize()
        nets.append(types.SimpleNamespace(store=store))
    stats = torch.linspace(-1, 1, 16)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), stats, nets)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["D_weights.npy", "G_bn_moving_stats.npy", "G_weights.npy", "R_bn_moving_stats.npy", "R_weights.npy",
                     "train_step_stats.npy"]
    assert all((tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes() for f in files)
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert all(a.dtype == np.float32 for a in got.values())
    assert np.array_equal(got["train_step_stats"], stats.numpy())
    assert np.array_equal(got["G_bn_moving_stats"], np.r_[np.zeros(8), np.ones(8)])
    assert got["G_weights"].shape == (bench.DUMP_WEIGHT_SAMPLE,) and np.isin(got["G_weights"], nets[0].store.w.numpy()).all()
    assert np.array_equal(got["R_weights"], nets[2].store.by_name["conv.w"].numpy().ravel())
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 64 << 20


def test_synthetic_loaders_keep_the_reference_interfaces():
    du = importlib.import_module("scrabble-gan_b200.bigacgan.data_utils")
    char_vec = "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ"
    gen = du.synthetic_word_batches((32, 160, 1), 4, char_vec, 10, seed=3)
    seen = set()
    for _ in range(40):
        imgs, labels = next(gen)
        length = labels.shape[1]
        seen.add(length)
        assert imgs.shape == (4, 32, 16 * length, 1) and imgs.dtype.name == "float32" and labels.dtype.name == "int32"
        assert -1.0 <= imgs.min() and imgs.max() <= 1.0 and 0 <= labels.min() and labels.max() < 52
    assert len(seen) > 3 and min(seen) >= 1 and max(seen) <= 10          # one bucket per batch, several buckets over time
    only5 = du.synthetic_word_batches((32, 160, 1), 2, char_vec, 10, bucket_weights=[0, 0, 0, 0, 1, 0, 0, 0, 0, 0])
    assert next(only5)[1].shape == (2, 5)
    words = du.synthetic_random_words(10, char_vec, words_per_bucket=7)
    assert len(words) == 10 and all(len(words[i]) == 7 and all(len(w) == i + 1 for w in words[i]) for i in range(10))
    assert du.STAT_NAMES[:3] == ("r_loss_fake", "r_loss_real", "r_loss_balanced") and len(du.STAT_NAMES) == 16


def test_conv_tile_plan_and_bucket_shards_host_only():
    """Host-only planning of the tensor-core conv launch (no GPU): wave quantisation is answered by splitting the k-range of the
    tiles of a partial last wave, never for short-k launches; and the shards of the gradient-bucket all-reduce tile the bucket."""
    import ctypes as C
    abi = importlib.import_module("scrabble-gan_b200._abi")
    ops = importlib.import_module("scrabble-gan_b200.ops")
    lib = abi.load()

    def plan(n, h, w, ci, co, k, sms=148, enabled=1):
        d = ops.desc_conv_fwd(n, h, w, ci, co, k, k, "same", in_dt=abi.SG_BF16)
        bn, split, tiles = C.c_int(), C.c_int(), C.c_int()
        assert lib.sg_conv_tc_plan(C.byref(d), sms, enabled, C.byref(bn), C.byref(split), C.byref(tiles)) == 0, abi.last_error()
        return bn.value, split.value, tiles.value
    # D.B4 on the fused batch: 128 images of 4x10 = 40 full pixel tiles x 4 column tiles = 160 tiles on 148 SMs: the 12 tiles of
    # the second wave are split along k (K = 9216 = 144 k-blocks) instead of running a second wave at 8 % occupancy
    bn, split, tiles = plan(128, 4, 10, 1024, 1024, 3)
    assert (bn, tiles) == (256, 160) and 4 <= split <= 8 and 12 * split <= 148
    assert plan(128, 4, 10, 1024, 1024, 3, enabled=0)[1] == 1
    # the half batch: 80 tiles on 148 SMs -> every tile is split (more, shorter units fill the machine)
    bn, split, tiles = plan(64, 4, 10, 1024, 1024, 3)
    assert (bn, tiles) == (256, 80) and split >= 2
    assert plan(128, 8, 20, 1024, 1024, 3)[1] > 1                      # 640 tiles = 4.32 waves: the tail is split
    assert plan(148, 8, 20, 1024, 1024, 3, sms=185)[1] == 1            # 740 tiles on 185 SMs: whole waves, nothing to split
    assert plan(128, 16, 40, 64, 512, 3)[1] == 1                       # K = 576 (9 k-blocks): the exchange would cost more
    assert plan(2, 4, 10, 64, 64, 3)[1] == 1
    # bucket shards: 16-byte aligned starts, cover [0, n) exactly once
    for n, world in ((1000003, 2), (5, 8), (4096, 3), (37336384, 8)):
        shard = int(lib.sg_peer_bucket_shard(n, world))
        assert shard % 4 == 0 and shard * world >= n and shard * (world - 1) < n + 4 * world
        covered = sum(max(0, min(n, (r + 1) * shard) - min(n, r * shard)) for r in range(world))
        assert covered == n
