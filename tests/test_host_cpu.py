"""CPU tests of the host-side mirror of the reference interface (no device work): layer walk / weight tables, npz
weight I/O and shape checking, the sample() diagnostic form, and the multi-GPU sharding logic -- the latter with real
world_size-2 gloo process groups (SURVEY 8e: independent sample batches, no collective on the data path)."""
import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import b200dm
from b200dm import sharding, weights as Wt
from oracle import init as OI, sampler as OS
from oracle.schedule import Betas as OBetas
from oracle.unet import UNet as OUNet
from oracle import first_stage as OF


# ----------------------------------------------------------------------------------------- layer walk / weight tables
@pytest.mark.parametrize("cond,S,C", [(False, 16, 8), (True, 32, 256), (True, 8, 16)])
def test_param_spec_equals_oracle_walk(cond, S, C):
    """The product's weight table (names, Keras-layout shapes, construction order) and the oracle's independent walk of
    build_model (dm3d.py:294-376 / conditional_dm3d.py:324-415) agree entry by entry."""
    net = b200dm.build_model(S, C, [64, 128, 256], [False, False, True, True], context_dim=1 if cond else None)
    ou = OUNet(S, C, [64, 128, 256], [False, False, True, True], first_conv_channels=32 if cond else 64, conditional=cond)
    assert [(n, tuple(s)) for n, s, _ in net.spec] == [(n, tuple(s)) for n, s, _ in ou.spec()]
    assert net.count_params() == sum(int(np.prod(s)) for _, s, _ in ou.spec())


def test_layer_counts_match_survey_appendix_a():
    """SURVEY 3.2: R=2, three widths -> 17 ResidualBlocks, 6 attention sites, 2 down + 2 up, 40 3^3 convs."""
    net = b200dm.build_model(32, 256, [64, 128, 256], [False, False, True, True], context_dim=1)
    kinds = [b["kind"] for b in net.blocks]
    assert kinds.count("res") == 17 and kinds.count("attn") == 6 and kinds.count("down") == 2 and kinds.count("up") == 2
    conv3 = sum(1 for n, s, _ in net.spec if n.endswith(".kernel") and len(s) == 5 and s[0] == 3)
    conv1 = sum(1 for n, s, _ in net.spec if n.endswith(".shortcut.kernel"))
    assert conv3 == 40 and conv1 == 12
    unc = b200dm.build_model(16, 8, [64, 128, 256], [False, False, True, True])
    assert sum(1 for n, s, _ in unc.spec if n.endswith(".shortcut.kernel")) == 11
    # duplicate widths: the reference compares widths by VALUE (dm3d.py:343) -> the downsample (and its skip push) is
    # dropped and the up path pops an empty skip stack, in the reference as here
    with pytest.raises(IndexError):
        b200dm.build_model(16, 8, [64, 64], [False, False])


def test_build_model_signature_and_errors():
    with pytest.raises(ValueError):
        b200dm.build_model(8, 8, [64], [False], has_cross_attention=[True])        # reference: context_dim required
    net = b200dm.build_model(8, 8, [64, 128], [False, True], num_res_blocks=1, norm_groups=8, interpolation="nearest")
    assert net.cfg.first_conv_channels == 64 and not net.cfg.conditional


def test_weights_roundtrip_and_shape_check(tmp_path):
    net = b200dm.build_model(8, 8, [64, 128, 256], [False, False, True, True])
    P = OI.make_params(OUNet(8, 8, [64, 128, 256], [False, False, True, True]).spec(), 3, "stress")
    p = tmp_path / "w.npz"
    Wt.save_npz(p, P)
    net.load_weights(str(p))
    for k, v in P.items():
        assert torch.equal(net.params[k], v)
    bad = dict(P)
    bad["in.kernel"] = bad["in.kernel"].permute(4, 3, 0, 1, 2).contiguous()                  # torch layout: must be rejected
    with pytest.raises(ValueError):
        net.set_weights(bad)
    del bad["in.kernel"]
    with pytest.raises(KeyError):
        net.set_weights(bad)


def test_keras_initialisers():
    net = b200dm.build_model(8, 8, [64, 128, 256], [False, False, True, True])
    P = net.params                                                                             # mode='keras'
    w = P["down.0.res.0.conv1.kernel"]
    lim = np.sqrt(3.0 / ((27 * 64 + 27 * 64) / 2))
    assert w.abs().max() <= lim and w.abs().max() > 0.9 * lim                                  # VarianceScaling(1, fan_avg, uniform)
    assert P["down.0.res.0.conv2.kernel"].abs().max() < 1e-5                                   # kernel_init(0.0) -> scale 1e-10
    assert torch.equal(P["out.norm.gamma"], torch.ones(64)) and torch.equal(P["out.norm.var"], torch.ones(64))


def test_first_stage_tables_match_oracle():
    vq = b200dm.VQGAN(num_channels=(32, 64, 128), num_embeddings=256, embedding_dim=64)
    od = OF.AttnCpDecoder(64, 1, (32, 64, 128))
    assert [(n, tuple(s)) for n, s, _ in vq.decoder.spec] == [(n, tuple(s)) for n, s, _ in od.spec()]
    mv = b200dm.VQVAE(in_channels=1, out_channels=1, num_channels=(32, 64), num_res_channels=(32, 64), num_res_layers=2,
                      num_embeddings=256, embedding_dim=64, latent_size=4)
    om = OF.MonaiDecoder(64, 1, (32, 64), 2, (32, 64), 4)
    assert [(n, tuple(s)) for n, s, _ in mv.decoder.spec] == [(n, tuple(s)) for n, s, _ in om.spec()]


@pytest.mark.parametrize("variant", ["vqgan", "gnorm", "stride"])
def test_vqgan_family_tables_match_oracle(variant):
    vq = b200dm.VQGAN(in_channels=2, out_channels=2, num_channels=(32, 64, 128), num_res_layers=3, num_res_channels=(32, 64, 128),
                      num_embeddings=256, embedding_dim=64, variant=variant)
    od = OF.VqganFamilyDecoder(variant, 64, 2, (32, 64, 128), 3, (32, 64, 128), 16)
    assert [(n, tuple(s)) for n, s, _ in vq.decoder.spec] == [(n, tuple(s)) for n, s, _ in od.spec()]
    assert vq.quantizer.layout == ("DK" if variant == "vqgan" else "KD")      # vqgan.py:164-170 vs vqgan_gnorm.py:164-170
    # an out_channels=1 gnorm/stride decoder asks for GroupNormalization(groups=0): unbuildable in the reference as well
    if variant != "vqgan":
        assert od.up_norm(1)[1] == 0


# ----------------------------------------------------------------------------------------- DiffusionModel host surface
def _args(T=20, n=1, bs=2):
    return types.SimpleNamespace(timesteps=T, num_gpus=n, kernel_resize=False, bs=bs)


def test_diffusion_model_surface_and_sample_form():
    dm = b200dm.DiffusionModel(8, 256, 8, None, _args())
    for attr in ("timesteps", "b", "network", "encoder", "quantizer", "decoder", "vqvae_trainer"):
        assert hasattr(dm, attr)
    ob = OBetas(20)
    assert np.array_equal(dm.b.alpha_bar, ob.alpha_bar) and np.array_equal(dm.b.sqrt_one_minus_alpha_bar, ob.sqrt_one_minus_alpha_bar)
    x, e = OI.normal((2, 8, 8, 8, 8), 1), OI.normal((2, 8, 8, 8, 8), 2)
    for t in (19, 7, 0):
        mean, var = dm.sample(x, e, torch.tensor([t, t]), x.shape)        # reference signature (dm3d.py:477)
        om, ov = OS.sample(ob, x, e, t)
        assert torch.equal(mean, om) and float(var.reshape(-1)[0]) == float(ov) and var.shape == (2, 1, 1, 1, 1)
    cdm = b200dm.ConditionalDiffusionModel(8, 64, 16, None, _args())
    assert cdm.network.cfg.conditional and cdm.network.cfg.first_conv_channels == 32
    assert cdm.quantizer.num_embeddings == 64 and cdm.quantizer.embedding_dim == 16            # conditional_dm3d.py:444-445
    assert dm.quantizer.num_embeddings == 1024 and dm.quantizer.embedding_dim == 256           # dm3d.py:405-406 (hard-coded)


# ----------------------------------------------------------------------------------------- sharding
def test_partition_properties():
    for total in (0, 1, 7, 8, 64, 1001):
        for world in (1, 2, 3, 4, 8):
            parts = [sharding.partition(total, world, r) for r in range(world)]
            assert sum(c for _, c in parts) == total
            assert parts[0][0] == 0 and all(parts[i][0] + parts[i][1] == parts[i + 1][0] for i in range(world - 1))
            assert max(c for _, c in parts) - min(c for _, c in parts) <= 1
    with pytest.raises(ValueError):
        sharding.partition(8, 2, 2)


class _FakeModel:
    """Records the generate() arguments; returns latents that depend only on (seed, global sample index), like the Philox stream."""

    def generate(self, shape, seed=0, sample_id0=0, context=None, **kw):
        ids = torch.arange(sample_id0, sample_id0 + shape[0], dtype=torch.float32)
        base = ids.view(-1, *([1] * (len(shape) - 1))).expand(*shape).clone() * 10 + seed
        if context is not None:
            base += torch.tensor(context, dtype=torch.float32).view(-1, *([1] * (len(shape) - 1)))
        return base


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, total, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ctx = [i % 2 for i in range(total)]
        lat, start = sharding.generate_sharded(_FakeModel(), total, (2, 2, 2, 3), context_ids=ctx, seed=5)
        # the data path has no collective; the TEST gathers on the host to compare with the single-process result
        out = [None] * world
        dist.all_gather_object(out, (start, None if lat is None else lat.numpy()))
        # bench.py's timing reduction: max over ranks
        t = torch.tensor([float(rank + 1)], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if rank == 0:
            q.put((out, float(t.item())))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("total", [8, 5, 1])
def test_sharded_generate_world2_gloo_matches_single_process(total):
    world, port = 2, _free_port()
    ctxm = mp.get_context("spawn")
    q = ctxm.SimpleQueue()
    procs = [ctxm.Process(target=_worker, args=(r, world, port, total, q)) for r in range(world)]
    for p in procs:
        p.start()
    out, tmax = q.get()
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert tmax == 2.0
    parts = [a for _, a in sorted(out, key=lambda e: e[0]) if a is not None]
    got = np.concatenate(parts, 0)
    ctx = [i % 2 for i in range(total)]
    want = _FakeModel().generate((total, 2, 2, 2, 3), seed=5, sample_id0=0, context=ctx).numpy()
    assert np.array_equal(got, want)              # identical regardless of how many ranks produced it


def test_tuning_switches_need_the_tuning_gate(monkeypatch):
    """Experiment switches of the Python layer are ignored unless B200DM_TUNING=1."""
    from b200dm import _lib as L
    monkeypatch.delenv("B200DM_TUNING", raising=False)
    monkeypatch.setenv("B200DM_CHAINS", "4")
    assert L.tuning_env("B200DM_CHAINS", "1") == "1"
    monkeypatch.setenv("B200DM_TUNING", "1")
    assert L.tuning_env("B200DM_CHAINS", "1") == "4"


def test_test_dm_script_flags(tmp_path):
    """tools/test_dm.py mirrors the --test_dm invocation of main.py:428-448 / main_conditional_dm.py:195-215: the reference's flag
    names parse with the reference's defaults, the modes outside the sampling path are accepted by the parser and refused at run
    time (no GPU needed for either)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("test_dm_tool", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "test_dm.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    a = mod.build_parser().parse_args(["--test_dm", "--suffix", "exp7", "--test_epoch", "100", "--timesteps", "300", "--vqvae_load_ckpt", "vq.ckpt"])
    assert a.test_dm and a.suffix == "exp7" and a.test_epoch == 100 and a.timesteps == 300 and a.vqvae_load_ckpt == "vq.ckpt"
    assert a.latent_size == 16 and a.num_embed == 256 and a.latent_channels == 64 and a.num_volumes == 10   # main.py:432-438, dm3d.py:539
    assert a.lbs == 5 and a.num_gpus == 2 and not a.kernel_resize                                            # main.py:451-505 defaults
    b = mod.build_parser().parse_args(["--train_dm", "--suffix", "x"])
    with pytest.raises(SystemExit, match="--test_dm only"):
        mod.run(b)
    img = np.arange(12, dtype=np.float32).reshape(3, 4)
    path = str(tmp_path / "slice.pgm")
    mod.write_pgm(path, img)
    raw = open(path, "rb").read()
    assert raw.startswith(b"P5\n4 3\n255\n") and len(raw) == len(b"P5\n4 3\n255\n") + 12 and raw[-1] == 255 and raw[len(b"P5\n4 3\n255\n")] == 0
