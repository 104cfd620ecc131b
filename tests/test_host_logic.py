"""CPU tests of the host-side logic: schedule tables, factory surface, state-dict handling, document sharding and the
world_size-2 gloo path."""
import os

import numpy as np
import pytest
import torch

from oracle import dvd_oracle as O
from oracle import synth


def test_schedule_matches_oracle_and_golden(golden_dir):
    from dvd_b200.sampler import create_gaussian_diffusion
    ka = np.load(os.path.join(golden_dir, "known_answers.npz"))
    for S, key in ((3, "betas3"), (10, "betas10")):
        d = create_gaussian_diffusion(steps=S, noise_schedule="cosine", predict_xstart=True, rescale_timesteps=True,
                                      rescale_learned_sigmas=True, timestep_respacing="")
        np.testing.assert_allclose(d.betas, ka[key], atol=1e-15)
        sch = O.Schedule(S)
        t_scaled, t_emb, a, b = d._plan()
        assert len(t_scaled) == S and t_scaled[-1] == 0.0
        for it, i in enumerate(range(S - 1, -1, -1)):
            assert t_scaled[it] == sch.scaled_t(i)
            assert t_emb[it] == O.remap_t(sch.scaled_t(i))
            np.testing.assert_allclose((a[it], b[it]), sch.ddim_ab(i), atol=1e-15)
    # S = 10: exact 600 / 300 fall through the strict thresholds
    d10 = create_gaussian_diffusion(steps=10, noise_schedule="cosine", predict_xstart=True, rescale_timesteps=True)
    ts, te, _, _ = d10._plan()
    assert ts[:5] == [900.0, 800.0, 700.0, 600.0, 500.0] and te[:5] == [2.0, 2.0, 2.0, 600.0, 1.0]
    assert te[6] == 300.0 and te[7] == 200.0


def test_linear_schedule_and_respacing():
    from dvd_b200.sampler import create_gaussian_diffusion, space_timesteps
    assert space_timesteps(10, [10]) == set(range(10))
    assert space_timesteps(100, "ddim10") == set(range(0, 100, 10))
    assert space_timesteps(300, [10, 15, 20]) is not None
    d = create_gaussian_diffusion(steps=100, noise_schedule="linear", predict_xstart=True, rescale_timesteps=True, timestep_respacing="ddim10")
    assert d.num_timesteps == 10 and d.timestep_map == list(range(0, 100, 10))
    assert d.scaled_t(9) == 900.0
    with pytest.raises(NotImplementedError):
        create_gaussian_diffusion(steps=3, noise_schedule="cosine", predict_xstart=False)


def test_factory_signature_matches_reference_call():
    """val_TDiff.py:46-51 calls create_model_and_diffusion(**args_to_dict(settings, defaults.keys()), device=..., train_mode=..., tv=...)."""
    from dvd_b200.script_util import args_to_dict, create_model_and_diffusion, model_and_diffusion_defaults

    class Env:      # admin/local.py values
        image_size = 64; num_channels = 128; num_res_blocks = 3; num_heads = 4; num_heads_upsample = -1
        attention_resolutions = "16,8"; dropout = 0.0; learn_sigma = False; sigma_small = False; class_cond = False
        diffusion_steps = 3; noise_schedule = "cosine"; timestep_respacing = ""; use_kl = False; predict_xstart = True
        rescale_timesteps = True; rescale_learned_sigmas = True; use_checkpoint = False; use_scale_shift_norm = True

    class S:
        env = Env()
    model, diffusion = create_model_and_diffusion(**args_to_dict(S, model_and_diffusion_defaults().keys()), device="cpu",
                                                  train_mode="stage_1_dit_cross", tv=True)
    assert diffusion.num_timesteps == 3 and hasattr(diffusion, "ddim_sample_loop")
    diffusion.settings = S          # val_TDiff.py:52
    with pytest.raises(ValueError):
        create_model_and_diffusion(**args_to_dict(S, model_and_diffusion_defaults().keys()), device="cpu", train_mode="stage_1", tv=True)


def test_state_dict_surface():
    from dvd_b200.model import DiT
    from dvd_b200.weights import required_keys
    spec = synth.state_dict_spec()
    assert set(required_keys()) <= set(spec)
    full = synth.make_state_dict(1234)                    # all 369 reference keys incl. dead blocks 0..10
    m = DiT(precision="fp32")
    res = m.load_state_dict(full, strict=False)
    assert res.missing_keys == [] and list(m.state_dict().keys()) == list(full.keys())
    n_params = sum(p.numel() for p in m.parameters())     # val_TDiff.py:35-38 prints this
    assert n_params > 150e6
    live = {k: v for k, v in full.items() if k in set(required_keys())}
    m.load_state_dict(live, strict=True)
    broken = dict(live); broken.pop("final_layer2.linear.weight")
    with pytest.raises(RuntimeError, match="Missing key"):
        m.load_state_dict(broken, strict=True)
    assert m.load_state_dict(broken, strict=False).missing_keys == ["final_layer2.linear.weight"]
    assert m.eval() is m and m.cpu() is m


def test_sampler_rejects_unsupported_configs():
    from dvd_b200.model import DiT
    from dvd_b200.sampler import create_gaussian_diffusion
    d = create_gaussian_diffusion(steps=3, noise_schedule="cosine", predict_xstart=True, rescale_timesteps=True)
    m = DiT(precision="fp32")
    kw = {"iter": True}
    with pytest.raises(NotImplementedError):
        d.ddim_sample_loop(m, (1, 2, 64, 64), clip_denoised=False, model_kwargs=kw, eta=0.5, n_batch=2, time_variant=True)
    with pytest.raises(NotImplementedError):
        d.ddim_sample_loop(m, (1, 2, 64, 64), clip_denoised=True, model_kwargs=kw, eta=0.0, n_batch=2, time_variant=True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        d.ddim_sample_loop(m, (1, 2, 64, 64), clip_denoised=False, model_kwargs=kw, eta=0.0, n_batch=2, time_variant=True)
    with pytest.raises(TypeError):
        d.ddim_sample_loop(torch.nn.Linear(1, 1), (1, 2, 64, 64), clip_denoised=False, model_kwargs=kw, eta=0.0, n_batch=2, time_variant=True)


def test_document_sharding():
    from dvd_b200.dist import batches, shard_documents
    for n, w in ((64, 8), (65, 8), (3, 8), (0, 2)):
        parts = [shard_documents(n, r, w) for r in range(w)]
        assert sorted(sum(parts, [])) == list(range(n))
        assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1
    assert batches([0, 1, 2, 3, 4], 2) == [[0, 1], [2, 3], [4]]
    with pytest.raises(ValueError):
        shard_documents(4, 2, 2)


def _gloo_worker(rank, world, port, q):
    os.environ.update({"RANK": str(rank), "WORLD_SIZE": str(world), "LOCAL_RANK": str(rank), "MASTER_ADDR": "127.0.0.1",
                       "MASTER_PORT": str(port)})
    import torch.distributed as dist
    from dvd_b200 import dist as D
    r, w, dev = D.setup_dist("gloo")
    mine = D.shard_documents(7, r, w)
    times = {d: 0.01 * (d + 1) for d in mine}            # stand-in for per-document device timings
    allt = {}
    for part in D.gather_metrics(times):
        allt.update(part)
    mx = D.max_over_ranks(float(sum(times.values())), torch.device("cpu"))
    D.barrier()
    q.put((r, mine, sorted(allt), mx))
    dist.destroy_process_group()


def test_world_size_2_gloo_sharding_and_gather():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res[0][1] == [0, 2, 4, 6] and res[1][1] == [1, 3, 5]
    assert res[0][2] == res[1][2] == list(range(7))        # every rank sees every document's timing
    assert abs(res[0][3] - res[1][3]) < 1e-12 and abs(res[0][3] - 0.16) < 1e-9     # max over ranks: 0.01*(1+3+5+7)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the UNMODIFIED reference from baseline/_ref or /root/reference on the host cores; the oracle port only
    when neither tree exists) prints ONE JSON line carrying the keys of the measurement contract; no GPU, no compiled extension involved."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--height", "96", "--width", "128"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "docs/s" and d["value"] > 0 and "workload" in d["config"]
    from oracle import ref_harness as RH
    assert d["cpu_baseline"]["kind"] == ("reference" if RH.available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert abs(d["ms_per_step"] * d["steps"] / 1e3 - d["steps"] / d["value"]) < 1e-6          # whole documents, no extrapolation
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_bench_dump_outputs_whole_or_fixed_sample(tmp_path):
    """bench.py --dump-outputs: small arrays are written whole in float32; one past the 64 MiB budget becomes the same seeded
    sample of distinct positions on every call, and the files stay under the budget together."""
    import bench
    g = torch.Generator().manual_seed(1)
    map64 = torch.rand(2, 2, 64, 64, generator=g) * 2 - 1
    image = torch.randint(0, 256, (2, 1500, 2000, 3), generator=g, dtype=torch.uint8)        # 72 MiB as float32
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"map64": map64, "image": image})
    m = np.load(tmp_path / "a" / "map64.npy")
    assert m.dtype == np.float32 and np.array_equal(m, map64.numpy())
    ia, ib = np.load(tmp_path / "a" / "image.npy"), np.load(tmp_path / "b" / "image.npy")
    assert ia.dtype == np.float32 and ia.ndim == 1 and np.array_equal(ia, ib)
    assert set(np.unique(ia)) <= set(range(256)) and len(np.unique(ia)) == 256
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    ramp = torch.arange(bench.DUMP_BYTES // 4 - 1000, dtype=torch.int32)      # just past the budget, every value exact in float32
    bench.dump_outputs(str(tmp_path / "r"), {"ramp": ramp})
    r = np.load(tmp_path / "r" / "ramp.npy")
    assert r.size < ramp.numel() and np.all(np.diff(r) > 0)                          # sorted positions, none drawn twice
    small = torch.randint(0, 256, (1, 96, 128, 3), generator=g, dtype=torch.uint8)
    bench.dump_outputs(str(tmp_path / "c"), {"map64": map64[:1], "image": small})
    assert np.array_equal(np.load(tmp_path / "c" / "image.npy"), small.float().numpy())


def test_committed_bench_lines_carry_the_contract():
    """profiles/r1_bench_lines.jsonl: every line of our arm has value / e2e / roofline / clocks / gpu_launches."""
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n = 0
    for l in open(os.path.join(root, "profiles", "r1_bench_lines.jsonl")):
        d = json.loads(l)
        if d.get("impl") == "reference":
            continue
        n += 1
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data", "config",
                  "e2e", "gpu_launches", "clocks", "roofline"):
            assert k in d, k
        assert d["gpu_launches"] > 0 and d["warmup"] >= 3 and d["scaling"] == "weak"
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
        assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert n >= 5


def test_split_f16_pair_reconstructs_weights():
    """weights.split_f16: hi + lo reproduces an fp32 weight to ~2^-22 relative (the fp16 pair of the two-pass q|k|v GEMM)."""
    import torch
    from dvd_b200.weights import split_f16, split_bf16
    g = torch.Generator().manual_seed(3)
    w = torch.randn(256, 384, generator=g) * 0.05
    hi, lo = split_f16(w)
    assert hi.dtype == torch.float16 and lo.dtype == torch.float16
    err = (hi.float() + lo.float() - w).abs().max() / w.abs().max()
    assert float(err) < 2e-6
    bh, bl = split_bf16(w)
    assert float((bh.float() + bl.float() - w).abs().max() / w.abs().max()) < 2e-5
    import pytest
    with pytest.raises(ValueError):
        split_f16(torch.full((2, 2), 1e5))
