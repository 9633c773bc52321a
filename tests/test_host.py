"""CPU-only tests: the C-ABI library loads and exports every symbol include/dne.h declares (no compute calls
without a GPU), the host-side network layouts agree with the oracle's independent restatement, the synthetic
environments, the sharding / collective host logic under gloo at world_size 2, and the CPU baseline worker."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "dne.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(dne_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    from dne import _ffi as F
    lib = F.lib()                                   # dlopen + struct-size ABI check
    syms = _header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/dne.h but not exported by libdne.so"
    assert set(F.EXPORTS) <= set(syms)
    assert lib.dne_version() >= 100
    a, b = C.c_int(), C.c_int()
    lib.dne_abi_sizes(C.byref(a), C.byref(b))
    assert (a.value, b.value) == (C.sizeof(F.LayerDesc), C.sizeof(F.NetDesc))


def test_no_cpu_fallback():
    import torch
    from dne import _ffi as F
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    h = C.c_void_p()
    assert F.lib().dne_ctx_create(0, C.byref(h)) == -2           # DNE_ERR_CUDA, reported not fatal
    assert b"dne_ctx_create" in F.lib().dne_last_error()
    with pytest.raises(F.DneError):
        F.Context(0)
    with pytest.raises(F.DneError):
        F.ptr(torch.zeros(3))


def test_ws_queries_run_without_gpu():
    from dne import _ffi as F, nets
    for name, slots in (("LargeModel", 256), ("ESAtariPolicy", 256), ("MujocoPolicy", 10000)):
        net = nets.make_net(name)
        nb = C.c_size_t()
        assert F.lib().dne_forward_ws_bytes(C.byref(net.desc), slots, C.byref(nb)) == 0
        assert 0 < nb.value < 4 << 30


@pytest.mark.parametrize("name", ["LargeModel", "Model", "GAAtariPolicy", "ESAtariPolicy", "MujocoPolicy", "ModelVirtualBN"])
def test_layouts_match_oracle(name):
    from dne import _ffi as F, nets
    net, ref = nets.make_net(name), O.make_net(name)
    assert net.num_params == ref.num_params
    for l, lo in zip(net.layers, ref.layers):
        offs = {v.kind: v.offset for v in lo.vars}
        assert l.off_w == offs["w"] and l.off_b == offs.get("b", -1)
        assert l.off_beta == offs.get("beta", -1) and l.off_gamma == offs.get("gamma", -1)
        if lo.kind == "conv":
            assert (l.hout, l.pad) == (lo.hout, lo.pad_before)
    d = net.desc
    assert d.num_params == net.num_params and d.n_layers == len(net.layers)
    assert d.vbn_len == sum(2 * l.cout for l in net.layers if l.bn != F.BN_NONE)


def test_synthetic_envs():
    from dne.envs import SyntheticAtariEnv, SyntheticVectorEnv
    env = SyntheticAtariEnv(8, episode_len=5, seed=1, pin=False)
    assert env.obs_block(0, 8).shape == (8, 84, 84, 4) and env.obs_block(0, 8).dtype.__str__() == "torch.uint8"
    env.reset(np.arange(8))
    done_at = None
    for t in range(5):
        rew, done = env.step(np.arange(8), np.zeros(8, dtype=np.int32))
        assert set(np.unique(rew)) <= {0.0, 10.0}
        env.advance()
        if done.all():
            done_at = t
    assert done_at == 4
    env2 = SyntheticAtariEnv(4, episode_len=(3, 9), seed=2, pin=False)
    env2.reset(np.arange(4))
    assert ((env2.ep_len >= 3) & (env2.ep_len <= 9)).all()
    v = SyntheticVectorEnv(4, episode_len=3, pin=False)
    v.reset(np.arange(4))
    r, d = v.step(np.arange(4), np.zeros((4, 17), np.float32))
    assert r.shape == (4,) and not d.any()


def test_shard_bounds_cover_everything():
    from dne.shard import shard_bounds
    for n in (0, 1, 7, 500, 501):
        for world in (1, 2, 3, 8):
            got = [shard_bounds(n, r, world) for r in range(world)]
            assert got[0][0] == 0 and got[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(got, got[1:]))
            assert max(h - l for l, h in got) - min(h - l for l, h in got) <= 1


_GLOO_WORKER = r'''
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path[:0] = [%(root)r, os.path.join(%(root)r, "deep-neuroevolution_b200")]
from dne import shard
from oracle import oracle as O
rank, world, _ = shard.init_from_env("gloo")
assert world == %(world)d
# one "generation": every rank draws the same index stream, evaluates its shard (fake returns = f(index)),
# gathers, ranks, forms its partial gradient with the GLOBAL denominator, all-reduces.
seed = shard.broadcast_seed(None if rank == 0 else 12345)
rs = np.random.RandomState(seed)
noise = O.noise_table(50_000)
P, n = 257, 21
idx = rs.randint(0, len(noise) - P + 1, size=n).astype(np.int64)
lo, hi = shard.shard_bounds(n, rank, world)
local = torch.from_numpy(np.stack([np.sin(idx[lo:hi] * 0.001), np.cos(idx[lo:hi] * 0.002)], axis=1).astype(np.float32))
allr = shard.all_gather_rows(local, n).numpy()
expect = np.stack([np.sin(idx * 0.001), np.cos(idx * 0.002)], axis=1).astype(np.float32)
assert np.array_equal(allr, expect), "gather order"
proc = O.compute_centered_ranks(allr)
part = np.zeros(P, dtype=np.float64)
for i in range(lo, hi):
    part += np.float64(np.float32(proc[i, 0] - proc[i, 1])) * noise[idx[i]:idx[i] + P].astype(np.float64)
g = torch.from_numpy((part / allr.size).astype(np.float32))
shard.all_reduce_sum_(g)
ref = O.es_gradient(proc, noise, idx, P, dtype=np.float64)
assert np.abs(g.numpy() - ref).max() <= 1e-5 * np.abs(ref).max()
# rank 0's host-side object everywhere (the NS-ES archive entries / parent choice use it)
bc = shard.broadcast_object(np.arange(12, dtype=np.uint8).reshape(3, 4) + 7 if rank == 0 else None)
assert bc.dtype == np.uint8 and bc.shape == (3, 4) and int(bc[0, 0]) == 7
assert shard.broadcast_object(41 + rank) == 41
shard.barrier()
if rank == 0:
    print("GLOO_OK", seed)
dist.destroy_process_group()
'''


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_generation_bookkeeping_gloo_world2(tmp_path, world):
    """world 2 and 3: 21 units -> ragged shards (10/11, 7/7/7), padded all_gather, partial gradients all-reduced."""
    script = tmp_path / "w.py"
    script.write_text(_GLOO_WORKER % {"root": ROOT, "world": world})
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", str(29569 + world), str(script)],
                       capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "GLOO_OK" in r.stdout


def test_cpu_worker_forward_matches_oracle():
    from oracle import cpu_worker as W
    rs = np.random.RandomState(0)
    for name in ("LargeModel", "ESAtariPolicy"):
        net = O.make_net(name)
        theta = (rs.randn(net.num_params) * 0.05).astype(np.float32)
        for v in net.variables():
            if v.kind == "gamma":
                theta[v.offset:v.offset + v.size] = 1.0
        obs = rs.randint(0, 256, size=(3, 84, 84, 4)).astype(np.uint8)
        prep = W.prepare(net, theta)
        stats = None
        kw = {}
        if name == "ESAtariPolicy":
            ref = rs.randint(0, 256, size=(8, 84, 84, 4)).astype(np.uint8)
            _, stats = W.forward_prepared(net, prep, ref, is_ref=True)
            _, ostats = O.forward(net, theta, ref, is_ref=True)
            kw = dict(vbn_stats=ostats)
            for (m, v), (mo, vo) in zip(stats, ostats):
                np.testing.assert_allclose(m.numpy(), mo, rtol=1e-4, atol=1e-5)
                np.testing.assert_allclose(v.numpy(), vo, rtol=1e-3, atol=1e-6)
        got, _ = W.forward_prepared(net, prep, obs, vbn_stats=stats)
        want, _ = O.forward(net, theta, obs, **kw)
        np.testing.assert_allclose(got.numpy(), want, rtol=1e-3, atol=1e-4)


def test_cpu_worker_sample_runs():
    from oracle import cpu_worker as W
    net = O.make_net("Model")
    noise = O.noise_table(net.num_params + 10_000)
    theta = noise[:net.num_params].copy() * np.float32(0.05)
    steps, wall, t_setup, t_step = W.measure_workers("Model", noise, theta, [3, 77], 4, 0.005, 2)
    assert steps == 2 * 2 * 4 and wall > 0 and t_setup > 0 and t_step > 0
    secs, g = W.measure_master_update(noise, theta, np.array([1, 5, 9]), np.arange(6, dtype=np.float32).reshape(3, 2))
    assert g.shape == (net.num_params,) and g.dtype == np.float32


def test_tensorboard_event_file(tmp_path):
    """tabular_logger.py:17-52,150-152: every dumped row also lands in a TensorBoard event file (TFRecord framing with
    masked CRC-32C, Event / Summary protobufs written without TensorFlow).  CRC-32C known answer: "123456789" -> 0xE3069283."""
    import glob
    from es_distributed import tabular_logger as tl
    assert tl._crc32c(b"123456789") == 0xE3069283
    tl.set_quiet(True)
    tl.start(str(tmp_path))
    for i in range(3):
        tl.record_tabular("EpRewMean", 10.5 * i)
        tl.record_tabular("TimestepsSoFar", 1000 * (i + 1))
        tl.record_tabular("Note", "text values are skipped")
        tl.dump_tabular()
    tl.stop()
    files = glob.glob(os.path.join(str(tmp_path), "events.out.tfevents.*"))
    assert len(files) == 1
    ev = tl.read_tb_events(files[0])
    assert [s for s, _ in ev] == [1, 2, 3]
    assert ev[2][1] == {"EpRewMean": 21.0, "TimestepsSoFar": 3000.0}


def test_tabular_logger(tmp_path):
    from es_distributed import tabular_logger as tl
    tl.start(str(tmp_path))
    tl.record_tabular("EpRewMean", 1.5)
    tl.record_tabular("TimestepsSoFar", 10)
    tl.dump_tabular()
    tl.stop()
    txt = (tmp_path / "log.txt").read_text()
    assert "EpRewMean" in txt and "TimestepsSoFar" in txt


def test_policy_reinitialize_matches_oracle():
    """Policy.reinitialize (policies.py:42-44 + tf_util.py:122-158) == oracle.ga_reinitialize on the flat vector."""
    import torch
    from es_distributed import policies
    from dne import nets
    from oracle import oracle
    for name in ("LargeModel", "Model", "MujocoPolicy"):
        net, onet = nets.make_net(name), oracle.make_net(name)
        th = np.random.RandomState(3).randn(net.num_params).astype(np.float32)
        got = policies.reinitialize_flat(net, torch.from_numpy(th)).numpy()
        want = oracle.ga_reinitialize(onet, th)
        np.testing.assert_allclose(got, want, rtol=2e-6, atol=1e-7)
    with pytest.raises(AttributeError):
        policies.reinitialize_flat(nets.make_net("ESAtariPolicy"), torch.zeros(nets.make_net("ESAtariPolicy").num_params))


def _cpu_policy_shell(cls, net):
    """A Policy object without a CUDA context: enough state for the host-side snapshot / flat-vector plumbing."""
    import torch
    p = object.__new__(cls)
    p.args, p.kwargs = (), {}
    p.net, p.num_params = net, net.num_params
    p.hidden_dims = [l.cout for l in net.layers[:-1]]          # MujocoPolicy names its layers l0..l{n-1}, out
    p.trainable_variables = p._variable_table()
    p.all_variables = list(p.trainable_variables)
    p.device = torch.device("cpu")
    p._theta = torch.zeros(net.num_params)
    p.ob_mean = p.ob_std = None
    return p


def test_snapshot_roundtrip_set_all_vars_and_initialize_from(tmp_path):
    """policies.py:36-40,49-67,219-249: variable-name keyed snapshot, set_all_vars order, growing initialize_from."""
    from es_distributed import policies as PO
    from es_distributed.es import RunningStat
    from dne import nets
    rs = np.random.RandomState(0)
    small = _cpu_policy_shell(PO.MujocoPolicy, nets.make_net("MujocoPolicy", ob_dim=5, hidden=(8, 8), ac_dim=3))
    small.set_trainable_flat(rs.randn(small.num_params).astype(np.float32))
    small.set_ob_stat(rs.randn(5).astype(np.float32), np.abs(rs.randn(5)).astype(np.float32) + 0.5)
    fn = str(tmp_path / "snap.h5")
    small.save(fn)
    name, blob, data = PO._read_snapshot(fn)
    assert name == "MujocoPolicy" and set(data) == {n for n, _, _ in small.all_variables} | {"MujocoPolicy/ob_mean:0", "MujocoPolicy/ob_std:0"}
    for n, shp, off in small.all_variables:
        assert data[n].shape == tuple(shp)
        np.testing.assert_array_equal(data[n].reshape(-1), small.get_trainable_flat()[off:off + data[n].size])
    # set_all_vars: all_variables order
    twin = _cpu_policy_shell(PO.MujocoPolicy, small.net)
    twin.set_all_vars(*[data[n] for n, _, _ in twin.all_variables])
    np.testing.assert_array_equal(twin.get_trainable_flat(), small.get_trainable_flat())
    with pytest.raises(AssertionError):
        twin.set_all_vars(*[data[n] for n, _, _ in twin.all_variables][:-1])
    # initialize_from into a wider policy: leading sub-arrays filled, the rest untouched; ob stat -> RunningStat
    big = _cpu_policy_shell(PO.MujocoPolicy, nets.make_net("MujocoPolicy", ob_dim=5, hidden=(16, 16), ac_dim=3))
    base = rs.randn(big.num_params).astype(np.float32)
    big.set_trainable_flat(base.copy())
    st = RunningStat((5,), eps=1e-2)
    big.initialize_from(fn, ob_stat=st)
    got = big.get_trainable_flat()
    for (n, shp, off), (_, sshp, _) in zip(big.all_variables, small.all_variables):
        cur = got[off:off + int(np.prod(shp))].reshape(shp)
        ref = base[off:off + int(np.prod(shp))].reshape(shp).copy()
        ref[tuple(np.s_[:k] for k in sshp)] = data[n]
        np.testing.assert_array_equal(cur, ref)
    np.testing.assert_allclose(st.mean, data["MujocoPolicy/ob_mean:0"], rtol=1e-6)
    np.testing.assert_allclose(big.ob_mean.numpy(), data["MujocoPolicy/ob_mean:0"])
    other = _cpu_policy_shell(PO.LargeModelPolicy, nets.make_net("LargeModel"))
    with pytest.raises(AssertionError):
        other.initialize_from(fn)


def test_get_ref_batch_host_env():
    """es.py:105-113 on the batched host env: `batch_size` frames, uint8 84x84x4, copies (not views of the pool)."""
    from dne.envs import SyntheticAtariEnv
    from es_distributed import es
    env = SyntheticAtariEnv(2, episode_len=3, seed=0, pin=False)
    rb = es.get_ref_batch(env, batch_size=5)
    assert len(rb) == 5 and all(f.shape == (84, 84, 4) and f.dtype == np.uint8 for f in rb)
    rb[0][:] = 7
    assert not np.all(env.pool.numpy()[:, 0] == 7)


def test_vine_export_files(tmp_path):
    """es_modified.py:140-199: per-generation offspring cloud and parent row in the visual inspector's layout."""
    from es_distributed.es import vine_export_cloud, vine_export_parent
    rs = np.random.RandomState(0)
    cloud = [(rs.randint(0, 256, size=(5, 128)).astype(np.uint8), 30.0, 5, 1234, 0, 1),
             (rs.randint(0, 256, size=128).astype(np.uint8), 10.0, 7, 1234, 0, -1)]
    path = vine_export_cloud(str(tmp_path), 3, cloud)
    rows = [l.split() for l in open(os.path.join(path, "snapshot_offspring_0003.dat"))]
    assert len(rows) == 2 and len(rows[0]) == 128 + 5
    assert [float(x) for x in rows[0][128:]] == [30.0, 5.0, 1234.0, 0.0, 1.0]
    assert [int(float(x)) for x in rows[0][:128]] == cloud[0][0][-1].tolist()      # bc_vec[-1]: the final BC row
    evals = [(cloud[0][0], 30.0, 5, 0), (cloud[1][0], 10.0, 7, 0), (cloud[1][0], 22.0, 6, 0)]
    vine_export_parent(str(tmp_path), 3, evals, [30.0, 10.0, 22.0], 0.02)
    row = open(os.path.join(path, "snapshot_parent_0003.dat")).read().split()
    assert float(row[128]) == 22.0 and float(row[-1]) == 0.02                      # closest to int(mean) = 20 is 22


def test_make_env_real_ids_need_opt_in(monkeypatch):
    """ADVICE r01: a real env id must not silently run on the synthetic stand-in."""
    from dne import envs
    monkeypatch.delenv("DNE_ALLOW_SYNTHETIC_ENV", raising=False)
    for env_id in ("FrostbiteNoFrameskip-v4", "Humanoid-v1"):
        with pytest.raises(KeyError, match="allow_synthetic_env"):
            envs.make_env(env_id, 4)
        e = envs.make_env(env_id, 4, allow_synthetic=True, episode_len=3)
        assert getattr(e, "synthetic", False) and e.n_slots == 4
    assert envs.make_env("SyntheticAtariFrostbite", 2, episode_len=3).n_slots == 2       # explicit synthetic ids need no flag
    with pytest.raises(KeyError):
        envs.make_env("NoSuchEnv-v0", 2)



def test_bench_clock_sampler_and_reference_arm_contract(tmp_path):
    """bench.py pieces that run without a GPU: the clock sampler degrades to a labelled record when nvidia-smi is missing or
    prints nothing useful, and `--impl reference` prints one JSON line with the driver's keys (a tiny sample here)."""
    import importlib.util
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    s = bench.ClockSampler(0)
    s.start()
    rec = s.stop()
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(rec)
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--pop", "8", "--episode-len", "20", "--cpu-sample-steps", "2", "--noise-count", "6000000"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "env-steps/s" and line["higher_is_better"] is True
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["kind"] in ("port", "reference")
    assert line["value"] > 0 and line["config"]["workload"].startswith("frostbite_es")


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "d"],
                                  ["--workload", "mlp", "--dump-outputs", "d"]])
def test_bench_rejects_arguments_it_cannot_honour(argv, tmp_path):
    """No timed step to report, or an output dump the chosen arm does not produce: an argument error, before any work."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py")] + argv, capture_output=True, text=True,
                         timeout=120, cwd=tmp_path)
    assert out.returncode == 2 and out.stdout == "", out.stderr[-2000:]
    assert not os.path.exists(tmp_path / "d")


def test_normc_initialiser_matches_reference_bit_exactly():
    """tf_util.normc_initializer (tf_util.py:108-119) executed by tests/golden/make_golden_policies.py on the global numpy stream
    vs the package's initialiser on a RandomState with the same seed."""
    import hashlib
    from es_distributed.policies import _normc
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_policies.npz"))
    for i in range(4):
        shape, std = tuple(int(d) for d in g[f"normc.{i}.shape"]), float(g[f"normc.{i}.std"])
        arr = _normc(np.random.RandomState(1000 + i), shape, std)
        assert arr.dtype == np.float32 and arr.shape == shape
        np.testing.assert_array_equal(arr.reshape(-1)[:16], g[f"normc.{i}.head"])
        assert hashlib.sha1(np.ascontiguousarray(arr).tobytes()).hexdigest() == str(g[f"normc.{i}.sha1"])


def test_raw_env_host_logic_matches_reference_wrappers():
    """dne/raw_env.py RawFrameAtariEnv (no-op reset, frame skip with break on game over, fire reset, last-two-frames buffer, episode
    restart) + the oracle's warp / frame stack, against the reference's own wrap_deepmind stack executed on the same emulator
    (tests/golden/make_golden_wrappers.py): raw step counter, rewards, dones and the sha1 of every uint8 frame stack."""
    import hashlib
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import wrappers_common as WC
    from dne.raw_env import RawFrameAtariEnv
    from oracle import oracle as O
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_wrappers.npz"))
    emu = WC.RedOnlyEmulator(WC.EMU_SEED, frames=WC.EMU_FRAMES)
    env = RawFrameAtariEnv([emu], noop_max=30, seed=WC.ENV_SEED, device="cpu")
    assert env.fire_reset                                        # action 1 is FIRE
    stack = np.zeros((1, 84, 84, 4), dtype=np.uint8)
    ev = [0]

    def check(kind, r, d):
        nonlocal stack
        i = ev[0]
        frame = O.warp_frame_cpu(np.maximum(env._raw_np[0, 0], env._raw_np[0, 1]))[None]       # max of the last two raw frames, then warp
        stack = O.max_and_stack(frame, frame, stack, env.fresh[:1].astype(bool), mode="cpu")
        env.fresh[:] = 0
        assert int(g["kind"][i]) == kind and int(g["emu_t"][i]) == emu.t, (i, kind, emu.t, int(g["emu_t"][i]))
        assert float(g["reward"][i]) == float(r) and bool(g["done"][i]) == bool(d), i
        if i == 0:
            np.testing.assert_array_equal(stack[0], g["first_stack"])
        assert hashlib.sha1(np.ascontiguousarray(stack[0]).tobytes()).hexdigest() == str(g["sha1"][i]), i
        ev[0] += 1

    env.reset([0])
    check(0, 0.0, False)
    for a in WC.ACTIONS:
        rew, done = env.step([0], [a])
        check(1, rew[0], done[0])
        if done[0]:
            env.reset([0])
            check(0, 0.0, False)
    assert ev[0] == len(g["kind"])


def test_vine_export_bytes_match_reference_functions(tmp_path):
    """The exact bytes es_modified.py `master_extract_cloud` / `master_extract_parent` wrote for the seeded input of
    tests/golden/make_golden_vine.py (the reference functions themselves, executed in the build container)."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_golden_vine as G
    from es_distributed.es import vine_export_cloud, vine_export_parent
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vine.npz"))
    _, cloud, evals, rets = G.inputs()
    path = vine_export_cloud(str(tmp_path), 7, cloud)
    vine_export_parent(str(tmp_path), 7, [e[:4] for e in evals], rets, evals[0][4])
    assert open(os.path.join(path, "snapshot_offspring_0007.dat"), "rb").read() == g["offspring"].tobytes()
    assert open(os.path.join(path, "snapshot_parent_0007.dat"), "rb").read() == g["parent"].tobytes()
    assert path.endswith(os.path.join("snapshots", "snapshot_gen_0007"))
    assert {"snapshot_offspring_0007.dat", "snapshot_parent_0007.dat"} <= {str(f) for f in g["files"]}


def test_log_txt_bytes_match_reference_logger(tmp_path):
    """log.txt of the package's tabular_logger vs the bytes the reference's own tabular_logger.py wrote for the same scripted calls
    (tests/golden/make_golden_logger.py): table layout, %-8.3g values, key truncation, back-to-back `log` strings."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_golden_logger as G
    from es_distributed import tabular_logger as L
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_logger.npz"))
    L.set_quiet(True)
    try:
        L.start(str(tmp_path))
        G.script(L)
    finally:
        L.stop()
        L.set_quiet(False)
    assert open(os.path.join(str(tmp_path), "log.txt"), "rb").read() == g["log_txt"].tobytes()


def test_logged_rows_carry_the_reference_keys_in_reference_order():
    """log.txt rows of the GA / NS-ES / RS / ES masters: every key the reference's master records, in its order
    (tests/golden/ref_log_keys.json = the record_tabular keys extracted from the reference sources), then the engine's extras.
    The masters only run on a GPU, so this checks (a) es.reference_row itself and (b) statically, that each master passes a value
    for every reference key that has no default -- a missing one would be a KeyError at run time."""
    import ast
    import json
    from es_distributed import es as ES
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref = json.load(open(os.path.join(root, "tests", "golden", "ref_log_keys.json")))
    for kind in ("ga", "nses", "rs"):
        assert ES.REF_ROW_KEYS[kind] == ref[kind]
        src = open(os.path.join(root, "deep-neuroevolution_b200", "es_distributed", kind + ".py")).read()
        passed = set()
        for node in ast.walk(ast.parse(src)):                  # keyword names of the `stats = dict(...)` call of the master
            if isinstance(node, ast.Assign) and getattr(node.targets[0], "id", None) == "stats" and isinstance(node.value, ast.Call) \
                    and getattr(node.value.func, "id", None) == "dict":
                passed |= {k.arg for k in node.value.keywords}
        need = [k for k in ref[kind] if k not in ES._ROW_DEFAULTS and k != "UniqueWorkers"]
        assert set(need) <= passed, (kind, sorted(set(need) - passed))
        assert 'reference_row("%s", stats, world)' % kind in src
        row = ES.reference_row(kind, dict({k: 1.0 for k in need}, Extra=5, NoveltyMean=2.0), world=3)
        assert list(row)[:len(ref[kind])] == ref[kind] and list(row)[len(ref[kind]):] == ["Extra", "NoveltyMean"]
        assert row["UniqueWorkers"] == 3 and row["EvalEpCount"] == 0 and np.isnan(row["EvalEpRewMean"])
    # ES: the master builds its row key by key in the reference's order
    es_src = open(os.path.join(root, "deep-neuroevolution_b200", "es_distributed", "es.py")).read()
    call = next(n for n in ast.walk(ast.parse(es_src)) if isinstance(n, ast.Call) and getattr(n.func, "id", None) == "GenerationStats")
    assert [k.arg for k in call.keywords] == ref["es"]
