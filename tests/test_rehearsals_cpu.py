"""Rehearsals: host-side code that will next run on a GPU, run here first against tests/engine_double.py (the CPU
oracle behind the Engine methods / C-ABI calls involved, decoding posted byte-form frames with `mrq_unpack8`, the
same inline decode the device kernel runs):

  * bench.py's whole N = 1 main path (`run_ours`) with its end-to-end leg (`bench_e2e`): the REAL orchestration code —
    frame building with `mrq_pack8` on a packer thread, the pipelined post / tick / drain loop, the commit-advance
    accumulation and the equality verdict (including a deliberately wrong decode, to show the verdict has teeth) —
    and the driver-facing contract of the JSON line it prints;
  * the bodies of the GPU tests written after round 1's GPU budget was spent (tests/test_zz_packed8_gpu.py,
    tests/test_zz_kat_gpu.py), so that when they first meet hardware a failure implicates the device path alone,
    not the test code.

What this cannot cover is the device kernels themselves and real PCIe timing."""
import argparse
import json

import pytest

from engine_double import FakeEngine, FakePinned


def _bench_on_the_double(monkeypatch, eng_cls, G=2048):
    import torch

    import bench
    import raftsql_b200
    import raftsql_b200.packed as packed

    made = []

    def make(*a, **kw):
        made.append(eng_cls(*a, **kw))
        return made[-1]

    monkeypatch.setattr(bench, "G_TOTAL", G)
    monkeypatch.setattr(raftsql_b200, "Engine", make)
    monkeypatch.setattr(packed, "PinnedArray", FakePinned)
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a: None)
    monkeypatch.setattr(bench, "bench_quorum_kernel", lambda *a, **k: {"bound": "hbm", "achieved": 1.0, "peak": 2.0, "frac": 0.5})
    monkeypatch.setattr(bench, "cpu_reference_ticks", lambda *a, **k: (80.0, 8, 3, 0.04, None))
    monkeypatch.setenv("MRQ_BENCH_REPS", "2")
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    return bench, made


def _args(**kw):
    d = dict(gpus=1, steps=6, warmup=3, impl="ours", gather="fused", l2=None, graph="auto", inbox="compact", write_back="every-tick",
             weak=False)
    d.update(kw)
    return argparse.Namespace(**d)


def test_rehearse_bench_main_path_e2e_leg_and_line_assembly(monkeypatch, capsys):
    """`python bench.py` at N = 1 on the engine double: the REAL run_ours() and bench_e2e() — dry run, byte frames posted to
    their slots, the repetitions of [rewind, warm-up, K timed ticks], the variant legs, and the end-to-end leg with its
    packer thread (mrq_pack8 on the clock), the pipelined post / tick / drain loop, the commit-advance accumulation and
    the equality verdict — one JSON line with the driver-facing contract."""
    from engine_double import FakeBenchEngine

    monkeypatch.delenv("MRQ_BENCH_FAST", raising=False)
    bench, made = _bench_on_the_double(monkeypatch, FakeBenchEngine)
    bench.run_ours(_args())
    out = capsys.readouterr().out.strip().splitlines()
    assert len(out) == 1, "exactly one JSON line"
    line = json.loads(out[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "clocks", "gpu_launches", "variants", "ms_per_step_reps"):
        assert k in line, k
    assert line["metric"] == "raft_ticks_per_sec_1Mx5" and line["unit"] == "ticks/s" and line["n_gpus"] == 1
    assert line["steps"] == 6 and line["warmup"] == 3 and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["value"] > 0 and abs(line["value"] - 1e3 / line["ms_per_step"]) < 1e-6 * line["value"]
    assert len(line["ms_per_step_reps"]) == 2 and line["config"]["tick_mode"] == 4 and "0 escaped" in line["config"]["inbox"]
    assert set(("bound", "achieved", "peak", "unit", "frac", "traffic")) <= set(line["roofline"])
    assert abs(line["roofline"]["frac"] - line["roofline"]["achieved"] / line["roofline"]["peak"]) < 1e-12
    assert set(("value", "unit", "cores", "kind", "sample")) <= set(line["cpu_baseline"])
    e = line["e2e"]
    assert set(("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "pack_us_per_tick", "preencoded")) <= set(e)
    assert e["encode_in_timed_region"] is True and e["equals_wide_form"] is True and e["escapes"] == 0
    assert e["h2d_bytes_per_step"] == 2048 * bench.R and e["d2h_bytes_per_step"] == 2048 and e["steps"] == 6
    assert "mrq_pack8" in e["api"] and "tick mode 4" in e["api"]
    assert set(line["variants"]) >= {"compact_per_tick_launches", "compact_batched_write_through", "wide_inbox_mode0"}
    assert "workload" in line["config"] and "model" not in line["config"]
    assert set(("sm_mhz", "sm_max_mhz", "reasons")) <= set(line["clocks"])


def test_a_wrong_decode_is_caught_by_the_e2e_legs_own_verdict(monkeypatch, capsys):
    """the leg's run-time check has teeth: a decode that is off by one entry on one sender makes it say False"""
    from engine_double import FakeBenchEngine

    class OffByOne(FakeBenchEngine):
        def _decode(self, frame, slot):
            super()._decode(frame, slot)
            if getattr(self, "sabotage", False):
                ack = (self.slots[slot]["type"][1] & 0x0F) == 4
                self.slots[slot]["index"][1][ack] += 1

    monkeypatch.delenv("MRQ_BENCH_FAST", raising=False)
    bench, made = _bench_on_the_double(monkeypatch, OffByOne)
    real = bench.bench_e2e

    def sabotaged(eng, *a, **k):
        eng.sabotage = True
        return real(eng, *a, **k)

    monkeypatch.setattr(bench, "bench_e2e", sabotaged)
    bench.run_ours(_args())
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["e2e"]["equals_wide_form"] is False


@pytest.mark.parametrize("G,R,cfg", [(1500, 7, 5), (1001, 5, 3), (300, 2, 5), (64, 1, 2)])
def test_rehearse_gpu_test_byte_form_decode_and_ticks(monkeypatch, G, R, cfg):
    import test_zz_packed8_gpu as t

    monkeypatch.setattr(t, "Engine", FakeEngine)
    t.test_byte_form_decodes_like_the_host_and_ticks_like_the_oracle(G, R, cfg)


@pytest.mark.parametrize("G,R,cfg", [(1200, 7, 5), (900, 5, 3), (300, 2, 5), (800, 3, 2)])
def test_rehearse_gpu_test_tick_mode_3(monkeypatch, G, R, cfg):
    import test_zz_packed8_gpu as t

    monkeypatch.setattr(t, "Engine", FakeEngine)
    t.test_tick_mode_3_consumes_the_bytes_itself(G, R, cfg)


def test_rehearse_gpu_test_sliding_window(monkeypatch):
    import test_zz_packed8_gpu as t

    monkeypatch.setattr(t, "Engine", FakeEngine)
    t.test_device_window_slides_by_itself_for_hundreds_of_ticks()


def test_rehearse_bench_inbox_forms_replay_the_same_ticks(monkeypatch, capsys):
    """`bench.py --inbox compact | bytes | wide` must drive the engine through exactly the same ticks: same commit indices at
    the end of the timed region, no escapes on the steady-state trace, and each form's byte count in the roofline."""
    import numpy as np

    from engine_double import FakeBenchEngine

    finals = {}
    for inbox in ("wide", "bytes", "compact"):

        class Eng(FakeBenchEngine):
            def timer_stop(self, _inbox=inbox):  # the end of a timed region
                finals[_inbox] = self.o.export()["committed"].copy()
                return super().timer_stop()

        monkeypatch.setenv("MRQ_BENCH_FAST", "1")  # kernels only: no e2e / cpu legs
        bench, made = _bench_on_the_double(monkeypatch, Eng)
        bench.run_ours(_args(inbox=inbox))
        line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
        tb = line["roofline"]["algorithmic_bytes_per_group"]["total"]
        if inbox == "bytes":
            assert "0 escaped" in line["config"]["inbox"] and "tick mode 3" in line["config"]["inbox"] and tb == 173
        elif inbox == "compact":
            assert "tick mode 4" in line["config"]["inbox"] and tb < 60  # one launch per 6 ticks: the state read is amortised
        else:
            assert tb == 217
    assert np.array_equal(finals["wide"], finals["bytes"]) and np.array_equal(finals["wide"], finals["compact"])
    assert (finals["wide"] > bench.steady_state(2048, bench.R, 0, bench.SEED)["committed"]).mean() > 0.9


def test_rehearse_bench_dump_outputs(monkeypatch, capsys, tmp_path):
    """`bench.py --dump-outputs DIR` writes what the last timed tick computed, as float32 / float64 .npy files"""
    import numpy as np

    from engine_double import FakeBenchEngine

    at_stop = []

    class Eng(FakeBenchEngine):
        def timer_stop(self):  # the end of a timed region
            at_stop.append(self.o.export())
            return super().timer_stop()

    monkeypatch.setenv("MRQ_BENCH_FAST", "1")  # the headline leg alone: its last rep is the last timed region
    bench, made = _bench_on_the_double(monkeypatch, Eng)
    bench.run_ours(_args(dump_outputs=str(tmp_path / "dump")))
    capsys.readouterr()
    got = {p.stem: np.load(p) for p in (tmp_path / "dump").glob("*.npy")}
    assert set(got) == {"committed", "out", "term", "role", "last_index", "commit_advance"}
    assert all(a.dtype in (np.float32, np.float64) and a.shape == (2048,) for a in got.values())
    want = at_stop[-1]
    for k in ("committed", "out", "term", "role", "last_index"):
        np.testing.assert_array_equal(got[k], want[k], err_msg=k)
    assert (got["committed"] > bench.steady_state(2048, bench.R, 0, bench.SEED)["committed"]).mean() > 0.9
    assert got["commit_advance"].max() > 0


@pytest.mark.parametrize("G,R,cfg", [(1200, 7, 5), (900, 5, 3), (300, 2, 5), (64, 1, 2)])
def test_rehearse_gpu_test_mode_4_per_tick(monkeypatch, G, R, cfg):
    import test_zz_compact_gpu as t

    monkeypatch.setattr(t, "Engine", FakeEngine)
    t.test_mode_4_per_tick_launches_equal_the_oracle(G, R, cfg)


@pytest.mark.parametrize("G,R,cfg,K", [(900, 5, 5, 6), (600, 7, 5, 5), (500, 3, 2, 8)])
def test_rehearse_gpu_test_mode_4_tick_many(monkeypatch, G, R, cfg, K):
    import test_zz_compact_gpu as t

    monkeypatch.setattr(t, "Engine", FakeEngine)
    t.test_mode_4_tick_many_runs_a_whole_slot_sequence_in_one_launch(G, R, cfg, K, 1)


def test_rehearse_gpu_test_mode_4_interop(monkeypatch):
    import test_zz_compact_gpu as t

    monkeypatch.setattr(t, "Engine", FakeEngine)
    t.test_mode_4_interoperates_with_every_entry_point_that_touches_wide_state()


def _engine_kat_cases():
    import test_zz_kat_gpu as t

    cases = []
    for name in sorted(n for n in dir(t) if n.startswith("test_")):
        fn = getattr(t, name)
        marks = [m for m in getattr(fn, "pytestmark", []) if m.name == "parametrize"]
        if not marks:
            cases.append(pytest.param(name, (), id=name))
            continue
        # expand the parametrize marks the same way pytest does (outer product, innermost mark first)
        import itertools

        names, values = [], []
        for m in marks:
            ns = [x.strip() for x in m.args[0].split(",")]
            names.append(ns)
            values.append([v if isinstance(v, (tuple, list)) and len(ns) > 1 else (v,) for v in m.args[1]])
        for combo in itertools.product(*values):
            kw = {}
            for ns, vs in zip(names, combo):
                kw.update(dict(zip(ns, vs)))
            cases.append(pytest.param(name, tuple(sorted(kw.items())), id=f"{name}-{'-'.join(str(v) for _, v in sorted(kw.items()))}"))
    return cases


@pytest.mark.parametrize("name,kwargs", _engine_kat_cases())
def test_rehearse_engine_kats(monkeypatch, name, kwargs):
    """the bodies of tests/test_zz_kat_gpu.py (upstream's tables through the engine, one message per tick) on the
    engine double: the adapter's way of raising MsgHup / MsgProp through the ABI must reproduce every table row"""
    import test_zz_kat_gpu as t

    monkeypatch.setattr(t, "Engine", FakeEngine)
    getattr(t, name)(**dict(kwargs))
