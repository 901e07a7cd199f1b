"""CPU: the in-box ``modal`` shim against the reference's pinned plumbing answers (SURVEY.md §8c):
hello_world sums, generators, spawn/gather + exception identity, batched ASCII round trip, async twins."""
import asyncio
import os
import subprocess
import sys
import threading
import time

import pytest

import modal
from oracle.stage_modal_examples import staged

PKG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "modal-examples_b200")


def make_app():
    app = modal.App("test-plumbing")

    @app.function()
    def f(i):
        return i * i

    @app.function()
    def where():
        return modal.is_local()

    @app.function()
    def gen(n):
        for i in range(n):
            yield i

    @app.function()
    def boom(x):
        if x == 3:
            raise ValueError("custom error")
        return x

    @app.function()
    async def af(i):
        await asyncio.sleep(0.001)
        return i * i

    return app, f, where, gen, boom, af


def test_local_remote_map_known_answers():
    app, f, where, *_ = make_app()
    with app.run():
        assert f.local(1000) == f.remote(1000) == 1_000_000  # hello_world.py:60-63
        assert sum(f.map(range(200))) == 2_646_700           # hello_world.py:66-70
        assert sum(f.map(range(1000))) == 332_833_500        # BASELINE config #1
        assert list(f.map(range(20))) == [i * i for i in range(20)]  # ordered by default
        assert sorted(f.map(range(50), order_outputs=False)) == sorted(i * i for i in range(50))
        assert modal.is_local() is True and where.remote() is False and where.local() is True


def test_starmap_for_each_kwargs_and_zip():
    app = modal.App("t2")
    seen = []

    @app.function()
    def add(a, b, scale=1):
        return (a + b) * scale

    @app.function()
    def note(x, tag=""):
        seen.append((x, tag))

    assert list(add.starmap([(1, 2), (3, 4)], kwargs={"scale": 10})) == [30, 70]
    assert list(add.map([1, 2, 3], [10, 20, 30])) == [11, 22, 33]  # multiple iterables are zipped (finetune_yolo.py:306)
    note.for_each(range(5), kwargs={"tag": "t"})
    assert sorted(seen) == [(i, "t") for i in range(5)]


def test_map_is_lazy_with_backpressure():
    app = modal.App("t3")
    release = threading.Event()

    @app.function(max_containers=2)
    def slow(i):
        release.wait(5)
        return i

    pulled = []

    def inputs():
        for i in range(10_000):
            pulled.append(i)
            yield i

    it = slow.map(inputs())
    t = threading.Thread(target=lambda: next(it))
    t.start()
    time.sleep(0.3)
    assert 0 < len(pulled) < 1000, "generator input must be consumed lazily, bounded by the in-flight window"
    release.set()
    t.join()


def test_generators_remote_gen():
    _, _, _, gen, *_ = make_app()
    assert list(gen.remote_gen(10)) == list(range(10))  # generators.py:13-22

    async def run():
        return [x async for x in gen.remote_gen.aio(5)]

    assert asyncio.run(run()) == [0, 1, 2, 3, 4]


def test_spawn_gather_and_exception_identity():
    app = modal.App("t4")

    @app.function()
    def step1(word):
        return word

    @app.function()
    def step2(n):
        return n

    @app.function()
    def bad():
        raise ValueError("custom error")

    a, b = step1.spawn("bar"), step2.spawn(4)
    assert modal.FunctionCall.gather(a, b) == ["bar", 4]  # parallel_execution.py:41-42
    with pytest.raises(ValueError, match="custom error"):  # parallel_execution.py:44-48
        modal.FunctionCall.gather(step1.spawn("x"), bad.spawn())
    call = step2.spawn(7)
    assert modal.FunctionCall.from_id(call.object_id).get(timeout=5) == 7  # poll_delayed_result.py:54-56


def test_get_timeout():
    app = modal.App("t5")
    ev = threading.Event()

    @app.function()
    def wait():
        ev.wait(5)
        return 1

    c = wait.spawn()
    with pytest.raises(TimeoutError):
        c.get(timeout=0.05)
    ev.set()
    assert c.get(timeout=5) == 1


def test_return_exceptions_and_raise():
    _, _, _, _, boom, _ = make_app()
    out = list(boom.map(range(5), return_exceptions=True))
    assert [o for o in out if not isinstance(o, Exception)] == [0, 1, 2, 4]
    assert isinstance(out[3], ValueError) and str(out[3]) == "custom error"
    with pytest.raises(ValueError, match="custom error"):
        list(boom.map(range(5)))
    boom.for_each(range(5), ignore_exceptions=True)  # inference_map.py:36


def test_async_twins():
    _, f, _, _, _, af = make_app()

    async def run():
        r = await f.remote.aio(12)
        s = 0
        async for x in f.map.aio(range(20)):  # hello_world_async.py:44-49
            s += x
        t = sum([x async for x in af.map.aio(range(20))])
        c = await f.spawn.aio(5)
        g = await modal.FunctionCall.gather.aio(c)
        return r, s, t, g

    assert asyncio.run(run()) == (144, 2470, 2470, [25])
    assert af.remote(9) == 81 and sum(af.map(range(20))) == 2470


def test_spawn_from_user_thread_pool():
    # amazon_embeddings.py:104-116 submits spawns from a ThreadPoolExecutor
    from concurrent.futures import ThreadPoolExecutor

    _, f, *_ = make_app()
    with ThreadPoolExecutor(8) as ex:
        calls = list(ex.map(f.spawn, range(64)))
    assert [c.get() for c in calls] == [i * i for i in range(64)]


def test_batched_ascii_round_trip():
    app = modal.App("t6")

    @app.function()
    @modal.batched(max_batch_size=4, wait_ms=50)
    def to_chr(codes: list[int]) -> list[str]:
        assert isinstance(codes, list) and 1 <= len(codes) <= 4
        return [chr(c) for c in codes]

    assert list(to_chr.map(range(33, 39))) == ["!", '"', "#", "$", "%", "&"]  # dynamic_batching.py:81-89


def test_cls_lifecycle_and_parameters():
    app = modal.App("t7")
    events = []

    @app.cls(gpu="B200:2", max_containers=3)
    @modal.concurrent(max_inputs=4)
    class Model:
        size: str = modal.parameter(default="base")

        @modal.enter()
        def load(self):
            events.append(("enter", self.size))
            self.w = {"base": 1, "large": 10}[self.size]

        @modal.enter()
        async def aload(self):
            events.append(("aenter", self.size))

        @modal.method()
        def run(self, x):
            return x * self.w

        @modal.method()
        async def arun(self, x):
            await asyncio.sleep(0)
            return -x * self.w

        @modal.exit()
        def bye(self):
            events.append(("exit", self.size))

    with app.run():
        m = Model()
        assert events == []  # lazy
        assert m.run.remote(3) == 3 and list(m.run.map([1, 2])) == [1, 2] and m.run.local(5) == 5
        assert sorted(m.arun.map([1, 2], order_outputs=False)) == [-2, -1]
        assert Model(size="large").run.remote(3) == 30
        assert events.count(("enter", "base")) == 1 and ("aenter", "base") in events
        assert Model.with_options(gpu="H100").options["gpu"] == "H100"
    assert ("exit", "base") in events and ("exit", "large") in events


def test_image_is_inert_but_env_applies():
    ran = []
    img = (modal.Image.from_registry("ghcr.io/x:1", add_python="3.10").dockerfile_commands("ENTRYPOINT []")
           .run_function(lambda: ran.append(1), gpu="A10G").uv_pip_install("httpx").env({"SHIM_TEST_ENV": "yes"}))
    assert ran == []  # run_function must NOT execute (text_embeddings_inference.py:70 would spawn TEI)
    with img.imports():
        import definitely_not_installed_module  # noqa: F401
    app = modal.App("t8", image=img)

    @app.function()
    def env():
        return os.environ.get("SHIM_TEST_ENV"), os.environ.get("MODAL_TASK_ID", "").startswith("ta-")

    assert env.remote() == ("yes", True)


def test_gpu_grammar_and_misc_surface():
    from modal.gpu import parse_gpu_count

    assert [parse_gpu_count(x) for x in ["H100", "a10g", "A100-80GB", "H100:2", "B200:8", "H100!", "any", ["h100", "a100", "any"],
                                          modal.gpu.L40S(count=4), None, False]] == [1, 1, 1, 2, 8, 1, 1, 1, 4, 0, 0]
    assert isinstance(modal.config._profile, str) and isinstance(modal.config.config["environment"], str)
    with pytest.raises(modal.exception.NotFoundError):
        modal.Cls.from_name("nope", "Nope")
    vol = modal.Volume.from_name("shim-test-vol", create_if_missing=True)
    vol.commit(); vol.reload()
    d = modal.Dict.from_name("shim-d", create_if_missing=True)
    d["k"] = 1
    assert d.get("k") == 1
    q = modal.Queue.from_name("shim-q", create_if_missing=True)
    q.put_many([1, 2, 3])
    assert q.get_many(10) == [1, 2, 3]
    assert modal.Retries(max_retries=3).max_retries == 3 and modal.Period(days=1).days == 1


def test_retries():
    app = modal.App("t9")
    n = {"c": 0}

    @app.function(retries=modal.Retries(max_retries=3, initial_delay=0.0))
    def flaky():
        n["c"] += 1
        if n["c"] < 3:
            raise RuntimeError("transient")
        return n["c"]

    assert flaky.remote() == 3


def _cli(*args, cwd=None):
    env = dict(os.environ, PYTHONPATH=PKG + os.pathsep + os.environ.get("PYTHONPATH", ""))
    return subprocess.run([sys.executable, "-m", "modal", *args], capture_output=True, text=True, env=env, cwd=cwd, timeout=120)


def test_cli_runs_entrypoint_with_kebab_options(tmp_path):
    script = tmp_path / "cli_demo.py"
    script.write_text(
        "import modal\napp = modal.App('cli-demo')\n"
        "@app.function()\ndef sq(x: int = 3):\n    return x * x\n"
        "@app.local_entrypoint()\ndef main(n_items: int = 4, loud: bool = False, name: str = 'w'):\n"
        "    print('SUM', sum(sq.map(range(n_items))), loud, name)\n")
    r = _cli("run", str(script), "--n-items", "10", "--loud", "--name", "z")
    assert r.returncode == 0, r.stderr
    assert "SUM 285 True z" in r.stdout
    r = _cli("run", f"{script}::sq", "--x", "7")
    assert r.returncode == 0 and r.stdout.strip().endswith("49")


@pytest.mark.parametrize("rel,expect", [
    ("01_getting_started/hello_world.py", "2646700"),
    ("01_getting_started/generators.py", "9"),
    ("08_advanced/hello_world_async.py", "2470"),
    ("03_scaling_out/dynamic_batching.py", "ASCII codes: [33, 34, 35, 36, 37, 38]"),
])
def test_reference_scripts_run_unchanged(rel, expect):
    r = _cli("run", staged(rel))
    assert r.returncode == 0, r.stderr[-2000:]
    assert expect in r.stdout


def test_reference_hot_path_scripts_import_unchanged():
    """The reference's own smoke test is `importlib.import_module` of every example
    (internal/examples_test.py:39-41); here over the embeddings directory with the shim as `modal`."""
    import importlib.util

    for fn in ["text_embeddings_inference.py", "amazon_embeddings.py", "image_embeddings_infinity.py", "qdrant.py"]:
        spec = importlib.util.spec_from_file_location("refmod_" + fn[:-3], staged("06_gpu_and_ml/embeddings/" + fn))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        assert any(isinstance(v, modal.App) for v in vars(mod).values())
