"""CPU: the reference's two other TEI fan-out scripts run VERBATIM through the `modal` shim (SURVEY.md section 8 f1, a9):

* `06_gpu_and_ml/embeddings/wikipedia/main.py::embed_dataset` (:262-333) -- three volumes mounted at /data, /checkpoint and
  /model, a secret, an async `@modal.method` that fans one map input out into concurrent `/embed` POSTs and returns
  `(chunks, np.ndarray)` (:147-161), `.map(..., order_outputs=False, return_exceptions=True, wrap_return_exceptions=False)`
  (:296-301), an Arrow checkpoint written under the mounted volume + `Volume.commit()` (:203-221);
* `06_gpu_and_ml/embeddings/amazon_embeddings.py` local entrypoint (:50-61) -- `launch_job.remote(...)`, `tei.embed.spawn`
  from a ThreadPoolExecutor and `FunctionCall.object_id` (:104-116), a class with `volumes=`, `retries=`,
  `scaledown_window=` (:180-189);
* `06_gpu_and_ml/embeddings/image_embeddings_infinity.py` local entrypoint (:393-415) -- app-level `volumes=`/`secrets=`,
  `Volume.listdir`, torchvision `read_image` on volume paths (:176-186, 318-320), an `async` `@modal.enter`/`@modal.exit`
  pair around a queue of engines and `embedder.embed.map(chunked(...))` (:288-356, 417-421);
* `06_gpu_and_ml/gpu_snapshot.py` (:25-77) -- `modal deploy` in one process, then the file run as a client in another:
  `modal.Cls.from_name(app_name, "SnapshotEmbedder")`, `@modal.enter(snap=True)`, `enable_memory_snapshot`,
  `experimental_options`, `embedder.run.remote(sentences=[...])`.

`text-embeddings-router` on PATH is the ORACLE-backed stand-in (tests/fake_tei); `datasets` and `huggingface_hub` are the
recording stand-ins under tests/stubs (this box has neither the package nor a network); `infinity_emb` is the ORACLE-backed
stand-in under tests/stubs_infinity (the product's adapter, modal-examples_b200/infinity_emb, has no CPU path and is tested
on the GPU in tests/test_gpu_vit.py); `sentence_transformers` (not installed) is the ORACLE-backed stand-in under tests/stubs_st.
No script is modified."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from oracle.stage_modal_examples import staged

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "modal-examples_b200")
EMB = "06_gpu_and_ml/embeddings/"


def _port_free(port):
    with socket.socket() as s:
        try:
            s.bind(("127.0.0.1", port))
            return True
        except OSError:
            return False


def _env(tmp_path, stubs=("stubs",)):
    state = tmp_path / "state"
    env = dict(os.environ, MODAL_SHIM_STATE=str(state), FAKE_TEI_LOG=str(tmp_path / "tei.jsonl"), FAKE_TEI_LAYERS="1",
               FAKE_HF_LOG=str(tmp_path / "hf.jsonl"), FAKE_DATASETS_DIR=str(tmp_path / "datasets"), HUGGINGFACE_TOKEN="hf_test",
               PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "tests", d) for d in stubs] + [PKG, os.environ.get("PYTHONPATH", "")]),
               PATH=os.path.join(ROOT, "tests", "fake_tei") + os.pathsep + os.environ["PATH"])
    return state, env


def _articles(n, seed):
    rng = np.random.default_rng(seed)
    words = ["embedding", "wikipedia", "volume", "gpu", "batch", "token", "vector", "search", "index", "article", "history", "river"]
    out = []
    for i in range(n):
        text = " ".join(rng.choice(words, size=int(rng.integers(60, 260))))
        out.append({"id": str(100 + i), "url": f"https://example.org/{i}", "title": f"Article {i}", "text": text})
    return out


@pytest.mark.timeout(600)
def test_wikipedia_embed_dataset_runs_unchanged(tmp_path):
    wiki = staged(EMB + "wikipedia/main.py")
    if not _port_free(8000):
        pytest.skip("port 8000 (hard-coded in the reference script) is taken on this box")
    state, env = _env(tmp_path)
    arts = _articles(5, 3)
    ds_dir = state / "volumes" / "embedding-wikipedia" / "wikipedia"  # what the script sees as /data/wikipedia (:22-27,182)
    os.makedirs(ds_dir)
    json.dump(arts, open(ds_dir / "train.json", "w"))
    chunks = [(a["id"], a["url"], a["title"], a["text"][s:s + 512]) for a in arts for s in range(0, len(a["text"]), 512)]
    batch_size = 4  # map inputs of 4 chunks (the script's default is 512 * 50)
    r = subprocess.run([sys.executable, "-m", "modal", "run", wiki + "::embed_dataset", "--down-scale", "1", "--batch-size", str(batch_size)],
                       env=env, capture_output=True, text=True, timeout=540)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
    assert "Webserver ready!" in r.stdout and "Saved checkpoint at /checkpoint/bge-small-en-v1.5-4" in r.stdout
    assert not os.path.exists("/checkpoint") and not os.path.exists("/data/wikipedia"), "mounts must stay virtual"
    # every chunk went to the router exactly once, in POSTs of at most one map input
    reqs = [json.loads(l) for l in open(tmp_path / "tei.jsonl")]
    assert sorted(t for q in reqs for t in q["inputs"]) == sorted(c[3] for c in chunks)
    assert len(reqs) == -(-len(chunks) // batch_size) and max(q["n"] for q in reqs) <= batch_size
    # the checkpoint under the mounted volume holds every chunk with the router's vector for its text
    import pyarrow.parquet as pq

    ck = state / "volumes" / "checkpoint" / "bge-small-en-v1.5-4"
    table = pq.read_table(ck / "data.parquet").to_pylist()
    assert sorted((row["id"], row["text"]) for row in table) == sorted((c[0], c[3]) for c in chunks)
    head = {t: h for q in reqs for t, h in zip(q["inputs"], q["head"])}
    for row in table:
        assert len(row["embedding"]) == 768
        assert np.allclose(row["embedding"][:4], head[row["text"]], rtol=0, atol=1e-7)
        assert abs(float(np.linalg.norm(row["embedding"])) - 1.0) < 1e-4
    # the upload step ran against the (recorded) hub with the secret's token and the checkpoint folder
    hf = [json.loads(l) for l in open(tmp_path / "hf.jsonl")]
    assert [h["call"] for h in hf] == ["create_repo", "upload_folder"] and hf[0]["token"] == "hf_test"
    assert hf[1]["folder_path"] == "/checkpoint/bge-small-en-v1.5-4" and "data.parquet" in hf[1]["files"]


@pytest.mark.timeout(600)
def test_amazon_embeddings_entrypoint_runs_unchanged(tmp_path):
    amazon = staged(EMB + "amazon_embeddings.py")
    if not _port_free(8000):
        pytest.skip("port 8000 (the reference script's default) is taken on this box")
    state, env = _env(tmp_path)
    rng = np.random.default_rng(5)
    rows = [{"asin": f"B{i:05d}", "user_id": f"u{i % 7}", "timestamp": 1_600_000_000 + i, "title": f"review {i}",
             "text": " ".join(rng.choice(["good", "bad", "magazine", "late", "glossy", "renewal"], size=int(rng.integers(5, 200))))}
            for i in range(300)]
    os.makedirs(tmp_path / "datasets")
    json.dump(rows, open(tmp_path / "datasets" / "raw_review_Magazine_Subscriptions.full.json", "w"))
    # expected batches: the script's own generator semantics (:238-268) restated -- chunks of 512 characters, batches of 256
    chunks = [(i, k, d["asin"], d["user_id"], d["timestamp"], d["title"], d["text"][s:s + 512])
              for i, d in enumerate(rows) for k, s in enumerate(range(0, len(d["text"]), 512))]
    n_batches = -(-len(chunks) // 256)
    out_path = "/tmp/embeddings-example-fc-ids.json"  # written by the script's entrypoint (:55-61)
    if os.path.exists(out_path):
        os.remove(out_path)
    r = subprocess.run([sys.executable, "-m", "modal", "run", "--detach", amazon, "--dataset-subset", "raw_review_Magazine_Subscriptions",
                        "--down-scale", "1"], env=env, capture_output=True, text=True, timeout=540)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
    assert "Inference server ready!" in r.stdout and "output handles saved to" in r.stdout
    ids = json.load(open(out_path))
    os.remove(out_path)
    assert len(ids) == n_batches and len(set(ids)) == n_batches and all(i.startswith("fc-") for i in ids)
    # image-build steps are recorded, never executed in-box (`run_function(download_model, volumes=...)`, :128-131,157-166)
    assert not os.path.exists(tmp_path / "hf.jsonl")
    # every spawned batch reached the router before the app exited (the shim drains spawned calls on exit)
    reqs = [json.loads(l) for l in open(tmp_path / "tei.jsonl")]
    assert sorted(q["n"] for q in reqs) == sorted([256] * (len(chunks) // 256) + ([len(chunks) % 256] if len(chunks) % 256 else []))
    assert sorted(t for q in reqs for t in q["inputs"]) == sorted(c[-1] for c in chunks)


@pytest.mark.timeout(600)
def test_image_embeddings_infinity_entrypoint_runs_unchanged(tmp_path):
    infinity = staged(EMB + "image_embeddings_infinity.py")
    pytest.importorskip("torchvision")
    from PIL import Image

    state, env = _env(tmp_path, stubs=("stubs_infinity",))  # ahead of the product's adapter on the path
    env["FAKE_INFINITY_LOG"] = str(tmp_path / "infinity.jsonl")
    env["FAKE_INFINITY_LAYERS"] = "1"
    # the volume already holds the preprocessed JPEGs `catalog_jpegs` would have written (:168-186): no dataset download
    img_dir = state / "volumes" / "example-embedding-data" / "extracted" / "microsoft" / "cats_vs_dogs"
    os.makedirs(img_dir)
    rng = np.random.default_rng(9)
    n = 7
    for i in range(n):
        Image.fromarray(rng.integers(0, 256, (224, 224, 3), dtype=np.uint8)).save(img_dir / f"img{i:07d}.jpg", quality=95)
    r = subprocess.run([sys.executable, "-m", "modal", "run", infinity], env=env, capture_output=True, text=True, timeout=540)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
    assert f"Found {n} JPEGs in the Volume." in r.stdout and "Loading 4 models..." in r.stdout
    assert f"n_ims={n}::concurrency=4" in r.stdout and "Embedding-only throughput (avg)" in r.stdout
    assert not os.path.exists("/data/extracted"), "mounts must stay virtual"
    calls = [json.loads(l) for l in open(tmp_path / "infinity.jsonl")]
    assert [c["n"] for c in calls] == [n] and all(sz == [224, 224] for sz in calls[0]["sizes"])  # one map input of <= 100 images


@pytest.mark.timeout(600)
def test_gpu_snapshot_deploy_then_client_process(tmp_path):
    snapshot = staged("06_gpu_and_ml/gpu_snapshot.py")
    state, env = _env(tmp_path, stubs=("stubs_st",))
    env["FAKE_ST_LAYERS"] = "1"
    # a client before any deployment: the script's own NotFoundError branch (:73-77)
    r = subprocess.run([sys.executable, snapshot], env=env, capture_output=True, text=True, timeout=300)
    # (the app object exists in the client process because the client IS the app's file; it must still run)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    r = subprocess.run([sys.executable, "-m", "modal", "deploy", snapshot], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "deployed app 'example-gpu-snapshot'" in r.stdout, (r.stdout[-2000:], r.stderr[-3000:])
    reg = json.load(open(state / "deployed.json"))
    assert reg["example-gpu-snapshot"]["path"] == snapshot
    r = subprocess.run([sys.executable, snapshot], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    assert "calling Modal Function" in r.stdout and "loading model" in r.stdout and "snapshotting v1" in r.stdout
    vec = json.loads(r.stdout.strip().splitlines()[-1])
    assert len(vec) == 1 and len(vec[0]) == 768 and abs(float(np.linalg.norm(vec[0])) - 1.0) < 1e-4
    # a different client process (no app object of its own) finds the deployed class through the state directory
    code = ("import json, modal\n"
            "E = modal.Cls.from_name('example-gpu-snapshot', 'SnapshotEmbedder')\n"
            "print(json.dumps(E().run.remote(sentences=['what is the meaning of life?'])))\n")
    r2 = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300, cwd=str(tmp_path))
    assert r2.returncode == 0, (r2.stdout[-2000:], r2.stderr[-3000:])
    assert np.allclose(json.loads(r2.stdout.strip().splitlines()[-1]), vec, atol=1e-6)
    # and an app nobody deployed is NotFoundError
    r3 = subprocess.run([sys.executable, "-c", "import modal\nmodal.Cls.from_name('no-such-app', 'X')"], env=env, capture_output=True, text=True, cwd=str(tmp_path))
    assert r3.returncode != 0 and "NotFoundError" in r3.stderr
