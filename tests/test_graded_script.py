"""CPU: the graded reference script runs VERBATIM through the `modal` shim --
`modal run 06_gpu_and_ml/embeddings/text_embeddings_inference.py::embed_dataset` (:141-169): the volume at
/data (virtual mount, nothing created under /), `spawn_server()` Popen + TCP readiness (:37-51), the `@app.cls` /
`@modal.concurrent` / `@modal.enter` / async `@modal.method` class (:79-104), `generate_batches()` (batches of 32, remainder
dropped, :156-163) and `model.embed.map(..., order_outputs=False)` (:167).  The `text-embeddings-router` on PATH is the
ORACLE-backed stand-in under tests/fake_tei (this box has no GPU and the product router has no CPU path); the product
router is driven the same way on the GPU in tests/test_gpu_router.py."""
import json
import os
import socket
import subprocess
import sys

import pytest

from oracle.stage_modal_examples import staged

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "modal-examples_b200")


def _port_free(port):
    with socket.socket() as s:
        try:
            s.bind(("127.0.0.1", port))
            return True
        except OSError:
            return False


@pytest.mark.timeout(600)
def test_text_embeddings_inference_embed_dataset_runs_unchanged(tmp_path):
    script = staged("06_gpu_and_ml/embeddings/text_embeddings_inference.py")
    if not _port_free(8000):
        pytest.skip("port 8000 (hard-coded in the reference script) is taken on this box")
    state = tmp_path / "state"
    env = dict(os.environ, PYTHONPATH=PKG + os.pathsep + os.environ.get("PYTHONPATH", ""), MODAL_SHIM_STATE=str(state),
               PATH=os.path.join(ROOT, "tests", "fake_tei") + os.pathsep + os.environ["PATH"], FAKE_TEI_LOG=str(tmp_path / "tei.jsonl"),
               FAKE_TEI_LAYERS="1")  # (httpx default timeout in the reference script is 5 s: keep the CPU stand-in quick)
    rows = 70  # -> 2 batches of 32, the last 6 items are dropped by generate_batches (:156-163)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "make_hn_dataset.py"), "--rows", str(rows)], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    data = json.load(open(state / "volumes" / "tei-hn-data" / "dataset.jsonl"))
    assert len(data) == rows and not os.path.exists("/data/dataset.jsonl")
    r = subprocess.run([sys.executable, "-m", "modal", "run", script + "::embed_dataset"], env=env, capture_output=True, text=True, timeout=540)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
    assert "Webserver ready!" in r.stdout
    reqs = [json.loads(l) for l in open(tmp_path / "tei.jsonl")]
    assert [q["n"] for q in reqs] == [32, 32], "two full batches, remainder dropped"
    seen = sorted(t for q in reqs for t in q["inputs"])
    assert seen == sorted(t for _, t in data[:64])
    assert all(len(q["head"]) == 32 for q in reqs)
