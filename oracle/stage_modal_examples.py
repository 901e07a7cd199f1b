"""Stages the upstream modal-examples scripts that tests run verbatim through the `modal` shim (tests/test_shim.py,
tests/test_graded_script.py, tests/test_sibling_scripts.py) under oracle/_ref/modal-examples/.  Their source is not part of
this repository: build() copies them from a modal-examples checkout -- $MODAL_EXAMPLES_DIR, else /root/reference -- and,
without one, keeps a copy staged earlier.  A test that needs a script that was never staged fails (see `staged`)."""
import os
import shutil

STAGED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "modal-examples")
SCRIPTS = [
    "01_getting_started/hello_world.py",
    "01_getting_started/generators.py",
    "03_scaling_out/dynamic_batching.py",
    "08_advanced/hello_world_async.py",
    "06_gpu_and_ml/gpu_snapshot.py",
    "06_gpu_and_ml/embeddings/text_embeddings_inference.py",
    "06_gpu_and_ml/embeddings/amazon_embeddings.py",
    "06_gpu_and_ml/embeddings/image_embeddings_infinity.py",
    "06_gpu_and_ml/embeddings/qdrant.py",
    "06_gpu_and_ml/embeddings/wikipedia/main.py",
    "06_gpu_and_ml/embeddings/wikipedia/download.py",
]


def stage() -> bool:
    """Copies SCRIPTS from the checkout into STAGED; False (and nothing touched) when there is no complete checkout."""
    src = os.environ.get("MODAL_EXAMPLES_DIR") or "/root/reference"
    if not all(os.path.isfile(os.path.join(src, rel)) for rel in SCRIPTS):
        return False
    for rel in SCRIPTS:
        dst = os.path.join(STAGED, rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        shutil.copyfile(os.path.join(src, rel), dst)
    return True


def staged(rel: str) -> str:
    """Path of the staged copy of upstream script `rel`; raises when build() has not staged it."""
    path = os.path.join(STAGED, rel)
    if not os.path.isfile(path):
        raise FileNotFoundError(f"{path} is not staged: run build() with a modal-examples checkout in $MODAL_EXAMPLES_DIR")
    return path
