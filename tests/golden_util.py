"""Load tests/golden/*.json.gz and regenerate their inputs; the reference's recorded answers."""
import gzip
import hashlib
import json
import re
import tempfile
from pathlib import Path

import numpy as np

import checker as C
from dump1090_b200 import synth

GOLDEN_DIR = Path(__file__).resolve().parent / "golden"
NAMES = sorted(p.name[: -len(".json.gz")] for p in GOLDEN_DIR.glob("*.json.gz"))
ANSWERS_PATH = GOLDEN_DIR / "reference_answers.json"
_answers = None


def digest(obj) -> str:
    """sha256 of an answer: raw bytes as they are, anything else as canonical JSON."""
    if isinstance(obj, np.ndarray):
        obj = np.ascontiguousarray(obj).tobytes()
    if not isinstance(obj, bytes):
        obj = json.dumps(obj, sort_keys=True, separators=(",", ":")).encode()
    return hashlib.sha256(obj).hexdigest()


def answer(key):
    """What the unmodified reference answered for test case `key` (recorded by
    tests/golden/make_reference_answers.py): the answer itself or its digest()."""
    global _answers
    if _answers is None:
        _answers = json.loads(ANSWERS_PATH.read_text())
    return _answers[key]


def write_answer(value, stream) -> None:
    """An answer in a form two of them can be diffed in: bytes as they are, anything else as indented JSON."""
    if isinstance(value, np.ndarray):
        value = value.tolist()
    stream.write(value if isinstance(value, bytes) else (json.dumps(value, indent=1, sort_keys=True) + "\n").encode())


def assert_answer(key, got) -> None:
    """`got` must be the reference's answer for `key`, which is recorded as its digest().  On a mismatch
    `got` is written to a file, to be diffed with what `make_reference_answers.py --show KEY` prints."""
    if digest(got) == answer(key):
        return
    path = Path(tempfile.gettempdir()) / ("answer_" + re.sub(r"[^A-Za-z0-9_.-]+", "_", key))
    with open(path, "wb") as f:
        write_answer(got, f)
    raise AssertionError(f"{key}: differs from the reference's recorded answer. This run's answer is in {path}; "
                         f"`python tests/golden/make_reference_answers.py --show '{key}'` prints the reference's "
                         "(oracle/_ref must be built)")


def load(name):
    with gzip.open(GOLDEN_DIR / f"{name}.json.gz", "rb") as f:
        return json.loads(f.read().decode())


def make_input(doc) -> np.ndarray:
    if doc["generator"] == "modes1":
        data = C.modes1()
    else:
        data = getattr(synth, doc["generator"])(**doc["args"])
    assert data.size == doc["nbytes"]
    assert hashlib.sha256(data.tobytes()).hexdigest() == doc["sha256"], "golden input drifted"
    return data


def cases():
    for name in NAMES:
        doc = load(name)
        for cid, case in doc["cases"].items():
            yield name, cid


CASES = list(cases())
