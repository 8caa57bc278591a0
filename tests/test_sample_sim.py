"""The GPU sampler's kernel (csrc/sample.cu) executed on the CPU emulator (tests/cusim) against the UNMODIFIED reference
sampler (src/inference/sampler.cpp; its draws recorded in tests/golden/ref_host.json by tests/golden/make_ref_golden.py) and
our host sampler, on the same logits / settings / seed.  The kernel follows the reference's float operations in order, so draws
must be identical whenever no ties straddle the top-k cut."""
import ctypes as C
import json
import subprocess
from pathlib import Path

import numpy as np
import pytest

from ntransformer_b200._lib import lib

ROOT = Path(__file__).resolve().parent.parent
SIM_DIR = ROOT / "tests" / "cusim"
SIG = [C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_float, C.c_float, C.c_int, C.c_void_p, C.c_int, C.c_ulonglong]


@pytest.fixture(scope="module")
def sim():
    r = subprocess.run(["make", "-C", str(SIM_DIR)], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.fail("tests/cusim does not build:\n" + r.stderr[-3000:])
    s = C.CDLL(str(SIM_DIR / "_sim" / "libsample_sim.so"))
    s.sample_sim.argtypes = SIG
    return s


def args_for(logits, temperature, top_k, top_p, penalty, window, recent, seed):
    return (logits.ctypes.data_as(C.c_void_p), len(logits), temperature, top_k, top_p, penalty, window,
            recent.ctypes.data_as(C.c_void_p) if len(recent) else None, len(recent), seed)


def draw_cases():
    """Arguments of sample_sim / ref_sample_token / nt_sample_token (test_draws_match_the_reference_sampler)."""
    rng = np.random.default_rng(11)
    for trial in range(40):
        n = int(rng.choice([300, 2048, 5000, 33000]))
        logits = (rng.standard_normal(n) * rng.choice([0.5, 2.0, 6.0])).astype(np.float32)
        temperature = float(rng.choice([0.3, 0.7, 1.0, 1.5]))
        top_k = int(rng.choice([1, 2, 5, 40, 64, 100, 1000 if n > 1024 else 200]))
        top_p = float(rng.choice([0.0, 0.5, 0.9, 0.95, 1.0]))
        penalty = float(rng.choice([1.0, 1.1, 1.5]))
        window = int(rng.choice([0, 4, 64]))
        recent = rng.integers(-1, n + 1, size=int(rng.integers(0, 90))).astype(np.int32)
        if trial % 5 == 0 and len(recent) > 3:
            recent[-1] = recent[-2] = int(np.argmax(logits))             # the top token twice in the window: penalised twice
        seed = int(rng.integers(0, 2**31))
        yield logits, temperature, top_k, top_p, penalty, window, recent, seed


def test_draws_match_the_reference_sampler(sim):
    wants = json.loads((ROOT / "tests" / "golden" / "ref_host.json").read_text())["sample_sim"]
    checked = 0
    for trial, (case, want) in enumerate(zip(draw_cases(), wants, strict=True)):
        logits, temperature, top_k, top_p, penalty, window, recent, seed = case
        a = args_for(*case)
        got = sim.sample_sim(*a)
        ours = lib().nt_sample_token(*a)
        assert got == want == ours, (trial, len(logits), temperature, top_k, top_p, penalty, window, seed, got, want, ours)
        checked += 1
    assert checked == 40


def test_uncovered_settings_are_declined(sim):
    logits = np.zeros(100, dtype=np.float32)
    none = np.zeros(0, dtype=np.int32)
    for temperature, top_k in ((0.0, 40), (0.7, 0), (0.7, 100), (0.7, 2000), (0.7, -1)):
        assert sim.sample_sim(*args_for(logits, temperature, top_k, 0.9, 1.0, 0, none, 1)) == -1


def test_ties_at_the_cut_pick_the_lowest_ids_and_stay_valid(sim):
    """All-equal logits, and a block of equal values straddling the top-k cut: the reference's partial_sort leaves the choice
    among ties unspecified; the kernel takes the lowest token ids.  The draw must come from exactly that candidate set with the
    reference's probabilities (uniform here)."""
    n, k = 3000, 7
    none = np.zeros(0, dtype=np.int32)
    logits = np.full(n, 1.25, dtype=np.float32)
    seen = set()
    for seed in range(60):
        t = sim.sample_sim(*args_for(logits, 0.8, k, 1.0, 1.0, 0, none, seed))
        assert 0 <= t < k, t                                              # lowest ids win the tie
        seen.add(t)
    assert len(seen) >= 5                                                 # and the draw is spread over them
    logits = np.linspace(-3, 3, n).astype(np.float32)
    logits[100:140] = 9.0                                                 # 40 equal maxima, k = 7 of them survive
    logits[2999] = 10.0                                                   # one strictly larger candidate
    picks = {sim.sample_sim(*args_for(logits, 1.0, k, 1.0, 1.0, 0, none, seed)) for seed in range(80)}
    assert picks <= ({2999} | set(range(100, 106))) and 2999 in picks
